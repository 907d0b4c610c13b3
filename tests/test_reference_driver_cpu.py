"""The multi-step reference that tests/test_gpu_train_step.py holds the fused training step to -- oracle gradients
(`train_step_grads`) plus the float64 Adam (`adam_step_f64`), driven by `train_steps` -- checked here against an
independent formulation: torch autograd through the coalesced COO operators and torch.optim.Adam
(`TorchCpuBaseline`).  A wrong reference would otherwise bless a wrong kernel."""
import numpy as np
import pytest
import torch

import credgcn_oracle as orc
from conftest import rel_err


def _tiny(tag):
    from credgcn import synth
    sg = synth.make_graph("C1", num_users=60, num_items=45, num_edges=600, duplicate_edges=20)
    ops = orc.Operators(sg.train_edges, sg.num_users, sg.num_items, sg.cred, tag)
    rng = np.random.default_rng(5)
    e0u = (rng.standard_normal((sg.num_users, 16)) * 0.3).astype(np.float32)
    e0i = (rng.standard_normal((sg.num_items, 16)) * 0.3).astype(np.float32)
    u, i = sg.train_edges[0].astype(np.int64), sg.train_edges[1].astype(np.int64)
    batches = []
    for t in range(3):
        sel = rng.integers(0, u.size, size=50 + 7 * t)
        batches.append((u[sel], i[sel], rng.integers(0, sg.num_items, size=sel.size)))
    return sg, ops, e0u, e0i, batches


@pytest.mark.parametrize("tag,fair", [("v2", 0.0), ("cu", 0.05)])
def test_reference_driver_matches_torch_autograd_and_adam(tag, fair):
    sg, ops, e0u, e0i, batches = _tiny(tag)
    order = "gs" if tag == "v2" else "jacobi"
    pop = (ops.deg_i / max(float(ops.deg_i.max()), 1.0)).astype(np.float32) if fair else None
    lr, reg = 1e-2, 1e-3
    ref = orc.train_steps(ops, e0u, e0i, batches, 2, order, reg, fair, pop, lr=lr)
    base = orc.TorchCpuBaseline(ops, e0u, e0i, 2, order, lr=lr)
    pop_t = None if pop is None else torch.from_numpy(pop)
    for t, (users, pos, neg) in enumerate(batches):
        p_before = (base.eu.detach().clone(), base.ei.detach().clone())
        loss = base.step(users, pos, neg, reg, fair, pop_t)
        r = ref[t]
        assert abs(loss - r["loss"]) <= 1e-5 * abs(r["loss"]), (t, loss, r["loss"])
        assert rel_err(base.eu.grad.numpy(), r["g_u"]) < 1e-5
        assert rel_err(base.ei.grad.numpy(), r["g_i"]) < 1e-5
        # the Adam update itself, element by element: both sides step from (nearly) the same parameters with (nearly)
        # the same gradients, so the updates agree to the gradient error -- where a gradient is not near zero (Adam
        # normalises a gradient, and the update of a near-zero one has an arbitrary size)
        for w, got, p0, g in ((r["p_u"], base.eu, p_before[0], r["g_u"]), (r["p_i"], base.ei, p_before[1], r["g_i"])):
            d_ref = w.astype(np.float64) - p0.numpy()
            d_got = got.detach().numpy().astype(np.float64) - p0.numpy()
            big = np.abs(g) > 1e-3 * np.abs(g).max()
            assert big.mean() > 0.5
            assert np.all(np.abs(d_got - d_ref)[big] <= 1e-3 * lr), (t, float(np.abs(d_got - d_ref)[big].max()))
            assert np.all(np.abs(d_got) <= lr * 1.01) and np.all(np.abs(d_ref) <= lr * 1.01)
    assert rel_err(base.eu.detach().numpy(), ref[-1]["p_u"]) < 1e-3 * lr


def test_adam_step_f64_is_torch_adam():
    """adam_step_f64 == torch.optim.Adam run in float64, over steps with zero, tiny and large gradients."""
    rng = np.random.default_rng(0)
    p0 = rng.standard_normal(400)
    q = torch.nn.Parameter(torch.tensor(p0))
    opt = torch.optim.Adam([q], lr=3e-3)
    p, m, v = p0.copy(), np.zeros(400), np.zeros(400)
    for t in range(1, 41):
        g = rng.standard_normal(400) * np.array([0.0, 1e-8, 1.0, 1e4])[np.arange(400) % 4]
        if 10 <= t < 20:
            g[:200] = 0.0
        q.grad = torch.tensor(g)
        opt.step()
        p, m, v = orc.adam_step_f64(p, g, m, v, t, lr=3e-3)
        np.testing.assert_allclose(p - p0, q.detach().numpy() - p0, rtol=1e-12, atol=1e-15)
