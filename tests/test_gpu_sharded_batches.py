"""The device side of the user-sharded epoch loop on one GPU: batch selection (cgx_batch_select) against NumPy, and
the count / slot / row-base arguments of the sampler, the scatter plan, the fused loss, the batch frontier and the
sampled-evaluation candidates against the same kernels on the whole or truncated batch, bit for bit."""
import pathlib
import sys

import numpy as np
import pytest
import torch

ROOT = pathlib.Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))
pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def cg():
    from credgcn import _lib, evaluate, graph, model, sampler, synth
    sg = synth.make_graph("C1", num_users=700, num_items=500, num_edges=30_000, duplicate_edges=20)
    gr = graph.build_graph(sg.train_edges, sg.num_users, sg.num_items, sg.cred, "v2", DEV)
    return dict(lib=_lib, ev=evaluate, graph=graph, m=model, smp=sampler, sg=sg, gr=gr)


def _select(cg, perm, step, B, lo, hi):
    lib = cg["lib"]
    d = torch.device(DEV)
    perm_d = torch.as_tensor(perm, dtype=torch.int64, device=d)
    step_d = torch.tensor([step], dtype=torch.int64, device=d)
    users = torch.full((B,), -7, dtype=torch.int64, device=d)
    slots = torch.full((B,), -7, dtype=torch.int64, device=d)
    cnt, tot = torch.full((1,), -7, dtype=torch.int64, device=d), torch.full((1,), -7, dtype=torch.int64, device=d)
    lib.check(lib.lib().cgx_batch_select(lib.ptr(perm_d), perm_d.numel(), lib.ptr(step_d), B, lo, hi, lib.ptr(users),
                                         lib.ptr(slots), lib.ptr(cnt), lib.ptr(tot), lib.stream_ptr(d)))
    c = int(cnt.item())
    return users.cpu().numpy(), slots.cpu().numpy(), c, int(tot.item())


@pytest.mark.parametrize("n_train,B", [(1000, 256), (1024, 256), (100, 4096), (9000, 4096), (4097, 1)])
def test_batch_select_matches_numpy(cg, n_train, B):
    rng = np.random.default_rng(n_train + B)
    U = n_train + 50
    perm = rng.permutation(U)[:n_train].astype(np.int64)
    steps = -(-n_train // B)
    ranges = [(0, U), (0, 0), (U // 3, U // 3 + 40), (perm[0], perm[0] + 1), (U - 1, U), (10, U // 2)]
    for s in list(range(min(steps, 3))) + [steps - 1, steps]:          # the tail batch, and one past the epoch
        batch = perm[s * B:(s + 1) * B]
        for lo, hi in ranges:
            users, slots, c, tot = _select(cg, perm, s, B, lo, hi)
            keep = np.flatnonzero((batch >= lo) & (batch < hi))
            assert tot == len(batch)
            assert c == keep.size
            np.testing.assert_array_equal(users[:c], batch[keep] - lo)
            np.testing.assert_array_equal(slots[:c], keep)
            assert (users[c:] == -7).all() and (slots[c:] == -7).all()     # padding is not written


def _sample(cg, users, tick, slots=None, count=None, fill=-5):
    smp = cg["smp"].TripleSampler(cg["gr"], 0.7, 0.75, 50, seed=42)
    B = users.numel()
    out = (torch.full((B,), fill, dtype=torch.int64, device=DEV), torch.full((B,), fill, dtype=torch.int64, device=DEV))
    t = torch.tensor([tick], dtype=torch.int64, device=DEV)
    return smp.sample(users, offset=0, offset_dev=t, slots=slots, count=count, out=out)


def test_sampler_slots_and_count_equal_whole_batch(cg):
    gr = cg["gr"]
    train_users = torch.nonzero(gr.deg_u > 0).flatten()
    whole = train_users[:512]
    pw, nw = _sample(cg, whole, 3)
    sel = torch.tensor([3, 4, 17, 100, 101, 511], dtype=torch.int64, device=DEV)
    cap = 16
    users = torch.full((cap,), 10**9, dtype=torch.int64, device=DEV)         # garbage ids in the padding
    users[: sel.numel()] = whole[sel]
    slots = torch.full((cap,), -1, dtype=torch.int64, device=DEV)
    slots[: sel.numel()] = sel
    count = torch.tensor([sel.numel()], dtype=torch.int64, device=DEV)
    p, n = _sample(cg, users, 3, slots, count)
    assert torch.equal(p[: sel.numel()], pw[sel]) and torch.equal(n[: sel.numel()], nw[sel])
    assert (p[sel.numel():] == -5).all() and (n[sel.numel():] == -5).all()
    # without slots / count: the old call
    p0, n0 = _sample(cg, whole, 3, None, None)
    assert torch.equal(p0, pw) and torch.equal(n0, nw)


def _loss_call(cg, users, pos, neg, count=None, total=None, batch_total=0, fair=0.0, pop=None):
    m, gr = cg["m"], cg["gr"]
    torch.manual_seed(1)
    d = 64
    f_u = torch.randn(gr.num_users, d, device=DEV) * 0.3
    f_i = torch.randn(gr.num_items, d, device=DEV) * 0.3
    e_u = torch.randn(gr.num_users, d, device=DEV) * 0.3
    e_i = torch.randn(gr.num_items, d, device=DEV) * 0.3
    plan = m.bpr_plan(gr, users, pos, neg, count=count)
    loss, g_u, g_i, er, ec = m.bpr_fused(gr, f_u, f_i, e_u, e_i, users, pos, neg, 1e-4, fair, pop, plan=plan,
                                         batch_total=batch_total, count=count, total=total)
    return loss.clone(), g_u, g_i, er.clone(), ec.clone()


@pytest.mark.parametrize("n,cap", [(300, 512), (512, 512), (1, 4096), (4000, 4096), (700, 5000)])
def test_loss_with_count_equals_truncated_batch(cg, n, cap):
    gr = cg["gr"]
    rng = np.random.default_rng(n)
    U, I = gr.num_users, gr.num_items
    users = torch.as_tensor(rng.integers(0, U, cap), device=DEV)
    pos = torch.as_tensor(rng.integers(0, I, cap), device=DEV)
    neg = torch.as_tensor(rng.integers(0, I, cap), device=DEV)
    pop = torch.rand(I, device=DEV)
    users[n:], pos[n:], neg[n:] = -3, 10**9, -10**9                 # garbage in the padding: no NaN
    cnt = torch.tensor([n], dtype=torch.int64, device=DEV)
    tot = torch.tensor([n + 57], dtype=torch.int64, device=DEV)
    want = _loss_call(cg, users[:n], pos[:n], neg[:n], batch_total=n + 57, fair=0.3, pop=pop)
    got = _loss_call(cg, users, pos, neg, count=cnt, total=tot, fair=0.3, pop=pop)
    assert torch.isfinite(got[0]).all()
    assert torch.equal(got[0], want[0])
    assert torch.equal(got[1], want[1]) and torch.equal(got[2], want[2])
    assert torch.equal(got[3][: 3 * n], want[3]) and (got[3][3 * n:] == -1).all()
    heads = want[3] >= 0
    assert torch.equal(got[4][: 3 * n][heads], want[4][heads])
    # row flags: mark_rows over the padded list flags what the truncated list flags
    lib = cg["lib"]
    flags = []
    for er in (got[3], want[3]):
        nu = torch.zeros(U, dtype=torch.uint8, device=DEV)
        ni = torch.zeros(I, dtype=torch.uint8, device=DEV)
        lib.check(lib.lib().cgx_bpr_mark_rows(lib.ptr(er), er.numel(), U, lib.ptr(nu), lib.ptr(ni),
                                              lib.stream_ptr(torch.device(DEV))))
        flags.append((nu, ni))
    assert torch.equal(flags[0][0], flags[1][0]) and torch.equal(flags[0][1], flags[1][1])


def test_loss_count_zero_and_bad_ids(cg):
    gr = cg["gr"]
    cap = 64
    users = torch.full((cap,), -1, dtype=torch.int64, device=DEV)
    pos = torch.full((cap,), 10**9, dtype=torch.int64, device=DEV)
    neg = torch.full((cap,), -1, dtype=torch.int64, device=DEV)
    zero = torch.zeros(1, dtype=torch.int64, device=DEV)
    tot = torch.tensor([100], dtype=torch.int64, device=DEV)
    loss, g_u, g_i, er, _ = _loss_call(cg, users, pos, neg, count=zero, total=tot)
    assert float(loss.item()) == 0.0
    assert not g_u.any() and not g_i.any() and (er == -1).all()
    # a bad id in a REAL entry still gives NaN
    users[:3] = torch.tensor([0, 1, 2], device=DEV)
    pos[:3] = torch.tensor([0, 1, 10**9], device=DEV)
    neg[:3] = torch.tensor([3, 4, 5], device=DEV)
    three = torch.tensor([3], dtype=torch.int64, device=DEV)
    loss, *_ = _loss_call(cg, users, pos, neg, count=three, total=tot)
    assert torch.isnan(loss).all()
    pos[2] = 7
    loss, *_ = _loss_call(cg, users, pos, neg, count=three, total=tot)
    assert torch.isfinite(loss).all()


def test_frontier_with_count(cg):
    m, gr = cg["m"], cg["gr"]
    rng = np.random.default_rng(5)
    cap, n = 256, 77
    users = torch.as_tensor(rng.integers(0, gr.num_users, cap), device=DEV)
    pos = torch.as_tensor(rng.integers(0, gr.num_items, cap), device=DEV)
    neg = torch.as_tensor(rng.integers(0, gr.num_items, cap), device=DEV)
    users[n:], pos[n:] = 10**9, -4
    fu_w = torch.zeros(gr.num_users, dtype=torch.uint8, device=DEV)
    fu_g = torch.zeros_like(fu_w)
    want = m.batch_frontier(gr, users[:n], pos[:n], neg[:n], flags_u=fu_w).clone()
    got = m.batch_frontier(gr, users, pos, neg, flags_u=fu_g,
                           count=torch.tensor([n], dtype=torch.int64, device=DEV)).clone()
    assert torch.equal(got, want) and torch.equal(fu_g, fu_w)
    none = m.batch_frontier(gr, users, pos, neg, count=torch.zeros(1, dtype=torch.int64, device=DEV))
    assert not none.any()


def test_candidates_row_base(cg):
    ev, gr, graph_mod, sg = cg["ev"], cg["gr"], cg["graph"], cg["sg"]
    U, I = sg.num_users, sg.num_items
    te = graph_mod.user_csr_device(sg.test_edges, U, I, DEV)
    tr = (gr.samp_indptr, gr.samp_idx)
    users = torch.nonzero(te[0][1:] > te[0][:-1]).flatten()
    whole = ev.sampled_candidates_device(tr, te, users, I, 99, 42)
    for a, b in ((0, 5), (7, 40), (users.numel() - 3, users.numel())):
        part = ev.sampled_candidates_device(tr, te, users[a:b], I, 99, 42, row_base=a)
        assert torch.equal(part, whole[a:b])
