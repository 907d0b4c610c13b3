"""The plain LightGCN baseline (RawLightGCN, lightgcn.py) trained through the fused TrainStep and train_on_arrays /
train_lightgcn(cfg.variant = "raw").

RawLightGCN keeps ONE table over users + items; TrainStep trains its row blocks [0, U) and [U, U + I) as the user and
item tables, in Jacobi order, with the gradient in the same blocks of one emb.weight.grad and one FusedAdam launch over
both blocks (torch.optim.Adam on emb.weight: Adam is elementwise).

* Six injected steps on C1 and C2, d in {32, 64}, K in {1, 3}, against the oracle's multi-step run (orc.train_steps on
  the credibility-1 "cu" operators): loss and gradients, the Adam update against torch.optim.Adam fed the same
  gradients, the state carried between steps.
* Five steps against the route a user has without TrainStep: autograd through RawLightGCN + torch.optim.Adam.
* capture(B) replays == eager sampled steps bit for bit (both plan paths), with phase_events on the eager side.
* Tables forced beyond L2: the item frontier and the deferred last layer, bit for bit against the non-deferred step
  and an eager forward.
* End to end: train_on_arrays in both eval modes, the best_model.pt checkpoint, train_lightgcn from files."""
import pickle
import re

import numpy as np
import pytest
import torch

import credgcn_oracle as orc
from conftest import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-4                       # the suite's bar for loss / gradients of the whole step (relative to the table max)
STEPS, LR, REG = 6, 1e-2, 1e-4
# Adam: FusedAdam's update against torch.optim.Adam fed the same gradients, per element (derivation of both bounds in
# test_gpu_train_step.py)
ADAM_RTOL = 1e-5
ADAM_ATOL = 1e-6


@pytest.fixture(scope="module")
def cg():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from credgcn import _lib, config, evaluate, graph, model, sampler, synth, train
    return dict(lib=_lib, config=config, evaluate=evaluate, graph=graph, model=model, sampler=sampler, synth=synth,
                train=train)


@pytest.fixture(scope="module")
def graphs(cg):
    """(SynthGraph, NormAdj, oracle operators) per shape: RAW's operator is the "cu" one with credibility 1."""
    cache = {}

    def get(shape):
        if shape not in cache:
            sg = cg["synth"].make_graph(shape)
            adj = cg["graph"].build_norm_adj(sg.train_edges, sg.num_users, sg.num_items, DEV)
            ops = orc.Operators(sg.train_edges, sg.num_users, sg.num_items, np.ones(sg.num_users, np.float32), "cu")
            cache[shape] = (sg, adj, ops)
        return cache[shape]
    return get


def _net(cg, sg, adj, d, K, seed=42):
    torch.manual_seed(seed)
    return cg["model"].RawLightGCN(sg.num_users, sg.num_items, d, K, adj).to(DEV)


def _injected_batches(sg, batch, steps=STEPS, seed=7):
    """`steps` triple lists.  Step t+1 re-touches the users of the first half of step t, leaves the others alone and
    adds users step t did not have; one user and one item occur in step 1 only (one triple)."""
    rng = np.random.default_rng(seed)
    ip, ix = orc.edges_to_user_csr(sg.train_edges, sg.num_users)
    deg_u = np.diff(ip)
    deg_i = np.bincount(ix, minlength=sg.num_items)
    once_i = int(np.argmin(deg_i))
    owners = np.flatnonzero(deg_u > 0)
    owners = owners[[once_i not in ix[ip[u]:ip[u + 1]] for u in owners]]
    once_u = int(owners[rng.integers(owners.size)])
    pool = owners[owners != once_u]

    def pos_of(us):
        return ix[ip[us] + (rng.random(us.size) * deg_u[us]).astype(np.int64)]

    def neg_of(n):                                        # uniform, never once_i
        x = rng.integers(0, sg.num_items - 1, size=n)
        return x + (x >= once_i)

    out, prev = [], None
    for t in range(steps):
        if prev is None:
            us = np.concatenate([[once_u], rng.choice(pool, size=batch - 1)])
        else:
            fresh = np.setdiff1d(pool, prev)
            us = np.concatenate([prev[prev != once_u][: batch // 2], rng.choice(fresh, size=batch - batch // 2)])
        ps, ns = pos_of(us), neg_of(us.size)
        if t == 0:
            ns[0] = once_i
        out.append((us.astype(np.int64), ps.astype(np.int64), ns.astype(np.int64)))
        prev = us
    return out, once_u, once_i


def _spacing(a):
    a = a.abs()
    return torch.nextafter(a, torch.full_like(a, float("inf"))) - a


def _assert_adam_update(p_new, q_new, p_old, lr, what):
    """p_new: FusedAdam's parameters, q_new: torch.optim.Adam's, both stepped from p_old with the same gradients."""
    err = (p_new - q_new).abs()
    bound = ADAM_RTOL * (q_new - p_old).abs() + ADAM_ATOL * lr + _spacing(torch.maximum(p_old.abs(), q_new.abs()))
    worst = float((err / bound).max())
    assert worst <= 1.0, (what, worst)


def _same_bits(a, b):
    return len(a) == len(b) and all(torch.equal(x.detach().view(torch.int32), y.detach().view(torch.int32))
                                    for x, y in zip(a, b))


def _state(st, loss):
    w = st.model.emb.weight
    return [loss.reshape(1), w, w.grad, *st.opt.m, *st.opt.v]


# ------------------------------------------------------------------------------------------------
# 1. multi-step parity against the oracle
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("d", [32, 64])
@pytest.mark.parametrize("shape", ["C1", "C2"])
def test_injected_steps_vs_oracle(cg, graphs, shape, d, K):
    sg, adj, ops = graphs(shape)
    U = sg.num_users
    net = _net(cg, sg, adj, d, K)
    w = net.emb.weight
    st = cg["model"].TrainStep(net, lr=LR, reg_weight=REG)
    assert w.grad is not None and w.grad.shape == w.shape
    batches, once_u, once_i = _injected_batches(sg, 4096 if shape == "C2" else 1024)
    assert sum(int((b[0] == once_u).sum()) for b in batches) == 1
    assert sum(int((b[1] == once_i).sum() + (b[2] == once_i).sum()) for b in batches) == 1
    e0 = w.detach().cpu().numpy()
    ref = orc.train_steps(ops, e0[:U], e0[U:], batches, K, "jacobi", REG, lr=LR)
    q = torch.nn.Parameter(torch.empty_like(w))           # torch.optim.Adam on ONE parameter, as lightgcn.py
    adam = torch.optim.Adam([q], lr=LR)
    for t, (trip, r) in enumerate(zip(batches, ref), start=1):
        p_old = w.detach().clone()
        loss = float(st(*trip).item())
        assert abs(loss - r["loss"]) <= TOL * abs(r["loss"]), (t, loss, r["loss"])
        g = w.grad.cpu().numpy()
        assert rel_err(g[:U], r["g_u"]) < TOL, t
        assert rel_err(g[U:], r["g_i"]) < TOL, t
        q.data.copy_(p_old)
        q.grad = w.grad.clone()
        adam.step()
        _assert_adam_update(w.detach(), q.detach(), p_old, LR, t)
        # state carried into the next step
        assert not st.g_u.any() and not st.g_i.any(), t
        assert not st.nz_u.any() and not st.nz_i.any(), t
        assert int(st.opt.step_dev.item()) == t
    assert torch.isfinite(st.f_u).all() and torch.isfinite(st.f_i).all()


# ------------------------------------------------------------------------------------------------
# 2. against the route a user has without TrainStep
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", ["C1", "C2"])
def test_matches_autograd_and_torch_adam(cg, graphs, shape):
    """RawLightGCN.get_user_item_emb + bpr_loss + backward (the autograd wrappers) + torch.optim.Adam over emb.weight,
    five steps on the same triples: loss, gradient and parameters after every step within 1e-4."""
    sg, adj, _ = graphs(shape)
    d, K, lr = 64, 3, 1e-3
    a, b = _net(cg, sg, adj, d, K), _net(cg, sg, adj, d, K)
    assert torch.equal(a.emb.weight, b.emb.weight)
    st = cg["model"].TrainStep(a, lr=lr, reg_weight=REG)
    opt = torch.optim.Adam(b.parameters(), lr=lr)
    batches, _, _ = _injected_batches(sg, 4096 if shape == "C2" else 1024, steps=5, seed=11)
    for t, trip in enumerate(batches, start=1):
        la = float(st(*trip).item())
        opt.zero_grad()
        users, pos, neg = (torch.tensor(x, device=DEV) for x in trip)
        ue, ie = b.get_user_item_emb()
        lb = b.bpr_loss(users, pos, neg, ue, ie, REG)
        lb.backward()
        opt.step()
        assert abs(la - lb.item()) <= TOL * abs(lb.item()), (t, la, lb.item())
        assert rel_err(a.emb.weight.grad.cpu().numpy(), b.emb.weight.grad.cpu().numpy()) < TOL, t
        assert rel_err(a.emb.weight.detach().cpu().numpy(), b.emb.weight.detach().cpu().numpy()) < TOL, t


# ------------------------------------------------------------------------------------------------
# 3. CUDA-graph replay
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("batch", [1024, 6000])
def test_captured_steps_equal_eager_steps(cg, graphs, batch):
    """capture(B) + step() against a TrainStep that steps eagerly from the same parameters with a sampler of the same
    seed: every loss, parameter, gradient, Adam moment and final table bit for bit.  B = 6000 puts the global-sort
    plan (3B > 12,288 keys) inside the graph.  The capture's warm-up leaves parameters, moments and counters as they
    were; the eager side collects phase_events."""
    sg, adj, _ = graphs("C1")
    gr = adj.graph
    S = cg["sampler"]
    a, b = _net(cg, sg, adj, 64, 3), _net(cg, sg, adj, 64, 3)
    sa = cg["model"].TrainStep(a, lr=LR, reg_weight=REG, sampler=S.TripleSampler(gr, None, seed=13))
    sb = cg["model"].TrainStep(b, lr=LR, reg_weight=REG, sampler=S.TripleSampler(gr, None, seed=13))
    w0 = a.emb.weight.detach().clone()
    sa.capture(batch)
    assert torch.equal(a.emb.weight, w0)
    assert int(sa.tick.item()) == 0 and int(sa.opt.step_dev.item()) == 0
    assert not any(x.any() for x in (*sa.opt.m, *sa.opt.v))
    owners = np.flatnonzero(gr.deg_u.cpu().numpy() > 0)
    rng = np.random.default_rng(batch)
    sb.phase_events = []
    for t in range(1, 5):
        users = torch.tensor(rng.choice(owners, size=batch), device=DEV)
        la, lb = sa.step(users), sb.step(users)
        assert _same_bits(_state(sa, la), _state(sb, lb)), t
        assert _same_bits([sa.f_u, sa.f_i], [sb.f_u, sb.f_i]), t
        assert int(sa.tick.item()) == int(sb.tick.item()) == t
        assert int(sa.opt.step_dev.item()) == int(sb.opt.step_dev.item()) == t
    torch.cuda.synchronize()
    assert len(sb.phase_events) == 4 and all(len(m) == 4 for m in sb.phase_events)
    assert all(m[0].elapsed_time(m[3]) > 0 for m in sb.phase_events)


# ------------------------------------------------------------------------------------------------
# 4. tables beyond L2: item frontier and deferred last layer
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [2, 3])
def test_beyond_l2_paths(cg, graphs, K):
    """L2_TABLE_BYTES = 0 puts C2's tables beyond L2 (hot-row hints on): the step uses the item frontier and, K >= 2,
    computes the last layer only on the rows the loss reads.  Against a TrainStep forced to the full last layer: loss,
    parameters, gradients and moments bit for bit; after each step f_u / f_i equal an eager forward of the step's
    parameters bit for bit on first read, and the gradients are the oracle's."""
    L, m = cg["lib"], cg["model"]
    sg, adj, ops = graphs("C2")
    gr, U, d = adj.graph, sg.num_users, 64
    batches, _, _ = _injected_batches(sg, 1024, steps=3, seed=5)
    gr.propagate_workspace(d, "jacobi")                   # sized now: the hints below are set for this width
    try:
        L.set_option("L2_TABLE_BYTES", 0)
        gr.set_emb_dim(d, hot_bytes=4 * d * 300)
        assert gr.by_user.idx_hint is not None
        a, b = _net(cg, sg, adj, d, K), _net(cg, sg, adj, d, K)
        sa, sb = m.TrainStep(a, lr=LR, reg_weight=REG), m.TrainStep(b, lr=LR, reg_weight=REG)
        sb._defer_final = False
        for t, trip in enumerate(batches):
            p_old = a.emb.weight.detach().clone()
            la, lb = sa(*trip), sb(*trip)
            assert sa._defer_final is True and sa._pending and not sb._pending, t
            n_front = int(sa.front_i.sum())
            assert 0 < n_front < sg.num_items, t
            assert _same_bits(_state(sa, la), _state(sb, lb)), t
            f_u, f_i = m.propagate_forward(gr, p_old[:U], p_old[U:], K, "jacobi")
            assert _same_bits([sa.f_u, sa.f_i], [f_u, f_i]), t
            assert _same_bits([sb.f_u, sb.f_i], [f_u, f_i]), t
            e0 = p_old.cpu().numpy()
            o_loss, o_gu, o_gi, _, _ = orc.train_step_grads(ops, e0[:U], e0[U:], *trip, K, "jacobi", REG)
            assert abs(float(la.item()) - o_loss) <= TOL * abs(o_loss), t
            g = a.emb.weight.grad.cpu().numpy()
            assert rel_err(g[:U], o_gu) < TOL and rel_err(g[U:], o_gi) < TOL, t
    finally:
        L.set_option("L2_TABLE_BYTES", -1)
        gr.set_emb_dim(d)


# ------------------------------------------------------------------------------------------------
# 5. end to end
# ------------------------------------------------------------------------------------------------
def _raw_cfg(cg, mode):
    cfg = cg["config"].CFG()
    cfg.device, cfg.variant, cfg.epochs, cfg.batch_size, cfg.eval_mode, cfg.lr = DEV, "raw", 15, 128, mode, 5e-3
    cfg.eval_every, cfg.emb_dim = 5, 64
    return cfg


def _evaluate(cg, cfg, net, train_csr, csr, num_items):
    ev = cg["evaluate"]
    if cfg.eval_mode == "full":
        return ev.evaluate_full_ranking(net, train_csr, csr, num_items, DEV)
    return ev.evaluate_sampled(net, train_csr, csr, num_items, DEV)


@pytest.mark.parametrize("mode", ["sampled", "full"])
def test_train_on_arrays_raw(cg, mode, tmp_path, capsys, monkeypatch):
    """train_on_arrays(variant="raw"): the loss falls, test Recall@20 beats the untrained model (same seed), the
    state_dict is {"emb.weight"}, and model/best_model.pt reproduces the returned test metrics in a fresh model.
    Batches of 128 over ~280 train users: CUDA-graph replays and an eager tail every epoch."""
    config, train = cg["config"], cg["train"]
    sg = cg["synth"].make_graph("C1", num_users=300, num_items=200, num_edges=12_000)
    cfg = _raw_cfg(cg, mode)
    monkeypatch.setattr(config, "cfg", cfg)               # the evaluators read the module-global cfg
    U, I = sg.num_users, sg.num_items
    adj = cg["graph"].build_norm_adj(sg.train_edges, U, I, DEV)
    train_csr, test_csr = adj.graph.user_csr_numpy(), train.evaluate_csr(sg.test_edges, U, I, DEV)   # as the loop's
    untrained = _evaluate(cg, cfg, _net(cg, sg, adj, cfg.emb_dim, cfg.num_layers, seed=0), train_csr, test_csr, I)

    torch.manual_seed(0)
    model, res = train.train_on_arrays(sg.train_edges, sg.val_edges, sg.test_edges, U, I, None, tmp_path, cfg)
    out = capsys.readouterr().out
    losses = [float(x) for x in re.findall(r"Epoch \d+ \| loss=([0-9.]+)", out)]
    assert len(losses) == cfg.epochs and losses[-1] < losses[0], losses
    assert isinstance(model, cg["model"].RawLightGCN)
    assert set(model.state_dict().keys()) == {"emb.weight"}
    assert res[20]["recall"] > untrained[20]["recall"], (res[20], untrained[20])
    assert res[20]["mode"] == untrained[20]["mode"]

    sd = torch.load(tmp_path / "model" / "best_model.pt", map_location="cpu")
    assert set(sd) == {"emb.weight"} and sd["emb.weight"].shape == (U + I, cfg.emb_dim)
    fresh = _net(cg, sg, adj, cfg.emb_dim, cfg.num_layers, seed=1)
    fresh.load_state_dict(sd)
    assert _evaluate(cg, cfg, fresh, train_csr, test_csr, I) == res


def test_train_lightgcn_raw_from_files(cg, tmp_path, capsys, monkeypatch):
    """train_lightgcn() with cfg.variant = "raw" from <out_dir>/npy/*.npy + model/*.pkl, and no credibility CSV: the
    configured path holds a file whose header the CSV reader rejects, so reading it would fail the run."""
    config, train = cg["config"], cg["train"]
    sg = cg["synth"].make_graph("C1", num_users=300, num_items=200, num_edges=12_000)
    (tmp_path / "npy").mkdir()
    (tmp_path / "model").mkdir()
    for split, e in (("train", sg.train_edges), ("val", sg.val_edges), ("test", sg.test_edges)):
        np.save(tmp_path / "npy" / f"{split}_edges.npy", e)
    for what, n in (("user", sg.num_users), ("item", sg.num_items)):
        with open(tmp_path / "model" / f"{what}2idx.pkl", "wb") as f:
            pickle.dump({f"{what}{k}": k for k in range(n)}, f)
    (tmp_path / "cred.csv").write_text("not,a,credibility,header\n")
    cfg = _raw_cfg(cg, "full")
    cfg.out_dir, cfg.cred_csv_path, cfg.epochs, cfg.eval_every = str(tmp_path), str(tmp_path / "cred.csv"), 4, 2
    monkeypatch.setattr(config, "cfg", cfg)
    res = train.train_lightgcn()
    out = capsys.readouterr().out
    assert "[CRED]" not in out and "TEST metrics" in out
    assert res[20]["mode"] == "full" and 0.0 <= res[20]["recall"] <= 1.0
    sd = torch.load(tmp_path / "model" / "best_model.pt", map_location="cpu")
    assert set(sd) == {"emb.weight"} and torch.isfinite(sd["emb.weight"]).all()
