"""The fused training step (sampler -> forward -> fused BPR loss -> adjoint -> Adam) over SEVERAL steps, and its parts
at the shapes and layouts where they can go wrong, against plain NumPy / SciPy references (float64 where it matters).

* Multi-step parity of TrainStep, injected triples and CUDA-graph replays of sampled ones: each step's loss and
  gradients against the oracle at that step's own parameters, the Adam update against torch.optim.Adam fed the same
  gradients, and the state carried between steps (gradient tables and row flags all-zero, device step counters).
* The fused loss at every width (d = 16 ... 256), batch sizes on both sides of the one-CTA plan (3B <= 12,288 keys),
  with the fairness term and a batch that is a shard of a larger one; the scatter plan bit-exact; adversarial run
  layouts; every gradient element against the float64 value with a bound set by its own sum of absolute terms.
* Sampler edges: a user who owns all items but one, a single degree class, zero-degree items, empty rows.
* Adam at the level of the update, over thousands of steps, on tables where the grid-stride loop iterates."""
import types

import numpy as np
import pytest
import torch

import credgcn_oracle as orc
from conftest import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-4                       # the suite's bar for loss / gradients of the whole step (relative to the table max)
U24 = 2.0 ** -24                 # unit roundoff of fp32

# Adam: the update p_new - p_old of FusedAdam against torch.optim.Adam fed the same gradients, per element.
# torch decays v with 0.999f but adds (1 - beta2) = 0.001f, and takes the bias correction 1 - 0.999^t in double; the
# kernel adds 1 - 0.999f = 0.001 * (1 - 1.29e-5) and divides by 1 - 0.999f^t, i.e. its weights sum to one.  torch's
# v-hat is therefore high by up to 0.001f / (1 - 0.999f) - 1 = 1.29e-5 (the limit for large t), sqrt(v-hat) by half
# of that, and its update low by up to 6.4e-6 relative.  ADAM_RTOL leaves 3.6e-6 on top for fp32 rounding: of the two
# moments and the quotient, and of the kernel's 1 - powf(0.999f, t), which cancels at small t (half an ulp of 0.998
# over 0.002 is 1.5e-5 in v-hat at t = 2, 3.3e-6 in the update for a constant gradient).  Measured on a B200 over the
# 2,500 steps below: 9.2e-6 worst relative error among updates above lr / 10.  Where m is a cancelling sum of
# gradients of both signs its absolute rounding is a few ulp of the gradients, i.e. a few 1e-7 of lr in the update:
# ADAM_ATOL (times lr).
ADAM_RTOL = 1e-5
ADAM_ATOL = 1e-6


@pytest.fixture(scope="module")
def cg():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from credgcn import _lib, graph, model, sampler, synth
    return dict(lib=_lib, graph=graph, model=model, sampler=sampler, synth=synth)


@pytest.fixture(scope="module")
def graphs(cg):
    cache = {}

    def get(shape, tag):
        if (shape, tag) not in cache:
            sg = cg["synth"].make_graph(shape)
            gr = cg["graph"].build_graph(sg.train_edges, sg.num_users, sg.num_items, sg.cred, tag, DEV)
            ops = orc.Operators(sg.train_edges, sg.num_users, sg.num_items, sg.cred, tag)
            cache[(shape, tag)] = (sg, gr, ops)
        return cache[(shape, tag)]
    return get


def _bits_for(n):
    """bits_for() of common.cuh: bits that hold 0 .. n-1, at least 1."""
    return max(1, (int(n) - 1).bit_length())


def _f32bits(x):
    return x.contiguous().view(torch.int32)


# ------------------------------------------------------------------------------------------------
# 1. multi-step parity of TrainStep
# ------------------------------------------------------------------------------------------------
CASES = {                        # shape, operator variant (order), fairness weight, mix of the sampler
    "C1-gs": ("C1", "v2", 0.0, None),
    "C1-jacobi-fair": ("C1", "cu", 0.01, 0.7),
    "C2-gs": ("C2", "v2", 0.0, 0.7),
}
STEPS, LR, REG, D, K = 6, 1e-2, 1e-4, 64, 3


def _net(cg, sg, gr, tag, fair, sampler=None):
    m = cg["model"]
    torch.manual_seed(42)
    if tag == "cu":
        net = m.CredLightGCN(sg.num_users, sg.num_items, D, K, gr.operator("C"), gr.operator("A"))
    else:
        net = m.LightGCN(sg.num_users, sg.num_items, D, K, gr.operator("A"), gr.operator("C"))
    net = net.to(DEV)
    pop = None
    if fair:
        deg = gr.deg_i_float()
        pop = (deg / max(float(deg.max()), 1.0)).astype(np.float32)
    st = m.TrainStep(net, lr=LR, reg_weight=REG, fair_weight=fair, pop=pop, sampler=sampler)
    return net, st, pop


def _injected_batches(sg, batch, seed=7):
    """STEPS triple lists.  Step t+1 re-touches the users of the first half of step t, leaves the others alone and
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
    for t in range(STEPS):
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
    """p_new: FusedAdam's parameters, q_new: torch.optim.Adam's, both stepped from p_old with the same gradients.
    Both are p_old - update rounded to fp32, so they may differ by one ulp of the parameter on top of the update."""
    err = (p_new - q_new).abs()
    bound = ADAM_RTOL * (q_new - p_old).abs() + ADAM_ATOL * lr + _spacing(torch.maximum(p_old.abs(), q_new.abs()))
    worst = float((err / bound).max())
    assert worst <= 1.0, (what, worst)


class _AdamMirror:
    """torch.optim.Adam on copies of the two tables, stepped from the kernel's parameters with the kernel's gradients."""

    def __init__(self, eu, ei, lr):
        self.q = [torch.nn.Parameter(torch.empty_like(eu)), torch.nn.Parameter(torch.empty_like(ei))]
        self.opt = torch.optim.Adam(self.q, lr=lr)

    def step(self, p_old, grads):
        for q, p, g in zip(self.q, p_old, grads):
            q.data.copy_(p)
            q.grad = g.clone()
        self.opt.step()
        return [q.detach() for q in self.q]


def _check_step(st, net, ops, order, fair, pop, mirror, p_old, triples, loss, t, sampled):
    eu, ei = net.user_emb.weight, net.item_emb.weight
    users, pos, neg = triples
    pu0, pi0 = (p.cpu().numpy() for p in p_old)
    o_loss, o_gu, o_gi, _, _ = orc.train_step_grads(ops, pu0, pi0, users, pos, neg, K, order, REG, fair, pop)
    assert abs(loss - o_loss) <= TOL * abs(o_loss), (t, loss, o_loss)
    assert rel_err(eu.grad.cpu().numpy(), o_gu) < TOL, t
    assert rel_err(ei.grad.cpu().numpy(), o_gi) < TOL, t
    q_u, q_i = mirror.step(p_old, (eu.grad, ei.grad))
    _assert_adam_update(eu.detach(), q_u, p_old[0], LR, ("user", t))
    _assert_adam_update(ei.detach(), q_i, p_old[1], LR, ("item", t))
    # state carried into the next step
    assert not st.g_u.any() and not st.g_i.any(), t
    assert not st.nz_u.any() and not st.nz_i.any(), t
    assert int(st.opt.step_dev.item()) == t
    if sampled:
        assert int(st.tick.item()) == t


@pytest.mark.parametrize("case", list(CASES))
def test_injected_steps_vs_oracle(cg, graphs, case):
    shape, tag, fair, _ = CASES[case]
    sg, gr, ops = graphs(shape, tag)
    order = "jacobi" if tag == "cu" else "gs"
    net, st, pop = _net(cg, sg, gr, tag, fair)
    batch = 4096 if shape == "C2" else 1024
    batches, once_u, once_i = _injected_batches(sg, batch)
    assert sum(int((b[0] == once_u).sum()) for b in batches) == 1
    assert sum(int((b[1] == once_i).sum() + (b[2] == once_i).sum()) for b in batches) == 1
    mirror = _AdamMirror(net.user_emb.weight, net.item_emb.weight, LR)
    for t, (users, pos, neg) in enumerate(batches, start=1):
        p_old = (net.user_emb.weight.detach().clone(), net.item_emb.weight.detach().clone())
        loss = float(st(users, pos, neg).item())
        _check_step(st, net, ops, order, fair, pop, mirror, p_old, (users, pos, neg), loss, t, sampled=False)


def _decode_plan(plan, B, U):
    """(users, pos, neg) a scatter plan was built from: key = (row << entry_bits) | entry, entry = type * B + slot."""
    eb = _bits_for(3 * B)
    k = plan.cpu().numpy().view(np.uint64)
    e, row = (k & np.uint64((1 << eb) - 1)).astype(np.int64), (k >> np.uint64(eb)).astype(np.int64)
    np.testing.assert_array_equal(np.sort(e), np.arange(3 * B))
    out = [np.empty(B, np.int64) for _ in range(3)]
    for typ in range(3):
        sel = (e // B) == typ
        out[typ][e[sel] % B] = row[sel] - (U if typ else 0)
    return out


@pytest.mark.parametrize("case,batch", [("C1-gs", 1024), ("C1-gs", 6000), ("C1-jacobi-fair", 1024),
                                        ("C1-jacobi-fair", 6000), ("C2-gs", 6000)])
def test_captured_steps_vs_oracle(cg, graphs, case, batch):
    """capture(B) + step(): every replay's triples are regenerated from the counter-based sampler (offset = step),
    must be the ones the replay's scatter plan holds, and the replayed step must match the oracle.  B = 6000 puts
    the global-sort plan (3B > 12,288 keys) inside the graph."""
    shape, tag, fair, mix = CASES[case]
    sg, gr, ops = graphs(shape, tag)
    order = "jacobi" if tag == "cu" else "gs"
    samp = cg["sampler"].TripleSampler(gr, mix, 0.75, 50, seed=13)
    net, st, pop = _net(cg, sg, gr, tag, fair, sampler=samp)
    owners = np.flatnonzero(gr.deg_u.cpu().numpy() > 0)
    rng = np.random.default_rng(batch)
    st.capture(batch)
    assert int(st.tick.item()) == 0 and int(st.opt.step_dev.item()) == 0
    mirror = _AdamMirror(net.user_emb.weight, net.item_emb.weight, LR)
    for t in range(1, STEPS + 1):
        users = torch.tensor(rng.choice(owners, size=batch), device=DEV)
        p_old = (net.user_emb.weight.detach().clone(), net.item_emb.weight.detach().clone())
        loss = float(st.step(users).item())
        torch.cuda.synchronize()
        pos, neg = samp.sample(users, offset=t)
        used = _decode_plan(st._bufs[batch][0], batch, sg.num_users)
        want = (users.cpu().numpy(), pos.cpu().numpy(), neg.cpu().numpy())
        for a, b in zip(used, want):
            np.testing.assert_array_equal(a, b)
        _check_step(st, net, ops, order, fair, pop, mirror, p_old, want, loss, t, sampled=True)


# ------------------------------------------------------------------------------------------------
# 2. the fused loss: plan, gradients, L2 rows, repeats
# ------------------------------------------------------------------------------------------------
def _fake_graph(U, I):
    """What bpr_plan / bpr_fused / apply_ego read of a graph: its sizes and device."""
    return types.SimpleNamespace(num_users=int(U), num_items=int(I), device=torch.device(DEV))


def _run_loss(cg, g, tabs, users, pos, neg, reg, fair, pop, bt):
    m = cg["model"]
    f_u, f_i, e_u, e_i = tabs
    plan = m.bpr_plan(g, users, pos, neg)
    loss, g_u, g_i, rows, coef = m.bpr_fused(g, f_u, f_i, e_u, e_i, users, pos, neg, reg, fair, pop, plan=plan,
                                             batch_total=bt)
    d_u, d_i = torch.zeros_like(e_u), torch.zeros_like(e_i)
    m.apply_ego(g, rows, coef, e_u, e_i, d_u, d_i)
    return dict(plan=plan, loss=loss, g_u=g_u, g_i=g_i, rows=rows, coef=coef, d_u=d_u, d_i=d_i)


def _check_loss(cg, U, I, d, users, pos, neg, fair, bt, seed):
    rng = np.random.default_rng(seed)

    def table(n):     # rows at scales 1e-2 .. 1: a wrong small row must not hide under a large one
        x = rng.standard_normal((n, d)) / np.sqrt(d)
        return (x * 10.0 ** rng.uniform(-2.0, 0.0, (n, 1))).astype(np.float32)
    tabs_h = [table(U), table(I), table(U), table(I)]
    pop = rng.random(I).astype(np.float32) if fair else None
    reg = 1e-3
    tabs = [torch.tensor(x, device=DEV) for x in tabs_h]
    g = _fake_graph(U, I)
    args = (users, pos, neg, reg, fair, None if pop is None else torch.tensor(pop, device=DEV), bt)
    got = _run_loss(cg, g, tabs, *args)
    B = len(users)
    Bt = bt or B

    # the plan: a host sort of the same keys
    eb = _bits_for(3 * B)
    rows_all = np.concatenate([users, U + pos, U + neg]).astype(np.uint64)
    keys = (rows_all << np.uint64(eb)) | np.arange(3 * B, dtype=np.uint64)
    np.testing.assert_array_equal(got["plan"].cpu().numpy().view(np.uint64), np.sort(keys))

    ref = orc.bpr_rows_f64(*tabs_h, users, pos, neg, reg, fair, pop, bt)
    assert abs(float(got["loss"].item()) - ref["loss"]) <= 1e-5 * ref["loss_abs"], (float(got["loss"].item()), ref)
    # every element against its own sum of absolute terms S.  The scatter adds a run of L entries in segments of 8
    # and then the L / 8 segment sums in order: ~(L / 8 + 24) fp32 roundings on the longest chain.  That stays below
    # 1e-5 * S up to L ~ 1,150; only longer runs (a whole batch on one row) get the derived allowance.
    for name, dref, s, mult in (("g_u", ref["d_fu"], ref["s_u"], ref["mult_u"]),
                                ("g_i", ref["d_fi"], ref["s_i"], ref["mult_i"])):
        tol = np.maximum(1e-5, (mult / 8.0 + 24.0) * U24)[:, None]
        err = np.abs(got[name].cpu().numpy().astype(np.float64) - dref)
        bad = err > tol * s
        assert not bad.any(), (name, np.argwhere(bad)[:5], float((err / np.maximum(tol * s, 1e-300)).max()))
    # the L2 rows: each distinct row once, with mult * 2 reg / batch_total, and no unfinished (-2) head
    rows, coef = got["rows"].cpu().numpy(), got["coef"].cpu().numpy()
    assert rows.min() >= -1
    head = rows >= 0
    mult_all = np.concatenate([ref["mult_u"], ref["mult_i"]])
    np.testing.assert_array_equal(np.sort(rows[head]), np.flatnonzero(mult_all))
    want_c = mult_all[rows[head]] * 2.0 * reg / Bt
    np.testing.assert_allclose(coef[head], want_c, rtol=1e-6)
    for name, e, mult in (("d_u", tabs_h[2], ref["mult_u"]), ("d_i", tabs_h[3], ref["mult_i"])):
        want = (mult * 2.0 * reg / Bt)[:, None] * e.astype(np.float64)
        np.testing.assert_allclose(got[name].cpu().numpy(), want, rtol=1e-6, atol=0.0, err_msg=name)
    # repeats: identical bits
    again = _run_loss(cg, g, tabs, *args)
    for k in ("plan", "rows"):
        assert torch.equal(got[k], again[k]), k
    for k in ("loss", "g_u", "g_i", "d_u", "d_i"):
        assert torch.equal(_f32bits(got[k]), _f32bits(again[k])), k
    sel = torch.tensor(head, device=DEV)
    assert torch.equal(_f32bits(got["coef"][sel]), _f32bits(again["coef"][sel]))


def _zipf_items(rng, I, n):
    """Item ids with p ~ rank^-1 over a random permutation: popular items give long runs."""
    p = 1.0 / np.arange(1, I + 1)
    return rng.permutation(I)[rng.choice(I, size=n, p=p / p.sum())].astype(np.int64)


@pytest.mark.parametrize("mode", ["plain", "fair-shard"])
@pytest.mark.parametrize("B", [1, 7, 4095, 4096, 4097, 20_000])
@pytest.mark.parametrize("d", [16, 32, 64, 128, 256])
def test_fused_loss_vs_f64(cg, d, B, mode):
    """Both plan paths (3B <= 12,288 keys: one CTA; above: global radix sort), every width (d = 256 is the only
    two-float4-per-lane instantiation), the fairness term, and a shard of a larger batch (batch_total != B)."""
    U, I = 3000, 5000
    rng = np.random.default_rng(d * 100_003 + B)
    users = rng.integers(0, U, B).astype(np.int64)
    pos, neg = _zipf_items(rng, I, B), _zipf_items(rng, I, B)
    fair, bt = (0.0, 0) if mode == "plain" else (0.05, 3 * B + 5)
    _check_loss(cg, U, I, d, users, pos, neg, fair, bt, seed=d + B)


@pytest.mark.parametrize("B", [1, 7, 4095, 4096, 4097, 20_000])
@pytest.mark.parametrize("UI", [(100, 155), (100, 156), (100, 157), (40_000, 30_000)])
def test_bpr_plan_is_the_host_sort(cg, UI, B):
    """255 / 256 / 257 rows put the row bits at 8, 8, 9 (one or two 8-bit digit passes of the one-CTA sort);
    70,000 rows need 17 bits (three passes)."""
    U, I = UI
    rng = np.random.default_rng(B + U + I)
    users, pos, neg = rng.integers(0, U, B), rng.integers(0, I, B), rng.integers(0, I, B)
    users[0], pos[-1] = U - 1, I - 1
    plan = cg["model"].bpr_plan(_fake_graph(U, I), users, pos, neg)
    eb = _bits_for(3 * B)
    rows = np.concatenate([users, U + pos, U + neg]).astype(np.uint64)
    keys = (rows << np.uint64(eb)) | np.arange(3 * B, dtype=np.uint64)
    np.testing.assert_array_equal(plan.cpu().numpy().view(np.uint64), np.sort(keys))


def _layout(name, U, I, rng):
    if name.startswith("single-run"):       # one user and one negative in every triple: a run of B entries each
        B = int(name.split("-")[-1])
        return np.full(B, 5), rng.integers(0, I, B), np.full(B, 7)
    if name == "ladder":                    # consecutive rows with runs of 1 .. 20: every start offset mod 8
        lens = np.arange(1, 21)
        users = np.repeat(np.arange(20), lens)
        pos = np.repeat(np.arange(20), lens[::-1])
        neg = np.repeat(np.arange(20, 40), rng.permutation(lens))
        return users, pos, neg
    # pos == neg, user U-1 next to item row 0 (the +U offset), item I-1
    B = 61
    users, pos, neg = rng.integers(0, U, B), rng.integers(0, I, B), rng.integers(0, I, B)
    users[:9] = U - 1
    pos[3:12] = 0
    neg[10:14] = pos[10:14]
    neg[20:29] = I - 1
    pos[40] = neg[40] = I - 1
    return users, pos, neg


@pytest.mark.parametrize("layout", ["single-run-4096", "single-run-20000", "ladder", "edges"])
@pytest.mark.parametrize("d", [16, 32, 64, 128, 256])
def test_fused_loss_adversarial_layouts(cg, d, layout):
    U, I = 3000, 5000
    rng = np.random.default_rng(d)
    users, pos, neg = (np.asarray(x, np.int64) for x in _layout(layout, U, I, rng))
    _check_loss(cg, U, I, d, users, pos, neg, 0.05, 0, seed=d + 1)


# ------------------------------------------------------------------------------------------------
# 3. sampler edges
# ------------------------------------------------------------------------------------------------
def _sampler_graph(cg, edges, U, I):
    return cg["graph"].build_graph(np.asarray(edges, np.int32), U, I, np.ones(U, np.float32), "v2", DEV)


@pytest.mark.parametrize("max_tries", [0, 50])
@pytest.mark.parametrize("mix", [None, 0.7, 1.0])
def test_sampler_almost_full_row(cg, mix, max_tries):
    """User 0 owns every item but one: that item is every negative -- also when the popularity draws give up after
    max_tries and the uniform draws take over."""
    U, I, free = 40, 64, 37
    rng = np.random.default_rng(1)
    own = [j for j in range(I) if j != free]
    eu = np.concatenate([np.zeros(len(own), np.int64), rng.integers(1, U, 600)])
    ei = np.concatenate([own, rng.integers(0, I, 600)])
    gr = _sampler_graph(cg, np.stack([eu, ei]), U, I)
    s = cg["sampler"].TripleSampler(gr, mix, 0.75, max_tries, seed=3)
    pos, neg = s.sample(torch.zeros(8192, dtype=torch.int64, device=DEV), offset=1)
    assert bool((neg == free).all())
    assert bool((pos != free).all()) and int(pos.min()) >= 0 and int(pos.max()) < I


def _chi2_one_user(cg, gr, user, mix, I):
    N = 400_000
    s = cg["sampler"].TripleSampler(gr, mix, 0.75, 50, seed=7)
    _, neg = s.sample(torch.full((N,), user, device=DEV, dtype=torch.int64), offset=2)
    counts = np.bincount(neg.cpu().numpy(), minlength=I).astype(np.float64)
    ip, ix = gr.user_csr_numpy()
    pop = orc.popularity_law(gr.deg_i.cpu().numpy(), 0.75)
    law = orc.negative_law_for_user(I, ix[ip[user]:ip[user + 1]], pop, mix)
    assert counts[law == 0].sum() == 0
    order = np.argsort(-law, kind="stable")
    bins = np.array_split(order[law[order] > 0], 40)
    obs = np.array([counts[b].sum() for b in bins])
    exp = np.array([law[b].sum() for b in bins]) * N
    chi2 = ((obs - exp) ** 2 / exp).sum()
    assert chi2 < 90.0, chi2          # 39 dof: P(chi2 > 90) ~ 5e-6
    return s


@pytest.mark.parametrize("mix", [0.7, 1.0])
def test_sampler_single_degree_class(cg, mix):
    """A regular bipartite graph (every item has degree 2): one degree class, so the popularity law is uniform."""
    U, I = 400, 2000
    u = np.repeat(np.arange(U), 10)
    i = (u * 10 + np.tile(np.arange(10), U)) % I
    gr = _sampler_graph(cg, np.stack([u, i]), U, I)
    assert set(gr.deg_i.cpu().numpy().tolist()) == {2}
    s = _chi2_one_user(cg, gr, 3, mix, I)
    assert int(s.n_classes.item()) == 1


@pytest.mark.parametrize("mix", [0.7, 1.0])
def test_sampler_zero_degree_items(cg, mix):
    """150 items without any train edge: weight (0 + 1)^gamma in the popularity law, one class of their own."""
    sg = cg["synth"].make_graph("C1", num_users=200, num_items=500, num_edges=8000)
    I = 650
    gr = _sampler_graph(cg, sg.train_edges, sg.num_users, I)
    deg = gr.deg_i.cpu().numpy()
    assert (deg == 0).sum() >= 150
    user = int(np.argmax(gr.deg_u.cpu().numpy()))
    _chi2_one_user(cg, gr, user, mix, I)


@pytest.mark.parametrize("mix", [None, 0.7])
def test_sampler_empty_rows_give_minus_one(cg, mix):
    e = np.array([[0, 0, 1, 3, 3, 3], [1, 4, 2, 0, 5, 6]])
    gr = _sampler_graph(cg, e, 6, 8)                    # users 2, 4 and 5 have no train item
    s = cg["sampler"].TripleSampler(gr, mix, 0.75, 50, seed=1)
    users = torch.tensor([0, 2, 1, 4, 3, 5], device=DEV)
    pos, neg = (x.cpu().numpy() for x in s.sample(users, offset=4))
    np.testing.assert_array_equal(pos[[1, 3, 5]], -1)
    np.testing.assert_array_equal(neg[[1, 3, 5]], -1)
    rows = {0: {1, 4}, 1: {2}, 3: {0, 5, 6}}
    for k, u in ((0, 0), (2, 1), (4, 3)):
        assert pos[k] in rows[u] and neg[k] not in rows[u] and 0 <= neg[k] < 8


# ------------------------------------------------------------------------------------------------
# 4. Adam at the level of the update
# ------------------------------------------------------------------------------------------------
def _grad_source(n, seed):
    """Per element: a scale class -- ordinary (1), of the order of eps (1e-8), large (1e4) -- and a switch that
    zeroes some elements for long stretches (steps 300..899 and 1600..2199)."""
    gen = torch.Generator(device=DEV).manual_seed(seed)
    cls = torch.randint(0, 4, (n,), device=DEV, generator=gen)
    scale = torch.tensor([1.0, 1e-8, 1e4, 1.0], device=DEV)[cls]
    gated = cls == 3

    def grad(t):
        g = torch.randn(n, device=DEV, generator=gen) * scale
        if 300 <= t < 900 or 1600 <= t < 2200:
            g[gated] = 0.0
        if 1200 <= t < 1300:                             # every gradient zero: m decays, v carries the update
            g.zero_()
        return g
    return grad


@pytest.mark.parametrize("form", ["two-tables-device-step", "one-table-host-step"])
def test_fused_adam_update_matches_torch_adam(cg, form):
    """2,500 steps.  Tables above 148 * 16 * 256 * 4 = 2,424,832 floats, so the grid-stride loop runs a second
    iteration, and not a multiple of that stride.  Before every step both sides' parameters are set to zero: the
    parameter after the step is then the update itself, to full fp32 precision (p enters no other Adam term)."""
    from credgcn._lib import check, lib, ptr, stream_ptr
    lr, T = 1e-3, 2500
    sizes = [40_627 * 64, 39_999 * 64] if form.startswith("two") else [2_600_132]
    p = [torch.zeros(n, device=DEV) for n in sizes]
    grads = [_grad_source(n, seed=k + 1) for k, n in enumerate(sizes)]
    m = [torch.zeros(n, device=DEV) for n in sizes]
    v = [torch.zeros(n, device=DEV) for n in sizes]
    q = [torch.nn.Parameter(torch.zeros(n, device=DEV)) for n in sizes]
    ref = torch.optim.Adam(q, lr=lr)
    step_dev = torch.zeros(1, dtype=torch.int64, device=DEV)
    worst = torch.zeros((), device=DEV)
    worst_rel = torch.zeros((), device=DEV)          # reported only: relative error where |update| > lr / 10
    for t in range(1, T + 1):
        g = [src(t) for src in grads]
        for x in p + q:
            x.data.zero_()
        for qq, gg in zip(q, g):
            qq.grad = gg
        ref.step()
        st = stream_ptr(DEV)
        if len(sizes) == 2:
            check(lib().cgx_tick(ptr(step_dev), st))
            check(lib().cgx_adam_step(ptr(p[0]), ptr(g[0]), ptr(m[0]), ptr(v[0]), sizes[0], ptr(p[1]), ptr(g[1]),
                                      ptr(m[1]), ptr(v[1]), sizes[1], lr, 0.9, 0.999, 1e-8, ptr(step_dev), 0, st))
        else:
            check(lib().cgx_adam_step(ptr(p[0]), ptr(g[0]), ptr(m[0]), ptr(v[0]), sizes[0], None, None, None, None, 0,
                                      lr, 0.9, 0.999, 1e-8, None, t, st))
        for pp, qq in zip(p, q):
            err = (pp - qq.detach()).abs()
            bound = ADAM_RTOL * qq.detach().abs() + ADAM_ATOL * lr
            worst = torch.maximum(worst, (err / bound).max())
            rel = torch.where(qq.detach().abs() > 0.1 * lr, err / qq.detach().abs(), 0.0)
            worst_rel = torch.maximum(worst_rel, rel.max())
    print(f"adam {form}: worst err / bound {float(worst):.3f}, worst relative error of updates > lr/10 "
          f"{float(worst_rel):.2e}")
    if len(sizes) == 2:
        assert int(step_dev.item()) == T
    for mm, qq in zip(m, q):                              # the moments themselves
        assert rel_err(mm.cpu().numpy(), ref.state[qq]["exp_avg"].cpu().numpy()) < 1e-5
    assert float(worst) <= 1.0, float(worst)
