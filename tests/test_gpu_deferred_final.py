"""TrainStep's deferred last layer: the step computes the last layer's products only on the rows the loss reads
(batch users; pos, neg and the batch users' train items), and the first read of f_u / f_i computes the rest.  A
deferring TrainStep and one forced eager, from identical parameters, must agree bit for bit -- loss, gradients,
parameters, Adam moments, and the final tables on first read -- for both orders, K = 1..4, every width, both SpMM
regimes and hot hints on and off, on a graph with chunked and huge rows inside and outside the masks."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda"

HALF_U, HALF_I = 20_000, 17_000     # two disconnected halves: a batch from one half never reaches the other
EMPTY_U = 100                        # users without train edges, after both halves
U, I = 2 * HALF_U + EMPTY_U, 2 * HALF_I


@pytest.fixture(scope="module")
def cg():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import credgcn  # noqa: F401
    from credgcn import _lib, graph, model, sampler
    return dict(lib=_lib, graph=graph, model=model, sampler=sampler)


def _edges():
    """Per half h: item 0 of the half is rated by all 20 000 of its users and user 0 of the half rates all 17 000 of
    its items (huge rows, > 16 384 non-zeros); items 1..8 are rated by 1 000 users each and users 1..8 rate 1 000
    items each (chunked rows); every user rates 4 random items of the half."""
    rng = np.random.default_rng(7)
    us, its = [], []
    for h in range(2):
        u0, i0 = h * HALF_U, h * HALF_I
        users, items = np.arange(u0, u0 + HALF_U), np.arange(i0, i0 + HALF_I)
        us += [users, np.full(HALF_I, u0)]
        its += [np.full(HALF_U, i0), items]
        for j in range(1, 9):
            us += [rng.choice(users, 1000, replace=False), np.full(1000, u0 + j)]
            its += [np.full(1000, i0 + j), rng.choice(items, 1000, replace=False)]
        us.append(np.repeat(users, 4))
        its.append(rng.integers(i0 + 9, i0 + HALF_I, 4 * HALF_U))
    key = np.unique(np.concatenate(us).astype(np.int64) * I + np.concatenate(its))
    return np.stack([key // I, key % I]).astype(np.int32)


@pytest.fixture(scope="module")
def gr(cg):
    g = cg["graph"].build_graph(_edges(), U, I, np.linspace(0.2, 1.0, U, dtype=np.float32), "v2", DEV)
    assert g.by_item.n_huge == 2 and g.by_item.n_long > 2 and g.by_user.n_huge == 2 and g.by_user.n_long > 2
    indptr, idx = g.by_user.indptr.cpu().numpy(), g.by_user.idx.cpu().numpy()
    g.host_rows = [idx[indptr[u]:indptr[u + 1]] for u in range(U)]
    return g


def _batch(gr, rng, B, half=0, users=None):
    """Triples of one half, with the half's huge and chunked user rows among the batch users."""
    if users is None:
        users = np.concatenate([np.arange(half * HALF_U, half * HALF_U + 3),
                                rng.integers(half * HALF_U, (half + 1) * HALF_U, B - 3)])
    pos = np.array([rng.choice(gr.host_rows[u]) if len(gr.host_rows[u]) else half * HALF_I for u in users])
    neg = rng.integers(half * HALF_I, (half + 1) * HALF_I, len(users))
    return users.astype(np.int64), pos.astype(np.int64), neg.astype(np.int64)


def _pair(cg, gr, order, K, d):
    """(deferring, eager) TrainSteps over identical parameters."""
    m = cg["model"]
    out = []
    for defer in (True, False):
        torch.manual_seed(0)
        net = (m.LightGCN(U, I, d, K, gr.operator("A"), gr.operator("C")) if order == "gs" else
               m.CredLightGCN(U, I, d, K, gr.operator("C"), gr.operator("A"))).to(DEV)
        st = m.TrainStep(net, lr=1e-2, reg_weight=1e-4)
        st._defer_final = defer
        out.append(st)
    return out


def _state(st, loss):
    m = st.model
    return [loss.reshape(1), m.user_emb.weight, m.item_emb.weight, m.user_emb.weight.grad, m.item_emb.weight.grad,
            *st.opt.m, *st.opt.v]


def _same_bits(a, b):
    return len(a) == len(b) and all(torch.equal(x.detach().view(torch.int32), y.detach().view(torch.int32))
                                    for x, y in zip(a, b))


def _poison(st):
    nan = float("nan")
    st._f_u.fill_(nan)
    st._f_i.fill_(nan)
    if st._fws is not None:
        st._fws.fill_(0xFF)                                           # every float of the workspace is NaN


def _check_steps(a, b, batches, K, read_every=True):
    """Injected triples through both steps; a is the deferring one."""
    for t, trip in enumerate(batches):
        _poison(a)
        la, lb = a(*trip), b(*trip)
        assert a._pending == (K >= 2) and not b._pending
        assert _same_bits(_state(a, la), _state(b, lb)), t
        if read_every or t == len(batches) - 1:
            assert _same_bits([a.f_u, a.f_i], [b.f_u, b.f_i]), t
            assert not a._pending
            assert torch.isfinite(a.f_u).all() and torch.isfinite(a.f_i).all()


def _regimes(cg, gr, d):
    L = cg["lib"]

    def in_l2():
        L.set_option("L2_TABLE_BYTES", -1)
        L.set_option("HOT_ROWS", 1)
        gr.set_emb_dim(d)

    def beyond(hot):
        def f():
            L.set_option("L2_TABLE_BYTES", 0)
            L.set_option("HOT_ROWS", hot)
            gr.set_emb_dim(d, hot_bytes=4 * d * 300)                  # 300 hot rows per side
            assert gr.by_user.idx_hint is not None
        return f
    return [("in_l2", in_l2), ("beyond_l2_hot", beyond(1)), ("beyond_l2_cold", beyond(0))]


def _restore(cg, gr, d):
    cg["lib"].set_option("L2_TABLE_BYTES", -1)
    cg["lib"].set_option("HOT_ROWS", -1)
    gr.set_emb_dim(d)


@pytest.mark.parametrize("d", [16, 32, 64, 128, 256])
@pytest.mark.parametrize("order", ["gs", "jacobi"])
def test_deferred_same_bits_as_eager(cg, gr, order, d):
    """Two steps per case: a batch of half 0 (its huge and chunked rows inside the masks, half 1's outside), then one
    of half 1.  f_u, f_i and the forward workspace are NaN before every step; the forward overwrites every row the
    last layer reads, so this shows only that no unwritten buffer is read -- the masks themselves are checked by the
    bit-for-bit comparison with the eager step (a row missing from them would change the loss)."""
    rng = np.random.default_rng(d)
    batches = [_batch(gr, rng, 256, 0), _batch(gr, rng, 256, 1)]
    for o in ("gs", "jacobi"):
        gr.propagate_workspace(d, o)                                  # sized now: the regimes below set the hints
    try:
        for name, setup in _regimes(cg, gr, d):
            setup()
            for K in (1, 2, 3, 4):
                a, b = _pair(cg, gr, order, K, d)
                _check_steps(a, b, batches, K)
    finally:
        _restore(cg, gr, d)


@pytest.mark.parametrize("order", ["gs", "jacobi"])
def test_edge_batches(cg, gr, order):
    """Duplicate users, B = 1, pos = neg, users without train edges, and a frontier that is every item."""
    rng = np.random.default_rng(3)
    batches = [
        (np.array([5, 5, 5, HALF_U, 7, 2 * HALF_U]), np.array([9, 9, I - 1, HALF_I, I - 1, 0]),
         np.array([9, 1, I - 1, HALF_I, I - 1, I - 1])),
        (np.array([HALF_U + 3]), np.array([I - 1]), np.array([I - 1])),
        (np.array([2 * HALF_U + 1]), np.array([0]), np.array([I - 1])),
        (rng.integers(0, 2 * HALF_U, I), np.arange(I), rng.integers(0, I, I)),
    ]
    batches = [tuple(x.astype(np.int64) for x in t) for t in batches]
    try:
        cg["lib"].set_option("L2_TABLE_BYTES", 0)
        a, b = _pair(cg, gr, order, 3, 64)
        _check_steps(a, b, batches, 3)
    finally:
        _restore(cg, gr, 64)


def test_reads_after_every_replay_or_only_the_last(cg, gr):
    """CUDA-graph replays of the default TrainStep (beyond L2: deferring) against one forced eager: tables read after
    every replay in one run, only after the last in another."""
    m, S = cg["model"], cg["sampler"]
    d, K = 64, 3
    users = torch.as_tensor(np.random.default_rng(0).choice(2 * HALF_U, 512, replace=False), device=DEV)
    try:
        cg["lib"].set_option("L2_TABLE_BYTES", 0)
        for read_every in (True, False):
            steps = []
            for defer in (None, False):
                torch.manual_seed(0)
                net = m.LightGCN(U, I, d, K, gr.operator("A"), gr.operator("C")).to(DEV)
                st = m.TrainStep(net, lr=1e-2, reg_weight=1e-4, sampler=S.TripleSampler(gr, 0.7, 0.75, 50, seed=9))
                st._defer_final = defer
                st.capture(users.numel())
                steps.append(st)
            a, b = steps
            assert a._defer_final is True and a._g_pending
            for t in range(4):
                la, lb = a.step(users), b.step(users)
                assert a._pending and not b._pending
                assert _same_bits(_state(a, la), _state(b, lb)), t
                if read_every or t == 3:
                    assert _same_bits([a.f_u, a.f_i], [b.f_u, b.f_i]), t
    finally:
        _restore(cg, gr, d)


def test_second_read_launches_nothing(cg, gr):
    L = cg["lib"].lib()
    try:
        cg["lib"].set_option("L2_TABLE_BYTES", 0)
        a, b = _pair(cg, gr, "gs", 3, 32)
        trip = _batch(gr, np.random.default_rng(1), 128, 0)
        a(*trip)
        b(*trip)
        n0 = L.cgx_launch_count()
        fu = a.f_u
        n1 = L.cgx_launch_count()
        fu2, fi, fi2 = a.f_u, a.f_i, a.f_i
        n2 = L.cgx_launch_count()
        assert n1 > n0 and n2 == n1
        assert fu is fu2 and fi is fi2 and fu is a._f_u
        assert _same_bits([fu, fi], [b.f_u, b.f_i])
    finally:
        _restore(cg, gr, 32)


def test_other_work_on_the_graph_before_the_read(cg, gr):
    """propagate_forward() and a second TrainStep's step on the same graph run between a step and the read: they
    share the graph's workspace, not the deferring step's."""
    m = cg["model"]
    rng = np.random.default_rng(2)
    try:
        cg["lib"].set_option("L2_TABLE_BYTES", 0)
        for order in ("gs", "jacobi"):
            a, b = _pair(cg, gr, order, 3, 64)
            c, _ = _pair(cg, gr, order, 2, 64)
            trip = _batch(gr, rng, 256, 0)
            a(*trip)
            b(*trip)
            e0 = torch.randn(U, 64, device=DEV), torch.randn(I, 64, device=DEV)
            m.propagate_forward(gr, *e0, 3, order)
            c(*_batch(gr, rng, 256, 1))
            assert _same_bits([a.f_i, a.f_u], [b.f_i, b.f_u]), order
    finally:
        _restore(cg, gr, 64)


def test_default_decision_and_memory_fallback(cg, gr, monkeypatch):
    """Beyond L2 with K >= 2 the step defers; inside L2, with K = 1, or without room for its own forward workspace
    it does not -- and the fallback computes the same bits."""
    m = cg["model"]
    trip = _batch(gr, np.random.default_rng(4), 256, 0)

    def decided(K, l2):
        cg["lib"].set_option("L2_TABLE_BYTES", l2)
        torch.manual_seed(0)
        st = m.TrainStep(m.LightGCN(U, I, 64, K, gr.operator("A"), gr.operator("C")).to(DEV), lr=1e-2)
        return st, st(*trip)
    try:
        assert decided(3, 0)[0]._defer_final is True
        assert decided(3, -1)[0]._defer_final is False
        assert decided(1, 0)[0]._defer_final is False
        a, la = decided(3, 0)
        monkeypatch.setattr(torch.cuda, "mem_get_info", lambda *_: (0, 180 << 30))
        b, lb = decided(3, 0)
        assert b._defer_final is False and b._fws is None and not b._pending
        assert _same_bits(_state(a, la), _state(b, lb))
        assert _same_bits([a.f_u, a.f_i], [b.f_u, b.f_i])
    finally:
        _restore(cg, gr, 64)
