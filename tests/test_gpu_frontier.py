"""The item frontier of a triple batch (cgx_batch_frontier) and the backward propagation restricted to it
(cgx_propagate_bwd_frontier): the flags equal the set computed on the host, and the restricted backward returns the
bits of cgx_propagate_bwd_flagged -- both orders, every width, both SpMM regimes, hot hints on and off, on a graph
with chunked and huge item rows inside and outside the frontier -- without reading a stale row of its workspace."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda"

HALF_U, HALF_I = 20_000, 2_000      # two disconnected halves: a batch from one half never reaches the other
EMPTY_U = 100                        # users without train edges, after both halves
U, I = 2 * HALF_U + EMPTY_U, 2 * HALF_I


@pytest.fixture(scope="module")
def cg():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import credgcn  # noqa: F401
    from credgcn import _lib, graph, model
    return dict(lib=_lib, graph=graph, model=model)


def _edges():
    """Per half: item 0 of the half is rated by all 20 000 of its users (a huge row, > 16 384 non-zeros), items 1..8
    by 1 000 each (chunked rows), and every user rates 4 random items of the half."""
    rng = np.random.default_rng(7)
    us, its = [], []
    for h in range(2):
        u0, i0 = h * HALF_U, h * HALF_I
        users = np.arange(u0, u0 + HALF_U)
        us.append(users)
        its.append(np.full(HALF_U, i0))
        for j in range(1, 9):
            us.append(rng.choice(users, 1000, replace=False))
            its.append(np.full(1000, i0 + j))
        us.append(np.repeat(users, 4))
        its.append(rng.integers(i0 + 9, i0 + HALF_I, 4 * HALF_U))
    key = np.unique(np.concatenate(us).astype(np.int64) * I + np.concatenate(its))
    return np.stack([key // I, key % I]).astype(np.int32)


@pytest.fixture(scope="module")
def gr(cg):
    e = _edges()
    g = cg["graph"].build_graph(e, U, I, np.linspace(0.2, 1.0, U, dtype=np.float32), "v2", DEV)
    assert g.by_item.n_huge == 2 and g.by_item.n_long > 2        # both huge rows and chunked rows are exercised
    indptr, idx = g.by_user.indptr.cpu().numpy(), g.by_user.idx.cpu().numpy()
    g.host_rows = [idx[indptr[u]:indptr[u + 1]] for u in range(U)]
    return g


def _front_host(gr, users, pos, neg):
    f = np.zeros(I, np.uint8)
    for u in users:
        f[gr.host_rows[u]] = 1
    f[pos] = 1
    f[neg] = 1
    return f


def _batch(gr, rng, B, half=0, users=None):
    """Triples of one half: positives from the user's row, negatives uniform over the half's items."""
    if users is None:
        users = rng.integers(half * HALF_U, (half + 1) * HALF_U, B)
    pos = np.array([rng.choice(gr.host_rows[u]) if len(gr.host_rows[u]) else half * HALF_I for u in users])
    neg = rng.integers(half * HALF_I, (half + 1) * HALF_I, len(users))
    return users.astype(np.int64), pos.astype(np.int64), neg.astype(np.int64)


def test_frontier_flags_equal_host_set(cg, gr):
    m = cg["model"]
    rng = np.random.default_rng(1)
    last_empty = 2 * HALF_U + EMPTY_U - 1
    cases = [
        _batch(gr, rng, 4096, 0), _batch(gr, rng, 4096, 1), _batch(gr, rng, 333, 1),
        # duplicate users, users without edges, pos == neg, the first and last item ids
        (np.array([5, 5, 5, 2 * HALF_U, 7, last_empty]), np.array([0, 0, I - 1, 3, I - 1, 0]),
         np.array([0, 1, I - 1, 3, I - 1, I - 1])),
        (np.array([HALF_U + 3]), np.array([I - 1]), np.array([I - 1])),                       # B = 1, pos = neg
        (np.array([2 * HALF_U]), np.array([0]), np.array([I - 1])),                           # B = 1, empty row
    ]
    flags = torch.full((I,), 7, dtype=torch.uint8, device=DEV)       # cgx_batch_frontier zeroes it first
    for users, pos, neg in cases:
        m.batch_frontier(gr, users, pos, neg, flags)
        assert np.array_equal(flags.cpu().numpy(), _front_host(gr, users, pos, neg))


def _grads(users, pos, neg, d, gen):
    g_u = torch.zeros(U, d, device=DEV)
    g_i = torch.zeros(I, d, device=DEV)
    ut = torch.as_tensor(users, device=DEV)
    it = torch.as_tensor(np.concatenate([pos, neg]), device=DEV)
    g_u[ut] = torch.randn(len(users), d, device=DEV, generator=gen)
    g_i[it] = torch.randn(len(it), d, device=DEV, generator=gen)
    nz_u = torch.zeros(U, dtype=torch.uint8, device=DEV)
    nz_i = torch.zeros(I, dtype=torch.uint8, device=DEV)
    nz_u[ut] = 1
    nz_i[it] = 1
    return g_u, g_i, nz_u, nz_i


class _Bwd:
    """Both backward entry points on one NaN-able workspace."""

    def __init__(self, cg, gr, d, order):
        self.cg, self.gr, self.d, self.order = cg, gr, d, cg["lib"].ORDERS[order]
        lib = cg["lib"].lib()
        n = lib.cgx_propagate_workspace_bytes_for(gr.by_user.ref(), gr.by_item.ref(), d, self.order)
        self.ws = cg["lib"].workspace(n, DEV)

    def __call__(self, K, g_u, g_i, nz_u, nz_i, front=None, nan=True):
        L = self.cg["lib"]
        if nan:
            self.ws.fill_(0xFF)                                       # every float of the workspace is NaN
        d_u, d_i = torch.empty_like(g_u), torch.empty_like(g_i)
        args = [self.gr.by_user.ref(), self.gr.by_item.ref(), self.order, K, self.d, L.ptr(g_u), L.ptr(g_i),
                L.ptr(nz_u), L.ptr(nz_i)]
        tail = [L.ptr(d_u), L.ptr(d_i), L.ptr(self.ws), self.ws.numel(), L.stream_ptr(DEV)]
        if front is None:
            L.check(L.lib().cgx_propagate_bwd_flagged(*args, *tail))
        else:
            L.check(L.lib().cgx_propagate_bwd_frontier(*args, L.ptr(front), *tail))
        return d_u, d_i


def _same_bits(a, b):
    return all(torch.equal(x.view(torch.int32), y.view(torch.int32)) for x, y in zip(a, b))


def _regimes(cg, gr, d):
    """(name, setter): the in-L2 geometry with no hints, the beyond-L2 geometry with hot hints on and off."""
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


@pytest.mark.parametrize("d", [16, 32, 64, 128, 256])
@pytest.mark.parametrize("order", ["gs", "jacobi"])
def test_frontier_backward_same_bits_as_flagged(cg, gr, order, d):
    """K = 1..4 under every regime; the frontier of the batch holds the huge row and chunked rows of half 0, the
    other half's huge and chunked rows are outside it.  Then a batch of half 1 (a disjoint frontier) on the same
    workspace, not refilled: the rows the first call left behind must not be read."""
    m, L = cg["model"], cg["lib"]
    rng = np.random.default_rng(d)
    gen = torch.Generator(device=DEV).manual_seed(d)
    bwd = _Bwd(cg, gr, d, order)
    a = _batch(gr, rng, 512, 0)
    b = _batch(gr, rng, 512, 1)
    fa = m.batch_frontier(gr, *a)
    fb = m.batch_frontier(gr, *b)
    assert fa[0] == 1 and fa[HALF_I] == 0 and not (fa.bool() & fb.bool()).any()
    ga, gb = _grads(*a, d, gen), _grads(*b, d, gen)
    try:
        for name, setup in _regimes(cg, gr, d):
            setup()
            for K in (1, 2, 3, 4):
                want_a, want_b = bwd(K, *ga), bwd(K, *gb)
                got_a = bwd(K, *ga, front=fa)
                got_b = bwd(K, *gb, front=fb, nan=False)
                assert torch.isfinite(got_a[0]).all() and torch.isfinite(got_b[0]).all(), (name, K)
                assert _same_bits(got_a, want_a), (name, K)
                assert _same_bits(got_b, want_b), (name, K)
    finally:
        L.set_option("L2_TABLE_BYTES", -1)
        L.set_option("HOT_ROWS", -1)
        gr.set_emb_dim(d)


@pytest.mark.parametrize("order", ["gs", "jacobi"])
def test_frontier_seed_edge_cases(cg, gr, order):
    """Users without train edges only (F = pos + neg), and a batch whose frontier is every item."""
    m = cg["model"]
    d = 64
    rng = np.random.default_rng(3)
    gen = torch.Generator(device=DEV).manual_seed(3)
    bwd = _Bwd(cg, gr, d, order)
    empty = np.arange(2 * HALF_U, 2 * HALF_U + EMPTY_U, dtype=np.int64)
    pos, neg = rng.integers(0, I, EMPTY_U), rng.integers(0, I, EMPTY_U)
    everything = rng.integers(0, 2 * HALF_U, I), np.arange(I), rng.integers(0, I, I)
    for users, p, n in ((empty, pos, neg), everything):
        f = m.batch_frontier(gr, users, p, n)
        want_f = np.zeros(I, np.uint8)
        if users is empty:
            want_f[p], want_f[n] = 1, 1
        else:
            want_f[:] = 1
        assert np.array_equal(f.cpu().numpy(), want_f)
        g = _grads(users, p, n, d, gen)
        for K in (1, 2, 3):
            assert _same_bits(bwd(K, *g, front=f), bwd(K, *g))


def test_train_step_uses_the_frontier_beyond_l2(cg, gr):
    """TrainStep computes the frontier of its batch only when the item table is beyond L2 (inside L2 the restricted
    backward does not pay), and both forms leave the same gradients."""
    m, L = cg["model"], cg["lib"]
    users, pos, neg = _batch(gr, np.random.default_rng(5), 256, 1)
    grads = []
    for l2 in (-1, 0):
        L.set_option("L2_TABLE_BYTES", l2)
        try:
            torch.manual_seed(0)
            net = m.LightGCN(U, I, 32, 2, gr.operator("A"), gr.operator("C")).to(DEV)
            st = m.TrainStep(net, lr=1e-2, reg_weight=1e-4)
            assert np.isfinite(float(st.forward_backward(users, pos, neg)))
            want = _front_host(gr, users, pos, neg) if l2 == 0 else np.zeros(I, np.uint8)
            assert np.array_equal(st.front_i.cpu().numpy(), want)
            grads.append((net.user_emb.weight.grad.clone(), net.item_emb.weight.grad.clone()))
        finally:
            L.set_option("L2_TABLE_BYTES", -1)
            gr.set_emb_dim(32)
    assert _same_bits(grads[0], grads[1])
