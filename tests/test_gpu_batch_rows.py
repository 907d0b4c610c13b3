"""The deferring TrainStep's last user product runs over the batch list itself (one block per batch entry, a repeated
user computed by one entry only), and with num_layers >= 3 its last layer adds layer K - 1 into the final tables.
Batches that repeat users -- a huge user (> 16 384 non-zeros, combined as the finishing kernel does), chunked users
(combined in chunk order) and short ones -- must give the eager step's bits: loss, gradients, parameters, Adam
moments, and the final tables on first read, for both orders, K = 2..4, widths of both lane layouts and both SpMM
regimes."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda"

NU, NI = 20_000, 17_000      # user 0 rates every item (huge row); users 1..8 rate 1 000 items each (chunked rows)


@pytest.fixture(scope="module")
def cg():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import credgcn  # noqa: F401
    from credgcn import _lib, graph, model
    return dict(lib=_lib, graph=graph, model=model)


@pytest.fixture(scope="module")
def gr(cg):
    rng = np.random.default_rng(11)
    users, items = np.arange(NU), np.arange(NI)
    us = [users, np.zeros(NI, np.int64), np.repeat(users, 3)]
    its = [np.zeros(NU, np.int64), items, rng.integers(9, NI, 3 * NU)]
    for j in range(1, 9):
        us += [rng.choice(users, 700, replace=False), np.full(1000, j)]
        its += [np.full(700, j), rng.choice(items, 1000, replace=False)]
    key = np.unique(np.concatenate(us).astype(np.int64) * NI + np.concatenate(its))
    edges = np.stack([key // NI, key % NI]).astype(np.int32)
    g = cg["graph"].build_graph(edges, NU, NI, np.linspace(0.2, 1.0, NU, dtype=np.float32), "v2", DEV)
    deg = (g.by_user.indptr[1:] - g.by_user.indptr[:-1]).cpu().numpy()
    assert deg[0] > 16_384 and all(256 < deg[j] <= 16_384 for j in range(1, 9))
    indptr, idx = g.by_user.indptr.cpu().numpy(), g.by_user.idx.cpu().numpy()
    g.host_rows = [idx[indptr[u]:indptr[u + 1]] for u in range(NU)]
    return g


def _batches(gr):
    rng = np.random.default_rng(5)
    lists = [
        np.array([0, 0, 3, 3, 3, 17, 0, 17, 4]),                                  # huge, chunked and short, repeated
        np.concatenate([np.zeros(40, np.int64), np.repeat(np.arange(1, 9), 5), rng.integers(9, NU, 300),
                        rng.integers(9, 200, 100)]),                              # + many repeats of short users
        np.full(64, 2),                                                           # one chunked user only
    ]
    out = []
    for users in lists:
        users = rng.permutation(users)
        pos = np.array([rng.choice(gr.host_rows[u]) for u in users])
        neg = rng.integers(0, NI, len(users))
        out.append(tuple(x.astype(np.int64) for x in (users, pos, neg)))
    return out


def _same_bits(a, b):
    return len(a) == len(b) and all(torch.equal(x.detach().view(torch.int32), y.detach().view(torch.int32))
                                    for x, y in zip(a, b))


def _state(st, loss):
    m = st.model
    return [loss.reshape(1), m.user_emb.weight, m.item_emb.weight, m.user_emb.weight.grad, m.item_emb.weight.grad,
            *st.opt.m, *st.opt.v]


@pytest.mark.parametrize("d", [16, 64, 128, 256])
@pytest.mark.parametrize("order", ["gs", "jacobi"])
def test_repeated_batch_users_same_bits_as_eager(cg, gr, order, d):
    m, L = cg["model"], cg["lib"]
    try:
        for l2 in (-1, 0):                                   # tables inside / beyond L2: both lane layouts at d >= 64
            L.set_option("L2_TABLE_BYTES", l2)
            gr.set_emb_dim(d)
            for K in (2, 3, 4):
                steps = []
                for defer in (True, False):
                    torch.manual_seed(0)
                    net = (m.LightGCN(NU, NI, d, K, gr.operator("A"), gr.operator("C")) if order == "gs" else
                           m.CredLightGCN(NU, NI, d, K, gr.operator("C"), gr.operator("A"))).to(DEV)
                    st = m.TrainStep(net, lr=1e-2, reg_weight=1e-4)
                    st._defer_final = defer
                    steps.append(st)
                a, b = steps
                for t, trip in enumerate(_batches(gr)):
                    a._f_u.fill_(float("nan"))                # every row the step reads must be written by it
                    la, lb = a(*trip), b(*trip)
                    assert a._pending and not b._pending
                    assert _same_bits(_state(a, la), _state(b, lb)), (l2, K, t)
                    assert _same_bits([a.f_u, a.f_i], [b.f_u, b.f_i]), (l2, K, t)
    finally:
        L.set_option("L2_TABLE_BYTES", -1)
        gr.set_emb_dim(d)
