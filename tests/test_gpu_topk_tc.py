"""The tensor-core full-rank top-K (csrc/eval_tc.cu) at its edges.  bf16x3 promises the ids and score bits of the fp32
kernel; bf16 a selection that is exact whenever the bf16 scores are.  Here both meet inputs where the candidate
selection can go wrong: users with fewer unseen items than the candidate lists hold, all-negative scores next to the
zero-filled columns of the last item tile, dead rows of the last CTA, train items that are every user's best items,
and inputs built to stress the completeness proof exact[K-1] > max_g thr_g + 2^-13 |u| max|i|.

cgx_eval_topk is called through _lib with outputs pre-filled with a sentinel (id -7, score NaN) and two spare rows, so
that a slot the kernels never write, or a write past the last row, fails deterministically.  Where the expected list
must be exact the scores are exactly representable (small integers in one non-zero column); elsewhere the fp32 kernel
is compared with the oracle under the tie rule of test_gpu_topk_deep and bf16x3 must return the fp32 bits."""
import contextlib
import re
import types

import numpy as np
import pytest
import torch

import credgcn_oracle as orc
from test_gpu_topk_deep import _check_topk, _expect_exact, _train_rows

pytestmark = pytest.mark.gpu
DEV = "cuda"
# every candidate-list configuration of the tensor-core kernel: (K, CGX_OPT_EVAL_GROUPS).  K <= 20 keeps 2 x 24
# candidates per user with two scanning groups and 32 with one; 20 < K <= 52 keeps 64.
CONFIGS = [(5, 1), (5, 2), (20, 1), (20, 2), (21, 0), (40, 0), (52, 0)]
MASKED = np.float32(-1e9)


@pytest.fixture(scope="module")
def cg():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from credgcn import _lib, config, evaluate, graph, model, synth
    return dict(lib=_lib, config=config, evaluate=evaluate, graph=graph, model=model, synth=synth)


def _kprime(K, groups):
    """Candidates kept per user: 2 x 24 with two scanning groups, 32 with one, 64 for K > 20."""
    return 64 if K > 20 else (48 if groups != 1 else 32)


@contextlib.contextmanager
def _option(lib, name, value):
    keep = lib.get_option(name)
    lib.set_option(name, value)
    try:
        yield
    finally:
        lib.set_option(name, keep)


def _topk(cg, fu, fi, users, csr, K, prec):
    """cgx_eval_topk with sentinel-filled outputs: every slot of the n rows must be written with an id in [0, I) and
    a score that is not NaN, and the two rows past them must stay untouched."""
    lib = cg["lib"]
    h = lib.lib()
    p = lib.PRECISIONS[prec]
    users = torch.as_tensor(np.asarray(users, np.int64)).to(DEV)
    n, I, d = users.numel(), fi.shape[0], fi.shape[1]
    if prec != "fp32":
        assert h.cgx_eval_topk_uses_tensor_cores(d, K, p) == 1, (d, K, prec)
    ids = torch.full((n + 2, K), -7, dtype=torch.int32, device=DEV)
    sc = torch.full((n + 2, K), float("nan"), dtype=torch.float32, device=DEV)
    ws = lib.workspace(h.cgx_eval_topk_workspace_bytes(n, I, d, K, p), DEV)
    ip, ix = csr
    lib.check(h.cgx_eval_topk(lib.ptr(users), n, lib.ptr(fu), lib.ptr(fi), I, d, lib.ptr(ip), lib.ptr(ix), K, p,
                              lib.ptr(ids), lib.ptr(sc), lib.ptr(ws), ws.numel(), lib.stream_ptr(DEV)))
    ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
    assert (ids[n:] == -7).all() and np.isnan(sc[n:]).all(), f"{prec} K={K}: wrote past its {n} rows"
    ids, sc = ids[:n], sc[:n]
    bad = np.argwhere((ids < 0) | (ids >= I) | np.isnan(sc))
    assert bad.size == 0, (f"{prec} K={K}: unwritten or invalid slots (row, col, id, score)",
                           [(int(r), int(c), int(ids[r, c]), float(sc[r, c])) for r, c in bad[:5]])
    return ids, sc


def _csr(rows):
    indptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    idx = np.concatenate([np.asarray(r, np.int64) for r in rows]) if indptr[-1] else np.zeros(0, np.int64)
    return indptr, idx


def _int_tables(vals, pattern, d):
    """Exactly representable scores: item i carries vals[p, i] in column p, the user of table row u has 1 in column
    pattern[u] -- one non-zero product per dot product, exact in fp32, bf16 and bf16x3."""
    P, I = vals.shape
    fi = np.zeros((I, d), np.float32)
    fi[:, :P] = vals.T
    fu = np.zeros((len(pattern), d), np.float32)
    fu[np.arange(len(pattern)), pattern] = 1.0
    return torch.tensor(fu, device=DEV), torch.tensor(fi, device=DEV)


def _expect(vals, pattern, users, train, K):
    """(ids, scores) of the exact answer for table rows `users`: (score desc, id asc), train items at -1e9 last."""
    scores = [vals[pattern[u]].astype(np.float32) for u in users]
    masked = [train[u] for u in users]
    ids = _expect_exact(scores, masked, K)
    sc = np.stack([np.where(np.isin(w, m), MASKED, s[w]) for w, s, m in zip(ids, scores, masked)])
    return ids, sc.astype(np.float32)


def _assert_exact(ids, sc, want_ids, want_sc, what):
    bad = np.argwhere(ids != want_ids)
    assert bad.size == 0, (what, [(int(r), int(c), int(ids[r, c]), int(want_ids[r, c])) for r, c in bad[:5]])
    np.testing.assert_array_equal(sc.view(np.uint32), want_sc.view(np.uint32), err_msg=str(what))


def _assert_exact_scores(ids, sc, want_sc, vals, pattern, users, train, what):
    """bf16 without a proof: the kept list holds the best K' approximate scores, but among items that tie at the list's
    weakest score it keeps whichever arrived or was evicted last, not the lowest ids.  With exact scores the K scores
    must still be the exact ones, bit for bit and in order, every id must carry its own score, ids must not repeat, and
    equal scores must come in ascending id order: so ids can differ from the fp32 answer only inside the tie group at
    the K-th score."""
    np.testing.assert_array_equal(sc.view(np.uint32), want_sc.view(np.uint32), err_msg=str(what))
    for r, u in enumerate(users):
        own = np.where(np.isin(ids[r], train[u]), MASKED, vals[pattern[u]][ids[r]].astype(np.float32))
        np.testing.assert_array_equal(own.view(np.uint32), sc[r].view(np.uint32), err_msg=str((what, r)))
        assert np.unique(ids[r]).size == ids.shape[1], (what, r)
        assert not ((sc[r, 1:] == sc[r, :-1]) & (ids[r, 1:] <= ids[r, :-1])).any(), (what, r)


def _assert_same_bits(ids, sc, ids0, sc0, what):
    bad = np.argwhere((ids != ids0) | (sc.view(np.uint32) != sc0.view(np.uint32)))
    assert bad.size == 0, (what, [(int(r), int(c), int(ids[r, c]), int(ids0[r, c]), float(sc[r, c]), float(sc0[r, c]))
                                  for r, c in bad[:5]])


# ------------------------------------------------------------------------------------------------
# 1. users with fewer unseen items than the candidate lists hold
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,groups", CONFIGS)
@pytest.mark.parametrize("d", [16, 32, 64, 128])
@pytest.mark.parametrize("prec", ["bf16x3", "bf16"])
def test_short_catalogue_rows(cg, prec, d, K, groups):
    """Users who have seen every item but 0, 1, K-1, K, K+1, K'-1, K' or K'+1 of them (K' = candidates kept per
    user), the unseen ones in the first item tile, across the boundary of tiles 2 and 3, in the last partial tile or
    scattered, and a user without train items.  Such a list holds fewer real candidates than K or than K': the row
    must still be the fp32 answer -- the unseen items, then the train items at -1e9 in id order."""
    I, P = 1013, 4                                              # 7 full tiles + one of 117 items
    Kp = _kprime(K, groups)
    rng = np.random.default_rng(1000 * K + 10 * d + groups)
    vals = rng.integers(-20, 21, (P, I)).astype(np.float32)     # ties on purpose: the id rule decides
    place = {"first": lambda n: np.arange(n), "boundary": lambda n: np.arange(384 - n // 2, 384 - n // 2 + n),
             "last": lambda n: np.arange(I - n, I), "scattered": lambda n: np.sort(rng.choice(I, n, replace=False))}
    unseen = [f(n) for n in sorted({0, 1, K - 1, K, K + 1, Kp - 1, Kp, Kp + 1}) for f in place.values()]
    train = [np.setdiff1d(np.arange(I), u) for u in unseen] + [np.zeros(0, np.int64)]
    U = len(train)
    pattern = np.arange(U) % P
    fu, fi = _int_tables(vals, pattern, d)
    csr = cg["evaluate"]._device_csr(_csr(train), DEV)
    users = np.arange(U)
    want_ids, want_sc = _expect(vals, pattern, users, train, K)
    with _option(cg["lib"], "EVAL_GROUPS", groups):
        ids0, sc0 = _topk(cg, fu, fi, users, csr, K, "fp32")
        _assert_exact(ids0, sc0, want_ids, want_sc, "fp32")
        ids, sc = _topk(cg, fu, fi, users, csr, K, prec)
        _assert_exact(ids, sc, want_ids, want_sc, prec)


# ------------------------------------------------------------------------------------------------
# 2. zero-filled columns of the last tile, dead rows of the last CTA
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_users", [1, 127, 129, 300])
@pytest.mark.parametrize("I", ["K", 127, 128, 129, 257, 1013])
def test_negative_scores_tail_columns_and_dead_rows(cg, I, n_users):
    """Every real score is strictly negative, so a column past I (zero-filled by the tile load, score 0) would win
    if the tail mask let it through; rows past n_users in the last 128-user CTA must write nothing.  The users array
    is unsorted and repeats users.  Exact integer scores (bf16x3 exact, bf16 exact up to ties at the K-th score),
    then random negative scores: fp32 vs the oracle, bf16x3 bit-identical to fp32."""
    d = {1: 16, 127: 32, 129: 64, 300: 128}[n_users]
    P = 4
    for K, groups in CONFIGS:
        n_items = K if I == "K" else I
        if K > n_items:
            continue
        rng = np.random.default_rng(n_items * 7 + n_users + K)
        users = rng.integers(0, n_users, n_users) if n_users > 1 else np.zeros(1, np.int64)
        lens = rng.integers(0, max(n_items // 3, 2), n_users)
        lens[::5] = 0
        train = [np.sort(rng.choice(n_items, ln, replace=False)) for ln in lens]
        csr = cg["evaluate"]._device_csr(_csr(train), DEV)
        pattern = np.arange(n_users) % P
        vals = -rng.integers(1, 40, (P, n_items)).astype(np.float32)
        fu, fi = _int_tables(vals, pattern, d)
        want_ids, want_sc = _expect(vals, pattern, users, train, K)
        fu_np = np.abs(rng.standard_normal((n_users, d))).astype(np.float32) * 0.2
        fi_np = -np.abs(rng.standard_normal((n_items, d))).astype(np.float32) * 0.2
        fu_r, fi_r = torch.tensor(fu_np, device=DEV), torch.tensor(fi_np, device=DEV)
        o_ids, o_sc = orc.full_rank_topk(fu_np, fi_np, users, _csr(train), K)
        with _option(cg["lib"], "EVAL_GROUPS", groups):
            for prec in ("fp32", "bf16x3"):
                ids, sc = _topk(cg, fu, fi, users, csr, K, prec)
                _assert_exact(ids, sc, want_ids, want_sc, (prec, K, groups))
            ids, sc = _topk(cg, fu, fi, users, csr, K, "bf16")
            _assert_exact_scores(ids, sc, want_sc, vals, pattern, users, train, ("bf16", K, groups))
            ids0, sc0 = _topk(cg, fu_r, fi_r, users, csr, K, "fp32")
            _check_topk(ids0, sc0, o_ids, o_sc, fu_np, fi_np, users)
            ids, sc = _topk(cg, fu_r, fi_r, users, csr, K, "bf16x3")
            _assert_same_bits(ids, sc, ids0, sc0, ("random", K, groups))
            _topk(cg, fu_r, fi_r, users, csr, K, "bf16")          # approximate, but every slot written and valid


# ------------------------------------------------------------------------------------------------
# 3. train items that are every user's best items
# ------------------------------------------------------------------------------------------------
def _mask_adversary_train(order_rows, I, U):
    """Train row of user u: its best T_u items (T from 4 to 4,900, far more tiles than the 4-tile mask ring), every
    third row also every item of one whole tile."""
    lens = [4, 20, 60, 128, 300, 1000, 3000, 4900]
    train = []
    for u in range(U):
        t = set(order_rows[u][:lens[u % len(lens)]].tolist())
        if u % 3 == 0:
            tile = (u // 3) % (I // 128)
            t.update(range(tile * 128, tile * 128 + 128))
        train.append(np.array(sorted(t), np.int64))
    return train


@pytest.mark.parametrize("d", [64, 128])
def test_train_items_are_the_best_items(cg, d):
    """Each user's train items are exactly its highest-scoring items, items 0, 127, 128 and I-1 first among them; the
    kernel must skip every one of them through the train-item bits and rank the next best.  Exact integer scores for
    both precisions (bf16 has no proof or redo to hide a mask error; it is exact up to ties at the K-th score), then
    random tables: fp32 vs the oracle, bf16x3 bit-identical to fp32."""
    I, U, P = 5000, 200, 4
    rng = np.random.default_rng(d)
    top = np.array([0, 127, 128, I - 1])
    vals = rng.integers(-100, 101, (P, I)).astype(np.float32)
    vals[:, top] = 120.0
    pattern = np.arange(U) % P
    order = [np.lexsort((np.arange(I), -vals[pattern[u]].astype(np.float64))) for u in range(U)]
    train = _mask_adversary_train(order, I, U)
    assert all(np.isin(top, t).all() for t in train)
    csr = cg["evaluate"]._device_csr(_csr(train), DEV)
    users = rng.permutation(U)
    fu, fi = _int_tables(vals, pattern, d)

    m = np.abs(rng.standard_normal(d)).astype(np.float32)
    m /= np.linalg.norm(m)
    fu_np = (rng.standard_normal((U, d)) * 0.05 + m).astype(np.float32)
    fi_np = (rng.standard_normal((I, d)) * 0.2).astype(np.float32)
    fi_np[top] = 3.0 * m + 0.01 * rng.standard_normal((4, d)).astype(np.float32)
    s = fu_np.astype(np.float64) @ fi_np.astype(np.float64).T
    order_r = [np.lexsort((np.arange(I), -s[u])) for u in range(U)]
    assert all(set(o[:4]) == set(top) for o in order_r)
    train_r = _mask_adversary_train(order_r, I, U)
    csr_r = cg["evaluate"]._device_csr(_csr(train_r), DEV)
    fu_r, fi_r = torch.tensor(fu_np, device=DEV), torch.tensor(fi_np, device=DEV)
    o_ids, o_sc = orc.full_rank_topk(fu_np, fi_np, users, _csr(train_r), 52)
    for K, groups in CONFIGS:
        want_ids, want_sc = _expect(vals, pattern, users, train, K)
        with _option(cg["lib"], "EVAL_GROUPS", groups):
            for prec in ("fp32", "bf16x3"):
                ids, sc = _topk(cg, fu, fi, users, csr, K, prec)
                _assert_exact(ids, sc, want_ids, want_sc, (prec, K, groups))
            ids, sc = _topk(cg, fu, fi, users, csr, K, "bf16")
            _assert_exact_scores(ids, sc, want_sc, vals, pattern, users, train, ("bf16", K, groups))
            ids0, sc0 = _topk(cg, fu_r, fi_r, users, csr_r, K, "fp32")
            _check_topk(ids0, sc0, o_ids[:, :K], o_sc[:, :K], fu_np, fi_np, users)
            ids, sc = _topk(cg, fu_r, fi_r, users, csr_r, K, "bf16x3")
            _assert_same_bits(ids, sc, ids0, sc0, ("random", K, groups))


# ------------------------------------------------------------------------------------------------
# 4. the completeness proof under stress
# ------------------------------------------------------------------------------------------------
def _fam_near_ties(rng, U, I, d, K):
    """All-positive vectors (sum |u_k i_k| = |u . i|: the 2^-13 bound is at its tightest) with K // 2 clear winners,
    then a cluster of 600 items whose scores are spread over +-16 eps around the K-th score: hundreds of items lie
    within 1-8 eps of it."""
    w = (1.0 + 0.25 * rng.random(d)).astype(np.float32)
    fu = (0.5 + rng.random((U, d))).astype(np.float32)
    scale = 0.3 + 0.9 * rng.random(I)
    pos = rng.permutation(I)
    scale[pos[:K // 2]] = 1.4 + 0.1 * rng.random(K // 2)
    cl = pos[K // 2:K // 2 + 600]
    scale[cl] = 1.3 * (1.0 + rng.uniform(-16, 16, cl.size) * 2.0 ** -13 * 1.5 / 1.3)
    fi = (scale[:, None] * (w + 2.0 ** -13 * rng.random((I, d)))).astype(np.float32)
    return fu, fi


def _fam_midpoints(rng, U, I, d, K):
    """fp32 values whose low 16 bits sit at or next to the bf16 rounding midpoint of the value (0x8000) or of its
    low part (0x0080, 0x8080), mixed signs."""
    def mid(shape):
        b = (rng.standard_normal(shape) * 0.2).astype(np.float32).view(np.uint32)
        low = rng.choice(np.array([0x8000, 0x7FFF, 0x8001, 0x0080, 0x8080, 0x7F80, 0x4000], np.uint32), shape)
        return ((b & np.uint32(0xFFFF0000)) | low).view(np.float32)
    return mid((U, d)), mid((I, d))


def _fam_large_and_tiny(rng, U, I, d, K):
    """One component of size ~1 next to d-1 components of ~1e-3: the large products tie in groups, the tiny ones
    (far below the bf16 resolution of the large ones) decide the order."""
    fu = (1e-3 * rng.standard_normal((U, d))).astype(np.float32)
    fu[:, 0] = 1.0
    fi = (1e-3 * rng.standard_normal((I, d))).astype(np.float32)
    fi[:, 0] = rng.choice(np.array([0.5, 0.75, 1.0], np.float32), I)
    return fu, fi


def _fam_norm_spread(rng, U, I, d, K):
    """Item norms spread over four decades."""
    fu = (rng.standard_normal((U, d)) * 0.2).astype(np.float32)
    fi = (rng.standard_normal((I, d)) * 0.2 * 10.0 ** rng.uniform(0, 4, (I, 1))).astype(np.float32)
    return fu, fi


def _fam_ties(rng, U, I, d, K):
    """K // 2 copies of 2v, then 150 exact copies of v (more than any candidate list holds) every 19th item from
    item 7 on, so over tiles of both parities; every user scores v positively."""
    m = np.abs(rng.standard_normal(d)).astype(np.float32)
    m /= np.linalg.norm(m)
    fu = (m + 0.3 * rng.standard_normal((U, d)) / np.sqrt(d)).astype(np.float32)
    fi = (0.05 * rng.standard_normal((I, d)) / np.sqrt(d)).astype(np.float32)
    ties = np.arange(7, 7 + 19 * 150, 19)
    fi[ties] = m
    fi[rng.choice(np.setdiff1d(np.arange(I), ties), K // 2, replace=False)] = 2 * m
    return fu, fi


def _fam_zero_users(rng, U, I, d, K):
    """Zero user vectors: every score is 0, eps is 0, no proof can hold -- every row is redone."""
    return np.zeros((U, d), np.float32), (rng.standard_normal((I, d)) * 0.2).astype(np.float32)


FAMILIES = {"near_ties": _fam_near_ties, "midpoints": _fam_midpoints, "large_and_tiny": _fam_large_and_tiny,
            "norm_spread": _fam_norm_spread, "ties": _fam_ties, "zero_users": _fam_zero_users}
_REDO = re.compile(r"\[cgx eval\] rows=(\d+) redo=(\d+)")


@pytest.mark.parametrize("K,groups", [(5, 2), (20, 2), (20, 1), (40, 0), (52, 0)])
@pytest.mark.parametrize("d", [64, 128])
def test_completeness_proof_under_stress(cg, capfd, d, K, groups):
    """Each family: fp32 against the oracle, bf16x3 bit-identical to fp32.  The redo count (CGX_OPT_EVAL_DEBUG bit 0)
    shows the proof both held and failed; the zero users send all 400 rows, more than the 296 CTAs of the persistent
    redo grid, through the redo loop."""
    U, I = 400, 3001
    counts = {}
    for f, (name, fam) in enumerate(FAMILIES.items()):
        rng = np.random.default_rng(100 * d + 10 * K + f)
        fu_np, fi_np = fam(rng, U, I, d, K)
        tr = _train_rows(rng, U, I)
        csr = cg["evaluate"]._device_csr(tr, DEV)
        users = np.arange(U)
        fu, fi = torch.tensor(fu_np, device=DEV), torch.tensor(fi_np, device=DEV)
        with _option(cg["lib"], "EVAL_GROUPS", groups):
            ids0, sc0 = _topk(cg, fu, fi, users, csr, K, "fp32")
            capfd.readouterr()
            with _option(cg["lib"], "EVAL_DEBUG", 1):
                ids, sc = _topk(cg, fu, fi, users, csr, K, "bf16x3")
            found = _REDO.findall(capfd.readouterr().err)
        assert len(found) == 1 and int(found[0][0]) == U, found
        counts[name] = int(found[0][1])
        o_ids, o_sc = orc.full_rank_topk(fu_np, fi_np, users, tr, K)
        _check_topk(ids0, sc0, o_ids, o_sc, fu_np, fi_np, users)
        _assert_same_bits(ids, sc, ids0, sc0, (name, d, K, groups))
    print("redo rows of", U, counts)
    assert counts["zero_users"] == U > 296
    assert any(c < U for c in counts.values()), counts          # the proof held for some rows
    assert any(c > 0 for n, c in counts.items() if n != "zero_users"), counts   # and failed on a non-zero user


# ------------------------------------------------------------------------------------------------
# 5. realistic tables at full size
# ------------------------------------------------------------------------------------------------
def test_c2_propagated_tables_all_users(cg):
    """C2-shaped tables after propagate_forward of a seeded Xavier init (the tables bench.py ranks), every user, K = 20
    and 50: bf16x3 returns the fp32 ids and score bits."""
    sg = cg["synth"].make_graph("C2")
    gr = cg["graph"].build_graph(sg.train_edges, sg.num_users, sg.num_items, sg.cred, "v2", DEV)
    torch.manual_seed(0)
    e0u = torch.nn.init.xavier_uniform_(torch.empty(sg.num_users, 64, device=DEV))
    e0i = torch.nn.init.xavier_uniform_(torch.empty(sg.num_items, 64, device=DEV))
    fu, fi = cg["model"].propagate_forward(gr, e0u, e0i, 3, "gs")
    users = np.arange(sg.num_users)
    csr = (gr.samp_indptr, gr.samp_idx)
    for K in (20, 50):
        ids0, sc0 = _topk(cg, fu, fi, users, csr, K, "fp32")
        ids, sc = _topk(cg, fu, fi, users, csr, K, "bf16x3")
        _assert_same_bits(ids, sc, ids0, sc0, ("C2", K))


def test_catalogue_of_two_million_items(cg):
    """2^21 items at d = 128 on 4,096 users, K = 20 and 50: low-rank tables with popularity-skewed item norms (the
    shape propagated embeddings take) rather than iid normals; bf16x3 returns the fp32 ids and score bits."""
    U, I, d = 4096, 1 << 21, 128
    g = torch.Generator(device=DEV).manual_seed(2)
    basis = torch.randn(16, d, device=DEV, generator=g) / 4
    fu = (torch.randn(U, 16, device=DEV, generator=g) @ basis + 0.05 * torch.randn(U, d, device=DEV, generator=g))
    norm_i = 1.0 + torch.rand(I, 1, device=DEV, generator=g).pow(-0.5).clamp(max=30.0)
    fi = (torch.randn(I, 16, device=DEV, generator=g) @ basis + 0.05 * torch.randn(I, d, device=DEV, generator=g))
    fi = (fi * norm_i / fi.norm(dim=1, keepdim=True)).contiguous()
    fu = fu.contiguous()
    csr = cg["evaluate"]._device_csr(_train_rows(np.random.default_rng(2), U, I, max_len=400), DEV)
    users = np.arange(U)
    for K in (20, 50):
        ids0, sc0 = _topk(cg, fu, fi, users, csr, K, "fp32")
        ids, sc = _topk(cg, fu, fi, users, csr, K, "bf16x3")
        _assert_same_bits(ids, sc, ids0, sc0, ("2^21 items", K))


# ------------------------------------------------------------------------------------------------
# 6. end to end
# ------------------------------------------------------------------------------------------------
def test_evaluate_full_ranking_with_short_catalogue_users(cg):
    """evaluate_full_ranking at the default precision on a graph whose test users include users with 0, 1, K-1, K,
    K+1, 47, 48 and 49 unseen items (K = 20), against the oracle, with the ranking metrics on the device and on the
    host.  The top-K ids are checked to lie in [0, I) first: the device metrics index item tables with them."""
    config, ev = cg["config"], cg["evaluate"]
    rng = np.random.default_rng(17)
    U, I, d = 300, 700, 64
    fu_np = (rng.standard_normal((U, d)) * 0.3).astype(np.float32)
    fi_np = (rng.standard_normal((I, d)) * 0.3).astype(np.float32)
    tr_rows = [np.unique(rng.integers(0, I, rng.integers(0, 60))) for _ in range(U)]
    te_rows = [np.setdiff1d(np.unique(rng.integers(0, I, rng.integers(1, 20))), r) for r in tr_rows]
    for j, n in enumerate([0, 1, 19, 20, 21, 47, 48, 49] * 2):   # short catalogues, their test items among the unseen
        unseen = np.sort(rng.choice(I, n, replace=False)) if j < 8 else np.arange(I - n, I)
        tr_rows[j] = np.setdiff1d(np.arange(I), unseen)
        te_rows[j] = unseen[: max(n // 2, 1)] if n else np.array([int(tr_rows[j][3])])
    tr, te = _csr(tr_rows), _csr(te_rows)
    item_pop = np.bincount(tr[1], minlength=I).astype(np.int64)
    total = int(item_pop.sum())
    cred = rng.random(U)
    fu, fi = torch.tensor(fu_np, device=DEV), torch.tensor(fi_np, device=DEV)
    net = types.SimpleNamespace(final_embeddings=lambda: (fu, fi))
    test_users = np.flatnonzero(np.diff(te[0]) > 0)
    cfg0 = config.CFG()
    ids, _ = ev.topk_device(fu, fi, torch.from_numpy(test_users), ev._device_csr(tr, DEV), max(cfg0.Ks),
                            cfg0.score_precision)
    ids = ids.cpu().numpy()
    assert ((ids >= 0) & (ids < I)).all(), "top-K ids outside the catalogue"
    want = orc.evaluate_full_ranking(fu_np, fi_np, tr, te, I, cfg0.Ks, item_pop, total, cred)
    keep = config.cfg
    try:
        for on_device in (True, False):
            cfg = config.CFG()
            cfg.metrics_on_device = on_device
            config.cfg = cfg
            got = ev.evaluate_full_ranking(net, tr, te, I, DEV, item_pop, total, cred)
            for K in cfg.Ks:
                assert set(want[K]) <= set(got[K])
                for k, v in want[K].items():
                    if isinstance(v, float):
                        assert got[K][k] == pytest.approx(v, rel=1e-4, abs=1e-6), (on_device, K, k)
                    else:
                        assert got[K][k] == v, (on_device, K, k)
    finally:
        config.cfg = keep
