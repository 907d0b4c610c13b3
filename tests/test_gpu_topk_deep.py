"""Deep full-rank top-K (128 < k <= 4096, csrc/eval_deep.cu) and ranking metrics at deep cut-offs, against the CPU
oracle.  The deep path is exact fp32 for every precision, so bf16x3 and bf16 must return the bits of fp32, and its
first columns must equal the k <= 128 kernels' lists."""
import types

import numpy as np
import pytest
import torch

import credgcn_oracle as orc

pytestmark = pytest.mark.gpu
DEV = "cuda"
PRECS = ("fp32", "bf16x3", "bf16")


@pytest.fixture(scope="module")
def cg():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from credgcn import _lib, config, evaluate, synth, train
    return dict(lib=_lib, config=config, evaluate=evaluate, synth=synth, train=train)


def _check_topk(ids, sc, o_ids, o_sc, f_u, f_i, users):
    """The tie-aware comparison of tests/test_gpu_parity.py (ids may differ only where the oracle's own scores tie),
    with the bar widened to the fp32 error bound of a d-term dot product, 2 * d * 2^-24 * sum_k |u_k i_k| (both the
    device's fmaf chain and NumPy's sum round).  Deep lists reach scores near zero, where that bound and not 1e-6 of
    the score decides what counts as a tie."""
    gamma = 2.0 * f_u.shape[1] * 2.0 ** -24
    au, ai = np.abs(f_u.astype(np.float64)), np.abs(f_i.astype(np.float64))
    bound = np.stack([gamma * np.maximum(ai[ids[r]] @ au[u], ai[o_ids[r]] @ au[u]) for r, u in enumerate(users)])
    a, b = o_sc.astype(np.float64), sc.astype(np.float64)
    diff = ids != o_ids
    tie = np.abs(a - b) <= np.maximum(1e-6 * np.maximum(np.abs(a), 1e-3), bound)
    bad = np.argwhere(diff & ~tie)
    assert bad.size == 0, [(int(r), int(c), a[r, c], b[r, c], bound[r, c]) for r, c in bad[:5]]
    close = np.abs(a - b) <= 1e-5 * np.abs(a) + np.maximum(1e-7, bound)
    assert close.all(), [(int(r), int(c), a[r, c], b[r, c]) for r, c in np.argwhere(~close)[:5]]


def _train_rows(rng, U, I, max_len=60):
    rows = [np.unique(rng.integers(0, I, rng.integers(0, max_len))) for _ in range(U)]
    indptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    return indptr, np.concatenate(rows).astype(np.int64)


def _topk(cg, fu, fi, users, csr_dev, K, prec="fp32"):
    ids, sc = cg["evaluate"].topk_device(fu, fi, torch.as_tensor(users), csr_dev, K, prec)
    return ids, sc


def _expect_exact(scores, masked_rows, K):
    """Best K of exactly representable scores: (score desc, id asc), masked items at -1e9."""
    out = []
    for s, m in zip(scores, masked_rows):
        s = s.astype(np.float32).copy()
        s[m] = np.float32(-1e9)
        out.append(np.lexsort((np.arange(s.size), -s.astype(np.float64)))[:K])
    return np.stack(out)


@pytest.mark.parametrize("d", [16, 32, 64, 128, 256])
def test_deep_topk_matches_oracle_all_widths_and_precisions(cg, d):
    """k in {129, 200, 256, 257, 1000, 4096} on I = 5,003 items (not a multiple of the 128-item tile) and 150 users
    (not a multiple of the CTA's 64), and k = I on the first 4,001 items: fp32 against the oracle with its tie rule,
    bf16x3 and bf16 bit-identical to fp32, and the prefix property against the k = 128 fp32 and k = 20 bf16x3
    lists."""
    U, I = 150, 5003
    rng = np.random.default_rng(100 + d)
    fu_np = (rng.standard_normal((U, d)) * 0.2).astype(np.float32)
    fi_np = (rng.standard_normal((I, d)) * 0.2).astype(np.float32)
    fi_np[::7] = fi_np[3]                                        # exact ties across many items
    tr = _train_rows(rng, U, I)
    users = np.arange(U, dtype=np.int64)
    fu, fi = torch.tensor(fu_np, device=DEV), torch.tensor(fi_np, device=DEV)
    csr = cg["evaluate"]._device_csr(tr, DEV)
    o_ids, o_sc = orc.full_rank_topk(fu_np, fi_np, users, tr, I)   # total order: every top-K is a prefix
    ids128, sc128 = _topk(cg, fu, fi, users, csr, 128)
    ids20, sc20 = _topk(cg, fu, fi, users, csr, 20, "bf16x3")
    for K in (129, 200, 256, 257, 1000, 4096):
        ids, sc = _topk(cg, fu, fi, users, csr, K)
        _check_topk(ids.cpu().numpy(), sc.cpu().numpy(), o_ids[:, :K], o_sc[:, :K], fu_np, fi_np, users)
        assert torch.equal(ids[:, :128], ids128) and torch.equal(sc[:, :128].view(torch.int32), sc128.view(torch.int32))
        assert torch.equal(ids[:, :20], ids20) and torch.equal(sc[:, :20].view(torch.int32), sc20.view(torch.int32))
        for prec in PRECS[1:]:
            ids_p, sc_p = _topk(cg, fu, fi, users, csr, K, prec)
            assert torch.equal(ids_p, ids), (K, prec)
            assert torch.equal(sc_p.view(torch.int32), sc.view(torch.int32)), (K, prec)
    I2 = 4001                                                    # k = I: the whole catalogue in order
    rows2 = [r[r < I2] for r in np.split(tr[1], tr[0][1:-1])]
    tr2 = (np.concatenate([[0], np.cumsum([len(r) for r in rows2])]).astype(np.int64), np.concatenate(rows2))
    csr2 = cg["evaluate"]._device_csr(tr2, DEV)
    ids, sc = _topk(cg, fu, fi[:I2].contiguous(), users, csr2, I2)
    o_ids, o_sc = orc.full_rank_topk(fu_np, fi_np[:I2], users, tr2, I2)
    _check_topk(ids.cpu().numpy(), sc.cpu().numpy(), o_ids, o_sc, fu_np, fi_np[:I2], users)
    for prec in PRECS[1:]:
        ids_p, sc_p = _topk(cg, fu, fi[:I2].contiguous(), users, csr2, I2, prec)
        assert torch.equal(ids_p, ids) and torch.equal(sc_p.view(torch.int32), sc.view(torch.int32)), prec


@pytest.mark.parametrize("K", [129, 300, 1000, 4093])
def test_deep_topk_adversarial_scores(cg, K):
    """Exactly representable scores (one non-zero column of small integers), so the expected lists are exact:
    all-equal scores, runs of equal scores that straddle compactions in rising and falling order, a user who has
    seen all but five items (masked items fill the tail in id order at -1e9), a user without train items, and
    k = I."""
    d, I = 16, 4093                                             # k = I is a valid call
    rows = {
        "all-equal": np.ones(I),
        "rising-runs": np.arange(I) // 37,
        "falling-runs": (I - np.arange(I)) // 53,
        "two-levels": (np.arange(I) % 2).astype(np.float64),
        "sawtooth": np.arange(I) % 300,
    }
    users_cols = list(rows.values())
    U = len(users_cols) * 3
    fu = torch.zeros(U, d, device=DEV)
    fi = torch.zeros(I, d, device=DEV)
    # item i carries its score for user pattern p in column p (exact: one non-zero product per chain)
    for p, v in enumerate(users_cols):
        fi[:, p] = torch.tensor(v, dtype=torch.float32, device=DEV)
    masked = []
    indptr, idx = [0], []
    scores = []
    keep = np.array([5, 999, 3000, 4001, 4092])
    for u in range(U):
        p = u % len(users_cols)
        fu[u, p] = 1.0
        scores.append(users_cols[p])
        kind = u // len(users_cols)
        m = np.zeros(0, np.int64) if kind == 0 else (np.setdiff1d(np.arange(I), keep) if kind == 1
                                                        else np.arange(0, I, 3))
        masked.append(m)
        idx.append(m)
        indptr.append(indptr[-1] + m.size)
    tr = (np.array(indptr, np.int64), np.concatenate(idx).astype(np.int64))
    csr = cg["evaluate"]._device_csr(tr, DEV)
    users = np.arange(U, dtype=np.int64)
    for k in (K, I):
        want = _expect_exact(scores, masked, k)
        ids, sc = _topk(cg, fu, fi, users, csr, k)
        ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
        np.testing.assert_array_equal(ids, want)
        want_sc = np.stack([np.where(np.isin(w, m), np.float32(-1e9), np.asarray(s, np.float32)[w])
                            for w, s, m in zip(want, scores, masked)])
        np.testing.assert_array_equal(sc.view(np.uint32), want_sc.astype(np.float32).view(np.uint32))
    r = len(users_cols)                                          # the user who has seen all but `keep`
    np.testing.assert_array_equal(np.sort(ids[r, :5]), keep)
    np.testing.assert_array_equal(ids[r, 5:], np.setdiff1d(np.arange(I), keep))
    assert (sc[r, 5:] == np.float32(-1e9)).all()


def test_deep_topk_chunking_and_repeats_are_bit_identical(cg):
    """CGX_OPT_TOPK_CHUNK_USERS = 1, 7 and the library's choice give the same bits; so do two repeated calls."""
    lib = cg["lib"]
    U, I, d = 150, 3001, 64
    rng = np.random.default_rng(7)
    fu = torch.tensor((rng.standard_normal((U, d)) * 0.2).astype(np.float32), device=DEV)
    fi = torch.tensor((rng.standard_normal((I, d)) * 0.2).astype(np.float32), device=DEV)
    fi[::5] = fi[1]
    csr = cg["evaluate"]._device_csr(_train_rows(rng, U, I), DEV)
    users = np.arange(U, dtype=np.int64)
    keep = lib.get_option("TOPK_CHUNK_USERS")
    try:
        for K in (129, 777):
            lib.set_option("TOPK_CHUNK_USERS", 0)
            ids0, sc0 = _topk(cg, fu, fi, users, csr, K)
            ids0b, sc0b = _topk(cg, fu, fi, users, csr, K)
            assert torch.equal(ids0, ids0b) and torch.equal(sc0.view(torch.int32), sc0b.view(torch.int32))
            for chunk in (1, 7):
                lib.set_option("TOPK_CHUNK_USERS", chunk)
                n_ws = lib.lib().cgx_eval_topk_workspace_bytes(U, I, d, K, 0)
                lib.set_option("TOPK_CHUNK_USERS", 0)
                assert n_ws < lib.lib().cgx_eval_topk_workspace_bytes(U, I, d, K, 0)
                lib.set_option("TOPK_CHUNK_USERS", chunk)
                ids, sc = _topk(cg, fu, fi, users, csr, K)
                assert torch.equal(ids, ids0) and torch.equal(sc.view(torch.int32), sc0.view(torch.int32)), chunk
    finally:
        lib.set_option("TOPK_CHUNK_USERS", keep)


def test_deep_topk_workspace_is_bounded_and_unchanged_up_to_128(cg):
    lib = cg["lib"].lib()
    P = cg["lib"].PRECISIONS
    assert lib.cgx_eval_topk_workspace_bytes(10_000_000, 2_000_000, 128, 20, P["fp32"]) == 256
    assert lib.cgx_eval_topk_workspace_bytes(10_000_000, 2_000_000, 128, 128, P["fp32"]) == 256
    big = [lib.cgx_eval_topk_workspace_bytes(10_000_000, 2_000_000, 128, k, p) for k in (129, 1000, 4096)
           for p in P.values()]
    assert max(big) <= (1 << 30) + (1 << 20)
    assert lib.cgx_eval_topk_uses_tensor_cores(64, 500, P["bf16x3"]) == 0


def test_deep_topk_catalogue_beyond_l2(cg):
    """I = 2^21 items at d = 128 (1 GiB item table), 300 users, k = 1000: the oracle on a sample of users, the
    prefix property against the k = 128 fp32 list on all of them."""
    U, I, d, K = 300, 1 << 21, 128, 1000
    g = torch.Generator(device=DEV).manual_seed(21)
    fu = torch.randn(U, d, device=DEV, generator=g) * 0.2
    fi = torch.randn(I, d, device=DEV, generator=g) * 0.2
    rng = np.random.default_rng(21)
    tr = _train_rows(rng, U, I, max_len=400)
    csr = cg["evaluate"]._device_csr(tr, DEV)
    users = np.arange(U, dtype=np.int64)
    ids, sc = _topk(cg, fu, fi, users, csr, K)
    ids128, sc128 = _topk(cg, fu, fi, users, csr, 128)
    assert torch.equal(ids[:, :128], ids128) and torch.equal(sc[:, :128].view(torch.int32), sc128.view(torch.int32))
    sample = np.array([0, 137, 299])
    fu_np, fi_np = fu.cpu().numpy(), fi.cpu().numpy()
    o_ids, o_sc = orc.full_rank_topk(fu_np, fi_np, sample, tr, K)
    _check_topk(ids.cpu().numpy()[sample], sc.cpu().numpy()[sample], o_ids, o_sc, fu_np, fi_np, sample)


def test_device_metrics_at_deep_cutoffs(cg):
    """cgx_eval_metrics with cut-offs up to 4096 equals the oracle's metrics_from_topk, and the sums of the cut-offs
    <= 256 are bit-identical to those of a call without the deep ones."""
    ev = cg["evaluate"]
    rng = np.random.default_rng(11)
    U, I, n, ld = 400, 6000, 180, 4096
    users = np.sort(rng.choice(U, n, replace=False)).astype(np.int64)
    rows = [np.sort(rng.choice(I, rng.integers(1, 300), replace=False)) for _ in range(U)]
    te_indptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    te_idx = np.concatenate(rows).astype(np.int64)
    ranked = np.stack([rng.permutation(I)[:ld] for _ in range(n)]).astype(np.int32)
    item_pop = rng.integers(0, 500, I).astype(np.int64)
    cred = rng.random(U)
    total = int(item_pop.sum())
    Ks = [10, 20, 300, 1000, 4096]
    te_dev = (torch.tensor(te_indptr, device=DEV), torch.tensor(te_idx, device=DEV, dtype=torch.int32))
    ranked_dev = torch.tensor(ranked, device=DEV)
    got = ev.metrics_device(ranked_dev, users, te_dev, I, Ks, "full", item_pop, total, cred)
    want = orc.metrics_from_topk(ranked.astype(np.int64), users, (te_indptr, te_idx), I, Ks, item_pop, total, cred)
    for K in Ks:
        for k, v in want[K].items():
            if isinstance(v, float):
                assert got[K][k] == pytest.approx(v, rel=1e-10, abs=1e-12), (K, k)
            else:
                assert got[K][k] == v, (K, k)
    users_dev = torch.tensor(users, device=DEV)
    pop_dev = torch.tensor(item_pop, device=DEV)
    flags = torch.tensor((np.arange(n) % 3).astype(np.uint8), device=DEV)
    deep, _ = ev.metrics_sums_device(ranked_dev, users_dev, te_dev, I, Ks, pop_dev, total, flags)
    shallow, _ = ev.metrics_sums_device(ranked_dev[:, :256].contiguous(), users_dev, te_dev, I, [10, 20, 256], pop_dev,
                                        total, flags)
    assert torch.equal(deep[:2].view(torch.int64), shallow[:2].view(torch.int64))
    from credgcn._lib import CgxError
    with pytest.raises(CgxError):
        ev.metrics_sums_device(torch.zeros(4, 4097, dtype=torch.int32, device=DEV), users_dev[:4], te_dev, I, [4097])


def test_evaluate_full_ranking_deep_cutoffs_match_oracle(cg):
    """evaluate_full_ranking with cfg.Ks = (20, 500), V2 extra keys included, against the oracle's
    evaluate_full_ranking; the host metrics path gives the same dict."""
    config, ev = cg["config"], cg["evaluate"]
    rng = np.random.default_rng(5)
    U, I, d = 500, 2500, 64
    fu_np = (rng.standard_normal((U, d)) * 0.3).astype(np.float32)
    fi_np = (rng.standard_normal((I, d)) * 0.3).astype(np.float32)
    tr = _train_rows(rng, U, I)
    te = _train_rows(rng, U, I, max_len=30)
    item_pop = np.bincount(tr[1], minlength=I).astype(np.int64)
    total = int(item_pop.sum())
    cred = rng.random(U)
    net = types.SimpleNamespace(final_embeddings=lambda: (torch.tensor(fu_np, device=DEV),
                                                          torch.tensor(fi_np, device=DEV)))
    keep = config.cfg
    try:
        for on_device in (True, False):
            cfg = config.CFG()
            cfg.Ks, cfg.metrics_on_device = (20, 500), on_device
            config.cfg = cfg
            got = ev.evaluate_full_ranking(net, tr, te, I, DEV, item_pop, total, cred)
            want = orc.evaluate_full_ranking(fu_np, fi_np, tr, te, I, (20, 500), item_pop, total, cred)
            for K in (20, 500):
                assert set(want[K]) <= set(got[K])
                for k, v in want[K].items():
                    if isinstance(v, float):
                        assert got[K][k] == pytest.approx(v, rel=1e-4, abs=1e-6), (on_device, K, k)
                    else:
                        assert got[K][k] == v, (on_device, K, k)
    finally:
        config.cfg = keep


def test_training_loop_with_deep_cutoff(cg):
    """train_on_arrays validates and tests with cfg.Ks = (20, 200) under eval_mode = "full"."""
    sg = cg["synth"].make_graph("C1", num_users=300, num_items=400, num_edges=12_000)
    config = cg["config"]
    cfg = config.CFG()
    cfg.device, cfg.variant, cfg.epochs, cfg.batch_size, cfg.eval_mode = DEV, "v2", 2, 128, "full"
    cfg.eval_every, cfg.Ks = 1, (20, 200)
    keep = config.cfg
    config.cfg = cfg
    try:
        torch.manual_seed(0)
        _, res = cg["train"].train_on_arrays(sg.train_edges, sg.val_edges, sg.test_edges, sg.num_users, sg.num_items,
                                             sg.cred, None, cfg)
    finally:
        config.cfg = keep
    assert res[200]["mode"] == "full" and res[200]["recall"] >= res[20]["recall"]


def test_deep_topk_errors(cg):
    from credgcn._lib import CgxError
    U, I, d = 4, 5000, 32
    fu, fi = torch.zeros(U, d, device=DEV), torch.zeros(I, d, device=DEV)
    csr = cg["evaluate"]._device_csr((np.zeros(U + 1, np.int64), np.zeros(0, np.int64)), DEV)
    with pytest.raises(CgxError, match="4096"):
        _topk(cg, fu, fi, np.arange(U), csr, 4097)
    with pytest.raises(CgxError):
        _topk(cg, fu, fi[:300], np.arange(U), csr, 301)
