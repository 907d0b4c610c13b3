"""Evaluation with the reference's entry points: the per-user Python loops of the reference
become one device top-K (or candidate-scoring) call plus vectorised NumPy metrics.

    metrics_at_k                 lightgcn_cu.py:469-484, Version-2/lighgcn_cu_pop.py:514-530
    evaluate_sampled             lightgcn_cu.py:487-546, lighgcn_cu_pop.py:536-650
    evaluate_full_ranking        lighgcn_cu_pop.py:653-752 (version_1/lightgcn_cu_message.py:535-585 short form)
    compute_item_popularity / novelty_stats_for_items / make_cred_groups   lighgcn_cu_pop.py:382-423
"""
from __future__ import annotations

import ctypes
import math

import numpy as np
import torch

from . import _lib, config
from ._lib import check, lib, ptr, stream_ptr, workspace
from .sampler import user_has_item


def metrics_at_k(ranked_items, gt_set, K):
    topk = ranked_items[:K]
    hits = [1 if int(x) in gt_set else 0 for x in topk]
    n_hit = sum(hits)
    dcg = sum(1.0 / math.log2(r + 2) for r, h in enumerate(hits) if h)
    idcg = sum(1.0 / math.log2(r + 2) for r in range(min(len(gt_set), K)))
    return n_hit / K, n_hit / max(len(gt_set), 1), (dcg / idcg) if idcg > 0 else 0.0


def compute_item_popularity(train_edges_2xE: np.ndarray, num_items: int):
    pop = np.bincount(np.asarray(train_edges_2xE[1], dtype=np.int64), minlength=num_items).astype(np.int64)
    return pop, int(pop.sum())


def novelty_stats_for_items(item_ids, pop: np.ndarray, total_train: int, num_items: int):
    item_ids = np.asarray(item_ids, dtype=np.int64)
    if item_ids.size == 0:
        return 0.0, 0.0
    p = pop[item_ids]
    return float(np.log(p + 1.0).mean()), float((-np.log2((p + 1.0) / (total_train + num_items))).mean())


def make_cred_groups(users: np.ndarray, cred: np.ndarray, pct: float):
    if users.size == 0:
        return np.array([], dtype=np.int64), np.array([], dtype=np.int64)
    k = max(int(round(users.size * pct)), 1)
    order = np.argsort(cred[users])
    return users[order[-k:]].astype(np.int64), users[order[:k]].astype(np.int64)


# ------------------------------------------------------------------------------------------
def _device_csr(csr, device):
    indptr, indices = csr
    ip = torch.as_tensor(indptr).to(device=device, dtype=torch.int64).contiguous()
    ix = torch.as_tensor(indices).to(device=device, dtype=torch.int32).contiguous()
    if ix.numel() == 0:
        ix = torch.zeros(1, dtype=torch.int32, device=device)
    return ip, ix


def topk_device(f_u, f_i, users, train_csr_dev, K: int, precision: str = "fp32"):
    """ids int32[n, K], scores float32[n, K] for `users` (int64 CUDA tensor): train items masked to
    -1e9, order = (score desc, item id asc)."""
    dev = f_u.device
    f_u, f_i = f_u.detach().contiguous(), f_i.detach().contiguous()
    users = torch.as_tensor(users, device=dev).to(torch.int64).contiguous()
    n, I, d = users.numel(), f_i.shape[0], f_i.shape[1]
    ids = torch.empty(n, K, dtype=torch.int32, device=dev)
    sc = torch.empty(n, K, dtype=torch.float32, device=dev)
    ip, ix = train_csr_dev
    prec = _lib.PRECISIONS[precision]
    ws = workspace(lib().cgx_eval_topk_workspace_bytes(n, I, d, K, prec), dev)
    with torch.cuda.device(dev):
        check(lib().cgx_eval_topk(ptr(users), n, ptr(f_u), ptr(f_i), I, d, ptr(ip), ptr(ix), K, prec, ptr(ids),
                                  ptr(sc), ptr(ws), ws.numel(), stream_ptr(dev)))
    return ids, sc


def score_candidates_device(f_u, f_i, users, cands):
    dev = f_u.device
    f_u, f_i = f_u.detach().contiguous(), f_i.detach().contiguous()
    users = torch.as_tensor(users, device=dev).to(torch.int64).contiguous()
    cands = torch.as_tensor(cands, device=dev).to(torch.int64).contiguous()
    n, c = cands.shape
    out = torch.empty(n, c, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        check(lib().cgx_score_candidates(ptr(users), ptr(cands), n, c, f_i.shape[1], ptr(f_u), ptr(f_i), ptr(out),
                                         stream_ptr(dev)))
    return out


def _hits_matrix(ranked: np.ndarray, users: np.ndarray, test_csr, num_items: int, gt_single=None) -> np.ndarray:
    """hits[r, j] = ranked[r, j] is a ground-truth item of users[r]."""
    if gt_single is not None:
        return ranked == gt_single[:, None]
    indptr, indices = test_csr
    rows = np.repeat(np.arange(len(indptr) - 1, dtype=np.int64), np.diff(indptr))
    keys = rows * num_items + np.asarray(indices, dtype=np.int64)         # sorted: CSR is (user, item) ordered
    q = users[:, None].astype(np.int64) * num_items + ranked.astype(np.int64)
    pos = np.searchsorted(keys, q)
    pos = np.minimum(pos, max(keys.size - 1, 0))
    return keys[pos] == q if keys.size else np.zeros_like(q, dtype=bool)


def metrics_from_ranked(ranked: np.ndarray, users: np.ndarray, test_csr, num_items: int, Ks, mode: str,
                        item_pop=None, total_train=0, cred_np=None, group_pct=0.20, gt_single=None, extra_keys=None):
    """The reference's result dict from a [n_users, >=max(Ks)] matrix of ranked item ids."""
    n = len(users)
    hits = _hits_matrix(ranked[:, : max(Ks)], users, test_csr, num_items, gt_single)
    n_gt = np.ones(n, np.int64) if gt_single is not None else np.diff(test_csr[0])[users]
    disc = 1.0 / np.log2(np.arange(max(Ks)) + 2.0)
    idcg_tab = np.concatenate([[0.0], np.cumsum(disc)])
    extra = item_pop is not None and cred_np is not None
    if extra:
        hi, lo = make_cred_groups(users, cred_np, group_pct)
        in_hi, in_lo = np.isin(users, hi), np.isin(users, lo)
    out = {}
    for K in Ks:
        h = hits[:, :K]
        nh = h.sum(1)
        recall = nh / np.maximum(n_gt, 1)
        idcg = idcg_tab[np.minimum(n_gt, K)]
        ndcg = np.where(idcg > 0, (h * disc[:K]).sum(1) / np.where(idcg > 0, idcg, 1.0), 0.0)
        res = {"precision": float((nh / K).mean()), "recall": float(recall.mean()), "ndcg": float(ndcg.mean())}
        if extra:
            top = ranked[:, :K].astype(np.int64)
            p = item_pop[top].astype(np.float64)
            res.update({
                "item_coverage": np.unique(top).size / max(num_items, 1),
                "avg_log_popularity": float(np.log(p + 1.0).mean(1).mean()),
                "avg_self_information": float((-np.log2((p + 1.0) / (total_train + num_items))).mean(1).mean()),
                "cred_utility": float(np.asarray(cred_np, np.float64)[users].mean()),
                "high_cred_recall": float(recall[in_hi].sum() / max(int(in_hi.sum()), 1)),
                "low_cred_recall": float(recall[in_lo].sum() / max(int(in_lo.sum()), 1)),
                "high_users": int(in_hi.sum()), "low_users": int(in_lo.sum()),
            })
        res.update({"users_eval": n, "mode": mode})
        if extra_keys:
            res.update(extra_keys)
        out[K] = res
    return out


def metrics_sums_device(ranked_dev: torch.Tensor, users_dev, test_csr_dev, num_items: int, ks, item_pop_dev=None,
                        total_train=0, flags_dev=None, gt_single_dev=None, with_coverage=False):
    """(sums float64[len(ks), 7], bitmaps int32[len(ks), ceil(I/32)] | None) on the device: the per-rank part of
    the metrics (cgx_eval_metrics); `ks` ascending."""
    dev = ranked_dev.device
    n = ranked_dev.shape[0]
    out = torch.zeros(len(ks), 7, dtype=torch.float64, device=dev)
    bitmaps = torch.zeros(len(ks), (num_items + 31) // 32, dtype=torch.int32, device=dev) if with_coverage else None
    if n == 0:
        return out, bitmaps
    ranked_dev = ranked_dev.to(torch.int32).contiguous()
    ks_host = (ctypes.c_int32 * len(ks))(*ks)
    ws = workspace(lib().cgx_eval_metrics_workspace_bytes(n, len(ks)), dev)
    gt = None if gt_single_dev is None else gt_single_dev.to(torch.int32).contiguous()
    ip, ix = test_csr_dev if test_csr_dev is not None else (None, None)
    opt = lambda t: None if t is None else ptr(t)   # noqa: E731
    with torch.cuda.device(dev):
        check(lib().cgx_eval_metrics(ptr(ranked_dev), n, ranked_dev.shape[1], opt(users_dev), opt(ip), opt(ix), opt(gt),
                                     num_items, ks_host, len(ks), opt(item_pop_dev), int(total_train), opt(flags_dev),
                                     opt(bitmaps), ptr(out), ptr(ws), ws.numel(), stream_ptr(dev)))
    return out, bitmaps


def coverage_counts_device(bitmaps: torch.Tensor, num_items: int) -> torch.Tensor:
    counts = torch.empty(bitmaps.shape[0], dtype=torch.int64, device=bitmaps.device)
    with torch.cuda.device(bitmaps.device):
        check(lib().cgx_eval_coverage(ptr(bitmaps), num_items, bitmaps.shape[0], ptr(counts),
                                      stream_ptr(bitmaps.device)))
    return counts


def metrics_result(Ks, ks, sums, counts, n: int, num_items: int, mode: str, groups=None, extra_keys=None):
    """The reference's result dict from the device sums; groups = (n_high, n_low, cred_utility) or None."""
    res_all = {}
    for K in Ks:
        ki = ks.index(int(K))
        s = sums[ki]
        res = {"precision": float(s[0] / n), "recall": float(s[1] / n), "ndcg": float(s[2] / n)}
        if groups is not None:
            n_hi, n_lo, cred_utility = groups
            res.update({
                "item_coverage": int(counts[ki]) / max(num_items, 1),
                "avg_log_popularity": float(s[3] / n),
                "avg_self_information": float(s[4] / n),
                "cred_utility": float(cred_utility),
                "high_cred_recall": float(s[5] / max(n_hi, 1)),
                "low_cred_recall": float(s[6] / max(n_lo, 1)),
                "high_users": int(n_hi), "low_users": int(n_lo),
            })
        res.update({"users_eval": n, "mode": mode})
        if extra_keys:
            res.update(extra_keys)
        res_all[K] = res
    return res_all


def metrics_device(ranked_dev: torch.Tensor, users, test_csr_dev, num_items: int, Ks, mode: str, item_pop=None,
                   total_train=0, cred_np=None, group_pct=0.20, gt_single_dev=None, extra_keys=None):
    """metrics_from_ranked computed on the device (cgx_eval_metrics + cgx_eval_coverage): the ranked ids stay
    in HBM and 7 sums + one count per cut-off come back.  Same result dict (double accumulation; the means
    agree with the NumPy path to ~1e-13 relative, the order of the additions differs)."""
    dev = ranked_dev.device
    users_np = np.asarray(users, dtype=np.int64)
    ks = sorted(set(int(k) for k in Ks))
    extra = item_pop is not None and cred_np is not None
    pop_dev = flags_dev = groups = None
    if extra:
        hi, lo = make_cred_groups(users_np, cred_np, group_pct)
        in_hi, in_lo = np.isin(users_np, hi), np.isin(users_np, lo)
        flags_dev = torch.from_numpy(in_hi.astype(np.uint8) + 2 * in_lo.astype(np.uint8)).to(dev)   # bit 0 high, bit 1 low
        pop_dev = torch.as_tensor(np.asarray(item_pop, dtype=np.int64)).to(dev)
        groups = (int(in_hi.sum()), int(in_lo.sum()), np.asarray(cred_np, np.float64)[users_np].mean())
    sums, bitmaps = metrics_sums_device(ranked_dev, torch.from_numpy(users_np).to(dev), test_csr_dev, num_items, ks,
                                        pop_dev, total_train, flags_dev, gt_single_dev, with_coverage=extra)
    counts = coverage_counts_device(bitmaps, num_items).cpu().numpy() if extra else None
    return metrics_result(Ks, ks, sums.cpu().numpy(), counts, users_np.size, num_items, mode, groups, extra_keys)


def _final_tables(model):
    with torch.no_grad():
        return model.final_embeddings() if hasattr(model, "final_embeddings") else model.get_user_item_emb()


@torch.no_grad()
def evaluate_full_ranking(model, train_csr, test_csr, num_items: int, device=None, item_pop=None,
                          total_train_interactions: int = 0, cred_np=None, precision: str | None = None):
    """Full-catalogue ranking of every user with >= 1 test item; train items masked (val items
    are NOT masked when testing, as in the reference, lighgcn_cu_pop.py:699-702)."""
    cfg = config.cfg
    f_u, f_i = _final_tables(model)
    indptr_te = np.asarray(test_csr[0])
    users = np.flatnonzero(np.diff(indptr_te) > 0).astype(np.int64)
    if users.size == 0:
        raise RuntimeError("No users with test interactions. Check your split or threshold.")
    K = max(cfg.Ks)
    ids, _ = topk_device(f_u, f_i, torch.from_numpy(users), _device_csr(train_csr, f_u.device), K,
                         precision or cfg.score_precision)
    if cfg.metrics_on_device:
        return metrics_device(ids, users, _device_csr(test_csr, f_u.device), num_items, cfg.Ks, "full", item_pop,
                              total_train_interactions, cred_np, cfg.cred_group_pct)
    ranked = ids.cpu().numpy()
    return metrics_from_ranked(ranked, users, (indptr_te, np.asarray(test_csr[1])), num_items, cfg.Ks, "full",
                               item_pop, total_train_interactions, cred_np, cfg.cred_group_pct)


def sampled_candidates(train_csr, test_csr, num_items: int, n_neg: int, seed: int):
    """Candidate lists of the sampled protocol, drawn exactly as the reference draws them
    (default_rng(seed + 999), 1 test positive + n_neg negatives outside test U train;
    lightgcn_cu.py:496-521) so that both sides rank identical candidates."""
    indptr_tr, indices_tr = train_csr
    indptr_te, indices_te = test_csr
    rng = np.random.default_rng(seed + 999)
    users = np.flatnonzero(np.diff(indptr_te) > 0).astype(np.int64)
    cands = np.empty((users.size, 1 + n_neg), dtype=np.int64)
    for r, u in enumerate(users):
        gt = indices_te[indptr_te[u]:indptr_te[u + 1]]
        gt_set = set(map(int, gt.tolist()))
        cands[r, 0] = int(gt[rng.integers(0, len(gt))])
        k = 1
        while k <= n_neg:
            j = int(rng.integers(0, num_items))
            if j in gt_set or user_has_item(indptr_tr, indices_tr, int(u), j):
                continue
            cands[r, k] = j
            k += 1
    return users, cands


def sampled_candidates_device(train_csr_dev, test_csr_dev, users, num_items: int, n_neg: int, seed: int,
                              row_base: int = 0):
    """Candidate lists of the sampled protocol drawn by one kernel (cgx_eval_candidates).  row_base: the rows of
    this call are rows row_base.. of a whole list (a shard gets the lists the whole call gives the same rows)."""
    dev = train_csr_dev[0].device
    users = torch.as_tensor(users, device=dev).to(torch.int64).contiguous()
    cand = torch.empty(users.numel(), 1 + n_neg, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        check(lib().cgx_eval_candidates(ptr(users), users.numel(), ptr(train_csr_dev[0]), ptr(train_csr_dev[1]),
                                        ptr(test_csr_dev[0]), ptr(test_csr_dev[1]), num_items, n_neg,
                                        (int(seed) + 999) & 0xFFFFFFFFFFFFFFFF, ptr(cand), stream_ptr(dev),
                                        int(row_base)))
    return cand


def rank_candidates_device(scores: torch.Tensor, cands: torch.Tensor) -> torch.Tensor:
    ranked = torch.empty_like(cands)
    with torch.cuda.device(scores.device):
        check(lib().cgx_rank_candidates(ptr(scores.contiguous()), ptr(cands.contiguous()), cands.shape[0],
                                        cands.shape[1], ptr(ranked), stream_ptr(scores.device)))
    return ranked


@torch.no_grad()
def evaluate_sampled(model, train_csr, test_csr, num_items: int, device=None, item_pop=None,
                     total_train_interactions: int = 0, cred_np=None, candidates=None, on_device=None):
    """1 positive + cfg.sampled_negatives negatives per test user, ranked by score.
    `candidates=(users, cands)` injects a candidate list (parity tests); `on_device` (default
    cfg.sampled_eval_on_device) draws the candidates with the device kernel instead of the host PCG64 loop."""
    cfg = config.cfg
    f_u, f_i = _final_tables(model)
    tr = (np.asarray(train_csr[0]), np.asarray(train_csr[1]))
    te = (np.asarray(test_csr[0]), np.asarray(test_csr[1]))
    on_device = cfg.sampled_eval_on_device if on_device is None else on_device
    if candidates is not None:
        users, cands = candidates
        cands_dev = torch.from_numpy(np.ascontiguousarray(cands)).to(f_u.device)
    elif on_device:
        users = np.flatnonzero(np.diff(te[0]) > 0).astype(np.int64)
        if len(users) == 0:
            raise RuntimeError("No users with test interactions.")
        cands_dev = sampled_candidates_device(_device_csr(tr, f_u.device), _device_csr(te, f_u.device), users,
                                              num_items, cfg.sampled_negatives, cfg.seed)
    else:
        users, cands = sampled_candidates(tr, te, num_items, cfg.sampled_negatives, cfg.seed)
        cands_dev = torch.from_numpy(cands).to(f_u.device) if len(users) else None
    if len(users) == 0:
        raise RuntimeError("No users with test interactions.")
    scores = score_candidates_device(f_u, f_i, torch.from_numpy(np.asarray(users)), cands_dev)
    ranked_dev = rank_candidates_device(scores, cands_dev)
    if cfg.metrics_on_device:
        return metrics_device(ranked_dev, users, None, num_items, cfg.Ks, "sampled(1pos+neg)", item_pop,
                              total_train_interactions, cred_np, cfg.cred_group_pct, gt_single_dev=cands_dev[:, 0],
                              extra_keys={"negatives": cfg.sampled_negatives})
    ranked = ranked_dev.cpu().numpy()
    cands = cands_dev.cpu().numpy()
    return metrics_from_ranked(ranked, users, te, num_items, cfg.Ks, "sampled(1pos+neg)", item_pop,
                               total_train_interactions, cred_np, cfg.cred_group_pct, gt_single=cands[:, 0],
                               extra_keys={"negatives": cfg.sampled_negatives})
