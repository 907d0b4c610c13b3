"""CPU oracle for the credibility-aware LightGCN hot path.  TEST INFRASTRUCTURE ONLY.

This file restates, in NumPy (+ SciPy CSR products, + a torch-CPU autograd leg used only
as the timed CPU baseline), what the reference computes on the path named by
BASELINE.json.  Nothing under the product package imports it: only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference` legs may.

Pinning: the reference has no tests or golden vectors of its own (SURVEY.md section 8c), so the
oracle is pinned against OUTPUTS OF THE REFERENCE ITSELF, produced in the build container
by `tests/golden/make_golden.py` (imports /root/reference/*.py by path) and committed as
`tests/golden/*.npz`; `tests/test_oracle_golden.py` replays them.  Versions the fixtures
were made with: torch 2.11.0+cu128, numpy 2.3.5.

Reference files (relative to /root/reference):
    CU  = lightgcn_cu.py
    V2  = Version-2/lighgcn_cu_pop.py
    DA  = version_1/lightgcn_cu_pop_Degree-Aware Message.py

Naming used here (the reference swaps M_ui/M_iu between CU and V2, so neither is used):
    A : [U x I] user-row operator, base weight           (CU `M_iu`, V2 `M_ui`)
    C : [I x U] item-row operator, credibility weighted  (CU `M_ui`, V2 `M_iu`)
"""
from __future__ import annotations

import math

import numpy as np
import scipy.sparse as sp

F32 = np.float32


# --------------------------------------------------------------------------------------
# a1. user-row CSR used by the samplers and the evaluators           (CU:259-276, V2:309-327)
# --------------------------------------------------------------------------------------
def edges_to_user_csr(edges_2xE: np.ndarray, num_users: int):
    """Rows = users, neighbours ascending, duplicate (u, i) pairs kept.

    The reference does a stable sort by user followed by a per-row sort (CU:263-275); a
    single lexicographic sort on (user, item) yields the same arrays."""
    u = np.asarray(edges_2xE[0], dtype=np.int64)
    it = np.asarray(edges_2xE[1], dtype=np.int64)
    order = np.lexsort((it, u))
    indptr = np.zeros(num_users + 1, dtype=np.int64)
    np.cumsum(np.bincount(u, minlength=num_users), out=indptr[1:])
    return indptr, it[order]


def row_contains(indptr, indices, user: int, item: int) -> bool:
    """Binary-search membership test on one CSR row (CU:279-285)."""
    lo, hi = int(indptr[user]), int(indptr[user + 1])
    if lo == hi:
        return False
    j = lo + int(np.searchsorted(indices[lo:hi], item))
    return j < hi and int(indices[j]) == item


# --------------------------------------------------------------------------------------
# a3 / a4 / a5. degrees and per-edge weights, NumPy float32 semantics
# --------------------------------------------------------------------------------------
def degrees(edges_2xE: np.ndarray, num_users: int, num_items: int):
    """bincount -> float32, duplicates counted (CU:383-384, V2:433-434)."""
    u = np.asarray(edges_2xE[0], dtype=np.int64)
    i = np.asarray(edges_2xE[1], dtype=np.int64)
    return (np.bincount(u, minlength=num_users).astype(F32),
            np.bincount(i, minlength=num_items).astype(F32))


def damping_alpha(deg_i: np.ndarray) -> np.ndarray:
    """DA:379-380: alpha_i = 1 / log1p(max(deg_i, 1)), float32 (NumPy's log1p, not libdevice's)."""
    return (F32(1.0) / np.log1p(np.maximum(deg_i.astype(F32), F32(1.0)))).astype(F32)


def edge_weights(variant: str, u: np.ndarray, i: np.ndarray, deg_u: np.ndarray, deg_i: np.ndarray,
                 cred: np.ndarray):
    """Per-edge (w_A, w_C) for the three builders.

    cu : denom = sqrt(max(du*di, 1e-12)); w_C = c_u/denom; w_A = 1/denom          (CU:386-389)
    v2 : w_A = (1/sqrt(max(du,1))) * (1/sqrt(max(di,1))); w_C = c_u * w_A          (V2:436-446)
    da : w_A = v2.w_A * alpha_i; w_C = c_u * w_A                                   (DA:365-392)
    Every op is a correctly rounded float32 op; no fused multiply-add."""
    cred = np.asarray(cred, dtype=F32)
    if variant == "cu":
        denom = np.sqrt(np.maximum(deg_u[u] * deg_i[i], F32(1e-12))).astype(F32)
        w_c = (cred[u] / denom).astype(F32)
        w_a = (F32(1.0) / denom).astype(F32)
        return w_a, w_c
    if variant not in ("v2", "da"):
        raise ValueError(f"unknown variant {variant!r}")
    isu = (F32(1.0) / np.sqrt(np.maximum(deg_u, F32(1.0)))).astype(F32)
    isi = (F32(1.0) / np.sqrt(np.maximum(deg_i, F32(1.0)))).astype(F32)
    w_a = (isu[u] * isi[i]).astype(F32)
    if variant == "da":
        w_a = (w_a * damping_alpha(deg_i)[i]).astype(F32)
    w_c = (cred[u] * w_a).astype(F32)
    return w_a, w_c


def coalesce(rows: np.ndarray, cols: np.ndarray, vals: np.ndarray):
    """torch `.coalesce()` on CPU: sort by (row, col), add duplicates left to right in fp32
    (CU:393,397; V2:443,450).  Explicit zeros stay in the pattern."""
    order = np.lexsort((cols, rows))
    r, c, v = rows[order], cols[order], vals[order].astype(F32)
    if r.size == 0:
        return r, c, v
    head = np.ones(r.size, dtype=bool)
    head[1:] = (r[1:] != r[:-1]) | (c[1:] != c[:-1])
    if head.all():
        return r, c, v
    starts = np.flatnonzero(head)
    mult = np.diff(np.append(starts, r.size))
    out = v[starts].copy()
    for k in range(1, int(mult.max())):           # k-th repeat of each run, in order
        sel = mult > k
        out[sel] = (out[sel] + v[starts[sel] + k]).astype(F32)
    return r[starts], c[starts], out


class Operators:
    """Both coalesced operators of one graph, plus everything the reference derives from it."""

    def __init__(self, edges_2xE, num_users, num_items, cred, variant: str):
        self.U, self.I, self.variant = int(num_users), int(num_items), variant
        u = np.asarray(edges_2xE[0], dtype=np.int64)
        i = np.asarray(edges_2xE[1], dtype=np.int64)
        self.deg_u, self.deg_i = degrees(edges_2xE, num_users, num_items)
        w_a, w_c = edge_weights(variant, u, i, self.deg_u, self.deg_i, cred)
        self.A_row, self.A_col, self.A_val = coalesce(u, i, w_a)     # [U x I]
        self.C_row, self.C_col, self.C_val = coalesce(i, u, w_c)     # [I x U]
        self.A = sp.csr_matrix((self.A_val, (self.A_row, self.A_col)), shape=(self.U, self.I), dtype=F32)
        self.C = sp.csr_matrix((self.C_val, (self.C_row, self.C_col)), shape=(self.I, self.U), dtype=F32)
        self.At = self.A.T.tocsr()
        self.Ct = self.C.T.tocsr()


# --------------------------------------------------------------------------------------
# a7 / a8. K-layer propagation + layer mean; a9. its backward
# --------------------------------------------------------------------------------------
def propagate(ops: Operators, e0_u: np.ndarray, e0_i: np.ndarray, num_layers: int, order: str):
    """order='jacobi' -> CU:429-437 (both products read layer k);
    order='gs' -> V2:482-486 (user update reads the NEW item layer).  Mean over K+1 layers
    as stack(...).mean(0) (CU:446-447, V2:488-489)."""
    u, i = e0_u.astype(F32), e0_i.astype(F32)
    us, is_ = [u], [i]
    for _ in range(num_layers):
        if order == "jacobi":
            i_new = (ops.C @ u).astype(F32)
            u_new = (ops.A @ i).astype(F32)
        elif order == "gs":
            i_new = (ops.C @ u).astype(F32)
            u_new = (ops.A @ i_new).astype(F32)
        else:
            raise ValueError(order)
        u, i = u_new, i_new
        us.append(u)
        is_.append(i)
    fu = np.stack(us, 0).mean(0, dtype=F32)
    fi = np.stack(is_, 0).mean(0, dtype=F32)
    return fu, fi


def propagate_backward(ops: Operators, g_u: np.ndarray, g_i: np.ndarray, num_layers: int, order: str):
    """Adjoint of `propagate` (what autograd does for CU:651 / V2:862); SURVEY.md appendix C."""
    s = F32(1.0 / (num_layers + 1))
    su, si = (s * g_u).astype(F32), (s * g_i).astype(F32)
    if order == "jacobi":
        bu, bi = su, si
        for _ in range(num_layers):
            bu, bi = (su + ops.Ct @ bi).astype(F32), (si + ops.At @ bu).astype(F32)
        return bu, bi
    bu = su
    for _ in range(num_layers):
        bi = (si + ops.At @ bu).astype(F32)
        bu = (su + ops.Ct @ bi).astype(F32)
    return bu, si


# --------------------------------------------------------------------------------------
# a10 / a11. BPR + L2 (+ fairness) on a triple batch, value and gradients
# --------------------------------------------------------------------------------------
def bpr_loss(f_u, f_i, e0_u, e0_i, users, pos, neg, reg_weight, fair_weight=0.0, pop=None):
    """L = -mean(log(sigmoid(y+ - y-) + 1e-12)) + fair*mean(pop[pos]*y+) + reg*mean(|e0_u|^2+|e0_p|^2+|e0_n|^2)
    (CU:635-648 with CU:450-463; V2:495-508 is the fair_weight=0 case).

    Returns loss and the four dense gradients (d f_u, d f_i, d e0_u, d e0_i) of L with the
    propagated tables treated as independent inputs."""
    B = len(users)
    fu, fp, fn = f_u[users].astype(F32), f_i[pos].astype(F32), f_i[neg].astype(F32)
    y_pos = (fu * fp).sum(1, dtype=F32)
    y_neg = (fu * fn).sum(1, dtype=F32)
    x = (y_pos - y_neg).astype(np.float64)
    sig = 1.0 / (1.0 + np.exp(-x))
    l_bpr = -np.log(sig + 1e-12).mean()
    l_fair = float((pop[pos].astype(np.float64) * y_pos).mean()) if (pop is not None and fair_weight) else 0.0
    eu, ep, en = e0_u[users].astype(np.float64), e0_i[pos].astype(np.float64), e0_i[neg].astype(np.float64)
    l_reg = ((eu ** 2).sum(1) + (ep ** 2).sum(1) + (en ** 2).sum(1)).mean()
    loss = l_bpr + fair_weight * l_fair + reg_weight * l_reg

    gx = (-(sig * (1.0 - sig)) / (sig + 1e-12) / B)                    # dL/dx
    gyp = gx + (fair_weight * pop[pos].astype(np.float64) / B if (pop is not None and fair_weight) else 0.0)
    gyn = -gx
    d_fu = np.zeros(f_u.shape, np.float64)
    d_fi = np.zeros(f_i.shape, np.float64)
    np.add.at(d_fu, users, gyp[:, None] * fp + gyn[:, None] * fn)
    np.add.at(d_fi, pos, gyp[:, None] * fu)
    np.add.at(d_fi, neg, gyn[:, None] * fu)
    d_e0u = np.zeros(e0_u.shape, np.float64)
    d_e0i = np.zeros(e0_i.shape, np.float64)
    c = 2.0 * reg_weight / B
    np.add.at(d_e0u, users, c * eu)
    np.add.at(d_e0i, pos, c * ep)
    np.add.at(d_e0i, neg, c * en)
    return float(loss), d_fu.astype(F32), d_fi.astype(F32), d_e0u.astype(F32), d_e0i.astype(F32)


def train_step_grads(ops, e0_u, e0_i, users, pos, neg, num_layers, order, reg_weight,
                     fair_weight=0.0, pop=None):
    """Loss and d loss / d ego tables for one step: forward, loss, backward (CU:632-651)."""
    f_u, f_i = propagate(ops, e0_u, e0_i, num_layers, order)
    loss, d_fu, d_fi, d_e0u, d_e0i = bpr_loss(f_u, f_i, e0_u, e0_i, users, pos, neg,
                                              reg_weight, fair_weight, pop)
    b_u, b_i = propagate_backward(ops, d_fu, d_fi, num_layers, order)
    return loss, (b_u + d_e0u).astype(F32), (b_i + d_e0i).astype(F32), f_u, f_i


def bpr_rows_f64(f_u, f_i, e0_u, e0_i, users, pos, neg, reg_weight, fair_weight=0.0, pop=None, batch_total=0):
    """The fused loss of `bpr_loss` in float64 throughout, with the means over `batch_total` triples (a shard of a
    larger batch; 0 = len(users)).  Besides the loss and d f_u / d f_i it returns, per gradient element, the sum of
    the absolute values of the terms that make it up (S_u, S_i): the scale an fp32 sum of those terms is accurate
    to, row by row, whatever the other rows hold.  `mult_u` / `mult_i`: how many plan entries each row has (the
    L2 gradient of a row is mult * 2 reg / batch_total * e0)."""
    users, pos, neg = (np.asarray(x, np.int64) for x in (users, pos, neg))
    Bt = float(batch_total or len(users))
    fu, fp, fn = (np.asarray(x, np.float64) for x in (f_u[users], f_i[pos], f_i[neg]))
    y_pos, y_neg = (fu * fp).sum(1), (fu * fn).sum(1)
    sig = 1.0 / (1.0 + np.exp(-(y_pos - y_neg)))
    pw = fair_weight * np.asarray(pop, np.float64)[pos] if (pop is not None and fair_weight) else np.zeros(len(users))
    l2 = sum((np.asarray(e[r], np.float64) ** 2).sum(1) for e, r in ((e0_u, users), (e0_i, pos), (e0_i, neg)))
    terms = -np.log(sig + 1e-12) + pw * y_pos + reg_weight * l2
    gx = -(sig * (1.0 - sig)) / (sig + 1e-12) / Bt
    cp, cn = gx + pw / Bt, -gx
    d_fu, s_u = np.zeros(f_u.shape), np.zeros(f_u.shape)
    d_fi, s_i = np.zeros(f_i.shape), np.zeros(f_i.shape)
    for d, s, rows, a, b in ((d_fu, s_u, users, cp[:, None] * fp, cn[:, None] * fn), (d_fi, s_i, pos, cp[:, None] * fu, 0),
                             (d_fi, s_i, neg, cn[:, None] * fu, 0)):
        np.add.at(d, rows, a + b)
        np.add.at(s, rows, np.abs(a) + np.abs(b))
    mult_u = np.bincount(users, minlength=f_u.shape[0])
    mult_i = np.bincount(pos, minlength=f_i.shape[0]) + np.bincount(neg, minlength=f_i.shape[0])
    return dict(loss=float(terms.sum() / Bt), loss_abs=float(np.abs(terms).sum() / Bt), d_fu=d_fu, d_fi=d_fi,
                s_u=s_u, s_i=s_i, mult_u=mult_u, mult_i=mult_i)


# --------------------------------------------------------------------------------------
# Adam (torch.optim.Adam defaults: no weight decay, no amsgrad) and a multi-step driver
# --------------------------------------------------------------------------------------
def adam_step_f64(p, g, m, v, t, lr=1e-3, betas=(0.9, 0.999), eps=1e-8):
    """Step t (1-based) of torch.optim.Adam in float64 on one table; returns the new (p, m, v)."""
    b1, b2 = betas
    g = np.asarray(g, np.float64)
    m = b1 * m + (1.0 - b1) * g
    v = b2 * v + (1.0 - b2) * g * g
    step = lr / (1.0 - b1 ** t) * m / (np.sqrt(v) / math.sqrt(1.0 - b2 ** t) + eps)
    return np.asarray(p, np.float64) - step, m, v


def train_steps(ops, e0_u, e0_i, batches, num_layers, order, reg_weight, fair_weight=0.0, pop=None, lr=1e-3):
    """Reference for a run of training steps (CU:608-652 repeated): per (users, pos, neg) batch, loss and gradients
    from `train_step_grads` at the current parameters, then `adam_step_f64` on both tables.  The parameters are
    rounded to float32 after every step, as the stored tables are.  Returns one dict per step: the loss, the
    gradients and the parameters after the step."""
    p = [np.array(e0_u, F32), np.array(e0_i, F32)]
    mv = [[np.zeros(x.shape), np.zeros(x.shape)] for x in p]
    out = []
    for t, (users, pos, neg) in enumerate(batches, start=1):
        loss, g_u, g_i, _, _ = train_step_grads(ops, p[0], p[1], users, pos, neg, num_layers, order, reg_weight,
                                                fair_weight, pop)
        for k, g in enumerate((g_u, g_i)):
            q, mv[k][0], mv[k][1] = adam_step_f64(p[k], g, mv[k][0], mv[k][1], t, lr)
            p[k] = q.astype(F32)
        out.append(dict(loss=loss, g_u=g_u, g_i=g_i, p_u=p[0].copy(), p_i=p[1].copy()))
    return out


# --------------------------------------------------------------------------------------
# a12 / a13 / a14. samplers (sequential, NumPy Generator -- same draw order as the reference)
# --------------------------------------------------------------------------------------
def popularity_law(deg_i: np.ndarray, gamma: float) -> np.ndarray:
    """V2:805-810: p_i = (deg_i + 1)^gamma / (sum + 1e-12), float64."""
    w = np.power(deg_i.astype(np.float64) + 1.0, gamma)
    return (w / (w.sum() + 1e-12)).astype(np.float64)


def draw_positive(indptr, indices, user, rng):
    lo, hi = indptr[user], indptr[user + 1]                    # CU:288-292
    if lo == hi:
        return None
    return int(indices[rng.integers(lo, hi)])


def draw_negative_uniform(indptr, indices, user, num_items, rng):
    while True:                                                # CU:295-299
        j = int(rng.integers(0, num_items))
        if not row_contains(indptr, indices, user, j):
            return j


def draw_negative_popmix(indptr, indices, user, num_items, rng, pop_prob, mix_pop, max_tries):
    for _ in range(max_tries):                                 # V2:364-371
        if rng.random() < mix_pop:
            j = int(rng.choice(num_items, p=pop_prob))
        else:
            j = int(rng.integers(0, num_items))
        if not row_contains(indptr, indices, user, j):
            return j
    return draw_negative_uniform(indptr, indices, user, num_items, rng)   # V2:373-376


def sample_batch(indptr, indices, batch_users, num_items, rng, pop_prob=None, mix_pop=0.7, max_tries=50):
    """One (user, pos, neg) triple per batch user with >=1 train item (CU:615-622, V2:835-849)."""
    us, ps, ns = [], [], []
    for u in batch_users:
        p = draw_positive(indptr, indices, int(u), rng)
        if p is None:
            continue
        if pop_prob is None:
            n = draw_negative_uniform(indptr, indices, int(u), num_items, rng)
        else:
            n = draw_negative_popmix(indptr, indices, int(u), num_items, rng, pop_prob, mix_pop, max_tries)
        us.append(int(u)); ps.append(p); ns.append(n)
    return np.asarray(us, np.int64), np.asarray(ps, np.int64), np.asarray(ns, np.int64)


def negative_law_for_user(num_items, train_row, pop_prob=None, mix_pop=0.7):
    """Exact distribution of an accepted negative when max_tries is not hit: the proposal
    mix*pop + (1-mix)*uniform restricted to items outside the user's train row, renormalised."""
    q = np.full(num_items, 1.0 / num_items)
    if pop_prob is not None:
        q = mix_pop * pop_prob + (1.0 - mix_pop) * q
    q = q.copy()
    q[np.unique(train_row)] = 0.0
    return q / q.sum()


# --------------------------------------------------------------------------------------
# a15 / a16. evaluation
# --------------------------------------------------------------------------------------
def metrics_at_k(ranked, gt_set, K):
    """precision = hits/K, recall = hits/max(|gt|,1), ndcg with 1/log2(rank+2) gains and
    idcg over min(|gt|, K)  (CU:469-484, V2:514-530)."""
    hits = [1 if int(x) in gt_set else 0 for x in ranked[:K]]
    h = sum(hits)
    dcg = sum(1.0 / math.log2(r + 2) for r, f in enumerate(hits) if f)
    idcg = sum(1.0 / math.log2(r + 2) for r in range(min(len(gt_set), K)))
    return h / K, h / max(len(gt_set), 1), (dcg / idcg if idcg > 0 else 0.0)


def novelty(item_ids, pop, total_train, num_items):
    """V2:390-404: mean log(pop+1) and mean -log2((pop+1)/(total+I))."""
    item_ids = np.asarray(item_ids, np.int64)
    if item_ids.size == 0:
        return 0.0, 0.0
    p = pop[item_ids].astype(np.float64)
    return float(np.log(p + 1.0).mean()), float((-np.log2((p + 1.0) / (total_train + num_items))).mean())


def cred_groups(users, cred, pct):
    """V2:407-423 (np.argsort default order; only meaningful when cred values are distinct)."""
    if users.size == 0:
        return np.empty(0, np.int64), np.empty(0, np.int64)
    k = max(int(round(users.size * pct)), 1)
    order = np.argsort(cred[users])
    return users[order[-k:]].astype(np.int64), users[order[:k]].astype(np.int64)


def full_rank_topk(f_u, f_i, users, train_csr, K):
    """Per user: fp32 scores against every item, train items -> -1e9, best K by
    (score desc, item id asc)  (V2:696-704; the reference's argsort leaves ties unordered --
    the id rule is the contract BASELINE.json states)."""
    indptr, indices = train_csr
    ids = np.empty((len(users), K), np.int64)
    sc = np.empty((len(users), K), F32)
    item_ids = np.arange(f_i.shape[0])
    for r, u in enumerate(users):
        s = (f_u[int(u)][None, :].astype(F32) * f_i.astype(F32)).sum(1, dtype=F32)
        s[indices[indptr[u]:indptr[u + 1]]] = F32(-1e9)
        top = np.lexsort((item_ids, -s))[:K]
        ids[r], sc[r] = top, s[top]
    return ids, sc


def evaluate_full_ranking(f_u, f_i, train_csr, test_csr, num_items, Ks=(10, 20), item_pop=None,
                          total_train=0, cred=None, group_pct=0.20):
    """V2:653-752 (extra keys only when item_pop / cred are given; MSG:535-585 is the short form)."""
    ind_te, idx_te = test_csr
    users = np.flatnonzero(np.diff(ind_te) > 0).astype(np.int64)
    if users.size == 0:
        raise RuntimeError("No users with test interactions.")
    ids, _ = full_rank_topk(f_u, f_i, users, train_csr, max(Ks))
    return metrics_from_topk(ids, users, test_csr, num_items, Ks, item_pop, total_train, cred, group_pct,
                             mode="full")


def metrics_from_topk(ids, users, test_csr, num_items, Ks, item_pop=None, total_train=0, cred=None,
                      group_pct=0.20, mode="full", gt_override=None):
    ind_te, idx_te = test_csr
    extra = item_pop is not None and cred is not None
    hi, lo = (cred_groups(users, cred, group_pct) if extra else (np.empty(0), np.empty(0)))
    hi, lo = set(map(int, hi)), set(map(int, lo))
    out = {}
    for K in Ks:
        sp_, sr, sn, slp, ssi = 0.0, 0.0, 0.0, 0.0, 0.0
        cover = set()
        gh = gl = 0.0
        nh = nl = 0
        for r, u in enumerate(users):
            gt = gt_override[r] if gt_override is not None else set(map(int, idx_te[ind_te[u]:ind_te[u + 1]]))
            p, rc, nd = metrics_at_k(ids[r], gt, K)
            sp_ += p; sr += rc; sn += nd
            if extra:
                top = ids[r][:K]
                cover.update(map(int, top))
                a, b = novelty(top, item_pop, total_train, num_items)
                slp += a; ssi += b
                if int(u) in hi:
                    gh += rc; nh += 1
                if int(u) in lo:
                    gl += rc; nl += 1
        n = len(users)
        res = {"precision": sp_ / n, "recall": sr / n, "ndcg": sn / n, "users_eval": n, "mode": mode}
        if extra:
            res.update({
                "item_coverage": len(cover) / max(num_items, 1),
                "avg_log_popularity": slp / n, "avg_self_information": ssi / n,
                "cred_utility": float(sum(float(cred[int(u)]) for u in users) / n),
                "high_cred_recall": gh / max(nh, 1), "low_cred_recall": gl / max(nl, 1),
                "high_users": nh, "low_users": nl,
            })
        out[K] = res
    return out


def sampled_candidates(train_csr, test_csr, num_items, n_neg, seed):
    """Candidate lists of the sampled protocol: 1 test positive + n_neg negatives outside
    test ∪ train, default_rng(seed + 999) (CU:496-521, V2:554-591)."""
    ind_tr, idx_tr = train_csr
    ind_te, idx_te = test_csr
    rng = np.random.default_rng(seed + 999)
    users = np.flatnonzero(np.diff(ind_te) > 0).astype(np.int64)
    cands = np.empty((users.size, 1 + n_neg), np.int64)
    for r, u in enumerate(users):
        gt = idx_te[ind_te[u]:ind_te[u + 1]]
        gts = set(map(int, gt))
        cands[r, 0] = int(gt[rng.integers(0, len(gt))])
        k = 1
        while k <= n_neg:
            j = int(rng.integers(0, num_items))
            if j in gts or row_contains(ind_tr, idx_tr, int(u), j):
                continue
            cands[r, k] = j
            k += 1
    return users, cands


def rank_candidates(f_u, f_i, users, cands):
    """Scores of each user's candidates, ranked by np.argsort(-scores) (CU:523-527)."""
    ranked = np.empty_like(cands)
    for r, u in enumerate(users):
        s = (f_u[int(u)][None, :] * f_i[cands[r]]).sum(1, dtype=F32)
        ranked[r] = cands[r][np.argsort(-s, kind="stable")]
    return ranked


# --------------------------------------------------------------------------------------
# timed CPU baseline: the reference's own execution strategy (COO torch.sparse.mm + autograd)
# --------------------------------------------------------------------------------------
class TorchCpuBaseline:
    """Port of the reference's CPU path for timing: coalesced COO operators, K layers of
    torch.sparse.mm (CU:429-437 / V2:482-486), stack+mean, BPR+L2, autograd backward, Adam."""

    def __init__(self, ops: Operators, e0_u, e0_i, num_layers, order, lr=1e-3, device="cpu"):
        """device="cuda": the same script-level code on the GPU, i.e. stock ATen / cuSPARSE kernels -- the
        reference's own GPU path (its scripts run with cfg.device = "cuda" when a GPU is present)."""
        import torch
        self.torch = torch
        self.K, self.order = num_layers, order
        self.device = torch.device(device)
        mk = lambda r, c, v, shape: torch.sparse_coo_tensor(
            torch.from_numpy(np.vstack([r, c])), torch.from_numpy(v), size=shape).coalesce().to(self.device)
        self.A = mk(ops.A_row, ops.A_col, ops.A_val, (ops.U, ops.I))
        self.C = mk(ops.C_row, ops.C_col, ops.C_val, (ops.I, ops.U))
        self.eu = torch.nn.Parameter(torch.from_numpy(np.array(e0_u, dtype=F32)).to(self.device))
        self.ei = torch.nn.Parameter(torch.from_numpy(np.array(e0_i, dtype=F32)).to(self.device))
        self.opt = torch.optim.Adam([self.eu, self.ei], lr=lr)

    def forward(self):
        torch = self.torch
        u, i = self.eu, self.ei
        us, is_ = [u], [i]
        for _ in range(self.K):
            i_new = torch.sparse.mm(self.C, u)
            u_new = torch.sparse.mm(self.A, i if self.order == "jacobi" else i_new)
            u, i = u_new, i_new
            us.append(u); is_.append(i)
        return torch.stack(us, 0).mean(0), torch.stack(is_, 0).mean(0)

    def loss(self, fu, fi, users, pos, neg, reg, fair=0.0, pop=None):
        torch = self.torch
        u, p, n = fu[users], fi[pos], fi[neg]
        yp, yn = (u * p).sum(1), (u * n).sum(1)
        out = -torch.log(torch.sigmoid(yp - yn) + 1e-12).mean()
        if fair and pop is not None:
            out = out + fair * (pop[pos] * yp).mean()
        r = (self.eu[users].norm(2, dim=1).pow(2) + self.ei[pos].norm(2, dim=1).pow(2)
             + self.ei[neg].norm(2, dim=1).pow(2)).mean()
        return out + reg * r

    def step(self, users, pos, neg, reg, fair=0.0, pop=None, optimize=True):
        torch = self.torch
        users, pos, neg = (torch.as_tensor(x, dtype=torch.long).to(self.device) for x in (users, pos, neg))
        fu, fi = self.forward()
        loss = self.loss(fu, fi, users, pos, neg, reg, fair, pop)
        self.opt.zero_grad()
        loss.backward()
        if optimize:
            self.opt.step()
        return float(loss.item())
