"""Seeded synthetic bipartite interaction graphs with injected fake-user blocks.

The reference ships no data (its dataset directory is git-ignored), so every parity
test and every bench line runs on graphs made here.  Shapes follow BASELINE.json's
configs (SURVEY.md section 8d):

    C1  943 x 1,682 x 100k        (ML-100K-shaped,  lightgcn_cu.py,          d=64  K=3)
    C2  31,668 x 38,048 x 1.56M   (Yelp2018-shaped, Version-2/lighgcn_cu_pop, d=64  K=3)
    C3  52,643 x 91,599 x 2.98M   (Amazon-Book-shaped, degree-aware variant,  d=64  K=4)
    C4  10M x 2M x 200M           (power law, d=128 K=3)
    C5  50M x 10M x 1B            (power law, d=64  K=3)

Law: item popularity p_i ~ rank^-0.8, user activity log-normal, unique (u, i) pairs,
a fake-user population (5 % of users, in clusters) whose edges concentrate on a
small target set of items, credibility Beta(5,2) for genuine and Beta(1,8) for fake
users with exact 0.0 / 1.0 values present, 80/10/10 split by a seeded permutation.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

SHAPES = {
    "C1": dict(num_users=943, num_items=1_682, num_edges=100_000, emb_dim=64, num_layers=3,
               variant="cu", order="jacobi", cluster=0),
    "C2": dict(num_users=31_668, num_items=38_048, num_edges=1_560_000, emb_dim=64, num_layers=3,
               variant="v2", order="gs", cluster=0),
    "C3": dict(num_users=52_643, num_items=91_599, num_edges=2_980_000, emb_dim=64, num_layers=4,
               variant="da", order="gs", cluster=0),
    "C4": dict(num_users=10_000_000, num_items=2_000_000, num_edges=200_000_000, emb_dim=128,
               num_layers=3, variant="v2", order="gs", cluster=1000),
    "C5": dict(num_users=50_000_000, num_items=10_000_000, num_edges=1_000_000_000, emb_dim=64,
               num_layers=3, variant="v2", order="gs", cluster=1000),
}
_CFG_ID = {"C1": 1, "C2": 2, "C3": 3, "C4": 4, "C5": 5}


@dataclass
class SynthGraph:
    name: str
    num_users: int
    num_items: int
    train_edges: np.ndarray          # int32 [2, E_train]
    val_edges: np.ndarray            # int32 [2, E_val]
    test_edges: np.ndarray           # int32 [2, E_test]
    cred: np.ndarray                 # float32 [U] in [0, 1]
    is_fake: np.ndarray              # bool [U]
    meta: dict = field(default_factory=dict)

    @property
    def all_edges(self) -> np.ndarray:
        return np.concatenate([self.train_edges, self.val_edges, self.test_edges], axis=1)


def _zipf_cdf(num_items: int, exponent: float, rng: np.random.Generator) -> tuple[np.ndarray, np.ndarray]:
    """CDF over items whose ids are a random permutation of the popularity ranks."""
    ranks = np.arange(1, num_items + 1, dtype=np.float64)
    p = ranks ** (-exponent)
    p /= p.sum()
    perm = rng.permutation(num_items)            # rank r -> item id perm[r]
    return np.cumsum(p), perm


def _user_counts(num_users: int, total: int, rng: np.random.Generator, sigma: float = 1.0) -> np.ndarray:
    a = rng.lognormal(mean=0.0, sigma=sigma, size=num_users)
    c = np.maximum(np.floor(a * (total / a.sum())).astype(np.int64), 1)
    return c


def make_graph(
    name: str = "C1",
    *,
    num_users: int | None = None,
    num_items: int | None = None,
    num_edges: int | None = None,
    seed: int | None = None,
    fake_frac: float = 0.05,
    cluster: int | None = None,
    duplicate_edges: int = 0,
    split=(0.8, 0.1, 0.1),
    item_seed: int | None = None,
) -> SynthGraph:
    """Build one synthetic graph.  `name` picks a BASELINE shape; explicit sizes override it.

    duplicate_edges > 0 appends that many repeated (u, i) pairs to the train split
    (legal in the reference: SURVEY.md appendix B-1) -- correctness tests only.
    """
    shp = dict(SHAPES.get(name, SHAPES["C1"]))
    U = int(num_users if num_users is not None else shp["num_users"])
    I = int(num_items if num_items is not None else shp["num_items"])
    E = int(num_edges if num_edges is not None else shp["num_edges"])
    E = min(E, (U * I) // 2)
    cl = int(cluster if cluster is not None else shp["cluster"])
    rng = np.random.default_rng(20240 + _CFG_ID.get(name, 9) if seed is None else seed)

    n_fake = int(round(U * fake_frac))
    n_gen = U - n_fake
    is_fake = np.zeros(U, dtype=bool)
    if n_fake:
        if cl <= 0:                               # one contiguous block at the top of the id range
            is_fake[n_gen:] = True
        else:                                     # clusters of `cl` consecutive ids spread over the range
            n_cl = max(n_fake // cl, 1)
            starts = np.sort(rng.choice(max(U // cl, 1), size=min(n_cl, max(U // cl, 1)), replace=False)) * cl
            for s in starts:
                is_fake[s:s + cl] = True
    fake_ids = np.flatnonzero(is_fake)
    gen_ids = np.flatnonzero(~is_fake)

    E_fake = int(E * fake_frac) if fake_ids.size else 0
    E_gen = E - E_fake

    # genuine edges: log-normal activity x Zipf item choice, de-duplicated
    # item_seed fixes the popularity ranking independently of `seed` (user shards of one catalogue)
    cdf, perm = _zipf_cdf(I, 0.8, rng if item_seed is None else np.random.default_rng(item_seed))
    keys = np.empty(0, dtype=np.int64)
    want = E_gen
    for _ in range(8):
        need = want - keys.size
        if need <= 0:
            break
        cnt = _user_counts(gen_ids.size, int(need * 1.25) + 16, rng)
        uu = np.repeat(gen_ids, cnt)
        ii = perm[np.minimum(np.searchsorted(cdf, rng.random(uu.size)), I - 1)]
        keys = np.unique(np.concatenate([keys, uu.astype(np.int64) * I + ii]))
    if keys.size > want:
        keys = keys[np.sort(rng.choice(keys.size, size=want, replace=False))]

    # fake edges: every cluster hammers its own small target set
    fkeys = np.empty(0, dtype=np.int64)
    if fake_ids.size:
        group = cl if cl > 0 else fake_ids.size
        per_user = max(E_fake // fake_ids.size, 1)
        parts = []
        for g0 in range(0, fake_ids.size, group):
            members = fake_ids[g0:g0 + group]
            t = int(np.clip(rng.integers(50, 501), per_user + 1, max(I - 1, per_user + 1)))
            t = min(t, I)
            targets = rng.choice(I, size=t, replace=False)
            k = min(per_user, t)
            # each member takes k distinct targets: argpartition of random scores
            pick = np.argpartition(rng.random((members.size, t)), k - 1, axis=1)[:, :k]
            parts.append((np.repeat(members, k).astype(np.int64) * I + targets[pick].ravel()))
        fkeys = np.unique(np.concatenate(parts))
        fkeys = np.setdiff1d(fkeys, keys, assume_unique=True)

    all_keys = np.concatenate([keys, fkeys])
    all_keys = all_keys[rng.permutation(all_keys.size)]
    u = (all_keys // I).astype(np.int32)
    i = (all_keys % I).astype(np.int32)
    edges = np.stack([u, i])

    n = edges.shape[1]
    n_tr = int(n * split[0])
    n_va = int(n * split[1])
    train, val, test = edges[:, :n_tr], edges[:, n_tr:n_tr + n_va], edges[:, n_tr + n_va:]
    if duplicate_edges:
        sel = rng.integers(0, train.shape[1], size=duplicate_edges)
        train = np.concatenate([train, train[:, sel]], axis=1)
        train = train[:, rng.permutation(train.shape[1])]

    cred = rng.beta(5.0, 2.0, size=U)
    if fake_ids.size:
        cred[fake_ids] = rng.beta(1.0, 8.0, size=fake_ids.size)
    cred = np.clip(cred, 0.0, 1.0).astype(np.float32)
    if U >= 4:                                    # exact end points must be exercised
        cred[gen_ids[0]] = 1.0
        cred[(fake_ids if fake_ids.size else gen_ids)[-1]] = 0.0

    return SynthGraph(
        name=name, num_users=U, num_items=I,
        train_edges=np.ascontiguousarray(train), val_edges=np.ascontiguousarray(val),
        test_edges=np.ascontiguousarray(test), cred=cred, is_fake=is_fake,
        meta=dict(shp, num_users=U, num_items=I, num_edges=int(n), fake_users=int(n_fake)),
    )


def make_graph_device(name: str = "C4", device="cuda", *, num_users=None, num_items=None, num_edges=None,
                      seed: int | None = None, fake_frac: float = 0.05, split=(0.8, 0.1, 0.1),
                      item_seed: int | None = None) -> SynthGraph:
    """Same law as make_graph, generated with torch on `device` for the shapes NumPy is too slow for
    (C4: 200M edges, C5: 1B edges).  Edge count is approximate (+-1 %): de-duplication is done by one
    sort instead of top-up rounds.  Edge arrays stay on the device (SynthGraph fields hold tensors)."""
    import torch
    shp = dict(SHAPES.get(name, SHAPES["C4"]))
    U = int(num_users if num_users is not None else shp["num_users"])
    I = int(num_items if num_items is not None else shp["num_items"])
    E = int(num_edges if num_edges is not None else shp["num_edges"])
    cl = int(shp["cluster"]) or 1000
    dev = torch.device(device)
    gen = torch.Generator(device=dev).manual_seed(20240 + _CFG_ID.get(name, 9) if seed is None else seed)
    rnd = lambda n: torch.rand(n, device=dev, generator=gen)

    # fake clusters: `cl` consecutive ids each, spread over the id range
    n_cl = max(int(round(U * fake_frac)) // cl, 1)
    starts = torch.randperm(max(U // cl, 1), device=dev, generator=gen)[:n_cl] * cl
    is_fake = torch.zeros(U, dtype=torch.bool, device=dev)
    fake_ids = (starts[:, None] + torch.arange(cl, device=dev)[None, :]).reshape(-1)
    fake_ids = fake_ids[fake_ids < U]
    is_fake[fake_ids] = True
    n_fake = int(fake_ids.numel())
    E_fake = int(E * fake_frac)
    E_gen = E - E_fake

    # genuine edges: log-normal activity x Zipf(0.8) items
    ranks = torch.arange(1, I + 1, device=dev, dtype=torch.float64)
    cdf = torch.cumsum(ranks.pow(-0.8), 0)
    cdf = (cdf / cdf[-1]).to(torch.float32)
    if item_seed is None:
        perm = torch.randperm(I, device=dev, generator=gen)
    else:       # popularity ranking fixed independently of `seed`: user shards of one catalogue
        perm = torch.randperm(I, device=dev, generator=torch.Generator(device=dev).manual_seed(item_seed))
    act = torch.exp(torch.randn(U, device=dev, generator=gen))
    act[is_fake] = 0.0
    cnt = torch.floor(act * (E_gen * 1.12 / act.sum())).to(torch.int64)
    cnt[~is_fake] = cnt[~is_fake].clamp(min=1)
    uu = torch.repeat_interleave(torch.arange(U, device=dev), cnt)
    del act, cnt
    ii = perm[torch.searchsorted(cdf, rnd(uu.numel())).clamp(max=I - 1)]
    keys = torch.unique(uu * I + ii)
    del uu, ii
    if keys.numel() > E_gen:
        keys = keys[rnd(keys.numel()) < (E_gen / keys.numel())]

    # fake edges: each cluster hammers its own 50..500 target items
    per_user = max(E_fake // max(n_fake, 1), 1)
    t_c = torch.randint(50, 501, (n_cl,), device=dev, generator=gen)
    targets = torch.randint(0, I, (n_cl, 500), device=dev, generator=gen)
    fu = torch.repeat_interleave(fake_ids, per_user)
    fc = torch.repeat_interleave(torch.arange(n_cl, device=dev).repeat_interleave(cl)[: fake_ids.numel()], per_user)
    fj = (rnd(fu.numel()) * t_c[fc]).to(torch.int64)
    fkeys = torch.unique(fu * I + targets[fc, fj])
    del fu, fc, fj

    all_keys = torch.cat([keys, fkeys])
    del keys, fkeys
    all_keys = all_keys[torch.randperm(all_keys.numel(), device=dev, generator=gen)]
    edges = torch.stack([(all_keys // I).to(torch.int32), (all_keys % I).to(torch.int32)])
    del all_keys
    n = edges.shape[1]
    n_tr, n_va = int(n * split[0]), int(n * split[1])

    g1 = torch._standard_gamma(torch.where(is_fake, 1.0, 5.0).to(torch.float32), generator=gen)
    g2 = torch._standard_gamma(torch.where(is_fake, 8.0, 2.0).to(torch.float32), generator=gen)
    cred = (g1 / (g1 + g2)).clamp(0.0, 1.0).to(torch.float32)
    cred[0], cred[-1] = 1.0, 0.0
    return SynthGraph(name=name, num_users=U, num_items=I, train_edges=edges[:, :n_tr].contiguous(),
                      val_edges=edges[:, n_tr:n_tr + n_va].contiguous(), test_edges=edges[:, n_tr + n_va:].contiguous(),
                      cred=cred, is_fake=is_fake,
                      meta=dict(shp, num_users=U, num_items=I, num_edges=int(n), fake_users=n_fake, on_device=True))


def make_triples(graph: SynthGraph, batch: int, seed: int = 7):
    """An injected (user, pos, neg) list: users with >=1 train edge, pos from their row,
    neg uniform outside the row.  Used wherever parity needs identical triples on both sides."""
    rng = np.random.default_rng(seed)
    u, i = graph.train_edges[0].astype(np.int64), graph.train_edges[1].astype(np.int64)
    sel = rng.integers(0, u.size, size=batch)
    users, pos = u[sel], i[sel]
    have = set((u * graph.num_items + i).tolist()) if u.size < 5_000_000 else None
    neg = rng.integers(0, graph.num_items, size=batch)
    if have is not None:
        for k in range(batch):
            while int(users[k]) * graph.num_items + int(neg[k]) in have:
                neg[k] = rng.integers(0, graph.num_items)
    return users.astype(np.int64), pos.astype(np.int64), neg.astype(np.int64)
