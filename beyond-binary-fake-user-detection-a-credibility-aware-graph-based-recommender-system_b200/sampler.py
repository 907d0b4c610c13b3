"""Triple samplers.  Reference names kept for the scalar helpers; the batch path runs on device.

    user_has_item / sample_pos_item / sample_neg_item      lightgcn_cu.py:279-299
    sample_neg_item_popmix + popularity law                 Version-2/lighgcn_cu_pop.py:349-376, 805-810

The reference draws from one sequential PCG64 stream inside a per-user Python loop; that stream is
not reproducible on a GPU, so parity is defined as (a) identical model/loss results under an
injected triple list and (b) the sampled negatives following the same law (tests check both).
"""
from __future__ import annotations

import numpy as np
import torch

from ._lib import check, lib, ptr, stream_ptr, workspace
from .graph import CredGraph


# ---- scalar helpers with the reference's signatures (host, NumPy) -- for scripts that call them
def user_has_item(indptr, indices, user: int, item: int) -> bool:
    lo, hi = int(indptr[user]), int(indptr[user + 1])
    if lo == hi:
        return False
    j = lo + int(np.searchsorted(indices[lo:hi], item))
    return j < hi and int(indices[j]) == item


def sample_pos_item(indptr, indices, user: int, rng: np.random.Generator):
    lo, hi = indptr[user], indptr[user + 1]
    if lo == hi:
        return None
    return int(indices[rng.integers(lo, hi)])


def sample_neg_item(indptr, indices, user: int, num_items: int, rng: np.random.Generator):
    while True:
        j = int(rng.integers(0, num_items))
        if not user_has_item(indptr, indices, user, j):
            return j


def sample_neg_item_popmix(indptr, indices, user: int, num_items: int, rng: np.random.Generator,
                           pop_prob: np.ndarray, mix_pop: float, max_tries: int):
    for _ in range(max_tries):
        j = int(rng.choice(num_items, p=pop_prob)) if rng.random() < mix_pop else int(rng.integers(0, num_items))
        if not user_has_item(indptr, indices, user, j):
            return j
    return sample_neg_item(indptr, indices, user, num_items, rng)


def popularity_probabilities(item_deg: np.ndarray, gamma: float) -> np.ndarray:
    """pop_prob of lighgcn_cu_pop.py:805-810 (float64)."""
    w = np.power(np.asarray(item_deg, dtype=np.float64) + 1.0, gamma)
    return (w / (w.sum() + 1e-12)).astype(np.float64)


# ---- device sampler -------------------------------------------------------------------------
class TripleSampler:
    """(user, pos, neg) for a batch of users in one kernel.  mix_pop=None -> uniform negatives
    (lightgcn_cu.py), otherwise the Method-E mixture with exponent `gamma` on (deg_i + 1)."""

    def __init__(self, graph: CredGraph, mix_pop: float | None = None, gamma: float = 0.75, max_tries: int = 50,
                 seed: int = 42):
        self.graph, self.mix_pop, self.gamma, self.max_tries, self.seed = graph, mix_pop, gamma, int(max_tries), seed
        self.calls = 0
        dev, I = graph.device, graph.num_items
        self.tables = None
        if mix_pop is not None:
            i32 = dict(dtype=torch.int32, device=dev)
            self.items_by_deg = torch.empty(I, **i32)
            self.class_start = torch.empty(I + 1, **i32)
            self.class_prob = torch.empty(I, dtype=torch.float32, device=dev)
            self.class_alias = torch.empty(I, **i32)
            self.n_classes = torch.zeros(1, **i32)
            ws = workspace(lib().cgx_sampler_build_workspace_bytes(I), dev)
            with torch.cuda.device(dev):
                check(lib().cgx_sampler_build(ptr(graph.deg_i), I, float(gamma), ptr(self.items_by_deg),
                                              ptr(self.class_start), ptr(self.class_prob), ptr(self.class_alias),
                                              ptr(self.n_classes), ptr(ws), ws.numel(), stream_ptr(dev)))
            self.tables = (self.items_by_deg, self.class_start, self.class_prob, self.class_alias, self.n_classes)

    def sample(self, users: torch.Tensor, offset: int | None = None, offset_dev: torch.Tensor | None = None,
               slots: torch.Tensor | None = None, count: torch.Tensor | None = None, out=None):
        """users: int64 CUDA tensor of batch users, each with >= 1 train item.  Returns (pos, neg).
        offset_dev: int64[1] device counter added to the offset (CUDA-graph replay).
        slots: int64[B] device tensor -- entry k draws the triple of global batch slot slots[k] (a sharded rank's part
        of a batch draws what the whole-batch call draws for those users); count: int64[1] device tensor -- entries at
        or past it are absent and their outputs are left untouched; out: (pos, neg) buffers to write."""
        g, dev = self.graph, self.graph.device
        users = torch.as_tensor(users, device=dev).to(torch.int64).contiguous()
        B = users.numel()
        pos, neg = out if out is not None else (torch.empty(B, dtype=torch.int64, device=dev),
                                                torch.empty(B, dtype=torch.int64, device=dev))
        if offset is None:
            offset = self.calls
        self.calls += 1
        t = self.tables or (None,) * 5
        with torch.cuda.device(dev):
            check(lib().cgx_sample_triples(ptr(users), B, ptr(g.samp_indptr), ptr(g.samp_idx), g.num_items,
                                           ptr(t[0]), ptr(t[1]), ptr(t[2]), ptr(t[3]), ptr(t[4]),
                                           -1.0 if self.mix_pop is None else float(self.mix_pop), self.max_tries,
                                           int(self.seed) & 0xFFFFFFFFFFFFFFFF, int(offset), ptr(offset_dev),
                                           ptr(pos), ptr(neg), stream_ptr(dev), ptr(slots), ptr(count)))
        return pos, neg
