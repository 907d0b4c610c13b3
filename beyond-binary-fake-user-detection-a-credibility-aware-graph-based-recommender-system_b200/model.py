"""Model classes with the reference's names and methods over the fused device kernels.

    CredLightGCN   lightgcn_cu.py:405-463            Jacobi layer order, loss assembled by the caller
    LightGCN       Version-2/lighgcn_cu_pop.py:458-508 Gauss-Seidel layer order, bpr_loss method
                   (also version_1/lightgcn_cu_message.py:408-430 and the degree-aware script)

state_dict keys are exactly `user_emb.weight`, `item_emb.weight` (the operators are plain
attributes, lightgcn_cu.py:411-412), so checkpoints interchange with the reference classes.
Initialisation stays torch (xavier_uniform_ on user_emb then item_emb) so seeds reproduce.
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import check, lib, ptr, stream_ptr, workspace
from .graph import CredGraph, graph_of


def _f32c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        raise _lib.CgxError(f"credgcn kernels are fp32, got {t.dtype}")
    return t.contiguous()


def _i64c(t, device) -> torch.Tensor:
    return torch.as_tensor(t, device=device).to(torch.int64).contiguous()


# ------------------------------------------------------------------------------------------
# raw ops (no autograd)
# ------------------------------------------------------------------------------------------
def propagate_forward(graph: CredGraph, e0_u, e0_i, num_layers: int, order: str):
    e0_u, e0_i = _f32c(e0_u), _f32c(e0_i)
    d = e0_u.shape[1]
    out_u, out_i = torch.empty_like(e0_u), torch.empty_like(e0_i)
    ws = graph.propagate_workspace(d, order)
    with torch.cuda.device(graph.device):
        check(lib().cgx_propagate_fwd(graph.by_user.ref(), graph.by_item.ref(), _lib.ORDERS[order], num_layers, d,
                                      ptr(e0_u), ptr(e0_i), ptr(out_u), ptr(out_i), ptr(ws), ws.numel(),
                                      stream_ptr(graph.device)))
    return out_u, out_i


def propagate_backward(graph: CredGraph, g_u, g_i, num_layers: int, order: str):
    g_u, g_i = _f32c(g_u), _f32c(g_i)
    d = g_u.shape[1]
    d_u, d_i = torch.empty_like(g_u), torch.empty_like(g_i)
    ws = graph.propagate_workspace(d, order)
    with torch.cuda.device(graph.device):
        check(lib().cgx_propagate_bwd(graph.by_user.ref(), graph.by_item.ref(), _lib.ORDERS[order], num_layers, d,
                                      ptr(g_u), ptr(g_i), ptr(d_u), ptr(d_i), ptr(ws), ws.numel(),
                                      stream_ptr(graph.device)))
    return d_u, d_i


def spmm(csr, x, use_bwd_values=False):
    """y = M @ x for one row order of the graph (one layer of the reference's torch.sparse.mm)."""
    x = _f32c(x)
    d = x.shape[1]
    y = torch.empty(csr.n_rows, d, dtype=torch.float32, device=x.device)
    ws = workspace(lib().cgx_spmm_workspace_bytes(csr.ref(), d), x.device)
    with torch.cuda.device(x.device):
        check(lib().cgx_spmm(csr.ref(), int(use_bwd_values), d, ptr(x), ptr(y), None, None, 1.0, ptr(ws),
                             ws.numel(), stream_ptr(x.device)))
    return y


def row_flags(x):
    """uint8[n_rows]: 1 where the row of x has a non-zero entry (cgx_row_flags)."""
    x = _f32c(x)
    flags = torch.empty(x.shape[0], dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        check(lib().cgx_row_flags(ptr(x), x.shape[0], x.shape[1], ptr(flags), stream_ptr(x.device)))
    return flags


def spmm_sparse_rows(csr, x, flags=None, use_bwd_values=False):
    """spmm() for an x whose rows are mostly zero: rows with flags == 0 are not gathered (same result)."""
    x = _f32c(x)
    flags = row_flags(x) if flags is None else flags
    d = x.shape[1]
    y = torch.empty(csr.n_rows, d, dtype=torch.float32, device=x.device)
    ws = workspace(lib().cgx_spmm_workspace_bytes(csr.ref(), d), x.device)
    with torch.cuda.device(x.device):
        check(lib().cgx_spmm_sparse_rows(csr.ref(), int(use_bwd_values), d, ptr(x), ptr(flags), ptr(y), None, None,
                                         1.0, ptr(ws), ws.numel(), stream_ptr(x.device)))
    return y


def bpr_plan(graph: CredGraph, users, pos, neg, plan=None):
    """Sorted (row, entry) keys of a triple batch: the scatter plan of the fused loss (indices only)."""
    dev = graph.device
    users, pos, neg = _i64c(users, dev), _i64c(pos, dev), _i64c(neg, dev)
    B = users.numel()
    if plan is None:
        plan = torch.empty(3 * B, dtype=torch.int64, device=dev)      # uint64 keys, stored as int64 bits
    ws = workspace(lib().cgx_bpr_plan_workspace_bytes(B), dev)
    with torch.cuda.device(dev):
        check(lib().cgx_bpr_plan(ptr(users), ptr(pos), ptr(neg), B, graph.num_users, graph.num_items, ptr(plan),
                                 ptr(ws), ws.numel(), stream_ptr(dev)))
    return plan


def batch_frontier(graph: CredGraph, users, pos, neg, flags=None, flags_u=None):
    """uint8[I]: 1 on the items of pos, neg and the train rows of the batch users (cgx_batch_frontier), the only
    rows where the first item-side adjoint of the batch's loss can be non-zero.  flags_u (uint8[U], optional) is
    set to 1 on the batch users."""
    dev = graph.device
    users, pos, neg = _i64c(users, dev), _i64c(pos, dev), _i64c(neg, dev)
    if flags is None:
        flags = torch.empty(graph.num_items, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        check(lib().cgx_batch_frontier(graph.by_user.ref(), ptr(users), ptr(pos), ptr(neg), users.numel(), ptr(flags),
                                       ptr(flags_u), stream_ptr(dev)))
    return flags


def bpr_fused(graph: CredGraph, f_u, f_i, e0_u, e0_i, users, pos, neg, reg_weight, fair_weight=0.0, pop=None,
              g_u=None, g_i=None, plan=None, bufs=None, batch_total=0):
    """Loss value + gradients w.r.t. the propagated tables + compact ego (L2) gradient.
    g_u / g_i, when given, must be zero-filled [U,d] / [I,d] buffers; `plan` = bpr_plan(...) of the
    same batch (built here when absent); `bufs` = reusable (loss, ego_rows, ego_coef, ws)."""
    dev = f_u.device
    f_u, f_i, e0_u, e0_i = _f32c(f_u), _f32c(f_i), _f32c(e0_u), _f32c(e0_i)
    users, pos, neg = _i64c(users, dev), _i64c(pos, dev), _i64c(neg, dev)
    B, d = users.numel(), f_u.shape[1]
    if plan is None:
        plan = bpr_plan(graph, users, pos, neg)
    if g_u is None:
        g_u = torch.zeros_like(f_u)
    if g_i is None:
        g_i = torch.zeros_like(f_i)
    if bufs is None:
        bufs = bpr_buffers(graph, B, dev)
    loss, ego_rows, ego_coef, ws = bufs
    pop_t = None if pop is None else _f32c(torch.as_tensor(pop, device=dev))
    with torch.cuda.device(dev):
        check(lib().cgx_bpr_fwd_bwd(ptr(users), ptr(pos), ptr(neg), B, int(batch_total), ptr(plan), graph.num_users,
                                    graph.num_items,
                                    d, ptr(f_u), ptr(f_i), ptr(e0_u), ptr(e0_i), ptr(pop_t), float(reg_weight),
                                    float(fair_weight), ptr(loss), ptr(g_u), ptr(g_i), ptr(ego_rows),
                                    ptr(ego_coef), ptr(ws), ws.numel(), stream_ptr(dev)))
    return loss, g_u, g_i, ego_rows, ego_coef


def bpr_buffers(graph: CredGraph, B: int, dev):
    return (torch.empty(1, dtype=torch.float32, device=dev), torch.empty(3 * B, dtype=torch.int32, device=dev),
            torch.empty(3 * B, dtype=torch.float32, device=dev),
            workspace(lib().cgx_bpr_workspace_bytes(B, graph.num_users, graph.num_items), dev))


def apply_ego(graph: CredGraph, ego_rows, ego_coef, e0_u, e0_i, d_e0_u, d_e0_i):
    with torch.cuda.device(e0_u.device):
        check(lib().cgx_bpr_apply_ego(ptr(ego_rows), ptr(ego_coef), ego_rows.numel(), graph.num_users,
                                      e0_u.shape[1], ptr(_f32c(e0_u)), ptr(_f32c(e0_i)), ptr(d_e0_u), ptr(d_e0_i),
                                      stream_ptr(e0_u.device)))


# ------------------------------------------------------------------------------------------
# autograd wrappers
# ------------------------------------------------------------------------------------------
class _Propagate(torch.autograd.Function):
    """final = mean_{k=0..K} layer_k, with the adjoint of SURVEY.md appendix C as backward."""

    @staticmethod
    def forward(ctx, e0_u, e0_i, graph, num_layers, order):
        ctx.graph, ctx.num_layers, ctx.order = graph, num_layers, order
        return propagate_forward(graph, e0_u.detach(), e0_i.detach(), num_layers, order)

    @staticmethod
    def backward(ctx, g_u, g_i):
        d_u, d_i = propagate_backward(ctx.graph, g_u, g_i, ctx.num_layers, ctx.order)
        return d_u, d_i, None, None, None


class _SpMM(torch.autograd.Function):
    """One layer product y = M x; backward is the same kernel on the transposed value array."""

    @staticmethod
    def forward(ctx, x, graph, which):
        ctx.graph, ctx.which = graph, which
        return spmm(graph.by_user if which == "A" else graph.by_item, x.detach(), False)

    @staticmethod
    def backward(ctx, gy):
        # (A)^T lives in item-row order, (C)^T in user-row order
        csr = ctx.graph.by_item if ctx.which == "A" else ctx.graph.by_user
        return spmm(csr, gy, True), None, None


class _BprLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, f_u, f_i, e0_u, e0_i, graph, users, pos, neg, reg_weight, fair_weight, pop):
        loss, g_u, g_i, ego_rows, ego_coef = bpr_fused(graph, f_u.detach(), f_i.detach(), e0_u.detach(),
                                                        e0_i.detach(), users, pos, neg, reg_weight, fair_weight, pop)
        ctx.graph = graph
        ctx.save_for_backward(g_u, g_i, ego_rows, ego_coef, e0_u.detach(), e0_i.detach())
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g):
        g_u, g_i, ego_rows, ego_coef, e0_u, e0_i = ctx.saved_tensors
        d_e0_u, d_e0_i = torch.zeros_like(e0_u), torch.zeros_like(e0_i)
        apply_ego(ctx.graph, ego_rows, ego_coef, e0_u, e0_i, d_e0_u, d_e0_i)
        return g_u * g, g_i * g, d_e0_u * g, d_e0_i * g, None, None, None, None, None, None, None


def fused_bpr_loss(graph, f_u, f_i, e0_u, e0_i, users, pos, neg, reg_weight, fair_weight=0.0, pop=None):
    return _BprLoss.apply(f_u, f_i, e0_u, e0_i, graph, users, pos, neg, reg_weight, fair_weight, pop)


# ------------------------------------------------------------------------------------------
# modules
# ------------------------------------------------------------------------------------------
class _Base(torch.nn.Module):
    ORDER = "gs"

    def __init__(self, num_users, num_items, emb_dim, num_layers, M_ui, M_iu):
        super().__init__()
        self.num_users, self.num_items, self.num_layers = num_users, num_items, num_layers
        self.M_ui, self.M_iu = M_ui, M_iu
        self.graph = graph_of(M_ui, M_iu)
        if (self.graph.num_users, self.graph.num_items) != (num_users, num_items):
            raise ValueError("operator shapes do not match num_users / num_items")
        if not lib().cgx_emb_dim_supported(emb_dim):
            raise _lib.CgxError(f"emb_dim={emb_dim} unsupported: use 16, 32, 64, 128 or 256")
        self.user_emb = torch.nn.Embedding(num_users, emb_dim)
        self.item_emb = torch.nn.Embedding(num_items, emb_dim)
        torch.nn.init.xavier_uniform_(self.user_emb.weight)
        torch.nn.init.xavier_uniform_(self.item_emb.weight)

    def ego_tables(self):
        """(user table, item table, user gradient, item gradient) as TrainStep updates them: the storage of the two
        weights, and fresh [U, d] / [I, d] buffers installed as their .grad."""
        eu, ei = self.user_emb.weight, self.item_emb.weight
        eu.grad, ei.grad = torch.empty_like(eu), torch.empty_like(ei)
        return eu.data, ei.data, eu.grad, ei.grad

    def _final(self):
        return _Propagate.apply(self.user_emb.weight, self.item_emb.weight, self.graph, self.num_layers, self.ORDER)

    def _layers(self):
        """Every layer table, one SpMM launch each (the reference's Python loop, kept for API parity)."""
        u, i = self.user_emb.weight, self.item_emb.weight
        us, is_ = [u], [i]
        for _ in range(self.num_layers):
            i_new = _SpMM.apply(u, self.graph, "C")
            u_new = _SpMM.apply(i if self.ORDER == "jacobi" else i_new, self.graph, "A")
            u, i = u_new, i_new
            us.append(u)
            is_.append(i)
        return us, is_


class CredLightGCN(_Base):
    """lightgcn_cu.py:405.  M_ui = [I x U] credibility operator, M_iu = [U x I] base operator."""
    ORDER = "jacobi"

    def propagate_all_layers(self):
        return self._layers()

    def final_embeddings(self):
        return self._final()

    def score(self, users, items, e_u, e_i):
        return (e_u[users] * e_i[items]).sum(dim=1)

    def l2_reg(self, users, pos_items, neg_items):
        eu, ep, en = self.user_emb.weight[users], self.item_emb.weight[pos_items], self.item_emb.weight[neg_items]
        return (eu.norm(2, dim=1).pow(2) + ep.norm(2, dim=1).pow(2) + en.norm(2, dim=1).pow(2)).mean()

    def fused_loss(self, users, pos_items, neg_items, e_u, e_i, lambda_reg, lambda_fair=0.0, pop=None):
        """L_bpr + lambda_fair * L_fair + lambda_reg * L_reg (lightgcn_cu.py:635-648) in one kernel."""
        return fused_bpr_loss(self.graph, e_u, e_i, self.user_emb.weight, self.item_emb.weight, users, pos_items,
                              neg_items, lambda_reg, lambda_fair, pop)


class LightGCN(_Base):
    """Version-2/lighgcn_cu_pop.py:458.  M_ui = [U x I] base operator, M_iu = [I x U] credibility operator."""
    ORDER = "gs"

    def propagate(self):
        return self._final()

    def get_user_item_emb(self):
        return self.propagate()

    def bpr_loss(self, users, pos_items, neg_items, user_emb, item_emb, reg_weight: float):
        return fused_bpr_loss(self.graph, user_emb, item_emb, self.user_emb.weight, self.item_emb.weight, users,
                              pos_items, neg_items, reg_weight)


class RawLightGCN(torch.nn.Module):
    """Plain LightGCN of lightgcn.py:306-349 (the thesis' ablation baseline): ONE embedding table over
    users + items and the symmetric normalised adjacency; x <- A x on a bipartite graph is the Jacobi
    schedule on the two blocks of the table.  state_dict key: `emb.weight`."""
    ORDER = "jacobi"

    def __init__(self, num_users, num_items, emb_dim, num_layers, norm_adj):
        super().__init__()
        from .graph import NormAdj
        if not isinstance(norm_adj, NormAdj):
            raise TypeError("expected the handle returned by credgcn.graph.build_norm_adj")
        self.num_users, self.num_items, self.num_layers = num_users, num_items, num_layers
        self.num_nodes = num_users + num_items
        self.norm_adj, self.graph = norm_adj, norm_adj.graph
        if not lib().cgx_emb_dim_supported(emb_dim):
            raise _lib.CgxError(f"emb_dim={emb_dim} unsupported: use 16, 32, 64, 128 or 256")
        self.emb = torch.nn.Embedding(self.num_nodes, emb_dim)
        torch.nn.init.xavier_uniform_(self.emb.weight)

    def ego_tables(self):
        """(user table, item table, user gradient, item gradient) as TrainStep updates them: the row blocks [0, U) and
        [U, U + I) of the one table's storage, and the same blocks of a fresh buffer installed as its .grad."""
        w, U = self.emb.weight, self.num_users
        w.grad = torch.empty_like(w)
        return w.data[:U], w.data[U:], w.grad[:U], w.grad[U:]

    def propagate(self):
        w = self.emb.weight
        fu, fi = _Propagate.apply(w[: self.num_users], w[self.num_users:], self.graph, self.num_layers, self.ORDER)
        return torch.cat([fu, fi], dim=0)

    def get_user_item_emb(self):
        x = self.propagate()
        return x[: self.num_users], x[self.num_users:]

    def bpr_loss(self, users, pos_items, neg_items, user_emb, item_emb, reg_weight: float):
        w = self.emb.weight
        return fused_bpr_loss(self.graph, user_emb, item_emb, w[: self.num_users], w[self.num_users:], users,
                              pos_items, neg_items, reg_weight)


# ------------------------------------------------------------------------------------------
# optimiser + fused training step (sampler -> forward -> loss -> backward -> Adam), no autograd graph
# ------------------------------------------------------------------------------------------
class FusedAdam:
    """torch.optim.Adam(params, lr) semantics (defaults: betas (0.9, 0.999), eps 1e-8; lightgcn_cu.py:587)
    for the two embedding tables, one kernel launch per step.  The step count lives on the device so
    that a captured CUDA graph keeps advancing it.  `grads`, when given, are the two gradient buffers to read instead
    of the weights' .grad: the tables may be the two row blocks of ONE parameter (RawLightGCN), which is then
    torch.optim.Adam on that parameter, Adam being elementwise."""

    def __init__(self, user_weight: torch.Tensor, item_weight: torch.Tensor, lr=1e-3, betas=(0.9, 0.999), eps=1e-8,
                 grads=None):
        self.params = (user_weight, item_weight)
        self.grads = grads
        self.lr, self.betas, self.eps = float(lr), (float(betas[0]), float(betas[1])), float(eps)
        self.m = [torch.zeros_like(p) for p in self.params]
        self.v = [torch.zeros_like(p) for p in self.params]
        self.step_dev = torch.zeros(1, dtype=torch.int64, device=user_weight.device)   # steps taken so far

    def _grads(self):
        return self.grads if self.grads is not None else tuple(p.grad for p in self.params)

    def zero_grad(self, set_to_none: bool = False):
        for g in self._grads():
            if g is not None:
                g.zero_()

    @torch.no_grad()
    def step(self):
        pu, pi = self.params
        gu, gi = self._grads()
        dev = pu.device
        with torch.cuda.device(dev):
            st = stream_ptr(dev)
            check(lib().cgx_tick(ptr(self.step_dev), st))
            check(lib().cgx_adam_step(ptr(pu.data), ptr(_f32c(gu)), ptr(self.m[0]), ptr(self.v[0]), pu.numel(),
                                      ptr(pi.data), ptr(_f32c(gi)), ptr(self.m[1]), ptr(self.v[1]), pi.numel(),
                                      self.lr, self.betas[0], self.betas[1], self.eps, ptr(self.step_dev), 0, st))

    def state_dict(self):
        return {"step": int(self.step_dev.item()), "exp_avg": self.m, "exp_avg_sq": self.v, "lr": self.lr,
                "betas": self.betas, "eps": self.eps}


class TrainStep:
    """One full training step on pre-allocated buffers.  Equivalent to lightgcn_cu.py:608-652 /
    lighgcn_cu_pop.py:826-863: one (user, pos, neg) triple per batch user, final embeddings, BPR (+fair) + L2
    loss, backward, dense Adam.  The model hands over its ego tables with `ego_tables()` and its layer order as
    `ORDER`: the two weights of CredLightGCN / LightGCN, or the user and item row blocks of RawLightGCN's one table
    (lightgcn.py's loop: Jacobi order, one Adam over `emb.weight`), whose gradient fills the same blocks of its .grad.

    `step(users)` samples on device and updates the parameters; `forward_backward(users, pos, neg)` runs
    on an injected triple list and leaves the gradients in `.grad` (parity tests).  `capture(batch)` records
    the whole step as ONE CUDA graph (sampler offsets and the Adam step count are device-side counters), which
    removes the ~25 per-step launch calls from the host's critical path.

    `f_u` / `f_i` are the final embeddings of the last step.  The loss reads only the batch users' rows of f_u and
    the pos / neg rows of f_i, so when the item table is beyond L2 (the SpMM's regime switch), num_layers >= 2 and
    the device has room for a second forward workspace ((U + I) d floats) with DEFER_HEADROOM to spare, the step
    computes the last layer's products only on the batch users and on the item frontier (pos, neg and the
    batch users' train items: all that the batch users' last-layer rows gather).  The first read of `f_u` or `f_i`
    after a step computes the other rows, on the current stream, with the same bits as an eager forward.  The
    properties return the same tensor objects every time: a reference held across a later step() is not completed
    by it; read the attribute again."""

    # free device memory that must remain after the deferred path's own forward workspace, else the step stays eager
    DEFER_HEADROOM = 2 << 30

    def __init__(self, model: _Base | RawLightGCN, lr=1e-3, reg_weight=1e-4, fair_weight=0.0, pop=None, optimizer=None,
                 sampler=None):
        self.model, self.graph = model, model.graph
        self.reg, self.fair = float(reg_weight), float(fair_weight)
        # the ego tables and their gradients: two parameters, or the two row blocks of RawLightGCN's one table
        self._eu, self._ei, self._gu, self._gi = model.ego_tables()
        eu, ei = self._eu, self._ei
        dev = eu.device
        self.pop = None if pop is None else torch.as_tensor(pop, dtype=torch.float32, device=dev).contiguous()
        self._f_u, self._f_i = torch.empty_like(eu), torch.empty_like(ei)
        # dL/d(final tables): dense, but kept ALL-ZERO between steps -- the loss writes <= 3 * batch rows, flags them
        # for the adjoint (cgx_bpr_mark_rows) and the rows are zeroed again after use (cgx_bpr_clear_rows): no fill of
        # (U + I) d floats and no scan for non-zero rows per step
        self.g_u, self.g_i = torch.zeros_like(eu), torch.zeros_like(ei)
        self.nz_u = torch.zeros(eu.shape[0], dtype=torch.uint8, device=dev)
        self.nz_i = torch.zeros(ei.shape[0], dtype=torch.uint8, device=dev)
        self.front_i = torch.zeros(ei.shape[0], dtype=torch.uint8, device=dev)   # item frontier of the batch
        self.batch_u = torch.zeros(eu.shape[0], dtype=torch.uint8, device=dev)   # users of the batch
        self.opt = optimizer or FusedAdam(eu, ei, lr=lr, grads=(self._gu, self._gi))
        self.sampler = sampler
        self.phase_events = None      # set to a list to collect (start, fwd_end, loss_end, bwd_end) CUDA events
        self.side = torch.cuda.Stream(device=dev)     # plan (+ item frontier) overlap the forward
        self.tick = torch.zeros(1, dtype=torch.int64, device=dev)   # sampler offset counter (device side)
        self._bufs = {}
        self._graph = None
        # Deferred last layer: decided by the first forward (_defers_final).  Its layer buffers must survive the
        # backward, which overwrites the graph's shared workspace, so the deferred path owns a forward workspace.
        self._defer_final = None
        self._fws = self._all_rows = None
        self._pending = False         # f_u / f_i lack the rows outside the last step's masks
        self._final_error = None      # a failed completion: f_u / f_i are unusable until the next step

    @property
    def f_u(self) -> torch.Tensor:
        """[U, d] final user embeddings of the last step."""
        self._complete_final()
        return self._f_u

    @property
    def f_i(self) -> torch.Tensor:
        """[I, d] final item embeddings of the last step."""
        self._complete_final()
        return self._f_i

    def _defers_final(self, d, order, beyond_l2):
        """Whether steps restrict the last layer (see the class doc).  Inside L2 the masked products' per-entry flag
        lookup costs more than the rows they skip (C2: 0.479 ms per step with it against 0.463 without); and the
        deferred path needs (U + I) d floats more device memory, which C5 on one GPU does not have."""
        if self.model.num_layers < 2 or not beyond_l2:
            return False
        g = self.graph
        need = lib().cgx_propagate_workspace_bytes_for(g.by_user.ref(), g.by_item.ref(), d, order)
        free, _ = torch.cuda.mem_get_info(g.device)
        return free >= need + self.DEFER_HEADROOM

    @torch.no_grad()
    def _complete_final(self):
        """The last layer's products on the rows the last step left out: the complement of its masks, as the
        epilogue adds into f_u / f_i in place (a row computed twice would be added twice)."""
        if self._final_error is not None:
            raise self._final_error
        if not self._pending:
            return
        m, g = self.model, self.graph
        eu, ei = self._eu, self._ei
        d, K, order = eu.shape[1], m.num_layers, _lib.ORDERS[m.ORDER]
        dev = eu.device
        with torch.cuda.device(dev):
            rest_u = torch.eq(self.batch_u, 0).view(torch.uint8)
            rest_i = torch.eq(self.front_i, 0).view(torch.uint8)
            try:
                check(lib().cgx_propagate_fwd_layers(g.by_user.ref(), g.by_item.ref(), order, K, d, ptr(eu), ptr(ei),
                                                     ptr(self._f_u), ptr(self._f_i), K - 1, K, ptr(rest_u),
                                                     ptr(rest_i), ptr(self._all_rows), ptr(self._fws),
                                                     self._fws.numel(), stream_ptr(dev)))
            except _lib.CgxError as e:
                # part of the rows may have been added already, so a retry could add them twice: every read raises
                # until the next step recomputes the tables
                self._final_error = e
                raise
        self._pending = False

    def _mark(self, marks):
        if self.phase_events is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record(torch.cuda.current_stream(self.graph.device))
            marks.append(ev)

    def _batch_bufs(self, B, dev):
        if B not in self._bufs:
            self._bufs[B] = (torch.empty(3 * B, dtype=torch.int64, device=dev), bpr_buffers(self.graph, B, dev))
        return self._bufs[B]

    @torch.no_grad()
    def forward_backward(self, users, pos, neg):
        m, g = self.model, self.graph
        eu, ei = self._eu, self._ei
        d, K, order = eu.shape[1], m.num_layers, _lib.ORDERS[m.ORDER]
        ws = g.propagate_workspace(d, order)
        dev = eu.device
        users, pos, neg = _i64c(users, dev), _i64c(pos, dev), _i64c(neg, dev)
        plan, bufs = self._batch_bufs(users.numel(), dev)
        # The item frontier pays only when the item table is beyond L2 (the SpMM's regime switch): inside L2 the
        # masked gather's per-entry flag lookup costs more than the gathers it saves (C2: +9 us per backward).
        beyond_l2 = g.num_items * d * 4 > _lib.get_option("L2_TABLE_BYTES")
        if self._defer_final is None:
            self._defer_final = self._defers_final(d, order, beyond_l2)
        defer = bool(self._defer_final) and K >= 2     # K = 1: the last layer reads E^0, which Adam overwrites
        if defer and self._fws is None:
            self._fws = workspace(lib().cgx_propagate_workspace_bytes_for(g.by_user.ref(), g.by_item.ref(), d, order),
                                  dev)
            self._all_rows = torch.ones(max(g.num_users, g.num_items), dtype=torch.uint8, device=dev)
        front = self.front_i if beyond_l2 or defer else None
        marks = []
        self._pending, self._final_error = False, None
        with torch.cuda.device(dev):
            main = torch.cuda.current_stream(dev)
            self._mark(marks)
            self.side.wait_stream(main)                 # the indices are ready
            with torch.cuda.stream(self.side):
                bpr_plan(g, users, pos, neg, plan)      # scatter plan: beside the forward
                if front is not None:
                    batch_frontier(g, users, pos, neg, front, self.batch_u if defer else None)
            st = stream_ptr(dev)
            if defer:
                # layers 1..K-1 beside the plan and frontier, then layer K on the rows the loss reads
                fws = self._fws
                check(lib().cgx_propagate_fwd_layers(g.by_user.ref(), g.by_item.ref(), order, K, d, ptr(eu), ptr(ei),
                                                     ptr(self._f_u), ptr(self._f_i), 0, K - 1, None, None, None,
                                                     ptr(fws), fws.numel(), st))
                main.wait_stream(self.side)
                check(lib().cgx_propagate_fwd_layers(g.by_user.ref(), g.by_item.ref(), order, K, d, ptr(eu), ptr(ei),
                                                     ptr(self._f_u), ptr(self._f_i), K - 1, K, ptr(self.batch_u),
                                                     ptr(self.front_i), ptr(self._all_rows), ptr(fws), fws.numel(),
                                                     st))
                self._mark(marks)
                self._pending = True
            else:
                check(lib().cgx_propagate_fwd(g.by_user.ref(), g.by_item.ref(), order, K, d, ptr(eu), ptr(ei),
                                              ptr(self._f_u), ptr(self._f_i), ptr(ws), ws.numel(), st))
                self._mark(marks)
                main.wait_stream(self.side)
            loss, _, _, ego_rows, ego_coef = bpr_fused(g, self._f_u, self._f_i, eu, ei, users, pos, neg, self.reg,
                                                       self.fair, self.pop, self.g_u, self.g_i, plan, bufs)
            n_ent = ego_rows.numel()
            check(lib().cgx_bpr_mark_rows(ptr(ego_rows), n_ent, g.num_users, ptr(self.nz_u), ptr(self.nz_i), st))
            self._mark(marks)
            check(lib().cgx_propagate_bwd_frontier(g.by_user.ref(), g.by_item.ref(), order, K, d, ptr(self.g_u),
                                                   ptr(self.g_i), ptr(self.nz_u), ptr(self.nz_i), ptr(front),
                                                   ptr(self._gu), ptr(self._gi), ptr(ws), ws.numel(), st))
            self._mark(marks)
            apply_ego(g, ego_rows, ego_coef, eu, ei, self._gu, self._gi)
            check(lib().cgx_bpr_clear_rows(ptr(ego_rows), n_ent, g.num_users, d, ptr(self.g_u), ptr(self.g_i),
                                           ptr(self.nz_u), ptr(self.nz_i), st))
        if self.phase_events is not None:
            self.phase_events.append(marks)
        return loss

    def __call__(self, users, pos, neg):
        """Injected triples: forward, loss, backward, optimiser step."""
        loss = self.forward_backward(users, pos, neg)
        self.opt.step()
        return loss

    # ---- sampling step, optionally as one CUDA graph --------------------------------------------
    @torch.no_grad()
    def _sampled_step(self, users):
        dev = self.graph.device
        with torch.cuda.device(dev):
            check(lib().cgx_tick(ptr(self.tick), stream_ptr(dev)))
        pos, neg = self.sampler.sample(users, offset=0, offset_dev=self.tick)
        return self.__call__(users, pos, neg)

    def capture(self, batch: int, preserve_state: bool = True):
        """Record sample + forward + loss + backward + Adam for `batch` users as one CUDA graph.  The two warm-up
        steps before the capture do not count: parameters, optimiser state and counters are restored afterwards --
        unless preserve_state=False (three more copies of both tables do not fit next to the 1 B-edge shape)."""
        if self.sampler is None:
            raise _lib.CgxError("TrainStep.capture needs a TripleSampler (pass sampler=...)")
        dev = self.graph.device
        self._g_users = torch.zeros(batch, dtype=torch.int64, device=dev)
        keep = self.phase_events
        self.phase_events = None
        warm = torch.cuda.Stream(device=dev)
        warm.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(warm):                       # warm-up outside capture (allocations, attributes)
            state = opt_state = None
            if preserve_state:
                state = [self._eu.clone(), self._ei.clone()]
                opt_state = ([t.clone() for t in self.opt.m], [t.clone() for t in self.opt.v],
                             self.opt.step_dev.clone(), self.tick.clone()) if isinstance(self.opt, FusedAdam) else None
            for _ in range(2):
                self._sampled_step(self._g_users)
            # the warm-up steps must not count: restore parameters, optimiser state and counters
            if state is not None:
                self._eu.copy_(state[0])
                self._ei.copy_(state[1])
            if opt_state is not None:
                for dst, src in zip(self.opt.m, opt_state[0]):
                    dst.copy_(src)
                for dst, src in zip(self.opt.v, opt_state[1]):
                    dst.copy_(src)
                self.opt.step_dev.copy_(opt_state[2])
                self.tick.copy_(opt_state[3])
        torch.cuda.current_stream(dev).wait_stream(warm)
        torch.cuda.synchronize(dev)
        self._graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._graph):
            self._g_loss = self._sampled_step(self._g_users)
        self._g_pending = self._pending           # what each replay leaves of f_u / f_i
        self.phase_events = keep
        return self

    def step(self, users):
        """users: int64 batch of users with >= 1 train item (CUDA or pinned host tensor)."""
        if self.sampler is None:
            raise _lib.CgxError("TrainStep.step needs a TripleSampler (pass sampler=...)")
        if self._graph is not None and users.numel() == self._g_users.numel() and self.phase_events is None:
            self._g_users.copy_(users, non_blocking=True)
            self._graph.replay()
            self._pending, self._final_error = self._g_pending, None
            return self._g_loss
        return self._sampled_step(_i64c(users, self.graph.device))
