"""User-sharded propagation / training over several GPUs of one node (one process per GPU).

The reference is single-device; this is the row partition BASELINE.json names (SURVEY.md section 8e):

  * users are split into contiguous ranges balanced by non-zeros; each rank owns the user table,
    the user rows of the operator pattern and the sampling CSR of its range;
  * the item table is replicated;
  * user <- item products (A x_i, C^T x_i) read the replicated item table: no communication;
  * item <- user products (C x_u, A^T x_u) give every rank a PARTIAL item table (the sum over its own
    users); one exchange per layer makes it whole again (csrc/comm.cu over NVLink peer memory: pushed / pull /
    NVLS form, or a torch.distributed all-reduce).  Forward: K exchanges of [I, d]; backward: K, plus ONE
    all-gather of the compact loss gradient (the <= 2 * batch item rows each rank's triples touched).
  * evaluation is user-sharded with no exchange (only metric sums are reduced).

`ShardedPropagation` is written against a two-method backend so that the host-side schedule can
be exercised on CPU with the gloo backend (tests/test_sharded_gloo.py injects an oracle backend);
the product backend is `CudaBackend` (libcredgcn.so) and there is no CPU backend in this package.
"""
from __future__ import annotations

import json
import os
import time

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from ._lib import check, lib, ptr, stream_ptr, workspace
from .graph import CredGraph, build_graph
from .model import FusedAdam, apply_ego, bpr_buffers, bpr_fused, bpr_plan
from .sampler import TripleSampler


def partition_users(deg_u: np.ndarray, world: int) -> np.ndarray:
    """bounds[world + 1]: contiguous user ranges with (nearly) equal numbers of non-zeros."""
    deg_u = np.asarray(deg_u, dtype=np.int64)
    csum = np.concatenate([[0], np.cumsum(deg_u)])
    targets = csum[-1] * np.arange(1, world, dtype=np.float64) / world
    cuts = np.searchsorted(csum, targets, side="left")
    bounds = np.concatenate([[0], cuts, [deg_u.size]]).astype(np.int64)
    return np.maximum.accumulate(bounds)


def shard_edges(edges_2xE: np.ndarray, bounds: np.ndarray, rank: int) -> np.ndarray:
    """Edges of the users owned by `rank`, user ids rebased to the shard."""
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    u = edges_2xE[0]
    keep = (u >= lo) & (u < hi)
    out = edges_2xE[:, keep].copy()
    out[0] -= lo
    return out


def _world(group=None) -> int:
    return dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1


def all_reduce_sum(t: torch.Tensor, group=None) -> torch.Tensor:
    if _world(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


class CollectiveExchange:
    """Partial item table -> whole item table through torch.distributed (NCCL on GPUs, gloo in the CPU tests)."""

    def __init__(self, group=None):
        self.group = group

    def partial_buffer(self, shape, device):
        return torch.empty(shape, dtype=torch.float32, device=device)

    def reduce(self, buf):
        return all_reduce_sum(buf, self.group)

    def allgather(self, block: torch.Tensor) -> torch.Tensor:
        """[n] float32 per rank -> [world, n], rank order."""
        world = _world(self.group)
        out = torch.empty(world, block.numel(), dtype=block.dtype, device=block.device)
        if world > 1:
            dist.all_gather_into_tensor(out.view(-1), block.contiguous().view(-1), group=self.group)
        else:
            out[0] = block
        return out


class _RawCuda:
    def __init__(self, address, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (address, False),
                                         "version": 3, "strides": None}


class P2PExchange:
    """Same contract over NVLink peer memory (csrc/comm.cu): partials are written straight into a peer-mapped
    buffer and summed by a kernel of the library -- in rank order by the pull kernel (one- or two-shot) or, when the
    product pushed its rows to their owners, by the pushed form; inside the NVSwitch by the NVLS form when the
    buffers have a multicast mapping.  Needs all ranks on one node with peer access (NVSwitch); the process group is
    only used to hand out the mappings and to agree on failures."""

    REGION_ALIGN = 1 << 16

    # Backing of the communication buffers: "ipc" = cudaMalloc + cudaIpc handles; "symm" / "auto" = torch symmetric
    # memory (peer mappings + the NVSwitch multicast mapping the NVLS form needs), falling back to "ipc" when any rank
    # cannot.  (The classes read no environment; `bench.py --gpus N` maps its experiment switches onto these attributes.)
    DEFAULT_BACKING = "ipc"

    def __init__(self, max_floats: int, device, group=None, gather_floats: int = 0, backing: str | None = None):
        """max_floats: largest table exchanged; gather_floats: largest per-rank block of allgather(); backing: see
        DEFAULT_BACKING.
        Collective over `group`: EVERY rank issues the same sequence of torch.distributed calls whether or not
        its own CUDA calls succeed (a failure is agreed on after each phase and raised on all ranks together), so a
        rank without peer access can never leave the others waiting inside a mismatched collective."""
        import ctypes as C
        backing = backing or self.DEFAULT_BACKING
        self.group, self.device = group, torch.device(device)
        self.world = _world(group)
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        self.region = (4 * int(max_floats) + self.REGION_ALIGN - 1) // self.REGION_ALIGN * self.REGION_ALIGN
        self.flag_off = 4 * self.region
        self.gather_off = self.flag_off + 4096
        self.gather_block = (4 * int(gather_floats) + 15) // 16 * 16
        total = self.gather_off + self.world * self.gather_block + 256
        self.base = C.c_void_p()
        self.bases = (C.c_void_p * self.world)()
        self._opened = []
        handle = (C.c_char * 64)()

        def agree(phase, err):
            """All ranks learn whether ANY rank failed `phase`; all raise together."""
            bad = torch.tensor([0.0 if err is None else 1.0], device=self.device)
            if self.world > 1:
                dist.all_reduce(bad, op=dist.ReduceOp.MAX, group=group)
            if bad.item() != 0:
                self.close()
                raise _lib.CgxError(f"P2PExchange: {phase} failed on " +
                                    (f"this rank: {err}" if err is not None else "another rank"))

        self.mc = 0                 # multicast (NVSwitch) mapping of the buffers: 0 = none (IPC backing)
        self._symm = None
        self.bytes = None
        if backing in ("auto", "symm") and self.world > 1:
            self._try_symmetric_memory(total, group, agree_soft=lambda bad: self._any(bad, group))
        if self._symm is None:
            self._ipc_backing(total, group, handle, agree)
        self.epoch_dev = torch.zeros(1, dtype=torch.int64, device=self.device)   # exchanges done so far
        self.slot = 0                                                          # region of the next exchange
        if self.world > 1:
            dist.barrier(group=group)          # every rank has mapped every buffer before the first exchange

    def _any(self, bad: bool, group) -> bool:
        t = torch.tensor([1.0 if bad else 0.0], device=self.device)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
        return t.item() != 0

    def _try_symmetric_memory(self, total, group, agree_soft):
        """Back the buffers with torch symmetric memory: peer mappings AND -- where the fabric has it -- one NVSwitch
        multicast mapping, which the NVLS form of the exchange needs.  Any failure on any rank (agreed after each
        phase) leaves every rank on the cudaIpc backing."""
        import ctypes as C
        t = hdl = None
        try:
            import torch.distributed._symmetric_memory as symm
            t = symm.empty(int(total), dtype=torch.uint8, device=self.device)
        except Exception as e:                      # noqa: BLE001
            self._symm_error = f"{type(e).__name__}: {e}"
        if agree_soft(t is None):
            return
        try:
            hdl = symm.rendezvous(t, group if group is not None else dist.group.WORLD)
            ptrs = [int(x) for x in hdl.buffer_ptrs]
            mc = int(getattr(hdl, "multicast_ptr", 0) or 0)
            assert len(ptrs) == self.world and all(ptrs)
        except Exception as e:                      # noqa: BLE001
            self._symm_error = f"{type(e).__name__}: {e}"
            hdl = None
        if agree_soft(hdl is None):
            return
        if agree_soft(mc == 0):                     # multicast on every rank or on none
            mc = 0
        t.zero_()
        for r in range(self.world):
            self.bases[r] = ptrs[r]
        self.base = C.c_void_p(ptrs[self.rank])
        self.bytes, self._symm, self.mc = t, (t, hdl), mc
        with torch.cuda.device(self.device):
            check(lib().cgx_spmm_set_push_peers(self.bases, self.world))
            torch.cuda.synchronize(self.device)

    def _ipc_backing(self, total, group, handle, agree):
        import ctypes as C
        err = None
        with torch.cuda.device(self.device):
            try:                                    # phase 1: allocate + export
                check(lib().cgx_comm_alloc(total, C.byref(self.base)))
                check(lib().cgx_comm_ipc_handle(self.base, handle))
            except Exception as e:                  # noqa: BLE001
                err = f"{type(e).__name__}: {e}"
            agree("allocating the communication buffer", err)
            handles = [None] * self.world
            if self.world > 1:                      # outside any try: every rank takes part
                dist.all_gather_object(handles, bytes(handle.raw), group=group)
            try:                                    # phase 2: map the peers
                for p in range(self.world):
                    if p == self.rank:
                        self.bases[p] = self.base.value
                    else:
                        peer = C.c_void_p()
                        check(lib().cgx_comm_ipc_open(C.c_char_p(handles[p]), C.byref(peer)))
                        self._opened.append(peer)
                        self.bases[p] = peer.value
                check(lib().cgx_spmm_set_push_peers(self.bases, self.world))   # targets of the fused product + exchange
            except Exception as e:                  # noqa: BLE001
                err = f"{type(e).__name__}: {e}"
            agree("mapping the peers' buffers (no NVLink / IPC peer access?)", err)
        self.bytes = torch.as_tensor(_RawCuda(self.base.value, total), device=self.device)

    def check(self):
        """Raise if a cross-GPU barrier of an exchange timed out (a peer died or lost step): the kernels then gave up
        instead of hanging the job, and every table exchanged since is unusable.  Synchronises the device."""
        import ctypes as C
        if self.base is None or not self.base.value:
            return
        code = C.c_uint32(0)
        with torch.cuda.device(self.device):
            check(lib().cgx_comm_status(self.base, self.flag_off, self.world, C.byref(code)))
        if code.value:
            raise _lib.CgxError(f"P2PExchange: rank {self.rank} gave up waiting for rank {(code.value & 0xff) - 1} at "
                                f"barrier {'AB'[(code.value >> 8) - 1]} of an exchange "
                                f"(time-out {_lib.get_option('P2P_TIMEOUT_MS')} ms)")

    def close(self):
        """Unmap the peers' buffers and free the own one (after all ranks are done with the exchange)."""
        self.bytes = None
        if self._symm is not None:                  # symmetric memory: torch owns the mappings
            torch.cuda.synchronize(self.device)
            self._symm, self.base, self.mc = None, None, 0
            return
        with torch.cuda.device(self.device):
            torch.cuda.synchronize(self.device)
            for peer in self._opened:
                lib().cgx_comm_ipc_close(peer)
            self._opened = []
            if self.base is not None and self.base.value:
                lib().cgx_comm_free(self.base)
            self.base = None

    def _view(self, offset, shape):
        n = int(np.prod(shape))
        return self.bytes[offset: offset + 4 * n].view(torch.float32).view(shape)

    def begin_step(self):
        """Restart the region alternation: every step then uses the same addresses (CUDA-graph replay)."""
        self.slot = 0

    def partial_buffer(self, shape, device=None):
        """The `in` region of the NEXT exchange: fill it, then call reduce() on it."""
        if 4 * int(np.prod(shape)) > self.region:
            raise _lib.CgxError("P2PExchange: payload larger than the communication regions")
        return self._view(self.slot * self.region, shape)

    def push_enabled(self, avg_row_nnz=None) -> bool:
        """Fused SpMM -> owner push + local reduce (cgx_spmm_push / cgx_comm_allreduce_pushed): the default above
        2 ranks (C2 shards, 4 ranks: 0.896 vs 0.975 ms/step) and for tables of 64 MB and more at any rank count (the
        reduce-scatter half then hides under the product).  At 2 ranks and 10 MB tables the one-shot pull kernel has
        one barrier less and wins (0.793 vs 0.812 ms).  force_push = True / False forces it on / off."""
        if self.world < 2:
            return False
        if self.force_push is not None:
            return bool(self.force_push)
        if self.region < (64 << 20):                # small tables: latency-bound exchange
            return self.world > 2
        # large tables: pushing pays while the product is long next to the table it produces -- its posted stores
        # need (R-1)/R x table bytes of NVLink per product time.  C4 shards (80 non-zeros per item row) gain
        # (134.6 vs 137.8 ms at 2 ranks); C5 shards (10 per row, 256-byte rows) lose badly: the product itself becomes
        # NVLink-bound (134.5 ms per step pushed vs 97.6 pulled vs 85.8 NCCL at 8 ranks).
        return avg_row_nnz is None or avg_row_nnz >= 32

    force_push = None       # True / False overrides the default choice (tests, bench experiments)

    def exchange_pushed(self, shape, push_product):
        """One item-table exchange in pushed form.  `push_product(stage_off, rank, world, rows_per)` must launch the
        product whose rows are pushed to their owners (CudaBackend.item_rows_push); returns the reduced table."""
        n_rows, d = int(shape[0]), int(shape[1])
        rows_per = (n_rows + self.world - 1) // self.world
        if 4 * self.world * rows_per * d > self.region:
            raise _lib.CgxError("P2PExchange: payload larger than the communication regions")
        par = self.slot
        self.slot ^= 1
        push_product(par * self.region, self.rank, self.world, rows_per)
        with torch.cuda.device(self.device):
            st = stream_ptr(self.device)
            check(lib().cgx_tick(ptr(self.epoch_dev), st))
            check(lib().cgx_comm_allreduce_pushed(self.rank, self.world, self.bases, par * self.region,
                                                  (2 + par) * self.region, self.flag_off, n_rows, d, rows_per,
                                                  ptr(self.epoch_dev), st))
        return self._view((2 + par) * self.region, (n_rows, d))

    def allgather(self, block: torch.Tensor) -> torch.Tensor:
        """[n] float32 per rank -> [world, n] (a view of the gather region; valid until the next allgather)."""
        nbytes = (4 * block.numel() + 15) // 16 * 16
        if nbytes > self.gather_block:
            raise _lib.CgxError("P2PExchange.allgather: block larger than the gather region (gather_floats)")
        block = block.contiguous()
        with torch.cuda.device(self.device):
            st = stream_ptr(self.device)
            check(lib().cgx_tick(ptr(self.epoch_dev), st))
            check(lib().cgx_comm_allgather(self.rank, self.world, self.bases, ptr(block), self.gather_off,
                                           self.flag_off, nbytes, ptr(self.epoch_dev), st))
        out = self.bytes[self.gather_off: self.gather_off + self.world * nbytes].view(torch.float32)
        return out.view(self.world, nbytes // 4)[:, : block.numel()]

    use_nvls = None         # None: automatic (below); True / False force it on / off

    def nvls_enabled(self, nbytes: int) -> bool:
        """NVLS form of reduce(): needs the multicast mapping.  Automatic choice: tables of 64 MB and more on 4+
        ranks -- at 2 ranks the one-shot pull kernel moves the same bytes per direction and is faster (2.56 GB:
        3.84 vs 6.46 ms), and small tables are latency-bound (9.7 MB: 36 vs 54 us)."""
        if not self.mc or self.world < 2:
            return False
        if self.use_nvls is not None:
            return bool(self.use_nvls)
        return self.world >= 4 and nbytes >= (64 << 20)

    def reduce(self, buf):
        par = self.slot
        self.slot ^= 1
        n_pad = (buf.numel() + 3) // 4 * 4
        with torch.cuda.device(self.device):
            st = stream_ptr(self.device)
            check(lib().cgx_tick(ptr(self.epoch_dev), st))
            if self.nvls_enabled(4 * n_pad):
                import ctypes as C
                check(lib().cgx_comm_allreduce_nvls(self.rank, self.world, self.bases, C.c_void_p(self.mc),
                                                    par * self.region, (2 + par) * self.region, self.flag_off, n_pad,
                                                    ptr(self.epoch_dev), st))
                return self._view((2 + par) * self.region, tuple(buf.shape))
            check(lib().cgx_comm_allreduce(self.rank, self.world, self.bases, par * self.region,
                                           (2 + par) * self.region, self.flag_off, n_pad, ptr(self.epoch_dev), st))
        return self._view((2 + par) * self.region, tuple(buf.shape))


class BackendBase:
    """A shard backend provides item_rows(x_u, bwd) and user_rows(x_i, bwd); the fused form below has
    a generic default so that test doubles only implement the two products."""

    def user_rows_acc(self, x_i, bwd, acc_in, scale, need_y=True):
        """y = user_rows(x_i); acc = scale * (acc_in + y).  Returns (y or None, acc)."""
        y = self.user_rows(x_i, bwd)
        return (y if need_y else None), (acc_in + y).mul_(scale)


class CudaBackend(BackendBase):
    """The two products of one shard, on libcredgcn.so."""
    supports_sparse_rows = True
    supports_row_flags = True

    def __init__(self, graph: CredGraph):
        self.graph = graph
        self._ws = {}

    def _flags_of(self, x):
        """Row flags of x computed on device (a scan of the whole table)."""
        fkey = ("flags", x.shape[0])
        if fkey not in self._ws:
            self._ws[fkey] = torch.empty(x.shape[0], dtype=torch.uint8, device=x.device)
        flags = self._ws[fkey]
        check(lib().cgx_row_flags(ptr(x), x.shape[0], x.shape[1], ptr(flags), stream_ptr(x.device)))
        return flags

    def _spmm(self, csr, x, bwd, y=None, acc_in=None, acc_out=None, scale=1.0, sparse=False, x_flags=None,
              acc_flags=None):
        """sparse=True: x is a loss gradient (rows mostly zero) -- skip its zero rows, using x_flags (uint8 per row)
        when the caller has them, else flags scanned from x.  acc_flags: the same promise for acc_in."""
        x = x.contiguous()
        d = x.shape[1]
        if y is None and acc_out is None:
            y = torch.empty(csr.n_rows, d, dtype=torch.float32, device=x.device)
        key = (id(csr), d)
        if key not in self._ws:
            self._ws[key] = workspace(lib().cgx_spmm_workspace_bytes(csr.ref(), d), x.device)
        ws = self._ws[key]
        with torch.cuda.device(x.device):
            flags = None
            if sparse:
                flags = x_flags if x_flags is not None else self._flags_of(x)
            check(lib().cgx_spmm_ex(csr.ref(), int(bwd), d, ptr(x), ptr(flags), ptr(y), ptr(acc_in), ptr(acc_flags),
                                    ptr(acc_out), float(scale), ptr(ws), ws.numel(), stream_ptr(x.device)))
        return y if y is not None else acc_out

    def item_rows(self, x_u, bwd=False, out=None, sparse=False, x_flags=None):
        """Partial [I, d]: C x_u (bwd: A^T x_u) summed over THIS shard's users (written into `out` if given)."""
        return self._spmm(self.graph.by_item, x_u, bwd, y=out, sparse=sparse, x_flags=x_flags)

    def item_rows_push(self, x_u, bwd, stage_off, rank, world, rows_per, sparse=False, x_flags=None):
        """item_rows whose output rows go straight to their owner rank's staging area (cgx_spmm_push)."""
        csr = self.graph.by_item
        x = x_u.contiguous()
        d = x.shape[1]
        key = (id(csr), d)
        if key not in self._ws:
            self._ws[key] = workspace(lib().cgx_spmm_workspace_bytes(csr.ref(), d), x.device)
        ws = self._ws[key]
        with torch.cuda.device(x.device):
            flags = None
            if sparse:
                flags = x_flags if x_flags is not None else self._flags_of(x)
            check(lib().cgx_spmm_push(csr.ref(), int(bwd), d, ptr(x), None if flags is None else ptr(flags), stage_off,
                                      rank, world, rows_per, ptr(ws), ws.numel(), stream_ptr(x.device)))

    def user_rows(self, x_i, bwd=False):
        """[U_local, d]: A x_i (bwd: C^T x_i) for this shard's users."""
        return self._spmm(self.graph.by_user, x_i, bwd)

    def user_rows_acc(self, x_i, bwd, acc_in, scale, need_y=True, sparse=False, acc_flags=None, acc_out=None):
        """Same product with the running sum / gradient seed fused into the SpMM epilogue (acc_out: where to write
        the sum; acc_flags: row flags of acc_in, whose unflagged rows are then not read)."""
        csr = self.graph.by_user
        y = torch.empty(csr.n_rows, x_i.shape[1], dtype=torch.float32, device=x_i.device) if need_y else None
        acc = acc_out if acc_out is not None else torch.empty(csr.n_rows, x_i.shape[1], dtype=torch.float32,
                                                              device=x_i.device)
        self._spmm(csr, x_i, bwd, y=y, acc_in=acc_in.contiguous(), acc_out=acc, scale=scale, sparse=sparse,
                   acc_flags=acc_flags)
        return y, acc


class ShardedPropagation:
    """K-layer propagation and its adjoint over user shards (lightgcn_cu.py:420-448 /
    Version-2/lighgcn_cu_pop.py:472-490 and their autograd; SURVEY.md appendix C)."""

    def __init__(self, backend, num_layers: int, order: str, group=None, exchange=None):
        if order not in ("jacobi", "gs"):
            raise ValueError(order)
        self.b, self.K, self.order, self.group = backend, int(num_layers), order, group
        self.ex = exchange or CollectiveExchange(group)

    def _push(self) -> bool:
        fn = getattr(self.ex, "push_enabled", None)
        if fn is None:
            return False
        g = getattr(self.b, "graph", None)
        avg = (g.by_item.nnz / max(g.by_item.n_rows, 1)) if g is not None else None
        return fn(avg)

    def _flags_ok(self):
        return getattr(self.b, "supports_row_flags", False)

    def _hint(self, sparse):
        """`sparse=True` keyword for backends that can skip zero rows of the input (an optimisation hint)."""
        return {"sparse": True} if sparse and getattr(self.b, "supports_sparse_rows", False) else {}

    def _item_exchange(self, x_u, bwd, shape, sparse=False, x_flags=None):
        """Partial item table of this shard -> whole item table (one exchange).  sparse: x_u is the loss
        gradient itself (rows mostly zero; x_flags = its row flags when the caller has them)."""
        fl = {"x_flags": x_flags} if (sparse and x_flags is not None and self._flags_ok()) else {}
        if hasattr(self.b, "item_rows_push") and self._push():
            return self.ex.exchange_pushed(
                shape, lambda off, rank, world, rows_per: self.b.item_rows_push(x_u, bwd, off, rank, world, rows_per,
                                                                              sparse, **fl))
        buf = self.ex.partial_buffer(shape, x_u.device)
        res = self.b.item_rows(x_u, bwd, out=buf, **self._hint(sparse), **fl)
        if res is not buf:                      # backends without an `out` argument return a fresh tensor
            buf.copy_(res)
        return self.ex.reduce(buf)

    def forward(self, e0_u: torch.Tensor, e0_i: torch.Tensor):
        """e0_u: this shard's user rows; e0_i: the replicated item table.  Returns (final_u shard, final_i)."""
        s = 1.0 / (self.K + 1)
        acc_u, acc_i = e0_u, e0_i
        u, i = e0_u, e0_i
        for k in range(self.K):
            last = k == self.K - 1
            i_new = self._item_exchange(u, False, tuple(e0_i.shape))
            u_new, acc_u = self.b.user_rows_acc(i if self.order == "jacobi" else i_new, False, acc_u,
                                                s if last else 1.0, need_y=not last)
            acc_i = acc_i + i_new if k == 0 else acc_i.add_(i_new)
            u, i = u_new, i_new
        return acc_u, acc_i.mul_(s)

    def backward(self, g_u: torch.Tensor, g_i_total: torch.Tensor, seed_rows=None, g_u_flags=None, out_u=None):
        """g_u: dL/d(final_u) rows of this shard; g_i_total: dL/d(final_i) already summed over ranks.
        seed_rows: optional (rows int64[n], keep bool[n]) -- g_i_total is zero outside rows[keep] (distinct rows): the
        seed is then added to each adjoint layer row by row instead of by a pass over the whole table, and in
        Gauss-Seidel order the item result (s * g_i_total, just as sparse) is left to the caller (None).
        g_u_flags: optional uint8 row flags of g_u (unflagged rows are all zero and are then never read);
        out_u: optional buffer for dL/dE0_u.
        Returns (dL/dE0_u shard, dL/dE0_i replicated)."""
        s = 1.0 / (self.K + 1)
        fl = {"acc_flags": g_u_flags} if (g_u_flags is not None and self._flags_ok()) else {}

        def last_out(last):
            return {"acc_out": out_u} if (last and out_u is not None and self._flags_ok()) else {}

        def add_seed(t):
            if seed_rows is None:
                return t.add_(g_i_total)
            rows, keep = seed_rows
            return t.index_add_(0, rows, g_i_total[rows] * keep[:, None])

        if self.order == "gs":
            bu = g_u
            for k in range(self.K):   # only the first product gathers the (row-sparse) loss gradient itself
                bi = add_seed(self._item_exchange(bu, True, tuple(g_i_total.shape), sparse=k == 0,
                                                  x_flags=g_u_flags))
                _, bu = self.b.user_rows_acc(bi, True, g_u, s if k == self.K - 1 else 1.0, need_y=False, **fl,
                                             **last_out(k == self.K - 1))
            return bu, (g_i_total.mul(s) if seed_rows is None else None)
        bu, bi = g_u, g_i_total
        for k in range(self.K):
            last = k == self.K - 1
            _, nu = self.b.user_rows_acc(bi, True, g_u, s if last else 1.0, need_y=False, **self._hint(k == 0), **fl,
                                         **last_out(last))
            ni = add_seed(self._item_exchange(bu, True, tuple(g_i_total.shape), sparse=k == 0, x_flags=g_u_flags))
            bu, bi = nu, (ni.mul_(s) if last else ni)
        return bu, bi


def build_local_graph(local_edges, num_local_users, num_items, cred_local, variant, device, group=None) -> CredGraph:
    """One shard's CredGraph; item degrees (weights, popularity law, alpha_i) are all-reduced."""
    return build_graph(local_edges, num_local_users, num_items, cred_local, variant, device,
                       reduce_item_degrees=lambda d: all_reduce_sum(d, group))


# ------------------------------------------------------------------------------------------
# compact loss gradient of the sharded step: pack / unpack (pure tensor code)
# ------------------------------------------------------------------------------------------
def item_gradient_block_floats(B: int, d: int) -> int:
    """[2B, d] gradient rows | 2B L2 coefficients | 2B row ids (int32 bits) | loss (+ 3 floats of padding)."""
    return 2 * B * (d + 2) + 4


def pack_item_gradient(ego_rows, ego_coef, gi_local, loss, B: int, Bm: int, U: int, d: int, count=None) -> torch.Tensor:
    """One rank's block.  ego_rows int32[3B] / ego_coef float[3B] come from cgx_bpr_fwd_bwd: entry k names the row of
    the k-th position of the scatter plan when that position starts a run (users < U, items offset by U), else -1; the
    plan is sorted by row with the B user entries first, so the item runs live in positions [B, 3B) -- or, when the
    batch has a device count c (int64[1] tensor `count`: triples at or past it are padding), in [c, 3c), the absent
    entries sorting last.  gi_local [I, d] holds the gradient rows the loss wrote.  Blocks have the size of
    Bm = max_batch on every rank (ranks may hold different batch sizes): unused slots carry row id -1 and zeros."""
    dev = gi_local.device
    if count is None:
        er, ec = ego_rows[B:], ego_coef[B:]
    else:                                   # positions c .. c + 2B - 1 (clamped; those past 3c hold -1)
        at = (torch.arange(2 * B, device=dev) + count).clamp_(max=3 * B - 1)
        er, ec = ego_rows[at], ego_coef[at]
    valid = er >= U
    rows = torch.where(valid, er - U, torch.zeros_like(er)).to(torch.int64)
    block = torch.zeros(item_gradient_block_floats(Bm, d), dtype=torch.float32, device=dev)
    block[: 2 * B * d].view(2 * B, d).copy_(torch.where(valid[:, None], gi_local[rows], 0.0))
    o_coef, o_rows, o_loss = 2 * Bm * d, 2 * Bm * (d + 1), 2 * Bm * (d + 2)
    block[o_coef: o_coef + 2 * B] = torch.where(valid, ec, 0.0)   # (non-head slots are uninitialised)
    rid_local = torch.full((2 * Bm,), -1, dtype=torch.int32, device=dev)
    rid_local[: 2 * B] = torch.where(valid, rows, torch.full_like(rows, -1)).to(torch.int32)
    block[o_rows: o_rows + 2 * Bm] = rid_local.view(torch.float32)
    block[o_loss] = loss.reshape(-1)[0]
    return block


def unpack_item_gradient(blocks: torch.Tensor, Bm: int, d: int, I: int):
    """blocks [world, n] (rank order) -> (vals [world, 2Bm, d], coef [world, 2Bm], rows [world, 2Bm] with invalid
    slots mapped to the dummy row I, ok [world, 2Bm], total loss [1])."""
    world = blocks.shape[0]
    o_coef, o_rows, o_loss = 2 * Bm * d, 2 * Bm * (d + 1), 2 * Bm * (d + 2)
    vals = blocks[:, : 2 * Bm * d].reshape(world, 2 * Bm, d)
    coef = blocks[:, o_coef: o_coef + 2 * Bm]
    rid = blocks[:, o_rows: o_rows + 2 * Bm].contiguous().view(torch.int32).to(torch.int64)
    ok = rid >= 0
    rows_all = torch.where(ok, rid, torch.full_like(rid, I))
    return vals, coef, rows_all, ok, blocks[:, o_loss].sum().reshape(1)


def distinct_rows(rows_all: torch.Tensor, ok: torch.Tensor, owner: torch.Tensor, I: int):
    """(rows int64[n] clamped to [0, I), keep bool[n]): keep marks ONE slot per distinct valid row (which of the
    duplicates wins is irrelevant: callers read the row's value from a dense table).  owner: int64[I + 1] scratch."""
    flat = rows_all.reshape(-1)
    ar = torch.arange(flat.numel(), device=flat.device)
    owner.scatter_(0, flat, ar)
    keep = (owner[flat] == ar) & ok.reshape(-1)
    return flat.clamp(max=I - 1), keep


class ShardedTrainStep:
    """One training step over user shards: local sampling, sharded forward, fused loss on the local
    triples (means over the GLOBAL batch), sharded backward, Adam on (local users, replicated items).

    Exchanges per step: K item tables forward, K backward, and ONE all-gather of the compact loss gradient -- the
    loss touches <= 2 * batch item rows per rank, so the gradient seed dL/d(final_i), the item L2 gradient and the loss
    value travel as (row id, coefficient, d floats) blocks of a few MB instead of two dense [I, d] tables, and every
    rank adds the blocks in rank order (identical bits on every rank)."""

    def __init__(self, graph: CredGraph, user_emb: torch.Tensor, item_emb: torch.Tensor, num_layers, order,
                 lr=1e-3, reg_weight=1e-4, mix_pop=0.7, gamma=0.75, max_tries=50, seed=42, group=None,
                 exchange: str = "p2p", max_batch: int = 4096, fair_weight: float = 0.0, pop=None):
        """fair_weight / pop: the fairness term of lightgcn_cu.py (pop: float[I], deg_i / max(deg_i) of the GLOBAL
        item degrees); its gradient rides in the loss gradient the step exchanges."""
        self.graph, self.group = graph, group
        self.eu = torch.nn.Parameter(user_emb.contiguous())
        self.ei = torch.nn.Parameter(item_emb.contiguous())
        dev = self.ei.device
        I, d = self.ei.shape
        self.max_batch = int(max_batch)
        # The loss gradient travels compact (rows the batch touched) when the item table is large; for small tables
        # (C2 shards: 10 MB) one dense exchange of [seed ; L2 gradient ; loss] is cheaper than the ~40 small launches
        # of packing, gathering and unpacking (C2 x 2: 0.78 vs 1.06 ms per step).
        self.compact = I * d * 4 >= (64 << 20) if self.force_compact is None else bool(self.force_compact)
        self.ex = None
        if exchange == "auto":
            exchange = self.choose_exchange(graph, I, d, _world(group))
        if not isinstance(exchange, str):          # an exchange object made by the caller (tests share one)
            self.ex = exchange
        elif exchange == "p2p" and _world(group) > 1:
            # peer mapping can be unavailable (no NVLink/IPC between the ranks): P2PExchange agrees on the outcome
            # over `group` and raises on ALL ranks together, which then all use the collective exchange.
            # Big tables with short item rows take the NVLS form, which needs the multicast mapping of symmetric memory.
            try:
                self.ex = P2PExchange(max((I + _world(group)) * d, 0 if self.compact else 2 * I * d + 4), dev, group,
                                      gather_floats=self._block_floats(self.max_batch, d),
                                      backing="auto" if self.wants_nvls(graph, I, d, _world(group)) else None)
            except _lib.CgxError as e:
                self._p2p_error = str(e)
        if self.ex is None:
            self.ex = CollectiveExchange(group)
        graph.set_emb_dim(d)          # hot-row hints of the SpMMs for this width
        self.prop = ShardedPropagation(CudaBackend(graph), num_layers, order, group, self.ex)
        self.sampler = TripleSampler(graph, mix_pop, gamma, max_tries, seed)
        self.reg, self.fair = float(reg_weight), float(fair_weight)
        self.pop = None if pop is None else torch.as_tensor(pop, dtype=torch.float32, device=dev).contiguous()
        self.eu.grad, self.ei.grad = torch.zeros_like(self.eu), torch.zeros_like(self.ei)
        self.opt = FusedAdam(self.eu, self.ei, lr=lr)
        # dense gradient tables kept ZERO outside the rows of the current batch (flagged for the adjoint by
        # cgx_bpr_mark_rows, cleared row by row after use): no per-step fill or scan of whole tables
        self.g_u = torch.zeros_like(self.eu)
        self.nz_u = torch.zeros(self.eu.shape[0], dtype=torch.uint8, device=dev)
        self.nz_i_local = torch.zeros(I, dtype=torch.uint8, device=dev)
        self.gi_local = torch.zeros_like(self.ei)            # bpr writes whole rows; only those rows are read back
        self.g_i = torch.zeros_like(self.ei)                 # dL/d(final_i), summed over ranks
        self.owner = torch.full((I + 1,), -1, dtype=torch.int64, device=dev)
        self.tick = torch.zeros(1, dtype=torch.int64, device=dev)
        self._ego_u = None          # dense form only: user L2 gradient buffer
        self._bufs = {}
        self._graph = None
        self._sel = None            # device-side batch selection of an epoch (plan_epochs)
        self._g_selected = False    # the captured graph is the epoch step (capture(selected=True))

    # Tables of 256 MB and more whose item rows are short (C5 shards: 10 non-zeros per row -- the pushed form makes
    # the product NVLink-bound there).  Measured on 8 B200s, C5, ms per step: pushed 134.5, pull kernel 97.6, NCCL 85.8,
    # this library's NVLS kernel (inside the CUDA graph) 85.4 -- so the peer-memory exchange stays, in its NVLS form.
    BIG_SHORT_ROWS_EXCHANGE = "p2p"

    force_compact = None        # tests: True / False overrides the size rule of the loss-gradient exchange

    @staticmethod
    def wants_nvls(graph, I, d, world) -> bool:
        big = I * d * 4 >= (256 << 20)
        short = graph.by_item.nnz / max(graph.by_item.n_rows, 1) < 32
        return world >= 4 and big and short

    @classmethod
    def choose_exchange(cls, graph, I, d, world) -> str:
        if world < 2:
            return "p2p"
        big = I * d * 4 >= (256 << 20)
        short = graph.by_item.nnz / max(graph.by_item.n_rows, 1) < 32
        return cls.BIG_SHORT_ROWS_EXCHANGE if (big and short) else "p2p"

    @staticmethod
    def _block_floats(B: int, d: int) -> int:
        return item_gradient_block_floats(B, d)

    @torch.no_grad()
    def __call__(self, users_local: torch.Tensor, batch_total: int | None = None, triples=None, count=None,
                 total=None, slots=None):
        """batch_total: global batch size (default: every rank holds a batch of this size).
        triples: optional injected (pos, neg) for users_local instead of sampling (parity tests).
        count / total / slots: int64 device tensors of a padded batch (cgx_batch_select): entries at or past count[0]
        are absent, total[0] is the global batch size, slots the entries' positions in the global batch (their
        sampler streams)."""
        g, dev = self.graph, self.eu.device
        B = users_local.numel()
        world = _world(self.group)
        B_total = 0 if total is not None else int(batch_total) if batch_total is not None else B * world
        U, (I, d) = g.num_users, self.ei.shape
        if B not in self._bufs:
            self._bufs[B] = (torch.empty(3 * B, dtype=torch.int64, device=dev), bpr_buffers(g, B, dev),
                             (torch.zeros(B, dtype=torch.int64, device=dev), torch.zeros(B, dtype=torch.int64,
                                                                                           device=dev)))
        plan, bufs, pn = self._bufs[B]
        if hasattr(self.ex, "begin_step"):
            self.ex.begin_step()
        with torch.cuda.device(dev):
            check(lib().cgx_tick(ptr(self.tick), stream_ptr(dev)))
        if triples is None:
            pos, neg = self.sampler.sample(users_local, offset=0, offset_dev=self.tick, slots=slots, count=count,
                                           out=pn)
        else:
            pos, neg = (torch.as_tensor(t, device=dev).to(torch.int64) for t in triples)
        bpr_plan(g, users_local, pos, neg, plan, count=count)
        f_u, f_i = self.prop.forward(self.eu.data, self.ei.data)
        if not self.compact:
            return self._finish_dense(users_local, pos, neg, plan, bufs, f_u, f_i, B_total, count, total)
        loss, _, _, ego_rows, ego_coef = bpr_fused(g, f_u, f_i, self.eu.data, self.ei.data, users_local, pos, neg,
                                                   self.reg, self.fair, self.pop, self.g_u, self.gi_local, plan, bufs,
                                                   B_total, count=count, total=total)
        with torch.cuda.device(dev):
            check(lib().cgx_bpr_mark_rows(ptr(ego_rows), ego_rows.numel(), U, ptr(self.nz_u), ptr(self.nz_i_local),
                                          stream_ptr(dev)))
        # ---- compact item part (pack -> all-gather -> unpack: pure tensor code, unit-tested on the CPU with gloo) ----
        Bm = self.max_batch
        if B > Bm:
            raise _lib.CgxError(f"ShardedTrainStep: batch of {B} users exceeds max_batch={Bm}")
        block = pack_item_gradient(ego_rows, ego_coef, self.gi_local, loss, B, Bm, U, d, count)
        blocks = self.ex.allgather(block)                                   # [world, n], rank order
        vals, coef, rows_all, ok, total_loss = unpack_item_gradient(blocks, Bm, d, I)
        for r in range(world):                                              # rank order: same bits on every rank
            self.g_i.index_add_(0, rows_all[r].clamp(max=I - 1), torch.where(ok[r][:, None], vals[r], 0.0))
        flat_c, keep = distinct_rows(rows_all, ok, self.owner, I)
        d_u, d_i = self.prop.backward(self.g_u, self.g_i, seed_rows=(flat_c, keep), g_u_flags=self.nz_u,
                                      out_u=self.eu.grad)
        if d_u is not self.eu.grad:
            self.eu.grad.copy_(d_u)
        # user part of the L2 gradient stays local (item entries masked out: rows >= U); added after the adjoint
        ego_user = torch.where(ego_rows < U, ego_rows, torch.full_like(ego_rows, -1))
        apply_ego(g, ego_user, ego_coef, self.eu.data, self.ei.data, self.eu.grad, self.gi_local)
        # item gradient: in Gauss-Seidel order it is s * seed + L2 term, non-zero on the batch's rows only
        if d_i is None:
            s = 1.0 / (self.prop.K + 1)
            self.ei.grad.index_add_(0, flat_c, self.g_i[flat_c] * (keep[:, None] * s))
        else:
            self.ei.grad.copy_(d_i)
        for r in range(world):
            rr = rows_all[r].clamp(max=I - 1)
            self.ei.grad.index_add_(0, rr, self.ei.data[rr] * (coef[r] * ok[r])[:, None])
        self.opt.step()
        # restore the all-zero invariant of the dense gradient tables, row by row
        with torch.cuda.device(dev):
            check(lib().cgx_bpr_clear_rows(ptr(ego_rows), ego_rows.numel(), U, d, ptr(self.g_u), ptr(self.gi_local),
                                           ptr(self.nz_u), ptr(self.nz_i_local), stream_ptr(dev)))
        self.g_i.index_fill_(0, flat_c, 0.0)            # (index_fill_: `t[idx] = 0.0` would copy a host scalar, which a
        if d_i is None:                                 #  CUDA-graph capture does not allow)
            self.ei.grad.index_fill_(0, flat_c, 0.0)
        return total_loss

    def _finish_dense(self, users_local, pos, neg, plan, bufs, f_u, f_i, B_total, count=None, total=None):
        """Loss, adjoint and Adam with ONE dense exchange of [item gradient seed ; item L2 gradient ; loss] -- the
        small-table form of the step (2 I d + 4 floats through the same exchange as the item tables)."""
        g, dev = self.graph, self.eu.device
        n = self.ei.numel()
        red = self.ex.partial_buffer((2 * n + 4,), dev)
        gi2 = red[: 2 * n].view(2, *self.ei.shape)
        self.g_u.zero_()
        red.zero_()
        if self._ego_u is None:
            self._ego_u = torch.zeros_like(self.eu)
        self._ego_u.zero_()
        bufs = (red[2 * n: 2 * n + 1],) + tuple(bufs[1:])
        _, _, _, ego_rows, ego_coef = bpr_fused(g, f_u, f_i, self.eu.data, self.ei.data, users_local, pos, neg,
                                                self.reg, self.fair, self.pop, self.g_u, gi2[0], plan, bufs, B_total,
                                                count=count, total=total)
        apply_ego(g, ego_rows, ego_coef, self.eu.data, self.ei.data, self._ego_u, gi2[1])
        # cloned: the exchange's output region is recycled two exchanges later, the seed is needed by every layer
        red = self.ex.reduce(red).clone()
        gi2 = red[: 2 * n].view(2, *self.ei.shape)
        d_u, d_i = self.prop.backward(self.g_u, gi2[0])
        self.eu.grad.copy_(d_u.add_(self._ego_u))
        self.ei.grad.copy_(d_i.add_(gi2[1]))
        self.opt.step()
        return red[2 * n: 2 * n + 1]

    def capture(self, batch: int, selected: bool = False):
        """Record the whole sharded step as one CUDA graph.  Only with the peer-memory exchange: every launch
        of the step is then a kernel of this library or a torch elementwise op, and the exchange epochs are
        device-side counters.  (Capturing the NCCL variant hung on this stack: torch 2.11 / NCCL 2.28.9.)
        selected=True records the epoch step of plan_epochs() instead -- batch selection on the device, then the step
        over the padded local batch of capacity max_batch -- which step_selected() replays: every batch of an epoch,
        the tail batch included, runs the same graph with no host work."""
        if not isinstance(self.ex, P2PExchange):
            raise _lib.CgxError("ShardedTrainStep.capture needs exchange='p2p'")
        if selected and self._sel is None:
            raise _lib.CgxError("ShardedTrainStep.capture(selected=True) needs plan_epochs() first")
        dev = self.eu.device
        self._g_users = torch.zeros(batch, dtype=torch.int64, device=dev)
        run = self._selected_step if selected else (lambda: self(self._g_users))
        state = (self.eu.data, self.ei.data, self.opt.m[0], self.opt.m[1], self.opt.v[0], self.opt.v[1],
                 self.opt.step_dev, self.tick) + ((self._sel["step"],) if selected else ())
        warm = torch.cuda.Stream(device=dev)
        warm.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(warm):
            keep = [t.clone() for t in state]
            for _ in range(2):                     # every rank runs the same two steps: exchanges stay matched
                run()
            for dst, src in zip(state, keep):
                dst.copy_(src)
        torch.cuda.current_stream(dev).wait_stream(warm)
        torch.cuda.synchronize(dev)
        self._graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._graph):
            self._g_loss = run()
        self._g_selected = selected
        return self

    # ---- epochs with device-side batch selection (train_on_arrays_sharded) ----------------------------------------
    def plan_epochs(self, n_train: int, lo: int, hi: int):
        """Buffers of the epoch step: the epoch's permutation of the n_train GLOBAL train users (begin_epoch), a device
        batch counter, and the selection outputs of capacity max_batch.  This rank owns the users [lo, hi)."""
        dev = self.eu.device
        i64 = dict(dtype=torch.int64, device=dev)
        self._sel = dict(perm=torch.zeros(int(n_train), **i64), n_train=int(n_train), lo=int(lo), hi=int(hi),
                         step=torch.zeros(1, **i64), users=torch.zeros(self.max_batch, **i64),
                         slots=torch.zeros(self.max_batch, **i64), count=torch.zeros(1, **i64),
                         total=torch.zeros(1, **i64))
        return self

    def begin_epoch(self, perm):
        """Upload the epoch's permutation of the global train users (identical on every rank) and restart at batch 0."""
        sel = self._sel
        p = torch.as_tensor(np.ascontiguousarray(perm, dtype=np.int64) if not isinstance(perm, torch.Tensor) else perm)
        if p.numel() != sel["n_train"]:
            raise _lib.CgxError(f"begin_epoch: permutation of {p.numel()} users, planned {sel['n_train']}")
        sel["perm"].copy_(p.to(torch.int64))
        sel["step"].zero_()

    def _selected_step(self):
        sel, dev = self._sel, self.eu.device
        with torch.cuda.device(dev):
            st = stream_ptr(dev)
            check(lib().cgx_batch_select(ptr(sel["perm"]), sel["n_train"], ptr(sel["step"]), self.max_batch,
                                         sel["lo"], sel["hi"], ptr(sel["users"]), ptr(sel["slots"]), ptr(sel["count"]),
                                         ptr(sel["total"]), st))
            check(lib().cgx_tick(ptr(sel["step"]), st))
        return self(sel["users"], count=sel["count"], total=sel["total"], slots=sel["slots"])

    def step_selected(self):
        """The next batch of the epoch (begin_epoch): the captured graph when capture(..., selected=True) ran, else
        the same launches eagerly.  Returns the global loss of the batch (float[1] device tensor)."""
        if self._graph is not None and self._g_selected:
            self._graph.replay()
            return self._g_loss
        return self._selected_step()

    def last_batch(self):
        """(global users, global slots, pos, neg) of this rank's part of the last selected batch (host NumPy)."""
        sel = self._sel
        c = int(sel["count"].item())
        pos, neg = self._bufs[self.max_batch][2]
        return ((sel["users"][:c] + sel["lo"]).cpu().numpy(), sel["slots"][:c].cpu().numpy(),
                pos[:c].cpu().numpy(), neg[:c].cpu().numpy())

    def step(self, users):
        if self._graph is not None and not self._g_selected and users.numel() == self._g_users.numel():
            self._g_users.copy_(users, non_blocking=True)
            self._graph.replay()
            return self._g_loss
        return self(torch.as_tensor(users).to(self.eu.device, non_blocking=True))

    def check(self):
        """Raise if an exchange gave up waiting for a peer (P2PExchange.check; synchronises)."""
        if isinstance(self.ex, P2PExchange):
            self.ex.check()

    def close(self):
        self._graph = None
        if isinstance(self.ex, P2PExchange):
            self.ex.close()


@torch.no_grad()
def evaluate_full_ranking_sharded(f_u_local, f_i, graph: CredGraph, test_edges_local, num_items, Ks=(10, 20),
                                  item_pop=None, total_train=0, cred_local=None, group_pct=0.20, group=None,
                                  precision="fp32"):
    """User-sharded full-rank evaluation (Version-2/lighgcn_cu_pop.py:653-752): every rank ranks ITS users
    against the replicated item table -- no embedding traffic -- and reduces them to metric sums on the device
    (cgx_eval_metrics).  Across ranks go: the 7 sums per cut-off (all-reduce, double), the coverage bitmaps
    (all-gather, OR-ed locally) and one credibility value per evaluated user (all-gather; the high / low groups are
    percentiles of the GLOBAL credibility order, V2:406-423).
    `graph` is the rank's local CredGraph (train mask = its duplicate-keeping user rows); `test_edges_local`
    holds the rank's users with shard-local ids."""
    from . import evaluate as ev
    from .graph import user_csr_device
    dev = f_u_local.device
    U_loc = graph.num_users
    te = user_csr_device(test_edges_local, U_loc, num_items, dev)
    users_dev = torch.nonzero(te[0][1:] > te[0][:-1]).flatten()
    n_loc = int(users_dev.numel())
    world = _world(group)
    K = max(Ks)
    ks = sorted(set(int(k) for k in Ks))
    extra = item_pop is not None and cred_local is not None

    def gather(x: np.ndarray):
        if world == 1:
            return [x]
        parts = [None] * world
        dist.all_gather_object(parts, x, group=group)
        return parts

    flags_dev = pop_dev = groups = None
    counts = gather(np.int64(n_loc))
    n = int(sum(int(c) for c in counts))
    if n == 0:
        raise RuntimeError("No users with test interactions. Check your split or threshold.")
    if extra:
        users_np = users_dev.cpu().numpy()
        parts = gather(np.asarray(cred_local)[users_np])
        rank = dist.get_rank(group) if world > 1 else 0
        first = int(sum(len(p) for p in parts[:rank]))
        cred_all = np.concatenate(parts)
        hi, lo = ev.make_cred_groups(np.arange(n), cred_all, group_pct)
        mine = np.arange(first, first + n_loc)
        in_hi, in_lo = np.isin(mine, hi), np.isin(mine, lo)
        flags_dev = torch.from_numpy(in_hi.astype(np.uint8) + 2 * in_lo.astype(np.uint8)).to(dev)
        pop_dev = torch.as_tensor(np.asarray(item_pop, dtype=np.int64)).to(dev)
        groups = (len(hi), len(lo), cred_all.astype(np.float64).mean())
    if n_loc:
        ids, _ = ev.topk_device(f_u_local, f_i, users_dev, (graph.samp_indptr, graph.samp_idx), K, precision)
    else:
        ids = torch.zeros(0, K, dtype=torch.int32, device=dev)
    sums, bitmaps = ev.metrics_sums_device(ids, users_dev, te, num_items, ks, pop_dev, total_train, flags_dev,
                                           with_coverage=extra)
    sums, cover = _reduce_metric_sums(sums, bitmaps, num_items, group)
    return ev.metrics_result(Ks, ks, sums, cover, n, num_items, "full", groups)


def _reduce_metric_sums(sums, bitmaps, num_items, group):
    """Per-rank metric sums -> global sums (all-reduce) and, with bitmaps, the global coverage counts (host)."""
    from . import evaluate as ev
    world = _world(group)
    if world > 1:
        dist.all_reduce(sums, group=group)
        if bitmaps is not None:   # NCCL has no bitwise-OR reduction: gather the (small) bitmaps and OR them here
            parts = [torch.empty_like(bitmaps) for _ in range(world)]
            dist.all_gather(parts, bitmaps, group=group)
            for p in parts[1:]:
                parts[0] |= p
            bitmaps = parts[0]
    cover = ev.coverage_counts_device(bitmaps, num_items).cpu().numpy() if bitmaps is not None else None
    return sums.cpu().numpy(), cover


@torch.no_grad()
def evaluate_sampled_sharded(f_u_local, f_i, graph: CredGraph, lo: int, hi: int, train_csr, test_csr, num_items,
                             Ks=(10, 20), n_neg=99, seed=42, on_device=False, item_pop=None, total_train=0, cred=None,
                             group_pct=0.20, group=None):
    """The sampled protocol (1 test positive + n_neg negatives per test user, lightgcn_cu.py:487-546) over user
    shards: every rank scores and ranks the candidate lists of ITS test users against the replicated item table,
    and only metric sums cross ranks.  train_csr / test_csr: host CSRs (indptr, indices) of the WHOLE graph;
    `graph` is the rank's local CredGraph (users [lo, hi)); cred: the GLOBAL credibility vector (None: no
    popularity / credibility metrics).  Candidates: on_device=False draws the reference's PCG64 list over all test
    users -- identical on every rank -- and keeps the rank's rows; on_device=True draws the rank's rows with
    cgx_eval_candidates keyed by their row in the whole list.  Either way each user ranks the candidates the
    single-GPU evaluate_sampled gives it, and the credibility groups are percentiles of the global order."""
    from . import evaluate as ev
    from .graph import user_csr_device
    dev = f_u_local.device
    te_ip = np.asarray(test_csr[0])
    users_all = np.flatnonzero(np.diff(te_ip) > 0).astype(np.int64)
    if users_all.size == 0:
        raise RuntimeError("No users with test interactions.")
    first, last = np.searchsorted(users_all, lo), np.searchsorted(users_all, hi)
    users = users_all[first:last]
    if on_device:
        te_loc = user_csr_device(np.stack([np.repeat(np.arange(hi - lo), np.diff(te_ip[lo:hi + 1])),
                                           np.asarray(test_csr[1])[te_ip[lo]:te_ip[hi]]]), hi - lo, num_items, dev)
        cands_dev = (ev.sampled_candidates_device((graph.samp_indptr, graph.samp_idx), te_loc, users - lo, num_items,
                                                  n_neg, seed, row_base=int(first)) if users.size else None)
    else:
        _, cands = ev.sampled_candidates(train_csr, test_csr, num_items, n_neg, seed)
        cands_dev = torch.from_numpy(np.ascontiguousarray(cands[first:last])).to(dev) if users.size else None
    ks = sorted(set(int(k) for k in Ks))
    extra = item_pop is not None and cred is not None
    pop_dev = flags_dev = groups = None
    if extra:
        hi_g, lo_g = ev.make_cred_groups(users_all, cred, group_pct)
        in_hi, in_lo = np.isin(users, hi_g), np.isin(users, lo_g)
        flags_dev = torch.from_numpy(in_hi.astype(np.uint8) + 2 * in_lo.astype(np.uint8)).to(dev)
        pop_dev = torch.as_tensor(np.asarray(item_pop, dtype=np.int64)).to(dev)
        groups = (len(hi_g), len(lo_g), np.asarray(cred, np.float64)[users_all].mean())
    users_dev = torch.from_numpy(users - lo).to(dev)
    if users.size:
        scores = ev.score_candidates_device(f_u_local, f_i, users_dev, cands_dev)
        ranked = ev.rank_candidates_device(scores, cands_dev)
        gt = cands_dev[:, 0]
    else:
        ranked = torch.zeros(0, 1 + n_neg, dtype=torch.int64, device=dev)
        gt = None
    sums, bitmaps = ev.metrics_sums_device(ranked, users_dev, None, num_items, ks, pop_dev, total_train, flags_dev,
                                           gt_single_dev=gt, with_coverage=extra)
    sums, cover = _reduce_metric_sums(sums, bitmaps, num_items, group)
    return ev.metrics_result(Ks, ks, sums, cover, int(users_all.size), num_items, "sampled(1pos+neg)", groups,
                             extra_keys={"negatives": n_neg})


# ------------------------------------------------------------------------------------------
# the reference's training loop over user shards (train_lightgcn() under torchrun)
# ------------------------------------------------------------------------------------------
def initial_tables(variant: str, num_users: int, num_items: int, emb_dim: int):
    """The initial (user, item) tables of the single-GPU model, drawn from torch's CPU generator in the same order as
    the model's constructor draws them (nn.Embedding's normal_ fill, then xavier_uniform_): RawLightGCN's one
    (U + I) x d table, or the two tables of CredLightGCN / LightGCN."""
    if variant == "raw":
        w = torch.empty(num_users + num_items, emb_dim)
        torch.nn.init.normal_(w)
        torch.nn.init.xavier_uniform_(w)
        return w[:num_users], w[num_users:]
    eu, ei = torch.empty(num_users, emb_dim), torch.empty(num_items, emb_dim)
    torch.nn.init.normal_(eu)
    torch.nn.init.normal_(ei)
    torch.nn.init.xavier_uniform_(eu)
    torch.nn.init.xavier_uniform_(ei)
    return eu, ei


def _gather_users(eu_local: torch.Tensor, bounds, group) -> torch.Tensor:
    """The user shards of all ranks in rank order (every rank takes part; the result is used on rank 0)."""
    world = _world(group)
    if world == 1:
        return eu_local.clone()
    rows = int(max(bounds[r + 1] - bounds[r] for r in range(world)))
    pad = torch.zeros(rows, eu_local.shape[1], dtype=eu_local.dtype, device=eu_local.device)
    pad[: eu_local.shape[0]] = eu_local
    parts = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(parts, pad, group=group)
    return torch.cat([parts[r][: int(bounds[r + 1] - bounds[r])] for r in range(world)])


def train_on_arrays_sharded(train_edges, val_edges, test_edges, num_users, num_items, cred_np, out_dir=None, cfg=None,
                            group=None, on_step=None):
    """train.train_on_arrays over the users of `group`'s ranks (one process per GPU, the current CUDA device): the
    same model, batches and triples as the single-GPU loop -- losses, metrics and tables agree up to the order of
    floating-point sums -- for every cfg.variant.

    Every rank computes the same train users and the same default_rng(cfg.seed) shuffle per epoch and runs
    ceil(n_train / batch_size) steps; the ShardedTrainStep selects each global batch's entries of the rank's users
    on the device (cgx_batch_select), samples the triple of each entry from the stream of its slot in the global
    batch, and divides by the global batch size, so the tail batch needs nothing special.  Evaluation follows
    cfg.eval_mode (full-rank: evaluate_full_ranking_sharded at cfg.score_precision; sampled:
    evaluate_sampled_sharded), with only metric sums crossing ranks.  Prints come from rank 0.  The best-validation
    checkpoint (same file name and keys as the single-GPU loop: the user shards in rank order and the item table)
    is written by rank 0 and restored on every rank before the test evaluation.  on_step(step, epoch, s): optional
    callback after every step (e.g. ShardedTrainStep.last_batch()).
    Returns (state_dict on rank 0 / None on the other ranks, test results -- identical on every rank)."""
    from pathlib import Path

    from . import config
    from . import evaluate as ev
    from .train import _GRAPH_VARIANT, _POPMIX, _print_metrics, evaluate_csr
    cfg = cfg or config.cfg
    variant = cfg.variant
    world = _world(group)
    rank = dist.get_rank(group) if world > 1 else 0
    dev = torch.device("cuda", torch.cuda.current_device())
    say = print if rank == 0 else (lambda *a, **k: None)
    say("Using device:", dev, f"(user-sharded over {world} ranks)")

    train_edges = np.asarray(train_edges)
    U, I = int(num_users), int(num_items)
    deg_u = np.bincount(train_edges[0].astype(np.int64), minlength=U)
    bounds = partition_users(deg_u, world)
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    raw = variant == "raw"
    cred = np.ones(U, dtype=np.float32) if raw else np.asarray(cred_np, dtype=np.float32)
    gl = build_local_graph(shard_edges(train_edges, bounds, rank), hi - lo, I, cred[lo:hi],
                           "cu" if raw else _GRAPH_VARIANT[variant], dev, group)
    rich = variant == "v2"
    item_pop, total_train = ev.compute_item_popularity(train_edges, I) if rich else (None, 0)
    train_users = np.flatnonzero(deg_u > 0)
    if len(train_users) == 0:
        raise RuntimeError("No train users with interactions. Check your threshold/split.")

    pop_fair = None
    if variant == "cu" and cfg.lambda_fair:
        deg_i = gl.deg_i_float()
        pop_fair = (deg_i / max(float(deg_i.max()), 1.0)).astype(np.float32)      # lightgcn_cu.py:583
    popmix = variant in _POPMIX
    if popmix:
        item_deg = gl.deg_i.cpu().numpy().astype(np.float64)
        p10, p50, p90, p99 = np.percentile(item_deg, [10, 50, 90, 99])
        say(f"[NEG-E] item_deg percentiles: p10={p10:.0f} p50={p50:.0f} p90={p90:.0f} p99={p99:.0f} "
            f"max={item_deg.max():.0f}")
        say(f"[NEG-E] mix_pop={cfg.neg_mix_pop} gamma={cfg.neg_pop_gamma}")
    eu0, ei0 = initial_tables(variant, U, I, cfg.emb_dim)
    step = ShardedTrainStep(gl, eu0[lo:hi].to(dev), ei0.to(dev), cfg.num_layers,
                            "jacobi" if variant in ("cu", "raw") else "gs", lr=cfg.lr,
                            reg_weight=cfg.lambda_reg if variant == "cu" else cfg.reg,
                            mix_pop=cfg.neg_mix_pop if popmix else None, gamma=cfg.neg_pop_gamma,
                            max_tries=cfg.neg_max_tries, seed=cfg.seed, group=group, exchange="auto",
                            max_batch=cfg.batch_size, fair_weight=cfg.lambda_fair if variant == "cu" else 0.0,
                            pop=pop_fair)
    del eu0, ei0
    n_train, B = len(train_users), int(cfg.batch_size)
    steps = -(-n_train // B)
    step.plan_epochs(n_train, lo, hi)

    full = cfg.eval_mode == "full" and variant != "cu"
    train_csr_host = None if full else evaluate_csr(train_edges, U, I, dev)    # the reference's candidate draw

    def run_eval(edges):
        f_u, f_i = step.prop.forward(step.eu.data, step.ei.data)
        f_u, f_i = f_u.contiguous(), f_i.contiguous()
        if full:
            return evaluate_full_ranking_sharded(f_u, f_i, gl, shard_edges(np.asarray(edges), bounds, rank), I,
                                                 cfg.Ks, item_pop, total_train, cred[lo:hi] if rich else None,
                                                 cfg.cred_group_pct, group, cfg.score_precision)
        return evaluate_sampled_sharded(f_u, f_i, gl, lo, hi, train_csr_host, evaluate_csr(edges, U, I, dev), I, cfg.Ks,
                                        cfg.sampled_negatives, cfg.seed, cfg.sampled_eval_on_device, item_pop,
                                        total_train, cred if rich else None, cfg.cred_group_pct, group)

    def state_dict():
        eu_all = _gather_users(step.eu.data, bounds, group)
        if rank != 0:
            return None
        if raw:
            return {"emb.weight": torch.cat([eu_all, step.ei.data.clone()])}
        return {"user_emb.weight": eu_all, "item_emb.weight": step.ei.data.clone()}

    best_val, best = -1.0, None
    best_path = None
    if out_dir is not None:
        best_path = Path(out_dir) / "model" / ("best_model_cred.pt" if variant == "cu" else "best_model.pt")
        if rank == 0:
            best_path.parent.mkdir(parents=True, exist_ok=True)

    rng = np.random.default_rng(cfg.seed)
    captured = False
    for epoch in range(1, cfg.epochs + 1):
        rng.shuffle(train_users)
        step.begin_epoch(train_users)
        if not captured and isinstance(step.ex, P2PExchange):
            step.capture(B, selected=True)       # every rank: the exchange kind is agreed on by all ranks
            captured = True
        losses = []
        for s in range(steps):
            losses.append(step.step_selected().clone())
            if on_step is not None:
                on_step(step, epoch, s)
        avg_loss = float(torch.stack(losses).mean().item()) if losses else 0.0
        say(f"Epoch {epoch:03d} | loss={avg_loss:.6f}" if variant == "cu" else f"Epoch {epoch:02d} | loss={avg_loss:.6f}")

        if epoch % cfg.eval_every == 0:
            val_res = run_eval(val_edges)
            selK = max(cfg.Ks)
            if rank == 0:
                _print_metrics("VAL metrics:", val_res, cfg.Ks, rich)
            if val_res[selK]["recall"] > best_val:
                best_val = val_res[selK]["recall"]
                best = (step.eu.data.clone(), step.ei.data.clone())
                sd = state_dict()
                if best_path is not None and rank == 0:
                    torch.save(sd, best_path)
                    print(f"  ✅ Saved best model to {best_path} (val Recall@{selK}={best_val:.4f})")
    step.check()
    if best is not None:
        step.eu.data.copy_(best[0])
        step.ei.data.copy_(best[1])
    test_res = run_eval(test_edges)
    if rank == 0:
        _print_metrics("\nTEST metrics:", test_res, cfg.Ks, rich)
    sd = state_dict()
    if world > 1:
        dist.barrier(group=group)
    step.close()
    return sd, test_res


# ------------------------------------------------------------------------------------------
# parity of the sharded path against the single-GPU path (tests/test_gpu_multi.py, bench.py --gpus N)
# ------------------------------------------------------------------------------------------
@torch.no_grad()
def parity_vs_single_gpu(rank: int, world: int, dev, variant="v2", order="gs", exchange=None, d=64, K=3,
                         batch=2048, graph_kwargs=None):
    """max relative error of the user-sharded forward / loss / gradients over `world` ranks against the single-GPU
    path on the WHOLE graph (a C1-shaped graph split by partition_users), for one injected triple list.  Every rank
    computes the single-GPU truth itself; the result is the maximum over ranks and quantities."""
    from . import synth
    from .graph import build_graph
    from .model import CredLightGCN, LightGCN, TrainStep
    sg = synth.make_graph("C1", **(graph_kwargs or dict(duplicate_edges=100)))
    U, I = sg.num_users, sg.num_items
    bounds = partition_users(np.bincount(sg.train_edges[0], minlength=U), world)
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    users, pos, neg = synth.make_triples(sg, batch)
    mine = (users >= lo) & (users < hi)
    torch.manual_seed(0)
    eu = torch.nn.init.xavier_uniform_(torch.empty(U, d))
    ei = torch.nn.init.xavier_uniform_(torch.empty(I, d))
    gl = build_local_graph(shard_edges(sg.train_edges, bounds, rank), hi - lo, I, sg.cred[lo:hi], variant, dev)
    ex = exchange or CollectiveExchange()
    prop = ShardedPropagation(CudaBackend(gl), K, order, exchange=ex)
    if hasattr(ex, "begin_step"):
        ex.begin_step()
    eu_l, ei_d = eu[lo:hi].to(dev).contiguous(), ei.to(dev)
    f_u, f_i = prop.forward(eu_l, ei_d)
    f_u, f_i = f_u.clone(), f_i.clone()
    g_u = torch.zeros_like(eu_l)
    gi2 = ex.partial_buffer((2, I, d), dev).zero_()
    ego_u = torch.zeros_like(eu_l)
    ul = torch.as_tensor(users[mine] - lo, device=dev)
    if ul.numel() == 0:            # bpr_fused needs >= 1 triple: contribute a zero-weight dummy via batch_total only
        loss = torch.zeros(1, device=dev)
    else:
        loss, _, _, ego_rows, ego_coef = bpr_fused(gl, f_u, f_i, eu_l, ei_d, ul, torch.as_tensor(pos[mine], device=dev),
                                                   torch.as_tensor(neg[mine], device=dev), 1e-4, 0.0, None, g_u, gi2[0],
                                                   batch_total=len(users))
        apply_ego(gl, ego_rows, ego_coef, eu_l, ei_d, ego_u, gi2[1])
    gi2 = ex.reduce(gi2).clone()
    loss = all_reduce_sum(loss.clone())
    d_u, d_i = prop.backward(g_u, gi2[0])
    d_u, d_i = d_u + ego_u, d_i + gi2[1]
    # single-GPU truth
    gr = build_graph(sg.train_edges, U, I, sg.cred, variant, dev)
    Net = CredLightGCN if order == "jacobi" else LightGCN
    ops = (gr.operator("C"), gr.operator("A")) if order == "jacobi" else (gr.operator("A"), gr.operator("C"))
    net = Net(U, I, d, K, *ops)
    net.load_state_dict({"user_emb.weight": eu, "item_emb.weight": ei})
    net = net.to(dev)
    st = TrainStep(net, reg_weight=1e-4)
    want = st.forward_backward(users, pos, neg)
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))
    errs = dict(loss=abs(float(loss.item()) - float(want.item())) / abs(float(want.item())),
                f_i=rel(f_i, st.f_i), d_i=rel(d_i, net.item_emb.weight.grad),
                deg_i=float((gl.deg_i != gr.deg_i).sum().item()))
    if hi > lo:
        errs["f_u"] = rel(f_u, st.f_u[lo:hi])
        errs["d_u"] = rel(d_u, net.user_emb.weight.grad[lo:hi])
    # the whole sharded training step (compact loss-gradient all-gather, row bookkeeping, Adam) on the same triples:
    # Adam's first-moment buffers after one step are 0.1 x the gradients the step used
    if hasattr(ex, "allgather"):         # (every rank of the C1 split owns users and triples; all ranks must take part)
        assert hi > lo and int(mine.sum()) > 0, "parity graph too small for this many ranks"
        st.opt.step()
        for form, compact in (("compact", True), ("dense", False)):
            ShardedTrainStep.force_compact = compact
            try:
                sh = ShardedTrainStep(gl, eu[lo:hi].to(dev), ei.to(dev), K, order, reg_weight=1e-4,
                                      mix_pop=None if variant == "cu" else 0.7, exchange=ex, max_batch=batch)
            finally:
                ShardedTrainStep.force_compact = None
            if not compact and isinstance(ex, P2PExchange) and ex.region < 4 * (2 * ei.numel() + 4):
                continue                  # the caller's exchange has no room for the dense form
            loss2 = sh(ul, batch_total=len(users), triples=(pos[mine], neg[mine]))
            errs[f"step_{form}_loss"] = abs(float(loss2.item()) - float(want.item())) / abs(float(want.item()))
            errs[f"step_{form}_m_u"] = rel(sh.opt.m[0], st.opt.m[0][lo:hi])
            errs[f"step_{form}_m_i"] = rel(sh.opt.m[1], st.opt.m[1])
            if compact:
                errs["step_tables_clean"] = float(sh.g_u.abs().max().item() + sh.g_i.abs().max().item()
                                                  + sh.gi_local.abs().max().item() + sh.nz_u.sum().item())
    worst = torch.tensor([max(errs.values())], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)
    return float(worst.item()), errs, (f_u, f_i, d_u, d_i)


# ------------------------------------------------------------------------------------------
# bench.py --gpus N (N > 1): weak scaling, one user shard of the workload per rank (C5: ONE graph split over the ranks)
# ------------------------------------------------------------------------------------------
def bench_main(args, rank: int, world: int, dev: torch.device):
    import pathlib
    import sys
    from . import synth
    root = pathlib.Path(__file__).resolve().parents[1]
    name = args.workload or "C4"
    shp = synth.SHAPES[name]
    strong = name == "C5"
    # experiment switches of this benchmark command (the classes themselves read no environment):
    #   CGX_EXCHANGE=auto|p2p|nccl, CGX_P2P_BACKING=ipc|symm|auto, CGX_P2P_PUSH=0|1, CGX_P2P_NVLS=0|1
    ex_kind = os.environ.get("CGX_EXCHANGE", "auto")
    if "CGX_P2P_BACKING" in os.environ:
        P2PExchange.DEFAULT_BACKING = os.environ["CGX_P2P_BACKING"]
    if "CGX_P2P_PUSH" in os.environ:
        P2PExchange.force_push = os.environ["CGX_P2P_PUSH"] == "1"
    if "CGX_P2P_NVLS" in os.environ:
        P2PExchange.use_nvls = os.environ["CGX_P2P_NVLS"] == "1"

    # ---- parity of this very exchange against the single-GPU path, before anything is timed ----
    par_ex = None
    if ex_kind in ("p2p", "auto"):
        try:
            par_ex = P2PExchange(2 * synth.SHAPES["C1"]["num_items"] * 64 + 4, dev,
                                 gather_floats=ShardedTrainStep._block_floats(2048, 64))
        except _lib.CgxError:
            par_ex = None
    parity, parity_detail, _ = parity_vs_single_gpu(rank, world, dev, "v2", "gs", exchange=par_ex)
    if par_ex is not None:
        par_ex.check()
        dist.barrier()
        par_ex.close()

    if strong:
        # BASELINE configs[4]: THE 50M x 10M x 1B-edge graph.  Every rank generates the same seeded graph on its own
        # GPU, partition_users cuts the users into `world` contiguous ranges of equal non-zeros, and the rank keeps
        # the edges (ids rebased), credibilities and test edges of its range.
        full = synth.make_graph_device("C5", dev)
        deg_all = torch.bincount(full.train_edges[0].to(torch.int64), minlength=full.num_users)
        bounds = partition_users(deg_all.cpu().numpy(), world)
        lo, hi = int(bounds[rank]), int(bounds[rank + 1])
        del deg_all

        def mine(e):
            keep = (e[0] >= lo) & (e[0] < hi)
            out = e[:, keep].clone()
            out[0] -= lo
            return out

        sg = synth.SynthGraph(name="C5", num_users=hi - lo, num_items=full.num_items, train_edges=mine(full.train_edges),
                              val_edges=full.val_edges[:, :0], test_edges=mine(full.test_edges),
                              cred=full.cred[lo:hi].contiguous(), is_fake=full.is_fake[lo:hi], meta=dict(full.meta))
        del full
        torch.cuda.empty_cache()
    elif name == "C4":
        sg = synth.make_graph_device(name, dev, seed=20240 + 1000 * (rank + 1), item_seed=20242)
    else:
        sg = synth.make_graph(name, seed=20240 + 1000 * (rank + 1), item_seed=20242)
    U, I, d, K = sg.num_users, sg.num_items, shp["emb_dim"], shp["num_layers"]
    E_local = int(sg.train_edges.shape[1])
    gr = build_local_graph(sg.train_edges, U, I, sg.cred, shp["variant"], dev)
    torch.manual_seed(42)
    item_emb = torch.nn.init.xavier_uniform_(torch.empty(I, d, device=dev))      # identical on every rank
    torch.manual_seed(1000 + rank)
    user_emb = torch.nn.init.xavier_uniform_(torch.empty(U, d, device=dev))
    n_eval = int(os.environ.get("CGX_BENCH_EVAL_USERS", "0"))   # per rank; 0 = no evaluation leg
    test_edges = None
    if n_eval:
        te = torch.as_tensor(sg.test_edges, device=dev)
        test_edges = te[:, te[0] < n_eval].contiguous()
        del te
    del sg
    torch.cuda.empty_cache()
    step = ShardedTrainStep(gr, user_emb, item_emb, K, shp["order"], mix_pop=None if shp["variant"] == "cu" else 0.7,
                            exchange=ex_kind, max_batch=args.batch)
    train_users = torch.nonzero(gr.deg_u > 0).reshape(-1).cpu().numpy()
    np.random.default_rng(42 + rank).shuffle(train_users)
    nb = min(len(train_users) // args.batch, 64)
    host_batches = [train_users[s * args.batch:(s + 1) * args.batch] for s in range(max(nb, 1))]
    dev_batches = [torch.from_numpy(b).to(dev) for b in host_batches]
    pinned = [torch.from_numpy(b).pin_memory() for b in host_batches]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    graphed = isinstance(step.ex, P2PExchange) and os.environ.get("CGX_SHARDED_GRAPH", "1") == "1"
    if graphed:
        try:
            step.capture(args.batch)
        except Exception as e:          # noqa: BLE001
            graphed, step._graph = False, None
            print(f"[bench] rank {rank}: CUDA-graph capture failed ({type(e).__name__}: {e}); eager launches",
                  file=sys.stderr)
        flag = torch.tensor([1.0 if graphed else 0.0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if flag.item() == 0:            # every rank must take the same path
            graphed, step._graph = False, None
    c0 = lib().cgx_launch_count()
    step(dev_batches[0])                         # one eager step: how many kernels of the library a step launches
    launches_per_step = lib().cgx_launch_count() - c0
    for s in range(max(args.warmup, 3)):
        step.step(dev_batches[s % len(dev_batches)])
    clocks = None
    if rank == 0:                                # nvidia-smi clocks / throttle reasons of rank 0's GPU during the timed steps
        sys.path.insert(0, str(root))
        import bench as _bench
        clocks = _bench.ClockSampler(dev.index if dev.index is not None else 0)
        clocks.__enter__()
    torch.cuda.synchronize()
    dist.barrier()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    for s in range(args.steps):
        flush.fill_(s & 0xff)
        starts[s].record()
        step.step(dev_batches[s % len(dev_batches)])
        ends[s].record()
    torch.cuda.synchronize()
    dist.barrier()
    total_ms = torch.tensor([sum(a.elapsed_time(b) for a, b in zip(starts, ends))], device=dev)
    dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)

    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    loss_host = 0.0
    for s in range(args.steps):
        loss_host = float(step.step(pinned[s % len(pinned)]).item())
    torch.cuda.synchronize()
    if clocks is not None:
        clocks.__exit__(None, None, None)
    e2e = torch.tensor([1e3 * (time.perf_counter() - t0)], device=dev)
    dist.all_reduce(e2e, op=dist.ReduceOp.MAX)
    step.check()                                 # no exchange gave up on a peer

    # ---- where the step's time goes: the propagation alone (products + exchanges), and one exchange alone ----
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    prop_f, prop_b = [], []
    g_u = torch.zeros_like(step.eu.data)
    g_i = torch.zeros_like(step.ei.data)
    g_u[:64] = 1e-3
    for _ in range(3):
        if hasattr(step.ex, "begin_step"):
            step.ex.begin_step()
        dist.barrier()
        ev[0].record()
        step.prop.forward(step.eu.data, step.ei.data)
        ev[1].record()
        step.prop.backward(g_u, g_i)
        ev[2].record()
        torch.cuda.synchronize()
        prop_f.append(ev[0].elapsed_time(ev[1]))
        prop_b.append(ev[1].elapsed_time(ev[2]))
    del g_u
    xs = []
    buf = step.ex.partial_buffer(tuple(step.ei.shape), dev)
    if hasattr(step.ex, "begin_step"):
        step.ex.begin_step()
    for _ in range(4):
        dist.barrier()
        buf = step.ex.partial_buffer(tuple(step.ei.shape), dev)
        ev[0].record()
        step.ex.reduce(buf)
        ev[1].record()
        torch.cuda.synchronize()
        xs.append(ev[0].elapsed_time(ev[1]))
    ps = [0.0]
    pushed = step.prop._push()
    if pushed:
        # the pushed form's own part (barrier, local reduce of the staged rows, delivery, barrier) without a product
        ps = []
        for _ in range(4):
            step.ex.begin_step()
            dist.barrier()
            ev[0].record()
            step.ex.exchange_pushed(tuple(step.ei.shape), lambda *a: None)
            ev[1].record()
            torch.cuda.synchronize()
            ps.append(ev[0].elapsed_time(ev[1]))
        ps = ps[1:]
    t3 = torch.tensor([min(prop_f), min(prop_b), min(xs[1:]), min(ps)], device=dev)
    dist.all_reduce(t3, op=dist.ReduceOp.MAX)
    prop_f_ms, prop_b_ms, xchg_ms, push_ms = (float(v) for v in t3.tolist())
    edges = torch.tensor([E_local], dtype=torch.int64, device=dev)
    dist.all_reduce(edges)
    nnz_t = torch.tensor([gr.nnz], dtype=torch.int64, device=dev)
    tu = torch.tensor([len(train_users)], dtype=torch.int64, device=dev)
    dist.all_reduce(tu, op=dist.ReduceOp.MAX)
    if rank == 0:
        ms = float(total_ms.item()) / args.steps
        e2e_ms = float(e2e.item()) / args.steps
        E = int(edges.item())
        hbm_peak, peak_src = _bench.peaks()
        nvl_peak = 770.0          # GB/s per direction per GPU, measured peer copy (B200_PROFILING.md)
        r = 4 * d
        table_bytes = I * r
        # per rank: what its own products move (gather model / compulsory) and what crosses NVLink
        gather = _bench.gather_model_bytes(U, I, int(nnz_t.item()), d, K)
        comp = _bench.compulsory_bytes(U, I, int(nnz_t.item()), d, K)
        traffic, traffic_src = _bench.traffic_per_step(name)
        prop_ms = prop_f_ms + prop_b_ms
        n_x = 2 * K              # item-table exchanges (the loss gradient travels as one small all-gather)
        link_bytes = (world - 1) / world * table_bytes          # per direction, per rank, per exchange
        steps_per_epoch = -(-int(tu.item()) // args.batch)
        line = {
            "metric": "edges/sec (3-layer cred-weighted LightGCN fwd+bwd)", "value": E / (ms / 1e3), "unit": "edges/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": _bench.workload_config(name, args.batch, world),
            "train_edges": E, "users_per_rank": U, "items": I,
            "e2e": {"value": E / (e2e_ms / 1e3), "unit": "edges/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(host_batches[0].nbytes) * world, "d2h_bytes_per_step": 4 * world,
                    "api": "ShardedTrainStep.step(pinned_host_users) + loss.item() on every rank"},
            "gpu_launches": int(launches_per_step * args.steps),
            "gpu_launches_note": f"{launches_per_step} kernels of libcredgcn.so per step and rank",
            "loss": loss_host,
            "collectives_per_step": f"{2 * K} item-table exchanges + 1 all-gather of the compact loss gradient",
            "cuda_graph": graphed, "exchange": type(step.ex).__name__ +
            (" (rows pushed from the SpMM epilogue + local reduce)" if pushed else
             " (NVLS: multimem.ld_reduce / multimem.st through the switch)" if
             (getattr(step.ex, "nvls_enabled", lambda n: False)(4 * step.ei.numel())) else
             " (pull kernel)" if isinstance(step.ex, P2PExchange) else ""),
            "parity_vs_1gpu": parity, "parity_vs_1gpu_detail": {k: float(v) for k, v in parity_detail.items()},
            "roofline": {
                "bound": "hbm + nvlink", "peak": hbm_peak, "unit": "GB/s", "peak_source": peak_src,
                "propagate_ms": {"fwd": prop_f_ms, "bwd": prop_b_ms,
                                 "note": "products + exchanges of one step, eager launches, max over ranks"},
                "frac_dram_bytes": (traffic / (prop_ms / 1e3) / 1e9 / hbm_peak) if traffic else None,
                "traffic_source": traffic_src,
                "frac_gather_model": gather / (prop_ms / 1e3) / 1e9 / hbm_peak,
                "frac_compulsory": comp / (prop_ms / 1e3) / 1e9 / hbm_peak,
                "frac": (traffic if traffic else gather) / (prop_ms / 1e3) / 1e9 / hbm_peak,
                "achieved": (traffic if traffic else gather) / (prop_ms / 1e3) / 1e9,
                "nvlink": {"bytes_per_exchange_per_direction": link_bytes, "exchange_ms": xchg_ms,
                           "achieved_gbs": link_bytes / (xchg_ms / 1e3) / 1e9, "peak_gbs": nvl_peak,
                           "frac": link_bytes / (xchg_ms / 1e3) / 1e9 / nvl_peak,
                           "exchanges_per_step": n_x, "exchange_share_of_step": n_x * xchg_ms / ms,
                           "pushed_form_reduce_deliver_ms": push_ms if push_ms > 0 else None,
                           "note": "exchange_ms: one item-table exchange timed alone in its stand-alone (pull / "
                                   "collective) form, max over ranks; pushed_form_reduce_deliver_ms: what the pushed "
                                   "form adds after the product (its reduce-scatter half rides on the SpMM epilogue)"},
            },
            "steps_per_epoch": steps_per_epoch, "epoch_ms": ms * steps_per_epoch,
            "epoch_ms_kind": f"extrapolated: {steps_per_epoch} steps x the timed mean step",
            "clocks": clocks.summary(),
        }
        print(json.dumps(line))
    if n_eval:      # user-sharded full-rank evaluation of the first n_eval users of every shard (second JSON line)
        with torch.no_grad():
            f_u, f_i = step.prop.forward(step.eu.detach(), step.ei.detach())
        f_u, f_i = f_u.contiguous(), f_i.contiguous()
        res = None
        times = []
        for _ in range(2):
            torch.cuda.synchronize()
            dist.barrier()
            t0 = time.perf_counter()
            res = evaluate_full_ranking_sharded(f_u, f_i, gr, test_edges, I, (10, 20), precision="bf16x3")
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        t = torch.tensor([times[-1]], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if rank == 0:
            n = res[20]["users_eval"]
            sec = float(t.item())
            print(json.dumps({"eval": "user-sharded full-rank Recall/NDCG@{10,20}, tcgen05 scores (bf16x3), device metrics",
                              "users_eval": n, "items": I, "emb_dim": d, "n_gpus": world, "seconds": sec,
                              "users_per_s": n / sec, "useful_TFLOPs_per_gpu": 2.0 * n * I * d / sec / world / 1e12,
                              "recall@20": res[20]["recall"], "ndcg@20": res[20]["ndcg"],
                              "projected_seconds_all_users": sec * (U * world * 0.85) / max(n, 1)}))
    dist.barrier()
    step.close()
    dist.destroy_process_group()
