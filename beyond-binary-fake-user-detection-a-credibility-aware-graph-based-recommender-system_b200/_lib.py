"""ctypes binding of libcredgcn.so (include/credgcn.h).  No CPU fallback: a missing library or a
non-CUDA tensor is an error, raised loudly."""
from __future__ import annotations

import ctypes as C
import os
import pathlib
import subprocess

import torch

PKG_DIR = pathlib.Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "libcredgcn.so"
CSRC_DIR = PKG_DIR / "csrc"

VARIANTS = {"cu": 0, "v2": 1, "da": 2}
ORDERS = {"jacobi": 0, "gs": 1}
PRECISIONS = {"fp32": 0, "bf16x3": 1, "bf16": 2}
# cgx_option (include/credgcn.h).  The library reads no environment variables; for experiments this binding maps
# CGX_OPT_<NAME>=<int> onto cgx_set_option when the library is loaded.
OPTIONS = {"L2_TABLE_BYTES": 0, "SPARSE_FIRST_ADJOINT": 1, "PDL": 2, "P2P_ONESHOT_MAX": 3, "P2P_TIMING": 4,
           "P2P_TIMEOUT_MS": 5, "EVAL_DEBUG": 6, "HOT_ROWS": 7, "EVAL_GROUPS": 8,
           "TOPK_CHUNK_USERS": 9}
LONG_ROW = 256
CHUNK = 256


class CgxError(RuntimeError):
    pass


class CsrStruct(C.Structure):
    """struct cgx_csr"""
    _fields_ = [
        ("n_rows", C.c_int32), ("n_cols", C.c_int32), ("nnz", C.c_int64),
        ("indptr", C.c_void_p), ("idx", C.c_void_p), ("val_fwd", C.c_void_p), ("val_bwd", C.c_void_p),
        ("perm", C.c_void_p), ("n_long", C.c_int32), ("n_chunks", C.c_int32),
        ("chunk_ptr", C.c_void_p), ("chunk_row", C.c_void_p),
        ("n_huge", C.c_int32), ("reserved_", C.c_int32), ("arrive", C.c_void_p), ("work", C.c_void_p),
        ("idx_hint", C.c_void_p),
    ]


_P = C.c_void_p
_CSR = C.POINTER(CsrStruct)
_SIGNATURES = {
    "cgx_last_error": (C.c_char_p, []),
    "cgx_version": (C.c_int, []),
    "cgx_launch_count": (C.c_uint64, []),
    "cgx_emb_dim_supported": (C.c_int, [C.c_int32]),
    "cgx_set_option": (C.c_int, [C.c_int, C.c_int64, C.POINTER(C.c_int64)]),
    "cgx_get_option": (C.c_int64, [C.c_int]),
    "cgx_hot_hints_workspace_bytes": (C.c_size_t, [C.c_int32]),
    "cgx_hot_hints": (C.c_int, [_P, C.c_int64, C.c_int32, _P, C.c_int32, _P, _P, C.c_size_t, _P]),
    "cgx_comm_status": (C.c_int, [_P, C.c_size_t, C.c_int, C.POINTER(C.c_uint32)]),
    "cgx_graph_build_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32, C.c_int32]),
    "cgx_graph_build": (C.c_int, [_P, _P, C.c_int64, C.c_int32, C.c_int32, _P, C.c_int, _P, _P, _P, _P, _P, _P,
                                  _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int, _P, C.c_size_t, _P]),
    "cgx_user_csr": (C.c_int, [_P, _P, C.c_int64, C.c_int32, C.c_int32, _P, _P, _P, C.c_size_t, _P]),
    "cgx_row_schedule_workspace_bytes": (C.c_size_t, [C.c_int32]),
    "cgx_row_schedule": (C.c_int, [_P, C.c_int32, _P, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                   C.POINTER(C.c_int32), _P, C.c_size_t, _P]),
    "cgx_row_schedule_chunks": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, C.c_size_t, _P]),
    "cgx_row_schedule_work": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "cgx_spmm_workspace_bytes": (C.c_size_t, [_CSR, C.c_int32]),
    "cgx_spmm": (C.c_int, [_CSR, C.c_int, C.c_int32, _P, _P, _P, _P, C.c_float, _P, C.c_size_t, _P]),
    "cgx_spmm_sparse_rows": (C.c_int, [_CSR, C.c_int, C.c_int32, _P, _P, _P, _P, _P, C.c_float, _P, C.c_size_t, _P]),
    "cgx_row_flags": (C.c_int, [_P, C.c_int64, C.c_int32, _P, _P]),
    "cgx_spmm_ex": (C.c_int, [_CSR, C.c_int, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_float, _P, C.c_size_t, _P]),
    "cgx_spmm_set_l2_table_bytes": (C.c_int64, [C.c_int64]),
    "cgx_propagate_workspace_bytes": (C.c_size_t, [_CSR, _CSR, C.c_int32]),
    "cgx_propagate_workspace_bytes_for": (C.c_size_t, [_CSR, _CSR, C.c_int32, C.c_int]),
    "cgx_propagate_fwd": (C.c_int, [_CSR, _CSR, C.c_int, C.c_int32, C.c_int32, _P, _P, _P, _P, _P,
                                    C.c_size_t, _P]),
    "cgx_propagate_fwd_layers": (C.c_int, [_CSR, _CSR, C.c_int, C.c_int32, C.c_int32, _P, _P, _P, _P, C.c_int32,
                                           C.c_int32, C.c_int, _P, _P, _P, C.c_int64, _P, _P, _P, C.c_size_t, _P]),
    "cgx_propagate_bwd": (C.c_int, [_CSR, _CSR, C.c_int, C.c_int32, C.c_int32, _P, _P, _P, _P, _P,
                                    C.c_size_t, _P]),
    "cgx_propagate_bwd_flagged": (C.c_int, [_CSR, _CSR, C.c_int, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P,
                                            C.c_size_t, _P]),
    "cgx_propagate_bwd_frontier": (C.c_int, [_CSR, _CSR, C.c_int, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P,
                                             _P, _P, C.c_size_t, _P]),
    "cgx_batch_frontier": (C.c_int, [_CSR, _P, _P, _P, C.c_int64, _P, _P, _P, _P, _P]),
    "cgx_bpr_mark_rows": (C.c_int, [_P, C.c_int64, C.c_int32, _P, _P, _P]),
    "cgx_bpr_clear_rows": (C.c_int, [_P, C.c_int64, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    "cgx_bpr_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32, C.c_int32]),
    "cgx_bpr_plan_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "cgx_bpr_plan": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, C.c_int32, _P, _P, C.c_size_t, _P, _P]),
    "cgx_bpr_fwd_bwd": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, _P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P,
                                  _P, _P,
                                  C.c_float, C.c_float, _P, _P, _P, _P, _P, _P, C.c_size_t, _P, _P, _P]),
    "cgx_bpr_apply_ego": (C.c_int, [_P, _P, C.c_int64, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    "cgx_sampler_build_workspace_bytes": (C.c_size_t, [C.c_int32]),
    "cgx_sampler_build": (C.c_int, [_P, C.c_int32, C.c_double, _P, _P, _P, _P, _P, _P, C.c_size_t, _P]),
    "cgx_sample_triples": (C.c_int, [_P, C.c_int64, _P, _P, C.c_int32, _P, _P, _P, _P, _P, C.c_float,
                                     C.c_int32, C.c_uint64, C.c_uint64, _P, _P, _P, _P, _P, _P]),
    "cgx_batch_select": (C.c_int, [_P, C.c_int64, _P, C.c_int64, C.c_int64, C.c_int64, _P, _P, _P, _P, _P]),
    "cgx_tick": (C.c_int, [_P, _P]),
    "cgx_adam_step": (C.c_int, [_P, _P, _P, _P, C.c_int64, _P, _P, _P, _P, C.c_int64, C.c_float, C.c_float,
                                C.c_float, C.c_float, _P, C.c_int64, _P]),
    "cgx_comm_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "cgx_comm_free": (C.c_int, [_P]),
    "cgx_comm_ipc_handle": (C.c_int, [_P, _P]),
    "cgx_comm_ipc_open": (C.c_int, [_P, C.POINTER(C.c_void_p)]),
    "cgx_comm_ipc_close": (C.c_int, [_P]),
    "cgx_comm_allreduce": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_void_p), C.c_size_t, C.c_size_t, C.c_size_t,
                                     C.c_int64, _P, _P]),
    "cgx_comm_allgather": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_void_p), _P, C.c_size_t, C.c_size_t, C.c_int64,
                                     _P, _P]),
    "cgx_comm_allreduce_nvls": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_void_p), _P, C.c_size_t, C.c_size_t,
                                          C.c_size_t, C.c_int64, _P, _P]),
    "cgx_comm_timing": (C.c_int, [_P]),
    "cgx_spmm_set_push_peers": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "cgx_spmm_push": (C.c_int, [_CSR, C.c_int, C.c_int32, _P, _P, C.c_size_t, C.c_int, C.c_int, C.c_int32, _P,
                                C.c_size_t, _P]),
    "cgx_comm_allreduce_pushed": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_void_p), C.c_size_t, C.c_size_t,
                                            C.c_size_t, C.c_int64, C.c_int32, C.c_int32, _P, _P]),
    "cgx_eval_topk_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int]),
    "cgx_eval_topk": (C.c_int, [_P, C.c_int64, _P, _P, C.c_int32, C.c_int32, _P, _P, C.c_int32, C.c_int, _P,
                                _P, _P, C.c_size_t, _P]),
    "cgx_score_candidates": (C.c_int, [_P, _P, C.c_int64, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "cgx_eval_candidates": (C.c_int, [_P, C.c_int64, _P, _P, _P, _P, C.c_int32, C.c_int32, C.c_uint64, _P, _P,
                                      C.c_int64]),
    "cgx_rank_candidates": (C.c_int, [_P, _P, C.c_int64, C.c_int32, _P, _P]),
    "cgx_eval_topk_uses_tensor_cores": (C.c_int, [C.c_int32, C.c_int32, C.c_int]),
    "cgx_eval_metrics_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32]),
    "cgx_eval_metrics": (C.c_int, [_P, C.c_int64, C.c_int32, _P, _P, _P, _P, C.c_int32, _P, C.c_int32, _P, C.c_int64,
                                   _P, _P, _P, _P, C.c_size_t, _P]),
    "cgx_eval_coverage": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P]),
}
EXPORTED = tuple(_SIGNATURES)

_lib = None


def build_library(verbose: bool = False) -> pathlib.Path:
    """Compile csrc/*.cu for sm_100a into libcredgcn.so (nvcc cross-compiles without a GPU)."""
    out = subprocess.run(["make", "-C", str(CSRC_DIR), "-j8"], capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout[-4000:], out.stderr[-4000:])
    if out.returncode != 0:
        raise CgxError("building libcredgcn.so failed (see output above)")
    return LIB_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise CgxError(
                f"{LIB_PATH} is missing: the sm_100a extension has not been built. Run "
                f"`python -c 'import __graft_entry__ as g; g.build()'` (or `make -C {CSRC_DIR}`). "
                "There is no CPU fallback.")
        handle = C.CDLL(str(LIB_PATH))
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)        # AttributeError here = header/library drift: fail loudly
            fn.restype, fn.argtypes = res, args
        _lib = handle
        for name, key in OPTIONS.items():
            env = os.environ.get(f"CGX_OPT_{name}")
            if env is not None:
                handle.cgx_set_option(key, int(env), None)
    return _lib


def set_option(name: str, value: int) -> int:
    """cgx_set_option by name; returns the previous value (negative value = restore the default)."""
    prev = C.c_int64(0)
    check(lib().cgx_set_option(OPTIONS[name], int(value), C.byref(prev)))
    return int(prev.value)


def get_option(name: str) -> int:
    return int(lib().cgx_get_option(OPTIONS[name]))


def check(status: int) -> None:
    if status != 0:
        raise CgxError(f"libcredgcn error {status}: {lib().cgx_last_error().decode()}")


def ptr(t: torch.Tensor | None):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise CgxError("credgcn ops need CUDA tensors: there is no CPU fallback")
    if not t.is_contiguous():
        raise CgxError("credgcn ops need contiguous tensors")
    return C.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def workspace(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
