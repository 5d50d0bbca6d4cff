"""ctypes binding of libhgr.so (include/hgr.h).  No CPU fallback: a missing or broken library raises."""
from __future__ import annotations

import ctypes as C
import os

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "libhgr.so")

HGR_MAX_ADDENDS = 8
HGR_MAX_GATHER = 8


class HgrError(RuntimeError):
    pass


class CsrDesc(C.Structure):
    """hgr_csr_t"""
    _fields_ = [
        ("n_rows", C.c_int32), ("n_cols", C.c_int32), ("nnz", C.c_int64),
        ("indptr", C.c_void_p), ("indices", C.c_void_p), ("values", C.c_void_p),
        ("chunk_nnz", C.c_int32), ("n_heavy_rows", C.c_int32), ("n_chunks", C.c_int64),
        ("heavy_rows", C.c_void_p), ("heavy_chunk_ptr", C.c_void_p), ("chunk_owner", C.c_void_p),
        ("work_order", C.c_void_p), ("n_work", C.c_int64),
        ("chunk_start", C.c_void_p),
    ]


class Epilogue(C.Structure):
    """hgr_epilogue_t"""
    _fields_ = [
        ("use_leaky", C.c_int32), ("leaky_slope", C.c_float),
        ("ln_gamma", C.c_void_p), ("ln_beta", C.c_void_p), ("ln_eps", C.c_float),
        ("residual", C.c_void_p),
        ("n_addends", C.c_int32), ("addends", C.c_void_p * HGR_MAX_ADDENDS),
        ("scale", C.c_float), ("scale_always", C.c_int32),
        ("pre", C.c_void_p),
        ("n_gather", C.c_int32), ("gather_out", C.c_void_p * HGR_MAX_GATHER), ("gather_row_offset", C.c_int64),
        ("gather_mc", C.c_void_p),
    ]


class Gather(C.Structure):
    """hgr_gather_t"""
    _fields_ = [("n_gather", C.c_int32), ("out", C.c_void_p * HGR_MAX_GATHER), ("row_offset", C.c_int64), ("mc", C.c_void_p)]


def make_gather(ptrs, row_offset: int, mc: int = 0) -> Gather:
    g = Gather()
    g.n_gather = len(ptrs)
    for j, p in enumerate(ptrs):
        g.out[j] = int(p)
    g.row_offset = int(row_offset)
    g.mc = int(mc) or None
    return g


_lib = None

# name -> (restype, argtypes); every symbol include/hgr.h declares
_VP, _I32, _I64, _F32, _SZ = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_size_t
SIGNATURES = {
    "hgr_last_error": (C.c_char_p, []),
    "hgr_version": (C.c_int, []),
    "hgr_launch_count": (C.c_uint64, []),
    "hgr_spmm_workspace_bytes": (_SZ, [C.POINTER(CsrDesc), _I32]),
    "hgr_spmm_f32": (C.c_int, [C.POINTER(CsrDesc), _VP, _VP, _I32, C.POINTER(Epilogue), _VP, _SZ, _VP]),
    "hgr_hgconv_f32": (C.c_int, [C.POINTER(CsrDesc), C.POINTER(CsrDesc), _VP, _VP, _VP, _I32, C.POINTER(Epilogue), _VP, _SZ, _VP]),
    "hgr_lightgcn_forward_f32": (C.c_int, [C.POINTER(CsrDesc), _VP, _VP, _VP, _I32, _I32, _I32, _VP, _SZ, _VP]),
    "hgr_layer_norm_f32": (C.c_int, [_VP, _VP, _VP, _F32, _I64, _I32, _VP, _VP]),
    "hgr_ln_bwd_partial_rows": (_I32, [_I64]),
    "hgr_leaky_ln_bwd_f32": (C.c_int, [_VP, _VP, _VP, _F32, _I32, _F32, _I64, _I32, _VP, _VP, _VP, _VP, _VP]),
    "hgr_leaky_ln_bwd_gather_f32": (C.c_int, [_VP, _VP, _VP, _F32, _I32, _F32, _I64, _I32, _VP, _VP, _VP, _VP, C.POINTER(Gather), _VP]),
    "hgr_publish_rows_f32": (C.c_int, [_VP, _I64, _I32, C.POINTER(Gather), _VP]),
    "hgr_tall_skinny_workspace_bytes": (_SZ, [_I64, _I32, _I32]),
    "hgr_tall_skinny_tn_f32": (C.c_int, [_VP, _VP, _I64, _I32, _I32, _VP, _VP, _SZ, _VP]),
    "hgr_rows_times_small_f32": (C.c_int, [_VP, _I32, _VP, _I32, _VP, _I32, _I64, _VP, _VP]),
    "hgr_rows_times_small_bias_f32": (C.c_int, [_VP, _I32, _VP, _I32, _VP, _I32, _I64, _VP, _VP, _I32, _VP]),
    "hgr_rows_times_small_gather_f32": (C.c_int, [_VP, _I32, _VP, _I32, _VP, _I32, _I64, _VP, _VP, _I32, C.POINTER(Gather), _VP]),
    "hgr_add_rows_f32": (C.c_int, [_VP, _VP, _I64, _I32, _VP, C.POINTER(Gather), _VP]),
    "hgr_build_csr_workspace_bytes": (_SZ, [_I64]),
    "hgr_coo_to_csr": (C.c_int, [_VP, _VP, _I64, _I32, _I32, _VP, _VP, _VP, _VP, _VP, _VP, _SZ, _VP]),
    "hgr_bipartite_to_csr": (C.c_int, [_VP, _VP, _I64, _I32, _I32, _VP, _VP, _VP, _VP, _VP, _VP, _SZ, _VP]),
    "hgr_degree_scale": (C.c_int, [_VP, _I64, _VP, _I32, _VP, _VP, _VP]),
    "hgr_csr_scale": (C.c_int, [_VP, _VP, _VP, _I32, _VP, _VP, _VP]),
    "hgr_bpr_l2_workspace_bytes": (_SZ, [_I64]),
    "hgr_bpr_l2_fwd_f32": (C.c_int, [_VP, _VP, _I64, _I64, _I32, _VP, _VP, _VP, _I64, _F32, _F32, _VP, _VP, _SZ, _VP, _VP]),
    "hgr_rank_metrics": (C.c_int, [_VP, _I64, _I32, _VP, _VP, _VP, _I32, _VP, _VP, _VP, _VP]),
    "hgr_drop_edges_f32": (C.c_int, [_VP, _VP, _VP, _I32, _I64, _I64, _F32, C.c_uint64, _VP, _VP, _VP, _I32, _VP, _VP]),
    "hgr_window_split_count": (C.c_int, [_VP, _VP, _I32, _I32, _I32, _I32, _I32, _VP, _VP]),
    "hgr_window_split_fill": (C.c_int, [_VP, _VP, _VP, _VP, _I32, _I32, _I32, _I32, _I32, _VP, _VP]),
    "hgr_rank_metric_sums": (C.c_int, [_VP, _VP, _VP, _I64, _I32, _VP, _VP, _I32, _I32, _VP, _VP, _VP, _VP]),
    "hgr_bpr_sample": (C.c_int, [_VP, _VP, _I64, _VP, _I64, _I64, _I32, _VP, _VP, _I32, C.c_uint64, C.c_uint64, _VP, _VP, _VP, _VP, _VP]),
    "hgr_ssl_workspace_bytes": (_SZ, [_I64, _I32]),
    "hgr_ssl_loss_fwd_f32": (C.c_int, [_VP, _VP, _I64, _I64, _I32, _VP, _I64, _F32, _I32, _I32, _VP, _VP, _SZ, _VP, _VP]),
    "hgr_ssl_loss_bwd_f32": (C.c_int, [_I64, _I64, _I32, _VP, _I64, _F32, _I32, _VP, _SZ, _VP, _VP, _VP, _VP]),
    "hgr_bpr_l2_fwd_owned_f32": (C.c_int, [_VP, _I64, _I32, _VP, _VP, _VP, _I64, _I64, _I64, _VP, _VP, _SZ, _VP, _VP]),
    "hgr_bpr_l2_finish_f32": (C.c_int, [_VP, _I64, _F32, _F32, _VP, _VP, _VP]),
    "hgr_bpr_l2_bwd_owned_f32": (C.c_int, [_VP, _I64, _I32, _VP, _VP, _VP, _I64, _F32, _F32, _VP, _VP, _I64, _I64, _VP, _VP]),
    "hgr_bpr_l2_bwd_window_f32": (C.c_int, [_VP, _I64, _I32, _VP, _VP, _VP, _I64, _F32, _F32, _VP, _VP, _I64, _I64, _VP, _VP]),
    "hgr_fullrank_topk_workspace_bytes": (_SZ, [_I64, _I64, _I32, _I32, _I32]),
    "hgr_fullrank_topk_f32": (C.c_int, [_VP, _I64, _VP, _I64, _I32, _VP, _I64, _VP, _VP, _I32, _I32, _I32, _VP, _VP, _VP, _VP, _SZ, _VP]),
    "hgr_bpr_l2_bwd_f32": (C.c_int, [_VP, _VP, _I64, _I64, _I32, _VP, _VP, _VP, _I64, _F32, _F32, _VP, _VP, _VP, _VP, _VP]),
}


def lib():
    """Load libhgr.so once.  Raises HgrError when it is missing: there is no other code path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise HgrError(
                "libhgr.so not found at %s -- build it with `python -m hypergraph_diffusion_for_recommendation_b200.build` "
                "(nvcc, sm_100a).  This package has no CPU or PyTorch fallback." % LIB_PATH)
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the symbol is not exported
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise HgrError("libhgr error %d: %s" % (rc, lib().hgr_last_error().decode()))


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr():
    import torch

    return torch.cuda.current_stream().cuda_stream


def launch_count() -> int:
    return int(lib().hgr_launch_count())
