"""ctypes binding of csrc/liblrs_pnp.so (C ABI declared in include/lrs_pnp.h).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C
lrs_pnp_dip_b200/csrc``.  There is no CPU or PyTorch fallback: if the shared
object is missing, or a compute entry point is called without a CUDA device,
the call raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
# LRS_PNP_LIB: developer switch for A/B runs of kernel variants (scripts/ab_fused.py); unset in normal use
LIB_PATH = os.environ.get("LRS_PNP_LIB") or os.path.join(_HERE, "csrc", "liblrs_pnp.so")

STEP_SPECTRAL, STEP_FROB4 = 0, 1
ENGINE_AUTO, ENGINE_SIMT, ENGINE_TC = 0, 1, 2
ENGINES = {"auto": ENGINE_AUTO, "simt": ENGINE_SIMT, "tc": ENGINE_TC}
ENGINE_DYNAMIC_TILES = 0x100          # OR-ed into the engine: work items claimed dynamically (include/lrs_pnp.h)
DENOISERS = {"soft": 0, "nlm": 1, "identity": 2}
MAX_BATCH = 65535                     # LRS_MAX_BATCH: largest cube count of the batched entry points

_p = C.c_void_p
_i64 = C.c_int64
_int = C.c_int
_f = C.c_float

# name -> (restype, argtypes); mirrors include/lrs_pnp.h one to one
SIGNATURES = {
    "lrs_last_error": (C.c_char_p, []),
    "lrs_version": (_int, []),
    "lrs_launch_count": (C.c_uint64, []),
    "lrs_axis_count": (_i64, [_i64, _int, _int]),
    "lrs_axis_starts": (_int, [_i64, _int, _int, C.POINTER(_i64), _i64]),
    "lrs_patch_index_i64": (_int, [_i64, _i64, _int, _int, _p, _p, _p, _p]),
    "lrs_im2col_f32": (_int, [_p, _p, _f, _i64, _i64, _int, _int, _p, _p]),
    "lrs_col2im_accum_f32": (_int, [_p, _i64, _i64, _int, _int, _p, _p]),
    "lrs_im2col_batch_f32": (_int, [_p, _p, _f, _i64, _i64, _i64, _int, _int, _p, _p]),
    "lrs_col2im_accum_batch_f32": (_int, [_p, _i64, _i64, _i64, _int, _int, _p, _p]),
    "lrs_col2im_accum_range_f32": (_int, [_p, _i64, _i64, _int, _int, _i64, _i64, _p, _p]),
    "lrs_coverage_weight_f32": (_int, [_i64, _i64, _int, _int, _p, _p]),
    "lrs_soft_f32": (_int, [_p, _f, _p, _i64, _p]),
    "lrs_axpy_f32": (_int, [_p, _p, _f, _p, _i64, _p]),
    "lrs_step_frob4_f32": (_int, [_p, _p, _int, _int, _i64, _p, _p]),
    "lrs_patch_mask_words_u64": (_int, [_p, _i64, _i64, _int, _int, _i64, _i64, _p, _p]),
    "lrs_spectral_patterns_workspace_bytes": (C.c_size_t, [_int]),
    "lrs_spectral_patterns_f32": (_int, [_p, _int, _int, _p, _i64, _p, _int, _p, _p, C.c_size_t, _p]),
    "lrs_ista_workspace_bytes": (C.c_size_t, [_int, _int, _i64]),
    "lrs_ista_soft_f32": (_int, [_p, _p, _p, _p, _f, _int, _int, _int, _i64, _p, _p, _p, C.c_size_t, _p]),
    "lrs_ista_pnp_f32": (_int, [_p, _p, _p, _p, _f, _int, _int, _int, _i64, _int, _f, _p, _p, _p, C.c_size_t, _p]),
    "lrs_sparse_step_fused_f32": (_int, [_p, _p, _f, _p, _p, _int, _p, _p, _f, _int, _i64, _i64, _int, _int, _i64,
                                         _i64, _p, _int, _p]),
    "lrs_admm_update_f32": (_int, [_p, _p, _p, _p, _p, _p, _p, _f, _f, _f, _i64, _i64, _i64, _i64, _int, _int, _p]),
    "lrs_admm_update_batch_f32": (_int, [_p, _p, _p, _p, _p, _p, _p, _f, _f, _f, _i64, _i64, _i64, _int, _int, _p]),
    "lrs_gram_f64": (_int, [_p, _p, _f, _i64, _i64, _p, _p]),
    "lrs_gram_batch_f64": (_int, [_p, _p, _f, _i64, _i64, _i64, _p, _p]),
    "lrs_sym_eig_jacobi_f64": (_int, [_p, _int, _p, _p, _p, _p]),
    "lrs_sym_eig_jacobi_batch_f64": (_int, [_p, _i64, _int, _p, _p, _p, _p]),
    "lrs_svt_weights_f64": (_int, [_p, _p, _i64, _i64, _int, _int, C.c_double, _int, _p, _p]),
    "lrs_svt_weights_batch_f64": (_int, [_p, _p, _i64, _i64, _i64, _i64, _int, _int, C.c_double, _int, _p, _p]),
    "lrs_svt_apply_f32": (_int, [_p, _p, _f, _p, _i64, _i64, _p, _p]),
    "lrs_svt_apply_batch_f32": (_int, [_p, _p, _f, _p, _i64, _i64, _i64, _p, _p]),
}

# diagnostics build only (include/lrs_pnp_diag.h, csrc/liblrs_pnp_diag.so): never loaded by the product path
DIAG_SIGNATURES = {
    "lrs_tc_probe_f32": (_int, [_p, _p, _p, _int, _int, _int, _int, _int, _p]),
    "lrs_tc_timing_read": (_int, [C.POINTER(C.c_uint64)]),
    "lrs_debug_tile_walk": (_int, [_i64, _i64, _int, _int, _i64, _i64, _int, _p, _p]),
    "lrs_debug_tile_walk_ordered": (_int, [_i64, _i64, _int, _int, _i64, _i64, _int, _p, _p, _p, _p]),
    "lrs_debug_jacobi_schedule": (_int, [_int, _p, _p, _p]),
    "lrs_debug_ista_plan": (_int, [_int, _int, _i64, _p]),
    "lrs_tc_microbench": (_int, [_int, _int, _int, _int, _int, _int, _int, _int, _int, _p, _p]),
}
DIAG_LIB_PATH = os.path.join(_HERE, "csrc", "liblrs_pnp_diag.so")

_lib: Optional[C.CDLL] = None
_diag: Optional[C.CDLL] = None


class LrsError(RuntimeError):
    pass


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if os.environ.get("LRS_PNP_DIAGNOSTICS") == "1":      # developer switch (scripts/tc_timing.py): instrumented build
            _lib = diag_lib()
            return _lib
        if not os.path.isfile(LIB_PATH):
            raise LrsError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C lrs_pnp_dip_b200/csrc`. There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError here = header / library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def diag_lib() -> C.CDLL:
    """The diagnostics build (tests/ and scripts/ only): the product entry points compiled with -DLRS_DIAGNOSTICS plus
    the tcgen05 probes, the host replay of the tile walk and the barrier-wait counters."""
    global _diag
    if _diag is None:
        if not os.path.isfile(DIAG_LIB_PATH):
            raise LrsError(f"{DIAG_LIB_PATH} not found: build it with `make -C lrs_pnp_dip_b200/csrc`")
        L = C.CDLL(DIAG_LIB_PATH)
        for name, (res, args) in {**SIGNATURES, **DIAG_SIGNATURES}.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _diag = L
    return _diag


def check(rc: int, what: str = "", L: Optional[C.CDLL] = None) -> None:
    if rc != 0:
        msg = (L or lib()).lrs_last_error()
        raise LrsError(f"{what or 'liblrs_pnp'} failed (code {rc}): {msg.decode() if msg else ''}")


def require_cuda():
    import torch

    if not torch.cuda.is_available():
        raise LrsError("lrs_pnp_dip_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


def stream_ptr() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream


def ptr(t) -> Optional[int]:
    return None if t is None else t.data_ptr()
