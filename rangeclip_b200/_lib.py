"""ctypes binding of ``librangeclip_b200.so`` (the C ABI declared in include/rangeclip_b200.h).

The shared library is built in-tree by ``rangeclip_b200/csrc/Makefile`` (or
``__graft_entry__.build()``).  There is NO fallback: if the library is missing, or a call
returns a non-zero status, a ``RuntimeError`` is raised.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RANGECLIP_B200_LIB", os.path.join(_HERE, "librangeclip_b200.so"))
CSRC = os.path.join(_HERE, "csrc")

RC_F32, RC_BF16 = 0, 1

_vp, _i32, _i64, _f32 = C.c_void_p, C.c_int, C.c_int64, C.c_float

# name -> argtypes (restype is int unless listed in _RESTYPES); mirrors include/rangeclip_b200.h
PROTOTYPES = {
    "rc_abi_version": [],
    "rc_last_error": [],
    "rc_launch_count": [],
    "rc_infonce_workspace_bytes": [_i32, _i32, _i64, _i32, _i32],
    "rc_infonce_workspace_bytes_dt": [_i32, _i32, _i64, _i32, _i32],
    "rc_infonce_f32": [_vp, _i32, _i32, _i64, _i64, _vp, _i32, _vp, _vp, _f32, _vp, _vp, _vp, _vp, _vp,
                       _vp, _vp, _vp, _vp],
    "rc_infonce_bf16": [_vp, _i32, _i32, _i32, _i64, _vp, _vp, _i32, _vp, _vp, _f32, _vp, _vp, _vp, _vp, _vp,
                        _vp, _vp, _vp, _vp, _i64, _i32, _vp],
    "rc_infonce_bf16_rep4": [_vp, _i32, _i32, _i32, _i64, _vp, _vp, _i32, _vp, _vp, _f32, _vp, _vp, _vp, _vp, _vp,
                             _vp, _vp, _vp, _vp, _i64, _i32, _vp],
    "rc_infonce_bf16_dyn": [_vp, _i32, _i32, _i32, _i64, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp,
                            _vp, _vp, _vp, _i64, _i32, _vp],
    "rc_infonce_bf16_dyn_kblock": [_vp, _i32, _i32, _i32, _i64, _vp, _vp, _i32, _vp, _i32, _vp, _vp, _vp, _i32, _vp, _vp, _vp,
                                   _vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp],
    "rc_contrast_build": [_vp, _i32, _vp, _vp, _i32, _i32, _i32, C.c_uint64, _vp, _i32, _vp, _vp, _vp, _vp],
    "rc_infonce_bf16_kblocks": [_vp, _i32, _i32, _i64, _vp, _vp, _i32, _i32, _vp, _vp, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                _vp, _i64, _i32, _vp],
    "rc_infonce_prepass": [_vp, _i32, _i32, _i32, _i64, _vp, _i64, _vp],
    "rc_infonce_prepass_tv": [_vp, _i32, _i32, _i32, _i32, _vp, _i64, _vp, _vp, _vp],
    "rc_tv_bwd_codes": [_vp, _i64, _i32, _i32, _vp, _vp, _i32, _vp, _vp, _vp],
    "rc_text_prepare": [_vp, _i64, _i64, _vp, _i32, _i32, _vp, _vp, _vp, _vp],
    "rc_weight_sum": [_vp, _vp, _i64, _vp, _vp],
    "rc_sample_weights": [_vp, _vp, _i32, _i64, _i64, _vp, _i32, _vp, _vp, _vp],
    "rc_sample_label_counts": [_vp, _vp, _i32, _i64, _i64, _i32, _vp, _vp],
    "rc_scale": [_vp, _i32, _i64, _vp, _vp],
    "rc_scale_to": [_vp, _i32, _vp, _i32, _i64, _vp, _vp],
    "rc_clip_crops": [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp],
    "rc_pool_fwd": [_vp, _i32, _i32, _i32, _i64, _vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp],
    "rc_pool_finish": [_vp, _vp, _i32, _i32, _vp],
    "rc_pool_bwd": [_vp, _vp, _i32, _i32, _i64, _vp, _vp, _i64, _i32, _i32, _vp, _i32, _i32, _vp],
    "rc_normalize_rows_fwd": [_vp, _i32, _i32, _i32, _i64, _vp, _vp, _vp],
    "rc_normalize_rows_bwd": [_vp, _vp, _vp, _i32, _i32, _i32, _i64, _vp, _vp],
    "rc_tv_normalize_bwd": [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp],
    "rc_tv_fwd": [_vp, _i32, _i64, _i32, _i32, _vp, _vp],
    "rc_tv_bwd": [_vp, _i32, _i64, _i32, _i32, _vp, _vp, _i32, _vp, _vp],
    "rc_tv_bwd_from": [_vp, _i32, _i64, _i32, _i32, _vp, _vp, _i32, _vp, _vp, _vp],
    "rc_eval_topk_f32": [_vp, _i32, _i32, _i64, _i64, _vp, _i32, _vp, _i32, _vp, _vp],
    "rc_eval_topk_bf16": [_vp, _i32, _i32, _i32, _i64, _vp, _i32, _vp, _i32, _vp, _vp, _i64, _vp],
    "rc_eval_topk_hist_bf16": [_vp, _i32, _i32, _i32, _i64, _vp, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _i32, _vp, _vp,
                               _vp, _i64, _vp],
    "rc_eval_topk_dyn_bf16": [_vp, _i32, _i32, _i32, _i64, _vp, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _i32, _vp, _vp,
                              _vp, _i64, _vp],
    "rc_eval_topk_bf16_rep4": [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _i32, _vp, _vp,
                               _vp, _i64, _vp],
    "rc_eval_hist": [_vp, _vp, _i32, _i64, _i32, _vp, _vp, _i32, _vp, _vp, _vp],
    "rc_eval_fold": [_vp, _i32, _i32, _vp, _vp, _vp],
}
# entry points that exist only in the bring-up build (librangeclip_b200_bringup.so, -DRC_BRINGUP)
BRINGUP_PROTOTYPES = {
    "rc_debug_set_timing_buffer": [_vp],
    "rc_debug_max_active_clusters": [_i32, _i32, _i32],
    "rc_debug_umma_gemm_2sm": [_vp, _vp, _i32, _i32, _vp, _vp],
    "rc_debug_umma_gemm_ts_2sm": [_vp, _vp, _i32, _i32, _vp, _vp],
    "rc_debug_umma_gemm": [_vp, _vp, _i32, _i32, _i32, _vp, _vp],
}
_RESTYPES = {"rc_last_error": C.c_char_p, "rc_launch_count": _i64, "rc_infonce_workspace_bytes": _i64,
             "rc_infonce_workspace_bytes_dt": _i64}

BRINGUP_LIB_PATH = os.path.join(_HERE, "librangeclip_b200_bringup.so")
_lib = None
_bringup = None


def build(verbose: bool = False) -> str:
    """Compile the CUDA sources for sm_100a (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(["make", "-C", CSRC, "-j8", "all", "bringup"], capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout[-4000:], r.stderr[-4000:])
    if r.returncode != 0:
        raise RuntimeError("building librangeclip_b200.so failed")
    return LIB_PATH


def lib() -> C.CDLL:
    """The loaded library; raises if it has not been built (no CPU / PyTorch fallback exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: run `make -C rangeclip_b200/csrc` (or __graft_entry__.build()); "
                "rangeclip_b200 has no fallback path")
        l = C.CDLL(LIB_PATH)
        for name, argtypes in PROTOTYPES.items():
            fn = getattr(l, name)
            fn.argtypes = argtypes
            fn.restype = _RESTYPES.get(name, C.c_int)
        if l.rc_abi_version() != 1:
            raise RuntimeError("librangeclip_b200.so: ABI version mismatch")
        _lib = l
    return _lib


def bringup_lib() -> C.CDLL:
    """The bring-up build of the same sources (adds the rc_debug_* entry points and the RANGECLIP_B200_* environment
    switches); used by the tcgen05 building-block tests and the tools, never by the drop-ins."""
    global _bringup
    if _bringup is None:
        if not os.path.exists(BRINGUP_LIB_PATH):
            raise RuntimeError(f"{BRINGUP_LIB_PATH} is missing: run `make -C rangeclip_b200/csrc bringup`")
        l = C.CDLL(BRINGUP_LIB_PATH)
        for name, argtypes in {**PROTOTYPES, **BRINGUP_PROTOTYPES}.items():
            fn = getattr(l, name)
            fn.argtypes = argtypes
            fn.restype = _RESTYPES.get(name, C.c_int)
        _bringup = l
    return _bringup


def check(status: int, what: str) -> None:
    if status != 0:
        msg = lib().rc_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (status {status}): {msg}")


def launch_count() -> int:
    return int(lib().rc_launch_count())
