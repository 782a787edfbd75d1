"""Loader for libfwb200.so.  Fails loudly: no CPU or eager fallback exists for any op."""
from __future__ import annotations

import ctypes as C
import re
from pathlib import Path

_HERE = Path(__file__).resolve().parent
_LIB_PATH = _HERE / "libfwb200.so"
_HEADER = _HERE.parent.parent / "include" / "fwb200.h"


class FwbError(RuntimeError):
    pass


def library_path() -> Path:
    return _LIB_PATH


def abi_symbols() -> list[str]:
    """Every function name declared in include/fwb200.h (used by the symbol-export test)."""
    text = _HEADER.read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(fwb_[a-z0-9_]+)\s*\(", text)))


class Epilogue(C.Structure):
    _fields_ = [
        ("bias", C.c_void_p), ("scale1", C.c_void_p), ("shift1", C.c_void_p), ("scale2", C.c_void_p),
        ("resid", C.c_void_p), ("resid_ld", C.c_int64), ("resid_dtype", C.c_int),
        ("out", C.c_void_p), ("out_ld", C.c_int64), ("out_dtype", C.c_int),
        ("act", C.c_int), ("round_flags", C.c_int),
    ]


class Tensor4(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("sb", C.c_int64), ("sl", C.c_int64), ("sh", C.c_int64)]


def _load():
    if not _LIB_PATH.exists():
        raise FwbError(
            f"{_LIB_PATH} is missing: build it with `python fantasy-world_b200/build.py` "
            "(or __graft_entry__.build()). There is no fallback path.")
    lib = C.CDLL(str(_LIB_PATH))
    lib.fwb_last_error.restype = C.c_char_p
    lib.fwb_abi_version.restype = C.c_int
    lib.fwb_device_ok.restype = C.c_int
    vp, i32, i64, f32 = C.c_void_p, C.c_int, C.c_int64, C.c_float
    lib.fwb_gemm_bf16.argtypes = [vp, i64, vp, i64, i32, i32, i32, C.POINTER(Epilogue), vp]
    lib.fwb_gemm_set_mode.argtypes = [i32]
    lib.fwb_attn_set_variant.argtypes = [i32]
    lib.fwb_attn_set_tail_split.argtypes = [i32]
    lib.fwb_attn_set_exp2_poly.argtypes = [i32]
    lib.fwb_attn_set_mufu_pingpong.argtypes = [i32, i32]
    lib.fwb_attn_set_pv_n96.argtypes = [i32]
    lib.fwb_attn_set_multicast.argtypes = [i32]
    lib.fwb_attn_set_short_kv_max.argtypes = [i32]
    lib.fwb_attn_fwd.argtypes = [C.POINTER(Tensor4)] * 4 + [i32, i32, i32, i32, i32, f32, i32, vp, C.c_size_t, vp]
    lib.fwb_attn_fwd_partial.argtypes = [C.POINTER(Tensor4)] * 3 + [vp, vp, i32, i32, i32, i32, i32, f32, vp, C.c_size_t, vp]
    lib.fwb_attn_merge.argtypes = [vp, vp, C.POINTER(Tensor4), i32, i32, i32, i32, i32, vp]
    lib.fwb_bringup_mma.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp, vp]
    lib.fwb_bringup_mma_pv_n.argtypes = [vp, vp, vp, i32, i32, i32, vp]
    lib.fwb_rowwise_set_ctas_per_sm.argtypes = [i32]
    lib.fwb_ln_modulate.argtypes = [vp, i32, i64, i32, i32, f32, vp, vp, vp, vp, vp, i64, vp]
    lib.fwb_rmsnorm_rope.argtypes = [vp, i64, i32, i32, vp, f32, vp, i32, vp]
    lib.fwb_rmsnorm_rope_periodic.argtypes = [vp, i64, i32, i32, vp, f32, vp, i32, i32, vp]
    lib.fwb_ln64_rope2d.argtypes = [vp, i64, i32, i32, f32, vp, vp, vp, vp, vp, vp, vp]
    lib.fwb_ln64_rope2d_periodic.argtypes = [vp, i64, i32, i32, f32, vp, vp, vp, vp, vp, vp, i32, vp]
    lib.fwb_cfg_euler_step.argtypes = [vp, vp, vp, i64, f32, f32, vp]
    for name in abi_symbols():
        fn = getattr(lib, name)  # raises AttributeError if a declared symbol is not exported
        if name not in ("fwb_last_error",):
            fn.restype = C.c_int if name != "fwb_last_error" else C.c_char_p
    lib.fwb_last_error.restype = C.c_char_p
    lib.fwb_attn_workspace_bytes.restype = C.c_size_t
    lib.fwb_attn_workspace_bytes.argtypes = []
    lib.fwb_attn_plan.argtypes = [i32, i32, i32, i32, i32, C.c_size_t, i32, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    return lib


lib = _load()


def check(rc: int, what: str):
    if rc != 0:
        msg = lib.fwb_last_error()
        raise FwbError(f"{what} failed (code {rc}): {msg.decode() if msg else '?'}")
