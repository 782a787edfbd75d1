"""Thin torch-tensor wrappers over the C ABI (include/fwb200.h).  Device pointers + sizes only cross the boundary."""
from __future__ import annotations

import ctypes as C
import math

import torch

from ._lib import Epilogue, Tensor4, check, lib

ACT_NONE, ACT_GELU_TANH, ACT_GELU_ERF, ACT_RELU, ACT_SILU = 0, 1, 2, 3, 4
ROUND_AFTER_BIAS, ROUND_AFTER_ACT, ROUND_AFTER_AFFINE, ROUND_AFTER_SCALE2 = 1, 2, 4, 8
DT_BF16, DT_F32 = 0, 1

__all__ = [
    "ACT_NONE", "ACT_GELU_TANH", "ACT_GELU_ERF", "ACT_RELU", "ACT_SILU",
    "ROUND_AFTER_BIAS", "ROUND_AFTER_ACT", "ROUND_AFTER_AFFINE", "ROUND_AFTER_SCALE2",
    "device_ok", "require_device", "linear", "attention", "attention_partial", "attention_merge", "bringup_mma",
    "ln_modulate", "rmsnorm_rope_", "ln64_rope2d_", "cfg_euler_step_", "launch_count", "reset_launch_count",
    "prof_enable", "prof_disable",
]

_LAUNCHES = 0


def launch_count() -> int:
    """Number of fwb200 kernel launches issued through this binding since the last reset."""
    return _LAUNCHES


def reset_launch_count():
    global _LAUNCHES
    _LAUNCHES = 0


def _count(n=1):
    global _LAUNCHES
    _LAUNCHES += n


# ---- optional per-launch CUDA-event timing (bench.py: roofline of the dominant kernel, step breakdown) -------------
_PROF = None


def prof_enable(prefixes=None):
    """Record a CUDA-event pair around every fwb200 launch whose tag starts with one of `prefixes` (None = all)."""
    global _PROF
    _PROF = {"prefixes": tuple(prefixes) if prefixes else None, "rec": {}}


def prof_disable():
    """Stop recording; returns {tag: (launches, total_ms)} (synchronises the device)."""
    global _PROF
    prof, _PROF = _PROF, None
    if prof is None:
        return {}
    torch.cuda.synchronize()
    return {tag: (len(ev), sum(a.elapsed_time(b) for a, b in ev)) for tag, ev in prof["rec"].items()}


import os as _os

_DEBUG_NAN = bool(int(_os.environ.get("FWB_DEBUG_NAN", "0")))


def _nan_check(tag, *tensors):
    """FWB_DEBUG_NAN=1: synchronise after every launch and report the first op that produces a non-finite value."""
    if _DEBUG_NAN:
        torch.cuda.synchronize()
        for i, t in enumerate(tensors):
            if t is not None and not torch.isfinite(t.float()).all():
                raise FloatingPointError(f"non-finite values in output {i} of {tag}")


class _Rec:
    __slots__ = ("tag", "a")

    def __init__(self, tag):
        self.tag = tag

    def __enter__(self):
        p = _PROF
        self.a = None
        if p is not None and (p["prefixes"] is None or self.tag.startswith(p["prefixes"])):
            self.a = torch.cuda.Event(enable_timing=True)
            self.a.record()
        return self

    def __exit__(self, *exc):
        if self.a is not None and _PROF is not None:
            b = torch.cuda.Event(enable_timing=True)
            b.record()
            _PROF["rec"].setdefault(self.tag, []).append((self.a, b))
        return False


def device_ok() -> bool:
    return bool(lib.fwb_device_ok())


def require_device():
    if not device_ok():
        msg = lib.fwb_last_error()
        raise RuntimeError("fwb200 needs a B200 (sm_100) device: " + (msg.decode() if msg else ""))


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _dt(t: torch.dtype) -> int:
    if t == torch.bfloat16:
        return DT_BF16
    if t == torch.float32:
        return DT_F32
    raise TypeError(f"unsupported dtype {t}")


def _f32vec(v, n, name):
    if v is None:
        return None
    if not (v.is_cuda and v.dtype == torch.float32 and v.is_contiguous() and v.numel() == n):
        raise ValueError(f"{name} must be a contiguous fp32 CUDA vector of {n} elements")
    return v


def linear(x: torch.Tensor, w: torch.Tensor, *, bias=None, act: int = ACT_NONE, scale1=None, shift1=None, scale2=None,
           resid=None, out=None, out_dtype=torch.bfloat16, round_flags: int = 0) -> torch.Tensor:
    """out = resid + scale2 * (scale1 * act(x @ w.T + bias) + shift1); x [..., K] bf16, w [N, K] bf16."""
    if not (x.is_cuda and w.is_cuda):
        raise RuntimeError("fwb200.linear: CUDA tensors required (no CPU fallback)")
    if x.dtype != torch.bfloat16 or w.dtype != torch.bfloat16:
        raise TypeError("fwb200.linear: x and w must be bf16")
    K = x.shape[-1]
    N = w.shape[0]
    assert w.shape[1] == K and w.stride(1) == 1
    x2 = x.reshape(-1, K)
    if x2.stride(1) != 1:
        x2 = x2.contiguous()
    M = x2.shape[0]
    if out is None:
        out = torch.empty((M, N), device=x.device, dtype=out_dtype)
    out2 = out.view(-1, N) if out.dim() != 2 else out
    assert out2.shape == (M, N) and out2.stride(1) == 1
    ep = Epilogue()
    bias = _f32vec(bias, N, "bias")
    scale1 = _f32vec(scale1, N, "scale1")
    shift1 = _f32vec(shift1, N, "shift1")
    scale2 = _f32vec(scale2, N, "scale2")
    ep.bias = bias.data_ptr() if bias is not None else None
    ep.scale1 = scale1.data_ptr() if scale1 is not None else None
    ep.shift1 = shift1.data_ptr() if shift1 is not None else None
    ep.scale2 = scale2.data_ptr() if scale2 is not None else None
    if resid is not None:
        r2 = resid.reshape(-1, N)
        assert r2.shape == (M, N) and r2.stride(1) == 1
        ep.resid, ep.resid_ld, ep.resid_dtype = r2.data_ptr(), r2.stride(0), _dt(r2.dtype)
    else:
        ep.resid, ep.resid_ld, ep.resid_dtype = None, 0, 0
    ep.out, ep.out_ld, ep.out_dtype = out2.data_ptr(), out2.stride(0), _dt(out2.dtype)
    ep.act, ep.round_flags = act, round_flags
    _count()
    with _Rec(f"gemm:M{M}:N{N}:K{K}"):
        check(lib.fwb_gemm_bf16(x2.data_ptr(), x2.stride(0), w.data_ptr(), w.stride(0), M, N, K, C.byref(ep), _stream()),
              "fwb_gemm_bf16")
    _nan_check(f"gemm:M{M}:N{N}:K{K}:act{act}", out)
    return out.view(*x.shape[:-1], N) if out.dim() == 2 and x.dim() != 2 else out


def _t4(t: torch.Tensor) -> Tensor4:
    # t: [B, L, H, D] view with unit stride on D
    assert t.dim() == 4 and t.stride(3) == 1 and t.dtype == torch.bfloat16 and t.is_cuda
    r = Tensor4()
    r.ptr, r.sb, r.sl, r.sh = t.data_ptr(), t.stride(0), t.stride(1), t.stride(2)
    return r


_attn_ws: dict = {}


_ATTN_WS_MAX = 8


def _attn_workspace(device):
    """Scratch for the tail split of the attention tile schedule (fwb_attn_workspace_bytes, ~78 MB), one per (device, stream).
    Stream handles are recycled by the driver and a process may create many side streams, so the cache is bounded: beyond
    _ATTN_WS_MAX entries the least recently used one is dropped (its memory returns to the caching allocator once the kernels
    already queued on it have run: the allocator keeps a block alive until its recorded stream uses are complete)."""
    stream = torch.cuda.current_stream(device)
    key = (device.index, stream.cuda_stream)
    ws = _attn_ws.pop(key, None)
    if ws is None:
        ws = torch.empty(int(lib.fwb_attn_workspace_bytes()), device=device, dtype=torch.uint8)
        while len(_attn_ws) >= _ATTN_WS_MAX:
            old = _attn_ws.pop(next(iter(_attn_ws)))
            old.record_stream(stream)
    _attn_ws[key] = ws          # re-insert: dict order = recency
    return ws


def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, *, scale: float | None = None, out=None,
              accumulate: bool = False) -> torch.Tensor:
    """softmax(scale * q k^T) v, non-causal. q [B, Lq, H, D], k/v [B, Lk, H, D] (bf16 views, D contiguous)."""
    B, Lq, H, D = q.shape
    Lk = k.shape[1]
    assert k.shape == (B, Lk, H, D) and v.shape == (B, Lk, H, D)
    if scale is None:
        scale = 1.0 / math.sqrt(D)
    if out is None:
        out = torch.empty((B, Lq, H, D), device=q.device, dtype=torch.bfloat16)
    tq, tk, tv, to = _t4(q), _t4(k), _t4(v), _t4(out)
    _count()
    with _Rec(f"attn:B{B}:H{H}:Lq{Lq}:Lk{Lk}:D{D}"):
        ws = _attn_workspace(q.device)
        check(lib.fwb_attn_fwd(C.byref(tq), C.byref(tk), C.byref(tv), C.byref(to), B, H, Lq, Lk, D, float(scale), int(accumulate),
                               ws.data_ptr(), ws.numel(), _stream()), "fwb_attn_fwd")
    _nan_check(f"attn:B{B}:H{H}:Lq{Lq}:Lk{Lk}:D{D}:acc{int(accumulate)}", out)
    return out


def attention_partial(q, k, v, part_out: torch.Tensor, part_lse: torch.Tensor, *, scale: float | None = None):
    """Attention of q over ONE subset of the keys: fp32 subset-normalised result into part_out [B, Lq, H, D] and the base-2 row
    log-sum-exp into part_lse [B, H, Lq] (see attention_merge)."""
    B, Lq, H, D = q.shape
    Lk = k.shape[1]
    if scale is None:
        scale = 1.0 / math.sqrt(D)
    assert part_out.shape == (B, Lq, H, D) and part_out.dtype == torch.float32 and part_out.is_contiguous()
    assert part_lse.shape == (B, H, Lq) and part_lse.dtype == torch.float32 and part_lse.is_contiguous()
    tq, tk, tv = _t4(q), _t4(k), _t4(v)
    _count()
    with _Rec(f"attn:B{B}:H{H}:Lq{Lq}:Lk{Lk}:D{D}"):
        ws = _attn_workspace(q.device)
        check(lib.fwb_attn_fwd_partial(C.byref(tq), C.byref(tk), C.byref(tv), part_out.data_ptr(), part_lse.data_ptr(), B, H, Lq, Lk,
                                       D, float(scale), ws.data_ptr(), ws.numel(), _stream()), "fwb_attn_fwd_partial")


def attention_merge(part: torch.Tensor, lse: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    """Combine S partial attentions (part [S, B, L, H, D] fp32, lse [S, B, H, L]) into the bf16 result [B, L, H, D]."""
    S, B, L, H, D = part.shape
    assert lse.shape == (S, B, H, L) and part.is_contiguous() and lse.is_contiguous()
    if out is None:
        out = torch.empty((B, L, H, D), device=part.device, dtype=torch.bfloat16)
    to = _t4(out)
    _count()
    with _Rec(f"attnmerge:S{S}:L{L}:H{H}:D{D}"):
        check(lib.fwb_attn_merge(part.data_ptr(), lse.data_ptr(), C.byref(to), S, B, H, L, D, _stream()), "fwb_attn_merge")
    return out


def bringup_mma(A: torch.Tensor, Bm: torch.Tensor, N: int, K: int, a_in_tmem: bool, b_mn_major: bool, overrides=None):
    D = torch.empty((128, N), device=A.device, dtype=torch.float32)
    ov = None
    if overrides is not None:
        arr = (C.c_uint32 * 8)(*[0xFFFFFFFF if o is None else int(o) for o in overrides])
        ov = C.cast(arr, C.c_void_p)
    check(lib.fwb_bringup_mma(A.data_ptr(), Bm.data_ptr(), D.data_ptr(), N, K, int(a_in_tmem), int(b_mn_major), ov,
                              _stream()), "fwb_bringup_mma")
    return D


def _vec(v, n, name):
    return None if v is None else _f32vec(v, n, name).data_ptr()


def ln_modulate(x: torch.Tensor, *, eps: float, w=None, b=None, mul=None, add=None, out=None) -> torch.Tensor:
    """out = bf16((LN(x) * w + b) * mul + add); x [..., C] bf16 or fp32 (last dim contiguous)."""
    if not x.is_cuda:
        raise RuntimeError("fwb200.ln_modulate: CUDA tensor required (no CPU fallback)")
    C = x.shape[-1]
    x2 = x.reshape(-1, C)
    if x2.stride(1) != 1:
        x2 = x2.contiguous()
    rows = x2.shape[0]
    if out is None:
        out = torch.empty((rows, C), device=x.device, dtype=torch.bfloat16)
    o2 = out.view(-1, C)
    _count()
    with _Rec(f"ln:R{rows}:C{C}:in{x2.element_size()}"):
      check(lib.fwb_ln_modulate(x2.data_ptr(), _dt(x2.dtype), x2.stride(0), rows, C, float(eps), _vec(w, C, "w"),
                              _vec(b, C, "b"), _vec(mul, C, "mul"), _vec(add, C, "add"), o2.data_ptr(), o2.stride(0),
                              _stream()), "fwb_ln_modulate")
    _nan_check(f"ln:R{rows}:C{C}", out)
    return out.view(*x.shape[:-1], C)


def rmsnorm_rope_(x: torch.Tensor, *, w=None, eps: float = 1e-6, cos_sin=None, head_dim: int = 0) -> torch.Tensor:
    """In place on bf16 x [rows, C] (row stride allowed): full-row RMSNorm(+w) then interleaved-pair RoPE.  cos_sin
    [T, head_dim/2, 2] with T dividing rows: row r uses table row r % T (a batch of B samples shares one per-position table)."""
    assert x.dim() == 2 and x.stride(1) == 1 and x.dtype == torch.bfloat16 and x.is_cuda
    rows, C = x.shape
    table_rows = rows
    if cos_sin is not None:
        table_rows = cos_sin.shape[0]
        assert cos_sin.dtype == torch.float32 and cos_sin.is_contiguous() and cos_sin.shape[1:] == (head_dim // 2, 2)
        if rows % table_rows:
            raise ValueError(f"rmsnorm_rope_: RoPE table of {table_rows} rows does not divide {rows} token rows")
    _count()
    with _Rec(f"rmsrope:R{rows}:C{C}"):
      check(lib.fwb_rmsnorm_rope_periodic(x.data_ptr(), x.stride(0), rows, C, _vec(w, C, "w"), float(eps),
                                        None if cos_sin is None else cos_sin.data_ptr(), table_rows, head_dim, _stream()),
            "fwb_rmsnorm_rope_periodic")
    _nan_check(f"rmsrope:R{rows}:C{C}", x)
    return x


def ln64_rope2d_(qkv: torch.Tensor, H: int, *, eps: float, qw, qb, kw, kb, cosT, sinT) -> torch.Tensor:
    """In place on packed qkv bf16 [rows, 3*H*64]: per-head LayerNorm + 2-D RoPE on the q and k thirds.  cosT / sinT [T, 64]
    with T dividing rows: row r uses table row r % T."""
    assert qkv.dim() == 2 and qkv.stride(1) == 1 and qkv.dtype == torch.bfloat16 and qkv.is_cuda
    rows = qkv.shape[0]
    table_rows = cosT.shape[0]
    assert cosT.shape == (table_rows, 64) and sinT.shape == (table_rows, 64) and cosT.is_contiguous() and sinT.is_contiguous()
    if rows % table_rows:
        raise ValueError(f"ln64_rope2d_: RoPE table of {table_rows} rows does not divide {rows} token rows")
    _count()
    with _Rec(f"ln64rope:R{rows}:H{H}"):
      check(lib.fwb_ln64_rope2d_periodic(qkv.data_ptr(), qkv.stride(0), rows, H, float(eps), _vec(qw, 64, "qw"), _vec(qb, 64, "qb"),
                                       _vec(kw, 64, "kw"), _vec(kb, 64, "kb"), cosT.data_ptr(), sinT.data_ptr(), table_rows,
                                       _stream()),
          "fwb_ln64_rope2d_periodic")
    _nan_check(f"ln64rope:R{rows}", qkv)
    return qkv


def cfg_euler_step_(latents: torch.Tensor, pred_pos: torch.Tensor, pred_neg: torch.Tensor, cfg_scale: float,
                    dsigma: float) -> torch.Tensor:
    for t in (latents, pred_pos, pred_neg):
        assert t.is_cuda and t.dtype == torch.bfloat16 and t.is_contiguous()
    _count()
    check(lib.fwb_cfg_euler_step(latents.data_ptr(), pred_pos.data_ptr(), pred_neg.data_ptr(), latents.numel(),
                                 float(cfg_scale), float(dsigma), _stream()), "fwb_cfg_euler_step")
    return latents
