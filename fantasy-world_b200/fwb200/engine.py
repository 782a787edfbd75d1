"""engine.py — the fused execution of the hot-path blocks on top of the C-ABI kernels.

The nn.Module classes under fantasy-world_b200/FantasyWorld/ (same names, signatures and state_dict keys as the
reference) own the parameters; their forward() bodies delegate here.  Everything below launches only fwb200 kernels
for the token-sized work; torch is used for allocation and for O(C)-sized vector prep (modulation vectors, tables).

Rounding points follow the reference's CUDA-autocast run (SURVEY.md Appendix A) — see oracle/fw_oracle.py, which
restates the same points on the CPU.
"""
from __future__ import annotations

import torch

from . import ops
from .ops import (ACT_GELU_ERF, ACT_GELU_TANH, ACT_RELU, ACT_SILU, ROUND_AFTER_ACT, ROUND_AFTER_AFFINE, ROUND_AFTER_BIAS)

BF16 = torch.bfloat16

# Sequence-parallel context (fwb200.sp.SPContext) for the duration of a joint_forward, or None on a single GPU.
SP = None
SP_GLOBAL_ATTN = False   # set by IRGBlock around the VGGT *global* block so that it gathers K|V across ranks


# ------------------------------------------------------------------------------------------------------------------
# identity caches.  Entries hold STRONG references to their source tensors and hit only on object identity + version:
# a freed tensor's address can be handed to a new tensor by the caching allocator, so (data_ptr, shape) alone is not a
# safe key.
# ------------------------------------------------------------------------------------------------------------------
class IdCache:
    def __init__(self, max_entries=8):
        self.max_entries = max_entries
        self.entries = {}

    def lookup(self, srcs, extra=None):
        key = (tuple(id(s) for s in srcs), extra)
        hit = self.entries.get(key)
        if hit is not None and all(a is b and a._version == v for a, b, v in zip(hit[0], srcs, hit[1])):
            return hit[2]
        return None

    def store(self, srcs, extra, value):
        if len(self.entries) >= self.max_entries:
            self.entries.pop(next(iter(self.entries)))
        self.entries[(tuple(id(s) for s in srcs), extra)] = (tuple(srcs), tuple(s._version for s in srcs), value)
        return value

    def get(self, srcs, extra, fn):
        hit = self.lookup(srcs, extra)
        if hit is None:
            with torch.no_grad():
                hit = self.store(srcs, extra, fn())
        return hit


def derived(owner, name, fn, *srcs):
    """Cache fn(*srcs) on `owner` (an nn.Module): fp32 copies of bias / norm vectors, padded or concatenated weights.
    Recomputed when a source tensor object is replaced or modified in place."""
    cache = owner.__dict__.setdefault("_fwb_cache", {})
    hit = cache.get(name)
    if hit is not None and len(hit[0]) == len(srcs) and all(a is b and a._version == v for a, b, v in zip(hit[0], srcs, hit[1])):
        return hit[2]
    with torch.no_grad():
        val = fn(*srcs)
    cache[name] = (tuple(srcs), tuple(s._version for s in srcs), val)
    return val


def f32(owner, name, t):
    return derived(owner, "f32:" + name, lambda s: s.detach().float().contiguous().view(-1), t)


def w16(owner, name, t):
    """bf16 contiguous [N, K] view of a Linear / 1x1 conv weight."""
    return derived(owner, "w16:" + name, lambda s: s.detach().to(BF16).reshape(s.shape[0], -1).contiguous(), t)


def _pad8(n):
    return (n + 7) // 8 * 8


def lin(x, layer, *, tag="", **kw):
    """fwb200.linear on an nn.Linear / 1x1 conv's parameters (bias as cached fp32).  Shapes whose N or K is not a
    multiple of 8 (TMA needs 16-byte rows) are zero-padded — exact — and the result is sliced back."""
    wt = layer.weight
    N, K = wt.shape[0], wt[0].numel()
    if N % 8 == 0 and K % 8 == 0:
        w = w16(layer, tag + "w", wt)
        b = f32(layer, tag + "b", layer.bias) if layer.bias is not None else None
        return ops.linear(x, w, bias=b, **kw)
    Np, Kp = _pad8(N), _pad8(K)

    def padw(s):
        o = torch.zeros(Np, Kp, device=s.device, dtype=BF16)
        o[:N, :K] = s.detach().to(BF16).reshape(N, K)
        return o

    def padb(s):
        o = torch.zeros(Np, device=s.device, dtype=torch.float32)
        o[:N] = s.detach().float()
        return o

    w = derived(layer, tag + "wpad", padw, wt)
    b = derived(layer, tag + "bpad", padb, layer.bias) if layer.bias is not None else None
    assert not any(kw.get(k) is not None for k in ("scale1", "shift1", "scale2", "resid", "out")), "padded path: plain epilogue only"
    x2 = x.reshape(-1, K)
    if Kp != K:
        xp = torch.zeros(x2.shape[0], Kp, device=x.device, dtype=BF16)
        xp[:, :K] = x2
        x2 = xp
    y = ops.linear(x2, w, bias=b, **kw)
    return y[:, :N].contiguous().view(*x.shape[:-1], N)


def as_bf16(x):
    return x if x.dtype == BF16 else x.to(BF16)


# ------------------------------------------------------------------------------------------------------------------
# RoPE tables
# ------------------------------------------------------------------------------------------------------------------
_cs_cache = IdCache(16)
_r2d_cache = IdCache(8)


def complex_to_cos_sin(freqs: torch.Tensor, device) -> torch.Tensor:
    """complex [L, 1, hd/2] (reference layout) -> fp32 [L, hd/2, 2] (cos, sin) on `device`; cached per tensor object."""
    def build():
        f = freqs.reshape(freqs.shape[0], -1)
        return torch.stack([f.real, f.imag], dim=-1).to(torch.float32).contiguous().to(device)

    return _cs_cache.get((freqs,), str(device), build)


ROPE2D_FP32_ANGLES = bool(int(__import__("os").environ.get("FWB_ROPE2D_FP32_ANGLES", "0")))


def rope2d_expanded(pos: torch.Tensor, base: float = 100.0):
    """VGGT 2-D RoPE tables expanded per token: pos int [rows, 2] -> (cos, sin) fp32 [rows, 64].
    Same arithmetic as vggt/layers/rope.py:82-110,153-167 (integer gather of per-position tables).

    Rounding point: the reference builds the angle table with `torch.einsum("i,j->ij", positions, inv_freq)` on first use,
    i.e. INSIDE the sampler's `torch.cuda.amp.autocast(bf16)` region (inference_wan21.py:310), where einsum is an
    autocast-to-bf16 op: angle = bf16(bf16(pos) * bf16(inv_freq)), then cos/sin in fp32.  That is what the released
    weights were trained and are run with, so it is reproduced here explicitly (independent of any ambient autocast).
    FWB_ROPE2D_FP32_ANGLES=1 (or engine.ROPE2D_FP32_ANGLES = True) selects the reference's no-autocast (fp32) arithmetic.

    A position tensor whose base carries `_fwb_period` (Aggregator._positions at batch > 1: every sample has the same
    positions) gets tables of that many rows only; ops.ln64_rope2d_ applies them periodically."""
    fp32_angles = ROPE2D_FP32_ANGLES
    base_t = pos._base if pos._base is not None else pos   # views of one position tensor share the tables
    period = getattr(base_t, "_fwb_period", None)

    def build():
        p = pos.reshape(-1, 2).long()
        if period is not None:
            p = p[:period]
        dim = 32
        with torch.autocast(device_type=p.device.type, enabled=False):
            exponents = torch.arange(0, dim, 2, device=p.device).float() / dim
            inv_freq = 1.0 / (base ** exponents)
            max_pos = int(p.max()) + 1
            positions = torch.arange(max_pos, device=p.device, dtype=inv_freq.dtype)
            if fp32_angles:
                ang = positions[:, None] * inv_freq[None, :]
            else:
                ang = (positions.to(BF16)[:, None] * inv_freq.to(BF16)[None, :]).float()
            ang = torch.cat((ang, ang), dim=-1)
            cos_t, sin_t = ang.cos(), ang.sin()
            cosT = torch.cat([cos_t[p[:, 0]], cos_t[p[:, 1]]], dim=-1).contiguous()
            sinT = torch.cat([sin_t[p[:, 0]], sin_t[p[:, 1]]], dim=-1).contiguous()
        return cosT, sinT

    return _r2d_cache.get((base_t,), (pos.numel(), base, fp32_angles, period), build)


# ------------------------------------------------------------------------------------------------------------------
# batch: every sample of a call shares the timestep
# ------------------------------------------------------------------------------------------------------------------
SHARED_TIMESTEP_MSG = ("samples of one batch must share the timestep: the reference's joint_forward has no per-sample "
                       "timestep semantics (at timesteps [900, 500] its batch-2 outputs differ from its own batch-1 runs by up to 1.46)")


def shared_timestep(timestep: torch.Tensor, batch: int) -> torch.Tensor:
    """Validate the timestep of a batch-`batch` call and return it as one element ([1]).  A timestep with 1 element, or with
    `batch` equal elements, is accepted; anything else raises ValueError.  Pure tensor logic, checked before any launch."""
    t = timestep.reshape(-1)
    if t.numel() not in (1, batch):
        raise ValueError(f"timestep has {t.numel()} elements for a batch of {batch}: give 1, or {batch} equal values")
    if t.numel() > 1 and not bool((t == t[:1]).all()):
        raise ValueError(SHARED_TIMESTEP_MSG + f"; got {t.tolist()}")
    return t[:1]


def shared_rows(m: torch.Tensor, what: str) -> torch.Tensor:
    """m [B, ...] -> m[:1] when all B rows are equal (a shared timestep), else ValueError.  B == 1 is returned as is."""
    if m.shape[0] > 1 and not bool((m == m[:1]).all()):
        raise ValueError(f"{what}: " + SHARED_TIMESTEP_MSG)
    return m[:1]


def _heads(t, B, H, D):
    """[B*L, H*D] row view -> [B, L, H, D] view (no copy)."""
    return t.unflatten(1, (H, D)).unflatten(0, (B, -1))


# ------------------------------------------------------------------------------------------------------------------
# DiT block pieces (reference: diffsynth_wan21/models/wan_video_dit.py DiTBlock / SelfAttention / CrossAttention)
# ------------------------------------------------------------------------------------------------------------------
def dit_mod_vectors(block, t_mod):
    """(modulation + t_mod).chunk(6) as fp32 vectors: shift, (1+scale) [rounded to bf16 first], gate — twice.
    t_mod [B, 6, C] must have equal rows (shared timestep, see shared_timestep)."""
    m = shared_rows(block.modulation.to(BF16) + t_mod.to(BF16), "dit_mod_vectors")  # [1, 6, C] bf16 add, as under autocast
    one_plus = (1 + m[0, [1, 4]]).float()              # bf16(1 + scale)
    mf = m[0].float()
    return dict(shift_msa=mf[0].contiguous(), mul_msa=one_plus[0].contiguous(), gate_msa=mf[2].contiguous(),
                shift_mlp=mf[3].contiguous(), mul_mlp=one_plus[1].contiguous(), gate_mlp=mf[5].contiguous())


def dit_self_attn(sa, h, cos_sin, x_resid, gate, n_batch=1):
    """x_resid + gate * o(attn(rope(norm_q(q(h))), rope(norm_k(k(h))), v(h)))  — wan_video_dit.py:175-182, 301.
    h [n_batch * L, C]: each sample attends over its own L tokens; cos_sin holds the L per-position rows."""
    rows = h.shape[0]
    H, D = sa.num_heads, sa.head_dim
    C = H * D
    if SP is None:
        q = lin(h, sa.q)
        k = lin(h, sa.k)
        v = lin(h, sa.v)
        ops.rmsnorm_rope_(q, w=f32(sa.norm_q, "w", sa.norm_q.weight), eps=sa.norm_q.eps, cos_sin=cos_sin, head_dim=D)
        ops.rmsnorm_rope_(k, w=f32(sa.norm_k, "w", sa.norm_k.weight), eps=sa.norm_k.eps, cos_sin=cos_sin, head_dim=D)
        o = ops.attention(_heads(q, n_batch, H, D), _heads(k, n_batch, H, D), _heads(v, n_batch, H, D))
    else:
        # sequence parallel: h holds this rank's L/P tokens.  K and V are written side by side into one packed buffer so
        # that a single exchange moves both; queries stay local.
        L = rows
        kv = torch.empty((L, 2 * C), device=h.device, dtype=BF16)
        lin(h, sa.k, out=kv[:, :C])
        lin(h, sa.v, out=kv[:, C:])
        ops.rmsnorm_rope_(kv[:, :C], w=f32(sa.norm_k, "w", sa.norm_k.weight), eps=sa.norm_k.eps, cos_sin=cos_sin, head_dim=D)
        rows = SP.layout.video_rows
        S = SP.kv_chunks if (len(set(rows)) == 1 and L >= 256 * SP.kv_chunks) else 1

        def heads(t):
            return t.unflatten(1, (H, D)).unsqueeze(0)

        if S == 1:
            kv_all = SP.all_gather_rows(kv, rows)
            q = ops.rmsnorm_rope_(lin(h, sa.q), w=f32(sa.norm_q, "w", sa.norm_q.weight), eps=sa.norm_q.eps, cos_sin=cos_sin, head_dim=D)
            o = ops.attention(q.view(1, L, H, D), heads(kv_all[:, :C]), heads(kv_all[:, C:]))
        else:
            # pipelined exchange: gather the K|V rows in S slices on a side stream; the q projection and then the attention
            # over slice c (split-KV partials) run while slice c+1 is still in flight; one merge at the end.  Keys form a set,
            # so the slice order is irrelevant to the result.
            pending = SP.gather_chunks_async(kv, S)
            q = ops.rmsnorm_rope_(lin(h, sa.q), w=f32(sa.norm_q, "w", sa.norm_q.weight), eps=sa.norm_q.eps, cos_sin=cos_sin, head_dim=D)
            q4 = q.view(1, L, H, D)
            part = torch.empty((S, 1, L, H, D), device=h.device, dtype=torch.float32)
            lse = torch.empty((S, 1, H, L), device=h.device, dtype=torch.float32)
            main = torch.cuda.current_stream()
            for c, (buf, ev) in enumerate(pending):
                main.wait_event(ev)
                ops.attention_partial(q4, heads(buf[:, :C]), heads(buf[:, C:]), part[c], lse[c])
            o = ops.attention_merge(part, lse)
    return lin(o.view(rows, C), sa.o, scale1=gate, resid=x_resid, round_flags=ROUND_AFTER_BIAS | ROUND_AFTER_AFFINE)


def cross_kv(ca, context):
    """Loop-invariant K/V of the text / CLIP context (SURVEY Appendix E) — cached per context tensor.
    context [B, n_ctx, C] -> per-sample K/V [B, n, H, D] (text, then CLIP or None)."""
    cache = ca.__dict__.get("_fwb_kv")
    if cache is None:
        cache = ca.__dict__["_fwb_kv"] = IdCache(4)

    def build():
        ctx = as_bf16(context)
        B, C = ctx.shape[0], ctx.shape[-1]
        H, D = ca.num_heads, ca.head_dim
        if ca.has_image_input:
            img, txt = ctx[:, :257], ctx[:, 257:]
        else:
            img, txt = None, ctx
        txt = txt.reshape(-1, C).contiguous()
        k = lin(txt, ca.k)
        ops.rmsnorm_rope_(k, w=f32(ca.norm_k, "w", ca.norm_k.weight), eps=ca.norm_k.eps)
        v = lin(txt, ca.v)
        out = [k.view(B, -1, H, D), v.view(B, -1, H, D), None, None]
        if img is not None:
            img = img.reshape(-1, C).contiguous()
            ki = lin(img, ca.k_img)
            ops.rmsnorm_rope_(ki, w=f32(ca.norm_k_img, "w", ca.norm_k_img.weight), eps=ca.norm_k_img.eps)
            vi = lin(img, ca.v_img)
            out[2], out[3] = ki.view(B, -1, H, D), vi.view(B, -1, H, D)
        return out

    srcs = (context, ca.k.weight, ca.v.weight)
    return cache.get(srcs, None, build)


def dit_cross_attn_core(ca, n3, context):
    """q-projection + text attention (+ CLIP attention, summed in bf16) — wan_video_dit.py:185-201.  n3 [B * L, C] against the
    context of each sample ([B, n_ctx, C]).  Returns [B * L, C]."""
    rows = n3.shape[0]
    H, D = ca.num_heads, ca.head_dim
    k, v, ki, vi = cross_kv(ca, context)
    if rows % k.shape[0]:
        raise ValueError(f"cross attention: {rows} query rows do not split over a context batch of {k.shape[0]}")
    q = lin(n3, ca.q)
    ops.rmsnorm_rope_(q, w=f32(ca.norm_q, "w", ca.norm_q.weight), eps=ca.norm_q.eps)
    q4 = _heads(q, k.shape[0], H, D)
    o = ops.attention(q4, k, v)
    if ki is not None:
        ops.attention(q4, ki, vi, out=o, accumulate=True)
    return o.view(rows, H * D)


def dit_ffn(block, x, mods):
    """x + gate_mlp * ffn(modulate(norm2(x)))  — wan_video_dit.py:288-294."""
    h = ops.ln_modulate(x, eps=block.norm2.eps, mul=mods["mul_mlp"], add=mods["shift_mlp"])
    h = lin(h, block.ffn[0], act=ACT_GELU_TANH, round_flags=ROUND_AFTER_BIAS | ROUND_AFTER_ACT)
    return lin(h, block.ffn[2], scale1=mods["gate_mlp"], resid=x, round_flags=ROUND_AFTER_BIAS | ROUND_AFTER_AFFINE)


# ------------------------------------------------------------------------------------------------------------------
# VGGT block pieces (reference: vggt/layers/block.py Block, vggt/layers/attention.py Attention)
# ------------------------------------------------------------------------------------------------------------------
def vggt_mod_vectors(block, e0):
    """(modulation + e0).chunk(6) in fp32 — vggt/layers/block.py:95-104.  e0 [B, 6, C] must have equal rows (shared timestep)."""
    assert e0 is not None
    e = shared_rows(block.modulation.float() + e0.float(), "vggt_mod_vectors")[0]  # [6, C]
    return dict(add1=e[0].contiguous(), mul1=(1 + e[1]).contiguous(), add2=e[3].contiguous(),
                mul2=(1 + e[4]).contiguous(), e5=e[5].contiguous())


def vggt_attn_part(block, x, tables, mods, n_batch):
    """x + ls1(proj(attn(norm1(x)*(1+e1)+e0)))  with x [rows, C] (rows = n_batch * tokens) — block.py:73-76."""
    rows, C = x.shape
    at = block.attn
    H = at.num_heads
    mul = mods["mul1"] if mods is not None else None
    add = mods["add1"] if mods is not None else None
    h = ops.ln_modulate(x, eps=block.norm1.eps, w=f32(block.norm1, "w", block.norm1.weight),
                        b=f32(block.norm1, "b", block.norm1.bias), mul=mul, add=add)
    qkv = lin(h, at.qkv)
    if tables is not None:  # aggregator configuration: per-head LayerNorm(64) + 2-D RoPE on q, k
        cosT, sinT = tables
        ops.ln64_rope2d_(qkv, H, eps=at.q_norm.eps, qw=f32(at.q_norm, "w", at.q_norm.weight),
                         qb=f32(at.q_norm, "b", at.q_norm.bias), kw=f32(at.k_norm, "w", at.k_norm.weight),
                         kb=f32(at.k_norm, "b", at.k_norm.bias), cosT=cosT, sinT=sinT)
    q5 = qkv.view(n_batch, rows // n_batch, 3, H, C // H)
    if SP is not None and SP_GLOBAL_ATTN:
        # global attention under sequence parallelism: local queries, K|V gathered from the frame-aligned shards
        kv_all = SP.all_gather_rows(qkv[:, C:].contiguous(), SP.layout.geo_rows())
        o = ops.attention(q5[:, :, 0], kv_all[:, :C].unflatten(1, (H, C // H)).unsqueeze(0),
                          kv_all[:, C:].unflatten(1, (H, C // H)).unsqueeze(0))
    else:
        o = ops.attention(q5[:, :, 0], q5[:, :, 1], q5[:, :, 2])
    gamma = f32(block.ls1, "g", block.ls1.gamma)
    return lin(o.view(rows, C), at.proj, scale1=gamma, resid=x, out_dtype=x.dtype,
               round_flags=ROUND_AFTER_BIAS | ROUND_AFTER_AFFINE)


def vggt_ffn_part(block, x, mods):
    """x + ls2(mlp(norm2(x)) * (1+e4) + e3) * e5  (modulation AFTER the MLP; fp32 stream) — block.py:78-81."""
    h = ops.ln_modulate(x, eps=block.norm2.eps, w=f32(block.norm2, "w", block.norm2.weight),
                        b=f32(block.norm2, "b", block.norm2.bias))
    h = lin(h, block.mlp.fc1, act=ACT_GELU_ERF, round_flags=ROUND_AFTER_BIAS | ROUND_AFTER_ACT)
    gamma = f32(block.ls2, "g", block.ls2.gamma)
    if mods is None:
        return lin(h, block.mlp.fc2, scale1=gamma, resid=x, out_dtype=x.dtype,
                   round_flags=ROUND_AFTER_BIAS | ROUND_AFTER_AFFINE)
    return lin(h, block.mlp.fc2, scale1=mods["mul2"], shift1=mods["add2"], scale2=gamma * mods["e5"], resid=x,
               out_dtype=torch.float32, round_flags=ROUND_AFTER_BIAS)


# ------------------------------------------------------------------------------------------------------------------
# bidirectional adapter (reference: fusion/layer/block.py CrossModalityBiAttentionBlock / BiMultiHeadAttention)
# ------------------------------------------------------------------------------------------------------------------
def bicross(blk, x1, x2, cs_dit, cs_agg, n_batch=1):
    """x1 [B*L1, C1] bf16 (video), x2 [B*L2, C2] fp32|bf16 (geometry) -> updated (x1, x2); sample b's video tokens attend to
    sample b's geometry tokens and back.  cs_dit / cs_agg hold the L1 / L2 per-position rows."""
    ca = blk.cross_attn
    H, D, E = ca.num_heads, ca.head_dim, ca.embed_dim
    L1, L2 = x1.shape[0], x2.shape[0]
    n1 = ops.ln_modulate(x1, eps=blk.attn_norm_m1.eps)
    n2 = ops.ln_modulate(x2, eps=blk.attn_norm_m2.eps)
    # one GEMM per stream: [q | v1] and [k | v2]
    w1 = derived(ca, "w_qv1", lambda a, b: torch.cat([a, b], 0).to(BF16).contiguous(), ca.m1_proj.weight, ca.values_m1_proj.weight)
    b1 = derived(ca, "b_qv1", lambda a, b: torch.cat([a, b], 0).float().contiguous(), ca.m1_proj.bias, ca.values_m1_proj.bias)
    w2 = derived(ca, "w_kv2", lambda a, b: torch.cat([a, b], 0).to(BF16).contiguous(), ca.m2_proj.weight, ca.values_m2_proj.weight)
    b2 = derived(ca, "b_kv2", lambda a, b: torch.cat([a, b], 0).float().contiguous(), ca.m2_proj.bias, ca.values_m2_proj.bias)
    qv1 = ops.linear(n1, w1, bias=b1)
    kv2 = ops.linear(n2, w2, bias=b2)
    ops.rmsnorm_rope_(qv1[:, :E], cos_sin=cs_dit, head_dim=D)
    ops.rmsnorm_rope_(kv2[:, :E], cos_sin=cs_agg, head_dim=D)
    q = _heads(qv1[:, :E], n_batch, H, D)
    v1 = _heads(qv1[:, E:], n_batch, H, D)
    k = _heads(kv2[:, :E], n_batch, H, D)
    v2 = _heads(kv2[:, E:], n_batch, H, D)
    if SP is None:
        o1 = ops.attention(q, k, v2)   # video <- geometry
        o2 = ops.attention(k, q, v1)   # geometry <- video
    else:
        def heads(t):
            return t.unflatten(1, (H, D)).unsqueeze(0)

        # both exchanges start on the side stream; the [q|v1] rows (needed by the geometry queries) travel in slices while the
        # video queries already attend over the gathered [k|v2]
        finish_kv2 = SP.all_gather_rows_async(kv2, SP.layout.geo_rows())                 # ragged frame-aligned shards
        rows = SP.layout.video_rows
        S = SP.kv_chunks if (len(set(rows)) == 1 and L1 >= 256 * SP.kv_chunks) else 1
        if S == 1:
            finish_qv1 = SP.all_gather_rows_async(qv1, rows)
            kv2_all = finish_kv2()                                                        # [N, 2E]
            o1 = ops.attention(q, heads(kv2_all[:, :E]), heads(kv2_all[:, E:]))           # local video queries x all geometry keys
            qv1_all = finish_qv1()                                                        # [L, 2E]
            o2 = ops.attention(k, heads(qv1_all[:, :E]), heads(qv1_all[:, E:]))           # local geometry queries x all video keys
        else:
            pending = SP.gather_chunks_async(qv1, S)
            kv2_all = finish_kv2()
            o1 = ops.attention(q, heads(kv2_all[:, :E]), heads(kv2_all[:, E:]))
            part = torch.empty((S, 1, L2, H, D), device=x1.device, dtype=torch.float32)
            lse = torch.empty((S, 1, H, L2), device=x1.device, dtype=torch.float32)
            main = torch.cuda.current_stream()
            for c, (buf, ev) in enumerate(pending):
                main.wait_event(ev)
                ops.attention_partial(k, heads(buf[:, :E]), heads(buf[:, E:]), part[c], lse[c])
            o2 = ops.attention_merge(part, lse)
    rf = ROUND_AFTER_BIAS | ROUND_AFTER_AFFINE
    x1 = lin(o1.view(L1, E), ca.out_m1_proj, scale1=f32(blk, "g1", blk.gamma_m1), resid=x1, round_flags=rf)
    x2 = lin(o2.view(L2, E), ca.out_m2_proj, scale1=f32(blk, "g2", blk.gamma_m2), resid=x2, out_dtype=x2.dtype,
             round_flags=rf)
    return x1, x2


# small MLPs on a handful of rows (time embeddings etc.)
def mlp_silu(x, l0, l2):
    h = lin(as_bf16(x), l0, act=ACT_SILU, round_flags=ROUND_AFTER_BIAS | ROUND_AFTER_ACT)
    return lin(h, l2, round_flags=ROUND_AFTER_BIAS)


__all__ = [n for n in dir() if not n.startswith("_")]
