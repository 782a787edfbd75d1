"""B200-native mirror of FantasyWorld/diffsynth_wan21/models/wan_video_dit.py (reference).

Same public names, constructor / forward signatures and state_dict keys as the reference module; the bodies are
written from scratch and run the token-sized work on the fwb200 sm_100a kernels (tcgen05 GEMM + flash attention,
fused LN/RMSNorm/RoPE).  No flash-attn / SDPA / cuBLAS dispatch, no CPU fallback: forward() needs a B200.

Reference call sites replaced are cited inline as `ref: wan_video_dit.py:<line>`.
"""
from __future__ import annotations

import math
from typing import Optional, Tuple

import torch
import torch.nn as nn

from fwb200 import engine as E
from fwb200 import ops

BF16 = torch.bfloat16


# ----------------------------------------------------------------------------------------------------------------------
# functional API kept for compatibility with callers of the reference module
# ----------------------------------------------------------------------------------------------------------------------
def flash_attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, num_heads: int, compatibility_mode=False):
    """[b, s, (n d)] attention through fwb_attn_fwd.  ref: wan_video_dit.py:28-66 (backend dispatch removed)."""
    b, s, c = q.shape
    d = c // num_heads
    o = ops.attention(E.as_bf16(q).view(b, s, num_heads, d), E.as_bf16(k).view(b, -1, num_heads, d),
                      E.as_bf16(v).view(b, -1, num_heads, d))
    return o.view(b, s, c)


def modulate(x: torch.Tensor, shift: torch.Tensor, scale: torch.Tensor):
    return x * (1 + scale) + shift


def sinusoidal_embedding_1d(dim, position):
    """cos|sin embedding evaluated in fp64, returned in position.dtype.  ref: wan_video_dit.py:73-77."""
    half = dim // 2
    inv = torch.pow(10000.0, -torch.arange(half, dtype=torch.float64, device=position.device) / half)
    ang = position.to(torch.float64)[:, None] * inv[None, :]
    return torch.cat([ang.cos(), ang.sin()], dim=1).to(position.dtype)


def precompute_freqs_cis(dim: int, end: int = 1024, theta: float = 10000.0):
    """complex128 table [end, dim // 2].  ref: wan_video_dit.py:88-94."""
    idx = torch.arange(0, dim, 2)[: dim // 2].double()
    ang = torch.outer(torch.arange(end).double(), 1.0 / (theta ** (idx / dim)))
    return torch.polar(torch.ones_like(ang), ang)


def precompute_freqs_cis_3d(dim: int, end: int = 1024, theta: float = 10000.0):
    """(f, h, w) tables with the head dim split (dim - 2*(dim//3), dim//3, dim//3).  ref: wan_video_dit.py:80-85."""
    third = dim // 3
    return (precompute_freqs_cis(dim - 2 * third, end, theta), precompute_freqs_cis(third, end, theta),
            precompute_freqs_cis(third, end, theta))


def _grid_freqs(freqs_3d, f, h, w):
    tf, th, tw = freqs_3d
    parts = (tf[:f].view(f, 1, 1, -1).expand(f, h, w, -1), th[:h].view(1, h, 1, -1).expand(f, h, w, -1),
             tw[:w].view(1, 1, w, -1).expand(f, h, w, -1))
    return torch.cat(parts, dim=-1)


def build_freqs_3d_with_extra_cis(freqs_3d, f: int, h: int, w: int, n_extra: int, device=None):
    """Per-frame [n_extra identity rotations | h*w patch rotations] -> [f*(n_extra+h*w), 1, D/2].
    ref: wan_video_dit.py:105-132."""
    patch = _grid_freqs(freqs_3d, f, h, w).reshape(f, h * w, -1)
    ident = torch.ones(f, n_extra, patch.shape[-1], dtype=patch.dtype, device=patch.device)
    full = torch.cat([ident, patch], dim=1).reshape(f * (n_extra + h * w), 1, -1)
    return full.to(device) if device is not None else full


def rope_apply(x, freqs, num_heads):
    """Interleaved-pair RoPE through fwb_rmsnorm_rope (norm disabled).  ref: wan_video_dit.py:97-102."""
    b, s, c = x.shape
    d = c // num_heads
    y = E.as_bf16(x).clone().view(b * s, c)
    cs = E.complex_to_cos_sin(freqs, x.device)          # [s] rows, applied to every sample
    ops.rmsnorm_rope_(y, cos_sin=cs, head_dim=d)
    return y.view(b, s, c).to(x.dtype)


# ----------------------------------------------------------------------------------------------------------------------
# modules
# ----------------------------------------------------------------------------------------------------------------------
class RMSNorm(nn.Module):
    """Full-channel RMSNorm.  In the fused block path it is folded into fwb_rmsnorm_rope; this forward is the
    standalone form.  ref: wan_video_dit.py:135-146."""

    def __init__(self, dim, eps=1e-5):
        super().__init__()
        self.eps = eps
        self.weight = nn.Parameter(torch.ones(dim))

    def forward(self, x):
        y = E.as_bf16(x).clone().view(-1, x.shape[-1])
        ops.rmsnorm_rope_(y, w=E.f32(self, "w", self.weight), eps=self.eps)
        return y.view(x.shape).to(x.dtype)


class AttentionModule(nn.Module):
    def __init__(self, num_heads):
        super().__init__()
        self.num_heads = num_heads

    def forward(self, q, k, v):
        return flash_attention(q=q, k=k, v=v, num_heads=self.num_heads)


class SelfAttention(nn.Module):
    """ref: wan_video_dit.py:159-182."""

    def __init__(self, dim: int, num_heads: int, eps: float = 1e-6):
        super().__init__()
        self.dim, self.num_heads, self.head_dim = dim, num_heads, dim // num_heads
        self.q = nn.Linear(dim, dim)
        self.k = nn.Linear(dim, dim)
        self.v = nn.Linear(dim, dim)
        self.o = nn.Linear(dim, dim)
        self.norm_q = RMSNorm(dim, eps=eps)
        self.norm_k = RMSNorm(dim, eps=eps)
        self.attn = AttentionModule(self.num_heads)

    def forward(self, x, freqs):
        b, s, c = x.shape
        h = E.as_bf16(x).reshape(b * s, c)
        cs = E.complex_to_cos_sin(freqs, x.device)
        q, k, v = E.lin(h, self.q), E.lin(h, self.k), E.lin(h, self.v)
        ops.rmsnorm_rope_(q, w=E.f32(self.norm_q, "w", self.norm_q.weight), eps=self.norm_q.eps, cos_sin=cs, head_dim=self.head_dim)
        ops.rmsnorm_rope_(k, w=E.f32(self.norm_k, "w", self.norm_k.weight), eps=self.norm_k.eps, cos_sin=cs, head_dim=self.head_dim)
        o = ops.attention(q.view(b, s, self.num_heads, -1), k.view(b, s, self.num_heads, -1), v.view(b, s, self.num_heads, -1))
        return E.lin(o.view(b * s, c), self.o, round_flags=ops.ROUND_AFTER_BIAS).view(b, s, c)


class CrossAttentionProcessor:
    """Text (+CLIP) cross attention followed by the output projection.  ref: wan_video_dit.py:185-201."""

    def __call__(self, attn, x: torch.Tensor, y: torch.Tensor):
        b, s, c = x.shape
        o = E.dit_cross_attn_core(attn, E.as_bf16(x).reshape(b * s, c), y)
        return E.lin(o, attn.o, round_flags=ops.ROUND_AFTER_BIAS).view(b, s, c)

    # fused-block hook: returns o(o_attn) + resid without materialising the intermediate
    def fused(self, attn, n3, context, x_resid, **kwargs):
        o = E.dit_cross_attn_core(attn, n3, context)
        return E.lin(o, attn.o, resid=x_resid, round_flags=ops.ROUND_AFTER_BIAS)


class CrossAttention(nn.Module):
    """ref: wan_video_dit.py:204-243."""

    def __init__(self, dim: int, num_heads: int, eps: float = 1e-6, has_image_input: bool = False):
        super().__init__()
        self.dim, self.num_heads, self.head_dim = dim, num_heads, dim // num_heads
        self.q = nn.Linear(dim, dim)
        self.k = nn.Linear(dim, dim)
        self.v = nn.Linear(dim, dim)
        self.o = nn.Linear(dim, dim)
        self.norm_q = RMSNorm(dim, eps=eps)
        self.norm_k = RMSNorm(dim, eps=eps)
        self.has_image_input = has_image_input
        if has_image_input:
            self.k_img = nn.Linear(dim, dim)
            self.v_img = nn.Linear(dim, dim)
            self.norm_k_img = RMSNorm(dim, eps=eps)
        self.attn = AttentionModule(self.num_heads)
        self.set_processor(CrossAttentionProcessor())

    def set_processor(self, processor):
        self.processor = processor

    def get_processor(self):
        return self.processor

    def forward(self, x: torch.Tensor, y: torch.Tensor, **kwargs):
        if isinstance(self.processor, CrossAttentionProcessor):
            return self.processor(self, x, y)
        return self.processor(self, x, y, **kwargs)


class GateModule(nn.Module):
    """x + gate * residual (folded into the GEMM epilogues in the fused path).  ref: wan_video_dit.py:246-251."""

    def forward(self, x, gate, residual):
        return x + gate * residual


class DiTBlock(nn.Module):
    """WanDiT block with the reference's split-forward switches.  ref: wan_video_dit.py:254-321.

    Kernel sequence per call (L tokens, C = 5120):
      ln_modulate -> q,k,v GEMMs -> rmsnorm_rope x2 -> attention -> o GEMM(+gate,+resid)
      ln(affine) -> q GEMM -> rmsnorm -> attention(text) -> attention(CLIP, accumulate) [-> camera AdaLN GEMMs]
      -> o GEMM(+resid) | ln_modulate -> ffn.0 GEMM(+GELU) -> ffn.2 GEMM(+gate,+resid)
    """

    def __init__(self, has_image_input: bool, dim: int, num_heads: int, ffn_dim: int, eps: float = 1e-6):
        super().__init__()
        self.dim, self.num_heads, self.ffn_dim = dim, num_heads, ffn_dim
        self.self_attn = SelfAttention(dim, num_heads, eps)
        self.cross_attn = CrossAttention(dim, num_heads, eps, has_image_input=has_image_input)
        self.norm1 = nn.LayerNorm(dim, eps=eps, elementwise_affine=False)
        self.norm2 = nn.LayerNorm(dim, eps=eps, elementwise_affine=False)
        self.norm3 = nn.LayerNorm(dim, eps=eps)
        self.ffn = nn.Sequential(nn.Linear(dim, ffn_dim), nn.GELU(approximate='tanh'), nn.Linear(ffn_dim, dim))
        self.modulation = nn.Parameter(torch.randn(1, 6, dim) / dim ** 0.5)
        self.gate = GateModule()

    def forward(self, x, context=None, t_mod=None, freqs=None, *, return_partial: bool = False,
                run_remaining: bool = False, modifiers: tuple | None = None, **kwargs):
        b, s, c = x.shape
        xs = E.as_bf16(x).reshape(b * s, c)
        if run_remaining:
            assert modifiers is not None, "modifiers must provide"
            return E.dit_ffn(self, xs, modifiers).view(b, s, c)

        mods = E.dit_mod_vectors(self, t_mod)
        cs = E.complex_to_cos_sin(freqs, x.device)
        if E.SP is not None and cs.shape[0] != s:      # sequence parallel: x holds this rank's rows of the token grid
            r0, r1 = E.SP.layout.video_range(E.SP.rank)
            cs = cs[r0:r1]
        h = ops.ln_modulate(xs, eps=self.norm1.eps, mul=mods["mul_msa"], add=mods["shift_msa"])
        xs = E.dit_self_attn(self.self_attn, h, cs, xs, mods["gate_msa"], n_batch=b)
        n3 = ops.ln_modulate(xs, eps=self.norm3.eps, w=E.f32(self.norm3, "w", self.norm3.weight),
                             b=E.f32(self.norm3, "b", self.norm3.bias))
        proc = self.cross_attn.processor
        xs = proc.fused(self.cross_attn, n3, context, xs, **kwargs)
        if return_partial:
            return xs.view(b, s, c), mods
        if modifiers is not None:
            mods = modifiers
        return E.dit_ffn(self, xs, mods).view(b, s, c)

    def forward_partial(self, *args, **kwargs):
        return self.forward(*args, **kwargs, return_partial=True)

    def forward_remaining(self, x, shift_mlp, scale_mlp, gate_mlp):
        raise NotImplementedError("use forward(run_remaining=True, modifiers=<dict returned by return_partial>)")


class MLP(torch.nn.Module):
    """CLIP feature projector: LN, Linear, GELU, Linear, LN.  ref: wan_video_dit.py:324-341."""

    def __init__(self, in_dim, out_dim, has_pos_emb=False):
        super().__init__()
        self.proj = torch.nn.Sequential(nn.LayerNorm(in_dim), nn.Linear(in_dim, in_dim), nn.GELU(),
                                        nn.Linear(in_dim, out_dim), nn.LayerNorm(out_dim))
        self.has_pos_emb = has_pos_emb
        if has_pos_emb:
            self.emb_pos = torch.nn.Parameter(torch.zeros((1, 514, 1280)))

    def forward(self, x):
        if self.has_pos_emb:
            x = x + self.emb_pos.to(dtype=x.dtype, device=x.device)
        shp = x.shape
        ln0, l1, _, l3, ln4 = self.proj
        h = ops.ln_modulate(x.reshape(-1, shp[-1]), eps=ln0.eps, w=E.f32(ln0, "w", ln0.weight), b=E.f32(ln0, "b", ln0.bias))
        h = E.lin(h, l1, act=ops.ACT_GELU_ERF, round_flags=ops.ROUND_AFTER_BIAS | ops.ROUND_AFTER_ACT)
        h = E.lin(h, l3, round_flags=ops.ROUND_AFTER_BIAS)
        h = ops.ln_modulate(h, eps=ln4.eps, w=E.f32(ln4, "w", ln4.weight), b=E.f32(ln4, "b", ln4.bias))
        return h.view(*shp[:-1], -1)


class Head(nn.Module):
    """ref: wan_video_dit.py:344-358."""

    def __init__(self, dim: int, out_dim: int, patch_size: Tuple[int, int, int], eps: float):
        super().__init__()
        self.dim, self.patch_size = dim, patch_size
        self.norm = nn.LayerNorm(dim, eps=eps, elementwise_affine=False)
        self.head = nn.Linear(dim, out_dim * math.prod(patch_size))
        self.modulation = nn.Parameter(torch.randn(1, 2, dim) / dim ** 0.5)

    def forward(self, x, t_mod):
        b, s, c = x.shape
        t_mod = E.shared_rows(t_mod.reshape(-1, 1, c), "Head")                                      # shared timestep
        m = self.modulation.to(dtype=t_mod.dtype, device=t_mod.device) + t_mod  # [1,2,C]
        shift = m[0, 0].float().contiguous()
        mul = (1 + m[0, 1]).float().contiguous()
        h = ops.ln_modulate(E.as_bf16(x).reshape(b * s, c), eps=self.norm.eps, mul=mul, add=shift)
        return E.lin(h, self.head, round_flags=ops.ROUND_AFTER_BIAS).view(b, s, -1)


class WanModel(torch.nn.Module):
    """ref: wan_video_dit.py:361-560."""

    def __init__(self, dim: int, in_dim: int, ffn_dim: int, out_dim: int, text_dim: int, freq_dim: int, eps: float,
                 patch_size: Tuple[int, int, int], num_heads: int, num_layers: int, has_image_input: bool,
                 has_image_pos_emb: bool = False, has_ref_conv: bool = False, add_control_adapter: bool = False,
                 in_dim_control_adapter: int = 24):
        super().__init__()
        self.dim, self.freq_dim, self.has_image_input, self.patch_size = dim, freq_dim, has_image_input, patch_size
        self.patch_embedding = nn.Conv3d(in_dim, dim, kernel_size=patch_size, stride=patch_size)
        self.text_embedding = nn.Sequential(nn.Linear(text_dim, dim), nn.GELU(approximate='tanh'), nn.Linear(dim, dim))
        self.time_embedding = nn.Sequential(nn.Linear(freq_dim, dim), nn.SiLU(), nn.Linear(dim, dim))
        self.time_projection = nn.Sequential(nn.SiLU(), nn.Linear(dim, dim * 6))
        self.blocks = nn.ModuleList([DiTBlock(has_image_input, dim, num_heads, ffn_dim, eps) for _ in range(num_layers)])
        self.head = Head(dim, out_dim, patch_size, eps)
        self.freqs = precompute_freqs_cis_3d(dim // num_heads)
        if has_image_input:
            self.img_emb = MLP(1280, dim, has_pos_emb=has_image_pos_emb)
        if has_ref_conv:
            self.ref_conv = nn.Conv2d(16, dim, kernel_size=(2, 2), stride=(2, 2))
        self.has_image_pos_emb, self.has_ref_conv = has_image_pos_emb, has_ref_conv
        if add_control_adapter:
            from .wan_video_camera_controller import SimpleAdapter
            self.control_adapter = SimpleAdapter(in_dim_control_adapter, dim, kernel_size=patch_size[1:], stride=patch_size[1:])
        else:
            self.control_adapter = None

    # -- embeddings ---------------------------------------------------------------------------------------------------
    def embed_time(self, timestep):
        """t [1, dim] and t_mod [1, 6, dim] (bf16).  ref: model_wan21.py:119-122 / wan_video_dit.py:468-470."""
        s = sinusoidal_embedding_1d(self.freq_dim, timestep)
        t = E.mlp_silu(s, self.time_embedding[0], self.time_embedding[2])
        tp = E.lin(torch.nn.functional.silu(t), self.time_projection[1], round_flags=ops.ROUND_AFTER_BIAS)
        return t, tp.unflatten(1, (6, self.dim))

    def embed_text(self, context):
        """ref: wan_video_dit.py:387-391, 471."""
        shp = context.shape
        h = E.lin(E.as_bf16(context).reshape(-1, shp[-1]), self.text_embedding[0], act=ops.ACT_GELU_TANH,
                  round_flags=ops.ROUND_AFTER_BIAS | ops.ROUND_AFTER_ACT)
        return E.lin(h, self.text_embedding[2], round_flags=ops.ROUND_AFTER_BIAS).view(*shp[:-1], self.dim)

    # -- token <-> latent layout --------------------------------------------------------------------------------------
    def patchify(self, x: torch.Tensor, control_camera_latents_input: torch.Tensor = None):
        """Conv3d(k = s = patch) as one GEMM over unfolded patches; tokens in (f h w) order.
        ref: wan_video_dit.py:424-435."""
        b, cin, F_, H_, W_ = x.shape
        pf, ph, pw = self.patch_size
        f, h, w = F_ // pf, H_ // ph, W_ // pw
        cols = E.as_bf16(x).view(b, cin, f, pf, h, ph, w, pw).permute(0, 2, 4, 6, 1, 3, 5, 7).reshape(b * f * h * w, cin * pf * ph * pw)
        tok = E.lin(cols.contiguous(), self.patch_embedding, round_flags=ops.ROUND_AFTER_BIAS)
        if self.control_adapter is not None and control_camera_latents_input is not None:
            y_camera = self.control_adapter(control_camera_latents_input)  # [b, dim, f, h, w]
            tok = tok + y_camera[0].permute(1, 2, 3, 0).reshape(f * h * w, -1).to(tok.dtype)
        return tok.view(b, f * h * w, self.dim), (f, h, w)

    def unpatchify(self, x: torch.Tensor, grid_size):
        """'b (f h w) (x y z c) -> b c (f x) (h y) (w z)'.  ref: wan_video_dit.py:437-442 (pure index shuffle)."""
        f, h, w = grid_size
        px, py, pz = self.patch_size
        b = x.shape[0]
        c = x.shape[-1] // (px * py * pz)
        return x.view(b, f, h, w, px, py, pz, c).permute(0, 7, 1, 4, 2, 5, 3, 6).reshape(b, c, f * px, h * py, w * pz)

    def grid_freqs(self, f, h, w, device):
        key = (f, h, w, str(device))
        cache = self.__dict__.setdefault("_freq_cache", {})
        if key not in cache:
            cache[key] = _grid_freqs(self.freqs, f, h, w).reshape(f * h * w, 1, -1).to(device)
        return cache[key]

    def forward(self, x: torch.Tensor, timestep: torch.Tensor, context: torch.Tensor,
                clip_feature: Optional[torch.Tensor] = None, y: Optional[torch.Tensor] = None,
                use_gradient_checkpointing: bool = False, use_gradient_checkpointing_offload: bool = False,
                plucker_fea: Optional[torch.Tensor] = None, plucker_context_lens: Optional[torch.Tensor] = None, **kwargs):
        """Plain WanDiT forward (all blocks).  ref: wan_video_dit.py:444-502."""
        t, t_mod = self.embed_time(timestep)
        context = self.embed_text(context)
        if self.has_image_input:
            x = torch.cat([x, y], dim=1)
            context = torch.cat([self.img_emb(clip_feature), context], dim=1)
        x, (f, h, w) = self.patchify(x)
        freqs = self.grid_freqs(f, h, w, x.device)
        kw = dict(plucker_fea=plucker_fea, plucker_context_lens=plucker_context_lens)
        for block in self.blocks:
            x = block(x, context, t_mod, freqs, **kw)
        return self.unpatchify(self.head(x, t), (f, h, w))

    # -- attention-processor plumbing (used by CameraConditionModel) -----------------------------------------------------
    @property
    def attn_processors(self):
        """{'blocks.<i>.cross_attn.processor': processor} for block index <= 24.  ref: wan_video_dit.py:508-529."""
        out = {}
        for name, module in self.named_modules():
            if hasattr(module, "set_processor") and "blocks." in name:
                if int(name.split("blocks.", 1)[1].split(".", 1)[0]) <= 24:
                    out[f"{name}.processor"] = module.processor
        return out

    def set_attn_processor(self, processor):
        """ref: wan_video_dit.py:531-572."""
        targets = self.attn_processors
        if isinstance(processor, dict) and len(processor) != len(targets):
            raise ValueError(f"A dict of processors was passed, but the number of processors {len(processor)} does not match "
                             f"the number of attention layers: {len(targets)}.")
        for name, module in self.named_modules():
            key = f"{name}.processor"
            if key in targets:
                module.set_processor(processor[key] if isinstance(processor, dict) else processor)
