"""B200-native mirror of FantasyWorld/fusion/layer/block.py (reference): the IRG (Integrated Reconstruction and
Generation) block = WanDiT block (Imagination-Prior branch) || VGGT global block (Geometry-Consistent branch), coupled
mid-block by a bidirectional cross-attention adapter.  Same class names, signatures and state_dict keys.

Adapter kernel sequence (fwb200): ln x2 -> [q|v1] GEMM, [k|v2] GEMM -> RoPE(q), RoPE(k) in place ->
attention(q,k,v2), attention(k,q,v1) -> out_m1 / out_m2 GEMMs with gamma*dx + residual fused in the epilogue.
Only the 'sdpa' numerics of the reference (the only implementation it actually uses, block.py:170) are provided.
"""
from __future__ import annotations

from typing import Literal, Optional, Tuple

import torch
import torch.nn as nn

from fwb200 import engine as E

from ...diffsynth_wan21.models.wan_video_dit import DiTBlock
from ...vggt.layers.block import Block


class BiMultiHeadAttention(nn.Module):
    """Two attentions over one score matrix: O1 = softmax(q k^T) v2 and O2 = softmax(k q^T) v1.
    ref: block.py:316-373 (parameters), 532-625 (forward_sdpa)."""

    def __init__(self, m1_dim, m2_dim, embed_dim, num_heads, dropout=0.0,
                 attn_implementation: Literal['eager', 'sdpa', 'flash_attn_2'] = 'sdpa'):
        super().__init__()
        self.embed_dim, self.num_heads, self.head_dim = embed_dim, num_heads, embed_dim // num_heads
        self.m1_dim, self.m2_dim = m1_dim, m2_dim
        assert self.head_dim * num_heads == embed_dim, "embed_dim must be divisible by num_heads"
        self.scale = self.head_dim ** (-0.5)
        self.dropout = dropout
        self.m1_proj = nn.Linear(m1_dim, embed_dim)
        self.m2_proj = nn.Linear(m2_dim, embed_dim)
        self.values_m1_proj = nn.Linear(m1_dim, embed_dim)
        self.values_m2_proj = nn.Linear(m2_dim, embed_dim)
        self.out_m1_proj = nn.Linear(embed_dim, m1_dim)
        self.out_m2_proj = nn.Linear(embed_dim, m2_dim)
        self.attn_implementation = attn_implementation
        for proj in (self.m1_proj, self.values_m1_proj, self.out_m1_proj, self.m2_proj, self.values_m2_proj, self.out_m2_proj):
            nn.init.xavier_uniform_(proj.weight)
            proj.bias.data.fill_(0)


class CrossModalityBiAttentionBlock(nn.Module):
    """x1 += gamma_m1 * dx1, x2 += gamma_m2 * dx2 with LayerNorm(no affine) inputs.  ref: block.py:146-221."""

    def __init__(self, m1_dim, m2_dim, hidden_size, num_heads, drop_path=0.0, enable_layernorm_kernel=False,
                 enable_flash_attn=False, init_values=1e-4, bica_mode: Literal['overall', 'temporal'] = 'overall'):
        super().__init__()
        if bica_mode != 'overall':
            raise NotImplementedError("only bica_mode='overall' (the reference's configuration) is implemented")
        self.m1_dim, self.m2_dim, self.hidden_size, self.num_heads = m1_dim, m2_dim, hidden_size, num_heads
        self.attn_norm_m1 = nn.LayerNorm(m1_dim, 1e-6, elementwise_affine=False)
        self.attn_norm_m2 = nn.LayerNorm(m2_dim, 1e-6, elementwise_affine=False)
        self.cross_attn = BiMultiHeadAttention(m1_dim, m2_dim, hidden_size, num_heads, dropout=0.0, attn_implementation='sdpa')
        self.gamma_m1 = nn.Parameter(torch.zeros(m1_dim), requires_grad=True)
        self.gamma_m2 = nn.Parameter(torch.zeros(m2_dim), requires_grad=True)
        self.drop_path = nn.Identity()
        self.bica_mode = bica_mode

    def forward(self, xs: Tuple[torch.Tensor], attention_masks: Optional[Tuple[torch.Tensor]] = (None, None), T: int = None,
                S: int = None, R: int = None, M: int = None, freqs=None, freqs_dit=None, freqs_agg=None):
        x1, x2 = xs
        if attention_masks[0] is not None or attention_masks[1] is not None:
            raise NotImplementedError('attention mask is currently unsupported for video-audio cross attention')
        B = x1.shape[0]
        if x2.shape[0] != B:
            raise ValueError(f"video batch {B} != geometry batch {x2.shape[0]}")
        a = E.as_bf16(x1).reshape(-1, x1.shape[-1])
        g = x2.reshape(-1, x2.shape[-1])
        if g.dtype not in (torch.float32, torch.bfloat16):
            g = g.float()
        cs_dit, cs_agg = E.complex_to_cos_sin(freqs_dit, x1.device), E.complex_to_cos_sin(freqs_agg, x1.device)
        if E.SP is not None:   # sequence parallel (batch 1): both streams hold this rank's rows only
            lay, rk = E.SP.layout, E.SP.rank
            if cs_dit.shape[0] != a.shape[0]:
                cs_dit = cs_dit[slice(*lay.video_range(rk))]
            if cs_agg.shape[0] != g.shape[0]:
                cs_agg = cs_agg[slice(*lay.geo_range(rk))]
        a, g = E.bicross(self, a, g, cs_dit, cs_agg, n_batch=B)
        return a.view(B, -1, a.shape[-1]), g.view(B, -1, g.shape[-1])


class IRGBlock(nn.Module):
    """ref: block.py:18-143."""

    def __init__(self, x_dit_block: DiTBlock, x_agg_block: Block, m1_dim, m2_dim, hidden_size, num_heads, drop_path=0.0,
                 enable_layernorm_kernel=False, enable_flash_attn=False, init_values=1e-4,
                 bica_mode: Literal['overall', 'temporal'] = 'overall'):
        super().__init__()
        self.x_dit = x_dit_block
        self.x_agg = x_agg_block
        self.bicross_attention = CrossModalityBiAttentionBlock(m1_dim, m2_dim, hidden_size, num_heads, drop_path=drop_path,
                                                               init_values=init_values, bica_mode=bica_mode)

    def forward(self, x_dit: torch.Tensor, x_agg: torch.Tensor, *, context: torch.Tensor, t_mod: torch.Tensor,
                freqs: torch.Tensor, freqs_dit: torch.Tensor, freqs_agg: torch.Tensor, pos: torch.Tensor | None = None,
                e0: torch.Tensor | None = None, uncond=False, **kwargs):
        """x_dit [B, L, 5120]; x_agg [(B S), P, 1024]; pos [(B S), P, 2].  Returns (x_dit, x_agg [B, S*P, C],
        [x_agg viewed as [B, S, P, C]]).  ref: block.py:43-94."""
        _, P, D = x_agg.shape
        B = x_dit.size(0)
        xd, mod_dit = self.x_dit(x_dit, context, t_mod, freqs, return_partial=True, **kwargs)
        pos_g = pos.reshape(B, -1, pos.shape[-1])
        E.SP_GLOBAL_ATTN = True     # (only consulted under sequence parallelism) this VGGT block attends over ALL frames
        try:
            xa, mod_agg = self.x_agg(x_agg.reshape(B, -1, D), pos=pos_g, e0=e0, return_partial=True)
        finally:
            E.SP_GLOBAL_ATTN = False
        if uncond is not True:
            xd, xa = self.bicross_attention([xd, xa], freqs=freqs, freqs_dit=freqs_dit, freqs_agg=freqs_agg)
        xd = self.x_dit(xd, context, t_mod, freqs, run_remaining=True, modifiers=mod_dit, **kwargs)
        xa = self.x_agg(xa, run_remaining=True, modifiers=mod_agg)
        return xd, xa, [xa.view(B, -1, P, D)]
