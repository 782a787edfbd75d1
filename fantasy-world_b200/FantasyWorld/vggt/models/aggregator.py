"""B200-native mirror of FantasyWorld/vggt/models/aggregator.py (reference).

Token assembly (camera + 4 register + h*w patch tokens per frame), integer positions, and the frame / global attention
drivers.  The integer / index work is plain torch (bit-exact by construction); the blocks run on the fwb200 kernels.
Same state_dict keys (camera_token, register_token, CamTokenProjector.*, frame_blocks.*, global_blocks.*).
"""
from __future__ import annotations

from typing import List, Tuple

import torch
import torch.nn as nn

from FantasyWorld.vggt.layers.block import Block, CamTokenProjector
from FantasyWorld.vggt.layers.rope import PositionGetter, RotaryPositionEmbedding2D
from FantasyWorld.wan.modules.model import rope_params


def slice_expand_and_flatten(token_tensor, B, S):
    """[1, 2, X, C] -> [(B S), X, C]: slot 0 for the first frame of every sequence, slot 1 for the other S-1 frames.
    ref: aggregator.py:283-306."""
    first = token_tensor[:, 0:1].expand(B, 1, *token_tensor.shape[2:])
    rest = token_tensor[:, 1:2].expand(B, S - 1, *token_tensor.shape[2:])
    return torch.cat([first, rest], dim=1).reshape(B * S, *token_tensor.shape[2:])


class Aggregator(nn.Module):
    def __init__(self, img_size=518, patch_size=14, embed_dim=1024, depth=24, num_heads=16, mlp_ratio=4.0,
                 num_register_tokens=4, block_fn=Block, qkv_bias=True, proj_bias=True, ffn_bias=True,
                 aa_order=["frame", "cross", "global"], aa_block_size=1, qk_norm=True, rope_freq=100, init_values=0.01,
                 cross_hidden_dim=1024, cross_num_heads=16, spatial_time=21):
        super().__init__()
        self.spatial_time = spatial_time
        self.rope = RotaryPositionEmbedding2D(frequency=rope_freq) if rope_freq > 0 else None
        self.position_getter = PositionGetter() if self.rope is not None else None
        self.CamTokenProjector = CamTokenProjector(out_dim=embed_dim)

        def make():
            return block_fn(dim=embed_dim, num_heads=num_heads, mlp_ratio=mlp_ratio, qkv_bias=qkv_bias, proj_bias=proj_bias,
                            ffn_bias=ffn_bias, init_values=init_values, qk_norm=qk_norm, rope=self.rope)

        self.frame_blocks = nn.ModuleList([make() for _ in range(depth)])
        self.global_blocks = nn.ModuleList([make() for _ in range(depth)])
        self.depth, self.aa_order, self.patch_size, self.aa_block_size = depth, aa_order, patch_size, aa_block_size
        d = cross_hidden_dim // cross_num_heads
        self.freqs = torch.cat([rope_params(1024, d - 4 * (d // 6)), rope_params(1024, 2 * (d // 6)),
                                rope_params(1024, 2 * (d // 6))], dim=1)
        if self.depth % self.aa_block_size != 0:
            raise ValueError(f"depth ({depth}) must be divisible by aa_block_size ({aa_block_size})")
        self.aa_block_num = self.depth // self.aa_block_size
        self.camera_token = nn.Parameter(torch.randn(1, 2, 1, embed_dim))
        self.register_token = nn.Parameter(torch.randn(1, 2, num_register_tokens, embed_dim))
        self.patch_start_idx = 1 + num_register_tokens
        nn.init.normal_(self.camera_token, std=1e-6)
        nn.init.normal_(self.register_token, std=1e-6)
        self.use_reentrant = False

    # -- token assembly ------------------------------------------------------------------------------------------------
    def _process_aggregator_input(self, patch_tokens: torch.Tensor, camera_token: torch.Tensor = None, frame_range=None):
        """patch_tokens [B, T, h, w, C] -> tokens [(B T), 5 + h*w, C], pos int64 [(B T), 5 + h*w, 2]
        (patch positions shifted by +1, specials at (0, 0)).  ref: aggregator.py:261-281.
        `frame_range=(f0, f1)` (sequence parallelism, B == 1): patch_tokens holds only frames f0..f1 of the clip; the
        "first frame" variants of the camera / register tokens are used for global frame 0 only."""
        B, T, gh, gw, C = patch_tokens.shape
        flat = patch_tokens.reshape(B * T, gh * gw, C)
        if frame_range is None:
            if camera_token is not None:
                cam = self.CamTokenProjector(camera_token).to(flat.dtype)
            else:
                cam = slice_expand_and_flatten(self.camera_token, B, T).to(flat.dtype)
            reg = slice_expand_and_flatten(self.register_token, B, T).to(flat.dtype)
        else:
            assert B == 1 and camera_token is None
            f0, f1 = frame_range
            slot = torch.tensor([0 if fr == 0 else 1 for fr in range(f0, f1)], device=flat.device)
            cam = self.camera_token[0, slot].to(flat.dtype)       # [T, 1, C]
            reg = self.register_token[0, slot].to(flat.dtype)     # [T, 4, C]
        tokens = torch.cat([cam, reg, flat], dim=1)
        return tokens, self._positions(B * T, gh, gw, flat.device, batch=B)

    def _positions(self, n, gh, gw, device, batch=1):
        """int64 [n, 5 + gh*gw, 2]; loop-invariant, so built once per (n, gh, gw) and reused (stable identity lets the
        RoPE tables derived from it be cached too).  At batch > 1 every sample has the same positions: the tensor is marked
        with the rows of one sample (`_fwb_period`), so the RoPE tables are built for one sample and shared."""
        if self.rope is None:
            return None
        cache = self.__dict__.setdefault("_pos_cache", {})
        key = (n, gh, gw, str(device), batch)
        if key not in cache:
            pos = self.position_getter(n, gh, gw, device=device)
            if self.patch_start_idx > 0:
                special = torch.zeros(n, self.patch_start_idx, 2, device=device, dtype=pos.dtype)
                pos = torch.cat([special, pos + 1], dim=1)
            pos = pos.contiguous()
            if batch > 1:
                pos._fwb_period = (n // batch) * pos.shape[1]
            cache[key] = pos
        return cache[key]

    # -- attention drivers ---------------------------------------------------------------------------------------------
    def _process_frame_attention(self, tokens, B, S, P, C, frame_idx, pos=None, e0=None):
        """Per-frame attention: tokens as [(B S), P, C].  ref: aggregator.py:215-237."""
        tokens = tokens.reshape(B * S, P, C)
        if pos is not None:
            pos = pos.reshape(B * S, P, 2)
        inter = []
        for _ in range(self.aa_block_size):
            tokens = self.frame_blocks[frame_idx](tokens, pos=pos, e0=e0)
            frame_idx += 1
            inter.append(tokens.view(B, S, P, C))
        return tokens, frame_idx, inter

    def _process_global_attention(self, tokens, B, S, P, C, global_idx, pos=None, e0=None):
        """All-frames attention: tokens as [B, (S P), C].  ref: aggregator.py:239-260."""
        tokens = tokens.reshape(B, S * P, C)
        if pos is not None:
            pos = pos.reshape(B, S * P, 2)
        inter = []
        for _ in range(self.aa_block_size):
            tokens = self.global_blocks[global_idx](tokens, pos=pos, e0=e0)
            global_idx += 1
            inter.append(tokens.view(B, S, P, C))
        return tokens, global_idx, inter

    def forward(self, patch_tokens: torch.Tensor, camera_token: torch.Tensor = None, e0: torch.Tensor = None) -> Tuple[List[torch.Tensor], int]:
        """Stand-alone geometry branch (no adapter): alternate frame / global blocks and collect
        [B, S, P, 2C] intermediates.  ref: aggregator.py:150-213."""
        B, T = patch_tokens.shape[:2]
        tokens, pos = self._process_aggregator_input(patch_tokens, camera_token)
        _, P, C = tokens.shape
        fi = gi = 0
        out = []
        for _ in range(self.aa_block_num):
            f_int = g_int = None
            for kind in self.aa_order:
                if kind == "frame":
                    tokens, fi, f_int = self._process_frame_attention(tokens, B, T, P, C, fi, pos=pos, e0=e0)
                elif kind == "global":
                    tokens, gi, g_int = self._process_global_attention(tokens, B, T, P, C, gi, pos=pos, e0=e0)
            out.extend(torch.cat([a, b], dim=-1) for a, b in zip(f_int, g_int))
        return out, self.patch_start_idx
