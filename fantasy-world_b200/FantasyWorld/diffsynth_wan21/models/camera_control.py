"""B200-native mirror of FantasyWorld/diffsynth_wan21/models/camera_control.py (reference).

Camera conditioning of the DiT cross-attention ('adaln' injection): after the text/CLIP attention, an MLP of the
token-aligned Plücker features and the attention output produces a per-token shift that is added before the output
projection (ref: camera_control.py:92-148).  Same class names and state_dict keys; the five small Linear layers run
as fwb200 GEMMs with fused ReLU / residual epilogues, and the loop-invariant parts (group1(plucker_fea), the
all-zeros test that costs the reference one host sync per call, camera_control.py:111) are hoisted and cached.
Only pose_inject_method == 'adaln' (the released configuration, inference_wan21.py:196-202) is implemented.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from fwb200 import engine as E
from fwb200 import ops

from .wan_video_dit import WanModel


class PoseProjModel(nn.Module):
    def __init__(self, pose_in_dim=1024, cross_attention_dim=1024):
        super().__init__()
        self.cross_attention_dim = cross_attention_dim
        self.proj = torch.nn.Linear(pose_in_dim, cross_attention_dim, bias=False)
        self.norm = torch.nn.LayerNorm(cross_attention_dim)

    def forward(self, pose_embeds):
        shp = pose_embeds.shape
        h = E.lin(E.as_bf16(pose_embeds).reshape(-1, shp[-1]), self.proj)
        h = ops.ln_modulate(h, eps=self.norm.eps, w=E.f32(self.norm, "w", self.norm.weight), b=E.f32(self.norm, "b", self.norm.bias))
        return h.view(*shp[:-1], -1)


class GroupLinearDualK(nn.Module):
    """ref: camera_control.py:24-39."""

    def __init__(self, context_dim, hidden_dim, groups=2):
        super().__init__()
        self.group1 = nn.Linear(context_dim, context_dim)
        mid = min(hidden_dim, context_dim) // 2
        self.group2 = nn.Sequential(nn.Linear(hidden_dim, mid), nn.ReLU(), nn.Linear(mid, context_dim))


class GroupLinearDualV(nn.Module):
    """ref: camera_control.py:42-63 (the 'scale' branch is the constant 0.0; only the shift MLP has weights)."""

    def __init__(self, context_dim, hidden_dim, groups=2):
        super().__init__()
        reduced = context_dim // 5
        self.group2 = nn.Sequential(nn.Linear(context_dim, reduced), nn.ReLU(), nn.Linear(reduced, hidden_dim))
        nn.init.zeros_(self.group2[-1].weight)
        nn.init.zeros_(self.group2[-1].bias)


def get_processor(method, context_dim, hidden_dim):
    if method != 'adaln':
        raise NotImplementedError("only pose_inject_method='adaln' is implemented (released configuration)")
    return GroupLinearDualK(context_dim, hidden_dim), GroupLinearDualV(context_dim, hidden_dim)


def _pad8(n):
    return (n + 7) // 8 * 8


class CrossAttentionAdapterProcessor(nn.Module):
    """ref: camera_control.py:79-148."""

    def __init__(self, context_dim, hidden_dim, pose_inject_method='latent_split'):
        super().__init__()
        self.context_dim, self.hidden_dim, self.pose_inject_method = context_dim, hidden_dim, pose_inject_method
        self.k_proj, self.v_proj = get_processor(pose_inject_method, context_dim, hidden_dim)

    # loop-invariant: group1(plucker_fea) and the all-zero flag, cached per plucker tensor
    def _plucker(self, plucker_fea):
        cache = self.__dict__.get("_fwb_pl")
        if cache is None:
            cache = self.__dict__["_fwb_pl"] = E.IdCache(2)

        def build():
            # the reference tests the WHOLE tensor (camera_control.py:111); a sequence-parallel rank only holds its row slice, so
            # FusionCore._local_rows stamps the slice with the flag of the full tensor (a rank whose slice happens to be all
            # zero must still apply the shift: it is group1's bias + group2(x), not zero)
            flag = getattr(plucker_fea, "_fwb_all_zero", None)
            all_zero = bool(torch.all(plucker_fea == 0).item()) if flag is None else bool(flag)
            p1 = None if all_zero else E.lin(E.as_bf16(plucker_fea).reshape(-1, plucker_fea.shape[-1]), self.k_proj.group1,
                                             round_flags=ops.ROUND_AFTER_BIAS)
            return all_zero, p1

        return cache.get((plucker_fea, self.k_proj.group1.weight), None, build)

    def _shift_weights(self):
        """v_proj.group2: Linear(2048->409), ReLU, Linear(409->5120).  409 is not a multiple of 8: zero-pad to 416
        (exact: padded hidden units are relu(0)=0 and meet zero weights)."""
        l0, l2 = self.v_proj.group2[0], self.v_proj.group2[2]
        r, rp = l0.out_features, _pad8(l0.out_features)

        def pad0(w, b):
            wp = torch.zeros(rp, w.shape[1], device=w.device, dtype=torch.bfloat16)
            wp[:r] = w.to(torch.bfloat16)
            bp = torch.zeros(rp, device=w.device, dtype=torch.float32)
            bp[:r] = b.float()
            return wp, bp

        def pad2(w):
            wp = torch.zeros(w.shape[0], rp, device=w.device, dtype=torch.bfloat16)
            wp[:, :r] = w.to(torch.bfloat16)
            return wp

        w0, b0 = E.derived(self, "v0", pad0, l0.weight, l0.bias)
        w2 = E.derived(self, "v2", pad2, l2.weight)
        return w0, b0, w2, E.f32(l2, "b", l2.bias)

    def _adaln(self, o, plucker_fea):
        """o [B*L, C] bf16 (text+CLIP attention output) -> o + shift; plucker_fea [B, L, 2048].  As in the reference, one
        all-zero test covers the whole batch: a batch with one all-zero sample still shifts every sample."""
        all_zero, p1 = self._plucker(plucker_fea)
        if all_zero:
            return o
        g2 = self.k_proj.group2
        h = E.lin(o, g2[0], act=ops.ACT_RELU, round_flags=ops.ROUND_AFTER_BIAS)
        comb = E.lin(h, g2[2], resid=p1, round_flags=ops.ROUND_AFTER_BIAS)
        w0, b0, w2, b2 = self._shift_weights()
        h2 = ops.linear(comb, w0, bias=b0, act=ops.ACT_RELU, round_flags=ops.ROUND_AFTER_BIAS)
        return ops.linear(h2, w2, bias=b2, resid=o, round_flags=ops.ROUND_AFTER_BIAS)

    def fused(self, attn, n3, context, x_resid, plucker_fea=None, plucker_context_lens=None, pose_scale: float = 1.0, **kw):
        assert pose_scale == 1.0, "pose_scale != 1 is not used by the reference sampler"
        o = E.dit_cross_attn_core(attn, n3, context)
        if plucker_fea is not None:
            o = self._adaln(o, plucker_fea)
        return E.lin(o, attn.o, resid=x_resid, round_flags=ops.ROUND_AFTER_BIAS)

    def __call__(self, attn: nn.Module, x: torch.Tensor, y: torch.Tensor, plucker_fea: torch.Tensor = None,
                 plucker_context_lens: torch.Tensor = None, pose_scale: float = 1.0):
        b, s, c = x.shape
        assert pose_scale == 1.0, "pose_scale != 1 is not used by the reference sampler"
        o = E.dit_cross_attn_core(attn, E.as_bf16(x).reshape(b * s, c), y)
        if plucker_fea is not None:
            o = self._adaln(o, plucker_fea)
        return E.lin(o, attn.o, round_flags=ops.ROUND_AFTER_BIAS).view(b, s, c)


class CameraConditionModel(nn.Module):
    """Installs the adapter processors on DiT blocks 0..24 and owns the pose encoder.  ref: camera_control.py:152-234."""

    def __init__(self, wan_dit: WanModel, pose_in_dim: int, plucker_fea_dim: int, pose_inject_method: str, use_info: str):
        super().__init__()
        self.pose_in_dim, self.plucker_fea_dim, self.pose_inject_method = pose_in_dim, plucker_fea_dim, pose_inject_method
        self.proj_model = nn.Identity()
        self.set_pose_processor(wan_dit)
        in_channels = {"all": 12, "rgb_conf": 4, "plucker": 6}.get(use_info)
        if in_channels is None:
            raise NotImplementedError(use_info)
        from .pose_adaptor_ac3d import CameraPoseEncoder
        self.pose_encoder = CameraPoseEncoder(context_dim=plucker_fea_dim, in_channels=in_channels, downscale_coef=8,
                                              pose_inject_method=pose_inject_method)

    def set_pose_processor(self, wan_dit):
        procs = {name: CrossAttentionAdapterProcessor(context_dim=self.plucker_fea_dim, hidden_dim=wan_dit.dim,
                                                      pose_inject_method=self.pose_inject_method)
                 for name in wan_dit.attn_processors.keys()}
        wan_dit.set_attn_processor(procs)

    def get_proj_fea(self, pose_fea=None):
        return self.proj_model(pose_fea) if pose_fea is not None else None

    def get_pose_fea(self, plucker=None):
        return self.pose_encoder(plucker) if plucker is not None else None
