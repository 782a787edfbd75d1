"""B200-native mirror of FantasyWorld/fusion/model_wan21.py (reference): FantasyWorldFusionModel — 16 frozen WanDiT
Preconditioning Blocks + 24 IRG blocks (DiT block || VGGT global block + bidirectional adapter) with the 24 VGGT frame
blocks in between, the DiT head, the geometry heads on the last step, and the 50-step CFG flow-matching sampler.

Same constructor / joint_forward / generate_video signatures, attributes (`pipe`, `vggt`, `IRGBlock`,
`camera_condition`) and state_dict keys as the reference, so inference_wan21.py and the released checkpoints drop in.
What differs is execution: all token-sized work runs on the fwb200 sm_100a kernels, loop-invariant work is hoisted
(SURVEY Appendix E: context embeddings and cross-attention K/V, RoPE tables, positions, camera-feature projections,
`output_list` on non-final steps) and the host syncs the reference pays inside the loop are gone (Appendix D-5).
Results are the same tensors the reference computes, at the reference's own rounding points.
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn as nn

from fwb200 import ops

from ..diffsynth_wan21 import ModelManager, WanVideoPipeline
from ..diffsynth_wan21.models.camera_control import CameraConditionModel
from ..diffsynth_wan21.models.wan_video_dit import (build_freqs_3d_with_extra_cis, precompute_freqs_cis_3d,
                                                    sinusoidal_embedding_1d, _grid_freqs)
from ..fusion.core import FusionCore
from ..fusion.layer.block import IRGBlock
from ..vggt.models.vggt import VGGT

LATENT_MEAN = [-0.7571, -0.7089, -0.9113, 0.1075, -0.1745, 0.9653, -0.1517, 1.5508,
               0.4134, -0.0715, 0.5517, -0.3632, -0.1922, -0.9497, 0.2503, -0.2921]
LATENT_STD = [2.8184, 1.4541, 2.3275, 2.6558, 1.2196, 1.7708, 2.6052, 2.0743,
              3.2687, 2.1526, 2.8652, 1.5579, 1.6382, 1.1253, 2.8251, 1.9160]


class FantasyWorldFusionModel(FusionCore):
    def __init__(self, start_index: int = 16, use_gradient_checkpointing: bool = True,
                 use_gradient_checkpointing_offload: bool = False, cross_attention_list: list = [0], dit_path=None,
                 vggt_cfg: dict | None = None, camera_control: bool = False, camera_cfg: dict | None = None,
                 drop_ratio: float = 0.17, dit_config: dict | None = None, device: str = "cuda"):
        """`dit_config` (extension): WanModel kwargs for a random-init / reduced-depth DiT when no checkpoint is given."""
        super().__init__()
        manager = ModelManager(torch_dtype=torch.bfloat16, device="cpu", dit_config=dit_config)
        manager.load_models(dit_path, torch_dtype=torch.bfloat16)
        self.pipe = WanVideoPipeline.from_model_manager(manager, device='cpu')
        self.vggt = VGGT(**(vggt_cfg or {}))
        self.vggt.to(torch.bfloat16)
        self.camera_control = camera_control
        if self.camera_control:
            self.camera_condition = CameraConditionModel(self.pipe.dit, **{k: v for k, v in camera_cfg.items()})
        self.start_index = start_index
        self.use_gradient_checkpointing = use_gradient_checkpointing
        self.use_gradient_checkpointing_offload = use_gradient_checkpointing_offload
        self.cross_attention_list = cross_attention_list
        self.device = device
        self.bicross_dim, self.bicross_num_heads = 1152, 12
        self.freqs_bicross = precompute_freqs_cis_3d(self.bicross_dim // self.bicross_num_heads)

        # model surgery (ref: model_wan21.py:69-87): DiT block start_index+i and VGGT global block i move into IRGBlock[i]
        irg = nn.ModuleList()
        for idx in self.cross_attention_list:
            dit_blk = self.pipe.dit.blocks[idx + self.start_index]
            agg_blk = self.vggt.aggregator.global_blocks[idx]
            self.pipe.dit.blocks[idx + self.start_index] = nn.Identity()
            self.vggt.aggregator.global_blocks[idx] = nn.Identity()
            irg.append(IRGBlock(x_agg_block=agg_blk, x_dit_block=dit_blk, m1_dim=self.pipe.dit.dim, m2_dim=self.vggt.embed_dim,
                                hidden_size=self.bicross_dim, num_heads=self.bicross_num_heads, drop_path=None))
        self.IRGBlock = irg
        self.mean = torch.tensor(LATENT_MEAN)
        self.std = torch.tensor(LATENT_STD)
        self.scale = [self.mean, 1.0 / self.std]
        self.use_info = (camera_cfg or {}).get('use_info')
        self.drop_ratio = drop_ratio
        self.to(torch.bfloat16)

    # ------------------------------------------------------------------------------------------------------------------
    def joint_forward(self, x: torch.Tensor, timestep: torch.Tensor, context: torch.Tensor,
                      clip_feature: Optional[torch.Tensor] = None, y: Optional[torch.Tensor] = None,
                      use_gradient_checkpointing: bool = True, camera_token=None, plucker_fea: Optional[torch.Tensor] = None,
                      plucker_context_lens: Optional[torch.Tensor] = None, uncond=False, return_prediction=False, **kwargs):
        """One denoiser evaluation.  ref: model_wan21.py:104-224.  With `self.sp` set (fwb200.sp.SPContext, world > 1) the
        tokens are sharded over the ranks of that group; inputs and outputs are replicated either way."""
        ops.require_device()
        ctx = self.embed_context(context, clip_feature)
        if self.pipe.dit.has_image_input:
            x = torch.cat([x, y], dim=1)
        return self._joint_core(x, timestep, ctx, dict(plucker_context_lens=plucker_context_lens), plucker_fea=plucker_fea,
                                camera_token=camera_token, uncond=uncond, return_prediction=return_prediction)

    # ------------------------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def generate_video(self, context_pos: torch.Tensor, context_neg: Optional[torch.Tensor] = None,
                       clip_feature: Optional[torch.Tensor] = None, y: Optional[torch.Tensor] = None,
                       use_gradient_checkpointing: bool = False, camera_token=None, height=480, width=832, num_frames=81,
                       num_inference_steps=50, cfg_scale=5.0, seed=None, device="cuda", plucker_embedding=None,
                       geo_prior=None, latents: Optional[torch.Tensor] = None, batch_cfg: bool = False, **kwargs):
        """50-step CFG flow-matching sampler.  ref: model_wan21.py:227-324.  `latents` (extension) injects the initial
        noise instead of drawing it (GPU RNG streams are not reproducible across devices, SURVEY Appendix D-6).
        Batch (extension): the batch is that of `latents`, or of `context_pos` when the noise is drawn here; every
        per-sample input (contexts, clip_feature, y, plucker_embedding, geo_prior) must have that batch.  `batch_cfg`: see
        denoise_step."""
        pipe = self.pipe
        if num_frames % 4 != 1:
            num_frames = (num_frames + 2) // 4 * 4 + 1
        pipe.scheduler.set_timesteps(num_inference_steps)
        if latents is None:
            if seed is not None:
                torch.manual_seed(1024)
            noise = pipe.generate_noise((context_pos.shape[0], 16, (num_frames - 1) // 4 + 1, height // 8, width // 8), seed=seed,
                                        device=device, dtype=torch.float32)
            latents = noise.to(dtype=pipe.torch_dtype, device=pipe.device)
        latents = latents.to(dtype=torch.bfloat16, device=pipe.device).contiguous().clone()

        plucker_fea = plucker_context_lens = None
        if self.camera_control:
            if self.use_info == 'rgb_conf':
                guide = geo_prior
            elif self.use_info == 'all':
                guide = torch.cat([geo_prior, plucker_embedding], dim=-1)
            elif self.use_info == 'plucker':
                guide = plucker_embedding
            else:
                raise NotImplementedError
            plucker_fea = self.camera_condition.get_pose_fea(guide)
            plucker_context_lens = torch.ones(guide.shape[1] // 4 + 1, dtype=torch.long, device=plucker_fea.device)
            plucker_context_lens[1:] = 4

        clip_feature = clip_feature.to(pipe.device) if clip_feature is not None else None
        y = y.to(pipe.device) if y is not None else None
        extra = pipe.prepare_extra_input(latents)
        final_prediction = None
        for step in range(num_inference_steps):
            latents, pred = self.denoise_step(latents, step, context_pos, context_neg, clip_feature=clip_feature, y=y,
                                              camera_token=camera_token, plucker_fea=plucker_fea,
                                              plucker_context_lens=plucker_context_lens, cfg_scale=cfg_scale,
                                              return_prediction=(step == num_inference_steps - 1), batch_cfg=batch_cfg, **extra)
            if pred is not None:
                final_prediction = pred
        return latents, final_prediction

    @torch.no_grad()
    def denoise_step(self, latents: torch.Tensor, step: int, context_pos: torch.Tensor, context_neg: Optional[torch.Tensor] = None,
                     clip_feature: Optional[torch.Tensor] = None, y: Optional[torch.Tensor] = None, camera_token=None,
                     plucker_fea: Optional[torch.Tensor] = None, plucker_context_lens: Optional[torch.Tensor] = None,
                     cfg_scale: float = 5.0, return_prediction: bool = False, batch_cfg: bool = False, **extra):
        """One iteration of the sampler loop (ref: model_wan21.py:289-322): conditional + unconditional joint_forward,
        classifier-free guidance and the flow-matching Euler update (fused in fwb_cfg_euler_step).  `latents` may live on
        the host (pinned): it is copied to the device here; the updated latents are returned on the device.
        Uses the schedule set by `self.pipe.scheduler.set_timesteps`.
        latents [B, ...] with per-sample contexts [B, ...] (one shared timestep).  batch_cfg=True evaluates the conditional
        and unconditional forwards as ONE forward of batch 2B (same results; off by default, see DESIGN.md §1 "Batch")."""
        pipe, sched = self.pipe, self.pipe.scheduler
        dev = pipe.device
        if latents.device.type != "cuda":
            latents = latents.to(device=dev, dtype=torch.bfloat16, non_blocking=True)
        latents = latents.contiguous()
        t_host = sched.timesteps[step]
        t = t_host.unsqueeze(0).to(dtype=pipe.torch_dtype, device=dev)   # bf16 timestep, as the reference (:292-293)
        kw = dict(clip_feature=clip_feature, y=y, use_gradient_checkpointing=False, camera_token=camera_token,
                  plucker_fea=plucker_fea, plucker_context_lens=plucker_context_lens)
        dsigma = sched.dsigma(t_host)
        if cfg_scale != 1.0 and context_neg is not None:
            pred_pos, pred_neg, pred = self._cfg_forwards(latents, t, context_pos, context_neg, {**kw, **extra}, return_prediction,
                                                          batch_cfg=batch_cfg)
            ops.cfg_euler_step_(latents, pred_pos.contiguous(), pred_neg.contiguous(), cfg_scale, dsigma)
        else:
            assert self.cfgp is None, "CFG parallelism needs cfg_scale != 1 and a negative context"
            self.check_batch(latents, context_pos, None, kw)
            pred_pos, pred = self.joint_forward(latents, timestep=t, context=context_pos, return_prediction=return_prediction, **kw, **extra)
            ops.cfg_euler_step_(latents, pred_pos.contiguous(), pred_pos.contiguous(), 1.0, dsigma)
        return latents, pred
