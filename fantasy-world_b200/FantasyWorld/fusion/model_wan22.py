"""B200-native mirror of FantasyWorld/fusion/model_wan22.py (reference): the Wan2.2-Fun-A14B-Control-Camera fusion model.
Differences from the Wan2.1 model (ref: model_wan22.py:226-348 vs model_wan21.py:104-224): no CLIP context
(`has_image_input=False`, 512 text tokens), the camera enters through `control_camera_latents_input` -> `SimpleAdapter`
added to the patch embedding, no camera AdaLN processors, reward-LoRA merged into the DiT weights at load time.  The
PCB / IRG schedule, the geometry branch and the heads are the shared fwb200-backed core (fusion/core.py).  inference_wan22.py
holds two such models (high-noise / low-noise experts, switched at t = 900); `denoise_step_experts` below is that switch.
Same constructor / joint_forward signature and state_dict keys as the reference.
"""
from __future__ import annotations

from collections import defaultdict
from typing import Optional

import torch
import torch.nn as nn

from fwb200 import ops

from ..diffsynth_wan22.models.wan_video_dit import build_freqs_3d_with_extra_cis, precompute_freqs_cis_3d, sinusoidal_embedding_1d  # noqa: F401
from ..diffsynth_wan22.pipelines.wan_video_new import ModelConfig, WanVideoPipeline
from ..fusion.core import FusionCore
from ..fusion.layer.block import IRGBlock
from ..vggt.models.vggt import VGGT


def load_lora(pipeline, lora_path, multiplier, sub_transformer_name):
    """Merge a LoRA (W += multiplier * alpha/r * up @ down) into the Linear / 1x1 conv weights of `pipeline.<sub_transformer_name>`.
    ref: model_wan22.py:18-118.  The reference resolves the flattened `lora_unet_a_b_c` layer names by trial and error over
    attribute paths; here every module path is flattened the same way once and looked up directly."""
    if lora_path is None:
        return
    from safetensors.torch import load_file
    root = getattr(pipeline, sub_transformer_name)
    table = {name.replace(".", "_"): mod for name, mod in root.named_modules() if hasattr(mod, "weight")}
    groups = defaultdict(dict)
    for key, value in load_file(lora_path).items():
        if ".lora_A.default." in key or ".lora_B.default." in key:
            # reference behaviour (model_wan22.py:33-36): it strips 21 of the 22 characters of `_lora_A_default_weight`, cannot
            # resolve the resulting layer name and skips the entry; a drop-in must leave those weights untouched too
            continue
        k = key
        for a, b in ((".lora_A.default.", ".lora_down."), (".lora_B.default.", ".lora_up."), (".lora_A.", ".lora_down."), (".lora_B.", ".lora_up.")):
            k = k.replace(a, b)
        if ".lora_down." in k:
            layer, elem = k.split(".lora_down.")[0], "down"
        elif ".lora_up." in k:
            layer, elem = k.split(".lora_up.")[0], "up"
        elif k.endswith(".alpha"):
            layer, elem = k[:-6], "alpha"
        else:
            continue
        layer = layer.replace(".", "_")
        for prefix in ("lora_unet__", "lora_unet_", "diffusion_model_", "transformer_"):
            if layer.startswith(prefix):
                layer = layer[len(prefix):]
        groups[layer][elem] = value
    device, dtype = getattr(pipeline, "device", "cpu"), getattr(pipeline, "torch_dtype", torch.bfloat16)
    for layer, el in groups.items():
        mod = table.get(layer)
        if mod is None or "up" not in el or "down" not in el:
            continue
        # arithmetic as the reference does it (model_wan22.py:100-117): factors cast to the pipeline dtype (bf16), the rank-r product
        # in that dtype, scaled and accumulated into the weight in that dtype — so merged checkpoints are bit-identical
        up, down = el["up"].to(device, dtype), el["down"].to(device, dtype)
        alpha = (el["alpha"].item() / up.shape[1]) if "alpha" in el else 1.0
        w = mod.weight.data.to(device, dtype)
        if up.dim() == 4:
            w += multiplier * alpha * torch.mm(up.squeeze(3).squeeze(2), down.squeeze(3).squeeze(2)).unsqueeze(2).unsqueeze(3)
        else:
            w += multiplier * alpha * torch.mm(up, down)
        mod.weight.data = w.to(mod.weight.device, mod.weight.dtype)


def select_high_noise_expert(t_host: torch.Tensor, timestep_boundary: float = 900.0, dtype=torch.bfloat16) -> bool:
    """Expert choice of inference_wan22.py:229-240: the timestep is cast to the sampler dtype (bf16) first, then compared —
    `t.item() > boundary` picks the high-noise expert."""
    return float(t_host.to(dtype)) > timestep_boundary


class FantasyWorldFusionModel(FusionCore):
    def __init__(self, start_index=16, use_gradient_checkpointing=True, use_gradient_checkpointing_offload=False,
                 cross_attention_list=[0], dit_path=None, lora_path=None, origin_file_pattern=None,
                 model_id="PAI/Wan2.2-Fun-A14B-Control-Camera", vggt_cfg: dict | None = None, camera_control: bool = False,
                 camera_cfg: dict | None = None, min_timestep_boundary=0, max_timestep_boundary=1, load_vae=False,
                 load_text_encoder=False, dit_config: dict | None = None):
        super().__init__()
        self.device = "cuda"
        configs = [ModelConfig(model_id=model_id, origin_file_pattern=origin_file_pattern, local_model_path=dit_path)]
        extra = dict(tokenizer_config=None)
        if load_vae and load_text_encoder:       # the expert that also serves the conditioning call and the final decode (ref: :144-163)
            configs += [ModelConfig(model_id=model_id, origin_file_pattern="models_t5_umt5-xxl-enc-bf16.pth", local_model_path=dit_path),
                        ModelConfig(model_id=model_id, origin_file_pattern="Wan2.1_VAE.pth", local_model_path=dit_path)]
            extra = {}                             # default tokenizer_config: the google/umt5-xxl directory
        pipe = WanVideoPipeline.from_pretrained(torch_dtype=torch.bfloat16, device="cpu", dit_config=dit_config, model_configs=configs,
                                                **extra)
        pipe.device = "cpu"
        load_lora(pipe, lora_path, 0.55, "dit")
        self.pipe = pipe
        self.min_timestep_boundary, self.max_timestep_boundary = min_timestep_boundary, max_timestep_boundary
        self.vggt = VGGT(**(vggt_cfg or {}))
        self.vggt.to(torch.bfloat16)
        self.camera_control = camera_control
        self.start_index = start_index
        self.use_gradient_checkpointing = use_gradient_checkpointing
        self.use_gradient_checkpointing_offload = use_gradient_checkpointing_offload
        self.cross_attention_list = cross_attention_list
        self.bicross_dim, self.bicross_num_heads = 1152, 12
        self.freqs_bicross = precompute_freqs_cis_3d(self.bicross_dim // self.bicross_num_heads)
        irg = nn.ModuleList()
        for idx in self.cross_attention_list:      # model surgery, ref: model_wan22.py:204-222
            dit_blk = self.pipe.dit.blocks[idx + self.start_index]
            agg_blk = self.vggt.aggregator.global_blocks[idx]
            self.pipe.dit.blocks[idx + self.start_index] = nn.Identity()
            self.vggt.aggregator.global_blocks[idx] = nn.Identity()
            irg.append(IRGBlock(x_dit_block=dit_blk, x_agg_block=agg_blk, m1_dim=self.pipe.dit.dim, m2_dim=self.vggt.embed_dim,
                                hidden_size=self.bicross_dim, num_heads=self.bicross_num_heads, drop_path=None))
        self.IRGBlock = irg
        self.use_info = (camera_cfg or {}).get('use_info')
        self.to(dtype=torch.bfloat16)

    def joint_forward(self, x: torch.Tensor, timestep: torch.Tensor, context: torch.Tensor, y: Optional[torch.Tensor] = None,
                      use_gradient_checkpointing: bool = True, camera_token=None,
                      control_camera_latents_input: Optional[torch.Tensor] = None, uncond=False, return_prediction=False, **kwargs):
        """ref: model_wan22.py:226-348."""
        ops.require_device()
        ctx = self.embed_context(context, None)
        if y is not None and self.pipe.dit.require_vae_embedding:
            x = torch.cat([x, y], dim=1)
        return self._joint_core(x, timestep, ctx, {}, control=control_camera_latents_input, camera_token=camera_token,
                                uncond=uncond, return_prediction=return_prediction)


@torch.no_grad()
def denoise_step_experts(model_high: FantasyWorldFusionModel, model_low: FantasyWorldFusionModel, latents, step, context_pos,
                         context_neg, y, control_camera_latents_input, timestep_boundary=900.0, cfg_scale=5.0,
                         return_prediction=False, batch_cfg=False):
    """One iteration of inference_wan22.py's loop (ref: inference_wan22.py:229-280): pick the high-noise or low-noise expert
    by timestep, two forwards (CFG), fused guidance + Euler update.  Batched latents / contexts and `batch_cfg` as in the
    Wan2.1 model's denoise_step."""
    sched = model_high.pipe.scheduler
    t_host = sched.timesteps[step]
    model = model_high if select_high_noise_expert(t_host, timestep_boundary) else model_low
    t = t_host.unsqueeze(0).to(dtype=torch.bfloat16, device=latents.device)
    kw = dict(y=y, use_gradient_checkpointing=False, camera_token=None, control_camera_latents_input=control_camera_latents_input)
    if cfg_scale != 1.0 and context_neg is not None:
        pos, neg, pred = model._cfg_forwards(latents, t, context_pos, context_neg, kw, return_prediction, batch_cfg=batch_cfg)
        ops.cfg_euler_step_(latents, pos.contiguous(), neg.contiguous(), cfg_scale, sched.dsigma(t_host))
    else:
        model.check_batch(latents, context_pos, None, kw)
        pos, pred = model.joint_forward(latents, timestep=t, context=context_pos, return_prediction=return_prediction, **kw)
        ops.cfg_euler_step_(latents, pos.contiguous(), pos.contiguous(), 1.0, sched.dsigma(t_host))
    return latents, pred
