"""Test-only import shim for the UNMODIFIED reference (SURVEY.md §8c).

The reference's package __init__ files star-import modules that need `imageio`, `modelscope`, `ftfy`, `diffusers`
(absent here, no network).  None of them is used by the denoising hot path, so we register inert stub modules and
then import the reference normally.  Used ONLY to (a) validate oracle/ against the real reference, (b) generate the
golden vectors under tests/golden/, (c) run the reference itself on the GPU box as the bf16 parity target and the GPU /
CPU baseline (oracle/ref_runner.py, always in its OWN process: the reference's package is called `FantasyWorld`, like
this repo's mirror, so the two never share an interpreter).  Lives under tools/ (it is an import helper for the reference, not part
of the oracle): the golden generators import it directly, oracle/ref_runner.py loads it by path.

Where the reference comes from: the byte-for-byte copy staged by oracle/make_ref.py under oracle/_ref/ (git-ignored).
"""
from __future__ import annotations

import importlib
import sys
import types

import torch
import torch.nn as nn

from pathlib import Path

REF_ROOT = str(Path(__file__).resolve().parent.parent / "oracle" / "_ref")


def reference_available() -> bool:
    return Path(REF_ROOT, "FantasyWorld").exists()


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    m.__path__ = []  # behave like a package
    sys.modules[name] = m
    return m


def install_stubs():
    if "diffusers" not in sys.modules:
        try:
            importlib.import_module("diffusers")
        except Exception:
            _stub("diffusers")
            _stub("diffusers.configuration_utils", ConfigMixin=type("ConfigMixin", (), {}),
                  register_to_config=lambda f: f)
            _stub("diffusers.models")
            _stub("diffusers.models.modeling_utils", ModelMixin=nn.Module)
    for name in ("imageio", "modelscope", "ftfy"):
        if name not in sys.modules:
            try:
                importlib.import_module(name)
            except Exception:
                m = _stub(name)
                if name == "modelscope":
                    m.snapshot_download = lambda *a, **k: None
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)


def import_reference(flash_attn: bool = False):
    """Returns a namespace with the reference modules the hot path uses.  flash_attn=False (CPU, or the SDPA leg on the
    GPU) clears the reference's FLASH_ATTN_2_AVAILABLE switch so that flash_attention() falls to
    F.scaled_dot_product_attention (wan_video_dit.py:60-65); flash_attn=True leaves the module's own detection alone
    (flash-attn 2.8 is installed in this image, so the DiT attention then goes through flash_attn_func)."""
    if not reference_available():
        raise RuntimeError(f"reference not found at {REF_ROOT}: run `python oracle/make_ref.py` in the build container")
    install_stubs()
    ns = types.SimpleNamespace()
    ns.dit = importlib.import_module("FantasyWorld.diffsynth_wan21.models.wan_video_dit")
    if not flash_attn:
        ns.dit.FLASH_ATTN_2_AVAILABLE = False
    ns.dit.FLASH_ATTN_3_AVAILABLE = False
    ns.dit.SAGE_ATTN_AVAILABLE = False
    ns.camera = importlib.import_module("FantasyWorld.diffsynth_wan21.models.camera_control")
    ns.fusion_block = importlib.import_module("FantasyWorld.fusion.layer.block")
    ns.fusion = importlib.import_module("FantasyWorld.fusion.model_wan21")
    ns.vggt = importlib.import_module("FantasyWorld.vggt.models.vggt")
    ns.vggt_block = importlib.import_module("FantasyWorld.vggt.layers.block")
    ns.sched = importlib.import_module("FantasyWorld.diffsynth_wan21.schedulers.flow_match")
    return ns


VGGT_CFG = dict(img_size=518, patch_size=16, embed_dim=1024, number_frame=81, freq_dim=256, enable_camera=True,
                enable_depth=True, enable_point=True, enable_track=False, DPT_patch_size=16)
CAMERA_CFG = dict(pose_in_dim=1024, plucker_fea_dim=2048, pose_inject_method="adaln", use_info="plucker")


def randomize_zero_init(model: nn.Module, seed: int = 1):
    """SURVEY Appendix D-1: zero / tiny initialised tensors hide whole sub-paths.  Overwrite them."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith("gamma_m1") or name.endswith("gamma_m2") or name.endswith("ls1.gamma") or name.endswith(
                    "ls2.gamma"):
                p.copy_(torch.rand(p.shape, generator=g) + 0.5)
            elif p.numel() > 0 and float(p.abs().max()) == 0.0:
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
            elif name.endswith("camera_token") or name.endswith("register_token"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)


def build_reference_fusion(num_dit_layers: int = 3, start_index: int = 1, heads: bool = True, seed: int = 0,
                           dtype=torch.float32, flash_attn: bool = False):
    """Assemble a reduced-depth FantasyWorldFusionModel exactly as model_wan21.py:38-102 does, but without
    ModelManager / checkpoints / .to('cuda').  Width is fixed by the reference (5120 / 1024)."""
    ns = import_reference(flash_attn=flash_attn)
    torch.manual_seed(seed)
    n_irg = num_dit_layers - start_index
    model = ns.fusion.FantasyWorldFusionModel.__new__(ns.fusion.FantasyWorldFusionModel)
    nn.Module.__init__(model)
    pipe = types.SimpleNamespace()
    pipe.dit = ns.dit.WanModel(dim=5120, in_dim=36, ffn_dim=13824, out_dim=16, text_dim=4096, freq_dim=256, eps=1e-6,
                               patch_size=(1, 2, 2), num_heads=40, num_layers=num_dit_layers, has_image_input=True)
    pipe.scheduler = ns.sched.FlowMatchScheduler(shift=5, sigma_min=0.0, extra_one_step=True)
    pipe.torch_dtype = dtype
    pipe.device = "cpu"

    class _Pipe(nn.Module):
        pass

    pm = _Pipe()
    pm.dit = pipe.dit
    pm.scheduler = pipe.scheduler
    pm.torch_dtype = dtype
    pm.device = "cpu"
    model.pipe = pm
    cfg = dict(VGGT_CFG)
    if not heads:
        cfg.update(enable_camera=False, enable_depth=False, enable_point=False)
    model.vggt = ns.vggt.VGGT(**cfg)
    # shrink the aggregator to n_irg blocks (it always builds 24)
    model.vggt.aggregator.frame_blocks = nn.ModuleList(list(model.vggt.aggregator.frame_blocks)[:n_irg])
    model.vggt.aggregator.global_blocks = nn.ModuleList(list(model.vggt.aggregator.global_blocks)[:n_irg])
    model.camera_control = True
    model.camera_condition = ns.camera.CameraConditionModel(pm.dit, **CAMERA_CFG)
    model.start_index = start_index
    model.use_gradient_checkpointing = False
    model.use_gradient_checkpointing_offload = False
    model.cross_attention_list = list(range(n_irg))
    model.device = "cpu"
    model.bicross_dim = 1152
    model.bicross_num_heads = 12
    model.freqs_bicross = ns.dit.precompute_freqs_cis_3d(1152 // 12)
    import copy
    irg = nn.ModuleList()
    for idx in model.cross_attention_list:
        src_dit = pm.dit.blocks[idx + start_index]
        src_agg = model.vggt.aggregator.global_blocks[idx]
        d, a = copy.deepcopy(src_dit), copy.deepcopy(src_agg)
        pm.dit.blocks[idx + start_index] = nn.Identity()
        model.vggt.aggregator.global_blocks[idx] = nn.Identity()
        irg.append(ns.fusion_block.IRGBlock(x_agg_block=a, x_dit_block=d, m1_dim=5120, m2_dim=1024, hidden_size=1152,
                                            num_heads=12, drop_path=None))
    model.IRGBlock = irg
    model.use_info = CAMERA_CFG["use_info"]
    model.drop_ratio = 0.17
    if dtype is not None:          # dtype=None: meta-device construction (the caller materialises and initialises)
        randomize_zero_init(model)
        model.to(dtype)
    model.eval()
    return model, ns
