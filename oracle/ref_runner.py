"""oracle/ref_runner.py — runs the UNMODIFIED reference (staged under oracle/_ref, through tools/ref_shim.py) in its
own process, on the CPU or on the GPU box's B200.  TEST / BENCH INFRASTRUCTURE ONLY; nothing in the product path imports it.

Why a separate process: the reference's package is called `FantasyWorld`, exactly like this repo's drop-in mirror, and it
uses absolute `FantasyWorld.*` imports, so the two cannot live in one interpreter.  Callers (tests/test_gpu_ref_parity.py,
bench.py) spawn `python oracle/ref_runner.py <cmd> ...`; tensors come back through a directory of .pt files, timings as
one JSON line on stdout.

Commands
  blocks  one PCB DiTBlock (wan_video_dit.py:254-321, camera AdaLN processor camera_control.py:92-148), one VGGT frame Block
          (vggt/layers/block.py:82-116 via aggregator.py:215-237) and one IRGBlock (fusion/layer/block.py:43-94) in isolation
          at a token grid f,h,w, on the per-key synthetic weights and seeded inputs of fwb_synth (identical in the caller).
  joint   reduced-depth FantasyWorldFusionModel.joint_forward (model_wan21.py:104-224), optional geometry heads.
  step    K denoise steps = 2 x joint_forward + CFG + FlowMatchScheduler.step, exactly the loop body of
          model_wan21.py:289-322, timed (CUDA events on the GPU, perf_counter on the CPU).
  schema  state_dict key -> shape of the fusion model at a given depth (meta device), for the drop-in schema test.
Modes (precision / attention backend; SURVEY §8c, BASELINE.md §4)
  bf16_fa2   model.to(bf16) + torch.autocast(bf16)  (inference_wan21.py:224, :310), flash_attention() -> flash_attn_func
  bf16_sdpa  same with FLASH_ATTN_2_AVAILABLE cleared -> F.scaled_dot_product_attention (wan_video_dit.py:60-65)
  fp32       bf16-valued weights upcast to fp32, no autocast, TF32 off: the "golden fp32" of the parity protocol
"""
from __future__ import annotations

import argparse
import contextlib
import importlib.util
import json
import os
import sys
import time
from pathlib import Path

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent


def _load_by_path(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


# neither the repo root nor fantasy-world_b200/ may be on sys.path here (the mirror package would shadow the reference)
sys.path[:] = [p for p in sys.path if Path(p or ".").resolve() not in (ROOT, ROOT / "fantasy-world_b200")]
S = _load_by_path("fwb_synth", ROOT / "fantasy-world_b200" / "fwb_synth.py")
shim = _load_by_path("fwb_ref_shim", ROOT / "tools" / "ref_shim.py")

import torch  # noqa: E402

MODES = ("bf16_fa2", "bf16_sdpa", "fp32")


def build(n_layers, start_index, heads, device, seed=0):
    """Reference fusion model (14B widths, reduced or full depth) with the per-key synthetic weights, fp32 master on `device`."""
    if torch.device(device).type == "cpu" and not heads:
        # CPU: skip the default initialisers (minutes of kaiming_uniform_ over ~1e9 values that synth_init overwrites anyway):
        # construct on the meta device, give storage, rebuild the plain (non-parameter) RoPE tables the constructors made.
        with torch.device("meta"):
            model, ns = shim.build_reference_fusion(num_dit_layers=n_layers, start_index=start_index, heads=False, seed=seed,
                                                    flash_attn=True, dtype=None)
        S.materialize(model, "cpu", torch.float32)
        model.pipe.dit.freqs = ns.dit.precompute_freqs_cis_3d(5120 // 40)
        model.freqs_bicross = ns.dit.precompute_freqs_cis_3d(1152 // 12)
        rope_params = sys.modules["FantasyWorld.wan.modules.model"].rope_params
        d = 1024 // 16
        model.vggt.aggregator.freqs = torch.cat([rope_params(1024, d - 4 * (d // 6)), rope_params(1024, 2 * (d // 6)),
                                                 rope_params(1024, 2 * (d // 6))], dim=1)
        model.eval()
    else:
        # the constructors' own initialisers run on `device` (fast on the GPU); dtype=None skips the shim's CPU-generator
        # randomisation of zero-initialised tensors — synth_init below overwrites every parameter anyway
        with torch.device(device):
            model, ns = shim.build_reference_fusion(num_dit_layers=n_layers, start_index=start_index, heads=heads, seed=seed,
                                                    flash_attn=True, dtype=None)
        model.to(device=device, dtype=torch.float32)
    S.synth_init(model, seed)          # generator on the parameter's device: the caller does the same -> identical weights
    model.pipe.device = device
    return model, ns


def clear_rope_caches(model):
    """RotaryPositionEmbedding2D caches its angle tables keyed by (dim, len, device, token dtype) (vggt/layers/rope.py:101):
    a table built under autocast (bf16 einsum) would otherwise be reused by the fp32 run of the same process."""
    for m in model.modules():
        if hasattr(m, "frequency_cache"):
            m.frequency_cache.clear()


@contextlib.contextmanager
def mode_ctx(model, ns, mode, device):
    """Put the model into `mode` (see module docstring) for the duration of the block."""
    dev_type = torch.device(device).type
    clear_rope_caches(model)
    flash_detected = ns.dit.FLASH_ATTN_2_AVAILABLE
    tf32 = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    try:
        if mode == "fp32":
            model.to(torch.bfloat16).to(torch.float32)       # bf16-valued weights, fp32 arithmetic
            model.pipe.torch_dtype = torch.float32
            ns.dit.FLASH_ATTN_2_AVAILABLE = False
            torch.backends.cuda.matmul.allow_tf32 = False
            torch.backends.cudnn.allow_tf32 = False
            with torch.no_grad():
                yield torch.float32
        else:
            model.to(torch.bfloat16)
            model.pipe.torch_dtype = torch.bfloat16
            ns.dit.FLASH_ATTN_2_AVAILABLE = flash_detected and mode == "bf16_fa2" and dev_type == "cuda"
            with torch.no_grad(), torch.autocast(dev_type, dtype=torch.bfloat16):
                yield torch.bfloat16
    finally:
        ns.dit.FLASH_ATTN_2_AVAILABLE = flash_detected
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf32


def _sync(device):
    if torch.device(device).type == "cuda":
        torch.cuda.synchronize()


def timed(fn, device, reps):
    """(result of the last call, [ms per call]) — CUDA events on the GPU, perf_counter on the CPU."""
    out, ms = None, []
    cuda = torch.device(device).type == "cuda"
    for _ in range(reps):
        if cuda:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            out = fn()
            b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
        else:
            t0 = time.perf_counter()
            out = fn()
            ms.append((time.perf_counter() - t0) * 1e3)
    return out, ms


def grid_tables(model, ns, f, h, w, device):
    """freqs / freqs_bi_dit / freqs_bi_agg / pos exactly as joint_forward builds them (model_wan21.py:132-147, aggregator.py:274-280)."""
    def grid(fr):
        return torch.cat([fr[0][:f].view(f, 1, 1, -1).expand(f, h, w, -1), fr[1][:h].view(1, h, 1, -1).expand(f, h, w, -1),
                          fr[2][:w].view(1, 1, w, -1).expand(f, h, w, -1)], dim=-1).reshape(f * h * w, 1, -1).to(device)
    freqs, fbd = grid(model.pipe.dit.freqs), grid(model.freqs_bicross)
    fba = ns.dit.build_freqs_3d_with_extra_cis(model.freqs_bicross, f, h, w, n_extra=5, device=device)
    agg = model.vggt.aggregator
    pos = agg.position_getter(f, h, w, device=device) + 1
    pos = torch.cat([torch.zeros(f, agg.patch_start_idx, 2, device=device, dtype=pos.dtype), pos], dim=1)
    return freqs, fbd, fba, pos


def run_blocks_once(model, ns, inp, f, h, w, device, dt, which=("pcb", "frame", "irg"), reps=1):
    """Returns ({name: tensor}, {name: [ms]}).  `inp`: fwb_synth.synth_block_inputs (fp32 CPU, bf16-valued)."""
    freqs, fbd, fba, pos = grid_tables(model, ns, f, h, w, device)
    d = {k: v.to(device=device, dtype=(torch.float32 if k == "e0" else dt)) for k, v in inp.items()}
    lens = torch.ones(f, dtype=torch.long, device=device)
    lens[1:] = 4
    kw = dict(plucker_fea=d["plucker"], plucker_context_lens=lens)
    agg = model.vggt.aggregator
    P, C = d["x_agg"].shape[1], d["x_agg"].shape[2]
    outs, times = {}, {}
    if "pcb" in which:
        outs["pcb"], times["pcb"] = timed(lambda: model.pipe.dit.blocks[0](d["x_dit"], d["context"], d["t_mod"], freqs, **kw), device, reps)
    if "frame" in which:
        r, times["frame"] = timed(lambda: agg._process_frame_attention(d["x_agg"], 1, f, P, C, 0, pos=pos, e0=d["e0"]), device, reps)
        outs["frame"] = r[0]
    if "irg" in which:
        r, times["irg"] = timed(lambda: model.IRGBlock[0](x_dit=d["x_dit"], x_agg=d["x_agg"], context=d["context"], t_mod=d["t_mod"],
                                                           freqs=freqs, freqs_dit=fbd, freqs_agg=fba, pos=pos, e0=d["e0"], uncond=False, **kw),
                                device, reps)
        outs["irg_x"], outs["irg_tokens"] = r[0], r[1]
    return outs, times


def cmd_blocks(a):
    f, h, w = a.grid
    model, ns = build(2, 1, False, a.device)
    inp = S.synth_block_inputs(f, h, w, a.text_len, a.seed)
    out_dir = Path(a.out) if a.out else None
    if out_dir:
        out_dir.mkdir(parents=True, exist_ok=True)
    report = {"cmd": "blocks", "grid": [f, h, w], "device": a.device, "flash_attn_detected": bool(ns.dit.FLASH_ATTN_2_AVAILABLE),
              "torch": torch.__version__, "ref_root": shim.REF_ROOT, "modes": {}}
    for mode in a.modes:
        with mode_ctx(model, ns, mode, a.device) as dt:
            if a.warmup:
                run_blocks_once(model, ns, inp, f, h, w, a.device, dt, reps=1)
            outs, times = run_blocks_once(model, ns, inp, f, h, w, a.device, dt, reps=a.reps)
            backend = "flash_attn_func" if ns.dit.FLASH_ATTN_2_AVAILABLE else "F.scaled_dot_product_attention"
        _sync(a.device)
        report["modes"][mode] = {"ms": {k: min(v) for k, v in times.items()}, "dit_attention_backend": backend,
                                 "dtypes": {k: str(v.dtype) for k, v in outs.items()}}
        if out_dir:
            torch.save({k: v.detach().cpu() for k, v in outs.items()}, out_dir / f"blocks_{mode}.pt")
        del outs
    print(json.dumps(report))


def joint_inputs(f, h, w, text_len, device, dt):
    inp = S.synth_inputs(f, h, w, device="cpu", seed=1024, text_len=text_len, dtype=torch.bfloat16)
    return {k: v.to(device=device, dtype=dt) for k, v in inp.items()}


def cmd_joint(a):
    f, h, w = a.grid
    model, ns = build(a.pcb + a.irg, a.pcb, a.heads, a.device)
    if a.heads:
        idx = [min(a.irg - 1, i) for i in a.head_layers]
        model.vggt.depth_head.intermediate_layer_idx = idx
        model.vggt.point_head.intermediate_layer_idx = idx
    out_dir = Path(a.out) if a.out else None
    if out_dir:
        out_dir.mkdir(parents=True, exist_ok=True)
    report = {"cmd": "joint", "grid": [f, h, w], "pcb": a.pcb, "irg": a.irg, "heads": a.heads, "device": a.device, "modes": {}}
    lens = torch.ones(f, dtype=torch.long, device=a.device)
    lens[1:] = 4
    for mode in a.modes:
        with mode_ctx(model, ns, mode, a.device) as dt:
            d = joint_inputs(f, h, w, a.text_len, a.device, dt)
            ts = torch.tensor([a.timestep], device=a.device, dtype=dt)

            def fwd():
                return model.joint_forward(d["latents"], timestep=ts, context=d["context_pos"], clip_feature=d["clip_feature"], y=d["y"],
                                           use_gradient_checkpointing=False, plucker_fea=d["plucker_fea"], plucker_context_lens=lens,
                                           return_prediction=a.heads)
            (out, pred), ms = timed(fwd, a.device, a.reps)
        report["modes"][mode] = {"ms": min(ms)}
        if out_dir:
            blob = {"out": out.detach().cpu()}
            if pred is not None:
                blob["pred"] = {k: v.detach().cpu() for k, v in pred.items()}
            torch.save(blob, out_dir / f"joint_{mode}.pt")
        del out, pred
    print(json.dumps(report))


def cmd_step(a):
    """K denoise steps through the reference's own joint_forward + scheduler (loop body of model_wan21.py:289-322), once per
    requested mode (the model is built once; e.g. bf16_fa2 then bf16_sdpa = both FLASH_ATTN_2_AVAILABLE settings)."""
    f, h, w = a.grid
    model, ns = build(a.pcb + a.irg, a.pcb, False, a.device)
    lens = torch.ones(f, dtype=torch.long, device=a.device)
    lens[1:] = 4
    sched = model.pipe.scheduler
    sched.set_timesteps(50)
    runs = {}
    for mode in a.modes:
        with mode_ctx(model, ns, mode, a.device) as dt:
            d = joint_inputs(f, h, w, a.text_len, a.device, dt)
            lat = d["latents"].clone()
            kw = dict(clip_feature=d["clip_feature"], y=d["y"], use_gradient_checkpointing=False, plucker_fea=d["plucker_fea"],
                      plucker_context_lens=lens)

            def one(i, lat):
                t = sched.timesteps[i % len(sched.timesteps)].unsqueeze(0).to(dtype=dt, device=a.device)
                pos, _ = model.joint_forward(lat, timestep=t, context=d["context_pos"], **kw)
                neg, _ = model.joint_forward(lat, timestep=t, context=d["context_neg"], **kw)
                pred = neg + 5.0 * (pos - neg)
                return sched.step(pred, sched.timesteps[i % len(sched.timesteps)], lat)

            for i in range(a.warmup):
                lat = one(i, lat)
            _sync(a.device)
            ms = []
            for i in range(a.steps):
                (lat), m = timed(lambda: one(a.warmup + i, lat), a.device, 1)
                ms.append(m[0])
            backend = "flash_attn_func" if ns.dit.FLASH_ATTN_2_AVAILABLE else "F.scaled_dot_product_attention"
        runs[mode] = {"ms_per_step": sum(ms) / len(ms), "ms_each": ms, "dit_attention_backend": backend,
                      "finite": bool(torch.isfinite(lat.float()).all())}
        del d, lat
    mem = torch.cuda.max_memory_allocated() / 2**30 if torch.device(a.device).type == "cuda" else None
    first = runs[a.modes[0]]
    print(json.dumps({"cmd": "step", "grid": [f, h, w], "pcb": a.pcb, "irg": a.irg, "mode": a.modes[0], "device": a.device, "steps": a.steps,
                      "warmup": a.warmup, "ms_per_step": first["ms_per_step"], "ms_each": first["ms_each"],
                      "dit_attention_backend": first["dit_attention_backend"], "finite": first["finite"], "modes": runs,
                      "max_mem_gib": mem, "threads": torch.get_num_threads()}))


def cmd_schema(a):
    """state_dict key -> shape of the reference fusion model at the given depth, built on the meta device (no storage)."""
    with torch.device("meta"):
        model, ns = shim.build_reference_fusion(num_dit_layers=a.pcb + a.irg, start_index=a.pcb, heads=True, flash_attn=False, dtype=None)
    schema = {k: list(v.shape) for k, v in model.state_dict().items()}
    if a.out:
        Path(a.out).write_text(json.dumps(schema))
    import hashlib
    digest = hashlib.sha256(json.dumps(sorted(schema.items())).encode()).hexdigest()
    print(json.dumps({"cmd": "schema", "pcb": a.pcb, "irg": a.irg, "keys": len(schema), "sha256": digest}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("cmd", choices=["blocks", "joint", "step", "schema"])
    ap.add_argument("--device", default="cuda" if torch.cuda.is_available() else "cpu")
    ap.add_argument("--grid", type=int, nargs=3, default=[1, 4, 4])
    ap.add_argument("--text-len", type=int, default=512)
    ap.add_argument("--seed", type=int, default=1024)
    ap.add_argument("--modes", default="bf16_fa2,bf16_sdpa,fp32")
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=1)
    ap.add_argument("--warmup", type=int, default=0)
    ap.add_argument("--steps", type=int, default=1)
    ap.add_argument("--pcb", type=int, default=1)
    ap.add_argument("--irg", type=int, default=1)
    ap.add_argument("--heads", action="store_true")
    ap.add_argument("--head-layers", type=int, nargs=4, default=[3, 2, 1, 0])
    ap.add_argument("--timestep", type=float, default=996.0)
    ap.add_argument("--threads", type=int, default=0)
    a = ap.parse_args()
    a.modes = [m for m in a.modes.split(",") if m]
    assert all(m in MODES for m in a.modes), a.modes
    if a.threads:
        torch.set_num_threads(a.threads)
    real_stdout = os.dup(1)          # the reference prints; keep stdout for the one JSON line
    os.dup2(2, 1)
    import io
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        {"blocks": cmd_blocks, "joint": cmd_joint, "step": cmd_step, "schema": cmd_schema}[a.cmd](a)
    os.write(real_stdout, buf.getvalue().strip().splitlines()[-1].encode() + b"\n")


if __name__ == "__main__":
    main()
