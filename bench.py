"""bench.py — denoise-steps/sec of the FantasyWorld hot path (BASELINE.json metric) on N B200 GPUs of one node.

    python bench.py --gpus 1 --steps 3 --warmup 3                     # our CUDA path (default workload = configs[1])
    python bench.py --impl reference --steps 1 --warmup 0             # the reference's CPU path (oracle port) on host cores
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...  # N > 1: see DESIGN.md §multi-GPU

Workload (configs[1]): Wan2.1-I2V-14B-480P shape, random-init, latents [1,16,21,60,104] (81 frames, 480x832),
16 Preconditioning Blocks + 24 IRG blocks, one step = conditional + unconditional joint_forward + CFG + Euler update
(geometry heads excluded from the per-step metric, as in SURVEY §8d).  Synthetic inputs, synthetic weights.

One JSON line on stdout (rank 0).  `value`: inputs resident in HBM.  `e2e`: the same step through the public module API
(FantasyWorldFusionModel.denoise_step) from pinned HOST buffers, H2D of the step's latents and D2H of the result inside
the timed region (conditioning tensors are uploaded once per run inside the timed region and amortised over the steps).
`roofline`: the dominant kernel (DiT self-attention, fwb_attn_fwd D=128) timed per launch with CUDA events during the
timed steps.  `cpu_baseline`: oracle port on the host cores, bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
PKG = ROOT / "fantasy-world_b200"
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))
# NOTE: fantasy-world_b200/ (the kernel-backed `FantasyWorld` mirror + fwb200) is put on sys.path by run_ours() only.  The
# reference arm (--impl reference) imports the UNMODIFIED reference, whose package is also called `FantasyWorld`, and must
# neither see the mirror nor map libfwb200.so.

STEP_FLOP_C2 = 4.267e15          # algorithmic FLOP per denoise step at C2 (SURVEY Appendix C / BASELINE.md §2)


def forward_flops(f, h, w, n_pcb, n_irg, text_len=512, clip=True, camera_adaln=True):
    """Algorithmic FLOPs of one joint_forward (attention 4*H*Lq*Lk*D, GEMM 2*M*N*K), same accounting as SURVEY App. C.
    Wan2.2: clip=False (512 text tokens only), camera_adaln=False (the camera enters through the hoisted control adapter)."""
    L, P = f * h * w, 5 + h * w
    N = f * P
    C, Fd = 5120, 13824
    ctx = text_len + (257 if clip else 0)
    dit = 2 * L * C * C * 4 + 4 * 40 * L * L * 128                        # qkvo + self-attn
    dit += 2 * L * C * C * 2 + 4 * 40 * L * ctx * 128                      # cross q,o + attn (K/V of the context are hoisted)
    dit += 2 * L * C * Fd * 2                                              # FFN
    cam = 2 * L * (C * 1024 + 1024 * 2048 + 2048 * 409 + 409 * C) if camera_adaln else 0   # camera AdaLN MLPs (group1 hoisted)
    vg_lin = 2 * N * 1024 * (3072 + 1024 + 4096 + 4096)
    frame = vg_lin + 4 * 16 * f * P * P * 64
    glob = vg_lin + 4 * 16 * N * N * 64
    adapter = 2 * L * C * 2304 + 2 * N * 1024 * 2304 + 2 * L * 1152 * C + 2 * N * 1152 * 1024 + 2 * 4 * 12 * L * N * 96
    total = n_pcb * (dit + cam) + n_irg * (frame + dit + glob + adapter) + min(n_irg, 9) * cam
    total += 2 * L * C * 1024                                              # projection head
    return float(total)


def vggt_forward_flops(f, h, w, n_blocks=24):
    """Aggregator of the stand-alone geometry branch: projection + n_blocks x (frame block + global block).  The heads'
    convolutions are not counted (they run on cuDNN, once per video)."""
    L, P = f * h * w, 5 + h * w
    N = f * P
    vg_lin = 2 * N * 1024 * (3072 + 1024 + 4096 + 4096)
    return float(2 * L * 5120 * 1024 + n_blocks * (2 * vg_lin + 4 * 16 * f * P * P * 64 + 4 * 16 * N * N * 64))


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index=0):
        super().__init__(daemon=True)
        self.gpu, self.stop_flag, self.rows = gpu_index, threading.Event(), []

    def run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured (MEASURED_PEAKS.json)"
    return 1590.0, 1400.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference's algorithm on the host cores (bounded sample)
# ----------------------------------------------------------------------------------------------------------------------
def usable_cores():
    """Host threads this process can really use: the affinity mask, capped by the cgroup CPU quota when there is one
    (os.cpu_count() reports the machine, and oversubscribing a quota makes the CPU arm look worse than it is)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = Path(path).read_text().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                per = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read_text())
                if q > 0:
                    n = min(n, max(1, int(q / per + 0.5)))
            break
        except Exception:
            continue
    return n


def sample_flops(f, h, w, text_len=512):
    """Algorithmic FLOPs of the CPU sample (1 PCB DiT block + 1 VGGT frame block + 1 IRG block at f,h,w).  The reference
    recomputes the context K/V and the camera group1 projection inside every block (no hoisting): counted."""
    L = f * h * w
    extra_kv = 2 * 2 * (text_len + 257) * 5120 * 5120 * 2 + 2 * 2 * L * 2048 * 2048
    return forward_flops(f, h, w, 1, 1, text_len) - 2 * L * 5120 * 1024 + extra_kv


class CpuReference:
    """The reference's own modules on the host cores (fp32, F.scaled_dot_product_attention, all usable threads).

    kind "reference": the UNMODIFIED reference staged under oracle/_ref through oracle/ref_runner.py —
    one PCB DiTBlock, one VGGT frame Block and one IRGBlock at full 14B widths.  kind "port": oracle/fw_oracle.py, used only
    when no reference is staged.  Only this class and tests/ touch oracle/."""

    def __init__(self):
        import torch
        torch.set_num_threads(usable_cores())
        self.torch = torch
        self.kind = "port"
        self.model = self.ns = self.R = None
        try:
            from oracle import ref_runner as R          # strips the mirror from sys.path, loads fwb_synth + the shim by path
            if R.shim.reference_available():
                self.R = R
                self.model, self.ns = R.build(2, 1, False, "cpu")
                self.kind = "reference"
        except Exception as e:                           # staged copy missing / broken: fall back to the port, say so
            self.err = f"{type(e).__name__}: {e}"
        if self.kind == "port":
            self._init_port()

    def _init_port(self):
        import importlib.util
        spec = importlib.util.spec_from_file_location("fwb_synth", PKG / "fwb_synth.py")
        S = sys.modules.get("fwb_synth") or importlib.util.module_from_spec(spec)
        if "fwb_synth" not in sys.modules:
            sys.modules["fwb_synth"] = S
            spec.loader.exec_module(S)
        schema = json.loads((ROOT / "tests" / "golden" / "schema_reduced.json").read_text())
        keys = [k for k in schema if k.startswith(("pipe.dit.blocks.0.", "vggt.aggregator.frame_blocks.0.", "IRGBlock.0.",
                                                    "vggt.aggregator.camera_token", "vggt.aggregator.register_token"))]
        self.sd = {k: S.synth_tensor(k, schema[k], 0, "cpu") for k in keys}
        self.S = S

    def sample(self, f=1, h=30, w=52, text_len=512):
        """Seconds for one sample at f,h,w; returns (seconds, algorithmic FLOPs, description)."""
        torch = self.torch
        if self.kind == "reference":
            R = self.R
            inp = R.S.synth_block_inputs(f, h, w, text_len)
            with R.mode_ctx(self.model, self.ns, "fp32", "cpu") as dt:
                t0 = time.perf_counter()
                R.run_blocks_once(self.model, self.ns, inp, f, h, w, "cpu", dt)
                sec = time.perf_counter() - t0
            what = "UNMODIFIED reference modules (oracle/_ref)"
        else:
            from oracle import fw_oracle as O
            inp = self.S.synth_block_inputs(f, h, w, text_len)
            tab, tab_d, tab_a = O.rope_table_3d(128, f, h, w), O.rope_table_3d(96, f, h, w), O.rope_table_3d_with_extra(96, f, h, w, 5)
            _, pos = O.aggregator_input(self.sd, "vggt.aggregator", torch.zeros(1, f, h, w, 1024))
            O.USE_TORCH_SDPA = True      # time what the reference runs on CPU (F.scaled_dot_product_attention)
            t0 = time.perf_counter()
            with torch.no_grad():
                x1 = O.dit_block(self.sd, "pipe.dit.blocks.0", inp["x_dit"], inp["context"], inp["t_mod"], tab, inp["plucker"])
                tk = O.vggt_block(self.sd, "vggt.aggregator.frame_blocks.0", inp["x_agg"], pos, inp["e0"])
                O.irg_block(self.sd, "IRGBlock.0", x1, tk, inp["context"], inp["t_mod"], tab, tab_d, tab_a, pos, inp["e0"], inp["plucker"])
            sec = time.perf_counter() - t0
            O.USE_TORCH_SDPA = False
            what = "fp32 oracle port (no reference staged)"
        return sec, sample_flops(f, h, w, text_len), (f"1 PCB DiT block + 1 VGGT frame block + 1 IRG block at f,h,w={f},{h},{w} "
                                                       f"(L={f * h * w}), fp32, {what}")

    def reduced_e2e(self, f=3, h=30, w=52, text_len=512):
        """A COMPLETE reduced problem, not extrapolated: one denoise step (2 x joint_forward + CFG + scheduler.step) of the
        1 PCB + 1 IRG model at f,h,w through the reference's own joint_forward (BASELINE.md §3 item 3)."""
        if self.kind != "reference":
            return None
        R, torch = self.R, self.torch
        model = self.model
        lens = torch.ones(f, dtype=torch.long)
        lens[1:] = 4
        sched = model.pipe.scheduler
        sched.set_timesteps(50)
        with R.mode_ctx(model, self.ns, "fp32", "cpu") as dt:
            d = R.joint_inputs(f, h, w, text_len, "cpu", dt)
            kw = dict(clip_feature=d["clip_feature"], y=d["y"], use_gradient_checkpointing=False, plucker_fea=d["plucker_fea"],
                      plucker_context_lens=lens)
            t = sched.timesteps[0].unsqueeze(0).to(dt)
            t0 = time.perf_counter()
            pos, _ = model.joint_forward(d["latents"], timestep=t, context=d["context_pos"], **kw)
            neg, _ = model.joint_forward(d["latents"], timestep=t, context=d["context_neg"], **kw)
            lat = sched.step(neg + 5.0 * (pos - neg), sched.timesteps[0], d["latents"])
            sec = time.perf_counter() - t0
        fl = 2 * (forward_flops(f, h, w, 1, 1, text_len))
        return {"grid": [f, h, w], "depth": "1 PCB + 1 IRG (14B widths)", "seconds_per_step": sec, "flop_per_step": fl,
                "achieved_tflops": fl / sec / 1e12, "finite": bool(torch.isfinite(lat).all()), "extrapolated": False}


def pick_sample_frames(sec_f1, n_samples, budget_s):
    """Largest sample (frames of the full 30x52 token grid) whose n_samples repetitions fit the time budget, from the measured
    1-frame sample and the FLOP ratio.  h,w are never reduced: every sample works on full C2 frames."""
    best = 1
    for f in (2, 3, 4, 6, 8, 12, 21):
        if sec_f1 * sample_flops(f, 30, 52) / sample_flops(1, 30, 52) * n_samples <= budget_s:
            best = f
    return best


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores.  Every timed "step" is one
    bounded sample of the C2 workload (contract ④); `ms_per_step` is the measured time of a sample, `value` the implied
    denoise-steps/s of the FULL C2 step (measured FLOP/s of the reference's algorithm / 4.27 PFLOP per step) and is labelled
    as extrapolated.  Two non-extrapolated points are added once: the same three blocks at the FULL C2 token count, and a
    complete reduced denoise step through joint_forward."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t_start = time.perf_counter()
    cpu = CpuReference()
    cores = usable_cores()
    n = args.warmup + args.steps
    sec1, _, _ = cpu.sample(f=1)
    fs = pick_sample_frames(sec1, n, args.cpu_budget)
    times, flops, desc = [], 0.0, ""
    for i in range(n):
        dt, flops, desc = cpu.sample(f=fs)
        if i >= args.warmup:
            times.append(dt)
    dt = sum(times) / len(times)
    rate = flops / dt                                   # FLOP/s of the reference algorithm on this host
    steps_per_s = rate / STEP_FLOP_C2
    extras = {}
    spent = time.perf_counter() - t_start
    est_full = dt * sample_flops(21, 30, 52) / flops
    if not args.no_cpu_full and est_full < max(60.0, 420.0 - spent):
        fdt, ffl, fdesc = cpu.sample(f=21)
        extras["full_token_sample"] = {"sample": fdesc, "seconds": fdt, "achieved_tflops": ffl / fdt / 1e12,
                                       "implied_steps_per_s": ffl / fdt / STEP_FLOP_C2, "extrapolated_from_blocks": True}
    else:
        extras["full_token_sample"] = {"skipped": "--no-cpu-full" if args.no_cpu_full else f"estimated {est_full:.0f} s exceeds the remaining budget"}
    if not args.no_cpu_full:
        try:
            extras["reduced_e2e"] = cpu.reduced_e2e()
        except Exception as e:
            extras["reduced_e2e"] = {"error": f"{type(e).__name__}: {e}"}
    line = {"metric": "denoise_steps_per_sec", "value": steps_per_s, "unit": "steps/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": "Wan2.1-I2V-14B-480P shape, latents 1x16x21x60x104 (81 frames), 16 PCB + 24 IRG, CFG 2 forwards/step",
                       "note": "each timed step is ONE bounded sample (ms_per_step = its measured time); value = measured FLOP/s of the "
                               "reference's algorithm / 4.267 PFLOP per C2 step, i.e. EXTRAPOLATED to the full step",
                       "same_config": False, "sample_frames": fs},
            "cpu_baseline": {"value": steps_per_s, "unit": "steps/s", "cores": cores, "kind": cpu.kind, "sample": desc,
                             "sample_seconds": dt, "achieved_tflops": rate / 1e12, **extras},
            "e2e": {"value": steps_per_s, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ----------------------------------------------------------------------------------------------------------------------
# GPU path
# ----------------------------------------------------------------------------------------------------------------------
def dominant_tag(L, world, H=40):
    """Profiling-tag prefix of the dominant kernel's launches: the self-attention (H heads) of this rank's L / world query rows.
    Under sequence parallelism every attention runs as split-KV partials over slices of the keys, and the slices may be ragged
    (4095 rows per rank in 4 slices = 1024, 1024, 1024, 1023), so the match is on the query side only."""
    return f"attn:B1:H{H}:Lq{L // world}:Lk"


def roofline_from_prof(prof, L, world, step_ms_total, sustained_peak, peak_src, H=40, D=128, kernel=None):
    """The `roofline` object from the CUDA-event records {tag: (launches, total_ms)} of the timed region (pure function)."""
    tag = dominant_tag(L, world, H)

    def lk(t):
        return int(t.split(":Lk")[1].split(":")[0])

    # the text / CLIP cross-attentions share the prefix (same q) but have 512 / 257 keys: not the dominant kernel
    dom = {t: v for t, v in prof.items() if t.startswith(tag) and t.endswith(f":D{D}") and lk(t) > 1024}
    if not dom:
        return None
    cnt = sum(c for c, _ in dom.values())
    tot = sum(ms_ for _, ms_ in dom.values())
    fl_total = sum(c * 4.0 * H * (L // world) * lk(t) * D for t, (c, _) in dom.items())
    ach = fl_total / (tot * 1e-3) / 1e12
    traffic, traffic_src = None, None
    tp = ROOT / "profiles" / "attn_d128_dram_bytes.json"
    if tp.exists() and world == 1 and L == 32760 and D == 128:        # the ncu capture is of the full-size single-GPU launch
        try:
            rec = json.loads(tp.read_text())
            traffic = rec.get("dram_bytes_per_launch")
            traffic_src = rec.get("source", "ncu --set full capture, see profiles/")
        except Exception:
            traffic = None
    return {"kernel": kernel or "attn_fwd_mc_kernel<128> (DiT self-attention: aliased S/P kernel in K/V-multicast CTA pairs, fwb_attn_fwd / fwb_attn_fwd_partial)", "bound": "tensor",
            "achieved": ach, "peak": sustained_peak, "unit": "TFLOP/s", "frac": ach / sustained_peak, "traffic": traffic,
            "traffic_source": traffic_src,
            "launches_timed": cnt, "ms_per_launch": tot / cnt, "flop_per_launch": fl_total / cnt,
            "peak_source": peak_src + ", sustained figure (kernel timed inside a long step)",
            "share_of_step": tot / step_ms_total}


DUMP_BYTES = 64 << 20


def dump_outputs(outs, out_dir):
    """Write {name: tensor} as out_dir/<name>.npy in float32, DUMP_BYTES in all.  A tensor larger than its share is written as
    the fixed sample (arange(n) * 2654435761 + 40503) mod numel of its flattened elements: the same positions on every run."""
    import numpy as np
    import torch
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    share = DUMP_BYTES // 4 // len(outs)
    for name, t in outs.items():
        t = t.detach()
        if t.numel() > share:
            t = t.reshape(-1)[(torch.arange(share, device=t.device) * 2654435761 + 40503) % t.numel()]
        np.save(out_dir / f"{name}.npy", t.float().cpu().numpy())


def _subprocess_json(cmd, timeout):
    """Run a helper process and parse the last stdout line as JSON ({"error": ...} on failure — a baseline leg must never
    take the measurement down with it)."""
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "PYTHONPATH"):
        env.pop(k, None)
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
        if r.returncode != 0:
            return {"error": f"rc {r.returncode}: {r.stderr.strip()[-400:]}"}
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"}


def gpu_reference_step(f, h, w, n_pcb, n_irg):
    """The UNMODIFIED reference on this same B200 (BASELINE.md §4): full-depth model under torch.autocast(bf16), one timed
    denoise step through its own joint_forward + scheduler (oracle/ref_runner.py `step`, separate process), after one warm-up."""
    if not (ROOT / "oracle" / "_ref" / "FantasyWorld").exists():
        return {"unavailable": "reference not staged (python oracle/make_ref.py)"}
    out = _subprocess_json([sys.executable, str(ROOT / "oracle" / "ref_runner.py"), "step", "--device", "cuda", "--grid", str(f), str(h), str(w),
                            "--pcb", str(n_pcb), "--irg", str(n_irg), "--steps", "1", "--warmup", "1", "--modes", "bf16_fa2,bf16_sdpa"], timeout=1200)
    if "ms_per_step" in out:
        out["steps_per_s"] = 1e3 / out["ms_per_step"]          # the reference's default path on this box (flash-attn for the DiT)
        for m in out.get("modes", {}).values():
            m["steps_per_s"] = 1e3 / m["ms_per_step"]
        out["what"] = "unmodified reference (oracle/_ref), model.to(bf16) + torch.autocast(cuda, bf16), same synthetic shapes, same GPU"
    return out


def run_ours(args):
    if str(PKG) not in sys.path:
        sys.path.insert(0, str(PKG))
    import torch
    import fwb200
    from fwb200.synth import build_fusion_model, synth_inputs

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    fwb200.require_device()
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    f, h, w = args.frames, args.h, args.w
    n_pcb, n_irg = args.pcb, args.irg
    wan22 = args.workload == "wan22_720p"
    model_low = None
    if wan22:
        # BASELINE configs[3]: Wan2.2-Fun-A14B-Control-Camera, two experts resident (high-noise / low-noise), switched by timestep
        from fwb200.synth import build_fusion_model_wan22
        from FantasyWorld.fusion.model_wan22 import denoise_step_experts
        model = build_fusion_model_wan22(num_dit_layers=n_pcb + n_irg, start_index=n_pcb, device=dev, seed=0)
        model_low = build_fusion_model_wan22(num_dit_layers=n_pcb + n_irg, start_index=n_pcb, device=dev, seed=1)
        model_low.pipe.device = dev
    else:
        model = build_fusion_model(num_dit_layers=n_pcb + n_irg, start_index=n_pcb, device=dev, seed=0, heads=False)
    model.pipe.device = dev
    inp = synth_inputs(f, h, w, device=dev, seed=1024, text_len=512)       # one sample, replicated inputs
    if wan22:
        g = torch.Generator(device="cpu").manual_seed(77)
        inp["control"] = torch.randn(1, 24, f, 16 * h, 16 * w, generator=g, dtype=torch.bfloat16).to(dev)   # Pluecker rays folded 4:1 in time
        inp.pop("clip_feature"), inp.pop("plucker_fea")
    par = "single"
    if world > 1:
        par = args.parallel if args.parallel != "auto" else ("cfg" if world % 2 == 0 else "sp")
        if par == "cfg":
            model.enable_cfg_parallel()       # pos / neg forwards on the two halves of the node, each half token-sharded (SURVEY §8e)
        else:
            from fwb200.sp import SPContext
            model.sp = SPContext()                                           # tokens sharded over all ranks
    if model_low is not None:
        model_low.sp, model_low.cfgp = model.sp, model.cfgp                  # one set of process groups for both experts
    lens = torch.ones(f, dtype=torch.long, device=dev)
    lens[1:] = 4
    sched = model.pipe.scheduler
    sched.set_timesteps(50)
    n_sched = len(sched.timesteps)

    def step_api(lat, i, c):
        """One denoise step through the public API on conditioning dict `c`; `lat` may be a pinned host tensor."""
        if wan22:
            # steps 0, 17, 34, 1, ... of the 50-step schedule: both experts are exercised inside any timed window (18 of 50 steps
            # lie above the t = 900 boundary)
            lat_dev = lat if lat.is_cuda else lat.to(dev, non_blocking=True)
            return denoise_step_experts(model, model_low, lat_dev.contiguous(), (i * 17) % n_sched, c["context_pos"], c["context_neg"],
                                        c["y"], c["control"], cfg_scale=5.0)[0]
        return model.denoise_step(lat, i % n_sched, c["context_pos"], c["context_neg"], clip_feature=c["clip_feature"],
                                  y=c["y"], plucker_fea=c["plucker_fea"], plucker_context_lens=lens, cfg_scale=5.0)[0]

    def one_step(lat, i):
        return step_api(lat, i, inp)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    lat = inp["latents"].clone()
    for i in range(args.warmup):
        lat = one_step(lat, i)
    barrier()

    # ---- timed region: device-resident inputs --------------------------------------------------------------------------
    L = f * h * w
    shards = world // 2 if par == "cfg" else world          # ranks one forward's tokens are sharded over
    dom_tag = dominant_tag(L, shards)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    fwb200.reset_launch_count()
    fwb200.prof_enable(prefixes=[dom_tag] if not args.breakdown else None)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if args.profiler_range:
        torch.cuda.profiler.start()             # ncu --profile-from-start off: capture exactly the timed steps
    e0.record()
    for i in range(args.steps):
        lat = one_step(lat, args.warmup + i)
    e1.record()
    barrier()
    if args.profiler_range:
        torch.cuda.profiler.stop()
    launches = fwb200.launch_count()
    prof = fwb200.prof_disable()
    ms = e0.elapsed_time(e1)
    if dist is not None:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    sampler.stop_flag.set()
    if args.dump_outputs and rank == 0:
        dump_outputs({"latents": lat}, args.dump_outputs)        # what denoise_step returned in the last timed step

    # ---- e2e: host buffers through the public API ------------------------------------------------------------------------
    host = {k: v.cpu().pin_memory() for k, v in inp.items()}
    lat_host = host["latents"].clone().pin_memory()
    out_host = torch.empty_like(lat_host).pin_memory()
    barrier()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    cond = {k: host[k].to(dev, non_blocking=True) for k in host if k != "latents"}
    h2d = sum(host[k].numel() * host[k].element_size() for k in cond)
    d2h = 0
    for i in range(args.steps):
        cur = step_api(lat_host, args.warmup + i, cond)
        out_host.copy_(cur, non_blocking=True)
        torch.cuda.current_stream().synchronize()       # the host needs the step's result before it can feed the next step
        lat_host.copy_(out_host)
        h2d += lat_host.numel() * lat_host.element_size()
        d2h += out_host.numel() * out_host.element_size()
    t1.record()
    barrier()
    ms_e2e = t0.elapsed_time(t1)
    if dist is not None:
        t = torch.tensor([ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = float(t)
        # all measurements are in: tear the NCCL groups down TOGETHER (rank 0 goes on alone to the CPU / reference legs, which take
        # minutes; a late one-sided destroy against peers that have already exited is what must not happen)
        dist.barrier()
        torch.cuda.synchronize()
        dist.destroy_process_group()

    if rank != 0:
        return
    steps_per_s = args.steps / (ms / 1e3)               # strong scaling: all ranks denoise ONE sample (sequence parallel)
    e2e_sps = args.steps / (ms_e2e / 1e3)
    burst, sustained, peak_src = peaks()
    roof = roofline_from_prof(prof, L, shards, ms, sustained, peak_src)
    fwd_fl = forward_flops(f, h, w, n_pcb, n_irg, clip=not wan22, camera_adaln=not wan22)
    full = (f, h, w, n_pcb, n_irg) == ((21, 45, 80, 16, 24) if wan22 else (21, 30, 52, 16, 24))
    sp_stats = (model.sp.n_gathers, model.sp.gather_bytes) if model.sp is not None else (0, 0)
    if par == "cfg":
        par_desc = (f"cfg2 x sp{world // 2}: conditional / unconditional forward on the two halves of the node, each half token-sharded "
                    f"sequence parallel (1 all-gather of packed K|V per attention inside a half), 1 prediction swap per step")
    elif par == "sp":
        par_desc = f"sp{world} (token-sharded sequence parallel, 1 all-gather of packed K|V per attention)"
    else:
        par_desc = "single"
    cpu = None
    if not args.no_cpu_baseline:
        # the reference's CPU path, in its own process (its package is called FantasyWorld like the mirror loaded here):
        # 2 bounded samples (1 warm-up) sized for ~20 s of CPU work
        ref = _subprocess_json([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                                "--cpu-budget", "30", "--no-cpu-full"], timeout=900)
        cpu = ref.get("cpu_baseline") or ref
        if isinstance(cpu, dict):
            cpu.pop("reduced_e2e", None), cpu.pop("full_token_sample", None)
    gpu_ref = None
    if world == 1 and args.gpu_reference != "off" and not wan22:
        del model, inp, host, cond
        torch.cuda.empty_cache()
        gpu_ref = gpu_reference_step(f, h, w, n_pcb, n_irg)
    line = {"metric": "denoise_steps_per_sec", "value": steps_per_s, "unit": "steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": ((("Wan2.2-Fun-A14B-Control-Camera 720p shape (BASELINE configs[3]), two experts resident, switched at t=900: "
                                      if wan22 else "Wan2.1-I2V-14B-480P shape (BASELINE configs[1]): ") if full
                                     else "REDUCED (not the headline config): ") +
                                    f"latents 1x16x{f}x{2 * h}x{2 * w}, {n_pcb} PCB + {n_irg} IRG blocks, 2 forwards/step (CFG 5.0), random-init"),
                       "tokens_video": L, "tokens_geometry": f * (5 + h * w), "flop_per_step": 2 * fwd_fl,
                       "achieved_tflops_per_gpu": 2 * fwd_fl * args.steps / (ms / 1e3) / 1e12 / world,
                       "parallelism": par_desc,
                       "sp_gathers_per_step": sp_stats[0] / max(1, args.warmup + 2 * args.steps),
                       "sp_gather_bytes_per_step": sp_stats[1] / max(1, args.warmup + 2 * args.steps),
                       "l2": "per-step working set (37 GB weights + >1 GB activations) exceeds the 126 MB L2; no flush needed"},
            "e2e": {"value": e2e_sps, "unit": "steps/s", "h2d_bytes_per_step": h2d / args.steps, "d2h_bytes_per_step": d2h / args.steps,
                    "api": ("denoise_step_experts" if wan22 else "FantasyWorldFusionModel.denoise_step") +
                           " from pinned host latents; conditioning uploaded once per run inside the timed region",
                    "note": "its own timed region of the same K steps, run after `value`'s; the copies (41 MB in, 4 MB out per step) are "
                            "0.01 % of a step, so the two differ by the board's run-to-run spread under its power cap (about +-1.5 %)"},
            "gpu_launches": launches, "clocks": sampler.summary(), "roofline": roof, "cpu_baseline": cpu,
            "gpu_reference": gpu_ref}
    if args.breakdown:
        agg = sorted(((t, c, ms_) for t, (c, ms_) in prof.items()), key=lambda r: -r[2])
        line["breakdown_ms_per_step"] = [{"tag": t, "launches_per_step": c / args.steps, "ms_per_step": m / args.steps} for t, c, m in agg[:40]]
    emit(line)


def run_vggt_only(args):
    """--workload vggt_only (BASELINE configs[4]): the stand-alone geometry branch — VGGT.forward(patch_token[1,5120,21,30,52], t) =
    5120->1024 projection, 24 x (frame block + global block) without the adapter, camera / depth / point heads for 81 frames at
    480x832 (reference: vggt/models/vggt.py:45-117).  One "step" = one such forward.  Single GPU (the path is once per video)."""
    if str(PKG) not in sys.path:
        sys.path.insert(0, str(PKG))
    import torch
    import fwb200
    from fwb200.synth import build_vggt
    assert int(os.environ.get("WORLD_SIZE", "1")) == 1, "vggt_only is a single-GPU workload"
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    fwb200.require_device()
    f, h, w = args.frames, args.h, args.w
    vggt = build_vggt(device=dev, seed=0, heads=True)
    g = torch.Generator(device="cpu").manual_seed(1024)
    patch_host = torch.randn(1, 5120, f, h, w, generator=g, dtype=torch.float32).to(torch.bfloat16).pin_memory()
    patch = patch_host.to(dev)
    t = torch.tensor([500.0], device=dev)

    def step(p_in):
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            return vggt(p_in, t=t)

    for _ in range(args.warmup):
        pred = step(patch)
    torch.cuda.synchronize()
    L, N = f * h * w, f * (5 + h * w)
    sampler = ClockSampler(0)
    sampler.start()
    fwb200.reset_launch_count()
    tag = dominant_tag(N, 1, H=16)
    fwb200.prof_enable(prefixes=[tag] if not args.breakdown else None)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        pred = step(patch)
    e1.record()
    torch.cuda.synchronize()
    launches = fwb200.launch_count()
    prof = fwb200.prof_disable()
    ms = e0.elapsed_time(e1)
    sampler.stop_flag.set()
    if args.dump_outputs:
        dump_outputs(pred, args.dump_outputs)                     # VGGT.forward's head outputs of the last timed step
    # e2e: patch tokens from pinned host memory, every head output read back
    outs = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in pred.items()}
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.steps):
        pred = step(patch_host.to(dev, non_blocking=True))
        for k, v in pred.items():
            outs[k].copy_(v, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    t1.record()
    torch.cuda.synchronize()
    ms_e2e = t0.elapsed_time(t1)
    burst, sustained, peak_src = peaks()
    roof = roofline_from_prof(prof, N, 1, ms, sustained, peak_src, H=16, D=64,
                              kernel="attn2_kernel<64,128> (VGGT global attention, H16 D64, fwb_attn_fwd)")
    fl = vggt_forward_flops(f, h, w)
    line = {"metric": "geometry_forwards_per_sec", "value": args.steps / (ms / 1e3), "unit": "forwards/s", "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"VGGT geometry branch only (BASELINE configs[4]): patch tokens 1x5120x{f}x{h}x{w}, 24 frame + 24 global blocks, "
                                   f"camera / depth / point heads for {4 * (f - 1) + 1} frames at {16 * h}x{16 * w}, random-init",
                       "tokens_geometry": N, "flop_per_step_aggregator": fl, "achieved_tflops_aggregator": fl * args.steps / (ms / 1e3) / 1e12,
                       "outputs": {k: list(v.shape) for k, v in pred.items()},
                       "l2": "activations (135 MB fp32 tokens, 0.4 GB qkv) and 2.4 GB of weights exceed the 126 MB L2; no flush needed"},
            "e2e": {"value": args.steps / (ms_e2e / 1e3), "unit": "forwards/s", "h2d_bytes_per_step": patch_host.numel() * 2,
                    "d2h_bytes_per_step": sum(v.numel() * v.element_size() for v in outs.values()),
                    "api": "VGGT.forward(patch_token, t) from a pinned host tensor; all head outputs copied back"},
            "gpu_launches": launches, "clocks": sampler.summary(), "roofline": roof, "cpu_baseline": None}
    if args.breakdown:
        agg = sorted(((tg, c, m_) for tg, (c, m_) in prof.items()), key=lambda r: -r[2])
        line["breakdown_ms_per_step"] = [{"tag": tg, "launches_per_step": c / args.steps, "ms_per_step": m / args.steps} for tg, c, m in agg[:30]]
    emit(line)


_JSON_FD = None


def protect_stdout():
    """Libraries (NCCL's version banner, torch warnings) may write to fd 1; the driver expects ONE JSON line there.  Keep a
    private copy of stdout for the result and point fd 1 at stderr for everything else."""
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_JSON_FD, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="wan21_480p", choices=["wan21_480p", "wan22_720p", "vggt_only"],
                    help="wan21_480p = BASELINE configs[1] (the headline metric); wan22_720p = configs[3] (meant for 8 GPUs); "
                         "vggt_only = configs[4], the stand-alone geometry branch with heads")
    ap.add_argument("--frames", type=int, default=21)
    ap.add_argument("--h", type=int, default=None)
    ap.add_argument("--w", type=int, default=None)
    ap.add_argument("--pcb", type=int, default=16)
    ap.add_argument("--irg", type=int, default=24)
    ap.add_argument("--breakdown", action="store_true", help="time every fwb200 launch with CUDA events and add a per-kernel table")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profiler-range", action="store_true",
                    help="cudaProfilerStart/Stop around the timed steps (for `ncu --profile-from-start off`; never a bench value)")
    ap.add_argument("--parallel", default="auto", choices=["auto", "cfg", "sp"],
                    help="N > 1: cfg = CFG-parallel x sequence-parallel halves (default for even N), sp = sequence parallel over all ranks")
    ap.add_argument("--gpu-reference", default="auto", choices=["auto", "off"],
                    help="N=1: also time the unmodified reference (oracle/_ref) on the same GPU, in its own process")
    ap.add_argument("--cpu-budget", type=float, default=200.0, help="--impl reference: seconds for warmup + steps samples")
    ap.add_argument("--no-cpu-full", action="store_true", help="--impl reference: skip the extra full-token-count sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (float32, 64 MB in all; a larger "
                         "output as a fixed sample of its elements), to compare two builds on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.h is None:
        args.h, args.w = (45, 80) if args.workload == "wan22_720p" else (30, 52)
    protect_stdout()
    if args.workload == "vggt_only" and args.impl != "reference":
        run_vggt_only(args)
        return
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
