"""Batch on one B200: ms per denoise step (Wan2.1-I2V-14B shapes, 16 PCB + 24 IRG blocks, CFG 5.0, random-init weights) for

    serial      batch 1, the two CFG forwards one after the other (the default path)
    batch_cfg   batch 1, the two CFG forwards as ONE forward of batch 2 (denoise_step(batch_cfg=True))
    two_per_call  batch 2 (two samples per call), serial CFG — compared with two batch-1 calls (2 x serial)

at the C2 grid (f,h,w = 21,30,52) and at a short clip (f = 5).  The boards run at their power cap, so the modes are timed as
in-step A/Bs: alternating one-step segments in one process, each mode warmed up first, CUDA events around each step, and the
median per mode reported.  Peak memory per mode is torch.cuda.max_memory_allocated over the mode's warm-up step: the 37 GB of
weights included and, at the second grid, the first grid's cached context K/V and RoPE tables too.  Outputs of serial and
batch_cfg from the same input are compared (with the attention tail split on, as in production).

    python tools/bench_batch.py [--rounds 4] [--pcb 16 --irg 24] [--grids 21,30,52 5,30,52] [--out FILE]

The report is printed as JSON (one line per grid, then the whole report) and, with --out, also written to FILE.
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
for p in (ROOT, ROOT / "fantasy-world_b200"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))


def gpu_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = None
    return info


def bench_grid(model, grid, rounds, lens_dev):
    import torch
    from fwb200.synth import synth_inputs
    f, h, w = grid
    one = synth_inputs(f, h, w, device="cuda", seed=1024, text_len=512)
    two_in = [one, synth_inputs(f, h, w, device="cuda", seed=1025, text_len=512)]
    two = {k: torch.cat([d[k] for d in two_in]) for k in one}
    lens = torch.ones(f, dtype=torch.long, device=lens_dev)
    lens[1:] = 4

    def step(d, i, **kw):
        return model.denoise_step(d["latents"].clone(), i, d["context_pos"], d["context_neg"], clip_feature=d["clip_feature"], y=d["y"],
                                  plucker_fea=d["plucker_fea"], plucker_context_lens=lens, cfg_scale=5.0, **kw)[0]

    modes = {"serial": lambda i: step(one, i), "batch_cfg": lambda i: step(one, i, batch_cfg=True),
             "two_per_call": lambda i: step(two, i)}
    res = {m: {"ms": []} for m in modes}
    outs = {}
    for m, fn in modes.items():                       # warm-up (every shape) + peak memory of the mode
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        outs[m] = fn(0)
        torch.cuda.synchronize()
        res[m]["peak_mem_gib"] = round(torch.cuda.max_memory_allocated() / 2 ** 30, 2)
    for r in range(rounds):                           # alternating one-step segments
        for m, fn in modes.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            fn(1 + r)
            b.record()
            torch.cuda.synchronize()
            res[m]["ms"].append(round(a.elapsed_time(b), 2))
    for m in modes:
        res[m]["ms_per_step"] = statistics.median(res[m]["ms"])
    s, bc, tw = (res[m]["ms_per_step"] for m in modes)
    diff = (outs["batch_cfg"].float() - outs["serial"].float())
    return {"grid": list(grid), "tokens_video": f * h * w, "modes": res,
            "batch_cfg_vs_serial": {"speedup": round(s / bc, 4), "max_abs_diff_after_one_step": float(diff.abs().max()),
                                    "rel_l2_diff": float(diff.norm() / outs["serial"].float().norm())},
            "two_per_call_vs_two_calls": {"ms_two_calls": 2 * s, "ms_one_call": tw, "speedup": round(2 * s / tw, 4)},
            "two_per_call_sample0_equals_serial": bool(torch.equal(outs["two_per_call"][:1], outs["serial"]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pcb", type=int, default=16)
    ap.add_argument("--irg", type=int, default=24)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--grids", nargs="+", default=["21,30,52", "5,30,52"])
    ap.add_argument("--out", default=None, help="also write the report to this JSON file")
    a = ap.parse_args()
    import torch
    import fwb200
    from fwb200.synth import build_fusion_model
    fwb200.require_device()
    torch.cuda.set_device(0)
    model = build_fusion_model(num_dit_layers=a.pcb + a.irg, start_index=a.pcb, device="cuda", seed=0, heads=False)
    model.pipe.scheduler.set_timesteps(50)
    rep = {"what": "ms per denoise step, one B200: serial CFG vs batch_cfg (batch 1), and two samples per call vs two calls",
           "model": f"Wan2.1-I2V-14B widths, {a.pcb} PCB + {a.irg} IRG blocks, random-init, CFG 5.0, text 512 tokens",
           "method": "alternating one-step segments in one process after a warm-up step per mode; CUDA events; median",
           "gpu": gpu_info(), "rounds": a.rounds, "torch": torch.__version__, "grids": []}
    with torch.no_grad():
        for g in a.grids:
            rep["grids"].append(bench_grid(model, tuple(int(x) for x in g.split(",")), a.rounds, "cuda"))
            print(json.dumps(rep["grids"][-1]), flush=True)
    print(json.dumps(rep))
    if a.out:
        out = Path(a.out)
        out.parent.mkdir(parents=True, exist_ok=True)
        out.write_text(json.dumps(rep, indent=1) + "\n")


if __name__ == "__main__":
    main()
