"""Golden of the UNMODIFIED reference at batch 2 (staged under oracle/_ref by oracle/make_ref.py, run through
oracle/ref_runner.py's model builder and precision modes in a process of its own), for tests/test_batch_cpu.py and
tests/test_gpu_batch.py:

    python tools/make_golden_batch.py [OUT]        # OUT defaults to tests/golden; writes batch_joint.pt (a few CPU minutes)

Configuration: 1 PCB + 1 IRG block at 14B widths, geometry heads on (head layers [0, 0, 0, 0]), fp32 on the CPU (the
"golden fp32" mode of ref_runner), token grid f,h,w = 2,2,3, text length 16, per-key synthetic weights generated on the CPU.
Sample i has the seeded inputs fwb_synth.synth_inputs(seed=1024 + i): its own latents, y, context, CLIP feature and Plücker
features.  Runs, each stored per sample as the fixed element sample of tests/_common.py:take_sample:

  single       the two samples as two batch-1 joint_forward calls, timestep 996
  batch        one batch-2 call, timestep 996 (shared)
  zero_cam     batch 2 with sample 1's Plücker features all zero (the reference tests the whole tensor for all-zero,
               camera_control.py:111, so sample 1 still gets the camera shift)
  zero_cam_single1   sample 1 alone with all-zero Plücker features (the shift is skipped)
  distinct_t   batch 2 with timesteps [900, 500], and single_t the two batch-1 runs at 900 and 500

Each per-sample tensor is kept as take_sample(t, N_SAMPLE); config["n_sample"] records N_SAMPLE for the tests.
"""
from __future__ import annotations

import importlib.util
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
GRID = (2, 2, 3)
TEXT_LEN = 16
SEEDS = (1024, 1025)
TIMESTEP = 996.0
DISTINCT_T = (900.0, 500.0)
HEAD_LAYERS = [0, 0, 0, 0]       # min(irg - 1, i) for the default [3, 2, 1, 0] at one IRG block
N_SAMPLE = 2048                  # elements kept per tensor (take_sample), so that the eleven runs stay under 1 MB


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def child(out_path):
    """Runs in its own process: oracle/ref_runner.py takes the repository off sys.path so that `FantasyWorld` is the reference."""
    rr = _load("fwb_ref_runner", ROOT / "oracle" / "ref_runner.py")
    common = _load("fwb_tests_common", ROOT / "tests" / "_common.py")
    torch = rr.torch
    torch.set_num_threads(max(1, torch.get_num_threads()))
    f, h, w = GRID
    model, ns = rr.build(2, 1, True, "cpu")
    model.vggt.depth_head.intermediate_layer_idx = list(HEAD_LAYERS)
    model.vggt.point_head.intermediate_layer_idx = list(HEAD_LAYERS)
    lens = torch.ones(f, dtype=torch.long)
    lens[1:] = 4
    res = {"config": {"grid": list(GRID), "text_len": TEXT_LEN, "pcb": 1, "irg": 1, "heads": True, "head_layers": HEAD_LAYERS,
                      "seeds": list(SEEDS), "timestep": TIMESTEP, "n_sample": N_SAMPLE, "distinct_timesteps": list(DISTINCT_T), "mode": "fp32",
                      "device": "cpu", "torch": torch.__version__}}
    with rr.mode_ctx(model, ns, "fp32", "cpu") as dt:
        inp = [{k: v.to(dt) for k, v in rr.S.synth_inputs(f, h, w, device="cpu", seed=s, text_len=TEXT_LEN, dtype=torch.bfloat16).items()}
               for s in SEEDS]

        def fwd(samples, ts, zero_plucker=()):
            d = {k: torch.cat([s[k] for s in samples]) for k in samples[0]}
            for i in zero_plucker:
                d["plucker_fea"][i] = 0
            t = torch.tensor(ts, dtype=dt)
            out, pred = model.joint_forward(d["latents"], timestep=t, context=d["context_pos"], clip_feature=d["clip_feature"], y=d["y"],
                                            use_gradient_checkpointing=False, plucker_fea=d["plucker_fea"], plucker_context_lens=lens,
                                            return_prediction=True)
            return [{"out": out[i].detach().clone(), "pred": {k: v[i].detach().clone() for k, v in pred.items()}}
                    for i in range(len(samples))]

        full = {"single": fwd(inp[:1], [TIMESTEP]) + fwd(inp[1:], [TIMESTEP]),
                "batch": fwd(inp, [TIMESTEP]),
                "zero_cam": fwd(inp, [TIMESTEP], zero_plucker=(1,)),
                "zero_cam_single1": fwd(inp[1:], [TIMESTEP], zero_plucker=(0,)),
                "distinct_t": fwd(inp, list(DISTINCT_T)),
                "single_t": fwd(inp[:1], [DISTINCT_T[0]]) + fwd(inp[1:], [DISTINCT_T[1]])}

    def diff(a, b):
        return max([float((a["out"] - b["out"]).abs().max())] + [float((a["pred"][k] - b["pred"][k]).abs().max()) for k in a["pred"]])

    res["report"] = {
        "batch_vs_single_max_abs": [diff(full["batch"][i], full["single"][i]) for i in range(2)],
        "zero_cam_sample0_vs_single_max_abs": diff(full["zero_cam"][0], full["single"][0]),
        "zero_cam_sample1_vs_zero_cam_single1_max_abs": diff(full["zero_cam"][1], full["zero_cam_single1"][0]),
        "distinct_t_vs_single_t_max_abs": [diff(full["distinct_t"][i], full["single_t"][i]) for i in range(2)],
    }
    ex = full["single"][0]
    res["shape"] = {"out": list(ex["out"].shape), **{f"pred/{k}": list(v.shape) for k, v in ex["pred"].items()}}
    for run, samples in full.items():
        res[run] = [{"out": common.take_sample(s["out"], N_SAMPLE), "pred": {k: common.take_sample(v, N_SAMPLE) for k, v in s["pred"].items()}}
                    for s in samples]
    torch.save(res, out_path)
    print(json.dumps(res["report"]))


def main():
    out = Path(sys.argv[1]).resolve() if len(sys.argv) > 1 else ROOT / "tests" / "golden"
    out.mkdir(parents=True, exist_ok=True)
    assert (ROOT / "oracle" / "_ref" / "FantasyWorld").exists(), "reference not staged: python oracle/make_ref.py"
    r = subprocess.run([sys.executable, __file__, "--child", str(out / "batch_joint.pt")], cwd=str(out), capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    print(r.stdout.strip().splitlines()[-1])


if __name__ == "__main__":
    if sys.argv[1:2] == ["--child"]:
        child(Path(sys.argv[2]))
    else:
        main()
