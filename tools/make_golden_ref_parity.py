"""Goldens from the UNMODIFIED reference (staged under oracle/_ref by oracle/make_ref.py), run through oracle/ref_runner.py in
its own process, for the tests that compare this repo with the reference:

    python tools/make_golden_ref_parity.py cpu [OUT]   # ref_runner_blocks_cpu.pt, reference_cli_imports.json, pose_enc_ref.pt
    python tools/make_golden_ref_parity.py gpu [OUT]   # on a B200: ref_parity_blocks_<name>.pt, ref_parity_joint_<mode>.pt,
                                                       #            ref_parity_deep.pt

OUT defaults to tests/golden.  The GPU outputs at the C2 token count run to hundreds of MB, so each tensor is reduced to the
fixed element sample of tests/_common.py:take_sample; tests/test_gpu_ref_parity.py takes the same elements of its own outputs.
"""
from __future__ import annotations

import ast
import json
import os
import subprocess
import sys
import tempfile
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tests"))
from _common import take_sample  # noqa: E402

REF = ROOT / "oracle" / "_ref"
C2 = (21, 30, 52)


def run_ref(args, out):
    env = dict(os.environ)
    env.pop("PYTHONPATH", None)
    r = subprocess.run([sys.executable, str(ROOT / "oracle" / "ref_runner.py"), *map(str, args), "--out", str(out)], capture_output=True,
                       text=True, env=env)
    assert r.returncode == 0, r.stderr[-3000:]
    rep = json.loads(r.stdout.strip().splitlines()[-1])
    rep.pop("ref_root", None)
    return rep


def sampled(blob):
    """{"out": tensor, "pred": {k: tensor}} -> the same structure of element samples, plus every full shape."""
    res = {"out": take_sample(blob["out"]), "shape": {"out": list(blob["out"].shape)}}
    if blob.get("pred") is not None:
        res["pred"] = {k: take_sample(v) for k, v in blob["pred"].items()}
        res["shape"].update({f"pred/{k}": list(v.shape) for k, v in blob["pred"].items()})
    return res


def gpu(out_dir):
    with tempfile.TemporaryDirectory() as tmp:
        d = Path(tmp)
        # test_block_at_c2_token_count_vs_reference_cuda_bf16: one file per block output, all three modes
        rep = run_ref(["blocks", "--device", "cuda", "--grid", *C2, "--text-len", 512, "--modes", "bf16_fa2,bf16_sdpa,fp32",
                       "--warmup", 1, "--reps", 2], d / "blocks")
        modes = {m: torch.load(d / "blocks" / f"blocks_{m}.pt") for m in ("bf16_fa2", "bf16_sdpa", "fp32")}
        for name in ("pcb", "frame", "irg_x", "irg_tokens"):
            torch.save({"report": rep, "grid": C2, "shape": list(modes["fp32"][name].shape),
                        **{m: take_sample(t[name]) for m, t in modes.items()}}, out_dir / f"ref_parity_blocks_{name}.pt")
        del modes
        # test_reduced_joint_forward_with_heads_at_c2_vs_reference_cuda_bf16: 2 PCB + 2 IRG with the heads, one file per mode
        rep = run_ref(["joint", "--device", "cuda", "--grid", *C2, "--text-len", 512, "--modes", "bf16_fa2,bf16_sdpa,fp32",
                       "--pcb", 2, "--irg", 2, "--heads", "--head-layers", 3, 2, 1, 0], d / "joint")
        for m in ("bf16_fa2", "bf16_sdpa", "fp32"):
            torch.save({"report": rep, "grid": C2, **sampled(torch.load(d / "joint" / f"joint_{m}.pt"))},
                       out_dir / f"ref_parity_joint_{m}.pt")
        # test_depth_drift_4pcb_4irg_vs_reference_cuda_bf16: small enough to keep whole
        rep = run_ref(["joint", "--device", "cuda", "--grid", 3, 8, 12, "--text-len", 64, "--modes", "bf16_fa2,fp32", "--pcb", 4,
                       "--irg", 4], d / "deep")
        torch.save({"report": rep, **{m: torch.load(d / "deep" / f"joint_{m}.pt")["out"] for m in ("bf16_fa2", "fp32")}},
                   out_dir / "ref_parity_deep.pt")


def cpu(out_dir):
    with tempfile.TemporaryDirectory() as tmp:
        # tests/test_ref_runner_cpu.py: the three blocks at f,h,w = 1,4,4 in fp32 on the CPU
        rep = run_ref(["blocks", "--device", "cpu", "--grid", 1, 4, 4, "--text-len", 64, "--modes", "fp32"], tmp)
        blob = torch.load(Path(tmp) / "blocks_fp32.pt")
        torch.save({"report": rep, **{k: v.clone() for k, v in blob.items()}}, out_dir / "ref_runner_blocks_cpu.pt")
    # tests/test_dropin.py: every `from FantasyWorld... import ...` of the reference's two CLIs
    imports = {}
    for cli in ("inference_wan21.py", "inference_wan22.py"):
        rows = []
        for node in ast.walk(ast.parse((REF / cli).read_text())):
            if isinstance(node, ast.ImportFrom) and node.module and node.module.startswith("FantasyWorld"):
                rows.append([node.module, [a.name for a in node.names]])
        imports[cli] = rows
    (out_dir / "reference_cli_imports.json").write_text(json.dumps(imports, indent=1) + "\n")
    # tests/test_dropin.py: the reference's pose-encoding helpers on the test's inputs
    code = f"""
import sys, importlib, torch
sys.path[:0] = [{str(ROOT / 'tests')!r}, {str(ROOT / 'fantasy-world_b200')!r}]
from test_dropin import pose_inputs
d = {str(REF / 'FantasyWorld' / 'vggt' / 'utils')!r}
import importlib.util
spec = importlib.util.spec_from_file_location("ref_vggt_utils", d + "/__init__.py", submodule_search_locations=[d])
pkg = importlib.util.module_from_spec(spec); sys.modules["ref_vggt_utils"] = pkg; spec.loader.exec_module(pkg)
pe, rot = importlib.import_module("ref_vggt_utils.pose_enc"), importlib.import_module("ref_vggt_utils.rotation")
q, R, ext, K = pose_inputs()
enc = pe.extri_intri_to_pose_encoding(ext, K, (480, 832))
e, k = pe.pose_encoding_to_extri_intri(enc, (480, 832))
torch.save({{"mat_to_quat": rot.mat_to_quat(R), "quat_to_mat": rot.quat_to_mat(q), "encoding": enc, "extri": e, "intri": k}},
           {str(out_dir / 'pose_enc_ref.pt')!r})
"""
    subprocess.run([sys.executable, "-c", code], check=True, cwd=str(ROOT / "tests"))


if __name__ == "__main__":
    which = sys.argv[1]
    out = Path(sys.argv[2]) if len(sys.argv) > 2 else ROOT / "tests" / "golden"
    out.mkdir(parents=True, exist_ok=True)
    assert (REF / "FantasyWorld").exists(), "reference not staged: python oracle/make_ref.py"
    {"cpu": cpu, "gpu": gpu}[which](out)
