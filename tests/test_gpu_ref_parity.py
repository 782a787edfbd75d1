"""bf16 parity against the UNMODIFIED reference running on the same B200 (SURVEY §8c, VERDICT r1 item 1).

The reference ran on a B200 (tools/make_golden_ref_parity.py: oracle/ref_runner.py on the unmodified reference) under
`torch.autocast("cuda", bf16)` — exactly how inference_wan21.py:310 runs it — on the same per-key synthetic weights and seeded
inputs as this repo's CUDA path, at the BASELINE C2 token count (f,h,w = 21,30,52: L = 32760 video tokens, N = 32865 geometry
tokens).  Its outputs are stored as goldens, each tensor as the fixed sample of elements of _common.take_sample (the full
tensors run to hundreds of MB); the statistics below are taken over the same elements of this repo's outputs:

  * one PCB DiT block, one VGGT frame block, one IRG block in isolation,
  * a reduced-depth joint_forward (2 PCB + 2 IRG) with the geometry heads (depth / point / camera at 81 x 480 x 832).

Protocol (SURVEY §8c; rtol 1e-3 is below one bf16 ulp = 2^-8, so two correct bf16 implementations cannot agree on every
element):
  (i)  pass-fraction of assert_close(ours, ref_cuda_bf16, rtol=1e-3, atol=1e-4) and the bf16-ulp distance histogram, next to
       the SAME statistics between the reference's own two attention backends (flash_attn_func vs F.sdpa) as the yardstick;
       asserted: ours is at least as close to the reference as 0.9 x that yardstick allows, and above the stated floors;
  (ii) || ours - golden_fp32 ||  <=  1.5 x || ref_cuda_bf16 - golden_fp32 ||   (never less accurate than the reference),
       golden_fp32 = the reference with the same bf16-valued weights in fp32, TF32 off; no additive slack.
The full report is written to gpurun_out/r02_ref_parity.json (committed under profiles/).
"""
import json
from pathlib import Path

import pytest
import torch

from _common import gold, take_sample

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
GRID = (21, 30, 52)
TEXT_LEN = 512
RTOL, ATOL = 1e-3, 1e-4
REPORT = {}


def _bf16_ord(t):
    """Monotone integer image of bf16 values (sign-magnitude -> two's complement order), for ulp distances."""
    b = t.to(torch.bfloat16).view(torch.int16).to(torch.int32)
    return torch.where(b < 0, -(b & 0x7FFF), b)


def metrics(ours, ref, gold=None):
    """SURVEY §8c statistics of `ours` against `ref` (+ both against the fp32 golden)."""
    o, r = ours.float().cuda().reshape(-1), ref.float().cuda().reshape(-1)
    diff = (o - r).abs()
    m = {"pass_frac": float((diff <= ATOL + RTOL * r.abs()).float().mean()), "max_abs": float(diff.max()),
         "rel_fro": float(diff.norm() / r.norm())}
    if ours.dtype == torch.bfloat16 and ref.dtype == torch.bfloat16:
        u = (_bf16_ord(ours.cuda().reshape(-1)) - _bf16_ord(ref.cuda().reshape(-1))).abs()
        m["ulp"] = {"max": int(u.max()), "eq": float((u == 0).float().mean()), "le1": float((u <= 1).float().mean()),
                    "le2": float((u <= 2).float().mean()), "le4": float((u <= 4).float().mean())}
    if gold is not None:
        g = gold.float().cuda().reshape(-1)
        m["err_vs_fp32"] = float((o - g).norm() / g.norm())
        m["ref_err_vs_fp32"] = float((r - g).norm() / g.norm())
        m["err_ratio"] = m["err_vs_fp32"] / max(m["ref_err_vs_fp32"], 1e-30)
    return m


def check(name, ours, fa2, sdpa, gold, floor):
    """Record + assert the protocol for one tensor.  `floor`: stated lower bound on pass_frac for this tensor."""
    ours = ours.reshape(fa2.shape)
    m = metrics(ours, fa2, gold)
    yard = metrics(sdpa, fa2, gold) if sdpa is not None else None
    REPORT[name] = {"ours_vs_ref_fa2": m, "ref_sdpa_vs_ref_fa2": yard, "shape": list(fa2.shape), "dtype": str(fa2.dtype),
                    "pass_frac_floor": floor}
    print(f"[ref-parity] {name}: pass_frac {m['pass_frac']:.4f} (yardstick {yard['pass_frac'] if yard else float('nan'):.4f}) "
          f"ulp {m.get('ulp')} err/ref_err vs fp32 {m['err_vs_fp32']:.3e}/{m['ref_err_vs_fp32']:.3e} = {m['err_ratio']:.3f}")
    assert m["err_ratio"] <= 1.5, f"{name}: less accurate than the reference: {m}"
    assert m["pass_frac"] >= floor, f"{name}: pass fraction {m['pass_frac']:.4f} below the stated floor {floor}"
    if yard is not None and yard["pass_frac"] < 0.999:
        assert m["pass_frac"] >= 0.9 * yard["pass_frac"], f"{name}: farther from the reference than its own two backends are apart"
    return m


@pytest.fixture(scope="module", autouse=True)
def _write_report():
    yield
    out = ROOT / "gpurun_out"
    out.mkdir(exist_ok=True)
    (out / "r02_ref_parity.json").write_text(json.dumps(REPORT, indent=1))


@pytest.fixture(scope="module")
def ours_blocks():
    """This repo's path on the same weights / inputs: the three blocks through the reference-shaped modules."""
    import fwb200
    from fwb200.synth import build_fusion_model
    from fwb_synth import synth_block_inputs
    fwb200.require_device()
    f, h, w = GRID
    model = build_fusion_model(num_dit_layers=2, start_index=1, device="cuda", seed=0, heads=False)   # weights generated on the GPU
    inp = synth_block_inputs(f, h, w, TEXT_LEN)
    bf = torch.bfloat16
    d = {k: v.to("cuda", torch.float32 if k == "e0" else bf) for k, v in inp.items()}
    fr, fd, fa = model.rope_tables(f, h, w, "cuda")
    agg = model.vggt.aggregator
    pos = agg._positions(f, h, w, torch.device("cuda"))
    lens = torch.ones(f, dtype=torch.long, device="cuda")
    lens[1:] = 4
    P, C = d["x_agg"].shape[1:]
    out = {}
    with torch.no_grad():
        out["pcb"] = model.pipe.dit.blocks[0](d["x_dit"], d["context"], d["t_mod"], fr, plucker_fea=d["plucker"], plucker_context_lens=lens)
        out["frame"] = agg._process_frame_attention(d["x_agg"], 1, f, P, C, 0, pos=pos, e0=d["e0"])[0]
        xd, xa, _ = model.IRGBlock[0](x_dit=d["x_dit"], x_agg=d["x_agg"], context=d["context"], t_mod=d["t_mod"], freqs=fr, freqs_dit=fd,
                                      freqs_agg=fa, pos=pos, e0=d["e0"], uncond=False, plucker_fea=d["plucker"], plucker_context_lens=lens)
        out["irg_x"], out["irg_tokens"] = xd, xa
    torch.cuda.synchronize()
    out = {k: v.detach().cpu() for k, v in out.items()}
    del model
    torch.cuda.empty_cache()
    return out


# stated floors on the rtol=1e-3 / atol=1e-4 pass fraction (measured values are in profiles/r02_ref_parity.json; floors sit a few
# points below them).  bf16 outputs: an element passes only if it rounds to the SAME bf16 value as the reference's (1 ulp = 3.9e-3
# relative > rtol), so the fraction is the share of bit-equal elements; fp32 outputs (geometry stream) are compared at fp32 grain.
FLOORS = {"pcb": 0.55, "frame": 0.30, "irg_x": 0.45, "irg_tokens": 0.30}


@pytest.mark.parametrize("name", ["pcb", "frame", "irg_x", "irg_tokens"])
def test_block_at_c2_token_count_vs_reference_cuda_bf16(name, ours_blocks):
    g = gold(f"ref_parity_blocks_{name}.pt")
    rep = g["report"]
    REPORT["reference_run_blocks"] = rep
    assert tuple(rep["grid"]) == GRID
    assert rep["modes"]["bf16_fa2"]["dit_attention_backend"] == "flash_attn_func", rep     # what the reference takes on a B200
    assert rep["modes"]["bf16_sdpa"]["dit_attention_backend"] == "F.scaled_dot_product_attention"
    ours = ours_blocks[name]
    assert ours.numel() == torch.Size(g["shape"]).numel(), (ours.shape, g["shape"])
    assert ours.dtype == g["bf16_fa2"].dtype, (name, ours.dtype, g["bf16_fa2"].dtype)   # same stream dtypes as the reference (SURVEY Appendix A)
    check(f"block/{name}", take_sample(ours), g["bf16_fa2"], g["bf16_sdpa"], g["fp32"], FLOORS[name])


JOINT = dict(pcb=2, irg=2)
HEAD_LAYERS = [1, 1, 1, 0]      # = min(irg - 1, i) for the reference default [3, 2, 1, 0] pattern at reduced depth


def test_reduced_joint_forward_with_heads_at_c2_vs_reference_cuda_bf16():
    import fwb200
    from fwb200.synth import build_fusion_model
    from fwb_synth import synth_inputs
    ref, sdpa, gold32 = (gold(f"ref_parity_joint_{m}.pt") for m in ("bf16_fa2", "bf16_sdpa", "fp32"))
    REPORT["reference_run_joint"] = rep = ref["report"]
    assert tuple(rep["grid"]) == GRID and (rep["pcb"], rep["irg"], rep["heads"]) == (JOINT["pcb"], JOINT["irg"], True)
    f, h, w = GRID
    fwb200.require_device()
    model = build_fusion_model(num_dit_layers=JOINT["pcb"] + JOINT["irg"], start_index=JOINT["pcb"], device="cuda", seed=0, heads=True)
    model.vggt.depth_head.intermediate_layer_idx = HEAD_LAYERS
    model.vggt.point_head.intermediate_layer_idx = HEAD_LAYERS
    inp = synth_inputs(f, h, w, device="cuda", seed=1024, text_len=TEXT_LEN)
    lens = torch.ones(f, dtype=torch.long, device="cuda")
    lens[1:] = 4
    ts = torch.tensor([996.0], device="cuda", dtype=torch.bfloat16)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        out, pred = model.joint_forward(inp["latents"], timestep=ts, context=inp["context_pos"], clip_feature=inp["clip_feature"], y=inp["y"],
                                        use_gradient_checkpointing=False, plucker_fea=inp["plucker_fea"], plucker_context_lens=lens,
                                        return_prediction=True)
    torch.cuda.synchronize()
    assert list(out.shape) == ref["shape"]["out"] == [1, 16, f, 2 * h, 2 * w] and out.dtype == ref["out"].dtype
    # after 4 DiT blocks + head the bf16 roundings of two correct implementations have decorrelated: ~27 % bit-equal elements,
    # the same as between the reference's own flash-attn and SDPA runs (yardstick); the floor sits below both
    check("joint/latent_out", take_sample(out), ref["out"], sdpa["out"], gold32["out"], 0.20)
    assert set(pred) == set(ref["pred"]), (sorted(pred), sorted(ref["pred"]))
    for k in sorted(ref["pred"]):                       # depth, depth_conf, world_points, world_points_conf, pose_enc
        assert list(pred[k].shape) == ref["shape"][f"pred/{k}"], (k, pred[k].shape, ref["shape"][f"pred/{k}"])
        o, r, g = take_sample(pred[k]).float(), ref["pred"][k].float(), gold32["pred"][k].float()
        m = metrics(o, r, g)
        REPORT[f"joint/pred/{k}"] = m
        print(f"[ref-parity] joint/pred/{k}: {m}")
        assert torch.isfinite(pred[k]).all(), k
        assert m["err_ratio"] <= 1.5, (k, m)


DEEP = dict(pcb=4, irg=4, grid=(3, 8, 12))


def test_depth_drift_4pcb_4irg_vs_reference_cuda_bf16():
    """Error growth over depth: 4 PCB + 4 IRG blocks (8 DiT blocks, 4 frame + 4 global VGGT blocks, 4 adapters).  After 8 blocks the
    bf16 streams of two correct implementations have decorrelated roundings, so element-wise agreement is meaningless; what
    must hold is protocol (ii): our distance to the fp32 golden stays within 1.5x of the reference's own bf16 distance."""
    import fwb200
    from fwb200.synth import build_fusion_model
    from fwb_synth import synth_inputs
    g = gold("ref_parity_deep.pt")
    f, h, w = DEEP["grid"]
    REPORT["reference_run_deep"] = rep = g["report"]
    assert rep["grid"] == [f, h, w] and (rep["pcb"], rep["irg"]) == (DEEP["pcb"], DEEP["irg"])
    fwb200.require_device()
    model = build_fusion_model(num_dit_layers=DEEP["pcb"] + DEEP["irg"], start_index=DEEP["pcb"], device="cuda", seed=0, heads=False)
    inp = synth_inputs(f, h, w, device="cuda", seed=1024, text_len=64)
    lens = torch.ones(f, dtype=torch.long, device="cuda")
    lens[1:] = 4
    ts = torch.tensor([996.0], device="cuda", dtype=torch.bfloat16)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        out, _ = model.joint_forward(inp["latents"], timestep=ts, context=inp["context_pos"], clip_feature=inp["clip_feature"], y=inp["y"],
                                     use_gradient_checkpointing=False, plucker_fea=inp["plucker_fea"], plucker_context_lens=lens)
    m = metrics(out.cpu(), g["bf16_fa2"], g["fp32"])
    REPORT["deep/latent_out"] = m
    print(f"[ref-parity] deep 4+4: {m}")
    assert m["err_ratio"] <= 1.5, m
