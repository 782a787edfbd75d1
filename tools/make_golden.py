"""Generate the golden vectors under tests/golden/ by running the UNMODIFIED reference (/root/reference, imported through
tools/ref_shim.py) on CPU in fp32.  Run in the build container only (the GPU box has no /root/reference):

    python tools/make_golden.py

Weights and inputs are NOT stored (a single 5120-wide block is 1.7 GB): both come from per-key / seeded generators in
fantasy-world_b200/fwb200/synth.py, so the tests regenerate exactly the tensors the reference saw here.  Stored: the
state_dict schema (key -> shape) and the reference's outputs (small).

Cases (SURVEY §8c/§8d):
  irg_block_c1   BASELINE config 1 — one IRG block forward at f,h,w = 1,4,4 (L = 16 video tokens, N = 21 geometry tokens)
  joint_forward  reduced depth (1 PCB + 1 IRG, 14B widths), f,h,w = 2,4,4, with geometry heads (81-frame analogue: 5 frames)
  denoise_step   one CFG Euler step (2 forwards + scheduler) at the same size
  scheduler      FlowMatchScheduler(shift=5, sigma_min=0, extra_one_step) sigmas / timesteps for 50 steps
"""
from __future__ import annotations

import json
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tools"))
sys.path.insert(0, str(ROOT / "fantasy-world_b200"))
GOLD = ROOT / "tests" / "golden"

F, H, W = 2, 4, 4            # token grid of the reduced joint_forward
TEXT_LEN = 64                # the text-context length is free; 64 keeps the fixture run short
TIMESTEP = 996.0             # bf16-representable (the reference casts the timestep to bf16, model_wan21.py:292-293)
HEAD_LAYER_IDX = [0, 0, 0, 0]  # reduced depth has a single intermediate; DPT default [23,17,11,7] needs 24


def main():
    from ref_shim import build_reference_fusion
    from fwb_synth import synth_init, synth_inputs  # per-key seeded init shared with the tests

    torch.manual_seed(0)
    torch.set_grad_enabled(False)
    t0 = time.time()
    model, ns = build_reference_fusion(num_dit_layers=2, start_index=1, heads=True)
    synth_init(model, seed=0, gen_device="cpu")
    model.vggt.depth_head.intermediate_layer_idx = HEAD_LAYER_IDX
    model.vggt.point_head.intermediate_layer_idx = HEAD_LAYER_IDX
    print(f"reference built + synthetic weights in {time.time() - t0:.0f}s")
    GOLD.mkdir(parents=True, exist_ok=True)
    schema = {k: list(v.shape) for k, v in model.state_dict().items()}
    (GOLD / "schema_reduced.json").write_text(json.dumps(schema, indent=0))

    # ---------------- scheduler ----------------
    sched = ns.sched.FlowMatchScheduler(shift=5, sigma_min=0.0, extra_one_step=True)
    sched.set_timesteps(50)
    torch.save({"sigmas": sched.sigmas.clone(), "timesteps": sched.timesteps.clone()}, GOLD / "scheduler.pt")

    # ---------------- irg_block_c1 ----------------
    g = torch.Generator().manual_seed(1024)
    f, h, w = 1, 4, 4
    L, N = f * h * w, f * (5 + h * w)
    x_dit = torch.randn(1, L, 5120, generator=g)
    x_agg = torch.randn(f, 5 + h * w, 1024, generator=g)
    context = torch.randn(1, 257 + TEXT_LEN, 5120, generator=g)
    t_mod = torch.randn(1, 6, 5120, generator=g) * 0.1
    e0 = torch.randn(1, 6, 1024, generator=g) * 0.1
    plucker = torch.randn(1, L, 2048, generator=g)
    dit = ns.dit
    freqs3 = dit.precompute_freqs_cis_3d(128)
    freqs = torch.cat([freqs3[0][:f].view(f, 1, 1, -1).expand(f, h, w, -1), freqs3[1][:h].view(1, h, 1, -1).expand(f, h, w, -1),
                       freqs3[2][:w].view(1, 1, w, -1).expand(f, h, w, -1)], dim=-1).reshape(L, 1, -1)
    fb = model.freqs_bicross
    freqs_bi_dit = torch.cat([fb[0][:f].view(f, 1, 1, -1).expand(f, h, w, -1), fb[1][:h].view(1, h, 1, -1).expand(f, h, w, -1),
                              fb[2][:w].view(1, 1, w, -1).expand(f, h, w, -1)], dim=-1).reshape(L, 1, -1)
    freqs_bi_agg = dit.build_freqs_3d_with_extra_cis(fb, f, h, w, n_extra=5)
    pos = model.vggt.aggregator.position_getter(f, h, w, device="cpu") + 1
    pos = torch.cat([torch.zeros(f, 5, 2, dtype=pos.dtype), pos], dim=1)
    lens = torch.ones(1, dtype=torch.long)
    xd, xa, inter = model.IRGBlock[0](x_dit=x_dit, x_agg=x_agg, context=context, t_mod=t_mod, freqs=freqs,
                                      freqs_dit=freqs_bi_dit, freqs_agg=freqs_bi_agg, pos=pos, e0=e0, uncond=False,
                                      plucker_fea=plucker, plucker_context_lens=lens)
    torch.save({"x_dit_out": xd.clone(), "x_agg_out": xa.clone(), "seed": 1024, "text_len": TEXT_LEN}, GOLD / "irg_block_c1.pt")
    print("irg_block_c1 done", xd.abs().mean().item(), xa.abs().mean().item())

    # ---------------- joint_forward (with intermediates and heads) ----------------
    inp = synth_inputs(F, H, W, device="cpu", seed=1024, text_len=TEXT_LEN, dtype=torch.float32)
    ts = torch.tensor([TIMESTEP])
    lens = torch.ones(F, dtype=torch.long)
    lens[1:] = 4
    taps = {}
    hooks = [model.pipe.dit.blocks[0].register_forward_hook(lambda m, i, o: taps.__setitem__("after_pcb", o.clone())),
             model.vggt.aggregator.frame_blocks[0].register_forward_hook(lambda m, i, o: taps.__setitem__("after_frame", o.clone())),
             model.IRGBlock[0].register_forward_hook(lambda m, i, o: taps.update(after_irg_x=o[0].clone(), after_irg_tokens=o[1].clone()))]
    out, pred = model.joint_forward(inp["latents"], timestep=ts, context=inp["context_pos"], clip_feature=inp["clip_feature"],
                                    y=inp["y"], use_gradient_checkpointing=False, plucker_fea=inp["plucker_fea"],
                                    plucker_context_lens=lens, return_prediction=True)
    for hk in hooks:
        hk.remove()
    parts = {"after_pcb": "joint_forward_after_pcb.pt", "after_irg_x": "joint_forward_after_irg_x.pt"}     # each file under 1 MB
    for k, name in parts.items():
        torch.save({k: taps.pop(k)}, GOLD / name)
    torch.save({"out": out.clone(), "pred": {k: v.clone() for k, v in pred.items()}, "taps": taps, "parts": list(parts.values()),
                "grid": (F, H, W), "text_len": TEXT_LEN, "timestep": TIMESTEP, "head_layer_idx": HEAD_LAYER_IDX}, GOLD / "joint_forward.pt")
    print("joint_forward done", out.abs().mean().item(), {k: tuple(v.shape) for k, v in pred.items()})

    # ---------------- one denoise step (CFG 5.0) ----------------
    model.pipe.scheduler.set_timesteps(50)
    step = 3
    t = model.pipe.scheduler.timesteps[step].to(torch.bfloat16).float().unsqueeze(0)
    lat = inp["latents"]
    p, _ = model.joint_forward(lat, timestep=t, context=inp["context_pos"], clip_feature=inp["clip_feature"], y=inp["y"],
                               use_gradient_checkpointing=False, plucker_fea=inp["plucker_fea"], plucker_context_lens=lens)
    n, _ = model.joint_forward(lat, timestep=t, context=inp["context_neg"], clip_feature=inp["clip_feature"], y=inp["y"],
                               use_gradient_checkpointing=False, plucker_fea=inp["plucker_fea"], plucker_context_lens=lens)
    pred_v = n + 5.0 * (p - n)
    new_lat = model.pipe.scheduler.step(pred_v, model.pipe.scheduler.timesteps[step], lat)
    torch.save({"latents_next": new_lat.clone(), "pred_pos": p.clone(), "pred_neg": n.clone(), "step": step,
                "timestep": float(t)}, GOLD / "denoise_step.pt")
    print("denoise_step done", new_lat.abs().mean().item(), f"total {time.time() - t0:.0f}s")


if __name__ == "__main__":
    main()
