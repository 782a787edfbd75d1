"""CPU tests of the host-side logic that needs no kernel: RoPE / position tables, scheduler, token layout, the temporal
up-sampler's whole-clip formulation, and the DPT head (pure torch) against the reference golden."""
import pytest
import torch

from _common import gold, rel_err, synth_state_dict
from oracle import fw_oracle as O


def test_scheduler_mirror():
    from FantasyWorld.diffsynth_wan21.schedulers.flow_match import FlowMatchScheduler
    g = gold("scheduler.pt")
    s = FlowMatchScheduler(shift=5, sigma_min=0.0, extra_one_step=True)
    s.set_timesteps(50)
    assert torch.equal(s.sigmas, g["sigmas"]) and torch.equal(s.timesteps, g["timesteps"])
    d = s.dsigma(s.timesteps[3])
    assert d == float(g["sigmas"][4] - g["sigmas"][3])
    assert s.dsigma(s.timesteps[49]) == float(0.0 - g["sigmas"][49])
    x = torch.randn(4, 4)
    v = torch.randn(4, 4)
    assert torch.equal(s.step(v, s.timesteps[7], x), x + v * (float(s.sigmas[8]) - float(s.sigmas[7])))


def test_rope_tables_match_oracle():
    from FantasyWorld.diffsynth_wan21.models.wan_video_dit import (_grid_freqs, build_freqs_3d_with_extra_cis,
                                                                   precompute_freqs_cis_3d, sinusoidal_embedding_1d)
    f, h, w = 3, 4, 5
    for hd in (128, 96):
        mine = _grid_freqs(precompute_freqs_cis_3d(hd), f, h, w).reshape(f * h * w, -1)
        assert torch.equal(mine, O.rope_table_3d(hd, f, h, w))
    extra = build_freqs_3d_with_extra_cis(precompute_freqs_cis_3d(96), f, h, w, n_extra=5).reshape(f * (5 + h * w), -1)
    assert torch.equal(extra, O.rope_table_3d_with_extra(96, f, h, w, 5))
    t = torch.tensor([996.0, 3.0])
    assert torch.equal(sinusoidal_embedding_1d(256, t), O.sinusoidal_embedding_1d(256, t).to(t.dtype))


def test_positions_and_token_assembly_bit_exact():
    from FantasyWorld.vggt.models.aggregator import Aggregator, slice_expand_and_flatten
    from FantasyWorld.vggt.layers.rope import PositionGetter
    sd = synth_state_dict()
    f, h, w = 3, 4, 6
    pg = PositionGetter()
    pos = pg(f, h, w, device=torch.device("cpu"))
    _, opos = O.aggregator_input(sd, "vggt.aggregator", torch.zeros(1, f, h, w, 1024))
    assert torch.equal(pos + 1, opos[:, 5:]) and pos.dtype == torch.int64
    tok = sd["vggt.aggregator.register_token"]
    out = slice_expand_and_flatten(tok, 1, f)
    assert torch.equal(out[0], tok[0, 0]) and torch.equal(out[1], tok[0, 1]) and torch.equal(out[2], tok[0, 1])


def test_rope2d_expanded_tables_follow_reference_arithmetic():
    import fwb200.engine as E
    pos = torch.tensor([[0, 0], [1, 1], [3, 7], [30, 52]])
    for fp32_angles, nm in ((False, O.BF16), (True, O.FP32)):   # autocast-faithful (default) and no-autocast arithmetic
        E.ROPE2D_FP32_ANGLES = fp32_angles
        try:
            with torch.autocast("cpu", dtype=torch.bfloat16):   # the result must not depend on ambient autocast
                cosT, sinT = E.rope2d_expanded(pos.clone())
        finally:
            E.ROPE2D_FP32_ANGLES = False
        ct, st = O.rope2d_tables(32, 53, nm=nm)
        assert torch.equal(cosT[:, :32], ct[pos[:, 0]]) and torch.equal(cosT[:, 32:], ct[pos[:, 1]])
        assert torch.equal(sinT[:, :32], st[pos[:, 0]]) and torch.equal(sinT[:, 32:], st[pos[:, 1]])


def test_unpatchify_and_patch_unfold_layout():
    from FantasyWorld.diffsynth_wan21.models.wan_video_dit import WanModel
    m = WanModel.__new__(WanModel)
    m.patch_size = (1, 2, 2)
    f, h, w = 2, 3, 4
    x = torch.arange(f * h * w * 64, dtype=torch.float32).view(1, f * h * w, 64)
    assert torch.equal(WanModel.unpatchify(m, x, (f, h, w)), O.unpatchify(x, (f, h, w)))
    # the im2col used by patchify reproduces Conv3d(k = s = (1,2,2))
    cin, dim = 5, 16
    conv = torch.nn.Conv3d(cin, dim, kernel_size=(1, 2, 2), stride=(1, 2, 2))
    v = torch.randn(1, cin, f, 2 * h, 2 * w)
    cols = v.view(1, cin, f, 1, h, 2, w, 2).permute(0, 2, 4, 6, 1, 3, 5, 7).reshape(f * h * w, cin * 4)
    ref = conv(v).permute(0, 2, 3, 4, 1).reshape(f * h * w, dim)
    assert torch.allclose(cols @ conv.weight.view(dim, -1).t() + conv.bias, ref, atol=1e-5)


def test_temporal_upsampler_whole_clip_equals_streaming():
    """WanVAE_(location='DPT').decode: our whole-clip causal evaluation vs a literal frame-by-frame streaming
    re-statement of the reference's cache protocol (vae_modified.py:81-125, 207-225, 454-476)."""
    from FantasyWorld.wan.modules.vae_modified import WanVAE_
    torch.manual_seed(0)
    C, T = 8, 5
    up = WanVAE_(z_dim=C, location="DPT")
    for p in up.parameters():
        torch.nn.init.normal_(p, std=0.3)
    z = torch.randn(1, C, T, 3, 4)
    ours = up.decode(z)
    assert ours.shape[2] == 4 * (T - 1) + 1

    def stream(up, z):
        x = up.conv2(z)
        layers = list(up.decoder.upsamples)
        cache = [None] * 4
        outs = []
        for i in range(x.shape[2]):
            cur = x[:, :, i:i + 1]
            for li, layer in enumerate(layers):
                if li % 2 == 0:  # Resample
                    b, c, t, hh, ww = cur.shape
                    if cache[li] is None:
                        cache[li] = "Rep"
                    else:
                        cx = cur[:, :, -2:].clone()
                        if cx.shape[2] < 2:
                            prev = torch.zeros_like(cx) if isinstance(cache[li], str) else cache[li][:, :, -1:]
                            cx = torch.cat([prev, cx], dim=2)
                        y = layer.time_conv(cur) if isinstance(cache[li], str) else layer.time_conv(cur, cache[li])
                        cache[li] = cx
                        y = y.reshape(b, 2, c, t, hh, ww)
                        cur = torch.stack((y[:, 0], y[:, 1]), 3).reshape(b, c, t * 2, hh, ww)
                else:  # ResidualBlock_Half
                    hres = cur
                    y = layer.residual[1](layer.residual[0](cur))
                    cx = y[:, :, -2:].clone()
                    if cx.shape[2] < 2 and cache[li] is not None:
                        cx = torch.cat([cache[li][:, :, -1:], cx], dim=2)
                    y = layer.residual[2](y, cache[li])
                    cache[li] = cx
                    cur = y + hres
            outs.append(cur)
        return torch.cat(outs, dim=2)

    ref = stream(up, z)
    assert ours.shape == ref.shape and torch.allclose(ours, ref, atol=1e-5)


def test_dpt_head_matches_reference_golden():
    """The DPT head mirror is pure torch: run it on CPU fp32 on the reference's own intermediates-equivalent produced by
    the oracle and compare with the reference's depth / point outputs (index chunking 4 / 16, temporal 4x, activations)."""
    import torch.nn as nn
    from FantasyWorld.vggt.heads.dpt_head import DPTHead_3D_Causal
    from fwb_synth import synth_inputs
    g = gold("joint_forward.pt")
    sd = synth_state_dict()
    f, h, w = g["grid"]
    inp = synth_inputs(f, h, w, device="cpu", seed=1024, text_len=g["text_len"], dtype=torch.float32)
    _, inter, patch = O.joint_forward(sd, inp["latents"], torch.tensor([g["timestep"]]), inp["context_pos"], inp["clip_feature"],
                                      inp["y"], inp["plucker_fea"], start_index=1, n_irg=1, collect_intermediates=True)
    for name, odim, act in (("depth_head", 2, "exp"), ("point_head", 4, "inv_log")):
        head = DPTHead_3D_Causal(dim_in=2048, output_dim=odim, activation=act, conf_activation="expp1", patch_size=16,
                                 intermediate_layer_idx=g["head_layer_idx"])
        head.load_state_dict({k[len("vggt." + name) + 1:]: v for k, v in sd.items() if k.startswith("vggt." + name + ".")}, strict=True)
        with torch.no_grad():
            pred, conf = head(inter, images=patch, patch_start_idx=5)
        key = "depth" if name == "depth_head" else "world_points"
        assert pred.shape == g["pred"][key].shape and conf.shape == g["pred"][key + "_conf"].shape
        assert rel_err(pred, g["pred"][key]) < 1e-3, (name, rel_err(pred, g["pred"][key]))
        assert rel_err(conf, g["pred"][key + "_conf"]) < 1e-3


def test_bench_reference_arm_prints_one_json_line():
    """bench.py --impl reference (the CPU arm the driver runs beside ours): exactly one JSON line on stdout with the contract's
    keys, whatever libraries print (stdout is re-pointed at stderr inside bench.py)."""
    import json
    import subprocess
    import sys
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    r = subprocess.run([sys.executable, str(root / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-budget", "5",
                        "--no-cpu-full"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "cpu_baseline", "impl"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "denoise_steps_per_sec" and d["unit"] == "steps/s"
    staged = (root / "oracle" / "_ref" / "FantasyWorld").exists()
    # the unmodified reference when it is staged (oracle/make_ref.py), the oracle port only as the fallback
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == ("reference" if staged else "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["ms_per_step"] == pytest.approx(1e3 * d["cpu_baseline"]["sample_seconds"])      # the measured sample, not the extrapolation
    assert d["config"]["same_config"] is False
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_bench_roofline_aggregation():
    """bench.roofline_from_prof: the dominant-kernel figure from the CUDA-event records, single GPU and sequence parallel with
    ragged K|V slices; cross-attention launches (same q, 512 / 257 keys) must not be counted."""
    import sys
    from pathlib import Path
    sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
    import bench
    L = 32760
    prof = {"attn:B1:H40:Lq32760:Lk32760:D128": (240, 240 * 20.0), "attn:B1:H40:Lq32760:Lk512:D128": (240, 160.0),
            "attn:B1:H12:Lq32760:Lk32865:D96": (144, 700.0)}
    r = bench.roofline_from_prof(prof, L, 1, 12600.0, 1421.6, "measured")
    assert r["launches_timed"] == 240 and abs(r["ms_per_launch"] - 20.0) < 1e-9
    assert abs(r["achieved"] - 4 * 40 * L * L * 128 / 20e-3 / 1e12) < 1e-6 and abs(r["frac"] - r["achieved"] / 1421.6) < 1e-12
    assert abs(r["share_of_step"] - 4800.0 / 12600.0) < 1e-12
    prof8 = {"attn:B1:H40:Lq4095:Lk8192:D128": (720, 720 * 0.6), "attn:B1:H40:Lq4095:Lk8184:D128": (240, 240 * 0.6),
             "attn:B1:H40:Lq4095:Lk257:D128": (240, 10.0)}
    r8 = bench.roofline_from_prof(prof8, L, 8, 2200.0, 1421.6, "measured")
    assert r8["launches_timed"] == 960 and r8["traffic"] is None
    fl = (720 * 8192 + 240 * 8184) * 4.0 * 40 * 4095 * 128
    assert abs(r8["achieved"] - fl / (960 * 0.6e-3) / 1e12) < 1e-6
    assert bench.roofline_from_prof({}, L, 8, 1.0, 1421.6, "x") is None


def _compare_head_records(rec, gold_rec, only_prefix=None):
    gold_rec = [r for r in gold_rec if only_prefix is None or r[0].startswith(only_prefix)]
    assert [(n, tuple(s)) for n, s, _ in rec] == [(n, tuple(s)) for n, s, _ in gold_rec]
    for (n, _, v), (_, _, gv) in zip(rec, gold_rec):
        assert (v is None) == (gv is None), n
        if v is not None:
            assert torch.equal(v, gv), n          # the SAME tokens, in the same order, reach this stage


def test_dpt_head_index_selection_and_chunking_match_reference():
    """SURVEY §8 a19: layer selection [23,17,11,7], the [:, f0:f1, 5:] slices of the 4-latent-frame chunks and the 16-video-frame
    chunks of the fusion stage, recorded by hooks on integer-coded tokens, are identical to the reference's (golden written by
    tools/make_golden_head_index.py from the unmodified reference)."""
    from _head_index import record_head_indexing
    from FantasyWorld.vggt.heads.dpt_head import DPTHead_3D_Causal
    from fwb_synth import synth_init
    g = gold("head_index.pt")
    wrap = torch.nn.Module()
    wrap.vggt = torch.nn.Module()
    wrap.vggt.depth_head = DPTHead_3D_Causal(dim_in=2048, output_dim=2, activation="exp", conf_activation="expp1", patch_size=16)
    synth_init(wrap, seed=0, gen_device="cpu")
    rec = record_head_indexing(wrap.vggt.depth_head.eval())
    _compare_head_records(rec, g["records"], only_prefix="dpt.")


def test_lora_merge_and_expert_switch_match_reference(tmp_path):
    """SURVEY §8f N4: `load_lora` (reference: fusion/model_wan22.py:18-118) merges kohya- and PEFT-style LoRA files into the DiT
    weights bit-identically to the unmodified reference, and the high-/low-noise expert choice over the 50-step schedule
    (inference_wan22.py:229-240) is the reference's.  Golden: tools/make_golden_lora.py."""
    import types
    from safetensors.torch import save_file
    from FantasyWorld.diffsynth_wan22.models.wan_video_dit import WanModel
    from FantasyWorld.diffsynth_wan22.schedulers.flow_match import FlowMatchScheduler
    from FantasyWorld.fusion.model_wan22 import load_lora, select_high_noise_expert
    from fwb_synth import synth_init
    g = gold("lora_merge.pt")
    for style, sd in g["loras"].items():
        model = WanModel(**g["cfg"])
        wrap = torch.nn.Module()
        wrap.dit = model
        synth_init(wrap, seed=0, gen_device="cpu")
        model.to(torch.bfloat16)
        before = {k: v.clone() for k, v in model.state_dict().items()}
        f = tmp_path / f"{style}.safetensors"
        save_file({k: v.contiguous() for k, v in sd.items()}, str(f))
        load_lora(types.SimpleNamespace(device="cpu", torch_dtype=torch.bfloat16, dit=model), str(f), 0.55, "dit")
        after = model.state_dict()
        changed = 0
        for k, ref in g["merged"][style].items():
            assert torch.equal(after[k], ref), (style, k)
            changed += int(not torch.equal(after[k], before[k]))
        assert changed == (0 if style == "peft_default" else 3), (style, changed)   # the three named layers; `.default` keys: skipped, as the reference
    sched = FlowMatchScheduler(shift=5, sigma_min=0.0, extra_one_step=True)
    sched.set_timesteps(50)
    assert [select_high_noise_expert(t) for t in sched.timesteps] == g["high_noise_steps"]
    assert 0 < sum(g["high_noise_steps"]) < 50
