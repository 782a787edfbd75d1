"""Batch > 1 on the B200: the periodic RoPE entry points, joint_forward at batch 2 against per-sample batch-1 calls and against the
unmodified reference's batch-2 golden (tools/make_golden_batch.py), the whole-batch all-zero camera rule, and the sampler with
batched latents and batched CFG (`batch_cfg`).

Exactness: GEMM rows and the row kernels are row-independent and every attention tile is computed the same way at any batch, so
with the key-split tail of the attention schedule off (it merges partials of whichever tiles land in the last wave, and that
set depends on the batch) a batch-2 call is bit-identical to its batch-1 calls."""
import ctypes as C
from contextlib import contextmanager

import pytest
import torch

from _common import gold, rel_err, take_sample

pytestmark = pytest.mark.gpu

BF = torch.bfloat16
HEADS = ("pose_enc", "depth", "depth_conf", "world_points", "world_points_conf")


@contextmanager
def tail_split_off():
    import fwb200
    fwb200.lib.fwb_attn_set_tail_split(0)
    try:
        yield
    finally:
        fwb200.lib.fwb_attn_set_tail_split(1)


def _lens(f):
    lens = torch.ones(f, dtype=torch.long, device="cuda")
    lens[1:] = 4
    return lens


def _inputs(f, h, w, seeds, text_len):
    from fwb_synth import synth_inputs
    per = [synth_inputs(f, h, w, device="cuda", seed=s, text_len=text_len) for s in seeds]
    return per, {k: torch.cat([p[k] for p in per]) for k in per[0]}


def _joint(model, d, ts, heads=True):
    with torch.no_grad(), torch.autocast("cuda", dtype=BF):
        return model.joint_forward(d["latents"], timestep=ts, context=d["context_pos"], clip_feature=d["clip_feature"], y=d["y"],
                                   use_gradient_checkpointing=False, plucker_fea=d["plucker_fea"],
                                   plucker_context_lens=_lens(d["latents"].shape[2]), return_prediction=heads)


# ---------------------------------------------------------------------------------------------------------------------------
# kernels
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [2, 3])
def test_periodic_rmsnorm_rope_equals_repeated_table(B):
    import fwb200
    from fwb200 import ops
    torch.manual_seed(B)
    L, C_, D = 288, 5120, 128
    x = torch.randn(B * L, C_, device="cuda").to(BF)
    wt = torch.rand(C_, device="cuda") + 0.5
    cs = torch.randn(L, D // 2, 2, device="cuda")
    rep = cs.repeat(B, 1, 1).contiguous()
    ref = x.clone()
    s = torch.cuda.current_stream().cuda_stream
    assert fwb200.lib.fwb_rmsnorm_rope(ref.data_ptr(), ref.stride(0), B * L, C_, wt.data_ptr(), C.c_float(1e-6), rep.data_ptr(), D, s) == 0
    out = ops.rmsnorm_rope_(x.clone(), w=wt, eps=1e-6, cos_sin=cs, head_dim=D)
    assert torch.equal(out, ref)
    # rope only on a strided [q | v] view (the adapter's buffer), head_dim 96
    buf = torch.randn(B * L, 2304, device="cuda").to(BF)
    cs96 = torch.randn(L, 48, 2, device="cuda")
    ref = buf.clone()
    assert fwb200.lib.fwb_rmsnorm_rope(ref.data_ptr(), ref.stride(0), B * L, 1152, None, C.c_float(1e-6),
                                       cs96.repeat(B, 1, 1).contiguous().data_ptr(), 96, s) == 0
    out = buf.clone()
    ops.rmsnorm_rope_(out[:, :1152], cos_sin=cs96, head_dim=96)
    torch.cuda.synchronize()
    assert torch.equal(out, ref)
    with pytest.raises(ValueError, match="does not divide"):
        ops.rmsnorm_rope_(x[:L + 1], cos_sin=cs, head_dim=D)


@pytest.mark.parametrize("B", [2, 4])
def test_periodic_ln64_rope2d_equals_repeated_table(B):
    import fwb200
    from fwb200 import ops
    torch.manual_seed(10 + B)
    rows1, H = 3 * (5 + 8 * 12), 16
    qkv = torch.randn(B * rows1, 3 * H * 64, device="cuda").to(BF)
    qw, qb, kw, kb = (torch.randn(64, device="cuda") for _ in range(4))
    cosT, sinT = torch.randn(rows1, 64, device="cuda"), torch.randn(rows1, 64, device="cuda")
    ref = qkv.clone()
    s = torch.cuda.current_stream().cuda_stream
    assert fwb200.lib.fwb_ln64_rope2d(ref.data_ptr(), ref.stride(0), B * rows1, H, C.c_float(1e-5), qw.data_ptr(), qb.data_ptr(),
                                      kw.data_ptr(), kb.data_ptr(), cosT.repeat(B, 1).contiguous().data_ptr(),
                                      sinT.repeat(B, 1).contiguous().data_ptr(), s) == 0
    out = ops.ln64_rope2d_(qkv.clone(), H, eps=1e-5, qw=qw, qb=qb, kw=kw, kb=kb, cosT=cosT, sinT=sinT)
    torch.cuda.synchronize()
    assert torch.equal(out, ref)


# ---------------------------------------------------------------------------------------------------------------------------
# joint_forward at batch 2 against per-sample batch-1 calls
# ---------------------------------------------------------------------------------------------------------------------------
def test_joint_forward_batch2_equals_two_batch1_calls():
    """2 PCB + 2 IRG blocks with the heads; two samples with their own latents, y, context, CLIP and camera features, one timestep."""
    import fwb200
    from fwb200.synth import build_fusion_model
    fwb200.require_device()
    f, h, w = 3, 8, 12
    model = build_fusion_model(num_dit_layers=4, start_index=2, device="cuda", seed=0, heads=True)
    for head in (model.vggt.depth_head, model.vggt.point_head):
        head.intermediate_layer_idx = [1, 1, 1, 0]
    per, both = _inputs(f, h, w, (1024, 1025), 64)
    ts = torch.tensor([996.0], device="cuda", dtype=BF)
    with tail_split_off():
        singles = [_joint(model, p, ts) for p in per]
        out, pred = _joint(model, both, ts)
    torch.cuda.synchronize()
    assert out.shape == (2, 16, f, 2 * h, 2 * w) and set(pred) == set(HEADS)
    for i, (o1, p1) in enumerate(singles):
        assert torch.equal(out[i:i + 1], o1), i
        for k in HEADS:
            assert pred[k].shape[0] == 2 and pred[k][i:i + 1].shape == p1[k].shape, k
            assert torch.isfinite(pred[k]).all(), k
            assert rel_err(pred[k][i:i + 1], p1[k]) <= 1e-3, (i, k, rel_err(pred[k][i:i + 1], p1[k]))
    # default schedule (tail split on): partials merged in a different order
    out_d, pred_d = _joint(model, both, ts)
    ts2 = torch.tensor([996.0, 996.0], device="cuda", dtype=BF)       # the same timestep given per sample
    out_t2, _ = _joint(model, both, ts2, heads=False)
    for i, (o1, p1) in enumerate(singles):
        assert rel_err(out_d[i:i + 1], o1) <= 1e-3
        for k in HEADS:
            assert rel_err(pred_d[k][i:i + 1], p1[k]) <= 1e-3, k
    assert torch.equal(out_t2, out_d)
    with pytest.raises(ValueError, match="share the timestep"):
        _joint(model, both, torch.tensor([900.0, 500.0], device="cuda", dtype=BF), heads=False)
    with pytest.raises(ValueError, match="context has batch 1"):     # no broadcasting of one sample's context over the batch
        _joint(model, {**both, "context_pos": per[0]["context_pos"], "clip_feature": per[0]["clip_feature"]}, ts, heads=False)


# ---------------------------------------------------------------------------------------------------------------------------
# against the unmodified reference (fp32 CPU golden) at batch 2
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def golden_model():
    import fwb200
    from fwb200.synth import build_fusion_model
    fwb200.require_device()
    g = gold("batch_joint.pt")
    cfg = g["config"]
    # the golden's weights were generated on the CPU: same generator here
    model = build_fusion_model(num_dit_layers=cfg["pcb"] + cfg["irg"], start_index=cfg["pcb"], device="cuda", seed=0, heads=True,
                               gen_device="cpu")
    for head in (model.vggt.depth_head, model.vggt.point_head):
        head.intermediate_layer_idx = list(cfg["head_layers"])
    per, both = _inputs(*cfg["grid"], cfg["seeds"], cfg["text_len"])
    yield g, model, per, both
    del model
    torch.cuda.empty_cache()


def _errs(res, i, gsample):
    """rel. L2 error vs the golden, per output (same sampled elements as the golden)."""
    out, pred = res
    n = gold("batch_joint.pt")["config"]["n_sample"]
    e = {"out": rel_err(take_sample(out[i], n), gsample["out"])}
    e.update({k: rel_err(take_sample(pred[k][i], n), gsample["pred"][k]) for k in HEADS})
    return e


def test_joint_forward_batch2_vs_reference_golden(golden_model):
    """err-vs-fp32 protocol of test_gpu_ref_parity: for each sample and output, the batch-2 error against the reference's fp32
    golden is at most 1.5x the batch-1 error against the same golden."""
    g, model, per, both = golden_model
    ts = torch.tensor([g["config"]["timestep"]], device="cuda", dtype=BF)
    res2 = _joint(model, both, ts)
    for i in range(2):
        e1 = _errs(_joint(model, per[i], ts), 0, g["single"][i])
        e2 = _errs(res2, i, g["single"][i])
        e2b = _errs(res2, i, g["batch"][i])
        print(f"[batch-golden] sample {i}: batch-1 err {e1}, batch-2 err {e2}")
        assert e1["out"] < 0.1, (i, e1)
        for k in e1:
            assert e2[k] <= 1.5 * e1[k] + 1e-7, (i, k, e1[k], e2[k])
            assert e2b[k] <= 1.5 * e1[k] + 1e-5, (i, k, e1[k], e2b[k])


def test_all_zero_camera_sample_in_a_batch_keeps_the_shift(golden_model):
    """The all-zero test covers the whole plucker tensor (reference camera_control.py:111): sample 1 with all-zero features inside
    a batch whose other sample has features gets the camera shift, as in the reference's batch run, not the skip of a batch-1 call."""
    g, model, per, both = golden_model
    ts = torch.tensor([g["config"]["timestep"]], device="cuda", dtype=BF)
    zc = dict(both, plucker_fea=both["plucker_fea"].clone())
    zc["plucker_fea"][1] = 0
    res = _joint(model, zc, ts)
    alone = _joint(model, dict(per[1], plucker_fea=torch.zeros_like(per[1]["plucker_fea"])), ts)
    base = _errs(_joint(model, per[1], ts), 0, g["single"][1])["out"]
    e_batch = _errs(res, 1, g["zero_cam"][1])["out"]
    e_skip = _errs(res, 1, g["zero_cam_single1"][0])["out"]
    e_alone = _errs(alone, 0, g["zero_cam_single1"][0])["out"]
    print(f"[batch-golden] zero camera: vs reference batch {e_batch:.3e}, vs reference skip {e_skip:.3e}, alone {e_alone:.3e}")
    assert e_batch <= 1.5 * base + 1e-7
    assert e_alone <= 1.5 * base + 1e-7
    assert e_skip > 5 * e_batch          # the reference's shift-vs-skip distance is 0.28 (rel. L2) on this output
    assert _errs(res, 0, g["zero_cam"][0])["out"] <= 1.5 * _errs(_joint(model, per[0], ts), 0, g["single"][0])["out"] + 1e-7


# ---------------------------------------------------------------------------------------------------------------------------
# sampler
# ---------------------------------------------------------------------------------------------------------------------------
def _sampler_model(pcb=1, irg=1):
    import fwb200
    from fwb200.synth import build_fusion_model
    fwb200.require_device()
    return build_fusion_model(num_dit_layers=pcb + irg, start_index=pcb, device="cuda", seed=0, heads=False)


def _step(model, lat, d, step, **kw):
    return model.denoise_step(lat.clone(), step, d["context_pos"], d["context_neg"], clip_feature=d["clip_feature"], y=d["y"],
                              plucker_fea=d["plucker_fea"], plucker_context_lens=_lens(lat.shape[2]), cfg_scale=5.0, **kw)[0]


def test_denoise_step_batch_cfg_and_batched_generate_video():
    f, h, w = 3, 8, 12
    model = _sampler_model()
    model.pipe.scheduler.set_timesteps(50)
    per, both = _inputs(f, h, w, (1024, 1025), 16)
    with tail_split_off():
        serial = _step(model, per[0]["latents"], per[0], 3)
        batched = _step(model, per[0]["latents"], per[0], 3, batch_cfg=True)
        assert torch.equal(batched, serial)
        b2 = _step(model, both["latents"], both, 3)
        b2_cfg = _step(model, both["latents"], both, 3, batch_cfg=True)
        assert torch.equal(b2[:1], serial) and torch.equal(b2_cfg, b2)
        # 2 steps of the whole sampler (pose encoder on the camera rays included) on batch-2 latents vs per-sample calls
        g = torch.Generator().manual_seed(7)
        rays = torch.randn(2, 4 * (f - 1) + 1, 16 * h, 16 * w, 6, generator=g).to("cuda", BF)
        kw = dict(height=16 * h, width=16 * w, num_frames=4 * (f - 1) + 1, num_inference_steps=2, cfg_scale=5.0, device="cuda")

        def gen(d, r, **extra):
            return model.generate_video(context_pos=d["context_pos"], context_neg=d["context_neg"], clip_feature=d["clip_feature"],
                                        y=d["y"], plucker_embedding=r, latents=d["latents"], **kw, **extra)[0]
        one = [gen(per[i], rays[i:i + 1]) for i in range(2)]
        two = gen(both, rays)
        two_cfg = gen(both, rays, batch_cfg=True)
    for i in range(2):
        assert torch.equal(two[i:i + 1], one[i]), i
    assert torch.equal(two_cfg, two)
    with pytest.raises(ValueError, match="latents have batch 2"):
        _step(model, both["latents"], dict(both, context_neg=per[0]["context_neg"]), 0)


def test_batch_cfg_at_c2_token_count():
    """One batch_cfg step at the BASELINE C2 token count (f,h,w = 21,30,52: L = 32760) at 1 PCB + 1 IRG block: a forward of batch 2
    over 65520 video and 65730 geometry token rows, equal to the serial step; peak memory printed."""
    f, h, w = 21, 30, 52
    model = _sampler_model()
    model.pipe.scheduler.set_timesteps(50)
    per, _ = _inputs(f, h, w, (1024,), 512)
    d = per[0]
    with tail_split_off():
        serial = _step(model, d["latents"], d, 0)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        batched = _step(model, d["latents"], d, 0, batch_cfg=True)
        torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() / 2 ** 30
    print(f"[batch] C2 batch_cfg step at 1+1 blocks: peak {peak:.2f} GiB on {torch.cuda.get_device_name(0)}")
    assert torch.equal(batched, serial)
    assert torch.isfinite(batched.float()).all()
