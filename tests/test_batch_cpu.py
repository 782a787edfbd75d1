"""Batch > 1 without a device: what the unmodified reference does with a batch (golden from tools/make_golden_batch.py), the
attention tile schedule at batch 2 and 4, and the batch / timestep validation that runs before any launch."""
import ctypes as C

import pytest
import torch

from _common import gold

BATCH_TOL = 5e-5          # the reference's own batch-2 vs batch-1 distance measured at most 8e-6


def _max_abs(a, b):
    return max([float((a["out"] - b["out"]).abs().max())] + [float((a["pred"][k] - b["pred"][k]).abs().max()) for k in a["pred"]])


@pytest.fixture(scope="module")
def g():
    return gold("batch_joint.pt")


def test_reference_batch_equals_its_batch_1_runs(g):
    """The reference at batch 2 with a shared timestep: every sample's latent output and all five head outputs equal the
    sample's own batch-1 run (fp32 on the CPU), so batch is a pure per-sample map there."""
    assert g["config"]["grid"] == [2, 2, 3] and g["config"]["heads"]
    assert set(g["single"][0]["pred"]) == {"pose_enc", "depth", "depth_conf", "world_points", "world_points_conf"}
    for i in range(2):
        assert _max_abs(g["batch"][i], g["single"][i]) <= BATCH_TOL, i
    # the two samples really are different inputs
    assert float((g["single"][0]["out"] - g["single"][1]["out"]).abs().max()) > 0.1


def test_reference_all_zero_camera_test_covers_the_whole_batch(g):
    """camera_control.py:111 tests the WHOLE plucker tensor for all-zero: a batch in which one sample's features are all zero still
    applies the camera shift to that sample (unlike the same sample alone, where the shift is skipped)."""
    assert _max_abs(g["zero_cam"][0], g["single"][0]) <= BATCH_TOL
    shifted, skipped = g["zero_cam"][1], g["zero_cam_single1"][0]
    assert float((shifted["out"] - skipped["out"]).abs().max()) > 1e-2


def test_reference_has_no_per_sample_timestep(g):
    """With distinct timesteps the reference's batch outputs are NOT the per-sample batch-1 runs at those timesteps, which is why
    a batch here must share its timestep."""
    assert g["config"]["distinct_timesteps"] == [900.0, 500.0]
    assert max(_max_abs(g["distinct_t"][i], g["single_t"][i]) for i in range(2)) > 0.1


@pytest.mark.parametrize("B", [2, 4])
@pytest.mark.parametrize("H,Lq,Lk,D", [(40, 32760, 32760, 128), (12, 32760, 32865, 96), (16, 32865, 32865, 64), (16, 1565, 1565, 64),
                                       (40, 1560, 1560, 128), (40, 32760, 512, 128)])
def test_attention_plan_covers_every_batched_tile_once(B, H, Lq, Lk, D):
    """fwb_attn_plan at batch B: the B*H*ceil(Lq/256) tiles (tile -> q block, head, batch as the kernels decode it) and, for the
    split tail, every key tile of every split, are each covered exactly once."""
    import fwb200
    sms, ws = 148, int(fwb200.lib.fwb_attn_workspace_bytes())
    n_full, S = C.c_int(), C.c_int()
    assert fwb200.lib.fwb_attn_plan(B, H, Lq, Lk, D, ws, sms, C.byref(n_full), C.byref(S)) == 0
    nq = -(-Lq // 256)
    n_tiles = nq * H * B
    n_kv = -(-Lk // 128)
    assert 0 <= n_full.value <= n_tiles
    seen = torch.zeros(B, H, nq, n_kv, dtype=torch.int32)
    for tile in range(n_tiles):
        q, h, b = tile % nq, (tile // nq) % H, tile // (nq * H)
        splits = 1 if tile < n_full.value else S.value
        for sp in range(splits):
            kv0, kv1 = sp * n_kv // splits, (sp + 1) * n_kv // splits
            seen[b, h, q, kv0:kv1] += 1
    assert bool((seen == 1).all())
    if S.value > 1:
        assert n_full.value % sms == 0 and n_tiles - n_full.value < sms


def test_shared_timestep_validation_is_host_only():
    from fwb200 import engine as E
    assert E.shared_timestep(torch.tensor([996.0]), 3).tolist() == [996.0]
    assert E.shared_timestep(torch.tensor([700.0, 700.0]), 2).tolist() == [700.0]
    assert E.shared_timestep(torch.tensor(500.0), 1).tolist() == [500.0]
    with pytest.raises(ValueError, match="share the timestep"):
        E.shared_timestep(torch.tensor([900.0, 500.0]), 2)
    with pytest.raises(ValueError, match="3 elements for a batch of 2"):
        E.shared_timestep(torch.tensor([900.0, 900.0, 900.0]), 2)
    with pytest.raises(ValueError, match="share the timestep"):
        E.shared_rows(torch.stack([torch.zeros(6, 8), torch.ones(6, 8)]), "dit_mod_vectors")
    m = torch.ones(3, 6, 8)
    assert E.shared_rows(m, "x").shape == (1, 6, 8)


class _Core:
    """The sampler's batch checks need only `sp` / `cfgp` and tensor shapes."""


def _core(sp=None, cfgp=None):
    from FantasyWorld.fusion.core import FusionCore
    c = _Core()
    c.sp, c.cfgp, c.PER_SAMPLE_KW = sp, cfgp, FusionCore.PER_SAMPLE_KW
    c.check_batch = FusionCore.check_batch.__get__(c)
    return c


def test_sampler_batch_checks():
    lat, ctx = torch.zeros(2, 16, 3, 4, 6), torch.zeros(2, 16, 4096)
    kw = dict(clip_feature=torch.zeros(2, 257, 1280), y=torch.zeros(2, 20, 3, 4, 6), plucker_fea=torch.zeros(2, 36, 2048),
              plucker_context_lens=torch.ones(2, dtype=torch.long))
    assert _core().check_batch(lat, ctx, ctx, kw) == 2
    assert _core().check_batch(lat, ctx, ctx, kw, batch_cfg=True) == 2
    # per-sample inputs must have the batch of the latents: no broadcasting of a batch-1 context
    with pytest.raises(ValueError, match="context_neg has batch 1"):
        _core().check_batch(lat, ctx, ctx[:1], kw)
    with pytest.raises(ValueError, match="y has batch 1"):
        _core().check_batch(lat, ctx, ctx, {**kw, "y": kw["y"][:1]})

    class SP:
        world = 2
    with pytest.raises(ValueError, match="batch_cfg=True"):
        _core(cfgp=object()).check_batch(lat[:1], ctx[:1], ctx[:1], {}, batch_cfg=True)
    with pytest.raises(ValueError, match="batch_cfg=True"):
        _core(sp=SP()).check_batch(lat[:1], ctx[:1], ctx[:1], {}, batch_cfg=True)
    with pytest.raises(ValueError, match="batch of 2 is not supported"):
        _core(sp=SP()).check_batch(lat, ctx, ctx, kw)
    assert _core(sp=SP()).check_batch(lat[:1], ctx[:1], ctx[:1], {}) == 1
