"""2-GPU sequence-parallel equivalence: joint_forward sharded over 2 ranks (NCCL) == the single-GPU joint_forward.
Every kernel is row-independent and the gathers only move bytes, so the results must be bit-identical."""
import os
import socket

import pytest
import torch

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from fwb200.sp import SPContext
        from fwb200.synth import build_fusion_model, synth_inputs
        dev = torch.device("cuda", rank)
        model = build_fusion_model(num_dit_layers=3, start_index=1, device=dev, seed=0, heads=True, gen_device="cpu")
        model.pipe.device = dev
        for head in (model.vggt.depth_head, model.vggt.point_head):
            head.intermediate_layer_idx = [1, 1, 0, 0]
        f, h, w = 3, 4, 6                                  # 3 frames over 2 ranks: ragged geometry shards (2 + 1)
        inp = synth_inputs(f, h, w, device=dev, seed=1024, text_len=64)
        ts = torch.tensor([996.0], device=dev, dtype=torch.bfloat16)
        kw = dict(timestep=ts, context=inp["context_pos"], clip_feature=inp["clip_feature"], y=inp["y"],
                  use_gradient_checkpointing=False, plucker_fea=inp["plucker_fea"], return_prediction=True)
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            ref, ref_pred = model.joint_forward(inp["latents"], **kw)
            model.sp = SPContext()
            out, pred = model.joint_forward(inp["latents"], **kw)
            out2, _ = model.joint_forward(inp["latents"], **{**kw, "return_prediction": False})
        assert torch.isfinite(out.float()).all()
        assert torch.equal(out, ref), float((out.float() - ref.float()).abs().max())
        assert torch.equal(out2, ref)
        for k in ref_pred:
            a, b = pred[k].float(), ref_pred[k].float()
            assert a.shape == b.shape and float((a - b).abs().max()) <= 1e-2 * float(b.abs().max()) + 1e-6, k
        assert model.sp.n_gathers > 0
        # larger grid: the pipelined exchange (K|V gathered in slices on a side stream, split-KV partial attentions + merge)
        f, h, w = 2, 16, 32                                 # L = 1024 -> 512 rows per rank -> 2 slices
        inp = synth_inputs(f, h, w, device=dev, seed=7, text_len=64)
        kw = dict(timestep=ts, context=inp["context_pos"], clip_feature=inp["clip_feature"], y=inp["y"],
                  use_gradient_checkpointing=False, plucker_fea=inp["plucker_fea"])
        with torch.no_grad():
            sp = model.sp
            model.sp = None
            ref, _ = model.joint_forward(inp["latents"], **kw)
            model.sp = sp
            assert sp.kv_chunks == 2
            out, _ = model.joint_forward(inp["latents"], **kw)
        rel = float((out.float() - ref.float()).norm() / ref.float().norm())
        assert rel < 1e-2, rel                              # merge re-association flips a few bf16 roundings, which then propagate
        # CFG parallelism at 2 ranks: rank 0 = conditional forward, rank 1 = unconditional forward (no sharding inside a half),
        # one swap of the predictions: the step must be BIT-IDENTICAL to the serial two-forward step on one GPU
        model.sp = None
        sched = model.pipe.scheduler
        sched.set_timesteps(50)
        lens = torch.ones(f, dtype=torch.long, device=dev)
        lens[1:] = 4
        skw = dict(clip_feature=inp["clip_feature"], y=inp["y"], plucker_fea=inp["plucker_fea"], plucker_context_lens=lens, cfg_scale=5.0)
        lat_ref, _ = model.denoise_step(inp["latents"].clone(), 3, inp["context_pos"], inp["context_neg"], **skw)
        cp = model.enable_cfg_parallel()
        assert cp.role == rank and model.sp is None
        lat_cp, _ = model.denoise_step(inp["latents"].clone(), 3, inp["context_pos"], inp["context_neg"], **skw)
        assert torch.equal(lat_cp, lat_ref), float((lat_cp.float() - lat_ref.float()).abs().max())
        assert cp.n_exchanges == 1
        ret[rank] = True
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sequence_parallel_2gpu_matches_single_gpu():
    import torch.multiprocessing as mp
    port = _free_port()
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(2, port, ret), nprocs=2, join=True)
    assert ret.get(0) and ret.get(1)
