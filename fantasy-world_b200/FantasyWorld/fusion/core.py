"""Shared execution core of the two fusion models (Wan2.1: FantasyWorld/fusion/model_wan21.py, Wan2.2:
FantasyWorld/fusion/model_wan22.py): token embedding, the PCB / frame-block / IRG-block schedule, the head, hoisting of
loop-invariant work and the sequence-parallel variant.  The two reference joint_forward bodies (model_wan21.py:104-224,
model_wan22.py:226-348) differ only in how the latent is turned into tokens (CLIP context + camera AdaLN features vs the
control-adapter added in patchify); everything after that is identical and lives here once.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from fwb200 import engine as E
from fwb200 import ops

from ..diffsynth_wan21.models.wan_video_dit import _grid_freqs, build_freqs_3d_with_extra_cis


class FusionCore(nn.Module):
    """Mixin holding everything both fusion models share.  Subclasses provide `pipe.dit`, `vggt`, `IRGBlock`,
    `start_index`, `cross_attention_list`, `freqs_bicross`; optional `sp` (fwb200.sp.SPContext) turns on sequence parallelism."""

    sp = None
    cfgp = None     # fwb200.sp.CFGParallel: the two CFG forwards of a step on the two halves of the node (sets .sp itself)

    def enable_cfg_parallel(self):
        """Collective over the default process group: split the ranks into a conditional and an unconditional half
        (each sequence-parallel inside) — see fwb200.sp.CFGParallel.  denoise_step then evaluates ONE forward per rank."""
        from fwb200.sp import CFGParallel
        self.cfgp = CFGParallel()
        self.sp = self.cfgp.sp
        return self.cfgp

    # per-sample keyword inputs of joint_forward (batch dimension first); everything else is shared by the batch
    PER_SAMPLE_KW = ("clip_feature", "y", "plucker_fea", "control_camera_latents_input", "camera_token")

    def check_batch(self, latents, context_pos, context_neg, kw, batch_cfg=False):
        """Batch size of a sampler call, validated: every per-sample input has the batch size of `latents` (no implicit
        broadcasting), and a batch > 1 or `batch_cfg` is refused under sequence or CFG parallelism."""
        b = latents.shape[0]
        named = [("context_pos", context_pos), ("context_neg", context_neg)] + [(k, kw.get(k)) for k in self.PER_SAMPLE_KW]
        for name, v in named:
            if v is not None and v.shape[0] != b:
                raise ValueError(f"{name} has batch {v.shape[0]}, latents have batch {b}: every per-sample input needs the same batch")
        parallel = self.cfgp is not None or (self.sp is not None and self.sp.world > 1)
        if batch_cfg and parallel:
            raise ValueError("batch_cfg=True runs both CFG forwards as one batch on one GPU; it cannot be combined with "
                             "enable_cfg_parallel() or sequence parallelism (model.sp)")
        if b > 1 and parallel:
            raise ValueError(f"a batch of {b} is not supported under sequence or CFG parallelism: run batch 1 per call")
        return b

    def _cat_cached(self, *ts):
        """torch.cat(ts) of loop-invariant inputs, cached per tensor tuple (stable identity keeps the context / K-V caches warm)."""
        cache = self.__dict__.get("_fwb_cat")
        if cache is None:
            cache = self.__dict__["_fwb_cat"] = E.IdCache(8)
        return cache.get(ts, None, lambda: torch.cat(ts))

    def _cfg_forwards(self, latents, t, context_pos, context_neg, kw, return_prediction, batch_cfg=False):
        """(pred_pos, pred_neg, prediction) of one step.  Serial: both forwards here (reference order, model_wan21.py:295-317).
        CFG-parallel: this rank evaluates only its half's forward and the halves swap predictions; the geometry-head
        prediction exists on the conditional half only (the reference takes it from the conditional pass).
        batch_cfg: ONE forward of batch 2B over cat([latents, latents]) with cat([context_pos, context_neg]); the two
        predictions are the contiguous halves of its output and the head prediction comes from the conditional half."""
        b = self.check_batch(latents, context_pos, context_neg, kw, batch_cfg)
        if batch_cfg:
            kw2 = {k: (self._cat_cached(v, v) if k in self.PER_SAMPLE_KW and v is not None else v) for k, v in kw.items()}
            out, pred = self.joint_forward(torch.cat([latents, latents]), timestep=t, context=self._cat_cached(context_pos, context_neg),
                                           return_prediction=return_prediction, **kw2)
            if pred is not None:
                pred = {k: v[:b] for k, v in pred.items()}
            return out[:b], out[b:], pred
        if self.cfgp is None:
            pred_pos, pred = self.joint_forward(latents, timestep=t, context=context_pos, return_prediction=return_prediction, **kw)
            pred_neg, _ = self.joint_forward(latents, timestep=t, context=context_neg, **kw)
            return pred_pos, pred_neg, pred
        role = self.cfgp.role
        mine, pred = self.joint_forward(latents, timestep=t, context=context_pos if role == 0 else context_neg,
                                        return_prediction=return_prediction and role == 0, **kw)
        pred_pos, pred_neg = self.cfgp.exchange(mine)
        return pred_pos, pred_neg, pred

    # ---- loop-invariant inputs (SURVEY Appendix E) ------------------------------------------------------------------------
    def embed_context(self, context, clip_feature=None):
        """text_embedding(context) (+ img_emb(clip) in front for Wan2.1-I2V): depends only on the prompt / first frame, so it
        is computed once per (context, clip) tensor pair instead of once per forward.  ref: model_wan21.py:123-128."""
        dit = self.pipe.dit
        cache = self.__dict__.get("_fwb_ctx")
        if cache is None:
            cache = self.__dict__["_fwb_ctx"] = E.IdCache(4)

        def build():
            ctx = dit.embed_text(context)
            if dit.has_image_input:
                ctx = torch.cat([dit.img_emb(clip_feature).to(ctx.dtype), ctx], dim=1)
            return ctx.contiguous()

        srcs = (context,) + ((clip_feature,) if (dit.has_image_input and clip_feature is not None) else ()) + (dit.text_embedding[0].weight,)
        return cache.get(srcs, None, build)

    def rope_tables(self, f, h, w, device):
        """freqs (D=128), freqs_bi_dit (D=96), freqs_bi_agg (D=96 with 5 identity rotations per frame).
        ref: model_wan21.py:132-147."""
        store = self.__dict__.setdefault("_fwb_rope", {})
        key = (f, h, w, str(device))
        if key not in store:
            dit = self.pipe.dit
            store[key] = (_grid_freqs(dit.freqs, f, h, w).reshape(f * h * w, 1, -1).to(device),
                          _grid_freqs(self.freqs_bicross, f, h, w).reshape(f * h * w, 1, -1).to(device),
                          build_freqs_3d_with_extra_cis(self.freqs_bicross, f, h, w, n_extra=5, device=device))
        return store[key]

    def _local_rows(self, t: torch.Tensor, r0: int, r1: int):
        """Cached row slice t[:, r0:r1] of a loop-invariant [1, L, C] tensor (stable identity keeps downstream caches warm)."""
        cache = self.__dict__.get("_fwb_rows")
        if cache is None:
            cache = self.__dict__["_fwb_rows"] = E.IdCache(4)
        def build():
            loc = t[:, r0:r1].contiguous()
            loc._fwb_all_zero = bool(torch.all(t == 0).item())     # all-zero test of the FULL tensor (camera AdaLN skip, see processor)
            return loc

        return cache.get((t,), (r0, r1), build)

    def _control_tokens(self, control):
        """Wan2.2 control adapter output as tokens [L, dim]: a conv stack over the camera latents that depends only on the
        camera path (71 TFLOP per forward at 720p in the reference, SURVEY Appendix E) — evaluated once per sample."""
        dit = self.pipe.dit
        cache = self.__dict__.get("_fwb_ctrl")
        if cache is None:
            cache = self.__dict__["_fwb_ctrl"] = E.IdCache(2)

        def build():
            yc = dit.control_adapter(control)                    # [b, dim, f, h, w] -> [(b f h w), dim]
            return E.as_bf16(yc.permute(0, 2, 3, 4, 1).reshape(-1, yc.shape[1])).contiguous()

        return cache.get((control, dit.control_adapter.conv.weight), None, build)

    # ---- the shared forward -----------------------------------------------------------------------------------------------
    def _joint_core(self, x, timestep, ctx, block_kw, plucker_fea=None, control=None, camera_token=None, uncond=False,
                    return_prediction=False):
        """x: the concatenated latent [B, C_in, F, H, W]; ctx: embedded context [B, n_ctx, dim].  Single GPU when self.sp is
        None (or world 1), otherwise token-sharded (SURVEY §8e, batch 1 only): video rows L/P per rank, frame-aligned geometry
        shards, one all-gather of packed K|V per attention, one gather of the projected tokens and one of the head output per
        forward.  At batch B every sample has its own latents, context and camera inputs and all share the timestep; each
        sample's tokens attend only to its own (B*L token rows, [B, L, H, D] attention views)."""
        sp = self.sp if (self.sp is not None and self.sp.world > 1) else None
        dit, vggt, agg = self.pipe.dit, self.vggt, self.vggt.aggregator
        b, cin, F_, H_, W_ = x.shape
        timestep = E.shared_timestep(timestep, b)
        if sp is not None and b > 1:
            raise ValueError(f"a batch of {b} is not supported under sequence parallelism")
        for name, v in (("context", ctx), ("plucker_fea", plucker_fea), ("control_camera_latents_input", control)):
            if v is not None and v.shape[0] != b:
                raise ValueError(f"{name} has batch {v.shape[0]}, the latents have batch {b}")
        t, t_mod = dit.embed_time(timestep)
        pf, ph, pw = dit.patch_size
        f, h, w = F_ // pf, H_ // ph, W_ // pw
        L = f * h * w
        if sp is not None:
            assert camera_token is None, "camera_token conditioning is not sharded (not used by the sampler)"
            lay = sp.set_grid(f, h, w)
            r0, r1 = lay.video_range(sp.rank)
            f0, f1 = lay.frame_range(sp.rank)
        else:
            r0, r1, f0, f1 = 0, L, 0, f
        # patchify: Conv3d(k = s = patch) as a GEMM over unfolded patches, only this rank's rows (ref: wan_video_dit.py:424-435)
        cols = E.as_bf16(x).view(b, cin, f, pf, h, ph, w, pw).permute(0, 2, 4, 6, 1, 3, 5, 7).reshape(b * L, cin * pf * ph * pw)
        resid = None
        if control is not None and dit.control_adapter is not None:
            resid = self._control_tokens(control)
            resid = resid[r0:r1] if sp is not None else resid
        cols = cols[r0:r1] if sp is not None else cols
        xl = E.lin(cols.contiguous(), dit.patch_embedding, resid=resid, round_flags=ops.ROUND_AFTER_BIAS).view(b, -1, dit.dim)
        freqs, freqs_bi_dit, freqs_bi_agg = self.rope_tables(f, h, w, xl.device)
        kw = dict(block_kw)
        if plucker_fea is not None:
            kw["plucker_fea"] = self._local_rows(plucker_fea, r0, r1) if sp is not None else plucker_fea

        E.SP = sp
        try:
            for i in range(self.start_index):                                   # Preconditioning Blocks
                xl = dit.blocks[i](xl, ctx, t_mod, freqs, **kw)
            # 5120 -> 1024 projection on local rows (then, under SP, one gather so that every rank can pick its frames)
            proj = vggt.project_tokens(xl)
            if sp is not None:
                proj = sp.all_gather_rows(proj[0], lay.video_rows)
            patch_all = proj.view(b, f, h, w, -1)
            e0 = vggt.time_modulation(timestep)
            if sp is not None:
                tokens, pos = agg._process_aggregator_input(patch_all[:, f0:f1], None, frame_range=(f0, f1))
            else:
                tokens, pos = agg._process_aggregator_input(patch_all, camera_token)
            S, (_, P, C) = f1 - f0, tokens.shape
            n_layers = len(dit.blocks) - self.start_index
            keep = None
            if return_prediction and sp is not None:                            # gather only what the heads read
                keep = {n_layers - 1}
                for head in (vggt.depth_head, vggt.point_head):
                    if head is not None:
                        keep |= {li % n_layers for li in head.intermediate_layer_idx}
            frame_idx = global_idx = 0
            output_list = []
            for i in range(n_layers):
                tokens, frame_idx, frame_inter = agg._process_frame_attention(tokens, b, S, P, C, frame_idx, pos=pos, e0=e0)
                if i in self.cross_attention_list:
                    xl, tokens, global_inter = self.IRGBlock[i](x_dit=xl, x_agg=tokens, context=ctx, t_mod=t_mod, freqs=freqs,
                                                                freqs_dit=freqs_bi_dit, freqs_agg=freqs_bi_agg, pos=pos, e0=e0,
                                                                uncond=uncond, **kw)
                    global_idx += 1
                else:
                    assert sp is None, "sequence parallel path expects every post-PCB block to be an IRG block"
                    xl = dit.blocks[i + self.start_index](xl, ctx, t_mod, freqs, **kw)
                    tokens, global_idx, global_inter = agg._process_global_attention(tokens, b, S, P, C, global_idx, pos=pos, e0=e0)
                if return_prediction:  # only the last step consumes these 2C-wide intermediates (ref: :208-212, :217-222)
                    if sp is None:
                        output_list.extend(torch.cat([a, b_], dim=-1) for a, b_ in zip(frame_inter, global_inter))
                    elif i in keep:
                        loc = torch.cat([frame_inter[0].reshape(S * P, C), global_inter[0].reshape(S * P, C)], dim=-1).contiguous()
                        output_list.append(sp.all_gather_rows(loc, lay.geo_rows()).view(1, f, P, 2 * C))
                    else:
                        output_list.append(None)
            out = dit.head(xl, t)
        finally:
            E.SP = None
        if sp is not None:
            out = sp.all_gather_rows(out[0].contiguous(), lay.video_rows).unsqueeze(0)
        out = dit.unpatchify(out, (f, h, w))
        if not return_prediction:
            return out, None
        if b == 1:
            return out, vggt._head_predction(patch_all, agg.patch_start_idx, output_list)
        # the heads run per sample: their convolutions then see the batch-1 shapes of a single call
        preds = [vggt._head_predction(patch_all[i:i + 1], agg.patch_start_idx, [o[i:i + 1] for o in output_list]) for i in range(b)]
        return out, {k: torch.cat([p[k] for p in preds]) for k in preds[0]}
