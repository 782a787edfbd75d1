/* fwb200.h — C ABI of libfwb200.so, the B200 (sm_100a) kernel library behind the FantasyWorld denoising hot path.
 *
 * The reference (Fantasy-AMAP/fantasy-world) has no native code and no FFI: its "operator API" for this path is the
 * set of PyTorch library calls listed in SURVEY.md §2.1 (K1..K11).  Each entry point below replaces one family of those
 * call sites; the file:line it replaces is cited per function.  The host side (Python, package
 * `fantasy-world_b200/FantasyWorld`) mirrors the reference's nn.Module surface and calls these through ctypes.
 *
 * Conventions
 *   - plain pointers + sizes; every pointer is a DEVICE pointer unless stated; no torch types
 *   - the caller owns all memory (outputs are pre-allocated); kernels never allocate
 *   - all launches go to `stream` (a cudaStream_t); no host synchronisation inside
 *   - return value: 0 = ok, non-zero = error; `fwb_last_error()` returns a thread-local message
 *   - bf16 tensors are row-major with the stated leading dimensions (in ELEMENTS)
 */
#ifndef FWB200_H_
#define FWB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FWB_ABI_VERSION 3

typedef struct CUstream_st* fwb_stream_t; /* == cudaStream_t */

enum { FWB_DT_BF16 = 0, FWB_DT_F32 = 1 };
enum { FWB_ACT_NONE = 0, FWB_ACT_GELU_TANH = 1, FWB_ACT_GELU_ERF = 2, FWB_ACT_RELU = 3, FWB_ACT_SILU = 4 };

/* bits of fwb_epilogue_t.round_flags: round the running value to bf16 (as CUDA autocast does between ops) */
enum {
  FWB_ROUND_AFTER_BIAS = 1,   /* nn.Linear output is bf16 under autocast */
  FWB_ROUND_AFTER_ACT = 2,    /* activation output bf16 */
  FWB_ROUND_AFTER_AFFINE = 4, /* after *scale1 + shift1 */
  FWB_ROUND_AFTER_SCALE2 = 8
};

/* ---- introspection ------------------------------------------------------------------------------------------- */
const char* fwb_last_error(void);
int fwb_abi_version(void);
/* 1 if a sm_100 device is current, else 0 (and fwb_last_error() says why). Product paths refuse to run without it. */
int fwb_device_ok(void);

/* ---- K6/K10: Linear (+bias, activation, column affine, gate, residual) -------------------------------------------
 * out[m,n] = resid[m,n] + scale2[n] * ( scale1[n] * act( sum_k A[m,k] W[n,k] + bias[n] ) + shift1[n] )
 * Replaces: nn.Linear call sites wan_video_dit.py:166-169,216-225,274-275 ; GateModule wan_video_dit.py:246-251 ;
 *           fusion/layer/block.py:340-346,218-219 ; vggt/layers/attention.py:42,46 ; vggt/layers/mlp.py:29-31 ;
 *           vggt/layers/block.py:73-81 (LayerScale / post-MLP modulation) ; camera_control.py:27-51 ; vggt.py:32.
 * A: [M,K] bf16 (lda), W: [N,K] bf16 (ldw) — nn.Linear weight layout.  K, lda, ldw, N, out_ld, resid_ld % 8 == 0.
 * All column vectors are fp32 [N] (NULL = absent).  Accumulation fp32 on tcgen05 tensor cores. */
typedef struct {
  const float* bias;
  const float* scale1;
  const float* shift1;
  const float* scale2;
  const void* resid; /* [M,N] or NULL */
  int64_t resid_ld;
  int resid_dtype; /* FWB_DT_* */
  void* out;       /* [M,N] */
  int64_t out_ld;
  int out_dtype; /* FWB_DT_* */
  int act;       /* FWB_ACT_* */
  int round_flags;
} fwb_epilogue_t;

int fwb_gemm_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, int M, int N, int K, const fwb_epilogue_t* ep,
                  fwb_stream_t stream);
/* Test / tuning hook: force the kernel variant (-1 automatic, 0 single-CTA 128x128, 1 single-CTA 128x256,
 * 2 CTA-pair 256x256 cta_group::2).  Results are identical across variants up to fp32 summation order. */
int fwb_gemm_set_mode(int mode);

/* ---- K1..K5: non-causal softmax attention ------------------------------------------------------------------------
 * out[b,l,h,:] = softmax_j( scale * q[b,l,h,:] . k[b,j,h,:] ) v[b,j,h,:]      (no mask, no dropout)
 * Replaces: flash_attention() wan_video_dit.py:28-66 (DiT self/cross attention), F.scaled_dot_product_attention at
 *           fusion/layer/block.py:598-605 (adapter, both directions) and vggt/layers/attention.py:61 (frame/global).
 * q,k,v,out: bf16, head_dim D in {64, 96, 128} contiguous; element strides given per tensor for batch (sb),
 * token (sl) and head (sh); all strides % 8 == 0.  scale is the softmax scale (reference: 1/sqrt(D)).
 * fp32 softmax statistics, P rounded to bf16 before PV (as flash-attn / cuDNN do), fp32 accumulation.
 * accumulate != 0: out = bf16(out + bf16(result)) — the text + CLIP attention sum of wan_video_dit.py:197-200. */
typedef struct {
  const void* ptr;
  int64_t sb, sl, sh;
} fwb_tensor4_t;

/* workspace (optional, may be NULL / 0): device scratch of fwb_attn_workspace_bytes() bytes, 16-byte aligned, private to the
 * stream.  With it, when the tile count (ceil(Lq/256) * H * B) leaves the last wave of CTAs partly empty, the tiles of that
 * wave are split along the keys over the idle SMs and merged (same result up to one rounding of the merge weights).  This is
 * what keeps the sequence-parallel shards (Lq = L / ranks) from losing up to a full wave per attention. */
size_t fwb_attn_workspace_bytes(void);
/* The schedule fwb_attn_fwd would choose (pure host arithmetic, no device needed): how many tiles run unsplit and into how many
 * key splits each remaining tile is cut (1 = no split), for n_sms SMs and a workspace of workspace_bytes. */
int fwb_attn_plan(int B, int H, int Lq, int Lk, int D, size_t workspace_bytes, int n_sms, int* n_unsplit_tiles, int* key_splits);
int fwb_attn_fwd(const fwb_tensor4_t* q, const fwb_tensor4_t* k, const fwb_tensor4_t* v, const fwb_tensor4_t* out, int B,
                 int H, int Lq, int Lk, int D, float scale, int accumulate, void* workspace, size_t workspace_bytes,
                 fwb_stream_t stream);

/* Split-KV attention (sequence-parallel pipelining: attention over the key chunk that has already arrived overlaps the
 * all-gather of the next chunk).  fwb_attn_fwd_partial writes, for one disjoint subset of the keys, the subset-normalised
 * result in fp32 (part_out [B, Lq, H, D]) and the row log-sum-exp in base 2 with the scale folded in (part_lse [B, H, Lq]);
 * fwb_attn_merge combines S such partials (part [S, B, Lq, H, D], lse [S, B, H, Lq]) into the bf16 output:
 * out = sum_s 2^(lse_s - max) part_s / sum_s 2^(lse_s - max).  Mathematically identical to one fwb_attn_fwd over all keys. */
int fwb_attn_fwd_partial(const fwb_tensor4_t* q, const fwb_tensor4_t* k, const fwb_tensor4_t* v, float* part_out, float* part_lse,
                         int B, int H, int Lq, int Lk, int D, float scale, void* workspace, size_t workspace_bytes,
                         fwb_stream_t stream);
int fwb_attn_merge(const float* part, const float* lse, const fwb_tensor4_t* out, int S, int B, int H, int L, int D,
                   fwb_stream_t stream);
/* Why there is no `fwb_attn_fwd_sp(..., ncclComm_t, kv_chunks)` / `fwb_allgather_kv` entry point (SURVEY §8b lists them as an
 * option): the exchange itself is ONE NCCL all-gather of the packed K|V rows per attention, and the host side of this path is
 * PyTorch (north star), which already owns the NCCL communicator (ProcessGroupNCCL, one per process / GPU).  Pulling a raw
 * ncclComm_t through a C ABI would either duplicate that communicator (a second NVLS / ring set-up per process and a second
 * stream-ordering domain) or reach into torch internals.  So the collective is issued by the host layer on a side stream
 * (fwb200/sp.py: all_gather_into_tensor in `kv_chunks` row slices) and what the ABI exports is the compute half of the
 * pipeline: fwb_attn_fwd_partial consumes slice c while slice c+1 is in flight, fwb_attn_merge combines the slices.  The pair
 * (host all-gather slice, fwb_attn_fwd_partial) is the `attn_fwd_sp` of the survey, split at the library boundary. */

/* Tuning / test hooks (process-wide; one process drives one GPU).  None of them changes what is computed beyond fp32
 * re-association or the sub-bf16 error of the exp2 polynomial; they select between measured kernel variants.
 *   fwb_attn_set_variant        0 = default per head_dim (64 -> decoupled S/P kernel, 96 / 128 -> aliased S/P kernel), 1 / 2 = force
 *   fwb_attn_set_tail_split     key-split tail of the tile schedule on (1, default) / off (0)
 *   fwb_attn_set_exp2_poly      pairs out of every 8 softmax element pairs whose 2^x comes from the packed FMA-pipe polynomial
 *                               instead of MUFU.EX2: -1 = default (2), 0 = MUFU only, 2 (max rel. error 8.6e-5 before P is rounded
 *                               to bf16; larger shares were measured slower and are not built)
 *   fwb_attn_set_mufu_pingpong  kernel 1 (aliased) / 2 (decoupled): alternate the exp2 phases of the two Q tiles of a CTA */
int fwb_attn_set_variant(int variant);
int fwb_attn_set_tail_split(int enabled);
int fwb_attn_set_exp2_poly(int pairs_of_8);
int fwb_attn_set_mufu_pingpong(int kernel, int enabled);
/* head_dim 96 (runs on the 128-wide instance with zero-filled columns): issue the PV MMAs with N = 96 instead of 128
 * (default on: bit-identical result, no MMA work on the padded columns; 0 = off for the A/B) */
int fwb_attn_set_pv_n96(int enabled);
/* aliased kernel, head_dim 128, >= 2048 keys, even number of 256-row query blocks, no key-split tail: run as clusters of two CTAs on
 * adjacent query blocks of one head that share every K/V tile through TMA multicast (halves the L2 -> SM traffic); bit-identical
 * results; default on (0 = off for the A/B) */
int fwb_attn_set_multicast(int enabled);
/* default kernel policy: problems with at most max_keys keys run the aliased kernel with ONE 128-row Q tile per CTA and two CTAs per SM
 * (prologue / epilogue of one CTA overlap the main loop of the other); 0 disables, default 2048 */
int fwb_attn_set_short_kv_max(int max_keys);

/* ---- K7: LayerNorm (+affine) (+modulate) -> bf16 ------------------------------------------------------------------
 * out[r,:] = bf16( (LN(x[r,:]) * w + b) * mul + add ), any of (w,b), mul, add may be NULL.  fp32 statistics.
 * Replaces: modulate(norm(x), shift, scale) wan_video_dit.py:69-70,301,311 (mul = 1+scale, add = shift); norm3 (:302);
 *           Head (:353-358); vggt Block norm1/norm2 (+e-modulation) vggt/layers/block.py:73-81; adapter input norms
 *           fusion/layer/block.py:197; img_emb LayerNorms wan_video_dit.py:324-341.
 * x: [rows,C] bf16 or fp32 (x_dtype), C % 8 == 0, C <= 5120; vectors fp32 [C]; out bf16 [rows,C]. */
int fwb_ln_modulate(const void* x, int x_dtype, int64_t ldx, int rows, int C, float eps, const float* w, const float* b,
                    const float* mul, const float* add, void* out, int64_t ldo, fwb_stream_t stream);
/* Tuning hook: 128-thread CTAs per SM of the persistent row kernels (fwb_ln_modulate, fwb_rmsnorm_rope): 0 = one full wave of as many
 * as fit (occupancy query per kernel, default), 1..16 = forced (A/B measurements) */
int fwb_rowwise_set_ctas_per_sm(int n);

/* ---- K8+K9 (DiT / adapter): full-channel RMSNorm then interleaved-pair RoPE, in place --------------------------------
 * x[r,:] <- rope( bf16( bf16(x * rsqrt(mean(x^2)+eps)) * w ) ), w == NULL skips the norm, cos_sin == NULL skips RoPE.
 * cos_sin: fp32 [rows, head_dim/2, 2] = (cos, sin) of the per-token 3-D RoPE angle, shared by all heads.
 * Replaces: RMSNorm wan_video_dit.py:135-146 (norm_q/norm_k :176-177, :192-196) and rope_apply :97-102
 *           (DiT :178-179; adapter fusion/layer/block.py:545-550). */
int fwb_rmsnorm_rope(void* x, int64_t ldx, int rows, int C, const float* w, float eps, const float* cos_sin, int head_dim,
                     fwb_stream_t stream);
/* Batched form: row r reads cos_sin row (r % table_rows); table_rows must divide rows.  At batch B the token rows are B*L
 * while the table is per position (L rows), so one cached table serves every sample.  fwb_rmsnorm_rope is this call with
 * table_rows = rows (same results).
 * Call sites: the DiT self-attention q/k (wan_video_dit.py:176-179) and the adapter q/k (fusion/layer/block.py:545-550)
 * at batch > 1 (fwb200/engine.py dit_self_attn, bicross). */
int fwb_rmsnorm_rope_periodic(void* x, int64_t ldx, int rows, int C, const float* w, float eps, const float* cos_sin,
                              int table_rows, int head_dim, fwb_stream_t stream);

/* ---- K8+K9 (VGGT): per-head LayerNorm(64) + 2-D rotate-half RoPE on q and k of a packed qkv buffer, in place --------
 * qkv: bf16 [rows, 3*H*64] laid out (3, H, 64); cosT/sinT: fp32 [rows, 64] expanded tables (first 32 = y, last 32 = x).
 * Replaces: q_norm/k_norm + rope vggt/layers/attention.py:52-58, vggt/layers/rope.py:133-188. */
int fwb_ln64_rope2d(void* qkv, int64_t ld, int rows, int H, float eps, const float* qw, const float* qb, const float* kw,
                    const float* kb, const float* cosT, const float* sinT, fwb_stream_t stream);
/* Batched form: row r reads cosT / sinT row (r % table_rows); table_rows must divide rows.  fwb_ln64_rope2d is this call with
 * table_rows = rows (same results).
 * Call sites: the VGGT frame and global blocks (vggt/layers/attention.py:52-58) at batch > 1, where the positions of every
 * sample are the same (fwb200/engine.py vggt_attn_part, tables from FantasyWorld/vggt/models/aggregator.py _positions). */
int fwb_ln64_rope2d_periodic(void* qkv, int64_t ld, int rows, int H, float eps, const float* qw, const float* qb, const float* kw,
                             const float* kb, const float* cosT, const float* sinT, int table_rows, fwb_stream_t stream);

/* ---- a1/a18: classifier-free guidance + flow-matching Euler update, in place on bf16 latents ------------------------
 * latents <- latents + (neg + cfg*(pos-neg)) * dsigma with the reference's bf16 rounding after every op.
 * Replaces: fusion/model_wan21.py:318-322, diffsynth_wan21/schedulers/flow_match.py:43-53. */
int fwb_cfg_euler_step(void* latents, const void* pred_pos, const void* pred_neg, int64_t n, float cfg_scale, float dsigma,
                       fwb_stream_t stream);

/* ---- bring-up micro-test (tests only; pins tcgen05 descriptor encodings on hardware) ------------------------------ */
int fwb_bringup_mma(const void* A, const void* B, float* D, int N, int K, int a_in_tmem, int b_mn_major,
                    const uint32_t* overrides, fwb_stream_t stream);
/* PV configuration (A in TMEM, B MN-major) with an MMA N narrower than the loaded tile (mma_n = 96: native head_dim-96 PV). */
int fwb_bringup_mma_pv_n(const void* A, const void* B, float* D, int N, int K, int mma_n, fwb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* FWB200_H_ */
