// fwb_rowwise.cu — HBM-bound row kernels that sit between the GEMMs and the attentions (SURVEY §2.1 K7, K8, K9).
//
//   fwb_ln_modulate     y = bf16( (LN(x) * w + b) * mul + add )          wan_video_dit.py:69-70,301,311 ;
//                                                                         vggt/layers/block.py:73-81 ; fusion/layer/block.py:197
//   fwb_rmsnorm_rope    full-channel RMSNorm (+weight) then interleaved-pair RoPE, in place
//                                                                         wan_video_dit.py:135-146,97-102,176-181 ;
//                                                                         fusion/layer/block.py:545-550
//   fwb_ln64_rope2d     per-head LayerNorm(64) + 2-D rotate-half RoPE on the q and k thirds of a packed qkv buffer
//                                                                         vggt/layers/attention.py:52-58 ; vggt/layers/rope.py:133-188
//   *_periodic          the same two RoPE kernels reading table row (row % table_rows): at batch B the token rows are B*L
//                       while the RoPE table is per position (L rows), so one table serves every sample
//   fwb_cfg_euler_step  latents += (neg + s*(pos-neg)) * dsigma           fusion/model_wan21.py:318-322 ; flow_match.py:43-53
//
// All are bandwidth bound: one pass over the row, 128-bit loads/stores, fp32 statistics with warp-shuffle reductions.
// Algorithmic bytes per element: read 2 (bf16) or 4 (fp32) + write 2.
#include "../../include/fwb200.h"
#include "fwb_common.cuh"
#include "fwb_host.h"

using namespace fwb;

namespace {

constexpr int kRowThreads = 128;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// block-wide sum for kRowThreads threads through a 4-float smem scratch, ONE barrier.  The scratch is not protected against the
// next call: consecutive reductions must alternate between two scratch buffers (a thread can only overwrite buffer A after the
// barrier of the reduction on buffer B, which every thread reaches after it has read A).
__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  return red[0] + red[1] + red[2] + red[3];
}

__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    f[2 * j] = __uint_as_float(w[j] << 16);
    f[2 * j + 1] = __uint_as_float(w[j] & 0xFFFF0000u);
  }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 u;
  u.x = pack_bf16x2(f[0], f[1]);
  u.y = pack_bf16x2(f[2], f[3]);
  u.z = pack_bf16x2(f[4], f[5]);
  u.w = pack_bf16x2(f[6], f[7]);
  return u;
}
__device__ __forceinline__ void load8_f32(const float* p, float (&f)[8]) {
  float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}

// ------------------------------------------------------------------------------------------------------------
// LayerNorm (+affine) (+modulate) -> bf16.  Persistent CTAs (a few per SM) walk the rows with a grid stride; thread t owns
// the 8-element chunks t, t+128, ...  The NEXT row's raw 16-byte chunks are loaded before the current row is reduced, so
// every CTA always has a full row of loads in flight while it sits in its two block-wide reductions (round 1 launched one
// CTA per row: the loads of a CTA came in one burst followed by ~1 us of reduction latency with nothing outstanding —
// 4.0 TB/s of the 6.57 TB/s copy bandwidth).  Per-thread element ownership and reduction order are unchanged, so results are
// bit-identical to the one-CTA-per-row version.
// ------------------------------------------------------------------------------------------------------------
template <int CHUNKS, bool IN_F32>
struct RowRaw {
  uint4 q[CHUNKS][IN_F32 ? 2 : 1];
};

template <int CHUNKS, bool IN_F32>
__device__ __forceinline__ void row_load(RowRaw<CHUNKS, IN_F32>& r, const void* __restrict__ x, long long ldx, int row, int nchunks) {
#pragma unroll
  for (int i = 0; i < CHUNKS; ++i) {
    const int ch = threadIdx.x + i * kRowThreads;
    if (ch < nchunks) {
      if (IN_F32) {
        const uint4* p = reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(x) + (size_t)row * ldx + ch * 8);
        r.q[i][0] = p[0];
        r.q[i][IN_F32 ? 1 : 0] = p[1];
      } else {
        r.q[i][0] = *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(x) + (size_t)row * ldx + ch * 8);
      }
    }
  }
}

template <int CHUNKS, bool IN_F32>
__device__ __forceinline__ void row_unpack(const RowRaw<CHUNKS, IN_F32>& r, int i, float (&f)[8]) {
  if (IN_F32) {
    const uint4 a = r.q[i][0], b = r.q[i][IN_F32 ? 1 : 0];
    f[0] = __uint_as_float(a.x); f[1] = __uint_as_float(a.y); f[2] = __uint_as_float(a.z); f[3] = __uint_as_float(a.w);
    f[4] = __uint_as_float(b.x); f[5] = __uint_as_float(b.y); f[6] = __uint_as_float(b.z); f[7] = __uint_as_float(b.w);
  } else {
    unpack8(r.q[i][0], f);
  }
}

template <int CHUNKS, bool IN_F32>
__global__ void __launch_bounds__(kRowThreads)
ln_modulate_kernel(const void* __restrict__ x, long long ldx, int rows, int C, float eps, const float* __restrict__ w,
                   const float* __restrict__ b, const float* __restrict__ mul, const float* __restrict__ add,
                   __nv_bfloat16* __restrict__ out, long long ldo) {
  __shared__ float red[4], red2[4];     // mean / variance reductions alternate (see block_sum)
  const int nchunks = C >> 3;
  RowRaw<CHUNKS, IN_F32> cur, nxt;
  int row = blockIdx.x;
  if (row >= rows) return;
  row_load(cur, x, ldx, row, nchunks);
  for (; row < rows; row += gridDim.x) {
    const int next = row + gridDim.x;
    if (next < rows) row_load(nxt, x, ldx, next, nchunks);
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) {
      if ((int)threadIdx.x + i * kRowThreads < nchunks) {
        float v[8];
        row_unpack(cur, i, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) s += v[j];
      }
    }
    const float mean = block_sum(s, red) / (float)C;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) {
      if ((int)threadIdx.x + i * kRowThreads < nchunks) {
        float v[8];
        row_unpack(cur, i, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float d = v[j] - mean;
          q += d * d;
        }
      }
    }
    const float rstd = rsqrtf(block_sum(q, red2) / (float)C + eps);
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) {
      const int ch = threadIdx.x + i * kRowThreads;
      if (ch < nchunks) {
        const int c0 = ch * 8;
        float v[8], y[8];
        row_unpack(cur, i, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) y[j] = (v[j] - mean) * rstd;
        if (w) {
          float ww[8], bb[8];
          load8_f32(w + c0, ww);
          load8_f32(b + c0, bb);
#pragma unroll
          for (int j = 0; j < 8; ++j) y[j] = y[j] * ww[j] + bb[j];
        }
        if (mul) {
          float mm[8];
          load8_f32(mul + c0, mm);
#pragma unroll
          for (int j = 0; j < 8; ++j) y[j] *= mm[j];
        }
        if (add) {
          float aa[8];
          load8_f32(add + c0, aa);
#pragma unroll
          for (int j = 0; j < 8; ++j) y[j] += aa[j];
        }
        *reinterpret_cast<uint4*>(out + (size_t)row * ldo + c0) = pack8(y);
      }
    }
    cur = nxt;
  }
}

// ------------------------------------------------------------------------------------------------------------
// RMSNorm over the full row (+weight) then RoPE on interleaved pairs, in place on bf16.
// Rounding points follow the reference: bf16(x*rstd) -> bf16(* w) -> rope in fp32 -> bf16.
// ------------------------------------------------------------------------------------------------------------
template <int CHUNKS>
__global__ void __launch_bounds__(kRowThreads)
rmsnorm_rope_kernel(__nv_bfloat16* __restrict__ x, long long ldx, int rows, int C, const float* __restrict__ w,
                    float eps, const float2* __restrict__ cs, int table_rows, int head_dim) {
  // persistent rows with the next row prefetched, as ln_modulate_kernel (in place: a row is only ever touched by one CTA)
  __shared__ float red[2][4];           // one reduction per row: alternate by row (see block_sum)
  int flip = 0;
  const int nchunks = C >> 3;
  const int half = head_dim >> 1;
  RowRaw<CHUNKS, false> cur, nxt;
  int row = blockIdx.x;
  if (row >= rows) return;
  row_load(cur, x, ldx, row, nchunks);
  for (; row < rows; row += gridDim.x) {
    const int next = row + gridDim.x;
    if (next < rows) row_load(nxt, x, ldx, next, nchunks);
    float rstd = 1.f;
    if (w) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < CHUNKS; ++i) {
        if ((int)threadIdx.x + i * kRowThreads < nchunks) {
          float v[8];
          row_unpack(cur, i, v);
#pragma unroll
          for (int j = 0; j < 8; ++j) s += v[j] * v[j];
        }
      }
      rstd = rsqrtf(block_sum(s, red[flip]) / (float)C + eps);
      flip ^= 1;
    }
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) {
      const int ch = threadIdx.x + i * kRowThreads;
      if (ch < nchunks) {
        const int c0 = ch * 8;
        float v[8], y[8];
        row_unpack(cur, i, v);
        if (w) {
          float ww[8];
          load8_f32(w + c0, ww);
#pragma unroll
          for (int j = 0; j < 8; ++j) y[j] = bf16_round(bf16_round(v[j] * rstd) * ww[j]);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) y[j] = v[j];
        }
        if (cs) {
          const int d0 = (c0 % head_dim) >> 1;  // first pair index inside the head
          const float2* t = cs + (size_t)(row % table_rows) * half + d0;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 c = __ldg(t + j);  // (cos, sin)
            const float a = y[2 * j], bq = y[2 * j + 1];
            y[2 * j] = a * c.x - bq * c.y;
            y[2 * j + 1] = a * c.y + bq * c.x;
          }
        }
        *reinterpret_cast<uint4*>(x + (size_t)row * ldx + c0) = pack8(y);
      }
    }
    cur = nxt;
  }
}

// ------------------------------------------------------------------------------------------------------------
// VGGT q/k: per-head LayerNorm(64, affine, eps) + 2-D rotate-half RoPE.  qkv row layout [3][H][64] bf16.
// 8 lanes per head (8 elements each).  cos/sin: per-row expanded tables [rows][64] fp32 (built on the host by the
// reference's own arithmetic: F.embedding gather by integer position).
// rot(f)[d] = -f[d+16] for (d%32) < 16, +f[d-16] otherwise  -> partner lane = lane ^ 2.
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
ln64_rope2d_kernel(__nv_bfloat16* __restrict__ qkv, long long ld, int rows, int H, float eps,
                   const float* __restrict__ qw, const float* __restrict__ qb, const float* __restrict__ kw,
                   const float* __restrict__ kb, const float* __restrict__ cosT, const float* __restrict__ sinT, int table_rows) {
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long group = gid >> 3;  // (row, which in {q,k}, head)
  const int g = (int)(gid & 7);
  const long long total = (long long)rows * 2 * H;
  const bool active = group < total;
  long long row = 0;
  int which = 0, head = 0;
  if (active) {
    row = group / (2 * H);
    const int rem = (int)(group % (2 * H));
    which = rem / H;
    head = rem % H;
  }
  __nv_bfloat16* p = qkv + row * ld + (size_t)which * H * 64 + head * 64 + g * 8;
  float f[8];
  if (active) {
    unpack8(*reinterpret_cast<const uint4*>(p), f);
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = 0.f;
  }
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) s += f[j];
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  s += __shfl_xor_sync(0xffffffffu, s, 4);
  const float mean = s * (1.f / 64.f);
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float d = f[j] - mean;
    q += d * d;
  }
  q += __shfl_xor_sync(0xffffffffu, q, 1);
  q += __shfl_xor_sync(0xffffffffu, q, 2);
  q += __shfl_xor_sync(0xffffffffu, q, 4);
  const float rstd = rsqrtf(q * (1.f / 64.f) + eps);
  const float* w = which ? kw : qw;
  const float* b = which ? kb : qb;
  float y[8], ww[8], bb[8];
  load8_f32(w + g * 8, ww);
  load8_f32(b + g * 8, bb);
#pragma unroll
  for (int j = 0; j < 8; ++j) y[j] = (f[j] - mean) * rstd * ww[j] + bb[j];
  float part[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) part[j] = __shfl_xor_sync(0xffffffffu, y[j], 2);
  if (active) {
    float cc[8], ss[8];
    const long long trow = (int)row % table_rows;    // row < rows (int): 32-bit modulo
    load8_f32(cosT + trow * 64 + g * 8, cc);
    load8_f32(sinT + trow * 64 + g * 8, ss);
    const float sign = (g & 2) ? 1.f : -1.f;
    float o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = y[j] * cc[j] + sign * part[j] * ss[j];
    *reinterpret_cast<uint4*>(p) = pack8(o);
  }
}

// latents <- bf16( latents + bf16( bf16( neg + bf16( s * bf16(pos - neg) ) ) * dsigma ) )
__global__ void cfg_euler_kernel(__nv_bfloat16* __restrict__ lat, const __nv_bfloat16* __restrict__ pos,
                                 const __nv_bfloat16* __restrict__ neg, long long n, float cfg, float dsigma) {
  long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8;
  if (i + 8 <= n) {
    float a[8], p[8], q[8];
    unpack8(*reinterpret_cast<const uint4*>(lat + i), a);
    unpack8(*reinterpret_cast<const uint4*>(pos + i), p);
    unpack8(*reinterpret_cast<const uint4*>(neg + i), q);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float pred = bf16_round(q[j] + bf16_round(cfg * bf16_round(p[j] - q[j])));
      a[j] = a[j] + bf16_round(pred * dsigma);
    }
    *reinterpret_cast<uint4*>(lat + i) = pack8(a);
  } else {
    for (; i < n; ++i) {
      const float p = __bfloat162float(pos[i]), q = __bfloat162float(neg[i]);
      const float pred = bf16_round(q + bf16_round(cfg * bf16_round(p - q)));
      lat[i] = __float2bfloat16_rn(__bfloat162float(lat[i]) + bf16_round(pred * dsigma));
    }
  }
}

int g_row_ctas_per_sm = 0;   // 0 = as many as fit (occupancy query per kernel); n > 0 forces n (fwb_rowwise_set_ctas_per_sm, A/B only)

// Grid of a persistent row kernel: (resident CTAs per SM) x #SMs — exactly one wave, so no CTA waits for a slot and the rows are dealt
// evenly (measured: a grid of 8 CTAs/SM when only 6 fit costs +27 %) — and never more than one CTA per row.
template <auto Kernel>
inline int row_grid(int rows) {
  static int occ[64] = {0};                       // per kernel instantiation and device ordinal
  int per_sm = g_row_ctas_per_sm;
  if (per_sm <= 0) {
    const int dev = current_device();
    int* slot = (dev >= 0 && dev < 64) ? &occ[dev] : nullptr;
    if (slot && *slot > 0) {
      per_sm = *slot;
    } else {
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, Kernel, kRowThreads, 0) != cudaSuccess || per_sm <= 0) per_sm = 4;
      if (slot) *slot = per_sm;
    }
  }
  const long long g = (long long)(num_sms() > 0 ? num_sms() : 148) * per_sm;
  return (int)(g < rows ? g : rows);
}

}  // namespace

extern "C" int fwb_rowwise_set_ctas_per_sm(int n) {
  FWB_CHECK(n >= 0 && n <= 16, "rowwise_set_ctas_per_sm: 0 (automatic) or 1..16");
  g_row_ctas_per_sm = n;
  return FWB_OK;
}

extern "C" int fwb_ln_modulate(const void* x, int x_dtype, int64_t ldx, int rows, int C, float eps, const float* w,
                               const float* b, const float* mul, const float* add, void* out, int64_t ldo,
                               cudaStream_t stream) {
  FWB_CHECK(x && out, "ln_modulate: null pointer");
  FWB_CHECK(rows > 0 && C > 0, "ln_modulate: empty problem rows=%d C=%d", rows, C);
  FWB_CHECK(C % 8 == 0 && C <= 5120, "ln_modulate: C=%d must be a multiple of 8 and <= 5120", C);
  FWB_CHECK(ldx % 8 == 0 && ldo % 8 == 0, "ln_modulate: leading dims must be multiples of 8");
  FWB_CHECK((w == nullptr) == (b == nullptr), "ln_modulate: affine weight and bias must come together");
  const int chunks = (C / 8 + kRowThreads - 1) / kRowThreads;
  const bool f32 = x_dtype == FWB_DT_F32;
  __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out);
#define LAUNCH(CH)                                                                                                \
  do {                                                                                                            \
    if (f32)                                                                                                      \
      ln_modulate_kernel<CH, true><<<row_grid<ln_modulate_kernel<CH, true>>(rows), kRowThreads, 0, stream>>>(     \
          x, ldx, rows, C, eps, w, b, mul, add, o, ldo);                                                          \
    else                                                                                                          \
      ln_modulate_kernel<CH, false><<<row_grid<ln_modulate_kernel<CH, false>>(rows), kRowThreads, 0, stream>>>(   \
          x, ldx, rows, C, eps, w, b, mul, add, o, ldo);                                                          \
  } while (0)
  if (chunks <= 1) LAUNCH(1);
  else if (chunks <= 2) LAUNCH(2);
  else LAUNCH(5);
#undef LAUNCH
  FWB_CUDA(cudaGetLastError());
  return FWB_OK;
}

extern "C" int fwb_rmsnorm_rope_periodic(void* x, int64_t ldx, int rows, int C, const float* w, float eps, const float* cos_sin,
                                         int table_rows, int head_dim, cudaStream_t stream) {
  FWB_CHECK(x, "rmsnorm_rope: null pointer");
  FWB_CHECK(rows > 0 && C > 0, "rmsnorm_rope: empty problem");
  FWB_CHECK(C % 8 == 0 && C <= 5120 && ldx % 8 == 0, "rmsnorm_rope: C=%d must be a multiple of 8 and <= 5120", C);
  FWB_CHECK(!cos_sin || (head_dim > 0 && head_dim % 8 == 0 && C % head_dim == 0), "rmsnorm_rope: bad head_dim %d", head_dim);
  FWB_CHECK(!cos_sin || (table_rows > 0 && rows % table_rows == 0),
            "rmsnorm_rope: table_rows=%d must divide rows=%d", table_rows, rows);
  if (!cos_sin) table_rows = 1;
  const int chunks = (C / 8 + kRowThreads - 1) / kRowThreads;
  __nv_bfloat16* xp = reinterpret_cast<__nv_bfloat16*>(x);
  const float2* cs = reinterpret_cast<const float2*>(cos_sin);
  if (chunks <= 1) rmsnorm_rope_kernel<1><<<row_grid<rmsnorm_rope_kernel<1>>(rows), kRowThreads, 0, stream>>>(xp, ldx, rows, C, w, eps, cs, table_rows, head_dim);
  else if (chunks <= 2) rmsnorm_rope_kernel<2><<<row_grid<rmsnorm_rope_kernel<2>>(rows), kRowThreads, 0, stream>>>(xp, ldx, rows, C, w, eps, cs, table_rows, head_dim);
  else rmsnorm_rope_kernel<5><<<row_grid<rmsnorm_rope_kernel<5>>(rows), kRowThreads, 0, stream>>>(xp, ldx, rows, C, w, eps, cs, table_rows, head_dim);
  FWB_CUDA(cudaGetLastError());
  return FWB_OK;
}

extern "C" int fwb_rmsnorm_rope(void* x, int64_t ldx, int rows, int C, const float* w, float eps, const float* cos_sin,
                                int head_dim, cudaStream_t stream) {
  return fwb_rmsnorm_rope_periodic(x, ldx, rows, C, w, eps, cos_sin, rows, head_dim, stream);
}

extern "C" int fwb_ln64_rope2d_periodic(void* qkv, int64_t ld, int rows, int H, float eps, const float* qw, const float* qb,
                                        const float* kw, const float* kb, const float* cosT, const float* sinT, int table_rows,
                                        cudaStream_t stream) {
  FWB_CHECK(qkv && qw && qb && kw && kb && cosT && sinT, "ln64_rope2d: null pointer");
  FWB_CHECK(rows > 0 && H > 0 && ld % 8 == 0 && ld >= 3LL * H * 64, "ln64_rope2d: bad shape rows=%d H=%d ld=%lld", rows, H, (long long)ld);
  FWB_CHECK(table_rows > 0 && rows % table_rows == 0, "ln64_rope2d: table_rows=%d must divide rows=%d", table_rows, rows);
  const long long threads = (long long)rows * 2 * H * 8;
  const long long blocks = (threads + 255) / 256;
  FWB_CHECK(blocks < 2147483647LL, "ln64_rope2d: too many rows");
  ln64_rope2d_kernel<<<(unsigned)blocks, 256, 0, stream>>>(reinterpret_cast<__nv_bfloat16*>(qkv), ld, rows, H, eps, qw, qb,
                                                         kw, kb, cosT, sinT, table_rows);
  FWB_CUDA(cudaGetLastError());
  return FWB_OK;
}

extern "C" int fwb_ln64_rope2d(void* qkv, int64_t ld, int rows, int H, float eps, const float* qw, const float* qb,
                               const float* kw, const float* kb, const float* cosT, const float* sinT,
                               cudaStream_t stream) {
  return fwb_ln64_rope2d_periodic(qkv, ld, rows, H, eps, qw, qb, kw, kb, cosT, sinT, rows, stream);
}

extern "C" int fwb_cfg_euler_step(void* latents, const void* pred_pos, const void* pred_neg, int64_t n, float cfg_scale,
                                  float dsigma, cudaStream_t stream) {
  FWB_CHECK(latents && pred_pos && pred_neg && n > 0, "cfg_euler_step: bad arguments");
  const long long blocks = ((n + 7) / 8 + 255) / 256;
  cfg_euler_kernel<<<(unsigned)blocks, 256, 0, stream>>>(reinterpret_cast<__nv_bfloat16*>(latents),
                                                       reinterpret_cast<const __nv_bfloat16*>(pred_pos),
                                                       reinterpret_cast<const __nv_bfloat16*>(pred_neg), n, cfg_scale,
                                                       dsigma);
  FWB_CUDA(cudaGetLastError());
  return FWB_OK;
}
