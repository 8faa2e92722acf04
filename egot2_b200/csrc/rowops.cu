// rowops.cu — HBM-bound row-wise kernels: LayerNorm fwd/bwd, token pooling, column reductions,
// dropout, casts, Adam, token-table helpers, SlowFast map pooling.
// One warp owns one row of H (H = 32*NPL, NPL in {1,2,4,8,16,32,64}); all statistics in fp32.
// Loads/stores are coalesced (lane-strided columns); grids are sized to a multiple of the SM count.
#include <math.h>

#include <stdlib.h>
#define EGOT2_FILE_ID 1
#include "ops.h"

namespace egot2 {

namespace {

constexpr int kWarpsPerCta = 8;

inline int row_grid(int rows) {
  int ctas = (rows + kWarpsPerCta - 1) / kWarpsPerCta;
  int cap = sm_count() * 8;
  return ctas < cap ? (ctas > 0 ? ctas : 1) : cap;
}

// ------------------------------------------------------------------ LayerNorm forward
template <typename TX, typename TY, int NPL>
__global__ void __launch_bounds__(kWarpsPerCta * 32) ln_fwd_kernel(const LayerNormArgs a) {
  EGOT2_PDL_ENTER();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int H = NPL * 32;
  const float inv_keep = a.p_drop > 0.f ? 1.f / (1.f - a.p_drop) : 1.f;
  float g[NPL], b[NPL];
#pragma unroll
  for (int i = 0; i < NPL; ++i) { g[i] = a.g[lane + 32 * i]; b[i] = a.b[lane + 32 * i]; }
  for (int row = blockIdx.x * kWarpsPerCta + warp; row < a.rows; row += gridDim.x * kWarpsPerCta) {
    const TX* x = (const TX*)a.x + (size_t)row * H;
    float v[NPL], s = 0.f;
#pragma unroll
    for (int i = 0; i < NPL; ++i) { v[i] = to_f32(x[lane + 32 * i]); s += v[i]; }
    const float mean = warp_sum(s) * (1.f / H);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NPL; ++i) { const float d = v[i] - mean; q += d * d; }
    const float rstd = rsqrtf(warp_sum(q) * (1.f / H) + a.eps);
    if (a.stat && lane == 0) { a.stat[2 * (size_t)row] = mean; a.stat[2 * (size_t)row + 1] = rstd; }
    const float* tab = a.table ? a.table + (size_t)(row % a.table_rows) * H : nullptr;
    TY* y = (TY*)a.y + (size_t)row * H;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      float o = (v[i] - mean) * rstd * g[i] + b[i];
      if (tab) o += tab[c];
      if (a.p_drop > 0.f) o *= drop_scale(a.drop_key ^ egot2_ep, (uint64_t)row * H + c, a.p_drop, inv_keep);
      y[c] = from_f32<TY>(o);
    }
  }
}

// ------------------------------------------------------------------ LayerNorm backward
template <typename TX, typename TDY, typename TDX, typename TR, int NPL>
__global__ void __launch_bounds__(kWarpsPerCta * 32) ln_bwd_kernel(const LayerNormBwdArgs a) {
  EGOT2_PDL_ENTER();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int H = NPL * 32;
  __shared__ float sdg[NPL * 32], sdb[NPL * 32];
  for (int i = threadIdx.x; i < H; i += blockDim.x) { sdg[i] = 0.f; sdb[i] = 0.f; }
  __syncthreads();
  float g[NPL], dg[NPL], db[NPL];
#pragma unroll
  for (int i = 0; i < NPL; ++i) { g[i] = a.g[lane + 32 * i]; dg[i] = 0.f; db[i] = 0.f; }
  for (int row = blockIdx.x * kWarpsPerCta + warp; row < a.rows; row += gridDim.x * kWarpsPerCta) {
    const TX* x = (const TX*)a.x + (size_t)row * H;
    const TDY* dy = (const TDY*)a.dy + (size_t)row * H;
    const float mean = a.stat[2 * (size_t)row], rstd = a.stat[2 * (size_t)row + 1];
    float xh[NPL], dyg[NPL], s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      const float d = to_f32(dy[c]);
      xh[i] = (to_f32(x[c]) - mean) * rstd;
      dyg[i] = d * g[i];
      dg[i] += d * xh[i];
      db[i] += d;
      s1 += dyg[i];
      s2 += dyg[i] * xh[i];
    }
    s1 = warp_sum(s1) * (1.f / H);
    s2 = warp_sum(s2) * (1.f / H);
    TDX* dx = (TDX*)a.dx + (size_t)row * H;
    const TR* dres = a.dres ? (const TR*)a.dres + (size_t)row * H : nullptr;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      float o = rstd * (dyg[i] - s1 - xh[i] * s2);
      if (dres) o += to_f32(dres[c]);
      dx[c] = from_f32<TDX>(o);
    }
  }
  if (a.dg) {
#pragma unroll
    for (int i = 0; i < NPL; ++i) { atomicAdd(&sdg[lane + 32 * i], dg[i]); atomicAdd(&sdb[lane + 32 * i], db[i]); }
    __syncthreads();
    for (int i = threadIdx.x; i < H; i += blockDim.x) { atomicAdd(a.dg + i, sdg[i]); atomicAdd(a.db + i, sdb[i]); }
  }
}

// ------------------------------------------------------------------ misc elementwise / reductions
__device__ __forceinline__ float* seg_target(const SegOut& so, int t) {
  int seg = 0, d = t;
  while (seg < so.n - 1 && d >= so.tokens[seg]) { d -= so.tokens[seg]; ++seg; }
  return seg < so.n ? so.out[seg] : nullptr;
}
template <typename TT>
__global__ void table_grad_kernel(int B, int T, int H, int clips_per_cta, const TT* __restrict__ dy,
                                  float* __restrict__ dtable, const SegOut so, float p_drop, uint64_t drop_key) {
  EGOT2_PDL_ENTER();
  // CTA (t, chunk): sums its chunk of clips for token t, then one atomic per column
  const int t = blockIdx.x;
  const int b0 = blockIdx.y * clips_per_cta, b1 = min(B, b0 + clips_per_cta);
  float* seg_out = seg_target(so, t);
  for (int c = threadIdx.x; c < H; c += blockDim.x) {
    float s = 0.f;
    if (p_drop > 0.f) {       // dy is read BEFORE the embedding dropout's mask was applied: apply it on the fly
      const float inv_keep = 1.f / (1.f - p_drop);
      for (int b = b0; b < b1; ++b) {
        const size_t idx = ((size_t)b * T + t) * H + c;
        s += to_f32(dy[idx]) * drop_scale(drop_key ^ egot2_ep, idx, p_drop, inv_keep);
      }
    } else {
      for (int b = b0; b < b1; ++b) s += to_f32(dy[((size_t)b * T + t) * H + c]);
    }
    if (dtable) atomicAdd(dtable + (size_t)t * H + c, s);
    if (seg_out) atomicAdd(seg_out + c, s);
  }
}
// bf16, H = 8 * LPR with LPR a power of two <= 128: LPR lanes x 16 B cover a token row, the CTA's 128 / LPR lane groups
// stride over the clips (independent 16 B loads), the partial rows meet in shared memory
__global__ void __launch_bounds__(128) table_grad_vec_kernel(int B, int T, int H, int clips_per_cta, const bf16* __restrict__ dy,
                                                             float* __restrict__ dtable, const SegOut so, float p_drop,
                                                             uint64_t drop_key) {
  EGOT2_PDL_ENTER();
  __shared__ float part[1024];
  const int lpr = H >> 3, groups = 128 / lpr;
  const int cg = threadIdx.x % lpr, g = threadIdx.x / lpr;
  const int t = blockIdx.x;
  const int b0 = blockIdx.y * clips_per_cta, b1 = min(B, b0 + clips_per_cta);
  const float inv_keep = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  for (int b = b0 + g; b < b1; b += groups) {
    const size_t idx = ((size_t)b * T + t) * H + cg * 8;
    const uint4 v = *reinterpret_cast<const uint4*>(dy + idx);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    float dm[8];
    if (p_drop > 0.f) drop_scale_n<8>(drop_key ^ egot2_ep, idx, p_drop, inv_keep, dm);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float lo = __uint_as_float(w[k] << 16), hi = __uint_as_float(w[k] & 0xffff0000u);
      if (p_drop > 0.f) { lo *= dm[2 * k]; hi *= dm[2 * k + 1]; }
      acc[2 * k] += lo; acc[2 * k + 1] += hi;
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) part[g * H + cg * 8 + i] = acc[i];
  __syncthreads();
  float* seg_out = seg_target(so, t);
  for (int c = threadIdx.x; c < H; c += 128) {
    float s = 0.f;
    for (int k = 0; k < groups; ++k) s += part[k * H + c];
    if (dtable) atomicAdd(dtable + (size_t)t * H + c, s);
    if (seg_out) atomicAdd(seg_out + c, s);
  }
}

template <typename T> struct Pair;
template <> struct Pair<float> { typedef float2 type; };
template <> struct Pair<bf16> { typedef __nv_bfloat162 type; };
__device__ __forceinline__ float2 pair_f32(float2 v) { return v; }
__device__ __forceinline__ float2 pair_f32(__nv_bfloat162 v) { return __bfloat1622float2(v); }

template <typename T>
__global__ void colsum_kernel(int M, int N, const T* __restrict__ x, int ldx, int rpg, int gstride,
                              float* __restrict__ out, int rows_per_cta) {
  EGOT2_PDL_ENTER();
  // blockDim = (32 column pairs, 8 row lanes): a warp reads 64 consecutive columns of one row per load
  typedef typename Pair<T>::type P2;
  const int n = (blockIdx.x * 32 + threadIdx.x) * 2;
  const int mbeg = blockIdx.y * rows_per_cta, mend = min(M, mbeg + rows_per_cta);
  float s0 = 0.f, s1 = 0.f;
  const bool vec = (n + 1 < N) && ((ldx & 1) == 0) && ((reinterpret_cast<uintptr_t>(x) & (2 * sizeof(T) - 1)) == 0);
  if (n < N) {
    for (int mb = mbeg + threadIdx.y; mb < mend; mb += 32) {
      float2 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int m = mb + 8 * u;
        v[u] = make_float2(0.f, 0.f);
        if (m < mend) {
          const long long r = rpg > 0 ? (long long)(m / rpg) * gstride + (m % rpg) : m;
          if (vec) v[u] = pair_f32(*reinterpret_cast<const P2*>(x + r * ldx + n));
          else { v[u].x = to_f32(x[r * ldx + n]); if (n + 1 < N) v[u].y = to_f32(x[r * ldx + n + 1]); }
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) { s0 += v[u].x; s1 += v[u].y; }
    }
  }
  __shared__ float red[8][65];
  red[threadIdx.y][2 * threadIdx.x] = s0;
  red[threadIdx.y][2 * threadIdx.x + 1] = s1;
  __syncthreads();
  if (threadIdx.y < 2) {
    const int c = 2 * threadIdx.x + threadIdx.y, nn = blockIdx.x * 64 + c;
    if (nn < N) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) t += red[i][c];
      atomicAdd(out + nn, t);
    }
  }
}

// fp32 (M, N) -> bf16 copy AND column sums in one pass (the decoder's attention gradients arrive in fp32 because several
// queries add into the same key rows; the GEMMs behind them want bf16, the bias gradient wants the column sums): N even,
// both row pitches even.  Same block shape and summation order as colsum_kernel<float>.
__global__ void colsum_cast_kernel(int M, int N, const float* __restrict__ x, int ldx, bf16* __restrict__ y, int ldy,
                                   float* __restrict__ out, int rows_per_cta) {
  EGOT2_PDL_ENTER();
  const int n = (blockIdx.x * 32 + threadIdx.x) * 2;
  const int mbeg = blockIdx.y * rows_per_cta, mend = min(M, mbeg + rows_per_cta);
  float s0 = 0.f, s1 = 0.f;
  if (n < N) {
    for (int mb = mbeg + threadIdx.y; mb < mend; mb += 32) {
      float2 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int m = mb + 8 * u;
        v[u] = make_float2(0.f, 0.f);
        if (m < mend) {
          v[u] = *reinterpret_cast<const float2*>(x + (size_t)m * ldx + n);
          *reinterpret_cast<__nv_bfloat162*>(y + (size_t)m * ldy + n) = __floats2bfloat162_rn(v[u].x, v[u].y);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) { s0 += v[u].x; s1 += v[u].y; }
    }
  }
  __shared__ float red[8][65];
  red[threadIdx.y][2 * threadIdx.x] = s0;
  red[threadIdx.y][2 * threadIdx.x + 1] = s1;
  __syncthreads();
  if (threadIdx.y < 2) {
    const int c = 2 * threadIdx.x + threadIdx.y, nn = blockIdx.x * 64 + c;
    if (nn < N) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) t += red[i][c];
      atomicAdd(out + nn, t);
    }
  }
}

// bf16 fast path: 128-bit loads, CW = 8 * lanes_per_row columns per CTA (N % 8 == 0, 16 B-aligned rows)
__global__ void __launch_bounds__(256) colsum_bf16_vec_kernel(int M, int N, const bf16* __restrict__ x, int ldx, int rpg,
                                                              int gstride, float* __restrict__ out, int rows_per_cta,
                                                              int lanes_per_row) {
  EGOT2_PDL_ENTER();
  const int cg = threadIdx.x % lanes_per_row, rl = threadIdx.x / lanes_per_row, nrl = 256 / lanes_per_row;
  const int n = (blockIdx.x * lanes_per_row + cg) * 8;
  const int mbeg = blockIdx.y * rows_per_cta, mend = min(M, mbeg + rows_per_cta);
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  if (n < N) {
    for (int m0 = mbeg + rl; m0 < mend; m0 += 4 * nrl) {
      uint4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int m = m0 + u * nrl;
        v[u] = make_uint4(0u, 0u, 0u, 0u);
        if (m < mend) {
          const long long r = rpg > 0 ? (long long)(m / rpg) * gstride + (m % rpg) : m;
          v[u] = __ldg(reinterpret_cast<const uint4*>(x + r * ldx + n));
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t w[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          acc[2 * k] += __uint_as_float(w[k] << 16);
          acc[2 * k + 1] += __uint_as_float(w[k] & 0xffff0000u);
        }
      }
    }
  }
  __shared__ float red[256 * 8];
#pragma unroll
  for (int i = 0; i < 8; ++i) red[(rl * lanes_per_row + cg) * 8 + i] = acc[i];
  __syncthreads();
  const int cw = lanes_per_row * 8;
  for (int c = threadIdx.x; c < cw; c += 256) {
    float t = 0.f;
    for (int r = 0; r < nrl; ++r) t += red[r * cw + c];
    const int nn = blockIdx.x * cw + c;
    if (nn < N) atomicAdd(out + nn, t);
  }
}

template <typename T>
__global__ void dropout_kernel(T* x, size_t n, float p, float inv_keep, uint64_t key) {
  EGOT2_PDL_ENTER();
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    x[i] = from_f32<T>(to_f32(x[i]) * drop_scale(key ^ egot2_ep, i, p, inv_keep));
}

template <typename TT>
__global__ void pool_fwd_kernel(int B, int T, int H, int pool, int row_tokens, const TT* __restrict__ x,
                                float* __restrict__ pooled) {
  EGOT2_PDL_ENTER();
  if (pool) {
    const int b = blockIdx.x;
    for (int c = threadIdx.x; c < H; c += blockDim.x) {
      float s = 0.f;
      for (int t = 0; t < T; ++t) s += to_f32(x[((size_t)b * T + t) * H + c]);
      pooled[(size_t)b * H + c] = s / (float)T;
    }
  } else {
    const int r = blockIdx.x, b = r / row_tokens, t = r % row_tokens;
    for (int c = threadIdx.x; c < H; c += blockDim.x)
      pooled[(size_t)r * H + c] = to_f32(x[((size_t)b * T + t) * H + c]);
  }
}

template <typename TT>
__global__ void pool_bwd_kernel(int B, int T, int H, int pool, int row_tokens, const float* __restrict__ dpooled,
                                TT* __restrict__ dx) {
  EGOT2_PDL_ENTER();
  const int r = blockIdx.x, b = r / T, t = r % T;     // one CTA per token row of dx
  for (int c = threadIdx.x; c < H; c += blockDim.x) {
    float v;
    if (pool) v = dpooled[(size_t)b * H + c] / (float)T;
    else v = t < row_tokens ? dpooled[((size_t)b * row_tokens + t) * H + c] : 0.f;
    dx[(size_t)r * H + c] = from_f32<TT>(v);
  }
}

__global__ void cast_to_bf16_kernel(const float* __restrict__ s, bf16* __restrict__ d, size_t n) {
  EGOT2_PDL_ENTER();
  size_t i = (blockIdx.x * (size_t)blockDim.x + threadIdx.x) * 4;
  const size_t stride = (size_t)gridDim.x * blockDim.x * 4;
  for (; i + 3 < n; i += stride) {
    const float4 v = *reinterpret_cast<const float4*>(s + i);
    __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 o; o.x = *reinterpret_cast<uint32_t*>(&lo); o.y = *reinterpret_cast<uint32_t*>(&hi);
    *reinterpret_cast<uint2*>(d + i) = o;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0)
    for (size_t j = n & ~(size_t)3; j < n; ++j) d[j] = __float2bfloat16_rn(s[j]);
}
__global__ void cast_rows_kernel(const float* __restrict__ s, int rows, int n, bf16* __restrict__ d, int ld) {
  EGOT2_PDL_ENTER();
  const size_t total = (size_t)rows * ld;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t r = i / ld; const int c = (int)(i % ld);
    d[i] = c < n ? __float2bfloat16_rn(s[r * n + c]) : __float2bfloat16_rn(0.f);
  }
}
__global__ void cast_to_f32_kernel(const bf16* __restrict__ s, float* __restrict__ d, size_t n) {
  EGOT2_PDL_ENTER();
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    d[i] = __bfloat162float(s[i]);
}
__global__ void copy_f32_kernel(const float* __restrict__ s, float* __restrict__ d, size_t n) {
  EGOT2_PDL_ENTER();
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) d[i] = s[i];
}
__global__ void zero_kernel(float* p, size_t n) {
  EGOT2_PDL_ENTER();
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = 0.f;
}

// DECOUPLED = torch.optim.AdamW: the weight decay scales the parameter (p *= 1 - lr*wd) instead of joining the gradient
template <bool DECOUPLED>
__global__ void adam_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, size_t n, float lr, float b1, float b2, float eps, float wd,
                            float bc1, float bc2_sqrt, float gscale, bf16* __restrict__ shadow, int zero_grad,
                            const int32_t* __restrict__ step_dev, const float* __restrict__ lr_dev,
                            const egot2_grad_guard* __restrict__ guard) {
  EGOT2_PDL_ENTER();
  if (guard) {               // egot2_grad_norm ran before: clip, or skip the update and only clear the gradient
    if (guard->skip) {
      if (zero_grad)
        for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) g[i] = 0.f;
      return;
    }
    gscale *= guard->coef;
  }
  if (step_dev) {            // step count kept on the device (whole-step CUDA graphs): bias corrections computed here
    const float t = (float)*step_dev;
    bc1 = 1.f - powf(b1, t);
    bc2_sqrt = sqrtf(1.f - powf(b2, t));
  }
  if (lr_dev) lr = *lr_dev;  // learning-rate schedule evaluated on the device (egot2_opt_advance)
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float grad = g[i] * gscale;
    float w = p[i];
    if (DECOUPLED) w *= 1.f - lr * wd;
    else if (wd != 0.f) grad += wd * w;
    const float mi = b1 * m[i] + (1.f - b1) * grad;
    const float vi = b2 * v[i] + (1.f - b2) * grad * grad;
    m[i] = mi; v[i] = vi;
    // torch.optim.Adam: denom = sqrt(v)/sqrt(bias_correction2) + eps ; step = lr / bias_correction1
    const float wn = w - (lr / bc1) * mi / (sqrtf(vi) / bc2_sqrt + eps);
    p[i] = wn;
    if (shadow) shadow[i] = __float2bfloat16_rn(wn);     // the bf16 copy the next forward's GEMMs read
    if (zero_grad) g[i] = 0.f;                           // the next backward accumulates into a clean arena
  }
}

// lr_at of include/egot2.h, without the warm-up
__device__ double lr_policy(const egot2_lr_sched& s, long long t) {
  if (s.kind == EGOT2_LR_COSINE) {
    if (t >= s.total_steps) return s.end_lr;
    return s.end_lr + (s.base_lr - s.end_lr) * (1.0 + cos(M_PI * (double)t / (double)s.total_steps)) * 0.5;
  }
  if (s.kind == EGOT2_LR_STEPS) {
    int i = 0;
    while (i < s.n_milestones && i < 8 && s.milestones[i] <= t) ++i;
    return s.base_lr * s.factors[i];
  }
  return s.base_lr;
}
__global__ void opt_advance_kernel(int32_t* __restrict__ step, const egot2_lr_sched* __restrict__ sched, float* __restrict__ lr) {
  EGOT2_PDL_ENTER();
  const egot2_lr_sched s = *sched;
  const int32_t t = *step + 1;
  const long long k = t - 1;           // lr of optimizer step t = lr_at(t - 1)
  double v;
  if (k < s.warmup_steps) {
    const double w0 = s.warmup_start_lr;
    v = w0 + (lr_policy(s, s.warmup_steps) - w0) * (double)k / (double)s.warmup_steps;
  } else {
    v = lr_policy(s, k);
  }
  *step = t;
  *lr = (float)v;
}

// egot2_grad_norm: a fixed grid (not sm_count-dependent, so every GPU adds in the same order), fp64 squares per thread in
// index order, a fixed-order CTA sum, and the last CTA to finish adds the per-CTA sums in CTA order.
constexpr int kNormCtas = 512, kNormThreads = 256;
__global__ void __launch_bounds__(kNormThreads) grad_norm_kernel(const float* __restrict__ g, size_t n, float scale,
                                                                 egot2_grad_guard* __restrict__ guard, int32_t* step_dev,
                                                                 double* part, unsigned int* ctr) {
  EGOT2_PDL_ENTER();
  __shared__ double sh[kNormThreads / 32];
  __shared__ unsigned int s_last;
  const size_t tid = blockIdx.x * (size_t)kNormThreads + threadIdx.x, stride = (size_t)kNormCtas * kNormThreads;
  double s = 0.0;
  size_t tail = 0;
  if ((reinterpret_cast<uintptr_t>(g) & 15) == 0) {
    const float4* g4 = reinterpret_cast<const float4*>(g);
    const size_t n4 = n / 4;
    constexpr int U = 4;                 // independent loads in flight per thread
    for (size_t q = tid; q < n4; q += stride * U) {
      float4 x[U];
#pragma unroll
      for (int u = 0; u < U; ++u) x[u] = q + u * stride < n4 ? g4[q + u * stride] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        s += (double)x[u].x * x[u].x; s += (double)x[u].y * x[u].y;
        s += (double)x[u].z * x[u].z; s += (double)x[u].w * x[u].w;
      }
    }
    tail = n4 * 4;
  }
  for (size_t i = tail + tid; i < n; i += stride) s += (double)g[i] * g[i];
  s = block_sum_f64(s, sh);
  if (threadIdx.x == 0) {
    part[blockIdx.x] = s;
    __threadfence();
    s_last = atomicAdd(ctr, 1u) == kNormCtas - 1 ? 1u : 0u;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();                       // every CTA's fenced partial is visible to the last one
  double t = 0.0;
  for (int c = threadIdx.x; c < kNormCtas; c += kNormThreads) t += reinterpret_cast<volatile double*>(part)[c];
  t = block_sum_f64(t, sh);
  if (threadIdx.x == 0) {
    grad_guard_finalize(t, scale, guard, step_dev);
    *ctr = 0;                            // ready for the next launch (graph replays)
  }
}

struct SegList { int n; int tokens[EGOT2_MAX_SEG]; int task[EGOT2_MAX_SEG]; };

__global__ void hhi_tok_table_fwd_kernel(const float* __restrict__ task_embed, const float* __restrict__ pe,
                                         SegList s, int H, float* __restrict__ table) {
  EGOT2_PDL_ENTER();
  // one CTA per token; d restarts at 0 for every task (PositionalEncoding applied per task before the concat)
  int t = blockIdx.x, seg = 0, d = t;
  while (seg < s.n - 1 && d >= s.tokens[seg]) { d -= s.tokens[seg]; ++seg; }
  for (int c = threadIdx.x; c < H; c += blockDim.x)
    table[(size_t)t * H + c] = task_embed[(size_t)s.task[seg] * H + c] + pe[(size_t)d * H + c];
}
__global__ void hhi_tok_table_bwd_kernel(const float* __restrict__ dtable, SegList s, int H,
                                         float* __restrict__ d_task_embed) {
  EGOT2_PDL_ENTER();
  // one CTA per segment: d_task_embed[task] += sum over the segment's tokens
  const int seg = blockIdx.x;
  int off = 0;
  for (int i = 0; i < seg; ++i) off += s.tokens[i];
  for (int c = threadIdx.x; c < H; c += blockDim.x) {
    float acc = 0.f;
    for (int d = 0; d < s.tokens[seg]; ++d) acc += dtable[(size_t)(off + d) * H + c];
    atomicAdd(d_task_embed + (size_t)s.task[seg] * H + c, acc);
  }
}

// AdaptiveAvgPool3d((Tout,1,1)) + permute: in (B,C,Tin,hw) -> out (B,Tout,C).  One warp per (b,c,to):
// the Tin/Tout*hw contiguous elements are read coalesced.
template <typename TI, typename TO>
__global__ void slowfast_pool_kernel(const TI* __restrict__ in, int B, int C, int Tin, int hw, int Tout,
                                     TO* __restrict__ out) {
  EGOT2_PDL_ENTER();
  const int lane = threadIdx.x & 31;
  const size_t warp = (blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5;
  const size_t total = (size_t)B * C * Tout;
  if (warp >= total) return;
  const int to = warp % Tout;
  const int c = (warp / Tout) % C;
  const int b = warp / ((size_t)Tout * C);
  const int win = Tin / Tout, n = win * hw;
  const TI* src = in + (((size_t)b * C + c) * Tin + (size_t)to * win) * hw;
  float s = 0.f;
  for (int i = lane; i < n; i += 32) s += to_f32(src[i]);
  s = warp_sum(s);
  if (lane == 0) out[((size_t)b * Tout + to) * C + c] = from_f32<TO>(s / (float)n);
}


// ------------------------------------------------------------------ bf16 vector LayerNorm (H in {128,256,512,1024})
// A row is read with 128-bit loads: LPR = min(32, H/8) lanes cover one 256-column segment, so a warp holds 32/LPR rows.
template <int HH> struct LnVec {
  static constexpr int LPR = HH / 8 < 32 ? HH / 8 : 32;      // lanes per row
  static constexpr int RPW = 32 / LPR;                        // rows per warp
  static constexpr int SEG = HH / (LPR * 8);                  // 8-column segments per lane
};
__device__ __forceinline__ void unpack8(const uint4& v, float (&o)[8]) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int k = 0; k < 4; ++k) { o[2 * k] = __uint_as_float(w[k] << 16); o[2 * k + 1] = __uint_as_float(w[k] & 0xffff0000u); }
}
__device__ __forceinline__ uint4 pack8(const float (&v)[8]) {
  uint4 o;
  __nv_bfloat162 p0 = __floats2bfloat162_rn(v[0], v[1]), p1 = __floats2bfloat162_rn(v[2], v[3]);
  __nv_bfloat162 p2 = __floats2bfloat162_rn(v[4], v[5]), p3 = __floats2bfloat162_rn(v[6], v[7]);
  o.x = *reinterpret_cast<uint32_t*>(&p0); o.y = *reinterpret_cast<uint32_t*>(&p1);
  o.z = *reinterpret_cast<uint32_t*>(&p2); o.w = *reinterpret_cast<uint32_t*>(&p3);
  return o;
}
template <int LPR> __device__ __forceinline__ float row_sum(float v) {
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int HH>
__global__ void __launch_bounds__(256) ln_fwd_vec_kernel(const LayerNormArgs a) {
  EGOT2_PDL_ENTER();
  typedef LnVec<HH> V;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane / V::LPR, cl = lane % V::LPR;
  const float inv_keep = a.p_drop > 0.f ? 1.f / (1.f - a.p_drop) : 1.f;
  float g[V::SEG][8], b[V::SEG][8];
#pragma unroll
  for (int s = 0; s < V::SEG; ++s)
#pragma unroll
    for (int i = 0; i < 8; ++i) { const int c = (s * V::LPR + cl) * 8 + i; g[s][i] = a.g[c]; b[s][i] = a.b[c]; }
  const int rows_per_iter = gridDim.x * 8 * V::RPW;
  // the loop bound is warp-uniform (row0); a warp's last sub-row may be past the end: it computes on zeros and stores nothing.
  // The next iteration's row is requested before this one is processed (a warp only walks a few rows; without the
  // prefetch every iteration starts with an exposed global-load round trip).
  int row0 = (blockIdx.x * 8 + warp) * V::RPW;
  uint4 xq[V::SEG];
  if (row0 < a.rows) {
    const bf16* x = (const bf16*)a.x + (size_t)(row0 + sub < a.rows ? row0 + sub : row0) * HH;
#pragma unroll
    for (int s = 0; s < V::SEG; ++s) xq[s] = __ldg(reinterpret_cast<const uint4*>(x) + s * V::LPR + cl);
  }
  for (; row0 < a.rows; row0 += rows_per_iter) {
    const int row = row0 + sub;
    const bool valid = row < a.rows;
    float v[V::SEG][8], sum = 0.f;
#pragma unroll
    for (int s = 0; s < V::SEG; ++s) {
      unpack8(xq[s], v[s]);
#pragma unroll
      for (int i = 0; i < 8; ++i) sum += v[s][i];
    }
    if (row0 + rows_per_iter < a.rows) {
      const int rn = row0 + rows_per_iter;
      const bf16* x = (const bf16*)a.x + (size_t)(rn + sub < a.rows ? rn + sub : rn) * HH;
#pragma unroll
      for (int s = 0; s < V::SEG; ++s) xq[s] = __ldg(reinterpret_cast<const uint4*>(x) + s * V::LPR + cl);
    }
    const float mean = row_sum<V::LPR>(sum) * (1.f / HH);
    float q = 0.f;
#pragma unroll
    for (int s = 0; s < V::SEG; ++s)
#pragma unroll
      for (int i = 0; i < 8; ++i) { const float d = v[s][i] - mean; q += d * d; }
    const float rstd = rsqrtf(row_sum<V::LPR>(q) * (1.f / HH) + a.eps);
    if (!valid) continue;                 // no warp-level operation below this point
    if (a.stat && cl == 0) { a.stat[2 * (size_t)row] = mean; a.stat[2 * (size_t)row + 1] = rstd; }
    const float* tab = a.table ? a.table + (size_t)(row % a.table_rows) * HH : nullptr;
    bf16* y = (bf16*)a.y + (size_t)row * HH;
#pragma unroll
    for (int s = 0; s < V::SEG; ++s) {
      const int c0 = (s * V::LPR + cl) * 8;
      float o[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = (v[s][i] - mean) * rstd * g[s][i] + b[s][i];
      if (tab) {
        const float4 t0 = __ldg(reinterpret_cast<const float4*>(tab + c0)), t1 = __ldg(reinterpret_cast<const float4*>(tab + c0 + 4));
        o[0] += t0.x; o[1] += t0.y; o[2] += t0.z; o[3] += t0.w; o[4] += t1.x; o[5] += t1.y; o[6] += t1.z; o[7] += t1.w;
      }
      if (a.p_drop > 0.f) {
        float dm[8];
        drop_scale_n<8>(a.drop_key ^ egot2_ep, (uint64_t)row * HH + c0, a.p_drop, inv_keep, dm);
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] *= dm[i];
      }
      reinterpret_cast<uint4*>(y)[s * V::LPR + cl] = pack8(o);
    }
  }
}

template <int HH>
__global__ void __launch_bounds__(256) ln_bwd_vec_kernel(const LayerNormBwdArgs a) {
  EGOT2_PDL_ENTER();
  typedef LnVec<HH> V;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane / V::LPR, cl = lane % V::LPR;
  __shared__ float sred[8][2][HH];
  const float dy_keep = a.dy_p_drop > 0.f ? 1.f / (1.f - a.dy_p_drop) : 1.f;
  const float dx2_keep = a.dx2_p_drop > 0.f ? 1.f / (1.f - a.dx2_p_drop) : 1.f;
  float g[V::SEG][8], dg[V::SEG][8], db[V::SEG][8], dcs[V::SEG][8];
#pragma unroll
  for (int s = 0; s < V::SEG; ++s)
#pragma unroll
    for (int i = 0; i < 8; ++i) { g[s][i] = a.g[(s * V::LPR + cl) * 8 + i]; dg[s][i] = 0.f; db[s][i] = 0.f; dcs[s][i] = 0.f; }
  const int rows_per_iter = gridDim.x * 8 * V::RPW;
  // warp-uniform loop bound (row0): a sub-row past the end reads row0 again and contributes nothing
  // x, dy and the row statistics of the NEXT iteration are requested before this one is processed (see ln_fwd_vec_kernel)
  int row0 = (blockIdx.x * 8 + warp) * V::RPW;
  uint4 xq[V::SEG], dq[V::SEG];
  float2 stq = make_float2(0.f, 0.f);
  if (row0 < a.rows) {
    const size_t rr = row0 + sub < a.rows ? row0 + sub : row0;
#pragma unroll
    for (int s = 0; s < V::SEG; ++s) {
      xq[s] = __ldg(reinterpret_cast<const uint4*>((const bf16*)a.x + rr * HH) + s * V::LPR + cl);
      dq[s] = __ldg(reinterpret_cast<const uint4*>((const bf16*)a.dy + rr * HH) + s * V::LPR + cl);
    }
    stq = __ldg(reinterpret_cast<const float2*>(a.stat) + rr);
  }
  for (; row0 < a.rows; row0 += rows_per_iter) {
    const int row = row0 + sub;
    const bool valid = row < a.rows;
    const float mean = stq.x, rstd = stq.y;
    uint4 xc[V::SEG], dc[V::SEG];
#pragma unroll
    for (int s = 0; s < V::SEG; ++s) { xc[s] = xq[s]; dc[s] = dq[s]; }
    if (row0 + rows_per_iter < a.rows) {
      const int rn = row0 + rows_per_iter;
      const size_t rr = rn + sub < a.rows ? rn + sub : rn;
#pragma unroll
      for (int s = 0; s < V::SEG; ++s) {
        xq[s] = __ldg(reinterpret_cast<const uint4*>((const bf16*)a.x + rr * HH) + s * V::LPR + cl);
        dq[s] = __ldg(reinterpret_cast<const uint4*>((const bf16*)a.dy + rr * HH) + s * V::LPR + cl);
      }
      stq = __ldg(reinterpret_cast<const float2*>(a.stat) + rr);
    }
    float xh[V::SEG][8], dyg[V::SEG][8], s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int s = 0; s < V::SEG; ++s) {
      float xv[8], d[8];
      unpack8(xc[s], xv);
      unpack8(dc[s], d);
      const int c0 = (s * V::LPR + cl) * 8;
      if (a.dy_p_drop > 0.f) {
        float dm[8];
        drop_scale_n<8>(a.dy_drop_key ^ egot2_ep, (uint64_t)row * HH + c0, a.dy_p_drop, dy_keep, dm);
#pragma unroll
        for (int i = 0; i < 8; ++i) d[i] *= dm[i];
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (!valid) d[i] = 0.f;
        xh[s][i] = (xv[i] - mean) * rstd;
        dyg[s][i] = d[i] * g[s][i];
        dg[s][i] += d[i] * xh[s][i];
        db[s][i] += d[i];
        s1 += dyg[s][i];
        s2 += dyg[s][i] * xh[s][i];
      }
    }
    s1 = row_sum<V::LPR>(s1) * (1.f / HH);
    s2 = row_sum<V::LPR>(s2) * (1.f / HH);
    if (!valid) continue;                 // no warp-level operation in the rest of the iteration
    uint4* dxp = reinterpret_cast<uint4*>((bf16*)a.dx + (size_t)row * HH);
    const uint4* drp = a.dres ? reinterpret_cast<const uint4*>((const bf16*)a.dres + (size_t)row * HH) : nullptr;
    uint4* dx2p = a.dx2 ? reinterpret_cast<uint4*>((bf16*)a.dx2 + (size_t)row * HH) : nullptr;
#pragma unroll
    for (int s = 0; s < V::SEG; ++s) {
      const int c0 = (s * V::LPR + cl) * 8;
      float o[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = rstd * (dyg[s][i] - s1 - xh[s][i] * s2);
      if (drp) {
        float r8[8];
        unpack8(__ldg(drp + s * V::LPR + cl), r8);
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] += r8[i];
      }
      const uint4 packed = pack8(o);
      dxp[s * V::LPR + cl] = packed;
      if (dx2p) {
        float o2[8];
        unpack8(packed, o2);        // the unfused sequence masks the bf16-rounded dx
        float dm2[8];
        drop_scale_n<8>(a.dx2_drop_key ^ egot2_ep, (uint64_t)row * HH + c0, a.dx2_p_drop, dx2_keep, dm2);
#pragma unroll
        for (int i = 0; i < 8; ++i) o2[i] *= dm2[i];
        const uint4 packed2 = pack8(o2);
        dx2p[s * V::LPR + cl] = packed2;
        if (a.dcol) {               // column sums of what the next Linear's backward sees (the rounded values)
          unpack8(packed2, o2);
#pragma unroll
          for (int i = 0; i < 8; ++i) dcs[s][i] += o2[i];
        }
      } else if (a.dcol) {
        float o1[8];
        unpack8(packed, o1);
#pragma unroll
        for (int i = 0; i < 8; ++i) dcs[s][i] += o1[i];
      }
    }
  }
  if (a.dg) {
    // fold the RPW rows a warp holds side by side, then the 8 warps through shared memory, then one atomic per column
#pragma unroll
    for (int s = 0; s < V::SEG; ++s)
#pragma unroll
      for (int i = 0; i < 8; ++i) {
#pragma unroll
        for (int o = V::LPR; o < 32; o <<= 1) {
          dg[s][i] += __shfl_xor_sync(0xffffffffu, dg[s][i], o);
          db[s][i] += __shfl_xor_sync(0xffffffffu, db[s][i], o);
        }
        if (sub == 0) { sred[warp][0][(s * V::LPR + cl) * 8 + i] = dg[s][i]; sred[warp][1][(s * V::LPR + cl) * 8 + i] = db[s][i]; }
      }
    __syncthreads();
    for (int c = threadIdx.x; c < 2 * HH; c += 256) {
      const int which = c / HH, col = c % HH;
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) t += sred[w][which][col];
      atomicAdd((which ? a.db : a.dg) + col, t);
    }
  }
  if (a.dcol) {
    __syncthreads();                           // sred is reused
#pragma unroll
    for (int s = 0; s < V::SEG; ++s)
#pragma unroll
      for (int i = 0; i < 8; ++i) {
#pragma unroll
        for (int o = V::LPR; o < 32; o <<= 1) dcs[s][i] += __shfl_xor_sync(0xffffffffu, dcs[s][i], o);
        if (sub == 0) sred[warp][0][(s * V::LPR + cl) * 8 + i] = dcs[s][i];
      }
    __syncthreads();
    for (int col = threadIdx.x; col < HH; col += 256) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) t += sred[w][0][col];
      atomicAdd(a.dcol + col, t);
    }
  }
}

template <int HH> int ln_fwd_vec_launch(const LayerNormArgs& a, cudaStream_t st) {
  const int rows_per_cta = 8 * LnVec<HH>::RPW;
  int grid = (a.rows + rows_per_cta - 1) / rows_per_cta;
  static int occ = 0;                         // resident CTAs per SM: the grid is ONE wave of them (grid-stride loop inside)
  if (occ == 0 && (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ln_fwd_vec_kernel<HH>, 256, 0) != cudaSuccess || occ < 1)) occ = 4;
  const int cap = sm_count() * occ;
  if (grid > cap) grid = cap;
  ProfScope prof(st, "ln_fwd rows%d H%d", a.rows, a.H);
  launch(ln_fwd_vec_kernel<HH>, dim3(grid), dim3(256), 0, st, a);
  EGOT2_LAUNCH_CHECK();
  return 0;
}
template <int HH> int ln_bwd_vec_launch(const LayerNormBwdArgs& a, cudaStream_t st) {
  const int rows_per_cta = 8 * LnVec<HH>::RPW;
  int grid = (a.rows + rows_per_cta - 1) / rows_per_cta;
  static int occ = 0;                         // one wave of resident CTAs, at most 4 per SM: every CTA ends with 2H global
  if (occ == 0) {                             // atomics on the same addresses
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ln_bwd_vec_kernel<HH>, 256, 0) != cudaSuccess || occ < 1) occ = 2;
    if (occ > 4) occ = 4;
    if (getenv("EGOT2_LN_BWD_OCC") && atoi(getenv("EGOT2_LN_BWD_OCC")) > 0) occ = atoi(getenv("EGOT2_LN_BWD_OCC"));      // experiments
  }
  const int cap = sm_count() * occ;
  if (grid > cap) grid = cap;
  ProfScope prof(st, "ln_bwd rows%d H%d", a.rows, a.H);
  launch(ln_bwd_vec_kernel<HH>, dim3(grid), dim3(256), 0, st, a);
  EGOT2_LAUNCH_CHECK();
  return 0;
}
inline bool ln_vec_ok(int dtype, int H, const void* p0, const void* p1, const void* p2, const void* p3) {
  auto al = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  return dtype == EGOT2_BF16 && (H == 128 || H == 256 || H == 512 || H == 1024) && al(p0) && al(p1) && al(p2) && al(p3);
}

template <int NPL> int ln_fwd_dispatch(const LayerNormArgs& a, cudaStream_t st) {
  const int grid = row_grid(a.rows);
  ProfScope prof(st, "ln_fwd rows%d H%d", a.rows, a.H);
  if (a.dtype == EGOT2_F32) launch(ln_fwd_kernel<float, float, NPL>, dim3(grid), dim3(kWarpsPerCta * 32), 0, st, a);
  else if (a.x_is_f32) launch(ln_fwd_kernel<float, bf16, NPL>, dim3(grid), dim3(kWarpsPerCta * 32), 0, st, a);
  else launch(ln_fwd_kernel<bf16, bf16, NPL>, dim3(grid), dim3(kWarpsPerCta * 32), 0, st, a);
  EGOT2_LAUNCH_CHECK();
  return 0;
}

template <int NPL> int ln_bwd_dispatch(const LayerNormBwdArgs& a, cudaStream_t st) {
  const int grid = row_grid(a.rows);
  const int nt = kWarpsPerCta * 32;
  ProfScope prof(st, "ln_bwd rows%d H%d", a.rows, a.H);
  if (a.dtype == EGOT2_F32) {
    launch(ln_bwd_kernel<float, float, float, float, NPL>, dim3(grid), dim3(nt), 0, st, a);
  } else {
    // bf16 activations; the pooled-vector LN of the head runs with fp32 x / dy / dx
    if (a.x_is_f32 && a.dy_is_f32 && a.dx_is_f32) launch(ln_bwd_kernel<float, float, float, bf16, NPL>, dim3(grid), dim3(nt), 0, st, a);
    else if (a.x_is_f32 && !a.dy_is_f32 && a.dx_is_f32) launch(ln_bwd_kernel<float, bf16, float, bf16, NPL>, dim3(grid), dim3(nt), 0, st, a);
    else if (!a.x_is_f32 && !a.dy_is_f32 && !a.dx_is_f32) launch(ln_bwd_kernel<bf16, bf16, bf16, bf16, NPL>, dim3(grid), dim3(nt), 0, st, a);
    else EGOT2_CHECK(false, "layernorm_bwd: unsupported dtype mix");
  }
  EGOT2_LAUNCH_CHECK();
  return 0;
}

}  // namespace

int layernorm_fwd(const LayerNormArgs& a, cudaStream_t st) {
  EGOT2_CHECK(a.H % 32 == 0 && a.H <= 2048, "layernorm: H=%d must be a multiple of 32 and <= 2048", a.H);
  if (a.rows == 0) return 0;
  if (!a.x_is_f32 && ln_vec_ok(a.dtype, a.H, a.x, a.y, a.table, nullptr)) {
    switch (a.H) {
      case 128: return ln_fwd_vec_launch<128>(a, st);
      case 256: return ln_fwd_vec_launch<256>(a, st);
      case 512: return ln_fwd_vec_launch<512>(a, st);
      case 1024: return ln_fwd_vec_launch<1024>(a, st);
    }
  }
  switch (a.H / 32) {
    case 1: return ln_fwd_dispatch<1>(a, st);
    case 2: return ln_fwd_dispatch<2>(a, st);
    case 4: return ln_fwd_dispatch<4>(a, st);
    case 8: return ln_fwd_dispatch<8>(a, st);
    case 16: return ln_fwd_dispatch<16>(a, st);
    case 32: return ln_fwd_dispatch<32>(a, st);
    case 64: return ln_fwd_dispatch<64>(a, st);       // H = 2048: the LTA 2-task translator's shipped width
  }
  EGOT2_CHECK(false, "layernorm: H=%d not in {32,64,128,256,512,1024,2048}", a.H);
}

int layernorm_bwd(const LayerNormBwdArgs& a, cudaStream_t st) {
  EGOT2_CHECK(a.H % 32 == 0 && a.H <= 2048, "layernorm_bwd: H=%d must be a multiple of 32 and <= 2048", a.H);
  if (a.rows == 0) return 0;
  if (!a.x_is_f32 && !a.dy_is_f32 && !a.dx_is_f32 && ln_vec_ok(a.dtype, a.H, a.x, a.dy, a.dx, a.dres) &&
      (reinterpret_cast<uintptr_t>(a.dx2) & 15) == 0) {
    switch (a.H) {
      case 128: return ln_bwd_vec_launch<128>(a, st);
      case 256: return ln_bwd_vec_launch<256>(a, st);
      case 512: return ln_bwd_vec_launch<512>(a, st);     // H = 1024 would need 64 KB of static reduction smem
    }
  }
  // generic path: the fused dropout sites / column sums become separate launches around the LayerNorm kernel
  if (a.dcol) {
    LayerNormBwdArgs b = a;
    b.dcol = nullptr;
    EGOT2_TRY(layernorm_bwd(b, st));
    EGOT2_CHECK(!a.dx_is_f32, "layernorm_bwd: fused column sums need dtype dx");
    return colsum_accum(a.dtype, a.rows, a.H, a.dx2 ? a.dx2 : a.dx, a.H, 0, 0, a.dcol, st);
  }
  if (a.dy_p_drop > 0.f || a.dx2) {
    LayerNormBwdArgs b = a;
    b.dy_p_drop = 0.f; b.dx2 = nullptr;
    const size_t n = (size_t)a.rows * a.H;
    if (a.dy_p_drop > 0.f) {
      EGOT2_CHECK(!a.dy_is_f32, "layernorm_bwd: fused dy dropout needs dtype dy");
      EGOT2_TRY(dropout_inplace(a.dtype, const_cast<void*>(a.dy), n, a.dy_p_drop, a.dy_drop_key, st));
    }
    EGOT2_TRY(layernorm_bwd(b, st));
    if (a.dx2) {
      EGOT2_CHECK(!a.dx_is_f32, "layernorm_bwd: fused dx2 dropout needs dtype dx");
      EGOT2_CUDA(cudaMemcpyAsync(a.dx2, a.dx, n * dtype_size(a.dtype), cudaMemcpyDeviceToDevice, st));
      EGOT2_TRY(dropout_inplace(a.dtype, a.dx2, n, a.dx2_p_drop, a.dx2_drop_key, st));
    }
    return 0;
  }
  switch (a.H / 32) {
    case 1: return ln_bwd_dispatch<1>(a, st);
    case 2: return ln_bwd_dispatch<2>(a, st);
    case 4: return ln_bwd_dispatch<4>(a, st);
    case 8: return ln_bwd_dispatch<8>(a, st);
    case 16: return ln_bwd_dispatch<16>(a, st);
    case 32: return ln_bwd_dispatch<32>(a, st);
    case 64: return ln_bwd_dispatch<64>(a, st);
  }
  EGOT2_CHECK(false, "layernorm_bwd: H=%d not in {32,64,128,256,512,1024,2048}", a.H);
}

int table_grad(int dtype, int B, int T, int H, const void* dy, float* dtable, const SegOut& so, float p_drop, uint64_t drop_key,
               cudaStream_t st) {
  const int nt = H < 256 ? ((H + 31) / 32 * 32) : 256;
  int chunks = (4 * sm_count() + T - 1) / T;           // ~4 CTAs per SM
  if (chunks > B) chunks = B;
  if (chunks < 1) chunks = 1;
  const int per = (B + chunks - 1) / chunks;
  dim3 grid(T, (B + per - 1) / per);
  ProfScope prof(st, "table_grad B%d T%d H%d", B, T, H);
  const int lpr = H / 8;
  if (dtype == EGOT2_BF16 && H % 8 == 0 && lpr <= 128 && (lpr & (lpr - 1)) == 0 && (reinterpret_cast<uintptr_t>(dy) & 15) == 0)
    launch(table_grad_vec_kernel, grid, dim3(128), 0, st, B, T, H, per, (const bf16*)dy, dtable, so, p_drop, drop_key);
  else if (dtype == EGOT2_F32) launch(table_grad_kernel<float>, grid, dim3(nt), 0, st, B, T, H, per, (const float*)dy, dtable, so, p_drop, drop_key);
  else launch(table_grad_kernel<bf16>, grid, dim3(nt), 0, st, B, T, H, per, (const bf16*)dy, dtable, so, p_drop, drop_key);
  EGOT2_LAUNCH_CHECK();
  return 0;
}

int colsum_accum(int dtype, int M, int N, const void* x, int ldx, int rpg, int gstride, float* out, cudaStream_t st) {
  if (M == 0 || N == 0) return 0;
  if (dtype == EGOT2_BF16 && N % 8 == 0 && ldx % 8 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0) {
    const int lanes_per_row = N >= 256 ? 32 : (N >= 128 ? 16 : (N >= 64 ? 8 : (N >= 32 ? 4 : (N >= 16 ? 2 : 1))));
    const int col_blocks = (N + lanes_per_row * 8 - 1) / (lanes_per_row * 8);
    int row_blocks = (sm_count() * 4 + col_blocks - 1) / col_blocks;
    int rows_per_cta = (M + row_blocks - 1) / row_blocks;
    const int min_rows = 4 * (256 / lanes_per_row);
    if (rows_per_cta < min_rows) rows_per_cta = min_rows;
    row_blocks = (M + rows_per_cta - 1) / rows_per_cta;
    ProfScope prof(st, "colsum M%d N%d", M, N);
    launch(colsum_bf16_vec_kernel, dim3(col_blocks, row_blocks), dim3(256), 0, st, M, N, (const bf16*)x, ldx, rpg, gstride, out,
                                                                        rows_per_cta, lanes_per_row);
    EGOT2_LAUNCH_CHECK();
    return 0;
  }
  const int col_blocks = (N + 63) / 64;
  int row_blocks = (sm_count() * 8 + col_blocks - 1) / col_blocks;
  int rows_per_cta = (M + row_blocks - 1) / row_blocks;
  if (rows_per_cta < 64) rows_per_cta = 64;
  row_blocks = (M + rows_per_cta - 1) / rows_per_cta;
  dim3 grid(col_blocks, row_blocks), block(32, 8);
  ProfScope prof(st, "colsum M%d N%d", M, N);
  if (dtype == EGOT2_F32) launch(colsum_kernel<float>, dim3(grid), dim3(block), 0, st, M, N, (const float*)x, ldx, rpg, gstride, out, rows_per_cta);
  else launch(colsum_kernel<bf16>, dim3(grid), dim3(block), 0, st, M, N, (const bf16*)x, ldx, rpg, gstride, out, rows_per_cta);
  EGOT2_LAUNCH_CHECK();
  return 0;
}

// y (bf16) = x (fp32) and out += column sums of x, one launch
int colsum_cast_bf16(int M, int N, const float* x, int ldx, void* y, int ldy, float* out, cudaStream_t st) {
  if (M == 0 || N == 0) return 0;
  EGOT2_CHECK((N & 1) == 0 && (ldx & 1) == 0 && (ldy & 1) == 0 && (reinterpret_cast<uintptr_t>(x) & 7) == 0 &&
              (reinterpret_cast<uintptr_t>(y) & 3) == 0, "colsum_cast: N and the row pitches must be even");
  const int col_blocks = (N + 63) / 64;
  int row_blocks = (sm_count() * 8 + col_blocks - 1) / col_blocks;
  int rows_per_cta = (M + row_blocks - 1) / row_blocks;
  if (rows_per_cta < 64) rows_per_cta = 64;
  row_blocks = (M + rows_per_cta - 1) / rows_per_cta;
  ProfScope prof(st, "colsum_cast M%d N%d", M, N);
  launch(colsum_cast_kernel, dim3(col_blocks, row_blocks), dim3(32, 8), 0, st, M, N, x, ldx, (bf16*)y, ldy, out, rows_per_cta);
  EGOT2_LAUNCH_CHECK();
  return 0;
}

static inline int ew_grid(size_t n, int per_thread = 1) {
  size_t ctas = (n / per_thread + 255) / 256;
  size_t cap = (size_t)sm_count() * 16;
  if (ctas > cap) ctas = cap;
  return ctas ? (int)ctas : 1;
}

int dropout_inplace(int dtype, void* x, size_t n, float p, uint64_t key, cudaStream_t st) {
  if (p <= 0.f || n == 0) return 0;
  const float inv_keep = 1.f / (1.f - p);
  ProfScope prof(st, "dropout_inplace n%zu", n);
  if (dtype == EGOT2_F32) launch(dropout_kernel<float>, dim3(ew_grid(n)), dim3(256), 0, st, (float*)x, n, p, inv_keep, key);
  else launch(dropout_kernel<bf16>, dim3(ew_grid(n)), dim3(256), 0, st, (bf16*)x, n, p, inv_keep, key);
  EGOT2_LAUNCH_CHECK();
  return 0;
}

int pool_fwd(int dtype, int B, int T, int H, int pool, int row_tokens, const void* x, float* pooled, cudaStream_t st) {
  const int rows = pool ? B : B * row_tokens;
  if (rows == 0) return 0;
  const int nt = H < 256 ? ((H + 31) / 32 * 32) : 256;
  ProfScope prof(st, "pool_fwd B%d T%d H%d", B, T, H);
  if (dtype == EGOT2_F32) launch(pool_fwd_kernel<float>, dim3(rows), dim3(nt), 0, st, B, T, H, pool, row_tokens, (const float*)x, pooled);
  else launch(pool_fwd_kernel<bf16>, dim3(rows), dim3(nt), 0, st, B, T, H, pool, row_tokens, (const bf16*)x, pooled);
  EGOT2_LAUNCH_CHECK();
  return 0;
}

int pool_bwd(int dtype, int B, int T, int H, int pool, int row_tokens, const float* dpooled, void* dx, cudaStream_t st) {
  if (B * T == 0) return 0;
  const int nt = H < 256 ? ((H + 31) / 32 * 32) : 256;
  ProfScope prof(st, "pool_bwd B%d T%d H%d", B, T, H);
  if (dtype == EGOT2_F32) launch(pool_bwd_kernel<float>, dim3(B * T), dim3(nt), 0, st, B, T, H, pool, row_tokens, dpooled, (float*)dx);
  else launch(pool_bwd_kernel<bf16>, dim3(B * T), dim3(nt), 0, st, B, T, H, pool, row_tokens, dpooled, (bf16*)dx);
  EGOT2_LAUNCH_CHECK();
  return 0;
}

int cast_f32_to(int dtype, const float* src, void* dst, size_t n, cudaStream_t st) {
  if (n == 0) return 0;
  ProfScope prof(st, "cast_f32_to n%zu", n);
  if (dtype == EGOT2_BF16) {
    EGOT2_CHECK(((uintptr_t)src % 16 == 0) && ((uintptr_t)dst % 8 == 0), "cast: unaligned buffers");
    launch(cast_to_bf16_kernel, dim3(ew_grid(n, 4)), dim3(256), 0, st, src, (bf16*)dst, n);
  } else {
    launch(copy_f32_kernel, dim3(ew_grid(n)), dim3(256), 0, st, src, (float*)dst, n);
  }
  EGOT2_LAUNCH_CHECK();
  return 0;
}

int cast_to_f32(int dtype, const void* src, float* dst, size_t n, cudaStream_t st) {
  if (n == 0) return 0;
  ProfScope prof(st, "cast_to_f32 n%zu", n);
  if (dtype == EGOT2_BF16) launch(cast_to_f32_kernel, dim3(ew_grid(n)), dim3(256), 0, st, (const bf16*)src, dst, n);
  else launch(copy_f32_kernel, dim3(ew_grid(n)), dim3(256), 0, st, (const float*)src, dst, n);
  EGOT2_LAUNCH_CHECK();
  return 0;
}

int cast_rows_f32_to_bf16(const float* src, int rows, int n, void* dst, int ld, cudaStream_t st) {
  if (rows == 0 || n == 0) return 0;
  ProfScope prof(st, "cast_rows rows%d n%d", rows, n);
  launch(cast_rows_kernel, dim3(ew_grid((size_t)rows * ld)), dim3(256), 0, st, src, rows, n, (bf16*)dst, ld);
  EGOT2_LAUNCH_CHECK();
  return 0;
}

int zero_f32(float* p, size_t n, cudaStream_t st) {
  if (n == 0) return 0;
  EGOT2_CUDA(cudaMemsetAsync(p, 0, n * sizeof(float), st));
  return 0;
}

}  // namespace egot2

// ---------------------------------------------------------------------------------- C ABI (utilities)
using namespace egot2;

extern "C" int egot2_cast_f32_to_bf16(const float* src, void* dst, size_t n, void* stream) {
  return cast_f32_to(EGOT2_BF16, src, dst, n, (cudaStream_t)stream);
}
extern "C" int egot2_cast_bf16_to_f32(const void* src, float* dst, size_t n, void* stream) {
  if (n == 0) return 0;
  launch(cast_to_f32_kernel, dim3(ew_grid(n)), dim3(256), 0, (cudaStream_t)stream, (const bf16*)src, dst, n);
  EGOT2_LAUNCH_CHECK();
  return 0;
}

static int adam_launch(float* param, float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr, float beta1,
                       float beta2, float eps, float weight_decay, int32_t step, float grad_scale, void* shadow,
                       int zero_grad, void* stream, const int32_t* step_dev = nullptr, bool decoupled = false,
                       const float* lr_dev = nullptr, const egot2_grad_guard* guard = nullptr) {
  EGOT2_CHECK(step >= 1 || step_dev, "adam: step must be >= 1");
  if (n == 0) return 0;
  const float bc1 = 1.f - powf(beta1, (float)step);
  const float bc2 = 1.f - powf(beta2, (float)step);
  ProfScope prof((cudaStream_t)stream, "adam n%zu", n);
  if (decoupled)
    launch(adam_kernel<true>, dim3(ew_grid(n)), dim3(256), 0, (cudaStream_t)stream, param, grad, exp_avg, exp_avg_sq, n, lr,
           beta1, beta2, eps, weight_decay, bc1, sqrtf(bc2), grad_scale, (bf16*)shadow, zero_grad, step_dev, lr_dev, guard);
  else
    launch(adam_kernel<false>, dim3(ew_grid(n)), dim3(256), 0, (cudaStream_t)stream, param, grad, exp_avg, exp_avg_sq, n, lr,
           beta1, beta2, eps, weight_decay, bc1, sqrtf(bc2), grad_scale, (bf16*)shadow, zero_grad, step_dev, lr_dev, guard);
  EGOT2_LAUNCH_CHECK();
  return 0;
}
extern "C" int egot2_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                               float beta1, float beta2, float eps, float weight_decay, int32_t step, float grad_scale,
                               void* stream) {
  return adam_launch(param, const_cast<float*>(grad), exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay, step,
                     grad_scale, nullptr, 0, stream);
}
extern "C" int egot2_adam_step_fused(float* param, float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                                     float beta1, float beta2, float eps, float weight_decay, int32_t step,
                                     float grad_scale, void* shadow_bf16, int32_t zero_grad, void* stream) {
  return adam_launch(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay, step, grad_scale, shadow_bf16,
                     zero_grad, stream);
}

// torch.optim.AdamW (HOI EgoT2-g: lr 1e-4, weight decay 1e-4, HOI/tasks/multitask/video_task.py:265-268), same fusions
extern "C" int egot2_adamw_step_fused(float* param, float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                                      float beta1, float beta2, float eps, float weight_decay, int32_t step,
                                      float grad_scale, void* shadow_bf16, int32_t zero_grad, void* stream) {
  return adam_launch(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay, step, grad_scale, shadow_bf16,
                     zero_grad, stream, nullptr, true);
}

extern "C" int egot2_adam_step_fused_dev(float* param, float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                                         float beta1, float beta2, float eps, float weight_decay,
                                         const int32_t* step_dev, float grad_scale, void* shadow_bf16, int32_t zero_grad,
                                         void* stream) {
  EGOT2_CHECK(step_dev != nullptr, "adam: step_dev is null");
  return adam_launch(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay, 1, grad_scale, shadow_bf16,
                     zero_grad, stream, step_dev);
}

extern "C" int egot2_adam_step_fused_sched(float* param, float* grad, float* exp_avg, float* exp_avg_sq, size_t n,
                                           const float* lr_dev, float beta1, float beta2, float eps, float weight_decay,
                                           const int32_t* step_dev, float grad_scale, void* shadow_bf16, int32_t zero_grad,
                                           int32_t decoupled, void* stream) {
  EGOT2_CHECK(step_dev != nullptr && lr_dev != nullptr, "adam: step_dev / lr_dev is null");
  return adam_launch(param, grad, exp_avg, exp_avg_sq, n, 0.f, beta1, beta2, eps, weight_decay, 1, grad_scale, shadow_bf16,
                     zero_grad, stream, step_dev, decoupled != 0, lr_dev);
}

extern "C" int egot2_adam_step_fused_guard(float* param, float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                                           const float* lr_dev, float beta1, float beta2, float eps, float weight_decay,
                                           const int32_t* step_dev, float grad_scale, void* shadow_bf16, int32_t zero_grad,
                                           int32_t decoupled, const egot2_grad_guard* guard, void* stream) {
  EGOT2_CHECK(step_dev != nullptr && guard != nullptr, "adam: step_dev / guard is null");
  return adam_launch(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay, 1, grad_scale, shadow_bf16,
                     zero_grad, stream, step_dev, decoupled != 0, lr_dev, guard);
}

extern "C" size_t egot2_grad_norm_workspace_bytes(void) { return kNormCtas * sizeof(double) + 16; }

extern "C" int egot2_grad_norm(const float* grad, size_t n, float grad_scale, egot2_grad_guard* guard, int32_t* step_dev,
                               void* workspace, size_t ws_bytes, void* stream) {
  EGOT2_CHECK(guard && workspace && (grad || n == 0), "grad_norm: grad / guard / workspace is null");
  EGOT2_CHECK(ws_bytes >= egot2_grad_norm_workspace_bytes() && reinterpret_cast<uintptr_t>(workspace) % 8 == 0,
              "grad_norm: workspace of %zu bytes (8-byte aligned) needed, got %zu", egot2_grad_norm_workspace_bytes(), ws_bytes);
  double* part = (double*)workspace;
  unsigned int* ctr = (unsigned int*)(part + kNormCtas);
  ProfScope prof((cudaStream_t)stream, "grad_norm n%zu", n);
  launch(grad_norm_kernel, dim3(kNormCtas), dim3(kNormThreads), 0, (cudaStream_t)stream, grad, n, grad_scale, guard, step_dev,
         part, ctr);
  EGOT2_LAUNCH_CHECK();
  return 0;
}

extern "C" int egot2_opt_advance(int32_t* step_dev, const egot2_lr_sched* sched, float* lr_dev, void* stream) {
  EGOT2_CHECK(step_dev && sched && lr_dev, "opt_advance: step_dev / sched / lr_dev is null");
  launch(opt_advance_kernel, dim3(1), dim3(1), 0, (cudaStream_t)stream, step_dev, sched, lr_dev);
  EGOT2_LAUNCH_CHECK();
  return 0;
}

extern "C" int egot2_hhi_tok_table_fwd(const float* task_embed, const float* pe, int32_t pe_len, int32_t n_seg,
                                       const int32_t* seg_tokens, const int32_t* seg_task_id, int32_t H,
                                       float* tok_table, void* stream) {
  EGOT2_CHECK(n_seg >= 1 && n_seg <= EGOT2_MAX_SEG, "tok_table: n_seg=%d", n_seg);
  SegList s; s.n = n_seg; int T = 0;
  for (int i = 0; i < n_seg; ++i) {
    EGOT2_CHECK(seg_tokens[i] <= pe_len, "tok_table: segment of %d tokens exceeds the pe table (%d)", seg_tokens[i], pe_len);
    s.tokens[i] = seg_tokens[i]; s.task[i] = seg_task_id[i]; T += seg_tokens[i];
  }
  if (T == 0) return 0;
  ProfScope prof((cudaStream_t)stream, "hhi_tok_table_fwd T%d H%d", T, H);
  launch(hhi_tok_table_fwd_kernel, dim3(T), dim3(128), 0, (cudaStream_t)stream, task_embed, pe, s, H, tok_table);
  EGOT2_LAUNCH_CHECK();
  return 0;
}
extern "C" int egot2_hhi_tok_table_bwd(const float* d_tok_table, int32_t n_seg, const int32_t* seg_tokens,
                                       const int32_t* seg_task_id, int32_t H, float* d_task_embed, void* stream) {
  EGOT2_CHECK(n_seg >= 1 && n_seg <= EGOT2_MAX_SEG, "tok_table: n_seg=%d", n_seg);
  SegList s; s.n = n_seg;
  for (int i = 0; i < n_seg; ++i) { s.tokens[i] = seg_tokens[i]; s.task[i] = seg_task_id[i]; }
  ProfScope prof((cudaStream_t)stream, "hhi_tok_table_bwd H%d", H);
  launch(hhi_tok_table_bwd_kernel, dim3(n_seg), dim3(128), 0, (cudaStream_t)stream, d_tok_table, s, H, d_task_embed);
  EGOT2_LAUNCH_CHECK();
  return 0;
}

extern "C" int egot2_slowfast_pool_fwd(const void* in, int32_t in_dtype, int32_t B, int32_t C, int32_t Tin, int32_t hw,
                                       int32_t Tout, void* out, int32_t out_dtype, void* stream) {
  EGOT2_CHECK(Tout > 0 && Tin % Tout == 0, "slowfast_pool: Tin=%d must be a multiple of Tout=%d", Tin, Tout);
  const size_t warps = (size_t)B * C * Tout;
  if (warps == 0) return 0;
  const int grid = (int)((warps * 32 + 255) / 256);
  cudaStream_t st = (cudaStream_t)stream;
  ProfScope prof(st, "slowfast_pool B%d C%d Tin%d hw%d", B, C, Tin, hw);
  if (in_dtype == EGOT2_F32 && out_dtype == EGOT2_F32)
    launch(slowfast_pool_kernel<float, float>, dim3(grid), dim3(256), 0, st, (const float*)in, B, C, Tin, hw, Tout, (float*)out);
  else if (in_dtype == EGOT2_F32 && out_dtype == EGOT2_BF16)
    launch(slowfast_pool_kernel<float, bf16>, dim3(grid), dim3(256), 0, st, (const float*)in, B, C, Tin, hw, Tout, (bf16*)out);
  else if (in_dtype == EGOT2_BF16 && out_dtype == EGOT2_BF16)
    launch(slowfast_pool_kernel<bf16, bf16>, dim3(grid), dim3(256), 0, st, (const bf16*)in, B, C, Tin, hw, Tout, (bf16*)out);
  else EGOT2_CHECK(false, "slowfast_pool: unsupported dtypes %d -> %d", in_dtype, out_dtype);
  EGOT2_LAUNCH_CHECK();
  return 0;
}

extern "C" int egot2_layernorm_fwd(int32_t dtype, int32_t rows, int32_t H, const void* x, const float* g, const float* b,
                                   float eps, void* y, float* stat, void* stream) {
  LayerNormArgs a; a.rows = rows; a.H = H; a.dtype = dtype; a.x = x; a.g = g; a.b = b; a.eps = eps; a.y = y; a.stat = stat;
  return layernorm_fwd(a, (cudaStream_t)stream);
}
