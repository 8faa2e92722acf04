// stats.cu — per-parameter gradient and weight statistics of the parameter arena (egot2_param_stats): num, finite min / max,
// fp64 sum and sum of squares, non-finite count, L2 norm and the bucket counts of TensorBoard's default histogram, for the
// gradient the optimizer applies and for the parameters before the update, in one launch that decides on the device whether
// the step is due.
#include <math.h>

#define EGOT2_FILE_ID 12
#include "ops.h"

namespace egot2 {
namespace {

constexpr int kStatsThreads = 256;
constexpr int kBuckets = EGOT2_STATS_BUCKETS;
constexpr int kEdges = kBuckets + 1;
constexpr int kPosEdges = (kEdges - 1) / 2;          // 774 positive edges 1e-12 * 1.1^k; edge kPosEdges is 0

// float -> unsigned key whose unsigned order is the float order (-0.0 just below +0.0): max keeps atomicMax(key),
// min keeps atomicMax(~key), so 0 is "nothing seen" for both and the scratch is zero when idle
__device__ __forceinline__ unsigned int order_key(float f) {
  const unsigned int b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float from_order_key(unsigned int k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// np.histogram's bucket of d over the edges e[0..kBuckets] (shared memory): e[i] <= d < e[i+1], the last bucket closed on
// the right; -1 outside [e[0], e[kBuckets]].  The candidate from the logarithm is off by at most one; the exact edges decide.
__device__ __forceinline__ int bucket_of(double d, const double* e) {
  if (!(d >= e[0] && d <= e[kBuckets])) return -1;
  if (d == e[kBuckets]) return kBuckets - 1;
  const float a = fabsf((float)d);
  int i;
  if (a < 1e-12f) {
    i = d < 0.0 ? kPosEdges - 1 : kPosEdges;
  } else {
    int k = (int)((__logf(a) + 27.6310211f) * 10.4920587f);      // log(a / 1e-12) / log(1.1)
    k = k < 0 ? 0 : (k > kPosEdges - 1 ? kPosEdges - 1 : k);
    i = d > 0.0 ? kPosEdges + 1 + k : kPosEdges - 2 - k;
    i = i < 0 ? 0 : i;
  }
  while (i > 0 && d < e[i]) --i;
  while (i < kBuckets - 1 && d >= e[i + 1]) ++i;
  return i;
}

struct StatsScratch {
  double* part;            // [n_units][2]: sum, sum of squares of every unit
  unsigned int* max_key;   // [2P]
  unsigned int* min_key;   // [2P] (~key)
  unsigned int* nonfinite; // [2P]
  unsigned int* nan_seen;  // [2P]
  unsigned int* pair_ctr;  // [2P]: units of the pair finished
  unsigned int* cta_ctr;   // [1]
  int32_t* counts;         // [2P][kBuckets]
};

inline size_t stats_align(size_t x) { return (x + 255) / 256 * 256; }
// byte offsets of the counter words and of the scratch counts inside the workspace (the unit partials come first)
inline size_t stats_words_off(int n_units) { return stats_align((size_t)n_units * 2 * sizeof(double)); }
inline size_t stats_counts_off(int P, int n_units) {
  return stats_words_off(n_units) + stats_align((10 * (size_t)P + 1) * sizeof(unsigned int));
}

inline StatsScratch stats_scratch(void* ws, int P, int n_units) {
  StatsScratch s;
  char* base = (char*)ws;
  s.part = (double*)base;
  unsigned int* w = (unsigned int*)(base + stats_words_off(n_units));
  s.max_key = w; s.min_key = w + 2 * P; s.nonfinite = w + 4 * P; s.nan_seen = w + 6 * P; s.pair_ctr = w + 8 * P;
  s.cta_ctr = w + 10 * P;
  s.counts = (int32_t*)(base + stats_counts_off(P, n_units));
  return s;
}

__global__ void __launch_bounds__(kStatsThreads) param_stats_kernel(
    const float* __restrict__ grad, const float* __restrict__ param, float scale, const int32_t* __restrict__ step_dev,
    egot2_param_stats_desc* __restrict__ desc, const egot2_stats_param* __restrict__ params, const egot2_stats_unit* __restrict__ units,
    int n_units, const double* __restrict__ edges, egot2_param_stat* __restrict__ out, int32_t* __restrict__ out_counts,
    StatsScratch ws) {
  EGOT2_PDL_ENTER();
  __shared__ double s_edges[kEdges];
  __shared__ int32_t s_hist[kBuckets];
  __shared__ double s_red[kStatsThreads / 32];
  __shared__ double s_part[kStatsThreads][2];
  __shared__ unsigned int s_flag;
  const int32_t t = *step_dev;
  const int every = desc->every;
  if (t < 1 || every < 1 || (t - 1) % every != 0) return;            // not due: every CTA leaves at once
  const int P = desc->n_params;
  const bool hist = desc->histograms != 0 && out_counts != nullptr;
  const int tid = threadIdx.x;
  if (hist) {
    for (int i = tid; i < kEdges; i += kStatsThreads) s_edges[i] = edges[i];
    for (int i = tid; i < kBuckets; i += kStatsThreads) s_hist[i] = 0;
  }
  __syncthreads();
  for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
    const egot2_stats_unit un = units[u];
    const int q = un.array * P + un.param;                             // pair: array 0 = gradient, 1 = parameters
    const float* src = un.array == 0 ? grad : param;
    const float mul = un.array == 0 ? scale : 1.f;
    double sum = 0.0, sq = 0.0;
    float mn = INFINITY, mx = -INFINITY;
    unsigned int nonfin = 0, nan = 0;
    constexpr int U = 4;                                               // independent loads in flight per thread
    for (int64_t i0 = un.begin + tid; i0 < un.end; i0 += (int64_t)U * kStatsThreads) {
      float x[U];
#pragma unroll
      for (int k = 0; k < U; ++k) {
        const int64_t i = i0 + (int64_t)k * kStatsThreads;
        x[k] = i < un.end ? src[i] * mul : 0.f;
      }
#pragma unroll
      for (int k = 0; k < U; ++k) {
        const float v = x[k];
        if (i0 + (int64_t)k * kStatsThreads >= un.end) {
        } else if (isfinite(v)) {
          const double d = (double)v;
          sum += d;
          sq += d * d;
          mn = fminf(mn, v);
          mx = fmaxf(mx, v);
          if (hist) {
            const int b = bucket_of(d, s_edges);
            if (b >= 0) atomicAdd(&s_hist[b], 1);
          }
        } else {
          ++nonfin;
          nan |= isnan(v) ? 1u : 0u;
        }
      }
    }
    // min / max / non-finite: exact, so atomics in any order give the same result
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      nonfin += __shfl_xor_sync(0xffffffffu, nonfin, o);
      nan |= __shfl_xor_sync(0xffffffffu, nan, o);
    }
    if ((tid & 31) == 0) {
      if (mx >= mn) {                                                   // the warp saw a finite element
        atomicMax(&ws.max_key[q], order_key(mx));
        atomicMax(&ws.min_key[q], ~order_key(mn));
      }
      if (nonfin) atomicAdd(&ws.nonfinite[q], nonfin);
      if (nan) atomicOr(&ws.nan_seen[q], 1u);
    }
    sum = block_sum_f64(sum, s_red);                                   // fixed order: the unit's partials are reproducible
    sq = block_sum_f64(sq, s_red);
    if (tid == 0) {
      ws.part[2 * u] = sum;
      ws.part[2 * u + 1] = sq;
    }
    __syncthreads();                                                    // s_hist complete
    if (hist) {
      int32_t* dst = ws.counts + (size_t)q * kBuckets;
      for (int b = tid; b < kBuckets; b += kStatsThreads) {
        const int32_t c = s_hist[b];
        if (c) {
          atomicAdd(&dst[b], c);
          s_hist[b] = 0;
        }
      }
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) {
      const egot2_stats_param& pr = params[un.param];
      s_flag = atomicAdd(&ws.pair_ctr[q], 1u) == (unsigned int)pr.n_units[un.array] - 1 ? 1u : 0u;
    }
    __syncthreads();
    if (!s_flag) continue;
    // the last unit of this pair: add the unit partials in unit order, write the record, hand the counts over
    __threadfence();
    const egot2_stats_param& pr = params[un.param];
    const int u0 = pr.first_unit[un.array], nu = pr.n_units[un.array];
    double tsum = 0.0, tsq = 0.0;
    for (int base = 0; base < nu; base += kStatsThreads) {
      if (base + tid < nu) {
        s_part[tid][0] = __ldcg(&ws.part[2 * (u0 + base + tid)]);
        s_part[tid][1] = __ldcg(&ws.part[2 * (u0 + base + tid) + 1]);
      }
      __syncthreads();
      if (tid == 0) {
        const int m = nu - base < kStatsThreads ? nu - base : kStatsThreads;
        for (int j = 0; j < m; ++j) { tsum += s_part[j][0]; tsq += s_part[j][1]; }
      }
      __syncthreads();
    }
    if (hist) {
      int32_t* scr = ws.counts + (size_t)q * kBuckets;
      int32_t* dst = out_counts + (size_t)q * kBuckets;
      for (int b = tid; b < kBuckets; b += kStatsThreads) {
        dst[b] = __ldcg(&scr[b]);
        scr[b] = 0;
      }
    }
    if (tid == 0) {
      const unsigned int kmax = __ldcg(&ws.max_key[q]), kmin = __ldcg(&ws.min_key[q]);
      const unsigned int nf = __ldcg(&ws.nonfinite[q]), nanq = __ldcg(&ws.nan_seen[q]);
      egot2_param_stat* r = out + q;
      r->sum = tsum;
      r->sum_squares = tsq;
      r->min = kmax ? from_order_key(~kmin) : INFINITY;                // no finite element: +inf / -inf
      r->max = kmax ? from_order_key(kmax) : -INFINITY;
      r->norm = nanq ? NAN : (nf ? INFINITY : (float)sqrt(tsq));       // torch.linalg.vector_norm over every element
      r->nonfinite = (int32_t)nf;
      r->num = pr.numel;
      ws.max_key[q] = ws.min_key[q] = ws.nonfinite[q] = ws.nan_seen[q] = ws.pair_ctr[q] = 0;
    }
  }
  // the last CTA: total gradient norm over the parameters with a gradient (parameter order), then the stamp
  __threadfence();
  __syncthreads();
  if (tid == 0) s_flag = atomicAdd(ws.cta_ctr, 1u) == gridDim.x - 1 ? 1u : 0u;
  __syncthreads();
  if (!s_flag || tid != 0) return;
  __threadfence();
  double tot = 0.0;
  bool any_nan = false, any_inf = false;
  for (int p = 0; p < P; ++p) {
    if (!params[p].has_grad) continue;
    tot += __ldcg(&out[p].sum_squares);
    const float nrm = __ldcg(&out[p].norm);
    any_nan |= isnan(nrm);
    any_inf |= isinf(nrm);
  }
  desc->grad_norm = any_nan ? NAN : (any_inf ? INFINITY : (float)sqrt(tot));
  desc->step = t;
  *ws.cta_ctr = 0;
}

}  // namespace
}  // namespace egot2

using namespace egot2;

extern "C" size_t egot2_param_stats_workspace_bytes(int32_t n_params, int32_t n_units) {
  if (n_params <= 0 || n_units <= 0) return 0;
  return stats_counts_off(n_params, n_units) + (size_t)2 * n_params * kBuckets * sizeof(int32_t);
}

extern "C" int egot2_param_stats(const float* grad, const float* param, float grad_scale, const int32_t* step_dev,
                                 egot2_param_stats_desc* desc, const egot2_stats_param* params, int32_t n_params,
                                 const egot2_stats_unit* units, int32_t n_units, const double* edges,
                                 egot2_param_stat* stats, int32_t* counts, void* workspace, size_t ws_bytes, void* stream) {
  EGOT2_CHECK(grad && param && step_dev && desc && params && units && stats && workspace,
              "param_stats: grad / param / step_dev / desc / params / units / stats / workspace is null");
  EGOT2_CHECK(n_params > 0 && n_units > 0, "param_stats: n_params %d and n_units %d must be positive", n_params, n_units);
  EGOT2_CHECK((edges == nullptr) == (counts == nullptr), "param_stats: edges and counts go together (histograms)");
  EGOT2_CHECK(isfinite(grad_scale), "param_stats: grad_scale %g is not finite", grad_scale);
  const size_t need = egot2_param_stats_workspace_bytes(n_params, n_units);
  EGOT2_CHECK(ws_bytes >= need && reinterpret_cast<uintptr_t>(workspace) % 256 == 0,
              "param_stats: workspace of %zu bytes (256-byte aligned) needed, got %zu", need, ws_bytes);
  const StatsScratch s = stats_scratch(workspace, n_params, n_units);
  const int grid = n_units < 2 * sm_count() ? n_units : 2 * sm_count();
  ProfScope prof((cudaStream_t)stream, "param_stats P%d units%d", n_params, n_units);
  launch(param_stats_kernel, dim3(grid), dim3(kStatsThreads), 0, (cudaStream_t)stream, grad, param, grad_scale, step_dev,
         desc, params, units, (int)n_units, edges, stats, counts, s);
  EGOT2_LAUNCH_CHECK();
  return 0;
}
