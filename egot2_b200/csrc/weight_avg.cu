// weight_avg.cu — the averaged copy of the parameter arena (egot2_weight_avg_update): torch.optim.swa_utils.AveragedModel's
// EMA and SWA updates, in one launch after the optimizer's, that decides on the device whether the step is due.
#define EGOT2_FILE_ID 18
#include "ops.h"

namespace egot2 {
namespace {

constexpr int kAvgThreads = 256;
constexpr int kAvgUnroll = 4;        // independent 16-byte loads of each array in flight per thread

// ATen's lerp (ATen/native/Lerp.h) as torch's CUDA _foreach_lerp_ compiles it for fp32: nvcc contracts both branches into
// one FMA each, a + w * (p - a) and p + (-(p - a)) * (1 - w).  one_minus_w = 1 - w, rounded once.
__device__ __forceinline__ float lerp_aten(float a, float p, float w, float one_minus_w) {
  const float d = __fsub_rn(p, a);
  return w < 0.5f ? __fmaf_rn(w, d, a) : __fmaf_rn(-d, one_minus_w, p);
}

__global__ void __launch_bounds__(kAvgThreads) weight_avg_kernel(const float4* __restrict__ param, float4* __restrict__ avg,
                                                                 size_t n4, int kind, float ema_w, int every, int start,
                                                                 const int32_t* __restrict__ step_dev,
                                                                 const egot2_grad_guard* __restrict__ guard) {
  EGOT2_PDL_ENTER();
  if (guard && guard->skip) return;                    // a skipped step: the guard took the step count back
  const int32_t t = *step_dev;
  if (t < start || (t - start) % every != 0) return;  // not due: every CTA leaves at once
  const int32_t k = (t - start) / every;              // earlier updates (AveragedModel.n_averaged)
  const size_t stride = (size_t)gridDim.x * kAvgThreads;
  size_t i0 = blockIdx.x * (size_t)kAvgThreads + threadIdx.x;
  if (k == 0) {                                        // the first update copies the parameters
    for (; i0 < n4; i0 += stride) avg[i0] = param[i0];
    return;
  }
  const float w = kind == EGOT2_AVG_SWA ? __fdiv_rn(1.f, (float)(k + 1)) : ema_w;
  const float omw = __fsub_rn(1.f, w);
  for (; i0 < n4; i0 += stride * kAvgUnroll) {
    float4 p[kAvgUnroll], a[kAvgUnroll];
#pragma unroll
    for (int u = 0; u < kAvgUnroll; ++u) {
      const size_t i = i0 + u * stride;
      if (i < n4) {
        p[u] = param[i];
        a[u] = avg[i];
      }
    }
#pragma unroll
    for (int u = 0; u < kAvgUnroll; ++u) {
      const size_t i = i0 + u * stride;
      if (i < n4) {
        float4 r;
        r.x = lerp_aten(a[u].x, p[u].x, w, omw);
        r.y = lerp_aten(a[u].y, p[u].y, w, omw);
        r.z = lerp_aten(a[u].z, p[u].z, w, omw);
        r.w = lerp_aten(a[u].w, p[u].w, w, omw);
        avg[i] = r;
      }
    }
  }
}

}  // namespace
}  // namespace egot2

using namespace egot2;

extern "C" int egot2_weight_avg_update(const float* param, float* avg, size_t n, int32_t kind, float ema_weight,
                                       int32_t every, int32_t start, const int32_t* step_dev, const egot2_grad_guard* guard,
                                       void* stream) {
  EGOT2_CHECK(param && avg && step_dev, "weight_avg_update: param / avg / step_dev is null");
  EGOT2_CHECK(kind == EGOT2_AVG_EMA || kind == EGOT2_AVG_SWA, "weight_avg_update: unknown kind %d", (int)kind);
  EGOT2_CHECK(every > 0 && start > 0, "weight_avg_update: every %d and start %d must be positive", (int)every, (int)start);
  EGOT2_CHECK(kind != EGOT2_AVG_EMA || (ema_weight >= 0.f && ema_weight <= 1.f),
              "weight_avg_update: ema_weight %g must be in [0, 1]", (double)ema_weight);
  EGOT2_CHECK(n % 4 == 0 && reinterpret_cast<uintptr_t>(param) % 16 == 0 && reinterpret_cast<uintptr_t>(avg) % 16 == 0,
              "weight_avg_update: n %zu must be a multiple of 4 and both arrays 16-byte aligned", n);
  if (n == 0) return 0;
  const size_t n4 = n / 4;
  size_t grid = (n4 + (size_t)kAvgThreads * kAvgUnroll - 1) / ((size_t)kAvgThreads * kAvgUnroll);
  const size_t cap = (size_t)sm_count() * 2;
  if (grid > cap) grid = cap;
  ProfScope prof((cudaStream_t)stream, "weight_avg_update n%zu", n);
  launch(weight_avg_kernel, dim3((unsigned)grid), dim3(kAvgThreads), 0, (cudaStream_t)stream,
         reinterpret_cast<const float4*>(param), reinterpret_cast<float4*>(avg), n4, (int)kind, ema_weight, (int)every,
         (int)start, step_dev, guard);
  EGOT2_LAUNCH_CHECK();
  return 0;
}
