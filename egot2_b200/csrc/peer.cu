// peer.cu — the data-parallel exchange step as ONE kernel over NVLink / NVSwitch peer memory:
//
//     gradient reduce-scatter  ->  Adam on this rank's slice  ->  all-gather of the updated parameters (fp32 + bf16 shadow)
//
// replaces [NCCL all-reduce of the flat gradient arena] + [fused Adam launch] of the reference's DDP step
// (HOI/scripts/lta/run_lta.py:249 DDPPlugin, HHI/tasks/ttm/video_task.py:64-66 Adam).  Every rank keeps its parameter arena,
// gradient arena and bf16 shadow in one cudaMalloc'd SLAB whose IPC handle the ranks exchange once (egot2_peer_*), so that every
// GPU can address every other GPU's slab.  Per step and rank r (world N, arena of n floats, slice_r = [r*ceil(n/N), ...)):
//   1. tell every peer "my gradients of epoch e are complete" (a release store of e into the peer's flag word for r);
//   2. wait until every rank said so; then for every element of slice_r: g = (1/N) * sum_p grad_p[i] in rank order (N-1 of the
//      loads cross NVLink), the Adam update on the LOCAL moments, and the new parameter written as fp32 and bf16 into ALL N slabs;
//   3. fence, tell every peer "my slice of epoch e is in your arena", and leave only when every rank said so.
// With a gradient guard (egot2_dp_desc.guard) step 2 is split at the global norm: dp_guard_reduce_kernel, then
// dp_guard_adam_kernel (one more flag round trip, for the per-rank partial sums of squares).  With parameter groups
// (egot2_dp_desc.groups) every quad takes its group's lr and weight decay, frozen quads are neither updated nor gathered
// (only their gradient is cleared) and stay out of the guard's norm.  With egot2_dp_desc.sgd the update is torch.optim.SGD
// (dp_reduce_sgd_kernel, or dp_guard_reduce_kernel + dp_guard_sgd_kernel) on the local momentum buffer; everything else is the same.
// After the kernel every rank holds bit-identical parameters (each slice is computed once, by its owner), no rank reads a
// peer's gradients any more (so the caller may clear its gradient arena), and nothing went through the host: the kernel sits in
// the step's CUDA graph behind the backward pass.  The message is latency-bound for the translators (0.7-9 M parameters), which
// is exactly where two NCCL calls + an eager optimizer launch per step cost 13 % at 8 GPUs (round 1).
// All spin waits are bounded (~4 s): a rank that never arrives makes the others trap instead of hanging the box.
#define EGOT2_FILE_ID 16
#include <math.h>
#include <string.h>

#include "ops.h"

namespace egot2 {
namespace {

constexpr int kMaxRanks = 8;
constexpr int kChannels = 2;           // independent exchanges in flight (e.g. [embed_numel, n) during the embedding backward, then [0, embed_numel))
// u32 words per channel: arrive[8] @0, done[8] @8, epoch @16, grid counter @17; with a gradient guard also the phase-A grid
// counter @18, norm_arrive[8] @24 (rank p's partial sum of squares of that epoch is in norm_part[p]) and norm_part[8] (fp64) @32
constexpr int kChanWords = 64;
constexpr int kFlagWords = kChannels * kChanWords;
constexpr int kWordCtrA = 18, kWordNormArrive = 24, kWordNormPart = 32;
// after the channels' words: per channel, the phase-A per-CTA fp64 partial sums (the grid is capped at this)
constexpr int kMaxCtas = 1024;

struct DpArgs {
  int world, rank;
  size_t n;                            // arena elements
  size_t lo, hi;                       // the element range this launch exchanges (multiples of 4), split over the ranks
  int channel;
  int zero_remote;                     // 1: the owner of a slice clears that slice of EVERY rank's gradient arena right after
                                       // reading it (small arenas: saves the caller's separate clear launch)
  char* slab[kMaxRanks];               // every rank's slab as THIS process addresses it (slab[rank] = the local one)
  size_t off_param, off_grad, off_shadow, off_flags;     // byte offsets inside a slab (identical on every rank)
  float* m; float* v;                  // local Adam moments (full arena layout; only this rank's slice is used)
  float lr, b1, b2, eps, wd, bc1, bc2_sqrt;
  const int32_t* step_dev;             // optional: optimizer step count on the device (graph replays)
  const float* lr_dev;                 // optional: learning rate on the device (egot2_opt_advance)
  int decoupled;
  egot2_grad_guard* guard;             // optional: global-norm clip / non-finite skip (two launches, see dp_guard_reduce_kernel)
  const egot2_param_groups* groups;    // optional: parameter groups, with the arena's block map
  const uint8_t* block_group;
  // last, so that the Adam kernels keep their parameter offsets: torch.optim.SGD instead of Adam (m = the momentum buffer or
  // NULL, v unused); first_step: the host step count is 1 (used without step_dev)
  int sgd;
  float momentum, dampening;
  int nesterov, first_step;
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// wait until *p >= want (epochs only grow); bounded
__device__ __forceinline__ void spin_until(const uint32_t* p, uint32_t want) {
  const long long t0 = clock64();
  while ((int32_t)(ld_acquire_sys(p) - want) < 0) {
    __nanosleep(64);
    if (clock64() - t0 > 8000000000LL) __trap();       // ~4 s at 2 GHz: a peer never arrived
  }
}

// this rank's slice of [lo, hi) in units of 4 floats (the arena is padded to a multiple of 64)
__device__ __forceinline__ void slice_quads(const DpArgs& a, size_t& q0, size_t& q1) {
  const size_t n4 = (a.hi - a.lo) / 4, per = (n4 + a.world - 1) / a.world, base = a.lo / 4;
  q0 = base + per * a.rank;
  q1 = (per * (a.rank + 1) < n4 ? per * (a.rank + 1) : n4) + base;
}
// the arithmetic of adam_kernel (rowops.cu), element for element; lr and wd of the quad's parameter group (quad_hp)
__device__ __forceinline__ void adam_quad(const DpArgs& a, float lr, float wd, float bc1, float bc2_sqrt, const float* gg,
                                          float* w, float* mm, float* vv) {
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    float grad = gg[k];
    float wk = w[k];
    if (a.decoupled) wk *= 1.f - lr * wd;
    else if (wd != 0.f) grad += wd * wk;
    mm[k] = a.b1 * mm[k] + (1.f - a.b1) * grad;
    vv[k] = a.b2 * vv[k] + (1.f - a.b2) * grad * grad;
    w[k] = wk - (lr / bc1) * mm[k] / (sqrtf(vv[k]) / bc2_sqrt + a.eps);
  }
}
// Quad q (global, in units of 4 floats) never straddles a 64-element block: its group's lr (the step's lr times lr_mult) and
// weight decay, and whether it is frozen.  Without groups: the step's lr, the desc's weight decay, never frozen.
__device__ __forceinline__ bool quad_hp(const DpArgs& a, size_t q, float lr, float& lr_q, float& wd_q) {
  lr_q = lr;
  wd_q = a.wd;
  if (!a.groups) return false;
  const int k = a.block_group[q >> 4];
  if (a.groups->frozen[k]) return true;
  lr_q = lr * a.groups->lr_mult[k];
  wd_q = a.groups->weight_decay[k];
  return false;
}
__device__ __forceinline__ void clear_grad_quad(const DpArgs& a, size_t q) {
  for (int p = 0; p < a.world; ++p) reinterpret_cast<float4*>(a.slab[p] + a.off_grad)[q] = make_float4(0.f, 0.f, 0.f, 0.f);
}
// local moments, then the all-gather: the owner writes its slice (fp32 + bf16 shadow) into every arena
__device__ __forceinline__ void store_and_gather(const DpArgs& a, size_t q, const float* w, const float* mm, const float* vv,
                                                 int zero_remote) {
  reinterpret_cast<float4*>(a.m)[q] = make_float4(mm[0], mm[1], mm[2], mm[3]);
  reinterpret_cast<float4*>(a.v)[q] = make_float4(vv[0], vv[1], vv[2], vv[3]);
  const float4 wn = make_float4(w[0], w[1], w[2], w[3]);
  __nv_bfloat162 s0 = __floats2bfloat162_rn(w[0], w[1]), s1 = __floats2bfloat162_rn(w[2], w[3]);
  uint2 sh; sh.x = *reinterpret_cast<uint32_t*>(&s0); sh.y = *reinterpret_cast<uint32_t*>(&s1);
  for (int p = 0; p < a.world; ++p) {
    reinterpret_cast<float4*>(a.slab[p] + a.off_param)[q] = wn;
    if (a.off_shadow != (size_t)-1) reinterpret_cast<uint2*>(a.slab[p] + a.off_shadow)[q] = sh;
    if (zero_remote) reinterpret_cast<float4*>(a.slab[p] + a.off_grad)[q] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}
// the arithmetic of sgd_kernel (rowops.cu), element for element: bb is the momentum buffer (unused without momentum)
__device__ __forceinline__ void sgd_quad(const DpArgs& a, float lr, float wd, bool first, const float* gg, float* w,
                                         float* bb) {
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    float d = gg[k];
    if (wd != 0.f) d += wd * w[k];
    if (a.m) {
      bb[k] = first ? d : a.momentum * bb[k] + (1.f - a.dampening) * d;
      d = a.nesterov ? d + a.momentum * bb[k] : bb[k];
    }
    w[k] = w[k] - lr * d;
  }
}
// SGD's store_and_gather: the local momentum buffer (if any), then the same all-gather of fp32 + bf16 shadow
__device__ __forceinline__ void store_and_gather_sgd(const DpArgs& a, size_t q, const float* w, const float* bb,
                                                     int zero_remote) {
  if (a.m) reinterpret_cast<float4*>(a.m)[q] = make_float4(bb[0], bb[1], bb[2], bb[3]);
  const float4 wn = make_float4(w[0], w[1], w[2], w[3]);
  __nv_bfloat162 s0 = __floats2bfloat162_rn(w[0], w[1]), s1 = __floats2bfloat162_rn(w[2], w[3]);
  uint2 sh; sh.x = *reinterpret_cast<uint32_t*>(&s0); sh.y = *reinterpret_cast<uint32_t*>(&s1);
  for (int p = 0; p < a.world; ++p) {
    reinterpret_cast<float4*>(a.slab[p] + a.off_param)[q] = wn;
    if (a.off_shadow != (size_t)-1) reinterpret_cast<uint2*>(a.slab[p] + a.off_shadow)[q] = sh;
    if (zero_remote) reinterpret_cast<float4*>(a.slab[p] + a.off_grad)[q] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}
// 3. everything this rank wrote is visible system-wide before it says so: the CTA barrier orders the CTA's writes before
//    thread 0's system-scope fence (cumulativity), which precedes the grid counter; one fence per CTA, not per thread.  The
//    last CTA announces "my slice of epoch e is in your arena" and leaves when every rank did, then advances the epoch.
__device__ __forceinline__ void finish_epoch(const DpArgs& a, uint32_t* grid_ctr, const uint32_t* done, uint32_t* epoch_w,
                                             uint32_t e) {
  __syncthreads();
  __shared__ uint32_t s_last;
  if (threadIdx.x == 0) {
    __threadfence_system();
    s_last = atomicAdd(grid_ctr, 1u) == gridDim.x - 1 ? 1u : 0u;
  }
  __syncthreads();
  if (!s_last) return;
  // the last CTA of this rank: every CTA's writes are fenced
  if (threadIdx.x < a.world) {
    __threadfence_system();                       // acquire side of the counter: the other CTAs' fenced writes, then the flag
    st_release_sys(reinterpret_cast<uint32_t*>(a.slab[threadIdx.x] + a.off_flags) + a.channel * kChanWords + kMaxRanks + a.rank, e);
    spin_until(done + threadIdx.x, e);           // ... and every rank's slice is in THIS arena before the launch completes
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    *grid_ctr = 0;
    *epoch_w = e;
    __threadfence();
  }
}

__global__ void __launch_bounds__(256) dp_reduce_adam_kernel(const DpArgs a) {
  EGOT2_PDL_ENTER();
  uint32_t* my_flags = reinterpret_cast<uint32_t*>(a.slab[a.rank] + a.off_flags) + a.channel * kChanWords;
  uint32_t* arrive = my_flags;                 // arrive[p]: rank p's gradients of that epoch are complete
  uint32_t* done = my_flags + kMaxRanks;       // done[p]:   rank p's slice of that epoch is in this rank's arena
  uint32_t* epoch_w = my_flags + 2 * kMaxRanks;
  uint32_t* grid_ctr = my_flags + 2 * kMaxRanks + 1;
  const uint32_t e = *reinterpret_cast<volatile uint32_t*>(epoch_w) + 1;      // advanced by the last CTA of this launch

  // 1. announce (the backward kernels that produced the gradients precede this launch in stream order)
  if (blockIdx.x == 0 && threadIdx.x < a.world) {
    st_release_sys(reinterpret_cast<uint32_t*>(a.slab[threadIdx.x] + a.off_flags) + a.channel * kChanWords + a.rank, e);
  }
  // 2. every CTA waits for every rank's announcement
  if (threadIdx.x < a.world) spin_until(arrive + threadIdx.x, e);
  __syncthreads();

  float bc1 = a.bc1, bc2_sqrt = a.bc2_sqrt;
  if (a.step_dev) {
    const float t = (float)*a.step_dev;
    bc1 = 1.f - powf(a.b1, t);
    bc2_sqrt = sqrtf(1.f - powf(a.b2, t));
  }
  const float lr = a.lr_dev ? *a.lr_dev : a.lr;
  const float inv_world = 1.f / (float)a.world;
  size_t q0, q1;
  slice_quads(a, q0, q1);
  constexpr int U = 2;                           // independent quads per thread and iteration: 2 * world loads in flight
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t qb = q0 + blockIdx.x * (size_t)blockDim.x + threadIdx.x; qb < q1; qb += stride * U) {
    float4 g[U], w4[U], m4[U], v4[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t q = qb + u * stride;
      g[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (q < q1) {
        for (int p = 0; p < a.world; ++p) {      // rank order: the same sum on whichever rank owns the slice
          const float4 x = reinterpret_cast<const float4*>(a.slab[p] + a.off_grad)[q];
          g[u].x += x.x; g[u].y += x.y; g[u].z += x.z; g[u].w += x.w;
        }
        w4[u] = reinterpret_cast<const float4*>(a.slab[a.rank] + a.off_param)[q];
        m4[u] = reinterpret_cast<float4*>(a.m)[q];
        v4[u] = reinterpret_cast<float4*>(a.v)[q];
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t q = qb + u * stride;
      if (q >= q1) continue;
      float lr_q, wd_q;
      if (quad_hp(a, q, lr, lr_q, wd_q)) {       // frozen: parameters, shadow and moments stay; the gradient is cleared
        if (a.zero_remote) clear_grad_quad(a, q);
        continue;
      }
      float gg[4] = {g[u].x * inv_world, g[u].y * inv_world, g[u].z * inv_world, g[u].w * inv_world};
      float w[4] = {w4[u].x, w4[u].y, w4[u].z, w4[u].w};
      float mm[4] = {m4[u].x, m4[u].y, m4[u].z, m4[u].w}, vv[4] = {v4[u].x, v4[u].y, v4[u].z, v4[u].w};
      adam_quad(a, lr_q, wd_q, bc1, bc2_sqrt, gg, w, mm, vv);
      store_and_gather(a, q, w, mm, vv, a.zero_remote);
    }
  }
  finish_epoch(a, grid_ctr, done, epoch_w, e);
}

// dp_reduce_adam_kernel with the SGD update: the same flags, slice, rank-order sum and frozen quads
__global__ void __launch_bounds__(256) dp_reduce_sgd_kernel(const DpArgs a) {
  EGOT2_PDL_ENTER();
  uint32_t* my_flags = reinterpret_cast<uint32_t*>(a.slab[a.rank] + a.off_flags) + a.channel * kChanWords;
  uint32_t* arrive = my_flags;
  uint32_t* done = my_flags + kMaxRanks;
  uint32_t* epoch_w = my_flags + 2 * kMaxRanks;
  uint32_t* grid_ctr = my_flags + 2 * kMaxRanks + 1;
  const uint32_t e = *reinterpret_cast<volatile uint32_t*>(epoch_w) + 1;

  if (blockIdx.x == 0 && threadIdx.x < a.world) {
    st_release_sys(reinterpret_cast<uint32_t*>(a.slab[threadIdx.x] + a.off_flags) + a.channel * kChanWords + a.rank, e);
  }
  if (threadIdx.x < a.world) spin_until(arrive + threadIdx.x, e);
  __syncthreads();

  const bool first = a.step_dev ? *a.step_dev == 1 : a.first_step != 0;
  const float lr = a.lr_dev ? *a.lr_dev : a.lr;
  const float inv_world = 1.f / (float)a.world;
  size_t q0, q1;
  slice_quads(a, q0, q1);
  constexpr int U = 2;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t qb = q0 + blockIdx.x * (size_t)blockDim.x + threadIdx.x; qb < q1; qb += stride * U) {
    float4 g[U], w4[U], b4[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t q = qb + u * stride;
      g[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      b4[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (q < q1) {
        for (int p = 0; p < a.world; ++p) {      // rank order, as dp_reduce_adam_kernel
          const float4 x = reinterpret_cast<const float4*>(a.slab[p] + a.off_grad)[q];
          g[u].x += x.x; g[u].y += x.y; g[u].z += x.z; g[u].w += x.w;
        }
        w4[u] = reinterpret_cast<const float4*>(a.slab[a.rank] + a.off_param)[q];
        if (a.m && !first) b4[u] = reinterpret_cast<float4*>(a.m)[q];
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t q = qb + u * stride;
      if (q >= q1) continue;
      float lr_q, wd_q;
      if (quad_hp(a, q, lr, lr_q, wd_q)) {       // frozen: parameters, shadow and buffer stay; the gradient is cleared
        if (a.zero_remote) clear_grad_quad(a, q);
        continue;
      }
      float gg[4] = {g[u].x * inv_world, g[u].y * inv_world, g[u].z * inv_world, g[u].w * inv_world};
      float w[4] = {w4[u].x, w4[u].y, w4[u].z, w4[u].w};
      float bb[4] = {b4[u].x, b4[u].y, b4[u].z, b4[u].w};
      sgd_quad(a, lr_q, wd_q, first, gg, w, bb);
      store_and_gather_sgd(a, q, w, bb, a.zero_remote);
    }
  }
  finish_epoch(a, grid_ctr, done, epoch_w, e);
}

// ---- guarded exchange (egot2_dp_desc.guard): the global norm must be known before any rank updates its slice, so the
// exchange runs as two launches on the same channel and epoch.
// Phase A: announce / wait as above; reduce this rank's slice in rank order and write g = (1/N) * sum into the LOCAL gradient
// arena (only the owner ever reads its slice, so in place is safe; zero_remote clears the peers' copies, not this one); sum
// the slice's squares in fp64 (per CTA, then the last CTA in CTA order); publish that partial to every peer; wait for all N
// and add them in rank order, so every rank computes the identical total_norm / coef / skip.
__global__ void __launch_bounds__(256) dp_guard_reduce_kernel(const DpArgs a) {
  EGOT2_PDL_ENTER();
  uint32_t* my_flags = reinterpret_cast<uint32_t*>(a.slab[a.rank] + a.off_flags) + a.channel * kChanWords;
  uint32_t* arrive = my_flags;
  uint32_t* epoch_w = my_flags + 2 * kMaxRanks;
  uint32_t* ctr_a = my_flags + kWordCtrA;
  uint32_t* norm_arrive = my_flags + kWordNormArrive;
  const double* norm_part = reinterpret_cast<const double*>(my_flags + kWordNormPart);
  double* cta_part = reinterpret_cast<double*>(reinterpret_cast<uint32_t*>(a.slab[a.rank] + a.off_flags) + kFlagWords) +
                     a.channel * kMaxCtas;
  const uint32_t e = *reinterpret_cast<volatile uint32_t*>(epoch_w) + 1;      // phase B's last CTA advances it

  if (blockIdx.x == 0 && threadIdx.x < a.world) {
    st_release_sys(reinterpret_cast<uint32_t*>(a.slab[threadIdx.x] + a.off_flags) + a.channel * kChanWords + a.rank, e);
  }
  if (threadIdx.x < a.world) spin_until(arrive + threadIdx.x, e);
  __syncthreads();

  const float inv_world = 1.f / (float)a.world;
  size_t q0, q1;
  slice_quads(a, q0, q1);
  constexpr int U = 2;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  double s = 0.0;
  for (size_t qb = q0 + blockIdx.x * (size_t)blockDim.x + threadIdx.x; qb < q1; qb += stride * U) {
    float4 g[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t q = qb + u * stride;
      g[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (q < q1) {
        for (int p = 0; p < a.world; ++p) {      // rank order, as dp_reduce_adam_kernel
          const float4 x = reinterpret_cast<const float4*>(a.slab[p] + a.off_grad)[q];
          g[u].x += x.x; g[u].y += x.y; g[u].z += x.z; g[u].w += x.w;
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t q = qb + u * stride;
      if (q >= q1) continue;
      const float4 gg = make_float4(g[u].x * inv_world, g[u].y * inv_world, g[u].z * inv_world, g[u].w * inv_world);
      reinterpret_cast<float4*>(a.slab[a.rank] + a.off_grad)[q] = gg;
      if (!(a.groups && a.groups->frozen[a.block_group[q >> 4]])) {      // frozen groups stay out of the norm
        s += (double)gg.x * gg.x; s += (double)gg.y * gg.y; s += (double)gg.z * gg.z; s += (double)gg.w * gg.w;
      }
      if (a.zero_remote)
        for (int p = 0; p < a.world; ++p)
          if (p != a.rank) reinterpret_cast<float4*>(a.slab[p] + a.off_grad)[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  __shared__ double sh[8];
  __shared__ uint32_t s_last;
  __shared__ double s_part;
  s = block_sum_f64(s, sh);
  if (threadIdx.x == 0) {
    cta_part[blockIdx.x] = s;
    __threadfence_system();              // also orders this CTA's zero_remote stores before phase B's done flags
    s_last = atomicAdd(ctr_a, 1u) == gridDim.x - 1 ? 1u : 0u;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  double t = 0.0;
  for (int c = threadIdx.x; c < (int)gridDim.x; c += blockDim.x) t += reinterpret_cast<volatile const double*>(cta_part)[c];
  t = block_sum_f64(t, sh);
  if (threadIdx.x == 0) s_part = t;
  __syncthreads();
  if (threadIdx.x < a.world) {           // publish this rank's partial to every peer, then wait for every peer's
    uint32_t* peer_flags = reinterpret_cast<uint32_t*>(a.slab[threadIdx.x] + a.off_flags) + a.channel * kChanWords;
    reinterpret_cast<double*>(peer_flags + kWordNormPart)[a.rank] = s_part;
    st_release_sys(peer_flags + kWordNormArrive + a.rank, e);       // release: the partial is visible before the flag
    spin_until(norm_arrive + threadIdx.x, e);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = 0.0;
    for (int p = 0; p < a.world; ++p) tot += reinterpret_cast<volatile const double*>(norm_part)[p];
    grad_guard_finalize(tot, 1.f, a.guard, const_cast<int32_t*>(a.step_dev));
    *ctr_a = 0;
    __threadfence();
  }
}

// Phase B: Adam on this rank's slice with the gradient phase A left in the local arena times guard->coef, the all-gather and
// the done flags; on a skip nothing is updated or gathered (every rank still holds the same parameters) and only the local
// slice of the gradient is cleared (zero_remote).
__global__ void __launch_bounds__(256) dp_guard_adam_kernel(const DpArgs a) {
  EGOT2_PDL_ENTER();
  uint32_t* my_flags = reinterpret_cast<uint32_t*>(a.slab[a.rank] + a.off_flags) + a.channel * kChanWords;
  uint32_t* done = my_flags + kMaxRanks;
  uint32_t* epoch_w = my_flags + 2 * kMaxRanks;
  uint32_t* grid_ctr = my_flags + 2 * kMaxRanks + 1;
  const uint32_t e = *reinterpret_cast<volatile uint32_t*>(epoch_w) + 1;
  const bool skip = a.guard->skip != 0;
  const float coef = a.guard->coef;
  float bc1 = a.bc1, bc2_sqrt = a.bc2_sqrt;
  if (a.step_dev) {
    const float t = (float)*a.step_dev;
    bc1 = 1.f - powf(a.b1, t);
    bc2_sqrt = sqrtf(1.f - powf(a.b2, t));
  }
  const float lr = a.lr_dev ? *a.lr_dev : a.lr;
  size_t q0, q1;
  slice_quads(a, q0, q1);
  float4* grad = reinterpret_cast<float4*>(a.slab[a.rank] + a.off_grad);
  for (size_t q = q0 + blockIdx.x * (size_t)blockDim.x + threadIdx.x; q < q1; q += (size_t)gridDim.x * blockDim.x) {
    float lr_q, wd_q;
    if (!skip && !quad_hp(a, q, lr, lr_q, wd_q)) {
      const float4 g4 = grad[q], w4 = reinterpret_cast<const float4*>(a.slab[a.rank] + a.off_param)[q];
      const float4 m4 = reinterpret_cast<float4*>(a.m)[q], v4 = reinterpret_cast<float4*>(a.v)[q];
      float gg[4] = {g4.x * coef, g4.y * coef, g4.z * coef, g4.w * coef};
      float w[4] = {w4.x, w4.y, w4.z, w4.w};
      float mm[4] = {m4.x, m4.y, m4.z, m4.w}, vv[4] = {v4.x, v4.y, v4.z, v4.w};
      adam_quad(a, lr_q, wd_q, bc1, bc2_sqrt, gg, w, mm, vv);
      store_and_gather(a, q, w, mm, vv, 0);
    }
    if (a.zero_remote) grad[q] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  finish_epoch(a, grid_ctr, done, epoch_w, e);
}

// Phase B of the guarded exchange with the SGD update (phase A, dp_guard_reduce_kernel, does not depend on the optimizer).
// The step count phase A left is that of the applied steps, so a skipped first step leaves the buffer's initialisation to
// the next applied one.
__global__ void __launch_bounds__(256) dp_guard_sgd_kernel(const DpArgs a) {
  EGOT2_PDL_ENTER();
  uint32_t* my_flags = reinterpret_cast<uint32_t*>(a.slab[a.rank] + a.off_flags) + a.channel * kChanWords;
  uint32_t* done = my_flags + kMaxRanks;
  uint32_t* epoch_w = my_flags + 2 * kMaxRanks;
  uint32_t* grid_ctr = my_flags + 2 * kMaxRanks + 1;
  const uint32_t e = *reinterpret_cast<volatile uint32_t*>(epoch_w) + 1;
  const bool skip = a.guard->skip != 0;
  const float coef = a.guard->coef;
  const bool first = a.step_dev ? *a.step_dev == 1 : a.first_step != 0;
  const float lr = a.lr_dev ? *a.lr_dev : a.lr;
  size_t q0, q1;
  slice_quads(a, q0, q1);
  float4* grad = reinterpret_cast<float4*>(a.slab[a.rank] + a.off_grad);
  for (size_t q = q0 + blockIdx.x * (size_t)blockDim.x + threadIdx.x; q < q1; q += (size_t)gridDim.x * blockDim.x) {
    float lr_q, wd_q;
    if (!skip && !quad_hp(a, q, lr, lr_q, wd_q)) {
      const float4 g4 = grad[q], w4 = reinterpret_cast<const float4*>(a.slab[a.rank] + a.off_param)[q];
      const float4 b4 = a.m && !first ? reinterpret_cast<float4*>(a.m)[q] : make_float4(0.f, 0.f, 0.f, 0.f);
      float gg[4] = {g4.x * coef, g4.y * coef, g4.z * coef, g4.w * coef};
      float w[4] = {w4.x, w4.y, w4.z, w4.w};
      float bb[4] = {b4.x, b4.y, b4.z, b4.w};
      sgd_quad(a, lr_q, wd_q, first, gg, w, bb);
      store_and_gather_sgd(a, q, w, bb, 0);
    }
    if (a.zero_remote) grad[q] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  finish_epoch(a, grid_ctr, done, epoch_w, e);
}

}  // namespace
}  // namespace egot2

using namespace egot2;

// ---------------------------------------------------------------- slabs and their IPC handles
extern "C" int egot2_peer_alloc(size_t bytes, void** ptr) {
  EGOT2_CHECK(ptr && bytes > 0, "peer_alloc: bad arguments");
  EGOT2_CUDA(cudaMalloc(ptr, bytes));
  EGOT2_CUDA(cudaMemset(*ptr, 0, bytes));
  return 0;
}
extern "C" int egot2_peer_free(void* ptr) {
  if (ptr) EGOT2_CUDA(cudaFree(ptr));
  return 0;
}
extern "C" int egot2_peer_handle_bytes(void) { return (int)sizeof(cudaIpcMemHandle_t); }
extern "C" int egot2_peer_export(void* ptr, void* handle_out) {
  EGOT2_CHECK(ptr && handle_out, "peer_export: bad arguments");
  cudaIpcMemHandle_t h;
  EGOT2_CUDA(cudaIpcGetMemHandle(&h, ptr));
  memcpy(handle_out, &h, sizeof(h));
  return 0;
}
extern "C" int egot2_peer_import(const void* handle, void** ptr) {
  EGOT2_CHECK(handle && ptr, "peer_import: bad arguments");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  EGOT2_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return 0;
}
extern "C" int egot2_peer_unimport(void* ptr) {
  if (ptr) EGOT2_CUDA(cudaIpcCloseMemHandle(ptr));
  return 0;
}
extern "C" size_t egot2_dp_flag_bytes(void) { return kFlagWords * sizeof(uint32_t) + kChannels * kMaxCtas * sizeof(double); }

static int dp_launch(const egot2_dp_desc* d, long long lo, long long hi, int channel, void* stream);
extern "C" int egot2_dp_reduce_adam(const egot2_dp_desc* d, void* stream) { return dp_launch(d, 0, d ? d->numel : 0, 0, stream); }
extern "C" int egot2_dp_reduce_adam_range(const egot2_dp_desc* d, int64_t lo, int64_t hi, int32_t channel, void* stream) {
  return dp_launch(d, lo, hi, channel, stream);
}
static int dp_launch(const egot2_dp_desc* d, long long lo, long long hi, int channel, void* stream) {
  EGOT2_CHECK(d && d->world >= 1 && d->world <= kMaxRanks && d->rank >= 0 && d->rank < d->world, "dp_reduce_adam: world/rank");
  EGOT2_CHECK(d->numel > 0 && d->numel % 4 == 0, "dp_reduce_adam: arena (numel %% 4 == 0)");
  if (d->sgd) {
    EGOT2_CHECK(d->momentum >= 0.f && isfinite(d->momentum) && isfinite(d->dampening) && !d->decoupled,
                "dp_reduce_adam (sgd): momentum %g / dampening %g / decoupled %d", d->momentum, d->dampening, d->decoupled);
    EGOT2_CHECK(!d->nesterov || (d->momentum > 0.f && d->dampening == 0.f),
                "dp_reduce_adam (sgd): nesterov needs momentum > 0 and dampening 0");
    EGOT2_CHECK((d->exp_avg == nullptr) == (d->momentum == 0.f),
                "dp_reduce_adam (sgd): exp_avg (the momentum buffer) must be given exactly when momentum != 0");
  } else {
    EGOT2_CHECK(d->exp_avg && d->exp_avg_sq, "dp_reduce_adam: moments");
  }
  EGOT2_CHECK(lo >= 0 && hi <= d->numel && lo <= hi && lo % 4 == 0 && hi % 4 == 0 && channel >= 0 && channel < kChannels,
              "dp_reduce_adam: range [%lld, %lld) / channel %d", lo, hi, channel);
  if (lo == hi) return 0;
  DpArgs a;
  a.world = d->world; a.rank = d->rank; a.n = (size_t)d->numel;
  a.lo = (size_t)lo; a.hi = (size_t)hi; a.channel = channel;
  for (int p = 0; p < d->world; ++p) {
    EGOT2_CHECK(d->slab[p] != nullptr, "dp_reduce_adam: slab of rank %d missing", p);
    a.slab[p] = (char*)d->slab[p];
  }
  for (int p = d->world; p < kMaxRanks; ++p) a.slab[p] = nullptr;
  a.off_param = (size_t)d->off_param; a.off_grad = (size_t)d->off_grad;
  a.off_shadow = d->off_shadow < 0 ? (size_t)-1 : (size_t)d->off_shadow;
  a.off_flags = (size_t)d->off_flags;
  EGOT2_CHECK(a.off_param % 16 == 0 && a.off_grad % 16 == 0 && (d->off_shadow < 0 || d->off_shadow % 8 == 0) && a.off_flags % 16 == 0,
              "dp_reduce_adam: slab offsets must be 16-byte aligned");
  a.m = d->exp_avg; a.v = d->exp_avg_sq;
  a.lr = d->lr; a.b1 = d->beta1; a.b2 = d->beta2; a.eps = d->eps; a.wd = d->weight_decay;
  a.bc1 = 1.f - powf(d->beta1, (float)d->step);
  a.bc2_sqrt = sqrtf(1.f - powf(d->beta2, (float)d->step));
  a.step_dev = d->step_dev;
  a.lr_dev = d->lr_dev;
  a.decoupled = d->decoupled;
  a.guard = d->guard;
  EGOT2_CHECK(!d->groups == !d->block_group, "dp_reduce_adam: groups and block_group go together");
  a.groups = d->groups;
  a.block_group = d->block_group;
  a.sgd = d->sgd ? 1 : 0;
  a.momentum = d->momentum;
  a.dampening = d->dampening;
  a.nesterov = d->nesterov ? 1 : 0;
  a.first_step = d->step == 1 ? 1 : 0;
  EGOT2_CHECK(!a.sgd || d->step >= 1 || d->step_dev, "dp_reduce_adam (sgd): step must be >= 1");
  // a few CTAs per rank: the message is latency-bound, and the spinning CTAs must never crowd out other work
  const size_t per4 = ((size_t)(hi - lo) / 4 + d->world - 1) / d->world;
  // latency-bound for the small arenas (a few CTAs), bandwidth-bound for the large ones (two waves of resident CTAs)
  int grid = (int)((per4 + 511) / 512);
  const int cap = sm_count() * 4;
  if (grid > cap) grid = cap;
  if (grid > kMaxCtas) grid = kMaxCtas;
  if (grid < 1) grid = 1;
  a.zero_remote = d->zero_grads_remote ? 1 : 0;
  cudaStream_t st = (cudaStream_t)stream;
  ProfScope prof(st, a.sgd ? "dp_reduce_sgd n%lld world%d ch%d" : "dp_reduce_adam n%lld world%d ch%d", (long long)(hi - lo),
                 d->world, channel);
  if (a.guard) {
    launch(dp_guard_reduce_kernel, dim3(grid), dim3(256), 0, st, a);
    EGOT2_LAUNCH_CHECK();
    launch(a.sgd ? dp_guard_sgd_kernel : dp_guard_adam_kernel, dim3(grid), dim3(256), 0, st, a);
  } else {
    launch(a.sgd ? dp_reduce_sgd_kernel : dp_reduce_adam_kernel, dim3(grid), dim3(256), 0, st, a);
  }
  EGOT2_LAUNCH_CHECK();
  return 0;
}
