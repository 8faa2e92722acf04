// ops.h — internal launchers shared by the stage-level C ABI (api.cu).
#pragma once
#include "common.cuh"

namespace egot2 {

// C[M,N] = epilogue( op(A)[M,K] . op(B)[K,N] )
struct GemmArgs {
  int M = 0, N = 0, K = 0;
  const void* A = nullptr; int lda = 0; int trans_a = 0;   // trans_a: stored (K,M)
  const void* B = nullptr; int ldb = 0; int trans_b = 0;   // trans_b: stored (N,K)  [nn.Linear weight]
  void* C = nullptr;       int ldc = 0;
  int in_dtype = EGOT2_F32;      // dtype of A and B
  int out_dtype = EGOT2_F32;     // dtype of C (and of residual / mask)
  // storage-row remap (segment scatter/gather inside (B,T,H) tensors):
  //   physical row = (r / rpg) * gstride + (r % rpg)   when rpg > 0
  int a_rpg = 0, a_gstride = 0;
  int b_rpg = 0, b_gstride = 0;
  int c_rpg = 0, c_gstride = 0;
  // epilogue, applied in this order
  const float* bias = nullptr;   // + bias[n]
  int relu = 0;                  // max(.,0)
  const void* mask = nullptr; int ldm = 0; float mask_scale = 1.f;   // * (mask[m,n] > 0 ? mask_scale : 0)
  float p_drop = 0.f; uint64_t drop_key = 0;                         // * dropmask(m*N+n)/(1-p)
  int trans_c = 0;               // fp32 split-K accumulation into the TRANSPOSE: element (m, n) is added to C[n * ldc + m] (tcgen05 kernel only)
  int drop_bit_mode = 0;         // FFN hidden site: one random bit per element when p == 0.5 (common.cuh drop_keep)
  const void* residual = nullptr; int ldr = 0;                       // + residual[m,n]
  int accumulate = 0;            // C += value (fp32 C only); split-K uses atomics
  int split_k = 1;
  // split_stride > 0 (fp32 C, no accumulate): split z WRITES its partial product to C + z * split_stride (elements) instead
  // of adding atomically - a deterministic split-K whose slabs the consumer sums in a fixed order (embed stage); the number
  // of splits actually launched (<= split_k) is returned through *splits_out
  long long split_stride = 0;
  int* splits_out = nullptr;
  // LayerNorm fused behind the epilogue (tcgen05 path only, see gemm_sm100_ln_ok): ln_out[row] = LN(C[row]) * ln_g + ln_b
  // (+ ln_table[(row + ln_row0) % ln_table_rows]) (* dropout(ln_p_drop)); statistics to ln_stat[row + ln_row0]; rows = C's storage rows
  const float* ln_g = nullptr; const float* ln_b = nullptr; float ln_eps = 1e-5f;
  void* ln_out = nullptr; float* ln_stat = nullptr; const float* ln_table = nullptr; int ln_table_rows = 0; int ln_row0 = 0;
  float ln_p_drop = 0.f; uint64_t ln_drop_key = 0;
};
bool gemm_sm100_ln_ok(const GemmArgs& a);
int gemm(const GemmArgs& a, cudaStream_t st);          // dispatch: tcgen05 (bf16, supported shapes) or CUDA-core
int gemm_simt(const GemmArgs& a, cudaStream_t st);     // gemm_simt.cu
int gemm_sm100(const GemmArgs& a, cudaStream_t st);    // gemm_sm100.cu; returns -1 if the shape is not handled
int suggest_split_k(int M, int N, int K);
// which implementation handled the last bf16 GEMM ("tcgen05" | "simt"); diagnostics only
const char* gemm_last_impl();

// y = LN(x [+ res]) * g + b (+ table[row % table_rows]); optional dropout after; stat = (mean, rstd)
struct LayerNormArgs {
  int rows = 0, H = 0; int dtype = EGOT2_F32;
  const void* x = nullptr; const float* g = nullptr; const float* b = nullptr; float eps = 1e-5f;
  void* y = nullptr; float* stat = nullptr;
  const float* table = nullptr; int table_rows = 0;
  float p_drop = 0.f; uint64_t drop_key = 0;
  int x_is_f32 = 0;              // x is fp32 regardless of dtype (pooled vectors)
};
int layernorm_fwd(const LayerNormArgs& a, cudaStream_t st);
// dx = LN'(dy) (+ dres);  dg += sum dy*xhat;  db += sum dy
struct LayerNormBwdArgs {
  int rows = 0, H = 0; int dtype = EGOT2_F32;
  const void* x = nullptr; const float* stat = nullptr; const float* g = nullptr;
  const void* dy = nullptr;      // dtype (fp32 if dy_is_f32)
  void* dx = nullptr;            // dtype (fp32 if dx_is_f32); may alias dy
  const void* dres = nullptr;    // optional (dtype): dx += dres, the gradient arriving through a residual branch
  float* dg = nullptr; float* db = nullptr;
  int x_is_f32 = 0; int dx_is_f32 = 0; int dy_is_f32 = 0;
  // fused dropout sites (bf16 vector path; the generic path emulates them with extra launches):
  float dy_p_drop = 0.f; uint64_t dy_drop_key = 0;       // dy *= dropmask(row*H+c)/(1-p) on load (a dropout that FOLLOWED the LN)
  float* dcol = nullptr;         // optional (H) +=: column sums of the gradient handed on (dx2 if given, else dx) = the bias
                                 // gradient of the Linear layer that produced the LN input's residual branch
  void* dx2 = nullptr; float dx2_p_drop = 0.f; uint64_t dx2_drop_key = 0;   // second output: dx * dropmask/(1-p) (a dropout that PRECEDED
                                                                            // the residual add feeding this LN)
};
int layernorm_bwd(const LayerNormBwdArgs& a, cudaStream_t st);

int attention_simt_fwd(int dtype, int B, int T, int H, int heads, const void* qkv, void* out, float* lse,
                       float p_drop, uint64_t drop_key, cudaStream_t st);
int attention_simt_bwd(int dtype, int B, int T, int H, int heads, const void* qkv, const void* out, const float* lse,
                       const void* dout, void* dqkv, float p_drop, uint64_t drop_key, void* ws, size_t ws_bytes,
                       cudaStream_t st);
bool attention_mma_supported(int dtype, int T, int H, int heads);           // attention_mma.cu (bf16, T <= 128)
int attention_mma_fwd(int B, int T, int H, int heads, const void* qkv, void* out, float* lse, float p_drop,
                      uint64_t drop_key, cudaStream_t st);
int attention_mma_bwd(int B, int T, int H, int heads, const void* qkv, const void* out, const float* lse,
                      const void* dout, void* dqkv, float p_drop, uint64_t drop_key, cudaStream_t st);
// attention_long.cu: tensor-core kernels for 128 < T <= 512 (bf16, head dim 16 / 32 / 64; online softmax over key blocks)
bool attention_long_supported(int dtype, int T, int H, int heads);
int attention_long_fwd(int B, int T, int H, int heads, const void* qkv, void* out, float* lse, float p_drop, uint64_t drop_key,
                       cudaStream_t st);
int attention_long_bwd(int B, int T, int H, int heads, const void* qkv, const void* out, const float* lse, const void* dout,
                       void* dqkv, float p_drop, uint64_t drop_key, cudaStream_t st);
// attention_wide.cu: head dim > 128 over T <= 32 tokens (LTA 2-task at H = 2048, 4 heads)
int attention_wide_fwd(int dtype, int B, int T, int H, int heads, const void* qkv, void* out, float* lse, float p_drop,
                       uint64_t drop_key, cudaStream_t st);
int attention_wide_bwd(int dtype, int B, int T, int H, int heads, const void* qkv, const void* out, const float* lse,
                       const void* dout, void* dqkv, float p_drop, uint64_t drop_key, cudaStream_t st);
int attention_fwd(int dtype, int B, int T, int H, int heads, const void* qkv, void* out, float* lse,
                  float p_drop, uint64_t drop_key, cudaStream_t st);
size_t attention_bwd_workspace(int dtype, int B, int T, int H, int heads);
int attention_bwd(int dtype, int B, int T, int H, int heads, const void* qkv, const void* out, const float* lse,
                  const void* dout, void* dqkv, float p_drop, uint64_t drop_key, void* ws, size_t ws_bytes,
                  cudaStream_t st);

// EgoT2-g decoder attention (attention_small.cu): S query tokens per row against M keys per row
struct SmallAttnArgs {
  int dtype = EGOT2_F32;
  int rows = 0, S = 0, M = 0, H = 0, heads = 0, causal = 0;
  const void* q = nullptr; int ldq = 0;                       // (rows*S, .) queries, head h = columns h*dh..
  const void* k = nullptr; const void* v = nullptr; int ldkv = 0;   // key/value rows, see the row mapping
  int kv_inner = 1, kv_outer = 0, kv_jstride = 1, kv_istride = 0;
  void* out = nullptr; int ldo = 0;                           // (rows*S, H)
  float* lse = nullptr;                                       // (rows*heads*S) or null
  float p_drop = 0.f; uint64_t drop_key = 0;
  // backward
  const void* dout = nullptr;                                 // (rows*S, .) with ldo
  float* dq = nullptr; int ld_dq = 0;                         // fp32, += (atomics)
  float* dk = nullptr; float* dv = nullptr; int ld_dkv = 0;   // fp32, += (atomics), indexed by kv row
};
int small_attn_fwd(const SmallAttnArgs& a, cudaStream_t st);
int small_attn_bwd(const SmallAttnArgs& a, cudaStream_t st);

// dtable[t,:] += sum_b dy[b,t,:]   (gradient of the (T,H) token table added after the embed LN)
// p_drop > 0: dy has NOT had the embedding dropout's mask applied yet; the kernel applies it while reading
// dtable[t,:] += sum_b dy[b,t,:] (dtable may be null); seg_out[k][:] += the same sums over segment k's tokens (null entries skipped)
struct SegOut { int n = 0; int tokens[EGOT2_MAX_SEG] = {}; float* out[EGOT2_MAX_SEG] = {}; };
int table_grad(int dtype, int B, int T, int H, const void* dy, float* dtable, const SegOut& so, float p_drop, uint64_t drop_key,
               cudaStream_t st);
// column sums: out[n] += sum_m x[m,n]   (bias gradients)
int colsum_accum(int dtype, int M, int N, const void* x, int ldx, int rpg, int gstride, float* out, cudaStream_t st);
int colsum_cast_bf16(int M, int N, const float* x, int ldx, void* y, int ldy, float* out, cudaStream_t st);   // y = bf16(x), out += colsum(x)
// in-place x *= dropmask/(1-p) over n elements (idx = linear element index)
int dropout_inplace(int dtype, void* x, size_t n, float p, uint64_t key, cudaStream_t st);
// pooled[b,:] = mean_t x[b,t,:]   or gather of the first row_tokens tokens (pool==0)
int pool_fwd(int dtype, int B, int T, int H, int pool, int row_tokens, const void* x, float* pooled, cudaStream_t st);
int pool_bwd(int dtype, int B, int T, int H, int pool, int row_tokens, const float* dpooled, void* dx, cudaStream_t st);
int cast_f32_to(int dtype, const float* src, void* dst, size_t n, cudaStream_t st);
int cast_to_f32(int dtype, const void* src, float* dst, size_t n, cudaStream_t st);
int zero_f32(float* p, size_t n, cudaStream_t st);
// x[i] = z[i] + table[i % table_elems]   (embed_extra.cu: the embed stage without LayerNorm)
int add_table(int dtype, size_t n, size_t table_elems, const void* z, const float* table, void* x, cudaStream_t st);
// embed stage after deterministic split-K projections (embed_extra.cu): sum of the slabs -> feature dropout -> z, LN,
// + table, embedding dropout -> x, one pass
bool embed_finish_supported(int dtype, int H);
struct EmbedSrc {      // where segment k's projected rows are: `splits` fp32 slabs of (B*tokens, H), or the bf16 features themselves
  int n = 0; int tok_begin[EGOT2_MAX_SEG] = {}; int tokens[EGOT2_MAX_SEG] = {}; int splits[EGOT2_MAX_SEG] = {};
  const float* slab[EGOT2_MAX_SEG] = {}; const void* direct[EGOT2_MAX_SEG] = {};
  int direct_f32[EGOT2_MAX_SEG] = {};      // the pass-through features are fp32 (caller hands fp32 features to a bf16 engine)
};
int embed_finish(int B, int T, int H, const EmbedSrc& src, int drop_tokens, float p_feat, uint64_t key_feat, const float* g,
                 const float* b, float eps, const float* table, float p_embed, uint64_t key_embed, void* z, float* stat, void* x,
                 cudaStream_t st);
// dst += a (+ b); a (and b) cleared (embed_extra.cu)
int sum_into_clear(float* dst, float* a, float* b, size_t n, cudaStream_t st);
// in-place dropout of the first `prefix` elements of every `period`-element clip (mask index = linear element index)
int dropout_prefix_inplace(int dtype, void* x, size_t n, size_t period, size_t prefix, float p, uint64_t key, cudaStream_t st);
// dst[r, 0..ld) = bf16(src[r, 0..n)) followed by zeros (ld >= n)
int cast_rows_f32_to_bf16(const float* src, int rows, int n, void* dst, int ld, cudaStream_t st);

// fused FFN block on tcgen05 (ffn_sm100.cu): x_out = LN2(x1 + drop2(drop(relu(x1 W1^T + b1)) W2^T + b2))
bool ffn_fused_supported(int dtype, int H, int FF);
int ffn_fused_fwd(int M, int FF, const void* x1, const void* W1, const float* b1, const void* W2, const float* b2,
                  const float* ln_g, const float* ln_b, float eps, void* hid, void* hmask, void* y2, float* stat2, void* x_out,
                  float p_drop, uint64_t key_ffn, uint64_t key_drop2, float* scratch, cudaStream_t st);
size_t ffn_scratch_bytes(int M);      // zeroed fp32 scratch that enables the FF-split of the last partial wave (may be 0)
// dhid = (d2 . W2) * gate(hmask) / (1-p);  d3 = dhid . W1 + (d1 ? d1 : d2);  db1 (optional) += column sums of dhid
int ffn_fused_bwd_dx(int M, int FF, const void* d2, const void* d1, const void* hmask, const void* W1, const void* W2,
                     float p_drop, void* dhid, void* d3, float* scratch, float* db1, cudaStream_t st);

// fused small heads (head_fused.cu): pool + LN + Linear(n_out <= 32) in one kernel per direction
bool head_fused_supported(const egot2_head_desc& d);
int head_fused_fwd(const egot2_head_desc& d, const egot2_head_in& in, const egot2_head_out& out, cudaStream_t st);
// fwd also emits the per-row loss terms + argmax when d.loss != NONE; bwd then derives d(loss)/d(logits) itself (written to
// `dlogits`, which is only READ when d.loss == NONE)
int loss_reduce(const egot2_head_desc& d, int rows, const float* row_loss, float* loss, cudaStream_t st);
int head_fused_bwd(const egot2_head_desc& d, const egot2_head_in& in, const egot2_head_out& saved, float* dlogits, float dloss_scale,
                   void* dx, const egot2_head_grads& g, cudaStream_t st);

// batched PNR / OSCC evaluation metrics on the device (loss.cu)
int pnr_metrics(int B, int n, const float* logits, const int64_t* label_idx, const float* label_onehot,
                const int64_t* sc_label, const double* fps, const int64_t* start, const int64_t* end, const int64_t* pnr,
                double* err_sec, long long* out_i64, double* out_f64, cudaStream_t st);
// losses on fp32 logits (rows, n_out)
int loss_fwd(const egot2_head_desc& d, int rows, const float* logits, const int64_t* labels, const float* class_weight,
             float* row_loss, float* loss, int32_t* argmax, cudaStream_t st);
// loss2 = the (2,) buffer written by loss_fwd: [loss, total weight]
int loss_bwd(const egot2_head_desc& d, int rows, const float* logits, const int64_t* labels, const float* class_weight,
             const float* loss2, float dloss_scale, float* dlogits, cudaStream_t st);

// ---- gradient guard (egot2_grad_guard): shared by egot2_grad_norm (rowops.cu) and the guarded peer exchange (peer.cu)
// Sum of v over the CTA in a fixed order (shuffle tree per warp, then the warp sums in warp order); the result is valid in
// thread 0.  `sh` holds blockDim.x / 32 doubles; every thread of the CTA must call it.
__device__ __forceinline__ double block_sum_f64(double v, double* sh) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();                     // `sh` may still be read by a previous call
  if ((threadIdx.x & 31) == 0) sh[warp] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < nw; ++w) s += sh[w];
  return s;
}
// total_norm = sqrt(sumsq) * |scale|; a finite norm gives the clip coefficient, a non-finite one skips the step and
// takes back the step-count increment of this step (so the count, the bias corrections and the lr schedule count applied
// steps only).  One thread.
__device__ __forceinline__ void grad_guard_finalize(double sumsq, float scale, egot2_grad_guard* guard, int32_t* step_dev) {
  const double tot = sqrt(sumsq) * fabs((double)scale);
  const float tn = (float)tot;
  guard->total_norm = tn;
  if (isfinite(tot)) {
    guard->coef = fminf(1.f, guard->max_norm / (tn + 1e-6f));      // clip_grad_norm_: clamp(max_norm / (norm + 1e-6), max=1)
    guard->skip = 0;
  } else {
    guard->coef = 0.f;
    guard->skip = 1;
    guard->skipped += 1;
    if (step_dev) *step_dev -= 1;
  }
}

}  // namespace egot2
