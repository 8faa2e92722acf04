/*
 * egot2.h — C ABI of libegot2.so: the B200 (sm_100a) implementation of EgoT2's task-translation
 * hot path (per-task projection -> LayerNorm + task/positional embedding -> TransformerEncoder over
 * the task x frame tokens -> task-of-interest head + loss, forward and backward).
 *
 * The reference (facebookresearch/EgoT2) is pure PyTorch: there is no FFI on this path.  The
 * boundary these entry points replace is the arithmetic that the reference's nn.Module classes
 * delegate to torch.nn / ATen (paths relative to the reference root):
 *
 *   egot2_embed_fwd/bwd          proj_* + self.ln + task_embed/pe (+dropouts)
 *                                HHI/models/ttm/model_taskspecific.py:178-182,188-190,222-226,238-241
 *                                HHI/models/asd/model_taskspecific.py:133-137,151-154
 *                                HOI/models/pnr/video_model_transfer_3task.py:249-254
 *                                HOI/models/lta/lta_models_lta_transfer.py:355-360
 *   egot2_hhi_tok_table_fwd/bwd  task_embed[:,k,:] + PositionalEncoding.pe[:D]
 *                                HHI/models/ttm/model_taskspecific.py:131-151,179-181
 *   egot2_encoder_layer_fwd/bwd  one nn.TransformerEncoderLayer (post-norm, ReLU, eps 1e-5)
 *                                HHI/models/ttm/model_taskspecific.py:168-171,191,242
 *                                HOI/models/pnr/video_model_transfer_3task.py:231-235,255
 *                                HOI/models/lta/lta_models_lta_transfer.py:272-275,361
 *   egot2_head_loss_fwd/bwd      mean over tokens + linear_head (+ loss)
 *                                HHI/models/ttm/model_taskspecific.py:192-193,243-244
 *                                HHI/tasks/ttm/video_task.py:23-24,36 (weighted CE)
 *                                HHI/tasks/asd/loss.py:11-30 (lossAV: FC + CE[1,4])
 *                                HOI/models/pnr/video_model_transfer_3task.py:256-257
 *                                HOI/tasks/pnr/video_taskspecific_pnr.py:29-31,143-146 (sigmoid+BCE / CE)
 *                                HOI/models/lta/head_helper.py:262-290, lta_models_lta_transfer.py:348-352
 *                                HOI/tasks/lta/long_term_anticipation_taskspecfic.py:177-183 (sum of 40 CE)
 *   egot2_slowfast_pool_fwd      AdaptiveAvgPool3d of the raw SlowFast maps
 *                                HOI/models/pnr/video_model_transfer_3task.py:226-227,245-247
 *   egot2_vit_layer_fwd/bwd      one simple_vit Transformer layer (pre-norm, GELU, bias-free attention)
 *                                HOI/models/pnr/simple_vit.py:55-107, HOI/models/pnr/video_model_transfer_3task.py:128-164
 *   egot2_adam_step              torch.optim.Adam over the flat translator parameter arena
 *                                HHI/tasks/ttm/video_task.py:64-66
 *   egot2_opt_advance            the optimizer step count and the learning rate of that step, on the device: the
 *                                warm-up + cosine / step-wise schedules of the HOI recipes (SURVEY.md §3.5,
 *                                HOI/optimizers/lta/lr_scheduler.py:21-26,67-91), read by egot2_adam_step_fused_sched
 *                                and by egot2_dp_reduce_adam (egot2_dp_desc.lr_dev) when they execute
 *   egot2_grad_norm              torch.nn.utils.clip_grad_norm_ (Lightning's gradient_clip_val) and GradScaler's skip of
 *                                non-finite steps, on the device, read by egot2_adam_step_fused_guard and by
 *                                egot2_dp_reduce_adam (egot2_dp_desc.guard)
 *   egot2_adam_step_fused_groups torch.optim param groups (per-group weight decay / lr multiplier, frozen parameters) over the
 *                                flat arena in the same one launch (SlowFast's construct_optimizer, HOI/optimizers/)
 *   egot2_sgd_step_fused         torch.optim.SGD (momentum, dampening, Nesterov, coupled weight decay) over the flat arena,
 *                                with the same device lr / guard / groups as the Adam entries and in egot2_dp_reduce_adam
 *                                (egot2_dp_desc.sgd); SlowFast's construct_optimizer builds it (HOI/optimizers/)
 *   egot2_param_stats            the add_histogram(name, weight) / add_histogram(name.grad, weight.grad) of the HOI LTA task's
 *                                gradient logging every LOG_GRADIENT_PERIOD steps (HOI/tasks/lta/video_task.py:112-125)
 *                                and Lightning's grad_norm, per parameter, on the device
 *   egot2_weight_avg_update      torch.optim.swa_utils.AveragedModel's update_parameters over the flat arena: the EMA of
 *                                get_ema_multi_avg_fn and the equal-weight SWA mean (Lightning's StochasticWeightAveraging)
 *
 * Conventions
 *   - every pointer is a DEVICE pointer (row-major, contiguous) unless the name ends in _host;
 *   - every call only enqueues work on `stream` (a cudaStream_t passed as void*); no hidden
 *     allocation, no host sync; scratch comes from the caller via workspace/ws_bytes;
 *   - return 0 on success; otherwise a non-zero code and egot2_last_error() (thread-local text);
 *   - "dtype" is the activation / GEMM-operand type of the call: EGOT2_F32 runs fp32 CUDA-core
 *     arithmetic (parity mode: logits within 1e-3 of the reference, argmax bit-exact);
 *     EGOT2_BF16 runs bf16 tensor-core GEMMs (tcgen05/TMEM) with fp32 accumulation and fp32
 *     LayerNorm/softmax statistics.  Matrix weights are passed in `dtype`; vectors (bias, LN
 *     gamma/beta, embeddings), statistics, losses and ALL gradients are fp32;
 *   - gradients are ACCUMULATED (+=) into the caller's buffers: zero the gradient arena once per
 *     step (this is also what lets `ln` be shared by two uses in the HOI PNR translator);
 *   - dropout masks are a pure function of (seed, site, element index), so forward and backward
 *     regenerate the same mask; nothing is stored.
 */
#ifndef EGOT2_H_
#define EGOT2_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EGOT2_MAX_SEG 8
#define EGOT2_MAX_GROUPS 4

enum { EGOT2_F32 = 0, EGOT2_BF16 = 1 };
enum { EGOT2_LOSS_NONE = 0, EGOT2_LOSS_CE = 1, EGOT2_LOSS_BCE_SIGMOID = 2, EGOT2_LOSS_CE_GROUPS = 3 };

const char* egot2_version(void);
const char* egot2_last_error(void);
/* SM count of the current device (cached per device). */
int egot2_sm_count(void);
/* Number of kernels this library has launched in this process so far (all streams). */
uint64_t egot2_launch_count(void);
/* Launcher timing for the benchmark's roofline: while enabled, every launcher of the library brackets the kernels it
 * enqueues with CUDA events on the launch stream (eager launches only; ignored during stream capture).
 * egot2_prof_report writes "<launcher tag>\t<launches>\t<total microseconds>\n" lines (host buffer). */
/* Dropout epoch: a device-resident counter XORed (times a constant) into every dropout key when the kernels EXECUTE, so
 * that a CUDA graph replayed every step draws fresh masks although its kernel arguments (the keys derived from `seed`)
 * were frozen at capture.  enable(1) allocates the 8-byte slot and switches all kernels to it (call outside stream
 * capture; single GPU context per process); set/advance enqueue on `stream` and are graph-capturable;
 * egot2_dropout_epoch_host(v) folds the same term into the keys on the HOST side instead (tests: host epoch v with the
 * device epoch off must reproduce device epoch v bit for bit). */
int egot2_dropout_epoch_enable(int on);
int egot2_dropout_epoch_set(uint64_t value, void* stream);
int egot2_dropout_epoch_advance(void* stream);
int egot2_dropout_epoch_host(uint64_t value);
int egot2_prof_enable(int on);
/* Deferred joins of the library's side streams (the parameter-gradient branches of egot2_encoder_layer_bwd).  While
 * egot2_side_defer(1) is in effect (per device), egot2_encoder_layer_bwd returns WITHOUT making `stream` wait for its
 * weight-gradient / bias-sum launches, so that they overlap the next layer's (or the embedding stage's) data-gradient
 * chain; a later egot2_encoder_layer_bwd that is handed the same `workspace` pointer first waits for them (callers
 * alternate two workspaces).  The caller MUST call egot2_side_join_all(stream) before anything on `stream` (or the host)
 * consumes the parameter gradients or reuses the saved activations, and before a stream capture ends.  Default off:
 * every call joins before returning (reference semantics: loss.backward() leaves every .grad complete). */
int egot2_side_defer(int on);
int egot2_side_join_all(void* stream);
/* Diagnostics, -DEGOT2_TIMELINE builds only (otherwise returns an error): every kernel stamps %globaltimer when it starts
 * (after its programmatic-dependent-launch wait) into dev_buf: u64[0] = number of stamps, then (ns, file_id*100000+line)
 * pairs, at most 2000.  Works inside CUDA-graph replays; NULL switches it off.  See tools/timeline.py. */
int egot2_timeline_set(void* dev_buf);
int egot2_prof_report(char* buf_host, size_t buf_bytes);

/* ------------------------------------------------------------------ embed stage */
typedef struct {
  int32_t dtype;                      /* token dtype */
  int32_t feat_dtype;                 /* dtype of the per-task feature tensors */
  int32_t B, T, H;                    /* clips, tokens per clip, hidden */
  int32_t n_seg;
  int32_t seg_tokens[EGOT2_MAX_SEG];  /* D_k: tokens this task contributes per clip */
  int32_t seg_in_dim[EGOT2_MAX_SEG];  /* K_k: feature width */
  int32_t seg_offset[EGOT2_MAX_SEG];  /* first token index of the task inside a clip */
  int32_t seg_has_proj[EGOT2_MAX_SEG];/* 0: feature is already H wide and is copied through */
  int32_t training;
  float p_feat;                       /* dropout on the projected features BEFORE the LN (HOI self.dp) */
  float p_embed;                      /* dropout AFTER the embedding add (HHI PositionalEncoding.dropout) */
  float ln_eps;
  uint64_t seed;
  int32_t no_ln;                      /* 1: no LayerNorm - tokens = projected features + tok_table (the 2-task simple_vit
                                       * sibling, HOI/models/pnr/video_model_transfer.py:63); needs p_feat = p_embed = 0 */
  int32_t feat_drop_tokens;           /* > 0: p_feat applies to the first feat_drop_tokens tokens of every clip only (the
                                       * 2-task PNR translator's FEAT_DROPOUT_MODE > 0 drops the PNR segment alone,
                                       * HOI/models/pnr/video_model_transfer.py:95-96); 0 = all tokens */
} egot2_embed_desc;

typedef struct {
  const void* feat[EGOT2_MAX_SEG];    /* (B, D_k, K_k), feat_dtype */
  const void* proj_w[EGOT2_MAX_SEG];  /* (H, K_k), dtype */
  const float* proj_b[EGOT2_MAX_SEG]; /* (H) */
  const float* ln_g;                  /* (H) shared self.ln */
  const float* ln_b;
  const float* tok_table;             /* (T, H): added after the LN */
} egot2_embed_in;

typedef struct {
  void* z;                            /* (B,T,H) dtype: projected (+feature-dropped) features, LN input  [saved] */
  float* stat;                        /* (B*T, 2): mean, rstd                                              [saved] */
  void* x;                            /* (B,T,H) dtype: tokens handed to the encoder */
} egot2_embed_out;

typedef struct {
  float* proj_w[EGOT2_MAX_SEG];
  float* proj_b[EGOT2_MAX_SEG];
  float* ln_g;
  float* ln_b;
  float* tok_table;                   /* (T,H); may be NULL when the table itself is not a parameter (HHI: use seg_embed) */
  float* dfeat[EGOT2_MAX_SEG];        /* optional (B,D_k,K_k) fp32 gradient w.r.t. a feature stream; NULL = frozen */
  float* seg_embed[EGOT2_MAX_SEG];    /* optional (H) +=: sum over clips and over segment k's tokens of the gradient that
                                       * reaches the token table, i.e. d(task_embed[task_k]) of the HHI translators whose
                                       * table rows are task_embed[task_k] + a fixed sinusoid (no (T,H) detour) */
} egot2_embed_grads;

size_t egot2_embed_workspace_bytes(const egot2_embed_desc* d, int backward);
int egot2_embed_fwd(const egot2_embed_desc* d, const egot2_embed_in* in, const egot2_embed_out* out,
                    void* workspace, size_t ws_bytes, void* stream);
int egot2_embed_bwd(const egot2_embed_desc* d, const egot2_embed_in* in, const egot2_embed_out* saved,
                    const void* dx /* (B,T,H) dtype; left intact */, const egot2_embed_grads* g,
                    void* workspace, size_t ws_bytes, void* stream);

/* HHI: tok_table[off_k + d, :] = task_embed[task_id_k, :] + pe[d, :]  (d restarts per task; `pe` is the module's
 * registered sinusoid buffer pos_embed.pe viewed as (pe_len,H); seg_* are HOST arrays) */
int egot2_hhi_tok_table_fwd(const float* task_embed /* (n_task,H) */, const float* pe, int32_t pe_len, int32_t n_seg,
                            const int32_t* seg_tokens_host, const int32_t* seg_task_id_host, int32_t H,
                            float* tok_table /* (T,H) */, void* stream);
int egot2_hhi_tok_table_bwd(const float* d_tok_table, int32_t n_seg, const int32_t* seg_tokens_host,
                            const int32_t* seg_task_id_host, int32_t H, float* d_task_embed /* += */, void* stream);

/* ------------------------------------------------------------------ encoder layer */
typedef struct {
  int32_t dtype;
  int32_t B, T, H, FF, heads;
  int32_t training;
  int32_t layer_index;                /* decorrelates dropout masks between layers */
  float p_drop;                       /* the layer's `dropout=`: attention probs, dropout1, dropout, dropout2 */
  float ln_eps;
  uint64_t seed;
} egot2_layer_desc;

typedef struct {
  const void* in_proj_w;              /* (3H,H) dtype */
  const void* out_proj_w;             /* (H,H)  */
  const void* lin1_w;                 /* (FF,H) */
  const void* lin2_w;                 /* (H,FF) */
  const float *in_proj_b, *out_proj_b, *lin1_b, *lin2_b;
  const float *norm1_g, *norm1_b, *norm2_g, *norm2_b;
} egot2_layer_params;

typedef struct {
  float *in_proj_w, *out_proj_w, *lin1_w, *lin2_w;
  float *in_proj_b, *out_proj_b, *lin1_b, *lin2_b;
  float *norm1_g, *norm1_b, *norm2_g, *norm2_b;
} egot2_layer_grads;

typedef struct {                      /* activations kept for backward; caller-allocated */
  void* qkv;                          /* (B*T, 3H) dtype */
  void* attn;                         /* (B*T, H)  dtype: concat of per-head P.V, input of out_proj */
  float* lse;                         /* (B, heads, T): log-sum-exp of the scaled scores */
  void* y1;                           /* (B*T, H) dtype: x + dropout1(attn out), LN1 input */
  float* stat1;                       /* (B*T, 2) */
  void* x1;                           /* (B*T, H) dtype: LN1 output */
  void* hid;                          /* (B*T, FF) dtype: dropout(relu(linear1(x1))) */
  void* y2;                           /* (B*T, H) dtype: x1 + dropout2(linear2(hid)), LN2 input */
  float* stat2;                       /* (B*T, 2) */
  void* hid_mask;                     /* optional (FF/64, B*T) x 64 bit: hid != 0 (ReLU gate x dropout keep).  Written by the
                                         fused tcgen05 FFN (bf16, H = 128, FF % 128 == 0); with it the backward runs the fused
                                         data-gradient kernel.  NULL: unfused backward from `hid`. */
  float* ffn_scratch;                 /* optional, egot2_ffn_scratch_bytes(B*T) bytes, ALL ZERO on entry and left all zero on
                                         exit: lets the fused FFN kernels cut the token tiles of their last, partial wave
                                         into FF slices that meet here (fp32).  NULL: tiles are never split. */
} egot2_layer_saved;

size_t egot2_ffn_scratch_bytes(int32_t M /* B*T tokens */);
size_t egot2_encoder_layer_workspace_bytes(const egot2_layer_desc* d, int backward);
int egot2_encoder_layer_fwd(const egot2_layer_desc* d, const egot2_layer_params* p, const void* x_in,
                            void* x_out, const egot2_layer_saved* s, void* workspace, size_t ws_bytes,
                            void* stream);
/* dx_out is clobbered; dx_in may alias dx_out. */
int egot2_encoder_layer_bwd(const egot2_layer_desc* d, const egot2_layer_params* p, const void* x_in,
                            const egot2_layer_saved* s, void* dx_out, void* dx_in,
                            const egot2_layer_grads* g, void* workspace, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------ simple_vit layer (HOI PNR "simple_vit" siblings)
 * One layer of the simple_vit Transformer (HOI/models/pnr/simple_vit.py:55-107; used by
 * HOI/models/pnr/video_model_transfer_3task.py:128-164 with dim 256, depth 3, heads 8, dim_head 128, mlp_dim 512):
 *     x1 = to_out(softmax(q k^T * dim_head^-0.5) v) + x,  [q|k|v] = to_qkv(LayerNorm(x))     (pre-norm, bias-free)
 *     x2 = W2 gelu(W1 LayerNorm(x1) + b1) + b2 + x1                                         (exact erf GELU)
 * no dropout; dim_head is independent of the model width D (inner = heads * dim_head). */
typedef struct {
  int32_t dtype;
  int32_t B, T, D;                    /* clips, tokens per clip, model width */
  int32_t heads, dim_head;
  int32_t mlp;                        /* hidden width of the FeedForward */
  int32_t layer_index;
  float ln_eps;
} egot2_vit_desc;

typedef struct {
  const void *qkv_w, *out_w;          /* layers.i.0.to_qkv.weight (3*inner, D), layers.i.0.to_out.weight (D, inner); dtype */
  const void *ff1_w, *ff2_w;          /* layers.i.1.net.1.weight (mlp, D), layers.i.1.net.3.weight (D, mlp); dtype */
  const float *norm_a_g, *norm_a_b;   /* layers.i.0.norm */
  const float *norm_f_g, *norm_f_b;   /* layers.i.1.net.0 */
  const float *ff1_b, *ff2_b;
} egot2_vit_params;

typedef struct {                      /* fp32, accumulated (+=) */
  float *qkv_w, *out_w, *ff1_w, *ff2_w;
  float *norm_a_g, *norm_a_b, *norm_f_g, *norm_f_b, *ff1_b, *ff2_b;
} egot2_vit_grads;

typedef struct {                      /* activations kept for backward; caller-allocated; M = B*T, inner = heads*dim_head */
  void* h; float* stat_a;             /* (M, D) LayerNorm_a output, (M, 2) */
  void* qkv;                          /* (M, 3*inner) */
  void* attn; float* lse;             /* (M, inner), (B, heads, T) */
  void* x1;                           /* (M, D) */
  void* h2; float* stat_f;            /* (M, D), (M, 2) */
  void* u; void* act;                 /* (M, mlp) pre-activation and gelu(u) */
} egot2_vit_saved;

size_t egot2_vit_layer_workspace_bytes(const egot2_vit_desc* d);
int egot2_vit_layer_fwd(const egot2_vit_desc* d, const egot2_vit_params* p, const void* x_in /* (M,D) */, void* x_out,
                        const egot2_vit_saved* s, void* stream);
/* dx_in may alias dx_out */
int egot2_vit_layer_bwd(const egot2_vit_desc* d, const egot2_vit_params* p, const void* x_in, const egot2_vit_saved* s,
                        const void* dx_out, void* dx_in, const egot2_vit_grads* g, void* workspace, size_t ws_bytes,
                        void* stream);

/* ------------------------------------------------------------------ EgoT2-g decoder (task-prompt transformer)
 * One nn.TransformerDecoderLayer (post-norm, ReLU; CustomDecoderLayer only forces need_weights) over the S-token task
 * prompt of every row, attending to that row's encoder memory:
 *     HHI/models/multitask/task_prompt_model.py:163-172,187-194,260-269
 * Row n, memory key j reads encoder token  (n / kv_inner) * kv_outer + j * kv_jstride + (n % kv_inner) * kv_istride :
 *     'lam' / 'ttm' (memory = the clip's M tokens):  kv_inner 1, kv_outer M, kv_jstride 1, kv_istride 0
 *     'asd' (:251-257, 3-token memory per frame):    kv_inner T, kv_outer 3T, kv_jstride T, kv_istride 1, rows = B*T */
typedef struct {
  int32_t dtype;
  int32_t rows, S;                    /* decoder rows, prompt tokens per row */
  int32_t mem_rows, M;                /* encoder tokens in `mem`, memory tokens per row */
  int32_t kv_inner, kv_outer, kv_jstride, kv_istride;
  int32_t H, FF, heads;
  int32_t training, layer_index;
  float p_drop, ln_eps;
  uint64_t seed;
} egot2_decoder_desc;

typedef struct {
  const void *sa_in_w, *sa_out_w;     /* self_attn.in_proj_weight (3H,H), out_proj.weight (H,H); dtype */
  const void *ca_in_w, *ca_out_w;     /* multihead_attn.* */
  const void *lin1_w, *lin2_w;        /* (FF,H), (H,FF) */
  const float *sa_in_b, *sa_out_b, *ca_in_b, *ca_out_b, *lin1_b, *lin2_b;
  const float *norm1_g, *norm1_b, *norm2_g, *norm2_b, *norm3_g, *norm3_b;
} egot2_decoder_params;

typedef struct {
  float *sa_in_w, *sa_out_w, *ca_in_w, *ca_out_w, *lin1_w, *lin2_w;
  float *sa_in_b, *sa_out_b, *ca_in_b, *ca_out_b, *lin1_b, *lin2_b;
  float *norm1_g, *norm1_b, *norm2_g, *norm2_b, *norm3_g, *norm3_b;
} egot2_decoder_grads;

typedef struct {                      /* activations kept for backward; caller-allocated; R = rows*S */
  void* qkv;                          /* (R, 3H) dtype */
  void* a1;                           /* (R, H): self-attention heads, input of out_proj */
  void* y1; float* stat1; void* x1;   /* (R, H) LN1 input, (R,2), LN1 output */
  void* qc;                           /* (R, H): cross-attention queries */
  void* kvc;                          /* (mem_rows, 2H): cross-attention keys | values of every encoder token */
  void* a2;                           /* (R, H) */
  void* y2; float* stat2; void* x2;
  void* hid;                          /* (R, FF) */
  void* y3; float* stat3;
} egot2_decoder_saved;

size_t egot2_decoder_layer_workspace_bytes(const egot2_decoder_desc* d);
int egot2_decoder_layer_fwd(const egot2_decoder_desc* d, const egot2_decoder_params* p, const void* y_in /* (R,H) */,
                            const void* mem /* (mem_rows,H) */, void* y_out, const egot2_decoder_saved* s, void* stream);
/* dy_out is clobbered; dy_in may alias it; dmem (mem_rows,H) fp32 is ACCUMULATED (+=) over the decoder layers */
int egot2_decoder_layer_bwd(const egot2_decoder_desc* d, const egot2_decoder_params* p, const void* y_in, const void* mem,
                            const egot2_decoder_saved* s, void* dy_out, void* dy_in, float* dmem,
                            const egot2_decoder_grads* g, void* workspace, size_t ws_bytes, void* stream);
/* prompt tokens: y[n,s,:] = embedding[tok[n,s],:] * sqrt(H) + pe[s,:], then Dropout(p) (decode(), :262-264) */
int egot2_prompt_embed_fwd(int32_t dtype, int32_t rows, int32_t S, int32_t H, const int64_t* tokens,
                           const float* embedding, const float* pe, float p_drop, int32_t training, uint64_t seed,
                           void* y, void* stream);
int egot2_prompt_embed_bwd(int32_t dtype, int32_t rows, int32_t S, int32_t H, const int64_t* tokens, const void* dy,
                           float p_drop, int32_t training, uint64_t seed, float* d_embedding /* (V,H) += */, void* stream);

/* ------------------------------------------------------------------ head + loss */
typedef struct {
  int32_t dtype;
  int32_t B, T, H;                    /* rows are mean-pooled over T when pool != 0 */
  int32_t pool;                       /* 1: rows = B clips (mean over T tokens); 0: rows = B*T tokens (ASD) */
  int32_t row_tokens;                 /* pool==0: use only the first row_tokens tokens of each clip */
  int32_t use_ln;                     /* LayerNorm before the Linear (linear_head.0) */
  int32_t n_out;                      /* width of the Linear: 2 | 16 | Z*593 */
  int32_t loss;                       /* EGOT2_LOSS_* */
  int32_t n_groups;                   /* CE_GROUPS: class groups inside each sub-row (verbs, nouns) */
  int32_t group_size[EGOT2_MAX_GROUPS];
  int32_t sub_rows;                   /* CE_GROUPS: Z sub-rows per row (n_out = sub_rows * sum(group_size)) */
  int32_t training;
  float p_head;                       /* dropout on the pooled vector (LTA MultiTaskHead) */
  float ln_eps;
  uint64_t seed;
} egot2_head_desc;

typedef struct {
  const void* x;                      /* (B,T,H) dtype encoder output */
  const float *ln_g, *ln_b;           /* (H) or NULL */
  const void* w;                      /* (n_out,H) dtype */
  const float* b;                     /* (n_out) */
  const int64_t* labels;              /* CE: (rows); BCE: (rows) index of the 1 in the one-hot; CE_GROUPS: (rows, sub_rows, n_groups) */
  const float* class_weight;          /* CE: (n_out) or NULL */
} egot2_head_in;

typedef struct {
  float* pooled;                      /* (rows,H) fp32: mean over tokens (or gathered tokens)  [saved] */
  float* stat;                        /* (rows,2)                                             [saved] */
  void* g;                            /* (rows,H) dtype: LN'd (+dropped) vector fed to the Linear [saved] */
  float* logits;                      /* (rows,n_out) fp32 */
  float* loss;                        /* (2): [0] the scalar loss, [1] its normaliser (sum of class weights | rows) */
  int32_t* argmax;                    /* (rows*sub_rows*max(1,n_groups)) index of the max logit (per group) or NULL */
  float* row_loss;                    /* (rows,2) scratch: weighted nll, weight */
} egot2_head_out;

typedef struct {
  float *ln_g, *ln_b, *w, *b;
} egot2_head_grads;

int egot2_head_rows(const egot2_head_desc* d);
int egot2_head_loss_fwd(const egot2_head_desc* d, const egot2_head_in* in, const egot2_head_out* out, void* stream);
/* If d->loss != NONE, dlogits is derived from the loss scaled by *dloss_scale_host (usually 1.0f) and
 * written to out->logits' gradient buffer `dlogits`; otherwise the caller provides dlogits. */
int egot2_head_loss_bwd(const egot2_head_desc* d, const egot2_head_in* in, const egot2_head_out* saved,
                        float* dlogits /* (rows,n_out) fp32 in/out */, float dloss_scale,
                        void* dx /* (B,T,H) dtype, written (=, not +=) */, const egot2_head_grads* g,
                        void* workspace, size_t ws_bytes, void* stream);
size_t egot2_head_workspace_bytes(const egot2_head_desc* d);

/* ------------------------------------------------------------------ utilities */
/* AdaptiveAvgPool3d of raw SlowFast maps: in (B,C,Tin,h,w) -> out (B,Tout,C), mean over h,w and Tin/Tout frames. */
int egot2_slowfast_pool_fwd(const void* in, int32_t in_dtype, int32_t B, int32_t C, int32_t Tin, int32_t hw,
                            int32_t Tout, void* out, int32_t out_dtype, void* stream);
/* fp32 -> bf16 shadow copy of (part of) the parameter arena. */
int egot2_cast_f32_to_bf16(const float* src, void* dst, size_t n, void* stream);
/* dst[i] += a[i] (+ b[i], b may be NULL), then a (and b) are cleared; n %% 4 == 0.  Joins the per-branch gradient arenas of an
 * EgoT2-g step (three forwards of one model on three streams, HHI/tasks/multitask/video_tasktranslation.py:48-61). */
int egot2_sum_into_f32(float* dst, float* a, float* b, size_t n, void* stream);
int egot2_cast_bf16_to_f32(const void* src, float* dst, size_t n, void* stream);
/* torch.optim.Adam (no amsgrad) over a flat arena; grad_scale multiplies the gradient first (1/world for DP mean). */
int egot2_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                    float beta1, float beta2, float eps, float weight_decay, int32_t step, float grad_scale,
                    void* stream);
/* Same update, and in the same pass: the bf16 shadow of the updated parameters (shadow_bf16, n elements; NULL = skip) and,
 * if zero_grad, the gradient arena is cleared for the next step's accumulation (replaces a cast launch and a fill). */
int egot2_adam_step_fused(float* param, float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                          float beta1, float beta2, float eps, float weight_decay, int32_t step, float grad_scale,
                          void* shadow_bf16, int32_t zero_grad, void* stream);
/* Same, with the step count t >= 1 read from DEVICE memory at execution time (bias corrections 1 - beta^t computed in the
 * kernel): the launch can sit inside a CUDA graph that is replayed every step while a counter kernel advances *step_dev. */
int egot2_adam_step_fused_dev(float* param, float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                              float beta1, float beta2, float eps, float weight_decay, const int32_t* step_dev,
                              float grad_scale, void* shadow_bf16, int32_t zero_grad, void* stream);
/* torch.optim.AdamW: decoupled weight decay (param *= 1 - lr*weight_decay before the Adam update); otherwise as
 * egot2_adam_step_fused (HOI EgoT2-g optimizer: HOI/tasks/multitask/video_task.py:265-268) */
int egot2_adamw_step_fused(float* param, float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                           float beta1, float beta2, float eps, float weight_decay, int32_t step, float grad_scale,
                           void* shadow_bf16, int32_t zero_grad, void* stream);

/* Learning-rate schedule, evaluated on the device.  lr_at(s) for optimizer step s = 0, 1, ... (fp64, rounded once to float):
 *   CONSTANT  base_lr
 *   COSINE    end_lr + (base_lr - end_lr) * (1 + cos(pi * s / total_steps)) / 2, and end_lr for s >= total_steps
 *   STEPS     base_lr * factors[i], i = the number of milestones <= s (SlowFast's steps-with-relative-lrs; MultiStepLR
 *             when factors[i] = gamma^i); milestones increasing, n_milestones <= 8, factors[0..n_milestones] used
 * and, for every kind, a linear warm-up over s < warmup_steps:
 *             warmup_start_lr + (lr_at(warmup_steps) - warmup_start_lr) * s / warmup_steps.
 * The lr of optimizer step t (1-based) is lr_at(t - 1): torch.optim.lr_scheduler.LambdaLR stepped after every
 * optimizer.step(). */
enum { EGOT2_LR_CONSTANT = 0, EGOT2_LR_COSINE = 1, EGOT2_LR_STEPS = 2 };
typedef struct {
  int32_t kind, n_milestones;           /* EGOT2_LR_*; STEPS: <= 8 */
  int64_t warmup_steps, total_steps;    /* in optimizer steps; total_steps > 0 for COSINE */
  double base_lr, warmup_start_lr, end_lr;
  int64_t milestones[8];
  double factors[9];
} egot2_lr_sched;
/* One thread: t = ++*step_dev; *lr_dev = (float) lr_at(*sched, t - 1).  All three are DEVICE pointers, read when the kernel
 * executes, so a CUDA graph that contains the launch follows a schedule rewritten between replays. */
int egot2_opt_advance(int32_t* step_dev, const egot2_lr_sched* sched, float* lr_dev, void* stream);
/* egot2_adam_step_fused_dev with the learning rate read from DEVICE memory (*lr_dev, e.g. written by egot2_opt_advance) at
 * execution time; decoupled = 1 runs AdamW (param *= 1 - lr*weight_decay with the same device lr). */
int egot2_adam_step_fused_sched(float* param, float* grad, float* exp_avg, float* exp_avg_sq, size_t n, const float* lr_dev,
                                float beta1, float beta2, float eps, float weight_decay, const int32_t* step_dev,
                                float grad_scale, void* shadow_bf16, int32_t zero_grad, int32_t decoupled, void* stream);

/* Gradient-norm clipping and skipping of non-finite steps, on the device (torch.nn.utils.clip_grad_norm_, and the step skip of
 * torch.amp.GradScaler).  A DEVICE-resident descriptor: max_norm is the input (> 0, +inf = never clip), the rest is written by
 * egot2_grad_norm (or by the guarded peer exchange) when it executes:
 *   total_norm = ||grad_scale * grad||_2 over the whole arena (squares summed in fp64, fixed order: bit-reproducible);
 *   finite total_norm:     coef = min(1, max_norm / (total_norm + 1e-6)) (fp32, clip_grad_norm_'s formula), skip = 0;
 *   non-finite total_norm: skip = 1, ++skipped, and the optimizer step count is decremented (*step_dev, when given), so
 *                          that it, the Adam bias corrections and the lr schedule count applied steps only. */
typedef struct {
  float max_norm;
  float total_norm;
  float coef;
  int32_t skip;
  int32_t skipped;
} egot2_grad_guard;
/* Bytes of the egot2_grad_norm workspace.  Zero-fill it once before its first use; every call leaves it that way again
 * (its grid counter resets itself), so the call can sit in a CUDA graph. */
size_t egot2_grad_norm_workspace_bytes(void);
/* One launch of a fixed grid (independent of the device and of timing): per-CTA fp64 sums of squares, and the last CTA adds
 * them in CTA order and writes total_norm / coef / skip (/ skipped, *step_dev) of *guard.  No host sync; graph-capturable. */
int egot2_grad_norm(const float* grad, size_t n, float grad_scale, egot2_grad_guard* guard, int32_t* step_dev, void* workspace,
                    size_t ws_bytes, void* stream);
/* egot2_adam_step_fused_sched with the guard applied: the gradient is multiplied by grad_scale * guard->coef; with
 * guard->skip the parameters, the moments and the shadow stay as they are and only the gradient is cleared (zero_grad).
 * lr_dev NULL: the learning rate is `lr`.  decoupled = 1 runs AdamW. */
int egot2_adam_step_fused_guard(float* param, float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                                const float* lr_dev, float beta1, float beta2, float eps, float weight_decay,
                                const int32_t* step_dev, float grad_scale, void* shadow_bf16, int32_t zero_grad,
                                int32_t decoupled, const egot2_grad_guard* guard, void* stream);

/* Parameter groups (torch.optim param groups: per-group weight decay and lr multiplier, and frozen parameters), on the device.
 * A DEVICE-resident descriptor plus a DEVICE map block_group[ceil(n / 64)]: element i belongs to group block_group[i / 64]
 * (< n_groups).  For the elements of group k, with lr the step's learning rate (by value or from lr_dev):
 *   Adam:   grad += weight_decay[k] * param;                  AdamW: param *= 1 - lr * lr_mult[k] * weight_decay[k];
 *   the step size is lr * lr_mult[k] (lr_mult[k] = 0 still updates the moments, as torch does with lr = 0);
 *   frozen[k] != 0 (requires_grad=False): parameters, shadow and moments are left as they are, the gradient is only cleared
 *   (zero_grad), and egot2_grad_norm_groups leaves it out of the norm.
 * The descriptor is read when a kernel executes, so a CUDA graph follows a descriptor rewritten between replays. */
#define EGOT2_MAX_PARAM_GROUPS 8
typedef struct {
  int32_t n_groups;                     /* 1..EGOT2_MAX_PARAM_GROUPS */
  float lr_mult[8];
  float weight_decay[8];
  int32_t frozen[8];
} egot2_param_groups;
/* egot2_adam_step_fused_guard with parameter groups: every element takes its group's lr multiplier, weight decay and frozen
 * flag (there is no arena-wide weight_decay argument).  lr_dev NULL: the learning rate is `lr`; guard NULL: no clipping or
 * skipping (with a guard, egot2_grad_norm_groups runs first).  step_dev is required.  decoupled = 1 runs AdamW. */
int egot2_adam_step_fused_groups(float* param, float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                                 const float* lr_dev, float beta1, float beta2, float eps, const int32_t* step_dev,
                                 float grad_scale, void* shadow_bf16, int32_t zero_grad, int32_t decoupled,
                                 const egot2_grad_guard* guard, const egot2_param_groups* groups,
                                 const uint8_t* block_group, void* stream);
/* egot2_grad_norm over the elements of non-frozen groups only (clip_grad_norm_ over the trainable parameters): a NaN / inf in
 * a frozen gradient neither clips nor skips.  Same fixed grid and summation order as egot2_grad_norm, with frozen elements
 * counted as 0. */
int egot2_grad_norm_groups(const float* grad, size_t n, float grad_scale, egot2_grad_guard* guard, int32_t* step_dev,
                           const egot2_param_groups* groups, const uint8_t* block_group, void* workspace, size_t ws_bytes,
                           void* stream);

/* torch.optim.SGD (maximize=False) over the flat arena in one launch.  For the elements of group k (without groups: one group
 * with lr_mult 1 and `weight_decay`), with lr the step's learning rate (by value, or *lr_dev when lr_dev is not NULL) and
 * g = grad * grad_scale (* guard->coef with a guard):
 *   if wd != 0:    g += wd * param                                      (coupled weight decay)
 *   if momentum:   buf = g on the first applied step, else momentum * buf + (1 - dampening) * g
 *                  d = nesterov ? g + momentum * buf : buf
 *   else           d = g
 *   param -= lr * lr_mult[k] * d;  shadow = bf16(param) (shadow_bf16 not NULL);  grad = 0 (zero_grad)
 * The first applied step is the one whose count is 1: *step_dev when step_dev is not NULL (read when the kernel executes,
 * after a guard took back a skipped step), else `step`.  momentum_buf is NULL exactly when momentum == 0.  momentum >= 0,
 * dampening finite, nesterov needs momentum > 0 and dampening == 0.  guard (needs step_dev): egot2_grad_norm[_groups] ran
 * first; on a skip parameters, shadow and buffer stay and the gradient is only cleared.  groups (with block_group):
 * egot2_adam_step_fused_groups' per-group lr_mult / weight_decay (`weight_decay` is then unused) / frozen, where a frozen
 * group also keeps its buffer. */
int egot2_sgd_step_fused(float* param, float* grad, float* momentum_buf, size_t n, float lr, const float* lr_dev,
                         float momentum, float dampening, int32_t nesterov, float weight_decay,
                         int32_t step, const int32_t* step_dev, float grad_scale, void* shadow_bf16, int32_t zero_grad,
                         const egot2_grad_guard* guard, const egot2_param_groups* groups, const uint8_t* block_group,
                         void* stream);

/* Per-parameter statistics of the gradient and of the weights (the histograms and gradient norms a training loop logs every
 * LOG_GRADIENT_PERIOD steps), on the device.  Array 0 is the gradient the optimizer applies, fp32(grad[i] * grad_scale);
 * array 1 is the fp32 parameters.  A step t (*step_dev, read when the kernel executes) is due when (t - 1) % every == 0; on
 * any other step every CTA returns at once and no output changes.  A DEVICE-resident descriptor: every, histograms and
 * n_params are inputs, grad_norm and step are written on a due step, step last. */
#define EGOT2_STATS_BUCKETS 1548      /* TensorBoard's default histogram: 1549 edges, see egot2_param_stats */
typedef struct {
  int32_t every;                      /* > 0 */
  int32_t histograms;                 /* 1: bucket counts as well (needs edges and counts) */
  int32_t n_params;                   /* P */
  int32_t step;                       /* out: t of the last due step, 0 before the first */
  float grad_norm;                    /* out: L2 norm of array 0 over the parameters with has_grad (NaN / inf as torch) */
} egot2_param_stats_desc;
/* One parameter of the arena: elements [offset, offset + numel).  has_grad = 0 (a frozen parameter): no gradient statistics,
 * no units in array 0, and no share in grad_norm.  first_unit[a] / n_units[a]: its units of array a, consecutive. */
typedef struct {
  int64_t offset;
  int64_t numel;
  int32_t has_grad;
  int32_t first_unit[2];
  int32_t n_units[2];
} egot2_stats_param;
/* One work unit: arena elements [begin, end) of parameter `param` in array `array` (0 gradient, 1 weights).  Units are
 * enumerated on the host, ordered by (array, param, begin); a unit never covers two parameters. */
typedef struct {
  int32_t param;
  int32_t array;
  int64_t begin, end;
} egot2_stats_unit;
/* The statistics of one (array, parameter); stats[a * P + p].  min / max / sum / sum_squares cover the finite elements (sums
 * in fp64, added in a fixed order: bit-reproducible); nonfinite counts NaN and +-inf; norm = sqrt(sum_squares) as fp32, or NaN
 * when a NaN is present, else +inf when an inf is; no finite element: min = +inf, max = -inf.  num = numel. */
typedef struct {
  double sum;
  double sum_squares;
  float min, max;
  float norm;
  int32_t nonfinite;
  int64_t num;
} egot2_param_stat;
/* Bytes of the egot2_param_stats workspace for P parameters and n_units units.  Zero-fill it once (256-byte aligned); every
 * call leaves it that way again, so the call can sit in a CUDA graph. */
size_t egot2_param_stats_workspace_bytes(int32_t n_params, int32_t n_units);
/* One launch of a grid fixed at launch: every unit's fp64 partial sums (fixed order), exact min / max / counts through integer
 * atomics, the unit partials of a parameter added in unit order by the CTA that finishes its last unit.  With histograms,
 * counts[a * P + p][b] = the number of finite values x with edges[b] <= (double)x < edges[b + 1] (the last bucket closed on
 * the right; np.histogram's rule; -0.0 counts as 0).  edges: the 1549 doubles of TensorBoard's default bins
 * (SummaryWriter.default_bins: v = 1e-12, times 1.1 while v < 1e20, mirrored, with 0).  edges and counts are both NULL
 * without histograms.  No host sync; graph-capturable. */
int egot2_param_stats(const float* grad, const float* param, float grad_scale, const int32_t* step_dev,
                      egot2_param_stats_desc* desc, const egot2_stats_param* params, int32_t n_params,
                      const egot2_stats_unit* units, int32_t n_units, const double* edges, egot2_param_stat* stats,
                      int32_t* counts, void* workspace, size_t ws_bytes, void* stream);

/* Weight averaging (torch.optim.swa_utils.AveragedModel) of the fp32 arena, after the optimizer launch of a step.  A step t
 * (*step_dev, the applied-step count, read when the kernel executes) is due when t >= start and (t - start) % every == 0;
 * on a due step, with n = (t - start) / every the number of earlier updates:
 *   n == 0:  avg = param                                            (AveragedModel's first update_parameters copies)
 *   n > 0:   avg = lerp(avg, param, w),  w = ema_weight (EGOT2_AVG_EMA: float(1 - decay), get_ema_multi_avg_fn)
 *                                        w = 1 / (n + 1) in fp32     (EGOT2_AVG_SWA: the running mean; ema_weight unused)
 * lerp is ATen's: w < 0.5 ? a + w * (p - a) : p - (p - a) * (1 - w), in fp32 with each product-and-sum fused into one FMA,
 * as torch's CUDA _foreach_lerp_ rounds it.  guard (NULL: none): when guard->skip is set the step was skipped and nothing
 * changes, whatever *step_dev holds.  On a step that is not due every CTA returns at once.  n is a multiple of 4 and both
 * arrays are 16-byte aligned.  No host sync; graph-capturable. */
enum { EGOT2_AVG_EMA = 0, EGOT2_AVG_SWA = 1 };
int egot2_weight_avg_update(const float* param, float* avg, size_t n, int32_t kind, float ema_weight, int32_t every,
                            int32_t start, const int32_t* step_dev, const egot2_grad_guard* guard, void* stream);

/* ------------------------------------------------------------------ data-parallel exchange over NVLink peer memory
 * The reference trains under DDP / DP (HOI/scripts/lta/run_lta.py:249, HOI/tasks/pnr/video_task.py:39-42): an all-reduce of the
 * translator gradients after backward, then the optimizer on every rank.  Here that is ONE kernel (csrc/peer.cu): gradient
 * reduce-scatter over peer memory -> Adam on this rank's slice -> all-gather of the updated fp32 parameters and bf16 shadow.
 *
 * Every rank keeps parameters, gradients and shadow in one "slab" allocated by egot2_peer_alloc (cudaMalloc; zero-filled) with
 * the same byte offsets on every rank, followed by egot2_dp_flag_bytes() bytes of flag words.  The ranks exchange the
 * egot2_peer_handle_bytes()-byte IPC handles (egot2_peer_export) through their own channel (torch.distributed) and map each
 * other's slabs (egot2_peer_import).  All ranks must call egot2_dp_reduce_adam the same number of times; a rank that never
 * does makes the others trap after ~4 s (no hang).  After the call (stream order) this rank's arena holds the new parameters,
 * identical bit for bit on every rank, and no peer reads this rank's gradients any more (the caller clears them). */
typedef struct {
  int32_t world, rank;
  int64_t numel;                      /* arena elements (a multiple of 4) */
  void* slab[8];                      /* slab[p]: rank p's slab as mapped in THIS process; slab[rank] = the local one */
  int64_t off_param, off_grad;        /* byte offsets of the fp32 parameter / gradient arenas inside a slab (16-byte aligned) */
  int64_t off_shadow;                 /* byte offset of the bf16 shadow, or -1 (fp32 engines) */
  int64_t off_flags;                  /* byte offset of the flag words */
  float* exp_avg; float* exp_avg_sq;  /* LOCAL Adam moments, arena layout (only this rank's slice is touched) */
  float lr, beta1, beta2, eps, weight_decay;
  int32_t step;                       /* optimizer step count (1-based) for the bias corrections, unless step_dev */
  const int32_t* step_dev;            /* optional: the count lives on the device (CUDA-graph replays) */
  int32_t decoupled;                  /* 1: AdamW */
  int32_t zero_grads_remote;          /* 1: the owner of a slice clears that slice of every rank's gradient arena after reading
                                       * it (small arenas: no separate clear launch); 0: the caller clears its arena afterwards */
  const float* lr_dev;                /* optional: the learning rate lives on the device (egot2_opt_advance); NULL: `lr` */
  egot2_grad_guard* guard;            /* optional: clip by the global norm of the rank-averaged gradient / skip non-finite
                                       * steps (egot2_grad_norm's semantics; every rank reaches the same decision).  The exchange
                                       * then runs as two launches with one more flag round trip: reduce + norm, then the update */
  const egot2_param_groups* groups;   /* optional, with block_group: parameter groups (egot2_adam_step_fused_groups' semantics;
                                       * `weight_decay` above is then unused, and the guard's norm leaves frozen groups out) */
  const uint8_t* block_group;         /* the group of every 64-element block of the WHOLE arena (also for a [lo, hi) range) */
  int32_t sgd;                        /* 1: torch.optim.SGD (egot2_sgd_step_fused's semantics) instead of Adam: exp_avg is the
                                       * LOCAL momentum buffer, NULL exactly when momentum == 0; exp_avg_sq may be NULL; beta1,
                                       * beta2 and eps are unused; decoupled must be 0.  0: Adam / AdamW as above */
  float momentum, dampening;
  int32_t nesterov;
} egot2_dp_desc;
int egot2_peer_alloc(size_t bytes, void** ptr);
int egot2_peer_free(void* ptr);
int egot2_peer_handle_bytes(void);
int egot2_peer_export(void* ptr, void* handle_out);
int egot2_peer_import(const void* handle, void** ptr);
int egot2_peer_unimport(void* ptr);
size_t egot2_dp_flag_bytes(void);
int egot2_dp_reduce_adam(const egot2_dp_desc* d, void* stream);
/* The same exchange restricted to arena elements [lo, hi) (multiples of 4) on flag channel 0 or 1: two exchanges may be in
 * flight at once on different channels and streams - e.g. everything but the embedding-stage gradients while the embedding
 * backward still runs, then the embedding prefix (the arena keeps those parameters first for exactly this purpose). */
int egot2_dp_reduce_adam_range(const egot2_dp_desc* d, int64_t lo, int64_t hi, int32_t channel, void* stream);

/* Batched PNR / OSCC evaluation metrics in one launch (replaces the per-clip `.item()` loops of
 * HOI/evaluation/pnr/metrics.py:11-80: state_change_accuracy, keyframe_accuracy, keyframe_distance).
 * logits (B,n) fp32; label_idx (B) int64 OR label_onehot (B,n) fp32; sc_label (B) int64 or NULL (every clip counts);
 * fps (B) f64 + start/end/pnr frames (B) int64, or fps NULL to skip the time error.
 * out_counts[2] = {correct, total}; out_dist_sum[1] = sum over counted clips of
 * |float32((end-start)/16 * argmax) - (pnr-start)| / fps; err_sec (B, optional) = per-clip error, -1 for skipped clips. */
int egot2_pnr_metrics(int32_t B, int32_t n, const float* logits, const int64_t* label_idx, const float* label_onehot,
                      const int64_t* sc_label, const double* fps, const int64_t* start_frame, const int64_t* end_frame,
                      const int64_t* pnr_frame, double* err_sec, int64_t* out_counts, double* out_dist_sum, void* stream);

/* TTM evaluation (HHI/utils/ttm/utils.py:71-80, PostProcessor._merge_output): out[s, :] = softmax(mean over rows
 * [seg_offsets[s], seg_offsets[s+1]) of logits (rows, n_cls)), one launch for all segments; the TTM score is out[s, 1].
 * n_cls <= 8; device pointers; seg_offsets has n_seg + 1 entries. */
int egot2_segment_softmax_mean(int32_t n_seg, int32_t n_cls, const float* logits, const int32_t* seg_offsets, float* out,
                               void* stream);
/* out = softmax(in) over the n columns of every row (fp32; may alias): the eval-mode activation of the LTA MultiTaskHead
 * (HOI/models/lta/head_helper.py:284-286) and lossAV's predScore (HHI/tasks/asd/loss.py:24). */
int egot2_row_softmax(int64_t rows, int32_t n, const float* in, float* out, void* stream);
/* LTA / AR evaluation (HOI/evaluation/lta/lta_metrics.py:39-73, topks_correct): correct[i] = number of rows whose label is among
 * the ks[i] largest of preds (N, C) (ties resolved towards the smaller class index); ks is a HOST array of n_k <= 8 values;
 * correct is a device array of n_k int64, overwritten. */
int egot2_topk_correct(int32_t N, int32_t C, const float* preds, const int64_t* labels, int32_t n_k, const int32_t* ks_host,
                       int64_t* correct, void* stream);
/* LTA evaluation (lta_metrics.py:87-110, edit_distance / AUED; `editdistance.eval` = Levenshtein distance): for every clip n and
 * prefix length z = 1..Z, min over the K sampled sequences of lev(preds[n, :z, k], labels[n, :z]) -> min_dist[n, z-1] (optional)
 * and sum_min[z-1] = sum over the clips (int64, overwritten).  preds (N, Z, K) and labels (N, Z) int64; Z <= 64.
 * ED_z of the reference = sum_min[z-1] / (z * N); AUED = trapz(ED) / (Z - 1). */
int egot2_edit_distance_prefix(int32_t N, int32_t Z, int32_t K, const int64_t* preds, const int64_t* labels, int32_t* min_dist,
                               int64_t* sum_min, void* stream);

/* ------------------------------------------------------------------ op-level entry points (diagnostics / unit tests) */
/* C[M,N] = op(A)[M,K] . op(B)[K,N] (+bias[N]) ; A stored (M,K) or, if trans_a, (K,M); B stored (K,N) or, if
 * trans_b, (N,K) [nn.Linear weight layout]; relu optional; C fp32 or bf16 per `dtype` (A,B in `dtype`). */
int egot2_gemm(int32_t dtype, int32_t M, int32_t N, int32_t K, const void* A, int32_t trans_a, const void* B,
               int32_t trans_b, const float* bias, int32_t relu, void* C, int32_t c_is_f32, int32_t accumulate,
               void* stream);
/* "tcgen05" | "simt": which GEMM implementation served the most recent GEMM of this thread (diagnostics). */
const char* egot2_gemm_last_impl(void);
int egot2_layernorm_fwd(int32_t dtype, int32_t rows, int32_t H, const void* x, const float* g, const float* b,
                        float eps, void* y, float* stat, void* stream);
/* self-attention over (B,T,3H) packed q|k|v -> (B,T,H); lse (B,heads,T). */
int egot2_attention_fwd(int32_t dtype, int32_t B, int32_t T, int32_t H, int32_t heads, const void* qkv, void* out,
                        float* lse, float p_drop, int32_t training, uint64_t seed, void* stream);
int egot2_attention_bwd(int32_t dtype, int32_t B, int32_t T, int32_t H, int32_t heads, const void* qkv,
                        const void* out, const float* lse, const void* dout, void* dqkv, float p_drop,
                        int32_t training, uint64_t seed, void* workspace, size_t ws_bytes, void* stream);

size_t egot2_attention_bwd_workspace_bytes(int32_t dtype, int32_t B, int32_t T, int32_t H, int32_t heads);
/* pooled[b,:] = mean_t x[b,t,:] (pool=1) or the first row_tokens tokens of every clip (pool=0; the ASD-of-interest
 * translator returns encoder tokens, HHI/models/asd/model_taskspecific.py:156-157); pooled is fp32. */
int egot2_pool_fwd(int32_t dtype, int32_t B, int32_t T, int32_t H, int32_t pool, int32_t row_tokens, const void* x,
                   float* pooled, void* stream);
int egot2_pool_bwd(int32_t dtype, int32_t B, int32_t T, int32_t H, int32_t pool, int32_t row_tokens,
                   const float* dpooled, void* dx, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EGOT2_H_ */
