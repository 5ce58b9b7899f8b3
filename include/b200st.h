/* libb200st — C ABI of the B200-native SpeechTransformer hot path.
 *
 * Drop-in boundary for bytedance/neurst (reference @ /root/reference).  The reference is pure Python; its
 * "FFI" for this path is the class registry (neurst/utils/registry.py:24-137) through which Trainer and the
 * models reach the neurst/layers and neurst/criterions packages.  Each entry point below replaces the TF/PyTorch
 * library ops behind one reference function (file:line cited per function); INTEGRATION.md shows the
 * ctypes binding a maintainer adds.
 *
 * Conventions: every pointer is a DEVICE pointer owned by the caller (weights, activations, workspace);
 * every call is asynchronous on the given cudaStream_t (passed as void*); return 0 = ok, non-zero = error
 * with a thread-local message from b200st_last_error(); no exceptions cross the ABI; the library never
 * allocates device memory.  dtype codes: 0 = fp32, 1 = bf16.
 */
#ifndef B200ST_H_
#define B200ST_H_
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define B200ST_F32 0
#define B200ST_BF16 1
#define B200ST_F16 2   /* IEEE half: forward values of the mixed16 precision */

const char* b200st_last_error(void);
int b200st_version(void);
/* number of hand-written kernels launched by this process so far (bench.py "gpu_launches") */
int64_t b200st_launch_count(void);

/* ---- generic contraction (tf.einsum / Dense / tf.matmul sites; neurst/layers/common_layers.py:270,276-288,
 *      multi_head_attention.py:145,215; text_modalities.py:104-108) ---------------------------------------
 * C[b2][b1][m][n] = epi(alpha * sum_k A(m,k) B(n,k)); operands K-major (mn_major=0) or MN-major (1).
 * bf16 operands -> tcgen05/TMEM/TMA kernel; fp32 operands -> fp32 FMA kernel (parity mode). */
typedef struct {
  const void* ptr; int32_t dtype; int32_t mn_major; int64_t ld, sb1, sb2;
} b200st_operand;
typedef struct {
  int32_t M, N, K, nb1, nb2;
  b200st_operand A, B;
  void* C; int32_t c_dtype; int64_t ldc, c_sb1, c_sb2;
  float alpha;
  const float* bias;
  int32_t relu;
  const void* mask_src; int32_t mask_dtype; int64_t mask_ld, mask_sb1, mask_sb2;
  float dropout_p; uint64_t dropout_seed, dropout_stream;
  const float* residual; int64_t res_ld, res_sb1, res_sb2;
  int32_t accumulate;
  int32_t splitk;        /* 1 = none, 0 = auto (linear fp32 accumulate epilogues only) */
  int32_t force_simt;    /* tests: run the fp32-FMA kernel even on bf16 operands */
} b200st_gemm_args;
int b200st_gemm(const b200st_gemm_args* args, void* stream);


/* ---- model handle ------------------------------------------------------------------------------------
 * model_type: 0 = SpeechTransformer (neurst/models/speech_transformer.py:27-280), 1 = text Transformer
 * (neurst/models/transformer.py), 2 = TransformerEncoder stack only (layers/encoders/transformer_encoder.py:23-136),
 * 3 = TransformerDecoder stack only (layers/decoders/transformer_decoder.py:23-228), 4 = MultiHeadAttention /
 * MultiHeadSelfAttention (layers/attentions/multi_head_attention.py:21-290).
 * precision: B200ST_F32 = fp32 FMA kernels (parity mode, any shape); B200ST_F16 / B200ST_BF16 = tcgen05 kernels with every
 * 16-bit tensor (weights shadow, activations, activation gradients) in that type, fp32 accumulation, fp32 master weights,
 * fp32 parameter gradients.  B200ST_F16 is the reference's own mixed precision (mixed_float16 + dynamic loss scaling,
 * neurst/training/training_utils.py:73-81,413-416): 11-bit significands, needs loss scaling (b200st_batch.loss_scale_dev +
 * b200st_optimizer_step); B200ST_BF16 needs none but carries 8-bit significands. */
typedef struct b200st_model* b200st_handle;
typedef struct {
  int32_t model_type;
  int32_t d, heads, ffn, enc_layers, dec_layers, vocab, src_vocab;
  int32_t feat, in_channels, channels, conv_layer_norm;
  int32_t precision;
  float ln_eps, attention_dropout, ffn_dropout, postprocess_dropout, label_smoothing;
  int32_t share_src_trg_embedding;
  int32_t mha_self, mha_din, mha_dmem, mha_dout;
  int32_t with_cross_attention;
  int32_t disable_fused_attention;   /* tests: materialised attention (GEMM + softmax kernels) and unfused FFN in the 16-bit modes */
  int32_t deterministic;             /* 1: the hidden-dimension slices of the fused FFN kernel reduce into the output in slice
                                      * order (ticket per row tile) instead of arrival order: bit-reproducible steps for a few
                                      * microseconds per FFN launch (default 0: fp32 sums in arrival order) */
} b200st_config;

int b200st_create(const b200st_config* cfg, b200st_handle* out);   /* host object only; no device memory */
int b200st_destroy(b200st_handle h);

/* Parameter arena: one flat fp32 buffer; tensors in the reference's TF layouts (dense [in,out], conv HWIO,
 * embedding [V,d]; SURVEY.md Appendix B), each starting at a multiple of 8 elements. */
int64_t b200st_param_arena_numel(b200st_handle h);
int32_t b200st_param_count(b200st_handle h);
int b200st_param_info(b200st_handle h, int32_t i, char* name, int32_t name_cap, int64_t* offset, int32_t* ndim,
                      int64_t* shape4);

typedef struct {
  const float* params;      /* fp32 master arena */
  const void* shadow;       /* 16-bit copy of the arena in the handle's precision (b200st_refresh_shadow / b200st_optimizer_step) */
  float* grads;             /* fp32, same layout; gradients are ACCUMULATED into it */
  void* workspace; uint64_t workspace_bytes;   /* >= b200st_workspace_bytes(...) , 256-byte aligned */
} b200st_buffers;

/* One batch in the reference's input-dict form (neurst/tasks/speech2text.py:135-161). */
typedef struct {
  const float* src;             /* speech: fp32 [B,T,feat,in_channels] */
  const int64_t* src_ids;       /* text:   [B,T] */
  const int64_t* src_length;    /* speech: [B] frames */
  const float* src_padding;     /* text:   [B,T] 1.0 = pad */
  const int64_t* trg_input;     /* [B,L] */
  const int64_t* trg;           /* [B,L] or NULL */
  const int64_t* trg_length;    /* [B]   or NULL */
  int32_t B, T, L;
  int32_t training;             /* dropout on */
  uint64_t seed;                /* dropout seed of this step */
  const uint64_t* seed_dev;     /* optional device-resident seed (read at kernel run time: CUDA-graph replay) */
  float loss_scale;             /* multiplies the loss gradient (0 => 1) */
  const float* loss_scale_dev;  /* optional device word, multiplied in too: the dynamic loss scale (element 0 of the
                                 * b200st_optimizer_step state), read at kernel run time so CUDA-graph replays follow it */
  float* logits;                /* out, optional: fp32 [B,L,V] */
  float* loss;                  /* out, optional: [1] = sum(nll)/sum(tokens) (label_smoothed_cross_entropy.py:46-53) */
  float* nll_sum;               /* out, optional: [B] */
  float* n_tokens;              /* out, optional: [B] */
  float* enc_out;               /* out, optional: fp32 [B,T',d] */
} b200st_batch;

int64_t b200st_workspace_bytes(b200st_handle h, int32_t B, int32_t T, int32_t L, int32_t training);
/* EncoderDecoderModel.call (+ criterion when trg given): neurst/models/encoder_decoder_model.py:263-279 */
int b200st_forward(b200st_handle h, const b200st_buffers* buf, const b200st_batch* batch, void* stream);
/* forward + label-smoothed CE + full backward (GradAccumKerasModel.train_step, gradaccum_keras_model.py:190-245) */
int b200st_forward_backward(b200st_handle h, const b200st_buffers* buf, const b200st_batch* batch, void* stream);

/* ---- data-parallel training step (SURVEY.md 8b/8e): NCCL over NVLink only, inside the library -----------------------------
 * One process per GPU.  Rank 0 calls b200st_comm_unique_id, the 128 bytes travel to the other ranks by any host channel,
 * every rank calls b200st_comm_init (ncclCommInitRank; libnccl.so.2 is dlopen'ed from the process or the system).
 * b200st_train_step = forward + loss + backward (+ allreduce_grads: ncclAllReduce(sum) of the fp32 gradient arena in
 * reverse-order buckets — decoder+output layer / upper encoder half / lower encoder half / front-end — each issued on the
 * library's communication stream the moment its last gradient kernel has been enqueued, so the transfers run under the
 * rest of the backward pass; `stream` waits for them at the end) (+ optim != NULL: b200st_optimizer_step with
 * grad_scale = 1/(replicas * update_cycle) = hvd.Average, neurst/training/hvd_utils.py:48-62).
 * b200st_comm_broadcast: rank-0 parameters to all (neurst/exps/trainer.py:285). */
int b200st_comm_unique_id(char* out128);
int b200st_comm_init(b200st_handle h, const char* id128, int32_t nranks, int32_t rank);
int b200st_comm_broadcast(b200st_handle h, float* buf, int64_t numel, int32_t root, void* stream);
/* call on every rank before the process group goes away; destroy every CUDA graph that captured b200st_train_step with
 * allreduce_grads first: ncclCommDestroy waits for the graphs that reference the communicator */
int b200st_comm_destroy(b200st_handle h);
int b200st_comm_stats(b200st_handle h, int64_t* reduced_elems, int32_t* calls, int32_t* world);   /* of the last step */
struct b200st_optim_args_;
typedef struct {
  int32_t allreduce_grads;
  const struct b200st_optim_args_* optim;     /* NULL: no optimizer step (gradient accumulation micro-step) */
} b200st_step_opts;
int b200st_train_step(b200st_handle h, const b200st_buffers* buf, const b200st_batch* batch, const b200st_step_opts* opts,
                      void* stream);

/* ---- inference: encoder pass, cached decoder step, greedy search (SURVEY.md 8 f1, BASELINE cfg-5) ---------------------
 * b200st_encode: modality + TransformerEncoder only (EncoderDecoderModel.get_symbols_to_logits_fn up to
 * create_decoding_internal_cache, neurst/models/encoder_decoder_model.py:230-241): enc_out fp32 [B,T',d], enc_bias fp32
 * [B,T'] = the additive memory bias (0 / -1e9).  Uses batch->src, src_length (speech) or src_ids, src_padding (text). */
int b200st_encode(b200st_handle h, const b200st_buffers* buf, const b200st_batch* batch, float* enc_out, float* enc_bias,
                  void* stream);
int64_t b200st_encode_workspace_bytes(b200st_handle h, int32_t B, int32_t T);
/* Decoding state, caller-owned device buffers (nothing grows during decoding):
 *   cross_kv  fp32 [dec_layers][B][Tm][2d]: memory keys | values, projected once (transformer_layers.py:156-170)
 *   self_kv   fp32 [dec_layers][2][B][max_len][d]: self-attention key / value cache (multi_head_attention.py:271-289)
 *   scratch   b200st_decode_scratch_floats(h, B) floats
 * use_shadow 0: weights read from the fp32 master arena (token ids identical to an fp32 reference); 1: 16-bit shadow. */
typedef struct {
  int32_t B, Tm, max_len;
  float* cross_kv; float* self_kv;
  const float* memory_bias;
  float* scratch;
  int32_t use_shadow;
} b200st_decode_state;
int64_t b200st_decode_scratch_floats(b200st_handle h, int32_t B);
/* TransformerDecoder.create_decoding_internal_cache + memorize_memory (transformer_decoder.py:105-147) */
int b200st_decode_init(b200st_handle h, const b200st_buffers* buf, const float* enc_out, const b200st_decode_state* st, void* stream);
/* symbols_to_logits_fn(symbols, cache, time) (encoder_decoder_model.py:243-253): symbols int64 [B] and the position *time_dev
 * are device-resident; appends this position's keys/values to self_kv; logits fp32 [B,V]. */
int b200st_decode_step(b200st_handle h, const b200st_buffers* buf, const b200st_decode_state* st, const int64_t* symbols,
                       const int32_t* time_dev, float* logits, void* stream);
/* sequence_beam_search with beam_size = 1 (neurst/layers/search/beam_search.py:254-439): log_softmax, finished rows emit EOS,
 * UNK masked unless unk_id < 0, EOS masked before min_len, argmax (lowest index on ties), stop when every row has finished
 * or after max_steps = min(T' + extra_decode_length, maximum_decode_length); out_ids [B,max_steps] is padded with EOS.
 * The step is captured once into a CUDA graph and replayed (use_graph); `stream` must not be capturing. */
typedef struct {
  const int64_t* bos_ids;
  int32_t eos_id, unk_id, min_len, max_steps;
  int64_t* out_ids; int32_t* out_len; float* out_logprob;
  void* state_words;            /* >= 256 bytes of device memory */
  int32_t use_graph;            /* 2: ONE persistent cooperative kernel for the whole search (grid-wide barriers between the
                                 * phases of a token; falls back to 1 when the grid cannot be co-scheduled); 1: one captured
                                 * CUDA graph of ~40 kernels replayed per token; 0: eager launches */
} b200st_greedy_args;
int b200st_greedy_search(b200st_handle h, const b200st_buffers* buf, const b200st_decode_state* st, const b200st_greedy_args* a,
                         void* stream);
/* mode the last b200st_greedy_search actually ran in: 2 persistent kernel, 1 captured graph, 0 eager launches */
int32_t b200st_greedy_used_graph(void);

/* 16-bit shadow of the parameter arena (tcgen05 operands); shadow_dtype = B200ST_BF16 or B200ST_F16 */
int b200st_refresh_shadow(const float* params, void* shadow, int32_t shadow_dtype, int64_t numel, void* stream);

/* Optimizer step of GradAccumKerasModel.train_step (neurst/training/gradaccum_keras_model.py:222-240): unscale ->
 * tf.clip_by_value / tf.clip_by_norm PER GRADIENT TENSOR -> Keras Adam (epsilon-hat form), with the 16-bit shadow refresh and
 * gradient zeroing in the same pass.  loss_scale_state != NULL enables the reference's dynamic loss scale
 * (neurst/training/revised_dynamic_loss_scale.py:60-107): device float[8] = {scale, finite steps in a row, last step skipped,
 * skipped steps, applied steps, global gradient norm, 1/scale latch, reserved}; a step whose gradients are not all finite
 * is skipped (parameters untouched, gradients zeroed) and halves the scale; `growth_steps` finite steps double it.
 * h may be NULL (whole arena = one tensor). tensor_sumsq: device float[param_count + 1] scratch (clip_norm / loss scale). */
typedef struct b200st_optim_args_ {
  float* params; float* grads; float* m; float* v;
  void* shadow; int32_t shadow_dtype;
  int64_t numel;
  float lr, beta1, beta2, eps;
  int64_t step_t;               /* Adam's t (from 1) when loss_scale_state is NULL; else t = applied steps on the device */
  float grad_scale;             /* 1 / (replicas * update_cycle) */
  int32_t zero_grad;
  float clip_value, clip_norm;  /* <= 0: off */
  float* tensor_sumsq;
  float* loss_scale_state;
  float growth_steps, multiplier;   /* 0 => 2000, 2 */
} b200st_optim_args;
int b200st_optimizer_step(b200st_handle h, const b200st_optim_args* a, void* stream);
/* legacy form: plain Keras Adam with a bf16 shadow, epsilon-hat form (neurst/optimizers/__init__.py:21; hparams speech_transformer.py:265-270):
 * g' = g*grad_scale; m,v update; p -= lr*sqrt(1-b2^t)/(1-b1^t) * m/(sqrt(v)+eps); optional bf16 shadow refresh + g=0 */
int b200st_adam_step(float* params, float* grads, float* m, float* v, void* shadow, int64_t numel, float lr, float beta1,
                     float beta2, float eps, int64_t step_t, float grad_scale, int32_t zero_grad, void* stream);

/* layer-level forward (reference layer API).  need_bytes != NULL: only report the workspace size. */
int b200st_encoder_forward(b200st_handle h, const b200st_buffers* buf, const float* x, const float* padding, int32_t B,
                           int32_t T, float* out, int32_t training, uint64_t seed, void* stream, uint64_t* need_bytes);
int b200st_decoder_forward(b200st_handle h, const b200st_buffers* buf, const float* x, const float* memory,
                           const float* memory_padding, int32_t B, int32_t L, int32_t Tm, float* out, int32_t training,
                           uint64_t seed, void* stream, uint64_t* need_bytes);
int b200st_mha_forward(b200st_handle h, const b200st_buffers* buf, const float* query, const float* memory,
                       const float* bias_2d, int32_t B, int32_t Tq, int32_t Tk, float* out, void* stream,
                       uint64_t* need_bytes);

/* criterion alone: LabelSmoothedCrossEntropy.__call__/reduce_loss (label_smoothed_cross_entropy.py:94-157,46-53) */
int b200st_lsce(const float* logits, const int64_t* trg, const int64_t* trg_length, int32_t B, int32_t L, int32_t V,
                float label_smoothing, float* nll_sum, float* n_tokens, float* loss, void* dlogits, int32_t dlogits_dtype,
                float loss_scale, void* stream);
/* LayerNormalization (common_layers.py:64-65) */
int b200st_layernorm_fwd(const void* x, int32_t x_dtype, const float* gamma, const float* beta, float eps, void* y,
                         int32_t y_dtype, float* mean, float* rstd, int64_t rows, int32_t cols, int32_t relu, void* stream);
int b200st_layernorm_bwd(const void* dy, int32_t dy_dtype, const void* x, int32_t x_dtype, const float* mean,
                         const float* rstd, const float* gamma, const float* beta, const float* dres, void* dx,
                         int32_t dx_dtype, float* dgamma, float* dbeta, int64_t rows, int32_t cols, int32_t relu, void* stream);
/* softmax over keys with additive [B,Tk] bias / causal mask (multi_head_attention.py:147-160); S fp32 [B,H,Tq,ldS] */
int b200st_softmax_fwd(const float* S, int64_t ldS, const float* bias_2d, int32_t causal, void* P, int32_t p_dtype,
                       int64_t ldP, int32_t B, int32_t H, int32_t Tq, int32_t Tk, void* stream);
/* conv subsampling front-end pieces (audio_modalities.py:84-109) */
int b200st_conv1_ln_relu_fwd(const float* src, const float* w, const float* b, const float* gamma, const float* beta,
                             void* y1, int32_t dtype, int32_t B, int32_t T, int32_t F, int32_t Cin, int32_t C,
                             int32_t use_ln, void* stream);

/* dropout bookkeeping for tests: the keep-mask (uint8) of site `stream_id` under `seed`, element i in [0,n) */
uint64_t b200st_dropout_stream_id(const char* site);
int b200st_dropout_mask(uint64_t seed, uint64_t stream_id, int64_t n, float p, uint8_t* out, void* stream);

/* tests only: the fused 16-bit attention and FFN kernels called on their own (dt = 1 bf16, 2 fp16).
 * Dropout is a probability plus a caller-owned keep bitmap: byte g holds the keep bits of elements 8g .. 8g+7 (bit j =
 * element 8g+j, the packing of b200st_dropout_mask); a bitmap is required when p > 0.
 * Attention (head dim 64): q/k/v/ctx/dq/dk/dv are [B*T, ld] row views, head h at columns [64h, 64h+64); bias [B, Tk]
 * additive or NULL; kv_len [B] or NULL (keys >= kv_len[b] carry the -1e9 bias: whole key blocks past it are skipped);
 * keep_bits [B, H, Tq, round8(Tk)]; lse [B, H, Tq] (natural log); dq_scratch fp32 with B*Tq*H*64 + B*H*Tq elements. */
int b200st_attention_fwd(int32_t dt, const void* q, int64_t q_ld, const void* k, int64_t k_ld, const void* v, int64_t v_ld,
                         int32_t B, int32_t H, int32_t Tq, int32_t Tk, const float* bias, const int32_t* kv_len,
                         int32_t causal, float drop_p, const uint8_t* keep_bits, void* ctx, int64_t ctx_ld, float* lse,
                         void* stream);
int b200st_attention_bwd(int32_t dt, const void* q, int64_t q_ld, const void* k, int64_t k_ld, const void* v, int64_t v_ld,
                         int32_t B, int32_t H, int32_t Tq, int32_t Tk, const float* bias, const int32_t* kv_len,
                         int32_t causal, float drop_p, const uint8_t* keep_bits, const void* ctx, int64_t ctx_ld,
                         const void* dctx, int64_t dctx_ld, const float* lse, float* dq_scratch, void* dq, int64_t dq_ld,
                         void* dk, int64_t dk_ld, void* dv, int64_t dv_ld, void* stream);
/* FFN (d in {128, 256}, ffn % 128 == 0), all row-major and packed: X [M, d], W1 [d, ffn], W2 [ffn, d] in dt; b1 [ffn],
 * b2 [d] fp32 or NULL; ffn_bits [M, ffn], post_bits [M, d].  Forward: F1 = dropout(relu(X W1 + b1)) [M, ffn] in dt,
 * x_out [M, d] fp32 += post-dropout(F1 W2 + b2).  Backward: dF1 = scale * (dY W2^T) where F1 > 0 [M, ffn] in dt,
 * dH [M, d] fp32 += dF1 W1^T.  tickets: NULL, or int [ceil(M / 128)] all zero (slices then add in a fixed order; the
 * kernel leaves them zero).  splits_out (may be NULL): the number of hidden slices the launch used. */
int b200st_ffn_fwd(int32_t dt, const void* X, int32_t M, int32_t d, int32_t ffn, const void* W1, const float* b1,
                   const void* W2, const float* b2, float drop_ffn_p, const uint8_t* ffn_bits, float drop_post_p,
                   const uint8_t* post_bits, void* F1, float* x_out, int32_t* tickets, int32_t* splits_out, void* stream);
int b200st_ffn_bwd(int32_t dt, const void* dY, int32_t M, int32_t d, int32_t ffn, const void* W1, const void* W2,
                   const void* F1, float scale, void* dF1, float* dH, int32_t* tickets, int32_t* splits_out, void* stream);

/* tests/bench only: time `iters` back-to-back launches of one GEMM with CUDA events on `stream` (no host overhead) */
int b200st_gemm_bench(const b200st_gemm_args* args, int32_t iters, float* ms_per_iter, void* stream);

/* bench only: per-launch CUDA-event timing of the tcgen05 GEMM launches issued between begin and end
 * (sum of kernel durations in ms, sum of their algorithmic FLOPs, number of launches) */
int b200st_profile_begin(void);
int b200st_profile_end(double* gemm_ms, double* gemm_flops, int64_t* gemm_launches);

#ifdef __cplusplus
}
#endif
#endif /* B200ST_H_ */
