// extern "C" surface of libb200st (see include/b200st.h).
#include "../../include/b200st.h"
#include "gemm.cuh"
#include "kernels.cuh"
#include "pdl.cuh"
#include "model.cuh"
#include <cstring>
#include <cstdlib>
#include "pdl.cuh"
#include <cmath>

namespace b200st {
static thread_local std::string g_last_error;
void set_last_error(const std::string& s) { g_last_error = s; }
int64_t g_kernel_launches = 0;
cudaError_t& pdl_launch_error() { static thread_local cudaError_t e = cudaSuccess; return e; }
bool pdl_enabled() { static const bool on = getenv("B200ST_NO_PDL") == nullptr; return on; }
}  // namespace b200st

using namespace b200st;

extern "C" {

const char* b200st_last_error(void) { return g_last_error.c_str(); }
int b200st_version(void) { return 201; }
int64_t b200st_launch_count(void) { return g_kernel_launches + tc_launch_count(); }

static GemmOperand to_operand(const b200st_operand& o) {
  GemmOperand r;
  r.ptr = o.ptr; r.dtype = o.dtype; r.mn_major = o.mn_major; r.ld = o.ld; r.sb1 = o.sb1; r.sb2 = o.sb2;
  return r;
}

static int convert_gemm(const b200st_gemm_args* a, GemmArgs& g);

int b200st_gemm(const b200st_gemm_args* a, void* stream) {
  if (!a) B200ST_FAIL("null args");
  GemmArgs g;
  B200ST_TRY(convert_gemm(a, g));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (a->force_simt) { if (g.splitk != 1) g.splitk = 1; return gemm_simt_f32(g, s); }
  return gemm(g, s);
}

int b200st_gemm_bench(const b200st_gemm_args* a, int32_t iters, float* ms_per_iter, void* stream) {
  if (!a || !ms_per_iter || iters <= 0) B200ST_FAIL("bad args");
  GemmArgs g;
  B200ST_TRY(convert_gemm(a, g));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  cudaEvent_t e0, e1;
  B200ST_CUDA(cudaEventCreate(&e0));
  B200ST_CUDA(cudaEventCreate(&e1));
  for (int i = 0; i < 3; ++i) B200ST_TRY(gemm(g, s));
  B200ST_CUDA(cudaEventRecord(e0, s));
  for (int i = 0; i < iters; ++i) B200ST_TRY(gemm(g, s));
  B200ST_CUDA(cudaEventRecord(e1, s));
  B200ST_CUDA(cudaEventSynchronize(e1));
  float ms = 0.f;
  B200ST_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  *ms_per_iter = ms / iters;
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  return 0;
}

static int convert_gemm(const b200st_gemm_args* a, GemmArgs& g) {
  g = gemm_defaults();
  g.M = a->M; g.N = a->N; g.K = a->K; g.nb1 = a->nb1 > 0 ? a->nb1 : 1; g.nb2 = a->nb2 > 0 ? a->nb2 : 1;
  g.A = to_operand(a->A); g.B = to_operand(a->B);
  g.C = a->C; g.c_dtype = a->c_dtype; g.ldc = a->ldc; g.c_sb1 = a->c_sb1; g.c_sb2 = a->c_sb2;
  g.epi.alpha = a->alpha;
  g.epi.bias = a->bias;
  g.epi.relu = a->relu;
  g.epi.mask_src = a->mask_src; g.epi.mask_dtype = a->mask_dtype;
  g.epi.mask_ld = a->mask_ld; g.epi.mask_sb1 = a->mask_sb1; g.epi.mask_sb2 = a->mask_sb2;
  if (a->dropout_p > 0.f) {
    B200ST_CHECK(a->dropout_p < 1.f, "dropout_p must be < 1");
    g.epi.drop = DropoutSpec{a->dropout_p, 1.f / (1.f - a->dropout_p), a->dropout_seed, a->dropout_stream, nullptr, nullptr};
  }
  g.epi.residual = a->residual; g.epi.res_ld = a->res_ld; g.epi.res_sb1 = a->res_sb1; g.epi.res_sb2 = a->res_sb2;
  g.epi.accumulate = a->accumulate;
  g.splitk = a->splitk;
  return 0;
}

int b200st_profile_begin(void) { tc_profile_begin(); return 0; }
int b200st_profile_end(double* gemm_ms, double* gemm_flops, int64_t* gemm_launches) {
  return tc_profile_end(gemm_ms, gemm_flops, gemm_launches);
}


struct b200st_model { Model m; };

int b200st_create(const b200st_config* cfg, b200st_handle* out) {
  if (!cfg || !out) B200ST_FAIL("null argument");
  b200st_model* h = new b200st_model();
  Config& c = h->m.cfg;
  c.model_type = cfg->model_type;
  c.d = cfg->d; c.heads = cfg->heads; c.ffn = cfg->ffn; c.enc_layers = cfg->enc_layers; c.dec_layers = cfg->dec_layers;
  c.vocab = cfg->vocab; c.src_vocab = cfg->src_vocab;
  c.feat = cfg->feat; c.in_channels = cfg->in_channels; c.channels = cfg->channels; c.conv_layer_norm = cfg->conv_layer_norm;
  c.precision = cfg->precision;
  c.ln_eps = cfg->ln_eps > 0.f ? cfg->ln_eps : 1e-6f;
  c.attention_dropout = cfg->attention_dropout; c.ffn_dropout = cfg->ffn_dropout; c.postprocess_dropout = cfg->postprocess_dropout;
  c.label_smoothing = cfg->label_smoothing;
  c.share_src_trg_embedding = cfg->share_src_trg_embedding;
  c.mha_self = cfg->mha_self; c.mha_din = cfg->mha_din; c.mha_dmem = cfg->mha_dmem; c.mha_dout = cfg->mha_dout;
  c.with_cross_attention = cfg->with_cross_attention;
  c.disable_fused_attention = cfg->disable_fused_attention;
  c.deterministic = cfg->deterministic;
  if (c.model_type < 0 || c.model_type > MODEL_MHA) { delete h; B200ST_FAIL("unknown model_type"); }
  if (c.attention_dropout < 0 || c.attention_dropout >= 1 || c.ffn_dropout < 0 || c.ffn_dropout >= 1 ||
      c.postprocess_dropout < 0 || c.postprocess_dropout >= 1) { delete h; B200ST_FAIL("dropout rates must be in [0,1)"); }
  if (int r = build_param_table(h->m)) { delete h; return r; }
  *out = h;
  return 0;
}
static Batch to_batch(const b200st_batch* b);
static Buffers to_buffers(const b200st_buffers* b);
int b200st_comm_unique_id(char* out128) {
  if (!out128) B200ST_FAIL("null argument");
  return comm_unique_id(out128);
}
int b200st_comm_init(b200st_handle h, const char* id128, int32_t nranks, int32_t rank) {
  if (!h || !id128) B200ST_FAIL("null argument");
  if (h->m.sync) { comm_destroy(h->m.sync); h->m.sync = nullptr; }
  return comm_init(&h->m.sync, id128, nranks, rank);
}
int b200st_comm_destroy(b200st_handle h) {
  if (!h) B200ST_FAIL("null handle");
  if (h->m.sync) { comm_destroy(h->m.sync); h->m.sync = nullptr; }
  return 0;
}
int b200st_comm_stats(b200st_handle h, int64_t* reduced_elems, int32_t* calls, int32_t* world) {
  if (!h) B200ST_FAIL("null handle");
  if (reduced_elems) *reduced_elems = comm_reduced_elems(h->m.sync);
  if (calls) *calls = comm_calls(h->m.sync);
  if (world) *world = comm_world(h->m.sync);
  return 0;
}
int b200st_comm_broadcast(b200st_handle h, float* buf, int64_t numel, int32_t root, void* stream) {
  if (!h || !buf) B200ST_FAIL("null argument");
  if (!h->m.sync) B200ST_FAIL("b200st_comm_init has not been called on this handle");
  return comm_broadcast(h->m.sync, buf, numel, root, reinterpret_cast<cudaStream_t>(stream));
}
int b200st_train_step(b200st_handle h, const b200st_buffers* buf, const b200st_batch* batch, const b200st_step_opts* opts, void* stream) {
  if (!h || !buf || !batch) B200ST_FAIL("null argument");
  if (batch->B <= 0 || batch->T <= 0 || batch->L <= 0) B200ST_FAIL("empty batch");
  Batch b = to_batch(batch);
  b.allreduce_grads = (opts && opts->allreduce_grads) ? 1 : 0;
  B200ST_TRY(model_forward(h->m, to_buffers(buf), b, true, reinterpret_cast<cudaStream_t>(stream)));
  if (opts && opts->optim) return b200st_optimizer_step(h, opts->optim, stream);
  return 0;
}
int b200st_destroy(b200st_handle h) {
  // a still-open communicator is left to the process teardown: ncclCommDestroy from a destructor that runs while the other
  // ranks (or the CUDA context) are already gone can block — b200st_comm_destroy is the explicit, collective-ordered exit
  delete h;
  return 0;
}
int64_t b200st_param_arena_numel(b200st_handle h) { return h ? h->m.arena_numel : -1; }
int32_t b200st_param_count(b200st_handle h) { return h ? (int32_t)h->m.params.size() : -1; }
int b200st_param_info(b200st_handle h, int32_t i, char* name, int32_t name_cap, int64_t* offset, int32_t* ndim, int64_t* shape4) {
  if (!h || i < 0 || i >= (int)h->m.params.size()) B200ST_FAIL("bad parameter index");
  const ParamInfo& p = h->m.params[i];
  if (name && name_cap > 0) { strncpy(name, p.name.c_str(), name_cap - 1); name[name_cap - 1] = 0; }
  if (offset) *offset = p.offset;
  if (ndim) *ndim = p.ndim;
  if (shape4) for (int k = 0; k < 4; ++k) shape4[k] = p.shape[k];
  return 0;
}

static Buffers to_buffers(const b200st_buffers* b) {
  Buffers r{};
  if (b) {
    r.params = b->params; r.shadow = b->shadow; r.grads = b->grads;
    r.workspace = b->workspace; r.workspace_bytes = (size_t)b->workspace_bytes;
  }
  return r;
}
static Batch to_batch(const b200st_batch* b) {
  Batch r{};
  r.src = b->src; r.src_ids = b->src_ids; r.src_length = b->src_length; r.src_padding = b->src_padding;
  r.trg_input = b->trg_input; r.trg = b->trg; r.trg_length = b->trg_length;
  r.B = b->B; r.T = b->T; r.L = b->L; r.training = b->training; r.seed = b->seed; r.seed_dev = b->seed_dev; r.loss_scale = b->loss_scale; r.loss_scale_dev = b->loss_scale_dev;
  r.logits = b->logits; r.loss = b->loss; r.nll_sum = b->nll_sum; r.n_tokens = b->n_tokens; r.enc_out = b->enc_out;
  return r;
}

int64_t b200st_workspace_bytes(b200st_handle h, int32_t B, int32_t T, int32_t L, int32_t training) {
  if (!h) return -1;
  return (int64_t)model_workspace_bytes(h->m, B, T, L, training);
}
int b200st_forward(b200st_handle h, const b200st_buffers* buf, const b200st_batch* batch, void* stream) {
  if (!h || !buf || !batch) B200ST_FAIL("null argument");
  if (batch->B <= 0 || batch->T <= 0 || batch->L <= 0) B200ST_FAIL("empty batch");
  return model_forward(h->m, to_buffers(buf), to_batch(batch), false, reinterpret_cast<cudaStream_t>(stream));
}
int b200st_forward_backward(b200st_handle h, const b200st_buffers* buf, const b200st_batch* batch, void* stream) {
  if (!h || !buf || !batch) B200ST_FAIL("null argument");
  if (batch->B <= 0 || batch->T <= 0 || batch->L <= 0) B200ST_FAIL("empty batch");
  return model_forward(h->m, to_buffers(buf), to_batch(batch), true, reinterpret_cast<cudaStream_t>(stream));
}
int b200st_encode(b200st_handle h, const b200st_buffers* buf, const b200st_batch* batch, float* enc_out, float* enc_bias,
                  void* stream) {
  if (!h || !buf || !batch || !enc_out) B200ST_FAIL("null argument");
  if (batch->B <= 0 || batch->T <= 0) B200ST_FAIL("empty batch");
  Batch b = to_batch(batch);
  b.L = 1; b.trg = nullptr; b.trg_length = nullptr; b.logits = nullptr;
  b.enc_out = enc_out; b.stop_after_encoder = 1; b.enc_bias_out = enc_bias;
  return model_forward(h->m, to_buffers(buf), b, false, reinterpret_cast<cudaStream_t>(stream));
}
int64_t b200st_encode_workspace_bytes(b200st_handle h, int32_t B, int32_t T) {
  if (!h) return -1;
  return (int64_t)model_workspace_bytes(h->m, B, T, 1, 0);
}
static DecodeState to_state(const b200st_decode_state* s) {
  DecodeState d{};
  d.B = s->B; d.Tm = s->Tm; d.max_len = s->max_len;
  d.cross_kv = s->cross_kv; d.self_kv = s->self_kv; d.memory_bias = s->memory_bias; d.scratch = s->scratch;
  d.use_shadow = s->use_shadow;
  return d;
}
int64_t b200st_decode_scratch_floats(b200st_handle h, int32_t B) {
  if (!h) return -1;
  return decode_scratch_floats(h->m, B);
}
int b200st_decode_init(b200st_handle h, const b200st_buffers* buf, const float* enc_out, const b200st_decode_state* st, void* stream) {
  if (!h || !buf || !st) B200ST_FAIL("null argument");
  return decode_init(h->m, to_buffers(buf), enc_out, to_state(st), reinterpret_cast<cudaStream_t>(stream));
}
int b200st_decode_step(b200st_handle h, const b200st_buffers* buf, const b200st_decode_state* st, const int64_t* symbols,
                       const int32_t* time_dev, float* logits, void* stream) {
  if (!h || !buf || !st) B200ST_FAIL("null argument");
  return decode_step(h->m, to_buffers(buf), to_state(st), symbols, time_dev, logits, reinterpret_cast<cudaStream_t>(stream));
}
int b200st_greedy_search(b200st_handle h, const b200st_buffers* buf, const b200st_decode_state* st, const b200st_greedy_args* a,
                         void* stream) {
  if (!h || !buf || !st || !a) B200ST_FAIL("null argument");
  GreedyArgs g{};
  g.bos_ids = a->bos_ids; g.eos_id = a->eos_id; g.unk_id = a->unk_id; g.min_len = a->min_len; g.max_steps = a->max_steps;
  g.out_ids = a->out_ids; g.out_len = a->out_len; g.out_logprob = a->out_logprob; g.state_words = a->state_words;
  g.use_graph = a->use_graph;
  return greedy_search(h->m, to_buffers(buf), to_state(st), g, reinterpret_cast<cudaStream_t>(stream));
}
int32_t b200st_greedy_used_graph(void) { return last_greedy_used_graph(); }
int b200st_refresh_shadow(const float* params, void* shadow, int32_t shadow_dtype, int64_t numel, void* stream) {
  if (!params || !shadow) B200ST_FAIL("null argument");
  return cast_f32_to_16(params, shadow, shadow_dtype, numel, reinterpret_cast<cudaStream_t>(stream));
}
static void fill_tensor_table(const Model& m, TensorTable& tt) {
  tt.n = 0;
  if (m.params.size() > 512) return;
  for (const ParamInfo& p : m.params) tt.off8[tt.n++] = (uint32_t)(p.offset >> 3);
  tt.off8[tt.n] = (uint32_t)(m.arena_numel >> 3);
}
int b200st_optimizer_step(b200st_handle h, const b200st_optim_args* a, void* stream) {
  if (!a || !a->params || !a->grads || !a->m || !a->v) B200ST_FAIL("bad optimizer arguments");
  if (!a->loss_scale_state && a->step_t < 1) B200ST_FAIL("step_t counts from 1");
  OptimArgs o{};
  o.p = a->params; o.g = a->grads; o.m = a->m; o.v = a->v;
  o.shadow = a->shadow; o.shadow_dtype = a->shadow_dtype;
  o.n = a->numel;
  o.lr = a->lr; o.beta1 = a->beta1; o.beta2 = a->beta2; o.eps = a->eps; o.step_t = a->step_t;
  o.grad_scale = a->grad_scale; o.zero_grad = a->zero_grad;
  o.clip_value = a->clip_value; o.clip_norm = a->clip_norm;
  o.tensor_sumsq = a->tensor_sumsq; o.ctl = a->loss_scale_state;
  o.growth_steps = a->growth_steps; o.multiplier = a->multiplier;
  TensorTable tt{};
  if (h) {
    if (a->numel != h->m.arena_numel) B200ST_FAIL("numel does not match the handle's parameter arena");
    fill_tensor_table(h->m, tt);
  } else if (a->clip_norm > 0.f || a->loss_scale_state) {
    // no handle: the whole arena is one tensor
    tt.n = 1; tt.off8[0] = 0; tt.off8[1] = (uint32_t)((a->numel + 7) >> 3);
  }
  return optimizer_step(o, tt, reinterpret_cast<cudaStream_t>(stream));
}
int b200st_adam_step(float* params, float* grads, float* m, float* v, void* shadow, int64_t numel, float lr, float beta1,
                     float beta2, float eps, int64_t step_t, float grad_scale, int32_t zero_grad, void* stream) {
  b200st_optim_args a{};
  a.params = params; a.grads = grads; a.m = m; a.v = v; a.shadow = shadow; a.shadow_dtype = B200ST_BF16; a.numel = numel;
  a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.step_t = step_t; a.grad_scale = grad_scale; a.zero_grad = zero_grad;
  return b200st_optimizer_step(nullptr, &a, stream);
}
int b200st_encoder_forward(b200st_handle h, const b200st_buffers* buf, const float* x, const float* padding, int32_t B,
                           int32_t T, float* out, int32_t training, uint64_t seed, void* stream, uint64_t* need_bytes) {
  if (!h) B200ST_FAIL("null handle");
  size_t need = 0;
  int r = encoder_forward_api(h->m, to_buffers(buf), x, padding, B, T, out, training, seed, reinterpret_cast<cudaStream_t>(stream),
                              need_bytes ? &need : nullptr);
  if (need_bytes) *need_bytes = need;
  return r;
}
int b200st_decoder_forward(b200st_handle h, const b200st_buffers* buf, const float* x, const float* memory,
                           const float* memory_padding, int32_t B, int32_t L, int32_t Tm, float* out, int32_t training,
                           uint64_t seed, void* stream, uint64_t* need_bytes) {
  if (!h) B200ST_FAIL("null handle");
  size_t need = 0;
  int r = decoder_forward_api(h->m, to_buffers(buf), x, memory, memory_padding, B, L, Tm, out, training, seed,
                              reinterpret_cast<cudaStream_t>(stream), need_bytes ? &need : nullptr);
  if (need_bytes) *need_bytes = need;
  return r;
}
int b200st_mha_forward(b200st_handle h, const b200st_buffers* buf, const float* query, const float* memory,
                       const float* bias_2d, int32_t B, int32_t Tq, int32_t Tk, float* out, void* stream, uint64_t* need_bytes) {
  if (!h) B200ST_FAIL("null handle");
  size_t need = 0;
  int r = mha_forward_api(h->m, to_buffers(buf), query, memory, bias_2d, B, Tq, Tk, out, reinterpret_cast<cudaStream_t>(stream),
                          need_bytes ? &need : nullptr);
  if (need_bytes) *need_bytes = need;
  return r;
}
int b200st_lsce(const float* logits, const int64_t* trg, const int64_t* trg_length, int32_t B, int32_t L, int32_t V,
                float label_smoothing, float* nll_sum, float* n_tokens, float* loss, void* dlogits, int32_t dlogits_dtype,
                float loss_scale, void* stream) {
  if (!logits || !trg || !trg_length || !nll_sum || !n_tokens || !loss) B200ST_FAIL("null argument");
  return lsce_fwd_bwd(logits, trg, trg_length, B, L, V, label_smoothing, nll_sum, n_tokens, loss, dlogits, dlogits_dtype,
                      loss_scale > 0.f ? loss_scale : 1.f, nullptr, reinterpret_cast<cudaStream_t>(stream));
}
int b200st_layernorm_fwd(const void* x, int32_t x_dtype, const float* gamma, const float* beta, float eps, void* y,
                         int32_t y_dtype, float* mean, float* rstd, int64_t rows, int32_t cols, int32_t relu, void* stream) {
  return layernorm_fwd(x, x_dtype, gamma, beta, eps, y, y_dtype, nullptr, mean, rstd, rows, cols, relu,
                       reinterpret_cast<cudaStream_t>(stream));
}
int b200st_layernorm_bwd(const void* dy, int32_t dy_dtype, const void* x, int32_t x_dtype, const float* mean,
                         const float* rstd, const float* gamma, const float* beta, const float* dres, void* dx,
                         int32_t dx_dtype, float* dgamma, float* dbeta, int64_t rows, int32_t cols, int32_t relu, void* stream) {
  return layernorm_bwd(dy, dy_dtype, x, x_dtype, mean, rstd, gamma, beta, dres, dx, dx_dtype, dgamma, dbeta, rows, cols, relu,
                       reinterpret_cast<cudaStream_t>(stream));
}
int b200st_softmax_fwd(const float* S, int64_t ldS, const float* bias_2d, int32_t causal, void* P, int32_t p_dtype,
                       int64_t ldP, int32_t B, int32_t H, int32_t Tq, int32_t Tk, void* stream) {
  if (!S || !P) B200ST_FAIL("null argument");
  return softmax_fwd(S, ldS, bias_2d, causal, P, nullptr, p_dtype, ldP, B, H, Tq, Tk, no_dropout(), reinterpret_cast<cudaStream_t>(stream));
}
int b200st_conv1_ln_relu_fwd(const float* src, const float* w, const float* b, const float* gamma, const float* beta,
                             void* y1, int32_t dtype, int32_t B, int32_t T, int32_t F, int32_t Cin, int32_t C,
                             int32_t use_ln, void* stream) {
  return conv1_ln_relu_fwd(src, w, b, gamma, beta, 1e-6f, y1, dtype, B, T, F, Cin, C, use_ln, reinterpret_cast<cudaStream_t>(stream));
}

uint64_t b200st_dropout_stream_id(const char* site) { return site ? dropout_stream_id(site) : 0; }

}  // extern "C"

namespace b200st {
__global__ void dropout_mask_kernel(uint64_t seed, uint64_t stream_id, int64_t n, float p, uint8_t* out) {
  pdl_wait();
  pdl_trigger();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = dropout_keep(seed, stream_id, (uint64_t)i, p) ? 1 : 0;
}
}  // namespace b200st

extern "C" int b200st_dropout_mask(uint64_t seed, uint64_t stream_id, int64_t n, float p, uint8_t* out, void* stream) {
  if (!out || n < 0) B200ST_FAIL("bad arguments");
  if (n == 0) return 0;
  int64_t g = (n + 255) / 256;
  if (g > 148 * 16) g = 148 * 16;
  launch_pdl(b200st::dropout_mask_kernel, (int)g, 256, 0, reinterpret_cast<cudaStream_t>(stream), seed, stream_id, n, p, out);
  B200ST_LAUNCH_CHECK();
  return 0;
}

