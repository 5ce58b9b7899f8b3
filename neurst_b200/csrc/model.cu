// Forward / backward orchestration of the SpeechTransformer hot path on top of the GEMM and elementwise kernels.
//
// Reference call stack being replaced (SURVEY.md §3.2): EncoderDecoderModel.call
// (neurst/models/encoder_decoder_model.py:263-279) -> SpeechTransformer.get_symbols_to_logits_fn
// (neurst/models/speech_transformer.py:179-189) -> AudioConv2dSubsamplingLayer / TransformerEncoder /
// TransformerDecoder / WordEmbeddingSharedWeights -> LabelSmoothedCrossEntropy.reduce_loss, and the backward
// TF autodiff derives from them (GradAccumKerasModel.train_step, gradaccum_keras_model.py:190-255).
#include "model.cuh"

#include <cmath>

namespace b200st {

// =============================================================================================
// parameter table
// =============================================================================================
static void add_param(Model& m, const std::string& name, std::initializer_list<int64_t> shape) {
  ParamInfo p;
  p.name = name;
  p.ndim = (int)shape.size();
  p.numel = 1;
  int i = 0;
  for (int64_t s : shape) { p.shape[i++] = s; p.numel *= s; }
  for (; i < 4; ++i) p.shape[i] = 1;
  p.offset = m.arena_numel;
  m.arena_numel += (p.numel + 7) / 8 * 8;
  m.index[name] = (int)m.params.size();
  m.params.push_back(p);
}

static void add_attention(Model& m, const std::string& pre, bool cross, int din, int dmem, int units, int dout, bool with_ln) {
  if (with_ln) { add_param(m, pre + ".ln.gamma", {din}); add_param(m, pre + ".ln.beta", {din}); }
  if (cross) {
    add_param(m, pre + ".q.kernel", {din, units}); add_param(m, pre + ".q.bias", {units});
    add_param(m, pre + ".kv.kernel", {dmem, 2 * units}); add_param(m, pre + ".kv.bias", {2 * units});
  } else {
    add_param(m, pre + ".qkv.kernel", {din, 3 * units}); add_param(m, pre + ".qkv.bias", {3 * units});
  }
  add_param(m, pre + ".out.kernel", {units, dout}); add_param(m, pre + ".out.bias", {dout});
}
static void add_ffn(Model& m, const std::string& pre, int d, int ffn) {
  add_param(m, pre + ".ln.gamma", {d}); add_param(m, pre + ".ln.beta", {d});
  add_param(m, pre + ".w1", {d, ffn}); add_param(m, pre + ".b1", {ffn});
  add_param(m, pre + ".w2", {ffn, d}); add_param(m, pre + ".b2", {d});
}

int build_param_table(Model& m) {
  const Config& c = m.cfg;
  m.params.clear(); m.index.clear(); m.arena_numel = 0;
  B200ST_CHECK(c.precision == F32 || c.precision == BF16 || c.precision == F16, "precision must be 0 (fp32), 1 (bf16) or 2 (fp16)");
  m.adt = c.precision;
  if (c.model_type == MODEL_MHA) {
    B200ST_CHECK(c.heads > 0 && c.d % c.heads == 0, "num_units must be divisible by heads");
    add_attention(m, "att", !c.mha_self, c.mha_din, c.mha_dmem, c.d, c.mha_dout, false);
    return 0;
  }
  B200ST_CHECK(c.d > 0 && c.heads > 0 && c.d % c.heads == 0, "hidden size must be divisible by heads");
  const bool has_enc = c.model_type != MODEL_DECODER, has_dec = c.model_type != MODEL_ENCODER;
  if (c.model_type == MODEL_SPEECH) {
    const int C = c.channels, F2 = ((c.feat + 1) / 2 + 1) / 2;
    add_param(m, "src.conv1.kernel", {3, 3, c.in_channels, C}); add_param(m, "src.conv1.bias", {C});
    add_param(m, "src.ln1.gamma", {C}); add_param(m, "src.ln1.beta", {C});
    add_param(m, "src.conv2.kernel", {3, 3, C, C}); add_param(m, "src.conv2.bias", {C});
    add_param(m, "src.ln2.gamma", {C}); add_param(m, "src.ln2.beta", {C});
    add_param(m, "src.dense.kernel", {(int64_t)F2 * C, c.d}); add_param(m, "src.dense.bias", {c.d});
  } else if (c.model_type == MODEL_TEXT && !c.share_src_trg_embedding) {
    add_param(m, "srcemb.emb", {c.src_vocab, c.d});
  }
  if (has_enc) {
    for (int i = 0; i < c.enc_layers; ++i) {
      const std::string p = "enc." + std::to_string(i);
      add_attention(m, p + ".att", false, c.d, c.d, c.d, c.d, true);
      add_ffn(m, p + ".ffn", c.d, c.ffn);
    }
    add_param(m, "enc.out_ln.gamma", {c.d}); add_param(m, "enc.out_ln.beta", {c.d});
  }
  if (has_dec) {
    for (int i = 0; i < c.dec_layers; ++i) {
      const std::string p = "dec." + std::to_string(i);
      add_attention(m, p + ".self", false, c.d, c.d, c.d, c.d, true);
      if (c.with_cross_attention) add_attention(m, p + ".cross", true, c.d, c.d, c.d, c.d, true);
      add_ffn(m, p + ".ffn", c.d, c.ffn);
    }
    add_param(m, "dec.out_ln.gamma", {c.d}); add_param(m, "dec.out_ln.beta", {c.d});
  }
  if (c.model_type == MODEL_SPEECH || c.model_type == MODEL_TEXT) {
    add_param(m, "trg.emb", {c.vocab, c.d}); add_param(m, "trg.bias", {c.vocab});
  }
  if (is16(c.precision)) {
    B200ST_CHECK(c.d % 8 == 0 && c.ffn % 8 == 0 && (c.d / c.heads) % 8 == 0, "bf16 mode needs d, ffn, head dim % 8 == 0");
    if (c.model_type == MODEL_SPEECH) B200ST_CHECK(c.channels % 8 == 0, "bf16 mode needs channels % 8 == 0");
    if (c.model_type <= MODEL_TEXT) B200ST_CHECK(c.vocab % 8 == 0, "bf16 mode needs vocab % 8 == 0");
  }
  return 0;
}

uint64_t dropout_stream_id(const std::string& site) {
  // "enc.in_drop" -> 1, "dec.in_drop" -> 2,
  // "enc.<i>.att.attn_drop" 1000+10i, ".att.post_drop" +1, ".ffn.ffn_drop" +2, ".ffn.post_drop" +3
  // "dec.<i>.self.attn_drop" 2000+10i, ".self.post_drop" +1, ".cross.attn_drop" +2, ".cross.post_drop" +3,
  // ".ffn.ffn_drop" +4, ".ffn.post_drop" +5
  if (site == "enc.in_drop") return 1;
  if (site == "dec.in_drop") return 2;
  const bool enc = site.rfind("enc.", 0) == 0;
  const size_t p1 = 4, p2 = site.find('.', p1);
  if (p2 == std::string::npos) return 0;
  const int layer = atoi(site.substr(p1, p2 - p1).c_str());
  const std::string rest = site.substr(p2 + 1);
  int code = -1;
  if (enc) {
    if (rest == "att.attn_drop") code = 0; else if (rest == "att.post_drop") code = 1;
    else if (rest == "ffn.ffn_drop") code = 2; else if (rest == "ffn.post_drop") code = 3;
  } else {
    if (rest == "self.attn_drop") code = 0; else if (rest == "self.post_drop") code = 1;
    else if (rest == "cross.attn_drop") code = 2; else if (rest == "cross.post_drop") code = 3;
    else if (rest == "ffn.ffn_drop") code = 4; else if (rest == "ffn.post_drop") code = 5;
  }
  if (code < 0) return 0;
  return (enc ? 1000 : 2000) + 10 * (uint64_t)layer + code;
}

// =============================================================================================
// execution context
// =============================================================================================
namespace {

struct Arena {
  char* base = nullptr;
  size_t cap = 0, off = 0;
  void* take(size_t bytes) {
    off = (off + 255) & ~(size_t)255;
    void* p = base + off;
    off += bytes;
    return p;
  }
};

// Weight / bias gradients are off the backward critical path (nothing in the step reads them before the optimizer), so
// they run on a second stream and fill the SMs the latency-bound dgrad chain leaves idle.  One process-wide stream +
// three events; inside a CUDA-graph capture the event edges become graph dependencies (fork / join).
struct SideStream {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, done[2] = {nullptr, nullptr}, bits_done = nullptr;
  bool ok = false;
};
static SideStream& side_stream() {
  static SideStream ss;
  static bool init = false;
  if (!init) {
    init = true;
    ss.ok = cudaStreamCreateWithFlags(&ss.stream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaEventCreateWithFlags(&ss.fork, cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&ss.done[0], cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&ss.done[1], cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&ss.bits_done, cudaEventDisableTiming) == cudaSuccess;
  }
  return ss;
}

struct Ctx {
  const Model& m;
  Buffers buf;
  cudaStream_t st;
  // ---- side stream for weight gradients (backward of the full model only) ----
  SideStream* side = nullptr;
  bool side_pending[2] = {false, false};
  int bwd_blocks = 0;
  int cur_par = 0;
  // Start of a backward block: picks the gradient-scratch parity and waits for the side-stream readers of that parity
  // (issued two blocks ago) before the block overwrites it.
  int begin_bwd_block() {
    cur_par = (bwd_blocks++) & 1;
    if (side && !dry && side_pending[cur_par]) {
      if (cudaStreamWaitEvent(st, side->done[cur_par], 0) != cudaSuccess) launch_failed = true;
      side_pending[cur_par] = false;
    }
    return cur_par;
  }
  // stream for a weight-gradient launch whose inputs were produced on `st` so far
  cudaStream_t wgrad_stream() {
    if (!side || dry) return st;
    if (cudaEventRecord(side->fork, st) != cudaSuccess || cudaStreamWaitEvent(side->stream, side->fork, 0) != cudaSuccess) {
      launch_failed = true;
      return st;
    }
    return side->stream;
  }
  void wgrad_done(cudaStream_t s) {
    if (!side || dry || s == st) return;
    if (cudaEventRecord(side->done[cur_par], s) != cudaSuccess) launch_failed = true;
    side_pending[cur_par] = true;
  }
  // Fused hand-over between backward blocks: the final LayerNorm-backward of a block also writes the NEXT block's
  // dY = cast(dropout'(dx)) into that block's parity buffer (set by the stack loop through `next_drop`).
  const DropoutSpec* next_drop = nullptr;   // post-dropout site of the block that runs next (null: no fused hand-over)
  bool dy_ready = false;                    // the previous block already produced this block's dY
  // parity the next block will select; its side-stream readers (two blocks ago) must be done before it is overwritten
  int next_parity_ready() {
    const int par = bwd_blocks & 1;
    if (side && !dry && side_pending[par]) {
      if (cudaStreamWaitEvent(st, side->done[par], 0) != cudaSuccess) launch_failed = true;
      side_pending[par] = false;
    }
    return par;
  }
  void join_side() {
    if (!side || dry) return;
    for (int i = 0; i < 2; ++i)
      if (side_pending[i]) {
        if (cudaStreamWaitEvent(st, side->done[i], 0) != cudaSuccess) launch_failed = true;
        side_pending[i] = false;
      }
  }
  // ---- data-parallel gradient buckets (comm.cu): [lo, hi) of the arena is final -> all-reduce it on the comm stream ----
  GradSync* sync = nullptr;
  int64_t sync_hi = 0;       // everything at or above this arena offset has already been handed to NCCL
  int reduce_down_to(const std::string& first_param) {
    if (!sync || dry) return 0;
    const ParamInfo* p = first_param.empty() ? nullptr : info(first_param);
    const int64_t lo = p ? p->offset : 0;
    if (lo >= sync_hi) return 0;
    // weight gradients of this range may still be running on the side stream: the comm stream waits for them directly
    cudaEvent_t e0 = (side && side_pending[0]) ? side->done[0] : nullptr, e1 = (side && side_pending[1]) ? side->done[1] : nullptr;
    const int rc = comm_reduce_range(sync, buf.grads, lo, sync_hi, st, e0, e1);
    sync_hi = lo;
    return rc;
  }
  // ragged batches: number of leading non-padded encoder positions per utterance; applies to attention calls whose key
  // bias is the encoder padding bias (encoder self-attention, decoder cross-attention)
  const float* klen_bias = nullptr;
  const int32_t* klen = nullptr;
  const int32_t* klen_for(const float* bias) const { return (bias && bias == klen_bias) ? klen : nullptr; }
  // deterministic mode: ticket words of the fused FFN kernel (one array per call, zeroed once, self-resetting)
  int* tickets = nullptr;
  int* mlp_tickets(int M) {
    if (!m.cfg.deterministic) return nullptr;
    if (!tickets) {
      tickets = reinterpret_cast<int*>(ar.take(sizeof(int) * 4096));
      if (!dry && cudaMemsetAsync(tickets, 0, sizeof(int) * 4096, st) != cudaSuccess) launch_failed = true;
    }
    return (M + 127) / 128 <= 4096 ? tickets : nullptr;
  }
  // weight gradients of the current backward block, launched together by flush_wgrads()
  struct PendingWgrad { GemmArgs g; float* db; const void* dY; int M, N; int64_t ldy; };
  std::vector<PendingWgrad> pending_wgrads;
  bool defer_wgrads = false;
  bool dry;        // planning pass: allocate only, launch nothing
  bool training;
  uint64_t seed;
  const uint64_t* seed_dev = nullptr;
  Arena ar;
  int adt;
  Ctx(const Model& mm, const Buffers& b, cudaStream_t s, bool d) : m(mm), buf(b), st(s), dry(d), training(false), seed(0), adt(mm.adt) {
    ar.base = reinterpret_cast<char*>(b.workspace);
    ar.cap = b.workspace_bytes;
  }
  size_t esz() const { return (size_t)dtype_size(adt); }
  void* act(int64_t n) { return ar.take((size_t)n * esz()); }
  float* f32(int64_t n) { return reinterpret_cast<float*>(ar.take((size_t)n * 4)); }
  std::unordered_map<uint64_t, DropoutSpec> drop_memo;
  bool launch_failed = false;
  struct DropSite { uint64_t stream; float p; int64_t groups; size_t arena_off; };
  std::vector<DropSite> drop_sites;      // recorded in allocation order (planning pass -> one batched generator launch)
  bool bits_pregenerated = false;
  // Dropout site `stream`.  The first (forward) use passes the element count: the keep-bits of the whole site are then
  // generated once into the workspace (one Philox call per 8 elements, full-occupancy kernel) and every consumer —
  // GEMM epilogues, fused attention, the backward pass — just reads bits.  Later uses return the memoised spec.
  cudaEvent_t bits_event = nullptr;      // keep-bit generation running on the side stream: the first consumer waits
  void wait_bits() {
    if (bits_event) {
      if (cudaStreamWaitEvent(st, bits_event, 0) != cudaSuccess) launch_failed = true;
      bits_event = nullptr;
    }
  }
  DropoutSpec drop(float p, uint64_t stream, int64_t n_elems = 0) {
    if (!training || p <= 0.f) return no_dropout();
    if (!dry) wait_bits();
    auto it = drop_memo.find(stream);
    if (it != drop_memo.end()) return it->second;
    DropoutSpec d{p, 1.f / (1.f - p), seed, stream, seed_dev, nullptr};
    if (n_elems > 0) {
      uint8_t* bits = reinterpret_cast<uint8_t*>(ar.take((size_t)((n_elems + 7) / 8 + 4)));
      drop_sites.push_back(DropSite{stream, p, (n_elems + 7) / 8, (size_t)(reinterpret_cast<char*>(bits) - ar.base)});
      if (!dry && !bits_pregenerated && dropout_bits(d, n_elems, bits, st) != 0) launch_failed = true;
      d.bits = bits;
      drop_memo[stream] = d;
    }
    return d;
  }
  const ParamInfo* info(const std::string& n) const {
    const int i = m.find(n);
    return i < 0 ? nullptr : &m.params[i];
  }
  const float* P(const std::string& n) const { const ParamInfo* p = info(n); return p ? buf.params + p->offset : nullptr; }
  float* G(const std::string& n) const { const ParamInfo* p = info(n); return (p && buf.grads) ? buf.grads + p->offset : nullptr; }
  // weight as GEMM operand in the compute dtype
  GemmOperand W(const std::string& n, int mn_major, int64_t ld) const {
    const ParamInfo* p = info(n);
    GemmOperand o{};
    if (!p) return o;
    if (is16(adt)) { o.ptr = reinterpret_cast<const uint16_t*>(buf.shadow) + p->offset; o.dtype = adt; }
    else { o.ptr = buf.params + p->offset; o.dtype = F32; }
    o.mn_major = mn_major; o.ld = ld;
    return o;
  }
  void* act_off(void* base, int64_t elems) const { return reinterpret_cast<char*>(base) + (size_t)elems * esz(); }
  const void* act_off(const void* base, int64_t elems) const { return reinterpret_cast<const char*>(base) + (size_t)elems * esz(); }
};

#define RUN(expr)                         \
  do {                                    \
    if (!c.dry) B200ST_TRY(expr);         \
  } while (0)

static int need_param(const Ctx& c, const std::string& n) {
  if (!c.info(n)) B200ST_FAIL("parameter '" + n + "' not in this model");
  return 0;
}

struct Scratch;
// final LayerNorm-backward of a block (+ fused production of the next block's dY when the stack loop announced one)
static int block_ln_bwd(Ctx& c, Scratch& sc, const float* dh, const float* x_in, const float* mean, const float* rstd,
                        const std::string& pre, const float* dx_out, float* dx_in, int M, int d);

// ---- dense layers:  weights stored [K_in, N_out] (TF layout) -----------------------------------
// Y[M,N] = epi(X[M,K] W)
static int linear_fwd(Ctx& c, const void* X, int64_t ldx, int M, int K, int N, const std::string& w, const std::string& b,
                      GemmEpilogue epi, void* Y, int ydt, int64_t ldy) {
  B200ST_TRY(need_param(c, w));
  GemmArgs g = gemm_defaults();
  g.M = M; g.N = N; g.K = K;
  g.A = GemmOperand{X, c.adt, 0, ldx, 0, 0};
  g.B = c.W(w, 1, N);
  g.C = Y; g.c_dtype = ydt; g.ldc = ldy;
  g.epi = epi;
  g.epi.bias = b.empty() ? nullptr : c.P(b);
  RUN(gemm(g, c.st));
  return 0;
}
// dX[M,K] = epi(dY[M,N] W^T)
static int linear_dgrad(Ctx& c, const void* dY, int64_t ldy, int M, int N, int K, const std::string& w, GemmEpilogue epi,
                        void* dX, int dxdt, int64_t lddx) {
  B200ST_TRY(need_param(c, w));
  GemmArgs g = gemm_defaults();
  g.M = M; g.N = K; g.K = N;
  g.A = GemmOperand{dY, c.adt, 0, ldy, 0, 0};
  g.B = c.W(w, 0, N);
  g.C = dX; g.c_dtype = dxdt; g.ldc = lddx;
  g.epi = epi;
  RUN(gemm(g, c.st));
  return 0;
}
// dW[K,N] += X^T dY ; db[N] += colsum(dY)
static int linear_wgrad(Ctx& c, const void* X, int64_t ldx, const void* dY, int64_t ldy, int M, int K, int N,
                        const std::string& w, const std::string& b) {
  B200ST_TRY(need_param(c, w));
  GemmArgs g = gemm_defaults();
  g.M = K; g.N = N; g.K = M;
  g.A = GemmOperand{X, c.adt, 1, ldx, 0, 0};
  g.B = GemmOperand{dY, c.adt, 1, ldy, 0, 0};
  g.C = c.G(w); g.c_dtype = F32; g.ldc = N;
  g.epi.accumulate = 1;
  g.splitk = 0;
  if (c.defer_wgrads) {      // inside a backward block: launched together at the end of the block (flush_wgrads)
    c.pending_wgrads.push_back(Ctx::PendingWgrad{g, b.empty() ? nullptr : c.G(b), dY, M, N, ldy});
    return 0;
  }
  cudaStream_t ws = c.wgrad_stream();
  RUN(gemm(g, ws));
  if (!b.empty()) RUN(colsum_accum(dY, c.adt, M, N, ldy, c.G(b), ws));
  c.wgrad_done(ws);
  return 0;
}
// End of a backward block: the block's weight gradients as ONE grouped launch (tc_gemm.cu: tc_wgrad_group_kernel) when they
// qualify, one by one otherwise; the bias gradients behind it.  All their inputs (the block's dY buffers in the current
// scratch parity, saved activations) were produced on `st` before this point and stay untouched until block i+2.
static int flush_wgrads(Ctx& c) {
  if (c.pending_wgrads.empty()) return 0;
  std::vector<Ctx::PendingWgrad> pend;
  pend.swap(c.pending_wgrads);
  cudaStream_t ws = c.wgrad_stream();
  if (!c.dry) {
    GemmArgs gs[4];
    const int n = (int)pend.size();
    int grouped = 2;           // 2 = not grouped: one launch per product
    if (n >= 2 && n <= 4 && is16(c.adt)) {
      for (int i = 0; i < n; ++i) gs[i] = pend[i].g;
      grouped = gemm_wgrad_group(gs, n, ws);
      if (grouped != 0 && grouped != 2) return grouped;
    }
    if (grouped != 0)
      for (const auto& w : pend) B200ST_TRY(gemm(w.g, ws));
    for (const auto& w : pend)
      if (w.db) B200ST_TRY(colsum_accum(w.dY, c.adt, w.M, w.N, w.ldy, w.db, ws));
  }
  c.wgrad_done(ws);
  return 0;
}
struct WgradBlock {          // scope of one backward block: defers linear_wgrad launches until flush()
  Ctx& c;
  explicit WgradBlock(Ctx& cc) : c(cc) { c.defer_wgrads = true; }
  int flush() { c.defer_wgrads = false; return flush_wgrads(c); }
  ~WgradBlock() { c.defer_wgrads = false; }
};

// ---- attention core on projected q/k/v views ----------------------------------------------------
struct View { void* ptr; int64_t ld; };   // [B*T, ld] row-major, heads at column offset h*dh
struct AttnDims { int B, H, Tq, Tk, units; };

static GemmOperand head_op(const Ctx& c, View v, int T, int dh, int mn_major) {
  return GemmOperand{v.ptr, c.adt, mn_major, v.ld, dh, (int64_t)T * v.ld};
}
static int round8(int x) { return (x + 7) / 8 * 8; }

static bool use_fused_attention(const Ctx& c, const AttnDims& a) {
  return is16(c.adt) && a.units / a.H == 64 && !c.m.cfg.disable_fused_attention;
}

static int attention_fwd(Ctx& c, const AttnDims& a, View q, View k, View v, const float* bias, int causal, DropoutSpec drop,
                         float* S, void* p_pre, void* p_drop, void* ctx, float* lse) {
  if (use_fused_attention(c, a)) {
    RUN(attention_fwd_fused(c.adt, q.ptr, q.ld, k.ptr, k.ld, v.ptr, v.ld, a.B, a.H, a.Tq, a.Tk, bias, causal, drop, ctx, a.units, lse, c.st,
                            c.klen_for(bias)));
    return 0;
  }
  const int dh = a.units / a.H, Tkp = round8(a.Tk);
  GemmArgs g = gemm_defaults();
  g.M = a.Tq; g.N = a.Tk; g.K = dh; g.nb1 = a.H; g.nb2 = a.B;
  g.A = head_op(c, q, a.Tq, dh, 0);
  g.B = head_op(c, k, a.Tk, dh, 0);
  g.C = S; g.c_dtype = F32; g.ldc = Tkp; g.c_sb1 = (int64_t)a.Tq * Tkp; g.c_sb2 = (int64_t)a.H * a.Tq * Tkp;
  g.epi.alpha = 1.0f / sqrtf((float)dh);     // q * dh^-0.5 (multi_head_attention.py:203)
  RUN(gemm(g, c.st));
  RUN(softmax_fwd(S, Tkp, bias, causal, p_pre, drop.p > 0.f ? p_drop : nullptr, c.adt, Tkp, a.B, a.H, a.Tq, a.Tk, drop, c.st));
  GemmArgs o = gemm_defaults();
  o.M = a.Tq; o.N = dh; o.K = a.Tk; o.nb1 = a.H; o.nb2 = a.B;
  o.A = GemmOperand{drop.p > 0.f ? p_drop : p_pre, c.adt, 0, Tkp, (int64_t)a.Tq * Tkp, (int64_t)a.H * a.Tq * Tkp};
  o.B = head_op(c, v, a.Tk, dh, 1);
  o.C = ctx; o.c_dtype = c.adt; o.ldc = a.units; o.c_sb1 = dh; o.c_sb2 = (int64_t)a.Tq * a.units;
  RUN(gemm(o, c.st));
  return 0;
}

// dctx (act dtype) [B*Tq, units]  ->  dq, dk, dv views (act dtype)
static int attention_bwd(Ctx& c, const AttnDims& a, View q, View k, View v, const void* p_pre, const void* p_drop,
                         DropoutSpec drop, const void* dctx, float* dP, void* dS, View dq, View dk, View dv, const void* ctx,
                         const float* lse, const float* bias, int causal, float* dq32) {
  if (use_fused_attention(c, a)) {
    RUN(attention_bwd_fused(c.adt, q.ptr, q.ld, k.ptr, k.ld, v.ptr, v.ld, ctx, a.units, dctx, a.units, lse, a.B, a.H, a.Tq, a.Tk, bias, causal,
                            drop, dq32, dq.ptr, dq.ld, dk.ptr, dk.ld, dv.ptr, dv.ld, c.st, c.klen_for(bias)));
    return 0;
  }
  const int dh = a.units / a.H, Tkp = round8(a.Tk);
  const int64_t psb1 = (int64_t)a.Tq * Tkp, psb2 = (int64_t)a.H * a.Tq * Tkp;
  const float alpha = 1.0f / sqrtf((float)dh);
  View dctx_v{const_cast<void*>(dctx), a.units};
  // dP = dctx V^T
  GemmArgs g = gemm_defaults();
  g.M = a.Tq; g.N = a.Tk; g.K = dh; g.nb1 = a.H; g.nb2 = a.B;
  g.A = head_op(c, dctx_v, a.Tq, dh, 0);
  g.B = head_op(c, v, a.Tk, dh, 0);
  g.C = dP; g.c_dtype = F32; g.ldc = Tkp; g.c_sb1 = psb1; g.c_sb2 = psb2;
  RUN(gemm(g, c.st));
  // dV = P_drop^T dctx
  GemmArgs gv = gemm_defaults();
  gv.M = a.Tk; gv.N = dh; gv.K = a.Tq; gv.nb1 = a.H; gv.nb2 = a.B;
  gv.A = GemmOperand{drop.p > 0.f ? p_drop : p_pre, c.adt, 1, Tkp, psb1, psb2};
  gv.B = head_op(c, dctx_v, a.Tq, dh, 1);
  gv.C = dv.ptr; gv.c_dtype = c.adt; gv.ldc = dv.ld; gv.c_sb1 = dh; gv.c_sb2 = (int64_t)a.Tk * dv.ld;
  RUN(gemm(gv, c.st));
  // dS = softmax'(dP)
  RUN(softmax_bwd(dP, Tkp, p_pre, dS, c.adt, Tkp, (int64_t)a.B * a.H * a.Tq, a.Tk, drop, c.st));
  // dQ = alpha dS K
  GemmArgs gq = gemm_defaults();
  gq.M = a.Tq; gq.N = dh; gq.K = a.Tk; gq.nb1 = a.H; gq.nb2 = a.B;
  gq.A = GemmOperand{dS, c.adt, 0, Tkp, psb1, psb2};
  gq.B = head_op(c, k, a.Tk, dh, 1);
  gq.C = dq.ptr; gq.c_dtype = c.adt; gq.ldc = dq.ld; gq.c_sb1 = dh; gq.c_sb2 = (int64_t)a.Tq * dq.ld;
  gq.epi.alpha = alpha;
  RUN(gemm(gq, c.st));
  // dK = alpha dS^T Q
  GemmArgs gk = gemm_defaults();
  gk.M = a.Tk; gk.N = dh; gk.K = a.Tq; gk.nb1 = a.H; gk.nb2 = a.B;
  gk.A = GemmOperand{dS, c.adt, 1, Tkp, psb1, psb2};
  gk.B = head_op(c, q, a.Tq, dh, 1);
  gk.C = dk.ptr; gk.c_dtype = c.adt; gk.ldc = dk.ld; gk.c_sb1 = dh; gk.c_sb2 = (int64_t)a.Tk * dk.ld;
  gk.epi.alpha = alpha;
  RUN(gemm(gk, c.st));
  return 0;
}

// ---- saved activations ---------------------------------------------------------------------------
struct AttnSave {
  const float* x_in = nullptr;
  void* h = nullptr; float* mean = nullptr; float* rstd = nullptr;
  void* qkv = nullptr;      // self: [M,3u]; cross: q [M,u]
  void* kv = nullptr;       // cross: [Mk,2u]
  void* p_pre = nullptr; void* p_drop = nullptr; void* ctx = nullptr;
  float* lse = nullptr;     // fused attention: per-row log-sum-exp [B,H,Tq]
  const void* mem = nullptr; // cross: memory in act dtype [Mk, d]
  const float* bias = nullptr; int causal = 0;
  AttnDims dims{};
  uint64_t s_attn = 0, s_post = 0;
};
struct FfnSave {
  const float* x_in = nullptr;
  void* h = nullptr; float* mean = nullptr; float* rstd = nullptr;
  void* f1 = nullptr;
  int M = 0;
  uint64_t s_ffn = 0, s_post = 0;
};

struct Scratch {   // shared transient buffers (sized for the largest sublayer)
  float* S = nullptr;       // [B,H,Tq,Tkp] fp32 logits / dP
  void* dS = nullptr;
  // gradient operands of the weight-gradient GEMMs: double-buffered by backward-block parity (side-stream readers)
  void* dY2[2] = {nullptr, nullptr};       // [M,d]
  void* dqkv2[2] = {nullptr, nullptr};     // [M,3d]
  void* dkv2[2] = {nullptr, nullptr};      // [Mk,2d]
  void* dF12[2] = {nullptr, nullptr};      // [M,ffn]
  void* dY = nullptr; void* dqkv = nullptr; void* dkv = nullptr; void* dF1 = nullptr;   // current block's buffers
  void select(int par) { dY = dY2[par]; dqkv = dqkv2[par]; dkv = dkv2[par]; dF1 = dF12[par]; }
  void* dctx = nullptr;     // [M,d]
  float* dh = nullptr;      // [M,d] fp32
  float* dq32 = nullptr;    // [M,d] fp32 (fused attention: dQ reduction across kv blocks)
};

static int block_ln_bwd(Ctx& c, Scratch& sc, const float* dh, const float* x_in, const float* mean, const float* rstd,
                        const std::string& pre, const float* dx_out, float* dx_in, int M, int d) {
  void* dnext = nullptr;
  DropoutSpec nd = no_dropout();
  if (c.next_drop) {
    dnext = sc.dY2[c.next_parity_ready()];
    nd = *c.next_drop;
    c.next_drop = nullptr;
    c.dy_ready = true;
  }
  RUN(layernorm_bwd_next(dh, F32, x_in, F32, mean, rstd, c.P(pre + ".ln.gamma"), c.P(pre + ".ln.beta"), dx_out, dx_in, F32,
                         c.G(pre + ".ln.gamma"), c.G(pre + ".ln.beta"), M, d, 0, dnext, c.adt, nd, c.st));
  return 0;
}

// x_out = x_in + dropout(Attn(LN(x_in)))  — pre-norm block (common_layers.py:73-85)
static int self_attn_block_fwd(Ctx& c, const std::string& pre, const float* x_in, float* x_out, int B, int T, const float* bias,
                               int causal, Scratch& sc, AttnSave& sv) {
  const Config& cf = c.m.cfg;
  const int d = cf.d, M = B * T, Tkp = round8(T);
  sv.x_in = x_in;
  sv.dims = AttnDims{B, cf.heads, T, T, d};
  sv.bias = bias; sv.causal = causal;
  sv.s_attn = dropout_stream_id(pre + ".attn_drop"); sv.s_post = dropout_stream_id(pre + ".post_drop");
  sv.h = c.act((int64_t)M * d); sv.mean = c.f32(M); sv.rstd = c.f32(M);
  sv.qkv = c.act((int64_t)M * 3 * d);
  const DropoutSpec adrop = c.drop(cf.attention_dropout, sv.s_attn, (int64_t)B * cf.heads * T * Tkp);
  if (use_fused_attention(c, sv.dims)) {
    sv.lse = c.f32((int64_t)B * cf.heads * T);
  } else {
    sv.p_pre = c.act((int64_t)B * cf.heads * T * Tkp);
    sv.p_drop = adrop.p > 0.f ? c.act((int64_t)B * cf.heads * T * Tkp) : nullptr;
  }
  sv.ctx = c.act((int64_t)M * d);
  RUN(layernorm_fwd(x_in, F32, c.P(pre + ".ln.gamma"), c.P(pre + ".ln.beta"), cf.ln_eps, sv.h, c.adt, nullptr, sv.mean, sv.rstd,
                    M, d, 0, c.st));
  GemmEpilogue e0 = gemm_defaults().epi;
  B200ST_TRY(linear_fwd(c, sv.h, d, M, d, 3 * d, pre + ".qkv.kernel", pre + ".qkv.bias", e0, sv.qkv, c.adt, 3 * d));
  View q{sv.qkv, 3 * d}, k{c.act_off(sv.qkv, d), 3 * d}, v{c.act_off(sv.qkv, 2 * d), 3 * d};
  B200ST_TRY(attention_fwd(c, sv.dims, q, k, v, bias, causal, adrop, sc.S, sv.p_pre, sv.p_drop, sv.ctx, sv.lse));
  GemmEpilogue e1 = gemm_defaults().epi;
  e1.drop = c.drop(cf.postprocess_dropout, sv.s_post, (int64_t)M * d);
  e1.residual = x_in; e1.res_ld = d;
  B200ST_TRY(linear_fwd(c, sv.ctx, d, M, d, d, pre + ".out.kernel", pre + ".out.bias", e1, x_out, F32, d));
  return 0;
}

static int self_attn_block_bwd(Ctx& c, const std::string& pre, const float* dx_out, float* dx_in, Scratch& sc, const AttnSave& sv) {
  sc.select(c.begin_bwd_block());
  WgradBlock wb(c);
  const Config& cf = c.m.cfg;
  const int d = cf.d, M = sv.dims.B * sv.dims.Tq;
  if (c.dy_ready) c.dy_ready = false;      // produced by the previous block's LayerNorm-backward
  else RUN(cast_dropout(dx_out, sc.dY, c.adt, (int64_t)M * d, c.drop(cf.postprocess_dropout, sv.s_post), c.st));
  B200ST_TRY(linear_wgrad(c, sv.ctx, d, sc.dY, d, M, d, d, pre + ".out.kernel", pre + ".out.bias"));
  GemmEpilogue e0 = gemm_defaults().epi;
  B200ST_TRY(linear_dgrad(c, sc.dY, d, M, d, d, pre + ".out.kernel", e0, sc.dctx, c.adt, d));
  View q{sv.qkv, 3 * d}, k{c.act_off(sv.qkv, d), 3 * d}, v{c.act_off(sv.qkv, 2 * d), 3 * d};
  View dq{sc.dqkv, 3 * d}, dk{c.act_off(sc.dqkv, d), 3 * d}, dv{c.act_off(sc.dqkv, 2 * d), 3 * d};
  B200ST_TRY(attention_bwd(c, sv.dims, q, k, v, sv.p_pre, sv.p_drop, c.drop(cf.attention_dropout, sv.s_attn), sc.dctx, sc.S, sc.dS,
                           dq, dk, dv, sv.ctx, sv.lse, sv.bias, sv.causal, sc.dq32));
  B200ST_TRY(linear_wgrad(c, sv.h, d, sc.dqkv, 3 * d, M, d, 3 * d, pre + ".qkv.kernel", pre + ".qkv.bias"));
  B200ST_TRY(wb.flush());      // every dY of the block exists: the side stream starts under the rest of the chain
  B200ST_TRY(linear_dgrad(c, sc.dqkv, 3 * d, M, 3 * d, d, pre + ".qkv.kernel", e0, sc.dh, F32, d));
  B200ST_TRY(block_ln_bwd(c, sc, sc.dh, sv.x_in, sv.mean, sv.rstd, pre, dx_out, dx_in, M, d));
  return wb.flush();
}

// cross attention: q from LN(x), k/v from memory (act dtype, [B*Tm, d]); memory_bias [B,Tm]
static int cross_attn_block_fwd(Ctx& c, const std::string& pre, const float* x_in, float* x_out, int B, int L, const void* mem,
                                int Tm, const float* mem_bias, Scratch& sc, AttnSave& sv) {
  const Config& cf = c.m.cfg;
  const int d = cf.d, M = B * L, Mk = B * Tm, Tkp = round8(Tm);
  sv.x_in = x_in; sv.mem = mem;
  sv.dims = AttnDims{B, cf.heads, L, Tm, d};
  sv.bias = mem_bias; sv.causal = 0;
  sv.s_attn = dropout_stream_id(pre + ".attn_drop"); sv.s_post = dropout_stream_id(pre + ".post_drop");
  sv.h = c.act((int64_t)M * d); sv.mean = c.f32(M); sv.rstd = c.f32(M);
  sv.qkv = c.act((int64_t)M * d);
  sv.kv = c.act((int64_t)Mk * 2 * d);
  const DropoutSpec adrop = c.drop(cf.attention_dropout, sv.s_attn, (int64_t)B * cf.heads * L * Tkp);
  if (use_fused_attention(c, sv.dims)) {
    sv.lse = c.f32((int64_t)B * cf.heads * L);
  } else {
    sv.p_pre = c.act((int64_t)B * cf.heads * L * Tkp);
    sv.p_drop = adrop.p > 0.f ? c.act((int64_t)B * cf.heads * L * Tkp) : nullptr;
  }
  sv.ctx = c.act((int64_t)M * d);
  RUN(layernorm_fwd(x_in, F32, c.P(pre + ".ln.gamma"), c.P(pre + ".ln.beta"), cf.ln_eps, sv.h, c.adt, nullptr, sv.mean, sv.rstd,
                    M, d, 0, c.st));
  GemmEpilogue e0 = gemm_defaults().epi;
  B200ST_TRY(linear_fwd(c, sv.h, d, M, d, d, pre + ".q.kernel", pre + ".q.bias", e0, sv.qkv, c.adt, d));
  B200ST_TRY(linear_fwd(c, mem, d, Mk, d, 2 * d, pre + ".kv.kernel", pre + ".kv.bias", e0, sv.kv, c.adt, 2 * d));
  View q{sv.qkv, d}, k{sv.kv, 2 * d}, v{c.act_off(sv.kv, d), 2 * d};
  B200ST_TRY(attention_fwd(c, sv.dims, q, k, v, mem_bias, 0, adrop, sc.S, sv.p_pre, sv.p_drop, sv.ctx, sv.lse));
  GemmEpilogue e1 = gemm_defaults().epi;
  e1.drop = c.drop(cf.postprocess_dropout, sv.s_post, (int64_t)M * d);
  e1.residual = x_in; e1.res_ld = d;
  B200ST_TRY(linear_fwd(c, sv.ctx, d, M, d, d, pre + ".out.kernel", pre + ".out.bias", e1, x_out, F32, d));
  return 0;
}

static int cross_attn_block_bwd(Ctx& c, const std::string& pre, const float* dx_out, float* dx_in, float* dmem, Scratch& sc,
                                const AttnSave& sv) {
  sc.select(c.begin_bwd_block());
  WgradBlock wb(c);
  const Config& cf = c.m.cfg;
  const int d = cf.d, M = sv.dims.B * sv.dims.Tq, Mk = sv.dims.B * sv.dims.Tk;
  if (c.dy_ready) c.dy_ready = false;      // produced by the previous block's LayerNorm-backward
  else RUN(cast_dropout(dx_out, sc.dY, c.adt, (int64_t)M * d, c.drop(cf.postprocess_dropout, sv.s_post), c.st));
  B200ST_TRY(linear_wgrad(c, sv.ctx, d, sc.dY, d, M, d, d, pre + ".out.kernel", pre + ".out.bias"));
  GemmEpilogue e0 = gemm_defaults().epi;
  B200ST_TRY(linear_dgrad(c, sc.dY, d, M, d, d, pre + ".out.kernel", e0, sc.dctx, c.adt, d));
  View q{sv.qkv, d}, k{sv.kv, 2 * d}, v{c.act_off(sv.kv, d), 2 * d};
  View dq{sc.dqkv, d}, dk{sc.dkv, 2 * d}, dv{c.act_off(sc.dkv, d), 2 * d};
  B200ST_TRY(attention_bwd(c, sv.dims, q, k, v, sv.p_pre, sv.p_drop, c.drop(cf.attention_dropout, sv.s_attn), sc.dctx, sc.S, sc.dS,
                           dq, dk, dv, sv.ctx, sv.lse, sv.bias, 0, sc.dq32));
  B200ST_TRY(linear_wgrad(c, sv.h, d, sc.dqkv, d, M, d, d, pre + ".q.kernel", pre + ".q.bias"));
  B200ST_TRY(linear_wgrad(c, sv.mem, d, sc.dkv, 2 * d, Mk, d, 2 * d, pre + ".kv.kernel", pre + ".kv.bias"));
  B200ST_TRY(wb.flush());
  B200ST_TRY(linear_dgrad(c, sc.dqkv, d, M, d, d, pre + ".q.kernel", e0, sc.dh, F32, d));
  B200ST_TRY(block_ln_bwd(c, sc, sc.dh, sv.x_in, sv.mean, sv.rstd, pre, dx_out, dx_in, M, d));
  GemmEpilogue ea = gemm_defaults().epi;
  ea.accumulate = 1;                              // memory gradient accumulates over decoder layers
  B200ST_TRY(linear_dgrad(c, sc.dkv, 2 * d, Mk, 2 * d, d, pre + ".kv.kernel", ea, dmem, F32, d));
  return wb.flush();
}

// x_out = x_in + dropout(W2 dropout(relu(W1 LN(x_in)))) (common_layers.py:145-160)
static int ffn_block_fwd(Ctx& c, const std::string& pre, const float* x_in, float* x_out, int M, FfnSave& sv) {
  const Config& cf = c.m.cfg;
  const int d = cf.d, f = cf.ffn;
  sv.x_in = x_in; sv.M = M;
  sv.s_ffn = dropout_stream_id(pre + ".ffn_drop"); sv.s_post = dropout_stream_id(pre + ".post_drop");
  sv.h = c.act((int64_t)M * d); sv.mean = c.f32(M); sv.rstd = c.f32(M);
  sv.f1 = c.act((int64_t)M * f);
  if (fused_mlp_supported(M, d, f, c.adt) && !c.m.cfg.disable_fused_attention) {
    // one kernel for FFN1 -> ReLU -> dropout -> FFN2 -> dropout -> +residual (SURVEY K11): the LayerNorm kernel also seeds
    // x_out with the residual, the fused kernel reduce-adds the rest
    B200ST_TRY(need_param(c, pre + ".w1")); B200ST_TRY(need_param(c, pre + ".w2"));
    RUN(layernorm_fwd_copy(x_in, F32, c.P(pre + ".ln.gamma"), c.P(pre + ".ln.beta"), cf.ln_eps, sv.h, c.adt, nullptr, sv.mean, sv.rstd,
                           M, d, 0, x_out, c.st));
    const DropoutSpec d1 = c.drop(cf.ffn_dropout, sv.s_ffn, (int64_t)M * f);
    const DropoutSpec d2 = c.drop(cf.postprocess_dropout, sv.s_post, (int64_t)M * d);
    int* tk = c.mlp_tickets(M);
    RUN(fused_mlp_fwd(sv.h, c.adt, M, d, f, c.W(pre + ".w1", 1, f).ptr, c.P(pre + ".b1"), c.W(pre + ".w2", 1, d).ptr, c.P(pre + ".b2"),
                      d1, d2, sv.f1, x_out, c.st, tk));
    return 0;
  }
  RUN(layernorm_fwd(x_in, F32, c.P(pre + ".ln.gamma"), c.P(pre + ".ln.beta"), cf.ln_eps, sv.h, c.adt, nullptr, sv.mean, sv.rstd,
                    M, d, 0, c.st));
  GemmEpilogue e1 = gemm_defaults().epi;
  e1.relu = 1;
  e1.drop = c.drop(cf.ffn_dropout, sv.s_ffn, (int64_t)M * f);
  B200ST_TRY(linear_fwd(c, sv.h, d, M, d, f, pre + ".w1", pre + ".b1", e1, sv.f1, c.adt, f));
  GemmEpilogue e2 = gemm_defaults().epi;
  e2.drop = c.drop(cf.postprocess_dropout, sv.s_post, (int64_t)M * d);
  e2.residual = x_in; e2.res_ld = d;
  B200ST_TRY(linear_fwd(c, sv.f1, f, M, f, d, pre + ".w2", pre + ".b2", e2, x_out, F32, d));
  return 0;
}

static int ffn_block_bwd(Ctx& c, const std::string& pre, const float* dx_out, float* dx_in, Scratch& sc, const FfnSave& sv) {
  sc.select(c.begin_bwd_block());
  WgradBlock wb(c);
  const Config& cf = c.m.cfg;
  const int d = cf.d, f = cf.ffn, M = sv.M;
  if (c.dy_ready) c.dy_ready = false;      // produced by the previous block's LayerNorm-backward
  else RUN(cast_dropout(dx_out, sc.dY, c.adt, (int64_t)M * d, c.drop(cf.postprocess_dropout, sv.s_post), c.st));
  B200ST_TRY(linear_wgrad(c, sv.f1, f, sc.dY, d, M, f, d, pre + ".w2", pre + ".b2"));
  if (fused_mlp_supported(M, d, f, c.adt) && !c.m.cfg.disable_fused_attention) {
    // data-gradient chain in one kernel: dF1 = (dY W2^T) * relu'/dropout' (written for the W1 weight gradient), dh = dF1 W1^T
    const DropoutSpec fd = c.drop(cf.ffn_dropout, sv.s_ffn);
    RUN(cudaMemsetAsync(sc.dh, 0, sizeof(float) * (size_t)M * d, c.st) == cudaSuccess ? 0 : 1);
    int* tk = c.mlp_tickets(M);
    RUN(fused_mlp_bwd(sc.dY, c.adt, M, d, f, c.W(pre + ".w1", 0, f).ptr, c.W(pre + ".w2", 0, d).ptr, sv.f1,
                      fd.p > 0.f ? fd.scale : 1.f, sc.dF1, sc.dh, c.st, tk));
    B200ST_TRY(linear_wgrad(c, sv.h, d, sc.dF1, f, M, d, f, pre + ".w1", pre + ".b1"));
    B200ST_TRY(wb.flush());
    B200ST_TRY(block_ln_bwd(c, sc, sc.dh, sv.x_in, sv.mean, sv.rstd, pre, dx_out, dx_in, M, d));
    return wb.flush();
  }
  GemmEpilogue e1 = gemm_defaults().epi;
  e1.mask_src = sv.f1; e1.mask_dtype = c.adt; e1.mask_ld = f;      // relu' and ffn-dropout mask: stored f1 > 0
  const DropoutSpec fd = c.drop(cf.ffn_dropout, sv.s_ffn);
  e1.alpha = fd.p > 0.f ? fd.scale : 1.f;
  B200ST_TRY(linear_dgrad(c, sc.dY, d, M, d, f, pre + ".w2", e1, sc.dF1, c.adt, f));
  B200ST_TRY(linear_wgrad(c, sv.h, d, sc.dF1, f, M, d, f, pre + ".w1", pre + ".b1"));
  GemmEpilogue e0 = gemm_defaults().epi;
  B200ST_TRY(linear_dgrad(c, sc.dF1, f, M, f, d, pre + ".w1", e0, sc.dh, F32, d));
  B200ST_TRY(block_ln_bwd(c, sc, sc.dh, sv.x_in, sv.mean, sv.rstd, pre, dx_out, dx_in, M, d));
  return wb.flush();
}

// ---- stacks ----------------------------------------------------------------------------------------
struct EncoderSave {
  std::vector<AttnSave> att; std::vector<FfnSave> ffn;
  const float* x_last = nullptr; float* mean = nullptr; float* rstd = nullptr;
  void* out = nullptr;       // act dtype [M,d]
  int B = 0, T = 0;
};

static void alloc_scratch(Ctx& c, Scratch& sc, int B, int Tq_max, int Tk_max, int Mq_max, int Mk_max, bool backward) {
  const Config& cf = c.m.cfg;
  const int64_t pl = (int64_t)B * cf.heads * Tq_max * round8(Tk_max);
  sc.S = c.f32(pl);
  if (backward) {
    sc.dS = c.act(pl);
    for (int par = 0; par < 2; ++par) {
      sc.dY2[par] = c.act((int64_t)Mq_max * cf.d);
      sc.dqkv2[par] = c.act((int64_t)Mq_max * 3 * cf.d);
      sc.dkv2[par] = c.act((int64_t)Mk_max * 2 * cf.d);
      sc.dF12[par] = c.act((int64_t)Mq_max * cf.ffn);
    }
    sc.select(0);
    sc.dctx = c.act((int64_t)Mq_max * cf.d);
    sc.dh = c.f32((int64_t)Mq_max * cf.d);
    sc.dq32 = c.f32((int64_t)Mq_max * (cf.d + cf.heads));   // + rowsum(dO * O) per (row, head)
  }
}

// x0: embedded input fp32 [B*T,d] (dropout already applied); bias [B,T]; out: act-dtype (+ optional fp32 copy)
static int encoder_fwd(Ctx& c, const float* x0, const float* bias, int B, int T, Scratch& sc, EncoderSave& sv, float* out32) {
  const Config& cf = c.m.cfg;
  const int M = B * T, d = cf.d;
  sv.B = B; sv.T = T;
  sv.att.resize(cf.enc_layers); sv.ffn.resize(cf.enc_layers);
  const float* x = x0;
  for (int i = 0; i < cf.enc_layers; ++i) {
    const std::string p = "enc." + std::to_string(i);
    float* x1 = c.f32((int64_t)M * d);
    B200ST_TRY(self_attn_block_fwd(c, p + ".att", x, x1, B, T, bias, 0, sc, sv.att[i]));
    float* x2 = c.f32((int64_t)M * d);
    B200ST_TRY(ffn_block_fwd(c, p + ".ffn", x1, x2, M, sv.ffn[i]));
    x = x2;
  }
  sv.x_last = x;
  sv.mean = c.f32(M); sv.rstd = c.f32(M);
  sv.out = c.act((int64_t)M * d);
  RUN(layernorm_fwd(x, F32, c.P("enc.out_ln.gamma"), c.P("enc.out_ln.beta"), cf.ln_eps, sv.out, c.adt, out32, sv.mean, sv.rstd, M, d, 0,
                    c.st));
  return 0;
}

// d_out: fp32 [M,d] gradient wrt encoder output; returns gradient wrt x0 in dx (fp32 [M,d])
static int encoder_bwd(Ctx& c, const float* d_out, float* dx, float* dx_tmp, Scratch& sc, const EncoderSave& sv, bool buckets = false) {
  const Config& cf = c.m.cfg;
  const int M = sv.B * sv.T, d = cf.d;
  RUN(layernorm_bwd(d_out, F32, sv.x_last, F32, sv.mean, sv.rstd, c.P("enc.out_ln.gamma"), c.P("enc.out_ln.beta"), nullptr, dx, F32,
                    c.G("enc.out_ln.gamma"), c.G("enc.out_ln.beta"), M, d, 0, c.st));
  for (int i = cf.enc_layers - 1; i >= 0; --i) {
    const std::string p = "enc." + std::to_string(i);
    // each block's LayerNorm-backward also emits the next block's dY = cast(dropout'(dx)) (same M for the whole stack)
    const DropoutSpec nd_att = c.drop(cf.postprocess_dropout, sv.att[i].s_post);
    c.next_drop = &nd_att;
    B200ST_TRY(ffn_block_bwd(c, p + ".ffn", dx, dx_tmp, sc, sv.ffn[i]));
    DropoutSpec nd_ffn = no_dropout();
    if (i > 0) { nd_ffn = c.drop(cf.postprocess_dropout, sv.ffn[i - 1].s_post); c.next_drop = &nd_ffn; }
    B200ST_TRY(self_attn_block_bwd(c, p + ".att", dx_tmp, dx, sc, sv.att[i]));
    // gradient bucket: the upper half of the encoder stack (+ its final LayerNorm) is final after layer enc_layers / 2
    if (buckets && i == cf.enc_layers / 2 && i > 0) B200ST_TRY(c.reduce_down_to(p + ".att.ln.gamma"));
  }
  return 0;
}

struct DecoderSave {
  std::vector<AttnSave> self, cross; std::vector<FfnSave> ffn;
  const float* x_last = nullptr; float* mean = nullptr; float* rstd = nullptr;
  void* out = nullptr;
  int B = 0, L = 0, Tm = 0;
};

static int decoder_fwd(Ctx& c, const float* x0, int B, int L, const void* mem, int Tm, const float* mem_bias, Scratch& sc,
                       DecoderSave& sv, float* out32) {
  const Config& cf = c.m.cfg;
  const int M = B * L, d = cf.d;
  sv.B = B; sv.L = L; sv.Tm = Tm;
  sv.self.resize(cf.dec_layers); sv.cross.resize(cf.dec_layers); sv.ffn.resize(cf.dec_layers);
  const float* x = x0;
  for (int i = 0; i < cf.dec_layers; ++i) {
    const std::string p = "dec." + std::to_string(i);
    float* x1 = c.f32((int64_t)M * d);
    B200ST_TRY(self_attn_block_fwd(c, p + ".self", x, x1, B, L, nullptr, 1, sc, sv.self[i]));
    x = x1;
    if (cf.with_cross_attention && mem) {
      float* x2 = c.f32((int64_t)M * d);
      B200ST_TRY(cross_attn_block_fwd(c, p + ".cross", x, x2, B, L, mem, Tm, mem_bias, sc, sv.cross[i]));
      x = x2;
    }
    float* x3 = c.f32((int64_t)M * d);
    B200ST_TRY(ffn_block_fwd(c, p + ".ffn", x, x3, M, sv.ffn[i]));
    x = x3;
  }
  sv.x_last = x;
  sv.mean = c.f32(M); sv.rstd = c.f32(M);
  sv.out = c.act((int64_t)M * d);
  RUN(layernorm_fwd(x, F32, c.P("dec.out_ln.gamma"), c.P("dec.out_ln.beta"), cf.ln_eps, sv.out, c.adt, out32, sv.mean, sv.rstd, M, d, 0,
                    c.st));
  return 0;
}

static int decoder_bwd(Ctx& c, const float* d_out, float* dx, float* dx_tmp, float* dmem, bool has_mem, Scratch& sc,
                       const DecoderSave& sv) {
  const Config& cf = c.m.cfg;
  const int M = sv.B * sv.L, d = cf.d;
  RUN(layernorm_bwd(d_out, F32, sv.x_last, F32, sv.mean, sv.rstd, c.P("dec.out_ln.gamma"), c.P("dec.out_ln.beta"), nullptr, dx, F32,
                    c.G("dec.out_ln.gamma"), c.G("dec.out_ln.beta"), M, d, 0, c.st));
  float* a = dx; float* b = dx_tmp;
  for (int i = cf.dec_layers - 1; i >= 0; --i) {
    const std::string p = "dec." + std::to_string(i);
    const bool cross = cf.with_cross_attention && has_mem;
    const DropoutSpec nd1 = c.drop(cf.postprocess_dropout, cross ? sv.cross[i].s_post : sv.self[i].s_post);
    c.next_drop = &nd1;
    B200ST_TRY(ffn_block_bwd(c, p + ".ffn", a, b, sc, sv.ffn[i]));
    std::swap(a, b);
    if (cross) {
      const DropoutSpec nd2 = c.drop(cf.postprocess_dropout, sv.self[i].s_post);
      c.next_drop = &nd2;
      B200ST_TRY(cross_attn_block_bwd(c, p + ".cross", a, b, dmem, sc, sv.cross[i]));
      std::swap(a, b);
    }
    DropoutSpec nd3 = no_dropout();
    if (i > 0) { nd3 = c.drop(cf.postprocess_dropout, sv.ffn[i - 1].s_post); c.next_drop = &nd3; }
    B200ST_TRY(self_attn_block_bwd(c, p + ".self", a, b, sc, sv.self[i]));
    std::swap(a, b);
  }
  if (a != dx) RUN(cudaMemcpyAsync(dx, a, sizeof(float) * (size_t)M * d, cudaMemcpyDeviceToDevice, c.st) == cudaSuccess ? 0 : 1);
  return 0;
}

// ---- speech front-end ------------------------------------------------------------------------------
struct FrontSave {
  void* y1 = nullptr; void* col = nullptr; void* z2 = nullptr; void* y2 = nullptr;
  float* mean2 = nullptr; float* rstd2 = nullptr;
  float* rstd1 = nullptr;    // normalised-save mode: y1 holds xhat of conv1's LayerNorm, rstd1 its 1/sigma
  int B = 0, T = 0, T1 = 0, F1 = 0, T2 = 0, F2 = 0;
  uint64_t s_in = 0;
};

// conv1's LayerNorm output is saved normalised (xhat + 1/sigma) instead of post-ReLU when the fast kernels apply
static bool front_saves_xhat(const Config& cf) { return cf.conv_layer_norm && cf.channels == 256 && cf.in_channels == 1; }

// src fp32 [B,T,F,Cin] -> x0 fp32 [B*T2, d] = dropout((dense(flatten(conv stack))) * sqrt(d) + pos)
static int speech_front_fwd(Ctx& c, const float* src, int B, int T, float* x0, FrontSave& sv) {
  const Config& cf = c.m.cfg;
  const int F = cf.feat, C = cf.channels, d = cf.d;
  const int T1 = (T + 1) / 2, F1 = (F + 1) / 2, T2 = (T1 + 1) / 2, F2 = (F1 + 1) / 2;
  sv.B = B; sv.T = T; sv.T1 = T1; sv.F1 = F1; sv.T2 = T2; sv.F2 = F2;
  sv.s_in = dropout_stream_id("enc.in_drop");
  const int64_t R1 = (int64_t)B * T1 * F1, R2 = (int64_t)B * T2 * F2;
  sv.y1 = c.act(R1 * C);
  sv.col = c.act(R2 * 9 * C);
  sv.z2 = c.act(R2 * C);
  sv.y2 = c.act(R2 * C);
  sv.mean2 = c.f32(R2); sv.rstd2 = c.f32(R2);
  float* e0 = c.f32((int64_t)B * T2 * d);
  if (front_saves_xhat(cf)) {
    sv.rstd1 = c.f32(R1);
    RUN(conv1_norm_fwd(src, c.P("src.conv1.kernel"), c.P("src.conv1.bias"), 1e-6f, sv.y1, c.adt, sv.rstd1, B, T, F, cf.in_channels, C,
                       c.st));
    RUN(im2col_3x3s2_affine(sv.y1, sv.col, c.adt, B, T1, F1, C, c.W("src.ln1.gamma", 0, C).ptr, c.W("src.ln1.beta", 0, C).ptr, c.st));
  } else {
    RUN(conv1_ln_relu_fwd(src, c.P("src.conv1.kernel"), c.P("src.conv1.bias"), c.P("src.ln1.gamma"), c.P("src.ln1.beta"), 1e-6f,
                          sv.y1, c.adt, B, T, F, cf.in_channels, C, cf.conv_layer_norm, c.st));
    RUN(im2col_3x3s2(sv.y1, sv.col, c.adt, B, T1, F1, C, c.st));
  }
  GemmEpilogue ez = gemm_defaults().epi;
  if (cf.conv_layer_norm) {
    B200ST_TRY(linear_fwd(c, sv.col, 9 * C, (int)R2, 9 * C, C, "src.conv2.kernel", "src.conv2.bias", ez, sv.z2, c.adt, C));
    RUN(layernorm_fwd(sv.z2, c.adt, c.P("src.ln2.gamma"), c.P("src.ln2.beta"), 1e-6f, sv.y2, c.adt, nullptr, sv.mean2, sv.rstd2, R2, C,
                      1, c.st));
  } else {
    ez.relu = 1;
    B200ST_TRY(linear_fwd(c, sv.col, 9 * C, (int)R2, 9 * C, C, "src.conv2.kernel", "src.conv2.bias", ez, sv.y2, c.adt, C));
  }
  GemmEpilogue ed = gemm_defaults().epi;
  B200ST_TRY(linear_fwd(c, sv.y2, (int64_t)F2 * C, B * T2, F2 * C, d, "src.dense.kernel", "src.dense.bias", ed, e0, F32, d));
  const DropoutSpec in_drop = c.drop(cf.postprocess_dropout, sv.s_in, (int64_t)B * T2 * d);   // outside RUN: allocates in the planning pass too
  RUN(posenc_fwd(e0, x0, B, T2, d, sqrtf((float)d), 0, in_drop, c.st));
  return 0;
}

static int speech_front_bwd(Ctx& c, const float* src, const float* dx0, const FrontSave& sv) {
  const Config& cf = c.m.cfg;
  const int F = cf.feat, C = cf.channels, d = cf.d, B = sv.B;
  const int64_t R1 = (int64_t)B * sv.T1 * sv.F1, R2 = (int64_t)B * sv.T2 * sv.F2;
  const int Mx = B * sv.T2;
  void* de0 = c.act((int64_t)Mx * d);
  void* dy2 = c.act(R2 * C);
  void* dz2 = c.act(R2 * C);
  // conv2's data gradient: implicit GEMMs straight from dz2 into class-major tiles (no [rows, 9C] column gradient), or the
  // explicit dcol = dz2 W^T + gather in conv1's backward
  const bool implicit_dgrad = front_saves_xhat(cf) && is16(c.adt) && C == 256 && sv.F2 <= 128;
  void* dcol = c.act(implicit_dgrad ? conv2_dgrad_implicit_elems(B, sv.T2, sv.F2, C) : R2 * 9 * C);
  void* dz1 = c.act(R1 * C);
  const int K1p = (9 * cf.in_channels + 7) / 8 * 8;
  void* col1 = c.act(R1 * K1p);
  RUN(posenc_bwd(dx0, de0, c.adt, (int64_t)Mx * d, sqrtf((float)d), c.drop(cf.postprocess_dropout, sv.s_in), c.st));
  B200ST_TRY(linear_wgrad(c, sv.y2, (int64_t)sv.F2 * C, de0, d, Mx, sv.F2 * C, d, "src.dense.kernel", "src.dense.bias"));
  GemmEpilogue e0 = gemm_defaults().epi;
  B200ST_TRY(linear_dgrad(c, de0, d, Mx, d, sv.F2 * C, "src.dense.kernel", e0, dy2, c.adt, (int64_t)sv.F2 * C));
  if (cf.conv_layer_norm) {
    RUN(layernorm_bwd(dy2, c.adt, sv.z2, c.adt, sv.mean2, sv.rstd2, c.P("src.ln2.gamma"), c.P("src.ln2.beta"), nullptr, dz2, c.adt,
                      c.G("src.ln2.gamma"), c.G("src.ln2.beta"), R2, C, 1, c.st));
  } else {
    B200ST_FAIL("training without conv layer norm is not implemented");
  }
  B200ST_TRY(linear_wgrad(c, sv.col, 9 * C, dz2, C, (int)R2, 9 * C, C, "src.conv2.kernel", "src.conv2.bias"));
  if (implicit_dgrad) RUN(conv2_dgrad_implicit(dz2, c.W("src.conv2.kernel", 0, C).ptr, dcol, c.adt, B, sv.T2, sv.F2, C, c.st));
  else B200ST_TRY(linear_dgrad(c, dz2, C, (int)R2, C, 9 * C, "src.conv2.kernel", e0, dcol, c.adt, 9 * C));
  // fused: col2im gather + ReLU' + LN' -> dz1, fbank im2col rows, db/dgamma/dbeta (xhat read back, or z1 recomputed)
  if (front_saves_xhat(cf)) {
    RUN(conv1_bwd_from_xhat(src, c.W("src.ln1.gamma", 0, C).ptr, c.W("src.ln1.beta", 0, C).ptr, sv.y1, sv.rstd1, dcol, c.adt, dz1, col1, K1p,
                            c.G("src.conv1.bias"), c.G("src.ln1.gamma"), c.G("src.ln1.beta"), B, sv.T, F, C, c.st, implicit_dgrad ? 1 : 0));
  } else {
    RUN(conv1_bwd_fused(src, c.P("src.conv1.kernel"), c.P("src.conv1.bias"), c.P("src.ln1.gamma"), c.P("src.ln1.beta"), 1e-6f, sv.y1,
                        dcol, c.adt, dz1, col1, K1p, c.G("src.conv1.bias"), c.G("src.ln1.gamma"), c.G("src.ln1.beta"), B, sv.T, F,
                        cf.in_channels, C, cf.conv_layer_norm, c.st));
  }
  {
    // dW1[9*Cin, C] += col1^T dz1   (split-K tcgen05 GEMM over all B*T1*F1 positions)
    GemmArgs g = gemm_defaults();
    g.M = 9 * cf.in_channels; g.N = C; g.K = (int)R1;
    g.A = GemmOperand{col1, c.adt, 1, K1p, 0, 0};
    g.B = GemmOperand{dz1, c.adt, 1, C, 0, 0};
    g.C = c.G("src.conv1.kernel"); g.c_dtype = F32; g.ldc = C;
    g.epi.accumulate = 1; g.splitk = 0;
    RUN(gemm(g, c.st));
  }
  return 0;
}

static int model_run(Ctx& c, const Batch& b, bool backward) {
  const Config& cf = c.m.cfg;
  B200ST_CHECK(cf.model_type == MODEL_SPEECH || cf.model_type == MODEL_TEXT, "not a full encoder-decoder model handle");
  const int B = b.B, L = b.L, d = cf.d, V = cf.vocab;
  const bool speech = cf.model_type == MODEL_SPEECH;
  const int Ts = speech ? (((b.T + 1) / 2) + 1) / 2 : b.T;     // encoder length
  const int Ms = B * Ts, Md = B * L;
  c.training = b.training != 0;
  c.seed = b.seed;
  c.seed_dev = b.seed_dev;
  if (backward) B200ST_CHECK(c.buf.grads != nullptr && b.trg != nullptr && b.trg_length != nullptr, "backward needs grads and targets");
  if (is16(c.adt)) B200ST_CHECK(c.buf.shadow != nullptr, "16-bit precision needs the 16-bit shadow arena");

  Scratch sc;
  alloc_scratch(c, sc, B, Ts > L ? Ts : L, Ts > L ? Ts : L, Ms > Md ? Ms : Md, Ms, backward);

  // ---- encoder side ----
  float* enc_bias = c.f32((int64_t)B * Ts);
  float* x0 = c.f32((int64_t)Ms * d);
  FrontSave fs;
  if (speech) {
    B200ST_CHECK(c.dry || (b.src && b.src_length), "speech model needs src and src_length");
    int32_t* klen = reinterpret_cast<int32_t*>(c.f32(B));
    RUN(length_to_bias(b.src_length, enc_bias, B, Ts, 2, c.st, klen));
    c.klen_bias = enc_bias; c.klen = klen;
    B200ST_TRY(speech_front_fwd(c, b.src, B, b.T, x0, fs));
  } else {
    B200ST_CHECK(c.dry || (b.src_ids && b.src_padding), "text model needs src ids and src_padding");
    RUN(padding_to_bias(b.src_padding, enc_bias, (int64_t)B * Ts, c.st));
    const std::string tab = cf.share_src_trg_embedding ? "trg.emb" : "srcemb.emb";
    RUN(embed_fwd(b.src_ids, c.P(tab), x0, B, Ts, d, cf.share_src_trg_embedding ? V : cf.src_vocab, 0,
                  c.drop(cf.postprocess_dropout, dropout_stream_id("enc.in_drop")), c.st));
  }
  EncoderSave es;
  B200ST_TRY(encoder_fwd(c, x0, enc_bias, B, Ts, sc, es, b.enc_out));
  if (b.stop_after_encoder) {
    if (b.enc_bias_out)
      RUN(cudaMemcpyAsync(b.enc_bias_out, enc_bias, sizeof(float) * (size_t)B * Ts, cudaMemcpyDeviceToDevice, c.st) == cudaSuccess ? 0 : 1);
    return 0;
  }

  // ---- decoder side ----
  float* y0 = c.f32((int64_t)Md * d);
  RUN(embed_fwd(b.trg_input, c.P("trg.emb"), y0, B, L, d, V, 0, c.drop(cf.postprocess_dropout, dropout_stream_id("dec.in_drop")), c.st));
  DecoderSave ds;
  B200ST_TRY(decoder_fwd(c, y0, B, L, es.out, Ts, enc_bias, sc, ds, nullptr));

  // ---- logits + loss ----
  const bool want_loss = b.trg != nullptr && b.trg_length != nullptr;
  float* logits = b.logits;
  if (!logits && want_loss) logits = c.f32((int64_t)Md * V);
  if (logits) {
    GemmArgs g = gemm_defaults();
    g.M = Md; g.N = V; g.K = d;
    g.A = GemmOperand{ds.out, c.adt, 0, d, 0, 0};
    g.B = c.W("trg.emb", 0, d);
    g.C = logits; g.c_dtype = F32; g.ldc = V;
    g.epi.bias = c.P("trg.bias");
    RUN(gemm(g, c.st));
  }
  void* dlogits = nullptr;
  if (want_loss) {
    float* nll = b.nll_sum ? b.nll_sum : c.f32(B);
    float* ntok = b.n_tokens ? b.n_tokens : c.f32(B);
    float* loss = b.loss ? b.loss : c.f32(1);
    if (backward) dlogits = c.act((int64_t)Md * V);
    RUN(lsce_fwd_bwd(logits, b.trg, b.trg_length, B, L, V, cf.label_smoothing, nll, ntok, loss, dlogits, c.adt,
                     b.loss_scale > 0.f ? b.loss_scale : 1.f, b.loss_scale_dev, c.st));
  }
  if (!backward) return 0;

  // =========================== backward ===========================
  if (!c.dry && side_stream().ok && !tc_profile_active()) c.side = &side_stream();
  if (!c.dry && b.allreduce_grads) {
    B200ST_CHECK(c.m.sync != nullptr, "allreduce_grads needs b200st_comm_init on this handle");
    c.sync = c.m.sync;
    c.sync_hi = c.m.arena_numel;
    comm_begin_step(c.sync);
    // the persistent GEMM grids assign tiles statically to `gridDim.x` CTAs: size them to the SMs NCCL leaves free, or the
    // CTAs that find no SM run as a second wave after the others have finished
    gemm_set_reserved_sms(comm_reserved_sms(c.sync));
  }
  // reverse-arena-order buckets only when no tensor receives gradient later than its bucket (text models may tie the
  // source and target embeddings: one all-reduce at the end)
  const bool buckets = speech;
  // logits layer: dE += dlogits^T dec_out ; db += colsum ; d_dec_out = dlogits E
  {
    GemmArgs g = gemm_defaults();
    g.M = V; g.N = d; g.K = Md;
    g.A = GemmOperand{dlogits, c.adt, 1, V, 0, 0};
    g.B = GemmOperand{ds.out, c.adt, 1, d, 0, 0};
    g.C = c.G("trg.emb"); g.c_dtype = F32; g.ldc = d;
    g.epi.accumulate = 1; g.splitk = 0;
    c.cur_par = 1;                       // dlogits is never reused: let the first backward block (parity 0) run ahead
    cudaStream_t ws = c.wgrad_stream();
    RUN(gemm(g, ws));
    RUN(colsum_accum(dlogits, c.adt, Md, V, V, c.G("trg.bias"), ws));
    c.wgrad_done(ws);
  }
  float* d_dec = c.f32((int64_t)Md * d);
  {
    GemmArgs g = gemm_defaults();
    g.M = Md; g.N = d; g.K = V;
    g.A = GemmOperand{dlogits, c.adt, 0, V, 0, 0};
    g.B = c.W("trg.emb", 1, d);
    g.C = d_dec; g.c_dtype = F32; g.ldc = d;
    if (is16(c.adt)) {
      // K = V = 8192 against only (B*L / 128) x (d / 64) output tiles: split-K with fp32 reduce-add into a zeroed buffer
      RUN(cudaMemsetAsync(d_dec, 0, sizeof(float) * (size_t)Md * d, c.st) == cudaSuccess ? 0 : 1);
      g.epi.accumulate = 1;
      g.splitk = 0;
    }
    RUN(gemm(g, c.st));
  }
  float* dy = c.f32((int64_t)Md * d);
  float* dy_tmp = c.f32((int64_t)Md * d);
  float* d_enc = c.f32((int64_t)Ms * d);
  RUN(fill_f32(d_enc, 0.f, (int64_t)Ms * d, c.st));
  B200ST_TRY(decoder_bwd(c, d_dec, dy, dy_tmp, d_enc, true, sc, ds));
  RUN(embed_bwd(b.trg_input, dy, c.G("trg.emb"), B, L, d, V, c.drop(cf.postprocess_dropout, dropout_stream_id("dec.in_drop")), c.st));
  if (buckets) B200ST_TRY(c.reduce_down_to("dec.0.self.ln.gamma"));     // decoder + output layer: ~40 MB under the encoder backward
  float* dx = c.f32((int64_t)Ms * d);
  float* dx_tmp = c.f32((int64_t)Ms * d);
  B200ST_TRY(encoder_bwd(c, d_enc, dx, dx_tmp, sc, es, buckets));
  if (buckets) B200ST_TRY(c.reduce_down_to("enc.0.att.ln.gamma"));
  if (speech) {
    B200ST_TRY(speech_front_bwd(c, b.src, dx, fs));
  } else {
    const std::string tab = cf.share_src_trg_embedding ? "trg.emb" : "srcemb.emb";
    RUN(embed_bwd(b.src_ids, dx, c.G(tab), B, Ts, d, cf.share_src_trg_embedding ? V : cf.src_vocab,
                  c.drop(cf.postprocess_dropout, dropout_stream_id("enc.in_drop")), c.st));
  }
  c.join_side();        // the optimizer / all-reduce on `st` must see every weight gradient
  if (c.sync) {
    gemm_set_reserved_sms(0);
    B200ST_TRY(c.reduce_down_to(""));        // the rest (front-end, or everything when not bucketed)
    B200ST_TRY(comm_join(c.sync, c.st));
  }
  return 0;
}

// Runs `body` twice: a planning pass (no launches) that sizes the workspace, then the real pass.
template <class F>
static int run_planned(const Model& m, const Buffers& buf, cudaStream_t st, F&& body, size_t* need_out) {
  static char dummy[64];
  Buffers fake = buf;
  if (!fake.params) fake.params = reinterpret_cast<const float*>(dummy);
  if (!fake.shadow) fake.shadow = dummy;
  if (need_out && !fake.grads) fake.grads = reinterpret_cast<float*>(dummy);
  fake.workspace = nullptr; fake.workspace_bytes = 0;
  Ctx dry(m, fake, nullptr, true);
  B200ST_TRY(body(dry));
  const size_t need = dry.ar.off + 512;
  if (need_out) { *need_out = need; return 0; }
  B200ST_CHECK(buf.params != nullptr && buf.workspace != nullptr, "params / workspace missing");
  B200ST_CHECK((reinterpret_cast<uintptr_t>(buf.workspace) & 255) == 0, "workspace must be 256-byte aligned");
  B200ST_CHECK(buf.workspace_bytes >= need, "workspace too small: need " + std::to_string(need) + " bytes, have " +
                                                std::to_string(buf.workspace_bytes));
  if (is16(m.adt)) B200ST_CHECK(buf.shadow != nullptr, "16-bit precision needs the 16-bit shadow arena");
  Ctx real(m, buf, st, false);
  // All dropout keep-bits of the call in ONE launch: the planning pass recorded every site in allocation order (the real
  // pass allocates identically), the table travels as a kernel argument.
  if (!dry.drop_sites.empty() && dry.drop_sites.size() <= 128) {
    DropBitsTable t{};
    t.n = (int)dry.drop_sites.size();
    int64_t g = 0;
    for (int i = 0; i < t.n; ++i) {
      const auto& ds = dry.drop_sites[i];
      t.stream[i] = ds.stream; t.thresh[i] = dropout_thresh16(ds.p); t.goff[i] = g; t.boff[i] = (int64_t)ds.arena_off;
      g += ds.groups;
    }
    t.goff[t.n] = g;
    // The generator is pure ALU work: it runs on the side stream under the (bandwidth-bound) kernels that precede the
    // first dropout consumer; Ctx::drop() makes `st` wait for it at that first consumer.
    SideStream& ss = side_stream();
    cudaStream_t bs = st;
    if (ss.ok && cudaEventRecord(ss.fork, st) == cudaSuccess && cudaStreamWaitEvent(ss.stream, ss.fork, 0) == cudaSuccess) bs = ss.stream;
    B200ST_TRY(dropout_bits_multi(t, dry.seed, dry.seed_dev, reinterpret_cast<uint8_t*>(buf.workspace), bs));
    if (bs != st) {
      B200ST_CUDA(cudaEventRecord(ss.bits_done, bs));
      real.bits_event = ss.bits_done;
    }
    real.bits_pregenerated = true;
  }
  const int body_rc = body(real);
  real.wait_bits();                     // no consumer ran (or an error unwound): still join the side stream
  B200ST_TRY(body_rc);
  B200ST_CHECK(!real.launch_failed, "dropout bitmap kernel launch failed");
  if (real.bits_pregenerated) {
    B200ST_CHECK(real.drop_sites.size() == dry.drop_sites.size(),
                 "dropout site plan mismatch: real " + std::to_string(real.drop_sites.size()) + " vs planned " +
                     std::to_string(dry.drop_sites.size()));
    for (size_t i = 0; i < real.drop_sites.size(); ++i)
      B200ST_CHECK(real.drop_sites[i].arena_off == dry.drop_sites[i].arena_off && real.drop_sites[i].stream == dry.drop_sites[i].stream,
                   "dropout site plan mismatch");
  }
  return 0;
}

}  // namespace

size_t model_workspace_bytes(const Model& m, int B, int T, int L, int training) {
  static const int64_t dummy = 0;
  Batch b{};
  b.B = B; b.T = T; b.L = L; b.training = training;
  b.trg = &dummy; b.trg_length = &dummy;     // plan with the loss (and the backward pass when training)
  Buffers buf{};
  size_t need = 0;
  if (run_planned(m, buf, nullptr, [&](Ctx& c) { return model_run(c, b, training != 0); }, &need) != 0) return 0;
  return need;
}

int model_forward(const Model& m, const Buffers& buf, const Batch& b, bool backward, cudaStream_t st) {
  return run_planned(m, buf, st, [&](Ctx& c) { return model_run(c, b, backward); }, nullptr);
}

// ---- stack-level API (forward only) ---------------------------------------------------------------
namespace {

int encoder_api_body(Ctx& c, const float* x, const float* padding, int B, int T, float* out, int training, uint64_t seed) {
  const Config& cf = c.m.cfg;
  c.training = training != 0; c.seed = seed;
  Scratch sc;
  alloc_scratch(c, sc, B, T, T, B * T, B * T, false);
  float* bias = c.f32((int64_t)B * T);
  RUN(padding_to_bias(padding, bias, (int64_t)B * T, c.st));
  float* x0 = c.f32((int64_t)B * T * cf.d);
  // encoder input dropout (transformer_encoder.py:125-127)
  RUN(cast_dropout(x, x0, F32, (int64_t)B * T * cf.d, c.drop(cf.postprocess_dropout, dropout_stream_id("enc.in_drop")), c.st));
  EncoderSave es;
  return encoder_fwd(c, x0, bias, B, T, sc, es, out);
}

int decoder_api_body(Ctx& c, const float* x, const float* memory, const float* memory_padding, int B, int L, int Tm, float* out,
                     int training, uint64_t seed) {
  const Config& cf = c.m.cfg;
  c.training = training != 0; c.seed = seed;
  const int d = cf.d;
  Scratch sc;
  const int Tmax = L > Tm ? L : Tm;
  alloc_scratch(c, sc, B, L, Tmax, B * L, B * Tm, false);
  float* x0 = c.f32((int64_t)B * L * d);
  RUN(cast_dropout(x, x0, F32, (int64_t)B * L * d, c.drop(cf.postprocess_dropout, dropout_stream_id("dec.in_drop")), c.st));
  void* mem = nullptr; float* mbias = nullptr;
  if (memory) {
    mem = c.act((int64_t)B * Tm * d);
    RUN(cast_dropout(memory, mem, c.adt, (int64_t)B * Tm * d, no_dropout(), c.st));
    mbias = c.f32((int64_t)B * Tm);
    RUN(padding_to_bias(memory_padding, mbias, (int64_t)B * Tm, c.st));
  }
  DecoderSave ds;
  return decoder_fwd(c, x0, B, L, mem, Tm, mbias, sc, ds, out);
}

int mha_api_body(Ctx& c, const float* query, const float* memory, const float* bias, int B, int Tq, int Tk, float* out) {
  const Config& cf = c.m.cfg;
  const int u = cf.d;
  const int64_t Mq = (int64_t)B * Tq, Mk = (int64_t)B * Tk;
  void* qin = c.act(Mq * cf.mha_din);
  RUN(cast_dropout(query, qin, c.adt, Mq * cf.mha_din, no_dropout(), c.st));
  float* S = c.f32((int64_t)B * cf.heads * Tq * round8(Tk));
  void* p_pre = c.act((int64_t)B * cf.heads * Tq * round8(Tk));
  void* ctx = c.act(Mq * u);
  float* lse = c.f32((int64_t)B * cf.heads * Tq);
  GemmEpilogue e0 = gemm_defaults().epi;
  AttnDims dims{B, cf.heads, Tq, Tk, u};
  if (cf.mha_self) {
    void* qkv = c.act(Mq * 3 * u);
    B200ST_TRY(linear_fwd(c, qin, cf.mha_din, (int)Mq, cf.mha_din, 3 * u, "att.qkv.kernel", "att.qkv.bias", e0, qkv, c.adt, 3 * u));
    View q{qkv, 3 * u}, k{c.act_off(qkv, u), 3 * u}, v{c.act_off(qkv, 2 * u), 3 * u};
    B200ST_TRY(attention_fwd(c, dims, q, k, v, bias, 0, no_dropout(), S, p_pre, nullptr, ctx, lse));
  } else {
    void* min = c.act(Mk * cf.mha_dmem);
    RUN(cast_dropout(memory, min, c.adt, Mk * cf.mha_dmem, no_dropout(), c.st));
    void* qb = c.act(Mq * u);
    void* kv = c.act(Mk * 2 * u);
    B200ST_TRY(linear_fwd(c, qin, cf.mha_din, (int)Mq, cf.mha_din, u, "att.q.kernel", "att.q.bias", e0, qb, c.adt, u));
    B200ST_TRY(linear_fwd(c, min, cf.mha_dmem, (int)Mk, cf.mha_dmem, 2 * u, "att.kv.kernel", "att.kv.bias", e0, kv, c.adt, 2 * u));
    View q{qb, u}, k{kv, 2 * u}, v{c.act_off(kv, u), 2 * u};
    B200ST_TRY(attention_fwd(c, dims, q, k, v, bias, 0, no_dropout(), S, p_pre, nullptr, ctx, lse));
  }
  return linear_fwd(c, ctx, u, (int)Mq, u, cf.mha_dout, "att.out.kernel", "att.out.bias", e0, out, F32, cf.mha_dout);
}

}  // namespace

int encoder_forward_api(const Model& m, const Buffers& buf, const float* x, const float* padding, int B, int T, float* out,
                        int training, uint64_t seed, cudaStream_t st, size_t* need) {
  B200ST_CHECK(m.cfg.model_type != MODEL_DECODER && m.cfg.model_type != MODEL_MHA, "handle has no encoder");
  return run_planned(m, buf, st, [&](Ctx& c) { return encoder_api_body(c, x, padding, B, T, out, training, seed); }, need);
}
int decoder_forward_api(const Model& m, const Buffers& buf, const float* x, const float* memory, const float* memory_padding,
                        int B, int L, int Tm, float* out, int training, uint64_t seed, cudaStream_t st, size_t* need) {
  B200ST_CHECK(m.cfg.model_type != MODEL_ENCODER && m.cfg.model_type != MODEL_MHA, "handle has no decoder");
  return run_planned(m, buf, st,
                     [&](Ctx& c) { return decoder_api_body(c, x, memory, memory_padding, B, L, Tm, out, training, seed); }, need);
}
int mha_forward_api(const Model& m, const Buffers& buf, const float* query, const float* memory, const float* bias, int B, int Tq,
                    int Tk, float* out, cudaStream_t st, size_t* need) {
  B200ST_CHECK(m.cfg.model_type == MODEL_MHA, "not a MultiHeadAttention handle");
  return run_planned(m, buf, st, [&](Ctx& c) { return mha_api_body(c, query, memory, bias, B, Tq, Tk, out); }, need);
}

}  // namespace b200st
