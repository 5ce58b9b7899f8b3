// GEMM problem description shared by the tcgen05 (bf16) and the SIMT (fp32) kernels.
//
//   C[b2][b1][m][n] (op)= epilogue( alpha * sum_k A[b2][b1](m,k) * B[b2][b1](n,k) )
//
// A is logically [M,K], B is logically [N,K] ("NT" form, the tcgen05 native form).  Each operand is
// either K-major (k contiguous, ld = stride between rows m / n) or MN-major (m / n contiguous,
// ld = stride between successive k).  Every contraction of the model (dense fwd / dgrad / wgrad,
// QK^T, PV and their backward products, conv2 as im2col GEMM) is one GemmArgs.
#pragma once
#include "common.cuh"

namespace b200st {

struct GemmOperand {
  const void* ptr;
  int dtype;        // F32 (SIMT path) or BF16 (tcgen05 path)
  int mn_major;     // 0: K contiguous, 1: M/N contiguous
  int64_t ld;       // elements
  int64_t sb1, sb2; // batch strides (elements)
};

struct GemmEpilogue {
  float alpha;
  const float* bias;        // [N] fp32 or null (added after alpha)
  int relu;                 // max(v,0) after bias
  const void* mask_src;     // optional: v *= (mask_src[m,n] > 0); indexed like C with mask_ld/sb
  int mask_dtype;
  int64_t mask_ld, mask_sb1, mask_sb2;
  DropoutSpec drop;         // applied after relu/mask; element index = ((b2*nb1+b1)*M + m)*N + n
  const float* residual;    // optional fp32, added last; indexed with res_ld/sb (sb may be 0)
  int64_t res_ld, res_sb1, res_sb2;
  int accumulate;           // C += v (fp32 C only); forced (atomic) when splitk > 1
};

struct GemmArgs {
  int M, N, K;
  int nb1, nb2;
  GemmOperand A, B;
  void* C;
  int c_dtype;
  int64_t ldc, c_sb1, c_sb2;
  GemmEpilogue epi;
  int splitk;               // >=1 ; >1 requires fp32 C, accumulate semantics, no nonlinear epilogue
};

inline GemmArgs gemm_defaults() {
  GemmArgs g{};
  g.nb1 = g.nb2 = 1;
  g.epi.alpha = 1.f;
  g.epi.drop = no_dropout();
  g.splitk = 1;
  return g;
}

// Applies the epilogue to one accumulator value.  `e_idx` is the dropout element index.
__device__ __forceinline__ float gemm_epilogue_value(const GemmEpilogue& ep, float acc, int m, int n, int64_t boff_mask,
                                                     int64_t boff_res, uint64_t e_idx) {
  float v = acc * ep.alpha;
  if (ep.bias) v += __ldg(ep.bias + n);
  if (ep.relu) v = fmaxf(v, 0.f);
  if (ep.mask_src) {
    float s = load_as_f32(ep.mask_src, ep.mask_dtype, boff_mask + (int64_t)m * ep.mask_ld + n);
    v = s > 0.f ? v : 0.f;
  }
  if (ep.drop.p > 0.f) v = drop_keep1(ep.drop, e_idx) ? v * ep.drop.scale : 0.f;
  if (ep.residual) v += __ldg(ep.residual + boff_res + (int64_t)m * ep.res_ld + n);
  return v;
}

// Host launchers (return 0 on success; message via set_last_error).
int gemm_simt_f32(const GemmArgs& g, cudaStream_t stream);
int gemm_tc_bf16(const GemmArgs& g, cudaStream_t stream);
// weight gradients of one backward block in one launch; returns 2 when the group does not qualify (nothing launched), 1 on error
int gemm_wgrad_group(const GemmArgs* gs, int n, cudaStream_t stream);
// Dispatch on operand dtype: F32 operands -> SIMT fp32 FMA kernel, BF16 operands -> tcgen05 kernel.
int gemm(const GemmArgs& g, cudaStream_t stream);

// Fused FFN forward (tc_gemm.cu: fused_mlp_fwd_kernel): x_out(fp32, pre-initialised with the residual) += post-dropout of
// (dropout(relu(X W1 + b1)) W2 + b2); the hidden activations are also written to F1 for the backward pass.
bool fused_mlp_supported(int M, int d, int ffn, int dtype);
int fused_mlp_fwd(const void* X, int dtype, int M, int d, int ffn, const void* W1, const float* b1, const void* W2, const float* b2,
                  DropoutSpec drop_ffn, DropoutSpec drop_post, void* F1, float* x_out, cudaStream_t stream, int* tickets = nullptr);
// tickets (optional): int [ceil(M / 128)], zero before the first use: hidden slices reduce in slice order (deterministic)

int fused_mlp_bwd(const void* dY, int dtype, int M, int d, int ffn, const void* W1, const void* W2, const void* F1, float scale,
                  void* dF1, float* dH, cudaStream_t stream, int* tickets = nullptr);

// SMs the persistent tcgen05 grids leave to concurrent communication kernels (set by the model while gradient all-reduces
// overlap the backward pass; 0 = none)
void gemm_set_reserved_sms(int n);
int64_t tc_launch_count();
void tc_count_launch();
void tc_profile_begin();
bool tc_profile_active();   // per-launch event timing on: the model keeps every launch on one stream
int tc_profile_end(double* ms, double* flops, int64_t* launches);

}  // namespace b200st
