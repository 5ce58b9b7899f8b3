// Conv2d-subsampling front-end kernels (reference: neurst/layers/modalities/audio_modalities.py:84-109).
//
// conv1 (Cin small, K = 9*Cin) is a direct CUDA-core convolution with the channel LayerNorm fused in — one warp per
// output position, 8 contiguous channels per lane (16-byte loads/stores along the feature axis), warp-shuffle
// statistics.  Production shape (C = 256, Cin = 1): filter taps in registers, and the training path stores the
// NORMALISED activation xhat + 1/sigma ("normalised-save"): gamma/beta/ReLU are applied by the im2col in flight and the
// backward reads xhat back, so it needs neither the convolution recompute nor the statistics.  Other shapes use the
// generic kernels (filter in shared memory, post-ReLU activation stored, z1 recomputed in the backward).
// conv2 is lowered to tcgen05 GEMMs through im2col (forward / wgrad) and a dcol GEMM (dgrad); the dgrad's col2im
// gather is fused with the ReLU mask, the LayerNorm backward of conv1 and the parameter-gradient partial sums.
// conv1's filter gradient is one more split-K GEMM over the tiny im2col of the fbank (written by the same kernel).
#include "kernels.cuh"
#include "pdl.cuh"

namespace b200st {

#define DISPATCH_DTYPE(dt, T, ...)                                   \
  do {                                                               \
    if ((dt) == F32) { using T = float; __VA_ARGS__; }               \
    else if ((dt) == BF16) { using T = __nv_bfloat16; __VA_ARGS__; } \
    else if ((dt) == F16) { using T = __half; __VA_ARGS__; }         \
    else B200ST_FAIL("bad dtype");                                   \
  } while (0)

namespace {

template <typename T> __device__ __forceinline__ void ld8(const T* src, float (&v)[8]);
template <> __device__ __forceinline__ void ld8<float>(const float* src, float (&v)[8]) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(src)), b = __ldg(reinterpret_cast<const float4*>(src) + 1);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
template <int DT> __device__ __forceinline__ void unpack8_16(const uint4& pk, float (&v)[8]) {
  const uint32_t w[4] = {pk.x, pk.y, pk.z, pk.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float2 f = unpack2_16(w[i], DT); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
}
template <> __device__ __forceinline__ void ld8<__nv_bfloat16>(const __nv_bfloat16* src, float (&v)[8]) {
  unpack8_16<BF16>(__ldg(reinterpret_cast<const uint4*>(src)), v);
}
template <> __device__ __forceinline__ void ld8<__half>(const __half* src, float (&v)[8]) {
  unpack8_16<F16>(__ldg(reinterpret_cast<const uint4*>(src)), v);
}
template <typename T> __device__ __forceinline__ void st8(T* dst, const float (&v)[8]);
template <> __device__ __forceinline__ void st8<float>(float* dst, const float (&v)[8]) {
  *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(dst + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
template <int DT> __device__ __forceinline__ void st8_16(void* dst, const float (&v)[8]) {
  uint4 pk;
  pk.x = pack2_16(v[0], v[1], DT); pk.y = pack2_16(v[2], v[3], DT);
  pk.z = pack2_16(v[4], v[5], DT); pk.w = pack2_16(v[6], v[7], DT);
  *reinterpret_cast<uint4*>(dst) = pk;
}
template <> __device__ __forceinline__ void st8<__nv_bfloat16>(__nv_bfloat16* dst, const float (&v)[8]) { st8_16<BF16>(dst, v); }
template <> __device__ __forceinline__ void st8<__half>(__half* dst, const float (&v)[8]) { st8_16<F16>(dst, v); }

// 8 consecutive elements held in raw form (prefetch registers: 16 B for bf16, 32 B for fp32)
template <typename T> struct Vec8;
template <typename T16, int DT> struct Vec8_16 {
  uint4 r;
  __device__ __forceinline__ void load(const T16* p) { r = __ldg(reinterpret_cast<const uint4*>(p)); }
  __device__ __forceinline__ void zero() { r = make_uint4(0, 0, 0, 0); }
  __device__ __forceinline__ void get(float (&v)[8]) const { unpack8_16<DT>(r, v); }
};
template <> struct Vec8<__nv_bfloat16> : Vec8_16<__nv_bfloat16, BF16> {};
template <> struct Vec8<__half> : Vec8_16<__half, F16> {};
template <> struct Vec8<float> {
  float4 a, b;
  __device__ __forceinline__ void load(const float* p) { a = __ldg(reinterpret_cast<const float4*>(p)); b = __ldg(reinterpret_cast<const float4*>(p) + 1); }
  __device__ __forceinline__ void zero() { a = make_float4(0.f, 0.f, 0.f, 0.f); b = a; }
  __device__ __forceinline__ void get(float (&v)[8]) const {
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
};

// Channel owned by (lane, i): VEC => 8 contiguous channels per lane per 256-channel group; else lane-strided.
template <bool VEC> __device__ __forceinline__ int chan(int lane, int i) {
  return VEC ? (8 * lane + 256 * (i >> 3) + (i & 7)) : (lane + 32 * i);
}
// Shared-memory slot of channel c within a per-channel table: permuted so that the 32 lanes of a warp reading
// "their i-th channel" hit 32 consecutive banks (the natural order would be an 8-way bank conflict for VEC).
template <bool VEC> __device__ __forceinline__ int slot_of_channel(int c) {
  return VEC ? ((c & ~255) + ((c & 7) << 5) + ((c & 255) >> 3)) : c;
}
template <bool VEC> __device__ __forceinline__ int slot(int lane, int i) {
  return VEC ? (256 * (i >> 3) + 32 * (i & 7) + lane) : (lane + 32 * i);
}

// Loads / stores the CPL channels a lane owns at row pointer p (C channels per row).
template <typename T, bool VEC, int CPL>
__device__ __forceinline__ void load_row(const T* p, int lane, int C, float (&v)[CPL]) {
  if (VEC) {
#pragma unroll
    for (int g = 0; g < CPL / 8; ++g) {
      float t[8];
      const int c0 = 8 * lane + 256 * g;
      if (c0 < C) ld8<T>(p + c0, t);
      else {
#pragma unroll
        for (int j = 0; j < 8; ++j) t[j] = 0.f;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) v[8 * g + j] = t[j];
    }
  } else {
#pragma unroll
    for (int i = 0; i < CPL; ++i) { const int c = lane + 32 * i; v[i] = c < C ? to_f32(p[c]) : 0.f; }
  }
}
template <typename T, bool VEC, int CPL>
__device__ __forceinline__ void store_row(T* p, int lane, int C, const float (&v)[CPL]) {
  if (VEC) {
#pragma unroll
    for (int g = 0; g < CPL / 8; ++g) {
      const int c0 = 8 * lane + 256 * g;
      if (c0 < C) {
        float t[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) t[j] = v[8 * g + j];
        st8<T>(p + c0, t);
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < CPL; ++i) { const int c = lane + 32 * i; if (c < C) p[c] = from_f32<T>(v[i]); }
  }
}

// z[i] = bias + sum_taps x * w  for the lane's channels.  The filter ([9*Cin][C] fp32) and bias live in shared memory
// (registers are needed for occupancy: these kernels are latency-bound on global loads).
template <bool VEC, int CPL, bool CIN1>
struct ConvTaps {
  const float* sw;      // smem [9*Cin][C]
  const float* sb;      // smem [C]
  int cp;               // padded channel count of one table row
  __device__ __forceinline__ void init(float* smem, const float* __restrict__ w, const float* __restrict__ bias, int Cin, int C) {
    const int Cp = VEC ? ((C + 255) & ~255) : C;       // padded row so that permuted slots stay in range
    const int nw = 9 * Cin * Cp;
    for (int i = threadIdx.x; i < 9 * Cin * C; i += blockDim.x) smem[(i / C) * Cp + slot_of_channel<VEC>(i % C)] = w[i];
    for (int i = threadIdx.x; i < C; i += blockDim.x) smem[nw + slot_of_channel<VEC>(i)] = bias[i];
    sw = smem; sb = smem + nw; cp = Cp;
    __syncthreads();
  }
  // xv: the 9*Cin input taps of this position (zero outside), in (kh,kw,ci) order
  __device__ __forceinline__ void apply(const float* xv, int lane, int Cin, int C, float (&z)[CPL]) const {
#pragma unroll
    for (int i = 0; i < CPL; ++i) { const int c = chan<VEC>(lane, i); z[i] = c < C ? sb[slot<VEC>(lane, i)] : 0.f; }
    if (CIN1) {
#pragma unroll
      for (int tp = 0; tp < 9; ++tp) {
        const float x = xv[tp];
        const float* wr = sw + tp * cp;
#pragma unroll
        for (int i = 0; i < CPL; ++i) { const int c = chan<VEC>(lane, i); if (c < C) z[i] = fmaf(x, wr[slot<VEC>(lane, i)], z[i]); }
      }
    } else {
      for (int k = 0; k < 9 * Cin; ++k) {
        const float x = xv[k];
        const float* wr = sw + k * cp;
#pragma unroll
        for (int i = 0; i < CPL; ++i) { const int c = chan<VEC>(lane, i); if (c < C) z[i] = fmaf(x, wr[slot<VEC>(lane, i)], z[i]); }
      }
    }
  }
};

constexpr int MAX_TAPS = 36;   // 9 * Cin, Cin <= 4

__device__ __forceinline__ void gather_taps(const float* __restrict__ src, int b, int t1, int f1, int Tn, int F, int Cin, float* xv) {
  for (int tp = 0; tp < 9; ++tp) {
    const int t = 2 * t1 + tp / 3 - 1, f = 2 * f1 + tp % 3 - 1;
    const bool ok = t >= 0 && t < Tn && f >= 0 && f < F;
    for (int ci = 0; ci < Cin; ++ci) xv[tp * Cin + ci] = ok ? __ldg(&src[(((int64_t)b * Tn + t) * F + f) * Cin + ci]) : 0.f;
  }
}

template <int CPL, bool VEC>
__device__ __forceinline__ void ln_stats(const float (&z)[CPL], int lane, int C, float eps, float& mean, float& rstd) {
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < CPL; ++i) if (chan<VEC>(lane, i) < C) sum += z[i];
  mean = warp_sum(sum) / C;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < CPL; ++i) if (chan<VEC>(lane, i) < C) { const float dl = z[i] - mean; sq += dl * dl; }
  rstd = 1.0f / sqrtf(warp_sum(sq) / C + eps);
}

// ---------------------------------------------------------------------------------------------
// conv1 + LN + ReLU forward
// ---------------------------------------------------------------------------------------------
template <typename T, bool VEC, int CPL, bool CIN1>
__global__ void __launch_bounds__(256, (CPL <= 8 ? 3 : 1)) conv1_fwd_kernel(const float* __restrict__ src, const float* __restrict__ w,
                                                         const float* __restrict__ bias, const float* __restrict__ gamma,
                                                         const float* __restrict__ beta, float eps, T* __restrict__ y, int B,
                                                         int Tn, int F, int Cin, int C, int T1, int F1, int use_ln,
                                                         float* __restrict__ rstd_out) {
  pdl_wait();
  pdl_trigger();
  extern __shared__ float conv_smem[];
  const int lane = threadIdx.x & 31;
  ConvTaps<VEC, CPL, CIN1> taps;
  taps.init(conv_smem, w, bias, CIN1 ? 1 : Cin, C);
  float greg[CPL], bereg[CPL];
#pragma unroll
  for (int i = 0; i < CPL; ++i) {
    const int c = chan<VEC>(lane, i);
    greg[i] = (use_ln && c < C) ? gamma[c] : 1.f; bereg[i] = (use_ln && c < C) ? beta[c] : 0.f;
  }
  const int64_t npos = (int64_t)B * T1 * F1;
  const int64_t warps_total = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t pos = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); pos < npos; pos += warps_total) {
    const int f1 = (int)(pos % F1);
    const int t1 = (int)((pos / F1) % T1);
    const int b = (int)(pos / ((int64_t)F1 * T1));
    float xv[CIN1 ? 9 : MAX_TAPS];
    gather_taps(src, b, t1, f1, Tn, F, CIN1 ? 1 : Cin, xv);
    float z[CPL];
    taps.apply(xv, lane, Cin, C, z);
    if (rstd_out) {
      // normalised-save mode: store xhat and 1/sigma only; gamma, beta and the ReLU are applied by the consumers
      // (im2col forward, conv1 backward), which removes the convolution recompute from the backward pass
      float mean, rstd;
      ln_stats<CPL, VEC>(z, lane, C, eps, mean, rstd);
#pragma unroll
      for (int i = 0; i < CPL; ++i) z[i] = (z[i] - mean) * rstd;
      if (lane == 0) rstd_out[pos] = rstd;
      store_row<T, VEC, CPL>(y + pos * C, lane, C, z);
      continue;
    }
    if (use_ln) {
      float mean, rstd;
      ln_stats<CPL, VEC>(z, lane, C, eps, mean, rstd);
#pragma unroll
      for (int i = 0; i < CPL; ++i) z[i] = (z[i] - mean) * rstd * greg[i] + bereg[i];
    }
#pragma unroll
    for (int i = 0; i < CPL; ++i) z[i] = fmaxf(z[i], 0.f);
    store_row<T, VEC, CPL>(y + pos * C, lane, C, z);
  }
}

// ---------------------------------------------------------------------------------------------
// conv1 forward, production shape (C == 256, Cin == 1): the lane's 9 x 8 filter taps live in registers (no shared-memory
// traffic: the generic kernel is LDS-bound), the 9 fbank taps of a position are fetched by lanes 0..8 one position
// ahead and broadcast with shuffles, each warp walks a contiguous range of positions.
// SAVE: store xhat + 1/sigma (normalised-save mode); else y = relu(LN(z) * gamma + beta).
// ---------------------------------------------------------------------------------------------
// d{0,1} += a * b{0,1} as one packed fp32x2 instruction (FFMA2, sm_100): half the issue slots of two FFMAs, and the same
// rounding (one fma.rn per element); B200 cfg-2 step 6.155 ms vs 6.173 ms with scalar fmaf (profiles/r02_bench_cfg2_ffma2.json)
__device__ __forceinline__ void ffma2_bcast(float& d0, float& d1, float a, float b0, float b1) {
  uint64_t av, bv, cv;
  asm("mov.b64 %0, {%1, %1};" : "=l"(av) : "f"(a));
  asm("mov.b64 %0, {%1, %2};" : "=l"(bv) : "f"(b0), "f"(b1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(cv) : "f"(d0), "f"(d1));
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(cv) : "l"(av), "l"(bv));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d0), "=f"(d1) : "l"(cv));
}

template <typename T, bool SAVE>
__global__ void __launch_bounds__(256, 2) conv1_fwd_c256_kernel(const float* __restrict__ src, const float* __restrict__ w,
                                                                const float* __restrict__ bias, const float* __restrict__ gamma,
                                                                const float* __restrict__ beta, float eps, T* __restrict__ y,
                                                                float* __restrict__ rstd_out, int B, int Tn, int F, int T1, int F1) {
  pdl_wait();
  pdl_trigger();
  constexpr int C = 256;
  const int lane = threadIdx.x & 31;
  float wreg[9][8], breg[8], greg[8], bereg[8];
#pragma unroll
  for (int tp = 0; tp < 9; ++tp) ld8<float>(w + tp * C + 8 * lane, wreg[tp]);
  ld8<float>(bias + 8 * lane, breg);
  if (!SAVE) { ld8<float>(gamma + 8 * lane, greg); ld8<float>(beta + 8 * lane, bereg); }
  const int64_t npos = (int64_t)B * T1 * F1;
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  // each warp walks a contiguous range of positions: neighbouring positions share fbank taps (L1 hits); the warp-interleaved
  // order was measured slower here (233 vs 203 us) although it helps the backward kernel slightly
  const int64_t per = (npos + nwarps - 1) / nwarps;
  const int64_t wid = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int64_t pos = wid * per;
  const int64_t pos_end = (pos + per < npos) ? pos + per : npos;
  if (pos >= pos_end) return;
  int f1 = (int)(pos % F1);
  int t1 = (int)((pos / F1) % T1);
  int b = (int)(pos / ((int64_t)F1 * T1));
  const int tap_dt = lane / 3 - 1, tap_df = lane % 3 - 1;      // lanes 0..8 own one fbank tap each
  auto load_tap = [&](int bb, int tt1, int ff1) {
    float v = 0.f;
    if (lane < 9) {
      const int t = 2 * tt1 + tap_dt, f = 2 * ff1 + tap_df;
      if (t >= 0 && t < Tn && f >= 0 && f < F) v = __ldg(&src[((int64_t)bb * Tn + t) * F + f]);
    }
    return v;
  };
  // the taps of the next RING-1 positions are in flight during the math of the current one (one position ahead left the
  // warps waiting on L2: 203 us for 0.28 GB of traffic, ncu round 2)
  constexpr int RING = 4;
  int64_t ipos = pos;
  int ib = b, it1 = t1, if1 = f1;
  auto issue_next = [&]() {
    float v = 0.f;
    if (ipos < pos_end) {
      v = load_tap(ib, it1, if1);
      ++ipos;
      if (++if1 == F1) { if1 = 0; if (++it1 == T1) { it1 = 0; ++ib; } }
    }
    return v;
  };
  auto process = [&](int64_t pp, float xv) {
    float z[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) z[i] = breg[i];
#pragma unroll
    for (int tp = 0; tp < 9; ++tp) {
      const float x = __shfl_sync(0xffffffffu, xv, tp);
#pragma unroll
      for (int i = 0; i < 8; i += 2) ffma2_bcast(z[i], z[i + 1], x, wreg[tp][i], wreg[tp][i + 1]);
    }
    float s1 = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s1 += z[i];
    const float mean = warp_sum(s1) * (1.0f / C);
    float s2 = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { z[i] -= mean; s2 = fmaf(z[i], z[i], s2); }
    const float rstd = 1.0f / sqrtf(warp_sum(s2) * (1.0f / C) + eps);
    if (SAVE) {
#pragma unroll
      for (int i = 0; i < 8; ++i) z[i] *= rstd;
      if (lane == 0) rstd_out[pp] = rstd;
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) z[i] = fmaxf(fmaf(z[i] * rstd, greg[i], bereg[i]), 0.f);
    }
    st8<T>(y + pp * C + 8 * lane, z);
  };
  float ring[RING];
#pragma unroll
  for (int j = 0; j < RING - 1; ++j) ring[j] = issue_next();
  while (pos < pos_end) {
#pragma unroll
    for (int j = 0; j < RING; ++j) {
      if (pos < pos_end) {
        ring[(j + RING - 1) % RING] = issue_next();
        process(pos, ring[j]);
        ++pos;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// fused conv2-dgrad gather (col2im) + ReLU' + LN' of conv1 (recompute) -> dz1, im2col of src, db/dgamma/dbeta
// ---------------------------------------------------------------------------------------------
template <typename T, bool VEC, int CPL, bool CIN1>
__global__ void __launch_bounds__(256, (CPL <= 8 ? 2 : 1)) conv1_bwd_fused_kernel(
    const float* __restrict__ src, const float* __restrict__ w, const float* __restrict__ bias, const float* __restrict__ gamma,
    const float* __restrict__ beta, float eps, const T* __restrict__ y1, const T* __restrict__ dcol, T* __restrict__ dz1,
    T* __restrict__ col1, int K1p, float* __restrict__ db, float* __restrict__ dgamma, float* __restrict__ dbeta, int B, int Tn,
    int F, int Cin, int C, int T1, int F1, int T2, int F2, int use_ln) {
  pdl_wait();
  pdl_trigger();
  extern __shared__ float conv_smem[];   // filter | bias | [3][C] block partials: db | dgamma | dbeta
  float* sacc = conv_smem + (9 * (CIN1 ? 1 : Cin) + 1) * (VEC ? ((C + 255) & ~255) : C);
  for (int i = threadIdx.x; i < 3 * C; i += blockDim.x) sacc[i] = 0.f;
  const int lane = threadIdx.x & 31;
  ConvTaps<VEC, CPL, CIN1> taps;
  taps.init(conv_smem, w, bias, CIN1 ? 1 : Cin, C);
  float greg[CPL], bereg[CPL], a_db[CPL], a_dg[CPL], a_dbe[CPL];
#pragma unroll
  for (int i = 0; i < CPL; ++i) {
    const int c = chan<VEC>(lane, i);
    greg[i] = (use_ln && c < C) ? gamma[c] : 1.f; bereg[i] = (use_ln && c < C) ? beta[c] : 0.f;
    a_db[i] = a_dg[i] = a_dbe[i] = 0.f;
  }
  const int K1 = 9 * (CIN1 ? 1 : Cin);
  const int64_t npos = (int64_t)B * T1 * F1;
  const int64_t warps_total = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t pos = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); pos < npos; pos += warps_total) {
    const int f1 = (int)(pos % F1);
    const int t1 = (int)((pos / F1) % T1);
    const int b = (int)(pos / ((int64_t)F1 * T1));
    // ---- dy1 = col2im gather of dcol (<= 4 taps for stride 2) ----
    float d[CPL];
#pragma unroll
    for (int i = 0; i < CPL; ++i) d[i] = 0.f;
#pragma unroll
    for (int kh = 0; kh < 3; ++kh) {
      const int tt = t1 + 1 - kh;
      if (tt < 0 || (tt & 1) || (tt >> 1) >= T2) continue;
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const int ff = f1 + 1 - kw;
        if (ff < 0 || (ff & 1) || (ff >> 1) >= F2) continue;
        const int64_t row = ((int64_t)b * T2 + (tt >> 1)) * F2 + (ff >> 1);
        float t[CPL];
        load_row<T, VEC, CPL>(dcol + (row * 9 + kh * 3 + kw) * C, lane, C, t);
#pragma unroll
        for (int i = 0; i < CPL; ++i) d[i] += t[i];
      }
    }
    // ---- ReLU mask from the stored output ----
    {
      float yv[CPL];
      load_row<T, VEC, CPL>(y1 + pos * C, lane, C, yv);
#pragma unroll
      for (int i = 0; i < CPL; ++i) if (!(yv[i] > 0.f)) d[i] = 0.f;
    }
    // ---- recompute z1 and LayerNorm backward ----
    float xv[CIN1 ? 9 : MAX_TAPS];
    gather_taps(src, b, t1, f1, Tn, F, CIN1 ? 1 : Cin, xv);
    if (use_ln) {
      float z[CPL];
      taps.apply(xv, lane, Cin, C, z);
      float mean, rstd;
      ln_stats<CPL, VEC>(z, lane, C, eps, mean, rstd);
      float c1 = 0.f, c2 = 0.f;
#pragma unroll
      for (int i = 0; i < CPL; ++i) {
        z[i] = (z[i] - mean) * rstd;                 // xhat
        if (chan<VEC>(lane, i) < C) {
          const float g = d[i] * greg[i];
          c1 += g; c2 += g * z[i];
          a_dg[i] += d[i] * z[i]; a_dbe[i] += d[i];
        }
      }
      c1 = warp_sum(c1) / C; c2 = warp_sum(c2) / C;
#pragma unroll
      for (int i = 0; i < CPL; ++i) d[i] = (chan<VEC>(lane, i) < C) ? rstd * (d[i] * greg[i] - c1 - z[i] * c2) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < CPL; ++i) a_db[i] += d[i];
    store_row<T, VEC, CPL>(dz1 + pos * C, lane, C, d);
    // ---- im2col row of the fbank (operand of the filter-gradient GEMM) ----
    if (CIN1) {
      float val = 0.f;
#pragma unroll
      for (int tp = 0; tp < 9; ++tp) if (lane == tp) val = xv[tp];
      if (lane < K1p) col1[pos * K1p + lane] = from_f32<T>(val);
    } else {
      if (lane < K1p) col1[pos * K1p + lane] = from_f32<T>(lane < K1 ? xv[lane] : 0.f);
      if (K1p > 32 && lane + 32 < K1p) col1[pos * K1p + lane + 32] = from_f32<T>(lane + 32 < K1 ? xv[lane + 32] : 0.f);
    }
  }
#pragma unroll
  for (int i = 0; i < CPL; ++i) {
    const int c = chan<VEC>(lane, i);
    if (c < C) { atomicAdd(&sacc[c], a_db[i]); atomicAdd(&sacc[C + c], a_dg[i]); atomicAdd(&sacc[2 * C + c], a_dbe[i]); }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    atomicAdd(&db[i], sacc[i]);
    if (use_ln) { atomicAdd(&dgamma[i], sacc[C + i]); atomicAdd(&dbeta[i], sacc[2 * C + i]); }
  }
}


// ---------------------------------------------------------------------------------------------
// Backward from the saved normalised activations (C == 256, Cin == 1): col2im gather of dcol + ReLU' + LN' with xhat and
// 1/sigma read back (no convolution recompute, no statistics), db/dgamma/dbeta partials, fbank im2col rows for dW1.
// ---------------------------------------------------------------------------------------------
// IMPLICIT: `dcol` is the class-major tiled input gradient written by the implicit conv2 data-gradient GEMMs
// (tc_gemm.cu: conv2_dgrad_implicit) — one row per position instead of up to four tap rows to gather.
template <typename T, bool IMPLICIT>
__global__ void __launch_bounds__(256, 2) conv1_bwd_xhat_c256_kernel(
    const float* __restrict__ src, const T* __restrict__ gamma, const T* __restrict__ beta, const T* __restrict__ xhat,
    const float* __restrict__ rstd, const T* __restrict__ dcol, T* __restrict__ dz1, T* __restrict__ col1, int K1p,
    float* __restrict__ db, float* __restrict__ dgamma, float* __restrict__ dbeta, int B, int Tn, int F, int T1, int F1, int T2,
    int F2, int tu, int ub) {
  pdl_wait();
  pdl_trigger();
  constexpr int C = 256;
  __shared__ float sacc[3 * C];
  for (int i = threadIdx.x; i < 3 * C; i += blockDim.x) sacc[i] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  float greg[8], breg[8], a_db[8], a_dg[8], a_dbe[8];
  ld8<T>(gamma + 8 * lane, greg);       // affine parameters exactly as the forward used them (bf16 shadow in bf16 mode)
  ld8<T>(beta + 8 * lane, breg);
#pragma unroll
  for (int i = 0; i < 8; ++i) a_db[i] = a_dg[i] = a_dbe[i] = 0.f;
  const int64_t npos = (int64_t)B * T1 * F1;
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t wid = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int64_t pos = wid;                       // warp-interleaved positions: the grid sweeps one contiguous window of xhat / dz1 (-10 us vs a range per warp)
  const int64_t pos_end = npos;
  const int step_f = (int)(nwarps % F1), step_t = (int)((nwarps / F1) % T1), step_b = (int)(nwarps / ((int64_t)F1 * T1));
  if (pos < pos_end) {
    int f1 = (int)(pos % F1);
    int t1 = (int)((pos / F1) % T1);
    int b = (int)(pos / ((int64_t)F1 * T1));
    const int tap_dt = lane / 3 - 1, tap_df = lane % 3 - 1;      // lanes 0..8 own one fbank tap each
    // every global load of a position (fbank tap, xhat row, 1/sigma, dcol rows) is issued RING-1 positions ahead: the kernel is
    // bound by bytes in flight, not by bandwidth (ncu, round 2: 2.8 TB/s with one position ahead) — the implicit variant loads
    // one gradient row instead of four and spends the freed registers on a deeper ring
    constexpr int NDC = IMPLICIT ? 1 : 4;
    constexpr int RING = IMPLICIT ? 4 : 2;
    struct Loads { Vec8<T> xh, dc[NDC]; float rs, xv; };
    auto issue = [&](int64_t p, int bb, int tt1, int ff1, Loads& L) {
      L.xv = 0.f;
      if (lane < 9) {
        const int t = 2 * tt1 + tap_dt, f = 2 * ff1 + tap_df;
        if (t >= 0 && t < Tn && f >= 0 && f < F) L.xv = __ldg(&src[((int64_t)bb * Tn + t) * F + f]);
      }
      L.xh.load(xhat + p * C + 8 * lane);
      L.rs = __ldg(rstd + p);
      if constexpr (IMPLICIT) {
        const int cls = ((tt1 & 1) << 1) | (ff1 & 1), u = tt1 >> 1, v = ff1 >> 1;
        const int64_t row = (((int64_t)cls * B + bb) * ub + u / tu) * 128 + (u % tu) * F2 + v;
        L.dc[0].load(dcol + row * C + 8 * lane);
      } else {
        // col2im: t1 even -> kh = 1 ; t1 odd -> kh in {0, 2} (same along f); slot = 2 * a + c2
        const int kh0 = (tt1 & 1) ? 0 : 1, kw0 = (ff1 & 1) ? 0 : 1;
#pragma unroll
        for (int a = 0; a < 2; ++a) {
#pragma unroll
          for (int c2 = 0; c2 < 2; ++c2) {
            const int kh = kh0 + 2 * a, kw = kw0 + 2 * c2;
            const int t2 = (tt1 + 1 - kh) >> 1, f2 = (ff1 + 1 - kw) >> 1;
            const bool ok = (a == 0 || (tt1 & 1)) && (c2 == 0 || (ff1 & 1)) && t2 < T2 && f2 < F2;
            if (ok) L.dc[2 * a + c2].load(dcol + ((((int64_t)bb * T2 + t2) * F2 + f2) * 9 + kh * 3 + kw) * C + 8 * lane);
            else L.dc[2 * a + c2].zero();
          }
        }
      }
    };
    auto process = [&](int64_t pp, const Loads& cur) {
      float xh[8], d[8];
      cur.xh.get(xh);
      cur.dc[0].get(d);
#pragma unroll
      for (int k = 1; k < NDC; ++k) {
        float t8[8];
        cur.dc[k].get(t8);
#pragma unroll
        for (int i = 0; i < 8; ++i) d[i] += t8[i];
      }
      const float rs = cur.rs;
      float c1 = 0.f, c2s = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (!(fmaf(xh[i], greg[i], breg[i]) > 0.f)) d[i] = 0.f;      // ReLU' on y = xhat * gamma + beta
        const float g = d[i] * greg[i];
        c1 += g; c2s = fmaf(g, xh[i], c2s);
        a_dg[i] = fmaf(d[i], xh[i], a_dg[i]); a_dbe[i] += d[i];
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) { c1 += __shfl_xor_sync(0xffffffffu, c1, o); c2s += __shfl_xor_sync(0xffffffffu, c2s, o); }
      c1 *= (1.0f / C); c2s *= (1.0f / C);
#pragma unroll
      for (int i = 0; i < 8; ++i) { d[i] = rs * (d[i] * greg[i] - c1 - xh[i] * c2s); a_db[i] += d[i]; }
      st8<T>(dz1 + pp * C + 8 * lane, d);
      if (lane < K1p) col1[pp * K1p + lane] = from_f32<T>(lane < 9 ? cur.xv : 0.f);
    };
    // issue cursor (position whose loads are issued next) runs RING-1 positions ahead of the compute cursor `pos`
    int64_t ipos = pos;
    int ib = b, it1 = t1, if1 = f1;
    auto issue_next = [&](Loads& L) {
      if (ipos < pos_end) {
        issue(ipos, ib, it1, if1, L);
        ipos += nwarps;
        if1 += step_f; if (if1 >= F1) { if1 -= F1; ++it1; }
        it1 += step_t; if (it1 >= T1) { it1 -= T1; ++ib; }
        ib += step_b;
      }
    };
    Loads ring[RING];
#pragma unroll
    for (int j = 0; j < RING - 1; ++j) issue_next(ring[j]);
    while (pos < pos_end) {
#pragma unroll
      for (int j = 0; j < RING; ++j) {
        if (pos < pos_end) {
          issue_next(ring[(j + RING - 1) % RING]);
          process(pos, ring[j]);
          pos += nwarps;
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int c = 8 * lane + i;
    atomicAdd(&sacc[c], a_db[i]); atomicAdd(&sacc[C + c], a_dg[i]); atomicAdd(&sacc[2 * C + c], a_dbe[i]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    atomicAdd(&db[i], sacc[i]); atomicAdd(&dgamma[i], sacc[C + i]); atomicAdd(&dbeta[i], sacc[2 * C + i]);
  }
}

// ---------------------------------------------------------------------------------------------
// im2col for the 3x3 stride-2 pad-1 conv2 (NHWC): one warp per (row, tap) chunk of C channels
// ---------------------------------------------------------------------------------------------
// y = relu(x * gamma + beta) on one 16-byte vector (affine parameters in the activation dtype: for bf16 they come from
// the bf16 shadow arena and the math is packed HFMA2.BF16 / HMNMX2 — the same rounding the backward's ReLU mask assumes)
__device__ __forceinline__ uint4 affine_relu_vec(uint4 v, const __nv_bfloat162 (&g)[4], const __nv_bfloat162 (&b)[4]) {
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&v);
  const __nv_bfloat162 zero = __floats2bfloat162_rn(0.f, 0.f);
#pragma unroll
  for (int j = 0; j < 4; ++j) h[j] = __hmax2(__hfma2(h[j], g[j], b[j]), zero);
  return v;
}
__device__ __forceinline__ uint4 affine_relu_vec(uint4 v, const __half2 (&g)[4], const __half2 (&b)[4]) {
  __half2* h = reinterpret_cast<__half2*>(&v);
  const __half2 zero = __floats2half2_rn(0.f, 0.f);
#pragma unroll
  for (int j = 0; j < 4; ++j) h[j] = __hmax2(__hfma2(h[j], g[j], b[j]), zero);
  return v;
}
__device__ __forceinline__ uint4 affine_relu_vec(uint4 v, const float (&g)[4], const float (&b)[4]) {
  float* f = reinterpret_cast<float*>(&v);
#pragma unroll
  for (int j = 0; j < 4; ++j) f[j] = fmaxf(fmaf(f[j], g[j], b[j]), 0.f);
  return v;
}
template <typename T> struct AffineRegs;
template <> struct AffineRegs<__nv_bfloat16> {
  __nv_bfloat162 g[4], b[4];
  __device__ __forceinline__ void load(const __nv_bfloat16* gamma, const __nv_bfloat16* beta, int c) {
    const uint4 gv = __ldg(reinterpret_cast<const uint4*>(gamma + c)), bv = __ldg(reinterpret_cast<const uint4*>(beta + c));
#pragma unroll
    for (int j = 0; j < 4; ++j) { g[j] = reinterpret_cast<const __nv_bfloat162*>(&gv)[j]; b[j] = reinterpret_cast<const __nv_bfloat162*>(&bv)[j]; }
  }
};
template <> struct AffineRegs<__half> {
  __half2 g[4], b[4];
  __device__ __forceinline__ void load(const __half* gamma, const __half* beta, int c) {
    const uint4 gv = __ldg(reinterpret_cast<const uint4*>(gamma + c)), bv = __ldg(reinterpret_cast<const uint4*>(beta + c));
#pragma unroll
    for (int j = 0; j < 4; ++j) { g[j] = reinterpret_cast<const __half2*>(&gv)[j]; b[j] = reinterpret_cast<const __half2*>(&bv)[j]; }
  }
};
template <> struct AffineRegs<float> {
  float g[4], b[4];
  __device__ __forceinline__ void load(const float* gamma, const float* beta, int c) {
    const float4 gv = __ldg(reinterpret_cast<const float4*>(gamma + c)), bv = __ldg(reinterpret_cast<const float4*>(beta + c));
    g[0] = gv.x; g[1] = gv.y; g[2] = gv.z; g[3] = gv.w; b[0] = bv.x; b[1] = bv.y; b[2] = bv.z; b[3] = bv.w;
  }
};

// gamma != null: the source holds the normalised conv1 activations; y = relu(x * gamma + beta) is applied in flight.
// ONE: C == 32 vectors, i.e. each lane owns exactly one 16-byte vector of the row (affine parameters stay in registers).
template <typename T, bool VEC, bool ONE>
__global__ void __launch_bounds__(256) im2col_kernel(const T* __restrict__ y1, T* __restrict__ col, int B, int T1, int F1,
                                                      int C, int T2, int F2, const T* __restrict__ gamma,
                                                      const T* __restrict__ beta) {
  pdl_wait();
  pdl_trigger();
  const int64_t nchunks = (int64_t)B * T2 * F2 * 9;
  const int lane = threadIdx.x & 31;
  const int64_t warps_total = (int64_t)gridDim.x * (blockDim.x >> 5);
  constexpr int EPV = 16 / sizeof(T);            // elements per 16-byte vector
  AffineRegs<T> ar;
  if (VEC && ONE && gamma) ar.load(gamma, beta, lane * EPV);
  for (int64_t ch = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); ch < nchunks; ch += warps_total) {
    const int tap = (int)(ch % 9);
    const int64_t row = ch / 9;
    const int f2 = (int)(row % F2);
    const int t2 = (int)((row / F2) % T2);
    const int b = (int)(row / ((int64_t)F2 * T2));
    const int t = 2 * t2 + tap / 3 - 1, f = 2 * f2 + tap % 3 - 1;
    const bool inside = t >= 0 && t < T1 && f >= 0 && f < F1;
    T* dst = col + (row * 9 + tap) * C;
    const T* srcp = y1 + (((int64_t)b * T1 + (inside ? t : 0)) * F1 + (inside ? f : 0)) * C;
    if (VEC && ONE) {
      uint4 v = make_uint4(0, 0, 0, 0);
      if (inside) {
        v = __ldg(reinterpret_cast<const uint4*>(srcp + lane * EPV));
        if (gamma) v = affine_relu_vec(v, ar.g, ar.b);
      }
      *reinterpret_cast<uint4*>(dst + lane * EPV) = v;
    } else if (VEC) {
      for (int c = lane * EPV; c < C; c += 32 * EPV) {
        uint4 v = make_uint4(0, 0, 0, 0);
        if (inside) {
          v = __ldg(reinterpret_cast<const uint4*>(srcp + c));
          if (gamma) { AffineRegs<T> a2; a2.load(gamma, beta, c); v = affine_relu_vec(v, a2.g, a2.b); }
        }
        *reinterpret_cast<uint4*>(dst + c) = v;
      }
    } else {
      for (int c = lane; c < C; c += 32) {
        float x = inside ? to_f32(srcp[c]) : 0.f;
        if (inside && gamma) x = fmaxf(fmaf(x, to_f32(gamma[c]), to_f32(beta[c])), 0.f);
        dst[c] = from_f32<T>(x);
      }
    }
  }
}


// Production shape (one 16-byte vector per lane and row, i.e. C * sizeof(T) == 512): one warp per OUTPUT row, the
// position is decoded once and the 9 tap loads are all in flight before the 9 stores (the generic kernel spends more
// instructions on index arithmetic than on the copy).
template <typename T>
__global__ void __launch_bounds__(256) im2col_row_kernel(const T* __restrict__ y1, T* __restrict__ col, int B, int T1, int F1,
                                                          int T2, int F2, const T* __restrict__ gamma, const T* __restrict__ beta) {
  pdl_wait();
  pdl_trigger();
  constexpr int EPV = 16 / sizeof(T);
  constexpr int C = 32 * EPV;
  const int lane = threadIdx.x & 31;
  const int64_t nrows = (int64_t)B * T2 * F2;
  const int64_t warps_total = (int64_t)gridDim.x * (blockDim.x >> 5);
  AffineRegs<T> ar;
  if (gamma) ar.load(gamma, beta, lane * EPV);
  for (int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < nrows; row += warps_total) {
    const int f2 = (int)(row % F2);
    const int t2 = (int)((row / F2) % T2);
    const int b = (int)(row / ((int64_t)F2 * T2));
    const T* base = y1 + ((int64_t)b * T1 * F1) * C + lane * EPV;
    uint4 v[9];
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      const int t = 2 * t2 + tap / 3 - 1, f = 2 * f2 + tap % 3 - 1;
      const bool inside = t >= 0 && t < T1 && f >= 0 && f < F1;
      v[tap] = make_uint4(0, 0, 0, 0);
      if (inside) v[tap] = __ldg(reinterpret_cast<const uint4*>(base + ((int64_t)t * F1 + f) * C));
    }
    T* dst = col + row * 9 * C + lane * EPV;
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      const int t = 2 * t2 + tap / 3 - 1, f = 2 * f2 + tap % 3 - 1;
      const bool inside = t >= 0 && t < T1 && f >= 0 && f < F1;
      uint4 o = v[tap];
      if (gamma && inside) o = affine_relu_vec(o, ar.g, ar.b);
      *reinterpret_cast<uint4*>(dst + tap * C) = o;
    }
  }
}

}  // namespace

static int pick_grid(int64_t npos, int per_block, int cap) {
  int64_t g = (npos + per_block - 1) / per_block;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

static int conv1_fwd_launch(const float* src, const float* w, const float* b, const float* gamma, const float* beta, float eps,
                            void* y1, int y_dtype, int B, int T, int F, int Cin, int C, int use_ln, float* rstd_out, cudaStream_t s);

int conv1_ln_relu_fwd(const float* src, const float* w, const float* b, const float* gamma, const float* beta, float eps,
                      void* y1, int y_dtype, int B, int T, int F, int Cin, int C, int use_ln, cudaStream_t s) {
  return conv1_fwd_launch(src, w, b, gamma, beta, eps, y1, y_dtype, B, T, F, Cin, C, use_ln, nullptr, s);
}
// normalised-save forward: xhat = LN-normalised conv1 output (no gamma/beta/ReLU) + 1/sigma per position
int conv1_norm_fwd(const float* src, const float* w, const float* b, float eps, void* xhat, int dtype, float* rstd, int B, int T,
                   int F, int Cin, int C, cudaStream_t s) {
  if (ablate_mask() & ABL_CONV) return 0;
  B200ST_CHECK(rstd != nullptr, "conv1_norm_fwd needs the rstd buffer");
  return conv1_fwd_launch(src, w, b, nullptr, nullptr, eps, xhat, dtype, B, T, F, Cin, C, 0, rstd, s);
}

static int conv1_fwd_launch(const float* src, const float* w, const float* b, const float* gamma, const float* beta, float eps,
                            void* y1, int y_dtype, int B, int T, int F, int Cin, int C, int use_ln, float* rstd_out, cudaStream_t s) {
  B200ST_CHECK(C <= 512 && Cin >= 1 && Cin <= 4, "conv front-end supports C <= 512 and 1..4 input channels");
  const int T1 = (T + 1) / 2, F1 = (F + 1) / 2;
  const int64_t npos = (int64_t)B * T1 * F1;
  if (npos == 0) return 0;
  const int grid = pick_grid(npos, 8 * 4, 148 * 12);
  const bool vec = (C % 8 == 0) && ((reinterpret_cast<uintptr_t>(y1) & 15) == 0);
  if (vec && C == 256 && Cin == 1 && (use_ln || rstd_out) && ((reinterpret_cast<uintptr_t>(w) & 15) == 0) &&
      ((reinterpret_cast<uintptr_t>(b) & 15) == 0) && (rstd_out || (((reinterpret_cast<uintptr_t>(gamma) | reinterpret_cast<uintptr_t>(beta)) & 15) == 0))) {
    const int grid1 = pick_grid(npos, 8 * 16, 148 * 2);
    if (rstd_out) DISPATCH_DTYPE(y_dtype, TT, (launch_pdl(conv1_fwd_c256_kernel<TT, true>, grid1, 256, 0, s, src, w, b, gamma, beta, eps, (TT*)y1, rstd_out, B, T, F, T1, F1)));
    else DISPATCH_DTYPE(y_dtype, TT, (launch_pdl(conv1_fwd_c256_kernel<TT, false>, grid1, 256, 0, s, src, w, b, gamma, beta, eps, (TT*)y1, rstd_out, B, T, F, T1, F1)));
    ++g_kernel_launches;
    B200ST_LAUNCH_CHECK();
    return 0;
  }
  const size_t smem = (size_t)(9 * Cin + 1) * ((C + 255) & ~255) * sizeof(float);
  B200ST_CHECK(smem <= 48 * 1024, "conv1 filter does not fit the default shared memory");
#define FWD(VEC, CPL, CIN1)                                                                                             \
  DISPATCH_DTYPE(y_dtype, TT, (launch_pdl(conv1_fwd_kernel<TT, VEC, CPL, CIN1>, grid, 256, smem, s, src, w, b, gamma, beta, eps, (TT*)y1, \
                                                                                        B, T, F, Cin, C, T1, F1, use_ln, rstd_out)))
  if (vec && C <= 256) { if (Cin == 1) FWD(true, 8, true); else FWD(true, 8, false); }
  else if (vec) { if (Cin == 1) FWD(true, 16, true); else FWD(true, 16, false); }
  else if (C <= 256) { if (Cin == 1) FWD(false, 8, true); else FWD(false, 8, false); }
  else { if (Cin == 1) FWD(false, 16, true); else FWD(false, 16, false); }
#undef FWD
  ++g_kernel_launches;
  B200ST_LAUNCH_CHECK();
  return 0;
}

int conv1_bwd_fused(const float* src, const float* w, const float* b, const float* gamma, const float* beta, float eps,
                    const void* y1, const void* dcol, int dtype, void* dz1, void* col1, int K1p, float* db, float* dgamma,
                    float* dbeta, int B, int T, int F, int Cin, int C, int use_ln, cudaStream_t s) {
  B200ST_CHECK(C <= 512 && Cin >= 1 && Cin <= 4, "conv front-end supports C <= 512 and 1..4 input channels");
  B200ST_CHECK(K1p >= 9 * Cin && K1p <= 64, "bad col1 row stride");
  const int T1 = (T + 1) / 2, F1 = (F + 1) / 2, T2 = (T1 + 1) / 2, F2 = (F1 + 1) / 2;
  const int64_t npos = (int64_t)B * T1 * F1;
  if (npos == 0) return 0;
  const int grid = pick_grid(npos, 8 * 4, 148 * 8);
  const size_t smem = (size_t)(9 * Cin + 1 + 3) * ((C + 255) & ~255) * sizeof(float);
  B200ST_CHECK(smem <= 48 * 1024, "conv1 filter does not fit the default shared memory");
  const bool vec = (C % 8 == 0) && ((reinterpret_cast<uintptr_t>(y1) & 15) == 0) && ((reinterpret_cast<uintptr_t>(dcol) & 15) == 0) &&
                   ((reinterpret_cast<uintptr_t>(dz1) & 15) == 0);
#define BWD(VEC, CPL, CIN1)                                                                                             \
  DISPATCH_DTYPE(dtype, TT, (launch_pdl(conv1_bwd_fused_kernel<TT, VEC, CPL, CIN1>, grid, 256, smem, s,                           \
      src, w, b, gamma, beta, eps, (const TT*)y1, (const TT*)dcol, (TT*)dz1, (TT*)col1, K1p, db, dgamma, dbeta, B, T, F, Cin, C, \
      T1, F1, T2, F2, use_ln)))
  if (vec && C <= 256) { if (Cin == 1) BWD(true, 8, true); else BWD(true, 8, false); }
  else if (vec) { if (Cin == 1) BWD(true, 16, true); else BWD(true, 16, false); }
  else if (C <= 256) { if (Cin == 1) BWD(false, 8, true); else BWD(false, 8, false); }
  else { if (Cin == 1) BWD(false, 16, true); else BWD(false, 16, false); }
#undef BWD
  ++g_kernel_launches;
  B200ST_LAUNCH_CHECK();
  return 0;
}

// backward of the normalised-save front-end (C == 256, Cin == 1, 16-byte aligned rows)
int conv1_bwd_from_xhat(const float* src, const void* gamma, const void* beta, const void* xhat, const float* rstd,
                        const void* dcol, int dtype, void* dz1, void* col1, int K1p, float* db, float* dgamma, float* dbeta, int B,
                        int T, int F, int C, cudaStream_t s, int implicit_tiles) {
  if (ablate_mask() & ABL_CONV) return 0;
  B200ST_CHECK(C == 256 && K1p >= 9 && K1p <= 32, "conv1_bwd_from_xhat supports C == 256, Cin == 1");
  B200ST_CHECK(((reinterpret_cast<uintptr_t>(xhat) | reinterpret_cast<uintptr_t>(dcol) | reinterpret_cast<uintptr_t>(dz1) |
                 reinterpret_cast<uintptr_t>(gamma) | reinterpret_cast<uintptr_t>(beta)) & 15) == 0, "conv1 backward buffers must be 16-byte aligned");
  const int T1 = (T + 1) / 2, F1 = (F + 1) / 2, T2 = (T1 + 1) / 2, F2 = (F1 + 1) / 2;
  const int64_t npos = (int64_t)B * T1 * F1;
  if (npos == 0) return 0;
  const int grid = pick_grid(npos, 8 * 16, 148 * 2);
  const int tu = F2 > 0 && F2 <= 128 ? 128 / F2 : 1, ub = (T2 + tu - 1) / tu;
  if (implicit_tiles) {
    B200ST_CHECK(F2 <= 128, "implicit conv2 dgrad layout needs F2 <= 128");
    DISPATCH_DTYPE(dtype, TT, (launch_pdl(conv1_bwd_xhat_c256_kernel<TT, true>, grid, 256, 0, s, src, (const TT*)gamma, (const TT*)beta, (const TT*)xhat, rstd,
                                          (const TT*)dcol, (TT*)dz1, (TT*)col1, K1p, db, dgamma, dbeta, B, T, F, T1, F1, T2, F2, tu, ub)));
  } else {
    DISPATCH_DTYPE(dtype, TT, (launch_pdl(conv1_bwd_xhat_c256_kernel<TT, false>, grid, 256, 0, s, src, (const TT*)gamma, (const TT*)beta, (const TT*)xhat, rstd,
                                          (const TT*)dcol, (TT*)dz1, (TT*)col1, K1p, db, dgamma, dbeta, B, T, F, T1, F1, T2, F2, tu, ub)));
  }
  ++g_kernel_launches;
  B200ST_LAUNCH_CHECK();
  return 0;
}

int im2col_3x3s2(const void* y1, void* col, int dtype, int B, int T1, int F1, int C, cudaStream_t s) {
  return im2col_3x3s2_affine(y1, col, dtype, B, T1, F1, C, nullptr, nullptr, s);
}

// gamma/beta != null (in the activation dtype): col = im2col(relu(y1 * gamma + beta)) (y1 = normalised conv1 output)
int im2col_3x3s2_affine(const void* y1, void* col, int dtype, int B, int T1, int F1, int C, const void* gamma, const void* beta,
                        cudaStream_t s) {
  const int T2 = (T1 + 1) / 2, F2 = (F1 + 1) / 2;
  const int64_t nchunks = (int64_t)B * T2 * F2 * 9;
  if (nchunks == 0 || (ablate_mask() & ABL_CONV)) return 0;
  const int grid = pick_grid(nchunks, 8 * 8, 148 * 16);
  const int esz = dtype_size(dtype);
  const bool vec = ((C * esz) % 16 == 0) && ((reinterpret_cast<uintptr_t>(y1) & 15) == 0) && ((reinterpret_cast<uintptr_t>(col) & 15) == 0) &&
                   ((reinterpret_cast<uintptr_t>(gamma) & 15) == 0) && ((reinterpret_cast<uintptr_t>(beta) & 15) == 0);
  const bool one = vec && C * esz == 32 * 16;
  if (one) {
    const int grid_r = pick_grid(nchunks / 9, 8 * 4, 148 * 8);
    DISPATCH_DTYPE(dtype, TT, (launch_pdl(im2col_row_kernel<TT>, grid_r, 256, 0, s, (const TT*)y1, (TT*)col, B, T1, F1, T2, F2, (const TT*)gamma, (const TT*)beta)));
  }
  else if (vec) DISPATCH_DTYPE(dtype, TT, (launch_pdl(im2col_kernel<TT, true, false>, grid, 256, 0, s, (const TT*)y1, (TT*)col, B, T1, F1, C, T2, F2, (const TT*)gamma, (const TT*)beta)));
  else DISPATCH_DTYPE(dtype, TT, (launch_pdl(im2col_kernel<TT, false, false>, grid, 256, 0, s, (const TT*)y1, (TT*)col, B, T1, F1, C, T2, F2, (const TT*)gamma, (const TT*)beta)));
  ++g_kernel_launches;
  B200ST_LAUNCH_CHECK();
  return 0;
}

}  // namespace b200st
