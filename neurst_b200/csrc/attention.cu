// Fused multi-head attention for sm_100a (head dim 64): S = QK^T and O = PV on tcgen05 with fp32 accumulators in
// TMEM, operands staged by TMA, online softmax with one thread per (query row, half of a key block), additive key bias /
// causal mask exactly as the reference (multi_head_attention.py:145-160: logits + bias, FLOAT_MIN = -1e9), dropout on
// the probabilities (:207-208) from the precomputed keep-bit bitmap.  The [B,H,Tq,Tk] score / probability tensors never
// touch HBM: forward keeps only the per-row log-sum-exp; backward recomputes P from Q, K and the LSE (flash-attention
// style).
//
// forward : grid (q tiles of 128, H, B), 320 threads: warp 0 TMA producer, warp 1 MMA issuer, warps 2-9 softmax
//           (2 per TMEM lane quadrant); two CTAs per SM.
// backward: attn_bwd_prep_kernel (zero dQ, D = rowsum(dO * O)), then grid (kv blocks of 128, H, B), 320 threads: K_j / V_j
//           resident; loops over q tiles; dK_j, dV_j accumulate in TMEM, dQ tiles are reduced across kv blocks with fp32
//           vector RED into a scratch buffer (cast_rows_kernel -> bf16).
// Measurement history and ncu findings: profiles/r01_attention_notes.md.
#include "gemm.cuh"
#include "kernels.cuh"
#include "pdl.cuh"
#include "ptx.cuh"

namespace b200st {

int make_tma_map_16(const void* ptr, int dtype, uint64_t inner, uint64_t rows, int nb1, int nb2, int64_t ld, int64_t sb1, int64_t sb2,
                    uint32_t box_rows, CUtensorMap* out);

namespace {

constexpr int BQ = 128, BKV = 128, DH = 64;
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;
constexpr float kMaskMin = -1.0e9f;   // neurst/utils/compat.py:24
constexpr uint32_t kTile16K = 128 * 64 * 2;      // [128 rows x 64 bf16] swizzled tile

struct AttnParams {
  int B, H, Tq, Tk, Tkp;
  float alpha;                 // dh^-0.5
  const float* bias;           // [B, Tk] additive or null
  const int32_t* kv_len;       // [B] or null: keys >= kv_len[b] are padding (bias -1e9): their key blocks are skipped
  int causal;
  DropoutSpec drop;
  uint16_t* ctx; int64_t ctx_ld;          // [B*Tq, H*64], 16-bit type DT (bf16 or fp16)
  float* lse;                  // [B, H, Tq]  (natural log)
  // backward only
  const uint16_t* dctx; int64_t dctx_ld;
  float* dq_acc; int64_t dq_ld;           // fp32 [B*Tq, H*64] (zeroed by attn_bwd_prep_kernel)
  const float* dvec;                      // [B, H, Tq] rowsum(dO * O) (attn_bwd_prep_kernel)
  uint16_t* dk; int64_t dk_ld;            // [B*Tk, ...] view base already offset to the K columns; + h*64
  uint16_t* dv; int64_t dv_ld;
};

__device__ __forceinline__ float logit(const AttnParams& p, float s, const float* bias_row, int k, int q) {
  float x = s * p.alpha;
  if (bias_row) x += __ldg(bias_row + k);
  if (p.causal && k > q + (p.Tk - p.Tq)) x += kMaskMin;
  return x;
}

// byte offset of element (row, col) inside a [128 x 64*NCB] bf16 operand stored as NCB column blocks of
// [128 rows x 128 B] with the 128B swizzle (16-byte chunk index XOR (row & 7))
__device__ __forceinline__ uint32_t swz_off(int row, int col) {
  const int cb = col >> 6, c = col & 63;
  return (uint32_t)(cb * kTile16K + row * 128 + ((((c >> 3) ^ (row & 7)) & 7) << 4) + ((c & 7) << 1));
}

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
// every kernel below is templated on DT, the 16-bit operand type (BF16 or F16): it only selects the MMA operand format
// bits and the fp32 <-> 16-bit conversions
#define pack_bf16(a, b) pack2_16((a), (b), DT)

// ==============================================================================================================
// forward: 320 threads = TMA warp + MMA warp + 8 softmax warps (2 per TMEM lane quadrant, each owning 64 of the 128
// key columns of a block); ~100 KB smem and 256 TMEM columns so that two CTAs share an SM.  K is double-buffered (the
// next S = QK^T is issued right behind PV), V single-buffered (only needed after the next softmax).
// Element math is branch-free: the key bias (times log2 e, -inf beyond Tk) sits in a shared-memory table read with
// broadcast LDS.128, the logit is one FFMA, exp is one MUFU.EX2, the dropout scale is folded into the final 1/l.
// ==============================================================================================================
__device__ __forceinline__ void softmax_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// 64 keep-bits (keys k0 .. k0+63 of one query row) from the precomputed bitmap [B, H, Tq, Tkp] (the host refuses p > 0
// without one); bits of keys >= Tkp read as 1
__device__ __forceinline__ void load_keep64(const uint8_t* row_bits, int k0, int Tkp, uint32_t (&keep)[2]) {
  keep[0] = keep[1] = 0xffffffffu;
  if (!row_bits) return;
  if ((Tkp & 63) == 0) {                  // rows are 8-byte aligned in the bitmap: one 64-bit load
    if (k0 < Tkp) {
      const uint2 w = __ldg(reinterpret_cast<const uint2*>(row_bits + (k0 >> 3)));
      keep[0] = w.x; keep[1] = w.y;
    }
    return;
  }
  uint32_t byte[8];                       // unaligned rows: 8 byte loads (all issued before the first use)
  const uint8_t* bp = row_bits + (k0 >> 3);
#pragma unroll
  for (int g = 0; g < 8; ++g) byte[g] = (k0 + 8 * g < Tkp) ? (uint32_t)__ldg(bp + g) : 0xffu;
  keep[0] = byte[0] | (byte[1] << 8) | (byte[2] << 16) | (byte[3] << 24);
  keep[1] = byte[4] | (byte[5] << 8) | (byte[6] << 16) | (byte[7] << 24);
}
// keep-bit row of (b, h, query row) in the bitmap, or null when the row takes no dropout
__device__ __forceinline__ const uint8_t* keep_row(const AttnParams& p, bool row_ok, int64_t row_g) {
  return (p.drop.p > 0.f && row_ok) ? p.drop.bits + row_g * (p.Tkp >> 3) : nullptr;
}

template <bool CAUSAL, int DT>
__global__ void __launch_bounds__(320, 2)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                const __grid_constant__ CUtensorMap tmV, const AttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const int nblk_all = (p.Tk + BKV - 1) / BKV;       // sizes the bias table (launch-time shared memory)
  // key blocks that hold at least one non-padded key (kv_len is written at the very start of the step, many kernels back:
  // complete and visible before this kernel's predecessor could start, so it may be read ahead of griddepcontrol.wait)
  const int nblk = p.kv_len ? max(1, min(nblk_all, (__ldg(p.kv_len + blockIdx.z) + BKV - 1) / BKV)) : nblk_all;
  const uint32_t sQ = base;                          // 16 KB
  const uint32_t sK = sQ + kTile16K;                 // 2 x 16 KB
  const uint32_t sV = sK + 2 * kTile16K;             // 16 KB
  const uint32_t sP = sV + kTile16K;                 // 32 KB
  const uint32_t sX = sP + 2 * kTile16K;             // exchange: max [2][2][128] + sum [2][128] floats = 3 KB
  const uint32_t sB = sX + 3072;                     // key bias * log2(e), [nblk * 128] floats
  const uint32_t bars = sB + (uint32_t)nblk_all * 512u;
  const uint32_t q_full = bars, v_full = bars + 8, v_empty = bars + 16, s_full = bars + 24, s_empty = bars + 32,
                 p_full = bars + 40, p_empty = bars + 48, o_ready = bars + 56, tmem_slot = bars + 64;
  auto k_full = [&](int s2) { return bars + 72u + 8u * s2; };
  auto k_empty = [&](int s2) { return bars + 88u + 8u * s2; };
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - ptx::smem_u32(smem_raw)));
  float* xch = reinterpret_cast<float*>(smem_raw + (sX - ptx::smem_u32(smem_raw)));
  float* btab = reinterpret_cast<float*>(smem_raw + (sB - ptx::smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tmQ); ptx::prefetch_tensormap(&tmK); ptx::prefetch_tensormap(&tmV);
    ptx::mbar_init(q_full, 1);
    ptx::mbar_init(v_full, 1); ptx::mbar_init(v_empty, 1);
    for (int s2 = 0; s2 < 2; ++s2) { ptx::mbar_init(k_full(s2), 1); ptx::mbar_init(k_empty(s2), 1); }
    ptx::mbar_init(s_full, 1); ptx::mbar_init(s_empty, 8);
    ptx::mbar_init(p_full, 8); ptx::mbar_init(p_empty, 1);
    ptx::mbar_init(o_ready, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) { ptx::tmem_alloc_n<256>(tmem_slot); ptx::tmem_relinquish(); }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = *tmem_slot_ptr;
  pdl_wait();      // everything above (barriers, TMEM, descriptor prefetch) overlaps the previous kernel's tail
  pdl_trigger();
  const uint32_t tS = tmem;            // 128 columns
  const uint32_t tO = tmem + 128;      // 64 columns

  if (warp == 0) {
    if (lane == 0) {
      ptx::mbar_arrive_expect_tx(q_full, kTile16K);
      ptx::tma_load_4d(sQ, &tmQ, q_full, 0, qt * BQ, h, b);
      for (int j = 0; j < nblk; ++j) {
        const int s2 = j & 1;
        ptx::mbar_wait(k_empty(s2), (((uint32_t)j >> 1) & 1u) ^ 1u);
        ptx::mbar_arrive_expect_tx(k_full(s2), kTile16K);
        ptx::tma_load_4d(sK + s2 * kTile16K, &tmK, k_full(s2), 0, j * BKV, h, b);
        ptx::mbar_wait(v_empty, ((uint32_t)j & 1u) ^ 1u);
        ptx::mbar_arrive_expect_tx(v_full, kTile16K);
        ptx::tma_load_4d(sV, &tmV, v_full, 0, j * BKV, h, b);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr int kBf = DT == BF16 ? 1 : 0;
      const uint32_t idesc_s = ptx::make_idesc_16(BKV, 0, 0, kBf, kBf);    // S[128 x 128] = Q K^T, both K-major
      const uint32_t idesc_o = ptx::make_idesc_16(DH, 0, 1, kBf, kBf);     // O[128 x 64] += P V, V as MN-major B
      ptx::mbar_wait(q_full, 0);
      for (int j = 0; j < nblk; ++j) {
        const uint32_t ph = (uint32_t)j & 1u;
        const uint32_t k_s = sK + (uint32_t)(j & 1) * kTile16K;
        ptx::mbar_wait(k_full(j & 1), ((uint32_t)j >> 1) & 1u);
        ptx::mbar_wait(s_empty, ph ^ 1u);
        ptx::tc_fence_after();
#pragma unroll
        for (int k = 0; k < DH / 16; ++k)
          ptx::mma_f16_ss(tS, ptx::make_smem_desc_sw128(sQ + k * 32, 16, 1024), ptx::make_smem_desc_sw128(k_s + k * 32, 16, 1024),
                          idesc_s, k > 0 ? 1u : 0u);
        ptx::mma_commit(s_full);
        ptx::mma_commit(k_empty(j & 1));
        ptx::mbar_wait(v_full, ph);
        ptx::mbar_wait(p_full, ph);
        ptx::tc_fence_after();
#pragma unroll
        for (int k = 0; k < BKV / 16; ++k)
          ptx::mma_f16_ss(tO, ptx::make_smem_desc_sw128(sP + (k >> 2) * kTile16K + (k & 3) * 32, 16, 1024),
                          ptx::make_smem_desc_sw128(sV + k * 2048, 8192, 1024), idesc_o, (j > 0 || k > 0) ? 1u : 0u);
        ptx::mma_commit(v_empty);
        ptx::mma_commit(p_empty);
        ptx::mma_commit(o_ready);
      }
    }
  } else {
    // ---------------- softmax warps: thread = (query row, half of the key columns) ----------------
    const int quad = warp & 3;
    const int half = (warp - 2) >> 2;
    const int row = quad * 32 + lane;
    const int q = qt * BQ + row;
    const int64_t row_g = ((int64_t)b * p.H + h) * p.Tq + q;
    const uint32_t lane_addr = (uint32_t)(quad * 32) << 16;
    const float a2 = p.alpha * kLog2e;
    const int qlim = q + (p.Tk - p.Tq);               // causal: keys k > qlim get the additive FLOAT_MIN
    const float cmask = kMaskMin * kLog2e;
    {
      const float* bias_row = p.bias ? p.bias + (int64_t)b * p.Tk : nullptr;
#pragma unroll 1          // unrolled, this one-off loop costs the causal instantiation extra spill slots
      for (int k = threadIdx.x - 64; k < nblk * BKV; k += 256)
        btab[k] = (k < p.Tk) ? (bias_row ? __ldg(bias_row + k) * kLog2e : 0.f) : -INFINITY;
      softmax_bar();
    }
    float m = -INFINITY, l = 0.f;      // running row max (log2 domain, shared by both halves) and this half's partial sum
    uint32_t keep[2], keep_next[2];
    const uint8_t* krow = keep_row(p, q < p.Tq, row_g);
    load_keep64(krow, half * 64, p.Tkp, keep);
    for (int j = 0; j < nblk; ++j) {
      const uint32_t ph = (uint32_t)j & 1u;
      const int kbase = j * BKV + half * 64;          // first key of this thread's 64 columns
      ptx::mbar_wait(s_full, ph);
      ptx::tc_fence_after();
      // logits (log2 domain) of this thread's 64 columns, kept in registers
      uint32_t r[64];
      {
        uint32_t (&r0)[32] = *reinterpret_cast<uint32_t (*)[32]>(&r[0]);
        uint32_t (&r1)[32] = *reinterpret_cast<uint32_t (*)[32]>(&r[32]);
        __syncwarp();
        ptx::tmem_ld_32x32b_x32(tS + lane_addr + half * 64, r0);
        ptx::tmem_ld_32x32b_x32(tS + lane_addr + half * 64 + 32, r1);
        if (j + 1 < nblk) load_keep64(krow, kbase + BKV, p.Tkp, keep_next);   // in flight during the math
        __syncwarp();
        ptx::tmem_ld_wait();
      }
      float bmax = -INFINITY;
      const float4* bt4 = reinterpret_cast<const float4*>(btab + kbase);
#pragma unroll
      for (int i4 = 0; i4 < 16; ++i4) {
        const float4 bb = bt4[i4];
        float x0 = fmaf(__uint_as_float(r[4 * i4 + 0]), a2, bb.x), x1 = fmaf(__uint_as_float(r[4 * i4 + 1]), a2, bb.y);
        float x2 = fmaf(__uint_as_float(r[4 * i4 + 2]), a2, bb.z), x3 = fmaf(__uint_as_float(r[4 * i4 + 3]), a2, bb.w);
        if (CAUSAL) {
          const int k = kbase + 4 * i4;
          x0 = (k + 0 > qlim) ? x0 + cmask : x0; x1 = (k + 1 > qlim) ? x1 + cmask : x1;
          x2 = (k + 2 > qlim) ? x2 + cmask : x2; x3 = (k + 3 > qlim) ? x3 + cmask : x3;
        }
        r[4 * i4 + 0] = __float_as_uint(x0); r[4 * i4 + 1] = __float_as_uint(x1);
        r[4 * i4 + 2] = __float_as_uint(x2); r[4 * i4 + 3] = __float_as_uint(x3);
        bmax = fmaxf(fmaxf(bmax, fmaxf(x0, x1)), fmaxf(x2, x3));
      }
      xch[(ph * 2 + half) * 128 + row] = bmax;
      softmax_bar();
      bmax = fmaxf(bmax, xch[(ph * 2 + (half ^ 1)) * 128 + row]);
      const float m_new = fmaxf(m, bmax);
      const float corr = ex2_approx(m - m_new);       // 0 on the first block (m = -inf)
      // probabilities -> bf16 P tile in shared memory (A operand of the PV product); dropout scale applied at the end
      ptx::mbar_wait(p_empty, ph ^ 1u);
      float bsum = 0.f;
#pragma unroll
      for (int g8 = 0; g8 < 8; ++g8) {
        const uint32_t kb = keep[g8 >> 2] >> (8 * (g8 & 3));
        float pv[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float pr = ex2_approx(__uint_as_float(r[g8 * 8 + i]) - m_new);
          bsum += pr;
          pv[i] = ((kb >> i) & 1u) ? pr : 0.f;
        }
        st_shared_v4(sP + swz_off(row, half * 64 + g8 * 8), pack_bf16(pv[0], pv[1]), pack_bf16(pv[2], pv[3]), pack_bf16(pv[4], pv[5]),
                     pack_bf16(pv[6], pv[7]));
      }
      l = l * corr + bsum;
      m = m_new;
      keep[0] = keep_next[0]; keep[1] = keep_next[1];
      // rescale this half's 32 output columns (after the logits registers are dead) once the previous PV product has landed
      if (j > 0) {
        ptx::mbar_wait(o_ready, ph ^ 1u);
        ptx::tc_fence_after();
        uint32_t ro[32];
        __syncwarp();
        ptx::tmem_ld_32x32b_x32(tO + lane_addr + half * 32, ro);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) ro[i] = __float_as_uint(__uint_as_float(ro[i]) * corr);
        ptx::tmem_st_32x32b_x32(tO + lane_addr + half * 32, ro);
        ptx::tmem_st_wait();
      }
      ptx::fence_proxy_async_smem();       // P (generic-proxy writes) -> visible to the tensor-core (async) proxy
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) { ptx::mbar_arrive(s_empty); ptx::mbar_arrive(p_full); }
    }
    // ---- epilogue: O * scale / l -> ctx, LSE ----
    float* xsum = xch + 512;
    xsum[half * 128 + row] = l;
    softmax_bar();
    l += xsum[(half ^ 1) * 128 + row];
    ptx::mbar_wait(o_ready, (uint32_t)(nblk - 1) & 1u);
    ptx::tc_fence_after();
    const float inv_l = ((p.drop.p > 0.f) ? p.drop.scale : 1.0f) / l;
    uint16_t* dst = p.ctx + ((int64_t)b * p.Tq + q) * p.ctx_ld + h * DH + half * 32;
    {
      uint32_t ro[32];
      __syncwarp();
      ptx::tmem_ld_32x32b_x32(tO + lane_addr + half * 32, ro);
      ptx::tmem_ld_wait();
      if (q < p.Tq) {
#pragma unroll
        for (int i = 0; i < 32; i += 8) {
          uint4 pk;
          pk.x = pack_bf16(__uint_as_float(ro[i]) * inv_l, __uint_as_float(ro[i + 1]) * inv_l);
          pk.y = pack_bf16(__uint_as_float(ro[i + 2]) * inv_l, __uint_as_float(ro[i + 3]) * inv_l);
          pk.z = pack_bf16(__uint_as_float(ro[i + 4]) * inv_l, __uint_as_float(ro[i + 5]) * inv_l);
          pk.w = pack_bf16(__uint_as_float(ro[i + 6]) * inv_l, __uint_as_float(ro[i + 7]) * inv_l);
          *reinterpret_cast<uint4*>(dst + i) = pk;
        }
      }
    }
    if (half == 0 && q < p.Tq && p.lse) p.lse[row_g] = m * kLn2 + logf(l);
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) { ptx::tc_fence_after(); ptx::tmem_dealloc(tmem, 256); }
}

// ==============================================================================================================
// backward: one CTA per (kv block, head, batch)
// ==============================================================================================================
__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

constexpr int kBwdThreads = 64 + 512;     // TMA warp + MMA warp + 16 compute warps (4 per TMEM lane quadrant, 32 key columns each)
__device__ __forceinline__ void bwd_bar() { asm volatile("bar.sync 1, 512;" ::: "memory"); }

template <bool CAUSAL, int DT>
__global__ void __launch_bounds__(kBwdThreads, 1)
attn_bwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmdO, const AttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sK = base;                          // 16 KB
  const uint32_t sV = sK + kTile16K;                 // 16 KB
  const uint32_t sQ = sV + kTile16K;                 // 2 x 16 KB
  const uint32_t sdO = sQ + 2 * kTile16K;            // 2 x 16 KB
  const uint32_t sP = sdO + 2 * kTile16K;            // 32 KB  [128 q x 128 keys] as 2 column blocks
  const uint32_t sdS = sP + 2 * kTile16K;            // 32 KB
  const uint32_t bars = sdS + 2 * kTile16K;
  const uint32_t kv_full = bars;
  auto qdo_full = [&](int s) { return bars + 8u * (1 + s); };
  auto qdo_empty = [&](int s) { return bars + 8u * (3 + s); };
  const uint32_t sdp_full = bars + 8u * 5;
  const uint32_t pds_full = bars + 8u * 6;
  const uint32_t dq_full = bars + 8u * 7;
  const uint32_t dq_empty = bars + 8u * 8;
  const uint32_t tmem_slot = bars + 8u * 9;
  const uint32_t sB = bars + 128;                    // key bias * log2(e) of this kv block, 128 floats
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - ptx::smem_u32(smem_raw)));
  float* btab = reinterpret_cast<float*>(smem_raw + (sB - ptx::smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int jb = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int nq = (p.Tq + BQ - 1) / BQ;
  if (p.kv_len && jb > 0 && jb * BKV >= __ldg(p.kv_len + b)) {
    // every key of this block is padding: P = 0 exactly, so dK = dV = 0 and the block adds nothing to dQ
    pdl_wait();
    pdl_trigger();
    for (int i = threadIdx.x; i < BKV * (DH / 8); i += blockDim.x) {
      const int r = i / (DH / 8), c8 = (i % (DH / 8)) * 8, kk = jb * BKV + r;
      if (kk < p.Tk) {
        *reinterpret_cast<uint4*>(p.dv + ((int64_t)b * p.Tk + kk) * p.dv_ld + h * DH + c8) = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4*>(p.dk + ((int64_t)b * p.Tk + kk) * p.dk_ld + h * DH + c8) = make_uint4(0, 0, 0, 0);
      }
    }
    return;
  }

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tmQ); ptx::prefetch_tensormap(&tmK); ptx::prefetch_tensormap(&tmV); ptx::prefetch_tensormap(&tmdO);
    ptx::mbar_init(kv_full, 1);
    for (int s = 0; s < 2; ++s) { ptx::mbar_init(qdo_full(s), 1); ptx::mbar_init(qdo_empty(s), 1); }
    ptx::mbar_init(sdp_full, 1); ptx::mbar_init(pds_full, 16);
    ptx::mbar_init(dq_full, 1); ptx::mbar_init(dq_empty, 16);
    ptx::fence_mbar_init();
  }
  if (warp == 1) { ptx::tmem_alloc_n<512>(tmem_slot); ptx::tmem_relinquish(); }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = *tmem_slot_ptr;
  pdl_wait();      // everything above (barriers, TMEM, descriptor prefetch) overlaps the previous kernel's tail
  pdl_trigger();
  const uint32_t tS = tmem, tdP = tmem + 128, tdV = tmem + 256, tdK = tmem + 320, tdQ = tmem + 384;

  if (warp == 0) {
    if (lane == 0) {
      ptx::mbar_arrive_expect_tx(kv_full, 2 * kTile16K);
      ptx::tma_load_4d(sK, &tmK, kv_full, 0, jb * BKV, h, b);
      ptx::tma_load_4d(sV, &tmV, kv_full, 0, jb * BKV, h, b);
      for (int i = 0; i < nq; ++i) {
        const int st = i & 1;
        ptx::mbar_wait(qdo_empty(st), (((uint32_t)i >> 1) & 1u) ^ 1u);
        ptx::mbar_arrive_expect_tx(qdo_full(st), 2 * kTile16K);
        ptx::tma_load_4d(sQ + st * kTile16K, &tmQ, qdo_full(st), 0, i * BQ, h, b);
        ptx::tma_load_4d(sdO + st * kTile16K, &tmdO, qdo_full(st), 0, i * BQ, h, b);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr int kBf = DT == BF16 ? 1 : 0;
      const uint32_t idesc_s = ptx::make_idesc_16(BKV, 0, 0, kBf, kBf);    // [128q x 128k], A,B K-major
      const uint32_t idesc_kv = ptx::make_idesc_16(DH, 1, 1, kBf, kBf);    // dV/dK [128k x 64] = X^T Y : A, B MN-major
      const uint32_t idesc_q = ptx::make_idesc_16(DH, 0, 1, kBf, kBf);     // dQ [128q x 64] = dS K : A K-major, B MN-major
      ptx::mbar_wait(kv_full, 0);
      for (int i = 0; i < nq; ++i) {
        const int st = i & 1;
        const uint32_t q_s = sQ + st * kTile16K, do_s = sdO + st * kTile16K;
        ptx::mbar_wait(qdo_full(st), ((uint32_t)i >> 1) & 1u);
        ptx::tc_fence_after();
        // S = Q K^T ; dP = dO V^T    (S / dP TMEM is free: the compute warps finished tile i-1 before pds_full(i-1))
#pragma unroll
        for (int k = 0; k < DH / 16; ++k) {
          ptx::mma_f16_ss(tS, ptx::make_smem_desc_sw128(q_s + k * 32, 16, 1024), ptx::make_smem_desc_sw128(sK + k * 32, 16, 1024),
                          idesc_s, k > 0 ? 1u : 0u);
        }
#pragma unroll
        for (int k = 0; k < DH / 16; ++k) {
          ptx::mma_f16_ss(tdP, ptx::make_smem_desc_sw128(do_s + k * 32, 16, 1024), ptx::make_smem_desc_sw128(sV + k * 32, 16, 1024),
                          idesc_s, k > 0 ? 1u : 0u);
        }
        ptx::mma_commit(sdp_full);
        ptx::mbar_wait(pds_full, (uint32_t)i & 1u);
        ptx::mbar_wait(dq_empty, ((uint32_t)i & 1u) ^ 1u);
        ptx::tc_fence_after();
#pragma unroll
        for (int k = 0; k < BQ / 16; ++k) {       // contraction over the 128 query rows
          const uint64_t a_p = ptx::make_smem_desc_sw128(sP + k * 2048, 16384, 1024);
          const uint64_t a_ds = ptx::make_smem_desc_sw128(sdS + k * 2048, 16384, 1024);
          const uint64_t b_do = ptx::make_smem_desc_sw128(do_s + k * 2048, 8192, 1024);
          const uint64_t b_q = ptx::make_smem_desc_sw128(q_s + k * 2048, 8192, 1024);
          ptx::mma_f16_ss(tdV, a_p, b_do, idesc_kv, (i > 0 || k > 0) ? 1u : 0u);
          ptx::mma_f16_ss(tdK, a_ds, b_q, idesc_kv, (i > 0 || k > 0) ? 1u : 0u);
        }
#pragma unroll
        for (int k = 0; k < BKV / 16; ++k) {      // contraction over the 128 keys
          const uint64_t a_ds = ptx::make_smem_desc_sw128(sdS + (k >> 2) * kTile16K + (k & 3) * 32, 16, 1024);
          const uint64_t b_k = ptx::make_smem_desc_sw128(sK + k * 2048, 8192, 1024);
          ptx::mma_f16_ss(tdQ, a_ds, b_k, idesc_q, k > 0 ? 1u : 0u);
        }
        ptx::mma_commit(qdo_empty(st));
        ptx::mma_commit(dq_full);
      }
    }
  } else {
    // 16 compute warps: thread = (row of the tile, quarter of the key columns) — four warps per scheduler hide the TMEM /
    // shared-memory latencies of the per-pair softmax recompute; no cross-warp reductions are needed in backward.
    // Branch-free element math as in the forward kernel (bias table in smem, one FFMA + one MUFU per probability); the
    // dropout scale is folded into dS (FFMA) and into the dV epilogue.
    const int quad = warp & 3;
    const int quarter = (warp - 2) >> 2;             // 0..3: key columns [32 * quarter, +32)
    const int row = quad * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(quad * 32) << 16;
    const float a2 = p.alpha * kLog2e;
    const float cmask = kMaskMin * kLog2e;
    const float dscale = (p.drop.p > 0.f) ? p.drop.scale : 1.0f;
    {
      const float* bias_row = p.bias ? p.bias + (int64_t)b * p.Tk : nullptr;
      const int t = threadIdx.x - 64;
      if (t < BKV) {
        const int k = jb * BKV + t;
        btab[t] = (k < p.Tk) ? (bias_row ? __ldg(bias_row + k) * kLog2e : 0.f) : -INFINITY;
      }
      bwd_bar();
    }
    const int c0 = quarter * 32;
    const int kbase64 = jb * BKV + (quarter >> 1) * 64;      // keep-bits come as aligned 64-key words
    const float4* bt4 = reinterpret_cast<const float4*>(btab + c0);
    // per-tile row scalars (D = rowsum(dO * O), LSE in the log2 domain: +inf on padding rows => P = 0, keep bits) are
    // prefetched one tile ahead so their global-load latency hides behind the previous tile's math
    // A row whose every key carries the -1e9 bias (a length-0 sequence): in fp32 each logit the forward pass visited
    // equals that bias (s is absorbed), so its softmax is uniform over those keys, but the stored LSE (-1e9) has absorbed
    // log(l) as well and exp2(x - lse2) gives 1 for every key.  Such rows scale P by 1 / (keys the forward pass visited).
    const int kv_vis = p.kv_len ? min(p.Tk, max(1, (__ldg(p.kv_len + b) + BKV - 1) / BKV) * BKV) : p.Tk;
    auto load_row = [&](int i, float& Dq, float& lse2, float& prs, uint32_t& keep) {
      const int q = i * BQ + row;
      const bool qv = q < p.Tq;
      const int64_t row_g = ((int64_t)b * p.H + h) * p.Tq + q;
      Dq = qv ? __ldg(p.dvec + row_g) : 0.f;
      lse2 = qv ? __ldg(p.lse + row_g) * kLog2e : INFINITY;
      prs = lse2 < 0.5f * cmask ? 1.f / (float)(CAUSAL ? min(kv_vis, q + (p.Tk - p.Tq) + 1) : kv_vis) : 1.f;
      uint32_t k2[2];
      load_keep64(keep_row(p, qv, row_g), kbase64, p.Tkp, k2);
      keep = k2[quarter & 1];
    };
    float Dq, lse2, prs, Dq_n = 0.f, lse2_n = INFINITY, prs_n = 1.f;
    uint32_t keep, keep_n = 0xffffffffu;
    load_row(0, Dq, lse2, prs, keep);
    for (int i = 0; i < nq; ++i) {
      const int q = i * BQ + row;
      const bool qv = q < p.Tq;
      const int qlim = q + (p.Tk - p.Tq);
      if (i + 1 < nq) load_row(i + 1, Dq_n, lse2_n, prs_n, keep_n);
      __syncwarp();
      ptx::mbar_wait(sdp_full, (uint32_t)i & 1u);
      ptx::tc_fence_after();
      {
        uint32_t rs[32], rp[32];
        __syncwarp();
        ptx::tmem_ld_32x32b_x32(tS + lane_addr + c0, rs);
        ptx::tmem_ld_32x32b_x32(tdP + lane_addr + c0, rp);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int g8 = 0; g8 < 4; ++g8) {
          const float4 b0 = bt4[g8 * 2], b1 = bt4[g8 * 2 + 1];
          const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
          const uint32_t kb = keep >> (8 * g8);
          float pd[8], ds[8];
#pragma unroll
          for (int t = 0; t < 8; ++t) {
            float x = fmaf(__uint_as_float(rs[g8 * 8 + t]), a2, bb[t]);
            if (CAUSAL) x = (jb * BKV + c0 + g8 * 8 + t > qlim) ? x + cmask : x;
            const float pr = ex2_approx(x - lse2) * prs;
            const bool kp = (kb >> t) & 1u;
            const float dpv = kp ? __uint_as_float(rp[g8 * 8 + t]) : 0.f;
            pd[t] = kp ? pr : 0.f;
            ds[t] = pr * fmaf(dpv, dscale, -Dq);
          }
          const uint32_t off = swz_off(row, c0 + g8 * 8);
          st_shared_v4(sP + off, pack_bf16(pd[0], pd[1]), pack_bf16(pd[2], pd[3]), pack_bf16(pd[4], pd[5]), pack_bf16(pd[6], pd[7]));
          st_shared_v4(sdS + off, pack_bf16(ds[0], ds[1]), pack_bf16(ds[2], ds[3]), pack_bf16(ds[4], ds[5]), pack_bf16(ds[6], ds[7]));
        }
      }
      ptx::fence_proxy_async_smem();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(pds_full);
      // ---- dQ tile (this warp's 16 columns) -> fp32 reduction across kv blocks ----
      ptx::mbar_wait(dq_full, (uint32_t)i & 1u);
      ptx::tc_fence_after();
      float* dq_row = p.dq_acc + ((int64_t)b * p.Tq + q) * p.dq_ld + h * DH + quarter * 16;
      {
        uint32_t r[16];
        __syncwarp();
        ptx::tmem_ld_32x32b_x16(tdQ + lane_addr + quarter * 16, r);
        ptx::tmem_ld_wait();
        if (qv) {
#pragma unroll
          for (int t = 0; t < 16; t += 4)
            red_add_v4(dq_row + t, __uint_as_float(r[t]) * p.alpha, __uint_as_float(r[t + 1]) * p.alpha,
                       __uint_as_float(r[t + 2]) * p.alpha, __uint_as_float(r[t + 3]) * p.alpha);
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(dq_empty);
      Dq = Dq_n; lse2 = lse2_n; prs = prs_n; keep = keep_n;
    }
    // ---- dV, dK of this kv block (all MMAs retired: the last dq_full commit covers them); 16 columns per warp ----
    const int kk = jb * BKV + row;
    uint16_t* dv_row = p.dv + ((int64_t)b * p.Tk + kk) * p.dv_ld + h * DH + quarter * 16;
    uint16_t* dk_row = p.dk + ((int64_t)b * p.Tk + kk) * p.dk_ld + h * DH + quarter * 16;
    {
      uint32_t rv[16], rk[16];
      __syncwarp();
      ptx::tmem_ld_32x32b_x16(tdV + lane_addr + quarter * 16, rv);
      ptx::tmem_ld_32x32b_x16(tdK + lane_addr + quarter * 16, rk);
      ptx::tmem_ld_wait();
      if (kk < p.Tk) {
#pragma unroll
        for (int t = 0; t < 16; t += 8) {
          uint4 a, c;
          a.x = pack_bf16(__uint_as_float(rv[t]) * dscale, __uint_as_float(rv[t + 1]) * dscale);
          a.y = pack_bf16(__uint_as_float(rv[t + 2]) * dscale, __uint_as_float(rv[t + 3]) * dscale);
          a.z = pack_bf16(__uint_as_float(rv[t + 4]) * dscale, __uint_as_float(rv[t + 5]) * dscale);
          a.w = pack_bf16(__uint_as_float(rv[t + 6]) * dscale, __uint_as_float(rv[t + 7]) * dscale);
          c.x = pack_bf16(__uint_as_float(rk[t]) * p.alpha, __uint_as_float(rk[t + 1]) * p.alpha);
          c.y = pack_bf16(__uint_as_float(rk[t + 2]) * p.alpha, __uint_as_float(rk[t + 3]) * p.alpha);
          c.z = pack_bf16(__uint_as_float(rk[t + 4]) * p.alpha, __uint_as_float(rk[t + 5]) * p.alpha);
          c.w = pack_bf16(__uint_as_float(rk[t + 6]) * p.alpha, __uint_as_float(rk[t + 7]) * p.alpha);
          *reinterpret_cast<uint4*>(dv_row + t) = a;
          *reinterpret_cast<uint4*>(dk_row + t) = c;
        }
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) { ptx::tc_fence_after(); ptx::tmem_dealloc(tmem, 512); }
}

constexpr size_t kBwdSmem = 1024 + (size_t)(2 + 2 + 2 + 2 + 2) * kTile16K + 128 + 512 + 64;

// One warp per (b, q) row: zero the fp32 dQ accumulator row and compute D[b,h,q] = sum_c dO[b,q,h,c] * O[b,q,h,c].
template <int DT>
__global__ void attn_bwd_prep_kernel(const uint16_t* __restrict__ o, int64_t o_ld, const uint16_t* __restrict__ dout,
                                     int64_t do_ld, float* __restrict__ dq_acc, float* __restrict__ dvec, int B, int H, int Tq) {
  pdl_wait();
  pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int64_t rows = (int64_t)B * Tq;
  const int chunks = H * (DH / 8);                  // 16-byte chunks per row; 8 chunks per head
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += (int64_t)gridDim.x * (blockDim.x >> 5)) {
    const int b = (int)(r / Tq), q = (int)(r % Tq);
    for (int c0 = 0; c0 < chunks; c0 += 32) {
      const int c = c0 + lane;
      float part = 0.f;
      if (c < chunks) {
        const uint4 a = __ldg(reinterpret_cast<const uint4*>(o + r * o_ld + 8 * c)), d = __ldg(reinterpret_cast<const uint4*>(dout + r * do_ld + 8 * c));
        const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, dw[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const float2 x = unpack2_16(aw[t], DT), y = unpack2_16(dw[t], DT);
          part = fmaf(x.x, y.x, fmaf(x.y, y.y, part));
        }
        float4* z = reinterpret_cast<float4*>(dq_acc + r * (int64_t)H * DH + 8 * c);
        z[0] = make_float4(0.f, 0.f, 0.f, 0.f); z[1] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      part += __shfl_xor_sync(0xffffffffu, part, 1);
      part += __shfl_xor_sync(0xffffffffu, part, 2);
      part += __shfl_xor_sync(0xffffffffu, part, 4);
      if (c < chunks && (lane & 7) == 0) dvec[((int64_t)b * H + (c >> 3)) * Tq + q] = part;
    }
  }
}

// dst(bf16)[r, 0..cols) = src(fp32)[r, 0..cols)   (dq scratch -> the q columns of the fused dqkv buffer)
template <int DT>
__global__ void cast_rows_kernel(const float* __restrict__ src, int64_t ld_src, uint16_t* __restrict__ dst, int64_t ld_dst,
                                 int64_t rows, int cols) {
  pdl_wait();
  pdl_trigger();
  const int64_t n8 = rows * (cols / 8);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / (cols / 8);
    const int c = (int)(i % (cols / 8)) * 8;
    const float4 a = *reinterpret_cast<const float4*>(src + r * ld_src + c), b2 = *reinterpret_cast<const float4*>(src + r * ld_src + c + 4);
    uint4 pk;
    pk.x = pack_bf16(a.x, a.y); pk.y = pack_bf16(a.z, a.w); pk.z = pack_bf16(b2.x, b2.y); pk.w = pack_bf16(b2.z, b2.w);
    *reinterpret_cast<uint4*>(dst + r * ld_dst + c) = pk;
  }
}

constexpr size_t kFwdSmemFixed = 1024 + (size_t)(1 + 2 + 1 + 2) * kTile16K + 3072 + 8 * 14 + 64;   // + 512 B per kv block (bias table)

}  // namespace

// q/k/v: bf16 views [B*T, ld] with head h at columns [h*64, h*64+64)
int attention_fwd_fused(int dt, const void* q, int64_t q_ld, const void* k, int64_t k_ld, const void* v, int64_t v_ld, int B, int H,
                        int Tq, int Tk, const float* bias, int causal, DropoutSpec drop, void* ctx, int64_t ctx_ld, float* lse,
                        cudaStream_t s, const int32_t* kv_len) {
  if (ablate_mask() & ABL_ATTN_FWD) return 0;
  B200ST_CHECK(Tq > 0 && Tk > 0 && B > 0 && H > 0, "empty attention");
  B200ST_CHECK(B <= 65535 && H <= 65535, "attention grid too large");
  B200ST_CHECK(is16(dt), "fused attention needs a 16-bit operand type");
  if (drop.p > 0.f) B200ST_CHECK(drop.bits != nullptr, "fused attention needs precomputed dropout bits");
  CUtensorMap tq, tk, tv;
  B200ST_TRY(make_tma_map_16(q, dt, DH, Tq, H, B, q_ld, DH, (int64_t)Tq * q_ld, BQ, &tq));
  B200ST_TRY(make_tma_map_16(k, dt, DH, Tk, H, B, k_ld, DH, (int64_t)Tk * k_ld, BKV, &tk));
  B200ST_TRY(make_tma_map_16(v, dt, DH, Tk, H, B, v_ld, DH, (int64_t)Tk * v_ld, BKV, &tv));
  AttnParams p{};
  p.B = B; p.H = H; p.Tq = Tq; p.Tk = Tk; p.Tkp = (Tk + 7) / 8 * 8;
  p.alpha = 0.125f;                     // 64^-0.5 (multi_head_attention.py:203)
  p.bias = bias; p.causal = causal; p.drop = drop; p.kv_len = kv_len;
  p.ctx = reinterpret_cast<uint16_t*>(ctx); p.ctx_ld = ctx_ld; p.lse = lse;
  B200ST_CHECK((reinterpret_cast<uintptr_t>(ctx) & 15) == 0 && ctx_ld % 8 == 0, "ctx must be 16-byte aligned");
  const size_t smem = kFwdSmemFixed + (size_t)((Tk + BKV - 1) / BKV) * 512;
  B200ST_CHECK(smem <= 227 * 1024, "fused attention: Tk too large for the shared-memory bias table");
  auto kern = causal ? (dt == F16 ? attn_fwd_kernel<true, F16> : attn_fwd_kernel<true, BF16>)
                     : (dt == F16 ? attn_fwd_kernel<false, F16> : attn_fwd_kernel<false, BF16>);
  static size_t attr[4] = {0, 0, 0, 0};
  const int ai = (causal ? 1 : 0) + (dt == F16 ? 2 : 0);
  if (smem > attr[ai]) {
    B200ST_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr[ai] = smem;
  }
  dim3 grid((Tq + BQ - 1) / BQ, H, B);
  launch_pdl(kern, grid, 320, smem, s, tq, tk, tv, p);
  tc_count_launch();
  B200ST_LAUNCH_CHECK();
  return 0;
}


// dq_scratch: fp32 [B*Tq, H*64] (overwritten).  dq/dk/dv: bf16 views like q/k/v.  lse / ctx from the forward pass.
int attention_bwd_fused(int dt, const void* q, int64_t q_ld, const void* k, int64_t k_ld, const void* v, int64_t v_ld, const void* ctx,
                        int64_t ctx_ld, const void* dctx, int64_t dctx_ld, const float* lse, int B, int H, int Tq, int Tk,
                        const float* bias, int causal, DropoutSpec drop, float* dq_scratch, void* dq, int64_t dq_ld, void* dk,
                        int64_t dk_ld, void* dv, int64_t dv_ld, cudaStream_t s, const int32_t* kv_len) {
  if (ablate_mask() & ABL_ATTN_BWD) return 0;
  B200ST_CHECK(Tq > 0 && Tk > 0 && B > 0 && H > 0 && B <= 65535 && H <= 65535, "bad attention shape");
  B200ST_CHECK(is16(dt), "fused attention needs a 16-bit operand type");
  if (drop.p > 0.f) B200ST_CHECK(drop.bits != nullptr, "fused attention needs precomputed dropout bits");
  CUtensorMap tq, tk, tv, tdo;
  B200ST_TRY(make_tma_map_16(q, dt, DH, Tq, H, B, q_ld, DH, (int64_t)Tq * q_ld, BQ, &tq));
  B200ST_TRY(make_tma_map_16(k, dt, DH, Tk, H, B, k_ld, DH, (int64_t)Tk * k_ld, BKV, &tk));
  B200ST_TRY(make_tma_map_16(v, dt, DH, Tk, H, B, v_ld, DH, (int64_t)Tk * v_ld, BKV, &tv));
  B200ST_TRY(make_tma_map_16(dctx, dt, DH, Tq, H, B, dctx_ld, DH, (int64_t)Tq * dctx_ld, BQ, &tdo));
  AttnParams p{};
  p.B = B; p.H = H; p.Tq = Tq; p.Tk = Tk; p.Tkp = (Tk + 7) / 8 * 8;
  p.alpha = 0.125f;
  p.bias = bias; p.causal = causal; p.drop = drop; p.kv_len = kv_len;
  p.ctx = reinterpret_cast<uint16_t*>(const_cast<void*>(ctx)); p.ctx_ld = ctx_ld;
  p.lse = const_cast<float*>(lse);
  p.dctx = reinterpret_cast<const uint16_t*>(dctx); p.dctx_ld = dctx_ld;
  p.dq_acc = dq_scratch; p.dq_ld = (int64_t)H * DH;
  p.dk = reinterpret_cast<uint16_t*>(dk); p.dk_ld = dk_ld;
  p.dv = reinterpret_cast<uint16_t*>(dv); p.dv_ld = dv_ld;
  B200ST_CHECK(((reinterpret_cast<uintptr_t>(dk) | reinterpret_cast<uintptr_t>(dv) | reinterpret_cast<uintptr_t>(dq) |
                 reinterpret_cast<uintptr_t>(dq_scratch)) & 15) == 0, "attention gradient buffers must be 16-byte aligned");
  static bool attr = false;
  if (!attr) {
    B200ST_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<false, BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBwdSmem));
    B200ST_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<true, BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBwdSmem));
    B200ST_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<false, F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBwdSmem));
    B200ST_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<true, F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBwdSmem));
    attr = true;
  }
  const int64_t rows = (int64_t)B * Tq;
  float* dvec = dq_scratch + rows * H * DH;
  p.dvec = dvec;
  B200ST_CHECK((reinterpret_cast<uintptr_t>(ctx) & 15) == 0 && (reinterpret_cast<uintptr_t>(dctx) & 15) == 0 && ctx_ld % 8 == 0 &&
               dctx_ld % 8 == 0, "attention ctx / dctx must be 16-byte aligned");
  {
    int64_t gp = (rows + 7) / 8;
    if (gp > 148 * 8) gp = 148 * 8;
    launch_pdl(dt == F16 ? attn_bwd_prep_kernel<F16> : attn_bwd_prep_kernel<BF16>, (int)gp, 256, 0, s,
               reinterpret_cast<const uint16_t*>(ctx), ctx_ld, reinterpret_cast<const uint16_t*>(dctx), dctx_ld, dq_scratch, dvec, B, H, Tq);
    g_kernel_launches += 1;
    B200ST_LAUNCH_CHECK();
  }
  dim3 grid((Tk + BKV - 1) / BKV, H, B);
  auto kern = causal ? (dt == F16 ? attn_bwd_kernel<true, F16> : attn_bwd_kernel<true, BF16>)
                     : (dt == F16 ? attn_bwd_kernel<false, F16> : attn_bwd_kernel<false, BF16>);
  launch_pdl(kern, grid, kBwdThreads, kBwdSmem, s, tq, tk, tv, tdo, p);
  B200ST_LAUNCH_CHECK();
  const int64_t n8 = rows * (H * DH / 8);
  int64_t g = (n8 + 255) / 256;
  if (g > 148 * 8) g = 148 * 8;
  launch_pdl(dt == F16 ? cast_rows_kernel<F16> : cast_rows_kernel<BF16>, (int)g, 256, 0, s, dq_scratch, (int64_t)H * DH,
             reinterpret_cast<uint16_t*>(dq), dq_ld, rows, H * DH);
  tc_count_launch();
  g_kernel_launches += 1;
  B200ST_LAUNCH_CHECK();
  return 0;
}

}  // namespace b200st
