// tcgen05 / TMEM / TMA bf16 GEMM for sm_100a.
//
// Persistent, warp-specialised kernel (one CTA per SM, 320 threads):
//   warp 0      : TMA producer  (cp.async.bulk.tensor -> 128B-swizzled smem ring, mbarrier complete_tx)
//   warp 1      : TMEM allocator + single-thread tcgen05.mma issuer (fp32 accumulators in TMEM, 2 stages)
//   warps 2..9  : epilogue (tcgen05.ld 32x32b -> registers -> fused epilogue -> 128B-swizzled smem staging box -> TMA
//                 store, or TMA reduce-add for split-K / accumulate), 2 warps per TMEM lane quadrant
// Tile: 128 x BN x 64 (BN in {64,128,256}); operands may be K-major or MN-major (wgrad / PV products),
// batched through 4-D tensor maps; optional split-K.  Every launch is a programmatic dependent launch (pdl.cuh).
// Measurements behind the design choices: profiles/r01_gemm_notes.md.
//
// Replaces the cuBLAS calls behind tf.einsum / Dense / Conv2D at the reference sites listed in
// SURVEY.md §2.3 (K3,K4,K8,K9,K10,K11,K13,K15), e.g. neurst/layers/common_layers.py:270,276-288.
#include "gemm.cuh"
#include "pdl.cuh"
#include "ptx.cuh"

#include <mutex>
#include <unordered_map>
#include <vector>
#include <cstring>
#include <cstdlib>

namespace b200st {

namespace {

constexpr int BM = 128;
constexpr int BK = 64;                  // 64 bf16 = 128 B = one swizzle row
constexpr int kThreads = 320;              // TMA warp + MMA warp + 8 epilogue warps
constexpr int kSmemLimit = 232448;      // 227 KB
constexpr uint32_t kABytes = BM * BK * 2;
constexpr uint32_t kStagingBytes = 8 * 2 * 4096;   // per epilogue warp: two 32-row x 128-byte boxes (ping-pong)

struct TcParams {
  int M, N, K;
  int nb1, nb2;
  int m_tiles, n_tiles, splitk, kb_total, kb_per_split;
  int64_t num_tiles;
  int stages;
  uint32_t a_lbo, a_sbo, b_lbo, b_sbo;   // descriptor byte offsets
  uint32_t a_kstep, b_kstep;             // smem byte advance per UMMA_K=16
  uint32_t idesc;
  void* C;
  int c_dtype;
  int64_t ldc, c_sb1, c_sb2;
  GemmEpilogue epi;
  int atomic;
  int use_tma_store;    // epilogue writes C through per-warp smem boxes + TMA store (aligned, non-ragged tiles)
  int c_reduce;         // C += (atomic / accumulate): cp.reduce.async.bulk.tensor .add
  // implicit transposed-convolution A operand (conv2 data gradient, see gemm_conv2_dgrad): A tile = a [conv_tu x conv_v]
  // patch of positions x 64 channels of dY[B, T2, F2, C], shifted by the tap; k-block kb = (tap, 64-channel chunk)
  int conv;             // 0 = off
  int conv_ub;          // row tiles per utterance
  int conv_tu;          // time rows per tile
  int conv_kpc;         // k-blocks per tap (C / 64)
  int conv_dt[4], conv_df[4], conv_wrow[4];   // per tap: time / frequency shift into dY, first row of the tap in the weight matrix
  uint32_t conv_a_bytes;                      // bytes one A box delivers (64 ch x conv_v x conv_tu x 2)
};

struct TileCoord { int b2, b1, m_blk, n_blk, split; };

__device__ __forceinline__ TileCoord decode_tile(const TcParams& p, int64_t tile) {
  TileCoord t;
  t.split = (int)(tile % p.splitk); tile /= p.splitk;
  t.n_blk = (int)(tile % p.n_tiles); tile /= p.n_tiles;
  t.m_blk = (int)(tile % p.m_tiles); tile /= p.m_tiles;
  t.b1 = (int)(tile % p.nb1);
  t.b2 = (int)(tile / p.nb1);
  return t;
}

enum OutMode : int { OUT_BF16 = 0, OUT_F32 = 1, OUT_ATOMIC = 2, OUT_F16 = 3 };
__host__ __device__ constexpr bool out_is16(int o) { return o == OUT_BF16 || o == OUT_F16; }

// Cold path (ragged N, unaligned rows, on-the-fly Philox): compact, not unrolled, out of line — keeps the kernel's hot
// code small enough for the instruction cache (the first version inlined every variant: 17 k SASS instructions).
__device__ __noinline__ void epilogue_chunk_general(const TcParams& p, const float* acc, int m, int n0, int64_t bidx,
                                                    int64_t boff_c, int64_t boff_mask, int64_t boff_res) {
  const GemmEpilogue& ep = p.epi;
#pragma unroll 1
  for (int j = 0; j < 32; ++j) {
    const int n = n0 + j;
    if (n >= p.N) break;
    const uint64_t e_idx = (uint64_t)((bidx * p.M + m) * (int64_t)p.N + n);
    const float v = gemm_epilogue_value(ep, acc[j], m, n, boff_mask, boff_res, e_idx);
    const int64_t idx = boff_c + (int64_t)m * p.ldc + n;
    if (p.atomic) atomicAdd(reinterpret_cast<float*>(p.C) + idx, v);
    else if (p.c_dtype == F32) reinterpret_cast<float*>(p.C)[idx] = ep.accumulate ? reinterpret_cast<float*>(p.C)[idx] + v : v;
    else store_from_f32(p.C, p.c_dtype, idx, v);
  }
}

// Per-row epilogue context: everything that does not change between the 32-column chunks of one tile row.
struct EpiRow {
  const float* bias;    // at n_base or null
  const char* mask;     // at n_base or null
  const float* res;     // at n_base or null
  const uint8_t* bits;  // dropout keep-bits at element (row, n_base) or null
  bool row_ok;          // m < M (rows beyond M are clipped by the TMA store; their loads are skipped)
};

// alpha / bias / relu / relu-mask / dropout bits / residual on one 32-column chunk (thread = one output row)
template <int OUT>
__device__ __forceinline__ void epilogue_math(const TcParams& p, const uint32_t (&r)[32], const EpiRow& e, int co, float relu_floor,
                                              float (&v)[32]) {
  const GemmEpilogue& ep = p.epi;
  if (e.bias) {
    const float4* b4 = reinterpret_cast<const float4*>(e.bias + co);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 bb = __ldg(b4 + j);
      v[4 * j + 0] = fmaxf(fmaf(__uint_as_float(r[4 * j + 0]), ep.alpha, bb.x), relu_floor);
      v[4 * j + 1] = fmaxf(fmaf(__uint_as_float(r[4 * j + 1]), ep.alpha, bb.y), relu_floor);
      v[4 * j + 2] = fmaxf(fmaf(__uint_as_float(r[4 * j + 2]), ep.alpha, bb.z), relu_floor);
      v[4 * j + 3] = fmaxf(fmaf(__uint_as_float(r[4 * j + 3]), ep.alpha, bb.w), relu_floor);
    }
  } else if (ep.relu || ep.alpha != 1.f) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = fmaxf(__uint_as_float(r[j]) * ep.alpha, relu_floor);
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
  }
  if (OUT == OUT_ATOMIC || !e.row_ok) return;
  if (e.mask) {
    if (ep.mask_dtype != F32) {
      // 16-bit mask source (bf16 or fp16): "> 0" <=> sign bit clear and magnitude bits non-zero, format-independent
      const uint4* mp = reinterpret_cast<const uint4*>(e.mask + co * 2);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint4 pk = __ldg(mp + j);
        const uint32_t w[4] = {pk.x, pk.y, pk.z, pk.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint32_t lo = w[i] & 0xffffu, hi = w[i] >> 16;
          if (!(lo != 0u && lo < 0x8000u)) v[8 * j + 2 * i] = 0.f;
          if (!(hi != 0u && hi < 0x8000u)) v[8 * j + 2 * i + 1] = 0.f;
        }
      }
    } else {
      const float4* mp = reinterpret_cast<const float4*>(e.mask + co * 4);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 f = __ldg(mp + j);
        if (!(f.x > 0.f)) v[4 * j] = 0.f;
        if (!(f.y > 0.f)) v[4 * j + 1] = 0.f;
        if (!(f.z > 0.f)) v[4 * j + 2] = 0.f;
        if (!(f.w > 0.f)) v[4 * j + 3] = 0.f;
      }
    }
  }
  if (e.bits) {
    const uint32_t keep32 = __ldg(reinterpret_cast<const uint32_t*>(e.bits + (co >> 3)));
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = ((keep32 >> j) & 1u) ? v[j] * ep.drop.scale : 0.f;
  }
  if (e.res) {
    const float4* rp = reinterpret_cast<const float4*>(e.res + co);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 rr = __ldg(rp + j);
      v[4 * j + 0] += rr.x; v[4 * j + 1] += rr.y; v[4 * j + 2] += rr.z; v[4 * j + 3] += rr.w;
    }
  }
}

// Writes this lane's row of a 32-column chunk into the warp's staging box ([32 rows x 128 B], 128B-swizzled, i.e. the
// layout the C tensor map expects): bf16 = half a row (64 B) at chunk-in-box `cb`, fp32 = the whole 128-byte row.
template <int OUT>
__device__ __forceinline__ void stage_chunk(uint32_t buf, int lane, int cb, const float (&v)[32]) {
  const uint32_t row = buf + (uint32_t)lane * 128u;
  const uint32_t sw = (uint32_t)(lane & 7);
  if (out_is16(OUT)) {
    constexpr int dt = OUT == OUT_F16 ? F16 : BF16;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t h0 = pack2_16(v[8 * j], v[8 * j + 1], dt), h1 = pack2_16(v[8 * j + 2], v[8 * j + 3], dt);
      const uint32_t h2 = pack2_16(v[8 * j + 4], v[8 * j + 5], dt), h3 = pack2_16(v[8 * j + 6], v[8 * j + 7], dt);
      const uint32_t addr = row + ((((uint32_t)(cb * 4 + j)) ^ sw) << 4);
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(h0), "r"(h1), "r"(h2), "r"(h3) : "memory");
    }
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t addr = row + ((((uint32_t)j) ^ sw) << 4);
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(__float_as_uint(v[4 * j])), "r"(__float_as_uint(v[4 * j + 1])),
                   "r"(__float_as_uint(v[4 * j + 2])), "r"(__float_as_uint(v[4 * j + 3]))
                   : "memory");
    }
  }
}

template <int BN, bool A_MN, bool B_MN, int OUT>
__global__ void __launch_bounds__(kThreads, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmC, const TcParams p) {
  extern __shared__ uint8_t smem_raw[];
  constexpr uint32_t kBBytes = BN * BK * 2;
  constexpr uint32_t kStageBytes = kABytes + kBBytes;
  constexpr uint32_t kTmemCols = (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;

  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const int stages = p.stages;
  const uint32_t stage_out = smem_base + stages * kStageBytes;   // 8 warps x 2 x 4 KB epilogue staging boxes
  const uint32_t bar_base = stage_out + kStagingBytes;           // 8-byte barriers
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (stages + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * stages + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * stages + 2 + s); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * stages + 4);
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - ptx::smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tmA);
    ptx::prefetch_tensormap(&tmB);
    if (p.use_tma_store) ptx::prefetch_tensormap(&tmC);
    for (int s = 0; s < stages; ++s) { ptx::mbar_init(full_bar(s), 1); ptx::mbar_init(empty_bar(s), 1); }
    for (int s = 0; s < 2; ++s) { ptx::mbar_init(tfull_bar(s), 1); ptx::mbar_init(tempty_bar(s), 8); }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, kTmemCols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  pdl_wait();      // everything above (barriers, TMEM, descriptor prefetch) overlaps the previous kernel's tail
  pdl_trigger();

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        const TileCoord t = decode_tile(p, tile);
        const int kb0 = t.split * p.kb_per_split;
        const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb) {
          ptx::mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t sa = smem_base + stage * kStageBytes;
          const uint32_t sb = sa + kABytes;
          if constexpr (!A_MN && !B_MN) {
            if (p.conv) {
              const int tap = kb / p.conv_kpc, c0 = (kb - tap * p.conv_kpc) * BK;
              ptx::mbar_arrive_expect_tx(full_bar(stage), p.conv_a_bytes + kBBytes);
              ptx::tma_load_4d(sa, &tmA, full_bar(stage), c0, p.conv_df[tap], (t.m_blk % p.conv_ub) * p.conv_tu + p.conv_dt[tap],
                               t.m_blk / p.conv_ub);
              ptx::tma_load_4d(sb, &tmB, full_bar(stage), c0, p.conv_wrow[tap] + t.n_blk * BN, 0, 0);
              if (++stage == stages) { stage = 0; phase ^= 1u; }
              continue;
            }
          }
          ptx::mbar_arrive_expect_tx(full_bar(stage), kStageBytes);
          if (A_MN) {
#pragma unroll
            for (int c = 0; c < BM / 64; ++c)
              ptx::tma_load_4d(sa + c * (64 * BK * 2), &tmA, full_bar(stage), t.m_blk * BM + c * 64, kb * BK, t.b1, t.b2);
          } else {
            ptx::tma_load_4d(sa, &tmA, full_bar(stage), kb * BK, t.m_blk * BM, t.b1, t.b2);
          }
          if (B_MN) {
#pragma unroll
            for (int c = 0; c < BN / 64; ++c)
              ptx::tma_load_4d(sb + c * (64 * BK * 2), &tmB, full_bar(stage), t.n_blk * BN + c * 64, kb * BK, t.b1, t.b2);
          } else {
            ptx::tma_load_4d(sb, &tmB, full_bar(stage), kb * BK, t.n_blk * BN, t.b1, t.b2);
          }
          if (++stage == stages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        const TileCoord t = decode_tile(p, tile);
        const int kb0 = t.split * p.kb_per_split;
        const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        ptx::mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        ptx::tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
        for (int kb = kb0; kb < kb1; ++kb) {
          ptx::mbar_wait(full_bar(stage), phase);
          ptx::tc_fence_after();
          const uint32_t sa = smem_base + stage * kStageBytes;
          const uint32_t sb = sa + kABytes;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint64_t da = ptx::make_smem_desc_sw128(sa + k * p.a_kstep, p.a_lbo, p.a_sbo);
            const uint64_t db = ptx::make_smem_desc_sw128(sb + k * p.b_kstep, p.b_lbo, p.b_sbo);
            ptx::mma_f16_ss(tmem_d, da, db, p.idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          ptx::mma_commit(empty_bar(stage));     // frees the smem slot when these MMAs retire
          if (++stage == stages) { stage = 0; phase ^= 1u; }
        }
        ptx::mma_commit(tfull_bar(acc));         // accumulator ready for the epilogue warps
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else {
    // ===================== epilogue warps (2..9) =====================
    // warp w may only touch TMEM lanes [32*(w%4), +32); the two warps sharing a quadrant split the columns.
    const int quad = warp & 3;
    const int half = (warp - 2) >> 2;              // 0 or 1
    const int row_in_tile = quad * 32 + lane;
    int acc = 0; uint32_t acc_phase = 0;
    const GemmEpilogue& ep = p.epi;
    const float relu_floor = ep.relu ? 0.f : -INFINITY;
    for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      const TileCoord t = decode_tile(p, tile);
      ptx::mbar_wait(tfull_bar(acc), acc_phase);
      ptx::tc_fence_after();
      const int m = t.m_blk * BM + row_in_tile;
      const int64_t bidx = (int64_t)t.b2 * p.nb1 + t.b1;
      const int64_t boff_c = (int64_t)t.b2 * p.c_sb2 + (int64_t)t.b1 * p.c_sb1;
      const int64_t boff_mask = (int64_t)t.b2 * ep.mask_sb2 + (int64_t)t.b1 * ep.mask_sb1;
      const int64_t boff_res = (int64_t)t.b2 * ep.res_sb2 + (int64_t)t.b1 * ep.res_sb1;
      const uint32_t taddr_row = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN);
      const int n_base = t.n_blk * BN;
      const int c_begin = half * (BN / 2);
      const bool tile_tma = p.use_tma_store && (n_base + BN <= p.N);     // warp-uniform
      if (tile_tma) {
        // ---- TMA-store path: TMEM -> registers -> fused math -> swizzled smem box -> cp.async.bulk.tensor store ----
        EpiRow er;
        er.row_ok = m < p.M;
        er.bias = ep.bias ? ep.bias + n_base : nullptr;
        er.mask = (ep.mask_src && er.row_ok) ? reinterpret_cast<const char*>(ep.mask_src) +
                                                   (size_t)(boff_mask + (int64_t)m * ep.mask_ld + n_base) * (ep.mask_dtype == F32 ? 4 : 2)
                                             : nullptr;
        er.res = (ep.residual && er.row_ok) ? ep.residual + boff_res + (int64_t)m * ep.res_ld + n_base : nullptr;
        er.bits = (ep.drop.p > 0.f && er.row_ok) ? ep.drop.bits + ((uint64_t)((bidx * p.M + m) * (int64_t)p.N + n_base) >> 3) : nullptr;
        constexpr int kColsPerBox = out_is16(OUT) ? 64 : 32;
        // BN = 64 with bf16 output: one 64-column box per quadrant, written by the half-0 warp alone
        constexpr bool kSingle = (BN / 2 < kColsPerBox);
        constexpr int kBoxes = kSingle ? 1 : BN / 2 / kColsPerBox;
        const int c_begin_box = kSingle ? 0 : c_begin;
        const int n_boxes = (kSingle && half == 1) ? 0 : kBoxes;
        const uint32_t my_stage = stage_out + (uint32_t)(warp - 2) * 8192u;
#pragma unroll 1
        for (int bx = 0; bx < n_boxes; ++bx) {
          const uint32_t buf = my_stage + (uint32_t)(bx & 1) * 4096u;
          if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");   // the box written 2 iterations ago is drained
          __syncwarp();
#pragma unroll
          for (int cb = 0; cb < kColsPerBox / 32; ++cb) {
            const int co = c_begin_box + bx * kColsPerBox + cb * 32;
            uint32_t r[32];
            ptx::tmem_ld_32x32b_x32(taddr_row + (uint32_t)co, r);
            ptx::tmem_ld_wait();
            float v[32];
            epilogue_math<OUT>(p, r, er, co, relu_floor, v);
            stage_chunk<OUT>(buf, lane, cb, v);
          }
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            const int cn = n_base + c_begin_box + bx * kColsPerBox, cm = t.m_blk * BM + quad * 32;
            if (p.c_reduce)
              asm volatile("cp.reduce.async.bulk.tensor.4d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                           ::"l"(&tmC), "r"(buf), "r"(cn), "r"(cm), "r"(t.b1), "r"(t.b2) : "memory");
            else
              asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                           ::"l"(&tmC), "r"(buf), "r"(cn), "r"(cm), "r"(t.b1), "r"(t.b2) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        }
      } else {
        // ---- general path (ragged N, unaligned operands, on-the-fly Philox): per-element, compact ----
#pragma unroll 1
        for (int co = c_begin; co < c_begin + BN / 2; co += 32) {
          if (n_base + co >= p.N) break;
          uint32_t r[32];
          __syncwarp();
          ptx::tmem_ld_32x32b_x32(taddr_row + (uint32_t)co, r);
          ptx::tmem_ld_wait();
          if (m < p.M) {
            float acc_v[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) acc_v[j] = __uint_as_float(r[j]);
            epilogue_chunk_general(p, acc_v, m, n_base + co, bidx, boff_c, boff_mask, boff_res);
          }
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(tempty_bar(acc));
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // all of this warp's TMA stores are complete
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}


// =============================================================================================================
// Grouped weight-gradient GEMM: up to kMaxGroup products  dW_g[K_in, N_out] += X_g^T dY_g  of one backward block in ONE
// persistent launch (TF autodiff of the Dense / einsum sites of a sublayer: neurst/layers/common_layers.py:270-288,
// multi_head_attention.py:145-215).  Each product alone has 2..16 output tiles and needs split-K over the B*T rows to fill
// 148 SMs, i.e. every CTA reduce-adds a full 128 x 256 fp32 tile for a handful of k-blocks of MMA work and every launch pays
// the fixed ~6 us; together the products of a block give one wave of work units with k-ranges 3-4x longer (tools/ablate_step.py:
// the weight-gradient launches cost 0.84 ms of the 6.46 ms cfg-2 step although they run on the side stream).
// Same pipeline as tc_gemm_kernel<256, true, true, OUT_ATOMIC>; a work unit = (product, m tile, n tile, k split).
// =============================================================================================================
constexpr int kMaxGroup = 4;
struct TcGroupProb {
  CUtensorMap ta, tb, tc;
  int m_tiles, n_tiles, splitk, kb_total, kb_per_split, tile_begin;
  float alpha;
  int pad_;
};
struct TcGroup {
  TcGroupProb prob[kMaxGroup];
  int n, num_tiles, stages;
  uint32_t idesc;
};
struct GroupTile { int gi, m_blk, n_blk, kb0, kb1; };
__device__ __forceinline__ GroupTile group_tile(const TcGroup& g, int tile) {
  GroupTile t;
  t.gi = 0;
#pragma unroll
  for (int i = 1; i < kMaxGroup; ++i)
    if (i < g.n && tile >= g.prob[i].tile_begin) t.gi = i;
  const TcGroupProb& q = g.prob[t.gi];
  int local = tile - q.tile_begin;
  const int split = local % q.splitk; local /= q.splitk;
  t.n_blk = local % q.n_tiles;
  t.m_blk = local / q.n_tiles;
  t.kb0 = split * q.kb_per_split;
  t.kb1 = min(q.kb_total, t.kb0 + q.kb_per_split);
  return t;
}

__global__ void __launch_bounds__(kThreads, 1) tc_wgrad_group_kernel(const __grid_constant__ TcGroup grp) {
  extern __shared__ uint8_t smem_raw[];
  constexpr int BN = 256;
  constexpr uint32_t kBBytes = BN * BK * 2;
  constexpr uint32_t kStageBytes = kABytes + kBBytes;
  constexpr uint32_t kMnLbo = 64u * BK * 2, kMnSbo = 1024u, kMnKstep = 16u * 128u;

  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const int stages = grp.stages;
  const uint32_t stage_out = smem_base + stages * kStageBytes;
  const uint32_t bar_base = stage_out + kStagingBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (stages + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * stages + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * stages + 2 + s); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * stages + 4);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - ptx::smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    for (int i = 0; i < grp.n; ++i) {
      ptx::prefetch_tensormap(&grp.prob[i].ta);
      ptx::prefetch_tensormap(&grp.prob[i].tb);
      ptx::prefetch_tensormap(&grp.prob[i].tc);
    }
    for (int s = 0; s < stages; ++s) { ptx::mbar_init(full_bar(s), 1); ptx::mbar_init(empty_bar(s), 1); }
    for (int s = 0; s < 2; ++s) { ptx::mbar_init(tfull_bar(s), 1); ptx::mbar_init(tempty_bar(s), 8); }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, 512);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  pdl_wait();
  pdl_trigger();

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < grp.num_tiles; tile += gridDim.x) {
        const GroupTile t = group_tile(grp, tile);
        const CUtensorMap* ma = &grp.prob[t.gi].ta;
        const CUtensorMap* mb = &grp.prob[t.gi].tb;
        for (int kb = t.kb0; kb < t.kb1; ++kb) {
          ptx::mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t sa = smem_base + stage * kStageBytes;
          const uint32_t sb = sa + kABytes;
          ptx::mbar_arrive_expect_tx(full_bar(stage), kStageBytes);
#pragma unroll
          for (int c = 0; c < BM / 64; ++c)
            ptx::tma_load_4d(sa + c * (64 * BK * 2), ma, full_bar(stage), t.m_blk * BM + c * 64, kb * BK, 0, 0);
#pragma unroll
          for (int c = 0; c < BN / 64; ++c)
            ptx::tma_load_4d(sb + c * (64 * BK * 2), mb, full_bar(stage), t.n_blk * BN + c * 64, kb * BK, 0, 0);
          if (++stage == stages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int tile = blockIdx.x; tile < grp.num_tiles; tile += gridDim.x) {
        const GroupTile t = group_tile(grp, tile);
        ptx::mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        ptx::tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
        for (int kb = t.kb0; kb < t.kb1; ++kb) {
          ptx::mbar_wait(full_bar(stage), phase);
          ptx::tc_fence_after();
          const uint32_t sa = smem_base + stage * kStageBytes;
          const uint32_t sb = sa + kABytes;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint64_t da = ptx::make_smem_desc_sw128(sa + k * kMnKstep, kMnLbo, kMnSbo);
            const uint64_t db = ptx::make_smem_desc_sw128(sb + k * kMnKstep, kMnLbo, kMnSbo);
            ptx::mma_f16_ss(tmem_d, da, db, grp.idesc, (kb > t.kb0 || k > 0) ? 1u : 0u);
          }
          ptx::mma_commit(empty_bar(stage));
          if (++stage == stages) { stage = 0; phase ^= 1u; }
        }
        ptx::mma_commit(tfull_bar(acc));
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else {
    const int quad = warp & 3;
    const int half = (warp - 2) >> 2;
    int acc = 0; uint32_t acc_phase = 0;
    const uint32_t my_stage = stage_out + (uint32_t)(warp - 2) * 8192u;
    for (int tile = blockIdx.x; tile < grp.num_tiles; tile += gridDim.x) {
      const GroupTile t = group_tile(grp, tile);
      const CUtensorMap* mc = &grp.prob[t.gi].tc;
      const float alpha = grp.prob[t.gi].alpha;
      ptx::mbar_wait(tfull_bar(acc), acc_phase);
      ptx::tc_fence_after();
      const uint32_t taddr_row = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN);
      const int c_begin = half * (BN / 2);
#pragma unroll 1
      for (int bx = 0; bx < BN / 2 / 32; ++bx) {
        const uint32_t buf = my_stage + (uint32_t)(bx & 1) * 4096u;
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        __syncwarp();
        const int co = c_begin + bx * 32;
        uint32_t r[32];
        ptx::tmem_ld_32x32b_x32(taddr_row + (uint32_t)co, r);
        ptx::tmem_ld_wait();
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]) * alpha;
        stage_chunk<OUT_ATOMIC>(buf, lane, 0, v);
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          const int cn = t.n_blk * BN + co, cm = t.m_blk * BM + quad * 32;
          asm volatile("cp.reduce.async.bulk.tensor.4d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                       ::"l"(mc), "r"(buf), "r"(cn), "r"(cm), "r"(0), "r"(0) : "memory");
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(tempty_bar(acc));
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 512);
  }
}


// =============================================================================================================
// Fused Transformer FFN forward (SURVEY K11):  x_out += dropout_post( dropout_ffn(relu(X W1 + b1)) W2 + b2 )
//   neurst/layers/common_layers.py:145-160 (TransformerFFN) inside the pre-norm wrapper (:73-85); X = LN(x_in) (16-bit),
//   x_out is pre-initialised with the residual x_in by the LayerNorm kernel.
// One CTA = (128-row tile, slice of the hidden dimension).  The X tile (128 x d, d <= 256) stays in shared memory; the hidden
// activations of a 128-column chunk are produced in TMEM (GEMM1), turned into the 16-bit A operand of GEMM2 in shared
// memory by the epilogue warps (bias, ReLU, dropout) — and TMA-stored to HBM only because the backward pass needs them —
// while GEMM2 accumulates the [128 x d] output tile in TMEM across all chunks.  Only the weights stream (L2 -> smem):
// 2 x 64 KB per chunk for 2 x 1024 MMA cycles, vs 4 x that for the two unfused GEMMs, and the [M, ffn] hidden tensor is
// never read back.  Slices of the hidden dimension reduce into x_out with fp32 TMA reduce-add (dropout is a mask: linear).
//   warp 0: TMA producer (X once, then weight stages in consumption order)     warp 1: MMA issuer
//   warps 2-9: epilogue (hidden chunk: TMEM -> regs -> smem operand + TMA store; final: TMEM -> regs -> smem -> reduce-add)
//   TMEM: [0,256) output accumulator, [256,384) / [384,512) hidden accumulators (double buffered)
//   smem: X 64 KB | H 2 x 32 KB | weight ring 3 x 32 KB (reused as the output staging boxes at the end)
// =============================================================================================================
struct MlpParams {
  int M, d, ffn;
  int chunks_per_cta;          // 128-column hidden chunks per CTA
  int splits;                  // hidden slices (gridDim.x = m_tiles * splits)
  const float* b1; const float* b2;
  DropoutSpec drop_ffn, drop_post;
  uint32_t idesc_g1, idesc_g2;
  // backward (dgrad chain) variant: hidden epilogue = alpha * acc masked by (mask_src > 0), no bias / ReLU / dropout bits
  int relu;
  float alpha;
  const void* mask_src; int64_t mask_ld;
  int* tickets;                // deterministic mode: [m_tiles] zero-initialised; slice s adds after slices < s (self-resetting)
};
constexpr int kMlpStages = 3;
constexpr uint32_t kMlpStageBytes = 32768;
constexpr uint32_t kMlpXBytes = 65536, kMlpHBytes = 32768;
constexpr size_t kMlpSmem = 1024 + kMlpXBytes + 2 * kMlpHBytes + kMlpStages * kMlpStageBytes + 256 + 1024;

// B_MN: weights as MN-major B operands (forward: W1 [d, ffn], W2 [ffn, d] in the TF [in, out] layout) or K-major (backward:
// the same arrays read transposed: G1 uses W2 rows = hidden units, G2 uses W1 rows = model dims)
template <int DT, bool B_MN>
__global__ void __launch_bounds__(kThreads, 1)
fused_mlp_fwd_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW1,
                     const __grid_constant__ CUtensorMap tmW2, const __grid_constant__ CUtensorMap tmF1,
                     const __grid_constant__ CUtensorMap tmOut, const MlpParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sX = base;
  const uint32_t sH = sX + kMlpXBytes;
  const uint32_t sW = sH + 2 * kMlpHBytes;
  const uint32_t bars = sW + kMlpStages * kMlpStageBytes;
  const uint32_t x_full = bars;
  auto w_full = [&](int s2) { return bars + 8u * (1 + s2); };
  auto w_empty = [&](int s2) { return bars + 8u * (1 + kMlpStages + s2); };
  auto ht_full = [&](int b) { return bars + 8u * (1 + 2 * kMlpStages + b); };        // hidden accumulator ready (MMA -> epilogue)
  auto ht_empty = [&](int b) { return bars + 8u * (3 + 2 * kMlpStages + b); };       // hidden accumulator drained (epilogue -> MMA)
  auto hs_full = [&](int b) { return bars + 8u * (5 + 2 * kMlpStages + b); };        // hidden operand in smem (epilogue -> MMA)
  auto hs_empty = [&](int b) { return bars + 8u * (7 + 2 * kMlpStages + b); };       // GEMM2 finished reading it (MMA -> epilogue)
  const uint32_t out_full = bars + 8u * (9 + 2 * kMlpStages);
  const uint32_t tmem_slot = bars + 8u * (10 + 2 * kMlpStages);
  const uint32_t bias_off = bars + 256u;           // 1 KB: [2][128] bias floats of the current / next hidden chunk
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - ptx::smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_blk = blockIdx.x / p.splits, split = blockIdx.x % p.splits;
  const int C = p.chunks_per_cta;
  const int chunk0 = split * C;
  const int kbx = p.d / BK;                    // k-blocks of GEMM1 (<= 4)

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tmX); ptx::prefetch_tensormap(&tmW1); ptx::prefetch_tensormap(&tmW2);
    ptx::prefetch_tensormap(&tmF1); ptx::prefetch_tensormap(&tmOut);
    ptx::mbar_init(x_full, 1);
    for (int s2 = 0; s2 < kMlpStages; ++s2) { ptx::mbar_init(w_full(s2), 1); ptx::mbar_init(w_empty(s2), 1); }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(ht_full(b), 1); ptx::mbar_init(ht_empty(b), 8);
      ptx::mbar_init(hs_full(b), 8); ptx::mbar_init(hs_empty(b), 1);
    }
    ptx::mbar_init(out_full, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) { ptx::tmem_alloc_n<512>(tmem_slot); ptx::tmem_relinquish(); }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = *tmem_slot_ptr;
  pdl_wait();
  pdl_trigger();
  const uint32_t tOut = tmem, tH0 = tmem + 256;

  if (warp == 0) {
    if (lane == 0) {
      ptx::mbar_arrive_expect_tx(x_full, (uint32_t)kbx * kABytes);
      for (int kb = 0; kb < kbx; ++kb) ptx::tma_load_4d(sX + kb * kABytes, &tmX, x_full, kb * BK, m_blk * BM, 0, 0);
      int it = 0;
      auto stage_wait = [&](int& st, uint32_t& dst) {
        st = it % kMlpStages;
        ptx::mbar_wait(w_empty(st), (((uint32_t)(it / kMlpStages)) & 1u) ^ 1u);
        dst = sW + st * kMlpStageBytes;
        ++it;
      };
      auto load_w1 = [&](int c) {          // GEMM1 B operand of chunk c: [K = d rows, N = 128 cols] as 2 k-blocks per stage
        const int n0 = (chunk0 + c) * 128;
        for (int s2 = 0; s2 < kbx; s2 += 2) {
          int st; uint32_t dst;
          stage_wait(st, dst);
          const int nkb = min(2, kbx - s2);
          ptx::mbar_arrive_expect_tx(w_full(st), (uint32_t)nkb * 16384u);
          for (int j = 0; j < nkb; ++j) {
            if (B_MN) {
              for (int i = 0; i < 2; ++i)
                ptx::tma_load_4d(dst + j * 16384 + i * 8192, &tmW1, w_full(st), n0 + i * 64, (s2 + j) * BK, 0, 0);
            } else {
              ptx::tma_load_4d(dst + j * 16384, &tmW1, w_full(st), (s2 + j) * BK, n0, 0, 0);      // [128 rows x 64 k]
            }
          }
        }
      };
      auto load_w2 = [&](int c) {          // GEMM2 B operand of chunk c: [K = 128 hidden rows, N = d cols], one k-block per stage
        const int k0 = (chunk0 + c) * 128;
        for (int kb = 0; kb < 2; ++kb) {
          int st; uint32_t dst;
          stage_wait(st, dst);
          ptx::mbar_arrive_expect_tx(w_full(st), (uint32_t)(p.d / 64) * 8192u);
          if (B_MN) {
            for (int i = 0; i < p.d / 64; ++i)
              ptx::tma_load_4d(dst + i * 8192, &tmW2, w_full(st), i * 64, k0 + kb * BK, 0, 0);
          } else {
            ptx::tma_load_4d(dst, &tmW2, w_full(st), k0 + kb * BK, 0, 0, 0);                        // [d rows x 64 k]
          }
        }
      };
      // consumption order of the MMA warp: GEMM1 runs two chunks ahead of GEMM2 (see there)
      load_w1(0);
      if (C > 1) load_w1(1);
      for (int c = 0; c < C; ++c) { if (c + 2 < C) load_w1(c + 2); load_w2(c); }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      int it = 0;
      auto stage_get = [&](uint32_t& src) {
        const int st = it % kMlpStages;
        ptx::mbar_wait(w_full(st), ((uint32_t)(it / kMlpStages)) & 1u);
        ptx::tc_fence_after();
        src = sW + st * kMlpStageBytes;
        ++it;
        return st;
      };
      auto gemm1 = [&](int c) {
        const int b = c & 1;
        ptx::mbar_wait(ht_empty(b), (((uint32_t)c >> 1) & 1u) ^ 1u);
        ptx::tc_fence_after();
        const uint32_t tH = tH0 + (uint32_t)b * 128u;
        for (int s2 = 0; s2 < kbx; s2 += 2) {
          uint32_t src;
          const int st = stage_get(src);
          const int nkb = min(2, kbx - s2);
          for (int j = 0; j < nkb; ++j) {
            const uint32_t sa = sX + (uint32_t)(s2 + j) * kABytes, sb = src + (uint32_t)j * 16384u;
#pragma unroll
            for (int k = 0; k < BK / 16; ++k)
              ptx::mma_f16_ss(tH, ptx::make_smem_desc_sw128(sa + k * 32, 16, 1024),
                              B_MN ? ptx::make_smem_desc_sw128(sb + k * 2048, 8192, 1024) : ptx::make_smem_desc_sw128(sb + k * 32, 16, 1024),
                              p.idesc_g1, (s2 + j > 0 || k > 0) ? 1u : 0u);
          }
          ptx::mma_commit(w_empty(st));
        }
        ptx::mma_commit(ht_full(b));
      };
      auto gemm2 = [&](int c) {
        const int b = c & 1;
        ptx::mbar_wait(hs_full(b), ((uint32_t)c >> 1) & 1u);
        ptx::tc_fence_after();
        for (int kb = 0; kb < 2; ++kb) {
          uint32_t src;
          const int st = stage_get(src);
          const uint32_t sa = sH + (uint32_t)b * kMlpHBytes + (uint32_t)kb * kABytes;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k)
            ptx::mma_f16_ss(tOut, ptx::make_smem_desc_sw128(sa + k * 32, 16, 1024),
                            B_MN ? ptx::make_smem_desc_sw128(src + k * 2048, 8192, 1024) : ptx::make_smem_desc_sw128(src + k * 32, 16, 1024),
                            p.idesc_g2, (c > 0 || kb > 0 || k > 0) ? 1u : 0u);
          ptx::mma_commit(w_empty(st));
        }
        ptx::mma_commit(hs_empty(b));
      };
      ptx::mbar_wait(x_full, 0);
      ptx::tc_fence_after();
      // GEMM1 of chunk c + 2 is issued BEFORE GEMM2 of chunk c: GEMM2(c) has to wait for the epilogue warps to turn the hidden
      // accumulator of chunk c into its smem operand, and the tensor pipe spends that time on the next-but-one GEMM1 (its TMEM
      // buffer (c & 1) is free as soon as the epilogue of chunk c has loaded its registers)
      gemm1(0);
      if (C > 1) gemm1(1);
      for (int c = 0; c < C; ++c) { if (c + 2 < C) gemm1(c + 2); gemm2(c); }
      ptx::mma_commit(out_full);
    }
  } else {
    const int quad = warp & 3, half = (warp - 2) >> 2;
    const int m = m_blk * BM + quad * 32 + lane;
    const bool row_ok = m < p.M;
    const uint32_t lane_addr = (uint32_t)(quad * 32) << 16;
    // ---- hidden chunks: TMEM -> bias, ReLU, dropout (forward) / relu'-dropout' mask (backward) -> 16-bit A operand of GEMM2
    // (+ TMA store: the backward pass / the W1 weight gradient need it).  With 230 KB of shared memory there is no L1 left, so
    // every global operand of the epilogue is fetched one chunk AHEAD: the 64 bias values of each column half go through a
    // 1 KB double buffer in shared memory (loaded by the quad-0 warps), the dropout keep-words / the 16-bit mask row of the
    // thread sit in registers across the wait for the accumulator.
    float* bias_s = reinterpret_cast<float*>(smem_raw + (bias_off - ptx::smem_u32(smem_raw)));      // [2][128]
    const bool use_bits = p.drop_ffn.p > 0.f;
    const float dscale = use_bits ? p.drop_ffn.scale : 1.f;
    const float hidden_floor = p.relu ? 0.f : -INFINITY;
    auto epi_bar = [] { asm volatile("bar.sync 1, 256;" ::: "memory"); };
    uint32_t keep_n[2] = {0xffffffffu, 0xffffffffu};
    uint4 mask_n[B_MN ? 1 : 8];
    auto prefetch = [&](int c) {          // global operands of chunk c
      const int n0 = (chunk0 + c) * 128 + half * 64;
      if (quad == 0 && p.b1) {
        bias_s[(c & 1) * 128 + half * 64 + lane] = __ldg(p.b1 + n0 + lane);
        bias_s[(c & 1) * 128 + half * 64 + 32 + lane] = __ldg(p.b1 + n0 + 32 + lane);
      }
      if (use_bits && row_ok) {
        const uint2 w = __ldg(reinterpret_cast<const uint2*>(p.drop_ffn.bits + ((uint64_t)((int64_t)m * p.ffn + n0) >> 3)));
        keep_n[0] = w.x; keep_n[1] = w.y;
      }
      if (!B_MN) {
        if (p.mask_src && row_ok) {
          const uint4* mp = reinterpret_cast<const uint4*>(reinterpret_cast<const char*>(p.mask_src) + ((int64_t)m * p.mask_ld + n0) * 2);
#pragma unroll
          for (int j = 0; j < 8; ++j) mask_n[j] = __ldg(mp + j);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) mask_n[j] = make_uint4(0, 0, 0, 0);
        }
      }
    };
    prefetch(0);
    epi_bar();
    for (int c = 0; c < C; ++c) {
      const int b = c & 1;
      const int n0 = (chunk0 + c) * 128 + half * 64;          // this warp's 64 hidden columns
      const uint32_t keep[2] = {keep_n[0], keep_n[1]};
      uint4 mask_c[B_MN ? 1 : 8];
      if (!B_MN) {
#pragma unroll
        for (int j = 0; j < 8; ++j) mask_c[j] = mask_n[j];
      }
      if (c + 1 < C) prefetch(c + 1);                          // in flight across the wait for the accumulator
      ptx::mbar_wait(ht_full(b), ((uint32_t)c >> 1) & 1u);
      ptx::tc_fence_after();
      float v[2][32];
      {
        uint32_t r0[32], r1[32];
        __syncwarp();
        ptx::tmem_ld_32x32b_x32(tH0 + (uint32_t)b * 128u + lane_addr + (uint32_t)(half * 64), r0);
        ptx::tmem_ld_32x32b_x32(tH0 + (uint32_t)b * 128u + lane_addr + (uint32_t)(half * 64 + 32), r1);
        ptx::tmem_ld_wait();
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(ht_empty(b));           // the accumulator can be overwritten by GEMM1 of chunk c + 2
        const float* bs = bias_s + b * 128 + half * 64;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const uint32_t (&r)[32] = hh ? r1 : r0;
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            float4 bb = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p.b1) bb = *reinterpret_cast<const float4*>(bs + hh * 32 + 4 * j4);          // broadcast LDS.128
            v[hh][4 * j4 + 0] = fmaxf(fmaf(__uint_as_float(r[4 * j4 + 0]), p.alpha, bb.x), hidden_floor);
            v[hh][4 * j4 + 1] = fmaxf(fmaf(__uint_as_float(r[4 * j4 + 1]), p.alpha, bb.y), hidden_floor);
            v[hh][4 * j4 + 2] = fmaxf(fmaf(__uint_as_float(r[4 * j4 + 2]), p.alpha, bb.z), hidden_floor);
            v[hh][4 * j4 + 3] = fmaxf(fmaf(__uint_as_float(r[4 * j4 + 3]), p.alpha, bb.w), hidden_floor);
          }
          if (use_bits) {
            const uint32_t k32 = keep[hh];
#pragma unroll
            for (int j = 0; j < 32; ++j) v[hh][j] = ((k32 >> j) & 1u) ? v[hh][j] * dscale : 0.f;
          }
          if (!B_MN) {
            // 16-bit mask source (bf16 / fp16): "> 0" <=> sign clear and magnitude bits non-zero
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint4 pk = mask_c[hh * 4 + j];
              const uint32_t w[4] = {pk.x, pk.y, pk.z, pk.w};
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const uint32_t lo = w[i] & 0xffffu, hi = w[i] >> 16;
                if (!(lo != 0u && lo < 0x8000u)) v[hh][8 * j + 2 * i] = 0.f;
                if (!(hi != 0u && hi < 0x8000u)) v[hh][8 * j + 2 * i + 1] = 0.f;
              }
            }
          }
        }
      }
      // operand buffer b: GEMM2 of chunk c - 2 has finished reading it, and this warp's own TMA store of chunk c - 2 too
      ptx::mbar_wait(hs_empty(b), (((uint32_t)c >> 1) & 1u) ^ 1u);
      if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
      __syncwarp();
      const uint32_t tile = sH + (uint32_t)b * kMlpHBytes + (uint32_t)half * kABytes + (uint32_t)(quad * 32) * 128u;
      stage_chunk<DT == F16 ? OUT_F16 : OUT_BF16>(tile, lane, 0, v[0]);
      stage_chunk<DT == F16 ? OUT_F16 : OUT_BF16>(tile, lane, 1, v[1]);
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        ptx::mbar_arrive(hs_full(b));
        asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                     ::"l"(&tmF1), "r"(tile), "r"(n0), "r"(m_blk * BM + quad * 32), "r"(0), "r"(0) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
      epi_bar();                 // bias of chunk c + 1 is in shared memory; buffer (c & 1) may be refilled next iteration
    }
    // output bias (slice 0 only) through the same 1 KB of shared memory, keep-words of the output tile in registers
    const int ncol = p.d / 2;                                    // columns per half
    const bool add_b2 = split == 0 && p.b2 != nullptr;
    if (add_b2 && (int)threadIdx.x - 64 < p.d) bias_s[threadIdx.x - 64] = __ldg(p.b2 + (threadIdx.x - 64));
    uint32_t keep_o[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
    if (p.drop_post.p > 0.f && row_ok) {
      const uint32_t* kp = reinterpret_cast<const uint32_t*>(p.drop_post.bits + ((uint64_t)((int64_t)m * p.d + half * ncol) >> 3));
#pragma unroll
      for (int j = 0; j < 4; ++j) if (j < ncol / 32) keep_o[j] = __ldg(kp + j);
    }
    epi_bar();
    // ---- output tile: TMEM -> (+ b2 on slice 0) -> post dropout -> fp32 reduce-add into x_out ----
    ptx::mbar_wait(out_full, 0);
    ptx::tc_fence_after();
    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncwarp();
    const float pscale = p.drop_post.p > 0.f ? p.drop_post.scale : 1.f;
    const uint32_t my_stage = sW + (uint32_t)(warp - 2) * 8192u;  // weight ring is free now: 8 warps x 2 x 4 KB boxes
    if (p.tickets && p.splits > 1) {
      // deterministic reduction order: slice s adds only after slices 0 .. s-1 of this row tile have completed theirs
      if (lane == 0) {
        const volatile int* tk = p.tickets + m_blk;
        while (*tk != split) { }
        __threadfence();
      }
      __syncwarp();
    }
#pragma unroll 1
    for (int bx = 0; bx < ncol / 32; ++bx) {
      const int co = half * ncol + bx * 32;
      const uint32_t buf = my_stage + (uint32_t)(bx & 1) * 4096u;
      if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
      __syncwarp();
      uint32_t r[32];
      ptx::tmem_ld_32x32b_x32(tOut + lane_addr + (uint32_t)co, r);
      ptx::tmem_ld_wait();
      float v[32];
      const uint32_t k32 = keep_o[bx & 3];
#pragma unroll
      for (int j4 = 0; j4 < 8; ++j4) {
        float4 bb = make_float4(0.f, 0.f, 0.f, 0.f);
        if (add_b2) bb = *reinterpret_cast<const float4*>(bias_s + co + 4 * j4);
        v[4 * j4 + 0] = __uint_as_float(r[4 * j4 + 0]) + bb.x; v[4 * j4 + 1] = __uint_as_float(r[4 * j4 + 1]) + bb.y;
        v[4 * j4 + 2] = __uint_as_float(r[4 * j4 + 2]) + bb.z; v[4 * j4 + 3] = __uint_as_float(r[4 * j4 + 3]) + bb.w;
      }
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = ((k32 >> j) & 1u) ? v[j] * pscale : 0.f;
      stage_chunk<OUT_F32>(buf, lane, 0, v);
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        asm volatile("cp.reduce.async.bulk.tensor.4d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                     ::"l"(&tmOut), "r"(buf), "r"(co), "r"(m_blk * BM + quad * 32), "r"(0), "r"(0) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    if (p.tickets && p.splits > 1) {
      __threadfence();
      epi_bar();                                   // all 8 warps' reductions have been performed
      if (threadIdx.x == 64) atomicExch(p.tickets + m_blk, split + 1 == p.splits ? 0 : split + 1);
    }
    ptx::tc_fence_before();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) { ptx::tc_fence_after(); ptx::tmem_dealloc(tmem, 512); }
}

// -------------------------------------------------------------------------------------------
// Host side: tensor-map construction (driver entry point fetched at run time; no libcuda link)
// -------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

struct MapKey {
  uint64_t v[10];
  bool operator==(const MapKey& o) const { return std::memcmp(v, o.v, sizeof(v)) == 0; }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    uint64_t h = 1469598103934665603ull;
    for (uint64_t x : k.v) { h ^= x; h *= 1099511628211ull; }
    return (size_t)h;
  }
};
std::mutex g_map_mu;
std::unordered_map<MapKey, CUtensorMap, MapKeyHash> g_map_cache;

// Operand tensor map: dims (inner, outer, nb1, nb2); inner = K (K-major) or M/N (MN-major).
int make_operand_map(const GemmOperand& op, int rows, int K, int nb1, int nb2, int box_rows_kmajor, CUtensorMap* out) {
  EncodeTiledFn fn = get_encode_fn();
  B200ST_CHECK(fn != nullptr, "cuTensorMapEncodeTiled unavailable (no CUDA driver?)");
  const uint64_t es = 2;
  uint64_t inner = op.mn_major ? (uint64_t)rows : (uint64_t)K;
  uint64_t outer = op.mn_major ? (uint64_t)K : (uint64_t)rows;
  uint64_t sb1 = nb1 > 1 ? (uint64_t)op.sb1 : (uint64_t)op.ld * outer;
  uint64_t sb2 = nb2 > 1 ? (uint64_t)op.sb2 : sb1 * (uint64_t)nb1;
  if (sb1 == 0) sb1 = (uint64_t)op.ld * outer;   // broadcast batch strides are not used by callers of the TC path
  if (sb2 == 0) sb2 = sb1 * (uint64_t)nb1;
  cuuint64_t dims[4] = {inner, outer, (cuuint64_t)nb1, (cuuint64_t)nb2};
  cuuint64_t strides[3] = {(cuuint64_t)op.ld * es, sb1 * es, sb2 * es};
  cuuint32_t box[4] = {64u, (cuuint32_t)(op.mn_major ? BK : box_rows_kmajor), 1u, 1u};
  cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
  B200ST_CHECK((reinterpret_cast<uintptr_t>(op.ptr) & 15) == 0, "TMA operand base must be 16-byte aligned");
  B200ST_CHECK(strides[0] % 16 == 0 && strides[1] % 16 == 0 && strides[2] % 16 == 0,
               "TMA operand strides must be multiples of 16 bytes (ld % 8 == 0 for bf16)");
  MapKey key{{(uint64_t)(uintptr_t)op.ptr, inner, outer, (uint64_t)nb1, (uint64_t)nb2, strides[0], strides[1], strides[2],
              box[1], (uint64_t)op.mn_major | ((uint64_t)op.dtype << 8)}};
  {
    std::lock_guard<std::mutex> lk(g_map_mu);
    auto it = g_map_cache.find(key);
    if (it != g_map_cache.end()) { *out = it->second; return 0; }
  }
  CUresult r = fn(out, op.dtype == F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4,
                  const_cast<void*>(op.ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) B200ST_FAIL("cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
  std::lock_guard<std::mutex> lk(g_map_mu);
  if (g_map_cache.size() > 65536) g_map_cache.clear();
  g_map_cache.emplace(key, *out);
  return 0;
}

// Output tensor map: dims (N, M, nb1, nb2); box = {128 bytes of columns, 32 rows} (one epilogue warp), 128B swizzle.
int make_out_map(const void* C, int c_dtype, int N, int M, int nb1, int nb2, int64_t ldc, int64_t sb1, int64_t sb2, CUtensorMap* out) {
  EncodeTiledFn fn = get_encode_fn();
  B200ST_CHECK(fn != nullptr, "cuTensorMapEncodeTiled unavailable (no CUDA driver?)");
  const uint64_t es = c_dtype == F32 ? 4 : 2;
  uint64_t s1 = nb1 > 1 ? (uint64_t)sb1 : (uint64_t)ldc * M;
  uint64_t s2 = nb2 > 1 ? (uint64_t)sb2 : s1 * (uint64_t)nb1;
  if (s1 == 0) s1 = (uint64_t)ldc * M;
  if (s2 == 0) s2 = s1 * (uint64_t)nb1;
  cuuint64_t dims[4] = {(cuuint64_t)N, (cuuint64_t)M, (cuuint64_t)nb1, (cuuint64_t)nb2};
  cuuint64_t strides[3] = {(cuuint64_t)ldc * es, s1 * es, s2 * es};
  cuuint32_t box[4] = {(cuuint32_t)(128 / es), 32u, 1u, 1u};
  cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
  if (strides[1] % 16 != 0) strides[1] = (strides[1] + 15) / 16 * 16;   // size-1 batch dims: any legal stride
  if (strides[2] % 16 != 0) strides[2] = (strides[2] + 15) / 16 * 16;
  MapKey key{{(uint64_t)(uintptr_t)C, (uint64_t)N, (uint64_t)M, (uint64_t)nb1, (uint64_t)nb2, strides[0], strides[1], strides[2],
              0x1000u + es, 7u | ((uint64_t)c_dtype << 8)}};
  {
    std::lock_guard<std::mutex> lk(g_map_mu);
    auto it = g_map_cache.find(key);
    if (it != g_map_cache.end()) { *out = it->second; return 0; }
  }
  CUresult r = fn(out, c_dtype == F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : c_dtype == F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(C), dims,
                  strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) B200ST_FAIL("cuTensorMapEncodeTiled (output) failed with CUresult " + std::to_string((int)r));
  std::lock_guard<std::mutex> lk(g_map_mu);
  g_map_cache.emplace(key, *out);
  return 0;
}

int g_num_sms = 0;
int g_reserved_sms = 0;
int64_t g_launches = 0;

// SMs a persistent grid may occupy: the device's SMs less those reserved for concurrent communication kernels (a
// reservation that would leave none is ignored)
int usable_sms(int* out) {
  if (g_num_sms == 0) {
    int dev = 0;
    B200ST_CUDA(cudaGetDevice(&dev));
    B200ST_CUDA(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev));
  }
  *out = g_reserved_sms > 0 && g_reserved_sms < g_num_sms ? g_num_sms - g_reserved_sms : g_num_sms;
  return 0;
}
}  // namespace

// 16-bit 4-D tensor map (inner, rows, nb1, nb2) with a {box_inner<=64, box_rows} box, 128B swizzle.
int make_tma_map_16(const void* ptr, int dtype, uint64_t inner, uint64_t rows, int nb1, int nb2, int64_t ld, int64_t sb1, int64_t sb2,
                    uint32_t box_rows, CUtensorMap* out) {
  GemmOperand op{ptr, dtype, 0, ld, sb1, sb2};
  return make_operand_map(op, (int)rows, (int)inner, nb1, nb2, (int)box_rows, out);
}
void tc_count_launch() { ++g_launches; }

namespace {

// optional GEMM profile (bench.py roofline pass; off in the timed region): every tcgen05 GEMM issued between begin and
// end is RECORDED (arguments only); tc_profile_end() then replays each recorded GEMM back to back (1 warm-up + kReps timed
// launches bracketed by one event pair, no host gap between them) and reports the per-launch average.  The buffers of the
// step are still alive (same workspace), accumulate / reduce epilogues only add into gradients nobody reads afterwards.
// conv2 data gradient as an implicit GEMM (see conv2_dgrad_implicit): replaces the A tensor map and the k-block -> coordinates rule
struct ConvA {
  const void* dy; int B, T2, F2, C;     // dY [B, T2, F2, C]
  int tu, ub, ntaps;
  int dt[4], df[4], wrow[4];
};
struct ProfRec { GemmArgs g; cudaStream_t stream; int bn, splitk; int group_n = 0; GemmArgs rest[3]; bool has_conv = false; ConvA conv; };   // group_n > 1: grouped weight-gradient launch (g + rest)
bool g_prof = false;
std::vector<ProfRec> g_prof_recs;

template <int BN, bool A_MN, bool B_MN, int OUT>
int launch_out(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const TcParams& p, int grid, size_t smem,
               cudaStream_t stream) {
  auto kern = tc_gemm_kernel<BN, A_MN, B_MN, OUT>;
  static bool attr_set = false;
  if (!attr_set) {
    B200ST_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
    attr_set = true;
  }
  launch_pdl(kern, grid, kThreads, smem, stream, ta, tb, tc, p);
  B200ST_LAUNCH_CHECK();
  return 0;
}

template <int BN, bool A_MN, bool B_MN>
int launch_variant(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const TcParams& p, int grid, size_t smem,
                   cudaStream_t stream) {
  if (p.atomic) return launch_out<BN, A_MN, B_MN, OUT_ATOMIC>(ta, tb, tc, p, grid, smem, stream);
  if (p.c_dtype == F32) return launch_out<BN, A_MN, B_MN, OUT_F32>(ta, tb, tc, p, grid, smem, stream);
  if (p.c_dtype == F16) return launch_out<BN, A_MN, B_MN, OUT_F16>(ta, tb, tc, p, grid, smem, stream);
  return launch_out<BN, A_MN, B_MN, OUT_BF16>(ta, tb, tc, p, grid, smem, stream);
}

template <int BN>
int launch_bn(bool a_mn, bool b_mn, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const TcParams& p, int grid,
              size_t smem, cudaStream_t stream) {
  if (!a_mn && !b_mn) return launch_variant<BN, false, false>(ta, tb, tc, p, grid, smem, stream);
  if (!a_mn && b_mn) return launch_variant<BN, false, true>(ta, tb, tc, p, grid, smem, stream);
  if (a_mn && !b_mn) return launch_variant<BN, true, false>(ta, tb, tc, p, grid, smem, stream);
  return launch_variant<BN, true, true>(ta, tb, tc, p, grid, smem, stream);
}

}  // namespace

void gemm_set_reserved_sms(int n) { g_reserved_sms = n; }
int64_t tc_launch_count() { return g_launches; }

namespace {
int gemm_tc_impl(const GemmArgs& g, cudaStream_t stream, const ConvA* conv);
}  // namespace
int gemm_tc_bf16(const GemmArgs& g, cudaStream_t stream) { return gemm_tc_impl(g, stream, nullptr); }

namespace {
int gemm_tc_impl(const GemmArgs& g, cudaStream_t stream, const ConvA* conv) {
  B200ST_CHECK(is16(g.A.dtype) && is16(g.B.dtype), "tcgen05 GEMM needs 16-bit (bf16 / fp16) operands");
  // measured on B200 (round 2): a kind::f16 MMA whose A and B formats differ raises an illegal-instruction fault, although
  // the instruction descriptor encodes them separately — so the library refuses mixed products up front
  B200ST_CHECK(g.A.dtype == g.B.dtype, "tcgen05 kind::f16 needs A and B in the same 16-bit format (both bf16 or both fp16)");
  B200ST_CHECK(g.M > 0 && g.N > 0 && g.K > 0 && g.nb1 > 0 && g.nb2 > 0, "empty GEMM");
  if (const int abl = ablate_mask()) {
    const bool wgrad = g.A.mn_major && g.B.mn_major;
    if ((wgrad && (abl & ABL_WGRAD)) || (!wgrad && (abl & ABL_GEMM))) return 0;
  }
  int num_sms = 0;
  B200ST_TRY(usable_sms(&num_sms));

  TcParams p{};
  p.M = g.M; p.N = g.N; p.K = g.K; p.nb1 = g.nb1; p.nb2 = g.nb2;
  p.m_tiles = ceil_div(g.M, BM);
  p.kb_total = ceil_div(g.K, BK);
  const int64_t batch = (int64_t)g.nb1 * g.nb2;

  // ---- joint choice of the N tile and the split-K factor ----
  // Per k-block a CTA needs max(tensor time, L2->smem fill time): 4 MMAs of 128 x c x 16 take 2c cycles; the operand
  // bytes (16 KB + 128c B) arrive at ~44 B/cycle/SM (measured, profiles/r01_gemm_notes.md).  The epilogue overlaps the
  // next tile's main loop.  Split-K (fp32 TMA reduce-add epilogue) is allowed for linear accumulate epilogues only and is
  // chosen so that the tile count fills the 148 SMs once.
  const bool linear_epi = !g.epi.relu && !g.epi.mask_src && g.epi.drop.p == 0.f && !g.epi.residual && !g.epi.bias;
  const bool split_ok = linear_epi && g.c_dtype == F32 && g.epi.accumulate;
  if (g.splitk > 1) B200ST_CHECK(split_ok, "split-K needs a linear fp32 accumulate epilogue");
  int bn, splitk = g.splitk >= 1 ? g.splitk : 1;
  {
    double best = 1e30;
    int best_bn = 0, best_sk = 1;
    const int cands[3] = {256, 128, 64};
    for (int c : cands) {
      if (conv && c != 256) continue;
      if (c > 64 && c >= 2 * ((g.N + 63) / 64 * 64)) continue;   // do not pad N by 2x or more
      const int64_t tiles0 = batch * p.m_tiles * ceil_div(g.N, c);
      int sk_lo = splitk, sk_hi = splitk;
      if (g.splitk == 0 && split_ok) {
        sk_lo = 1;
        sk_hi = (int)(num_sms / tiles0);
        const int cap = p.kb_total / 4 > 0 ? p.kb_total / 4 : 1;
        if (sk_hi > cap) sk_hi = cap;
        if (sk_hi < 1) sk_hi = 1;
      }
      for (int sk = sk_hi; sk >= sk_lo; sk = (sk > sk_lo && sk > 1) ? (sk == sk_hi && sk_hi > 2 ? sk / 2 : sk - 1) : sk_lo - 1) {
        const int kb_per = ceil_div(p.kb_total, sk);
        const int64_t tiles = tiles0 * ceil_div(p.kb_total, kb_per);
        const int64_t waves = (tiles + num_sms - 1) / num_sms;
        const double fill = (16384.0 + 128.0 * c) / 44.0, mma = 2.0 * c;
        const double mainloop = kb_per * (fill > mma ? fill : mma);
        const double epi = (sk > 1 ? 14.0 : 10.0) * c + 600.0;
        const double cost = (double)waves * ((mainloop > epi ? mainloop : epi) + 800.0) + (sk > 1 ? 500.0 : 0.0);
        if (cost < best) { best = cost; best_bn = c; best_sk = sk; }
        if (sk <= sk_lo) break;
      }
    }
    bn = best_bn;
    splitk = best_sk;
  }
  if (splitk > p.kb_total) splitk = p.kb_total;
  p.kb_per_split = ceil_div(p.kb_total, splitk);
  splitk = ceil_div(p.kb_total, p.kb_per_split);   // no empty trailing split
  p.splitk = splitk;
  p.atomic = (splitk > 1) ? 1 : 0;
  p.n_tiles = ceil_div(g.N, bn);
  p.num_tiles = batch * p.m_tiles * p.n_tiles * splitk;

  // one CTA per SM (two co-resident CTAs were measured: no gain, see profiles/r01_gemm_notes.md)
  const uint32_t stage_bytes = kABytes + (uint32_t)bn * BK * 2;
  int stages = (int)((kSmemLimit - (int)kStagingBytes - 2048) / stage_bytes);
  if (stages > 8) stages = 8;
  p.stages = stages;
  const size_t smem = 1024 + (size_t)stages * stage_bytes + kStagingBytes + 8 * (2 * stages + 5) + 16;
  B200ST_CHECK(smem <= (size_t)kSmemLimit, "smem budget exceeded");

  // descriptors
  const uint32_t mn_lbo = 64u * BK * 2;   // next 64-wide MN chunk (TMA box)
  const uint32_t mn_sbo = 1024u;          // next group of 8 k-rows
  const uint32_t k_lbo = 16u;             // ignored for swizzled K-major
  const uint32_t k_sbo = 1024u;           // next group of 8 rows
  p.a_lbo = g.A.mn_major ? mn_lbo : k_lbo;  p.a_sbo = g.A.mn_major ? mn_sbo : k_sbo;
  p.b_lbo = g.B.mn_major ? mn_lbo : k_lbo;  p.b_sbo = g.B.mn_major ? mn_sbo : k_sbo;
  p.a_kstep = g.A.mn_major ? 16u * 128u : 32u;
  p.b_kstep = g.B.mn_major ? 16u * 128u : 32u;
  p.idesc = ptx::make_idesc_16(bn, g.A.mn_major, g.B.mn_major, g.A.dtype == BF16, g.B.dtype == BF16);

  p.C = g.C; p.c_dtype = g.c_dtype; p.ldc = g.ldc; p.c_sb1 = g.c_sb1; p.c_sb2 = g.c_sb2;
  p.epi = g.epi;
  if (g.epi.accumulate) B200ST_CHECK(g.c_dtype == F32, "accumulate needs fp32 C");

  // ---- output path: TMA store through per-warp staging boxes when everything is 16-byte aligned ----
  const uint64_t esz_c = g.c_dtype == F32 ? 4 : 2;
  auto al16 = [](const void* ptr) { return (reinterpret_cast<uintptr_t>(ptr) & 15) == 0; };
  bool tma_ok = al16(g.C) && (g.ldc * esz_c) % 16 == 0 && (g.nb1 == 1 || (g.c_sb1 * esz_c) % 16 == 0) &&
                (g.nb2 == 1 || (g.c_sb2 * esz_c) % 16 == 0) && g.N >= bn;
  if (g.epi.bias) tma_ok = tma_ok && al16(g.epi.bias);
  if (g.epi.mask_src) {
    const uint64_t em = g.epi.mask_dtype == F32 ? 4 : 2;   // bf16 and fp16 masks are both read as sign/magnitude words
    tma_ok = tma_ok && al16(g.epi.mask_src) && (g.epi.mask_ld * em) % 16 == 0 && (g.epi.mask_sb1 * em) % 16 == 0 &&
             (g.epi.mask_sb2 * em) % 16 == 0;
  }
  if (g.epi.residual)
    tma_ok = tma_ok && al16(g.epi.residual) && (g.epi.res_ld * 4) % 16 == 0 && (g.epi.res_sb1 * 4) % 16 == 0 && (g.epi.res_sb2 * 4) % 16 == 0;
  if (g.epi.drop.p > 0.f) tma_ok = tma_ok && g.epi.drop.bits != nullptr && (g.N % 32 == 0);
  p.use_tma_store = tma_ok ? 1 : 0;
  p.c_reduce = (p.atomic || g.epi.accumulate) ? 1 : 0;
  CUtensorMap tc;
  std::memset(&tc, 0, sizeof(tc));
  if (tma_ok) B200ST_TRY(make_out_map(g.C, g.c_dtype, g.N, g.M, g.nb1, g.nb2, g.ldc, g.c_sb1, g.c_sb2, &tc));

  CUtensorMap ta, tb;
  if (conv) {
    B200ST_CHECK(bn == 256 && splitk == 1 && !g.A.mn_major && !g.B.mn_major && g.nb1 == 1 && g.nb2 == 1 && conv->C % BK == 0 &&
                     g.K == conv->ntaps * conv->C && g.M == conv->B * conv->ub * BM && conv->F2 * conv->tu <= BM && conv->ntaps <= 4,
                 "implicit conv dgrad: unsupported shape");
    p.conv = 1; p.conv_ub = conv->ub; p.conv_tu = conv->tu; p.conv_kpc = conv->C / BK;
    for (int i = 0; i < conv->ntaps; ++i) { p.conv_dt[i] = conv->dt[i]; p.conv_df[i] = conv->df[i]; p.conv_wrow[i] = conv->wrow[i]; }
    p.conv_a_bytes = (uint32_t)(BK * conv->F2 * conv->tu * 2);
    // A: dY as a 4-D tensor (C, F2, T2, B); one box = 64 channels x all F2 frequencies x tu time rows of one utterance — rows
    // beyond the tensor (the shifted taps at the far edge) are zero-filled by the TMA unit, i.e. the convolution's border
    EncodeTiledFn fn = get_encode_fn();
    B200ST_CHECK(fn != nullptr, "cuTensorMapEncodeTiled unavailable (no CUDA driver?)");
    B200ST_CHECK((reinterpret_cast<uintptr_t>(conv->dy) & 15) == 0, "TMA operand base must be 16-byte aligned");
    cuuint64_t dims[4] = {(cuuint64_t)conv->C, (cuuint64_t)conv->F2, (cuuint64_t)conv->T2, (cuuint64_t)conv->B};
    cuuint64_t strides[3] = {(cuuint64_t)conv->C * 2, (cuuint64_t)conv->F2 * conv->C * 2, (cuuint64_t)conv->T2 * conv->F2 * conv->C * 2};
    cuuint32_t box[4] = {(cuuint32_t)BK, (cuuint32_t)conv->F2, (cuuint32_t)conv->tu, 1u};
    cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
    CUresult r = fn(&ta, g.A.dtype == F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(conv->dy),
                    dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) B200ST_FAIL("cuTensorMapEncodeTiled (conv dY) failed with CUresult " + std::to_string((int)r));
    B200ST_TRY(make_operand_map(g.B, 9 * conv->C, conv->C, 1, 1, bn, &tb));      // all 9 taps of the [9C, C] weight matrix
  } else {
    B200ST_TRY(make_operand_map(g.A, g.M, g.K, g.nb1, g.nb2, BM, &ta));
    B200ST_TRY(make_operand_map(g.B, g.N, g.K, g.nb1, g.nb2, bn, &tb));
  }

  const int grid = (int)(p.num_tiles < num_sms ? p.num_tiles : num_sms);
  ++g_launches;
  if (g_prof) {
    ProfRec r{g, stream, bn, splitk};
    if (conv) { r.has_conv = true; r.conv = *conv; }
    g_prof_recs.push_back(r);
  }
  int rc = 0;
  switch (bn) {
    case 64: rc = launch_bn<64>(g.A.mn_major, g.B.mn_major, ta, tb, tc, p, grid, smem, stream); break;
    case 128: rc = launch_bn<128>(g.A.mn_major, g.B.mn_major, ta, tb, tc, p, grid, smem, stream); break;
    case 256: rc = launch_bn<256>(g.A.mn_major, g.B.mn_major, ta, tb, tc, p, grid, smem, stream); break;
    default: B200ST_FAIL("unsupported BN");
  }
  return rc;
}
}  // namespace

// Data gradient of the 3x3 / stride-2 / pad-1 convolution (Conv2D#2 of AudioConv2dSubsamplingLayer,
// neurst/layers/modalities/audio_modalities.py:96-104) as four implicit GEMMs, one per parity class (t1 & 1, f1 & 1) of the
// input position: dA[b, t1, f1, :] = sum over the taps (kh, kw) with t1 = 2 t2 + kh - 1, f1 = 2 f2 + kw - 1 of
// dY[b, t2, f2, :] W[kh, kw]^T — 1 tap for (even, even), 2 for the mixed classes, 4 for (odd, odd).  The A operand is read
// straight out of dY by 4-D TMA boxes shifted by the tap (zero fill = border), so neither the [rows, 9C] column gradient
// (737 MB at cfg-2) nor its col2im gather exist.  Output: class-major padded tiles
//   dA[cls][b][tile][128 rows = tu x F2 positions (+ unused rows)][C],   tile = (t1 >> 1) / tu,   row = ((t1 >> 1) % tu) * F2 + (f1 >> 1)
// which conv1's backward kernel reads back with the same arithmetic.
int conv2_dgrad_implicit(const void* dy, const void* w16, void* da, int dtype, int B, int T2, int F2, int C, cudaStream_t stream) {
  B200ST_CHECK(is16(dtype) && C == 256 && F2 >= 1 && F2 <= BM, "implicit conv2 dgrad: 16-bit, C == 256, F2 <= 128");
  ConvA ca{};
  ca.dy = dy; ca.B = B; ca.T2 = T2; ca.F2 = F2; ca.C = C;
  ca.tu = BM / F2;
  ca.ub = ceil_div(T2, ca.tu);
  const int64_t cls_elems = (int64_t)B * ca.ub * BM * C;
  for (int cls = 0; cls < 4; ++cls) {
    const int pt = cls >> 1, pf = cls & 1;
    // per axis: even position -> centre tap, same index; odd position -> tap 2 at the same index and tap 0 at index + 1
    const int nt = pt ? 2 : 1, nf = pf ? 2 : 1;
    const int kh_of[2] = {pt ? 2 : 1, 0}, dt_of[2] = {0, 1};
    const int kw_of[2] = {pf ? 2 : 1, 0}, df_of[2] = {0, 1};
    ca.ntaps = nt * nf;
    for (int a = 0; a < nt; ++a)
      for (int b2 = 0; b2 < nf; ++b2) {
        const int i = a * nf + b2;
        ca.dt[i] = dt_of[a]; ca.df[i] = df_of[b2]; ca.wrow[i] = (kh_of[a] * 3 + kw_of[b2]) * C;
      }
    GemmArgs g = gemm_defaults();
    g.M = B * ca.ub * BM; g.N = C; g.K = ca.ntaps * C;
    g.A = GemmOperand{dy, dtype, 0, C, 0, 0};
    g.B = GemmOperand{w16, dtype, 0, C, 0, 0};
    g.C = reinterpret_cast<char*>(da) + (size_t)cls * cls_elems * 2; g.c_dtype = dtype; g.ldc = C;
    B200ST_TRY(gemm_tc_impl(g, stream, &ca));
  }
  return 0;
}
int64_t conv2_dgrad_implicit_elems(int B, int T2, int F2, int C) {
  const int tu = BM / F2;
  return 4 * (int64_t)B * ceil_div(T2, tu) * BM * C;
}


// One launch for the weight gradients of a backward block (see tc_wgrad_group_kernel).  Every product must be a plain
// fp32-accumulate MN-major x MN-major 16-bit GEMM with M % 128 == 0 and N % 256 == 0; returns 2 (nothing launched) when the
// group does not qualify, so that the caller issues the products one by one.
int gemm_wgrad_group(const GemmArgs* gs, int n, cudaStream_t stream) {
  if (n < 2 || n > kMaxGroup) return 2;
  for (int i = 0; i < n; ++i) {
    const GemmArgs& g = gs[i];
    const bool plain = !g.epi.relu && !g.epi.mask_src && g.epi.drop.p == 0.f && !g.epi.residual && !g.epi.bias && g.epi.accumulate;
    if (!(is16(g.A.dtype) && g.A.dtype == g.B.dtype && g.A.dtype == gs[0].A.dtype && g.A.mn_major && g.B.mn_major && plain &&
          g.c_dtype == F32 && g.nb1 == 1 && g.nb2 == 1 && g.M % BM == 0 && g.N % 256 == 0 && g.K > 0 && g.splitk <= 1 &&
          (reinterpret_cast<uintptr_t>(g.C) & 15) == 0 && (g.ldc * 4) % 16 == 0))
      return 2;
  }
  if (ablate_mask() & ABL_WGRAD) return 0;
  int num_sms = 0;
  B200ST_TRY(usable_sms(&num_sms));
  TcGroup grp;
  std::memset(&grp, 0, sizeof(grp));
  grp.n = n;
  int64_t work = 0;
  int tiles0[kMaxGroup], kbt[kMaxGroup];
  for (int i = 0; i < n; ++i) {
    tiles0[i] = (gs[i].M / BM) * (gs[i].N / 256);
    kbt[i] = ceil_div(gs[i].K, BK);
    work += (int64_t)tiles0[i] * kbt[i];
  }
  // smallest common k-range L (in 64-row blocks) whose work units fit one wave of `num_sms` CTAs
  int L = (int)((work + num_sms - 1) / num_sms);
  if (L < 2) L = 2;
  for (;; ++L) {
    int64_t units = 0;
    for (int i = 0; i < n; ++i) units += (int64_t)tiles0[i] * ceil_div(kbt[i], L);
    if (units <= num_sms || L >= 4096) break;
  }
  int tile = 0;
  for (int i = 0; i < n; ++i) {
    const GemmArgs& g = gs[i];
    TcGroupProb& q = grp.prob[i];
    q.m_tiles = g.M / BM; q.n_tiles = g.N / 256; q.kb_total = kbt[i];
    q.kb_per_split = L < kbt[i] ? L : kbt[i];
    q.splitk = ceil_div(kbt[i], q.kb_per_split);
    q.tile_begin = tile;
    q.alpha = g.epi.alpha;
    tile += q.m_tiles * q.n_tiles * q.splitk;
    B200ST_TRY(make_operand_map(g.A, g.M, g.K, 1, 1, BM, &q.ta));
    B200ST_TRY(make_operand_map(g.B, g.N, g.K, 1, 1, 256, &q.tb));
    B200ST_TRY(make_out_map(g.C, F32, g.N, g.M, 1, 1, g.ldc, 0, 0, &q.tc));
  }
  grp.num_tiles = tile;
  const uint32_t stage_bytes = kABytes + 256u * BK * 2;
  int stages = (int)((kSmemLimit - (int)kStagingBytes - 2048) / stage_bytes);
  if (stages > 8) stages = 8;
  grp.stages = stages;
  grp.idesc = ptx::make_idesc_16(256, 1, 1, gs[0].A.dtype == BF16, gs[0].B.dtype == BF16);
  const size_t smem = 1024 + (size_t)stages * stage_bytes + kStagingBytes + 8 * (2 * stages + 5) + 16;
  B200ST_CHECK(smem <= (size_t)kSmemLimit, "smem budget exceeded");
  static bool attr_set = false;
  if (!attr_set) {
    B200ST_CUDA(cudaFuncSetAttribute(tc_wgrad_group_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
    attr_set = true;
  }
  const int grid = grp.num_tiles < num_sms ? grp.num_tiles : num_sms;
  ++g_launches;
  if (g_prof) {
    ProfRec r{gs[0], stream, 256, grp.prob[0].splitk};
    r.group_n = n;
    for (int i = 1; i < n; ++i) r.rest[i - 1] = gs[i];
    g_prof_recs.push_back(r);
  }
  launch_pdl(tc_wgrad_group_kernel, grid, kThreads, smem, stream, grp);
  B200ST_LAUNCH_CHECK();
  return 0;
}


// Fused FFN forward (see fused_mlp_fwd_kernel).  X: 16-bit [M, d] (LayerNorm output); W1 [d, ffn], W2 [ffn, d] in the same
// 16-bit type (TF layouts); F1 out [M, ffn] (saved for the backward pass); x_out fp32 [M, d] must already hold the residual.
bool fused_mlp_supported(int M, int d, int ffn, int dtype) {
  return is16(dtype) && (d == 128 || d == 256) && ffn % 128 == 0 && M > 0;
}
namespace {
// slices of the hidden dimension: the most CTAs that still fit one wave, with an equal number of 128-column chunks per slice
int mlp_splits(int M, int ffn, int* splits) {
  int num_sms = 0;
  B200ST_TRY(usable_sms(&num_sms));
  const int m_tiles = ceil_div(M, BM), chunks = ffn / 128;
  *splits = 1;
  for (int s = 1; s <= chunks; ++s)
    if (chunks % s == 0 && (int64_t)m_tiles * s <= num_sms) *splits = s;
  return 0;
}
}  // namespace
int fused_mlp_fwd(const void* X, int dtype, int M, int d, int ffn, const void* W1, const float* b1, const void* W2, const float* b2,
                  DropoutSpec drop_ffn, DropoutSpec drop_post, void* F1, float* x_out, cudaStream_t stream, int* tickets,
                  int* splits_out) {
  if (ablate_mask() & ABL_MLP_FWD) return 0;
  B200ST_CHECK(fused_mlp_supported(M, d, ffn, dtype), "fused MLP: unsupported shape / dtype");
  if (drop_ffn.p > 0.f) B200ST_CHECK(drop_ffn.bits != nullptr, "fused MLP needs precomputed dropout bits");
  if (drop_post.p > 0.f) B200ST_CHECK(drop_post.bits != nullptr, "fused MLP needs precomputed dropout bits");
  const int m_tiles = ceil_div(M, BM), chunks = ffn / 128;
  int splits = 1;
  B200ST_TRY(mlp_splits(M, ffn, &splits));
  MlpParams p{};
  p.M = M; p.d = d; p.ffn = ffn; p.splits = splits; p.chunks_per_cta = chunks / splits;
  p.b1 = b1; p.b2 = b2; p.drop_ffn = drop_ffn; p.drop_post = drop_post;
  p.relu = 1; p.alpha = 1.f; p.mask_src = nullptr; p.mask_ld = 0; p.tickets = tickets;
  p.idesc_g1 = ptx::make_idesc_16(128, 0, 1, dtype == BF16, dtype == BF16);
  p.idesc_g2 = ptx::make_idesc_16(d, 0, 1, dtype == BF16, dtype == BF16);
  CUtensorMap tx, tw1, tw2, tf1, tout;
  B200ST_TRY(make_operand_map(GemmOperand{X, dtype, 0, d, 0, 0}, M, d, 1, 1, BM, &tx));
  B200ST_TRY(make_operand_map(GemmOperand{W1, dtype, 1, ffn, 0, 0}, ffn, d, 1, 1, 64, &tw1));
  B200ST_TRY(make_operand_map(GemmOperand{W2, dtype, 1, d, 0, 0}, d, ffn, 1, 1, 64, &tw2));
  B200ST_TRY(make_out_map(F1, dtype, ffn, M, 1, 1, ffn, 0, 0, &tf1));
  B200ST_TRY(make_out_map(x_out, F32, d, M, 1, 1, d, 0, 0, &tout));
  auto kern = dtype == F16 ? fused_mlp_fwd_kernel<F16, true> : fused_mlp_fwd_kernel<BF16, true>;
  static bool attr[2] = {false, false};
  if (!attr[dtype == F16]) {
    B200ST_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMlpSmem));
    attr[dtype == F16] = true;
  }
  launch_pdl(kern, m_tiles * splits, kThreads, kMlpSmem, stream, tx, tw1, tw2, tf1, tout, p);
  ++g_launches;
  B200ST_LAUNCH_CHECK();
  if (splits_out) *splits_out = splits;
  return 0;
}

// Fused FFN backward, data-gradient chain: dF1 = scale * (dY W2^T) masked by (F1 > 0)  [written for the W1 weight gradient],
// dH += dF1 W1^T (fp32 reduce-add into what dH holds; the model zero-initialises it).  Same kernel, weights read as K-major B operands.
int fused_mlp_bwd(const void* dY, int dtype, int M, int d, int ffn, const void* W1, const void* W2, const void* F1, float scale,
                  void* dF1, float* dH, cudaStream_t stream, int* tickets, int* splits_out) {
  if (ablate_mask() & ABL_MLP_BWD) return 0;
  B200ST_CHECK(fused_mlp_supported(M, d, ffn, dtype), "fused MLP: unsupported shape / dtype");
  const int m_tiles = ceil_div(M, BM), chunks = ffn / 128;
  int splits = 1;
  B200ST_TRY(mlp_splits(M, ffn, &splits));
  MlpParams p{};
  p.M = M; p.d = d; p.ffn = ffn; p.splits = splits; p.chunks_per_cta = chunks / splits;
  p.b1 = nullptr; p.b2 = nullptr; p.drop_ffn = no_dropout(); p.drop_post = no_dropout();
  p.relu = 0; p.alpha = scale; p.mask_src = F1; p.mask_ld = ffn; p.tickets = tickets;
  p.idesc_g1 = ptx::make_idesc_16(128, 0, 0, dtype == BF16, dtype == BF16);
  p.idesc_g2 = ptx::make_idesc_16(d, 0, 0, dtype == BF16, dtype == BF16);
  CUtensorMap tx, tw1, tw2, tf1, tout;
  B200ST_TRY(make_operand_map(GemmOperand{dY, dtype, 0, d, 0, 0}, M, d, 1, 1, BM, &tx));
  B200ST_TRY(make_operand_map(GemmOperand{W2, dtype, 0, d, 0, 0}, ffn, d, 1, 1, 128, &tw1));     // G1: rows = hidden units, k = d
  B200ST_TRY(make_operand_map(GemmOperand{W1, dtype, 0, ffn, 0, 0}, d, ffn, 1, 1, d, &tw2));      // G2: rows = model dims, k = hidden
  B200ST_TRY(make_out_map(dF1, dtype, ffn, M, 1, 1, ffn, 0, 0, &tf1));
  B200ST_TRY(make_out_map(dH, F32, d, M, 1, 1, d, 0, 0, &tout));
  auto kern = dtype == F16 ? fused_mlp_fwd_kernel<F16, false> : fused_mlp_fwd_kernel<BF16, false>;
  static bool attr[2] = {false, false};
  if (!attr[dtype == F16]) {
    B200ST_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMlpSmem));
    attr[dtype == F16] = true;
  }
  launch_pdl(kern, m_tiles * splits, kThreads, kMlpSmem, stream, tx, tw1, tw2, tf1, tout, p);
  ++g_launches;
  B200ST_LAUNCH_CHECK();
  if (splits_out) *splits_out = splits;
  return 0;
}

void tc_profile_begin() {
  g_prof_recs.clear();
  g_prof = true;
}
bool tc_profile_active() { return g_prof; }
int tc_profile_end(double* ms, double* flops, int64_t* launches) {
  g_prof = false;
  constexpr int kReps = 4;
  double tms = 0, tf = 0;
  FILE* dump = getenv("B200ST_PROFILE_CSV") ? fopen(getenv("B200ST_PROFILE_CSV"), "w") : nullptr;
  if (dump) fprintf(dump, "M,N,K,batch,bn,splitk,a_mn,b_mn,epi,us,tflops\n");
  cudaEvent_t e0, e1;
  B200ST_CUDA(cudaEventCreate(&e0));
  B200ST_CUDA(cudaEventCreate(&e1));
  std::vector<ProfRec> recs;
  recs.swap(g_prof_recs);
  for (const ProfRec& r : recs) {
    const cudaStream_t st = r.stream;
    GemmArgs grp_args[4];
    grp_args[0] = r.g;
    for (int i = 1; i < r.group_n; ++i) grp_args[i] = r.rest[i - 1];
    auto run = [&]() -> int {
      if (r.has_conv) return gemm_tc_impl(r.g, st, &r.conv);
      return r.group_n > 1 ? gemm_wgrad_group(grp_args, r.group_n, st) : gemm_tc_bf16(r.g, st);
    };
    B200ST_TRY(run());                                          // warm-up (tensor maps, instruction cache)
    B200ST_CUDA(cudaEventRecord(e0, st));
    for (int i = 0; i < kReps; ++i) B200ST_TRY(run());
    B200ST_CUDA(cudaEventRecord(e1, st));
    B200ST_CUDA(cudaEventSynchronize(e1));
    float t = 0.f;
    B200ST_CUDA(cudaEventElapsedTime(&t, e0, e1));
    t /= kReps;
    double fl = 2.0 * (double)r.g.M * r.g.N * r.g.K * (double)r.g.nb1 * r.g.nb2;
    for (int i = 1; i < r.group_n; ++i) fl += 2.0 * (double)grp_args[i].M * grp_args[i].N * grp_args[i].K;
    const int epi = (r.g.epi.bias ? 1 : 0) | (r.g.epi.relu ? 2 : 0) | (r.g.epi.mask_src ? 4 : 0) | (r.g.epi.drop.p > 0.f ? 8 : 0) |
                    (r.g.epi.residual ? 16 : 0) | (r.g.c_dtype == F32 ? 32 : 0);
    if (dump) fprintf(dump, "%d,%d,%d,%d,%d,%d,%d,%d,%d,%.2f,%.1f\n", r.g.M, r.g.N, r.g.K, r.group_n > 1 ? -r.group_n : r.g.nb1 * r.g.nb2, r.bn,
                      r.splitk, r.g.A.mn_major, r.g.B.mn_major, epi, t * 1e3, fl / (t * 1e-3) / 1e12);   // batch = -n: grouped launch of n products (first one listed)
    tms += t; tf += fl;
  }
  if (dump) fclose(dump);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  if (ms) *ms = tms;
  if (flops) *flops = tf;
  if (launches) *launches = (int64_t)recs.size();
  return 0;
}

}  // namespace b200st
