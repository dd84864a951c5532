// Flash attention backward on tcgen05/TMEM (sm_100a), head_dim 64, non-causal.
// Autograd of eager_attention_forward (reference modeling_videomae.py:196-223):
//   P = softmax(Q K^T * scale) ; O = P V ; D = rowsum(dO . O)
//   dV = P^T dO ; dP = dO V^T ; dS = P . (dP - D) * scale ; dK = dS^T Q ; dQ = dS K
//
// DEFAULT: flash_attn_bwd_fused_kernel (further down) — ONE pass per (key block, query block) pair, dQ summed across key
// blocks by fp32 bulk reductions.  DETERMINISTIC MODE: the two kernels below, both "pure TMEM" (no thread-written operand
// tiles, no atomics -> bit-deterministic):
//
//  flash_attn_bwd_dkdv_kernel : one CTA owns 128 keys (K_j, V_j in smem) and streams the query blocks i.
//        S^T  = K_j Q_i^T   (SS)  TMEM [0,128)        dP^T = V_j dO_i^T  (SS)  TMEM [128,256)     key index = TMEM lane
//        (both with a fifth K-step that subtracts lse/scale resp. D inside the product: see the fused kernel)
//        P^T, dS^T -> bf16 -> TMEM [256,320), [320,384)
//        dV  += P^T  dO_i   (TS, B = dO_i tile read MN-major)  TMEM [384,448)
//        dK  += dS^T Q_i    (TS, B = Q_i  tile read MN-major)  TMEM [448,512)
//  flash_attn_bwd_dq_kernel   : one CTA owns 128 queries (Q_i, dO_i in smem) and streams the key blocks j.
//        S = Q_i K_j^T (SS) [0,128)   dP = dO_i V_j^T (SS) [128,256)   dS -> bf16 -> TMEM [256,320)   query = TMEM lane
//        dQ += dS K_j  (TS, B = K_j tile read MN-major)  TMEM [320,384)
// Recomputing S/dP in the second kernel costs 2 extra products and a second set of exponentials per tile pair; the fused
// kernel avoids both at the price of an order-dependent fp32 dQ reduction (profiles/r02_attn_notes.md).
// Roles in both: warp 0 lane 0 TMA producer; warp 1 lane 0 issues the score products, warp 3 lane 0 the gradient
// products; warp 2 stages lse/D (dkdv only); warpgroups 1,2 = 256 math threads, thread = TMEM lane, each warpgroup takes
// 64 of the 128 score columns.  Scores of block n+1 and the gradient products of block n run under the math of block n+1.
#include "common.cuh"
#include "../../include/smbv_b200.h"

namespace smbv {

constexpr uint32_t EX2_EMU_PAIRS = 0xA4A4u;  // pairs (of every 16) whose exponentials run on the FMA / ALU pipes instead of MUFU
constexpr int AB_THREADS = 384;
constexpr int AB_TILE = 128 * 64 * 2;  // 16 KB
constexpr int AB_STAGES = 5;  // K/V (dQ kernel) or Q/dO (dK/dV kernel) prefetch depth: a 32 KB block takes ~1700 cycles from L2 under load
constexpr int AB_SMEM = AB_TILE * (2 + 2 * AB_STAGES) + AB_STAGES * 1024 + 1024 + 256;

constexpr int AF_XT = 128 * 16 * 2;  // 4 KB: one [128 x 16] bf16 K-major, NON-swizzled operand tile (the fifth K-step of the score products)
constexpr int DK_STAGES = 4;         // dK/dV kernel: Q/dO prefetch depth (one less than the dQ kernel: the statistic tiles need the room)
constexpr int DK_SMEM = AB_TILE * (2 + 2 * DK_STAGES) + (1 + 2 * DK_STAGES) * AF_XT + 1024 + 256;

// fp32 value as three bf16 terms (hi + mid + lo reproduces it to fp32 accuracy), the first three K entries of an operand row
__device__ __forceinline__ uint4 split3_bf16(float v) {
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  const float r1 = v - __bfloat162float(h);
  const __nv_bfloat16 m = __float2bfloat16_rn(r1);
  const __nv_bfloat16 l = __float2bfloat16_rn(r1 - __bfloat162float(m));
  return make_uint4((uint32_t)__bfloat16_as_ushort(h) | ((uint32_t)__bfloat16_as_ushort(m) << 16), (uint32_t)__bfloat16_as_ushort(l), 0u, 0u);
}

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__global__ void __launch_bounds__(AB_THREADS, 1)
flash_attn_bwd_dkdv_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                           const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmDO, int H, int N,
                           float scale, const float* __restrict__ lse, const float* __restrict__ Dsum,
                           __nv_bfloat16* __restrict__ dk, __nv_bfloat16* __restrict__ dv, int zero) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sK = smem;
  uint8_t* sV = sK + AB_TILE;
  uint8_t* sQ = sV + AB_TILE;                   // DK_STAGES tiles
  uint8_t* sDO = sQ + DK_STAGES * AB_TILE;      // DK_STAGES tiles
  // softmax statistics through a fifth K-step of the score products (see the fused kernel below): no statistic loads in the math loop
  uint8_t* sX1 = sDO + DK_STAGES * AB_TILE;      // the ones tile [1 1 1 0 ... 0] per key row
  uint8_t* sXL = sX1 + AF_XT;                    // [DK_STAGES] -lse/scale of the stage's 128 queries (3-term bf16 split)
  uint8_t* sXD = sXL + DK_STAGES * AF_XT;        // [DK_STAGES] -D
  uint64_t* bars = reinterpret_cast<uint64_t*>(sXD + DK_STAGES * AF_XT);
  uint64_t* kv_full = bars;                        // 1
  uint64_t* qdo_full = kv_full + 1;                // [STAGES] count 2: TMA (expect_tx) + stats warp
  uint64_t* qdo_empty = qdo_full + DK_STAGES;      // [STAGES] count 2 (one commit from each MMA issuer)
  // every score / product barrier exists once per 64-column HALF of the tile = once per math warpgroup, so the two
  // warpgroups run as two independent, naturally staggered pipelines (one's TMEM load / store phases fall into the
  // other's MUFU phase) instead of in lockstep
  uint64_t* s_full = qdo_empty + DK_STAGES;        // [2] 1
  uint64_t* s_free = s_full + 2;                   // [2] 4 warps
  uint64_t* p_full = s_free + 2;                   // [2] 4 warps
  uint64_t* pd_done = p_full + 2;                  // [2] 1: the gradient products of that half have retired
  uint64_t* acc_full = pd_done + 2;                // 1
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kv0 = blockIdx.x * 128;
  const int bh = blockIdx.y;
  const int nq = (N + 127) / 128;
  const float scale_log2 = scale * 1.4426950408889634f;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmDO);
    mbar_init(smem_u32(kv_full), 1);
    for (int s = 0; s < DK_STAGES; ++s) mbar_init(smem_u32(&qdo_full[s]), 2), mbar_init(smem_u32(&qdo_empty[s]), 2);
    for (int w = 0; w < 2; ++w) {
      mbar_init(smem_u32(&s_full[w]), 1);
      mbar_init(smem_u32(&s_free[w]), 4);
      mbar_init(smem_u32(&p_full[w]), 4);
      mbar_init(smem_u32(&pd_done[w]), 1);
    }
    mbar_init(smem_u32(acc_full), 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t T_ST = tmem_base, T_DPT = tmem_base + 128, T_PT = tmem_base + 256, T_DST = tmem_base + 320,
                 T_DV = tmem_base + 384, T_DK = tmem_base + 448;

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
    if (warp == 0 && lane == 0) {  // ===== TMA producer =====
      mbar_expect_tx(smem_u32(kv_full), 2 * AB_TILE);
      tma_load_3d(smem_u32(sK), &tmK, smem_u32(kv_full), 0, kv0, bh);
      tma_load_3d(smem_u32(sV), &tmV, smem_u32(kv_full), 0, kv0, bh);
      uint32_t s = 0, ph = 0;
      for (int i = 0; i < nq; ++i) {
        mbar_wait(smem_u32(&qdo_empty[s]), ph ^ 1);
        mbar_expect_tx(smem_u32(&qdo_full[s]), 2 * AB_TILE);
        tma_load_3d(smem_u32(sQ + s * AB_TILE), &tmQ, smem_u32(&qdo_full[s]), 0, i * 128, bh);
        tma_load_4d(smem_u32(sDO + s * AB_TILE), &tmDO, smem_u32(&qdo_full[s]), 0, i * 128, bh % H, bh / H);
        if (++s == DK_STAGES) s = 0, ph ^= 1;
      }
    } else if (warp == 2) {  // ===== statistics: -lse/scale and -D of the stage's 128 queries as MMA operand rows, 4 per lane =====
#pragma unroll
      for (int q = 0; q < 4; ++q) {  // once: the ones tile and the k = 8..15 halves (always zero) of every stage tile
        const int r = lane * 4 + q;
        const uint32_t off = (uint32_t)((r >> 3) * 256 + (r & 7) * 16);
        *reinterpret_cast<uint4*>(sX1 + off) = make_uint4(0x3F803F80u, 0x00003F80u, 0u, 0u);  // bf16 1, 1, 1, 0 ...
        *reinterpret_cast<uint4*>(sX1 + off + 128) = make_uint4(0u, 0u, 0u, 0u);
        for (int st = 0; st < 2 * DK_STAGES; ++st) *reinterpret_cast<uint4*>(sXL + st * AF_XT + off + 128) = make_uint4(0u, 0u, 0u, 0u);
      }
      const float neg_inv_scale = -1.f / scale;
      uint32_t s = 0, ph = 0;
      for (int i = 0; i < nq; ++i) {
        mbar_wait(smem_u32(&qdo_empty[s]), ph ^ 1);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int r = lane * 4 + q, row = i * 128 + r;
          const bool ok = row < N;
          // out-of-range query rows: a huge negative score offset -> P = 0, so they contribute nothing to dK / dV
          const float L = ok ? lse[(int64_t)bh * N + row] * neg_inv_scale : -1e30f;
          const float Dn = ok ? -Dsum[(int64_t)bh * N + row] : 0.f;
          const uint32_t off = (uint32_t)(s * AF_XT + (r >> 3) * 256 + (r & 7) * 16);
          *reinterpret_cast<uint4*>(sXL + off) = split3_bf16(L);
          *reinterpret_cast<uint4*>(sXD + off) = split3_bf16(Dn);
        }
        fence_proxy_async_smem();  // generic-proxy stores -> visible to the tensor core's (async proxy) operand reads
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&qdo_full[s]));
        if (++s == DK_STAGES) s = 0, ph ^= 1;
      }
    } else if (warp == 1 && elect_one()) {  // ===== MMA issuer A: the score products S^T, dP^T, one 64-query half at a time =====
      constexpr uint32_t id_s = umma_idesc(UMMA_BF16, 128, 128, 0, 0);
      const uint64_t dK_k = umma_desc(smem_u32(sK), 16, 1024, UMMA_SW_128B);
      const uint64_t dV_k = umma_desc(smem_u32(sV), 16, 1024, UMMA_SW_128B);
      const uint64_t dQ_k = umma_desc(smem_u32(sQ), 16, 1024, UMMA_SW_128B);
      const uint64_t dDO_k = umma_desc(smem_u32(sDO), 16, 1024, UMMA_SW_128B);
      const uint64_t dX1 = umma_desc(smem_u32(sX1), 128, 256, UMMA_SW_NONE);
      const uint64_t dXL = umma_desc(smem_u32(sXL), 128, 256, UMMA_SW_NONE);
      const uint64_t dXD = umma_desc(smem_u32(sXD), 128, 256, UMMA_SW_NONE);
      mbar_wait(smem_u32(kv_full), 0);
      uint32_t s = 0, ph = 0;
      for (int i = 0; i < nq; ++i) {
        mbar_wait(smem_u32(&qdo_full[s]), ph);
        if (i > 0) {  // both halves of block i-1 are in registers
          mbar_wait(smem_u32(&s_free[0]), (i - 1) & 1);
          mbar_wait(smem_u32(&s_free[1]), (i - 1) & 1);
        }
        tc_fence_after();
        const uint64_t off = (uint64_t)((s * AB_TILE) >> 4), xoff = (uint64_t)((s * AF_XT) >> 4);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_f16_ss(T_ST, dK_k + 2 * k, dQ_k + off + 2 * k, id_s, k != 0);
        umma_f16_ss(T_ST, dX1, dXL + xoff, id_s, 1);   // fifth K-step: S^T - lse/scale
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_f16_ss(T_DPT, dV_k + 2 * k, dDO_k + off + 2 * k, id_s, k != 0);
        umma_f16_ss(T_DPT, dX1, dXD + xoff, id_s, 1);  // fifth K-step: dP^T - D
        umma_commit(smem_u32(&s_full[0]));     // both math warpgroups wait on this one (N = 128: half the MMA issues)
        umma_commit(smem_u32(&qdo_empty[s]));  // (second arrival comes from issuer B)
        if (++s == DK_STAGES) s = 0, ph ^= 1;
      }
    } else if (warp == 3 && elect_one()) {  // ===== MMA issuer B: dV += P^T dO_i, dK += dS^T Q_i, per half =====
      constexpr uint32_t id_g = umma_idesc(UMMA_BF16, 128, 64, 0, 1);  // A in TMEM, B tile read MN-major
      const uint64_t dQ_mn = umma_desc(smem_u32(sQ), AB_TILE, 1024, UMMA_SW_128B);
      const uint64_t dDO_mn = umma_desc(smem_u32(sDO), AB_TILE, 1024, UMMA_SW_128B);
      uint32_t s = 0;
      for (int i = 0; i < nq; ++i) {
        const uint64_t off = (uint64_t)((s * AB_TILE) >> 4);
#pragma unroll
        for (int w = 0; w < 2; ++w) {
          mbar_wait(smem_u32(&p_full[w]), i & 1);
          tc_fence_after();
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int kk = w * 4 + k;  // 16-query reduction step
            umma_f16_ts(T_DV, T_PT + kk * 8, dDO_mn + off + (uint64_t)(kk * 128), id_g, (i | kk) != 0);
          }
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int kk = w * 4 + k;
            umma_f16_ts(T_DK, T_DST + kk * 8, dQ_mn + off + (uint64_t)(kk * 128), id_g, (i | kk) != 0);
          }
          umma_commit(smem_u32(&pd_done[w]));
        }
        umma_commit(smem_u32(&qdo_empty[s]));
        if (++s == DK_STAGES) s = 0;
      }
      umma_commit(smem_u32(acc_full));
    }
    __syncwarp();
  } else {  // ===== the two math warpgroups: thread = key row, warpgroup = 64 query columns =====
    asm volatile("setmaxnreg.inc.sync.aligned.u32 216;");
    int n_local = N;  // re-derived inside this register region (see DESIGN.md: setmaxnreg + live-through scalars)
    asm volatile("" : "+r"(n_local));
    const int nq_m = (n_local + 127) / 128;
    const int wg = (warp >> 2) - 1;
    const int quad = warp & 3;
    const int r = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    const bool kv_ok = kv0 + r < n_local;
    const uint64_t sc2_c = pack2(scale_log2, scale_log2);
    uint32_t s = 0;
    for (int i = 0; i < nq_m; ++i) {
      mbar_wait(smem_u32(&s_full[0]), i & 1);  // also implies stage s (lse, D) has landed (issuer A waited on qdo_full)
      tc_fence_after();
      uint32_t pp[32], dd[32];
      // pull this warpgroup's 64 columns of S^T and dP^T into registers first and release the TMEM columns at once:
      // the next block's score products then run under this block's math
      uint32_t sv[64], dpv[64];
      tmem_ld32(T_ST + lane_base + wg * 64, *reinterpret_cast<uint32_t(*)[32]>(&sv[0]));
      tmem_ld32(T_ST + lane_base + wg * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&sv[32]));
      tmem_ld32(T_DPT + lane_base + wg * 64, *reinterpret_cast<uint32_t(*)[32]>(&dpv[0]));
      tmem_ld32(T_DPT + lane_base + wg * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&dpv[32]));
      tmem_wait_ld();
      tc_fence_before();
      __syncwarp();
      // the token dependency keeps ptxas from hoisting the exponentials above the arrive (see the dQ kernel)
      uint32_t tok = 0;
      if (lane == 0) tok = mbar_arrive_tok(smem_u32(&s_free[wg]));
      const float zf = __uint_as_float(tok & (uint32_t)zero);  // +0.0f at run time
      const uint64_t sc2 = fadd2(sc2_c, pack2(zf, zf));
#pragma unroll
      for (int c = 0; c < 4; ++c) {
#pragma unroll
        for (int q = 0; q < 8; ++q) {  // packed f32x2 math: one FFMA2 / FADD2 / FMUL2 per PAIR of elements
          const int col = c * 16 + 2 * q;
          // sv = S^T - lse/scale, dpv = dP^T - D (the statistics came in through the fifth K-step of the score products)
          const uint64_t x2 = fmul2(pack2(__uint_as_float(sv[col]), __uint_as_float(sv[col + 1])), sc2);
          float p0, p1;  // key rows past N (zero K/V rows) only feed accumulator rows that are never stored
          if ((EX2_EMU_PAIRS >> ((c * 8 + q) & 15)) & 1u) {
            ex2_emu2(x2, p0, p1);
          } else {
            float a0, a1;
            unpack2(x2, a0, a1);
            p0 = ex2f(a0), p1 = ex2f(a1);
          }
          const uint64_t p2 = pack2(p0, p1);
          // dS^T without the softmax scale: it is applied once to dK in the epilogue
          float d0, d1;
          unpack2(fmul2(p2, pack2(__uint_as_float(dpv[col]), __uint_as_float(dpv[col + 1]))), d0, d1);
          pp[c * 8 + q] = pack_bf16(p0, p1);
          dd[c * 8 + q] = pack_bf16(d0, d1);
        }
      }
      // the gradient products of block i-1 read P^T / dS^T from TMEM: they must have retired before we overwrite them
      // (issued a whole math phase ago, so this wait is normally free)
      if (i > 0) {
        mbar_wait(smem_u32(&pd_done[wg]), (i - 1) & 1);
        tc_fence_after();
      }
      tmem_st32(T_PT + lane_base + wg * 32, pp);
      tmem_st32(T_DST + lane_base + wg * 32, dd);
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&p_full[wg]));
      if (++s == DK_STAGES) s = 0;
    }
    // ---- epilogue: warpgroup 0 writes dV_j, warpgroup 1 writes dK_j (bf16, head-major [BH, N, 64]) ----
    mbar_wait(smem_u32(acc_full), 0);
    tc_fence_after();
    __nv_bfloat16* outp = (wg == 0 ? dv : dk) + ((int64_t)bh * n_local + kv0 + r) * 64;
    const uint32_t tacc = (wg == 0 ? T_DV : T_DK) + lane_base;
    const float osc = wg == 0 ? 1.f : scale;  // dK = scale * (unscaled dS)^T Q
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      uint32_t o[32];
      tmem_ld32(tacc + c * 32, o);
      tmem_wait_ld();
#pragma unroll
      for (int q = 0; q < 32; ++q) o[q] = __float_as_uint(__uint_as_float(o[q]) * osc);
      if (kv_ok) {
        uint4* dst = reinterpret_cast<uint4*>(outp + c * 32);
#pragma unroll
        for (int q = 0; q < 4; ++q)
          dst[q] = make_uint4(pack_bf16(__uint_as_float(o[8 * q]), __uint_as_float(o[8 * q + 1])),
                              pack_bf16(__uint_as_float(o[8 * q + 2]), __uint_as_float(o[8 * q + 3])),
                              pack_bf16(__uint_as_float(o[8 * q + 4]), __uint_as_float(o[8 * q + 5])),
                              pack_bf16(__uint_as_float(o[8 * q + 6]), __uint_as_float(o[8 * q + 7])));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------------------------
// dQ kernel: CTA = 128 queries, streams key blocks
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(AB_THREADS, 1)
flash_attn_bwd_dq_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                         const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmDO, int H, int N,
                         float scale, const float* __restrict__ lse, const float* __restrict__ Dsum,
                         __nv_bfloat16* __restrict__ dq, int zero) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sDO = sQ + AB_TILE;
  uint8_t* sK = sDO + AB_TILE;                  // AB_STAGES tiles
  uint8_t* sV = sK + AB_STAGES * AB_TILE;       // AB_STAGES tiles
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + AB_STAGES * AB_TILE);
  uint64_t* q_full = bars;                         // 1
  uint64_t* k_full = q_full + 1;                   // [STAGES]
  uint64_t* k_empty = k_full + AB_STAGES;          // [STAGES] count 2 (scores + dQ product both read K_j)
  uint64_t* v_full = k_empty + AB_STAGES;          // [STAGES]
  uint64_t* v_empty = v_full + AB_STAGES;          // [STAGES] count 1
  uint64_t* s_full = v_empty + AB_STAGES;          // [2] per 64-key half / math warpgroup (see the dK/dV kernel)
  uint64_t* s_free = s_full + 2;                   // [2] 4 warps
  uint64_t* p_full = s_free + 2;                   // [2] 4 warps
  uint64_t* pd_done = p_full + 2;                  // [2]
  uint64_t* acc_full = pd_done + 2;                // 1
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * 128;
  const int bh = blockIdx.y;
  const int nkv = (N + 127) / 128;
  const float scale_log2 = scale * 1.4426950408889634f;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmDO);
    mbar_init(smem_u32(q_full), 1);
    for (int s = 0; s < AB_STAGES; ++s) {
      mbar_init(smem_u32(&k_full[s]), 1), mbar_init(smem_u32(&k_empty[s]), 2);
      mbar_init(smem_u32(&v_full[s]), 1), mbar_init(smem_u32(&v_empty[s]), 1);
    }
    for (int w = 0; w < 2; ++w) {
      mbar_init(smem_u32(&s_full[w]), 1);
      mbar_init(smem_u32(&s_free[w]), 4);
      mbar_init(smem_u32(&p_full[w]), 4);
      mbar_init(smem_u32(&pd_done[w]), 1);
    }
    mbar_init(smem_u32(acc_full), 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t T_S = tmem_base, T_DP = tmem_base + 128, T_DS = tmem_base + 256, T_DQ = tmem_base + 320;

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
    if (warp == 0 && lane == 0) {  // ===== TMA producer =====
      mbar_expect_tx(smem_u32(q_full), 2 * AB_TILE);
      tma_load_3d(smem_u32(sQ), &tmQ, smem_u32(q_full), 0, q0, bh);
      tma_load_4d(smem_u32(sDO), &tmDO, smem_u32(q_full), 0, q0, bh % H, bh / H);
      uint32_t s = 0, ph = 0;
      for (int j = 0; j < nkv; ++j) {
        mbar_wait(smem_u32(&k_empty[s]), ph ^ 1);
        mbar_expect_tx(smem_u32(&k_full[s]), AB_TILE);
        tma_load_3d(smem_u32(sK + s * AB_TILE), &tmK, smem_u32(&k_full[s]), 0, j * 128, bh);
        mbar_expect_tx(smem_u32(&v_full[s]), AB_TILE);
        tma_load_3d(smem_u32(sV + s * AB_TILE), &tmV, smem_u32(&v_full[s]), 0, j * 128, bh);
        if (++s == AB_STAGES) s = 0, ph ^= 1;
      }
    } else if (warp == 1 && elect_one()) {  // ===== MMA issuer A: S = Q K_j^T, dP = dO V_j^T for the whole 128-key block =====
      // A tcgen05.mma costs the issuing thread ~75 cycles regardless of its size (timeline trace, profiles/r01_attn_notes.md):
      // with 64-key halves (N = 64, 32 tensor-pipe cycles each) the 16 issues + 4 commits per block WERE the 1790-cycle block
      // period.  N = 128 halves the issue count; one commit serves both math warpgroups.
      constexpr uint32_t id_s = umma_idesc(UMMA_BF16, 128, 128, 0, 0);
      const uint64_t dQ_k = umma_desc(smem_u32(sQ), 16, 1024, UMMA_SW_128B);
      const uint64_t dDO_k = umma_desc(smem_u32(sDO), 16, 1024, UMMA_SW_128B);
      const uint64_t dK_k = umma_desc(smem_u32(sK), 16, 1024, UMMA_SW_128B);
      const uint64_t dV_k = umma_desc(smem_u32(sV), 16, 1024, UMMA_SW_128B);
      mbar_wait(smem_u32(q_full), 0);
      uint32_t s = 0, ph = 0;
      for (int j = 0; j < nkv; ++j) {
        mbar_wait(smem_u32(&k_full[s]), ph);
        mbar_wait(smem_u32(&v_full[s]), ph);
        if (j > 0) {  // both halves of block j-1 are in registers
          mbar_wait(smem_u32(&s_free[0]), (j - 1) & 1);
          mbar_wait(smem_u32(&s_free[1]), (j - 1) & 1);
        }
        tc_fence_after();
        const uint64_t off = (uint64_t)((s * AB_TILE) >> 4);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_f16_ss(T_S, dQ_k + 2 * k, dK_k + off + 2 * k, id_s, k != 0);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_f16_ss(T_DP, dDO_k + 2 * k, dV_k + off + 2 * k, id_s, k != 0);
        umma_commit(smem_u32(&s_full[0]));      // both math warpgroups wait on this one
        umma_commit(smem_u32(&k_empty[s]));     // (second arrival: issuer B; V_j is only read here, so k_empty covers it too)
        if (++s == AB_STAGES) s = 0, ph ^= 1;
      }
    } else if (warp == 3 && elect_one()) {  // ===== MMA issuer B: dQ += dS K_j, per half =====
      constexpr uint32_t id_g = umma_idesc(UMMA_BF16, 128, 64, 0, 1);
      const uint64_t dK_mn = umma_desc(smem_u32(sK), AB_TILE, 1024, UMMA_SW_128B);
      uint32_t s = 0;
      for (int j = 0; j < nkv; ++j) {
        const uint64_t off = (uint64_t)((s * AB_TILE) >> 4);
#pragma unroll
        for (int w = 0; w < 2; ++w) {
          mbar_wait(smem_u32(&p_full[w]), j & 1);
          tc_fence_after();
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int kk = w * 4 + k;
            umma_f16_ts(T_DQ, T_DS + kk * 8, dK_mn + off + (uint64_t)(kk * 128), id_g, (j | kk) != 0);
          }
          umma_commit(smem_u32(&pd_done[w]));
        }
        umma_commit(smem_u32(&k_empty[s]));
        if (++s == AB_STAGES) s = 0;
      }
      umma_commit(smem_u32(acc_full));
    }
    __syncwarp();
  } else {  // ===== math: thread = query row, warpgroup = 64 key columns =====
    asm volatile("setmaxnreg.inc.sync.aligned.u32 216;");
    int n_local = N;
    asm volatile("" : "+r"(n_local));
    const int nkv_m = (n_local + 127) / 128;
    const int wg = (warp >> 2) - 1;
    const int quad = warp & 3;
    const int r = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    const int qrow = q0 + r;
    const bool q_ok = qrow < n_local;
    // out-of-range query rows: lse = +inf -> P = 0
    const float neg_l2 = q_ok ? -lse[(int64_t)bh * n_local + qrow] * 1.4426950408889634f : -INFINITY;
    const float dsum = q_ok ? Dsum[(int64_t)bh * n_local + qrow] : 0.f;
    const uint64_t sc2 = pack2(scale_log2, scale_log2), nl2_row = pack2(neg_l2, neg_l2), nds2 = pack2(-dsum, -dsum);
    for (int j = 0; j < nkv_m; ++j) {
      mbar_wait(smem_u32(&s_full[0]), j & 1);
      tc_fence_after();
      uint32_t dd[32];
      uint32_t sv[64], dpv[64];
      tmem_ld32(T_S + lane_base + wg * 64, *reinterpret_cast<uint32_t(*)[32]>(&sv[0]));
      tmem_ld32(T_S + lane_base + wg * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&sv[32]));
      tmem_ld32(T_DP + lane_base + wg * 64, *reinterpret_cast<uint32_t(*)[32]>(&dpv[0]));
      tmem_ld32(T_DP + lane_base + wg * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&dpv[32]));
      tmem_wait_ld();
      tc_fence_before();
      __syncwarp();
      // the next block's scores run under this block's math — provided the arrive really precedes the math in the SASS:
      // the token dependency below keeps ptxas from hoisting the exponentials above it (it did: 63 of 64 MUFU.EX2)
      uint32_t tok = 0;
      if (lane == 0) tok = mbar_arrive_tok(smem_u32(&s_free[wg]));
      const float zf = __uint_as_float(tok & (uint32_t)zero);  // +0.0f at run time
      const uint64_t nl2 = fadd2(nl2_row, pack2(zf, zf));
#pragma unroll
      for (int c = 0; c < 4; ++c) {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const int col = c * 16 + 2 * q;
          const uint64_t x2 = ffma2(pack2(__uint_as_float(sv[col]), __uint_as_float(sv[col + 1])), sc2, nl2);
          float a0, a1, p0, p1;
          unpack2(x2, a0, a1);
          if ((EX2_EMU_PAIRS >> ((c * 8 + q) & 15)) & 1u) {
            ex2_emu2(x2, p0, p1);
          } else {
            p0 = ex2f(a0), p1 = ex2f(a1);
          }
          // key rows past N need no masking: TMA zero-fills K_j there, so whatever (finite) dS those columns get is
          // multiplied by zero rows in dQ += dS K_j  (the per-element selects cost 134 of 327 instructions per block)
          float d0, d1;  // dS without the softmax scale: applied once to dQ in the epilogue
          unpack2(fmul2(pack2(p0, p1), fadd2(pack2(__uint_as_float(dpv[col]), __uint_as_float(dpv[col + 1])), nds2)), d0, d1);
          dd[c * 8 + q] = pack_bf16(d0, d1);
        }
      }
      if (j > 0) {
        mbar_wait(smem_u32(&pd_done[wg]), (j - 1) & 1);
        tc_fence_after();
      }
      tmem_st32(T_DS + lane_base + wg * 32, dd);
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&p_full[wg]));
    }
    // ---- epilogue: dQ tile -> bf16 head-major [BH, N, 64]; each warpgroup writes 32 of the 64 columns ----
    mbar_wait(smem_u32(acc_full), 0);
    tc_fence_after();
    uint32_t o[32];
    tmem_ld32(T_DQ + lane_base + wg * 32, o);
    tmem_wait_ld();
    if (q_ok) {
      uint4* dst = reinterpret_cast<uint4*>(dq + ((int64_t)bh * n_local + qrow) * 64 + wg * 32);
#pragma unroll
      for (int q = 0; q < 4; ++q)
        dst[q] = make_uint4(pack_bf16(__uint_as_float(o[8 * q]) * scale, __uint_as_float(o[8 * q + 1]) * scale),
                            pack_bf16(__uint_as_float(o[8 * q + 2]) * scale, __uint_as_float(o[8 * q + 3]) * scale),
                            pack_bf16(__uint_as_float(o[8 * q + 4]) * scale, __uint_as_float(o[8 * q + 5]) * scale),
                            pack_bf16(__uint_as_float(o[8 * q + 6]) * scale, __uint_as_float(o[8 * q + 7]) * scale));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------------------------
// Fused backward ("one pass"): the dK/dV kernel above additionally forms dQ_i = dS_i K_j for every block pair, so S / dP / the
// exponentials are computed ONCE per pair (5 products per pair instead of 4 + 3, half the MUFU work of the two-kernel path).
//   dS^T (bf16) goes to a 128B-swizzled shared-memory tile [2 x (128 keys x 64 queries)] instead of TMEM and is read twice:
//        dK += dS^T Q_i   (SS, A = the tile K-major, B = Q_i tile MN-major)                      TMEM [384,448)
//        dQ_i = dS K_j    (SS, A = the SAME tile MN-major (M = queries), B = K_j tile MN-major)  TMEM [448,512)
//   dQ_i leaves through the math threads one block late: TMEM -> registers -> swizzled fp32 slab -> cp.reduce.async.bulk
//   (.add.f32) into the fp32 accumulator dq_acc [BH, N, 64]; a finishing pass scales and rounds it to bf16.
// The cross-CTA fp32 reduction makes dQ order-dependent in its last bits (dK / dV stay bit-deterministic); the two-kernel path
// remains available as the deterministic mode (smbv_flash_attn_bwd_ex).  Every CTA of a head walks the query blocks from a
// different start so that concurrent reductions land on different accumulator rows.
// ------------------------------------------------------------------------------------------------------------------
constexpr int AF_STAGES = 3;
constexpr int AF_SMEM = AB_TILE * (2 + 2 * AF_STAGES + 2 + 2) + (1 + 2 * AF_STAGES) * AF_XT + 1024 + 256;

// Work decomposition of the fused backward (1-D grid).  Unit u = (key block u % nkv, head u / nkv).  CTAs [0, n_full) take one
// whole unit each (n_full = a multiple of the SM count: complete waves).  The units of the partial last wave are cut into
// `parts` query ranges, one CTA each, so that the last wave costs 1/parts .. of a unit instead of a whole one (960 units on
// 148 SMs: 6.5 rounds instead of 7).  A split CTA leaves fp32 partial dK / dV in part_ws; attn_bwd_combine_kernel sums them.
struct FusedWork {
  int kvblk, bh, qb0, qb1, part;  // part = index of the partial-result slot, -1 for a whole unit
};
__device__ __forceinline__ FusedWork fused_work(int cta, int nkv, int n_full, int parts, int nq_all) {
  FusedWork w;
  int unit = cta;
  w.qb0 = 0, w.qb1 = nq_all, w.part = -1;
  if (cta >= n_full) {
    const int t = cta - n_full, pi = t % parts;
    unit = n_full + t / parts;
    w.qb0 = (int)((int64_t)nq_all * pi / parts);
    w.qb1 = (int)((int64_t)nq_all * (pi + 1) / parts);
    w.part = t;
  }
  w.kvblk = unit % nkv;
  w.bh = unit / nkv;
  return w;
}

__device__ __forceinline__ void tma_reduce_add_3d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.reduce.async.bulk.tensor.3d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(src), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void sts_u4(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}

__global__ void __launch_bounds__(AB_THREADS, 1)
flash_attn_bwd_fused_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                            const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmDO,
                            const __grid_constant__ CUtensorMap tmDQ, int H, int N, float scale,
                            const float* __restrict__ lse, const float* __restrict__ Dsum, __nv_bfloat16* __restrict__ dk,
                            __nv_bfloat16* __restrict__ dv, float* __restrict__ part_ws, int nkv,
                            int n_full, int parts, int zero) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sK = smem;
  uint8_t* sV = sK + AB_TILE;
  uint8_t* sQ = sV + AB_TILE;                   // AF_STAGES tiles
  uint8_t* sDO = sQ + AF_STAGES * AB_TILE;      // AF_STAGES tiles
  uint8_t* sDS = sDO + AF_STAGES * AB_TILE;     // dS^T bf16: 2 sub-tiles [128 keys x 64 queries], one per math warpgroup
  uint8_t* sDQ = sDS + 2 * AB_TILE;             // dQ fp32 slabs: 2 x [128 queries x 32 d], one per math warpgroup
  // The per-query softmax statistics enter through the score products themselves: a fifth K-step (K = 16) multiplies a
  // constant A tile [1 1 1 0 ... 0] (per key row) with a B tile whose query row holds -lse/scale (resp. -D) split into three
  // bf16 terms (hi + mid + lo = the fp32 value), so the accumulators come back as S^T - lse/scale and dP^T - D.  The math
  // threads then need no statistics at all: 64 broadcast LDS.64 per thread and block (40 % of the kernel's shared-memory
  // wavefronts: ncu l1tex__data_pipe_lsu_wavefronts 60 %) and 32 FADD2 disappear; cost: 2 x 64 tensor cycles per block.
  // Tile layout (no swizzle, K-major): element (row, k) at (row/8)*256 + (k/8)*128 + (row%8)*16 + (k%8)*2, LBO 128, SBO 256.
  uint8_t* sX1 = sDQ + 2 * AB_TILE;             // the ones tile
  uint8_t* sXL = sX1 + AF_XT;                   // [AF_STAGES] -lse/scale of the stage's 128 queries
  uint8_t* sXD = sXL + AF_STAGES * AF_XT;       // [AF_STAGES] -D
  uint64_t* bars = reinterpret_cast<uint64_t*>(sXD + AF_STAGES * AF_XT);
  uint64_t* kv_full = bars;                        // 1
  uint64_t* qdo_full = kv_full + 1;                // [STAGES] count 2: TMA (expect_tx) + stats warp
  uint64_t* qdo_empty = qdo_full + AF_STAGES;      // [STAGES] count 2 (one commit from each MMA issuer)
  uint64_t* s_full = qdo_empty + AF_STAGES;        // 1: S^T and dP^T of the block (both warpgroups wait on it)
  uint64_t* s_free = s_full + 1;                   // [2] 4 warps: that half of S^T / dP^T is in registers
  uint64_t* p_full = s_free + 2;                   // [2] 4 warps: P^T (TMEM) and dS^T (smem) of that half are written
  uint64_t* pd_done = p_full + 2;                  // 1: every product that reads P^T / dS^T of the block has retired
  uint64_t* dq_full = pd_done + 1;                 // 1: dQ_i complete in TMEM
  uint64_t* dq_free = dq_full + 1;                 // 8 warps: dQ_i is in registers
  uint64_t* acc_full = dq_free + 1;                // 1
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const FusedWork wk = fused_work((int)blockIdx.x, nkv, n_full, parts, (N + 127) / 128);
  const int kv0 = wk.kvblk * 128;
  const int bh = wk.bh;
  const int nq = wk.qb1 - wk.qb0;  // query blocks this CTA walks: [qb0, qb1), starting at qb0 + q_rot
  const int q_rot = (int)((wk.kvblk * 37u) % (unsigned)nq);
  const float scale_log2 = scale * 1.4426950408889634f;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmDO);
    tma_prefetch_desc(&tmDQ);
    mbar_init(smem_u32(kv_full), 1);
    for (int s = 0; s < AF_STAGES; ++s) mbar_init(smem_u32(&qdo_full[s]), 2), mbar_init(smem_u32(&qdo_empty[s]), 2);
    mbar_init(smem_u32(s_full), 1);
    for (int w = 0; w < 2; ++w) mbar_init(smem_u32(&s_free[w]), 4), mbar_init(smem_u32(&p_full[w]), 4);
    mbar_init(smem_u32(pd_done), 1);
    mbar_init(smem_u32(dq_full), 1);
    mbar_init(smem_u32(dq_free), 8);
    mbar_init(smem_u32(acc_full), 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t T_ST = tmem_base, T_DPT = tmem_base + 128, T_PT = tmem_base + 256, T_DV = tmem_base + 320,
                 T_DK = tmem_base + 384, T_DQ = tmem_base + 448;

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
    if (warp == 0 && lane == 0) {  // ===== TMA producer =====
      mbar_expect_tx(smem_u32(kv_full), 2 * AB_TILE);
      tma_load_3d(smem_u32(sK), &tmK, smem_u32(kv_full), 0, kv0, bh);
      tma_load_3d(smem_u32(sV), &tmV, smem_u32(kv_full), 0, kv0, bh);
      uint32_t s = 0, ph = 0;
      int iq = wk.qb0 + q_rot;
      for (int i = 0; i < nq; ++i) {
        mbar_wait(smem_u32(&qdo_empty[s]), ph ^ 1);
        mbar_expect_tx(smem_u32(&qdo_full[s]), 2 * AB_TILE);
        tma_load_3d(smem_u32(sQ + s * AB_TILE), &tmQ, smem_u32(&qdo_full[s]), 0, iq * 128, bh);
        tma_load_4d(smem_u32(sDO + s * AB_TILE), &tmDO, smem_u32(&qdo_full[s]), 0, iq * 128, bh % H, bh / H);
        if (++s == AF_STAGES) s = 0, ph ^= 1;
        if (++iq == wk.qb1) iq = wk.qb0;
      }
    } else if (warp == 2) {  // ===== statistics: -lse/scale and -D of the stage's 128 queries as MMA operand rows, 4 per lane =====
      {  // once: the ones tile and the k = 8..15 halves (always zero) of every stage tile
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int r = lane * 4 + q;
          const uint32_t off = (uint32_t)((r >> 3) * 256 + (r & 7) * 16);
          *reinterpret_cast<uint4*>(sX1 + off) = make_uint4(0x3F803F80u, 0x00003F80u, 0u, 0u);  // bf16 1, 1, 1, 0 ...
          *reinterpret_cast<uint4*>(sX1 + off + 128) = make_uint4(0u, 0u, 0u, 0u);
          for (int st = 0; st < 2 * AF_STAGES; ++st) *reinterpret_cast<uint4*>(sXL + st * AF_XT + off + 128) = make_uint4(0u, 0u, 0u, 0u);
        }
      }
      const float neg_inv_scale = -1.f / scale;
      uint32_t s = 0, ph = 0;
      int iq = wk.qb0 + q_rot;
      for (int i = 0; i < nq; ++i) {
        mbar_wait(smem_u32(&qdo_empty[s]), ph ^ 1);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int r = lane * 4 + q, row = iq * 128 + r;
          const bool ok = row < N;
          // out-of-range query rows: a huge negative score offset -> P = 0 -> dS = 0: nothing reaches dK / dV / dQ
          const float L = ok ? lse[(int64_t)bh * N + row] * neg_inv_scale : -1e30f;
          const float Dn = ok ? -Dsum[(int64_t)bh * N + row] : 0.f;
          const uint32_t off = (uint32_t)(s * AF_XT + (r >> 3) * 256 + (r & 7) * 16);
          *reinterpret_cast<uint4*>(sXL + off) = split3_bf16(L);
          *reinterpret_cast<uint4*>(sXD + off) = split3_bf16(Dn);
        }
        fence_proxy_async_smem();  // generic-proxy stores -> visible to the tensor core's (async proxy) operand reads
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&qdo_full[s]));
        if (++s == AF_STAGES) s = 0, ph ^= 1;
        if (++iq == wk.qb1) iq = wk.qb0;
      }
    } else if (warp == 1 && elect_one()) {  // ===== MMA issuer A: S^T = K_j Q_i^T, dP^T = V_j dO_i^T =====
      constexpr uint32_t id_s = umma_idesc(UMMA_BF16, 128, 128, 0, 0);
      const uint64_t dK_k = umma_desc(smem_u32(sK), 16, 1024, UMMA_SW_128B);
      const uint64_t dV_k = umma_desc(smem_u32(sV), 16, 1024, UMMA_SW_128B);
      const uint64_t dQ_k = umma_desc(smem_u32(sQ), 16, 1024, UMMA_SW_128B);
      const uint64_t dDO_k = umma_desc(smem_u32(sDO), 16, 1024, UMMA_SW_128B);
      const uint64_t dX1 = umma_desc(smem_u32(sX1), 128, 256, UMMA_SW_NONE);
      const uint64_t dXL = umma_desc(smem_u32(sXL), 128, 256, UMMA_SW_NONE);
      const uint64_t dXD = umma_desc(smem_u32(sXD), 128, 256, UMMA_SW_NONE);
      mbar_wait(smem_u32(kv_full), 0);
      uint32_t s = 0, ph = 0;
      for (int i = 0; i < nq; ++i) {
        mbar_wait(smem_u32(&qdo_full[s]), ph);
        if (i > 0) {  // both halves of block i-1 are in registers
          mbar_wait(smem_u32(&s_free[0]), (i - 1) & 1);
          mbar_wait(smem_u32(&s_free[1]), (i - 1) & 1);
        }
        tc_fence_after();
        const uint64_t off = (uint64_t)((s * AB_TILE) >> 4), xoff = (uint64_t)((s * AF_XT) >> 4);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_f16_ss(T_ST, dK_k + 2 * k, dQ_k + off + 2 * k, id_s, k != 0);
        umma_f16_ss(T_ST, dX1, dXL + xoff, id_s, 1);   // fifth K-step: S^T - lse/scale
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_f16_ss(T_DPT, dV_k + 2 * k, dDO_k + off + 2 * k, id_s, k != 0);
        umma_f16_ss(T_DPT, dX1, dXD + xoff, id_s, 1);  // fifth K-step: dP^T - D
        umma_commit(smem_u32(s_full));
        umma_commit(smem_u32(&qdo_empty[s]));  // (second arrival comes from issuer B)
        if (++s == AF_STAGES) s = 0, ph ^= 1;
      }
    } else if (warp == 3 && elect_one()) {  // ===== MMA issuer B: dV, dK per half, then dQ_i for the whole block =====
      constexpr uint32_t id_g = umma_idesc(UMMA_BF16, 128, 64, 0, 1);  // A K-major (TMEM / dS^T tile), B tile MN-major
      constexpr uint32_t id_q = umma_idesc(UMMA_BF16, 128, 64, 1, 1);  // A = dS^T tile read MN-major, B = K_j MN-major
      const uint64_t dQ_mn = umma_desc(smem_u32(sQ), AB_TILE, 1024, UMMA_SW_128B);
      const uint64_t dDO_mn = umma_desc(smem_u32(sDO), AB_TILE, 1024, UMMA_SW_128B);
      const uint64_t dDS_k = umma_desc(smem_u32(sDS), 16, 1024, UMMA_SW_128B);
      const uint64_t dDS_mn = umma_desc(smem_u32(sDS), AB_TILE, 1024, UMMA_SW_128B);  // LBO = the next 64-query sub-tile
      const uint64_t dK_mn = umma_desc(smem_u32(sK), AB_TILE, 1024, UMMA_SW_128B);
      mbar_wait(smem_u32(kv_full), 0);
      uint32_t s = 0;
      for (int i = 0; i < nq; ++i) {
        const uint64_t off = (uint64_t)((s * AB_TILE) >> 4);
        // the loop-invariant descriptors are re-derived from these opaque copies every iteration: hoisted out of the loop,
        // their 24 per-step variants exceeded this warp's 72-register budget and were spilled (LDL in front of the MMA issues)
        uint64_t ds_k = dDS_k, ds_mn = dDS_mn, k_mn = dK_mn;
        asm volatile("" : "+l"(ds_k), "+l"(ds_mn), "+l"(k_mn));
#pragma unroll
        for (int w = 0; w < 2; ++w) {
          mbar_wait(smem_u32(&p_full[w]), i & 1);
          tc_fence_after();
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int kk = w * 4 + k;  // 16-query reduction step
            umma_f16_ts(T_DV, T_PT + kk * 8, dDO_mn + off + (uint64_t)(kk * 128), id_g, (i | kk) != 0);
          }
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int kk = w * 4 + k;
            umma_f16_ss(T_DK, ds_k + (uint64_t)(w * (AB_TILE >> 4) + 2 * k), dQ_mn + off + (uint64_t)(kk * 128), id_g, (i | kk) != 0);
          }
        }
        if (i > 0) {  // dQ_{i-1} has been pulled out of TMEM
          mbar_wait(smem_u32(dq_free), (i - 1) & 1);
          tc_fence_after();
        }
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)  // 16-key reduction step
          umma_f16_ss(T_DQ, ds_mn + (uint64_t)(kk * 128), k_mn + (uint64_t)(kk * 128), id_q, kk != 0);
        umma_commit(smem_u32(dq_full));
        umma_commit(smem_u32(pd_done));
        umma_commit(smem_u32(&qdo_empty[s]));
        if (++s == AF_STAGES) s = 0;
      }
      umma_commit(smem_u32(acc_full));
    }
    __syncwarp();
  } else {  // ===== the two math warpgroups: thread = key row, warpgroup = 64 query columns =====
    asm volatile("setmaxnreg.inc.sync.aligned.u32 216;");
    int n_local = N;  // re-derived inside this register region (see DESIGN.md: setmaxnreg + live-through scalars)
    asm volatile("" : "+r"(n_local));
    const FusedWork wm = fused_work((int)blockIdx.x, nkv, n_full, parts, (n_local + 127) / 128);
    const int nq_m = wm.qb1 - wm.qb0;
    const int wg = (warp >> 2) - 1;
    const int quad = warp & 3;
    const int r = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    const bool kv_ok = kv0 + r < n_local;
    const uint32_t ds_row = smem_u32(sDS) + wg * AB_TILE + r * 128;   // this key's 64 dS^T values of this half
    const uint32_t dq_slab = smem_u32(sDQ) + wg * AB_TILE;            // [128 queries x 32 d] fp32, 128B swizzle
    const uint32_t dq_row = dq_slab + r * 128;
    const uint32_t swz = (uint32_t)(r & 7);
    const uint64_t sc2_c = pack2(scale_log2, scale_log2);
    int iq_prev = 0;  // query block whose dQ sits in TMEM
    auto drain_dq = [&](int b, int iq_b) {  // dQ of pipeline step b: TMEM -> fp32 slab -> TMA reduce-add
      mbar_wait(smem_u32(dq_full), b & 1);
      tc_fence_after();
      uint32_t o[32];
      tmem_ld32(T_DQ + lane_base + wg * 32, o);
      tmem_wait_ld();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(dq_free));
      // per-warp slab [32 queries x 32 d] and per-warp reduction: no cross-warp barrier, the four warps of a warpgroup keep
      // their natural stagger (a 128-thread bar.sync + one [128 x 32] slab version was 4 % slower; reducing straight from registers
      // with red.global.add.v4.f32 — half-used 32-byte sectors at the L2 — 38 % slower: profiles/r02_attn_notes.md)
      if (lane == 0) tma_wait_group_read<0>();  // this warp's previous reduction has finished reading its slab
      __syncwarp();
#pragma unroll
      for (int c = 0; c < 8; ++c) sts_u4(dq_row + ((c ^ swz) << 4), o[4 * c], o[4 * c + 1], o[4 * c + 2], o[4 * c + 3]);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        tma_reduce_add_3d(&tmDQ, dq_slab + quad * 4096, wg * 32, iq_b * 128 + quad * 32, bh);
        tma_commit_group();
      }
    };
    uint32_t s = 0;
    int iq = wm.qb0 + (int)((wm.kvblk * 37u) % (unsigned)nq_m);
    for (int i = 0; i < nq_m; ++i) {
      mbar_wait(smem_u32(s_full), i & 1);
      tc_fence_after();
      uint32_t pp[32], dd[32];
      uint32_t sv[64], dpv[64];
      tmem_ld32(T_ST + lane_base + wg * 64, *reinterpret_cast<uint32_t(*)[32]>(&sv[0]));
      tmem_ld32(T_ST + lane_base + wg * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&sv[32]));
      tmem_ld32(T_DPT + lane_base + wg * 64, *reinterpret_cast<uint32_t(*)[32]>(&dpv[0]));
      tmem_ld32(T_DPT + lane_base + wg * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&dpv[32]));
      tmem_wait_ld();
      tc_fence_before();
      __syncwarp();
      uint32_t tok = 0;  // the token dependency keeps ptxas from hoisting the exponentials above the arrive
      if (lane == 0) tok = mbar_arrive_tok(smem_u32(&s_free[wg]));
      const float zf = __uint_as_float(tok & (uint32_t)zero);  // +0.0f at run time
      const uint64_t sc2 = fadd2(sc2_c, pack2(zf, zf));
#pragma unroll
      for (int c = 0; c < 4; ++c) {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const int col = c * 16 + 2 * q;
          // sv = S^T - lse/scale, dpv = dP^T - D (the statistics came in through the fifth K-step of the score products)
          const uint64_t x2 = fmul2(pack2(__uint_as_float(sv[col]), __uint_as_float(sv[col + 1])), sc2);
          float p0, p1;
          if ((EX2_EMU_PAIRS >> ((c * 8 + q) & 15)) & 1u) {
            ex2_emu2(x2, p0, p1);
          } else {
            float a0, a1;
            unpack2(x2, a0, a1);
            p0 = ex2f(a0), p1 = ex2f(a1);
          }
          const uint64_t p2 = pack2(p0, p1);
          float d0, d1;  // dS^T without the softmax scale: applied to dK in the epilogue and to dQ in the finishing pass
          unpack2(fmul2(p2, pack2(__uint_as_float(dpv[col]), __uint_as_float(dpv[col + 1]))), d0, d1);
          pp[c * 8 + q] = pack_bf16(p0, p1);
          dd[c * 8 + q] = pack_bf16(d0, d1);
        }
      }
      if (i > 0) {  // the products of block i-1 read P^T (TMEM) and dS^T (smem): they must have retired
        mbar_wait(smem_u32(pd_done), (i - 1) & 1);
        tc_fence_after();
      }
      tmem_st32(T_PT + lane_base + wg * 32, pp);
#pragma unroll
      for (int c = 0; c < 8; ++c) sts_u4(ds_row + ((c ^ swz) << 4), dd[4 * c], dd[4 * c + 1], dd[4 * c + 2], dd[4 * c + 3]);
      tmem_wait_st();
      fence_proxy_async_smem();  // dS^T tile -> visible to the tensor core's (async proxy) reads
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&p_full[wg]));
      if (i > 0) drain_dq(i - 1, iq_prev);
      iq_prev = iq;
      if (++iq == wm.qb1) iq = wm.qb0;
      if (++s == AF_STAGES) s = 0;
    }
    drain_dq(nq_m - 1, iq_prev);
    // ---- epilogue: warpgroup 0 writes dV_j, warpgroup 1 writes dK_j (bf16, head-major [BH, N, 64]) ----
    mbar_wait(smem_u32(acc_full), 0);
    tc_fence_after();
    __nv_bfloat16* outp = (wg == 0 ? dv : dk) + ((int64_t)bh * n_local + kv0 + r) * 64;
    float* outf = part_ws + (((int64_t)wm.part * 2 + wg) * 128 + r) * 64;  // split CTA: fp32 partial [part][dV | dK][128][64]
    const uint32_t tacc = (wg == 0 ? T_DV : T_DK) + lane_base;
    const float osc = wg == 0 ? 1.f : scale;  // dK = scale * (unscaled dS)^T Q
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      uint32_t o[32];
      tmem_ld32(tacc + c * 32, o);
      tmem_wait_ld();
#pragma unroll
      for (int q = 0; q < 32; ++q) o[q] = __float_as_uint(__uint_as_float(o[q]) * osc);
      if (wm.part >= 0) {
#pragma unroll
        for (int q = 0; q < 8; ++q)
          reinterpret_cast<uint4*>(outf + c * 32)[q] = make_uint4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
      } else if (kv_ok) {
        uint4* dst = reinterpret_cast<uint4*>(outp + c * 32);
#pragma unroll
        for (int q = 0; q < 4; ++q)
          dst[q] = make_uint4(pack_bf16(__uint_as_float(o[8 * q]), __uint_as_float(o[8 * q + 1])),
                              pack_bf16(__uint_as_float(o[8 * q + 2]), __uint_as_float(o[8 * q + 3])),
                              pack_bf16(__uint_as_float(o[8 * q + 4]), __uint_as_float(o[8 * q + 5])),
                              pack_bf16(__uint_as_float(o[8 * q + 6]), __uint_as_float(o[8 * q + 7])));
      }
    }
    if (lane == 0) tma_wait_group<0>();  // the last reductions have left shared memory and are globally performed
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 512);
}

// dK / dV of the split units: sum of the `parts` fp32 partials -> bf16.  grid (split units, 2), 256 threads, 8 elements each.
__global__ void __launch_bounds__(256) attn_bwd_combine_kernel(const float* __restrict__ part_ws, int parts, int nkv, int n_full, int N,
                                                               __nv_bfloat16* __restrict__ dk, __nv_bfloat16* __restrict__ dv) {
  const int unit = n_full + blockIdx.x, which = blockIdx.y;  // which: 0 = dV, 1 = dK
  const int kvblk = unit % nkv, bh = unit / nkv;
  __nv_bfloat16* out = which == 0 ? dv : dk;
  for (int e8 = threadIdx.x; e8 < 128 * 64 / 8; e8 += 256) {
    const int row = e8 >> 3, c8 = e8 & 7;
    if (kvblk * 128 + row >= N) continue;
    float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int p = 0; p < parts; ++p) {  // fixed order: deterministic
      const float* src = part_ws + ((((int64_t)blockIdx.x * parts + p) * 2 + which) * 128 + row) * 64 + c8 * 8;
      const float4 x = ldg_stream_f4(src), y = ldg_stream_f4(src + 4);
      a[0] += x.x, a[1] += x.y, a[2] += x.z, a[3] += x.w, a[4] += y.x, a[5] += y.y, a[6] += y.z, a[7] += y.w;
    }
    reinterpret_cast<uint4*>(out + ((int64_t)bh * N + kvblk * 128 + row) * 64)[c8] =
        make_uint4(pack_bf16(a[0], a[1]), pack_bf16(a[2], a[3]), pack_bf16(a[4], a[5]), pack_bf16(a[6], a[7]));
  }
}

// dq[i] = bf16(scale * acc[i]): the finishing pass of the fused backward (8 elements per thread)
__global__ void __launch_bounds__(256) attn_bwd_dq_finish_kernel(const float* __restrict__ acc, __nv_bfloat16* __restrict__ dq,
                                                                 int64_t n8, float scale) {
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n8) return;
  const float4 a = ldg_stream_f4(acc + i * 8), b = ldg_stream_f4(acc + i * 8 + 4);
  reinterpret_cast<uint4*>(dq)[i] = make_uint4(pack_bf16(a.x * scale, a.y * scale), pack_bf16(a.z * scale, a.w * scale),
                                              pack_bf16(b.x * scale, b.y * scale), pack_bf16(b.z * scale, b.w * scale));
}

// D[bh, q] = sum_d dO[b, q, h*64 + d] * O[b, q, h*64 + d].  Eight threads per (token, head) row, one 16-byte chunk of O and of
// dO each (round 1 used a whole warp per row with 4-byte loads: 1.7 TB/s); o / dout are token-major, so row r = token * H + head
// starts at element 64 r.
__global__ void __launch_bounds__(256) attn_bwd_prep_kernel(const __nv_bfloat16* __restrict__ o, const __nv_bfloat16* __restrict__ dout,
                                                            int B, int H, int N, float* __restrict__ Dsum) {
  const int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x;
  const int64_t row = idx >> 3;
  const int c8 = (int)(idx & 7);
  const bool ok = row < (int64_t)B * N * H;
  float s = 0.f;
  if (ok) {
    const uint4 a = ldg_stream_u4(o + row * 64 + c8 * 8), b = ldg_stream_u4(dout + row * 64 + c8 * 8);
    const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, bw[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      s = fmaf(__uint_as_float(aw[i] << 16), __uint_as_float(bw[i] << 16), s);
      s = fmaf(__uint_as_float(aw[i] & 0xFFFF0000u), __uint_as_float(bw[i] & 0xFFFF0000u), s);
    }
  }
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  s += __shfl_xor_sync(0xffffffffu, s, 4);
  if (ok && c8 == 0) {
    const int h = (int)(row % H);
    const int64_t tok = row / H;  // b*N + n
    const int bb = (int)(tok / N), n = (int)(tok % N);
    Dsum[((int64_t)bb * H + h) * N + n] = s;
  }
}

static int head_tmap(CUtensorMap* m, const void* base, int BH, int N) {  // head-major [BH, N, 64]
  uint64_t dims[3] = {64, (uint64_t)N, (uint64_t)BH};
  uint64_t str[2] = {64 * 2, (uint64_t)N * 64 * 2};
  uint32_t box[3] = {64, 128, 1};
  return make_tmap(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

}  // namespace smbv

using namespace smbv;

extern "C" int smbv_flash_attn_bwd_ex(const smbv_bf16* q, const smbv_bf16* k, const smbv_bf16* v, const smbv_bf16* o,
                                      const smbv_bf16* dout, const float* lse, int B, int H, int N, float scale,
                                      float* dsum_ws, smbv_bf16* dq, smbv_bf16* dk, smbv_bf16* dv, void* ev_dkdv_start,
                                      void* ev_dkdv_stop, smbv_stream_t st) {
  SMBV_ARG(q && k && v && o && dout && lse && dsum_ws && dq && dk && dv, "flash_attn_bwd: null pointer");
  SMBV_ARG(B >= 1 && (int64_t)B * H <= 65535, "flash_attn_bwd: bad batch B=%d (B*H must be <= 65535)", B);
  SMBV_ARG(H > 0 && N > 0 && scale > 0.f, "flash_attn_bwd: bad sizes H=%d N=%d", H, N);
  cudaStream_t s = (cudaStream_t)st;
  const int BH = B * H;
  const int64_t nwarps = (int64_t)B * N * H;
  attn_bwd_prep_kernel<<<(unsigned)((nwarps * 8 + 255) / 256), 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(o),
                                                                     reinterpret_cast<const __nv_bfloat16*>(dout), B, H, N, dsum_ws);
  SMBV_LAUNCH_CHECK("attn_bwd_prep");
  CUtensorMap tq, tk, tv, tdo;
  int r;
  if ((r = head_tmap(&tq, q, BH, N))) return r;
  if ((r = head_tmap(&tk, k, BH, N))) return r;
  if ((r = head_tmap(&tv, v, BH, N))) return r;
  {  // dO is token-major [B, N, H*64]: per (sample, head) a [N, 64] matrix with row stride H*64
    uint64_t dims[4] = {64, (uint64_t)N, (uint64_t)H, (uint64_t)B};
    uint64_t str[3] = {(uint64_t)H * 64 * 2, 64 * 2, (uint64_t)N * H * 64 * 2};
    uint32_t box[4] = {64, 128, 1, 1};
    if ((r = make_tmap(&tdo, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, dout, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B))) return r;
  }
  static bool attr_set = false;
  if (!attr_set) {
    SMBV_CUDA(cudaFuncSetAttribute(flash_attn_bwd_dkdv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DK_SMEM));
    SMBV_CUDA(cudaFuncSetAttribute(flash_attn_bwd_dq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AB_SMEM));
    attr_set = true;
  }
  dim3 grid((N + 127) / 128, BH);
  // The dK/dV and dQ kernels are independent (both only read q, k, v, dO, lse, D) and each runs one CTA per SM, so their
  // grids rarely fill whole waves (960 CTAs = 6.49 waves at H=6, N=20480).  Launching dQ on a forked stream lets its CTAs
  // start on the SMs the last dK/dV wave leaves idle: 13 waves instead of 7 + 7.  Fork/join is by events (no host sync).
  static thread_local cudaStream_t s2 = nullptr;
  static thread_local cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  const bool fork = ((int64_t)grid.x * grid.y) % num_sms() != 0;
  if (fork && !s2) {
    SMBV_CUDA(cudaStreamCreateWithFlags(&s2, cudaStreamNonBlocking));
    SMBV_CUDA(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
    SMBV_CUDA(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
  }
  cudaStream_t sq = s;
  if (fork) {
    SMBV_CUDA(cudaEventRecord(ev_fork, s));  // after the prep kernel (D) and everything that produced the inputs
    SMBV_CUDA(cudaStreamWaitEvent(s2, ev_fork, 0));
    sq = s2;
  }
  if (ev_dkdv_start) SMBV_CUDA(cudaEventRecord((cudaEvent_t)ev_dkdv_start, s));
  flash_attn_bwd_dkdv_kernel<<<grid, AB_THREADS, DK_SMEM, s>>>(tq, tk, tv, tdo, H, N, scale, lse, dsum_ws,
                                                               reinterpret_cast<__nv_bfloat16*>(dk), reinterpret_cast<__nv_bfloat16*>(dv), 0);
  SMBV_LAUNCH_CHECK("flash_attn_bwd_dkdv");
  if (ev_dkdv_stop) SMBV_CUDA(cudaEventRecord((cudaEvent_t)ev_dkdv_stop, s));
  flash_attn_bwd_dq_kernel<<<grid, AB_THREADS, AB_SMEM, sq>>>(tq, tk, tv, tdo, H, N, scale, lse, dsum_ws,
                                                             reinterpret_cast<__nv_bfloat16*>(dq), 0);
  SMBV_LAUNCH_CHECK("flash_attn_bwd_dq");
  if (fork) {
    SMBV_CUDA(cudaEventRecord(ev_join, s2));
    SMBV_CUDA(cudaStreamWaitEvent(s, ev_join, 0));
  }
  return 0;
}

// split of the partial last wave (see FusedWork): n_full whole units, the rest cut into `parts` query ranges
static void fused_plan(int B, int H, int N, int* n_full, int* parts) {
  const int nkv = (N + 127) / 128, U = nkv * B * H, sms = num_sms();
  int nf = (U / sms) * sms, R = U - nf, best = 1;
  if (R > 0) {  // tail cost in units of one whole CTA: rounds(k) * (1/k + fixed/nq); fixed = per-CTA prologue + epilogue ~ 4 blocks
    const double fixed = 4.0 / nkv;
    double best_cost = 1.0 + fixed;
    for (int k = 2; k <= 8 && k <= nkv; ++k) {
      const double cost = (double)((R * k + sms - 1) / sms) * (1.0 / k + fixed);
      if (cost < best_cost * 0.97) best_cost = cost, best = k;
    }
  }
  if (best == 1) nf = U;
  *n_full = nf, *parts = best;
}

extern "C" int64_t smbv_flash_attn_bwd_fused_workspace_bytes(int B, int H, int N) {
  if (B < 1 || H < 1 || N < 1) return 0;
  int n_full, parts;
  fused_plan(B, H, N, &n_full, &parts);
  const int64_t U = (int64_t)((N + 127) / 128) * B * H;
  return (int64_t)B * H * N * 64 * 4 + (U - n_full) * parts * 2 * 128 * 64 * 4;
}

extern "C" int smbv_flash_attn_bwd_fused(const smbv_bf16* q, const smbv_bf16* k, const smbv_bf16* v, const smbv_bf16* o,
                                         const smbv_bf16* dout, const float* lse, int B, int H, int N, float scale,
                                         float* dsum_ws, void* workspace, int64_t workspace_bytes, smbv_bf16* dq,
                                         smbv_bf16* dk, smbv_bf16* dv, void* ev_start, void* ev_stop, smbv_stream_t st) {
  SMBV_ARG(q && k && v && o && dout && lse && dsum_ws && workspace && dq && dk && dv, "flash_attn_bwd_fused: null pointer");
  SMBV_ARG(B >= 1 && (int64_t)B * H <= 65535, "flash_attn_bwd_fused: bad batch B=%d (B*H must be <= 65535)", B);
  SMBV_ARG(H > 0 && N > 0 && scale > 0.f, "flash_attn_bwd_fused: bad sizes H=%d N=%d", H, N);
  SMBV_ARG(workspace_bytes >= smbv_flash_attn_bwd_fused_workspace_bytes(B, H, N), "flash_attn_bwd_fused: workspace too small");
  cudaStream_t s = (cudaStream_t)st;
  const int BH = B * H;
  const int64_t nwarps = (int64_t)B * N * H;
  const int64_t nacc = (int64_t)BH * N * 64;
  float* dq_acc_ws = reinterpret_cast<float*>(workspace);
  float* part_ws = dq_acc_ws + nacc;
  int n_full, parts;
  fused_plan(B, H, N, &n_full, &parts);
  const int nkv = (N + 127) / 128, U = nkv * BH, n_split = U - n_full;
  SMBV_CUDA(cudaMemsetAsync(dq_acc_ws, 0, (size_t)nacc * sizeof(float), s));
  attn_bwd_prep_kernel<<<(unsigned)((nwarps * 8 + 255) / 256), 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(o),
                                                                     reinterpret_cast<const __nv_bfloat16*>(dout), B, H, N, dsum_ws);
  SMBV_LAUNCH_CHECK("attn_bwd_prep");
  CUtensorMap tq, tk, tv, tdo, tdq;
  int r;
  if ((r = head_tmap(&tq, q, BH, N))) return r;
  if ((r = head_tmap(&tk, k, BH, N))) return r;
  if ((r = head_tmap(&tv, v, BH, N))) return r;
  {  // dO is token-major [B, N, H*64]: per (sample, head) a [N, 64] matrix with row stride H*64
    uint64_t dims[4] = {64, (uint64_t)N, (uint64_t)H, (uint64_t)B};
    uint64_t str[3] = {(uint64_t)H * 64 * 2, 64 * 2, (uint64_t)N * H * 64 * 2};
    uint32_t box[4] = {64, 128, 1, 1};
    if ((r = make_tmap(&tdo, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, dout, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B))) return r;
  }
  {  // fp32 dQ accumulator [BH, N, 64], reduced into by [32 queries x 32 d] slabs (one per math warp)
    uint64_t dims[3] = {64, (uint64_t)N, (uint64_t)BH};
    uint64_t str[2] = {64 * 4, (uint64_t)N * 64 * 4};
    uint32_t box[3] = {32, 32, 1};
    if ((r = make_tmap(&tdq, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, dq_acc_ws, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B))) return r;
  }
  static bool attr_set = false;
  if (!attr_set) {
    SMBV_CUDA(cudaFuncSetAttribute(flash_attn_bwd_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AF_SMEM));
    attr_set = true;
  }
  const unsigned grid = (unsigned)(n_full + n_split * parts);
  if (ev_start) SMBV_CUDA(cudaEventRecord((cudaEvent_t)ev_start, s));
  flash_attn_bwd_fused_kernel<<<grid, AB_THREADS, AF_SMEM, s>>>(tq, tk, tv, tdo, tdq, H, N, scale, lse, dsum_ws,
                                                                reinterpret_cast<__nv_bfloat16*>(dk), reinterpret_cast<__nv_bfloat16*>(dv),
                                                                part_ws, nkv, n_full, parts, 0);
  SMBV_LAUNCH_CHECK("flash_attn_bwd_fused");
  if (n_split > 0) {
    attn_bwd_combine_kernel<<<dim3((unsigned)n_split, 2), 256, 0, s>>>(part_ws, parts, nkv, n_full, N, reinterpret_cast<__nv_bfloat16*>(dk),
                                                                       reinterpret_cast<__nv_bfloat16*>(dv));
    SMBV_LAUNCH_CHECK("attn_bwd_combine");
  }
  if (ev_stop) SMBV_CUDA(cudaEventRecord((cudaEvent_t)ev_stop, s));
  attn_bwd_dq_finish_kernel<<<(unsigned)((nacc / 8 + 255) / 256), 256, 0, s>>>(dq_acc_ws, reinterpret_cast<__nv_bfloat16*>(dq),
                                                                              nacc / 8, scale);
  SMBV_LAUNCH_CHECK("attn_bwd_dq_finish");
  return 0;
}

extern "C" int smbv_flash_attn_bwd(const smbv_bf16* q, const smbv_bf16* k, const smbv_bf16* v, const smbv_bf16* o,
                                   const smbv_bf16* dout, const float* lse, int B, int H, int N, float scale,
                                   float* dsum_ws, smbv_bf16* dq, smbv_bf16* dk, smbv_bf16* dv, smbv_stream_t st) {
  return smbv_flash_attn_bwd_ex(q, k, v, o, dout, lse, B, H, N, scale, dsum_ws, dq, dk, dv, nullptr, nullptr, st);
}
