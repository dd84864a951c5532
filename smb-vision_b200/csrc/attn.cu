// Flash attention forward on tcgen05/TMEM (sm_100a): non-causal MHA, head_dim 64, online softmax.
// Semantics: eager_attention_forward, reference modeling_videomae.py:196-223 (softmax in fp32, probabilities cast
// to the value dtype before P@V, output [B,N,H,64]).
//
// flash_attn_fwd2_kernel: two query tiles (256 rows) per CTA, two softmax warpgroups, everything but K/V/Q in TMEM.
//   warpgroup 0 : warp 0 lane 0 = TMA producer (Q once; K and V tiles through 4-stage mbarrier rings, 128B swizzle),
//                 warp 1 / warp 2 lane 0 = MMA issuer of tile A / tile B
//   warpgroup 1 : softmax of tile A (rows q0 .. q0+127), one row per thread;  warpgroup 2 : tile B
//   TMEM        : S_A [0,128) S_B [128,256) | P_A [256,320) P_B [320,384) (bf16 pairs) | O_A [384,448) O_B [448,512)
// The softmax releases S as soon as it sits in registers (s_free), so S(j+1) = Q K(j+1)^T is computed WHILE the
// softmax of block j runs; P is written back to TMEM and feeds O += P V as the TMEM A operand (no smem round trip).
// Each tile has its own issuing thread (blocking mbarrier waits in the tile's natural event order s_free, p_full, ...),
// so neither tile queues behind the other's softmax.  Running max with lazy rescaling: O is rescaled in TMEM only when
// the max grows by more than 2^8.  Packed f32x2 math (FFMA2/FADD2) + FMNMX3.
#include "common.cuh"
#include "../../include/smbv_b200.h"

namespace smbv {

constexpr int ATT_BQ = 128, ATT_BK = 128, ATT_D = 64;
constexpr int ATT_TILE_BYTES = 128 * 64 * 2;  // 16 KB: one [128 x 64] bf16 tile (Q, K or V)
constexpr float ATT_RESCALE_LOG2 = 8.f;

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

constexpr int A2_THREADS = 384;
constexpr int A2_KSTAGES = 4, A2_VSTAGES = 4;
constexpr int A2_SMEM = ATT_TILE_BYTES * (2 + A2_KSTAGES + A2_VSTAGES) + 1024 + 256;

// Pair i of every 16-pair chunk of exponentials runs as ex2_emu2 on the FMA / ALU pipes when bit i is set, else on MUFU.EX2.
// 6 of every 16 pairs (37.5 %): measured on one box, same run: 1.52 ms vs 1.60 ms all-MUFU at H=12, N=20480 (-5 %; also -5 % at
// H=6 and at N=7168); 25 % and 31 % gain less, 44 % and 50 % fall off a cliff (1.78 / 1.85 ms: the softmax warps become
// issue-bound), other placements of the six pairs are 1-7 % slower.
constexpr uint32_t EX2_EMU_PAIRS = 0xA4A4u;

__global__ void __launch_bounds__(A2_THREADS, 1)
flash_attn_fwd2_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                       const __grid_constant__ CUtensorMap tmV, int H, int N, float scale_log2, float scale,
                       __nv_bfloat16* __restrict__ out, float* __restrict__ lse, int n_full, int n_split, int parts, int pairs_per_head,
                       float* __restrict__ ws) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;  // 2 tiles
  uint8_t* sK = sQ + 2 * ATT_TILE_BYTES;
  uint8_t* sV = sK + A2_KSTAGES * ATT_TILE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + A2_VSTAGES * ATT_TILE_BYTES);
  uint64_t* q_full = bars;
  uint64_t* k_full = q_full + 1;
  uint64_t* k_empty = k_full + A2_KSTAGES;
  uint64_t* v_full = k_empty + A2_KSTAGES;
  uint64_t* v_empty = v_full + A2_VSTAGES;
  uint64_t* s_full = v_empty + A2_VSTAGES;  // [2] per tile
  uint64_t* s_free = s_full + 2;            // [2]
  uint64_t* p_full = s_free + 2;            // [2]
  uint64_t* pv_done = p_full + 2;           // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(pv_done + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // Work decomposition.  A unit = a PAIR of adjacent 128-row query tiles of one head (the ping-pong mode).  The first
  // n_full CTAs run whole units.  The units that would form a last, partial wave are each split over `parts` CTAs by key
  // range (wave-quantisation fix: the tail then costs 1/parts .. of a CTA time); those CTAs leave un-normalised partial results
  // (O, max, sum) in `ws` and flash_attn_combine_kernel merges the halves.  A head with an odd number of tiles ends with
  // one single-tile CTA.
  int q0, bh, ntiles = 2, kv_begin = 0, split_slot = -1;
  const int nkv_total = (N + ATT_BK - 1) / ATT_BK;
  int nkv = nkv_total;
  {
    const int b = blockIdx.x;
    if (b < n_full) {
      bh = b / pairs_per_head, q0 = 2 * (b % pairs_per_head) * ATT_BQ;
    } else if (b < n_full + parts * n_split) {
      const int s1 = b - n_full, pr = n_full + s1 / parts, part = s1 % parts;
      bh = pr / pairs_per_head, q0 = 2 * (pr % pairs_per_head) * ATT_BQ;
      kv_begin = (int)((int64_t)nkv_total * part / parts);
      nkv = (int)((int64_t)nkv_total * (part + 1) / parts) - kv_begin;
      split_slot = s1;  // (unit, part)
    } else {  // odd leftover tile of a head
      bh = b - n_full - parts * n_split, q0 = ((N + ATT_BQ - 1) / ATT_BQ - 1) * ATT_BQ, ntiles = 1;
    }
  }

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    mbar_init(smem_u32(q_full), 1);
    for (int s = 0; s < A2_KSTAGES; ++s) mbar_init(smem_u32(&k_full[s]), 1), mbar_init(smem_u32(&k_empty[s]), ntiles);
    for (int s = 0; s < A2_VSTAGES; ++s) mbar_init(smem_u32(&v_full[s]), 1), mbar_init(smem_u32(&v_empty[s]), ntiles);
    for (int t = 0; t < 2; ++t) {
      mbar_init(smem_u32(&s_full[t]), 1);
      mbar_init(smem_u32(&s_free[t]), 4);
      mbar_init(smem_u32(&p_full[t]), 4);
      mbar_init(smem_u32(&pv_done[t]), 1);
    }
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
    if (warp == 0 && lane == 0) {  // ===== TMA producer =====
      mbar_expect_tx(smem_u32(q_full), ntiles * ATT_TILE_BYTES);
      tma_load_3d(smem_u32(sQ), &tmQ, smem_u32(q_full), 0, q0, bh);
      if (ntiles == 2) tma_load_3d(smem_u32(sQ + ATT_TILE_BYTES), &tmQ, smem_u32(q_full), 0, q0 + ATT_BQ, bh);
      uint32_t ks = 0, kph = 0, vs = 0, vph = 0;
      for (int j = 0; j < nkv; ++j) {
        mbar_wait(smem_u32(&k_empty[ks]), kph ^ 1);
        mbar_expect_tx(smem_u32(&k_full[ks]), ATT_TILE_BYTES);
        tma_load_3d(smem_u32(sK + ks * ATT_TILE_BYTES), &tmK, smem_u32(&k_full[ks]), 0, (kv_begin + j) * ATT_BK, bh);
        if (++ks == A2_KSTAGES) ks = 0, kph ^= 1;
        mbar_wait(smem_u32(&v_empty[vs]), vph ^ 1);
        mbar_expect_tx(smem_u32(&v_full[vs]), ATT_TILE_BYTES);
        tma_load_3d(smem_u32(sV + vs * ATT_TILE_BYTES), &tmV, smem_u32(&v_full[vs]), 0, (kv_begin + j) * ATT_BK, bh);
        if (++vs == A2_VSTAGES) vs = 0, vph ^= 1;
      }
    } else if ((warp == 1 || (warp == 2 && ntiles == 2)) && elect_one()) {  // ===== MMA issuers: warp 1 -> tile A, warp 2 -> tile B =====
      // elect.sync, not `lane == 0`: with a threadIdx-derived predicate ptxas cannot prove a single active lane and wraps every
      // tcgen05.mma in an ELECT / R2UR / BRA.U.ANY waterfall loop (~75 cycles of issue per MMA, 12 MMAs per score tile)
      const int t = warp - 1;
      constexpr uint32_t idesc_s = umma_idesc(UMMA_BF16, 128, 128);
      constexpr uint32_t idesc_o = umma_idesc(UMMA_BF16, 128, 64, 0, 1);  // V is the MN-major B operand
      // descriptor templates: only the 14-bit start-address field changes (+ bytes >> 4)
      const uint64_t dQ = umma_desc(smem_u32(sQ + t * ATT_TILE_BYTES), 16, 1024, UMMA_SW_128B);
      const uint64_t dK = umma_desc(smem_u32(sK), 16, 1024, UMMA_SW_128B);
      const uint64_t dV = umma_desc(smem_u32(sV), ATT_TILE_BYTES, 1024, UMMA_SW_128B);
      const uint32_t tS = tmem_base + t * 128, tP = tmem_base + 256 + t * 64, tO = tmem_base + 384 + t * 64;
      uint32_t ks = 0, kph = 0, vs = 0, vph = 0;
      auto issue_S = [&]() {  // S_t = Q_t K(stage ks)^T, then release the K stage (both issuers arrive on k_empty)
        mbar_wait(smem_u32(&k_full[ks]), kph);
        tc_fence_after();
        const uint64_t b = dK + (uint64_t)((ks * ATT_TILE_BYTES) >> 4);
#pragma unroll
        for (int k = 0; k < ATT_D / 16; ++k) umma_f16_ss(tS, dQ + 2 * k, b + 2 * k, idesc_s, k != 0);
        umma_commit(smem_u32(&s_full[t]));
        umma_commit(smem_u32(&k_empty[ks]));
        if (++ks == A2_KSTAGES) ks = 0, kph ^= 1;
      };
      mbar_wait(smem_u32(q_full), 0);
      issue_S();
      for (int j = 0; j < nkv; ++j) {
        if (j + 1 < nkv) {  // S(j+1) as soon as the softmax has pulled S(j) into registers: runs under softmax(j)
          mbar_wait(smem_u32(&s_free[t]), j & 1);
          issue_S();
        }
        mbar_wait(smem_u32(&v_full[vs]), vph);
        mbar_wait(smem_u32(&p_full[t]), j & 1);
        tc_fence_after();
        const uint64_t b = dV + (uint64_t)((vs * ATT_TILE_BYTES) >> 4);
#pragma unroll
        for (int k = 0; k < ATT_BK / 16; ++k)  // A = P[128 x 16] as bf16 pairs in 8 TMEM columns
          umma_f16_ts(tO, tP + k * 8, b + (uint64_t)(k * 128), idesc_o, (j | k) != 0);
        umma_commit(smem_u32(&pv_done[t]));
        umma_commit(smem_u32(&v_empty[vs]));
        if (++vs == A2_VSTAGES) vs = 0, vph ^= 1;
      }
    }
    __syncwarp();
  } else if ((warp >> 2) - 1 < ntiles) {  // ===== softmax warpgroups (the second one idles in a single-tile CTA) =====
    asm volatile("setmaxnreg.inc.sync.aligned.u32 216;");
    const int t = (warp >> 2) - 1;  // tile 0 / 1
    const int quad = warp & 3;
    const int r = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    const uint32_t tS = tmem_base + lane_base + t * 128;
    const uint32_t tP = tmem_base + lane_base + 256 + t * 64;
    const uint32_t tO = tmem_base + lane_base + 384 + t * 64;
    const uint64_t sc2 = pack2(scale_log2, scale_log2);
    float m_used = -INFINITY, l = 0.f;
    // barrier addresses as 32-bit shared-window offsets held in registers of THIS register region: the generic `bars`
    // pointer lives across the setmaxnreg boundary and was re-loaded from local memory (LDL) in front of every arrive / wait
    uint32_t b_sfull = smem_u32(&s_full[t]), b_sfree = smem_u32(&s_free[t]), b_pfull = smem_u32(&p_full[t]), b_pvdone = smem_u32(&pv_done[t]);
    asm volatile("" : "+r"(b_sfull), "+r"(b_sfree), "+r"(b_pfull), "+r"(b_pvdone));
    for (int j = 0; j < nkv; ++j) {
      mbar_wait(b_sfull, j & 1);
      tc_fence_after();
      uint32_t s[4][32];
#pragma unroll
      for (int c = 0; c < 4; ++c) tmem_ld32(tS + c * 32, s[c]);
      tmem_wait_ld();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(b_sfree);  // S(j+1) may now overwrite the S columns
      const int kv_valid = N - (kv_begin + j) * ATT_BK;
      if (kv_valid < ATT_BK) {
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (c * 32 + i >= kv_valid) s[c][i] = __float_as_uint(-INFINITY);
      }
      // row maximum of the block: EIGHT independent FMNMX3 chains of 8 (ncu source view: the four 16-deep chains were 16 % of a
      // softmax warp's stall samples — every FMNMX3 waits ~5 cycles for its predecessor); max is exact, so the result is unchanged
      float mx[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) mx[q] = -INFINITY;
#pragma unroll
      for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int i = 0; i < 32; i += 16)
#pragma unroll
          for (int q = 0; q < 8; ++q) mx[q] = fmax3(mx[q], __uint_as_float(s[c][i + 2 * q]), __uint_as_float(s[c][i + 2 * q + 1]));
      const float m_blk = fmaxf(fmax3(mx[0], mx[1], mx[2]), fmax3(fmax3(mx[3], mx[4], mx[5]), mx[6], mx[7]));
      bool need = false;
      float alpha = 1.f;
      uint64_t acc[4] = {0ull, 0ull, 0ull, 0ull};
      uint32_t pk[4][16];
      auto chunk = [&](int c, uint64_t nm2, uint64_t (&a4)[4]) {  // 32 columns: p = 2^(s * scale_log2 + nm), packed bf16 + row-sum terms
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const uint64_t x2 = ffma2(pack2(__uint_as_float(s[c][2 * i]), __uint_as_float(s[c][2 * i + 1])), sc2, nm2);
          float p0, p1;
          if ((EX2_EMU_PAIRS >> i) & 1u) {
            ex2_emu2(x2, p0, p1);
          } else {
            float a, b;
            unpack2(x2, a, b);
            p0 = ex2(a), p1 = ex2(b);
          }
          a4[i & 3] = fadd2(a4[i & 3], pack2(p0, p1));
          pk[c][i] = pack_bf16(p0, p1);
        }
      };
      if (j == 0) {
        m_used = m_blk;
      } else if ((m_blk - m_used) * scale_log2 > ATT_RESCALE_LOG2) {
        need = true;
        alpha = ex2((m_used - m_blk) * scale_log2);
        m_used = m_blk;
        l *= alpha;
      }
      const float nm = -m_used * scale_log2;
      const uint64_t nm2 = pack2(nm, nm);
#pragma unroll
      for (int c = 0; c < 4; ++c) chunk(c, nm2, acc);
      {
        float a0, a1, b0, b1, c0, c1, d0, d1;
        unpack2(acc[0], a0, a1), unpack2(acc[1], b0, b1), unpack2(acc[2], c0, c1), unpack2(acc[3], d0, d1);
        l += ((a0 + a1) + (b0 + b1)) + ((c0 + c1) + (d0 + d1));
      }
      // PV(j-1) must have retired before P is overwritten / O is rescaled; by now it has had a whole softmax to do so
      if (j > 0) {
        mbar_wait(b_pvdone, (j - 1) & 1);
        tc_fence_after();
      }
      if (__any_sync(0xffffffffu, need)) {
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          uint32_t o[32];
          tmem_ld32(tO + c * 32, o);
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
          tmem_st32(tO + c * 32, o);
        }
      }
#pragma unroll
      for (int c = 0; c < 4; ++c) tmem_st16(tP + c * 16, pk[c]);
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(b_pfull);
    }
    mbar_wait(b_pvdone, (nkv - 1) & 1);
    tc_fence_after();
    const float inv_l = 1.f / l;
    const int row = q0 + t * ATT_BQ + r;
    const int bidx = bh / H, h = bh - bidx * H;
    if (split_slot >= 0) {  // key-range half of a split unit: leave (O un-normalised, max, sum) for the combine kernel
      float* wo = ws + ((int64_t)(split_slot * 2 + t) * ATT_BQ + r) * 68;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t o[32];
        tmem_ld32(tO + c * 32, o);
        tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 8; ++i)
          *reinterpret_cast<float4*>(wo + c * 32 + 4 * i) = make_float4(__uint_as_float(o[4 * i]), __uint_as_float(o[4 * i + 1]),
                                                                         __uint_as_float(o[4 * i + 2]), __uint_as_float(o[4 * i + 3]));
      }
      wo[64] = m_used * scale;  // natural-log units
      wo[65] = l;
    } else {
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      uint32_t o[32];
      tmem_ld32(tO + c * 32, o);
      tmem_wait_ld();
      if (row < N) {
        uint4* dst = reinterpret_cast<uint4*>(out + ((int64_t)bidx * N + row) * (H * ATT_D) + h * ATT_D + c * 32);
#pragma unroll
        for (int i = 0; i < 4; ++i)
          dst[i] = make_uint4(pack_bf16(__uint_as_float(o[8 * i]) * inv_l, __uint_as_float(o[8 * i + 1]) * inv_l),
                              pack_bf16(__uint_as_float(o[8 * i + 2]) * inv_l, __uint_as_float(o[8 * i + 3]) * inv_l),
                              pack_bf16(__uint_as_float(o[8 * i + 4]) * inv_l, __uint_as_float(o[8 * i + 5]) * inv_l),
                              pack_bf16(__uint_as_float(o[8 * i + 6]) * inv_l, __uint_as_float(o[8 * i + 7]) * inv_l));
      }
    }
    if (lse && row < N) lse[(int64_t)bh * N + row] = m_used * scale + logf(l);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 512);
}

// merges the `parts` key-range pieces of every split unit: one warp per query row, 2 columns per lane
__global__ void __launch_bounds__(256) flash_attn_combine_kernel(const float* __restrict__ ws, int n_full, int n_split, int parts,
                                                                 int pairs_per_head, int H, int N,
                                                                 __nv_bfloat16* __restrict__ out, float* __restrict__ lse) {
  const int w = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (w >= n_split * 2 * ATT_BQ) return;
  const int u = w / (2 * ATT_BQ), rem = w - u * 2 * ATT_BQ, t = rem / ATT_BQ, r = rem - t * ATT_BQ;
  const int pr = n_full + u, bh = pr / pairs_per_head;
  const int row = (2 * (pr % pairs_per_head) + t) * ATT_BQ + r;
  if (row >= N) return;
  const float* p0 = ws + ((int64_t)((u * parts) * 2 + t) * ATT_BQ + r) * 68;  // piece p at p0 + p * stride
  const int64_t stride = (int64_t)2 * ATT_BQ * 68;
  float m = -INFINITY;
  for (int p = 0; p < parts; ++p) m = fmaxf(m, p0[p * stride + 64]);
  float L = 0.f, ax = 0.f, ay = 0.f;
  for (int p = 0; p < parts; ++p) {  // fixed order: deterministic
    const float wp = __expf(p0[p * stride + 64] - m);
    const float2 a = *reinterpret_cast<const float2*>(p0 + p * stride + 2 * lane);
    L += p0[p * stride + 65] * wp, ax += a.x * wp, ay += a.y * wp;
  }
  const float inv = 1.f / L;
  const int bidx = bh / H, h = bh - bidx * H;
  *reinterpret_cast<uint32_t*>(out + ((int64_t)bidx * N + row) * (H * ATT_D) + h * ATT_D + 2 * lane) = pack_bf16(ax * inv, ay * inv);
  if (lse && lane == 0) lse[(int64_t)bh * N + row] = m + logf(L);
}

static int attn_tmap(CUtensorMap* m, const void* base, int BH, int N, int box_rows) {
  uint64_t dims[3] = {64, (uint64_t)N, (uint64_t)BH};
  uint64_t str[2] = {64 * 2, (uint64_t)N * 64 * 2};
  uint32_t box[3] = {64, (uint32_t)box_rows, 1};
  return make_tmap(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

}  // namespace smbv

using namespace smbv;

// split of the partial last wave: `rest` units cut into `parts` key ranges each (0 = no split).  Cost of the tail in units of one
// whole CTA: rounds(k) * (1/k + fixed/nkv), fixed = the per-CTA prologue + epilogue in key-block times (Q load, TMEM allocation,
// pipeline fill, O write-back ~ 3 blocks): short units (1960 tokens = 16 blocks) must not be cut into 3-block pieces
static int attn_fwd_parts(int64_t num_pairs, int nkv_total) {
  const int W = num_sms();
  const int rest = (int)(num_pairs % W);
  if (rest == 0) return 0;
  const double fixed = 3.0 / nkv_total;
  int best = 0;
  double best_cost = 1.0 + fixed;
  for (int k = 2; k <= 8 && k <= nkv_total; ++k) {
    const double cost = (double)((rest * k + W - 1) / W) * (1.0 / k + fixed);
    if (cost < best_cost * 0.97) best_cost = cost, best = k;
  }
  return best;
}

extern "C" int64_t smbv_flash_attn_fwd_workspace_bytes(int B, int H, int N) {
  const int64_t pairs = (int64_t)B * H * (((N + ATT_BQ - 1) / ATT_BQ) / 2);
  const int64_t rest = pairs % num_sms();
  return rest * 8 * 2 * ATT_BQ * 68 * (int64_t)sizeof(float);  // up to 8 pieces per split unit
}

extern "C" int smbv_flash_attn_fwd_ex(const smbv_bf16* q, const smbv_bf16* k, const smbv_bf16* v, int B, int H, int N,
                                      float scale, smbv_bf16* out, float* lse, int variant, void* workspace,
                                      int64_t workspace_bytes, smbv_stream_t st) {
  SMBV_ARG(q && k && v && out, "flash_attn_fwd: null pointer");
  SMBV_ARG(B > 0 && H > 0 && N > 0, "flash_attn_fwd: bad sizes B=%d H=%d N=%d", B, H, N);
  SMBV_ARG(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v) |
             reinterpret_cast<uintptr_t>(out)) & 15) == 0,
           "flash_attn_fwd: pointers must be 16-byte aligned");
  SMBV_ARG(scale > 0.f, "flash_attn_fwd: scale must be positive");
  SMBV_ARG(variant == 0, "flash_attn_fwd: variant=%d is reserved and must be 0", variant);
  const int BH = B * H;
  CUtensorMap tq, tk, tv;
  int r;
  if ((r = attn_tmap(&tq, q, BH, N, ATT_BQ))) return r;
  if ((r = attn_tmap(&tk, k, BH, N, ATT_BK))) return r;
  if ((r = attn_tmap(&tv, v, BH, N, ATT_BK))) return r;
  static bool attr_set = false;
  if (!attr_set) {
    SMBV_CUDA(cudaFuncSetAttribute(flash_attn_fwd2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, A2_SMEM));
    attr_set = true;
  }
  const float scale_log2 = scale * 1.4426950408889634f;
  __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out);
  // whole units in complete waves; the units of a partial last wave are split by key range (see the kernel)
  const int t128 = (N + ATT_BQ - 1) / ATT_BQ, pph = t128 / 2, num_pairs = BH * pph, odd = BH * (t128 & 1);
  const int nkv_total = (N + ATT_BK - 1) / ATT_BK;
  const int W = num_sms();
  int n_full = num_pairs, n_split = 0, parts = 2;
  {
    const int rest = num_pairs % W, k = attn_fwd_parts(num_pairs, nkv_total);
    const int64_t need = (int64_t)rest * k * 2 * ATT_BQ * 68 * (int64_t)sizeof(float);
    if (k >= 2 && workspace && workspace_bytes >= need) n_split = rest, n_full = num_pairs - rest, parts = k;
  }
  dim3 grid2(n_full + parts * n_split + odd);
  const int pph_arg = pph > 0 ? pph : 1;
  float* wsf = reinterpret_cast<float*>(workspace);
  flash_attn_fwd2_kernel<<<grid2, A2_THREADS, A2_SMEM, (cudaStream_t)st>>>(tq, tk, tv, H, N, scale_log2, scale, o, lse, n_full,
                                                                            n_split, parts, pph_arg, wsf);
  SMBV_LAUNCH_CHECK("flash_attn_fwd2");
  if (n_split > 0) {
    flash_attn_combine_kernel<<<(n_split * 2 * ATT_BQ + 7) / 8, 256, 0, (cudaStream_t)st>>>(wsf, n_full, n_split, parts, pph_arg, H, N, o, lse);
    SMBV_LAUNCH_CHECK("flash_attn_combine");
  }
  return 0;
}

extern "C" int smbv_flash_attn_fwd(const smbv_bf16* q, const smbv_bf16* k, const smbv_bf16* v, int B, int H, int N,
                                   float scale, smbv_bf16* out, float* lse, smbv_stream_t st) {
  return smbv_flash_attn_fwd_ex(q, k, v, B, H, N, scale, out, lse, 0, nullptr, 0, st);
}
