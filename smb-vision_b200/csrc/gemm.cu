// tcgen05 GEMM for every nn.Linear on the path: C[M,N] = A[M,K] * W[N,K]^T, bf16 operands, fp32 accumulators in TMEM,
// fused epilogues (bias, exact-erf GELU, residual add, head-major QKV split, positional gather).
//
// Persistent, warp-specialised (sm_100a):
//   warp 0 lane 0 : TMA producer  (cp.async.bulk.tensor, 128B-swizzled K-major tiles, STAGES-deep mbarrier ring)
//   warp 1 lane 0 : MMA issuer    (tcgen05.mma cta_group::1 kind::f16, M=128 x N=BN x K=16 per instruction)
//   warps 2..17   : epilogue      (tcgen05.ld 32x32b -> registers -> swizzled smem slab -> TMA store / reduce-add; four groups of four
//                                  warps), double-buffered TMEM accumulators so the epilogue of tile i overlaps the main loop of tile i+1
//                                  (modes with a per-element side input: warps 2..5, registers -> global)
#include <cstring>

#include <cstdlib>

#include "common.cuh"
#include "../../include/smbv_b200.h"

namespace smbv {

constexpr int GEMM_BM = 128;
constexpr int GEMM_BK = 64;  // 64 bf16 = 128 B = one swizzle-128B row
constexpr int GEMM_THREADS_REG = 192;  // warp 0 TMA, warp 1 MMA, warps 2-5: register epilogue
constexpr int GEMM_THREADS_TMA = 576;  // warp 0 TMA, warp 1 MMA, warps 2-17: four epilogue groups (two per slab buffer)

constexpr int EPI_SLAB_BYTES = GEMM_BM * 128;  // [128 rows x 128 B] 128B-swizzled staging slab of the TMA epilogue
// EPI4: the GELU (+ saved pre-activation) and dGELU epilogues — two slab transfers per slab — get FOUR slab buffers (an input / second-output
// buffer beside the output buffer of each group pair) and pay for them with one main-loop stage: those GEMMs are epilogue-bound.
template <int BN, bool EPI4 = false>
struct GemmCfg {
  static constexpr int STAGES = EPI4 ? (BN == 256 ? 3 : 4) : (BN == 256 ? 4 : 6);
  static constexpr int SLABS = EPI4 ? 4 : 2;
  static constexpr int A_BYTES = GEMM_BM * GEMM_BK * 2;
  static constexpr int B_BYTES = BN * GEMM_BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int TMEM_COLS = 2 * BN;  // two accumulator stages (256 or 512 columns, power of two)
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + SLABS * EPI_SLAB_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
};

struct GemmEpi {
  int M, N, K;
  int split_k;           // > 1: the K range is split over blockIdx-derived slices, epilogue must be a reducing one
  int n_whole;           // output tiles [0, n_whole) run their whole K range, only the rest is cut into split_k slices (0: all are cut)
  const void* aux;       // EPI_DGELU_BF16: pre-activation, bf16 [M, ldo]
  const float* alpha;    // optional device scalar multiplied into the accumulator (EPI_ATOMIC_F32 / EPI_BF16 / EPI_F32)
  const float* bias;
  int mode;
  void* out;
  int64_t ldo;
  const float* residual;
  int heads, tokens;
  const float* pos;
  int64_t ldpos;
  const int32_t* row_map;
};

// erf by Abramowitz & Stegun 7.1.28: erf(x) = 1 - (1 + a1 x + ... + a6 x^6)^-16 for x >= 0, odd extension.  |error| <= 3e-7
// analytically, 1.8e-6 in fp32 (measured over [-8, 8]) => GELU absolute error <= 5.5e-7, far below the bf16 rounding of the
// output (hidden_act = "gelu" is the exact-erf GELU, reference :368-370).  7 FMA + 4 FMUL + one MUFU.RCP, branch-free: the
// library erff (two divergent branches, ~30 instructions) made the epilogue, not the MMA main loop, bound the fc1 GEMM.
__device__ __forceinline__ float erf_as(float x) {
  const float ax = fabsf(x);
  float p = fmaf(ax, 0.0000430638f, 0.0002765672f);
  p = fmaf(p, ax, 0.0001520143f);
  p = fmaf(p, ax, 0.0092705272f);
  p = fmaf(p, ax, 0.0422820123f);
  p = fmaf(p, ax, 0.0705230784f);
  p = fmaf(p, ax, 1.f);
  p *= p, p *= p, p *= p, p *= p;  // ^16 (inf for |x| > ~60: rcp(inf) = 0, erf = 1)
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(p));
  return copysignf(1.f - r, x);
}
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.f + erf_as(x * 0.70710678118654752f)); }
// the same on a PAIR in packed f32x2 math (FFMA2 / FMUL2 / FADD2: half the issue slots of the polynomial; the fc1 epilogue was
// issue-bound: ~6400 issue cycles per 128x256 tile on two epilogue warps per scheduler against a 6144-cycle main loop at K = 768).
// Same operations in the same order as gelu_erf on each half -> bit-identical results.
__device__ __forceinline__ void gelu_erf2(float& x0, float& x1) {
  const uint64_t x2 = pack2(x0, x1);
  const uint64_t z2 = fmul2(x2, pack2(0.70710678118654752f, 0.70710678118654752f));
  float z0, z1;
  unpack2(z2, z0, z1);
  const uint64_t a2 = pack2(fabsf(z0), fabsf(z1));
  uint64_t p2 = ffma2(a2, pack2(0.0000430638f, 0.0000430638f), pack2(0.0002765672f, 0.0002765672f));
  p2 = ffma2(p2, a2, pack2(0.0001520143f, 0.0001520143f));
  p2 = ffma2(p2, a2, pack2(0.0092705272f, 0.0092705272f));
  p2 = ffma2(p2, a2, pack2(0.0422820123f, 0.0422820123f));
  p2 = ffma2(p2, a2, pack2(0.0705230784f, 0.0705230784f));
  p2 = ffma2(p2, a2, pack2(1.f, 1.f));
  p2 = fmul2(p2, p2), p2 = fmul2(p2, p2), p2 = fmul2(p2, p2), p2 = fmul2(p2, p2);
  float p0, p1, r0, r1;
  unpack2(p2, p0, p1);
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r0) : "f"(p0));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r1) : "f"(p1));
  const float e0 = copysignf(1.f - r0, z0), e1 = copysignf(1.f - r1, z1);
  // 0.5f * x * (1.f + erf): (0.5 x) first, as the scalar version evaluates left to right
  const uint64_t h2 = fmul2(x2, pack2(0.5f, 0.5f));
  unpack2(fmul2(h2, fadd2(pack2(1.f, 1.f), pack2(e0, e1))), x0, x1);
}
__device__ __forceinline__ float dgelu_erf(float x) {
  return 0.5f * (1.f + erf_as(x * 0.70710678118654752f)) + x * __expf(-0.5f * x * x) * 0.3989422804014327f;
}

// gelu'(x) on a pair, packed like gelu_erf2 (the dGELU epilogue of the fc2 dgrad)
__device__ __forceinline__ void dgelu_erf2(float x0, float x1, float& g0, float& g1) {
  const uint64_t x2 = pack2(x0, x1);
  const uint64_t z2 = fmul2(x2, pack2(0.70710678118654752f, 0.70710678118654752f));
  float z0, z1;
  unpack2(z2, z0, z1);
  const uint64_t a2 = pack2(fabsf(z0), fabsf(z1));
  uint64_t p2 = ffma2(a2, pack2(0.0000430638f, 0.0000430638f), pack2(0.0002765672f, 0.0002765672f));
  p2 = ffma2(p2, a2, pack2(0.0001520143f, 0.0001520143f));
  p2 = ffma2(p2, a2, pack2(0.0092705272f, 0.0092705272f));
  p2 = ffma2(p2, a2, pack2(0.0422820123f, 0.0422820123f));
  p2 = ffma2(p2, a2, pack2(0.0705230784f, 0.0705230784f));
  p2 = ffma2(p2, a2, pack2(1.f, 1.f));
  p2 = fmul2(p2, p2), p2 = fmul2(p2, p2), p2 = fmul2(p2, p2), p2 = fmul2(p2, p2);
  float p0, p1, r0, r1, t0, t1, q0, q1;
  unpack2(p2, p0, p1);
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r0) : "f"(p0));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r1) : "f"(p1));
  const float e0 = copysignf(1.f - r0, z0), e1 = copysignf(1.f - r1, z1);
  // x * exp(-x^2 / 2) / sqrt(2 pi): exp as ex2(-0.5 x^2 log2 e)
  unpack2(fmul2(fmul2(x2, x2), pack2(-0.72134752044448170f, -0.72134752044448170f)), t0, t1);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(q0) : "f"(t0));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(q1) : "f"(t1));
  const uint64_t c2 = fmul2(fmul2(x2, pack2(q0, q1)), pack2(0.3989422804014327f, 0.3989422804014327f));
  unpack2(ffma2(fadd2(pack2(1.f, 1.f), pack2(e0, e1)), pack2(0.5f, 0.5f), c2), g0, g1);
}
// one thread = one output row, 32 consecutive columns [col, col+32)
__device__ __forceinline__ void epilogue_store(const GemmEpi& e, int row, int col, const uint32_t (&r)[32]) {
  float v[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
  if (e.alpha) {
    const float al = __ldg(e.alpha);
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] *= al;
  }
  if (e.bias) {
    const float4* b4 = reinterpret_cast<const float4*>(e.bias + col);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float4 b = __ldg(b4 + i);
      v[4 * i] += b.x, v[4 * i + 1] += b.y, v[4 * i + 2] += b.z, v[4 * i + 3] += b.w;
    }
  }
  switch (e.mode) {
    case SMBV_EPI_ATOMIC_F32: {  // split-K / gradient accumulation: out += acc (fp32 reductions in L2)
      float* o = reinterpret_cast<float*>(e.out) + (int64_t)row * e.ldo + col;
#pragma unroll
      for (int i = 0; i < 8; ++i)
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(o + 4 * i), "f"(v[4 * i]), "f"(v[4 * i + 1]),
                     "f"(v[4 * i + 2]), "f"(v[4 * i + 3])
                     : "memory");
      break;
    }
    case SMBV_EPI_DGELU_BF16: {  // out = acc * gelu'(pre)
      const uint4* ax = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(e.aux) + (int64_t)row * e.ldo + col);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint4 a = ax[i];
        const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const __nv_bfloat162 pv = *reinterpret_cast<const __nv_bfloat162*>(&w[q]);
          v[8 * i + 2 * q] *= dgelu_erf(__low2float(pv));
          v[8 * i + 2 * q + 1] *= dgelu_erf(__high2float(pv));
        }
      }
      uint4* o = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(e.out) + (int64_t)row * e.ldo + col);
#pragma unroll
      for (int i = 0; i < 4; ++i)
        o[i] = make_uint4(pack_bf16(v[8 * i], v[8 * i + 1]), pack_bf16(v[8 * i + 2], v[8 * i + 3]),
                          pack_bf16(v[8 * i + 4], v[8 * i + 5]), pack_bf16(v[8 * i + 6], v[8 * i + 7]));
      break;
    }
    case SMBV_EPI_GELU_BF16:
      if (e.aux) {  // training: also keep the pre-activation (bf16) for the backward pass
        uint4* pa = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(const_cast<void*>(e.aux)) + (int64_t)row * e.ldo + col);
#pragma unroll
        for (int i = 0; i < 4; ++i)
          pa[i] = make_uint4(pack_bf16(v[8 * i], v[8 * i + 1]), pack_bf16(v[8 * i + 2], v[8 * i + 3]),
                             pack_bf16(v[8 * i + 4], v[8 * i + 5]), pack_bf16(v[8 * i + 6], v[8 * i + 7]));
      }
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = gelu_erf(v[i]);
      // fallthrough
    case SMBV_EPI_BF16: {
      uint4* o = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(e.out) + (int64_t)row * e.ldo + col);
#pragma unroll
      for (int i = 0; i < 4; ++i)
        o[i] = make_uint4(pack_bf16(v[8 * i], v[8 * i + 1]), pack_bf16(v[8 * i + 2], v[8 * i + 3]),
                          pack_bf16(v[8 * i + 4], v[8 * i + 5]), pack_bf16(v[8 * i + 6], v[8 * i + 7]));
      break;
    }
    case SMBV_EPI_QKV_HEADS: {
      const int hd = e.heads * 64;
      const int part = col / hd, rem = col - part * hd;
      const int head = rem >> 6, d = rem & 63;
      const int b = row / e.tokens, n = row - b * e.tokens;
      const int batch = e.M / e.tokens;
      int64_t off = ((((int64_t)part * batch + b) * e.heads + head) * e.tokens + n) * 64 + d;
      uint4* o = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(e.out) + off);
#pragma unroll
      for (int i = 0; i < 4; ++i)
        o[i] = make_uint4(pack_bf16(v[8 * i], v[8 * i + 1]), pack_bf16(v[8 * i + 2], v[8 * i + 3]),
                          pack_bf16(v[8 * i + 4], v[8 * i + 5]), pack_bf16(v[8 * i + 6], v[8 * i + 7]));
      break;
    }
    case SMBV_EPI_RESID_F32: {
      const float4* rs = reinterpret_cast<const float4*>(e.residual + (int64_t)row * e.ldo + col);
      float4 rr[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) rr[i] = rs[i];
      float4* o = reinterpret_cast<float4*>(reinterpret_cast<float*>(e.out) + (int64_t)row * e.ldo + col);
#pragma unroll
      for (int i = 0; i < 8; ++i)
        o[i] = make_float4(v[4 * i] + rr[i].x, v[4 * i + 1] + rr[i].y, v[4 * i + 2] + rr[i].z, v[4 * i + 3] + rr[i].w);
      break;
    }
    case SMBV_EPI_POS_GATHER_F32: {
      const float4* ps = reinterpret_cast<const float4*>(e.pos + (int64_t)e.row_map[row] * e.ldpos + col);
      float4* o = reinterpret_cast<float4*>(reinterpret_cast<float*>(e.out) + (int64_t)row * e.ldo + col);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float4 p = __ldg(ps + i);
        o[i] = make_float4(v[4 * i] + p.x, v[4 * i + 1] + p.y, v[4 * i + 2] + p.z, v[4 * i + 3] + p.w);
      }
      break;
    }
    default: {  // SMBV_EPI_F32
      float4* o = reinterpret_cast<float4*>(reinterpret_cast<float*>(e.out) + (int64_t)row * e.ldo + col);
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    }
  }
}

// A_MN / B_MN: operand is "MN-major" (its M resp. N index is the contiguous one in memory: transposed activations /
// weights for dgrad and wgrad).  Such tiles are loaded as [64 k-rows x 64 mn] 128B-swizzled sub-tiles (8 KB each).
// A3D: A is the head-major Q/K/V-gradient buffer [3][batch][heads][tokens][64] of ONE sample, seen through a 4-D tensor map
// (64, tokens, heads, 3): K-major -> the k-block index selects (part, head); MN-major -> the 64-wide m chunk does.
// TMA_EPI: the epilogue stages [128 x 128 B] slabs (64 bf16 / 32 fp32 columns) in swizzled shared memory and one thread
// hands them to the TMA unit: plain stores for bf16 / fp32 outputs, **reduce-add** (cp.reduce.async.bulk .add.f32) for the
// in-place residual update X += acc + bias and for the split-K weight gradients.  No row-strided global accesses, no
// residual read by the SM at all.  Modes that need a per-element side input keep the register epilogue.
template <int BN, bool A_MN, bool B_MN, bool A3D, bool TMA_EPI, bool EPI4 = false>
__global__ void __launch_bounds__(TMA_EPI ? GEMM_THREADS_TMA : GEMM_THREADS_REG, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmAux, const GemmEpi e, int tiles_m,
                 int tiles_n) {
  using Cfg = GemmCfg<BN, EPI4>;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* slab = smem + Cfg::STAGES * Cfg::STAGE_BYTES;  // SLABS x EPI_SLAB_BYTES (1024-aligned): output buffer of pair 0, 1 [, side buffer of pair 0, 1]
  uint8_t* bar_area = slab + Cfg::SLABS * EPI_SLAB_BYTES;
  uint64_t* full = reinterpret_cast<uint64_t*>(bar_area);
  uint64_t* empty = full + Cfg::STAGES;
  uint64_t* tfull = empty + Cfg::STAGES;
  uint64_t* tempty = tfull + 2;
  uint64_t* slab_free = tempty + 2;  // [2] per epilogue group: the pre-activation slab of the dGELU epilogue has landed (TMA load)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(slab_free + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total_kb = (e.K + GEMM_BK - 1) / GEMM_BK;
  const int kb_per = (total_kb + e.split_k - 1) / e.split_k;
  // work-unit id t: t < n_whole = output tile t with its whole K range; above = (output tile, K slice), slice fastest.  The reducing
  // epilogues (fp32 TMA reduce-add: residual update, weight gradients) make a K split free of any workspace, so the output tiles of a
  // PARTIAL LAST ROUND are cut into slices (480 tiles on 148 SMs: 3 rounds + 36 tiles x 4 slices = 3.25 rounds instead of 4)
  const int n_whole = e.n_whole;
  const int num_tiles = n_whole + (tiles_m * tiles_n - n_whole) * e.split_k;
  auto decode = [&](int t, int& mn, int& slice, int& kb0, int& kb1) {
    if (t < n_whole) {
      mn = t, slice = 0, kb0 = 0, kb1 = total_kb;
    } else {
      const int u = t - n_whole, q = u / e.split_k;
      mn = n_whole + q, slice = u - q * e.split_k, kb0 = slice * kb_per, kb1 = min(total_kb, kb0 + kb_per);
    }
  };

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < Cfg::STAGES; ++s) {
      mbar_init(smem_u32(&full[s]), 1);
      mbar_init(smem_u32(&empty[s]), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(smem_u32(&tfull[s]), 1);
      mbar_init(smem_u32(&tempty[s]), TMA_EPI ? 16 : 4);  // one arrive per epilogue warp
      mbar_init(smem_u32(&slab_free[s]), 1);
    }
    if (TMA_EPI) tma_prefetch_desc(&tmC);
    if (TMA_EPI && e.aux) tma_prefetch_desc(&tmAux);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), Cfg::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {  // ===== TMA producer =====
      uint32_t s = 0, ph = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        int mn, slice, kb0, kb1;
        decode(t, mn, slice, kb0, kb1);
        const int m0 = (mn / tiles_n) * GEMM_BM, n0 = (mn % tiles_n) * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(smem_u32(&empty[s]), ph ^ 1);
          const uint32_t fb = smem_u32(&full[s]);
          mbar_expect_tx(fb, Cfg::STAGE_BYTES);
          const uint32_t sa = smem_u32(smem + s * Cfg::STAGE_BYTES);
          const uint32_t sb = sa + Cfg::A_BYTES;
          if (!A_MN) {
            if (A3D) tma_load_4d(sa, &tmA, fb, 0, m0, kb % e.heads, kb / e.heads);
            else tma_load_2d(sa, &tmA, fb, kb * GEMM_BK, m0);
          } else {
#pragma unroll
            for (int c = 0; c < GEMM_BM / 64; ++c) {
              if (A3D) tma_load_4d(sa + c * 8192, &tmA, fb, 0, kb * GEMM_BK, (m0 / 64 + c) % e.heads, (m0 / 64 + c) / e.heads);
              else tma_load_2d(sa + c * 8192, &tmA, fb, m0 + c * 64, kb * GEMM_BK);
            }
          }
          if (!B_MN) {
            tma_load_2d(sb, &tmB, fb, kb * GEMM_BK, n0);
          } else {
#pragma unroll
            for (int c = 0; c < BN / 64; ++c) tma_load_2d(sb + c * 8192, &tmB, fb, n0 + c * 64, kb * GEMM_BK);
          }
          if (++s == Cfg::STAGES) s = 0, ph ^= 1;
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (elect_one()) {  // ===== MMA issuer (elect.sync: no per-MMA waterfall loop, see profiles/r01_attn_notes.md) =====
      constexpr uint32_t idesc = umma_idesc(UMMA_BF16, GEMM_BM, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
      uint32_t s = 0, ph = 0, it = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
        const uint32_t as = it & 1, aph = (it >> 1) & 1;
        int mn, slice, kb0, kb1;
        decode(t, mn, slice, kb0, kb1);
        mbar_wait(smem_u32(&tempty[as]), aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(smem_u32(&full[s]), ph);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + s * Cfg::STAGE_BYTES);
          const uint32_t sb = sa + Cfg::A_BYTES;
#pragma unroll
          for (int k = 0; k < GEMM_BK / 16; ++k) {
            // K-major: +32 B per 16-element k step inside the 128 B row; MN-major: +16 rows of 128 B, LBO = next 64-wide chunk
            const uint64_t ad = A_MN ? umma_desc(sa + k * 2048, 8192, 1024, UMMA_SW_128B) : umma_desc(sa + k * 32, 16, 1024, UMMA_SW_128B);
            const uint64_t bd = B_MN ? umma_desc(sb + k * 2048, 8192, 1024, UMMA_SW_128B) : umma_desc(sb + k * 32, 16, 1024, UMMA_SW_128B);
            umma_f16_ss(d_tmem, ad, bd, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit(smem_u32(&empty[s]));  // frees the smem stage when these MMAs retire
          if (++s == Cfg::STAGES) s = 0, ph ^= 1;
        }
        umma_commit(smem_u32(&tfull[as]));  // accumulator complete -> epilogue
      }
    }
    __syncwarp();
  } else if (TMA_EPI) {  // ===== four epilogue groups (warps 2-5, 6-9, 10-13, 14-17), TMA store / reduce path =====
    // Two [128 x 128 B] swizzled slab buffers, each shared by a PAIR of groups: pair p = groups p and p + 2 takes every other slab
    // of the tile, and inside a slab each group converts one 64-byte half of every row (32 bf16 / 16 fp32 columns): accumulator ->
    // registers -> (+bias, GELU, bf16) -> slab -> one thread hands it to the TMA unit.  The math of the next slab runs while the
    // TMA unit still reads the previous one.  Sixteen warps = four per scheduler: the exact-erf GELU / dGELU epilogues need
    // ~6400 issue cycles per 128x256 tile, more than the main loop at K <= 768 (K = 384 in the decoder: 3250 cycles) — with two
    // groups those GEMMs ran at the epilogue's speed, not the tensor core's (tools/gemm_small_sweep.py).
    const int grp = (warp - 2) >> 2;                // 0 .. 3
    const int pair = grp & 1;                       // slab buffer, slab parity
    const int half = grp >> 1;                      // which 64-byte half of the slab rows
    const int quad = warp & 3;
    const int prow = quad * 32 + lane;              // accumulator row of this thread
    const bool leader = half == 0 && ((threadIdx.x - 64) & 127) == 0;
    const bool f32out = (e.mode == SMBV_EPI_RESID_F32 || e.mode == SMBV_EPI_F32 || e.mode == SMBV_EPI_ATOMIC_F32);
    const bool reduce = (e.mode == SMBV_EPI_RESID_F32 || e.mode == SMBV_EPI_ATOMIC_F32);
    const int wcols = f32out ? 32 : 64;             // columns per 128-byte slab row
    const float alpha = e.alpha ? __ldg(e.alpha) : 1.f;
    const uint32_t sbase = smem_u32(slab + pair * EPI_SLAB_BYTES);
    const uint32_t srow = sbase + prow * 128;
    // EPI4: the pair's SIDE buffer — the pre-activation slab of the dGELU epilogue arrives there (prefetched one slab ahead), the
    // saved pre-activation of the GELU epilogue leaves from there; without EPI4 both share the output buffer
    const uint32_t xbase = EPI4 ? smem_u32(slab + (2 + pair) * EPI_SLAB_BYTES) : sbase;
    const uint32_t xrow = xbase + prow * 128;
    bool prefetched = false;  // EPI4 dGELU: this slab's pre-activation load was issued during the previous slab
    const uint32_t bar_id = 1 + pair;
    const bool dgelu = e.mode == SMBV_EPI_DGELU_BF16;
    const bool save_pre = e.mode == SMBV_EPI_GELU_BF16 && e.aux != nullptr;
    uint32_t aux_ph = 0;
    uint32_t it = 0;
    auto slab_store16 = [&](uint32_t row_addr, const uint32_t (&w)[16]) {  // this group's four 16-byte chunks of its row (128B swizzle)
#pragma unroll
      for (int i = 0; i < 4; ++i)
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(row_addr + (((4 * half + i) ^ (prow & 7)) << 4)), "r"(w[4 * i]),
                     "r"(w[4 * i + 1]), "r"(w[4 * i + 2]), "r"(w[4 * i + 3])
                     : "memory");
    };
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
      const uint32_t as = it & 1, aph = (it >> 1) & 1;
      int mn, slice, kb0_, kb1_;
      decode(t, mn, slice, kb0_, kb1_);
      const int m0 = (mn / tiles_n) * GEMM_BM, n0 = (mn % tiles_n) * BN;
      mbar_wait(smem_u32(&tfull[as]), aph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + as * BN;
      const int nslab = min(BN / wcols, (e.N - n0 + wcols - 1) / wcols);  // slabs that exist in this tile
      const int my_last = ((nslab - 1 - pair) / 2) * 2 + pair;            // last slab of this pair (< pair if none)
      if (nslab <= pair) {  // nothing for this pair in this tile: just release the accumulator
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&tempty[as]));
        continue;
      }
#pragma unroll 1
      for (int sl = pair; sl < nslab; sl += 2) {
        const int col0 = n0 + sl * wcols;
        uint32_t pk[16];  // the 64 B this thread will put into its slab row
        uint32_t ax[16];
        if (f32out) {
          const int c0 = col0 + half * 16;
          uint32_t r[16];
          tmem_ld16(taddr + sl * 32 + half * 16, r);
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            float4 v = make_float4(__uint_as_float(r[4 * i]) * alpha, __uint_as_float(r[4 * i + 1]) * alpha,
                                   __uint_as_float(r[4 * i + 2]) * alpha, __uint_as_float(r[4 * i + 3]) * alpha);
            if (e.bias && slice == 0) {  // (K slices > 0 of a split tile add only their partial sums)
              const float4 bb = __ldg(reinterpret_cast<const float4*>(e.bias + c0) + i);
              v.x += bb.x, v.y += bb.y, v.z += bb.z, v.w += bb.w;
            }
            pk[4 * i] = __float_as_uint(v.x), pk[4 * i + 1] = __float_as_uint(v.y), pk[4 * i + 2] = __float_as_uint(v.z),
                   pk[4 * i + 3] = __float_as_uint(v.w);
          }
        } else {
          const int c0 = col0 + half * 32;
          // side input of the dGELU epilogue (dH = acc * gelu'(pre)): the [128 x 64] pre-activation slab comes by TMA into this
          // pair's slab buffer (it is free: the wait below), every thread reads ITS half row (same 128B swizzle), and the result
          // goes back into the same place -> no row-strided global accesses (the register epilogue ran these GEMMs at ~400 TFLOP/s)
          if (dgelu) {
            if (leader && !(EPI4 && prefetched)) {
              if (!EPI4) tma_wait_group_read<0>();  // the previous store of this pair has finished reading the (shared) slab
              mbar_expect_tx(smem_u32(&slab_free[pair]), EPI_SLAB_BYTES);
              tma_load_2d(xbase, &tmAux, smem_u32(&slab_free[pair]), col0, m0);
            }
            mbar_wait(smem_u32(&slab_free[pair]), aux_ph);
            aux_ph ^= 1;
#pragma unroll
            for (int i = 0; i < 4; ++i)
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                           : "=r"(ax[4 * i]), "=r"(ax[4 * i + 1]), "=r"(ax[4 * i + 2]), "=r"(ax[4 * i + 3])
                           : "r"(xrow + (((4 * half + i) ^ (prow & 7)) << 4)));
            if (EPI4) {
              // every thread of the pair has its pre-activation values: the side buffer takes the NEXT slab of this pair (same tile, or
              // the first one of the CTA's next tile) while this slab is converted; the output buffer is free once the previous store
              // has read it
              if (leader) tma_wait_group_read<0>();
              asm volatile("bar.sync %0, 256;" ::"r"(bar_id) : "memory");
              int nt = t, nsl = sl + 2;
              if (nsl >= nslab) nt = t + gridDim.x, nsl = pair;
              prefetched = false;
              if (nt < num_tiles) {
                int mn2, slice2, ka, kb;
                decode(nt, mn2, slice2, ka, kb);
                const int nm0 = (mn2 / tiles_n) * GEMM_BM, nn0 = (mn2 % tiles_n) * BN;
                if (nsl < min(BN / 64, (e.N - nn0 + 63) / 64)) {
                  prefetched = true;
                  if (leader) {
                    mbar_expect_tx(smem_u32(&slab_free[pair]), EPI_SLAB_BYTES);
                    tma_load_2d(xbase, &tmAux, smem_u32(&slab_free[pair]), nn0 + nsl * 64, nm0);
                  }
                }
              }
            }
          }
          uint32_t r[32];
          tmem_ld32(taddr + sl * 64 + half * 32, r);
          tmem_wait_ld();
          float v[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]) * alpha;
          // (K slices > 0 of a split tile add only their partial sums.)  c0 < N: with N % 64 == 32 the second half of the last slab
          // lies past N; its values are clipped by the TMA store, and bias[N .. N+31] may lie outside the caller's allocation
          if (e.bias && slice == 0 && c0 < e.N) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 bb = __ldg(reinterpret_cast<const float4*>(e.bias + c0) + i);
              v[4 * i] += bb.x, v[4 * i + 1] += bb.y, v[4 * i + 2] += bb.z, v[4 * i + 3] += bb.w;
            }
          }
          if (dgelu) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const uint32_t w = ax[i];
              float g0, g1;
              dgelu_erf2(__uint_as_float(w << 16), __uint_as_float(w & 0xFFFF0000u), g0, g1);
              v[2 * i] *= g0, v[2 * i + 1] *= g1;
            }
          }
          if (e.mode == SMBV_EPI_GELU_BF16) {
            if (save_pre) {  // training: the pre-activation (bf16) is a second output (its own slab store below)
#pragma unroll
              for (int i = 0; i < 16; ++i) ax[i] = pack_bf16(v[2 * i], v[2 * i + 1]);
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) gelu_erf2(v[2 * i], v[2 * i + 1]);
          }
#pragma unroll
          for (int i = 0; i < 16; ++i) pk[i] = pack_bf16(v[2 * i], v[2 * i + 1]);
          if (save_pre && !EPI4) {  // first hand the pre-activation slab to the TMA unit, then (below) the GELU output
            if (leader) tma_wait_group_read<0>();
            asm volatile("bar.sync %0, 256;" ::"r"(bar_id) : "memory");
            slab_store16(srow, ax);
            fence_proxy_async_smem();
            asm volatile("bar.sync %0, 256;" ::"r"(bar_id) : "memory");
            if (leader) {
              tma_store_2d(&tmAux, sbase, col0, m0);
              tma_commit_group();
            }
          }
        }
        if (sl == my_last) {  // this group's share of the accumulator is in registers: release the TMEM stage
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(smem_u32(&tempty[as]));
        }
        if (!dgelu) {  // (dGELU: the output buffer is free already — EPI4: waited for above; else each thread overwrites its own half row)
          if (leader) tma_wait_group_read<0>();          // the previous store(s) of this pair have finished reading the slab buffer(s)
          asm volatile("bar.sync %0, 256;" ::"r"(bar_id) : "memory");
        }
        if (EPI4 && save_pre) slab_store16(xrow, ax);    // second output: the pre-activation, from the side buffer
        slab_store16(srow, pk);
        fence_proxy_async_smem();                        // slab writes -> visible to the TMA unit
        asm volatile("bar.sync %0, 256;" ::"r"(bar_id) : "memory");
        if (leader) {
          if (EPI4 && save_pre) tma_store_2d(&tmAux, xbase, col0, m0);
          if (e.mode == SMBV_EPI_QKV_HEADS) {
            const int hd = e.heads * 64;
            const int part = col0 / hd, head = (col0 - part * hd) >> 6;
            const int bsmp = m0 / e.tokens, nn = m0 - bsmp * e.tokens;
            tma_store_5d(&tmC, sbase, 0, nn, head, bsmp, part);
          } else if (reduce) {
            tma_reduce_add_2d(&tmC, sbase, col0, m0);
          } else {
            tma_store_2d(&tmC, sbase, col0, m0);
          }
          tma_commit_group();
        }
      }
    }
    if (leader) tma_wait_group<0>();  // global writes complete before the kernel ends
  } else if (warp < 6) {  // ===== epilogue warps 2..5, register path (modes with a per-element side input) =====
    const int quad = warp & 3;  // TMEM lane quadrant this warp may access
    uint32_t it = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
      const uint32_t as = it & 1, aph = (it >> 1) & 1;
      int mn, slice, kb0_, kb1_;
      decode(t, mn, slice, kb0_, kb1_);
      const int m0 = (mn / tiles_n) * GEMM_BM, n0 = (mn % tiles_n) * BN;
      mbar_wait(smem_u32(&tfull[as]), aph);
      tc_fence_after();
      const int row = m0 + quad * 32 + lane;
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + as * BN;
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        uint32_t r[32];
        tmem_ld32(taddr + c * 32, r);
        tmem_wait_ld();
        const int col = n0 + c * 32;
        if (row < e.M && col < e.N) epilogue_store(e, row, col, r);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&tempty[as]));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

struct GemmHost {
  const void* A; int64_t lda; int a_layout;   // SMBV_A_*
  const void* W; int64_t ldw; int w_layout;   // 0: [N,K] row-major (K-major), 1: [K,N] row-major (MN-major)
  int64_t a_part_stride;                      // head-major A: elements between the q/k/v parts
  GemmEpi e;
};

static bool use_tma_epilogue(const GemmEpi& e) {
  switch (e.mode) {
    case SMBV_EPI_BF16:
    case SMBV_EPI_F32:
    case SMBV_EPI_ATOMIC_F32:
      return true;
    case SMBV_EPI_GELU_BF16:   // (+ the saved pre-activation of the training forward: a second slab store)
    case SMBV_EPI_DGELU_BF16:  // (the pre-activation slab comes in by TMA)
      return true;
    case SMBV_EPI_RESID_F32:
      return e.residual == e.out;  // in place: X += acc + bias as a TMA reduce-add
    case SMBV_EPI_QKV_HEADS:
      return e.tokens % GEMM_BM == 0;
    default:
      return false;
  }
}

static int make_out_tmap(CUtensorMap* m, const GemmEpi& e) {
  if (e.mode == SMBV_EPI_QKV_HEADS) {  // [3][batch][heads][tokens][64] bf16
    const uint64_t batch = (uint64_t)(e.M / e.tokens);
    uint64_t dims[5] = {64, (uint64_t)e.tokens, (uint64_t)e.heads, batch, 3};
    uint64_t str[4] = {128, (uint64_t)e.tokens * 128, (uint64_t)e.heads * e.tokens * 128, batch * e.heads * e.tokens * 128};
    uint32_t box[5] = {64, GEMM_BM, 1, 1, 1};
    return make_tmap(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, e.out, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
  }
  const bool f32 = (e.mode == SMBV_EPI_RESID_F32 || e.mode == SMBV_EPI_F32 || e.mode == SMBV_EPI_ATOMIC_F32);
  uint64_t dims[2] = {(uint64_t)e.N, (uint64_t)e.M};
  uint64_t str[1] = {(uint64_t)e.ldo * (f32 ? 4 : 2)};
  uint32_t box[2] = {(uint32_t)(f32 ? 32 : 64), GEMM_BM};
  return make_tmap(m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, e.out, dims, str, box,
                   CU_TENSOR_MAP_SWIZZLE_128B);
}

template <int BN, bool A_MN, bool B_MN, bool A3D, bool TMA_EPI, bool EPI4 = false>
static int launch_gemm(const GemmHost& h, cudaStream_t st) {
  using Cfg = GemmCfg<BN, EPI4>;
  const GemmEpi& e = h.e;
  CUtensorMap tmA, tmB, tmC, tmAux;
  int r;
  memset(&tmAux, 0, sizeof(tmAux));
  if (TMA_EPI) {
    if ((r = make_out_tmap(&tmC, e))) return r;
    if (e.aux && (e.mode == SMBV_EPI_GELU_BF16 || e.mode == SMBV_EPI_DGELU_BF16)) {  // bf16 [M, ldo] pre-activation, same geometry as out
      uint64_t dims[2] = {(uint64_t)e.N, (uint64_t)e.M};
      uint64_t str[1] = {(uint64_t)e.ldo * 2};
      uint32_t box[2] = {64, GEMM_BM};
      if ((r = make_tmap(&tmAux, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, e.aux, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B))) return r;
    }
  } else {
    memset(&tmC, 0, sizeof(tmC));
  }
  if (A3D) {  // [3][.][heads][tokens][64]; M (K-major) or K (MN-major) is the token axis
    const int tokens = A_MN ? e.K : e.M;
    uint64_t dims[4] = {64, (uint64_t)tokens, (uint64_t)e.heads, 3};
    uint64_t str[3] = {64 * 2, (uint64_t)tokens * 64 * 2, (uint64_t)h.a_part_stride * 2};
    uint32_t box[4] = {64, (uint32_t)(A_MN ? 64 : GEMM_BM), 1, 1};
    r = make_tmap(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, h.A, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
  } else if (A_MN) {  // memory [K][M]
    uint64_t dims[2] = {(uint64_t)e.M, (uint64_t)e.K};
    uint64_t str[1] = {(uint64_t)h.lda * 2};
    uint32_t box[2] = {64, 64};
    r = make_tmap(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, h.A, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
  } else {  // memory [M][K]
    uint64_t dims[2] = {(uint64_t)e.K, (uint64_t)e.M};
    uint64_t str[1] = {(uint64_t)h.lda * 2};
    uint32_t box[2] = {GEMM_BK, GEMM_BM};
    r = make_tmap(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, h.A, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
  }
  if (r) return r;
  if (B_MN) {  // memory [K][N]
    uint64_t dims[2] = {(uint64_t)e.N, (uint64_t)e.K};
    uint64_t str[1] = {(uint64_t)h.ldw * 2};
    uint32_t box[2] = {64, 64};
    r = make_tmap(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, h.W, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
  } else {  // memory [N][K]
    uint64_t dims[2] = {(uint64_t)e.K, (uint64_t)e.N};
    uint64_t str[1] = {(uint64_t)h.ldw * 2};
    uint32_t box[2] = {GEMM_BK, (uint32_t)BN};
    r = make_tmap(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, h.W, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
  }
  if (r) return r;
  const int tiles_m = (e.M + GEMM_BM - 1) / GEMM_BM, tiles_n = (e.N + BN - 1) / BN;
  static bool attr_set = false;
  if (!attr_set) {
    SMBV_CUDA(cudaFuncSetAttribute(gemm_bf16_kernel<BN, A_MN, B_MN, A3D, TMA_EPI, EPI4>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    attr_set = true;
  }
  const int grid = min(e.n_whole + (tiles_m * tiles_n - e.n_whole) * e.split_k, num_sms());
  gemm_bf16_kernel<BN, A_MN, B_MN, A3D, TMA_EPI, EPI4><<<grid, TMA_EPI ? GEMM_THREADS_TMA : GEMM_THREADS_REG, Cfg::SMEM_BYTES, st>>>(tmA, tmB, tmC, tmAux, e, tiles_m, tiles_n);
  SMBV_LAUNCH_CHECK("gemm_bf16");
  return 0;
}

static int dispatch_gemm(GemmHost& h, cudaStream_t st) {
  GemmEpi& e = h.e;
  const bool a_mn = h.a_layout == SMBV_A_TRANSPOSED || h.a_layout == SMBV_A_HEADS_T;
  const bool a3d = h.a_layout == SMBV_A_HEADS || h.a_layout == SMBV_A_HEADS_T;
  const bool b_mn = h.w_layout == 1;
  const int total_kb = (e.K + GEMM_BK - 1) / GEMM_BK;
  // fewer than two waves of 128x256 tiles: BN=128 gives more tiles (better SM fill); otherwise BN=256 halves the A re-reads
  // (measured with tools/gemm_bn_sweep.py after the elect.sync issue fix: 7168x768 outputs 477/849 vs 439/812 TF/s)
  const int64_t tiles256 = (int64_t)((e.M + 127) / 128) * ((e.N + 255) / 256);
  const bool bn256 = (e.N % 256 == 0) && tiles256 * (e.split_k > 0 ? e.split_k : 1) >= 2 * num_sms();
  int bn = bn256 ? 256 : 128;
  {  // developer override for A/B timing (tools/gemm_bn_sweep.py): SMBV_GEMM_BN=128|256
    static const int forced = [] { const char* v = getenv("SMBV_GEMM_BN"); return v ? atoi(v) : 0; }();
    if (forced == 128 || (forced == 256 && e.N % 256 == 0)) bn = forced;
  }
  if (e.split_k == 0) {  // auto: fill the machine when the output has few tiles (weight gradients)
    const int64_t tiles = (int64_t)((e.M + 127) / 128) * ((e.N + bn - 1) / bn);
    int sk = 1;
    if (e.mode == SMBV_EPI_ATOMIC_F32 && tiles < num_sms()) { int64_t want = (2 * (int64_t)num_sms() + tiles - 1) / tiles; sk = (int)(want < total_kb ? want : total_kb); }
    e.split_k = sk < 1 ? 1 : sk;
  }
  if (e.mode == SMBV_EPI_RESID_F32 && e.residual == e.out && e.split_k <= 1) {
    // in-place residual update = fp32 TMA reduce-add: the tiles of a partial last round are cut into K slices (see the kernel).
    // tail cost in units of one whole tile: rounds(k) * (1/k + fixed / total_kb), fixed ~ 3 k-blocks of epilogue + pipeline fill
    // OPT-IN (SMBV_GEMM_TAIL_SPLIT=1): the slices of one tile reduce into X in arbitrary order, so the residual stream — and with it
    // the embeddings — would no longer be bit-reproducible run to run; measured gain 8-15 % on the fc2 GEMMs = 0.5 % of a step.
    static const bool on = [] { const char* v = getenv("SMBV_GEMM_TAIL_SPLIT"); return v && v[0] == '1'; }();
    const int W = num_sms();
    const int64_t tiles = (int64_t)((e.M + 127) / 128) * ((e.N + bn - 1) / bn);
    const int R = (int)(tiles % W);
    if (on && tiles > W && R > 0) {
      const double fixed = 3.0 / total_kb;
      double best_cost = 1.0 + fixed;
      int best = 1;
      for (int k = 2; k <= 8 && k <= total_kb; ++k) {
        if ((int64_t)((total_kb + k - 1) / k) * (k - 1) >= total_kb) continue;  // would leave an empty slice
        const double cost = (double)(((int64_t)R * k + W - 1) / W) * (1.0 / k + fixed);
        if (cost < best_cost * 0.97) best_cost = cost, best = k;
      }
      if (best > 1) e.split_k = best, e.n_whole = (int)(tiles - R);
    }
  }
  while (e.split_k > 1 && (int64_t)((total_kb + e.split_k - 1) / e.split_k) * (e.split_k - 1) >= total_kb) --e.split_k;  // no empty slice
  const bool tma_epi = use_tma_epilogue(e);
  // the two-transfer epilogues (dGELU: pre-activation slab in, gradient slab out; GELU with the saved pre-activation: two slabs out)
  // run on the four-slab-buffer variant (plain row-major A; W [N,K] for the forward fc1, W [K,N] for the fc2 dgrad)
  static const bool epi4_on = [] { const char* v = getenv("SMBV_GEMM_EPI4"); return !(v && v[0] == '0'); }();
  // (measured, tools/gemm_small_sweep.py: dGELU 51.9 -> 47.6 us at M=7168, K=768 and 68.4 -> 57.8 us at M=20480, K=384; GELU + pre 51.5 -> 49.3 us
  //  at K=384 but 43.6 -> 45.3 us at K=768, where the third stage is missed: only short main loops take it)
  if (epi4_on && tma_epi && !a_mn && !a3d && e.aux && (e.mode == SMBV_EPI_DGELU_BF16 || (e.mode == SMBV_EPI_GELU_BF16 && e.K <= 512))) {
    if (bn == 256) return b_mn ? launch_gemm<256, false, true, false, true, true>(h, st) : launch_gemm<256, false, false, false, true, true>(h, st);
    return b_mn ? launch_gemm<128, false, true, false, true, true>(h, st) : launch_gemm<128, false, false, false, true, true>(h, st);
  }
#define SMBV_GEMM_CASE(BN_, AMN, BMN, A3)                                                  \
  if (bn == BN_ && a_mn == AMN && b_mn == BMN && a3d == A3)                                \
    return tma_epi ? launch_gemm<BN_, AMN, BMN, A3, true>(h, st) : launch_gemm<BN_, AMN, BMN, A3, false>(h, st);
  SMBV_GEMM_CASE(256, false, false, false) SMBV_GEMM_CASE(128, false, false, false)
  SMBV_GEMM_CASE(256, false, true, false)  SMBV_GEMM_CASE(128, false, true, false)
  SMBV_GEMM_CASE(256, true, true, false)   SMBV_GEMM_CASE(128, true, true, false)
  SMBV_GEMM_CASE(256, false, true, true)   SMBV_GEMM_CASE(128, false, true, true)
  SMBV_GEMM_CASE(256, true, true, true)    SMBV_GEMM_CASE(128, true, true, true)
#undef SMBV_GEMM_CASE
  set_error("gemm: unsupported operand layout combination a_layout=%d w_layout=%d", h.a_layout, h.w_layout);
  return -1;
}

}  // namespace smbv

using namespace smbv;

static int check_common(const void* A, const void* W, const void* out, int M, int N, int K, const float* bias, int epilogue) {
  SMBV_ARG(A && W && out, "gemm: null pointer");
  SMBV_ARG(M > 0 && N > 0 && K > 0, "gemm: bad shape M=%d N=%d K=%d", M, N, K);
  SMBV_ARG(N % 32 == 0, "gemm: N=%d must be a multiple of 32", N);
  SMBV_ARG((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0 &&
               (reinterpret_cast<uintptr_t>(out) & 15) == 0,
           "gemm: A/W/out must be 16-byte aligned");
  SMBV_ARG(epilogue >= SMBV_EPI_BF16 && epilogue <= SMBV_EPI_DGELU_BF16, "gemm: unknown epilogue %d", epilogue);
  if (bias) SMBV_ARG((reinterpret_cast<uintptr_t>(bias) & 15) == 0, "gemm: bias must be 16-byte aligned");
  return 0;
}

extern "C" int smbv_gemm_bf16(const smbv_gemm_args* a, smbv_stream_t st) {
  SMBV_ARG(a != nullptr, "gemm_bf16: null args");
  if (int r = check_common(a->A, a->W, a->out, a->M, a->N, a->K, a->bias, a->epilogue)) return r;
  SMBV_ARG(a->epilogue <= SMBV_EPI_POS_GATHER_F32, "gemm_bf16: epilogue %d needs smbv_gemm_ex", a->epilogue);
  SMBV_ARG(a->K % 8 == 0 && a->lda % 8 == 0 && a->ldw % 8 == 0 && a->lda >= a->K && a->ldw >= a->K,
           "gemm_bf16: K/lda/ldw must be multiples of 8 (16-byte TMA rows): K=%d lda=%lld ldw=%lld", a->K,
           (long long)a->lda, (long long)a->ldw);
  if (a->epilogue == SMBV_EPI_QKV_HEADS) {
    SMBV_ARG(a->heads > 0 && a->tokens > 0 && a->N == 3 * a->heads * 64 && a->M % a->tokens == 0,
             "gemm_bf16: QKV epilogue needs N == 3*heads*64 and M %% tokens == 0 (N=%d heads=%d M=%d tokens=%d)", a->N,
             a->heads, a->M, a->tokens);
  } else {
    SMBV_ARG(a->ldo >= a->N && a->ldo % 8 == 0, "gemm_bf16: ldo=%lld must be >= N and a multiple of 8", (long long)a->ldo);
  }
  if (a->epilogue == SMBV_EPI_RESID_F32) SMBV_ARG(a->residual != nullptr, "gemm_bf16: residual epilogue without residual");
  if (a->epilogue == SMBV_EPI_POS_GATHER_F32)
    SMBV_ARG(a->pos && a->row_map && a->ldpos >= a->N && a->ldpos % 4 == 0, "gemm_bf16: pos-gather epilogue needs pos,row_map,ldpos");
  GemmHost h{};
  h.A = a->A, h.lda = a->lda, h.a_layout = SMBV_A_ROWMAJOR, h.W = a->W, h.ldw = a->ldw, h.w_layout = 0;
  h.e = GemmEpi{a->M, a->N, a->K, 1, 0, nullptr, nullptr, a->bias, a->epilogue, a->out, a->ldo, a->residual, a->heads, a->tokens, a->pos, a->ldpos, a->row_map};
  return dispatch_gemm(h, (cudaStream_t)st);
}

extern "C" int smbv_gemm_ex(const smbv_gemm_ex_args* a, smbv_stream_t st) {
  SMBV_ARG(a != nullptr, "gemm_ex: null args");
  if (int r = check_common(a->A, a->W, a->out, a->M, a->N, a->K, a->bias, a->epilogue)) return r;
  SMBV_ARG(a->a_layout >= SMBV_A_ROWMAJOR && a->a_layout <= SMBV_A_HEADS_T, "gemm_ex: bad a_layout %d", a->a_layout);
  SMBV_ARG(a->w_layout == 0 || a->w_layout == 1, "gemm_ex: bad w_layout %d", a->w_layout);
  SMBV_ARG(a->epilogue == SMBV_EPI_BF16 || a->epilogue == SMBV_EPI_F32 || a->epilogue == SMBV_EPI_ATOMIC_F32 ||
               a->epilogue == SMBV_EPI_DGELU_BF16 || a->epilogue == SMBV_EPI_RESID_F32 || a->epilogue == SMBV_EPI_GELU_BF16,
           "gemm_ex: epilogue %d not supported here", a->epilogue);
  SMBV_ARG(a->ldo >= a->N && a->ldo % 8 == 0, "gemm_ex: ldo=%lld must be >= N and a multiple of 8", (long long)a->ldo);
  SMBV_ARG(a->split_k >= 0 && (a->split_k <= 1 || a->epilogue == SMBV_EPI_ATOMIC_F32), "gemm_ex: split_k > 1 needs the atomic epilogue");
  if (a->a_layout == SMBV_A_ROWMAJOR) SMBV_ARG(a->lda >= a->K && a->lda % 8 == 0, "gemm_ex: bad lda");
  if (a->a_layout == SMBV_A_TRANSPOSED) SMBV_ARG(a->lda >= a->M && a->lda % 8 == 0, "gemm_ex: bad lda (transposed A)");
  if (a->a_layout == SMBV_A_HEADS) SMBV_ARG(a->heads > 0 && a->K == 3 * a->heads * 64, "gemm_ex: head-major A needs K == 3*heads*64");
  if (a->a_layout == SMBV_A_HEADS_T) SMBV_ARG(a->heads > 0 && a->M == 3 * a->heads * 64, "gemm_ex: head-major A^T needs M == 3*heads*64");
  if (a->w_layout == 0) SMBV_ARG(a->ldw >= a->K && a->ldw % 8 == 0, "gemm_ex: bad ldw");
  else SMBV_ARG(a->ldw >= a->N && a->ldw % 8 == 0, "gemm_ex: bad ldw (transposed W)");
  if (a->epilogue == SMBV_EPI_DGELU_BF16) SMBV_ARG(a->aux != nullptr, "gemm_ex: dGELU epilogue needs aux (pre-activation)");
  if (a->epilogue == SMBV_EPI_RESID_F32) SMBV_ARG(a->residual != nullptr, "gemm_ex: residual epilogue without residual");
  GemmHost h{};
  h.A = a->A, h.lda = a->lda, h.a_layout = a->a_layout, h.W = a->W, h.ldw = a->ldw, h.w_layout = a->w_layout;
  h.a_part_stride = a->a_part_stride;
  h.e = GemmEpi{a->M, a->N, a->K, a->split_k, 0, a->aux, a->alpha, a->bias, a->epilogue, a->out, a->ldo, a->residual, a->heads, 0, nullptr, 0, nullptr};
  return dispatch_gemm(h, (cudaStream_t)st);
}
