// V-JEPA2-3D rotary position embedding of the queries and keys (SURVEY.md §8f rank 4; reference
// src/models/vjepa/modeling_vjepa.py:204-228 `rotate_queries_or_keys`, :297-330 `get_position_ids` /
// `apply_rotary_embeddings`), in place on the head-major bf16 Q/K sections the QKV GEMM epilogue writes.
//
// Semantics restated: the head dimension D is cut into three segments of S = 2*((D/3)/2) elements (frame, height, width
// position) and a tail of D - 3S elements that is passed through.  Inside a segment, with h = S/2 and
// omega_j = 10000^(-j/h), element e (segment-local) is paired with e^1 and
//     out[e] = x[e] * cos(p * omega[e mod h]) + (e even ? -x[e+1] : x[e-1]) * sin(p * omega[e mod h])
// — the reference tiles the h angles twice (`.repeat(1,1,1,2)`) while pairing adjacent elements, so the two elements of a
// pair use DIFFERENT angles (e mod h and (e+1) mod h).  That is kept exactly; it makes the map a general 2x2 block per
// pair rather than a rotation, so the backward pass needs the explicit transpose (`transpose` = 1).
// The position p of a token is derived from its id (ids[b, t], or t when ids == NULL):
//     frame = id / (gs*gs), height = (id - frame*gs*gs) / gs, width = the remainder   (gs = crop_size / patch_size).
//
// Roofline: HBM, 2 B read + 2 B written per element, one 16-byte chunk (8 elements) per thread; the cos/sin table of the
// first `max_pos` positions is built once per CTA in shared memory (positions beyond it — the reference allows
// extrapolating ids — fall back to sincosf).  rope3d_kernel (round 1) measured 931 GB/s = 14 % of the HBM peak — its
// per-element segment / angle index arithmetic divides by run-time values; rope3d_v2_kernel below is the default.
#include "common.cuh"
#include "../../include/smbv_b200.h"

namespace smbv {

struct RopeArgs {
  int64_t chunks;        // total 16-byte chunks = G*B*H*n*D/8
  int B, H, n, D;
  int seg, half;         // S and h
  int gs, max_pos;
  int transpose;
};

__device__ __forceinline__ float rope_omega(int j, int half) { return 1.0f / powf(10000.0f, (float)j / (float)half); }

__global__ void __launch_bounds__(256) rope3d_kernel(__nv_bfloat16* __restrict__ x, const int32_t* __restrict__ ids, RopeArgs a) {
  extern __shared__ float2 cs[];  // [max_pos][half] (cos, sin)
  for (int i = threadIdx.x; i < a.max_pos * a.half; i += blockDim.x) {
    const int p = i / a.half, j = i - p * a.half;
    float s, c;
    sincosf((float)p * rope_omega(j, a.half), &s, &c);
    cs[i] = make_float2(c, s);
  }
  __syncthreads();
  const int cpr = a.D / 8;  // chunks per row
  for (int64_t ch = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; ch < a.chunks; ch += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = ch / cpr;
    const int e0 = (int)(ch - row * cpr) * 8;
    if (e0 >= 3 * a.seg) continue;  // pass-through tail
    const int t = (int)(row % a.n);
    const int b = (int)((row / ((int64_t)a.n * a.H)) % a.B);
    const int id = ids ? ids[(int64_t)b * a.n + t] : t;
    const int frame = id / (a.gs * a.gs);
    const int rem = id - frame * a.gs * a.gs;
    const int hh = rem / a.gs;
    const int pos3[3] = {frame, hh, rem - hh * a.gs};
    uint4* p4 = reinterpret_cast<uint4*>(x + row * a.D + e0);
    uint4 raw = *p4;
    __nv_bfloat16* v = reinterpret_cast<__nv_bfloat16*>(&raw);
    float in[8], c[8], s[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      in[i] = __bfloat162float(v[i]);
      const int e = e0 + i;
      if (e < 3 * a.seg) {
        const int sg = e / a.seg, l = e - sg * a.seg, j = l % a.half;
        const int p = sg == 0 ? pos3[0] : sg == 1 ? pos3[1] : pos3[2];
        if (p < a.max_pos) {
          const float2 t2 = cs[p * a.half + j];
          c[i] = t2.x, s[i] = t2.y;
        } else {
          sincosf((float)p * rope_omega(j, a.half), &s[i], &c[i]);
        }
      } else {
        c[i] = 1.f, s[i] = 0.f;
      }
    }
#pragma unroll
    for (int i = 0; i < 8; i += 2) {
      if (e0 + i >= 3 * a.seg) continue;  // pass-through pair (3*seg is even): keep its bits, -0.0 included
      float o0, o1;
      // explicit products / fused adds: both kernels round identically (no compiler-chosen FMA contraction)
      if (!a.transpose) {
        o0 = __fmaf_rn(in[i], c[i], -__fmul_rn(in[i + 1], s[i]));
        o1 = __fmaf_rn(in[i + 1], c[i + 1], __fmul_rn(in[i], s[i + 1]));
      } else {
        o0 = __fmaf_rn(in[i], c[i], __fmul_rn(in[i + 1], s[i + 1]));
        o1 = __fmaf_rn(in[i + 1], c[i + 1], -__fmul_rn(in[i], s[i]));
      }
      v[i] = __float2bfloat16_rn(o0), v[i + 1] = __float2bfloat16_rn(o1);
    }
    *p4 = raw;
  }
}

// ---- default kernel -----------------------------------------------------------------------------------------------
// Same map without the per-element divisions that held rope3d_kernel at 14 % of the HBM peak (46 MUFU.RCP per 16-byte
// chunk): a 2-D grid (x: blocks of ROPE2_ROWS tokens, y: the (section, batch, head) row group) so that no thread decomposes
// a flat chunk index; a per-CTA table of (segment, angle index) codes for the D head elements, read back 8 codes at a time
// and kept in registers for all rows of the thread; the token position is decoded by two multiply-shift divisions (exact
// for id < 2^24, divisor < 2^16: magic = ceil(2^40 / d)); four rows per thread are in flight (loads first, then math, then
// stores) so that the in-place read-modify-write does not serialise on its own stores.
constexpr int ROPE2_ROWS = 512;
constexpr int ROPE2_BATCH = 4;

__device__ __noinline__ float2 rope_cs_slow(int p, int j, int half) {  // positions beyond the table (extrapolated ids)
  float s, c;
  sincosf((float)p * rope_omega(j, half), &s, &c);
  return make_float2(c, s);
}
__device__ __forceinline__ float2 rope_cs(const float2* cs, int p, int j, int half, int max_pos) {
  return p < max_pos ? cs[p * half + j] : rope_cs_slow(p, j, half);
}
__device__ __forceinline__ int rope_div(int x, uint64_t magic) { return (int)(((uint64_t)(uint32_t)x * magic) >> 40); }

__global__ void __launch_bounds__(256, 3) rope3d_v2_kernel(__nv_bfloat16* __restrict__ x, const int32_t* __restrict__ ids, RopeArgs a,
                                                        uint64_t magic_g2, uint64_t magic_gs) {
  extern __shared__ float2 cs[];                       // [max_pos][half] (cos, sin)
  __shared__ __align__(16) uint16_t el[256];           // per head element: (segment << 8) | angle index; 0xFFFF = pass-through
  for (int i = threadIdx.x; i < a.max_pos * a.half; i += blockDim.x) {
    const int p = i / a.half, j = i - p * a.half;
    float s, c;
    sincosf((float)p * rope_omega(j, a.half), &s, &c);
    cs[i] = make_float2(c, s);
  }
  for (int e = threadIdx.x; e < a.D; e += blockDim.x) {
    if (e < 3 * a.seg) {
      const int sg = e / a.seg, l = e - sg * a.seg;
      el[e] = (uint16_t)((sg << 8) | (l % a.half));
    } else {
      el[e] = 0xFFFFu;
    }
  }
  __syncthreads();
  const int cpr = a.D / 8;                             // chunks per row
  const int rpp = 256 / cpr;                           // rows per pass
  const int r = threadIdx.x / cpr, c8 = threadIdx.x - r * cpr;
  if (r >= rpp || c8 * 8 >= 3 * a.seg) return;         // idle lanes (256 % cpr != 0) and the pass-through tail chunks
  const int b = (int)((blockIdx.y / a.H) % a.B);
  const int g2 = a.gs * a.gs;
  int ee[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) ee[i] = el[c8 * 8 + i];
  const int t_end = min(a.n, ((int)blockIdx.x + 1) * ROPE2_ROWS);
  __nv_bfloat16* base = x + (int64_t)blockIdx.y * a.n * a.D + c8 * 8;
  const int32_t* idrow = ids ? ids + (int64_t)b * a.n : nullptr;
  for (int t0 = (int)blockIdx.x * ROPE2_ROWS + r; t0 < t_end; t0 += rpp * ROPE2_BATCH) {
    uint4 raw[ROPE2_BATCH];
    int id[ROPE2_BATCH];
#pragma unroll
    for (int u = 0; u < ROPE2_BATCH; ++u) {
      const int t = t0 + u * rpp;
      if (t < t_end) {
        raw[u] = *reinterpret_cast<const uint4*>(base + (int64_t)t * a.D);
        id[u] = idrow ? idrow[t] : t;
      }
    }
#pragma unroll
    for (int u = 0; u < ROPE2_BATCH; ++u) {
      const int t = t0 + u * rpp;
      if (t >= t_end) continue;
      const int p0 = rope_div(id[u], magic_g2);
      const int rem = id[u] - p0 * g2;
      const int p1 = rope_div(rem, magic_gs);
      const int p2 = rem - p1 * a.gs;
      uint32_t* w = reinterpret_cast<uint32_t*>(&raw[u]);
      const bool fast = max(p0, max(p1, p2)) < a.max_pos;  // all three positions inside the table: no per-element branch
      const int pb0 = p0 * a.half, pb1 = p1 * a.half, pb2 = p2 * a.half;
#pragma unroll
      for (int i = 0; i < 4; ++i) {  // one adjacent pair per 32-bit word
        const int code0 = ee[2 * i], code1 = ee[2 * i + 1];
        if (code0 == 0xFFFF) continue;  // pass-through pair (3*seg is even, so code1 is 0xFFFF too): keep its bits, -0.0 included
        const float x0 = __uint_as_float(w[i] << 16), x1 = __uint_as_float(w[i] & 0xFFFF0000u);
        float2 a0 = make_float2(1.f, 0.f), a1 = make_float2(1.f, 0.f);
        if (fast) {
          if (code0 != 0xFFFF) a0 = cs[((code0 >> 8) == 0 ? pb0 : (code0 >> 8) == 1 ? pb1 : pb2) + (code0 & 0xFF)];
          if (code1 != 0xFFFF) a1 = cs[((code1 >> 8) == 0 ? pb0 : (code1 >> 8) == 1 ? pb1 : pb2) + (code1 & 0xFF)];
        } else {
          if (code0 != 0xFFFF) a0 = rope_cs(cs, (code0 >> 8) == 0 ? p0 : (code0 >> 8) == 1 ? p1 : p2, code0 & 0xFF, a.half, a.max_pos);
          if (code1 != 0xFFFF) a1 = rope_cs(cs, (code1 >> 8) == 0 ? p0 : (code1 >> 8) == 1 ? p1 : p2, code1 & 0xFF, a.half, a.max_pos);
        }
        float o0, o1;
        if (!a.transpose) {
          o0 = __fmaf_rn(x0, a0.x, -__fmul_rn(x1, a0.y));
          o1 = __fmaf_rn(x1, a1.x, __fmul_rn(x0, a1.y));
        } else {
          o0 = __fmaf_rn(x0, a0.x, __fmul_rn(x1, a1.y));
          o1 = __fmaf_rn(x1, a1.x, -__fmul_rn(x0, a0.y));
        }
        w[i] = pack_bf16(o0, o1);
      }
      *reinterpret_cast<uint4*>(base + (int64_t)t * a.D) = raw[u];
    }
  }
}

}  // namespace smbv

using namespace smbv;

extern "C" int smbv_rope3d(smbv_bf16* x, const int32_t* ids, int G, int B, int H, int n, int D, int grid_size, int max_pos,
                           int transpose, smbv_stream_t st) {
  SMBV_ARG(x, "rope3d: null pointer");
  SMBV_ARG(G > 0 && B > 0 && H > 0 && n > 0, "rope3d: bad sizes G=%d B=%d H=%d n=%d", G, B, H, n);
  SMBV_ARG(D >= 8 && D % 8 == 0 && D <= 256, "rope3d: head_dim %d must be a multiple of 8 (<= 256)", D);
  SMBV_ARG(grid_size > 0 && max_pos > 0, "rope3d: grid_size and max_pos must be positive");
  SMBV_ARG((reinterpret_cast<uintptr_t>(x) & 15) == 0, "rope3d: x must be 16-byte aligned");
  RopeArgs a;
  a.B = B, a.H = H, a.n = n, a.D = D;
  a.seg = 2 * ((D / 3) / 2), a.half = a.seg / 2;
  if (a.seg == 0) return 0;  // head_dim < 6: nothing is rotated
  a.gs = grid_size, a.max_pos = max_pos, a.transpose = (transpose & 1) ? 1 : 0;
  a.chunks = (int64_t)G * B * H * n * (D / 8);
  const size_t smem = (size_t)max_pos * a.half * sizeof(float2);
  SMBV_ARG(smem <= 40 * 1024, "rope3d: max_pos=%d too large for the shared-memory table", max_pos);
  // ids are token indices of a grid_size^2 x frames lattice: < 2^24 for every volume this library takes (512x512x320 -> 20480);
  // `transpose` & 2 selects the first-generation kernel (kept as the independent cross-check of tests/test_gpu_vjepa.py)
  if (!(transpose & 2) && (int64_t)G * B * H <= 65535 && grid_size < 256) {  // gs^2 < 2^16: the multiply-shift division is exact
    const uint64_t g2 = (uint64_t)grid_size * grid_size;
    const uint64_t magic_g2 = ((1ull << 40) + g2 - 1) / g2, magic_gs = ((1ull << 40) + grid_size - 1) / (uint64_t)grid_size;
    dim3 grid2((unsigned)((n + ROPE2_ROWS - 1) / ROPE2_ROWS), (unsigned)(G * B * H));
    rope3d_v2_kernel<<<grid2, 256, smem, (cudaStream_t)st>>>(reinterpret_cast<__nv_bfloat16*>(x), ids, a, magic_g2, magic_gs);
    SMBV_LAUNCH_CHECK("rope3d_v2");
    return 0;
  }
  const int64_t want = (a.chunks + 255) / 256;
  const int grid = (int)(want < (int64_t)num_sms() * 8 ? want : (int64_t)num_sms() * 8);
  rope3d_kernel<<<grid, 256, smem, (cudaStream_t)st>>>(reinterpret_cast<__nv_bfloat16*>(x), ids, a);
  SMBV_LAUNCH_CHECK("rope3d");
  return 0;
}
