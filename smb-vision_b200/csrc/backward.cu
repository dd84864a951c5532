// HBM-bound kernels of the backward pass: LayerNorm backward (fused with the residual-gradient accumulation and the
// bf16 re-cast the next GEMM needs), bias / mask-token gradients (column sums), visible-patch gather for the
// patch-embedding weight gradient.  Autograd semantics of the reference modules (modeling_videomae.py:402-431, :495-505).
#include "common.cuh"
#include "../../include/smbv_b200.h"

namespace smbv {

// ------------------------------------------------------------------------------------------------
// LayerNorm backward, two kernels (a fused single kernel needed ~190 registers -> 8 warps/SM):
//  (rows)    one warp per row:  xhat = (x - mean) rstd ; g = dy * gamma ; dx = rstd (g - mean(g) - xhat mean(g xhat))
//            dres (fp32 residual-stream gradient) (+)= dx (+ extra) ; optional bf16 copy of the updated dres for the next GEMM.
//            `extra` (or NULL): a second fp32 addend of the same shape — the gradient of a hidden state returned by
//            `output_hidden_states`, which joins the residual-stream gradient at this layer boundary
//  (columns) dgamma[c] += sum_rows dy * xhat ; dbeta[c] += sum_rows dy   (lane = 8 columns, warps stride over rows)
// ------------------------------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(256) layernorm_bwd_rows_kernel(const __nv_bfloat16* __restrict__ dy, const float* __restrict__ x,
                                                                 const float* __restrict__ mean, const float* __restrict__ rstd,
                                                                 const float* __restrict__ gamma, int M, int d,
                                                                 float* __restrict__ dres, int accumulate,
                                                                 __nv_bfloat16* __restrict__ dres_bf16,
                                                                 const float* __restrict__ extra) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= M) return;
  const int nvec = d >> 2;
  const float inv_d = 1.f / (float)d;
  const float mu = mean[row], rs = rstd[row];
  const float4* xr = reinterpret_cast<const float4*>(x + (int64_t)row * d);
  const uint2* dyr = reinterpret_cast<const uint2*>(dy + (int64_t)row * d);
  float4* dr = reinterpret_cast<float4*>(dres + (int64_t)row * d);
  const float4* er = extra ? reinterpret_cast<const float4*>(extra + (int64_t)row * d) : nullptr;
  float4 xh[NV], g[NV], prev[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) {  // every load of the row is issued before the first use
    const int c = lane + 32 * i;
    xh[i] = c < nvec ? xr[c] : make_float4(0.f, 0.f, 0.f, 0.f);
    const uint2 dv = c < nvec ? dyr[c] : make_uint2(0u, 0u);
    const __nv_bfloat162 d01 = *reinterpret_cast<const __nv_bfloat162*>(&dv.x), d23 = *reinterpret_cast<const __nv_bfloat162*>(&dv.y);
    g[i] = make_float4(__low2float(d01), __high2float(d01), __low2float(d23), __high2float(d23));
    prev[i] = (accumulate && c < nvec) ? dr[c] : make_float4(0.f, 0.f, 0.f, 0.f);
    if (er && c < nvec) {
      const float4 e = er[c];
      prev[i] = make_float4(prev[i].x + e.x, prev[i].y + e.y, prev[i].z + e.z, prev[i].w + e.w);
    }
  }
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = lane + 32 * i;
    if (c < nvec) {
      const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma) + c);
      xh[i] = make_float4((xh[i].x - mu) * rs, (xh[i].y - mu) * rs, (xh[i].z - mu) * rs, (xh[i].w - mu) * rs);
      g[i] = make_float4(g[i].x * gm.x, g[i].y * gm.y, g[i].z * gm.z, g[i].w * gm.w);
      s1 += (g[i].x + g[i].y) + (g[i].z + g[i].w);
      s2 += (g[i].x * xh[i].x + g[i].y * xh[i].y) + (g[i].z * xh[i].z + g[i].w * xh[i].w);
    }
  }
  const float c1 = warp_sum(s1) * inv_d, c2 = warp_sum(s2) * inv_d;
  uint2* drb = dres_bf16 ? reinterpret_cast<uint2*>(dres_bf16 + (int64_t)row * d) : nullptr;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = lane + 32 * i;
    if (c < nvec) {
      const float4 o = make_float4(rs * (g[i].x - c1 - xh[i].x * c2) + prev[i].x, rs * (g[i].y - c1 - xh[i].y * c2) + prev[i].y,
                                   rs * (g[i].z - c1 - xh[i].z * c2) + prev[i].z, rs * (g[i].w - c1 - xh[i].w * c2) + prev[i].w);
      dr[c] = o;
      if (drb) drb[c] = make_uint2(pack_bf16(o.x, o.y), pack_bf16(o.z, o.w));
    }
  }
}

__global__ void __launch_bounds__(256) layernorm_bwd_params_kernel(const __nv_bfloat16* __restrict__ dy, const float* __restrict__ x,
                                                                   const float* __restrict__ mean, const float* __restrict__ rstd,
                                                                   int M, int d, float* __restrict__ dgamma, float* __restrict__ dbeta) {
  __shared__ float sh[8][256];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int col = blockIdx.x * 256 + lane * 8;
  float ag[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, ab[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (col < d) {
    for (int r = blockIdx.y * 8 + warp; r < M; r += gridDim.y * 8) {
      const float mu = mean[r], rs = rstd[r];
      const uint4 dv = ldg_stream_u4(dy + (int64_t)r * d + col);
      const float4 x0 = ldg_stream_f4(x + (int64_t)r * d + col), x1 = ldg_stream_f4(x + (int64_t)r * d + col + 4);
      const uint32_t w[4] = {dv.x, dv.y, dv.z, dv.w};
      const float xv[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const __nv_bfloat162 p = *reinterpret_cast<const __nv_bfloat162*>(&w[q]);
        const float d0 = __low2float(p), d1 = __high2float(p);
        ag[2 * q] += d0 * (xv[2 * q] - mu) * rs, ag[2 * q + 1] += d1 * (xv[2 * q + 1] - mu) * rs;
        ab[2 * q] += d0, ab[2 * q + 1] += d1;
      }
    }
  }
#pragma unroll
  for (int pass = 0; pass < 2; ++pass) {
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 8; ++q) sh[warp][lane * 8 + q] = pass == 0 ? ag[q] : ab[q];
    __syncthreads();
    float s = 0.f;
#pragma unroll
    for (int w2 = 0; w2 < 8; ++w2) s += sh[w2][threadIdx.x];
    const int c = blockIdx.x * 256 + threadIdx.x;
    if (c < d) atomicAdd((pass == 0 ? dgamma : dbeta) + c, s);
  }
}

// ------------------------------------------------------------------------------------------------
// column sums (bias gradients): out[n] += sum_m x[m, n]
// ------------------------------------------------------------------------------------------------
// zH > 0: x is the head-major [3][zB][zH][M][64] buffer; blockIdx.z = (part, b, h) and out is [3*zH*64]
__global__ void __launch_bounds__(256) colsum_bf16_kernel(const __nv_bfloat16* __restrict__ x, int M, int N, int64_t ld,
                                                          float* __restrict__ out, int zB, int zH, int skip_part) {
  __shared__ float sh[8][256];
  if (zH > 0) {
    const int z = blockIdx.z;
    if (z / (zB * zH) == skip_part) return;
    x += (int64_t)z * M * 64;
    out += ((z / (zB * zH)) * zH + z % zH) * 64;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int col = blockIdx.x * 256 + lane * 8;  // 8 bf16 = 16 B per lane
  float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (col < N) {
    int r = blockIdx.y * 8 + warp;
    const int step = gridDim.y * 8;
    for (; r + step < M; r += 2 * step) {  // two independent rows in flight per warp
      const uint4 v0 = ldg_stream_u4(x + (int64_t)r * ld + col), v1 = ldg_stream_u4(x + (int64_t)(r + step) * ld + col);
      const uint32_t w0[4] = {v0.x, v0.y, v0.z, v0.w}, w1[4] = {v1.x, v1.y, v1.z, v1.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const __nv_bfloat162 p = *reinterpret_cast<const __nv_bfloat162*>(&w0[q]), t = *reinterpret_cast<const __nv_bfloat162*>(&w1[q]);
        a[2 * q] += __low2float(p) + __low2float(t), a[2 * q + 1] += __high2float(p) + __high2float(t);
      }
    }
    if (r < M) {
      const uint4 v0 = ldg_stream_u4(x + (int64_t)r * ld + col);
      const uint32_t w0[4] = {v0.x, v0.y, v0.z, v0.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const __nv_bfloat162 p = *reinterpret_cast<const __nv_bfloat162*>(&w0[q]);
        a[2 * q] += __low2float(p), a[2 * q + 1] += __high2float(p);
      }
    }
  }
#pragma unroll
  for (int q = 0; q < 8; ++q) sh[warp][lane * 8 + q] = a[q];
  __syncthreads();
  float s = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) s += sh[w][threadIdx.x];
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c < N) atomicAdd(out + c, s);
}

__global__ void __launch_bounds__(256) colsum_f32_kernel(const float* __restrict__ x, int M, int N, int64_t ld,
                                                         float* __restrict__ out) {
  __shared__ float sh[8][128];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int col = blockIdx.x * 128 + lane * 4;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  if (col < N) {
    for (int r = blockIdx.y * 8 + warp; r < M; r += gridDim.y * 8) {
      const float4 v = *reinterpret_cast<const float4*>(x + (int64_t)r * ld + col);
      a.x += v.x, a.y += v.y, a.z += v.z, a.w += v.w;
    }
  }
  sh[warp][lane * 4] = a.x, sh[warp][lane * 4 + 1] = a.y, sh[warp][lane * 4 + 2] = a.z, sh[warp][lane * 4 + 3] = a.w;
  __syncthreads();
  if (threadIdx.x < 128) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += sh[w][threadIdx.x];
    const int c = blockIdx.x * 128 + threadIdx.x;
    if (c < N) atomicAdd(out + c, s);
  }
}

// ------------------------------------------------------------------------------------------------
// visible-patch gather: out[b*nv + i, k] = bf16(volume patch vis_idx[b,i], voxel k)   (k = dz*256 + dy*16 + dx)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gather_patches_kernel(const float* __restrict__ vol, int T, int H, int W,
                                                             const int32_t* __restrict__ idx, int n_sel, int idx_stride,
                                                             __nv_bfloat16* __restrict__ out) {
  const int i = blockIdx.x, b = blockIdx.y, t = threadIdx.x;
  const int n = idx[(int64_t)b * idx_stride + i];
  const int gy = H >> 4, gx = W >> 4;
  const int tx = n % gx, ty = (n / gx) % gy, tz = n / (gx * gy);
  const int dz = t >> 4, dy = t & 15;
  const float* src = vol + (((int64_t)b * T + (tz * 16 + dz)) * H + (ty * 16 + dy)) * W + tx * 16;
  uint32_t w[8];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float4 v = ldg_stream_f4(src + 4 * q);
    w[2 * q] = pack_bf16(v.x, v.y), w[2 * q + 1] = pack_bf16(v.z, v.w);
  }
  uint4* dst = reinterpret_cast<uint4*>(out + ((int64_t)b * n_sel + i) * 4096 + t * 16);
  dst[0] = make_uint4(w[0], w[1], w[2], w[3]);
  dst[1] = make_uint4(w[4], w[5], w[6], w[7]);
}

}  // namespace smbv

using namespace smbv;

static int layernorm_bwd_launch(const smbv_bf16* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                                int M, int d, float* dres, int accumulate, smbv_bf16* dres_bf16, float* dgamma, float* dbeta,
                                const float* extra, cudaStream_t s) {
  const int nv = (d / 4 + 31) / 32;
  const __nv_bfloat16* dyy = reinterpret_cast<const __nv_bfloat16*>(dy);
  __nv_bfloat16* db = reinterpret_cast<__nv_bfloat16*>(dres_bf16);
  const int grid = (M + 7) / 8;
#define LNB_CASE(NV)                                                                                                  \
  case NV:                                                                                                            \
    layernorm_bwd_rows_kernel<NV><<<grid, 256, 0, s>>>(dyy, x, mean, rstd, gamma, M, d, dres, accumulate, db, extra);  \
    break;
  switch (nv <= 1 ? 1 : nv <= 2 ? 2 : nv <= 3 ? 3 : nv <= 4 ? 4 : nv <= 6 ? 6 : 8) {
    LNB_CASE(1) LNB_CASE(2) LNB_CASE(3) LNB_CASE(4) LNB_CASE(6) LNB_CASE(8)
  }
#undef LNB_CASE
  SMBV_LAUNCH_CHECK("layernorm_bwd_rows");
  dim3 pgrid((d + 255) / 256, max(1, min(256, M / 32)));
  layernorm_bwd_params_kernel<<<pgrid, 256, 0, s>>>(dyy, x, mean, rstd, M, d, dgamma, dbeta);
  SMBV_LAUNCH_CHECK("layernorm_bwd_params");
  return 0;
}

extern "C" int smbv_layernorm_bwd(const smbv_bf16* dy, const float* x, const float* mean, const float* rstd,
                                  const float* gamma, int M, int d, float* dres, int accumulate, smbv_bf16* dres_bf16,
                                  float* dgamma, float* dbeta, float* workspace, smbv_stream_t st) {
  (void)workspace;  // kept in the ABI; the two-kernel version needs none
  SMBV_ARG(dy && x && mean && rstd && gamma && dres && dgamma && dbeta, "layernorm_bwd: null pointer");
  SMBV_ARG(M > 0 && d > 0 && d % 8 == 0 && d <= 1024, "layernorm_bwd: need d %% 8 == 0 and d <= 1024 (got M=%d d=%d)", M, d);
  SMBV_ARG(((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dres)) & 15) == 0,
           "layernorm_bwd: pointers must be 16-byte aligned");
  return layernorm_bwd_launch(dy, x, mean, rstd, gamma, M, d, dres, accumulate, dres_bf16, dgamma, dbeta, nullptr,
                              (cudaStream_t)st);
}

extern "C" int smbv_layernorm_bwd_add(const smbv_bf16* dy, const float* x, const float* mean, const float* rstd,
                                      const float* gamma, int M, int d, float* dres, int accumulate, smbv_bf16* dres_bf16,
                                      float* dgamma, float* dbeta, const float* extra, smbv_stream_t st) {
  SMBV_ARG(dy && x && mean && rstd && gamma && dres && dgamma && dbeta, "layernorm_bwd_add: null pointer");
  SMBV_ARG(M > 0 && d > 0 && d % 8 == 0 && d <= 1024, "layernorm_bwd_add: need d %% 8 == 0 and d <= 1024 (got M=%d d=%d)", M, d);
  SMBV_ARG(((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dres) |
             reinterpret_cast<uintptr_t>(extra)) & 15) == 0,
           "layernorm_bwd_add: pointers must be 16-byte aligned");
  return layernorm_bwd_launch(dy, x, mean, rstd, gamma, M, d, dres, accumulate, dres_bf16, dgamma, dbeta, extra,
                              (cudaStream_t)st);
}

extern "C" int smbv_layernorm_bwd_blocks(void) { return 4 * num_sms(); }

extern "C" int smbv_colsum_bf16(const smbv_bf16* x, int M, int N, int64_t ld, float* out, smbv_stream_t st) {
  SMBV_ARG(x && out && M > 0 && N > 0 && N % 8 == 0 && ld >= N && ld % 8 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0,
           "colsum_bf16: need N, ld multiples of 8 and a 16-byte aligned x (M=%d N=%d ld=%lld)", M, N, (long long)ld);
  dim3 grid((N + 255) / 256, max(1, min(512, M / 32)));
  colsum_bf16_kernel<<<grid, 256, 0, (cudaStream_t)st>>>(reinterpret_cast<const __nv_bfloat16*>(x), M, N, ld, out, 0, 0, -1);
  SMBV_LAUNCH_CHECK("colsum_bf16");
  return 0;
}

extern "C" int smbv_colsum_heads_bf16(const smbv_bf16* x, int B, int H, int n, float* out, int skip_k, smbv_stream_t st) {
  SMBV_ARG(x && out && B > 0 && H > 0 && n > 0, "colsum_heads_bf16: bad args");
  dim3 grid(1, max(1, min(64, n / 32)), 3 * B * H);
  colsum_bf16_kernel<<<grid, 256, 0, (cudaStream_t)st>>>(reinterpret_cast<const __nv_bfloat16*>(x), n, 64, 64, out, B, H, skip_k ? 1 : -1);
  SMBV_LAUNCH_CHECK("colsum_heads_bf16");
  return 0;
}

extern "C" int smbv_colsum_f32(const float* x, int M, int N, int64_t ld, float* out, smbv_stream_t st) {
  SMBV_ARG(x && out && M > 0 && N > 0 && N % 4 == 0 && ld >= N && ld % 4 == 0, "colsum_f32: bad args M=%d N=%d ld=%lld", M, N, (long long)ld);
  dim3 grid((N + 127) / 128, max(1, min(256, M / 64)));
  colsum_f32_kernel<<<grid, 256, 0, (cudaStream_t)st>>>(x, M, N, ld, out);
  SMBV_LAUNCH_CHECK("colsum_f32");
  return 0;
}

extern "C" int smbv_gather_patches_bf16(const float* volume, int B, int T, int H, int W, int P, const int32_t* idx,
                                        int n_sel, int idx_stride, smbv_bf16* out, smbv_stream_t st) {
  SMBV_ARG(volume && idx && out, "gather_patches: null pointer");
  SMBV_ARG(P == 16 && T % 16 == 0 && H % 16 == 0 && W % 16 == 0 && B > 0 && n_sel > 0 && idx_stride >= n_sel, "gather_patches: bad sizes");
  SMBV_ARG(((reinterpret_cast<uintptr_t>(volume) | reinterpret_cast<uintptr_t>(out)) & 15) == 0, "gather_patches: pointers must be 16-byte aligned");
  dim3 grid(n_sel, B);
  gather_patches_kernel<<<grid, 256, 0, (cudaStream_t)st>>>(volume, T, H, W, idx, n_sel, idx_stride, reinterpret_cast<__nv_bfloat16*>(out));
  SMBV_LAUNCH_CHECK("gather_patches");
  return 0;
}
