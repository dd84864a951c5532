// HBM-bound kernels of the MIM path: mask upsample + index lists, sin-cos table, LayerNorm, mask-token fill,
// fused norm-pix masked loss + gradient, casts.  Coalesced 128-bit accesses, warp-shuffle reductions, grids sized
// well above 148 SMs x resident CTAs.  No tensor cores here by design (byte/row work, see DESIGN.md).
#include "common.cuh"
#include "../../include/smbv_b200.h"

namespace smbv {

// ------------------------------------------------------------------------------------------------
// mask upsample: fine[b, z, y, x] = coarse[b, z/s, y/s, x/s]            (src/dataloader/mim.py:66-69)
// ------------------------------------------------------------------------------------------------
__global__ void mask_upsample_kernel(const uint8_t* __restrict__ coarse, uint8_t* __restrict__ fine, int cz, int cy,
                                     int cx, int s, int64_t total) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int fx = cx * s, fy = cy * s, fz = cz * s;
  int x = (int)(i % fx);
  int64_t r = i / fx;
  int y = (int)(r % fy);
  r /= fy;
  int z = (int)(r % fz);
  int b = (int)(r / fz);
  fine[i] = coarse[(((int64_t)b * cz + z / s) * cy + y / s) * cx + x / s] ? 1 : 0;
}

// ------------------------------------------------------------------------------------------------
// mask index lists: one 1024-thread CTA per sample, ordered compaction by block scan (ascending n).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) mask_index_kernel(const uint8_t* __restrict__ fine, int N,
                                                         int32_t* __restrict__ vis_idx, int32_t* __restrict__ msk_idx,
                                                         int32_t* __restrict__ slot, int32_t* __restrict__ counts) {
  __shared__ int warp_tot[32];
  __shared__ int base_sh;
  const int b = blockIdx.x, t = threadIdx.x;
  const uint8_t* m = fine + (int64_t)b * N;
  const int per = (N + 1023) / 1024;
  const int lo = t * per, hi = min(N, lo + per);
  int nvis = 0;
  for (int n = lo; n < hi; ++n) nvis += (m[n] == 0);
  // inclusive scan of nvis over the block
  int v = nvis;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int u = __shfl_up_sync(0xffffffffu, v, o);
    if ((t & 31) >= o) v += u;
  }
  if ((t & 31) == 31) warp_tot[t >> 5] = v;
  __syncthreads();
  if (t < 32) {
    int w = warp_tot[t];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int u = __shfl_up_sync(0xffffffffu, w, o);
      if (t >= o) w += u;
    }
    warp_tot[t] = w;
    if (t == 31) base_sh = w;
  }
  __syncthreads();
  int vis_before = v - nvis + ((t >> 5) ? warp_tot[(t >> 5) - 1] : 0);
  int msk_before = lo < N ? lo - vis_before : 0;
  for (int n = lo; n < hi; ++n) {
    if (m[n] == 0) {
      vis_idx[(int64_t)b * N + vis_before] = n;
      slot[(int64_t)b * N + n] = vis_before++;
    } else {
      msk_idx[(int64_t)b * N + msk_before] = n;
      slot[(int64_t)b * N + n] = msk_before++;
    }
  }
  if (t == 0) {
    counts[2 * b] = base_sh;
    counts[2 * b + 1] = N - base_sh;
  }
}

// ------------------------------------------------------------------------------------------------
// sin-cos table in float64 (modeling_videomae.py:95-106)
// ------------------------------------------------------------------------------------------------
__global__ void sincos_kernel(float* __restrict__ out, int n, int d) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)n * d) return;
  int j = (int)(i % d);
  int p = (int)(i / d);
  double ang = (double)p / pow(10000.0, (double)(2 * (j / 2)) / (double)d);
  out[i] = (float)((j & 1) ? cos(ang) : sin(ang));
}

// ------------------------------------------------------------------------------------------------
// LayerNorm forward: one warp per row, the row lives in registers (NV float4 per lane), two-pass statistics.
// x_copy (or NULL): the input row is also stored there — the per-layer hidden state of `output_hidden_states`, taken from
// the registers of block k's first LayerNorm instead of a second pass over the residual stream.
// ------------------------------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(256) layernorm_fwd_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, float eps, int M, int d,
                                                            __nv_bfloat16* __restrict__ y, float* __restrict__ mean_out,
                                                            float* __restrict__ rstd_out, float* __restrict__ x_copy) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  const int lane = threadIdx.x & 31;
  const int nvec = d >> 2;
  const float4* xr = reinterpret_cast<const float4*>(x + (int64_t)row * d);
  float4 v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    int c = lane + 32 * i;
    v[i] = c < nvec ? xr[c] : make_float4(0.f, 0.f, 0.f, 0.f);
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  if (x_copy) {
    float4* xc = reinterpret_cast<float4*>(x_copy + (int64_t)row * d);
#pragma unroll
    for (int i = 0; i < NV; ++i)
      if (lane + 32 * i < nvec) xc[lane + 32 * i] = v[i];
  }
  const float mean = warp_sum(s) / (float)d;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    int c = lane + 32 * i;
    if (c < nvec) {
      float a = v[i].x - mean, b = v[i].y - mean, cc = v[i].z - mean, dd = v[i].w - mean;
      q += (a * a + b * b) + (cc * cc + dd * dd);
    }
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)d + eps);
  if (lane == 0) {
    if (mean_out) mean_out[row] = mean;
    if (rstd_out) rstd_out[row] = rstd;
  }
  const float4* g4 = reinterpret_cast<const float4*>(gamma);
  const float4* b4 = reinterpret_cast<const float4*>(beta);
  uint2* yr = reinterpret_cast<uint2*>(y + (int64_t)row * d);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    int c = lane + 32 * i;
    if (c < nvec) {
      float4 g = __ldg(g4 + c), bb = __ldg(b4 + c);
      uint2 o;
      o.x = pack_bf16((v[i].x - mean) * rstd * g.x + bb.x, (v[i].y - mean) * rstd * g.y + bb.y);
      o.y = pack_bf16((v[i].z - mean) * rstd * g.z + bb.z, (v[i].w - mean) * rstd * g.w + bb.w);
      yr[c] = o;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// decoder mask rows: x_dec[b, n_vis + j, :] = mask_token + pos[msk_idx[b, j], :]   (modeling_videomae.py:812-815)
// ------------------------------------------------------------------------------------------------
__global__ void fill_mask_tokens_kernel(float* __restrict__ x_dec, const float* __restrict__ mask_token,
                                        const float* __restrict__ pos, const int32_t* __restrict__ msk_idx, int N,
                                        int n_vis, int d4, int idx_stride, int64_t total) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int c = (int)(i % d4);
  int64_t r = i / d4;
  int n_mask = N - n_vis;
  int j = (int)(r % n_mask);
  int b = (int)(r / n_mask);
  int src = msk_idx[(int64_t)b * idx_stride + j];
  float4 p = reinterpret_cast<const float4*>(pos)[(int64_t)src * d4 + c];
  float4 m = __ldg(reinterpret_cast<const float4*>(mask_token) + c);
  reinterpret_cast<float4*>(x_dec)[((int64_t)b * N + n_vis + j) * d4 + c] =
      make_float4(p.x + m.x, p.y + m.y, p.z + m.z, p.w + m.w);
}

// ------------------------------------------------------------------------------------------------
// fused norm-pix masked loss + gradient (P = 16: 4096 voxels per patch, 256 threads x 16 voxels).
// thread t owns voxel row (dz = t/16, dy = t%16): 16 contiguous floats of the volume (two full 32 B sectors)
// and logits/dlogits elements [16t, 16t+16) (32 B, fully coalesced across the warp).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float block_sum_256(float v, float* sh) {
  v = warp_sum(v);
  __syncthreads();  // protect sh reuse
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) t += sh[i];
  return t;
}

template <int LOSS_KIND, bool WRITE_GRAD>
__global__ void __launch_bounds__(256) normpix_loss_p16_kernel(const float* __restrict__ vol, int T, int H, int W,
                                                               const int32_t* __restrict__ msk_idx, int n_mask,
                                                               int idx_stride, const __nv_bfloat16* __restrict__ logits,
                                                               __nv_bfloat16* __restrict__ dlogits,
                                                               float* __restrict__ partial, float grad_scale) {
  __shared__ float sh[8];
  const int j = blockIdx.x, b = blockIdx.y, t = threadIdx.x;
  const int n = msk_idx[(int64_t)b * idx_stride + j];
  const int gy = H >> 4, gx = W >> 4;
  const int tx = n % gx, ty = (n / gx) % gy, tz = n / (gx * gy);
  const int dz = t >> 4, dy = t & 15;
  const float* src = vol + (((int64_t)b * T + (tz * 16 + dz)) * H + (ty * 16 + dy)) * W + tx * 16;
  float x[16];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float4 v = ldg_stream_f4(src + 4 * i);
    x[4 * i] = v.x, x[4 * i + 1] = v.y, x[4 * i + 2] = v.z, x[4 * i + 3] = v.w;
  }
  // logits for this thread's 16 targets (issue before the reductions to overlap latency)
  const int64_t row = (int64_t)b * n_mask + j;
  const uint4* lp = reinterpret_cast<const uint4*>(logits + row * 4096 + t * 16);
  uint4 l0 = ldg_stream_u4(lp), l1 = ldg_stream_u4(lp + 1);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += x[i];
  const float mean = block_sum_256(s, sh) * (1.f / 4096.f);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    x[i] -= mean;
    q += x[i] * x[i];
  }
  const float var = block_sum_256(q, sh) * (1.f / 4095.f);  // UNBIASED (modeling_videomae.py:860)
  const float inv = 1.f / (sqrtf(var) + 1e-6f);             // eps outside the sqrt (:859-861)
  uint32_t lw[8] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w};
  uint32_t gw[8];
  float acc = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    __nv_bfloat162 lv = *reinterpret_cast<__nv_bfloat162*>(&lw[i]);
    float d0 = __low2float(lv) - x[2 * i] * inv;
    float d1 = __high2float(lv) - x[2 * i + 1] * inv;
    if (LOSS_KIND == 0) {
      acc += d0 * d0 + d1 * d1;
      if (WRITE_GRAD) gw[i] = pack_bf16(2.f * grad_scale * d0, 2.f * grad_scale * d1);
    } else {
      acc += fabsf(d0) + fabsf(d1);
      if (WRITE_GRAD)
        gw[i] = pack_bf16(d0 > 0.f ? grad_scale : (d0 < 0.f ? -grad_scale : 0.f),
                          d1 > 0.f ? grad_scale : (d1 < 0.f ? -grad_scale : 0.f));
    }
  }
  if (WRITE_GRAD) {
    uint4* gp = reinterpret_cast<uint4*>(dlogits + row * 4096 + t * 16);
    gp[0] = make_uint4(gw[0], gw[1], gw[2], gw[3]);
    gp[1] = make_uint4(gw[4], gw[5], gw[6], gw[7]);
  }
  const float tot = block_sum_256(acc, sh);
  if (t == 0) partial[row] = tot;
}

// Warp-per-patch variant (default for P = 16): one warp owns a whole masked patch -- 128 voxels and 128 logits per lane,
// every load of the patch issued before the first use, statistics by warp shuffles only (no block barriers), 8 patches
// per 256-thread CTA.  The block-per-patch kernel above spent its time in three __syncthreads-separated reductions.
//   lane l, load i (0..31): voxel row r = 8 i + l / 4 (dz = r / 16, dy = r % 16), floats [4 (l % 4), 4 (l % 4) + 4)
//                           -> k = 16 r + 4 (l % 4) .. : a warp-wide load covers 8 rows x 64 B (full sectors)
//   logits / dlogits: the same k, read as 8-byte pieces (4 bf16), 256 B contiguous per warp-wide access
template <int LOSS_KIND, bool WRITE_GRAD>
__global__ void __launch_bounds__(256) normpix_loss_p16_warp_kernel(const float* __restrict__ vol, int T, int H, int W,
                                                                    const int32_t* __restrict__ msk_idx, int n_mask,
                                                                    int idx_stride, const __nv_bfloat16* __restrict__ logits,
                                                                    __nv_bfloat16* __restrict__ dlogits,
                                                                    float* __restrict__ partial, float grad_scale) {
  const int lane = threadIdx.x & 31;
  const int j = blockIdx.x * 8 + (threadIdx.x >> 5), b = blockIdx.y;
  if (j >= n_mask) return;
  const int n = msk_idx[(int64_t)b * idx_stride + j];
  const int gy = H >> 4, gx = W >> 4;
  const int tx = n % gx, ty = (n / gx) % gy, tz = n / (gx * gy);
  const float* base = vol + (((int64_t)b * T + tz * 16) * H + ty * 16) * W + tx * 16 + 4 * (lane & 3);
  const int64_t row = (int64_t)b * n_mask + j;
  const __nv_bfloat16* lrow = logits + row * 4096 + 4 * (lane & 3);
  float4 x[32];
  uint2 lg[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int r = 8 * i + (lane >> 2);
    x[i] = ldg_stream_f4(base + ((int64_t)(r >> 4) * H + (r & 15)) * W);
  }
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int r = 8 * i + (lane >> 2);
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(lg[i].x), "=r"(lg[i].y) : "l"(lrow + 16 * r));
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 32; ++i) s += (x[i].x + x[i].y) + (x[i].z + x[i].w);
  const float mean = warp_sum(s) * (1.f / 4096.f);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    x[i].x -= mean, x[i].y -= mean, x[i].z -= mean, x[i].w -= mean;
    q += (x[i].x * x[i].x + x[i].y * x[i].y) + (x[i].z * x[i].z + x[i].w * x[i].w);
  }
  const float var = warp_sum(q) * (1.f / 4095.f);  // UNBIASED (modeling_videomae.py:860)
  const float inv = 1.f / (sqrtf(var) + 1e-6f);     // eps outside the sqrt (:859-861)
  __nv_bfloat16* drow = WRITE_GRAD ? dlogits + row * 4096 + 4 * (lane & 3) : nullptr;
  float acc = 0.f;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int r = 8 * i + (lane >> 2);
    const __nv_bfloat162 l01 = *reinterpret_cast<const __nv_bfloat162*>(&lg[i].x), l23 = *reinterpret_cast<const __nv_bfloat162*>(&lg[i].y);
    const float d0 = __low2float(l01) - x[i].x * inv, d1 = __high2float(l01) - x[i].y * inv;
    const float d2 = __low2float(l23) - x[i].z * inv, d3 = __high2float(l23) - x[i].w * inv;
    uint2 g;
    if (LOSS_KIND == 0) {
      acc += (d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3);
      const float gs2 = 2.f * grad_scale;
      g = make_uint2(pack_bf16(gs2 * d0, gs2 * d1), pack_bf16(gs2 * d2, gs2 * d3));
    } else {
      acc += (fabsf(d0) + fabsf(d1)) + (fabsf(d2) + fabsf(d3));
      auto sg = [&](float d) { return d > 0.f ? grad_scale : (d < 0.f ? -grad_scale : 0.f); };
      g = make_uint2(pack_bf16(sg(d0), sg(d1)), pack_bf16(sg(d2), sg(d3)));
    }
    if (WRITE_GRAD) *reinterpret_cast<uint2*>(drow + 16 * r) = g;
  }
  const float tot = warp_sum(acc);
  if (lane == 0) partial[row] = tot;
}

// deterministic final reduction of the per-patch partials (fp64), loss = sum / count
__global__ void __launch_bounds__(1024) loss_reduce_kernel(const float* __restrict__ partial, int n, double inv_count,
                                                           float* __restrict__ loss_out) {
  __shared__ double sh[32];
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += 1024) s += (double)partial[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    s = sh[threadIdx.x];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (threadIdx.x == 0) loss_out[0] = (float)(s * inv_count);
  }
}

// generic-P fallback (any patch size with P^3 <= 32768): one CTA per masked patch, three passes through L1/L2.
template <int LOSS_KIND, bool WRITE_GRAD>
__global__ void __launch_bounds__(256) normpix_loss_generic_kernel(const float* __restrict__ vol, int T, int H, int W,
                                                                   int P, const int32_t* __restrict__ msk_idx,
                                                                   int n_mask, int idx_stride,
                                                                   const __nv_bfloat16* __restrict__ logits,
                                                                   __nv_bfloat16* __restrict__ dlogits,
                                                                   float* __restrict__ partial, float grad_scale) {
  __shared__ float sh[8];
  const int j = blockIdx.x, b = blockIdx.y, t = threadIdx.x;
  const int n = msk_idx[(int64_t)b * idx_stride + j];
  const int gy = H / P, gx = W / P, K = P * P * P;
  const int tx = n % gx, ty = (n / gx) % gy, tz = n / (gx * gy);
  const float* base = vol + (((int64_t)b * T + tz * P) * H + ty * P) * W + tx * P;
  auto at = [&](int k) { return base[((int64_t)(k / (P * P)) * H + (k / P) % P) * W + k % P]; };
  float s = 0.f;
  for (int k = t; k < K; k += 256) s += at(k);
  const float mean = block_sum_256(s, sh) / (float)K;
  float q = 0.f;
  for (int k = t; k < K; k += 256) {
    float d = at(k) - mean;
    q += d * d;
  }
  const float var = block_sum_256(q, sh) / (float)(K - 1);
  const float inv = 1.f / (sqrtf(var) + 1e-6f);
  const int64_t row = (int64_t)b * n_mask + j;
  float acc = 0.f;
  for (int k = t; k < K; k += 256) {
    float d = __bfloat162float(logits[row * K + k]) - (at(k) - mean) * inv;
    float g;
    if (LOSS_KIND == 0) {
      acc += d * d;
      g = 2.f * grad_scale * d;
    } else {
      acc += fabsf(d);
      g = d > 0.f ? grad_scale : (d < 0.f ? -grad_scale : 0.f);
    }
    if (WRITE_GRAD) dlogits[row * K + k] = __float2bfloat16(g);
  }
  const float tot = block_sum_256(acc, sh);
  if (t == 0) partial[row] = tot;
}

__global__ void cast_f32_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int64_t n) {
  int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i + 3 < n) {
    float4 v = *reinterpret_cast<const float4*>(src + i);
    uint2 o;
    o.x = pack_bf16(v.x, v.y);
    o.y = pack_bf16(v.z, v.w);
    *reinterpret_cast<uint2*>(dst + i) = o;
  } else {
    for (; i < n; ++i) dst[i] = __float2bfloat16(src[i]);
  }
}

__global__ void cast_bf16_f32_scale_kernel(const __nv_bfloat16* __restrict__ src, float* __restrict__ dst, int64_t n, float scale) {
  int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i + 3 < n) {
    const uint2 v = *reinterpret_cast<const uint2*>(src + i);
    const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&v.x), b = *reinterpret_cast<const __nv_bfloat162*>(&v.y);
    *reinterpret_cast<float4*>(dst + i) = make_float4(scale * __low2float(a), scale * __high2float(a), scale * __low2float(b), scale * __high2float(b));
  } else {
    for (; i < n; ++i) dst[i] = scale * __bfloat162float(src[i]);
  }
}

// x = scale * x + addend, then the bf16 copy of the result (every part optional).  Joins the gradient of a returned hidden
// state to the residual-stream gradient at a boundary that has no LayerNorm backward pass, and applies the upstream
// d(loss) factor there (device scalar: no host synchronisation).
__global__ void scale_add_recast_kernel(float* __restrict__ x, int64_t n4, const float* __restrict__ scale,
                                        const float* __restrict__ addend, __nv_bfloat16* __restrict__ x_bf16) {
  const float sc = scale ? *scale : 1.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 v = reinterpret_cast<const float4*>(x)[i];
    if (scale) v = make_float4(sc * v.x, sc * v.y, sc * v.z, sc * v.w);
    if (addend) {
      const float4 a = reinterpret_cast<const float4*>(addend)[i];
      v = make_float4(v.x + a.x, v.y + a.y, v.z + a.z, v.w + a.w);
    }
    reinterpret_cast<float4*>(x)[i] = v;
    if (x_bf16) reinterpret_cast<uint2*>(x_bf16)[i] = make_uint2(pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
  }
}

}  // namespace smbv

using namespace smbv;

extern "C" int smbv_mask_upsample(const uint8_t* coarse, uint8_t* fine, int B, int cz, int cy, int cx, int scale,
                                  smbv_stream_t st) {
  SMBV_ARG(coarse && fine, "mask_upsample: null pointer");
  SMBV_ARG(B > 0 && cz > 0 && cy > 0 && cx > 0 && scale > 0, "mask_upsample: bad sizes B=%d grid=%dx%dx%d scale=%d", B,
           cz, cy, cx, scale);
  int64_t total = (int64_t)B * cz * cy * cx * scale * scale * scale;
  mask_upsample_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)st>>>(coarse, fine, cz, cy, cx, scale,
                                                                                      total);
  SMBV_LAUNCH_CHECK("mask_upsample");
  return 0;
}

extern "C" int smbv_mask_index(const uint8_t* fine, int B, int N, int32_t* vis_idx, int32_t* msk_idx, int32_t* slot,
                               int32_t* counts, smbv_stream_t st) {
  SMBV_ARG(fine && vis_idx && msk_idx && slot && counts, "mask_index: null pointer");
  SMBV_ARG(B > 0 && N > 0, "mask_index: bad sizes B=%d N=%d", B, N);
  mask_index_kernel<<<B, 1024, 0, (cudaStream_t)st>>>(fine, N, vis_idx, msk_idx, slot, counts);
  SMBV_LAUNCH_CHECK("mask_index");
  return 0;
}

extern "C" int smbv_sincos_table(float* out, int n, int d, smbv_stream_t st) {
  SMBV_ARG(out && n > 0 && d > 0, "sincos_table: bad args");
  int64_t total = (int64_t)n * d;
  sincos_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)st>>>(out, n, d);
  SMBV_LAUNCH_CHECK("sincos_table");
  return 0;
}

static int layernorm_fwd_launch(const float* x, const float* gamma, const float* beta, float eps, int M, int d, smbv_bf16* y,
                                float* mean, float* rstd, float* x_copy, cudaStream_t s) {
  const int nv = (d / 4 + 31) / 32;
  dim3 grid((M + 7) / 8), block(256);
  __nv_bfloat16* yy = reinterpret_cast<__nv_bfloat16*>(y);
#define LN_CASE(NV)                                                                                         \
  case NV:                                                                                                  \
    layernorm_fwd_kernel<NV><<<grid, block, 0, s>>>(x, gamma, beta, eps, M, d, yy, mean, rstd, x_copy);     \
    break;
  switch (nv <= 1 ? 1 : nv <= 2 ? 2 : nv <= 3 ? 3 : nv <= 4 ? 4 : nv <= 6 ? 6 : nv <= 8 ? 8 : nv <= 16 ? 16 : 32) {
    LN_CASE(1) LN_CASE(2) LN_CASE(3) LN_CASE(4) LN_CASE(6) LN_CASE(8) LN_CASE(16) LN_CASE(32)
  }
#undef LN_CASE
  SMBV_LAUNCH_CHECK("layernorm_fwd");
  return 0;
}

extern "C" int smbv_layernorm_fwd(const float* x, const float* gamma, const float* beta, float eps, int M, int d,
                                  smbv_bf16* y, float* mean, float* rstd, smbv_stream_t st) {
  SMBV_ARG(x && gamma && beta && y, "layernorm_fwd: null pointer");
  SMBV_ARG(M > 0 && d > 0 && d % 4 == 0 && d <= 4096, "layernorm_fwd: need d %% 4 == 0 and d <= 4096 (got M=%d d=%d)", M, d);
  return layernorm_fwd_launch(x, gamma, beta, eps, M, d, y, mean, rstd, nullptr, (cudaStream_t)st);
}

extern "C" int smbv_layernorm_fwd_copy(const float* x, const float* gamma, const float* beta, float eps, int M, int d,
                                       smbv_bf16* y, float* mean, float* rstd, float* x_copy, smbv_stream_t st) {
  SMBV_ARG(x && gamma && beta && y, "layernorm_fwd_copy: null pointer");
  SMBV_ARG(M > 0 && d > 0 && d % 4 == 0 && d <= 4096, "layernorm_fwd_copy: need d %% 4 == 0 and d <= 4096 (got M=%d d=%d)", M, d);
  SMBV_ARG(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(x_copy)) & 15) == 0,
           "layernorm_fwd_copy: x and x_copy must be 16-byte aligned");
  return layernorm_fwd_launch(x, gamma, beta, eps, M, d, y, mean, rstd, x_copy, (cudaStream_t)st);
}

extern "C" int smbv_fill_mask_tokens(float* x_dec, const float* mask_token, const float* pos, const int32_t* msk_idx,
                                     int B, int N, int n_vis, int d, int idx_stride, smbv_stream_t st) {
  SMBV_ARG(x_dec && mask_token && pos && msk_idx, "fill_mask_tokens: null pointer");
  SMBV_ARG(B > 0 && N > 0 && n_vis >= 0 && n_vis <= N && d > 0 && d % 4 == 0, "fill_mask_tokens: bad sizes");
  int64_t total = (int64_t)B * (N - n_vis) * (d / 4);
  if (total == 0) return 0;
  fill_mask_tokens_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)st>>>(x_dec, mask_token, pos, msk_idx,
                                                                                         N, n_vis, d / 4, idx_stride, total);
  SMBV_LAUNCH_CHECK("fill_mask_tokens");
  return 0;
}

extern "C" int smbv_normpix_loss(const float* volume, int B, int T, int H, int W, int P, const int32_t* msk_idx,
                                 int n_mask, int idx_stride, const smbv_bf16* logits, smbv_bf16* dlogits, float* partial,
                                 float* loss_out, int loss_kind, smbv_stream_t st) {
  SMBV_ARG(volume && msk_idx && logits && partial && loss_out, "normpix_loss: null pointer");
  SMBV_ARG(B > 0 && P > 0 && T % P == 0 && H % P == 0 && W % P == 0, "normpix_loss: volume %dx%dx%d not divisible by patch %d", T, H, W, P);
  SMBV_ARG(n_mask > 0 && idx_stride >= n_mask, "normpix_loss: bad n_mask=%d idx_stride=%d", n_mask, idx_stride);
  SMBV_ARG(loss_kind == 0 || loss_kind == 1 || loss_kind == 16 || loss_kind == 17, "normpix_loss: loss_kind must be 0 (mse) or 1 (l1)");
  const bool force_block = loss_kind >= 16;  // 16/17: the block-per-patch kernel (kept for A/B measurements)
  loss_kind &= 1;
  SMBV_ARG((int64_t)P * P * P <= 32768 && P * P * P > 1, "normpix_loss: unsupported patch size %d", P);
  cudaStream_t s = (cudaStream_t)st;
  const double count = (double)B * n_mask * P * P * P;
  const float gs = (float)(1.0 / count);
  const __nv_bfloat16* lg = reinterpret_cast<const __nv_bfloat16*>(logits);
  __nv_bfloat16* dl = reinterpret_cast<__nv_bfloat16*>(dlogits);
  dim3 grid(n_mask, B);
  const bool fast = (P == 16) && (W % 4 == 0) && ((reinterpret_cast<uintptr_t>(volume) & 15) == 0) &&
                    ((reinterpret_cast<uintptr_t>(logits) & 15) == 0) && ((reinterpret_cast<uintptr_t>(dlogits) & 15) == 0);
#define LOSS_LAUNCH(KERNEL, ...)                                                                         \
  if (loss_kind == 0) {                                                                                  \
    if (dl) KERNEL<0, true><<<grid, 256, 0, s>>>(__VA_ARGS__);                                           \
    else KERNEL<0, false><<<grid, 256, 0, s>>>(__VA_ARGS__);                                             \
  } else {                                                                                               \
    if (dl) KERNEL<1, true><<<grid, 256, 0, s>>>(__VA_ARGS__);                                           \
    else KERNEL<1, false><<<grid, 256, 0, s>>>(__VA_ARGS__);                                             \
  }
  if (fast && force_block) {
    LOSS_LAUNCH(normpix_loss_p16_kernel, volume, T, H, W, msk_idx, n_mask, idx_stride, lg, dl, partial, gs)
  } else if (fast) {
    grid = dim3((n_mask + 7) / 8, B);
    LOSS_LAUNCH(normpix_loss_p16_warp_kernel, volume, T, H, W, msk_idx, n_mask, idx_stride, lg, dl, partial, gs)
  } else {
    LOSS_LAUNCH(normpix_loss_generic_kernel, volume, T, H, W, P, msk_idx, n_mask, idx_stride, lg, dl, partial, gs)
  }
#undef LOSS_LAUNCH
  SMBV_LAUNCH_CHECK("normpix_loss");
  loss_reduce_kernel<<<1, 1024, 0, s>>>(partial, B * n_mask, 1.0 / count, loss_out);
  SMBV_LAUNCH_CHECK("loss_reduce");
  return 0;
}

extern "C" int smbv_cast_f32_bf16(const float* src, smbv_bf16* dst, int64_t n, smbv_stream_t st) {
  SMBV_ARG(src && dst && n >= 0, "cast_f32_bf16: bad args");
  if (n == 0) return 0;
  SMBV_ARG((reinterpret_cast<uintptr_t>(src) & 15) == 0 && (reinterpret_cast<uintptr_t>(dst) & 7) == 0,
           "cast_f32_bf16: pointers must be 16/8-byte aligned");
  int64_t nthreads = (n + 3) / 4;
  cast_f32_bf16_kernel<<<(unsigned)((nthreads + 255) / 256), 256, 0, (cudaStream_t)st>>>(
      src, reinterpret_cast<__nv_bfloat16*>(dst), n);
  SMBV_LAUNCH_CHECK("cast_f32_bf16");
  return 0;
}

extern "C" int smbv_cast_bf16_f32_scale(const smbv_bf16* src, float* dst, int64_t n, float scale, smbv_stream_t st) {
  SMBV_ARG(src && dst && n >= 0, "cast_bf16_f32_scale: bad args");
  if (n == 0) return 0;
  SMBV_ARG((reinterpret_cast<uintptr_t>(src) & 7) == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0,
           "cast_bf16_f32_scale: pointers must be 8/16-byte aligned");
  int64_t nthreads = (n + 3) / 4;
  cast_bf16_f32_scale_kernel<<<(unsigned)((nthreads + 255) / 256), 256, 0, (cudaStream_t)st>>>(
      reinterpret_cast<const __nv_bfloat16*>(src), dst, n, scale);
  SMBV_LAUNCH_CHECK("cast_bf16_f32_scale");
  return 0;
}

extern "C" int smbv_scale_add_recast_f32(float* x, int64_t n, const float* scale_dev, const float* addend, smbv_bf16* x_bf16,
                                         smbv_stream_t st) {
  SMBV_ARG(x, "scale_add_recast_f32: null pointer");
  SMBV_ARG(n > 0 && n % 4 == 0, "scale_add_recast_f32: n=%lld must be a positive multiple of 4", (long long)n);
  SMBV_ARG(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(addend)) & 15) == 0 &&
               (reinterpret_cast<uintptr_t>(x_bf16) & 7) == 0,
           "scale_add_recast_f32: x and addend must be 16-byte aligned, x_bf16 8-byte aligned");
  const int64_t n4 = n / 4, want = (n4 + 255) / 256, cap = (int64_t)num_sms() * 8;
  scale_add_recast_kernel<<<(unsigned)(want < cap ? want : cap), 256, 0, (cudaStream_t)st>>>(
      x, n4, scale_dev, addend, reinterpret_cast<__nv_bfloat16*>(x_bf16));
  SMBV_LAUNCH_CHECK("scale_add_recast_f32");
  return 0;
}
