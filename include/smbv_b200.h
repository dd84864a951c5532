/* smbv_b200 — C ABI of the B200-native (sm_100a) kernels behind smb-vision's 3D-ViT MIM hot path.
 *
 * The reference (standardmodelbio/smb-vision) has NO native/FFI boundary of its own: the path sits
 * behind two Python interfaces (SURVEY.md §8b) — the module API
 * `VideoMAEForPreTraining.forward(pixel_values, bool_masked_pos)` / `model.videomae(x)`
 * (src/models/videomae/modeling_videomae.py:753-908, :537-658) and the attention plug-in registry
 * `ALL_ATTENTION_FUNCTIONS[config._attn_implementation]` (:270-289).  This header is the C-ABI those
 * Python bindings call (ctypes; see INTEGRATION.md).  Each entry cites the reference code it replaces.
 *
 * Conventions: raw device pointers + explicit sizes, a `cudaStream_t` passed as `void*`, no allocation
 * inside, no hidden host synchronisation, thread-safe per stream.  Return 0 = ok; negative = argument
 * error detected on the host before any launch; positive = cudaError_t.  `smbv_last_error()` returns a
 * thread-local message for the last non-zero return.  bf16 = raw uint16 bits (__nv_bfloat16).
 */
#ifndef SMBV_B200_H
#define SMBV_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef void* smbv_stream_t; /* cudaStream_t */
typedef uint16_t smbv_bf16;

int smbv_version(void);              /* 100 * major + minor */
int smbv_sm_arch(void);              /* 100 : compiled for sm_100a only */
const char* smbv_last_error(void);
int smbv_device_ok(void);            /* 0 if the current device is compute capability 10.x, else -1 */

/* ---- a1 / K15: src/dataloader/mim.py:66-69 — coarse cell mask -> patch-resolution mask (np.repeat x scale on z,y,x) */
int smbv_mask_upsample(const uint8_t* coarse /*[B,cz,cy,cx]*/, uint8_t* fine /*[B,cz*s,cy*s,cx*s]*/,
                       int B, int cz, int cy, int cx, int scale, smbv_stream_t st);

/* ---- K3: replaces the boolean-mask gathers `x[~mask]`, `x[mask]` (modeling_videomae.py:134-137, :811-812, :893-894).
 * Builds, per sample, ascending index lists and the inverse map in one launch, with no host sync:
 *   vis_idx[b, i] = i-th visible token, msk_idx[b, j] = j-th masked token (both rows have stride N),
 *   slot[b, n]    = rank of token n inside its own group, counts[b] = {n_visible, n_masked}. */
int smbv_mask_index(const uint8_t* fine /*[B,N]*/, int B, int N, int32_t* vis_idx, int32_t* msk_idx, int32_t* slot,
                    int32_t* counts /*[B,2]*/, smbv_stream_t st);

/* ---- a3 / K2: get_sinusoid_encoding_table (modeling_videomae.py:95-106), computed in float64 on device then cast */
int smbv_sincos_table(float* out /*[n,d]*/, int n, int d, smbv_stream_t st);

/* ---- a5+a4 / K1+K2+K3: Conv3d(1->D, k=s=P) patch embedding (modeling_videomae.py:172-192) as an implicit GEMM: the fp32
 * volume is read once by coalesced loads, converted to bf16 on the way into shared memory, and multiplied on tcgen05 with
 * the bf16 weight (fp32 accumulate) — the operand precision of the reference's bf16-autocast Conv3d; epilogue + bias + pos[n]
 * and, when `slot`/`fine` are given, compaction of the visible rows (`emb[~mask]`, :134-137).
 * weight: bf16 [D, P^3] (the Conv3d weight viewed as a matrix, cast once by the caller).
 * out: fp32 [B, n_out, D] where n_out = N (fine == NULL) or n_visible. */
int smbv_patch_embed_fwd(const float* volume /*[B,T,H,W]*/, const smbv_bf16* weight /*[D,P^3] bf16*/, const float* bias /*[D]*/,
                         const float* pos /*[N,D] or NULL*/, const uint8_t* fine /*[B,N] or NULL*/, const int32_t* slot /*[B,N] or NULL*/,
                         int B, int T, int H, int W, int P, int D, int n_out, float* out, smbv_stream_t st);

/* ---- north-star variant ("SimMIM mask-token blending ... fused into its epilogue"): the same implicit GEMM with the epilogue
 * out[b,n,:] = (fine[b,n] ? mask_token : emb[b,n,:] + bias) + pos[n] — `torch.where(bool_masked_pos, mask_token, embeddings)` followed
 * by the position add (the only SimMIM-style blend in the reference: src/models/dinov2/modeling_dinov2.py:104-107, :113).
 * All N rows are written (no compaction).  mask_token: fp32 [D].  out: fp32 [B, N, D]. */
int smbv_patch_embed_select_fwd(const float* volume /*[B,T,H,W]*/, const smbv_bf16* weight /*[D,P^3] bf16*/, const float* bias /*[D]*/,
                                const float* pos /*[N,D] or NULL*/, const uint8_t* fine /*[B,N]*/, const float* mask_token /*[D]*/,
                                int B, int T, int H, int W, int P, int D, float* out, smbv_stream_t st);

/* ---- K4: nn.LayerNorm over the last dim (modeling_videomae.py:402-403, :412, :423; decoder.norm :676, :721).
 * x fp32 [M,d] (rows may be gathered through row_idx), y bf16 [M,d]; mean/rstd optional (saved for backward). */
int smbv_layernorm_fwd(const float* x, const float* gamma, const float* beta, float eps, int M, int d,
                       smbv_bf16* y, float* mean /*[M] or NULL*/, float* rstd /*[M] or NULL*/, smbv_stream_t st);
/* the same, and the fp32 input rows are also stored to x_copy [M,d] (or NULL): block k's input is the hidden state k of
 * `output_hidden_states` (VideoMAEModel.forward returns the input of every layer and the last output), written from the registers that
 * already hold it.  x and x_copy 16-byte aligned. */
int smbv_layernorm_fwd_copy(const float* x, const float* gamma, const float* beta, float eps, int M, int d, smbv_bf16* y,
                            float* mean /*[M] or NULL*/, float* rstd /*[M] or NULL*/, float* x_copy /*[M,d] or NULL*/,
                            smbv_stream_t st);

/* ---- K5, K7-K10, K12: nn.Linear (F.linear, modeling_videomae.py:262-264, :311, :368, :382, :801-803, :722) as a
 * tcgen05 GEMM  C[M,N] = A[M,K] * W[N,K]^T  (bf16 operands, fp32 accumulate in TMEM) with a fused epilogue. */
enum {
  SMBV_EPI_BF16 = 0,        /* out bf16 [M,ldo] = acc + bias                                                      */
  SMBV_EPI_GELU_BF16 = 1,   /* out bf16 = gelu_erf(acc + bias)                      (:368-370, hidden_act="gelu") */
  SMBV_EPI_RESID_F32 = 2,   /* out fp32 = residual + acc + bias  (residual may alias out)           (:420, :385) */
  SMBV_EPI_QKV_HEADS = 3,   /* out bf16 [3, rows/tokens, heads, tokens, 64] head-major Q,K,V        (:253-268)   */
  SMBV_EPI_F32 = 4,         /* out fp32 = acc + bias                                                              */
  SMBV_EPI_POS_GATHER_F32 = 5, /* out fp32 = acc + bias + pos[row_map[row], :]      (encoder_to_decoder + PE, :801-815) */
  SMBV_EPI_ATOMIC_F32 = 6,  /* out fp32 += acc  (weight gradients, split-K; red.global.add)                       */
  SMBV_EPI_DGELU_BF16 = 7   /* out bf16 = acc * gelu_erf'(aux)      (backward of :368-370 fused into the fc2 dgrad) */
};
typedef struct {
  const smbv_bf16* A; int64_t lda;   /* [M,K] row-major */
  const smbv_bf16* W; int64_t ldw;   /* [N,K] row-major (nn.Linear weight) */
  int32_t M, N, K;
  const float* bias;                 /* [N] or NULL */
  int32_t epilogue;
  void* out; int64_t ldo;
  const float* residual;             /* EPI_RESID_F32: [M,ldo] */
  int32_t heads, tokens;             /* EPI_QKV_HEADS: N == 3*heads*64, M == batch*tokens */
  const float* pos; int64_t ldpos;   /* EPI_POS_GATHER_F32 */
  const int32_t* row_map;            /* EPI_POS_GATHER_F32: [M] */
} smbv_gemm_args;
int smbv_gemm_bf16(const smbv_gemm_args* a, smbv_stream_t st);

/* Backward of the same nn.Linear layers (autograd of F.linear: dX = dY W, dW = dY^T X), on the same tcgen05 kernel with
 * transposed ("MN-major") operand views instead of transpose passes:
 *   C[M,N] (+)= sum_k A(m,k) * Wt(n,k)
 *   a_layout: ROWMAJOR   A is [M,K] row-major           TRANSPOSED  A is stored [K,M] row-major (A = X^T)
 *             HEADS      A is the head-major dQ/dK/dV buffer [3][.][heads][M tokens][64] of one sample, K = 3*heads*64
 *             HEADS_T    the transpose of that buffer: M = 3*heads*64, K = tokens
 *   w_layout: 0  W is [N,K] row-major                   1  W is stored [K,N] row-major
 *   split_k : 0 = choose automatically (fills the SMs for small outputs), needs SMBV_EPI_ATOMIC_F32 when > 1 */
enum { SMBV_A_ROWMAJOR = 0, SMBV_A_TRANSPOSED = 1, SMBV_A_HEADS = 2, SMBV_A_HEADS_T = 3 };
typedef struct {
  const smbv_bf16* A; int64_t lda; int32_t a_layout; int64_t a_part_stride;
  const smbv_bf16* W; int64_t ldw; int32_t w_layout;
  int32_t M, N, K, heads, split_k;
  const float* bias;                 /* [N] or NULL */
  const float* alpha;                /* optional device scalar multiplied into the accumulator */
  int32_t epilogue;                  /* BF16, GELU_BF16, F32, ATOMIC_F32, DGELU_BF16, RESID_F32 */
  void* out; int64_t ldo;
  const float* residual;             /* RESID_F32 */
  const smbv_bf16* aux;              /* DGELU_BF16: pre-activation [M,ldo] (input); GELU_BF16: optional pre-activation OUTPUT */
} smbv_gemm_ex_args;
int smbv_gemm_ex(const smbv_gemm_ex_args* a, smbv_stream_t st);

/* ---- a6+a7 / K6: non-causal multi-head attention, head_dim 64 (eager_attention_forward, modeling_videomae.py:196-223;
 * the AttentionInterface contract of :270-289).  q,k,v bf16 [BH, N, 64]; out bf16 [B, N, H*64]; lse fp32 [BH,N] or NULL
 * (natural-log sum-exp of the scaled scores, saved for backward).  Online-softmax flash tiling on tcgen05/TMEM. */
int smbv_flash_attn_fwd(const smbv_bf16* q, const smbv_bf16* k, const smbv_bf16* v, int B, int H, int N, float scale,
                        smbv_bf16* out, float* lse, smbv_stream_t st);
/* same, with an optional workspace of smbv_flash_attn_fwd_workspace_bytes(B,H,N) bytes: with it, the query-tile pairs of
 * a partial last wave are split over 2..8 CTAs by key range and merged by a combine kernel (wave-quantisation fix).
 * `variant` is reserved and must be 0; any other value is rejected with an argument error. */
int64_t smbv_flash_attn_fwd_workspace_bytes(int B, int H, int N);
int smbv_flash_attn_fwd_ex(const smbv_bf16* q, const smbv_bf16* k, const smbv_bf16* v, int B, int H, int N, float scale,
                           smbv_bf16* out, float* lse, int variant, void* workspace, int64_t workspace_bytes,
                           smbv_stream_t st);

/* ---- backward of K6 (autograd of eager_attention_forward, modeling_videomae.py:196-223).
 * q,k,v bf16 head-major [B,H,N,64]; o, dout bf16 token-major [B,N,H*64]; lse fp32 [B,H,N] from the forward.
 * Workspace: dsum_ws fp32 [B*H*N].  dq, dk, dv bf16 [B,H,N,64].  Deterministic (no atomics).  The dQ kernel runs on an
 * internal forked stream joined back to `st` by events before the call returns (no host synchronisation). */
int smbv_flash_attn_bwd(const smbv_bf16* q, const smbv_bf16* k, const smbv_bf16* v, const smbv_bf16* o,
                        const smbv_bf16* dout, const float* lse, int B, int H, int N, float scale, float* dsum_ws,
                        smbv_bf16* dq, smbv_bf16* dk, smbv_bf16* dv, smbv_stream_t st);
/* same; ev_dkdv_start / ev_dkdv_stop (cudaEvent_t or NULL) are recorded on `st` immediately before / after the dK/dV kernel
 * launch, so that a caller can time that kernel alone although dQ runs beside it on the forked stream (bench.py's roofline). */
int smbv_flash_attn_bwd_ex(const smbv_bf16* q, const smbv_bf16* k, const smbv_bf16* v, const smbv_bf16* o,
                           const smbv_bf16* dout, const float* lse, int B, int H, int N, float scale, float* dsum_ws,
                           smbv_bf16* dq, smbv_bf16* dk, smbv_bf16* dv, void* ev_dkdv_start, void* ev_dkdv_stop,
                           smbv_stream_t st);

/* Fused one-pass backward (default of the Python host side): ONE kernel computes S, dP and the exponentials once per
 * (key block, query block) pair and forms dV, dK (accumulated in tensor memory, bit-deterministic) and dQ, whose per-pair
 * partial products are summed across key blocks by fp32 bulk reductions (cp.reduce.async.bulk .add.f32) — so dQ is
 * order-dependent in its last fp32 bits (like torch's default flash / cuDNN backward); smbv_flash_attn_bwd stays the
 * deterministic mode.  The (key block, head) units of a partial last wave are cut into query ranges (one CTA each) whose fp32
 * partial dK / dV are summed in fixed order by a combine kernel.  Workspaces: dsum_ws fp32 [B*H*N]; `workspace` of
 * smbv_flash_attn_bwd_fused_workspace_bytes(B,H,N) bytes (fp32 dQ accumulator, zeroed by the call, + the partials).
 * ev_start / ev_stop (cudaEvent_t or NULL) are recorded on `st` around the fused kernel (+ combine). */
int64_t smbv_flash_attn_bwd_fused_workspace_bytes(int B, int H, int N);
int smbv_flash_attn_bwd_fused(const smbv_bf16* q, const smbv_bf16* k, const smbv_bf16* v, const smbv_bf16* o,
                              const smbv_bf16* dout, const float* lse, int B, int H, int N, float scale, float* dsum_ws,
                              void* workspace, int64_t workspace_bytes, smbv_bf16* dq, smbv_bf16* dk, smbv_bf16* dv,
                              void* ev_start, void* ev_stop, smbv_stream_t st);

/* ---- the same attention (forward + backward) for SMALL head dimensions (8, 16, 32), e.g. the reference's CPU-runnable tiny
 * config (BASELINE.json configs[0]: 64/4 and 32/2 = head_dim 16).  fp32 CUDA-core kernels, deterministic.  q, k, v (and dq,
 * dk, dv) are addressed through (batch, head, token) ELEMENT strides: the fused token-major QKV GEMM output [B,N,3,H,hd]
 * (stride_b = N*3*H*hd, stride_h = hd, stride_n = 3*H*hd) or head-major [B,H,N,hd].  out / o / dout: [B,N,H*hd]; lse and
 * dsum_ws: fp32 [B,H,N]. */
int smbv_attn_small_fwd(const smbv_bf16* q, const smbv_bf16* k, const smbv_bf16* v, int64_t stride_b, int64_t stride_h,
                        int64_t stride_n, int B, int H, int N, int head_dim, float scale, smbv_bf16* out, float* lse,
                        smbv_stream_t st);
int smbv_attn_small_bwd(const smbv_bf16* q, const smbv_bf16* k, const smbv_bf16* v, int64_t stride_b, int64_t stride_h,
                        int64_t stride_n, const smbv_bf16* o, const smbv_bf16* dout, const float* lse, int B, int H, int N,
                        int head_dim, float scale, float* dsum_ws, smbv_bf16* dq, smbv_bf16* dk, smbv_bf16* dv,
                        int64_t dstride_b, int64_t dstride_h, int64_t dstride_n, smbv_stream_t st);

/* ---- a12 / K11: rows [n_vis, N) of the decoder input = mask_token + PE[msk_idx] (modeling_videomae.py:812-815) */
int smbv_fill_mask_tokens(float* x_dec /*[B,N,d]*/, const float* mask_token /*[d]*/, const float* pos /*[N,d]*/,
                          const int32_t* msk_idx /*[B, idx_stride]*/, int B, int N, int n_vis, int d, int idx_stride,
                          smbv_stream_t st);

/* ---- a14+a15 / K13+K14: label patchify + per-patch normalise (unbiased var, +1e-6 outside sqrt) + masked mean loss
 * (modeling_videomae.py:822-897) fused with its gradient.  One CTA per masked patch reads its P^3 voxels once.
 *   loss_kind 0 = MSE (reference), 1 = L1 (north-star variant).  logits bf16 [B,n_mask,P^3];
 *   dlogits (nullable) = dloss/dlogits for dloss = 1; partial fp32 [B*n_mask] workspace; loss_out fp32 [1]. */
int smbv_normpix_loss(const float* volume /*[B,T,H,W]*/, int B, int T, int H, int W, int P,
                      const int32_t* msk_idx /*[B, idx_stride]*/, int n_mask, int idx_stride,
                      const smbv_bf16* logits, smbv_bf16* dlogits, float* partial, float* loss_out, int loss_kind,
                      smbv_stream_t st);

/* ---- backward of K4 (nn.LayerNorm autograd): dres (+)= dLN/dx, optional bf16 copy of the updated dres, dgamma += , dbeta +=.
 * workspace: fp32 [smbv_layernorm_bwd_blocks() * 2 * d].  mean/rstd are the statistics smbv_layernorm_fwd saved. */
int smbv_layernorm_bwd(const smbv_bf16* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                       int M, int d, float* dres, int accumulate, smbv_bf16* dres_bf16 /*or NULL*/, float* dgamma,
                       float* dbeta, float* workspace, smbv_stream_t st);
int smbv_layernorm_bwd_blocks(void);
/* the same with a second fp32 addend: dres = (accumulate ? dres : 0) + dLN/dx + extra, bf16 copy of that sum.  `extra` [M,d]
 * (or NULL) is the gradient of the hidden state that enters this LayerNorm (`output_hidden_states`); no
 * workspace. */
int smbv_layernorm_bwd_add(const smbv_bf16* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                           int M, int d, float* dres, int accumulate, smbv_bf16* dres_bf16 /*or NULL*/, float* dgamma,
                           float* dbeta, const float* extra /*[M,d] or NULL*/, smbv_stream_t st);

/* ---- bias / mask-token gradients: out[n] += sum_m x[m,n]  (x row-major with leading dimension ld) */
int smbv_colsum_bf16(const smbv_bf16* x, int M, int N, int64_t ld, float* out, smbv_stream_t st);
int smbv_colsum_f32(const float* x, int M, int N, int64_t ld, float* out, smbv_stream_t st);
/* q_bias / v_bias gradients from the head-major dQ/dK/dV buffer [3,B,H,n,64]: out[3*H*64] += sum over b, n.
 * skip_k != 0 leaves the middle third (the K part: k_bias is a constant zero, reference :261) untouched. */
int smbv_colsum_heads_bf16(const smbv_bf16* x, int B, int H, int n, float* out, int skip_k, smbv_stream_t st);

/* ---- patch-embedding weight gradient operand: out[b*n_sel + i, :] = bf16(P^3 voxels of patch idx[b,i])
 * (the im2col rows of the visible tokens only; reference Conv3d autograd, modeling_videomae.py:172-192) */
int smbv_gather_patches_bf16(const float* volume, int B, int T, int H, int W, int P, const int32_t* idx /*[B,idx_stride]*/,
                             int n_sel, int idx_stride, smbv_bf16* out /*[B*n_sel, P^3]*/, smbv_stream_t st);

/* ---- SURVEY.md §8f rank 1: classification head of VideoMAEForVideoClassification (modeling_videomae.py:917-1023):
 *   h = fc_norm(pooled * inv_n)  (nn.LayerNorm eps; gamma == NULL: no norm, the use_mean_pooling=False branch :976-977)
 *   logits = [h, feats] W^T + bias          (torch.cat with `additional_features`, :979-989)
 *   loss (:995-1012): REGRESSION  = MSE (mean over B*L; labels fp32 [B,L]),
 *                     SINGLE_LABEL = cross entropy (mean over B; labels int64 [B]),
 *                     MULTI_LABEL  = BCE with logits (mean over B*L; labels fp32 [B,L]),  NONE = logits only.
 * `pooled` fp32 [B,d] is the token SUM of the encoder output (smbv_colsum_f32 per sample) with inv_n = 1/N.
 * With dpooled != NULL the same launch also runs the head's backward for dloss = 1: dW [L,d+F] +=, dbias [L] +=,
 * dgamma/dbeta [d] +=, and dpooled [B,d] = dloss/d(token row) (already divided by N; identical for every token). */
enum { SMBV_CLS_NONE = 0, SMBV_CLS_REGRESSION = 1, SMBV_CLS_SINGLE_LABEL = 2, SMBV_CLS_MULTI_LABEL = 3 };
int smbv_cls_head(const float* pooled, float inv_n, const float* gamma, const float* beta, float eps, const float* feats,
                  const float* W, const float* bias, const void* labels, int B, int d, int F, int L, int problem,
                  float* logits /*[B,L]*/, float* loss /*[1]*/, float* dW, float* dbias, float* dgamma, float* dbeta,
                  float* dpooled, smbv_stream_t st);
/* out[b,:] = sum over the N token rows of x[b] (numerator of `.mean(1)`, :975); deterministic two-stage sum, no atomics.
 * workspace: fp32 [B * smbv_token_sum_chunks(N) * d]. */
int smbv_token_sum_chunks(int N);
int smbv_token_sum(const float* x /*[B,N,d]*/, int B, int N, int d, float* workspace, float* out /*[B,d]*/, smbv_stream_t st);
/* dx[b,n,:] = g[b,:] for all n (autograd of `.mean(1)`, :975) + optional bf16 copy */
int smbv_broadcast_rows(const float* g /*[B,d]*/, int B, int N, int d, float* dx /*[B,N,d]*/, smbv_bf16* dx_bf16 /*or NULL*/,
                        smbv_stream_t st);

/* ---- SURVEY.md §8f rank 2: the optimiser step HF Trainer runs after backward (src/run_mim.py:445;
 * scripts/training/run_mim.sh:17-21: AdamW lr 5e-5, weight_decay 0.01, max_grad_norm 1.0) over flat fp32 arenas that
 * share one layout (parameters, gradients, both Adam moments) + the bf16 operand copy the GEMMs read.
 *   smbv_sumsq_f32 : out[0] = sum x^2 (the squared global gradient norm of clip_grad_norm_), deterministic;
 *                    workspace fp32 [smbv_sumsq_workspace_floats()].
 *   smbv_adamw_step: torch.nn.utils.clip_grad_norm_(max_grad_norm) folded in as a scale read from the DEVICE scalar
 *                    grad_norm_sq (NULL = no clipping; no host sync), then torch.optim.AdamW semantics (decoupled decay,
 *                    bias correction with `step` 1-based), then param_bf16[i] = bf16(param[i]) (NULL = skip).
 *                    Segment k covers float4 groups [seg_start4[k], seg_start4[k+1]) (last one to n/4); seg_nodecay[k] = 1
 *                    switches weight decay off (biases and LayerNorm weights, Trainer.get_decay_parameter_names), = 2
 *                    marks a frozen segment (requires_grad=False: neither updated nor decayed, like torch.optim).
 *   smbv_scale_f32 : x[i] *= *scale_dev (device scalar; the upstream d(loss) factor of loss.backward() — gradient
 *                    accumulation, loss scaling — applied to the flat gradient arena in fp32). */
int smbv_sumsq_workspace_floats(void);
int smbv_sumsq_f32(const float* x, int64_t n, float* workspace, float* out, smbv_stream_t st);
int smbv_scale_f32(float* x, int64_t n, const float* scale_dev, smbv_stream_t st);
int smbv_adamw_step(float* param, smbv_bf16* param_bf16, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                    const int32_t* seg_start4, const uint8_t* seg_nodecay, int nseg, float lr, float beta1, float beta2,
                    float eps, float weight_decay, int step, const float* grad_norm_sq, float max_grad_norm, smbv_stream_t st);

/* ---- SURVEY.md §8f rank 2: on-device tail of the data pipeline, src/dataloader/mim.py:154-170 + PermuteImage :86-91:
 * ScaleIntensityRanged(a_min,a_max,b_min,b_max,clip) -> SpatialPadd(symmetric, 0) -> CenterSpatialCropd((H,W,T)) ->
 * permute(3,0,1,2), fused into one tiled-transpose pass.  src: resampled volume [X,Y,Z], Z contiguous, fp32 or int16 HU;
 * out: fp32 [T,H,W] (= pixel_values[b, :, 0] of the model), out[z',x',y'] <- src[x,y,z].  Bit-exact fp32 arithmetic. */
enum { SMBV_SRC_F32 = 0, SMBV_SRC_I16 = 1 };
int smbv_prepare_volume(const void* src, int src_dtype, int X, int Y, int Z, float a_min, float a_max, float b_min, float b_max,
                        int clip, int H, int W, int T, float* out /*[T,H,W]*/, smbv_stream_t st);

/* ---- SURVEY.md §8f rank 4 (first slice): V-JEPA target-encoder momentum update (src/run_vjepa.py:87-99,
 * `param_k.mul_(m).add_(param_q, alpha=1-m)` for every parameter) as one pass over two flat arenas; bit-exact fp32. */
int smbv_ema_update(float* target, const float* source, int64_t n, float momentum, float one_minus_momentum /* (float)(1.0 - m) */,
                    smbv_stream_t st);

/* ---- SURVEY.md §8f rank 4: V-JEPA2-3D rotary embedding of queries and keys (src/models/vjepa/modeling_vjepa.py:204-228
 * rotate_queries_or_keys, :297-330 get_position_ids / apply_rotary_embeddings), in place on x = bf16 [G,B,H,n,D] (e.g. the
 * Q and K sections of the head-major QKV buffer, G = 2).  Three segments of 2*((D/3)/2) elements rotate by the frame /
 * height / width index of the token id (ids int32 [B,n], or NULL = arange(n)); grid_size = crop_size / patch_size;
 * max_pos = positions tabulated in shared memory (larger ones are computed directly).  transpose bit 0 = 1 applies the
 * transposed map (the backward pass: the reference's pairing is not an orthogonal rotation, see rope.cu); bit 1 selects
 * the first-generation kernel (flat-index decode; kept as the bit-exact cross-check of the default one). */
int smbv_rope3d(smbv_bf16* x, const int32_t* ids, int G, int B, int H, int n, int D, int grid_size, int max_pos, int transpose,
                smbv_stream_t st);

/* ---- SURVEY.md §8f rank 4: `apply_masks` (src/models/vjepa/modeling_vjepa.py:543-557): out[b,k,:] = src[b, idx[b,k], :];
 * src fp32 [B,N,d], idx int32 [B,K] (values in [0,N)), out fp32 [B,K,d]; d % 4 == 0. */
int smbv_gather_rows_f32(const float* src, const int32_t* idx, int B, int N, int K, int d, float* out, smbv_stream_t st);
/* adjoint of the gather: out[b, idx[b*ldidx + k], :] = src[b,k,:] for k < K (other rows of out are left untouched: zero-fill first);
 * src fp32 [B,K,d], out fp32 [B,N,d].  Used by the SimMIM-style decoder backward (head gradient -> masked rows). */
int smbv_scatter_rows_f32(const float* src, const int32_t* idx, int B, int N, int K, int ldidx, int d, float* out, smbv_stream_t st);

/* ---- SURVEY.md §8f rank 4: head_dim 32 (the V-JEPA predictor, 384 / 12 heads; modeling_vjepa.py:629-657) on the head_dim-64 tcgen05
 * attention kernels by zero padding.  head_major = 1: [outer, H/2, n, 64] ("double heads": what the fused QKV epilogue writes with
 * heads = H/2) <-> [outer, H, n, 64] rows {head, 0..0};  head_major = 0: token-major [outer*n, H*32] <-> [outer*n, H*64].
 * expand = 1 pads, expand = 0 drops the pad.  bf16. */
int smbv_heads32_convert(const smbv_bf16* in, smbv_bf16* out, int64_t outer, int H, int n, int head_major, int expand, smbv_stream_t st);

/* ---- SURVEY.md §8f rank 4: `torch.argsort(position_masks, dim=1)` of the predictor (modeling_vjepa.py:718-720) and what
 * sort_tokens / unsort_tokens (:658-697) derive from it, as one index kernel (stable counting rank):
 * order[b, r] = index of the r-th smallest position, inv[b, i] = rank of element i (the reverse argsort), sorted[b, r] = pos[b, order[b, r]],
 * sorted2 (optional, [B, 2n]) = every sorted id twice (rotary ids of the two 32-wide heads of a 64-wide row).  All int32. */
int smbv_position_sort(const int32_t* pos /*[B,n]*/, int B, int n, int32_t* order, int32_t* inv, int32_t* sorted, int32_t* sorted2 /*or NULL*/,
                       smbv_stream_t st);

/* ---- SURVEY.md §8f rank 4: the V-JEPA loss, nn.L1Loss() (src/run_vjepa.py:108, :137): loss[0] = mean |pred - target| over n
 * fp32 elements (deterministic two-stage sum, fp64 final) and, when dpred != NULL, dpred = sign(pred - target) * upstream / n
 * in the same pass (sign(0) = 0, as torch); any n > 0 (the n % 4 trailing elements take a scalar tail).  workspace:
 * smbv_l1_workspace_floats() floats. */
int smbv_l1_workspace_floats(void);
int smbv_l1_loss_f32(const float* pred, const float* target, int64_t n, float* workspace, float* loss, float* dpred /* or NULL */,
                     float upstream, smbv_stream_t st);

/* ---- helpers on the path: fp32 -> bf16 cast of weights (autocast, SURVEY.md §8 a′ dtype notes) */
int smbv_cast_f32_bf16(const float* src, smbv_bf16* dst, int64_t n, smbv_stream_t st);
/* dst[i] = scale * float(src[i])   (gradient all-reduce wire format bf16 -> fp32 master gradients, with the 1/world mean) */
int smbv_cast_bf16_f32_scale(const smbv_bf16* src, float* dst, int64_t n, float scale, smbv_stream_t st);
/* x[i] = (*scale_dev) * x[i] + addend[i], then x_bf16[i] = bf16(x[i]); scale_dev NULL = 1, addend NULL = 0, x_bf16 NULL =
 * no copy.  n a multiple of 4.  The gradient of a hidden state (`output_hidden_states`) joins
 * the residual-stream gradient at the encoder output, and the upstream d(loss) factor is applied there. */
int smbv_scale_add_recast_f32(float* x, int64_t n, const float* scale_dev /*or NULL*/, const float* addend /*or NULL*/,
                              smbv_bf16* x_bf16 /*or NULL*/, smbv_stream_t st);

#ifdef __cplusplus
}
#endif
#endif
