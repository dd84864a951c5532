"""Tensor-level wrappers over the C-ABI (``include/smbv_b200.h``).

PyTorch is used only for device memory and streams: every wrapper checks dtype/device/contiguity, allocates
the outputs, and hands raw pointers plus the current CUDA stream to the library.  There is no fallback: a CPU
tensor or a missing library raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

from . import _lib
from ._lib import (A_HEADS, A_HEADS_T, A_ROWMAJOR, A_TRANSPOSED, CLS_MULTI_LABEL, CLS_NONE, CLS_REGRESSION, CLS_SINGLE_LABEL, EPI_ATOMIC_F32, EPI_BF16, EPI_DGELU_BF16, EPI_F32,
                   EPI_GELU_BF16, EPI_POS_GATHER_F32, EPI_QKV_HEADS, EPI_RESID_F32, GemmArgs, GemmExArgs, SmbvError, call)


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _chk(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise SmbvError(f"{name}: expected a CUDA tensor (smb_vision_b200 has no CPU path)")
    if t.dtype != dtype:
        raise SmbvError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise SmbvError(f"{name}: expected a contiguous tensor")
    return t


def _ptr(t) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


def mask_upsample(coarse: torch.Tensor, scale: int) -> torch.Tensor:
    """uint8 [B,cz,cy,cx] -> uint8 [B, N] at patch resolution (src/dataloader/mim.py:66-69)."""
    _chk(coarse, torch.uint8, "coarse")
    B, cz, cy, cx = coarse.shape
    fine = torch.empty((B, cz * scale * cy * scale * cx * scale), dtype=torch.uint8, device=coarse.device)
    call("smbv_mask_upsample", _ptr(coarse), _ptr(fine), B, cz, cy, cx, scale, _stream())
    return fine


def mask_index(fine: torch.Tensor):
    """uint8 [B,N] -> (vis_idx, msk_idx, slot, counts), all int32; no host synchronisation."""
    _chk(fine, torch.uint8, "fine")
    B, N = fine.shape
    dev = fine.device
    vis = torch.empty((B, N), dtype=torch.int32, device=dev)
    msk = torch.empty((B, N), dtype=torch.int32, device=dev)
    slot = torch.empty((B, N), dtype=torch.int32, device=dev)
    counts = torch.empty((B, 2), dtype=torch.int32, device=dev)
    call("smbv_mask_index", _ptr(fine), B, N, _ptr(vis), _ptr(msk), _ptr(slot), _ptr(counts), _stream())
    return vis, msk, slot, counts


def sincos_table(n: int, d: int, device) -> torch.Tensor:
    out = torch.empty((n, d), dtype=torch.float32, device=device)
    call("smbv_sincos_table", _ptr(out), n, d, _stream())
    return out


def _w16(weight: torch.Tensor) -> torch.Tensor:
    """the patch-embedding weight as the kernel reads it: bf16 [D, 4096], contiguous."""
    if isinstance(weight, torch.Tensor) and weight.dtype == torch.float32:
        weight = cast_bf16(_chk(weight, torch.float32, "weight"))
    return _chk(weight, torch.bfloat16, "weight")


def patch_embed_fwd(volume, weight, bias, pos, fine=None, slot=None, n_out=None) -> torch.Tensor:
    """volume fp32 [B,T,H,W]; weight bf16 [D,4096] (an fp32 weight is cast here: callers on a hot path pass the cached bf16
    copy); returns fp32 [B, n_out, D]."""
    _chk(volume, torch.float32, "volume")
    weight = _w16(weight)
    _chk(bias, torch.float32, "bias")
    if pos is not None:  # None: no position table (V-JEPA: positions enter through RoPE)
        _chk(pos, torch.float32, "pos")
    B, T, H, W = volume.shape
    D = weight.shape[0]
    N = (T // 16) * (H // 16) * (W // 16)
    if fine is not None:
        _chk(fine, torch.uint8, "fine")
        _chk(slot, torch.int32, "slot")
        if n_out is None:
            raise SmbvError("patch_embed_fwd: n_out (visible tokens per sample) is required with a mask")
    else:
        n_out = N
    out = torch.empty((B, n_out, D), dtype=torch.float32, device=volume.device)
    call("smbv_patch_embed_fwd", _ptr(volume), _ptr(weight), _ptr(bias), _ptr(pos), _ptr(fine), _ptr(slot),
         B, T, H, W, 16, D, n_out, _ptr(out), _stream())
    return out


def patch_embed_select_fwd(volume, weight, bias, pos, fine, mask_token) -> torch.Tensor:
    """SimMIM-style blend in the patch-embed epilogue: out[b,n] = (fine[b,n] ? mask_token : emb[b,n] + bias) + pos[n]; fp32 [B,N,D]."""
    for t, nme in ((volume, "volume"), (bias, "bias"), (mask_token, "mask_token")):
        _chk(t, torch.float32, nme)
    weight = _w16(weight)
    if pos is not None:
        _chk(pos, torch.float32, "pos")
    _chk(fine, torch.uint8, "fine")
    B, T, H, W = volume.shape
    D = weight.shape[0]
    N = (T // 16) * (H // 16) * (W // 16)
    if tuple(fine.shape) != (B, N) or mask_token.numel() != D:
        raise SmbvError(f"patch_embed_select_fwd: fine must be [{B},{N}] and mask_token [{D}]")
    out = torch.empty((B, N, D), dtype=torch.float32, device=volume.device)
    call("smbv_patch_embed_select_fwd", _ptr(volume), _ptr(weight), _ptr(bias), _ptr(pos), _ptr(fine), _ptr(mask_token),
         B, T, H, W, 16, D, _ptr(out), _stream())
    return out


def layernorm_fwd(x, gamma, beta, eps: float, save_stats: bool = False, out=None, x_copy=None):
    """x fp32 [..., d] -> bf16 [..., d] (+ mean, rstd fp32 [M] when save_stats).  x_copy: fp32 like x, receives a copy of x
    (written from the registers the LayerNorm reads x into)."""
    _chk(x, torch.float32, "x")
    _chk(gamma, torch.float32, "gamma")
    _chk(beta, torch.float32, "beta")
    d = x.shape[-1]
    M = x.numel() // d
    y = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device) if out is None else _chk(out, torch.bfloat16, "out")
    mean = rstd = None
    if save_stats:
        mean = torch.empty((M,), dtype=torch.float32, device=x.device)
        rstd = torch.empty((M,), dtype=torch.float32, device=x.device)
    if x_copy is None:
        call("smbv_layernorm_fwd", _ptr(x), _ptr(gamma), _ptr(beta), float(eps), M, d, _ptr(y), _ptr(mean), _ptr(rstd), _stream())
    else:
        if _chk(x_copy, torch.float32, "x_copy").shape != x.shape:
            raise SmbvError(f"layernorm_fwd: x_copy must be shaped like x {tuple(x.shape)}")
        call("smbv_layernorm_fwd_copy", _ptr(x), _ptr(gamma), _ptr(beta), float(eps), M, d, _ptr(y), _ptr(mean), _ptr(rstd),
             _ptr(x_copy), _stream())
    return (y, mean, rstd) if save_stats else y


def gemm(a, w, bias=None, epilogue=EPI_BF16, out=None, residual=None, heads=0, tokens=0, pos=None, row_map=None):
    """C = a[M,K] @ w[N,K]^T with a fused epilogue; a, w bf16.  Returns the output tensor."""
    _chk(a, torch.bfloat16, "a")
    _chk(w, torch.bfloat16, "w")
    K = a.shape[-1]
    M = a.numel() // K
    N = w.shape[0]
    if w.shape[1] != K:
        raise SmbvError(f"gemm: K mismatch a[..,{K}] vs w[{N},{w.shape[1]}]")
    if bias is not None:
        _chk(bias, torch.float32, "bias")
    dev = a.device
    if out is None:
        if epilogue in (EPI_BF16, EPI_GELU_BF16):
            out = torch.empty((*a.shape[:-1], N), dtype=torch.bfloat16, device=dev)
        elif epilogue == EPI_QKV_HEADS:
            out = torch.empty((3, M // tokens, heads, tokens, 64), dtype=torch.bfloat16, device=dev)
        elif epilogue == EPI_RESID_F32:
            out = residual  # in place on the residual stream
        else:
            out = torch.empty((*a.shape[:-1], N), dtype=torch.float32, device=dev)
    g = GemmArgs()
    g.A, g.lda, g.W, g.ldw = a.data_ptr(), K, w.data_ptr(), K
    g.M, g.N, g.K = M, N, K
    g.bias = 0 if bias is None else bias.data_ptr()
    g.epilogue = epilogue
    g.out, g.ldo = out.data_ptr(), N
    g.residual = 0
    if epilogue == EPI_RESID_F32:
        _chk(residual, torch.float32, "residual")
        _chk(out, torch.float32, "out")
        g.residual = residual.data_ptr()
    g.heads, g.tokens = heads, tokens
    g.pos, g.ldpos, g.row_map = 0, 0, 0
    if epilogue == EPI_POS_GATHER_F32:
        _chk(pos, torch.float32, "pos")
        _chk(row_map, torch.int32, "row_map")
        g.pos, g.ldpos, g.row_map = pos.data_ptr(), pos.shape[-1], row_map.data_ptr()
    call("smbv_gemm_bf16", C.byref(g), _stream())
    return out


def flash_attn_fwd(q, k, v, scale: float, return_lse: bool = False):
    """q,k,v bf16 [B,H,N,64] -> out bf16 [B,N,H*64]."""
    _chk(q, torch.bfloat16, "q")
    _chk(k, torch.bfloat16, "k")
    _chk(v, torch.bfloat16, "v")
    B, H, N, D = q.shape
    if D != 64:
        raise SmbvError(f"flash_attn_fwd: head_dim {D} not supported (64 only)")
    out = torch.empty((B, N, H * 64), dtype=torch.bfloat16, device=q.device)
    lse = torch.empty((B, H, N), dtype=torch.float32, device=q.device) if return_lse else None
    wsb = int(_lib.load().smbv_flash_attn_fwd_workspace_bytes(B, H, N))
    ws = torch.empty((wsb,), dtype=torch.uint8, device=q.device) if wsb else None
    call("smbv_flash_attn_fwd_ex", _ptr(q), _ptr(k), _ptr(v), B, H, N, float(scale), _ptr(out), _ptr(lse),
         0, _ptr(ws), wsb, _stream())
    return (out, lse) if return_lse else out


def fill_mask_tokens(x_dec, mask_token, pos, msk_idx, n_vis: int) -> None:
    _chk(x_dec, torch.float32, "x_dec")
    _chk(mask_token, torch.float32, "mask_token")
    _chk(pos, torch.float32, "pos")
    _chk(msk_idx, torch.int32, "msk_idx")
    B, N, d = x_dec.shape
    call("smbv_fill_mask_tokens", _ptr(x_dec), _ptr(mask_token), _ptr(pos), _ptr(msk_idx), B, N, n_vis, d,
         msk_idx.shape[1], _stream())


def normpix_loss(volume, msk_idx, n_mask: int, logits, want_grad: bool, loss_kind: int = 0, patch: int = 16):
    """volume fp32 [B,T,H,W]; logits bf16 [B,n_mask,P^3] -> (loss fp32 [], dlogits bf16 or None)."""
    _chk(volume, torch.float32, "volume")
    _chk(msk_idx, torch.int32, "msk_idx")
    _chk(logits, torch.bfloat16, "logits")
    B, T, H, W = volume.shape
    dl = torch.empty_like(logits) if want_grad else None
    partial = torch.empty((B * n_mask,), dtype=torch.float32, device=volume.device)
    loss = torch.empty((1,), dtype=torch.float32, device=volume.device)
    call("smbv_normpix_loss", _ptr(volume), B, T, H, W, patch, _ptr(msk_idx), n_mask, msk_idx.shape[1], _ptr(logits),
         _ptr(dl), _ptr(partial), _ptr(loss), loss_kind, _stream())
    return loss[0], dl


def cast_bf16(src: torch.Tensor, out=None) -> torch.Tensor:
    _chk(src, torch.float32, "src")
    dst = torch.empty(src.shape, dtype=torch.bfloat16, device=src.device) if out is None else _chk(out, torch.bfloat16, "out")
    call("smbv_cast_f32_bf16", _ptr(src), _ptr(dst), src.numel(), _stream())
    return dst


# ----------------------------------------------------------------------------------------------
# backward
# ----------------------------------------------------------------------------------------------
def gemm_ex(A, W, M, N, K, epilogue, out, a_layout=A_ROWMAJOR, w_layout=0, lda=None, ldw=None, heads=0, a_part_stride=0,
            split_k=0, bias=None, alpha=None, residual=None, aux=None, ldo=None):
    """out[M,N] (+)= sum_k A(m,k) W(n,k) with transposed / head-major operand views (see include/smbv_b200.h)."""
    _chk(A, torch.bfloat16, "A")
    _chk(W, torch.bfloat16, "W")
    g = GemmExArgs()
    g.A, g.a_layout, g.a_part_stride = A.data_ptr(), a_layout, a_part_stride
    g.lda = lda if lda is not None else (K if a_layout == A_ROWMAJOR else M)
    g.W, g.w_layout = W.data_ptr(), w_layout
    g.ldw = ldw if ldw is not None else (K if w_layout == 0 else N)
    g.M, g.N, g.K, g.heads, g.split_k = M, N, K, heads, split_k
    g.bias = 0 if bias is None else _chk(bias, torch.float32, "bias").data_ptr()
    g.alpha = 0 if alpha is None else _chk(alpha, torch.float32, "alpha").data_ptr()
    g.epilogue = epilogue
    g.out, g.ldo = out.data_ptr(), (ldo if ldo is not None else N)
    g.residual = 0 if residual is None else residual.data_ptr()
    g.aux = 0 if aux is None else _chk(aux, torch.bfloat16, "aux").data_ptr()
    call("smbv_gemm_ex", C.byref(g), _stream())
    return out


def linear_dgrad(dy, w, out_dtype=torch.bfloat16, aux=None, out=None):
    """dX[M,K] = dY[M,N] @ W[N,K]  (W is the nn.Linear weight, bf16 [N,K]); aux -> multiply by gelu'(aux)."""
    N, K = w.shape
    M = dy.numel() // N
    if out is None:
        out = torch.empty((*dy.shape[:-1], K), dtype=out_dtype, device=dy.device)
    epi = EPI_DGELU_BF16 if aux is not None else (EPI_BF16 if out.dtype == torch.bfloat16 else EPI_F32)
    return gemm_ex(dy, w, M, K, N, epi, out, a_layout=A_ROWMAJOR, w_layout=1, lda=N, ldw=K, aux=aux)


def linear_wgrad(dy, x, dw):
    """dW[N,K] += dY[M,N]^T @ X[M,K]  (fp32 accumulate into dw, split-K atomics)."""
    N, K = dw.shape
    M = dy.numel() // N
    _chk(dw, torch.float32, "dw")
    return gemm_ex(dy, x, N, K, M, EPI_ATOMIC_F32, dw, a_layout=A_TRANSPOSED, w_layout=1, lda=N, ldw=K)


def qkv_dgrad(dqkv, w, tokens, heads, batch_index=0, batch=1, out=None):
    """dH[tokens, d] = dQKV (head-major [3,B,H,tokens,64], sample `batch_index`) @ Wqkv[3d, d]."""
    N3, d = w.shape
    if out is None:
        out = torch.empty((tokens, d), dtype=torch.bfloat16, device=w.device)
    A = dqkv[0, batch_index]
    return gemm_ex(A, w, tokens, d, N3, EPI_BF16, out, a_layout=A_HEADS, w_layout=1, ldw=d, heads=heads,
                   a_part_stride=batch * heads * tokens * 64)


def qkv_wgrad(dqkv, x, dw, tokens, heads, batch_index=0, batch=1):
    """dWqkv[3d, d] += dQKV^T @ X[tokens, d]."""
    N3, d = dw.shape
    A = dqkv[0, batch_index]
    return gemm_ex(A, x, N3, d, tokens, EPI_ATOMIC_F32, dw, a_layout=A_HEADS_T, w_layout=1, ldw=d, heads=heads,
                   a_part_stride=batch * heads * tokens * 64)


_ln_ws = {}


def layernorm_bwd(dy, x, mean, rstd, gamma, dres, accumulate, dgamma, dbeta, want_bf16=True, extra=None):
    """dres (+)= dLN/dx (+ extra, fp32 like x); returns the bf16 copy of the updated dres (or None)."""
    _chk(dy, torch.bfloat16, "dy")
    _chk(x, torch.float32, "x")
    _chk(dres, torch.float32, "dres")
    d = x.shape[-1]
    M = x.numel() // d
    db = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device) if want_bf16 else None
    if extra is not None:
        if _chk(extra, torch.float32, "extra").shape != x.shape:
            raise SmbvError(f"layernorm_bwd: extra must be shaped like x {tuple(x.shape)}")
        call("smbv_layernorm_bwd_add", _ptr(dy), _ptr(x), _ptr(mean), _ptr(rstd), _ptr(gamma), M, d, _ptr(dres),
             1 if accumulate else 0, _ptr(db), _ptr(dgamma), _ptr(dbeta), _ptr(extra), _stream())
        return db
    key = (str(x.device), d)
    if key not in _ln_ws:
        _ln_ws[key] = torch.empty((_lib.load().smbv_layernorm_bwd_blocks() * 2 * d,), dtype=torch.float32, device=x.device)
    call("smbv_layernorm_bwd", _ptr(dy), _ptr(x), _ptr(mean), _ptr(rstd), _ptr(gamma), M, d, _ptr(dres), 1 if accumulate else 0,
         _ptr(db), _ptr(dgamma), _ptr(dbeta), _ptr(_ln_ws[key]), _stream())
    return db


def colsum(x, out, M=None, N=None, ld=None):
    """out[N] += column sums of x[M,N] (bf16 or fp32)."""
    N = x.shape[-1] if N is None else N
    M = x.numel() // x.shape[-1] if M is None else M
    ld = x.shape[-1] if ld is None else ld
    _chk(out, torch.float32, "out")
    call("smbv_colsum_bf16" if x.dtype == torch.bfloat16 else "smbv_colsum_f32", _ptr(x), M, N, ld, _ptr(out), _stream())


def colsum_heads(dqkv, out, skip_k: bool = False):
    """out[3*H*64] += sum over batch and tokens of the head-major [3,B,H,n,64] buffer (skip_k: leave the K third alone)."""
    _chk(dqkv, torch.bfloat16, "dqkv")
    _chk(out, torch.float32, "out")
    _, B, H, n, _ = dqkv.shape
    call("smbv_colsum_heads_bf16", _ptr(dqkv), B, H, n, _ptr(out), 1 if skip_k else 0, _stream())


def gather_patches(volume, idx, n_sel):
    _chk(volume, torch.float32, "volume")
    _chk(idx, torch.int32, "idx")
    B, T, H, W = volume.shape
    out = torch.empty((B * n_sel, 4096), dtype=torch.bfloat16, device=volume.device)
    call("smbv_gather_patches_bf16", _ptr(volume), B, T, H, W, 16, _ptr(idx), n_sel, idx.shape[1], _ptr(out), _stream())
    return out


def cast_f32_scaled(src: torch.Tensor, dst: torch.Tensor, scale: float) -> torch.Tensor:
    _chk(src, torch.bfloat16, "src")
    _chk(dst, torch.float32, "dst")
    call("smbv_cast_bf16_f32_scale", _ptr(src), _ptr(dst), src.numel(), float(scale), _stream())
    return dst


def scale_add_recast_(x: torch.Tensor, scale: Optional[torch.Tensor] = None, addend: Optional[torch.Tensor] = None,
                      want_bf16: bool = True):
    """x = scale * x + addend in place (scale: a 1-element tensor, moved to the device as fp32 without a host sync; None = 1;
    addend fp32 like x or None); returns the bf16 copy of the result (or None)."""
    _chk(x, torch.float32, "x")
    if addend is not None and _chk(addend, torch.float32, "addend").shape != x.shape:
        raise SmbvError(f"scale_add_recast_: addend must be shaped like x {tuple(x.shape)}")
    sc = None if scale is None else scale.detach().to(device=x.device, dtype=torch.float32).reshape(1).contiguous()
    xb = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device) if want_bf16 else None
    call("smbv_scale_add_recast_f32", _ptr(x), x.numel(), _ptr(sc), _ptr(addend), _ptr(xb), _stream())
    return xb


# measurement hook (bench.py): a callable returning two raw cudaEvent_t handles that the library records around the dK/dV
# kernel of the next attention-backward call; None (the default) = no events
attn_bwd_event_source = None


def scale_f32_(x: torch.Tensor, scale: torch.Tensor) -> torch.Tensor:
    """x *= scale in place; scale = a 0-d / 1-element tensor (moved to the device as fp32 without a host sync)."""
    _chk(x, torch.float32, "x")
    sc = scale.detach().to(device=x.device, dtype=torch.float32).reshape(1).contiguous()
    call("smbv_scale_f32", _ptr(x), x.numel(), _ptr(sc), _stream())
    return x


# deterministic attention backward (two kernels, no cross-CTA reduction) instead of the fused one-pass kernel: process-wide
# default, overridable per call
ATTN_BWD_DETERMINISTIC = os.environ.get("SMBV_ATTN_BWD_DETERMINISTIC", "0") == "1"


def flash_attn_bwd(q, k, v, o, dout, lse, scale, dq=None, dk=None, dv=None, deterministic=None):
    """q,k,v bf16 [B,H,N,64] (or [H,N,64] for one sample); o,dout bf16 [B,N,H*64]; lse fp32 [B,H,N] -> (dq, dk, dv) like q.
    deterministic=False (default): fused one-pass kernel, dQ summed across key blocks by fp32 bulk reductions (dK, dV exact
    run to run, dQ equal up to fp32 summation order); True: the two-kernel path, bit-deterministic."""
    for t, nme in ((q, "q"), (k, "k"), (v, "v"), (o, "o"), (dout, "dout")):
        _chk(t, torch.bfloat16, nme)
    _chk(lse, torch.float32, "lse")
    B = 1 if q.dim() == 3 else q.shape[0]
    H, N = q.shape[-3], q.shape[-2]
    dev = q.device
    dsum = torch.empty((B, H, N), dtype=torch.float32, device=dev)
    outs = []
    for t, nme in ((dq, "dq"), (dk, "dk"), (dv, "dv")):
        outs.append(torch.empty(q.shape, dtype=torch.bfloat16, device=dev) if t is None else _chk(t, torch.bfloat16, nme))
    dq, dk, dv = outs
    ev = attn_bwd_event_source() if attn_bwd_event_source is not None else (None, None)
    if ATTN_BWD_DETERMINISTIC if deterministic is None else deterministic:
        call("smbv_flash_attn_bwd_ex", _ptr(q), _ptr(k), _ptr(v), _ptr(o), _ptr(dout), _ptr(lse), B, H, N, float(scale), _ptr(dsum),
             _ptr(dq), _ptr(dk), _ptr(dv), C.c_void_p(ev[0]), C.c_void_p(ev[1]), _stream())
    else:
        wsb = int(_lib.load().smbv_flash_attn_bwd_fused_workspace_bytes(B, H, N))
        ws = torch.empty((wsb,), dtype=torch.uint8, device=dev)  # fp32 dQ accumulator + partial dK / dV of the split last wave
        call("smbv_flash_attn_bwd_fused", _ptr(q), _ptr(k), _ptr(v), _ptr(o), _ptr(dout), _ptr(lse), B, H, N, float(scale),
             _ptr(dsum), _ptr(ws), wsb, _ptr(dq), _ptr(dk), _ptr(dv), C.c_void_p(ev[0]), C.c_void_p(ev[1]), _stream())
    return dq, dk, dv


# ----------------------------------------------------------------------------------------------
# classification head (reference VideoMAEForVideoClassification, modeling_videomae.py:917-1023)
# ----------------------------------------------------------------------------------------------
def token_sum(x: torch.Tensor) -> torch.Tensor:
    """x fp32 [B,N,d] -> fp32 [B,d] column sums per sample (the numerator of `sequence_output.mean(1)`, :975)."""
    _chk(x, torch.float32, "x")
    B, N, d = x.shape
    out = torch.empty((B, d), dtype=torch.float32, device=x.device)
    ws = torch.empty((B * int(_lib.load().smbv_token_sum_chunks(N)) * d,), dtype=torch.float32, device=x.device)
    call("smbv_token_sum", _ptr(x), B, N, d, _ptr(ws), _ptr(out), _stream())  # deterministic (no atomics)
    return out


def cls_head(pooled, inv_n: float, gamma, beta, eps: float, feats, W, bias, labels, problem: int, grads=None):
    """fc_norm -> cat(features) -> classifier -> loss, and (with `grads`) the head's whole backward in the same launch.

    pooled fp32 [B,d]; feats fp32 [B,F] or None; W fp32 [L,d+F]; labels int64 [B] (single label) / fp32 [B,L] / None.
    grads: dict(dW, dbias, dgamma, dbeta) of fp32 accumulators -> returns (loss, logits, dpooled [B,d])."""
    _chk(pooled, torch.float32, "pooled")
    _chk(W, torch.float32, "W")
    _chk(bias, torch.float32, "bias")
    B, d = pooled.shape
    L, D = W.shape
    F = D - d
    if F < 0 or (F > 0 and feats is None):
        raise SmbvError(f"cls_head: classifier expects {F} additional features")
    if feats is not None:
        _chk(feats, torch.float32, "additional_features")
        if tuple(feats.shape) != (B, F):
            raise SmbvError(f"cls_head: additional_features must be [{B},{F}], got {tuple(feats.shape)}")
    if gamma is not None:
        _chk(gamma, torch.float32, "gamma")
        _chk(beta, torch.float32, "beta")
    if problem != CLS_NONE:
        _chk(labels, torch.int64 if problem == CLS_SINGLE_LABEL else torch.float32, "labels")
        want = B if problem == CLS_SINGLE_LABEL else B * L
        if labels.numel() != want:
            raise SmbvError(f"cls_head: labels has {labels.numel()} elements, expected {want}")
    dev = pooled.device
    logits = torch.empty((B, L), dtype=torch.float32, device=dev)
    loss = torch.empty((1,), dtype=torch.float32, device=dev) if problem != CLS_NONE else None
    dpooled = None
    g = {}
    if grads is not None:
        dpooled = torch.empty((B, d), dtype=torch.float32, device=dev)
        g = {k: (None if v is None else _chk(v, torch.float32, k)) for k, v in grads.items()}
    call("smbv_cls_head", _ptr(pooled), float(inv_n), _ptr(gamma), _ptr(beta), float(eps), _ptr(feats), _ptr(W), _ptr(bias),
         _ptr(labels), B, d, F, L, problem, _ptr(logits), _ptr(loss), _ptr(g.get("dW")), _ptr(g.get("dbias")),
         _ptr(g.get("dgamma")), _ptr(g.get("dbeta")), _ptr(dpooled), _stream())
    return (None if loss is None else loss[0]), logits, dpooled


def broadcast_rows(g: torch.Tensor, N: int, want_bf16: bool = True):
    """g fp32 [B,d] -> (dx fp32 [B,N,d], dx bf16 or None) with dx[b,n,:] = g[b,:]."""
    _chk(g, torch.float32, "g")
    B, d = g.shape
    dx = torch.empty((B, N, d), dtype=torch.float32, device=g.device)
    dxb = torch.empty((B, N, d), dtype=torch.bfloat16, device=g.device) if want_bf16 else None
    call("smbv_broadcast_rows", _ptr(g), B, N, d, _ptr(dx), _ptr(dxb), _stream())
    return dx, dxb


# ----------------------------------------------------------------------------------------------
# input pipeline tail (reference src/dataloader/mim.py:154-170 + PermuteImage :86-91)
# ----------------------------------------------------------------------------------------------
def prepare_volume(raw: torch.Tensor, H: int, W: int, T: int, a_min: float, a_max: float, b_min: float, b_max: float,
                   clip: bool, out=None) -> torch.Tensor:
    """raw [X,Y,Z] fp32 / int16 (Z contiguous) -> fp32 [T,H,W]: scale-intensity + symmetric pad + centre crop + permute."""
    if not raw.is_cuda or not raw.is_contiguous() or raw.dim() != 3:
        raise SmbvError("prepare_volume: expected a contiguous CUDA tensor [X,Y,Z]")
    if raw.dtype not in (torch.float32, torch.int16):
        raise SmbvError(f"prepare_volume: dtype {raw.dtype} not supported (float32 or int16)")
    X, Y, Z = raw.shape
    if out is None:
        out = torch.empty((T, H, W), dtype=torch.float32, device=raw.device)
    else:
        _chk(out, torch.float32, "out")
        if tuple(out.shape) != (T, H, W):
            raise SmbvError(f"prepare_volume: out must be [{T},{H},{W}]")
    call("smbv_prepare_volume", _ptr(raw), 0 if raw.dtype == torch.float32 else 1, X, Y, Z, float(a_min), float(a_max), float(b_min),
         float(b_max), 1 if clip else 0, H, W, T, _ptr(out), _stream())
    return out


# ----------------------------------------------------------------------------------------------
# V-JEPA2-3D rotary embedding (reference src/models/vjepa/modeling_vjepa.py:204-228, :297-330)
# ----------------------------------------------------------------------------------------------
def rope3d_(x: torch.Tensor, grid_size: int, ids: Optional[torch.Tensor] = None, max_pos: int = 64, transpose: bool = False,
            first_generation_kernel: bool = False) -> torch.Tensor:
    """In place on x = bf16 [G,B,H,n,D] (or [B,H,n,D]): rotate the frame / height / width segments of every head row by
    the position of its token (ids int32 [B,n]; None = arange(n)).  transpose=True applies the transposed map (backward)."""
    _chk(x, torch.bfloat16, "x")
    if x.dim() == 4:
        G, (B, H, n, D) = 1, x.shape
    elif x.dim() == 5:
        G, B, H, n, D = x.shape
    else:
        raise SmbvError("rope3d_: x must be [G,B,H,n,D] or [B,H,n,D]")
    if ids is not None:
        _chk(ids, torch.int32, "ids")
        if tuple(ids.shape) != (B, n):
            raise SmbvError(f"rope3d_: ids must be [{B},{n}]")
    call("smbv_rope3d", _ptr(x), _ptr(ids), G, B, H, n, D, int(grid_size), int(max_pos),
         (1 if transpose else 0) | (2 if first_generation_kernel else 0), _stream())
    return x


def gather_rows(src: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    """`apply_masks` (modeling_vjepa.py:543-557): src fp32 [B,N,d], idx int32 [B,K] -> fp32 [B,K,d]."""
    _chk(src, torch.float32, "src")
    _chk(idx, torch.int32, "idx")
    B, N, d = src.shape
    if idx.dim() != 2 or idx.shape[0] != B:
        raise SmbvError(f"gather_rows: idx must be [{B}, K]")
    K = idx.shape[1]
    out = torch.empty((B, K, d), dtype=torch.float32, device=src.device)
    if K == 0:
        return out
    call("smbv_gather_rows_f32", _ptr(src), _ptr(idx), B, N, K, d, _ptr(out), _stream())
    return out


def scatter_rows(src: torch.Tensor, idx: torch.Tensor, N: int, K: Optional[int] = None) -> torch.Tensor:
    """adjoint of gather_rows: src fp32 [B,K,d], idx int32 [B, >= K] -> fp32 [B,N,d], zero except out[b, idx[b,k]] = src[b,k]."""
    _chk(src, torch.float32, "src")
    _chk(idx, torch.int32, "idx")
    B, Ks, d = src.shape
    K = Ks if K is None else K
    out = torch.zeros((B, N, d), dtype=torch.float32, device=src.device)
    if K:
        call("smbv_scatter_rows_f32", _ptr(src), _ptr(idx), B, N, K, idx.shape[1], d, _ptr(out), _stream())
    return out


def heads32_expand(x: torch.Tensor) -> torch.Tensor:
    """head-major bf16 [..., H/2, n, 64] (two 32-wide heads per row) -> [..., H, n, 64] rows {head, 0...0}."""
    _chk(x, torch.bfloat16, "x")
    *outer, H2, n, w = x.shape
    if w != 64:
        raise SmbvError("heads32_expand: rows must be 64 wide")
    o = 1
    for v in outer:
        o *= v
    out = torch.empty((*outer, 2 * H2, n, 64), dtype=torch.bfloat16, device=x.device)
    call("smbv_heads32_convert", _ptr(x), _ptr(out), o, 2 * H2, n, 1, 1, _stream())
    return out


def heads32_squeeze(x: torch.Tensor) -> torch.Tensor:
    """inverse of heads32_expand: [..., H, n, 64] -> [..., H/2, n, 64] (the zero pad is dropped)."""
    _chk(x, torch.bfloat16, "x")
    *outer, H, n, w = x.shape
    o = 1
    for v in outer:
        o *= v
    out = torch.empty((*outer, H // 2, n, 64), dtype=torch.bfloat16, device=x.device)
    call("smbv_heads32_convert", _ptr(x), _ptr(out), o, H, n, 1, 0, _stream())
    return out


def heads32_tokens(x: torch.Tensor, H: int, expand: bool) -> torch.Tensor:
    """token-major bf16 [B, n, H*32] -> [B, n, H*64] zero-padded per head (expand) or back (not expand)."""
    _chk(x, torch.bfloat16, "x")
    B, n, w = x.shape
    out = torch.empty((B, n, H * (64 if expand else 32)), dtype=torch.bfloat16, device=x.device)
    call("smbv_heads32_convert", _ptr(x), _ptr(out), B, H, n, 0, 1 if expand else 0, _stream())
    return out


def position_sort(pos: torch.Tensor, doubled: bool = False):
    """int32 [B,n] -> (order, inv, sorted[, sorted2 [B,2n]]): argsort, reverse argsort, sorted ids (see include/smbv_b200.h)."""
    _chk(pos, torch.int32, "pos")
    B, n = pos.shape
    order, inv, srt = (torch.empty((B, n), dtype=torch.int32, device=pos.device) for _ in range(3))
    s2 = torch.empty((B, 2 * n), dtype=torch.int32, device=pos.device) if doubled else None
    call("smbv_position_sort", _ptr(pos), B, n, _ptr(order), _ptr(inv), _ptr(srt), _ptr(s2), _stream())
    return (order, inv, srt, s2) if doubled else (order, inv, srt)


_l1_ws = {}


def l1_loss(pred: torch.Tensor, target: torch.Tensor, want_grad: bool = False, upstream: float = 1.0):
    """nn.L1Loss (src/run_vjepa.py:108): mean |pred - target| as a device scalar [1] (+ d loss / d pred when want_grad)."""
    _chk(pred, torch.float32, "pred")
    _chk(target, torch.float32, "target")
    if pred.shape != target.shape:
        raise SmbvError(f"l1_loss: shapes differ {tuple(pred.shape)} vs {tuple(target.shape)}")
    key = str(pred.device)
    if key not in _l1_ws:
        _l1_ws[key] = torch.empty((int(_lib.load().smbv_l1_workspace_floats()),), dtype=torch.float32, device=pred.device)
    loss = torch.empty((1,), dtype=torch.float32, device=pred.device)
    dpred = torch.empty_like(pred) if want_grad else None
    call("smbv_l1_loss_f32", _ptr(pred), _ptr(target), pred.numel(), _ptr(_l1_ws[key]), _ptr(loss), _ptr(dpred), float(upstream), _stream())
    return (loss, dpred) if want_grad else loss


# ----------------------------------------------------------------------------------------------
# small head dimensions (8/16/32): fused token-major QKV [B,n,3,H,hd]
# ----------------------------------------------------------------------------------------------
def attn_small_fwd(qkv: torch.Tensor, heads: int, scale: float, return_lse: bool = False):
    """qkv bf16 [B,n,3*d] (the plain QKV GEMM output, d = heads*hd) -> out bf16 [B,n,d] (+ lse fp32 [B,heads,n])."""
    _chk(qkv, torch.bfloat16, "qkv")
    B, n, d3 = qkv.shape
    d = d3 // 3
    hd = d // heads
    out = torch.empty((B, n, d), dtype=torch.bfloat16, device=qkv.device)
    lse = torch.empty((B, heads, n), dtype=torch.float32, device=qkv.device) if return_lse else None
    p = qkv.data_ptr()
    call("smbv_attn_small_fwd", C.c_void_p(p), C.c_void_p(p + 2 * d), C.c_void_p(p + 4 * d), n * d3, hd, d3, B, heads, n, hd, float(scale),
         _ptr(out), _ptr(lse), _stream())
    return (out, lse) if return_lse else out


def attn_small_bwd(qkv, out, dout, lse, heads: int, scale: float) -> torch.Tensor:
    """-> dqkv bf16 [B,n,3*d] in the layout of `qkv` (rows of the QKV GEMM output gradient)."""
    for t, nme in ((qkv, "qkv"), (out, "out"), (dout, "dout")):
        _chk(t, torch.bfloat16, nme)
    _chk(lse, torch.float32, "lse")
    B, n, d3 = qkv.shape
    d = d3 // 3
    hd = d // heads
    dqkv = torch.empty_like(qkv)
    dsum = torch.empty((B, heads, n), dtype=torch.float32, device=qkv.device)
    p, g = qkv.data_ptr(), dqkv.data_ptr()
    call("smbv_attn_small_bwd", C.c_void_p(p), C.c_void_p(p + 2 * d), C.c_void_p(p + 4 * d), n * d3, hd, d3, _ptr(out), _ptr(dout), _ptr(lse),
         B, heads, n, hd, float(scale), _ptr(dsum), C.c_void_p(g), C.c_void_p(g + 2 * d), C.c_void_p(g + 4 * d), n * d3, hd, d3, _stream())
    return dqkv


def attn_small_fwd_strided(q, k, v, scale: float):
    """q,k,v bf16 [B,H,N,hd] contiguous (head-major) -> (out bf16 [B,N,H*hd], lse fp32 [B,H,N])."""
    for t, nme in ((q, "q"), (k, "k"), (v, "v")):
        _chk(t, torch.bfloat16, nme)
    B, H, N, hd = q.shape
    out = torch.empty((B, N, H * hd), dtype=torch.bfloat16, device=q.device)
    lse = torch.empty((B, H, N), dtype=torch.float32, device=q.device)
    call("smbv_attn_small_fwd", _ptr(q), _ptr(k), _ptr(v), H * N * hd, N * hd, hd, B, H, N, hd, float(scale), _ptr(out), _ptr(lse), _stream())
    return out, lse


def attn_small_bwd_strided(q, k, v, out, dout, lse, scale: float):
    """head-major inputs as above; out / dout bf16 [B,N,H*hd] -> (dq, dk, dv) bf16 [B,H,N,hd]."""
    for t, nme in ((q, "q"), (k, "k"), (v, "v"), (out, "out"), (dout, "dout")):
        _chk(t, torch.bfloat16, nme)
    _chk(lse, torch.float32, "lse")
    B, H, N, hd = q.shape
    dq, dk, dv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
    dsum = torch.empty((B, H, N), dtype=torch.float32, device=q.device)
    call("smbv_attn_small_bwd", _ptr(q), _ptr(k), _ptr(v), H * N * hd, N * hd, hd, _ptr(out), _ptr(dout), _ptr(lse), B, H, N, hd, float(scale),
         _ptr(dsum), _ptr(dq), _ptr(dk), _ptr(dv), H * N * hd, N * hd, hd, _stream())
    return dq, dk, dv
