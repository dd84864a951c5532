"""Developer harness for the B200 box: runs every kernel family against a torch reference in its OWN subprocess
(a trapped kernel poisons the CUDA context) with a timeout, and writes gpurun_out/gpu_check.json.

    python tools/gpu_check.py all            # everything
    python tools/gpu_check.py gemm attn      # selected groups
"""
from __future__ import annotations

import json
import os
import subprocess
import sys
import time
import traceback

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "gpurun_out")

RESULTS = []


def rec(name, ok, **kw):
    RESULTS.append(dict(name=name, ok=bool(ok), **kw))
    print(("PASS " if ok else "FAIL ") + name + " " + json.dumps(kw, default=str)[:600], flush=True)


def relerr(a, b):
    import torch
    a, b = a.double(), b.double()
    return (torch.linalg.norm(a - b) / (torch.linalg.norm(b) + 1e-30)).item(), (a - b).abs().max().item()


def timeit(fn, iters=10, warmup=3):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


# ------------------------------------------------------------------------------------------
def g_bandwidth():
    import numpy as np
    import torch
    from oracle.mim_mask import OracleMaskGenerator
    from oracle import videomae_oracle as vo
    from smb_vision_b200 import ops
    dev = "cuda"
    # mask upsample + index
    for size, depth in [(96, 96), (512, 320)]:
        np.random.seed(0)
        g = OracleMaskGenerator(size, depth, 32, 16, 0.65)
        coarse = np.stack([g.coarse(), g.coarse()])
        fine_ref = np.stack([g.upsample(c, g.scale) for c in coarse])
        fine = ops.mask_upsample(torch.from_numpy(coarse).to(dev), g.scale)
        ok = np.array_equal(fine.cpu().numpy(), fine_ref)
        vis, msk, slot, counts = ops.mask_index(fine)
        torch.cuda.synchronize()
        for b in range(2):
            nv, nm = counts[b].tolist()
            ok &= nv == int((fine_ref[b] == 0).sum()) and nm == int(fine_ref[b].sum())
            ok &= np.array_equal(vis[b, :nv].cpu().numpy(), np.nonzero(fine_ref[b] == 0)[0])
            ok &= np.array_equal(msk[b, :nm].cpu().numpy(), np.nonzero(fine_ref[b])[0])
            s = slot[b].cpu().numpy()
            ok &= np.array_equal(s[np.nonzero(fine_ref[b] == 0)[0]], np.arange(nv)) and np.array_equal(s[np.nonzero(fine_ref[b])[0]], np.arange(nm))
        rec(f"mask_{size}x{depth}", ok)
    # sincos
    for n, d in [(216, 64), (20480, 768), (20480, 384)]:
        t = ops.sincos_table(n, d, dev)
        ref = vo.sinusoid_table(n, d)[0].to(dev)
        rec(f"sincos_{n}x{d}", (t - ref).abs().max().item() <= 1.2e-7, maxabs=(t - ref).abs().max().item(),
            exact=bool(torch.equal(t, ref)))
    # layernorm
    for M, d, eps in [(216, 64, 1e-12), (72, 32, 1e-5), (20480, 768, 1e-12), (13312, 384, 1e-5), (1000, 1024, 1e-6)]:
        x = torch.randn(M, d, device=dev) * 2 + 0.5
        gm, bt = torch.randn(d, device=dev), torch.randn(d, device=dev)
        y, mean, rstd = ops.layernorm_fwd(x, gm, bt, eps, save_stats=True)
        ref = torch.nn.functional.layer_norm(x, (d,), gm, bt, eps)
        fr, mx = relerr(y.float(), ref)
        rec(f"layernorm_{M}x{d}", fr < 3e-3, frob=fr, maxabs=mx, mean_err=(mean - x.mean(1)).abs().max().item())
    x = torch.randn(20480, 768, device=dev)
    gm, bt = torch.ones(768, device=dev), torch.zeros(768, device=dev)
    ms = timeit(lambda: ops.layernorm_fwd(x, gm, bt, 1e-12))
    rec("layernorm_time_20480x768", True, ms=ms, gbs=(x.numel() * 6) / ms / 1e6)
    # cast
    s = torch.randn(1000003, device=dev)[:1000000]
    rec("cast_bf16", torch.equal(ops.cast_bf16(s.contiguous()), s.to(torch.bfloat16)))
    # fill mask tokens
    B, N, d, nv = 2, 216, 32, 72
    xd = torch.zeros(B, N, d, device=dev)
    mt, pos = torch.randn(d, device=dev), torch.randn(N, d, device=dev)
    midx = torch.stack([torch.randperm(N, device=dev)[: N - nv].sort().values for _ in range(B)]).int()
    midx_p = torch.zeros(B, N, dtype=torch.int32, device=dev)
    midx_p[:, : N - nv] = midx
    ops.fill_mask_tokens(xd, mt, pos, midx_p, nv)
    ref = mt[None, None] + pos[midx.long()]
    rec("fill_mask_tokens", torch.equal(xd[:, nv:], ref) and xd[:, :nv].abs().max().item() == 0)
    # loss
    for name, cfgd, B in [("tiny", vo.TINY, 2), ("full", {}, 1)]:
        cfg = vo.OracleConfig(**cfgd)
        x = vo.synthetic_volume(cfg, B, 7)
        np.random.seed(0)
        g = OracleMaskGenerator(cfg.image_size, cfg.num_frames, 32, 16, 0.65)
        mask = torch.from_numpy(np.stack([g() for _ in range(B)]))
        nm = int(mask[0].sum())
        lab = vo.labels_normpix(x, cfg)[mask].reshape(B, nm, -1)
        logits = (0.3 * torch.randn(B, nm, 4096)).to(torch.bfloat16)
        xg = x[:, :, 0].contiguous().to(dev)
        _, midx, _, _ = ops.mask_index(mask.to(torch.uint8).to(dev))
        for kind, kname in [(0, "mse"), (1, "l1")]:
            loss, dl = ops.normpix_loss(xg, midx, nm, logits.to(dev), True, kind)
            lf = logits.float().requires_grad_(True)
            lref = torch.nn.functional.mse_loss(lf, lab) if kind == 0 else torch.nn.functional.l1_loss(lf, lab)
            lref.backward()
            fr, mx = relerr(dl.float().cpu(), lf.grad)
            lrel = abs(loss.item() - lref.item()) / lref.item()
            rec(f"loss_{name}_{kname}", lrel < 1e-5 and fr < 4e-3, loss=loss.item(), ref=lref.item(), rel=lrel, grad_frob=fr)
        if name == "full":
            lg = logits.to(dev)
            ms = timeit(lambda: ops.normpix_loss(xg, midx, nm, lg, True, 0))
            bytes_alg = nm * 4096 * (4 + 2 + 2)
            rec("loss_time_full_fwd_bwd", True, ms=ms, gbs=bytes_alg / ms / 1e6, alg_mb=bytes_alg / 1e6)
            ms = timeit(lambda: ops.normpix_loss(xg, midx, nm, lg, False, 0))
            rec("loss_time_full_fwd", True, ms=ms, gbs=nm * 4096 * 6 / ms / 1e6)
            ms = timeit(lambda: ops.normpix_loss(xg, midx, nm, lg, True, 16))
            rec("loss_time_full_fwd_bwd_blockkernel", True, ms=ms, gbs=bytes_alg / ms / 1e6)


def g_gemm():
    import torch
    from smb_vision_b200 import ops
    dev = "cuda"
    torch.manual_seed(0)
    shapes = [(128, 128, 64), (128, 256, 128), (256, 128, 768), (216, 192, 64), (72, 32, 64), (144, 4096, 32),
              (1000, 768, 3072), (7168, 2304, 768), (20480, 768, 3072)]
    for M, N, K in shapes:
        a = (torch.randn(M, K, device=dev)).to(torch.bfloat16)
        w = (torch.randn(N, K, device=dev) * 0.05).to(torch.bfloat16)
        bias = torch.randn(N, device=dev)
        ref = a.float() @ w.float().t() + bias
        out = ops.gemm(a, w, bias, ops.EPI_F32)
        fr, mx = relerr(out, ref)
        extra = {}
        if fr > 1e-3:
            extra = dict(got=out[:2, :6].tolist(), want=ref[:2, :6].tolist())
        rec(f"gemm_f32_{M}x{N}x{K}", fr < 1e-3, frob=fr, maxabs=mx, **extra)
    M, N, K = 512, 768, 768
    a = torch.randn(M, K, device=dev).to(torch.bfloat16)
    w = (torch.randn(N, K, device=dev) * 0.05).to(torch.bfloat16)
    bias = torch.randn(N, device=dev)
    ref = a.float() @ w.float().t() + bias
    fr, _ = relerr(ops.gemm(a, w, bias, ops.EPI_BF16).float(), ref)
    rec("gemm_epi_bf16", fr < 5e-3, frob=fr)
    fr, _ = relerr(ops.gemm(a, w, None, ops.EPI_BF16).float(), ref - bias)
    rec("gemm_epi_bf16_nobias", fr < 5e-3, frob=fr)
    fr, _ = relerr(ops.gemm(a, w, bias, ops.EPI_GELU_BF16).float(), torch.nn.functional.gelu(ref))
    rec("gemm_epi_gelu", fr < 5e-3, frob=fr)
    res = torch.randn(M, N, device=dev)
    res0 = res.clone()
    ops.gemm(a, w, bias, ops.EPI_RESID_F32, residual=res)
    fr, _ = relerr(res, res0 + ref)
    rec("gemm_epi_resid_inplace", fr < 1e-3, frob=fr)
    # qkv heads
    B, T, H = 2, 256, 4
    a = torch.randn(B * T, 256, device=dev).to(torch.bfloat16)
    w = (torch.randn(3 * H * 64, 256, device=dev) * 0.05).to(torch.bfloat16)
    bias = torch.randn(3 * H * 64, device=dev)
    out = ops.gemm(a, w, bias, ops.EPI_QKV_HEADS, heads=H, tokens=T)
    ref = (a.float() @ w.float().t() + bias).view(B, T, 3, H, 64).permute(2, 0, 3, 1, 4)
    fr, _ = relerr(out.float(), ref)
    rec("gemm_epi_qkv_heads", fr < 5e-3, frob=fr)
    # pos gather
    M, N, K = 144, 32, 64
    a = torch.randn(M, K, device=dev).to(torch.bfloat16)
    w = (torch.randn(N, K, device=dev) * 0.05).to(torch.bfloat16)
    pos = torch.randn(216, N, device=dev)
    rm = torch.randperm(216, device=dev)[:M].int()
    out = ops.gemm(a, w, None, ops.EPI_POS_GATHER_F32, pos=pos, row_map=rm)
    fr, _ = relerr(out, a.float() @ w.float().t() + pos[rm.long()])
    rec("gemm_epi_pos_gather", fr < 1e-3, frob=fr)
    # timing at the model's shapes
    for M, N, K, epi in [(20480, 2304, 768, "qkv"), (20480, 768, 768, "resid"), (20480, 3072, 768, "gelu"),
                         (20480, 768, 3072, "resid"), (13312, 4096, 384, "bf16"), (7168, 3072, 768, "gelu")]:
        a = torch.randn(M, K, device=dev).to(torch.bfloat16)
        w = (torch.randn(N, K, device=dev) * 0.05).to(torch.bfloat16)
        bias = torch.randn(N, device=dev)
        res = torch.zeros(M, N, device=dev) if epi == "resid" else None
        if epi == "qkv":
            fn = lambda: ops.gemm(a, w, bias, ops.EPI_QKV_HEADS, heads=N // 192, tokens=M)
        elif epi == "resid":
            fn = lambda: ops.gemm(a, w, bias, ops.EPI_RESID_F32, residual=res)
        elif epi == "gelu":
            fn = lambda: ops.gemm(a, w, bias, ops.EPI_GELU_BF16)
        else:
            fn = lambda: ops.gemm(a, w, bias, ops.EPI_BF16)
        ms = timeit(fn)
        ms_t = timeit(lambda: a @ w.t())
        rec(f"gemm_time_{M}x{N}x{K}_{epi}", True, ms=ms, tflops=2 * M * N * K / ms / 1e9, torch_matmul_ms=ms_t,
            torch_tflops=2 * M * N * K / ms_t / 1e9)


def _attn_case(B, H, N, scale=0.125, seed=0):
    import torch
    from smb_vision_b200 import ops
    dev = "cuda"
    torch.manual_seed(seed)
    q = torch.randn(B, H, N, 64, device=dev).to(torch.bfloat16)
    k = torch.randn(B, H, N, 64, device=dev).to(torch.bfloat16)
    v = torch.randn(B, H, N, 64, device=dev).to(torch.bfloat16)
    out, lse = ops.flash_attn_fwd(q, k, v, scale, return_lse=True)
    s = (q.float() @ k.float().transpose(-1, -2)) * scale
    ref = (torch.softmax(s, -1) @ v.float()).transpose(1, 2).reshape(B, N, H * 64)
    lref = torch.logsumexp(s, -1)
    fr, mx = relerr(out.float(), ref)
    extra = {}
    if not fr < 1e-2:
        extra = dict(got=out[0, :2, :4].tolist(), want=ref[0, :2, :4].tolist())
    rec(f"attn_B{B}H{H}N{N}", fr < 1e-2, frob=fr, maxabs=mx, lse_err=(lse - lref).abs().max().item(), **extra)


def g_attn():
    for B, H, N in [(1, 1, 128), (1, 2, 256), (2, 3, 1024), (1, 2, 216), (1, 1, 72), (1, 1, 384), (1, 2, 3000)]:
        _attn_case(B, H, N)


def g_attn_big():
    import torch
    from smb_vision_b200 import ops
    dev = "cuda"
    # large-magnitude scores exercise the lazy rescale path
    torch.manual_seed(1)
    B, H, N = 1, 2, 2048
    q = (torch.randn(B, H, N, 64, device=dev) * 3).to(torch.bfloat16)
    k = (torch.randn(B, H, N, 64, device=dev) * 3).to(torch.bfloat16)
    v = torch.randn(B, H, N, 64, device=dev).to(torch.bfloat16)
    out = ops.flash_attn_fwd(q, k, v, 0.125)
    s = (q.float() @ k.float().transpose(-1, -2)) * 0.125
    ref = (torch.softmax(s, -1) @ v.float()).transpose(1, 2).reshape(B, N, H * 64)
    fr, mx = relerr(out.float(), ref)
    rec("attn_large_scores", fr < 1e-2, frob=fr, maxabs=mx)
    for H, N in [(12, 20480), (12, 7168), (6, 20480)]:
        q = torch.randn(1, H, N, 64, device=dev).to(torch.bfloat16)
        k = torch.randn(1, H, N, 64, device=dev).to(torch.bfloat16)
        v = torch.randn(1, H, N, 64, device=dev).to(torch.bfloat16)
        out = ops.flash_attn_fwd(q, k, v, 0.125)
        ref = torch.nn.functional.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(1, N, H * 64)
        fr, mx = relerr(out.float(), ref.float())
        ms = timeit(lambda: ops.flash_attn_fwd(q, k, v, 0.125), iters=5, warmup=2)
        ms_t = timeit(lambda: torch.nn.functional.scaled_dot_product_attention(q, k, v), iters=5, warmup=2)
        fl = 4.0 * N * N * 64 * H
        rec(f"attn_time_H{H}N{N}", fr < 1e-2, frob_vs_sdpa=fr, ms=ms, tflops=fl / ms / 1e9, torch_sdpa_ms=ms_t,
            torch_sdpa_tflops=fl / ms_t / 1e9)


def g_patch():
    import numpy as np
    import torch
    from oracle import videomae_oracle as vo
    from oracle.mim_mask import OracleMaskGenerator
    from smb_vision_b200 import ops
    dev = "cuda"
    for name, cfgd, B in [("tiny", vo.TINY, 2), ("full", {}, 1)]:
        cfg = vo.OracleConfig(**cfgd)
        D = cfg.hidden_size
        x = vo.synthetic_volume(cfg, B, 7)
        torch.manual_seed(3)
        w = torch.randn(D, 4096) * 0.02
        b = torch.randn(D) * 0.1
        P = vo.patchify(x, cfg)
        pos = vo.sinusoid_table(cfg.num_patches, D)[0]
        ref = (P.double() @ w.double().t() + b.double() + pos.double()).float()
        xg = x[:, :, 0].contiguous().to(dev)
        wg, bg, pg = w.to(dev).bfloat16(), b.to(dev), pos.to(dev)  # the kernel's operand: bf16 weight (cast once)
        out = ops.patch_embed_fwd(xg, wg, bg, pg)
        fr, mx = relerr(out.cpu(), ref)
        extra = {}
        if not fr < 2e-3:
            extra = dict(got=out[0, :2, :4].tolist(), want=ref[0, :2, :4].tolist(), got_last=out[0, -1, :4].tolist(), want_last=ref[0, -1, :4].tolist())
        rec(f"patch_embed_{name}_all", fr < 5e-3, frob=fr, maxabs=mx, **extra)
        np.random.seed(0)
        g = OracleMaskGenerator(cfg.image_size, cfg.num_frames, 32, 16, 0.65)
        mask = torch.from_numpy(np.stack([g() for _ in range(B)]))
        fine = mask.to(torch.uint8).to(dev)
        vis, msk, slot, counts = ops.mask_index(fine)
        nv = int((~mask[0]).sum())
        out = ops.patch_embed_fwd(xg, wg, bg, pg, fine, slot, nv)
        refv = ref[~mask].reshape(B, nv, D)
        fr, mx = relerr(out.cpu(), refv)
        rec(f"patch_embed_{name}_visible", fr < 5e-3, frob=fr, maxabs=mx)
        if name == "full":
            ms = timeit(lambda: ops.patch_embed_fwd(xg, wg, bg, pg), iters=5, warmup=2)
            rec("patch_embed_time_full", True, ms=ms, tflops=2 * 20480 * 4096 * 768 / ms / 1e9,
                gbs=(xg.numel() * 4 + 20480 * 768 * 8 + 768 * 4096 * 2) / ms / 1e6, algorithmic_mb=(xg.numel() * 4 + 20480 * 768 * 8 + 768 * 4096 * 2) / 1e6)


def g_bwd_gemm():
    import torch
    from smb_vision_b200 import ops
    dev = "cuda"
    torch.manual_seed(0)
    for M, N, K in [(256, 128, 64), (216, 384, 128), (7168, 768, 3072), (20480, 3072, 768), (13312, 4096, 384)]:
        dy = torch.randn(M, N, device=dev).to(torch.bfloat16)
        w = (torch.randn(N, K, device=dev) * 0.05).to(torch.bfloat16)
        x = torch.randn(M, K, device=dev).to(torch.bfloat16)
        ref = dy.float() @ w.float()
        got = ops.linear_dgrad(dy, w)
        fr, _ = relerr(got.float(), ref)
        rec(f"dgrad_{M}x{N}x{K}", fr < 5e-3, frob=fr)
        got32 = ops.linear_dgrad(dy, w, out_dtype=torch.float32)
        fr, _ = relerr(got32, ref)
        rec(f"dgrad_f32_{M}x{N}x{K}", fr < 1e-4, frob=fr)
        pre = torch.randn(M, K, device=dev).to(torch.bfloat16)
        got = ops.linear_dgrad(dy, w, aux=pre)
        pf = pre.float().requires_grad_(True)
        torch.nn.functional.gelu(pf).backward(ref)
        fr, _ = relerr(got.float(), pf.grad)
        rec(f"dgrad_dgelu_{M}x{N}x{K}", fr < 6e-3, frob=fr)
        dw = torch.zeros(N, K, device=dev)
        ops.linear_wgrad(dy, x, dw)
        refw = dy.float().t() @ x.float()
        fr, _ = relerr(dw, refw)
        rec(f"wgrad_{M}x{N}x{K}", fr < 1e-4, frob=fr)
        if M >= 7168:
            ms = timeit(lambda: ops.linear_dgrad(dy, w))
            ms2 = timeit(lambda: ops.linear_wgrad(dy, x, dw))
            rec(f"bwd_gemm_time_{M}x{N}x{K}", True, dgrad_ms=ms, dgrad_tflops=2 * M * N * K / ms / 1e9, wgrad_ms=ms2, wgrad_tflops=2 * M * N * K / ms2 / 1e9)
    # head-major views
    B, H, T, d = 2, 2, 216, 128
    dqkv = torch.randn(3, B, H, T, 64, device=dev).to(torch.bfloat16)
    w = (torch.randn(3 * H * 64, d, device=dev) * 0.05).to(torch.bfloat16)
    x = torch.randn(B, T, d, device=dev).to(torch.bfloat16)
    dw = torch.zeros(3 * H * 64, d, device=dev)
    for b in range(B):
        flat = dqkv[:, b].permute(2, 0, 1, 3).reshape(T, 3 * H * 64).float()  # [T, (part, h, dd)]
        got = ops.qkv_dgrad(dqkv, w, T, H, batch_index=b, batch=B)
        fr, _ = relerr(got.float(), flat @ w.float())
        rec(f"qkv_dgrad_b{b}", fr < 5e-3, frob=fr)
        ops.qkv_wgrad(dqkv, x[b].contiguous(), dw, T, H, batch_index=b, batch=B)
    refw = sum(dqkv[:, b].permute(2, 0, 1, 3).reshape(T, 3 * H * 64).float().t() @ x[b].float() for b in range(B))
    fr, _ = relerr(dw, refw)
    rec("qkv_wgrad", fr < 1e-4, frob=fr)
    out = torch.zeros(3 * H * 64, device=dev)
    ops.colsum_heads(dqkv, out)
    fr, _ = relerr(out, dqkv.float().sum(dim=(1, 3)).reshape(-1))
    rec("colsum_heads", fr < 1e-5, frob=fr)
    for M, N in [(216, 128), (13312, 4096), (7168, 768)]:
        xx = torch.randn(M, N, device=dev)
        o1, o2 = torch.zeros(N, device=dev), torch.zeros(N, device=dev)
        ops.colsum(xx, o1)
        ops.colsum(xx.to(torch.bfloat16), o2)
        f1, _ = relerr(o1, xx.sum(0))
        f2, _ = relerr(o2, xx.to(torch.bfloat16).float().sum(0))
        rec(f"colsum_{M}x{N}", f1 < 1e-5 and f2 < 1e-5, f32=f1, bf16=f2)
    # layernorm backward
    for M, d in [(216, 128), (72, 64), (7168, 768), (20480, 384)]:
        x = (torch.randn(M, d, device=dev) * 2 + 0.3).requires_grad_(True)
        gm = torch.randn(d, device=dev, requires_grad=True)
        bt = torch.randn(d, device=dev, requires_grad=True)
        dy = torch.randn(M, d, device=dev).to(torch.bfloat16)
        torch.nn.functional.layer_norm(x, (d,), gm, bt, 1e-6).backward(dy.float())
        _, mean, rstd = ops.layernorm_fwd(x.detach(), gm.detach(), bt.detach(), 1e-6, save_stats=True)
        dres0 = torch.randn(M, d, device=dev)
        dres = dres0.clone()
        dg, dbt = torch.zeros(d, device=dev), torch.zeros(d, device=dev)
        dbf = ops.layernorm_bwd(dy, x.detach(), mean, rstd, gm.detach(), dres, True, dg, dbt)
        f1, _ = relerr(dres - dres0, x.grad)
        f2, _ = relerr(dg, gm.grad)
        f3, _ = relerr(dbt, bt.grad)
        f4, _ = relerr(dbf.float(), dres)
        rec(f"ln_bwd_{M}x{d}", f1 < 1e-4 and f2 < 1e-4 and f3 < 1e-4 and f4 < 4e-3, dx=f1, dgamma=f2, dbeta=f3, bf16=f4)
    # patch gather
    import numpy as np
    from oracle import videomae_oracle as vo
    cfg = vo.OracleConfig(**vo.TINY)
    xv = vo.synthetic_volume(cfg, 2, 3)
    P = vo.patchify(xv, cfg)
    idx = torch.stack([torch.randperm(216)[:72].sort().values for _ in range(2)]).int()
    idxp = torch.zeros(2, 216, dtype=torch.int32)
    idxp[:, :72] = idx
    got = ops.gather_patches(xv[:, :, 0].contiguous().to(dev), idxp.to(dev), 72)
    ref = torch.stack([P[b, idx[b].long()] for b in range(2)]).reshape(144, 4096).to(torch.bfloat16)
    rec("gather_patches", torch.equal(got.cpu(), ref))


def _attn_bwd_case(H, N, seed=0, mag=1.0):
    import torch
    from smb_vision_b200 import ops
    dev = "cuda"
    torch.manual_seed(seed)
    q = (mag * torch.randn(H, N, 64, device=dev)).to(torch.bfloat16)
    k = (mag * torch.randn(H, N, 64, device=dev)).to(torch.bfloat16)
    v = torch.randn(H, N, 64, device=dev).to(torch.bfloat16)
    dout = torch.randn(N, H * 64, device=dev).to(torch.bfloat16)
    o, lse = ops.flash_attn_fwd(q[None], k[None], v[None], 0.125, return_lse=True)
    dq, dk, dv = ops.flash_attn_bwd(q, k, v, o[0], dout, lse[0], 0.125)
    qf, kf, vf = (t.float().requires_grad_(True) for t in (q, k, v))
    s = (qf @ kf.transpose(-1, -2)) * 0.125
    of = (torch.softmax(s, -1) @ vf).transpose(0, 1).reshape(N, H * 64)
    of.backward(dout.float())
    f1, _ = relerr(dq.float(), qf.grad)
    f2, _ = relerr(dk.float(), kf.grad)
    f3, _ = relerr(dv.float(), vf.grad)
    rec(f"attn_bwd_H{H}N{N}", f1 < 1e-2 and f2 < 1e-2 and f3 < 1e-2, dq=f1, dk=f2, dv=f3)


def g_attn_bwd():
    import torch
    from smb_vision_b200 import ops
    for H, N in [(1, 128), (2, 256), (2, 216), (1, 72), (3, 1024), (2, 1000)]:
        _attn_bwd_case(H, N)
    _attn_bwd_case(2, 512, seed=1, mag=2.5)
    dev = "cuda"
    for H, N in [(12, 7168), (6, 20480)]:
        q, k, v = (torch.randn(H, N, 64, device=dev).to(torch.bfloat16) for _ in range(3))
        dout = torch.randn(N, H * 64, device=dev).to(torch.bfloat16)
        o, lse = ops.flash_attn_fwd(q[None], k[None], v[None], 0.125, return_lse=True)
        ms = timeit(lambda: ops.flash_attn_bwd(q, k, v, o[0], dout, lse[0], 0.125), iters=3, warmup=1)
        rec(f"attn_bwd_time_H{H}N{N}", True, ms=ms, tflops=10.0 * N * N * 64 * H / ms / 1e9)


def g_neighbours():
    """HBM-bound kernels either side of the hot path (SURVEY.md §8f): achieved GB/s against MEASURED_PEAKS.json."""
    import ctypes as C

    import torch
    from smb_vision_b200 import ops
    from smb_vision_b200._lib import call
    dev = "cuda"
    peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"] if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def report(name, nbytes, fn, iters=20):
        ms = timeit(fn, iters=iters)
        gbs = nbytes / ms / 1e6
        rec(name, True, ms=round(ms, 4), gbs=round(gbs, 1), frac_of_hbm_peak=round(gbs / peak, 3), algorithmic_mb=round(nbytes / 1e6, 1))

    # optimiser over the smb-vision-base arena (97.2 M parameters)
    n = 97_161_088 // 64 * 64 + 4096
    p, g_, m, v = (torch.randn(n, device=dev) * 0.02 for _ in range(4))
    v.abs_()
    pb = torch.empty(n, dtype=torch.bfloat16, device=dev)
    starts = torch.tensor([0, n // 8, n // 4], dtype=torch.int32, device=dev)
    flags = torch.tensor([0, 1, 0], dtype=torch.uint8, device=dev)
    ws = torch.empty(int(ops._lib.load().smbv_sumsq_workspace_floats()), device=dev)
    nsq = torch.zeros(1, device=dev)
    report("sumsq_97M", n * 4, lambda: call("smbv_sumsq_f32", ops._ptr(g_), n, ops._ptr(ws), ops._ptr(nsq), st))
    report("adamw_97M", n * 30, lambda: call("smbv_adamw_step", ops._ptr(p), ops._ptr(pb), ops._ptr(g_), ops._ptr(m), ops._ptr(v), n,
                                              ops._ptr(starts), ops._ptr(flags), 3, 5e-5, 0.9, 0.999, 1e-8, 0.01, 3, ops._ptr(nsq), 1.0, st))
    del p, g_, m, v, pb
    # input pipeline tail at 512x512x320
    for dt, nb in ((torch.int16, 2), (torch.float32, 4)):
        raw = (torch.randint(-1200, 1500, (512, 512, 320), device=dev).to(dt))
        out = torch.empty((320, 512, 512), device=dev)
        report(f"prepare_volume_{'i16' if nb == 2 else 'f32'}", raw.numel() * (nb + 4),
               lambda: ops.prepare_volume(raw, 512, 512, 320, -1000.0, 1000.0, 0.0, 1.0, True, out=out))
    # ragged: pad + crop (530 x 470 x 350 -> 512 x 512 x 320)
    raw = torch.randint(-1200, 1500, (530, 470, 350), device=dev).to(torch.int16)
    report("prepare_volume_i16_padcrop", 512 * 470 * 320 * 2 + 512 * 512 * 320 * 4,
           lambda: ops.prepare_volume(raw, 512, 512, 320, -1000.0, 1000.0, 0.0, 1.0, True, out=out))
    # classification head neighbours at BASELINE configs[3] size: batch 4, 224x224x160 -> 1960 tokens, d 768
    X = torch.randn(4, 1960, 768, device=dev)
    report("token_sum_b4_n1960", X.numel() * 4, lambda: ops.token_sum(X))
    gp = torch.randn(4, 768, device=dev)
    report("broadcast_rows_b4_n1960", X.numel() * 6, lambda: ops.broadcast_rows(gp, 1960))
    X = torch.randn(1, 20480, 768, device=dev)
    report("token_sum_n20480", X.numel() * 4, lambda: ops.token_sum(X))
    W, bias = torch.randn(3, 770, device=dev), torch.randn(3, device=dev)
    pooled, feats, labels = torch.randn(4, 768, device=dev), torch.randn(4, 2, device=dev), torch.tensor([0, 1, 2, 1], device=dev)
    gam, bet = torch.ones(768, device=dev), torch.zeros(768, device=dev)
    grads = dict(dW=torch.zeros_like(W), dbias=torch.zeros_like(bias), dgamma=torch.zeros(768, device=dev), dbeta=torch.zeros(768, device=dev))
    ms = timeit(lambda: ops.cls_head(pooled, 1 / 1960, gam, bet, 1e-5, feats, W, bias, labels, 2, grads), iters=50)
    rec("cls_head_fwd_bwd_b4", True, us=round(ms * 1e3, 2))


def g_vjepa():
    """HBM-bound kernels of the V-JEPA step (SURVEY.md §8f rank 4) at ViT-L / 512x512x320 sizes: achieved GB/s against
    MEASURED_PEAKS.json.  (Added at the end of round 1 after the GPU budget was spent: first thing to run in round 2.)"""
    import torch
    from smb_vision_b200 import ops
    dev = "cuda"
    peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"] if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0

    def report(name, nbytes, fn, iters=20):
        ms = timeit(fn, iters=iters)
        gbs = nbytes / ms / 1e6
        rec(name, True, ms=round(ms, 4), gbs=round(gbs, 1), frac_of_hbm_peak=round(gbs / peak, 3), algorithmic_mb=round(nbytes / 1e6, 1))

    qk = torch.randn(2, 1, 16, 20480, 64, device=dev).bfloat16()  # Q and K of 16 heads x 20480 tokens
    report("rope3d_vitl_n20480", qk.numel() * 2 * 2 * 60 // 64, lambda: ops.rope3d_(qk, 32, max_pos=32))  # the 4-element tail is not touched
    report("rope3d_transpose_vitl_n20480", qk.numel() * 2 * 2 * 60 // 64, lambda: ops.rope3d_(qk, 32, max_pos=32, transpose=True))
    seq = torch.randn(1, 20480, 1024, device=dev)
    idx = torch.randperm(20480, device=dev)[:12288].sort().values.int()[None].contiguous()
    report("gather_rows_12288_of_20480x1024", 12288 * 1024 * 8, lambda: ops.gather_rows(seq, idx))
    p, t = torch.randn(1, 12288, 1024, device=dev), torch.randn(1, 12288, 1024, device=dev)
    report("l1_loss_12288x1024", p.numel() * 8, lambda: ops.l1_loss(p, t))
    report("l1_loss_with_grad_12288x1024", p.numel() * 12, lambda: ops.l1_loss(p, t, want_grad=True))


GROUPS = {"vjepa": g_vjepa, "neighbours": g_neighbours, "bwd_gemm": g_bwd_gemm, "attn_bwd": g_attn_bwd, "bandwidth": g_bandwidth, "gemm": g_gemm, "attn": g_attn, "attn_big": g_attn_big, "patch": g_patch}


def run_group(name):
    import torch
    assert torch.cuda.is_available(), "no GPU"
    try:
        GROUPS[name]()
        torch.cuda.synchronize()
    except Exception as e:  # noqa
        rec(f"{name}_exception", False, error=repr(e)[:800], tb=traceback.format_exc()[-1500:])
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, f"gpu_check_{name}.json"), "w") as f:
        json.dump(RESULTS, f, indent=1, default=str)


def main():
    args = sys.argv[1:] or ["all"]
    if args[0] == "--group":
        run_group(args[1])
        return
    names = list(GROUPS) if args == ["all"] else args
    os.makedirs(OUT, exist_ok=True)
    summary = {}
    for n in names:
        t0 = time.time()
        try:
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--group", n], timeout=420, capture_output=True, text=True)
            rc, tail = p.returncode, (p.stdout[-6000:] + "\n--stderr--\n" + p.stderr[-3000:])
        except subprocess.TimeoutExpired as e:
            rc, tail = -999, "TIMEOUT " + str(e.stdout)[-2000:]
        print(f"===== group {n}: rc={rc} ({time.time() - t0:.1f}s)\n{tail}", flush=True)
        with open(os.path.join(OUT, f"gpu_check_{n}.log"), "w") as f:
            f.write(tail)
        try:
            res = json.load(open(os.path.join(OUT, f"gpu_check_{n}.json")))
        except Exception:
            res = []
        summary[n] = dict(rc=rc, n=len(res), failed=[r["name"] for r in res if not r["ok"]])
    with open(os.path.join(OUT, "gpu_check_summary.json"), "w") as f:
        json.dump(summary, f, indent=1)
    print("SUMMARY", json.dumps(summary))


if __name__ == "__main__":
    main()
