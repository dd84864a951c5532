"""Encoder-side (7168-token) and decoder-side GEMM shapes of the MIM training step vs torch.matmul (cuBLAS, no epilogue), forward / dgrad / wgrad.
usage: python tools/gemm_small_sweep.py [tag]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from smb_vision_b200 import ops
tag = sys.argv[1] if len(sys.argv) > 1 else ""
dev = "cuda"
torch.manual_seed(0)


def timeit(fn, n=50):
    for _ in range(5): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3  # us


rows = []
for M, d, m in [(7168, 768, 3072), (20480, 384, 1536)]:
    H = d // 64
    x = torch.randn(M, d, device=dev).bfloat16()
    h = torch.randn(M, m, device=dev).bfloat16()
    wqkv = (torch.randn(3 * d, d, device=dev) * 0.05).bfloat16()
    wo = (torch.randn(d, d, device=dev) * 0.05).bfloat16()
    w1 = (torch.randn(m, d, device=dev) * 0.05).bfloat16()
    w2 = (torch.randn(d, m, device=dev) * 0.05).bfloat16()
    b3, bd, bm = torch.randn(3 * d, device=dev), torch.randn(d, device=dev), torch.randn(m, device=dev)
    res = torch.zeros(M, d, device=dev)
    pre = torch.empty(M, m, device=dev, dtype=torch.bfloat16)
    f = torch.empty(M, m, device=dev, dtype=torch.bfloat16)
    dw1 = torch.zeros(m, d, device=dev)
    dw2 = torch.zeros(d, m, device=dev)
    dwo = torch.zeros(d, d, device=dev)
    cases = [
        ("qkv fwd", lambda: ops.gemm(x, wqkv, b3, ops.EPI_QKV_HEADS, heads=H, tokens=M), lambda: x @ wqkv.t(), 2 * M * 3 * d * d),
        ("out-proj fwd (resid)", lambda: ops.gemm(x, wo, bd, ops.EPI_RESID_F32, residual=res), lambda: x @ wo.t(), 2 * M * d * d),
        ("fc1 fwd (gelu+pre)", lambda: ops.gemm_ex(x, w1, M, m, d, ops.EPI_GELU_BF16, f, bias=bm, aux=pre), lambda: x @ w1.t(), 2 * M * m * d),
        ("fc2 fwd (resid)", lambda: ops.gemm(h, w2, bd, ops.EPI_RESID_F32, residual=res), lambda: h @ w2.t(), 2 * M * m * d),
        ("fc2 dgrad (dgelu)", lambda: ops.linear_dgrad(x, w2, aux=pre), lambda: x @ w2, 2 * M * m * d),
        ("fc1 dgrad", lambda: ops.linear_dgrad(h, w1), lambda: h @ w1, 2 * M * m * d),
        ("out-proj dgrad", lambda: ops.linear_dgrad(x, wo), lambda: x @ wo, 2 * M * d * d),
        ("fc2 wgrad", lambda: ops.linear_wgrad(x, h, dw2), lambda: x.t() @ h, 2 * M * m * d),
        ("fc1 wgrad", lambda: ops.linear_wgrad(h, x, dw1), lambda: h.t() @ x, 2 * M * m * d),
        ("out-proj wgrad", lambda: ops.linear_wgrad(x, x, dwo), lambda: x.t() @ x, 2 * M * d * d),
    ]
    for name, ours, ref, fl in cases:
        t, tr = timeit(ours), timeit(ref)
        rows.append((M, d, name, t, tr, fl / t / 1e6, fl / tr / 1e6))
print(tag)
tot = tot_r = 0
for M, d, name, t, tr, tf, tfr in rows:
    print(f"M={M:5d} d={d:3d} {name:24s} ours {t:7.1f} us ({tf:6.0f} TF/s) | torch.matmul {tr:7.1f} us ({tfr:6.0f} TF/s) | ratio {t / tr:.2f}")
    layers = 12 if M == 7168 else 4
    tot += t * layers; tot_r += tr * layers
print(f"sum over layers (12 encoder, 4 decoder): ours {tot / 1e3:.2f} ms, torch.matmul {tot_r / 1e3:.2f} ms")
