"""Forward GEMMs with their fused epilogues at the model shapes: parity vs fp32 torch + CUDA-event timings next to torch.matmul
(cuBLAS, no epilogue).
usage: python tools/gemm_ab.py [tag]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from smb_vision_b200 import ops
tag = sys.argv[1] if len(sys.argv) > 1 else ""
dev = "cuda"
torch.manual_seed(0)
def timeit(fn, iters=20, warmup=5):
    for _ in range(warmup): fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters
def frob(a, b): return ((a.float() - b.float()).norm() / b.float().norm()).item()
for M, N, K, epi in [(20480, 768, 768, "resid"), (20480, 768, 3072, "resid"), (7168, 768, 768, "resid"), (7168, 768, 3072, "resid"),
                     (20480, 384, 384, "resid"), (20480, 384, 1536, "resid"), (20000, 768, 776, "resid"),
                     (20480, 3072, 768, "gelu"), (7168, 3072, 768, "gelu"), (20480, 1536, 384, "gelu"), (20480, 2304, 768, "bf16")]:
    a, w, bias = (torch.randn(M, K, device=dev)).bfloat16(), (torch.randn(N, K, device=dev) * 0.05).bfloat16(), torch.randn(N, device=dev)
    ref = a.float() @ w.float().t() + bias
    if epi == "resid":
        res = torch.randn(M, N, device=dev)
        x = res.clone(); ops.gemm(a, w, bias, ops.EPI_RESID_F32, residual=x); got = x; ref = ref + res
        fn = lambda: ops.gemm(a, w, bias, ops.EPI_RESID_F32, residual=x)
    elif epi == "gelu":
        got = ops.gemm(a, w, bias, ops.EPI_GELU_BF16); ref = torch.nn.functional.gelu(ref)
        fn = lambda: ops.gemm(a, w, bias, ops.EPI_GELU_BF16)
    else:
        got = ops.gemm(a, w, bias, ops.EPI_BF16)
        fn = lambda: ops.gemm(a, w, bias, ops.EPI_BF16)
    torch.cuda.synchronize()
    err = frob(got, ref)
    ms = timeit(fn)
    tm = timeit(lambda: torch.matmul(a, w.t()))
    print(tag, f"M{M} N{N} K{K} {epi}: err {err:.2e}  {ms*1e3:.1f} us = {2.0*M*N*K/ms/1e9:.0f} TF/s   (torch.matmul {tm*1e3:.1f} us = {2.0*M*N*K/tm/1e9:.0f})", flush=True)
