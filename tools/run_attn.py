"""Run the flash-attention kernel alone (for ncu).  usage: python tools/run_attn.py [H] [N] [iters]"""
import ctypes as C
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from smb_vision_b200 import _lib

H = int(sys.argv[1]) if len(sys.argv) > 1 else 12
N = int(sys.argv[2]) if len(sys.argv) > 2 else 20480
iters = int(sys.argv[3]) if len(sys.argv) > 3 else 3
torch.manual_seed(0)
q, k, v = (torch.randn(1, H, N, 64, device="cuda").to(torch.bfloat16) for _ in range(3))
o = torch.empty(1, N, H * 64, device="cuda", dtype=torch.bfloat16)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
for i in range(iters):
    if i == iters - 1:
        e0.record()
    _lib.call("smbv_flash_attn_fwd_ex", C.c_void_p(q.data_ptr()), C.c_void_p(k.data_ptr()), C.c_void_p(v.data_ptr()), 1, H, N, 0.125,
              C.c_void_p(o.data_ptr()), None, 0, None, 0, C.c_void_p(torch.cuda.current_stream().cuda_stream))
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1)
print(f"attn H={H} N={N}: {ms:.3f} ms, {4.0*N*N*64*H/ms/1e9:.1f} TFLOP/s")
