"""ctypes binding of the C-ABI library ``lib/libsmbv_b200.so`` (declared in ``include/smbv_b200.h``).

The product path has no CPU or PyTorch fallback: if the library is missing or a call fails, a
:class:`SmbvError` is raised.  Build it with ``make`` or ``python -c 'import __graft_entry__ as g; g.build()'``.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SMBV_LIB") or os.path.join(_HERE, "lib", "libsmbv_b200.so")  # SMBV_LIB: developer A/B of two builds

# epilogue ids (include/smbv_b200.h)
EPI_BF16, EPI_GELU_BF16, EPI_RESID_F32, EPI_QKV_HEADS, EPI_F32, EPI_POS_GATHER_F32 = range(6)


class SmbvError(RuntimeError):
    pass


class GemmArgs(C.Structure):
    _fields_ = [
        ("A", C.c_void_p), ("lda", C.c_int64),
        ("W", C.c_void_p), ("ldw", C.c_int64),
        ("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32),
        ("bias", C.c_void_p),
        ("epilogue", C.c_int32),
        ("out", C.c_void_p), ("ldo", C.c_int64),
        ("residual", C.c_void_p),
        ("heads", C.c_int32), ("tokens", C.c_int32),
        ("pos", C.c_void_p), ("ldpos", C.c_int64),
        ("row_map", C.c_void_p),
    ]


class GemmExArgs(C.Structure):
    _fields_ = [
        ("A", C.c_void_p), ("lda", C.c_int64), ("a_layout", C.c_int32), ("a_part_stride", C.c_int64),
        ("W", C.c_void_p), ("ldw", C.c_int64), ("w_layout", C.c_int32),
        ("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32), ("heads", C.c_int32), ("split_k", C.c_int32),
        ("bias", C.c_void_p), ("alpha", C.c_void_p),
        ("epilogue", C.c_int32),
        ("out", C.c_void_p), ("ldo", C.c_int64),
        ("residual", C.c_void_p),
        ("aux", C.c_void_p),
    ]


A_ROWMAJOR, A_TRANSPOSED, A_HEADS, A_HEADS_T = range(4)
CLS_NONE, CLS_REGRESSION, CLS_SINGLE_LABEL, CLS_MULTI_LABEL = range(4)
EPI_ATOMIC_F32, EPI_DGELU_BF16 = 6, 7

_P, _I, _F, _L = C.c_void_p, C.c_int, C.c_float, C.c_int64
# name -> argtypes; every symbol include/smbv_b200.h declares (tests/test_cabi.py checks the two lists agree)
SIGNATURES = {
    "smbv_version": [],
    "smbv_sm_arch": [],
    "smbv_device_ok": [],
    "smbv_mask_upsample": [_P, _P, _I, _I, _I, _I, _I, _P],
    "smbv_mask_index": [_P, _I, _I, _P, _P, _P, _P, _P],
    "smbv_sincos_table": [_P, _I, _I, _P],
    "smbv_patch_embed_fwd": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P],
    "smbv_patch_embed_select_fwd": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _P],
    "smbv_layernorm_fwd": [_P, _P, _P, _F, _I, _I, _P, _P, _P, _P],
    "smbv_layernorm_fwd_copy": [_P, _P, _P, _F, _I, _I, _P, _P, _P, _P, _P],
    "smbv_gemm_bf16": [C.POINTER(GemmArgs), _P],
    "smbv_gemm_ex": [C.POINTER(GemmExArgs), _P],
    "smbv_flash_attn_bwd": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _F, _P, _P, _P, _P, _P],
    "smbv_flash_attn_bwd_ex": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _F, _P, _P, _P, _P, _P, _P, _P],
    "smbv_flash_attn_bwd_fused": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _F, _P, _P, _L, _P, _P, _P, _P, _P, _P],
    "smbv_layernorm_bwd": [_P, _P, _P, _P, _P, _I, _I, _P, _I, _P, _P, _P, _P, _P],
    "smbv_layernorm_bwd_blocks": [],
    "smbv_layernorm_bwd_add": [_P, _P, _P, _P, _P, _I, _I, _P, _I, _P, _P, _P, _P, _P],
    "smbv_colsum_bf16": [_P, _I, _I, _L, _P, _P],
    "smbv_colsum_f32": [_P, _I, _I, _L, _P, _P],
    "smbv_colsum_heads_bf16": [_P, _I, _I, _I, _P, _I, _P],
    "smbv_gather_patches_bf16": [_P, _I, _I, _I, _I, _I, _P, _I, _I, _P, _P],
    "smbv_flash_attn_fwd": [_P, _P, _P, _I, _I, _I, _F, _P, _P, _P],
    "smbv_flash_attn_fwd_ex": [_P, _P, _P, _I, _I, _I, _F, _P, _P, _I, _P, _L, _P],
    "smbv_flash_attn_fwd_workspace_bytes": [_I, _I, _I],
    "smbv_flash_attn_bwd_fused_workspace_bytes": [_I, _I, _I],
    "smbv_attn_small_fwd": [_P, _P, _P, _L, _L, _L, _I, _I, _I, _I, _F, _P, _P, _P],
    "smbv_attn_small_bwd": [_P, _P, _P, _L, _L, _L, _P, _P, _P, _I, _I, _I, _I, _F, _P, _P, _P, _P, _L, _L, _L, _P],
    "smbv_fill_mask_tokens": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    "smbv_normpix_loss": [_P, _I, _I, _I, _I, _I, _P, _I, _I, _P, _P, _P, _P, _I, _P],
    "smbv_cls_head": [_P, _F, _P, _P, _F, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P],
    "smbv_broadcast_rows": [_P, _I, _I, _I, _P, _P, _P],
    "smbv_token_sum_chunks": [_I],
    "smbv_token_sum": [_P, _I, _I, _I, _P, _P, _P],
    "smbv_prepare_volume": [_P, _I, _I, _I, _I, _F, _F, _F, _F, _I, _I, _I, _I, _P, _P],
    "smbv_sumsq_workspace_floats": [],
    "smbv_sumsq_f32": [_P, _L, _P, _P, _P],
    "smbv_scale_f32": [_P, _L, _P, _P],
    "smbv_adamw_step": [_P, _P, _P, _P, _P, _L, _P, _P, _I, _F, _F, _F, _F, _F, _I, _P, _F, _P],
    "smbv_ema_update": [_P, _P, _L, _F, _F, _P],
    "smbv_rope3d": [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P],
    "smbv_gather_rows_f32": [_P, _P, _I, _I, _I, _I, _P, _P],
    "smbv_scatter_rows_f32": [_P, _P, _I, _I, _I, _I, _I, _P, _P],
    "smbv_heads32_convert": [_P, _P, _L, _I, _I, _I, _I, _P],
    "smbv_position_sort": [_P, _I, _I, _P, _P, _P, _P, _P],
    "smbv_l1_workspace_floats": [],
    "smbv_l1_loss_f32": [_P, _P, _L, _P, _P, _P, _F, _P],
    "smbv_cast_f32_bf16": [_P, _P, _L, _P],
    "smbv_cast_bf16_f32_scale": [_P, _P, _L, _F, _P],
    "smbv_scale_add_recast_f32": [_P, _L, _P, _P, _P, _P],
}

_lib = None


def load() -> C.CDLL:
    """Load the library once; raise loudly if it is not built (no fallback path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SmbvError(
            f"{LIB_PATH} is missing: the sm_100a CUDA extension is not built. Run `make` at the repo root "
            "(or __graft_entry__.build()). smb_vision_b200 has no CPU/PyTorch fallback."
        )
    lib = C.CDLL(LIB_PATH)
    lib.smbv_last_error.restype = C.c_char_p
    lib.smbv_last_error.argtypes = []
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = C.c_int64 if name.endswith("_workspace_bytes") else C.c_int
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().smbv_last_error().decode(errors="replace")
        kind = "argument error" if rc < 0 else f"CUDA error {rc}"
        raise SmbvError(f"{what}: {kind}: {msg}")


# kernels launched per C-ABI call (for bench.py's gpu_launches count)
LAUNCHES_PER_CALL = {"smbv_normpix_loss": 2, "smbv_layernorm_bwd": 2, "smbv_layernorm_bwd_add": 2, "smbv_flash_attn_bwd": 3, "smbv_flash_attn_bwd_ex": 3, "smbv_flash_attn_bwd_fused": 4, "smbv_sumsq_f32": 2, "smbv_l1_loss_f32": 2, "smbv_token_sum": 2, "smbv_attn_small_bwd": 2}
launch_count = 0
# optional hook(name) -> context manager, used by bench.py to bracket one kernel family with CUDA events
event_hook = None


def call(name: str, *args) -> None:
    global launch_count
    launch_count += LAUNCHES_PER_CALL.get(name, 1)
    if event_hook is not None:
        with event_hook(name):
            check(getattr(load(), name)(*args), name)
    else:
        check(getattr(load(), name)(*args), name)
