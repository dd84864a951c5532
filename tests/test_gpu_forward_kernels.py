"""Kernel-level parity of the FORWARD pass (run with -m gpu on the B200 box): every epilogue and dispatch path of the forward
GEMM (`gemm.cu`), the implicit-GEMM patch embedding (`patch_embed.cu`), LayerNorm forward, the three norm-pix loss kernels,
the decoder's mask-token fill and the fp32 -> bf16 weight cast (`bandwidth.cu`).  The model-level tests allow whole-tensor
Frobenius norms of 3e-3 .. 5e-3 against fp32; one k-block missing from one 128x256 tile of the fc1 GEMM moves such a norm
by less than that.  Here each kernel is compared on its own with a float64 reference computed ON THE DEVICE from the exact
operands it reads (bf16-rounded A, W and volume; fp32 bias, position table and residual), per tile and per element.  Every
output the kernel overwrites is a NaN-prefilled view between guard regions that must come back untouched.

Bounds (the worst value measured on one NVIDIA B200 at a 1000 W power limit in brackets):
  GEMM fp32 outputs (F32, RESID_F32, POS_GATHER_F32): Frobenius-rel <= 2e-5 [3.1e-6], max-abs-rel <= 1e-4 [3.5e-6], worst
      128x128 tile <= 2e-5 [3.2e-6] (the bounds of tests/test_gpu_backward_kernels.py; the worst case is K = 4096);
  GEMM bf16 outputs (BF16, GELU, saved pre-activation, QKV_HEADS, DGELU): every element within 1 bf16 ulp of the fp64
      value, plus 1e-5 of the output's max as floor [0.50 ulp];
  GELU / dGELU epilogue math over every finite bf16 input (W = I): within 1 ulp of the bf16 rounding of the fp64 GELU /
      GELU' plus an absolute floor of 1e-6 [GELU 0.79, GELU' 0.19; with a bias, off the bf16 grid: <= 1 ulp]; beyond the
      output rounding the GELU is off by at most 5.2e-7, GELU' by 1.5e-8; the saved pre-activation equals the input in
      value (-0 comes back as +0: the accumulator adds signed zeros);
  patch embedding: the fp32 GEMM bounds [Frobenius 4.4e-6, max-abs-rel 5.7e-6, tile 4.6e-6] over 4096-long dot products;
  LayerNorm: mean within MEAN_ULPS = 4 fp32 ulps of the row's rms [1.08], rstd within RSTD_ULPS = 4 fp32 ulps of the
      two-pass value for the kernel's own mean [1.33], y within 1 bf16 ulp (+ 1e-5 of the max) of the fp64 result for
      those statistics [0.50];
  norm-pix loss: loss relative error <= LOSS_REL = 1e-5 [1.2e-6]; MSE dlogits within 1 bf16 ulp + 2/count * LABEL_TOL of
      the fp64 gradient [0.50]; L1 dlogits exactly sign(d) / count wherever |d| > LABEL_TOL [no exception].  The warp,
      block and generic kernels sum the patch statistics in different orders, so their labels differ in the last fp32
      bits: their losses agree within REPRO_LOSS = 2e-6 [3.9e-7], their MSE dlogits within 1 bf16 ulp (at most 2682 elements
      differ in one call), their L1 dlogits wherever |d| > LABEL_TOL;
  mask-token fill and cast: bit-exact.
Every family runs a negative control: the comparison against a deliberately wrong reference must fail its local bound by
>= 100x [measured margin over the bound in brackets]: one k-block of one tile dropped (GEMM) [4.4e3x], two heads of one
sample swapped (QKV) [4.4e4x], identity row_map in one row (POS_GATHER) [3.8e4x], one dz plane of one tile dropped (patch
embedding) [8.3e3x], one-pass variance (LayerNorm rstd) [7.3e7x], biased variance (norm-pix loss, logits = bf16(label))
[167x L1, 497x MSE].

Reproducibility (README, "Determinism"): no forward kernel here has a cross-CTA reduction; each output is checked
bit-identical on a second call.
"""
import math
import re
import types

import pytest
import torch
import torch.nn.functional as F

from oracle import videomae_oracle as vo

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

F32_FROB, F32_MAX, F32_LOCAL = 2e-5, 1e-4, 2e-5
BF16_ULPS = 1.0
GELU_FLOOR = 1e-6  # absolute floor of the exhaustive GELU / GELU' check (GELU(-7) ~ -7e-12 comes out as -0)
MEAN_ULPS, RSTD_ULPS = 4.0, 4.0
LOSS_REL = 1e-5
LABEL_TOL = 4e-6  # absolute error of a normalised fp32 label
REPRO_LOSS = 2e-6  # relative loss difference between the norm-pix kernels (fp32 summation order)
CONTROL = 100.0
GUARD, SENTINEL = 256, 7.0


@pytest.fixture(scope="module")
def ops():
    assert torch.cuda.is_available()
    from smb_vision_b200 import load, ops as _ops

    lib = load()
    assert lib.smbv_device_ok() == 0, lib.smbv_last_error()
    return _ops


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def frob(a, b):
    a, b = a.double(), b.double()
    return (torch.linalg.norm(a - b) / torch.linalg.norm(b)).item()


def maxrel(a, b):
    a, b = a.double(), b.double()
    return ((a - b).abs().max() / b.abs().max()).item()


def tile_frob(a, b, tr=128, tc=128):
    """worst Frobenius-rel over the [tr x tc] tiles of a 2-D output (tr=1, tc=width: worst row)."""
    a, b = a.double(), b.double()
    R, C = b.shape
    pad = (0, (-C) % tc, 0, (-R) % tr)
    e, r = F.pad((a - b) ** 2, pad), F.pad(b ** 2, pad)
    shape = (e.shape[0] // tr, tr, e.shape[1] // tc, tc)
    e, r = e.view(shape).sum((1, 3)), r.view(shape).sum((1, 3))
    return (e.sqrt() / r.sqrt().clamp_min(1e-300)).max().item()


def ulp_bf16(ref):
    ref = ref.double()
    return torch.exp2(torch.floor(torch.log2(ref.abs())) - 7)  # 8 significant bits; 0 at ref == 0


def bf16_ulps(got, ref, floor=None):
    """max over elements of |got - ref| / (1 bf16 ulp of ref + floor); floor defaults to 1e-5 max|ref|."""
    ref = ref.double()
    floor = 1e-5 * ref.abs().max() if floor is None else floor
    return ((got.double() - ref).abs() / (ulp_bf16(ref) + floor)).max().item()


def check_f32(got, ref, worst, local=None):
    assert torch.isfinite(got).all()
    f, m = frob(got, ref), maxrel(got, ref)
    loc = tile_frob(got, ref) if local is None else local(got, ref)
    worst["frob"], worst["maxrel"], worst["local"] = max(worst.get("frob", 0), f), max(worst.get("maxrel", 0), m), max(worst.get("local", 0), loc)
    assert f <= F32_FROB and m <= F32_MAX and loc <= F32_LOCAL, (f, m, loc)


def check_bf16(got, ref, worst, key="ulps", floor=None):
    assert torch.isfinite(got.float()).all()
    u = bf16_ulps(got, ref, floor)
    worst[key] = max(worst.get(key, 0), u)
    assert u <= BF16_ULPS, (key, u)


def report(name, worst, bounds):
    print(f"{name}: " + ", ".join(f"{k} {worst[k]:.2e} (bound {bounds[k]:.0e})" for k in bounds if k in worst))


def rnd(shape, g, dtype=torch.bfloat16, scale=1.0, shift=0.0):
    return (torch.randn(shape, device=DEV, generator=g) * scale + shift).to(dtype)


def guarded(shape, dtype=torch.float32):
    """(buffer, view): a NaN-prefilled view between two guard regions of SENTINEL (16-byte aligned)."""
    n = math.prod(shape)
    buf = torch.full((n + 2 * GUARD,), float("nan"), dtype=dtype, device=DEV)
    buf[:GUARD] = SENTINEL
    buf[GUARD + n:] = SENTINEL
    return buf, buf[GUARD:GUARD + n].view(shape)


def guards_ok(buf):
    return bool((buf[:GUARD] == SENTINEL).all() and (buf[-GUARD:] == SENTINEL).all())


def gelu64(z):
    return 0.5 * z * (1 + torch.special.erf(z / math.sqrt(2)))


def dgelu64(z):
    return 0.5 * (1 + torch.special.erf(z / math.sqrt(2))) + z * torch.exp(-0.5 * z * z) / math.sqrt(2 * math.pi)


# =====================================================================================================================
# 1. dispatch replica of the forward GEMM (gemm.cu: dispatch_gemm, use_tma_epilogue)
# =====================================================================================================================
def gemm_plan(kind, M, N, K, tokens=0, sms=148):
    """what `dispatch_gemm` launches for one call form: template arguments <BN, A_MN, B_MN, A3D, TMA_EPI, EPI4>, the tile
    count, the grid and the most tiles one CTA runs."""
    tiles256 = -(-M // 128) * -(-N // 256)
    bn = 256 if N % 256 == 0 and tiles256 >= 2 * sms else 128
    tma = kind in ("bf16", "f32", "gelu", "gelu_pre", "dgelu", "resid_in") or (kind == "qkv" and tokens % 128 == 0)
    epi4 = kind == "dgelu" or (kind == "gelu_pre" and K <= 512)
    tiles = -(-M // 128) * -(-N // bn)
    grid = min(tiles, sms)
    return dict(targs=(bn, False, kind == "dgelu", False, tma, epi4), bn=bn, tma=tma, epi4=epi4, tiles=tiles, grid=grid,
                per_cta=-(-tiles // grid))


# (name, kind, M, N, K, extra).  Model shapes: encoder 768 / 3072 / 2304, decoder 384 / 1536 / 1152, decoder head 4096,
# V-JEPA ViT-L 1024 / 4096 / 3072, at 1960 x 4 (classification), 7168 (visible), 13312 (masked) and 20480 tokens.
# qkv: extra = (batch, heads); pos: extra = rows of the position table; dgelu: (M, N, K) of the GEMM, K = fc2 output.
GEMM_CASES = [
    ("enc-qkv-20480", "qkv", 20480, 2304, 768, (1, 12)),
    ("enc-oproj-20480", "resid_in", 20480, 768, 768, None),
    ("enc-fc1-20480", "gelu_pre", 20480, 3072, 768, None),
    ("enc-fc2-20480", "resid_in", 20480, 768, 3072, None),
    ("enc-fc1-7168-infer", "gelu", 7168, 3072, 768, None),
    ("enc-qkv-7840-b4", "qkv", 7840, 2304, 768, (4, 12)),
    ("enc-fc1-7840-infer", "gelu", 7840, 3072, 768, None),
    ("enc-oproj-7840-outofplace", "resid_out", 7840, 768, 768, None),
    ("dec-qkv-20480", "qkv", 20480, 1152, 384, (1, 6)),
    ("dec-fc1-20480", "gelu_pre", 20480, 1536, 384, None),
    ("dec-fc2-20480", "resid_in", 20480, 384, 1536, None),
    ("dec-head-13312", "bf16", 13312, 4096, 384, None),
    ("dec-embed-7168", "pos", 7168, 384, 768, 20480),
    ("dec-f32-7168", "f32", 7168, 384, 768, None),
    ("vjepa-qkv-7840-b4", "qkv", 7840, 3072, 1024, (4, 16)),
    ("vjepa-qkv-7168-b2", "qkv", 7168, 3072, 1024, (2, 16)),
    ("vjepa-fc1-7840", "gelu_pre", 7840, 4096, 1024, None),
    ("vjepa-fc2-7840", "resid_in", 7840, 1024, 4096, None),
    ("fc2-dgelu-7168", "dgelu", 7168, 3072, 768, None),
    ("dec-fc2-dgelu-20480", "dgelu", 20480, 1536, 384, None),
    ("dgelu-1000", "dgelu", 1000, 3072, 768, None),
    ("dgelu-n160", "dgelu", 300, 160, 96, None),
    ("gelu-pre-epi4-1000", "gelu_pre", 1000, 1536, 384, None),
    ("gelu-pre-1000", "gelu_pre", 1000, 3072, 768, None),
    ("gelu-pre-n160", "gelu_pre", 130, 160, 640, None),
    ("f32-n96", "f32", 300, 96, 32, None),
    ("bf16-n160", "bf16", 300, 160, 64, None),
    ("bf16-n800", "bf16", 1000, 800, 256, None),
    ("resid-in-n160", "resid_in", 300, 160, 64, None),
    ("resid-out-1000", "resid_out", 1000, 768, 768, None),
    ("qkv-reg-216-b2", "qkv", 432, 384, 128, (2, 2)),
    ("qkv-tma-256-b2", "qkv", 512, 384, 128, (2, 2)),
    ("qkv-tma-128-b4", "qkv", 512, 192, 64, (4, 1)),
    ("qkv-reg-1000-b4", "qkv", 4000, 1152, 384, (4, 6)),
    ("qkv-tma-1024-b2", "qkv", 2048, 1152, 384, (2, 6)),
    ("pos-small", "pos", 100, 96, 64, 300),
]
CASE_IDS = [c[0] for c in GEMM_CASES]

REQUIRED = {"BF16", "F32", "GELU", "GELU+pre", "RESID in place", "RESID out of place", "QKV TMA", "QKV register",
            "POS_GATHER", "DGELU", "TMA BN128", "TMA BN256", "GELU+pre EPI4 BN128", "GELU+pre EPI4 BN256",
            "GELU+pre BN128", "GELU+pre BN256", "DGELU BN128", "DGELU BN256", "ragged M", "N%64==32", "N%BN!=0",
            "1 tile/CTA", "2 tiles/CTA", ">=3 tiles/CTA", "partial last wave", "QKV batch>1 TMA", "QKV batch>1 register"}
MODE_TAG = {"bf16": "BF16", "f32": "F32", "gelu": "GELU", "gelu_pre": "GELU+pre", "resid_in": "RESID in place",
            "resid_out": "RESID out of place", "pos": "POS_GATHER", "dgelu": "DGELU"}


def plan_tags(kind, M, N, K, extra, p):
    tags = {MODE_TAG.get(kind) or ("QKV TMA" if p["tma"] else "QKV register")}
    if kind == "qkv" and extra[0] > 1:
        tags.add("QKV batch>1 " + ("TMA" if p["tma"] else "register"))
    if p["tma"]:
        tags.add(f"TMA BN{p['bn']}")
    if kind == "gelu_pre":
        tags.add(f"GELU+pre {'EPI4 ' if p['epi4'] else ''}BN{p['bn']}")
    if kind == "dgelu":
        tags.add(f"DGELU BN{p['bn']}")
    if M % 128:
        tags.add("ragged M")
    if N % 64 == 32:
        tags.add("N%64==32")
    if N % p["bn"]:
        tags.add("N%BN!=0")
    tags.add({1: "1 tile/CTA", 2: "2 tiles/CTA"}.get(p["per_cta"], ">=3 tiles/CTA"))
    if p["tiles"] > p["grid"] and p["tiles"] % p["grid"]:
        tags.add("partial last wave")
    return tags


def make_case(case, seed):
    """inputs of one GEMM case (bf16 operands at realistic scales, fp32 side inputs)."""
    name, kind, M, N, K, extra = case
    g = torch.Generator(device=DEV).manual_seed(seed)
    c = dict(g=g)
    if kind == "dgelu":  # dX[M,N] = (dY[M,K] W2[K,N]) * gelu'(pre[M,N]); W2 is the fc2 weight [K, N]
        c["a"], c["w"] = rnd((M, K), g), rnd((K, N), g, scale=0.05)
        c["pre"] = rnd((M, N), g, scale=1.5)
        return c
    c["a"], c["w"] = rnd((M, K), g), rnd((N, K), g, scale=0.05)
    c["bias"] = torch.randn(N, device=DEV, generator=g)
    if kind in ("resid_in", "resid_out"):
        c["res"] = torch.randn(M, N, device=DEV, generator=g) * 3
    if kind == "pos":
        rows = extra
        c["pos"] = torch.randn(rows, N, device=DEV, generator=g)
        c["vis"] = torch.stack([torch.randperm(rows, device=DEV, generator=g) for _ in range(2)]).to(torch.int32)  # [2, rows]
        c["bias"] = None if M >= 1000 else c["bias"]  # the decoder embedding has no bias; the small case has one
    return c


def run_case(ops, case, c):
    """one call in the model's call form; returns {output name: (view, guarded buffer)}."""
    name, kind, M, N, K, extra = case
    a, w = c["a"], c["w"]
    if kind in ("bf16", "gelu"):
        buf, out = guarded((M, N), torch.bfloat16)
        ops.gemm(a, w, c["bias"], ops.EPI_BF16 if kind == "bf16" else ops.EPI_GELU_BF16, out=out)
        return {"out": (out, buf)}
    if kind == "f32":
        buf, out = guarded((M, N))
        ops.gemm(a, w, c["bias"], ops.EPI_F32, out=out)
        return {"out": (out, buf)}
    if kind == "gelu_pre":
        buf, out = guarded((M, N), torch.bfloat16)
        pbuf, pre = guarded((M, N), torch.bfloat16)
        ops.gemm_ex(a, w, M, N, K, ops.EPI_GELU_BF16, out, bias=c["bias"], aux=pre)
        return {"out": (out, buf), "pre": (pre, pbuf)}
    if kind == "resid_in":
        buf, x = guarded((M, N))
        x.copy_(c["res"])
        ops.gemm(a, w, c["bias"], ops.EPI_RESID_F32, residual=x)
        return {"out": (x, buf)}
    if kind == "resid_out":
        buf, out = guarded((M, N))
        ops.gemm(a, w, c["bias"], ops.EPI_RESID_F32, out=out, residual=c["res"])
        return {"out": (out, buf)}
    if kind == "qkv":
        B, H = extra
        buf, out = guarded((3, B, H, M // B, 64), torch.bfloat16)
        ops.gemm(a, w, c["bias"], ops.EPI_QKV_HEADS, out=out, heads=H, tokens=M // B)
        return {"out": (out, buf)}
    if kind == "pos":  # as the decoder calls it: rows [0, M) of sample 1 of a [2, rows, N] buffer, row_map = a row of vis
        buf, xd = guarded((2, extra, N))
        ops.gemm(a, w, c["bias"], ops.EPI_POS_GATHER_F32, out=xd[1, :M], pos=c["pos"], row_map=c["vis"][1])
        return {"out": (xd[1, :M], buf), "rest": (xd[1, M:], None), "other": (xd[0], None)}
    if kind == "dgelu":
        buf, out = guarded((M, N), torch.bfloat16)
        ops.linear_dgrad(a, w, aux=c["pre"], out=out)
        return {"out": (out, buf)}
    raise AssertionError(kind)


def test_gemm_dispatch_replica_matches_the_launched_kernel(ops):
    """Each case runs once under torch.profiler (kernel activity only, nothing written): the launched
    gemm_bf16_kernel<BN, A_MN, B_MN, A3D, TMA_EPI, EPI4> must be the replica's prediction, and the case list must reach
    every REQUIRED path on this device's SM count."""
    sms = sm_count()
    reached, bad = set(), []
    print(f"\n{'case':28s} {'M':>6s} {'N':>5s} {'K':>5s}  predicted <BN,A_MN,B_MN,A3D,TMA,EPI4>  tiles grid /CTA  launched")
    for i, case in enumerate(GEMM_CASES):
        name, kind, M, N, K, extra = case
        p = gemm_plan(kind, M, N, K, tokens=M // extra[0] if kind == "qkv" else 0, sms=sms)
        c = make_case(case, i)
        run_case(ops, case, c)  # warm-up (first launches set kernel attributes)
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            run_case(ops, case, c)
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if "gemm_bf16_kernel" in e.name]
        launched = []
        for nm in names:
            args = [s.strip() for s in re.search(r"gemm_bf16_kernel<([^>]*)>", nm).group(1).split(",")]
            args = [int(args[0])] + [s == "true" for s in args[1:]] + [False] * (6 - len(args))
            launched.append(tuple(args))
        ok = launched == [p["targs"]]
        bad += [] if ok else [(name, p["targs"], launched)]
        tags = plan_tags(kind, M, N, K, extra, p)
        reached |= tags
        fmt = lambda t: "<" + ",".join(str(int(v)) if isinstance(v, bool) else str(v) for v in t) + ">"  # noqa: E731
        print(f"{name:28s} {M:6d} {N:5d} {K:5d}  {fmt(p['targs']):38s} {p['tiles']:5d} {p['grid']:4d} {p['per_cta']:4d}  "
              f"{' '.join(fmt(t) for t in launched)}{'' if ok else '  MISMATCH'}")
    print(f"REQUIRED paths reached: {len(REQUIRED & reached)}/{len(REQUIRED)}; missing: {sorted(REQUIRED - reached)}")
    assert not bad, bad
    assert REQUIRED <= reached, sorted(REQUIRED - reached)


# =====================================================================================================================
# 2. GEMM epilogue parity
# =====================================================================================================================
def tile_block(a, b, kb, r=slice(0, 128), c=slice(0, 128)):
    """contribution of k-block kb (64 along the contraction) of a[R,K] @ b[K,C] to the output tile [r, c], fp64."""
    ks = slice(64 * kb, 64 * kb + 64)
    return a[r, ks].double() @ b[ks, c].double()


@pytest.mark.parametrize("case", GEMM_CASES, ids=CASE_IDS)
def test_gemm_epilogue_matches_fp64(ops, case):
    name, kind, M, N, K, extra = case
    c = make_case(case, CASE_IDS.index(name))
    outs = run_case(ops, case, c)
    for v, buf in outs.values():
        assert buf is None or guards_ok(buf), "guard region overwritten"
    a, w = c["a"], c["w"]
    wt = w.double() if kind == "dgelu" else w.double().t()  # [K, N]
    acc = a.double() @ wt
    kb = ((K + 63) // 64) // 2
    blk = torch.zeros_like(acc)
    blk[:128, :128] = tile_block(a, wt, kb)  # negative control: this k-block missing from the first output tile
    bias = c.get("bias")
    z = acc + (bias.double() if bias is not None and kind != "dgelu" else 0)
    worst, got = {}, outs["out"][0]
    if kind in ("f32", "resid_in", "resid_out"):
        ref = z + (c["res"].double() if kind != "f32" else 0)
        check_f32(got, ref, worst)
        ctrl = tile_frob(got, ref - blk)
        bounds, cbound = dict(frob=F32_FROB, maxrel=F32_MAX, local=F32_LOCAL), CONTROL * F32_LOCAL
    elif kind == "pos":
        vis = c["vis"][1, :M].long()
        ref = z + c["pos"].double()[vis]
        check_f32(got, ref, worst)
        assert torch.isnan(outs["rest"][0]).all() and torch.isnan(outs["other"][0]).all(), "rows outside out= written"
        bad = ref.clone()
        r = M // 2
        bad[r] = z[r] + c["pos"].double()[r]  # negative control: identity row_map in one row
        ctrl = tile_frob(got, bad, 1, N)
        bounds, cbound = dict(frob=F32_FROB, maxrel=F32_MAX, local=F32_LOCAL), CONTROL * F32_LOCAL
    elif kind == "qkv":
        B, H = extra
        hm = lambda t: t.view(B, M // B, 3, H, 64).permute(2, 0, 3, 1, 4)  # noqa: E731  token-major -> [3,B,H,n,64]
        ref = hm(z)
        check_bf16(got, ref, worst)
        bad = ref.clone()
        if H > 1:  # negative control: heads 0 and 1 of the last sample swapped
            bad[:, B - 1, [0, 1]] = ref[:, B - 1, [1, 0]]
        else:  # one head: Q and K of the last sample swapped
            bad[[0, 1], B - 1] = ref[[1, 0], B - 1]
        ctrl = bf16_ulps(got, bad)
        bounds, cbound = dict(ulps=BF16_ULPS), CONTROL * BF16_ULPS
    else:
        if kind == "bf16":
            ref, badref = z, z - blk
        elif kind in ("gelu", "gelu_pre"):
            ref, badref = gelu64(z), gelu64(z - blk)
            if kind == "gelu_pre":
                check_bf16(outs["pre"][0], z, worst, key="pre ulps")
        else:  # dgelu
            gp = dgelu64(c["pre"].double())
            ref, badref = acc * gp, (acc - blk) * gp
        check_bf16(got, ref, worst)
        ctrl = bf16_ulps(got, badref)
        bounds, cbound = dict(ulps=BF16_ULPS), CONTROL * BF16_ULPS
        if kind == "gelu_pre":
            bounds["pre ulps"] = BF16_ULPS
    # reproducibility: a second call is bit-identical (no cross-CTA reduction)
    outs2 = run_case(ops, case, c)
    for k in ("out", "pre"):
        assert k not in outs or torch.equal(outs2[k][0], outs[k][0]), k
    report(f"gemm {name} ({kind}, M={M} N={N} K={K})", worst, bounds)
    print(f"  negative control ({'two heads swapped' if kind == 'qkv' else 'identity row_map in one row' if kind == 'pos' else 'one k-block missing in one tile'}): "
          f"{ctrl:.2e} (must be >= {cbound:.0e})")
    assert ctrl >= cbound


# ---------------------------------------------------------------------------------------------------------------------
# GELU / dGELU epilogue math over every finite bf16 value: W = I and bias = 0, so the accumulator IS the bf16 input
# ---------------------------------------------------------------------------------------------------------------------
def all_finite_bf16():
    bits = torch.arange(-32768, 32768, dtype=torch.int32, device=DEV).to(torch.int16).view(torch.bfloat16)
    return bits[torch.isfinite(bits.float())]


def _exhaustive_shape(variant, sms):
    """(kind, M, N) of a GEMM that takes the named variant (see gemm_plan) and holds every finite bf16 value."""
    n_all = 65280
    kind, epi4, bn = variant
    if kind == "gelu":
        N = 384
    elif kind == "dgelu":
        N = 384 if bn == 128 else 512
    else:
        N = {(True, 128): 384, (True, 256): 512, (False, 128): 640, (False, 256): 768}[(epi4, bn)]
    M = -(-n_all // N)
    if bn == 256:  # at least two waves of 128x256 tiles
        M = max(M, -(-2 * sms // (N // 256)) * 128)
    return kind, M, N


EXHAUSTIVE = [("gelu", False, 128), ("gelu_pre", True, 128), ("gelu_pre", True, 256), ("gelu_pre", False, 128),
              ("gelu_pre", False, 256), ("dgelu", True, 128), ("dgelu", True, 256)]


@pytest.mark.parametrize("variant", EXHAUSTIVE, ids=[f"{k}-{'epi4-' if e else ''}bn{b}" for k, e, b in EXHAUSTIVE])
def test_gelu_epilogues_on_every_bf16_input(ops, variant):
    """fc1 GELU (plain and with the saved pre-activation) and fc2 dGELU epilogue on every finite bf16 value, on each variant
    the fc1 / fc2 GEMMs can take (EPI4 or not, BN 128 or 256): within 1 ulp of the bf16 rounding of the fp64 GELU / GELU'
    plus GELU_FLOOR.  GELU: A = the values, W = I, bias 0; dGELU: dY W == 1 exactly, pre = the values."""
    sms = sm_count()
    kind, M, N = _exhaustive_shape(variant, sms)
    K = N if kind != "dgelu" else 64
    p = gemm_plan(kind, M, N, K, sms=sms)
    assert (p["epi4"], p["bn"]) == variant[1:] or kind == "gelu", (p, variant)
    vals = all_finite_bf16()
    x = vals.repeat(-(-M * N // vals.numel()))[:M * N].view(M, N).contiguous()
    buf, out = guarded((M, N), torch.bfloat16)
    if kind == "dgelu":
        dy = torch.zeros(M, K, dtype=torch.bfloat16, device=DEV)
        dy[:, 0] = 1
        w2 = torch.zeros(K, N, dtype=torch.bfloat16, device=DEV)
        w2[0] = 1
        ops.linear_dgrad(dy, w2, aux=x, out=out)
        ref = dgelu64(x.double())
    else:
        eye = torch.eye(N, dtype=torch.bfloat16, device=DEV)
        if kind == "gelu":
            ops.gemm(x, eye, None, ops.EPI_GELU_BF16, out=out)
        else:
            pbuf, pre = guarded((M, N), torch.bfloat16)
            ops.gemm_ex(x, eye, M, N, N, ops.EPI_GELU_BF16, out, aux=pre)
            assert guards_ok(pbuf)
            assert torch.equal(pre, x), "saved pre-activation differs from the accumulator"
            nbits = int((pre.view(torch.int16) != x.view(torch.int16)).sum())
            print(f"  saved pre-activation: equal in value; {nbits} elements differ in bits (-0 in -> +0 out)")
        ref = gelu64(x.double())
    assert guards_ok(buf)
    refb = ref.bfloat16().double()  # (fp64 -> bf16 goes through fp32: a tie may round either way, within the 1 ulp)
    assert torch.isfinite(out.float()).all()
    err = (out.double() - refb).abs()
    u = (err / (ulp_bf16(refb) + GELU_FLOOR)).max().item()
    beyond = ((out.double() - ref).abs() - 0.5 * ulp_bf16(ref)).clamp_min(0)  # error beyond the output rounding (fp32 math + erf approximation)
    print(f"{kind} {variant} M={M} N={N}: {u:.3f} ulps (bound {BF16_ULPS} ulp + {GELU_FLOOR:.0e}); max abs error beyond the "
          f"bf16 rounding {beyond.max().item():.2e}; max abs error {err.max().item():.2e} at |x| <= 1: "
          f"{err[x.float().abs() <= 1].max().item():.2e}")
    assert u <= BF16_ULPS


def test_gelu_epilogue_with_bias_near_the_minimum_and_in_the_tails(ops):
    """bias moves the pre-activation off the bf16 grid: x in [-1, -0.5] (the GELU minimum at -0.75) and |x| in [3, 10],
    saved pre-activation = bf16(fp32(x + b)) bit for bit, GELU within 1 ulp + GELU_FLOOR, on the EPI4 and plain variants."""
    g = torch.Generator(device=DEV).manual_seed(5)
    worst = {}
    for N in (384, 640):
        M = 512
        xs = torch.cat([torch.rand(M * N // 2, device=DEV, generator=g) * -0.5 - 0.5,
                        (torch.rand(M * N // 2, device=DEV, generator=g) * 7 + 3) * (torch.randint(0, 2, (M * N // 2,), device=DEV, generator=g) * 2 - 1)])
        x = xs.view(M, N).bfloat16()
        bias = (torch.rand(N, device=DEV, generator=g) - 0.5) * 0.02
        buf, out = guarded((M, N), torch.bfloat16)
        pbuf, pre = guarded((M, N), torch.bfloat16)
        ops.gemm_ex(x, torch.eye(N, dtype=torch.bfloat16, device=DEV), M, N, N, ops.EPI_GELU_BF16, out, bias=bias, aux=pre)
        assert guards_ok(buf) and guards_ok(pbuf)
        zf = x.float() + bias
        assert torch.equal(pre, zf.bfloat16())
        refb = gelu64(zf.double()).bfloat16().double()
        u = ((out.double() - refb).abs() / (ulp_bf16(refb) + GELU_FLOOR)).max().item()
        worst["ulps"] = max(worst.get("ulps", 0), u)
        assert u <= BF16_ULPS
    report("GELU with bias (minimum and tails)", worst, dict(ulps=BF16_ULPS))


# =====================================================================================================================
# 3. patch embedding
# =====================================================================================================================
def pe_call(ops, vol, w16, bias, pos, out, fine=None, slot=None, n_out=None, mask_token=None):
    from smb_vision_b200._lib import call

    B, T, H, W = vol.shape
    D = w16.shape[0]
    if mask_token is not None:
        call("smbv_patch_embed_select_fwd", ops._ptr(vol), ops._ptr(w16), ops._ptr(bias), ops._ptr(pos), ops._ptr(fine),
             ops._ptr(mask_token), B, T, H, W, 16, D, ops._ptr(out), ops._stream())
    else:
        n = (T // 16) * (H // 16) * (W // 16) if n_out is None else n_out
        call("smbv_patch_embed_fwd", ops._ptr(vol), ops._ptr(w16), ops._ptr(bias), ops._ptr(pos), ops._ptr(fine),
             ops._ptr(slot), B, T, H, W, 16, D, n, ops._ptr(out), ops._stream())


PE_VOLUMES = [(96, 96, 96), (160, 224, 224), (32, 80, 592)]  # 6^3 tokens; 10 x 14 x 14 (gx = gy = 14); gy = 5, gx = 37
PE_DIMS = (32, 64, 128, 192, 384, 768, 1024)


@pytest.mark.parametrize("vshape", PE_VOLUMES, ids=["96cube", "224x224x160", "gy5-gx37"])
def test_patch_embed_matches_fp64(ops, vshape):
    """fp64 patchify(bf16 volume) @ bf16 W^T + bias (+ pos) for B = 1, 2, 4 and every D (D % 192 != 0: a narrow last N tile),
    pos = None on some, the visible-token compaction (nothing masked, one token visible, B >= 2 with equal counts) and the
    SimMIM blend; per 128-token x 128-column tile and per element; bit-reproducible."""
    T, H, W = vshape
    cfg = types.SimpleNamespace(tubelet_size=16, patch_size=16)
    N = (T // 16) * (H // 16) * (W // 16)
    worst, ctrl = {}, float("inf")
    for B in (1, 2, 4):
        g = torch.Generator(device=DEV).manual_seed(B * 1000 + N)
        vol = torch.rand(B, T, H, W, device=DEV, generator=g) * 2 - 0.5
        P = vo.patchify(vol.bfloat16().double()[:, :, None], cfg)  # [B, N, 4096]
        for D in PE_DIMS:
            w16 = rnd((D, 4096), g, scale=0.02)
            bias = torch.randn(D, device=DEV, generator=g) * 0.1
            pos = None if D == 1024 else torch.randn(N, D, device=DEV, generator=g)  # V-JEPA (ViT-L): positions through RoPE
            emb = P @ w16.double().t()
            ref = emb + bias.double() + (pos.double() if pos is not None else 0)
            buf, out = guarded((B, N, D))
            pe_call(ops, vol, w16, bias, pos, out)
            assert guards_ok(buf)
            check_f32(out.reshape(B * N, D), ref.reshape(B * N, D), worst)
            buf2, out2 = guarded((B, N, D))
            pe_call(ops, vol, w16, bias, pos, out2)
            assert torch.equal(out2, out)
            # negative control: dz plane 7 (k in [7*256, 8*256)) of the first 128 tokens x 128 channels dropped
            bad = ref.clone().reshape(B * N, D)
            ks = slice(7 * 256, 8 * 256)
            Pr = P.reshape(B * N, 4096)
            bad[:128, :128] -= Pr[:128, ks] @ w16.double()[:128, ks].t()
            ctrl = min(ctrl, tile_frob(out.reshape(B * N, D), bad))
        # compaction and blend at D = 384 (decoder / encoder widths are covered above)
        D = 384
        w16 = rnd((D, 4096), g, scale=0.02)
        bias, pos = torch.randn(D, device=DEV, generator=g) * 0.1, torch.randn(N, D, device=DEV, generator=g)
        full = P @ w16.double().t() + bias.double() + pos.double()
        masks = []
        if B == 1:
            masks += [torch.zeros(1, N, dtype=torch.bool, device=DEV), torch.ones(1, N, dtype=torch.bool, device=DEV)]
            masks[-1][0, N // 2] = False  # all but one masked
        n_vis = max(1, N // 3)
        masks.append(torch.stack([torch.randperm(N, device=DEV, generator=g) >= n_vis for _ in range(B)]))
        for mask in masks:
            nv = int((~mask[0]).sum())
            fine = mask.to(torch.uint8)
            _, _, slot, _ = ops.mask_index(fine)
            buf, out = guarded((B, nv, D))
            pe_call(ops, vol, w16, bias, pos, out, fine=fine, slot=slot, n_out=nv)
            assert guards_ok(buf)
            ref = torch.stack([full[b][~mask[b]] for b in range(B)])
            check_f32(out.reshape(B * nv, D), ref.reshape(B * nv, D), worst)
            mt = torch.randn(D, device=DEV, generator=g)
            buf, out = guarded((B, N, D))
            pe_call(ops, vol, w16, bias, pos, out, fine=fine, mask_token=mt)
            assert guards_ok(buf)
            ref = torch.where(mask[..., None], mt.double() + pos.double(), full)
            check_f32(out.reshape(B * N, D), ref.reshape(B * N, D), worst)
            buf2, out2 = guarded((B, N, D))
            pe_call(ops, vol, w16, bias, pos, out2, fine=fine, mask_token=mt)
            assert torch.equal(out2, out)
    report(f"patch_embed {T}x{H}x{W} (N={N})", worst, dict(frob=F32_FROB, maxrel=F32_MAX, local=F32_LOCAL))
    print(f"  negative control (one dz plane missing in one tile): worst-tile frob-rel {ctrl:.2e}")
    assert ctrl >= CONTROL * F32_LOCAL


# =====================================================================================================================
# 4. LayerNorm forward
# =====================================================================================================================
LN_DIMS = (64, 128, 256, 384, 512, 768, 1024, 2048, 4096, 100, 260)  # NV = 1, 1, 2, 3, 4, 6, 8, 16, 32; 100, 260: idle lanes


def _ln_rows(kind, M, d, g):
    if kind == "randn":
        return torch.randn(M, d, device=DEV, generator=g) * 3 + 1
    if kind == "offset":  # |mean| >> std: a one-pass E[x^2] - mean^2 cancels catastrophically
        return torch.randn(M, d, device=DEV, generator=g) * 1e-2 + 1e3
    x = torch.full((M, d), 0.75, device=DEV)  # constant rows: var = 0, rstd = eps^-1/2
    x[1::2] = -3.5
    return x


def ln_call(ops, x, gamma, beta, eps, y):
    """smbv_layernorm_fwd into y (bf16 [M, d]) with NaN-prefilled, guarded mean / rstd; returns (mean, rstd)."""
    from smb_vision_b200._lib import call

    M, d = x.shape
    bm, mean = guarded((M,))
    br, rstd = guarded((M,))
    call("smbv_layernorm_fwd", ops._ptr(x), ops._ptr(gamma), ops._ptr(beta), float(eps), M, d, ops._ptr(y), ops._ptr(mean),
         ops._ptr(rstd), ops._stream())
    assert guards_ok(bm) and guards_ok(br), "guard region of mean / rstd overwritten"
    return mean, rstd


@pytest.mark.parametrize("d", LN_DIMS)
def test_layernorm_forward_matches_fp64(ops, d):
    """every NV instantiation, M % 8 != 0, `out=` row views, every eps the models use (1e-12 VideoMAE, 1e-6 V-JEPA, 1e-5
    decoder norm / fc_norm).  mean: error in fp32 ulps of the row's rms; rstd: in fp32 ulps of the two-pass value computed
    in fp64 for the kernel's mean; y: bf16 ulps of the fp64 LayerNorm with those statistics.  Bit-reproducible."""
    worst, ctrl = {}, 0.0
    for kind in ("randn", "offset", "constant"):
        for eps in (1e-12, 1e-6, 1e-5):
            M = 1031 if d <= 1024 else 203
            g = torch.Generator(device=DEV).manual_seed(d * 7 + M + int(-math.log10(eps)))
            x = _ln_rows(kind, M, d, g)
            gamma, beta = torch.randn(d, device=DEV, generator=g), torch.randn(d, device=DEV, generator=g)
            buf, y = guarded((M + 5, d), torch.bfloat16)
            yv = y[3:3 + M]  # a row range of a larger buffer, as the decoder norm writes hN[b]
            mean, rstd = ln_call(ops, x, gamma, beta, eps, yv)
            assert guards_ok(buf) and torch.isnan(y[:3].float()).all() and torch.isnan(y[3 + M:].float()).all()
            xd = x.double()
            mu = xd.mean(1)
            rms = xd.pow(2).mean(1).sqrt()
            eps32 = float(torch.tensor(eps, dtype=torch.float32))
            m_ulps = ((mean.double() - mu).abs() / (rms * 2.0 ** -23)).max().item()
            mk = mean.double()[:, None]
            r2 = 1 / torch.sqrt((xd - mk).pow(2).mean(1) + eps32)  # two-pass rstd for the kernel's mean
            r_ulps = ((rstd.double() - r2).abs() / (r2 * 2.0 ** -23)).max().item()
            ref = (xd - mk) * rstd.double()[:, None] * gamma.double() + beta.double()
            worst["mean ulps"] = max(worst.get("mean ulps", 0), m_ulps)
            worst["rstd ulps"] = max(worst.get("rstd ulps", 0), r_ulps)
            check_bf16(yv, ref, worst, key="y ulps")
            assert m_ulps <= MEAN_ULPS and r_ulps <= RSTD_ULPS, (kind, eps, m_ulps, r_ulps)
            if kind == "constant":
                assert torch.equal(mean, x[:, 0]) and torch.equal(yv, beta.bfloat16().expand(M, d))
            buf2, y2 = guarded((M, d), torch.bfloat16)
            mean2, rstd2 = ln_call(ops, x, gamma, beta, eps, y2)
            assert guards_ok(buf2) and torch.equal(y2, yv) and torch.equal(mean2, mean) and torch.equal(rstd2, rstd)
            if kind == "offset":  # negative control: one-pass variance E[x^2] - mean^2 in fp32
                xf = x.float()
                var1 = (xf * xf).mean(1) - mean * mean
                r1 = torch.rsqrt(var1.clamp_min(0) + eps).double()
                ctrl = max(ctrl, ((rstd.double() - r1).abs() / (r1 * 2.0 ** -23)).max().item())
    report(f"layernorm_fwd d={d}", worst, {"mean ulps": MEAN_ULPS, "rstd ulps": RSTD_ULPS, "y ulps": BF16_ULPS})
    print(f"  negative control (one-pass variance, |mean| = 1e3, std = 1e-2): rstd {ctrl:.2e} fp32 ulps")
    assert ctrl >= CONTROL * RSTD_ULPS


# =====================================================================================================================
# 5. norm-pix loss, mask-token fill, cast
# =====================================================================================================================
def _normpix_ref(vol, idx, n_mask, logits, P, kind, unbiased=True):
    """fp64 per-patch normalised labels -> (loss, dlogits, d, labels) for the masked patches idx[:, :n_mask]."""
    B = vol.shape[0]
    cfg = types.SimpleNamespace(tubelet_size=P, patch_size=P)
    X = vo.patchify(vol.double()[:, :, None], cfg)
    X = torch.stack([X[b, idx[b, :n_mask].long()] for b in range(B)])  # [B, n_mask, P^3]
    mean = X.mean(-1, keepdim=True)
    var = X.var(-1, keepdim=True, unbiased=unbiased)
    lab = (X - mean) / (var.sqrt() + 1e-6)
    d = logits.double() - lab
    count = d.numel()
    if kind == 0:
        return (d * d).sum() / count, 2 * d / count, d, lab
    return d.abs().sum() / count, torch.sign(d) / count, d, lab


def _normpix_grad_metric(dl, ref_dl, d, lab, count, kind):
    if kind == 0:
        return bf16_ulps(dl, ref_dl, floor=2 / count * LABEL_TOL * (1 + lab.abs()))
    gs = float(torch.tensor(1 / count, dtype=torch.float32).bfloat16())
    sure = d.abs() > LABEL_TOL * (1 + lab.abs())
    want = torch.sign(d) * gs
    wrong = (sure & (dl.double() != want)) | ((d == 0) & (dl != 0))
    return float(wrong.sum())


def normpix_call(ops, vol, idx, n_mask, logits, loss_kind, P):
    """smbv_normpix_loss with NaN-prefilled, guarded dlogits, per-patch partials and loss: every element must be written,
    nothing past them (the warp kernel's last CTA has warps past n_mask when n_mask % 8 != 0).  Returns (loss, dlogits)."""
    from smb_vision_b200._lib import call

    B, T, H, W = vol.shape
    bd, dl = guarded(tuple(logits.shape), torch.bfloat16)
    bp, partial = guarded((B * n_mask,))
    bl, loss = guarded((1,))
    call("smbv_normpix_loss", ops._ptr(vol), B, T, H, W, P, ops._ptr(idx), n_mask, idx.shape[1], ops._ptr(logits), ops._ptr(dl),
         ops._ptr(partial), ops._ptr(loss), loss_kind, ops._stream())
    assert guards_ok(bd) and guards_ok(bp) and guards_ok(bl), "guard region overwritten"
    assert not torch.isnan(dl.float()).any() and not torch.isnan(partial).any(), "dlogits / partials not fully written"
    # the loss is the fp64 sum of the partials over the element count, rounded to fp32
    want = partial.double().sum() / logits.numel()
    assert abs(loss.double().item() - want.item()) <= 2.0 ** -23 * abs(want.item()), (loss.item(), want.item())
    return loss[0], dl


def _mask_idx(Np, stride, B, pins, g):
    """int32 [B, stride] rows of distinct patch ids, pins[(b, j)] = patch id at position j of sample b."""
    rows = []
    for b in range(B):
        pin = {j: p for (bb, j), p in pins.items() if bb == b}
        rest = [i for i in torch.randperm(Np, device=DEV, generator=g).tolist() if i not in pin.values()]
        rows.append([pin[j] if j in pin else rest.pop() for j in range(stride)])
    return torch.tensor(rows, dtype=torch.int32, device=DEV)


@pytest.mark.parametrize("kind", [0, 1], ids=["mse", "l1"])
def test_normpix_loss_three_kernels_match_fp64(ops, kind):
    """warp-per-patch (default), block-per-patch (loss_kind 16 / 17) and generic-P kernels (patch = 8, and P = 16 on a volume
    view that is not 16-byte aligned): B = 1, 2, n_mask % 8 != 0, idx_stride > n_mask, constant patches, logits = 0.5 randn
    and logits = bf16(label) (d = 0 on the constant patches: L1 sign at 0).  Loss within LOSS_REL of fp64, dlogits per
    element; the three P = 16 kernels agree up to fp32 summation order (loss) and 1 bf16 ulp (dlogits)."""
    T, H, W = 32, 48, 64
    worst, ctrl, ndiff = {}, float("inf"), 0
    for B in (1, 2):
        g = torch.Generator(device=DEV).manual_seed(B + 10 * kind)
        vol = torch.randn(B, T, H, W, device=DEV, generator=g) * 2 + 0.5
        vol[0, :16, :16, :16] = 0.25  # patch 0 of sample 0: constant (label 0 / (0 + 1e-6))
        vol[B - 1, 16:, 32:, 48:] = -1.5  # the last patch of the last sample: constant
        for P, n_mask, stride in ((16, 13, 20), (8, 37, 50)):
            Np = (T // P) * (H // P) * (W // P)
            # the constant patches (patch 0 of sample 0, the last patch of the last sample) are among the masked ones
            pins = {(0, 3): 0, (B - 1, n_mask - 1): Np - 1}
            idx = _mask_idx(Np, stride, B, pins, g)
            _, _, _, lab = _normpix_ref(vol, idx, n_mask, torch.zeros(B, n_mask, P ** 3, device=DEV), P, kind)
            for fam, logits in (("randn", rnd((B, n_mask, P ** 3), g, scale=0.5)), ("label", lab.bfloat16())):
                ref_loss, ref_dl, d, _ = _normpix_ref(vol, idx, n_mask, logits, P, kind)
                count = d.numel()
                variants = [("generic P=8", vol, kind)] if P == 8 else [("warp", vol, kind), ("block", vol, kind + 16)]
                if P == 16:  # the same volume at an address that is 4 bytes past a 16-byte boundary -> generic kernel
                    big = torch.empty(vol.numel() + 4, device=DEV)
                    vmis = big[1:1 + vol.numel()].view(vol.shape)
                    vmis.copy_(vol)
                    variants.append(("generic misaligned", vmis, kind))
                res = {}
                for vname, v, lk in variants:
                    loss, dl = normpix_call(ops, v, idx, n_mask, logits, lk, P)
                    lrel = abs(loss.item() - ref_loss.item()) / ref_loss.item()
                    gm = _normpix_grad_metric(dl, ref_dl, d, lab, count, kind)
                    key = "dl ulps" if kind == 0 else "dl wrong signs"
                    worst["loss rel"], worst[key] = max(worst.get("loss rel", 0), lrel), max(worst.get(key, 0), gm)
                    assert lrel <= LOSS_REL and gm <= (BF16_ULPS if kind == 0 else 0), (vname, B, P, fam, lrel, gm)
                    if fam == "label":  # constant patches: d == 0
                        assert (dl.double()[d == 0] == 0).all()
                    loss2, dl2 = normpix_call(ops, v, idx, n_mask, logits, lk, P)
                    assert loss2.item() == loss.item() and torch.equal(dl2, dl)
                    res[vname] = (loss.item(), dl)
                    if fam == "label" and vname in ("warp", "generic P=8"):
                        # negative control: labels with the biased variance.  They move by sqrt(K / (K - 1)) - 1 = 1.2e-4
                        # of |label| (P = 16), against d ~ 2^-9 |label| for logits = bf16(label): the loss moves by 0.2 % (L1) to 0.5 % (MSE)
                        bl, _, _, _ = _normpix_ref(vol, idx, n_mask, logits, P, kind, unbiased=False)
                        ctrl = min(ctrl, abs(loss.item() - bl.item()) / bl.item() / LOSS_REL)
                if P == 16:  # the three kernels sum in different orders: labels may differ in the last fp32 bits
                    l0, d0 = res["warp"]
                    for vname, (lv, dv) in res.items():
                        agree = abs(lv - l0) / abs(l0)
                        nd = int((dv != d0).sum())
                        worst["kernels agree"] = max(worst.get("kernels agree", 0), agree)
                        ndiff = max(ndiff, nd)
                        if kind == 0:
                            dd = bf16_ulps(dv, d0.double(), floor=2 / count * LABEL_TOL)
                        else:
                            dd = float(((dv != d0) & (d.abs() > LABEL_TOL * (1 + lab.abs()))).sum())
                        assert agree <= REPRO_LOSS and dd <= (BF16_ULPS if kind == 0 else 0), (vname, agree, nd, dd)
    report(f"normpix_loss {'mse' if kind == 0 else 'l1'}", worst,
           {"loss rel": LOSS_REL, "dl ulps": BF16_ULPS, "dl wrong signs": 0.0, "kernels agree": REPRO_LOSS})
    print(f"  dlogits elements that differ between the warp, block and generic kernels: at most {ndiff} per call")
    print(f"  negative control (biased variance, logits = label): loss error {ctrl:.1f} x the bound")
    assert ctrl >= CONTROL


def test_fill_mask_tokens_is_exact(ops):
    """x_dec[b, n_vis + j] = pos[msk_idx[b, j]] + mask_token, bit-exact in fp32, idx_stride > n_mask; rows < n_vis keep their
    sentinel."""
    for B, N, n_vis, d in ((1, 300, 100, 384), (2, 1000, 357, 388), (3, 64, 0, 4)):
        g = torch.Generator(device=DEV).manual_seed(N + d)
        n_mask, stride = N - n_vis, N - n_vis + 7
        pos = torch.randn(N, d, device=DEV, generator=g)
        mt = torch.randn(d, device=DEV, generator=g)
        idx = torch.stack([torch.randperm(N, device=DEV, generator=g)[:n_mask] for _ in range(B)])
        idx = torch.cat([idx, idx[:, :7] if n_mask >= 7 else torch.zeros(B, 7, dtype=idx.dtype, device=DEV)], 1).to(torch.int32)
        buf, x = guarded((B, N, d))
        x[:, :n_vis] = -2.0
        ops.fill_mask_tokens(x, mt, pos, idx, n_vis)
        assert guards_ok(buf) and (x[:, :n_vis] == -2.0).all()
        want = pos[idx[:, :n_mask].long()] + mt
        assert torch.equal(x[:, n_vis:], want)
        assert not torch.equal(x[:, n_vis:], pos[:n_mask].expand(B, n_mask, d) + mt)  # negative control: identity index


def test_cast_bf16_is_round_to_nearest_even(ops):
    """fp32 -> bf16 weight cast (every bf16 weight copy, the AdamW arena's too): bit-exact against torch's .bfloat16() for
    n % 4 = 0..3 (the scalar tail), +-0, denormals, +-inf, values exactly at the rounding tie (both parities) and random
    values; NaN stays NaN (payload free); nothing past n written."""
    g = torch.Generator(device=DEV).manual_seed(1)
    special = torch.tensor([0.0, -0.0, float("inf"), float("-inf"), 1e-40, -1e-40, 1.4e-45, 3.4e38, -3.4e38, 1.17549435e-38],
                           device=DEV)
    ties = torch.tensor([0x3F808000, 0x3F818000, 0xBF808000, 0xBF818000, 0x00008000, 0x00018000, 0x7F7F8000, 0x3F80FFFF,
                         0x3F807FFF, 0x3F808001], dtype=torch.int64, device=DEV).to(torch.int32).view(torch.float32)
    for n in (4096, 4097, 4098, 4099, 1, 2, 3, 1000003):
        src = torch.randn(n, device=DEV, generator=g) * torch.exp2(torch.randint(-140, 120, (n,), device=DEV, generator=g).float())
        k = min(n, special.numel() + ties.numel())
        src[:k] = torch.cat([special, ties])[:k]
        if n > 40:
            src[-1] = float("nan")
        buf, out = guarded((n,), torch.bfloat16)
        ops.cast_bf16(src, out=out)
        assert guards_ok(buf)
        fin = ~torch.isnan(src)
        assert torch.equal(out[fin].view(torch.int16), src[fin].bfloat16().view(torch.int16)), n
        assert torch.isnan(out[~fin].float()).all()
        assert not torch.equal(out[fin].view(torch.int16), (src[fin].view(torch.int32) >> 16).to(torch.int16)) or n < 40  # control: truncation
