"""Kernel-level parity of the training BACKWARD (run with -m gpu on the B200 box): the gradient GEMM views of `gemm_ex`
(transposed / head-major A, W seen [K,N], split-K reduce-add), LayerNorm backward, the column sums behind every bias
gradient and the data-movement kernels of the backward pass.  Whole-model gradient tests allow 2e-2 .. 5e-2; one k-block
missing from one output tile of the patch-embedding weight gradient moves that tensor by only ~9e-3, so these tests
compare each kernel on its own with a float64 reference computed ON THE DEVICE from the same bf16 operands the kernel
reads: the bounds then measure accumulation and output rounding only.

Bounds:
  fp32 / reduce-add outputs: Frobenius-rel <= 2e-5, max-abs-rel <= 1e-4, plus a local bound (worst 128x128 tile, worst row,
      or per column relative to the column's L2 norm) so that one wrong tile, row or k-block cannot hide in a global norm;
  bf16 outputs: Frobenius-rel <= 4e-3 and every element within 1 bf16 ulp of the fp64 reference (+ 1e-5 of the max as floor);
  data movement and casts: bit-exact.
Every test also runs a negative control: the same comparison against a reference with one k-block / head / row / row
block removed must fail its local bound by >= 100x.

Reproducibility (README, "Determinism"): kernels without a cross-CTA reduction (dgrad GEMMs, LayerNorm-backward rows, token
sum, gathers, casts) are checked bit-identical on a second call; the reduce-add ones (weight gradients, column sums, dgamma /
dbeta) are checked equal up to fp32 summation order (REPRO_TOL).
"""
import types

import pytest
import torch
import torch.nn.functional as F

from oracle import videomae_oracle as vo

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

F32_FROB, F32_MAX, F32_LOCAL = 2e-5, 1e-4, 2e-5
# the fp32 tensor-core accumulator loses ~1e-9 per k-step: a tile that runs more than 8192 k-steps in one accumulator gets
# 5e-5 (Frobenius-rel / worst tile; measured on B200 at 1000 W: 2.3e-5 for the [768,4096] weight gradient over 20480 tokens,
# 192 output tiles -> no K split)
F32_LONG_K = 5e-5
COL_REL = 1e-4  # column sums: |err| / L2 norm of the summed terms
BF16_FROB, BF16_ULPS = 4e-3, 1.0
REPRO_TOL = 2e-6  # Frobenius-rel between two calls of a reduce-add kernel (fp32 summation order only)
CONTROL = 100.0


@pytest.fixture(scope="module")
def ops():
    assert torch.cuda.is_available()
    from smb_vision_b200 import load, ops as _ops

    lib = load()
    assert lib.smbv_device_ok() == 0, lib.smbv_last_error()
    return _ops


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


def col_rel(got, ref, scale):
    """max over elements of |got - ref| / scale, scale = L2 norm of the terms summed into that element."""
    return ((got.double() - ref.double()).abs() / scale.double().clamp_min(1e-300)).max().item()


def bf16_ulps(got, ref):
    """max over elements of |got - ref| / (1 bf16 ulp of ref + 1e-5 max|ref|)."""
    ref = ref.double()
    ulp = torch.exp2(torch.floor(torch.log2(ref.abs())) - 7)  # 8 significant bits; 0 at ref == 0
    return ((got.double() - ref).abs() / (ulp + 1e-5 * ref.abs().max())).max().item()


def check_f32(got, ref, worst, local=None):
    """fp32 output against the fp64 reference; returns the local metric (worst 128x128 tile unless given)."""
    assert torch.isfinite(got).all()
    f, m = frob(got, ref), maxrel(got, ref)
    loc = tile_frob(got, ref) if local is None else local(got, ref)
    worst["frob"], worst["maxrel"], worst["local"] = max(worst.get("frob", 0), f), max(worst.get("maxrel", 0), m), max(worst.get("local", 0), loc)
    return f, m, loc


def check_bf16(got, ref, worst):
    assert torch.isfinite(got.float()).all()
    f, u = frob(got, ref), bf16_ulps(got, ref)
    worst["frob"], worst["ulps"] = max(worst.get("frob", 0), f), max(worst.get("ulps", 0), u)
    return f, u


def report(name, worst, bounds):
    print(f"{name}: " + ", ".join(f"{k} {worst[k]:.2e} (bound {bounds[k]:.0e})" for k in bounds if k in worst))


def rnd(shape, g, dtype=torch.bfloat16, scale=1.0):
    return (torch.randn(shape, device=DEV, generator=g) * scale).to(dtype)


def tile_block(a, b, kb, r=slice(0, 128), c=slice(0, 128)):
    """contribution of k-block kb (64 along the contraction) of a[R,K] @ b[K,C] to the output tile [r, c], fp64."""
    ks = slice(64 * kb, 64 * kb + 64)
    return a[r, ks].double() @ b[ks, c].double()


# =====================================================================================================================
# 1. gradient GEMMs
# =====================================================================================================================
TOKENS = [1, 63, 65, 200, 1000, 7168, 13312, 20480]  # ragged last k-block; 7168 / 13312 / 20480 = encoder / masked / full


@pytest.mark.parametrize("N,K", [(768, 768), (3072, 768), (768, 3072), (384, 768), (1152, 384), (384, 1536), (4096, 384),
                                 (768, 4096), (768, 96), (384, 160), (96, 768)])
def test_linear_wgrad_matches_fp64(ops, N, K):
    """dW[N,K] += dY[M,N]^T X[M,K]: transposed A, W seen [K,N], fp32 reduce-add epilogue, automatic split-K.  Every output
    shape of the model (decoder head [4096,384], patch embedding [768,4096]) at every token count, plus N % 64 == 32 and an
    output with 96 rows."""
    worst, ctrl = {}, float("inf")
    for M in TOKENS:
        tol = F32_FROB if M <= 8192 else F32_LONG_K
        g = torch.Generator(device=DEV).manual_seed(N * 7 + K * 13 + M)
        dy, x = rnd((M, N), g), rnd((M, K), g)
        prefill = torch.randn(N, K, device=DEV, generator=g) * M ** 0.5  # accumulate semantics: same scale as the product
        dw = prefill.clone()
        ops.linear_wgrad(dy, x, dw)
        got = dw.double() - prefill.double()
        ref = dy.double().t() @ x.double()
        f, m, t = check_f32(got, ref, worst)
        assert f <= tol and m <= F32_MAX and t <= tol, (M, f, m, t)
        dw2 = prefill.clone()
        ops.linear_wgrad(dy, x, dw2)
        rep = frob(dw2, dw)
        worst["repro"] = max(worst.get("repro", 0), rep)
        assert rep <= REPRO_TOL, (M, rep)
        # negative control: k-block (middle one) dropped from the first 128x128 output tile
        bad = ref.clone()
        bad[:128, :128] -= tile_block(dy.t(), x, ((M + 63) // 64) // 2)
        ctrl = min(ctrl, tile_frob(got, bad))
    report(f"wgrad [{N},{K}]", worst, dict(frob=F32_LONG_K, maxrel=F32_MAX, local=F32_LONG_K, repro=REPRO_TOL))
    print(f"  (bound 2e-5 up to 8192 tokens)  negative control (one k-block missing in one tile): worst-tile frob-rel >= {ctrl:.2e}")
    assert ctrl >= CONTROL * F32_LONG_K


@pytest.mark.parametrize("N,K,M,splits", [(768, 768, 7168, [0, 1, 2, 3, 7, 112]),    # 36 tiles < 148 SMs: auto split
                                          (384, 1536, 300, [0, 1, 2, 3, 4, 5, 7]),  # 5 k-blocks: 4 and 7 leave an empty slice
                                          (1152, 384, 1000, [1, 2, 3, 7, 16])])
def test_explicit_split_k_matches_fp64_and_agrees(ops, N, K, M, splits):
    """`gemm_ex(..., EPI_ATOMIC_F32, split_k=s)`: every split (the no-empty-slice loop lowers s = 4 and 7 at 5 k-blocks) matches
    the reference, and all splits agree with each other within the fp32 accumulation bound (a split regroups the tensor-core
    sums, not only the order of the reduce-adds: measured 5.6e-6 between 1 and 112 slices at 112 k-blocks)."""
    g = torch.Generator(device=DEV).manual_seed(M)
    dy, x = rnd((M, N), g), rnd((M, K), g)
    prefill = torch.randn(N, K, device=DEV, generator=g) * M ** 0.5
    ref = dy.double().t() @ x.double()
    worst, outs = {}, {}
    for s in splits:
        dw = prefill.clone()
        ops.gemm_ex(dy, x, N, K, M, ops.EPI_ATOMIC_F32, dw, a_layout=ops.A_TRANSPOSED, w_layout=1, lda=N, ldw=K, split_k=s)
        got = dw.double() - prefill.double()
        f, m, t = check_f32(got, ref, worst)
        assert f <= F32_FROB and m <= F32_MAX and t <= F32_LOCAL, (s, f, m, t)
        outs[s] = dw
    agree = max(frob(o, outs[1]) for o in outs.values())
    worst["agree"] = agree
    assert agree <= F32_FROB
    report(f"split-K {splits} [{N},{K}] x {M}", worst, dict(frob=F32_FROB, maxrel=F32_MAX, local=F32_LOCAL, agree=F32_FROB))
    bad = ref.clone()
    bad[:128, :128] -= tile_block(dy.t(), x, 0)
    ctrl = tile_frob(outs[splits[-1]].double() - prefill.double(), bad)
    print(f"  negative control (k-block 0 missing in one tile): {ctrl:.2e}")
    assert ctrl >= CONTROL * F32_LOCAL


def test_gemm_ex_bias_alpha_and_strided_views(ops):
    """C-ABI extras of `gemm_ex`: bias under a K split (added once, by slice 0), the device-scalar alpha (reduce-add, fp32 and
    bf16 epilogues), ldo > N (columns past N untouched) and lda > M on the transposed A."""
    g = torch.Generator(device=DEV).manual_seed(11)
    N, K, M = 384, 160, 1000
    dy, x = rnd((M, N), g), rnd((M, K), g)
    bias = torch.randn(K, device=DEV, generator=g) * 10
    alpha = torch.tensor([0.3125], device=DEV)
    ref = dy.double().t() @ x.double()
    worst = {}
    for s in (1, 4, 0):
        dw = torch.zeros(N, K, device=DEV)
        ops.gemm_ex(dy, x, N, K, M, ops.EPI_ATOMIC_F32, dw, a_layout=ops.A_TRANSPOSED, w_layout=1, lda=N, ldw=K, split_k=s, bias=bias)
        f, m, t = check_f32(dw, ref + bias.double(), worst)
        assert f <= F32_FROB and m <= F32_MAX and t <= F32_LOCAL, (s, f, m, t)
        dw = torch.zeros(N, K, device=DEV)
        ops.gemm_ex(dy, x, N, K, M, ops.EPI_ATOMIC_F32, dw, a_layout=ops.A_TRANSPOSED, w_layout=1, lda=N, ldw=K, split_k=s, alpha=alpha)
        f, m, t = check_f32(dw, 0.3125 * ref, worst)
        assert f <= F32_FROB and m <= F32_MAX and t <= F32_LOCAL, (s, f, m, t)
    # alpha (+ bias) on the plain fp32 / bf16 outputs of a row-major A
    a, w = rnd((M, K), g), rnd((N, K), g, scale=0.05)
    refo = a.double() @ w.double().t()
    bias_n = torch.randn(N, device=DEV, generator=g)
    out = torch.full((M, N), float("nan"), device=DEV)
    ops.gemm_ex(a, w, M, N, K, ops.EPI_F32, out, alpha=alpha, bias=bias_n)
    f, m, t = check_f32(out, 0.3125 * refo + bias_n.double(), worst)
    assert f <= F32_FROB and m <= F32_MAX and t <= F32_LOCAL
    outb = torch.full((M, N), float("nan"), dtype=torch.bfloat16, device=DEV)
    ops.gemm_ex(a, w, M, N, K, ops.EPI_BF16, outb, alpha=alpha)
    wb = {}
    f, u = check_bf16(outb, 0.3125 * refo, wb)
    assert f <= BF16_FROB and u <= BF16_ULPS
    # ldo > N: the fp32 columns past N keep their sentinel
    ldo = N + 40
    wide = torch.full((M, ldo), 7.0, device=DEV)
    wide[:, :N] = float("nan")
    ops.gemm_ex(a, w, M, N, K, ops.EPI_F32, wide, ldo=ldo)
    f, m, t = check_f32(wide[:, :N], refo, worst)
    assert f <= F32_FROB and m <= F32_MAX and t <= F32_LOCAL
    assert torch.equal(wide[:, N:], torch.full((M, ldo - N), 7.0, device=DEV))
    # lda > M on the transposed A: dY stored [tokens][lda] with only the first N columns used
    lda = N + 64
    dyw = rnd((M, lda), g)
    dw = torch.zeros(N, K, device=DEV)
    ops.gemm_ex(dyw, x, N, K, M, ops.EPI_ATOMIC_F32, dw, a_layout=ops.A_TRANSPOSED, w_layout=1, lda=lda, ldw=K)
    f, m, t = check_f32(dw, dyw[:, :N].double().t() @ x.double(), worst)
    assert f <= F32_FROB and m <= F32_MAX and t <= F32_LOCAL
    report("gemm_ex bias / alpha / ldo / lda", worst, dict(frob=F32_FROB, maxrel=F32_MAX, local=F32_LOCAL))
    report("gemm_ex alpha, bf16 output", wb, dict(frob=BF16_FROB, ulps=BF16_ULPS))
    # negative control: bias added by every one of the 4 K slices instead of once
    dw = torch.zeros(N, K, device=DEV)
    ops.gemm_ex(dy, x, N, K, M, ops.EPI_ATOMIC_F32, dw, a_layout=ops.A_TRANSPOSED, w_layout=1, lda=N, ldw=K, split_k=4, bias=bias)
    ctrl = tile_frob(dw, ref + 4 * bias.double())
    print(f"  negative control (bias once per slice): {ctrl:.2e}")
    assert ctrl >= CONTROL * F32_LOCAL


@pytest.mark.parametrize("N,K", [(768, 96), (1536, 384), (3072, 768), (384, 1536), (768, 3072)])
def test_linear_dgrad_bf16_and_f32_match_fp64(ops, N, K):
    """dX[M,K] = dY[M,N] W[N,K] (W = the nn.Linear weight seen [K,N]) with the bf16 and fp32 epilogues at ragged M; M = 7168
    with K = 1536 / 3072 takes BN = 256 (two or more waves of 128x256 tiles).  No cross-CTA reduction: bit-identical on a
    second call."""
    g = torch.Generator(device=DEV).manual_seed(N + K)
    w = rnd((N, K), g, scale=0.05)
    wb, w32, ctrl_b, ctrl_f = {}, {}, float("inf"), float("inf")
    for M in (1, 130, 1000, 7168):
        dy = rnd((M, N), g)
        ref = dy.double() @ w.double()
        kb = (N // 64) // 2
        bad = ref.clone()
        bad[:128, :128] -= tile_block(dy, w, kb)
        out = torch.full((M, K), float("nan"), dtype=torch.bfloat16, device=DEV)
        ops.linear_dgrad(dy, w, out=out)
        f, u = check_bf16(out, ref, wb)
        assert f <= BF16_FROB and u <= BF16_ULPS, (M, f, u)
        assert torch.equal(ops.linear_dgrad(dy, w), out)
        ctrl_b = min(ctrl_b, bf16_ulps(out, bad))
        out = torch.full((M, K), float("nan"), device=DEV)
        ops.linear_dgrad(dy, w, out=out)
        f, m, t = check_f32(out, ref, w32)
        assert f <= F32_FROB and m <= F32_MAX and t <= F32_LOCAL, (M, f, m, t)
        assert torch.equal(ops.linear_dgrad(dy, w, out_dtype=torch.float32), out)
        ctrl_f = min(ctrl_f, tile_frob(out, bad))
    report(f"dgrad bf16 [{N}->{K}]", wb, dict(frob=BF16_FROB, ulps=BF16_ULPS))
    report(f"dgrad f32  [{N}->{K}]", w32, dict(frob=F32_FROB, maxrel=F32_MAX, local=F32_LOCAL))
    print(f"  negative control (one k-block missing in one tile): bf16 {ctrl_b:.2e} ulps, f32 worst-tile {ctrl_f:.2e}")
    assert ctrl_b >= CONTROL * BF16_ULPS and ctrl_f >= CONTROL * F32_LOCAL


def _token_major(dqkv):
    """head-major [3,B,H,n,64] -> token-major [B, n, 3*H*64] (the layout of the plain QKV GEMM output)."""
    _, B, H, n, _ = dqkv.shape
    return dqkv.permute(1, 3, 0, 2, 4).reshape(B, n, 3 * H * 64)


def _qkv_case(ops, dqkv, heads, worst_d, worst_w, g):
    """qkv_dgrad / qkv_wgrad for every sample of a head-major buffer; returns the weakest negative-control ratios."""
    _, B, _, n, _ = dqkv.shape
    d = heads * 64
    w = rnd((3 * d, d), g, scale=0.05)
    tok = _token_major(dqkv).double()
    cd, cw = float("inf"), float("inf")
    for b in range(B):
        ref = tok[b] @ w.double()
        out = torch.full((n, d), float("nan"), dtype=torch.bfloat16, device=DEV)
        ops.qkv_dgrad(dqkv, w, n, heads, batch_index=b, batch=B, out=out)
        f, u = check_bf16(out, ref, worst_d)
        assert f <= BF16_FROB and u <= BF16_ULPS, (b, f, u)
        out2 = torch.empty_like(out)
        ops.qkv_dgrad(dqkv, w, n, heads, batch_index=b, batch=B, out=out2)
        assert torch.equal(out, out2)
        x = rnd((n, d), g)
        prefill = torch.randn(3 * d, d, device=DEV, generator=g) * n ** 0.5
        dw = prefill.clone()
        ops.qkv_wgrad(dqkv, x, dw, n, heads, batch_index=b, batch=B)
        got = dw.double() - prefill.double()
        refw = tok[b].t() @ x.double()
        f, m, t = check_f32(got, refw, worst_w)
        assert f <= F32_FROB and m <= F32_MAX and t <= F32_LOCAL, (b, f, m, t)
        # negative controls: the neighbouring sample when there is one, else the Q gradient of head 0 dropped
        if B > 1:
            o = (b + 1) % B
            badd, badw = tok[o] @ w.double(), tok[o].t() @ x.double()
        else:
            t0 = tok[b].clone()
            t0[:, :64] = 0
            badd, badw = t0 @ w.double(), t0.t() @ x.double()
        cd, cw = min(cd, bf16_ulps(out, badd)), min(cw, tile_frob(got, badw))
    return cd, cw


QKV_SHAPES = [(H, n) for H in (1, 2, 6, 12, 16) for n in (72, 130, 216, 1000, 7168)] + [(6, 20480)]


@pytest.mark.parametrize("H,n", QKV_SHAPES)
def test_qkv_dgrad_and_wgrad_head_major_match_fp64(ops, H, n):
    """QKV input and weight gradients read straight from the head-major [3,B,H,n,64] attention-gradient buffer (4-D tensor map,
    a_part_stride across the batch) for B = 1, 2, 3 and every batch_index, against the token-major fp64 products."""
    worst_d, worst_w, cd, cw = {}, {}, float("inf"), float("inf")
    for B in (1, 2, 3):
        g = torch.Generator(device=DEV).manual_seed(H * 100003 + n * 7 + B)
        dqkv = rnd((3, B, H, n, 64), g)
        a, b = _qkv_case(ops, dqkv, H, worst_d, worst_w, g)
        cd, cw = min(cd, a), min(cw, b)
    report(f"qkv_dgrad H={H} n={n}", worst_d, dict(frob=BF16_FROB, ulps=BF16_ULPS))
    report(f"qkv_wgrad H={H} n={n}", worst_w, dict(frob=F32_FROB, maxrel=F32_MAX, local=F32_LOCAL))
    print(f"  negative control (wrong sample / head dropped): dgrad {cd:.2e} ulps, wgrad worst-tile {cw:.2e}")
    assert cd >= CONTROL * BF16_ULPS and cw >= CONTROL * F32_LOCAL


@pytest.mark.parametrize("H,n", [(12, 216), (12, 1000), (6, 130)])
def test_qkv_gradients_heads32_call_pattern(ops, H, n):
    """head_dim 32 (V-JEPA predictor): the attention gradient [3,B,H,n,64] rows {head, pad} are squeezed to [3,B,H/2,n,64]
    (two heads per row, bit-exact) and the QKV gradients are taken with H // 2 heads."""
    B = 2
    g = torch.Generator(device=DEV).manual_seed(H + n)
    full = rnd((3, B, H, n, 64), g)
    full[..., 32:] = 0
    sq = ops.heads32_squeeze(full)
    want = full.view(3, B, H // 2, 2, n, 64)[..., :32].permute(0, 1, 2, 4, 3, 5).reshape(3, B, H // 2, n, 64)
    assert torch.equal(sq, want)
    worst_d, worst_w = {}, {}
    cd, cw = _qkv_case(ops, sq, H // 2, worst_d, worst_w, g)
    report(f"heads32 qkv_dgrad H={H} n={n}", worst_d, dict(frob=BF16_FROB, ulps=BF16_ULPS))
    report(f"heads32 qkv_wgrad H={H} n={n}", worst_w, dict(frob=F32_FROB, maxrel=F32_MAX, local=F32_LOCAL))
    print(f"  negative control (wrong sample): dgrad {cd:.2e} ulps, wgrad worst-tile {cw:.2e}")
    assert cd >= CONTROL * BF16_ULPS and cw >= CONTROL * F32_LOCAL


# =====================================================================================================================
# 2. LayerNorm backward
# =====================================================================================================================
def _ln_bwd_ref(dy, x, mean, rstd, gamma):
    """closed-form LayerNorm backward in fp64 with the given statistics -> (dx, dgamma, dbeta, dgamma / dbeta term norms)."""
    x, dy, gamma = x.double(), dy.double(), gamma.double()
    mu, rs = mean.double()[:, None], rstd.double()[:, None]
    xh = (x - mu) * rs
    gg = dy * gamma
    dx = rs * (gg - gg.mean(1, keepdim=True) - xh * (gg * xh).mean(1, keepdim=True))
    return dx, (dy * xh).sum(0), dy.sum(0), ((dy * xh) ** 2).sum(0).sqrt(), (dy ** 2).sum(0).sqrt()


LN_CASES = [(d, (1, 5, 7, 9, 33, 1031)) for d in (8, 40, 136, 384, 512, 520, 768, 896, 1024)] + [(768, (7168,)), (384, (20480, 13312))]


@pytest.mark.parametrize("d,Ms", LN_CASES)
def test_layernorm_backward_matches_fp64(ops, d, Ms):
    """rows kernel (dres (+)= dx and its bf16 copy, every NV case incl. the rounded-up d = 520 / 896) and the reduce-add
    dgamma / dbeta kernel, with the statistics `layernorm_fwd(save_stats=True)` returned; accumulate and want_bf16 both ways."""
    eps = 1e-6
    row = lambda a, b: tile_frob(a, b, 1, d)  # noqa: E731
    wd, wp, ctrl = {}, {}, float("inf")
    for M in Ms:
        g = torch.Generator(device=DEV).manual_seed(M * 1009 + d)
        x = torch.randn(M, d, device=DEV, generator=g) * 3 + 1
        gamma, beta = torch.randn(d, device=DEV, generator=g), torch.randn(d, device=DEV, generator=g)
        _, mean, rstd = ops.layernorm_fwd(x, gamma, beta, eps, save_stats=True)
        dy = rnd((M, d), g)
        if M == Ms[0]:  # the closed form is the autograd of F.layer_norm (fp64, exact statistics)
            xr = x.double().requires_grad_(True)
            F.layer_norm(xr, (d,), gamma.double(), beta.double(), eps).backward(dy.double())
            mu, var = x.double().mean(1), x.double().var(1, unbiased=False)
            assert frob(_ln_bwd_ref(dy, x, mu, 1 / torch.sqrt(var + eps), gamma)[0], xr.grad) <= 1e-10
        dx, dgr, dbr, sg, sb = _ln_bwd_ref(dy, x, mean, rstd, gamma)
        for accumulate in (False, True):
            for want_bf16 in (True, False):
                prev = torch.randn(M, d, device=DEV, generator=g) * float(dx.abs().max())
                dres = prev.clone() if accumulate else torch.full((M, d), float("nan"), device=DEV)
                # accumulators at the scale of what is added, so that their own rounding stays below the bound
                pg, pb = torch.randn(d, device=DEV, generator=g) * sg.float(), torch.randn(d, device=DEV, generator=g) * sb.float()
                dgam, dbet = pg.clone(), pb.clone()
                db = ops.layernorm_bwd(dy, x, mean, rstd, gamma, dres, accumulate, dgam, dbet, want_bf16=want_bf16)
                got = dres.double() - (prev.double() if accumulate else 0)
                f, m, r = check_f32(got, dx, wd, local=row)
                assert f <= F32_FROB and m <= F32_MAX and r <= F32_LOCAL, (M, accumulate, f, m, r)
                assert (db is None) != want_bf16 and (db is None or torch.equal(db, dres.bfloat16()))
                for gotp, prevp, refp, scale in ((dgam, pg, dgr, sg), (dbet, pb, dbr, sb)):
                    gp = gotp.double() - prevp.double()
                    f, m, c = check_f32(gp, refp, wp, local=lambda a, b, s=scale: col_rel(a, b, s))
                    assert f <= F32_FROB and m <= F32_MAX and c <= COL_REL, (M, f, m, c)
                # reproducibility: the rows kernel is bit-identical, dgamma / dbeta equal up to summation order
                dres2 = prev.clone() if accumulate else torch.empty(M, d, device=DEV)
                dgam2, dbet2 = pg.clone(), pb.clone()
                db2 = ops.layernorm_bwd(dy, x, mean, rstd, gamma, dres2, accumulate, dgam2, dbet2, want_bf16=want_bf16)
                assert torch.equal(dres2, dres) and (db is None or torch.equal(db2, db))
                rep = max(frob(dgam2, dgam), frob(dbet2, dbet))
                wp["repro"] = max(wp.get("repro", 0), rep)
                assert rep <= REPRO_TOL
        # negative control: the mean of one row shifted by one standard deviation
        mb = mean.clone()
        mb[M // 2] += 1 / rstd[M // 2]
        ctrl = min(ctrl, row(got, _ln_bwd_ref(dy, x, mb, rstd, gamma)[0]))
    report(f"layernorm_bwd dres d={d}", wd, dict(frob=F32_FROB, maxrel=F32_MAX, local=F32_LOCAL))
    report(f"layernorm_bwd dgamma/dbeta d={d}", wp, dict(frob=F32_FROB, maxrel=F32_MAX, local=COL_REL, repro=REPRO_TOL))
    print(f"  negative control (one row's mean shifted by 1 std): worst-row frob-rel {ctrl:.2e}")
    assert ctrl >= CONTROL * F32_LOCAL


# =====================================================================================================================
# 3. reductions and data movement
# =====================================================================================================================
def _colsum_check(ops, x2d, M, N, ld, worst):
    """ops.colsum over x2d (rows of ld elements, the first N used) vs fp64; returns the negative-control ratio."""
    g = torch.Generator(device=DEV).manual_seed(M * 31 + N)
    rows = x2d[:M, :N].double()
    ref, scale = rows.sum(0), (rows ** 2).sum(0).sqrt()
    prefill = torch.randn(N, device=DEV, generator=g)
    out = prefill.clone()
    ops.colsum(x2d, out, M=M, N=N, ld=ld)
    got = out.double() - prefill.double()
    f, m, c = check_f32(got, ref, worst, local=lambda a, b: col_rel(a, b, scale))
    assert f <= F32_FROB and m <= F32_MAX and c <= COL_REL, (M, N, ld, f, m, c)
    out2 = prefill.clone()
    ops.colsum(x2d, out2, M=M, N=N, ld=ld)
    rep = frob(out2, out)
    worst["repro"] = max(worst.get("repro", 0), rep)
    assert rep <= REPRO_TOL
    r0 = (M // 2) // 64 * 64  # negative control: one 64-row block missing
    return col_rel(got, ref - rows[r0:r0 + 64].sum(0), scale)


@pytest.mark.parametrize("dtype", ["bf16", "f32"])
def test_colsum_matches_fp64(ops, dtype):
    """bias / mask-token gradients: out[N] += column sums.  bf16: one row block (M < 64) with warps on the two-rows-in-flight
    loop next to warps on the single-row tail (M = 9, 17); fp32: N % 4 == 0 but not % 128.  Both with ld > N, fp32 also on a
    row range of a wider buffer (the mask-token gradient reads rows n_vis.. of the decoder gradient)."""
    worst, ctrl = {}, float("inf")
    if dtype == "bf16":
        Ns, Ms, dt, lds = (8, 40, 264, 768, 4096), (1, 2, 9, 17, 31, 33, 1000, 20480), torch.bfloat16, (0, 24)
    else:
        Ns, Ms, dt, lds = (4, 36, 388, 900), (1, 7, 64, 65, 1000, 13312), torch.float32, (0, 12)
    for N in Ns:
        for M in Ms:
            for extra in lds:
                g = torch.Generator(device=DEV).manual_seed(N * M + extra)
                x = rnd((M, N + extra), g, dtype=dt)
                ctrl = min(ctrl, _colsum_check(ops, x, M, N, N + extra, worst))
    if dtype == "f32":  # a row range [r0:] of a wider [R, ld] buffer
        g = torch.Generator(device=DEV).manual_seed(5)
        big = rnd((2000, 400), g, dtype=dt)
        ctrl = min(ctrl, _colsum_check(ops, big[700:], 1300, 388, 400, worst))
    report(f"colsum {dtype}", worst, dict(frob=F32_FROB, maxrel=F32_MAX, local=COL_REL, repro=REPRO_TOL))
    print(f"  negative control (one 64-row block missing): per-column error {ctrl:.2e}")
    assert ctrl >= CONTROL * COL_REL


@pytest.mark.parametrize("skip_k", [False, True])
def test_colsum_heads_matches_fp64(ops, skip_k):
    """q / v bias gradients straight from the head-major [3,B,H,n,64] buffer; with skip_k the K third stays bit-identical."""
    worst, ctrl = {}, float("inf")
    for B in (1, 3):
        for H in (1, 12):
            for n in (1, 37, 130, 1000):
                g = torch.Generator(device=DEV).manual_seed(B * 1000 + H * 10 + n)
                dqkv = rnd((3, B, H, n, 64), g)
                xd = dqkv.double()
                ref, scale = xd.sum((1, 3)).reshape(-1), (xd ** 2).sum((1, 3)).sqrt().reshape(-1)
                prefill = torch.randn(3 * H * 64, device=DEV, generator=g)
                out = prefill.clone()
                ops.colsum_heads(dqkv, out, skip_k=skip_k)
                got = out.double() - prefill.double()
                parts = [0, 2] if skip_k else [0, 1, 2]
                sel = torch.cat([torch.arange(p * H * 64, (p + 1) * H * 64, device=DEV) for p in parts])
                f, m, c = check_f32(got[sel], ref[sel], worst, local=lambda a, b: col_rel(a, b, scale[sel]))
                assert f <= F32_FROB and m <= F32_MAX and c <= COL_REL, (B, H, n, f, m, c)
                if skip_k:
                    assert torch.equal(out[H * 64:2 * H * 64], prefill[H * 64:2 * H * 64])
                bad = ref.clone()  # negative control: a 64-token block of (part 0, sample 0, head 0) missing
                bad[:64] -= xd[0, 0, 0, :64].sum(0)
                ctrl = min(ctrl, col_rel(got[:64], bad[:64], scale[:64]))
    report(f"colsum_heads skip_k={skip_k}", worst, dict(frob=F32_FROB, maxrel=F32_MAX, local=COL_REL))
    print(f"  negative control (one 64-token block missing): per-column error {ctrl:.2e}")
    assert ctrl >= CONTROL * COL_REL


def test_token_sum_matches_fp64_and_is_bit_reproducible(ops):
    """per-sample token sums (numerator of the mean pooling) at ragged N; fixed-order reduction, so a second call is
    bit-identical."""
    worst, ctrl = {}, float("inf")
    for B in (1, 3):
        for N in (1, 127, 129, 1000, 20480):
            for d in (4, 388, 768):
                g = torch.Generator(device=DEV).manual_seed(B + N + d)
                x = torch.randn(B, N, d, device=DEV, generator=g)
                xd = x.double()
                ref, scale = xd.sum(1), (xd ** 2).sum(1).sqrt()
                out = ops.token_sum(x)
                f, m, c = check_f32(out, ref, worst, local=lambda a, b: col_rel(a, b, scale))
                assert f <= F32_FROB and m <= F32_MAX and c <= COL_REL, (B, N, d, f, m, c)
                assert torch.equal(ops.token_sum(x), out)
                r0 = (N // 2) // 64 * 64
                ctrl = min(ctrl, col_rel(out, ref - xd[:, r0:r0 + 64].sum(1), scale))
    report("token_sum", worst, dict(frob=F32_FROB, maxrel=F32_MAX, local=COL_REL))
    print(f"  negative control (one 64-row block missing): per-column error {ctrl:.2e}")
    assert ctrl >= CONTROL * COL_REL


def test_gather_patches_is_patchify_rounded_to_bf16(ops):
    """im2col rows of the patch-embedding weight gradient: bit-exact `patchify` rows (bf16) of the selected tokens, B = 2, a
    non-cubic volume, idx_stride > n_sel."""
    B, T, H, W = 2, 48, 32, 64  # 3 x 2 x 4 = 24 patches per sample
    g = torch.Generator(device=DEV).manual_seed(3)
    vol = torch.randn(B, T, H, W, device=DEV, generator=g)
    n_sel, stride = 9, 16
    idx = torch.stack([torch.randperm(24, device=DEV, generator=g)[:stride] for _ in range(B)]).to(torch.int32)
    out = ops.gather_patches(vol, idx, n_sel)
    cfg = types.SimpleNamespace(tubelet_size=16, patch_size=16)
    P = vo.patchify(vol[:, :, None], cfg)  # [B, 24, 4096]
    want = torch.cat([P[b, idx[b, :n_sel].long()] for b in range(B)]).bfloat16()
    assert out.shape == (B * n_sel, 4096) and torch.equal(out, want)
    assert torch.equal(ops.gather_patches(vol, idx, n_sel), out)
    wrong = torch.cat([P[b, idx[b, 1:n_sel + 1].long()] for b in range(B)]).bfloat16()  # negative control: rows shifted by one
    assert not torch.equal(out, wrong)


def test_scatter_rows_is_the_adjoint_of_gather_rows(ops):
    """out[b, idx[b,k]] = src[b,k] for k < K, zero elsewhere; K < idx.shape[1] (the decoder's masked rows) and K = 0."""
    B, N, d, L = 2, 300, 388, 120
    g = torch.Generator(device=DEV).manual_seed(8)
    idx = torch.stack([torch.randperm(N, device=DEV, generator=g)[:L] for _ in range(B)]).to(torch.int32)
    for K in (L, 77, 0):
        src = torch.randn(B, K, d, device=DEV, generator=g)
        out = ops.scatter_rows(src, idx, N, K)
        want = torch.zeros(B, N, d, device=DEV)
        for b in range(B):
            want[b, idx[b, :K].long()] = src[b]
        assert torch.equal(out, want)
        if K:
            assert torch.equal(ops.gather_rows(out, idx[:, :K].contiguous()), src)
            assert not torch.equal(out, torch.roll(want, 1, dims=1))  # negative control


def test_cast_f32_scaled_and_scale_f32_are_exact(ops):
    """gradient casts: bf16 -> fp32 times a host scale (odd n: the scalar tail), and the in-place fp32 x *= device scalar;
    both bit-exact, nothing past n written."""
    g = torch.Generator(device=DEV).manual_seed(4)
    scale = 0.3333333432674408  # an fp32 value: the product of a bf16 and it is exact in fp64, so both roundings agree
    for n in (1, 3, 5, 4097, 1000003):
        src = rnd((n,), g)
        buf = torch.full((n + 8,), -7.0, device=DEV)
        buf[:n] = float("nan")
        ops.cast_f32_scaled(src, buf[:n], scale)
        assert torch.equal(buf[:n], src.float() * scale) and torch.equal(buf[n:], torch.full((8,), -7.0, device=DEV))
        assert not torch.equal(buf[:n], src.float() * 0.33)  # negative control: another scale
    for n in (4, 4 * 1000003):  # grid-stride: more float4 than the capped grid
        x = torch.randn(n, device=DEV, generator=g)
        s = torch.tensor(0.7, device=DEV)
        want = x * s
        assert torch.equal(ops.scale_f32_(x, s), want)
