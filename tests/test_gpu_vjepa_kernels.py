"""Kernel-level parity of the V-JEPA path (run with -m gpu on the B200 box): the rotary embedding `smbv_rope3d` (both
kernels, both directions, the predictor's doubled-row view), `smbv_heads32_convert`, `smbv_position_sort`,
`smbv_gather_rows_f32` / `smbv_scatter_rows_f32`, `smbv_l1_loss_f32`, and the rotary attention sublayer of
`training.block_forward_train` / `training.block_backward` stage by stage.  The whole-model tests of test_gpu_vjepa.py allow
2e-2 .. 1.5e-1 at a 64^3 fixture; here each kernel is compared with a float64 reference computed ON THE DEVICE from the exact
bf16 / fp32 operands it reads, at the ViT-L (512x512x320: 20 480 tokens, 16 heads of 64) and predictor (384 / 12) sizes.

Bounds (worst measured on one NVIDIA B200 at a 1000 W power limit in brackets):
  rotary map, both kernels, forward and transposed, per element: |got - ref| <= ROPE_BOUND x (1 bf16 ulp of ref + floor)
      [0.50 in every case], where floor = (|x_a| + |x_b|) (OMEGA_ULPS |theta| + SINCOS_ULPS + PRODUCT_ULPS) 2^-24 (1 + 2^-7)
      is what fp32 arithmetic can lose before the one bf16 rounding: omega = 1 / powf(10000, j / half) is off by <= 14.2
      units of 2^-24 (0.5 for j / half, amplified ln(10^4) = 9.2x by the power, 4 for powf, 0.5 for the reciprocal) and
      theta = p omega by 0.5 more; sincosf adds <= 2 ulp; the product and the fused add <= 1 unit each (x_a, x_b: the two
      inputs of the pair); pass-through tail elements, -0.0 among them, bit-unchanged;
  heads32 expand / squeeze (head-major and token-major), position sort, row gather / scatter: bit-exact, pad columns +0.0,
      rows a scatter does not list untouched;
  L1 loss: relative error of the mean <= (fp32 additions on the longest path + 18) 2^-24 (a sum of non-negative terms)
      [4.3e-8 at n = 1031, bound 1.1e-6; 2.2e-8 at 27 M elements, bound 2.4e-6]; dpred bit-exact sign(p - t) fp32(upstream / n);
  attention sublayer, each stage fed the kernels' own output of the stage before:
      rotated Q / K: the rotary bound  [0.50];
      attention output per element <= O_ULPS bf16 ulps with a 2^-8 row-rms floor (o_ulps of test_gpu_attention_kernels.py)
      [0.85], lse <= LSE_ABS  [1.9e-5];
      dQ / dK / dV per element <= D_ULPS with the term floors of test_gpu_attention_kernels.py  [1.97];
      after the transposed map: the rotary bound  [0.50];
      dh1 (the QKV dgrad GEMM) <= 1 bf16 ulp + 1e-5 max  [0.50];
      fused QKV bias gradient (Q, K and V slots) <= COL_REL of the L2 norm of the summed terms  [4.8e-5].
  K bias against the TRUE gradient (fp64 dK of the fp64 attention backward, fp64 transposed map, fp64 sum), per feature:
      <= 2 x 2^-8 sum_t |dK_t,f| (the two bf16 roundings of dK: attention-backward output, then the transposed map) + the
      colsum bound + sum_t of the attention-backward element bound, each over the feature and its rotation partner
      [2.3e-3 of the bound; Frobenius-rel to the true gradient 5.3e-3].
      A "K slot zeroed" control cannot be separated from this bound, and the bound is kept as derived: every feature of the K
      slot is a cancelling sum (sum_t dK_t is exactly 0 without the rotary map, because each row of the softmax backward sums
      to zero), and what the rotation leaves is only 1.6 - 4.6x the worst case of the two roundings alone, 0.20 - 0.58x once
      the attention-backward bound is added (at 1999 and at 20 480 tokens).  This cancellation is also why the whole-model tests
      of test_gpu_vjepa.py need 1.5e-1 for `key.bias` against an fp32 oracle, where the 2e-2 .. 7e-2 bounds cover every
      other tensor: every bf16 rounding upstream of dK is amplified by sum_t |dK_t| / |sum_t dK_t|.  At the stage level, against
      the kernels' own dK, a zeroed K slot fails the colsum bound by 2.7e4x.
Negative controls (each must fail its bound by >= 100x; smallest measured): the forward rotary map where the transpose belongs
5.9e5; `ids` tiled ([ids, ids]) in place of ids2 on the doubled view 1.5e6; wrong positions on the sublayer's Q / K 1.1e6;
dh1 without the dK third 1.4e4; K slot zeroed (stage bound) 2.7e4; L1 reference without the tail elements 4.2e3.  For the
exact kernels the control is a mismatch: a swapped real-head pair (99.9 % of the elements), ties in reverse order (>= 2268
ranks), the rows of the other sample (all elements), idx read with stride K instead of ldidx (>= 30 % of the rows).
Every output is written into a NaN-prefilled view (int32: -7) between guard regions that are checked afterwards; every
kernel here except the attention backward has a fixed partition, so a second call must give bit-identical output.  The module
runs in about 15 s on the B200.
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

GUARD, SENTINEL, INT_FILL = 256, 1232.0, -7
U24 = 2.0 ** -24
CONTROL = 100.0

ROPE_BOUND = 1.0
OMEGA_ULPS, SINCOS_ULPS, PRODUCT_ULPS = 15.0, 2.0, 2.0
O_ULPS, LSE_ABS, D_ULPS = 5.0, 2.5e-4, 5.0  # test_gpu_attention_kernels.py: o_ulps, lse, d_ulps
ROW_FLOOR = 2.0 ** -8
BF16_ULPS = 1.0
COL_REL = 1e-4

L1_BLOCKS, CTA_THREADS = 1184, 256  # vjepa_ops.cu: L1_BLOCKS; 256 threads per CTA
VITL = dict(gs=32, frames=320)  # 512 x 512 x 320 with 16^3 patches: 32 x 32 x 20 = 20 480 tokens
N_VITL = 20480


@pytest.fixture(scope="module")
def lib():
    assert torch.cuda.is_available()
    from smb_vision_b200 import load

    lib = load()
    assert lib.smbv_device_ok() == 0, lib.smbv_last_error()
    return lib


def call(name, *args):
    from smb_vision_b200._lib import call as _call

    _call(name, *args, torch.cuda.current_stream().cuda_stream)


def ptr(t):
    return 0 if t is None else t.data_ptr()


def guarded(shape, dtype):
    """(buffer, view): a view prefilled with NaN (int32: INT_FILL) between two guard regions of SENTINEL (16-byte aligned)."""
    n = math.prod(shape)
    buf = torch.full((n + 2 * GUARD,), SENTINEL, dtype=dtype, device=DEV)
    buf[GUARD:GUARD + n] = INT_FILL if dtype == torch.int32 else float("nan")
    return buf, buf[GUARD:GUARD + n].view(shape)


def guards_ok(buf):
    return bool((buf[:GUARD] == SENTINEL).all() and (buf[-GUARD:] == SENTINEL).all())


def bits(t):
    return t.view({torch.float32: torch.int32, torch.bfloat16: torch.int16, torch.int32: torch.int32}[t.dtype])


def same_bits(a, b):
    return torch.equal(bits(a), bits(b))


def report(name, worst, bound, ctrl=None):
    print(f"{name}: {worst:.3g} (bound {bound:.3g})" + ("" if ctrl is None else f"; negative control {ctrl:.3g} x bound"))


def ulp_bf16(ref):
    """one bf16 ulp (8 significant bits) of each element of a float64 tensor; 0 at ref == 0."""
    return torch.exp2(torch.floor(torch.log2(ref.abs())) - 7)


def max_ratio(err, den):
    return (err / den.clamp_min(1e-300)).max().item()


def kernel_names(fn):
    """names of the CUDA kernels `fn` launches (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events()}


def vjepa_max_pos(gs, frames, n_tokens=0):
    """vjepa.py's table length: min(max(grid, frames / 16, tokens / grid^2 + 1), 256) (encoder: n_tokens = 0)."""
    return min(max(gs, frames // 16, n_tokens // (gs * gs) + 1 if n_tokens else 0), 256)


# =====================================================================================================================
# 1. rotary embedding: smbv_rope3d
# =====================================================================================================================
def positions(ids, n, gs):
    t = torch.arange(n, device=DEV) if ids is None else ids.long()
    f = t // (gs * gs)
    rem = t - f * gs * gs
    hh = rem // gs
    return f, hh, rem - hh * gs


def rope_ref64(x, ids, gs, transpose):
    """float64 map of x [..., B, H, n, D] (any float dtype, read exactly) with ids [B, n] or None = arange(n), and the
    per-element fp32 floor of the module docstring.  Element e of a segment uses angle p omega[e mod S/2] (the reference
    tiles the S/2 angles twice while pairing adjacent elements)."""
    D, n = x.shape[-1], x.shape[-2]
    S = 2 * ((D // 3) // 2)
    h = S // 2
    xd = x.double()
    out, floor = xd.clone(), torch.zeros_like(xd)
    omega = torch.pow(10000.0, -torch.arange(h, dtype=torch.float64, device=DEV) / h)
    for k, p in enumerate(positions(ids, n, gs)):
        th = p.double()[..., None] * omega
        th = torch.cat([th, th], -1)
        if ids is not None:
            th = th[:, None]  # [B, 1, n, S]: the same ids for every head
        c, s = th.cos(), th.sin()
        seg = xd[..., k * S:(k + 1) * S]
        x0, x1 = seg[..., 0::2], seg[..., 1::2]
        c0, c1, s0, s1 = c[..., 0::2], c[..., 1::2], s[..., 0::2], s[..., 1::2]
        if not transpose:
            o0, o1 = x0 * c0 - x1 * s0, x1 * c1 + x0 * s1
        else:
            o0, o1 = x0 * c0 + x1 * s1, x1 * c1 - x0 * s0
        out[..., k * S:(k + 1) * S:2], out[..., k * S + 1:(k + 1) * S:2] = o0, o1
        eps = (OMEGA_ULPS * torch.maximum(th[..., 0::2], th[..., 1::2]) + SINCOS_ULPS + PRODUCT_ULPS) * U24
        e = (x0.abs() + x1.abs()) * eps * (1 + 2.0 ** -7)
        floor[..., k * S:(k + 1) * S:2], floor[..., k * S + 1:(k + 1) * S:2] = e, e
    return out, floor


def rope_metric(got, ref, floor):
    """max over elements of |got - ref| / (1 bf16 ulp of ref + floor)."""
    assert not torch.isnan(got).any()
    return max_ratio((got.double() - ref).abs(), ulp_bf16(ref) + floor)


def run_rope(x, gs, ids, max_pos, transpose, first_gen=False):
    """smbv_rope3d in place on a copy of x [G,B,H,n,D] inside a guarded buffer; returns the result."""
    G, B, H, n, D = x.shape
    buf, y = guarded(x.shape, torch.bfloat16)
    y.copy_(x)
    call("smbv_rope3d", ptr(y), ptr(ids), G, B, H, n, D, gs, max_pos, (1 if transpose else 0) | (2 if first_gen else 0))
    assert guards_ok(buf)
    return y


def rope_input(shape, g):
    """bf16 N(0,1) with -0.0 and +0.0 sprinkled through every column (the pass-through tail too)."""
    x = torch.randn(shape, device=DEV, generator=g).bfloat16()
    x.view(-1)[3::37] = -0.0
    x.view(-1)[5::41] = 0.0
    return x


def sorted_ids_with_ties(B, n, N, g):
    """sorted positions of a context and a target mask drawn independently from N tokens (overlaps = duplicate ids)."""
    a = n // 2
    rows = [torch.cat([torch.randperm(N, device=DEV, generator=g)[:a], torch.randperm(N, device=DEV, generator=g)[:n - a]])
            for _ in range(B)]
    return torch.stack(rows).sort(1).values.int().contiguous()


def check_rope(x, gs, ids, max_pos, name, v1_bits=True):
    """both directions of the default dispatch against fp64, tail bits, bit-identical repeat, the first-generation kernel's
    bits, and the control: the forward map where the transpose belongs.  Returns the worst metric."""
    D = x.shape[-1]
    tail = 3 * 2 * ((D // 3) // 2)
    worst, ctrl = 0.0, float("inf")
    for tr in (False, True):
        y = run_rope(x, gs, ids, max_pos, tr)
        ref, floor = rope_ref64(x, ids, gs, tr)
        worst = max(worst, rope_metric(y, ref, floor))
        assert same_bits(y[..., tail:], x[..., tail:])
        assert same_bits(run_rope(x, gs, ids, max_pos, tr), y)
        if v1_bits:
            assert same_bits(run_rope(x, gs, ids, max_pos, tr, first_gen=True), y)
        if tr:
            ref_bad, _ = rope_ref64(x, ids, gs, False)
            ctrl = rope_metric(y, ref_bad, floor)
        del ref, floor
    report(f"rope {name}", worst, ROPE_BOUND, ctrl / ROPE_BOUND)
    assert worst <= ROPE_BOUND
    assert ctrl >= CONTROL * ROPE_BOUND
    return worst


def test_rope_encoder_full_size(lib):
    """ViT-L encoder at 512x512x320: Q and K [2,1,16,20480,64], ids = None, grid 32, max_pos by vjepa.py's rule."""
    g = torch.Generator(device=DEV).manual_seed(1)
    x = rope_input((2, 1, 16, N_VITL, 64), g)
    check_rope(x, VITL["gs"], None, vjepa_max_pos(VITL["gs"], VITL["frames"]), "encoder [2,1,16,20480,64]")


def beyond_table_ids(B, n, gs, max_pos, g):
    """ids whose frame is inside the table for rows with (t // 32) even and beyond it otherwise: every 4-row batch of a
    rope3d_v2 thread (rows t, t + rpp, t + 2 rpp, t + 3 rpp, rpp = 32 or 64) mixes the fast and the per-element branch."""
    t = torch.arange(n, device=DEV)
    inside = torch.randint(0, max_pos * gs * gs, (B, n), device=DEV, generator=g)
    beyond = torch.randint(max_pos * gs * gs, 40 * max_pos * gs * gs, (B, n), device=DEV, generator=g)
    return torch.where(((t // 32) % 2 == 0)[None], inside, beyond).int().contiguous()


ROPE_CASES = [  # (name, D, (G, B, H, n), gs, ids kind, frames of the clip)
    ("predictor hd64 ties", 64, (2, 2, 6, 3001), 24, "ties", 256),
    ("predictor hd32 ties", 32, (2, 2, 12, 3001), 32, "ties", 320),
    ("clamp 256 hd32", 32, (2, 2, 4, 1031), 16, "long", 4800),
    ("clamp 256 hd64", 64, (2, 2, 4, 1031), 16, "long", 4800),
    ("beyond table hd64", 64, (2, 2, 3, 1031), 4, "beyond", 128),
    ("beyond table hd32", 32, (2, 2, 3, 1031), 4, "beyond", 128),
    ("ragged 20479 hd64", 64, (2, 1, 4, 20479), 32, None, 320),
    ("ragged 20479 hd32", 32, (2, 1, 4, 20479), 32, None, 320),
    ("grid 255", 64, (2, 2, 2, 1031), 255, "ties", 48),
    ("grid 256", 64, (2, 2, 2, 1031), 256, "ties", 48),
]


@pytest.mark.parametrize("name,D,shape,gs,kind,frames", ROPE_CASES, ids=[c[0] for c in ROPE_CASES])
def test_rope_geometries(lib, name, D, shape, gs, kind, frames):
    """Predictor geometry (sorted ids with duplicates, max_pos by vjepa.py's rule: 24, 32, and the 256 clamp of a 300-frame
    clip whose later frames run past the table), ids beyond the table mixed with ids inside it in every 4-row batch, ragged
    n (not a multiple of 512 nor of the rows per pass), grid 255 (the multiply-shift kernel) and 256 (the first-generation
    kernel by the dispatch rule)."""
    G, B, H, n = shape
    g = torch.Generator(device=DEV).manual_seed(D * 7 + n + gs)
    x = rope_input((G, B, H, n, D), g)
    n_tok = frames // 16 * gs * gs
    max_pos = vjepa_max_pos(gs, frames, n_tok if kind else 0)
    if kind == "beyond":
        max_pos = 8
        ids = beyond_table_ids(B, n, gs, max_pos, g)
    elif kind in ("ties", "long"):
        ids = sorted_ids_with_ties(B, n, n_tok, g)
    else:
        ids = None
    if kind == "long":
        assert max_pos == 256 and int(ids.max()) // (gs * gs) > 256
    check_rope(x, gs, ids, max_pos, f"{name} max_pos={max_pos}")


@pytest.mark.parametrize("n", [3001, N_VITL])
def test_rope_doubled_row_view(lib, n):
    """The predictor's head_dim-32 wiring (modeling.attention32_forward, training.block_backward): the QKV GEMM writes
    [3, B, H/2, n, 64] double heads, the kernel runs on Q and K viewed as [2, B, H/2, 2n, 32] with ids2 (every sorted id
    twice).  Against fp64 in the reference layout: real head h is columns (h % 2) 32 ... +31 of double head h / 2 and is
    rotated with ids.  Controls: the forward map where the transpose belongs; `ids` tiled ([ids, ids]) in place of ids2."""
    from smb_vision_b200 import ops

    B, H = 2, 12
    g = torch.Generator(device=DEV).manual_seed(n)
    qkv2 = rope_input((3, B, H // 2, n, 64), g)
    pos = torch.randint(0, N_VITL, (B, n), device=DEV, generator=g, dtype=torch.int32)
    pos[:, 1::3] = pos[:, 0::3][:, :pos[:, 1::3].shape[1]]  # duplicates
    _, _, ids, ids2 = ops.position_sort(pos.contiguous(), doubled=True)
    gs, max_pos = VITL["gs"], vjepa_max_pos(VITL["gs"], VITL["frames"], N_VITL)
    real = qkv2[:2].view(2, B, H // 2, n, 2, 32).permute(0, 1, 2, 4, 3, 5).reshape(2, B, H, n, 32)

    def doubled(t):  # [2, B, H, n, 32] (real heads) -> [2, B, H/2, 2n, 32] (the kernel's view)
        return t.view(2, B, H // 2, 2, n, 32).permute(0, 1, 2, 4, 3, 5).reshape(2, B, H // 2, 2 * n, 32)

    view = qkv2[:2].contiguous().view(2, B, H // 2, 2 * n, 32)
    assert torch.equal(doubled(real), view)
    worst, ctrl_ids, ctrl_tr = 0.0, float("inf"), float("inf")
    for tr in (False, True):
        y = run_rope(view, gs, ids2, max_pos, tr)
        assert same_bits(run_rope(view, gs, ids2, max_pos, tr), y)
        ref, floor = rope_ref64(real, ids, gs, tr)
        worst = max(worst, rope_metric(y, doubled(ref), doubled(floor)))
        bad, _ = rope_ref64(view, torch.cat([ids, ids], 1), gs, tr)
        ctrl_ids = min(ctrl_ids, rope_metric(y, bad, doubled(floor)))
        if tr:
            bad, _ = rope_ref64(real, ids, gs, False)
            ctrl_tr = rope_metric(y, doubled(bad), doubled(floor))
        assert same_bits(y.view(2, B, H // 2, n, 64)[..., 30:32], qkv2[:2, ..., 30:32])  # the tails of both real heads
        assert same_bits(y.view(2, B, H // 2, n, 64)[..., 62:], qkv2[:2, ..., 62:])
        del ref, floor, bad
    report(f"rope doubled view n={n}", worst, ROPE_BOUND, min(ctrl_ids, ctrl_tr) / ROPE_BOUND)
    print(f"  controls: ids in place of ids2 {ctrl_ids:.3g}, forward map in place of the transpose {ctrl_tr:.3g}")
    assert worst <= ROPE_BOUND
    assert ctrl_ids >= CONTROL * ROPE_BOUND and ctrl_tr >= CONTROL * ROPE_BOUND


@pytest.mark.parametrize("G,B,H", [(1, 5, 13107), (2, 4, 8192)])
def test_rope_dispatch_boundary(lib, G, B, H):
    """G*B*H = 65535 runs rope3d_v2_kernel (grid.y = G*B*H), 65536 the first-generation kernel; both against fp64 at a
    ragged n = 3, per-sample ids.  At 65536 the result must carry the multiply-shift kernel's bits, which it gives on the
    two halves G = 0 and G = 1 (32768 rows each); at 65535 the explicitly selected first-generation kernel agrees."""
    n, D, gs, max_pos = 3, 64, 4, 8
    g = torch.Generator(device=DEV).manual_seed(G * B * H)
    x = rope_input((G, B, H, n, D), g)
    ids = torch.randint(0, 12 * gs * gs, (B, n), device=DEV, generator=g, dtype=torch.int32)
    names = kernel_names(lambda: run_rope(x, gs, ids, max_pos, False))
    rope_kernels = {k for k in names if "rope3d" in k}
    want = "rope3d_v2_kernel" if G * B * H <= 65535 else "rope3d_kernel"
    print(f"rope G*B*H={G * B * H}: {sorted(rope_kernels)}")
    assert rope_kernels and all(want in k and (want != "rope3d_kernel" or "v2" not in k) for k in rope_kernels)
    worst = 0.0
    for tr in (False, True):
        y = run_rope(x, gs, ids, max_pos, tr)
        ref, floor = rope_ref64(x, ids, gs, tr)
        worst = max(worst, rope_metric(y, ref, floor))
        if G * B * H > 65535:
            halves = torch.cat([run_rope(x[i:i + 1], gs, ids, max_pos, tr) for i in range(G)])
            assert same_bits(y, halves)
        else:
            assert same_bits(y, run_rope(x, gs, ids, max_pos, tr, first_gen=True))
    report(f"rope dispatch G*B*H={G * B * H}", worst, ROPE_BOUND)
    assert worst <= ROPE_BOUND


# =====================================================================================================================
# 2. smbv_heads32_convert
# =====================================================================================================================
@pytest.mark.parametrize("n", [N_VITL, N_VITL - 1])
def test_heads32_convert_exact(lib, n):
    """Predictor size (B' = 2, 12 heads of 32): head-major expand [3, B', 6, n, 64] -> [3, B', 12, n, 64] with +0.0 pad
    columns, squeeze back (a non-zero pad is dropped), token-major [B', n, 384] <-> [B', n, 768]; bit-exact, guarded,
    repeatable.  Control: a reference with the two real heads of each double head swapped."""
    B, H = 2, 12
    g = torch.Generator(device=DEV).manual_seed(n)
    x = torch.randn(3, B, H // 2, n, 64, device=DEV, generator=g).bfloat16()
    want = x.view(3, B, H // 2, n, 2, 32).permute(0, 1, 2, 4, 3, 5).reshape(3, B, H, n, 32)
    outs = []
    for _ in range(2):
        buf, e = guarded((3, B, H, n, 64), torch.bfloat16)
        call("smbv_heads32_convert", ptr(x), ptr(e), 3 * B, H, n, 1, 1)
        assert guards_ok(buf)
        assert same_bits(e[..., :32], want) and (bits(e[..., 32:]) == 0).all()
        outs.append(e)
    assert same_bits(outs[0], outs[1])
    swapped = want.view(3, B, H // 2, 2, n, 32).flip(3).reshape(3, B, H, n, 32)
    ctrl = (bits(outs[0][..., :32]) != bits(swapped)).double().mean().item()
    padded = outs[0].clone()
    padded[..., 32:] = torch.randn(3, B, H, n, 32, device=DEV, generator=g).bfloat16()
    buf, s = guarded((3, B, H // 2, n, 64), torch.bfloat16)
    call("smbv_heads32_convert", ptr(padded), ptr(s), 3 * B, H, n, 1, 0)
    assert guards_ok(buf) and same_bits(s, x)
    # token-major: [B', n, H*32] <-> [B', n, H*64]
    t = torch.randn(B, n, H * 32, device=DEV, generator=g).bfloat16()
    buf, te = guarded((B, n, H * 64), torch.bfloat16)
    call("smbv_heads32_convert", ptr(t), ptr(te), B, H, n, 0, 1)
    assert guards_ok(buf)
    te4 = te.view(B, n, H, 64)
    assert same_bits(te4[..., :32], t.view(B, n, H, 32)) and (bits(te4[..., 32:]) == 0).all()
    te4[..., 32:] = 3.0
    buf, ts = guarded((B, n, H * 32), torch.bfloat16)
    call("smbv_heads32_convert", ptr(te), ptr(ts), B, H, n, 0, 0)
    assert guards_ok(buf) and same_bits(ts, t)
    print(f"heads32 n={n}: bit-exact; negative control (swapped head pair) mismatches {ctrl:.3f} of the elements")
    assert ctrl > 0.9


# =====================================================================================================================
# 3. smbv_position_sort
# =====================================================================================================================
def run_sort(pos, doubled=True):
    B, n = pos.shape
    bufs, views = zip(*(guarded(s, torch.int32) for s in [(B, n)] * 3 + [(B, 2 * n)]))
    call("smbv_position_sort", ptr(pos), B, n, ptr(views[0]), ptr(views[1]), ptr(views[2]), ptr(views[3]) if doubled else 0)
    assert all(guards_ok(b) for b in bufs)
    return views


SORT_CASES = [("random ties", 4, N_VITL), ("default masks", 4, N_VITL), ("ragged", 4, N_VITL - 77), ("ragged small", 3, 1000),
              ("single token", 3, 1)]


@pytest.mark.parametrize("name,B,n", SORT_CASES, ids=[c[0] for c in SORT_CASES])
def test_position_sort_exact(lib, name, B, n):
    """order / inv / sorted / sorted2 exact against torch.argsort(stable=True) on the device, at B' = 2 samples x 2 mask
    pairs and n = 20 480 (random positions with ties; the reference's default masks, arange twice, so every id appears
    twice), n not a multiple of 256, and one-token rows; sorted2 = NULL leaves the other outputs unchanged; a second call
    gives the same bits.  Control: ties broken in reverse index order."""
    g = torch.Generator(device=DEV).manual_seed(n + B)
    if name == "default masks":
        pos = torch.arange(n // 2, device=DEV, dtype=torch.int32).repeat(B, 2)
    else:
        pos = torch.randint(0, max(2, n // 2), (B, n), device=DEV, generator=g, dtype=torch.int32)
    pos = pos.contiguous()
    order, inv, srt, s2 = run_sort(pos)
    want = torch.argsort(pos.long(), dim=1, stable=True)
    assert torch.equal(order.long(), want)
    assert torch.equal(inv.long(), torch.argsort(want, dim=1))
    assert torch.equal(srt, torch.gather(pos, 1, want))
    assert torch.equal(s2, srt.repeat_interleave(2, dim=1))
    again = run_sort(pos)
    assert all(same_bits(a, b) for a, b in zip(again, (order, inv, srt, s2)))
    o3, i3, s3, n3 = run_sort(pos, doubled=False)
    assert same_bits(o3, order) and same_bits(i3, inv) and same_bits(s3, srt) and bool((n3 == INT_FILL).all())
    idx = torch.arange(n, device=DEV)
    bad = torch.argsort(pos.long() * n + (n - 1 - idx), dim=1)
    ctrl = int((order.long() != bad).sum())
    print(f"position_sort {name} B={B} n={n}: exact; " + (f"negative control (reversed ties) {ctrl} mismatching ranks" if n > 1 else "no ties"))
    assert n == 1 or ctrl > 0


def test_position_sort_argument_checks(lib):
    """B > 65535 (the grid's y limit), B = 0 and n = 0 are refused on the host before any launch; the outputs stay as
    they were."""
    from smb_vision_b200._lib import SmbvError

    B = 65536
    pos = torch.zeros(B, dtype=torch.int32, device=DEV)
    outs = [torch.full((2 * B,), INT_FILL, dtype=torch.int32, device=DEV) for _ in range(4)]
    for b, n in ((B, 1), (0, 1), (1, 0)):
        with pytest.raises(SmbvError):
            call("smbv_position_sort", ptr(pos), b, n, *(ptr(o) for o in outs))
    torch.cuda.synchronize()
    assert all(bool((o == INT_FILL).all()) for o in outs)


# =====================================================================================================================
# 4. smbv_gather_rows_f32 / smbv_scatter_rows_f32
# =====================================================================================================================
def test_gather_rows_full_size(lib):
    """out[b, k] = src[b, idx[b, k]] at d = 1024, K = 12 345 of N = 20 480 (unsorted, distinct), bit-exact, guarded,
    repeatable.  Control: the rows of the other sample."""
    B, N, K, d = 2, N_VITL, 12345, 1024
    g = torch.Generator(device=DEV).manual_seed(4)
    src = torch.randn(B, N, d, device=DEV, generator=g)
    idx = torch.stack([torch.randperm(N, device=DEV, generator=g)[:K] for _ in range(B)]).int().contiguous()
    want = torch.gather(src, 1, idx.long()[..., None].expand(B, K, d))
    outs = []
    for _ in range(2):
        buf, out = guarded((B, K, d), torch.float32)
        call("smbv_gather_rows_f32", ptr(src), ptr(idx), B, N, K, d, ptr(out))
        assert guards_ok(buf) and same_bits(out, want)
        outs.append(out)
    assert same_bits(outs[0], outs[1])
    bad = torch.gather(src.flip(0), 1, idx.long()[..., None].expand(B, K, d))
    ctrl = (outs[0] != bad).double().mean().item()
    print(f"gather_rows K={K} d={d}: bit-exact; negative control (other sample) mismatches {ctrl:.3f} of the elements")
    assert ctrl > 0.9


SCATTER_CASES = [  # (name, B, N, K, ldidx, d)
    ("predictor dXt -> sorted rows", 2, N_VITL, 12345, 12345, 1024),
    ("MIM decoder dG -> masked rows, ldidx N", 2, N_VITL, 15360, N_VITL, 1024),
    ("ldidx > K, d 384", 3, 1000, 257, 999, 384),
]


@pytest.mark.parametrize("name,B,N,K,ldidx,d", SCATTER_CASES, ids=[c[0] for c in SCATTER_CASES])
def test_scatter_rows_exact(lib, name, B, N, K, ldidx, d):
    """out[b, idx[b, k]] = src[b, k] for k < K, reading idx with row stride ldidx: the predictor's
    scatter_rows(dXt, inv_tgt, n_tot) and the MIM decoder's scatter_rows(dG, msk, N, n_mask) (idx rows of N entries, the
    first n_mask of them used).  Into a NaN-prefilled guarded output: listed rows bit-exact, every other row still NaN (the
    kernel never writes it; ops.scatter_rows zero-fills it first, also checked); repeatable.  Control: idx read with stride
    K instead of ldidx."""
    from smb_vision_b200 import ops

    g = torch.Generator(device=DEV).manual_seed(K + ldidx)
    src = torch.randn(B, K, d, device=DEV, generator=g)
    idx = torch.stack([torch.randperm(N, device=DEV, generator=g)[:ldidx] for _ in range(B)]).int().contiguous()
    used = idx[:, :K].long()
    outs = []
    for _ in range(2):
        buf, out = guarded((B, N, d), torch.float32)
        call("smbv_scatter_rows_f32", ptr(src), ptr(idx), B, N, K, ldidx, d, ptr(out))
        assert guards_ok(buf)
        assert same_bits(torch.gather(out, 1, used[..., None].expand(B, K, d)), src)
        listed = torch.zeros(B, N, dtype=torch.bool, device=DEV).scatter_(1, used, True)
        assert bool(torch.isnan(out[~listed]).all())
        outs.append(out)
    assert same_bits(outs[0], outs[1])
    z = ops.scatter_rows(src, idx, N, K)
    assert same_bits(z[listed], outs[0][listed]) and bool((bits(z[~listed]) == 0).all())
    msg = "(ldidx = K: no stride control)"
    if ldidx != K:
        flat = idx.view(-1)[:B * K].view(B, K).long()
        bad = torch.zeros(B, N, d, device=DEV).scatter_(1, flat[..., None].expand(B, K, d), src)
        ctrl = (outs[0].nan_to_num(0.0) != bad).any(-1).double().mean().item()
        msg = f"negative control (idx read with stride K) rows differing {ctrl:.3f}"
        assert ctrl > 0
    print(f"scatter_rows {name}: bit-exact, unlisted rows untouched; {msg}")


# =====================================================================================================================
# 5. smbv_l1_loss_f32
# =====================================================================================================================
def l1_rel_bound(n):
    """fp32 additions on the longest path of one element into the loss (module docstring) x 2^-24."""
    iters = -(-(n // 4) // (L1_BLOCKS * CTA_THREADS))
    return (iters + 18) * U24


L1_FULL = 13312 * 1024 * 2  # predictor output [B' = 2, 13 312 target tokens, 1024]
L1_SIZES = [L1_FULL, L1_FULL - 1, L1_FULL - 2, L1_FULL - 3, 1, 2, 3, 1031, 4 * L1_BLOCKS * CTA_THREADS + 6]


@pytest.mark.parametrize("n", L1_SIZES)
def test_l1_loss_matches_fp64(lib, n):
    """mean |pred - target| against the fp64 mean, for n % 4 = 0 .. 3 (the n % 4 trailing elements belong to the last CTA;
    n < 4: nothing but the tail), upstream 3 and 0.37: dpred bit-exact sign(p - t) * fp32(upstream / n) with sign(0) = 0,
    guarded, a second call bit-identical.  The tail elements carry ~1 % of the sum, so that the control — the reference
    without them — is visible at every n."""
    g = torch.Generator(device=DEV).manual_seed(n)
    p = torch.randn(n, device=DEV, generator=g)
    t = torch.randn(n, device=DEV, generator=g)
    r = n % 4
    body = n - r
    t[:body:7] = p[:body:7]  # exact ties: gradient 0
    if r:
        t[body:] = p[body:] - torch.tensor([1.0, -1.0, 1.0], device=DEV)[:r] * (0.01 * n / r + 1.0)
    ad = (p.double() - t.double()).abs()
    ref = ad.mean().item()
    bound = l1_rel_bound(n)
    worst, ctrl = 0.0, None
    for up in (3.0, 0.37):
        res = []
        for _ in range(2):
            lb, loss = guarded((1,), torch.float32)
            db, dp = guarded((n,), torch.float32)
            wb, ws = guarded((L1_BLOCKS,), torch.float32)
            call("smbv_l1_loss_f32", ptr(p), ptr(t), n, ptr(ws), ptr(loss), ptr(dp), up)
            assert guards_ok(lb) and guards_ok(db) and guards_ok(wb)
            res.append((loss.clone(), dp.clone()))
        assert same_bits(res[0][0], res[1][0]) and same_bits(res[0][1], res[1][1])
        loss, dp = res[0]
        worst = max(worst, abs(loss.item() - ref) / ref)
        gscale = torch.tensor(torch.tensor(up, dtype=torch.float32).item() / n, dtype=torch.float32).item()  # fp32(fp32(up) / n)
        want = torch.sign(p.double() - t.double()).float() * gscale
        assert same_bits(dp, want), int((bits(dp) != bits(want)).sum())
        assert bool((dp[:body:7] == 0).all())
        if r:
            drop = ad[:body].sum().item() / n
            ctrl = abs(loss.item() - drop) / ref / bound
    report(f"l1_loss n={n} (n % 4 = {r})", worst, bound, ctrl)
    assert worst <= bound
    if r:
        assert ctrl >= CONTROL


# =====================================================================================================================
# 6. the rotary attention sublayer: training.block_forward_train / block_backward
# =====================================================================================================================
def heads_of(t, B, H):
    """token-major [B, n, H*W] -> [B*H, n, W]"""
    n = t.shape[1]
    return t.view(B, n, H, -1).permute(0, 2, 1, 3).reshape(B * H, n, -1)


def attn_ref64(q, k, v, o, do, lse, scale):
    """q, k, v, o, do [BH, N, 64] bf16 (o, lse: what the backward kernel reads, i.e. the forward kernel's), lse [BH, N] fp32.
    -> fp64 forward O, lse of softmax(scale q k^T) v; the backward from the given O and lse: dq, dk, dv and the L2 norms of
    the terms summed into each element tq, tk, tv (the definitions of test_gpu_attention_kernels.reference)."""
    BH, N, D = q.shape
    qd, kd, vd, dod, od = (t.double() for t in (q, k, v, do, o))
    z = lambda: torch.zeros(BH, N, D, dtype=torch.float64, device=DEV)  # noqa: E731
    r = dict(o=z(), lse=torch.zeros(BH, N, dtype=torch.float64, device=DEV), dq=z(), dk=z(), dv=z(), tq=z(), tk=z(), tv=z())
    R = max(128, (2 ** 26 // (BH * N)) // 128 * 128)
    for r0 in range(0, N, R):
        sl = slice(r0, min(N, r0 + R))
        s = torch.bmm(qd[:, sl], kd.transpose(1, 2)) * scale
        ls = torch.logsumexp(s, -1, keepdim=True)
        r["o"][:, sl], r["lse"][:, sl] = torch.bmm(torch.exp(s - ls), vd), ls[..., 0]
        p = torch.exp(s - lse[:, sl].double()[..., None])
        del s
        dp = torch.bmm(dod[:, sl], vd.transpose(1, 2))
        dsum = (dod[:, sl] * od[:, sl]).sum(-1, keepdim=True)
        ds = p * (dp - dsum)
        r["dq"][:, sl] = scale * torch.bmm(ds, kd)
        r["dk"] += scale * torch.bmm(ds.transpose(1, 2), qd[:, sl])
        r["dv"] += torch.bmm(p.transpose(1, 2), dod[:, sl])
        dabs = (dod[:, sl] * od[:, sl]).abs().sum(-1, keepdim=True)
        a2 = (ds.abs() + 2.0 ** -16 * p * (torch.bmm(dod[:, sl].abs(), vd.abs().transpose(1, 2)) + dabs)) ** 2
        r["tq"][:, sl] = scale * torch.bmm(a2, kd ** 2).sqrt()
        r["tk"] += torch.bmm(a2.transpose(1, 2), qd[:, sl] ** 2)
        r["tv"] += torch.bmm((p * p).transpose(1, 2), dod[:, sl] ** 2)
        del p, ds, dp, a2
    r["tk"], r["tv"] = scale * r["tk"].sqrt(), r["tv"].sqrt()
    return r


def ulps_floor(ref, term=None, row_floor=True):
    """per element: 1 bf16 ulp of ref + ROW_FLOOR x max(rms of the row, term) + 1e-5 max|ref| (rows = last dim)."""
    ref = ref.double()
    f = ulp_bf16(ref) + 1e-5 * ref.abs().max()
    if row_floor:
        rms = ref.pow(2).mean(-1, keepdim=True).sqrt()
        f = f + ROW_FLOOR * (rms if term is None else torch.maximum(rms, term.double()))
    return f


class Spy:
    """Records what the sublayer hands to the kernels it calls (ops.rope3d_, ops.flash_attn_bwd, ops.qkv_dgrad,
    ops.layernorm_bwd) without changing a bit of it."""

    def __init__(self, monkeypatch):
        from smb_vision_b200 import ops

        self.rope, self.bwd, self.dgrad, self.ln_dy = [], [], [], []
        real_rope, real_bwd, real_dgrad, real_lnb = ops.rope3d_, ops.flash_attn_bwd, ops.qkv_dgrad, ops.layernorm_bwd

        def rope(x, grid_size, ids=None, max_pos=64, transpose=False, first_generation_kernel=False):
            before = x.clone()
            real_rope(x, grid_size, ids, max_pos, transpose, first_generation_kernel)
            self.rope.append(dict(before=before, after=x.clone(), gs=grid_size, ids=ids, max_pos=max_pos, transpose=transpose))
            return x

        def bwd(q, k, v, o, dout, lse, scale, **kw):
            res = real_bwd(q, k, v, o, dout, lse, scale, **kw)
            self.bwd.append(dict(q=q, k=k, v=v, o=o, do=dout.clone(), lse=lse, scale=scale, d=[t.clone() for t in res]))
            return res

        def dgrad(dqkv, w, tokens, heads, batch_index=0, batch=1, out=None):
            if batch_index == 0:
                self.dgrad.append(dict(dqkv=dqkv.clone(), heads=heads))
            return real_dgrad(dqkv, w, tokens, heads, batch_index=batch_index, batch=batch, out=out)

        def lnb(dy, *a, **kw):
            self.ln_dy.append(dy.clone())
            return real_lnb(dy, *a, **kw)

        for name, fn in (("rope3d_", rope), ("flash_attn_bwd", bwd), ("qkv_dgrad", dgrad), ("layernorm_bwd", lnb)):
            monkeypatch.setattr(ops, name, fn)


BLOCK_CFG = {  # d, heads, pad32 (head_dim 32 on the head_dim-64 kernels), rotary ids
    "encoder hd64": (1024, 16, False, False),
    "predictor hd32": (384, 12, True, True),
    "predictor hd64": (384, 6, False, True),
}


def make_layer(d, H, pad32, g):
    from smb_vision_b200 import vjepa

    layer = vjepa._VJepaLayer(d, 4 * d, 1e-6, True).to(DEV)
    with torch.no_grad():
        for name, prm in layer.named_parameters():
            if name.endswith("weight") and prm.dim() == 2:
                prm.copy_(torch.randn(prm.shape, device=DEV, generator=g) / math.sqrt(prm.shape[1]))
            elif "norm" in name and name.endswith("weight"):
                prm.copy_(1.0 + 0.1 * torch.randn(prm.shape, device=DEV, generator=g))
            else:
                prm.copy_(0.2 * torch.randn(prm.shape, device=DEV, generator=g))
    p = vjepa._pack_layer(layer, H, 1e-6)
    p.pad32 = p.hd == 32 and pad32  # as VJepaPredictorRunner.packed sets it
    return layer, p


def real_heads(t, hd):
    """[..., H', n, 64] rows as the QKV GEMM wrote them -> [..., H, n, hd] real heads (hd 32: two per 64-wide row)."""
    if hd == 64:
        return t
    *o, H2, n, _ = t.shape
    return t.view(*o, H2, n, 2, 32).transpose(-3, -2).reshape(*o, 2 * H2, n, 32)


def gemm_layout(t, hd):
    """inverse of real_heads"""
    if hd == 64:
        return t
    *o, H, n, _ = t.shape
    return t.view(*o, H // 2, 2, n, 32).transpose(-3, -2).reshape(*o, H // 2, n, 64)


def pair_sum(a, D):
    """a + a[partner] over the rotated columns of head rows of width D (the transposed map mixes each adjacent pair)."""
    S3 = 3 * 2 * ((D // 3) // 2)
    out = a.clone()
    out[..., 0:S3:2] += a[..., 1:S3:2]
    out[..., 1:S3:2] += a[..., 0:S3:2]
    return out


@pytest.mark.parametrize("size", ["moderate", "full"])
@pytest.mark.parametrize("cfg", list(BLOCK_CFG))
def test_rotary_attention_sublayer_stages(lib, monkeypatch, cfg, size):
    """block_forward_train / block_backward on a vjepa._pack_layer with the rope tuple as vjepa.py builds it (encoder:
    (grid, None, max_pos); predictor: (grid, ids, max_pos, ids2) from smbv_position_sort of a context and a target mask with
    shared positions), at n = 1999 (B = 2) and 20 480 tokens.  Each stage against fp64 from the kernels' own output of the
    stage before: the saved rotated Q / K; the attention output and lse; dQ / dK / dV of the attention backward; the same
    after the transposed map, in the layout the QKV GEMM wrote; dh1; the fused [Q; K; V] bias gradient, and the K slot
    against the true fp64 gradient (module docstring).  Controls: wrong positions on Q / K, the forward map in place of the
    transpose, dh1 without the dK third, the K slot zeroed."""
    from smb_vision_b200 import ops, vjepa
    from smb_vision_b200.training import block_backward, block_forward_train, vjepa_block_names

    d, H, pad32, with_ids = BLOCK_CFG[cfg]
    hd = d // H
    B, n = (1 if cfg.startswith("encoder") else 2, N_VITL) if size == "full" else (2, 1999)
    g = torch.Generator(device=DEV).manual_seed(d + H + n)
    layer, p = make_layer(d, H, pad32, g)
    gs = VITL["gs"]
    if with_ids:
        N = VITL["frames"] // 16 * gs * gs
        a = n // 2
        ctx = torch.stack([torch.randperm(N, device=DEV, generator=g)[:a].sort().values for _ in range(B)])
        tgt = torch.stack([torch.randperm(N, device=DEV, generator=g)[:n - a].sort().values for _ in range(B)])
        _, _, ids, ids2 = ops.position_sort(torch.cat([ctx, tgt], 1).int().contiguous(), doubled=True)
        rope = (gs, ids, min(max(gs, VITL["frames"] // 16, int(N // (gs * gs)) + 1), 256), ids2)  # vjepa.py predictor rule
        ids_true = torch.cat([ctx, tgt], 1).sort(1).values  # independent of the kernel
        assert int((ids_true[:, 1:] == ids_true[:, :-1]).sum()) > 0  # ties
    else:
        rope = (gs, None, min(max(gs, VITL["frames"] // 16, VITL["frames"] // 16), 256))  # vjepa.py encoder rule
        ids_true = None
    X = torch.randn(B, n, d, device=DEV, generator=g)
    spy = Spy(monkeypatch)
    _, s = block_forward_train(X, p, rope)
    assert len(spy.rope) == 1 and not spy.rope[0]["transpose"]
    res = {}

    # ---- stage 1: rotated Q / K (saved); control: wrong positions ----
    pre = spy.rope[0]["before"].view(2, B, -1, n, 64)  # Q, K as the QKV GEMM wrote them
    pre_r = real_heads(pre, hd)  # [2, B, H, n, hd]
    ref, floor = rope_ref64(pre_r, ids_true, gs, False)
    got = s.qkv[:2, ..., :hd]  # saved, zero-padded for hd 32
    res["rotated q/k"] = rope_metric(got, ref, floor)
    if pad32:
        assert (bits(s.qkv[..., 32:]) == 0).all()
        bad, _ = rope_ref64(spy.rope[0]["before"], torch.cat([ids_true, ids_true], 1), gs, False)  # ids where ids2 belongs
        bad = real_heads(bad.view(2, B, H // 2, n, 64), hd)
    elif with_ids:
        bad, _ = rope_ref64(pre_r, None, gs, False)  # arange in place of the sorted ids
    else:
        bad, _ = rope_ref64(pre_r, None, gs - 1, False)  # the wrong grid
    ctrl_rope = rope_metric(got, bad, floor)
    del ref, floor, bad

    # ---- stage 2: attention forward from the saved (rotated, padded) q, k, v ----
    q, k, v = (s.qkv[i].reshape(B * H, n, 64) for i in range(3))
    scale = hd ** -0.5
    assert len(spy.bwd) == 0
    dX = torch.randn(B, n, d, device=DEV, generator=g)
    dXb = ops.cast_bf16(dX)
    sc = vjepa._ScratchGrads(dict(layer.named_parameters()), DEV)
    block_backward(dX, dXb, s, p, sc, "", vjepa_block_names(""), rope)
    bw = spy.bwd[0]
    o_k = heads_of(bw["o"], B, H)  # the forward kernel's O (a64 for hd 32), as the backward reads it
    lse_k = bw["lse"].reshape(B * H, n)
    r = attn_ref64(q, k, v, o_k, heads_of(bw["do"], B, H), lse_k, scale)
    o_ref = r["o"][..., :hd]
    got_a = heads_of(s.a, B, H)  # [BH, n, hd]: after heads32_tokens for hd 32
    res["attention O"] = max_ratio((got_a.double() - o_ref).abs(), ulps_floor(o_ref)) / O_ULPS
    res["lse"] = (lse_k.double() - r["lse"]).abs().max().item() / LSE_ABS

    # ---- stage 3: attention backward (dq, dk, dv as the kernel wrote them, padded for hd 32) ----
    dq_k, dk_k, dv_k = (t.reshape(B * H, n, 64) for t in bw["d"])
    dworst = 0.0
    for got_d, key, term in ((dq_k, "dq", "tq"), (dk_k, "dk", "tk"), (dv_k, "dv", "tv")):
        dworst = max(dworst, max_ratio((got_d.double() - r[key]).abs(), ulps_floor(r[key], r[term])))
    res["dq/dk/dv"] = dworst / D_ULPS
    if pad32:
        assert all(bool((bits(t[..., 32:]) == 0).all()) for t in (dq_k, dk_k, dv_k))

    # ---- stage 4: the transposed map on dQ / dK, in the QKV GEMM's layout; control: the forward map ----
    tr = [c for c in spy.rope if c["transpose"]]
    assert len(tr) == 1
    dpre = torch.stack([dq_k, dk_k]).view(2, B, H, n, 64)[..., :hd]  # the attention backward's own output, real heads
    assert same_bits(tr[0]["before"].view(2, B, -1, n, 64), gemm_layout(dpre, hd))  # heads32_squeeze (hd 32) is exact
    dpost = real_heads(tr[0]["after"].view(2, B, -1, n, 64), hd)
    ref, floor = rope_ref64(dpre, ids_true, gs, True)
    res["transposed map"] = rope_metric(dpost, ref, floor)
    bad, _ = rope_ref64(dpre, ids_true, gs, False)
    ctrl_tr = rope_metric(dpost, bad, floor)
    del ref, bad

    # ---- stage 5: dh1 = dQKV Wqkv (the dgrad GEMM); control: without the dK third ----
    dqkv = spy.dgrad[0]["dqkv"]  # [3, B, H', n, 64] as qkv_dgrad reads it
    assert same_bits(dqkv[:2], tr[0]["after"].view(2, B, -1, n, 64))
    dh1 = spy.ln_dy[-1]  # the LayerNorm-1 backward's input
    W = p.wqkv.double()
    tok = dqkv.permute(1, 3, 0, 2, 4).reshape(B, n, 3 * d).double()  # [B, n, 3d]: slot, head, column
    ref = tok @ W
    res["dh1"] = max_ratio((dh1.double() - ref).abs(), ulps_floor(ref, row_floor=False)) / BF16_ULPS
    tok[..., d:2 * d] = 0
    bad = tok @ W
    ctrl_dh1 = max_ratio((dh1.double() - bad).abs(), ulps_floor(ref, row_floor=False)) / BF16_ULPS
    del tok, ref, bad

    # ---- stage 6: fused bias gradient; K slot against the true gradient ----
    gb = sc.fused_qkv_bias("").double()  # [q; k; v] bias gradients, accumulated from zero
    dd = dqkv.double()
    ref_b = dd.sum((1, 3)).reshape(3 * d)  # slot, head, column
    col = dd.square().sum((1, 3)).sqrt().reshape(3 * d)
    res["bias colsum"] = max_ratio((gb - ref_b).abs(), col) / COL_REL
    ctrl_k = max_ratio(ref_b[d:2 * d].abs(), col[d:2 * d]) / COL_REL
    # true K-bias gradient: fp64 dK of the fp64 backward, fp64 transposed map, fp64 sum over the batch and the tokens
    dk_true = r["dk"].view(B, H, n, 64)[..., :hd]
    true_post, map_floor = rope_ref64(dk_true, ids_true, gs, True)
    true_bk = true_post.sum((0, 2)).reshape(d)
    a_bnd = D_ULPS * ulps_floor(r["dk"], r["tk"]).view(B, H, n, 64)[..., :hd]  # attention-backward element bound of dK
    dk_abs = dk_true.abs()
    rounding = (2 * 2.0 ** -8 * pair_sum(dk_abs, hd) + map_floor).sum((0, 2)).reshape(d) + COL_REL * col[d:2 * d]
    kb = rounding + pair_sum(a_bnd, hd).sum((0, 2)).reshape(d)
    res["K bias vs true"] = max_ratio((gb[d:2 * d] - true_bk).abs(), kb)
    ctrl_k_true = max_ratio(true_bk.abs(), kb)  # the true K-bias gradient over its bound = the "K slot zeroed" control
    ctrl_k_round = max_ratio(true_bk.abs(), rounding)
    k_frob = (torch.linalg.norm(gb[d:2 * d] - true_bk) / torch.linalg.norm(true_bk)).item()
    del r, dd

    name = f"sublayer {cfg} B={B} n={n}"
    for k_, v_ in res.items():
        report(f"{name}: {k_}", v_, 1.0)
    print(f"{name}: controls (x bound): rope positions {ctrl_rope:.3g}, forward map for the transpose {ctrl_tr:.3g}, dh1 without dK "
          f"{ctrl_dh1:.3g}, K slot zeroed {ctrl_k:.3g} (colsum bound)")
    print(f"{name}: K bias: true gradient / bound {ctrl_k_true:.3g} (= the K-slot-zeroed control against the true gradient; "
          f"against the two roundings and the colsum bound alone {ctrl_k_round:.3g}); Frobenius-rel to the true gradient {k_frob:.3g}")
    assert all(v_ <= 1.0 for v_ in res.values()), res
    assert ctrl_rope >= CONTROL and ctrl_tr >= CONTROL and ctrl_dh1 >= CONTROL and ctrl_k >= CONTROL
