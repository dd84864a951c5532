"""Kernel-level parity of flash attention (run with -m gpu on the B200 box): the tcgen05 forward (`smbv_flash_attn_fwd_ex`,
with and without the key-range split of its partial last wave), the fused one-pass backward and the deterministic two-kernel
backward, and the fp32 CUDA-core kernels for head_dim 8 / 16 / 32.  Each kernel is compared on its own with a float64
reference computed ON THE DEVICE from the same bf16 operands it reads (chunked by query rows): the backward reference takes
exactly the O (bf16) and lse (fp32) the backward reads, built from the fp64 forward and not from the forward kernel.

Error model (per element of an output; eps = 2^-9, the relative rounding error of bf16):
  * P is rounded to bf16 before the PV and dV products, dS before the dQ and dK products: relative error <= eps per term,
    independent across terms, so a sum of n comparable terms moves by ~ eps / sqrt(n) of its magnitude (more when the
    terms cancel, as in dS = P (dP - D) of a nearly one-hot row);
  * the emulated exponentials (`ex2_emu2`, 6 of every 16) have a relative error of about 1e-4 (code comment; not measured
    here), below the bf16 rounding of P;
  * accumulation is fp32 (tensor-core, cross-CTA reductions and the split combines), ~1e-7 relative;
  * each output is rounded to bf16 once: 0.5 ulp.
A correct kernel is thus within a few bf16 ulps of the fp64 value, relative to the size of the output row: the element-wise
metric is |got - ref| / (1 ulp(ref) + ROW_FLOOR * rms(ref row) + 1e-5 max|ref|).  The local metrics are the Frobenius-rel of
every 128-row tile and every row of every head (tiles and rows whose reference is tiny are judged against LOCAL_FLOOR of an
average tile / row, so that underflowed rows do not divide by zero).  A gradient element's error is measured relative to
the larger of the result and the norm of the terms summed into it (`reference`): where dQ_i = sum_j dS_ij k_j cancels
(aligned keys, a one-hot row), what remains is the rounding of each term.  The bounds below are about 2x the worst value
measured over every shape and family on a B200 at a 1000 W power limit (the measured value is beside each bound).

Input families (each through the forward and both backward kernels): N(0,1) (`random`, which also carries the negative
controls), a running maximum that rises slowly (never rescales O: P up to 2^7.9), fast (rescales at every key block) and in
irregular jumps, a maximum in the first block that falls until P underflows the 2^-126 clamp of `ex2_emu2`, a nearly
one-hot softmax with |lse| / scale in the hundreds (the fifth K-step of the fused backward carries -lse/scale and -D as a
three-term bf16 split), exact ties (Q = 0 rows, duplicated keys) and the zero-padded head_dim-32 layout of `heads32_expand`.

Shapes come from a Python replica of the two work plans (`attn_fwd_parts`, `fused_plan`), pinned to the library by the
exported workspace sizes, so that every split count of both plans is reached on the device under test.

Negative controls (random family): the comparison against a reference with one key block removed from one query tile (O,
lse, dQ) or one query block removed from one key tile (dK, dV) must fail the local bound by >= CONTROL_BF16.
"""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
LOG2E = 1.4426950408889634

# bounds: see the module docstring (measured values on B200, 1000 W, in the comments)
BND = dict(
    o_tile=6e-3,     # O: worst 128-row tile Frobenius-rel (measured 3.6e-3, heads32; 2.8e-3 random)
    o_row=1e-2,      # O: worst row (measured 4.8e-3, peaked)
    o_ulps=5.0,      # O: element-wise, in bf16 ulps with the row floor (measured 2.5, heads32)
    lse=2.5e-4,      # lse: max |got - ref| (measured 1.1e-4, peaked: |lse| ~ 60)
    d_tile=6e-3,     # dQ per query tile, dK / dV per key tile (measured 4.9e-3 rising-slow, 3.1e-3 random; < 2x: one query
                     # block missing from one key tile at N = 20480 moves a tile by only ~8 %, and its control needs 10x)
    d_ulps=5.0,      # dQ / dK / dV element-wise (measured 2.3, rising-jumps)
    comp=7e-3,       # (measured 3.5e-3, rising-slow) kernel forward -> kernel backward against the exact fp64 gradient: worst tile, less COMP_OWN x the
)                    # worst tile of the fp64 backward of the bf16-rounded O (D = rowsum(dO O) is ill-conditioned when P is
COMP_OWN = 4.0       # nearly one-hot: rounding O alone moves such dQ tiles by O(1))
ROW_FLOOR = 2.0 ** -8   # element floor: one bf16 ulp of the row's rms
LOCAL_FLOOR = 1e-3      # tile / row norms are floored at this fraction of an average tile / row of the tensor
REPRO_ULPS = 1.0        # fused backward dQ, second call: fp32 reduction order, then one bf16 rounding
# fp32 CUDA-core kernels (P not rounded): output rounding only (measured 3.5e-3, 0.43 ulps, 7.3e-7)
SMALL = dict(row=7e-3, ulps=1.0, lse=1.5e-6)
CONTROL_BF16 = 10.0
G = 4096                # guard elements on each side of every output
SENT = 1232.0           # guard sentinel (exact in bf16 and fp32)


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


def tile_frob(a, b, tr=128, term=None):
    """worst Frobenius-rel over the [tr x W] row tiles of every head of [BH, N, W] outputs (tr=1: worst row); a tile's
    reference norm is floored at LOCAL_FLOOR of the norm of an average tile and, for a gradient, at the norm of the terms
    summed into the tile's elements (`term` [BH, N, W], see `reference`): where those terms cancel, the rounding of each of
    them is what is left, so the error is measured relative to the terms."""
    a, b = a.double(), b.double()
    BH, N, W = b.shape
    pad = (0, 0, 0, (-N) % tr)
    e = F.pad((a - b) ** 2, pad).view(BH, -1, tr, W).sum((2, 3))
    r = F.pad(b ** 2, pad).view(BH, -1, tr, W).sum((2, 3))
    avg = (b ** 2).sum() / (BH * N) * tr
    den = torch.maximum(r.sqrt(), LOCAL_FLOOR * avg.sqrt())
    if term is not None:
        den = torch.maximum(den, F.pad(term.double() ** 2, pad).view(BH, -1, tr, W).sum((2, 3)).sqrt())
    return (e.sqrt() / den.clamp_min(1e-300)).max().item()


def bf16_ulps(got, ref, term=None):
    """max over elements of |got - ref| / (1 bf16 ulp of ref + ROW_FLOOR rms(ref row) + 1e-5 max|ref|), rows = last dim;
    for a gradient, the larger of the row's rms and the norm of the terms summed into the element (`term`, see tile_frob)."""
    ref = ref.double()
    ulp = torch.exp2(torch.floor(torch.log2(ref.abs())) - 7)  # 8 significant bits; 0 at ref == 0
    rms = ref.pow(2).mean(-1, keepdim=True).sqrt()
    if term is not None:
        rms = torch.maximum(rms, term.double())
    floor = ulp + ROW_FLOOR * rms + 1e-5 * ref.abs().max()
    return ((got.double() - ref).abs() / floor.clamp_min(1e-300)).max().item()


def report(name, worst, bounds):
    print(f"{name}: " + ", ".join(f"{k} {worst[k]:.2e} (bound {bounds[k]:.0e})" for k in bounds if k in worst))


def rnd(shape, g, scale=1.0):
    return (torch.randn(shape, device=DEV, generator=g) * scale).bfloat16()


def _vp(t, off_bytes=0):
    return C.c_void_p(0 if t is None else t.data_ptr() + off_bytes)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def guarded(n, dtype, regions=1):
    """flat buffer [G | n | G | n | ... | G] with NaN in the regions and SENT in the guards; returns (buffer, region views)."""
    buf = torch.full((G + regions * (n + G),), SENT, dtype=dtype, device=DEV)
    views = [buf[G + i * (n + G):G + i * (n + G) + n] for i in range(regions)]
    for v in views:
        v.fill_(float("nan"))
    return buf, views


def guards_intact(buf, n, regions=1):
    keep = torch.ones_like(buf, dtype=torch.bool)
    for i in range(regions):
        keep[G + i * (n + G):G + i * (n + G) + n] = False
    return bool((buf[keep] == SENT).all())


# =====================================================================================================================
# 0. replica of the work plans, shape lists
# =====================================================================================================================
def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def fwd_plan(B, H, N, sms):
    """attn.cu attn_fwd_parts: (key-range pieces per split unit (0 = whole units only), split units, query tiles, key blocks)."""
    t128 = (N + 127) // 128
    pairs = B * H * (t128 // 2)
    rest = pairs % sms
    if rest == 0:
        return 0, 0, t128, t128
    fixed, best, best_cost = 3.0 / t128, 0, 1.0 + 3.0 / t128
    for k in range(2, min(8, t128) + 1):
        cost = float((rest * k + sms - 1) // sms) * (1.0 / k + fixed)
        if cost < best_cost * 0.97:
            best_cost, best = cost, k
    return best, (rest if best else 0), t128, t128


def bwd_plan(B, H, N, sms):
    """attn_bwd.cu fused_plan: (query-range pieces per split unit, whole units, all units)."""
    nkv = (N + 127) // 128
    U = nkv * B * H
    nf = (U // sms) * sms
    R, best = U - nf, 1
    if R > 0:
        fixed, best_cost = 4.0 / nkv, 1.0 + 4.0 / nkv
        for k in range(2, min(8, nkv) + 1):
            cost = float((R * k + sms - 1) // sms) * (1.0 / k + fixed)
            if cost < best_cost * 0.97:
                best_cost, best = cost, k
    if best == 1:
        nf = U
    return best, nf, U


def bwd_workspace_bytes(B, H, N, sms):
    parts, nf, U = bwd_plan(B, H, N, sms)
    return B * H * N * 256 + (U - nf) * parts * 65536


def fwd_workspace_bytes(B, H, N, sms):
    return (B * H * (((N + 127) // 128) // 2)) % sms * 8 * 2 * 128 * 68 * 4


def _fwd_kinds(s, sms):
    parts, _, t128, nkv = fwd_plan(*s, sms)
    kinds = {f"fwd parts {parts}"} if parts else ({"fwd no split"} if t128 >= 2 else set())
    if parts and nkv % parts:
        kinds.add("fwd parts not dividing the key blocks")
    if parts and t128 % 2:
        kinds.add("fwd split with an odd last query tile")
    if s[2] <= 128:
        kinds.add("fwd N <= 128")
    return kinds


def _bwd_kinds(s, sms):
    parts, _, _ = bwd_plan(*s, sms)
    kinds = {f"bwd parts {parts}"}
    if parts > 1 and ((s[2] + 127) // 128) % parts:
        kinds.add("bwd parts not dividing the query blocks")
    return kinds


REQUIRED = ({"fwd no split", "fwd N <= 128", "fwd parts not dividing the key blocks", "fwd split with an odd last query tile"}
            | {f"fwd parts {k}" for k in range(2, 9)} | {f"bwd parts {k}" for k in range(1, 9)}
            | {"bwd parts not dividing the query blocks"})


def plan_shapes(sms):
    """the first single-sample shape (one head, N rising; then H heads at N = 256) that reaches each plan kind not reached yet"""
    cands = [(1, 1, n) for n in range(1, 2049)] + [(1, h, 256) for h in range(2, 2 * sms + 1)]
    got, out = set(), []
    for s in cands:
        k = (_fwd_kinds(s, sms) | _bwd_kinds(s, sms)) & REQUIRED
        if k - got:
            got |= k
            out.append(s)
    return out


MODEL_SHAPES = [(1, 12, 7168), (1, 6, 20480), (1, 12, 20480), (1, 16, 20480), (4, 12, 1960), (1, 16, 9216), (2, 12, 7168),
                (1, 2, 20480)]  # MIM encoder, decoder, full / V-JEPA encoder, classification, V-JEPA, batched, two heads
RAGGED_SHAPES = [(1, 1, 1), (1, 1, 64), (1, 1, 127), (1, 1, 128), (1, 1, 129), (1, 1, 255), (1, 1, 257), (3, 2, 129), (2, 3, 257)]
EXTRA_SHAPES = [(2, 3, 1000), (1, 4, 4096)]  # batched ragged, and a longer row for the non-random families


def shapes_for(family, sms):
    base = plan_shapes(sms) + RAGGED_SHAPES
    return base + (MODEL_SHAPES if family == "random" else EXTRA_SHAPES)


def test_plan_replica_and_shape_coverage(ops):
    """the replica predicts the library's workspace sizes exactly for every shape used, and the shape lists reach every
    split count of both plans on this device, a split count that does not divide the blocks, an odd last query tile
    under a split, whole units only, and N <= 128."""
    from smb_vision_b200 import load

    lib, sms = load(), sm_count()
    shapes = sorted({s for f in FAMILIES for s in shapes_for(f, sms)})
    for s in shapes:
        assert lib.smbv_flash_attn_bwd_fused_workspace_bytes(*s) == bwd_workspace_bytes(*s, sms), s
        assert lib.smbv_flash_attn_fwd_workspace_bytes(*s) == fwd_workspace_bytes(*s, sms), s
    reached = set().union(*(_fwd_kinds(s, sms) | _bwd_kinds(s, sms) for s in shapes))
    assert REQUIRED <= reached, sorted(REQUIRED - reached)
    print(f"plan replica ({sms} SMs): {len(shapes)} shapes; plan shapes {plan_shapes(sms)}")
    for s in MODEL_SHAPES:
        print(f"  {s}: fwd parts {fwd_plan(*s, sms)[0]}, bwd parts {bwd_plan(*s, sms)[0]}")


# =====================================================================================================================
# fp64 reference
# =====================================================================================================================
def reference(q, k, v, do, scale, backward=True, true_grad=False):
    """q, k, v, do [BH, N, D] (bf16, do per head) -> fp64 O, lse and the backward of (O rounded to bf16, lse rounded to
    fp32): dq, dk, dv; with true_grad also the exact gradient (dq_t, dk_t, dv_t) of softmax(scale q k^T) v.  tq, tk, tv
    [BH, N, D]: per output element, the L2 norm of the terms summed into it, tq_id = scale (sum_j a_ij^2 k_jd^2)^1/2,
    tk_jd = scale (sum_i a_ij^2 q_id^2)^1/2, tv_jd = (sum_i P_ij^2 dO_id^2)^1/2, with a_ij = |dS_ij| + 2^-16 P_ij
    (sum_d |dO_id V_jd| + sum_d |dO_id O_id|): dS plus the fp32 rounding of the two 64-term dot products dP_ij and D_i, whose
    difference cancels (to exactly 0 at N = 1, to ~1e-4 of the terms in a one-hot row) where dS is small."""
    BH, N, D = q.shape
    qd, kd, vd, dod = (t.double() for t in (q, k, v, do))
    z = lambda: torch.zeros(BH, N, D, dtype=torch.float64, device=DEV)  # noqa: E731
    r = dict(o=z(), lse=torch.zeros(BH, N, dtype=torch.float64, device=DEV), dq=z(), dk=z(), dv=z())
    if true_grad:
        r.update(dq_t=z(), dk_t=z(), dv_t=z())
    if backward:
        r.update(tq=z(), tk=z(), tv=z())
    R = max(128, (2 ** 26 // (BH * N)) // 128 * 128)
    for r0 in range(0, N, R):
        sl = slice(r0, min(N, r0 + R))
        s = torch.bmm(qd[:, sl], kd.transpose(1, 2)) * scale
        lse = torch.logsumexp(s, -1, keepdim=True)
        dp = torch.bmm(dod[:, sl], vd.transpose(1, 2)) if backward else None
        if true_grad:
            p = torch.exp(s - lse)
            o = torch.bmm(p, vd)
            ds = p * (dp - (dod[:, sl] * o).sum(-1, keepdim=True))
            r["dq_t"][:, sl] = scale * torch.bmm(ds, kd)
            r["dk_t"] += scale * torch.bmm(ds.transpose(1, 2), qd[:, sl])
            r["dv_t"] += torch.bmm(p.transpose(1, 2), dod[:, sl])
            del p, ds
        else:
            o = torch.bmm(torch.exp(s - lse), vd)
        r["o"][:, sl], r["lse"][:, sl] = o, lse[..., 0]
        if not backward:
            continue
        p = torch.exp(s - lse.float().double())  # what the backward reads: lse in fp32, O in bf16
        del s
        dsum = (dod[:, sl] * o.bfloat16().double()).sum(-1, keepdim=True)
        ds = p * (dp - dsum)
        r["dq"][:, sl] = scale * torch.bmm(ds, kd)
        r["dk"] += scale * torch.bmm(ds.transpose(1, 2), qd[:, sl])
        r["dv"] += torch.bmm(p.transpose(1, 2), dod[:, sl])
        dabs = (dod[:, sl] * o.bfloat16().double()).abs().sum(-1, keepdim=True)
        a2 = (ds.abs() + 2.0 ** -16 * p * (torch.bmm(dod[:, sl].abs(), vd.abs().transpose(1, 2)) + dabs)) ** 2
        r["tq"][:, sl] = scale * torch.bmm(a2, kd ** 2).sqrt()
        r["tk"] += torch.bmm(a2.transpose(1, 2), qd[:, sl] ** 2)
        r["tv"] += torch.bmm((p * p).transpose(1, 2), dod[:, sl] ** 2)
        del p, ds, dp, a2
    if backward:
        r["tk"], r["tv"] = scale * r["tk"].sqrt(), r["tv"].sqrt()
    return r


def _rows(q, k, v, do, o_in, lse_in, bh, rows, scale, drop_keys=None):
    """for query rows `rows` of head bh: (O, lse) of the softmax with keys `drop_keys` removed, and P, dS of the backward."""
    qd, kd, vd, dod = q[bh, rows].double(), k[bh].double(), v[bh].double(), do[bh, rows].double()
    s = qd @ kd.t() * scale
    sb = s.clone()
    if drop_keys is not None:
        sb[:, drop_keys] = float("-inf")
    lse = torch.logsumexp(sb, -1)
    o_bad = torch.softmax(sb, -1) @ vd
    p = torch.exp(s - lse_in[bh, rows].double()[:, None])
    ds = p * (dod @ vd.t() - (dod * o_in[bh, rows].double()).sum(-1, keepdim=True))
    return o_bad, lse, p, ds


# =====================================================================================================================
# input families
# =====================================================================================================================
FAMILIES = ["random", "rising-slow", "rising-fast", "rising-jumps", "falling", "peaked", "ties", "heads32"]


def _aligned(B, H, N, profile, g, scale):
    """q_i = a_i u, k_j = c_j u + noise: scores in log2 units ~ (a_i / 4) * profile[j] (profile in log2 units at a_i = 4)."""
    u = torch.randn(64, device=DEV, generator=g)
    u /= u.norm()
    a = 3.5 + torch.rand(B, H, N, 1, device=DEV, generator=g)
    q = a * u + 0.02 * torch.randn(B, H, N, 64, device=DEV, generator=g)
    c = profile / (scale * LOG2E * 4.0)
    k = c[None, None, :, None] * u + 0.05 * torch.randn(B, H, N, 64, device=DEV, generator=g)
    return q.bfloat16(), k.bfloat16()


def make_inputs(family, B, H, N, seed):
    """-> q, k, v [B,H,N,64] bf16, dO [B,N,H*64] bf16, scale"""
    g = torch.Generator(device=DEV).manual_seed(seed)
    scale = 0.125
    v, do = rnd((B, H, N, 64), g), rnd((B, N, H * 64), g)
    j = torch.arange(N, device=DEV, dtype=torch.float64)
    if family == "random":
        q, k = rnd((B, H, N, 64), g), rnd((B, H, N, 64), g)
    elif family == "rising-slow":    # the maximum rises by 6.8 log2 units over the whole row: never 2^8 above the first block's
        q, k = _aligned(B, H, N, (6.8 * j / N).float(), g, scale)
    elif family == "rising-fast":    # +12 log2 units per key block: O is rescaled at every block
        q, k = _aligned(B, H, N, (12.0 * j / 128).float(), g, scale)
    elif family == "rising-jumps":   # irregular jumps between blocks, some of which add up past 2^8 only together
        steps = torch.tensor([0.0, 2.0, 5.0, 9.0, 30.0], device=DEV)[torch.randint(0, 5, ((N + 127) // 128,), device=DEV, generator=g)]
        jb = (j // 128).long()
        q, k = _aligned(B, H, N, (torch.cumsum(steps, 0)[jb] + 0.5 * (j % 128) / 128).float(), g, scale)
    elif family == "falling":        # the maximum in the first block, then 300 log2 units down: P underflows past 2^-126
        q, k = _aligned(B, H, N, (-300.0 * j / N).float(), g, scale)
    elif family == "peaked":         # nearly one-hot rows on top of a shared component: |lse| / scale in the hundreds
        w = torch.randn(64, device=DEV, generator=g)
        w *= 20.0 / w.norm()
        q = (2.5 * torch.randn(B, H, N, 64, device=DEV, generator=g) + w).bfloat16()
        k = (2.5 * torch.randn(B, H, N, 64, device=DEV, generator=g) + w).bfloat16()
    elif family == "ties":           # Q = 0 rows (uniform attention), every key twice, key block 1 a copy of block 0
        q, k = rnd((B, H, N, 64), g), rnd((B, H, N, 64), g)
        q[:, :, ::4] = 0
        k[:, :, 1::2] = k[:, :, 0:N - 1:2]
        if N >= 256:
            k[:, :, 128:256] = k[:, :, :128]
    elif family == "heads32":        # heads32_expand layout: 32 real columns + 32 zero columns, scale 32^-0.5
        q, k = rnd((B, H, N, 64), g), rnd((B, H, N, 64), g)
        for t in (q, k, v):
            t[..., 32:] = 0
        do.view(B, N, H, 64)[..., 32:] = 0
        scale = 32 ** -0.5
    else:
        raise ValueError(family)
    return q.contiguous(), k.contiguous(), v, do, scale


def check_family_inputs(family, q, k, scale, N):
    """the fp64 scores of head 0 really do what the family is for (returns a description for the report)."""
    x = (q[0, 0].double() @ k[0, 0].double().t()) * scale * LOG2E  # log2 units
    nkv = N // 128  # full key blocks (a ragged last block rises less)
    if family.startswith("rising") and nkv >= 3:
        mb = x[:, :nkv * 128].reshape(N, nkv, 128).amax(-1)  # block maxima [rows, blocks]
        m_used, resc = mb[:, 0].clone(), torch.zeros(N, device=DEV)
        for b in range(1, nkv):  # the forward kernel's lazy-rescale decision over the whole key range
            jump = mb[:, b] - m_used > 8.0
            resc += jump
            m_used = torch.where(jump, mb[:, b], m_used)
        frac = (resc / (nkv - 1)).mean().item()
        if family == "rising-slow":
            rise = (mb.amax(1) - mb[:, 0]).max().item()
            assert frac == 0 and rise > 3.0, (frac, rise)
            return f"rescaled blocks 0, P up to 2^{rise:.1f}"
        elif family == "rising-fast":
            assert frac == 1.0, frac
        else:
            assert 0.15 < frac < 0.85, frac
        return f"rescaled blocks {frac:.2f}"
    if family == "falling":
        fall = (x.amax(1, keepdim=True) - x).amax(1).min().item()
        assert N < 128 or fall > 140, fall
        return f"min over rows of the fall {fall:.0f} log2 units"
    if family == "peaked":
        lse = torch.logsumexp(x / LOG2E, 1)
        pmax = torch.softmax(x / LOG2E, 1).amax(1)
        assert (lse / scale).abs().min() > 100 and pmax.median() > 0.5, (lse.min().item(), pmax.median().item())
        return f"|lse|/scale >= {(lse / scale).abs().min().item():.0f}, median max P {pmax.median().item():.2f}"
    return ""


def heads(t, B, H):
    """token-major [B, N, H*W] -> [B*H, N, W]"""
    N = t.shape[1]
    return t.view(B, N, H, -1).permute(0, 2, 1, 3).reshape(B * H, N, -1)


def tokens(t, B, H):
    """[B*H, N, W] -> token-major [B, N, H*W]"""
    _, N, W = t.shape
    return t.view(B, H, N, W).permute(0, 2, 1, 3).reshape(B, N, H * W)


# =====================================================================================================================
# kernel calls: outputs as NaN-prefilled views inside guarded buffers
# =====================================================================================================================
def run_fwd(lib, q, k, v, scale, split):
    """smbv_flash_attn_fwd_ex with the split workspace (split=True) or a null workspace (whole units only)."""
    from smb_vision_b200 import _lib

    Bn, H, N, _ = q.shape
    n_o, n_l = Bn * N * H * 64, Bn * H * N
    ob, (o,) = guarded(n_o, torch.bfloat16)
    lb, (lse,) = guarded(n_l, torch.float32)
    wsb = int(lib.smbv_flash_attn_fwd_workspace_bytes(Bn, H, N)) if split else 0
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV) if wsb else None
    _lib.call("smbv_flash_attn_fwd_ex", _vp(q), _vp(k), _vp(v), Bn, H, N, float(scale), _vp(o), _vp(lse), 0, _vp(ws), wsb, _stream())
    torch.cuda.synchronize()
    ok = guards_intact(ob, n_o) and guards_intact(lb, n_l)
    return o.view(Bn, N, H * 64), lse.view(Bn, H, N), ok


def run_bwd(ops, q, k, v, o, do, lse, scale, deterministic):
    """ops.flash_attn_bwd with dq / dk / dv as views into one guarded buffer (the [3,B,H,N,64] pattern of training.py, with
    guards between the three); B == 1 takes the one-sample 3-D call form."""
    Bn, H, N, _ = q.shape
    n = Bn * H * N * 64
    buf, views = guarded(n, torch.bfloat16, 3)
    if Bn == 1:
        dq, dk, dv = (t.view(H, N, 64) for t in views)
        ops.flash_attn_bwd(q[0], k[0], v[0], o[0], do[0], lse[0], scale, dq=dq, dk=dk, dv=dv, deterministic=deterministic)
    else:
        dq, dk, dv = (t.view(Bn, H, N, 64) for t in views)
        ops.flash_attn_bwd(q, k, v, o, do, lse, scale, dq=dq, dk=dk, dv=dv, deterministic=deterministic)
    torch.cuda.synchronize()
    return [t.view(Bn * H, N, 64) for t in views], guards_intact(buf, n, 3)


class Tally:
    """worst value per metric, and the checks that failed (reported together at the end of a test)"""

    def __init__(self):
        self.worst, self.fails = {}, []

    def add(self, key, val, bound, what):
        self.worst[key] = max(self.worst.get(key, 0.0), val)
        if not val <= bound:  # NaN fails
            self.fails.append(f"{what}: {key} {val:.3e} > {bound:.0e}")

    def expect(self, cond, what):
        if not cond:
            self.fails.append(what)


def _real(t, family):
    return t[..., :32] if family == "heads32" else t


def _check_pad(tl, t, family, what):
    if family == "heads32":
        tl.expect(bool((t[..., 32:] == 0).all()), f"{what}: pad columns not exactly zero")


def _largest_full_block(n):
    """index of the last 128-block of n rows that is full (the last block when n % 128 == 0)"""
    return n // 128 - 1


# =====================================================================================================================
# 1. forward
# =====================================================================================================================
@pytest.mark.parametrize("family", FAMILIES)
def test_flash_attention_forward_matches_fp64(ops, family):
    """O and lse of the default forward kernel, with the split workspace and without one, against fp64 softmax(scale QK^T)V;
    a second call is bit-identical; nothing outside out / lse is written and every element of them is."""
    from smb_vision_b200 import load

    lib, sms = load(), sm_count()
    tl, ctrl, notes = Tally(), float("inf"), set()
    for s in shapes_for(family, sms):
        Bn, H, N = s
        q, k, v, do, scale = make_inputs(family, *s, seed=N * 131 + H * 7 + Bn)
        notes.add(check_family_inputs(family, q, k, scale, N))
        ref = reference(q.view(-1, N, 64), k.view(-1, N, 64), v.view(-1, N, 64), heads(do, Bn, H), scale, backward=False)
        ro = _real(ref["o"], family)
        for split in (True, False):
            what = f"{s} {'split' if split else 'whole'} (fwd parts {fwd_plan(*s, sms)[0] if split else 0})"
            o, lse, ok = run_fwd(lib, q, k, v, scale, split)
            tl.expect(ok, f"{what}: guard bytes changed")
            tl.expect(bool(torch.isfinite(o.float()).all() and torch.isfinite(lse).all()), f"{what}: NaN left in the output")
            oh = heads(o, Bn, H)
            _check_pad(tl, oh, family, what)
            oh = _real(oh, family)
            tl.add("o_tile", tile_frob(oh, ro), BND["o_tile"], what)
            tl.add("o_row", tile_frob(oh, ro, 1), BND["o_row"], what)
            tl.add("o_ulps", bf16_ulps(oh, ro), BND["o_ulps"], what)
            tl.add("lse", (lse.view(-1, N).double() - ref["lse"]).abs().max().item(), BND["lse"], what)
            o2, lse2, _ = run_fwd(lib, q, k, v, scale, split)
            tl.expect(torch.equal(o2, o) and torch.equal(lse2, lse), f"{what}: second call not bit-identical")
            if family == "random" and N >= 1024 and split:
                # negative control: one key block missing from one query tile of the last head (a split unit when there are any)
                bh, t128 = Bn * H - 1, (N + 127) // 128
                qt = 2 * (t128 // 2 - 1)
                kb = _largest_full_block(N)
                rows, keys = slice(128 * qt, 128 * qt + 128), slice(128 * kb, 128 * kb + 128)
                o_bad, l_bad, _, _ = _rows(q.view(-1, N, 64), k.view(-1, N, 64), v.view(-1, N, 64), heads(do, Bn, H),
                                           ref["o"], ref["lse"].float(), bh, rows, scale, keys)
                c_o = tile_frob(oh[bh:bh + 1, rows], o_bad[None]) / BND["o_tile"]
                c_l = (lse.view(-1, N)[bh, rows].double() - l_bad).abs().max().item() / BND["lse"]
                ctrl = min(ctrl, c_o, c_l)
        del ref
    report(f"flash_attn_fwd {family}", tl.worst, BND)
    if notes - {""}:
        print(f"  inputs: {'; '.join(sorted(notes - {''}))}")
    if family == "random":
        print(f"  negative control (one key block missing from one query tile): worst tile / bound >= {ctrl:.1f}")
        tl.expect(ctrl >= CONTROL_BF16, f"negative control margin {ctrl:.1f} < {CONTROL_BF16}")
    assert not tl.fails, "\n".join(tl.fails[:20])


# =====================================================================================================================
# 2. backward: fused (default) and deterministic
# =====================================================================================================================
@pytest.mark.parametrize("family", FAMILIES)
def test_flash_attention_backward_matches_fp64(ops, family):
    """dQ, dK, dV of both backward paths for O = fp64 reference rounded to bf16 and lse = fp64 lse rounded to fp32, against
    the fp64 backward of exactly those inputs; determinism (fused: dK / dV bit-identical, dQ within one bf16 ulp of fp32
    reduction order; deterministic path: all bit-identical); guards and NaN prefills; and the composition kernel forward ->
    kernel backward against the true fp64 gradient."""
    from smb_vision_b200 import load

    lib, sms = load(), sm_count()
    tl, ctrl = Tally(), {"dq": float("inf"), "dk": float("inf"), "dv": float("inf")}
    for s in shapes_for(family, sms):
        Bn, H, N = s
        q, k, v, do, scale = make_inputs(family, *s, seed=N * 137 + H * 11 + Bn)
        qh, kh, vh, doh = q.view(-1, N, 64), k.view(-1, N, 64), v.view(-1, N, 64), heads(do, Bn, H)
        ref = reference(qh, kh, vh, doh, scale, true_grad=True)
        o_in = tokens(ref["o"].bfloat16(), Bn, H).contiguous()
        lse_in = ref["lse"].float().view(Bn, H, N).contiguous()
        for det in (False, True):
            what = f"{s} {'deterministic' if det else f'fused (bwd parts {bwd_plan(*s, sms)[0]})'}"
            got, ok = run_bwd(ops, q, k, v, o_in, do, lse_in, scale, det)
            tl.expect(ok, f"{what}: guard bytes changed")
            for name, t in zip(("dq", "dk", "dv"), got):
                tl.expect(bool(torch.isfinite(t.float()).all()), f"{what}: NaN left in {name}")
                _check_pad(tl, t, family, f"{what} {name}")
                term = _real(ref["t" + name[1]], family)
                tl.add("d_tile", tile_frob(_real(t, family), _real(ref[name], family), term=term), BND["d_tile"], f"{what} {name}")
                tl.add("d_ulps", bf16_ulps(_real(t, family), _real(ref[name], family), term), BND["d_ulps"], f"{what} {name}")
            got2, _ = run_bwd(ops, q, k, v, o_in, do, lse_in, scale, det)
            tl.expect(torch.equal(got2[1], got[1]) and torch.equal(got2[2], got[2]), f"{what}: dK / dV not bit-identical")
            if det:
                tl.expect(torch.equal(got2[0], got[0]), f"{what}: dQ not bit-identical")
            else:
                tl.add("dq_repro_ulps", bf16_ulps(got2[0], got[0]), REPRO_ULPS, what)
            if family == "random" and N >= 1024 and not det:
                # negative controls on the last head (a split unit when there are any): one query block missing from one
                # key tile of dK / dV; one key block missing from one query tile of dQ
                bh, nb = Bn * H - 1, _largest_full_block(N)
                rows = slice(128 * nb, 128 * nb + 128)
                _, _, p, ds = _rows(qh, kh, vh, doh, ref["o"].bfloat16(), ref["lse"].float(), bh, rows, scale)
                keys = rows  # key tile nb, query block nb
                bad_dv = ref["dv"][bh, keys] - p[:, keys].t() @ doh[bh, rows].double()
                bad_dk = ref["dk"][bh, keys] - scale * ds[:, keys].t() @ qh[bh, rows].double()
                bad_dq = ref["dq"][bh, rows] - scale * ds[:, keys] @ kh[bh, keys].double()
                for name, t, bad in (("dv", got[2], bad_dv), ("dk", got[1], bad_dk), ("dq", got[0], bad_dq)):
                    term = ref["t" + name[1]][bh:bh + 1, rows]
                    ctrl[name] = min(ctrl[name], tile_frob(t[bh:bh + 1, rows], bad[None], term=term) / BND["d_tile"])
        # composition: kernel forward, then the fused kernel backward, against the exact gradient
        o, lse, _ = run_fwd(lib, q, k, v, scale, True)
        got, _ = run_bwd(ops, q, k, v, o.contiguous(), do, lse.contiguous(), scale, False)
        for name, t in zip(("dq", "dk", "dv"), got):
            exact = _real(ref[name + "_t"], family)
            term = _real(ref["t" + name[1]], family)
            own = tile_frob(_real(ref[name], family), exact, term=term)  # what rounding O to bf16 alone does to the exact gradient
            tl.worst["comp_bf16_o"] = max(tl.worst.get("comp_bf16_o", 0.0), own)
            tl.add("comp", tile_frob(_real(t, family), exact, term=term) - COMP_OWN * own, BND["comp"], f"{s} composition {name}")
        del ref
    report(f"flash_attn_bwd {family}", tl.worst, dict(BND, dq_repro_ulps=REPRO_ULPS, comp_bf16_o=float("inf")))
    if family == "random":
        print("  negative controls, worst tile / bound: " + ", ".join(f"{k} {v:.1f}" for k, v in ctrl.items())
              + " (dK / dV: one query block missing from one key tile; dQ: one key block missing from one query tile)")
        tl.expect(min(ctrl.values()) >= CONTROL_BF16, f"negative control margin {ctrl} < {CONTROL_BF16}")
    assert not tl.fails, "\n".join(tl.fails[:20])


# =====================================================================================================================
# 4. small head dimensions (fp32 CUDA-core kernels)
# =====================================================================================================================
@pytest.mark.parametrize("hd", [8, 16, 32])
@pytest.mark.parametrize("layout", ["token-major", "head-major"])
def test_small_head_attention_matches_fp64(ops, hd, layout):
    """smbv_attn_small_fwd / _bwd on the fused token-major QKV buffer [B,N,3,H,hd] and on head-major [B,H,N,hd] inputs:
    per-row bounds against fp64, NaN-prefilled guarded outputs, bit-identical second calls, and a dropped-key-row control."""
    from smb_vision_b200 import _lib

    tl, ctrl = Tally(), float("inf")
    for Bn, H, N in [(1, 1, 1), (1, 2, 7), (1, 1, 31), (2, 3, 32), (1, 2, 33), (1, 4, 300), (3, 2, 300)]:
        g = torch.Generator(device=DEV).manual_seed(hd * 1000 + N * 10 + Bn)
        d, scale = H * hd, hd ** -0.5
        if layout == "token-major":
            qkv = rnd((Bn, N, 3 * d), g)
            src = (qkv, qkv, qkv)
            offs = (0, 2 * d, 4 * d)  # bytes
            strides = (N * 3 * d, hd, 3 * d)
            q, k, v = (qkv.view(Bn, N, 3, H, hd)[:, :, i].permute(0, 2, 1, 3).reshape(Bn * H, N, hd) for i in range(3))
        else:
            src = tuple(rnd((Bn, H, N, hd), g) for _ in range(3))
            offs = (0, 0, 0)
            strides = (H * N * hd, N * hd, hd)
            q, k, v = (t.view(Bn * H, N, hd) for t in src)
        do = rnd((Bn, N, d), g)
        ref = reference(q, k, v, heads(do, Bn, H), scale)
        what = f"B={Bn} H={H} N={N}"
        outs = []
        for _ in range(2):
            ob, (o,) = guarded(Bn * N * d, torch.bfloat16)
            lb, (lse,) = guarded(Bn * H * N, torch.float32)
            _lib.call("smbv_attn_small_fwd", *(_vp(t, b) for t, b in zip(src, offs)), *strides, Bn, H, N, hd, float(scale),
                      _vp(o), _vp(lse), _stream())
            torch.cuda.synchronize()
            tl.expect(guards_intact(ob, Bn * N * d) and guards_intact(lb, Bn * H * N), f"{what}: fwd guard bytes changed")
            tl.expect(bool(torch.isfinite(o.float()).all() and torch.isfinite(lse).all()), f"{what}: NaN left in out / lse")
            outs.append((o, lse))
        tl.expect(torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]), f"{what}: fwd not bit-identical")
        oh = heads(outs[0][0].view(Bn, N, d), Bn, H)
        tl.add("row", tile_frob(oh, ref["o"], 1), SMALL["row"], f"{what} O")
        tl.add("ulps", bf16_ulps(oh, ref["o"]), SMALL["ulps"], f"{what} O")
        tl.add("lse", (outs[0][1].view(-1, N).double() - ref["lse"]).abs().max().item(), SMALL["lse"], what)
        # backward from the fp64 O (rounded to bf16) and lse (rounded to fp32)
        o_in = tokens(ref["o"].bfloat16(), Bn, H).contiguous()
        lse_in = ref["lse"].float().contiguous()
        grads = []
        for _ in range(2):
            if layout == "token-major":
                db, (dqkv,) = guarded(Bn * N * 3 * d, torch.bfloat16)
                dst, n_g, reg = (dqkv, dqkv, dqkv), Bn * N * 3 * d, 1
            else:
                db, views = guarded(Bn * H * N * hd, torch.bfloat16, 3)
                dst, n_g, reg = tuple(views), Bn * H * N * hd, 3
            dsum = torch.empty(Bn * H * N, device=DEV)
            _lib.call("smbv_attn_small_bwd", *(_vp(t, b) for t, b in zip(src, offs)), *strides, _vp(o_in), _vp(do), _vp(lse_in),
                      Bn, H, N, hd, float(scale), _vp(dsum), *(_vp(t, b) for t, b in zip(dst, offs)), *strides, _stream())
            torch.cuda.synchronize()
            tl.expect(guards_intact(db, n_g, reg), f"{what}: bwd guard bytes changed")
            if layout == "token-major":
                gq, gk, gv = (dqkv.view(Bn, N, 3, H, hd)[:, :, i].permute(0, 2, 1, 3).reshape(Bn * H, N, hd) for i in range(3))
            else:
                gq, gk, gv = (t.view(Bn * H, N, hd) for t in views)
            grads.append((gq, gk, gv))
        tl.expect(all(torch.equal(a, b) for a, b in zip(*grads)), f"{what}: bwd not bit-identical")
        for name, t in zip(("dq", "dk", "dv"), grads[0]):
            tl.expect(bool(torch.isfinite(t.float()).all()), f"{what}: NaN left in {name}")
            term = ref["t" + name[1]]
            tl.add("row", tile_frob(t, ref[name], 1, term), SMALL["row"], f"{what} {name}")
            tl.add("ulps", bf16_ulps(t, ref[name], term), SMALL["ulps"], f"{what} {name}")
        if N == 300:  # negative control: key row 150 dropped from O (every query) and from dQ
            bad_o = torch.stack([_rows(q, k, v, heads(do, Bn, H), ref["o"], lse_in, bh, slice(0, N), scale, [150])[0]
                                 for bh in range(Bn * H)])
            _, _, _, ds = _rows(q, k, v, heads(do, Bn, H), ref["o"].bfloat16(), lse_in, 0, slice(0, N), scale)
            bad_dq = ref["dq"][0] - scale * ds[:, 150:151] @ k[0, 150:151].double()
            ctrl = min(ctrl, tile_frob(oh, bad_o, 1) / SMALL["row"], tile_frob(grads[0][0][:1], bad_dq[None], 1, ref["tq"][:1]) / SMALL["row"])
    report(f"attn_small hd={hd} {layout}", tl.worst, SMALL)
    print(f"  negative control (one key row dropped, O and dQ): worst row / bound >= {ctrl:.1f}")
    tl.expect(ctrl >= CONTROL_BF16, f"negative control margin {ctrl:.1f} < {CONTROL_BF16}")
    assert not tl.fails, "\n".join(tl.fails[:20])
