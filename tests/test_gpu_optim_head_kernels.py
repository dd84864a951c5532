"""Kernel-level parity of the optimiser step, the EMA target update and the classification head (run with -m gpu on the
B200 box): `smbv_sumsq_f32` (global gradient norm), `smbv_adamw_step` (clip + AdamW + bf16 operand refresh over the flat
arena), `smbv_ema_update`, `smbv_cls_head` (fc_norm -> classifier -> MSE / CE / BCE and its whole backward) and
`smbv_broadcast_rows`.  End-to-end tests compare weight matrices after a few steps at 5e-2; a wrong decay flag on one
segment moves a parameter by lr * wd * p ~ 1e-5 p per step, so each kernel is compared here on its own, through the C ABI,
with a float64 reference computed ON THE DEVICE from the exact fp32 operands the kernel reads.

Bounds (worst measured on one NVIDIA B200 at a 1000 W power limit in brackets):
  global norm: relative error of the sum of squares and of every per-CTA partial <= 1e-6  [total 5.7e-8, partial 2.4e-7];
  AdamW, one step from the kernel's own fp32 state, per element, in units of 2^-23 of the magnitude of the summed terms:
      p <= 2 (terms |p dk| + step_size (|b1 m| + |(1-b1) g| + |m'|) / denom)  [1.02],
      m <= 2 (terms |b1 m| + |(1-b1) g|)  [1.21],  v <= 2 (v')  [1.57];
      bf16 copy: bit-exact round-to-nearest-even of the new p; frozen segments and lr = 0: bit-unchanged;
      decay-flag isolation (g = m = v = 0, lr wd = 0.5): bit-exact p / 2 or p;
  EMA: bit-identical to torch's `t.mul_(m).add_(s, alpha=1-m)`; against fp64 <= 1 unit of 2^-23 of |m t| + |(1-m) s|, which
      two roundings cannot exceed  [1.0, at m = 1 - 2^-24];
  classification head, per row (logits: per element) relative to the L2 norm of the magnitudes of the summed terms:
      <= 1e-5  [logits 8.5e-7, loss 9.3e-8, dW 1.8e-7, dbias 1.5e-6, dgamma 1.8e-7, dbeta 1.1e-7, dpooled 5.0e-7];
      MSE with labels equal to the logits: every gradient exactly 0;
  broadcast rows: bit-exact fp32 and bf16 round-to-nearest-even.
Negative controls, worst (smallest) measured: global norm 1.8e-3 (1800x its bound, at 328 M elements, where the largest of
1184 partials is 0.18 % of the sum); AdamW flag flip 8.4e3 and clip ignored 8.4e12; EMA 1.2e4; head 0.030.  The whole
module runs in about 15 s.
Every output a kernel overwrites is a NaN-prefilled view between guard regions; accumulated outputs (dW, dbias, dgamma,
dbeta) are prefilled with random values and checked as prefill + increment; every output is bit-identical on a second call.
Each family has a negative control that must fail its bound by >= 100x: one partial dropped from the norm, one segment's
decay flag flipped, the clip ignored, the last float4 of the EMA target left unchanged, one label's dW row missing, one
broadcast row taken from the next sample.
"""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

GUARD, SENTINEL = 256, 7.0
U23 = 2.0 ** -23
CONTROL = 100.0
CHUNK = 1 << 24  # elements per fp64 reference chunk (a few hundred MB of temporaries)

SUMSQ_REL = 1e-6
ADAM_P, ADAM_M, ADAM_V = 2.0, 2.0, 2.0
EMA_U = 1.0
HEAD_REL = 1e-5

SUMSQ_CTAS, CTA_THREADS = 1184, 256  # optim.cu: SUMSQ_BLOCKS, and the AdamW / EMA grid cap (148 SMs x 8)
GRID_STRIDE4 = SUMSQ_CTAS * CTA_THREADS  # float4 groups per grid-stride step of adamw_kernel / ema_kernel
VITB_MIM_N, VJEPA_L_N = 97_171_840, 328_592_768  # the flat arenas of bench.py's MIM and V-JEPA models


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


def guarded(shape, dtype=torch.float32, fill=float("nan")):
    """(buffer, view): a view prefilled with `fill` between two guard regions of SENTINEL (16-byte aligned)."""
    n = math.prod(shape)
    buf = torch.full((n + 2 * GUARD,), fill, dtype=dtype, device=DEV)
    buf[:GUARD] = SENTINEL
    buf[GUARD + n:] = SENTINEL
    return buf, buf[GUARD:GUARD + n].view(shape)


def guards_ok(buf):
    return bool((buf[:GUARD] == SENTINEL).all() and (buf[-GUARD:] == SENTINEL).all())


def bits(t):
    return t.view({torch.float32: torch.int32, torch.bfloat16: torch.int16}[t.dtype])


def same_bits(a, b):
    return torch.equal(bits(a), bits(b))


def chunks(n):
    for s in range(0, n, CHUNK):
        yield slice(s, min(n, s + CHUNK))


def report(name, worst, bounds, ctrl=None):
    line = f"{name}: " + ", ".join(f"{k} {worst[k]:.3g} (bound {bounds[k]:.3g})" for k in bounds if k in worst)
    print(line + ("" if ctrl is None else f"; negative control {ctrl:.3g}"))


def spread_values(n, g):
    """randn scaled per 4096-element block by 10^U(-8, 3): gradients of layers several decades apart."""
    nb = (n + 4095) // 4096
    x = torch.randn(nb, 4096, device=DEV, generator=g)
    x *= torch.pow(10.0, torch.rand(nb, 1, device=DEV, generator=g) * 11 - 8)
    return x.view(-1)[:n]


# =====================================================================================================================
# 1. global gradient norm: smbv_sumsq_f32
# =====================================================================================================================
def sumsq_partials64(x):
    """fp64 sum of squares of what each of the 1184 CTAs of sumsq_partial_kernel reads (float4 i -> CTA (i / 256) % 1184)."""
    R = SUMSQ_CTAS * CTA_THREADS * 4
    n = x.numel()
    full = n // R
    part = torch.zeros(SUMSQ_CTAS, dtype=torch.float64, device=DEV)
    rows = max(1, CHUNK // R)
    for r0 in range(0, full, rows):
        r1 = min(full, r0 + rows)
        part += x[r0 * R:r1 * R].view(r1 - r0, SUMSQ_CTAS, CTA_THREADS * 4).double().square().sum((0, 2))
    if n > full * R:
        tail = torch.zeros(R, dtype=torch.float64, device=DEV)
        tail[:n - full * R] = x[full * R:].double()
        part += tail.view(SUMSQ_CTAS, CTA_THREADS * 4).square().sum(1)
    return part


@pytest.mark.parametrize("n", [4, GRID_STRIDE4 * 4 - 4, GRID_STRIDE4 * 4 + 4, VITB_MIM_N, VJEPA_L_N])
def test_sumsq_matches_fp64(lib, n):
    """Squared global gradient norm: every per-CTA partial and the final sum against fp64, with values spanning 1e-8 .. 1e3
    per block; the grid-stride partition is fixed to 1184 CTAs, so n = 1184*256*4 +- 4 puts one float4 more or less than
    a whole round on CTA 0, and the two real arena sizes run ~80 and ~270 float4 per thread."""
    g = torch.Generator(device=DEV).manual_seed(n % 100003)
    buf, x = guarded((n,))
    x.copy_(spread_values(n, g))
    ws_buf, ws = guarded((SUMSQ_CTAS,))
    out_buf, out = guarded((1,))
    call("smbv_sumsq_f32", ptr(x), n, ptr(ws), ptr(out))
    assert guards_ok(ws_buf) and guards_ok(out_buf) and guards_ok(buf)
    part = sumsq_partials64(x)
    ref = part.sum().item()
    assert torch.isfinite(ws).all() and math.isfinite(out.item())
    worst = {"partial": ((ws.double() - part).abs() / part.clamp_min(1e-300)).max().item(),
             "total": abs(out.item() - ref) / ref}
    ws2_buf, ws2 = guarded((SUMSQ_CTAS,))
    out2_buf, out2 = guarded((1,))
    call("smbv_sumsq_f32", ptr(x), n, ptr(ws2), ptr(out2))
    assert same_bits(ws2, ws) and same_bits(out2, out)
    # negative control: the reference without its largest partial
    ctrl = abs(out.item() - (ref - part.max().item())) / ref
    report(f"sumsq n={n}", worst, dict(partial=SUMSQ_REL, total=SUMSQ_REL), ctrl)
    if n <= CTA_THREADS * 4:
        assert (part[1:] == 0).all() and (ws[1:] == 0).all()  # CTAs with nothing to read contribute exact zeros
    assert worst["partial"] <= SUMSQ_REL and worst["total"] <= SUMSQ_REL
    assert ctrl >= CONTROL * SUMSQ_REL


# =====================================================================================================================
# 2. AdamW: smbv_adamw_step
# =====================================================================================================================
B1, B2, EPS = 0.9, 0.999, 1e-8


def f32(x):
    return float(torch.tensor(x, dtype=torch.float32))


def synthetic_table(n4, nseg, g, first_frozen=False, last_frozen=False):
    """A segment table of nseg entries over n4 float4 groups: one-float4 segments, starts on grid-stride multiples
    (k * 1184 * 256), adjacent equal flags left unmerged, flags 0 / 1 / 2."""
    assert n4 >= 4 * nseg
    fixed = {1, 2, 3}  # segments 1 and 2 are one float4 long
    fixed |= {k * GRID_STRIDE4 for k in range(1, n4 // GRID_STRIDE4 + 1) if k * GRID_STRIDE4 < n4}
    fixed |= {n4 - 1}  # the last segment is one float4 long
    fixed = sorted(fixed)[:max(0, nseg - 1)]
    need = nseg - 1 - len(fixed)
    pool = torch.randperm(n4 - 1, device=DEV, generator=g)[:need + len(fixed) + 8] + 1
    extra = [int(s) for s in pool.tolist() if int(s) not in fixed][:need]
    starts = [0] + sorted(fixed + extra)
    assert len(starts) == nseg and len(set(starts)) == nseg
    flags = torch.randint(0, 3, (nseg,), device=DEV, generator=g)
    if nseg >= 4:
        flags[1] = flags[2]  # equal neighbours, not merged
    flags[0] = 2 if first_frozen else 0
    if last_frozen:
        flags[-1] = 2
    elif nseg > 1:
        flags[-1] = 1
    return torch.tensor(starts, dtype=torch.int32, device=DEV), flags.to(torch.uint8)


def real_table(kind):
    """The decay-segment table of a full-size model, built on the meta device (no weights allocated)."""
    from transformers import VideoMAEConfig, VJEPA2Config

    from smb_vision_b200.training import ArenaLayout

    with torch.device("meta"):
        if kind == "vit-b-mim":
            from smb_vision_b200.modeling import B200VideoMAEForPreTraining

            c = VideoMAEConfig()
            c.update(dict(image_size=512, patch_size=16, num_channels=1, num_frames=320, tubelet_size=16))
            model = B200VideoMAEForPreTraining(c)
        else:
            from smb_vision_b200.vjepa import B200VJEPA2Model

            model = B200VJEPA2Model(VJEPA2Config(patch_size=16, crop_size=384, frames_per_clip=256, tubelet_size=16, in_chans=1))
    lay = ArenaLayout(model)
    starts, flags = lay.decay_segments()
    return lay.total, torch.tensor(starts, dtype=torch.int32, device=DEV), torch.tensor(flags, dtype=torch.uint8, device=DEV)


def element_flags(starts, flags, n):
    n4 = n // 4
    lens = torch.diff(torch.cat([starts.long(), torch.tensor([n4], device=DEV)]))
    assert (lens > 0).all()
    return torch.repeat_interleave(flags, lens).repeat_interleave(4)


class AdamState:
    """Guarded fp32 p / m / v, a guarded bf16 copy (NaN, SENTINEL where frozen) and the kernel's inputs kept for the reference."""

    def __init__(self, n, fl, g, m0="randn", v0="randn", zero_grad=False):
        self.n, self.fl = n, fl
        self.pbuf, self.p = guarded((n,))
        self.mbuf, self.m = guarded((n,))
        self.vbuf, self.v = guarded((n,))
        self.bbuf, self.pb = guarded((n,), torch.bfloat16)
        self.p.copy_(torch.randn(n, device=DEV, generator=g))
        self.grad = torch.zeros(n, device=DEV) if zero_grad else spread_values(n, g).contiguous()
        self.m.copy_(torch.zeros(n, device=DEV) if m0 == "zero" else torch.randn(n, device=DEV, generator=g) * 1e-3)
        self.v.copy_(torch.zeros(n, device=DEV) if v0 == "zero" else torch.rand(n, device=DEV, generator=g) * 1e-5)
        self.pb[fl == 2] = SENTINEL
        zero = torch.zeros(1, device=DEV).expand(n)  # zero moments are not copied (the full-size arenas)
        self.m0 = zero if m0 == "zero" else self.m.clone()
        self.v0 = zero if v0 == "zero" else self.v.clone()
        self.p0, self.pb0 = self.p.clone(), self.pb.clone()

    def run(self, starts, flags, lr, wd, step, nsq=None, max_norm=1.0, pb=True):
        call("smbv_adamw_step", ptr(self.p), ptr(self.pb) if pb else 0, ptr(self.grad), ptr(self.m), ptr(self.v), self.n, ptr(starts),
             ptr(flags), starts.numel(), lr, B1, B2, EPS, wd, step, ptr(nsq), max_norm)
        assert all(guards_ok(b) for b in (self.pbuf, self.mbuf, self.vbuf, self.bbuf))

    def outputs(self):
        return self.p.clone(), self.m.clone(), self.v.clone(), self.pb.clone()

    def restore(self):
        self.p.copy_(self.p0), self.m.copy_(self.m0), self.v.copy_(self.v0), self.pb.copy_(self.pb0)


def adam_check(st, lr, wd, step, clip, worst, decay_fl=None):
    """Per-element parity of one step against torch.optim.AdamW's formula in fp64 from the kernel's fp32 inputs; bf16 copy
    bit-exact RN of the new p; frozen (flag 2) p / m / v / bf16 bit-unchanged.  `decay_fl` overrides the per-element flags of
    the REFERENCE (negative control); returns the worst p metric of the elements whose reference flag differs."""
    b1, b2 = f32(B1), f32(B2)
    omb1, omb2 = 1.0 - b1, 1.0 - b2
    lr32, wd32, eps32 = f32(lr), f32(wd), f32(EPS)
    bc1 = 1.0 - b1 ** step
    step_size = lr32 / bc1
    bc2_rsqrt = 1.0 / math.sqrt(1.0 - b2 ** step)
    ctrl = 0.0
    for s in chunks(st.n):
        fl = st.fl[s]
        rfl = fl if decay_fl is None else decay_fl[s]
        frz = fl == 2
        p0, m0, v0, g = st.p0[s].double(), st.m0[s].double(), st.v0[s].double(), st.grad[s].double() * clip
        dk = torch.where(rfl == 0, 1.0 - lr32 * wd32, 1.0)
        m = b1 * m0 + omb1 * g
        v = b2 * v0 + omb2 * g * g
        denom = v.sqrt() * bc2_rsqrt + eps32
        p = p0 * dk - step_size * m / denom
        sm = (b1 * m0).abs() + (omb1 * g).abs()
        sp = (p0 * dk).abs() + step_size * (sm + m.abs()) / denom
        live = ~frz
        ep = ((st.p[s].double() - p).abs() / (U23 * sp).clamp_min(1e-300))
        if decay_fl is not None:
            diff = live & (rfl != fl)
            if diff.any():
                ctrl = max(ctrl, ep[diff].max().item())
            continue
        em = ((st.m[s].double() - m).abs() / (U23 * sm).clamp_min(1e-300))
        ev = ((st.v[s].double() - v).abs() / (U23 * v).clamp_min(1e-300))
        # exact zeros: an element whose reference is exactly 0 must come out exactly 0
        em = torch.where(sm == 0, (st.m[s] != 0).double() * 1e30, em)
        ev = torch.where(v == 0, (st.v[s] != 0).double() * 1e30, ev)
        if live.any():
            for k, e in (("p", ep), ("m", em), ("v", ev)):
                worst[k] = max(worst.get(k, 0.0), e[live].max().item())
        assert torch.isfinite(st.p[s]).all()
        assert same_bits(st.p[s][frz], st.p0[s][frz]) and same_bits(st.m[s][frz], st.m0[s][frz]) and same_bits(st.v[s][frz], st.v0[s][frz])
        assert (st.pb[s][frz] == SENTINEL).all()
        assert same_bits(st.pb[s][live], st.p[s][live].bfloat16())
    return ctrl


def assert_adam(worst):
    assert worst.get("p", 0) <= ADAM_P and worst.get("m", 0) <= ADAM_M and worst.get("v", 0) <= ADAM_V, worst


TABLES = [(1, 1 << 14, False, False), (5, 1 << 14, True, False), (255, 1 << 16, False, True), (256, 1 << 16, True, True),
          (257, 1 << 16, False, False), (582, GRID_STRIDE4 * 3 + 777, True, False), (4096, GRID_STRIDE4 * 2 + 5, False, True)]


@pytest.mark.parametrize("nseg,n4,first_frozen,last_frozen", TABLES)
def test_adamw_segment_tables(lib, nseg, n4, first_frozen, last_frozen):
    """Segment lookup (shared-memory table filled in a 256-stride loop, binary search per float4) for 1 .. 4096 segments:
    (a) decay-flag isolation, g = m = v = 0 and lr wd = 0.5: p must become exactly p / 2 where the flag is 0 and stay
    bit-unchanged where it is 1 or 2; (b) one ordinary step against the fp64 reference; (c) the bf16 copy and frozen
    segments; (d) bit-identical on a second call.  Control: a reference with one segment's flag flipped."""
    g = torch.Generator(device=DEV).manual_seed(nseg * 31 + n4)
    starts, flags = synthetic_table(n4, nseg, g, first_frozen, last_frozen)
    n = 4 * n4
    fl = element_flags(starts, flags, n)
    # (a) decay-flag isolation
    st = AdamState(n, fl, g, m0="zero", v0="zero", zero_grad=True)
    st.run(starts, flags, 0.5, 1.0, 1)
    want = torch.where(fl == 0, st.p0 * 0.5, st.p0)
    assert same_bits(st.p, want), int((bits(st.p) != bits(want)).sum())
    assert (st.m == 0).all() and (st.v == 0).all()
    assert same_bits(st.pb[fl != 2], st.p[fl != 2].bfloat16()) and (st.pb[fl == 2] == SENTINEL).all()
    # (b)-(d) an ordinary step, clipped
    worst = {}
    st = AdamState(n, fl, g)
    nsq = torch.tensor([float(st.grad.double().square().sum())], device=DEV)
    clip = min(1.0, 1.0 / (math.sqrt(nsq.item()) + 1e-6))
    st.run(starts, flags, 1e-2, 0.1, 7, nsq)
    adam_check(st, 1e-2, 0.1, 7, clip, worst)
    out = st.outputs()
    st.restore()
    st.run(starts, flags, 1e-2, 0.1, 7, nsq)
    assert all(same_bits(a, b) for a, b in zip(st.outputs(), out))
    # negative control: the reference with the largest non-frozen segment's decay flag flipped
    lens = torch.diff(torch.cat([starts.long(), torch.tensor([n4], device=DEV)]))
    k = int(torch.where(flags == 2, 0, lens).argmax())
    ctrl = 0.0
    if flags[k] != 2:
        bad = flags.clone()
        bad[k] = 1 - bad[k]
        ctrl = adam_check(st, 1e-2, 0.1, 7, clip, {}, element_flags(starts, bad, n))
    report(f"adamw nseg={nseg} n4={n4}", worst, dict(p=ADAM_P, m=ADAM_M, v=ADAM_V), ctrl)
    assert_adam(worst)
    assert flags[k] == 2 or ctrl >= CONTROL * ADAM_P


@pytest.mark.parametrize("kind", ["vit-b-mim", "vjepa-vit-l"])
def test_adamw_real_arena_tables(lib, kind):
    """The decay-segment tables of the two full-size arenas (132 segments over 97 171 840 elements, and V-JEPA ViT-L's over
    328 592 768): the first step (m = v = 0) against the fp64 reference, then decay-flag isolation on the same buffers."""
    n, starts, flags = real_table(kind)
    assert n == (VITB_MIM_N if kind == "vit-b-mim" else VJEPA_L_N)
    g = torch.Generator(device=DEV).manual_seed(n % 1000)
    fl = element_flags(starts, flags, n)
    st = AdamState(n, fl, g, m0="zero", v0="zero")
    worst = {}
    st.run(starts, flags, 5e-5, 0.01, 1)
    adam_check(st, 5e-5, 0.01, 1, 1.0, worst)
    report(f"adamw {kind} ({starts.numel()} segments)", worst, dict(p=ADAM_P, m=ADAM_M, v=ADAM_V))
    assert_adam(worst)
    st.grad.zero_(), st.m.zero_(), st.v.zero_()
    st.p0.copy_(st.p)
    st.run(starts, flags, 0.5, 1.0, 2)
    for s in chunks(n):
        assert same_bits(st.p[s], torch.where(fl[s] == 0, st.p0[s] * 0.5, st.p0[s])), s
        assert same_bits(st.pb[s], st.p[s].bfloat16())


STEP_CASES = [  # (step, lr, norm case)
    (1, 1e-3, "below"), (2, 1e-3, "above"), (10, 1e-3, "null"), (10_000, 1e-3, "zero"), (1_000_000, 1e-3, "above"),
    (1, 0.0, "above"), (3, 0.0, "null")]


@pytest.mark.parametrize("step,lr,norm", STEP_CASES)
def test_adamw_steps_and_clipping(lib, step, lr, norm):
    """Bias corrections at step 1, 2, 10, 1e4 and 1e6; lr = 0 (the first step of cosine_with_warmup: p bit-unchanged, m and v
    still move); gradient norm 0 (with zero gradients), below max_norm, 1e6 x above it, and grad_norm_sq = NULL.
    Control: the reference without the clip."""
    g = torch.Generator(device=DEV).manual_seed(step + int(lr * 1e6))
    n4 = GRID_STRIDE4 + 333
    starts, flags = synthetic_table(n4, 40, g, True, False)
    n = 4 * n4
    fl = element_flags(starts, flags, n)
    st = AdamState(n, fl, g, zero_grad=(norm == "zero"))
    true = float(st.grad.double().square().sum())
    sq = {"zero": 0.0, "below": 0.25, "above": 1e12, "null": None}[norm]
    if norm == "below":
        st.grad *= 0.5 / math.sqrt(true)
    elif norm == "above":
        st.grad *= 1e6 / math.sqrt(true)
    nsq = None if sq is None else torch.tensor([sq], device=DEV)
    n32 = None if sq is None else nsq.item()
    clip = 1.0 if sq is None else min(1.0, f32(1.0) / (math.sqrt(n32) + 1e-6))
    worst = {}
    st.run(starts, flags, lr, 0.05, step, nsq, 1.0)
    adam_check(st, lr, 0.05, step, clip, worst)
    if lr == 0.0:
        assert same_bits(st.p, st.p0)
        assert not torch.equal(st.m, st.m0) and not torch.equal(st.v, st.v0)
    out = st.outputs()
    st.restore()
    st.run(starts, flags, lr, 0.05, step, nsq, 1.0)
    assert all(same_bits(a, b) for a, b in zip(st.outputs(), out))
    ctrl = None
    if norm == "above":  # negative control: the m of a reference that ignores the clip (the gradient term 1e6 x too large)
        b1 = f32(B1)
        m_bad = b1 * st.m0.double() + (1.0 - b1) * st.grad.double()
        sm = (b1 * st.m0.double()).abs() + ((1.0 - b1) * st.grad.double() * clip).abs()
        ctrl = ((st.m.double() - m_bad).abs() / (U23 * sm).clamp_min(1e-300))[fl != 2].max().item()
    report(f"adamw step={step} lr={lr} norm={norm}", worst, dict(p=ADAM_P, m=ADAM_M, v=ADAM_V), ctrl)
    assert_adam(worst)
    if ctrl is not None:
        assert ctrl >= CONTROL * ADAM_M


def test_adamw_without_bf16_copy_and_argument_checks(lib):
    """param_bf16 = NULL skips the copy (the V-JEPA target arena has none); the C ABI rejects nseg = 0 / 4097 and step 0."""
    from smb_vision_b200._lib import SmbvError

    g = torch.Generator(device=DEV).manual_seed(5)
    starts, flags = synthetic_table(4096, 9, g)
    fl = element_flags(starts, flags, 4 * 4096)
    st = AdamState(4 * 4096, fl, g)
    worst = {}
    st.run(starts, flags, 1e-3, 0.01, 4, pb=False)
    assert same_bits(st.pb, st.pb0)
    st.pb[fl != 2] = st.p[fl != 2].bfloat16()  # what adam_check expects of a bf16 copy; p, m and v are checked as usual
    adam_check(st, 1e-3, 0.01, 4, 1.0, worst)
    assert_adam(worst)
    for nseg, step in ((0, 1), (4097, 1), (9, 0)):
        with pytest.raises(SmbvError):
            call("smbv_adamw_step", ptr(st.p), 0, ptr(st.grad), ptr(st.m), ptr(st.v), st.n, ptr(starts), ptr(flags), nseg, 1e-3, B1, B2,
                 EPS, 0.01, step, 0, 1.0)


# =====================================================================================================================
# 3. EMA: smbv_ema_update
# =====================================================================================================================
@pytest.mark.parametrize("n", [4, GRID_STRIDE4 * 4 + 4, VITB_MIM_N, VJEPA_L_N])
def test_ema_matches_torch_bitwise_and_fp64(lib, n):
    """target = m target + (1 - m) source for m = 0, 0.5, 0.99925 (V-JEPA), 1 - 2^-24 and 1: bit-identical to torch's
    `t.mul_(m).add_(s, alpha=1-m)` on the device, and against fp64 within the kernel's two roundings.
    Control (m = 0.5, 0.99925): the reference with the last float4 of the target left unchanged."""
    g = torch.Generator(device=DEV).manual_seed(n % 9973)
    src = torch.randn(n, device=DEV, generator=g)
    t0 = torch.randn(n, device=DEV, generator=g)
    buf, t = guarded((n,))
    for mom in (0.0, 0.5, 0.99925, 1.0 - 2.0 ** -24, 1.0):
        t.copy_(t0)
        call("smbv_ema_update", ptr(t), ptr(src), n, mom, float(1.0 - mom))
        assert guards_ok(buf)
        want = t0.clone().mul_(mom).add_(src, alpha=1.0 - mom)
        assert same_bits(t, want), (mom, int((bits(t) != bits(want)).sum()))
        t.copy_(t0)
        call("smbv_ema_update", ptr(t), ptr(src), n, mom, float(1.0 - mom))
        assert same_bits(t, want)  # second call: the same bits
        del want
        m32, om32 = f32(mom), f32(1.0 - mom)
        worst, ctrl = 0.0, float("inf")
        for s in chunks(n):
            a, b = m32 * t0[s].double(), om32 * src[s].double()
            ref, scale = a + b, a.abs() + b.abs()
            e = (t[s].double() - ref).abs() / (U23 * scale).clamp_min(1e-300)
            e = torch.where(scale == 0, (t[s] != 0).double() * 1e30, e)
            worst = max(worst, e.max().item())
            if s.stop == n and 0.0 < mom < 0.9999:
                bad = ref.clone()
                bad[-4:] = t0[s][-4:].double()
                ctrl = ((t[s][-4:].double() - bad[-4:]).abs() / (U23 * scale[-4:])).max().item()
        print(f"ema n={n} m={mom!r}: {worst:.3g} (bound {EMA_U})" + ("" if ctrl == float("inf") else f"; negative control {ctrl:.3g}"))
        assert worst <= EMA_U, mom
        assert ctrl >= CONTROL * EMA_U


# =====================================================================================================================
# 4. classification head: smbv_cls_head
# =====================================================================================================================
NONE, MSE, CE, BCE = 0, 1, 2, 3  # SMBV_CLS_*
HEAD_SHAPES = [  # (B, d, F, L, fc_norm, inv_n = 1)
    (1, 64, 0, 1, True, False), (4, 100, 1, 2, True, False), (33, 768, 300, 7, True, False), (4, 1000, 0, 8, False, True),
    (33, 1024, 1, 9, True, False), (4, 768, 2, 33, True, False), (1, 1024, 300, 1000, True, True), (33, 100, 0, 1000, False, False),
    (4, 64, 300, 33, False, False), (1, 768, 0, 9, False, True), (33, 1000, 1, 7, True, False), (4, 4096, 0, 3000, True, False)]


def head_inputs(B, d, F_, L, norm, inv_one, g, N=1960):
    pooled = torch.randn(B, d, device=DEV, generator=g) * (1.0 if inv_one else N ** 0.5) + 0.3
    inv_n = 1.0 if inv_one else 1.0 / N
    gamma = 1 + 0.1 * torch.randn(d, device=DEV, generator=g) if norm else None
    beta = 0.1 * torch.randn(d, device=DEV, generator=g) if norm else None
    feats = torch.randn(B, F_, device=DEV, generator=g) if F_ else None
    W = torch.randn(L, d + F_, device=DEV, generator=g) / math.sqrt(d + F_)
    bias = 0.1 * torch.randn(L, device=DEV, generator=g)
    return dict(pooled=pooled, inv_n=inv_n, gamma=gamma, beta=beta, feats=feats, W=W, bias=bias)


def head_labels(problem, B, L, g):
    if problem == CE:
        return torch.randint(0, L, (B,), device=DEV, generator=g)
    if problem == MSE:
        return torch.randn(B, L, device=DEV, generator=g)
    if problem == BCE:
        return (torch.rand(B, L, device=DEV, generator=g) > 0.5).float()
    return None


def prefill_scales(ref, d, D):
    """Per-element size of each accumulator's increment: the prefill gets the same size (as in the backward-kernel tests),
    so that the fp32 rounding of prefill + increment stays at the scale of the increment."""
    if "sdW" not in ref:
        return {}
    s = dict(dW=ref["sdW"][:, None] / math.sqrt(D), dbias=ref["sdbias"])
    if "sdgamma" in ref:
        s.update(dgamma=ref["sdgamma"] / math.sqrt(d), dbeta=ref["sdbeta"] / math.sqrt(d))
    return {k: v.float() for k, v in s.items()}


class HeadOut:
    def __init__(self, B, d, F_, L, norm, train, g, scales=None):
        self.lbuf, self.logits = guarded((B, L))
        self.sbuf, self.loss = guarded((1,))
        self.pbuf, self.dpooled = guarded((B, d))
        self.acc = {}
        shapes = dict(dW=(L, d + F_), dbias=(L,), dgamma=(d,), dbeta=(d,))
        for k, shp in shapes.items():
            if k in ("dgamma", "dbeta") and not norm:
                continue
            buf, v = guarded(shp)
            v.copy_(torch.randn(shp, device=DEV, generator=g) * (scales or {}).get(k, 1.0))
            self.acc[k] = (buf, v, v.clone())
        self.train = train

    def bufs(self):
        return [self.lbuf, self.sbuf, self.pbuf] + [b for b, _, _ in self.acc.values()]


def head_call(x, labels, problem, out, with_acc=True):
    a = {k: v for k, (_, v, _) in out.acc.items()} if with_acc else {}
    B, d = x["pooled"].shape
    L, D = x["W"].shape
    call("smbv_cls_head", ptr(x["pooled"]), x["inv_n"], ptr(x["gamma"]), ptr(x["beta"]), 1e-5, ptr(x["feats"]), ptr(x["W"]), ptr(x["bias"]),
         ptr(labels), B, d, D - d, L, problem, ptr(out.logits), ptr(out.loss) if problem != NONE else 0, ptr(a.get("dW")), ptr(a.get("dbias")),
         ptr(a.get("dgamma")), ptr(a.get("dbeta")), ptr(out.dpooled) if out.train else 0)
    assert all(guards_ok(b) for b in out.bufs())


def head_reference(x, labels, problem):
    """fp64 autograd of LayerNorm -> cat -> Linear -> loss from the fp32 operands, plus magnitude scales of each output."""
    d = x["pooled"].shape[1]
    inv_n = f32(x["inv_n"])
    P = x["pooled"].double().requires_grad_(True)
    W = x["W"].double().requires_grad_(True)
    b = x["bias"].double().requires_grad_(True)
    norm = x["gamma"] is not None
    ga = x["gamma"].double().requires_grad_(True) if norm else None
    be = x["beta"].double().requires_grad_(True) if norm else None
    h = P * inv_n
    if norm:
        mu = h.mean(1, keepdim=True)
        rstd = ((h - mu).square().mean(1, keepdim=True) + f32(1e-5)).rsqrt()
        xh = (h - mu) * rstd
        hn = xh * ga + be
    else:
        xh, rstd, hn = None, None, h
    z = torch.cat([hn, x["feats"].double()], 1) if x["feats"] is not None else hn
    lg = z @ W.t() + b
    B, L = lg.shape
    r = dict(logits=lg.detach())
    zd = z.detach().abs()
    Wd = W.detach()
    lscale = ((zd[:, None, :] * Wd[None].abs()).square().sum(-1)).sqrt() + b.detach().abs()  # [B, L]
    r["lscale"] = lscale
    if problem == NONE:
        return r
    lgd = lg.detach()
    if problem == CE:
        loss = F.cross_entropy(lg, labels)
        lse = torch.logsumexp(lgd, 1, keepdim=True)
        p = (lgd - lse).exp()
        oh = F.one_hot(labels, L).double()
        dlmag = (p * (2 + lgd.abs() + lse.abs() + lscale) + oh) / B
        lterms = (lse.squeeze(1).abs() + lgd.gather(1, labels[:, None]).squeeze(1).abs()).sum() / B
    elif problem == MSE:
        t = labels.double()
        loss = F.mse_loss(lg, t)
        dlmag = 2 * ((lgd - t).abs() + lscale) / (B * L)
        lterms = ((lgd - t).square() + 2 * (lgd - t).abs() * lscale).sum() / (B * L)
    else:
        t = labels.double()
        loss = F.binary_cross_entropy_with_logits(lg, t)
        sg = torch.sigmoid(lgd)
        dlmag = (sg + t + sg * (1 - sg) * (lgd.abs() + lscale)) / (B * L)
        lterms = (lgd.clamp_min(0) + (lgd * t).abs() + torch.log1p(torch.exp(-lgd.abs())) + (sg - t).abs() * lscale).sum() / (B * L)
    loss.backward()
    dlmag = dlmag + 2.0 ** -126  # what underflows in fp32 (exp of a logit ~100 below the maximum) is lost, not wrong
    r.update(loss=loss.detach(), lscale_loss=lterms, dW=W.grad, dbias=b.grad, dpooled=P.grad)
    r["sdW"] = ((dlmag.t()[:, :, None] * zd[None]).square().sum((1, 2))).sqrt()  # per label row
    r["sdbias"] = dlmag.square().sum(0).sqrt()
    dzmag = (dlmag[:, :, None] * Wd[None, :, :d].abs()).square().sum(1).sqrt()  # [B, d]
    if norm:
        xhd = xh.detach()
        r.update(dgamma=ga.grad, dbeta=be.grad)
        r["sdgamma"] = (dzmag * xhd.abs()).square().sum().sqrt()
        r["sdbeta"] = dzmag.square().sum().sqrt()
        gmag = dzmag * x["gamma"].double().abs()
        c1, c2 = gmag.mean(1, keepdim=True), (gmag * xhd.abs()).mean(1, keepdim=True)
        r["sdpooled"] = (inv_n * rstd.detach() * (gmag + c1 + xhd.abs() * c2)).square().sum(1).sqrt()
    else:
        r["sdpooled"] = inv_n * dzmag.square().sum(1).sqrt()
    return r


def head_errors(out, ref, problem, worst):
    e = {"logits": ((out.logits.double() - ref["logits"]).abs() / ref["lscale"]).max().item()}
    if problem != NONE:
        e["loss"] = abs(out.loss.item() - ref["loss"].item()) / ref["lscale_loss"].item()
    if out.train:
        _, dW, pre = out.acc["dW"]
        e["dW"] = ((dW.double() - pre.double() - ref["dW"]).abs().max(1).values / ref["sdW"]).max().item()
        _, db, pre = out.acc["dbias"]
        e["dbias"] = ((db.double() - pre.double() - ref["dbias"]).abs() / ref["sdbias"]).max().item()
        for k in ("dgamma", "dbeta"):
            if k in out.acc:
                _, v, pre = out.acc[k]
                e[k] = ((v.double() - pre.double() - ref[k]).abs().max() / ref["s" + k]).item()
        e["dpooled"] = ((out.dpooled.double() - ref["dpooled"]).abs().max(1).values / ref["sdpooled"]).max().item()
    for k, v in e.items():
        worst[k] = max(worst.get(k, 0.0), v)
    return e


@pytest.mark.parametrize("B,d,F_,L,norm,inv_one", HEAD_SHAPES)
def test_cls_head_matches_fp64(lib, B, d, F_, L, norm, inv_one):
    """Forward only (problem NONE; and each loss without dpooled): logits, loss, accumulators untouched; training, for MSE /
    CE / BCE: loss, logits, dW, dbias, dgamma, dbeta and dpooled against fp64 autograd; every output bit-identical on a
    second call.  L > 8 runs the one-warp-per-label loop more than once, L > 32 the lane loops of the losses; d = 4096,
    L = 3000 needs more than 48 KB of shared memory.  Control: the reference without the largest label row of dW."""
    g = torch.Generator(device=DEV).manual_seed(B * 1000003 + d * 1009 + F_ * 31 + L)
    x = head_inputs(B, d, F_, L, norm, inv_one, g)
    worst, ctrl = {}, float("inf")
    for problem in (NONE, MSE, CE, BCE):
        labels = head_labels(problem, B, L, g)
        ref = head_reference(x, labels, problem)
        for train in ((False,) if problem == NONE else (False, True)):
            out = HeadOut(B, d, F_, L, norm, train, g, prefill_scales(ref, d, d + F_))
            head_call(x, labels, problem, out)
            e = head_errors(out, ref, problem, worst)
            assert all(v <= HEAD_REL for v in e.values()), (problem, train, e)
            if not train:
                assert all(same_bits(v, pre) for _, v, pre in out.acc.values())  # forward only: accumulators untouched
                assert torch.isnan(out.dpooled).all()
                if problem == NONE:
                    assert torch.isnan(out.loss).all()
                continue
            again = HeadOut(B, d, F_, L, norm, train, torch.Generator(device=DEV).manual_seed(0))
            for k, (_, v, pre) in again.acc.items():
                v.copy_(out.acc[k][2])
            head_call(x, labels, problem, again)
            assert same_bits(again.logits, out.logits) and same_bits(again.loss, out.loss) and same_bits(again.dpooled, out.dpooled)
            assert all(same_bits(again.acc[k][1], out.acc[k][1]) for k in out.acc)
            # negative control: the label row of dW with the largest increment (relative to its scale) missing from the reference
            rel = ref["dW"].abs().max(1).values / ref["sdW"]
            l = int(rel.argmax())
            if rel[l] > 0:  # (CE with one class: every gradient is exactly 0)
                _, dW, pre = out.acc["dW"]
                ctrl = min(ctrl, ((dW[l].double() - pre[l].double()).abs().max() / ref["sdW"][l]).item())
    report(f"cls_head B={B} d={d} F={F_} L={L} norm={norm} inv_n={'1' if inv_one else '1/N'}", worst,
           {k: HEAD_REL for k in worst}, ctrl)
    assert ctrl >= CONTROL * HEAD_REL


@pytest.mark.parametrize("case", ["ce80", "ce_high", "ce_low", "bce30", "bce100"])
def test_cls_head_hard_logits(lib, case):
    """Peaked losses: CE with logits at +-80 (one class far above the rest) and with every logit near +95 or -95 (exp
    overflows / underflows without the max subtraction); BCE at |x| = 30 and 100 (the sigmoid saturates)."""
    g = torch.Generator(device=DEV).manual_seed(len(case) * 7 + ord(case[-1]))
    B, d, F_, L = 4, 768, 2, 41
    x = head_inputs(B, d, F_, L, True, False, g)
    x["W"] *= 1e-3
    lab = torch.arange(L, device=DEV)
    x["bias"] = {"ce80": torch.where(lab % 5 == 0, 80.0, -80.0), "ce_high": 95.0 + 3 * torch.randn(L, device=DEV, generator=g),
                 "ce_low": -95.0 + 3 * torch.randn(L, device=DEV, generator=g), "bce30": torch.where(lab % 2 == 0, 30.0, -30.0),
                 "bce100": torch.where(lab % 2 == 0, 100.0, -100.0)}[case].contiguous()
    problem = CE if case.startswith("ce") else BCE
    labels = head_labels(problem, B, L, g)
    ref = head_reference(x, labels, problem)
    worst = {}
    out = HeadOut(B, d, F_, L, True, True, g, prefill_scales(ref, d, d + F_))
    head_call(x, labels, problem, out)
    e = head_errors(out, ref, problem, worst)
    report(f"cls_head {case}", worst, {k: HEAD_REL for k in worst})
    assert all(v <= HEAD_REL for v in e.values()), e


def test_cls_head_mse_labels_equal_logits(lib):
    """MSE with labels equal to the kernel's own logits: loss, every gradient increment and dpooled exactly 0."""
    g = torch.Generator(device=DEV).manual_seed(3)
    B, d, F_, L = 4, 768, 2, 9
    x = head_inputs(B, d, F_, L, True, False, g)
    out = HeadOut(B, d, F_, L, True, False, g)
    head_call(x, None, NONE, out)
    labels = out.logits.clone()
    out = HeadOut(B, d, F_, L, True, True, g)
    head_call(x, labels, MSE, out)
    assert out.loss.item() == 0.0 and (out.dpooled == 0).all()
    assert all(same_bits(v, pre) for _, v, pre in out.acc.values())


# =====================================================================================================================
# 5. smbv_broadcast_rows
# =====================================================================================================================
@pytest.mark.parametrize("N", [1, 1960, 20480])
@pytest.mark.parametrize("d", [4, 100, 768, 1024])
def test_broadcast_rows_bit_exact(lib, N, d):
    """dx[b, n, :] = g[b, :] in fp32 and its bf16 RN copy for B = 4, bit-exact; dx_bf16 = NULL writes only dx.
    Control: one row of the reference taken from the next sample must be seen."""
    B = 4
    gen = torch.Generator(device=DEV).manual_seed(N + d)
    src = torch.randn(B, d, device=DEV, generator=gen) * torch.pow(10.0, torch.randn(B, d, device=DEV, generator=gen) * 3)
    want = src[:, None, :].expand(B, N, d)
    for with_bf16 in (True, False):
        outs = []
        for _ in range(2):
            fbuf, dx = guarded((B, N, d))
            bbuf, dxb = guarded((B, N, d), torch.bfloat16)
            call("smbv_broadcast_rows", ptr(src), B, N, d, ptr(dx), ptr(dxb) if with_bf16 else 0)
            assert guards_ok(fbuf) and guards_ok(bbuf)
            assert same_bits(dx, want.contiguous())
            if with_bf16:
                assert same_bits(dxb, want.bfloat16().contiguous())
            else:
                assert torch.isnan(dxb).all()
            outs.append((dx, dxb))
        assert same_bits(outs[0][0], outs[1][0]) and same_bits(outs[0][1], outs[1][1])
    bad = want.clone()
    bad[0, N - 1] = src[1]
    assert not torch.equal(outs[0][0], bad)
