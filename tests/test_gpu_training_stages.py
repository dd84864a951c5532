"""Stage-by-stage parity of the MIM and classification training step (run with -m gpu on the B200 box): how
`training.mim_forward_train` / `mim_backward` and `cls_forward_train` / `cls_backward` wire the kernels together.  The
kernel-level files (test_gpu_forward_kernels.py, test_gpu_backward_kernels.py, test_gpu_attention_kernels.py,
test_gpu_optim_head_kernels.py) check every kernel on its own; the whole-model tests compare each gradient with the fp32
oracle at a Frobenius-rel of 2e-2, which cannot see a junction that drops one of ~140 masked rows or hands one sample's
LayerNorm statistics to another.  Here the real entry points run unchanged while a `Spy` records what they hand to each
kernel (ops.* and training.block_forward_train / block_backward), and every junction is compared with a float64
reference computed ON THE DEVICE from the exact bf16 / fp32 operands that stage read:

  forward:  patch embedding with the visible-row compaction (the patchify is taken from the volume here, not from the
            kernel's gathered rows; the saved rows must be exactly those) or the SimMIM blend; every encoder / decoder
            block at its junctions (x_mid = x_in + a Wo^T + bo, the LayerNorm statistics of x_in and x_mid, x_out = x_mid
            + f W2^T + b2); the final encoder LayerNorm or S.xb = bf16(X); the decoder input [Z We2d^T + PE_d[vis] |
            mask_token + PE_d[msk]] (SimMIM: all N rows in natural order); the head LayerNorm of each sample's masked rows
            with that sample's statistics, the logits and the loss read at msk[b];
  backward: dhN; the decoder-norm backward (visible rows exactly 0, SimMIM: scattered to msk); in every block dpre =
            (dXb W2) * gelu'(pre), dh2, the LN2 backward added into dX, dO, the attention backward's inputs, dh1 and the
            LN1 backward; the decoder-input split (mask-token gradient over rows n_vis:, dX = dZb We2d in fp32); the
            final-LayerNorm backward and the SimMIM blend; the classification broadcast and the CLS-row path;
  arena:    every parameter view of GradArena.flat against the fp64 sum of its stage contributions (from the stage
            operands, not from the list of calls the code made), the K-bias pad slot exactly 0, the alignment padding
            between segments still NaN; a second backward into the unzeroed arena gives twice the first; every
            data-parallel bucket is complete (bit-identical to the final arena) when its hook fires, on both
            SMBV_WGRAD_STREAM settings; the forward repeats bit for bit.

Bounds, each derived from the roundings of the stage (u = 2^-24; acc(n) = LAM sqrt(n) u, LAM = 4: the probabilistic
bound of an fp32 sum of n terms, relative to the sum of their magnitudes; the products of bf16 operands are exact):
  bf16 output of a GEMM (dgrad, logits):  1 bf16 ulp of ref + acc(K) sum_k |a_k w_k| (the accumulation before the one
      output rounding); dGELU: + DGELU_ABS |acc| (the epilogue's gelu' is within 1.8e-6 analytically, csrc/gemm.cu);
  fp32 output of a GEMM epilogue (patch embedding, decoder input, residual junctions, the fp32 e2d dgrad):
      acc(K) sum_k |a_k w_k| + 2u (|ref| + |every addend|);
  LayerNorm statistics: mean within acc(d) mean|x|; rstd within (acc(d) + 4u) relative (two-pass variance, rsqrt);
  LayerNorm output (bf16), with the saved statistics as the operands: 1 ulp + 4u (|x| + |mean|) rstd |gamma| + 4u |beta|;
  LayerNorm backward (fp32, added into dres): acc(d) rstd (|g| + mean|g| + |xhat| mean|g xhat|) (g = gamma dy, the two
      row means) + 2u (|dres before| + |ref|);
  every arena element (split-K reduce-adds, column sums, dgamma / dbeta): acc(n) sum over its n terms of |term| + 2u |ref|;
      a weight gradient adds n u / 8 of the same sum: the tensor-core accumulator truncates the running fp32 sum once per
      16-deep k-step (up to 2^-23 of it, with a bias, so the error grows linearly in n: test_gpu_backward_kernels.py,
      F32_LONG_K); without this term the 7168-row patch-embedding weight gradient exceeds acc(n) alone by 1.6x;
  token sum: acc(N) sum|x|;  loss: LOSS_REL relative; dlogits: 1 ulp + 2 / count LABEL_TOL (1 + |label|) (the bounds of
      test_gpu_forward_kernels.py for the norm-pix kernel alone);
  data movement and casts (saved patches, bf16 copies, the classification broadcast, the CLS-row seed): bit-exact;
  second backward into the same arena: Frobenius-rel <= REPRO_TOL to twice the first, per parameter (the split-K spread of
  test_side_stream_gradients_match_single_stream).
No element floor beyond these terms is needed: an element whose terms are all zero must come out exactly 0.

Worst measured values over every configuration, from one run on one NVIDIA B200 at a 1000 W power limit (value / bound;
smallest negative control / bound in brackets): patch embedding 0.030 [7.5e3]; block x_mid 0.22 [753], x_out 0.20 [9.2e3];
LayerNorm statistics <= 0.08 (head LN [5.2e4]); final / head LayerNorm output 0.50 [5.6e4]; decoder input 0.054 [3.1e4],
masked rows 0.50; logits 0.50; loss value 9.1e-3; dlogits 0.50 [4.2e5]; dhN 0.49 [5.5e3]; decoder-norm backward 0.075
[9.9e4]; dpre 0.50 [740]; dh2 0.50 [3.6e3]; LN2 backward 0.23 [1.2e6]; dO 0.50 [4.2e3]; dh1 0.50 [188]; LN1 backward 0.24;
e2d dgrad 0.059 [1.0e4]; final-LayerNorm backward 0.044 [8.3e4], CLS row 0.028 [1.1e4]; token sum 0.042 [4.3e3]; arena
0.45 (patch-embedding weight at 512x512x320 [562], mask token [2.0e4], SimMIM encoder mask token [1.8e5], fused QKV
weight without the last sample [9.1e4]); second backward 0.037 of REPRO_TOL.  Every bucket was complete at its hook.
The module runs in about 15 s.
Negative controls (each must fail its bound by >= 100x): the visible rows of another sample in the patch embedding and in
the decoder input (B = 1: rows rolled by one token); another sample's (token's) attention output at x_mid and MLP output at
x_out; another sample's statistics in the final, head and decoder-norm LayerNorms; dlogits with the labels in reverse mask order; another
sample's dlogits for dhN; gelu' from another block's pre; the LN2 backward without the residual add; dO from another
sample's dXb; dh1 without the dK third; the e2d dgrad from another sample; the mask-token gradient summed over the visible
rows (SimMIM: the encoder mask token over the visible rows); the fused QKV weight gradient without the last sample (B > 1).
Configurations: tiny (head_dim 16: the small-head branch of block_backward), SMALL64 (MAE, SimMIM, final LayerNorm,
classification with mean pooling and with the CLS row), base width at 160x160x96 with 2 encoder and 1 decoder layer at
B = 3 (own mask per sample, n_vis = 208), and base width at 512x512x320, B = 1, 2 + 1 layers.
"""
import math
import types

import numpy as np
import pytest
import torch

import __graft_entry__ as ge
from oracle import videomae_oracle as vo

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

U24 = 2.0 ** -24
LAM = 4.0
BF16_ULPS = 1.0
DGELU_ABS = 2e-6
LOSS_REL = 1e-5
LABEL_TOL = 4e-6  # absolute error of a normalised fp32 label (test_gpu_forward_kernels.py)
REPRO_TOL = 2e-4
TC_STEP = U24 / 8  # per row of a tensor-core weight gradient: one 2^-23 truncation of the fp32 accumulator per 16-deep k-step
CONTROL = 100.0


@pytest.fixture(scope="module")
def lib():
    assert torch.cuda.is_available()
    from smb_vision_b200 import load

    lib = load()
    assert lib.smbv_device_ok() == 0, lib.smbv_last_error()
    return lib


# =====================================================================================================================
# helpers (same meaning as in the kernel-level parity files)
# =====================================================================================================================
def bits(t):
    return t.view({torch.float32: torch.int32, torch.bfloat16: torch.int16, torch.int32: torch.int32}[t.dtype])


def same_bits(a, b):
    return a.shape == b.shape and torch.equal(bits(a.contiguous()), bits(b.contiguous()))


def report(name, worst, bound, ctrl=None):
    print(f"{name}: {worst:.3g} (bound {bound:.3g})" + ("" if ctrl is None else f"; negative control {ctrl:.3g} x bound"))


def ulp_bf16(ref):
    """one bf16 ulp (8 significant bits) of each element of a float64 tensor; 0 at ref == 0."""
    return torch.exp2(torch.floor(torch.log2(ref.abs())) - 7)


def max_ratio(err, den):
    return (err / den.clamp_min(1e-300)).max().item()


def acc(n):
    return LAM * math.sqrt(n) * U24


def d64(t):
    return t.double()


def mm_terms(a, w):
    """fp64 a @ w^T and sum_k |a_k w_k| for a [..., K], w [N, K]."""
    a, w = d64(a), d64(w)
    return a @ w.t(), a.abs() @ w.abs().t()


def other(t):
    """the same tensor with its samples rotated (B > 1) or, for one sample, its rows rotated by one: the 'wrong sample'
    operand of the negative controls."""
    return t.roll(1, 0) if t.shape[0] > 1 else t.roll(1, 1)


def gelu_prime64(x):
    x = d64(x)
    return 0.5 * (1 + torch.erf(x / math.sqrt(2))) + x * torch.exp(-0.5 * x * x) / math.sqrt(2 * math.pi)


def ln_stats64(x):
    x = d64(x)
    m = x.mean(-1)
    return m, (x.var(-1, unbiased=False) + 0.0).clamp_min(0)


def ln_fwd64(x, m, r, gamma, beta):
    """LayerNorm of x with the given (saved) statistics, fp64, and its rounding term."""
    x, m, r = d64(x), d64(m).reshape(x.shape[:-1])[..., None], d64(r).reshape(x.shape[:-1])[..., None]
    y = (x - m) * r * d64(gamma) + d64(beta)
    term = 4 * U24 * ((x.abs() + m.abs()) * r * d64(gamma).abs() + d64(beta).abs())
    return y, term


def ln_bwd64(dy, x, m, r, gamma):
    """-> (dx, element term, xhat) of LayerNorm backward from the saved statistics (the operands the kernel reads)."""
    x = d64(x)
    m, r = d64(m).reshape(x.shape[:-1])[..., None], d64(r).reshape(x.shape[:-1])[..., None]
    xh = (x - m) * r
    g = d64(dy) * d64(gamma)
    mg, mgx = g.mean(-1, keepdim=True), (g * xh).mean(-1, keepdim=True)
    dx = r * (g - mg - xh * mgx)
    term = r * (g.abs() + g.abs().mean(-1, keepdim=True) + xh.abs() * (g * xh).abs().mean(-1, keepdim=True))
    return dx, term, xh


def patchify64(vol):
    """im2col rows of the bf16-rounded volume (what the patch embedding reads): fp64 [B, N, 4096]."""
    cfg = types.SimpleNamespace(tubelet_size=16, patch_size=16)
    return vo.patchify(vol.bfloat16().double()[:, :, None], cfg)


def rows(t, idx):
    """t [B, N, ...] -> [B, K, ...] rows idx[b] of each sample."""
    return torch.stack([t[b, idx[b].long()] for b in range(t.shape[0])])


class Results:
    """stage -> (worst / bound, control / bound); printed and asserted at the end of a test."""

    def __init__(self, name):
        self.name, self.res, self.ctrl = name, {}, {}

    def check(self, stage, got, ref, bound, bad=None):
        got = d64(got)
        assert torch.isfinite(got).all(), stage
        r = max_ratio((got - ref).abs(), bound)
        self.res[stage] = max(self.res.get(stage, 0.0), r)
        if bad is not None:
            c = max_ratio((got - bad).abs(), bound)
            self.ctrl[stage] = min(self.ctrl.get(stage, float("inf")), c)
        return r

    def exact(self, stage, ok):
        self.res[stage] = max(self.res.get(stage, 0.0), 0.0 if ok else float("inf"))

    def finish(self):
        for k, v in self.res.items():
            report(f"{self.name}: {k}", v, 1.0, self.ctrl.get(k))
        bad = {k: v for k, v in self.res.items() if not v <= 1.0}
        weak = {k: v for k, v in self.ctrl.items() if not v >= CONTROL}
        assert not bad, bad
        assert not weak, weak


class Expect:
    """fp64 expected arena contributions: name -> (sum, sum of |terms|, number of terms)."""

    def __init__(self):
        self.ref, self.l1, self.n, self.tc = {}, {}, {}, {}

    def add(self, key, ref, l1, n, tc=0):
        if key in self.ref:
            self.ref[key] = self.ref[key] + ref
            self.l1[key] = self.l1[key] + l1
            self.n[key] += n
            self.tc[key] += tc
        else:
            self.ref[key], self.l1[key], self.n[key], self.tc[key] = ref, l1, n, tc

    def wgrad(self, key, dy, x):
        """dW += dy^T x over the rows of dy [M, N], x [M, K]."""
        dy, x = d64(dy).reshape(-1, dy.shape[-1]), d64(x).reshape(-1, x.shape[-1])
        self.add(key, dy.t() @ x, dy.abs().t() @ x.abs(), dy.shape[0], dy.shape[0])

    def colsum(self, key, dy):
        dy = d64(dy).reshape(-1, dy.shape[-1])
        self.add(key, dy.sum(0), dy.abs().sum(0), dy.shape[0])

    def bound(self, key):
        return (acc(self.n[key]) + TC_STEP * self.tc[key]) * self.l1[key] + 2 * U24 * self.ref[key].abs()


# =====================================================================================================================
# the spy
# =====================================================================================================================
WATCH = ("layernorm_bwd", "linear_dgrad", "flash_attn_bwd", "attn_small_bwd", "qkv_dgrad", "gather_patches", "normpix_loss",
         "cast_bf16", "token_sum", "patch_embed_select_fwd")


class Spy:
    """Records what the training step hands to the kernels without changing a bit of it: `log` = every call of the
    WATCH ops (name, args, kwargs, result; for the LayerNorm backward its dres before and after), `fwd` / `bwd` = every
    block_forward_train / block_backward with its inputs, saves and outputs and the range of `log` entries it made."""

    def __init__(self, monkeypatch):
        from smb_vision_b200 import ops, training

        self.log, self.fwd, self.bwd = [], [], []
        for name in WATCH:
            monkeypatch.setattr(ops, name, self._wrap(name, getattr(ops, name)))
        real_f, real_b = training.block_forward_train, training.block_backward

        def fwd(X, p, rope=None):
            out, s = real_f(X, p, rope)
            self.fwd.append(dict(s=s, p=p, out=out))
            return out, s

        def bwd(dX, dXb, s, p, arena, prefix, names=None, rope=None, sq=None, extra=None):
            rec = dict(dX_before=dX.clone(), dXb=dXb.clone(), s=s, p=p, prefix=prefix, lo=len(self.log))
            res = real_b(dX, dXb, s, p, arena, prefix, names, rope, sq, extra)
            rec.update(dX_after=dX.clone(), ret=res, hi=len(self.log))
            self.bwd.append(rec)
            return res

        monkeypatch.setattr(training, "block_forward_train", fwd)
        monkeypatch.setattr(training, "block_backward", bwd)

    def _wrap(self, name, real):
        def fn(*args, **kw):
            rec = dict(name=name, args=args, kw=kw)
            if name == "layernorm_bwd":
                rec["dres_before"] = args[5].clone()
            res = real(*args, **kw)
            if name == "layernorm_bwd":
                rec["dres_after"] = args[5].clone()
            if name == "linear_dgrad" and res.dtype == torch.float32:  # the e2d dgrad's dX: updated in place later
                rec["snap"] = res.clone()
            if name == "flash_attn_bwd":
                res = tuple(res)
                rec["d"] = [t.clone() for t in res]
            rec["out"] = res
            self.log.append(rec)
            return res
        return fn

    def calls(self, name, lo=0, hi=None):
        return [c for c in self.log[lo:hi] if c["name"] == name]


# =====================================================================================================================
# models and inputs
# =====================================================================================================================
BASE = dict(hidden_size=768, num_attention_heads=12, intermediate_size=3072, decoder_hidden_size=384,
            decoder_num_attention_heads=6, decoder_intermediate_size=1536, num_hidden_layers=2, decoder_num_hidden_layers=1,
            patch_size=16, tubelet_size=16, num_channels=1)
CASES = {  # name -> (config, batch, mim_style)
    "tiny-mae": (dict(vo.TINY), 2, "mae"),
    "small64-mae": (dict(ge.SMALL64), 2, "mae"),
    "small64-simmim": (dict(ge.SMALL64), 2, "simmim"),
    "small64-final-ln": (dict(ge.SMALL64, use_mean_pooling=False), 2, "mae"),
    "base-160x160x96-B3": (dict(BASE, image_size=160, num_frames=96), 3, "mae"),
    "base-512x512x320-B1": (dict(BASE, image_size=512, num_frames=320), 1, "mae"),
}


def make_mim(cfgd, B, style, seed=1234):
    from smb_vision_b200.data import MaskGenerator
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining

    cfg = vo.OracleConfig(**cfgd)
    sd = vo.synthetic_state_dict(cfg, seed)
    if style == "simmim":
        sd["videomae.embeddings.mask_token"] = 0.3 * torch.randn(1, 1, cfg.hidden_size, generator=torch.Generator().manual_seed(9))
    model = B200VideoMAEForPreTraining(ge.hf_config(cfgd), mim_style=style).to(DEV).train()
    model.load_state_dict(sd, strict=True)
    vol = model.videomae._volume(vo.synthetic_volume(cfg, B, 7).to(DEV))
    np.random.seed(B)
    mp = MaskGenerator(cfg.image_size, cfg.num_frames, 32, 16, 0.65).device_batch(B, DEV)
    return model, vol, mp


def make_cls(cfgd, B):
    from smb_vision_b200.modeling import B200VideoMAEForVideoClassification

    cfg = vo.OracleConfig(**cfgd)
    hc = ge.hf_config(cfgd)
    hc.num_labels, hc.additional_features_size, hc.problem_type = 3, 2, "single_label_classification"
    model = B200VideoMAEForVideoClassification(hc).to(DEV).train()
    sd = {k: v for k, v in vo.synthetic_state_dict(cfg, 1234).items() if k.startswith("videomae.")}
    gsd = torch.Generator().manual_seed(2)
    sd["classifier.weight"] = 0.05 * torch.randn(3, cfg.hidden_size + 2, generator=gsd)
    sd["classifier.bias"] = 0.02 * torch.randn(3, generator=gsd)
    if model.fc_norm is not None:
        sd["fc_norm.weight"] = 1 + 0.1 * torch.randn(cfg.hidden_size, generator=gsd)
        sd["fc_norm.bias"] = 0.1 * torch.randn(cfg.hidden_size, generator=gsd)
    model.load_state_dict(sd, strict=True)
    vol = model.videomae._volume(vo.synthetic_volume(cfg, B, 5).to(DEV))
    feats = torch.randn(B, 2, generator=gsd).to(DEV)
    labels = torch.arange(B, dtype=torch.long).remainder(3).to(DEV)
    return model, vol, feats, labels


def nan_padded_arena(model):
    """GradArena whose alignment padding (elements no parameter or pad entry covers) holds NaN; -> (arena, padding mask)."""
    from smb_vision_b200.training import GradArena

    a = GradArena(model, DEV)
    covered = torch.zeros(a.flat.numel(), dtype=torch.bool, device=DEV)
    for o, n in a.offsets.values():
        covered[o:o + n] = True
    pad = ~covered
    a.flat[pad] = float("nan")
    return a, pad


# =====================================================================================================================
# stage checks shared by the MIM and the classification step
# =====================================================================================================================
def check_block_forward(R, tag, rec, other_rec):
    s, p, out = rec["s"], rec["p"], rec["out"]
    d = s.x_in.shape[-1]
    for st, x, m, r in (("LN1 stats", s.x_in, s.m1, s.r1), ("LN2 stats", s.x_mid, s.m2, s.r2)):
        m64, v64 = ln_stats64(x)
        r64 = (v64 + p.eps).rsqrt().reshape(-1)
        m64 = m64.reshape(-1)
        R.check(f"{tag} {st} (mean)", m, m64, acc(d) * d64(x).abs().mean(-1).reshape(-1))
        R.check(f"{tag} {st} (rstd)", r, r64, (acc(d) + 4 * U24) * r64)
    ref, T = mm_terms(s.a, p.wo)
    ref = ref + d64(p.bo) + d64(s.x_in)
    bnd = acc(d) * T + 2 * U24 * (ref.abs() + d64(p.bo).abs() + d64(s.x_in).abs())
    R.check(f"{tag} x_mid = x_in + a Wo^T + bo", s.x_mid, ref, bnd, d64(other(s.a)) @ d64(p.wo).t() + d64(p.bo) + d64(s.x_in))
    K = p.w2.shape[1]
    ref, T = mm_terms(s.f, p.w2)
    ref = ref + d64(p.b2) + d64(s.x_mid)
    bnd = acc(K) * T + 2 * U24 * (ref.abs() + d64(p.b2).abs() + d64(s.x_mid).abs())
    R.check(f"{tag} x_out = x_mid + f W2^T + b2", out, ref, bnd, d64(other(s.f)) @ d64(p.w2).t() + d64(p.b2) + d64(s.x_mid))


def check_block_backward(R, E, spy, tag, rec, names, pre_other=None):
    """one block_backward call: every stage from the operands it read; its parameter contributions go to E."""
    s, p = rec["s"], rec["p"]
    B, n, d = rec["dX_before"].shape
    lo, hi = rec["lo"], rec["hi"]
    dg = spy.calls("linear_dgrad", lo, hi)
    lnb = spy.calls("layernorm_bwd", lo, hi)
    assert len(dg) == (3 if p.hd == 64 else 4) and len(lnb) == 2, (len(dg), len(lnb))  # small heads: + the QKV dgrad
    dXb = rec["dXb"]
    R.exact(f"{tag} dXb = bf16(dX)", same_bits(dXb, rec["dX_before"].bfloat16()))
    # dpre = (dXb W2) * gelu'(pre)
    dpre = dg[0]["out"]
    assert dg[0]["kw"].get("aux") is not None
    acc_ref, T = d64(dXb) @ d64(p.w2), d64(dXb).abs() @ d64(p.w2).abs()
    gp = gelu_prime64(s.pre)
    ref = acc_ref * gp
    bnd = BF16_ULPS * ulp_bf16(ref) + acc(p.w2.shape[0]) * T * gp.abs() + DGELU_ABS * T
    R.check("block dpre = (dXb W2) gelu'(pre)", dpre, ref, bnd, None if pre_other is None else acc_ref * gelu_prime64(pre_other))
    # dh2 = dpre W1
    dh2 = dg[1]["out"]
    ref, T = d64(dpre) @ d64(p.w1), d64(dpre).abs() @ d64(p.w1).abs()
    R.check("block dh2 = dpre W1", dh2, ref, BF16_ULPS * ulp_bf16(ref) + acc(p.w1.shape[0]) * T, d64(other(dpre)) @ d64(p.w1))
    # LN2 backward added into dX
    c2 = lnb[0]
    R.exact("block LN2 backward reads dh2, x_mid and adds into dX", c2["args"][0] is dh2 and same_bits(c2["dres_before"], rec["dX_before"]))
    dx, term, xh2 = ln_bwd64(dh2, s.x_mid, s.m2, s.r2, p.g2)
    ref = dx + d64(rec["dX_before"])
    bnd = acc(d) * term + 2 * U24 * (d64(rec["dX_before"]).abs() + ref.abs())
    R.check("block LN2 backward (+ residual)", c2["dres_after"], ref, bnd, dx)
    dXb_mid = c2["out"]
    R.exact("block LN2 bf16 copy", same_bits(dXb_mid, c2["dres_after"].bfloat16()))
    # dO = dXb_mid Wo
    dO = dg[2]["out"]
    ref, T = d64(dXb_mid) @ d64(p.wo), d64(dXb_mid).abs() @ d64(p.wo).abs()
    R.check("block dO = dXb Wo", dO, ref, BF16_ULPS * ulp_bf16(ref) + acc(d) * T, d64(other(dXb_mid)) @ d64(p.wo))
    # the attention backward reads dO and the block's saves; dQKV token-major [B, n, 3d]
    if p.hd == 64:
        (fa,) = spy.calls("flash_attn_bwd", lo, hi)
        a = fa["args"]
        R.exact("block attention backward operands", all(a[j].data_ptr() == s.qkv[j].data_ptr() for j in range(3)) and a[3] is s.a
                and a[4] is dO and a[5] is s.lse)
        dqkv = torch.stack(fa["d"]).permute(1, 3, 0, 2, 4).reshape(B, n, 3 * d)
        dgr = spy.calls("qkv_dgrad", lo, hi)
        R.exact("block qkv_dgrad per sample", sorted(c["kw"]["batch_index"] for c in dgr) == list(range(B)))
    else:
        (sa,) = spy.calls("attn_small_bwd", lo, hi)
        a = sa["args"]
        R.exact("block attention backward operands", a[0] is s.qkv and a[1] is s.a and a[2] is dO and a[3] is s.lse)
        dqkv = sa["out"]
    # dh1 = dQKV Wqkv, then LN1 backward
    c1 = lnb[1]
    dh1 = c1["args"][0]
    ref, T = d64(dqkv) @ d64(p.wqkv), d64(dqkv).abs() @ d64(p.wqkv).abs()
    nok = dqkv.clone()
    nok[..., d:2 * d] = 0
    R.check("block dh1 = dQKV Wqkv", dh1, ref, BF16_ULPS * ulp_bf16(ref) + acc(3 * d) * T, d64(nok) @ d64(p.wqkv))
    R.exact("block LN1 backward adds into the LN2 result", same_bits(c1["dres_before"], c2["dres_after"]))
    dx, term, xh1 = ln_bwd64(dh1, s.x_in, s.m1, s.r1, p.g1)
    ref = dx + d64(c2["dres_after"])
    bnd = acc(d) * term + 2 * U24 * (d64(c2["dres_after"]).abs() + ref.abs())
    R.check("block LN1 backward (+ residual)", rec["dX_after"], ref, bnd)
    R.exact("block returns bf16(dX)", same_bits(rec["ret"], rec["dX_after"].bfloat16()))
    # parameter contributions, from the stage operands
    pre = rec["prefix"]
    E.wgrad(names["w2"], dXb, s.f)
    E.colsum(names["b2"], dXb)
    E.wgrad(names["w1"], dpre, s.h2)
    E.colsum(names["b1"], dpre)
    E.colsum(names["ln2w"], d64(dh2) * xh2)
    E.colsum(names["ln2b"], dh2)
    E.wgrad(names["wo"], dXb_mid, s.a)
    E.colsum(names["bo"], dXb_mid)
    E.wgrad(pre + "qkv", dqkv, s.h1)
    E.colsum(names["qkv_bias"], dqkv[..., :d])
    E.colsum(pre + "attention.attention.v_bias", dqkv[..., 2 * d:])
    E.colsum(names["ln1w"], d64(dh1) * xh1)
    E.colsum(names["ln1b"], dh1)
    return dqkv


def check_arena(R, E, arena, pad, bad=None):
    """every parameter view against its fp64 expectation; K pad slots exactly 0; the alignment padding still NaN.
    `bad`: {stage name: (key, wrong fp64 expectation)} negative controls."""
    from smb_vision_b200.training import PAD_SUFFIX

    seen = set()
    for name, (o, n) in arena.offsets.items():
        if name.endswith(PAD_SUFFIX):
            R.exact("arena K-bias pad slot exactly 0", bool((bits(arena.flat[o:o + n]) == 0).all()))
            continue
        if name.endswith(("query.weight", "key.weight", "value.weight")):
            pre = name[:name.index("attention.attention.")]
            key = pre + "qkv"
            if key in seen:
                continue
            got = arena.fused_qkv(pre)
        else:
            key, got = name, arena.views[name]
        seen.add(key)
        assert key in E.ref, f"no stage contribution recorded for {key}"
        ref = E.ref[key].reshape(got.shape)
        bnd = E.bound(key).reshape(got.shape)
        for st, (k2, wrong) in (bad or {}).items():
            if k2 == key:
                R.check(st, got, ref, bnd, wrong.reshape(got.shape))
        R.check("arena: every parameter = sum of its stage contributions", got, ref, bnd)
    R.exact("arena alignment padding still NaN", bool(torch.isnan(arena.flat[pad]).all()))


def check_patch_embedding_grads(R, E, vol, dX_enc, idx):
    """patch-embedding bias and weight contributions: rows idx of the encoder-input gradient against the patchify of the
    volume taken here."""
    P = rows(patchify64(vol), idx)
    dXr = rows(dX_enc, idx) if idx.shape[1] != dX_enc.shape[1] else dX_enc
    E.colsum("videomae.embeddings.patch_embeddings.projection.bias", dXr)
    E.wgrad("videomae.embeddings.patch_embeddings.projection.weight", dXr.bfloat16(), P)
    return P


# =====================================================================================================================
# the MIM step
# =====================================================================================================================
@pytest.mark.parametrize("case", list(CASES))
def test_mim_step_stages(lib, monkeypatch, case):
    """mim_forward_train + mim_backward on one config: every forward and backward junction, arena closure,
    accumulation and bit-repeatable forward (module docstring)."""
    from smb_vision_b200.training import mim_backward, mim_forward_train, videomae_block_names

    cfgd, B, style = CASES[case]
    simmim = style == "simmim"
    model, vol, mp = make_mim(cfgd, B, style)
    fine, vis, msk, slot, n_vis, n_mask = mp
    vm, c = model.videomae, model.config
    L, Ld = c.num_hidden_layers, c.decoder_num_hidden_layers
    N, d, dd = vm.num_patches, c.hidden_size, c.decoder_hidden_size
    pe, pd = vm.packed(), model.packed()
    visk, mskk = vis[:, :n_vis], msk[:, :n_mask]
    R = Results(f"MIM {case} B={B} n_vis={n_vis}")
    E = Expect()
    arena, pad = nan_padded_arena(model)
    spy = Spy(monkeypatch)
    with torch.no_grad():
        loss, logits, dlogits, S = mim_forward_train(model, vol, mp)
        n_fwd_log = len(spy.log)
        mim_backward(model, S, dlogits, arena)
    torch.cuda.synchronize()
    assert len(spy.fwd) == L + Ld and len(spy.bwd) == L + Ld

    # ---- F1: patch embedding ----
    P = patchify64(vol)  # [B, N, 4096]
    W16, bpe, pos = pe["wpe16"], pe["bpe"], vm.pos_table(d, DEV)
    X0 = spy.fwd[0]["s"].x_in
    emb, T = mm_terms(P, W16)
    emb = emb + d64(bpe)
    if simmim:
        (call,) = spy.calls("patch_embed_select_fwd", 0, n_fwd_log)
        fm = fine.bool()[..., None]
        mt = d64(pe["mask_token"])
        ref = torch.where(fm, mt, emb) + d64(pos)
        bnd = torch.where(fm, 0 * T, acc(4096) * T) + 2 * U24 * (ref.abs() + emb.abs() + mt.abs() + d64(pos).abs())
        R.check("F1 SimMIM blend: where(msk, mask_token, P W^T + b) + PE", X0, ref, bnd,
                torch.where(other(fm), mt, emb) + d64(pos))
    else:
        gp = spy.calls("gather_patches", 0, n_fwd_log)
        assert len(gp) == 1
        R.exact("F1 saved patches = patchify(vol)[vis]", same_bits(S.enc[0].view(B, n_vis, -1), rows(P, visk).bfloat16()))
        ref = rows(emb, visk) + d64(pos)[visk.long()]
        bnd = acc(4096) * rows(T, visk) + 2 * U24 * (ref.abs() + rows(emb, visk).abs() + d64(pos)[visk.long()].abs())
        bad_idx = other(visk)
        R.check("F1 X[b, j] = P[vis[b, j]] W^T + b + PE[vis[b, j]]", X0, ref, bnd,
                rows(emb, bad_idx) + d64(pos)[bad_idx.long()])
    # ---- F2: block junctions ----
    for i, rec in enumerate(spy.fwd):
        check_block_forward(R, "F2 block", rec, None)
        if i + 1 < len(spy.fwd) and i + 1 != L:
            R.exact("F2 block chaining", spy.fwd[i + 1]["s"].x_in is rec["out"])
    X = spy.fwd[L - 1]["out"]
    # ---- F3: final encoder LayerNorm / bf16(X) ----
    if vm.layernorm is not None:
        eps = c.layer_norm_eps
        m64, v64 = ln_stats64(X)
        r64 = (v64 + eps).rsqrt()
        R.check("F3 final LN stats (mean)", S.mE, m64.reshape(-1), acc(d) * d64(X).abs().mean(-1).reshape(-1))
        R.check("F3 final LN stats (rstd)", S.rE, r64.reshape(-1), (acc(d) + 4 * U24) * r64.reshape(-1))
        ref, term = ln_fwd64(X, S.mE, S.rE, vm.layernorm.weight, vm.layernorm.bias)
        bad, _ = ln_fwd64(X, other(S.mE.view(B, -1)), other(S.rE.view(B, -1)), vm.layernorm.weight, vm.layernorm.bias)
        R.check("F3 final encoder LayerNorm", S.xb, ref, BF16_ULPS * ulp_bf16(ref) + term, bad)
    else:
        R.exact("F3 S.xb = bf16(X)", same_bits(S.xb, X.bfloat16()))
    # ---- F4: decoder input ----
    Xd0 = spy.fwd[L]["s"].x_in
    pos_d = d64(vm.pos_table(dd, DEV))
    z, T = mm_terms(S.xb, pd["we2d"])
    if simmim:
        ref = z + pos_d
        R.check("F4 decoder input (SimMIM: all N rows, natural order)", Xd0, ref, acc(d) * T + 2 * U24 * (ref.abs() + pos_d.abs()),
                other(z) + pos_d)
    else:
        ref = z + pos_d[visk.long()]
        bnd = acc(d) * T + 2 * U24 * (ref.abs() + pos_d[visk.long()].abs())
        R.check("F4 decoder input, visible rows: xb We2d^T + PE_d[vis]", Xd0[:, :n_vis], ref, bnd, z + pos_d[other(visk).long()])
        mt = d64(pd["mask_token"]).reshape(-1)
        ref = mt + pos_d[mskk.long()]
        R.check("F4 decoder input, masked rows: mask_token + PE_d[msk]", Xd0[:, n_vis:], ref, 2 * U24 * (ref.abs() + mt.abs()),
                mt + pos_d[other(mskk).long()])
    # ---- F5: head LayerNorm per sample, logits, loss ----
    if simmim:
        R.exact("F5 SimMIM head rows = gather(xd, msk)", same_bits(S.g, rows(S.xd, mskk)))
        hrows = S.g
    else:
        hrows = S.xd[:, n_vis:]
    m64, v64 = ln_stats64(hrows)
    r64 = (v64 + 1e-5).rsqrt()
    R.check("F5 head LN stats (mean)", S.mN, m64, acc(dd) * d64(hrows).abs().mean(-1), other(m64))
    R.check("F5 head LN stats (rstd)", S.rN, r64, (acc(dd) + 4 * U24) * r64, other(r64))
    ref, term = ln_fwd64(hrows, S.mN, S.rN, pd["gn"], pd["bn"])
    bad, _ = ln_fwd64(hrows, other(S.mN), other(S.rN), pd["gn"], pd["bn"])
    R.check("F5 head LayerNorm with each sample's statistics", S.hN, ref, BF16_ULPS * ulp_bf16(ref) + term, bad)
    ref, T = mm_terms(S.hN, pd["wh"])
    ref = ref + d64(pd["bh"])
    R.check("F5 logits = hN Wh^T + bh", logits, ref, BF16_ULPS * ulp_bf16(ref) + acc(dd) * T + 2 * U24 * d64(pd["bh"]).abs())
    (npl,) = spy.calls("normpix_loss", 0, n_fwd_log)
    R.exact("F5 loss reads msk and the logits", npl["args"][1] is msk and npl["args"][3] is logits)

    def normpix64(idx):
        X_ = rows(vo.patchify(d64(vol)[:, :, None], types.SimpleNamespace(tubelet_size=16, patch_size=16)), idx)  # fp32 volume
        lab = (X_ - X_.mean(-1, keepdim=True)) / (X_.var(-1, keepdim=True, unbiased=True).sqrt() + 1e-6)
        dlt = d64(logits) - lab
        return (dlt * dlt).mean(), 2 * dlt / dlt.numel(), lab

    assert model.loss_kind == 0
    lref, dl_ref, lab = normpix64(mskk)
    _, dl_bad, _ = normpix64(mskk.flip(1))  # labels paired with the wrong logits rows
    # the loss value is a mean over every masked element: no row-assignment error moves it measurably, so its negative
    # control is the per-element dlogits below
    R.check("F5 loss value", loss.reshape(1), lref.reshape(1), LOSS_REL * lref.abs().reshape(1))
    R.check("F5 dlogits = 2 (logits - labels at msk[b]) / count", dlogits, dl_ref,
            BF16_ULPS * ulp_bf16(dl_ref) + 2 / dl_ref.numel() * LABEL_TOL * (1 + lab.abs()), dl_bad)

    # ---- B1: head ----
    bw = spy.calls("linear_dgrad", n_fwd_log)
    dhN = bw[0]["out"]
    R.exact("B1 head dgrad reads dlogits", bw[0]["args"][0] is dlogits)
    ref, T = d64(dlogits) @ d64(pd["wh"]), d64(dlogits).abs() @ d64(pd["wh"]).abs()
    R.check("B1 dhN = dlogits Wh", dhN, ref, BF16_ULPS * ulp_bf16(ref) + acc(pd["wh"].shape[0]) * T, d64(other(dlogits)) @ d64(pd["wh"]))
    E.wgrad("decoder.head.weight", dlogits, S.hN)
    E.colsum("decoder.head.bias", dlogits)
    # ---- B2: decoder norm backward ----
    dec = [r for r in spy.bwd if r["prefix"].startswith("decoder.")]
    enc = [r for r in spy.bwd if r["prefix"].startswith("videomae.")]
    dXd0 = dec[0]["dX_before"]
    dx, term, xh = ln_bwd64(dhN, hrows, S.mN, S.rN, pd["gn"])
    bad, _, _ = ln_bwd64(dhN, hrows, other(S.mN), other(S.rN), pd["gn"])
    bnd = acc(dd) * term + 2 * U24 * dx.abs()
    if simmim:
        R.check("B2 decoder norm backward, scattered to msk", rows(dXd0, mskk), dx, bnd, bad)
        keep = torch.ones(B, N, dtype=torch.bool, device=DEV)
        keep.scatter_(1, mskk.long(), False)
        R.exact("B2 rows outside msk exactly 0", bool((bits(dXd0[keep]) == 0).all()))
    else:
        R.check("B2 decoder norm backward, rows n_vis:", dXd0[:, n_vis:], dx, bnd, bad)
        R.exact("B2 visible rows exactly 0", bool((bits(dXd0[:, :n_vis]) == 0).all()))
    E.colsum("decoder.norm.weight", d64(dhN) * xh)
    E.colsum("decoder.norm.bias", dhN)
    # ---- B3: every block ----
    fwd_of = {id(r["s"]): i for i, r in enumerate(spy.fwd)}
    dqkv_last = None
    for rec in spy.bwd:
        i = fwd_of[id(rec["s"])]
        pre_other = spy.fwd[(i + 1) % L]["s"].pre if i < L and L > 1 else None
        dq = check_block_backward(R, E, spy, "B3", rec, videomae_block_names(rec["prefix"]), pre_other)
        if rec["prefix"] == "videomae.encoder.layer.0.":
            dqkv_last = (rec, dq)
    for a_, b_ in zip(spy.bwd[:-1], spy.bwd[1:]):
        if a_["prefix"].startswith("decoder.") == b_["prefix"].startswith("decoder."):
            R.exact("B3 block chaining", same_bits(b_["dX_before"], a_["dX_after"]) and same_bits(b_["dXb"], a_["ret"]))
    # ---- B4: decoder-input split ----
    dXdF = dec[-1]["dX_after"]  # [B, N, dd]
    n_enc = N if simmim else n_vis
    dZb_ref = dXdF[:, :n_enc].bfloat16()
    e2d = [cl for cl in bw if cl["args"][1].data_ptr() == pd["we2d"].data_ptr()]
    assert len(e2d) == 1
    dZb = e2d[0]["args"][0]
    R.exact("B4 dZb = bf16(dXd[:, :n_enc])", same_bits(dZb, dZb_ref))
    dXe = e2d[0]["snap"]
    ref, T = d64(dZb) @ d64(pd["we2d"]), d64(dZb).abs() @ d64(pd["we2d"]).abs()
    R.check("B4 dX = dZb We2d (fp32)", dXe, ref, acc(dd) * T + 2 * U24 * ref.abs(), d64(other(dZb)) @ d64(pd["we2d"]))
    E.wgrad("encoder_to_decoder.weight", dZb, S.xb)
    bad_arena = {}
    if simmim:
        E.add("mask_token", torch.zeros(dd, dtype=torch.float64, device=DEV), torch.zeros(dd, dtype=torch.float64, device=DEV), 1)
    else:
        E.colsum("mask_token", dXdF[:, n_vis:])
        bad_arena["B4 mask-token gradient = sum over rows n_vis:"] = ("mask_token", d64(dXdF[:, :n_vis]).reshape(-1, dd).sum(0))
    # ---- B5: final encoder LayerNorm backward / SimMIM blend ----
    dX_top = enc[0]["dX_before"]
    if vm.layernorm is not None:
        after = [cl for cl in spy.log[n_fwd_log:enc[0]["lo"]] if cl["name"] == "layernorm_bwd" and cl["args"][1] is S.x_pre]
        assert len(after) == 1
        fl = after[0]
        R.exact("B5 final LN backward reads bf16(dX)", same_bits(fl["args"][0], dXe.bfloat16()))
        dx, term, xh = ln_bwd64(fl["args"][0], S.x_pre, S.mE, S.rE, vm.layernorm.weight)
        bad, _, _ = ln_bwd64(fl["args"][0], S.x_pre, other(S.mE.view(B, -1)), other(S.rE.view(B, -1)), vm.layernorm.weight)
        R.check("B5 final encoder LayerNorm backward", fl["dres_after"], dx, acc(d) * term + 2 * U24 * dx.abs(), bad)
        R.exact("B5 encoder backward starts from it", same_bits(dX_top, fl["dres_after"]) and same_bits(enc[0]["dXb"], fl["out"]))
        E.colsum("videomae.layernorm.weight", d64(fl["args"][0]) * xh)
        E.colsum("videomae.layernorm.bias", fl["args"][0])
    else:
        R.exact("B5 encoder backward starts from dX", same_bits(dX_top, dXe))
    dXE = enc[-1]["dX_after"]
    if simmim:
        E.colsum("videomae.embeddings.mask_token", rows(dXE, mskk))
        bad_arena["B5 SimMIM encoder mask token = sum over msk rows"] = (
            "videomae.embeddings.mask_token", d64(rows(dXE, visk)).reshape(-1, d).sum(0))
        P_used = check_patch_embedding_grads(R, E, vol, dXE, visk)
        bad_w = d64(rows(dXE, other(visk)).bfloat16()).reshape(-1, d).t() @ d64(rows(P, visk)).reshape(-1, 4096)
    else:
        P_used = check_patch_embedding_grads(R, E, vol, dXE, visk)
        bad_w = d64(dXE.bfloat16()).reshape(-1, d).t() @ d64(rows(P, other(visk))).reshape(-1, 4096)
    bad_arena["B6 patch-embedding weight from the visible rows' patches"] = ("videomae.embeddings.patch_embeddings.projection.weight", bad_w)
    if B > 1 and dqkv_last is not None:
        rec, dq = dqkv_last
        pre = rec["prefix"]
        E_b = d64(dq[-1]).t() @ d64(rec["s"].h1[-1])
        bad_arena["B3 fused QKV weight gradient over every sample"] = (pre + "qkv", E.ref[pre + "qkv"] - E_b)
    # ---- arena closure, accumulation ----
    check_arena(R, E, arena, pad, bad_arena)
    first = arena.flat.clone()
    with torch.no_grad():
        mim_backward(model, S, dlogits, arena)
    torch.cuda.synchronize()
    worst = 0.0
    for name, v in arena.views.items():
        o, n = arena.offsets[name]
        f = first[o:o + n].double()
        nrm = torch.linalg.norm(2 * f).item()
        e = torch.linalg.norm(v.reshape(-1).double() - 2 * f).item()
        worst = max(worst, e / nrm if nrm > 0 else (0.0 if e == 0 else float("inf")))
    R.res["accumulation: second backward = 2x first (Frobenius-rel / REPRO_TOL)"] = worst / REPRO_TOL
    # ---- repeatability of the forward ----
    saved = [(r["s"], r["out"]) for r in spy.fwd]
    with torch.no_grad():
        loss2, logits2, dlogits2, S2 = mim_forward_train(model, vol, mp)
    ok = same_bits(loss2.reshape(1), loss.reshape(1)) and same_bits(logits2, logits) and same_bits(dlogits2, dlogits)
    for (s1, o1), r2 in zip(saved, spy.fwd[len(saved):]):
        s2 = r2["s"]
        ok = ok and same_bits(o1, r2["out"]) and all(same_bits(getattr(s1, k), getattr(s2, k))
                                                     for k in ("h1", "a", "lse", "x_mid", "h2", "pre", "f"))
    R.exact("forward repeats bit for bit", ok)
    R.finish()


# =====================================================================================================================
# the classification step
# =====================================================================================================================
@pytest.mark.parametrize("pooling", ["mean", "cls-row"])
def test_cls_step_stages(lib, monkeypatch, pooling):
    """cls_forward_train + cls_backward on SMALL64, B = 2: the token sum or the final LayerNorm, the broadcast of dpooled
    to every row (mean pooling) or the seed on row 0 only (CLS row), every encoder block, the patch embedding, arena
    closure (the classifier / fc_norm gradients of the forward launch stay untouched by the backward)."""
    from smb_vision_b200.training import cls_backward, cls_forward_train, videomae_block_names

    cfgd = dict(ge.SMALL64, use_mean_pooling=pooling == "mean")
    B = 2
    model, vol, feats, labels = make_cls(cfgd, B)
    vm, c = model.videomae, model.config
    L, N, d = c.num_hidden_layers, vm.num_patches, c.hidden_size
    R = Results(f"classification {pooling} B={B}")
    E = Expect()
    arena, pad = nan_padded_arena(model)
    spy = Spy(monkeypatch)
    with torch.no_grad():
        loss, logits, dpooled, S = cls_forward_train(model, vol, feats, labels, arena)
        torch.cuda.synchronize()
        head = arena.flat[:arena.bucket_bounds[1]].clone()
        n_fwd_log = len(spy.log)
        cls_backward(model, S, dpooled, arena)
    torch.cuda.synchronize()
    P = patchify64(vol)
    pe = vm.packed()
    emb, T = mm_terms(P, pe["wpe16"])
    pos = d64(vm.pos_table(d, DEV))
    ref = emb + d64(pe["bpe"]) + pos
    R.check("F1 patch embedding (all tokens)", spy.fwd[0]["s"].x_in, ref, acc(4096) * T + 2 * U24 * (ref.abs() + emb.abs() + pos.abs()),
            other(emb) + d64(pe["bpe"]) + pos)
    for rec in spy.fwd:
        check_block_forward(R, "F2 block", rec, None)
    X = spy.fwd[-1]["out"]
    enc = spy.bwd
    if pooling == "mean":
        (ts,) = spy.calls("token_sum", 0, n_fwd_log)
        ref = d64(X).sum(1)
        R.check("F3 token sum", ts["out"], ref, acc(N) * d64(X).abs().sum(1) + 2 * U24 * ref.abs(), d64(X[:, 1:]).sum(1))
        R.exact("B7 broadcast: dpooled on every row", same_bits(enc[0]["dX_before"], dpooled[:, None].expand(B, N, d)))
    else:
        fl = [cl for cl in spy.log[n_fwd_log:enc[0]["lo"]] if cl["name"] == "layernorm_bwd"]
        assert len(fl) == 1
        fl = fl[0]
        seed = torch.zeros(B, N, d, dtype=torch.bfloat16, device=DEV)
        seed[:, 0] = dpooled.bfloat16()
        R.exact("B7 CLS row: only row 0 of dY is non-zero, = bf16(dpooled)", same_bits(fl["args"][0], seed))
        m64, v64 = ln_stats64(X)
        r64 = (v64 + c.layer_norm_eps).rsqrt()
        R.check("F3 final LN stats (rstd)", S.rE, r64.reshape(-1), (acc(d) + 4 * U24) * r64.reshape(-1))
        dx, term, xh = ln_bwd64(fl["args"][0], S.x_pre, S.mE, S.rE, vm.layernorm.weight)
        bad, _, _ = ln_bwd64(fl["args"][0], S.x_pre, other(S.mE.view(B, -1)), other(S.rE.view(B, -1)), vm.layernorm.weight)
        R.check("B7 final LayerNorm backward of the CLS row", fl["dres_after"], dx, acc(d) * term + 2 * U24 * dx.abs(), bad)
        R.exact("B7 encoder backward starts from it", same_bits(enc[0]["dX_before"], fl["dres_after"]))
        E.colsum("videomae.layernorm.weight", d64(fl["args"][0]) * xh)
        E.colsum("videomae.layernorm.bias", fl["args"][0])
    for i, rec in enumerate(enc):
        j = L - 1 - i
        check_block_backward(R, E, spy, "B3", rec, videomae_block_names(rec["prefix"]), spy.fwd[(j + 1) % L]["s"].pre)
    idx = torch.arange(N, dtype=torch.int32, device=DEV).repeat(B, 1)
    (gp,) = spy.calls("gather_patches", n_fwd_log)
    R.exact("B6 gathered patches = patchify(vol)", same_bits(gp["out"].view(B, N, -1), P.bfloat16()))
    check_patch_embedding_grads(R, E, vol, enc[-1]["dX_after"], idx)
    # classifier / fc_norm: computed and accumulated by the head kernel in the forward launch
    for k in ("classifier.weight", "classifier.bias", "fc_norm.weight", "fc_norm.bias"):
        if k in arena.views:
            E.add(k, d64(arena.views[k]), torch.zeros_like(d64(arena.views[k])), 1)
    R.exact("B7 head gradients untouched by cls_backward", same_bits(arena.flat[:arena.bucket_bounds[1]], head))
    check_arena(R, E, arena, pad)
    R.finish()


# =====================================================================================================================
# data-parallel buckets
# =====================================================================================================================
@pytest.mark.parametrize("stream", ["0", "1"])
@pytest.mark.parametrize("variant", ["mae", "simmim", "mae-final-ln", "cls-mean", "cls-row"])
def test_bucket_complete_when_hook_fires(lib, monkeypatch, variant, stream):
    """on_bucket(i) clones flat[bounds[i]:bounds[i+1]] on the stream it is called on; after the backward and a
    synchronize every clone must be bit-identical to the final arena slice (a parameter whose gradient lands after its
    bucket's hook would make the data-parallel reducer send a partial gradient).  Every bucket fires exactly once, in
    order.  SMALL64, B = 2, both SMBV_WGRAD_STREAM settings."""
    from smb_vision_b200.training import GradArena, cls_backward, cls_forward_train, mim_backward, mim_forward_train

    monkeypatch.setenv("SMBV_WGRAD_STREAM", stream)
    B = 2
    if variant.startswith("cls"):
        model, vol, feats, labels = make_cls(dict(ge.SMALL64, use_mean_pooling=variant == "cls-mean"), B)
    else:
        cfgd = dict(ge.SMALL64, use_mean_pooling=variant != "mae-final-ln")
        model, vol, mp = make_mim(cfgd, B, "simmim" if variant == "simmim" else "mae")
    arena = GradArena(model, DEV)
    bounds = arena.bucket_bounds
    clones, order = {}, []

    def hook(i):
        order.append(i)
        clones[i] = arena.flat[bounds[i]:bounds[i + 1]].clone()  # on the current (hook) stream

    with torch.no_grad():
        if variant.startswith("cls"):
            _, _, dpooled, S = cls_forward_train(model, vol, feats, labels, arena)
            cls_backward(model, S, dpooled, arena, hook)
        else:
            _, _, dlogits, S = mim_forward_train(model, vol, mp)
            mim_backward(model, S, dlogits, arena, hook)
    torch.cuda.synchronize()
    assert order == list(range(len(bounds) - 1)), order
    partial = [i for i in order if not same_bits(clones[i], arena.flat[bounds[i]:bounds[i + 1]])]
    print(f"buckets {variant} SMBV_WGRAD_STREAM={stream}: {len(order)} buckets, incomplete at their hook: {partial}")
    assert not partial
