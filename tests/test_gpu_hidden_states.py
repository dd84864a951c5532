"""GPU: `output_hidden_states` of the VideoMAE models (run with -m gpu on the B200 box).

Kernel level against fp64 / bit-exact references: the LayerNorm forward that also stores its input row (the hidden-state
snapshot), the LayerNorm backward with an extra fp32 addend (a hidden state's gradient joining the residual-stream gradient),
and the fused scale + add + bf16 re-cast.  Model level against the CPU oracle's states (tests/test_hidden_states_cpu.py pins
them to upstream transformers): forward values, bit-identities with truncated models and with the flag off, and parameter
gradients of losses that read the states, with and without the model loss.

Tolerances (SURVEY.md §8c): embeddings Frobenius-rel <= 2e-2, max-abs-rel <= 5e-2; gradients Frobenius-rel <= 2e-2
(grad_tol: 5e-2 for the layer-0 Q / K gradients of the small fixtures, see test_gpu_parity.grad_tol); gradients of runs
that differ only in run-to-run split-K summation order <= 2e-4 (test_gpu_parity.test_side_stream_gradients_match_single_stream).
"""
import numpy as np
import pytest
import torch

import __graft_entry__ as ge
from oracle import videomae_oracle as vo
from test_hidden_states_cpu import _mask, oracle_states

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PE_W = "videomae.embeddings.patch_embeddings.projection.weight"


@pytest.fixture(scope="module")
def ops():
    assert torch.cuda.is_available()
    from smb_vision_b200 import load, ops as _ops

    assert load().smbv_device_ok() == 0
    return _ops


def frob(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return (torch.linalg.norm(a - b) / torch.linalg.norm(b)).item()


def maxrel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).abs().max() / b.abs().max()).item()


def grad_tol(name, tol):
    qk = any(t in name for t in ("attention.query.weight", "attention.key.weight", "attention.q_bias"))
    return 5e-2 if qk else tol


def _cfgd(name, **kw):
    return dict(vo.TINY if name == "tiny" else ge.SMALL64, **kw)


def _encoder_sd(sd):
    return {k[len("videomae."):]: v for k, v in sd.items() if k.startswith("videomae.")}


def _encoder(cfgd, sd):
    from smb_vision_b200.modeling import B200VideoMAEModel

    m = B200VideoMAEModel(ge.hf_config(cfgd)).to(DEV)
    m.load_state_dict(_encoder_sd(sd), strict=True)
    return m


# ---------------------------------------------------------------------------- kernels
SHAPES = [(M, d) for d in (64, 128, 384, 768, 1024) for M in (1, 37, 1031)]


@pytest.mark.parametrize("M,d", SHAPES)
def test_layernorm_fwd_copy(ops, M, d):
    g = torch.Generator().manual_seed(M * d)
    x = (torch.randn(M, d, generator=g) * 3 + 1).to(DEV)
    w, b = torch.randn(d, generator=g).to(DEV), torch.randn(d, generator=g).to(DEV)
    y0, m0, r0 = ops.layernorm_fwd(x, w, b, 1e-6, save_stats=True)
    cp = torch.full_like(x, float("nan"))
    y1, m1, r1 = ops.layernorm_fwd(x, w, b, 1e-6, save_stats=True, x_copy=cp)
    assert torch.equal(cp, x)  # the snapshot is the input, bit for bit
    assert torch.equal(y0, y1) and torch.equal(m0, m1) and torch.equal(r0, r1)
    # the copy entry with a NULL copy pointer is the old kernel
    from smb_vision_b200._lib import call

    y2, m2, r2 = torch.empty_like(y0), torch.empty_like(m0), torch.empty_like(r0)
    call("smbv_layernorm_fwd_copy", ops._ptr(x), ops._ptr(w), ops._ptr(b), 1e-6, M, d, ops._ptr(y2), ops._ptr(m2), ops._ptr(r2),
         None, ops._stream())
    assert torch.equal(y0, y2) and torch.equal(m0, m2) and torch.equal(r0, r2)
    ref = torch.nn.functional.layer_norm(x.double(), (d,), w.double(), b.double(), 1e-6)
    assert frob(y1.float(), ref) <= 3e-3


@pytest.mark.parametrize("M,d", SHAPES)
@pytest.mark.parametrize("accumulate", [True, False])
def test_layernorm_bwd_add(ops, M, d, accumulate):
    g = torch.Generator().manual_seed(M + d)
    x = (torch.randn(M, d, generator=g) * 2 + 0.5).to(DEV)
    w, b = torch.randn(d, generator=g).to(DEV), torch.randn(d, generator=g).to(DEV)
    _, mean, rstd = ops.layernorm_fwd(x, w, b, 1e-6, save_stats=True)
    dy = torch.randn(M, d, generator=g).to(DEV).bfloat16()
    dres0 = torch.randn(M, d, generator=g).to(DEV)
    extra = torch.randn(M, d, generator=g).to(DEV)

    def run(ex):
        dres = dres0.clone()
        dg, db = torch.zeros(d, device=DEV), torch.zeros(d, device=DEV)
        dxb = ops.layernorm_bwd(dy, x, mean, rstd, w, dres, accumulate, dg, db, extra=ex)
        return dres, dxb, dg, db

    old = run(None)
    # the new entry with a NULL addend is the old kernel, bit for bit
    from smb_vision_b200._lib import call

    dres, dg, db = dres0.clone(), torch.zeros(d, device=DEV), torch.zeros(d, device=DEV)
    dxb = torch.empty_like(dy)
    call("smbv_layernorm_bwd_add", ops._ptr(dy), ops._ptr(x), ops._ptr(mean), ops._ptr(rstd), ops._ptr(w), M, d, ops._ptr(dres),
         1 if accumulate else 0, ops._ptr(dxb), ops._ptr(dg), ops._ptr(db), None, ops._stream())
    assert torch.equal(old[0], dres) and torch.equal(old[1], dxb)
    # dgamma / dbeta: the column pass sums row blocks with atomics (order-dependent once M > 32 rows)
    for a, b_ in zip(old[2:], (dg, db)):
        assert torch.allclose(a, b_, rtol=1e-5, atol=1e-5 * float(a.abs().max()))
    new = run(extra)
    # old result + extra up to fp32 rounding: the kernel rounds prev + extra, then adds dLN/dx; old and new each round once more
    want = old[0].double() + extra.double()
    mag = new[0].double().abs() + old[0].double().abs() + extra.double().abs() + (dres0.double().abs() if accumulate else 0)
    assert ((new[0].double() - want).abs() <= 2.0 ** -23 * mag).all()
    assert torch.equal(new[1], new[0].bfloat16())  # the bf16 copy is the rounding of the fp32 result
    for a, b_ in zip(old[2:], new[2:]):  # dgamma / dbeta do not see the addend
        assert torch.allclose(a, b_, rtol=1e-5, atol=1e-5 * float(a.abs().max()))
    # fp64 reference of the whole update
    xd = x.double().requires_grad_(True)
    torch.nn.functional.layer_norm(xd, (d,), w.double(), b.double(), 1e-6).backward(dy.double())
    ref = xd.grad + (dres0.double() if accumulate else 0) + extra.double()
    assert frob(new[0], ref) <= 1e-5


@pytest.mark.parametrize("n", [4, 8 * 1031, 2 * 1031 * 768])
def test_scale_add_recast(ops, n):
    g = torch.Generator().manual_seed(n)
    x0, a = torch.randn(n, generator=g).to(DEV), torch.randn(n, generator=g).to(DEV)
    sc = torch.tensor([0.75], device=DEV)
    x = x0.clone()
    xb = ops.scale_add_recast_(x, None, a)
    assert torch.equal(x, x0 + a) and torch.equal(xb, x.bfloat16())  # one fp32 add: exact rounding
    x = x0.clone()
    xb = ops.scale_add_recast_(x, sc, a)
    want = 0.75 * x0.double() + a.double()
    assert ((x.double() - want).abs() <= 2.0 ** -23 * (want.abs() + a.double().abs())).all() and torch.equal(xb, x.bfloat16())
    x = x0.clone()
    assert ops.scale_add_recast_(x, sc, None, want_bf16=False) is None
    assert torch.equal(x, x0 * 0.75)  # 0.75 x is exact in fp32
    x = x0.clone()
    ops.scale_add_recast_(x, torch.zeros(1, device=DEV), a)
    assert torch.equal(x, a)


# ---------------------------------------------------------------------------- forward
@pytest.mark.parametrize("name", ["tiny", "small64"])
@pytest.mark.parametrize("B", [1, 2])
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("mean_pooling", [True, False])
def test_encoder_states_match_oracle(ops, name, B, masked, mean_pooling):
    cfgd = _cfgd(name, use_mean_pooling=mean_pooling)
    cfg = vo.OracleConfig(**cfgd)
    sd = vo.synthetic_state_dict(cfg, 1234)
    m = _encoder(cfgd, sd)
    x = vo.synthetic_volume(cfg, B, 7)
    mask = _mask(B) if masked else None
    mdev = None if mask is None else mask.to(DEV)
    with torch.no_grad():
        want = oracle_states(sd, cfg, x, mask)
        out = m(x.to(DEV), mdev, output_hidden_states=True)
        off = m(x.to(DEV), mdev)
    assert off.hidden_states is None and len(out.hidden_states) == cfg.num_hidden_layers + 1
    for k, (h, w) in enumerate(zip(out.hidden_states, want)):
        assert h.dtype == torch.float32 and h.shape == w.shape, k
        assert frob(h, w) <= 2e-2 and maxrel(h, w) <= 5e-2, k
    assert torch.equal(out.last_hidden_state, off.last_hidden_state)  # the flag changes no output
    if mean_pooling:
        assert out.hidden_states[-1] is out.last_hidden_state
    # state k == last_hidden_state of the same weights cut to k blocks (no final LayerNorm), bit for bit
    for k in range(cfg.num_hidden_layers + 1):
        cut = dict(cfgd, num_hidden_layers=k, use_mean_pooling=True)
        mk = _encoder(cut, {n: v for n, v in sd.items() if not n.startswith("videomae.layernorm.") and
                            not any(n.startswith(f"videomae.encoder.layer.{i}.") for i in range(k, cfg.num_hidden_layers))})
        with torch.no_grad():
            assert torch.equal(mk(x.to(DEV), mdev).last_hidden_state, out.hidden_states[k]), k


def test_config_flag_tuple_order_and_bf16(ops):
    from smb_vision_b200.modeling import B200VideoMAEModel

    cfg = vo.OracleConfig(**ge.SMALL64)
    sd = vo.synthetic_state_dict(cfg, 1234)
    m = _encoder(ge.SMALL64, sd)
    x = vo.synthetic_volume(cfg, 1, 7).to(DEV)
    with torch.no_grad():
        ref = m(x, output_hidden_states=True)
        m.config.output_hidden_states = True
        by_cfg = m(x)
        tup = m(x, return_dict=False)
        assert m(x, output_hidden_states=False).hidden_states is None
        m.config.output_hidden_states = False
    assert all(torch.equal(a, b) for a, b in zip(by_cfg.hidden_states, ref.hidden_states))
    assert len(tup) == 2 and torch.equal(tup[0], ref.last_hidden_state) and len(tup[1]) == cfg.num_hidden_layers + 1
    mb = B200VideoMAEModel(ge.hf_config(ge.SMALL64)).to(DEV)
    mb.load_state_dict(_encoder_sd(sd))
    mb.set_reduced_precision(torch.bfloat16)
    with torch.no_grad():
        ob = mb(x, output_hidden_states=True)
    assert all(h.dtype == torch.bfloat16 for h in ob.hidden_states) and ob.hidden_states[-1] is ob.last_hidden_state
    want = oracle_states(sd, cfg, x.cpu())
    for h, w in zip(ob.hidden_states, want):
        assert frob(h.float(), w) <= 2e-2


@pytest.mark.parametrize("style", ["mae", "simmim"])
def test_pretraining_and_classification_states(ops, style):
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining, B200VideoMAEForVideoClassification

    cfg = vo.OracleConfig(**ge.SMALL64)
    sd = vo.synthetic_state_dict(cfg, 1234)
    sd["videomae.embeddings.mask_token"] = 0.2 * torch.randn(1, 1, cfg.hidden_size, generator=torch.Generator().manual_seed(4))
    pre = B200VideoMAEForPreTraining(ge.hf_config(ge.SMALL64), mim_style=style).to(DEV)
    pre.load_state_dict({k: v for k, v in sd.items() if k in pre.state_dict()}, strict=True)
    x = vo.synthetic_volume(cfg, 2, 7)
    mask = _mask(2)
    with torch.no_grad():
        out = pre(x.to(DEV), mask, output_hidden_states=True)
        off = pre(x.to(DEV), mask)
        tup = pre(x.to(DEV), mask, output_hidden_states=True, return_dict=False)
    want = oracle_states(sd, cfg, x, mask, simmim=style == "simmim")
    assert len(out.hidden_states) == len(want)
    for h, w in zip(out.hidden_states, want):
        assert frob(h, w) <= 2e-2 and maxrel(h, w) <= 5e-2
    assert torch.equal(out.loss, off.loss) and torch.equal(out.logits, off.logits)
    assert len(tup) == 3 and torch.equal(tup[1], off.logits) and torch.equal(tup[2][0], out.hidden_states[0])
    hc = ge.hf_config(ge.SMALL64)
    hc.num_labels = 3
    cls = B200VideoMAEForVideoClassification(hc).to(DEV)
    csd = vo.synthetic_cls_state_dict(cfg, 3, 0, 1234)
    cls.load_state_dict(csd, strict=True)
    with torch.no_grad():
        co = cls(x.to(DEV), output_hidden_states=True)
        ct = cls(x.to(DEV), labels=torch.tensor([0, 2]), output_hidden_states=True, return_dict=False)
    assert len(ct) == 3 and ct[0].dim() == 0 and torch.equal(ct[2][0], co.hidden_states[0])
    for h, w in zip(co.hidden_states, oracle_states(csd, cfg, x)):
        assert frob(h, w) <= 2e-2 and maxrel(h, w) <= 5e-2


# ---------------------------------------------------------------------------- backward
def _probes(states, seed=5):
    """R_k for k in {0, 1, L}: loss term sum <R_k, H_k>, scaled so that it is of the order of the model losses."""
    g = torch.Generator().manual_seed(seed)
    L = len(states) - 1
    return {k: torch.randn(states[k].shape, generator=g) / states[k].numel() for k in sorted({0, 1, L})}


def _probe_loss(states, R):
    return sum((states[k].float() * R[k].to(states[k].device)).sum() for k in R)


def _check_grads(model, ref, prefix=""):
    bad = {}
    for k, p in model.named_parameters():
        r = ref.get(prefix + k)
        if r is None or float(r.abs().max()) == 0:  # the loss was not used: nothing reaches this parameter
            assert p.grad is None or float(p.grad.abs().max()) == 0, k
            continue
        e = frob(p.grad, r)
        if not e <= grad_tol(k, 2e-2):
            bad[k] = e
    assert not bad, bad


def _autocast_operands(sd, x):
    return {k: (v.bfloat16().float() if k == PE_W else v) for k, v in sd.items()}, x.bfloat16().float()


@pytest.mark.parametrize("name", ["tiny", "small64"])
@pytest.mark.parametrize("mean_pooling", [True, False])
@pytest.mark.parametrize("masked", [False, True])
def test_encoder_state_gradients(ops, name, mean_pooling, masked):
    cfgd = _cfgd(name, use_mean_pooling=mean_pooling)
    cfg = vo.OracleConfig(**cfgd)
    sd = vo.synthetic_state_dict(cfg, 1234)
    m = _encoder(cfgd, sd)
    x = vo.synthetic_volume(cfg, 1, 7)
    mask = _mask(1) if masked else None
    sdo, xo = _autocast_operands(sd, x)
    sdg = {k: v.clone().requires_grad_(True) for k, v in sdo.items() if k.startswith("videomae.")}
    states = oracle_states(sdg, cfg, xo, mask)
    R = _probes(states)
    last = vo.encoder(sdg, cfg, xo, mask)
    Rl = torch.randn(last.shape, generator=torch.Generator().manual_seed(9)) / last.numel()
    (_probe_loss(states, R) + (last * Rl).sum()).backward()
    ref = {k[len("videomae."):]: v.grad for k, v in sdg.items()}
    m.train()
    out = m(x.to(DEV), None if mask is None else mask.to(DEV), output_hidden_states=True)
    assert all(h.requires_grad for h in out.hidden_states)
    (_probe_loss(out.hidden_states, R) + (out.last_hidden_state * Rl.to(DEV)).sum()).backward()
    _check_grads(m, ref)
    # only the states, last_hidden_state unused
    m.zero_grad(set_to_none=True)
    for v in sdg.values():
        v.grad = None
    _probe_loss(oracle_states(sdg, cfg, xo, mask), R).backward()
    ref = {k[len("videomae."):]: v.grad for k, v in sdg.items()}
    out = m(x.to(DEV), None if mask is None else mask.to(DEV), output_hidden_states=True)
    _probe_loss(out.hidden_states, R).backward()
    _check_grads(m, ref)


def _mim(style, sd):
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining

    pre = B200VideoMAEForPreTraining(ge.hf_config(ge.SMALL64), mim_style=style).to(DEV)
    pre.load_state_dict({k: v for k, v in sd.items() if k in pre.state_dict()}, strict=True)
    return pre


@pytest.mark.parametrize("style", ["mae", "simmim"])
@pytest.mark.parametrize("loss_factor", [1.0, 3.0, None])
def test_pretraining_state_gradients(ops, style, loss_factor):
    """gradients = factor * d(loss) + sum_k d<R_k, H_k>: the upstream factor reaches the loss part only (None: loss unused)."""
    cfg = vo.OracleConfig(**ge.SMALL64)
    sd = vo.synthetic_state_dict(cfg, 1234)
    sd["videomae.embeddings.mask_token"] = 0.2 * torch.randn(1, 1, cfg.hidden_size, generator=torch.Generator().manual_seed(4))
    pre = _mim(style, sd)
    x = vo.synthetic_volume(cfg, 1, 7)
    mask = _mask(1)
    sdo, xo = _autocast_operands(sd, x)
    sdg = {k: v.clone().requires_grad_(True) for k, v in sdo.items() if k in pre.state_dict()}
    fwd = vo.pretrain_forward_simmim if style == "simmim" else vo.pretrain_forward
    loss, _, _ = fwd(sdg, cfg, xo, mask, "mse")  # mse: the L1 gradient sign(diff) flips near ties with bf16 logits
    states = oracle_states(sdg, cfg, xo, mask, simmim=style == "simmim")
    R = _probes(states)
    total = _probe_loss(states, R) + (0 if loss_factor is None else loss * loss_factor)
    total.backward()
    ref = {k: v.grad for k, v in sdg.items()}
    out = pre(x.to(DEV), mask, output_hidden_states=True)
    total = _probe_loss(out.hidden_states, R) + (0 if loss_factor is None else out.loss * loss_factor)
    total.backward()
    _check_grads(pre, ref)


@pytest.mark.parametrize("mean_pooling", [True, False])
@pytest.mark.parametrize("loss_factor", [1.0, 3.0, None])
def test_classification_state_gradients(ops, mean_pooling, loss_factor):
    from smb_vision_b200.modeling import B200VideoMAEForVideoClassification

    cfgd = _cfgd("small64", use_mean_pooling=mean_pooling)
    cfg = vo.OracleConfig(**cfgd)
    hc = ge.hf_config(cfgd)
    hc.num_labels = 3
    cls = B200VideoMAEForVideoClassification(hc).to(DEV)
    sd = {k: v for k, v in vo.synthetic_cls_state_dict(cfg, 3, 0, 1234).items() if k in cls.state_dict()}
    cls.load_state_dict(sd, strict=True)
    x = vo.synthetic_volume(cfg, 2, 7)
    labels = torch.tensor([0, 2])
    sdo, xo = _autocast_operands(sd, x)
    sdg = {k: v.clone().requires_grad_(True) for k, v in sdo.items()}
    loss, _ = vo.classify_forward(sdg, cfg, xo, None, labels, 3)
    states = oracle_states(sdg, cfg, xo)
    R = _probes(states)
    (_probe_loss(states, R) + (0 if loss_factor is None else loss * loss_factor)).backward()
    ref = {k: v.grad for k, v in sdg.items()}
    out = cls(x.to(DEV), labels=labels, output_hidden_states=True)
    (_probe_loss(out.hidden_states, R) + (0 if loss_factor is None else out.loss * loss_factor)).backward()
    _check_grads(cls, ref)


def test_unused_states_leave_gradients_unchanged(ops):
    cfg = vo.OracleConfig(**ge.SMALL64)
    sd = vo.synthetic_state_dict(cfg, 1234)
    pre = _mim("mae", sd)
    x = vo.synthetic_volume(cfg, 1, 7).to(DEV)
    mask = _mask(1)
    grads = []
    for flag in (False, True):
        pre.zero_grad(set_to_none=True)
        out = pre(x, mask, output_hidden_states=flag)
        assert (out.hidden_states is not None) == flag
        out.loss.backward()
        grads.append({k: p.grad.clone() for k, p in pre.named_parameters()})
    for k in grads[0]:
        assert frob(grads[1][k], grads[0][k]) <= 2e-4, k


def test_in_place_edit_of_a_state_raises(ops):
    cfg = vo.OracleConfig(**ge.SMALL64)
    m = _encoder(ge.SMALL64, vo.synthetic_state_dict(cfg, 1234))
    out = m(vo.synthetic_volume(cfg, 1, 7).to(DEV), output_hidden_states=True)
    out.hidden_states[1].mul_(2.0)
    with pytest.raises(RuntimeError, match="inplace"):
        out.hidden_states[0].sum().backward()


# ---------------------------------------------------------------------------- extraction
def test_embedding_runner_layers(ops):
    from smb_vision_b200.inference import EmbeddingRunner

    cfg = vo.OracleConfig(**dict(ge.SMALL64, use_mean_pooling=False))
    m = _encoder(dict(ge.SMALL64, use_mean_pooling=False), vo.synthetic_state_dict(cfg, 1234))
    vols = [vo.synthetic_volume(cfg, 1, 30 + i).pin_memory() for i in range(4)]
    layers = (2, 0, 1)
    with torch.no_grad():
        want = [torch.stack([m(v.to(DEV), output_hidden_states=True).hidden_states[k][0] for k in layers]).cpu() for v in vols]
    got = list(EmbeddingRunner(m, layers=layers).embed_stream(iter(vols), copy=True))
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert g.shape == (3, 216, cfg.hidden_size) and torch.equal(g, w)
    with torch.no_grad():
        plain = [m(v.to(DEV)).last_hidden_state.cpu() for v in vols]
    assert all(torch.equal(g, w) for g, w in zip(EmbeddingRunner(m).embed_stream(iter(vols), copy=True), plain))
    with pytest.raises(ValueError):
        EmbeddingRunner(m, layers=(3,))


# ---------------------------------------------------------------------------- full size
def test_full_size_states_are_deterministic(ops):
    """smb-vision-base at 512x512x320: all 13 states, bit-identical run to run; the last one is the flag-off output."""
    from smb_vision_b200.modeling import B200VideoMAEModel

    cfg = vo.OracleConfig()
    torch.manual_seed(0)
    m = B200VideoMAEModel(ge.hf_config({k: getattr(cfg, k) for k in cfg.__dataclass_fields__})).to(DEV)
    x = vo.synthetic_volume(cfg, 1, 7).to(DEV)
    with torch.no_grad():
        a = m(x, output_hidden_states=True).hidden_states
        b = m(x, output_hidden_states=True).hidden_states
        off = m(x).last_hidden_state
    assert len(a) == 13 and all(h.shape == (1, 20480, 768) for h in a)
    assert all(torch.equal(p, q) for p, q in zip(a, b))
    assert torch.equal(a[-1], off)
    assert all(torch.isfinite(h).all() for h in a)
