"""GPU parity of the native V-JEPA2-3D encoder path (SURVEY.md §8f rank 4): the rotary-embedding kernel and the whole
encoder against oracle/vjepa_oracle.py and against tests/golden/vjepa_small64.npz (outputs of the reference module).

Tolerances: the kernel rotates bf16 Q/K in fp32 and rounds once to bf16: |err| <= 2^-8 |ref| + 1e-5 elementwise against
the fp32 oracle on the same bf16-rounded input; encoder embeddings as in test_gpu_parity.py (Frobenius-rel <= 2e-2,
max-abs-rel <= 5e-2: bf16 operands vs the fp32 reference)."""
import os

import numpy as np
import pytest
import torch

from oracle import vjepa_oracle as vj

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def ops():
    assert torch.cuda.is_available()
    from smb_vision_b200 import load, ops as _ops

    assert load().smbv_device_ok() == 0
    return _ops


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "vjepa_small64.npz"))


def hf_config(cfgd):
    from transformers import VJEPA2Config

    return VJEPA2Config(**cfgd, pred_hidden_size=64, pred_num_attention_heads=2, pred_num_hidden_layers=1, pred_num_mask_tokens=2)


def frob(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return (torch.linalg.norm(a - b) / torch.linalg.norm(b)).item()


def maxrel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).abs().max() / b.abs().max()).item()


def close_bf16(got, ref):
    err = (got.float().cpu() - ref).abs()
    return bool((err <= 2.0**-8 * ref.abs() + 1e-5).all()), float(err.max())


@pytest.mark.parametrize("D,transpose,masked", [(64, False, False), (64, True, False), (64, False, True), (64, True, True),
                                                (32, False, False), (32, True, True), (128, False, True)])
def test_rope3d_matches_oracle(ops, D, transpose, masked):
    g = torch.Generator().manual_seed(D + 2 * transpose + masked)
    G, B, H, n, gs = 2, 2, 3, 80, 4  # ids up to 5*16: frames 0..4
    x = torch.randn(G, B, H, n, D, generator=g).bfloat16()
    ids = torch.stack([torch.randperm(5 * gs * gs, generator=g)[:n].sort().values for _ in range(B)]) if masked else None
    ref = torch.stack([vj.rope3d(x[i].float(), ids, gs, transpose) for i in range(G)])
    got = ops.rope3d_(x.to(DEV), gs, None if ids is None else ids.int().to(DEV), max_pos=8, transpose=transpose)
    ok, worst = close_bf16(got, ref)
    assert ok, worst
    S = 2 * ((D // 3) // 2)
    assert torch.equal(got[..., 3 * S:].cpu(), x[..., 3 * S:])  # pass-through tail: untouched bits


@pytest.mark.parametrize("D,n,gs,masked", [(64, 80, 4, True), (64, 1031, 8, False), (32, 513, 4, True), (128, 77, 4, False), (64, 20480, 32, False)])
def test_rope3d_kernels_agree_bit_for_bit(ops, D, n, gs, masked):
    """the default kernel (2-D grid, multiply-shift position decode, 4 rows in flight) against the first-generation kernel
    (flat index, integer divisions): same table, same arithmetic -> identical bits, forward and transposed, incl. ragged n."""
    g = torch.Generator().manual_seed(n + D)
    x = torch.randn(2, 2, 3, n, D, generator=g).bfloat16().to(DEV)
    ids = None
    if masked:
        ids = torch.stack([torch.randperm(4 * n, generator=g)[:n].sort().values for _ in range(2)]).int().to(DEV)
    for tr in (False, True):
        a = ops.rope3d_(x.clone(), gs, ids, max_pos=16, transpose=tr)
        b = ops.rope3d_(x.clone(), gs, ids, max_pos=16, transpose=tr, first_generation_kernel=True)
        assert torch.equal(a, b)


def test_rope3d_positions_beyond_the_table(ops):
    """the reference lets position masks extrapolate past the configured grid (modeling_vjepa.py:303): ids whose frame
    index exceeds max_pos take the direct sincosf path and must give the same numbers as the tabulated one."""
    g = torch.Generator().manual_seed(5)
    x = torch.randn(1, 1, 2, 64, 64, generator=g).bfloat16()
    ids = (torch.arange(64) * 37 % 997).sort().values[None]  # frames up to 62 with a 4x4 grid
    ref = vj.rope3d(x[0].float(), ids, 4)[None]
    a = ops.rope3d_(x.to(DEV), 4, ids.int().to(DEV), max_pos=4)
    b = ops.rope3d_(x.to(DEV), 4, ids.int().to(DEV), max_pos=64)
    assert close_bf16(a, ref)[0] and close_bf16(b, ref)[0]
    assert (a.float() - b.float()).abs().max().item() <= 2.0**-7 * ref.abs().max().item()


def test_rope3d_matches_reference_golden(ops, gold):
    """the reference's own apply_rotary_embeddings output and autograd gradient (fp32) — input and output rounded to bf16."""
    for case in ("arange", "masked"):
        ids = None if case == "arange" else torch.from_numpy(gold["rope_mask_ids"]).int().to(DEV)
        for src, dst, tr in ((f"rope_{case}_in", f"rope_{case}_out", False), (f"rope_{case}_upstream", f"rope_{case}_grad", True)):
            x, ref = torch.from_numpy(gold[src]), torch.from_numpy(gold[dst])
            got = ops.rope3d_(x.bfloat16().to(DEV), 4, ids, max_pos=4, transpose=tr)
            assert frob(got.float(), ref) <= 4e-3 and maxrel(got.float(), ref) <= 1e-2


def test_rope3d_full_size_properties(ops):
    """ViT-L at 512x512x320: Q and K of 16 heads x 20480 tokens.  Size-independent properties: token 0 and the 4 tail
    elements are bit-unchanged, the map is linear, and `transpose` is its adjoint (<R x, g> == <x, R^T g>)."""
    torch.manual_seed(0)
    shape = (2, 1, 16, 20480, 64)
    x = torch.randn(shape, device=DEV).bfloat16()
    g = torch.randn(shape, device=DEV).bfloat16()
    y = ops.rope3d_(x.clone(), 32, max_pos=32)
    assert torch.equal(y[..., 60:], x[..., 60:]) and torch.equal(y[:, :, :, 0], x[:, :, :, 0])
    assert not torch.equal(y[:, :, :, 1, :60], x[:, :, :, 1, :60])
    gt = ops.rope3d_(g.clone(), 32, max_pos=32, transpose=True)
    lhs, rhs = (y.double() * g.double()).sum().item(), (x.double() * gt.double()).sum().item()
    scale = (y.double().norm() * g.double().norm()).item()
    assert abs(lhs - rhs) <= 1e-4 * scale  # bf16 output rounding, 84M terms of random sign
    y2 = ops.rope3d_((2 * x).clone(), 32, max_pos=32)
    assert torch.equal(y2, 2 * y)  # scaling by 2 is exact in bf16


@pytest.fixture(scope="module")
def small_vjepa(ops):
    from smb_vision_b200.vjepa import B200VJEPA2Model

    cfg = vj.VJepaOracleConfig(**vj.SMALL64_VJEPA)
    sd = vj.synthetic_state_dict(cfg)
    model = B200VJEPA2Model(hf_config(vj.SMALL64_VJEPA)).to(DEV).eval()
    res = model.load_state_dict(sd, strict=False)
    assert not res.unexpected_keys and all(k.startswith("predictor.") for k in res.missing_keys)
    return cfg, sd, model


def test_vjepa_encoder_matches_reference_golden(small_vjepa, gold):
    """B200VJEPA2Model(x, context_mask, target_mask, skip_predictor=True) vs the reference model's outputs."""
    cfg, sd, model = small_vjepa
    x = vj.synthetic_video(cfg, 2)
    ctx, tgt = torch.from_numpy(gold["context_mask"]), torch.from_numpy(gold["target_mask"])
    out = model(x.to(DEV), context_mask=[ctx], target_mask=[tgt], skip_predictor=True)
    assert out.predictor_output is None and out.last_hidden_state.dtype == torch.float32
    for name in ("last_hidden_state", "masked_hidden_state", "target_hidden_state"):
        got, ref = getattr(out, name), torch.from_numpy(gold[name])
        assert got.shape == ref.shape
        assert frob(got, ref) <= 2e-2 and maxrel(got, ref) <= 5e-2, (name, frob(got, ref), maxrel(got, ref))
    feats = model.get_vision_features(x.to(DEV))  # inference path; `out` above came from the training forward (grads enabled)
    assert frob(feats, out.last_hidden_state.detach()) <= 1e-3
    with torch.no_grad():
        assert torch.equal(model(x.to(DEV), skip_predictor=True).last_hidden_state, feats)


def test_vjepa_encoder_is_sensitive_to_rope_and_key_bias(small_vjepa, gold):
    """negative control: dropping the K bias or the rotary step moves the output far outside the tolerance — the parity
    above is not vacuous."""
    from smb_vision_b200 import modeling

    cfg, sd, model = small_vjepa
    x = vj.synthetic_video(cfg, 2).to(DEV)
    ref = torch.from_numpy(gold["last_hidden_state"])
    vol = model._volume(x)
    pk = model.packed()
    X = modeling.ops.patch_embed_fwd(vol, pk["wpe"], pk["bpe"], None)
    for p in pk["layers"]:
        modeling._block_forward(X, p, None)  # no rope
    no_rope = modeling.ops.layernorm_fwd(X, pk["g"], pk["b"], cfg.layer_norm_eps).float()
    assert frob(no_rope, ref) > 0.2
    with torch.no_grad():
        saved = model.encoder.layer[0].attention.key.bias.clone()
        model.encoder.layer[0].attention.key.bias.add_(1.0)
        moved = model.get_vision_features(x)
        model.encoder.layer[0].attention.key.bias.copy_(saved)
    assert frob(moved, ref) > 0.08
    assert frob(model.get_vision_features(x), ref) <= 2e-2


def test_vjepa_forward_with_predictor_matches_upstream(small_vjepa):
    """skip_predictor=False: native encoder + the upstream predictor through the attention plug-in vs the upstream
    VJEPA2Model (fp32, sdpa) with the same weights."""
    from transformers import VJEPA2Model

    cfg, sd, model = small_vjepa
    torch.manual_seed(3)
    hf = hf_config(vj.SMALL64_VJEPA)
    hf._attn_implementation = "sdpa"
    up = VJEPA2Model(hf).to(DEV).eval()
    with torch.no_grad():
        for p in up.predictor.parameters():  # mask tokens / biases start at zero: perturb so that they matter
            p.add_(0.02 * torch.randn_like(p))
    model.load_state_dict(up.state_dict(), strict=True)
    x = vj.synthetic_video(cfg, 2).to(DEV)
    N = cfg.num_patches
    g = torch.Generator().manual_seed(1)
    perm = torch.stack([torch.randperm(N, generator=g) for _ in range(2)])
    ctx, tgt = perm[:, :30].sort(dim=1).values.to(DEV), perm[:, 30:].sort(dim=1).values.to(DEV)
    with torch.no_grad():
        want = up(pixel_values_videos=x, context_mask=[ctx], target_mask=[tgt])
    got = model(x, context_mask=[ctx], target_mask=[tgt])
    assert frob(got.last_hidden_state, want.last_hidden_state) <= 2e-2
    pw, pg = want.predictor_output.last_hidden_state, got.predictor_output.last_hidden_state
    assert pg.shape == pw.shape and frob(pg, pw) <= 3e-2, frob(pg, pw)
    want_tgt = torch.gather(want.last_hidden_state, 1, tgt.unsqueeze(-1).expand(-1, -1, want.last_hidden_state.size(-1)))
    assert frob(got.predictor_output.target_hidden_state, want_tgt) <= 2e-2
    model.load_state_dict(sd, strict=False)


def test_vjepa_embedding_runner(small_vjepa):
    """the overlapped H2D / compute / D2H extraction loop (src/run_inference.py:99-123 role) serves the V-JEPA encoder too."""
    from smb_vision_b200.inference import EmbeddingRunner

    cfg, sd, model = small_vjepa
    vols = [vj.synthetic_video(cfg, 1, 40 + i).pin_memory() for i in range(4)]
    want = [model.get_vision_features(v.to(DEV)).cpu() for v in vols]
    got = [e.clone() for e in EmbeddingRunner(model).embed_stream(iter(vols))]
    assert len(got) == 4 and all(torch.equal(g, w) for g, w in zip(got, want))


def test_vjepa_errors(small_vjepa):
    from smb_vision_b200 import SmbvError
    from smb_vision_b200.vjepa import B200VJEPA2Model

    cfg, sd, model = small_vjepa
    with pytest.raises(ValueError):
        model(None)
    with pytest.raises(ValueError):
        model(torch.zeros(1, 48, 3, 64, 64))
    bad = dict(vj.SMALL64_VJEPA, num_attention_heads=4)  # head_dim 32
    m = B200VJEPA2Model(hf_config(bad), with_predictor=False).to(DEV)
    with pytest.raises(SmbvError):
        m(torch.zeros(1, 48, 1, 64, 64), skip_predictor=True)
    with pytest.raises(SmbvError):
        m(torch.zeros(1, 48, 1, 64, 64))  # no predictor built


# ---------------------------------------------------------------------------- training: encoder backward
def test_vjepa_encoder_gradients_match_oracle_and_reference(small_vjepa, gold):
    """loss = <last_hidden_state, U>: the hand-written encoder backward (attention backward kernels, transposed rotary
    map, K-bias gradient, tubelet-embedding wgrad) against the oracle's autograd for EVERY encoder parameter, and against
    the reference model's own gradients for the stored selection.  Tolerance: Frobenius-rel 5e-2 per tensor (bf16
    operands and activations vs fp32; the MIM gradient test uses the same bound)."""
    cfg, sd, model = small_vjepa
    model.load_state_dict(sd, strict=False)
    x = vj.synthetic_video(cfg, 2)
    U = torch.from_numpy(gold["grad_upstream"])
    model.zero_grad(set_to_none=True)
    out = model(x.to(DEV), skip_predictor=True)
    assert out.last_hidden_state.requires_grad
    (out.last_hidden_state * U.to(DEV)).sum().backward()
    # the oracle sees the tubelet-embedding OPERANDS the way the kernel (and the reference's bf16-autocast Conv3d) does: volume and
    # weight rounded to bf16.  With this fixture's peaky attention (Q/K std 0.3) that 2^-9 input rounding alone moves the Q/K gradients
    # by 7e-2, which would mask what the test is about — the backward kernels.
    wk = "encoder.embeddings.patch_embeddings.proj_3d.weight"
    osd = {k: (v.bfloat16().float() if k == wk else v.clone()).requires_grad_(True) for k, v in sd.items()}
    (vj.encoder_forward(osd, cfg, x.bfloat16().float()) * U).sum().backward()
    got = {"encoder." + k: p.grad for k, p in model.encoder.named_parameters()}
    assert set(got) == set(osd) and all(g is not None for g in got.values())
    # K bias: sum_j dK_j vanishes identically without the rotary map (softmax-backward rows sum to zero), so with it the
    # gradient is a small residual of cancelling bf16 dK rows: measured 5.7e-2, bound 1.5e-1; everything else 5e-2
    # (round 2, bf16 tubelet-embedding operands: worst measured 5.8e-2 on a LayerNorm weight of this deliberately ill-conditioned fixture
    # — Q/K std 0.3 — where round 1's TF32 embedding gave 4.6e-2; bound 7e-2).
    # test_gpu_vjepa_kernels.py checks the K slot stage by stage (Frobenius-rel 5.3e-3 to the true gradient given the
    # kernels' own attention inputs) and shows why its bound cannot be derived tighter: the true K-bias gradient is only
    # 1.6 - 4.6x the worst case of the two bf16 roundings of dK alone
    tol = lambda k: 1.5e-1 if k.endswith("key.bias") else 7e-2
    errs = sorted(((frob(got[k], osd[k].grad), k) for k in osd), reverse=True)
    assert all(e <= tol(k) for e, k in errs), errs[:4]
    # the reference model's own (fp32) gradients: same bound plus the operand rounding of the embedding measured above
    for k in [f[len("grad::"):] for f in gold.files if f.startswith("grad::")]:
        assert frob(got[k], torch.from_numpy(gold["grad::" + k])) <= 2 * tol(k), k
    # the gradient reaches the masked views too, and a second backward accumulates
    model.zero_grad(set_to_none=True)
    ctx, tgt = torch.from_numpy(gold["context_mask"]).to(DEV), torch.from_numpy(gold["target_mask"]).to(DEV)
    o2 = model(x.to(DEV), context_mask=[ctx], target_mask=[tgt], skip_predictor=True)
    (o2.target_hidden_state.sum() + o2.masked_hidden_state.sum()).backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in model.encoder.parameters())


def test_vjepa_native_online_training_matches_plugin_route():
    """three optimisation steps of examples/train_vjepa.py: B200VJEPA2Model as the online model (native encoder forward
    AND backward, upstream predictor through the plug-in) against the upstream VJEPA2Model through the plug-in — the route
    already checked against the reference's plain-torch loop in tests/test_gpu_examples.py.  Same weights, same batches."""
    import sys

    import transformers

    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples"))
    import smb_vision_b200.attention_interface as ai
    import train_vjepa
    from smb_vision_b200.optim import EmaTarget, FusedAdamW
    from smb_vision_b200.vjepa import B200VJEPA2Model

    dev = torch.device(DEV)
    name = ai.register()
    kw = dict(patch_size=16, crop_size=64, frames_per_clip=64, tubelet_size=16, in_chans=1, hidden_size=128, num_attention_heads=2,
              num_hidden_layers=2, pred_hidden_size=64, pred_num_attention_heads=2, pred_num_hidden_layers=2, pred_num_mask_tokens=2)
    c = transformers.VJEPA2Config(**kw)
    c._attn_implementation = name
    torch.manual_seed(0)
    ma = transformers.VJEPA2Model(c).to(dev).train()
    with torch.no_grad():  # make attention matter (see oracle/vjepa_oracle.synthetic_state_dict)
        for k, p in ma.named_parameters():
            if k.startswith("encoder.") and k.endswith(("query.weight", "key.weight")):
                p.mul_(10.0)
    mb = B200VJEPA2Model(transformers.VJEPA2Config(**kw)).to(dev).train()
    mb.load_state_dict(ma.state_dict(), strict=True)
    g = torch.Generator().manual_seed(1)
    batches = []
    for _ in range(3):
        x = torch.rand(2, 64, 1, 64, 64, generator=g).to(dev)
        perm = torch.randperm(64, generator=g)
        batches.append((x, [perm[:40].sort().values[None].repeat(2, 1).to(dev)], [perm[40:].sort().values[None].repeat(2, 1).to(dev)]))
    losses = []
    for m in (ma, mb):
        opt = FusedAdamW(m, lr=1e-3, weight_decay=0.01, max_grad_norm=1.0)
        grads = opt.grad_arena()
        tgt = EmaTarget(m, momentum=0.99925)
        losses.append([float(train_vjepa.vjepa_step(m, tgt, opt, grads, *b)) for b in batches])
    for a, b in zip(*losses):
        assert abs(a - b) / a <= 2e-2, losses
    assert losses[1][-1] != losses[1][0]
    big = lambda t: t.dim() >= 2 and float(t.detach().abs().mean()) > 5e-3
    pa = dict(ma.named_parameters())
    worst = max((frob(p.detach(), pa[k.replace("proj_3d", "proj")].detach()), k) for k, p in mb.named_parameters() if big(p))
    assert worst[0] <= 5e-2, worst


@pytest.mark.parametrize("D,N", [(32, 1536), (16, 1100)])
def test_plugin_pads_small_heads_to_the_tcgen05_kernels(ops, D, N):
    """head_dim 32 (the V-JEPA predictor, 384/12) at >= 1024 tokens: Q, K, V are zero-padded to 64 and run on the tcgen05
    forward AND backward kernels; result and gradients vs fp32 SDPA.  Also times the predictor shape against the small-head
    route it replaces."""
    import smb_vision_b200.attention_interface as ai

    g = torch.Generator().manual_seed(D)
    B, H = 2, 3
    q, k, v, up = (torch.randn(B, H, N, D, generator=g).to(DEV) for _ in range(4))
    ref_in = [t.clone().requires_grad_(True) for t in (q, k, v)]
    ref = torch.nn.functional.scaled_dot_product_attention(*ref_in, scale=D ** -0.5)  # [B,H,N,D] fp32
    (ref * up).sum().backward()
    ins = [t.clone().requires_grad_(True) for t in (q, k, v)]
    out, _ = ai.b200_flash_attention(None, *ins, scaling=D ** -0.5)
    assert out.shape == (B, N, H, D) and out.is_contiguous() and out.dtype == torch.float32
    (out * up.transpose(1, 2)).sum().backward()
    assert frob(out.transpose(1, 2), ref) <= 1e-2
    for a, b in zip(ins, ref_in):
        assert frob(a.grad, b.grad) <= 2e-2
    # below the threshold the small-head kernels serve the call (exact fp32 softmax) and agree with the padded route
    old = ai.PAD_TO_64_MIN_TOKENS
    try:
        ai.PAD_TO_64_MIN_TOKENS = 1 << 30
        with torch.no_grad():
            small, _ = ai.b200_flash_attention(None, q, k, v, scaling=D ** -0.5)
    finally:
        ai.PAD_TO_64_MIN_TOKENS = old
    assert frob(small, out.detach()) <= 1e-2


def test_predictor_shape_speed_padded_vs_small_head(ops):
    """V-JEPA predictor attention at the full token count (12 heads x 32, 20 480 tokens): the padded tcgen05 route must be
    at least 3x faster than the small-head kernels (measured: see profiles/r01_vjepa.md)."""
    import smb_vision_b200.attention_interface as ai

    q, k, v = (torch.randn(1, 12, 20480, 32, device=DEV).bfloat16() for _ in range(3))

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    with torch.no_grad():
        t_pad = timed(lambda: ai.b200_flash_attention(None, q, k, v, scaling=32 ** -0.5))
        old = ai.PAD_TO_64_MIN_TOKENS
        try:
            ai.PAD_TO_64_MIN_TOKENS = 1 << 30
            t_small = timed(lambda: ai.b200_flash_attention(None, q, k, v, scaling=32 ** -0.5))
        finally:
            ai.PAD_TO_64_MIN_TOKENS = old
    print(f"predictor attention forward, H=12 D=32 N=20480: padded tcgen05 {t_pad:.2f} ms, small-head kernels {t_small:.2f} ms")
    assert t_pad * 3 <= t_small


# ---------------------------------------------------------------------------- index / loss kernels of the step
@pytest.mark.parametrize("B,N,K,d", [(2, 48, 20, 128), (1, 20480, 12345, 1024), (3, 64, 64, 4), (2, 48, 0, 128)])
def test_gather_rows_equals_torch_gather(ops, B, N, K, d):
    """apply_masks (modeling_vjepa.py:543-557): bit-exact row gather."""
    from smb_vision_b200.vjepa import apply_masks

    g = torch.Generator().manual_seed(K)
    src = torch.randn(B, N, d, generator=g).to(DEV)
    idx = torch.stack([torch.randperm(N, generator=g)[:K] for _ in range(B)]).to(DEV)  # int64, unsorted
    want = torch.gather(src, 1, idx.unsqueeze(-1).expand(-1, -1, d))
    assert torch.equal(ops.gather_rows(src, idx.int()), want)
    with torch.no_grad():
        assert torch.equal(apply_masks(src, [idx]), want)
        assert torch.equal(apply_masks(src, [idx, idx.flip(1)]), torch.cat([want, want.flip(1)], 0))
    s2 = src.clone().requires_grad_(True)  # a tensor that carries gradient keeps torch's differentiable gather
    if K:
        apply_masks(s2, [idx]).sum().backward()
        assert float(s2.grad.sum()) == B * K * d


@pytest.mark.parametrize("shape", [(2, 12, 128), (1, 13312, 1024), (4,), (3, 7, 5), (1,), (1031,)])  # incl. n % 4 != 0 (scalar tail)
def test_l1_loss_matches_torch(ops, shape):
    """nn.L1Loss (src/run_vjepa.py:108): value rel <= 1e-6 (fp64 final sum vs torch's fp32 tree), gradient = sign / n incl.
    sign(0) = 0, deterministic."""
    from smb_vision_b200.vjepa import l1_loss

    g = torch.Generator().manual_seed(len(shape))
    p = torch.randn(shape, generator=g).to(DEV)
    t = torch.randn(shape, generator=g).to(DEV)
    t.view(-1)[::7] = p.view(-1)[::7]  # exact ties: gradient 0 there
    pr = p.clone().requires_grad_(True)
    ref = torch.nn.functional.l1_loss(pr, t)
    (3.0 * ref).backward()
    pk = p.clone().requires_grad_(True)
    got = l1_loss(pk, t)
    (3.0 * got).backward()
    assert got.shape == () and abs(got.item() - ref.item()) <= 1e-6 * ref.item()
    assert torch.allclose(pk.grad, pr.grad, rtol=1e-6, atol=0) and bool((pk.grad.view(-1)[::7] == 0).all())
    a, b = ops.l1_loss(p, t), ops.l1_loss(p, t)
    assert torch.equal(a, b)
    with torch.no_grad():
        assert abs(l1_loss(p, t).item() - ref.item()) <= 1e-6 * ref.item()


# ---------------------------------------------------------------------------- native predictor (round 2)
def test_position_sort_and_heads32_layout_kernels(ops):
    """smbv_position_sort == torch.argsort (stable) + reverse argsort + sorted ids (modeling_vjepa.py:708, :674-679), incl. duplicate
    positions (the default masks are arange twice); smbv_heads32_convert pads / squeezes exactly."""
    g = torch.Generator().manual_seed(0)
    for B, n in [(2, 48), (1, 1000), (3, 257)]:
        pos = torch.randint(0, max(2, n // 2), (B, n), generator=g, dtype=torch.int32)  # many ties
        order, inv, srt, s2 = ops.position_sort(pos.to(DEV), doubled=True)
        want = torch.argsort(pos.long(), dim=1, stable=True)
        assert torch.equal(order.cpu().long(), want)
        assert torch.equal(inv.cpu().long(), torch.argsort(want, dim=1))
        assert torch.equal(srt.cpu(), torch.gather(pos, 1, want))
        assert torch.equal(s2.cpu(), torch.gather(pos, 1, want).repeat_interleave(2, dim=1))
    x = torch.randn(3, 2, 3, 50, 64, generator=g).bfloat16().to(DEV)  # [3, B, H/2, n, 64]
    e = ops.heads32_expand(x)  # [3, B, H, n, 64]
    assert e.shape == (3, 2, 6, 50, 64) and float(e[..., 32:].abs().max()) == 0.0
    assert torch.equal(e[:, :, 0::2, :, :32], x[..., :32]) and torch.equal(e[:, :, 1::2, :, :32], x[..., 32:])
    assert torch.equal(ops.heads32_squeeze(e), x)
    t = torch.randn(2, 50, 6 * 32, generator=g).bfloat16().to(DEV)
    te = ops.heads32_tokens(t, 6, expand=True)
    assert torch.equal(te.view(2, 50, 6, 64)[..., :32], t.view(2, 50, 6, 32)) and float(te.view(2, 50, 6, 64)[..., 32:].abs().max()) == 0.0
    assert torch.equal(ops.heads32_tokens(te, 6, expand=False), t)


@pytest.fixture(scope="module")
def small_vjepa_pred(ops):
    from smb_vision_b200.vjepa import B200VJEPA2Model

    cfgd = dict(vj.SMALL64_VJEPA, **vj.SMALL64_VJEPA_PRED)  # predictor 64 / 2 heads: head_dim 32 -> the zero-padded tcgen05 route
    cfg = vj.VJepaOracleConfig(**cfgd)
    sd = {**vj.synthetic_state_dict(cfg), **vj.synthetic_predictor_state_dict(cfg)}
    model = B200VJEPA2Model(hf_config(vj.SMALL64_VJEPA)).to(DEV)  # hf_config adds the SMALL64_VJEPA_PRED predictor sizes
    model.load_state_dict(sd, strict=True)
    return cfg, sd, model


def test_native_predictor_matches_reference_golden(small_vjepa_pred, gold):
    """whole forward with the NATIVE predictor (gather, Linear, mask token, position sort, rotary with sorted ids, head_dim-32
    attention on the padded tcgen05 kernels, LayerNorm, projection) vs the reference model's own predictor output (golden)."""
    cfg, sd, model = small_vjepa_pred
    x = vj.synthetic_video(cfg, 2).to(DEV)
    ctx, tgt = torch.from_numpy(gold["context_mask"]).to(DEV), torch.from_numpy(gold["target_mask"]).to(DEV)
    with torch.no_grad():
        out = model(x, context_mask=[ctx], target_mask=[tgt])
    ref = torch.from_numpy(gold["predictor_last_hidden_state"])
    got = out.predictor_output.last_hidden_state
    assert got.shape == ref.shape and got.dtype == torch.float32
    assert frob(got, ref) <= 3e-2, frob(got, ref)
    assert frob(out.predictor_output.target_hidden_state, torch.from_numpy(gold["predictor_target_hidden_state"])) <= 2e-2
    # the comparison sees what a port gets wrong: the other mask token moves the output far beyond the tolerance
    model._pred_runner.mask_index = 0
    model._pred_runner.invalidate()
    with torch.no_grad():
        wrong = model(x, context_mask=[ctx], target_mask=[tgt]).predictor_output.last_hidden_state
    model._pred_runner.mask_index = 1
    model._pred_runner.invalidate()
    assert frob(wrong, ref) > 0.1


def test_native_predictor_gradients_match_oracle(small_vjepa_pred, gold):
    """loss = <predictions, U>: every predictor parameter gradient and the gradient w.r.t. the encoder output against autograd
    over the oracle restatement (fp32) fed the SAME encoder output."""
    cfg, sd, model = small_vjepa_pred
    runner = model._pred_runner
    g = torch.Generator().manual_seed(11)
    ctx, tgt = torch.from_numpy(gold["context_mask"]), torch.from_numpy(gold["target_mask"])
    with torch.no_grad():
        enc = model.get_vision_features(vj.synthetic_video(cfg, 2).to(DEV)).cpu()
    U = torch.randn(2, tgt.shape[1], cfg.hidden_size, generator=g)
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items() if k.startswith("predictor.")}
    enc_ref = enc.clone().requires_grad_(True)
    (vj.predictor_forward({**sd, **sdg}, cfg, enc_ref, [ctx], [tgt]) * U).sum().backward()
    from smb_vision_b200.vjepa import _PredictorFunction

    enc_dev = enc.to(DEV).requires_grad_(True)
    named = list(model.predictor.named_parameters())
    model.zero_grad(set_to_none=True)
    pred = _PredictorFunction.apply(runner, enc_dev, [ctx.to(DEV)], [tgt.to(DEV)], tuple(n for n, _ in named), *[p for _, p in named])
    (pred * U.to(DEV)).sum().backward()
    assert frob(enc_dev.grad, enc_ref.grad) <= 3e-2, frob(enc_dev.grad, enc_ref.grad)
    bad = {}
    for n, p in named:
        ref = sdg["predictor." + n].grad
        if n == "embeddings.mask_tokens":  # only the chosen token (index 1) is used
            assert float(p.grad[0].abs().max()) == 0.0
        e = frob(p.grad, ref)
        # K bias: a residual of cancelling bf16 dK rows (see the encoder test and test_gpu_vjepa_kernels.py)
        if not e <= (1.5e-1 if n.endswith("key.bias") else 5e-2):
            bad[n] = e
    assert not bad, bad
    model.zero_grad(set_to_none=True)
