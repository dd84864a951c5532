"""GPU parity tests (run with -m gpu on the B200 box).  Every test calls the CUDA path through the C ABI
(smb_vision_b200.ops -> ctypes -> libsmbv_b200.so) and compares with the CPU oracle on the same seeded inputs.

Tolerances (SURVEY.md §8c, calibrated against the reference's own bf16-autocast-vs-fp32 deviation):
  mask / index lists: exact;   loss rel <= 1e-4 (model level), <= 1e-5 (loss kernel alone, fp32 logits path);
  logits Frobenius-rel <= 1e-2, max-abs-rel <= 2e-2;   embeddings Frobenius-rel <= 2e-2, max-abs-rel <= 5e-2.
"""
import json
import os

import numpy as np
import pytest
import torch

import __graft_entry__ as ge
from oracle import videomae_oracle as vo
from oracle.mim_mask import OracleMaskGenerator

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def ops():
    assert torch.cuda.is_available()
    from smb_vision_b200 import load, ops as _ops

    lib = load()
    assert lib.smbv_device_ok() == 0, lib.smbv_last_error()
    return _ops


def frob(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return (torch.linalg.norm(a - b) / torch.linalg.norm(b)).item()


def maxrel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).abs().max() / b.abs().max()).item()


PE_W = "videomae.embeddings.patch_embeddings.projection.weight"


def grad_tol(name, tol):
    """Frobenius-rel bound of one parameter gradient on the SMALL fixtures.  The layer-0 Q / K gradients are residuals of
    cancelling terms (every row of dS sums to zero) behind bf16 operands on both sides of the attention backward, so on the
    216-token, 2-head fixtures they carry 2-4e-2 of bf16 rounding noise when only a few rows receive gradient (measured on
    B200: q_bias 2.1e-2 through `.videomae`, 3.8e-2 with the CLS-row head); at the benchmark size the same gradients agree
    to 7e-3 (tests/test_gpu_fullsize.py).  Every other parameter keeps the tight bound."""
    qk = any(t in name for t in ("attention.query.weight", "attention.key.weight", "attention.q_bias"))
    return 5e-2 if qk else tol


def autocast_operands(sd, x):
    """the patch-embedding OPERANDS as the kernel (and the reference's bf16-autocast Conv3d) reads them: volume and Conv3d weight
    rounded to bf16.  Gradient comparisons against the fp32 oracle use them so that the 2^-9 input rounding — which the first
    attention layer amplifies into its Q/K gradients — is not mistaken for an error of the backward kernels."""
    return {k: (v.bfloat16().float() if k == PE_W else v) for k, v in sd.items()}, x.bfloat16().float()


# ---------------------------------------------------------------------------- masks (exact)
def test_mask_known_answers_on_device(ops, golden_dir):
    for kat in json.load(open(os.path.join(golden_dir, "mask_kat.json"))):
        np.random.seed(kat["seed"])
        g = OracleMaskGenerator(kat["input_size"], kat["depth"], kat["mask_patch_size"], kat["model_patch_size"], kat["mask_ratio"])
        coarse = g.coarse()
        fine = ops.mask_upsample(torch.from_numpy(coarse)[None].to(DEV), g.scale)
        ref = g.upsample(coarse, g.scale)
        assert np.array_equal(fine[0].cpu().numpy(), ref)  # exact mask equality
        vis, msk, slot, counts = ops.mask_index(fine)
        assert counts[0].tolist() == [kat["n"] - kat["n_mask"], kat["n_mask"]]
        assert msk[0, :10].tolist() == kat["first_masked"]
        assert np.array_equal(msk[0, : kat["n_mask"]].cpu().numpy(), np.nonzero(ref)[0])
        assert np.array_equal(vis[0, : kat["n"] - kat["n_mask"]].cpu().numpy(), np.nonzero(ref == 0)[0])


def test_mask_index_edge_cases(ops):
    for fine in [torch.zeros(1, 216, dtype=torch.uint8), torch.ones(2, 216, dtype=torch.uint8),
                 (torch.arange(3 * 1000).view(3, 1000) % 7 == 0).to(torch.uint8)]:
        vis, msk, slot, counts = ops.mask_index(fine.to(DEV))
        for b in range(fine.shape[0]):
            nz = torch.nonzero(fine[b]).flatten()
            z = torch.nonzero(fine[b] == 0).flatten()
            assert counts[b].tolist() == [len(z), len(nz)]
            assert torch.equal(msk[b, : len(nz)].cpu().long(), nz) and torch.equal(vis[b, : len(z)].cpu().long(), z)
            s = slot[b].cpu().long()
            assert torch.equal(s[nz], torch.arange(len(nz))) and torch.equal(s[z], torch.arange(len(z)))


# ---------------------------------------------------------------------------- bandwidth kernels
def test_sincos_table(ops):
    for n, d in [(216, 64), (216, 128), (20480, 768)]:
        got = ops.sincos_table(n, d, DEV).cpu()
        assert (got - vo.sinusoid_table(n, d)[0]).abs().max().item() <= 1.2e-7  # 1 ulp of fp32 at |x|<=1


@pytest.mark.parametrize("M,d,eps", [(216, 128, 1e-12), (72, 64, 1e-5), (5, 768, 1e-12), (1031, 384, 1e-5)])
def test_layernorm(ops, M, d, eps):
    g = torch.Generator().manual_seed(M + d)
    x = torch.randn(M, d, generator=g) * 3 + 1
    w, b = torch.randn(d, generator=g), torch.randn(d, generator=g)
    y, mean, rstd = ops.layernorm_fwd(x.to(DEV), w.to(DEV), b.to(DEV), eps, save_stats=True)
    ref = torch.nn.functional.layer_norm(x, (d,), w, b, eps)
    assert frob(y.float(), ref) <= 3e-3  # bf16 output rounding
    assert (mean.cpu() - x.mean(1)).abs().max() <= 1e-5
    assert ((rstd.cpu() - 1 / torch.sqrt(x.var(1, unbiased=False) + eps)).abs() / rstd.cpu()).max() <= 1e-4


@pytest.mark.parametrize("kind", ["mse", "l1"])
def test_normpix_loss_kernel_alone(ops, kind):
    """oracle logits in -> loss rel <= 1e-5 (SURVEY.md §8c), dlogits vs autograd."""
    cfg = vo.OracleConfig(**vo.TINY)
    B = 2
    x = vo.synthetic_volume(cfg, B, 11)
    x[1, :16, :, :16, :16] = 0.25  # a constant patch -> labels 0 (reference: 0 / (0 + 1e-6))
    np.random.seed(3)
    g = OracleMaskGenerator(96, 96, 32, 16, 0.65)
    mask = torch.from_numpy(np.stack([g(), g()]))
    if not mask[1, 0]:  # make sure the constant patch is a masked one, keeping the per-sample count equal
        j = torch.nonzero(mask[1]).flatten()[-1]
        mask[1, 0], mask[1, j] = True, False
    nm = int(mask[0].sum())
    assert int(mask[1].sum()) == nm
    lab = vo.labels_normpix(x, cfg)[mask].reshape(B, nm, -1)
    logits = (0.5 * torch.randn(B, nm, 4096, generator=torch.Generator().manual_seed(0))).to(torch.bfloat16)
    lf = logits.float().requires_grad_(True)
    ref = torch.nn.functional.mse_loss(lf, lab) if kind == "mse" else torch.nn.functional.l1_loss(lf, lab)
    ref.backward()
    _, midx, _, _ = ops.mask_index(mask.to(torch.uint8).to(DEV))
    loss, dl = ops.normpix_loss(x[:, :, 0].contiguous().to(DEV), midx, nm, logits.to(DEV), True, 0 if kind == "mse" else 1)
    assert abs(loss.item() - ref.item()) / ref.item() <= 1e-5
    assert frob(dl.float(), lf.grad) <= 5e-3  # bf16 gradient rounding
    loss2, none = ops.normpix_loss(x[:, :, 0].contiguous().to(DEV), midx, nm, logits.to(DEV), False, 0 if kind == "mse" else 1)
    assert none is None and loss2.item() == loss.item()  # deterministic reduction


def test_normpix_loss_full_size_closed_form(ops):
    """512x512x320: with logits == 0 the MSE is mean(label^2) = (K-1)/K * var/(sqrt(var)+1e-6)^2 ~ 4095/4096
    for every non-constant patch — a size-independent property, no CPU oracle needed at this size."""
    g = torch.Generator(device="cpu").manual_seed(5)
    vol = torch.rand(1, 320, 512, 512, generator=g).to(DEV)
    np.random.seed(0)
    mask = torch.from_numpy(OracleMaskGenerator(512, 320, 32, 16, 0.65)())[None]
    nm = int(mask.sum())
    _, midx, _, _ = ops.mask_index(mask.to(torch.uint8).to(DEV))
    logits = torch.zeros(1, nm, 4096, dtype=torch.bfloat16, device=DEV)
    loss, dl = ops.normpix_loss(vol, midx, nm, logits, True, 0)
    assert abs(loss.item() - 4095.0 / 4096.0) <= 2e-5
    # gradient of the mean: sum(dlogits) == -2/count * sum(labels) == 0 (zero-mean labels), |dl| small and finite
    assert torch.isfinite(dl.float()).all() and abs(dl.float().sum().item()) < 1e-3


# ---------------------------------------------------------------------------- tensor-core kernels
@pytest.mark.parametrize("M,N,K", [(216, 384, 128), (72, 128, 128), (144, 4096, 64), (300, 96, 32), (300, 160, 64), (1024, 768, 3072)])
def test_gemm_bias(ops, M, N, K):
    """N % 64 == 32 (96, 160): the bf16 epilogues' last slab is half outside the output (bias read only up to N)."""
    g = torch.Generator().manual_seed(M * N + K)
    a = torch.randn(M, K, generator=g).to(torch.bfloat16)
    w = (0.05 * torch.randn(N, K, generator=g)).to(torch.bfloat16)
    b = torch.randn(N, generator=g)
    ref = a.double() @ w.double().t() + b.double()
    out = ops.gemm(a.to(DEV), w.to(DEV), b.to(DEV), ops.EPI_F32)
    assert frob(out, ref) <= 2e-5  # fp32 accumulation of exact bf16 products
    out = ops.gemm(a.to(DEV), w.to(DEV), b.to(DEV), ops.EPI_BF16)
    assert frob(out.float(), ref) <= 4e-3
    out = ops.gemm(a.to(DEV), w.to(DEV), b.to(DEV), ops.EPI_GELU_BF16)
    assert frob(out.float(), torch.nn.functional.gelu(ref)) <= 4e-3
    res = torch.randn(M, N, generator=g)
    out = ops.gemm(a.to(DEV), w.to(DEV), b.to(DEV), ops.EPI_RESID_F32, residual=res.clone().to(DEV))
    assert frob(out, ref + res.double()) <= 2e-5


@pytest.mark.parametrize("M,N,K", [(1000, 512, 256), (7168, 3072, 768), (300, 1536, 384)])
def test_gemm_training_epilogues_gelu_with_saved_preactivation_and_dgelu(ops, M, N, K):
    """The two side-input epilogues of the training MLP, both on the TMA slab path since round 2 (ragged M included):
    fc1 forward = GELU(x W^T + b) AND the saved bf16 pre-activation (second slab store, reference :368-370 under autograd);
    fc2 dgrad  = (dY W) * gelu'(pre) with the pre-activation slab loaded by TMA (autograd of the exact-erf GELU)."""
    g = torch.Generator(device=DEV).manual_seed(M)
    a = torch.randn(M, K, device=DEV, generator=g).bfloat16()
    w = (torch.randn(N, K, device=DEV, generator=g) * 0.05).bfloat16()
    bias = torch.randn(N, device=DEV, generator=g)
    pre = torch.full((M, N), float("nan"), dtype=torch.bfloat16, device=DEV)
    h = torch.full((M, N), float("nan"), dtype=torch.bfloat16, device=DEV)
    ops.gemm_ex(a, w, M, N, K, ops.EPI_GELU_BF16, h, bias=bias, aux=pre)
    ref = a.float() @ w.float().t() + bias
    assert torch.isfinite(pre.float()).all() and torch.isfinite(h.float()).all()  # every element written, nothing past the ragged edge read back
    assert frob(pre, ref) <= 3e-3 and frob(h, torch.nn.functional.gelu(ref)) <= 3e-3
    assert torch.equal(h, ops.gemm(a, w, bias, ops.EPI_GELU_BF16))  # same GELU output as the inference epilogue (no aux)
    # dgrad with dGELU: dX[M,N] = (dY[M,K] @ W2[K,N]) * gelu'(pre)   (W2 = an nn.Linear weight [K, N] seen transposed)
    dy = torch.randn(M, K, device=DEV, generator=g).bfloat16()
    w2 = (torch.randn(K, N, device=DEV, generator=g) * 0.05).bfloat16()
    dh = ops.linear_dgrad(dy, w2, aux=pre)
    x = pre.float().requires_grad_(True)
    torch.nn.functional.gelu(x).backward(dy.float() @ w2.float())
    assert dh.shape == (M, N) and frob(dh, x.grad) <= 4e-3


def test_gemm_in_place_residual_epilogue_at_full_size(ops):
    """X += A W^T + b through the in-place residual epilogue (fp32 TMA reduce-add into X) at the fc2 shape of the full model:
    480 output tiles on 148 SMs, so the last round is partial."""
    g = torch.Generator(device=DEV).manual_seed(3)
    M, N, K = 20480, 768, 3072
    a = torch.randn(M, K, device=DEV, generator=g).bfloat16()
    w = (torch.randn(N, K, device=DEV, generator=g) * 0.05).bfloat16()
    b = torch.randn(N, device=DEV, generator=g)
    r = torch.randn(M, N, device=DEV, generator=g)
    x = r.clone()
    ops.gemm(a, w, b, ops.EPI_RESID_F32, residual=x)
    ref = r + b + a.float() @ w.float().t()
    err = ((x - ref).norm() / ref.norm()).item()
    assert err <= 1e-5, err


def test_gemm_identity_property(ops):
    """W = I -> out == A exactly (bf16 in, fp32 accumulate): holds at any size, checked at M = 20480."""
    a = torch.randn(20480, 768, generator=torch.Generator().manual_seed(1)).to(torch.bfloat16).to(DEV)
    w = torch.eye(768, dtype=torch.bfloat16, device=DEV)
    out = ops.gemm(a, w, None, ops.EPI_F32)
    assert torch.equal(out, a.float())


def test_gemm_qkv_head_layout(ops):
    B, T, H = 2, 216, 2
    g = torch.Generator().manual_seed(9)
    a = torch.randn(B * T, 128, generator=g).to(torch.bfloat16)
    w = (0.05 * torch.randn(3 * H * 64, 128, generator=g)).to(torch.bfloat16)
    b = torch.randn(3 * H * 64, generator=g)
    out = ops.gemm(a.to(DEV), w.to(DEV), b.to(DEV), ops.EPI_QKV_HEADS, heads=H, tokens=T)
    ref = (a.float() @ w.float().t() + b).view(B, T, 3, H, 64).permute(2, 0, 3, 1, 4)
    assert out.shape == (3, B, H, T, 64) and frob(out.float(), ref) <= 4e-3


@pytest.mark.parametrize("B,H,N", [(1, 2, 216), (2, 1, 72), (1, 3, 640), (1, 1, 1)])
def test_flash_attention_vs_eager(ops, B, H, N):
    """eager_attention_forward semantics (modeling_videomae.py:196-223), ragged N (KV tail masking) included."""
    g = torch.Generator().manual_seed(N)
    q, k, v = (torch.randn(B, H, N, 64, generator=g).to(torch.bfloat16) for _ in range(3))
    out, lse = ops.flash_attn_fwd(q.to(DEV), k.to(DEV), v.to(DEV), 0.125, return_lse=True)
    s = (q.double() @ k.double().transpose(-1, -2)) * 0.125
    ref = (torch.softmax(s, -1) @ v.double()).transpose(1, 2).reshape(B, N, H * 64)
    assert frob(out.float(), ref) <= 6e-3
    assert (lse.cpu().double() - torch.logsumexp(s, -1)).abs().max() <= 1e-4


def test_flash_attention_rows_sum_to_one_full_size(ops):
    """V = 1 -> out == 1 for any Q,K: softmax rows sum to one.  Checked at the full 20480 tokens."""
    g = torch.Generator().manual_seed(2)
    q = (2 * torch.randn(1, 2, 20480, 64, generator=g)).to(torch.bfloat16).to(DEV)
    k = (2 * torch.randn(1, 2, 20480, 64, generator=g)).to(torch.bfloat16).to(DEV)
    v = torch.ones(1, 2, 20480, 64, dtype=torch.bfloat16, device=DEV)
    out = ops.flash_attn_fwd(q, k, v, 0.125)
    assert (out.float() - 1).abs().max().item() <= 8e-3  # bf16 rounding of P and of the output


def test_patch_embed_vs_oracle(ops):
    cfg = vo.OracleConfig(**ge.SMALL64)
    sd = vo.synthetic_state_dict(cfg, 1234)
    x = vo.synthetic_volume(cfg, 2, 7)
    np.random.seed(0)
    g = OracleMaskGenerator(96, 96, 32, 16, 0.65)
    mask = torch.from_numpy(np.stack([g(), g()]))
    w = sd["videomae.embeddings.patch_embeddings.projection.weight"].reshape(cfg.hidden_size, -1).contiguous()
    b = sd["videomae.embeddings.patch_embeddings.projection.bias"]
    pos = ops.sincos_table(cfg.num_patches, cfg.hidden_size, DEV)
    vol = x[:, :, 0].contiguous().to(DEV)
    full = ops.patch_embed_fwd(vol, w.to(DEV), b.to(DEV), pos)
    # (i) against the fp32 oracle: bf16 operands (8-bit mantissa, what the reference's bf16-autocast Conv3d reads), fp32 accumulate
    assert frob(full, vo.embed(sd, cfg, x, None)) <= 5e-3
    # (ii) against the oracle fed the SAME bf16-rounded operands: only the fp32 summation order is left
    sdr = dict(sd)
    sdr["videomae.embeddings.patch_embeddings.projection.weight"] = sd["videomae.embeddings.patch_embeddings.projection.weight"].bfloat16().float()
    xr = x.bfloat16().float()
    assert frob(full, vo.embed(sdr, cfg, xr, None)) <= 2e-5
    fine = mask.to(torch.uint8).to(DEV)
    _, _, slot, _ = ops.mask_index(fine)
    vis = ops.patch_embed_fwd(vol, w.to(DEV), b.to(DEV), pos, fine, slot, int((~mask[0]).sum()))
    assert frob(vis, vo.embed(sdr, cfg, xr, mask)) <= 2e-5


def test_patch_embed_delta_weight_full_size(ops):
    """weight = delta at voxel (dz,dy,dx) of output channel c -> embedding[n, c] == volume[voxel of patch n] (+pos):
    pins the TMA tile -> K ordering at 512x512x320 without a CPU oracle."""
    vol = torch.rand(1, 320, 512, 512, generator=torch.Generator().manual_seed(4)).to(DEV)
    D = 32
    w = torch.zeros(D, 16, 16, 16)
    taps = [(0, 0, 0), (15, 15, 15), (3, 7, 11), (8, 0, 5)]
    for c, (dz, dy, dx) in enumerate(taps):
        w[c, dz, dy, dx] = 1.0
    pos = torch.zeros(20480, D, device=DEV)
    out = ops.patch_embed_fwd(vol, w.reshape(D, -1).contiguous().to(DEV), torch.zeros(D, device=DEV), pos)
    v5 = vol.view(20, 16, 32, 16, 32, 16)
    for c, (dz, dy, dx) in enumerate(taps):
        want = v5[:, dz, :, dy, :, dx].reshape(-1)
        assert torch.equal(out[0, :, c], want.bfloat16().float())  # exactly the bf16 rounding of the voxel value
    assert out[0, :, len(taps):].abs().max().item() == 0.0


# ---------------------------------------------------------------------------- model level
@pytest.fixture(scope="module")
def small_model(ops):
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining

    cfg = vo.OracleConfig(**ge.SMALL64)
    sd = vo.synthetic_state_dict(cfg, 1234)
    model = B200VideoMAEForPreTraining(ge.hf_config(ge.SMALL64)).to(DEV)
    model.load_state_dict(sd, strict=True)
    return cfg, sd, model


@pytest.mark.parametrize("B", [1, 2])
def test_mim_forward_matches_oracle(small_model, B):
    cfg, sd, model = small_model
    x = vo.synthetic_volume(cfg, B, 7)
    np.random.seed(0)
    g = OracleMaskGenerator(96, 96, 32, 16, 0.65)
    mask = torch.from_numpy(np.stack([g() for _ in range(B)]))
    out = model(x.to(DEV), mask)
    with torch.no_grad():
        loss, logits, _ = vo.pretrain_forward(sd, cfg, x, mask)
    assert out.logits.shape == logits.shape
    assert abs(out.loss.item() - loss.item()) / loss.item() <= 1e-4
    assert frob(out.logits.float(), logits) <= 1e-2 and maxrel(out.logits.float(), logits) <= 2e-2
    # tuple form + device mask with an explicit count (no sync) give the same numbers
    l2, lg2 = model(x.to(DEV), mask.to(DEV), return_dict=False, num_masked=int(mask[0].sum()))
    assert l2.item() == out.loss.item() and torch.equal(lg2, out.logits)


def test_embedding_extraction_matches_oracle(small_model):
    cfg, sd, model = small_model
    x = vo.synthetic_volume(cfg, 2, 21)
    with torch.no_grad():
        emb = model.videomae(x.to(DEV)).last_hidden_state
    with torch.no_grad():
        ref = vo.encoder(sd, cfg, x, None)
    assert emb.shape == ref.shape and emb.dtype == torch.float32
    assert frob(emb, ref) <= 2e-2 and maxrel(emb, ref) <= 5e-2


def test_l1_variant_matches_oracle(small_model):
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining

    cfg, sd, _ = small_model
    model = B200VideoMAEForPreTraining(ge.hf_config(ge.SMALL64), loss_kind="l1").to(DEV)
    model.load_state_dict(sd, strict=True)
    x = vo.synthetic_volume(cfg, 1, 7)
    np.random.seed(1)
    mask = torch.from_numpy(OracleMaskGenerator(96, 96, 32, 16, 0.65)())[None]
    out = model(x.to(DEV), mask)
    with torch.no_grad():
        loss, _, _ = vo.pretrain_forward(sd, cfg, x, mask, loss_kind="l1")
    assert abs(out.loss.item() - loss.item()) / loss.item() <= 1e-3


def test_full_size_embedding_runs_and_is_deterministic(ops):
    """smb-vision-base at 512x512x320: finite, right shape, bit-identical across two runs (no atomics on the path)."""
    from smb_vision_b200.modeling import B200VideoMAEModel

    cfg = vo.OracleConfig()
    torch.manual_seed(0)
    model = B200VideoMAEModel(ge.hf_config({k: getattr(cfg, k) for k in cfg.__dataclass_fields__})).to(DEV)
    x = vo.synthetic_volume(cfg, 1, 7).to(DEV)
    with torch.no_grad():
        a = model(x).last_hidden_state
    with torch.no_grad():
        b = model(x).last_hidden_state
    assert a.shape == (1, 20480, 768) and torch.isfinite(a).all()
    assert torch.equal(a, b)


# ---------------------------------------------------------------------------- training step (gradients)
def _oracle_grads(cfg, sd, x, mask, loss_kind="mse"):
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    loss, _, _ = vo.pretrain_forward(sdg, cfg, x, mask, loss_kind=loss_kind)
    loss.backward()
    return loss.item(), {k: v.grad for k, v in sdg.items()}


@pytest.mark.parametrize("B", [1, 2])
def test_mim_gradients_match_oracle(small_model, B):
    """loss.backward() through the CUDA backward vs autograd over the oracle (SURVEY.md §8c: grads Frobenius-rel <= 2e-2,
    zero-initialised parameters perturbed so their gradients are exercised)."""
    cfg, sd, model = small_model
    x = vo.synthetic_volume(cfg, B, 7)
    np.random.seed(0)
    g = OracleMaskGenerator(96, 96, 32, 16, 0.65)
    mask = torch.from_numpy(np.stack([g() for _ in range(B)]))
    ref_loss, ref = _oracle_grads(cfg, sd, x, mask)
    model.zero_grad(set_to_none=True)
    out = model(x.to(DEV), mask)
    assert out.loss.requires_grad
    out.loss.backward()
    assert abs(out.loss.item() - ref_loss) / ref_loss <= 1e-4
    worst = {}
    for k, p in model.named_parameters():
        assert p.grad is not None, k
        worst[k] = frob(p.grad, ref[k])
    bad = {k: v for k, v in worst.items() if not v <= 2e-2}
    assert not bad, bad


def test_data_parallel_step_single_rank(small_model):
    """DataParallelStep (world 1) == autograd path; gradients live in the flat arena assigned to .grad."""
    from smb_vision_b200.modeling import _prep_mask
    from smb_vision_b200.training import DataParallelStep

    cfg, sd, model = small_model
    x = vo.synthetic_volume(cfg, 1, 7)
    np.random.seed(0)
    mask = torch.from_numpy(OracleMaskGenerator(96, 96, 32, 16, 0.65)())[None]
    _, ref = _oracle_grads(cfg, sd, x, mask)
    dp = DataParallelStep(model)
    vol = model.videomae._volume(x.to(DEV))
    loss, _ = dp.step(vol, _prep_mask(mask, vol.device, None))
    for k, p in model.named_parameters():
        assert p.grad.data_ptr() == dp.arena.views[k].data_ptr()
        assert frob(p.grad, ref[k]) <= 2e-2, k
    model.zero_grad(set_to_none=True)


def test_embedding_runner_matches_direct_call(small_model):
    """EmbeddingRunner (H2D / compute / D2H overlapped on three streams) returns exactly what model.videomae(x) does,
    in order, for a stream longer than its buffer depth."""
    from smb_vision_b200.inference import EmbeddingRunner

    cfg, sd, model = small_model
    vols = [vo.synthetic_volume(cfg, 1, 30 + i).pin_memory() for i in range(5)]
    with torch.no_grad():
        want = [model.videomae(v.to(DEV)).last_hidden_state.cpu() for v in vols]
    got = [e.clone() for e in EmbeddingRunner(model).embed_stream(iter(vols))]
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert torch.equal(g, w)
    # documented lifetime: a yielded (zero-copy) result stays valid while the consumer holds the NEXT one
    prev = None
    for i, e in enumerate(EmbeddingRunner(model).embed_stream(iter(vols))):
        if prev is not None:
            torch.cuda.synchronize()  # everything that could overwrite `prev` has been enqueued and has run
            assert torch.equal(prev, want[i - 1]), i
        prev = e
    # copy=True hands out fresh tensors: collecting the whole stream is safe
    for g, w in zip(list(EmbeddingRunner(model).embed_stream(iter(vols), copy=True)), want):
        assert torch.equal(g, w)


# ---------------------------------------------------------------------------- committed reference fixtures (tests/golden)
def test_mim_matches_reference_golden(small_model, golden_dir):
    """CUDA path vs tests/golden/small64_mim.npz — outputs of the REFERENCE model itself (oracle/make_golden.py imports
    /root/reference/src/models/videomae/modeling_videomae.py): loss, logits, embeddings and selected gradients."""
    cfg, sd, model = small_model
    meta = json.load(open(os.path.join(golden_dir, "small64_mim.json")))
    gold = np.load(os.path.join(golden_dir, "small64_mim.npz"))
    assert meta["config"] == ge.SMALL64
    x = vo.synthetic_volume(cfg, 1, meta["volume_seed"])
    mask = torch.from_numpy(gold["mask"])
    model.zero_grad(set_to_none=True)
    out = model(x.to(DEV), mask)
    out.loss.backward()
    with torch.no_grad():
        emb = model.videomae(x.to(DEV)).last_hidden_state
    assert abs(out.loss.item() - float(gold["loss"])) / float(gold["loss"]) <= 1e-4
    lg, eg = torch.from_numpy(gold["logits"]), torch.from_numpy(gold["embeddings"])
    assert frob(out.logits.float(), lg) <= 1e-2 and maxrel(out.logits.float(), lg) <= 2e-2
    assert frob(emb, eg) <= 2e-2 and maxrel(emb, eg) <= 5e-2
    pairs = {"g_patch_w": "videomae.embeddings.patch_embeddings.projection.weight", "g_mask_token": "mask_token",
             "g_q_bias0": "videomae.encoder.layer.0.attention.attention.q_bias", "g_e2d": "encoder_to_decoder.weight",
             "g_head_b": "decoder.head.bias", "g_fc1_w_l1": "videomae.encoder.layer.1.intermediate.dense.weight"}
    params = dict(model.named_parameters())
    for gk, pk in pairs.items():
        assert frob(params[pk].grad, torch.from_numpy(gold[gk])) <= 2e-2, gk
    norms = np.array([float(params[k].grad.norm()) for k in meta["grad_keys"]])
    assert np.allclose(norms, gold["grad_norms"], rtol=2e-2, atol=1e-9)
    model.zero_grad(set_to_none=True)


# ---------------------------------------------------------------------------- classification head (SURVEY.md §8f rank 1)
CLS = {"single": ("single_label_classification", 3, torch.long), "multi": ("multi_label_classification", 3, torch.float32),
       "regression": ("regression", 1, torch.float32)}


def _cls_model(ptype, n_feat=2):
    from smb_vision_b200.modeling import B200VideoMAEForVideoClassification

    full, n_lab, _ = CLS[ptype]
    cfg = vo.OracleConfig(**ge.SMALL64)
    hc = ge.hf_config(ge.SMALL64)
    hc.num_labels, hc.additional_features_size, hc.problem_type = n_lab, n_feat, full
    model = B200VideoMAEForVideoClassification(hc).to(DEV)
    sd = vo.synthetic_cls_state_dict(cfg, n_lab, n_feat, 1234)
    model.load_state_dict(sd, strict=True)
    return cfg, sd, model


@pytest.mark.parametrize("ptype", list(CLS))
def test_classification_matches_reference_golden(ops, golden_dir, ptype):
    """forward(pixel_values, additional_features, labels) + loss.backward() vs the reference's own outputs
    (VideoMAEForVideoClassification, modeling_videomae.py:917-1023) stored in tests/golden/small64_cls.npz."""
    gold = np.load(os.path.join(golden_dir, "small64_cls.npz"))
    cfg, sd, model = _cls_model(ptype)
    feats = torch.from_numpy(gold["features"])
    labels = torch.from_numpy(gold[f"{ptype}_labels"]).to(CLS[ptype][2])
    x = vo.synthetic_volume(cfg, feats.shape[0], 11)
    out = model(x.to(DEV), additional_features=feats, labels=labels)
    assert out.logits.shape == gold[f"{ptype}_logits"].shape and out.loss.requires_grad
    out.loss.backward()
    ref_loss = float(gold[f"{ptype}_loss"])
    assert abs(out.loss.item() - ref_loss) / abs(ref_loss) <= 2e-3  # the loss IS the model output here (bf16 encoder noise)
    assert maxrel(out.logits, torch.from_numpy(gold[f"{ptype}_logits"])) <= 2e-2
    params = dict(model.named_parameters())
    for gk, pk in {"g_classifier_w": "classifier.weight", "g_classifier_b": "classifier.bias", "g_fc_norm_w": "fc_norm.weight",
                   "g_fc_norm_b": "fc_norm.bias", "g_patch_b": "videomae.embeddings.patch_embeddings.projection.bias",
                   "g_qw0": "videomae.encoder.layer.0.attention.attention.query.weight"}.items():
        assert frob(params[pk].grad, torch.from_numpy(gold[f"{ptype}_{gk}"])) <= 3e-2, gk
    # inference call (no labels) gives the same logits and no loss; tuple form
    with torch.no_grad():
        o2 = model(x.to(DEV), additional_features=feats)
        (lg3,) = model(x.to(DEV), additional_features=feats, return_dict=False)
    assert o2.loss is None and torch.allclose(o2.logits, out.logits, atol=1e-5) and torch.equal(lg3, o2.logits)


def test_classification_all_gradients_match_oracle(ops):
    """every parameter gradient of the classification model vs autograd over the oracle restatement (batch 3, 4 features)."""
    cfg, sd, model = _cls_model("single", n_feat=4)
    B = 3
    x = vo.synthetic_volume(cfg, B, 5)
    feats = torch.randn(B, 4, generator=torch.Generator().manual_seed(3))
    labels = torch.tensor([1, 2, 0])
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    loss, logits = vo.classify_forward(sdg, cfg, x, feats, labels, 3, "single_label_classification")
    loss.backward()
    out = model(x.to(DEV), additional_features=feats.to(DEV), labels=labels.to(DEV))
    (out.loss * 2.0).backward()  # a scaled loss (gradient accumulation) must scale every gradient
    assert abs(out.loss.item() - loss.item()) / loss.item() <= 2e-3
    bad = {k: frob(p.grad, 2.0 * sdg[k].grad) for k, p in model.named_parameters()}
    bad = {k: v for k, v in bad.items() if not v <= 3e-2}
    assert not bad, bad


def test_classification_data_parallel_step_and_errors(ops):
    from smb_vision_b200.training import DataParallelStep

    cfg, sd, model = _cls_model("multi")
    x = vo.synthetic_volume(cfg, 2, 11)
    feats = torch.randn(2, 2, generator=torch.Generator().manual_seed(5))
    labels = torch.tensor([[1.0, 0.0, 1.0], [0.0, 0.0, 1.0]])
    out = model(x.to(DEV), additional_features=feats, labels=labels)
    out.loss.backward()
    ref = {k: p.grad.clone() for k, p in model.named_parameters()}
    dp = DataParallelStep(model)
    vol = model.videomae._volume(x.to(DEV))
    loss, _ = dp.step(vol, feats.to(DEV), labels.to(DEV))
    assert abs(loss.item() - out.loss.item()) <= 1e-6
    for k, p in model.named_parameters():
        assert p.grad.data_ptr() == dp.arena.views[k].data_ptr()
        assert frob(p.grad, ref[k]) <= 1e-3, k
    with pytest.raises(ValueError):  # reference :983-986
        model(x.to(DEV), additional_features=torch.zeros(2, 5))
    with pytest.raises(ValueError):  # reference :181-184
        model(x.repeat(1, 1, 3, 1, 1).to(DEV), additional_features=feats)
    # fine-tuning loop: fused clip + AdamW over the classification model's arena (classifier + fc_norm bucket first)
    from smb_vision_b200.optim import FusedAdamW

    dp2 = DataParallelStep(model, optimizer=FusedAdamW(model, lr=1e-3, max_grad_norm=1.0))
    vol = model.videomae._volume(x.to(DEV))
    ls = [dp2.step(vol, feats.to(DEV), labels.to(DEV))[0].item() for _ in range(4)]
    assert all(np.isfinite(ls)) and ls[-1] < ls[0], ls


def test_cls_head_kernel_alone(ops):
    """smbv_cls_head vs torch fp32 (LayerNorm + Linear + the three losses), forward and every gradient, incl. the
    no-norm branch and the no-feature case."""
    import torch.nn.functional as F

    g = torch.Generator().manual_seed(0)
    for d, Fe, L, B, prob, norm in [(768, 2, 5, 4, 2, True), (128, 0, 1, 3, 1, True), (384, 3, 7, 2, 3, True), (64, 1, 4, 2, 2, False)]:
        N = 37
        pooled = torch.randn(B, d, generator=g) * N
        gamma, beta = 1 + 0.1 * torch.randn(d, generator=g), 0.1 * torch.randn(d, generator=g)
        feats = torch.randn(B, Fe, generator=g) if Fe else None
        W, bias = (0.1 * torch.randn(L, d + Fe, generator=g)).requires_grad_(True), (0.1 * torch.randn(L, generator=g)).requires_grad_(True)
        gam, bet, p = gamma.clone().requires_grad_(norm), beta.clone().requires_grad_(norm), pooled.clone().requires_grad_(True)
        h = p / N
        if norm:
            h = F.layer_norm(h, (d,), gam, bet, 1e-5)
        z = torch.cat([h, feats], -1) if Fe else h
        logits = F.linear(z, W, bias)
        if prob == 2:
            labels = torch.randint(0, L, (B,), generator=g)
            loss = F.cross_entropy(logits, labels)
        elif prob == 1:
            labels = torch.randn(B, L, generator=g)
            loss = F.mse_loss(logits, labels)
        else:
            labels = (torch.rand(B, L, generator=g) > 0.5).float()
            loss = F.binary_cross_entropy_with_logits(logits, labels)
        loss.backward()
        grads = dict(dW=torch.zeros(L, d + Fe, device=DEV), dbias=torch.zeros(L, device=DEV),
                     dgamma=torch.zeros(d, device=DEV) if norm else None, dbeta=torch.zeros(d, device=DEV) if norm else None)
        lo, lg, dp = ops.cls_head(pooled.to(DEV), 1.0 / N, gamma.to(DEV) if norm else None, beta.to(DEV) if norm else None, 1e-5,
                                  None if feats is None else feats.to(DEV), W.detach().to(DEV), bias.detach().to(DEV), labels.to(DEV), prob, grads)
        assert abs(lo.item() - loss.item()) <= 1e-5 * max(1.0, abs(loss.item()))
        assert torch.allclose(lg.cpu(), logits.detach(), atol=1e-4, rtol=1e-4)
        assert frob(grads["dW"], W.grad) <= 1e-4 and frob(grads["dbias"], bias.grad) <= 1e-4
        assert frob(dp, p.grad) <= 1e-4
        if norm:
            assert frob(grads["dgamma"], gam.grad) <= 1e-4 and frob(grads["dbeta"], bet.grad) <= 1e-4
        dx, dxb = ops.broadcast_rows(dp, 9)
        assert torch.equal(dx, dp[:, None, :].expand(B, 9, d)) and torch.equal(dxb, dx.bfloat16())


# ---------------------------------------------------------------------------- operator-level plug-in (SURVEY.md §8b.2)
def test_attention_interface_on_unmodified_upstream_model(ops):
    """The UNMODIFIED transformers VideoMAE (the class src/run_mim.py:19-20 imports) with
    config._attn_implementation = "b200_tcgen05": forward and backward through the registered tcgen05 kernels vs its own sdpa."""
    import transformers

    import smb_vision_b200.attention_interface as ai

    name = ai.register()
    cfg = vo.OracleConfig(**ge.SMALL64)
    sd = vo.synthetic_state_dict(cfg, 1234)
    x = vo.synthetic_volume(cfg, 2, 7).to(DEV)
    np.random.seed(0)
    g = OracleMaskGenerator(96, 96, 32, 16, 0.65)
    mask = torch.from_numpy(np.stack([g() for _ in range(2)])).to(DEV)
    res = {}
    for impl in ("sdpa", name):
        hc = ge.hf_config(ge.SMALL64)
        hc._attn_implementation = impl
        m = transformers.VideoMAEForPreTraining(hc).to(DEV)
        m.load_state_dict(sd, strict=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):  # HF Trainer bf16 (scripts/training/run_mim.sh)
            out = m(x, mask)
        out.loss.backward()
        res[impl] = (out.loss.item(), out.logits.float().detach(),
                     m.videomae.encoder.layer[0].attention.attention.query.weight.grad.clone(),
                     m.videomae.embeddings.patch_embeddings.projection.weight.grad.clone())
    a, b = res["sdpa"], res[name]
    assert abs(a[0] - b[0]) / a[0] <= 1e-4
    assert frob(b[1], a[1]) <= 1e-2
    assert frob(b[2], a[2]) <= 3e-2 and frob(b[3], a[3]) <= 3e-2
    with pytest.raises(Exception):
        z = torch.zeros(1, 1, 8, 48, device=DEV)
        ai.b200_flash_attention(None, z, z, z)  # head_dim 48: not implemented, no fallback


def test_vjepa_step_through_the_attention_plugin(ops):
    """SURVEY.md §8f rank 4 (first slice): the V-JEPA 3D model dispatches its RoPE attention through the same registry
    (reference modeling_vjepa.py:352-370), so the UNMODIFIED upstream VJEPA2Model runs every attention — encoder at
    head_dim 64 on the tcgen05 kernels, predictor at head_dim 32 on the small-head kernels — forward and backward on our
    CUDA path.  One training-style step (predictor output vs target L1, reference src/run_vjepa.py:108-137) vs sdpa."""
    import transformers

    import smb_vision_b200.attention_interface as ai

    name = ai.register()
    res = {}
    g = torch.Generator().manual_seed(0)
    x = torch.rand(2, 64, 1, 64, 64, generator=g).to(DEV)
    N = 4 * 4 * 4
    perm = torch.randperm(N, generator=g)
    ctx = [perm[:40].sort().values[None].repeat(2, 1).to(DEV)]
    tgt = [perm[40:].sort().values[None].repeat(2, 1).to(DEV)]
    for impl in ("sdpa", name):
        c = transformers.VJEPA2Config(patch_size=16, crop_size=64, frames_per_clip=64, tubelet_size=16, hidden_size=128, in_chans=1,
                                      num_attention_heads=2, num_hidden_layers=2, pred_hidden_size=64, pred_num_attention_heads=2,
                                      pred_num_hidden_layers=2, pred_num_mask_tokens=2)
        c._attn_implementation = impl
        torch.manual_seed(7)
        m = transformers.VJEPA2Model(c).to(DEV)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = m(pixel_values_videos=x, context_mask=ctx, target_mask=tgt)
            loss = torch.nn.functional.l1_loss(out.predictor_output.last_hidden_state.float(), out.predictor_output.target_hidden_state.float().detach())
        loss.backward()
        res[impl] = (loss.item(), out.last_hidden_state.float().detach(), m.encoder.layer[0].attention.query.weight.grad.clone(),
                     m.predictor.layer[1].attention.key.weight.grad.clone())
    a, b = res["sdpa"], res[name]
    assert abs(a[0] - b[0]) / a[0] <= 5e-3
    assert frob(b[1], a[1]) <= 1e-2
    assert frob(b[2], a[2]) <= 5e-2 and frob(b[3], a[3]) <= 5e-2


# ---------------------------------------------------------------------------- optimiser step (SURVEY.md §8f rank 2)
def test_adamw_kernel_matches_torch(ops):
    """smbv_sumsq_f32 + smbv_adamw_step vs clip_grad_norm_ + torch.optim.AdamW with Trainer's decay / no-decay groups."""
    import ctypes as C

    from smb_vision_b200._lib import call

    g = torch.Generator().manual_seed(0)
    sizes = [(4096, 0), (64, 1), (12288, 0), (192, 1), (640, 0)]  # (elements, nodecay)
    n = sum(s for s, _ in sizes)
    p0 = torch.randn(n, generator=g)
    ps = [torch.nn.Parameter(t.clone()) for t in p0.split([s for s, _ in sizes])]
    opt = torch.optim.AdamW([{"params": [p for p, (_, nd) in zip(ps, sizes) if not nd], "weight_decay": 0.01},
                             {"params": [p for p, (_, nd) in zip(ps, sizes) if nd], "weight_decay": 0.0}], lr=1e-3)
    p = p0.clone().to(DEV)
    pb = torch.empty(n, dtype=torch.bfloat16, device=DEV)
    m, v = torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    starts = torch.tensor(np.cumsum([0] + [s for s, _ in sizes[:-1]]) // 4, dtype=torch.int32, device=DEV)
    flags = torch.tensor([nd for _, nd in sizes], dtype=torch.uint8, device=DEV)
    ws = torch.empty(int(ops._lib.load().smbv_sumsq_workspace_floats()), device=DEV)
    nsq = torch.zeros(1, device=DEV)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for step in range(1, 6):
        grad = torch.randn(n, generator=g) * (3.0 if step % 2 else 0.001)  # clipped and unclipped steps
        for q, gq in zip(ps, grad.split([s for s, _ in sizes])):
            q.grad = gq.clone()
        tn = torch.nn.utils.clip_grad_norm_(ps, 1.0)
        opt.step()
        gd = grad.to(DEV)
        call("smbv_sumsq_f32", ops._ptr(gd), n, ops._ptr(ws), ops._ptr(nsq), st)
        assert abs(nsq.sqrt().item() - tn.item()) <= 1e-5 * tn.item()
        call("smbv_adamw_step", ops._ptr(p), ops._ptr(pb), ops._ptr(gd), ops._ptr(m), ops._ptr(v), n, ops._ptr(starts), ops._ptr(flags),
             len(sizes), 1e-3, 0.9, 0.999, 1e-8, 0.01, step, ops._ptr(nsq), 1.0, st)
        want = torch.cat([q.detach() for q in ps])
        assert (p.cpu() - want).abs().max().item() <= 2e-6, step
        assert torch.equal(pb, p.bfloat16())


def test_fused_adamw_training_steps_match_torch_adamw(ops):
    """3 optimiser steps of DataParallelStep + FusedAdamW (flat arenas, bf16 operand refresh in the update kernel) vs
    the autograd path + clip_grad_norm_ + torch.optim.AdamW with Trainer's parameter groups, from the same weights."""
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining, _prep_mask
    from smb_vision_b200.optim import FusedAdamW
    from smb_vision_b200.training import DataParallelStep

    cfg = vo.OracleConfig(**ge.SMALL64)
    sd = vo.synthetic_state_dict(cfg, 1234)
    x = vo.synthetic_volume(cfg, 1, 7).to(DEV)
    np.random.seed(0)
    mask = torch.from_numpy(OracleMaskGenerator(96, 96, 32, 16, 0.65)())[None]
    lr = 1e-3  # large enough that three steps move the loss well beyond bf16 noise

    ma = B200VideoMAEForPreTraining(ge.hf_config(ge.SMALL64)).to(DEV)
    ma.load_state_dict(sd, strict=True)
    nd = lambda n: ("bias" in n or "norm" in n)
    opt_a = torch.optim.AdamW([{"params": [p for n, p in ma.named_parameters() if not nd(n)], "weight_decay": 0.01},
                               {"params": [p for n, p in ma.named_parameters() if nd(n)], "weight_decay": 0.0}], lr=lr)
    losses_a = []
    for _ in range(3):
        opt_a.zero_grad(set_to_none=True)
        out = ma(x, mask)
        out.loss.backward()
        torch.nn.utils.clip_grad_norm_(ma.parameters(), 1.0)
        opt_a.step()
        losses_a.append(out.loss.item())

    mb = B200VideoMAEForPreTraining(ge.hf_config(ge.SMALL64)).to(DEV)
    opt_b = FusedAdamW(mb, lr=lr, weight_decay=0.01, max_grad_norm=1.0)  # adopts the parameters into a flat arena
    mb.load_state_dict(sd, strict=True)  # AFTER adoption: the bf16 copies must follow (sync on the next forward)
    keys = set(mb.state_dict().keys())
    assert keys == set(sd.keys())
    dp = DataParallelStep(mb, optimizer=opt_b)
    vol = mb.videomae._volume(x)
    mp = _prep_mask(mask, vol.device, None)
    losses_b = [dp.step(vol, mp)[0].item() for _ in range(3)]
    assert losses_a[0] != losses_a[2]  # the weights really moved
    for a, b in zip(losses_a, losses_b):
        assert abs(a - b) / a <= 1e-4, (losses_a, losses_b)
    pa, pb = dict(ma.named_parameters()), dict(mb.named_parameters())
    worst = max(frob(pb[k].detach(), pa[k].detach()) for k in pa)
    assert worst <= 2e-3, worst  # Adam's update is sign-like at step 1: tiny gradient noise moves single elements by ~lr
    # resume: optimiser state round-trips through state_dict
    st = opt_b.state_dict()
    opt_c = FusedAdamW(mb, lr=lr)
    opt_c.load_state_dict(st)
    assert opt_c.steps == 3 and torch.equal(opt_c.exp_avg, opt_b.exp_avg) and torch.equal(opt_c.exp_avg_sq, opt_b.exp_avg_sq)


# ---------------------------------------------------------------------------- data entry points (rows a1/a2, §8f rank 2)
def test_product_mask_generator_device_batch(ops, golden_dir):
    """MaskGenerator.device_batch: coarse cells from numpy's global RNG (reference stream), upsample + index lists on the
    GPU; equals the reference masks index for index, no host sync needed for the counts."""
    from smb_vision_b200.data import MaskGenerator

    np.random.seed(0)
    g = MaskGenerator(512, 320, 32, 16, 0.65)
    fine, vis, msk, slot, n_vis, n_mask = g.device_batch(2, DEV)
    np.random.seed(0)
    o = OracleMaskGenerator(512, 320, 32, 16, 0.65)
    want = np.stack([o(), o()])
    assert np.array_equal(fine.cpu().numpy().astype(bool), want)
    assert (n_vis, n_mask) == (7168, 13312)
    for b in range(2):
        assert np.array_equal(msk[b, :n_mask].cpu().numpy(), np.nonzero(want[b])[0])
        assert np.array_equal(vis[b, :n_vis].cpu().numpy(), np.nonzero(~want[b])[0])


@pytest.mark.parametrize("shape,img,depth,dtype", [((40, 52, 30), 64, 32, "i16"), ((70, 90, 50), 64, 32, "f32"), ((64, 64, 32), 64, 32, "i16"),
                                                   ((33, 97, 31), 48, 48, "f32"), ((101, 20, 77), 32, 64, "i16")])
def test_prepare_volume_matches_oracle_bit_exact(ops, shape, img, depth, dtype):
    """scale-intensity + symmetric pad + centre crop + permute in one kernel == the numpy restatement, bit for bit
    (padding, cropping and both at once; odd sizes; fp32 and int16 sources)."""
    from oracle import preprocess_oracle as po
    from smb_vision_b200.data import VolumePreprocessor

    rng = np.random.default_rng(1)
    raw = rng.integers(-1500, 2500, size=shape).astype(np.int16)
    if dtype == "f32":
        raw = (raw.astype(np.float32) + rng.random(shape, dtype=np.float32))
    want = po.prepare_volume(raw, img, depth)
    got = VolumePreprocessor(img, depth, device=DEV)(torch.from_numpy(raw)[None])
    assert got.shape == (depth, 1, img, img) and got.dtype == torch.float32
    assert np.array_equal(got.cpu().numpy(), want)


def test_prepare_volume_full_size_properties(ops):
    """512x512x320 from an int16 CT-like source: identity geometry (out[z,0,x,y] == f(src[x,y,z])), range [0,1],
    and the prepared batch feeds the model directly."""
    from smb_vision_b200.data import VolumePreprocessor

    g = torch.Generator().manual_seed(0)
    raw = torch.randint(-1200, 1200, (512, 512, 320), generator=g, dtype=torch.int16)
    pp = VolumePreprocessor(512, 320, device=DEV)
    out = pp.batch([raw.pin_memory()])
    assert out.shape == (1, 320, 1, 512, 512) and 0.0 <= out.min().item() and out.max().item() <= 1.0
    idx = torch.randint(0, 320, (64, 3), generator=g)
    for z, x, y in idx.tolist():
        x, y = x % 512 + 100, y % 512 + 50
        want = min(max((float(raw[x, y, z]) + 1000.0) / 2000.0, 0.0), 1.0)
        assert abs(out[0, z, 0, x, y].item() - want) <= 1e-6


# ---------------------------------------------------------------------------- BASELINE configs[0]: the tiny config (head_dim 16)
@pytest.mark.parametrize("B,H,N,hd", [(1, 4, 72, 16), (2, 2, 216, 16), (1, 3, 50, 32), (2, 1, 7, 8), (1, 2, 300, 32)])
def test_small_head_attention_vs_eager(ops, B, H, N, hd):
    """smbv_attn_small_fwd/bwd (token-major fused QKV) vs eager_attention_forward in fp32 (reference :196-223), fwd + grads."""
    g = torch.Generator().manual_seed(B * 1000 + N)
    d = H * hd
    qkv = torch.randn(B, N, 3 * d, generator=g).bfloat16()
    dout = torch.randn(B, N, d, generator=g).bfloat16()
    scale = hd ** -0.5
    x = qkv.float().requires_grad_(True)
    q, k, v = (t.reshape(B, N, H, hd).transpose(1, 2) for t in x.split(d, dim=-1))
    p = torch.softmax(q @ k.transpose(-1, -2) * scale, dim=-1)
    ref = (p @ v).transpose(1, 2).reshape(B, N, d)
    ref.backward(dout.float())
    out, lse = ops.attn_small_fwd(qkv.to(DEV), H, scale, return_lse=True)
    assert frob(out.float(), ref.detach()) <= 5e-3
    lse_ref = torch.logsumexp(q.detach() @ k.detach().transpose(-1, -2) * scale, dim=-1)
    assert (lse.cpu() - lse_ref).abs().max().item() <= 1e-4
    dqkv = ops.attn_small_bwd(qkv.to(DEV), out, dout.to(DEV), lse, H, scale)
    assert frob(dqkv.float(), x.grad) <= 1e-2
    assert torch.equal(dqkv, ops.attn_small_bwd(qkv.to(DEV), out, dout.to(DEV), lse, H, scale))  # deterministic


def test_tiny_config_matches_reference_golden(ops, golden_dir):
    """BASELINE.json configs[0] — tiny 3D ViT MIM forward + loss on the 96^3 volume, patch 16, mask_patch 32, ratio 0.65 —
    on the GPU against the REFERENCE's own outputs (tests/golden/tiny_mim.npz): loss, logits, embeddings, gradients."""
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining

    meta = json.load(open(os.path.join(golden_dir, "tiny_mim.json")))
    gold = np.load(os.path.join(golden_dir, "tiny_mim.npz"))
    cfg = vo.OracleConfig(**meta["config"])
    sd = vo.synthetic_state_dict(cfg, meta["weight_seed"])
    model = B200VideoMAEForPreTraining(ge.hf_config(meta["config"])).to(DEV)
    model.load_state_dict(sd, strict=True)
    x = vo.synthetic_volume(cfg, 1, meta["volume_seed"])
    mask = torch.from_numpy(gold["mask"])
    out = model(x.to(DEV), mask)
    out.loss.backward()
    with torch.no_grad():
        emb = model.videomae(x.to(DEV)).last_hidden_state
    assert abs(out.loss.item() - float(gold["loss"])) / float(gold["loss"]) <= 1e-4
    lg, eg = torch.from_numpy(gold["logits"]), torch.from_numpy(gold["embeddings"])
    assert frob(out.logits.float(), lg) <= 1e-2 and maxrel(out.logits.float(), lg) <= 2e-2
    assert frob(emb, eg) <= 2e-2 and maxrel(emb, eg) <= 5e-2
    params = dict(model.named_parameters())
    pairs = {"g_patch_w": "videomae.embeddings.patch_embeddings.projection.weight", "g_mask_token": "mask_token",
             "g_q_bias0": "videomae.encoder.layer.0.attention.attention.q_bias", "g_e2d": "encoder_to_decoder.weight",
             "g_head_b": "decoder.head.bias", "g_fc1_w_l1": "videomae.encoder.layer.1.intermediate.dense.weight"}
    for gk, pk in pairs.items():
        assert frob(params[pk].grad, torch.from_numpy(gold[gk])) <= 2e-2, gk
    norms = np.array([float(params[k].grad.norm()) for k in meta["grad_keys"]])
    assert np.allclose(norms, gold["grad_norms"], rtol=2e-2, atol=1e-9)


def test_tiny_config_classification_matches_reference_golden(ops, golden_dir):
    from smb_vision_b200.modeling import B200VideoMAEForVideoClassification

    gold = np.load(os.path.join(golden_dir, "tiny_cls.npz"))
    cfg = vo.OracleConfig(**vo.TINY)
    hc = ge.hf_config(vo.TINY)
    hc.num_labels, hc.additional_features_size, hc.problem_type = 3, 2, "single_label_classification"
    model = B200VideoMAEForVideoClassification(hc).to(DEV)
    model.load_state_dict(vo.synthetic_cls_state_dict(cfg, 3, 2, 1234), strict=True)
    feats, labels = torch.from_numpy(gold["features"]), torch.from_numpy(gold["single_labels"]).long()
    out = model(vo.synthetic_volume(cfg, 2, 11).to(DEV), additional_features=feats, labels=labels)
    out.loss.backward()
    assert abs(out.loss.item() - float(gold["single_loss"])) / float(gold["single_loss"]) <= 2e-3
    assert maxrel(out.logits, torch.from_numpy(gold["single_logits"])) <= 2e-2
    params = dict(model.named_parameters())
    for gk, pk in {"g_classifier_w": "classifier.weight", "g_fc_norm_w": "fc_norm.weight",
                   "g_qw0": "videomae.encoder.layer.0.attention.attention.query.weight"}.items():
        assert frob(params[pk].grad, torch.from_numpy(gold[f"single_{gk}"])) <= 3e-2, gk


def test_full_size_training_step_properties(ops):
    """smb-vision-base MIM step at 512x512x320 (BASELINE configs[2]): finite decreasing loss over optimiser steps, every
    parameter receives a finite gradient, the fused clip brings the global norm to max_grad_norm, and scaling the loss by 2
    scales the gradients by 2 (linearity of the hand-scheduled backward)."""
    from smb_vision_b200.data import MaskGenerator
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining
    from smb_vision_b200.optim import FusedAdamW
    from smb_vision_b200.training import DataParallelStep, GradArena, mim_backward, mim_forward_train

    cfg = vo.OracleConfig()
    torch.manual_seed(0)
    model = B200VideoMAEForPreTraining(ge.hf_config({k: getattr(cfg, k) for k in cfg.__dataclass_fields__})).to(DEV).train()
    vol = model.videomae._volume(vo.synthetic_volume(cfg, 1, 7).to(DEV))
    np.random.seed(0)
    mp = MaskGenerator(512, 320, 32, 16, 0.65).device_batch(1, DEV)
    assert (mp[4], mp[5]) == (7168, 13312)
    with torch.no_grad():
        a1, a2 = GradArena(model, DEV), GradArena(model, DEV)
        loss, logits, dlogits, S = mim_forward_train(model, vol, mp)
        d2 = dlogits * 2
        mim_backward(model, S, dlogits, a1)
        mim_backward(model, S, d2, a2)
    assert logits.shape == (1, 13312, 4096) and torch.isfinite(loss) and torch.isfinite(a1.flat).all()
    assert frob(a2.flat, 2 * a1.flat) <= 1e-4
    zero = [k for k, t in a1.views.items() if float(t.abs().max()) == 0.0]
    assert zero == ["mask_token"] or not zero, zero  # mask_token is zero-initialised but its GRADIENT is not zero
    opt = FusedAdamW(model, lr=1e-3, max_grad_norm=1.0)
    dp = DataParallelStep(model, optimizer=opt)
    losses = [dp.step(vol, mp)[0].item() for _ in range(4)]
    assert all(np.isfinite(losses)) and losses[-1] < losses[0]
    assert float(opt.grad_norm()) > 0


@pytest.mark.parametrize("deterministic", [False, True])
@pytest.mark.parametrize("B,H,N", [(2, 2, 216), (3, 1, 130), (4, 12, 1960), (1, 3, 20000)])
def test_flash_attention_backward_batched_vs_eager(ops, B, H, N, deterministic):
    """whole-batch backward launch (4-D dO tensor map) vs autograd over eager_attention_forward in fp32; (4,12,1960) is the
    classification fine-tuning shape of BASELINE configs[3] (224x224x160, batch 4); (1,3,20000) = 471 (key block, head)
    units on 148 SMs: the fused kernel splits its partial last wave by query range (ragged N).  Both modes: the fused one-pass
    kernel (default; dQ summed across key blocks by fp32 bulk reductions: dK / dV bit-identical run to run, dQ up to fp32
    summation order) and the deterministic two-kernel path (everything bit-identical)."""
    g = torch.Generator(device=DEV).manual_seed(N)
    q, k, v = (torch.randn(B, H, N, 64, device=DEV, generator=g).bfloat16() for _ in range(3))
    dout = torch.randn(B, N, H * 64, device=DEV, generator=g).bfloat16()
    out, lse = ops.flash_attn_fwd(q, k, v, 0.125, return_lse=True)
    dq, dk, dv = ops.flash_attn_bwd(q, k, v, out, dout, lse, 0.125, deterministic=deterministic)
    if N <= 2000:
        qf, kf, vf = (t.float().requires_grad_(True) for t in (q, k, v))
        p = torch.softmax(qf @ kf.transpose(-1, -2) * 0.125, dim=-1)
        ref = (p @ vf).transpose(1, 2).reshape(B, N, H * 64)
        ref.backward(dout.float())
        assert frob(out.float(), ref.detach()) <= 5e-3
        want = (qf.grad, kf.grad, vf.grad)
    else:  # fp32 autograd needs 3 x N^2 floats per head: check head by head in fp64 on a slice of the rows instead
        want = None
        qd, kd, vd, dod = q[0].double(), k[0].double(), v[0].double(), dout[0].double().reshape(N, H, 64).transpose(0, 1)
        p = torch.softmax(qd @ kd.transpose(-1, -2) * 0.125, dim=-1)          # [H, N, N] fp64 = 9.6 GB at H=3
        # forward at this shape: 234 query-tile pairs on 148 SMs -> the 86 units of the last wave are split 5-way by key range
        assert frob(out[0].double().reshape(N, H, 64).transpose(0, 1), p @ vd) <= 5e-3
        assert (lse[0].double() - torch.logsumexp(qd @ kd.transpose(-1, -2) * 0.125, dim=-1)).abs().max().item() <= 2e-3
        dvr = p.transpose(-1, -2) @ dod
        dp = dod @ vd.transpose(-1, -2)
        ds = p * (dp - (dp * p).sum(-1, keepdim=True)) * 0.125
        want = ((ds @ kd)[None], (ds.transpose(-1, -2) @ qd)[None], dvr[None])
        del p, dp, ds
    assert frob(dq.float(), want[0]) <= 2e-2 and frob(dk.float(), want[1]) <= 2e-2 and frob(dv.float(), want[2]) <= 2e-2
    dq2, dk2, dv2 = ops.flash_attn_bwd(q, k, v, out, dout, lse, 0.125, deterministic=deterministic)
    assert torch.equal(dk, dk2) and torch.equal(dv, dv2)
    if deterministic:
        assert torch.equal(dq, dq2)
    else:  # equal up to the order of the fp32 reductions (then one bf16 rounding)
        assert frob(dq2.float(), dq.float()) <= 1e-3
        d3 = ops.flash_attn_bwd(q, k, v, out, dout, lse, 0.125, deterministic=True)
        assert frob(dq.float(), d3[0].float()) <= 4e-3 and frob(dk.float(), d3[1].float()) <= 2e-3 and frob(dv.float(), d3[2].float()) <= 2e-3


def test_config_variants_qkv_bias_off_and_final_layernorm(ops):
    """VideoMAEConfig variants the reference model supports: qkv_bias=False (no q/v bias parameters, reference :242-251) and
    use_mean_pooling=False (final encoder LayerNorm, :517-520): embeddings, MIM forward and every gradient vs the oracle."""
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining

    np.random.seed(0)
    mask = torch.from_numpy(OracleMaskGenerator(96, 96, 32, 16, 0.65)())[None]
    for variant, train_ok in ((dict(qkv_bias=False), True), (dict(qkv_bias=False, use_mean_pooling=False), True)):
        cfgd = dict(ge.SMALL64, **variant)
        cfg = vo.OracleConfig(**cfgd)
        sd = vo.synthetic_state_dict(cfg, 1234)
        model = B200VideoMAEForPreTraining(ge.hf_config(cfgd)).to(DEV)
        model.load_state_dict(sd, strict=True)
        x = vo.synthetic_volume(cfg, 1, 7)
        with torch.no_grad():
            out = model(x.to(DEV), mask)
            emb = model.videomae(x.to(DEV)).last_hidden_state
            loss, logits, _ = vo.pretrain_forward(sd, cfg, x, mask)
            emb_ref = vo.encoder(sd, cfg, x, None)
        assert abs(out.loss.item() - loss.item()) / loss.item() <= 1e-4
        assert frob(out.logits.float(), logits) <= 1e-2 and frob(emb, emb_ref) <= 2e-2
        if train_ok:
            ref_loss, ref = _oracle_grads(cfg, sd, x, mask)
            model(x.to(DEV), mask).loss.backward()
            bad = {k: frob(p.grad, ref[k]) for k, p in model.named_parameters()}
            bad = {k: v for k, v in bad.items() if not v <= 2e-2}
            assert not bad, bad
        else:
            with pytest.raises(NotImplementedError):
                model(x.to(DEV), mask).loss.backward()


# ---------------------------------------------------------------------------- round-2 additions
def test_cuda_graph_step_equals_eager_step(small_model):
    """DataParallelStep(cuda_graph=True): forward + backward replayed from a CUDA graph, optimiser step outside it.  Four steps
    with a DIFFERENT volume and mask every step (the inputs go through the static buffers) give the eager path's losses and
    parameters (up to the fp32 summation order of dQ in the fused attention backward)."""
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining, _prep_mask
    from smb_vision_b200.optim import FusedAdamW
    from smb_vision_b200.training import DataParallelStep

    cfg, sd, _ = small_model
    vols = [vo.synthetic_volume(cfg, 2, 20 + i) for i in range(4)]
    np.random.seed(5)
    gen = OracleMaskGenerator(96, 96, 32, 16, 0.65)
    masks = [torch.from_numpy(np.stack([gen(), gen()])) for _ in range(4)]

    def run(graph):
        m = B200VideoMAEForPreTraining(ge.hf_config(ge.SMALL64)).to(DEV)
        opt = FusedAdamW(m, lr=1e-3, weight_decay=0.01, max_grad_norm=1.0)
        m.load_state_dict(sd, strict=True)
        dp = DataParallelStep(m, optimizer=opt, cuda_graph=graph)
        losses = []
        for x, mk in zip(vols, masks):
            vol = m.videomae._volume(x.to(DEV))
            loss, logits = dp.step(vol, _prep_mask(mk, vol.device, None))
            losses.append(loss.item())  # (static tensor in graph mode: read before the next step)
        assert dp.cuda_graph == graph and (len(dp._graphs) == 1) == graph
        return losses, {k: p.detach().clone() for k, p in m.named_parameters()}

    le, pe = run(False)
    lg, pg = run(True)
    assert len(set(le)) == 4  # different inputs, moving weights
    for a, b in zip(le, lg):
        assert abs(a - b) / a <= 1e-4, (le, lg)
    worst = max(frob(pg[k], pe[k]) for k in pe)
    assert worst <= 2e-3, worst


def test_torch_fused_optimizer_does_not_train_on_stale_operands(small_model):
    """`torch.optim.AdamW(fused=True)` (HF Trainer's default on torch >= 2.8) updates parameters WITHOUT bumping their version
    counters; the cached bf16 operands must still follow.  Three steps of `model(...).loss.backward()` + fused AdamW must give
    the losses of the same loop with the unfused optimiser (with and without a ParamArena behind the parameters)."""
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining
    from smb_vision_b200.training import ParamArena

    cfg, sd, _ = small_model
    x = vo.synthetic_volume(cfg, 1, 7).to(DEV)
    np.random.seed(0)
    mask = torch.from_numpy(OracleMaskGenerator(96, 96, 32, 16, 0.65)())[None]

    def run(fused, arena):
        m = B200VideoMAEForPreTraining(ge.hf_config(ge.SMALL64)).to(DEV)
        m.load_state_dict(sd, strict=True)
        if arena:
            ParamArena(m)
        opt = torch.optim.AdamW(m.parameters(), lr=2e-3, weight_decay=0.0, fused=fused, foreach=False if fused else None)
        losses = []
        for _ in range(4):
            opt.zero_grad(set_to_none=True)
            out = m(x, mask)
            out.loss.backward()
            opt.step()
            losses.append(out.loss.item())
        return losses

    ref = run(False, False)
    assert ref[0] - ref[3] > 1e-3  # the weights really move the loss
    for fused, arena in ((True, False), (True, True), (False, True)):
        got = run(fused, arena)
        for a, b in zip(ref, got):
            assert abs(a - b) / a <= 2e-4, (fused, arena, ref, got)


def test_encoder_forward_is_differentiable(small_model):
    """`model.videomae(x[, mask]).last_hidden_state` under enabled grad carries gradients to every encoder parameter
    (reference VideoMAEModel.forward under autograd, :537-658) — a user fine-tuning through `.videomae` must not get zeros."""
    cfg, sd, model = small_model
    x = vo.synthetic_volume(cfg, 2, 9)
    g = torch.randn(2, 216, cfg.hidden_size, generator=torch.Generator().manual_seed(1))
    np.random.seed(3)
    gen = OracleMaskGenerator(96, 96, 32, 16, 0.65)
    mask = torch.from_numpy(np.stack([gen(), gen()]))
    for m_ in (None, mask):
        gg = g if m_ is None else g[:, :72]
        sdr, xr = autocast_operands(sd, x)
        sdg = {k: v.clone().requires_grad_(True) for k, v in sdr.items() if k.startswith("videomae.")}
        (vo.encoder(sdg, cfg, xr, m_) * gg).sum().backward()
        model.zero_grad(set_to_none=True)
        emb = model.videomae(x.to(DEV), m_).last_hidden_state
        assert emb.requires_grad
        (emb * gg.to(DEV)).sum().backward()
        bad = {k: frob(p.grad, sdg["videomae." + k].grad) for k, p in model.videomae.named_parameters()}
        bad = {k: v for k, v in bad.items() if not v <= grad_tol(k, 2e-2)}
        assert not bad, bad
    with torch.no_grad():
        assert not model.videomae(x.to(DEV)).last_hidden_state.requires_grad
    model.zero_grad(set_to_none=True)


def test_upstream_gradient_scale_is_applied_in_fp32_and_backward_is_repeatable(small_model):
    """(loss / 3).backward() (gradient accumulation): every gradient = oracle / 3 to fp32 accuracy of the factor (a bf16-rounded
    1/3 would be 0.2 % off), and a second backward through the retained graph gives the same gradients again (the saved
    dlogits are not mutated)."""
    cfg, sd, model = small_model
    x = vo.synthetic_volume(cfg, 1, 7)
    np.random.seed(0)
    mask = torch.from_numpy(OracleMaskGenerator(96, 96, 32, 16, 0.65)())[None]
    model.zero_grad(set_to_none=True)
    out = model(x.to(DEV), mask)
    out.loss.backward(retain_graph=True)
    g1 = {k: p.grad.clone() for k, p in model.named_parameters()}
    model.zero_grad(set_to_none=True)
    (out.loss / 3.0).backward()
    for k, p in model.named_parameters():
        want = g1[k] / 3.0
        assert (p.grad - want).abs().max().item() <= 1e-6 * want.abs().max().item() + 1e-12, k
    model.zero_grad(set_to_none=True)


def test_classification_cls_row_head_trains(ops):
    """use_mean_pooling=False (reference :976-977: final encoder LayerNorm, first token's row, no fc_norm): forward and every
    gradient vs autograd over the oracle."""
    from smb_vision_b200.modeling import B200VideoMAEForVideoClassification

    cfgd = dict(ge.SMALL64, use_mean_pooling=False)
    cfg = vo.OracleConfig(**cfgd)
    hc = ge.hf_config(cfgd)
    hc.num_labels, hc.additional_features_size = 3, 2
    sd = {k: v for k, v in vo.synthetic_state_dict(cfg, 1234).items() if k.startswith("videomae.")}
    gsd = torch.Generator().manual_seed(2)
    sd["classifier.weight"] = 0.05 * torch.randn(3, cfg.hidden_size + 2, generator=gsd)
    sd["classifier.bias"] = 0.02 * torch.randn(3, generator=gsd)
    model = B200VideoMAEForVideoClassification(hc).to(DEV)
    assert model.fc_norm is None and model.videomae.layernorm is not None
    model.load_state_dict(sd, strict=True)
    B = 2
    x = vo.synthetic_volume(cfg, B, 5)
    feats = torch.randn(B, 2, generator=gsd)
    labels = torch.tensor([2, 0])
    sdr, xr = autocast_operands(sd, x)
    sdg = {k: v.clone().requires_grad_(True) for k, v in sdr.items()}
    loss, logits = vo.classify_forward(sdg, cfg, xr, feats, labels, 3, "single_label_classification")
    loss.backward()
    out = model(x.to(DEV), additional_features=feats.to(DEV), labels=labels.to(DEV))
    out.loss.backward()
    assert abs(out.loss.item() - loss.item()) / loss.item() <= 2e-3 and frob(out.logits, logits.detach()) <= 2e-2
    bad = {k: frob(p.grad, sdg[k].grad) for k, p in model.named_parameters()}
    bad = {k: v for k, v in bad.items() if not v <= grad_tol(k, 3e-2)}
    assert not bad, bad


def test_fused_adamw_leaves_frozen_parameters_alone(ops):
    """requires_grad=False parameters (a frozen patch embedding under a trained model) are neither updated nor decayed."""
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining, _prep_mask
    from smb_vision_b200.optim import FusedAdamW
    from smb_vision_b200.training import DataParallelStep

    cfg = vo.OracleConfig(**ge.SMALL64)
    model = B200VideoMAEForPreTraining(ge.hf_config(ge.SMALL64)).to(DEV)
    model.load_state_dict(vo.synthetic_state_dict(cfg, 1234), strict=True)
    frozen = ["videomae.embeddings.patch_embeddings.projection.weight", "decoder.norm.weight"]
    for k, p in model.named_parameters():
        if k in frozen:
            p.requires_grad = False
    before = {k: p.detach().clone() for k, p in model.named_parameters()}
    dp = DataParallelStep(model, optimizer=FusedAdamW(model, lr=1e-2, weight_decay=0.1))
    x = vo.synthetic_volume(cfg, 1, 7).to(DEV)
    np.random.seed(0)
    mask = torch.from_numpy(OracleMaskGenerator(96, 96, 32, 16, 0.65)())[None]
    vol = model.videomae._volume(x)
    dp.step(vol, _prep_mask(mask, vol.device, None))
    dp.step(vol, _prep_mask(mask, vol.device, None))
    for k, p in model.named_parameters():
        if k in frozen:
            assert torch.equal(p.detach(), before[k]), k
        else:
            assert not torch.equal(p.detach(), before[k]), k


def test_fused_adamw_clip_norm_ignores_frozen_parameters(ops):
    """With a frozen patch embedding and decoder head, the global norm FusedAdamW clips by is clip_grad_norm_ over the
    trainable parameters' gradients (a frozen parameter has no .grad under torch), although the native backward writes a
    gradient for every parameter.  Control: the norm over the whole gradient arena, frozen gradients included (what the
    optimiser computed before it zeroed them), is off by far more than the bound."""
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining, _prep_mask
    from smb_vision_b200.optim import FusedAdamW
    from smb_vision_b200.training import DataParallelStep

    cfg = vo.OracleConfig(**ge.SMALL64)
    model = B200VideoMAEForPreTraining(ge.hf_config(ge.SMALL64)).to(DEV)
    model.load_state_dict(vo.synthetic_state_dict(cfg, 1234), strict=True)
    # the patch embedding's gradient is small in this model, the decoder head's is not: freeze both
    frozen = ["videomae.embeddings.patch_embeddings.projection.weight", "decoder.head.weight"]
    for k in frozen:
        model.get_parameter(k).requires_grad = False
    opt = FusedAdamW(model, lr=1e-3)
    dp = DataParallelStep(model, optimizer=opt)
    x = vo.synthetic_volume(cfg, 1, 7).to(DEV)
    np.random.seed(0)
    mask = torch.from_numpy(OracleMaskGenerator(96, 96, 32, 16, 0.65)())[None]
    vol = model.videomae._volume(x)
    # the frozen weights' gradients as the backward writes them (before the optimiser step)
    dp._fwd_bwd(vol, _prep_mask(mask, vol.device, None))
    frozen_sq = sum(dp.arena.g(k).double().square().sum().item() for k in frozen)
    dp.step(vol, _prep_mask(mask, vol.device, None))
    trainable = []
    for k, p in model.named_parameters():
        if p.requires_grad:
            trainable.append(torch.nn.Parameter(torch.empty_like(p)))
            trainable[-1].grad = dp.arena.g(k).clone()
    want = torch.nn.utils.clip_grad_norm_(trainable, float("inf")).item()
    got = opt.grad_norm().item()
    whole = (want ** 2 + frozen_sq) ** 0.5
    print(f"clip norm with frozen parameters: {got:.6g}, clip_grad_norm_ {want:.6g}, rel {abs(got - want) / want:.2e} (bound 1e-6); "
          f"norm including the frozen gradients {whole:.6g} (rel {abs(whole - want) / want:.2e})")
    assert frozen_sq > 0 and abs(got - want) <= 1e-6 * want  # measured 1.2e-7 on B200 (1000 W)
    assert abs(whole - want) >= 100 * 1e-6 * want


def test_whole_model_reduced_precision_mode(ops, tmp_path):
    """`from_pretrained(..., torch_dtype=torch.bfloat16)` (run_inspect.py:106-111): weights held in bf16, outputs returned in
    bf16, numbers within the embedding tolerance of the fp32 oracle evaluated on the bf16-rounded weights."""
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining, B200VideoMAEModel

    cfg = vo.OracleConfig(**ge.SMALL64)
    sd = vo.synthetic_state_dict(cfg, 1234)
    m = B200VideoMAEForPreTraining(ge.hf_config(ge.SMALL64))
    m.load_state_dict(sd, strict=True)
    m.save_pretrained(tmp_path / "ck")
    enc = B200VideoMAEModel.from_pretrained(tmp_path / "ck", torch_dtype=torch.bfloat16, attn_implementation="flash_attention_2").to(DEV)
    x = vo.synthetic_volume(cfg, 1, 21)
    with torch.no_grad():
        emb = enc(x.bfloat16().to(DEV)).last_hidden_state  # bf16 volume in, like a model.to(bfloat16) caller passes
    assert emb.dtype == torch.bfloat16
    sdb = {k: v.bfloat16().float() for k, v in sd.items()}
    with torch.no_grad():
        ref = vo.encoder(sdb, cfg, x.bfloat16().float(), None)
    assert frob(emb.float(), ref) <= 2e-2 and maxrel(emb.float(), ref) <= 5e-2


@pytest.mark.parametrize("B,loss_kind", [(1, "l1"), (2, "mse")])
def test_simmim_style_matches_oracle(ops, B, loss_kind):
    """North-star variant (mim_style='simmim'): select(mask, mask_token, emb) + pos fused into the patch-embed epilogue
    (semantics of src/models/dinov2/modeling_dinov2.py:104-107), encoder / decoder over all N tokens, head + loss on the masked rows.
    Forward (loss, logits) and EVERY parameter gradient vs autograd over oracle.pretrain_forward_simmim."""
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining

    cfg = vo.OracleConfig(**ge.SMALL64)
    sd = vo.synthetic_state_dict(cfg, 1234)
    sd["videomae.embeddings.mask_token"] = 0.3 * torch.randn(1, 1, cfg.hidden_size, generator=torch.Generator().manual_seed(9))
    model = B200VideoMAEForPreTraining(ge.hf_config(ge.SMALL64), loss_kind=loss_kind, mim_style="simmim").to(DEV)
    model.load_state_dict(sd, strict=True)
    x = vo.synthetic_volume(cfg, B, 7)
    np.random.seed(2)
    g = OracleMaskGenerator(96, 96, 32, 16, 0.65)
    mask = torch.from_numpy(np.stack([g() for _ in range(B)]))
    # the epilogue alone: blended embeddings == torch.where(mask, mask_token, emb) + pos
    pk = model.videomae.packed()
    fine = mask.to(torch.uint8).to(DEV)
    pos = model.videomae.pos_table(cfg.hidden_size, torch.device(DEV))
    E = ops.patch_embed_select_fwd(x[:, :, 0].contiguous().to(DEV), pk["wpe"], pk["bpe"], pos, fine, pk["mask_token"])
    Eref = vo.embed(sd, cfg, x, None) - vo.sinusoid_table(cfg.num_patches, cfg.hidden_size)
    Eref = torch.where(mask.unsqueeze(-1), sd["videomae.embeddings.mask_token"], Eref) + vo.sinusoid_table(cfg.num_patches, cfg.hidden_size)
    assert frob(E, Eref) <= 2e-3
    assert torch.equal(E.cpu()[mask], (sd["videomae.embeddings.mask_token"].reshape(-1) + vo.sinusoid_table(cfg.num_patches, cfg.hidden_size)[0])[None].expand(B, -1, -1)[mask])
    # model level
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    loss, logits, _ = vo.pretrain_forward_simmim(sdg, cfg, x, mask, loss_kind=loss_kind)
    loss.backward()
    with torch.no_grad():
        out0 = model(x.to(DEV), mask)
    out = model(x.to(DEV), mask)
    out.loss.backward()
    assert out0.loss.item() == out.loss.item() and torch.equal(out0.logits, out.logits)  # no-grad and training forward agree
    assert abs(out.loss.item() - loss.item()) / loss.item() <= (1e-3 if loss_kind == "l1" else 1e-4)
    assert frob(out.logits.float(), logits.detach()) <= 1e-2 and maxrel(out.logits.float(), logits.detach()) <= 2e-2
    tol = 5e-2 if loss_kind == "l1" else 2e-2  # L1: the gradient is sign(diff) / n, elements near a tie flip with bf16 logits
    bad = {}
    for k, p in model.named_parameters():
        if k == "mask_token":  # the decoder-width token of the MAE path is unused here
            assert p.grad is None or float(p.grad.abs().max()) == 0.0
            continue
        e = frob(p.grad, sdg[k].grad)
        if not e <= tol:
            bad[k] = e
    assert not bad, bad


def test_side_stream_gradients_match_single_stream(ops, monkeypatch):
    """training.SideQueue: the weight / bias gradients queued on the second stream (default) equal the ones of the single-stream
    backward (SMBV_WGRAD_STREAM=0) — same kernels on the same inputs, only the launch stream differs; a missing dependency between
    the streams would show up as a wrong or partial gradient.  SMALL64 batch 2 (eager) and the CUDA-graph step."""
    from smb_vision_b200.data import MaskGenerator
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining
    from smb_vision_b200.training import DataParallelStep, GradArena, mim_backward, mim_forward_train

    cfg = vo.OracleConfig(**ge.SMALL64)
    torch.manual_seed(0)
    model = B200VideoMAEForPreTraining(ge.hf_config(ge.SMALL64)).to(DEV).train()
    model.load_state_dict(vo.synthetic_state_dict(cfg, 1234), strict=True)
    vol = model.videomae._volume(vo.synthetic_volume(cfg, 2, 7).to(DEV))
    np.random.seed(0)
    mp = MaskGenerator(96, 96, 32, 16, 0.65).device_batch(2, DEV)
    arenas = {}
    with torch.no_grad():
        loss, logits, dlogits, S = mim_forward_train(model, vol, mp)
        for mode in ("0", "1", "1", "1"):
            monkeypatch.setenv("SMBV_WGRAD_STREAM", mode)
            a = GradArena(model, DEV)
            mim_backward(model, S, dlogits, a)
            torch.cuda.synchronize()
            arenas.setdefault(mode, []).append(a.flat.clone())
    ref = arenas["0"][0]
    assert torch.isfinite(ref).all() and float(ref.abs().max()) > 0
    for a in arenas["1"]:
        # split-K reduce-adds may land in another order, so the two settings are not bit-exact by construction (full size: 4e-5 between
        # two single-stream runs); a missing dependency between the streams gives an O(1) difference
        assert frob(a, ref) <= 2e-4
    # the graph-captured step forks and joins the side stream inside the capture
    monkeypatch.setenv("SMBV_WGRAD_STREAM", "1")
    dp = DataParallelStep(model, cuda_graph=True)
    for _ in range(3):
        l, _ = dp.step(vol, mp)
        torch.cuda.synchronize()
        assert abs(float(l) - float(loss)) <= 1e-5 * abs(float(loss))
        assert frob(dp.arena.flat, ref) <= 2e-4
