"""Drop-in module API for the 3D-ViT MIM hot path, running on the sm_100a kernels.

Mirrors the reference interface (``/root/reference/src/models/videomae/modeling_videomae.py``):

* ``B200VideoMAEForPreTraining(config).forward(pixel_values, bool_masked_pos)`` -> ``(loss, logits)``
  (reference ``VideoMAEForPreTraining.forward``, :753-908)
* ``model.videomae(pixel_values[, bool_masked_pos]).last_hidden_state`` — the embedding-extraction API
  (reference ``VideoMAEModel.forward``, :537-658; callers ``src/run_inference.py:78-86``)

Same constructor (a ``VideoMAEConfig``), same parameter names/shapes (``load_state_dict(strict=True)`` both ways,
SURVEY.md §8b), same ``ValueError``s.  Parameters live in ordinary ``nn.Linear``/``nn.LayerNorm``/``nn.Conv3d``
containers whose ``forward`` is never called: all compute goes through ``ops`` -> C ABI -> CUDA.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional

import torch
from torch import nn

from . import ops
from ._lib import SmbvError

try:  # the reference's own output classes, when transformers is importable (it is a dependency of the reference)
    from transformers.modeling_outputs import BaseModelOutput, ImageClassifierOutput
    from transformers.models.videomae.modeling_videomae import VideoMAEForPreTrainingOutput
except Exception:  # pragma: no cover
    @dataclass
    class BaseModelOutput:  # type: ignore
        last_hidden_state: torch.Tensor = None
        hidden_states: Optional[tuple] = None
        attentions: Optional[tuple] = None

    @dataclass
    class ImageClassifierOutput:  # type: ignore
        loss: Optional[torch.Tensor] = None
        logits: torch.Tensor = None
        hidden_states: Optional[tuple] = None
        attentions: Optional[tuple] = None

    @dataclass
    class VideoMAEForPreTrainingOutput:  # type: ignore
        loss: Optional[torch.Tensor] = None
        logits: torch.Tensor = None
        hidden_states: Optional[tuple] = None
        attentions: Optional[tuple] = None


def _cfg(config, name, default=None):
    return getattr(config, name, default)


# ----------------------------------------------------------------------------------------------
# parameter containers (names == the reference checkpoint ABI)
# ----------------------------------------------------------------------------------------------
class _SelfAttention(nn.Module):  # reference :227-251
    def __init__(self, d, qkv_bias=True):
        super().__init__()
        self.query = nn.Linear(d, d, bias=False)
        self.key = nn.Linear(d, d, bias=False)
        self.value = nn.Linear(d, d, bias=False)
        if qkv_bias:
            self.q_bias = nn.Parameter(torch.zeros(d))
            self.v_bias = nn.Parameter(torch.zeros(d))
        else:
            self.q_bias = None
            self.v_bias = None


class _Dense(nn.Module):
    def __init__(self, i, o):
        super().__init__()
        self.dense = nn.Linear(i, o)


class _Attention(nn.Module):  # reference :319-355
    def __init__(self, d, qkv_bias):
        super().__init__()
        self.attention = _SelfAttention(d, qkv_bias)
        self.output = _Dense(d, d)


class _Layer(nn.Module):  # reference :392-431
    def __init__(self, d, m, eps, qkv_bias):
        super().__init__()
        self.attention = _Attention(d, qkv_bias)
        self.intermediate = _Dense(d, m)
        self.output = _Dense(m, d)
        self.layernorm_before = nn.LayerNorm(d, eps=eps)
        self.layernorm_after = nn.LayerNorm(d, eps=eps)


class _PatchEmbeddings(nn.Module):  # reference :143-192
    def __init__(self, config):
        super().__init__()
        p, t = config.patch_size, config.tubelet_size
        self.projection = nn.Conv3d(config.num_channels, config.hidden_size, kernel_size=(t, p, p), stride=(t, p, p))


class _Embeddings(nn.Module):
    def __init__(self, config, use_mask_token: bool = False):
        super().__init__()
        self.patch_embeddings = _PatchEmbeddings(config)
        if use_mask_token:  # SimMIM-style blend (north star; semantics of src/models/dinov2/modeling_dinov2.py:47, :104-107)
            self.mask_token = nn.Parameter(torch.zeros(1, 1, config.hidden_size))


class _Encoder(nn.Module):
    def __init__(self, n, d, m, eps, qkv_bias):
        super().__init__()
        self.layer = nn.ModuleList([_Layer(d, m, eps, qkv_bias) for _ in range(n)])


class _Decoder(nn.Module):  # reference :662-682
    def __init__(self, config):
        super().__init__()
        dd = config.decoder_hidden_size
        self.decoder_layers = nn.ModuleList(
            [_Layer(dd, config.decoder_intermediate_size, config.layer_norm_eps, config.qkv_bias)
             for _ in range(config.decoder_num_hidden_layers)])
        self.norm = nn.LayerNorm(dd)  # eps 1e-5 (reference :676)
        out = config.tubelet_size * config.patch_size**2 * config.num_channels
        self.head = nn.Linear(dd, out)


def _init_weights(module, std):
    """reference _init_weights :495-505."""
    for m in module.modules():
        if isinstance(m, (nn.Linear, nn.Conv3d)):
            nn.init.normal_(m.weight, mean=0.0, std=std)
            if m.bias is not None:
                nn.init.zeros_(m.bias)
        elif isinstance(m, nn.LayerNorm):
            nn.init.ones_(m.weight)
            nn.init.zeros_(m.bias)


# ----------------------------------------------------------------------------------------------
# packed (kernel-ready) weights
# ----------------------------------------------------------------------------------------------
class _PackedLayer:
    __slots__ = ("wqkv", "bqkv", "wo", "bo", "w1", "b1", "w2", "b2", "g1", "be1", "g2", "be2", "heads", "eps", "hd", "pad32")


def _f32(t):
    return t.detach().float().contiguous()


def _pack_layer(layer: _Layer, heads: int, eps: float, arena=None, prefix: str = "") -> _PackedLayer:
    """fp32 master -> bf16 operands (autocast semantics, SURVEY.md §8 a′); Q,K,V fused into one [3d,d] weight with
    bias [q_bias; 0; v_bias] (reference :261-264).  With a `training.ParamArena` the operands are VIEWS of its flat
    bf16 / fp32 buffers (kept current by FusedAdamW), so nothing is copied or cast here."""
    a = layer.attention.attention
    d = a.query.weight.shape[0]
    p = _PackedLayer()
    if arena is not None and a.q_bias is not None:
        p.wqkv, p.bqkv = arena.wqkv16(prefix), arena.bqkv(prefix)
        p.wo, p.bo = arena.w16(prefix + "attention.output.dense.weight"), _f32(layer.attention.output.dense.bias)
        p.w1, p.b1 = arena.w16(prefix + "intermediate.dense.weight"), _f32(layer.intermediate.dense.bias)
        p.w2, p.b2 = arena.w16(prefix + "output.dense.weight"), _f32(layer.output.dense.bias)
        p.g1, p.be1 = _f32(layer.layernorm_before.weight), _f32(layer.layernorm_before.bias)
        p.g2, p.be2 = _f32(layer.layernorm_after.weight), _f32(layer.layernorm_after.bias)
        p.heads, p.eps, p.hd = heads, eps, d // heads
        return p
    p.wqkv = ops.cast_bf16(torch.cat([_f32(a.query.weight), _f32(a.key.weight), _f32(a.value.weight)], 0))
    zeros = torch.zeros(d, dtype=torch.float32, device=a.query.weight.device)
    p.bqkv = torch.cat([_f32(a.q_bias) if a.q_bias is not None else zeros, zeros,
                        _f32(a.v_bias) if a.v_bias is not None else zeros]).contiguous()
    p.wo, p.bo = ops.cast_bf16(_f32(layer.attention.output.dense.weight)), _f32(layer.attention.output.dense.bias)
    p.w1, p.b1 = ops.cast_bf16(_f32(layer.intermediate.dense.weight)), _f32(layer.intermediate.dense.bias)
    p.w2, p.b2 = ops.cast_bf16(_f32(layer.output.dense.weight)), _f32(layer.output.dense.bias)
    p.g1, p.be1 = _f32(layer.layernorm_before.weight), _f32(layer.layernorm_before.bias)
    p.g2, p.be2 = _f32(layer.layernorm_after.weight), _f32(layer.layernorm_after.bias)
    p.heads, p.eps, p.hd = heads, eps, d // heads
    return p


def _block_forward(X: torch.Tensor, p: _PackedLayer, rope=None, x_copy=None) -> None:
    """One pre-LN transformer block, in place on the fp32 residual stream X [B, n, d]  (reference :405-431).
    `rope` = (grid_size, ids or None, max_pos): V-JEPA's rotary embedding of Q and K (modeling_vjepa.py:346-348).
    `x_copy`: fp32 like X, receives the block's input (stored by the first LayerNorm, which reads X anyway)."""
    B, n, d = X.shape
    h = ops.layernorm_fwd(X, p.g1, p.be1, p.eps, x_copy=x_copy)
    pad32 = p.hd == 32 and getattr(p, "pad32", False)
    if rope is not None and p.hd != 64 and not pad32:
        raise SmbvError("the rotary embedding kernel is wired to the tcgen05 attention paths (head_dim 64, or 32 zero-padded)")
    if pad32:  # head_dim 32 on the head_dim-64 kernels (V-JEPA predictor): see attention32_forward
        a = attention32_forward(h, p, n, rope)[0]
    elif p.hd == 64:
        qkv = ops.gemm(h, p.wqkv, p.bqkv, ops.EPI_QKV_HEADS, heads=p.heads, tokens=n)  # [3,B,H,n,64]
        if rope is not None:
            ops.rope3d_(qkv[:2], rope[0], rope[1], rope[2])  # Q and K sections, in place
        a = ops.flash_attn_fwd(qkv[0], qkv[1], qkv[2], 64 ** -0.5)  # [B,n,d] bf16
    else:  # small heads (tiny configs): token-major QKV + the CUDA-core attention kernels
        a = ops.attn_small_fwd(ops.gemm(h, p.wqkv, p.bqkv, ops.EPI_BF16), p.heads, p.hd ** -0.5)
    ops.gemm(a, p.wo, p.bo, ops.EPI_RESID_F32, residual=X)  # X += a Wo^T + bo
    h = ops.layernorm_fwd(X, p.g2, p.be2, p.eps)
    f = ops.gemm(h, p.w1, p.b1, ops.EPI_GELU_BF16)
    ops.gemm(f, p.w2, p.b2, ops.EPI_RESID_F32, residual=X)  # X += gelu(.) W2^T + b2


def attention32_forward(h: torch.Tensor, p: _PackedLayer, n: int, rope=None, return_lse: bool = False):
    """Attention of a head_dim-32 block (V-JEPA predictor, 384 / 12 heads) on the head_dim-64 tcgen05 kernels.
    The fused QKV GEMM writes H/2 "double heads" (64-wide head-major rows holding two real heads); the rotary kernel runs on
    them viewed as 32-wide rows (`rope` = (grid, ids, max_pos, ids_doubled)); the rows are split into H zero-padded 64-wide
    heads for the attention kernel (scale 32^-0.5; the pad changes neither q.k nor P.v) and the output is squeezed back.
    Returns (a bf16 [B,n,d], qkv_padded [3,B,H,n,64], a64 [B,n,H*64], lse)."""
    B, H = h.shape[0], p.heads
    qkv2 = ops.gemm(h, p.wqkv, p.bqkv, ops.EPI_QKV_HEADS, heads=H // 2, tokens=n)  # [3,B,H/2,n,64]
    if rope is not None:
        ops.rope3d_(qkv2[:2].view(2, B, H // 2, 2 * n, 32), rope[0], rope[3], rope[2])
    qkvp = ops.heads32_expand(qkv2)  # [3,B,H,n,64]
    res = ops.flash_attn_fwd(qkvp[0], qkvp[1], qkvp[2], 32 ** -0.5, return_lse=return_lse)
    a64, lse = res if return_lse else (res, None)
    return ops.heads32_tokens(a64, H, expand=False), qkvp, a64, lse


def _params_signature(module: nn.Module):
    return tuple((p.data_ptr(), p._version) for p in module.parameters())


def _prep_mask(bool_masked_pos: torch.Tensor, device, num_masked: Optional[int]):
    """bool [B,N] -> (fine uint8, vis_idx, msk_idx, slot, n_vis, n_mask).  A CPU mask is counted on the host (no
    device sync); a CUDA mask needs `num_masked` or one 8-byte D2H read of the counts (the reference syncs on
    every boolean gather, modeling_videomae.py:136, :811-812, :894)."""
    B, N = bool_masked_pos.shape
    if bool_masked_pos.dtype not in (torch.bool, torch.uint8):
        raise SmbvError("bool_masked_pos must be a bool tensor")
    if not bool_masked_pos.is_cuda:
        per = bool_masked_pos.to(torch.uint8).sum(dim=1)
        if num_masked is None:
            num_masked = int(per[0])
        if not bool((per == num_masked).all()):
            # same failure the reference hits at the reshape of modeling_videomae.py:137
            raise RuntimeError("bool_masked_pos must mask the same number of patches for every sample in the batch")
    fine = bool_masked_pos.to(device=device, dtype=torch.uint8, non_blocking=True).contiguous()
    vis, msk, slot, counts = ops.mask_index(fine)
    if num_masked is None:
        c = counts.cpu()
        num_masked = int(c[0, 1])
        if not bool((c[:, 1] == num_masked).all()):
            raise RuntimeError("bool_masked_pos must mask the same number of patches for every sample in the batch")
    return fine, vis, msk, slot, N - num_masked, num_masked


def _check_layers(layers, L: int):
    """hidden-state indices 0..L (0 = patch embedding, L = last block)."""
    layers = [int(k) for k in layers]
    bad = [k for k in layers if not 0 <= k <= L]
    if bad:
        raise ValueError(f"hidden-state indices {bad} outside 0..{L} (0 = patch embedding, {L} = last block)")
    return layers


def _want_states(output_hidden_states, config) -> bool:
    """`output_hidden_states=None` falls back to `config.output_hidden_states` (upstream PreTrainedModel semantics)."""
    return bool(_cfg(config, "output_hidden_states", False) if output_hidden_states is None else output_hidden_states)


def _out_states(states, dtype):
    return tuple(states) if dtype is None else tuple(h.to(dtype) for h in states)


class _PretrainedIO:
    """`from_pretrained` / `save_pretrained` with the checkpoint layout the reference's `PreTrainedModel` classes use
    (reference src/run_mim.py:345-357, src/run_inference.py:70, src/run_classification.py:495-504): a LOCAL directory with
    `config.json` + `model.safetensors` (or `pytorch_model.bin`, or a sharded `model.safetensors.index.json`).  Like
    HF, parameters the checkpoint lacks keep their fresh initialisation (e.g. `classifier.*` when fine-tuning from an MIM
    checkpoint) and checkpoint entries the model lacks are ignored; both lists are kept in `model.loading_info`."""

    # attention back ends a caller may name (reference src/run_mim.py:345-357 passes `attn_implementation`): they are all
    # the same function — softmax(QK^T * scale) V, reference :196-223 — and every one of them runs on the tcgen05 kernel here
    _ATTN_NAMES = (None, "eager", "sdpa", "flash_attention_2", "flash_attention_3", "flex_attention", "b200_tcgen05")
    _out_dtype = None  # set by `torch_dtype=torch.bfloat16/float16`: whole-model reduced precision (run_inspect.py:106-111)

    def set_reduced_precision(self, dtype) -> None:
        """`from_pretrained(..., torch_dtype=torch.bfloat16)` semantics (scripts/inference/inspect/run_inspect.py:106-111):
        the checkpoint is held in `dtype` — every parameter is rounded to it (stored in the fp32 master containers the
        kernels read, so the values are exactly the reference's bf16 weights) — and outputs are returned in `dtype`.
        Internally the residual stream, LayerNorm statistics and softmax stay fp32 (more exact than the reference's bf16
        pipeline, inside the same tolerance against the fp32 oracle)."""
        if dtype in (None, torch.float32):
            self._out_dtype = None
            return
        if dtype not in (torch.bfloat16, torch.float16):
            raise ValueError(f"torch_dtype {dtype} is not supported (float32, bfloat16, float16)")
        with torch.no_grad():
            for p in self.parameters():
                p.copy_(p.to(dtype).to(p.dtype))
        self._out_dtype = dtype
        for m in (self, getattr(self, "videomae", None)):
            if m is not None and hasattr(m, "refresh_operands"):
                m.refresh_operands()
                m._out_dtype = dtype

    @classmethod
    def from_pretrained(cls, pretrained_model_name_or_path, config=None, torch_dtype=None, attn_implementation=None, **kwargs):
        import json
        import os

        if attn_implementation not in cls._ATTN_NAMES:
            raise ValueError(f"attn_implementation={attn_implementation!r} is not one of {cls._ATTN_NAMES[1:]} "
                             "(all of them run on the tcgen05 flash-attention kernel in this build)")
        dtype = kwargs.pop("dtype", None) if torch_dtype is None else torch_dtype  # transformers >= 4.56 spells it `dtype`
        if isinstance(dtype, str):
            dtype = None if dtype == "auto" else getattr(torch, dtype)
        path = str(pretrained_model_name_or_path)
        if not os.path.isdir(path):
            raise OSError(f"{path} is not a local directory (this build has no hub access; download the checkpoint first)")
        if config is None:
            config = cls._config_from_dir(path)
        model = cls(config, **{k: v for k, v in kwargs.items() if k in ("loss_kind",)})
        sd = {}
        if os.path.exists(os.path.join(path, "model.safetensors.index.json")):
            from safetensors.torch import load_file

            idx = json.load(open(os.path.join(path, "model.safetensors.index.json")))
            for shard in sorted(set(idx["weight_map"].values())):
                sd.update(load_file(os.path.join(path, shard)))
        elif os.path.exists(os.path.join(path, "model.safetensors")):
            from safetensors.torch import load_file

            sd = load_file(os.path.join(path, "model.safetensors"))
        elif os.path.exists(os.path.join(path, "pytorch_model.bin")):
            sd = torch.load(os.path.join(path, "pytorch_model.bin"), map_location="cpu", weights_only=True)
        else:
            raise OSError(f"no model.safetensors / pytorch_model.bin under {path}")
        own = model.state_dict()
        sd = model._rename_checkpoint_keys(sd)
        if not any(k in own for k in sd) and any(("videomae." + k) in own for k in sd):
            sd = {"videomae." + k: v for k, v in sd.items()}  # a bare VideoMAEModel checkpoint (base_model_prefix)
        if not any(k in own for k in sd) and any(k.startswith("videomae.") and k[len("videomae."):] in own for k in sd):
            sd = {k[len("videomae."):]: v for k, v in sd.items() if k.startswith("videomae.")}  # head model -> bare encoder
        bad = [k for k in sd if k in own and tuple(sd[k].shape) != tuple(own[k].shape)]
        if bad:
            raise RuntimeError(f"size mismatch for {bad[:4]}{'...' if len(bad) > 4 else ''}")
        res = model.load_state_dict({k: v.float() for k, v in sd.items() if k in own}, strict=False)
        model.loading_info = {"missing_keys": list(res.missing_keys), "unexpected_keys": [k for k in sd if k not in own],
                              "attn_implementation": "b200_tcgen05", "requested_attn_implementation": attn_implementation}
        model.set_reduced_precision(dtype)  # float32 / None: fp32 masters + bf16 tensor-core operands (autocast semantics)
        return model

    @classmethod
    def _config_from_dir(cls, path):
        from transformers import VideoMAEConfig

        return VideoMAEConfig.from_pretrained(path)

    def _rename_checkpoint_keys(self, sd: dict) -> dict:
        return sd

    # ---- small PreTrainedModel surface HF `Trainer` and the reference scripts touch ----
    supports_gradient_checkpointing = True  # reference modeling_videomae.py:487-493

    def gradient_checkpointing_enable(self, gradient_checkpointing_kwargs=None):
        """Accepted for `--gradient_checkpointing true` (scripts/training/run_mim.sh:32) and ignored: the saved activations
        of one 512x512x320 volume are 6.5 GB of the 180 GB HBM3e, so nothing is recomputed."""
        self.is_gradient_checkpointing = False

    def gradient_checkpointing_disable(self):
        self.is_gradient_checkpointing = False

    @property
    def device(self):
        return next(self.parameters()).device

    @property
    def dtype(self):
        return next(self.parameters()).dtype

    def num_parameters(self, only_trainable: bool = False) -> int:
        return sum(p.numel() for p in self.parameters() if p.requires_grad or not only_trainable)

    def get_input_embeddings(self):
        vm = getattr(self, "videomae", self)
        return vm.embeddings.patch_embeddings

    def save_pretrained(self, save_directory, safe_serialization: bool = True, **kwargs):
        import os

        os.makedirs(save_directory, exist_ok=True)
        self.config.save_pretrained(save_directory)
        sd = {k: v.detach().to("cpu").contiguous().clone() for k, v in self.state_dict().items()}
        if safe_serialization:
            from safetensors.torch import save_file

            save_file(sd, os.path.join(save_directory, "model.safetensors"), metadata={"format": "pt"})
        else:
            torch.save(sd, os.path.join(save_directory, "pytorch_model.bin"))


class B200VideoMAEModel(_PretrainedIO, nn.Module):
    """Encoder (reference ``VideoMAEModel``, modeling_videomae.py:508-658)."""

    base_model_prefix = "videomae"
    main_input_name = "pixel_values"

    def __init__(self, config, use_mask_token: bool = False):
        super().__init__()
        self.config = config
        d = config.hidden_size
        if d % config.num_attention_heads != 0:
            raise ValueError(f"hidden size {d} is not a multiple of the number of attention heads {config.num_attention_heads}")
        self.embeddings = _Embeddings(config, use_mask_token)
        self.encoder = _Encoder(config.num_hidden_layers, d, config.intermediate_size, config.layer_norm_eps, config.qkv_bias)
        self.layernorm = None if _cfg(config, "use_mean_pooling", True) else nn.LayerNorm(d, eps=config.layer_norm_eps)
        _init_weights(self, _cfg(config, "initializer_range", 0.02))
        self._packed = None
        self._packed_sig = None
        self._arena = None  # training.ParamArena, when the parameters live in a flat arena
        self._pos = {}

    # ---- geometry ----
    @property
    def grid(self):
        c = self.config
        return (c.num_frames // c.tubelet_size, c.image_size // c.patch_size, c.image_size // c.patch_size)

    @property
    def num_patches(self):
        g = self.grid
        return g[0] * g[1] * g[2]

    def pos_table(self, d: int, device) -> torch.Tensor:
        """Fixed sin-cos table, generated once on the device (reference builds it in Python at init, :95-106, :121,
        and copies it host->device on every forward, :129-131)."""
        key = (d, str(device))
        if key not in self._pos:
            self._pos[key] = ops.sincos_table(self.num_patches, d, device)
        return self._pos[key]

    def _check_config(self):
        c = self.config
        if c.patch_size != 16 or c.tubelet_size != 16:
            raise SmbvError("smb_vision_b200 implements patch_size = tubelet_size = 16 (src/run_mim.py:322-330 sets both)")
        if c.num_channels != 1:
            raise SmbvError("smb_vision_b200 implements single-channel CT/MR volumes (num_channels=1, src/run_mim.py:326)")
        if c.hidden_size // c.num_attention_heads not in (8, 16, 32, 64):
            raise SmbvError("smb_vision_b200 attention implements head_dim 64 (tcgen05; smb-vision-base: 768/12, decoder 384/6) "
                            "and 8/16/32 (small-model kernels)")
        if _cfg(c, "hidden_act", "gelu") != "gelu":
            raise SmbvError("only hidden_act='gelu' (exact erf) is implemented")

    def packed(self):
        sig = _params_signature(self)
        if self._packed is None or sig != self._packed_sig:
            c = self.config
            proj = self.embeddings.patch_embeddings.projection
            ar = self._arena
            if ar is not None:  # parameters were edited through torch (load_state_dict, ...): refresh the bf16 copies
                ar.sync_bf16()
            self._packed = dict(
                wpe=_f32(proj.weight).reshape(c.hidden_size, -1).contiguous(), bpe=_f32(proj.bias),
                layers=[_pack_layer(l, c.num_attention_heads, c.layer_norm_eps, ar, f"videomae.encoder.layer.{i}.")
                        for i, l in enumerate(self.encoder.layer)],
            )
            # bf16 operand of the patch embedding (implicit-GEMM kernel and the visible-patch GEMM of the training forward):
            # a view of the arena's bf16 copy (kept current by smbv_adamw_step) or a cast made once per parameter version
            self._packed["wpe16"] = (ar.w16("videomae.embeddings.patch_embeddings.projection.weight").reshape(c.hidden_size, -1)
                                     if ar is not None else ops.cast_bf16(self._packed["wpe"]))
            if hasattr(self.embeddings, "mask_token"):
                self._packed["mask_token"] = _f32(self.embeddings.mask_token).reshape(-1)
            self._packed_sig = sig
        return self._packed

    def refresh_operands(self) -> None:
        """Re-derive the bf16 GEMM operands from the fp32 masters.  `packed()` keys its cache on torch's parameter version
        counters, which `torch.optim.AdamW(fused=True)` / foreach optimisers (HF Trainer's default) do NOT bump — so every
        differentiable forward calls this first (a 97 M-element cast, < 1 ms) instead of trusting the counters."""
        if self._arena is not None:
            self._arena.sync_bf16()  # the packed operands are views of the arena: nothing to re-pack
        else:
            self._packed = None

    def _volume(self, pixel_values: torch.Tensor) -> torch.Tensor:
        c = self.config
        if pixel_values.dim() != 5:
            raise ValueError("pixel_values must be [batch, frames, channels, height, width]")
        B, T, C, H, W = pixel_values.shape
        if C != c.num_channels:  # reference :181-184
            raise ValueError("Make sure that the channel dimension of the pixel values match with the one set in the configuration.")
        if H != c.image_size or W != c.image_size:  # reference :185-188
            raise ValueError(f"Input image size ({H}*{W}) doesn't match model ({c.image_size}*{c.image_size}).")
        if T != c.num_frames:
            raise ValueError(f"Input depth ({T}) doesn't match model ({c.num_frames}).")
        dev = self.embeddings.patch_embeddings.projection.weight.device
        v = pixel_values.to(device=dev, dtype=torch.float32, non_blocking=True)
        return v.reshape(B, T, H, W).contiguous()  # C == 1: permute(0,2,1,3,4) of reference :190 is free

    def encode(self, vol: torch.Tensor, mask_pack=None, blend: bool = False, keep=None):
        """fp32 volume [B,T,H,W] -> fp32 residual stream [B, n, d] after all encoder blocks.  `blend`: SimMIM style — masked
        tokens are replaced by the encoder mask token in the patch-embed epilogue and all N tokens are kept.
        `keep`: hidden-state indices (0 = patch embedding, k = output of block k-1, taken before the final LayerNorm) ->
        returns (X, states) with states[k] fp32 [B, n, d] for k in `keep` and None elsewhere (num_hidden_layers + 1 entries);
        state L is the residual stream itself, the others are copies written by the first LayerNorm of the next block."""
        self._check_config()
        pk = self.packed()
        pos = self.pos_table(self.config.hidden_size, vol.device)
        if blend:
            if "mask_token" not in pk:
                raise SmbvError("the SimMIM blend needs a model built with use_mask_token=True")
            X = ops.patch_embed_select_fwd(vol, pk["wpe16"], pk["bpe"], pos, mask_pack[0], pk["mask_token"])
        elif mask_pack is None:
            X = ops.patch_embed_fwd(vol, pk["wpe16"], pk["bpe"], pos)
        else:
            fine, _, _, slot, n_vis, _ = mask_pack
            X = ops.patch_embed_fwd(vol, pk["wpe16"], pk["bpe"], pos, fine, slot, n_vis)
        L = len(pk["layers"])
        keep = None if keep is None else set(_check_layers(keep, L))
        states = [None] * (L + 1)
        for i, p in enumerate(pk["layers"]):
            if keep is not None and i in keep:
                states[i] = torch.empty_like(X)
            _block_forward(X, p, x_copy=states[i])
        if keep is not None and L in keep:
            states[L] = X
        if self.layernorm is not None:  # use_mean_pooling=False only (reference :517-520, :648-649)
            X = ops.layernorm_fwd(X, _f32(self.layernorm.weight), _f32(self.layernorm.bias), self.config.layer_norm_eps).float()
        return X if keep is None else (X, states)

    def forward(self, pixel_values, bool_masked_pos=None, head_mask=None, output_attentions=None,
                output_hidden_states=None, return_dict=None, num_masked: Optional[int] = None, **kwargs):
        if head_mask is not None:
            raise ValueError("head_mask is not supported by the fused attention kernel")
        if output_attentions:
            raise ValueError("output_attentions is not supported by the fused attention kernel (same restriction as sdpa, reference :272-276)")
        with torch.no_grad():
            vol = self._volume(pixel_values)
            mp = None if bool_masked_pos is None else _prep_mask(bool_masked_pos, vol.device, num_masked)
        X, states = self._encode_states(vol, mp, _want_states(output_hidden_states, self.config))
        if self._out_dtype is not None:
            X = X.to(self._out_dtype)
        hs = None
        if states is not None:  # upstream: the last state IS last_hidden_state when no final LayerNorm follows
            hs = _out_states(states[:-1], self._out_dtype) + ((X,) if self.layernorm is None else _out_states(states[-1:], self._out_dtype))
        if return_dict is False:
            return (X,) if hs is None else (X, hs)
        return BaseModelOutput(last_hidden_state=X, hidden_states=hs, attentions=None)

    def _encode_states(self, vol, mask_pack, want: bool):
        """-> (X, states or None): the encoder output (after the final LayerNorm, if any) and, with `want`, the
        num_hidden_layers + 1 hidden states (the last one before that LayerNorm).  Differentiable when grad is enabled and a
        parameter requires it (one autograd node: CUDA forward with saves + hand-scheduled backward)."""
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            from .training import encoder_autograd_forward

            out = encoder_autograd_forward(self, vol, mask_pack, states=want)
            if not want:
                return out, None
            X, states = out[0], list(out[1:])
            return X, (states + [X] if self.layernorm is None else states)
        with torch.no_grad():
            if not want:
                return self.encode(vol, mask_pack), None
            return self.encode(vol, mask_pack, keep=range(self.config.num_hidden_layers + 1))


class B200VideoMAEForPreTraining(_PretrainedIO, nn.Module):
    """MIM pre-training model (reference ``VideoMAEForPreTraining``, modeling_videomae.py:733-908).

    ``loss_kind='mse'`` with norm-pix targets and ``mim_style='mae'`` (masked tokens dropped before the encoder, decoder-width
    mask token appended after it) are the reference path.  The north star's wording — "SimMIM mask-token blending ... fused
    into [the patch-embed] epilogue ... masked-L1 reconstruction loss" — is the switch ``mim_style='simmim', loss_kind='l1'``:
    ``select(mask, mask_token, emb) + pos`` in the patch-embed epilogue (``smbv_patch_embed_select_fwd``; semantics of
    src/models/dinov2/modeling_dinov2.py:104-107), encoder and decoder over all N tokens in natural order, head and loss on the
    masked rows; one extra parameter ``videomae.embeddings.mask_token`` [1,1,hidden].  Oracle: ``pretrain_forward_simmim``."""

    base_model_prefix = "videomae"
    main_input_name = "pixel_values"

    def __init__(self, config, loss_kind: str = "mse", mim_style: str = "mae"):
        super().__init__()
        self.config = config
        self.loss_kind = {"mse": 0, "l1": 1}[loss_kind]
        if mim_style not in ("mae", "simmim"):
            raise ValueError(f"mim_style must be 'mae' (the reference path) or 'simmim' (the north-star variant), got {mim_style!r}")
        self.mim_style = mim_style
        self.videomae = B200VideoMAEModel(config, use_mask_token=(mim_style == "simmim"))
        self.encoder_to_decoder = nn.Linear(config.hidden_size, config.decoder_hidden_size, bias=False)
        self.mask_token = nn.Parameter(torch.zeros(1, 1, config.decoder_hidden_size))
        self.decoder = _Decoder(config)
        std = _cfg(config, "initializer_range", 0.02)
        _init_weights(self.encoder_to_decoder, std)
        _init_weights(self.decoder, std)
        self.decoder.norm.eps = 1e-5
        self._packed = None
        self._packed_sig = None
        self._arena = None

    def packed(self):
        sig = _params_signature(self.decoder) + _params_signature(self.encoder_to_decoder) + ((self.mask_token.data_ptr(), self.mask_token._version),)
        if self._packed is None or sig != self._packed_sig:
            c = self.config
            ar = self._arena
            if ar is not None:
                ar.sync_bf16()
            self._packed = dict(
                we2d=ops.cast_bf16(_f32(self.encoder_to_decoder.weight)) if ar is None else ar.w16("encoder_to_decoder.weight"),
                mask_token=_f32(self.mask_token).reshape(-1).contiguous(),
                layers=[_pack_layer(l, c.decoder_num_attention_heads, c.layer_norm_eps, ar, f"decoder.decoder_layers.{j}.")
                        for j, l in enumerate(self.decoder.decoder_layers)],
                gn=_f32(self.decoder.norm.weight), bn=_f32(self.decoder.norm.bias),
                wh=ops.cast_bf16(_f32(self.decoder.head.weight)) if ar is None else ar.w16("decoder.head.weight"), bh=_f32(self.decoder.head.bias),
            )
            self._packed_sig = sig
        return self._packed

    def refresh_operands(self) -> None:
        """see B200VideoMAEModel.refresh_operands (encoder and decoder share one arena when there is one)."""
        if self._arena is not None:
            self._arena.sync_bf16()
        else:
            self._packed = None
            self.videomae.refresh_operands()

    def _check_config(self):
        c = self.config
        if c.decoder_hidden_size // c.decoder_num_attention_heads not in (8, 16, 32, 64):
            raise SmbvError("smb_vision_b200 attention implements head_dim 64 (tcgen05) and 8/16/32 (small-model kernels)")
        if not _cfg(c, "norm_pix_loss", True):
            # reference :868-874 raises for C != 3 when norm_pix_loss is False
            raise ValueError("Can't unnormalize non-RGB images. Consider setting config.norm_pix_loss to False.")

    def forward_no_grad(self, vol: torch.Tensor, mask_pack, want_dlogits: bool = False, states: bool = False):
        """Forward of reference :791-897 on device tensors.  Returns (loss, logits bf16 [B,n_mask,K], dlogits|None), and the
        encoder's hidden states as a fourth item with `states`."""
        self._check_config()
        keep = range(self.config.num_hidden_layers + 1) if states else None
        c = self.config
        fine, vis, msk, slot, n_vis, n_mask = mask_pack
        B = vol.shape[0]
        N, dd = self.videomae.num_patches, c.decoder_hidden_size
        pk = self.packed()
        pos_d = self.videomae.pos_table(dd, vol.device)
        if self.mim_style == "simmim":
            X = self.videomae.encode(vol, mask_pack, blend=True, keep=keep)  # [B, N, d] fp32, masked rows = mask token + PE
            X, hs = X if states else (X, None)
            Xb = ops.cast_bf16(X)
            Xd = torch.empty((B, N, dd), dtype=torch.float32, device=vol.device)
            every = torch.arange(N, dtype=torch.int32, device=vol.device)
            for b in range(B):  # encoder_to_decoder + PE, natural token order
                ops.gemm(Xb[b], pk["we2d"], None, ops.EPI_POS_GATHER_F32, out=Xd[b], pos=pos_d, row_map=every)
            for p in pk["layers"]:
                _block_forward(Xd, p)
            G = ops.gather_rows(Xd, msk[:, :n_mask].contiguous())  # masked rows, ascending n
            hN = ops.layernorm_fwd(G, pk["gn"], pk["bn"], 1e-5)
            logits = ops.gemm(hN, pk["wh"], pk["bh"], ops.EPI_BF16)
            loss, dlogits = ops.normpix_loss(vol, msk, n_mask, logits, want_dlogits, self.loss_kind, c.patch_size)
            return (loss, logits, dlogits, hs) if states else (loss, logits, dlogits)
        X = self.videomae.encode(vol, mask_pack, keep=keep)  # [B, n_vis, d] fp32
        X, hs = X if states else (X, None)
        Xb = ops.cast_bf16(X)
        Xd = torch.empty((B, N, dd), dtype=torch.float32, device=vol.device)
        for b in range(B):  # visible rows: encoder_to_decoder + PE[vis]  (reference :801-811, :815)
            ops.gemm(Xb[b], pk["we2d"], None, ops.EPI_POS_GATHER_F32, out=Xd[b, :n_vis], pos=pos_d, row_map=vis[b])
        ops.fill_mask_tokens(Xd, pk["mask_token"], pos_d, msk, n_vis)  # masked rows (reference :812-815)
        for p in pk["layers"]:
            _block_forward(Xd, p)
        hN = torch.empty((B, n_mask, dd), dtype=torch.bfloat16, device=vol.device)
        for b in range(B):  # last n_mask tokens -> LayerNorm(eps 1e-5) (reference :717-721)
            ops.layernorm_fwd(Xd[b, n_vis:], pk["gn"], pk["bn"], 1e-5, out=hN[b])
        logits = ops.gemm(hN, pk["wh"], pk["bh"], ops.EPI_BF16)  # [B, n_mask, 4096] bf16 (reference :722)
        loss, dlogits = ops.normpix_loss(vol, msk, n_mask, logits, want_dlogits, self.loss_kind, c.patch_size)
        return (loss, logits, dlogits, hs) if states else (loss, logits, dlogits)

    def forward(self, pixel_values, bool_masked_pos=None, head_mask=None, output_attentions=None,
                output_hidden_states=None, return_dict=None, num_masked: Optional[int] = None, **kwargs):
        if head_mask is not None:
            raise ValueError("head_mask is not supported by the fused attention kernel")
        if output_attentions:
            raise ValueError("output_attentions is not supported by the fused attention kernel")
        if bool_masked_pos is None:  # reference :807-808
            raise ValueError("One must provided a boolean mask ")
        with torch.no_grad():
            vol = self.videomae._volume(pixel_values)
            mp = _prep_mask(bool_masked_pos, vol.device, num_masked)
        want = _want_states(output_hidden_states, self.config)
        hs = None
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            from .training import autograd_forward  # differentiable path: one autograd node around the CUDA fwd/bwd

            self.refresh_operands()
            loss, logits, *states = autograd_forward(self, vol, mp, states=want)
        else:
            with torch.no_grad():
                loss, logits, _, *states = self.forward_no_grad(vol, mp, states=want)
                states = states[0] if want else []
        if want:  # the encoder's states (visible tokens; all N for mim_style="simmim")
            hs = _out_states(states, self._out_dtype)
        if return_dict is False:
            return (loss, logits) if hs is None else (loss, logits, hs)
        return VideoMAEForPreTrainingOutput(loss=loss, logits=logits, hidden_states=hs, attentions=None)


class B200VideoMAEForVideoClassification(_PretrainedIO, nn.Module):
    """Classification / regression fine-tuning model with optional additional features (age, sex, ...).

    Reference ``VideoMAEForVideoClassification`` (modeling_videomae.py:917-1023; callers src/run_classification.py:227-271,
    :452-504): encoder over ALL tokens -> mean over tokens -> ``fc_norm`` -> ``cat([h, additional_features])`` ->
    ``classifier`` -> MSE / cross-entropy / BCE-with-logits by ``config.problem_type``.  Same parameter names
    (``videomae.*``, ``fc_norm.*``, ``classifier.*``) and the same ``ValueError``s."""

    base_model_prefix = "videomae"
    main_input_name = "pixel_values"
    _PROBLEMS = {"regression": ops.CLS_REGRESSION, "single_label_classification": ops.CLS_SINGLE_LABEL,
                 "multi_label_classification": ops.CLS_MULTI_LABEL}

    def __init__(self, config):
        super().__init__()
        self.config = config
        self.num_labels = config.num_labels
        if self.num_labels <= 0:
            raise SmbvError("num_labels must be > 0 (the nn.Identity classifier of reference :932-937 has no loss to train)")
        self.videomae = B200VideoMAEModel(config)
        d = config.hidden_size
        self.fc_norm = nn.LayerNorm(d) if _cfg(config, "use_mean_pooling", True) else None  # eps 1e-5 (reference :925)
        extra = int(_cfg(config, "additional_features_size", 0) or 0)
        self.classifier = nn.Linear(d + extra, self.num_labels)  # reference :927-937
        _init_weights(self.classifier, _cfg(config, "initializer_range", 0.02))

    def head_params(self):
        fn = self.fc_norm
        return dict(gamma=None if fn is None else _f32(fn.weight), beta=None if fn is None else _f32(fn.bias),
                    eps=1e-5 if fn is None else fn.eps, W=_f32(self.classifier.weight), b=_f32(self.classifier.bias))

    def problem_id(self, labels) -> int:
        """reference :995-1002 (sets config.problem_type on first use, like the reference does)."""
        if labels is None:
            return ops.CLS_NONE
        c = self.config
        if _cfg(c, "problem_type") is None:
            if self.num_labels == 1:
                c.problem_type = "regression"
            elif labels.dtype in (torch.long, torch.int):
                c.problem_type = "single_label_classification"
            else:
                c.problem_type = "multi_label_classification"
        return self._PROBLEMS[c.problem_type]

    def _prep(self, additional_features, labels, dev):
        c = self.config
        feats = None
        if additional_features is not None:  # reference :980-987
            if not hasattr(c, "additional_features_size"):
                raise ValueError("Model config must have additional_features_size set when using additional_features")
            if additional_features.shape[-1] != c.additional_features_size:
                raise ValueError(f"Expected additional_features of size {c.additional_features_size}, got {additional_features.shape[-1]}")
            feats = additional_features.to(device=dev, dtype=torch.float32, non_blocking=True).contiguous()
        elif self.classifier.in_features != c.hidden_size:
            raise ValueError(f"Expected additional_features of size {self.classifier.in_features - c.hidden_size}, got none")
        lab = None
        if labels is not None:
            pid = self.problem_id(labels)
            lab = labels.to(device=dev, non_blocking=True)
            lab = (lab.to(torch.int64).reshape(-1) if pid == ops.CLS_SINGLE_LABEL else lab.to(torch.float32).reshape(-1, self.num_labels)).contiguous()
        return feats, lab

    def forward(self, pixel_values=None, additional_features=None, head_mask=None, labels=None, output_attentions=None,
                output_hidden_states=None, return_dict=None, **kwargs):
        if head_mask is not None:
            raise ValueError("head_mask is not supported by the fused attention kernel")
        if output_attentions:
            raise ValueError("output_attentions is not supported by the fused attention kernel")
        with torch.no_grad():
            vol = self.videomae._volume(pixel_values)
            feats, lab = self._prep(additional_features, labels, vol.device)
        want = _want_states(output_hidden_states, self.config)
        states = None
        if lab is not None and torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            from .training import cls_autograd_forward

            self.videomae.refresh_operands()
            loss, logits, *states = cls_autograd_forward(self, vol, feats, lab, states=want)
        else:
            if want:  # without labels there is no loss to train, but the states stay differentiable under grad
                X, states = self.videomae._encode_states(vol, None, True)
            with torch.no_grad():
                if not want:
                    X = self.videomae.encode(vol, None)  # [B, N, d] fp32 (already through videomae.layernorm if not mean pooling)
                X = X.detach()
                hp = self.head_params()
                if self.fc_norm is not None:  # reference :974-975
                    pooled, inv_n = ops.token_sum(X), 1.0 / X.shape[1]
                else:  # reference :976-977
                    pooled, inv_n = X[:, 0].contiguous(), 1.0
                loss, logits, _ = ops.cls_head(pooled, inv_n, hp["gamma"], hp["beta"], hp["eps"], feats, hp["W"], hp["b"], lab,
                                               self.problem_id(lab))
        if self._out_dtype is not None:
            logits = logits.to(self._out_dtype)
        hs = _out_states(states, self._out_dtype) if want else None
        if return_dict is False:
            return tuple(v for v in (loss, logits, hs) if v is not None)
        return ImageClassifierOutput(loss=loss, logits=logits, hidden_states=hs, attentions=None)
