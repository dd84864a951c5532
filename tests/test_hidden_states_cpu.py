"""CPU: the semantics of `output_hidden_states` for the VideoMAE models, pinned against upstream `transformers`, and the host-side
argument checks of the C entry points behind it.

`oracle_states` composes the oracle's own pieces (`embed`, `_layer`) into the encoder's hidden states: entry 0 is the
patch-embedding output (after the position add and the masked-token drop, or the SimMIM blend), entry k the output of block
k - 1, all taken before the final encoder LayerNorm of use_mean_pooling=False.  The GPU tests (test_gpu_hidden_states.py)
compare the CUDA path with it.
"""
import ctypes

import numpy as np
import pytest
import torch

import __graft_entry__ as ge
from oracle import videomae_oracle as vo
from oracle.mim_mask import OracleMaskGenerator


def oracle_states(sd, cfg, x, mask=None, simmim=False):
    """The num_hidden_layers + 1 encoder hidden states of the oracle (differentiable like the oracle itself)."""
    if simmim:  # pretrain_forward_simmim's blend: every token, masked ones replaced by the encoder mask token
        w = sd["videomae.embeddings.patch_embeddings.projection.weight"]
        E = torch.nn.functional.linear(vo.patchify(x, cfg).to(w.dtype), w.permute(0, 2, 3, 4, 1).reshape(w.shape[0], -1),
                                       sd["videomae.embeddings.patch_embeddings.projection.bias"])
        E = torch.where(mask.unsqueeze(-1), sd["videomae.embeddings.mask_token"].to(E.dtype), E)
        h = E + vo.sinusoid_table(cfg.num_patches, cfg.hidden_size).to(E.dtype)
    else:
        h = vo.embed(sd, cfg, x, mask)
    states = [h]
    for i in range(cfg.num_hidden_layers):
        h = vo._layer(h, sd, f"videomae.encoder.layer.{i}.", cfg.num_attention_heads, cfg.layer_norm_eps)
        states.append(h)
    return states


def _mask(batch, seed=0):
    np.random.seed(seed)
    g = OracleMaskGenerator(96, 96, 32, 16, 0.65)
    return torch.from_numpy(np.stack([g() for _ in range(batch)]))


def _upstream(cls, cfgd, sd, **extra):
    import transformers

    hc = ge.hf_config(cfgd)
    hc._attn_implementation = "eager"
    for k, v in extra.items():
        setattr(hc, k, v)
    m = getattr(transformers, cls)(hc).eval()
    own = m.state_dict()
    m.load_state_dict({k: v for k, v in sd.items() if k in own}, strict=False)
    return m


def _close(got, want):
    assert len(got) == len(want)
    for k, (a, b) in enumerate(zip(got, want)):
        assert a.shape == b.shape, k
        assert (a - b).abs().max().item() <= 1e-5, k


@pytest.mark.parametrize("name", ["tiny", "small64"])
@pytest.mark.parametrize("mean_pooling", [True, False])
def test_oracle_states_match_upstream(name, mean_pooling):
    """VideoMAEModel / ForPreTraining / ForVideoClassification(output_hidden_states=True) of upstream transformers against
    oracle_states, same weights, masked and unmasked."""
    cfgd = dict(vo.TINY if name == "tiny" else ge.SMALL64, use_mean_pooling=mean_pooling)
    cfg = vo.OracleConfig(**cfgd)
    sd = vo.synthetic_cls_state_dict(cfg, 3, 0, 1234)
    sd.update({k: v for k, v in vo.synthetic_state_dict(cfg, 1234).items() if not k.startswith("videomae.")})
    x = vo.synthetic_volume(cfg, 2, 7)
    mask = _mask(2)
    with torch.no_grad():
        want_full = oracle_states(sd, cfg, x)
        want_vis = oracle_states(sd, cfg, x, mask)
        enc = _upstream("VideoMAEModel", cfgd, {k[len("videomae."):]: v for k, v in sd.items() if k.startswith("videomae.")})
        out = enc(x, output_hidden_states=True)
        _close(out.hidden_states, want_full)
        if mean_pooling:  # the last state is last_hidden_state itself
            assert torch.equal(out.hidden_states[-1], out.last_hidden_state)
        _close(enc(x, bool_masked_pos=mask, output_hidden_states=True).hidden_states, want_vis)
        pre = _upstream("VideoMAEForPreTraining", cfgd, sd)
        assert pre(x, mask).hidden_states is None
        _close(pre(x, mask, output_hidden_states=True).hidden_states, want_vis)  # the encoder's states, visible tokens
        tup = pre(x, mask, output_hidden_states=True, return_dict=False)
        assert len(tup) == 3 and isinstance(tup[2], tuple)  # (loss, logits, hidden_states)
        cls = _upstream("VideoMAEForVideoClassification", cfgd, sd, num_labels=3)
        _close(cls(x, output_hidden_states=True).hidden_states, want_full)
        cls.config.output_hidden_states = True  # the config flag, no argument
        _close(cls(x).hidden_states, want_full)
    assert len(want_full) == cfg.num_hidden_layers + 1 and want_vis[0].shape[1] == int((~mask[0]).sum())


def test_oracle_states_end_in_the_encoder_output():
    """oracle_states is consistent with the oracle's encoder (both pooling modes) and its SimMIM variant feeds the decoder."""
    cfg = vo.OracleConfig(**vo.TINY)
    sd = vo.synthetic_state_dict(cfg, 3)
    sd["videomae.embeddings.mask_token"] = 0.2 * torch.randn(1, 1, cfg.hidden_size, generator=torch.Generator().manual_seed(4))
    x = vo.synthetic_volume(cfg, 1, 5)
    mask = _mask(1)
    with torch.no_grad():
        assert torch.equal(oracle_states(sd, cfg, x, mask)[-1], vo.encoder(sd, cfg, x, mask))
        s = oracle_states(sd, cfg, x, mask, simmim=True)
        assert s[0].shape == (1, cfg.num_patches, cfg.hidden_size)
        # the SimMIM states reproduce the SimMIM loss through the rest of the oracle's decoder path
        h = torch.nn.functional.linear(s[-1], sd["encoder_to_decoder.weight"]) + vo.sinusoid_table(cfg.num_patches, cfg.decoder_hidden_size)
        for j in range(cfg.decoder_num_hidden_layers):
            h = vo._layer(h, sd, f"decoder.decoder_layers.{j}.", cfg.decoder_num_attention_heads, cfg.layer_norm_eps)
        h = torch.nn.functional.layer_norm(h[mask].reshape(1, -1, cfg.decoder_hidden_size), (cfg.decoder_hidden_size,),
                                           sd["decoder.norm.weight"], sd["decoder.norm.bias"], 1e-5)
        logits = torch.nn.functional.linear(h, sd["decoder.head.weight"], sd["decoder.head.bias"])
        _, want, _ = vo.pretrain_forward_simmim(sd, cfg, x, mask, "l1")
    assert torch.equal(logits, want)


def test_new_entry_points_reject_bad_arguments_without_a_device():
    ge.build()
    import smb_vision_b200

    lib = smb_vision_b200.load()
    P16, P8 = ctypes.c_void_p(16), ctypes.c_void_p(8)
    # LayerNorm forward with the hidden-state copy
    assert lib.smbv_layernorm_fwd_copy(None, P16, P16, 1e-5, 4, 64, P16, None, None, P16, None) < 0
    assert b"null" in lib.smbv_last_error()
    assert lib.smbv_layernorm_fwd_copy(P16, P16, P16, 1e-5, 4, 64, P16, None, None, P8, None) < 0
    assert b"aligned" in lib.smbv_last_error()
    assert lib.smbv_layernorm_fwd_copy(P16, P16, P16, 1e-5, 4, 6, P16, None, None, P16, None) < 0
    assert b"d % 4" in lib.smbv_last_error()
    # LayerNorm backward with the extra addend
    args = [P16] * 5 + [4, 64, P16, 1, P16, P16, P16]
    assert lib.smbv_layernorm_bwd_add(*args[:4], None, *args[5:], P16, None) < 0 and b"null" in lib.smbv_last_error()
    assert lib.smbv_layernorm_bwd_add(*args, P8, None) < 0 and b"aligned" in lib.smbv_last_error()
    assert lib.smbv_layernorm_bwd_add(*args[:5], 4, 60, *args[7:], P16, None) < 0 and b"d % 8" in lib.smbv_last_error()
    # fused scale + add + bf16 re-cast
    assert lib.smbv_scale_add_recast_f32(None, 8, None, P16, P16, None) < 0 and b"null" in lib.smbv_last_error()
    assert lib.smbv_scale_add_recast_f32(P16, 6, None, P16, P16, None) < 0 and b"multiple of 4" in lib.smbv_last_error()
    assert lib.smbv_scale_add_recast_f32(P16, 8, None, P8, P16, None) < 0 and b"aligned" in lib.smbv_last_error()
    assert lib.smbv_scale_add_recast_f32(P16, 8, None, P16, ctypes.c_void_p(18), None) < 0 and b"aligned" in lib.smbv_last_error()


def test_hidden_state_indices_are_checked():
    from smb_vision_b200.modeling import _check_layers, _want_states

    assert _check_layers((0, 3, 12), 12) == [0, 3, 12]
    with pytest.raises(ValueError, match="outside 0..12"):
        _check_layers((3, 13), 12)
    hc = ge.hf_config(vo.TINY)
    assert not _want_states(None, hc) and _want_states(True, hc)
    hc.output_hidden_states = True
    assert _want_states(None, hc) and not _want_states(False, hc)
