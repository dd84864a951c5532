"""CPU: the C-ABI library builds, loads, and exports every symbol include/smbv_b200.h declares; the host binding
fails loudly (no fallback) without a GPU; the module keeps the reference checkpoint ABI and error behaviour."""
import ctypes
import os
import re

import pytest
import torch

import __graft_entry__ as ge
from oracle import videomae_oracle as vo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    ge.build()
    import smb_vision_b200

    return smb_vision_b200.load()


def header_symbols():
    src = open(os.path.join(ROOT, "include", "smbv_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(smbv_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(lib):
    syms = header_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/smbv_b200.h but not exported"


def test_binding_covers_header(lib):
    from smb_vision_b200 import _lib

    declared = set(header_symbols()) - {"smbv_last_error"}
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)


def test_version_and_arch(lib):
    assert lib.smbv_version() >= 100
    assert lib.smbv_sm_arch() == 100


def test_argument_errors_are_reported_before_launch(lib):
    # negative return + message, no CUDA call needed
    rc = lib.smbv_mask_index(None, 1, 8, None, None, None, None, None)
    assert rc < 0 and b"null" in lib.smbv_last_error()
    rc = lib.smbv_layernorm_fwd(ctypes.c_void_p(16), ctypes.c_void_p(16), ctypes.c_void_p(16), 1e-5, 4, 6, ctypes.c_void_p(16), None, None, None)
    assert rc < 0 and b"d % 4" in lib.smbv_last_error()
    from smb_vision_b200._lib import GemmArgs

    g = GemmArgs()
    g.A = g.W = g.out = 16
    g.M, g.N, g.K, g.lda, g.ldw, g.ldo = 128, 100, 64, 64, 64, 100
    assert lib.smbv_gemm_bf16(ctypes.byref(g), None) < 0 and b"multiple of 32" in lib.smbv_last_error()
    P16 = ctypes.c_void_p(16)
    assert lib.smbv_flash_attn_fwd_ex(P16, P16, P16, 1, 1, 128, 0.125, P16, None, 1, None, 0, None) < 0
    assert b"variant" in lib.smbv_last_error()
    # V-JEPA entry points (SURVEY.md §8f rank 4)
    assert lib.smbv_rope3d(P16, None, 2, 1, 2, 8, 60, 4, 4, 0, None) < 0 and b"multiple of 8" in lib.smbv_last_error()
    assert lib.smbv_rope3d(None, None, 2, 1, 2, 8, 64, 4, 4, 0, None) < 0 and b"null" in lib.smbv_last_error()
    assert lib.smbv_rope3d(P16, None, 2, 1, 2, 8, 64, 4, 100000, 0, None) < 0 and b"max_pos" in lib.smbv_last_error()
    assert lib.smbv_gather_rows_f32(P16, P16, 1, 8, 4, 6, P16, None) < 0 and b"multiple of 4" in lib.smbv_last_error()
    assert lib.smbv_l1_loss_f32(P16, P16, 0, P16, P16, None, 1.0, None) < 0 and b"positive" in lib.smbv_last_error()
    assert lib.smbv_l1_loss_f32(P16, None, 8, P16, P16, None, 1.0, None) < 0 and b"null" in lib.smbv_last_error()
    assert lib.smbv_l1_workspace_floats() >= 148


def test_no_cpu_fallback():
    from smb_vision_b200 import SmbvError, ops

    with pytest.raises(SmbvError):
        ops.layernorm_fwd(torch.zeros(4, 8), torch.ones(8), torch.zeros(8), 1e-5)
    with pytest.raises(SmbvError):
        ops.gemm(torch.zeros(4, 8, dtype=torch.bfloat16), torch.zeros(32, 8, dtype=torch.bfloat16))
    with pytest.raises(SmbvError):
        ops.rope3d_(torch.zeros(1, 2, 8, 64, dtype=torch.bfloat16), 4)
    with pytest.raises(SmbvError):
        ops.gather_rows(torch.zeros(1, 8, 4), torch.zeros(1, 2, dtype=torch.int32))
    with pytest.raises(SmbvError):
        ops.l1_loss(torch.zeros(8), torch.zeros(8))


def test_missing_library_fails_loudly(monkeypatch):
    from smb_vision_b200 import _lib

    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libsmbv_b200.so")
    with pytest.raises(_lib.SmbvError, match="not built"):
        _lib.load()


def test_product_package_never_imports_oracle():
    pkg = os.path.join(ROOT, "smb-vision_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt, f


@pytest.mark.parametrize("cfgd", [vo.TINY, ge.SMALL64, {}, dict(ge.SMALL64, qkv_bias=False, use_mean_pooling=False)])
def test_checkpoint_abi_matches_reference(cfgd):
    """state-dict keys/shapes == the reference's (SURVEY.md §8b), so load_state_dict(strict=True) works both ways."""
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining

    ocfg = vo.OracleConfig(**cfgd)
    full = {k: getattr(ocfg, k) for k in ocfg.__dataclass_fields__}
    with torch.device("meta"):
        m = B200VideoMAEForPreTraining(ge.hf_config(full))
    got = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    want = {k: tuple(v) for k, v in vo.param_shapes(ocfg).items()}
    assert got == want
    if cfgd and "qkv_bias" in cfgd:  # the config variants against the upstream class itself
        import transformers

        with torch.device("meta"):
            up = transformers.VideoMAEForPreTraining(ge.hf_config(full))
        assert got == {k: tuple(v.shape) for k, v in up.state_dict().items()}
    if not cfgd:
        assert sum(v.numel() for v in m.state_dict().values()) == 97_161_088  # SURVEY.md §8 a16
        assert sum(v.numel() for v in m.videomae.state_dict().values()) == 88_191_744


def test_reference_error_behaviour():
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining

    m = B200VideoMAEForPreTraining(ge.hf_config(ge.SMALL64))
    x = torch.zeros(1, 96, 1, 96, 96)
    with pytest.raises(ValueError, match="channel dimension"):  # modeling_videomae.py:181-184
        m.videomae(x.repeat(1, 1, 3, 1, 1))
    with pytest.raises(ValueError, match="doesn't match model"):  # :185-188
        m.videomae(x[..., :80])
    with pytest.raises(ValueError, match="boolean mask"):  # :807-808
        m(x, None)
    with pytest.raises(ValueError):
        m(x, torch.zeros(1, 216, dtype=torch.bool), head_mask=torch.ones(2))
    ragged = torch.zeros(2, 216, dtype=torch.bool)
    ragged[0, :8] = True
    with pytest.raises(RuntimeError):  # reshape failure of :137
        m(x.repeat(2, 1, 1, 1, 1), ragged)


def test_classification_checkpoint_abi_and_errors():
    """B200VideoMAEForVideoClassification: same keys/shapes as the reference's class (fc_norm.*, classifier.* with the
    additional-feature columns, modeling_videomae.py:925-937), the upstream class without features, and its ValueErrors."""
    import transformers
    from smb_vision_b200.modeling import B200VideoMAEForVideoClassification

    ocfg = vo.OracleConfig(**ge.SMALL64)
    hc = ge.hf_config(ge.SMALL64)
    hc.num_labels, hc.additional_features_size = 3, 2
    m = B200VideoMAEForVideoClassification(hc)
    want = {k: tuple(v.shape) for k, v in vo.synthetic_cls_state_dict(ocfg, 3, 2).items()}
    assert {k: tuple(v.shape) for k, v in m.state_dict().items()} == want
    hc0 = ge.hf_config(ge.SMALL64)
    hc0.num_labels = 4
    up = transformers.VideoMAEForVideoClassification(hc0)
    m0 = B200VideoMAEForVideoClassification(hc0)
    assert {k: tuple(v.shape) for k, v in m0.state_dict().items()} == {k: tuple(v.shape) for k, v in up.state_dict().items()}
    m0.load_state_dict(up.state_dict(), strict=True)
    x = torch.zeros(1, 96, 1, 96, 96)
    with pytest.raises(ValueError, match="Expected additional_features of size 2"):  # :983-986
        m(x, additional_features=torch.zeros(1, 5))
    with pytest.raises(ValueError, match="additional_features_size"):  # :981-982
        m0(x, additional_features=torch.zeros(1, 2))
    with pytest.raises(ValueError, match="channel dimension"):
        m(x.repeat(1, 1, 3, 1, 1), additional_features=torch.zeros(1, 2))


def test_attention_interface_registers_and_refuses_unsupported():
    import smb_vision_b200.attention_interface as ai
    from smb_vision_b200 import SmbvError
    from transformers.modeling_utils import ALL_ATTENTION_FUNCTIONS

    name = ai.register()
    assert ALL_ATTENTION_FUNCTIONS.get_interface(name, None) is ai.b200_flash_attention
    q = torch.zeros(1, 2, 8, 64)
    with pytest.raises(SmbvError, match="attention_mask"):
        ai.b200_flash_attention(None, q, q, q, attention_mask=torch.zeros(1))
    with pytest.raises(SmbvError, match="causal"):
        ai.b200_flash_attention(None, q, q, q, is_causal=True)
    with pytest.raises(SmbvError, match="head_dim"):
        ai.b200_flash_attention(None, q[..., :48], q, q)  # head_dim 48: neither the tcgen05 (64) nor the small-head (8/16/32) kernels
    with pytest.raises(SmbvError, match="CUDA tensor"):  # no CPU fallback
        ai.b200_flash_attention(None, q, q, q)


def test_from_pretrained_and_save_pretrained_round_trip_with_upstream(tmp_path):
    """checkpoint directories are interchangeable with the reference's PreTrainedModel classes, both directions
    (src/run_mim.py:345-357 loads with from_pretrained; HF Trainer saves with save_pretrained)."""
    import transformers
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining, B200VideoMAEForVideoClassification, B200VideoMAEModel

    hc = ge.hf_config(ge.SMALL64)
    up = transformers.VideoMAEForPreTraining(hc)
    up.save_pretrained(tmp_path / "up")
    m = B200VideoMAEForPreTraining.from_pretrained(tmp_path / "up")
    assert m.loading_info["missing_keys"] == [] and m.loading_info["unexpected_keys"] == []
    assert m.loading_info["attn_implementation"] == "b200_tcgen05"
    assert m.config.image_size == 96 and m.config.num_frames == 96
    for k, v in up.state_dict().items():
        assert torch.equal(m.state_dict()[k], v), k
    m.save_pretrained(tmp_path / "ours")
    back = transformers.VideoMAEForPreTraining.from_pretrained(tmp_path / "ours")
    for k, v in up.state_dict().items():
        assert torch.equal(back.state_dict()[k], v), k
    # fine-tuning from the MIM checkpoint: encoder loaded, head freshly initialised, decoder ignored (HF semantics)
    hcc = ge.hf_config(ge.SMALL64)
    hcc.num_labels, hcc.additional_features_size = 3, 2
    c = B200VideoMAEForVideoClassification.from_pretrained(tmp_path / "up", config=hcc)
    assert sorted(c.loading_info["missing_keys"]) == ["classifier.bias", "classifier.weight", "fc_norm.bias", "fc_norm.weight"]
    assert all(k.startswith(("decoder.", "encoder_to_decoder", "mask_token")) for k in c.loading_info["unexpected_keys"])
    assert torch.equal(c.videomae.encoder.layer[1].output.dense.weight, up.videomae.encoder.layer[1].output.dense.weight)
    enc = B200VideoMAEModel.from_pretrained(tmp_path / "up")  # bare encoder from a head-model checkpoint
    assert not enc.loading_info["missing_keys"]
    with pytest.raises(OSError):
        B200VideoMAEModel.from_pretrained("standardmodelbio/smb-vision-base")  # no hub access
    # the keyword arguments the reference scripts pass (src/run_mim.py:345-357, run_inspect.py:106-111) are honoured:
    # every attention back-end name maps to the tcgen05 kernel, an unknown one is an error; torch_dtype=bfloat16 holds the
    # checkpoint in bf16 (values rounded, fp32 containers) and returns outputs in bf16
    B200VideoMAEModel.from_pretrained(tmp_path / "up", attn_implementation="flash_attention_2", torch_dtype=torch.float32)
    with pytest.raises(ValueError, match="attn_implementation"):
        B200VideoMAEModel.from_pretrained(tmp_path / "up", attn_implementation="paged")
    with pytest.raises(ValueError, match="torch_dtype"):
        B200VideoMAEModel.from_pretrained(tmp_path / "up", torch_dtype=torch.float64)
    hb = B200VideoMAEModel.from_pretrained(tmp_path / "up", torch_dtype=torch.bfloat16, attn_implementation="sdpa")
    assert hb._out_dtype == torch.bfloat16 and hb.dtype == torch.float32
    for k, v in up.videomae.state_dict().items():
        assert torch.equal(hb.state_dict()[k], v.bfloat16().float()), k
    assert B200VideoMAEModel.from_pretrained(tmp_path / "up", dtype="bfloat16")._out_dtype == torch.bfloat16
    # the PreTrainedModel surface HF Trainer touches
    m.gradient_checkpointing_enable()
    assert m.supports_gradient_checkpointing and m.device.type == "cpu" and m.dtype == torch.float32
    assert m.num_parameters() == up.num_parameters() and m.get_input_embeddings() is m.videomae.embeddings.patch_embeddings
