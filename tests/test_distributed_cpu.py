"""CPU, world_size 2, gloo: the N>1 host logic — volume sharding (no collective) and the bucketed gradient reducer
(fp32 and bf16 wire formats) that the data-parallel MIM step drives from backward."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import __graft_entry__ as ge


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, wire, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from smb_vision_b200.distributed import BucketReducer, shard_volumes
        from smb_vision_b200.modeling import B200VideoMAEForPreTraining
        from smb_vision_b200.training import GradArena

        model = B200VideoMAEForPreTraining(ge.hf_config(ge.SMALL64))
        arena = GradArena(model, "cpu")
        g = torch.Generator().manual_seed(100 + rank)
        arena.flat.copy_(torch.randn(arena.flat.numel(), generator=g))
        mine = arena.flat.clone()
        red = BucketReducer(arena.flat, arena.bucket_bounds, wire_dtype=wire)
        red.overlap = (rank_overlap := os.environ.get("SMBV_TEST_DP_OVERLAP", "1") != "0")  # False: one exchange at finish()
        for i in range(len(arena.bucket_bounds) - 1):  # the order backward completes them
            red.reduce_bucket(i)
        red.finish()
        gathered = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(gathered, mine)
        if wire == torch.float32:
            want = sum(gathered) / world
            err = (arena.flat - want).abs().max().item()
        else:
            want = sum(t.to(torch.bfloat16).float() for t in gathered) / world
            err = ((arena.flat - want).abs() / (want.abs() + 1.0)).max().item()
        shard = shard_volumes(list(range(11)), rank, world)
        q.put((rank, err, shard, arena.views["decoder.head.bias"].data_ptr() == arena.flat.data_ptr() + 4 * arena.offsets["decoder.head.bias"][0]))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("overlap", [True, False])
@pytest.mark.parametrize("wire", [torch.float32, torch.bfloat16])
def test_bucket_reducer_world2_gloo(wire, overlap, monkeypatch):
    monkeypatch.setenv("SMBV_TEST_DP_OVERLAP", "1" if overlap else "0")  # (inherited by the spawned ranks)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, wire, q)) for r in range(2)]
    [p.start() for p in procs]
    res = sorted(q.get(timeout=180) for _ in range(2))
    [p.join(timeout=60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    tol = 1e-6 if wire == torch.float32 else 1e-2  # bf16 wire: one rounding of the summed value
    for rank, err, shard, view_ok in res:
        assert err <= tol and view_ok
    assert res[0][2] == [0, 1, 2, 3, 4, 5] and res[1][2] == [6, 7, 8, 9, 10]  # contiguous chunks, run_inspect.py:218-221


def test_shard_volumes_edges():
    from smb_vision_b200.distributed import shard_volumes

    assert shard_volumes([], 0, 4) == []
    assert [shard_volumes(list(range(3)), r, 4) for r in range(4)] == [[0], [1], [2], []]
    assert sum((shard_volumes(list(range(17)), r, 8) for r in range(8)), []) == list(range(17))
    with pytest.raises(ValueError):
        shard_volumes([1], 2, 2)


def test_grad_arena_layout():
    """Buckets are contiguous, aligned (TMA operand bases), cover every parameter once, in backward-completion order;
    [q_bias; zero pad; v_bias] and [Wq; Wk; Wv] are single views (the fused QKV GEMM's bias / weight)."""
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining, B200VideoMAEForVideoClassification
    from smb_vision_b200.training import ALIGN, PAD_SUFFIX, ArenaLayout, GradArena, order_groups

    model = B200VideoMAEForPreTraining(ge.hf_config(ge.SMALL64))
    arena = GradArena(model, "cpu")
    names = [n for g in order_groups(model) for n in g]
    real = [n for n in names if not n.endswith(PAD_SUFFIX)]
    assert sorted(real) == sorted(n for n, _ in model.named_parameters()) and len(set(names)) == len(names)
    prev_end = 0
    for n in names:
        off, cnt = arena.offsets[n]
        assert off % ALIGN == 0 and off >= prev_end
        prev_end = off + cnt
    assert arena.bucket_bounds[0] == 0 and arena.bucket_bounds[-1] == arena.flat.numel()
    assert names[0] == "decoder.head.weight" and names[-1].startswith("videomae.embeddings.patch_embeddings")
    pre = "videomae.encoder.layer.0."
    qkv = arena.fused_qkv(pre)
    assert qkv.shape == (3 * 128, 128) and qkv.data_ptr() == arena.views[pre + "attention.attention.query.weight"].data_ptr()
    assert qkv[256:].data_ptr() == arena.views[pre + "attention.attention.value.weight"].data_ptr()
    b = arena.fused_qkv_bias(pre)
    assert b.shape == (384,) and b.data_ptr() == arena.views[pre + "attention.attention.q_bias"].data_ptr()
    assert b[256:].data_ptr() == arena.views[pre + "attention.attention.v_bias"].data_ptr()
    # weight-decay segments: Trainer.get_decay_parameter_names (no decay for LayerNorm weights and *bias*)
    lay = arena.layout
    starts, flags = lay.decay_segments()
    assert starts[0] == 0 and starts == sorted(starts) and all(a != b for a, b in zip(flags, flags[1:]))

    def nodecay(name):
        o = lay.offsets[name][0] // 4
        k = max(i for i, s0 in enumerate(starts) if s0 <= o)
        return flags[k]

    assert nodecay("decoder.head.weight") == 0 and nodecay("mask_token") == 0 and nodecay(pre + "attention.attention.key.weight") == 0
    for n in ("decoder.head.bias", "decoder.norm.weight", pre + "layernorm_before.weight", pre + "attention.attention.q_bias",
              pre + "attention.attention.v_bias", pre + "output.dense.bias"):
        assert nodecay(n) == 1, n
    # classification model: classifier + fc_norm first
    hc = ge.hf_config(ge.SMALL64)
    hc.num_labels, hc.additional_features_size = 3, 2
    lc = ArenaLayout(B200VideoMAEForVideoClassification(hc))
    assert lc.order[0] == "classifier.weight" and lc.offsets["classifier.weight"] == (0, 3 * 130)


def _decay_models():
    import transformers
    from transformers import VJEPA2Config

    from smb_vision_b200.modeling import B200VideoMAEForPreTraining, B200VideoMAEForVideoClassification
    from smb_vision_b200.vjepa import B200VJEPA2Model

    def cls(mean_pooling):
        hc = ge.hf_config(ge.SMALL64)
        hc.num_labels, hc.additional_features_size, hc.use_mean_pooling = 3, 2, mean_pooling
        return B200VideoMAEForVideoClassification(hc)

    vc = VJEPA2Config(patch_size=16, crop_size=64, frames_per_clip=64, tubelet_size=16, in_chans=1, hidden_size=128, num_attention_heads=2,
                      num_hidden_layers=2, pred_hidden_size=64, pred_num_attention_heads=2, pred_num_hidden_layers=2, pred_num_mask_tokens=2)
    return {"videomae-pretraining": lambda: B200VideoMAEForPreTraining(ge.hf_config(ge.SMALL64)),
            "classification-mean-pooling": lambda: cls(True), "classification-cls-token": lambda: cls(False),
            "vjepa": lambda: B200VJEPA2Model(vc), "upstream-vjepa": lambda: transformers.VJEPA2Model(vc),
            "upstream-videomae-pretraining": lambda: transformers.VideoMAEForPreTraining(ge.hf_config(ge.SMALL64))}


@pytest.mark.parametrize("kind", list(_decay_models()))
def test_decay_segments_match_trainer(kind):
    """FusedAdamW's weight-decay set is transformers Trainer's: flag 0 exactly for the names
    Trainer.get_decay_parameter_names returns (which excludes every nn.LayerNorm parameter, so V-JEPA's norm1 / norm2
    weights too), flag 1 for the rest and for the k_bias_pad entries."""
    from transformers import Trainer

    from smb_vision_b200.training import PAD_SUFFIX, ArenaLayout

    model = _decay_models()[kind]()
    lay = ArenaLayout(model)
    starts, flags = lay.decay_segments()
    assert starts[0] == 0 and starts == sorted(starts) and all(a != b for a, b in zip(flags, flags[1:]))
    decay = set(Trainer.get_decay_parameter_names(None, model))
    assert decay and decay <= set(lay.shapes)

    def flag(name):
        o = lay.offsets[name][0] // 4
        return flags[max(i for i, s0 in enumerate(starts) if s0 <= o)]

    got = {n: flag(n) for n in lay.order}
    assert all(got[n] == 1 for n in lay.order if n.endswith(PAD_SUFFIX))
    wrong = sorted(n for n in lay.shapes if got[n] != (0 if n in decay else 1))
    assert not wrong, wrong
    frozen = sorted(lay.shapes)[::3]
    starts_f, flags_f = lay.decay_segments(frozen)
    o = lay.offsets[frozen[0]][0] // 4
    assert flags_f[max(i for i, s0 in enumerate(starts_f) if s0 <= o)] == 2


def test_cosine_schedule_matches_transformers():
    from transformers import get_cosine_schedule_with_warmup

    from smb_vision_b200.optim import cosine_with_warmup

    p = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.SGD([p], lr=5e-5)
    sch = get_cosine_schedule_with_warmup(opt, num_warmup_steps=7, num_training_steps=100)
    for step in range(100):
        assert abs(opt.param_groups[0]["lr"] - cosine_with_warmup(step, 5e-5, 7, 100)) < 1e-12, step
        opt.step()
        sch.step()


def _arena_worker(rank, world, port, wire, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from transformers import VJEPA2Config

        from smb_vision_b200.training import GradArena
        from smb_vision_b200.vjepa import B200VJEPA2Model

        torch.manual_seed(0)
        model = B200VJEPA2Model(VJEPA2Config(patch_size=16, crop_size=64, frames_per_clip=64, tubelet_size=16, in_chans=1, hidden_size=128,
                                             num_attention_heads=2, num_hidden_layers=2), with_predictor=False)
        arena = GradArena(model, "cpu")  # generic layout (reverse registration order, bucketed)
        arena.assign_to_params()
        for i, p in enumerate(model.parameters()):  # what autograd would have accumulated on this rank
            p.grad.fill_(float(rank + 1) * (i + 1))
        arena.all_reduce(wire_dtype=wire)
        want = [1.5 * (i + 1) for i, _ in enumerate(model.parameters())]
        err = max(float((p.grad - w).abs().max()) / w for p, w in zip(model.parameters(), want))
        q.put((rank, err, len(arena.bucket_bounds) - 1))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("wire", [torch.float32, torch.bfloat16])
def test_grad_arena_all_reduce_world2_gloo(wire):
    """GradArena.all_reduce (the data-parallel step of the autograd-driven V-JEPA routes): mean over two ranks of every
    parameter's gradient, through the flat arena views."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_arena_worker, args=(r, 2, port, wire, q)) for r in range(2)]
    [p.start() for p in procs]
    res = sorted(q.get(timeout=180) for _ in range(2))
    [p.join(timeout=60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    for rank, err, nb in res:
        assert err <= (1e-6 if wire == torch.float32 else 4e-3) and nb >= 1


def test_grad_arena_all_reduce_single_process_is_a_noop():
    from smb_vision_b200.modeling import B200VideoMAEForPreTraining
    from smb_vision_b200.training import GradArena

    arena = GradArena(B200VideoMAEForPreTraining(ge.hf_config(ge.SMALL64)), "cpu")
    arena.flat.fill_(2.0)
    arena.all_reduce()
    assert float(arena.flat.min()) == 2.0 and float(arena.flat.max()) == 2.0


def test_graph_step_input_flattening_and_signature():
    """DataParallelStep's CUDA-graph path keys its graphs on the input signature and feeds them through static buffers: the
    flattening of (vol, mask_pack) / (vol, feats, labels) must keep structure, order and the non-tensor leaves (host logic only)."""
    import torch

    from smb_vision_b200.training import DataParallelStep

    vol = torch.zeros(1, 4, 8, 8)
    pack = (torch.zeros(1, 6, dtype=torch.uint8), torch.zeros(1, 6, dtype=torch.int32), torch.ones(1, 6, dtype=torch.int32), torch.zeros(1, 6, dtype=torch.int32), 2, 4)
    leaves, rebuild, key = DataParallelStep._flatten(vol, (pack,))
    assert len(leaves) == 5 and leaves[0] is vol and leaves[3] is pack[2]
    repl = [t.clone() + 1 for t in leaves]
    args = rebuild(repl)
    assert args[0] is repl[0] and isinstance(args[1], tuple) and args[1][4:] == (2, 4) and args[1][2] is repl[3]
    # same shapes / dtypes / ints -> same key; another mask count or another volume shape -> another graph
    _, _, key2 = DataParallelStep._flatten(vol.clone(), (tuple(t.clone() if isinstance(t, torch.Tensor) else t for t in pack),))
    assert key2 == key
    _, _, key3 = DataParallelStep._flatten(vol, (pack[:4] + (3, 3),))
    _, _, key4 = DataParallelStep._flatten(torch.zeros(2, 4, 8, 8), (pack,))
    assert key3 != key and key4 != key
    # classification inputs: (vol, feats, labels)
    leaves_c, rebuild_c, _ = DataParallelStep._flatten(vol, (torch.zeros(1, 2), torch.zeros(1, dtype=torch.long)))
    assert len(leaves_c) == 3 and len(rebuild_c(leaves_c)) == 3


def test_side_queue_without_a_gpu_runs_inline_in_order():
    """training.SideQueue (second stream for the weight / bias gradients and the data-parallel bucket hook): on a CPU device — and with
    SMBV_WGRAD_STREAM=0 — it is a pass-through: work runs at the call, bucket hooks fire at block_done, in program order."""
    from smb_vision_b200.training import SideQueue

    sq, log = SideQueue("cpu"), []
    assert not sq.enabled and sq.mark() is None
    sq.run(None, lambda: log.append("w0"), torch.zeros(1))
    sq.block_done(lambda: log.append("b0"))
    sq.run(None, lambda: log.append("w1"))
    sq.block_done(None)
    sq.block_done(lambda: log.append("b2"))
    sq.finish()
    assert log == ["w0", "b0", "w1", "b2"] and not sq.keep and not sq.marks


def test_bucket_reducer_world1_is_a_no_op():
    from smb_vision_b200.distributed import BucketReducer

    flat = torch.arange(12, dtype=torch.float32)
    red = BucketReducer(flat, [0, 4, 12], group=False)
    red.reduce_bucket(0), red.reduce_bucket(1), red.finish()
    assert red.world == 1 and not red.pending and torch.equal(flat, torch.arange(12, dtype=torch.float32))
