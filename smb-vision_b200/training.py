"""MIM training step on the sm_100a kernels: forward with saved activations + hand-scheduled backward.

Replaces autograd over the reference graph (``VideoMAEForPreTraining.forward`` + ``loss.backward()``,
modeling_videomae.py:753-908) and the DDP gradient all-reduce HF ``Trainer`` triggers
(SURVEY.md §2c/§8e).  Gradients land in ONE flat fp32 arena laid out in backward-completion order, so
data-parallel buckets are contiguous slices that can be all-reduced (bf16 on the wire, NCCL) while the rest
of backward is still running.
"""
from __future__ import annotations

import re
from typing import Callable, Dict, List, Optional, Tuple

import torch

from . import ops


# ----------------------------------------------------------------------------------------------
# second stream for the gradient kernels that nothing downstream waits for
# ----------------------------------------------------------------------------------------------
_side_streams: Dict[str, "torch.cuda.Stream"] = {}


class SideQueue:
    """Weight- and bias-gradient kernels of the backward pass on a SECOND stream.

    The backward's critical path is dgrad -> LayerNorm backward -> attention backward -> dgrad ...; the weight-gradient GEMMs and
    the bias column sums (a third of the backward's GEMM time plus ~80 small bandwidth kernels per step) only feed the optimiser.
    Queued on a side stream they run beside the critical path: their CTAs take the SMs a persistent one-CTA-per-SM kernel
    leaves idle in its partial last round, and the column sums run under tensor-bound kernels.  (autograd over the reference graph
    has the same freedom; the reference leaves it to the CUDA caching allocator's single stream.)

    `mark()` records "everything queued so far on the main stream" BEFORE the next critical-path kernel is launched, `run(mark, fn,
    *tensors)` queues fn's launches behind that mark on the side stream and keeps `tensors` (what those launches read) alive,
    `block_done(cb)` closes a block: `cb` (the data-parallel bucket hook: cast + all-reduce launch) is queued on the side stream
    behind everything the block launched on either stream, and the main stream joins the side work of the PREVIOUS block (queued
    a whole block ago, so the join does not stall) and releases its tensors; `finish()` joins everything.
    SMBV_WGRAD_STREAM=0 keeps every launch on the main stream (A/B switch).  Works under CUDA-graph capture: the side stream
    forks from and joins the capturing stream through events."""

    def __init__(self, device):
        import os

        self.enabled = os.environ.get("SMBV_WGRAD_STREAM", "1") != "0" and torch.device(device).type == "cuda"
        self.cur = torch.cuda.current_stream(device) if self.enabled else None
        if self.enabled:
            key = str(device)
            if key not in _side_streams:
                _side_streams[key] = torch.cuda.Stream(device)
            self.side = _side_streams[key]
        self.keep: list = []
        self.marks: list = []
        self.queued = False  # side work queued since the last block_done

    def mark(self):
        if not self.enabled:
            return None
        ev = torch.cuda.Event()
        ev.record(self.cur)
        return ev

    def run(self, mark, fn: Callable[[], None], *tensors) -> None:
        if not self.enabled:
            fn()
            return
        self.side.wait_event(mark)
        with torch.cuda.stream(self.side):
            fn()
        self.keep.extend(tensors)
        self.queued = True

    def _settle(self, m) -> None:
        ev, keep = m
        self.cur.wait_event(ev)
        keep.clear()

    def block_done(self, cb: Optional[Callable[[], None]] = None) -> None:
        if not self.enabled:
            if cb is not None:
                cb()
            return
        if cb is not None:
            # the block's gradients are complete once the main stream's work so far AND the side queue's have run: `cb` (cast to
            # the wire format + all-reduce launch of the data-parallel bucket) goes onto the side stream behind both, so the
            # critical path carries neither the cast nor a wait
            self.side.wait_event(self.mark())
            with torch.cuda.stream(self.side):
                cb()
        ev = torch.cuda.Event()
        ev.record(self.side)
        self.marks.append((ev, self.keep))
        self.keep, self.queued = [], False
        while len(self.marks) > 1:
            self._settle(self.marks.pop(0))

    def finish(self) -> None:
        if not self.enabled:
            return
        if self.queued:
            self.block_done(None)
        while self.marks:
            self._settle(self.marks.pop(0))


# ----------------------------------------------------------------------------------------------
# flat arenas: ONE layout shared by the gradients, the fp32 master parameters, their bf16 operand copies and the
# Adam moments
# ----------------------------------------------------------------------------------------------
ALIGN = 64  # elements: 256 B in the fp32 arenas, 128 B in the bf16 one (TMA operand bases need 16 B)
PAD_SUFFIX = "k_bias_pad"  # pseudo entry between q_bias and v_bias: the constant zero k bias of reference :261
# transformers Trainer.get_decay_parameter_names: no weight decay for parameters of nn.LayerNorm modules or for names (lower
# case) matching one of these
NO_DECAY_PATTERNS = re.compile(r"bias|layernorm|rmsnorm|(?:^|\.)norm(?:$|\.)|_norm(?:$|\.)")


class ArenaLayout:
    """Offsets of every parameter in a flat buffer, ordered as backward finishes them (decoder head first, patch
    embedding last); buckets (= `order_groups`) are contiguous slices.  Between `q_bias` and `v_bias` of every block
    sits a zero pad of the same size so that [q_bias; 0; v_bias] — the bias of the fused QKV GEMM — is ONE view."""

    def __init__(self, model):
        self.shapes: Dict[str, torch.Size] = {k: p.shape for k, p in model.named_parameters()}
        self.layernorm_params = {f"{mn}.{pn}" if mn else pn for mn, m in model.named_modules() if isinstance(m, torch.nn.LayerNorm)
                                 for pn, _ in m.named_parameters()}
        groups = order_groups(model)
        real = [n for g in groups for n in g if not n.endswith(PAD_SUFFIX)]
        assert set(real) == set(self.shapes) and len(real) == len(self.shapes), set(real) ^ set(self.shapes)
        self.offsets: Dict[str, Tuple[int, int]] = {}
        self.bucket_bounds: List[int] = [0]
        self.order: List[str] = []
        off = end = 0  # `end` = first element after the previous entry (before alignment padding)
        tight = ("query.weight", "key.weight", "q_bias", PAD_SUFFIX)  # the NEXT entry follows these without padding
        prev = ""
        for group in groups:
            for name in group:
                n = self.shapes[name[:-len(PAD_SUFFIX)] + "q_bias"].numel() if name.endswith(PAD_SUFFIX) else self.shapes[name].numel()
                if prev.endswith(tight):  # [Wq; Wk; Wv] and [q_bias; 0; v_bias] must be single contiguous views
                    assert end % 8 == 0, f"{name}: fused Q/K/V views need sizes that are multiples of 8 elements"
                    off = end
                self.offsets[name] = (off, n)
                self.order.append(name)
                end = off + n
                off = (end + ALIGN - 1) // ALIGN * ALIGN
                prev = name
            self.bucket_bounds.append(off)
        self.total = off

    def views(self, flat: torch.Tensor) -> Dict[str, torch.Tensor]:
        return {k: flat[o:o + n].view(self.shapes[k]) for k, (o, n) in self.offsets.items() if k in self.shapes}

    def decay_segments(self, frozen=()):
        """(start4 int32[], flag uint8[]) for smbv_adamw_step: flag 1 = weight decay off, with the rule of transformers
        Trainer.get_decay_parameter_names (every parameter of an nn.LayerNorm module, and every name matching
        NO_DECAY_PATTERNS, e.g. "bias", "layernorm", ".norm.", "_norm."; the k_bias_pad entries count as biases), flag 2 =
        frozen (`frozen`: names with requires_grad=False — neither updated nor decayed, as torch.optim skips them); adjacent
        equal flags merged."""
        starts, flags = [], []
        frozen = set(frozen)
        for name in self.order:
            nd = 1 if (name in self.layernorm_params or NO_DECAY_PATTERNS.search(name.lower())) else 0
            if name in frozen:
                nd = 2
            if not flags or flags[-1] != nd:
                starts.append(self.offsets[name][0] // 4)
                flags.append(nd)
        return starts, flags


class GradArena:
    """Flat fp32 gradient buffer (layout: `ArenaLayout`)."""

    def __init__(self, model, device, layout: Optional[ArenaLayout] = None):
        self.layout = layout or ArenaLayout(model)
        self.named: Dict[str, torch.nn.Parameter] = dict(model.named_parameters())
        self.offsets, self.bucket_bounds = self.layout.offsets, self.layout.bucket_bounds
        self.flat = torch.zeros(self.layout.total, dtype=torch.float32, device=device)
        self.views = self.layout.views(self.flat)

    def zero(self):
        self.flat.zero_()

    def g(self, name):
        return self.views[name]

    def fused_qkv(self, prefix):
        """query/key/value weights are adjacent in the arena: one [3d, d] view for the fused wgrad."""
        q = prefix + "attention.attention.query.weight"
        o, n = self.offsets[q]
        d = self.named[q].shape[0]
        return self.flat[o:o + 3 * n].view(3 * d, d)

    def fused_qkv_bias(self, prefix):
        """[q_bias; k pad; v_bias] as one [3d] view (the K third stays zero: smbv_colsum_heads_bf16 skips it)."""
        o, n = self.offsets[prefix + "attention.attention.q_bias"]
        return self.flat[o:o + 3 * n]

    def assign_to_params(self):
        for k, p in self.named.items():
            p.grad = self.views[k]

    def all_reduce(self, wire_dtype=torch.bfloat16, process_group=None) -> None:
        """Data-parallel mean of the whole arena over the ranks, after backward — for modules differentiated by torch
        autograd (the V-JEPA routes of examples/train_vjepa.py; the reference gets this from accelerate's DDP wrapper,
        scripts/training/run_vjepa.sh:16).  One bucketed all-reduce (bf16 on the wire by default, like
        `DataParallelStep`, which additionally overlaps the buckets with backward).  No-op for a single process."""
        import torch.distributed as dist

        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(process_group) == 1:
            return
        if getattr(self, "_reducer", None) is None:
            from .distributed import BucketReducer

            cd = cu = None
            if self.flat.is_cuda and wire_dtype == torch.bfloat16:  # the library's cast kernels (bf16 <-> fp32 with the 1/world scale)
                cd = lambda src, dst: ops.cast_bf16(src, out=dst)
                cu = ops.cast_f32_scaled
            self._reducer = BucketReducer(self.flat, self.bucket_bounds, group=process_group, wire_dtype=wire_dtype, cast_down=cd, cast_up=cu)
        for i in range(len(self.bucket_bounds) - 1):
            self._reducer.reduce_bucket(i)
        self._reducer.finish()


class ParamArena:
    """fp32 master parameters of `model` moved into one flat buffer (every `p.data` becomes a view of it, so state-dict
    keys/shapes, `load_state_dict` and checkpoints are unchanged) + the bf16 operand copy of the whole buffer that the
    tcgen05 GEMMs read.  `model.packed()` then hands out views of these two buffers instead of re-packing per tensor, and
    `FusedAdamW` updates both in one pass."""

    def __init__(self, model, layout: Optional[ArenaLayout] = None, with_bf16: Optional[bool] = None):
        self.layout = layout or ArenaLayout(model)
        self.model = model
        dev = next(model.parameters()).device
        self.flat = torch.zeros(self.layout.total, dtype=torch.float32, device=dev)
        self.views = self.layout.views(self.flat)
        with torch.no_grad():
            for k, p in model.named_parameters():
                if p.dtype != torch.float32:
                    raise ValueError(f"ParamArena holds fp32 master parameters; {k} is {p.dtype}")
                self.views[k].copy_(p.data)
                p.data = self.views[k]
        own = hasattr(model, "videomae")  # our modules read bf16 operand views; foreign modules (autocast) do not
        self.bf16 = torch.empty(self.layout.total, dtype=torch.bfloat16, device=dev) if (own if with_bf16 is None else with_bf16) else None
        self.sync_bf16()
        if own:
            for m in (model, getattr(model, "videomae", None)):
                if m is not None:
                    m._arena, m._packed, m._packed_sig = self, None, None
        else:
            model._arena = self

    def sync_bf16(self):
        """re-derive the bf16 operand copy from the fp32 masters (after load_state_dict / any torch-side edit)."""
        if self.bf16 is not None:
            ops.cast_bf16(self.flat, out=self.bf16)

    def w16(self, name) -> torch.Tensor:
        o, n = self.layout.offsets[name]
        return self.bf16[o:o + n].view(self.layout.shapes[name])

    def wqkv16(self, prefix) -> torch.Tensor:
        q = prefix + "attention.attention.query.weight"
        o, n = self.layout.offsets[q]
        d = self.layout.shapes[q][0]
        return self.bf16[o:o + 3 * n].view(3 * d, d)

    def bqkv(self, prefix) -> torch.Tensor:
        o, n = self.layout.offsets[prefix + "attention.attention.q_bias"]
        return self.flat[o:o + 3 * n]


def _layer_names(prefix, qkv_bias=True):
    a = prefix + "attention.attention."
    names = [prefix + "output.dense.weight", prefix + "output.dense.bias", prefix + "intermediate.dense.weight",
             prefix + "intermediate.dense.bias", prefix + "layernorm_after.weight", prefix + "layernorm_after.bias",
             prefix + "attention.output.dense.weight", prefix + "attention.output.dense.bias",
             a + "query.weight", a + "key.weight", a + "value.weight"]  # q,k,v adjacent (fused wgrad)
    if qkv_bias:
        names += [a + "q_bias", a + PAD_SUFFIX, a + "v_bias"]
    names += [prefix + "layernorm_before.weight", prefix + "layernorm_before.bias"]
    return names


def generic_groups(model, bucket_elems: int = 8 << 20) -> List[List[str]]:
    """Any nn.Module (e.g. the reference's V-JEPA model driven through the attention plug-in): parameters in REVERSE
    registration order (≈ the order autograd finishes them), cut into buckets of about `bucket_elems` elements."""
    groups, cur, n = [], [], 0
    for name, p in reversed(list(model.named_parameters())):
        cur.append(name)
        n += p.numel()
        if n >= bucket_elems:
            groups.append(cur)
            cur, n = [], 0
    if cur:
        groups.append(cur)
    return groups


def order_groups(model) -> List[List[str]]:
    """Parameter names grouped into data-parallel buckets, in backward-completion order (MIM model: decoder head first;
    classification model: classifier + fc_norm first; both end with the encoder blocks and the patch embedding)."""
    if not hasattr(model, "videomae"):
        return generic_groups(model)
    c = model.config
    groups = []
    if hasattr(model, "decoder"):
        groups.append(["decoder.head.weight", "decoder.head.bias", "decoder.norm.weight", "decoder.norm.bias"])
        for j in reversed(range(c.decoder_num_hidden_layers)):
            groups.append(_layer_names(f"decoder.decoder_layers.{j}.", c.qkv_bias))
        groups.append(["mask_token", "encoder_to_decoder.weight"])
    elif hasattr(model, "classifier"):
        head = ["classifier.weight", "classifier.bias"]
        if model.fc_norm is not None:
            head += ["fc_norm.weight", "fc_norm.bias"]
        groups.append(head)
    for i in reversed(range(c.num_hidden_layers)):
        groups.append(_layer_names(f"videomae.encoder.layer.{i}.", c.qkv_bias))
    tail = ["videomae.embeddings.patch_embeddings.projection.weight", "videomae.embeddings.patch_embeddings.projection.bias"]
    if hasattr(model.videomae.embeddings, "mask_token"):  # SimMIM-style encoder mask token
        tail = ["videomae.embeddings.mask_token"] + tail
    if model.videomae.layernorm is not None:
        tail = ["videomae.layernorm.weight", "videomae.layernorm.bias"] + tail
    groups.append(tail)
    return groups


# ----------------------------------------------------------------------------------------------
# one transformer block: forward with saves / backward
# ----------------------------------------------------------------------------------------------
class _BlockSaved:
    __slots__ = ("x_in", "h1", "m1", "r1", "qkv", "a", "a64", "lse", "x_mid", "h2", "m2", "r2", "pre", "f")


def videomae_block_names(prefix: str) -> Dict[str, object]:
    """role -> parameter name of one reference VideoMAE block (modeling_videomae.py:392-431); K has no bias (:261)."""
    return dict(w2=prefix + "output.dense.weight", b2=prefix + "output.dense.bias", w1=prefix + "intermediate.dense.weight",
                b1=prefix + "intermediate.dense.bias", ln2w=prefix + "layernorm_after.weight", ln2b=prefix + "layernorm_after.bias",
                wo=prefix + "attention.output.dense.weight", bo=prefix + "attention.output.dense.bias",
                ln1w=prefix + "layernorm_before.weight", ln1b=prefix + "layernorm_before.bias",
                qkv_bias=prefix + "attention.attention.q_bias", skip_k=True)


def vjepa_block_names(prefix: str) -> Dict[str, object]:
    """role -> parameter name of one reference V-JEPA block (modeling_vjepa.py:429-485); Q, K and V all carry a bias."""
    return dict(w2=prefix + "mlp.fc2.weight", b2=prefix + "mlp.fc2.bias", w1=prefix + "mlp.fc1.weight", b1=prefix + "mlp.fc1.bias",
                ln2w=prefix + "norm2.weight", ln2b=prefix + "norm2.bias", wo=prefix + "attention.proj.weight",
                bo=prefix + "attention.proj.bias", ln1w=prefix + "norm1.weight", ln1b=prefix + "norm1.bias",
                qkv_bias=prefix + "attention.query.bias", skip_k=False)


def block_forward_train(X, p, rope=None) -> Tuple[torch.Tensor, _BlockSaved]:
    """Same math as modeling._block_forward (reference :405-431), out of place, keeping what backward needs.
    `rope` = (grid_size, ids, max_pos): V-JEPA's rotary embedding; the SAVED Q and K are the rotated ones."""
    B, n, d = X.shape
    s = _BlockSaved()
    s.x_in = X
    s.h1, s.m1, s.r1 = ops.layernorm_fwd(X, p.g1, p.be1, p.eps, save_stats=True)
    pad32 = p.hd == 32 and getattr(p, "pad32", False)
    if rope is not None and p.hd != 64 and not pad32:
        raise ops.SmbvError("the rotary embedding kernel is wired to the tcgen05 attention paths (head_dim 64, or 32 zero-padded)")
    if pad32:  # head_dim 32 on the head_dim-64 kernels; the SAVED q, k, v are the rotated, zero-padded ones
        from .modeling import attention32_forward

        s.a, s.qkv, s.a64, s.lse = attention32_forward(s.h1, p, n, rope, return_lse=True)
    elif p.hd == 64:
        s.qkv = ops.gemm(s.h1, p.wqkv, p.bqkv, ops.EPI_QKV_HEADS, heads=p.heads, tokens=n)
        if rope is not None:
            ops.rope3d_(s.qkv[:2], rope[0], rope[1], rope[2])
        s.a, s.lse = ops.flash_attn_fwd(s.qkv[0], s.qkv[1], s.qkv[2], 64 ** -0.5, return_lse=True)
    else:  # small heads: token-major [B,n,3d]
        s.qkv = ops.gemm(s.h1, p.wqkv, p.bqkv, ops.EPI_BF16)
        s.a, s.lse = ops.attn_small_fwd(s.qkv, p.heads, p.hd ** -0.5, return_lse=True)
    s.x_mid = X.clone()  # keep X_in for the LayerNorm backward; the update itself is an in-place TMA reduce-add
    ops.gemm(s.a, p.wo, p.bo, ops.EPI_RESID_F32, residual=s.x_mid)
    s.h2, s.m2, s.r2 = ops.layernorm_fwd(s.x_mid, p.g2, p.be2, p.eps, save_stats=True)
    M, m = B * n, p.w1.shape[0]
    s.pre = torch.empty((B, n, m), dtype=torch.bfloat16, device=X.device)
    s.f = torch.empty((B, n, m), dtype=torch.bfloat16, device=X.device)
    ops.gemm_ex(s.h2, p.w1, M, m, d, ops.EPI_GELU_BF16, s.f, bias=p.b1, aux=s.pre)
    x_out = s.x_mid.clone()
    ops.gemm(s.f, p.w2, p.b2, ops.EPI_RESID_F32, residual=x_out)
    return x_out, s


def block_backward(dX, dXb, s: _BlockSaved, p, arena, prefix: str, names: Optional[Dict[str, object]] = None, rope=None,
                   sq: Optional[SideQueue] = None, extra=None):
    """dX: fp32 [B,n,d] gradient of the block output (updated IN PLACE to the gradient of the block input);
    dXb: its bf16 copy.  Returns the bf16 copy of the updated dX.  `names`: role -> parameter name (default: the VideoMAE
    block under `prefix`); `rope`: as in block_forward_train — the gradients of the rotated Q, K go back through the
    transposed rotary map before the bias / weight / input gradients are formed.  `sq`: the caller's SideQueue — weight / bias
    gradients are queued there (each AFTER the critical-path kernel that starts from the same inputs has been launched); the
    caller closes the block with `sq.block_done` and ends with `sq.finish()`.  None = everything on the current stream.
    `extra`: fp32 like dX or None — the gradient of the block's input as a returned hidden state, added by the last LayerNorm
    backward (so both the updated dX and its bf16 copy include it)."""
    B, n, d = dX.shape
    H = p.heads
    g = arena.g
    nm = names or videomae_block_names(prefix)
    if sq is None:
        sq = SideQueue("cpu")  # disabled: runs everything in place

    def wb(mark, dy, x, w, b):  # weight + bias gradient of one nn.Linear
        gw, gb = g(w), g(b)  # (a scratch arena allocates on first use: on the main stream)

        def fn():
            ops.linear_wgrad(dy, x, gw)
            ops.colsum(dy, gb)
        sq.run(mark, fn, dy, x)

    def qkv_wb(mark, dqkv, heads):  # fused QKV weight gradient + bias gradient straight into [dq_bias; 0 | dk_bias; dv_bias]
        gb = arena.fused_qkv_bias(prefix) if nm["qkv_bias"] in arena.offsets else None
        dwqkv = arena.fused_qkv(prefix)

        def fn():
            if gb is not None:
                ops.colsum_heads(dqkv, gb, skip_k=bool(nm["skip_k"]))
            for b in range(B):
                ops.qkv_wgrad(dqkv, s.h1[b], dwqkv, n, heads, batch_index=b, batch=B)
        sq.run(mark, fn, dqkv, s.h1)

    # ---- MLP: X_out = X_mid + W2 gelu(W1 LN2(X_mid) + b1) + b2 ----
    mk = sq.mark()
    dpre = ops.linear_dgrad(dXb, p.w2, aux=s.pre)  # [B,n,4d] bf16, gelu' fused
    wb(mk, dXb, s.f, nm["w2"], nm["b2"])
    mk = sq.mark()
    dh2 = ops.linear_dgrad(dpre, p.w1)
    wb(mk, dpre, s.h2, nm["w1"], nm["b1"])
    dXb = ops.layernorm_bwd(dh2, s.x_mid, s.m2, s.r2, p.g2, dX, True, g(nm["ln2w"]), g(nm["ln2b"]))
    # ---- attention: X_mid = X_in + Wo Attn(LN1(X_in)) + bo ----
    mk = sq.mark()
    dO = ops.linear_dgrad(dXb, p.wo)  # [B,n,d] bf16 token-major
    wb(mk, dXb, s.a, nm["wo"], nm["bo"])
    if p.hd == 32 and getattr(p, "pad32", False):  # head_dim 32 on the head_dim-64 kernels (see modeling.attention32_forward)
        dqkvp = torch.empty_like(s.qkv)  # [3,B,H,n,64]; the pad columns of dq, dk, dv come out zero
        ops.flash_attn_bwd(s.qkv[0], s.qkv[1], s.qkv[2], s.a64, ops.heads32_tokens(dO, H, expand=True), s.lse, 32 ** -0.5,
                           dq=dqkvp[0], dk=dqkvp[1], dv=dqkvp[2])
        dqkv = ops.heads32_squeeze(dqkvp)  # [3,B,H/2,n,64]: the layout the fused QKV GEMM wrote
        if rope is not None:
            ops.rope3d_(dqkv[:2].view(2, B, H // 2, 2 * n, 32), rope[0], rope[3], rope[2], transpose=True)
        dh1 = torch.empty((B, n, d), dtype=torch.bfloat16, device=dX.device)
        mk = sq.mark()
        for b in range(B):
            ops.qkv_dgrad(dqkv, p.wqkv, n, H // 2, batch_index=b, batch=B, out=dh1[b])
        qkv_wb(mk, dqkv, H // 2)
    elif p.hd != 64:  # small heads: token-major dQKV [B,n,3d] -> plain row-major dgrad / wgrad
        dqkv = ops.attn_small_bwd(s.qkv, s.a, dO, s.lse, H, p.hd ** -0.5)
        if nm["qkv_bias"] in arena.offsets:
            bq = arena.fused_qkv_bias(prefix)
            ops.colsum(dqkv, bq)
            bq[d:2 * d].zero_()  # k_bias is a constant zero (reference :261): its slot is padding, not a parameter
        ops.linear_wgrad(dqkv, s.h1, arena.fused_qkv(prefix))
        dh1 = ops.linear_dgrad(dqkv, p.wqkv)
    else:
        dqkv = torch.empty_like(s.qkv)  # [3,B,H,n,64]
        ops.flash_attn_bwd(s.qkv[0], s.qkv[1], s.qkv[2], s.a, dO, s.lse, 64 ** -0.5, dq=dqkv[0], dk=dqkv[1], dv=dqkv[2])  # whole batch
        if rope is not None:
            ops.rope3d_(dqkv[:2], rope[0], rope[1], rope[2], transpose=True)
        dh1 = torch.empty((B, n, d), dtype=torch.bfloat16, device=dX.device)
        mk = sq.mark()
        for b in range(B):
            ops.qkv_dgrad(dqkv, p.wqkv, n, H, batch_index=b, batch=B, out=dh1[b])
        qkv_wb(mk, dqkv, H)
    dXb = ops.layernorm_bwd(dh1, s.x_in, s.m1, s.r1, p.g1, dX, True, g(nm["ln1w"]), g(nm["ln1b"]), extra=extra)
    return dXb


# ----------------------------------------------------------------------------------------------
# whole model
# ----------------------------------------------------------------------------------------------
class _ModelSaved:
    pass


def encoder_forward_train(vm, vol, mask_pack=None, blend: bool = False):
    """Patch embedding (+ visible-row compaction when masked) and the encoder blocks of reference :124-139, :442-483,
    keeping activations.  Returns (X fp32 [B,n,d], [per-block saves]).  `blend`: SimMIM style (all N tokens, masked ones
    replaced by the encoder mask token in the patch-embed epilogue)."""
    vm._check_config()
    pe = vm.packed()
    pos = vm.pos_table(vm.config.hidden_size, vol.device)
    patches = None
    if blend:
        X = ops.patch_embed_select_fwd(vol, pe["wpe16"], pe["bpe"], pos, mask_pack[0], pe["mask_token"])
    elif mask_pack is None:
        X = ops.patch_embed_fwd(vol, pe["wpe16"], pe["bpe"], pos)
    else:
        # training: only the visible 35 % of the patches are embedded.  Their im2col rows (bf16, what the reference's bf16
        # autocast conv sees) are gathered once, feed a plain tcgen05 GEMM whose epilogue adds bias + PE[vis], and are kept
        # for the weight gradient (the implicit-GEMM kernel would embed all 20480 tokens in TF32 and drop 65 % of them).
        _, vis, _, _, n_vis, _ = mask_pack
        B, d = vol.shape[0], vm.config.hidden_size
        patches = ops.gather_patches(vol, vis, n_vis)  # [B*n_vis, 4096] bf16
        wpe16 = pe["wpe16"]  # a view of the arena's bf16 operand copy (kept current by smbv_adamw_step) or the cached cast
        X = torch.empty((B, n_vis, d), dtype=torch.float32, device=vol.device)
        pv = patches.view(B, n_vis, -1)
        for b in range(B):
            ops.gemm(pv[b], wpe16, pe["bpe"], ops.EPI_POS_GATHER_F32, out=X[b], pos=pos, row_map=vis[b])
    saved = [patches]
    for p in pe["layers"]:
        X, sv = block_forward_train(X, p)
        saved.append(sv)
    return X, saved  # saved[0] = gathered visible patches (or None), saved[1:] = per-block activations


def encoder_backward(vm, vol, saved, dX, dXb, arena: GradArena, idx, n_sel: int, done: Callable[[], None], blend_pack=None,
                     sq: Optional[SideQueue] = None, dhidden=None):
    """dX fp32 [B,n,d] (+ bf16 copy) = gradient of the encoder output -> encoder-block and patch-embedding gradients.
    `idx` int32 [B, >= n_sel]: the tokens that reached the encoder (the visible ones; all of them without a mask).
    `sq`: the caller's SideQueue (its `done` closes the blocks on it and the caller finishes it).
    `dhidden`: gradients of the hidden states (fp32 [B,n,d] or None, index k = input of block k); entry k joins dX in
    block k's last LayerNorm backward.  Entries past the last block are the caller's (already in dX)."""
    pe = vm.packed()
    g = arena.g
    d = vm.config.hidden_size
    patches, blocks = saved[0], saved[1:]
    for i in reversed(range(len(blocks))):
        dXb = block_backward(dX, dXb, blocks[i], pe["layers"][i], arena, f"videomae.encoder.layer.{i}.", sq=sq,
                             extra=None if dhidden is None else dhidden[i])
        done()
    if blend_pack is not None:
        # SimMIM blend: E[b,n] = mask ? mask_token : conv(P[n]) + bias — the masked rows of dE sum into the mask token, the
        # visible rows carry the patch-embedding gradients
        _, vis, msk, _, n_vis, n_mask = blend_pack
        ops.colsum(ops.gather_rows(dX, msk[:, :n_mask].contiguous()), g("videomae.embeddings.mask_token").view(-1))
        dX = ops.gather_rows(dX, vis[:, :n_vis].contiguous())  # [B, n_vis, d]
        dXb, idx, n_sel = ops.cast_bf16(dX), vis, n_vis
    # patch embedding: only the tokens that were kept carry gradient (masked rows of E were dropped, reference :134-137)
    ops.colsum(dX, g("videomae.embeddings.patch_embeddings.projection.bias"))
    if patches is None:
        patches = ops.gather_patches(vol, idx, n_sel)  # [B*n_sel, 4096] bf16 im2col rows
    ops.linear_wgrad(dXb, patches, g("videomae.embeddings.patch_embeddings.projection.weight").view(d, -1))
    done()


def _encoder_states(S, X):
    """The encoder's hidden states (upstream `output_hidden_states`): every block's input — kept out of place by
    block_forward_train anyway — and the last block's output X, before the optional final LayerNorm."""
    return [sv.x_in for sv in S.enc[1:]] + [X]


def mim_forward_train(model, vol, mask_pack, states: bool = False):
    """Forward of reference :791-897 keeping activations.  Returns (loss, logits, dlogits, saved); with `states`, saved.states
    holds the encoder's hidden states."""
    model._check_config()
    vm = model.videomae
    vm._check_config()
    c = model.config
    fine, vis, msk, slot, n_vis, n_mask = mask_pack
    B = vol.shape[0]
    N, d, dd = vm.num_patches, c.hidden_size, c.decoder_hidden_size
    S = _ModelSaved()
    pd = model.packed()
    simmim = getattr(model, "mim_style", "mae") == "simmim"
    X, S.enc = encoder_forward_train(vm, vol, mask_pack, blend=simmim)
    if states:
        S.states = _encoder_states(S, X)
    if vm.layernorm is not None:  # use_mean_pooling=False: final encoder LayerNorm (reference :517-520, :648-649)
        _final_ln_forward(vm, X, S)
    else:
        S.xb = ops.cast_bf16(X)
    pos_d = vm.pos_table(dd, vol.device)
    Xd = torch.empty((B, N, dd), dtype=torch.float32, device=vol.device)
    if simmim:  # all N tokens, natural order
        every = torch.arange(N, dtype=torch.int32, device=vol.device)
        for b in range(B):
            ops.gemm(S.xb[b], pd["we2d"], None, ops.EPI_POS_GATHER_F32, out=Xd[b], pos=pos_d, row_map=every)
    else:
        for b in range(B):
            ops.gemm(S.xb[b], pd["we2d"], None, ops.EPI_POS_GATHER_F32, out=Xd[b, :n_vis], pos=pos_d, row_map=vis[b])
        ops.fill_mask_tokens(Xd, pd["mask_token"], pos_d, msk, n_vis)
    S.dec = []
    for p in pd["layers"]:
        Xd, sv = block_forward_train(Xd, p)
        S.dec.append(sv)
    S.xd = Xd
    S.hN = torch.empty((B, n_mask, dd), dtype=torch.bfloat16, device=vol.device)
    S.mN = torch.empty((B, n_mask), dtype=torch.float32, device=vol.device)
    S.rN = torch.empty((B, n_mask), dtype=torch.float32, device=vol.device)
    if simmim:
        S.g = ops.gather_rows(Xd, msk[:, :n_mask].contiguous())  # the masked rows, ascending n
    for b in range(B):
        _, m_, r_ = ops.layernorm_fwd(S.g[b] if simmim else Xd[b, n_vis:], pd["gn"], pd["bn"], 1e-5, save_stats=True, out=S.hN[b])
        S.mN[b], S.rN[b] = m_, r_
    logits = ops.gemm(S.hN, pd["wh"], pd["bh"], ops.EPI_BF16)
    loss, dlogits = ops.normpix_loss(vol, msk, n_mask, logits, True, model.loss_kind, c.patch_size)
    S.vol, S.mask_pack = vol, mask_pack
    return loss, logits, dlogits, S


def mim_backward(model, S, dlogits, arena: GradArena, on_bucket: Optional[Callable[[int], None]] = None, dhidden=None,
                 loss_scale=None):
    """Backward of the whole model into `arena` (gradients are ACCUMULATED: zero the arena first for a fresh step).
    `on_bucket(i)` is called as soon as bucket i of `order_groups` is complete (DP all-reduce hook).
    `dhidden` (list of num_hidden_layers + 1 fp32 tensors or None): gradients of the encoder's hidden states, added at their
    layer boundaries; the gradients are then loss_scale * d(loss) + the hidden-state terms — the loss gradient is scaled
    where it enters the encoder, and the decoder / head gradients behind it at the end."""
    vm = model.videomae
    c = model.config
    fine, vis, msk, slot, n_vis, n_mask = S.mask_pack
    B = S.vol.shape[0]
    N, d, dd = vm.num_patches, c.hidden_size, c.decoder_hidden_size
    pe, pd = vm.packed(), model.packed()
    g = arena.g
    dev = S.vol.device
    bucket = 0
    sq = SideQueue(dev)  # weight / bias gradients beside the critical path; a bucket is handed to `on_bucket` once they have landed

    def done():
        nonlocal bucket
        b = bucket
        bucket += 1
        sq.block_done((lambda: on_bucket(b)) if on_bucket is not None else None)

    # ---- head + final decoder LayerNorm (reference :717-722) ----
    mk = sq.mark()
    dhN = ops.linear_dgrad(dlogits, pd["wh"])  # [B, n_mask, dd] bf16
    gw, gb = g("decoder.head.weight"), g("decoder.head.bias")
    sq.run(mk, lambda: (ops.linear_wgrad(dlogits, S.hN, gw), ops.colsum(dlogits, gb)), dlogits, S.hN)
    simmim = getattr(model, "mim_style", "mae") == "simmim"
    if simmim:  # the head read the masked rows out of the natural-order sequence: scatter its gradient back
        dG = torch.empty((B, n_mask, dd), dtype=torch.float32, device=dev)
        for b in range(B):
            ops.layernorm_bwd(dhN[b], S.g[b], S.mN[b], S.rN[b], pd["gn"], dG[b], False,
                              g("decoder.norm.weight"), g("decoder.norm.bias"), want_bf16=False)
        dXd = ops.scatter_rows(dG, msk, N, n_mask)
    else:
        dXd = torch.zeros((B, N, dd), dtype=torch.float32, device=dev)  # visible rows get no gradient from the head
        for b in range(B):
            ops.layernorm_bwd(dhN[b], S.xd[b, n_vis:], S.mN[b], S.rN[b], pd["gn"], dXd[b, n_vis:], False,
                              g("decoder.norm.weight"), g("decoder.norm.bias"), want_bf16=False)
    done()
    dXb = ops.cast_bf16(dXd)
    for j in reversed(range(len(S.dec))):
        dXb = block_backward(dXd, dXb, S.dec[j], pd["layers"][j], arena, f"decoder.decoder_layers.{j}.", sq=sq)
        done()
    # ---- decoder input: cat([Z + PE_vis, mask_token + PE_msk]) (reference :801-815); SimMIM style: Z + PE for every token ----
    n_enc = N if simmim else n_vis
    dZb = torch.empty((B, n_enc, dd), dtype=torch.bfloat16, device=dev)
    gm = g("mask_token").view(-1)
    for b in range(B):
        if not simmim:
            ops.colsum(dXd[b, n_vis:], gm, M=n_mask, N=dd, ld=dd)
        ops.cast_bf16(dXd[b, :n_enc], out=dZb[b])
    mk = sq.mark()
    dX = ops.linear_dgrad(dZb, pd["we2d"], out_dtype=torch.float32)  # [B, n_vis, d] fp32
    ge2d = g("encoder_to_decoder.weight")
    sq.run(mk, lambda: ops.linear_wgrad(dZb, S.xb, ge2d), dZb, S.xb)
    done()
    if dhidden is None:
        dXb = ops.cast_bf16(dX)
    else:  # loss gradient * loss_scale (+ the last hidden state's gradient when no final LayerNorm follows it)
        dXb = ops.scale_add_recast_(dX, loss_scale, dhidden[-1] if vm.layernorm is None else None)
    if vm.layernorm is not None:  # back through the final encoder LayerNorm
        dX, dXb = _final_ln_backward(vm, S, dXb, arena, extra=None if dhidden is None else dhidden[-1])
    encoder_backward(vm, S.vol, S.enc, dX, dXb, arena, vis, n_vis, done, blend_pack=S.mask_pack if simmim else None, sq=sq,
                     dhidden=dhidden)
    sq.finish()
    if dhidden is not None:  # the loss-only gradients (head, decoder, mask_token, encoder_to_decoder: the buckets before the encoder's)
        ops.scale_f32_(arena.flat[:arena.bucket_bounds[c.decoder_num_hidden_layers + 2]], loss_scale)


# ----------------------------------------------------------------------------------------------
# autograd bridge (HF Trainer / plain loss.backward())
# ----------------------------------------------------------------------------------------------
def _hidden_grads(ctx, dH):
    """The gradients of the returned hidden states as contiguous fp32 tensors (None where unused), or None when all are
    unused.  Reading ctx.saved_tensors raises torch's in-place modification error if a returned state was edited: the
    hand-written backward reads the same tensors."""
    ctx.saved_tensors
    if all(g is None for g in dH):
        return None
    return [None if g is None else g.float().contiguous() for g in dH]


def _loss_scale(grad_loss, device):
    return torch.zeros(1, dtype=torch.float32, device=device) if grad_loss is None else grad_loss


class _MIMFunction(torch.autograd.Function):
    """One node for the whole model: forward runs the CUDA forward, backward runs `mim_backward` and hands every
    parameter its gradient, so `out.loss.backward()` works exactly like with the reference module.  With `states` the
    encoder's hidden states are further outputs, differentiable through the same backward."""

    @staticmethod
    def forward(ctx, model, vol, mask_pack, names, states, *params):
        loss, logits, dlogits, S = mim_forward_train(model, vol, mask_pack, states=states)
        ctx.model, ctx.S, ctx.dlogits, ctx.names = model, S, dlogits, names
        ctx.needs = [p.requires_grad for p in params]
        ctx.mark_non_differentiable(logits)
        ctx.set_materialize_grads(False)
        hs = S.states if states else []
        ctx.save_for_backward(*hs)
        return (loss, logits, *hs)

    @staticmethod
    def backward(ctx, grad_loss, _grad_logits, *dH):
        arena = GradArena(ctx.model, ctx.S.vol.device)  # fresh: autograd may adopt these views as p.grad
        dhidden = _hidden_grads(ctx, dH)
        if dhidden is None:
            mim_backward(ctx.model, ctx.S, ctx.dlogits, arena)  # gradients for d(loss) = 1; the saved dlogits stay untouched
            # upstream factor (gradient accumulation, loss scaling; 1.0 for a plain .backward()) applied in fp32 on the way out
            ops.scale_f32_(arena.flat, grad_loss)
        else:  # the factor must not reach the hidden-state terms: mim_backward applies it to the loss gradient only
            mim_backward(ctx.model, ctx.S, ctx.dlogits, arena, dhidden=dhidden, loss_scale=_loss_scale(grad_loss, arena.flat.device))
        grads = tuple(arena.views[n] if need else None for n, need in zip(ctx.names, ctx.needs))
        return (None, None, None, None, None) + grads


def autograd_forward(model, vol, mask_pack, states: bool = False):
    """-> (loss, logits[, hidden state 0, ..., hidden state L])."""
    names, params = zip(*model.named_parameters())
    return _MIMFunction.apply(model, vol, mask_pack, list(names), states, *params)


class _EncoderOnly(torch.nn.Module):
    """Name-space shim: a bare `B200VideoMAEModel` seen under the `videomae.` prefix the arena layout uses."""

    def __init__(self, vm):
        super().__init__()
        self.videomae = vm
        self.config = vm.config


def _final_ln_forward(vm, X, S):
    """use_mean_pooling=False: the encoder's final LayerNorm (reference :517-520, :648-649), keeping its statistics."""
    S.x_pre = X
    S.xb, S.mE, S.rE = ops.layernorm_fwd(X, vm.layernorm.weight.detach(), vm.layernorm.bias.detach(), vm.config.layer_norm_eps, save_stats=True)
    return S.xb


def _final_ln_backward(vm, S, dYb, arena, extra=None):
    """dYb bf16 [B,n,d] = gradient of the final LayerNorm's output -> (dX fp32, dX bf16) of its input (+ `extra`, the
    gradient of that input as the last hidden state)."""
    dX = torch.empty_like(S.x_pre)
    dXb = ops.layernorm_bwd(dYb, S.x_pre, S.mE, S.rE, vm.layernorm.weight.detach(), dX, False,
                            arena.g("videomae.layernorm.weight"), arena.g("videomae.layernorm.bias"), extra=extra)
    return dX, dXb


class _EncoderFunction(torch.autograd.Function):
    """`model.videomae(x[, mask]).last_hidden_state` with gradients (reference VideoMAEModel.forward, :537-658, under
    autograd): forward = the CUDA forward keeping activations, backward = `encoder_backward`.  With `states` the hidden
    states are further outputs: every block's input, and the last block's output when a final LayerNorm follows it (without
    one that output is X itself)."""

    @staticmethod
    def forward(ctx, vm, vol, mask_pack, names, states, *params):
        S = _ModelSaved()
        X, S.enc = encoder_forward_train(vm, vol, mask_pack)
        hs = _encoder_states(S, X) if states else []
        if vm.layernorm is not None:
            X = _final_ln_forward(vm, X, S).float()
        elif hs:
            hs.pop()  # state L is the returned X
        S.vol, S.mask_pack = vol, mask_pack
        ctx.vm, ctx.S, ctx.names, ctx.x_shape = vm, S, names, X.shape
        ctx.needs = [p.requires_grad for p in params]
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(*hs)
        return (X, *hs) if states else X

    @staticmethod
    def backward(ctx, dOut, *dH):
        vm, S = ctx.vm, ctx.S
        arena = GradArena(_EncoderOnly(vm), S.vol.device)
        dhidden = _hidden_grads(ctx, dH)
        if dhidden is not None and vm.layernorm is None:
            dhidden.append(None)  # the last state is X: its gradient is dOut
        B, n = ctx.x_shape[:2]
        if dOut is None:  # only hidden states were used
            dOut = torch.zeros(ctx.x_shape, dtype=torch.float32, device=S.vol.device)
        if vm.layernorm is not None:
            dX, dXb = _final_ln_backward(vm, S, ops.cast_bf16(dOut.float().contiguous()), arena,
                                         extra=None if dhidden is None else dhidden[-1])
        else:
            dX = dOut.float().clone()  # the block backward updates it in place
            dXb = ops.cast_bf16(dX)
        if S.mask_pack is None:
            idx = torch.arange(n, dtype=torch.int32, device=dX.device).repeat(B, 1).contiguous()
        else:
            idx = S.mask_pack[1]
        encoder_backward(vm, S.vol, S.enc, dX, dXb, arena, idx, n, lambda: None, dhidden=dhidden)
        grads = tuple(arena.views["videomae." + nm] if need else None for nm, need in zip(ctx.names, ctx.needs))
        return (None, None, None, None, None) + grads


def encoder_autograd_forward(vm, vol, mask_pack, states: bool = False):
    """-> X, or (X, hidden states ...) with `states` (see _EncoderFunction)."""
    vm.refresh_operands()
    names, params = zip(*vm.named_parameters())
    return _EncoderFunction.apply(vm, vol, mask_pack, list(names), states, *params)


# ----------------------------------------------------------------------------------------------
# data parallel step (one process per GPU; NCCL all-reduce overlapped with backward)
# ----------------------------------------------------------------------------------------------
class DataParallelStep:
    """`step(*inputs)` = forward + backward + bucketed gradient all-reduce (+ optional optimiser).

    MIM model: `step(vol, mask_pack)`; classification model: `step(vol, additional_features, labels)`.
    Each bucket (one transformer block) is cast to bf16, all-reduced on NCCL's stream while backward continues, and
    folded back into the fp32 arena as the mean over ranks.  world_size 1 (or no process group) skips communication.
    """

    def __init__(self, model, optimizer: Optional[torch.optim.Optimizer] = None, process_group=None, wire_dtype=torch.bfloat16,
                 cuda_graph: bool = False):
        """cuda_graph=True: forward + backward (+ the gradient all-reduce) of a step are captured ONCE per input signature into a
        CUDA graph and replayed — the step is ~475 launches (1975 for the classification shape), many of them 10-30 us kernels
        behind ~20 us of host work each (ctypes call, TMA descriptor encoding), so the eager step is partly launch-bound: the
        replay is 7 % faster at 512x512x320 (29.4 -> 27.3 ms, tools/graph_step.py).  Inputs are copied into static buffers
        (`static_inputs()` hands them out so that a producer kernel can write them in place); the returned loss / logits are
        static tensors overwritten by the next step.  The optimiser step (lr and bias corrections change every step) stays
        outside the graph.  Needs optim.FusedAdamW or no optimiser; falls back to eager otherwise."""
        from .distributed import BucketReducer

        self.model = model
        self.dev = next(model.parameters()).device
        self.fused_opt = hasattr(optimizer, "exp_avg_sq")  # optim.FusedAdamW (flat arenas) vs a torch.optim optimiser
        pa = getattr(model, "_arena", None)
        self.arena = GradArena(model, self.dev, optimizer.layout if self.fused_opt else (pa.layout if pa is not None else None))
        self.arena.assign_to_params()
        self.opt = optimizer
        self.reducer = BucketReducer(self.arena.flat, self.arena.bucket_bounds, process_group, wire_dtype,
                                     cast_down=lambda s, d: ops.cast_bf16(s, out=d), cast_up=ops.cast_f32_scaled)
        self.world = self.reducer.world
        self.is_cls = hasattr(model, "classifier")
        self.cuda_graph = bool(cuda_graph) and (self.fused_opt or optimizer is None)
        self._graphs = {}  # input signature -> (graph, static tensors, static loss, static logits)

    # ---- one forward + backward (+ all-reduce), eager; gradients land in the arena ----
    def _fwd_bwd(self, vol, *inputs):
        self.arena.zero()
        with torch.no_grad():
            if self.is_cls:
                feats, labels = inputs
                loss, logits, dpooled, S = cls_forward_train(self.model, vol, feats, labels, self.arena)
                cls_backward(self.model, S, dpooled, self.arena, self.reducer.reduce_bucket)
            else:
                (mask_pack,) = inputs
                loss, logits, dlogits, S = mim_forward_train(self.model, vol, mask_pack)
                mim_backward(self.model, S, dlogits, self.arena, self.reducer.reduce_bucket)
            self.reducer.finish()
        return loss, logits

    # ---- CUDA-graph path ----
    @staticmethod
    def _flatten(vol, inputs):
        """(tensors, rebuild): the tensor leaves of (vol, *inputs) in order, and a function that rebuilds the argument list
        from replacement tensors (ints / None / other leaves stay as they are: they are part of the signature)."""
        leaves, spec = [], []

        def walk(x):
            if isinstance(x, torch.Tensor):
                leaves.append(x)
                return ("t", len(leaves) - 1)
            if isinstance(x, (tuple, list)):
                return ("l", type(x), [walk(y) for y in x])
            return ("c", x)

        spec = [walk(vol)] + [walk(x) for x in inputs]

        def build(node, ts):
            if node[0] == "t":
                return ts[node[1]]
            if node[0] == "l":
                return node[1](build(y, ts) for y in node[2])
            return node[1]

        def sig(node):
            if node[0] == "t":
                t = leaves[node[1]]
                return ("t", tuple(t.shape), str(t.dtype))
            if node[0] == "l":
                return tuple(sig(y) for y in node[2])
            return ("c", node[1] if isinstance(node[1], (int, float, str, bool, type(None))) else id(node[1]))

        return leaves, (lambda ts: [build(n, ts) for n in spec]), tuple(sig(n) for n in spec)

    def static_inputs(self, vol, *inputs):
        """The static input buffers of the graph for this input signature, in the structure of (vol, *inputs) — captured on
        first use from the given example.  Tensors written in place there (e.g. `VolumePreprocessor(..., out=...)`) and passed
        back to `step` are not copied again."""
        leaves, rebuild, key = self._flatten(vol, inputs)
        if key not in self._graphs:
            self._capture(key, leaves, rebuild)
        return rebuild(self._graphs[key][1])

    def _capture(self, key, leaves, rebuild):
        static = [t.detach().clone() for t in leaves]
        args = rebuild(static)
        cur = torch.cuda.current_stream(self.dev)
        side = torch.cuda.Stream(self.dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):  # warm-up on a side stream (lazy initialisations must not happen under capture)
            for _ in range(2):
                self._fwd_bwd(*args)
        cur.wait_stream(side)
        torch.cuda.synchronize(self.dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            loss, logits = self._fwd_bwd(*args)
        self._graphs[key] = (g, static, loss, logits)

    def release_graphs(self):
        """Drop the captured graphs (call before destroying a process group whose all-reduces they captured: NCCL's communicator
        teardown hangs while such graphs are alive)."""
        self._graphs.clear()

    def _graph_fwd_bwd(self, vol, *inputs):
        leaves, rebuild, key = self._flatten(vol, inputs)
        if key not in self._graphs:
            self._capture(key, leaves, rebuild)
        g, static, loss, logits = self._graphs[key]
        for src, dst in zip(leaves, static):
            if src.data_ptr() != dst.data_ptr():
                dst.copy_(src, non_blocking=True)
        g.replay()
        return loss, logits

    def step(self, vol, *inputs):
        if not self.fused_opt:
            # a torch optimiser (or the caller) moved the fp32 masters; fused / foreach optimisers do not bump the version
            # counters packed() keys on, so the bf16 operands are re-derived every step (FusedAdamW refreshes them itself)
            vm = getattr(self.model, "videomae", None)
            (self.model if hasattr(self.model, "refresh_operands") else vm).refresh_operands()
        if self.cuda_graph:
            loss, logits = self._graph_fwd_bwd(vol, *inputs)
        else:
            loss, logits = self._fwd_bwd(vol, *inputs)
        if self.fused_opt:
            self.opt.step(self.arena)  # clip + AdamW + bf16 operand refresh, one pass over the arenas
        elif self.opt is not None:
            self.opt.step()
        return loss, logits


# ----------------------------------------------------------------------------------------------
# classification fine-tuning (SURVEY.md §8f rank 1; reference VideoMAEForVideoClassification :917-1023)
# ----------------------------------------------------------------------------------------------
def cls_forward_train(model, vol, feats, labels, arena: GradArena, states: bool = False):
    """Encoder (all tokens, no mask) -> token mean -> fc_norm -> [cat features] -> classifier -> loss.  The head's own
    gradients (classifier, fc_norm) are produced by the same launch as its forward and land in `arena`.
    Returns (loss, logits fp32 [B,L], dpooled fp32 [B,d], saved); with `states`, saved.states holds the encoder's hidden
    states."""
    vm = model.videomae
    S = _ModelSaved()
    X, S.enc = encoder_forward_train(vm, vol, None)
    if states:
        S.states = _encoder_states(S, X)
    B, N, d = X.shape
    hp = model.head_params()
    grads = dict(dW=arena.g("classifier.weight"), dbias=arena.g("classifier.bias"),
                 dgamma=arena.views.get("fc_norm.weight"), dbeta=arena.views.get("fc_norm.bias"))
    if model.fc_norm is not None:  # mean over tokens -> fc_norm (reference :974-975)
        pooled, inv_n = ops.token_sum(X), 1.0 / N
    else:  # use_mean_pooling=False: final encoder LayerNorm, then the FIRST token's row (reference :976-977)
        pooled, inv_n = _final_ln_forward(vm, X, S)[:, 0].float().contiguous(), 1.0
    loss, logits, dpooled = ops.cls_head(pooled, inv_n, hp["gamma"], hp["beta"], hp["eps"], feats, hp["W"], hp["b"],
                                         labels, model.problem_id(labels), grads)
    S.vol, S.n = vol, N
    return loss, logits, dpooled, S


def cls_backward(model, S, dpooled, arena: GradArena, on_bucket: Optional[Callable[[int], None]] = None, dhidden=None):
    """Broadcast d(loss)/d(mean token) to every token row, then the encoder / patch-embedding backward.  `dhidden`: as in
    mim_backward (the caller scales dpooled and the head's gradients)."""
    bucket = 0
    sq = SideQueue(S.vol.device)

    def done():
        nonlocal bucket
        b = bucket
        bucket += 1
        sq.block_done((lambda: on_bucket(b)) if on_bucket is not None else None)

    done()  # bucket 0 = classifier (+ fc_norm), finished in the forward launch
    B = S.vol.shape[0]
    vm = model.videomae
    if model.fc_norm is not None:
        dX, dXb = ops.broadcast_rows(dpooled, S.n)  # d mean / d token, every row
        if dhidden is not None and dhidden[-1] is not None:
            dXb = ops.scale_add_recast_(dX, None, dhidden[-1])
    else:  # only the first token's row of the final LayerNorm output carries gradient
        dYb = torch.zeros((B, S.n, dpooled.shape[1]), dtype=torch.bfloat16, device=dpooled.device)
        dYb[:, 0] = ops.cast_bf16(dpooled)
        dX, dXb = _final_ln_backward(vm, S, dYb, arena, extra=None if dhidden is None else dhidden[-1])
    idx = torch.arange(S.n, dtype=torch.int32, device=S.vol.device).repeat(B, 1).contiguous()
    encoder_backward(vm, S.vol, S.enc, dX, dXb, arena, idx, S.n, done, sq=sq, dhidden=dhidden)
    sq.finish()


class _ClsFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, vol, feats, labels, names, states, *params):
        arena = GradArena(model, vol.device)
        loss, logits, dpooled, S = cls_forward_train(model, vol, feats, labels, arena, states=states)
        ctx.model, ctx.S, ctx.dpooled, ctx.names, ctx.arena = model, S, dpooled, names, arena
        ctx.needs = [p.requires_grad for p in params]
        ctx.mark_non_differentiable(logits)
        ctx.set_materialize_grads(False)
        hs = S.states if states else []
        ctx.save_for_backward(*hs)
        return (loss, logits, *hs)

    @staticmethod
    def backward(ctx, grad_loss, _grad_logits, *dH):
        arena = ctx.arena
        dhidden = _hidden_grads(ctx, dH)
        if dhidden is None:
            cls_backward(ctx.model, ctx.S, ctx.dpooled, arena)  # everything for d(loss) = 1 (head gradients came with the forward)
            ops.scale_f32_(arena.flat, grad_loss)
        else:  # the upstream factor scales the loss seed and the head's gradients, not the hidden-state terms
            sc = _loss_scale(grad_loss, arena.flat.device)
            dpooled = ops.scale_f32_(ctx.dpooled.clone(), sc)
            cls_backward(ctx.model, ctx.S, dpooled, arena, dhidden=dhidden)
            ops.scale_f32_(arena.flat[:arena.bucket_bounds[1]], sc)  # bucket 0: classifier (+ fc_norm)
        grads = tuple(arena.views[n] if need else None for n, need in zip(ctx.names, ctx.needs))
        return (None, None, None, None, None, None) + grads


def cls_autograd_forward(model, vol, feats, labels, states: bool = False):
    """-> (loss, logits[, hidden state 0, ..., hidden state L])."""
    names, params = zip(*model.named_parameters())
    return _ClsFunction.apply(model, vol, feats, labels, list(names), states, *params)
