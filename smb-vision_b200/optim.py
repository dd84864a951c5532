"""Optimiser side of the training step (SURVEY.md §8f rank 2): what HF ``Trainer`` runs after ``loss.backward()``
(invoked at reference src/run_mim.py:445 with the hyper-parameters of scripts/training/run_mim.sh:17-21) —
``clip_grad_norm_(max_grad_norm=1.0)`` -> ``torch.optim.AdamW(lr=5e-5, weight_decay=0.01)`` -> cosine schedule with
``warmup_ratio=0.01`` — as two launches over the flat arenas of ``training.ParamArena`` / ``GradArena``:

* ``smbv_sumsq_f32``  : squared global gradient norm into a device scalar (deterministic, no host sync);
* ``smbv_adamw_step`` : clip scale + AdamW + refresh of the bf16 operand copy of every weight, one pass, 30 B / parameter.

Weight decay is applied to the same parameter set ``Trainer.get_decay_parameter_names`` selects: everything except the
parameters of ``nn.LayerNorm`` modules and names matching "bias", "layernorm", "rmsnorm", "norm" as a whole name
component or "_norm" at the end of one (``training.ArenaLayout.decay_segments``).  So V-JEPA's ``norm1`` / ``norm2``
LayerNorm weights are not decayed.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Callable, Optional

import torch

from . import ops
from ._lib import call, load
from .training import GradArena, ParamArena


def cosine_with_warmup(step: int, base_lr: float, warmup_steps: int, total_steps: int, num_cycles: float = 0.5) -> float:
    """transformers.get_cosine_schedule_with_warmup (``--lr_scheduler_type cosine --warmup_ratio 0.01``): the learning
    rate used BY optimiser step number `step` (0-based: the first update uses step 0 -> lr 0 when warmup_steps > 0)."""
    if step < warmup_steps:
        return base_lr * step / max(1, warmup_steps)
    progress = (step - warmup_steps) / max(1, total_steps - warmup_steps)
    return base_lr * max(0.0, 0.5 * (1.0 + math.cos(math.pi * num_cycles * 2.0 * progress)))


class FusedAdamW:
    """AdamW + global-norm clipping over a ``ParamArena`` (created on demand: the model's parameters become views of one
    flat fp32 buffer; state-dict keys/shapes are unchanged).

    ``step(grad_arena)`` consumes the flat gradient buffer (already all-reduced by ``DataParallelStep``).
    ``lr_schedule(step_index) -> lr`` overrides the constant ``lr`` (e.g. ``functools.partial(cosine_with_warmup, ...)``).
    """

    def __init__(self, model, lr: float = 5e-5, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.01,
                 max_grad_norm: Optional[float] = 1.0, lr_schedule: Optional[Callable[[int], float]] = None,
                 params: Optional[ParamArena] = None):
        self.params = params or getattr(model, "_arena", None) or ParamArena(model)
        self.layout = self.params.layout
        dev = self.params.flat.device
        self.lr, self.betas, self.eps, self.weight_decay = lr, betas, eps, weight_decay
        self.max_grad_norm, self.lr_schedule = max_grad_norm, lr_schedule
        self.exp_avg = torch.zeros_like(self.params.flat)
        self.exp_avg_sq = torch.zeros_like(self.params.flat)
        self.steps = 0
        # frozen parameters (requires_grad=False at construction, e.g. a frozen encoder under a fine-tuned head) are skipped
        frozen = [k for k, p in self.params.model.named_parameters() if not p.requires_grad]
        starts, flags = self.layout.decay_segments(frozen)
        # the native backward writes a gradient for every parameter; torch's clip_grad_norm_ never sees a frozen one (its
        # .grad is None), so those views are zeroed before the global norm
        self._frozen_views = [self.layout.offsets[k] for k in frozen]  # (offset, count)
        self.seg_start = torch.tensor(starts, dtype=torch.int32, device=dev)
        self.seg_nodecay = torch.tensor(flags, dtype=torch.uint8, device=dev)
        self.norm_sq = torch.zeros(1, dtype=torch.float32, device=dev)
        self.ws = torch.empty(int(load().smbv_sumsq_workspace_floats()), dtype=torch.float32, device=dev)

    def current_lr(self) -> float:
        return self.lr if self.lr_schedule is None else float(self.lr_schedule(self.steps))

    def grad_norm(self) -> torch.Tensor:
        """device scalar: the global L2 norm of the gradients seen by the last `step` (before clipping)."""
        return self.norm_sq.sqrt()

    def grad_arena(self) -> GradArena:
        """A gradient arena with this optimiser's layout, assigned to `p.grad` of every parameter: torch autograd then
        accumulates straight into the flat buffer (for modules that are differentiated by autograd, e.g. the reference's
        models driven through the attention plug-in).  Call `.zero()` on it before each backward."""
        ga = GradArena(self.params.model, self.params.flat.device, self.layout)
        ga.assign_to_params()
        return ga

    def step(self, grads: GradArena) -> None:
        if grads.layout.total != self.layout.total or grads.layout.offsets != self.layout.offsets:
            raise ValueError("FusedAdamW: gradient arena and parameter arena have different layouts")
        g = grads.flat
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        clip = self.max_grad_norm is not None and self.max_grad_norm > 0
        if clip:
            for o, n in self._frozen_views:
                g[o:o + n].zero_()
            call("smbv_sumsq_f32", ops._ptr(g), g.numel(), ops._ptr(self.ws), ops._ptr(self.norm_sq), st)
        lr = self.current_lr()
        self.steps += 1
        call("smbv_adamw_step", ops._ptr(self.params.flat), ops._ptr(self.params.bf16), ops._ptr(g), ops._ptr(self.exp_avg),
             ops._ptr(self.exp_avg_sq), g.numel(), ops._ptr(self.seg_start), ops._ptr(self.seg_nodecay), self.seg_start.numel(),
             float(lr), float(self.betas[0]), float(self.betas[1]), float(self.eps), float(self.weight_decay), self.steps,
             ops._ptr(self.norm_sq) if clip else C.c_void_p(0), float(self.max_grad_norm or 0.0), st)
        invalidate = getattr(self.params.model, "invalidate_packed", None)
        if invalidate is not None:  # modules that cache packed operands keyed on torch's version counters (vjepa.py)
            invalidate()

    # ---- checkpoint / resume (HF Trainer saves optimizer.pt next to the model, SURVEY.md §5) ----
    def state_dict(self) -> dict:
        v_m, v_v = self.layout.views(self.exp_avg), self.layout.views(self.exp_avg_sq)
        return {"step": self.steps, "exp_avg": {k: t.clone() for k, t in v_m.items()},
                "exp_avg_sq": {k: t.clone() for k, t in v_v.items()},
                "hyper": dict(lr=self.lr, betas=self.betas, eps=self.eps, weight_decay=self.weight_decay, max_grad_norm=self.max_grad_norm)}

    def load_state_dict(self, sd: dict) -> None:
        v_m, v_v = self.layout.views(self.exp_avg), self.layout.views(self.exp_avg_sq)
        with torch.no_grad():
            for k in v_m:
                v_m[k].copy_(sd["exp_avg"][k])
                v_v[k].copy_(sd["exp_avg_sq"][k])
        self.steps = int(sd["step"])


class EmaTarget:
    """Momentum (EMA) copy of a model — the V-JEPA target encoder (reference src/run_vjepa.py:87-107: `copy.deepcopy(model)`,
    `requires_grad = False`, `param_k.mul_(m).add_(param_q, alpha=1-m)` for every parameter after each step) as ONE launch over
    two flat arenas with the same layout (`smbv_ema_update`, bit-exact with the per-parameter torch loop)."""

    def __init__(self, model, momentum: float = 0.99925, source_params: Optional[ParamArena] = None):
        import copy

        self.momentum = float(momentum)
        self.source = source_params or getattr(model, "_arena", None) or ParamArena(model)
        arena, model._arena = getattr(model, "_arena", None), None  # the arena must not be deep-copied along with the module
        try:
            self.model = copy.deepcopy(model)
        finally:
            model._arena = arena
        for p in self.model.parameters():
            p.requires_grad = False
        self.params = ParamArena(self.model, self.source.layout, with_bf16=False)
        self._runner = None

    def encode(self, pixel_values_videos: torch.Tensor) -> torch.Tensor:
        """Target-encoder forward of a V-JEPA model (reference src/run_vjepa.py:126-135: `self.target_encoder(...,
        skip_predictor=True)` under no_grad) on the native encoder kernels, reading the momentum weights in place:
        fp32 last_hidden_state [B, N, d]."""
        if self._runner is None:
            from .vjepa import VJepaEncoderRunner

            self._runner = VJepaEncoderRunner(self.model.encoder, self.model.config)
        return self._runner(pixel_values_videos)

    def update(self) -> None:
        if self._runner is not None:
            self._runner.invalidate()  # the kernel below does not bump torch's parameter versions
        n = self.params.flat.numel()
        call("smbv_ema_update", ops._ptr(self.params.flat), ops._ptr(self.source.flat), n, self.momentum, float(1.0 - self.momentum),
             C.c_void_p(torch.cuda.current_stream().cuda_stream))
