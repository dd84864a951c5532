"""Embedding extraction runner: `model.videomae(x).last_hidden_state` over a stream of host volumes, with the
host->device copy of volume i+1 and the device->host copy of embedding i-1 overlapped with the compute of volume i
(three CUDA streams, double-buffered device and pinned host buffers).

Reference loop: src/run_inference.py:99-123 (`image.to(device)`; `model.videomae(image.unsqueeze(0))`;
`last_hidden_state.cpu().numpy()`), which serialises the three phases.
"""
from __future__ import annotations

from typing import Iterable, Iterator, Optional, Sequence

import torch


class EmbeddingRunner:
    def __init__(self, model, depth: int = 2, preprocess=None, layers: Optional[Sequence[int]] = None):
        """`preprocess`: optional `data.VolumePreprocessor`; the stream then carries RAW resampled volumes ([X,Y,Z] fp32 or
        int16 HU — half the PCIe bytes) and the scale/pad/crop/permute tail runs on the GPU in front of the encoder.
        `layers`: hidden-state indices of a VideoMAE encoder (0 = patch embedding, k = output of block k, before the final
        LayerNorm of use_mean_pooling=False) — each result is then [len(layers), N, d] instead of last_hidden_state; only the
        requested states are copied out of the residual stream."""
        self.model = model.videomae if hasattr(model, "videomae") else model
        self.layers = None
        if layers is not None:
            if hasattr(self.model, "get_vision_features"):
                raise ValueError("layers= is implemented for the VideoMAE encoder")
            from .modeling import _check_layers

            self.layers = _check_layers(layers, self.model.config.num_hidden_layers)
        self.preprocess = preprocess
        self.dev = next(self.model.parameters()).device
        self.depth = depth
        self.s_in, self.s_out = torch.cuda.Stream(self.dev), torch.cuda.Stream(self.dev)
        self.dev_in = [None] * depth
        # depth + 1 pinned result buffers: the one handed to the consumer is not a copy target again until the consumer
        # has asked for the result after the next one (see embed_stream)
        self.host_out = [None] * (depth + 1)
        self.ev_in = [torch.cuda.Event() for _ in range(depth)]
        self.ev_done = [torch.cuda.Event() for _ in range(depth)]
        self.ev_out = [torch.cuda.Event() for _ in range(depth + 1)]

    @torch.no_grad()  # inference: the differentiable encoder path (activations kept for backward) must never be taken here
    def _submit(self, i: int, vol: torch.Tensor) -> None:
        """Enqueue H2D + compute + D2H of volume i (host tensor [1,T,1,H,W] or [T,1,H,W], ideally pinned)."""
        k, ko = i % self.depth, i % (self.depth + 1)
        if self.preprocess is None and vol.dim() == 4:
            vol = vol.unsqueeze(0)
        compute = torch.cuda.current_stream(self.dev)
        with torch.cuda.stream(self.s_in):
            self.s_in.wait_event(self.ev_done[k])  # the previous user of this device buffer has been consumed
            if self.dev_in[k] is None or self.dev_in[k].shape != vol.shape or self.dev_in[k].dtype != vol.dtype:
                self.dev_in[k] = torch.empty(vol.shape, dtype=vol.dtype if self.preprocess is not None else torch.float32, device=self.dev)
            self.dev_in[k].copy_(vol, non_blocking=True)
            self.ev_in[k].record(self.s_in)
        compute.wait_event(self.ev_in[k])
        x = self.dev_in[k] if self.preprocess is None else self.preprocess(self.dev_in[k]).unsqueeze(0)
        if self.layers is not None:  # [1, N, d] states, copied into the rows of one [len(layers), N, d] result
            _, states = self.model.encode(self.model._volume(x), keep=self.layers)
            parts = [states[j] for j in self.layers]
            shape = (len(parts), *parts[0].shape[1:])
        else:
            # V-JEPA models expose the encoder-only pass as get_vision_features (modeling_vjepa.py:1151-1153)
            emb = self.model.get_vision_features(x) if hasattr(self.model, "get_vision_features") else self.model(x).last_hidden_state
            parts, shape = [emb], emb.shape
        self.ev_done[k].record(compute)
        with torch.cuda.stream(self.s_out):
            self.s_out.wait_event(self.ev_done[k])
            if self.host_out[ko] is None or self.host_out[ko].shape != shape:
                self.host_out[ko] = torch.empty(shape, dtype=torch.float32).pin_memory()
            if self.layers is None:
                self.host_out[ko].copy_(parts[0], non_blocking=True)
            else:
                for j, h in enumerate(parts):
                    self.host_out[ko][j].copy_(h[0], non_blocking=True)
            for h in parts:
                h.record_stream(self.s_out)
            self.ev_out[ko].record(self.s_out)

    def embed_stream(self, volumes: Iterable[torch.Tensor], copy: bool = False) -> Iterator[torch.Tensor]:
        """Yields the fp32 embedding [1, N, d] ([len(layers), N, d] with `layers`) of every volume, in order, as a pinned host
        tensor.

        Zero-copy by default: result i aliases one of `depth + 1` rotating pinned buffers and stays valid while the consumer
        holds result i + 1 (a one-item look-ahead is safe); it is overwritten once result i + 2 has been requested.  Keep a
        result longer by cloning it, or pass `copy=True` to receive fresh (unpinned) tensors — e.g. for
        `list(runner.embed_stream(...))`."""
        n_sub = 0
        n_out = 0
        hb = self.depth + 1

        def take(i):
            self.ev_out[i % hb].synchronize()
            return self.host_out[i % hb].clone() if copy else self.host_out[i % hb]

        for vol in volumes:
            if n_sub - n_out >= self.depth:  # keep at most `depth` volumes in flight
                yield take(n_out)
                n_out += 1
            self._submit(n_sub, vol)
            n_sub += 1
        while n_out < n_sub:
            yield take(n_out)
            n_out += 1
