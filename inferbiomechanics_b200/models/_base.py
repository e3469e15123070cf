"""Shared plumbing of the drop-in model classes: arena management and dict-input packing."""
from __future__ import annotations

from typing import Dict, Optional, Sequence

import torch
import torch.nn as nn

from .. import _lib, ops
from ..keys import LOSS_QUANTITIES, MODEL_INPUT_ORDER
from ..params import ParamArena


class EngineModule(nn.Module):
    """nn.Module whose parameters are views into a flat HBM arena read by libibm_b200 kernels."""

    LATENCY_BATCH = 16      # inference batches up to this size replay a captured CUDA graph (the viewers' batch-of-1 path)
    trains_by_diffusion = False     # True: the Trainer's step feeds noised labels and timesteps (GaussianDiffusion.q_sample)

    def _init_engine_state(self):
        self._arena: Optional[ParamArena] = None
        self._engine = None
        self._stage: Dict[tuple, torch.Tensor] = {}
        self._lat: Dict[tuple, dict] = {}

    def _device(self) -> torch.device:
        p = next(self.parameters())
        if not p.is_cuda:
            raise _lib.IbmError(
                f"{type(self).__name__} runs only on a B200: move it to CUDA with .to('cuda') "
                "(inferbiomechanics_b200 has no CPU fallback)")
        return p.device

    def _build_engine(self, arena: ParamArena):
        raise NotImplementedError

    def engine(self):
        dev = self._device()
        if self._arena is None or not self._arena.intact():
            self._arena = ParamArena(list(self.named_parameters()), dev)
            self._engine = self._build_engine(self._arena)
            # module loop (the reference's autograd + DDP idiom): every data-parallel rank draws its own dropout masks, as
            # per-process torch RNGs do; the native Trainer re-seeds with its own seed and step count (Trainer.seed_rng)
            from ..parallel import world
            self._engine.set_rng(0, world()[0], 0, None)
        else:
            self._arena.sync_shadow()
        return self._engine

    @property
    def arena(self) -> ParamArena:
        self.engine()
        return self._arena

    # ---- engine backward for the autograd bridges ------------------------------------------------------
    def _engine_backward(self, B: int, F: int) -> tuple:
        """Runs the engine backward (its dout already written) into the scratch gradient arena, leaving the ``.grad`` arena
        alone, and returns one gradient per parameter for autograd."""
        arena = self._arena
        scratch = arena.scratch_grad()
        scratch.zero_()
        arena.grad_target = scratch
        try:
            self._engine.backward(B, F)
        finally:
            arena.grad_target = arena.grad
        grads = []
        for n, p in zip(arena.names, arena.params):
            o, k = arena.offsets[n]
            grads.append(scratch[o:o + k].view(p.shape).clone())
        return tuple(grads)

    def _quantities(self, x: torch.Tensor, B: int, F: int, Fo: int) -> Dict[str, torch.Tensor]:
        """The output dict of an engine output (or a clone of one): the four quantities of the last Fo frames."""
        return dict(zip(LOSS_QUANTITIES, self._engine.quantity_views(x, B, F, Fo)))

    # ---- dict → packed bf16 rows ---------------------------------------------------------------
    def _pack_dict(self, input: Dict[str, torch.Tensor], layout, F: int, keys: Sequence[str] = MODEL_INPUT_ORDER) -> None:
        """torch.concat([...10 keys...], -1) of the reference (FeedForward…py:97-108), as one kernel
        writing bf16 rows into ``layout`` (an engine's ``input_layout``).  CPU tensors are concatenated into one pinned
        staging buffer and moved with a single H2D copy (the reference issues one copy per forward too, after its concat)."""
        dst_bf16, frame_stride, win_extra, col0 = layout
        dev = dst_bf16.device
        ts = [input[k] for k in keys]
        B = ts[0].shape[0]
        n_rows = B * F
        if all(not t.is_cuda for t in ts):
            C = sum(t.shape[-1] for t in ts)
            key = ("pin", n_rows, C)
            if key not in self._stage:
                self._stage[key] = torch.empty(n_rows, C, dtype=torch.float32).pin_memory()
                self._stage[("dev",) + key[1:]] = torch.empty(n_rows, C, dtype=torch.float32, device=dev)
            pin, devbuf = self._stage[key], self._stage[("dev",) + key[1:]]
            torch.cat([t.reshape(n_rows, -1).to(torch.float32) for t in ts], dim=-1, out=pin)
            devbuf.copy_(pin, non_blocking=True)
            srcs = [devbuf]
        else:
            srcs = [t.to(dev, torch.float32, non_blocking=True).contiguous().view(n_rows, -1) for t in ts]
        ops.pack_inputs(srcs, n_rows, F, out_bf16=dst_bf16, frame_stride=frame_stride, win_extra=win_extra, col0=col0)

    # ---- small-batch inference latency path (SURVEY §8f-4) -------------------------------------------------------
    def _latency_path(self, B: int) -> bool:
        """The per-window viewers (visualize.py:157-186, save_prediction_csv.py:91-113, review_file.py:72-100) call
        ``model(inputs)`` with a batch of ONE window under no_grad: a handful of 5-10 us kernels behind ~15 us of host work per
        launch.  Such calls replay one captured CUDA graph instead (IBM_INFER_GRAPHS=0 keeps the eager launches)."""
        import os
        return (not torch.is_grad_enabled() and not self.training and B <= self.LATENCY_BATCH
                and os.environ.get("IBM_INFER_GRAPHS", "1") != "0")

    def _graphed_inference(self, input: Dict[str, torch.Tensor], F: int, keys: Sequence[str] = MODEL_INPUT_ORDER) -> torch.Tensor:
        """Packs the inputs into the engine's input layout and runs the inference forward, returning a clone of the engine's
        output.  The first two calls per (batch, frames) run eagerly (every lazily created buffer exists afterwards), the
        third captures, later ones copy the inputs into the static staging rows and replay.  Weights are read through the
        arena's stable pointers; ``engine()`` has already refreshed the bf16 shadow if a parameter changed."""
        eng = self._engine
        dev = self._arena.device
        ts = [input[k] for k in keys]
        B = ts[0].shape[0]
        n_rows = B * F
        C = sum(t.shape[-1] for t in ts)

        def launch(rows):
            buf, fs, we, col0 = eng.input_layout(B, F, False)
            ops.pack_inputs([rows], n_rows, F, out_bf16=buf, frame_stride=fs, win_extra=we, col0=col0)
            return eng.forward(B, F, False)

        key = (B, F, C, id(eng))
        st = self._lat.get(key)
        if st is None:
            if len(self._lat) >= 8:
                self._lat.pop(next(iter(self._lat)))
            st = self._lat[key] = dict(pin=torch.empty(n_rows, C, dtype=torch.float32).pin_memory(),
                                       rows=torch.empty(n_rows, C, dtype=torch.float32, device=dev), graph=None, out=None, calls=0,
                                       engine=eng)
        if all(not t.is_cuda for t in ts):
            torch.cat([t.reshape(n_rows, -1).to(torch.float32) for t in ts], dim=-1, out=st["pin"])
            st["rows"].copy_(st["pin"], non_blocking=True)
        else:
            torch.cat([t.to(dev, torch.float32, non_blocking=True).reshape(n_rows, -1) for t in ts], dim=-1, out=st["rows"])
        if st["graph"] is None:
            if st["calls"] < 2:
                st["calls"] += 1
                return launch(st["rows"]).clone()
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                st["out"] = launch(st["rows"])
            st["graph"] = g
        eng.refresh_weights()               # re-laid-out weight copies are refreshed outside the graph
        st["graph"].replay()
        return st["out"].clone()
