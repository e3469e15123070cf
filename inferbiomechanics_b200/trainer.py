"""B200-native training step for the reference's training loop shape
(/root/reference/src/cli/train.py:240-284): zero_grad → forward → RegressionLossEvaluator → backward
→ (DDP allreduce) → optimizer.step, without autograd, without per-step host syncs:

    grads.zero_ (one memset of the flat arena)
    window packer  → bf16 activations            (1-2 kernels)
    forward engine → fp32 outputs                (tcgen05 GEMMs + fused elementwise)
    fused loss fwd → fp32[40] result on device   (1 kernel)
    fused loss bwd → bf16 d loss/d out           (1 kernel)
    backward engine → flat fp32 grad arena       (bucketed NCCL allreduce fired layer by layer)
    fused optimizer → params + state + bf16 shadow (1 kernel, 1/W folded in)

Works for ``FeedForwardBaseline``, ``Groundlink`` and ``DiffusionDenoiser`` through their engines' common step interface
(``input_layout``, ``forward``, ``dout``, ``quantity_views``, ``backward``, ``bucket_boundaries``, ``set_rng``).  The
drop-in classes remain usable with the reference's own autograd loop; this is the path bench.py times.
"""
from __future__ import annotations

import argparse
import contextlib
import gc
import math
import os
from typing import Dict, Iterator, List, Optional

import torch

from . import ops, parallel
from .data.window_store import WindowStore
from .diffusion import GaussianDiffusion
from .engine import quantity_split
from .keys import LOSS_QUANTITIES, MODEL_INPUT_ORDER
from .loss.RegressionLossEvaluator import COP_FORCE_THRESHOLD, component_weights

ALL_COMPONENTS = argparse.Namespace(predict_grf_components=list(range(6)), predict_cop_components=list(range(6)),
                                    predict_moment_components=list(range(6)), predict_wrench_components=list(range(12)))


def _time_kernel(fn, iters: int = 20) -> float:
    """Average GPU time of one launch: `iters` launches are captured in a CUDA graph and the replay is timed with
    events, so host-side launch overhead (ctypes marshalling is ~50-100 us per call, longer than these kernels)
    is not part of the number."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(iters):
            fn()
    g.replay()                                   # warm replay
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


LR_SCHEDULES = tuple(ops.LR_SCHEDULES)                # the kernel's schedule codes, in the order of their values


def lr_lambda(n: int, warmup_steps: int, schedule: str, total_steps: int, lr_ratio: float) -> float:
    """Learning-rate factor of the 1-based step n, the host twin of the optimizer kernel's (include/ibm_b200.h,
    ibm_optimizer_step_sched): n / W during a warm-up of W steps, then 1 (constant) or a cosine from 1 down to
    ``lr_ratio`` = lr_min / lr at step ``total_steps``.  ``LambdaLR(opt, lambda s: lr_lambda(s + 1, ...))`` hands the
    optimizer's n-th step() lr * lr_lambda(n)."""
    if warmup_steps > 0 and n <= warmup_steps:
        return n / warmup_steps
    if schedule == "constant":
        return 1.0
    p = min(max((n - warmup_steps) / (total_steps - warmup_steps), 0.0), 1.0)
    return lr_ratio + (1.0 - lr_ratio) * (0.5 * (1.0 + math.cos(math.pi * p)))


def check_clip_sched(lr: float, clip_grad_norm: float, lr_warmup_steps: int, lr_schedule: str, lr_min: float,
                     total_steps: Optional[int], flag: str = "") -> None:
    """ValueError for settings the scheduled optimizer cannot run; ``flag`` = '--' names the CLI flags instead."""
    def name(k):
        return f"--{k.replace('_', '-')}" if flag else k
    if not clip_grad_norm >= 0.0:
        raise ValueError(f"{name('clip_grad_norm')} must be >= 0 (0 = no clipping), got {clip_grad_norm}")
    if lr_warmup_steps < 0:
        raise ValueError(f"{name('lr_warmup_steps')} must be >= 0, got {lr_warmup_steps}")
    if lr_schedule not in LR_SCHEDULES:
        raise ValueError(f"{name('lr_schedule')} must be one of {LR_SCHEDULES}, got {lr_schedule!r}")
    if not lr_min >= 0.0:
        raise ValueError(f"{name('lr_min')} must be >= 0, got {lr_min}")
    if lr_min > lr:
        raise ValueError(f"{name('lr_min')} ({lr_min}) must not exceed the learning rate ({lr})")
    if total_steps is not None and total_steps < 0:
        raise ValueError(f"total_steps must be >= 0, got {total_steps}")
    if lr_schedule == "cosine" and (total_steps is None or total_steps <= lr_warmup_steps):
        raise ValueError(f"the cosine schedule needs total_steps > {name('lr_warmup_steps')} ({lr_warmup_steps}), got {total_steps}")


def check_cond_drop(cond_drop_prob: float, trains_by_diffusion: bool, flag: str = "") -> None:
    """ValueError for a condition-dropout probability outside [0, 1], or a nonzero one for a model that does not train by
    diffusion (only the denoiser has a condition to drop); ``flag`` = '--' names the CLI flag instead."""
    name = "--cond-drop-prob" if flag else "cond_drop_prob"
    if not 0.0 <= cond_drop_prob <= 1.0:
        raise ValueError(f"{name} must lie in [0, 1] (0 = off), got {cond_drop_prob}")
    if cond_drop_prob > 0.0 and not trains_by_diffusion:
        raise ValueError(f"{name} applies to the diffusion denoiser only (classifier-free guidance)")


class Trainer:
    COND_DROP_SEED = 0x63666764         # Philox key constant of the condition-dropout masks
    cond_drop_prob = 0.0

    def __init__(self, model, opt_type: str = "rmsprop", lr: float = 1e-4, args: Optional[argparse.Namespace] = None,
                 diffusion: Optional[GaussianDiffusion] = None, bucket_mb: float = 8.0, seed: int = 0, ema_decay: float = 0.0,
                 clip_grad_norm: float = 0.0, lr_warmup_steps: int = 0, lr_schedule: str = "constant", lr_min: float = 0.0,
                 total_steps: Optional[int] = None, cond_drop_prob: float = 0.0):
        if not 0.0 <= ema_decay < 1.0:
            raise ValueError(f"ema_decay must be in [0, 1) (0 = no EMA), got {ema_decay}")
        check_clip_sched(lr, clip_grad_norm, lr_warmup_steps, lr_schedule, lr_min, total_steps)
        check_cond_drop(cond_drop_prob, getattr(model, "trains_by_diffusion", False))
        self.model = model
        self.eng = model.engine()
        self.arena = model.arena
        self.opt_type, self.lr = opt_type, lr
        self.weights = component_weights(args or ALL_COMPONENTS)
        self.rank, self.world = parallel.world()
        self.step_count = 0
        self.seed = seed
        # diffusion training (the denoiser): noised labels as input, no graph capture, overlapped allreduce buckets
        self.diffusion = (diffusion or GaussianDiffusion(device=self.arena.device)) if model.trains_by_diffusion else None
        n = self.arena.total
        dev = self.arena.device
        self.state0 = torch.zeros(n, device=dev) if opt_type != "sgd" else None
        self.state1 = torch.zeros(n, device=dev) if opt_type in ("adam", "adadelta", "adamax") else None
        self.results: List[torch.Tensor] = []              # fp32[40] per step, device-resident
        self._result_ring = [torch.zeros(40, device=dev) for _ in range(8)]
        bucket_mb = float(os.environ.get("IBM_BUCKET_MB", bucket_mb))      # experiments: bucket size of the gradient allreduce
        # FeedForward / Groundlink gradients are a few MB: one allreduce of the whole arena after backward ("tail") costs less
        # than a bucket per layer group (0.46 vs 0.51 ms per B = 32 step on 2 GPUs) and leaves one point in the step where a
        # captured step is cut in two (see _train_step_graphed).  The denoiser keeps the overlapped buckets unless IBM_ALLREDUCE says otherwise.
        self.use_graphs = os.environ.get("IBM_TRAIN_GRAPHS", "1") != "0"
        self.dp_graphs = self.use_graphs and self.diffusion is None and os.environ.get("IBM_TRAIN_GRAPHS_DP", "1") != "0"
        buckets = parallel.make_buckets(self.eng.bucket_boundaries(), n, int(bucket_mb * (1 << 20) / 4))
        self.bucketer = parallel.GradBucketer(self.arena.grad, buckets,
                                              mode=None if self.diffusion is not None else os.environ.get("IBM_ALLREDUCE", "tail"))
        self.eng.bucket_hook = self.bucketer.group_done
        # DDP constructor semantics: everyone starts from rank 0's parameters (train.py:175)
        self.bucketer.broadcast_(self.arena.master)
        self.arena.sync_shadow(force=True)
        # exponential moving average of the weights, updated by the optimizer kernel: taken after the broadcast, it stays
        # identical across data-parallel ranks because their masters are bit-identical after every step
        self.ema_decay = float(ema_decay)
        self.ema: Optional[torch.Tensor] = self.arena.master.clone() if ema_decay > 0 else None
        self._in_ema = False
        # global-norm gradient clipping and the learning-rate schedule, both evaluated on the device by the optimizer kernel
        # from the device step counter, so captured steps replay with the values of their own step
        self.clip_grad_norm = float(clip_grad_norm)
        self.lr_warmup_steps, self.lr_schedule, self.lr_min = int(lr_warmup_steps), lr_schedule, float(lr_min)
        self.total_steps = int(total_steps) if total_steps is not None else 0
        self.scheduled = self.lr_warmup_steps > 0 or lr_schedule != "constant"
        self._clip_ws = ops.GradClipWorkspace(dev) if self.clip_grad_norm > 0 else None
        # classifier-free guidance training: the denoiser's condition is zeroed for a random fraction of the windows of each
        # step, Philox keyed by (COND_DROP_SEED ^ trainer seed) + rank and offset by the global step count, so every rank
        # draws its own masks and a resumed run continues the sequence
        self.cond_drop_prob = float(cond_drop_prob)
        self._cond_drop_seed = (self.COND_DROP_SEED ^ ((seed * 0x9E3779B1) & 0x7FFFFFFF)) + self.rank
        # device-resident 1-based step counter: incremented by a one-thread kernel at the start of every step, read by the
        # dropout kernels (Philox offset) and the optimizer kernel (Adam / Adamax bias correction), so that a captured step
        # can be replayed although those values change from step to step
        self.step_dev = torch.zeros(1, dtype=torch.int64, device=dev)
        self.seed_rng()
        self._store_labels: Dict[int, torch.Tensor] = {}       # batch size -> (B, Fo, 30) labels packed from a window store
        self._host_stage: Dict[tuple, tuple] = {}              # (batch size, slot) -> (device staging tensors, ready, consumed)
        self._host_labels: Dict[int, torch.Tensor] = {}        # batch size -> (B, Fo, 30) labels packed from host batches
        self._gen = torch.Generator(device=dev).manual_seed(seed + 7919 * self.rank)
        # CUDA-graph replay of the (launch-bound) FeedForward step: key -> [eager steps seen, graph, static idx, static result]
        self._graphs: Dict[tuple, list] = {}

    def seed_rng(self) -> None:
        """Dropout masks: Philox keyed by (engine constant ^ trainer seed) + rank, offset by the GLOBAL step count — every
        data-parallel rank draws its own mask (the reference's per-process torch RNG does), and a resumed run continues the
        sequence instead of replaying the masks of step 1."""
        self.eng.set_rng((self.seed * 0x9E3779B1) & 0x7FFFFFFF, self.rank, self.step_count, self.step_dev)
        self.step_dev.fill_(self.step_count)

    # ---- one optimisation step on windows idx of a store -------------------------------------------
    def _graphable(self) -> bool:
        """The FeedForward / Groundlink steps are 25-80 short launches: at the reference's batch sizes (32-64 windows,
        train.py:52) the host, not the GPU, paces them, so a step is captured once per (store, batch size) and replayed —
        with dropout and Adam/Adamax too, whose per-step values come from the device-resident step counter.  Data-parallel
        steps are captured as TWO graphs cut at the gradient allreduce, which stays an ordinary NCCL call between the two
        replays (a captured NCCL allreduce hung on replay in both attempts of round 2 — side-stream buckets and a single
        collective on the capture stream — so NCCL is kept out of the graphs).  Not captured: the denoiser (its step is
        GPU-bound and draws timesteps with a torch generator).  IBM_TRAIN_GRAPHS=0 switches replay off altogether,
        IBM_TRAIN_GRAPHS_DP=0 for data-parallel runs only."""
        if not self.use_graphs or self.diffusion is not None:
            return False
        return self.world == 1 or (self.dp_graphs and self.bucketer.mode == "tail")

    def train_step(self, store: WindowStore, idx: torch.Tensor) -> torch.Tensor:
        """Returns the device-resident fp32[40] result (loss at [0]); nothing is synchronised."""
        if self._graphable():
            return self._train_step_graphed(store, idx)
        return self._train_step_eager(store, idx)

    def _capture_step(self, store: WindowStore, idx: torch.Tensor) -> list:
        """Captures one eager step into CUDA graphs: one graph on a single rank; under data parallelism [everything up to the
        end of backward] and [optimizer], the bucketer's finish_hook closing the first graph and opening the second at the
        point where the eager step issues its allreduce.  Capture does not execute."""
        graphs = [torch.cuda.CUDAGraph()]
        mode = "thread_local" if self.world > 1 else "global"     # the NCCL watchdog thread may query events meanwhile
        # as torch.cuda.graph() does: collect garbage first — a CUDAGraph (or a tensor with cross-stream events) finalised by
        # the cyclic collector in the middle of the capture issues calls that invalidate it — and keep the collector off meanwhile
        gc.collect()
        torch.cuda.synchronize()
        gc_was_on = gc.isenabled()
        gc.disable()
        side = torch.cuda.Stream(device=self.arena.device)
        side.wait_stream(torch.cuda.current_stream())

        def cut():
            graphs[-1].capture_end()
            nxt = torch.cuda.CUDAGraph()
            nxt.capture_begin(pool=graphs[0].pool(), capture_error_mode=mode)
            graphs.append(nxt)

        self.bucketer.finish_hook = cut if self.world > 1 else None
        # the replays must re-derive cached weight layouts (Groundlink's conv GEMM layouts) from the masters the previous
        # step wrote: a stale weights version makes the captured forward record that refresh
        self.arena.bump_version()
        try:
            with torch.cuda.stream(side):
                graphs[0].capture_begin(capture_error_mode=mode)
                try:
                    self._train_step_eager(store, idx)
                finally:
                    graphs[-1].capture_end()
        finally:
            self.bucketer.finish_hook = None
            if gc_was_on:
                gc.enable()
        torch.cuda.current_stream().wait_stream(side)
        return graphs

    def _train_step_graphed(self, store: WindowStore, idx: torch.Tensor) -> torch.Tensor:
        # launch arguments baked into the captured step: the schedule's parameters, never a per-step learning rate
        key = (id(store), idx.numel(), self.lr, self.model.training, self._clip_sched_key())
        g = self._graphs.get(key)
        if g is None:
            if len(self._graphs) >= 8:
                self._graphs.pop(next(iter(self._graphs)))
            g = self._graphs[key] = [0, None, None, None, store]     # holds the store: its id() cannot be recycled
        if g[1] is None:
            if g[0] < 2:                         # two eager steps first: every lazily created buffer / attribute exists
                g[0] += 1
                return self._train_step_eager(store, idx)
            g[2] = idx.clone()
            g[3] = torch.zeros(40, device=idx.device)
            ring, self._result_ring = self._result_ring, [g[3]]
            count = self.step_count
            torch.cuda.synchronize()
            try:
                graphs = self._capture_step(store, g[2])
            finally:
                self._result_ring = ring
            self.step_count = count              # capture does not execute: the replay below is this step
            self.seed_rng()
            g[1] = graphs
        g[2].copy_(idx, non_blocking=True)
        g[1][0].replay()
        for graph in g[1][1:]:                   # data parallel: [... backward] -> allreduce of the arena -> [optimizer]
            self.bucketer.allreduce_all()
            graph.replay()
        self.step_count += 1
        self.arena.bump_version()                # the replayed optimizer wrote the masters
        result = self._result_ring[self.step_count % len(self._result_ring)]
        result.copy_(g[3], non_blocking=True)
        return result

    def _train_step_eager(self, store: WindowStore, idx: torch.Tensor) -> torch.Tensor:
        B, F = idx.numel(), store.F
        lab = self._labels(store, idx)
        self._begin_step()
        store.pack(idx, self.eng.input_layout(B, F, True))
        return self._step(B, F, lab)

    def _labels(self, store: WindowStore, idx: torch.Tensor) -> torch.Tensor:
        B = idx.numel()
        if B not in self._store_labels:
            self._store_labels[B] = torch.empty(B, store.Fo, 30, dtype=torch.float32, device=self.arena.device)
        return store.labels(idx, self._store_labels[B])

    def _begin_step(self) -> None:
        self.arena.zero_grad()
        self.bucketer.begin_step()
        ops.counter_add(self.step_dev, 1)        # the step that starts now: value step_count + 1 on the device

    def _step(self, B: int, F: int, lab: torch.Tensor) -> torch.Tensor:
        """The step after packing: forward, fused loss forward / backward on the (B, Fo, ·) quantity views of the output and
        of its gradient, backward into the flat gradient arena, allreduce, fused optimizer."""
        eng = self.eng
        if self.diffusion is not None:
            # x_t = q_sample(labels, t) into columns 0..29 of the input rows, t drawn per window
            t = eng.t_buffer(B, True)
            t.copy_(torch.randint(0, self.diffusion.T, (B,), device=t.device, generator=self._gen, dtype=torch.int32))
            xc, ld, _, _ = eng.input_layout(B, F, True)
            self.diffusion.q_sample(lab.view(B, -1), t, None, xt_bf16=xc, bf16_ld=ld, seed=self.seed + self.rank, offset=self.step_count)
            if self.cond_drop_prob > 0.0:
                # the null condition is all-zero kinematics; the in-projection's weight gradient reads the same zeroed rows
                ops.cond_dropout(xc, B, F, 30, eng.c_in, self.cond_drop_prob, self._cond_drop_seed, self.step_count)
        Fo = lab.shape[1]
        outs = eng.quantity_views(eng.forward(B, F, True), B, F, Fo)
        labs, gviews = quantity_split(lab), eng.quantity_views(eng.dout(B, F), B, F, Fo)
        result = self._result_ring[self.step_count % len(self._result_ring)]
        ops.regression_loss_fwd(outs, labs, self.weights, COP_FORCE_THRESHOLD, result=result)
        ops.regression_loss_bwd(outs, labs, self.weights, gviews, threshold=COP_FORCE_THRESHOLD)
        eng.backward(B, F)
        self.bucketer.finish()
        self.optimizer_step()
        return result

    def optimizer_step(self) -> None:
        """After ``bucketer.finish()``, on the compute stream: the gradient arena holds the allreduced sum.  With clipping on,
        the norm kernel reads it first and the scheduled optimizer applies the coefficient it wrote."""
        self.step_count += 1
        if self._clip_ws is None and not self.scheduled:
            ops.optimizer_step(self.opt_type, self.arena.master, self.arena.grad, self.state0, self.state1, self.arena.shadow,
                               self.lr, 1.0 / self.world, self.step_count, step_dev=self.step_dev, ema=self.ema,
                               ema_decay=self.ema_decay)
        else:
            clip = None
            if self._clip_ws is not None:
                clip = ops.grad_clip_coef(self.arena.grad, self.clip_grad_norm, 1.0 / self.world, self._clip_ws)
            ops.optimizer_step(self.opt_type, self.arena.master, self.arena.grad, self.state0, self.state1, self.arena.shadow,
                               self.lr, 1.0 / self.world, self.step_count, step_dev=self.step_dev, ema=self.ema,
                               ema_decay=self.ema_decay, clip=clip, schedule=self.lr_schedule,
                               warmup_steps=self.lr_warmup_steps, total_steps=self.total_steps, lr_min=self.lr_min)
        self.arena.mark_shadow_fresh()

    # ---- gradient clipping and learning-rate schedule ----------------------------------------------------------------
    def _clip_sched_key(self) -> Optional[tuple]:
        if self._clip_ws is None and not self.scheduled:
            return None
        return (self.clip_grad_norm, self.lr_warmup_steps, self.lr_schedule, self.total_steps, self.lr_min)

    def current_lr(self) -> float:
        """The learning rate the next step applies (the optimizer kernel derives the same value on the device)."""
        if not self.scheduled:
            return self.lr
        return self.lr * lr_lambda(self.step_count + 1, self.lr_warmup_steps, self.lr_schedule, self.total_steps,
                                   self.lr_min / self.lr if self.lr > 0 else 0.0)

    def grad_norm_stats(self, reset: bool = True) -> dict:
        """Mean pre-clip global gradient norm, the number of clipped steps and the number of steps since the last reset:
        one read of the device record (a synchronisation), meant for report time."""
        if self._clip_ws is None:
            raise RuntimeError("this Trainer does not clip gradients (construct it with clip_grad_norm > 0)")
        total, steps, clipped = self._clip_ws.record.tolist()
        if reset:
            self._clip_ws.record.zero_()
        return {"mean_norm": total / steps if steps else float("nan"), "clipped": int(clipped), "steps": int(steps)}

    # ---- exponential moving average of the weights -------------------------------------------------------------------
    def _require_ema(self) -> None:
        if self.ema is None:
            raise RuntimeError("this Trainer keeps no EMA of the weights (construct it with ema_decay > 0)")

    def ema_state_dict(self) -> dict:
        """``model.state_dict()``'s keys with the parameters taken from the EMA arena and the buffers (BatchNorm running
        statistics) copied from the model, so ``model.load_state_dict`` of any instance of the class accepts it."""
        self._require_ema()
        out = {}
        for k, v in self.model.state_dict().items():
            if k in self.arena.offsets:
                o, n = self.arena.offsets[k]
                out[k] = self.ema[o:o + n].view(v.shape).clone()
            else:
                out[k] = v.clone()
        return out

    def load_ema_state_dict(self, sd: Optional[dict]) -> None:
        """Inverse of ``ema_state_dict``: the parameters' entries go into the EMA arena (buffers are the model's own).
        ``None`` restarts the average at the current weights (a resumed run whose checkpoint holds no EMA)."""
        self._require_ema()
        if sd is None:
            self.ema.copy_(self.arena.master)
            return
        if all(k.startswith("module.") for k in sd):
            sd = {k[len("module."):]: v for k, v in sd.items()}
        keys = self.model.state_dict().keys()
        missing = [k for k in self.arena.names if k not in sd]
        unexpected = [k for k in sd if k not in keys]
        if missing or unexpected:
            raise ValueError(f"EMA state dict does not match the model: missing {missing}, unexpected {unexpected}")
        for name in self.arena.names:
            o, n = self.arena.offsets[name]
            if sd[name].numel() != n:
                raise ValueError(f"EMA entry {name} has {sd[name].numel()} elements, the parameter {n}")
            self.ema[o:o + n].copy_(sd[name].reshape(-1))

    def _swap_ema(self) -> None:
        """Exchanges the contents (never the storage: captured graphs hold the pointers) of the masters and the EMA arena,
        then re-derives the bf16 shadow, the padded copies and, through the version bump, every cache keyed on
        ``ParamArena.version``.  Parameters are views re-pointed into the masters, so a copy into the masters does not move
        their ``_version``: the bump is what makes the Groundlink conv layouts and the denoiser's time-MLP table refresh."""
        tmp = self.arena.master.clone()
        self.arena.master.copy_(self.ema)
        self.ema.copy_(tmp)
        self.arena.sync_shadow(force=True)
        self.arena.bump_version()

    @contextlib.contextmanager
    def ema_weights(self) -> Iterator[None]:
        """Evaluates (``eval_step``, the model's forward, sampling) with the EMA weights in the masters; the trained weights
        are back on exit."""
        self._require_ema()
        if self._in_ema:
            raise RuntimeError("already inside ema_weights()")
        self._in_ema = True
        self._swap_ema()
        try:
            yield
        finally:
            self._swap_ema()
            self._in_ema = False

    # ---- optimizer state in torch.optim's own state_dict layout (checkpoints, train.py:270-278) -----------------------
    _OPT_CLASS = {"adagrad": "Adagrad", "adam": "Adam", "sgd": "SGD", "rmsprop": "RMSprop", "adadelta": "Adadelta", "adamax": "Adamax"}
    _OPT_STATE = {"rmsprop": ("square_avg", None), "adam": ("exp_avg", "exp_avg_sq"), "sgd": (None, None), "adagrad": ("sum", None),
                  "adadelta": ("square_avg", "acc_delta"), "adamax": ("exp_avg", "exp_inf")}

    def optimizer_state_dict(self) -> dict:
        """What ``torch.optim.<Type>(model.parameters(), lr).state_dict()`` would hold after the same steps: per-parameter
        state tensors (CPU copies of this trainer's flat state arenas, cut at the parameter offsets) keyed by the
        parameter's position in ``model.parameters()``, plus torch's own ``param_groups`` defaults — so the reference's
        ``optimizer.load_state_dict(checkpoint['optimizer_state_dict'])`` (abstract_command.py:113-114) accepts it."""
        cls = getattr(torch.optim, self._OPT_CLASS[self.opt_type])
        sd = cls(self.arena.params, lr=self.lr).state_dict()         # param_groups with torch's defaults, empty state
        n0, n1 = self._OPT_STATE[self.opt_type]
        if self.step_count > 0 and n0 is not None:
            for i, name in enumerate(self.arena.names):
                o, k = self.arena.offsets[name]
                shape = self.arena.params[i].shape
                st = {"step": torch.tensor(float(self.step_count)), n0: self.state0[o:o + k].view(shape).cpu().clone()}
                if n1 is not None:
                    st[n1] = self.state1[o:o + k].view(shape).cpu().clone()
                sd["state"][i] = st
        elif self.step_count > 0:                                    # SGD without momentum keeps no tensors
            sd["state"] = {i: {"momentum_buffer": None} for i in range(len(self.arena.names))}
        sd["ibm_b200"] = {"opt_type": self.opt_type, "step": self.step_count}
        if self.scheduled:
            # what a torch optimizer's group holds after optimizer.step(); scheduler.step() under LambdaLR
            sd["param_groups"][0]["lr"] = self.current_lr()
            sd["param_groups"][0]["initial_lr"] = self.lr
        if self._clip_sched_key() is not None:
            sd["ibm_b200"].update(clip_grad_norm=self.clip_grad_norm, lr_warmup_steps=self.lr_warmup_steps,
                                  lr_schedule=self.lr_schedule, lr_min=self.lr_min, total_steps=self.total_steps)
        if self.cond_drop_prob > 0.0:
            sd["ibm_b200"]["cond_drop_prob"] = self.cond_drop_prob
        return sd

    def load_optimizer_state_dict(self, sd: dict) -> None:
        """Inverse of ``optimizer_state_dict``; also accepts a checkpoint written by the reference's torch optimizer of the
        same type (same parameter order) and the flat blob of earlier versions of this trainer."""
        if not sd:
            return
        if "state" not in sd:                                        # legacy flat blob {'opt_type','step','state0','state1'}
            if sd.get("opt_type") != self.opt_type:
                raise ValueError(f"checkpoint optimizer {sd.get('opt_type')!r} != --opt-type {self.opt_type!r}")
            for dst, src in ((self.state0, sd.get("state0")), (self.state1, sd.get("state1"))):
                if dst is not None and src is not None:
                    dst.copy_(src)
            self.step_count = int(sd.get("step", 0))
            self.seed_rng()
            return
        tag = sd.get("ibm_b200")
        if tag is not None and tag["opt_type"] != self.opt_type:
            raise ValueError(f"checkpoint optimizer {tag['opt_type']!r} != --opt-type {self.opt_type!r}")
        n0, n1 = self._OPT_STATE[self.opt_type]
        state = sd["state"]
        if len(state) not in (0, len(self.arena.names)):
            raise ValueError(f"optimizer state holds {len(state)} parameters, the model has {len(self.arena.names)}")
        steps = set()
        for i, name in enumerate(self.arena.names):
            st = state.get(i, state.get(str(i)))
            if st is None:
                continue
            if n0 is not None:
                if n0 not in st or (n1 is not None and n1 not in st):
                    raise ValueError(f"optimizer state of parameter {i} lacks {n0!r}/{n1!r}: not a {self._OPT_CLASS[self.opt_type]} checkpoint")
                o, k = self.arena.offsets[name]
                if st[n0].numel() != k:
                    raise ValueError(f"optimizer state of {name} has {st[n0].numel()} elements, the parameter {k}")
                self.state0[o:o + k].copy_(st[n0].reshape(-1))
                if n1 is not None:
                    self.state1[o:o + k].copy_(st[n1].reshape(-1))
            if "step" in st:
                steps.add(int(float(st["step"])))
        if len(steps) > 1:
            raise ValueError(f"per-parameter step counts differ ({sorted(steps)}): the fused optimizer keeps one")
        self.step_count = steps.pop() if steps else int(tag["step"]) if tag else 0
        self.seed_rng()
        self._graphs.clear()

    # ---- evaluation (no_grad forward + loss), used by analyze / dev-eval ------------------------------
    @torch.no_grad()
    def eval_step(self, store: WindowStore, idx: torch.Tensor) -> torch.Tensor:
        if self.diffusion is not None:
            raise NotImplementedError("denoiser evaluation = reverse sampling; use GaussianDiffusion.sample")
        B, F = idx.numel(), store.F
        lab = self._labels(store, idx)
        store.pack(idx, self.eng.input_layout(B, F, False))
        out = self.eng.forward(B, F, False)
        return ops.regression_loss_fwd(self.eng.quantity_views(out, B, F, store.Fo), quantity_split(lab), self.weights)

    # ---- host-fed step (the e2e path) ----------------------------------------------------------------------------
    def make_host_batch(self, B: int, seed: int = 0, frames: Optional[int] = None):
        """Synthetic pinned host tensors shaped like a reference DataLoader batch (SURVEY §8d)."""
        m = self.model
        g = torch.Generator().manual_seed(seed)
        # window length, root-history columns and output frames of the model family: FeedForward has num_frames and a
        # stride-long history, the denoiser a fixed frame count, Groundlink windows of any length (frames=T)
        F = frames if frames is not None else getattr(m, "num_frames", getattr(m, "frames", None))
        if F is None:
            raise ValueError("Groundlink windows have no fixed length: pass frames=T")
        hist = 3 * getattr(m, "stride", m.root_history_len)
        Fo = F if getattr(m, "output_data_format", "all_frames") == "all_frames" else 1
        widths = {"pos": 23, "vel": 23, "acc": 23, "rootLinearVelInRootFrame": 3, "rootAngularVelInRootFrame": 3,
                  "rootLinearAccInRootFrame": 3, "rootAngularAccInRootFrame": 3, "jointCentersInRootFrame": 36,
                  "rootPosHistoryInRootFrame": hist, "rootEulerHistoryInRootFrame": hist}
        inputs = {k: torch.randn(B, F, widths[k], generator=g).pin_memory() for k in MODEL_INPUT_ORDER}
        scale = {LOSS_QUANTITIES[0]: 1.0, LOSS_QUANTITIES[1]: 10.0, LOSS_QUANTITIES[2]: 1.0, LOSS_QUANTITIES[3]: 1.0}
        labels = {k: (torch.randn(B, Fo, 12 if i == 3 else 6, generator=g) * scale[k]).pin_memory() for i, k in enumerate(LOSS_QUANTITIES)}
        return {"inputs": inputs, "labels": labels}

    def train_step_host(self, inputs, labels) -> float:
        """One optimisation step fed from (pinned) host tensors: async H2D copies of the 14 tensors, one packing kernel for
        the ten inputs and one for the four label tensors, the native step, then a D2H read of the loss."""
        for loss in self.train_steps_host([(inputs, labels)]):
            return loss

    def train_steps_host(self, batches):
        """Generator over host batches ``(inputs, labels)`` (dicts of pinned CPU tensors, as a DataLoader with
        ``pin_memory=True`` yields them): one optimisation step per batch, yielding that step's loss as a python float.

        Every step: H2D copy of the step's 14 tensors, packing kernels, the native step, a D2H read of the loss — pipelined
        the way a prefetching loader feeds a training loop: the copies of batch i+1 run on a copy stream into the other half
        of a double-buffered staging area while step i computes, and the loss of step i is read back only after step i+1 has
        been enqueued, so the GPU never waits for Python to launch the next step."""
        dev = self.arena.device
        copy_stream = getattr(self, "_copy_stream", None)
        if copy_stream is None:
            copy_stream = self._copy_stream = torch.cuda.Stream(device=dev)
        main = torch.cuda.current_stream(dev)
        it = iter(batches)

        def upload(batch, slot):
            inputs, labels = batch
            B = inputs[MODEL_INPUT_ORDER[0]].shape[0]
            key = (B, slot)
            if key not in self._host_stage:
                self._host_stage[key] = ({k: torch.empty(v.shape, dtype=torch.float32, device=dev) for k, v in {**inputs, **labels}.items()},
                                         torch.cuda.Event(), torch.cuda.Event())
            stage, ready, consumed = self._host_stage[key]
            copy_stream.wait_event(consumed)                  # the step that last read this slot has packed it
            with torch.cuda.stream(copy_stream):
                for k, v in {**inputs, **labels}.items():
                    stage[k].copy_(v, non_blocking=True)
                ready.record(copy_stream)
            return B, stage, ready, consumed

        def launch(up):
            B, stage, ready, consumed = up
            main.wait_event(ready)
            F = stage[MODEL_INPUT_ORDER[0]].shape[1]
            Fo = stage[LOSS_QUANTITIES[0]].shape[1]
            if B not in self._host_labels:
                self._host_labels[B] = torch.empty(B, Fo, 30, dtype=torch.float32, device=dev)
            lab = self._host_labels[B]
            ops.pack_inputs([stage[k].view(B * Fo, -1) for k in LOSS_QUANTITIES], B * Fo, Fo, out_f32=lab.view(B * Fo, 30))
            self._begin_step()
            # the ten per-key input tensors (FeedForward…py:97-108 concat order) -> the engine's packed bf16 layout, one kernel
            buf, fs, we, col0 = self.eng.input_layout(B, F, True)
            ops.pack_inputs([stage[k].view(B * F, -1) for k in MODEL_INPUT_ORDER], B * F, F, out_bf16=buf, frame_stride=fs,
                            win_extra=we, col0=col0)
            consumed.record(main)                             # staging slot is free once both packers have run
            return self._step(B, F, lab)

        try:
            nxt = upload(next(it), 0)
        except StopIteration:
            return
        slot, pending = 0, None                               # pending: (result tensor, event) of the step enqueued last
        while nxt is not None:
            cur = nxt
            result = launch(cur)
            done = torch.cuda.Event()
            done.record(main)
            slot ^= 1
            try:
                nxt = upload(next(it), slot)                  # copies of the next batch overlap this step's kernels
            except StopIteration:
                nxt = None
            if pending is not None:
                pending[1].synchronize()
                yield float(pending[0][0].item())
            # the result ring holds 8 steps: cloning is not needed for a one-step delay
            pending = (result, done)
        pending[1].synchronize()
        yield float(pending[0][0].item())

    # ---- profiling helpers used by bench.py ------------------------------------------------------------------------
    def profile_gemms(self, store, idx):
        """One extra training step with CUDA events around every tcgen05 GEMM launch (on the launching stream):
        returns (total GEMM ms, total algorithmic FLOPs = 2*M*N*K per launch, number of launches)."""
        real = ops.gemm
        recs = []

        def timed(A, Bm, out, M, N, K, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = real(A, Bm, out, M, N, K, **kw)
            e1.record()
            recs.append((e0, e1, 2.0 * M * N * K, (M, N, K)))
            return r

        # every other C-ABI entry point is timed the same way (per-kernel ms of one step, live, no profiler)
        real_call = ops.call
        krecs = []

        def timed_call(name, *a):
            if name == "ibm_gemm_bf16":
                return real_call(name, *a)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            real_call(name, *a)
            e1.record()
            krecs.append((name, e0, e1))

        ops.gemm = timed
        ops.call = timed_call
        try:
            self.train_step(store, idx)
            torch.cuda.synchronize()
        finally:
            ops.gemm = real
            ops.call = real_call
        self.last_gemm_records = [(e0.elapsed_time(e1), fl, shp) for e0, e1, fl, shp in recs]
        per = {}
        for name, e0, e1 in krecs:
            p = per.setdefault(name, [0, 0.0])
            p[0] += 1
            p[1] += e0.elapsed_time(e1)
        self.last_kernel_ms = {k: {"launches": v[0], "ms": round(v[1], 4)} for k, v in sorted(per.items(), key=lambda kv: -kv[1][1])}
        return sum(r[0] for r in self.last_gemm_records), sum(r[1] for r in self.last_gemm_records), len(recs)

    def aux_measurements(self, store, idx, pk, world):
        """HBM-bound kernels against the measured copy bandwidth (inputs >= 300 MB exceed L2), the per-shape GEMM table and the
        per-kernel times of one training step.  Reverse sampling (BASELINE configs[3]) is bench_legs.sampling_leg."""
        B = idx.numel()
        dev = self.arena.device
        hbm = pk["hbm_gbs"]
        out = {}
        if self.diffusion is not None:
            eng, F = self.eng, self.eng.F
            # stream of 16384 windows (819 200 rows): every operand set is > 200 MB, i.e. larger than the 126 MB L2,
            # so consecutive timed launches cannot re-use each other's lines
            Bb = 16384
            M = Bb * F
            rows = torch.randn(M, 32, device=dev)
            lab = torch.randn(Bb, F, 30, device=dev) * 5
            outs, labs = quantity_split(rows.view(Bb, F, 32)), quantity_split(lab)
            res = torch.zeros(40, device=dev)
            g16buf = torch.zeros(M, 32, dtype=torch.bfloat16, device=dev)
            g16 = quantity_split(g16buf.view(Bb, F, 32))

            def entry(ms, by):
                return {"bound": "hbm", "ms": ms, "achieved": by / ms / 1e6, "peak": hbm, "unit": "GB/s", "frac": by / ms / 1e6 / hbm,
                        "algorithmic_bytes": by, "rows": M}

            out["loss_fwd"] = entry(_time_kernel(lambda: ops.regression_loss_fwd(outs, labs, self.weights, result=res)), M * 240.0)
            out["loss_bwd_bf16"] = entry(_time_kernel(lambda: ops.regression_loss_bwd(outs, labs, self.weights, g16)), M * 300.0)
            x0 = lab.view(Bb, -1)
            eps = torch.randn_like(x0)
            xt = torch.empty_like(x0)
            t = torch.randint(0, 1000, (Bb,), device=dev, dtype=torch.int32)
            d = self.diffusion
            out["q_sample"] = entry(_time_kernel(lambda: ops.q_sample(x0, eps, t, d.sqrt_abar, d.sqrt_one_minus_abar, xt_f32=xt)), M * 360.0)
            tdev = torch.full((1,), 500, dtype=torch.int32, device=dev)
            xp = torch.empty(M, 30, device=dev)
            out["posterior_step"] = entry(_time_kernel(lambda: ops.posterior_step(rows, 32, x0.view(M, 30), eps.view(M, 30), tdev, d.coef_x0,
                                                                                  d.coef_xt, d.sigma, M, x_prev=xp)), M * 480.0)
            del rows, lab, g16buf, eps, xt, xp
            # the same two kernels over an analysis-sized stream (65 536 windows = 3.3 M rows, 786 MB forward): the fixed costs of
            # a 40 us launch (ramp-up, last-block fp64 reduction) are amortised, which is the regime of the analyze pass
            Bs = 65536
            Ms = Bs * F
            rows = torch.randn(Ms, 32, device=dev)
            lab = torch.randn(Bs, F, 30, device=dev) * 5
            outs, labs = quantity_split(rows.view(Bs, F, 32)), quantity_split(lab)
            g16buf = torch.zeros(Ms, 32, dtype=torch.bfloat16, device=dev)
            g16 = quantity_split(g16buf.view(Bs, F, 32))
            e = entry(_time_kernel(lambda: ops.regression_loss_fwd(outs, labs, self.weights, result=res), iters=10), Ms * 240.0)
            e["rows"] = Ms
            out["loss_fwd_stream"] = e
            e = entry(_time_kernel(lambda: ops.regression_loss_bwd(outs, labs, self.weights, g16), iters=10), Ms * 300.0)
            e["rows"] = Ms
            out["loss_bwd_bf16_stream"] = e
            del rows, lab, g16buf, outs, labs, g16
            # per-shape table of the GEMM launches of one training step (from profile_gemms)
            shapes = {}
            for ms, fl, shp in getattr(self, "last_gemm_records", []):
                e = shapes.setdefault("x".join(str(v) for v in shp), [0, 0.0, 0.0])
                e[0] += 1; e[1] += ms; e[2] += fl
            out["other_kernels_ms_per_step"] = getattr(self, "last_kernel_ms", {})
            # the HBM-bound layer kernels as they run INSIDE the training step (power-capped clocks, cold L2, neighbours' tails):
            # algorithmic bytes per launch / in-step CUDA-event time per launch, against the measured copy bandwidth
            Mrows, d_ = B * F, eng.d
            per_launch = {"ibm_attention_fwd": 8.0 * d_ * Mrows, "ibm_attention_bwd": 14.0 * d_ * Mrows,
                          "ibm_layernorm_fwd": (4.0 * d_ + 8.0) * Mrows, "ibm_layernorm_bwd": (6.0 * d_ + 8.0) * Mrows,
                          "ibm_regression_loss_fwd": 240.0 * Mrows, "ibm_regression_loss_bwd": 300.0 * Mrows}
            tab = {}
            for name, by in per_launch.items():
                rec = out["other_kernels_ms_per_step"].get(name)
                if rec and rec["ms"] > 0:
                    us = rec["ms"] * 1e3 / rec["launches"]
                    tab[name] = {"launches": rec["launches"], "us_per_launch": round(us, 1), "algorithmic_bytes": by,
                                 "achieved": by / us / 1e3, "peak": hbm, "unit": "GB/s", "frac": by / us / 1e3 / hbm}
            out["hbm_kernels_in_step"] = tab
            out["gemm_shapes_MxNxK"] = {k: {"launches": v[0], "ms": round(v[1], 4), "tflops": round(v[2] / (v[1] * 1e-3) / 1e12, 1)}
                                        for k, v in shapes.items()}
        return out
