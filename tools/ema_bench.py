"""Cost of the exponential moving average of the weights (``Trainer(ema_decay=...)``), EMA off against EMA on:

* the fused optimizer kernel alone on an arena the size of the BASELINE configs[1] denoiser's (d=512, 8 heads, FFN 2048,
  8 layers: ~25 M parameters), RMSprop and Adam, each launch fed by the device step counter as the Trainer does.  Timed with
  CUDA events over a captured graph of 50 launches (``trainer._time_kernel``); the arenas (>= 450 MB) exceed the 126 MB L2.
  Bytes from the shapes: RMSprop reads param, grad, state (12 B) and writes param, state, bf16 shadow (10 B) per parameter,
  Adam 16 B + 14 B; the EMA adds 4 B read + 4 B written.  Rates are set against the 6 536.7 GB/s HBM copy figure
  DESIGN.md quotes;
* the configs[1] denoiser training step (B = 4096 windows, F = 50, RMSprop lr 1e-4 as bench.py), two identically seeded
  models, one Trainer each, the two arms alternated within each repeat (CUDA events around `--steps` steps);
* the configs[0] FeedForward step (T = 50, stride 5, hidden 512-512, sigmoid, B = 32), graph-replayed, alternated the same way.

Reports medians over `--repeats` with min / max, the device name and power limit.  Prints one JSON line (and writes it to
--out if given).

    python tools/ema_bench.py [--repeats 5] [--steps 10] [--out result.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from inferbiomechanics_b200 import ops
from inferbiomechanics_b200.data.window_store import WindowStore
from inferbiomechanics_b200.diffusion import GaussianDiffusion
from inferbiomechanics_b200.models.DiffusionDenoiser import DiffusionDenoiser
from inferbiomechanics_b200.models.FeedForwardRegressionBaseline import FeedForwardBaseline
from inferbiomechanics_b200.trainer import Trainer, _time_kernel

DESIGN_HBM_GBS = 6536.7
DECAY = 0.999


def device_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return dict(device=name, power_limit=power, torch_device=torch.cuda.get_device_name(0))


def stats(xs, digits=4):
    return dict(median=round(statistics.median(xs), digits), min=round(min(xs), digits), max=round(max(xs), digits), n=len(xs))


def kernel_leg(n, dev, repeats):
    g = torch.Generator(device=dev).manual_seed(0)
    p = torch.randn(n, device=dev, generator=g)
    grad = torch.randn(n, device=dev, generator=g) * 1e-3
    s0, s1, ema = torch.zeros(n, device=dev), torch.zeros(n, device=dev), p.clone()
    pb = torch.empty(n, dtype=torch.bfloat16, device=dev)
    counter = torch.full((1,), 1000, dtype=torch.int64, device=dev)
    per_param = {"rmsprop": 22.0, "adam": 30.0}
    cases = [(k, e) for k in ("rmsprop", "adam") for e in (False, True)]
    times = {c: [] for c in cases}
    for _ in range(repeats):
        for kind, on in cases:
            fn = (lambda k=kind: ops.optimizer_step(k, p, grad, s0, s1, pb, 1e-4, 1.0, 1, step_dev=counter, ema=ema, ema_decay=DECAY)) \
                if on else (lambda k=kind: ops.optimizer_step(k, p, grad, s0, s1, pb, 1e-4, 1.0, 1, step_dev=counter))
            times[(kind, on)].append(_time_kernel(fn, iters=50))
    out = []
    for (kind, on), ts in times.items():
        by = n * (per_param[kind] + (8.0 if on else 0.0))
        ms = statistics.median(ts)
        gbs = by / (ms * 1e-3) / 1e9
        out.append(dict(optimizer=kind, ema=on, params=n, bytes_per_launch=by, us=stats([1e3 * t for t in ts], 1),
                        achieved_gbs=round(gbs, 1), frac_of_design_hbm=round(gbs / DESIGN_HBM_GBS, 3)))
    return out


def step_leg(make, batches, steps, repeats, graphs_expected):
    """Two identically seeded (model, store, trainer) arms, EMA off / on, alternated per repeat; ms per step."""
    arms = {}
    for on in (False, True):
        model, store, tr_kw = make()
        arms[on] = (store, Trainer(model, ema_decay=DECAY if on else 0.0, **tr_kw))
    B = batches
    for on, (store, tr) in arms.items():
        idx = store.shard(0, 1)
        for i in range(4):                                   # warm-up: eager steps, capture, first replays
            tr.train_step(store, idx[(i % 4) * B:(i % 4 + 1) * B])
    torch.cuda.synchronize()
    times = {False: [], True: []}
    losses = {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(repeats):
        for on, (store, tr) in arms.items():
            idx = store.shard(0, 1)
            torch.cuda.synchronize()
            e0.record()
            for i in range(steps):
                res = tr.train_step(store, idx[(i % 4) * B:(i % 4 + 1) * B])
            e1.record()
            torch.cuda.synchronize()
            times[on].append(e0.elapsed_time(e1) / steps)
            losses[on] = res[0].item()
    replayed = {on: any(g[1] is not None for g in tr._graphs.values()) for on, (_, tr) in arms.items()}
    assert all(v == graphs_expected for v in replayed.values()), replayed
    off, on = statistics.median(times[False]), statistics.median(times[True])
    return dict(ema_off_ms=stats(times[False]), ema_on_ms=stats(times[True]), delta_us=round(1e3 * (on - off), 1),
                delta_frac=round((on - off) / off, 4), graph_replayed=graphs_expected,
                last_loss={"ema_off": losses[False], "ema_on": losses[True]})


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10, help="denoiser steps per timed window (the FeedForward leg runs 20x as many)")
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ema_bench needs a CUDA device")
    if args.repeats < 3:
        ap.error("--repeats must be at least 3")
    dev = torch.device("cuda", 0)

    def denoiser():
        torch.manual_seed(0)
        m = DiffusionDenoiser(frames=50, d_model=512, num_heads=8, dim_feedforward=2048, num_layers=8).to(dev)
        store = WindowStore.synthetic(4096 * 4, 50, 1, 177, "all_frames", seed=1234, device=dev)
        return m, store, dict(opt_type="rmsprop", lr=1e-4, diffusion=GaussianDiffusion(device=dev), seed=1234)

    def feedforward():
        torch.manual_seed(0)
        m = FeedForwardBaseline(23, 2, 50, "all_frames", "sigmoid", 5, 10, hidden_dims=[512, 512]).to(dev)
        store = WindowStore.synthetic(4096, 50, 5, 147, "all_frames", seed=3, device=dev)
        return m, store, dict(opt_type="rmsprop", lr=1e-4, seed=1234)

    n = denoiser()[0].arena.total
    torch.cuda.empty_cache()
    kern = kernel_leg(n, dev, args.repeats)
    den = step_leg(denoiser, 4096, args.steps, args.repeats, graphs_expected=False)
    torch.cuda.empty_cache()
    ff = step_leg(feedforward, 32, 20 * args.steps, args.repeats, graphs_expected=True)
    line = json.dumps(dict(bench="ema", ema_decay=DECAY, **device_info(), repeats=args.repeats,
                           design_hbm_gbs=DESIGN_HBM_GBS, optimizer_kernel=kern,
                           denoiser_step=dict(model="configs[1] denoiser d=512 h=8 ff=2048 L=8 F=50, B=4096, rmsprop 1e-4",
                                              steps_per_window=args.steps, **den),
                           feedforward_step=dict(model="configs[0] FeedForward T=50 stride 5 hidden 512-512 sigmoid, B=32, rmsprop 1e-4",
                                                 steps_per_window=20 * args.steps, **ff)))
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
