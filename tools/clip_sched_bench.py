"""Cost of global-norm gradient clipping and the learning-rate schedule (``Trainer(clip_grad_norm=..., lr_warmup_steps=...,
lr_schedule=...)``), options off against on:

* the norm kernel (``ibm_grad_clip_coef``) alone on gradient arenas the size of the BASELINE configs[1] denoiser's (d=512,
  8 heads, FFN 2048, 8 layers: 25.9 M parameters, 104 MB), timed over a captured graph of 48 launches
  (``trainer._time_kernel``).  One arena would fit the 126 MB L2 and be read from there after the first launch, so the
  launches rotate over three arenas (311 MB): each launch reads an arena two launches older than the lines L2 still holds.
  Bytes: one 4 B read per parameter, set against the 6 536.7 GB/s HBM copy figure DESIGN.md quotes;
* the scheduled optimizer kernel (clip coefficient + cosine schedule read on the device) against the current one, RMSprop
  and Adam, EMA off and on, on the same arena, each launch fed by the device step counter as the Trainer does;
* the configs[1] denoiser training step (B = 4096 windows, F = 50, RMSprop lr 1e-4 as bench.py) with
  ``--clip-grad-norm 1 --lr-warmup-steps 1000 --lr-schedule cosine`` against the defaults, two identically seeded models,
  one Trainer each, the two arms alternated within each repeat (CUDA events around ``--steps`` steps);
* the configs[0] FeedForward step (T = 50, stride 5, hidden 512-512, sigmoid, B = 32), graph-replayed, the same flags
  against the defaults, alternated the same way.

Reports medians over ``--repeats`` with min / max, the device name and power limit.  Prints one JSON line (and writes it
to --out if given).

    python tools/clip_sched_bench.py [--repeats 7] [--steps 10] [--out profiles/r05_clip_sched.json]
"""
import argparse
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch

from ema_bench import DESIGN_HBM_GBS, device_info, stats
from inferbiomechanics_b200 import ops
from inferbiomechanics_b200.data.window_store import WindowStore
from inferbiomechanics_b200.diffusion import GaussianDiffusion
from inferbiomechanics_b200.models.DiffusionDenoiser import DiffusionDenoiser
from inferbiomechanics_b200.models.FeedForwardRegressionBaseline import FeedForwardBaseline
from inferbiomechanics_b200.trainer import Trainer, _time_kernel

FLAGS = dict(clip_grad_norm=1.0, lr_warmup_steps=1000, lr_schedule="cosine", total_steps=100_000)
SCHED = dict(schedule="cosine", warmup_steps=1000, total_steps=100_000, lr_min=0.0)


def norm_leg(n, dev, repeats, arenas=3):
    gen = torch.Generator(device=dev).manual_seed(0)
    grads = [torch.randn(n, device=dev, generator=gen) * 1e-3 for _ in range(arenas)]
    ws = ops.GradClipWorkspace(dev)
    turn = [0]

    def launch():
        ops.grad_clip_coef(grads[turn[0] % arenas], 1.0, 1.0, ws)
        turn[0] += 1

    times = [_time_kernel(launch, iters=16 * arenas) for _ in range(repeats)]
    ms = statistics.median(times)
    gbs = 4.0 * n / (ms * 1e-3) / 1e9
    return dict(params=n, bytes_per_launch=4 * n, arenas_rotated=arenas, rotated_bytes=4 * n * arenas,
                us=stats([1e3 * t for t in times], 1), achieved_gbs=round(gbs, 1), frac_of_design_hbm=round(gbs / DESIGN_HBM_GBS, 3))


def optimizer_leg(n, dev, repeats):
    g = torch.Generator(device=dev).manual_seed(0)
    p = torch.randn(n, device=dev, generator=g)
    grad = torch.randn(n, device=dev, generator=g) * 1e-3
    s0, s1, ema = torch.zeros(n, device=dev), torch.zeros(n, device=dev), p.clone()
    pb = torch.empty(n, dtype=torch.bfloat16, device=dev)
    counter = torch.full((1,), 1500, dtype=torch.int64, device=dev)
    clip = torch.tensor([2.0, 0.5], device=dev)
    per_param = {"rmsprop": 22.0, "adam": 30.0}
    cases = [(k, e, s) for k in ("rmsprop", "adam") for e in (False, True) for s in (False, True)]
    times = {c: [] for c in cases}
    for _ in range(repeats):
        for kind, on, sched in cases:
            kw = dict(step_dev=counter, ema=ema if on else None, ema_decay=0.999 if on else 0.0)
            if sched:
                kw.update(clip=clip, **SCHED)
            times[(kind, on, sched)].append(_time_kernel(lambda k=kind, kw=kw: ops.optimizer_step(k, p, grad, s0, s1, pb, 1e-4, 1.0, 1,
                                                                                                    **kw), iters=50))
    out = []
    for (kind, on, sched), ts in times.items():
        by = n * (per_param[kind] + (8.0 if on else 0.0))
        ms = statistics.median(ts)
        gbs = by / (ms * 1e-3) / 1e9
        out.append(dict(optimizer=kind, ema=on, scheduled=sched, params=n, bytes_per_launch=by, us=stats([1e3 * t for t in ts], 1),
                        achieved_gbs=round(gbs, 1), frac_of_design_hbm=round(gbs / DESIGN_HBM_GBS, 3)))
    return out


def step_leg(make, B, steps, repeats, graphs_expected):
    """Two identically seeded (model, store, trainer) arms, defaults / clip + schedule, alternated per repeat; ms per step."""
    arms = {}
    for on in (False, True):
        model, store, tr_kw = make()
        arms[on] = (store, Trainer(model, **tr_kw, **(FLAGS if on else {})))
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
    replayed = {on: sum(g[1] is not None for g in tr._graphs.values()) for on, (_, tr) in arms.items()}
    assert all(v == (1 if graphs_expected else 0) for v in replayed.values()), replayed
    norms = arms[True][1].grad_norm_stats()
    off, on = statistics.median(times[False]), statistics.median(times[True])
    return dict(off_ms=stats(times[False]), clip_sched_ms=stats(times[True]), delta_us=round(1e3 * (on - off), 1),
                delta_frac=round((on - off) / off, 4), graph_replayed=graphs_expected, captures_per_arm=replayed[True],
                lr_at_end=arms[True][1].current_lr(), mean_preclip_norm=norms["mean_norm"],
                clipped_steps=norms["clipped"], steps_recorded=norms["steps"],
                last_loss={"off": losses[False], "clip_sched": losses[True]})


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--steps", type=int, default=10, help="denoiser steps per timed window (the FeedForward leg runs 20x as many)")
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("clip_sched_bench needs a CUDA device")
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
    norm = norm_leg(n, dev, args.repeats)
    opt = optimizer_leg(n, dev, args.repeats)
    torch.cuda.empty_cache()
    den = step_leg(denoiser, 4096, args.steps, args.repeats, graphs_expected=False)
    torch.cuda.empty_cache()
    ff = step_leg(feedforward, 32, 20 * args.steps, args.repeats, graphs_expected=True)
    line = json.dumps(dict(bench="clip_sched", flags=FLAGS, **device_info(), repeats=args.repeats, design_hbm_gbs=DESIGN_HBM_GBS,
                           norm_kernel=norm, optimizer_kernel=opt,
                           denoiser_step=dict(model="configs[1] denoiser d=512 h=8 ff=2048 L=8 F=50, B=4096, rmsprop 1e-4",
                                              steps_per_window=args.steps, **den),
                           feedforward_step=dict(model="configs[0] FeedForward T=50 stride 5 hidden 512-512 sigmoid, B=32, rmsprop 1e-4",
                                                 steps_per_window=20 * args.steps, **ff)))
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
