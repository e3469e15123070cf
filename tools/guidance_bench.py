"""Cost of classifier-free guidance (``Trainer(cond_drop_prob=...)``, ``GaussianDiffusion.sample(guidance_scale=...)``) on
the BASELINE configs[1] / configs[3] denoiser (d=512, 8 heads, FFN 2048, 8 layers, F=50):

* the condition-dropout kernel (``ibm_cond_dropout``) alone at the training shape: 4096 windows x 50 rows of the 208-column
  concat buffer, p = 0.1, timed over a captured graph of 50 launches (``trainer._time_kernel``).  The buffer (85 MB) fits
  the 126 MB L2, so this is an in-step figure, not an HBM one.  Bytes: the dropped windows' condition columns;
* the configs[1] training step (B = 4096, RMSprop lr 1e-4 as bench.py) with ``cond_drop_prob`` 0 and 0.1: two identically
  seeded models, one Trainer each, the two arms alternated within each repeat (CUDA events around ``--steps`` steps);
* one DDIM-50 sampling step (eta = 0) without guidance and with guidance scale 2.5, at 512 and 4096 windows: a 50-step
  call (graph-replayed after a warm-up call) timed with the host clock up to a device synchronise, divided by 50; the
  cases are interleaved per repeat.  Beside it the guided and unguided step kernels alone (``_time_kernel``, Philox noise)
  with their bytes computed from the shapes, against the 7 700 GB/s data-sheet HBM bandwidth and the 6 536.7 GB/s copy
  figure DESIGN.md quotes.

Reports medians over ``--repeats`` with min / max, the device name and power limit read in the same run.  Prints one JSON
line (and writes it to --out if given).

    python tools/guidance_bench.py [--repeats 5] [--steps 10] [--out profiles/r06_guidance.json]
"""
import argparse
import json
import os
import statistics
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch

from ema_bench import DESIGN_HBM_GBS, device_info, stats
from inferbiomechanics_b200 import ops
from inferbiomechanics_b200.data.window_store import WindowStore
from inferbiomechanics_b200.diffusion import GaussianDiffusion
from inferbiomechanics_b200.models.DiffusionDenoiser import DiffusionDenoiser
from inferbiomechanics_b200.trainer import Trainer, _time_kernel

DATASHEET_HBM_GBS = 7700.0
P_DROP, SCALE, S = 0.1, 2.5, 50
F, C_IN, LD = 50, 177, 208


def dropout_leg(dev, repeats):
    B = 4096
    xc = torch.randn(B * F, LD, device=dev).to(torch.bfloat16)
    keep = torch.empty(B, dtype=torch.uint8, device=dev)
    times = [_time_kernel(lambda: ops.cond_dropout(xc, B, F, 30, C_IN, P_DROP, 1234, 7), iters=50) for _ in range(repeats)]
    ops.cond_dropout(xc, B, F, 30, C_IN, P_DROP, 1234, 7, keep_out=keep)
    dropped = int((keep == 0).sum().item())
    by = dropped * F * C_IN * 2.0
    us = statistics.median(times) * 1e3
    return dict(windows=B, rows_per_window=F, ld=LD, p=P_DROP, dropped_windows=dropped, bytes_written=by, us=stats([1e3 * t for t in times], 2),
                achieved_gbs=round(by / (us * 1e-6) / 1e9, 1))


def step_leg(dev, steps, repeats):
    arms = {}
    for p in (0.0, P_DROP):
        torch.manual_seed(0)
        m = DiffusionDenoiser(frames=F, d_model=512, num_heads=8, dim_feedforward=2048, num_layers=8).to(dev)
        store = WindowStore.synthetic(4096 * 4, F, 1, C_IN, "all_frames", seed=1234, device=dev)
        arms[p] = (store, Trainer(m, opt_type="rmsprop", lr=1e-4, diffusion=GaussianDiffusion(device=dev), seed=1234, cond_drop_prob=p))
    B = 4096
    for store, tr in arms.values():
        idx = store.shard(0, 1)
        for i in range(3):
            tr.train_step(store, idx[(i % 4) * B:(i % 4 + 1) * B])
    torch.cuda.synchronize()
    times = {p: [] for p in arms}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(repeats):
        for p, (store, tr) in arms.items():
            idx = store.shard(0, 1)
            torch.cuda.synchronize()
            e0.record()
            for i in range(steps):
                tr.train_step(store, idx[(i % 4) * B:(i % 4 + 1) * B])
            e1.record()
            torch.cuda.synchronize()
            times[p].append(e0.elapsed_time(e1) / steps)
    off, on = statistics.median(times[0.0]), statistics.median(times[P_DROP])
    return dict(windows=B, steps_per_window=steps, p0_ms=stats(times[0.0]), p01_ms=stats(times[P_DROP]),
                delta_us=round(1e3 * (on - off), 1), delta_frac=round((on - off) / off, 4))


def step_kernel_leg(dev, B, repeats):
    """The guided and unguided DDIM step kernels alone at M = 50 B rows, Philox noise, fp32 state + bf16 rows written."""
    M = B * F
    gd = GaussianDiffusion(device=dev)
    tab = gd.ddim_tables(S, 0.0)
    t_dev = torch.tensor([int(tab["ts"][10])], dtype=torch.int32, device=dev)
    x0h = torch.randn(2 * M, 32, device=dev)
    x = torch.randn(M, 30, device=dev)
    xb = torch.zeros(2 * M, LD, dtype=torch.bfloat16, device=dev)
    args = (t_dev, tab["coef_x0"], tab["coef_xt"], tab["sigma"], M)
    kw = dict(x_prev=x, bf16_ld=LD, t_succ=tab["succ"], seed=3)
    unguided = [_time_kernel(lambda: ops.posterior_step(x0h, 32, x, None, *args, xprev_bf16=xb, **kw), iters=50) for _ in range(repeats)]
    guided = [_time_kernel(lambda: ops.guided_step(x0h, 32, x, None, *args, SCALE, xprev_bf16=xb, **kw), iters=50) for _ in range(repeats)]
    # algorithmic bytes per row: x0_hat 30 fp32 per half read, x_t read and x_prev written (30 fp32 each), 30 bf16 per half written
    by = {"unguided": M * (120 + 120 + 120 + 60.0), "guided": M * (240 + 120 + 120 + 120.0)}
    out = {}
    for name, ts in (("unguided", unguided), ("guided", guided)):
        us = statistics.median(ts) * 1e3
        gbs = by[name] / (us * 1e-6) / 1e9
        out[name] = dict(bytes=by[name], us=stats([1e3 * t for t in ts], 2), achieved_gbs=round(gbs, 1),
                         frac_of_datasheet_hbm=round(gbs / DATASHEET_HBM_GBS, 3), frac_of_design_hbm=round(gbs / DESIGN_HBM_GBS, 3))
    return out


def sampling_leg(dev, repeats):
    torch.manual_seed(0)
    model = DiffusionDenoiser(frames=F, d_model=512, num_heads=8, dim_feedforward=2048, num_layers=8).to(dev)
    model.eval()
    eng = model.engine()
    gd = GaussianDiffusion(device=dev)
    cases = [(B, s) for B in (512, 4096) for s in (1.0, SCALE)]
    for B in (512, 4096):
        eng.xc(B, False)[:, 30:30 + C_IN] = torch.randn(B * F, C_IN, device=dev).to(torch.bfloat16)

    def run(B, s):
        return gd.sample(model, B, seed=1, ddim_steps=S, guidance_scale=s)

    for c in cases:                                         # warm-up: captures each case's graph
        assert torch.isfinite(run(*c)).all()
    times = {c: [] for c in cases}
    for _ in range(repeats):
        for c in cases:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run(*c)
            torch.cuda.synchronize()
            times[c].append((time.perf_counter() - t0) * 1e3 / S)
    out = {}
    for B in (512, 4096):
        plain, guided = statistics.median(times[(B, 1.0)]), statistics.median(times[(B, SCALE)])
        out[str(B)] = dict(unguided_step_ms=stats(times[(B, 1.0)]), guided_step_ms=stats(times[(B, SCALE)]),
                           ratio=round(guided / plain, 3), step_kernels=step_kernel_leg(dev, B, repeats))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10, help="training steps per timed window")
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("guidance_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    info = device_info()
    drop = dropout_leg(dev, args.repeats)
    torch.cuda.empty_cache()
    step = step_leg(dev, args.steps, args.repeats)
    torch.cuda.empty_cache()
    samp = sampling_leg(dev, args.repeats)
    line = json.dumps(dict(bench="guidance", **info, repeats=args.repeats, datasheet_hbm_gbs=DATASHEET_HBM_GBS,
                           design_hbm_gbs=DESIGN_HBM_GBS, cond_dropout_kernel=drop,
                           training_step=dict(model="configs[1] denoiser d=512 h=8 ff=2048 L=8 F=50, B=4096, rmsprop 1e-4", **step),
                           ddim50_sampling=dict(eta=0.0, guidance_scale=SCALE, per_windows=samp)))
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
