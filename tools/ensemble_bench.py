"""Cost of ensemble sampling and scoring (``GaussianDiffusion.sample(num_samples=K)``, ``ops.ensemble_score``) on the BASELINE
configs[3] denoiser (d=512, 8 heads, FFN 2048, 8 layers, F=50):

* the scoring kernel (``ibm_ensemble_score``) alone at K = 4, 16, 64 on an analyze-sized launch of 4096 sampled windows
  (4096 / K windows x K draws, F = 50, all frames), timed over a captured graph of 20 launches (``trainer._time_kernel``).
  The draws (24.6 MB) stay in the 126 MB L2 across the replays, as they are right after the sampler writes them; one more
  case at K = 16 with 32768 sampled windows (197 MB of draws) is larger than the L2.  Bytes from the shapes: the draws and the
  labels read, the mean written;
* DDIM-50 sampling (eta = 0) of 4096 sampled windows as 4096 x 1, 1024 x 4 and 256 x 16 windows x draws: one call
  (graph-replayed after a warm-up call) timed with the host clock up to a device synchronise, the cases interleaved per repeat.

Reports medians over ``--repeats`` with min / max, against the 7 700 GB/s data-sheet HBM bandwidth and the 6 536.7 GB/s copy
figure DESIGN.md quotes, with the device name and power limit read in the same run.  Prints one JSON line (and writes it to
--out if given).

    python tools/ensemble_bench.py [--repeats 5] [--out profiles/r07_ensemble.json]
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
from inferbiomechanics_b200.diffusion import GaussianDiffusion
from inferbiomechanics_b200.models.DiffusionDenoiser import DiffusionDenoiser
from inferbiomechanics_b200.trainer import _time_kernel

DATASHEET_HBM_GBS = 7700.0
L2_BYTES = 126e6
F, C_IN, S = 50, 177, 50


def kernel_case(dev, K, sampled, repeats):
    B = sampled // K
    g = torch.Generator(device=dev).manual_seed(K)
    draws = torch.randn(K, B, F, 30, device=dev, generator=g)
    labels = torch.randn(B, F, 30, device=dev, generator=g) * 20
    acc = torch.zeros(5, 30, dtype=torch.float64, device=dev)
    mean = torch.empty_like(labels)
    ws = ops.EnsembleWorkspace(dev)
    times = [_time_kernel(lambda: ops.ensemble_score(draws, labels, acc, mean, ws), iters=20) for _ in range(repeats)]
    draw_bytes = draws.numel() * 4.0
    by = draw_bytes + 2 * labels.numel() * 4.0
    us = statistics.median(times) * 1e3
    gbs = by / (us * 1e-6) / 1e9
    return dict(K=K, windows=B, sampled_windows=K * B, frames=F, draw_bytes=draw_bytes, bytes=by,
                draws_l2_resident=draw_bytes + 2 * labels.numel() * 4.0 < L2_BYTES, us=stats([1e3 * t for t in times], 2),
                achieved_gbs=round(gbs, 1), frac_of_datasheet_hbm=round(gbs / DATASHEET_HBM_GBS, 3),
                frac_of_design_hbm=round(gbs / DESIGN_HBM_GBS, 3))


def sampling_leg(dev, repeats):
    torch.manual_seed(0)
    model = DiffusionDenoiser(frames=F, d_model=512, num_heads=8, dim_feedforward=2048, num_layers=8).to(dev)
    model.eval()
    eng = model.engine()
    gd = GaussianDiffusion(device=dev)
    cases = [(4096, None), (1024, 4), (256, 16)]
    for B, _ in cases:
        eng.xc(B, False)[:, 30:30 + C_IN] = torch.randn(B * F, C_IN, device=dev).to(torch.bfloat16)

    def run(B, K):
        return gd.sample(model, B, seed=1, ddim_steps=S, num_samples=K)

    for c in cases:                                         # warm-up: captures each case's graph (all at 4096 windows)
        assert torch.isfinite(run(*c)).all()
    times = {c: [] for c in cases}
    for _ in range(repeats):
        for c in cases:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run(*c)
            torch.cuda.synchronize()
            times[c].append((time.perf_counter() - t0) * 1e3)
    return {f"{B}x{K or 1}": dict(windows=B, draws=K or 1, call_ms=stats(times[(B, K)], 2)) for B, K in cases}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ensemble_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    info = device_info()
    kern = [kernel_case(dev, K, 4096, args.repeats) for K in (4, 16, 64)]
    kern.append(kernel_case(dev, 16, 32768, args.repeats))
    torch.cuda.empty_cache()
    samp = sampling_leg(dev, args.repeats)
    line = json.dumps(dict(bench="ensemble", **info, repeats=args.repeats, datasheet_hbm_gbs=DATASHEET_HBM_GBS,
                           design_hbm_gbs=DESIGN_HBM_GBS, score_kernel=kern,
                           ddim50_sampling=dict(model="configs[3] denoiser d=512 h=8 ff=2048 L=8 F=50", eta=0.0,
                                                sampled_windows=4096, per_case=samp)))
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
