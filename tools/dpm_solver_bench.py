"""Cost of DPM-Solver++(2M) sampling (``GaussianDiffusion.sample(dpm_steps=S)``) against DDIM at eta = 0 with the same step
count, on the BASELINE configs[3] denoiser (d=512, 8 heads, FFN 2048, 8 layers, F=50):

* whole sampling calls, DDIM-S and DPM-S for S in {10, 20, 50} at 512 and 4096 windows: one warm-up call per case (it
  captures the case's graph), then ``--repeats`` rounds in which every case runs once, in turn (DDIM-S right before DPM-S);
  each call is timed with the host clock up to a device synchronise and reported as windows/s;
* the step kernel alone at M = 25 600 and 204 800 rows (512 and 4096 windows): ``ibm_ddpm_respaced_step`` (DDIM) against
  ``ibm_ddpm_multistep_step`` on an interior step, timed with CUDA events over a captured graph of 50 launches
  (``trainer._time_kernel``), the two alternating per repeat.  Bytes are computed from the shapes: 420 B per row for DDIM
  (x0_hat and x_t read, x_prev written in fp32, the bf16 row written) and 660 B for the multistep step (plus the fp32
  previous prediction read and written), set against the 6 536.7 GB/s copy figure DESIGN.md quotes.

It also checks that DPM-2 equals DDIM-2 bit for bit on the model.  Reports medians with min / max, the device name and power
limit read in the same run, and prints one JSON line (also written to --out if given).

    python tools/dpm_solver_bench.py [--repeats 5] [--out profiles/r09_dpm_solver.json]
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

F, C_IN, LD = 50, 177, 208
WINDOWS = (512, 4096)
STEPS = (10, 20, 50)
BYTES_PER_ROW = {"ddim": 420.0, "dpm": 660.0}


def step_kernel_leg(dev, B, repeats):
    M = B * F
    gd = GaussianDiffusion(device=dev)
    ddim, dpm = gd.ddim_tables(20, 0.0), gd.dpm_tables(20)
    x0h = torch.randn(M, 32, device=dev)
    x = torch.randn(M, 30, device=dev)
    prev = torch.randn(M, 30, device=dev)
    xb = torch.zeros(M, LD, dtype=torch.bfloat16, device=dev)
    t_ddim = torch.tensor([int(ddim["ts"][10])], dtype=torch.int32, device=dev)
    t_dpm = torch.tensor([int(dpm["ts"][10])], dtype=torch.int32, device=dev)
    assert float(dpm["coef_prev"][int(dpm["ts"][10])]) != 0.0
    t_next = torch.zeros(1, dtype=torch.int32, device=dev)
    run = {"ddim": lambda: ops.posterior_step(x0h, 32, x, None, t_ddim, ddim["coef_x0"], ddim["coef_xt"], ddim["sigma"], M,
                                              x_prev=x, xprev_bf16=xb, bf16_ld=LD, seed=3, t_next=t_next, t_succ=ddim["succ"]),
           "dpm": lambda: ops.multistep_step(x0h, 32, x, t_dpm, dpm["coef_x0"], dpm["coef_xt"], dpm["coef_prev"], dpm["succ"], M,
                                             prev, x_prev=x, xprev_bf16=xb, bf16_ld=LD, t_next=t_next)}
    times = {k: [] for k in run}
    for _ in range(repeats):
        for k, fn in run.items():
            times[k].append(_time_kernel(fn, iters=50))
    out = dict(rows=M)
    for k in run:
        us = statistics.median(times[k]) * 1e3
        by = M * BYTES_PER_ROW[k]
        gbs = by / (us * 1e-6) / 1e9
        out[k] = dict(bytes_per_row=BYTES_PER_ROW[k], us=stats([1e3 * t for t in times[k]], 2), achieved_gbs=round(gbs, 1),
                      frac_of_design_hbm=round(gbs / DESIGN_HBM_GBS, 3))
    return out


def sampling_leg(dev, repeats):
    torch.manual_seed(0)
    model = DiffusionDenoiser(frames=F, d_model=512, num_heads=8, dim_feedforward=2048, num_layers=8).to(dev)
    model.eval()
    eng = model.engine()
    gd = GaussianDiffusion(device=dev)
    for B in WINDOWS:
        eng.xc(B, False)[:, 30:30 + C_IN] = torch.randn(B * F, C_IN, device=dev).to(torch.bfloat16)
    # DPM-2 is DDIM-2 at eta = 0, bit for bit
    a = gd.sample(model, WINDOWS[0], seed=1, dpm_steps=2)
    b = gd.sample(model, WINDOWS[0], seed=1, ddim_steps=2)
    assert torch.isfinite(a).all() and torch.equal(a, b), "DPM-2 != DDIM-2"

    def run(B, kind, S):
        kw = dict(dpm_steps=S) if kind == "dpm" else dict(ddim_steps=S)
        return gd.sample(model, B, seed=1, **kw)

    cases = [(B, kind, S) for B in WINDOWS for S in STEPS for kind in ("ddim", "dpm")]
    for c in cases:                                         # warm-up: captures each case's graph
        assert torch.isfinite(run(*c)).all(), c
    times = {c: [] for c in cases}
    for _ in range(repeats):
        for c in cases:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run(*c)
            torch.cuda.synchronize()
            times[c].append(time.perf_counter() - t0)
    out = {}
    for B in WINDOWS:
        row = {}
        for S in STEPS:
            w = {kind: [B / t for t in times[(B, kind, S)]] for kind in ("ddim", "dpm")}
            row[str(S)] = dict(ddim_windows_per_s=stats(w["ddim"], 1), dpm_windows_per_s=stats(w["dpm"], 1),
                               dpm_over_ddim=round(statistics.median(w["dpm"]) / statistics.median(w["ddim"]), 4))
        out[str(B)] = row
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dpm_solver_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    info = device_info()
    kern = {str(B): step_kernel_leg(dev, B, args.repeats) for B in WINDOWS}
    torch.cuda.empty_cache()
    samp = sampling_leg(dev, args.repeats)
    line = json.dumps(dict(bench="dpm_solver", **info, repeats=args.repeats, design_hbm_gbs=DESIGN_HBM_GBS,
                           dpm2_equals_ddim2=True,
                           step_kernel=dict(steps="interior step 10 of S=20, rows of F=50, bf16 ld 208", per_windows=kern),
                           sampling=dict(model="configs[3] denoiser d=512 h=8 ff=2048 L=8 F=50", ddim_eta=0.0,
                                         per_windows=samp)))
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
