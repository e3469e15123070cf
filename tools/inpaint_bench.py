"""Cost of inpainting (``GaussianDiffusion.sample(known=..., known_mask=...)``) on the BASELINE configs[3] denoiser (d=512,
8 heads, FFN 2048, 8 layers, F=50):

* the DDIM step kernel alone at 512 and 4096 windows (M = 50 B rows, Philox noise, fp32 state and bf16 rows written), today's
  ``ibm_ddpm_respaced_step`` against ``ibm_ddpm_inpaint_step`` with the force channels known (the ``analyze
  --given-quantities force`` mask) and with every channel known (the most the kernel reads), timed over a captured graph of
  50 launches (``trainer._time_kernel``).  Bytes are computed from the shapes: 420 B per row today (x0_hat and x_t read,
  x_prev written in fp32, the bf16 row written) plus 4 B for the row's mask word and 8 B per channel pair with a known bit,
  at most 124 B more.  They are set against the 7 700 GB/s data-sheet HBM bandwidth and the 6 536.7 GB/s copy figure
  DESIGN.md quotes.  The buffers of 512 windows fit the 126 MB L2; those of 4096 windows (about 160 MB with the 208-column
  bf16 buffer) do not;
* one DDIM-50 sampling step (eta = 0) without and with the force mask, at 512 and 4096 windows: a 50-step call (graph-replayed
  after a warm-up call) timed with the host clock up to a device synchronise, divided by 50; the two cases alternate per
  repeat.

Reports medians over ``--repeats`` with min / max, the device name and power limit read in the same run.  Prints one JSON
line (and writes it to --out if given).

    python tools/inpaint_bench.py [--repeats 7] [--out profiles/r08_inpaint.json]
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
from inferbiomechanics_b200.cli.train import known_quantity_mask
from inferbiomechanics_b200.diffusion import GaussianDiffusion, known_mask_words
from inferbiomechanics_b200.models.DiffusionDenoiser import DiffusionDenoiser
from inferbiomechanics_b200.trainer import _time_kernel

DATASHEET_HBM_GBS = 7700.0
S, F, C_IN, LD = 50, 50, 177, 208
WINDOWS = (512, 4096)
MASKS = {"force": known_quantity_mask(("force",)), "all": torch.ones(30, dtype=torch.bool)}


def step_kernel_leg(dev, B, repeats):
    M = B * F
    gd = GaussianDiffusion(device=dev)
    tab = gd.ddim_tables(S, 0.0)
    t_dev = torch.tensor([int(tab["ts"][10])], dtype=torch.int32, device=dev)
    x0h = torch.randn(M, 32, device=dev)
    x = torch.randn(M, 30, device=dev)
    y = torch.randn(M, 30, device=dev)
    xb = torch.zeros(M, LD, dtype=torch.bfloat16, device=dev)
    args = (x0h, 32, x, None, t_dev, tab["coef_x0"], tab["coef_xt"], tab["sigma"], M)
    kw = dict(x_prev=x, xprev_bf16=xb, bf16_ld=LD, t_succ=tab["succ"], seed=3)
    cases = {"today": ({}, 420.0)}
    for name, mask in MASKS.items():
        words = known_mask_words(mask.to(dev), M).contiguous()
        pairs = int(mask.view(15, 2).any(dim=1).sum())
        cases[name] = (dict(known=y, known_mask=words), 420.0 + 4 + 8 * pairs)
    times = {name: [] for name in cases}
    for _ in range(repeats):                                 # the cases alternate within each repeat
        for name, (kn, _) in cases.items():
            times[name].append(_time_kernel(lambda: ops.posterior_step(*args, **kw, **kn), iters=50))
    out = {}
    for name, (_, per_row) in cases.items():
        us = statistics.median(times[name]) * 1e3
        by = M * per_row
        gbs = by / (us * 1e-6) / 1e9
        out[name] = dict(bytes_per_row=per_row, bytes=by, us=stats([1e3 * t for t in times[name]], 2), achieved_gbs=round(gbs, 1),
                         frac_of_datasheet_hbm=round(gbs / DATASHEET_HBM_GBS, 3), frac_of_design_hbm=round(gbs / DESIGN_HBM_GBS, 3))
    return out


def sampling_leg(dev, repeats):
    torch.manual_seed(0)
    model = DiffusionDenoiser(frames=F, d_model=512, num_heads=8, dim_feedforward=2048, num_layers=8).to(dev)
    model.eval()
    eng = model.engine()
    gd = GaussianDiffusion(device=dev)
    known = {}
    for B in WINDOWS:
        eng.xc(B, False)[:, 30:30 + C_IN] = torch.randn(B * F, C_IN, device=dev).to(torch.bfloat16)
        known[B] = torch.randn(B, F, 30, device=dev)
    force = MASKS["force"].to(dev)

    def run(B, inpaint):
        kn = dict(known=known[B], known_mask=force) if inpaint else {}
        return gd.sample(model, B, seed=1, ddim_steps=S, **kn)

    cases = [(B, inpaint) for B in WINDOWS for inpaint in (False, True)]
    for c in cases:                                         # warm-up: captures each case's graph
        x = run(*c)
        assert torch.isfinite(x).all()
        if c[1]:
            assert torch.equal(x[..., 6:12], known[c[0]][..., 6:12])
    times = {c: [] for c in cases}
    for _ in range(repeats):
        for c in cases:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run(*c)
            torch.cuda.synchronize()
            times[c].append((time.perf_counter() - t0) * 1e3 / S)
    out = {}
    for B in WINDOWS:
        plain, inp = statistics.median(times[(B, False)]), statistics.median(times[(B, True)])
        out[str(B)] = dict(plain_step_ms=stats(times[(B, False)]), force_known_step_ms=stats(times[(B, True)]),
                           ratio=round(inp / plain, 4))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("inpaint_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    info = device_info()
    kern = {str(B): step_kernel_leg(dev, B, args.repeats) for B in WINDOWS}
    torch.cuda.empty_cache()
    samp = sampling_leg(dev, args.repeats)
    line = json.dumps(dict(bench="inpaint", **info, repeats=args.repeats, datasheet_hbm_gbs=DATASHEET_HBM_GBS,
                           design_hbm_gbs=DESIGN_HBM_GBS,
                           step_kernel=dict(sampler=f"DDIM-{S} eta 0, Philox noise, rows of F={F}", per_windows=kern),
                           ddim50_sampling=dict(model="configs[3] denoiser d=512 h=8 ff=2048 L=8 F=50", eta=0.0,
                                                known="force channels 6-11 of every row", per_windows=samp)))
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
