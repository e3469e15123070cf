"""Sampling throughput of the BASELINE configs[3] denoiser (d=512, 8 heads, FFN 2048, 8 layers, F=50) by sampler and step
count: the 1000-step DDPM chain against DDIM with S in {250, 50, 20}, at 512 and 4096 windows per GPU.

Each (windows, sampler) case is warmed up once (that call captures its CUDA graph), then timed with the host clock around
a call that ends in a device synchronise; the repeats are interleaved over all cases so drift on a shared host spreads
over every case alike.  In the same process it asserts that DDIM with S = T and eta = 1 reproduces the DDPM chain bit
for bit at the 512-window shape, and reads the device name and power limit the numbers were measured at.  Prints one
JSON line (and writes it to --out if given).

    python tools/sampling_steps_bench.py [--repeats 3] [--out result.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from inferbiomechanics_b200.diffusion import GaussianDiffusion
from inferbiomechanics_b200.models.DiffusionDenoiser import DiffusionDenoiser

WINDOWS = (512, 4096)
SAMPLERS = (("ddpm", 1000), ("ddim", 250), ("ddim", 50), ("ddim", 20))


def device_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return dict(device=name, power_limit=power, torch_device=torch.cuda.get_device_name(0))


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sampling_steps_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    model = DiffusionDenoiser(frames=50, d_model=512, num_heads=8, dim_feedforward=2048, num_layers=8).to(dev)
    model.eval()
    eng = model.engine()
    gd = GaussianDiffusion(device=dev)
    for B in WINDOWS:
        eng.xc(B, False)[:, 30:30 + eng.c_in] = torch.randn(B * eng.F, eng.c_in, device=dev).to(torch.bfloat16)

    def run(B, sampler, S):
        kw = dict(ddim_steps=S) if sampler == "ddim" else {}
        return gd.sample(model, B, seed=1, **kw)

    # DDIM over the full sequence at eta = 1 is the DDPM chain: same tables, same Philox draws
    ddpm = gd.sample(model, WINDOWS[0], seed=7)
    ddim = gd.sample(model, WINDOWS[0], seed=7, ddim_steps=gd.T, eta=1.0)
    assert torch.isfinite(ddpm).all()
    bit_equal = torch.equal(ddpm, ddim)
    assert bit_equal, f"DDIM(S=T, eta=1) differs from DDPM: max |diff| {(ddpm - ddim).abs().max().item()}"

    cases = [(B, s, S) for B in WINDOWS for s, S in SAMPLERS]
    for c in cases:
        run(*c)
    torch.cuda.synchronize()
    times = {c: [] for c in cases}
    for _ in range(args.repeats):
        for c in cases:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run(*c)
            torch.cuda.synchronize()
            times[c].append(time.perf_counter() - t0)

    results = []
    for (B, sampler, S), ts in times.items():
        med = statistics.median(ts)
        results.append(dict(windows=B, sampler=sampler, steps=S, s_per_batch=round(med, 5), s_min=round(min(ts), 5),
                            s_max=round(max(ts), 5), ms_per_step=round(1e3 * med / S, 4),
                            windows_per_s=round(B / med, 1), denoise_steps_per_s=round(S / med, 1)))
    line = json.dumps(dict(bench="sampling_steps", model="configs[3] denoiser d=512 h=8 ff=2048 L=8 F=50", **device_info(),
                           repeats=args.repeats, ddim_full_eta1_equals_ddpm_bitwise=bit_equal, results=results))
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
