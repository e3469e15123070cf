#!/usr/bin/env python
"""Benchmark of the InferBiomechanics hot path on B200 (contract: see task description / DESIGN.md §4).

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU under torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU arm: the reference path on host cores
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR  # also write the last timed step's outputs as .npy

Workload at every N: BASELINE.json configs[1]/[2] — motion-diffusion denoiser TRAINING on synthetic
AddBiomechanics-shaped windows (F=50 frames, 177 kinematic channels, 30 target channels), bf16 GEMMs,
per-GPU batch 4096 windows (weak scaling), d=512 / 8 heads / FFN 2048 / 8 layers, RMSprop 1e-4.
One step = window packer → q_sample → forward → fused regression loss → backward → (bucketed NCCL
allreduce) → fused optimizer.  `value` = windows/s with the frame store resident in HBM; `e2e` = the
same step fed from pinned HOST tensors through Trainer.train_steps_host (every step: H2D of the step's inputs and a
D2H read of its loss inside the timed region; the next batch's copies are prefetched on a copy stream).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "denoiser_train_windows_per_sec"
UNIT = "windows/s"
F, C_IN, D_MODEL, HEADS, FF, LAYERS = 50, 177, 512, 8, 2048, 8
PER_GPU_BATCH = 4096


def config(n_gpus: int, batch: int) -> dict:
    return {
        "workload": "BASELINE configs[1] (N=1) / configs[2] (N>1): diffusion denoiser training, synthetic kinematic windows",
        "frames": F, "cond_channels": C_IN, "target_channels": 30, "d_model": D_MODEL, "heads": HEADS, "ffn": FF,
        "layers": LAYERS, "per_gpu_batch_windows": batch, "global_batch_windows": batch * n_gpus,
        "optimizer": "rmsprop lr=1e-4", "parallelism": f"dp{n_gpus}",
        "l2": "per-step working set (~25 GB of activations) >> 126 MB L2; no explicit flush needed",
    }


def peaks() -> dict:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        d["_source"] = "measured (MEASURED_PEAKS.json)"
        return d
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "_source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled during the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.lines, self.proc, self.first = index, [], None, 0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        """Start of the timed region: samples taken before this point (warm-up) are dropped."""
        self.first = len(self.lines)

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines[self.first:]:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        busy = [c for c in sm if c > 0]
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


CPU_SAMPLE_WINDOWS = 256        # windows per CPU step: a bounded sample of the 4096-window GPU batch (BASELINE.md §3)


def _cpu_denoiser_loop(sample_b: int):
    """(step callable, kind, description).  Real reference modules when the oracle/_ref snapshot (or /root/reference) is there —
    reference TransformerLayer x 8 + reference RegressionLossEvaluator + torch.optim.RMSprop composed per the builder's denoiser
    spec (the reference has no denoiser: src/.gitignore:10 is its only trace) — else the functional CPU port (oracle/train.py)."""
    import torch
    from oracle import ref_cpu
    if ref_cpu.available():
        loop = ref_cpu.denoiser_loop(sample_b, C_IN, F, D_MODEL, HEADS, FF, LAYERS)
        return loop, "reference", ("reference TransformerLayer x8 (TransformerBaseline.py:8-38) + reference RegressionLossEvaluator.__call__ + "
                                   "torch.optim.RMSprop(1e-4) from the oracle/_ref snapshot, composed per the builder's denoiser spec "
                                   "(the reference has no diffusion model)")
    from oracle import ddpm as oddpm
    from oracle import train as otrain
    tr = otrain.PortTrainer(otrain.init_denoiser(C_IN, F, D_MODEL, FF, LAYERS, seed=0), lr=1e-4, opt="rmsprop")
    sched = oddpm.make_schedule()
    g = torch.Generator().manual_seed(1234)
    cond = torch.randn(sample_b, F, C_IN, generator=g)
    _, labels = otrain.synthetic_batch(sample_b, F, 23, 30, 1235)
    x0 = torch.cat([labels[k] for k in (otrain._loss.COP, otrain._loss.FORCE, otrain._loss.TORQUE, otrain._loss.WRENCH)], dim=-1)

    def step():
        t = torch.randint(0, 1000, (sample_b,), generator=g)
        eps = torch.randn(sample_b, F, 30, generator=g)
        tr.step_denoiser(sched, cond, x0, t, eps, labels, LAYERS, HEADS)
    return step, "port", "functional CPU port of the same step (oracle/train.py): oracle/_ref snapshot absent"


def run_reference_arm(args) -> None:
    """The reference's CPU implementation of the path on the box's host cores, all threads, at the requested --steps / --warmup,
    each step a bounded 256-window sample of the 4096-window GPU batch (CPU throughput is flat in the batch size beyond that)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from oracle import ref_cpu
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sample_b = CPU_SAMPLE_WINDOWS
    step, kind, what = _cpu_denoiser_loop(sample_b)
    warm, steps = max(1, args.warmup), max(1, args.steps)
    dt = ref_cpu.time_steps(step, warm, steps)
    v = sample_b / dt
    sample = (f"{sample_b} windows per step (of the {PER_GPU_BATCH}-window GPU batch), {warm} warm-up + {steps} timed steps, torch CPU fp32, "
              f"{cores} threads ({ref_cpu.host()['cpu_model']}); {what}")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": config(args.gpus, PER_GPU_BATCH),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def cpu_baseline_leg() -> dict:
    """Bounded CPU sample of the same workload on the host cores (~10-20 s): 2 warm-up + 8 timed steps of 256 windows."""
    import torch
    from oracle import ref_cpu
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step, kind, what = _cpu_denoiser_loop(CPU_SAMPLE_WINDOWS)
    dt = ref_cpu.time_steps(step, 2, 8)
    return {"value": CPU_SAMPLE_WINDOWS / dt, "unit": UNIT, "cores": cores, "kind": kind, "ms_per_step": dt * 1e3,
            "cpu_model": ref_cpu.host()["cpu_model"],
            "sample": f"{CPU_SAMPLE_WINDOWS} windows/step x 8 timed steps (2 warm-up) of the same denoiser training step, torch CPU fp32; {what}"}


def cpu_other_configs() -> dict:
    """The other BASELINE configs on the host cores, REAL reference modules (BASELINE.md §3: 5 warm-up, >= 30 timed steps for
    configs[0]); bounded so the whole block stays under ~40 s."""
    import torch
    from oracle import ref_cpu
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    out = {"cores": cores, "cpu_model": ref_cpu.host()["cpu_model"]}
    if not ref_cpu.available():
        out["unavailable"] = "oracle/_ref snapshot absent (python -m oracle.build_ref in the build container)"
        return out
    out["kind"] = "reference"
    ff = {}
    for B, warm, n in ((32, 5, 60), (4096, 3, 12)):
        dt = ref_cpu.time_steps(ref_cpu.feedforward_loop(B), warm, n)
        ff[f"batch_{B}"] = {"windows_per_s": B / dt, "ms_per_step": dt * 1e3, "warmup": warm, "steps_timed": n}
    out["feedforward_train"] = dict(ff, what="configs[0]: reference FeedForwardBaseline [512,512] sigmoid + RegressionLossEvaluator + RMSprop(1e-4), fp32")
    gl = {}
    for B, warm, n in ((32, 2, 10), (256, 1, 4)):
        dt = ref_cpu.time_steps(ref_cpu.groundlink_loop(B), warm, n)
        gl[f"batch_{B}"] = {"windows_per_s": B / dt, "ms_per_step": dt * 1e3, "warmup": warm, "steps_timed": n}
    out["groundlink_train"] = dict(gl, what="reference Groundlink(23,12,10) T=50, Dropout(0.2) active + evaluator + RMSprop, fp32")
    dt = ref_cpu.time_steps(ref_cpu.transformer_forward(32), 2, 10)
    out["transformer_analyze"] = {"windows_per_s": 32 / dt, "ms_per_batch": dt * 1e3, "batch": 32, "steps_timed": 10,
                                  "what": "configs[4]: reference TransformerBaseline stack + heads, T=200, fp64, no_grad"}
    sb = 64
    dt = ref_cpu.time_steps(ref_cpu.denoiser_sampler(sb, C_IN, F, D_MODEL, HEADS, FF, LAYERS), 1, 4)
    out["sampling"] = {"window_steps_per_s": sb / dt, "ms_per_denoise_step": dt * 1e3, "windows": sb, "steps_timed": 4,
                       "what": "configs[3]: one reverse step = composed denoiser forward (reference TransformerLayer x8) + posterior update, fp32"}
    return out


DUMP_SAMPLE = 4 << 20          # parameter / gradient elements kept per array: 2 x 16 MB of fp32, well under 64 MB in all


def dump_outputs(out_dir: str, result, arena) -> None:
    """What the last timed step hands its caller, for comparing two builds output for output:
    step_result.npy  the fp32[40] the step returns (loss at [0], then its per-channel and report metrics);
    params.npy       the fp32 parameters the step's optimizer update left in place;
    grads.npy        the fp32 parameter gradients of that step.
    Arenas larger than DUMP_SAMPLE elements are written as the same seeded, sorted sample of positions every run.
    The inputs are seeded, but the bias-gradient and LayerNorm reductions add with float atomics, so two runs differ in the
    last bits of every gradient and RMSprop compounds that over the steps: compare dumps with a tolerance."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    n = arena.total
    idx = None
    if n > DUMP_SAMPLE:
        idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values.to(arena.device)
    for name, t in (("step_result", result), ("params", arena.master), ("grads", arena.grad)):
        if name != "step_result" and idx is not None:
            t = t[idx]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=PER_GPU_BATCH, help="windows per GPU per step")
    ap.add_argument("--no-aux", action="store_true", help="skip the auxiliary sampling / elementwise roofline measurements")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sampling", action="store_true", help="skip the configs[3] reverse-sampling block")
    ap.add_argument("--sampling-steps", type=int, default=1000, help="denoise steps of the sampling block (configs[3]: 1000)")
    ap.add_argument("--sampling-windows", type=int, default=512, help="windows per GPU of the sampling block (configs[3]: 4096 / 8)")
    ap.add_argument("--dump-outputs", type=str, default=None, metavar="DIR",
                    help="GPU arm only: after the timed steps, write what the last timed step computed as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm only, not to --impl reference")
    if args.impl == "reference":
        run_reference_arm(args)
        return
    args.warmup = max(args.warmup, 3)
    # stdout carries exactly ONE JSON line: libraries that print to fd 1 (NCCL's "NCCL version ..." banner) go to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    from inferbiomechanics_b200 import _lib, ops, parallel
    from inferbiomechanics_b200.data.window_store import WindowStore
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    from inferbiomechanics_b200.models.DiffusionDenoiser import DiffusionDenoiser
    from inferbiomechanics_b200.trainer import Trainer

    rank, world, local = parallel.init_from_env("nccl")
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = parallel.bind_to_gpu_numa(local)      # before any pinned allocation: host staging lands on the GPU's NUMA node
    B = args.batch
    torch.manual_seed(0)
    model = DiffusionDenoiser(frames=F, d_model=D_MODEL, num_heads=HEADS, dim_feedforward=FF, num_layers=LAYERS).to(dev)
    diffusion = GaussianDiffusion(device=dev)
    trainer = Trainer(model, opt_type="rmsprop", lr=1e-4, diffusion=diffusion, seed=1234)
    n_batches = 4
    store = WindowStore.synthetic(B * n_batches, F, 1, C_IN, "all_frames", seed=1234 + rank, device=dev)
    idx_all = store.shard(0, 1)
    batches = [idx_all[i * B:(i + 1) * B] for i in range(n_batches)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ------------------------------------------------ value: HBM-resident inputs ---------------------------------
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()                      # nvidia-smi needs a moment to start: launch it before the warm-up
    for i in range(args.warmup):
        trainer.train_step(store, batches[i % n_batches])
    barrier()
    clocks.mark()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = _lib.launch_count
    barrier()
    e0.record()
    for i in range(args.steps):
        res = trainer.train_step(store, batches[i % n_batches])
    e1.record()
    barrier()
    launches = _lib.launch_count - launches0
    elapsed_ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(elapsed_ms, op=dist.ReduceOp.MAX)
    ms_per_step = elapsed_ms.item() / args.steps
    value = world * B / (ms_per_step * 1e-3)
    final_loss = res[0].item()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, model.arena)

    # ------------------------------------------------ e2e: host buffers through the public call ---------------------
    host = trainer.make_host_batch(B, seed=99 + rank)               # pinned CPU tensors (dict of 10 inputs + 4 labels)
    # the public host-fed loop: a generator over (inputs, labels) batches that prefetches the next batch's H2D copies on a
    # copy stream while the current step computes and reads each step's loss back (python float) one step late
    for _ in trainer.train_steps_host([(host["inputs"], host["labels"])] * 3):
        pass
    barrier()
    e0.record()
    for loss_host in trainer.train_steps_host([(host["inputs"], host["labels"])] * args.steps):
        pass
    e1.record()
    barrier()
    e2e_ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = world * B / (e2e_ms.item() / args.steps * 1e-3)
    clock_info = clocks.stop() if rank == 0 else None          # samples cover both timed regions (value and e2e)
    h2d = sum(t.numel() * t.element_size() for t in host["inputs"].values()) + sum(t.numel() * t.element_size() for t in host["labels"].values())

    # ------------------------------------------------ roofline of the dominant kernel (tcgen05 GEMM) ----------------
    pk = peaks()
    gemm_ms, gemm_flops, n_gemm = trainer.profile_gemms(store, batches[0])
    achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12
    peak = pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
    # DRAM traffic of the dominant kernel: ncu --set full captures of its four big shapes (48 of the 106 launches, ~75 % of
    # the GEMM time), committed under profiles/; per launch, like `achieved`
    traffic, traffic_detail = None, None
    tp = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp))
        per = {k: v["dram_read"] + v["dram_write"] for k, v in tj["shapes"].items()}
        traffic = sum(per.values()) / len(per)
        traffic_detail = {"source": tj["_source"], "round": tj["_round"], "per_shape_dram_bytes": per,
                          "per_shape_operand_bytes": {k: v["operand_bytes"] for k, v in tj["shapes"].items()},
                          "note": "traffic = mean over the four captured shapes; DRAM bytes are 0.95-1.12x the operand bytes (each operand "
                                  "crosses HBM once; part of the output stays in the 126 MB L2 for the consumer)"}
    roofline = {"bound": "tensor", "kernel": "ibm::gemm::gemm_kernel (tcgen05.mma + TMA, all shapes of one training step)",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic, "traffic_detail": traffic_detail,
                "peak_source": pk["_source"] + ", sustained figure (kernel timed inside a long step)",
                "launches_per_step": n_gemm, "gemm_ms_per_step": gemm_ms, "gemm_share_of_step": gemm_ms / ms_per_step,
                "step_model_flops_per_window": 3 * 2.57e9}

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic", "config": config(world, B),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "ms_per_step": e2e_ms.item() / args.steps, "api": "for loss in Trainer.train_steps_host(iterable of (inputs: Dict[str, pinned CPU Tensor], labels)): per step H2D of the 14 tensors + D2H loss read, next batch prefetched on a copy stream"},
        "gpu_launches": launches, "roofline": roofline, "final_loss": final_loss, "loss_host": loss_host,
    }
    out["host_affinity"] = None if numa_cpus is None else f"{len(numa_cpus)} cores local to the GPU's PCIe root (rank 0)"
    if rank == 0:
        out["clocks"] = clock_info
    from inferbiomechanics_b200 import bench_legs
    if not args.no_sampling:
        # the second half of BASELINE.json's metric ("train windows/sec & denoise steps/sec"): configs[3] exactly
        out["sampling"] = bench_legs.sampling_leg(dev, world, rank, pk, model, windows_per_gpu=args.sampling_windows,
                                                  steps=args.sampling_steps)
    if not args.no_aux:
        out["aux"] = trainer.aux_measurements(store, batches[0], pk, world)
        # the other BASELINE configs (not the headline metric): configs[0] model on the GPU, Groundlink, configs[4] stream
        del trainer, store
        torch.cuda.empty_cache()
        out["aux"]["feedforward_train"] = bench_legs.feedforward_train_leg(dev, world)
        out["aux"]["groundlink_train"] = bench_legs.groundlink_train_leg(dev, world)
        out["aux"]["transformer_analyze"] = bench_legs.transformer_analyze_leg(dev, world, pk)
        if rank == 0:
            out["aux"]["batch1_latency"] = bench_legs.batch1_latency_leg(dev)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline_leg()
        if "aux" in out:
            out["aux"]["cpu_other_configs"] = cpu_other_configs()
    if rank == 0:
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
