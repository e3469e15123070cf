"""Auxiliary measurements of bench.py for the BASELINE configs other than the headline one (which is the
denoiser training step): configs[0] FeedForward training (reference shape B=32 and a GPU-sized batch),
Groundlink training, and configs[4] the TransformerBaseline analysis pass over a long-window (T=200) stream.

Every leg is timed with CUDA events on the launching stream after warm-up, through the drop-in classes /
Trainer (the public calls), and reports its algorithmic FLOPs (SURVEY §8d figures) next to the time.
"""
from __future__ import annotations

from typing import Dict

import torch

from . import ops


def _events():
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def max_over_ranks(ms: float) -> float:
    """Every multi-GPU figure is computed from the SLOWEST rank's device time (all_reduce MAX), never rank 0's alone."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    return ms


def _barrier():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.barrier()
    torch.cuda.synchronize()


def _per_kernel(fn) -> Dict[str, dict]:
    """One extra instrumented pass: CUDA events around every C-ABI launch (live, no profiler)."""
    real_call = ops.call
    recs = []

    def timed_call(name, *a):
        e0, e1 = _events()
        e0.record()
        real_call(name, *a)
        e1.record()
        recs.append((name, e0, e1))

    ops.call = timed_call
    try:
        fn()
        torch.cuda.synchronize()
    finally:
        ops.call = real_call
    per: Dict[str, list] = {}
    for name, e0, e1 in recs:
        p = per.setdefault(name, [0, 0.0])
        p[0] += 1
        p[1] += e0.elapsed_time(e1)
    return {k: {"launches": v[0], "ms": round(v[1], 4)} for k, v in sorted(per.items(), key=lambda kv: -kv[1][1])}


def feedforward_train_leg(dev, world: int, steps: int = 20) -> dict:
    """BASELINE configs[0] shape on the GPU: FeedForwardBaseline 1470->512->512->300 (D=23, T=50, stride 5, sigmoid,
    RMSprop 1e-4; FeedForward...py:20-78, train.py:183-197), one Trainer.train_step per step (packer -> 3 tcgen05 GEMMs
    -> fused loss -> backward -> fused optimizer).  5 505 024 FLOP/window fwd+bwd (SURVEY §8d)."""
    from .data.window_store import WindowStore
    from .models.FeedForwardRegressionBaseline import FeedForwardBaseline
    from .trainer import Trainer
    torch.manual_seed(0)
    model = FeedForwardBaseline(23, 2, 50, "all_frames", "sigmoid", 5, 10, hidden_dims=[512, 512]).to(dev)
    trainer = Trainer(model, opt_type="rmsprop", lr=1e-4)
    out = {}
    for B in (32, 16384):
        store = WindowStore.synthetic(B * 2, 50, 5, 147, "all_frames", seed=77, device=dev)
        idx = store.shard(0, 1)
        batches = [idx[:B], idx[B:2 * B]]
        for i in range(3):
            trainer.train_step(store, batches[i % 2])
        e0, e1 = _events()
        _barrier()
        e0.record()
        for i in range(steps):
            trainer.train_step(store, batches[i % 2])
        e1.record()
        _barrier()
        ms = max_over_ranks(e0.elapsed_time(e1) / steps)
        out[f"batch_{B}"] = {"windows_per_s": world * B / (ms * 1e-3), "ms_per_step": ms,
                             "tflops": 5505024.0 * B / (ms * 1e-3) / 1e12}
        del store
    out["note"] = "configs[0] model on the GPU; batch 32 is launch-latency bound (about 20 launches per step), batch 16384 is the throughput shape"
    return out


def groundlink_train_leg(dev, world: int, steps: int = 10, B: int = 4096, T: int = 50) -> dict:
    """Groundlink (Groundlink.py:20-156) training: implicit-GEMM temporal CNN + per-frame MLP, forward + backward with
    Dropout(0.2) active, 110.0 MFLOP/window forward at T=50 (SURVEY §8d), ~3x for the step.  Two paths over the same
    kernels: the native ``Trainer`` step (window store -> padded-row packer -> fused loss -> fused RMSprop) and the reference's
    loop shape (module forward -> evaluator -> loss.backward() -> torch.optim.RMSprop.step())."""
    import argparse
    from .data.window_store import WindowStore
    from .keys import LOSS_QUANTITIES, MODEL_INPUT_ORDER
    from .loss.RegressionLossEvaluator import RegressionLossEvaluator
    from .models.Groundlink import Groundlink
    from .trainer import Trainer
    torch.manual_seed(0)
    out = {"batch": B, "frames": T}

    def timed(step):
        for _ in range(3):
            step()
        e0, e1 = _events()
        _barrier()
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        _barrier()
        ms = max_over_ranks(e0.elapsed_time(e1) / steps)
        return {"windows_per_s": world * B / (ms * 1e-3), "ms_per_step": ms, "tflops_model": 3 * 110.016e6 * B / (ms * 1e-3) / 1e12}

    store = WindowStore.synthetic(2 * B, T, 1, 177, "all_frames", seed=5, device=dev)
    idx = store.shard(0, 1)
    batches = [idx[:B], idx[B:2 * B]]
    m = Groundlink(23, 12, 10, "all_frames").to(dev).train()
    tr = Trainer(m, opt_type="rmsprop", lr=1e-4)
    it = [0]

    def native():
        it[0] += 1
        tr.train_step(store, batches[it[0] & 1])

    out["native_trainer"] = timed(native)
    del tr, m

    m = Groundlink(23, 12, 10, "all_frames").to(dev).train()
    opt = torch.optim.RMSprop(m.parameters(), lr=1e-4)
    ev = RegressionLossEvaluator(dataset=None, split="train", device=str(dev))
    args = argparse.Namespace(predict_grf_components=list(range(6)), predict_cop_components=list(range(6)),
                              predict_moment_components=list(range(6)), predict_wrench_components=list(range(12)))
    widths = [23, 23, 23, 3, 3, 3, 3, 36, 30, 30]
    x = dict(zip(MODEL_INPUT_ORDER, [t.contiguous() for t in torch.split(store.pack_f32(batches[0]), widths, dim=-1)]))
    labels = dict(zip(LOSS_QUANTITIES, [t.contiguous() for t in torch.split(store.labels(batches[0]), [6, 6, 6, 12], dim=-1)]))

    def module_loop():
        opt.zero_grad()
        loss = ev(x, m(x), labels, [], [], args, compute_report=False)
        loss.backward()
        opt.step()
        ev._reset_lists()

    out["module_loop"] = timed(module_loop)
    return out


def transformer_analyze_leg(dev, world: int, pk: dict, B: int = 2048, T: int = 200, n_batches: int = 6) -> dict:
    """BASELINE configs[4]: TransformerBaseline (TransformerBaseline.py:73-148; d=108, 3 heads, 3 layers, FFN 60) analysis
    pass over a stream of long windows (T=200), contiguous window shards per GPU, no collective.  142 065 600
    FLOP/window forward (SURVEY §8d).  `value`: inputs resident in HBM; `e2e`: inputs in pinned host memory, H2D of
    every batch and D2H of its three outputs inside the timed region.  fp32 parameters (ctor dtype argument)."""
    from .keys import InputDataKeys as K, OutputDataKeys as O
    from .models.TransformerBaseline import TransformerBaseline
    torch.manual_seed(0)
    D = 23
    m = TransformerBaseline(D, T, dtype=torch.float32).to(dev)
    g = torch.Generator(device=dev).manual_seed(11)
    chans = [(K.POS, D), (K.VEL, D), (K.ACC, D), (K.COM_POS, 3), (K.COM_VEL, 3), (K.COM_ACC, 3)]
    x = {k: torch.randn(B, c, T, device=dev, generator=g) for k, c in chans}
    torch.set_grad_enabled(False)                     # the analysis pass (analyze.py:112-156 runs under torch.no_grad())
    for _ in range(20):                               # ~50 ms of work: a GPU that was idle needs it to reach its clocks
        m(x)
    e0, e1 = _events()
    _barrier()
    e0.record()
    for _ in range(n_batches):
        out = m(x)
    e1.record()
    _barrier()
    ms = max_over_ranks(e0.elapsed_time(e1) / n_batches)
    kern = _per_kernel(lambda: m(x))
    torch.set_grad_enabled(True)
    kern_ms = sum(v["ms"] for v in kern.values())
    # end to end: pinned host inputs, outputs read back
    xh = {k: v.cpu().pin_memory() for k, v in x.items()}

    def e2e_pass(n):
        got = 0
        for o in m.forward_stream([xh] * n):         # pinned host inputs in, pinned host outputs out, copies overlapped
            got += 1
        assert got == n

    e2e_pass(3)
    _barrier()
    e0.record()
    e2e_pass(2 * n_batches)
    e1.record()
    _barrier()
    ms_e2e_f32 = max_over_ranks(e0.elapsed_time(e1) / (2 * n_batches))
    # the same stream pre-packed ONCE on the host to frame-major bf16 rows (TransformerBaseline.prepack): half the link bytes
    xp = TransformerBaseline.prepack(xh)
    xh_f32 = xh

    def e2e_packed(n):
        got = 0
        for o in m.forward_stream([xp] * n):
            got += 1
        assert got == n

    e2e_packed(3)
    _barrier()
    e0.record()
    e2e_packed(2 * n_batches)
    e1.record()
    _barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1) / (2 * n_batches))
    xh = {"packed": xp}
    oh = next(iter(m.forward_stream([xp])))
    # the host link on its own: the same pinned tensors copied H2D with nothing else running (explains the e2e figure, which is
    # bound by max(compute, H2D) per batch)
    xd = {k: torch.empty_like(v, device=dev) for k, v in xh.items()}
    for k, v in xh.items():
        xd[k].copy_(v, non_blocking=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(4):
        for k, v in xh.items():
            xd[k].copy_(v, non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    h2d_only_ms = max_over_ranks(e0.elapsed_time(e1) / 4)
    del xd
    h2d = sum(v.numel() * v.element_size() for v in xh.values())
    d2h = sum(v.numel() * v.element_size() for v in oh.values())
    fl = 142065600.0 * B
    return {"metric": "transformer_analyze_windows_per_sec", "value": world * B / (ms * 1e-3), "unit": "windows/s",
            "ms_per_batch": ms, "batch_windows": B, "window_frames": T, "tflops": fl / (ms * 1e-3) / 1e12,
            "kernel_ms_per_batch": kern_ms, "kernels": kern,
            "e2e": {"value": world * B / (ms_e2e * 1e-3), "unit": "windows/s", "ms_per_batch": ms_e2e, "h2d_bytes_per_batch": h2d,
                    "d2h_bytes_per_batch": d2h, "h2d_alone_ms_per_batch": h2d_only_ms,
                    "h2d_alone_gbs": sum(v.numel() * v.element_size() for v in xh.values()) / h2d_only_ms / 1e6,
                    "fp32_dict_feed": {"value": world * B / (ms_e2e_f32 * 1e-3), "ms_per_batch": ms_e2e_f32,
                                       "h2d_bytes_per_batch": sum(v.numel() * v.element_size() for v in xh_f32.values())},
                    "api": "TransformerBaseline.forward_stream(iterable of TransformerBaseline.prepack(batch) tensors): windows converted "
                           "once on the host to frame-major bf16 rows; H2D of every batch and D2H of its three outputs timed"},
            "full_stream": f"2^20 windows = {(1 << 20) / (world * B / (ms * 1e-3)):.2f} s at this rate on {world} GPU(s)",
            "note": "weak scaling (contiguous window shards, no collective); d=108 rows are padded to 112 bf16 columns, heads 36->48"}


def sampling_leg(dev, world: int, rank: int, pk: dict, model, windows_per_gpu: int = 512, steps: int = 1000) -> dict:
    """BASELINE configs[3] as stated: DDPM reverse sampling, the FULL 1000-step schedule, 4096 windows sharded over 8 GPUs =
    512 windows per GPU (weak scaling: every rank samples its own 512, no collective).  ``value``: kinematic conditions
    already packed in HBM, device-timed over the 1000 graph-replayed denoise steps, MAX over ranks.  ``e2e``: the public
    call ``GaussianDiffusion.sample_windows`` with the conditions in pinned HOST memory and the trajectories returned to
    pinned host memory (H2D + packing + 1000 steps + D2H inside the timed region).  ``roofline``: tensor-bound — algorithmic
    FLOPs of the GEMM launches of one denoise step / their summed CUDA-event time (one eager, instrumented step)."""
    from .diffusion import GaussianDiffusion
    eng = model.engine()
    F, C = eng.F, eng.c_in
    sb = windows_per_gpu
    gd = GaussianDiffusion(device=dev)
    g = torch.Generator().manual_seed(4242)
    cond_host = torch.randn(world * sb, F, C, generator=g).pin_memory()          # the whole job's windows; a rank reads its shard
    mine = slice(rank * sb, (rank + 1) * sb)
    buf, fs, we, col0 = eng.input_layout(sb, F, False)
    ops.pack_inputs([cond_host[mine].reshape(-1, C).to(dev)], sb * F, F, out_bf16=buf, frame_stride=fs, win_extra=we, col0=col0)
    seed = 1
    gd.sample(model, sb, steps=20, seed=seed + rank)                             # captures the 2-step graph, warms the clocks
    e0, e1 = _events()
    _barrier()
    e0.record()
    x0 = gd.sample(model, sb, steps=steps, seed=seed + rank)
    e1.record()
    _barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    assert torch.isfinite(x0).all()
    # end to end through the public sharded call
    gd.sample_windows(model, cond_host, batch=sb, steps=4, seed=seed)            # staging buffers, streams
    _barrier()
    e0.record()
    rng, traj = gd.sample_windows(model, cond_host, batch=sb, steps=steps, seed=seed)
    e1.record()
    _barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    assert len(rng) == sb and tuple(traj.shape) == (sb, F, 30) and not traj.is_cuda
    # GEMMs of one denoise step (eager, events around every launch)
    real = ops.gemm
    recs = []

    def timed(A, Bm, out, M, N, K, **kw):
        a, b = _events()
        a.record()
        r = real(A, Bm, out, M, N, K, **kw)
        b.record()
        recs.append((a, b, 2.0 * M * N * K))
        return r

    ops.gemm = timed
    try:
        gd.sample(model, sb, steps=2, seed=seed + rank, use_graph=False)
        torch.cuda.synchronize()
    finally:
        ops.gemm = real
    gemm_ms = sum(a.elapsed_time(b) for a, b, _ in recs) / 2
    gemm_fl = sum(f for _, _, f in recs) / 2
    peak = pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
    ach = gemm_fl / (gemm_ms * 1e-3) / 1e12
    ms_step = ms / steps
    return {
        "metric": "denoise_window_steps_per_sec", "value": world * sb * steps / (ms * 1e-3), "unit": "window-steps/s",
        "n_gpus": world, "higher_is_better": True, "scaling": "weak", "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "BASELINE configs[3]: DDPM reverse sampling of GRF/CoP/torque/wrench trajectories, full schedule",
                   "denoise_steps": steps, "windows_per_gpu": sb, "windows_total": world * sb, "frames": F, "cond_channels": C,
                   "d_model": eng.d, "heads": eng.H, "ffn": eng.ff, "layers": eng.L, "parallelism": f"window shards x{world}, no collective"},
        "ms_per_denoise_step": ms_step, "seconds_per_1000_step_batch": ms * 1e-3,
        "e2e": {"value": world * sb * steps / (ms_e2e * 1e-3), "unit": "window-steps/s", "h2d_bytes_per_step": sb * F * C * 4,
                "d2h_bytes_per_step": sb * F * 30 * 4, "seconds": ms_e2e * 1e-3,
                "api": "GaussianDiffusion.sample_windows(model, cond: pinned host (N, F, 177), batch=512): a step of this leg = one "
                       "512-window batch through all denoise steps; H2D conditions + pack + sampling + D2H trajectories timed"},
        "roofline": {"bound": "tensor", "kernel": "ibm::gemm::gemm_kernel (all GEMM launches of one denoise step, M = 25 600 rows)",
                     "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
                     "gemm_ms_per_step": gemm_ms, "gemm_launches_per_step": len(recs) // 2, "gemm_share_of_step": gemm_ms / ms_step,
                     "step_model_tflops": 2.57e9 * sb / (ms_step * 1e-3) / 1e12,
                     "note": "512 windows x 50 frames = 25 600 rows per GEMM: 13-54 GFLOP launches of 15-50 us; the step is a chain of "
                             "~60 short dependent launches replayed from a CUDA graph"},
    }


def batch1_latency_leg(dev) -> dict:
    """SURVEY §8f-4: latency of ``model(inputs)`` on ONE window from host tensors under no_grad, as the per-window viewers call
    it (visualize.py:157-186, save_prediction_csv.py:91-113): host wall-clock per call including the H2D copy of the window and
    a device synchronize (the caller reads the prediction), median of 200 calls; eager launches vs the captured graph."""
    import os
    import statistics
    import time
    from .keys import MODEL_INPUT_ORDER
    from .models.FeedForwardRegressionBaseline import FeedForwardBaseline
    from .models.Groundlink import Groundlink
    torch.manual_seed(0)
    out = {}
    widths = lambda hist: dict(zip(MODEL_INPUT_ORDER, [23, 23, 23, 3, 3, 3, 3, 36, hist, hist]))
    cases = {"feedforward": (FeedForwardBaseline(23, 2, 50, "all_frames", "sigmoid", 5, 10).to(dev).eval(), 10, 15),
             "groundlink": (Groundlink(23, 12, 10, "all_frames").to(dev).eval(), 50, 30)}
    prev = os.environ.get("IBM_INFER_GRAPHS")
    try:
        with torch.no_grad():
            for name, (m, F, hist) in cases.items():
                x = {k: torch.randn(1, F, w) for k, w in widths(hist).items()}
                res = {}
                for mode, flag in (("eager", "0"), ("graph", "1")):
                    os.environ["IBM_INFER_GRAPHS"] = flag
                    for _ in range(10):
                        m(x)
                    torch.cuda.synchronize()
                    ts = []
                    for _ in range(200):
                        t0 = time.perf_counter()
                        o = m(x)
                        torch.cuda.synchronize()
                        ts.append(time.perf_counter() - t0)
                    res[f"{mode}_us"] = round(statistics.median(ts) * 1e6, 1)
                out[name] = res
    finally:
        if prev is None:
            os.environ.pop("IBM_INFER_GRAPHS", None)
        else:
            os.environ["IBM_INFER_GRAPHS"] = prev
    out["note"] = "one window per call from CPU tensors; host wall-clock incl. concat + H2D + launches + synchronize, median of 200"
    return out
