"""Worker of tests/test_gpu_clip_sched.py: one process per GPU (torchrun), NCCL.  Every rank trains a FeedForward model with
global-norm clipping active on every step and a warm-up + cosine schedule, from DIFFERENT initial weights (the broadcast
equalises them), and writes the masters and the clip record {total, coefficient} after every step to <out>/rank<r>.pt.
The allreduce mode and graph replay come from the environment (IBM_ALLREDUCE, IBM_TRAIN_GRAPHS)."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))


def main(out_dir: str, steps: int, B: int):
    from inferbiomechanics_b200 import parallel
    from inferbiomechanics_b200.data.window_store import WindowStore
    from inferbiomechanics_b200.models.FeedForwardRegressionBaseline import FeedForwardBaseline
    from inferbiomechanics_b200.trainer import Trainer
    rank, world, local = parallel.init_from_env("nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    torch.manual_seed(100 + rank)
    model = FeedForwardBaseline(23, 2, 50, "all_frames", "sigmoid", 5, 10, hidden_dims=[64, 64]).to(dev)
    store = WindowStore.synthetic(2048, 50, 5, 147, "all_frames", seed=3, device=dev)
    tr = Trainer(model, opt_type="adam", lr=1e-3, seed=5, clip_grad_norm=1e-3, lr_warmup_steps=2, lr_schedule="cosine",
                 total_steps=steps, lr_min=1e-4)
    idx = store.shard(rank, world)
    masters, clips = [], []
    for s in range(steps):
        tr.train_step(store, idx[s * B:(s + 1) * B])
        masters.append(tr.arena.master.cpu())
        clips.append(tr._clip_ws.out.cpu())
    torch.save({"master": masters, "clip": clips, "stats": tr.grad_norm_stats(),
                "graphs": sum(g[1] is not None for g in tr._graphs.values())}, os.path.join(out_dir, f"rank{rank}.pt"))
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main(sys.argv[1], int(sys.argv[2]), int(sys.argv[3]))
