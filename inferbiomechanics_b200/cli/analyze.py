"""``analyze`` command: evaluates the latest checkpoint on the dev and train splits and prints the evaluator's
report, flags as in ``/root/reference/src/cli/analyze.py:20-242``.

The reference walks a ``DataLoader(batch_size=1)`` in one process (analyze.py:112,139-180); windows are
independent, so here each rank takes a CONTIGUOUS range of windows in large equal batches (SURVEY §8e: no
collective during the pass), keeps the per-batch fp32[40] results on the device and merges them once at the end —
equal batch sizes keep the reference's mean-of-batch-means aggregate (RegressionLossEvaluator.py:383-387) exact.
Per-window plots (matplotlib) and the names CSV are outside the hot path.  ``--model-type diffusion`` runs the
reverse sampler per batch (``--sampler ddpm``: the 1000-step chain; ``ddim``: ``--sampling-steps`` respaced steps;
``dpmpp2m``: ``--sampling-steps`` steps of the second-order multistep DPM-Solver++(2M) on log-SNR-spaced timesteps) and
scores the sampled trajectories with the same evaluator; ``--guidance-scale`` samples it with classifier-free guidance, which
needs a checkpoint trained with ``train --cond-drop-prob``.  ``--num-samples K`` (K >= 2) draws K samples per window: the
evaluator scores their mean and an ``EnsembleScorer`` block (CRPS, spread, spread-skill ratio, pairwise distance) follows
the report.  ``--given-quantities force ...`` gives the sampler the labels of those quantities as known values (inpainting):
they come back exactly, and the report's other quantities are the prediction conditioned on them.
"""
from __future__ import annotations

import argparse
import logging
import os

import torch
import torch.distributed as dist

from .. import parallel
from ..diffusion import MAX_NUM_SAMPLES, GaussianDiffusion, check_guidance_scale
from ..loss.RegressionLossEvaluator import RegressionLossEvaluator
from ..loss.ensemble import ENSEMBLE_GROUPS, EnsembleScorer
from ..trainer import Trainer
from . import _data
from .abstract_command import AbstractCommand
from .train import _ResultLog, input_dict, label_dict, sample_and_score


class AnalyzeCommand(AbstractCommand):
    def __init__(self):
        super().__init__()

    def register_subcommand(self, subparsers: argparse._SubParsersAction):
        sp = subparsers.add_parser('analyze', help='Evaluate the performance of a model on dataset.')
        sp.add_argument('--dataset-home', type=str, default='../data', help='The path to the AddBiomechanics dataset.')
        sp.add_argument('--model-type', type=str, default='feedforward', help='The model to train.')
        sp.add_argument('--no-wandb', action='store_true', default=False, help='Log this analysis to Weights and Biases.')
        sp.add_argument('--output-data-format', type=str, default='all_frames', choices=['all_frames', 'last_frame'],
                        help='Output for all frames in a window or only the last frame.')
        sp.add_argument('--checkpoint-dir', type=str, default='../checkpoints', help='Where the checkpoints of `train` live.')
        sp.add_argument('--geometry-folder', type=str, default=None, help='Path to the Geometry folder with bone mesh data.')
        sp.add_argument('--history-len', type=int, default=50,
                        help='The number of timesteps of context to show when constructing the inputs.')
        sp.add_argument('--stride', type=int, default=5,
                        help='The number of timesteps of context to show when constructing the inputs.')
        sp.add_argument('--hidden-dims', type=int, nargs='+', default=[512, 512], help='Hidden dims across different layers.')
        sp.add_argument('--activation', type=str, default='sigmoid', help='Which activation func?')
        sp.add_argument('--batchnorm', action='store_true', help='The checkpoint was trained with --batchnorm (else read off its keys).')
        sp.add_argument('--dropout', action='store_true', help='The checkpoint was trained with --dropout (else read off its keys).')
        sp.add_argument('--device', type=str, default='cuda', help='Accepted for compatibility; this path runs on the GPU only.')
        sp.add_argument('--short', type=bool, default=False, help='Use very short datasets to test without loading a bunch of data.')
        sp.add_argument('--data-loading-workers', type=int, default=3, help='Accepted for compatibility.')
        sp.add_argument('--predict-grf-components', type=int, nargs='+', default=[1], help='Which grf components to train.')
        sp.add_argument('--predict-cop-components', type=int, nargs='+', default=[], help='Which grf components to train.')
        sp.add_argument('--predict-moment-components', type=int, nargs='+', default=[], help='Which grf components to train.')
        sp.add_argument('--predict-wrench-components', type=int, nargs='+', default=[], help='Which grf components to train.')
        # additions of the B200 path
        sp.add_argument('--synthetic-windows', type=int, default=0, help='Analyze synthetic windows instead of *.ibmstore files.')
        sp.add_argument('--batch-size', type=int, default=4096, help='Windows per launch (the reference analyses one at a time).')
        sp.add_argument('--sampling-steps', type=int, default=1000,
                        help='Reverse-diffusion steps for --model-type diffusion.  --sampler ddpm: the first N steps of the '
                             '1000-step chain (N < 1000 truncates it and scores a partially denoised sample); --sampler ddim '
                             'and dpmpp2m: the number S of steps (1..1000).')
        sp.add_argument('--sampler', type=str, default='ddpm', choices=['ddpm', 'ddim', 'dpmpp2m'],
                        help='Reverse sampler for --model-type diffusion: the ancestral DDPM chain, few-step DDIM, or the '
                             'second-order multistep DPM-Solver++(2M) (deterministic given x_T, one forward per step like '
                             'DDIM, more accurate at the same S).')
        sp.add_argument('--eta', type=float, default=0.0,
                        help='DDIM noise scale in [0, 1] (0: deterministic given x_T; 1: respaced ancestral sampling); '
                             '--sampler ddim only.')
        sp.add_argument('--ema', action='store_true', default=False,
                        help="Evaluate the checkpoint's EMA weights (ema_state_dict, written by train --ema-decay) instead of "
                             "the trained ones.")
        sp.add_argument('--guidance-scale', type=float, default=1.0,
                        help='--model-type diffusion: classifier-free guidance scale s (x0 = u + s (c - u)) with either '
                             'sampler; 1 = no guidance, 0 = unconditional. s != 1 needs a checkpoint trained with '
                             'train --cond-drop-prob > 0.')
        sp.add_argument('--num-samples', type=int, default=1,
                        help=f'--model-type diffusion: samples drawn per window (1..{MAX_NUM_SAMPLES}).  K >= 2 scores the '
                             'ensemble mean with the evaluator and adds CRPS, spread, spread-skill ratio and mean pairwise '
                             'distance per quantity; each launch then samples batch-size // K windows x K draws.')
        sp.add_argument('--given-quantities', type=str, nargs='+', default=[], choices=list(ENSEMBLE_GROUPS),
                        help='--model-type diffusion: quantities whose labels the sampler is given and holds fixed '
                             '(inpainting); they read 0 error and the others are predicted conditionally on them.  Needs '
                             '--output-data-format all_frames and the whole chain (not --sampler ddpm with --sampling-steps < 1000).')

    def run(self, args: argparse.Namespace):
        if 'command' in args and args.command != 'analyze':
            return False
        if args.sampler != 'ddim' and args.eta != 0.0:
            raise ValueError("--eta applies to --sampler ddim only")
        model_type: str = args.model_type
        checkpoint_dir: str = os.path.join(os.path.abspath(args.checkpoint_dir), model_type)
        guidance = args.guidance_scale
        if guidance != 1.0:
            self.check_guidance_checkpoint(model_type, guidance, checkpoint_dir)
        K = args.num_samples
        self.check_num_samples(model_type, K, args.batch_size)
        given = tuple(args.given_quantities)
        self.check_given_quantities(given, model_type, args)
        # windows per launch: K draws each, so that every launch but the last holds the same number of windows
        per_launch = args.batch_size // K
        root_history_len = 10
        rank, world, local = parallel.init_from_env("nccl")
        torch.cuda.set_device(local)
        device = torch.device("cuda", local)
        # --batchnorm / --dropout shift the nn.Sequential positions of the checkpoint's keys (SURVEY §9.3; the reference's analyze has no
        # such flags and cannot load those checkpoints): taken from the flags, else read off the latest checkpoint's keys
        batchnorm, dropout = self.feedforward_layout(checkpoint_dir) if model_type == 'feedforward' else (False, False)
        model = self.get_model(_data.NUM_DOFS, 2, model_type, history_len=args.history_len, hidden_dims=args.hidden_dims,
                               activation=args.activation, stride=args.stride, batchnorm=args.batchnorm or batchnorm,
                               dropout=args.dropout or dropout, dropout_prob=0.0,
                               root_history_len=root_history_len, output_data_format=args.output_data_format,
                               device=str(device)).to(device)
        self.load_latest_checkpoint(model, checkpoint_dir=checkpoint_dir, state_key='ema_state_dict' if args.ema else 'model_state_dict')
        model.eval()
        native = model_type == 'feedforward'
        trainer = Trainer(model, args=args) if native else None
        diffusion = GaussianDiffusion(device=device) if model_type == 'diffusion' else None
        if not args.no_wandb:
            import wandb
            wandb.init(project="addbiomechanics-baseline", config=dict(args.__dict__))

        reports, ensemble_reports = {}, {}
        for split, seed in (('dev', 4321), ('train', 1234)):
            logging.info(f'## Loading {split} dataset:')
            store = _data.open_split(args, split, model_type, device, seed=seed)
            n = len(store)
            shard = parallel.contiguous_shard(n, rank, world)
            idx_all = torch.arange(shard.start, shard.stop, device=device)
            log, ev = _ResultLog(split), RegressionLossEvaluator(None, split, device=device)
            scorer = EnsembleScorer(K, split, device=device) if K > 1 else None
            with torch.no_grad():
                for i in range(0, idx_all.numel(), per_launch):
                    idx = idx_all[i:i + per_launch]
                    if native:
                        log.add(trainer.eval_step(store, idx))
                        continue
                    if model_type == 'diffusion':
                        ens = dict(num_samples=K, scorer=scorer) if scorer is not None else {}
                        if given:
                            ens["known_quantities"] = given
                        if args.sampler == 'ddim':
                            sample_and_score(diffusion, model, store, idx, ev, args, 1234 + rank, ddim_steps=args.sampling_steps,
                                             eta=args.eta, guidance_scale=guidance, **ens)
                        elif args.sampler == 'dpmpp2m':
                            sample_and_score(diffusion, model, store, idx, ev, args, 1234 + rank, dpm_steps=args.sampling_steps,
                                             guidance_scale=guidance, **ens)
                        else:
                            sample_and_score(diffusion, model, store, idx, ev, args, 1234 + rank, steps=args.sampling_steps,
                                             guidance_scale=guidance, **ens)
                        continue
                    inputs = input_dict(store, idx, model_type, args.stride, root_history_len)
                    ev(inputs, model(inputs), label_dict(store, idx), [], [], args)
            src = log.ev if native else ev
            # one merge of the per-rank batch results at the very end (≈ 40 floats per batch); no collective before
            if world > 1:
                mine = torch.stack(src._results) if src._results else torch.zeros(0, 40, device=device)
                counts = [torch.zeros(1, dtype=torch.long, device=device) for _ in range(world)]
                dist.all_gather(counts, torch.tensor([mine.shape[0]], device=device))
                mx = int(max(c.item() for c in counts))
                padded = torch.zeros(mx, 40, device=device)
                padded[:mine.shape[0]] = mine
                gathered = [torch.zeros_like(padded) for _ in range(world)]
                dist.all_gather(gathered, padded)
                merged = [g[:int(c.item())] for g, c in zip(gathered, counts)]
                src._results = [r for g in merged for r in g]
                src._wm_results = list(src._results)
            if scorer is not None:
                scorer.merge(world)
            if rank == 0:
                print(f'{split} set evaluation ({n} windows' + (f', guidance scale {guidance:g}' if guidance != 1.0 else '') +
                      (f', ensemble mean of {K} samples' if scorer is not None else '') +
                      (f', given {" ".join(given)}' if given else '') + '):')
                reports[split] = src.aggregate()
                src.print_report(args, log_to_wandb=not args.no_wandb)
                if scorer is not None:
                    ensemble_reports[split] = scorer.summary()
                    scorer.print_report(args, log_to_wandb=not args.no_wandb, summary=ensemble_reports[split], given=given)
        if dist.is_initialized():
            dist.destroy_process_group()
        self.last_reports = reports
        self.last_ensemble_reports = ensemble_reports
        return True

    @staticmethod
    def check_num_samples(model_type: str, num_samples: int, batch_size: int) -> None:
        """ValueError unless ``--num-samples`` can run: 1 <= K <= 64, K >= 2 for the diffusion model only, K <= --batch-size
        (each launch samples batch-size // K windows x K draws)."""
        if not 1 <= num_samples <= MAX_NUM_SAMPLES:
            raise ValueError(f"--num-samples must lie in [1, {MAX_NUM_SAMPLES}], got {num_samples}")
        if num_samples > 1 and model_type != 'diffusion':
            raise ValueError("--num-samples > 1 applies to --model-type diffusion only")
        if num_samples > batch_size:
            raise ValueError(f"--num-samples {num_samples} exceeds --batch-size {batch_size}: a launch samples batch-size // K "
                             "windows x K draws")

    @staticmethod
    def check_given_quantities(given, model_type: str, args) -> None:
        """ValueError unless ``--given-quantities`` can run: a diffusion model, labels of every frame (the known values are the
        labels) and the whole chain (a truncated DDPM chain stops before the step that returns the known values)."""
        if not given:
            return
        if model_type != 'diffusion':
            raise ValueError("--given-quantities applies to --model-type diffusion only")
        if args.output_data_format != 'all_frames':
            raise ValueError("--given-quantities needs --output-data-format all_frames: last_frame labels hold one frame")
        if args.sampler == 'ddpm' and args.sampling_steps < 1000:
            raise ValueError(f"--given-quantities needs the whole chain: --sampler ddpm --sampling-steps {args.sampling_steps} "
                             "truncates it")

    def check_guidance_checkpoint(self, model_type: str, guidance_scale: float, checkpoint_dir: str) -> None:
        """ValueError unless guidance can run: a diffusion model, a finite scale >= 0 and a latest checkpoint whose optimizer
        tag records cond_drop_prob > 0 (a denoiser never trained without its condition has no meaningful unconditional
        prediction)."""
        if model_type != 'diffusion':
            raise ValueError("--guidance-scale applies to --model-type diffusion only")
        check_guidance_scale(guidance_scale)
        path = self.latest_checkpoint_path(checkpoint_dir)
        if path is None:
            raise ValueError(f"--guidance-scale {guidance_scale:g} needs a checkpoint trained with --cond-drop-prob > 0; "
                             f"{checkpoint_dir} holds none")
        tag = (torch.load(path, map_location="cpu").get('optimizer_state_dict') or {}).get('ibm_b200') or {}
        if not tag.get('cond_drop_prob', 0.0) > 0.0:
            raise ValueError(f"--guidance-scale {guidance_scale:g} needs a checkpoint trained with --cond-drop-prob > 0; "
                             f"{path} records none")
