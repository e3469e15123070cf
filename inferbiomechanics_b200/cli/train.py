"""``train`` command: same flags, loop shape, report text and checkpoint format as
``/root/reference/src/cli/train.py:24-296``, on the B200 path.

What changes underneath (and nothing a caller of the command sees): the two DataLoaders become HBM-resident
``WindowStore``s sharded by the reference's DistributedSampler rule; model / loss / backward / optimizer are
one ``Trainer.train_step`` (explicit kernel launches over flat parameter arenas, bucketed NCCL allreduce
overlapped with backward, fused optimizer) instead of autograd + DDP + torch.optim; losses stay on the device
and are read back only at report time, for all three model types (``feedforward``, ``groundlink``, ``diffusion``).
Conscious fixes of reference defects that stop it running (SURVEY §0.4): ``DEV``/``mp``/``time`` are defined,
``any(params_to_optimize)`` is not evaluated on tensors.  One process per GPU under torchrun, as in the reference.
"""
from __future__ import annotations

import argparse
import contextlib
import logging
import os
from typing import List

import torch
import torch.distributed as dist

from .. import parallel
from ..data.window_store import WindowStore
from ..diffusion import GaussianDiffusion
from ..keys import LOSS_QUANTITIES, MODEL_INPUT_ORDER
from ..loss.RegressionLossEvaluator import RegressionLossEvaluator
from ..loss.ensemble import ENSEMBLE_GROUPS
from ..trainer import LR_SCHEDULES, Trainer, check_clip_sched, check_cond_drop
from . import _data
from .abstract_command import AbstractCommand

DEV = 'dev'


def input_dict(store: WindowStore, idx: torch.Tensor, model_type: str, stride: int, root_history_len: int):
    """A reference-shaped batch (Dict[str, Tensor(B,F,C)]) cut out of the packed fp32 window rows."""
    hist = stride * 3 if model_type == "feedforward" else root_history_len * 3
    widths = [_data.NUM_DOFS] * 3 + [3] * 4 + [3 * _data.NUM_JOINTS, hist, hist]
    x = store.pack_f32(idx)
    out, c = {}, 0
    for k, w in zip(MODEL_INPUT_ORDER, widths):
        out[k] = x[:, :, c:c + w]
        c += w
    return out


QUANTITY_CUTS = [(0, 6), (6, 12), (12, 18), (18, 30)]       # column ranges of the four loss quantities in a 30-wide row


def quantity_dict(rows: torch.Tensor):
    """The four loss quantities of (B, F, 30) rows30, as views."""
    return {k: rows[:, :, a:b] for k, (a, b) in zip(LOSS_QUANTITIES, QUANTITY_CUTS)}


def label_dict(store: WindowStore, idx: torch.Tensor):
    return quantity_dict(store.labels(idx))


def known_quantity_mask(quantities) -> torch.Tensor:
    """bool (30,): the rows30 channels of the named quantities (keys of ``ENSEMBLE_GROUPS``: force, cop, moment, wrench)."""
    mask = torch.zeros(30, dtype=torch.bool)
    for q in quantities:
        if q not in ENSEMBLE_GROUPS:
            raise ValueError(f"unknown quantity {q!r}: choose from {', '.join(ENSEMBLE_GROUPS)}")
        a, b = ENSEMBLE_GROUPS[q][0]
        mask[a:b] = True
    return mask


def sample_and_score(diffusion, model, store: WindowStore, idx: torch.Tensor, ev: RegressionLossEvaluator, args, seed: int,
                     *, steps=None, ddim_steps=None, eta: float = 0.0, guidance_scale: float = 1.0, num_samples: int = 1,
                     scorer=None, known_quantities=(), dpm_steps=None) -> None:
    """Reverse-sample the denoiser's trajectories for windows ``idx`` of ``store`` and score them with ``ev`` against the
    store's labels: the condition is the packed kinematics in the engine's concat buffer, x_T ~ Philox(``seed``), and
    ``steps`` / ``ddim_steps`` / ``eta`` / ``dpm_steps`` select the sampler and ``guidance_scale`` the classifier-free guidance as in
    ``GaussianDiffusion.sample``.  ``num_samples`` K >= 2 draws K samples per window: ``scorer`` (an ``EnsembleScorer`` for
    K draws) accumulates their probabilistic scores and ``ev`` scores the ensemble mean.  ``known_quantities`` (names of
    ``ENSEMBLE_GROUPS``): the store's labels of those quantities are given to the sampler as known values (inpainting), so
    the others are predicted conditionally on them; needs labels of every frame."""
    store.pack(idx, model.engine().input_layout(idx.numel(), store.F, False))
    given = {}
    if known_quantities:
        if store.Fo != store.F:
            raise ValueError("known quantities need labels of every frame (--output-data-format all_frames)")
        given = dict(known=store.labels(idx), known_mask=known_quantity_mask(known_quantities))
    if num_samples > 1:
        if scorer is None or scorer.K != num_samples:
            raise ValueError(f"num_samples={num_samples} needs an EnsembleScorer for {num_samples} draws")
        draws = diffusion.sample(model, idx.numel(), steps=steps, seed=seed, ddim_steps=ddim_steps, eta=eta,
                                 guidance_scale=guidance_scale, num_samples=num_samples, dpm_steps=dpm_steps, **given)
        labels = store.labels(idx)
        ev({}, quantity_dict(scorer.score(draws, labels)), quantity_dict(labels), [], [], args)
        return
    x0 = diffusion.sample(model, idx.numel(), steps=steps, seed=seed, ddim_steps=ddim_steps, eta=eta,
                          guidance_scale=guidance_scale, dpm_steps=dpm_steps, **given)
    if store.Fo == 1:                     # --output-data-format last_frame: labels hold the last frame only
        x0 = x0[:, -1:]
    ev({}, quantity_dict(x0), label_dict(store, idx), [], [], args)


class _ResultLog:
    """Device-resident fp32[40] results of ``Trainer`` steps, reported with the evaluator's own text/keys."""

    def __init__(self, split: str):
        self.ev = RegressionLossEvaluator(None, split)

    def add(self, result: torch.Tensor):
        r = result.clone()
        self.ev._results.append(r)
        self.ev._wm_results.append(r)

    def print_report(self, args, reset=True, log_to_wandb=False):
        self.ev.print_report(args, reset=reset, log_to_wandb=log_to_wandb)


def print_all_ranks_report(ev: RegressionLossEvaluator, args, rank: int, world: int, device) -> None:
    """Rank-0 aggregate over all data-parallel ranks, printed next to the per-rank report the reference prints
    (train.py:223-229,286-292 report per process).  One allreduce of the 40-float mean result; every rank must call it,
    BEFORE the evaluator's lists are reset."""
    if world == 1:
        return
    st = ev._stack()
    local = torch.from_numpy(st.mean(axis=0)).to(device) if st.shape[0] else torch.zeros(40, device=device)
    merged = parallel.mean_over_ranks(local)
    if rank == 0:
        tmp = RegressionLossEvaluator(None, ev.split)
        tmp._results = [merged.cpu()]
        tmp._wm_results = [merged.cpu()]
        print(f'[all {world} ranks] {ev.split} set:')
        tmp.print_report(args, reset=True)


class _TrainerOptimizer:
    """``optimizer``-shaped handle on a native ``Trainer`` for ``load_latest_checkpoint`` (abstract_command.py:113-114)."""

    def __init__(self, trainer: Trainer):
        self.trainer = trainer

    def state_dict(self):
        return self.trainer.optimizer_state_dict()

    def load_state_dict(self, sd):
        self.trainer.load_optimizer_state_dict(sd)


class TrainCommand(AbstractCommand):
    def __init__(self):
        super().__init__()

    def register_subcommand(self, subparsers: argparse._SubParsersAction):
        sp = subparsers.add_parser('train', help='Train a model on the AddBiomechanics dataset')
        sp.add_argument('--dataset-home', type=str, default='../data', help='The path to the AddBiomechanics dataset.')
        sp.add_argument('--no-wandb', action='store_true', default=False, help='Log this run to Weights and Biases.')
        sp.add_argument('--model-type', type=str, default='feedforward', choices=['feedforward', 'groundlink', 'diffusion'],
                        help='The model to train.')
        sp.add_argument('--output-data-format', type=str, default='all_frames', choices=['all_frames', 'last_frame'],
                        help='Output for all frames in a window or only the last frame.')
        sp.add_argument('--checkpoint-dir', type=str, default='../checkpoints',
                        help='The path to a model checkpoint to save during training. Also, starts from the latest '
                             'checkpoint in this directory.')
        sp.add_argument('--geometry-folder', type=str, default=None, help='Path to the Geometry folder with bone mesh data.')
        sp.add_argument('--history-len', type=int, default=50,
                        help='The number of timesteps of context to show when constructing the inputs.')
        sp.add_argument('--stride', type=int, default=5,
                        help='The timestep gap between frames in the context window to be used when constructing the inputs.')
        sp.add_argument('--learning-rate', type=float, default=1e-4, help='The learning rate for weight updates.')
        sp.add_argument('--dropout', action='store_true', help='Apply dropout?')
        sp.add_argument('--dropout-prob', type=float, default=0.5, help='Dropout prob')
        sp.add_argument('--hidden-dims', type=int, nargs='+', default=[512, 512], help='Hidden dims across different layers.')
        sp.add_argument('--batchnorm', action='store_true', help='Apply batchnorm?')
        sp.add_argument('--activation', type=str, default='sigmoid', help='Which activation func?')
        sp.add_argument('--epochs', type=int, default=10, help='The number of epochs to run training for.')
        sp.add_argument('--opt-type', type=str, default='rmsprop',
                        help='The optimizer to use when adapting the weights of the model during training.')
        sp.add_argument('--batch-size', type=int, default=64, help='The batch size to use when training the model.')
        sp.add_argument('--short', action='store_true', help='Use very short datasets to test without loading a bunch of data.')
        sp.add_argument('--data-loading-workers', type=int, default=1,
                        help='Accepted for compatibility; windows are gathered from HBM, there are no loader processes.')
        sp.add_argument('--predict-grf-components', type=int, nargs='+', default=[i for i in range(6)], help='Which grf components to train.')
        sp.add_argument('--predict-cop-components', type=int, nargs='+', default=[i for i in range(6)], help='Which cop components to train.')
        sp.add_argument('--predict-moment-components', type=int, nargs='+', default=[i for i in range(6)], help='Which moment components to train.')
        sp.add_argument('--predict-wrench-components', type=int, nargs='+', default=[i for i in range(12)], help='Which wrench components to train.')
        sp.add_argument('--trial-filter', type=str, nargs='+', default=[""], help='What kind of trials to train/test on.')
        sp.add_argument('--compute-report', action='store_true', default=False,
                        help='Compute inverse dynamics reports during loss evaluation (needs nimblephysics: not on this path).')
        # additions of the B200 path
        sp.add_argument('--synthetic-windows', type=int, default=0,
                        help='Train on this many synthetic AddBiomechanics-shaped windows instead of <dataset-home>/*.ibmstore.')
        sp.add_argument('--max-batches', type=int, default=0, help='Stop every epoch after this many batches (0 = all).')
        sp.add_argument('--dev-sampling-steps', type=int, default=0,
                        help='--model-type diffusion: score the dev set before each epoch on samples of this many DDIM steps '
                             '(eta = 0); 0 skips the dev pass of the denoiser.')
        sp.add_argument('--ema-decay', type=float, default=0.0,
                        help='Keep an exponential moving average of the weights with this decay (e.g. 0.999; warm-up '
                             'min(decay, (1 + n) / (10 + n)) at step n), evaluate the dev set with it and save it in the '
                             'checkpoints as ema_state_dict; 0 keeps none.')
        sp.add_argument('--clip-grad-norm', type=float, default=0.0,
                        help='Scale the gradient down to this global L2 norm when it is larger (torch.nn.utils.clip_grad_norm_); '
                             'each training report adds the mean pre-clip norm and the number of clipped steps. 0 = off.')
        sp.add_argument('--lr-warmup-steps', type=int, default=0,
                        help='Raise the learning rate linearly from lr / W to lr over the first W optimizer steps (0 = off).')
        sp.add_argument('--lr-schedule', type=str, default='constant', choices=list(LR_SCHEDULES),
                        help='Learning rate after the warm-up: constant, or a cosine decay to --lr-min at the last step of '
                             'the run (epochs x batches per epoch).')
        sp.add_argument('--lr-min', type=float, default=0.0, help='Final learning rate of the cosine schedule.')
        sp.add_argument('--cond-drop-prob', type=float, default=0.0,
                        help='--model-type diffusion: replace the kinematics of this fraction of the windows of every step by '
                             'zeros (e.g. 0.1, as MDM), so the denoiser also learns the unconditional prediction that '
                             'analyze --guidance-scale needs; recorded in the checkpoints. 0 = off.')

    def run(self, args: argparse.Namespace):
        if 'command' in args and args.command != 'train':
            return False
        if args.compute_report:
            raise NotImplementedError("--compute-report needs nimblephysics inverse dynamics (RegressionLossEvaluator.py:265-286)")
        if args.dev_sampling_steps < 0:
            raise ValueError(f"--dev-sampling-steps must be >= 0, got {args.dev_sampling_steps}")
        if not 0.0 <= args.ema_decay < 1.0:
            raise ValueError(f"--ema-decay must be in [0, 1), got {args.ema_decay}")
        # the cosine's length (epochs x batches per epoch) is checked once the training store is open
        check_clip_sched(args.learning_rate, args.clip_grad_norm, args.lr_warmup_steps, 'constant', args.lr_min, None, flag='--')
        check_cond_drop(args.cond_drop_prob, args.model_type == 'diffusion', flag='--')
        model_type: str = args.model_type
        checkpoint_dir: str = os.path.join(os.path.abspath(args.checkpoint_dir), model_type)
        root_history_len = 10
        log_to_wandb: bool = not args.no_wandb
        rank, world, local = parallel.init_from_env("nccl")
        torch.cuda.set_device(local)
        device = torch.device("cuda", local)
        print(f"Running on {world} GPUs.")
        print(f"Current device being used for model training and loss evaluation: {local}.")
        if log_to_wandb:
            import wandb
            wandb.init(project="addbiomechanics-baseline", config=dict(args.__dict__),
                       group=os.getenv('WANDB_RUN_GROUP', f'ddp_{wandb.util.generate_id()}'))

        print("Initializing training set...")
        train_store = _data.open_split(args, 'train', model_type, device, seed=1234)
        print("Initializing dev set...")
        dev_store = _data.open_split(args, DEV, model_type, device, seed=4321)

        print("Initializing model...")
        torch.manual_seed(0)
        model = self.get_model(_data.NUM_DOFS, 2, model_type, history_len=args.history_len, stride=args.stride,
                               hidden_dims=args.hidden_dims, activation=args.activation, batchnorm=args.batchnorm,
                               dropout=args.dropout, dropout_prob=args.dropout_prob, root_history_len=root_history_len,
                               output_data_format=args.output_data_format, device=str(device)).to(device)
        if args.opt_type not in ('adagrad', 'adam', 'sgd', 'rmsprop', 'adadelta', 'adamax'):
            logging.error('Invalid optimizer type: ' + args.opt_type)
            assert (False)

        train_batches = WindowStore.batches(train_store.shard(rank, world), args.batch_size)
        dev_batches = WindowStore.batches(dev_store.shard(rank, world), args.batch_size)
        if args.max_batches:
            train_batches, dev_batches = train_batches[:args.max_batches], dev_batches[:args.max_batches]

        native = model_type in ('feedforward', 'groundlink', 'diffusion')
        if native:
            # every rank holds an equal-sized shard, so every rank runs the same number of steps
            total_steps = args.epochs * len(train_batches) if args.lr_schedule == 'cosine' else None
            if total_steps is not None and total_steps <= args.lr_warmup_steps:
                raise ValueError(f"--lr-schedule cosine needs more steps than --lr-warmup-steps ({args.lr_warmup_steps}); "
                                 f"the run has {total_steps} ({args.epochs} epochs x {len(train_batches)} batches)")
            trainer = Trainer(model, opt_type=args.opt_type, lr=args.learning_rate, args=args, seed=1234, ema_decay=args.ema_decay,
                              clip_grad_norm=args.clip_grad_norm, lr_warmup_steps=args.lr_warmup_steps,
                              lr_schedule=args.lr_schedule, lr_min=args.lr_min, total_steps=total_steps,
                              cond_drop_prob=args.cond_drop_prob)
            optimizer = None
        else:
            if world > 1:
                model = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], output_device=local)
            optimizer = getattr(torch.optim, {'adagrad': 'Adagrad', 'adam': 'Adam', 'sgd': 'SGD', 'rmsprop': 'RMSprop',
                                              'adadelta': 'Adadelta', 'adamax': 'Adamax'}[args.opt_type])(model.parameters(),
                                                                                                       lr=args.learning_rate)
        # the native trainer exposes load_state_dict/state_dict in torch.optim's layout, so the same call restores it
        epoch_checkpoint, _ = self.load_latest_checkpoint(model, checkpoint_dir=checkpoint_dir,
                                                          optimizer=_TrainerOptimizer(trainer) if native else optimizer)
        if native and epoch_checkpoint >= 0:
            trainer.arena.sync_shadow(force=True)        # parameters were replaced under the engine
            if trainer.ema is not None:
                # the average resumes from the checkpoint, or starts at the loaded weights if that run kept none
                ck = torch.load(self.latest_checkpoint_path(checkpoint_dir), map_location="cpu")
                trainer.load_ema_state_dict(ck.get('ema_state_dict'))
        use_ema = native and trainer.ema is not None
        clipping = native and args.clip_grad_norm > 0

        train_log, dev_log = _ResultLog('train'), _ResultLog(DEV)
        train_ev, dev_ev = RegressionLossEvaluator(None, 'train', device=device), RegressionLossEvaluator(None, DEV, device=device)
        # the denoiser is evaluated by reverse sampling, as in analyze: a few DDIM steps per dev batch, or no dev pass
        dev_diffusion = GaussianDiffusion(device=device) if model_type == 'diffusion' and args.dev_sampling_steps else None

        for epoch in range(epoch_checkpoint + 1, args.epochs):
            print(f'[{rank=}] Evaluating Dev Set Before Epoch {epoch}')
            with torch.no_grad(), (trainer.ema_weights() if use_ema else contextlib.nullcontext()):
                model.eval()
                if model_type != 'diffusion' or dev_diffusion is not None:
                    for i, idx in enumerate(dev_batches):
                        if dev_diffusion is not None:
                            sample_and_score(dev_diffusion, model, dev_store, idx, dev_log.ev, args, 1234 + rank,
                                             ddim_steps=args.dev_sampling_steps)
                        elif native:
                            dev_log.add(trainer.eval_step(dev_store, idx))
                        else:
                            inputs = input_dict(dev_store, idx, model_type, args.stride, root_history_len)
                            dev_ev(inputs, model(inputs), label_dict(dev_store, idx), [], [], args)
                        if (i + 1) % 100 == 0 or i == len(dev_batches) - 1:
                            print('  - Dev Batch ' + str(i + 1) + '/' + str(len(dev_batches)))
                print(f'[{rank=}] Dev Set Evaluation' + (' (EMA weights)' if use_ema else '') + ': ')
                print_all_ranks_report(dev_log.ev if native else dev_ev, args, rank, world, device)
                (dev_log if native else dev_ev).print_report(args, log_to_wandb=log_to_wandb)
            if world > 1:
                dist.barrier()
            print(f'[{rank=}] Running Training Epoch {epoch}')
            model.train()
            for i, idx in enumerate(train_batches):
                if native:
                    train_log.add(trainer.train_step(train_store, idx))
                else:
                    optimizer.zero_grad()
                    inputs = input_dict(train_store, idx, model_type, args.stride, root_history_len)
                    loss = train_ev(inputs, model(inputs), label_dict(train_store, idx), [], [], args,
                                    log_reports_to_wandb=log_to_wandb)
                    loss.backward()
                    optimizer.step()
                if (i + 1) % 100 == 0 or i == len(train_batches) - 1:
                    logging.info(f'  - [{rank=}] Batch ' + str(i + 1) + '/' + str(len(train_batches)))
                if (i + 1) % 1000 == 0 or i == len(train_batches) - 1:
                    logging.info(f'[{rank=}] Batch {i} Training Set Evaluation: ')
                    (train_log if native else train_ev).print_report(args, reset=False)
                    if clipping:
                        st = trainer.grad_norm_stats()
                        print(f'[{rank=}] Gradient norm before clipping: mean {st["mean_norm"]:.6g} over {st["steps"]} steps, '
                              f'{st["clipped"]} clipped (max norm {args.clip_grad_norm:g})')
                    if rank == 0:                              # avoid redundant saving across processes
                        model_path = f"{checkpoint_dir}/epoch_{epoch}_batch_{i}.pt"
                        os.makedirs(os.path.dirname(model_path), exist_ok=True)
                        ck = {'epoch': epoch, 'model_state_dict': model.state_dict(),
                              'optimizer_state_dict': optimizer.state_dict() if optimizer is not None else
                              trainer.optimizer_state_dict()}
                        if use_ema:
                            ck['ema_state_dict'] = trainer.ema_state_dict()
                        torch.save(ck, model_path)
            logging.info('-' * 80)
            logging.info(f'[{rank=}] Epoch {epoch}/{args.epochs} Training Set Evaluation: ')
            logging.info('-' * 80)
            print_all_ranks_report(train_log.ev if native else train_ev, args, rank, world, device)
            (train_log if native else train_ev).print_report(args, log_to_wandb=log_to_wandb)
            logging.info('-' * 80)

        if log_to_wandb:
            import wandb
            wandb.finish()
        if dist.is_initialized():
            dist.destroy_process_group()
        return True
