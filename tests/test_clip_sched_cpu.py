"""Gradient clipping and learning-rate schedule surface without a GPU: the host schedule against torch's LambdaLR driving a
real SGD, the Trainer's and the train command's argument checks, the parser's defaults, and the optimizer checkpoint's
param_groups with the options off and on."""
import argparse
import math
from types import SimpleNamespace

import pytest
import torch


def _parser():
    from inferbiomechanics_b200.cli.train import TrainCommand
    p = argparse.ArgumentParser()
    sub = p.add_subparsers(dest="command")
    TrainCommand().register_subcommand(sub)
    return p


def _lam(n, W, cosine, S, r):
    """The schedule as the feature defines it, written out independently of the package."""
    if W > 0 and n <= W:
        return n / W
    if not cosine:
        return 1.0
    p = min(max((n - W) / (S - W), 0.0), 1.0)
    return r + (1 - r) * 0.5 * (1 + math.cos(math.pi * p))


@pytest.mark.parametrize("W,schedule,lr_min", [(10, "constant", 0.0), (10, "cosine", 0.0), (0, "cosine", 0.0),
                                               (10, "cosine", 2e-4)])
def test_host_schedule_equals_lambda_lr_on_a_real_optimizer(W, schedule, lr_min):
    """The n-th ``opt.step()`` under ``LambdaLR(opt, lambda s: lam(s + 1))`` runs at the rate the Trainer reports for its n-th
    step (``current_lr`` with n - 1 steps taken), over 3 W + 20 steps: the warm-up, the cosine to S = 2 W + 20 and the
    clamped tail after S."""
    from inferbiomechanics_b200.trainer import Trainer, lr_lambda
    lr, steps = 1e-3, 3 * W + 20
    S = 2 * W + 20 if schedule == "cosine" else 0
    p = torch.nn.Parameter(torch.zeros(3))
    opt = torch.optim.SGD([p], lr=lr)
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda s: _lam(s + 1, W, schedule == "cosine", S, lr_min / lr))
    tr = SimpleNamespace(scheduled=True, lr=lr, lr_warmup_steps=W, lr_schedule=schedule, total_steps=S, lr_min=lr_min)
    seen = []
    for n in range(1, steps + 1):
        tr.step_count = n - 1
        used = opt.param_groups[0]["lr"]
        assert Trainer.current_lr(tr) == pytest.approx(used, rel=1e-12, abs=0.0), n
        assert lr * lr_lambda(n, W, schedule, S, lr_min / lr) == pytest.approx(used, rel=1e-12, abs=0.0), n
        seen.append(used)
        p.grad = torch.ones(3)
        opt.step()
        sched.step()
    if W:
        assert seen[0] == pytest.approx(lr / W) and seen[W - 1] == pytest.approx(lr)
    if schedule == "cosine":
        assert seen[S - 1] == pytest.approx(lr_min, abs=1e-15) and seen[-1] == pytest.approx(lr_min, abs=1e-15)
        assert all(a >= b for a, b in zip(seen[W:], seen[W + 1:]))
    else:
        assert all(v == lr for v in seen[W:])


@pytest.mark.parametrize("kw,match", [({"clip_grad_norm": -1.0}, "clip_grad_norm"), ({"clip_grad_norm": float("nan")}, "clip_grad_norm"),
                                      ({"lr_warmup_steps": -1}, "lr_warmup_steps"), ({"lr_schedule": "step"}, "lr_schedule"),
                                      ({"lr_schedule": "cosine"}, "total_steps"),
                                      ({"lr_schedule": "cosine", "lr_warmup_steps": 10, "total_steps": 10}, "total_steps"),
                                      ({"lr_min": -1e-5}, "lr_min"), ({"lr_min": 2e-3}, "lr_min"), ({"total_steps": -3}, "total_steps")])
def test_trainer_rejects_bad_clip_and_schedule_settings(kw, match):
    from inferbiomechanics_b200.trainer import Trainer
    with pytest.raises(ValueError, match=match):
        Trainer(None, lr=1e-3, **kw)


def test_clip_and_schedule_flags_parse_with_defaults_off():
    a = _parser().parse_args(["train"])
    assert (a.clip_grad_norm, a.lr_warmup_steps, a.lr_schedule, a.lr_min) == (0.0, 0, "constant", 0.0)
    a = _parser().parse_args(["train", "--clip-grad-norm", "1", "--lr-warmup-steps", "1000", "--lr-schedule", "cosine",
                              "--lr-min", "1e-6"])
    assert (a.clip_grad_norm, a.lr_warmup_steps, a.lr_schedule, a.lr_min) == (1.0, 1000, "cosine", 1e-6)
    with pytest.raises(SystemExit):
        _parser().parse_args(["train", "--lr-schedule", "linear"])


@pytest.mark.parametrize("flags,match", [(["--clip-grad-norm", "-1"], "--clip-grad-norm"),
                                         (["--lr-warmup-steps", "-5"], "--lr-warmup-steps"),
                                         (["--lr-min", "-1"], "--lr-min"),
                                         (["--learning-rate", "1e-4", "--lr-min", "1e-3"], "--lr-min")])
def test_train_rejects_bad_clip_and_schedule_flags_before_gpu(flags, match):
    from inferbiomechanics_b200.cli.train import TrainCommand
    args = _parser().parse_args(["train", "--no-wandb", *flags])
    with pytest.raises(ValueError, match=match):
        TrainCommand().run(args)


def _stub_trainer(opt_type, **kw):
    """A Trainer's checkpoint surface on CPU tensors: the attributes optimizer_state_dict reads."""
    from inferbiomechanics_b200.trainer import Trainer
    tr = object.__new__(Trainer)
    params = [torch.nn.Parameter(torch.zeros(4, 3)), torch.nn.Parameter(torch.zeros(3))]
    tr.arena = SimpleNamespace(params=params, names=["w", "b"], offsets={"w": (0, 12), "b": (16, 3)})
    tr.opt_type, tr.lr, tr.step_count = opt_type, 1e-3, 0
    tr.state0, tr.state1 = torch.zeros(19), torch.zeros(19)
    tr.clip_grad_norm = kw.get("clip_grad_norm", 0.0)
    tr.lr_warmup_steps, tr.lr_schedule = kw.get("lr_warmup_steps", 0), kw.get("lr_schedule", "constant")
    tr.lr_min, tr.total_steps = kw.get("lr_min", 0.0), kw.get("total_steps", 0)
    tr.scheduled = tr.lr_warmup_steps > 0 or tr.lr_schedule != "constant"
    tr._clip_ws = object() if tr.clip_grad_norm > 0 else None
    return tr, params


@pytest.mark.parametrize("opt_type", ["rmsprop", "adam", "sgd"])
def test_checkpoint_param_groups_unchanged_with_options_off(opt_type):
    from inferbiomechanics_b200.trainer import Trainer
    tr, params = _stub_trainer(opt_type)
    sd = tr.optimizer_state_dict()
    ref = getattr(torch.optim, Trainer._OPT_CLASS[opt_type])(params, lr=1e-3).state_dict()
    assert sd["param_groups"] == ref["param_groups"]
    assert sd["ibm_b200"] == {"opt_type": opt_type, "step": 0}


def test_checkpoint_records_schedule_like_lambda_lr():
    """With a schedule, param_groups[0] holds the next step's rate as ``lr`` and the base rate as ``initial_lr``, what
    torch's group holds after ``opt.step(); sched.step()``; the ibm_b200 tag records the settings."""
    tr, params = _stub_trainer("adam", clip_grad_norm=1.0, lr_warmup_steps=4, lr_schedule="cosine", total_steps=10, lr_min=1e-4)
    opt = torch.optim.Adam(params, lr=1e-3)
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda s: _lam(s + 1, 4, True, 10, 0.1))
    for n in range(6):
        sd = tr.optimizer_state_dict()
        assert sd["param_groups"][0]["lr"] == pytest.approx(opt.param_groups[0]["lr"], rel=1e-12)
        assert sd["param_groups"][0]["initial_lr"] == opt.param_groups[0]["initial_lr"] == 1e-3
        tr.step_count += 1
        for p in params:
            p.grad = torch.zeros_like(p)
        opt.step()
        sched.step()
    assert sd["ibm_b200"] == {"opt_type": "adam", "step": 5, "clip_grad_norm": 1.0, "lr_warmup_steps": 4, "lr_schedule": "cosine",
                              "lr_min": 1e-4, "total_steps": 10}
