"""Classifier-free guidance surface without a GPU: the argument checks of the Trainer, the sampler and both commands (before
any device work), the parser defaults, the optimizer checkpoint tag, the checkpoint check behind ``analyze
--guidance-scale``, and the guidance oracle itself."""
import argparse
import math
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import cfg_oracle as ocfg
import ddim_oracle as odim
import philox_oracle as ph
from oracle import ddpm as oddpm


def _parser():
    from inferbiomechanics_b200.cli.analyze import AnalyzeCommand
    from inferbiomechanics_b200.cli.train import TrainCommand
    p = argparse.ArgumentParser()
    sub = p.add_subparsers(dest="command")
    for c in (TrainCommand(), AnalyzeCommand()):
        c.register_subcommand(sub)
    return p


def test_guidance_flags_parse_with_defaults_off():
    assert _parser().parse_args(["train"]).cond_drop_prob == 0.0
    assert _parser().parse_args(["train", "--cond-drop-prob", "0.1"]).cond_drop_prob == 0.1
    assert _parser().parse_args(["analyze"]).guidance_scale == 1.0
    assert _parser().parse_args(["analyze", "--guidance-scale", "2.5"]).guidance_scale == 2.5


@pytest.mark.parametrize("p", [-0.1, 1.5, float("nan")])
def test_trainer_rejects_drop_probability_outside_unit_interval(p):
    from inferbiomechanics_b200.trainer import Trainer
    with pytest.raises(ValueError, match=r"cond_drop_prob must lie in \[0, 1\]"):
        Trainer(SimpleNamespace(trains_by_diffusion=True), cond_drop_prob=p)


@pytest.mark.parametrize("model", [None, SimpleNamespace(trains_by_diffusion=False)])
def test_trainer_rejects_drop_probability_without_diffusion(model):
    from inferbiomechanics_b200.trainer import Trainer
    with pytest.raises(ValueError, match="diffusion denoiser only"):
        Trainer(model, cond_drop_prob=0.1)


@pytest.mark.parametrize("flags,match", [(["--cond-drop-prob", "0.1", "--model-type", "feedforward"], "diffusion denoiser only"),
                                         (["--cond-drop-prob", "0.1", "--model-type", "groundlink"], "diffusion denoiser only"),
                                         (["--cond-drop-prob", "1.5", "--model-type", "diffusion"], "--cond-drop-prob"),
                                         (["--cond-drop-prob", "-1", "--model-type", "diffusion"], "--cond-drop-prob")])
def test_train_rejects_bad_drop_probability_before_gpu(flags, match):
    from inferbiomechanics_b200.cli.train import TrainCommand
    with pytest.raises(ValueError, match=match):
        TrainCommand().run(_parser().parse_args(["train", "--no-wandb", *flags]))


@pytest.mark.parametrize("scale", [-0.5, float("nan"), float("inf")])
def test_sampler_rejects_negative_or_non_finite_scale(scale):
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    gd = GaussianDiffusion(num_timesteps=20, device="cpu")
    with pytest.raises(ValueError, match="guidance_scale"):
        gd.sample(None, 4, guidance_scale=scale)
    with pytest.raises(ValueError, match="guidance_scale"):
        gd.sample(None, 4, ddim_steps=5, eta=1.0, guidance_scale=scale)
    with pytest.raises(ValueError, match="guidance_scale"):
        gd.sample_windows(None, torch.zeros(4, 10, 177), guidance_scale=scale)


def _checkpoint(root, tag):
    d = os.path.join(root, "diffusion")
    os.makedirs(d, exist_ok=True)
    path = os.path.join(d, "epoch_0_batch_3.pt")
    torch.save({"epoch": 0, "model_state_dict": {}, "optimizer_state_dict": {"state": {}, "param_groups": [], "ibm_b200": tag}}, path)
    return path


@pytest.mark.parametrize("flags,match", [(["--model-type", "feedforward", "--guidance-scale", "2"], "diffusion only"),
                                         (["--model-type", "diffusion", "--guidance-scale", "-1"], "guidance_scale"),
                                         (["--model-type", "diffusion", "--guidance-scale", "nan"], "guidance_scale")])
def test_analyze_rejects_bad_guidance_before_gpu(tmp_path, flags, match):
    from inferbiomechanics_b200.cli.analyze import AnalyzeCommand
    _checkpoint(str(tmp_path), {"opt_type": "rmsprop", "step": 4, "cond_drop_prob": 0.1})
    args = _parser().parse_args(["analyze", "--no-wandb", "--checkpoint-dir", str(tmp_path), *flags])
    with pytest.raises(ValueError, match=match):
        AnalyzeCommand().run(args)


def test_analyze_guidance_needs_a_checkpoint_trained_with_condition_dropout(tmp_path):
    from inferbiomechanics_b200.cli.analyze import AnalyzeCommand
    ck = str(tmp_path / "ck")
    args = _parser().parse_args(["analyze", "--no-wandb", "--checkpoint-dir", ck, "--model-type", "diffusion", "--guidance-scale", "2"])
    with pytest.raises(ValueError, match="holds none"):
        AnalyzeCommand().run(args)
    path = _checkpoint(ck, {"opt_type": "rmsprop", "step": 4})
    with pytest.raises(ValueError, match=f"{path} records none"):
        AnalyzeCommand().run(args)
    _checkpoint(ck, {"opt_type": "rmsprop", "step": 4, "cond_drop_prob": 0.1})
    AnalyzeCommand().check_guidance_checkpoint("diffusion", 2.0, os.path.join(ck, "diffusion"))


def _stub_trainer(**kw):
    """The attributes optimizer_state_dict reads, on CPU tensors."""
    from inferbiomechanics_b200.trainer import Trainer
    tr = object.__new__(Trainer)
    params = [torch.nn.Parameter(torch.zeros(4, 3)), torch.nn.Parameter(torch.zeros(3))]
    tr.arena = SimpleNamespace(params=params, names=["w", "b"], offsets={"w": (0, 12), "b": (16, 3)})
    tr.opt_type, tr.lr, tr.step_count = "rmsprop", 1e-3, 0
    tr.state0, tr.state1 = torch.zeros(19), None
    tr.scheduled, tr._clip_ws = False, None
    for k, v in kw.items():
        setattr(tr, k, v)
    return tr


def test_checkpoint_tag_records_the_drop_probability_only_when_on():
    assert _stub_trainer().optimizer_state_dict()["ibm_b200"] == {"opt_type": "rmsprop", "step": 0}
    sd = _stub_trainer(cond_drop_prob=0.1).optimizer_state_dict()
    assert sd["ibm_b200"] == {"opt_type": "rmsprop", "step": 0, "cond_drop_prob": 0.1}


def test_drop_mask_follows_the_dropout_keep_rule():
    B, p, seed, offset = 5000, 0.1, 1234, 77
    keep = ocfg.cond_keep(B, p, seed, offset)
    word0 = ph.philox_words(B, seed, offset)[:, 0]
    assert np.array_equal(~keep, word0 < np.uint32(ph.keep_threshold(p)))
    assert abs((~keep).mean() - p) < 0.02
    assert not ocfg.cond_keep(B, 1.0, seed, offset).any()
    assert not np.array_equal(keep, ocfg.cond_keep(B, p, seed, offset + 1))


@pytest.mark.parametrize("t", [0, 1, 500, 999])
def test_guided_oracle_at_scale_one_is_the_conditional_step(t):
    g = torch.Generator().manual_seed(t)
    c, u, x, z = (torch.randn(50, 30, generator=g) for _ in range(4))
    sched = oddpm.make_schedule()
    dsched = {k: v.double() for k, v in sched.items()}
    want_c = oddpm.posterior_step(dsched, c.double(), x.double(), t, z.double())
    want_u = oddpm.posterior_step(dsched, u.double(), x.double(), t, z.double())
    assert torch.equal(ocfg.guided_ddpm_step(sched, c, u, x, t, z, 1.0), want_c)
    assert torch.equal(ocfg.guided_ddpm_step(sched, c, u, x, t, z, 0.0), want_u)
    ab = odim.abar()
    p = max(t - 100, -1)
    for eta in (0.0, 1.0):
        assert torch.equal(ocfg.guided_ddim_step(ab, c, u, x, t, p, eta, z, 1.0), odim.ddim_step(ab, c, x, t, p, eta, z))
        assert torch.equal(ocfg.guided_ddim_step(ab, c, u, x, t, p, eta, z, 0.0), odim.ddim_step(ab, u, x, t, p, eta, z))
    s = 2.5
    assert torch.allclose(ocfg.guided_x0(c, u, s), c.double() + (s - 1) * (c.double() - u.double()), rtol=0, atol=1e-12)
    assert math.isclose(float(ocfg.guided_x0(torch.ones(1), torch.zeros(1), s)), s)
