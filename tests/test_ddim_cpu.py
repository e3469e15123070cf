"""DDIM sampling schedule (no GPU): the library's per-timestep tables (``diffusion.ddim_schedule``) against the eps-form
DDIM oracle (``tests/ddim_oracle.py``), their identity with the DDPM posterior tables over the full sequence, the
timestep sequence, and the argument checks of the sampler and the analyze command."""
import argparse

import numpy as np
import pytest
import torch

import ddim_oracle as odim
from inferbiomechanics_b200.diffusion import GaussianDiffusion, ddim_schedule

T = 1000


@pytest.mark.parametrize("eta", [0.0, 0.5, 1.0])
@pytest.mark.parametrize("S", [1, 2, 7, 50, T])
def test_tables_reproduce_eps_form_oracle(S, eta):
    tab = ddim_schedule(S, eta)
    ab = odim.abar(T)
    ts = odim.ddim_timesteps(T, S)
    np.testing.assert_array_equal(tab["ts"], ts)
    g = torch.Generator().manual_seed(S)
    for i, t in enumerate(ts.tolist()):
        p = int(ts[i + 1]) if i + 1 < S else -1
        assert tab["succ"][t] == p
        x0, xt, z = (torch.randn(64, 30, generator=g, dtype=torch.float64) for _ in range(3))
        want = odim.ddim_step(ab, x0, xt, t, p, eta, z)
        c0, ct, sg = (float(tab[k][t]) for k in ("coef_x0", "coef_xt", "sigma"))
        got = c0 * x0 + ct * xt + (sg * z if t > 0 else 0.0)
        # each fp32 table entry carries at most half an ulp (2^-24 relative) of rounding
        bound = 2.0 ** -23 * (abs(c0) * x0.abs() + ct * xt.abs() + sg * z.abs()) + 1e-300
        assert ((got - want).abs() <= bound).all(), (S, eta, t, ((got - want).abs() / bound).max().item())


@pytest.mark.parametrize("num_timesteps", [12, 20, 1000])
def test_full_sequence_at_eta_one_is_the_ddpm_chain_bit_for_bit(num_timesteps):
    tab = ddim_schedule(num_timesteps, 1.0, num_timesteps)
    gd = GaussianDiffusion(num_timesteps=num_timesteps, device="cpu")
    np.testing.assert_array_equal(tab["ts"], np.arange(num_timesteps - 1, -1, -1))
    np.testing.assert_array_equal(tab["succ"], np.arange(num_timesteps) - 1)
    np.testing.assert_array_equal(tab["coef_x0"], gd.coef_x0.numpy())
    np.testing.assert_array_equal(tab["coef_xt"], gd.coef_xt.numpy())
    np.testing.assert_array_equal(tab["sigma"][1:], gd.sigma.numpy()[1:])      # the step at t = 0 draws no noise in either
    assert (tab["coef_x0"][0], tab["coef_xt"][0]) == (1.0, 0.0)


def test_timestep_sequences():
    for S in range(1, T + 1):
        ts = ddim_schedule(S, 0.0)["ts"]
        assert len(ts) == S and ts[0] == T - 1 and (np.diff(ts) < 0).all(), S
        if S >= 2:
            assert ts[-1] == 0, S


def test_single_step_returns_x0_hat():
    tab = ddim_schedule(1, 1.0)
    assert tab["ts"].tolist() == [T - 1] and tab["succ"][T - 1] == -1
    assert (tab["coef_x0"][T - 1], tab["coef_xt"][T - 1], tab["sigma"][T - 1]) == (1.0, 0.0, 0.0)
    assert not tab["coef_x0"][:T - 1].any() and not tab["coef_xt"][:T - 1].any()


@pytest.mark.parametrize("S", [1, 7, 50, T])
def test_eta_zero_draws_no_noise(S):
    tab = ddim_schedule(S, 0.0)
    assert not tab["sigma"].any()
    assert tab["sigma"].dtype == np.float32 and tab["succ"].dtype == np.int32


@pytest.mark.parametrize("kw", [dict(steps=10, ddim_steps=10), dict(ddim_steps=0), dict(ddim_steps=T + 1),
                                dict(ddim_steps=10, eta=-0.1), dict(ddim_steps=10, eta=1.5), dict(eta=0.5),
                                dict(steps=10, eta=0.5)])
def test_sampler_rejects_bad_schedules(kw):
    gd = GaussianDiffusion(device="cpu")
    with pytest.raises(ValueError):
        gd.sample(None, 4, **kw)                  # rejected before the model is touched
    with pytest.raises(ValueError):
        gd.sample_windows(None, torch.zeros(4, 10, 177), **kw)
    if "ddim_steps" in kw and "steps" not in kw:
        with pytest.raises(ValueError):
            ddim_schedule(kw["ddim_steps"], kw.get("eta", 0.0))


def test_analyze_sampler_flags():
    from inferbiomechanics_b200.cli.analyze import AnalyzeCommand
    from inferbiomechanics_b200.cli.train import TrainCommand
    p = argparse.ArgumentParser()
    sub = p.add_subparsers(dest="command")
    an = AnalyzeCommand()
    for c in (TrainCommand(), an):
        c.register_subcommand(sub)
    a = p.parse_args(["analyze"])
    assert (a.sampler, a.eta, a.sampling_steps) == ("ddpm", 0.0, 1000)
    a = p.parse_args("analyze --model-type diffusion --sampler ddim --sampling-steps 50 --eta 0.3".split())
    assert (a.sampler, a.eta, a.sampling_steps) == ("ddim", 0.3, 50)
    with pytest.raises(SystemExit):
        p.parse_args("analyze --sampler ddpmx".split())
    with pytest.raises(ValueError, match="--eta"):
        an.run(p.parse_args("analyze --model-type diffusion --sampler ddpm --eta 0.5".split()))
    assert p.parse_args(["train"]).dev_sampling_steps == 0
