"""DPM-Solver++(2M) sampling schedule (no GPU): the timestep rule, the library's tables (``diffusion.dpm_schedule``) against
the exp / lambda-form oracle (``tests/dpm_oracle.py``) and against DDIM's on the first-order steps, the convergence order
against the exact probability-flow solution of an analytic denoiser, and the argument checks of the sampler and the analyze
command."""
import argparse

import numpy as np
import pytest
import torch

import ddim_oracle as odim
import dpm_oracle as odpm
from inferbiomechanics_b200.diffusion import GaussianDiffusion, ddim_schedule, dpm_schedule, dpm_timesteps

T = 1000


def test_timestep_rule_for_every_step_count():
    ab = odim.abar(T)
    for S in range(1, T + 1):
        ts = dpm_timesteps(S, ab)
        assert len(ts) == S and len(set(ts.tolist())) == S, S
        assert ts[0] == T - 1 and ts[-1] == (0 if S >= 2 else T - 1) and (np.diff(ts) < 0).all(), S
        if S in (1, 2, 3, 10, 20, 57, 100, 999, T):
            np.testing.assert_array_equal(ts, odpm.dpm_timesteps(T, S, ab))
    assert dpm_timesteps(2, ab).tolist() == [999, 0]
    assert dpm_timesteps(10, ab).tolist() == [999, 886, 757, 603, 410, 202, 73, 22, 5, 0]
    np.testing.assert_array_equal(dpm_timesteps(T, ab), np.arange(T - 1, -1, -1))


@pytest.mark.parametrize("S", [1, 2, 3, 10, 20, 57, T])
def test_tables_match_the_exp_lambda_oracle(S):
    tab = dpm_schedule(S)
    ab = odim.abar(T)
    ts = odpm.dpm_timesteps(T, S, ab)
    np.testing.assert_array_equal(tab["ts"], ts)
    on = np.zeros(T, dtype=bool)
    on[ts] = True
    for k in ("coef_x0", "coef_xt", "coef_prev"):
        assert tab[k].dtype == np.float32 and not tab[k][~on].any(), k
    assert tab["succ"].dtype == np.int32
    for i, t in enumerate(ts.tolist()):
        assert tab["succ"][t] == (ts[i + 1] if i + 1 < S else -1)
        want = odpm.step_coefs(ab, ts, i)
        got = (tab["coef_x0"][t], tab["coef_prev"][t], tab["coef_xt"][t])
        np.testing.assert_allclose(np.array(got, dtype=np.float64), np.array(want), rtol=1e-6, atol=0, err_msg=f"S={S} i={i}")


@pytest.mark.parametrize("S", [2, 3, 10, 20, 57, T])
def test_first_and_last_steps_are_ddim_eta_zero_bit_for_bit(S):
    tab = dpm_schedule(S)
    ab = odim.abar(T)
    ts = tab["ts"]
    for i in (0, S - 1):
        t, p = int(ts[i]), (int(ts[i + 1]) if i + 1 < S else -1)
        # DDIM-eta-0's formula for the same (t, p), as ddim_schedule evaluates it
        a_t, a_p = ab[t], (ab[p] if p >= 0 else 1.0)
        c = np.sqrt(max(1.0 - a_p, 0.0))
        assert tab["coef_x0"][t] == np.float32(np.sqrt(a_p) - c * np.sqrt(a_t) / np.sqrt(1.0 - a_t)), (S, i)
        assert tab["coef_xt"][t] == np.float32(c / np.sqrt(1.0 - a_t)), (S, i)
        assert tab["coef_prev"][t] == 0.0, (S, i)
    assert (tab["coef_x0"][0], tab["coef_xt"][0], tab["coef_prev"][0]) == (1.0, 0.0, 0.0)
    if S > 2:
        assert (tab["coef_prev"][ts[1:-1]] != 0).all()


@pytest.mark.parametrize("S", [1, 2])
def test_one_and_two_steps_are_the_ddim_tables(S):
    dpm, ddim = dpm_schedule(S), ddim_schedule(S, 0.0)
    for k in ("coef_x0", "coef_xt", "succ", "ts"):
        np.testing.assert_array_equal(dpm[k], ddim[k])
    assert not dpm["coef_prev"].any()


# ---------------------------------------- convergence ----------------------------------------------------------------
MU, SD = 0.3, 0.5                       # Gaussian data x0 ~ N(MU, SD^2) per element: x0_hat and the flow are closed-form


def _x0_hat(ab, x, t):
    a = ab[t]
    return MU + np.sqrt(a) * SD * SD / (a * SD * SD + 1.0 - a) * (x - np.sqrt(a) * MU)


def _exact(ab, x_T):
    """The probability-flow ODE solution at t = 0 from x_T: xi = (x - sqrt(a) MU) / sqrt(a SD^2 + 1 - a) is constant along it."""
    s = lambda t: np.sqrt(ab[t] * SD * SD + 1.0 - ab[t])
    xi = (x_T - np.sqrt(ab[T - 1]) * MU) / s(T - 1)
    return _x0_hat(ab, np.sqrt(ab[0]) * MU + s(0) * xi, 0)


def _run(tab, x_T, ab):
    """The library's tables in an fp64 loop."""
    x, prev = x_T.copy(), None
    for t in tab["ts"].tolist():
        d = _x0_hat(ab, x, t)
        cp = float(tab.get("coef_prev", np.zeros(T))[t])
        x = float(tab["coef_x0"][t]) * d + float(tab["coef_xt"][t]) * x + (cp * prev if cp != 0.0 else 0.0)
        prev = d
    return x


def test_second_order_convergence_on_an_analytic_denoiser():
    ab = odim.abar(T)
    x_T = np.random.default_rng(0).standard_normal(200_000)
    ref = _exact(ab, x_T)
    err = lambda tab: np.abs(_run(tab, x_T, ab) - ref).max()
    dpm = {S: err(dpm_schedule(S)) for S in (20, 25, 50, 100)}
    ddim = {S: err(ddim_schedule(S, 0.0)) for S in (20, 25, 50, 100)}
    for lo, hi in ((25, 50), (50, 100)):
        assert dpm[lo] / dpm[hi] >= 3.5, (lo, dpm)
        assert ddim[lo] / ddim[hi] <= 2.2, (lo, ddim)
    assert dpm[20] <= ddim[20] / 5, (dpm[20], ddim[20])
    assert dpm[20] < ddim[100]


def test_oracle_loop_agrees_with_the_tables():
    ab = odim.abar(T)
    x_T = torch.from_numpy(np.random.default_rng(1).standard_normal(4096))
    for S in (3, 10, 20):
        want = odpm.dpm_sample_loop(ab, lambda x, t: torch.from_numpy(_x0_hat(ab, x.double().numpy(), t)), x_T.float(), S)
        got = _run(dpm_schedule(S), x_T.float().double().numpy(), ab)
        np.testing.assert_allclose(want.double().numpy(), got, rtol=0, atol=1e-5)


# ---------------------------------------- refusals --------------------------------------------------------------------
@pytest.mark.parametrize("kw", [dict(dpm_steps=0), dict(dpm_steps=T + 1), dict(dpm_steps=2.5), dict(dpm_steps=10, ddim_steps=10),
                                dict(dpm_steps=10, steps=10), dict(dpm_steps=10, eta=0.5)])
def test_sampler_rejects_bad_dpm_schedules(kw):
    gd = GaussianDiffusion(device="cpu")
    with pytest.raises(ValueError):
        gd.sample(None, 4, **kw)                  # rejected before the model is touched
    with pytest.raises(ValueError):
        gd.sample_windows(None, torch.zeros(4, 10, 177), **kw)
    if set(kw) == {"dpm_steps"}:
        with pytest.raises(ValueError):
            dpm_schedule(kw["dpm_steps"])


def test_sampler_rejects_supplied_noise_with_dpm():
    gd = GaussianDiffusion(device="cpu")
    with pytest.raises(ValueError, match="noise"):
        gd.sample(None, 4, dpm_steps=10, noise=lambda t: None)


def _parser():
    from inferbiomechanics_b200.cli.analyze import AnalyzeCommand
    from inferbiomechanics_b200.cli.train import TrainCommand
    p = argparse.ArgumentParser()
    sub = p.add_subparsers(dest="command")
    an = AnalyzeCommand()
    for c in (TrainCommand(), an):
        c.register_subcommand(sub)
    return p, an


def test_analyze_dpm_sampler_flags():
    p, an = _parser()
    a = p.parse_args("analyze --model-type diffusion --sampler dpmpp2m --sampling-steps 20".split())
    assert (a.sampler, a.eta, a.sampling_steps) == ("dpmpp2m", 0.0, 20)
    with pytest.raises(ValueError, match="--eta"):
        an.run(p.parse_args("analyze --model-type diffusion --sampler dpmpp2m --eta 0.5".split()))
