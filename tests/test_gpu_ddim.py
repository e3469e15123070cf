"""Few-step DDIM sampling on a B200: the respaced step kernel against the eps-form oracle (``tests/ddim_oracle.py``,
builder-owned, parity unpinned like all diffusion code), the full sequence at eta = 1 against the DDPM chain bit for
bit, the sampler loop against the oracle loop, CUDA-graph replay against eager launches, and the CLI paths."""
import math
import re

import numpy as np
import pytest
import torch

import ddim_oracle as odim
from oracle import models as om
from test_gpu_models import _small_denoiser, close

pytestmark = pytest.mark.gpu


def _cond(m, B):
    """Random conditioning kinematics in the denoiser's concat buffer (columns 30…)."""
    eng = m.engine()
    eng.xc(B, False)[:, 30:30 + eng.c_in] = torch.randn(B * eng.F, eng.c_in, device="cuda",
                                                       generator=torch.Generator("cuda").manual_seed(B)).to(torch.bfloat16)


@pytest.mark.parametrize("eta", [0.0, 1.0])
@pytest.mark.parametrize("which", ["middle", "last"])
def test_respaced_step_kernel_matches_oracle(which, eta):
    from inferbiomechanics_b200 import ops
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    S, M = 7, 4000
    gd = GaussianDiffusion(device="cuda")
    tab = gd.ddim_tables(S, eta)
    ts = tab["ts"].tolist()
    i = 3 if which == "middle" else S - 1
    t, p = ts[i], (ts[i + 1] if i + 1 < S else -1)
    g = torch.Generator().manual_seed(11)
    x0h = torch.randn(M, 32, generator=g)                  # the head GEMM's 32-float rows
    xt, z = torch.randn(M, 30, generator=g), torch.randn(M, 30, generator=g)
    t_dev = torch.tensor([t], dtype=torch.int32, device="cuda")
    t_next = torch.full((1,), 12345, dtype=torch.int32, device="cuda")
    out = torch.empty(M, 30, device="cuda")
    ops.posterior_step(x0h.cuda(), 32, xt.cuda(), z.cuda(), t_dev, tab["coef_x0"], tab["coef_xt"], tab["sigma"], M, x_prev=out,
                       t_next=t_next, t_succ=tab["succ"])
    want = odim.ddim_step(odim.abar(), x0h[:, :30], xt, t, p, eta, z)
    torch.testing.assert_close(out.cpu().double(), want, rtol=2e-6, atol=1e-6)
    assert t_next.item() == p


@pytest.mark.parametrize("use_graph", [False, True])
def test_full_sequence_at_eta_one_equals_ddpm(use_graph):
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F = 8, 10
    m, _ = _small_denoiser(F=F, L=1)
    _cond(m, B)
    gd = GaussianDiffusion(num_timesteps=20, device="cuda")
    a = gd.sample(m, B, seed=5, use_graph=use_graph)
    b = gd.sample(m, B, seed=5, use_graph=use_graph, ddim_steps=20, eta=1.0)
    assert torch.isfinite(a).all()
    torch.testing.assert_close(b, a, rtol=0, atol=0)


@pytest.mark.parametrize("eta", [0.0, 1.0])
def test_sampling_loop_matches_oracle_with_supplied_noise(eta):
    from inferbiomechanics_b200 import ops
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F, S = 4, 10, 6
    m, sd = _small_denoiser(F=F, L=1)
    cond = torch.randn(B, F, 177, generator=torch.Generator().manual_seed(2))
    eng = m.engine()
    ops.pack_inputs([cond.reshape(B * F, 177).cuda()], B * F, F, out_bf16=eng.xc(B, False), frame_stride=eng.ld_in, win_extra=0,
                    col0=30)
    gd = GaussianDiffusion(device="cuda")
    g = torch.Generator().manual_seed(3)
    x_T = torch.randn(B, F, 30, generator=g)
    ts = odim.ddim_timesteps(1000, S).tolist()
    zs = {t: torch.randn(B * F, 30, generator=g) for t in ts}
    seen = []
    got = gd.sample(m, B, x_T=x_T.cuda(), noise=lambda t: seen.append(t) or zs[t].cuda(), ddim_steps=S, eta=eta)
    assert seen == ts
    with torch.no_grad():
        denoise = lambda x, t: om.denoiser_forward(sd, cond, x.view(B, F, 30), torch.full((B,), t), 1, 2).reshape(B * F, 30)
        want = odim.ddim_sample_loop(odim.abar(), denoise, x_T.reshape(B * F, 30), S, eta, lambda t: zs[t])
    close(got.reshape(B * F, 30), want, 5e-2, "trajectory")


def test_single_step_returns_x0_hat():
    from inferbiomechanics_b200 import ops
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F = 8, 10
    m, _ = _small_denoiser(F=F, L=1)
    _cond(m, B)
    eng = m.engine()
    gd = GaussianDiffusion(device="cuda")
    x_T = torch.randn(B, F, 30, device="cuda", generator=torch.Generator("cuda").manual_seed(6))
    got = gd.sample(m, B, x_T=x_T, ddim_steps=1, eta=1.0, seed=3)
    # the denoiser's own x0_hat at t = T-1 for the same x_T
    ops.pack_inputs([x_T.reshape(B * F, 30)], B * F, F, out_bf16=eng.xc(B, False), frame_stride=eng.ld_in, win_extra=0, col0=0)
    t_dev = torch.tensor([gd.T - 1], dtype=torch.int32, device="cuda")
    with torch.no_grad():
        x0h = eng.forward(B, F, False, t_scalar=t_dev, t_count=gd.T)[:, :30].reshape(B, F, 30).clone()
    torch.testing.assert_close(got, x0h, rtol=0, atol=0)


@pytest.mark.parametrize("S", [7, 10])
def test_graph_replay_equals_eager(S):
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F = 8, 10
    m, _ = _small_denoiser(F=F, L=1)
    _cond(m, B)
    gd = GaussianDiffusion(num_timesteps=20, device="cuda")
    a = gd.sample(m, B, seed=5, ddim_steps=S, eta=1.0, use_graph=False)
    b = gd.sample(m, B, seed=5, ddim_steps=S, eta=1.0)
    graph = gd._graphs[(id(m), B, (S, 1.0))]["graph"]
    c = gd.sample(m, B, seed=5, ddim_steps=S, eta=1.0)        # second call replays the cached graph only
    assert graph is not None and gd._graphs[(id(m), B, (S, 1.0))]["graph"] is graph
    assert torch.isfinite(a).all()
    torch.testing.assert_close(b, a, rtol=0, atol=0)
    torch.testing.assert_close(c, a, rtol=0, atol=0)


def test_interleaved_schedules_never_share_a_graph():
    """DDPM, DDIM-7 and DDIM-10 on one model and batch size each capture their own graph (the tables are baked into
    the captured launches); in any order each result equals a fresh eager run of its schedule."""
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F = 8, 10
    m, _ = _small_denoiser(F=F, L=1)
    _cond(m, B)
    schedules = [dict(), dict(ddim_steps=7, eta=1.0), dict(ddim_steps=10)]
    want = [GaussianDiffusion(num_timesteps=20, device="cuda").sample(m, B, seed=5, use_graph=False, **kw) for kw in schedules]
    gd = GaussianDiffusion(num_timesteps=20, device="cuda")
    for k in (0, 1, 2, 1, 0, 2, 2, 1, 0):
        torch.testing.assert_close(gd.sample(m, B, seed=5, **schedules[k]), want[k], rtol=0, atol=0, msg=lambda s: f"{k}: {s}")
    assert len(gd._graphs) == 3
    assert not torch.equal(want[1], want[2]) and not torch.equal(want[0], want[1])


def test_eta_zero_is_deterministic_given_x_T():
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F = 8, 10
    m, _ = _small_denoiser(F=F, L=1)
    _cond(m, B)
    gd = GaussianDiffusion(device="cuda")
    x_T = torch.randn(B, F, 30, device="cuda", generator=torch.Generator("cuda").manual_seed(8))
    a = gd.sample(m, B, x_T=x_T, ddim_steps=9, seed=1)
    b = gd.sample(m, B, x_T=x_T, ddim_steps=9, seed=2)
    assert torch.isfinite(a).all()
    torch.testing.assert_close(a, b, rtol=0, atol=0)
    c = gd.sample(m, B, x_T=x_T, ddim_steps=9, eta=1.0, seed=1)
    d = gd.sample(m, B, x_T=x_T, ddim_steps=9, eta=1.0, seed=2)
    assert not torch.equal(c, d)                           # eta > 0 draws per-seed noise


def test_sample_windows_with_ddim_matches_direct_calls():
    from inferbiomechanics_b200 import ops
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    F, N, batch = 10, 21, 8
    m, _ = _small_denoiser(F=F, L=1)
    eng = m.engine()
    gd = GaussianDiffusion(num_timesteps=12, device="cuda")
    cond = torch.randn(N, F, 177, generator=torch.Generator().manual_seed(4)).pin_memory()
    shards = [gd.sample_windows(m, cond, batch=batch, seed=9, rank=r, world=2, ddim_steps=5, eta=1.0) for r in range(2)]
    assert [len(s[0]) for s in shards] == [11, 10]
    for r, (rng, x0) in enumerate(shards):
        assert tuple(x0.shape) == (len(rng), F, 30) and torch.isfinite(x0).all()
        for i, a in enumerate(range(rng.start, rng.stop, batch)):
            b = min(a + batch, rng.stop)
            ops.pack_inputs([cond[a:b].reshape(-1, 177).cuda()], (b - a) * F, F, out_bf16=eng.xc(b - a, False), frame_stride=eng.ld_in,
                            win_extra=0, col0=30)
            want = gd.sample(m, b - a, seed=9 + r + 7919 * i, ddim_steps=5, eta=1.0)
            torch.testing.assert_close(x0[a - rng.start:b - rng.start], want.cpu(), rtol=0, atol=0)


def _run(argv):
    from inferbiomechanics_b200.main import main
    return main(argv)


def test_cli_ddim_analyze_and_train_dev_pass(tmp_path, capsys):
    ck = str(tmp_path / "ck")
    common = ["--no-wandb", "--synthetic-windows", "512", "--checkpoint-dir", ck, "--history-len", "50", "--stride", "1",
              "--model-type", "diffusion", "--batch-size", "64"]
    assert _run(["train", *common, "--epochs", "1", "--max-batches", "2", "--dev-sampling-steps", "4"]) is not None
    out = capsys.readouterr().out
    dev = re.search(r"Dev Set Evaluation: \n(.*?)Running Training Epoch", out, re.S)
    assert dev is not None and "Force Avg Err" in dev.group(1), out
    for extra in ([], ["--output-data-format", "last_frame"]):
        an = _run(["analyze", *common, "--sampler", "ddim", "--sampling-steps", "10", *extra])
        loss = an.last_reports["dev"]["loss"]
        assert math.isfinite(loss) and loss > 0, (extra, loss)
    with pytest.raises(ValueError, match="--eta"):
        _run(["analyze", *common, "--sampler", "ddpm", "--eta", "0.5"])
