"""Ensemble sampling and scoring on a B200: ``ibm_ensemble_score`` against the fp64 oracle (``tests/ensemble_oracle.py``), its
determinism, accumulation and refusals, ``GaussianDiffusion.sample(num_samples=K)`` against the B*K-window call it is built
from, ``sample_windows(num_samples=K)``, and ``analyze --num-samples``."""
import math
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

import ensemble_oracle as oens
from test_gpu_guidance import _entry_points, _pack_cond
from test_gpu_models import _small_denoiser, close

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _case(K, B, F, Fo, seed):
    """Draws (K, B, F, 30) with per-channel offsets and spreads, labels (B, Fo, 30) whose force triples sit on, just above and
    well away from the 10 N contact threshold."""
    g = torch.Generator().manual_seed(seed)
    mu = torch.randn(30, generator=g) * 3
    sig = torch.rand(30, generator=g) + 0.2
    draws = mu + sig * torch.randn(K, B, F, 30, generator=g)
    lab = mu + sig * torch.randn(B, Fo, 30, generator=g)
    u = torch.randint(0, 4, (B, Fo, 2), generator=g)
    just = float(np.nextafter(np.float32(10), np.float32(11)))
    for foot in range(2):
        sl = slice(6 + 3 * foot, 9 + 3 * foot)
        for code, trip in ((0, (10.0, 0.0, 0.0)), (1, (6.0, 8.0, 0.0)), (2, (just, 0.0, 0.0))):
            lab[..., sl][u[..., foot] == code] = torch.tensor(trip)
        lab[..., sl][u[..., foot] == 3] *= 20
    return draws.float(), lab.float()


def _score(draws, lab):
    from inferbiomechanics_b200 import ops
    acc = torch.zeros(5, 30, dtype=torch.float64, device="cuda")
    mean = torch.empty(lab.shape, device="cuda")
    ops.ensemble_score(draws.cuda(), lab.cuda(), acc, mean, ops.EnsembleWorkspace("cuda"))
    return mean, acc


@pytest.mark.parametrize("Fo", ["F", 1])
@pytest.mark.parametrize("K,B", [(2, 37), (3, 5), (8, 129), (17, 64), (64, 23)])
def test_kernel_matches_fp64_oracle(K, B, Fo):
    from inferbiomechanics_b200.loss.RegressionLossEvaluator import RegressionLossEvaluator
    F = 10
    fo = F if Fo == "F" else 1
    draws, lab = _case(K, B, F, fo, seed=K * 1000 + B + fo)
    mean, acc = _score(draws, lab)
    m, want, con = oens.score(draws.numpy(), lab.numpy())
    # contact decisions: the oracle's, and those of the loss evaluator's own mask kernel, give the CoP counts exactly
    mask = RegressionLossEvaluator.get_mask_by_threes(lab[..., 6:12].cuda(), 10.0).cpu().numpy()
    assert np.array_equal(mask[..., ::3] > 0, con)
    assert 0 < con.sum() < con.size
    got = acc.cpu().numpy()
    assert np.array_equal(got[4], want[4]), (got[4], want[4])
    np.testing.assert_allclose(mean.cpu().numpy(), m, rtol=1e-6, atol=0)
    np.testing.assert_allclose(got[:4], want[:4], rtol=1e-5, atol=0)


def test_mean_out_sentinels_and_bitwise_repeat_and_accumulation():
    from inferbiomechanics_b200 import ops
    K, B, F = 16, 300, 50
    draws, lab = _case(K, B, F, F, seed=7)
    draws, lab = draws.cuda(), lab.cuda()
    n = B * F * 30
    big = torch.full((n + 64,), float("nan"), device="cuda")
    big.view(torch.int32)[:] = 0x7FC0BEEF
    mean = big[32:32 + n].view(B, F, 30)
    ws = ops.EnsembleWorkspace("cuda")
    a1 = torch.zeros(5, 30, dtype=torch.float64, device="cuda")
    ops.ensemble_score(draws, lab, a1, mean, ws)
    bits = big.view(torch.int32)
    assert (bits[:32] == 0x7FC0BEEF).all() and (bits[32 + n:] == 0x7FC0BEEF).all()
    assert torch.isfinite(mean).all()
    a2 = torch.zeros(5, 30, dtype=torch.float64, device="cuda")
    ops.ensemble_score(draws, lab, a2, torch.empty_like(lab), ws)
    assert torch.equal(a1, a2), "two launches on the same input differ"
    ops.ensemble_score(draws, lab, a2, torch.empty_like(lab), ops.EnsembleWorkspace("cuda"))
    assert torch.equal(a2, 2 * a1), "successive batches do not accumulate"
    # one batch scored as two halves matches one call within fp64 rounding
    h = torch.zeros(5, 30, dtype=torch.float64, device="cuda")
    for sl in (slice(0, 131), slice(131, B)):
        ops.ensemble_score(draws[:, sl].contiguous(), lab[sl].contiguous(), h, torch.empty_like(lab[sl]), ws)
    torch.testing.assert_close(h, a1, rtol=1e-12, atol=0)


@pytest.mark.parametrize("K", [2, 16])
def test_calibrated_device_draws_give_unbiased_crps_and_unit_spread_skill(K):
    from inferbiomechanics_b200.loss.ensemble import EnsembleScorer
    B, F, mu, sigma = 1000, 34, 20.0, 1.3                 # ~1e6 elements; label forces ~ 35 N/kg: every row a contact
    g = torch.Generator("cuda").manual_seed(K)
    sc = EnsembleScorer(K, device="cuda")
    for _ in range(2):
        sc.score(mu + sigma * torch.randn(K, B, F, 30, device="cuda", generator=g),
                 mu + sigma * torch.randn(B, F, 30, device="cuda", generator=g))
    acc = sc.acc.cpu().numpy().sum(axis=1)
    assert acc[4] == 2 * B * F * 30
    crps, ssr = acc[0] / acc[4], math.sqrt((K + 1) / K * acc[1] / acc[2])
    assert abs(crps / (sigma / math.sqrt(math.pi)) - 1) < 0.01, crps
    assert abs(ssr - 1) < 0.02, ssr
    s = sc.summary()
    assert all(abs(s[q]["spread_skill"] - 1) < 0.05 for q in ("force", "cop", "moment", "wrench"))


def test_refusals_launch_nothing():
    from inferbiomechanics_b200 import _lib, ops
    ws = ops.EnsembleWorkspace("cuda")
    acc = torch.zeros(5, 30, dtype=torch.float64, device="cuda")
    lab = torch.zeros(4, 10, 30, device="cuda")
    bad = [
        (torch.zeros(1, 4, 10, 30, device="cuda"), lab, acc, torch.empty_like(lab)),          # K = 1
        (torch.zeros(65, 4, 10, 30, device="cuda"), lab, acc, torch.empty_like(lab)),         # K = 65
        (torch.zeros(4, 4, 10, 30, device="cuda"), torch.zeros(4, 3, 30, device="cuda"), acc,
         torch.empty(4, 3, 30, device="cuda")),                                               # Fo not in {1, F}
        (torch.zeros(4, 5, 10, 30, device="cuda"), lab, acc, torch.empty_like(lab)),          # B mismatch
        (torch.zeros(4, 10, 4, 30, device="cuda").transpose(1, 2), lab, acc, torch.empty_like(lab)),   # non-contiguous
        (torch.zeros(4, 4, 10, 30, device="cuda", dtype=torch.float64), lab, acc, torch.empty_like(lab)),
        (torch.zeros(4, 4, 10, 30, device="cuda"), lab, acc.float(), torch.empty_like(lab)),
        (torch.zeros(4, 4, 10, 30, device="cuda"), lab, acc, torch.empty(4, 1, 30, device="cuda")),
    ]
    n = _lib.launch_count
    for args in bad:
        with pytest.raises(ValueError, match="ensemble_score"):
            ops.ensemble_score(*args, ws)
    assert _lib.launch_count == n
    # the C entry point refuses the same cases itself (IBM_E_ARG) before launching
    lib = _lib.load()
    d = torch.zeros(65, 4, 10, 30, device="cuda")
    out = torch.empty_like(lab)
    s = torch.cuda.current_stream().cuda_stream
    args = lambda K, Fo=10, dp=d.data_ptr(), lp=lab.data_ptr(), cp=ws.counter.data_ptr(): (
        dp, K, 4, 10, lp, Fo, 10.0, out.data_ptr(), acc.data_ptr(), ws.partials.data_ptr(), cp, s)
    for a in (args(1), args(65), args(4, Fo=3), args(4, dp=d.data_ptr() + 2), args(4, lp=0), args(4, cp=0)):
        assert lib.ibm_ensemble_score(*a) == 1, a
    torch.cuda.synchronize()
    assert not acc.any() and not ws.counter.any()


# ---------------------------------------- sampling ------------------------------------------------------------------------
def _replicate(m, B, K):
    eng = m.engine()
    src = eng.xc(B, False).clone()
    eng.xc(B * K, False).copy_(src.repeat(K, 1))


@pytest.mark.parametrize("kw", [dict(), dict(ddim_steps=7, eta=0.0), dict(ddim_steps=7, eta=1.0),
                                dict(ddim_steps=6, eta=1.0, guidance_scale=2.5), dict(guidance_scale=0.5)],
                         ids=["ddpm", "ddim-eta0", "ddim-eta1", "ddim-guided", "ddpm-guided"])
def test_num_samples_is_the_call_on_replicated_windows(kw):
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F, K = 6, 10, 4
    m, _ = _small_denoiser(F=F, L=1)
    _pack_cond(m, B, 3)
    gd = GaussianDiffusion(num_timesteps=15, device="cuda")
    got = gd.sample(m, B, seed=5, num_samples=K, **kw)
    assert tuple(got.shape) == (K, B, F, 30) and torch.isfinite(got).all()
    again = gd.sample(m, B, seed=5, num_samples=K, **kw)          # graph replay
    eager = gd.sample(m, B, seed=5, num_samples=K, use_graph=False, **kw)
    _replicate(m, B, K)
    want = GaussianDiffusion(num_timesteps=15, device="cuda").sample(m, B * K, seed=5, use_graph=False, **kw)
    assert torch.equal(got.reshape(B * K, F, 30), want)
    assert torch.equal(again, got) and torch.equal(eager, got)
    # draw 0 starts from the x_T and noise of the B-window call; the forward on B*K rows may round differently
    one = GaussianDiffusion(num_timesteps=15, device="cuda").sample(m, B, seed=5, use_graph=False, **kw)
    close(got[0], one, 5e-2, "draw 0 vs the B-window sample")
    for k in range(1, K):
        assert (got[k] != got[0]).reshape(B, -1).any(dim=1).all(), f"draw {k} equals draw 0 for some window"


def test_num_samples_none_and_one_launch_todays_sequence():
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F = 8, 10
    m, _ = _small_denoiser(F=F, L=1)
    _pack_cond(m, B, 6)
    gd = GaussianDiffusion(num_timesteps=20, device="cuda")
    gd.sample(m, B, seed=5, ddim_steps=8, use_graph=False)
    plain = _entry_points(lambda: gd.sample(m, B, seed=5, ddim_steps=8, use_graph=False))
    none = _entry_points(lambda: gd.sample(m, B, seed=5, ddim_steps=8, use_graph=False, num_samples=None))
    one = _entry_points(lambda: gd.sample(m, B, seed=5, ddim_steps=8, use_graph=False, num_samples=1))
    assert plain == none == one and "ibm_ensemble_score" not in plain
    a = gd.sample(m, B, seed=5, ddim_steps=8)
    b = gd.sample(m, B, seed=5, ddim_steps=8, num_samples=1)
    assert tuple(b.shape) == (1, B, F, 30) and torch.equal(a, b[0])


def test_sample_windows_with_num_samples_matches_direct_calls():
    from inferbiomechanics_b200 import ops
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    F, N, batch, K = 10, 21, 8, 3
    m, _ = _small_denoiser(F=F, L=1)
    eng = m.engine()
    gd = GaussianDiffusion(num_timesteps=12, device="cuda")
    cond = torch.randn(N, F, 177, generator=torch.Generator().manual_seed(4)).pin_memory()
    kw = dict(ddim_steps=5, eta=1.0)
    rng, x0 = gd.sample_windows(m, cond, batch=batch, seed=9, rank=0, world=1, num_samples=K, **kw)
    assert tuple(x0.shape) == (N, K, F, 30) and x0.is_pinned() and torch.isfinite(x0).all()
    for i, a in enumerate(range(0, N, batch)):
        b = min(a + batch, N)
        ops.pack_inputs([cond[a:b].reshape(-1, 177).cuda()], (b - a) * F, F, out_bf16=eng.xc(b - a, False), frame_stride=eng.ld_in,
                        win_extra=0, col0=30)
        want = gd.sample(m, b - a, seed=9 + 7919 * i, num_samples=K, **kw)
        assert torch.equal(x0[a:b], want.transpose(0, 1).cpu())


# ---------------------------------------- CLI -----------------------------------------------------------------------------
def _run(argv):
    from inferbiomechanics_b200.main import main
    return main(argv)


COMMON = ["--no-wandb", "--synthetic-windows", "512", "--history-len", "50", "--stride", "1", "--model-type", "diffusion",
          "--batch-size", "64"]


def _ensemble_lines(out):
    return [ln for ln in out.splitlines() if re.match(r"\t(force|cop|moment|wrench): CRPS ", ln)]


def test_cli_analyze_num_samples(tmp_path, capsys):
    ck = str(tmp_path / "ck")
    common = [*COMMON, "--checkpoint-dir", ck]
    _run(["train", *common, "--epochs", "1", "--max-batches", "3", "--cond-drop-prob", "0.1"])
    capsys.readouterr()
    ddpm = ["--sampler", "ddpm", "--sampling-steps", "20"]
    plain = _run(["analyze", *common, *ddpm])
    out_plain = capsys.readouterr().out
    one = _run(["analyze", *common, *ddpm, "--num-samples", "1"])
    assert capsys.readouterr().out == out_plain and one.last_ensemble_reports == {}
    assert "ensemble" not in out_plain.lower()
    for extra in (ddpm, ["--sampler", "ddim", "--sampling-steps", "10", "--guidance-scale", "2"]):
        an = _run(["analyze", *common, *extra, "--num-samples", "4"])
        out = capsys.readouterr().out
        assert re.search(r"dev set evaluation \(\d+ windows(, guidance scale 2)?, ensemble mean of 4 samples\):", out), out
        assert len(_ensemble_lines(out)) == 8, out                 # four quantities, dev and train
        for split in ("dev", "train"):
            rep = an.last_ensemble_reports[split]
            for q in ("force", "cop", "moment", "wrench"):
                assert all(math.isfinite(rep[q][k]) for k in ("crps", "rmse", "spread", "spread_skill", "pair_dist")), rep[q]
                assert rep[q]["count"] > 0
            assert math.isfinite(an.last_reports[split]["loss"])
    assert plain.last_reports["dev"]["loss"] != an.last_reports["dev"]["loss"]


def test_cli_analyze_num_samples_two_ranks(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ck = str(tmp_path / "ck")
    _run(["train", *COMMON, "--checkpoint-dir", ck, "--epochs", "1", "--max-batches", "2"])
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", PYTHONPATH=ROOT)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29741", "-m", "inferbiomechanics_b200.main", "analyze", *COMMON, "--checkpoint-dir", ck,
           "--sampler", "ddim", "--sampling-steps", "8", "--num-samples", "4"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = _ensemble_lines(r.stdout)
    assert len(lines) == 8, r.stdout
    assert all("nan" not in ln for ln in lines)
