"""Ensemble scoring without a GPU: the oracle's fair CRPS (pair form = sorted form = hand-computed cases), its calibration on
Gaussian draws against the biased K^2 estimator, the argument checks of the sampler, the ops wrapper, the scorer and
``analyze --num-samples`` (before any device work), the parser default, and ``EnsembleScorer``'s rank-order merge and metrics."""
import argparse
import math

import numpy as np
import pytest
import torch

import ensemble_oracle as oens


def _parser():
    from inferbiomechanics_b200.cli.analyze import AnalyzeCommand
    from inferbiomechanics_b200.cli.train import TrainCommand
    p = argparse.ArgumentParser()
    sub = p.add_subparsers(dest="command")
    for c in (TrainCommand(), AnalyzeCommand()):
        c.register_subcommand(sub)
    return p


def test_fair_crps_pair_form_equals_sorted_form_and_hand_cases():
    # K = 2: x = (1, 3), y = 0: (1 + 3)/2 - 2*|1-3| / (2*2*1) = 2 - 1 = 1
    assert oens.fair_crps(np.array([1.0, 3.0]), 0.0) == pytest.approx(1.0, abs=1e-15)
    assert oens.fair_crps_sorted(np.array([3.0, 1.0]), 0.0) == pytest.approx(1.0, abs=1e-15)
    # K = 3: x = (0, 1, 4), y = 2: mean |x - y| = (2 + 1 + 2)/3 = 5/3; sum_{i<j} = 1 + 4 + 3 = 8 -> 8 / (3*2) = 4/3; crps = 1/3
    assert oens.fair_crps(np.array([4.0, 0.0, 1.0]), 2.0) == pytest.approx(1.0 / 3.0, abs=1e-15)
    assert oens.fair_crps_sorted(np.array([4.0, 0.0, 1.0]), 2.0) == pytest.approx(1.0 / 3.0, abs=1e-15)
    assert oens.pair_sum(np.array([4.0, 0.0, 1.0])) == 8.0 == oens.pair_sum_sorted(np.array([4.0, 0.0, 1.0]))
    rng = np.random.default_rng(0)
    for K in (2, 3, 8, 17, 64):
        x, y = rng.normal(size=(K, 200)) * 3 + 1, rng.normal(size=200)
        np.testing.assert_allclose(oens.pair_sum(x), oens.pair_sum_sorted(x), rtol=1e-12)
        np.testing.assert_allclose(oens.fair_crps(x, y), oens.fair_crps_sorted(x, y), rtol=1e-10, atol=1e-12)


def _calibrated(K, n=100_000, mu=0.7, sigma=1.3, seed=1):
    rng = np.random.default_rng(seed + K)
    return rng.normal(mu, sigma, size=(K, n)), rng.normal(mu, sigma, size=n), sigma


@pytest.mark.parametrize("K", [2, 16])
def test_fair_crps_is_unbiased_and_spread_skill_is_one_on_calibrated_draws(K):
    x, y, sigma = _calibrated(K)
    want = sigma / math.sqrt(math.pi)
    assert abs(oens.fair_crps_sorted(x, y).mean() / want - 1) < 0.01
    m = x.mean(axis=0)
    ssr = math.sqrt((K + 1) / K * ((x - m) ** 2).sum(axis=0).sum() / (K - 1) / ((m - y) ** 2).sum())
    assert abs(ssr - 1) < 0.02
    if K == 2:    # the K^2 estimator's mean is sigma/sqrt(pi) (1 + 1/K): the 1 % check tells the two apart
        assert abs(oens.biased_crps(x, y).mean() / want - 1) > 0.01
        assert abs(oens.biased_crps(x, y).mean() / (want * (1 + 1 / K)) - 1) < 0.01


def test_oracle_score_scores_cop_on_contact_rows_only():
    rng = np.random.default_rng(3)
    K, B, F = 3, 4, 5
    draws = rng.normal(size=(K, B, F, 30))
    lab = rng.normal(size=(B, F, 30)).astype(np.float32)
    lab[..., 6:9] = [10.0, 0.0, 0.0]                    # on the threshold: no contact
    lab[0, 0, 6:9] = [np.nextafter(np.float32(10), np.float32(11)), 0, 0]
    lab[..., 9:12] = [6.0, 8.0, 0.0]                    # norm exactly 10: no contact
    lab[1, 2, 9:12] = [20.0, 0.0, 0.0]
    _, acc, con = oens.score(draws, lab)
    assert con[..., 0].sum() == 1 and con[..., 1].sum() == 1
    assert list(acc[4, :6]) == [1, 1, 1, 1, 1, 1] and (acc[4, 6:] == B * F).all()
    _, acc1, _ = oens.score(draws, lab[:, -1:])
    assert (acc1[4, 6:] == B).all() and (acc1[4, :6] == 0).all()


def test_num_samples_parses_with_default_one():
    assert _parser().parse_args(["analyze"]).num_samples == 1
    assert _parser().parse_args(["analyze", "--num-samples", "16"]).num_samples == 16


@pytest.mark.parametrize("flags,match", [(["--model-type", "diffusion", "--num-samples", "0"], r"\[1, 64\]"),
                                         (["--model-type", "diffusion", "--num-samples", "65"], r"\[1, 64\]"),
                                         (["--model-type", "feedforward", "--num-samples", "2"], "diffusion only"),
                                         (["--model-type", "groundlink", "--num-samples", "4"], "diffusion only"),
                                         (["--model-type", "diffusion", "--num-samples", "8", "--batch-size", "4"], "exceeds")])
def test_analyze_rejects_bad_num_samples_before_gpu(tmp_path, flags, match):
    from inferbiomechanics_b200.cli.analyze import AnalyzeCommand
    args = _parser().parse_args(["analyze", "--no-wandb", "--checkpoint-dir", str(tmp_path), *flags])
    with pytest.raises(ValueError, match=match):
        AnalyzeCommand().run(args)


@pytest.mark.parametrize("K", [0, 65, -1, 2.0])
def test_sampler_rejects_num_samples_outside_range(K):
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    gd = GaussianDiffusion(num_timesteps=20, device="cpu")
    with pytest.raises(ValueError, match="num_samples"):
        gd.sample(None, 4, num_samples=K)
    with pytest.raises(ValueError, match="num_samples"):
        gd.sample(None, 4, ddim_steps=5, eta=1.0, guidance_scale=2.0, num_samples=K)
    with pytest.raises(ValueError, match="num_samples"):
        gd.sample_windows(None, torch.zeros(4, 10, 177), num_samples=K)


def test_ensemble_score_rejects_cpu_tensors_and_scorer_rejects_k_below_two():
    from inferbiomechanics_b200 import _lib, ops
    from inferbiomechanics_b200.loss.ensemble import EnsembleScorer
    n = _lib.launch_count
    ws = ops.EnsembleWorkspace("cpu")
    with pytest.raises(ValueError, match="CUDA"):
        ops.ensemble_score(torch.zeros(4, 2, 5, 30), torch.zeros(2, 5, 30), torch.zeros(5, 30, dtype=torch.float64),
                           torch.zeros(2, 5, 30), ws)
    assert _lib.launch_count == n
    for K in (1, 65):
        with pytest.raises(ValueError, match="num_samples"):
            EnsembleScorer(K, device="cpu")


def test_merge_sums_the_ranks_in_rank_order(monkeypatch):
    import torch.distributed as dist
    from inferbiomechanics_b200.loss.ensemble import EnsembleScorer
    sc = EnsembleScorer(4, device="cpu")
    # values whose fp64 sum depends on the order: rank order gives ((1e16 + 1) + 1) - 1e16 = 0, other orders 2
    ranks = [torch.full((5, 30), v, dtype=torch.float64) for v in (1e16, 1.0, 1.0, -1e16)]

    def fake_all_gather(out, t):
        assert torch.equal(t, sc.acc)
        for o, r in zip(out, ranks):
            o.copy_(r)

    monkeypatch.setattr(dist, "all_gather", fake_all_gather)
    sc.merge(4)
    want = np.zeros((5, 30))
    for r in ranks:
        want += r.numpy()
    assert np.array_equal(sc.acc.numpy(), want)
    assert sc.acc[0, 0].item() == 0.0
    assert ((1.0 + 1.0) + 1e16) + -1e16 == 2.0          # another order gives another sum
    before = sc.acc.clone()
    sc.merge(1)                                          # one rank: nothing to gather
    assert torch.equal(sc.acc, before)


def test_summary_pools_the_channels_of_each_quantity():
    from inferbiomechanics_b200.loss.ensemble import EnsembleScorer, ensemble_metrics
    K = 4
    sc = EnsembleScorer(K, device="cpu")
    rng = np.random.default_rng(5)
    acc = rng.uniform(1, 2, size=(5, 30))
    acc[4] = rng.integers(10, 100, size=30)
    sc.acc.copy_(torch.from_numpy(acc))
    s = sc.summary()
    f = acc[:, 6:12].sum(axis=1)
    assert s["force"]["crps"] == pytest.approx(f[0] / f[4])
    assert s["force"]["rmse"] == pytest.approx(math.sqrt(f[2] / f[4]))
    assert s["force"]["spread"] == pytest.approx(math.sqrt(f[1] / f[4]))
    assert s["force"]["spread_skill"] == pytest.approx(math.sqrt((K + 1) / K * f[1] / f[2]))
    assert s["force"]["pair_dist"] == pytest.approx(f[3] / f[4])
    assert s["force"]["count"] == int(f[4])
    assert s["wrench"]["count"] == int(acc[4, 18:30].sum()) and s["cop"]["count"] == int(acc[4, :6].sum())
    assert s["channels"]["crps"][3] == pytest.approx(acc[0, 3] / acc[4, 3])
    assert math.isnan(ensemble_metrics(np.zeros(5), K)["crps"])
