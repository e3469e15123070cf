"""Inpainting surface without a GPU: the oracle's loops at the two ends of the mask, the mask → row-word packing and the
quantity → channel mapping, the argument checks of the sampler, the step wrappers and ``analyze --given-quantities`` (before
any device work), the parser default and the report's "given" marks."""
import argparse

import numpy as np
import pytest
import torch

import cfg_oracle as ocfg
import ddim_oracle as odim
import inpaint_oracle as oinp
from oracle import ddpm as oddpm

B, F = 3, 4


def _denoise(x, t):
    """A toy x0-predictor that depends on x and t and couples the channels of a row (the oracle loops only need a callable)."""
    x = x.double()
    return 0.7 * torch.tanh(x) + 0.3 * x.mean(-1, keepdim=True) + 0.01 * np.sin(t)


def _case(seed):
    g = torch.Generator().manual_seed(seed)
    x_T = torch.randn(B * F, 30, generator=g)
    y = torch.randn(B * F, 30, generator=g)
    zs = {t: torch.randn(B * F, 30, generator=g) for t in range(1000)}
    return x_T, y, zs


def _ddpm(denoise, x_T, zs):
    sched = {k: v.double() for k, v in oddpm.make_schedule().items()}
    return oddpm.sample_loop(sched, lambda x, t: denoise(x, t).double(), x_T.double(), lambda t: zs[t].double()).float()


def _ddim(denoise, x_T, zs, S, eta):
    return odim.ddim_sample_loop(odim.abar(), denoise, x_T, S, eta, lambda t: zs[t])


@pytest.mark.parametrize("guided", [False, True])
def test_oracle_loops_return_y_with_every_entry_known_and_the_plain_result_with_none(guided):
    x_T, y, zs = _case(1)
    den = ocfg.guided_denoiser(lambda x, t, cond: _denoise(x, t) + (0.2 if cond else 0.0), 2.5) if guided else _denoise
    everything, nothing = torch.ones(30, dtype=torch.bool), torch.zeros(30, dtype=torch.bool)
    assert torch.equal(_ddpm(oinp.known_denoiser(den, y, everything), x_T, zs), y)
    assert torch.equal(_ddpm(oinp.known_denoiser(den, y, nothing), x_T, zs), _ddpm(den, x_T, zs))
    for S, eta in ((1, 0.0), (2, 1.0), (7, 0.0), (50, 1.0)):
        assert torch.equal(_ddim(oinp.known_denoiser(den, y, everything), x_T, zs, S, eta), y), (S, eta)
        assert torch.equal(_ddim(oinp.known_denoiser(den, y, nothing), x_T, zs, S, eta), _ddim(den, x_T, zs, S, eta)), (S, eta)


def test_oracle_partial_mask_holds_known_entries_and_ignores_unknown_nan():
    x_T, y, zs = _case(2)
    mask = torch.rand(B * F, 30, generator=torch.Generator().manual_seed(3)) < 0.4
    y_nan = torch.where(mask, y, torch.full_like(y, float("nan")))
    out = _ddim(oinp.known_denoiser(_denoise, y_nan, mask), x_T, zs, 7, 1.0)
    assert torch.equal(out[mask], y[mask]) and torch.isfinite(out).all()
    plain = _ddim(_denoise, x_T, zs, 7, 1.0)
    assert not torch.equal(out[~mask], plain[~mask])          # the unknown entries are conditioned on the known ones


def test_mask_words_match_the_oracle_and_ignore_nothing():
    from inferbiomechanics_b200.diffusion import known_mask_words
    g = torch.Generator().manual_seed(5)
    mask = torch.rand(B, F, 30, generator=g) < 0.5
    assert torch.equal(known_mask_words(mask, B * F), oinp.mask_words(mask).view(-1))
    one = torch.zeros(30, dtype=torch.bool)
    one[[0, 7, 29]] = True
    w = known_mask_words(one, 5)
    assert w.dtype == torch.int32 and tuple(w.shape) == (5,) and (w == (1 | 1 << 7 | 1 << 29)).all()
    assert (known_mask_words(torch.ones(30, dtype=torch.bool), 2) == (1 << 30) - 1).all()
    assert (known_mask_words(torch.zeros(30, dtype=torch.bool), 2) == 0).all()


def test_quantity_bits():
    from inferbiomechanics_b200.cli.train import known_quantity_mask
    from inferbiomechanics_b200.diffusion import known_mask_words

    def word(*qs):
        return int(known_mask_words(known_quantity_mask(qs), 1)[0])

    assert word("force") == 0b111111 << 6
    assert word("cop") == 0b111111
    assert word("moment") == 0b111111 << 12
    assert word("wrench") == 0xFFF << 18
    assert word("force", "cop") == 0xFFF
    assert word("cop", "force", "moment", "wrench") == (1 << 30) - 1
    assert word() == 0
    with pytest.raises(ValueError, match="unknown quantity"):
        known_quantity_mask(("grf",))


def _y(shape=(B, F, 30), dtype=torch.float32):
    return torch.zeros(shape, dtype=dtype)


@pytest.mark.parametrize("kw,match", [
    (dict(known=_y()), "give both or neither"),
    (dict(known_mask=torch.ones(30, dtype=torch.bool)), "give both or neither"),
    (dict(known=_y(dtype=torch.float64), known_mask=torch.ones(30, dtype=torch.bool)), "known must be an fp32"),
    (dict(known=_y((B + 1, F, 30)), known_mask=torch.ones(30, dtype=torch.bool)), "known must be an fp32"),
    (dict(known=_y((B, F, 29)), known_mask=torch.ones(30, dtype=torch.bool)), "known must be an fp32"),
    (dict(known=_y((B, F * 30)), known_mask=torch.ones(30, dtype=torch.bool)), "known must be an fp32"),
    (dict(known=_y(), known_mask=torch.ones(30, dtype=torch.uint8)), "known_mask must be a bool"),
    (dict(known=_y(), known_mask=torch.ones(29, dtype=torch.bool)), "known_mask must be a bool"),
    (dict(known=_y(), known_mask=torch.ones(B, F, 6, dtype=torch.bool)), "known_mask must be a bool"),
    (dict(known=_y(), known_mask=torch.ones(30, dtype=torch.bool), steps=10), "whole chain"),
])
def test_sampler_rejects_bad_known_arguments(kw, match):
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    gd = GaussianDiffusion(num_timesteps=20, device="cpu")
    with pytest.raises(ValueError, match=match):
        gd.sample(None, B, **kw)
    if "known" in kw and kw["known"].dim() == 3:
        with pytest.raises(ValueError, match=match):
            gd.sample_windows(None, torch.zeros(B, F, 177), **kw)


def test_sampler_accepts_the_whole_ddpm_chain_and_rejects_known_values_off_the_device():
    from inferbiomechanics_b200.diffusion import GaussianDiffusion, check_known
    mask = torch.ones(30, dtype=torch.bool)
    assert check_known(_y(), mask, B, F, 20, 20)
    assert check_known(_y(), mask, B, F, 20, None)
    assert not check_known(None, None, B, F, 20, 5)
    with pytest.raises(ValueError, match="on meta"):
        check_known(_y(), mask, B, F, 20, None, device="meta")
    gd = GaussianDiffusion(num_timesteps=20, device="cpu")
    with pytest.raises(ValueError, match="known must be on"):
        gd.sample(None, B, known=_y().to("meta"), known_mask=mask)


def _step_args(M):
    x0h, x = torch.zeros(M, 32), torch.zeros(M, 30)
    t = torch.zeros(1, dtype=torch.int32)
    return (x0h, 32, x, None, t, torch.zeros(20), torch.zeros(20), torch.zeros(20), M)


@pytest.mark.parametrize("known,mask,match", [
    (torch.zeros(6, 30), None, "both or neither"),
    (None, torch.zeros(6, dtype=torch.int32), "both or neither"),
    (torch.zeros(6, 30), torch.zeros(6, dtype=torch.int32), "CUDA tensor"),             # host tensors
])
def test_step_wrappers_reject_bad_known_arguments_before_calling(known, mask, match):
    from inferbiomechanics_b200 import _lib, ops
    n = _lib.launch_count
    with pytest.raises(ValueError, match=match):
        ops.posterior_step(*_step_args(6), x_prev=torch.zeros(6, 30), known=known, known_mask=mask)
    with pytest.raises(ValueError, match=match):
        ops.guided_step(*_step_args(6), 2.5, x_prev=torch.zeros(6, 30), known=known, known_mask=mask)
    assert _lib.launch_count == n


def _parser():
    from inferbiomechanics_b200.cli.analyze import AnalyzeCommand
    p = argparse.ArgumentParser()
    AnalyzeCommand().register_subcommand(p.add_subparsers(dest="command"))
    return p


def test_given_quantities_parse_with_default_none():
    assert _parser().parse_args(["analyze"]).given_quantities == []
    assert _parser().parse_args(["analyze", "--given-quantities", "force", "cop"]).given_quantities == ["force", "cop"]
    with pytest.raises(SystemExit):
        _parser().parse_args(["analyze", "--given-quantities", "grf"])


@pytest.mark.parametrize("flags,match", [
    (["--model-type", "feedforward"], "diffusion only"),
    (["--model-type", "groundlink"], "diffusion only"),
    (["--model-type", "diffusion", "--output-data-format", "last_frame"], "all_frames"),
    (["--model-type", "diffusion", "--sampler", "ddpm", "--sampling-steps", "999"], "whole chain"),
])
def test_analyze_rejects_given_quantities_before_gpu(tmp_path, flags, match):
    from inferbiomechanics_b200.cli.analyze import AnalyzeCommand
    args = _parser().parse_args(["analyze", "--no-wandb", "--checkpoint-dir", str(tmp_path), "--given-quantities", "force", *flags])
    with pytest.raises(ValueError, match=match):
        AnalyzeCommand().run(args)


def test_analyze_accepts_given_quantities_on_the_whole_chain():
    from inferbiomechanics_b200.cli.analyze import AnalyzeCommand
    for flags in (["--sampler", "ddim", "--sampling-steps", "4"], ["--sampler", "ddpm"]):
        args = _parser().parse_args(["analyze", "--model-type", "diffusion", "--given-quantities", "force", *flags])
        AnalyzeCommand.check_given_quantities(tuple(args.given_quantities), "diffusion", args)


def test_sample_and_score_rejects_known_quantities_with_last_frame_labels():
    from types import SimpleNamespace

    from inferbiomechanics_b200.cli.train import sample_and_score
    model = SimpleNamespace(engine=lambda: SimpleNamespace(input_layout=lambda *a: None))
    store = SimpleNamespace(F=10, Fo=1, pack=lambda idx, layout: None)
    with pytest.raises(ValueError, match="every frame"):
        sample_and_score(None, model, store, torch.arange(4), None, None, 0, ddim_steps=4, known_quantities=("force",))


def test_ensemble_report_marks_given_quantities(capsys):
    from inferbiomechanics_b200.loss.ensemble import EnsembleScorer
    sc = EnsembleScorer(2, "dev", device="cpu")
    sc.acc[4] = 1.0
    sc.print_report(given=("force",))
    out = capsys.readouterr().out
    assert "\tforce (given): CRPS" in out and "\tcop: CRPS" in out and out.count("(given)") == 1
