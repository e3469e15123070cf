"""Weight EMA surface without a GPU: the train / analyze flags, the range check of the decay before any device work, and
the checkpoint loader behind ``analyze --ema``."""
import argparse
import os

import pytest
import torch


def _parser():
    from inferbiomechanics_b200.cli.analyze import AnalyzeCommand
    from inferbiomechanics_b200.cli.train import TrainCommand
    p = argparse.ArgumentParser()
    sub = p.add_subparsers(dest="command")
    for c in (TrainCommand(), AnalyzeCommand()):
        c.register_subcommand(sub)
    return p


def test_ema_flags_parse_with_defaults_off():
    assert _parser().parse_args(["train"]).ema_decay == 0.0
    assert _parser().parse_args(["train", "--ema-decay", "0.999"]).ema_decay == 0.999
    assert _parser().parse_args(["analyze"]).ema is False
    assert _parser().parse_args(["analyze", "--ema"]).ema is True


@pytest.mark.parametrize("decay", ["1.0", "-0.1", "1.5", "nan"])
def test_train_rejects_decay_outside_unit_interval_before_gpu(decay):
    from inferbiomechanics_b200.cli.train import TrainCommand
    args = _parser().parse_args(["train", "--no-wandb", "--ema-decay", decay])
    with pytest.raises(ValueError, match="--ema-decay"):
        TrainCommand().run(args)


@pytest.mark.parametrize("decay", [1.0, -0.5])
def test_trainer_rejects_decay_outside_unit_interval(decay):
    from inferbiomechanics_b200.trainer import Trainer
    with pytest.raises(ValueError, match="ema_decay"):
        Trainer(None, ema_decay=decay)


def test_checkpoint_loader_reads_ema_or_names_the_file(tmp_path, capsys):
    from inferbiomechanics_b200.cli.abstract_command import AbstractCommand
    cmd = AbstractCommand()
    model = torch.nn.Linear(3, 2)
    d = tmp_path / "ck"
    os.makedirs(d)
    raw = {k: torch.full_like(v, 1.0) for k, v in model.state_dict().items()}
    torch.save({"epoch": 0, "model_state_dict": raw, "optimizer_state_dict": {}}, d / "epoch_0_batch_9.pt")
    with pytest.raises(ValueError, match="epoch_0_batch_9.pt"):
        cmd.load_latest_checkpoint(model, checkpoint_dir=str(d), state_key="ema_state_dict")
    # the newest checkpoint carries an average: --ema loads it, the default still loads the trained weights
    ema = {k: torch.full_like(v, 2.0) for k, v in model.state_dict().items()}
    torch.save({"epoch": 1, "model_state_dict": raw, "optimizer_state_dict": {}, "ema_state_dict": ema}, d / "epoch_1_batch_3.pt")
    assert cmd.load_latest_checkpoint(model, checkpoint_dir=str(d), state_key="ema_state_dict") == (1, 3)
    assert float(model.weight.detach()[0, 0]) == 2.0
    assert cmd.load_latest_checkpoint(model, checkpoint_dir=str(d)) == (1, 3)
    assert float(model.weight.detach()[0, 0]) == 1.0
