"""The train / analyze commands end to end on a B200 (synthetic AddBiomechanics-shaped windows, BASELINE configs[0]
shape: FeedForward, T=50, stride 5, batch 32): flags as in the reference, checkpoint written in the reference format
and picked up by analyze, loss decreasing, window-store file round trip bit-exact."""
import argparse
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


def _run(argv):
    from inferbiomechanics_b200.main import main
    return main(argv)


def test_train_then_analyze_feedforward(tmp_path, capsys):
    ck = str(tmp_path / "ck")
    common = ["--no-wandb", "--synthetic-windows", "4096", "--checkpoint-dir", ck, "--history-len", "50", "--stride", "5",
              "--hidden-dims", "512", "512", "--activation", "sigmoid"]
    cmd = _run(["train", *common, "--model-type", "feedforward", "--epochs", "2", "--batch-size", "32", "--learning-rate", "1e-3"])
    assert cmd is not None
    files = sorted(os.listdir(os.path.join(ck, "feedforward")))
    # reference naming (train.py:271): one checkpoint at the last batch of each epoch (synthetic stores round the window
    # count up to whole trials, so the batch count is read back rather than assumed)
    assert len(files) == 2 and files[0].startswith("epoch_0_batch_") and files[1].startswith("epoch_1_batch_")
    assert files[0].split("_batch_")[1] == files[1].split("_batch_")[1]
    sd = torch.load(os.path.join(ck, "feedforward", files[-1]), map_location="cpu")
    assert set(sd) == {"epoch", "model_state_dict", "optimizer_state_dict"} and sd["epoch"] == 1
    assert set(sd["model_state_dict"]) == {"net.0.weight", "net.0.bias", "net.2.weight", "net.2.bias", "net.4.weight", "net.4.bias"}
    out = capsys.readouterr().out
    assert "Evaluating Dev Set Before Epoch 1" in out and "Force Avg Err" in out
    an = _run(["analyze", *common, "--model-type", "feedforward", "--predict-grf-components", "0", "1", "2", "3", "4", "5"])
    rep = an.last_reports
    assert set(rep) == {"dev", "train"} and all(r is not None and r["loss"] > 0 for r in rep.values())
    # resuming: a third epoch starts from the epoch-1 checkpoint (abstract_command.load_latest_checkpoint)
    _run(["train", *common, "--model-type", "feedforward", "--epochs", "3", "--batch-size", "32", "--max-batches", "4"])
    assert "epoch_2_batch_3.pt" in os.listdir(os.path.join(ck, "feedforward"))
    assert "Loaded checkpoint from epoch 1" in capsys.readouterr().out


def test_train_batchnorm_dropout_checkpoint_is_analyzable(tmp_path):
    """--batchnorm --dropout shift the state_dict positions (SURVEY §9.3); analyze reads the layout off the checkpoint."""
    ck = str(tmp_path / "ck")
    common = ["--no-wandb", "--synthetic-windows", "1024", "--checkpoint-dir", ck, "--history-len", "50", "--stride", "5",
              "--hidden-dims", "64", "64", "--activation", "relu"]
    _run(["train", *common, "--model-type", "feedforward", "--epochs", "1", "--batch-size", "64", "--batchnorm", "--dropout",
          "--dropout-prob", "0.1", "--opt-type", "adam"])
    sd = torch.load(os.path.join(ck, "feedforward", sorted(os.listdir(os.path.join(ck, "feedforward")))[-1]), map_location="cpu")
    assert "net.1.running_mean" in sd["model_state_dict"] and "net.2.weight" in sd["model_state_dict"]
    assert sd["optimizer_state_dict"]["ibm_b200"]["opt_type"] == "adam" and 0 in sd["optimizer_state_dict"]["state"]
    an = _run(["analyze", *common, "--model-type", "feedforward"])
    assert an.last_reports["dev"]["loss"] > 0


def test_train_groundlink_and_diffusion_smoke(tmp_path):
    ck = str(tmp_path / "ck")
    common = ["--no-wandb", "--synthetic-windows", "512", "--checkpoint-dir", ck, "--history-len", "50", "--stride", "1",
              "--epochs", "1", "--max-batches", "3"]
    assert _run(["train", *common, "--model-type", "groundlink", "--batch-size", "16"]) is not None
    assert _run(["train", *common, "--model-type", "diffusion", "--batch-size", "64"]) is not None
    an = _run(["analyze", "--no-wandb", "--synthetic-windows", "512", "--checkpoint-dir", ck, "--history-len", "50", "--stride", "1",
               "--model-type", "diffusion", "--batch-size", "64", "--sampling-steps", "20", "--predict-grf-components", "0", "1", "2"])
    assert an.last_reports["dev"]["loss"] > 0
    an = _run(["analyze", "--no-wandb", "--synthetic-windows", "256", "--checkpoint-dir", ck, "--history-len", "50", "--stride", "1",
               "--model-type", "diffusion", "--batch-size", "64", "--sampling-steps", "4", "--output-data-format", "last_frame"])
    assert an.last_reports["dev"]["loss"] > 0               # last_frame labels vs the last sampled frame


def test_window_store_file_roundtrip(tmp_path):
    from inferbiomechanics_b200.data.window_store import WindowStore
    a = WindowStore.synthetic(3000, 50, 5, 147, "all_frames", seed=5, device="cuda")
    p = str(tmp_path / "train.ibmstore")
    a.save(p)
    b = WindowStore.load(p, 50, 5, "all_frames", device="cuda")
    assert len(a) == len(b) and torch.equal(a.win_row0, b.win_row0)
    idx = torch.arange(0, len(a), 7, device="cuda")
    assert torch.equal(a.pack_f32(idx), b.pack_f32(idx)) and torch.equal(a.labels(idx), b.labels(idx))
    with open(p, "r+b") as f:
        f.write(b"XX")
    with pytest.raises(ValueError):
        WindowStore.load(p, 50, 5, "all_frames", device="cuda")


@pytest.mark.parametrize("opt", ["rmsprop", "adam", "adadelta", "sgd"])
def test_trainer_resume_continues_the_uninterrupted_run(tmp_path, opt):
    """Save after 3 native steps (model.state_dict() + Trainer.optimizer_state_dict(), the checkpoint train.py:270-278 writes),
    load both into a fresh model/Trainer, run 3 more: parameters equal those of 6 uninterrupted steps.  The optimizer blob
    is torch.optim's own layout — the matching torch optimizer loads it and holds the same tensors.
    Tolerance 2e-5 absolute on parameters of size ~0.03: split-K weight gradients are fp32 TMA reduce-adds whose order is
    not fixed, so two runs of the same step differ in the last bits."""
    from inferbiomechanics_b200.data.window_store import WindowStore
    from inferbiomechanics_b200.models.FeedForwardRegressionBaseline import FeedForwardBaseline
    from inferbiomechanics_b200.trainer import Trainer

    def fresh():
        torch.manual_seed(0)
        return FeedForwardBaseline(23, 2, 50, "all_frames", "sigmoid", 5, 10, hidden_dims=[64, 64]).cuda()

    store = WindowStore.synthetic(1024, 50, 5, 147, "all_frames", seed=3, device="cuda")
    idx = store.shard(0, 1)
    batches = [idx[i * 32:(i + 1) * 32] for i in range(6)]
    a = fresh()
    ta = Trainer(a, opt_type=opt, lr=1e-3)
    for b in batches:
        ta.train_step(store, b)
    m1 = fresh()
    t1 = Trainer(m1, opt_type=opt, lr=1e-3)
    for b in batches[:3]:
        t1.train_step(store, b)
    path = str(tmp_path / "epoch_0_batch_2.pt")
    torch.save({"epoch": 0, "model_state_dict": m1.state_dict(), "optimizer_state_dict": t1.optimizer_state_dict()}, path)
    ck = torch.load(path, map_location="cpu")
    m2 = fresh()
    m2.load_state_dict(ck["model_state_dict"])
    t2 = Trainer(m2, opt_type=opt, lr=1e-3)
    t2.load_optimizer_state_dict(ck["optimizer_state_dict"])
    assert t2.step_count == 3
    t2.arena.sync_shadow(force=True)
    for b in batches[3:]:
        t2.train_step(store, b)
    for (n, p), q in zip(a.named_parameters(), m2.parameters()):
        assert (p - q).abs().max().item() <= 2e-5, n
    # the reference side: torch.optim's own class accepts the blob (abstract_command.py:113-114)
    cls = getattr(torch.optim, Trainer._OPT_CLASS[opt])
    topt = cls(m2.parameters(), lr=1e-3)
    topt.load_state_dict({k: v for k, v in ck["optimizer_state_dict"].items() if k != "ibm_b200"})
    n0, _ = Trainer._OPT_STATE[opt]
    if n0 is not None:
        st = topt.state[next(iter(m2.parameters()))]
        o, k = t1.arena.offsets[t1.arena.names[0]]
        assert torch.equal(st[n0].reshape(-1).cpu(), t1.state0[o:o + k].cpu()) and int(st["step"]) == 3
    with pytest.raises(ValueError):
        Trainer(fresh(), opt_type="adagrad", lr=1e-3).load_optimizer_state_dict(ck["optimizer_state_dict"])


@pytest.mark.parametrize("kind,opt", [("feedforward_dropout_bn", "adam"), ("feedforward", "adamax"), ("groundlink", "rmsprop"),
                                      ("groundlink_eval", "rmsprop")])
def test_graph_replayed_steps_equal_eager_steps(monkeypatch, kind, opt):
    """Small-batch steps are captured once and replayed (Trainer._graphable): with dropout, BatchNorm, Adam/Adamax and for
    Groundlink too — the Philox offsets and the bias-correction step come from a device-resident counter.  Same seeds =>
    same masks => the replayed run equals the eager run (2e-5 absolute: fp32 reduce-add order of split-K weight gradients).
    ``groundlink_eval`` evaluates right before the capture and between replays: both the captured steps and the evaluations
    must read the conv weights the optimizer last wrote, not a cached GEMM layout of older ones."""
    from inferbiomechanics_b200.data.window_store import WindowStore
    from inferbiomechanics_b200.models.FeedForwardRegressionBaseline import FeedForwardBaseline
    from inferbiomechanics_b200.models.Groundlink import Groundlink
    from inferbiomechanics_b200.trainer import Trainer

    def run(graphs: bool):
        monkeypatch.setenv("IBM_TRAIN_GRAPHS", "1" if graphs else "0")
        torch.manual_seed(0)
        if kind.startswith("groundlink"):
            m = Groundlink(23, 12, 10, "all_frames").cuda().train()
            store = WindowStore.synthetic(512, 20, 1, 177, "all_frames", seed=3, device="cuda")
            B = 16
        else:
            bn = kind.endswith("_bn")
            m = FeedForwardBaseline(23, 2, 50, "all_frames", "relu", 5, 10, hidden_dims=[64, 64], batchnorm=bn, dropout=bn,
                                    dropout_prob=0.25).cuda().train()
            store = WindowStore.synthetic(1024, 50, 5, 147, "all_frames", seed=3, device="cuda")
            B = 32
        tr = Trainer(m, opt_type=opt, lr=1e-3, seed=9)
        idx = store.shard(0, 1)
        losses, evals = [], []
        for i in range(7):
            losses.append(tr.train_step(store, idx[(i % 4) * B:(i % 4 + 1) * B])[0].item())
            if kind == "groundlink_eval" and i in (1, 4):     # after the last eager step before the capture, and between replays
                evals.append(tr.eval_step(store, idx[:B])[0].item())
        replayed = any(g[1] is not None for g in tr._graphs.values())
        return {n: p.detach().clone() for n, p in m.named_parameters()}, losses + evals, replayed, tr

    pe, le, re_, _ = run(False)
    pg, lg, rg, tr = run(True)
    assert rg and not re_                                   # steps 3.. of the second run were graph replays
    assert int(tr.step_dev.item()) == tr.step_count == 7
    assert len(le) == len(lg) == (9 if kind == "groundlink_eval" else 7)
    for a, b in zip(le, lg):
        assert abs(a - b) <= 1e-4 * abs(a), (le, lg)
    for n in pe:
        assert (pe[n] - pg[n]).abs().max().item() <= 2e-5, n
