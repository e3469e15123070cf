"""Exponential moving average of the weights on a B200: the EMA instantiation of the fused optimizer kernel against the
non-EMA entry points (bit for bit) and an fp64 oracle, graph-replayed steps, ``Trainer.ema_weights()`` for the three models
(every weight cache follows the swap both ways), checkpoint resume, the CLI, and two data-parallel ranks."""
import os
import subprocess
import sys

import pytest
import torch

from test_gpu_models import _small_denoiser

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = ["rmsprop", "adam", "sgd", "adagrad", "adadelta", "adamax"]


# ---------------------------------------- kernel ----------------------------------------------------------------------
@pytest.mark.parametrize("by_counter", [False, True])
@pytest.mark.parametrize("kind", KINDS)
def test_ema_kernel_leaves_the_update_alone_and_matches_fp64_oracle(kind, by_counter):
    """20 steps on 10 007 parameters (a float4 body and a 3-element tail).  Parameters, state and bf16 shadow equal those of
    the non-EMA entry point bit for bit.  The EMA follows e += (1 - d_n)(p_n - e), d_n = min(decay, (1 + n)/(10 + n)), in
    fp64 on the kernel's own parameters: decay 0.5 covers the warm-up (d_1..d_3 = 2/11, 3/12, 4/13) and the cap (n >= 8).
    Bar: 2e-6 absolute on |e| <~ 4: about one fp32 rounding of |e| per step, damped by the contraction d_n <= 0.5."""
    from inferbiomechanics_b200 import ops
    n, decay = 10007, 0.5
    g = torch.Generator().manual_seed(3)
    p0 = torch.randn(n, generator=g).cuda()
    ref = [p0.clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda"), torch.zeros(n, dtype=torch.bfloat16, device="cuda")]
    got = [t.clone() for t in ref]
    ema = p0.clone()
    oracle = p0.double().cpu()
    counter = torch.zeros(1, dtype=torch.int64, device="cuda")
    for step in range(1, 21):
        grad = torch.randn(n, generator=g).cuda()
        counter.fill_(step)
        dev = counter if by_counter else None
        ops.optimizer_step(kind, ref[0], grad, ref[1], ref[2], ref[3], 1e-2, 0.5, step, step_dev=dev)
        # by counter: a wrong by-value step must not matter
        ops.optimizer_step(kind, got[0], grad, got[1], got[2], got[3], 1e-2, 0.5, 999 if by_counter else step, step_dev=dev,
                           ema=ema, ema_decay=decay)
        for a, b in zip(ref, got):
            assert torch.equal(a, b), step
        d = min(float(torch.tensor(decay, dtype=torch.float32)), (1.0 + step) / (10.0 + step))
        oracle = oracle + (1.0 - d) * (got[0].double().cpu() - oracle)
        err = (ema.double().cpu() - oracle).abs().max().item()
        assert err <= 2e-6, (step, err)
    assert (ema - got[0]).abs().max().item() > 1e-5                   # the average lags the parameters (Adadelta's by ~1e-4)


def test_ema_entry_point_rejects_bad_arguments():
    from inferbiomechanics_b200 import ops
    p, g, s = (torch.zeros(64, device="cuda") for _ in range(3))
    for decay in (0.0, 1.0, -0.5):
        with pytest.raises(ValueError):
            ops.optimizer_step("rmsprop", p, g, s, None, None, 1e-3, 1.0, 1, ema=torch.zeros(64, device="cuda"), ema_decay=decay)
    with pytest.raises(ValueError):                                  # not 16-byte aligned
        ops.optimizer_step("rmsprop", p, g, s, None, None, 1e-3, 1.0, 1, ema=torch.zeros(65, device="cuda")[1:], ema_decay=0.9)
    with pytest.raises(ValueError):                                  # wrong size
        ops.optimizer_step("rmsprop", p, g, s, None, None, 1e-3, 1.0, 1, ema=torch.zeros(32, device="cuda"), ema_decay=0.9)


# ---------------------------------------- models ----------------------------------------------------------------------
def _setup(kind, seed=0):
    """(model, store, batch size, optimizer) for the three trained model families at small shapes."""
    from inferbiomechanics_b200.data.window_store import WindowStore
    from inferbiomechanics_b200.models.FeedForwardRegressionBaseline import FeedForwardBaseline
    from inferbiomechanics_b200.models.Groundlink import Groundlink
    torch.manual_seed(seed)
    if kind == "feedforward":
        m = FeedForwardBaseline(23, 2, 50, "all_frames", "relu", 5, 10, hidden_dims=[64, 64], batchnorm=True, dropout=True,
                                dropout_prob=0.25).cuda().train()
        return m, WindowStore.synthetic(1024, 50, 5, 147, "all_frames", seed=3, device="cuda"), 32, "adam"
    if kind == "groundlink":
        m = Groundlink(23, 12, 10, "all_frames").cuda().train()
        return m, WindowStore.synthetic(512, 20, 1, 177, "all_frames", seed=3, device="cuda"), 16, "rmsprop"
    m, _ = _small_denoiser(F=10, L=2, seed=5 + seed)
    return m, WindowStore.synthetic(2048, 10, 1, 177, "all_frames", seed=3, device="cuda"), 32, "adam"


def _batch(store, B, i):
    idx = store.shard(0, 1)
    return idx[(i % 4) * B:(i % 4 + 1) * B]


def _cond(m, B):
    eng = m.engine()
    eng.xc(B, False)[:, 30:30 + eng.c_in] = torch.randn(B * eng.F, eng.c_in, device="cuda",
                                                       generator=torch.Generator("cuda").manual_seed(B)).to(torch.bfloat16)


@pytest.mark.parametrize("kind,opt", [("feedforward", "adam"), ("groundlink", "rmsprop")])
def test_graph_replayed_ema_equals_eager(monkeypatch, kind, opt):
    """Captured FeedForward (dropout + BatchNorm) and Groundlink steps replay with the EMA decay of the step the device counter
    holds: the replayed run's EMA equals the eager run's (2e-5: fp32 reduce-add order of split-K weight gradients)."""
    from inferbiomechanics_b200.trainer import Trainer

    def run(graphs):
        monkeypatch.setenv("IBM_TRAIN_GRAPHS", "1" if graphs else "0")
        m, store, B, _ = _setup(kind)
        tr = Trainer(m, opt_type=opt, lr=1e-3, seed=9, ema_decay=0.9)
        for i in range(7):
            tr.train_step(store, _batch(store, B, i))
        torch.cuda.synchronize()
        return tr, any(g[1] is not None for g in tr._graphs.values())

    te, re_ = run(False)
    tg, rg = run(True)
    assert rg and not re_
    assert int(tg.step_dev.item()) == tg.step_count == 7
    assert (te.ema - tg.ema).abs().max().item() <= 2e-5
    assert (tg.ema - tg.arena.master).abs().max().item() > 1e-5


def _evaluate(kind, tr, store, B):
    """eval_step's fp32[40] result (FeedForward, Groundlink), or a 4-step DDIM sample with a fixed seed (denoiser)."""
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    tr.model.eval()
    try:
        if kind == "diffusion":
            _cond(tr.model, B)
            if not hasattr(tr, "_test_gd"):
                tr._test_gd = GaussianDiffusion(device="cuda")
            return tr._test_gd.sample(tr.model, B, seed=21, ddim_steps=4)
        return tr.eval_step(store, _batch(store, B, 1)).clone()
    finally:
        tr.model.train()


@pytest.mark.parametrize("kind", ["feedforward", "groundlink", "diffusion"])
def test_ema_weights_swap_evaluates_the_average_and_restores_everything(kind):
    """Inside ``ema_weights()`` the evaluation equals that of a fresh model loaded with ``ema_state_dict()`` and differs from
    the raw-weight one; after exit master and shadow are bit-identical to before and a raw-weight evaluation repeats
    (for the denoiser: the time-MLP table and the sampling graph were rebuilt both ways).  Training around a swap equals
    training straight through."""
    from inferbiomechanics_b200.trainer import Trainer
    m, store, B, opt = _setup(kind)
    tr = Trainer(m, opt_type=opt, lr=1e-3, seed=9, ema_decay=0.9)
    for i in range(3):
        tr.train_step(store, _batch(store, B, i))
    raw = _evaluate(kind, tr, store, B)
    master, shadow = tr.arena.master.clone(), tr.arena.shadow.clone()
    with tr.ema_weights():
        with pytest.raises(RuntimeError):
            with tr.ema_weights():
                pass
        avg = _evaluate(kind, tr, store, B)
    assert torch.equal(tr.arena.master, master) and torch.equal(tr.arena.shadow, shadow)
    torch.testing.assert_close(_evaluate(kind, tr, store, B), raw, rtol=1e-6, atol=1e-7)
    assert (avg - raw).abs().max().item() > 1e-4

    f, _, _, _ = _setup(kind, seed=1)                                # different init: everything comes from the state dict
    f.load_state_dict(tr.ema_state_dict())
    tf = Trainer(f, opt_type=opt, lr=1e-3, seed=9)
    torch.testing.assert_close(_evaluate(kind, tf, store, B), avg, rtol=1e-5, atol=1e-6)

    for i in range(3, 6):
        tr.train_step(store, _batch(store, B, i))
    m2, _, _, _ = _setup(kind)
    t2 = Trainer(m2, opt_type=opt, lr=1e-3, seed=9, ema_decay=0.9)
    for i in range(6):
        t2.train_step(store, _batch(store, B, i))
    assert (tr.arena.master - t2.arena.master).abs().max().item() <= 2e-5
    assert (tr.ema - t2.ema).abs().max().item() <= 2e-5


def test_ema_weights_needs_an_ema():
    from inferbiomechanics_b200.trainer import Trainer
    m, _, _, _ = _setup("feedforward")
    tr = Trainer(m, opt_type="adam", lr=1e-3)
    with pytest.raises(RuntimeError):
        with tr.ema_weights():
            pass
    with pytest.raises(RuntimeError):
        tr.ema_state_dict()


@pytest.mark.parametrize("kind", ["feedforward", "groundlink"])
def test_resume_with_ema_continues_the_uninterrupted_run(tmp_path, kind):
    """Save model, optimizer and EMA after 3 steps, resume into a fresh Trainer, take 3 more: parameters and EMA equal those of
    6 uninterrupted steps (2e-5), the warm-up continuing from the restored step count.  A checkpoint without an EMA resumes
    with the average restarted at the loaded weights."""
    from inferbiomechanics_b200.trainer import Trainer
    m, store, B, opt = _setup(kind)
    ta = Trainer(m, opt_type=opt, lr=1e-3, seed=9, ema_decay=0.99)
    for i in range(6):
        ta.train_step(store, _batch(store, B, i))
    m1, _, _, _ = _setup(kind)
    t1 = Trainer(m1, opt_type=opt, lr=1e-3, seed=9, ema_decay=0.99)
    for i in range(3):
        t1.train_step(store, _batch(store, B, i))
    path = str(tmp_path / "epoch_0_batch_2.pt")
    torch.save({"epoch": 0, "model_state_dict": m1.state_dict(), "optimizer_state_dict": t1.optimizer_state_dict(),
                "ema_state_dict": t1.ema_state_dict()}, path)
    ck = torch.load(path, map_location="cpu")
    m2, _, _, _ = _setup(kind, seed=1)
    m2.load_state_dict(ck["model_state_dict"])
    t2 = Trainer(m2, opt_type=opt, lr=1e-3, seed=9, ema_decay=0.99)
    t2.load_optimizer_state_dict(ck["optimizer_state_dict"])
    t2.arena.sync_shadow(force=True)
    t2.load_ema_state_dict(ck["ema_state_dict"])
    assert t2.step_count == 3 and torch.equal(t2.ema, t1.ema)
    for i in range(3, 6):
        t2.train_step(store, _batch(store, B, i))
    assert (ta.arena.master - t2.arena.master).abs().max().item() <= 2e-5
    assert (ta.ema - t2.ema).abs().max().item() <= 2e-5
    with pytest.raises(ValueError):
        t2.load_ema_state_dict({k: v for k, v in ck["ema_state_dict"].items() if k != t2.arena.names[0]})

    m3, _, _, _ = _setup(kind, seed=1)
    m3.load_state_dict(ck["model_state_dict"])
    t3 = Trainer(m3, opt_type=opt, lr=1e-3, seed=9, ema_decay=0.99)
    t3.load_ema_state_dict(None)
    assert torch.equal(t3.ema, t3.arena.master) and torch.equal(t3.ema, t1.arena.master)


# ---------------------------------------- CLI -------------------------------------------------------------------------
def _run(argv):
    from inferbiomechanics_b200.main import main
    return main(argv)


def _latest(ck, kind):
    d = os.path.join(ck, kind)
    files = sorted(os.listdir(d), key=lambda x: (int(x.split("_")[1]), int(x.split("_")[3].split(".")[0])))
    return torch.load(os.path.join(d, files[-1]), map_location="cpu")


def test_cli_train_with_ema_and_analyze_with_ema(tmp_path, capsys):
    ck = str(tmp_path / "ck")
    ff = ["--no-wandb", "--synthetic-windows", "1024", "--checkpoint-dir", ck, "--history-len", "50", "--stride", "5",
          "--hidden-dims", "64", "64", "--activation", "relu", "--model-type", "feedforward"]
    _run(["train", *ff, "--epochs", "2", "--batch-size", "32", "--learning-rate", "1e-3", "--ema-decay", "0.99"])
    sd = _latest(ck, "feedforward")
    assert set(sd) == {"epoch", "model_state_dict", "optimizer_state_dict", "ema_state_dict"}
    assert list(sd["ema_state_dict"]) == list(sd["model_state_dict"])
    assert "Dev Set Evaluation (EMA weights)" in capsys.readouterr().out
    grf = ["--predict-grf-components", "0", "1", "2", "3", "4", "5"]
    raw = _run(["analyze", *ff, *grf]).last_reports
    avg = _run(["analyze", *ff, *grf, "--ema"]).last_reports
    assert avg["dev"]["loss"] > 0 and avg["dev"]["loss"] != raw["dev"]["loss"]

    dif = ["--no-wandb", "--synthetic-windows", "512", "--checkpoint-dir", ck, "--history-len", "50", "--stride", "1",
           "--model-type", "diffusion"]
    _run(["train", *dif, "--epochs", "1", "--max-batches", "3", "--batch-size", "64", "--ema-decay", "0.99"])
    assert "ema_state_dict" in _latest(ck, "diffusion")
    an = ["analyze", *dif, "--batch-size", "64", "--sampler", "ddim", "--sampling-steps", "4", "--predict-grf-components", "0", "1", "2"]
    raw = _run(an).last_reports
    avg = _run([*an, "--ema"]).last_reports
    assert avg["dev"]["loss"] > 0 and avg["dev"]["loss"] != raw["dev"]["loss"]

    gl = ["--no-wandb", "--synthetic-windows", "512", "--checkpoint-dir", ck, "--history-len", "50", "--stride", "1",
          "--model-type", "groundlink"]
    _run(["train", *gl, "--epochs", "1", "--max-batches", "3", "--batch-size", "16"])
    assert set(_latest(ck, "groundlink")) == {"epoch", "model_state_dict", "optimizer_state_dict"}
    with pytest.raises(ValueError, match="epoch_0_batch_2.pt"):
        _run(["analyze", *gl, "--ema"])
    # a run that turns the EMA on when resuming starts the average at the loaded weights
    _run(["train", *gl, "--epochs", "2", "--max-batches", "3", "--batch-size", "16", "--ema-decay", "0.9"])
    assert "ema_state_dict" in _latest(ck, "groundlink") and _latest(ck, "groundlink")["epoch"] == 1


# ---------------------------------------- data parallel ---------------------------------------------------------------
def test_two_ranks_keep_bit_identical_ema(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    worker = os.path.join(ROOT, "tests", "workers", "ema_rank_worker.py")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29737", worker, str(tmp_path), "4", "64"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stderr[-3000:]
    ranks = [torch.load(os.path.join(tmp_path, f"rank{i}.pt")) for i in range(2)]
    assert len(ranks[0]["ema"]) == 4
    for s, (a, b) in enumerate(zip(ranks[0]["ema"], ranks[1]["ema"])):
        assert torch.equal(a, b), f"EMA differs between ranks after step {s + 1}"
    assert not torch.equal(ranks[0]["ema"][-1], ranks[0]["master"])
