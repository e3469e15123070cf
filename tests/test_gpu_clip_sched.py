"""Global-norm gradient clipping and the learning-rate schedule on a B200: the norm kernel against an fp64 oracle, the
scheduled optimizer against the unscheduled entry points (bit for bit) and a one-step fp64 oracle, the Trainer against
torch's clip_grad_norm_ + torch.optim + LambdaLR for the three models, graph replay with a learning rate that changes every
step, resume mid-warm-up, the CLI, and two data-parallel ranks."""
import math
import os
import subprocess
import sys

import pytest
import torch

from test_gpu_models import _small_denoiser

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = ["rmsprop", "adam", "sgd", "adagrad", "adadelta", "adamax"]


def _lam(n, W, cosine, S, r):
    """The schedule as the feature defines it, written out independently of the package."""
    if W > 0 and n <= W:
        return n / W
    if not cosine:
        return 1.0
    p = min(max((n - W) / (S - W), 0.0), 1.0)
    return r + (1 - r) * 0.5 * (1 + math.cos(math.pi * p))


# ---------------------------------------- norm kernel -----------------------------------------------------------------
def _norm_oracle(g, scale, max_norm):
    total = scale * g.double().pow(2).sum().sqrt().item()
    t32 = torch.tensor(total, dtype=torch.float32)
    coef = torch.clamp(torch.tensor(max_norm, dtype=torch.float32) / (t32 + 1e-6), max=1.0)
    return total, coef.item()


@pytest.mark.parametrize("n", [1, 3, 4097, 10007, "denoiser"])
def test_norm_kernel_matches_fp64_and_repeats_bit_for_bit(n):
    """Sizes 1, 3 (no float4 body), 4097 and 10 007 (a body and a tail) and the 25.9 M-parameter arena of the configs[1]
    denoiser (larger than L2), at grad_scale 1 and 0.5 (a 2-rank average).  Rel. 1e-6 against fp64; a second launch on the
    same arena gives the same two floats bit for bit; a cap above the norm gives a coefficient of exactly 1."""
    from inferbiomechanics_b200 import ops
    if n == "denoiser":
        from inferbiomechanics_b200.models.DiffusionDenoiser import DiffusionDenoiser
        m = DiffusionDenoiser(frames=50, d_model=512, num_heads=8, dim_feedforward=2048, num_layers=8).cuda()
        g = m.arena.grad
        assert g.numel() > 25_000_000
        g.normal_(generator=torch.Generator("cuda").manual_seed(1))
        g.mul_(1e-3)
    else:
        g = torch.randn(n, generator=torch.Generator().manual_seed(n)).cuda()
    ws = ops.GradClipWorkspace("cuda")
    for scale in (1.0, 0.5):
        total, _ = _norm_oracle(g, scale, 1.0)
        for max_norm in (0.25 * total, 4.0 * total):
            out = ops.grad_clip_coef(g, max_norm, scale, ws).clone()
            again = ops.grad_clip_coef(g, max_norm, scale, ws).clone()
            assert torch.equal(out, again)
            ref_total, ref_coef = _norm_oracle(g, scale, max_norm)
            assert abs(out[0].item() - ref_total) <= 1e-6 * ref_total, (out[0].item(), ref_total)
            assert abs(out[1].item() - ref_coef) <= 1e-6 * ref_coef, (out[1].item(), ref_coef)
            if max_norm > total:
                assert out[1].item() == 1.0
            else:
                assert out[1].item() < 0.26
    rec = ws.record.tolist()
    assert rec[1] == 8 and rec[2] == 4                 # 8 launches, the 4 with the cap at a quarter of the norm clipped
    assert ws.counter.item() == 0                      # the last block left the counter ready for the next launch


def test_norm_kernel_rejects_bad_arguments():
    from inferbiomechanics_b200 import ops
    g = torch.zeros(65, device="cuda")
    with pytest.raises(ValueError):
        ops.grad_clip_coef(g, 0.0)
    with pytest.raises(ValueError):
        ops.grad_clip_coef(g[1:], 1.0)                 # not 16-byte aligned


# ---------------------------------------- scheduled optimizer ---------------------------------------------------------
def _step64(kind, p, g, s0, s1, lr, n):
    """One torch-default step of ``kind`` in fp64 (the optimizer kernel's update rules)."""
    if kind == "rmsprop":
        s0 = 0.99 * s0 + 0.01 * g * g
        return p - lr * g / (s0.sqrt() + 1e-8), s0, s1
    if kind == "adam":
        s0 = 0.9 * s0 + 0.1 * g
        s1 = 0.999 * s1 + 0.001 * g * g
        bc1, bc2 = 1 - 0.9 ** n, 1 - 0.999 ** n
        return p - (lr / bc1) * s0 / (s1.sqrt() / math.sqrt(bc2) + 1e-8), s0, s1
    if kind == "sgd":
        return p - lr * g, s0, s1
    if kind == "adagrad":
        s0 = s0 + g * g
        return p - lr * g / (s0.sqrt() + 1e-10), s0, s1
    if kind == "adadelta":
        s0 = 0.9 * s0 + 0.1 * g * g
        delta = (s1 + 1e-6).sqrt() / (s0 + 1e-6).sqrt() * g
        s1 = 0.9 * s1 + 0.1 * delta * delta
        return p - lr * delta, s0, s1
    s0 = 0.9 * s0 + 0.1 * g
    s1 = torch.maximum(0.999 * s1, g.abs() + 1e-8)
    return p - (lr / (1 - 0.9 ** n)) * s0 / s1, s0, s1


@pytest.mark.parametrize("scale", [0.5, 1.0 / 3.0])
@pytest.mark.parametrize("with_ema", [False, True])
@pytest.mark.parametrize("by_counter", [False, True])
@pytest.mark.parametrize("kind", KINDS)
def test_scheduled_optimizer_is_the_plain_step_at_unit_factors_and_matches_fp64(kind, by_counter, with_ema, scale):
    """20 steps on 10 007 parameters (a float4 body and a 3-element tail), grad_scale 0.5 (exact) and 1/3 (a 3-rank average:
    g * grad_scale rounds, so a product contracted differently in the two instantiations would show).
    (a) clip coefficient 1 and a constant schedule without warm-up: parameters, state, bf16 shadow and EMA equal those of
        ibm_optimizer_step / _dev / _ema bit for bit.
    (b) a coefficient in (0.3, 0.9) every step, 5 warm-up steps, then a cosine to lr_min at step 15 and the clamped tail: each
        step within 2e-6 of one fp64 step taken from the kernel's own previous parameters and state, at the rate lr * lam(n).
    By counter, the by-value step passed is wrong on purpose: only the device counter may matter."""
    from inferbiomechanics_b200 import ops
    n, lr = 10007, 1e-2
    g0 = torch.Generator().manual_seed(3)
    p0 = torch.randn(n, generator=g0).cuda()

    def arenas():
        return [p0.clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda"),
                torch.zeros(n, dtype=torch.bfloat16, device="cuda"), p0.clone() if with_ema else None]

    ref, got, sch = arenas(), arenas(), arenas()
    counter = torch.zeros(1, dtype=torch.int64, device="cuda")
    unit = torch.tensor([7.0, 1.0], device="cuda")
    clip = torch.zeros(2, device="cuda")
    ema_kw = lambda a: dict(ema=a[4], ema_decay=0.9 if with_ema else 0.0)       # noqa: E731
    for step in range(1, 21):
        grad = torch.randn(n, generator=g0).cuda()
        counter.fill_(step)
        dev = counter if by_counter else None
        val = 999 if by_counter else step
        ops.optimizer_step(kind, ref[0], grad, *ref[1:4], lr, scale, step, step_dev=dev, **ema_kw(ref))
        ops.optimizer_step(kind, got[0], grad, *got[1:4], lr, scale, val, step_dev=dev, clip=unit, schedule="constant",
                           **ema_kw(got))
        for a, b in zip(ref, got):
            if a is not None:
                assert torch.equal(a, b), (step, kind)

        coef = 0.3 + 0.6 * torch.rand(1, generator=g0).item()
        clip[1] = coef
        before = [t.double().cpu() for t in sch[:3]]
        ops.optimizer_step(kind, sch[0], grad, *sch[1:4], lr, scale, val, step_dev=dev, clip=clip, schedule="cosine", warmup_steps=5,
                           total_steps=15, lr_min=1e-3, **ema_kw(sch))
        g64 = (grad.double().cpu() * float(torch.tensor(scale, dtype=torch.float32))) * float(torch.tensor(coef, dtype=torch.float32))
        lr_n = lr * _lam(step, 5, True, 15, 0.1)
        p, s0, s1 = _step64(kind, before[0], g64, before[1], before[2], lr_n, step)
        err = (sch[0].double().cpu() - p).abs().max().item()
        assert err <= 2e-6, (step, kind, err)
        for got_s, want in ((sch[1], s0), (sch[2], s1)):
            if kind != "sgd":
                e = (got_s.double().cpu() - want).abs().max().item()
                assert e <= 2e-6 * max(1.0, want.abs().max().item()), (step, kind, e)
    assert not torch.equal(sch[0], ref[0])


def test_scheduled_optimizer_rejects_bad_arguments():
    from inferbiomechanics_b200 import ops
    p, g, s = (torch.zeros(64, device="cuda") for _ in range(3))
    bad = [dict(schedule="cosine", warmup_steps=5, total_steps=5), dict(schedule="cosine", total_steps=0),
           dict(schedule="constant", warmup_steps=-1), dict(schedule="constant", lr_min=1e-2), dict(schedule="constant", lr_min=-1.0),
           dict(schedule="linear")]
    for kw in bad:
        with pytest.raises(ValueError):
            ops.optimizer_step("rmsprop", p, g, s, None, None, 1e-3, 1.0, 1, **kw)
    with pytest.raises(ValueError):
        ops.optimizer_step("rmsprop", p, g, s, None, None, 1e-3, 1.0, 1, schedule="constant", ema=torch.zeros(64, device="cuda"),
                           ema_decay=1.0)


# ---------------------------------------- end to end against torch ----------------------------------------------------
STEPS, W, MAX_NORM = 12, 4, 1e-3


def _flags(lr, lr_min):
    return dict(clip_grad_norm=MAX_NORM, lr_warmup_steps=W, lr_schedule="cosine", total_steps=STEPS, lr_min=lr_min)


def _torch_opt(params, cls, lr, lr_min):
    opt = cls(params, lr=lr)
    return opt, torch.optim.lr_scheduler.LambdaLR(opt, lambda s: _lam(s + 1, W, True, STEPS, lr_min / lr))


@pytest.mark.parametrize("kind", ["feedforward", "groundlink"])
def test_trainer_matches_module_loop_with_clipping_and_schedule(kind, monkeypatch):
    """12 graph-replayed steps (two eager, one capture, nine replays) with clipping active on every step, a 4-step warm-up and
    a cosine to lr_min, against the drop-in module on the same weights and windows through autograd, clip_grad_norm_,
    torch.optim.SGD and LambdaLR.  Same kernels, so losses agree to 2e-3 and the parameters and BatchNorm buffers to the
    bar of the unclipped module-loop tests (1e-3 of each tensor's scale); the pre-clip norm the Trainer reports each step is
    clip_grad_norm_'s to 2e-3."""
    from inferbiomechanics_b200.data.window_store import WindowStore
    from inferbiomechanics_b200.keys import LOSS_QUANTITIES, MODEL_INPUT_ORDER
    from inferbiomechanics_b200.loss.RegressionLossEvaluator import RegressionLossEvaluator
    from inferbiomechanics_b200.models.FeedForwardRegressionBaseline import FeedForwardBaseline
    from inferbiomechanics_b200.models.Groundlink import Groundlink
    from inferbiomechanics_b200.trainer import ALL_COMPONENTS, Trainer
    monkeypatch.setenv("IBM_TRAIN_GRAPHS", "1")
    if kind == "feedforward":
        T, B, lr = 50, 64, 2.0
        store = WindowStore.synthetic(STEPS * B, T, 5, 147, "all_frames", seed=3, trial_len=400)
        torch.manual_seed(2)
        make = lambda: FeedForwardBaseline(23, 2, T, "all_frames", "tanh", 5, 10, hidden_dims=[64, 32],  # noqa: E731
                                           batchnorm=True).cuda().train()
        widths = [23, 23, 23, 3, 3, 3, 3, 36, 15, 15]
    else:
        T, B, lr = 20, 8, 2.0
        store = WindowStore.synthetic(STEPS * B + 8, T, 1, 177, "all_frames", seed=9, trial_len=120)
        torch.manual_seed(5)
        make = lambda: Groundlink(23, 12, 10, "all_frames", fc_dropout=0.0).cuda().train()  # noqa: E731
        widths = [23, 23, 23, 3, 3, 3, 3, 36, 30, 30]
    a, b = make(), make()
    b.load_state_dict(a.state_dict())
    init = {k: v.detach().clone() for k, v in b.state_dict().items()}
    tr = Trainer(a, opt_type="sgd", lr=lr, **_flags(lr, 0.1 * lr))
    opt, sched = _torch_opt(b.parameters(), torch.optim.SGD, lr, 0.1 * lr)
    ev = RegressionLossEvaluator(dataset=None, split="train", device="cuda")
    idx_all = store.shard(0, 1)
    for step in range(STEPS):
        idx = idx_all[step * B:(step + 1) * B]
        assert tr.current_lr() == pytest.approx(opt.param_groups[0]["lr"], rel=1e-12)
        res = tr.train_step(store, idx)
        st = tr.grad_norm_stats()
        x = store.pack_f32(idx)
        inputs = dict(zip(MODEL_INPUT_ORDER, torch.split(x, widths, dim=-1)))
        labels = dict(zip(LOSS_QUANTITIES, torch.split(store.labels(idx), [6, 6, 6, 12], dim=-1)))
        opt.zero_grad()
        loss = ev(inputs, b(inputs), labels, [], [], ALL_COMPONENTS)
        loss.backward()
        norm = torch.nn.utils.clip_grad_norm_(b.parameters(), MAX_NORM).item()
        opt.step()
        sched.step()
        assert res[0].item() == pytest.approx(loss.item(), rel=2e-3), step
        assert st["steps"] == 1 and st["clipped"] == 1 and norm > MAX_NORM
        assert st["mean_norm"] == pytest.approx(norm, rel=2e-3), step
    assert sum(g[1] is not None for g in tr._graphs.values()) == 1
    sa, sb = a.state_dict(), b.state_dict()
    for k in sa:
        if k.endswith("num_batches_tracked"):
            assert int(sa[k]) == int(sb[k]) == STEPS
            continue
        d0 = (sa[k].float() - sb[k].float()).abs().max().item()
        assert d0 <= 1e-3 * (sb[k].float().abs().max().item() + 1e-3), f"{k}: {d0}"
    moved = max((sb[k].float() - init[k].float()).abs().max().item() for k in sb if not k.endswith("num_batches_tracked"))
    assert moved > 1e-4


def test_denoiser_trainer_matches_torch_clip_adam_and_lambda_lr():
    """The denoiser's step draws its timesteps and noise on the device, so the oracle takes each step's allreduced gradient
    from the arena (its autograd parity is the subject of the denoiser tests) and applies torch's clip_grad_norm_, Adam and
    LambdaLR to an fp32 copy of the masters: 12 steps, clipping active on every step, within 2e-6 of the Trainer's masters,
    and the reported pre-clip norms are clip_grad_norm_'s to 1e-6."""
    from inferbiomechanics_b200.data.window_store import WindowStore
    from inferbiomechanics_b200.trainer import Trainer
    m, _ = _small_denoiser(F=10, L=2)
    store = WindowStore.synthetic(2048, 10, 1, 177, "all_frames", seed=3, trial_len=300)
    lr = 2e-3
    tr = Trainer(m, opt_type="adam", lr=lr, seed=11, **_flags(lr, 1e-4))
    q = torch.nn.Parameter(tr.arena.master.detach().clone())
    opt, sched = _torch_opt([q], torch.optim.Adam, lr, 1e-4)
    idx_all = store.shard(0, 1)
    for step in range(STEPS):
        tr.train_step(store, idx_all[(step % 8) * 32:(step % 8 + 1) * 32])
        st = tr.grad_norm_stats()
        q.grad = tr.arena.grad.detach().clone()
        norm = torch.nn.utils.clip_grad_norm_([q], MAX_NORM).item()
        opt.step()
        sched.step()
        assert st["clipped"] == 1 and st["mean_norm"] == pytest.approx(norm, rel=1e-6), step
        err = (tr.arena.master - q.detach()).abs().max().item()
        assert err <= 2e-6, (step, err)


@pytest.mark.parametrize("kind", ["feedforward", "groundlink"])
def test_graph_replay_equals_eager_with_a_changing_rate_and_captures_once(kind, monkeypatch):
    """With the learning rate changing every step (warm-up, then cosine) and clipping on, the replayed run's masters equal the
    eager run's (2e-5: fp32 reduce-add order of split-K weight gradients), and the step is captured once for the whole run."""
    from test_gpu_ema import _batch, _setup
    from inferbiomechanics_b200.trainer import Trainer
    captures = []
    real = Trainer._capture_step
    monkeypatch.setattr(Trainer, "_capture_step", lambda self, *a: captures.append(1) or real(self, *a))

    def run(graphs):
        monkeypatch.setenv("IBM_TRAIN_GRAPHS", "1" if graphs else "0")
        m, store, B, opt = _setup(kind)
        tr = Trainer(m, opt_type=opt, lr=1e-3, seed=9, **_flags(1e-3, 1e-4))
        for i in range(STEPS):
            tr.train_step(store, _batch(store, B, i))
        torch.cuda.synchronize()
        return tr

    te = run(False)
    assert not captures
    tg = run(True)
    assert len(captures) == 1 and sum(g[1] is not None for g in tg._graphs.values()) == 1
    assert int(tg.step_dev.item()) == tg.step_count == STEPS
    assert (te.arena.master - tg.arena.master).abs().max().item() <= 2e-5
    assert te.grad_norm_stats()["clipped"] == tg.grad_norm_stats()["clipped"] == STEPS


def test_huge_cap_without_schedule_is_bit_identical_to_options_off():
    """Two Trainers on the same FeedForward weights (Adam, EMA on), one with a cap of 1e30 and a constant schedule without
    warm-up: fed the same gradients through the Trainer's optimizer step, masters, state, shadow and EMA stay bit-identical
    (the coefficient is exactly 1 and lam = 1)."""
    from test_gpu_ema import _setup
    from inferbiomechanics_b200 import ops
    from inferbiomechanics_b200.trainer import Trainer
    trs = []
    for on in (False, True):
        m, _, _, _ = _setup("feedforward")
        trs.append(Trainer(m, opt_type="adam", lr=1e-3, seed=9, ema_decay=0.9, **(dict(clip_grad_norm=1e30) if on else {})))
    g = torch.Generator("cuda").manual_seed(4)
    for _ in range(6):
        grad = torch.randn(trs[0].arena.grad.numel(), device="cuda", generator=g)
        for tr in trs:
            tr.arena.grad.copy_(grad)
            ops.counter_add(tr.step_dev, 1)
            tr.optimizer_step()
    a, b = trs
    for x, y in ((a.arena.master, b.arena.master), (a.arena.shadow, b.arena.shadow), (a.state0, b.state0), (a.state1, b.state1),
                 (a.ema, b.ema)):
        assert torch.equal(x, y)
    assert b.grad_norm_stats()["clipped"] == 0 and not torch.equal(a.arena.master, a.ema)


def test_resume_mid_warmup_continues_the_schedule(tmp_path):
    """A checkpoint after 3 of 6 warm-up steps, resumed into a fresh Trainer, continues to step 12 like an uninterrupted run
    (2e-5), and its param_groups[0] holds LambdaLR's rate for step 4 and the base rate."""
    from test_gpu_ema import _batch, _setup
    from inferbiomechanics_b200.trainer import Trainer
    flags = dict(clip_grad_norm=MAX_NORM, lr_warmup_steps=6, lr_schedule="cosine", total_steps=STEPS, lr_min=1e-4)
    m, store, B, opt = _setup("feedforward")
    ta = Trainer(m, opt_type=opt, lr=1e-3, seed=9, **flags)
    for i in range(STEPS):
        ta.train_step(store, _batch(store, B, i))
    m1, _, _, _ = _setup("feedforward")
    t1 = Trainer(m1, opt_type=opt, lr=1e-3, seed=9, **flags)
    for i in range(3):
        t1.train_step(store, _batch(store, B, i))
    path = str(tmp_path / "epoch_0_batch_2.pt")
    torch.save({"epoch": 0, "model_state_dict": m1.state_dict(), "optimizer_state_dict": t1.optimizer_state_dict()}, path)
    ck = torch.load(path, map_location="cpu")
    p = torch.nn.Parameter(torch.zeros(1))
    o = torch.optim.Adam([p], lr=1e-3)
    s = torch.optim.lr_scheduler.LambdaLR(o, lambda k: _lam(k + 1, 6, True, STEPS, 0.1))
    for _ in range(3):
        p.grad = torch.zeros(1)
        o.step()
        s.step()
    group = ck["optimizer_state_dict"]["param_groups"][0]
    assert group["lr"] == pytest.approx(o.param_groups[0]["lr"], rel=1e-12) and group["initial_lr"] == 1e-3
    assert ck["optimizer_state_dict"]["ibm_b200"]["lr_warmup_steps"] == 6
    m2, _, _, _ = _setup("feedforward", seed=1)
    m2.load_state_dict(ck["model_state_dict"])
    t2 = Trainer(m2, opt_type=opt, lr=1e-3, seed=9, **flags)
    t2.load_optimizer_state_dict(ck["optimizer_state_dict"])
    t2.arena.sync_shadow(force=True)
    assert t2.step_count == 3 and t2.current_lr() == pytest.approx(group["lr"], rel=1e-12)
    for i in range(3, STEPS):
        t2.train_step(store, _batch(store, B, i))
    assert (ta.arena.master - t2.arena.master).abs().max().item() <= 2e-5


# ---------------------------------------- CLI -------------------------------------------------------------------------
def test_cli_train_with_clipping_and_cosine(tmp_path, capsys):
    from test_gpu_ema import _latest, _run
    ck = str(tmp_path / "ck")
    ff = ["--no-wandb", "--synthetic-windows", "1024", "--checkpoint-dir", ck, "--history-len", "50", "--stride", "5",
          "--hidden-dims", "64", "64", "--activation", "relu", "--model-type", "feedforward", "--batch-size", "32",
          "--learning-rate", "1e-3"]
    _run(["train", *ff, "--epochs", "2", "--max-batches", "6", "--clip-grad-norm", "1e-3", "--lr-warmup-steps", "4",
          "--lr-schedule", "cosine", "--lr-min", "1e-5"])
    out = capsys.readouterr().out
    lines = [ln for ln in out.splitlines() if "Gradient norm before clipping" in ln]
    assert len(lines) == 2 and all("over 6 steps, 6 clipped" in ln for ln in lines), lines
    sd = _latest(ck, "feedforward")["optimizer_state_dict"]
    assert sd["ibm_b200"] == {"opt_type": "rmsprop", "step": 12, "clip_grad_norm": 1e-3, "lr_warmup_steps": 4,
                              "lr_schedule": "cosine", "lr_min": 1e-5, "total_steps": 12}
    assert sd["param_groups"][0]["lr"] == pytest.approx(1e-5, rel=1e-9) and sd["param_groups"][0]["initial_lr"] == 1e-3

    dif = ["--no-wandb", "--synthetic-windows", "512", "--checkpoint-dir", ck, "--history-len", "50", "--stride", "1",
           "--model-type", "diffusion", "--batch-size", "64"]
    _run(["train", *dif, "--epochs", "1", "--max-batches", "3", "--clip-grad-norm", "1", "--lr-warmup-steps", "2"])
    assert "Gradient norm before clipping" in capsys.readouterr().out
    with pytest.raises(ValueError, match="--lr-warmup-steps"):
        _run(["train", *dif, "--epochs", "1", "--max-batches", "3", "--lr-schedule", "cosine", "--lr-warmup-steps", "3",
              "--checkpoint-dir", str(tmp_path / "other")])

    gl = ["--no-wandb", "--synthetic-windows", "512", "--checkpoint-dir", ck, "--history-len", "50", "--stride", "1",
          "--model-type", "groundlink"]
    _run(["train", *gl, "--epochs", "1", "--max-batches", "3", "--batch-size", "16"])
    assert "Gradient norm" not in capsys.readouterr().out
    sd = _latest(ck, "groundlink")["optimizer_state_dict"]
    assert sd["ibm_b200"] == {"opt_type": "rmsprop", "step": 3} and "initial_lr" not in sd["param_groups"][0]


# ---------------------------------------- data parallel ---------------------------------------------------------------
@pytest.mark.parametrize("mode,graphs", [("overlap", "0"), ("tail", "0"), ("tail", "1")])
def test_two_ranks_stay_bit_identical_with_clipping(tmp_path, mode, graphs):
    """Clipping active on every step (and a warm-up + cosine): both ranks compute the coefficient from the same reduced
    gradient, so masters and {total, coefficient} are bit-identical after every step, with overlapped buckets, one tail
    allreduce, and the data-parallel step replayed from its two graphs."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    worker = os.path.join(ROOT, "tests", "workers", "clip_sched_rank_worker.py")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", IBM_ALLREDUCE=mode, IBM_TRAIN_GRAPHS=graphs)
    port = {"overlap": 29741, "tail": 29742}[mode] + 2 * int(graphs)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), worker, str(tmp_path), "6", "64"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stderr[-3000:]
    ranks = [torch.load(os.path.join(tmp_path, f"rank{i}.pt")) for i in range(2)]
    assert ranks[0]["graphs"] == (1 if graphs == "1" else 0)
    for s in range(6):
        assert torch.equal(ranks[0]["master"][s], ranks[1]["master"][s]), f"masters differ after step {s + 1}"
        assert torch.equal(ranks[0]["clip"][s], ranks[1]["clip"][s]), f"clip record differs after step {s + 1}"
        assert ranks[0]["clip"][s][1].item() < 1.0
    assert ranks[0]["stats"]["clipped"] == 6
