"""Classifier-free guidance on a B200: the condition-dropout kernel against the Philox oracle bit for bit, the Trainer with
condition dropout against a Trainer fed host-zeroed kinematics, the guided step kernel against an fp64 oracle, the guided
sampling loop against the CPU oracle loop, CUDA-graph replay, sharded sampling and the CLI.  The oracle (``tests/
cfg_oracle.py``) is builder-owned and parity unpinned, like all diffusion code here."""
import math
import os
import re
from collections import Counter

import numpy as np
import pytest
import torch

import cfg_oracle as ocfg
import ddim_oracle as odim
import philox_oracle as ph
from oracle import ddpm as oddpm
from oracle import models as om
from test_gpu_models import _small_denoiser, close

pytestmark = pytest.mark.gpu

SEED_MIX = 0x9E3779B1


def _bits(x):
    return x.view(torch.int16)


def _random_bf16(rows, ld, seed):
    """bf16 rows of arbitrary finite bit patterns (no NaN, so a changed byte cannot hide)."""
    g = torch.Generator("cuda").manual_seed(seed)
    return (torch.randn(rows, ld, device="cuda", generator=g) * 3).to(torch.bfloat16)


# ---------------------------------------- condition dropout kernel ----------------------------------------------------
@pytest.mark.parametrize("B,F,ld,col0,ncols,p,seed,offset", [
    (1, 10, 208, 30, 177, 0.5, 1, 0),
    (37, 10, 208, 30, 177, 0.1, 5, 3),
    (512, 50, 208, 30, 177, 0.3, 1234, 99),
    (300, 7, 210, 30, 177, 0.6, 2, (1 << 33) + 5),          # rows not 16-byte aligned: the element-wise path
    (64, 4, 64, 16, 32, 0.5, 9, 1),                         # a range of whole 8-column groups
    (513, 3, 208, 30, 177, 1.0, 0, 0),                      # p = 1 drops every window
])
def test_cond_dropout_kernel_matches_oracle(B, F, ld, col0, ncols, p, seed, offset):
    from inferbiomechanics_b200 import ops
    xc = _random_bf16(B * F, ld, B + F)
    before = xc.clone()
    keep_out = torch.full((B,), 7, dtype=torch.uint8, device="cuda")
    ops.cond_dropout(xc, B, F, col0, ncols, p, seed, offset, keep_out=keep_out)
    keep = ocfg.cond_keep(B, p, seed, offset)
    want = before.clone().view(B, F, ld)
    want[torch.from_numpy(~keep).cuda(), :, col0:col0 + ncols] = 0
    assert torch.equal(_bits(xc), _bits(want.view(B * F, ld))), "bytes differ from the oracle"
    assert np.array_equal(keep_out.cpu().numpy(), keep.astype(np.uint8))
    if p >= 1.0:
        assert not keep.any()
    elif B >= 37:
        assert keep.any() and not keep.all()
    # without the record the same windows are dropped
    xc2 = before.clone()
    ops.cond_dropout(xc2, B, F, col0, ncols, p, seed, offset)
    assert torch.equal(_bits(xc2), _bits(xc))


def test_cond_dropout_rejects_p_zero_without_launching():
    from inferbiomechanics_b200 import _lib, ops
    xc = torch.zeros(10, 208, dtype=torch.bfloat16, device="cuda")
    n = _lib.launch_count
    with pytest.raises(ValueError):
        ops.cond_dropout(xc, 1, 10, 30, 177, 0.0, 0, 0)
    assert _lib.launch_count == n


# ---------------------------------------- Trainer ---------------------------------------------------------------------
def _denoiser_setup():
    from inferbiomechanics_b200.data.window_store import WindowStore
    m, _ = _small_denoiser(F=10, L=2, seed=5)
    return m, WindowStore.synthetic(2048, 10, 1, 177, "all_frames", seed=3, device="cuda")


def _drop_seed(seed, rank=0):
    """The trainer's documented key: (COND_DROP_SEED ^ mixed trainer seed) + rank."""
    from inferbiomechanics_b200.trainer import Trainer
    return (Trainer.COND_DROP_SEED ^ ((seed * SEED_MIX) & 0x7FFFFFFF)) + rank


class _ZeroedStore:
    """A window store whose packed kinematics have, at step i, the windows the oracle drops zeroed."""

    def __init__(self, store, p, seed):
        self.store, self.p, self.seed, self.step = store, p, seed, 0

    def __getattr__(self, k):
        return getattr(self.store, k)

    def pack(self, idx, layout):
        self.store.pack(idx, layout)
        buf = layout[0]
        B = idx.numel()
        drop = torch.from_numpy(~ocfg.cond_keep(B, self.p, self.seed, self.step)).cuda()
        buf.view(B, self.store.F, -1)[drop, :, 30:207] = 0
        self.step += 1


STEPS, B = 6, 32


def _batch(store, i):
    return store.shard(0, 1)[(i % 8) * B:(i % 8 + 1) * B]


def _sync(dst, src):
    """Gives Trainer ``dst`` the weights and optimizer state of ``src``, bit for bit (the shadow, the padded copies and every
    weight cache re-derived, as ``Trainer.ema_weights`` does)."""
    dst.arena.master.copy_(src.arena.master)
    for d, s in ((dst.state0, src.state0), (dst.state1, src.state1)):
        if d is not None:
            d.copy_(s)
    dst.arena.sync_shadow(force=True)
    dst.arena.bump_version()


def _same_step(a, b, what):
    """The backward's fp32 reductions (split-K reduce-adds, atomics) are not ordered, so two runs of one denoiser step from the
    same weights on the same input rows agree on the forward bit for bit and on the gradient only to rounding; an adaptive
    optimizer then turns a rounding-level difference of a near-zero gradient entry into a full step, so trained masters are
    not compared.  The gradients are, to 1e-5 of their largest entry."""
    ga, gb = a.arena.grad, b.arena.grad
    d, scale = (ga - gb).abs().max().item(), ga.abs().max().item()
    assert d <= 1e-5 * scale, f"{what}: gradients differ by {d:.3g} (largest entry {scale:.3g})"


def test_trainer_with_condition_dropout_equals_zeroed_store():
    """Store path: every step, Trainer(cond_drop_prob=0.25) and Trainer() fed windows whose kinematics the oracle's masks zero
    start from the same weights, train on bit-identical input rows (x_t and condition), reach the same loss bit for bit and
    the same gradient to rounding; without dropout the rows, the loss and the gradient differ."""
    from inferbiomechanics_b200.trainer import Trainer
    p, seed = 0.25, 11
    trs = {}
    for kind in ("drop", "zeroed", "plain"):
        m, store = _denoiser_setup()
        trs[kind] = Trainer(m, opt_type="adam", lr=2e-3, seed=seed, cond_drop_prob=p if kind == "drop" else 0.0)
    src = {"drop": store, "zeroed": _ZeroedStore(store, p, _drop_seed(seed)), "plain": store}
    for i in range(STEPS):
        for k in ("zeroed", "plain"):
            _sync(trs[k], trs["drop"])
        loss = {k: tr.train_step(src[k], _batch(store, i))[0].item() for k, tr in trs.items()}
        rows = {k: tr.eng.xc(B, True) for k, tr in trs.items()}
        assert torch.equal(_bits(rows["drop"]), _bits(rows["zeroed"])), f"input rows differ at step {i}"
        assert loss["drop"] == loss["zeroed"], (i, loss)
        _same_step(trs["drop"], trs["zeroed"], f"step {i}")
        assert not torch.equal(rows["drop"], rows["plain"]) and loss["drop"] != loss["plain"], (i, loss)
        gd, gp = trs["drop"].arena.grad, trs["plain"].arena.grad
        assert (gd - gp).abs().max().item() > 1e-3 * gd.abs().max().item()


def test_host_fed_trainer_with_condition_dropout_equals_host_zeroed_batches():
    """Host-fed path (train_step_host): the same masks, with the reference's kinematics zeroed in the pinned host tensors;
    every step from the same weights, bit-identical input rows and loss, the same gradient to rounding."""
    from inferbiomechanics_b200.keys import MODEL_INPUT_ORDER
    from inferbiomechanics_b200.trainer import Trainer
    p, seed = 0.3, 4
    trs = []
    for drop in (True, False):
        m, _ = _denoiser_setup()
        trs.append(Trainer(m, opt_type="rmsprop", lr=1e-3, seed=seed, cond_drop_prob=p if drop else 0.0))
    ta, tb = trs
    for i in range(4):
        _sync(tb, ta)
        a, b = ta.make_host_batch(B, seed=100 + i), tb.make_host_batch(B, seed=100 + i)
        dropped = torch.from_numpy(~ocfg.cond_keep(B, p, _drop_seed(seed), i))
        assert dropped.any()
        for k in MODEL_INPUT_ORDER:
            b["inputs"][k][dropped] = 0.0
        la = ta.train_step_host(a["inputs"], a["labels"])
        lb = tb.train_step_host(b["inputs"], b["labels"])
        assert torch.equal(_bits(ta.eng.xc(B, True)), _bits(tb.eng.xc(B, True))), f"input rows differ at step {i}"
        assert la == lb, (i, la, lb)
        _same_step(ta, tb, f"step {i}")


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return Counter(e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)


def test_drop_probability_zero_launches_the_plain_step():
    from inferbiomechanics_b200.trainer import Trainer
    names = []
    for kw in ({}, {"cond_drop_prob": 0.0}, {"cond_drop_prob": 0.1}):
        m, store = _denoiser_setup()
        tr = Trainer(m, opt_type="adam", lr=1e-3, seed=3, **kw)
        tr.train_step(store, _batch(store, 0))
        names.append(_kernel_names(lambda: tr.train_step(store, _batch(store, 1))))
    assert names[0] == names[1]
    assert not any("cond_dropout" in k for k in names[0])
    extra = names[2] - names[0]
    assert sum(extra.values()) == 1 and "cond_dropout_kernel" in next(iter(extra)), extra
    assert not names[0] - names[2]


def test_resume_with_condition_dropout_continues_the_masks(tmp_path):
    """A checkpoint after 3 of 6 steps, resumed into a fresh Trainer, continues like the run that wrote it: the masks continue
    from the stored step count, so steps 4-6 train on bit-identical input rows, and step 4 (same weights) reaches the same loss
    bit for bit and the same gradient to rounding.  The timestep generator is not part of a checkpoint, so its state is carried
    over by hand."""
    from inferbiomechanics_b200.trainer import Trainer
    flags = dict(opt_type="adam", lr=2e-3, seed=7, cond_drop_prob=0.4)
    m1, store = _denoiser_setup()
    t1 = Trainer(m1, **flags)
    for i in range(3):
        t1.train_step(store, _batch(store, i))
    gen = t1._gen.get_state()
    path = str(tmp_path / "epoch_0_batch_2.pt")
    torch.save({"epoch": 0, "model_state_dict": m1.state_dict(), "optimizer_state_dict": t1.optimizer_state_dict()}, path)
    ck = torch.load(path, map_location="cpu")
    assert ck["optimizer_state_dict"]["ibm_b200"]["cond_drop_prob"] == 0.4
    m2, _ = _small_denoiser(F=10, L=2, seed=9)
    m2.load_state_dict(ck["model_state_dict"])
    t2 = Trainer(m2, **flags)
    t2.load_optimizer_state_dict(ck["optimizer_state_dict"])
    t2.arena.sync_shadow(force=True)
    t2._gen.set_state(gen)
    assert t2.step_count == 3 and torch.equal(t2.arena.master, t1.arena.master)
    for i in range(3, STEPS):
        l1 = t1.train_step(store, _batch(store, i))[0].item()
        l2 = t2.train_step(store, _batch(store, i))[0].item()
        assert torch.equal(_bits(t2.eng.xc(B, True)), _bits(t1.eng.xc(B, True))), f"input rows differ at step {i}"
        if i == 3:
            assert l1 == l2, (l1, l2)
            _same_step(t1, t2, "first resumed step")


# ---------------------------------------- guided step kernel ----------------------------------------------------------
def _tables(gd, sampler, eta):
    if sampler == "ddpm":
        return gd.coef_x0, gd.coef_xt, gd.sigma, None
    tab = gd.ddim_tables(7, eta)
    return tab["coef_x0"], tab["coef_xt"], tab["sigma"], tab["succ"]


@pytest.mark.parametrize("noise", ["supplied", "philox"])
@pytest.mark.parametrize("sampler,eta", [("ddpm", 1.0), ("ddim", 0.0), ("ddim", 1.0)])
@pytest.mark.parametrize("s", [0.0, 0.5, 2.5])
def test_guided_step_kernel_matches_oracle(s, sampler, eta, noise):
    from inferbiomechanics_b200 import ops
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    M, seed, offset = 4000, 77, 5
    gd = GaussianDiffusion(device="cuda")
    c0, c1, sig, succ = _tables(gd, sampler, eta)
    if sampler == "ddpm":
        t, p = 500, 499
    else:
        ts = gd.ddim_tables(7, eta)["ts"].tolist()
        t, p = ts[3], ts[4]
    g = torch.Generator().manual_seed(11)
    x0h = torch.randn(2 * M, 32, generator=g)
    xt, z = torch.randn(M, 30, generator=g), torch.randn(M, 30, generator=g)
    t_dev = torch.tensor([t], dtype=torch.int32, device="cuda")
    t_next = torch.full((1,), 12345, dtype=torch.int32, device="cuda")
    out = torch.empty(M, 30, device="cuda")
    xb = torch.zeros(2 * M, 40, dtype=torch.bfloat16, device="cuda")
    ops.guided_step(x0h.cuda(), 32, xt.cuda(), z.cuda() if noise == "supplied" else None, t_dev, c0, c1, sig, M, s, x_prev=out,
                    xprev_bf16=xb, bf16_ld=40, seed=seed, offset=offset, t_next=t_next, t_succ=succ)
    zz = z if noise == "supplied" else torch.from_numpy(ph.normals(M * 30, seed, offset + t)).view(M, 30)
    c, u = x0h[:M, :30], x0h[M:, :30]
    if sampler == "ddpm":
        want = ocfg.guided_ddpm_step(oddpm.make_schedule(), c, u, xt, t, zz, s)
        sigma = float(gd.sigma[t])
    else:
        want = ocfg.guided_ddim_step(odim.abar(), c, u, xt, t, p, eta, zz, s)
        sigma = float(sig[t])
    atol = 1e-6 + (1e-4 * sigma if noise == "philox" else 0.0)      # __logf / __sincosf in the Philox normals
    torch.testing.assert_close(out.cpu().double(), want, rtol=2e-6, atol=atol)
    assert t_next.item() == p
    assert torch.equal(_bits(xb[:M]), _bits(xb[M:]))
    assert torch.equal(_bits(xb[:M, :30]), _bits(out.to(torch.bfloat16)))
    assert not xb[:, 30:].any()


@pytest.mark.parametrize("sampler,eta", [("ddpm", 1.0), ("ddim", 0.0), ("ddim", 1.0)])
@pytest.mark.parametrize("s", [0.0, 0.5, 2.5, 1.0])
def test_guided_step_with_equal_halves_is_the_unguided_step(s, sampler, eta):
    from inferbiomechanics_b200 import ops
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    M = 3000
    gd = GaussianDiffusion(device="cuda")
    c0, c1, sig, succ = _tables(gd, sampler, eta)
    t = 500 if sampler == "ddpm" else gd.ddim_tables(7, eta)["ts"].tolist()[2]
    g = torch.Generator("cuda").manual_seed(3)
    c = torch.randn(M, 32, device="cuda", generator=g)
    xt = torch.randn(M, 30, device="cuda", generator=g)
    for z in (None, torch.randn(M, 30, device="cuda", generator=g)):
        outs = []
        for guided in (False, True):
            t_next = torch.zeros(1, dtype=torch.int32, device="cuda")
            x = torch.empty(M, 30, device="cuda")
            xb = torch.zeros(2 * M, 208, dtype=torch.bfloat16, device="cuda")
            t_dev = torch.tensor([t], dtype=torch.int32, device="cuda")
            if guided:
                ops.guided_step(torch.cat([c, c]), 32, xt, z, t_dev, c0, c1, sig, M, s, x_prev=x, xprev_bf16=xb, bf16_ld=208,
                                seed=9, offset=2, t_next=t_next, t_succ=succ)
            else:
                ops.posterior_step(c, 32, xt, z, t_dev, c0, c1, sig, M, x_prev=x, xprev_bf16=xb, bf16_ld=208, seed=9, offset=2,
                                   t_next=t_next, t_succ=succ)
            outs.append((x, xb, t_next.item()))
        (xa, ba, na), (xg, bg, ng) = outs
        assert torch.equal(xa, xg) and na == ng
        assert torch.equal(_bits(ba[:M]), _bits(bg[:M])) and torch.equal(_bits(bg[:M]), _bits(bg[M:]))


def test_guided_step_rejects_bad_scale():
    from inferbiomechanics_b200 import ops
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    gd = GaussianDiffusion(device="cuda")
    x0h, x = torch.zeros(20, 32, device="cuda"), torch.zeros(10, 30, device="cuda")
    t_dev = torch.tensor([3], dtype=torch.int32, device="cuda")
    for s in (-1.0, float("nan"), float("inf")):
        with pytest.raises(ValueError, match="guidance scale"):
            ops.guided_step(x0h, 32, x, None, t_dev, gd.coef_x0, gd.coef_xt, gd.sigma, 10, s, x_prev=x)


# ---------------------------------------- guided sampling loop --------------------------------------------------------
def _pack_cond(m, B, seed):
    from inferbiomechanics_b200 import ops
    eng = m.engine()
    cond = torch.randn(B, eng.F, eng.c_in, generator=torch.Generator().manual_seed(seed))
    ops.pack_inputs([cond.reshape(B * eng.F, eng.c_in).cuda()], B * eng.F, eng.F, out_bf16=eng.xc(B, False),
                    frame_stride=eng.ld_in, win_extra=0, col0=30)
    return cond


@pytest.mark.parametrize("sampler", ["ddpm", "ddim"])
def test_guided_sampling_loop_matches_oracle_with_supplied_noise(sampler):
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F, s, eta = 4, 10, 2.5, 1.0
    m, sd = _small_denoiser(F=F, L=1)
    cond = _pack_cond(m, B, 2)
    gd = GaussianDiffusion(device="cuda")
    g = torch.Generator().manual_seed(3)
    x_T = torch.randn(B, F, 30, generator=g)
    ts = list(range(999, 993, -1)) if sampler == "ddpm" else odim.ddim_timesteps(1000, 10).tolist()
    zs = {t: torch.randn(B * F, 30, generator=g) for t in ts}
    seen = []
    kw = dict(steps=len(ts)) if sampler == "ddpm" else dict(ddim_steps=10, eta=eta)
    got = gd.sample(m, B, x_T=x_T.cuda(), noise=lambda t: seen.append(t) or zs[t].cuda(), guidance_scale=s, **kw)
    assert seen == ts

    def denoise(x, t, conditional):
        cc = cond if conditional else torch.zeros_like(cond)
        return om.denoiser_forward(sd, cc, x.float().view(B, F, 30), torch.full((B,), t), 1, 2).reshape(B * F, 30)

    guided = ocfg.guided_denoiser(denoise, s)
    with torch.no_grad():
        if sampler == "ddpm":
            sched = oddpm.make_schedule()
            x = x_T.reshape(B * F, 30)
            for t in ts:
                x = ocfg.guided_ddpm_step(sched, denoise(x, t, True), denoise(x, t, False), x, t, zs[t], s).float()
            want = x
        else:
            want = odim.ddim_sample_loop(odim.abar(), guided, x_T.reshape(B * F, 30), 10, eta, lambda t: zs[t])
            plain = odim.ddim_sample_loop(odim.abar(), lambda x, t: denoise(x, t, True), x_T.reshape(B * F, 30), 10, eta,
                                          lambda t: zs[t])
    close(got.reshape(B * F, 30), want, 5e-2, "guided trajectory")
    if sampler == "ddim":                                   # guidance moved the result away from the conditional sample
        assert (got.reshape(B * F, 30).cpu().double() - plain.double()).abs().max().item() > 0.1 * plain.abs().max().item()


@pytest.mark.parametrize("S", [7, 10])
def test_guided_graph_replay_equals_eager(S):
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F = 8, 10
    m, _ = _small_denoiser(F=F, L=1)
    _pack_cond(m, B, 4)
    gd = GaussianDiffusion(num_timesteps=20, device="cuda")
    a = gd.sample(m, B, seed=5, ddim_steps=S, eta=1.0, guidance_scale=2.5, use_graph=False)
    b = gd.sample(m, B, seed=5, ddim_steps=S, eta=1.0, guidance_scale=2.5)
    key = (id(m), B, (S, 1.0), 2.5)
    graph = gd._graphs[key]["graph"]
    c = gd.sample(m, B, seed=5, ddim_steps=S, eta=1.0, guidance_scale=2.5)
    assert graph is not None and gd._graphs[key]["graph"] is graph
    assert torch.isfinite(a).all()
    torch.testing.assert_close(b, a, rtol=0, atol=0)
    torch.testing.assert_close(c, a, rtol=0, atol=0)
    # the DDPM chain (odd step count: the last step runs eagerly)
    gd2 = GaussianDiffusion(num_timesteps=S, device="cuda")
    d = gd2.sample(m, B, seed=5, guidance_scale=0.5, use_graph=False)
    e = gd2.sample(m, B, seed=5, guidance_scale=0.5)
    torch.testing.assert_close(e, d, rtol=0, atol=0)


def test_each_scale_has_its_own_graph_and_scale_one_is_unguided():
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F = 8, 10
    m, _ = _small_denoiser(F=F, L=1)
    _pack_cond(m, B, 6)
    scales = [1.0, 2.5, 0.0, 0.5]
    want = [GaussianDiffusion(num_timesteps=20, device="cuda").sample(m, B, seed=5, ddim_steps=8, guidance_scale=s,
                                                                     use_graph=False) for s in scales]
    gd = GaussianDiffusion(num_timesteps=20, device="cuda")
    for k in (1, 0, 2, 3, 1, 0, 3, 2):
        torch.testing.assert_close(gd.sample(m, B, seed=5, ddim_steps=8, guidance_scale=scales[k]), want[k], rtol=0, atol=0)
    assert len(gd._graphs) == 4 and (id(m), B, (8, 0.0)) in gd._graphs
    assert all(not torch.equal(want[i], want[j]) for i in range(4) for j in range(i))
    # s = 1 is today's loop: the same launches, in the same order, none of the guidance entry points
    gd3 = GaussianDiffusion(num_timesteps=20, device="cuda")
    for s in (1.0, 2.0):                                    # first calls allocate the cache entries and upload the tables
        gd3.sample(m, B, seed=5, ddim_steps=8, guidance_scale=s, use_graph=False)
    plain = _entry_points(lambda: gd3.sample(m, B, seed=5, ddim_steps=8, use_graph=False))
    one = _entry_points(lambda: gd3.sample(m, B, seed=5, ddim_steps=8, guidance_scale=1.0, use_graph=False))
    assert plain == one and plain.count("ibm_ddpm_respaced_step") == 8
    assert "ibm_cond_dropout" not in one and "ibm_ddpm_guided_step" not in one
    guided = _entry_points(lambda: gd3.sample(m, B, seed=5, ddim_steps=8, guidance_scale=2.0, use_graph=False))
    assert guided.count("ibm_cond_dropout") == 1 and guided.count("ibm_ddpm_guided_step") == 8
    assert "ibm_ddpm_respaced_step" not in guided


def _entry_points(fn):
    """The library entry points ``fn`` calls, in order (each launches its kernels on the current stream)."""
    from inferbiomechanics_b200 import ops
    seen, real = [], ops.call
    ops.call = lambda name, *a: seen.append(name) or real(name, *a)
    try:
        fn()
        torch.cuda.synchronize()
    finally:
        ops.call = real
    return seen


def test_unconditional_sampling_ignores_the_condition():
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F = 8, 10
    m, _ = _small_denoiser(F=F, L=1)
    gd = GaussianDiffusion(num_timesteps=20, device="cuda")
    _pack_cond(m, B, 1)
    a = gd.sample(m, B, seed=5, ddim_steps=6, guidance_scale=0.0)
    _pack_cond(m, B, 2)
    b = gd.sample(m, B, seed=5, ddim_steps=6, guidance_scale=0.0)
    c = gd.sample(m, B, seed=5, ddim_steps=6)
    torch.testing.assert_close(a, b, rtol=0, atol=0)
    assert not torch.equal(a, c)


def test_sharded_guided_sample_windows_matches_direct_calls():
    from inferbiomechanics_b200 import ops
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    F, N, batch = 10, 21, 8
    m, _ = _small_denoiser(F=F, L=1)
    eng = m.engine()
    gd = GaussianDiffusion(num_timesteps=12, device="cuda")
    cond = torch.randn(N, F, 177, generator=torch.Generator().manual_seed(4)).pin_memory()
    kw = dict(ddim_steps=5, eta=1.0, guidance_scale=2.5)
    shards = [gd.sample_windows(m, cond, batch=batch, seed=9, rank=r, world=2, **kw) for r in range(2)]
    assert [len(s[0]) for s in shards] == [11, 10]
    for r, (rng, x0) in enumerate(shards):
        assert tuple(x0.shape) == (len(rng), F, 30) and torch.isfinite(x0).all()
        for i, a in enumerate(range(rng.start, rng.stop, batch)):
            b = min(a + batch, rng.stop)
            ops.pack_inputs([cond[a:b].reshape(-1, 177).cuda()], (b - a) * F, F, out_bf16=eng.xc(b - a, False), frame_stride=eng.ld_in,
                            win_extra=0, col0=30)
            want = gd.sample(m, b - a, seed=9 + r + 7919 * i, **kw)
            torch.testing.assert_close(x0[a - rng.start:b - rng.start], want.cpu(), rtol=0, atol=0)


# ---------------------------------------- CLI -------------------------------------------------------------------------
def _run(argv):
    from inferbiomechanics_b200.main import main
    return main(argv)


def test_cli_train_with_condition_dropout_then_guided_analyze(tmp_path, capsys):
    ck = str(tmp_path / "ck")
    common = ["--no-wandb", "--synthetic-windows", "512", "--checkpoint-dir", ck, "--history-len", "50", "--stride", "1",
              "--model-type", "diffusion", "--batch-size", "64"]
    _run(["train", *common, "--epochs", "1", "--max-batches", "3", "--cond-drop-prob", "0.1"])
    d = os.path.join(ck, "diffusion")
    last = sorted(os.listdir(d))[-1]
    tag = torch.load(os.path.join(d, last), map_location="cpu")["optimizer_state_dict"]["ibm_b200"]
    assert tag == {"opt_type": "rmsprop", "step": 3, "cond_drop_prob": 0.1}
    capsys.readouterr()
    an = _run(["analyze", *common, "--sampler", "ddim", "--sampling-steps", "10", "--guidance-scale", "2.5"])
    out = capsys.readouterr().out
    assert re.search(r"dev set evaluation \(\d+ windows, guidance scale 2\.5\):", out), out
    loss = an.last_reports["dev"]["loss"]
    assert math.isfinite(loss) and loss > 0
    an = _run(["analyze", *common, "--sampler", "ddpm", "--sampling-steps", "20", "--guidance-scale", "0"])
    assert math.isfinite(an.last_reports["dev"]["loss"])
    assert "guidance scale 0)" in capsys.readouterr().out
    an = _run(["analyze", *common, "--sampler", "ddim", "--sampling-steps", "10"])
    out = capsys.readouterr().out
    assert re.search(r"dev set evaluation \(\d+ windows\):", out) and "guidance" not in out
    # a checkpoint trained without condition dropout cannot be guided
    ck2 = str(tmp_path / "ck2")
    plain = [a if a != ck else ck2 for a in common]
    _run(["train", *plain, "--epochs", "1", "--max-batches", "1"])
    with pytest.raises(ValueError, match="records none"):
        _run(["analyze", *plain, "--sampler", "ddim", "--sampling-steps", "10", "--guidance-scale", "2.5"])
