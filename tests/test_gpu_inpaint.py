"""Inpainting on a B200: the known-value step kernel (``ibm_ddpm_inpaint_step``) against the fp64 oracle, the sampling loop
against the CPU oracle loop, the exactness of the known entries of a sample, the identities with today's sampler (empty mask,
graph replay, reused graphs, ``num_samples``, sharded ``sample_windows``), refusals and ``analyze --given-quantities``.  The
oracle (``tests/inpaint_oracle.py``) is builder-owned and parity unpinned, like all diffusion code here."""
import math
import re

import pytest
import torch

import cfg_oracle as ocfg
import ddim_oracle as odim
import inpaint_oracle as oinp
import philox_oracle as ph
from oracle import ddpm as oddpm
from oracle import models as om
from test_gpu_ensemble import _replicate
from test_gpu_guidance import _bits, _entry_points, _pack_cond, _tables
from test_gpu_models import _small_denoiser, close

pytestmark = pytest.mark.gpu

NAN = float("nan")


def _mask(kind, shape, seed):
    if kind == "all":
        return torch.ones(shape, dtype=torch.bool)
    if kind == "none":
        return torch.zeros(shape, dtype=torch.bool)
    return torch.rand(shape, generator=torch.Generator().manual_seed(seed)) < 0.4


def _with_nan(y, mask):
    """y where the mask is set, NaN elsewhere: an unknown entry must never reach the output."""
    return torch.where(mask, y, torch.full_like(y, NAN))


# ---------------------------------------- step kernel -----------------------------------------------------------------
@pytest.mark.parametrize("mask_kind", ["random", "all", "none"])
@pytest.mark.parametrize("noise", ["supplied", "philox"])
@pytest.mark.parametrize("guided", [False, True])
@pytest.mark.parametrize("sampler,eta", [("ddpm", 1.0), ("ddim", 0.0), ("ddim", 1.0)])
def test_inpaint_step_kernel_matches_oracle(sampler, eta, guided, noise, mask_kind):
    from inferbiomechanics_b200 import ops
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    M, seed, offset, s = 3000, 77, 5, 2.5
    gd = GaussianDiffusion(device="cuda")
    c0, c1, sig, succ = _tables(gd, sampler, eta)
    if sampler == "ddpm":
        t, p = 500, 499
    else:
        ts = gd.ddim_tables(7, eta)["ts"].tolist()
        t, p = ts[3], ts[4]
    g = torch.Generator().manual_seed(13)
    x0h = torch.randn((2 if guided else 1) * M, 32, generator=g)
    xt, z, y = (torch.randn(M, 30, generator=g) for _ in range(3))
    mask = _mask(mask_kind, (M, 30), 17)
    t_dev = torch.tensor([t], dtype=torch.int32, device="cuda")
    t_next = torch.full((1,), 12345, dtype=torch.int32, device="cuda")
    out = torch.empty(M, 30, device="cuda")
    xb = torch.zeros((2 if guided else 1) * M, 40, dtype=torch.bfloat16, device="cuda")
    kw = dict(x_prev=out, xprev_bf16=xb, bf16_ld=40, seed=seed, offset=offset, t_next=t_next, t_succ=succ,
              known=_with_nan(y, mask).cuda(), known_mask=oinp.mask_words(mask).cuda())
    zc = z.cuda() if noise == "supplied" else None
    if guided:
        ops.guided_step(x0h.cuda(), 32, xt.cuda(), zc, t_dev, c0, c1, sig, M, s, **kw)
        pred = ocfg.guided_x0(x0h[:M, :30], x0h[M:, :30], s)
    else:
        ops.posterior_step(x0h.cuda(), 32, xt.cuda(), zc, t_dev, c0, c1, sig, M, **kw)
        pred = x0h[:, :30].double()
    pred = oinp.known_x0(pred, y, mask)
    zz = z if noise == "supplied" else torch.from_numpy(ph.normals(M * 30, seed, offset + t)).view(M, 30)
    if sampler == "ddpm":
        sched = {k: v.double() for k, v in oddpm.make_schedule().items()}
        want = oddpm.posterior_step(sched, pred, xt.double(), t, zz.double())
        sigma = float(gd.sigma[t])
    else:
        want = odim.ddim_step(odim.abar(), pred, xt, t, p, eta, zz)
        sigma = float(sig[t])
    assert torch.isfinite(out).all()
    atol = 1e-6 + (1e-4 * sigma if noise == "philox" else 0.0)      # __logf / __sincosf in the Philox normals
    torch.testing.assert_close(out.cpu().double(), want, rtol=2e-6, atol=atol)
    assert t_next.item() == p
    assert torch.equal(_bits(xb[:M, :30]), _bits(out.to(torch.bfloat16)))
    if guided:
        assert torch.equal(_bits(xb[:M]), _bits(xb[M:]))
    assert not xb[:, 30:].any()


@pytest.mark.parametrize("guided", [False, True])
@pytest.mark.parametrize("sampler,eta", [("ddpm", 1.0), ("ddim", 0.0), ("ddim", 1.0)])
def test_empty_mask_is_todays_step_and_bits_30_31_change_nothing(sampler, eta, guided):
    from inferbiomechanics_b200 import ops
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    M = 2000
    gd = GaussianDiffusion(device="cuda")
    c0, c1, sig, succ = _tables(gd, sampler, eta)
    t = 500 if sampler == "ddpm" else gd.ddim_tables(7, eta)["ts"].tolist()[2]
    g = torch.Generator("cuda").manual_seed(3)
    x0h = torch.randn((2 if guided else 1) * M, 32, device="cuda", generator=g)
    xt = torch.randn(M, 30, device="cuda", generator=g)
    y = torch.randn(M, 30, device="cuda", generator=g)
    rand_words = oinp.mask_words(_mask("random", (M, 30), 4)).cuda()
    high = torch.full((M,), -(1 << 31), dtype=torch.int32, device="cuda") | (1 << 30)          # bits 30 and 31 only
    for z in (None, torch.randn(M, 30, device="cuda", generator=g)):
        outs = {}
        for name, kn in (("today", {}), ("empty", dict(known=torch.full_like(y, NAN), known_mask=torch.zeros_like(high))),
                         ("high", dict(known=torch.full_like(y, NAN), known_mask=high)),
                         ("random", dict(known=y, known_mask=rand_words)),
                         ("random+high", dict(known=y, known_mask=rand_words | high))):
            x = torch.empty(M, 30, device="cuda")
            xb = torch.zeros((2 if guided else 1) * M, 208, dtype=torch.bfloat16, device="cuda")
            t_next = torch.zeros(1, dtype=torch.int32, device="cuda")
            t_dev = torch.tensor([t], dtype=torch.int32, device="cuda")
            kw = dict(x_prev=x, xprev_bf16=xb, bf16_ld=208, seed=9, offset=2, t_next=t_next, t_succ=succ, **kn)
            if guided:
                ops.guided_step(x0h, 32, xt, z, t_dev, c0, c1, sig, M, 2.5, **kw)
            else:
                ops.posterior_step(x0h, 32, xt, z, t_dev, c0, c1, sig, M, **kw)
            outs[name] = (x, _bits(xb), t_next.item())
        for name in ("empty", "high"):
            assert torch.equal(outs[name][0], outs["today"][0]) and torch.equal(outs[name][1], outs["today"][1]), name
            assert outs[name][2] == outs["today"][2]
        assert torch.equal(outs["random+high"][0], outs["random"][0])
        assert not torch.equal(outs["random"][0], outs["today"][0])


def test_step_refusals_launch_nothing():
    from inferbiomechanics_b200 import _lib, ops
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    M = 100
    gd = GaussianDiffusion(device="cuda")
    x0h, xt = torch.zeros(2 * M, 32, device="cuda"), torch.zeros(M, 30, device="cuda")
    t_dev = torch.tensor([3], dtype=torch.int32, device="cuda")
    t_next = torch.full((1,), 777, dtype=torch.int32, device="cuda")
    out = torch.full((M, 30), 5.0, device="cuda")
    y, w = torch.zeros(M, 30, device="cuda"), torch.zeros(M, dtype=torch.int32, device="cuda")
    buf = torch.zeros(M * 30 + 1, device="cuda")
    bad = [(y, None), (None, w), (y.double(), w), (y, w.long()), (y[:, :29], w), (y[:M - 1], w), (y, w[:M - 1]),
           (y.cpu(), w), (y, w.cpu()), (torch.zeros(30, M, device="cuda").t(), w), (y.view(M, 30, 1), w)]
    n = _lib.launch_count
    for k, m in bad:
        with pytest.raises(ValueError):
            ops.posterior_step(x0h, 32, xt, None, t_dev, gd.coef_x0, gd.coef_xt, gd.sigma, M, x_prev=out, t_next=t_next,
                               known=k, known_mask=m)
        with pytest.raises(ValueError):
            ops.guided_step(x0h, 32, xt, None, t_dev, gd.coef_x0, gd.coef_xt, gd.sigma, M, 2.5, x_prev=out, t_next=t_next,
                            known=k, known_mask=m)
    assert _lib.launch_count == n
    # refused in C: known values 4-byte aligned only, a bad guidance scale, no output
    for call in (lambda: ops.posterior_step(x0h, 32, xt, None, t_dev, gd.coef_x0, gd.coef_xt, gd.sigma, M, x_prev=out,
                                            t_next=t_next, known=buf[1:].view(M, 30), known_mask=w),
                 lambda: ops.guided_step(x0h, 32, xt, None, t_dev, gd.coef_x0, gd.coef_xt, gd.sigma, M, -1.0, x_prev=out,
                                         t_next=t_next, known=y, known_mask=w),
                 lambda: ops.posterior_step(x0h, 32, xt, None, t_dev, gd.coef_x0, gd.coef_xt, gd.sigma, M, t_next=t_next,
                                            known=y, known_mask=w)):
        with pytest.raises(ValueError):
            call()
    torch.cuda.synchronize()
    assert (out == 5.0).all() and t_next.item() == 777


# ---------------------------------------- sampling loop ---------------------------------------------------------------
def _denoiser(sd, cond, B, F):
    def denoise(x, t, conditional=True):
        cc = cond if conditional else torch.zeros_like(cond)
        return om.denoiser_forward(sd, cc, x.float().view(B, F, 30), torch.full((B,), t), 1, 2).reshape(B * F, 30)
    return denoise


@pytest.mark.parametrize("sampler,s", [("ddpm", 1.0), ("ddim", 1.0), ("ddim", 2.5)])
def test_inpainted_sampling_loop_matches_oracle_with_supplied_noise(sampler, s):
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F, eta = 4, 10, 1.0
    m, sd = _small_denoiser(F=F, L=1)
    cond = _pack_cond(m, B, 2)
    T = 20 if sampler == "ddpm" else 1000
    gd = GaussianDiffusion(num_timesteps=T, device="cuda")
    g = torch.Generator().manual_seed(3)
    x_T = torch.randn(B, F, 30, generator=g)
    y = torch.randn(B, F, 30, generator=g)
    mask = _mask("random", (B, F, 30), 8)
    mask[:, 3:6] = True                                     # whole frames known, as around a gap
    ts = list(range(T - 1, -1, -1)) if sampler == "ddpm" else odim.ddim_timesteps(T, 10).tolist()
    zs = {t: torch.randn(B * F, 30, generator=g) for t in ts}
    kw = {} if sampler == "ddpm" else dict(ddim_steps=10, eta=eta)
    got = gd.sample(m, B, x_T=x_T.cuda(), noise=lambda t: zs[t].cuda(), guidance_scale=s, known=_with_nan(y, mask).cuda(),
                    known_mask=mask.cuda(), **kw)
    den = _denoiser(sd, cond, B, F)
    pred = ocfg.guided_denoiser(den, s) if s != 1.0 else den
    inp = oinp.known_denoiser(pred, y.reshape(B * F, 30), mask.reshape(B * F, 30))
    with torch.no_grad():
        if sampler == "ddpm":
            sched = {k: v.double() for k, v in oddpm.make_schedule(T).items()}
            want = oddpm.sample_loop(sched, lambda x, t: inp(x, t).double(), x_T.reshape(B * F, 30).double(),
                                     lambda t: zs[t].double()).float()
        else:
            want = odim.ddim_sample_loop(odim.abar(), inp, x_T.reshape(B * F, 30), 10, eta, lambda t: zs[t])
    assert torch.isfinite(got).all()
    close(got.reshape(B * F, 30), want, 5e-2, "inpainted trajectory")
    assert torch.equal(got.cpu()[mask], y[mask])


@pytest.mark.parametrize("sampler", [("ddpm", None, 0.0), ("ddim", 1, 0.0), ("ddim", 1, 1.0), ("ddim", 2, 0.0), ("ddim", 2, 1.0),
                                     ("ddim", 7, 0.0), ("ddim", 7, 1.0)], ids=lambda c: "-".join(map(str, c)))
def test_sample_equals_known_values_exactly(sampler):
    from inferbiomechanics_b200.cli.train import known_quantity_mask
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    kind, S, eta = sampler
    B, F = 6, 10
    m, _ = _small_denoiser(F=F, L=1)
    _pack_cond(m, B, 5)
    gd = GaussianDiffusion(device="cuda")
    y = torch.randn(B, F, 30, generator=torch.Generator().manual_seed(9)) * 4
    masks = [_mask("random", (B, F, 30), 10), known_quantity_mask(("force",))]
    kw = {} if kind == "ddpm" else dict(ddim_steps=S, eta=eta)
    for s in (1.0, 2.5):
        for K, mask in ((None, masks[0]), (3, masks[1])):
            full = mask.expand(B, F, 30)
            x = gd.sample(m, B, seed=4, guidance_scale=s, num_samples=K, known=_with_nan(y, full).cuda(), known_mask=mask.cuda(),
                          **kw).cpu()
            draws = x.unsqueeze(0) if K is None else x
            assert torch.isfinite(draws).all(), (s, K)
            for d in draws:
                assert torch.equal(d[full], y[full]), (s, K)
            assert not torch.equal(draws[0][~full], y[~full])


# ---------------------------------------- identities ------------------------------------------------------------------
@pytest.mark.parametrize("kw", [dict(ddim_steps=8, eta=1.0), dict(ddim_steps=8, eta=0.0, guidance_scale=2.5), dict()],
                         ids=["ddim", "ddim-guided", "ddpm"])
def test_empty_mask_sample_is_todays_sample(kw):
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F = 8, 10
    m, _ = _small_denoiser(F=F, L=1)
    _pack_cond(m, B, 6)
    empty = dict(known=torch.full((B, F, 30), NAN, device="cuda"), known_mask=torch.zeros(30, dtype=torch.bool))
    gd = GaussianDiffusion(num_timesteps=20, device="cuda")
    for use_graph in (False, True, True):
        today = gd.sample(m, B, seed=5, use_graph=use_graph, **kw)
        inp = gd.sample(m, B, seed=5, use_graph=use_graph, **kw, **empty)
        assert torch.equal(today, inp), use_graph
    # known=None launches today's sequence: no inpainting entry point
    calls = _entry_points(lambda: gd.sample(m, B, seed=5, use_graph=False, **kw))
    assert "ibm_ddpm_inpaint_step" not in calls
    calls = _entry_points(lambda: gd.sample(m, B, seed=5, use_graph=False, **kw, **empty))
    assert "ibm_ddpm_posterior_step" not in calls and "ibm_ddpm_respaced_step" not in calls and "ibm_ddpm_guided_step" not in calls
    assert calls.count("ibm_ddpm_inpaint_step") == (8 if kw else 20)


@pytest.mark.parametrize("S,s", [(7, 1.0), (10, 1.0), (10, 2.5)])
def test_inpainted_graph_replay_equals_eager_and_reuses_one_graph(S, s):
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F = 8, 10
    m, _ = _small_denoiser(F=F, L=1)
    _pack_cond(m, B, 4)
    g = torch.Generator().manual_seed(2)
    ys = [torch.randn(B, F, 30, generator=g).cuda() for _ in range(3)]
    masks = [_mask("random", (B, F, 30), 20).cuda(), _mask("random", (B, F, 30), 21).cuda(),
             torch.zeros(30, dtype=torch.bool, device="cuda")]
    masks[2][6:12] = True
    kw = dict(seed=5, ddim_steps=S, eta=1.0, guidance_scale=s)
    eager = [GaussianDiffusion(num_timesteps=20, device="cuda").sample(m, B, use_graph=False, known=y, known_mask=k, **kw)
             for y, k in zip(ys, masks)]
    gd = GaussianDiffusion(num_timesteps=20, device="cuda")
    key = (id(m), B, (S, 1.0)) + ((float(s),) if s != 1.0 else ()) + ("inpaint",)
    graph = None
    for i in (0, 1, 2, 0):
        got = gd.sample(m, B, known=ys[i], known_mask=masks[i], **kw)
        assert torch.equal(got, eager[i]), i
        graph = graph or gd._graphs[key]["graph"]
        assert graph is not None and gd._graphs[key]["graph"] is graph
    assert len(gd._graphs) == 1
    assert not torch.equal(eager[0], eager[1])


@pytest.mark.parametrize("kw", [dict(ddim_steps=7, eta=1.0), dict(ddim_steps=6, eta=0.0, guidance_scale=2.5), dict()],
                         ids=["ddim", "ddim-guided", "ddpm"])
def test_num_samples_is_the_call_on_replicated_windows_and_known_values(kw):
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F, K = 6, 10, 3
    m, _ = _small_denoiser(F=F, L=1)
    _pack_cond(m, B, 3)
    y = torch.randn(B, F, 30, generator=torch.Generator().manual_seed(1)).cuda()
    mask = _mask("random", (B, F, 30), 2).cuda()
    gd = GaussianDiffusion(num_timesteps=15, device="cuda")
    got = gd.sample(m, B, seed=5, num_samples=K, known=y, known_mask=mask, **kw)
    again = gd.sample(m, B, seed=5, num_samples=K, known=y, known_mask=mask, **kw)
    _replicate(m, B, K)
    want = GaussianDiffusion(num_timesteps=15, device="cuda").sample(m, B * K, seed=5, use_graph=False, known=y.repeat(K, 1, 1),
                                                                    known_mask=mask.repeat(K, 1, 1), **kw)
    assert torch.equal(got.reshape(B * K, F, 30), want) and torch.equal(again, got)


def test_sharded_sample_windows_with_known_values_matches_direct_calls():
    from inferbiomechanics_b200 import ops
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    F, N, batch = 10, 21, 8
    m, _ = _small_denoiser(F=F, L=1)
    eng = m.engine()
    gd = GaussianDiffusion(num_timesteps=12, device="cuda")
    g = torch.Generator().manual_seed(4)
    cond = torch.randn(N, F, 177, generator=g).pin_memory()
    y = torch.randn(N, F, 30, generator=g)
    for mask in (_mask("random", (N, F, 30), 5), torch.arange(30) < 6):
        known = _with_nan(y, mask.expand(N, F, 30)).pin_memory()
        kw = dict(ddim_steps=5, eta=1.0, guidance_scale=2.5)
        shards = [gd.sample_windows(m, cond, batch=batch, seed=9, rank=r, world=2, known=known, known_mask=mask, **kw)
                  for r in range(2)]
        assert [len(s[0]) for s in shards] == [11, 10]
        for r, (rng, x0) in enumerate(shards):
            assert tuple(x0.shape) == (len(rng), F, 30) and torch.isfinite(x0).all()
            for i, a in enumerate(range(rng.start, rng.stop, batch)):
                b = min(a + batch, rng.stop)
                ops.pack_inputs([cond[a:b].reshape(-1, 177).cuda()], (b - a) * F, F, out_bf16=eng.xc(b - a, False),
                                frame_stride=eng.ld_in, win_extra=0, col0=30)
                mk = mask[a:b].cuda() if mask.dim() == 3 else mask
                want = gd.sample(m, b - a, seed=9 + r + 7919 * i, known=known[a:b].cuda(), known_mask=mk, **kw)
                assert torch.equal(x0[a - rng.start:b - rng.start], want.cpu())


def test_sampler_refusals_launch_nothing():
    from inferbiomechanics_b200 import _lib
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F = 4, 10
    m, _ = _small_denoiser(F=F, L=1)
    gd = GaussianDiffusion(num_timesteps=20, device="cuda")
    mask = torch.ones(30, dtype=torch.bool)
    m.engine()
    n = _lib.launch_count
    for kw in (dict(known=torch.zeros(B, F + 1, 30, device="cuda"), known_mask=mask),
               dict(known=torch.zeros(B, F, 30), known_mask=mask),
               dict(known=torch.zeros(B, F, 30, device="cuda"), known_mask=mask, steps=10),
               dict(known=torch.zeros(B, F, 30, device="cuda"))):
        with pytest.raises(ValueError):
            gd.sample(m, B, **kw)
    with pytest.raises(ValueError):
        gd.sample_windows(m, torch.zeros(B, F, 177), known=torch.zeros(B, F, 30, device="cuda"), known_mask=mask)
    assert _lib.launch_count == n


# ---------------------------------------- CLI -------------------------------------------------------------------------
def _run(argv):
    from inferbiomechanics_b200.main import main
    return main(argv)


def test_cli_analyze_given_force(tmp_path, capsys):
    ck = str(tmp_path / "ck")
    common = ["--no-wandb", "--synthetic-windows", "512", "--checkpoint-dir", ck, "--history-len", "50", "--stride", "1",
              "--model-type", "diffusion", "--batch-size", "64"]
    _run(["train", *common, "--epochs", "1", "--max-batches", "3"])
    capsys.readouterr()
    ddim = ["--sampler", "ddim", "--sampling-steps", "4", "--given-quantities", "force"]
    an = _run(["analyze", *common, *ddim])
    out = capsys.readouterr().out
    assert re.search(r"dev set evaluation \(\d+ windows, given force\):", out), out
    for split in ("dev", "train"):
        rep = an.last_reports[split]
        assert rep["force_r"] == 0.0 and not rep["force"].any(), rep
        assert all(math.isfinite(rep[k]) for k in ("loss", "cop_r", "moment_r", "wrench_r")), rep
        assert rep["moment_r"] > 0
    an = _run(["analyze", *common, *ddim, "--num-samples", "2"])
    out = capsys.readouterr().out
    assert re.search(r"dev set evaluation \(\d+ windows, ensemble mean of 2 samples, given force\):", out), out
    assert len(re.findall(r"\tforce \(given\): CRPS ", out)) == 2 and "cop (given)" not in out
    for split in ("dev", "train"):
        rep = an.last_reports[split]
        assert rep["force_r"] == 0.0 and not rep["force"].any(), rep
        ens = an.last_ensemble_reports[split]
        assert ens["force"]["crps"] == 0.0 and ens["force"]["spread"] == 0.0 and ens["force"]["count"] > 0, ens["force"]
        for q in ("cop", "moment", "wrench"):
            assert all(math.isfinite(ens[q][k]) for k in ("crps", "rmse", "spread")), ens[q]
        assert ens["moment"]["spread"] > 0
