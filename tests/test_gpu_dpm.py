"""DPM-Solver++(2M) sampling on a B200: the multistep step kernel (``ibm_ddpm_multistep_step``) against the fp64 exp / lambda
oracle (``tests/dpm_oracle.py``, builder-owned and parity unpinned like all diffusion code here), its refusals, the sampling
loop against the oracle loop, the identities with DDIM at one and two steps, graph replay, graph separation per schedule,
exact known values, ``num_samples``, sharded ``sample_windows`` and ``analyze --sampler dpmpp2m``."""
import math
import re

import pytest
import torch

import cfg_oracle as ocfg
import ddim_oracle as odim
import dpm_oracle as odpm
import inpaint_oracle as oinp
from oracle import models as om
from test_gpu_ensemble import _replicate
from test_gpu_guidance import _bits, _pack_cond
from test_gpu_models import _small_denoiser, close

pytestmark = pytest.mark.gpu

NAN = float("nan")


# ---------------------------------------- step kernel -----------------------------------------------------------------
@pytest.mark.parametrize("known", [False, True])
@pytest.mark.parametrize("guided", [False, True])
@pytest.mark.parametrize("which", ["first", "interior", "last"])
def test_multistep_kernel_matches_oracle(which, guided, known):
    from inferbiomechanics_b200 import ops
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    S, M, s = 10, 3000, 2.5
    gd = GaussianDiffusion(device="cuda")
    tab = gd.dpm_tables(S)
    ts = tab["ts"]
    i = {"first": 0, "interior": 4, "last": S - 1}[which]
    t, p = int(ts[i]), (int(ts[i + 1]) if i + 1 < S else -1)
    g = torch.Generator().manual_seed(21 + i)
    x0h = torch.randn((2 if guided else 1) * M, 32, generator=g)      # the head GEMM's 32-float rows
    xt, prev, y = (torch.randn(M, 30, generator=g) for _ in range(3))
    mask = torch.rand(M, 30, generator=g) < 0.4
    # the first step must not read the previous prediction: NaN there would poison the output
    prev_dev = prev.cuda() if which == "interior" else torch.full((M, 30), NAN, device="cuda")
    t_dev = torch.tensor([t], dtype=torch.int32, device="cuda")
    t_next = torch.full((1,), 12345, dtype=torch.int32, device="cuda")
    out = torch.empty(M, 30, device="cuda")
    xb = torch.zeros((2 if guided else 1) * M, 40, dtype=torch.bfloat16, device="cuda")
    kn = dict(known=torch.where(mask, y, torch.full_like(y, NAN)).cuda(), known_mask=oinp.mask_words(mask).cuda()) if known else {}
    ops.multistep_step(x0h.cuda(), 32, xt.cuda(), t_dev, tab["coef_x0"], tab["coef_xt"], tab["coef_prev"], tab["succ"], M, prev_dev,
                       x_prev=out, xprev_bf16=xb, bf16_ld=40, t_next=t_next, guidance_scale=s if guided else None, **kn)
    pred = ocfg.guided_x0(x0h[:M, :30], x0h[M:, :30], s) if guided else x0h[:, :30].double()
    if known:
        pred = oinp.known_x0(pred, y, mask)
    want = odpm.dpm_step(odim.abar(), ts, i, pred, prev, xt)
    assert torch.isfinite(out).all()
    torch.testing.assert_close(out.cpu().double(), want, rtol=2e-6, atol=1e-6)
    assert t_next.item() == p == int(tab["succ"][t])
    # x0_prev now holds this step's prediction: after the guided combination and the known-entry select
    got_prev = prev_dev.cpu()
    if guided:
        torch.testing.assert_close(got_prev.double(), pred, rtol=2e-6, atol=1e-6)
    else:
        assert torch.equal(got_prev, pred.float())
    if known:
        assert torch.equal(got_prev[mask], y[mask])
    if which == "last":
        assert torch.equal(out.cpu(), got_prev)                    # the last step returns the prediction exactly
    assert torch.equal(_bits(xb[:M, :30]), _bits(out.to(torch.bfloat16)))
    if guided:
        assert torch.equal(_bits(xb[:M]), _bits(xb[M:]))
    assert not xb[:, 30:].any()


@pytest.mark.parametrize("guided", [False, True])
def test_first_and_last_steps_are_the_ddim_steps(guided):
    """On the first-order steps the multistep kernel computes exactly what the respaced DDIM-eta-0 step computes."""
    from inferbiomechanics_b200 import ops
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    M, s = 2000, 2.5
    gd = GaussianDiffusion(device="cuda")
    dpm, ddim = gd.dpm_tables(2), gd.ddim_tables(2, 0.0)
    g = torch.Generator("cuda").manual_seed(5)
    x0h = torch.randn((2 if guided else 1) * M, 32, device="cuda", generator=g)
    xt = torch.randn(M, 30, device="cuda", generator=g)
    for t in (gd.T - 1, 0):
        outs = []
        for kind in ("dpm", "ddim"):
            x = torch.empty(M, 30, device="cuda")
            xb = torch.zeros((2 if guided else 1) * M, 208, dtype=torch.bfloat16, device="cuda")
            t_dev = torch.tensor([t], dtype=torch.int32, device="cuda")
            t_next = torch.zeros(1, dtype=torch.int32, device="cuda")
            if kind == "dpm":
                ops.multistep_step(x0h, 32, xt, t_dev, dpm["coef_x0"], dpm["coef_xt"], dpm["coef_prev"], dpm["succ"], M,
                                   torch.full((M, 30), NAN, device="cuda"), x_prev=x, xprev_bf16=xb, bf16_ld=208, t_next=t_next,
                                   guidance_scale=s if guided else None)
            elif guided:
                ops.guided_step(x0h, 32, xt, None, t_dev, ddim["coef_x0"], ddim["coef_xt"], ddim["sigma"], M, s, x_prev=x,
                                xprev_bf16=xb, bf16_ld=208, seed=3, t_next=t_next, t_succ=ddim["succ"])
            else:
                ops.posterior_step(x0h, 32, xt, None, t_dev, ddim["coef_x0"], ddim["coef_xt"], ddim["sigma"], M, x_prev=x,
                                   xprev_bf16=xb, bf16_ld=208, seed=3, t_next=t_next, t_succ=ddim["succ"])
            outs.append((x, _bits(xb), t_next.item()))
        assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]) and outs[0][2] == outs[1][2], t


def _raw_args(M=100):
    """A valid argument set of ibm_ddpm_multistep_step (device tensors kept alive by the dict)."""
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    tab = GaussianDiffusion(device="cuda").dpm_tables(10)
    d = dict(x0h=torch.zeros(2 * M, 32, device="cuda"), xt=torch.zeros(M, 30, device="cuda"),
             t_dev=torch.tensor([int(tab["ts"][3])], dtype=torch.int32, device="cuda"),
             prev=torch.full((M, 30), 7.0, device="cuda"), out=torch.full((M, 30), 5.0, device="cuda"),
             xb=torch.full((2 * M, 40), 3.0, dtype=torch.bfloat16, device="cuda"),
             t_next=torch.full((1,), 777, dtype=torch.int32, device="cuda"), known=torch.zeros(M + 1, 30, device="cuda"),
             words=torch.zeros(M, dtype=torch.int32, device="cuda"), buf=torch.zeros(M * 30 + 1, device="cuda"), tab=tab)
    args = dict(x0_hat=d["x0h"].data_ptr(), x0_ld=32, x_t=d["xt"].data_ptr(), t_dev=d["t_dev"].data_ptr(),
                coef_x0=tab["coef_x0"].data_ptr(), coef_xt=tab["coef_xt"].data_ptr(), coef_prev=tab["coef_prev"].data_ptr(),
                t_succ=tab["succ"].data_ptr(), M=M, x0_prev=d["prev"].data_ptr(), x_prev=d["out"].data_ptr(),
                xprev_bf16=d["xb"].data_ptr(), bf16_ld=40, t_next=d["t_next"].data_ptr(), guidance_scale=2.5, guided=1,
                known=None, known_mask=None, stream=torch.cuda.current_stream().cuda_stream)
    return d, args


def test_step_refusals_launch_nothing():
    from inferbiomechanics_b200 import _lib, ops
    lib = _lib.load()
    d, ok = _raw_args()
    M = ok["M"]
    kp, wp = d["known"].data_ptr(), d["words"].data_ptr()
    bad = [dict(x0_hat=None), dict(x_t=None), dict(t_dev=None), dict(coef_x0=None), dict(coef_xt=None), dict(coef_prev=None),
           dict(t_succ=None), dict(x0_prev=None), dict(x0_prev=d["buf"].data_ptr() + 4), dict(x0_prev=ok["x_prev"]),
           dict(x0_prev=ok["x_t"]), dict(x0_prev=ok["x0_hat"]), dict(known=kp), dict(known_mask=wp),
           dict(known=kp + 4, known_mask=wp), dict(M=0), dict(x0_ld=29), dict(x0_ld=33), dict(bf16_ld=41), dict(bf16_ld=28),
           dict(x_prev=None, xprev_bf16=None), dict(guidance_scale=-1.0), dict(guidance_scale=NAN),
           dict(guidance_scale=float("inf")), dict(guidance_scale=-1.0, guided=0)]
    for kw in bad:
        a = {**ok, **kw}
        rc = lib.ibm_ddpm_multistep_step(*a.values())
        assert rc == 1, kw
    # refused by the wrapper before the call: the previous-prediction buffer and the known values
    n = _lib.launch_count
    tab = d["tab"]
    y, w = d["known"][:M], d["words"]
    for prev, kn in ((d["prev"][:M - 1], {}), (d["prev"].double(), {}), (d["prev"].cpu(), {}), (d["prev"].t().contiguous().t(), {}),
                     (d["prev"], dict(known=y)), (d["prev"], dict(known_mask=w)), (d["prev"], dict(known=y.double(), known_mask=w))):
        with pytest.raises(ValueError):
            ops.multistep_step(d["x0h"], 32, d["xt"], d["t_dev"], tab["coef_x0"], tab["coef_xt"], tab["coef_prev"], tab["succ"], M,
                               prev, x_prev=d["out"], t_next=d["t_next"], guidance_scale=2.5, **kn)
    assert _lib.launch_count == n
    torch.cuda.synchronize()
    assert (d["out"] == 5.0).all() and (d["prev"] == 7.0).all() and (d["xb"] == 3.0).all() and d["t_next"].item() == 777
    # the valid set runs
    assert lib.ibm_ddpm_multistep_step(*ok.values()) == 0
    torch.cuda.synchronize()
    assert d["t_next"].item() == int(tab["succ"][int(tab["ts"][3])]) and (d["prev"] == 0).all()


# ---------------------------------------- sampling loop ---------------------------------------------------------------
@pytest.mark.parametrize("S", [6, 10])
def test_sampling_loop_matches_oracle(S):
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F = 4, 10
    m, sd = _small_denoiser(F=F, L=1)
    cond = _pack_cond(m, B, 2)
    gd = GaussianDiffusion(device="cuda")
    x_T = torch.randn(B, F, 30, generator=torch.Generator().manual_seed(3))
    got = gd.sample(m, B, x_T=x_T.cuda(), dpm_steps=S)
    with torch.no_grad():
        denoise = lambda x, t: om.denoiser_forward(sd, cond, x.float().view(B, F, 30), torch.full((B,), t), 1, 2).reshape(B * F, 30)
        want = odpm.dpm_sample_loop(odim.abar(), denoise, x_T.reshape(B * F, 30), S)
    assert torch.isfinite(got).all()
    close(got.reshape(B * F, 30), want, 5e-2, "trajectory")


@pytest.mark.parametrize("S", [1, 2])
def test_one_and_two_steps_are_ddim_eta_zero_bit_for_bit(S):
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F, K = 6, 10, 3
    m, _ = _small_denoiser(F=F, L=1)
    _pack_cond(m, B, 7)
    y = torch.randn(B, F, 30, generator=torch.Generator().manual_seed(9)).cuda()
    mask = (torch.rand(B, F, 30, generator=torch.Generator().manual_seed(10)) < 0.4).cuda()
    gd = GaussianDiffusion(device="cuda")
    for kw in (dict(), dict(guidance_scale=2.5), dict(known=y, known_mask=mask), dict(num_samples=K),
               dict(num_samples=K, guidance_scale=2.5, known=y, known_mask=mask)):
        for use_graph in (False, True):
            a = gd.sample(m, B, seed=4, use_graph=use_graph, dpm_steps=S, **kw)
            b = gd.sample(m, B, seed=4, use_graph=use_graph, ddim_steps=S, eta=0.0, **kw)
            assert torch.isfinite(a).all() and torch.equal(a, b), (kw, use_graph)


@pytest.mark.parametrize("S", [7, 10])
@pytest.mark.parametrize("s", [1.0, 2.5])
def test_graph_replay_equals_eager(S, s):
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F = 8, 10
    m, _ = _small_denoiser(F=F, L=1)
    _pack_cond(m, B, 4)
    gd = GaussianDiffusion(num_timesteps=20, device="cuda")
    a = gd.sample(m, B, seed=5, dpm_steps=S, guidance_scale=s, use_graph=False)
    b = gd.sample(m, B, seed=5, dpm_steps=S, guidance_scale=s)
    key = (id(m), B, ("dpm", S)) + ((s,) if s != 1.0 else ())
    graph = gd._graphs[key]["graph"]
    c = gd.sample(m, B, seed=5, dpm_steps=S, guidance_scale=s)        # second call replays the cached graph only
    assert graph is not None and gd._graphs[key]["graph"] is graph
    assert torch.isfinite(a).all()
    assert torch.equal(b, a) and torch.equal(c, a)


def test_interleaved_samplers_never_share_a_graph():
    """DPM-7, DPM-10, DDIM-7 and DDPM on one model and batch size each capture their own graph; in any order each result
    equals a fresh eager run of its schedule."""
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F = 8, 10
    m, _ = _small_denoiser(F=F, L=1)
    _pack_cond(m, B, 1)
    schedules = [dict(dpm_steps=7), dict(dpm_steps=10), dict(ddim_steps=7), dict()]
    want = [GaussianDiffusion(num_timesteps=20, device="cuda").sample(m, B, seed=5, use_graph=False, **kw) for kw in schedules]
    gd = GaussianDiffusion(num_timesteps=20, device="cuda")
    for k in (0, 2, 3, 1, 0, 3, 2, 1, 1, 0):
        assert torch.equal(gd.sample(m, B, seed=5, **schedules[k]), want[k]), k
    assert len(gd._graphs) == 4
    assert all(not torch.equal(want[i], want[j]) for i in range(4) for j in range(i))


@pytest.mark.parametrize("S", [3, 10])
def test_sample_equals_known_values_exactly(S):
    from inferbiomechanics_b200.cli.train import known_quantity_mask
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F = 6, 10
    m, _ = _small_denoiser(F=F, L=1)
    _pack_cond(m, B, 5)
    gd = GaussianDiffusion(device="cuda")
    y = torch.randn(B, F, 30, generator=torch.Generator().manual_seed(9)) * 4
    rand = torch.rand(B, F, 30, generator=torch.Generator().manual_seed(10)) < 0.4
    for s in (1.0, 2.5):
        for K, mask in ((None, rand), (3, known_quantity_mask(("force",)))):
            full = mask.expand(B, F, 30)
            x = gd.sample(m, B, seed=4, guidance_scale=s, num_samples=K, dpm_steps=S,
                          known=torch.where(full, y, torch.full_like(y, NAN)).cuda(), known_mask=mask.cuda()).cpu()
            draws = x.unsqueeze(0) if K is None else x
            assert torch.isfinite(draws).all(), (s, K)
            for d in draws:
                assert torch.equal(d[full], y[full]), (s, K)
            assert not torch.equal(draws[0][~full], y[~full])


@pytest.mark.parametrize("kw", [dict(dpm_steps=7), dict(dpm_steps=6, guidance_scale=2.5)], ids=["plain", "guided"])
def test_num_samples_is_the_call_on_replicated_windows(kw):
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F, K = 6, 10, 3
    m, _ = _small_denoiser(F=F, L=1)
    _pack_cond(m, B, 3)
    gd = GaussianDiffusion(num_timesteps=15, device="cuda")
    got = gd.sample(m, B, seed=5, num_samples=K, **kw)
    again = gd.sample(m, B, seed=5, num_samples=K, **kw)
    _replicate(m, B, K)
    want = GaussianDiffusion(num_timesteps=15, device="cuda").sample(m, B * K, seed=5, use_graph=False, **kw)
    assert tuple(got.shape) == (K, B, F, 30)
    assert torch.equal(got.reshape(B * K, F, 30), want) and torch.equal(again, got)
    assert not torch.equal(got[0], got[1])                  # the draws start from different x_T


def test_sample_windows_with_dpm_matches_direct_calls():
    from inferbiomechanics_b200 import ops
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    F, N, batch = 10, 21, 8
    m, _ = _small_denoiser(F=F, L=1)
    eng = m.engine()
    gd = GaussianDiffusion(num_timesteps=12, device="cuda")
    cond = torch.randn(N, F, 177, generator=torch.Generator().manual_seed(4)).pin_memory()
    for kw in (dict(dpm_steps=5), dict(dpm_steps=4, guidance_scale=2.5)):
        shards = [gd.sample_windows(m, cond, batch=batch, seed=9, rank=r, world=2, **kw) for r in range(2)]
        assert [len(s[0]) for s in shards] == [11, 10]
        for r, (rng, x0) in enumerate(shards):
            assert tuple(x0.shape) == (len(rng), F, 30) and torch.isfinite(x0).all()
            for i, a in enumerate(range(rng.start, rng.stop, batch)):
                b = min(a + batch, rng.stop)
                ops.pack_inputs([cond[a:b].reshape(-1, 177).cuda()], (b - a) * F, F, out_bf16=eng.xc(b - a, False),
                                frame_stride=eng.ld_in, win_extra=0, col0=30)
                want = gd.sample(m, b - a, seed=9 + r + 7919 * i, **kw)
                assert torch.equal(x0[a - rng.start:b - rng.start], want.cpu()), (kw, r, i)


def test_sampler_refusals_launch_nothing():
    from inferbiomechanics_b200 import _lib
    from inferbiomechanics_b200.diffusion import GaussianDiffusion
    B, F = 4, 10
    m, _ = _small_denoiser(F=F, L=1)
    gd = GaussianDiffusion(num_timesteps=20, device="cuda")
    m.engine()
    n = _lib.launch_count
    for kw in (dict(dpm_steps=5, noise=lambda t: None), dict(dpm_steps=5, eta=0.5), dict(dpm_steps=5, ddim_steps=5),
               dict(dpm_steps=21), dict(dpm_steps=0)):
        with pytest.raises(ValueError):
            gd.sample(m, B, **kw)
    assert _lib.launch_count == n


# ---------------------------------------- CLI -------------------------------------------------------------------------
def _run(argv):
    from inferbiomechanics_b200.main import main
    return main(argv)


def test_cli_analyze_with_dpm(tmp_path, capsys):
    ck = str(tmp_path / "ck")
    common = ["--no-wandb", "--synthetic-windows", "512", "--checkpoint-dir", ck, "--history-len", "50", "--stride", "1",
              "--model-type", "diffusion", "--batch-size", "64"]
    _run(["train", *common, "--epochs", "1", "--max-batches", "3", "--cond-drop-prob", "0.1"])   # guidance needs cond-drop
    capsys.readouterr()
    dpm = ["--sampler", "dpmpp2m", "--sampling-steps", "10"]
    for extra in ([], ["--output-data-format", "last_frame"]):
        an = _run(["analyze", *common, *dpm, *extra])
        loss = an.last_reports["dev"]["loss"]
        assert math.isfinite(loss) and loss > 0, (extra, loss)
    out = capsys.readouterr().out
    assert re.search(r"dev set evaluation \(\d+ windows\):", out), out
    an = _run(["analyze", *common, *dpm, "--num-samples", "2"])
    out = capsys.readouterr().out
    assert re.search(r"dev set evaluation \(\d+ windows, ensemble mean of 2 samples\):", out), out
    assert math.isfinite(an.last_ensemble_reports["dev"]["force"]["crps"])
    an = _run(["analyze", *common, *dpm, "--given-quantities", "force"])
    out = capsys.readouterr().out
    assert re.search(r"dev set evaluation \(\d+ windows, given force\):", out), out
    for split in ("dev", "train"):
        rep = an.last_reports[split]
        assert rep["force_r"] == 0.0 and not rep["force"].any(), rep
        assert math.isfinite(rep["moment_r"]) and rep["moment_r"] > 0
    an = _run(["analyze", *common, *dpm, "--guidance-scale", "2.5"])
    out = capsys.readouterr().out
    assert re.search(r"dev set evaluation \(\d+ windows, guidance scale 2\.5\):", out), out
    assert math.isfinite(an.last_reports["dev"]["loss"])
    with pytest.raises(ValueError, match="--eta"):
        _run(["analyze", *common, *dpm, "--eta", "0.5"])
