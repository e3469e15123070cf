"""Every Philox4x32-10 draw on the device against the numpy oracle (tests/philox_oracle.py): the dropout masks of
``ibm_dropout_bf16`` / ``ibm_dropout_bf16_dev`` bit for bit, and the diffusion noise of ``q_sample`` (both kernel paths)
and of the posterior / respaced steps with ``z == NULL``.

The normals go through __logf / __sincosf, so they are compared at 1e-4 absolute: the intrinsics' documented errors are
a few 1e-7 on these arguments, which the Box-Muller radius sqrt(-2 ln u) amplifies only for u within ~1e-5 of 1 (measured
on these seeded draws: at most 4e-5).  A wrong counter layout, seed / offset word or lane order shows up as an O(1)
difference."""
import numpy as np
import pytest
import torch

import philox_oracle as ph

pytestmark = pytest.mark.gpu

HI_SEED, HI_OFFSET = (1 << 32) + 7, (1 << 33) + 5


def _seeds():
    from inferbiomechanics_b200.engine import FeedForwardEngine
    from inferbiomechanics_b200.engine_groundlink import GroundlinkEngine
    return [(HI_SEED, HI_OFFSET), (GroundlinkEngine.CNN_DROPOUT_SEED, 4 * 3 + 2), (GroundlinkEngine.FC_DROPOUT_SEED, 3 * 5 + 1),
            (FeedForwardEngine.DROPOUT_SEED + 1, 3 * 1000 + 2)]


def _bf16_input(n, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(n, generator=g) * 3).to(torch.bfloat16)


def _same_bits(got, want, what):
    got = got.cpu().view(torch.int16)
    want = want.view(torch.int16)
    bad = (got != want).nonzero()
    assert bad.numel() == 0, f"{what}: {bad.numel()} of {got.numel()} elements differ, first at {bad[0].item()}"


@pytest.mark.parametrize("p", [0.0, 0.2, 0.25, 0.5, 0.9])
@pytest.mark.parametrize("n", [4, 1020, (1 << 20) + 4])
def test_dropout_matches_oracle_bit_for_bit(n, p):
    from inferbiomechanics_b200 import ops
    x = _bf16_input(n, n)
    xd = x.cuda()
    for seed, offset in _seeds():
        y = torch.full_like(xd, float("nan"))
        ops.dropout(xd, y, p, seed, offset)
        _same_bits(y, ph.dropout_bf16(x, p, seed, offset), f"n={n} p={p} seed={seed:#x} offset={offset:#x}")


@pytest.mark.parametrize("p", [0.2, 0.5])
def test_dropout_dev_equals_dropout_at_the_stepped_offset(p):
    """``ibm_dropout_bf16_dev`` with *step_dev = s draws the mask of offset add + mul * s, including steps that carry into
    the high word of the offset."""
    from inferbiomechanics_b200 import ops
    n, add, mul = 4096 + 4, 2, 4
    x = _bf16_input(n, 3).cuda()
    step_dev = torch.zeros(1, dtype=torch.int64, device="cuda")
    for seed, _ in _seeds():
        for s in (0, 1, 7, 1000, (1 << 31) + 3):
            step_dev.fill_(s)
            a, b = torch.empty_like(x), torch.empty_like(x)
            ops.dropout(x, a, p, seed, add, step_dev, mul)
            ops.dropout(x, b, p, seed, add + mul * s)
            assert torch.equal(a.view(torch.int16), b.view(torch.int16)), (seed, s)
            _same_bits(a, ph.dropout_bf16(x, p, seed, add + mul * s), f"dev step {s}")


def _check_normals(got, n, seed, offset, what):
    err = np.abs(got.double().cpu().numpy().reshape(-1) - ph.normals(n, seed, offset))
    worst = int(np.argmax(err))
    print(f"{what}: max |err| {err[worst]:.3g}")
    assert err[worst] <= 1e-4, f"{what}: element {worst} off by {err[worst]:.3g}"


@pytest.mark.parametrize("F", [1, 2, 3])
@pytest.mark.parametrize("seed,offset", [(HI_SEED, HI_OFFSET), (7, 1)])
def test_q_sample_noise_matches_oracle(F, seed, offset):
    """per window 30 * F values: F = 2 (60, a multiple of 4) takes the float4 path, F = 1 and 3 the scalar one; an odd
    window count leaves the last draw partly used."""
    from inferbiomechanics_b200 import ops
    from oracle import ddpm as oddpm
    sched = {k: v.cuda() for k, v in oddpm.make_schedule().items()}
    B = 2001
    x0 = torch.randn(B, F, 30, device="cuda", generator=torch.Generator("cuda").manual_seed(F))
    t = torch.randint(0, 1000, (B,), device="cuda", generator=torch.Generator("cuda").manual_seed(F + 1)).int()
    xt = torch.empty_like(x0)
    eps = torch.full_like(x0, float("nan"))
    ops.q_sample(x0, None, t, sched["sqrt_abar"], sched["sqrt_one_minus_abar"], xt_f32=xt, seed=seed, offset=offset, eps_out=eps)
    _check_normals(eps, B * F * 30, seed, offset, f"q_sample F={F}")
    tl = t.long()
    want = sched["sqrt_abar"][tl].view(B, 1, 1).double() * x0.double() + sched["sqrt_one_minus_abar"][tl].view(B, 1, 1).double() * eps.double()
    torch.testing.assert_close(xt.double(), want, rtol=0, atol=1e-5 * want.abs().max().item())


@pytest.mark.parametrize("respaced", [False, True])
def test_posterior_step_noise_matches_oracle(respaced):
    """``z == NULL``: the step draws its noise at counter offset ``offset + t``.  Tables with coef_x0 = coef_xt = 0 and
    sigma = 1 make the step's output that noise exactly; t = 0 draws none."""
    from inferbiomechanics_b200 import ops
    T, M = 1000, 4001
    zeros = torch.zeros(T, device="cuda")
    sigma = torch.ones(T, device="cuda")
    succ = (torch.arange(T, dtype=torch.int32, device="cuda") - 3).clamp_min(-1)
    x0h = torch.randn(M, 32, device="cuda")
    xt = torch.randn(M, 30, device="cuda")
    for t in (0, 1, 37, 999):
        t_dev = torch.tensor([t], dtype=torch.int32, device="cuda")
        out = torch.full((M, 30), float("nan"), device="cuda")
        ops.posterior_step(x0h, 32, xt, None, t_dev, zeros, zeros, sigma, M, x_prev=out, seed=HI_SEED, offset=HI_OFFSET,
                           t_succ=succ if respaced else None)
        if t == 0:
            assert torch.all(out == 0)
        else:
            _check_normals(out, M * 30, HI_SEED, HI_OFFSET + t, f"{'respaced' if respaced else 'posterior'} t={t}")
