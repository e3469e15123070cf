"""The fp64 GEMM oracle (tests/gemm_oracle.py) against an independent torch statement of the same contract at tiny shapes:
taps through conv1d, activation derivatives through autograd, the bitmask through numpy.  No GPU needed."""
import itertools

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import gemm_oracle as go

TORCH_ACT = {"none": lambda x: x, "relu": F.relu, "sigmoid": torch.sigmoid, "tanh": torch.tanh, "elu": F.elu, "silu": F.silu}


def _bf16(*shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(torch.bfloat16)


def _valid(act, aux_mode, mask_mode):
    try:
        go.check_epilogue(act, aux_mode, mask_mode)
        return True
    except ValueError:
        return False


COMBOS = list(itertools.product(go.ACTS, (0, 1, 2), (0, 1, 2), (1, 3)))


@pytest.mark.parametrize("act,aux_mode,mask_mode,taps", COMBOS)
def test_oracle_matches_torch(act, aux_mode, mask_mode, taps):
    M, N, C = 11, 64, 72 if taps > 1 else 40
    K = taps * C
    Cp = (C + 63) // 64 * 64 if taps > 1 else C
    A = _bf16(M + taps - 1, C, seed=1)
    B = torch.zeros(N, taps * Cp, dtype=torch.bfloat16)
    W = _bf16(N, C, taps, seed=2, scale=0.2)                                # conv1d weight [out, in, tap]
    for j in range(taps):
        B[:, j * Cp:j * Cp + C] = W[:, :, j]
    bias = torch.randn(N, generator=torch.Generator().manual_seed(3))
    z = _bf16(M, N, seed=4).double()
    kw = dict(bias=bias, act=act, taps=taps, aux_mode=aux_mode, mask_mode=mask_mode)
    mask = torch.randint(0, 256, (M, N // 8), generator=torch.Generator().manual_seed(5), dtype=torch.uint8)
    if aux_mode == 1:
        kw["aux"] = z.to(torch.bfloat16)
    if aux_mode == 2:
        kw["aux"] = TORCH_ACT[act](z).to(torch.bfloat16)                     # a saved activation output
    if mask_mode == 2:
        kw["mask"] = mask
    if not _valid(act, aux_mode, mask_mode):
        with pytest.raises(ValueError):
            go.gemm_ref(A, B, M, N, K, **kw)
        return
    ref, bound = go.gemm_ref(A, B, M, N, K, **kw)

    x = A.double().t().unsqueeze(0)                                          # [1, C, M + taps - 1]
    pre = F.conv1d(x, W.double(), bias.double()).squeeze(0).t()             # [M, N]
    if aux_mode == 1:
        want = TORCH_ACT[act](pre) + z.to(torch.bfloat16).double()
    elif aux_mode == 2:
        # the from-output derivative formula, evaluated at act(z), is autograd's act'(z)
        zz = z.clone().requires_grad_(True)
        TORCH_ACT[act](zz).sum().backward()
        y = kw["aux"].double()
        g_formula = go.act_grad_from_output(TORCH_ACT[act](z), act)
        torch.testing.assert_close(g_formula, zz.grad, rtol=1e-9, atol=1e-12)
        want = pre * go.act_grad_from_output(y, act)
    elif mask_mode == 2:
        bits = torch.from_numpy(np.unpackbits(mask.numpy(), axis=1, bitorder="little")).bool()
        want = torch.where(bits, pre, torch.zeros_like(pre))
    else:
        want = TORCH_ACT[act](pre)
    torch.testing.assert_close(ref, want, rtol=1e-12, atol=1e-12)
    assert bool((bound >= 0).all())
    # the bound admits the output rounding of a bf16 result, and is far below an error of 1 %
    assert go.max_violation(ref.to(torch.bfloat16), ref, bound) == ""
    big = ref.abs() > 0.1
    assert bool((bound[big] < 1e-2 * ref[big].abs()).all())


@pytest.mark.parametrize("a_mn,b_mn", [(False, False), (True, False), (False, True), (True, True)])
def test_oracle_operand_layouts_and_accumulate(a_mn, b_mn):
    M, N, K = 9, 13, 21
    Al, Bl = _bf16(M, K, seed=11), _bf16(N, K, seed=12)
    A = Al.t().contiguous() if a_mn else Al
    B = Bl.t().contiguous() if b_mn else Bl
    d0 = torch.randn(M, N, generator=torch.Generator().manual_seed(13))
    ref, bound = go.gemm_ref(A, B, M, N, K, a_mn=a_mn, b_mn=b_mn, accumulate=True, d_init=d0, out_f32=True)
    torch.testing.assert_close(ref, d0.double() + Al.double() @ Bl.double().t(), rtol=1e-12, atol=1e-12)
    assert go.max_violation(ref.float(), ref, bound) == ""
    with pytest.raises(ValueError):
        go.gemm_ref(A, B, M, N, K, a_mn=a_mn, b_mn=b_mn, accumulate=True, d_init=d0, out_f32=False)


def test_oracle_taps_b_mn_layout():
    """MN-major B with taps: tap j's rows start at j * round_up(C, 64)."""
    M, N, C, taps = 7, 16, 72, 3
    A = _bf16(M + taps - 1, C, seed=21)
    W = _bf16(N, C, taps, seed=22)
    Bt = torch.zeros(taps * 128, N, dtype=torch.bfloat16)
    for j in range(taps):
        Bt[j * 128:j * 128 + C] = W[:, :, j].t()
    ref, _ = go.gemm_ref(A, Bt, M, N, taps * C, b_mn=True, taps=taps)
    want = F.conv1d(A.double().t().unsqueeze(0), W.double()).squeeze(0).t()
    torch.testing.assert_close(ref, want, rtol=1e-12, atol=1e-12)


def test_mask_bytes_and_colsum():
    g = torch.Generator().manual_seed(31)
    out = torch.randn(70, 128, generator=g).to(torch.bfloat16)
    out[3, 5] = 0.0
    want = np.packbits((out.float().numpy() > 0), axis=1, bitorder="little")
    assert np.array_equal(go.mask_bytes(out, 70, 128).numpy(), want)
    assert torch.equal(go.mask_bits(go.mask_bytes(out, 70, 128), 70, 128), out > 0)
    init = torch.full((128,), 2.0)
    ref, bound = go.colsum_ref(out, 65, 128, init)
    torch.testing.assert_close(ref, 2.0 + out[:65].double().sum(0), rtol=1e-12, atol=1e-12)
    assert bool((bound > 0).all()) and bool((bound < 1e-3).all())


def test_max_violation_reports_nan_and_worst():
    ref = torch.zeros(2, 3, dtype=torch.float64)
    bound = torch.full((2, 3), 0.1, dtype=torch.float64)
    out = torch.zeros(2, 3)
    assert go.max_violation(out, ref, bound) == ""
    out[1, 2] = 0.5
    assert "[1, 2]" in go.max_violation(out, ref, bound)
    out[0, 0] = float("nan")
    assert "[0, 0]" in go.max_violation(out, ref, bound)
