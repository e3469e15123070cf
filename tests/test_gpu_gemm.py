"""GPU parity: tcgen05 GEMM (through the C ABI) vs fp64 matmul of the same bf16-rounded operands.

Tolerance: operands are exact bf16 on both sides and accumulation is fp32 in TMEM, so the only
differences are fp32 summation order and the final output rounding: rtol 2e-2*|bf16 ulp| for bf16
outputs (one bf16 rounding = 2^-8 relative) and 1e-4 relative-to-scale for fp32 outputs.
"""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _mk(rows, cols, ld, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    buf = torch.zeros(rows, ld, dtype=torch.bfloat16)
    buf[:, :cols] = (torch.randn(rows, cols, generator=g) * scale).to(torch.bfloat16)
    return buf


ACTS = {
    "none": lambda x: x, "relu": lambda x: x.clamp_min(0), "sigmoid": torch.sigmoid, "tanh": torch.tanh,
    "elu": torch.nn.functional.elu, "silu": torch.nn.functional.silu,
}


def _check(out, ref, bf16_out, what):
    out = out.double().cpu()
    scale = ref.abs().max().item() + 1e-30
    err = (out - ref).abs().max().item()
    tol = (1.0 / 128 if bf16_out else 2e-4) * scale
    assert err <= tol, f"{what}: max abs err {err:.4g} > {tol:.4g} (scale {scale:.4g})"


@pytest.mark.parametrize("M,N,K,act,out_f32", [
    (128, 256, 64, "none", False),
    (256, 256, 128, "relu", False),
    (300, 300, 1470, "sigmoid", False),      # FeedForward layer shapes, ragged everything
    (32, 512, 1470, "sigmoid", False),       # BASELINE config 1 batch
    (1000, 512, 512, "tanh", True),
    (520, 30, 512, "none", True),            # 30-channel head, fp32 out
    (777, 1536, 512, "none", False),         # fused QKV
    (640, 2048, 512, "relu", False),
    (640, 512, 2048, "none", False),
    (130, 128, 208, "elu", False),
    (4096, 64, 72, "silu", False),
    (6, 40, 1470, "tanh", False),            # narrow bf16 outputs (hidden sizes 40 / 24 of the golden FeedForward case)
    (6, 24, 40, "tanh", False),
    (200, 8, 64, "none", False),
    (200, 12, 64, "none", True),
    (5000, 512, 1472, "sigmoid", False),     # K >= 1024 but 20 row blocks x 1 column-tile pair < 148: single column tiles
    (777, 1000, 2048, "none", True),
    (70000, 512, 1024, "relu", False),
    (40000, 1536, 512, "none", False),       # >= 148 row blocks, K <= 512 (also the A-stationary schedule when IBM_GEMM_AS=1)
    (50000, 600, 256, "relu", False),        # ... ragged N, K = 4 k-blocks
    (38011, 512, 328, "silu", False),        # ... ragged M and K
    (40000, 1000, 512, "tanh", True),        # ... fp32 output
])
def test_gemm_forward(M, N, K, act, out_f32):
    from inferbiomechanics_b200 import ops
    lda, ldb = ops.round_up(K, 8), ops.round_up(K, 8)
    A, B = _mk(M, K, lda, 1), _mk(N, K, ldb, 2, 1.0 / math.sqrt(K))
    bias = torch.randn(N, generator=torch.Generator().manual_seed(3))
    ldd = ops.round_up(N, 4 if out_f32 else 8)
    out = torch.full((M, ldd), 7.0, dtype=torch.float32 if out_f32 else torch.bfloat16, device="cuda")
    ops.gemm(A.cuda(), B.cuda(), out, M, N, K, bias=bias.cuda(), act=act)
    torch.cuda.synchronize()
    ref = ACTS[act](A[:, :K].double() @ B[:, :K].double().t() + bias.double())
    _check(out[:, :N], ref, not out_f32, f"fwd {M}x{N}x{K} {act}")
    # TMA clips stores at the tensor extent rounded up to a 16-byte chunk: columns beyond that are untouched
    gran = 4 if out_f32 else 8
    n_touched = (N + gran - 1) // gran * gran
    if ldd > n_touched:
        assert torch.all(out[:, n_touched:].float() == 7.0)


# of the K >= 1024 shapes only (20000, 1024, 1536) has enough work items for two-tile supertiles
@pytest.mark.parametrize("M,N,K", [(515, 512, 256), (300, 200, 128), (40000, 512, 512), (1000, 2048, 512),
                                   (3000, 512, 2048), (20000, 1024, 1536), (300, 504, 1024)])
def test_gemm_residual_and_dact(M, N, K):
    from inferbiomechanics_b200 import ops
    A, B = _mk(M, K, K, 4), _mk(N, K, K, 5, 1.0 / math.sqrt(K))
    bias = torch.randn(N, generator=torch.Generator().manual_seed(6))
    aux = _mk(M, N, N, 7)
    out = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
    ops.gemm(A.cuda(), B.cuda(), out, M, N, K, bias=bias.cuda(), aux=aux.cuda(), aux_mode=1)
    ref = A.double() @ B.double().t() + bias.double() + aux.double()
    _check(out, ref, True, "residual")
    for act, dfn in (("relu", lambda y: (y > 0).double()), ("sigmoid", lambda y: y * (1 - y)),
                     ("tanh", lambda y: 1 - y * y), ("elu", lambda y: torch.where(y > 0, torch.ones_like(y), y + 1))):
        y = ACTS[act](_mk(M, N, N, 8).float()).to(torch.bfloat16)
        ops.gemm(A.cuda(), B.cuda(), out, M, N, K, act=act, aux=y.cuda(), aux_mode=2)
        ref = (A.double() @ B.double().t()) * dfn(y.double())
        _check(out, ref, True, f"dact {act}")


@pytest.mark.parametrize("M,N,K", [(515, 512, 256), (4000, 2048, 512), (77, 200, 128), (130, 72, 64), (1000, 512, 1024)])
def test_gemm_fused_colsum(M, N, K):
    """colsum_out += column sums of the bf16 output rows < M (bias gradient of the producing layer), in the same launch."""
    from inferbiomechanics_b200 import ops
    A, B = _mk(M, K, K, 51), _mk(K, ops.round_up(N, 8), ops.round_up(N, 8), 52, 1.0 / math.sqrt(K))
    h = torch.relu(_mk(M, N, ops.round_up(N, 8), 53).float()).to(torch.bfloat16)
    bias = torch.randn(N, generator=torch.Generator().manual_seed(54))
    out = torch.empty(M, ops.round_up(N, 8), dtype=torch.bfloat16, device="cuda")
    cs = torch.full((N,), 2.0, device="cuda")
    # dgrad through relu (aux epilogue) and a plain biased forward (non-aux epilogue)
    ops.gemm(A.cuda(), B.cuda(), out, M, N, K, b_mn=True, act="relu", aux=h.cuda(), aux_mode=2, colsum=cs)
    want = 2.0 + out[:, :N].double().sum(0).cpu()
    torch.testing.assert_close(cs.double().cpu(), want, rtol=1e-4, atol=1e-3 * math.sqrt(M))
    ref = (A.double() @ B[:, :N].double()) * (h[:, :N].double() > 0)
    _check(out[:, :N], ref, True, "dact relu with colsum")
    cs.fill_(0.0)
    ops.gemm(A.cuda(), B.cuda(), out, M, N, K, b_mn=True, bias=bias.cuda(), colsum=cs)
    torch.testing.assert_close(cs.double().cpu(), out[:, :N].double().sum(0).cpu(), rtol=1e-4, atol=1e-3 * math.sqrt(M))


@pytest.mark.parametrize("M,N,K", [(256, 128, 192), (1000, 1470, 512), (333, 512, 300), (640, 208, 512), (6, 32, 30), (70, 24, 40),
                                   (45000, 512, 512)])       # out-proj dgrad shape, >= 148 row blocks
def test_gemm_dgrad_b_mn_major(M, N, K):
    """dX[M,N] = dY[M,K] · W[K,N]  with W stored row-major [K, N] (MN-major B operand)."""
    from inferbiomechanics_b200 import ops
    dY = _mk(M, K, ops.round_up(K, 8), 11)
    W = _mk(K, N, ops.round_up(N, 8), 12, 1.0 / math.sqrt(K))
    out = torch.empty(M, ops.round_up(N, 8), dtype=torch.bfloat16, device="cuda")
    ops.gemm(dY.cuda(), W.cuda(), out, M, N, K, b_mn=True)
    ref = dY[:, :K].double() @ W[:, :N].double()
    _check(out[:, :N], ref, True, f"dgrad {M}x{N}x{K}")


@pytest.mark.parametrize("Mtok,Nout,Kin,split", [(512, 128, 256, 1), (4000, 512, 512, 0), (1111, 300, 512, 3),
                                                 (2048, 512, 1472, 0), (6400, 30, 512, 0), (6, 30, 32, 0), (33, 48, 24, 0)])
def test_gemm_wgrad_mn_mn_accumulate(Mtok, Nout, Kin, split):
    """dW[Nout,Kin] += dY[Mtok,Nout]^T · X[Mtok,Kin]: both operands MN-major, split-K TMA reduce-add."""
    from inferbiomechanics_b200 import ops
    dY = _mk(Mtok, Nout, ops.round_up(Nout, 8), 21)
    X = _mk(Mtok, Kin, ops.round_up(Kin, 8), 22)
    init = torch.randn(Nout, Kin, generator=torch.Generator().manual_seed(23))
    dW = init.clone().cuda()
    ops.gemm(dY.cuda(), X.cuda(), dW, Nout, Kin, Mtok, a_mn=True, b_mn=True, accumulate=True, split_k=split)
    ref = init.double() + dY[:, :Nout].double().t() @ X[:, :Kin].double()
    _check(dW, ref, False, f"wgrad {Mtok} {Nout}x{Kin}")


@pytest.mark.parametrize("M,N,K", [(515, 512, 256), (4000, 2048, 512), (300, 128, 64), (40000, 2048, 512)])
def test_gemm_relu_sign_bitmask(M, N, K):
    """mask_mode 1 writes (relu output > 0) bits next to the forward output; mask_mode 2 applies them in the dgrad:
    identical to the aux_mode-2 path that re-reads the activation."""
    from inferbiomechanics_b200 import ops
    X, W = _mk(M, K, K, 61), _mk(N, K, K, 62, 1.0 / math.sqrt(K))
    bias = torch.randn(N, generator=torch.Generator().manual_seed(63))
    h = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
    mask = torch.full((M, N // 8), 0xAA, dtype=torch.uint8, device="cuda")
    ops.gemm(X.cuda(), W.cuda(), h, M, N, K, bias=bias.cuda(), act="relu", mask=mask, mask_mode=1)
    bits = torch.from_numpy(np.unpackbits(mask.cpu().numpy(), axis=1, bitorder="little")).bool()
    assert torch.equal(bits, h.cpu() > 0)                          # bit-exact: the sign of what was stored
    # dgrad: dY [M, Kd] · Wd [Kd, N]  gated by the bits  ==  the aux_mode-2 result, element for element
    Kd = 256
    dY, Wd = _mk(M, Kd, Kd, 64), _mk(Kd, N, N, 65, 1.0 / math.sqrt(Kd))
    a = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
    b = torch.empty_like(a)
    ca, cb = torch.zeros(N, device="cuda"), torch.zeros(N, device="cuda")
    ops.gemm(dY.cuda(), Wd.cuda(), a, M, N, Kd, b_mn=True, mask=mask, mask_mode=2, colsum=ca)
    ops.gemm(dY.cuda(), Wd.cuda(), b, M, N, Kd, b_mn=True, act="relu", aux=h, aux_mode=2, colsum=cb)
    assert torch.equal(a, b)
    torch.testing.assert_close(ca, cb, rtol=1e-4, atol=1e-3 * math.sqrt(M))
    with pytest.raises(ValueError):
        ops.gemm(X.cuda(), W.cuda(), h, M, N, K, mask=mask[:, :-1].contiguous(), mask_mode=1)      # ldmask*8 < N


def test_gemm_a_stationary_mode_parity():
    """The experimental A-stationary schedule (IBM_GEMM_AS=1, read once per process) gives the same results: run the QKV
    shape in a subprocess with the switch on and compare with this process (switch off)."""
    import subprocess
    import sys
    code = (
        "import torch, math, sys; sys.path.insert(0, '.');"
        "from inferbiomechanics_b200 import ops;"
        "g = torch.Generator().manual_seed(3);"
        "A = torch.randn(40000, 512, generator=g).to(torch.bfloat16).cuda();"
        "B = (torch.randn(1536, 512, generator=g) / math.sqrt(512)).to(torch.bfloat16).cuda();"
        "out = torch.empty(40000, 1536, dtype=torch.bfloat16, device='cuda');"
        "ops.gemm(A, B, out, 40000, 1536, 512, act='relu');"
        "torch.cuda.synchronize(); print(out.float().sum().item(), out.float().abs().max().item(), out[12345, 777].item())")
    import os
    outs = []
    for flag in ("0", "1"):
        env = dict(os.environ, IBM_GEMM_AS=flag)
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=os.path.dirname(os.path.dirname(__file__)))
        assert r.returncode == 0, r.stderr[-800:]
        outs.append([float(x) for x in r.stdout.split()])
    assert outs[0][1] == outs[1][1] and outs[0][2] == outs[1][2]          # same tile arithmetic: identical elements
    assert abs(outs[0][0] - outs[1][0]) <= 1e-6 * abs(outs[0][0]) + 1e-3


def test_gemm_taps_implicit_conv():
    """K = taps*C: k-block kb reads A rows m + kb // kb_per_tap (temporal convolution as a GEMM)."""
    from inferbiomechanics_b200 import ops
    rows, C, N, taps = 400, 128, 256, 7
    Xp = _mk(rows + taps - 1, C, C, 31)
    W = _mk(N, taps * C, taps * C, 32, 1.0 / math.sqrt(taps * C))
    out = torch.empty(rows, N, dtype=torch.bfloat16, device="cuda")
    ops.gemm(Xp.cuda(), W.cuda(), out, rows, N, taps * C, taps=taps)
    ref = torch.zeros(rows, N, dtype=torch.float64)
    for j in range(taps):
        ref += Xp[j:j + rows].double() @ W[:, j * C:(j + 1) * C].double().t()
    _check(out, ref, True, "taps")


def test_gemm_argument_errors():
    from inferbiomechanics_b200 import ops
    A = torch.zeros(8, 12, dtype=torch.bfloat16, device="cuda")
    out = torch.zeros(8, 8, dtype=torch.bfloat16, device="cuda")
    with pytest.raises(ValueError):
        ops.gemm(A, A, out, 8, 8, 12)                   # lda=12 is not a multiple of 8
    with pytest.raises(ValueError):
        ops.gemm(out, out, out, 0, 8, 8)                # empty problem


def test_gemm_pad_column_contract():
    """Header contract: when K % 8 != 0 the operand pad columns [K, ld) must be zero.  This test pins
    what the hardware does otherwise (TMA bounds-checks the inner dimension in 16-byte chunks), so a
    change in that behaviour is noticed: garbage in the last partial chunk DOES leak into the result,
    garbage beyond it does not."""
    from inferbiomechanics_b200 import ops
    M, N, K = 128, 128, 68                # 68 = 8*8 + 4: last chunk holds cols 64..71, ld = 80
    A, B = _mk(M, K, 80, 41), _mk(N, K, 80, 42)
    ref = A[:, :K].double() @ B[:, :K].double().t()
    out = torch.empty(M, N, dtype=torch.float32, device="cuda")
    A2, B2 = A.clone(), B.clone()
    A2[:, 72:] = 100.0; B2[:, 72:] = 100.0          # beyond the last partial chunk: must be ignored
    ops.gemm(A2.cuda(), B2.cuda(), out, M, N, K)
    _check(out, ref, False, "garbage beyond the partial chunk")
    A3, B3 = A.clone(), B.clone()
    A3[:, 68:72] = 1.0; B3[:, 68:72] = 1.0           # inside the partial chunk
    ops.gemm(A3.cuda(), B3.cuda(), out, M, N, K)
    leaked = (out.double().cpu() - ref).abs().max().item()
    assert leaked < 1e-3 or abs(leaked - 4.0) < 1e-2, leaked
    print("TMA inner-dimension bound granularity:", "16-byte chunk (pads must be zero)" if leaked > 1 else "element")


# ---------------------------------------------------------------------------------------------------
# The EXACT GEMM shapes of the benchmarked denoiser step (BASELINE configs[1]: 4096 windows x 50 frames = 204 800
# rows, d = 512, FFN 2048, fused QKV 1536): forward / dgrad epilogue variants as engine.EncoderLayerPlan issues
# them, and the weight gradients with their 204 800-long reduction (default split-K + TMA reduce-add).
# Operands are generated on the device and the fp64 reference product runs on the device too (the CPU would
# need minutes for 4 x 10^11 multiply-adds); same tolerance as above.
# ---------------------------------------------------------------------------------------------------
M_BENCH = 204800


def _dev(rows, cols, seed, scale=1.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(rows, cols, generator=g, device="cuda") * scale).to(torch.bfloat16)


def _check_dev(out, ref, bf16_out, what):
    scale = ref.abs().max().item() + 1e-30
    err = (out.double() - ref).abs().max().item()
    tol = (1.0 / 128 if bf16_out else 2e-4) * scale
    assert err <= tol, f"{what}: max abs err {err:.4g} > {tol:.4g} (scale {scale:.4g})"


@pytest.mark.parametrize("name,N,K,kind", [
    ("qkv", 1536, 512, "bias"), ("out_proj", 512, 512, "residual"), ("ffn1", 2048, 512, "relu_mask"), ("ffn2", 512, 2048, "residual"),
])
def test_gemm_bench_shapes_forward(name, N, K, kind):
    from inferbiomechanics_b200 import ops
    M = M_BENCH
    A, W = _dev(M, K, 1), _dev(N, K, 2, 1.0 / math.sqrt(K))
    bias = torch.randn(N, generator=torch.Generator(device="cuda").manual_seed(3), device="cuda")
    out = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
    ref = A.double() @ W.double().t() + bias.double()
    if kind == "bias":
        ops.gemm(A, W, out, M, N, K, bias=bias)
    elif kind == "residual":
        aux = _dev(M, N, 4)
        ops.gemm(A, W, out, M, N, K, bias=bias, aux=aux, aux_mode=1)
        ref += aux.double()
    else:
        mask = torch.zeros(M, N // 8, dtype=torch.uint8, device="cuda")
        ops.gemm(A, W, out, M, N, K, bias=bias, act="relu", mask=mask, mask_mode=1)
        ref.clamp_min_(0)
        bits = (mask.unsqueeze(-1) >> torch.arange(8, device="cuda", dtype=torch.uint8)) & 1
        assert torch.equal(bits.view(M, N).bool(), out > 0)
    _check_dev(out, ref, True, f"{name} forward at M={M}")


@pytest.mark.parametrize("name,N,K,kind", [
    ("ffn2_dgrad", 2048, 512, "mask_colsum"), ("ffn1_dgrad", 512, 2048, "residual"), ("out_proj_dgrad", 512, 512, "plain"),
    ("in_proj_dgrad", 512, 1536, "residual"),
])
def test_gemm_bench_shapes_dgrad(name, N, K, kind):
    """dX[M,N] = dY[M,K] · W[K,N] (W row-major = MN-major B operand), epilogues as in EncoderLayerPlan.backward."""
    from inferbiomechanics_b200 import ops
    M = M_BENCH
    dY, W = _dev(M, K, 11), _dev(K, N, 12, 1.0 / math.sqrt(K))
    out = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
    ref = dY.double() @ W.double()
    if kind == "plain":
        ops.gemm(dY, W, out, M, N, K, b_mn=True)
    elif kind == "residual":
        aux = _dev(M, N, 13)
        ops.gemm(dY, W, out, M, N, K, b_mn=True, aux=aux, aux_mode=1)
        ref += aux.double()
    else:
        g = torch.Generator(device="cuda").manual_seed(14)
        mask = torch.randint(0, 256, (M, N // 8), generator=g, device="cuda", dtype=torch.uint8)
        cs = torch.zeros(N, device="cuda")
        ops.gemm(dY, W, out, M, N, K, b_mn=True, mask=mask, mask_mode=2, colsum=cs)
        bits = ((mask.unsqueeze(-1) >> torch.arange(8, device="cuda", dtype=torch.uint8)) & 1).view(M, N)
        ref *= bits.double()
        torch.testing.assert_close(cs.double(), out.double().sum(0), rtol=1e-4, atol=1e-3 * math.sqrt(M))
    _check_dev(out, ref, True, f"{name} at M={M}")


@pytest.mark.parametrize("name,Nout,Kin", [("ffn2_wgrad", 512, 2048), ("ffn1_wgrad", 2048, 512), ("out_proj_wgrad", 512, 512),
                                           ("qkv_wgrad", 1536, 512), ("head_wgrad", 30, 512)])
def test_gemm_bench_shapes_wgrad(name, Nout, Kin):
    """dW[Nout,Kin] += dY^T · X over a 204 800-long reduction, the engine's default split-K."""
    from inferbiomechanics_b200 import ops
    M = M_BENCH
    ldn = ops.round_up(Nout, 8)
    dY = torch.zeros(M, ldn, dtype=torch.bfloat16, device="cuda")
    dY[:, :Nout] = _dev(M, Nout, 21)
    X = _dev(M, Kin, 22)
    init = torch.randn(Nout, Kin, generator=torch.Generator(device="cuda").manual_seed(23), device="cuda")
    dW = init.clone()
    ops.gemm(dY, X, dW, Nout, Kin, M, a_mn=True, b_mn=True, accumulate=True)
    ref = init.double() + dY[:, :Nout].double().t() @ X.double()
    # fp32 accumulation of 204 800 products of unit-variance terms: scale ~ sqrt(M); same relative bar as above
    _check_dev(dW, ref, False, f"{name} reduction {M}")
