"""fp64 oracle of the ibm_gemm_bf16 contract (include/ibm_b200.h).  TEST INFRASTRUCTURE ONLY.

``gemm_ref`` takes the arguments of ``ops.gemm`` (bf16 operands as stored, with their leading dimensions) and returns the
fp64 result of the full epilogue together with a per-element error bound for the kernel's output:

  pre       = sum_taps A_j · B_j^T (+ bias)            A_j = rows [j, j + M) of A, B_j = tap j's columns of B
  aux_mode 0: act(pre)            aux_mode 1: act(pre) + aux            aux_mode 2: pre · act'(aux), act' from the OUTPUT
  mask_mode 1: act(pre) (bits = stored output > 0)     mask_mode 2: pre where the bit is set, 0 elsewhere
  accumulate : D_init + A · B^T

  With taps the K range of B is taps blocks of round_up(K / taps, 64) columns (rows when B is MN-major): tap j's
  weights start at column j · round_up(K / taps, 64).  When K / taps is a multiple of 64 this is the plain [N, K] layout.

Error bound, per element (u = 2^-24, one fp32 rounding):
  accumulation   (K + 1) · u · (|A|·|B|^T + |bias|) · L,  L bounds |act'| (1 for none/relu/tanh/elu, 0.25 for sigmoid,
                 1.1 for silu); in aux_mode 2 the factor is |act'(aux)| itself, in mask_mode 2 the bit
  residual add   2u · (|act(pre)| + |aux|)                  (aux_mode 1)
  split-K        (splits + 1) · u · |D_init|                (accumulate; splits <= max(1, ceil(K / 64) / 8))
  activations    1e-6 · |ref|                               (__expf in sigmoid / silu)
  bf16 output    2^-8 · (|ref| + the above)                 (one round-to-nearest-even to 8 significant bits)
The accumulation term is the classical worst case of a K-term fp32 sum, so any tile-indexing error (a wrong row, column,
tap or k block) shows up as an error far above it, also in small outputs and in a single ragged tile.

``mask_bytes`` and ``colsum_ref`` judge the two side outputs from the output the kernel stored, as the kernel computes
them from it.
"""
from __future__ import annotations

import math

import torch

ACTS = ("none", "relu", "sigmoid", "tanh", "elu", "silu")
ACT_LIP = {"none": 1.0, "relu": 1.0, "tanh": 1.0, "elu": 1.0, "sigmoid": 0.25, "silu": 1.1}
U = 2.0 ** -24


def act_fwd(x: torch.Tensor, act: str) -> torch.Tensor:
    if act == "none":
        return x
    if act == "relu":
        return x.clamp_min(0)
    if act == "sigmoid":
        return torch.sigmoid(x)
    if act == "tanh":
        return torch.tanh(x)
    if act == "elu":
        return torch.where(x > 0, x, torch.expm1(x))
    if act == "silu":
        return x * torch.sigmoid(x)
    raise ValueError(act)


def act_grad_from_output(y: torch.Tensor, act: str) -> torch.Tensor:
    """act'(x) expressed through y = act(x) (the saved activation output of aux_mode 2)."""
    if act == "none":
        return torch.ones_like(y)
    if act == "relu":
        return (y > 0).to(y.dtype)
    if act == "sigmoid":
        return y * (1 - y)
    if act == "tanh":
        return 1 - y * y
    if act == "elu":
        return torch.where(y > 0, torch.ones_like(y), y + 1)
    raise ValueError(f"the derivative of {act} cannot be computed from its output")


def check_epilogue(act="none", aux_mode=0, mask_mode=0, out_f32=False, accumulate=False, bias=None, taps=1, a_mn=False):
    """The epilogue combinations ibm_gemm_bf16 computes; raises ValueError for the others, as the library does."""
    if act not in ACTS:
        raise ValueError(f"bad activation {act}")
    if aux_mode == 1 and act not in ("none", "relu", "elu"):
        raise ValueError("aux_mode 1 (residual) supports act none, relu, elu")
    if aux_mode == 2 and act == "silu":
        raise ValueError("aux_mode 2 needs an activation whose derivative follows from its output")
    if mask_mode and (out_f32 or accumulate or aux_mode):
        raise ValueError("the sign bitmask needs a bf16 output without aux")
    if mask_mode == 2 and act != "none":
        raise ValueError("mask_mode 2 gates acc + bias: no activation")
    if accumulate and (not out_f32 or act != "none" or aux_mode or bias is not None):
        raise ValueError("accumulate mode needs an fp32 output and a plain epilogue")
    if taps > 1 and a_mn:
        raise ValueError("taps needs a K-major A")


def tap_operands(A, B, M, N, K, a_mn=False, b_mn=False, taps=1):
    """[(A_j [M, C], B_j [N, C])] in fp64 for the taps of the product (one pair when taps == 1)."""
    if taps == 1:
        Al = A[:K, :M].t() if a_mn else A[:M, :K]
        Bl = B[:K, :N].t() if b_mn else B[:N, :K]
        return [(Al.double(), Bl.double())]
    C = K // taps
    Cp = (C + 63) // 64 * 64
    out = []
    for j in range(taps):
        Bj = B[j * Cp:j * Cp + C, :N].t() if b_mn else B[:N, j * Cp:j * Cp + C]
        out.append((A[j:j + M, :C].double(), Bj.double()))
    return out


def mask_bits(mask: torch.Tensor, M: int, N: int) -> torch.Tensor:
    """uint8 [M, >= N/8] -> bool [M, N]; bit (c & 7) of byte c >> 3 is column c."""
    sh = torch.arange(8, device=mask.device, dtype=torch.uint8)
    return ((mask[:M, :N // 8].unsqueeze(-1) >> sh) & 1).reshape(M, N).bool()


def mask_bytes(out: torch.Tensor, M: int, N: int) -> torch.Tensor:
    """The mask_mode-1 bytes the kernel must write for the stored output: bit = (out > 0)."""
    bits = (out[:M, :N] > 0).to(torch.int32).reshape(M, N // 8, 8)
    return (bits << torch.arange(8, device=out.device, dtype=torch.int32)).sum(-1).to(torch.uint8)


def colsum_ref(out: torch.Tensor, M: int, N: int, init: torch.Tensor):
    """(fp64 init + column sums of the stored output over rows < M, bound) for the fused colsum.  The kernel sums 32-row
    slices in fp32 and adds them to init with atomics: at most min(M, 32) + ceil(M / 32) + 1 roundings per column."""
    x = out[:M, :N].double()
    ref = init[:N].double() + x.sum(0)
    n_round = min(M, 32) + (M + 31) // 32 + 2
    return ref, n_round * U * (x.abs().sum(0) + init[:N].double().abs())


def gemm_ref(A, B, M, N, K, *, a_mn=False, b_mn=False, bias=None, act="none", aux=None, aux_mode=0, mask=None,
             mask_mode=0, taps=1, accumulate=False, d_init=None, out_f32=False):
    """(fp64 reference [M, N], per-element bound [M, N]) of ibm_gemm_bf16's output; see the module docstring.
    aux: bf16 [>= M, >= N]; mask (mask_mode 2): uint8 [>= M, >= N/8]; d_init (accumulate): D before the call."""
    check_epilogue(act, aux_mode, mask_mode, out_f32, accumulate, bias, taps, a_mn)
    if taps < 1:
        taps = 1
    pre = None
    absab = None
    for Aj, Bj in tap_operands(A, B, M, N, K, a_mn, b_mn, taps):
        p, q = Aj @ Bj.t(), Aj.abs() @ Bj.abs().t()
        pre = p if pre is None else pre + p
        absab = q if absab is None else absab + q
    if bias is not None:
        b = bias[:N].double()
        pre = pre + b
        absab = absab + b.abs()
    acc_err = (K + 1) * U * absab
    if accumulate:
        d0 = d_init[:M, :N].double()
        ref = d0 + pre
        splits = max(1, ((K + 63) // 64) // 8)
        err = acc_err + (splits + 1) * U * d0.abs()
    elif aux_mode == 1:
        y = act_fwd(pre, act)
        xa = aux[:M, :N].double()
        ref = y + xa
        err = ACT_LIP[act] * acc_err + 2 * U * (y.abs() + xa.abs())
    elif aux_mode == 2:
        g = act_grad_from_output(aux[:M, :N].double(), act)
        ref = pre * g
        err = g.abs() * acc_err
    elif mask_mode == 2:
        keep = mask_bits(mask, M, N).double()
        ref = pre * keep
        err = keep * acc_err
    else:
        ref = act_fwd(pre, act)
        err = ACT_LIP[act] * acc_err
    err = err + 1e-6 * ref.abs()
    if not out_f32:
        err = err + 2.0 ** -8 * (ref.abs() + err)
    return ref, err


def max_violation(out: torch.Tensor, ref: torch.Tensor, bound: torch.Tensor) -> str:
    """'' if |out - ref| <= bound everywhere (NaN counts as a violation), else a description of the worst element."""
    diff = (out.double() - ref).abs()
    bad = ~(diff <= bound)
    if not bool(bad.any()):
        return ""
    excess = torch.where(bad, torch.nan_to_num(diff - bound, nan=math.inf), torch.zeros_like(diff))
    i = int(excess.argmax())
    r, c = divmod(i, ref.shape[1])
    return (f"{int(bad.sum())} elements out of bound; worst at [{r}, {c}]: got {float(out[r, c]):.6g}, "
            f"want {float(ref[r, c]):.6g} +- {float(bound[r, c]):.3g}")
