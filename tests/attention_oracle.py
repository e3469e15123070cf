"""fp64 oracle of the attention contract (include/ibm_b200.h: ibm_attention_fwd, ibm_attention_bwd,
ibm_attention_bwd_long).  TEST INFRASTRUCTURE ONLY.

The inputs are the bf16 operands as stored, as 2-D row-major views (one row per (window, frame), head h at columns
[h*hd, (h+1)*hd)).  Every function returns fp64 results in the same 2-D layout together with a per-element bound on the
kernel's error.  Notation per (window, head), with u = 2^-24 (one fp32 rounding) and r = 2^-8 (one bf16 rounding):

  s_ij = sum_k q_ik k_jk     z_ij = scale log2(e) s_ij     p_ij = 2^(z_ij - max_j z_ij) / sum_j 2^(...)     o = p v

Forward.  The kernels form s in fp32 on the tensor cores, exponentiate with ex2.approx against a running row maximum,
round p (or the unnormalised exponentials) to bf16 for the product with v, keep the normaliser in fp32 from the
unrounded values, and round o to bf16.  The relative error of one p_ij is at most

  eps_ij = ln2 * [ scale log2(e) (hd_qk + 2) u sum_k |q_ik k_jk|        fp32 score accumulation (worst case)
                  + 4 u (|z_ij| + max_j |z_ij|) ]                        scale*log2(e) rounded, the fma against the
                                                                         maximum, the maximum times the scale and
                                                                         the difference of two running maxima
           + (2 + ceil(T / 32)) 2^-21                                    ex2.approx / lg2.approx (documented 2^-22
                                                                         relative / 2^-22.6 absolute, twice that here),
                                                                         once for p, once for a log-sum-exp, once per
                                                                         32-key chunk for the online rescale
           + (T + 4) u                                                   the fp32 normaliser, its reciprocal, the scale

A perturbation p_ij (1 + e_ij) moves o_ic by sum_j p_ij e_ij (v_jc - o_ic); rounding p to bf16 before p v moves it by at
most r sum_j p_ij |v_jc|; the fp32 accumulation of p v adds (T + 2) u sum_j p_ij |v_jc|.  So

  err_o = sum_j p_ij |v_jc - o_ic| eps_ij + (r + (T + 2) u) sum_j p_ij |v_jc|
  |o - ref| <= r |ref| + (1 + r) err_o                                   (the bf16 store of the computed value)

Backward.  dP = dO v^T, D_i = sum_c dO_ic O_ic, dS = p o (dP - D), dV = p^T dO, dQ = scale dS k, dK = scale dS^T q.
ibm_attention_bwd recomputes O on chip, so its D is that of the exact output (D_i = sum_j p_ij dP_ij);
ibm_attention_bwd_long is given the forward output o and forms D from it.  The kernels round p and scale*dS to bf16
before the second products, and accumulate everything in fp32:

  d_dP_ij = (max(hd_v, 16) + 2) u sum_c |dO_ic v_jc|                    fp32 accumulation (hd_v = 8 is padded to 16)
  d_D_i   = sum_j p_ij (|dP_ij| eps_ij + d_dP_ij) + (T + 2) u sum_j p_ij |dP_ij|      (D from the exact output)
          = (hd_v + 2) u sum_c |dO_ic o_ic|                                           (D from the stored o)
  e_ij    = scale p_ij [ eps_ij |dP_ij - D_i| + d_dP_ij + d_D_i + 3 u (|dP_ij| + |D_i|) ]
  E_ij    = r scale |dS_ij| + (1 + r) e_ij                               error of the bf16 scale*dS operand
  err_dV  = sum_i p_ij (r + (1 + r) eps_ij) |dO_ic| + (T + 2) u sum_i p_ij |dO_ic|
  err_dQ  = sum_j E_ij |k_jk| + (T + 2) u sum_j (scale |dS_ij| + E_ij) |k_jk|
  err_dK  = sum_i E_ij |q_ik| + (T + 2) u sum_i (scale |dS_ij| + E_ij) |q_ik|
  bound   = r |ref| + (1 + r) err

Bias sums.  The kernels add the column sums of dq / dk / dv over all rows to an fp32 vector with atomics (ibm_attention_bwd
on the tensor cores sums the bf16-rounded values, the others the fp32 ones; the bound above covers both).  Their bound is
the column sum of the element bounds plus (rows + 1) u (sum_rows |x| + |init|) for the fp32 additions in any order.  The
key-bias gradient is zero in exact arithmetic (every row of dS sums to zero), so its bound rests on exactly that
absolute sum of its summands.

Every term is a worst case, so a row, key, head or window indexing error (which moves an output by the size of a value,
not by a rounding of it) shows up far above the bound; tests/test_attention_oracle_cpu.py plants such faults and checks
that the bound flags each one.
"""
from __future__ import annotations

import math

import torch

U = 2.0 ** -24
R = 2.0 ** -8
LOG2E = 1.4426950408889634
LN2 = math.log(2.0)
TRANSC = 2.0 ** -21


def f32(x: float) -> float:
    """The fp32 value the library receives for a Python float."""
    return float(torch.tensor(x, dtype=torch.float32))


def heads(X: torch.Tensor, n_win: int, T: int, H: int, hd: int) -> torch.Tensor:
    """Rows [0, n_win*T), columns [0, H*hd) of a 2-D view -> fp64 [n_win, H, T, hd]."""
    return X[:n_win * T, :H * hd].double().reshape(n_win, T, H, hd).permute(0, 2, 1, 3)


def flat(X: torch.Tensor) -> torch.Tensor:
    """[n_win, H, T, hd] -> [n_win*T, H*hd]."""
    n_win, H, T, hd = X.shape
    return X.permute(0, 2, 1, 3).reshape(n_win * T, H * hd)


def _softmax_parts(q, k, scale):
    """(p, eps) of the module docstring, [n_win, H, T, T]."""
    T, hd = q.shape[-2], q.shape[-1]
    sl = scale * LOG2E
    z = (q @ k.transpose(-1, -2)) * sl
    a = q.abs() @ k.abs().transpose(-1, -2)
    p = torch.softmax(z * LN2, dim=-1)
    zmax = z.abs().amax(dim=-1, keepdim=True)
    eps = (LN2 * (sl * (hd + 2) * U * a + 4 * U * (z.abs() + zmax))
           + (2 + math.ceil(T / 32)) * TRANSC + (T + 4) * U)
    return p, eps


def attention_fwd_ref(q, k, v, n_win, T, H, hd_qk, hd_v, scale):
    """(o [n_win*T, H*hd_v], bound, p [n_win, H, T, T]) for ibm_attention_fwd."""
    Q, K, V = heads(q, n_win, T, H, hd_qk), heads(k, n_win, T, H, hd_qk), heads(v, n_win, T, H, hd_v)
    p, eps = _softmax_parts(Q, K, scale)
    o = p @ V
    # sum_j p_ij eps_ij |v_jc - o_ic|, one value column at a time (no [n_win, H, T, T, hd_v] temporary)
    pe = p * eps
    dev = torch.empty_like(o)
    for c in range(V.shape[-1]):
        dev[..., c] = (pe * (V[..., c].unsqueeze(-2) - o[..., c].unsqueeze(-1)).abs()).sum(-1)
    err = dev + (R + (T + 2) * U) * (p @ V.abs())
    bound = R * o.abs() + (1 + R) * err
    return flat(o), flat(bound), p


def attention_bwd_ref(q, k, v, d_o, n_win, T, H, hd_qk, hd_v, scale, o=None):
    """dict(dq, dk, dv, and their bounds 'b_dq', 'b_dk', 'b_dv'), 2-D, for the backward.  o None: D from the exact
    output (ibm_attention_bwd); otherwise D from the given bf16 forward output (ibm_attention_bwd_long)."""
    Q, K, V = heads(q, n_win, T, H, hd_qk), heads(k, n_win, T, H, hd_qk), heads(v, n_win, T, H, hd_v)
    G = heads(d_o, n_win, T, H, hd_v)
    p, eps = _softmax_parts(Q, K, scale)
    dP = G @ V.transpose(-1, -2)
    d_dP = (max(hd_v, 16) + 2) * U * (G.abs() @ V.abs().transpose(-1, -2))
    if o is None:
        D = (p * dP).sum(-1, keepdim=True)
        d_D = (p * (dP.abs() * eps + d_dP)).sum(-1, keepdim=True) + (T + 2) * U * (p * dP.abs()).sum(-1, keepdim=True)
    else:
        Og = heads(o, n_win, T, H, hd_v)
        D = (G * Og).sum(-1, keepdim=True)
        d_D = (hd_v + 2) * U * (G * Og).abs().sum(-1, keepdim=True)
    dS = p * (dP - D)
    e = scale * p * (eps * (dP - D).abs() + d_dP + d_D + 3 * U * (dP.abs() + D.abs()))
    E = R * scale * dS.abs() + (1 + R) * e
    sdS = scale * dS.abs() + E
    out = {}
    dv = p.transpose(-1, -2) @ G
    err = (p * (R + (1 + R) * eps)).transpose(-1, -2) @ G.abs() + (T + 2) * U * (p.transpose(-1, -2) @ G.abs())
    out["dv"], out["b_dv"] = flat(dv), flat(R * dv.abs() + (1 + R) * err)
    dq = scale * (dS @ K)
    err = E @ K.abs() + (T + 2) * U * (sdS @ K.abs())
    out["dq"], out["b_dq"] = flat(dq), flat(R * dq.abs() + (1 + R) * err)
    dk = scale * (dS.transpose(-1, -2) @ Q)
    err = E.transpose(-1, -2) @ Q.abs() + (T + 2) * U * (sdS.transpose(-1, -2) @ Q.abs())
    out["dk"], out["b_dk"] = flat(dk), flat(R * dk.abs() + (1 + R) * err)
    return out


def bias_ref(ref: torch.Tensor, bound: torch.Tensor, init: torch.Tensor):
    """(init + column sums of ref, bound) for a fused bias gradient; ref and bound [rows, n] fp64, init [n]."""
    rows = ref.shape[0]
    i = init.double()
    return i + ref.sum(0), bound.sum(0) + (rows + 1) * U * (ref.abs().sum(0) + bound.sum(0) + i.abs())


def max_violation(out: torch.Tensor, ref: torch.Tensor, bound: torch.Tensor) -> str:
    """'' if |out - ref| <= bound everywhere (NaN is a violation), else the worst element and the count."""
    out, ref, bound = out.reshape(ref.shape[0], -1), ref.reshape(ref.shape[0], -1), bound.reshape(ref.shape[0], -1)
    diff = (out.double() - ref).abs()
    bad = ~(diff <= bound)
    if not bool(bad.any()):
        return ""
    excess = torch.where(bad, torch.nan_to_num(diff / bound, nan=math.inf, posinf=math.inf), torch.zeros_like(diff))
    i = int(excess.argmax())
    r, c = divmod(i, ref.shape[1])
    return (f"{int(bad.sum())} elements out of bound; worst at [{r}, {c}]: got {float(out[r, c]):.6g}, "
            f"want {float(ref[r, c]):.6g} +- {float(bound[r, c]):.3g}")


def err_ratio(out: torch.Tensor, ref: torch.Tensor, bound: torch.Tensor) -> float:
    """max |out - ref| / bound: how close a kernel comes to its bound."""
    return float(((out.reshape(ref.shape).double() - ref).abs() / bound.clamp_min(1e-300)).max())
