"""Builder-owned DPM-Solver++(2M) oracle.  TEST INFRASTRUCTURE ONLY.

Builder-owned and **parity unpinned**, like ``ddim_oracle.py`` and ``oracle/ddpm.py``: the reference repository contains no
diffusion code.  It lives beside the tests that use it so that the ``oracle`` package stays as it is.

Spec (Lu et al. 2022, the multistep second-order data-prediction solver; DESIGN.md D-1), restated in fp64 in the paper's
exp / lambda form — deliberately *not* the per-timestep linear coefficients the library tabulates
(``inferbiomechanics_b200.diffusion.dpm_schedule``).  With a = abar, alpha = sqrt(a), sigma = sqrt(1 - a) and
lambda = ln(alpha / sigma):
  timesteps  S = 1: [T-1].  S >= 2: u_i = argmin_t |lambda(t) - target_i| for S targets equally spaced from lambda(T-1) to
             lambda(0) (the smaller t on a tie), u_i = min(u_i, T-1-i), u_{S-1} = 0, then u_i = max(u_i, u_{i+1} + 1) for
             i = S-2 .. 0.
  step i from t = ts[i] to p = ts[i+1] (p = -1 after the last: alpha = 1, sigma = 0), h = lambda_p - lambda_t:
             D   = x0_hat                                          (first and last steps)
             D   = (1 + 1/(2r)) x0_hat - 1/(2r) x0_hat_prev,  r = (lambda_t - lambda_q) / h,  q = ts[i-1]   (interior)
             x_p = (sigma_p / sigma_t) x_t - alpha_p (e^{-h} - 1) D     (x_p = D after the last step)
"""
from __future__ import annotations

from typing import Callable, Optional

import numpy as np
import torch

import ddim_oracle as odim


def lam(ab: np.ndarray, t: int) -> float:
    return 0.5 * float(np.log(ab[t] / (1.0 - ab[t])))


def dpm_timesteps(T: int, S: int, ab: Optional[np.ndarray] = None) -> np.ndarray:
    ab = odim.abar(T) if ab is None else ab
    if S == 1:
        return np.array([T - 1])
    lams = 0.5 * np.log(ab / (1.0 - ab))
    ts = []
    for i in range(S):
        target = lams[T - 1] + (lams[0] - lams[T - 1]) * i / (S - 1)
        ts.append(min(int(np.argmin(np.abs(lams - target))), T - 1 - i))
    ts[-1] = 0
    for i in range(S - 2, -1, -1):
        ts[i] = max(ts[i], ts[i + 1] + 1)
    return np.array(ts)


def step_coefs(ab: np.ndarray, ts, i: int):
    """(c_x0, c_prev, c_xt) of step i in the exp / lambda form: x_p = c_x0 x0_hat + c_prev x0_hat_prev + c_xt x_t."""
    S = len(ts)
    t = int(ts[i])
    sig_t = np.sqrt(1.0 - ab[t])
    if i == S - 1:
        return 1.0, 0.0, 0.0
    p = int(ts[i + 1])
    alpha_p, sig_p = np.sqrt(ab[p]), np.sqrt(1.0 - ab[p])
    h = lam(ab, p) - lam(ab, t)
    lin = -alpha_p * np.expm1(-h)
    if i == 0:
        return lin, 0.0, sig_p / sig_t
    r = (lam(ab, t) - lam(ab, int(ts[i - 1]))) / h
    return lin * (1.0 + 0.5 / r), -lin * 0.5 / r, sig_p / sig_t


def dpm_step(ab: np.ndarray, ts, i: int, x0_hat: torch.Tensor, x0_prev: Optional[torch.Tensor], x_t: torch.Tensor) -> torch.Tensor:
    """Step i of the sequence ``ts`` in fp64 (x0_prev is not used on the first and last steps)."""
    c0, cp, ct = step_coefs(ab, ts, i)
    out = c0 * x0_hat.double() + ct * x_t.double()
    if cp != 0.0:
        out = out + cp * x0_prev.double()
    return out


def dpm_sample_loop(ab: np.ndarray, denoise: Callable[[torch.Tensor, int], torch.Tensor], x_T: torch.Tensor, S: int) -> torch.Tensor:
    """x_T → x_0 over the S-step sequence; the state is rounded to fp32 between steps, as the CUDA path stores it, and so
    is the previous prediction."""
    ts = dpm_timesteps(len(ab), S, ab)
    x, prev = x_T, None
    for i, t in enumerate(ts.tolist()):
        d = denoise(x, t).float()
        x = dpm_step(ab, ts, i, d, prev, x).float()
        prev = d
    return x
