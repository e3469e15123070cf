"""Builder-owned DDIM oracle.  TEST INFRASTRUCTURE ONLY.

**PARITY UNPINNED — NOT FROM THE REFERENCE**, like ``oracle/ddpm.py``, whose schedule it uses: the reference
repository contains no diffusion code.  It lives beside the tests that use it so that the ``oracle`` package, which the
existing golden and parity tests are measured against, stays as it is.

Spec (DDIM, Song et al. 2021; DESIGN.md D-1), restated in fp64 from abar in the eps form — deliberately *not* the
per-timestep linear coefficients the library tabulates (``inferbiomechanics_b200.diffusion.ddim_schedule``):
  ts      = round(linspace(T-1, 0, S))                    (numpy's round; S distinct timesteps, ts[0] = T-1)
  step t → p (p = next entry of ts, -1 after the last, abar[-1] := 1):
    sigma   = eta sqrt((1-a_p)/(1-a_t)) sqrt(1 - a_t/a_p)
    c       = sqrt(max(1 - a_p - sigma^2, 0))
    eps_hat = (x_t - sqrt(a_t) x0_hat) / sqrt(1-a_t)
    x_p     = sqrt(a_p) x0_hat + c eps_hat + [t>0] sigma z
"""
from __future__ import annotations

from typing import Callable

import numpy as np
import torch

from oracle import ddpm as oddpm


def abar(num_timesteps: int = oddpm.NUM_TIMESTEPS) -> np.ndarray:
    return np.cumprod(1.0 - np.linspace(oddpm.BETA_START, oddpm.BETA_END, num_timesteps, dtype=np.float64))


def ddim_timesteps(T: int, S: int) -> np.ndarray:
    return np.round(np.linspace(T - 1, 0, S)).astype(np.int64)


def ddim_step(ab: np.ndarray, x0_hat: torch.Tensor, x_t: torch.Tensor, t: int, p: int, eta: float,
              z: torch.Tensor) -> torch.Tensor:
    """One DDIM step from timestep t to p (p = -1: to x_0), in fp64."""
    a_t = float(ab[t])
    a_p = float(ab[p]) if p >= 0 else 1.0
    sigma = eta * np.sqrt((1.0 - a_p) / (1.0 - a_t)) * np.sqrt(1.0 - a_t / a_p)
    c = np.sqrt(max(1.0 - a_p - sigma * sigma, 0.0))
    x0_hat, x_t = x0_hat.double(), x_t.double()
    eps_hat = (x_t - np.sqrt(a_t) * x0_hat) / np.sqrt(1.0 - a_t)
    x_p = np.sqrt(a_p) * x0_hat + c * eps_hat
    if t > 0:
        x_p = x_p + sigma * z.double()
    return x_p


def ddim_sample_loop(ab: np.ndarray, denoise: Callable[[torch.Tensor, int], torch.Tensor], x_T: torch.Tensor, S: int,
                     eta: float, noise: Callable[[int], torch.Tensor]) -> torch.Tensor:
    """x_T → x_0 over the S-step sequence; ``noise(t)`` supplies z at each timestep walked (parity tests feed the
    CUDA path the same noise).  The state is rounded to fp32 between steps, as the CUDA path stores it."""
    ts = ddim_timesteps(len(ab), S).tolist()
    x = x_T
    for i, t in enumerate(ts):
        p = ts[i + 1] if i + 1 < len(ts) else -1
        x = ddim_step(ab, denoise(x, t), x, t, p, eta, noise(t)).float()
    return x
