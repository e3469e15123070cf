"""Classifier-free guidance oracle.  TEST INFRASTRUCTURE ONLY.

Builder-owned and **parity unpinned**, like ``ddim_oracle.py`` and ``oracle/ddpm.py``: the reference repository contains no
diffusion code.  It lives beside the tests that use it so that the ``oracle`` package stays as it is.

Spec (Ho & Salimans 2022; DESIGN.md D-1):
  condition dropout  window b of a training step is dropped iff word 0 of Philox4x32-10 draw b at (seed, offset) is below
                     uint32(float64(float32 p) * 2^32) (``philox_oracle.keep_threshold``); p >= 1 drops every window.  A
                     dropped window's kinematics become +0 (the null condition).
  guided prediction  x0_hat = u + s (c - u), c the prediction on the condition, u the one on zero kinematics; the step
                     from t is then the DDPM posterior step or the DDIM step of ``ddim_oracle`` on x0_hat.
"""
from __future__ import annotations

from typing import Callable

import numpy as np
import torch

import ddim_oracle as odim
import philox_oracle as ph
from oracle import ddpm as oddpm


def cond_keep(B: int, p: float, seed: int, offset: int) -> np.ndarray:
    """bool [B]: True where window b keeps its condition."""
    if p >= 1.0:
        return np.zeros(B, dtype=bool)
    return ph.philox_words(B, seed, offset)[:, 0] >= np.uint32(ph.keep_threshold(p))


def guided_x0(c: torch.Tensor, u: torch.Tensor, s: float) -> torch.Tensor:
    c, u = c.double(), u.double()
    return u + s * (c - u)


def guided_ddpm_step(sched, c, u, x_t, t: int, z, s: float) -> torch.Tensor:
    """One DDPM posterior step on the guided prediction, in fp64 from the fp32 tables of ``oracle/ddpm.py``."""
    d = {k: v.double() for k, v in sched.items()}
    return oddpm.posterior_step(d, guided_x0(c, u, s), x_t.double(), t, z.double())


def guided_ddim_step(ab: np.ndarray, c, u, x_t, t: int, p: int, eta: float, z, s: float) -> torch.Tensor:
    return odim.ddim_step(ab, guided_x0(c, u, s), x_t, t, p, eta, z)


def guided_denoiser(denoise: Callable[[torch.Tensor, int, bool], torch.Tensor], s: float):
    """``denoise(x, t, conditional)`` → the guided x0_hat(x, t), for ``oddpm.sample_loop`` / ``odim.ddim_sample_loop``."""
    return lambda x, t: guided_x0(denoise(x, t, True), denoise(x, t, False), s)
