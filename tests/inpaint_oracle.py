"""Inpainting oracle.  TEST INFRASTRUCTURE ONLY.

Builder-owned and **parity unpinned**, like ``cfg_oracle.py``, ``ddim_oracle.py`` and ``oracle/ddpm.py``: the reference
repository contains no diffusion code.  It lives beside the tests that use it so that the ``oracle`` package stays as it is.

Spec (MDM's ``p_mean_variance`` for an x0-predicting model; DESIGN.md D-1): given known values y and a bool known-mask of the
state's shape, every reverse step replaces the known entries of the prediction, after the guided combination if any, by y:
  x0_hat = where(mask, y, denoise(x, t))
and then takes the unchanged DDPM or DDIM step.  A select, not a blend: an unknown entry of y (even NaN) never reaches x0_hat.
"""
from __future__ import annotations

from typing import Callable

import torch


def known_denoiser(denoise: Callable[[torch.Tensor, int], torch.Tensor], y: torch.Tensor, mask: torch.Tensor):
    """``denoise(x, t)`` → the inpainted x0_hat(x, t), for ``oddpm.sample_loop`` / ``odim.ddim_sample_loop`` (compose with
    ``cfg_oracle.guided_denoiser`` for a guided one)."""
    return lambda x, t: known_x0(denoise(x, t), y, mask)


def known_x0(x0_hat: torch.Tensor, y: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
    y = y.to(x0_hat.dtype)
    return torch.where(mask.expand_as(x0_hat), y.expand_as(x0_hat), x0_hat)


def mask_words(mask: torch.Tensor) -> torch.Tensor:
    """int32 row words of a bool (..., 30) mask: bit c set iff channel c is known (spelled out per channel)."""
    w = torch.zeros(mask.shape[:-1], dtype=torch.int64)
    for c in range(30):
        w |= mask[..., c].to(torch.int64) << c
    return w.to(torch.int32)
