"""Philox4x32-10 oracle for the dropout masks and the diffusion noise.  TEST INFRASTRUCTURE ONLY.

A vectorised numpy restatement of ``philox4x32_10`` / ``philox_normal4`` (csrc/common.cuh) and of the keep rule of
``dropout_kernel`` (csrc/elementwise.cu).  It lives beside the tests that use it, so the ``oracle`` package stays as it is.

Spec:
  counter  (i_lo, i_hi, off_lo, off_hi)   i = draw index, off = the 64-bit counter offset
  key      (seed_lo, seed_hi)
  round    c = (hi(M1 c2) ^ c1 ^ k0, lo(M1 c2), hi(M0 c0) ^ c3 ^ k1, lo(M0 c0));  k += (W0, W1);  10 rounds
  dropout  word k of draw i decides element 4i + k: kept iff word >= uint32(float64(float32 p) * 2^32); a kept value
           becomes bf16_rne(float32(x) * float32(1 / (1 - p))), the scale computed in fp32; a dropped one becomes +0
  normal4  u_k = (float32(r_k) + 0.5f) * 2^-32 in fp32;  Box-Muller on (u0, u1) and (u2, u3):
           (r0 cos 2pi u1, r0 sin 2pi u1, r1 cos 2pi u3, r1 sin 2pi u3),  r0 = sqrt(-2 ln u0), r1 = sqrt(-2 ln u2)
"""
from __future__ import annotations

import numpy as np
import torch

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK32 = 0xFFFFFFFF


def philox4x32_10(ctr, key):
    """ctr: four uint32 arrays (or ints), broadcast together; key: two ints.  Returns four uint32 arrays."""
    c = [np.asarray(v, dtype=np.uint64) & np.uint64(MASK32) for v in ctr]
    c = np.broadcast_arrays(*c)
    c = [v.copy() for v in c]
    k0, k1 = int(key[0]) & MASK32, int(key[1]) & MASK32
    m0, m1, lo = np.uint64(M0), np.uint64(M1), np.uint64(MASK32)
    s32 = np.uint64(32)
    for _ in range(10):
        p0, p1 = m0 * c[0], m1 * c[2]                # 32 x 32 -> 64-bit products, exact in uint64
        c = [(p1 >> s32) ^ c[1] ^ np.uint64(k0), p1 & lo, (p0 >> s32) ^ c[3] ^ np.uint64(k1), p0 & lo]
        k0, k1 = (k0 + W0) & MASK32, (k1 + W1) & MASK32
    return [v.astype(np.uint32) for v in c]


def philox_words(n_draws: int, seed: int, offset: int) -> np.ndarray:
    """(n_draws, 4) uint32: the four words of draws 0 .. n_draws-1 at counter offset ``offset``."""
    i = np.arange(n_draws, dtype=np.uint64)
    r = philox4x32_10((i & np.uint64(MASK32), i >> np.uint64(32), offset & MASK32, (offset >> 32) & MASK32),
                      (seed & MASK32, (seed >> 32) & MASK32))
    return np.stack(r, axis=1)


def keep_threshold(p: float) -> int:
    return int(float(np.float32(p)) * 4294967296.0)      # the kernel's (uint32_t)(p * 4294967296.0), p a float


def dropout_bf16(x: torch.Tensor, p: float, seed: int, offset: int) -> torch.Tensor:
    """Inverted dropout of a flat bf16 tensor (numel % 4 == 0), bit for bit as ``ibm_dropout_bf16`` computes it."""
    n = x.numel()
    assert n % 4 == 0
    keep = philox_words(n // 4, seed, offset).reshape(-1) >= np.uint32(keep_threshold(p))
    scale = np.float32(1.0) / (np.float32(1.0) - np.float32(p))
    xf = x.detach().cpu().reshape(-1).float().numpy()
    y = np.where(keep, xf * scale, np.float32(0.0)).astype(np.float32)
    return torch.from_numpy(y).to(torch.bfloat16)


def uniforms(n_draws: int, seed: int, offset: int) -> np.ndarray:
    """(n_draws, 4) fp32 uniforms in (0, 1] as ``philox_normal4`` forms them."""
    r = philox_words(n_draws, seed, offset)
    return (r.astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -32)


def normals(n: int, seed: int, offset: int) -> np.ndarray:
    """The first n normals of the flat stream (element e = lane e & 3 of draw e >> 2), in fp64 from the fp32 uniforms."""
    nd = (n + 3) // 4
    u = uniforms(nd, seed, offset).astype(np.float64)
    rad = np.sqrt(-2.0 * np.log(u[:, [0, 2]]))
    ang = 2.0 * np.pi * u[:, [1, 3]]
    return np.stack([rad[:, 0] * np.cos(ang[:, 0]), rad[:, 0] * np.sin(ang[:, 0]),
                     rad[:, 1] * np.cos(ang[:, 1]), rad[:, 1] * np.sin(ang[:, 1])], axis=1).reshape(-1)[:n]
