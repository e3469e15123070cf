"""Launch plans ("engines") for the model families: explicit forward/backward sequences of
libibm_b200 kernels over preallocated HBM buffers.  No autograd, no torch math: torch tensors are
only the memory the kernels read and write.

* ``FeedForwardEngine``  — /root/reference/src/models/FeedForwardRegressionBaseline.py:65-77,113
* ``EncoderLayerPlan``   — /root/reference/src/models/TransformerBaseline.py:8-38 (post-LN layer),
                            shared by the denoiser (d=512) and the TransformerBaseline (d=108 padded)
* ``DenoiserEngine``     — builder-owned DDPM denoiser (DESIGN.md D-1), forward + backward

The three model engines (and ``GroundlinkEngine``, engine_groundlink.py) share the step interface the Trainer and the
drop-in modules drive:

* ``input_layout(B, F, train)`` → ``(bf16 buffer, frame_stride, win_extra, col0)``: where the packers write frame t of
  window b (element ``(b*F + t)*frame_stride + b*win_extra + col0``);
* ``forward(B, F, train)`` → the fp32 output, ``dout(B, F)`` → the bf16 output-gradient buffer, ``backward(B, F)``;
* ``quantity_views(x, B, F, Fo)`` → the four (B, Fo, ·) loss-quantity views (cop, force, torque, wrench) of either;
* ``bucket_boundaries()`` → arena offsets of the gradient groups; backward calls ``bucket_hook(g)`` once group g and all
  later ones are complete;
* ``set_rng(seed_mix, rank, step, step_dev)`` seeds the dropout masks; ``refresh_weights()`` re-derives cached weight
  copies when ``ParamArena.version`` moved.
"""
from __future__ import annotations

import math
import os
from typing import Dict, List, Optional, Tuple

import torch

from . import ops
from .params import ParamArena

BF16 = torch.bfloat16
F32 = torch.float32


def _r8(x: int) -> int:
    return ops.round_up(x, 8)


def quantity_split(rows: torch.Tensor) -> List[torch.Tensor]:
    """(…, >=30) rows30 tensor → the four loss quantities (cop, force, torque, wrench) as views."""
    return [rows[..., 0:6], rows[..., 6:12], rows[..., 12:18], rows[..., 18:30]]


class _Buffers:
    """Per-batch-size cache of activation buffers (allocated once, reused every step)."""

    def __init__(self, device):
        self.device = device
        self._cache: Dict[Tuple, Dict[str, torch.Tensor]] = {}

    def get(self, key: Tuple) -> Dict[str, torch.Tensor]:
        if key not in self._cache:
            if len(self._cache) >= 16:          # bounded: ragged last batches come and go
                self._cache.pop(next(iter(self._cache)))
            self._cache[key] = {}
        return self._cache[key]

    def tensor(self, store: Dict[str, torch.Tensor], name: str, shape, dtype, zero=False) -> torch.Tensor:
        t = store.get(name)
        if t is None:
            t = (torch.zeros if zero else torch.empty)(shape, dtype=dtype, device=self.device)
            store[name] = t
        return t


# =============================================================================================
# FeedForward MLP
# =============================================================================================
class FeedForwardEngine:
    """dims = [K0, h1, …, N_out]; every layer y = act(x W^T + b) except the last (no act, fp32 out).

    Optional per-layer ``[Dropout][BatchNorm1d]`` on the layer INPUT (FeedForward…py:68-72): ``bn`` is a list with one
    entry per Linear (``None`` or ``(weight name, bias name, nn.BatchNorm1d module)`` — the module only holds the
    running-statistics buffers and eps/momentum), ``dropout_p`` the probability of the Philox inverted dropout.
    ``frame_width``: input columns per frame (a window is one row of F frames)."""

    DROPOUT_SEED = 0x66666e6e

    def __init__(self, arena: ParamArena, layers: List[Tuple[str, str, int, int]], activation: str, frame_width: int, bn=None,
                 dropout_p: float = 0.0):
        self.arena = arena
        self.frame_width = frame_width
        self.layers = layers                    # (weight name, bias name, N, K)
        self.act = activation
        self.buf = _Buffers(arena.device)
        self.bucket_hook = None                 # callable(layer_index) fired when a layer's grads are complete
        self.out_cols = layers[-1][2]
        self.in_cols = layers[0][3]
        self.in_ld = _r8(self.in_cols)
        self.bn = bn if bn is not None and any(b is not None for b in bn) else None
        self.dropout_p = float(dropout_p)
        self.set_rng(0, 0, 0, None)
        if self.bn is not None:
            maxc = max(K for (_, _, _, K) in layers)
            self.bn_ws = ops.batchnorm_workspace(maxc, arena.device)
            self.bn_stats = {i: (torch.zeros(K, device=arena.device), torch.ones(K, device=arena.device))
                             for i, (_, _, _, K) in enumerate(layers) if self.bn[i] is not None}

    def set_rng(self, seed_mix: int, rank: int, step: int, step_dev: Optional[torch.Tensor]) -> None:
        """Dropout masks: Philox keyed by (DROPOUT_SEED ^ seed_mix) + rank, offset by the training-forward count ``step`` —
        or, when ``step_dev`` (a device-resident step counter) is given, by its value, so that a captured step replays."""
        self.dropout_seed = (self.DROPOUT_SEED ^ seed_mix) + rank
        self.step, self.step_dev = step, step_dev

    def refresh_weights(self) -> None:
        """No derived weight copies beyond the arena's own (the GEMMs read the bf16 shadow)."""

    def bucket_boundaries(self) -> List[int]:
        """Arena offsets of the gradient groups: group i = Linear layer i (a layer's BatchNorm parameters precede it)."""
        offs = self.arena.offsets
        return [offs[self.bn[i][0] if self.bn is not None and self.bn[i] is not None else w][0]
                for i, (w, _, _, _) in enumerate(self.layers)]

    def input_buffer(self, B: int) -> torch.Tensor:
        s = self.buf.get((B,))
        return self.buf.tensor(s, "x0", (B, self.in_ld), BF16, zero=True)

    def input_layout(self, B: int, F: int, train: bool) -> Tuple[torch.Tensor, int, int, int]:
        """(buffer, frame_stride, win_extra, col0) for the packers: one row per window, frame-major (FeedForward…py:108)."""
        return self.input_buffer(B), self.frame_width, self.in_ld - self.in_cols, 0

    def dout(self, B: int, F: int) -> torch.Tensor:
        s = self.buf.get((B,))
        return self.buf.tensor(s, "dout", (B, _r8(self.out_cols)), BF16, zero=True)

    def quantity_views(self, x: torch.Tensor, B: int, F: int, Fo: int) -> List[torch.Tensor]:
        """(B, Fo, ·) views of the four quantities in an output / output-gradient row: quantity-then-frame blocks
        (FeedForward…py:116-121)."""
        def blk(a, b, c):
            return x[:, a * Fo:b * Fo].unflatten(1, (Fo, c))
        return [blk(0, 6, 6), blk(6, 12, 6), blk(12, 18, 6), blk(18, 30, 12)]

    def forward(self, B: int, F: int, train: bool) -> torch.Tensor:
        """Consumes input_buffer(B); returns fp32 [B, ld>=N_out] (first N_out columns valid).  ``train`` selects batch
        statistics (and updates the running ones) for BatchNorm and switches dropout on, like nn.Module.training.
        ``F`` is implied by the layer widths."""
        s = self.buf.get((B,))
        x = self.input_buffer(B)
        n_layers = len(self.layers)
        drop = train and self.dropout_p > 0.0
        if train:
            self.step += 1
        s["mode"] = (train, drop)
        for i, (wn, bn, N, K) in enumerate(self.layers):
            W = self.arena.weight_operand(wn, N, K)
            bias = self.arena.master_of(bn)
            last = i == n_layers - 1
            if drop:                                                    # nn.Dropout(p) on the layer input
                xd = self.buf.tensor(s, f"xd{i}", tuple(x.shape), BF16)
                if self.step_dev is not None:
                    ops.dropout(x, xd, self.dropout_p, self.dropout_seed, i, self.step_dev, n_layers)
                else:
                    ops.dropout(x, xd, self.dropout_p, self.dropout_seed, n_layers * self.step + i)
                x = xd
            if self.bn is not None and self.bn[i] is not None:          # nn.BatchNorm1d(h0) on the (dropped) input
                gname, bname, mod = self.bn[i]
                xb = self.buf.tensor(s, f"xb{i}", tuple(x.shape), BF16, zero=True)
                mean, rstd = self.bn_stats[i]
                mom = 0.1 if mod.momentum is None else float(mod.momentum)
                ops.batchnorm_fwd(x, xb, B, K, self.arena.master_of(gname), self.arena.master_of(bname), mod.running_mean,
                                  mod.running_var, mean, rstd, train, mom, float(mod.eps), self.bn_ws)
                if train:
                    mod.num_batches_tracked += 1
                s[f"prebn{i}"] = x
                x = xb
            s[f"in{i}"] = x                                             # what the GEMM consumed (weight-gradient operand)
            if last:
                y = self.buf.tensor(s, "out", (B, ops.round_up(N, 4)), F32)
                ops.gemm(x, W, y, B, N, K, bias=bias)
            else:
                y = self.buf.tensor(s, f"a{i}", (B, _r8(N)), BF16, zero=True)
                ops.gemm(x, W, y, B, N, K, bias=bias, act=self.act)
            x = y
        return x

    def backward(self, B: int, F: int) -> None:
        """Consumes dout(B, F) (bf16 d loss/d out); accumulates weight/bias grads into the arena."""
        arena = self.arena
        s = self.buf.get((B,))
        train, drop = s.get("mode", (False, False))
        dy = self.dout(B, F)
        n_layers = len(self.layers)
        bias_done = False                       # layer i's bias gradient already produced by BatchNorm i+1's backward
        for i in range(n_layers - 1, -1, -1):
            wn, bn, N, K = self.layers[i]
            x = s[f"in{i}"]
            has_bn = self.bn is not None and self.bn[i] is not None
            _wgrad(arena, wn, N, K, dy, x, B, self.buf, s)
            if not bias_done:
                ops.colsum(dy, B, N, arena.grad_of(bn))
            bias_done = False
            if i > 0 or has_bn:
                W = self.arena.weight_operand(wn, N, K)
                dx = self.buf.tensor(s, f"da{i - 1}" if i > 0 else "dx0", (B, _r8(K)), BF16, zero=True)
                prev = s[f"a{i - 1}"] if i > 0 else None             # activation OUTPUT of layer i-1 (its derivative gate)
                if not has_bn:
                    # dX = (dY · W) ∘ act'(x): W [N,K] row-major is the MN-major B operand [K_red=N, N_out=K]
                    ops.gemm(dy, W, dx, B, K, N, b_mn=True, act=self.act, aux=prev, aux_mode=2)
                else:
                    gname, bname, mod = self.bn[i]
                    ops.gemm(dy, W, dx, B, K, N, b_mn=True)
                    mean, rstd = self.bn_stats[i] if train else (mod.running_mean, mod.running_var)
                    ops.batchnorm_bwd(dx, s[f"prebn{i}"], dx if i > 0 else None, B, K, self.arena.master_of(gname), mean, rstd,
                                      train, float(mod.eps), arena.grad_of(gname), arena.grad_of(bname), self.bn_ws,
                                      act_out=prev, act=self.act if prev is not None else None,
                                      dx_colsum=arena.grad_of(self.layers[i - 1][1]) if i > 0 and not drop else None)
                    bias_done = i > 0 and not drop   # fp32 column sums of dx = bias gradient of layer i-1 (no mask in between)
                if drop and i > 0:                                      # same Philox (seed, offset) as the forward mask
                    if self.step_dev is not None:
                        ops.dropout(dx, dx, self.dropout_p, self.dropout_seed, i, self.step_dev, n_layers)
                    else:
                        ops.dropout(dx, dx, self.dropout_p, self.dropout_seed, n_layers * self.step + i)
                dy = dx
            if self.bucket_hook is not None:
                self.bucket_hook(i)               # layer i's gradients are complete


def _wgrad(arena: ParamArena, wname: str, N: int, K: int, dy: torch.Tensor, x: torch.Tensor, M: int, buf: _Buffers,
           store: Dict[str, torch.Tensor]) -> None:
    """dW[N,K] += dY[M,N]^T · X[M,K] (both operands MN-major, split-K TMA reduce-add into fp32).
    fp32 TMA rows must be 16-byte multiples: odd K goes through a padded scratch."""
    g = arena.grad_of(wname, (N, K))
    if K % 4 == 0:
        ops.gemm(dy, x, g, N, K, M, a_mn=True, b_mn=True, accumulate=True)
    else:
        tmp = buf.tensor(store, f"wg_{wname}", (N, ops.round_up(K, 4)), F32)
        tmp.zero_()
        ops.gemm(dy, x, tmp, N, K, M, a_mn=True, b_mn=True, accumulate=True)
        g.add_(tmp[:, :K])                                      # strided copy-add (plumbing)


# =============================================================================================
# Post-LN transformer encoder layer (reference TransformerLayer)
# =============================================================================================
class EncoderLayerPlan:
    """One ``TransformerLayer`` (TransformerBaseline.py:8-38): x1 = LN1(x + MHA(x)); x2 = LN2(x1 + FFN(x1)).

    Residual adds are fused into the out-proj / FFN-2 GEMM epilogues (aux_mode 1); ReLU into FFN-1's
    epilogue and its derivative into FFN-2's dgrad epilogue (aux_mode 2); bias gradients of out-proj and
    FFN-2 into the LayerNorm backward kernel.
    """

    def __init__(self, arena: ParamArena, prefix: str, d: int, heads: int, ff: int):
        self.arena, self.p, self.d, self.H, self.ff = arena, prefix, d, heads, ff
        self.hd = d // heads
        assert d % 8 == 0 and self.hd in (32, 48, 64), "engine supports head_dim 32/48/64 and d % 8 == 0"

    def n(self, s: str) -> str:
        return self.p + s

    def alloc(self, buf: _Buffers, st: Dict[str, torch.Tensor], tag: str, M: int, train: bool):
        d, ff = self.d, self.ff
        names = [("qkv", 3 * d), ("o", d), ("s1", d), ("x1", d), ("h", ff), ("s2", d), ("x2", d)]
        out = {k: buf.tensor(st, f"{tag}.{k}", (M, w), BF16) for k, w in names}
        # sign bits of h (1 bit per element): all the FFN-2 dgrad needs of the saved activation
        use_mask = train and ff % 64 == 0 and os.environ.get("IBM_NO_HMASK", "0") != "1"     # env switch: A/B measurements
        out["hmask"] = buf.tensor(st, f"{tag}.hmask", (M, ff // 8), torch.uint8) if use_mask else None
        for k in ("mean1", "rstd1", "mean2", "rstd2"):
            out[k] = buf.tensor(st, f"{tag}.{k}", (M,), F32)
        return out

    def forward(self, x: torch.Tensor, a: Dict[str, torch.Tensor], M: int, n_win: int, T: int) -> torch.Tensor:
        A, d, ff, n = self.arena, self.d, self.ff, self.n
        ops.gemm(x, A.shadow_of(n("multihead_attention.in_proj_weight"), (3 * d, d)), a["qkv"], M, 3 * d, d,
                 bias=A.master_of(n("multihead_attention.in_proj_bias")))
        ops.attention_fwd_fused(a["qkv"], d, a["o"], n_win, T, self.H, self.hd, 1.0 / math.sqrt(self.hd))
        ops.gemm(a["o"], A.shadow_of(n("multihead_attention.out_proj.weight"), (d, d)), a["s1"], M, d, d,
                 bias=A.master_of(n("multihead_attention.out_proj.bias")), aux=x, aux_mode=1)
        ops.layernorm_fwd(a["s1"], a["x1"], A.master_of(n("norm1.weight")), A.master_of(n("norm1.bias")), M, d,
                          mean=a["mean1"], rstd=a["rstd1"])
        ops.gemm(a["x1"], A.shadow_of(n("feedforward.0.weight"), (ff, d)), a["h"], M, ff, d,
                 bias=A.master_of(n("feedforward.0.bias")), act="relu", mask=a.get("hmask"), mask_mode=1)
        ops.gemm(a["h"], A.shadow_of(n("feedforward.2.weight"), (d, ff)), a["s2"], M, d, ff,
                 bias=A.master_of(n("feedforward.2.bias")), aux=a["x1"], aux_mode=1)
        ops.layernorm_fwd(a["s2"], a["x2"], A.master_of(n("norm2.weight")), A.master_of(n("norm2.bias")), M, d,
                          mean=a["mean2"], rstd=a["rstd2"])
        return a["x2"]

    def backward(self, x: torch.Tensor, a: Dict[str, torch.Tensor], dx2: torch.Tensor, sc: Dict[str, torch.Tensor],
                 M: int, n_win: int, T: int, dx_out: torch.Tensor) -> None:
        """dx2 = d loss/d x2 (bf16 [M,d]); writes d loss/d x into dx_out; accumulates parameter grads."""
        A, d, ff, n = self.arena, self.d, self.ff, self.n
        g = A.grad_of
        ds, dh, dx1, do, dqkv = sc["ds"], sc["dh"], sc["dx1"], sc["do"], sc["dqkv"]
        # LN2 backward (+ bias grad of FFN-2 as colsum(ds2))
        ops.layernorm_bwd(dx2, a["s2"], A.master_of(n("norm2.weight")), a["mean2"], a["rstd2"], M, d, ds,
                          g(n("norm2.weight")), g(n("norm2.bias")), g(n("feedforward.2.bias")))
        # FFN-2: dW2 += ds^T h ; dh = (ds · W2) ∘ relu'(h)
        ops.gemm(ds, a["h"], g(n("feedforward.2.weight"), (d, ff)), d, ff, M, a_mn=True, b_mn=True, accumulate=True)
        #        db1 = colsum(dh) accumulated by the same epilogue
        if a.get("hmask") is not None:
            ops.gemm(ds, A.shadow_of(n("feedforward.2.weight"), (d, ff)), dh, M, ff, d, b_mn=True, mask=a["hmask"], mask_mode=2,
                     colsum=g(n("feedforward.0.bias")))
        else:
            ops.gemm(ds, A.shadow_of(n("feedforward.2.weight"), (d, ff)), dh, M, ff, d, b_mn=True, act="relu", aux=a["h"],
                     aux_mode=2, colsum=g(n("feedforward.0.bias")))
        # FFN-1: dW1 += dh^T x1 ; dx1 = dh · W1 + ds (residual)
        ops.gemm(dh, a["x1"], g(n("feedforward.0.weight"), (ff, d)), ff, d, M, a_mn=True, b_mn=True, accumulate=True)
        ops.gemm(dh, A.shadow_of(n("feedforward.0.weight"), (ff, d)), dx1, M, d, ff, b_mn=True, aux=ds, aux_mode=1)
        # LN1 backward (+ bias grad of out-proj)
        ops.layernorm_bwd(dx1, a["s1"], A.master_of(n("norm1.weight")), a["mean1"], a["rstd1"], M, d, ds,
                          g(n("norm1.weight")), g(n("norm1.bias")), g(n("multihead_attention.out_proj.bias")))
        # out-proj: dWo += ds^T o ; do = ds · Wo
        ops.gemm(ds, a["o"], g(n("multihead_attention.out_proj.weight"), (d, d)), d, d, M, a_mn=True, b_mn=True,
                 accumulate=True)
        ops.gemm(ds, A.shadow_of(n("multihead_attention.out_proj.weight"), (d, d)), do, M, d, d, b_mn=True)
        # attention backward → dqkv, with dbqkv = colsum(dqkv) accumulated by the same kernel
        if T <= 64:
            ops.attention_bwd(a["qkv"], d, do, dqkv, n_win, T, self.H, self.hd, 1.0 / math.sqrt(self.hd),
                              dbias=g(n("multihead_attention.in_proj_bias")))
        else:                                     # whole windows of up to 256 frames (the TransformerBaseline's T = 200)
            qkv, db = a["qkv"], g(n("multihead_attention.in_proj_bias"))
            ops.attention_bwd_long(qkv[:, :d], qkv[:, d:2 * d], qkv[:, 2 * d:], a["o"], do, dqkv[:, :d], dqkv[:, d:2 * d],
                                   dqkv[:, 2 * d:], n_win, T, self.H, self.hd, self.hd, 1.0 / math.sqrt(self.hd),
                                   dbq=db[:d], dbk=db[d:2 * d], dbv=db[2 * d:])
        # in-proj: dWqkv += dqkv^T x ; dx = dqkv · Wqkv + ds (residual)
        ops.gemm(dqkv, x, g(n("multihead_attention.in_proj_weight"), (3 * d, d)), 3 * d, d, M, a_mn=True, b_mn=True,
                 accumulate=True)
        ops.gemm(dqkv, A.shadow_of(n("multihead_attention.in_proj_weight"), (3 * d, d)), dx_out, M, d, 3 * d, b_mn=True,
                 aux=ds, aux_mode=1)


# =============================================================================================
# Diffusion denoiser (builder-owned spec, DESIGN.md D-1)
# =============================================================================================
class DenoiserEngine:
    """x0_hat = out_proj(Layers(in_proj([x_t | cond]) + time_mlp(sin_emb(t)) + pos_embedding)).

    ``xc`` is the concat buffer [M, ld_in] bf16: columns 0..29 = x_t rows (written by q_sample /
    posterior_step), 30..30+C_in = packed kinematics (written by the window packer).
    """

    def __init__(self, arena: ParamArena, c_in: int, frames: int, d: int, heads: int, ff: int, num_layers: int):
        self.arena, self.c_in, self.F, self.d, self.H, self.ff, self.L = arena, c_in, frames, d, heads, ff, num_layers
        self.k_in = 30 + c_in
        self.ld_in = _r8(self.k_in)
        self.layers = [EncoderLayerPlan(arena, f"layers.{l}.", d, heads, ff) for l in range(num_layers)]
        self.buf = _Buffers(arena.device)
        self.bucket_hook = None          # callable(group) fired when a group's grads are complete: 0 = stem, l + 1 = layer l, L + 1 = head
        self._temb_key = None

    def set_rng(self, seed_mix: int, rank: int, step: int, step_dev: Optional[torch.Tensor]) -> None:
        """No dropout: nothing to seed."""

    def refresh_weights(self) -> None:
        """The time-MLP table is refreshed by ``temb_table`` itself."""

    def bucket_boundaries(self) -> List[int]:
        offs = self.arena.offsets
        first = [offs[f"layers.{l}.multihead_attention.in_proj_weight"][0] for l in range(self.L)]
        return [0] + first + [offs["out_proj.weight"][0]]

    # ---- buffers ----
    def state(self, B: int, train: bool) -> Dict[str, torch.Tensor]:
        return self.buf.get((B, train))

    def xc(self, B: int, train: bool = True) -> torch.Tensor:
        return self.buf.tensor(self.state(B, train), "xc", (B * self.F, self.ld_in), BF16, zero=True)

    def input_layout(self, B: int, F: int, train: bool) -> Tuple[torch.Tensor, int, int, int]:
        """(buffer, frame_stride, win_extra, col0) for the packers: the kinematics go to columns 30… of xc."""
        return self.xc(B, train), self.ld_in, 0, 30

    def t_buffer(self, B: int, train: bool = True) -> torch.Tensor:
        return self.buf.tensor(self.state(B, train), "t", (B,), torch.int32, zero=True)

    def dout(self, B: int, F: int) -> torch.Tensor:
        return self.buf.tensor(self.state(B, True), "dout", (B * self.F, 32), BF16, zero=True)

    def quantity_views(self, x: torch.Tensor, B: int, F: int, Fo: int) -> List[torch.Tensor]:
        """(B, Fo, ·) views of the four quantities of the last Fo frames of an [M, 32] output / output-gradient buffer."""
        return quantity_split(x.view(B, self.F, 32)[:, self.F - Fo:])

    def _check_frames(self, F: int) -> None:
        if F != self.F:
            raise ValueError(f"the denoiser was built for {self.F}-frame windows, got {F}")

    # ---- forward ----
    def temb_table(self, n_timesteps: int) -> torch.Tensor:
        """bf16 [n, d]: the time MLP (Linear·SiLU·Linear of the sinusoidal embedding, DESIGN D-1) of EVERY timestep,
        evaluated once per set of weights.  Reverse sampling runs all windows at the same timestep, so a denoise step
        only adds row t of this table (ibm_add_time_pos with t_row) instead of re-running two GEMMs per step."""
        A, d = self.arena, self.d
        key = (A.version, n_timesteps)
        if self._temb_key != key:
            n = n_timesteps
            t = torch.arange(n, dtype=torch.int32, device=A.device)
            emb, pre, act = (torch.empty(n, d, dtype=BF16, device=A.device) for _ in range(3))
            table = torch.empty(n, d, dtype=BF16, device=A.device)
            ops.timestep_embed(t, emb, d)
            ops.gemm(emb, A.shadow_of("time_mlp.0.weight", (d, d)), pre, n, d, d, bias=A.master_of("time_mlp.0.bias"))
            ops.act_fwd(pre, act, "silu")
            ops.gemm(act, A.shadow_of("time_mlp.2.weight", (d, d)), table, n, d, d, bias=A.master_of("time_mlp.2.bias"))
            self._temb_table, self._temb_key = table, key
        return self._temb_table

    def forward(self, B: int, F: int, train: bool, t_scalar: Optional[torch.Tensor] = None, t_count: int = 0) -> torch.Tensor:
        """Consumes xc(B) and t_buffer(B) (or a device scalar timestep); returns x0_hat fp32 [M, 32].
        ``t_count`` > 0 with ``t_scalar``: timesteps are < t_count and the time MLP comes from ``temb_table``."""
        self._check_frames(F)
        A, d = self.arena, self.d
        M = B * F
        st = self.state(B, train)
        T = self.buf.tensor
        xc = self.xc(B, train)
        h0 = T(st, "h0", (M, d), BF16)
        ops.gemm(xc, A.weight_operand("in_proj.weight", d, self.k_in), h0, M, d, self.k_in, bias=A.master_of("in_proj.bias"))
        if t_scalar is not None and t_count > 0 and not train:
            ops.add_time_pos(h0, self.temb_table(t_count), A.master_of("pos_embedding", (F, d)), M, F, d, t_row=t_scalar)
        else:
            emb, pre, act, temb = (T(st, k, (B, d), BF16) for k in ("emb", "tpre", "tact", "temb"))
            if t_scalar is not None:
                ops.timestep_embed(t_scalar, emb, d, scalar=True)
            else:
                ops.timestep_embed(self.t_buffer(B, train), emb, d)
            ops.gemm(emb, A.shadow_of("time_mlp.0.weight", (d, d)), pre, B, d, d, bias=A.master_of("time_mlp.0.bias"))
            ops.act_fwd(pre, act, "silu")
            ops.gemm(act, A.shadow_of("time_mlp.2.weight", (d, d)), temb, B, d, d, bias=A.master_of("time_mlp.2.bias"))
            ops.add_time_pos(h0, temb, A.master_of("pos_embedding", (F, d)), M, F, d)
        x = h0
        for l, layer in enumerate(self.layers):
            # inference re-uses one set of layer buffers; training keeps every layer's activations
            tag = f"L{l}" if train else "L"
            a = layer.alloc(self.buf, st, tag, M, train)
            if not train and l % 2 == 1:          # ping-pong the layer output so x (input) stays intact
                a = dict(a)
                a["x2"] = T(st, "L.x2b", (M, d), BF16)
            x = layer.forward(x, a, M, B, F)
        out = T(st, "out", (M, 32), F32)
        ops.gemm(x, A.shadow_of("out_proj.weight", (30, d)), out, M, 30, d, bias=A.master_of("out_proj.bias"))
        return out

    # ---- backward ----
    def backward(self, B: int, F: int) -> None:
        """Consumes dout(B, F) (bf16 d loss/d x0_hat rows, cols 30,31 zero); accumulates grads into the arena."""
        self._check_frames(F)
        A, d, ff = self.arena, self.d, self.ff
        M = B * F
        st = self.state(B, True)
        T = self.buf.tensor
        g = A.grad_of
        dout = self.dout(B, F)
        sc = {"ds": T(st, "ds", (M, d), BF16), "dh": T(st, "dh", (M, ff), BF16), "dx1": T(st, "dx1", (M, d), BF16),
              "do": T(st, "do", (M, d), BF16), "dqkv": T(st, "dqkv", (M, 3 * d), BF16)}
        dxa, dxb = T(st, "dxa", (M, d), BF16), T(st, "dxb", (M, d), BF16)
        x_last = st[f"L{self.L - 1}.x2"]
        ops.gemm(dout, x_last, g("out_proj.weight", (30, d)), 30, d, M, a_mn=True, b_mn=True, accumulate=True)
        ops.colsum(dout, M, 30, g("out_proj.bias"))
        ops.gemm(dout, A.shadow_of("out_proj.weight", (30, d)), dxa, M, d, 30, b_mn=True)
        if self.bucket_hook is not None:
            self.bucket_hook(self.L + 1)          # head gradients complete
        dx, other = dxa, dxb
        for l in range(self.L - 1, -1, -1):
            layer = self.layers[l]
            a = {k: st[f"L{l}.{k}"] for k in ("qkv", "o", "s1", "x1", "h", "s2", "x2", "mean1", "rstd1", "mean2", "rstd2")}
            a["hmask"] = st.get(f"L{l}.hmask")
            x_in = st["h0"] if l == 0 else st[f"L{l - 1}.x2"]
            layer.backward(x_in, a, dx, sc, M, B, F, other)
            dx, other = other, dx
            if self.bucket_hook is not None:
                self.bucket_hook(l + 1)
        # dx = d loss / d h0
        dtemb, dact, dpre = (T(st, k, (B, d), BF16) for k in ("dtemb", "dact", "dpre"))
        # one pass over dx: time-embedding gradient per window, positional-table gradient, in-projection bias gradient
        ops.add_time_pos_bwd(dx, dtemb, g("pos_embedding", (F, d)), M, F, d, dbias=g("in_proj.bias"))
        ops.gemm(dtemb, st["tact"], g("time_mlp.2.weight", (d, d)), d, d, B, a_mn=True, b_mn=True, accumulate=True)
        ops.colsum(dtemb, B, d, g("time_mlp.2.bias"))
        ops.gemm(dtemb, A.shadow_of("time_mlp.2.weight", (d, d)), dact, B, d, d, b_mn=True)
        ops.act_bwd(dact, st["tpre"], dpre, "silu")
        ops.gemm(dpre, st["emb"], g("time_mlp.0.weight", (d, d)), d, d, B, a_mn=True, b_mn=True, accumulate=True)
        ops.colsum(dpre, B, d, g("time_mlp.0.bias"))
        _wgrad(A, "in_proj.weight", d, self.k_in, dx, self.xc(B), M, self.buf, st)
        if self.bucket_hook is not None:
            self.bucket_hook(0)
