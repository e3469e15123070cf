"""Launch plan for the Groundlink CNN (/root/reference/src/models/Groundlink.py:20-77, 105-156):
4 x [Conv1d(k=7, padding=3, padding_mode="replicate") + ELU] over time, then per-frame
Linear(256,256)+ELU x2 and Linear(256,30, bias=False), with Dropout(0.2) before each Linear in training.

The temporal convolution is an implicit GEMM on tcgen05 (``ibm_gemm_bf16(taps=7)``): activations live in a
*padded row layout* — window b owns rows [b*Tp, (b+1)*Tp), Tp = T + 6, frame t at row b*Tp + 3 + t, the 3+3
pad rows holding copies of the first / last frame (replicate padding) — so tap j of output row r reads row
r + j and the whole convolution is one GEMM with K = 7 * C_in.  The GEMM's TMA store is pointed 3 rows down,
which drops each frame's output straight into its slot of the next layer's padded buffer; a tiny kernel then
refreshes the 6 pad rows per window.  Backward: dgrad is the same implicit GEMM with flipped taps and
transposed weights, wgrad is 7 MN-major split-K GEMMs (one per tap) accumulating into an fp32 scratch in GEMM
layout that is folded back into the (C_out, C_in, 7) parameter gradient.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import torch

from . import ops
from .engine import _Buffers, _r8, quantity_split
from .params import ParamArena

BF16, F32 = torch.bfloat16, torch.float32


class GroundlinkEngine:
    CNN_DROPOUT_SEED = 0x636e6e64
    FC_DROPOUT_SEED = 0x6c696e6b

    def __init__(self, arena: ParamArena, c_in: int, features: List[int], fc_dropout: float, cnn_dropout: float = 0.0,
                 cnn_kernel: int = 7, fc_depth: int = 3):
        """``cnn_kernel`` (odd) and ``fc_depth`` are the reference constructor's arguments (Groundlink.py:20): kernel taps of every
        Conv1d (padding = cnn_kernel // 2, replicate) and the number of Linear layers of the per-frame MLP (fc_depth - 1 hidden
        256 -> 256 + ELU layers, then 256 -> 30 without bias)."""
        assert cnn_kernel % 2 == 1 and cnn_kernel >= 1 and fc_depth >= 1
        self.kt, self.pad, self.fc_depth = cnn_kernel, cnn_kernel // 2, fc_depth
        self.arena = arena
        self.ch = [c_in] + list(features)                 # [177, 128, 128, 256, 256]
        self.ld = [_r8(c) for c in self.ch]               # row pitch of each layer's activation buffer
        self.cin_pad = [ops.round_up(self.ld[i], 64) for i in range(4)]       # per-tap K padded to whole 64-wide k blocks
        self.cout_pad = [ops.round_up(self.ch[i + 1], 64) for i in range(4)]
        self.conv_pos = (1, 4, 7, 10)                     # nn.Sequential positions (SURVEY §9.3)
        self.fc_pos = tuple(3 * j + 2 for j in range(fc_depth))     # [Transpose, (Dropout, Linear, ELU) x (depth-1), Dropout, Linear]
        self.fc_dropout = fc_dropout
        self.cnn_dropout = float(cnn_dropout)             # nn.Dropout before every Conv1d (Groundlink.py:41, default 0.0)
        self.buf = _Buffers(arena.device)
        self._w_version = None
        self._w: Dict[str, torch.Tensor] = {}
        self.set_rng(0, 0, 0, None)
        self.bucket_hook = None                 # callable(group) fired when a group's grads are complete: 0-3 = conv layers, 4 = the MLP

    def set_rng(self, seed_mix: int, rank: int, step: int, step_dev: Optional[torch.Tensor]) -> None:
        """Dropout masks: Philox keyed by (CNN/FC_DROPOUT_SEED ^ seed_mix) + rank, offset by the training-forward count
        ``step`` — or, when ``step_dev`` (a device-resident step counter) is given, by its value, so that a captured step
        replays."""
        self.cnn_seed = (self.CNN_DROPOUT_SEED ^ seed_mix) + rank
        self.fc_seed = (self.FC_DROPOUT_SEED ^ seed_mix) + rank
        self.step, self.step_dev = step, step_dev

    def bucket_boundaries(self) -> List[int]:
        offs = self.arena.offsets
        return [offs[f"cnn.{p}.weight"][0] for p in self.conv_pos] + [offs[f"fc.{self.fc_pos[0]}.weight"][0]]

    def _drop(self, x, y, p, seed, mul, add, step):
        """Philox offset = mul * step + add, the step taken from the device counter when the Trainer owns one."""
        if self.step_dev is not None:
            ops.dropout(x, y, p, seed, add, self.step_dev, mul)
        else:
            ops.dropout(x, y, p, seed, mul * step + add)

    # ---- weights in GEMM layouts (refreshed when the fp32 masters change) ---------------------------------
    def refresh_weights(self) -> Dict[str, torch.Tensor]:
        """Re-lays the conv weights out for the GEMMs if the arena's weights version moved.  The copies are updated in place,
        so a captured step that contains the re-layout keeps reading them."""
        ver = self.arena.version
        if self._w_version == ver and self._w:
            return self._w
        dev = self.arena.device
        for i, pos in enumerate(self.conv_pos):
            cout, cin = self.ch[i + 1], self.ch[i]
            KT = self.kt
            w = self.arena.master_of(f"cnn.{pos}.weight", (cout, cin, KT))
            fw = self._w.get(f"f{i}")
            if fw is None:
                fw = self._w[f"f{i}"] = torch.empty(cout, KT * self.cin_pad[i], dtype=BF16, device=dev)
                self._w[f"d{i}"] = torch.empty(cin, KT * self.cout_pad[i], dtype=BF16, device=dev)
            ops.conv_weight_to_gemm(w, fw, self.cin_pad[i])
            ops.conv_weight_to_dgrad(w, self._w[f"d{i}"], self.cout_pad[i])
        self._w_version = ver
        return self._w

    # ---- buffers ---------------------------------------------------------------------------------------------
    def _state(self, B: int, T: int):
        st = self.buf.get((B, T))
        PAD = self.pad
        Tp = T + 2 * PAD
        Mp = B * Tp
        if "x0" not in st:
            slack = max(8, ops.round_up(self.kt + 1, 8))   # rows of zeros before/after: tap shifts (+kt-1) and the +pad store shift
            for i in range(5):
                full = torch.zeros(Mp + 2 * slack, self.ld[i], dtype=BF16, device=self.arena.device)
                st[f"x{i}_full"] = full
                st[f"x{i}"] = full[slack:slack + Mp]
                gfull = torch.zeros(Mp + 2 * slack, self.ld[i], dtype=BF16, device=self.arena.device)
                st[f"g{i}_full"] = gfull
                st[f"g{i}"] = gfull[slack:slack + Mp]
            names = ["y4d"] + [f"{k}{j}" for j in range(1, self.fc_depth) for k in ("h", "hd", "dh")]
            for k in names:
                st[k] = torch.zeros(Mp, self.ch[-1], dtype=BF16, device=self.arena.device)
            st["out"] = torch.zeros(Mp, 32, dtype=F32, device=self.arena.device)
            st["dout"] = torch.zeros(Mp, 32, dtype=BF16, device=self.arena.device)
            st["slack"] = slack
        return st, Tp, Mp

    def input_layout(self, B: int, T: int, train: bool) -> Tuple[torch.Tensor, int, int, int]:
        """(buffer, frame_stride, win_extra, col0) for the packers: frame t of window b → row b*Tp + 3 + t."""
        st, Tp, Mp = self._state(B, T)
        ld = self.ld[0]
        return st["x0"], ld, 2 * self.pad * ld, self.pad * ld

    def _frames(self, name: str, B: int, T: int) -> torch.Tensor:
        st, Tp, Mp = self._state(B, T)
        return st[name].view(B, Tp, 32)[:, self.pad:self.pad + T, :]

    def dout(self, B: int, T: int) -> torch.Tensor:
        """(B, T, 32) bf16 view of the output-gradient rows (all other rows stay zero)."""
        return self._frames("dout", B, T)

    def quantity_views(self, x: torch.Tensor, B: int, T: int, Fo: int) -> List[torch.Tensor]:
        """(B, Fo, ·) views of the four quantities of a (B, T, 32) output / output-gradient view; Fo = 1 is the last
        frame, the only output of ``last_frame`` (Groundlink.py:147-148)."""
        return quantity_split(x[:, T - Fo:])

    # ---- forward ---------------------------------------------------------------------------------------------
    def forward(self, B: int, T: int, train: bool) -> torch.Tensor:
        """Consumes input_layout (frames written at rows b*Tp+3+t); returns the (B, T, 32) fp32 output view."""
        A = self.arena
        W = self.refresh_weights()
        st, Tp, Mp = self._state(B, T)
        PAD, KT, depth, C = self.pad, self.kt, self.fc_depth, self.ch[-1]
        self.step += 1
        cdrop = train and self.cnn_dropout > 0.0
        st["cnn_dropped"] = cdrop
        ops.replicate_pad_rows(st["x0"], B, T, PAD, self.ld[0])
        for i, pos in enumerate(self.conv_pos):
            x, y_full = st[f"x{i}"], st[f"x{i + 1}_full"]
            slack = st["slack"]
            if cdrop:
                # Dropout on the conv INPUT, before the (replicate) padding the conv applies itself: mask the whole buffer with
                # Philox(seed, 4*step + i) (zeros stay zeros), then let the pad rows replicate the DROPPED edge frames
                xd_full = st.get(f"xd{i}_full")
                if xd_full is None:
                    xd_full = st[f"xd{i}_full"] = torch.zeros_like(st[f"x{i}_full"])
                    st[f"xd{i}"] = xd_full[slack:slack + Mp]
                self._drop(st[f"x{i}_full"], xd_full, self.cnn_dropout, self.cnn_seed, 4, i, self.step)
                ops.replicate_pad_rows(st[f"xd{i}"], B, T, PAD, self.ld[i])
                x = st[f"xd{i}"]
            y_shift = y_full[slack + PAD: slack + PAD + Mp]             # the store lands 3 rows down: frame slots of layer i+1
            ops.gemm(x, W[f"f{i}"], y_shift, Mp, self.ch[i + 1], KT * self.ld[i], lda=self.ld[i], bias=A.master_of(f"cnn.{pos}.bias"),
                     act="elu", taps=KT)
            ops.replicate_pad_rows(st[f"x{i + 1}"], B, T, PAD, self.ld[i + 1])
        drop = train and self.fc_dropout > 0.0
        a = st["x4"]
        for j, pos in enumerate(self.fc_pos):                # Linear j reads the (dropped) output of layer j-1 / the CNN
            if drop:
                ad = st["y4d"] if j == 0 else st[f"hd{j}"]
                self._drop(a, ad, self.fc_dropout, self.fc_seed, depth, j, self.step)
                a = ad
            if j < depth - 1:
                ops.gemm(a, A.shadow_of(f"fc.{pos}.weight", (C, C)), st[f"h{j + 1}"], Mp, C, C, bias=A.master_of(f"fc.{pos}.bias"), act="elu")
                a = st[f"h{j + 1}"]
            else:
                ops.gemm(a, A.shadow_of(f"fc.{pos}.weight", (30, C)), st["out"], Mp, 30, C)
        st["dropped"] = drop
        return self._frames("out", B, T)

    # ---- backward ---------------------------------------------------------------------------------------------
    def backward(self, B: int, T: int) -> None:
        """Consumes dout(B, T) (bf16; all other rows zero); accumulates parameter grads."""
        A = self.arena
        W = self.refresh_weights()
        g = A.grad_of
        st, Tp, Mp = self._state(B, T)
        drop = st.get("dropped", False)
        cdrop = st.get("cnn_dropped", False)
        PAD, KT, depth, C = self.pad, self.kt, self.fc_depth, self.ch[-1]
        p, s = self.fc_dropout, self.step
        dy, n_out = st["dout"], 30
        for j in range(depth - 1, -1, -1):
            pos = self.fc_pos[j]
            pre = st["x4"] if j == 0 else st[f"h{j}"]                    # ELU output feeding Linear j (before its dropout)
            x_in = (st["y4d"] if j == 0 else st[f"hd{j}"]) if drop else pre
            ops.gemm(dy, x_in, g(f"fc.{pos}.weight", (n_out, C)), n_out, C, Mp, a_mn=True, b_mn=True, accumulate=True)
            if j < depth - 1:                                            # the last Linear has no bias (Groundlink.py:62)
                ops.colsum(dy, Mp, C, g(f"fc.{pos}.bias"))
            # gradient w.r.t. the ELU output below, through its derivative; for j == 0 that is the last conv layer's padded output
            dx = st["g4"] if j == 0 else st[f"dh{j}"]
            ops.gemm(dy, A.shadow_of(f"fc.{pos}.weight", (n_out, C)), dx, Mp, C, n_out, b_mn=True, act="elu", aux=pre, aux_mode=2)
            if drop:
                self._drop(dx, dx, p, self.fc_seed, depth, j, s)
            dy, n_out = dx, C
        if self.bucket_hook is not None:
            self.bucket_hook(4)
        slack = st["slack"]
        for i in range(3, -1, -1):
            pos = self.conv_pos[i]
            cout, cin = self.ch[i + 1], self.ch[i]
            G = st[f"g{i + 1}"]                              # d loss / d (ELU output of conv i), padded layout, already times ELU'
            ops.fold_pad_rows(G, B, T, PAD, self.ld[i + 1])  # replicate-pad adjoint; pad rows become zero
            if cdrop and i + 1 <= 3:
                # adjoint of the dropout in front of conv i+1: the same Philox mask over the identically shaped buffer (the ELU
                # derivative fused into the producing dgrad commutes with it, and with the fold because pads replicate x)
                Gfull = st[f"g{i + 1}_full"]
                self._drop(Gfull, Gfull, self.cnn_dropout, self.cnn_seed, 4, i + 1, s)
            ops.colsum(G, Mp, cout, g(f"cnn.{pos}.bias"))
            # wgrad: dW_j[co, ci] = sum_r G[r + 3, co] * Xp[r + j, ci]  (7 split-K MN-major GEMMs into GEMM-layout scratch)
            wg = self.buf.tensor(st, f"wg{i}", (cout, KT * self.cin_pad[i]), F32)
            wg.zero_()
            Gf, Xf = st[f"g{i + 1}_full"], st[f"xd{i}_full" if cdrop else f"x{i}_full"]
            for j in range(KT):
                ops.gemm(Gf[slack + PAD:], Xf[slack + j:], wg[:, j * self.cin_pad[i]:], cout, cin, Mp, lda=self.ld[i + 1], ldb=self.ld[i],
                         ldd=KT * self.cin_pad[i], a_mn=True, b_mn=True, accumulate=True)
            ops.conv_wgrad_from_gemm(wg, g(f"cnn.{pos}.weight", (cout, cin, KT)), self.cin_pad[i], accumulate=True)
            if i > 0:
                # dgrad: dXp[s] = sum_j G[s - j + 3] W_j^T  → taps GEMM over rows shifted up by 3, flipped/transposed weights,
                # times ELU'(x_i) in the epilogue (x_i = padded output of conv i-1, pad rows included)
                ops.gemm(Gf[slack - PAD:], W[f"d{i}"], st[f"g{i}"], Mp, cin, KT * self.ld[i + 1], lda=self.ld[i + 1], act="elu",
                         aux=st[f"x{i}"], aux_mode=2, taps=KT)
            if self.bucket_hook is not None:
                self.bucket_hook(i)
