"""Motion-diffusion denoiser (builder-owned spec — the reference has NO diffusion model; its only
trace is the ignored launcher name at /root/reference/src/.gitignore:10.  Spec frozen in DESIGN.md D-1).

x0-prediction (MDM style): given packed kinematics c (B,F,C_in), a noisy 30-channel target x_t
(B,F,30) and a timestep t (B,), predict x0_hat split into the four ``OutputDataKeys`` the reference's
``RegressionLossEvaluator`` consumes, so the training loss *is* the reference's regression loss.
The encoder layers are the reference's ``TransformerLayer`` (post-LN, nn.MultiheadAttention, ReLU FFN;
/root/reference/src/models/TransformerBaseline.py:8-38) at d=512, 8 heads, FFN 2048, 8 layers; the
parameter containers below reproduce its ``state_dict`` keys so a reference layer's weights load.

Classifier-free guidance (DESIGN.md D-1): the null condition is all-zero kinematics, so a model trained with
``Trainer(cond_drop_prob=p)`` (``train --cond-drop-prob``) gives its unconditional prediction when ``forward`` is passed zero
kinematics, and guided x0_hat = u + s (c - u) is two calls of this module.  No parameter is added: checkpoints trained either
way have the same keys.
"""
from __future__ import annotations

from typing import Dict

import torch
import torch.nn as nn

from .. import ops
from ..engine import DenoiserEngine
from ..keys import InputDataKeys
from ._base import EngineModule


class _TransformerLayerParams(nn.Module):
    """Parameter container with the reference TransformerLayer's module names (no forward)."""

    def __init__(self, d: int, heads: int, ff: int):
        super().__init__()
        self.multihead_attention = nn.MultiheadAttention(d, heads, dropout=0.0, batch_first=True)
        self.feedforward = nn.Sequential(nn.Linear(d, ff), nn.ReLU(), nn.Linear(ff, d))
        self.norm1 = nn.LayerNorm(d)
        self.norm2 = nn.LayerNorm(d)


class _DenoiserFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, B, train, *params):
        eng = model.engine()
        out = eng.forward(B, eng.F, train)     # train ⇒ keep every layer's activations for backward
        ctx.model, ctx.B = model, B
        return out.clone()

    @staticmethod
    def backward(ctx, grad_out):
        model, B = ctx.model, ctx.B
        eng = model._engine
        M = B * eng.F
        ops.cast_pad(grad_out.contiguous().view(M, 32), eng.dout(B, eng.F), M, 30)
        return (None, None, None, *model._engine_backward(B, eng.F))


class DiffusionDenoiser(EngineModule):
    trains_by_diffusion = True

    def __init__(self, num_dofs: int = 23, num_joints: int = 12, root_history_len: int = 10, frames: int = 50,
                 d_model: int = 512, num_heads: int = 8, dim_feedforward: int = 2048, num_layers: int = 8):
        super().__init__()
        self._init_engine_state()
        self.num_dofs, self.num_joints, self.root_history_len = num_dofs, num_joints, root_history_len
        self.frames, self.d_model, self.num_heads, self.dim_feedforward, self.num_layers = \
            frames, d_model, num_heads, dim_feedforward, num_layers
        self.cond_width = num_dofs * 3 + 12 + num_joints * 3 + root_history_len * 6           # 177 (Groundlink.py:26)
        self.in_proj = nn.Linear(30 + self.cond_width, d_model)
        self.time_mlp = nn.Sequential(nn.Linear(d_model, d_model), nn.SiLU(), nn.Linear(d_model, d_model))
        self.pos_embedding = nn.Parameter(torch.randn(frames, d_model) * 0.02)
        self.layers = nn.ModuleList([_TransformerLayerParams(d_model, num_heads, dim_feedforward) for _ in range(num_layers)])
        self.out_proj = nn.Linear(d_model, 30)

    def _build_engine(self, arena):
        return DenoiserEngine(arena, self.cond_width, self.frames, self.d_model, self.num_heads, self.dim_feedforward,
                              self.num_layers)

    def forward(self, input: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        """input: the 10 kinematic keys (B,F,·) + InputDataKeys.X_T (B,F,30) + InputDataKeys.TIMESTEP (B,)."""
        assert len(input[InputDataKeys.POS].shape) == 3
        assert input[InputDataKeys.POS].shape[-1] == self.num_dofs
        assert input[InputDataKeys.JOINT_CENTERS_IN_ROOT_FRAME].shape[-1] == self.num_joints * 3
        assert input[InputDataKeys.ROOT_POS_HISTORY_IN_ROOT_FRAME].shape[-1] == self.root_history_len * 3
        assert input[InputDataKeys.ROOT_EULER_HISTORY_IN_ROOT_FRAME].shape[-1] == self.root_history_len * 3
        B, F = input[InputDataKeys.POS].shape[0], input[InputDataKeys.POS].shape[1]
        assert F == self.frames and tuple(input[InputDataKeys.X_T].shape) == (B, F, 30)
        eng = self.engine()
        train = torch.is_grad_enabled()
        layout = eng.input_layout(B, F, train)
        self._pack_dict(input, layout, F)
        self._pack_dict(input, layout[:3] + (0,), F, keys=(InputDataKeys.X_T,))        # x_t: columns 0..29
        eng.t_buffer(B, train).copy_(input[InputDataKeys.TIMESTEP].to(torch.int32), non_blocking=True)
        return self.forward_packed(B)

    def forward_packed(self, B: int) -> Dict[str, torch.Tensor]:
        """Forward from already filled engine buffers xc(B, train), t_buffer(B, train) (window-store fast path)."""
        F = self.frames
        return self._quantities(_DenoiserFunction.apply(self, B, torch.is_grad_enabled(), *self.parameters()), B, F, F)
