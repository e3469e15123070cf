"""Drop-in ``FeedForwardBaseline`` running on libibm_b200 (tcgen05 GEMMs with fused bias+activation).

Same constructor signature, ``forward(Dict[str,Tensor]) -> Dict[str,Tensor]`` contract, assertions,
``state_dict`` keys (``net.{i}.weight/bias``) and default initialisation as
``/root/reference/src/models/FeedForwardRegressionBaseline.py:14-121``.  The ``nn.Sequential`` below
is only the parameter container (same modules in the same order, so the same RNG stream yields the
same initial weights and checkpoints load unchanged); the arithmetic is the engine's.
"""
from __future__ import annotations

import logging
from typing import Dict, List

import torch
import torch.nn as nn

from .. import ops
from ..engine import FeedForwardEngine
from ..keys import InputDataKeys
from ._base import EngineModule

ACTIVATION_FUNCS = {"relu": nn.ReLU(), "tanh": nn.Tanh(), "sigmoid": nn.Sigmoid()}


class _FeedForwardFunction(torch.autograd.Function):
    """Autograd bridge: forward/backward are engine launch sequences; parameter tensors are passed
    only so autograd (and DDP's hooks) see them."""

    @staticmethod
    def forward(ctx, model, B, F, *params):
        eng = model.engine()
        out = eng.forward(B, F, model.training)
        ctx.model, ctx.B, ctx.F = model, B, F
        return out[:, :eng.out_cols].clone()

    @staticmethod
    def backward(ctx, grad_out):
        model, B, F = ctx.model, ctx.B, ctx.F
        eng = model._engine
        ops.cast_pad(grad_out.contiguous(), eng.dout(B, F), B, eng.out_cols)
        return (None, None, None, *model._engine_backward(B, F))


class FeedForwardBaseline(EngineModule):
    num_dofs: int
    num_contact_bodies: int
    history_len: int
    root_history_len: int

    def __init__(self,
                 num_dofs: int,
                 num_contact_bodies: int,
                 history_len: int,
                 output_data_format: str,
                 activation: str,
                 stride: int,
                 root_history_len: int,
                 hidden_dims: List[int] = [512, 512],
                 batchnorm: bool = False,
                 dropout: bool = False,
                 dropout_prob: float = 0.0,
                 device: str = 'cpu'):
        super().__init__()
        self._init_engine_state()
        self.stride = stride
        self.activation = activation
        self.output_data_format = output_data_format
        self.num_dofs = num_dofs
        self.num_contact_bodies = num_contact_bodies
        self.history_len = history_len
        self.root_history_len = root_history_len
        self.device = device
        self.batchnorm, self.dropout, self.dropout_prob = batchnorm, dropout, dropout_prob

        self.num_frames = history_len // stride
        self.frame_width = 3 * num_dofs + 4 * 3 + 2 * stride * 3 + 12 * 3
        self.input_size = self.frame_width * self.num_frames            # FeedForward…py:52
        self.num_output_frames = self.num_frames if output_data_format == 'all_frames' else 1
        self.output_size = num_contact_bodies * (3 * 3 + 6) * self.num_output_frames   # FeedForward…py:62
        # num_contact_bodies != 2 follows the reference literally: the last Linear has num_contact_bodies * 15 * F outputs and the
        # split below still takes the first 30 * F of them (FeedForward...py:116-121), so 3+ bodies carry unused outputs and
        # 1 body fails in the reshape exactly as the reference does

        net = []
        dims = [self.input_size] + list(hidden_dims) + [self.output_size]
        self._linear_pos = []
        self._bn_pos = []
        for i, (h0, h1) in enumerate(zip(dims[:-1], dims[1:])):
            if dropout:
                net.append(nn.Dropout(dropout_prob))
            if batchnorm:
                self._bn_pos.append(len(net))
                net.append(nn.BatchNorm1d(h0))
            self._linear_pos.append((len(net), h1, h0))
            net.append(nn.Linear(h0, h1, dtype=torch.float32, device=device if device != 'cpu' else None))
            if i < len(dims) - 2:
                net.append(ACTIVATION_FUNCS[self.activation])
        self.net = nn.Sequential(*net)
        logging.info(f"{self.net=}")

    def _build_engine(self, arena):
        layers = [(f"net.{pos}.weight", f"net.{pos}.bias", n, k) for pos, n, k in self._linear_pos]
        # [Dropout][BatchNorm1d] sit on each Linear's input (FeedForward…py:68-72): BatchNorm1d over the packed bf16 rows
        # (ibm_batchnorm_fwd/bwd, batch statistics when self.training), Philox inverted dropout (ibm_dropout_bf16)
        bn = [(f"net.{p}.weight", f"net.{p}.bias", self.net[p]) for p in self._bn_pos] if self.batchnorm else None
        return FeedForwardEngine(arena, layers, self.activation, self.frame_width, bn=bn,
                                 dropout_p=self.dropout_prob if self.dropout else 0.0)

    def forward(self, input: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        # 1. same shape assertions as the reference (FeedForward…py:83-94)
        assert len(input[InputDataKeys.POS].shape) == 3
        assert input[InputDataKeys.POS].shape[-1] == self.num_dofs
        assert input[InputDataKeys.VEL].shape[-1] == self.num_dofs
        assert input[InputDataKeys.ACC].shape[-1] == self.num_dofs
        assert len(input[InputDataKeys.JOINT_CENTERS_IN_ROOT_FRAME].shape) == 3
        assert input[InputDataKeys.JOINT_CENTERS_IN_ROOT_FRAME].shape[-1] == 12 * 3
        assert len(input[InputDataKeys.ROOT_POS_HISTORY_IN_ROOT_FRAME].shape) == 3
        assert input[InputDataKeys.ROOT_POS_HISTORY_IN_ROOT_FRAME].shape[-1] == self.stride * 3
        assert len(input[InputDataKeys.ROOT_EULER_HISTORY_IN_ROOT_FRAME].shape) == 3
        assert input[InputDataKeys.ROOT_EULER_HISTORY_IN_ROOT_FRAME].shape[-1] == self.stride * 3
        eng = self.engine()
        B, F = input[InputDataKeys.POS].shape[0], input[InputDataKeys.POS].shape[1]
        assert F * self.frame_width == self.input_size, "window length does not match history_len // stride"
        if self._latency_path(B):
            # batch-of-1 viewers (visualize.py:181, save_prediction_csv.py:103): pack + 3 GEMMs replayed from one CUDA graph
            return self._quantities(self._graphed_inference(input, F)[:, :eng.out_cols], B, F, self.num_output_frames)
        # 2. concat + flatten + bf16 in one kernel (row-per-window layout, K padded to a multiple of 8)
        self._pack_dict(input, eng.input_layout(B, F, self.training), F)
        return self.forward_packed(B)

    def forward_packed(self, B: int) -> Dict[str, torch.Tensor]:
        """Forward from an already packed engine.input_buffer(B) (the window-store fast path); quantity-then-frame blocks
        of the output row (FeedForward…py:116-121)."""
        F = self.num_frames
        return self._quantities(_FeedForwardFunction.apply(self, B, F, *self.parameters()), B, F, self.num_output_frames)
