"""Drop-in ``Groundlink`` (temporal CNN + per-frame MLP) on libibm_b200.

Constructor signature, ``forward(Dict) -> Dict`` contract, assertions, Xavier initialisation and
``state_dict`` keys (``cnn.{1,4,7,10}.{weight,bias}``, ``fc.{2,5}.{weight,bias}``, ``fc.8.weight``) follow
``/root/reference/src/models/Groundlink.py:20-156``.  The ``nn.Sequential`` containers only hold the
parameters; the arithmetic is ``GroundlinkEngine`` (implicit-GEMM convolutions on tcgen05, see
engine_groundlink.py).  Note the reference's own factory call passes the wrong positional arguments
(``src/cli/abstract_command.py:74-79``, SURVEY §0.3); construct it directly with ``num_joints=12``.
"""
from __future__ import annotations

from typing import Dict

import torch
import torch.nn as nn

from ..engine_groundlink import GroundlinkEngine
from ..keys import InputDataKeys
from ._base import EngineModule


class Transpose(nn.Module):
    def __init__(self, dim1, dim2):
        super().__init__()
        self._dim1, self._dim2 = dim1, dim2

    def extra_repr(self):
        return "{}, {}".format(self._dim1, self._dim2)

    def forward(self, input):
        return input.transpose(self._dim1, self._dim2)


class _GroundlinkFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, B, T, train, *params):
        eng = model.engine()
        out = eng.forward(B, T, train)
        ctx.model, ctx.B, ctx.T = model, B, T
        return out.clone()

    @staticmethod
    def backward(ctx, grad_out):
        model, B, T = ctx.model, ctx.B, ctx.T
        dv = model._engine.dout(B, T)
        dv[:, :, :30] = grad_out[:, :, :30].to(torch.bfloat16)          # strided write into the padded-row gradient buffer
        return (None, None, None, None, *model._engine_backward(B, T))


class Groundlink(EngineModule):
    def __init__(self, num_dofs: int, num_joints: int, root_history_len: int, output_data_format: str = "all_frames",
                 cnn_kernel=7, cnn_dropout=0.0, fc_depth=3, fc_dropout=0.2):
        super().__init__()
        self._init_engine_state()
        self.num_dofs = num_dofs
        self.num_joints = num_joints
        self.root_history_len = root_history_len
        self.output_data_format = output_data_format
        if cnn_kernel % 2 == 0:
            # Conv1d(k, padding=k // 2) with an even k emits T + 1 frames per layer: the reference's own output slicing and
            # loss then fail on the frame count, so there is no behaviour to reproduce
            raise NotImplementedError("even cnn_kernel: Conv1d(padding=k//2) changes the number of frames (unusable in the reference too)")
        if fc_depth < 1:
            raise ValueError("fc_depth must be >= 1")
        self.cnn_kernel, self.fc_depth = cnn_kernel, fc_depth
        self.cnn_dropout, self.fc_dropout = cnn_dropout, fc_dropout
        input_size = (num_dofs * 3 + 12 + num_joints * 3 + root_history_len * 6)
        self.input_size = input_size
        cnn_features = [input_size, 128, 128, 256, 256]
        self.cnn_features = cnn_features
        features_out = 30

        pre_layers = [torch.nn.Flatten(start_dim=2, end_dim=-1), Transpose(-2, -1)]
        conv = lambda c_in, c_out: torch.nn.Conv1d(c_in, c_out, cnn_kernel, padding=cnn_kernel // 2, padding_mode="replicate")
        cnn_layers = []
        for c_in, c_out in zip(cnn_features[:-1], cnn_features[1:]):
            cnn_layers += [torch.nn.Dropout(p=cnn_dropout), conv(c_in, c_out), torch.nn.ELU()]
        fc_layers = [Transpose(-2, -1)]
        for _ in range(fc_depth - 1):
            fc_layers += [torch.nn.Dropout(p=fc_dropout), torch.nn.Linear(cnn_features[-1], cnn_features[-1]), torch.nn.ELU()]
        fc_layers += [torch.nn.Dropout(p=fc_dropout), torch.nn.Linear(cnn_features[-1], features_out, bias=False)]
        self.pre_net = self.initialize(nn.Sequential(*pre_layers))
        self.cnn = self.initialize(nn.Sequential(*cnn_layers))
        self.fc = self.initialize(nn.Sequential(*fc_layers))

    def initialize(self, net):
        """Xavier-normal with the ReLU gain for every Linear/Conv1d that is followed by an ELU, zero bias
        (Groundlink.py:79-103; layers not followed by an activation keep torch's default init)."""
        gain = torch.nn.init.calculate_gain("relu")
        mods = list(net)
        for layer, nxt in zip(mods[:-1], mods[1:]):
            if isinstance(layer, (torch.nn.Linear, torch.nn.Conv1d)) and isinstance(nxt, torch.nn.ELU):
                torch.nn.init.xavier_normal_(layer.weight, gain)
                if layer.bias is not None:
                    torch.nn.init.zeros_(layer.bias)
        return net

    def _build_engine(self, arena):
        return GroundlinkEngine(arena, self.input_size, self.cnn_features[1:], self.fc_dropout, self.cnn_dropout,
                                cnn_kernel=self.cnn_kernel, fc_depth=self.fc_depth)

    def forward(self, input: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        # 1. same shape assertions as the reference (Groundlink.py:107-118)
        assert len(input[InputDataKeys.POS].shape) == 3
        assert input[InputDataKeys.POS].shape[-1] == self.num_dofs
        assert len(input[InputDataKeys.VEL].shape) == 3
        assert input[InputDataKeys.VEL].shape[-1] == self.num_dofs
        assert len(input[InputDataKeys.ACC].shape) == 3
        assert input[InputDataKeys.ACC].shape[-1] == self.num_dofs
        assert len(input[InputDataKeys.JOINT_CENTERS_IN_ROOT_FRAME].shape) == 3
        assert input[InputDataKeys.JOINT_CENTERS_IN_ROOT_FRAME].shape[-1] == self.num_joints * 3
        assert len(input[InputDataKeys.ROOT_POS_HISTORY_IN_ROOT_FRAME].shape) == 3
        assert input[InputDataKeys.ROOT_POS_HISTORY_IN_ROOT_FRAME].shape[-1] == self.root_history_len * 3
        assert len(input[InputDataKeys.ROOT_EULER_HISTORY_IN_ROOT_FRAME].shape) == 3
        assert input[InputDataKeys.ROOT_EULER_HISTORY_IN_ROOT_FRAME].shape[-1] == self.root_history_len * 3
        eng = self.engine()
        B, T = input[InputDataKeys.POS].shape[0], input[InputDataKeys.POS].shape[1]
        if self._latency_path(B):
            # batch-of-1 viewers: packer + 4 implicit-GEMM convolutions + pad refreshes + MLP replayed from one CUDA graph
            return self._quantities(self._graphed_inference(input, T), B, T, self._output_frames(T))
        # 2. concat → bf16 rows in the padded-row layout (frame t of window b at row b*(T+6) + 3 + t)
        self._pack_dict(input, eng.input_layout(B, T, self.training), T)
        return self.forward_packed(B, T)

    def forward_packed(self, B: int, T: int) -> Dict[str, torch.Tensor]:
        out = _GroundlinkFunction.apply(self, B, T, self.training and torch.is_grad_enabled(), *self.parameters())
        return self._quantities(out, B, T, self._output_frames(T))

    def _output_frames(self, T: int) -> int:
        return T if self.output_data_format == 'all_frames' else 1      # Groundlink.py:147-148: last_frame keeps the last one
