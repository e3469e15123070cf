"""Flat parameter / gradient / bf16-shadow arenas.

All parameters of a model live in ONE contiguous fp32 tensor (each parameter 256-byte aligned), all
gradients in a second, and a bf16 shadow copy of the parameters (what the tcgen05 GEMMs read) in a
third with the same offsets.  ``nn.Parameter``s are ordinary contiguous views into the master arena
(and their ``.grad`` into the gradient arena), so ``state_dict``/``load_state_dict``, torch
optimizers and DDP keep working on them; the B200-native trainer instead treats each arena as one
buffer: one memset to zero gradients, one bucketed NCCL allreduce per contiguous slice (no
pack/unpack), one fused optimizer launch that also refreshes the shadow.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import torch

from . import ops

ALIGN = 64  # elements: 256 B in fp32, 128 B in bf16 (TMA needs 16-byte aligned bases)


class ParamArena:
    def __init__(self, named_params: List[Tuple[str, torch.nn.Parameter]], device: torch.device):
        self.device = torch.device(device)
        self.names: List[str] = []
        self.params: List[torch.nn.Parameter] = []
        self.offsets: Dict[str, Tuple[int, int]] = {}
        off = 0
        for n, p in named_params:
            if p.dtype != torch.float32:
                raise TypeError(f"parameter {n} is {p.dtype}; the B200 path keeps fp32 masters with bf16 shadows")
            self.names.append(n)
            self.params.append(p)
            self.offsets[n] = (off, p.numel())
            off += ops.round_up(p.numel(), ALIGN)
        self.total = max(off, ALIGN)
        self.master = torch.zeros(self.total, dtype=torch.float32, device=self.device)
        self.grad = torch.zeros(self.total, dtype=torch.float32, device=self.device)
        self.shadow = torch.zeros(self.total, dtype=torch.bfloat16, device=self.device)
        self.grad_target = self.grad
        self._scratch: Optional[torch.Tensor] = None
        with torch.no_grad():
            for n, p in zip(self.names, self.params):
                o, k = self.offsets[n]
                self.master[o:o + k].copy_(p.detach().reshape(-1))
                p.data = self.master[o:o + k].view(p.shape)
                p.grad = self.grad[o:o + k].view(p.shape)
        self._ptrs = [p.data_ptr() for p in self.params]
        self._versions: Optional[int] = None
        self._device_writes = 0
        self.padded: Dict[str, torch.Tensor] = {}      # bf16 copies with ld rounded up to 8 for odd-K weights
        self.sync_shadow(force=True)

    # -- validity -----------------------------------------------------------------------------
    def intact(self) -> bool:
        """False once someone re-pointed a parameter (model.to(), load_state_dict(assign=True) …)."""
        return all(p.data_ptr() == q and p.device == self.device for p, q in zip(self.params, self._ptrs))

    def _version_sum(self) -> int:
        return sum(p._version for p in self.params)

    @property
    def version(self) -> int:
        """Changes whenever the fp32 masters may have changed: torch's in-place writes (each parameter's ``_version``) plus
        device-side writes (``bump_version``).  Caches of weights derived from the masters key on it."""
        return self._version_sum() + self._device_writes

    def bump_version(self) -> None:
        """Records a write of the masters that torch does not see: the fused optimizer writes them through raw pointers,
        eagerly or from a replayed CUDA graph."""
        self._device_writes += 1

    # -- views ----------------------------------------------------------------------------------
    def shadow_of(self, name: str, shape=None) -> torch.Tensor:
        o, k = self.offsets[name]
        v = self.shadow[o:o + k]
        return v.view(shape) if shape is not None else v

    def grad_of(self, name: str, shape=None) -> torch.Tensor:
        """View into the current gradient target (the .grad arena for the native trainer, the scratch
        arena while an autograd.Function backward is running)."""
        o, k = self.offsets[name]
        v = self.grad_target[o:o + k]
        return v.view(shape) if shape is not None else v

    def scratch_grad(self) -> torch.Tensor:
        if self._scratch is None:
            self._scratch = torch.zeros_like(self.grad)
        return self._scratch

    def master_of(self, name: str, shape=None) -> torch.Tensor:
        o, k = self.offsets[name]
        v = self.master[o:o + k]
        return v.view(shape) if shape is not None else v

    def weight_operand(self, name: str, rows: int, cols: int) -> torch.Tensor:
        """bf16 [rows, ld] GEMM operand for a 2-D weight: the shadow itself when cols % 8 == 0, else a
        zero-padded copy (TMA needs 16-byte rows and zero pad columns)."""
        if cols % 8 == 0:
            return self.shadow_of(name, (rows, cols))
        if name not in self.padded:
            self.padded[name] = torch.zeros(rows, ops.round_up(cols, 8), dtype=torch.bfloat16, device=self.device)
            ops.cast_pad(self.master_of(name, (rows, cols)), self.padded[name], rows, cols)
        return self.padded[name]

    # -- maintenance ------------------------------------------------------------------------------
    def sync_shadow(self, force: bool = False) -> None:
        """Refresh the bf16 shadow if any parameter was modified in place since the last refresh
        (torch optimizers, load_state_dict, manual edits all bump ``_version``)."""
        v = self._version_sum()
        if force or v != self._versions:
            ops.cast_f32_bf16(self.master, self.shadow)
            self.refresh_padded()
            self._versions = v

    def refresh_padded(self) -> None:
        for name, buf in self.padded.items():
            o, k = self.offsets[name]
            rows = buf.shape[0]
            ops.cast_pad(self.master[o:o + k].view(rows, k // rows), buf, rows, k // rows)

    def mark_shadow_fresh(self) -> None:
        """Called after the fused optimizer kernel (which writes the masters and the shadow itself)."""
        self.refresh_padded()
        self._versions = self._version_sum()
        self.bump_version()

    def zero_grad(self) -> None:
        self.grad.zero_()
