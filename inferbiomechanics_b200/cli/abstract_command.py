"""Command base class: model factory and latest-checkpoint loader, same public methods as
``/root/reference/src/cli/abstract_command.py:11-120``.

Conscious fixes of reference defects (SURVEY §9.6), none of which change numerics:
* ``get_model('groundlink')`` passes ``num_joints=12`` (the reference call at :74-79 shifts the positional
  arguments and raises TypeError);
* ``'transformer'`` and ``'diffusion'`` are accepted model types;
* ``load_latest_checkpoint`` accepts state dicts saved from a DDP wrapper (``module.`` prefix, train.py:276).
``ensure_geometry`` (wget of bone meshes for the GUI) and ``AnalyticalBaseline`` are out of scope.
"""
from __future__ import annotations

import argparse
import logging
import os
from typing import List

import torch

from ..models.DiffusionDenoiser import DiffusionDenoiser
from ..models.FeedForwardRegressionBaseline import FeedForwardBaseline
from ..models.Groundlink import Groundlink
from ..models.TransformerBaseline import TransformerBaseline


class AbstractCommand:
    def register_subcommand(self, subparsers: argparse._SubParsersAction):
        pass

    def run(self, args: argparse.Namespace) -> bool:
        pass

    def register_model_options(self, parser: argparse.ArgumentParser):
        pass

    def get_model(self,
                  num_dofs: int,
                  num_contact_bodies: int,
                  model_type: str = 'feedforward',
                  history_len: int = 5,
                  stride: int = 1,
                  hidden_dims: List[int] = [512],
                  activation: str = 'relu',
                  batchnorm: bool = False,
                  dropout: bool = False,
                  dropout_prob: float = 0.0,
                  root_history_len: int = 10,
                  output_data_format: str = 'all_frames',
                  device: str = 'cpu'):
        if model_type == 'feedforward':
            model = FeedForwardBaseline(num_dofs, num_contact_bodies, history_len, output_data_format, activation, stride=stride,
                                        hidden_dims=hidden_dims, batchnorm=batchnorm, dropout=dropout, dropout_prob=dropout_prob,
                                        root_history_len=root_history_len, device=device)
        elif model_type == 'groundlink':
            model = Groundlink(num_dofs, 12, root_history_len, output_data_format)
        elif model_type == 'transformer':
            model = TransformerBaseline(num_dofs, history_len // stride)
        elif model_type == 'diffusion':
            model = DiffusionDenoiser(num_dofs, 12, root_history_len, frames=history_len // stride)
        else:
            raise ValueError(f"model type {model_type!r} is not available on the B200 path (analytical needs nimblephysics)")
        return model

    @staticmethod
    def latest_checkpoint_path(checkpoint_dir: str):
        if not os.path.exists(checkpoint_dir):
            return None
        checkpoints = [f for f in os.listdir(checkpoint_dir) if f.endswith(".pt")]
        if not checkpoints:
            return None
        checkpoints.sort(key=lambda x: (int(x.split('_')[1]), int(x.split('_')[3].split('.')[0])))
        return os.path.join(checkpoint_dir, checkpoints[-1])

    @classmethod
    def feedforward_layout(cls, checkpoint_dir: str):
        """(batchnorm, dropout) of the FeedForwardBaseline that wrote the latest checkpoint, read off its ``nn.Sequential``
        positions (FeedForward…py:68-75: per layer ``[Dropout][BatchNorm1d] Linear act``): BatchNorm leaves ``running_mean``
        buffers, and the first Linear sits at position ``int(dropout) + int(batchnorm)``."""
        path = cls.latest_checkpoint_path(checkpoint_dir)
        if path is None:
            return False, False
        sd = torch.load(path, map_location="cpu")['model_state_dict']
        keys = [k[len('module.'):] if k.startswith('module.') else k for k in sd]
        bn = any(k.endswith('running_mean') for k in keys)
        first_linear = min(int(k.split('.')[1]) for k, v in zip(keys, sd.values()) if k.endswith('.weight') and v.dim() == 2)
        return bn, first_linear - int(bn) == 1

    def load_latest_checkpoint(self, model, optimizer=None, checkpoint_dir="../checkpoints", *, state_key="model_state_dict"):
        """Loads the newest ``epoch_{e}_batch_{i}.pt`` into ``model`` (and ``optimizer``); returns (epoch, batch), or (-1, 0)
        if there is none.  ``state_key='ema_state_dict'`` loads the weight average ``train --ema-decay`` saved instead of
        the trained weights; a checkpoint without that entry is a ValueError."""
        if not os.path.exists(checkpoint_dir):
            print("Checkpoint directory does not exist!")
            return -1, 0
        checkpoints = [f for f in os.listdir(checkpoint_dir) if f.endswith(".pt")]
        if not checkpoints:
            print("No checkpoints available!")
            return -1, 0
        # epoch_{e}_batch_{i}.pt, newest by (epoch, batch)  (abstract_command.py:100)
        checkpoints.sort(key=lambda x: (int(x.split('_')[1]), int(x.split('_')[3].split('.')[0])))
        latest_checkpoint = os.path.join(checkpoint_dir, checkpoints[-1])
        logging.info(f"{latest_checkpoint=}")
        checkpoint = torch.load(latest_checkpoint, map_location="cpu")
        if state_key not in checkpoint:
            raise ValueError(f"{latest_checkpoint} holds no {state_key!r} (was it trained with --ema-decay?)")
        sd = checkpoint[state_key]
        if all(k.startswith('module.') for k in sd):
            sd = {k[len('module.'):]: v for k, v in sd.items()}
        model.load_state_dict(sd)
        if optimizer is not None and 'optimizer_state_dict' in checkpoint and hasattr(optimizer, 'load_state_dict'):
            optimizer.load_state_dict(checkpoint['optimizer_state_dict'])
        epoch = checkpoint['epoch']
        batch = checkpoints[-1].split('_')[3].split('.')[0]
        print(f"Loaded checkpoint from epoch {epoch}, batch {batch}")
        return epoch, int(batch)
