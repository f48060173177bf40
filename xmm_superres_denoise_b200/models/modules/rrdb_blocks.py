"""Parameter containers with the reference's names, shapes and construction order
(xmm_superres_denoise/models/modules/rrdb_blocks.py:10-70).

The convolutions are ``nn.Conv2d`` modules only so that ``state_dict()`` keys, OIHW fp32
shapes, default initialisation and optimizer / DDP behaviour are identical to the reference;
they are never called.  The arithmetic runs in ``engine.RRDBEngine`` (whole generator) --
a dense block on its own has no tensor to hand its activations to, so calling one directly
goes through a one-block engine (inference only).
"""
from __future__ import annotations

import torch
from torch import nn


def make_layer(block, n_layers):
    layers = []
    for _ in range(n_layers):
        layers.append(block())
    return nn.Sequential(*layers)


class ResidualDenseBlock_5C(nn.Module):
    def __init__(self, nf=64, gc=32, bias=True, memory_efficient: bool = False):
        super().__init__()
        # memory_efficient (activation checkpointing of the concats, rrdb_blocks.py:17-19,39-47): training reads the
        # GENERATOR's flag (engine_train.TrainEngine), keeps each dense block's input only and recomputes x1..x4 in the
        # backward pass.  A per-block mix is not supported: this block's own flag is kept for API compatibility only.
        # Inference ignores the flag, as checkpointing does.
        self.mem_efficient = memory_efficient
        self.nf, self.gc = nf, gc
        self.conv1 = nn.Conv2d(nf, gc, 3, 1, 1, bias=bias)
        self.conv2 = nn.Conv2d(nf + gc, gc, 3, 1, 1, bias=bias)
        self.conv3 = nn.Conv2d(nf + 2 * gc, gc, 3, 1, 1, bias=bias)
        self.conv4 = nn.Conv2d(nf + 3 * gc, gc, 3, 1, 1, bias=bias)
        self.conv5 = nn.Conv2d(nf + 4 * gc, nf, 3, 1, 1, bias=bias)
        self.lrelu = nn.LeakyReLU(negative_slope=0.2, inplace=True)

    def forward(self, x: torch.Tensor):
        from ...engine import standalone_block_forward

        return standalone_block_forward([self], x, rrdb=False)


class RRDB(nn.Module):
    """Residual in Residual Dense Block"""

    def __init__(self, nf, gc=32, memory_efficient: bool = False):
        super().__init__()
        self.RDB1 = ResidualDenseBlock_5C(nf, gc, memory_efficient=memory_efficient)
        self.RDB2 = ResidualDenseBlock_5C(nf, gc, memory_efficient=memory_efficient)
        self.RDB3 = ResidualDenseBlock_5C(nf, gc, memory_efficient=memory_efficient)

    def forward(self, x):
        from ...engine import standalone_block_forward

        return standalone_block_forward([self.RDB1, self.RDB2, self.RDB3], x, rrdb=True)
