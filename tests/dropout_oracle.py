"""ResNet-block dropout on top of the CPU oracle (oracle/cgan_oracle.py).  TEST INFRASTRUCTURE, NOT PRODUCT.

The reference's ResNetBlock.forward is x + block1(dropout(block0(x))) (model/blocks.py:68-88); with p > 0 the dropout is
nn.Dropout(p): x * mask / (1 - p) in train mode.  The masks come from the device run (ResNetBlock.dropout_mask), so that
both sides drop the same elements; `unpack_mask` turns the device bitmask into the oracle's bool [B, C, X, Y, Z]."""
from __future__ import annotations

from functools import partial
from typing import Dict, Optional, Tuple
from unittest import mock

import numpy as np
import torch

from oracle import cgan_oracle as O

Masks = Optional[Dict[str, Tuple[torch.Tensor, float]]]  # res0 layer name -> (bool mask [B, C, X, Y, Z], p)


def unpack_mask(bits: torch.Tensor, shape_cl) -> torch.Tensor:
    """Keep bitmask (bit e & 7 of byte e >> 3 for the channels-last index e) -> bool [B, C, X, Y, Z]."""
    n = int(np.prod(shape_cl))
    flat = np.unpackbits(bits.detach().cpu().numpy(), bitorder="little")[:n].astype(bool)
    return torch.from_numpy(flat.reshape(shape_cl)).permute(0, 4, 1, 2, 3).contiguous()


def generator_forward(params, buffers, x, layers=None, train: bool = True, dropout: Masks = None):
    """cgan_oracle.generator_forward with x * mask / (1 - p) applied after each res0 layer named in `dropout`."""
    layers = layers or O.generator_layers()
    skip = None
    for l in layers:
        if l["kind"] == "res0":
            skip = x
        x = O._conv_block(x, l, params, buffers, train)
        if l["kind"] == "res0" and dropout and l["name"] in dropout:
            m, p = dropout[l["name"]]
            x = x * m.to(x.dtype) / (1 - p)
        if l["kind"] == "res1":
            x = skip + x
    return x


def train_step(st: O.StepState, opt, low, high, mask_low, mask_high, iteration: int, dropout: Masks = None, **kw):
    """cgan_oracle.train_step whose generator pass applies the given dropout masks."""
    with mock.patch.object(O, "generator_forward", partial(generator_forward, dropout=dropout)):
        return O.train_step(st, opt, low, high, mask_low, mask_high, iteration, **kw)
