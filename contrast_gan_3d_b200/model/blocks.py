"""ConvBlock / ResNetBlock with the reference's constructor signatures, attribute names and
state_dict keys (reference model/blocks.py:4-88); forward runs on libcgan3d kernels.

`self.conv` / `self.normalization` are stock torch modules used ONLY as parameter containers
(identical default init, `.to()`, `state_dict()`); their own forward is never called.
"""
from __future__ import annotations

from typing import Optional

import torch
from torch import Tensor, nn

from .. import _lib, ops


def _act_code(activation_fn) -> int:
    if activation_fn in (nn.ReLU,):
        return _lib.ACT_RELU
    if activation_fn in (nn.LeakyReLU,):
        return _lib.ACT_LRELU
    if activation_fn in (nn.Identity,):
        return _lib.ACT_NONE
    raise NotImplementedError(f"activation {activation_fn} is not part of the hot path")


def to_channels_last(x: Tensor) -> Tensor:
    """[B, C, X, Y, Z] -> [B, X, Y, Z, C] (a free view when C == 1)."""
    if x.shape[1] == 1:
        return x.contiguous().reshape(x.shape[0], *x.shape[2:], 1)
    return x.permute(0, 2, 3, 4, 1).contiguous()


def from_channels_last(x: Tensor) -> Tensor:
    if x.shape[-1] == 1:
        return x.reshape(x.shape[0], 1, *x.shape[1:-1])
    return x.permute(0, 4, 1, 2, 3).contiguous()


class ConvBlock(nn.Module):
    def __init__(
        self,
        is_2D: bool,
        channels_in: int,
        channels_out: int,
        kernel_size: int,
        upsample: bool = False,
        output_padding: int = 0,
        padding_mode: str = "zeros",
        padding: int = 0,
        stride: int = 1,
        activation_fn: nn.Module = nn.ReLU,
        norm_layer: Optional[nn.Module] = None,
        **kwargs,
    ):
        super().__init__()
        if is_2D:
            raise NotImplementedError("2D variant (conf_2D.py) is outside the B200 hot path (SURVEY §8f rank 4)")
        if norm_layer is None:
            norm_layer = nn.BatchNorm3d
        if norm_layer not in (nn.BatchNorm3d, nn.Identity, nn.LayerNorm):
            raise NotImplementedError(f"norm layer {norm_layer} is not supported (BatchNorm3d, Identity, LayerNorm are)")
        if padding_mode not in ("zeros", "reflect"):
            raise NotImplementedError(f"padding_mode {padding_mode!r}")
        args = {}
        conv_class = nn.Conv3d
        if upsample:
            args = {"output_padding": output_padding}
            conv_class = nn.ConvTranspose3d
        self.conv = conv_class(channels_in, channels_out, kernel_size, stride=stride, bias=norm_layer == nn.Identity,
                               padding_mode=padding_mode, padding=padding, **args)
        # reference blocks.py:40-45: LayerNorm over the layer's whole output [C, W, H, D] when a patch size is given
        norm_shape, norm_args = channels_out, {}
        if norm_layer == nn.LayerNorm and (ps := kwargs.get("patch_size")):
            norm_shape = list(ps)
            if (affine := kwargs.get("elementwise_affine")) is not None:
                norm_args["elementwise_affine"] = affine
        self.normalization = norm_layer(norm_shape, **norm_args)
        activation_kwargs = {}
        self.negative_slope = 0.0
        if (ns := kwargs.get("negative_slope")) is not None:
            activation_kwargs["negative_slope"] = ns
        self.activation_fn = activation_fn(inplace=True, **activation_kwargs)
        if isinstance(self.activation_fn, nn.LeakyReLU):
            self.negative_slope = float(self.activation_fn.negative_slope)
        self.act_code = _act_code(activation_fn)
        self.spec = ops.ConvSpec(transposed=upsample, cin=channels_in, cout=channels_out, k=kernel_size, stride=stride,
                                 pad=padding, reflect=padding_mode == "reflect", out_pad=output_padding)
        self.compute_dtype = kwargs.get("compute_dtype", torch.float32)

    def forward_cl(self, x: Tensor, residual: Optional[Tensor] = None, pad_out: int = 0, dropout: float = 0.0):
        """pad_out > 0 returns the output with the reflection padding of its consumer already applied (fused into the
        normalise + activation pass); the consumer must then be told that its input is pre-padded.
        dropout = p > 0 (BatchNorm blocks) applies nn.Dropout(p) to the output in the same pass and returns
        (output, keep bitmask) (ops.ConvBlockFn)."""
        bn = self.normalization if isinstance(self.normalization, nn.BatchNorm3d) else None
        cfg = ops.BlockCfg(spec=self.spec, act=self.act_code, slope=self.negative_slope, dtype=self.compute_dtype,
                           training=self.training or (bn is not None and not bn.track_running_stats),
                           momentum=0.1 if bn is None or bn.momentum is None else bn.momentum,
                           eps=1e-5 if bn is None else bn.eps, pad_out=pad_out, dropout=dropout)
        if bn is not None:
            return ops.ConvBlockFn.apply(x, self.conv.weight, None, bn.weight, bn.bias, residual, bn.running_mean,
                                         bn.running_var, bn.num_batches_tracked, cfg)
        return ops.ConvBlockFn.apply(x, self.conv.weight, self.conv.bias, None, None, residual, None, None, None, cfg)

    def forward_cl_differentiable(self, x: Tensor) -> Tensor:
        """act(norm(conv(x))) built from the twice-differentiable conv Functions (ops.ConvGatherFn / ScatterFn / WgradFn)
        for critics WITHOUT BatchNorm (Identity or LayerNorm: the WGAN-GP configurations, reference
        experiments/gradient_penalty_conf.py:14, gp_layernorm.py:10-13).  The convolutions are libcgan3d kernels in every
        derivative order; bias / LayerNorm / LeakyReLU are plain ATen element-wise ops, which autograd differentiates twice."""
        y = ops.conv_differentiable(x, self.conv.weight, self.spec, self.compute_dtype)
        if self.conv.bias is not None:
            y = y + self.conv.bias.to(y.dtype)
        if isinstance(self.normalization, nn.LayerNorm):
            ln = self.normalization
            C = y.shape[-1]
            if tuple(ln.normalized_shape) != (C, *y.shape[1:4]):
                raise ValueError(f"LayerNorm shape {tuple(ln.normalized_shape)} does not match the layer output {(C, *y.shape[1:4])}")
            # same element set as the reference's [C, W, H, D]; affine parameters are stored in that layout
            wt = None if ln.weight is None else ln.weight.permute(1, 2, 3, 0)
            bs = None if ln.bias is None else ln.bias.permute(1, 2, 3, 0)
            y = torch.nn.functional.layer_norm(y.float(), y.shape[1:], wt, bs, ln.eps).to(y.dtype)
        elif not isinstance(self.normalization, nn.Identity):
            raise NotImplementedError("the twice-differentiable path has no BatchNorm (the reference pairs WGAN-GP with Identity / LayerNorm)")
        if self.act_code == _lib.ACT_LRELU:
            y = torch.nn.functional.leaky_relu(y, self.negative_slope)
        elif self.act_code == _lib.ACT_RELU:
            y = torch.relu(y)
        return y

    def forward(self, x: Tensor) -> Tensor:
        if isinstance(self.normalization, nn.LayerNorm):
            return from_channels_last(self.forward_cl_differentiable(to_channels_last(x)).float())
        return from_channels_last(self.forward_cl(to_channels_last(x)).float())


class ResNetBlock(nn.Module):
    """x + block1(dropout(block0(x))) (reference model/blocks.py:56-88).

    dropout_prob > 0: `self.dropout` is nn.Dropout(dropout_prob) (parameter-free: the state_dict is that of p = 0) and,
    while it is in train mode, runs fused into block0's normalise pass.  `self.dropout_mask` holds the keep bitmask of the
    last forward that drew one (uint8, bit e & 7 of byte e >> 3 for the channels-last index e of block0's output), else
    None; under a CUDA graph it is the graph's static tensor, rewritten by every replay."""

    def __init__(self, is_2D: bool, channels_in: int, channels_out: int, kernel_size: int = 3,
                 dropout_prob: float = 0.0, padding_mode: str = "zeros", **kwargs):
        super().__init__()
        padding_amount = 1
        self.block0 = ConvBlock(is_2D, channels_in, channels_out, kernel_size, padding_mode=padding_mode,
                                padding=padding_amount, activation_fn=nn.Identity, **kwargs)
        # nn.Dropout rejects p outside [0, 1] with torch's ValueError
        self.dropout = nn.Dropout(dropout_prob) if dropout_prob != 0 else nn.Identity()
        if isinstance(self.dropout, nn.Dropout) and not isinstance(self.block0.normalization, nn.BatchNorm3d):
            raise NotImplementedError("ResNet dropout is fused into block0's BatchNorm pass; blocks without BatchNorm have none")
        self.dropout_mask: Optional[Tensor] = None
        self.block1 = ConvBlock(is_2D, channels_out, channels_out, kernel_size, padding_mode=padding_mode,
                                padding=padding_amount, **kwargs)

    def forward_cl(self, x: Tensor) -> Tensor:
        # x + block1(dropout(block0(x))): the dropout is fused into block0's normalise pass, the skip add into block1's
        if isinstance(self.dropout, nn.Dropout) and self.dropout.training and self.dropout.p > 0:
            h, self.dropout_mask = self.block0.forward_cl(x, dropout=self.dropout.p)
        else:
            h = self.block0.forward_cl(x)
        return self.block1.forward_cl(h, residual=x)

    def forward(self, x: Tensor) -> Tensor:
        return from_channels_last(self.forward_cl(to_channels_last(x)).float())
