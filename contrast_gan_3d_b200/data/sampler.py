"""Patch sampler: the crop / pad index law of reference data/CCTADataLoader.py:76-108 (which delegates to
batchgenerators `pad_nd_image` + `crop(crop_type="random")`), with the pad + crop + int16->f32 + HU scaling
done by one device kernel per patch instead of a whole-volume float copy on CPU workers.  An optional `transform`
(data.augment.SpatialTransform2, the reference's SpatialTransform_2) is applied to each batch after its crops.

The integer index math is host-side Python and bit-exact with the oracle restatement; volumes are int16
[W, H, D, 2] (HU, centerline mask)."""
from __future__ import annotations

from typing import List, Sequence, Tuple

import numpy as np
import torch

from .. import ops
from .._lib import call
from .Scaler import FactorZeroCenterScaler


def pad_amounts(shape: Sequence[int], patch: Sequence[int]) -> List[Tuple[int, int]]:
    """Symmetric zero padding up to the patch size: below = d // 2, above = d // 2 + d % 2."""
    out = []
    for s, p in zip(shape, patch):
        d = max(p - s, 0)
        out.append((d // 2, d // 2 + d % 2))
    return out


def random_crop_lower_bounds(padded_shape: Sequence[int], patch: Sequence[int], rs=np.random) -> List[int]:
    """Per axis in W, H, D order: `randint(0, dim - size)` (high exclusive) when dim > size else (dim - size) // 2,
    drawn from the legacy global numpy RNG exactly as batchgenerators does."""
    lbs = []
    for d, c in zip(padded_shape, patch):
        lbs.append(int(rs.randint(0, d - c)) if d - c > 0 else (d - c) // 2)
    return lbs


class DevicePatchSampler:
    """Samples batches {"data": f32 [B,1,*patch], "seg": bool [B,1,*patch], "name", "path"} like
    CCTADataLoader.generate_train_batch, from device-resident int16 volumes.  With a `transform`, the batch passes
    through it after all its crops are drawn (the reference's loader-then-augmenter order), drawing from the same `rs`."""

    def __init__(self, volumes: List[torch.Tensor], patch_shape: Sequence[int], batch_size: int,
                 scaler: FactorZeroCenterScaler = None, names: List[str] = None, rs=np.random, transform=None):
        for v in volumes:
            if v.dtype != torch.int16 or v.dim() != 4 or v.shape[-1] != 2 or not v.is_cuda:
                raise ValueError("volumes must be CUDA int16 tensors [W, H, D, 2]")
        self.volumes = [v.contiguous() for v in volumes]
        self.patch = tuple(int(p) for p in patch_shape)
        self.batch_size = batch_size
        self.scaler = scaler or FactorZeroCenterScaler(-1024, 1500, 600)
        self.names = names or [f"vol{i}" for i in range(len(volumes))]
        self.rs = rs
        self.transform = transform

    def get_indices(self) -> np.ndarray:
        # batchgenerators DataLoader.get_indices with infinite=True
        return self.rs.choice(len(self.volumes), self.batch_size, replace=True)

    def sample_one(self, vol: torch.Tensor, data_out: torch.Tensor, mask_out: torch.Tensor) -> List[int]:
        X, Y, Z = vol.shape[:3]
        padded = [max(a, b) for a, b in zip((X, Y, Z), self.patch)]
        lbs = random_crop_lower_bounds(padded, self.patch, self.rs)
        call("cgan3d_crop_scale", vol.data_ptr(), X, Y, Z, *lbs, *self.patch, float(self.scaler.shift),
             float(self.scaler.factor), data_out.data_ptr(), mask_out.data_ptr(), ops._st())
        return lbs

    def generate_train_batch(self) -> dict:
        dev = self.volumes[0].device
        data = torch.empty((self.batch_size, 1, *self.patch), dtype=torch.float32, device=dev)
        seg = torch.empty((self.batch_size, 1, *self.patch), dtype=torch.uint8, device=dev)
        names, lbs = [], []
        for i, idx in enumerate(self.get_indices()):
            lbs.append(self.sample_one(self.volumes[idx], data[i], seg[i]))
            names.append(self.names[idx])
        batch = {"data": data, "seg": seg.view(torch.bool), "name": names, "path": names, "lbs": lbs}
        return batch if self.transform is None else self.transform(batch, rs=self.rs)

    def __next__(self):
        return self.generate_train_batch()

    def __iter__(self):
        return self
