"""Whole-volume inference with the reference's class name and call signature
(reference eval/CCTAContrastCorrector.py:24-135): tile -> patch - G(patch) -> stitch -> unscale to HU.

The int16 volume is uploaded once; tiling, int16->f32 scaling, stitching (average where tiles overlap) and the
HU unscale are device kernels.  Like the reference, the generator is NOT switched to eval mode: BatchNorm uses the
statistics of the tiles sharing a batch (SURVEY §8a, a14) and tiles go through in row-major (x, y, z) order.
For the same reason a generator built with resnet_dropout_prob > 0 keeps its dropout active here: two calls on the same
volume give different corrections, and torch.manual_seed before a call reproduces it."""
from __future__ import annotations

from dataclasses import dataclass, field
from pathlib import Path
from typing import Callable, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch
from torch import Tensor, nn

from .. import ops
from .._lib import call
from ..data.Scaler import FactorZeroCenterScaler
from ..model.utils import compute_convolution_filters_shape


def grid_tiles(volume_shape: Sequence[int], patch: Sequence[int]) -> List[Tuple[int, int, int]]:
    """Regular grid with step = patch, z fastest; a trailing partial tile is squeezed back inside the volume."""
    starts = []
    for s, p in zip(volume_shape, patch):
        if s < p:
            raise ValueError(f"volume extent {s} smaller than inference patch {p}")
        a = list(range(0, s - p + 1, p))
        if a[-1] + p < s:
            a.append(s - p)
        starts.append(a)
    return [(x, y, z) for x in starts[0] for y in starts[1] for z in starts[2]]


@dataclass
class CCTAContrastCorrector:
    model: Callable[[], nn.Module]
    scaler: FactorZeroCenterScaler
    device: torch.device
    inference_patch_size: Optional[Sequence[int]] = None
    checkpoint_path: Optional[Path] = None
    upsampler: Callable = field(init=False, default=None)  # nn.Upsample when the patch does not round-trip, else None

    def __post_init__(self):
        self.model = self.model()
        if self.checkpoint_path is not None:
            self.load_model(self.checkpoint_path)
        self.model = self.model.to(self.device)
        self.correct_scan = self.correct_scan_3D  # the reference's dispatch attribute (CCTAContrastCorrector.py:39-41)
        if self.inference_patch_size is None or len(self.inference_patch_size) < 3:
            raise NotImplementedError("2D slice-wise correction is outside the B200 hot path (SURVEY §8f rank 4)")
        out_shape = compute_convolution_filters_shape(self.model, (1, *self.inference_patch_size), show=False)
        # When the strided convs do not round-trip the patch size the reference resizes the attenuation map back with
        # nn.Upsample(size=inference_patch_size) (nearest) before subtracting it (CCTAContrastCorrector.py:42-52,79).
        self._att_shape = None
        if out_shape[1:] != list(self.inference_patch_size):
            self._att_shape = tuple(out_shape[1:])
            self.upsampler = nn.Upsample(size=tuple(self.inference_patch_size))  # parameter record only; see _corrected

    def load_model(self, checkpoint_path: Union[str, Path]):
        ckpt = torch.load(checkpoint_path, map_location="cpu")
        self.model.load_state_dict(ckpt["generator"])
        self.checkpoint_path = Path(checkpoint_path)

    def _corrected(self, xb: Tensor) -> Tensor:
        """patch - upsampler(G(patch)) for one batch of tiles (CCTAContrastCorrector.py:78-79)."""
        if self._att_shape is None:
            if hasattr(self.model, "forward_corrected"):
                return self.model.forward_corrected(xb)[1]
            return xb - self.model(xb)
        att = self.model(xb).contiguous()
        assert tuple(att.shape[2:]) == self._att_shape, (att.shape, self._att_shape)
        out = torch.empty_like(xb)
        call("cgan3d_sub_resized", xb.data_ptr(), att.data_ptr(), out.data_ptr(), xb.shape[0], *xb.shape[2:], *att.shape[2:],
             ops._st())
        return out

    def _accumulate(self, ccta, batch_size: int):
        if isinstance(ccta, Tensor) and not ccta.is_cuda and ccta.dtype == torch.int16 and ccta.is_pinned():
            vol = ccta.to(self.device, non_blocking=True)  # already page-locked: no staging copy
        elif isinstance(ccta, np.ndarray):
            if ccta.dtype != np.int16:
                ccta = np.rint(ccta).astype(np.int16) if np.issubdtype(ccta.dtype, np.floating) else ccta.astype(np.int16)
            # stage through a cached pinned buffer: the pageable->device path of a 134 MB volume costs several times the
            # PCIe time of the pinned copy
            host = self._pinned("in", ccta.shape, torch.int16)
            busy = self.__dict__.get("_in_copied")
            if busy is not None:
                busy.synchronize()  # the previous call's host->device copy must have left the pinned buffer
            host.numpy()[...] = ccta
            vol = host.to(self.device, non_blocking=True)
            self._in_copied = torch.cuda.Event()
            self._in_copied.record(torch.cuda.current_stream(self.device))
        else:
            vol = ccta.to(self.device).to(torch.int16).contiguous()
        X, Y, Z = vol.shape
        P = tuple(int(p) for p in self.inference_patch_size)
        tiles = grid_tiles((X, Y, Z), P)
        acc = torch.zeros((X, Y, Z), dtype=torch.float32, device=self.device)
        cnt = torch.zeros((X, Y, Z), dtype=torch.float32, device=self.device)
        st = ops._st
        for i in range(0, len(tiles), batch_size):
            chunk = tiles[i:i + batch_size]
            xb = torch.empty((len(chunk), 1, *P), dtype=torch.float32, device=self.device)
            for j, (x0, y0, z0) in enumerate(chunk):
                call("cgan3d_tile_extract", vol.data_ptr(), X, Y, Z, x0, y0, z0, *P, float(self.scaler.shift),
                     float(self.scaler.factor), xb[j].data_ptr(), st())
            corrected = self._corrected(xb)
            for j, (x0, y0, z0) in enumerate(chunk):
                call("cgan3d_tile_accumulate", corrected[j].data_ptr(), acc.data_ptr(), cnt.data_ptr(), X, Y, Z, x0, y0, z0,
                     *P, st())
        return acc, cnt

    @torch.no_grad()
    def correct_scan_3D(self, ccta, batch_size: int, desc: Optional[str] = None) -> Tensor:
        """The corrected scan in NETWORK units, [1, W, H, D] on the device (= the reference's aggregator.get_output(),
        CCTAContrastCorrector.py:60-81)."""
        acc, cnt = self._accumulate(ccta, batch_size)
        return (acc / cnt).unsqueeze(0)

    def _pinned(self, key: str, shape, dtype) -> Tensor:
        """Cached page-locked host staging tensor (allocating pinned memory costs more than the transfer itself)."""
        cache = self.__dict__.setdefault("_pinned_cache", {})
        t = cache.get(key)
        if t is None or tuple(t.shape) != tuple(shape) or t.dtype != dtype:
            t = torch.empty(tuple(shape), dtype=dtype, pin_memory=self.device.type == "cuda")
            cache[key] = t
        return t

    @torch.no_grad()
    def __call__(self, ccta, batch_size: int = 16, **kwargs) -> Tensor:
        """Corrected scan in HU on the host (a fresh tensor per call, like the reference)."""
        kwargs.pop("desc", None)
        acc, cnt = self._accumulate(ccta, batch_size)
        out = torch.empty_like(acc)
        call("cgan3d_tile_finalize", acc.data_ptr(), cnt.data_ptr(), out.data_ptr(), acc.numel(), float(self.scaler.shift),
             float(self.scaler.factor), ops._st())
        # a FRESH page-locked tensor per call (like the reference's `.cpu()` result, the caller owns it): torch's caching host
        # allocator hands the block of an earlier, released result back without a new cudaHostAlloc, so there is no
        # 268 MB host-side clone on the path
        host = torch.empty(out.shape, dtype=out.dtype, pin_memory=True)
        host.copy_(out, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return host

    @classmethod
    def from_checkpoint(cls, inference_patch_size, device, checkpoint_path, generator_class=None, scaler=None):
        if generator_class is None:
            from ..experiments.b200_conf import generator_class
        return cls(generator_class, scaler or FactorZeroCenterScaler(-1024, 1500, 600), device,
                   inference_patch_size=inference_patch_size, checkpoint_path=checkpoint_path)
