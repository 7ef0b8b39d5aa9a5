"""Whole-volume inference with the reference's class name and call signature
(reference eval/CCTAContrastCorrector.py:24-135): tile -> patch - G(patch) -> stitch -> unscale to HU.

The int16 volume is uploaded once; tiling, int16->f32 scaling, stitching and the HU unscale are device kernels: one
batched tile extraction per batch, and one stitch launch per volume that blends every corrected tile of the call (held
on the device until then: n_tiles * P^3 * 4 bytes, 268 MB for a 512 x 512 x 256 volume in disjoint 128^3 tiles).
Like the reference, the generator is NOT switched to eval mode by default: BatchNorm uses the statistics of the tiles
sharing a batch (SURVEY §8a, a14) and tiles go through in row-major (x, y, z) order.  For the same reason a generator
built with resnet_dropout_prob > 0 keeps its dropout active here: two calls on the same volume give different
corrections, and torch.manual_seed before a call reproduces it.

Seam smoothing, off by default (the reference has neither): `tile_step` < patch makes the tiles overlap, `blend=
"gaussian"` weights each tile's voxels by a Gaussian centred on the tile instead of averaging them, and `eval_mode=True`
runs the generator in eval() mode for the call (BatchNorm running statistics, no dropout), so that a tile's correction
does not depend on the tiles that share its batch."""
from __future__ import annotations

from dataclasses import dataclass, field
from numbers import Integral
from pathlib import Path
from typing import Callable, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch
from torch import Tensor, nn

from .. import _lib, ops
from .._lib import call
from ..data.Scaler import FactorZeroCenterScaler
from ..model.utils import compute_convolution_filters_shape

BLENDS = {"avg": _lib.BLEND_AVG, "gaussian": _lib.BLEND_GAUSSIAN}


def tile_steps(patch: Sequence[int], step: Optional[Union[int, Sequence[int]]] = None) -> Tuple[int, ...]:
    """Per-axis grid step: `patch` for None, an int for every axis, or one int per axis; each in 1..patch."""
    patch = tuple(int(p) for p in patch)
    if step is None:
        return patch
    if isinstance(step, Integral) and not isinstance(step, bool):
        steps = (int(step),) * len(patch)
    else:
        try:
            steps = tuple(step)
        except TypeError:
            raise ValueError(f"tile step {step!r} is neither an int nor a sequence") from None
        if len(steps) != len(patch) or not all(isinstance(s, Integral) and not isinstance(s, bool) for s in steps):
            raise ValueError(f"tile step {step!r} needs {len(patch)} ints")
        steps = tuple(int(s) for s in steps)
    if not all(1 <= s <= p for s, p in zip(steps, patch)):
        raise ValueError(f"tile step {steps} outside 1..patch {patch}")
    return steps


def grid_tiles(volume_shape: Sequence[int], patch: Sequence[int],
               step: Optional[Union[int, Sequence[int]]] = None) -> List[Tuple[int, int, int]]:
    """Tile origins of a regular grid with `step` per axis (default: step = patch, disjoint tiles), z fastest: starts
    0, step, 2 step, ... <= S - P, and S - P appended when the last of them stops short of the end (squeezed back inside
    the volume).  The device kernels (cgan3d_tile_extract_grid / cgan3d_tile_stitch) number the tiles the same way."""
    steps = tile_steps(patch, step)
    starts = []
    for s, p, d in zip(volume_shape, patch, steps):
        if s < p:
            raise ValueError(f"volume extent {s} smaller than inference patch {p}")
        a = list(range(0, s - p + 1, d))
        if a[-1] + p < s:
            a.append(s - p)
        starts.append(a)
    return [(x, y, z) for x in starts[0] for y in starts[1] for z in starts[2]]


@dataclass
class CCTAContrastCorrector:
    """The reference's corrector.  Optional seam smoothing (defaults reproduce the reference):

    tile_step: grid step per axis (int or 3 ints, 1..patch); None = patch, disjoint tiles.
    blend: "avg" or "gaussian".  Where tiles overlap, voxel v is sum_t w(v - o_t) c_t(v) / sum_t w(v - o_t) over the
        covering tiles t in ascending index, c_t = tile t's corrected values, o_t its origin.  "avg": w = 1.
        "gaussian": w = prod_a exp(-(i_a - (p_a - 1) / 2)^2 / (2 sigma_a^2)), sigma_a = p_a / 8, in fp32.  Over the
        patch sizes of this model it never reaches 0 (about 5e-11 at the corner of a 128^3 tile), so no clamp is needed.
    eval_mode: run the generator in eval() mode for the call (BatchNorm running statistics, dropout off) and restore
        every module's previous mode afterwards; each tile's correction is then independent of its batch.
    """
    model: Callable[[], nn.Module]
    scaler: FactorZeroCenterScaler
    device: torch.device
    inference_patch_size: Optional[Sequence[int]] = None
    checkpoint_path: Optional[Path] = None
    tile_step: Optional[Union[int, Sequence[int]]] = None
    blend: str = "avg"
    eval_mode: bool = False
    upsampler: Callable = field(init=False, default=None)  # nn.Upsample when the patch does not round-trip, else None

    def __post_init__(self):
        if self.blend not in BLENDS:
            raise ValueError(f"blend {self.blend!r} is not one of {sorted(BLENDS)}")
        self.model = self.model()
        if self.checkpoint_path is not None:
            self.load_model(self.checkpoint_path)
        self.model = self.model.to(self.device)
        self.correct_scan = self.correct_scan_3D  # the reference's dispatch attribute (CCTAContrastCorrector.py:39-41)
        if self.inference_patch_size is None or len(self.inference_patch_size) < 3:
            raise NotImplementedError("2D slice-wise correction is outside the B200 hot path (SURVEY §8f rank 4)")
        self._steps = tile_steps(self.inference_patch_size, self.tile_step)
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

    def _upload(self, ccta) -> Tensor:
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
        return vol

    def _stitch(self, ccta, batch_size: int, to_hu: bool) -> Tensor:
        """Corrects every grid tile, a batch per generator pass, and blends them into one [X, Y, Z] fp32 volume (HU with
        to_hu, else network units).  The corrected batches stay on the device until the single stitch launch."""
        vol = self._upload(ccta)
        X, Y, Z = vol.shape
        P = tuple(int(p) for p in self.inference_patch_size)
        n = len(grid_tiles((X, Y, Z), P, self._steps))
        shift, factor = float(self.scaler.shift), float(self.scaler.factor)
        st = ops._st
        modes = [(m, m.training) for m in self.model.modules()]
        if self.eval_mode:
            self.model.eval()
        try:
            batches = []
            for t0 in range(0, n, batch_size):
                xb = torch.empty((min(batch_size, n - t0), 1, *P), dtype=torch.float32, device=self.device)
                call("cgan3d_tile_extract_grid", vol.data_ptr(), X, Y, Z, *P, *self._steps, t0, xb.shape[0], shift, factor,
                     xb.data_ptr(), st())
                corrected = self._corrected(xb)
                assert corrected.is_contiguous() and corrected.shape == xb.shape, corrected.shape
                batches.append(corrected)
        finally:
            for m, training in modes:
                m.training = training
        tile_bytes = 4 * int(np.prod(P))
        ptrs = np.concatenate([b.data_ptr() + tile_bytes * np.arange(b.shape[0], dtype=np.int64) for b in batches])
        table = torch.from_numpy(ptrs).pin_memory().to(self.device, non_blocking=True)
        out = torch.empty((X, Y, Z), dtype=torch.float32, device=self.device)
        call("cgan3d_tile_stitch", table.data_ptr(), n, X, Y, Z, *P, *self._steps, BLENDS[self.blend], int(to_hu), shift,
             factor, out.data_ptr(), st())
        return out

    @torch.no_grad()
    def correct_scan_3D(self, ccta, batch_size: int, desc: Optional[str] = None) -> Tensor:
        """The corrected scan in NETWORK units, [1, W, H, D] on the device (= the reference's aggregator.get_output(),
        CCTAContrastCorrector.py:60-81)."""
        return self._stitch(ccta, batch_size, to_hu=False).unsqueeze(0)

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
        out = self._stitch(ccta, batch_size, to_hu=True)
        # a FRESH page-locked tensor per call (like the reference's `.cpu()` result, the caller owns it): torch's caching host
        # allocator hands the block of an earlier, released result back without a new cudaHostAlloc, so there is no
        # 268 MB host-side clone on the path
        host = torch.empty(out.shape, dtype=out.dtype, pin_memory=True)
        host.copy_(out, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return host

    @classmethod
    def from_checkpoint(cls, inference_patch_size, device, checkpoint_path, generator_class=None, scaler=None,
                        tile_step=None, blend: str = "avg", eval_mode: bool = False):
        if generator_class is None:
            from ..experiments.b200_conf import generator_class
        return cls(generator_class, scaler or FactorZeroCenterScaler(-1024, 1500, 600), device,
                   inference_patch_size=inference_patch_size, checkpoint_path=checkpoint_path, tile_step=tile_step,
                   blend=blend, eval_mode=eval_mode)
