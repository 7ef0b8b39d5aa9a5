"""Overlapping tiles and blended stitching of the corrector on top of the CPU oracle (oracle/cgan_oracle.py).  TEST
INFRASTRUCTURE, NOT PRODUCT.

Restates in NumPy / float64 what CCTAContrastCorrector(tile_step=, blend=, eval_mode=) computes: the tile grid with a
step, the separable Gaussian importance weight (sigma = patch / 8 per axis) and the weighted blend
out(v) = sum_t w(v - o_t) c_t(v) / sum_t w(v - o_t).  With step = patch and blend "avg" it is the reference's stitching
(cgan_oracle.correct_scan_3d)."""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple, Union

import numpy as np
import torch
import torch.nn.functional as F

from oracle import cgan_oracle as O


def grid_tiles(volume_shape: Sequence[int], patch: Sequence[int],
               step: Optional[Union[int, Sequence[int]]] = None) -> List[Tuple[int, int, int]]:
    """Starts 0, step, 2 step, ... <= S - P per axis, plus S - P when the last one stops short; z fastest."""
    if step is None:
        step = patch
    if np.isscalar(step):
        step = (step,) * 3
    axes = []
    for s, p, d in zip(volume_shape, patch, step):
        a = list(range(0, s - p + 1, d))
        if a[-1] + p < s:
            a.append(s - p)
        axes.append(a)
    return [(x, y, z) for x in axes[0] for y in axes[1] for z in axes[2]]


def weights(patch: Sequence[int], blend: str) -> np.ndarray:
    """w[i, j, k] (float64): 1 for "avg"; prod_a exp(-(i_a - (p_a - 1) / 2)^2 / (2 (p_a / 8)^2)) for "gaussian"."""
    if blend == "avg":
        return np.ones(tuple(patch))
    assert blend == "gaussian", blend
    g = [np.exp(-(np.arange(p) - (p - 1) / 2.0) ** 2 / (2.0 * (p / 8.0) ** 2)) for p in patch]
    return g[0][:, None, None] * g[1][None, :, None] * g[2][None, None, :]


def blend_tiles(tiles, origins, volume_shape, patch, blend: str) -> np.ndarray:
    """Weighted average of the tiles (any array-likes [PX, PY, PZ]) at their origins, float64."""
    w = weights(patch, blend)
    acc = np.zeros(tuple(volume_shape))
    wsum = np.zeros(tuple(volume_shape))
    for (x, y, z), c in zip(origins, tiles):
        sl = np.s_[x:x + patch[0], y:y + patch[1], z:z + patch[2]]
        acc[sl] += w * np.asarray(c, dtype=np.float64)
        wsum[sl] += w
    return acc / wsum


def correct_scan_3d(params, buffers, ccta: np.ndarray, patch=(128, 128, 128), batch_size=16, step=None, blend="avg",
                    eval_mode=False, layers=None) -> torch.Tensor:
    """CCTAContrastCorrector(tile_step=step, blend=blend, eval_mode=eval_mode)(ccta, batch_size): HU, float64."""
    layers = layers or O.generator_layers()
    tiles = grid_tiles(ccta.shape, patch, step)
    corrected = []
    with torch.no_grad():
        for i in range(0, len(tiles), batch_size):
            chunk = tiles[i:i + batch_size]
            xb = torch.stack([torch.from_numpy(O.scale_hu(ccta[x:x + patch[0], y:y + patch[1], z:z + patch[2]]
                                                          .astype(np.float32)).astype(np.float32))[None]
                              for (x, y, z) in chunk])
            att = O.generator_forward(params, buffers, xb, layers, train=eval_mode is False)
            if att.shape[2:] != xb.shape[2:]:  # nn.Upsample(size=inference_patch_size), mode "nearest"
                att = F.interpolate(att, size=tuple(patch))
            corrected += [c[0].numpy() for c in xb - att]
    return torch.from_numpy(O.unscale_hu(blend_tiles(corrected, tiles, ccta.shape, patch, blend)))
