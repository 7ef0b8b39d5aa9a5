"""NumPy / SciPy restatement of batchgenerators' `augment_spatial_2` [upstream, unpinned], the spatial stage of the
reference's training input pipeline (SpatialTransform_2, reference experiments/basic_conf.py:88-106).  It is the
checker for contrast_gan_3d_b200.data.augment and is never shipped or measured.

It calls the SciPy primitives batchgenerators calls: `map_coordinates` (prefilter=True) for the resampling and
`fourier_gaussian` on `np.fft.fftn` output for the elastic fields.  The draw order follows batchgenerators 0.25 from
its source as recalled, not checked against an installed upstream.  The reference runs this transform in 4 worker
processes per loader, each with its own RNG state, so its draw stream cannot be reproduced anyway: what is pinned is
this restatement, against which the device pipeline is tested.

One parameter upstream lacks: `noise_fn(shape)` supplies the uniform [0, 1) noise of each elastic field (upstream:
`np.random.random`, the default here).  The device pipeline draws that noise from a counter-based generator instead of
the legacy numpy stream; tests pass its values in through `noise_fn`."""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence

import numpy as np
from scipy.ndimage import fourier_gaussian, map_coordinates


def create_zero_centered_coordinate_mesh(shape: Sequence[int]) -> np.ndarray:
    tmp = tuple(np.arange(i) for i in shape)
    coords = np.array(np.meshgrid(*tmp, indexing="ij")).astype(float)
    for d in range(len(shape)):
        coords[d] -= ((np.array(shape).astype(float) - 1) / 2.0)[d]
    return coords


def smooth_noise(noise01: np.ndarray, sigmas: Sequence[float]) -> np.ndarray:
    """One unnormalised elastic field: ifftn(fourier_gaussian(fftn(noise * 2 - 1), sigmas)).real."""
    return np.fft.ifftn(fourier_gaussian(np.fft.fftn(noise01 * 2 - 1), sigmas)).real


def elastic_deform_coordinates_2(coords: np.ndarray, sigmas, magnitudes, noise_fn: Callable) -> np.ndarray:
    offsets = []
    for d in range(len(coords)):
        field = smooth_noise(noise_fn(coords.shape[1:]), sigmas)
        mx = np.max(np.abs(field))
        offsets.append(field / (mx / (magnitudes[d] + 1e-8)))
    return np.array(offsets) + coords


def rotation_matrix_3d(angle_x: float, angle_y: float, angle_z: float) -> np.ndarray:
    cx, sx, cy, sy, cz, sz = (np.cos(angle_x), np.sin(angle_x), np.cos(angle_y), np.sin(angle_y), np.cos(angle_z),
                              np.sin(angle_z))
    rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    return np.identity(3) @ rx @ ry @ rz


def rotate_coords_3d(coords: np.ndarray, angle_x: float, angle_y: float, angle_z: float) -> np.ndarray:
    rot = rotation_matrix_3d(angle_x, angle_y, angle_z)
    return np.dot(coords.reshape(len(coords), -1).transpose(), rot).transpose().reshape(coords.shape)


def crop_zero_filled(vol: np.ndarray, lbs: Sequence[int], size: Sequence[int]) -> np.ndarray:
    """vol[..., lb:lb+size] per spatial axis with zeros outside the volume (batchgenerators `crop`, constant 0 pad)."""
    out = np.zeros((*vol.shape[:-3], *size), dtype=vol.dtype)
    src, dst = [], []
    for lb, n, s in zip(lbs, size, vol.shape[-3:]):
        lo, hi = max(lb, 0), min(lb + n, s)
        src.append(slice(lo, max(hi, lo)))
        dst.append(slice(lo - lb, max(hi, lo) - lb))
    out[(..., *dst)] = vol[(..., *src)]
    return out


def augment_spatial_2(data: np.ndarray, seg: Optional[np.ndarray], patch_size: Sequence[int],
                      patch_center_dist_from_border=30, do_elastic_deform=True, deformation_scale=(0, 0.25),
                      do_rotation=True, angle_x=(0, 2 * np.pi), angle_y=(0, 2 * np.pi), angle_z=(0, 2 * np.pi),
                      do_scale=True, scale=(0.75, 1.25), border_mode_data="nearest", border_cval_data=0, order_data=3,
                      border_mode_seg="constant", border_cval_seg=0, order_seg=0, random_crop=True, p_el_per_sample=1,
                      p_scale_per_sample=1, p_rot_per_sample=1, independent_scale_for_each_axis=False,
                      p_rot_per_axis: float = 1, p_independent_scale_per_axis: int = 1,
                      noise_fn: Callable = None, record: Optional[List[dict]] = None):
    """data [B, C, X, Y, Z] float, seg [B, C, X, Y, Z] binary or None -> (data float32 [B, C, *patch], seg bool or None).
    With `record` a list, one dict of the sample's drawn parameters (and its sampling coordinates) is appended per
    sample."""
    if noise_fn is None:
        noise_fn = lambda s: np.random.random(s)  # noqa: E731
    patch_size = tuple(int(p) for p in patch_size)
    dim = len(patch_size)
    assert dim == 3
    pcdb = (list(patch_center_dist_from_border) if isinstance(patch_center_dist_from_border, (list, tuple, np.ndarray))
            else dim * [patch_center_dist_from_border])
    data_result = np.zeros((data.shape[0], data.shape[1], *patch_size), dtype=np.float32)
    seg_result = None if seg is None else np.zeros((seg.shape[0], seg.shape[1], *patch_size), dtype=bool)
    for b in range(data.shape[0]):
        rec = {"elastic": False, "rotation": False, "scale": False}
        coords = create_zero_centered_coordinate_mesh(patch_size)
        modified = False
        if np.random.uniform() < p_el_per_sample and do_elastic_deform:
            mag, sigmas = [], []
            def_scale = np.random.uniform(deformation_scale[0], deformation_scale[1])
            for d in range(dim):
                sigmas.append(def_scale * patch_size[d])
                mag.append(np.random.uniform(sigmas[-1] / 8, sigmas[-1] / 2))
            coords = elastic_deform_coordinates_2(coords, sigmas, mag, noise_fn)
            modified = True
            rec.update(elastic=True, sigmas=sigmas, mags=mag)
        if np.random.uniform() < p_rot_per_sample and do_rotation:
            a_x = np.random.uniform(angle_x[0], angle_x[1]) if np.random.uniform() <= p_rot_per_axis else 0
            a_y = np.random.uniform(angle_y[0], angle_y[1]) if np.random.uniform() <= p_rot_per_axis else 0
            a_z = np.random.uniform(angle_z[0], angle_z[1]) if np.random.uniform() <= p_rot_per_axis else 0
            coords = rotate_coords_3d(coords, a_x, a_y, a_z)
            modified = True
            rec.update(rotation=True, angles=(a_x, a_y, a_z))
        if np.random.uniform() < p_scale_per_sample and do_scale:
            if independent_scale_for_each_axis and np.random.uniform() < p_independent_scale_per_axis:
                sc = []
                for _ in range(dim):
                    if np.random.random() < 0.5 and scale[0] < 1:
                        sc.append(np.random.uniform(scale[0], 1))
                    else:
                        sc.append(np.random.uniform(max(scale[0], 1), scale[1]))
                for d in range(dim):
                    coords[d] *= sc[d]
            else:
                if np.random.random() < 0.5 and scale[0] < 1:
                    sc = np.random.uniform(scale[0], 1)
                else:
                    sc = np.random.uniform(max(scale[0], 1), scale[1])
                coords *= sc
            modified = True
            rec.update(scale=True, sc=sc)
        if modified:
            coords -= coords.mean(axis=tuple(range(1, len(coords.shape))), keepdims=True)
            ctr = []
            for d in range(dim):
                if random_crop:
                    ctr.append(np.random.uniform(pcdb[d], data.shape[d + 2] - pcdb[d]))
                else:
                    ctr.append(data.shape[d + 2] / 2.0 - 0.5)
                coords[d] += ctr[-1]
            rec["ctr"] = ctr
            rec["coords"] = coords
            for c in range(data.shape[1]):
                data_result[b, c] = map_coordinates(data[b, c].astype(float), coords, order=order_data,
                                                    mode=border_mode_data, cval=border_cval_data)
            if seg is not None:
                for c in range(seg.shape[1]):
                    seg_result[b, c] = map_coordinates((seg[b, c] == 1).astype(float), coords, order=order_seg,
                                                       mode=border_mode_seg, cval=border_cval_seg) >= 0.5
        else:
            shape = data.shape[2:]
            if random_crop:  # batchgenerators get_lbs_for_random_crop with margins
                margin = [pcdb[d] - patch_size[d] // 2 for d in range(dim)]
                lbs = [int(np.random.randint(margin[d], shape[d] - patch_size[d] - margin[d]))
                       if shape[d] - patch_size[d] - margin[d] > margin[d] else (shape[d] - patch_size[d]) // 2
                       for d in range(dim)]
            else:
                lbs = [(shape[d] - patch_size[d]) // 2 for d in range(dim)]
            rec["lbs"] = lbs
            data_result[b] = crop_zero_filled(data[b], lbs, patch_size)
            if seg is not None:
                seg_result[b] = crop_zero_filled(seg[b], lbs, patch_size) == 1
        if record is not None:
            record.append(rec)
    return data_result, seg_result
