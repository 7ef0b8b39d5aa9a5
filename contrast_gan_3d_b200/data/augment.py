"""batchgenerators' SpatialTransform_2 (the reference's training augmentation, experiments/basic_conf.py:88-106) on the
device: elastic deformation, rotation, scaling and the random-shift crop of `augment_spatial_2`.

Every scalar is drawn on the host from the legacy numpy stream in batchgenerators' order (tests/augment_oracle.py
restates it).  The device then runs three stages of csrc/augment.cu: elastic offset fields for the samples that drew
elastic deformation, cubic B-spline coefficients of every transformed sample, and one resampling launch for the batch.
The per-sample parameters and smoothing taps travel in one pinned host-to-device copy.

Deliberate divergence from upstream: the uniform noise of the elastic fields does not come from legacy `np.random`.
Upstream draws 3 x P^3 doubles there (6.3 M per sample at 128^3, tens of ms of host time); here each elastic sample
draws one 64-bit seed from `noise_rng`, a numpy Generator owned by the transform, and the device expands it with
Philox4x32-10.  The legacy stream therefore sees exactly the scalar draws of upstream, but elastic fields differ from
upstream's for the same legacy seed.

Supported: 3-D patches, data order 3 with border mode `nearest` (upstream's default) or `constant`, seg order 0 with
border mode `constant`.  Anything else raises NotImplementedError."""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import numpy as np
import torch

from .. import ops
from .._lib import (BORDER_CONSTANT, BORDER_NEAREST, SPATIAL_ELASTIC, SPATIAL_TRANSFORM, SpatialParams, call, lib)

_MODES = {"constant": BORDER_CONSTANT, "nearest": BORDER_NEAREST}


def gaussian_taps(n: int, sigma: float) -> np.ndarray:
    """Periodic taps h with circular_conv(x, h) == ifft(fourier_gaussian(fft(x), sigma)).real along one axis of n."""
    return np.fft.ifft(np.exp(-2.0 * np.pi ** 2 * float(sigma) ** 2 * np.fft.fftfreq(n) ** 2)).real


def rotation_matrix(a_x: float, a_y: float, a_z: float) -> np.ndarray:
    """batchgenerators rotate_coords_3d: coords -> R^T coords with R = Rx(a_x) Ry(a_y) Rz(a_z)."""
    cx, sx, cy, sy, cz, sz = np.cos(a_x), np.sin(a_x), np.cos(a_y), np.sin(a_y), np.cos(a_z), np.sin(a_z)
    rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    return rx @ ry @ rz


def _align(n: int, a: int = 16) -> int:
    return (n + a - 1) // a * a


class SpatialTransform2:
    """Keyword arguments and defaults of batchgenerators' SpatialTransform_2.  `__call__` takes and returns the sampler's
    {"data": f32 [B,1,*S], "seg": bool [B,1,*S], "name", "path"} dict of CUDA tensors (other keys pass through) and
    enqueues on the current stream; the result has spatial shape `patch_size`."""

    def __init__(self, patch_size: Sequence[int], patch_center_dist_from_border=30, do_elastic_deform=True,
                 deformation_scale=(0, 0.25), do_rotation=True, angle_x=(0, 2 * np.pi), angle_y=(0, 2 * np.pi),
                 angle_z=(0, 2 * np.pi), do_scale=True, scale=(0.75, 1.25), border_mode_data="nearest",
                 border_cval_data=0, order_data=3, border_mode_seg="constant", border_cval_seg=0, order_seg=0,
                 random_crop=True, p_el_per_sample=1, p_scale_per_sample=1, p_rot_per_sample=1,
                 independent_scale_for_each_axis=False, p_rot_per_axis: float = 1,
                 p_independent_scale_per_axis: int = 1, noise_rng: Optional[np.random.Generator] = None):
        if len(patch_size) != 3:
            raise NotImplementedError("SpatialTransform2: only 3-D patches are supported")
        if order_data != 3 or border_mode_data not in _MODES:
            raise NotImplementedError(f"SpatialTransform2: data order {order_data} / border mode {border_mode_data!r} "
                                      f"(order 3 with 'nearest' or 'constant' only)")
        if order_seg != 0 or border_mode_seg != "constant":
            raise NotImplementedError(f"SpatialTransform2: seg order {order_seg} / border mode {border_mode_seg!r} "
                                      f"(order 0 with 'constant' only)")
        self.patch_size = tuple(int(p) for p in patch_size)
        pcdb = patch_center_dist_from_border
        self.pcdb = list(pcdb) if isinstance(pcdb, (list, tuple, np.ndarray)) else 3 * [pcdb]
        self.do_elastic_deform, self.deformation_scale = do_elastic_deform, deformation_scale
        self.do_rotation, self.angles = do_rotation, (angle_x, angle_y, angle_z)
        self.do_scale, self.scale = do_scale, scale
        self.border_mode_data, self.border_cval_data = border_mode_data, float(border_cval_data)
        self.border_cval_seg = border_cval_seg
        self.random_crop = random_crop
        self.p_el, self.p_scale, self.p_rot = p_el_per_sample, p_scale_per_sample, p_rot_per_sample
        self.independent_scale_for_each_axis = independent_scale_for_each_axis
        self.p_rot_per_axis, self.p_independent_scale_per_axis = p_rot_per_axis, p_independent_scale_per_axis
        self.noise_rng = noise_rng if noise_rng is not None else np.random.default_rng()

    def draw(self, batch_size: int, rs=np.random, shape: Optional[Sequence[int]] = None) -> List[dict]:
        """Per-sample parameters, drawn from `rs` in augment_spatial_2's order for inputs of spatial `shape` (default:
        the patch size).  Keys as the oracle records them, plus `seed` for elastic samples (from `noise_rng`)."""
        patch = self.patch_size
        shape = tuple(shape) if shape is not None else patch
        out = []
        for _ in range(batch_size):
            rec = {"elastic": False, "rotation": False, "scale": False}
            if rs.uniform() < self.p_el and self.do_elastic_deform:
                def_scale = rs.uniform(self.deformation_scale[0], self.deformation_scale[1])
                sigmas = [def_scale * p for p in patch]
                mags = [rs.uniform(s / 8, s / 2) for s in sigmas]
                rec.update(elastic=True, sigmas=sigmas, mags=mags,
                           seed=int(self.noise_rng.integers(0, 2 ** 64, dtype=np.uint64)))
            if rs.uniform() < self.p_rot and self.do_rotation:
                angles = tuple(rs.uniform(a[0], a[1]) if rs.uniform() <= self.p_rot_per_axis else 0
                               for a in self.angles)
                rec.update(rotation=True, angles=angles)
            if rs.uniform() < self.p_scale and self.do_scale:
                lo, hi = self.scale

                def one():
                    return rs.uniform(lo, 1) if rs.random() < 0.5 and lo < 1 else rs.uniform(max(lo, 1), hi)

                if self.independent_scale_for_each_axis and rs.uniform() < self.p_independent_scale_per_axis:
                    sc = [one() for _ in range(3)]
                else:
                    sc = one()
                rec.update(scale=True, sc=sc)
            if rec["elastic"] or rec["rotation"] or rec["scale"]:
                rec["ctr"] = [rs.uniform(self.pcdb[d], shape[d] - self.pcdb[d]) if self.random_crop
                              else shape[d] / 2.0 - 0.5 for d in range(3)]
            elif self.random_crop:
                margin = [self.pcdb[d] - patch[d] // 2 for d in range(3)]
                rec["lbs"] = [int(rs.randint(margin[d], shape[d] - patch[d] - margin[d]))
                              if shape[d] - patch[d] - margin[d] > margin[d] else (shape[d] - patch[d]) // 2
                              for d in range(3)]
            else:
                rec["lbs"] = [(shape[d] - patch[d]) // 2 for d in range(3)]
            out.append(rec)
        return out

    def __call__(self, batch: dict, rs=np.random) -> dict:
        data, seg = batch["data"], batch["seg"]
        if (not data.is_cuda or data.dtype != torch.float32 or data.dim() != 5 or data.shape[1] != 1
                or seg is None or seg.shape != data.shape or seg.dtype != torch.bool):
            raise ValueError("SpatialTransform2: data must be CUDA float32 [B,1,X,Y,Z] with a bool seg of that shape")
        draws = self.draw(data.shape[0], rs, tuple(data.shape[2:]))
        out = self.apply(data, seg, draws)
        res = dict(batch)
        res["data"], res["seg"] = out
        return res

    def apply(self, data: torch.Tensor, seg: torch.Tensor, draws: List[dict]):
        """Run the device stages for already drawn parameters; returns (data f32, seg bool) [B,1,*patch]."""
        B, S, P = data.shape[0], tuple(int(s) for s in data.shape[2:]), self.patch_size
        dev = data.device
        el = [i for i, r in enumerate(draws) if r["elastic"]]
        tf = [i for i, r in enumerate(draws) if "ctr" in r]
        ntap = sum(P)
        params = (SpatialParams * B)()
        for i, r in enumerate(draws):
            p = params[i]
            if "ctr" in r:
                p.flags = SPATIAL_TRANSFORM | (SPATIAL_ELASTIC if r["elastic"] else 0)
                p.coef_slot = tf.index(i)
                p.field_slot = el.index(i) if r["elastic"] else -1
                a = rotation_matrix(*r["angles"]).T if r["rotation"] else np.identity(3)
                if r["scale"]:
                    a = np.diag(np.broadcast_to(np.asarray(r["sc"], dtype=float), (3,))) @ a
                p.A[:] = [float(v) for v in a.reshape(-1)]
                p.ctr[:] = [float(v) for v in r["ctr"]]
            else:
                p.flags, p.coef_slot, p.field_slot = 0, -1, -1
                p.shift[:] = r["lbs"]
        # one pinned upload: [params | samples i32 | seeds u64 | mags f64 | taps f64]
        o_smp = _align(C.sizeof(params))
        o_seed = _align(o_smp + 4 * len(tf))
        o_mag = _align(o_seed + 8 * len(el))
        o_tap = _align(o_mag + 24 * len(el))
        nbytes = o_tap + 8 * ntap * len(el)
        host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
        hv = host.numpy()
        C.memmove(hv.ctypes.data, C.addressof(params), C.sizeof(params))
        hv[o_smp:o_smp + 4 * len(tf)].view(np.int32)[:] = tf
        if el:
            hv[o_seed:o_seed + 8 * len(el)].view(np.uint64)[:] = [draws[i]["seed"] for i in el]
            hv[o_mag:o_mag + 24 * len(el)].view(np.float64)[:] = np.array([draws[i]["mags"] for i in el]).reshape(-1)
            taps = hv[o_tap:o_tap + 8 * ntap * len(el)].view(np.float64).reshape(len(el), ntap)
            for j, i in enumerate(el):
                taps[j] = np.concatenate([gaussian_taps(n, s) for n, s in zip(P, draws[i]["sigmas"])])
        dbuf = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        dbuf.copy_(host, non_blocking=True)
        base = dbuf.data_ptr()
        st = ops._st()
        field = sums = None
        if el:
            field = torch.empty((len(el), 3, *P), dtype=torch.float32, device=dev)
            sums = torch.empty((len(el), 3), dtype=torch.float64, device=dev)
            wsb = lib().cgan3d_elastic_workspace_bytes(len(el), *P)
            ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
            call("cgan3d_elastic_field", len(el), *P, base + o_seed, base + o_mag, base + o_tap, field.data_ptr(),
                 sums.data_ptr(), ws.data_ptr(), wsb, st)
        mode = _MODES[self.border_mode_data]
        coef = None
        if tf:
            cb = lib().cgan3d_spline_workspace_bytes(len(tf), *S, mode)
            coef = torch.empty(cb, dtype=torch.uint8, device=dev)
            call("cgan3d_spline_prefilter", data.data_ptr(), *S, len(tf), base + o_smp, mode, coef.data_ptr(), cb, st)
        out = torch.empty((B, 1, *P), dtype=torch.float32, device=dev)
        out_seg = torch.empty((B, 1, *P), dtype=torch.uint8, device=dev)
        seg_u8 = seg.contiguous().view(torch.uint8)
        call("cgan3d_spatial_resample", data.contiguous().data_ptr(), seg_u8.data_ptr(), B, *S, *P, base,
             field.data_ptr() if field is not None else None, sums.data_ptr() if sums is not None else None,
             coef.data_ptr() if coef is not None else None, mode, self.border_cval_data,
             int(self.border_cval_seg >= 0.5), out.data_ptr(), out_seg.data_ptr(), st)
        return out, out_seg.view(torch.bool)
