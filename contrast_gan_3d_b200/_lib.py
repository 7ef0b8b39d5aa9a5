"""ctypes binding of libcgan3d.so (the C ABI declared in include/cgan3d.h).

The library is mandatory: there is no CPU or ATen fallback for the hot path.  Loading
fails loudly (ImportError) when the shared object is missing and cannot be built.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libcgan3d.so"

F32, BF16 = 0, 1
ACT_NONE, ACT_RELU, ACT_LRELU, ACT_TANH = 0, 1, 2, 3
OP_GATHER, OP_SCATTER, OP_WGRAD = 0, 1, 2
IMPL_AUTO, IMPL_GENERIC, IMPL_TC = 0, 1, 2


class ConvGeom(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("B", "Xb", "Yb", "Zb", "Cb", "Xs", "Ys", "Zs", "Cs", "k", "stride", "pad")]

    def key(self):
        return tuple(getattr(self, n) for n, _ in self._fields_)


BORDER_CONSTANT, BORDER_NEAREST = 0, 1
SPATIAL_TRANSFORM, SPATIAL_ELASTIC = 1, 2


class SpatialParams(C.Structure):
    """cgan3d_spatial_params_t: per-sample record of cgan3d_spatial_resample."""
    _fields_ = [("flags", C.c_int32), ("coef_slot", C.c_int32), ("field_slot", C.c_int32), ("shift", C.c_int32 * 3),
                ("A", C.c_float * 9), ("ctr", C.c_float * 3)]


class Cgan3dError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libcgan3d error {code}: {msg}")
        self.code = code


_vp, _i, _i64, _f, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t
_G = C.POINTER(ConvGeom)

# name -> (restype, argtypes).  Every symbol of include/cgan3d.h must appear here (tested).
SIGNATURES = {
    "cgan3d_version": (_i, []),
    "cgan3d_last_error": (C.c_char_p, []),
    "cgan3d_capabilities": (C.c_uint32, []),
    "cgan3d_device_supports_tc": (_i, []),
    "cgan3d_pack_weights": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "cgan3d_conv_workspace_bytes": (_sz, [_G, _i, _i]),
    "cgan3d_conv_gather": (_i, [_G, _i, _vp, _vp, _vp, _vp, _vp, _sz, _i, _vp]),
    "cgan3d_conv_scatter": (_i, [_G, _i, _vp, _vp, _vp, _vp, _vp, _sz, _i, _vp]),
    "cgan3d_conv_wgrad": (_i, [_G, _i, _vp, _vp, _vp, _f, _vp, _sz, _i, _vp]),
    "cgan3d_conv_select": (_i, [_G, _i, _i]),
    "cgan3d_conv_fuses_bnstats": (_i, [_G, _i, _i]),
    "cgan3d_conv_bnstats": (_i, [_G, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "cgan3d_reflect_pad": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "cgan3d_reflect_pad_backward": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "cgan3d_bn_stats": (_i, [_vp, _i, _i64, _i, _vp, _vp]),
    "cgan3d_bn_finalize": (_i, [_vp, _i64, _i, _f, _f, _vp, _vp, _vp, _vp, _vp]),
    "cgan3d_bn_eval_params": (_i, [_vp, _vp, _i, _f, _vp, _vp]),
    "cgan3d_bn_apply": (_i, [_vp, _vp, _i, _i64, _i, _vp, _vp, _vp, _i, _f, _vp, _vp]),
    "cgan3d_bn_apply_pad": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _i, _f, _i, _vp]),
    "cgan3d_bn_backward_reduce": (_i, [_vp, _vp, _i, _i64, _i, _vp, _vp, _vp, _i, _f, _vp, _vp]),
    "cgan3d_bn_backward_apply": (_i, [_vp, _vp, _vp, _i, _i64, _i, _vp, _vp, _vp, _i, _f, _vp, _vp, _vp, _f, _vp]),
    "cgan3d_bn_apply_dropout": (_i, [_vp, _vp, _vp, _i, _i64, _i, _vp, _vp, _vp, _i, _f, _f, _vp, _vp]),
    "cgan3d_bn_backward_reduce_dropout": (_i, [_vp, _vp, _vp, _i, _i64, _i, _vp, _vp, _vp, _i, _f, _f, _vp, _vp]),
    "cgan3d_bn_backward_apply_dropout": (_i, [_vp, _vp, _vp, _vp, _i, _i64, _i, _vp, _vp, _vp, _i, _f, _f, _vp, _vp, _vp, _f, _vp]),
    "cgan3d_bias_act": (_i, [_vp, _vp, _i, _i64, _i, _vp, _i, _f, _vp]),
    "cgan3d_bias_act_backward": (_i, [_vp, _vp, _vp, _i, _i64, _i, _vp, _i, _f, _vp, _vp]),
    "cgan3d_col_sums": (_i, [_vp, _i, _i64, _i, _vp, _vp]),
    "cgan3d_sums_to_f32": (_i, [_vp, _vp, _i, _f, _f, _vp]),
    "cgan3d_tanh_residual": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i64, _vp]),
    "cgan3d_tanh_residual_backward": (_i, [_vp, _vp, _vp, _vp, _i, _i64, _vp, _vp]),
    "cgan3d_cast": (_i, [_vp, _i, _vp, _i, _i64, _vp]),
    "cgan3d_axpy": (_i, [_vp, _vp, _i, _i64, _vp]),
    "cgan3d_gen_loss_sums": (_i, [_vp, _vp, _vp, _i64, _f, _f, _vp, _vp]),
    "cgan3d_gen_loss_finalize": (_i, [_vp, _i64, _f, _f, _vp, _vp, _vp]),
    "cgan3d_gen_loss_backward": (_i, [_vp, _vp, _vp, _i64, _f, _f, _vp, _vp, _vp, _vp, _vp]),
    "cgan3d_mean": (_i, [_vp, _i, _i64, _f, _vp, _vp, _vp]),
    "cgan3d_fill": (_i, [_vp, _i, _i64, _vp, _f, _vp]),
    "cgan3d_adam_step": (_i, [_vp, _vp, _vp, _vp, _i64, _f, _f, _f, _f, _i, _f, _vp]),
    "cgan3d_adam_step_multi": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _f, _f, _f, _f, _i, _f, _vp]),
    "cgan3d_adam_tick": (_i, [_vp, _vp]),
    "cgan3d_adam_step_multi_dev": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _vp, _f, _f, _f, _f, _vp]),
    "cgan3d_rmsprop_step_multi": (_i, [_i, _vp, _vp, _vp, _vp, _f, _f, _f, _f, _vp]),
    "cgan3d_crop_scale": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _f, _vp, _vp, _vp]),
    "cgan3d_scale_i16": (_i, [_vp, _vp, _i64, _f, _f, _vp]),
    "cgan3d_tile_extract": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _f, _vp, _vp]),
    "cgan3d_tile_accumulate": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "cgan3d_tile_finalize": (_i, [_vp, _vp, _vp, _i64, _f, _f, _vp]),
    "cgan3d_sub_resized": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "cgan3d_elastic_noise": (_i, [_i, _i, _i, _i, _vp, _vp, _vp]),
    "cgan3d_elastic_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "cgan3d_elastic_field": (_i, [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "cgan3d_spline_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "cgan3d_spline_prefilter": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _vp, _sz, _vp]),
    "cgan3d_spatial_resample": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _f, _i, _vp, _vp, _vp]),
}

_lib = None
launch_count = 0  # number of library entry-point calls that enqueue at least one kernel (bench: gpu_launches)


def _ensure_built() -> Path:
    """Path of an up-to-date libcgan3d.so.  The library is git-ignored and travels separately from the sources, so an
    existing file is only trusted when its build stamp equals the digest of the current csrc/ + cgan3d.h (a stale binary
    would be called through ctypes signatures that no longer match its ABI).  With nvcc present a mismatch triggers a
    rebuild; without nvcc it is an error."""
    from . import build as _build

    if os.environ.get("CGAN3D_REBUILD"):
        return _build.build(force=True)
    if LIB_PATH.exists() and _build.is_current():
        return LIB_PATH
    if _build.have_nvcc():
        return _build.build()  # a no-op when the stamp matches
    if LIB_PATH.exists():
        raise RuntimeError(f"{LIB_PATH} does not match the sources (build stamp != source digest) and nvcc is not available "
                           f"to rebuild it")
    raise RuntimeError(f"{LIB_PATH} is missing and nvcc is not available")


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        try:
            path = _ensure_built()
            _lib = C.CDLL(str(path))
        except Exception as e:  # no fallback by design
            raise ImportError(f"libcgan3d.so is required (build with `python -m contrast_gan_3d_b200.build`): {e}") from e
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(_lib, name)
            fn.restype = res
            fn.argtypes = args
    return _lib


def last_error() -> str:
    return lib().cgan3d_last_error().decode(errors="replace")


def call(name: str, *args):
    """Invoke an int-returning entry point; raise Cgan3dError on failure."""
    global launch_count
    rc = getattr(lib(), name)(*args)
    if rc != 0:
        raise Cgan3dError(rc, last_error())
    launch_count += 1
    return rc
