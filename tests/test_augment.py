"""SpatialTransform2 (batchgenerators SpatialTransform_2 on the device) against the NumPy / SciPy restatement in
tests/augment_oracle.py: host draws and smoothing taps on the CPU, each device stage and the sampler end to end on the
GPU."""
from __future__ import annotations

import ctypes

import numpy as np
import pytest
import torch

from contrast_gan_3d_b200 import _lib
from contrast_gan_3d_b200.data.augment import SpatialTransform2, gaussian_taps, rotation_matrix
from tests import augment_oracle as AO

DEV = "cuda:0"


def _separable_smooth(noise01: np.ndarray, sigmas) -> np.ndarray:
    x = noise01 * 2 - 1
    for ax, (n, s) in enumerate(zip(x.shape, sigmas)):
        h = gaussian_taps(n, s)
        x = sum(h[k] * np.roll(x, k, axis=ax) for k in range(n))
    return x


@pytest.mark.parametrize("shape", [(16, 16, 16), (9, 9, 9), (128, 128, 32)])
def test_separable_periodic_taps_match_fft_path(shape):
    rng = np.random.default_rng(0)
    noise = rng.random(shape)
    for scale in (0.01 / 16, 0.1, 0.25, 32 / 128):
        for sig in ([0.01, 0.01, 0.01], [scale * n for n in shape], [32.0, 32.0, 32.0]):
            ref = AO.smooth_noise(noise, sig)
            got = _separable_smooth(noise, sig)
            assert np.abs(got - ref).max() <= 1e-12 * max(1.0, np.abs(ref).max()), (shape, sig)


@pytest.mark.parametrize("mode", ["nearest", "constant"])
def test_oracle_identity_parameters_return_the_input(mode):
    rng = np.random.default_rng(1)
    data = rng.normal(size=(2, 1, 12, 10, 9))
    seg = (rng.random(data.shape) < 0.3).astype(np.float32)
    # no branch fires, centre crop of an equal shape: the identity
    d, s = AO.augment_spatial_2(data, seg, data.shape[2:], p_el_per_sample=0, p_rot_per_sample=0,
                                p_scale_per_sample=0, random_crop=False, border_mode_data=mode)
    np.testing.assert_array_equal(d, data.astype(np.float32))
    np.testing.assert_array_equal(s, seg == 1)
    # the interpolation path at the integer grid (scale 1, centred): the input to float rounding
    d, s = AO.augment_spatial_2(data, seg, data.shape[2:], do_elastic_deform=False, do_rotation=False, scale=(1, 1),
                                random_crop=False, border_mode_data=mode)
    np.testing.assert_allclose(d, data.astype(np.float32), rtol=0, atol=1e-6)
    np.testing.assert_array_equal(s, seg == 1)


DRAW_CONFIGS = [
    dict(p_el_per_sample=0.5, p_rot_per_sample=0.5, p_scale_per_sample=0.5, p_rot_per_axis=0.5,
         independent_scale_for_each_axis=True, p_independent_scale_per_axis=0.5, patch_center_dist_from_border=6),
    dict(p_el_per_sample=0.3, p_rot_per_sample=0.3, p_scale_per_sample=0.3, scale=(1.1, 1.4), random_crop=False,
         angle_x=(-0.5, 0.5), deformation_scale=(0.05, 0.2)),
]


@pytest.mark.parametrize("cfg", range(len(DRAW_CONFIGS)))
def test_draw_matches_oracle_and_leaves_the_legacy_rng_alike(cfg):
    kw = DRAW_CONFIGS[cfg]
    patch, shape, B = (8, 8, 8), (12, 11, 10), 4
    t = SpatialTransform2(patch, **kw, noise_rng=np.random.default_rng(0))
    rng = np.random.default_rng(1)
    data = rng.normal(size=(B, 1, *shape))
    seg = (rng.random(data.shape) < 0.3).astype(np.float32)
    seen = set()
    for seed in range(60):
        np.random.seed(seed)
        draws = t.draw(B, np.random, shape)
        after_draw = np.random.get_state()
        np.random.seed(seed)
        rec = []
        noise = np.random.default_rng(seed)
        AO.augment_spatial_2(data, seg, patch, **kw, noise_fn=lambda s: noise.random(s), record=rec)
        after_oracle = np.random.get_state()
        assert after_draw[0] == after_oracle[0] and after_draw[2:] == after_oracle[2:]
        np.testing.assert_array_equal(after_draw[1], after_oracle[1])
        for d, r in zip(draws, rec):
            for k, v in r.items():
                if k != "coords":
                    np.testing.assert_array_equal(np.asarray(d[k], dtype=float), np.asarray(v, dtype=float), err_msg=k)
            assert ("seed" in d) == r["elastic"]
            seen.add((r["elastic"], r["rotation"], r["scale"], isinstance(r.get("sc"), list)))
    assert {k[:3] for k in seen} == {(a, b, c) for a in (False, True) for b in (False, True) for c in (False, True)}
    if kw.get("independent_scale_for_each_axis"):
        assert any(k[3] for k in seen)


def test_unsupported_configurations_raise():
    for kw in (dict(order_data=1), dict(border_mode_data="reflect"), dict(order_seg=1), dict(border_mode_seg="nearest")):
        with pytest.raises(NotImplementedError):
            SpatialTransform2((16, 16, 16), **kw)
    with pytest.raises(NotImplementedError):
        SpatialTransform2((16, 16))
    lib = _lib.lib()
    assert lib.cgan3d_spline_prefilter(1, 16, 16, 16, 1, 1, 2, 1, 1 << 30, None) == -5
    assert lib.cgan3d_spatial_resample(1, 1, 1, 16, 16, 16, 16, 16, 16, 1, None, None, 1, 3, 0.0, 0, 1, 1, None) == -5
    assert lib.cgan3d_elastic_field(1, 16, 16, 2, 1, 1, 1, 1, 1, 1, 1 << 30, None) == -5
    assert lib.cgan3d_spline_workspace_bytes(1, 16, 16, 16, 2) == 0


# ---- GPU ---------------------------------------------------------------------------------------------------------

def _mesh(P):
    return AO.create_zero_centered_coordinate_mesh(P)


def _resample(data, seg, P, params, field, sums, mode, cval=0.0, seg_fill=0):
    """prefilter + resample of every sample of data / seg (CUDA [B, *S]) with explicit records."""
    B, S = data.shape[0], tuple(data.shape[1:])
    m = _lib.BORDER_NEAREST if mode == "nearest" else _lib.BORDER_CONSTANT
    st = torch.cuda.current_stream().cuda_stream
    samples = torch.arange(B, dtype=torch.int32, device=DEV)
    cb = _lib.lib().cgan3d_spline_workspace_bytes(B, *S, m)
    coef = torch.empty(cb, dtype=torch.uint8, device=DEV)
    _lib.call("cgan3d_spline_prefilter", data.data_ptr(), *S, B, samples.data_ptr(), m, coef.data_ptr(), cb, st)
    pbuf = torch.frombuffer(bytearray(bytes(params)), dtype=torch.uint8).to(DEV)
    out = torch.empty((B, *P), dtype=torch.float32, device=DEV)
    oseg = torch.empty((B, *P), dtype=torch.uint8, device=DEV)
    _lib.call("cgan3d_spatial_resample", data.data_ptr(), seg.data_ptr(), B, *S, *P, pbuf.data_ptr(),
              field.data_ptr(), sums.data_ptr(), coef.data_ptr(), m, float(cval), int(seg_fill), out.data_ptr(),
              oseg.data_ptr(), st)
    torch.cuda.synchronize()
    return out.cpu().numpy(), oseg.cpu().numpy()


def _near_round(c, tol):
    f = c - np.floor(c)
    return np.abs(f - 0.5) < tol


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["nearest", "constant"])
@pytest.mark.parametrize("P", [(128, 128, 128), (128, 128, 32)])
def test_prefilter_and_resample_match_scipy(mode, P):
    rng = np.random.default_rng(7)
    S = P
    data = rng.uniform(-2, 2, size=S).astype(np.float32)
    seg = (rng.random(S) < 0.3).astype(np.uint8)
    # target coordinates per axis: uniform over [-3, n+2], integers, half-integers, within 1e-3 of the edges, outside
    want = np.empty((3, *P))
    for d in range(3):
        n = S[d]
        kind = rng.integers(0, 5, size=P)
        u = rng.uniform(-3, n + 2, size=P)
        cand = [u, np.round(u), np.floor(u) + 0.5,
                np.where(rng.random(P) < 0.5, 0.0, n - 1.0) + rng.uniform(-1e-3, 1e-3, size=P),
                np.where(rng.random(P) < 0.5, -rng.uniform(0, 40, size=P), n - 1 + rng.uniform(0, 40, size=P))]
        want[d] = np.choose(kind, cand)
    mesh32 = _mesh(P).astype(np.float32)
    off32 = (want - _mesh(P)).astype(np.float32)
    c32 = mesh32 + off32  # what the device computes: mesh + offset in fp32, identity map, no centring
    params = (_lib.SpatialParams * 1)()
    params[0].flags = _lib.SPATIAL_TRANSFORM | _lib.SPATIAL_ELASTIC
    params[0].coef_slot, params[0].field_slot = 0, 0
    params[0].A[:] = [1, 0, 0, 0, 1, 0, 0, 0, 1]
    field = torch.from_numpy(off32[None]).to(DEV)
    sums = torch.zeros((1, 3), dtype=torch.float64, device=DEV)
    cval = 0.25
    got, gseg = _resample(torch.from_numpy(data[None]).to(DEV), torch.from_numpy(seg[None]).to(DEV), P, params, field,
                          sums, mode, cval=cval)
    c64 = c32.astype(np.float64)
    ref = AO.map_coordinates(data.astype(np.float64), c64, order=3, mode=mode, cval=cval)
    rseg = AO.map_coordinates(seg.astype(np.float64), c64, order=0, mode="constant", cval=0) >= 0.5
    err = np.abs(got[0] - ref).max() / np.abs(ref).max()
    print(f"prefilter+resample {mode} {P}: max|d|/max|ref| = {err:.3g}")
    assert err <= 1e-5  # 8.2e-7 measured (constant, 128^3)
    ok = ~np.any(_near_round(c64, 1e-4), axis=0)
    assert ok.mean() > 0.5
    np.testing.assert_array_equal(gseg[0][ok].astype(bool), rseg[ok])


def _elastic(seeds, P, sigmas, mags):
    n = len(seeds)
    st = torch.cuda.current_stream().cuda_stream
    sd = torch.tensor(np.array(seeds, dtype=np.uint64).view(np.int64), device=DEV)
    mg = torch.tensor(np.array(mags, dtype=np.float64), device=DEV)
    taps = torch.tensor(np.stack([np.concatenate([gaussian_taps(p, s) for p, s in zip(P, sg)]) for sg in sigmas]),
                        device=DEV)
    field = torch.empty((n, 3, *P), dtype=torch.float32, device=DEV)
    sums = torch.empty((n, 3), dtype=torch.float64, device=DEV)
    wsb = _lib.lib().cgan3d_elastic_workspace_bytes(n, *P)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    _lib.call("cgan3d_elastic_field", n, *P, sd.data_ptr(), mg.data_ptr(), taps.data_ptr(), field.data_ptr(),
              sums.data_ptr(), ws.data_ptr(), wsb, st)
    torch.cuda.synchronize()
    return field, sums


def device_noise(seed, P):
    sd = torch.tensor(np.array([seed], dtype=np.uint64).view(np.int64), device=DEV)
    out = torch.empty((1, 3, *P), dtype=torch.float32, device=DEV)
    _lib.call("cgan3d_elastic_noise", 1, *P, sd.data_ptr(), out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return out[0].cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("P", [(128, 128, 128), (128, 128, 32)])
def test_elastic_field_matches_oracle_on_device_noise(P):
    seeds = [12345, 2 ** 63 + 7]
    sigmas = [[0.25 * p for p in P], [0.02 * p for p in P]]
    mags = [[s / 3 for s in sg] for sg in sigmas]
    field, sums = _elastic(seeds, P, sigmas, mags)
    f = field.cpu().numpy()
    for i, seed in enumerate(seeds):
        noise = device_noise(seed, P)
        assert noise.min() >= -1 and noise.max() < 1
        assert abs(noise.mean()) < 2e-3 and abs(noise.var() - 1 / 3) < 2e-3
        for d in range(3):
            g = AO.smooth_noise((noise[d].astype(np.float64) + 1) / 2, sigmas[i])
            ref = g / (np.abs(g).max() / (mags[i][d] + 1e-8))
            err = np.abs(f[i, d] - ref).max()
            print(f"elastic {P} seed {i} axis {d}: max|d| / mag = {err / mags[i][d]:.3g}")
            assert err <= 1e-5 * mags[i][d]
            # the sums give the mean offset that re-centres the coordinates
            assert abs(sums[i, d].item() - ref.sum()) / ref.size <= 1e-5 * mags[i][d]
    assert not np.array_equal(device_noise(seeds[0], P), device_noise(seeds[1], P))
    again, sums2 = _elastic(seeds, P, sigmas, mags)
    assert torch.equal(again, field) and torch.equal(sums2, sums)


def _volumes(shape, n, seed):
    rng = np.random.default_rng(seed)
    vols = []
    for _ in range(n):
        v = np.clip(rng.normal(100, 400, size=(*shape, 2)), -1024, 1500).astype(np.int16)
        v[..., 1] = rng.random(shape) < 0.05
        vols.append(v)
    return vols


E2E = [(el, rot, sc, mode, P) for P in [(128, 128, 32), (128, 128, 128)] for mode in ["nearest", "constant"]
       for el in (0, 1) for rot in (0, 1) for sc in (0, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(E2E)))
def test_sampler_with_transform_matches_oracle(case):
    from contrast_gan_3d_b200.data import DevicePatchSampler

    el, rot, sc, mode, P = E2E[case]
    B = 2
    vol_shape = tuple(p + 20 for p in P)
    vols = _volumes(vol_shape, 2, case)
    dvols = [torch.from_numpy(v).to(DEV) for v in vols]
    kw = dict(p_el_per_sample=el, p_rot_per_sample=rot, p_scale_per_sample=sc, border_mode_data=mode,
              angle_x=(-np.pi / 6, np.pi / 6), angle_y=(-np.pi / 6, np.pi / 6), angle_z=(-np.pi / 6, np.pi / 6),
              scale=(0.7, 1.4), independent_scale_for_each_axis=bool(case % 2), p_independent_scale_per_axis=1,
              random_crop=case % 3 != 0, border_cval_data=-0.5 if mode == "constant" else 0)
    t = SpatialTransform2(P, **kw, noise_rng=np.random.default_rng(1000 + case))
    np.random.seed(case)
    got = DevicePatchSampler(dvols, P, B, transform=t).generate_train_batch()
    torch.cuda.synchronize()
    after_device = np.random.get_state()
    np.random.seed(case)
    raw = DevicePatchSampler(dvols, P, B).generate_train_batch()  # the same crops
    seeds = np.random.default_rng(1000 + case)
    state = {"calls": 0, "noise": None}

    def noise_fn(shape):
        if state["calls"] % 3 == 0:
            state["noise"] = device_noise(int(seeds.integers(0, 2 ** 64, dtype=np.uint64)), P)
        d = state["calls"] % 3
        state["calls"] += 1
        return (state["noise"][d].astype(np.float64) + 1) / 2

    rec = []
    ref, rseg = AO.augment_spatial_2(raw["data"].cpu().numpy().astype(np.float64), raw["seg"].cpu().numpy(), P, **kw,
                                     noise_fn=noise_fn, record=rec)
    np.testing.assert_array_equal(np.random.get_state()[1], after_device[1])
    gd, gs = got["data"].cpu().numpy(), got["seg"].cpu().numpy()
    assert gd.shape == (B, 1, *P) and got["seg"].dtype == torch.bool and got["name"] == raw["name"]
    for b, r in enumerate(rec):
        if "coords" not in r:  # shifted zero-filled copy: bit-exact
            np.testing.assert_array_equal(gd[b], ref[b])
            np.testing.assert_array_equal(gs[b], rseg[b])
            continue
        c = r["coords"]
        S = raw["data"].shape[2:]
        edge = np.zeros(P, dtype=bool)
        for d in range(3):
            edge |= (np.abs(c[d]) < 1e-3) | (np.abs(c[d] - (S[d] - 1)) < 1e-3)
        ok = ~edge if mode == "constant" else np.ones(P, dtype=bool)
        err = np.abs(gd[b, 0] - ref[b, 0])[ok].max() / np.abs(ref[b, 0]).max()
        print(f"e2e {E2E[case]} sample {b}: max|d|/max|ref| = {err:.3g}")
        assert err <= 1e-4  # fp32 coordinates on the device against float64 in the oracle: 2.4e-5 measured
        sok = ~(np.any(_near_round(c, 1e-4), axis=0) | edge)
        np.testing.assert_array_equal(gs[b, 0][sok], rseg[b, 0][sok])


@pytest.mark.gpu
def test_bf16_trainer_trains_from_an_augmented_sampler():
    from functools import partial

    from contrast_gan_3d_b200.data import DevicePatchSampler
    from contrast_gan_3d_b200.model import HULoss, PatchGANDiscriminator, ResnetGenerator
    from contrast_gan_3d_b200.optim import FusedAdam
    from contrast_gan_3d_b200.trainer.Trainer import NullLogger, Trainer

    P = (128, 128, 128)
    dvols = [torch.from_numpy(v).to(DEV) for v in _volumes((150, 140, 130), 3, 0)]
    t = SpatialTransform2(P, p_el_per_sample=0.5, p_rot_per_sample=0.5, p_scale_per_sample=0.5,
                          angle_x=(-np.pi / 6, np.pi / 6), scale=(0.7, 1.4), noise_rng=np.random.default_rng(0))
    np.random.seed(0)
    samplers = [DevicePatchSampler(dvols, P, b, transform=t) for b in (2, 1, 1)]
    torch.manual_seed(0)
    dt = torch.bfloat16
    tr = Trainer(10, 2, None, 1, 1, 0, 0, partial(ResnetGenerator, 4, 2, 16, compute_dtype=dt),
                 partial(PatchGANDiscriminator, 1, 8, 3, negative_slope=0.2, compute_dtype=dt),
                 partial(FusedAdam, lr=2e-4, betas=(0.5, 0.999)), partial(FusedAdam, lr=2e-4, betas=(0.5, 0.999)),
                 HULoss(0.18666666666666668, 0.35333333333333333), NullLogger(), torch.device(DEV), weight_clip=0.01,
                 checkpoint_every=None)
    for it in range(3):
        batches = [s.generate_train_batch() for s in samplers]
        batches[0] = dict(batches[0], seg=None)
        logs = tr.train_step(batches, it)
        torch.cuda.synchronize()
        assert logs and all(np.isfinite(float(v.detach())) for v in logs.values()), logs


def test_rotation_matrix_matches_oracle():
    for a in ((0.1, -0.2, 0.3), (0, 0, 0), (np.pi / 6, 0, -np.pi / 6)):
        np.testing.assert_array_equal(rotation_matrix(*a), AO.rotation_matrix_3d(*a))
    assert ctypes.sizeof(_lib.SpatialParams) == 72
