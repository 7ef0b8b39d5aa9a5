"""Overlapping tiles, Gaussian blending and eval-mode inference in CCTAContrastCorrector: the tile grid and argument
checks on the CPU; on the GPU the batched extraction and the stitch kernel against the per-tile entry points and a
float64 NumPy restatement, and the corrector end to end against the CPU oracle (tests/overlap_oracle.py)."""
import ctypes
from functools import partial

import numpy as np
import pytest
import torch

from oracle import cgan_oracle as O
from tests import overlap_oracle as OO

DEV = "cuda:0"
SHIFT, FACTOR = 238.0, 600.0


def _hu_volume(shape, seed):
    return np.clip(np.random.default_rng(seed).normal(100, 300, size=shape), -1024, 1500).astype(np.int16)


# ---------------------------------------------------------------------------------------------------------------- CPU
GRID_CASES = [  # (volume, patch, step)
    ((512, 512, 256), (128, 128, 128), 64),           # divisible
    ((300, 260, 140), (128, 128, 128), 64),           # non-divisible: squeezed last tiles
    ((128, 128, 32), (128, 128, 32), (64, 32, 16)),   # anisotropic patch
    ((200, 150, 70), (128, 128, 32), (96, 100, 8)),
    ((40, 32, 48), (16, 16, 16), (8, 8, 12)),
    ((37, 16, 41), (16, 16, 16), 16),                 # step == patch
    ((37, 16, 41), (16, 16, 16), 1),
]


@pytest.mark.parametrize("vol, patch, step", GRID_CASES)
def test_grid_tiles_with_step_match_the_helper(vol, patch, step):
    from contrast_gan_3d_b200.eval import grid_tiles

    assert grid_tiles(vol, patch, step) == OO.grid_tiles(vol, patch, step)


@pytest.mark.parametrize("vol, patch", [((512, 512, 256), (128, 128, 128)), ((37, 16, 41), (16, 16, 16)),
                                        ((128, 128, 32), (128, 128, 32))])
def test_grid_tiles_default_step_is_the_patch(vol, patch):
    from contrast_gan_3d_b200.eval import grid_tiles

    assert grid_tiles(vol, patch) == grid_tiles(vol, patch, patch) == O.grid_tiles(vol, patch)


@pytest.mark.parametrize("step", [0, -4, 17, (8, 8), (8, 8, 0), (8, 8, 20), 2.5, (8, 8, 4.0), True, "8"])
def test_grid_tiles_rejects_bad_steps(step):
    from contrast_gan_3d_b200.eval import grid_tiles

    with pytest.raises(ValueError):
        grid_tiles((32, 32, 32), (16, 16, 16), step)


def test_grid_tiles_volume_smaller_than_patch_still_raises():
    from contrast_gan_3d_b200.eval import grid_tiles

    with pytest.raises(ValueError):
        grid_tiles((8, 16, 16), (16, 16, 16), 8)


def _cpu_corrector(**kw):
    from contrast_gan_3d_b200.data import FactorZeroCenterScaler
    from contrast_gan_3d_b200.eval import CCTAContrastCorrector
    from contrast_gan_3d_b200.model import ResnetGenerator

    return CCTAContrastCorrector(partial(ResnetGenerator, 4, 2, 16), FactorZeroCenterScaler(-1024, 1500, 600),
                                 torch.device("cpu"), inference_patch_size=(16, 16, 16), **kw)


def test_corrector_options_are_checked_on_construction():
    with pytest.raises(ValueError):
        _cpu_corrector(blend="median")
    for step in (0, 17, (8, 8)):
        with pytest.raises(ValueError):
            _cpu_corrector(tile_step=step)
    c = _cpu_corrector()
    assert (c.tile_step, c.blend, c.eval_mode) == (None, "avg", False)
    c = _cpu_corrector(tile_step=(8, 8, 12), blend="gaussian", eval_mode=True)
    assert c._steps == (8, 8, 12)


def test_gaussian_weight_stays_positive_over_a_128_tile():
    """The fp32 weight law of the stitch kernel: its smallest value (a corner of a 128^3 tile) is about 5e-11, far from
    underflow, so the normalisation needs no clamp."""
    f = np.float32
    i = np.arange(128, dtype=f)
    sig = f(128) * f(0.125)
    d = i - f(0.5) * f(127)
    g = np.exp(-(d * d) / (f(2) * sig * sig)).astype(f)
    corner = g[0] * g[0] * g[0]
    assert 1e-11 < corner < 1e-10
    np.testing.assert_allclose(OO.weights((128, 128, 128), "gaussian")[0, 0, 0], corner, rtol=1e-5)


# ---------------------------------------------------------------------------------------------------------------- GPU
def _lib():
    from contrast_gan_3d_b200 import _lib as L

    return L


def _st():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _stitch(tiles, vol_shape, patch, step, blend, to_hu=False):
    """cgan3d_tile_stitch over a [n][PX][PY][PZ] fp32 device stack."""
    L = _lib()
    n = tiles.shape[0]
    ptrs = torch.tensor([tiles.data_ptr() + 4 * tiles[0].numel() * t for t in range(n)], dtype=torch.int64, device=DEV)
    out = torch.empty(vol_shape, dtype=torch.float32, device=DEV)
    L.call("cgan3d_tile_stitch", ptrs.data_ptr(), n, *vol_shape, *patch, *step, L.BLEND_GAUSSIAN if blend == "gaussian"
           else L.BLEND_AVG, int(to_hu), SHIFT, FACTOR, out.data_ptr(), _st())
    torch.cuda.synchronize()
    return out


def _steps(step):
    return (step,) * 3 if np.isscalar(step) else tuple(step)


@pytest.mark.gpu
@pytest.mark.parametrize("vol, patch, step", [((37, 29, 41), (16, 12, 20), (5, 7, 20)), ((40, 32, 48), (16, 16, 16), (8, 8, 12)),
                                              ((32, 16, 40), (16, 16, 16), 16), ((20, 20, 20), (20, 20, 20), 20)])
def test_batched_extract_matches_per_tile_extract(vol, patch, step):
    L = _lib()
    hu = torch.from_numpy(_hu_volume(vol, 4)).to(DEV)
    origins = OO.grid_tiles(vol, patch, step)
    n = len(origins)
    t0 = min(3, n - 1)
    got = torch.full((n - t0, *patch), float("nan"), device=DEV)
    L.call("cgan3d_tile_extract_grid", hu.data_ptr(), *vol, *patch, *_steps(step), t0, n - t0, SHIFT, FACTOR,
           got.data_ptr(), _st())
    want = torch.empty_like(got)
    for j, (x, y, z) in enumerate(origins[t0:]):
        L.call("cgan3d_tile_extract", hu.data_ptr(), *vol, x, y, z, *patch, SHIFT, FACTOR, want[j].data_ptr(), _st())
    torch.cuda.synchronize()
    assert torch.equal(got, want)


@pytest.mark.gpu
def test_tile_entry_points_reject_bad_grids():
    L = _lib()
    hu = torch.zeros((32, 32, 32), dtype=torch.int16, device=DEV)
    buf = torch.zeros((64, 16, 16, 16), device=DEV)
    out = torch.zeros((32, 32, 32), device=DEV)
    for args in ((16, 16, 16, 0, 8, 8, 0, 1), (16, 16, 16, 8, 8, 17, 0, 1), (33, 16, 16, 8, 8, 8, 0, 1),
                 (16, 16, 16, 8, 8, 8, 26, 2), (16, 16, 16, 8, 8, 8, -1, 1)):
        with pytest.raises(L.Cgan3dError) as e:
            L.call("cgan3d_tile_extract_grid", hu.data_ptr(), 32, 32, 32, *args, SHIFT, FACTOR, buf.data_ptr(), _st())
        assert e.value.code == -2
    ptrs = torch.zeros(27, dtype=torch.int64, device=DEV)
    with pytest.raises(L.Cgan3dError):  # the 8-step grid of a 32^3 volume has 27 tiles, not 26
        L.call("cgan3d_tile_stitch", ptrs.data_ptr(), 26, 32, 32, 32, 16, 16, 16, 8, 8, 8, 0, 0, SHIFT, FACTOR,
               out.data_ptr(), _st())
    with pytest.raises(L.Cgan3dError):
        L.call("cgan3d_tile_stitch", ptrs.data_ptr(), 27, 32, 32, 32, 16, 16, 16, 8, 8, 8, 2, 0, SHIFT, FACTOR,
               out.data_ptr(), _st())


STITCH_CASES = [  # (volume, patch, step): overlaps 0 / 25 / 50 / 75 %, non-divisible and anisotropic
    ((40, 36, 44), (16, 16, 16), 16),
    ((40, 36, 44), (16, 16, 16), 12),
    ((40, 36, 44), (16, 16, 16), 8),
    ((40, 36, 44), (16, 16, 16), 4),
    ((70, 50, 21), (32, 24, 8), (16, 18, 6)),
    ((128, 128, 32), (64, 64, 16), (48, 32, 4)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("blend", ["avg", "gaussian"])
@pytest.mark.parametrize("vol, patch, step", STITCH_CASES)
def test_stitch_kernel_against_float64(vol, patch, step, blend):
    origins = OO.grid_tiles(vol, patch, step)
    g = torch.Generator().manual_seed(len(origins))
    tiles = torch.randn((len(origins), *patch), generator=g)
    ref = OO.blend_tiles(tiles.numpy(), origins, vol, patch, blend)
    dev = tiles.to(DEV)
    got = _stitch(dev, vol, patch, _steps(step), blend)
    err = np.abs(got.cpu().numpy().astype(np.float64) - ref).max()
    assert err <= 2e-6 * np.abs(ref).max(), (err, np.abs(ref).max())
    assert torch.equal(_stitch(dev, vol, patch, _steps(step), blend), got), "second launch differs"
    hu = _stitch(dev, vol, patch, _steps(step), blend, to_hu=True)  # fused unscale: within an ulp of the two-step one
    torch.testing.assert_close(hu, got * FACTOR + SHIFT, rtol=1e-6, atol=1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("blend, step", [("avg", 8), ("avg", 12), ("gaussian", 8), ("gaussian", 4), ("gaussian", 12)])
@pytest.mark.parametrize("value", [0.7134, -1.3e-3, 517.25])
def test_stitch_of_a_constant_gives_it_back(blend, step, value):
    """avg is a plain sum / count (at most 8 covering tiles here); gaussian a running weighted mean."""
    vol, patch = (40, 36, 44), (16, 16, 16)
    n = len(OO.grid_tiles(vol, patch, step))
    c = np.float32(value)
    got = _stitch(torch.full((n, *patch), float(c), device=DEV), vol, patch, _steps(step), blend).cpu().numpy()
    assert np.abs(got.astype(np.float64) - float(c)).max() <= 2 * float(np.spacing(np.abs(c)))


# --------------------------------------------------------------------------------------------------- corrector, GPU
def _corrector(patch=(16, 16, 16), dtype=torch.float32, dropout=0.0, **kw):
    from contrast_gan_3d_b200.data import FactorZeroCenterScaler
    from contrast_gan_3d_b200.eval import CCTAContrastCorrector
    from contrast_gan_3d_b200.model import ResnetGenerator

    torch.manual_seed(0)
    return CCTAContrastCorrector(partial(ResnetGenerator, 4, 2, 16, compute_dtype=dtype, resnet_dropout_prob=dropout),
                                 FactorZeroCenterScaler(-1024, 1500, 600), torch.device(DEV), inference_patch_size=patch, **kw)


def _recording(corr):
    """Wrap the corrector's per-batch generator step and keep copies of its inputs and outputs."""
    rec = []
    inner = corr._corrected

    def corrected(xb):
        c = inner(xb)
        rec.append((xb.clone(), c.clone()))
        return c

    corr._corrected = corrected
    return rec


def _old_stitch(rec, hu, patch, to_hu):
    """The per-tile cgan3d_tile_extract / _accumulate / _finalize loop of the previous corrector, on recorded outputs."""
    L = _lib()
    X, Y, Z = hu.shape
    acc = torch.zeros((X, Y, Z), device=DEV)
    cnt = torch.zeros_like(acc)
    origins = iter(O.grid_tiles((X, Y, Z), patch))
    for xb, corrected in rec:
        tile = torch.empty((1, *patch), device=DEV)
        for j in range(xb.shape[0]):
            x, y, z = next(origins)
            L.call("cgan3d_tile_extract", hu.data_ptr(), X, Y, Z, x, y, z, *patch, SHIFT, FACTOR, tile.data_ptr(), _st())
            assert torch.equal(tile, xb[j]), "batched extraction differs from cgan3d_tile_extract"
            L.call("cgan3d_tile_accumulate", corrected[j].data_ptr(), acc.data_ptr(), cnt.data_ptr(), X, Y, Z, x, y, z,
                   *patch, _st())
    if not to_hu:
        return acc / cnt
    out = torch.empty_like(acc)
    L.call("cgan3d_tile_finalize", acc.data_ptr(), cnt.data_ptr(), out.data_ptr(), acc.numel(), SHIFT, FACTOR, _st())
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("shape, patch, batch, dtype", [((32, 16, 40), (16, 16, 16), 3, torch.float32),
                                                        ((256, 256, 128), (128, 128, 128), 4, torch.bfloat16)],
                         ids=["small_f32", "c2_quarter_bf16"])
def test_defaults_are_bit_identical_to_the_per_tile_entry_points(shape, patch, batch, dtype):
    corr = _corrector(patch, dtype)
    rec = _recording(corr)
    ccta = _hu_volume(shape, 0)
    hu = torch.from_numpy(ccta).to(DEV)
    got = corr(ccta, batch_size=batch)
    assert got.shape == shape and got.device.type == "cpu" and got.dtype == torch.float32
    assert torch.equal(got, _old_stitch(rec, hu, patch, to_hu=True).cpu())
    rec.clear()
    net = corr.correct_scan_3D(ccta, batch)
    assert net.shape == (1, *shape) and net.is_cuda
    assert torch.equal(net[0], _old_stitch(rec, hu, patch, to_hu=False))


def _set_running_stats(corr, patch, n=3):
    """A few train-mode forwards on random input leave non-trivial BatchNorm running statistics."""
    g = torch.Generator(device=DEV).manual_seed(5)
    with torch.no_grad():
        for _ in range(n):
            corr.model(torch.randn((2, 1, *patch), device=DEV, generator=g) * 0.7 + 0.2)
    bn = corr.model.model.first.normalization
    assert float(bn.running_mean.abs().max()) > 1e-3 and float((bn.running_var - 1).abs().max()) > 1e-3


def _oracle_params(corr):
    """Oracle params (same seed as the corrector's generator) with the device generator's running statistics."""
    torch.manual_seed(0)
    gp, gb = O.init_params(O.generator_layers())
    sd = corr.model.state_dict()
    for k in gb:
        gb[k] = sd[k].detach().cpu().clone()
    for k in gp:
        assert torch.equal(gp[k], sd[k].detach().cpu()), k
    return gp, gb


@pytest.mark.gpu
@pytest.mark.parametrize("eval_mode", [False, True], ids=["train", "eval"])
@pytest.mark.parametrize("blend", ["avg", "gaussian"])
def test_overlapping_corrector_against_the_oracle(blend, eval_mode):
    patch, step = (16, 16, 16), (8, 8, 12)
    corr = _corrector(patch, tile_step=step, blend=blend, eval_mode=eval_mode)
    if eval_mode:
        _set_running_stats(corr, patch)
    gp, gb = _oracle_params(corr)
    ccta = _hu_volume((40, 32, 48), 1)
    ref = OO.correct_scan_3d(gp, gb, ccta, patch=patch, batch_size=5, step=step, blend=blend, eval_mode=eval_mode)
    got = corr(ccta, batch_size=5)
    err = (got.double() - ref).abs()
    assert bool((err <= 1e-4 * ref.abs() + 2e-2).all()), float(err.max())
    net = corr.correct_scan_3D(ccta, 5)
    if eval_mode:  # deterministic: the network-units result is the HU result before the unscale
        torch.testing.assert_close((net[0] * FACTOR + SHIFT).cpu(), got, rtol=1e-6, atol=1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("blend", ["avg", "gaussian"])
def test_overlapping_corrector_upsample_branch(blend):
    patch, step = (30, 32, 28), (15, 16, 10)
    corr = _corrector(patch, tile_step=step, blend=blend)
    assert corr.upsampler is not None
    gp, gb = _oracle_params(corr)
    ccta = _hu_volume((60, 40, 56), 2)
    ref = OO.correct_scan_3d(gp, gb, ccta, patch=patch, batch_size=4, step=step, blend=blend)
    got = corr(ccta, batch_size=4)
    err = (got.double() - ref).abs()
    assert bool((err <= 1e-4 * ref.abs() + 2e-2).all()), float(err.max())


@pytest.mark.gpu
def test_overlapping_corrector_c2_tiles_bf16():
    """128^3 tiles at step 64 with Gaussian blending, bf16 generator, against the fp32 oracle, with the bound of
    test_corrector_c2_shape_quarter_volume_bf16: 2e-2 of the attenuation range (600 HU) + rtol."""
    patch = (128, 128, 128)
    corr = _corrector(patch, torch.bfloat16, tile_step=64, blend="gaussian")
    gp, gb = _oracle_params(corr)
    ccta = _hu_volume((256, 192, 128), 3)
    ref = OO.correct_scan_3d(gp, gb, ccta, patch=patch, batch_size=4, step=64, blend="gaussian")
    got = corr(ccta, batch_size=4)
    err = (got.double() - ref).abs()
    att_ref = (ref - torch.from_numpy(ccta.astype(np.float64))).abs()
    assert float(err.max()) <= 2e-2 * 600 + 2e-2 * float(att_ref.max()), (float(err.max()), float(att_ref.max()))
    assert float(err.mean()) <= 2.0, float(err.mean())


@pytest.mark.gpu
def test_eval_mode_restores_modes_and_does_not_depend_on_the_batch(capsys):
    patch = (16, 16, 16)
    corr = _corrector(patch, tile_step=8, blend="gaussian", eval_mode=True)
    _set_running_stats(corr, patch)
    corr.model.model.downsampling[1].eval()  # a mixed state must come back as it was
    before = [m.training for m in corr.model.modules()]
    ccta = _hu_volume((40, 32, 48), 4)
    a = corr(ccta, batch_size=1)
    assert [m.training for m in corr.model.modules()] == before
    b = corr(ccta, batch_size=16)
    err = (a - b).abs()
    assert bool((err <= 1e-4 * b.abs() + 2e-2).all()), float(err.max())
    with capsys.disabled():
        print(f"\n[eval_mode] batch_size 1 vs 16: bit-identical={torch.equal(a, b)} max |diff| = {float(err.max()):.3e} HU")


@pytest.mark.gpu
def test_eval_mode_turns_dropout_off():
    patch = (16, 16, 16)
    corr = _corrector(patch, dropout=0.5, tile_step=8, eval_mode=True)
    _set_running_stats(corr, patch)
    ccta = _hu_volume((32, 16, 32), 5)
    a = corr(ccta, batch_size=2)
    b = corr(ccta, batch_size=2)
    assert torch.equal(a, b)
    assert corr.model.training
