"""ResNet-block dropout (resnet_dropout_prob > 0): module contract on the CPU; on the GPU the keep law against a NumPy
restatement of Philox4x32-10, the fused forward / backward passes, ResNetBlock and Trainer steps against the CPU oracle
on the same masks, and the train / eval / corrector mode rules."""
from functools import partial

import numpy as np
import pytest
import torch
from torch import nn

from oracle import cgan_oracle as O
from tests import dropout_oracle as DO

DEV = "cuda:0"
MASK32 = 0xFFFFFFFF


# ---------------------------------------------------------------------------------------------------- CPU
def test_generator_with_dropout_keeps_the_reference_module_tree_and_state_dict():
    from contrast_gan_3d_b200.model import ResnetGenerator

    torch.manual_seed(0)
    G = ResnetGenerator(4, 2, 16, resnet_dropout_prob=0.5)
    torch.manual_seed(0)
    G0 = ResnetGenerator(4, 2, 16)
    assert [(k, tuple(v.shape)) for k, v in G.state_dict().items()] == [(k, tuple(v.shape)) for k, v in G0.state_dict().items()]
    for blk in G.model.resnet_backbone:
        assert type(blk.dropout) is nn.Dropout and blk.dropout.p == 0.5 and blk.dropout_mask is None
    assert dict(G.named_modules())["model.resnet_backbone.3.dropout"] is G.model.resnet_backbone[3].dropout
    assert all(type(b.dropout) is nn.Identity for b in G0.model.resnet_backbone)


@pytest.mark.parametrize("p", [-0.1, 1.5])
def test_dropout_probability_outside_the_unit_interval_is_rejected(p):
    from contrast_gan_3d_b200.model import ResnetGenerator

    with pytest.raises(ValueError):
        ResnetGenerator(4, 2, 16, resnet_dropout_prob=p)


def test_dropout_in_a_block_without_batchnorm_is_not_implemented():
    from contrast_gan_3d_b200.model.blocks import ResNetBlock

    with pytest.raises(NotImplementedError):
        ResNetBlock(False, 8, 8, dropout_prob=0.5, norm_layer=nn.Identity)
    ResNetBlock(False, 8, 8, dropout_prob=0.0, norm_layer=nn.Identity)


def test_dropout_entry_points_are_bound():
    from contrast_gan_3d_b200 import _lib

    for name in ("cgan3d_bn_apply_dropout", "cgan3d_bn_backward_reduce_dropout", "cgan3d_bn_backward_apply_dropout"):
        assert name in _lib.SIGNATURES


def test_dropout_rejects_p_outside_the_unit_interval_without_a_gpu():
    from contrast_gan_3d_b200 import _lib

    lib = _lib.lib()
    rc = lib.cgan3d_bn_apply_dropout(1, 1, 1, _lib.F32, 8, 8, 1, 1, 1, _lib.ACT_NONE, 0.0, 1.5, 1, None)
    assert rc != 0 and b"outside [0, 1]" in lib.cgan3d_last_error()


# ---------------------------------------------------------------------------------------------------- keep law
def philox4x32_10(q: np.ndarray, seed: int):
    """The four words of Philox4x32-10 at counters (lo32 q, hi32 q, 0, 0) under the 64-bit key `seed` (uint64 arrays)."""
    c0, c1 = q & MASK32, q >> np.uint64(32)
    c2 = c3 = np.zeros_like(q)
    k0, k1 = np.uint64(seed & MASK32), np.uint64(seed >> 32)
    for _ in range(10):
        p0, p1 = c0 * np.uint64(0xD2511F53), c2 * np.uint64(0xCD9E8D57)
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & MASK32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & MASK32
        k0, k1 = np.uint64((int(k0) + 0x9E3779B9) & MASK32), np.uint64((int(k1) + 0xBB67AE85) & MASK32)
    return np.stack([c0, c1, c2, c3], axis=1)  # [len(q), 4]: word j of counter q belongs to element 4q + j


def keep_law(seed: int, n: int, p: float) -> np.ndarray:
    """kept(e) <=> word e & 3 of Philox4x32-10 at counter e >> 2 >= floor(p * 2^32), p as the fp32 the ABI takes."""
    u = philox4x32_10(np.arange((n + 3) // 4, dtype=np.uint64), seed % 2 ** 64).reshape(-1)[:n]
    return u >= np.uint64(int(np.floor(float(np.float32(p)) * 2 ** 32)))


def _bn_inputs(rows, C, dtype, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    y = torch.randn(rows, C, device=DEV, generator=g).to(dtype)
    mi = torch.cat([torch.randn(C, device=DEV, generator=g) * 0.1, torch.rand(C, device=DEV, generator=g) + 0.5])
    gamma = torch.rand(C, device=DEV, generator=g) + 0.5
    beta = torch.randn(C, device=DEV, generator=g) * 0.1
    return y, mi, gamma, beta


def _apply(y, mi, gamma, beta, act, p=None, seed=None):
    from contrast_gan_3d_b200 import _lib, ops

    rows, C = y.shape
    z = torch.empty_like(y)
    if p is None:
        ops.call("cgan3d_bn_apply", ops._p(y), ops._p(z), ops._dt(y.dtype), rows, C, ops._p(mi), ops._p(gamma), ops._p(beta),
                 act, 0.2, None, ops._st())
        return z, None
    keep = torch.empty((y.numel() + 7) // 8, dtype=torch.uint8, device=DEV)
    s = torch.tensor([seed], dtype=torch.int64, device=DEV)
    ops.call("cgan3d_bn_apply_dropout", ops._p(y), ops._p(z), ops._p(keep), ops._dt(y.dtype), rows, C, ops._p(mi), ops._p(gamma),
             ops._p(beta), act, 0.2, p, ops._p(s), ops._st())
    return z, keep


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("C,rows", [(64, 2 * 16 ** 3), (12, 2 * 16 ** 3 + 1)], ids=["vec8", "scalar"])
def test_keep_law_and_scaled_outputs(C, rows, dtype):
    """The bitmask equals the NumPy restatement bit for bit (padding bits of the last byte 0); kept outputs are the p = 0
    outputs times fp32(1 / (1 - p)) (fp32: exactly; bf16: within one ulp), dropped outputs are 0."""
    from contrast_gan_3d_b200 import _lib

    y, mi, gamma, beta = _bn_inputs(rows, C, dtype)
    n = rows * C
    z0, _ = _apply(y, mi, gamma, beta, _lib.ACT_LRELU)
    for p in (0.1, 0.5, 0.9):
        for seed in (0, 1, 0x0123456789ABCDEF, -(2 ** 63) + 12345):
            z, keep = _apply(y, mi, gamma, beta, _lib.ACT_LRELU, p, seed)
            raw = np.unpackbits(keep.cpu().numpy(), bitorder="little")
            ref = keep_law(seed, n, p)
            assert np.array_equal(raw[:n].astype(bool), ref), (p, seed)
            assert not raw[n:].any()
            kept = torch.from_numpy(ref).to(DEV).view(rows, C)
            scale = float(np.float32(1.0 / (1.0 - float(np.float32(p)))))
            want = torch.where(kept, z0.float() * np.float32(scale), torch.zeros((), device=DEV))
            if dtype == torch.float32:
                assert torch.equal(z, want), (p, seed)
            else:
                err = (z.float() - want).abs()
                assert bool((err <= 2 ** -7 * (1 + 2 ** -7) * want.abs()).all()), (p, seed, float(err.max()))


def _backward(dz, y, mi, gamma, beta, act, keep=None, p=0.0):
    from contrast_gan_3d_b200 import ops

    rows, C = y.shape
    sums = torch.empty(2 * C, dtype=torch.float64, device=DEV)
    dy = torch.empty_like(y)
    dg, db = torch.empty(C, device=DEV), torch.empty(C, device=DEV)
    dt = ops._dt(y.dtype)
    args = (ops._p(mi), ops._p(gamma), ops._p(beta), act, 0.2)
    if keep is None:
        ops.call("cgan3d_bn_backward_reduce", ops._p(dz), ops._p(y), dt, rows, C, *args, ops._p(sums), ops._st())
        ops.call("cgan3d_bn_backward_apply", ops._p(dz), ops._p(y), ops._p(dy), dt, rows, C, *args, ops._p(sums), ops._p(dg),
                 ops._p(db), 0.0, ops._st())
    else:
        ops.call("cgan3d_bn_backward_reduce_dropout", ops._p(dz), ops._p(y), ops._p(keep), dt, rows, C, *args, p, ops._p(sums),
                 ops._st())
        ops.call("cgan3d_bn_backward_apply_dropout", ops._p(dz), ops._p(y), ops._p(keep), ops._p(dy), dt, rows, C, *args, p,
                 ops._p(sums), ops._p(dg), ops._p(db), 0.0, ops._st())
    return dy, dg, db


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("C,rows", [(64, 2 * 16 ** 3), (12, 2 * 16 ** 3 + 1)], ids=["vec8", "scalar"])
def test_backward_reads_the_mask_and_ignores_dropped_gradients(C, rows, dtype):
    """The dropout backward equals the plain backward fed dz * keep / (1 - p); dropped elements contribute exactly nothing:
    NaN in dz at every dropped element leaves dy, dgamma and dbeta finite and unchanged.  p = 1: zeros everywhere."""
    from contrast_gan_3d_b200 import _lib

    y, mi, gamma, beta = _bn_inputs(rows, C, dtype, seed=3)
    dz = torch.randn(rows, C, device=DEV).to(dtype)
    act, p = _lib.ACT_NONE, 0.5
    _, keep = _apply(y, mi, gamma, beta, act, p, seed=77)
    kept = torch.from_numpy(keep_law(77, rows * C, p)).to(DEV).view(rows, C)
    got = _backward(dz, y, mi, gamma, beta, act, keep, p)
    want = _backward(torch.where(kept, dz * 2, torch.zeros((), device=DEV, dtype=dtype)), y, mi, gamma, beta, act)
    for a, b, nm in zip(got, want, ("dy", "dgamma", "dbeta")):
        tol = 1e-5 if dtype == torch.float32 else 1e-2
        assert torch.allclose(a.float(), b.float(), rtol=tol, atol=tol * float(b.float().abs().max())), nm
    nan = _backward(torch.where(kept, dz, torch.full((), float("nan"), device=DEV, dtype=dtype)), y, mi, gamma, beta, act, keep, p)
    for a, b, nm in zip(nan, got, ("dy", "dgamma", "dbeta")):
        # equal up to the order of the reductions' fp64 atomics
        assert bool(torch.isfinite(a).all()) and torch.allclose(a.float(), b.float(), rtol=1e-5, atol=1e-6), nm
    z1, keep1 = _apply(y, mi, gamma, beta, act, 1.0, seed=5)
    assert not bool(keep1.any()) and bool((z1 == 0).all())
    for t in _backward(dz, y, mi, gamma, beta, act, keep1, 1.0):
        assert bool((t == 0).all())


# ---------------------------------------------------------------------------------------------------- statistics, seeding
@pytest.mark.gpu
def test_mask_statistics_and_seeding_at_the_c3_resnet_shape():
    """16 x 32^3 x 64, p = 0.5: per-channel kept fraction within 6 sigma of the binomial; two forwards draw different
    masks; torch.manual_seed reproduces a mask."""
    from contrast_gan_3d_b200.model.blocks import ResNetBlock

    torch.manual_seed(0)
    blk = ResNetBlock(False, 64, 64, dropout_prob=0.5, compute_dtype=torch.bfloat16).to(DEV)
    x = torch.randn(16, 32, 32, 32, 64, device=DEV)
    with torch.no_grad():
        torch.manual_seed(11)
        blk.forward_cl(x)
        m1 = blk.dropout_mask.clone()
        blk.forward_cl(x)
        m2 = blk.dropout_mask.clone()
        torch.manual_seed(11)
        blk.forward_cl(x)
        m3 = blk.dropout_mask.clone()
    assert not torch.equal(m1, m2) and torch.equal(m1, m3)
    bits = np.unpackbits(m1.cpu().numpy(), bitorder="little").reshape(-1, 64)
    n = bits.shape[0]
    frac = bits.sum(0)
    sigma = (n * 0.25) ** 0.5
    assert np.all(np.abs(frac - n * 0.5) <= 6 * sigma), (frac.min(), frac.max(), n)


# ---------------------------------------------------------------------------------------------------- ResNetBlock vs oracle
def _cl(x):
    return x.permute(0, 2, 3, 4, 1).contiguous()


def _ncl(x):
    return x.permute(0, 4, 1, 2, 3).contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("C", [64, 4])
def test_resnet_block_forward_backward_against_oracle_on_the_same_mask(C, dtype):
    from contrast_gan_3d_b200.model.blocks import ResNetBlock

    torch.manual_seed(2)
    p = 0.3
    blk = ResNetBlock(False, C, C, dropout_prob=p, compute_dtype=dtype)
    with torch.no_grad():
        for b in (blk.block0, blk.block1):
            b.normalization.weight.uniform_(0.5, 1.5)
            b.normalization.bias.uniform_(-0.5, 0.5)
        if dtype == torch.bfloat16:
            # block1's ReLU away from its kink: a pre-activation within bf16 rounding of 0 takes the other branch than in
            # the fp32 oracle and moves that element's gradient by O(1), whatever the dropout does.  The dropout sits
            # before block1's convolution, so every element of dx and of block0's gradients still goes through the mask.
            blk.block1.normalization.bias.uniform_(6.0, 7.0)
    ref = {k: v.clone() for k, v in blk.state_dict().items()}
    x = torch.randn(2, C, 6, 7, 5)
    gy = torch.randn(2, C, 6, 7, 5)
    blk = blk.to(DEV)
    xd = _cl(x).to(DEV).requires_grad_(True)
    out = blk.forward_cl(xd)
    out.backward(_cl(gy).to(DEV).to(out.dtype))
    mask = DO.unpack_mask(blk.dropout_mask, (2, 6, 7, 5, C))

    params = {k: v.clone().requires_grad_(True) for k, v in ref.items() if "running" not in k and "num_batches" not in k}
    bufs = {k: v.clone() for k, v in ref.items() if k not in params}
    layers = [dict(name="block0", kind="res0", cin=C, cout=C, k=3, stride=1, pad=1, pad_mode="zeros", out_pad=0, norm=True,
                   act="none", bias=False),
              dict(name="block1", kind="res1", cin=C, cout=C, k=3, stride=1, pad=1, pad_mode="zeros", out_pad=0, norm=True,
                   act="relu", bias=False)]
    xr = x.clone().requires_grad_(True)
    yr = DO.generator_forward(params, bufs, xr, layers, train=True, dropout={"block0": (mask, p)})
    names = list(params)
    grads = torch.autograd.grad(yr, [xr] + [params[k] for k in names], gy)
    close = _close32 if dtype == torch.float32 else _close16
    close(_ncl(out), yr, "out")
    close(_ncl(xd.grad), grads[0], "dx")
    for k, g in zip(names, grads[1:]):
        got = dict(blk.named_parameters())[k].grad
        if dtype == torch.float32:
            # a parameter gradient is a sum over all B*X*Y*Z positions: its rounding error scales with the largest entry
            _close32(got, g, k, atol=1e-5 * float(g.abs().max()))
        else:
            close(got, g, k)
    for k, v in bufs.items():
        if "running" in k:
            close(blk.state_dict()[k], v, k)
    assert mask.float().mean().item() == pytest.approx(1 - p, abs=0.05)


def _close32(got, ref, msg, atol=1e-5):
    got, ref = got.detach().float().cpu(), ref.detach().float().cpu()
    err = (got - ref).abs()
    assert bool((err <= 1e-4 * ref.abs() + max(atol, 1e-5)).all()), f"{msg} max err {err.max().item():.3e}"


def _close16(got, ref, msg):
    got, ref = got.detach().float().cpu(), ref.detach().float().cpu()
    err = (got - ref).abs()
    assert bool((err <= 2e-2 * ref.abs() + 2e-2 * ref.abs().max()).all()), f"{msg} max err {err.max().item():.3e}"


# ---------------------------------------------------------------------------------------------------- Trainer steps
def _make_trainer(dtype, p):
    from contrast_gan_3d_b200.model import HULoss, PatchGANDiscriminator, ResnetGenerator
    from contrast_gan_3d_b200.optim import FusedAdam
    from contrast_gan_3d_b200.trainer.Trainer import NullLogger, Trainer

    torch.manual_seed(0)
    return Trainer(10, 2, None, 1, 1, 0, 0, partial(ResnetGenerator, 4, 2, 16, resnet_dropout_prob=p, compute_dtype=dtype),
                   partial(PatchGANDiscriminator, 1, 8, 3, negative_slope=0.2, compute_dtype=dtype),
                   partial(FusedAdam, lr=2e-4, betas=(0.5, 0.999)), partial(FusedAdam, lr=2e-4, betas=(0.5, 0.999)),
                   HULoss(0.18666666666666668, 0.35333333333333333), NullLogger(), torch.device(DEV), weight_clip=0.01,
                   checkpoint_every=None)


def _batch(gen, patch):
    opt = O.synthetic_patches(gen, (2, 1, *patch))
    low, high = O.synthetic_patches(gen, (1, 1, *patch)), O.synthetic_patches(gen, (1, 1, *patch))
    ml, mh = O.synthetic_masks(gen, (1, 1, *patch)), O.synthetic_masks(gen, (1, 1, *patch))
    return opt, low, high, ml, mh


def _step_masks(tr, p):
    out = {}
    for i, blk in enumerate(tr.generator.model.resnet_backbone):
        out[f"model.resnet_backbone.{i}.block0"] = (DO.unpack_mask(blk.dropout_mask, (2, 8, 8, 8, 64)), p)
    return out


KEYS = ("D", "G", "G-full", "sim", "HU")


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True], ids=["eager", "graph"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_train_steps_with_dropout_against_oracle(dtype, graph):
    """ResnetGenerator(4, 2, 16, resnet_dropout_prob=0.5) at 32^3, each step against oracle.train_step fed that step's masks.
    Graph: one eager warm-up, capture at the second step, replays after it; every replay draws new masks."""
    p, patch = 0.5, (32, 32, 32)
    st = O.StepState(seed=0)
    tr = _make_trainer(dtype, p)
    if graph:
        tr.enable_cuda_graph(warmup=1)
    steps = 5 if graph else 3
    gen = torch.Generator().manual_seed(1)
    seen = []
    atol16 = np.array([2e-3, 2e-3, 2e-3, 1e-3, 1e-3])
    for it in range(steps):
        opt, low, high, ml, mh = _batch(gen, patch)
        logs = tr.train_step([dict(data=opt, seg=None), dict(data=low, seg=ml), dict(data=high, seg=mh)], it)
        got = np.array([float(logs[k]) for k in KEYS])
        masks = _step_masks(tr, p)
        seen.append(torch.cat([m.flatten() for m, _ in masks.values()]))
        ref = DO.train_step(st, opt, low, high, ml, mh, it, dropout=masks)
        want = np.array([ref[k] for k in KEYS])
        if dtype == torch.float32:
            rt, at = (1e-4, 1e-5) if it == 0 else (5e-4, 5e-5)  # as tests/test_gpu_parity.py's multi-step oracle test
            assert np.all(np.abs(got - want) <= rt * np.abs(want) + at), (it, got, want)
        else:
            assert np.all(np.abs(got - want) <= 2e-2 * np.abs(want) + atol16), (it, got, want)
    for i in range(1, steps):
        assert not torch.equal(seen[i], seen[i - 1]), f"step {i} reused the masks of step {i - 1}"
    if graph:
        assert all(e["graph"] is not None for e in tr._graphs["entries"].values())


# ---------------------------------------------------------------------------------------------------- modes
@pytest.mark.gpu
def test_eval_mode_output_is_the_p0_output():
    from contrast_gan_3d_b200.model import ResnetGenerator

    torch.manual_seed(0)
    G = ResnetGenerator(4, 2, 16, resnet_dropout_prob=0.5).to(DEV)
    G0 = ResnetGenerator(4, 2, 16).to(DEV)
    G0.load_state_dict(G.state_dict())
    x = torch.randn(2, 1, 32, 32, 32, device=DEV)
    with torch.no_grad():
        G.train(); G0.train()
        G(x); G0(x)  # move the running statistics away from their initial values
        G0.load_state_dict(G.state_dict())
        G.eval(); G0.eval()
        assert torch.equal(G(x), G0(x))


@pytest.mark.gpu
def test_validate_draws_no_mask_and_graph_launches_do_not_change():
    tr = _make_trainer(torch.float32, 0.5)
    tr.val_iterations = 1
    gen = torch.Generator().manual_seed(21)
    opt, low, high, ml, mh = _batch(gen, (32, 32, 32))
    tr.train_step([dict(data=opt, seg=None), dict(data=low, seg=ml), dict(data=high, seg=mh)], 0)
    masks = [b.dropout_mask for b in tr.generator.model.resnet_backbone]
    rng = torch.cuda.get_rng_state()
    vb = [tuple(O.synthetic_patches(gen, (2, 1, 32, 32, 32)) for _ in range(3))]
    tr.validate({0: iter([dict(data=b[0]) for b in vb]), -1: iter([dict(data=b[1]) for b in vb]),
                 1: iter([dict(data=b[2]) for b in vb])}, 1)
    assert torch.equal(torch.cuda.get_rng_state(), rng), "validate drew random numbers"
    assert all(b.dropout_mask is m for b, m in zip(tr.generator.model.resnet_backbone, masks))

    launches = []
    for p in (0.0, 0.5):
        t = _make_trainer(torch.bfloat16, p)
        t.enable_cuda_graph(warmup=1)
        g = torch.Generator().manual_seed(3)
        for it in range(3):
            opt, low, high, ml, mh = _batch(g, (32, 32, 32))
            t.train_step([dict(data=opt, seg=None), dict(data=low, seg=ml), dict(data=high, seg=mh)], it)
        launches.append(t.graph_launches_per_step())
    assert launches[0] == launches[1] > 0, launches


@pytest.mark.gpu
def test_corrector_keeps_dropout_active_and_reseeding_reproduces():
    """Like BatchNorm, the dropout of a p > 0 generator stays in train mode in the corrector (the reference never calls
    .eval()): two calls differ, a call after torch.manual_seed reproduces the first."""
    from contrast_gan_3d_b200.data import FactorZeroCenterScaler
    from contrast_gan_3d_b200.eval import CCTAContrastCorrector
    from contrast_gan_3d_b200.model import ResnetGenerator

    torch.manual_seed(0)
    corr = CCTAContrastCorrector(partial(ResnetGenerator, 4, 2, 16, resnet_dropout_prob=0.5),
                                 FactorZeroCenterScaler(-1024, 1500, 600), torch.device(DEV), inference_patch_size=(16, 16, 16))
    ccta = np.clip(np.random.default_rng(0).normal(100, 300, size=(32, 16, 32)), -1024, 1500).astype(np.int16)
    torch.manual_seed(9)
    a = corr(ccta, batch_size=2)
    b = corr(ccta, batch_size=2)
    torch.manual_seed(9)
    c = corr(ccta, batch_size=2)
    assert float((a - b).abs().max()) > 1.0, "two calls drew the same masks"
    assert float((a - c).abs().max()) <= 1e-2, "re-seeding did not reproduce the masks"
