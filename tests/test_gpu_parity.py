"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle and the golden fixtures.

Tolerances (SURVEY Appendix E): fp32 path  |d| <= 1e-4*|ref| + 1e-5 ;
bf16 path  |d| <= 2e-2*|ref| + 2e-2*max|ref| on tensors and rtol 2e-2 on the logged losses
(the critic loss is a difference of two nearly equal means: its atol is scaled to the logit means)."""
import ctypes
from functools import partial

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import cgan_oracle as O

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _ops():
    from contrast_gan_3d_b200 import _lib, ops

    return _lib, ops


def cl(x):  # [B,C,X,Y,Z] -> channels-last
    return x.permute(0, 2, 3, 4, 1).contiguous()


def ncl(x):
    return x.permute(0, 4, 1, 2, 3).contiguous()


def assert_close32(got, ref, rtol=1e-4, atol=1e-5, msg=""):
    got, ref = got.detach().float().cpu(), ref.detach().float().cpu()
    err = (got - ref).abs()
    tol = rtol * ref.abs() + atol
    assert bool((err <= tol).all()), f"{msg} max err {err.max().item():.3e} (ref max {ref.abs().max().item():.3e})"


def assert_close16(got, ref, msg=""):
    got, ref = got.detach().float().cpu(), ref.detach().float().cpu()
    err = (got - ref).abs()
    tol = 2e-2 * ref.abs() + 2e-2 * ref.abs().max()
    assert bool((err <= tol).all()), f"{msg} max err {err.max().item():.3e} (ref max {ref.abs().max().item():.3e})"


CONV_CASES = [
    # (name, transposed, cin, cout, k, stride, pad, out_pad, spatial(input))
    ("g_first_like", False, 1, 16, 7, 1, 3, 0, (10, 9, 12)),
    ("g_down", False, 16, 32, 3, 2, 1, 0, (12, 10, 8)),
    ("g_down_odd", False, 8, 16, 3, 2, 1, 0, (11, 9, 7)),
    ("g_res", False, 64, 64, 3, 1, 1, 0, (6, 5, 9)),
    ("g_up", True, 32, 16, 3, 2, 1, 1, (5, 6, 4)),
    ("g_last_like", False, 16, 1, 7, 1, 3, 0, (9, 8, 10)),
    ("d_first", False, 1, 8, 4, 2, 1, 0, (12, 12, 10)),
    ("d_mid", False, 8, 16, 4, 2, 1, 0, (8, 10, 12)),
    ("d_last", False, 64, 1, 4, 1, 1, 0, (4, 5, 4)),
]


@pytest.mark.parametrize("case", CONV_CASES, ids=[c[0] for c in CONV_CASES])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_conv_primitives_generic(case, dtype):
    """gather / scatter / wgrad against ATen CPU conv3d / conv_transpose3d and their autograd."""
    _lib, ops = _ops()
    name, tr, cin, cout, k, s, p, op, sp = case
    gen = torch.Generator().manual_seed(hash(name) % 1000)
    B = 2
    x = torch.randn((B, cin, *sp), generator=gen)
    wshape = (cin, cout, k, k, k) if tr else (cout, cin, k, k, k)
    w = torch.randn(wshape, generator=gen) / (cin * k ** 3) ** 0.5
    if dtype == torch.bfloat16:  # compare against the same rounded operands
        x, w = x.bfloat16().float(), w.bfloat16().float()
    x.requires_grad_(True)
    w.requires_grad_(True)
    y = F.conv_transpose3d(x, w, stride=s, padding=p, output_padding=op) if tr else F.conv3d(x, w, stride=s, padding=p)
    gy = torch.randn(y.shape, generator=gen)
    if dtype == torch.bfloat16:
        gy = gy.bfloat16().float()
    gx_ref, gw_ref = torch.autograd.grad(y, (x, w), gy)

    spec = ops.ConvSpec(transposed=tr, cin=cin, cout=cout, k=k, stride=s, pad=p, out_pad=op)
    g, out_sp = spec.geometry(B, sp)
    assert tuple(out_sp) == tuple(y.shape[2:])
    xd = cl(x.detach()).to(DEV, dtype)
    gyd = cl(gy).to(DEV, dtype)
    wp = ops.pack_weights(w.detach().to(DEV), dtype)
    impl = _lib.IMPL_GENERIC
    if tr:
        yd = ops.conv_scatter(g, xd, wp, impl=impl)
        gxd = ops.conv_gather(g, gyd, wp, impl=impl)
        gwd = ops.conv_wgrad(g, gyd, xd, impl=impl)
    else:
        yd = ops.conv_gather(g, xd, wp, impl=impl)
        gxd = ops.conv_scatter(g, gyd, wp, impl=impl)
        gwd = ops.conv_wgrad(g, xd, gyd, impl=impl)
    torch.cuda.synchronize()
    if dtype == torch.float32:
        assert_close32(ncl(yd), y, msg="fprop")
        assert_close32(ncl(gxd), gx_ref, msg="dgrad")
        assert_close32(gwd, gw_ref, rtol=1e-4, atol=1e-4, msg="wgrad")
    else:  # operands identical, fp32 accumulate, only the bf16 output rounding differs
        assert_close32(ncl(yd), y, rtol=8e-3, atol=1e-3, msg="fprop")
        assert_close32(ncl(gxd), gx_ref, rtol=8e-3, atol=1e-3, msg="dgrad")
        assert_close32(gwd, gw_ref, rtol=1e-3, atol=1e-3, msg="wgrad")


@pytest.mark.parametrize("C,dtype", [(3, torch.float32), (4, torch.float32), (8, torch.float32), (16, torch.bfloat16), (1, torch.bfloat16)])
def test_reflect_pad_and_adjoint(C, dtype):
    """scalar (odd channel counts) and 16-byte-vector paths of the reflect pad and of its adjoint"""
    _lib, ops = _ops()
    gen = torch.Generator().manual_seed(3)
    x = torch.randn((2, C, 6, 5, 7), generator=gen).to(dtype).float().requires_grad_(True)
    y = F.pad(x, (3,) * 6, mode="reflect")
    gy = torch.randn(y.shape, generator=gen).to(dtype).float()
    gx, = torch.autograd.grad(y, x, gy)
    yd = ops.reflect_pad(cl(x.detach()).to(DEV, dtype), 3)
    gxd = ops.reflect_pad_backward(cl(gy).to(DEV, dtype), 3)
    assert torch.equal(ncl(yd).float().cpu(), y.detach())
    if dtype == torch.float32:
        assert_close32(ncl(gxd), gx, rtol=1e-6, atol=1e-6)
    else:
        assert_close32(ncl(gxd), gx, rtol=8e-3, atol=1e-3)


@pytest.mark.parametrize("act", ["relu", "lrelu", "none"])
@pytest.mark.parametrize("with_res", [False, True])
def test_conv_block_fn_matches_aten_batchnorm_train_and_backward(act, with_res):
    _lib, ops = _ops()
    from contrast_gan_3d_b200.model.blocks import ConvBlock
    from torch import nn

    torch.manual_seed(5)
    afn = {"relu": nn.ReLU, "lrelu": nn.LeakyReLU, "none": nn.Identity}[act]
    blk = ConvBlock(False, 8, 8, 3, padding=1, activation_fn=afn, negative_slope=0.2 if act == "lrelu" else None)
    with torch.no_grad():
        blk.normalization.weight.uniform_(0.5, 1.5)
        blk.normalization.bias.uniform_(-0.5, 0.5)
    ref = nn.Sequential(nn.Conv3d(8, 8, 3, padding=1, bias=False), nn.BatchNorm3d(8))
    ref[0].load_state_dict(blk.conv.state_dict())
    ref[1].load_state_dict(blk.normalization.state_dict())
    x = torch.randn(3, 8, 6, 7, 5, requires_grad=True)
    r = torch.randn(3, 8, 6, 7, 5, requires_grad=True)
    y = ref(x)
    y = {"relu": F.relu, "lrelu": lambda t: F.leaky_relu(t, 0.2), "none": lambda t: t}[act](y)
    if with_res:
        y = y + r
    gy = torch.randn_like(y)
    refs = torch.autograd.grad(y, [x, r] if with_res else [x], gy, retain_graph=True)
    pgr = torch.autograd.grad(y, list(ref.parameters()), gy)

    blk = blk.to(DEV)
    xd = cl(x.detach()).to(DEV).requires_grad_(True)
    rd = cl(r.detach()).to(DEV).requires_grad_(True)
    yd = blk.forward_cl(xd, residual=rd if with_res else None)
    got = torch.autograd.grad(yd, [xd, rd] if with_res else [xd], cl(gy).to(DEV), retain_graph=True)
    pg = torch.autograd.grad(yd, [blk.conv.weight, blk.normalization.weight, blk.normalization.bias], cl(gy).to(DEV))
    assert_close32(ncl(yd), y, msg="fwd")
    for a, b, n in zip(got, refs, ("dx", "dres")):
        assert_close32(ncl(a), b, rtol=1e-4, atol=2e-5, msg=n)
    for a, b, n in zip(pg, pgr, ("dw", "dgamma", "dbeta")):
        assert_close32(a, b, rtol=1e-4, atol=1e-4, msg=n)
    assert_close32(blk.normalization.running_mean, ref[1].running_mean, rtol=1e-5, atol=1e-6)
    assert_close32(blk.normalization.running_var, ref[1].running_var, rtol=1e-5, atol=1e-6)
    assert int(blk.normalization.num_batches_tracked) == 1


def _load_models(dtype=torch.float32):
    from contrast_gan_3d_b200.model import PatchGANDiscriminator, ResnetGenerator

    torch.manual_seed(0)
    G = ResnetGenerator(4, 2, 16, compute_dtype=dtype).to(DEV)
    D = PatchGANDiscriminator(1, 8, 3, negative_slope=0.2, compute_dtype=dtype).to(DEV)
    return G, D


def test_modules_forward_against_golden_fp32(golden_dir):
    g = np.load(golden_dir / "modules_forward.npz")
    G, D = _load_models()
    G.train(); D.train()
    yg = G(torch.from_numpy(g["xg"]).to(DEV))
    yd = D(torch.from_numpy(g["xd"]).to(DEV))
    yr = G(torch.from_numpy(g["xr"]).to(DEV))  # non-cubic patch
    assert yg.shape == (2, 1, 16, 16, 16) and yd.shape == (2, 1, 1, 1, 1)
    assert_close32(yg, torch.from_numpy(g["yg"]), msg="G")
    assert_close32(yd, torch.from_numpy(g["yd"]), msg="D")
    assert_close32(yr, torch.from_numpy(g["yr"]), msg="G non-cubic")
    G.eval()
    with torch.no_grad():
        ye = G(torch.from_numpy(g["xg"]).to(DEV))
    assert_close32(ye, torch.from_numpy(g["yg_eval"]), msg="G eval")
    sd = G.state_dict()
    for k in sd:  # running stats after the same sequence of train-mode calls
        v = sd[k].double().flatten().cpu()
        fp = np.array([v.sum().item(), v.abs().sum().item(), (v * v).sum().item(), v[0].item(), v[-1].item()])
        np.testing.assert_allclose(fp, g["G_after/" + k], rtol=1e-4, atol=1e-6, err_msg=k)


def test_modules_forward_bf16_against_golden(golden_dir):
    g = np.load(golden_dir / "modules_forward.npz")
    G, D = _load_models(torch.bfloat16)
    yg = G(torch.from_numpy(g["xg"]).to(DEV))
    yd = D(torch.from_numpy(g["xd"]).to(DEV))
    assert yg.dtype == torch.float32 and yd.dtype == torch.float32
    assert_close16(yg, torch.from_numpy(g["yg"]), msg="G bf16")
    assert_close16(yd, torch.from_numpy(g["yd"]), msg="D bf16")


def test_losses_against_golden(golden_dir):
    from contrast_gan_3d_b200.model import HULoss, WassersteinLoss, ZNCCLoss
    from contrast_gan_3d_b200.model.loss import fused_similarity_and_hu

    g = np.load(golden_dir / "losses.npz")
    a = torch.from_numpy(g["a"]).to(DEV).requires_grad_(True)
    b = torch.from_numpy(g["b"]).to(DEV)
    m = torch.from_numpy(g["m"]).to(DEV)
    z = ZNCCLoss()(a, b)
    gz, = torch.autograd.grad(z, a)
    assert z.item() == pytest.approx(g["zncc"].item(), rel=1e-5)
    assert_close32(gz, torch.from_numpy(g["zncc_grad"]), rtol=1e-4, atol=1e-8)
    hu = HULoss(0.18666666666666668, 0.35333333333333333, (2, 1, 8, 8, 8))
    h = hu(a, m)
    gh, = torch.autograd.grad(h, a)
    assert h.item() == pytest.approx(g["hu"].item(), rel=1e-5)
    assert_close32(gh, torch.from_numpy(g["hu_grad"]), rtol=1e-4, atol=1e-8)
    assert hu(a, torch.zeros_like(m)).item() == 0.0  # empty mask: no NaN
    s2, h2 = fused_similarity_and_hu(a, b, m, hu, 1.0, 1.0)
    gf, = torch.autograd.grad(s2 + h2, a)
    assert s2.item() == pytest.approx(g["zncc"].item(), rel=1e-5) and h2.item() == pytest.approx(g["hu"].item(), rel=1e-5)
    assert_close32(gf, torch.from_numpy(g["zncc_grad"] + g["hu_grad"]), rtol=1e-4, atol=1e-8)
    w = WassersteinLoss()(a.detach(), b)
    assert w.item() == pytest.approx(g["wass"].item(), rel=1e-5, abs=1e-7)
    assert WassersteinLoss()(a.detach()).item() == pytest.approx(g["wass_fake_only"].item(), rel=1e-5)
    la = a.detach().clone().requires_grad_(True)
    gw, = torch.autograd.grad(WassersteinLoss()(la, b) * 3.0, la)
    assert_close32(gw, torch.full_like(gw, 3.0 / la.numel()), rtol=1e-6, atol=0)


def test_fused_adam_matches_torch_adam():
    from contrast_gan_3d_b200.optim import FusedAdam

    torch.manual_seed(1)
    p0 = torch.randn(1000)
    pr = p0.clone().requires_grad_(True)
    pm = p0.clone().to(DEV).requires_grad_(True)
    o_ref = torch.optim.Adam([pr], lr=2e-4, betas=(0.5, 0.999))
    o_my = FusedAdam([pm], lr=2e-4, betas=(0.5, 0.999))
    for it in range(5):
        gr = torch.randn(1000) * (10.0 ** (it - 2))
        pr.grad = gr.clone()
        pm.grad = gr.clone().to(DEV)
        o_ref.step()
        o_my.step(clip=0.5)
        with torch.no_grad():
            pr.clamp_(-0.5, 0.5)
        assert_close32(pm, pr, rtol=1e-6, atol=1e-7, msg=f"step {it}")


def _make_trainer(dtype, n_sub_shape=None):
    from contrast_gan_3d_b200.model import HULoss, PatchGANDiscriminator, ResnetGenerator
    from contrast_gan_3d_b200.optim import FusedAdam
    from contrast_gan_3d_b200.trainer.Trainer import NullLogger, Trainer
    from torch.optim.lr_scheduler import MultiStepLR

    torch.manual_seed(0)
    return Trainer(10, 2, None, 1, 1, 1, 0,
                   partial(ResnetGenerator, 4, 2, 16, compute_dtype=dtype),
                   partial(PatchGANDiscriminator, 1, 8, 3, negative_slope=0.2, compute_dtype=dtype),
                   partial(FusedAdam, lr=2e-4, betas=(0.5, 0.999)), partial(FusedAdam, lr=2e-4, betas=(0.5, 0.999)),
                   HULoss(0.18666666666666668, 0.35333333333333333), NullLogger(), torch.device(DEV), weight_clip=0.01,
                   generator_lr_scheduler_class=partial(MultiStepLR, milestones=[6000, 8000], gamma=0.1),
                   critic_lr_scheduler_class=partial(MultiStepLR, milestones=[6000, 8000], gamma=0.1),
                   checkpoint_every=None)


def _batches(gen, patch, n_opt=2, n_low=1, n_high=1):
    opt = O.synthetic_patches(gen, (n_opt, 1, *patch))
    low = O.synthetic_patches(gen, (n_low, 1, *patch))
    high = O.synthetic_patches(gen, (n_high, 1, *patch))
    ml = O.synthetic_masks(gen, (n_low, 1, *patch))
    mh = O.synthetic_masks(gen, (n_high, 1, *patch))
    return opt, low, high, ml, mh


KEYS = ("D", "G", "G-full", "sim", "HU")


def _run(tr, patch, steps):
    gen = torch.Generator().manual_seed(1)
    rows = []
    tr.generator.train(); tr.critic.train()
    for it in range(steps):
        opt, low, high, ml, mh = _batches(gen, patch)
        logs = tr.train_step([dict(data=opt, seg=torch.zeros_like(opt, dtype=torch.bool), name=["o"]),
                              dict(data=low, seg=ml, name=["l"]), dict(data=high, seg=mh, name=["h"])], it)
        rows.append([float(logs[k].detach()) for k in KEYS])
    return np.array(rows)


@pytest.mark.parametrize("name,patch,steps", [("train_steps_32.npz", (32, 32, 32), 3), ("train_steps_c1_64.npz", (64, 64, 64), 2)])
def test_train_steps_fp32_against_reference_golden(golden_dir, name, patch, steps):
    """BASELINE config C1 (and a 32^3 variant): per-step losses and post-step weights vs the reference Trainer."""
    g = np.load(golden_dir / name)
    tr = _make_trainer(torch.float32)
    losses = _run(tr, patch, steps)
    ref = g["losses"]
    # Step 1 (identical weights): the stated fp32 criterion |d| <= 1e-4*|ref| + 1e-5 (D and G are differences of
    # logit means, SURVEY App. E).  Later steps run from weights that went through Adam, whose first updates are
    # lr*g/(|g|+eps) ~ lr*sign(g): summation-order noise of 1e-7 in a near-zero gradient moves that weight by up to
    # 2*lr, so two correct fp32 implementations drift apart by O(lr) per step; the criterion is relaxed accordingly.
    # The control run tests/test_oracle_golden.py::test_fp32_multi_step_drift_control_against_fp64 shows ATen's own fp32 vs
    # fp64 difference using 78 % of the strict criterion at step 2; the later steps are held to 5x the strict criterion.
    strict = 1e-4 * np.abs(ref) + 1e-5
    use = np.abs(losses - ref) / strict
    print(f"fraction of the strict fp32 criterion used per step / loss:\n{use}")
    assert np.all(use[0] <= 1.0), f"\n{losses}\n{ref}"
    assert np.all(use[1:] <= 5.0), f"\n{losses}\n{ref}\n{use}"
    lr = 2e-4
    for prefix, mod in (("G/", tr.generator), ("D/", tr.critic)):
        for k, v in mod.state_dict().items():
            v = v.double().flatten().cpu()
            fp = np.array([v.sum().item(), v.abs().sum().item(), (v * v).sum().item(), v[0].item(), v[-1].item()])
            w = g[prefix + k]
            n = v.numel()
            # sum-type fingerprints: per-element drift <= 2*lr*steps on a small fraction of n elements
            tol = np.array([2 * lr * steps * n ** 0.5, 2 * lr * steps * n ** 0.5, 2e-3 * abs(w[2]) + 1e-6, 2 * lr * steps, 2 * lr * steps])
            assert np.all(np.abs(fp - w) <= 2e-3 * np.abs(w) + tol), (k, fp, w)


def test_train_steps_bf16_against_reference_golden(golden_dir):
    g = np.load(golden_dir / "train_steps_32.npz")
    tr = _make_trainer(torch.bfloat16)
    losses = _run(tr, (32, 32, 32), 3)
    ref = g["losses"]
    # rtol 2e-2 on the losses; D/G are built from logit means of magnitude ~1e-2..1e-1 at init and shrink ~100x once the
    # critic is clipped, so their atol is 2e-2 of the first-step magnitude of those means
    atol = np.array([2e-3, 2e-3, 2e-3, 1e-3, 1e-3])
    assert np.all(np.abs(losses - ref) <= 2e-2 * np.abs(ref) + atol), f"\n{losses}\n{ref}"


def _make_gp_trainer(dtype, norm, patch):
    from contrast_gan_3d_b200.model import HULoss, PatchGANDiscriminator, ResnetGenerator
    from contrast_gan_3d_b200.optim import FusedAdam
    from contrast_gan_3d_b200.trainer.Trainer import NullLogger, Trainer
    from torch import nn

    cargs = dict(negative_slope=0.2, compute_dtype=dtype)
    if norm == "identity":
        cargs.update(norm_layer=nn.Identity)
    else:
        cargs.update(norm_layer=nn.LayerNorm, patch_size=(1, *patch), elementwise_affine=False)
    torch.manual_seed(0)
    return Trainer(10, 2, None, 1, 1, 1, 0, partial(ResnetGenerator, 4, 2, 16, compute_dtype=dtype),
                   partial(PatchGANDiscriminator, 1, 8, 3, **cargs),
                   partial(FusedAdam, lr=1e-4, betas=(0.0, 0.9)), partial(FusedAdam, lr=1e-4, betas=(0.0, 0.9)),
                   HULoss(0.18666666666666668, 0.35333333333333333), NullLogger(), torch.device(DEV), weight_clip=None,
                   checkpoint_every=None)


def _gp_eps(it):
    def f(n):
        torch.manual_seed(9000 + it)  # the recipe of tests/golden/make_golden_gp.py
        return torch.rand((n, 1, 1, 1, 1))
    return f


@pytest.mark.parametrize("name,norm", [("train_steps_gp_32.npz", "identity"), ("train_steps_gp_layernorm_32.npz", "layer")])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_wgan_gp_train_steps_against_reference_golden(golden_dir, name, norm, dtype):
    """WGAN-GP mode (weight_clip=None; reference Trainer.py:122-133, model/utils.py:12-41): three full steps against the
    reference Trainer's logged losses, Identity-norm critic (gradient_penalty_conf.py) and LayerNorm critic
    (gp_layernorm.py).  The penalty differentiates the critic's input gradient, i.e. runs every conv kernel of the critic
    in second order (ops.ConvGatherFn / ConvScatterFn / ConvWgradFn)."""
    g = np.load(golden_dir / name)
    patch = (32, 32, 32)
    tr = _make_gp_trainer(dtype, norm, patch)
    assert list(tr.critic.state_dict().keys()) == list(g["D_keys"])
    gen = torch.Generator().manual_seed(1)
    tr.generator.train(); tr.critic.train()
    rows = []
    for it in range(3):
        opt, low, high, ml, mh = _batches(gen, patch)
        tr.gp_eps_fn = _gp_eps(it)
        logs = tr.train_step([dict(data=opt, seg=None, name=[]), dict(data=low, seg=ml, name=[]), dict(data=high, seg=mh, name=[])], it)
        rows.append([float(logs[k].detach()) for k in KEYS])
    losses, ref = np.array(rows), g["losses"]
    if dtype == torch.float32:
        strict = 1e-4 * np.abs(ref) + 1e-5
        use = np.abs(losses - ref) / strict
        # Steps >= 1 run from weights that went through Adam(beta1 = 0): updates are lr * g / |g|-like, so fp32 rounding
        # noise moves whole weights.  tests/test_oracle_golden.py::test_wgan_gp_fp32_drift_control_against_fp64 measures
        # ATen's OWN fp32-vs-fp64 difference in these configurations: 0.33x the strict criterion (Identity critic) and 53x
        # (LayerNorm critic, whose normalisation amplifies the weight noise) at step 2.  Bound: 5x / 100x the strict criterion.
        later = 5.0 if norm == "identity" else 100.0
        assert np.all(use[0] <= 1.0) and np.all(use[1:] <= later), f"\n{losses}\n{ref}\n{use}"
        lr, steps = 1e-4, 3
        for prefix, mod in (("G/", tr.generator), ("D/", tr.critic)):
            for k, v in mod.state_dict().items():
                v = v.double().flatten().cpu()
                fp = np.array([v.sum().item(), v.abs().sum().item(), (v * v).sum().item(), v[0].item(), v[-1].item()])
                w, n = g[prefix + k], v.numel()
                tol = np.array([2 * lr * steps * n ** 0.5, 2 * lr * steps * n ** 0.5, 2e-3 * abs(w[2]) + 1e-6, 2 * lr * steps, 2 * lr * steps])
                assert np.all(np.abs(fp - w) <= 2e-3 * np.abs(w) + tol), (k, fp, w)
    else:
        # D is dominated by the penalty (~5-10 = lambda * (|grad| - 1)^2); G = -mean(logits) is a mean of logits whose
        # spread is O(1) under LayerNorm (unit-variance features) and O(0.1) otherwise: atol = 1 % of that spread
        atol = np.array([2e-2, 2e-3, 2e-3, 1e-3, 1e-3]) if norm == "identity" else np.array([5e-2, 1e-2, 1e-2, 1e-3, 1e-3])
        assert np.all(np.abs(losses - ref) <= 2e-2 * np.abs(ref) + atol), f"\n{losses}\n{ref}"


def test_gradient_penalty_second_order_gradients_vs_aten():
    """d(penalty)/d(weights) of a two-layer bias + LeakyReLU critic: the twice-differentiable conv Functions against ATen's
    double backward (fp32, CPU) on identical weights and inputs."""
    from contrast_gan_3d_b200 import ops
    from contrast_gan_3d_b200.model.utils import wgan_gradient_penalty

    gen = torch.Generator().manual_seed(4)
    w1 = (torch.randn((8, 1, 4, 4, 4), generator=gen) * 0.2).requires_grad_(True)
    b1 = (torch.randn(8, generator=gen) * 0.1).requires_grad_(True)
    w2 = (torch.randn((1, 8, 4, 4, 4), generator=gen) * 0.1).requires_grad_(True)
    real, fake = torch.randn((3, 1, 12, 10, 8), generator=gen), torch.randn((3, 1, 12, 10, 8), generator=gen)
    eps = torch.rand((3, 1, 1, 1, 1), generator=gen)

    def critic_ref(x):
        return F.conv3d(F.leaky_relu(F.conv3d(x, w1, b1, stride=2, padding=1), 0.2), w2, None, stride=1, padding=1)

    pen_ref = wgan_gradient_penalty(real, fake, critic_ref, eps_fn=lambda n: eps)
    gref = torch.autograd.grad(pen_ref, (w1, b1, w2))

    w1d, b1d, w2d = (t.detach().to(DEV).requires_grad_(True) for t in (w1, b1, w2))
    s1 = ops.ConvSpec(transposed=False, cin=1, cout=8, k=4, stride=2, pad=1)
    s2 = ops.ConvSpec(transposed=False, cin=8, cout=1, k=4, stride=1, pad=1)

    def critic_ours(x):  # [B, 1, X, Y, Z] -> channels-last
        h = x.reshape(x.shape[0], *x.shape[2:], 1)
        h = F.leaky_relu(ops.conv_differentiable(h, w1d, s1, torch.float32) + b1d, 0.2)
        h = ops.conv_differentiable(h, w2d, s2, torch.float32)
        return h.reshape(h.shape[0], 1, *h.shape[1:4])

    pen = wgan_gradient_penalty(real.to(DEV), fake.to(DEV), critic_ours, device=DEV, eps_fn=lambda n: eps)
    got = torch.autograd.grad(pen, (w1d, b1d, w2d))
    assert pen.item() == pytest.approx(pen_ref.item(), rel=1e-4)
    for a, b, nm in zip(got, gref, ("dw1", "db1", "dw2")):
        assert_close32(a, b, rtol=1e-3, atol=1e-4 * float(b.abs().max()) + 1e-7, msg=nm)


def test_train_step_against_oracle_other_shape():
    """Non-cubic patches and unequal low/high batch sizes, fp32, against the CPU oracle step."""
    patch = (32, 48, 32)
    st = O.StepState(seed=0)
    tr = _make_trainer(torch.float32)
    gen = torch.Generator().manual_seed(11)
    for it in range(2):
        opt, low, high, ml, mh = _batches(gen, patch, 3, 2, 1)
        ref = O.train_step(st, opt, low, high, ml, mh, it)
        logs = tr.train_step([dict(data=opt, seg=None, name=[]), dict(data=low, seg=ml, name=[]),
                              dict(data=high, seg=mh, name=[])], it)
        for k in KEYS:
            rt, at = (1e-4, 1e-5) if it == 0 else (5e-4, 5e-5)  # see test_train_steps_fp32_against_reference_golden
            assert abs(float(logs[k].detach()) - ref[k]) <= rt * abs(ref[k]) + at, (it, k, float(logs[k].detach()), ref[k])
    for k, v in tr.generator.state_dict().items():
        r = {**st.gp, **st.gb}[k]
        assert_close32(v, r, rtol=2e-3, atol=2 * 2e-4 * 2, msg=k)


@pytest.mark.parametrize("C,dtype,act", [(16, torch.bfloat16, "relu"), (8, torch.float32, "lrelu"), (64, torch.bfloat16, "none")])
def test_bn_apply_fused_with_reflect_pad(C, dtype, act):
    """cgan3d_bn_apply_pad == reflect_pad(bn_apply(y)) bit for bit (same arithmetic, only the store address changes)."""
    from contrast_gan_3d_b200 import _lib, ops
    B, X, Y, Z, p = 2, 9, 12, 10, 3
    gen = torch.Generator().manual_seed(3)
    y = torch.randn((B, X, Y, Z, C), generator=gen).to(DEV).to(dtype)
    mi = torch.cat([torch.randn(C, generator=gen) * 0.1, torch.rand(C, generator=gen) + 0.5]).to(DEV)
    gamma, beta = (torch.rand(C, generator=gen) + 0.5).to(DEV), (torch.randn(C, generator=gen) * 0.1).to(DEV)
    code = {"relu": _lib.ACT_RELU, "lrelu": _lib.ACT_LRELU, "none": _lib.ACT_NONE}[act]
    dt = _lib.BF16 if dtype == torch.bfloat16 else _lib.F32
    z = torch.empty_like(y)
    ops.call("cgan3d_bn_apply", ops._p(y), ops._p(z), dt, B * X * Y * Z, C, ops._p(mi), ops._p(gamma), ops._p(beta), code, 0.2, None, ops._st())
    want = ops.reflect_pad(z, p)
    got = torch.empty((B, X + 2 * p, Y + 2 * p, Z + 2 * p, C), dtype=dtype, device=DEV)
    ops.call("cgan3d_bn_apply_pad", ops._p(y), ops._p(got), dt, B, X, Y, Z, C, ops._p(mi), ops._p(gamma), ops._p(beta), code, 0.2, p, ops._st())
    assert torch.equal(got, want)
    ref = torch.nn.functional.pad(z.permute(0, 4, 1, 2, 3).float(), (p,) * 6, mode="reflect").permute(0, 2, 3, 4, 1).to(dtype)
    assert torch.equal(got, ref)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_conv_block_with_padded_output_backward_vs_aten(dtype):
    """ConvBlock whose output carries its consumer's reflection padding (pad_out = 3, the generator's last up-sampling
    block): forward and all gradients against ATen's conv_transpose3d -> batch_norm -> relu -> reflection_pad3d."""
    from contrast_gan_3d_b200.model.blocks import ConvBlock
    from torch import nn

    torch.manual_seed(6)
    blk = ConvBlock(False, 32, 16, 3, upsample=True, output_padding=1, padding=1, stride=2, compute_dtype=dtype)
    with torch.no_grad():
        blk.normalization.weight.uniform_(0.5, 1.5)
        blk.normalization.bias.uniform_(-0.5, 0.5)
    ref_conv = nn.ConvTranspose3d(32, 16, 3, stride=2, padding=1, output_padding=1, bias=False)
    ref_bn = nn.BatchNorm3d(16)
    ref_conv.load_state_dict(blk.conv.state_dict()); ref_bn.load_state_dict(blk.normalization.state_dict())
    x = torch.randn(2, 32, 5, 6, 4)
    if dtype == torch.bfloat16:
        x = x.bfloat16().float()
        with torch.no_grad():
            ref_conv.weight.copy_(ref_conv.weight.bfloat16().float())
            blk.conv.weight.copy_(ref_conv.weight)
    x.requires_grad_(True)
    yr = F.pad(F.relu(ref_bn(ref_conv(x))), (3,) * 6, mode="reflect")
    gy = torch.randn_like(yr)
    if dtype == torch.bfloat16:
        gy = gy.bfloat16().float()
    gx_r, gw_r, gg_r, gb_r = torch.autograd.grad(yr, [x, ref_conv.weight, ref_bn.weight, ref_bn.bias], gy)
    blk = blk.to(DEV)
    xd = cl(x.detach()).to(DEV).requires_grad_(True)
    yd = blk.forward_cl(xd, pad_out=3)
    gx, gw, gg, gb = torch.autograd.grad(yd, [xd, blk.conv.weight, blk.normalization.weight, blk.normalization.bias], cl(gy).to(DEV, yd.dtype))
    if dtype == torch.float32:
        assert_close32(ncl(yd), yr, msg="fwd")
        assert_close32(ncl(gx), gx_r, rtol=1e-4, atol=2e-5, msg="dx")
        for a_, b_, n in ((gw, gw_r, "dw"), (gg, gg_r, "dgamma"), (gb, gb_r, "dbeta")):
            assert_close32(a_, b_, rtol=1e-4, atol=1e-4, msg=n)
    else:
        assert_close16(ncl(yd), yr, msg="fwd")
        assert_close16(ncl(gx), gx_r, msg="dx")
        for a_, b_, n in ((gw, gw_r, "dw"), (gg, gg_r, "dgamma"), (gb, gb_r, "dbeta")):
            assert_close16(a_, b_, msg=n)


def test_fit_prefetches_next_batch_with_identical_results():
    """`fit` draws the next batch one iteration early and copies it under the running step (Trainer.prefetch).  The staged
    generator input must be exactly the host batch both when the step starts and when it ends (the next prefetch must not
    touch the buffer in flight), and the trained weights must match (to atomic-summation noise) those of calling train_step
    batch by batch (reference loop, trainer/Trainer.py:206-209)."""
    patch = (32, 32, 32)

    def loaders(seed, steps):
        gen = torch.Generator().manual_seed(seed)
        rows = [[], [], []]
        for _ in range(steps):
            opt, low, high, ml, mh = _batches(gen, patch)
            rows[0].append(dict(data=opt.pin_memory(), seg=None, name=[]))
            rows[1].append(dict(data=low.pin_memory(), seg=ml.pin_memory(), name=[]))
            rows[2].append(dict(data=high.pin_memory(), seg=mh.pin_memory(), name=[]))
        return rows

    steps = 4
    a, b = _make_trainer(torch.bfloat16), _make_trainer(torch.bfloat16)
    a.train_iterations = b.train_iterations = steps
    a.val_every = b.val_every = None
    rows = loaders(5, steps)
    a.generator.train(); a.critic.train()
    for it in range(steps):
        a.train_step([rows[0][it], rows[1][it], rows[2][it]], it)
    rows = loaders(5, steps)
    seen_begin, seen_end = [], []
    gen_fwd, gen_step = b._generate, b.train_generator

    def spy_generate(subopt):
        seen_begin.append(subopt.clone())
        return gen_fwd(subopt)

    def spy_generator_step(inputs, recon, masks):
        out = gen_step(inputs, recon, masks)
        seen_end.append(inputs.clone())
        return out

    b._generate, b.train_generator = spy_generate, spy_generator_step
    b.fit({0: iter(rows[0]), -1: iter(rows[1]), 1: iter(rows[2])}, {})
    assert getattr(b, "_prefetch_flip", None) is not None, "fit did not prefetch"
    torch.cuda.synchronize()
    assert len(seen_begin) == steps and len(seen_end) == steps
    for it in range(steps):
        want = torch.cat([rows[1][it]["data"], rows[2][it]["data"]]).to(DEV)
        assert torch.equal(seen_begin[it], want), f"step {it}: staged input differs at the start of the step"
        assert torch.equal(seen_end[it], want), f"step {it}: staged input was overwritten during the step"
    # the weight gradients are summed with floating-point atomics, so two runs agree to rounding noise, not bit for bit:
    # 4 Adam steps of 2e-4 bound the drift of one weight by 1.6e-3
    for (k, va), vb in zip(a.generator.state_dict().items(), b.generator.state_dict().values()):
        if "running_" in k or "num_batches" in k:
            continue
        assert_close32(va, vb, rtol=0, atol=1.7e-3, msg=k)
    d = (a.generator.state_dict()["model.first.conv.weight"] - b.generator.state_dict()["model.first.conv.weight"]).abs().mean()
    assert float(d) < 2e-4, float(d)


def test_raw_int16_hu_batches_scaled_on_device():
    """Batches may carry raw int16 HU (2 bytes per voxel across PCIe); Trainer(hu_scaler=...) applies the reference's
    FactorZeroCenterScaler on the device (data/Scaler.py:41-42): same losses as feeding the host-scaled fp32 patches."""
    from contrast_gan_3d_b200.data import FactorZeroCenterScaler

    sc = FactorZeroCenterScaler(-1024, 1500, 600)
    gen = torch.Generator().manual_seed(8)
    patch = (32, 32, 32)
    hu = [torch.randint(-1024, 1500, (n, 1, *patch), generator=gen, dtype=torch.int16) for n in (2, 1, 1)]
    ml, mh = O.synthetic_masks(gen, (1, 1, *patch)), O.synthetic_masks(gen, (1, 1, *patch))
    scaled = [torch.from_numpy(sc(h.numpy().astype(np.float32)).astype(np.float32)) for h in hu]
    a, b = _make_trainer(torch.float32), _make_trainer(torch.float32)
    b.hu_scaler = sc
    la = a.train_step([dict(data=scaled[0], seg=None), dict(data=scaled[1], seg=ml), dict(data=scaled[2], seg=mh)], 0)
    lb = b.train_step([dict(data=hu[0].pin_memory(), seg=None), dict(data=hu[1].pin_memory(), seg=ml), dict(data=hu[2].pin_memory(), seg=mh)], 0)
    for k in KEYS:
        assert float(lb[k]) == pytest.approx(float(la[k]), rel=1e-5, abs=1e-7), k
    with pytest.raises(ValueError, match="hu_scaler"):
        a.train_step([dict(data=hu[0], seg=None), dict(data=hu[1], seg=ml), dict(data=hu[2], seg=mh)], 0)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_cuda_graphed_step_equals_eager_step(dtype):
    """Trainer.enable_cuda_graph: the captured + replayed step (3 eager warm-ups, capture at the 4th step, replays after it)
    against the eager Trainer on the same batches, with an LR schedule that changes the rate while the graph is live
    (learning rate and Adam step count are device-resident in FusedAdam) and a generator trained every second iteration
    (two graph variants)."""
    from torch.optim.lr_scheduler import MultiStepLR

    def make():
        tr = _make_trainer(dtype)
        tr.lr_scheduler_G = MultiStepLR(tr.optimizer_G, milestones=[2, 4], gamma=0.5)
        tr.lr_scheduler_D = MultiStepLR(tr.optimizer_D, milestones=[5, 8], gamma=0.5)
        tr.train_generator_every = 2
        return tr

    a, b = make(), make()
    b.enable_cuda_graph(warmup=2)
    gen = torch.Generator().manual_seed(17)
    patch = (32, 32, 32)
    steps = 12
    la, lb = [], []
    for it in range(steps):
        opt, low, high, ml, mh = _batches(gen, patch)
        p = [dict(data=opt, seg=None, name=[]), dict(data=low, seg=ml, name=[]), dict(data=high, seg=mh, name=[])]
        ra = a.train_step(p, it)
        la.append({k: float(v) for k, v in ra.items()})
        rb = b.train_step(p, it)
        lb.append({k: float(v) for k, v in rb.items()})  # read before the next replay overwrites the static outputs
    ents = b._graphs["entries"]
    assert len(ents) == 2 and all(e["graph"] is not None for e in ents.values()), "both variants (critic only / critic + generator) captured"
    assert b.optimizer_G.param_groups[0]["lr"] == a.optimizer_G.param_groups[0]["lr"] == 2e-4 * 0.25
    assert b.optimizer_D.param_groups[0]["lr"] == a.optimizer_D.param_groups[0]["lr"] == 2e-4 * 0.25
    for o_a, o_b in ((a.optimizer_G, b.optimizer_G), (a.optimizer_D, b.optimizer_D)):
        sa = [o_a.state[p]["step"] for p in o_a.param_groups[0]["params"]]
        sb = [o_b.state[p]["step"] for p in o_b.param_groups[0]["params"]]
        assert sa == sb, "host-side Adam step counts follow the replays"
        hyper = o_b._dev[id(o_b.param_groups[0])]["hyper"].cpu()
        assert float(hyper[1]) == sa[0] and float(hyper[0]) == pytest.approx(o_b.param_groups[0]["lr"])
    rt, at = (2e-3, 1e-4) if dtype == torch.float32 else (2e-2, 2e-3)  # same kernels; fp atomics order differs between runs
    for it in range(steps):
        assert set(la[it]) == set(lb[it])
        for k in la[it]:
            assert abs(la[it][k] - lb[it][k]) <= rt * abs(la[it][k]) + at, (it, k, la[it][k], lb[it][k])
    for (k, va), vb in zip(a.generator.state_dict().items(), b.generator.state_dict().values()):
        if "num_batches" in k:
            assert int(va) == int(vb), k
        elif "running_" not in k:
            assert_close32(va, vb, rtol=0, atol=2 * 2e-4 * steps, msg=k)
            assert float((va.float() - vb.float()).abs().mean()) < 1e-4, k


def test_step_after_reset_to_initial_state_is_a_first_step():
    """What bench.py --dump-outputs relies on: after graph-replayed steps (which advance FusedAdam's device-side step
    count without running its Python code), releasing the graphs, loading the initial state_dicts and clearing the
    optimizers' state make the next step the first step of a fresh trainer (host and device step counts included)."""
    a, b = _make_trainer(torch.float32), _make_trainer(torch.float32)
    initial = [{k: v.detach().clone() for k, v in m.state_dict().items()} for m in (b.generator, b.critic)]
    opt, low, high, ml, mh = _batches(torch.Generator().manual_seed(17), (32, 32, 32))
    p = [dict(data=opt, seg=None, name=[]), dict(data=low, seg=ml, name=[]), dict(data=high, seg=mh, name=[])]
    la = {k: float(v) for k, v in a.train_step(p, 0).items()}
    b.enable_cuda_graph(warmup=2)
    for _ in range(4):  # two eager warm-ups, the capture, one replay
        b.train_step(p, 0)
    assert all(e["graph"] is not None for e in b._graphs["entries"].values())
    b.release_cuda_graphs()
    for m, sd in zip((b.generator, b.critic), initial):
        m.load_state_dict(sd)
    b.optimizer_G.state.clear(); b.optimizer_D.state.clear()
    lb = {k: float(v) for k, v in b.train_step(p, 0).items()}
    for k in la:  # same kernels; fp atomics order differs between runs
        assert abs(la[k] - lb[k]) <= 2e-3 * abs(la[k]) + 1e-4, (k, la[k], lb[k])
    for o in (b.optimizer_G, b.optimizer_D):
        assert {o.state[q]["step"] for q in o.param_groups[0]["params"]} == {1}
        assert float(o._dev[id(o.param_groups[0])]["hyper"][1]) == 1.0
    for ma, mb in ((a.generator, b.generator), (a.critic, b.critic)):
        for (k, va), vb in zip(ma.state_dict().items(), mb.state_dict().values()):
            if "num_batches" in k:
                assert int(va) == int(vb), k
            else:  # one Adam step moves a weight by at most lr; a near-zero gradient may flip its sign
                assert_close32(vb, va, rtol=1e-3, atol=2 * 2e-4, msg=k)
                assert float((va.float() - vb.float()).abs().mean()) < 1e-5, k


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_rmsprop_small_patch_configuration_against_oracle(dtype):
    """The reference's rmsprop_conf.py (RMSprop for both networks, which star-imports small_patch_size.py: non-cubic
    128 x 128 x 32 patches): two steps with FusedRMSprop (+ fused weight clip) against the oracle stepping with the
    torch.optim.RMSprop algorithm."""
    from contrast_gan_3d_b200.model import HULoss, PatchGANDiscriminator, ResnetGenerator
    from contrast_gan_3d_b200.optim import FusedRMSprop
    from contrast_gan_3d_b200.trainer.Trainer import NullLogger, Trainer

    patch = (128, 128, 32)
    st = O.StepState(seed=0)
    st.opt_g, st.opt_d = O.RMSpropState(st.gp, 2e-4), O.RMSpropState(st.dp, 2e-4)
    torch.manual_seed(0)
    tr = Trainer(10, 2, None, 1, 1, 1, 0, partial(ResnetGenerator, 4, 2, 16, compute_dtype=dtype),
                 partial(PatchGANDiscriminator, 1, 8, 3, negative_slope=0.2, compute_dtype=dtype),
                 partial(FusedRMSprop, lr=2e-4), partial(FusedRMSprop, lr=2e-4),
                 HULoss(0.18666666666666668, 0.35333333333333333), NullLogger(), torch.device(DEV), weight_clip=0.01,
                 checkpoint_every=None)
    gen = torch.Generator().manual_seed(23)
    for it in range(2):
        opt, low, high, ml, mh = _batches(gen, patch)
        ref = O.train_step(st, opt, low, high, ml, mh, it)
        logs = tr.train_step([dict(data=opt, seg=None, name=[]), dict(data=low, seg=ml, name=[]), dict(data=high, seg=mh, name=[])], it)
        for k in KEYS:
            got = float(logs[k].detach())
            if dtype == torch.float32:
                rt, at = (1e-4, 1e-5) if it == 0 else (5e-4, 5e-5)
            else:
                rt, at = 2e-2, (2e-3 if k in ("D", "G", "G-full") else 1e-3)
            assert abs(got - ref[k]) <= rt * abs(ref[k]) + at, (it, k, got, ref[k])
    if dtype == torch.float32:
        for k, v in tr.critic.state_dict().items():
            if "running_" in k or "num_batches" in k:
                continue
            assert float(v.abs().max()) <= 0.01 + 1e-7, k  # the clip is fused into the RMSprop kernel


def test_generator_only_iterations_and_cadence():
    tr = _make_trainer(torch.float32)
    tr.train_generator_every = 2
    gen = torch.Generator().manual_seed(2)
    opt, low, high, ml, mh = _batches(gen, (32, 32, 32))
    p = [dict(data=opt, seg=None, name=[]), dict(data=low, seg=ml, name=[]), dict(data=high, seg=mh, name=[])]
    assert set(tr.train_step(p, 0)) == {"D", "G", "G-full", "sim", "HU"}
    assert set(tr.train_step(p, 1)) == {"D"}


def test_device_sampler_bit_exact_against_oracle():
    from contrast_gan_3d_b200.data import DevicePatchSampler

    rng = np.random.default_rng(3)
    for shape, patch in (((40, 37, 20), (16, 16, 16)), ((10, 37, 13), (16, 16, 16)), ((16, 16, 16), (16, 16, 16)),
                         ((5, 6, 7), (8, 8, 8))):
        vol = rng.integers(-1024, 1500, size=(*shape, 2)).astype(np.int16)
        vol[..., 1] = rng.random(shape) < 0.05
        np.random.seed(42)
        data, seg, lbs = O.generate_one(vol, patch)
        smp = DevicePatchSampler([torch.from_numpy(vol).to(DEV)], patch, 1)
        d = torch.empty((1, 1, *patch), dtype=torch.float32, device=DEV)
        m = torch.empty((1, 1, *patch), dtype=torch.uint8, device=DEV)
        np.random.seed(42)
        got_lbs = smp.sample_one(smp.volumes[0], d[0], m[0])
        assert got_lbs == lbs
        np.testing.assert_array_equal(d.cpu().numpy(), data)  # bit-exact incl. the (hu-238)/600 rounding
        np.testing.assert_array_equal(m.cpu().numpy().astype(np.float32), seg)
    np.random.seed(0)
    b = DevicePatchSampler([torch.from_numpy(vol).to(DEV)] * 3, (8, 8, 8), 4).generate_train_batch()
    assert b["data"].shape == (4, 1, 8, 8, 8) and b["seg"].dtype == torch.bool and len(b["name"]) == 4


def test_corrector_against_oracle_small_volume():
    from contrast_gan_3d_b200.data import FactorZeroCenterScaler
    from contrast_gan_3d_b200.eval import CCTAContrastCorrector
    from contrast_gan_3d_b200.model import ResnetGenerator

    torch.manual_seed(0)
    gp, gb = O.init_params(O.generator_layers())
    rng = np.random.default_rng(0)
    ccta = np.clip(rng.normal(100, 300, size=(32, 16, 40)), -1024, 1500).astype(np.int16)  # z not divisible: overlap
    ref = O.correct_scan_3d(gp, gb, ccta, patch=(16, 16, 16), batch_size=3)
    torch.manual_seed(0)
    corr = CCTAContrastCorrector(partial(ResnetGenerator, 4, 2, 16), FactorZeroCenterScaler(-1024, 1500, 600),
                                 torch.device(DEV), inference_patch_size=(16, 16, 16))
    got = corr(ccta, batch_size=3)
    assert got.shape == ccta.shape and got.device.type == "cpu"
    assert_close32(got, ref, rtol=1e-4, atol=2e-2, msg="corrected HU")  # HU units: 2e-2 HU == 3e-5 network units


def test_corrector_upsample_branch_and_return_types():
    """A patch size that the strided convs do not round-trip (30 -> 15 -> 8 -> 16 -> 32): the reference resizes the
    attenuation map with nn.Upsample(size=patch) before subtracting it (eval/CCTAContrastCorrector.py:42-52,79).  Also the
    reference's call surface: `correct_scan` alias, correct_scan_3D returns [1, W, H, D] network units on the device."""
    from contrast_gan_3d_b200.data import FactorZeroCenterScaler
    from contrast_gan_3d_b200.eval import CCTAContrastCorrector
    from contrast_gan_3d_b200.model import ResnetGenerator

    torch.manual_seed(0)
    gp, gb = O.init_params(O.generator_layers())
    rng = np.random.default_rng(1)
    patch = (30, 32, 28)
    ccta = np.clip(rng.normal(100, 300, size=(60, 32, 56)), -1024, 1500).astype(np.int16)
    ref = O.correct_scan_3d(gp, gb, ccta, patch=patch, batch_size=2)
    torch.manual_seed(0)
    sc = FactorZeroCenterScaler(-1024, 1500, 600)
    corr = CCTAContrastCorrector(partial(ResnetGenerator, 4, 2, 16), sc, torch.device(DEV), inference_patch_size=patch)
    assert isinstance(corr.upsampler, torch.nn.Upsample) and corr.correct_scan == corr.correct_scan_3D
    got = corr(ccta, batch_size=2)
    assert_close32(got, ref, rtol=1e-4, atol=2e-2, msg="corrected HU (upsample branch)")
    torch.manual_seed(0)
    corr2 = CCTAContrastCorrector(partial(ResnetGenerator, 4, 2, 16), sc, torch.device(DEV), inference_patch_size=patch)
    net = corr2.correct_scan(ccta, 2)
    assert net.shape == (1, *ccta.shape) and net.is_cuda
    assert_close32(sc.unscale(net).squeeze().cpu(), ref, rtol=1e-4, atol=2e-2, msg="correct_scan_3D return value")


def test_corrector_c2_shape_quarter_volume_bf16():
    """BASELINE config C2's tiling at a quarter of the volume (256 x 256 x 128 in 128^3 tiles, batches of 4: several
    batches, so the train-mode BatchNorm grouping and the tile order matter), bf16 generator, against the fp32 oracle:
    corrected HU within 2e-2 of the attenuation range (600 HU) => 12 HU + rtol."""
    from contrast_gan_3d_b200.data import FactorZeroCenterScaler
    from contrast_gan_3d_b200.eval import CCTAContrastCorrector
    from contrast_gan_3d_b200.model import ResnetGenerator

    torch.manual_seed(0)
    gp, gb = O.init_params(O.generator_layers())
    rng = np.random.default_rng(2)
    ccta = np.clip(rng.normal(100, 300, size=(256, 256, 128)), -1024, 1500).astype(np.int16)
    ref = O.correct_scan_3d(gp, gb, ccta, patch=(128, 128, 128), batch_size=4)
    torch.manual_seed(0)
    corr = CCTAContrastCorrector(partial(ResnetGenerator, 4, 2, 16, compute_dtype=torch.bfloat16),
                                 FactorZeroCenterScaler(-1024, 1500, 600), torch.device(DEV), inference_patch_size=(128, 128, 128))
    got = corr(ccta, batch_size=4)
    assert got.shape == ccta.shape
    err = (got - ref).abs()
    att_ref = (ref - torch.from_numpy(ccta.astype(np.float32))).abs()  # |600 * G(x)|
    assert float(err.max()) <= 2e-2 * 600 + 2e-2 * float(att_ref.max()), (float(err.max()), float(att_ref.max()))
    assert float(err.mean()) <= 2.0, float(err.mean())  # HU


# ------------------------------------------------------------------------------------------------------------
# tcgen05 implicit-GEMM path
# ------------------------------------------------------------------------------------------------------------
TC_CASES = [
    # (name, cin, cout, B, spatial)
    ("tiny_64", 64, 64, 2, (8, 8, 8)),
    ("res_layer_32", 64, 64, 2, (32, 32, 32)),
    ("ztiled_16_32", 16, 32, 1, (6, 12, 70)),
    ("c128", 128, 128, 1, (9, 16, 16)),
    ("ragged_32_16", 32, 16, 3, (5, 13, 11)),
    ("c32_to_64", 32, 64, 2, (7, 9, 20)),
]


@pytest.mark.parametrize("case", TC_CASES, ids=[c[0] for c in TC_CASES])
def test_tcgen05_conv3_s1_fprop_and_dgrad(case):
    """tcgen05 kernel vs the generic CUDA-core kernel on identical bf16 operands (both fp32-accumulate: they may only
    differ by summation order and the final bf16 rounding) and vs ATen fp32 on CPU."""
    _lib, ops = _ops()
    name, cin, cout, B, sp = case
    gen = torch.Generator().manual_seed(len(name))
    x = torch.randn((B, cin, *sp), generator=gen).bfloat16().float()
    w = (torch.randn((cout, cin, 3, 3, 3), generator=gen) / (cin * 27) ** 0.5).bfloat16().float()
    gy = torch.randn((B, cout, *sp), generator=gen).bfloat16().float()
    spec = ops.ConvSpec(transposed=False, cin=cin, cout=cout, k=3, stride=1, pad=1)
    g, _ = spec.geometry(B, sp)
    assert _lib.lib().cgan3d_conv_select(ctypes.byref(g), _lib.BF16, 0) == 2, "tcgen05 path should be selected"
    xd = cl(x).to(DEV, torch.bfloat16)
    gyd = cl(gy).to(DEV, torch.bfloat16)
    wp = ops.pack_weights(w.to(DEV), torch.bfloat16)
    y_tc = ops.conv_gather(g, xd, wp, impl=_lib.IMPL_TC)
    y_gen = ops.conv_gather(g, xd, wp, impl=_lib.IMPL_GENERIC)
    dx_tc = ops.conv_scatter(g, gyd, wp, impl=_lib.IMPL_TC)
    dx_gen = ops.conv_scatter(g, gyd, wp, impl=_lib.IMPL_GENERIC)
    torch.cuda.synchronize()
    xr = x.clone().requires_grad_(True)
    y_ref = F.conv3d(xr, w, padding=1)
    dx_ref, = torch.autograd.grad(y_ref, xr, gy)
    if _lib.lib().cgan3d_conv_select(ctypes.byref(g), _lib.BF16, 2) == 2:  # tcgen05 wgrad (Cout in {32, 64}, Cin <= 64)
        dw_tc = ops.conv_wgrad(g, xd, gyd, impl=_lib.IMPL_TC)
        wr = w.clone().requires_grad_(True)
        dw_ref, = torch.autograd.grad(F.conv3d(x, wr, padding=1), wr, gy)
        assert_close32(dw_tc, dw_ref, rtol=2e-3, atol=2e-3 * float(dw_ref.abs().max()), msg="wgrad vs ATen")
    else:
        assert cout not in (32, 64) or cin > 64 or sp[2] > 62
    for got, gen_, ref, nm in ((y_tc, y_gen, y_ref, "fprop"), (dx_tc, dx_gen, dx_ref, "dgrad")):
        assert torch.isfinite(got.float()).all(), nm
        assert_close32(ncl(got), ref, rtol=8e-3, atol=2e-3, msg=nm + " vs ATen")
        d = (got.float() - gen_.float()).abs()
        # one bf16 ulp of disagreement at most (different summation order before the rounding)
        assert bool((d <= 2 ** -7 * gen_.float().abs() + 1e-3).all()), f"{nm} vs generic: {d.max().item()}"


S2_CASES = [
    # (name, transposed module?, cin, cout, k, out_pad, B, spatial_in)
    ("down0_like", False, 16, 32, 3, 0, 2, (16, 12, 20)),
    ("down1_like", False, 32, 64, 3, 0, 1, (12, 16, 72)),
    ("down_odd", False, 16, 16, 3, 0, 2, (9, 11, 13)),
    ("critic_mid_k4", False, 16, 32, 4, 0, 2, (12, 16, 8)),
    ("critic_first_k4", False, 1, 8, 4, 0, 2, (12, 16, 8)),
    ("critic_first_big", False, 1, 8, 4, 0, 1, (20, 70, 44)),
    ("critic_first_odd", False, 1, 8, 4, 0, 2, (9, 11, 14)),
    ("critic_mid0_k4", False, 8, 16, 4, 0, 2, (12, 16, 8)),
    ("critic_mid0_big", False, 8, 16, 4, 0, 1, (20, 24, 40)),
    ("down_c8_k3", False, 8, 16, 3, 0, 2, (10, 12, 14)),
    ("critic_mid2_k4", False, 32, 64, 4, 0, 2, (16, 16, 16)),
    ("up0_like", True, 64, 32, 3, 1, 1, (6, 8, 10)),
    ("up1_like", True, 32, 16, 3, 1, 2, (8, 6, 36)),
]


@pytest.mark.parametrize("case", S2_CASES, ids=[c[0] for c in S2_CASES])
def test_tcgen05_strided_and_transposed_convs(case):
    """Strided gather / scatter tcgen05 kernels (tap-program kernel) vs the generic kernels and vs ATen, both directions of
    each module (fprop and dgrad)."""
    _lib, ops = _ops()
    name, tr, cin, cout, k, op, B, sp = case
    gen = torch.Generator().manual_seed(len(name) + 7)
    x = torch.randn((B, cin, *sp), generator=gen).bfloat16().float().requires_grad_(True)
    wshape = (cin, cout, k, k, k) if tr else (cout, cin, k, k, k)
    w = (torch.randn(wshape, generator=gen) / (cin * k ** 3) ** 0.5).bfloat16().float()
    y = F.conv_transpose3d(x, w, stride=2, padding=1, output_padding=op) if tr else F.conv3d(x, w, stride=2, padding=1)
    gy = torch.randn(y.shape, generator=gen).bfloat16().float()
    gx_ref, = torch.autograd.grad(y, x, gy)
    spec = ops.ConvSpec(transposed=tr, cin=cin, cout=cout, k=k, stride=2, pad=1, out_pad=op)
    g, out_sp = spec.geometry(B, sp)
    xd = cl(x.detach()).to(DEV, torch.bfloat16)
    gyd = cl(gy).to(DEV, torch.bfloat16)
    wp = ops.pack_weights(w.to(DEV), torch.bfloat16)
    fwd_op, bwd_op = (1, 0) if tr else (0, 1)
    assert _lib.lib().cgan3d_conv_select(ctypes.byref(g), _lib.BF16, fwd_op) == 2, "tcgen05 path should cover the forward"
    fwd = (lambda impl: ops.conv_scatter(g, xd, wp, impl=impl)) if tr else (lambda impl: ops.conv_gather(g, xd, wp, impl=impl))
    bwd = (lambda impl: ops.conv_gather(g, gyd, wp, impl=impl)) if tr else (lambda impl: ops.conv_scatter(g, gyd, wp, impl=impl))
    pairs = [(fwd(_lib.IMPL_TC), fwd(_lib.IMPL_GENERIC), y.detach(), "fprop")]
    if _lib.lib().cgan3d_conv_select(ctypes.byref(g), _lib.BF16, bwd_op) == 2:
        pairs.append((bwd(_lib.IMPL_TC), bwd(_lib.IMPL_GENERIC), gx_ref, "dgrad"))
    else:
        assert "odd" in name, f"{name}: dgrad of this layer should run on the tcgen05 path"
    torch.cuda.synchronize()
    for got, gen_, ref, nm in pairs:
        assert torch.isfinite(got.float()).all(), nm
        assert_close32(ncl(got), ref, rtol=8e-3, atol=2e-3, msg=nm + " vs ATen")
        d = (got.float() - gen_.float()).abs()
        assert bool((d <= 2 ** -7 * gen_.float().abs() + 1e-3).all()), f"{nm} vs generic: {d.max().item()}"
    # weight gradient (same formula for both module kinds: small side x big side)
    wr = w.clone().requires_grad_(True)
    yr = F.conv_transpose3d(x.detach(), wr, stride=2, padding=1, output_padding=op) if tr else F.conv3d(x.detach(), wr, stride=2, padding=1)
    dw_ref, = torch.autograd.grad(yr, wr, gy)
    big, small = (gyd, xd) if tr else (xd, gyd)
    if _lib.lib().cgan3d_conv_select(ctypes.byref(g), _lib.BF16, 2) == 2:
        dw_tc = ops.conv_wgrad(g, big, small, impl=_lib.IMPL_TC)
        assert_close32(dw_tc, dw_ref, rtol=2e-3, atol=2e-3 * float(dw_ref.abs().max()), msg="strided wgrad (tcgen05) vs ATen")
    else:
        assert g.Cs not in (16, 32, 64) and "critic_first" not in name, "tcgen05 wgrad should cover Cs in {16, 32, 64} and the critic's first layer"
    dw_gen = ops.conv_wgrad(g, big, small, impl=_lib.IMPL_GENERIC)
    assert_close32(dw_gen, dw_ref, rtol=2e-3, atol=2e-3 * float(dw_ref.abs().max()), msg="strided wgrad (generic) vs ATen")


THIN_CASES = [
    # (name, B, spatial_in, pad)   7x7x7 stride-1 thin-channel layers of the generator
    ("thin_small_valid", 2, (10, 9, 12), 0),
    ("thin_zeropad", 1, (9, 16, 8), 3),
    ("thin_tiled", 2, (20, 150, 37), 0),
    ("thin_c1_like", 1, (38, 38, 38), 0),
]


@pytest.mark.parametrize("case", THIN_CASES, ids=[c[0] for c in THIN_CASES])
def test_tcgen05_thin_7x7x7_layers(case):
    """tcgen05 kernels of model.first (1->16) and model.last_conv (16->1): fprop, dgrad and wgrad vs the generic
    kernels (same bf16 operands) and vs ATen fp32."""
    _lib, ops = _ops()
    name, B, sp, pad = case
    gen = torch.Generator().manual_seed(len(name) + 3)
    for cin, cout in ((1, 16), (16, 1)):
        x = torch.randn((B, cin, *sp), generator=gen).bfloat16().float().requires_grad_(True)
        w = (torch.randn((cout, cin, 7, 7, 7), generator=gen) / (cin * 343) ** 0.5).bfloat16().float().requires_grad_(True)
        y = F.conv3d(x, w, padding=pad)
        gy = torch.randn(y.shape, generator=gen).bfloat16().float()
        gx_ref, gw_ref = torch.autograd.grad(y, (x, w), gy)
        spec = ops.ConvSpec(transposed=False, cin=cin, cout=cout, k=7, stride=1, pad=pad)
        g, _ = spec.geometry(B, sp)
        xd = cl(x.detach()).to(DEV, torch.bfloat16)
        gyd = cl(gy).to(DEV, torch.bfloat16)
        wp = ops.pack_weights(w.detach().to(DEV), torch.bfloat16)
        sel = [_lib.lib().cgan3d_conv_select(ctypes.byref(g), _lib.BF16, op) for op in range(3)]
        checks = []
        if sel[0] == 2:
            checks.append((ops.conv_gather(g, xd, wp, impl=_lib.IMPL_TC), ops.conv_gather(g, xd, wp, impl=_lib.IMPL_GENERIC), y.detach(), "fprop"))
        if sel[1] == 2:
            checks.append((ops.conv_scatter(g, gyd, wp, impl=_lib.IMPL_TC), ops.conv_scatter(g, gyd, wp, impl=_lib.IMPL_GENERIC), gx_ref, "dgrad"))
        torch.cuda.synchronize()
        for got, gen_, ref, nm in checks:
            assert torch.isfinite(got.float()).all(), f"{cin}->{cout} {nm}"
            assert_close32(ncl(got), ref, rtol=8e-3, atol=2e-3, msg=f"{cin}->{cout} {nm} vs ATen")
            d = (got.float() - gen_.float()).abs()
            assert bool((d <= 2 ** -7 * gen_.float().abs() + 1e-3).all()), f"{cin}->{cout} {nm} vs generic: {d.max().item()}"
        if sel[2] == 2:
            dw = ops.conv_wgrad(g, xd, gyd, impl=_lib.IMPL_TC)
            assert_close32(dw, gw_ref, rtol=2e-3, atol=2e-3 * float(gw_ref.abs().max()), msg=f"{cin}->{cout} wgrad vs ATen")
    # which ops the tcgen05 path must cover for these layers (extended as kernels land)
    for cin, cout in ((1, 16), (16, 1)):
        spec = ops.ConvSpec(transposed=False, cin=cin, cout=cout, k=7, stride=1, pad=pad)
        g, _ = spec.geometry(B, sp)
        assert _lib.lib().cgan3d_conv_select(ctypes.byref(g), _lib.BF16, 0) == 2
        assert _lib.lib().cgan3d_conv_select(ctypes.byref(g), _lib.BF16, 1) == 2


def test_train_step_bf16_full_patch_size_against_oracle():
    """BASELINE patch size (128^3, the shape every tcgen05 tiling of bench.py runs at), 2 pairs, bf16 path: the four
    logged losses of one full G+D step against the fp32 CPU oracle, rtol 2e-2 (atol as in the 32^3 test)."""
    patch = (128, 128, 128)
    st = O.StepState(seed=0)
    tr = _make_trainer(torch.bfloat16)
    gen = torch.Generator().manual_seed(5)
    opt, low, high, ml, mh = _batches(gen, patch, 2, 1, 1)
    ref = O.train_step(st, opt, low, high, ml, mh, 0)
    logs = tr.train_step([dict(data=opt, seg=None, name=[]), dict(data=low, seg=ml, name=[]), dict(data=high, seg=mh, name=[])], 0)
    atol = dict(zip(KEYS, (2e-3, 2e-3, 2e-3, 1e-3, 1e-3)))
    for k in KEYS:
        got = float(logs[k].detach())
        assert abs(got - ref[k]) <= 2e-2 * abs(ref[k]) + atol[k], (k, got, ref[k])


def test_full_size_layers_tcgen05_vs_generic():
    """Every generator layer shape of BASELINE config C3 (B = 1): tcgen05 fprop vs the CUDA-core kernel on identical bf16
    operands (<= 1 bf16 ulp), and linearity conv(2x) == 2 conv(x) bit-exactly (a power-of-two scale commutes with every
    rounding step), which is size independent."""
    _lib, ops = _ops()
    layers = [  # (transposed, cin, cout, k, stride, pad, out_pad, spatial_in)
        (False, 1, 16, 7, 1, 0, 0, (134, 134, 134)), (False, 16, 32, 3, 2, 1, 0, (128, 128, 128)),
        (False, 32, 64, 3, 2, 1, 0, (64, 64, 64)), (False, 64, 64, 3, 1, 1, 0, (32, 32, 32)),
        (True, 64, 32, 3, 2, 1, 1, (32, 32, 32)), (True, 32, 16, 3, 2, 1, 1, (64, 64, 64)),
        (False, 16, 1, 7, 1, 0, 0, (134, 134, 134)),
    ]
    gen = torch.Generator().manual_seed(9)
    for tr, cin, cout, k, s, p, op, sp in layers:
        spec = ops.ConvSpec(transposed=tr, cin=cin, cout=cout, k=k, stride=s, pad=p, out_pad=op)
        g, _ = spec.geometry(1, sp)
        x = torch.randn((1, *sp, cin), generator=gen).to(DEV, torch.bfloat16)
        wshape = (cin, cout, k, k, k) if tr else (cout, cin, k, k, k)
        w = (torch.randn(wshape, generator=gen) / (cin * k ** 3) ** 0.5).to(DEV)
        wp = ops.pack_weights(w, torch.bfloat16)
        f = (lambda xx, impl: ops.conv_scatter(g, xx, wp, impl=impl)) if tr else (lambda xx, impl: ops.conv_gather(g, xx, wp, impl=impl))
        opi = 1 if tr else 0
        assert _lib.lib().cgan3d_conv_select(ctypes.byref(g), _lib.BF16, opi) == 2, (cin, cout, k, s)
        y_tc = f(x, _lib.IMPL_TC).float()
        y_gen = f(x, _lib.IMPL_GENERIC).float()
        d = (y_tc - y_gen).abs()
        assert bool((d <= 2 ** -7 * y_gen.abs() + 1e-3).all()), f"{cin}->{cout} k{k} s{s}: {d.max().item()}"
        y2 = f(x * 2, _lib.IMPL_TC).float()
        assert torch.equal(y2, 2 * y_tc), f"{cin}->{cout} k{k} s{s}: linearity"


@pytest.mark.parametrize("case", [("first7", False, 1, 16, 7, 1, 0, 2, (12, 20, 15)), ("s1_64", False, 64, 64, 3, 1, 0, 2, (9, 10, 12)), ("s1_32_16", False, 32, 16, 3, 1, 0, 1, (6, 13, 11)),
                                  ("down", False, 16, 32, 3, 2, 0, 2, (12, 10, 16)), ("critic_mid", False, 8, 16, 4, 2, 0, 2, (12, 16, 8)),
                                  ("up", True, 32, 16, 3, 2, 1, 2, (6, 5, 8)), ("critic_mid2", False, 32, 64, 4, 2, 0, 1, (16, 16, 16))],
                         ids=lambda c: c[0])
def test_conv_with_fused_batchnorm_statistics(case):
    """cgan3d_conv_bnstats: identical output to the plain tcgen05 conv, and per-channel sum / sum of squares equal to those of
    the fp32 ATen result (they are taken from the fp32 accumulators, before the bf16 storage rounding)."""
    _lib, ops = _ops()
    name, tr, cin, cout, k, s, op, B, sp = case
    gen = torch.Generator().manual_seed(len(name))
    x = torch.randn((B, cin, *sp), generator=gen).bfloat16().float()
    wshape = (cin, cout, k, k, k) if tr else (cout, cin, k, k, k)
    w = (torch.randn(wshape, generator=gen) / (cin * k ** 3) ** 0.5).bfloat16().float()
    pad = 0 if k == 7 else 1
    y = F.conv_transpose3d(x, w, stride=s, padding=pad, output_padding=op) if tr else F.conv3d(x, w, stride=s, padding=pad)
    spec = ops.ConvSpec(transposed=tr, cin=cin, cout=cout, k=k, stride=s, pad=pad, out_pad=op)
    g, _ = spec.geometry(B, sp)
    assert ops.conv_fuses_bnstats(g, torch.bfloat16, tr), "this layer should fuse its BatchNorm statistics"
    xd = cl(x).to(DEV, torch.bfloat16)
    wp = ops.pack_weights(w.to(DEV), torch.bfloat16)
    plain = ops.conv_scatter(g, xd, wp, impl=_lib.IMPL_TC) if tr else ops.conv_gather(g, xd, wp, impl=_lib.IMPL_TC)
    fused, sums = ops.conv_bnstats(g, xd, wp, tr)
    torch.cuda.synchronize()
    assert torch.equal(fused, plain)
    yc = y.double().permute(1, 0, 2, 3, 4).reshape(cout, -1)
    ref = torch.cat([yc.sum(1), (yc * yc).sum(1)])
    assert_close32(sums, ref, rtol=1e-4, atol=1e-4 * float(ref.abs().max()), msg="fused statistics")


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_validate_against_oracle(dtype):
    """Trainer.validate (eval-mode BatchNorm from the running statistics, non-cubic validation patches as in the reference's
    (256, 256, 128) setting, scaled down) after one training step, against the oracle's restatement."""
    st = O.StepState(seed=0)
    tr = _make_trainer(dtype)
    tr.val_iterations = 2
    gen = torch.Generator().manual_seed(21)
    opt, low, high, ml, mh = _batches(gen, (32, 32, 32))
    O.train_step(st, opt, low, high, ml, mh, 0)
    tr.train_step([dict(data=opt, seg=None, name=[]), dict(data=low, seg=ml, name=[]), dict(data=high, seg=mh, name=[])], 0)
    vpatch = (64, 64, 32)
    vb = [tuple(O.synthetic_patches(gen, (2, 1, *vpatch)) for _ in range(3)) for _ in range(2)]
    ref = O.validate(st, vb)
    loaders = {0: iter([dict(data=b[0]) for b in vb]), -1: iter([dict(data=b[1]) for b in vb]), 1: iter([dict(data=b[2]) for b in vb])}
    got = tr.validate(loaders, 400)
    assert tr.generator.training and tr.critic.training  # validate() restores train mode (Trainer.py:297-298)
    rt, at = (2e-3, 1e-4) if dtype == torch.float32 else (2e-2, 2e-3)  # weights went through one Adam step (see above)
    for k in ("D", "G", "sim"):
        assert abs(float(got[k]) - ref[k]) <= rt * abs(ref[k]) + at, (k, float(got[k]), ref[k])
