"""Pin the CPU oracle (oracle/cgan_oracle.py) against fixtures produced by the unmodified
reference (tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest
import torch

from oracle import cgan_oracle as O

# The reference produced the goldens on CPU with 8 intra-op threads.  ATen splits its CPU reductions by thread count, so
# the oracle reproduces them bit for bit only at that count; at others the fp32 summation order alone exceeds the
# tolerances below.
GOLDEN_THREADS = 8


@pytest.fixture(autouse=True)
def _golden_thread_count():
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


def _fp(v):
    v = v.detach().double().flatten()
    return np.array([v.sum().item(), v.abs().sum().item(), (v * v).sum().item(), v[0].item(), v[-1].item()])


@pytest.fixture(scope="module")
def mods(golden_dir):
    return np.load(golden_dir / "modules_forward.npz")


def _init():
    torch.manual_seed(0)
    gp, gb = O.init_params(O.generator_layers())
    dp, db = O.init_params(O.critic_layers())
    return gp, gb, dp, db


def test_state_dict_contract_and_seeded_init(mods):
    gp, gb, dp, db = _init()
    gkeys = O.state_dict_order(O.generator_layers())
    dkeys = O.state_dict_order(O.critic_layers())
    assert gkeys == list(mods["G_keys"])
    assert dkeys == list(mods["D_keys"])
    allg = {**gp, **gb}
    alld = {**dp, **db}
    assert [str(tuple(allg[k].shape)) for k in gkeys] == list(mods["G_shapes"])
    assert [str(tuple(alld[k].shape)) for k in dkeys] == list(mods["D_shapes"])
    for k in gkeys:  # bit-identical seeded init (same RNG draws, same order)
        np.testing.assert_array_equal(_fp(allg[k]), mods["G/" + k], err_msg=k)
    for k in dkeys:
        np.testing.assert_array_equal(_fp(alld[k]), mods["D/" + k], err_msg=k)
    n_g = sum(v.numel() for v in gp.values())
    n_d = sum(v.numel() for v in dp.values())
    assert [n_g, n_d] == list(mods["n_params"]) == [1035297, 176873]


def test_generator_and_critic_forward(mods):
    gp, gb, dp, db = _init()
    yg = O.generator_forward(gp, gb, torch.from_numpy(mods["xg"]))
    yd = O.critic_forward(dp, db, torch.from_numpy(mods["xd"]))
    np.testing.assert_allclose(yg.numpy(), mods["yg"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(yd.numpy(), mods["yd"], rtol=1e-5, atol=1e-6)
    yr = O.generator_forward(gp, gb, torch.from_numpy(mods["xr"]))
    np.testing.assert_allclose(yr.numpy(), mods["yr"], rtol=1e-5, atol=1e-6)
    ye = O.generator_forward(gp, gb, torch.from_numpy(mods["xg"]), train=False)
    np.testing.assert_allclose(ye.numpy(), mods["yg_eval"], rtol=1e-5, atol=1e-6)
    # running statistics after the two train-mode calls match the reference's buffers
    for k, v in {**gp, **gb}.items():
        np.testing.assert_allclose(_fp(v), mods["G_after/" + k], rtol=1e-6, atol=1e-9, err_msg=k)


def test_losses(golden_dir):
    g = np.load(golden_dir / "losses.npz")
    a = torch.from_numpy(g["a"]).requires_grad_(True)
    b = torch.from_numpy(g["b"])
    m = torch.from_numpy(g["m"])
    z = O.zncc_loss(a, b)
    gz, = torch.autograd.grad(z, a)
    assert z.item() == pytest.approx(g["zncc"].item(), rel=1e-6)
    np.testing.assert_allclose(gz.numpy(), g["zncc_grad"], rtol=1e-5, atol=1e-9)
    h = O.hu_loss(a, m, 0.18666666666666668, 0.35333333333333333)
    gh, = torch.autograd.grad(h, a)
    assert h.item() == pytest.approx(g["hu"].item(), rel=1e-6)
    np.testing.assert_allclose(gh.numpy(), g["hu_grad"], rtol=1e-5, atol=1e-9)
    assert O.hu_loss(a, torch.zeros_like(m), 0.18666666666666668, 0.35333333333333333).item() == g["hu_empty"].item() == 0.0
    assert O.wasserstein_loss(a.detach(), b).item() == pytest.approx(g["wass"].item(), rel=1e-6)
    assert O.wasserstein_loss(a.detach()).item() == pytest.approx(g["wass_fake_only"].item(), rel=1e-6)


def _run_steps(patch, n_steps):
    st = O.StepState(seed=0)
    gen = torch.Generator().manual_seed(1)
    logs = []
    for it in range(n_steps):
        opt = O.synthetic_patches(gen, (2, 1, *patch))
        low = O.synthetic_patches(gen, (1, 1, *patch))
        high = O.synthetic_patches(gen, (1, 1, *patch))
        ml = O.synthetic_masks(gen, (1, 1, *patch))
        mh = O.synthetic_masks(gen, (1, 1, *patch))
        logs.append(O.train_step(st, opt, low, high, ml, mh, it))
    return st, np.array([[l[k] for k in ("D", "G", "G-full", "sim", "HU")] for l in logs])


@pytest.mark.parametrize("name,patch,steps", [("train_steps_32.npz", (32, 32, 32), 3),
                                              ("train_steps_c1_64.npz", (64, 64, 64), 2)])
def test_train_steps_match_reference_trainer(golden_dir, name, patch, steps):
    g = np.load(golden_dir / name)
    st, losses = _run_steps(patch, steps)
    # the critic loss is a difference of nearly equal means: absolute tolerance scaled to the logits
    np.testing.assert_allclose(losses, g["losses"], rtol=2e-4, atol=2e-6)
    for k, v in {**st.gp, **st.gb}.items():
        np.testing.assert_allclose(_fp(v), g["G/" + k], rtol=1e-4, atol=1e-6, err_msg=k)
    for k, v in {**st.dp, **st.db}.items():
        np.testing.assert_allclose(_fp(v), g["D/" + k], rtol=1e-4, atol=1e-6, err_msg=k)


def test_integer_helpers(golden_dir):
    g = np.load(golden_dir / "integer_helpers.npz")
    for row in g["conv_shapes"]:
        dims, (k, p, s, op), want = list(row[:4]), row[4:8], list(row[8:])
        got = O.convolution_output_shape(dims, 5, int(k), int(p), int(s),
                                         transpose_output_padding=None if op < 0 else int(op))
        assert got == want
    assert O.scaler_shift() == int(g["scaler_shift"]) == 238
    np.testing.assert_array_equal(O.scale_hu(g["scaler_in"]), g["scaler_out"])
    np.testing.assert_array_equal(O.unscale_hu(O.scale_hu(g["scaler_in"])), g["unscale"])
    assert list(g["scan_type_order"]) == [0, -1, 1]
    assert list(g["g_out_shape"]) == [1, 128, 128, 128]
    assert list(g["d_out_shape"]) == [1, 7, 7, 7]


def test_aten_primitives_against_naive_restatement():
    rng = np.random.default_rng(0)
    x = rng.standard_normal((2, 3, 7, 6, 5)).astype(np.float32)
    for (k, s, p, mode) in ((3, 1, 1, "zeros"), (3, 2, 1, "zeros"), (4, 2, 1, "zeros"), (5, 1, 2, "reflect")):
        w = rng.standard_normal((4, 3, k, k, k)).astype(np.float32)
        ref = O.naive_conv3d(x, w, s, p, mode)
        xt = torch.from_numpy(x)
        if mode == "reflect":
            xt = torch.nn.functional.pad(xt, (p,) * 6, mode="reflect")
            got = torch.nn.functional.conv3d(xt, torch.from_numpy(w), stride=s)
        else:
            got = torch.nn.functional.conv3d(xt, torch.from_numpy(w), stride=s, padding=p)
        np.testing.assert_allclose(got.numpy(), ref, rtol=1e-4, atol=1e-4)
    wt = rng.standard_normal((3, 4, 3, 3, 3)).astype(np.float32)
    ref = O.naive_conv_transpose3d(x, wt, 2, 1, 1)
    got = torch.nn.functional.conv_transpose3d(torch.from_numpy(x), torch.from_numpy(wt), stride=2, padding=1,
                                               output_padding=1)
    np.testing.assert_allclose(got.numpy(), ref, rtol=1e-4, atol=1e-4)


def test_sampler_index_law():
    rng = np.random.default_rng(3)
    # bigger and smaller than the patch, odd differences
    for shape, patch in (((40, 37, 20), (16, 16, 16)), ((10, 37, 13), (16, 16, 16)), ((16, 16, 16), (16, 16, 16))):
        vol = rng.integers(-1024, 1500, size=(*shape, 2)).astype(np.int16)
        vol[..., 1] = rng.random(shape) < 0.01
        np.random.seed(42)
        data, seg, lbs = O.generate_one(vol, patch)
        assert data.shape == seg.shape == (1, 1, *patch)
        padded_shape, pads = O.pad_nd_image_shape((1, 1, *shape, 2), (*patch, 2))
        assert padded_shape[2:5] == [max(a, b) for a, b in zip(shape, patch)]
        for (lo, hi), s, p in zip(pads[2:5], shape, patch):
            d = max(p - s, 0)
            assert (lo, hi) == (d // 2, d // 2 + d % 2)
        np.random.seed(42)
        want = [int(np.random.randint(0, d - c)) if d - c > 0 else (d - c) // 2 for d, c in zip(padded_shape[2:5], patch)]
        assert lbs == want
        # the last valid offset is never drawn (high-exclusive randint)
        for lb, d, c in zip(lbs, padded_shape[2:5], patch):
            assert lb < max(d - c, 1)
        padded = O.pad_nd_image(vol[None, None], (*patch, 2)).astype(np.float32)
        sl = tuple(slice(lb, lb + c) for lb, c in zip(lbs, patch))
        np.testing.assert_array_equal(data[0, 0], ((padded[0, 0][sl][..., 0] - 238) / 600).astype(np.float32))
        np.testing.assert_array_equal(seg[0, 0], padded[0, 0][sl][..., 1])


def test_grid_tiles_divisible_and_squeeze():
    t = O.grid_tiles((512, 512, 256), (128, 128, 128))
    assert len(t) == 32 and t[0] == (0, 0, 0) and t[1] == (0, 0, 128) and t[2] == (0, 128, 0)
    t = O.grid_tiles((20, 16, 16), (16, 16, 16))
    assert t == [(0, 0, 0), (4, 0, 0)]


def test_oracle_validate_against_reference_golden(golden_dir):
    """Trainer.validate of the unmodified reference (tests/golden/make_golden_validate.py) vs the oracle's restatement."""
    g = np.load(golden_dir / "validate_32.npz")
    st = O.StepState(seed=0)
    gen = torch.Generator().manual_seed(21)
    patch = (32, 32, 32)
    opt = O.synthetic_patches(gen, (2, 1, *patch))
    low = O.synthetic_patches(gen, (1, 1, *patch))
    high = O.synthetic_patches(gen, (1, 1, *patch))
    ml = O.synthetic_masks(gen, (1, 1, *patch))
    mh = O.synthetic_masks(gen, (1, 1, *patch))
    O.train_step(st, opt, low, high, ml, mh, 0)
    vb = [tuple(O.synthetic_patches(gen, (2, 1, 64, 64, 32)) for _ in range(3)) for _ in range(2)]
    got = O.validate(st, vb)
    ref = dict(zip(("D", "G", "sim"), g["val"]))
    for k in ref:
        assert abs(got[k] - ref[k]) <= 1e-4 * abs(ref[k]) + 1e-6, (k, got[k], ref[k])


def test_fp32_multi_step_drift_control_against_fp64():
    """Control run for the multi-step fp32 tolerance of tests/test_gpu_parity.py: the SAME oracle (ATen CPU) in fp32 and in
    fp64 from identical seeded weights and inputs, three full G+D steps at 32^3.

    Step 0 runs from identical weights and agrees to ~1e-6 relative.  From step 1 on the fp32 run has been through Adam,
    whose first updates are lr * sign(g): rounding noise in near-zero gradients flips whole weight updates, and the
    fp32-vs-fp64 loss difference grows by two orders of magnitude.  It uses most of the strict single-step criterion
    |d| <= 1e-4 |ref| + 1e-5 (here: 78 % of it on the HU loss of step 2; asserted > 30 % to allow for other CPUs), so a second, independent fp32
    implementation (another summation order: our CUDA kernels) cannot be held to that criterion after step 0; the GPU tests
    use 5x the strict criterion for the later steps."""
    def run(dt):
        st = O.StepState(seed=0)
        for d in (st.gp, st.gb, st.dp, st.db):
            for k in d:
                if d[k].is_floating_point():
                    d[k] = d[k].to(dt)
        st.opt_g, st.opt_d = O.AdamState(st.gp), O.AdamState(st.dp)
        gen = torch.Generator().manual_seed(1)
        rows = []
        for it in range(3):
            opt, low, high = (O.synthetic_patches(gen, (n, 1, 32, 32, 32)).to(dt) for n in (2, 1, 1))
            ml, mh = (O.synthetic_masks(gen, (1, 1, 32, 32, 32)) for _ in range(2))
            r = O.train_step(st, opt, low, high, ml, mh, it)
            rows.append([r[k] for k in ("D", "G", "G-full", "sim", "HU")])
        return np.array(rows)

    a, b = run(torch.float32), run(torch.float64)
    strict = 1e-4 * np.abs(b) + 1e-5
    use = np.abs(a - b) / strict  # fraction of the strict criterion consumed by fp32 rounding alone
    assert use[0].max() < 0.05, use[0]
    assert use[1:].max() > 0.3, use            # the reference's own arithmetic nearly exhausts the strict criterion ...
    assert use[1:].max() < 5.0, use            # ... and stays inside the relaxed one (5x) used for steps >= 1
    rel = np.abs(a - b) / np.abs(b)
    assert rel[1:].max() > 20 * rel[0].max(), rel  # the drift is produced by the optimizer steps, not by one forward pass


@pytest.mark.parametrize("name,norm", [("train_steps_gp_32.npz", "identity"), ("train_steps_gp_layernorm_32.npz", "layer")])
def test_wgan_gp_train_steps_against_reference_golden(golden_dir, name, norm):
    """WGAN-GP mode (weight_clip=None): oracle vs the reference Trainer's logged losses and post-step weights for the
    Identity-norm critic (gradient_penalty_conf.py) and the LayerNorm critic (gp_layernorm.py)."""
    g = np.load(golden_dir / name)
    st = O.StepState(seed=0, lr=1e-4, betas=(0.0, 0.9), d_layers=O.critic_layers(norm=norm))
    assert O.state_dict_order(st.d_layers) == list(g["D_keys"])
    gen = torch.Generator().manual_seed(1)
    rows = []
    for it in range(3):
        opt, low, high = (O.synthetic_patches(gen, (n, 1, 32, 32, 32)) for n in (2, 1, 1))
        ml, mh = (O.synthetic_masks(gen, (1, 1, 32, 32, 32)) for _ in range(2))
        torch.manual_seed(9000 + it)
        eps = torch.rand((2, 1, 1, 1, 1))
        r = O.train_step(st, opt, low, high, ml, mh, it, weight_clip=None, gp_eps=eps)
        rows.append([r[k] for k in ("D", "G", "G-full", "sim", "HU")])
    np.testing.assert_allclose(np.array(rows), g["losses"], rtol=2e-5, atol=2e-6)
    for prefix, d in (("G/", {**st.gp, **st.gb}), ("D/", {**st.dp, **st.db})):
        for k, v in d.items():
            np.testing.assert_allclose(_fp(v), g[prefix + k], rtol=1e-4, atol=1e-6, err_msg=k)


def test_wgan_gp_fp32_drift_control_against_fp64():
    """Control for the multi-step fp32 bound of the WGAN-GP GPU tests: the oracle (ATen CPU) in fp32 vs fp64 from the same
    seeded state, LayerNorm critic.  With Adam(beta1 = 0) and a LayerNorm critic ATen's own rounding noise grows to tens of
    times the strict single-step criterion |d| <= 1e-4 |ref| + 1e-5 within three steps (53x on the generator's adversarial
    loss here), so an independent fp32 implementation is held to 100x that criterion after step 0 in this configuration."""
    def run(dt):
        st = O.StepState(seed=0, lr=1e-4, betas=(0.0, 0.9), d_layers=O.critic_layers(norm="layer"))
        for d in (st.gp, st.gb, st.dp, st.db):
            for k in d:
                if d[k].is_floating_point():
                    d[k] = d[k].to(dt)
        st.opt_g, st.opt_d = O.AdamState(st.gp, 1e-4, (0.0, 0.9)), O.AdamState(st.dp, 1e-4, (0.0, 0.9))
        gen = torch.Generator().manual_seed(1)
        rows = []
        for it in range(3):
            opt, low, high = (O.synthetic_patches(gen, (n, 1, 32, 32, 32)).to(dt) for n in (2, 1, 1))
            ml, mh = (O.synthetic_masks(gen, (1, 1, 32, 32, 32)) for _ in range(2))
            torch.manual_seed(9000 + it)
            eps = torch.rand((2, 1, 1, 1, 1)).to(dt)
            r = O.train_step(st, opt, low, high, ml, mh, it, weight_clip=None, gp_eps=eps)
            rows.append([r[k] for k in ("D", "G", "G-full", "sim", "HU")])
        return np.array(rows)

    a, b = run(torch.float32), run(torch.float64)
    use = np.abs(a - b) / (1e-4 * np.abs(b) + 1e-5)
    assert use[0].max() < 0.05, use[0]
    assert 5.0 < use[2].max() < 100.0, use


def test_oracle_rmsprop_matches_torch_rmsprop():
    """The oracle's RMSprop (experiments/rmsprop_conf.py:8-9 constructs torch.optim.RMSprop(lr=lr)) against torch itself."""
    torch.manual_seed(0)
    p = {"a": torch.randn(50)}
    q = p["a"].clone().requires_grad_(True)
    opt = torch.optim.RMSprop([q], lr=2e-4)
    st = O.RMSpropState(p, 2e-4)
    for i in range(4):
        g = torch.randn(50) * 10.0 ** (i - 2)
        q.grad = g.clone()
        opt.step()
        st.apply(p, {"a": g})
    assert torch.equal(p["a"], q.detach())
