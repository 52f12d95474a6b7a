"""img2img (SDEdit) and latent-blend inpainting on the DDIM sampler (DESIGN.md §7 row f5; definition in
oracle/img2img_oracle.py). CPU: the oracle against its fixture and its own invariants. GPU: the CUDA path through the C ABI
against the fixture, bit for bit against text-to-image, and its launch / graph-cache / error behaviour."""
import math
import os

import numpy as np
import pytest
import torch

from stable_diffusion_burn_b200 import synth, topology

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "img2img.npz")


def rel(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def small_inputs(n=1, seed=0):
    """64x64 images (latent 8x8, the smallest encoder size): cheap enough for the CPU oracle."""
    g = np.random.Generator(np.random.Philox(500 + seed))
    rgb = g.integers(0, 256, (n, 64, 64, 3), dtype=np.uint8)
    return rgb, synth.make_context(n, 5, seed=8), synth.make_context(1, 2, seed=99)[0], synth.make_latent(n, 8, 8, seed=61)


# ------------------------------------------------------------------------------------------------ CPU
@pytest.fixture(scope="module")
def P():
    from oracle import sd_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    return O.Params(synth.make_params(0, which=topology.unet_params() + topology.vae_encoder_params()))


def test_oracle_rederives_fixture(P):
    from oracle import img2img_oracle as I
    g = np.load(GOLD)
    x0 = I.encode_x0(P, g["rgb"])
    assert np.allclose(x0, g["x0"], rtol=0, atol=2e-5 * np.abs(g["x0"]).max())
    for case, mask in (("plain", None), ("masked", g["mask"])):
        want = g[f"latent:{case}"]
        lat = I.img2img_latent(P, g["rgb"], g["context"], g["uncond"], float(g["scale"]), int(g["n_steps"]), float(g["strength"]),
                               g["noise"], mask=mask, x0=g["x0"])
        assert np.allclose(lat, want, rtol=0, atol=2e-5 * np.abs(want).max()), case
    # the kept cells of the masked case are x0 itself
    keep = I.latent_mask(g["mask"])[:, None].repeat(4, 1) == 0
    assert np.array_equal(g["latent:masked"][keep], g["x0"][keep])


def test_mask_all_ones_is_no_mask_and_all_zeros_is_x0(P):
    from oracle import img2img_oracle as I
    rgb, c, u, noise = small_inputs()
    x0 = I.encode_x0(P, rgb)
    plain = I.img2img_latent(P, rgb, c, u, 7.5, 2, 1.0, noise, x0=x0)
    ones = I.img2img_latent(P, rgb, c, u, 7.5, 2, 1.0, noise, mask=np.ones((1, 64, 64), np.uint8), x0=x0)
    zeros = I.img2img_latent(P, rgb, c, u, 7.5, 2, 1.0, noise, mask=np.zeros((1, 64, 64), np.uint8), x0=x0)
    assert np.array_equal(plain, ones)
    assert np.array_equal(zeros, x0)
    assert not np.array_equal(plain, x0)


def test_strength_zero_returns_x0(P):
    from oracle import img2img_oracle as I
    rgb, c, u, noise = small_inputs()
    x0 = I.encode_x0(P, rgb)
    assert np.array_equal(I.img2img_latent(P, rgb, c, u, 7.5, 20, 0.0, noise, x0=x0), x0)
    assert np.array_equal(I.img2img_latent(P, rgb, c, u, 7.5, 20, 0.04, noise, x0=x0), x0)  # floor(0.8) = 0 steps


def test_latent_mask_is_8x8_max_pool():
    from oracle import img2img_oracle as I
    mask = np.zeros((3, 64, 128), np.uint8)
    mask[0, :, :64] = 1
    mask[1, 13:30, 37:101] = 200  # edges off the 8-pixel grid
    mask[2, 63, 127] = 1          # one pixel in the last block
    want = np.zeros((3, 8, 16), np.uint8)
    for n in range(3):
        for y in range(8):
            for x in range(16):
                want[n, y, x] = 1 if mask[n, 8 * y:8 * y + 8, 8 * x:8 * x + 8].any() else 0
    got = I.latent_mask(mask)
    assert got.dtype == np.uint8 and np.array_equal(got, want)
    assert want[1, 1, 4] == 1 and want[1, 3, 12] == 1 and want[1, 4, 4] == 0  # rows 8..15 touched by 13, cols 96..103 by 100


@pytest.mark.parametrize("strength,n_steps,i0", [
    (0.5, 4, 2), (1.0, 4, 0), (0.75, 20, 5), (0.0, 20, 20),
    (1.0, 3, 0), (0.75, 3, 1), (0.3, 3, 3), (0.5, 3, 2),  # n_steps = 3: T = 4 (999, 666, 333, 0)
    (0.29, 100, 71),  # 0.29 * 100 = 28.999999999999996: the 1e-9 keeps it at 29 steps
    (0.999, 1, 1), (0.7, 10, 3),
])
def test_n_run_rounding(strength, n_steps, i0):
    from oracle import img2img_oracle as I
    ts, step, got = I.img2img_schedule(n_steps, strength)
    assert got == i0, (strength, n_steps, got)
    assert len(ts) - got == min(len(ts), math.floor(strength * len(ts) + 1e-9))


def test_image_from_rgb8():
    from oracle import img2img_oracle as I
    v = np.arange(256, dtype=np.uint8).reshape(1, 16, 16, 1).repeat(3, -1)
    x = I.image_from_rgb8(v)
    assert x.shape == (1, 3, 16, 16) and x.dtype == np.float32
    assert x[0, 0, 0, 0] == -1.0 and x[0, 0, 15, 15] == 1.0
    assert np.abs(x[0, 1].reshape(-1) - (np.arange(256) / 127.5 - 1)).max() < 1e-6


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def sd(ctx):
    ctx.init_synthetic(0)
    ctx.finalize_weights()
    return ctx


def _x0_gpu(sd, rgb):
    """0.18215f x sdb_encode_image(image_from_rgb8(rgb)) in numpy fp32: the x0 the img2img path must compute."""
    from oracle import img2img_oracle as I
    return sd.encode_image(I.image_from_rgb8(rgb)) * np.float32(0.18215)


def _u8_ok(got, want, region):
    d = np.abs(got.astype(np.int16) - want.astype(np.int16))[region]
    return float((d <= 1).mean()), int(d.max())


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["plain", "masked"])
def test_fixture_parity(sd, case):
    g = np.load(GOLD)
    mask = g["mask"] if case == "masked" else None
    lat, rgb = sd.img2img(g["context"], g["uncond"], float(g["scale"]), int(g["n_steps"]), g["rgb"], float(g["strength"]),
                          mask=mask, noise=g["noise"])
    want = g[f"latent:{case}"]
    if mask is None:
        e = rel(lat, want)
        region = np.ones(g[f"u8_sub:{case}"].shape, bool)
    else:
        from oracle import img2img_oracle as I
        rep = I.latent_mask(mask)[:, None].repeat(4, 1) != 0
        e = rel(lat[rep], want[rep])
        region = np.broadcast_to((mask[:, ::2, ::2] != 0)[..., None], g[f"u8_sub:{case}"].shape)
    frac, dmax = _u8_ok(rgb[:, ::2, ::2, :], g[f"u8_sub:{case}"], region)
    print(f"img2img {case}: latent rel L2 {e:.3e}; u8 within 1 LSB {frac:.5f}, max diff {dmax}")
    assert e <= 2e-3
    assert frac >= 0.998 and dmax <= 4


@pytest.mark.gpu
@pytest.mark.parametrize("graphs", [1, 0])
def test_strength_one_is_text_to_image_bit_for_bit(sd, graphs):
    """img2img at strength 1 without a mask = sample_latent from x_T = fl(fl(a x0) + fl(b eps)) at t = 999, computed in numpy."""
    g = np.load(GOLD)
    x0 = _x0_gpu(sd, g["rgb"])
    alpha = float(sd.get_tensor("alpha_cumulative_products", (1000,))[999])
    xT = np.float32(math.sqrt(alpha)) * x0 + np.float32(math.sqrt(1.0 - alpha)) * g["noise"]
    sd.set_option("graphs", graphs)
    try:
        lat, _ = sd.img2img(g["context"], g["uncond"], 5.0, 2, g["rgb"], 1.0, noise=g["noise"], image=False)
        want = sd.sample_latent(g["context"], g["uncond"], 5.0, 2, init_latent=xT)
    finally:
        sd.set_option("graphs", 1)
    assert np.isfinite(lat).all() and np.array_equal(lat, want)


@pytest.mark.gpu
def test_masked_keeps_known_cells_and_pixels(sd):
    from oracle import img2img_oracle as I
    g = np.load(GOLD)
    x0 = _x0_gpu(sd, g["rgb"])
    lat, rgb = sd.img2img(g["context"], g["uncond"], 5.0, 4, g["rgb"], 0.5, mask=g["mask"], noise=g["noise"])
    keep = I.latent_mask(g["mask"])[:, None].repeat(4, 1) == 0
    assert np.array_equal(lat[keep], x0[keep])
    assert (lat[~keep] != x0[~keep]).any()
    kept_px = g["mask"] == 0
    assert np.array_equal(rgb[kept_px], g["rgb"][kept_px])


@pytest.mark.gpu
def test_graph_cache_is_not_disturbed(sd):
    g = np.load(GOLD)
    init = synth.make_latent(2, 32, 32, seed=5)
    a = sd.sample_latent(g["context"], g["uncond"], 5.0, 4, init_latent=init)
    sd.img2img(g["context"], g["uncond"], 5.0, 4, g["rgb"], 0.5, mask=g["mask"], noise=g["noise"])
    b = sd.sample_latent(g["context"], g["uncond"], 5.0, 4, init_latent=init)
    assert np.array_equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("masked", [False, True])
def test_launch_accounting(sd, masked):
    """Each step of img2img issues the launches of a text-to-image step, with or without a mask; strength 0 runs no UNet."""
    g = np.load(GOLD)
    mask = g["mask"] if masked else None

    def count(fn):
        before = sd.launch_count()
        fn()
        return sd.launch_count() - before

    i2i = lambda s: count(lambda: sd.img2img(g["context"], g["uncond"], 5.0, 4, g["rgb"], s, mask=mask, noise=g["noise"],
                                             image=False))
    t2i = lambda steps: count(lambda: sd.sample_latent(g["context"], g["uncond"], 5.0, steps, init_latent=g["noise"]))
    i2i(1.0), t2i(4)  # the step graph of this shape exists before anything is counted
    d_i2i = i2i(1.0) - i2i(0.5)
    d_t2i = t2i(4) - t2i(2)
    assert d_i2i == d_t2i and d_t2i > 0, (d_i2i, d_t2i)
    step = t2i(2) - t2i(1)
    assert i2i(0.25) - i2i(0.0) >= step  # one step (T = 4, n_run = 1) against none: a whole UNet pass


@pytest.mark.gpu
def test_seeded_noise_and_batch_invariance(sd):
    g = np.load(GOLD)
    run = lambda sl, **kw: sd.img2img(g["context"][sl], g["uncond"], 5.0, 4, g["rgb"][sl], 0.5, image=False, **kw)[0]
    a, b, c = run(slice(0, 2), seed=7), run(slice(0, 2), seed=7), run(slice(0, 2), seed=8)
    assert np.array_equal(a, b) and not np.array_equal(a, c)
    assert rel(run(slice(0, 1), seed=7), a[0:1]) < 1e-3  # image 0 draws the first elements of the seeded stream
    both = run(slice(0, 2), noise=g["noise"])
    for i in range(2):
        one = run(slice(i, i + 1), noise=g["noise"][i:i + 1])
        assert rel(both[i:i + 1], one) < 1e-3, i


@pytest.mark.gpu
def test_error_paths(sd):
    from stable_diffusion_burn_b200._lib import SdbError
    g = np.load(GOLD)
    args = (g["context"], g["uncond"], 5.0, 4)
    for s in (-0.1, 1.5, float("nan")):
        with pytest.raises(SdbError, match="strength"):
            sd.img2img(*args, g["rgb"], s)
    with pytest.raises(SdbError, match="both null"):
        sd.img2img(*args, g["rgb"], 0.5, latent=False, image=False)
    with pytest.raises(SdbError):  # 264 px: latent 33, not a multiple of 8
        sd.img2img(*args, np.zeros((2, 264, 256, 3), np.uint8), 0.5)
    with pytest.raises(SdbError):  # 128 px: latent 16, the UNet's deepest level would have 4 tokens
        sd.img2img(*args, np.zeros((2, 128, 128, 3), np.uint8), 0.5)
    with pytest.raises(SdbError, match="n_steps"):
        sd.img2img(g["context"], g["uncond"], 5.0, 0, g["rgb"], 0.5)
    # the context is still usable after the failures
    lat, _ = sd.img2img(*args, g["rgb"], 0.0, noise=g["noise"], image=False)
    assert np.array_equal(lat, _x0_gpu(sd, g["rgb"]))
