"""Selectable samplers: DDIM with eta in [0, 1] and DPM-Solver++(2M) on the reference's schedule (DESIGN.md §7 row f6; definition
in oracle/sampler_oracle.py). CPU: the oracle against its fixture, against the exact solution of a Gaussian toy, and its own
invariants. GPU: the CUDA path through the C ABI against the fixture, step for step against a numpy f32 replay of the update
kernels, and its noise / launch / graph-cache / error behaviour."""
import math
import os

import numpy as np
import pytest
import torch

from stable_diffusion_burn_b200 import synth, topology

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "sampler.npz")
CASES = {"dpmpp_2m": ("dpmpp_2m", 0.0), "ddim_eta1": ("ddim", 1.0)}


def rel(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


# ------------------------------------------------------------------------------------------------ CPU
@pytest.fixture(scope="module")
def P():
    from oracle import sd_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    return O.Params(synth.make_params(0, which=topology.unet_params()))


def test_oracle_rederives_fixture(P):
    from oracle import sampler_oracle as S
    g = np.load(GOLD)
    for case, (sampler, eta) in CASES.items():
        want = g[f"latent:{case}"]
        lat = S.sample_latent(P, g["context"], g["uncond"], float(g["scale"]), int(g["n_steps"]), torch.from_numpy(g["init_latent"]),
                              sampler, eta=eta, step_noise=g["step_noise"] if eta > 0 else None).numpy()
        assert np.allclose(lat, want, rtol=0, atol=2e-5 * np.abs(want).max()), case


# Gaussian toy with an exact noise prediction: data ~ N(mu, s^2), eps(x, t) = sqrt(1-a) (x - sqrt(a) mu) / (a s^2 + 1 - a).
# The probability-flow ODE moves xbar = x / sqrt(a) as xbar - mu ∝ sqrt(s^2 + sigma^2), sigma^2 = (1 - a) / a.
MU, SD = 0.7, 0.3
ALPHAS = synth.alpha_cumulative_products()


def _toy_eps(x, t):
    a = float(ALPHAS[t])
    return math.sqrt(1.0 - a) * (x - math.sqrt(a) * MU) / (a * SD * SD + 1.0 - a)


def _toy_exact(xT, aT, a):
    scale = math.sqrt(SD * SD + (1.0 - a) / a) / math.sqrt(SD * SD + (1.0 - aT) / aT)
    return math.sqrt(a) * (MU + (xT / math.sqrt(aT) - MU) * scale)


def _toy_errors(sampler, n_steps):
    """-> (rel error of the latent before the last step, rel error of the result) against the exact solution."""
    from oracle import sampler_oracle as S
    ts, _ = S.O.ddim_timesteps(n_steps)
    aT, a_last = float(ALPHAS[ts[0]]), float(ALPHAS[ts[-1]])
    g = np.random.default_rng(0)
    xT = torch.from_numpy(math.sqrt(aT) * MU + math.sqrt(aT * SD * SD + 1.0 - aT) * g.standard_normal(4096))
    taps = {}
    out = S.sample_latent(None, None, None, 1.0, n_steps, xT, sampler, taps=taps, eps_fn=_toy_eps, alphas=ALPHAS)
    before = taps[f"step{len(ts) - 2}/latent"]
    return rel(before, _toy_exact(xT, aT, a_last)), rel(out, _toy_exact(xT, aT, 1.0))


def test_gaussian_toy_dpmpp_2m_beats_ddim():
    """Measured (4096 samples, mu 0.7, s 0.3), before the last step / result: N=5 2.5e-2 vs 1.2e-2 / 0.218 vs 0.214;
    N=10 2.5e-2 vs 5.5e-3 / 0.146 vs 0.136; N=20 2.1e-2 vs 9.0e-4 / 9.1e-2 vs 7.7e-2; N=50 1.4e-2 vs 1.5e-3 / 4.6e-2 vs 3.3e-2.
    The final jump to sigma = 0 (a first-order step for both) dominates the result."""
    for n in (5, 10, 20, 50):
        (d_before, d_final), (p_before, p_final) = _toy_errors("ddim", n), _toy_errors("dpmpp_2m", n)
        assert p_before < d_before, (n, p_before, d_before)
        if n == 5:
            assert p_final <= 1.02 * d_final, (n, p_final, d_final)
        else:
            assert p_final < d_final, (n, p_final, d_final)
        if n == 20:
            assert p_before * 5 <= d_before, (p_before, d_before)


def test_dpmpp_2m_step0_is_ddim_step0():
    """The first-order DPM-Solver++ step is DDIM: (s_n/s_t) x - alpha_n expm1(-h) x0 = alpha_n x0 + s_n pred."""
    from oracle import sampler_oracle as S
    x = torch.from_numpy(np.random.default_rng(1).standard_normal(512))
    for n_steps in (3, 10, 50):
        t_d, t_p = {}, {}
        S.sample_latent(None, None, None, 1.0, n_steps, x, "ddim", taps=t_d, eps_fn=_toy_eps, alphas=ALPHAS)
        S.sample_latent(None, None, None, 1.0, n_steps, x, "dpmpp_2m", taps=t_p, eps_fn=_toy_eps, alphas=ALPHAS)
        assert torch.allclose(t_p["step0/latent"], t_d["step0/latent"], rtol=1e-12, atol=1e-12), n_steps
        assert not torch.allclose(t_p["step1/latent"], t_d["step1/latent"], rtol=1e-6, atol=0)  # second order from step 1


def test_ddim_eta0_is_sd_oracle_sample_latent(monkeypatch):
    """With eta = 0 the DDIM sampler is sd_oracle.sample_latent (the reference's loop) exactly; a cheap stand-in for
    forward_diffuser keeps the UNet out of it."""
    from oracle import sampler_oracle as S
    from oracle import sd_oracle as O
    monkeypatch.setattr(O, "forward_diffuser", lambda P, x, t, c, u, scale, taps=None: torch.tanh(x * (1.0 + t / 1000.0)) * scale)
    P = O.Params({"alpha_cumulative_products": ALPHAS})
    x = torch.from_numpy(synth.make_latent(2, 8, 8, seed=3))
    for n_steps in (1, 4, 20):
        want = O.sample_latent(P, None, None, 0.8, n_steps, x)
        got = S.sample_latent(P, np.zeros((2, 1, 768), np.float32), np.zeros((1, 768), np.float32), 0.8, n_steps, x, "ddim")
        assert torch.equal(got, want), n_steps


@pytest.mark.parametrize("n_steps", [1, 2, 4, 20, 50, 333, 1000])
def test_sigma_vanishes_at_the_last_step(n_steps):
    from oracle import sampler_oracle as S
    ks = S.coeffs("ddim", ALPHAS, n_steps, eta=1.0)
    assert ks[-1]["sigma"] == 0.0
    assert all(k["sigma"] > 0 for k in ks[:-1])
    for k, (_, a_t, a_next) in zip(ks, S.schedule(ALPHAS, n_steps)):
        assert abs(k["dir"] ** 2 + k["sigma"] ** 2 + a_next - 1.0) < 1e-12
        assert k["sigma"] ** 2 <= 1.0 - a_next + 1e-15
    assert all(k["sigma"] == 0.0 for k in S.coeffs("ddim", ALPHAS, n_steps, eta=0.0))
    dk = S.coeffs("dpmpp_2m", ALPHAS, n_steps)
    assert dk[-1]["kind"] == "final" and all(k["kind"] == "second" for k in dk[1:-1])
    assert len(dk) == 1 or dk[0]["kind"] == "first"


def test_update_f32_agrees_with_f64_math():
    from oracle import sampler_oracle as S
    g = np.random.default_rng(2)
    x, u, c, z, prev = (g.standard_normal(4096).astype(np.float32) for _ in range(5))
    scale = 5.0
    x64, u64, c64, z64, p64 = (v.astype(np.float64) for v in (x, u, c, z, prev))
    pred = u64 + (c64 - u64) * scale
    for k in S.coeffs("ddim", ALPHAS, 10, eta=1.0):
        x0 = (x64 - pred * k["sqrt_1m_at"]) / k["sqrt_at"]
        want = x0 * k["sqrt_anext"] + pred * k["dir"] + k["sigma"] * z64
        got = S.ddim_update_f32(x, u, c, scale, k, z)
        assert got.dtype == np.float32 and rel(got, want) < 1e-5
    for k in S.coeffs("dpmpp_2m", ALPHAS, 10):
        x0 = (x64 - pred * k["sqrt_1m_at"]) / k["sqrt_at"]
        if k["kind"] == "final":
            want = x0
        else:
            D = x0 if k["kind"] == "first" else (1 + k["w1"]) * x0 - k["w1"] * p64
            want = x64 * k["ratio"] - D * k["coef"]
        got, got_x0 = S.dpmpp_2m_update_f32(x, u, c, scale, k, prev)
        assert got.dtype == np.float32 and rel(got, want) < 1e-5 and rel(got_x0, x0) < 1e-5, k["kind"]


def test_step_seed():
    from oracle import sampler_oracle as S
    assert S.step_seed(0, 0) == 0x9E3779B97F4A7C15
    assert S.step_seed(5, 1) == 5 ^ ((2 * 0x9E3779B97F4A7C15) % 2 ** 64)
    assert S.step_seed(2 ** 64 - 1, 2) == (2 ** 64 - 1) ^ ((3 * 0x9E3779B97F4A7C15) % 2 ** 64)
    assert len({S.step_seed(7, i) for i in range(1000)}) == 1000


def test_oracle_argument_rules():
    from oracle import sampler_oracle as S
    x = torch.zeros(4, dtype=torch.float64)
    run = lambda sampler, **kw: S.sample_latent(None, None, None, 1.0, 4, x, sampler, eps_fn=_toy_eps, alphas=ALPHAS, **kw)
    for bad in (dict(sampler="euler"), dict(sampler="ddim", eta=1.5), dict(sampler="ddim", eta=float("nan")),
                dict(sampler="ddim", eta=0.5), dict(sampler="ddim", step_noise=np.zeros((4, 4))),
                dict(sampler="dpmpp_2m", step_noise=np.zeros((4, 4)))):
        with pytest.raises(ValueError):
            run(**bad)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def sd(ctx):
    ctx.init_synthetic(0)
    ctx.finalize_weights()
    return ctx


def _sample(sd, g, case, **kw):
    sampler, eta = CASES[case]
    args = dict(init_latent=g["init_latent"], step_noise=g["step_noise"] if eta > 0 else None)
    args.update(kw)
    return sd.sample_ex(g["context"], g["uncond"], float(g["scale"]), int(g["n_steps"]), sampler=sampler, eta=eta, **args)[0]


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_fixture_parity(sd, case):
    g = np.load(GOLD)
    lat = _sample(sd, g, case)
    e = rel(lat, g[f"latent:{case}"])
    print(f"sampler {case}: latent rel L2 {e:.3e}")
    assert e <= 2e-3


@pytest.mark.gpu
@pytest.mark.parametrize("graphs", [1, 0])
@pytest.mark.parametrize("case", list(CASES))
def test_exact_step_replay(sd, case, graphs):
    """The chain driven from the same initial latent by sdb_forward_diffuser's two UNet outputs (the batch-2n pass the loop
    replays) and the numpy f32 update of oracle/sampler_oracle.py equals sample_ex bit for bit."""
    from oracle import sampler_oracle as S
    g = np.load(GOLD)
    sampler, eta = CASES[case]
    scale, n_steps = float(g["scale"]), int(g["n_steps"])
    alphas = sd.get_tensor("alpha_cumulative_products", (1000,))
    sd.set_option("graphs", graphs)
    try:
        got = _sample(sd, g, case)
        x, prev = g["init_latent"].copy(), None
        for i, ((t, _, _), k) in enumerate(zip(S.schedule(alphas, n_steps), S.coeffs(sampler, alphas, n_steps, eta))):
            _, u, c = sd.forward_diffuser(x, t, g["context"], g["uncond"], scale)
            if sampler == "ddim":
                x = S.ddim_update_f32(x, u, c, scale, k, g["step_noise"][i])
            else:
                x, prev = S.dpmpp_2m_update_f32(x, u, c, scale, k, prev)
    finally:
        sd.set_option("graphs", 1)
    assert np.isfinite(got).all()
    diff = np.abs(got.astype(np.float64) - x)
    assert np.array_equal(got, x), f"{int((diff > 0).sum())} elements differ, max {diff.max():.3e}"


@pytest.mark.gpu
def test_ddim_eta0_is_sample_latent_bit_for_bit(sd):
    g = np.load(GOLD)
    want = sd.sample_latent(g["context"], g["uncond"], 5.0, 4, init_latent=g["init_latent"])
    got = sd.sample_ex(g["context"], g["uncond"], 5.0, 4, "ddim", 0.0, init_latent=g["init_latent"])[0]
    assert np.array_equal(got, want)
    seeded = sd.sample_ex(g["context"], g["uncond"], 5.0, 4, "ddim", 0.0, seed=11, H=32, W=32)[0]
    assert np.array_equal(seeded, sd.sample_latent(g["context"], g["uncond"], 5.0, 4, seed=11, H=32, W=32))


@pytest.mark.gpu
def test_seeded_noise_streams(sd):
    from oracle import sampler_oracle as S
    g = np.load(GOLD)
    n, le, T = 2, 2 * 4 * 32 * 32, 4
    # sdb_randn is an element-wise stream, and it is the initial latent of sample_latent
    r = sd.randn(42, le)
    assert np.array_equal(sd.randn(42, 100), r[:100]) and abs(float(r.mean())) < 0.05 and abs(float(r.std()) - 1) < 0.05
    lat = lambda **kw: sd.sample_latent(g["context"], g["uncond"], 5.0, 4, H=32, W=32, **kw)
    assert np.array_equal(lat(seed=42), lat(init_latent=r.reshape(n, 4, 32, 32)))
    # the in-kernel draw of DDIM eta > 0 is slice i = sdb_randn(seed_i) of an explicit step_noise
    run = lambda **kw: sd.sample_ex(g["context"], g["uncond"], 5.0, 4, "ddim", 1.0, H=32, W=32, **kw)[0]
    noise = np.stack([sd.randn(S.step_seed(42, i), le) for i in range(T)]).reshape(T, n, 4, 32, 32)
    internal = run(seed=42)
    assert np.array_equal(internal, run(seed=42, step_noise=noise))
    assert np.array_equal(internal, run(init_latent=r.reshape(n, 4, 32, 32), step_noise=noise))
    assert np.array_equal(internal, run(seed=42)) and not np.array_equal(internal, run(seed=43))
    # eta scales the noise: eta = 1 differs from eta = 0 from the same initial latent
    assert not np.array_equal(internal, lat(seed=42))


@pytest.mark.gpu
def test_launch_accounting(sd):
    """Each step issues the launches of a DDIM step whatever the sampler: the UNet graph and one update kernel."""
    g = np.load(GOLD)

    def count(sampler, eta, steps):
        before = sd.launch_count()
        sd.sample_ex(g["context"], g["uncond"], 5.0, steps, sampler, eta, init_latent=g["init_latent"])
        return sd.launch_count() - before

    for s, e in (("ddim", 0.0), ("ddim", 1.0), ("dpmpp_2m", 0.0)):
        count(s, e, 4)  # the step graph of this shape exists before anything is counted
    d = {(s, e): count(s, e, 4) - count(s, e, 2) for s, e in (("ddim", 0.0), ("ddim", 1.0), ("dpmpp_2m", 0.0))}
    assert len(set(d.values())) == 1 and min(d.values()) > 0, d


@pytest.mark.gpu
def test_graph_cache_is_not_disturbed(sd):
    g = np.load(GOLD)
    a = sd.sample_latent(g["context"], g["uncond"], 5.0, 4, init_latent=g["init_latent"])
    _sample(sd, g, "dpmpp_2m")
    b = sd.sample_latent(g["context"], g["uncond"], 5.0, 4, init_latent=g["init_latent"])
    _sample(sd, g, "ddim_eta1")
    c = sd.sample_latent(g["context"], g["uncond"], 5.0, 4, init_latent=g["init_latent"])
    assert np.array_equal(a, b) and np.array_equal(a, c)


@pytest.mark.gpu
def test_batch_invariance(sd):
    g = np.load(GOLD)
    both = _sample(sd, g, "dpmpp_2m")
    for i in range(2):
        one = sd.sample_ex(g["context"][i:i + 1], g["uncond"], 5.0, 4, "dpmpp_2m", init_latent=g["init_latent"][i:i + 1])[0]
        assert rel(both[i:i + 1], one) < 1e-3, i


@pytest.mark.gpu
def test_pipeline_keywords(sd):
    """StableDiffusion.sample_latent / sample_image take sampler / eta / step_noise; the defaults stay on sdb_sample_latent."""
    from stable_diffusion_burn_b200.pipeline import StableDiffusion
    g = np.load(GOLD)
    pipe = StableDiffusion.__new__(StableDiffusion)
    pipe.ctx = sd
    kw = dict(init_latent=g["init_latent"], height=256, width=256)
    assert np.array_equal(pipe.sample_latent(g["context"], g["uncond"], 5.0, 4, **kw),
                          sd.sample_latent(g["context"], g["uncond"], 5.0, 4, init_latent=g["init_latent"]))
    assert np.array_equal(pipe.sample_latent(g["context"], g["uncond"], 5.0, 4, sampler="dpmpp_2m", **kw), _sample(sd, g, "dpmpp_2m"))
    assert np.array_equal(pipe.sample_latent(g["context"], g["uncond"], 5.0, 4, sampler="ddim", eta=1.0, step_noise=g["step_noise"],
                                             **kw), _sample(sd, g, "ddim_eta1"))
    imgs = pipe.sample_image(g["context"], g["uncond"], 5.0, 4, sampler="dpmpp_2m", **kw)
    want = sd.latent_to_image(_sample(sd, g, "dpmpp_2m"))
    assert len(imgs) == 2 and np.array_equal(np.stack(imgs), want.reshape(2, -1))


@pytest.mark.gpu
def test_error_paths(sd):
    from stable_diffusion_burn_b200._lib import SdbError
    g = np.load(GOLD)
    args = (g["context"], g["uncond"], 5.0, 4)
    kw = dict(init_latent=g["init_latent"])
    with pytest.raises(SdbError, match="unknown sampler"):
        sd.sample_ex(*args, 7, **kw)
    with pytest.raises(ValueError):
        sd.sample_ex(*args, "euler", **kw)
    for eta in (-0.1, 1.5, float("nan")):
        with pytest.raises(SdbError, match="eta must lie"):
            sd.sample_ex(*args, "ddim", eta, **kw)
    with pytest.raises(SdbError, match="eta applies to DDIM only"):
        sd.sample_ex(*args, "dpmpp_2m", 0.5, **kw)
    for sampler, eta in (("ddim", 0.0), ("dpmpp_2m", 0.0)):
        with pytest.raises(SdbError, match="step_noise"):
            sd.sample_ex(*args, sampler, eta, step_noise=g["step_noise"], **kw)
    with pytest.raises(SdbError, match="both null"):
        sd.sample_ex(*args, "dpmpp_2m", latent=False, image=False, **kw)
    with pytest.raises(SdbError, match="n_steps"):
        sd.sample_ex(g["context"], g["uncond"], 5.0, 0, "dpmpp_2m", **kw)
    with pytest.raises(SdbError):  # latent 33: not a multiple of 8
        sd.sample_ex(*args, "dpmpp_2m", H=33, W=32)
    # the context is still usable after the failures
    assert np.array_equal(_sample(sd, g, "dpmpp_2m"), _sample(sd, g, "dpmpp_2m"))
    assert rel(_sample(sd, g, "dpmpp_2m"), g["latent:dpmpp_2m"]) <= 2e-3
