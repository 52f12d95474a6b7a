"""CPU suite: pins the oracle (against the committed fixtures it generated and against library forms of the
same ops), the host logic (topology, synthetic stream, DDIM schedule), and the C ABI surface."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import sd_oracle as O
from stable_diffusion_burn_b200 import _lib, synth, topology

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def P():
    torch.set_num_threads(os.cpu_count() or 1)
    return O.Params(synth.make_params(0))


# ------------------------------------------------------------------ oracle formulas == library forms
def test_groupnorm_matches_library():
    x = torch.randn(2, 64, 5, 7)
    g = torch.rand(64) + 0.5
    b = torch.randn(64)
    Pm = O.Params({"n/weight": g.numpy(), "n/bias": b.numpy()})
    assert torch.allclose(O.group_norm(Pm, "n", x), F.group_norm(x, 32, g, b, 1e-5), atol=2e-6)


def test_attention_matches_sdpa():
    q, k, v = torch.randn(2, 50, 64), torch.randn(2, 9, 64), torch.randn(2, 9, 64)
    ref = F.scaled_dot_product_attention(q.view(2, 50, 4, 16).transpose(1, 2), k.view(2, 9, 4, 16).transpose(1, 2),
                                         v.view(2, 9, 4, 16).transpose(1, 2)).transpose(1, 2).reshape(2, 50, 64)
    assert torch.allclose(O.qkv_attention(q, k, v, 4), ref, atol=2e-6)


def test_upsample_and_gelu_and_silu():
    x = torch.randn(1, 3, 4, 5)
    assert torch.equal(O.upsample_nearest2x(x), F.interpolate(x, scale_factor=2, mode="nearest"))
    assert torch.allclose(O.gelu_erf(x), F.gelu(x), atol=1e-6)
    assert torch.allclose(O.silu(x), F.silu(x), atol=1e-6)


def test_timestep_embedding_layout():
    e = O.timestep_embedding(7)
    assert e.shape == (1, 320)
    f = torch.exp(torch.arange(160, dtype=torch.float32) * (-np.log(10000.0) / 160))
    assert torch.allclose(e[0, :160], torch.cos(7 * f)) and torch.allclose(e[0, 160:], torch.sin(7 * f))


def test_ddim_schedule():
    ts, step = O.ddim_timesteps(20)
    assert step == 50 and ts[0] == 999 and ts[-1] == 49 and len(ts) == 20
    ts, step = O.ddim_timesteps(50)
    assert step == 20 and ts[-1] == 19 and len(ts) == 50
    ts, step = O.ddim_timesteps(1)
    assert ts == [999]
    ts, step = O.ddim_timesteps(3)  # 1000 // 3 = 333 -> 4 iterations (999, 666, 333, 0) like step_by
    assert ts == [999, 666, 333, 0]


def test_u8_cast_truncates_and_clamps():
    v = torch.tensor([-3.0, 0.0, 0.999, 1.0, 254.999, 255.0, 300.0, float("nan")])
    assert O.to_u8(v).tolist() == [0, 0, 0, 1, 254, 255, 255, 255]


# ------------------------------------------------------------------ oracle vs committed fixtures
def test_unet_fixture_batch2_32(P):
    g = np.load(os.path.join(GOLD, "unet_batch2_32.npz"))
    with torch.no_grad():
        y = O.unet_forward(P, torch.from_numpy(synth.make_latent(2, 32, 32, seed=7)), 321, torch.from_numpy(synth.make_context(2, 5, seed=5)))
    assert np.allclose(y.numpy(), g["out"], rtol=0, atol=2e-5 * np.abs(g["out"]).max())


def test_vae_fixture_16(P):
    g = np.load(os.path.join(GOLD, "vae_16.npz"))
    with torch.no_grad():
        img = O.decode_latent(P, torch.from_numpy(synth.make_latent(1, 16, 16, seed=21)))
    assert np.allclose(img.numpy(), g["img"], rtol=0, atol=2e-5 * np.abs(g["img"]).max())


def test_cfg_batching_equals_two_passes(P):
    """The CUDA path evaluates cond+uncond as one batch-2n pass; the reference does two passes. Same result."""
    x = torch.from_numpy(synth.make_latent(1, 8, 8, seed=2))
    c = torch.from_numpy(synth.make_context(1, 5, seed=8))
    with torch.no_grad():
        two = torch.cat([O.unet_forward(P, x, 10, c), O.unet_forward(P, x, 10, c * 0.5)])
        one = O.unet_forward(P, torch.cat([x, x]), 10, torch.cat([c, c * 0.5]))
    assert torch.allclose(one, two, atol=1e-5)


# ------------------------------------------------------------------ host logic
def test_topology_counts():
    ps = topology.all_params()
    names = [p[0] for p in ps]
    assert len(set(names)) == len(names)
    unet = sum(int(np.prod(s)) for n, s, _, _ in ps if n.startswith("unet/"))
    assert abs(unet - 859.5e6) < 1.0e6  # SURVEY §6: UNet ~ 859.5 M params
    assert "unet/output_blocks/rtu2/upsample/conv/weight" in names
    assert "autoencoder/decoder/blocks/2/upsampler/weight" in names and "autoencoder/decoder/blocks/3/upsampler/weight" not in names


def test_synth_stream_is_stable():
    a = synth.make_tensor("unet/conv_out/bias", (4,), "conv_b", 2880, 0)
    assert a.dtype == np.float32 and np.all(np.abs(a) <= 1 / np.sqrt(2880))
    assert synth.fnv1a32("abc") == 0x1A47E90B
    u = synth.uniform01("x", 5, 0)
    assert np.all((u >= 0) & (u < 1))
    al = synth.alpha_cumulative_products()
    assert al.shape == (1000,) and abs(al[0] - 0.99915) < 1e-5 and abs(al[-1] - 0.00466) < 1e-4


# ------------------------------------------------------------------ C ABI surface (no GPU needed)
def test_abi_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "sdb200.h")).read()
    declared = set(re.findall(r"\b(sdb_[a-z0-9_]+)\s*\(", hdr))
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for sym in sorted(declared):
        assert hasattr(lib, sym), sym
    assert declared == {s[0] for s in _lib.SIGNATURES}


def test_no_cpu_fallback():
    """Without a CUDA device the library refuses to create a context. The devices are hidden from a child process, so the
    check runs the same on machines with and without a GPU."""
    code = ("import ctypes; from stable_diffusion_burn_b200 import _lib; lib = _lib.load(); h = ctypes.c_void_p(); "
            "print(lib.sdb_create(0, ctypes.byref(h)), lib.sdb_last_error(None).decode())")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, check=True).stdout
    rc, msg = out.split(" ", 1)
    assert int(rc) != 0
    assert "no CUDA device" in msg
