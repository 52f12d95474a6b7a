"""Generates tests/golden/sampler.npz from the sampler oracle (oracle/sampler_oracle.py) on the synthetic weights (seed 0).

Batch 2, latent 32x32 (the smallest UNet size), L = 5, Lu = 2, n_steps = 4, guidance 5.0, initial latent
synth.make_latent(2, 32, 32, seed=23). Two cases: DPM-Solver++(2M), and DDIM with eta = 1 whose step noise
[T=4, 2, 4, 32, 32] (synth.make_latent(8, 32, 32, seed=29)) is stored with it. Stored: the inputs and both result latents.
Run from the repo root:  python tests/golden/make_sampler_golden.py
"""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import sampler_oracle as S  # noqa: E402
from stable_diffusion_burn_b200 import synth, topology  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "sampler.npz")
N_STEPS, SCALE = 4, 5.0
CASES = (("dpmpp_2m", S.DPMPP_2M, 0.0), ("ddim_eta1", S.DDIM, 1.0))


def inputs():
    T = len(S.O.ddim_timesteps(N_STEPS)[0])
    return dict(context=synth.make_context(2, 5, seed=3), uncond=synth.make_context(1, 2, seed=99)[0],
                init_latent=synth.make_latent(2, 32, 32, seed=23),
                step_noise=synth.make_latent(2 * T, 32, 32, seed=29).reshape(T, 2, 4, 32, 32))


def params():
    return S.O.Params(synth.make_params(0, which=topology.unet_params()))


def run_case(P, g, sampler, eta):
    return S.sample_latent(P, g["context"], g["uncond"], SCALE, N_STEPS, torch.from_numpy(g["init_latent"]), sampler, eta=eta,
                           step_noise=g["step_noise"] if eta > 0 else None).numpy()


def main():
    torch.set_num_threads(os.cpu_count() or 1)
    t0 = time.time()
    P = params()
    g = inputs()
    keep = dict(g, n_steps=np.int32(N_STEPS), scale=np.float64(SCALE))
    for case, sampler, eta in CASES:
        lat = run_case(P, g, sampler, eta)
        keep[f"latent:{case}"] = lat
        print(case, time.time() - t0, "rms", float(np.sqrt((lat ** 2).mean())), flush=True)
    np.savez_compressed(OUT, **keep)
    print("done", time.time() - t0)


if __name__ == "__main__":
    main()
