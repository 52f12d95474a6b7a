"""Generates tests/golden/img2img.npz from the img2img oracle (oracle/img2img_oracle.py) on the synthetic weights (seed 0).

Batch 2 of smooth synthetic 256x256 images (latent 32x32, the smallest UNet size), n_steps = 4 and strength 0.5 (the two
steps from t = 499), guidance 5.0, explicit noise synth.make_latent(2, 32, 32, seed=41). Two cases: img2img without a mask,
and inpainting where image 0 repaints its left half and image 1 a box whose edges are not on the 8-pixel grid (so the 8x8
max-pool is exercised). Stored: the inputs, x0, both result latents and the u8 images subsampled by 2.
Run from the repo root:  python tests/golden/make_img2img_golden.py
"""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import img2img_oracle as I  # noqa: E402
from stable_diffusion_burn_b200 import synth, topology  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "img2img.npz")
N_STEPS, STRENGTH, SCALE = 4, 0.5, 5.0


def inputs():
    """The fixture's inputs, all RNG-free except the synth streams: rgb [2,256,256,3], mask [2,256,256], context, uncond, noise."""
    y, x = np.meshgrid(np.arange(256, dtype=np.float64), np.arange(256, dtype=np.float64), indexing="ij")
    imgs = []
    for i in range(2):
        ch = [np.sin(x / (23.0 + 7 * i) + c) * np.cos(y / (31.0 - 5 * i) - 0.7 * c) for c in range(3)]
        imgs.append(np.stack(ch, -1))
    rgb = np.clip(np.rint(127.5 + 110.0 * np.stack(imgs)), 0, 255).astype(np.uint8)
    mask = np.zeros((2, 256, 256), np.uint8)
    mask[0, :, :128] = 1
    mask[1, 37:150, 61:203] = 255
    return dict(rgb=rgb, mask=mask, context=synth.make_context(2, 7, seed=3), uncond=synth.make_context(1, 2, seed=99)[0],
                noise=synth.make_latent(2, 32, 32, seed=41))


def params(decoder=True):
    which = topology.unet_params() + topology.vae_encoder_params() + (topology.vae_decoder_params() if decoder else [])
    return I.O.Params(synth.make_params(0, which=which))


def main():
    torch.set_num_threads(os.cpu_count() or 1)
    t0 = time.time()
    P = params()
    g = inputs()
    x0 = I.encode_x0(P, g["rgb"])
    print("x0", time.time() - t0, flush=True)
    keep = dict(g, x0=x0, n_steps=np.int32(N_STEPS), strength=np.float64(STRENGTH), scale=np.float64(SCALE))
    for case, mask in (("plain", None), ("masked", g["mask"])):
        lat = I.img2img_latent(P, g["rgb"], g["context"], g["uncond"], SCALE, N_STEPS, STRENGTH, g["noise"], mask=mask, x0=x0)
        u8 = I.img2img_image(P, lat, g["rgb"], mask)
        keep[f"latent:{case}"] = lat
        keep[f"u8_sub:{case}"] = u8[:, ::2, ::2, :].copy()
        print(case, time.time() - t0, "rms", float(np.sqrt((lat ** 2).mean())), flush=True)
    np.savez_compressed(OUT, **keep)
    print("done", time.time() - t0)


if __name__ == "__main__":
    main()
