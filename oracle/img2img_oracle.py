"""CPU ORACLE for img2img and inpainting — TEST INFRASTRUCTURE ONLY (never imported by the product path).

THIS PART HAS NO REFERENCE COUNTERPART. Gadersd/stable-diffusion-burn @ 893fb095 samples text-to-image only. What follows is
the standard SDEdit (img2img) and legacy latent-blend inpainting construction applied to the reference's own schedule and
sampler (src/model/stablediffusion/mod.rs:102-160), built on the arithmetic of oracle/sd_oracle.py (encode_image,
forward_diffuser, ddim_timesteps, latent_to_image_f32, to_u8). It is this project's definition, stated once, here:

  1. x = fl(fl(v * fl32(2/255)) - 1) per channel of the u8 image [n,8H,8W,3], NCHW, no FMA (numpy fp32 reproduces the kernel).
  2. x0 = fl(encode_image(x) * 0.18215f): the inverse of latent_to_image's `latent * (1/0.18215)`; the encoder returns the
     posterior mean, as the reference's encode_image does.
  3. ts, step = ddim_timesteps(n_steps), T = len(ts); n_run = min(T, floor(strength * T + 1e-9)); i0 = T - n_run.
     n_run == 0: the result latent is x0 (no UNet evaluation).
  4. a = fl32(sqrt(f64(alpha[ts[i0]]))), b = fl32(sqrt(1 - f64(alpha[ts[i0]]))); x_t0 = fl(fl(a*x0) + fl(b*eps)), no FMA.
  5. The DDIM / CFG loop of sample_latent over ts[i0:], unchanged.
  6. With a pixel mask (nonzero = repaint): the latent mask m is the max over each 8x8 pixel block. After each step's update
     the cells with m == 0 are SELECTED from known = fl(fl(sqrt(a_prev)*x0) + fl(sqrt(1-a_prev)*eps)); a_prev = 1 at the
     last step, so the kept cells of the result equal x0 exactly.
  7. Decode + u8 as latent_to_image; with a mask, pixels whose mask is 0 are then copied from the input image unchanged.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from oracle import sd_oracle as O

LATENT_SCALE = np.float32(0.18215)


def image_from_rgb8(rgb):
    """u8 [n,H,W,3] -> fp32 [n,3,H,W] in [-1,1]: fl(fl(v * fl32(2/255)) - 1) (step 1)."""
    v = np.asarray(rgb, np.uint8).astype(np.float32).transpose(0, 3, 1, 2)
    return np.ascontiguousarray(v * np.float32(2.0 / 255.0) - np.float32(1.0))


def latent_mask(mask):
    """pixel mask [n,8H,8W] (nonzero = repaint) -> latent mask [n,H,W] u8 in {0,1}: max over each 8x8 block (step 6)."""
    m = np.asarray(mask) != 0
    n, hp, wp = m.shape
    return m.reshape(n, hp // 8, 8, wp // 8, 8).any(axis=(2, 4)).astype(np.uint8)


def img2img_schedule(n_steps, strength):
    """-> (ts, step, i0): the steps that run are ts[i0:] (step 3)."""
    ts, step = O.ddim_timesteps(n_steps)
    T = len(ts)
    n_run = min(T, int(math.floor(strength * T + 1e-9)))
    return ts, step, T - n_run


def encode_x0(P, rgb):
    """x0 = fl(encode_image(image_from_rgb8(rgb)) * 0.18215f) [n,4,H,W] (step 2)."""
    with torch.no_grad():
        enc = O.encode_image(P, torch.from_numpy(image_from_rgb8(rgb))).to(torch.float32).numpy()
    return enc * LATENT_SCALE


def noised(x0, eps, alpha):
    """fl(fl(fl32(sqrt(alpha)) * x0) + fl(fl32(sqrt(1 - alpha)) * eps)), alpha a float widened from f32 (steps 4 and 6)."""
    a, b = np.float32(math.sqrt(float(alpha))), np.float32(math.sqrt(1.0 - float(alpha)))
    return a * np.asarray(x0, np.float32) + b * np.asarray(eps, np.float32)


def img2img_latent(P, rgb, context, uncond, scale, n_steps, strength, noise, mask=None, x0=None):
    """Result latent [n,4,H,W] of img2img (mask None) or inpainting (steps 1-6). context [n,L,768], uncond [Lu,768], noise
    [n,4,H,W] (numpy or torch); `x0` may be passed to skip the encoder when it is already known."""
    if x0 is None:
        x0 = encode_x0(P, rgb)
    ts, step, i0 = img2img_schedule(n_steps, strength)
    if i0 == len(ts):
        return np.array(x0, np.float32)
    alphas = P("alpha_cumulative_products").to(torch.float32)
    eps = np.asarray(noise, np.float32)
    keep = None if mask is None else torch.from_numpy(latent_mask(mask)[:, None] == 0)
    context = torch.as_tensor(context).to(P.dtype)
    uncond = torch.as_tensor(uncond).to(P.dtype)
    latent = torch.from_numpy(noised(x0, eps, alphas[ts[i0]])).to(P.dtype)
    with torch.no_grad():
        for t in ts[i0:]:
            # the body of sd_oracle.sample_latent (stablediffusion/mod.rs:124-156, sigma = 0)
            a_t = float(alphas[t])
            a_prev = float(alphas[t - step]) if t >= step else 1.0
            pred = O.forward_diffuser(P, latent, t, context, uncond, scale)
            predx0 = (latent - pred * math.sqrt(1.0 - a_t)) / math.sqrt(a_t)
            latent = predx0 * math.sqrt(a_prev) + pred * math.sqrt(1.0 - a_prev)
            if keep is not None:
                latent = torch.where(keep, torch.from_numpy(noised(x0, eps, a_prev)).to(P.dtype), latent)
    return latent.numpy()


def img2img_image(P, latent, rgb, mask=None):
    """u8 [n,8H,8W,3] of a result latent: latent_to_image, then the pixels with mask == 0 copied from rgb (step 7)."""
    with torch.no_grad():
        u8 = O.to_u8(O.latent_to_image_f32(P, torch.as_tensor(latent)))
    if mask is not None:
        u8 = np.where((np.asarray(mask) != 0)[..., None], u8, np.asarray(rgb, np.uint8))
    return u8
