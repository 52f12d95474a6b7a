"""Host-side mirror of the reference's Rust interface for the hot path, over the C ABI.

Same names, argument meaning and error behaviour as
  StableDiffusion::{sample_image, sample_latent, latent_to_image}  src/model/stablediffusion/mod.rs:51-160
  UNet::forward                                                    src/model/unet/mod.rs:109-142
  Autoencoder::decode_latent                                       src/model/autoencoder/mod.rs:68-71
Tensors are numpy fp32 arrays with the reference's shapes (NCHW, [n, L, 768]); errors raise
(the reference panics). No computation happens in Python and there is no fallback path: every call
goes to libsdb200.so and fails loudly if the CUDA library or a B200 is missing.

Differences forced by the tier (documented in DESIGN.md): the initial latent is an explicit argument
(the reference draws it from an unseeded backend RNG) and H/W are parameters (the reference hard-codes 64x64).
"""
from __future__ import annotations

import numpy as np

from ._lib import Context


class UNet:
    def __init__(self, ctx: Context):
        self._c = ctx

    def forward(self, x: np.ndarray, timesteps, context: np.ndarray) -> np.ndarray:
        """x [n,4,H,W]; timesteps Int[1] (one t for the batch); context [n,L,768] -> [n,4,H,W]."""
        ts = np.asarray(timesteps).reshape(-1)
        if ts.size != 1:
            raise ValueError("timesteps must hold exactly one value (reference: Tensor<B,1,Int> of length 1)")
        return self._c.unet_forward(x, int(ts[0]), context)


class Autoencoder:
    def __init__(self, ctx: Context):
        self._c = ctx

    def decode_latent(self, latent: np.ndarray) -> np.ndarray:
        """latent [n,4,H,W] -> image [n,3,8H,8W]."""
        return self._c.decode_latent(latent)

    def encode_image(self, img: np.ndarray) -> np.ndarray:
        """Autoencoder::encode_image (src/model/autoencoder/mod.rs:60-66): image [n,3,H,W] -> latent [n,4,H/8,W/8]."""
        return self._c.encode_image(img)

    def forward(self, img: np.ndarray) -> np.ndarray:
        """Autoencoder::forward (:56-58) = decode_latent(encode_image(x))."""
        return self.decode_latent(self.encode_image(img))


class CLIP:
    def __init__(self, ctx: Context):
        self._c = ctx

    def forward(self, tokens) -> np.ndarray:
        """CLIP::forward (src/model/clip/mod.rs:56-75): int ids [n,L] (L <= 77, unpadded) -> [n,L,768]."""
        return self._c.clip_forward(tokens)


class StableDiffusion:
    """Owns the device context; `diffusion`, `autoencoder` and `clip` mirror the reference's fields."""

    def __init__(self, device: int = 0):
        self.ctx = Context(device)
        self.diffusion = UNet(self.ctx)
        self.autoencoder = Autoencoder(self.ctx)
        self.clip = CLIP(self.ctx)

    # ---- prompt -> context (reference stablediffusion/mod.rs:194-211)
    def context(self, tokenizer, text: str) -> np.ndarray:
        """[1, L, 768]: CLIP of "<|startoftext|>{text}<|endoftext|>" (no padding to 77, like the reference)."""
        ids = tokenizer.encode(f"<|startoftext|>{text}<|endoftext|>")
        return self.clip.forward(np.asarray(ids, np.int32)[None])

    def unconditional_context(self, tokenizer) -> np.ndarray:
        """[Lu, 768] = context("").squeeze(0); Lu = 2 for the empty prompt."""
        return self.context(tokenizer, "")[0]

    # ---- weights (reference: load_stable_diffusion / load_record)
    def init_synthetic(self, seed: int = 0):
        self.ctx.init_synthetic(seed)
        self.ctx.finalize_weights()
        return self

    def load_dump_dir(self, path: str):
        """load_stable_diffusion(path, device) (src/model/stablediffusion/load.rs:16-33): the reference's dump-dir tree."""
        self.ctx.load_dump_dir(path)
        self.ctx.finalize_weights()
        return self

    def load_arrays(self, arrays: dict):
        for name, a in arrays.items():
            self.ctx.set_tensor(name, a)
        self.ctx.finalize_weights()
        return self

    # ---- hot path
    # sampler = "ddim" (eta in [0,1]; the reference's sampler is eta = 0) or "dpmpp_2m" (DPM-Solver++(2M), eta = 0); step_noise
    # [T,n,4,H/8,W/8] is the per-step noise of DDIM with eta > 0 (None: the seeded stream). DESIGN.md §7 row f6. The defaults
    # take the reference's own entry points.
    def sample_image(self, context, unconditional_context, unconditional_guidance_scale: float, n_steps: int,
                     init_latent=None, seed: int = 0, height: int = 512, width: int = 512, sampler: str = "ddim",
                     eta: float = 0.0, step_noise=None):
        """-> list of n flat uint8 arrays of H*W*3 (HWC RGB), like the reference's Vec<Vec<u8>>."""
        if sampler == "ddim" and eta == 0.0 and step_noise is None:
            rgb = self.ctx.sample_image(context, unconditional_context, unconditional_guidance_scale, n_steps,
                                        init_latent=init_latent, seed=seed, H=height // 8, W=width // 8)
        else:
            _, rgb = self.ctx.sample_ex(context, unconditional_context, unconditional_guidance_scale, n_steps, sampler=sampler,
                                        eta=eta, init_latent=init_latent, step_noise=step_noise, seed=seed, H=height // 8,
                                        W=width // 8, latent=False, image=True)
        return [rgb[i].reshape(-1) for i in range(rgb.shape[0])]

    def sample_latent(self, context, unconditional_context, unconditional_guidance_scale: float, n_steps: int,
                      init_latent=None, seed: int = 0, height: int = 512, width: int = 512, sampler: str = "ddim",
                      eta: float = 0.0, step_noise=None) -> np.ndarray:
        if sampler == "ddim" and eta == 0.0 and step_noise is None:
            return self.ctx.sample_latent(context, unconditional_context, unconditional_guidance_scale, n_steps,
                                          init_latent=init_latent, seed=seed, H=height // 8, W=width // 8)
        lat, _ = self.ctx.sample_ex(context, unconditional_context, unconditional_guidance_scale, n_steps, sampler=sampler,
                                    eta=eta, init_latent=init_latent, step_noise=step_noise, seed=seed, H=height // 8,
                                    W=width // 8)
        return lat

    def img2img(self, context, unconditional_context, unconditional_guidance_scale: float, n_steps: int, image, strength: float,
                mask=None, noise=None, seed: int = 0):
        """img2img (SDEdit) and, with `mask`, latent-blend inpainting on the same DDIM sampler (DESIGN.md §7 row f5; the reference
        has no img2img). image [n,H,W,3] uint8 (H, W multiples of 64, the layout sample_image returns), strength in [0,1] (the
        share of the n_steps schedule that runs), mask [n,H,W] (nonzero = repaint) or None, noise [n,4,H/8,W/8] or None (the
        seeded stream sample_image draws from). -> list of n flat uint8 arrays of H*W*3, like sample_image."""
        _, rgb = self.ctx.img2img(context, unconditional_context, unconditional_guidance_scale, n_steps, image, strength,
                                  mask=mask, noise=noise, seed=seed, latent=False)
        return [rgb[i].reshape(-1) for i in range(rgb.shape[0])]

    def latent_to_image(self, latent):
        rgb = self.ctx.latent_to_image(latent)
        return [rgb[i].reshape(-1) for i in range(rgb.shape[0])]

    def close(self):
        self.ctx.close()
