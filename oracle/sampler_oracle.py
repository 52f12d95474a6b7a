"""CPU ORACLE for the selectable samplers — TEST INFRASTRUCTURE ONLY (never imported by the product path).

THE REFERENCE HAS NO COUNTERPART BEYOND ITS `sigma` LINE. Gadersd/stable-diffusion-burn @ 893fb095 samples with DDIM at eta = 0:
`sigma` is fixed to 0 (src/model/stablediffusion/mod.rs:119) and the noise term of the update (:155) never runs. What follows
is this project's definition of DDIM with eta > 0 (that term switched on) and of DPM-Solver++(2M), stated once, here. Both
use the reference's schedule unchanged (oracle/sd_oracle.py, sample_latent):
  ts, step = ddim_timesteps(n_steps), T = len(ts); a_t = alphas[t] read as f32 and widened to f64;
  a_next = alphas[t - step] if t >= step else 1.0.

DDIM, eta in [0, 1] (stablediffusion/mod.rs:152-155 with sigma no longer 0):
  sigma_i = eta * sqrt((1 - a_next) / (1 - a_t)) * sqrt(1 - a_t / a_next)       (0 at the last step: a_next = 1)
  x0  = (x - pred * sqrt(1 - a_t)) / sqrt(a_t)
  x'  = x0 * sqrt(a_next) + pred * sqrt(1 - a_next - sigma_i^2) + sigma_i * z_i   (z_i: step i's slice of the noise)
  eta = 0 is the reference's sampler exactly.

DPM-Solver++(2M), data prediction, multistep (the k-diffusion / diffusers convention):
  alpha = sqrt(a), s = sqrt(1 - a), lambda = log(alpha / s); x0_i = (x - pred * s_t) / alpha_t; h_i = lambda_next - lambda_t
  step 0:        D = x0_0                                                   (first order)
  middle step i: r = h_{i-1} / h_i, D = (1 + 1/(2r)) * x0_i - (1/(2r)) * x0_{i-1}   (second order)
  x' = (s_next / s_t) * x - alpha_next * expm1(-h_i) * D
  last step:     a_next = 1 (s = 0, h = inf): x' = x0_i                     (first order, as diffusers forces at a zero final sigma)

Every scalar coefficient is computed in f64 and rounded to f32 once. The CUDA kernels apply them with one rounding per operation
and no contraction, in the order of ddim_update_f32 / dpmpp_2m_update_f32 below, which therefore reproduce them bit for bit.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from oracle import sd_oracle as O

DDIM, DPMPP_2M = "ddim", "dpmpp_2m"
SAMPLERS = (DDIM, DPMPP_2M)
SEED_MUL = 0x9E3779B97F4A7C15


def step_seed(seed, i):
    """Seed of step i's slice of the library's internal noise stream: seed ^ ((i + 1) * 0x9E3779B97F4A7C15) mod 2^64."""
    return (int(seed) ^ ((i + 1) * SEED_MUL)) & 0xFFFFFFFFFFFFFFFF


def schedule(alphas, n_steps):
    """-> [(t, a_t, a_next)] for the T steps: alphas read as f32, widened to f64."""
    a = np.asarray(alphas, np.float32)
    ts, step = O.ddim_timesteps(n_steps)
    return [(t, float(a[t]), float(a[t - step]) if t >= step else 1.0) for t in ts]


def ddim_sigma(a_t, a_next, eta):
    return eta * math.sqrt((1.0 - a_next) / (1.0 - a_t)) * math.sqrt(1.0 - a_t / a_next)


def ddim_coeffs(a_t, a_next, eta):
    """f64 coefficients of one DDIM step."""
    sigma = ddim_sigma(a_t, a_next, eta)
    return dict(sqrt_1m_at=math.sqrt(1.0 - a_t), sqrt_at=math.sqrt(a_t), sqrt_anext=math.sqrt(a_next),
                dir=math.sqrt(max(0.0, 1.0 - a_next - sigma * sigma)), sigma=sigma)


def _lam(a):
    return math.log(math.sqrt(a) / math.sqrt(1.0 - a))


def dpmpp_2m_coeffs(a_t, a_next, h_prev):
    """f64 coefficients of one DPM-Solver++(2M) step; h_prev = h_{i-1} or None at step 0. -> (coeffs, h_i); h_i is None at the
    last step. kind: "first", "second" or "final"."""
    k = dict(sqrt_1m_at=math.sqrt(1.0 - a_t), sqrt_at=math.sqrt(a_t))
    if a_next >= 1.0:
        return dict(k, kind="final"), None
    h = _lam(a_next) - _lam(a_t)
    k.update(ratio=math.sqrt(1.0 - a_next) / math.sqrt(1.0 - a_t), coef=math.sqrt(a_next) * math.expm1(-h))
    if h_prev is None:
        return dict(k, kind="first"), h
    r = h_prev / h
    return dict(k, kind="second", w0=1.0 + 1.0 / (2.0 * r), w1=1.0 / (2.0 * r)), h


def coeffs(sampler, alphas, n_steps, eta=0.0):
    """The per-step f64 coefficients of a whole run: [dict] of length T."""
    out, h_prev = [], None
    for _, a_t, a_next in schedule(alphas, n_steps):
        if sampler == DDIM:
            out.append(ddim_coeffs(a_t, a_next, eta))
        elif sampler == DPMPP_2M:
            k, h_prev = dpmpp_2m_coeffs(a_t, a_next, h_prev)
            out.append(k)
        else:
            raise ValueError(f"unknown sampler {sampler!r}")
    return out


# ---------------------------------------------------------------------------------------------- f32 replay of the kernels
def _cfg_x0_f32(x, u, c, scale, k):
    f = np.float32
    x, u, c = (np.asarray(v, np.float32) for v in (x, u, c))
    pred = u + (c - u) * f(scale)
    return pred, (x - pred * f(k["sqrt_1m_at"])) / f(k["sqrt_at"])


def ddim_update_f32(x, u, c, scale, k, z=None):
    """cfg_ddim_eta_kernel: pred = u + (c - u)*scale; x0 = (x - pred*s_t)/sqrt(a_t); x' = x0*sqrt(a_next) + pred*dir
    (+ sigma*z when sigma != 0), numpy f32, one rounding per operation."""
    f = np.float32
    pred, x0 = _cfg_x0_f32(x, u, c, scale, k)
    out = x0 * f(k["sqrt_anext"]) + pred * f(k["dir"])
    if f(k["sigma"]) != 0:
        out = out + f(k["sigma"]) * np.asarray(z, np.float32)
    return out


def dpmpp_2m_update_f32(x, u, c, scale, k, prev=None):
    """cfg_dpmpp2m_kernel -> (x', x0): D = x0 (first) or x0*w0 - prev*w1 (second); x' = x*ratio - D*coef; final: x' = x0.
    numpy f32, one rounding per operation; `prev` (x0 of the previous step) is read by the second-order variant only."""
    f = np.float32
    _, x0 = _cfg_x0_f32(x, u, c, scale, k)
    if k["kind"] == "final":
        return x0, x0
    D = x0 if k["kind"] == "first" else x0 * f(k["w0"]) - np.asarray(prev, np.float32) * f(k["w1"])
    return np.asarray(x, np.float32) * f(k["ratio"]) - D * f(k["coef"]), x0


# ---------------------------------------------------------------------------------------------- the samplers
def sample_latent(P, context, uncond, scale, n_steps, init_latent, sampler, eta=0.0, step_noise=None, taps=None, eps_fn=None,
                  alphas=None):
    """Result latent of `sampler` ("ddim" or "dpmpp_2m") from init_latent [n,4,H,W] (torch). The arithmetic runs in the dtype of
    init_latent (P.dtype for the UNet) with the f64 coefficients applied as tensor-by-scalar ops, as sd_oracle.sample_latent.
    step_noise [T,n,4,H,W]: slice i is z_i of DDIM with eta > 0 (required there, rejected elsewhere).
    eps_fn(x, t) -> guided prediction replaces forward_diffuser (P, context, uncond are then unused; pass `alphas`).
    taps: dict receiving f"step{i}/pred", f"step{i}/x0" and f"step{i}/latent" (the latent after step i)."""
    if sampler not in SAMPLERS:
        raise ValueError(f"unknown sampler {sampler!r}")
    if not (0.0 <= eta <= 1.0):
        raise ValueError("eta must lie in [0, 1]")
    noisy = sampler == DDIM and eta > 0
    if noisy and step_noise is None:
        raise ValueError("DDIM with eta > 0 needs step_noise")
    if not noisy and step_noise is not None:
        raise ValueError("step_noise is used only by DDIM with eta > 0")
    if alphas is None:
        alphas = P("alpha_cumulative_products").to(torch.float32).numpy()
    if eps_fn is None:
        context = torch.as_tensor(context).to(P.dtype)
        uncond = torch.as_tensor(uncond).to(P.dtype)
        eps_fn = lambda x, t: O.forward_diffuser(P, x, t, context, uncond, scale)
    latent = torch.as_tensor(init_latent)
    ks = coeffs(sampler, alphas, n_steps, eta)
    prev = None
    with torch.no_grad():
        for i, ((t, _, _), k) in enumerate(zip(schedule(alphas, n_steps), ks)):
            pred = eps_fn(latent, t)
            x0 = (latent - pred * k["sqrt_1m_at"]) / k["sqrt_at"]
            if sampler == DDIM:
                latent = x0 * k["sqrt_anext"] + pred * k["dir"]
                if k["sigma"] != 0:
                    latent = latent + torch.as_tensor(step_noise[i]).to(latent.dtype) * k["sigma"]
            elif k["kind"] == "final":
                latent = x0
            else:
                D = x0 if k["kind"] == "first" else x0 * k["w0"] - prev * k["w1"]
                latent = latent * k["ratio"] - D * k["coef"]
            prev = x0
            if taps is not None:
                taps[f"step{i}/pred"], taps[f"step{i}/x0"], taps[f"step{i}/latent"] = pred, x0, latent
    return latent
