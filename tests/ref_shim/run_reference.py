"""Runs the reference's own Python model (<reference checkout>/python/dump.py, imported unmodified) on the tinygrad stand-in.

TEST INFRASTRUCTURE. What is reference-authored here: the model topology and op sequence (python/dump.py:24-350, 352-461),
the savers that define the dump-dir names, transposes and metadata the Rust loaders read (python/save.py, unet.py,
autoencoder.py, clip.py, stablediffusion.py). What is not: the primitive tensor ops (torch, behind tests/ref_shim/tinygrad).
"""
from __future__ import annotations

import contextlib
import hashlib
import io
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))


def load_dump_module(ref_dir: str):
    """import <ref_dir>/python/dump.py with the stand-in `tinygrad` package ahead of everything else."""
    ref_py = os.path.join(ref_dir, "python")
    if not os.path.isfile(os.path.join(ref_py, "dump.py")):
        raise FileNotFoundError(f"{ref_py}/dump.py: not a checkout of the reference")
    for p in (HERE, ref_py):
        if p not in sys.path:
            sys.path.insert(0, p)
    if ROOT not in sys.path:
        sys.path.append(ROOT)
    import dump  # noqa: E402  (the reference file)
    return dump


def _params_of(obj, seen, out):
    """every stand-in parameter tensor reachable from `obj` (model objects, lists, dicts, namedtuples)."""
    from tinygrad.tensor import Tensor
    if id(obj) in seen:
        return
    seen.add(id(obj))
    if isinstance(obj, Tensor):
        out.append(obj)
    elif isinstance(obj, (list, tuple)):
        for o in obj:
            _params_of(o, seen, out)
    elif isinstance(obj, dict):
        for o in obj.values():
            _params_of(o, seen, out)
    elif hasattr(obj, "__dict__") and not isinstance(obj, type) and not callable(getattr(obj, "__code__", None)):
        for o in vars(obj).values():
            _params_of(o, seen, out)


SMALL_FILE = 8192  # dump-dir files up to this size are compared by value, larger ones by size


def tree_manifest(root: str) -> dict:
    """relative path -> [size, digest of the stored values (files up to SMALL_FILE bytes) or None] for every file under `root`."""
    out = {}
    for d, _, fs in os.walk(root):
        for f in fs:
            p = os.path.join(d, f)
            size = os.path.getsize(p)
            digest = None
            if size <= SMALL_FILE:
                a = np.load(p)
                digest = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()[:16]
            out[os.path.relpath(p, root)] = [size, digest]
    return out


def _fingerprint(a: np.ndarray):
    f = np.ascontiguousarray(a, np.float32).reshape(-1)
    return (tuple(a.shape), f[:6].tobytes(), f[-6:].tobytes())


class Reference:
    """The reference StableDiffusion object (python/dump.py:565-570) with random stand-in weights, plus the dump-dir name of
    every parameter, DERIVED by running the reference's own saver and matching what it wrote against the parameters."""

    def __init__(self, ref_dir: str, seed: int = 0, verbose: bool = False):
        self.dump = load_dump_module(ref_dir)
        from tinygrad import nn
        from tinygrad.tensor import Tensor
        self.Tensor = Tensor
        Tensor.no_grad = True
        nn.set_seed(seed)
        self.model = self.dump.StableDiffusion()
        self.unet = self.model.model.diffusion_model
        self.vae = self.model.first_stage_model
        self.clip = self.model.cond_stage_model.transformer.text_model
        self.verbose = verbose
        self.names = None  # dump-dir name -> (param, transposed)

    def set_alphas(self, alphas: np.ndarray):
        self.model.alphas_cumprod.t = torch.from_numpy(np.asarray(alphas, np.float32).copy())

    def save(self, path: str):
        """python/stablediffusion.py:8-14 save_stable_diffusion — the reference's writer of the tree the Rust side loads."""
        sink = io.StringIO()
        with contextlib.redirect_stdout(sys.stdout if self.verbose else sink):
            self.dump.sdsave.save_stable_diffusion(self.model, path)

    def derive_names(self, path: str):
        """Matches every tensor file under `path` (written by save()) to the parameter it came from."""
        from stable_diffusion_burn_b200 import dumpdir
        params = []
        _params_of(self.model, set(), params)
        table = {}
        for p in params:
            a = p.numpy()
            table.setdefault(_fingerprint(a), []).append((p, False))
            if a.ndim == 2:
                table.setdefault(_fingerprint(a.T), []).append((p, True))
        names, used = {}, set()
        for dirpath, _, files in os.walk(path):
            for f in files:
                if not f.endswith(".npy"):
                    continue
                rel = os.path.relpath(os.path.join(dirpath, f), path)[:-4]
                try:
                    a = dumpdir.read_tensor(os.path.join(dirpath, f))
                except ValueError:
                    continue  # scalars ([1.0, v]) and small metadata vectors that are not tensors
                hits = table.get(_fingerprint(a))
                if not hits:
                    continue
                p, tr = hits[0]
                if not np.array_equal(a, p.numpy().T if tr else p.numpy()):
                    continue
                names[rel] = (p, tr)
                used.add(id(p))
        missing = [p.shape for p in params if id(p) not in used]
        assert not missing, f"parameters the reference saver did not write: {missing[:5]}"
        self.names = names
        return names

    def assign(self, arrays: dict):
        """loads weights by dump-dir name (registry names; the schedule is 'alpha_cumulative_products')."""
        assert self.names is not None, "derive_names() first"
        done = 0
        for name, (p, tr) in self.names.items():
            key = "alpha_cumulative_products" if name == "alphas_cumprod" else name
            if key not in arrays:
                continue
            a = np.asarray(arrays[key], np.float32)
            p.t = torch.from_numpy(np.ascontiguousarray(a.T if tr else a).copy())
            done += 1
        return done

    # ---- forwards (the reference's __call__ methods)
    def unet_forward(self, x, t, context):
        """python/dump.py:326-350 UNetModel.__call__(x, timesteps, context); timesteps = Tensor([t]) as in :631."""
        T = self.Tensor
        with torch.no_grad():
            return self.unet(T(np.asarray(x, np.float32)), T([float(t)]), T(np.asarray(context, np.float32))).numpy()

    def decode_latent(self, latent):
        """python/dump.py:149-150: post_quant_conv then decoder (== Autoencoder::decode_latent, autoencoder/mod.rs:68-71)."""
        T = self.Tensor
        with torch.no_grad():
            return self.vae.decoder(self.vae.post_quant_conv(T(np.asarray(latent, np.float32)))).numpy()

    def encode_image(self, img):
        """python/dump.py:145-148: encoder, quant_conv, [:, 0:4] (== Autoencoder::encode_image, autoencoder/mod.rs:60-66)."""
        T = self.Tensor
        with torch.no_grad():
            lat = self.vae.quant_conv(self.vae.encoder(T(np.asarray(img, np.float32))))
            return lat[:, 0:4].numpy()

    def autoencoder_forward(self, img):
        """python/dump.py:144-150 AutoencoderKL.__call__ as written (encode + decode)."""
        with torch.no_grad():
            return self.vae(self.Tensor(np.asarray(img, np.float32))).numpy()

    def clip_forward(self, tokens):
        """python/dump.py:449-454 CLIPTextTransformer.__call__(input_ids[n, L])."""
        with torch.no_grad():
            return self.clip(self.Tensor(torch.from_numpy(np.asarray(tokens, np.int64)))).numpy()

    def timestep_embedding(self, t):
        """python/dump.py:274-278."""
        with torch.no_grad():
            return self.dump.timestep_embedding(self.Tensor([float(t)]), 320).numpy()
