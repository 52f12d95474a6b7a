"""Generates tests/golden/ref_python.npz: outputs of the REFERENCE'S OWN Python model (<reference checkout>/python/dump.py, run
unmodified on tests/ref_shim/tinygrad) on this repo's synthetic weights (seed 0). Needs a checkout of the reference.

  python tests/ref_shim/make_ref_golden.py <reference checkout>

How the synthetic weights get into the reference model: the reference's saver (python/stablediffusion.py:8-14) writes the
randomly initialised model as a dump-dir; every file it wrote is matched back to the parameter it came from, which yields the
dump-dir name (and orientation) of every parameter; the synthetic tensors are then assigned by that name.
"""
import os
import shutil
import sys
import tempfile
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, HERE]
import run_reference as R  # noqa: E402
from stable_diffusion_burn_b200 import synth  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "ref_python.npz")
CLIP_PROMPT = [49406, 550, 5810, 617, 8661, 2441, 13, 27, 347, 40786, 4160, 91, 285, 49407]


def inputs():
    g = np.random.Generator(np.random.Philox(2024))
    return {
        "unet32:x": synth.make_latent(2, 32, 32, seed=3), "unet32:ctx": synth.make_context(2, 7, seed=4), "unet32:t": np.int32(321),
        "unet64:x": synth.make_latent(1, 64, 64, seed=1234), "unet64:ctx": synth.make_context(1, 77, seed=77), "unet64:t": np.int32(999),
        "dec16:lat": synth.make_latent(1, 16, 16, seed=21),
        "dec64:lat": synth.make_latent(1, 64, 64, seed=22),
        "enc64:img": g.standard_normal((1, 3, 64, 64), dtype=np.float32),
        "clip:tok": np.asarray([CLIP_PROMPT], np.int32),
        "clip:tok2": np.asarray([[49406, 49407]], np.int32),
    }


def main():
    torch.set_num_threads(os.cpu_count())
    t0 = time.time()
    ref = R.Reference(sys.argv[1], seed=0)
    tmp = tempfile.mkdtemp(prefix="sdb200_ref_dump")
    try:
        ref.save(tmp)
        ref.derive_names(tmp)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    print("reference model built, saved by its own saver, names derived:", len(ref.names), f"{time.time() - t0:.0f}s", flush=True)
    n = ref.assign(synth.make_params(0))
    assert n == len(ref.names), (n, len(ref.names))
    print("synthetic weights assigned", f"{time.time() - t0:.0f}s", flush=True)
    keep = dict(inputs())
    keep["unet32:out"] = ref.unet_forward(keep["unet32:x"], int(keep["unet32:t"]), keep["unet32:ctx"])
    keep["unet64:out"] = ref.unet_forward(keep["unet64:x"], int(keep["unet64:t"]), keep["unet64:ctx"])
    keep["dec16:img"] = ref.decode_latent(keep["dec16:lat"])
    img = ref.decode_latent(keep["dec64:lat"])
    keep["dec64:img_sub"] = img[:, :, ::8, ::8].copy()
    keep["dec64:img_rows"] = img[:, :, 250:254, :].copy()
    keep["enc64:lat"] = ref.encode_image(keep["enc64:img"])
    keep["clip:out"] = ref.clip_forward(keep["clip:tok"])
    keep["clip:out2"] = ref.clip_forward(keep["clip:tok2"])
    for t in (1, 500, 999):
        keep[f"temb:{t}"] = ref.timestep_embedding(t)
    for k, v in keep.items():
        if k.split(":")[1] in ("out", "img", "img_sub", "lat", "out2"):
            print(k, v.shape, "rms", float(np.sqrt((v.astype(np.float64) ** 2).mean())))
    np.savez_compressed(OUT, **keep)
    print("wrote", OUT, os.path.getsize(OUT), "bytes", f"{time.time() - t0:.0f}s")


if __name__ == "__main__":
    main()
