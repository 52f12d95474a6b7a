"""Generates the fixtures through which the CPU suite checks this repo against the reference without a checkout of it:

  python tests/ref_shim/make_ref_fixtures.py <reference checkout>

* tests/golden/reference_line_counts.json: the line count of every .rs / .py file of the reference (citations in this repo
  point at those lines, tests/test_citations_cpu.py).
* tests/golden/bpe_simple_vocab_16e6.txt.xz: the part of the reference's BPE vocabulary file the tokenizer reads, the header
  line and the 48894 merges after it (src/tokenizer.rs:92-93; tests/test_tokenizer_cpu.py).
* tests/golden/ref_dump_tree.json.xz: the dump-dir names the reference's saver writes, and the tree it writes for the model with
  the synthetic weights (seed 0): every file's size, and a digest of the values of every file up to 8 KiB
  (tests/test_ref_pin_cpu.py::test_fixture_dump_dir_tree).
* tests/golden/ref_python_forwards.npz: further outputs of the reference's own Python model on the synthetic weights
  (tests/test_ref_pin_cpu.py::test_fixture_forwards).

It also re-derives one entry of tests/golden/ref_python.npz from the reference model and fails if that fixture has moved.
"""
import json
import lzma
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

GOLD = os.path.join(ROOT, "tests", "golden")
N_MERGES = 49152 - 256 - 2  # merges the tokenizer keeps after the header line


def forwards_inputs():
    """Inputs of test_fixture_forwards (the UNet and CLIP cases it also runs are those of ref_python.npz)."""
    return {"dec16:lat": synth.make_latent(1, 16, 16, seed=5),
            "enc64:img": np.random.default_rng(0).standard_normal((1, 3, 64, 64)).astype(np.float32),
            "temb:t": np.int32(321)}


def line_counts(ref_dir):
    out = {}
    for d, _, fs in os.walk(ref_dir):
        if "/.git" in d:
            continue
        for f in fs:
            if f.endswith((".rs", ".py")):
                p = os.path.join(d, f)
                out[os.path.relpath(p, ref_dir)] = sum(1 for _ in open(p, encoding="utf-8", errors="replace"))
    return dict(sorted(out.items()))


def main():
    ref_dir = sys.argv[1]
    torch.set_num_threads(os.cpu_count())
    t0 = time.time()
    with open(os.path.join(GOLD, "reference_line_counts.json"), "w") as f:
        json.dump(line_counts(ref_dir), f, indent=0, sort_keys=True)
        f.write("\n")
    with open(os.path.join(ref_dir, "bpe_simple_vocab_16e6.txt"), encoding="utf-8") as f:
        head = [next(f) for _ in range(1 + N_MERGES)]
    with lzma.open(os.path.join(GOLD, "bpe_simple_vocab_16e6.txt.xz"), "wt", encoding="utf-8", preset=9) as f:
        f.write("".join(head))

    ref = R.Reference(ref_dir, seed=0)
    tmp = tempfile.mkdtemp(prefix="sdb200_ref_dump")
    try:
        ref.save(tmp)
        ref.derive_names(tmp)
        shutil.rmtree(tmp)
        n = ref.assign(synth.make_params(0))
        assert n == len(ref.names), (n, len(ref.names))
        print("synthetic weights assigned", f"{time.time() - t0:.0f}s", flush=True)
        ref.save(tmp)
        tree = {"names": sorted(ref.names), "files": R.tree_manifest(tmp)}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    with lzma.open(os.path.join(GOLD, "ref_dump_tree.json.xz"), "wt", encoding="utf-8", preset=9) as f:
        json.dump(tree, f, indent=0, sort_keys=True)
        f.write("\n")
    print("tree:", len(tree["files"]), "files", f"{time.time() - t0:.0f}s", flush=True)

    G = np.load(os.path.join(GOLD, "ref_python.npz"))
    got = ref.decode_latent(G["dec16:lat"]).astype(np.float64)
    e = float(np.linalg.norm(got - G["dec16:img"]) / np.linalg.norm(G["dec16:img"]))
    assert e < 1e-6, f"tests/golden/ref_python.npz is not what the reference model outputs any more: dec16 {e:.3e}"

    keep = dict(forwards_inputs())
    # images are kept at every second pixel of each axis
    keep["dec16:img_sub"] = ref.decode_latent(keep["dec16:lat"])[:, :, ::2, ::2].copy()
    keep["enc64:lat"] = ref.encode_image(keep["enc64:img"])
    keep["ae64:img_sub"] = ref.autoencoder_forward(keep["enc64:img"])[:, :, ::2, ::2].copy()
    keep["temb:out"] = ref.timestep_embedding(int(keep["temb:t"]))
    del keep["enc64:img"]  # regenerated from its seed by the test
    np.savez_compressed(os.path.join(GOLD, "ref_python_forwards.npz"), **keep)
    print("done", f"{time.time() - t0:.0f}s")


if __name__ == "__main__":
    main()
