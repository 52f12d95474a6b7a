"""Cost of the selectable samplers on the device entry point (sdb_sample_ex_dev), all configurations alternated in one process.

Setup: 512x512 images (latent 64x64), guidance 7.5, L = 77, Lu = 2, u8 output, batch 1 and batch 8 (BATCHES=1,8):
  ddim_20      DDIM eta = 0 at 20 steps (the reference's sampler; the cfg_ddim_kernel path of sdb_sample_image)
  ddim_eta1_20 DDIM eta = 1 at 20 steps, step noise drawn inside the update kernel
  dpmpp_20     DPM-Solver++(2M) at 20 steps
  dpmpp_10     DPM-Solver++(2M) at 10 steps (the step count it is used at in place of DDIM at 20)
  ddim_10      DDIM eta = 0 at 10 steps (with ddim_20: the per-step cost of DDIM)
Every configuration is timed with CUDA events around one library call, REPS times per round, and the rounds alternate all
configurations so drift hits them alike; medians over all repetitions, also per image (/ n). Per-step cost of a sampler =
(its 20-step time - its 10-step time) / 10, for DDIM and DPM++. Then, in a separate pass with torch.profiler (not mixed into
the timings), the per-launch device time of the three update kernels. Prints one JSON line with the device name and power limit
read in the same process.
Usage: [BATCHES=1,8 REPS=5 ROUNDS=3] python tools/sampler_time.py
"""
import ctypes as C
import json
import os
import re
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from stable_diffusion_burn_b200 import _lib, synth

SCALE, L, H = 7.5, 77, 64
BATCHES = [int(b) for b in os.environ.get("BATCHES", "1,8").split(",")]
REPS, ROUNDS = int(os.environ.get("REPS", 5)), int(os.environ.get("ROUNDS", 3))
CONFIGS = {"ddim_20": (0, 0.0, 20), "ddim_eta1_20": (0, 1.0, 20), "dpmpp_20": (1, 0.0, 20), "dpmpp_10": (1, 0.0, 10),
           "ddim_10": (0, 0.0, 10)}
KERNELS = ("cfg_ddim_kernel", "cfg_ddim_eta_kernel", "cfg_dpmpp2m_kernel")


def device_info():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def main():
    dev = torch.device("cuda:0")
    c = _lib.Context(0)
    c.init_synthetic(0)
    c.finalize_weights()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    vp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    out = {"config": dict(px=8 * H, L=L, Lu=2, scale=SCALE, reps=REPS, rounds=ROUNDS, configs=CONFIGS), **device_info(),
           "batches": {}}
    for n in BATCHES:
        ctx = torch.from_numpy(synth.make_context(n, L)).to(dev)
        unc = torch.from_numpy(synth.make_context(1, 2, seed=99)[0]).to(dev)
        lat0 = torch.from_numpy(synth.make_latent(n, H, H)).to(dev)
        rgb = torch.empty((n, 8 * H, 8 * H, 3), dtype=torch.uint8, device=dev)

        def run(sampler, eta, steps):
            c.check(c.lib.sdb_sample_ex_dev(c.h, vp(ctx), n, L, vp(unc), 2, SCALE, steps, sampler, eta, vp(lat0), None, 1234, H, H,
                                            None, vp(rgb), st))

        fns = {k: (lambda a=a: run(*a)) for k, a in CONFIGS.items()}
        for k, fn in fns.items():  # warm-up: modules, the step graph of the shape, grow-only buffers
            fn(), fn()
            torch.cuda.synchronize()
            print(f"batch {n}: warmed up {k}", file=sys.stderr, flush=True)
        ms = {k: [] for k in fns}
        for r in range(ROUNDS):
            for k, fn in fns.items():
                for _ in range(REPS):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record(); fn(); b.record(); torch.cuda.synchronize()
                    ms[k].append(a.elapsed_time(b))
            print(f"batch {n}: round {r + 1}/{ROUNDS} " + json.dumps({k: round(v[-1], 3) for k, v in ms.items()}), file=sys.stderr,
                  flush=True)
        med = {k: float(np.median(v)) for k, v in ms.items()}
        res = {
            "median_ms": med,
            "median_ms_per_image": {k: v / n for k, v in med.items()},
            "min_max_ms": {k: [float(min(v)), float(max(v))] for k, v in ms.items()},
            "ddim_step_ms": (med["ddim_20"] - med["ddim_10"]) / 10,
            "dpmpp_step_ms": (med["dpmpp_20"] - med["dpmpp_10"]) / 10,
            "ddim_eta1_minus_ddim_20_ms": med["ddim_eta1_20"] - med["ddim_20"],
            "dpmpp_20_minus_ddim_20_ms": med["dpmpp_20"] - med["ddim_20"],
        }
        # per-launch device time of the update kernels, in a profiled pass of its own
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for k in ("ddim_20", "ddim_eta1_20", "dpmpp_20"):
                fns[k]()
            torch.cuda.synchronize()
        name = lambda s: (lambda m: m and m.group(1) + (m.group(2) or ""))(
            re.search(r"\b(" + "|".join(KERNELS) + r")(<\d>)?\(", s))  # demangled "void sdb::<name>[<kind>](args)"
        kern = {}
        for e in prof.key_averages():
            if name(e.key):
                dt = getattr(e, "device_time", None) or getattr(e, "cuda_time", 0.0)  # average per launch, us
                kern[name(e.key)] = {"launches": int(e.count), "avg_us": float(dt)}
        per_launch = {}  # the spread behind each average: one device interval per launch
        for e in prof.events():
            if str(getattr(e, "device_type", "")).endswith("CUDA") and name(e.name):
                per_launch.setdefault(name(e.name), []).append(e.time_range.elapsed_us())
        for k, v in per_launch.items():
            if k in kern:
                kern[k].update(min_us=float(min(v)), median_us=float(np.median(v)), max_us=float(max(v)))
        res["kernels"] = kern
        out["batches"][str(n)] = res
        print(f"batch {n}: " + json.dumps(res), file=sys.stderr, flush=True)
    c.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
