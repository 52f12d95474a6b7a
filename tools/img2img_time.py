"""img2img / inpainting cost on the device entry points (sdb_img2img_dev), against text-to-image in the same process.

Setup: 512x512 images (latent 64x64), 20 DDIM steps, strength 0.75 (15 steps run), guidance 7.5, L = 77, Lu = 2, batch 1 and
batch 8 (BATCHES=1,8). Every configuration is timed with CUDA events around one library call, REPS times per round, and the
rounds alternate all configurations (text-to-image included) so drift hits them alike; the medians over all repetitions are
reported. The split into stages comes from calls that stop early:
  encode      = img2img at strength 0, latent output only (u8 -> planes, encoder, x0 scale)
  steps       = img2img at strength 0.75, latent output only, minus `encode`
  decode_u8   = img2img at strength 0, u8 output, minus `encode`
  total       = img2img at strength 0.75 with u8 output, without and with a mask (left half repainted)
  t2i_total   = sample_image_dev at 20 steps; t2i_step = (t2i_total - t2i_5 steps) / 15
Then, in a separate pass with torch.profiler (not mixed into the timings above), the per-launch device time of the
sampler's elementwise kernels: cfg_ddim_kernel (no mask) and cfg_ddim_blend_kernel (mask), and the img2img boundary kernels.
Prints one JSON line with the device name and power limit read in the same process.
Usage: [BATCHES=1,8 REPS=5 ROUNDS=3] python tools/img2img_time.py
"""
import ctypes as C
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from stable_diffusion_burn_b200 import _lib, synth

STEPS, STRENGTH, SCALE, L, H = 20, 0.75, 7.5, 77, 64
BATCHES = [int(b) for b in os.environ.get("BATCHES", "1,8").split(",")]
REPS, ROUNDS = int(os.environ.get("REPS", 5)), int(os.environ.get("ROUNDS", 3))


def device_info():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def smooth_rgb(n):
    y, x = np.meshgrid(np.arange(8 * H, dtype=np.float64), np.arange(8 * H, dtype=np.float64), indexing="ij")
    imgs = [np.stack([np.sin(x / (40.0 + 9 * i) + ch) * np.cos(y / (55.0 - 3 * i) - ch) for ch in range(3)], -1) for i in range(n)]
    return np.clip(np.rint(127.5 + 110.0 * np.stack(imgs)), 0, 255).astype(np.uint8)


def main():
    dev = torch.device("cuda:0")
    c = _lib.Context(0)
    c.init_synthetic(0)
    c.finalize_weights()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    vp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    out = {"config": dict(steps=STEPS, strength=STRENGTH, steps_run=int(np.floor(STRENGTH * STEPS + 1e-9)), px=8 * H, L=L, Lu=2,
                          reps=REPS, rounds=ROUNDS), **device_info(), "batches": {}}
    for n in BATCHES:
        ctx = torch.from_numpy(synth.make_context(n, L)).to(dev)
        unc = torch.from_numpy(synth.make_context(1, 2, seed=99)[0]).to(dev)
        lat0 = torch.from_numpy(synth.make_latent(n, H, H)).to(dev)
        rgb = torch.from_numpy(smooth_rgb(n)).to(dev)
        mask = torch.zeros((n, 8 * H, 8 * H), dtype=torch.uint8, device=dev)
        mask[:, :, : 4 * H] = 1
        lat = torch.empty((n, 4, H, H), dtype=torch.float32, device=dev)
        out_rgb = torch.empty_like(rgb)

        def i2i(strength, latent_out, rgb_out, m=None):
            c.check(c.lib.sdb_img2img_dev(c.h, vp(rgb), vp(m), vp(ctx), n, L, vp(unc), 2, SCALE, STEPS, strength, None, 1234, H, H,
                                          vp(latent_out), vp(rgb_out), st))

        def t2i(steps):
            c.check(c.lib.sdb_sample_image_dev(c.h, vp(ctx), n, L, vp(unc), 2, SCALE, steps, vp(lat0), H, H, vp(out_rgb), st))

        configs = {
            "encode": lambda: i2i(0.0, lat, None),
            "encode_decode_u8": lambda: i2i(0.0, None, out_rgb),
            "encode_steps": lambda: i2i(STRENGTH, lat, None),
            "total": lambda: i2i(STRENGTH, None, out_rgb),
            "total_masked": lambda: i2i(STRENGTH, None, out_rgb, mask),
            "t2i_total": lambda: t2i(STEPS),
            "t2i_5steps": lambda: t2i(5),
        }
        for fn in configs.values():  # warm-up: modules, graphs of the shape, grow-only buffers
            fn(), fn()
        torch.cuda.synchronize()
        ms = {k: [] for k in configs}
        for _ in range(ROUNDS):
            for k, fn in configs.items():
                for _ in range(REPS):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record(); fn(); b.record(); torch.cuda.synchronize()
                    ms[k].append(a.elapsed_time(b))
        med = {k: float(np.median(v)) for k, v in ms.items()}
        spread = {k: [float(min(v)), float(max(v))] for k, v in ms.items()}
        t2i_step = (med["t2i_total"] - med["t2i_5steps"]) / (STEPS - 5)
        steps_run = out["config"]["steps_run"]
        res = {
            "median_ms": med, "min_max_ms": spread,
            "encode_ms": med["encode"],
            "steps_ms": med["encode_steps"] - med["encode"],
            "decode_u8_ms": med["encode_decode_u8"] - med["encode"],
            "t2i_step_ms": t2i_step,
            "expected_total_ms": steps_run * t2i_step + (med["encode_decode_u8"] - med["encode"]) + med["encode"],
            "mask_overhead_ms": med["total_masked"] - med["total"],
        }
        # per-kernel device time in a profiled pass of its own
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            configs["total"]()
            configs["total_masked"]()
            torch.cuda.synchronize()
        kern = {}
        for e in prof.key_averages():
            for key in ("cfg_ddim_kernel", "cfg_ddim_blend_kernel", "rgb8_to_planes4_kernel", "latent_mask_kernel", "scale_kernel",
                        "noise_latent_kernel", "to_rgb8_paste_kernel", "to_rgb8_kernel", "randn_kernel"):
                if key + "(" in e.key:  # demangled "void sdb::<name>(args)"
                    dt = getattr(e, "device_time", None) or getattr(e, "cuda_time", 0.0)  # average per launch, us
                    kern[key] = {"launches": int(e.count), "avg_us": float(dt)}
        res["kernels"] = kern
        out["batches"][str(n)] = res
        print(f"batch {n}: " + json.dumps(res), file=sys.stderr, flush=True)
    c.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
