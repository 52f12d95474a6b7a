#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (BASELINE.json: 512x512 images/sec @ 20 DDIM steps).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one process per GPU)
  python bench.py --impl reference --steps K --warmup W    # reference arm: CPU port (oracle/) on the host cores

A "step" is one pass of the hot path over one batch: StableDiffusion::sample_image for `--batch` images
(20 DDIM steps x (cond+uncond UNet) + VAE decode + u8 pack). Default workload = BASELINE configs[1]
(batch 1, 512x512, 20 steps, cfg 7.5) on every rank (weak scaling: per-GPU work is fixed).
Prints ONE JSON line on rank 0. With --dump-outputs DIR, the images the last timed step produced are written to DIR as
float32 .npy (same arguments -> same inputs, so two builds can be compared output for output).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: no __pycache__ from this process

DUMP_BUDGET_BYTES = 64 << 20  # all files of one --dump-outputs directory together

METRIC = "images_per_sec_512x512_20steps"
UNIT = "images/s"
FLOP_PER_IMAGE = 34_695e9  # algorithmic, SURVEY §8d: 40 x 804.4 + 2518.4 GFLOP


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(tflops=float(p["bf16_tflops_sustained"]), tflops_burst=float(p["bf16_tflops"]), hbm=float(p["hbm_gbs"]), src="measured")
    except Exception:
        return dict(tflops=1400.0, tflops_burst=1590.0, hbm=6650.0, src="fallback")


def gemm_traffic_per_launch():
    """DRAM bytes per gemm_tc launch from the committed ncu capture (profiles/r2_gemm_traffic.json, else round 1's), or None."""
    for name in ("r2_gemm_traffic.json", "r1_gemm_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return float(json.load(f)["traffic_bytes_per_launch"])
        except Exception:
            continue
    return None


def workload_config(args, n):
    """`config` of the JSON line — identical in both arms (the reference arm runs on this arm's config)."""
    return {"workload": f"SDv1-4 txt2img {args.size}x{args.size}, {args.ddim_steps} steps, cfg=7.5, batch={n} per GPU",
            "context_len": args.context_len, "precision_option": args.precision,
            "l2": "inputs larger than L2: >1.9 GB of packed weights stream from HBM every UNet step (L2 = 126 MB)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def window(self, t0, t1):
        """clocks / throttle reasons of the samples taken in [t0, t1] (one nvidia-smi process serves every timed region of the
        run: forking a second one from a process that holds a CUDA context, pinned buffers and NCCL threads hung rank 0)"""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        rows = [r for (t, r) in list(self.rows) if t0 <= t <= t1 + 0.25]
        sm = [float(r[0]) for r in rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()


def host_threads():
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    return max(1, min(n, 32))  # torch-CPU stops scaling (and shared hosts oversubscribe) beyond a few dozen threads


# algorithmic GFLOP of the CPU port's work items (SURVEY §8d; the 32x32 figures scale conv/linear by 1/4, self-attention by 1/16)
GF_UNET_64, GF_UNET_32 = 804.4, 178.2
GF_DEC_64, GF_DEC_32 = 2518.4, 631.6


def cpu_port_times(n_steps=1, latent=64, ddim_steps_total=20):
    """Times the CPU port of the reference path (oracle/, torch fp32 on the host cores): `n_steps` REAL DDIM steps (cond + uncond
    UNet at the full latent size, L = 77 / Lu = 2, the timesteps a `ddim_steps_total`-step schedule starts with) and one REAL
    decode_latent. Nothing is extrapolated. Returns (seconds per DDIM step [list], seconds per decode, threads, description)."""
    import torch

    from oracle import sd_oracle as O
    from stable_diffusion_burn_b200 import synth
    threads = host_threads()
    torch.set_num_threads(threads)
    P = O.Params(synth.make_params(0))
    ctx = torch.from_numpy(synth.make_context(1, 77))
    unc = torch.from_numpy(synth.make_context(1, 2, seed=99))[0]
    ts, _ = O.ddim_timesteps(ddim_steps_total)
    with torch.no_grad():
        lat = torch.from_numpy(synth.make_latent(1, latent, latent))
        O.unet_forward(P, lat[:, :, :16, :16].contiguous(), 999, ctx)  # thread pool / allocator warm-up, not a step
        steps = []
        for i in range(n_steps):
            t0 = time.perf_counter()
            O.forward_diffuser(P, lat, ts[i % len(ts)], ctx, unc, 7.5)
            steps.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        O.decode_latent(P, lat * (1.0 / 0.18215))
        dec = time.perf_counter() - t0
    what = f"{n_steps} real {latent}x{latent} DDIM step(s) (cond+uncond UNet, L=77/Lu=2) + 1 real decode_latent, timed directly on {threads} threads"
    return steps, dec, threads, what


def gpu_eager_times():
    """OPTIONAL, labelled secondary comparator (SURVEY §8d): the same torch restatement with its tensors on cuda:0, i.e. what
    torch 2.11 eager (cuDNN convs with TF32 allowed, cuBLAS fp32 matmuls, materialised attention scores) does with the
    reference's op sequence on this GPU. It is NOT the reference (which cannot be built here) and not this repo's path."""
    import torch

    from oracle import sd_oracle as O
    from stable_diffusion_burn_b200 import synth
    dev = torch.device("cuda:0")
    P = O.Params({})
    P.t = {k: torch.from_numpy(v).to(dev) for k, v in synth.make_params(0).items()}
    ctx = torch.from_numpy(synth.make_context(1, 77)).to(dev)
    unc = torch.from_numpy(synth.make_context(1, 2, seed=99))[0].to(dev)
    lat = torch.from_numpy(synth.make_latent(1, 64, 64)).to(dev)

    def timed(fn, reps):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    with torch.no_grad():
        step_ms = timed(lambda: O.forward_diffuser(P, lat, 999, ctx, unc, 7.5), 5)
        dec_ms = timed(lambda: O.decode_latent(P, lat * (1.0 / 0.18215)), 3)
    return {"ms_per_ddim_step": step_ms, "ms_decode": dec_ms, "images_per_s": 1000.0 / (20 * step_ms + dec_ms),
            "what": "torch 2.11 eager on cuda:0 running the oracle's op sequence (cuDNN conv, TF32 allowed; cuBLAS fp32 matmul): "
                    "a labelled secondary comparator, not the reference and not this repo's path"}


def dump_outputs(out_dir, name, a, budget_bytes):
    """Writes `a` as out_dir/<name>.npy in float32; above `budget_bytes`, a fixed seeded sample of its flattened values instead,
    as out_dir/<name>_sample.npy (the same positions for the same shape, so samples of two runs compare element for element)."""
    import numpy as np
    a = np.ascontiguousarray(a, np.float32)
    if a.nbytes > budget_bytes:
        keep = np.sort(np.random.default_rng(0).choice(a.size, budget_bytes // 4, replace=False))
        a, name = a.reshape(-1)[keep], name + "_sample"
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), a)


def run_reference(args):
    """Reference arm: the reference's own implementation cannot be built here (Rust, no toolchain; DESIGN.md §2), so this times
    the CPU port of the same path on the host cores. A bench "step" of this arm is ONE real DDIM step of the workload (2 UNet
    evaluations at the full latent size) — a bounded sample of the 20-step image; warm-up and timed steps are all real, and one
    real decode is timed beside them. value = 1 / (ddim_steps * mean_step + decode)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    total = args.warmup + args.steps
    step_s, dec, threads, what = cpu_port_times(total, latent=args.size // 8, ddim_steps_total=args.ddim_steps)
    timed = step_s[args.warmup:]
    mean_step = sum(timed) / len(timed)
    img_s = args.ddim_steps * mean_step + dec
    value = 1.0 / img_s
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": mean_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.batch),
        "impl_note": "CPU port of the Burn path (oracle/, torch-CPU fp32; the Rust reference cannot be built in this image). Each timed "
                     "step is ONE real DDIM step (cond+uncond UNet); value = 1/(ddim_steps*mean_step + decode), decode timed once",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{what} ({mean_step:.2f} s/step, decode {dec:.2f} s)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.ref_cuda:
        try:
            line["secondary_gpu_eager"] = gpu_eager_times()
        except Exception as e:  # the comparator is optional: never let it take the reference line down
            line["secondary_gpu_eager"] = {"unavailable": repr(e)[:200]}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="sdb200")
    ap.add_argument("--batch", type=int, default=1, help="images per rank per step (BASELINE configs[1] = 1; configs[4] = 8)")
    ap.add_argument("--ddim-steps", type=int, default=20)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--context-len", type=int, default=77)
    ap.add_argument("--precision", type=int, default=0, help="0 = per-layer policy (meets 1e-3), 1/2/3 = force passes")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--no-c5", action="store_true", help="multi-GPU runs: skip the BASELINE configs[4] sub-record (8 images per rank)")
    ap.add_argument("--ref-cuda", action="store_true",
                    help="with --impl reference: also time the torch restatement on cuda:0 (labelled secondary comparator)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the u8 images of the last timed step as float32 DIR/images.npy (images_rank<r>.npy per rank "
                         "with several GPUs; a seeded sample when above 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to this repo's CUDA path")
    if args.impl == "reference":
        return run_reference(args)
    if args.warmup < 3:
        args.warmup = 3

    import numpy as np
    import torch

    from stable_diffusion_burn_b200 import _lib, synth

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # stdout must carry exactly one JSON line: NCCL_DEBUG=VERSION would print the NCCL banner there
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from stable_diffusion_burn_b200 import parallel
    ctx = _lib.Context(local)
    # ---- weights: rank 0 fills the fp32 master arena; ONE NCCL broadcast, issued by the library itself
    # (sdb_broadcast_weights, include/sdb200.h), ships it over NVLink. No collective on the sampling path.
    if rank == 0:
        ctx.init_synthetic(0)
    bcast_ms = None
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        parallel.broadcast_weights(ctx, rank, world)
        bcast_ms = (time.perf_counter() - t0) * 1e3  # includes ncclCommInitRank
    ctx.finalize_weights()
    if args.precision:
        ctx.set_option("precision", args.precision)

    Hl = args.size // 8
    L, Lu = args.context_len, 2
    dev = torch.device("cuda", local)
    stream = torch.cuda.current_stream()

    def make_steps(n):
        """(device-resident step, host-buffer end-to-end step, h2d bytes, d2h bytes) for a batch of n images per rank;
        image index = rank*n + i: every rank samples different images."""
        h_ctx = synth.make_context(n, L, seed=77 + rank)
        h_unc = synth.make_context(1, Lu, seed=99)[0]
        h_lat = synth.make_latent(n, Hl, Hl, seed=1234 + rank * n)
        d_ctx, d_unc, d_lat = (torch.from_numpy(a).to(dev) for a in (h_ctx, h_unc, h_lat))
        d_rgb = torch.empty((n, 8 * Hl, 8 * Hl, 3), dtype=torch.uint8, device=dev)
        p_ctx, p_unc, p_lat = (torch.from_numpy(a).pin_memory() for a in (h_ctx, h_unc, h_lat))
        p_rgb = torch.empty((n, 8 * Hl, 8 * Hl, 3), dtype=torch.uint8).pin_memory()
        keep = (d_ctx, d_unc, d_lat, d_rgb, p_ctx, p_unc, p_lat, p_rgb)

        def dev_step(_k=keep):
            ctx.check(ctx.lib.sdb_sample_image_dev(ctx.h, d_ctx.data_ptr(), n, L, d_unc.data_ptr(), Lu, 7.5, args.ddim_steps,
                                                   d_lat.data_ptr(), Hl, Hl, d_rgb.data_ptr(), stream.cuda_stream))

        def e2e_step(_k=keep):
            # the public host-buffer call: H2D of context/uncond/latent, sampling, D2H of the u8 images — all inside
            ctx.check(ctx.lib.sdb_sample_image(ctx.h, _lib.ptr(p_ctx.numpy()), n, L, _lib.ptr(p_unc.numpy()), Lu, 7.5, args.ddim_steps,
                                               _lib.ptr(p_lat.numpy()), 0, Hl, Hl, p_rgb.numpy().ctypes.data_as(_lib._u8p)))
        return dev_step, e2e_step, int(h_ctx.nbytes + h_unc.nbytes + h_lat.nbytes), int(p_rgb.numel()), d_rgb

    n = args.batch
    step_dev, step_e2e, h2d, d2h, d_rgb = make_steps(n)

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        e0.record(stream)
        for _ in range(k):
            fn()
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        if dist:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # one sampler process for the whole run, started before any timed region
    for _ in range(args.warmup):
        step_dev()
    l0 = ctx.launch_count()
    w0 = time.time()
    ms = timed(step_dev, args.steps)
    w1 = time.time()
    launches = ctx.launch_count() - l0
    clocks = sampler.window(w0, w1) if rank == 0 else None
    value = world * n * args.steps / (ms * 1e-3)
    if args.dump_outputs:  # d_rgb holds what the last timed step wrote; nothing has run since
        dump_outputs(args.dump_outputs, "images" if world == 1 else f"images_rank{rank}", d_rgb.cpu().numpy(),
                     DUMP_BUDGET_BYTES // world)

    # ---- end to end through the host-buffer C ABI
    step_e2e()
    barrier()
    t0 = time.perf_counter()
    ms_e2e_dev = timed(step_e2e, args.steps)
    wall = time.perf_counter() - t0
    ms_e2e = max(ms_e2e_dev, 0.0)
    # the host-buffer call is synchronous: wall clock covers the copies too; take the larger of the two clocks
    ms_e2e = max(ms_e2e, wall * 1e3) if not dist else ms_e2e
    e2e_value = world * n * args.steps / (ms_e2e * 1e-3)

    # ---- BASELINE configs[4] (64 images sharded 8 per rank over 8 GPUs) as a sub-record whenever the job is multi-GPU:
    # the same call with 8 images per rank (world * 8 images per step), its own clocks sample; the headline stays configs[1]
    c5 = None
    if world > 1 and args.batch != 8 and not args.no_c5:
        c5_dev, c5_e2e, c5_h2d, c5_d2h, _ = make_steps(8)
        for _ in range(2):
            c5_dev()
        k5 = max(2, min(args.steps, 5))
        w0 = time.time()
        ms5 = timed(c5_dev, k5)
        clk5 = sampler.window(w0, time.time()) if rank == 0 else None
        c5_e2e()
        ms5e = timed(c5_e2e, k5)
        c5 = {"workload": f"BASELINE configs[4]: SDv1-4 txt2img {args.size}x{args.size}, {args.ddim_steps} steps, cfg=7.5, "
                          f"{8 * world} images sharded 8 per rank over {world} GPUs",
              "value": world * 8 * k5 / (ms5 * 1e-3), "unit": UNIT, "steps": k5, "warmup": 2, "ms_per_step": ms5 / k5,
              "images_per_step": 8 * world, "clocks": clk5,
              "e2e": {"value": world * 8 * k5 / (ms5e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": c5_h2d, "d2h_bytes_per_step": c5_d2h}}

    # ---- per-kernel-class device time (graphs bypassed, every launch bracketed by events) for the roofline
    roof, classes = None, None
    if rank == 0 and not args.no_profile:
        ctx.profile(True)
        ctx.profile_reset()
        step_dev()
        torch.cuda.synchronize()
        classes = ctx.profile_table()
        ctx.profile(False)
        g = classes["gemm_tc"]
        pk = peaks()
        tot_ms = sum(v["ms"] for v in classes.values())
        ach = g["flops"] / (g["ms"] * 1e-3) / 1e12 if g["ms"] > 0 else 0.0
        roof = {"bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05 implicit GEMM, all conv/linear layers of one sample_image)",
                "achieved": ach, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": ach / pk["tflops"], "peak_source": pk["src"] + " bf16 cuBLAS sustained (same tensor rate as fp16)",
                "traffic": gemm_traffic_per_launch(), "algorithmic_bytes_per_launch": g["bytes"] / max(1, g["launches"]),
                "launches": g["launches"], "avg_launch_us": g["ms"] * 1e3 / max(1, g["launches"]),
                "algorithmic_tflop_per_step": g["flops"] / 1e12, "issued_tflop_per_step": g["issued_flops"] / 1e12,
                # share of the REPLAYED step (the timed value), from event-bracketed launches: an upper bound, each bracket
                # carries ~3 us of event overhead that graph replay does not pay
                "share_of_step": g["ms"] / (ms / args.steps), "profile_mode_total_ms": tot_ms,
                "whole_image_tflops": value / world * FLOP_PER_IMAGE / 1e12 if args.size == 512 and args.ddim_steps == 20 else None}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        step_s, dec, threads, what = cpu_port_times(1, latent=Hl, ddim_steps_total=args.ddim_steps)
        cpu_img_s = args.ddim_steps * step_s[0] + dec
        cpu = {"value": 1.0 / cpu_img_s, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"{what}; {step_s[0]:.2f} s/step x {args.ddim_steps} + decode {dec:.2f} s = {cpu_img_s:.1f} s/image"}

    if rank == 0:
        sampler.stop()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp16 tensor-core operands (3-term split-fp16 on the two high-res UNet levels), fp32 accumulate",
            "data": "synthetic",
            "config": workload_config(args, n),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches),
            "roofline": roof,
            "cpu_baseline": cpu,
            "kernel_classes": classes,
            "weights_broadcast_ms": bcast_ms,
        }
        if c5 is not None:
            line["c5"] = c5
        print(json.dumps(line), flush=True)
    if dist:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
