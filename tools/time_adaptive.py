#!/usr/bin/env python
"""Time adaptive Algorithm B frames (rt_render_path_adaptive) against the uniform frame, on the complex scene.

Alternating in one process: the uniform frame (path kernel + resolve, --spp samples) and adaptive frames (min_spp,
max_spp, each tolerance), CUDA events around whole frames.  For every frame: median ms, mean samples per pixel and the
RMSE of the resolved image (levels, 0-255) against a uniform --ref-spp frame rendered with another seed.  Then one
profiled frame per tolerance gives the device time of each round and the active fraction entering it, and the list
launches' ms per G pixel-samples against the uniform launch's.  The card's name and power limit are printed first.

    python tools/time_adaptive.py [--reps 5] [--tolerances 1,2,4,8]
"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import ray_tracer_v1_b200 as rtb
from ray_tracer_v1_b200 import _native as nat, scenes


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                      # noqa: BLE001
        q = f"unknown ({e})"
    return f"{name}, power limit / max SM clock: {q}"


class Frames:
    def __init__(self, sc, spec, W, H):
        self.sc, self.spec, self.W, self.H = sc, spec, W, H
        dev = "cuda"
        self.accum = torch.zeros((H, W, 4), dtype=torch.float32, device=dev)
        self.moments = torch.zeros((H, W, 4), dtype=torch.float64, device=dev)
        self.list = torch.zeros(H * W + 1, dtype=torch.int32, device=dev)
        self.image = torch.zeros((H, W, 3), dtype=torch.float32, device=dev)
        self.var = torch.zeros((H, W, 3), dtype=torch.float32, device=dev)
        self.counts = torch.zeros((H, W), dtype=torch.int32, device=dev)
        self.stats = torch.zeros(8, dtype=torch.int64, device=dev)

    def params(self, spp, seed):
        s = self.spec
        return self.sc.path_params(s.camera, self.W, self.H, spp, s.max_bounces, s.mirror_threshold, seed=seed)

    def uniform(self, spp, seed):
        self.stats.zero_()
        self.sc.render_path(self.params(spp, seed), self.accum, nat.F32, stats=self.stats)
        self.sc.resolve(self.accum, self.W, self.H, spp, self.image, nat.F32)

    def adaptive(self, min_spp, max_spp, tol, seed):
        self.stats.zero_()
        self.sc.render_path_adaptive(self.params(max_spp, seed), min_spp, tol, self.accum, self.moments, self.list,
                                     self.image, nat.F32, var=self.var, counts=self.counts, stats=self.stats)


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--w", type=int, default=1920)
    ap.add_argument("--h", type=int, default=1080)
    ap.add_argument("--spp", type=int, default=64, help="samples per pixel of the uniform frame")
    ap.add_argument("--min-spp", type=int, default=16)
    ap.add_argument("--max-spp", type=int, default=256)
    ap.add_argument("--tolerances", default="1,2,4,8", help="comma-separated, colour levels")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--ref-spp", type=int, default=4096)
    args = ap.parse_args()
    print(card(), flush=True)
    spec = scenes.build_complex()
    sc = nat.DeviceScene(rtb.flatten_scene(spec.spheres, background_colour=spec.background))
    W, H = args.w, args.h
    F = Frames(sc, spec, W, H)
    tols = [float(t) for t in args.tolerances.split(",")]

    # reference: the mean of a long uniform frame with another seed, in levels (as the resolve floors it)
    F.uniform(args.ref_spp, seed=1000)
    torch.cuda.synchronize()
    ref = torch.floor(F.accum[..., :3].double() / args.ref_spp).cpu().numpy()

    def rmse():
        return float(np.sqrt(np.mean((F.image.double().cpu().numpy() * 255.0 - ref) ** 2)))

    variants = [("uniform", args.spp, lambda: F.uniform(args.spp, seed=1))]
    for t in tols:
        variants.append((f"adaptive tol {t:g}", t, (lambda t=t: F.adaptive(args.min_spp, args.max_spp, t, seed=1))))
    for _, _, fn in variants:                                      # warm-up: module loads, shared-memory opt-in
        fn()
    torch.cuda.synchronize()
    times = {name: [] for name, _, _ in variants}
    for _ in range(args.reps):
        for name, _, fn in variants:
            times[name].append(timed(fn))
    print(f"\ncomplex {W}x{H}, uniform {args.spp} spp against adaptive min {args.min_spp} max {args.max_spp}; "
          f"RMSE in levels against a uniform {args.ref_spp}-spp frame (seed 1000); {args.reps} alternating reps")
    print(f"{'frame':>20} {'median ms':>10} {'min ms':>8} {'mean spp':>9} {'RMSE':>7} {'rays':>12}")
    for name, arg, fn in variants:
        fn()
        torch.cuda.synchronize()
        spp = float(args.spp) if name == "uniform" else float(F.counts.double().mean())
        print(f"{name:>20} {np.median(times[name]):10.3f} {min(times[name]):8.3f} {spp:9.2f} {rmse():7.3f} "
              f"{int(F.stats[0]):12d}", flush=True)

    # rounds: device time of every kernel of one frame (a profiled run of its own), grouped by round
    from torch.profiler import ProfilerActivity, profile
    print("\nrounds (one profiled frame each): active = fraction of pixels entering the round; Gps = G pixel-samples")
    for name, arg, fn in variants:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        evs = sorted((e for e in prof.events() if e.device_type.name == "CUDA"), key=lambda e: e.time_range.start)
        kern = [(e.name, e.device_time) for e in evs if "memset" not in e.name.lower() and "memcpy" not in e.name.lower()]
        paths = [(n, t / 1000.0) for n, t in kern if "path_kernel" in n]
        other = sum(t for n, t in kern if "path_kernel" not in n) / 1000.0
        if name == "uniform":
            gps = W * H * args.spp / 1e9
            print(f"  {name}: path kernel {paths[0][1]:.3f} ms = {paths[0][1] / gps:.3f} ms/Gps; other kernels {other:.3f} ms")
            continue
        counts = F.counts.cpu().numpy()
        c, lo = args.min_spp, 0
        rows = []
        for r, (_, ms) in enumerate(paths):
            active = float(np.mean(counts > lo)) if r else 1.0
            hi = c
            n_ps = int(np.sum(np.minimum(counts, hi) - np.minimum(counts, lo)))
            rows.append(f"r{r} [{lo},{hi}) active {active:.4f} {ms:.3f} ms {ms / (n_ps / 1e9) if n_ps else 0:.3f} ms/Gps")
            lo, c = hi, min(2 * hi, args.max_spp)
        list_ms = sum(ms for _, ms in paths[1:])
        list_ps = float(np.sum(counts - np.minimum(counts, args.min_spp))) / 1e9
        print(f"  {name}: " + "; ".join(rows) + f"; select + resolve {other:.3f} ms; list launches together "
              f"{(list_ms / list_ps) if list_ps else 0:.3f} ms/Gps", flush=True)
    sc.close()


if __name__ == "__main__":
    main()
