#!/usr/bin/env python
"""Time and score the variance-guided non-local-means filter (rt_denoise) on the complex scene.

Alternating in one process, CUDA events around whole frames: uniform frames at each --spp, noisy (path kernel + resolve)
and denoised (path kernel with moments + variance resolve + rt_denoise) with each filter setting, and one adaptive frame
(min 16, max 256 spp, tolerance --tolerance) denoised with each setting.  For every frame: median ms, mean samples per
pixel and the RMSE of the image (levels, 0-255) against the floored mean of a uniform --ref-spp frame rendered with seed
1000, as tools/time_adaptive.py measures it.  Then the filter's own kernel time per setting (CUDA events around --kernel-reps
launches), with the pipe that bounds it from the operation counts over that time.  The card's name and power limit are
printed first.

    python tools/time_denoise.py [--reps 5] [--spp 16,32,64] [--settings 10:3:0.45,10:1:0.7]
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

    def params(self, spp, seed):
        s = self.spec
        return self.sc.path_params(s.camera, self.W, self.H, spp, s.max_bounces, s.mirror_threshold, seed=seed)

    def noisy(self, spp, seed):
        self.sc.render_path(self.params(spp, seed), self.accum, nat.F32)
        self.sc.resolve(self.accum, self.W, self.H, spp, self.image, nat.F32)

    def denoised(self, spp, seed, setting):
        self.sc.render_path(self.params(spp, seed), self.accum, nat.F32, moments=self.moments)
        self.sc.resolve_variance(self.accum, self.moments, self.W, self.H, self.var, nat.F32)
        self.filter(setting)

    def adaptive(self, tol, seed, setting):
        self.sc.render_path_adaptive(self.params(256, seed), 16, tol, self.accum, self.moments, self.list, self.image, nat.F32,
                                     var=self.var, counts=self.counts)
        self.filter(setting)

    def filter(self, setting):
        r, f, k = setting
        self.sc.denoise(self.accum, self.var, self.W, self.H, self.image, nat.F32, radius=r, patch_radius=f, k=k)


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def op_counts(W, H, r, f):
    """FP32, MUFU and 4-byte shared-memory load operations of one filter launch, counted from denoise_nlm_kernel's
    source (16 x 16 tiles): per offset and tile, (16 + 2f)^2 patch distances of 3 channels (2 loads; sub, mul, add, min,
    add, fma, the divide's multiply and the channel sum -> 9 FP32 and one MUFU.RCP each, plus the 1/3 scale),
    (16 + 2f) x 16 row sums and 16 x 16 column sums of 2f + 1 loads and adds, and per pixel 3 loads, a mul, max, the
    MUFU.EX2 input scale, one add and three FMA."""
    tiles = ((W + 15) // 16) * ((H + 15) // 16)
    R, P, offsets = 16 + 2 * f, 2 * f + 1, (2 * r + 1) ** 2
    fp32 = tiles * offsets * (R * R * (3 * 9 + 1) + (R * 16 + 256) * P + 256 * 7)
    mufu = tiles * offsets * (R * R * 3 + 256)
    lds = tiles * offsets * (R * R * 6 + (R * 16 + 256) * P + 256 * 3)
    return fp32, mufu, lds


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--w", type=int, default=1920)
    ap.add_argument("--h", type=int, default=1080)
    ap.add_argument("--spp", default="16,32,64", help="comma-separated samples per pixel of the uniform frames")
    ap.add_argument("--tolerance", type=float, default=8.0, help="adaptive frame tolerance, colour levels")
    ap.add_argument("--settings", default="10:3:0.45,10:1:0.7", help="filter settings radius:patch_radius:k")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--kernel-reps", type=int, default=20)
    ap.add_argument("--ref-spp", type=int, default=4096)
    args = ap.parse_args()
    print(card(), flush=True)
    spec = scenes.build_complex()
    sc = nat.DeviceScene(rtb.flatten_scene(spec.spheres, background_colour=spec.background))
    W, H = args.w, args.h
    F = Frames(sc, spec, W, H)
    spps = [int(s) for s in args.spp.split(",")]
    settings = [tuple(t(v) for t, v in zip((int, int, float), s.split(":"))) for s in args.settings.split(",")]

    F.noisy(args.ref_spp, seed=1000)
    torch.cuda.synchronize()
    ref = torch.floor(F.accum[..., :3].double() / args.ref_spp).cpu().numpy()

    def rmse():
        return float(np.sqrt(np.mean((F.image.double().cpu().numpy() * 255.0 - ref) ** 2)))

    def name(s):
        return f"r{s[0]} f{s[1]} k{s[2]:g}"

    variants = []
    for spp in spps:
        variants.append((f"{spp} spp noisy", spp, lambda spp=spp: F.noisy(spp, seed=1)))
        for s in settings:
            variants.append((f"{spp} spp {name(s)}", spp, lambda spp=spp, s=s: F.denoised(spp, 1, s)))
    for s in settings:
        variants.append((f"adaptive {args.tolerance:g} {name(s)}", None, lambda s=s: F.adaptive(args.tolerance, 1, s)))
    for _, _, fn in variants:                                      # warm-up: module loads, shared-memory opt-in
        fn()
    torch.cuda.synchronize()
    times = {v[0]: [] for v in variants}
    for _ in range(args.reps):
        for label, _, fn in variants:
            times[label].append(timed(fn))

    # the filter alone, on the last frame's sums and variance
    kernel_ms = {}
    for s in settings:
        F.filter(s)
        torch.cuda.synchronize()
        kernel_ms[s] = float(np.median([timed(lambda s=s: F.filter(s)) for _ in range(args.kernel_reps)]))

    print(f"\ncomplex {W}x{H}, FP32 accum; RMSE in levels against a uniform {args.ref_spp}-spp frame (seed 1000); "
          f"{args.reps} alternating reps")
    print(f"{'frame':>28} {'median ms':>10} {'min ms':>8} {'filter ms':>9} {'mean spp':>9} {'RMSE':>7}")
    for label, spp, fn in variants:
        fn()
        torch.cuda.synchronize()
        mean_spp = float(spp) if spp else float(F.counts.double().mean())
        s = next((s for s in settings if label.endswith(name(s))), None)
        filt = f"{kernel_ms[s]:9.3f}" if s else f"{'-':>9}"
        print(f"{label:>28} {np.median(times[label]):10.3f} {min(times[label]):8.3f} {filt} {mean_spp:9.2f} {rmse():7.3f}",
              flush=True)

    print("\nfilter kernel (denoise_nlm_kernel) alone: operations counted from the source over the median kernel time")
    for s in settings:
        fp32, mufu, lds = op_counts(W, H, s[0], s[1])
        t = kernel_ms[s] / 1e3
        print(f"  {name(s)}: {kernel_ms[s]:.3f} ms, {fp32 / 1e9:.1f} G FP32 ops = {fp32 / t / 1e12:.1f} T/s, "
              f"{mufu / 1e9:.2f} G MUFU ops = {mufu / t / 1e12:.2f} T/s, {lds / 1e9:.1f} G shared loads = "
              f"{4 * lds / t / 1e12:.1f} TB/s", flush=True)
    sc.close()


if __name__ == "__main__":
    main()
