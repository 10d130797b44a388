#!/usr/bin/env python
"""Time and score the first-hit features (rt_render_features) and the feature-guided filter (rt_denoise_features).

For the complex scene and the chandelier at --w x --h and each --spp, with the DESIGN §4.8c protocol (CUDA events around
whole frames, alternating reps, medians; RMSE of the image in levels against the floored mean of a uniform --ref-spp
frame rendered with seed 1000):
  - the noisy frame (path kernel + resolve),
  - the colour-only filter at the library defaults (r 10, f 3, k 0.45),
  - the feature-guided filter over the grid f x k x k_f (r 10, tau 1e-3), each frame's features taken over its first
    min(spp, --feature-spp) samples.
Then the feature kernel alone at FEATURE_SPP 4 / 8 / 16 (camera rays and nearest-hit queries per second) and the filter
kernel with and without features.  The card's name, power limit and clock are printed first.

    python tools/time_features.py [--reps 3] [--spp 4,16,64] [--f 1,3] [--k 0.45,0.7,1.0] [--kf 0.3,0.6,1.2]
"""
import argparse
import itertools
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
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm,clocks.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                      # noqa: BLE001
        q = f"unknown ({e})"
    return f"{name}, power limit / max SM clock / SM clock: {q}"


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


class Frames:
    def __init__(self, sc, spec, W, H, feature_spp):
        self.sc, self.spec, self.W, self.H, self.feature_spp = sc, spec, W, H, feature_spp
        z = lambda shape, dt=torch.float32: torch.zeros(shape, dtype=dt, device="cuda")    # noqa: E731
        self.accum, self.moments = z((H, W, 4)), z((H, W, 4), torch.float64)
        self.image, self.var = z((H, W, 3)), z((H, W, 3))
        self.features = (z((H, W, 3)), z((H, W, 3)), z((H, W)), z((H, W, 3)))

    def params(self, spp, seed, samples=None):
        s = self.spec
        return self.sc.path_params(s.camera, self.W, self.H, spp, s.max_bounces, s.mirror_threshold, seed=seed,
                                   samples=samples)

    def noisy(self, spp, seed):
        self.sc.render_path(self.params(spp, seed), self.accum, nat.F32)
        self.sc.resolve(self.accum, self.W, self.H, spp, self.image, nat.F32)

    def render_features(self, spp, seed, nf=None):
        nf = min(spp, self.feature_spp) if nf is None else nf
        self.sc.render_features(self.params(nf, seed, samples=(0, nf)), *self.features, precision=nat.F32)

    def denoised(self, spp, seed, setting):
        self.sc.render_path(self.params(spp, seed), self.accum, nat.F32, moments=self.moments)
        self.sc.resolve_variance(self.accum, self.moments, self.W, self.H, self.var, nat.F32)
        if setting[3] is not None:
            self.render_features(spp, seed)
        self.filter(setting)

    def filter(self, setting):
        r, f, k, kf = setting
        extra = {} if kf is None else dict(features=self.features, k_f=kf)
        self.sc.denoise(self.accum, self.var, self.W, self.H, self.image, nat.F32, radius=r, patch_radius=f, k=k, **extra)


def name(s):
    return f"r{s[0]} f{s[1]} k{s[2]:g}" + ("" if s[3] is None else f" kf{s[3]:g}")


def run_scene(label, spec, args):
    sc = nat.DeviceScene(rtb.flatten_scene(spec.spheres, background_colour=spec.background))
    if sc.n > 256:
        sc.build_lbvh()
    W, H = args.w, args.h
    F = Frames(sc, spec, W, H, args.feature_spp)
    F.noisy(args.ref_spp, seed=1000)
    torch.cuda.synchronize()
    ref = torch.floor(F.accum[..., :3].double() / args.ref_spp).cpu().numpy()

    def rmse():
        torch.cuda.synchronize()
        return float(np.sqrt(np.mean((F.image.double().cpu().numpy() * 255.0 - ref) ** 2)))

    colour = (10, 3, 0.45, None)
    grid = [(10, f, k, kf) for f, k, kf in itertools.product([int(v) for v in args.f.split(",")],
                                                             [float(v) for v in args.k.split(",")],
                                                             [float(v) for v in args.kf.split(",")])]
    print(f"\n{label} {W}x{H}, FP32 accum, {sc.n} spheres; RMSE in levels against a uniform {args.ref_spp}-spp frame "
          f"(seed 1000); features over the first min(spp, {args.feature_spp}) samples; {args.reps} alternating reps")
    print(f"{'frame':>34} {'median ms':>10} {'RMSE':>7}")
    for spp in [int(s) for s in args.spp.split(",")]:
        variants = [(f"{spp} spp noisy", lambda spp=spp: F.noisy(spp, 1))]
        variants += [(f"{spp} spp {name(s)}", lambda spp=spp, s=s: F.denoised(spp, 1, s)) for s in [colour] + grid]
        for _, fn in variants:
            fn()
        torch.cuda.synchronize()
        times = {v[0]: [] for v in variants}
        for _ in range(args.reps):
            for lab, fn in variants:
                times[lab].append(timed(fn))
        for lab, fn in variants:
            fn()
            print(f"{lab:>34} {np.median(times[lab]):10.3f} {rmse():7.3f}", flush=True)

    # the feature kernel alone: camera rays and nearest-hit queries (one per ray) per second
    print(f"feature kernel alone ({label}):")
    for nf in (4, 8, 16):
        F.render_features(nf, 1, nf)
        ms = float(np.median([timed(lambda nf=nf: F.render_features(nf, 1, nf)) for _ in range(args.kernel_reps)]))
        rays = W * H * nf
        print(f"  FEATURE_SPP {nf:2d}: {ms:.3f} ms, {rays / 1e6:.1f} M rays = {rays / ms / 1e6:.2f} G rays/s, "
              f"{rays * sc.n / ms / 1e9:.2f} T brute-force sphere tests/s equivalent", flush=True)
    print(f"filter kernel alone ({label}, on the last 64-spp frame and its 8-sample features):")
    F.denoised(64, 1, (10, 3, 0.45, 0.6))
    for s in (colour, (10, 3, 0.45, 0.6), (10, 1, 0.7, None), (10, 1, 0.7, 0.6)):
        F.filter(s)
        ms = float(np.median([timed(lambda s=s: F.filter(s)) for _ in range(args.kernel_reps)]))
        print(f"  {name(s):>22}: {ms:.3f} ms", flush=True)
    sc.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--w", type=int, default=1920)
    ap.add_argument("--h", type=int, default=1080)
    ap.add_argument("--spp", default="4,16,64")
    ap.add_argument("--f", default="1,3", help="patch radii of the feature grid")
    ap.add_argument("--k", default="0.45,0.7,1.0", help="colour k of the feature grid")
    ap.add_argument("--kf", default="0.3,0.6,1.2", help="k_f of the feature grid")
    ap.add_argument("--feature-spp", type=int, default=8)
    ap.add_argument("--scenes", default="complex,chandelier")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--kernel-reps", type=int, default=20)
    ap.add_argument("--ref-spp", type=int, default=4096)
    args = ap.parse_args()
    print(card(), flush=True)
    for label in args.scenes.split(","):
        run_scene(label, {"complex": scenes.build_complex, "chandelier": scenes.build_chandelier}[label](), args)


if __name__ == "__main__":
    main()
