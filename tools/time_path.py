#!/usr/bin/env python
"""Device-time the path kernel alone (CUDA events) for scene / spp / ksplit variants and the diagnostic schedule bits
(rt_path_params.schedule: 2 = no camera-ray candidate lists, 4 = no parameter-block kernel).  Development aid.

--moments: the plain launch and the launch that also stores the per-pixel second moments (rt_render_path_moments),
alternately in one process; prints both times, the overhead, and whether the two accumulation buffers are the same."""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hashlib
import numpy as np
import torch

import ray_tracer_v1_b200 as rtb
from ray_tracer_v1_b200 import _native as nat, scenes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scene", default="complex")
    ap.add_argument("--spp", type=int, default=16)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--w", type=int, default=1920)
    ap.add_argument("--h", type=int, default=1080)
    ap.add_argument("--lbvh", action="store_true")
    ap.add_argument("--ksplit", type=int, default=-1, help="-1 auto, 0 off, k = lanes per pixel")
    ap.add_argument("--schedules", default="0", help="comma-separated schedule values, e.g. 0,2,4")
    ap.add_argument("--no-stats", action="store_true", help="launch without the statistics counters")
    ap.add_argument("--save", default=None, help="write the last accumulation buffer to this .npy")
    ap.add_argument("--moments", action="store_true", help="time the plain and the moments launch alternately")
    args = ap.parse_args()
    if args.scene.startswith("scaled"):           # scaled1000 / scaled10000 / scaled100000: SURVEY 8d's LBVH variant of C4
        spec = scenes.build_chandelier()
        fs = scenes.build_many_spheres_flat(int(args.scene[6:]), seed=0)
        args.lbvh = True
    else:
        spec = scenes.build_complex() if args.scene == "complex" else scenes.build_chandelier()
        fs = rtb.flatten_scene(spec.spheres, background_colour=spec.background)
    sc = nat.DeviceScene(fs)
    if args.lbvh:
        sc.build_lbvh(50.0)
    W, H = args.w, args.h
    accum = torch.zeros((H, W, 4), dtype=torch.float32, device="cuda")
    stats = torch.zeros(8, dtype=torch.int64, device="cuda")
    ref = None
    if args.moments:
        time_moments(sc, spec, args, accum, stats)
        return
    for schedule in [int(v) for v in args.schedules.split(',')]:
        p = sc.path_params(spec.camera, W, H, args.spp, spec.max_bounces, spec.mirror_threshold, seed=1, schedule=schedule, ksplit=args.ksplit)
        sc.render_path(p, accum, nat.F32, stats=stats)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(args.reps):
            stats.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); sc.render_path(p, accum, nat.F32, stats=None if args.no_stats else stats); b.record()
            torch.cuda.synchronize()
            best = min(best, a.elapsed_time(b))
        st = stats.cpu().numpy()
        img = accum.cpu().numpy()
        same = None if ref is None else bool(np.array_equal(ref, img))
        ref = img if ref is None else ref
        if args.save:
            np.save(args.save, img)
        print(f"{args.scene} {W}x{H} spp {args.spp} schedule {schedule} ksplit {args.ksplit}: {best:.3f} ms  {st[4] / best / 1e6:.2f} Gqueries/s "
              f"rays/sample {st[0] / (W * H * args.spp):.3f}  tests/query {st[5] / st[4]:.1f} boxes/query {st[6] / st[4]:.1f} same_image={same} "
              f"sha1 {hashlib.sha1(np.ascontiguousarray(img).tobytes()).hexdigest()[:12]}", flush=True)


def time_moments(sc, spec, args, accum, stats):
    W, H = args.w, args.h
    moments = torch.zeros((H, W, 4), dtype=torch.float64, device="cuda")
    sha = lambda t: hashlib.sha1(np.ascontiguousarray(t.cpu().numpy()).tobytes()).hexdigest()[:12]      # noqa: E731
    for schedule in [int(v) for v in args.schedules.split(',')]:
        p = sc.path_params(spec.camera, W, H, args.spp, spec.max_bounces, spec.mirror_threshold, seed=1, schedule=schedule, ksplit=args.ksplit)
        variants = (("plain", None), ("moments", moments))
        for _, m in variants:                                              # warm-up: module load, smem opt-in
            sc.render_path(p, accum, nat.F32, stats=stats, moments=m)
        torch.cuda.synchronize()
        times, digest = {k: [] for k, _ in variants}, {}
        for _ in range(args.reps):
            for name, m in variants:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); sc.render_path(p, accum, nat.F32, stats=None if args.no_stats else stats, moments=m); b.record()
                torch.cuda.synchronize()
                times[name].append(a.elapsed_time(b))
                digest[name] = sha(accum)
        t0, t1 = np.median(times["plain"]), np.median(times["moments"])
        print(f"{args.scene} {W}x{H} spp {args.spp} schedule {schedule} ksplit {args.ksplit} ({args.reps} alternating reps, "
              f"median / min): plain {t0:.3f} / {min(times['plain']):.3f} ms  moments {t1:.3f} / {min(times['moments']):.3f} ms  "
              f"overhead {100.0 * (t1 / t0 - 1):+.2f} %  accum sha1 plain {digest['plain']} moments {digest['moments']} "
              f"same={digest['plain'] == digest['moments']}", flush=True)


if __name__ == "__main__":
    main()
