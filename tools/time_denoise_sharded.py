#!/usr/bin/env python
"""Time the row-band filters (rt_denoise_rows, rt_denoise_features_rows; DESIGN §4.8e) and the denoised sharded frame.

One GPU (plain ``python``): the complex scene at --w x --h, one --spp frame with its variance and features.  For each
N in --ranks, the band of row_bands(H, N) with the largest window (the slowest rank) is filtered two ways, for both
filters at the library defaults:
  band    the band kernel over the band's rows (``DeviceScene.denoise(rows=)``),
  window  the whole-frame kernel run on the band's halo'd window [y0 - h, y1 + h), pointers shifted to its first row
          (the alternative that needs no new kernel, and also filters the halo rows).
CUDA events around --launches launches, the two arms alternating over --reps, medians.  Both outputs are checked bit
for bit against the same rows of the whole-frame filter while it runs.

Under ``torchrun --nproc-per-node N``: ShardedPathRenderer frames of the complex scene at --w x --h and --frame-spp,
in tiles and samples modes: the plain frame, the denoised frame and the feature-denoised frame, alternating, host clock
around each frame after a device synchronise and a barrier (medians over --reps).  Rank 0 checks each denoised image
bit for bit against FrameContext.render_path(denoise=True) of the same frame on one GPU.

The card's name, power limit and max SM clock are printed first.

    python tools/time_denoise_sharded.py [--ranks 1,2,4,8] [--reps 9]
    torchrun --nproc-per-node 8 tools/time_denoise_sharded.py [--frame-spp 64]
"""
import argparse
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import ray_tracer_v1_b200 as rtb
from ray_tracer_v1_b200 import _native as nat, scenes
from ray_tracer_v1_b200.distributed import row_bands


def card(device=0):
    name = torch.cuda.get_device_name(device)
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                      # noqa: BLE001
        q = f"unknown ({e})"
    return f"{name}, power limit / max SM clock: {q}"


def complex_scene():
    spec = scenes.build_complex()
    return spec, rtb.flatten_scene(spec.spheres, background_colour=spec.background)


def one_gpu(args):
    spec, fs = complex_scene()
    W, H = args.w, args.h
    sc = nat.DeviceScene(fs)
    if sc.n > 256:
        sc.build_lbvh()
    z = lambda shape, dt=torch.float32: torch.zeros(shape, dtype=dt, device="cuda")    # noqa: E731
    acc, mom, var = z((H, W, 4)), z((H, W, 4), torch.float64), z((H, W, 3))
    feats = (z((H, W, 3)), z((H, W, 3)), z((H, W)), z((H, W, 3)))
    p = sc.path_params(spec.camera, W, H, args.spp, spec.max_bounces, spec.mirror_threshold, seed=1)
    sc.render_path(p, acc, nat.F32, moments=mom)
    sc.resolve_variance(acc, mom, W, H, var, nat.F32)
    sc.render_features(sc.path_params(spec.camera, W, H, args.spp, 1, 0.0, seed=1, samples=(0, min(args.spp, 8))),
                       *feats, precision=nat.F32)
    print(f"# {card()}")
    print(f"# complex scene {W}x{H}, {args.spp} spp, {args.launches} launches per measurement, median of {args.reps}")
    print("| filter | N | band rows | window rows | band CTAs | window CTAs | band ms | window ms | window / band |")
    print("|---|---|---|---|---|---|---|---|---|")
    for features in (False, True):
        fb = feats if features else None
        full = z((H, W, 3))
        sc.denoise(acc, var, W, H, full, nat.F32, features=fb)
        full = full.cpu().numpy()
        h = nat.denoise_halo(features=features)
        for n in args.ranks:
            bands = row_bands(H, n)
            y0, y1 = max(bands, key=lambda b: (min(H, b[1] + h) - max(0, b[0] - h), b[1] - b[0]))
            lo, hi = max(0, y0 - h), min(H, y1 + h)
            img_b, img_w = z((H, W, 3)), z((hi - lo, W, 3))
            fw = None if fb is None else tuple(f[lo:hi] for f in fb)

            def band():
                sc.denoise(acc, var, W, H, img_b, nat.F32, features=fb, rows=(y0, y1))

            def window():
                sc.denoise(acc[lo:hi], var[lo:hi], W, hi - lo, img_w, nat.F32, features=fw)

            arms = {"band": (band, []), "window": (window, [])}
            for fn, _ in arms.values():                      # warm-up, and the check against the whole frame
                fn()
            torch.cuda.synchronize()
            assert np.array_equal(img_b.cpu().numpy()[y0:y1], full[y0:y1]), ("band", n)
            assert np.array_equal(img_w.cpu().numpy()[y0 - lo:y1 - lo], full[y0:y1]), ("window", n)
            for rep in range(args.reps):
                for name in (("band", "window") if rep % 2 == 0 else ("window", "band")):
                    fn, times = arms[name]
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    for _ in range(args.launches):
                        fn()
                    b.record()
                    torch.cuda.synchronize()
                    times.append(a.elapsed_time(b) / args.launches)
            mb, mw = (statistics.median(arms[k][1]) for k in ("band", "window"))
            tiles_x = (W + 15) // 16
            print(f"| {'features' if features else 'colour'} | {n} | {y1 - y0} | {hi - lo} | "
                  f"{tiles_x * ((y1 - y0 + 15) // 16)} | {tiles_x * ((hi - lo + 15) // 16)} | {mb:.3f} | {mw:.3f} | "
                  f"{mw / mb:.3f} |", flush=True)
    sc.close()


def sharded(args):
    import torch.distributed as dist
    from ray_tracer_v1_b200.distributed import ShardedPathRenderer
    from ray_tracer_v1_b200.frames import FrameContext
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    spec, fs = complex_scene()
    W, H, spp = args.w, args.h, args.frame_spp
    frame = (spec.camera, W, H, spp, spec.max_bounces, spec.mirror_threshold)
    r = ShardedPathRenderer(device=local)
    r.set_scene(fs)
    kinds = {"plain": {}, "denoise": {"denoise": True}, "features": {"denoise": True, "features": True}}
    if rank == 0:
        print(f"# {card(local)}")
        print(f"# complex scene {W}x{H}, {spp} spp, {world} ranks, host clock per frame, median of {args.reps}")
        fc = FrameContext(local)
        fc.set_scene(fs)
        refs = {k: np.array(fc.render_path(*frame, seed=3, denoise=True, features=(k == "features"))[0])
                for k in ("denoise", "features")}
        fc.close()
        print("| mode | plain ms | denoised ms | feature-denoised ms |")
        print("|---|---|---|---|")
    for mode in ("tiles", "samples"):
        times = {k: [] for k in kinds}
        for k, kw in kinds.items():                              # warm-up and the bit-for-bit check
            img, _ = r.render(*frame, seed=3, mode=mode, **kw)
            if rank == 0 and k in refs:
                assert np.array_equal(img.cpu().numpy(), refs[k]), (mode, k)
        for rep in range(args.reps):
            order = list(kinds) if rep % 2 == 0 else list(reversed(kinds))
            for k in order:
                torch.cuda.synchronize()
                dist.barrier()
                t0 = time.perf_counter()
                r.render(*frame, seed=3, mode=mode, **kinds[k])
                torch.cuda.synchronize()
                dist.barrier()
                times[k].append((time.perf_counter() - t0) * 1e3)
        if rank == 0:
            m = {k: statistics.median(v) for k, v in times.items()}
            print(f"| {mode} | {m['plain']:.2f} | {m['denoise']:.2f} | {m['features']:.2f} |", flush=True)
    r.close()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--w", type=int, default=1920)
    ap.add_argument("--h", type=int, default=1080)
    ap.add_argument("--spp", type=int, default=16, help="samples of the frame the one-GPU mode filters")
    ap.add_argument("--frame-spp", type=int, default=64, help="samples of the sharded frames")
    ap.add_argument("--ranks", type=lambda s: [int(x) for x in s.split(",")], default=[1, 2, 4, 8])
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--launches", type=int, default=5)
    args = ap.parse_args()
    if "WORLD_SIZE" in os.environ:             # under torchrun (at --nproc-per-node 1 too)
        sharded(args)
    else:
        one_gpu(args)


if __name__ == "__main__":
    main()
