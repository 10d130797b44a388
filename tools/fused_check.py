#!/usr/bin/env python
"""Fused multi-GPU sinks (single launch per rank and frame; the round-1 launch chain) vs the NCCL paths: same frame bit
for bit, device-timed side by side.

    python tools/fused_check.py                                   # 1 GPU (peers = self)
    torchrun --nproc-per-node N --master-addr 127.0.0.1 tools/fused_check.py [--spp 64]

--variance: per-pixel variance through every path instead.  For each mode, rank 0's variance from render and from
render_fused (single launch and chain) is compared bit for bit with the 1-GPU render_path(..., variance=True), each
image with the same call without variance, and plain and variance frames of every path are timed alternately.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
    os.environ["NCCL_DEBUG"] = "WARN"
import numpy as np
import torch
import torch.distributed as dist

import ray_tracer_v1_b200 as rtb
from ray_tracer_v1_b200 import _native as nat, scenes
from ray_tracer_v1_b200.distributed import ShardedPathRenderer


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--spp", type=int, default=16)
    ap.add_argument("--w", type=int, default=1920)
    ap.add_argument("--h", type=int, default=1080)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--scene", default="complex")
    ap.add_argument("--variance", action="store_true", help="check and time the per-pixel variance of every path")
    args = ap.parse_args()
    rank, world, local = (int(os.environ.get(k, d)) for k, d in (("RANK", 0), ("WORLD_SIZE", 1), ("LOCAL_RANK", 0)))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    spec = scenes.build_complex() if args.scene == "complex" else scenes.build_chandelier()
    fs = rtb.flatten_scene(spec.spheres, background_colour=spec.background)
    r = ShardedPathRenderer(device=local)
    r.set_scene(fs)
    W, H, spp = args.w, args.h, args.spp
    depth, thr = spec.max_bounces, spec.mirror_threshold

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    out = {"world": world, "scene": args.scene, "spp": spp}
    if args.variance:
        out["variance"] = True
        check_variance(args, r, spec, fs, rank, world, sync, out)
        out["timed_out"] = r.fused_timed_out()
        if rank == 0:
            print(json.dumps(out), flush=True)
        r.close()
        if world > 1:
            dist.destroy_process_group()
        return
    for mode in ("tiles", "samples"):
        ref, _ = r.render(spec.camera, W, H, spp, depth, thr, seed=3, mode=mode)
        ref = ref.clone() if rank == 0 else None
        img, _ = r.render_fused(spec.camera, W, H, spp, depth, thr, seed=3, mode=mode)
        sync()
        if rank == 0:
            out[f"{mode}_identical"] = bool(torch.equal(ref, img))
            out[f"{mode}_maxdiff"] = float((ref - img).abs().max())
        chain = lambda *a, **k: r.render_fused(*a, in_kernel=False, **k)      # round-1 chain of wait / signal / resolve launches
        img2, _ = chain(spec.camera, W, H, spp, depth, thr, seed=3, mode=mode)
        sync()
        if rank == 0:
            out[f"{mode}_chain_identical"] = bool(torch.equal(ref, img2))
        for name, fn in (("nccl", r.render), ("chain", chain), ("fused", r.render_fused)):
            for i in range(2):
                fn(spec.camera, W, H, spp, depth, thr, seed=10 + i, mode=mode)
            sync()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(args.reps):
                fn(spec.camera, W, H, spp, depth, thr, seed=20 + i, mode=mode)
            b.record()
            sync()
            t = torch.tensor([a.elapsed_time(b) / args.reps], device="cuda")
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            out[f"{mode}_{name}_ms"] = float(t)
    out["timed_out"] = r.fused_timed_out()
    if rank == 0:
        print(json.dumps(out), flush=True)
    r.close()
    if world > 1:
        dist.destroy_process_group()


def check_variance(args, r, spec, fs, rank, world, sync, out):
    """Bit-exactness of every path's variance against one GPU, and plain vs variance ms/frame of every path."""
    W, H, spp = args.w, args.h, args.spp
    depth, thr = spec.max_bounces, spec.mirror_threshold
    cam = spec.camera
    ref_var = None
    if rank == 0:
        from ray_tracer_v1_b200.renderers import render_path
        _, _, ref_var = render_path(fs, cam, W, H, spp, depth, thr, seed=3, variance=True)
    paths = {"nccl": r.render, "fused": r.render_fused,
             "chain": lambda *a, **k: r.render_fused(*a, in_kernel=False, **k)}
    for mode in ("tiles", "samples"):
        for name, fn in paths.items():
            img, _ = fn(cam, W, H, spp, depth, thr, seed=3, mode=mode)
            img = img.clone() if rank == 0 else None
            img_v, _, var = fn(cam, W, H, spp, depth, thr, seed=3, mode=mode, variance=True)
            sync()
            if rank == 0:
                out[f"{mode}_{name}_var_identical"] = bool(np.array_equal(var.cpu().numpy(), ref_var))
                out[f"{mode}_{name}_image_identical"] = bool(torch.equal(img, img_v))
        for name, fn in paths.items():
            for variance in (False, True):                  # warm both kernels
                fn(cam, W, H, spp, depth, thr, seed=10, mode=mode, variance=variance)
            sync()
            times = {False: [], True: []}
            for i in range(2 * args.reps):                    # alternate plain and variance frames
                variance = bool(i & 1)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn(cam, W, H, spp, depth, thr, seed=20 + i, mode=mode, variance=variance)
                b.record()
                sync()
                times[variance].append(a.elapsed_time(b))
            for variance, key in ((False, "ms"), (True, "var_ms")):
                t = torch.tensor([float(np.median(times[variance]))], device="cuda")
                if world > 1:
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                out[f"{mode}_{name}_{key}"] = round(float(t), 3)


if __name__ == "__main__":
    main()
