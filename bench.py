#!/usr/bin/env python
"""Headline benchmark: Mrays/s and ms/frame of the traditional path tracer (Algorithm B, TraditionalRenderer.render)
on the complex scene, 1920x1080, 64 spp (BASELINE.json configs[2]) at N = 1/2/4/8 B200, tile-sharded.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # own arm (CUDA)
    python bench.py ... --dump-outputs DIR                         # + the last timed step's frame and counters as .npy
    python bench.py --impl reference [...]                         # the CPU port of the reference (oracle/, OpenMP)
    torchrun --nproc-per-node N ... bench.py --gpus N ...          # N > 1, one rank per GPU over NCCL

A step = one frame.  A ray = one nearest-hit query (SURVEY.md 8d); `rays_ref_compatible` counts like the reference's
own `total_rays` (every trace_ray_traditional call, including the ones that return at the depth check).
`value` is device-timed with inputs resident in HBM; `e2e` goes through the reference-facing API with host buffers
(scene flattening + upload in, float32 image out, every step).  One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# stdout carries ONE JSON line.  Libraries write banners to fd 1 behind Python's back (NCCL prints "NCCL version ..."
# there whenever NCCL_DEBUG >= VERSION), so fd 1 is pointed at stderr for the whole run and the JSON line goes to a
# private duplicate of the original stdout.
JSON_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)

import numpy as np  # noqa: E402

W, H, SPP, DEPTH, THRESHOLD, FOV = 1920, 1080, 64, 5, 0.9, 60.0
NCU_SUMMARY = os.path.join(ROOT, "profiles", "ncu_path_kernel_r2.txt")     # `ncu --set full` summary of one 64-spp launch of the committed kernel
SUSTAINED_SECONDS = 5.0
CPU_W, CPU_H, CPU_SPP = 960, 540, 16          # bounded CPU sample: 1/16 of the frame's pixel-samples
METRIC, UNIT = "Mrays/s (complex scene, 1920x1080, 64 spp)", "Mrays/s"
WORKLOAD = "complex scene (54 spheres, 3 lights) 1920x1080 64 spp depth 5, Algorithm B (TraditionalRenderer)"


def complex_scene():
    import ray_tracer_v1_b200 as rtb
    from ray_tracer_v1_b200 import scenes
    spec = scenes.build_complex()
    fs = rtb.flatten_scene(spec.spheres, background_colour=spec.background)
    return spec, fs


def ncu_dram_bytes():
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel, read from the committed ncu
    summary (profiles/); None when the summary is absent.  (DRAM counters cannot be read outside a profiler; a number
    measured under ncu is never a bench value, so this is the one figure of the line that comes from a capture.)"""
    unit = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    try:
        tot, seen = 0.0, 0
        for line in open(NCU_SUMMARY):
            f = line.split()
            if len(f) >= 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                tot += float(f[1]) * unit.get(f[2], 1); seen += 1
        return int(tot) if seen == 2 else None
    except OSError:
        return None


def flop_per_query(n_spheres, n_lights):
    """SURVEY.md 8d: 20 FLOP per ray-sphere test x N, + hit point/normal 15 + 25 per light + bounce/TBN/fold 70."""
    return 20 * n_spheres + 15 + 25 * n_lights + 70


def dump_outputs(out_dir, image, stats):
    """--dump-outputs: the frame and counters one timed step returned to its caller, whole (25 MB), so that two builds
    can be compared output for output.  Step i renders with seed i, so equal arguments give equal inputs.
      image.npy  float32 [H, W, 3], the resolved frame
      stats.npy  float64 [8], the path kernel's uint64 counter block (exact: every count is far below 2**53)"""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "image.npy"), image.detach().cpu().numpy().astype(np.float32, copy=False))
    np.save(os.path.join(out_dir, "stats.npy"), stats.detach().cpu().numpy().astype(np.float64))


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
    NOTE = {"sw_power_cap": 0x4}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        while self.ok and not self._stop_evt.is_set():
            try:
                self.samples.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                try:
                    mask = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for name, bit in {**self.BAD, **self.NOTE}.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(0.01)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        return {"sm_mhz": (statistics.median(self.samples) if self.samples else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------ CPU legs
def cpu_port_run(fs, spec, width, height, spp, seed, threads):
    """The oracle's C restatement of TraditionalRenderer.render on the host cores (OpenMP).  -> (queries, rays, seconds)"""
    from oracle import oracle as orc
    t0 = time.perf_counter()
    _, st = orc.render_path(fs, spec.camera, width, height, spp, DEPTH, THRESHOLD, seed=seed, fov=FOV, nthreads=threads)
    dt = time.perf_counter() - t0
    return st["queries"], st["total_rays"], dt


def host_threads():
    from oracle import oracle as orc
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    return max(1, min(avail, orc.max_threads() if orc.max_threads() > 1 else avail))


def cpu_baseline(fs, spec):
    """Bounded sample of the SAME workload (same scene, depth, camera): 960x540 x 16 spp = 1/16 of the frame's
    pixel-samples, ~40 M queries, ~30 core-seconds of CPU work."""
    threads = host_threads()
    cpu_port_run(fs, spec, 96, 54, 2, 1, threads)        # warm the library / thread pool
    q, r, dt = cpu_port_run(fs, spec, CPU_W, CPU_H, CPU_SPP, 0, threads)
    return {"value": q / dt / 1e6, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{CPU_W}x{CPU_H} x {CPU_SPP} spp of the same scene/depth/camera ({q} queries, {r} reference-counted rays, {dt:.2f} s); "
                      "oracle/rt_oracle.c (C, FP64, OpenMP) -- the reference itself is single-threaded Python "
                      "(3.3-7.4 krays/s published, BASELINE.md)",
            "rays_ref_compatible_per_s": r / dt / 1e6}


def run_reference_arm(args):
    """--impl reference: the CPU port of the reference's path on all host threads, same metric/config; each step a
    bounded sample (960x540 x 16 spp, 1/16 of the frame) of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    spec, fs = complex_scene()
    threads = host_threads()
    sw, sh, sspp = CPU_W, CPU_H, CPU_SPP
    for i in range(args.warmup):
        cpu_port_run(fs, spec, 96, 54, 2, 100 + i, threads)
    q_tot = r_tot = 0
    t_tot = 0.0
    for i in range(args.steps):
        q, r, dt = cpu_port_run(fs, spec, sw, sh, sspp, i, threads)
        q_tot += q; r_tot += r; t_tot += dt
    value = q_tot / t_tot / 1e6
    sample = f"{sw}x{sh} x {sspp} spp of the same scene/depth/camera per step"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample": sample},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "rays_ref_compatible_per_s": r_tot / t_tot / 1e6, "gpu_launches": 0}
    print(json.dumps(line), file=JSON_OUT, flush=True)
    return 0


# ------------------------------------------------------------------------------------------------ per-shape extras
def _max_over_ranks(torch, dist, world, values):
    t = torch.tensor(values, dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t]


def _sum_over_ranks(torch, dist, world, values):
    t = torch.tensor(values, dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return [float(v) for v in t]


def extras(torch, dist, rank, world, local, fused_ok, peak, reps=3):
    """Every BASELINE shape at this GPU count (north_star: 'throughput on synthetic scenes of each named shape is reported
    at 1, 2, 4 and 8 GPUs'), device-timed, max over ranks:
      C3          the headline frame back to back (no flush): tile-sharded (BASELINE config 3) as fused stripes (path-kernel
                  stores over NVLink) and as contiguous bands + one NCCL gather; sample-sharded (fused reduce-scatter / NCCL)
      C4          chandelier 1920x1080 64 spp, sample-range sharded (fused reduce-scatter; NCCL reduce beside it)
      C5          65,536 envs env-sharded (no collective): steady-state env-steps/s through rt_env_step_auto graph replay,
                  and each shard checked against the same rows of the unsharded batch
      C1, C2      Algorithm-A frames are sub-millisecond: frame-parallel (each rank renders its own frames of a sequence)"""
    import ray_tracer_v1_b200 as rtb
    from ray_tracer_v1_b200 import _native as nat, scenes
    from ray_tracer_v1_b200.distributed import ShardedPathRenderer
    from ray_tracer_v1_b200.ray_tracer_env import BatchedRayTracerEnv
    out = {}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        fn(); fn()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        barrier()
        return _max_over_ranks(torch, dist, world, [a.elapsed_time(b) / n])[0]

    def path_leg(spec, spp, depth, thr, modes):
        fs = rtb.flatten_scene(spec.spheres, background_colour=spec.background)
        r = ShardedPathRenderer(device=local)
        r.set_scene(fs)
        leg = {}
        q = None
        for mode, collective in modes:
            if collective == "fused" and not fused_ok:
                continue
            fn = (lambda m=mode: r.render_fused(spec.camera, W, H, spp, depth, thr, seed=5, fov=FOV, mode=m)) if collective == "fused" \
                else (lambda m=mode: r.render(spec.camera, W, H, spp, depth, thr, seed=5, fov=FOV, mode=m))
            ms = timed(fn, reps)
            r.stats.zero_()
            fn()
            barrier()
            q = _sum_over_ranks(torch, dist, world, [float(r.stats[4])])[0] if world > 1 else float(r.stats[4])
            leg[f"{mode}_{collective}"] = {"ms_per_frame": ms, "Mrays_per_s": q / ms / 1e3}
        n, nL = int(fs.radius.shape[0]), int(fs.l_index.shape[0])
        best = min(v["ms_per_frame"] for v in leg.values())
        leg["roofline_frac"] = q * flop_per_query(n, nL) / world / (best * 1e-3) / 1e12 / peak
        r.close()
        return leg

    # ---- C3: the headline frame, tile-sharded
    modes = [("tiles", "fused"), ("tiles", "nccl"), ("samples", "fused"), ("samples", "nccl")] if world > 1 else [("tiles", "nccl")]
    out["C3_complex_1920x1080_spp64"] = path_leg(scenes.build_complex(), SPP, DEPTH, THRESHOLD, modes)
    # ---- C4: chandelier, sample-range sharded
    modes = [("samples", "fused"), ("samples", "nccl")] if world > 1 else [("samples", "nccl")]
    out["C4_chandelier_1920x1080_spp64_samples"] = path_leg(scenes.build_chandelier(), 64, 8, 0.0, modes)

    # ---- C5: env-sharded rollouts
    for flavour in ("fb", "rl"):
        if flavour == "fb":
            spec = scenes.build_balls_in_space(as_rendered=False)
            kw = dict(image_width=800, image_height=600, camera_position=(0.0, 0.0, 1.0), fov=90, max_bounces=5, flavour="fb")
        else:
            spec = scenes.build_optimized_env_scene()
            kw = dict(image_width=320, image_height=240, camera_position=(0.0, 0.0, 0.0), fov=80, max_bounces=6, flavour="rl")
        fs = rtb.flatten_scene(spec.spheres, spec.global_lights, spec.point_lights, spec.background)
        B = 65536
        env = BatchedRayTracerEnv.shard(fs, B, rank=rank, world=world, device=local, seed=3, **kw)
        b0 = env.env_offset
        lo = torch.as_tensor(env.action_space.low, device="cuda")
        hi = torch.as_tensor(env.action_space.high, device="cuda")
        g = torch.Generator(device="cuda").manual_seed(7)
        acts = lo + (hi - lo) * torch.rand((8, B, 2), device="cuda", generator=g)         # the same actions on every rank
        mine = acts[:, b0:b0 + env.n_envs].contiguous()
        env.reset(seed=3)
        # shard == the same rows of the unsharded batch (device-drawn pixels are keyed by the global env index)
        whole = BatchedRayTracerEnv(fs, B, device=local, seed=3, **kw)
        whole.reset(seed=3)
        same = bool(torch.equal(whole.obs[b0:b0 + env.n_envs], env.obs))
        for t in range(kw["max_bounces"] + 2):
            ow, rw_, _, _, _ = whole.step_auto(acts[t % 8])
            os_, rs_, _, _, _ = env.step_auto(mine[t % 8])
            same = same and bool(torch.equal(ow[b0:b0 + env.n_envs], os_)) and bool(torch.equal(rw_[b0:b0 + env.n_envs], rs_))
        whole.close()
        # steady state: actions written in place, the step replayed from a CUDA graph (one launch, finished episodes restart in it)
        steps = 200
        k = [0]

        def one():
            env.actions.copy_(mine[k[0] % 8]); k[0] += 1
            env.step_auto(None, graph=True)
        for _ in range(10):
            one()
        barrier()
        env.stats.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            one()
        b.record()
        barrier()
        ms = _max_over_ranks(torch, dist, world, [a.elapsed_time(b)])[0]
        q = _sum_over_ranks(torch, dist, world, [float(env.stats[4])])[0]
        ok = _sum_over_ranks(torch, dist, world, [1.0 if same else 0.0])[0] == world
        out[f"C5_env_{flavour}_65536_env_sharded"] = {
            "envs_per_rank": env.n_envs, "us_per_step": 1e3 * ms / steps, "env_steps_per_s": B * steps / (ms * 1e-3),
            "Mrays_per_s": q / ms / 1e3, "launches_per_step": 2, "shards_equal_unsharded_rows": bool(ok),
            "note": "one action copy + one graph-replayed rt_env_step_auto launch per step; no collective"}
        env.close()

    # ---- C1 / C2: Algorithm A, frame-parallel
    def whitted_leg(spec, Wd, Hd, spp, depth, grid):
        fs = rtb.flatten_scene(spec.spheres, spec.global_lights, spec.point_lights, background_colour=spec.background)
        sc = nat.DeviceScene(fs, local)
        X, Y = grid
        accum = torch.zeros((Hd, Wd, 4), dtype=torch.float32, device="cuda")
        image = torch.zeros((Hd, Wd, 3), dtype=torch.float32, device="cuda")
        stats = torch.zeros(8, dtype=torch.int64, device="cuda")
        params = [sc.whitted_params(spec.camera, X, Y, spp=spp, max_bounces=depth, miss=[spec.miss.r, spec.miss.g, spec.miss.b],
                                    seed=rank * 1000 + f) for f in range(4)]
        k = [0]

        def frame():
            sc.render_whitted(params[k[0] % 4], accum, nat.F32, stats=stats); k[0] += 1
            sc.resolve(accum, Wd, Hd, spp, image, nat.F32)
        ms = timed(frame, 20)
        stats.zero_()
        frame()
        torch.cuda.synchronize()
        q = float(stats[4])
        qs = _sum_over_ranks(torch, dist, world, [q])[0]
        sc.close()
        return {"ms_per_frame_per_rank": ms, "frames_per_s": world * 1e3 / ms, "Mrays_per_s": qs / ms / 1e3,
                "sharding": "frame-parallel (independent frames per rank, no collective)"}

    balls = scenes.build_balls_in_space()
    out["C1_balls_320x240_spp1"] = whitted_leg(balls, 320, 240, 1, 1, scenes.custom_scene_grid(320, 240))
    for nm, spec in (("marbles4", scenes.build_marbles4()), ("planets2", scenes.build_planets2())):
        kk = 640 * spec.ray_step
        out[f"C2_{nm}_1280x720_spp16"] = whitted_leg(spec, 1280, 720, 16, 4, (np.linspace(-kk * 16 / 9, kk * 16 / 9, 1280),
                                                                                np.linspace(kk, -kk, 720)))
    return out


# ------------------------------------------------------------------------------------------------ own arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="auto", choices=["auto", "tiles", "samples"],
                    help="auto = tiles: at N=1 one band is the frame; at N>1 every rank renders interleaved 8-row stripes "
                         "(BASELINE config 3 is tile-sharded); the sample-range split is timed beside it under extra")
    ap.add_argument("--collective", default="fused", choices=["fused", "nccl", "chain"],
                    help="N>1: fused = ONE path-kernel launch per rank and frame, its stores/reductions and the epoch protocol "
                         "over NVLink peer memory; chain = the round-1 launch chain around the kernel; nccl = gather/reduce")
    ap.add_argument("--spp", type=int, default=SPP)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the per-shape table and the sustained run")
    ap.add_argument("--flush-mib", type=int, default=256, help="size of the L2 flush between timed steps (diagnostic; 0 = none)")
    ap.add_argument("--debug-ranks", action="store_true", help="every rank prints its own per-step times to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's frame and counters to DIR/image.npy and DIR/stats.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the CUDA arm only")
        return run_reference_arm(args)
    args.warmup = max(args.warmup, 3)
    if args.mode == "auto":
        args.mode = "tiles"          # BASELINE config 3: "tile-sharded at 2/4/8 GPUs" (the sample split is timed under extra)

    import torch
    import torch.distributed as dist
    import ray_tracer_v1_b200 as rtb
    from ray_tracer_v1_b200 import _native as nat
    from ray_tracer_v1_b200.distributed import ShardedPathRenderer, row_bands, sample_ranges

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    nat.lib()      # fail loudly if the CUDA extension is missing

    spec, fs = complex_scene()
    spp = args.spp
    r = ShardedPathRenderer(device=local)
    r.set_scene(fs)
    cam = spec.camera
    flush = torch.empty(max(args.flush_mib, 1) << 20, dtype=torch.uint8, device="cuda")     # default 256 MiB > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    fused = world > 1 and args.collective in ("fused", "chain")
    in_kernel = args.collective == "fused"
    fused_note = None
    if fused:
        # peer mappings are set up collectively; if any rank cannot (no IPC / no peer access) every rank raises and
        # the whole job uses the NCCL collective instead
        try:
            r._ensure_fabric(W, H)
        except Exception as e:      # noqa: BLE001
            fused, fused_note = False, f"fused collective unavailable, NCCL used: {e}"
            print(fused_note, file=sys.stderr, flush=True)

    def step(i, **kw):
        if fused:
            return r.render_fused(cam, W, H, spp, DEPTH, THRESHOLD, seed=i, fov=FOV, mode=args.mode, in_kernel=in_kernel, **kw)
        return r.render(cam, W, H, spp, DEPTH, THRESHOLD, seed=i, fov=FOV, mode=args.mode, **kw)

    # FP32 roofline denominator, measured here, with the SM clock it ran at
    peak_clock = ClockSampler(local)
    peak_clock.start()
    fp32_peak, _ = nat.measure_fp32_peak(local, 25)
    peak_clock = peak_clock.stop()
    counters = torch.zeros(8, dtype=torch.int64, device="cuda")
    launches = 0

    def one_step(i, ev_i, kev_i):
        """One step of the benchmark: [L2 flush, untimed] [event] the frame [event] [counters].  The warm-up steps run this
        very function, so nothing in the timed region is a first use (the first `counters += r.stats` alone loads a
        torch kernel module: 15 ms of idle GPU after which the next two frames of every rank ran 3-5 % slow).
        -> (image, stats): what the renderer hands its caller (the [H,W,3] float32 frame on rank 0, None elsewhere)."""
        nonlocal launches, counters
        # L2 flush between the timed steps (untimed: outside the step's event pair).  The K steps are bracketed by a
        # barrier + synchronize on both sides, not individually: inside, the frame protocol itself keeps the ranks together
        if args.flush_mib:
            flush.zero_()
        ev_i[0].record()
        # the step, with the dominant kernel bracketed separately for the roofline
        image = None
        if fused:
            image, _ = r.render_fused(cam, W, H, spp, DEPTH, THRESHOLD, seed=i, fov=FOV, mode=args.mode, kernel_events=kev_i,
                                      in_kernel=in_kernel)
            launches += r.launches
        else:
            r._ensure(W, H)
            rows = row_bands(H, world)[rank] if args.mode == "tiles" else (0, H)
            smp = sample_ranges(spp, world)[rank] if args.mode == "samples" else (0, spp)
            r.stats.zero_()
            p = r.scene.path_params(cam, W, H, spp, DEPTH, THRESHOLD, seed=i, fov=FOV, rows=rows, samples=smp)
            kev_i[0].record()
            r.scene.render_path(p, r.accum, nat.F32, stats=r.stats)
            kev_i[1].record()
            if args.mode == "tiles":
                r.scene.resolve(r.accum, W, H, spp, r.image, nat.F32, rows=rows)
                launches += 2
                if world > 1:
                    from ray_tracer_v1_b200.distributed import gather_row_bands
                    gather_row_bands(r.image, row_bands(H, world))
            else:
                from ray_tracer_v1_b200.distributed import reduce_sample_sums
                reduce_sample_sums(r.accum)
                launches += 1
                if rank == 0:
                    r.scene.resolve(r.accum, W, H, spp, r.image, nat.F32)
                    launches += 1
            if rank == 0:
                image = r.image
        ev_i[1].record()
        counters += r.stats
        return image, r.stats

    mk_ev = lambda: (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))      # noqa: E731
    for i in range(args.warmup):
        one_step(1000 + i, mk_ev(), mk_ev())
    barrier()

    # ---- device-timed steps (inputs resident in HBM); L2 flushed, untimed, between steps
    sampler = ClockSampler(local)
    sampler.start()
    ev = [mk_ev() for _ in range(args.steps)]
    kev = [mk_ev() for _ in range(args.steps)]
    counters.zero_()
    launches = 0
    barrier()
    for i in range(args.steps):
        last = one_step(i, ev[i], kev[i])
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)
    step_ms = [a.elapsed_time(b) for a, b in ev]
    kern_ms = [a.elapsed_time(b) for a, b in kev]
    if args.debug_ranks:
        gaps = [ev[i][1].elapsed_time(ev[i + 1][0]) for i in range(args.steps - 1)]
        print(f"[rank {rank}] step ms {' '.join(f'{v:.3f}' for v in step_ms)} | kernel ms {' '.join(f'{v:.3f}' for v in kern_ms)} "
              f"| gap (flush) ms {' '.join(f'{v:.3f}' for v in gaps)}", file=sys.stderr, flush=True)
    t = torch.tensor([sum(step_ms), sum(kern_ms)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(counters, op=dist.ReduceOp.SUM)
    total_ms, kernel_ms = float(t[0]), float(t[1])
    c = counters.cpu().numpy()
    rays_ref, queries, tests = int(c[0]), int(c[4]), int(c[5])
    value = queries / (total_ms * 1e-3) / 1e6

    # ---- end to end through the reference-facing API: host scene objects in, host image out, every step
    barrier()
    if world == 1:
        # the class a user of the reference calls: ComplexTraditionalRenderer.render(width, height, spp, max_bounces)
        # (FB/fb_vs_traditional_complex.py:391) -- every call re-flattens the 54 Python sphere objects, uploads the scene,
        # renders, resolves and brings the float32 image to host memory before it returns
        from ray_tracer_v1_b200.renderers import ComplexTraditionalRenderer
        rend = ComplexTraditionalRenderer(device=local, seed=0)
        rend.scene = spec.spheres
        rend.light_sources = [sph for sph in spec.spheres if sph.material.emitive]
        rend.small_lights = [sph for sph in rend.light_sources if sph.radius < 0.5]
        rend.camera_position = rtb.Vector(*cam)
        for i in range(2):
            rend.seed = 2000 + i
            rend.render(W, H, spp, DEPTH)
        torch.cuda.synchronize()
        e2e_queries, checksum = 0, 0.0
        t0 = time.perf_counter()
        for i in range(args.steps):
            rend.seed = i
            img = rend.render(W, H, spp, DEPTH)               # synchronous: the host image is complete on return
            checksum += float(img[0, 0, 0])
            e2e_queries += int(rend._ctx.host_stats.array[4])
        e2e_s = time.perf_counter() - t0
        e2e_value = e2e_queries / e2e_s / 1e6
        e2e_h2d, e2e_d2h = int(rend._ctx.h2d_bytes), int(rend._ctx.d2h_bytes)
        e2e_how = ("ComplexTraditionalRenderer.render(1920, 1080, 64, 5) per step (the reference's own class API): scene "
                   "re-flattened and uploaded, path kernel, resolve, D2H of the float32 image into pinned host memory, "
                   "synchronous return of the host image")
    else:
        e2e_q = torch.zeros(1, dtype=torch.int64, device="cuda")
        for i in range(2):
            r.set_scene(fs)
            step(2000 + i, to_host=True)
        barrier()
        t0 = time.perf_counter()
        pending, checksum = None, 0.0
        marks = []
        for i in range(args.steps):
            marks.append(time.perf_counter() - t0)
            # the reference-facing objects (54 Sphere / Material / Colour instances) are re-flattened EVERY frame, as the
            # drop-in classes do (scenes are mutable lists: SURVEY 8b) -- host work that overlaps the previous frame's render
            fs_i = rtb.flatten_scene(spec.spheres, background_colour=spec.background)
            r.set_scene(fs_i)                                     # H2D: the flattened scene, re-uploaded every frame
            img, st = step(i, to_host="async")                     # D2H: the float32 image into pinned host memory, on the
            e2e_q += st[4:5]                                       # copy stream while the next frame renders ...
            if pending is not None:
                checksum += float(pending.result()[0, 0, 0])       # ... and every frame IS read on the host, one frame later
            pending = img
        if pending is not None:
            checksum += float(pending.result()[0, 0, 0])
        marks.append(time.perf_counter() - t0)
        barrier()
        e2e_s = time.perf_counter() - t0
        if args.debug_ranks:
            print(f"[rank {rank}] e2e host marks (ms since start, one per step issue, then after the last read): "
                  f"{' '.join(f'{1e3 * v:.2f}' for v in marks)} | total {1e3 * e2e_s:.2f}", file=sys.stderr, flush=True)
        te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        dist.all_reduce(e2e_q, op=dist.ReduceOp.SUM)
        e2e_s = float(te[0])
        e2e_value = int(e2e_q[0]) / e2e_s / 1e6
        e2e_h2d, e2e_d2h = int(r.h2d_bytes), int(W * H * 3 * 4)
        e2e_how = ("ShardedPathRenderer (one process per GPU): scene re-flattened and re-uploaded on every rank, ONE fused "
                   "launch per rank, frame f copied to pinned host memory on rank 0's copy stream while frame f+1 renders; "
                   "every frame's host image is read inside the timed region")

    # ---- sustained: >= 5 s of frames back to back (no flush, no host sync), clocks sampled throughout
    sustained = None
    if world == 1 and not args.no_extra:
        r._ensure(W, H)
        p = r.scene.path_params(cam, W, H, spp, DEPTH, THRESHOLD, seed=77, fov=FOV)
        n_frames = max(10, int(SUSTAINED_SECONDS * 1e3 / (total_ms / args.steps)) + 1)
        sus = ClockSampler(local)
        torch.cuda.synchronize()
        sus.start()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n_frames):
            r.scene.render_path(p, r.accum, nat.F32, stats=None)
            r.scene.resolve(r.accum, W, H, spp, r.image, nat.F32)
        b.record()
        torch.cuda.synchronize()
        sc_ = sus.stop()
        sus_ms = a.elapsed_time(b)
        sustained = {"frames": n_frames, "seconds": sus_ms * 1e-3, "ms_per_frame": sus_ms / n_frames,
                     "Mrays_per_s": (queries / args.steps) * n_frames / (sus_ms * 1e-3) / 1e6, "clocks": sc_,
                     "note": "the same frame back to back (path kernel + resolve), no L2 flush, no host synchronisation"}

    extra = None
    if not args.no_extra:
        extra = extras(torch, dist, rank, world, local, fused or world == 1, fp32_peak)
        if world > 1 and fused:
            # the launch chain of round 1 beside the single launch, same frame (what the in-kernel protocol buys)
            def chain():
                r.render_fused(cam, W, H, spp, DEPTH, THRESHOLD, seed=9, fov=FOV, mode=args.mode, in_kernel=False)

            def single():
                r.render_fused(cam, W, H, spp, DEPTH, THRESHOLD, seed=9, fov=FOV, mode=args.mode, in_kernel=True)
            res = {}
            for name, fn in (("launch_chain_ms", chain), ("single_launch_ms", single)):
                fn(); fn()
                barrier()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(5):
                    fn()
                b.record()
                barrier()
                res[name] = _max_over_ranks(torch, dist, world, [a.elapsed_time(b) / 5])[0]
            # NVLink payload of the fused sample reduce: every pixel's (r, g, b, n) goes to its owner as one 16-byte red
            # NVLink payload per frame: samples = every rank's (r,g,b,n) of every pixel to its owner (one 16-byte red each)
            # + the resolved bands to rank 0; tiles = the resolved float32 stripes of ranks 1.. to rank 0
            res["nvlink_bytes_per_frame"] = int(W * H * 16 * (world - 1) + W * H * 12 * (world - 1) / world) if args.mode == "samples" \
                else int(W * H * 12 * (world - 1) / world)
            extra["C3_fused_protocol"] = res

    if rank == 0:
        n_sph, n_l = int(fs.radius.shape[0]), int(fs.l_index.shape[0])
        fpq = flop_per_query(n_sph, n_l)
        # roofline of the dominant kernel (path_kernel<float>): algorithmic FLOP per launch / its mean duration,
        # per GPU (this rank's launches; all ranks run the same kernel on equal shares)
        q_rank0 = queries / world
        achieved = q_rank0 * fpq / (kernel_ms * 1e-3) / 1e12
        # the same with the sphere tests the kernel actually executed (camera rays skip the spheres outside their warp
        # tile's cone; secondary rays test all N): never above `achieved`
        tests_per_query = tests / max(queries, 1)
        fpq_exec = 20.0 * tests_per_query + 15 + 25 * n_l + 70
        achieved_exec = q_rank0 * fpq_exec / (kernel_ms * 1e-3) / 1e12
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "width": W, "height": H, "spp": spp, "max_bounces": DEPTH,
                       "sharding": args.mode if world == 1 else f"{args.mode}, {args.collective if fused else 'nccl'} collective "
                       + ("(ONE path-kernel launch per rank and frame: epilogue stores/reductions over NVLink peer memory, epoch "
                          "protocol, band resolve and collection inside the launch)" if fused and in_kernel else
                          "(path-kernel epilogue over NVLink peer memory, flag / resolve launches around it)" if fused else "(NCCL)"),
                       "l2": (f"flushed between steps ({args.flush_mib} MiB memset, untimed)" if args.flush_mib else "NOT flushed (diagnostic run)") + "; inputs are a 3 KB scene",
                       "ray_definition": "one nearest-hit query over the scene (SURVEY 8d)"},
            "rays_ref_compatible_per_s": rays_ref / (total_ms * 1e-3) / 1e6,
            "rays_per_pixel_sample": rays_ref / (args.steps * W * H * spp),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": e2e_h2d,
                    "d2h_bytes_per_step": e2e_d2h, "ms_per_step": 1e3 * e2e_s / args.steps, "through": e2e_how},
            "gpu_launches": launches,
            "roofline": {"bound": "fp32", "kernel": "path_kernel<float, 3, true, false> (persistent warps, sphere/light pairs as uniform operands, "
                                                      "warp-vote skip of the sqrt/key half of a pair, camera-ray candidate lists, integer fold, lock-step)",
                         "achieved": achieved, "peak": fp32_peak,
                         "unit": "TFLOP/s", "frac": achieved / fp32_peak,
                         "peak_source": "rt_measure_fp32_peak (FFMA issue-rate micro-benchmark, best of 25 launches, measured in this "
                                        "run; MEASURED_PEAKS.json has no FP32 figure)",
                         "peak_clock_mhz": peak_clock.get("sm_mhz"), "peak_theoretical": None,
                         "flop_per_query": fpq, "queries_per_launch": q_rank0 / args.steps,
                         "sphere_tests_per_query_executed": tests_per_query, "flop_per_query_executed": fpq_exec,
                         "achieved_executed": achieved_exec, "frac_executed": achieved_exec / fp32_peak,
                         "kernel_ms": kernel_ms / args.steps,
                         # dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed ncu summary
                         # (the 33 MB framebuffer write mostly stays in the 126 MB L2 past the end of the kernel)
                         "traffic": ncu_dram_bytes(), "traffic_source": os.path.relpath(NCU_SUMMARY, ROOT),
                         "hbm_algorithmic_bytes_per_launch": W * H * 16 // world},
            "clocks": clocks,
        }
        try:
            props = nat.device_props(local)
            line["roofline"]["peak_theoretical"] = props["sm_count"] * 128 * 2 * (clocks.get("sm_max_mhz") or 0) * 1e6 / 1e12
        except Exception:      # noqa: BLE001
            pass
        if fused:
            line["config"]["fused_wait_timed_out"] = bool(r.fused_timed_out())
        if fused_note:
            line["config"]["note"] = fused_note
        if sustained:
            line["extra_sustained"] = sustained
        if extra:
            line["extra"] = extra
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(fs, spec)
        print(json.dumps(line), file=JSON_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
