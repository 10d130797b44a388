"""The row-band halo exchange of denoised sharded frames (ray-tracer-v1_b200/distributed.py, DESIGN §4.8e) on CPU.

``halo_plan`` is a pure function: every rank must receive each row of its window it does not own exactly once, from
the rank that owns it, also when the halo is deeper than a neighbour's band and when bands are empty.  Over ``gloo`` at
world 2 and 3, ``reduce_row_bands`` + ``exchange_halos`` + a NumPy stand-in stencil (the mean over a clamped window of
depth h) computed per band and gathered onto rank 0 must equal the stencil of the whole, unsharded frame."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT

CASES = [(1080, 8), (117, 8), (27, 2), (5, 8), (64, 3)]


@pytest.mark.parametrize("H,world", CASES)
@pytest.mark.parametrize("h", [0, 1, 13, 20])
def test_halo_plan_covers_every_window_once(H, world, h):
    from ray_tracer_v1_b200.distributed import halo_plan, halo_windows, row_bands
    bands, windows, plan = row_bands(H, world), halo_windows(H, world, h), halo_plan(H, world, h)
    for dst in range(world):
        y0, y1 = bands[dst]
        lo, hi = windows[dst]
        if y0 == y1:
            assert lo == hi
        else:
            assert (lo, hi) == (max(0, y0 - h), min(H, y1 + h))
        got = []
        for src, d, a, b in plan:
            if d != dst:
                continue
            assert src != dst and a < b
            assert bands[src][0] <= a and b <= bands[src][1], "rows are sent by their owner"
            got += range(a, b)
        want = [y for y in range(lo, hi) if not y0 <= y < y1]
        assert sorted(got) == want, (dst, sorted(got), want)
    if (H, world, h) == (117, 8, 20):       # bands of 14-15 rows: a 20-row halo takes rows from two ranks on each side
        assert len({src for src, d, _, _ in plan if d == 3}) == 4


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _stencil(x, h):
    """The mean over rows [y - h, y + h] clamped into the frame, for every row of x [H, W, C]."""
    H = x.shape[0]
    idx = np.clip(np.arange(H)[:, None] + np.arange(-h, h + 1)[None, :], 0, H - 1)
    return x[idx].mean(axis=1)


def _worker(rank, world, port, q):
    try:
        sys.path.insert(0, ROOT)
        os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
        dist.init_process_group("gloo", rank=rank, world_size=world)
        from ray_tracer_v1_b200.distributed import (row_bands, halo_plan, exchange_halos, reduce_row_bands,
                                                    gather_row_bands)
        results = []
        for H, h in ((27, 3), (27, 20), (5, 2), (64, 13), (2, 1)):
            W = 4
            rng = np.random.default_rng(H * 100 + h)
            parts = rng.integers(0, 255, (world, H, W, 4)).astype(np.float32)    # each rank's partial sums
            whole = parts.sum(axis=0)
            t = torch.from_numpy(parts[rank].copy())
            v = torch.from_numpy(rng.random((H, W, 3)).astype(np.float32))       # the same "variance" on every rank
            bands = row_bands(H, world)
            y0, y1 = bands[rank]
            reduce_row_bands(t, bands)
            mine = torch.zeros_like(v)
            mine[y0:y1] = v[y0:y1]                                               # this rank computed its band only
            exchange_halos([t, mine], halo_plan(H, world, h))
            out = torch.zeros((H, W, 7), dtype=torch.float64)
            if y1 > y0:
                lo, hi = max(0, y0 - h), min(H, y1 + h)
                window = np.concatenate([t.numpy(), mine.numpy()], axis=-1).astype(np.float64)
                win = np.full_like(window, np.nan)
                win[lo:hi] = window[lo:hi]                                       # rows outside the window are unknown
                idx = np.clip(np.arange(y0, y1)[:, None] + np.arange(-h, h + 1)[None, :], lo, hi - 1)
                out[y0:y1] = torch.from_numpy(win[idx].mean(axis=1))
            gather_row_bands(out, bands)
            if rank == 0:
                ref = _stencil(np.concatenate([whole, v.numpy()], axis=-1).astype(np.float64), h)
                results.append((H, h, bool(np.array_equal(out.numpy(), ref))))
        if rank == 0:
            q.put(results)
        dist.barrier()
        dist.destroy_process_group()
    except Exception as e:      # surface the failure in the parent
        q.put(("error", repr(e)))
        raise


@pytest.mark.parametrize("world", [2, 3])
def test_band_stencil_over_gloo_equals_the_whole_frame(world):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = q.get(timeout=240)
    for p in procs:
        p.join(timeout=120)
    assert isinstance(res, list) and all(ok for _, _, ok in res), res
    assert all(p.exitcode == 0 for p in procs)
