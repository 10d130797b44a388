"""Per-pixel variance through the fused multi-GPU sinks (rt_render_path_sink_moments, rt_resolve_clear_moments) and
through ShardedPathRenderer.

One GPU stands in for every rank (peers = self, as in test_gpu_parity.py): the sinks address the "peers'" buffers with
plain device pointers.  Every variance must equal, bit for bit, rt_render_path_moments + rt_resolve_variance of the
unsharded frame, and every image the same frame rendered without variance."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def nat(rt):
    from ray_tracer_v1_b200 import _native
    return _native


@pytest.fixture(scope="module")
def complex_scene(rt):
    import ray_tracer_v1_b200 as pkg
    from ray_tracer_v1_b200 import scenes
    spec = scenes.build_complex()
    return spec, pkg.flatten_scene(spec.spheres, background_colour=spec.background)


def zeros(shape, dtype):
    import torch
    return torch.zeros(shape, dtype=dtype, device="cuda")


def reference(nat, sc, p):
    """The unsharded frame: rt_render_path_moments + rt_resolve + rt_resolve_variance -> (image, var, accum, moments)."""
    import torch
    W, H, spp = p.W, p.H, p.s1 - p.s0
    acc, mom = zeros((H, W, 4), torch.float32), zeros((H, W, 4), torch.float64)
    img, var = zeros((H, W, 3), torch.float32), zeros((H, W, 3), torch.float32)
    sc.render_path(p, acc, nat.F32, moments=mom)
    sc.resolve(acc, W, H, spp, img, nat.F32)
    sc.resolve_variance(acc, mom, W, H, var, nat.F32)
    torch.cuda.synchronize()
    return img.cpu().numpy(), var.cpu().numpy(), acc.cpu().numpy(), mom.cpu().numpy()


def last_error(nat):
    return nat.load_symbols().rt_last_error().decode()


# ------------------------------------------------------------------ image sink (tile sharding)
@pytest.mark.parametrize("W,H,spp,col_split", [(200, 117, 6, 0), (192, 117, 6, 1), (200, 117, 1, 0), (192, 117, 1, 1)])
def test_image_sink_variance(nat, complex_scene, W, H, spp, col_split):
    """Three "ranks" render interleaved stripes (or, with col_split, column segments of every stripe) into one image
    and one variance image: the variance equals the unsharded one bit for bit, the image the plain sink's image."""
    import torch
    spec, fs = complex_scene
    sc = nat.DeviceScene(fs)
    p = sc.path_params(spec.camera, W, H, spp, 5, 0.9, seed=4)
    ref_img, ref_var, _, _ = reference(nat, sc, p)
    img, var, plain = zeros((H, W, 3), torch.float32), zeros((H, W, 3), torch.float32), zeros((H, W, 3), torch.float32)
    stats, stats_plain = zeros(8, torch.int64), zeros(8, torch.int64)
    for r in range(3):
        sink = nat.PathSink()
        sink.mode, sink.tile_first, sink.tile_step, sink.col_split = nat.SINK_IMAGE, r, 3, col_split
        ms = nat.PathMomentsSink()
        ms.var = var.data_ptr()
        sink.image = img.data_ptr()
        sc.render_path_sink(p, sink, stats=stats, moments_sink=ms)
        sink.image = plain.data_ptr()
        sc.render_path_sink(p, sink, stats=stats_plain)
    torch.cuda.synchronize()
    assert np.array_equal(var.cpu().numpy(), ref_var)
    assert np.array_equal(img.cpu().numpy(), plain.cpu().numpy()) and np.array_equal(img.cpu().numpy(), ref_img)
    assert torch.equal(stats, stats_plain)
    if spp == 1:
        assert not var.any()
    else:
        assert float(var.max()) > 0
    sc.close()


# ------------------------------------------------------------------ scatter-add sink (sample sharding)
@pytest.mark.parametrize("ranges", [((0, 4), (4, 6)), ((0, 4), (4, 4), (4, 6))])
def test_scatter_add_sink_moments(nat, complex_scene, ranges):
    """The "ranks" add their sample ranges (one of them empty) into the owners' sums and moments: the moments equal the
    unsharded ones bit for bit, rt_resolve_clear_moments yields the reference image and variance and leaves both
    buffers zero."""
    import torch
    from ray_tracer_v1_b200.distributed import row_bands
    spec, fs = complex_scene
    sc = nat.DeviceScene(fs)
    W, H, spp, world = 200, 117, 6, len(ranges)
    ref_img, ref_var, ref_acc, ref_mom = reference(nat, sc, sc.path_params(spec.camera, W, H, spp, 5, 0.9, seed=4))
    acc, mom = zeros((H, W, 4), torch.float32), zeros((H, W, 4), torch.float64)
    bands = row_bands(H, world)
    for s0, s1 in ranges:
        q = sc.path_params(spec.camera, W, H, spp, 5, 0.9, seed=4, samples=(s0, s1))
        sink, ms = nat.PathSink(), nat.PathMomentsSink()
        sink.mode, sink.world = nat.SINK_SCATTER_ADD, world
        for k in range(world):
            sink.accum[k], ms.moments[k] = acc.data_ptr(), mom.data_ptr()
            sink.band_y[k] = bands[k][0]
        sink.band_y[world] = H
        sc.render_path_sink(q, sink, moments_sink=ms)
    torch.cuda.synchronize()
    assert np.array_equal(acc.cpu().numpy(), ref_acc) and np.array_equal(mom.cpu().numpy(), ref_mom)
    img, var = zeros((H, W, 3), torch.float32), zeros((H, W, 3), torch.float32)
    for y0, y1 in bands:
        nat.check(nat.lib().rt_resolve_clear_moments(0, acc.data_ptr(), mom.data_ptr(), W, H, y0, y1, spp, img.data_ptr(),
                                                     var.data_ptr(), 1, None))
    torch.cuda.synchronize()
    assert np.array_equal(img.cpu().numpy(), ref_img) and np.array_equal(var.cpu().numpy(), ref_var)
    assert not acc.any() and not mom.any()
    sc.close()


# ------------------------------------------------------------------ single-launch protocol (rt_path_sink.sync)
@pytest.mark.parametrize("mode", ["tiles", "samples"])
def test_single_launch_protocol_variance(nat, complex_scene, mode):
    """The in-kernel frame protocol of test_single_launch_frame_protocol (3 co-resident "ranks", rank 0 launched last,
    four frames through both buffer parities) with variance on frames 1, 2 and 4 and off on frame 3: every frame's
    image and variance equal the unsharded ones, no flag wait times out, and the moments bands are zero after each
    variance frame."""
    import torch
    from ray_tracer_v1_b200.distributed import row_bands, sample_ranges
    spec, fs = complex_scene
    sc = nat.DeviceScene(fs)
    W, H, spp, world = 384, 216, 7, 3
    dev = torch.device("cuda", 0)
    images = [zeros((H, W, 3), torch.float32) for _ in (0, 1)]
    vars_ = [zeros((H, W, 3), torch.float32) for _ in (0, 1)]
    accum = [[zeros((H, W, 4), torch.float32) for _ in range(world)] for _ in (0, 1)]
    moments = [[zeros((H, W, 4), torch.float64) for _ in range(world)] for _ in (0, 1)]
    flags = [zeros(nat.FLAG_WORDS, torch.int32) for _ in range(world)]
    timed_out = zeros(1, torch.int32)
    streams = [torch.cuda.Stream(device=dev) for _ in range(world)]
    bands = row_bands(H, world)
    torch.cuda.synchronize()
    for e in range(1, 5):
        buf, variance = e & 1, e != 3
        vars_[buf].fill_(-1.0)
        p = sc.path_params(spec.camera, W, H, spp, 5, 0.9, seed=100 + e)
        ref_img, ref_var, _, _ = reference(nat, sc, p)
        for rank in reversed(range(world)):
            p = sc.path_params(spec.camera, W, H, spp, 5, 0.9, seed=100 + e)
            sink = nat.PathSink()
            sink.world, sink.rank, sink.sync, sink.epoch, sink.spp_total = world, rank, 1, e, spp
            sink.go_epoch = e - 1 if rank == 0 else 0
            sink.image = images[buf].data_ptr()
            sink.timed_out, sink.timeout_ms, sink.max_ctas = timed_out.data_ptr(), 4000, 148
            for k in range(world):
                sink.flags[k] = flags[k].data_ptr()
            ms = nat.PathMomentsSink()
            ms.var = vars_[buf].data_ptr()
            if mode == "tiles":
                sink.mode, sink.tile_first, sink.tile_step = nat.SINK_IMAGE, rank, world
            else:
                sink.mode = nat.SINK_SCATTER_ADD
                p.s0, p.s1 = sample_ranges(spp, world)[rank]
                for k in range(world):
                    sink.accum[k] = accum[buf][k].data_ptr()
                    ms.moments[k] = moments[buf][k].data_ptr()
                    sink.band_y[k] = bands[k][0]
                sink.band_y[world] = H
            sc.render_path_sink(p, sink, stream=streams[rank].cuda_stream, moments_sink=ms if variance else None)
        streams[0].synchronize()
        assert int(timed_out.item()) == 0, "a flag wait timed out: the launches did not run concurrently"
        assert np.array_equal(images[buf].cpu().numpy(), ref_img), f"frame {e}"
        torch.cuda.synchronize()
        if variance:
            assert np.array_equal(vars_[buf].cpu().numpy(), ref_var), f"frame {e}"
        else:
            assert bool((vars_[buf] == -1.0).all()), "a frame without variance leaves the variance image alone"
        if mode == "samples":
            assert not any(bool(a.any()) for a in accum[buf])
            assert not any(bool(m.any()) for m in moments[buf]), "moments bands are cleared for the frame after next"
    assert [int(f[32]) for f in flags] == [3] * world
    sc.close()


# ------------------------------------------------------------------ ShardedPathRenderer (one rank)
def _host(x):
    """A returned image / variance as numpy, whatever to_host made of it."""
    if hasattr(x, "result"):
        x = x.result()
    if hasattr(x, "cpu"):
        x = x.cpu().numpy()
    return np.array(x)


@pytest.mark.parametrize("to_host", [False, True, "async"])
def test_sharded_renderer_variance(nat, complex_scene, to_host):
    """render and render_fused (in-kernel protocol and launch chain), tiles and samples: the variance equals
    render_path(..., variance=True) bit for bit, the image the same call without variance; a variance frame between two
    plain frames leaves their images and launch counts unchanged."""
    import torch
    from ray_tracer_v1_b200.distributed import ShardedPathRenderer
    from ray_tracer_v1_b200.renderers import render_path
    spec, fs = complex_scene
    W, H, spp = 160, 90, 6
    args = (spec.camera, W, H, spp, spec.max_bounces, spec.mirror_threshold)
    ref_img, _, ref_var = render_path(fs, *args, seed=7, variance=True)
    plain_ref = {s: render_path(fs, *args, seed=s)[0] for s in (6, 8)}
    r = ShardedPathRenderer()
    r.set_scene(fs)
    calls = {"nccl": r.render, "fused": r.render_fused,
             "chain": lambda *a, **k: r.render_fused(*a, in_kernel=False, **k)}
    for name, fn in calls.items():
        for mode in ("tiles", "samples"):
            out = fn(*args, seed=6, mode=mode, to_host=to_host)
            assert len(out) == 2
            before, launches = _host(out[0]), r.launches
            img, stats, var = fn(*args, seed=7, mode=mode, to_host=to_host, variance=True)
            img, var = _host(img), _host(var)
            torch.cuda.synchronize()
            assert np.array_equal(var, ref_var), (name, mode)
            assert np.array_equal(img, ref_img), (name, mode)
            out = fn(*args, seed=8, mode=mode, to_host=to_host)
            assert len(out) == 2 and r.launches == launches, (name, mode)
            assert np.array_equal(before, plain_ref[6]) and np.array_equal(_host(out[0]), plain_ref[8]), (name, mode)
    assert not r.fused_timed_out()
    r.close()


def test_sharded_renderer_variance_fp64(nat, complex_scene):
    """The NCCL path in FP64: the variance equals the FP64 render_path(..., variance=True) bit for bit."""
    from ray_tracer_v1_b200.distributed import ShardedPathRenderer
    from ray_tracer_v1_b200.renderers import render_path
    spec, fs = complex_scene
    W, H, spp = 96, 54, 5
    args = (spec.camera, W, H, spp, spec.max_bounces, spec.mirror_threshold)
    ref_img, _, ref_var = render_path(fs, *args, seed=9, precision="f64", variance=True)
    r = ShardedPathRenderer(precision="f64")
    r.set_scene(fs)
    for mode in ("tiles", "samples"):
        img, _, var = r.render(*args, seed=9, mode=mode, to_host=True, variance=True)
        assert np.array_equal(var, ref_var) and np.array_equal(img, ref_img), mode
        assert var.max() > 0
    r.close()


# ------------------------------------------------------------------ rejections
def test_moments_sink_rejections(nat, complex_scene):
    """Missing pointers and a bad band are RT_ERR_INVALID, and rt_last_error names the cause."""
    import torch
    spec, fs = complex_scene
    sc = nat.DeviceScene(fs)
    W, H, spp = 64, 32, 4
    L = nat.lib()
    p = sc.path_params(spec.camera, W, H, spp, 5, 0.9, seed=1)
    img, var = zeros((H, W, 3), torch.float32), zeros((H, W, 3), torch.float32)
    acc, mom = zeros((H, W, 4), torch.float32), zeros((H, W, 4), torch.float64)
    flags = [zeros(nat.FLAG_WORDS, torch.int32) for _ in range(2)]
    INVALID = 1

    def call(sink, ms):
        return L.rt_render_path_sink_moments(sc.handle, C.byref(p), C.byref(sink), C.byref(ms), None, None)

    sink = nat.PathSink()
    sink.mode, sink.tile_first, sink.tile_step, sink.image = nat.SINK_IMAGE, 0, 1, img.data_ptr()
    assert call(sink, nat.PathMomentsSink()) == INVALID and "variance image" in last_error(nat)
    assert L.rt_render_path_sink_moments(sc.handle, C.byref(p), C.byref(sink), None, None, None) == INVALID
    assert "NULL argument" in last_error(nat)
    sink = nat.PathSink()
    sink.mode, sink.world = nat.SINK_SCATTER_ADD, 2
    sink.accum[0] = sink.accum[1] = acc.data_ptr()
    sink.band_y[0], sink.band_y[1], sink.band_y[2] = 0, H // 2, H
    ms = nat.PathMomentsSink()
    ms.moments[0] = mom.data_ptr()
    assert call(sink, ms) == INVALID and "peer moments" in last_error(nat)
    ms.moments[1] = mom.data_ptr()
    sink.sync, sink.rank, sink.epoch, sink.spp_total, sink.image = 1, 0, 1, spp, img.data_ptr()
    sink.flags[0], sink.flags[1] = flags[0].data_ptr(), flags[1].data_ptr()
    assert call(sink, ms) == INVALID and "variance image" in last_error(nat)
    torch.cuda.synchronize()
    assert not img.any() and not var.any() and not acc.any() and not mom.any(), "a rejected call launches nothing"
    a, m, i, v = acc.data_ptr(), mom.data_ptr(), img.data_ptr(), var.data_ptr()
    assert L.rt_resolve_clear_moments(0, a, m, W, H, 0, H + 1, spp, i, v, 1, None) == INVALID
    assert "row band" in last_error(nat)
    assert L.rt_resolve_clear_moments(0, a, m, W, H, 9, 3, spp, i, v, 1, None) == INVALID
    assert "row band" in last_error(nat)
    assert L.rt_resolve_clear_moments(0, a, m, W, H, 0, H, 0, i, v, 1, None) == INVALID and "spp" in last_error(nat)
    assert L.rt_resolve_clear_moments(0, a, None, W, H, 0, H, spp, i, v, 1, None) == INVALID
    assert L.rt_resolve_clear_moments(0, a, m, W, H, 0, H, spp, i, None, 1, None) == INVALID
    assert "NULL argument" in last_error(nat)
    sc.close()
