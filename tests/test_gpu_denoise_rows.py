"""The row-band filters (rt_denoise_rows, rt_denoise_features_rows; DESIGN §4.8e) and the denoised sharded frame.

- band = whole frame: rows [y0, y1) of the band filter equal those rows of rt_denoise / rt_denoise_features bit for
  bit, for every band of row_bands(H, N), N in {1, 2, 3, 8}, single rows, bands shorter than the halo, bands at both
  edges, bands not a multiple of the 16-row tile and the whole frame;
- window: with every row outside [y0 - h, y1 + h) poisoned (NaN sums at count 1, NaN variance and features) the band
  does not change, and no image row outside the band is written;
- ranks emulated on one GPU: each "rank" renders its share into its own buffers, band sums are formed as
  reduce_row_bands forms them, halo_plan is applied with device copies, and the assembled bands equal the unsharded
  DeviceScene.denoise frame bit for bit;
- ShardedPathRenderer.render(denoise=True) at world 1 equals FrameContext.render_path(denoise=True) bit for bit;
- every rejection is RT_ERR_INVALID with a message naming the cause.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import load_golden
from test_gpu_denoise_edges import synthetic, synthetic_features

pytestmark = pytest.mark.gpu

PAIRS = [(10, 3), (3, 1), (15, 5), (0, 0), (1, 0), (0, 2)]
SENTINEL = -5.0


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


def dev(x, dtype=None):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(x))
    return (t if dtype is None else t.to(dtype)).cuda()


def ft(nat, prec):
    import torch
    return torch.float64 if prec == nat.F64 else torch.float32


def golden_inputs(nat):
    """The complex golden frame at 8 spp: (name, accum [H,W,4] float64, var, features) on the host."""
    import torch
    z, fs = load_golden("path_complex_48x27")
    W, H = int(z["W"]), int(z["H"])
    sc = nat.DeviceScene(fs)
    p = sc.path_params(z["cam"], W, H, 8, int(z["max_bounces"]), float(z["mirror_threshold"]), seed=3)
    acc, mom = torch.zeros((H, W, 4), device="cuda"), torch.zeros((H, W, 4), dtype=torch.float64, device="cuda")
    var = torch.zeros((H, W, 3), device="cuda")
    feats = [torch.zeros(s, device="cuda") for s in ((H, W, 3), (H, W, 3), (H, W), (H, W, 3))]
    sc.render_path(p, acc, nat.F32, moments=mom)
    sc.resolve_variance(acc, mom, W, H, var, nat.F32)
    sc.render_features(p, *feats, precision=nat.F32)
    torch.cuda.synchronize()
    sc.close()
    return "complex", acc.double().cpu().numpy(), var.cpu().numpy(), [f.cpu().numpy() for f in feats]


def frames(nat):
    yield golden_inputs(nat)
    for H, W in ((35, 47), (113, 200)):
        acc, var = synthetic(H, W, seed=H)
        yield f"synthetic {W}x{H}", acc, var, synthetic_features(H, W, seed=H)


def bands_of(H, h):
    """Every band the tests filter: row_bands(H, N) for N in {1, 2, 3, 8}, single rows at the edges and the middle,
    bands shorter than the halo, bands touching either edge, bands not a multiple of 16 rows, and the whole frame."""
    from ray_tracer_v1_b200.distributed import row_bands
    out = {b for n in (1, 2, 3, 8) for b in row_bands(H, n) if b[1] > b[0]}
    out |= {(0, 1), (H - 1, H), (H // 2, H // 2 + 1), (0, H)}
    short = max(1, min(h - 1, H // 3)) if h > 1 else 1
    out |= {(0, short), (H - short, H), (H // 3, H // 3 + short)}
    out |= {(1, min(H, 18)), (max(0, H - 17), H - 1), (5, min(H, 22))}
    return sorted(b for b in out if 0 <= b[0] < b[1] <= H)


class Filter:
    """Device inputs of one frame and one filter; full() and band() run the whole-frame and the band kernel."""

    def __init__(self, nat, sc, acc, var, feats, prec, features, r, f):
        import torch
        self.nat, self.sc, self.prec, self.r, self.f = nat, sc, prec, r, f
        self.H, self.W = acc.shape[:2]
        self.host = (acc, var, feats)
        self.acc, self.var = dev(acc, ft(nat, prec)), dev(var)
        self.feats = [dev(x) for x in feats] if features else None
        self.features = features
        self.halo = nat.denoise_halo(r, f, features)
        self.torch = torch

    def _run(self, acc, var, feats, rows):
        img = self.torch.full((self.H, self.W, 3), SENTINEL, device="cuda")
        self.sc.denoise(acc, var, self.W, self.H, img, self.prec, radius=self.r, patch_radius=self.f, features=feats,
                        rows=rows)
        return img.cpu().numpy()

    def full(self):
        return self._run(self.acc, self.var, self.feats, None)

    def band(self, rows):
        return self._run(self.acc, self.var, self.feats, rows)

    def band_poisoned(self, rows):
        """The band with every input row outside its window replaced by NaN (sums; count 1) and NaN variance and
        features."""
        acc, var, feats = np.array(self.host[0], copy=True), np.array(self.host[1], copy=True), None
        y0, y1 = rows
        lo, hi = max(0, y0 - self.halo), min(self.H, y1 + self.halo)
        out = np.ones(self.H, bool)
        out[lo:hi] = False
        acc[out, :, :3], acc[out, :, 3], var[out] = np.nan, 1, np.nan
        if self.features:
            feats = []
            for x in self.host[2]:
                x = np.array(x, copy=True)
                x[out] = np.nan
                feats.append(dev(x))
        return self._run(dev(acc, ft(self.nat, self.prec)), dev(var), feats, rows)


def check_band(img, ref, rows, what):
    y0, y1 = rows
    assert np.array_equal(img[y0:y1], ref[y0:y1]), (what, rows)
    assert (img[:y0] == SENTINEL).all() and (img[y1:] == SENTINEL).all(), (what, rows, "a row outside the band was written")


@pytest.mark.parametrize("features", [False, True], ids=["colour", "features"])
@pytest.mark.parametrize("precision", ["F32", "F64"])
def test_band_equals_whole_frame(nat, features, precision):
    """Rows [y0, y1) of the band filter equal the whole-frame filter's, for every band of bands_of and every (r, f)."""
    prec = getattr(nat, precision)
    sc = nat.DeviceScene(load_golden("path_complex_48x27")[1])
    n = 0
    for name, acc, var, feats in frames(nat):
        for r, f in PAIRS:
            flt = Filter(nat, sc, acc, var, feats, prec, features, r, f)
            ref = flt.full()
            assert not (ref == SENTINEL).any() and np.isfinite(ref).all()
            for rows in bands_of(flt.H, flt.halo):
                check_band(flt.band(rows), ref, rows, (name, r, f))
                n += 1
    assert n > 300
    sc.close()


@pytest.mark.parametrize("features", [False, True], ids=["colour", "features"])
@pytest.mark.parametrize("precision", ["F32", "F64"])
def test_band_reads_only_its_window(nat, features, precision):
    """With every row outside the band's window poisoned, the band is unchanged and no other image row is written."""
    prec = getattr(nat, precision)
    sc = nat.DeviceScene(load_golden("path_complex_48x27")[1])
    for name, acc, var, feats in frames(nat):
        for r, f in ((10, 3), (15, 5), (0, 0), (1, 0), (0, 2)):
            flt = Filter(nat, sc, acc, var, feats, prec, features, r, f)
            ref = flt.full()
            bands = bands_of(flt.H, flt.halo)
            for rows in bands if name.startswith("complex") else bands[::3]:
                check_band(flt.band_poisoned(rows), ref, rows, (name, r, f))
    sc.close()


# ------------------------------------------------------------------ ranks emulated on one GPU
def emulate(nat, sc, spec, W, H, spp, world, mode, prec, features, params, seed=2):
    """Each "rank" renders its share into its own full-frame buffers (rows outside what it computed hold NaN), forms
    its band sums as reduce_row_bands does, resolves its band's variance, receives its halo by halo_plan with device
    copies, renders its window's features and filters its band into one shared image."""
    import torch
    from ray_tracer_v1_b200.distributed import row_bands, sample_ranges, halo_plan, halo_windows
    T = ft(nat, prec)
    bands = row_bands(H, world)
    h = nat.denoise_halo(params.get("radius", 10), params.get("patch_radius", 3), features)
    nan = float("nan")
    acc = [torch.full((H, W, 4), nan, dtype=T, device="cuda") for _ in range(world)]
    mom = [torch.full((H, W, 4), nan, dtype=torch.float64, device="cuda") for _ in range(world)]
    var = [torch.full((H, W, 3), nan, device="cuda") for _ in range(world)]
    for k in range(world):
        acc[k][..., 3] = 1
        rows, samples = (bands[k], (0, spp)) if mode == "tiles" else ((0, H), sample_ranges(spp, world)[k])
        if samples[0] == samples[1]:
            acc[k].zero_(), mom[k].zero_()
        p = sc.path_params(spec.camera, W, H, spp, spec.max_bounces, spec.mirror_threshold, seed=seed, rows=rows,
                           samples=samples)
        sc.render_path(p, acc[k], prec, moments=mom[k])
    if mode == "samples":
        total_a, total_m = sum(acc), sum(mom)
        for k, (a, b) in enumerate(bands):
            keep = torch.zeros(H, dtype=torch.bool, device="cuda")
            keep[a:b] = True
            acc[k] = torch.where(keep[:, None, None], total_a, torch.full_like(total_a, nan))
            acc[k][~keep, :, 3] = 1
            mom[k] = torch.where(keep[:, None, None], total_m, torch.full_like(total_m, nan))
    for k, (a, b) in enumerate(bands):
        if b > a:
            sc.resolve_variance(acc[k], mom[k], W, H, var[k], prec, rows=(a, b))
    for src, dst, a, b in halo_plan(H, world, h):
        acc[dst][a:b] = acc[src][a:b]
        var[dst][a:b] = var[src][a:b]
    image = torch.full((H, W, 3), SENTINEL, device="cuda")
    for k, (a, b) in enumerate(bands):
        lo, hi = halo_windows(H, world, h)[k]
        fb = None
        if features:
            fb = [torch.full(s, nan, device="cuda") for s in ((H, W, 3), (H, W, 3), (H, W), (H, W, 3))]
            if hi > lo:
                p = sc.path_params(spec.camera, W, H, spp, 1, 0.0, seed=seed, rows=(lo, hi), samples=(0, min(spp, 8)))
                sc.render_features(p, *fb, precision=prec)
        if b > a:
            sc.denoise(acc[k], var[k], W, H, image, prec, features=fb, rows=(a, b), **params)
    return image.cpu().numpy()


def unsharded(nat, sc, spec, W, H, spp, prec, features, params, seed=2):
    import torch
    acc = torch.zeros((H, W, 4), dtype=ft(nat, prec), device="cuda")
    mom = torch.zeros((H, W, 4), dtype=torch.float64, device="cuda")
    var, image = torch.zeros((H, W, 3), device="cuda"), torch.zeros((H, W, 3), device="cuda")
    p = sc.path_params(spec.camera, W, H, spp, spec.max_bounces, spec.mirror_threshold, seed=seed)
    sc.render_path(p, acc, prec, moments=mom)
    sc.resolve_variance(acc, mom, W, H, var, prec)
    fb = None
    if features:
        fb = [torch.zeros(s, device="cuda") for s in ((H, W, 3), (H, W, 3), (H, W), (H, W, 3))]
        pf = sc.path_params(spec.camera, W, H, spp, 1, 0.0, seed=seed, samples=(0, min(spp, 8)))
        sc.render_features(pf, *fb, precision=prec)
    sc.denoise(acc, var, W, H, image, prec, features=fb, **params)
    return image.cpu().numpy()


@pytest.mark.parametrize("world", [2, 3, 8])
def test_ranks_emulated_on_one_gpu(nat, complex_scene, world):
    """tiles and samples, H = 117 and H = 5 (empty bands at world 8), the defaults and (15, 5), FP32 and FP64, colour
    and features: the assembled bands equal the unsharded frame bit for bit."""
    spec, fs = complex_scene
    sc = nat.DeviceScene(fs)
    W, spp = 64, 6
    for H in (117, 5):
        for precision in ("F32", "F64"):
            prec = getattr(nat, precision)
            for features in (False, True):
                for params in ({}, {"radius": 15, "patch_radius": 5}):
                    ref = unsharded(nat, sc, spec, W, H, spp, prec, features, params)
                    assert np.isfinite(ref).all()
                    for mode in ("tiles", "samples"):
                        got = emulate(nat, sc, spec, W, H, spp, world, mode, prec, features, params)
                        assert np.array_equal(got, ref), (H, precision, features, params, mode)
    sc.close()


# ------------------------------------------------------------------ ShardedPathRenderer (one rank)
def _host(x):
    if hasattr(x, "result"):
        x = x.result()
    if hasattr(x, "cpu"):
        x = x.cpu().numpy()
    return np.array(x)


@pytest.mark.parametrize("to_host", [False, True, "async"])
def test_sharded_renderer_denoise(nat, complex_scene, to_host):
    """render(denoise=True[, features=True]) equals FrameContext.render_path(denoise=True[, features=True]) bit for
    bit in both modes, with and without the variance; a plain frame before and after keeps its image and launch
    count; features without denoise is a ValueError."""
    import torch
    from ray_tracer_v1_b200.distributed import ShardedPathRenderer
    from ray_tracer_v1_b200.frames import FrameContext
    from ray_tracer_v1_b200.renderers import render_path
    spec, fs = complex_scene
    W, H, spp = 160, 90, 6
    args = (spec.camera, W, H, spp, spec.max_bounces, spec.mirror_threshold)
    fc = FrameContext()
    fc.set_scene(fs)
    ref = {}
    for features in (False, True):
        img, _, var = fc.render_path(*args, seed=7, denoise=True, features=features, variance=True)
        ref[features] = (np.array(img), np.array(var))
    ref[(True, "params")] = np.array(fc.render_path(*args, seed=7, denoise=True, features=True)[0])
    fc.close()
    plain_ref = {s: render_path(fs, *args, seed=s)[0] for s in (6, 8)}
    assert not np.array_equal(ref[False][0], ref[True][0])
    r = ShardedPathRenderer()
    r.set_scene(fs)
    for mode in ("tiles", "samples"):
        out = r.render(*args, seed=6, mode=mode, to_host=to_host)
        before, launches = _host(out[0]), r.launches
        for features in (False, True):
            out = r.render(*args, seed=7, mode=mode, to_host=to_host, denoise=True, features=features)
            assert len(out) == 2
            assert np.array_equal(_host(out[0]), ref[features][0]), (mode, features)
            assert r.launches == 3 + features, (mode, features, r.launches)
            img, _, var = r.render(*args, seed=7, mode=mode, to_host=to_host, denoise=True, features=features,
                                   variance=True)
            img, var = _host(img), _host(var)
            assert np.array_equal(img, ref[features][0]) and np.array_equal(var, ref[features][1]), (mode, features)
        out = r.render(*args, seed=7, mode=mode, to_host=to_host, denoise=True, features=True,
                       denoise_params={"radius": 10, "patch_radius": 3, "k": 1.0, "k_f": 1.2, "tau": 1e-3})
        assert np.array_equal(_host(out[0]), ref[(True, "params")])
        out = r.render(*args, seed=7, mode=mode, to_host=to_host, denoise=True, denoise_params={"radius": 2})
        assert not np.array_equal(_host(out[0]), ref[False][0])
        out = r.render(*args, seed=8, mode=mode, to_host=to_host)
        torch.cuda.synchronize()
        assert len(out) == 2 and r.launches == launches, mode
        assert np.array_equal(before, plain_ref[6]) and np.array_equal(_host(out[0]), plain_ref[8]), mode
    with pytest.raises(ValueError, match="denoise"):
        r.render(*args, features=True)
    with pytest.raises(nat.NativeLibraryError, match="radius"):
        r.render(*args, denoise=True, denoise_params={"radius": 16})
    r.close()


# ------------------------------------------------------------------ rejections
def test_rows_rejections(nat):
    """NULL pointers, bad sizes and parameters as the whole-frame calls, and every band outside 0 <= y0 < y1 <= H, are
    RT_ERR_INVALID with a message naming the cause; a rejected call writes nothing."""
    import torch
    W, H = 20, 10
    L = nat.lib()
    acc, var = torch.ones((H, W, 4), device="cuda"), torch.zeros((H, W, 3), device="cuda")
    img = torch.full((H, W, 3), SENTINEL, device="cuda")
    fb = [torch.zeros(s, device="cuda") for s in ((H, W, 3), (H, W, 3), (H, W), (H, W, 3))]
    a, v, i = acc.data_ptr(), var.data_ptr(), img.data_ptr()
    fp = [x.data_ptr() for x in fb]
    INVALID = 1

    def colour(prec=nat.F32, w=W, h=H, y0=0, y1=H, r=10, f=3, k=0.45, ptrs=(a, v, i), params=True):
        d = nat.DenoiseParams()
        d.radius, d.patch_radius, d.k = r, f, k
        return L.rt_denoise_rows(0, prec, ptrs[0], ptrs[1], w, h, y0, y1, C.byref(d) if params else None, ptrs[2], None)

    def feature(prec=nat.F32, w=W, h=H, y0=0, y1=H, r=10, f=3, k=1.0, k_f=1.2, tau=1e-3, feats=fp, ptrs=(a, v, i)):
        d = nat.DenoiseFeaturesParams()
        d.radius, d.patch_radius, d.k, d.k_f, d.tau = r, f, k, k_f, tau
        return L.rt_denoise_features_rows(0, prec, ptrs[0], ptrs[1], *feats, w, h, y0, y1, C.byref(d), ptrs[2], None)

    def rejected(rc, msg):
        assert rc == INVALID and msg in L.rt_last_error().decode(), (rc, L.rt_last_error().decode(), msg)

    for call in (colour, feature):
        rejected(call(ptrs=(None, v, i)), "NULL argument")
        rejected(call(ptrs=(a, None, i)), "NULL argument")
        rejected(call(ptrs=(a, v, None)), "NULL argument")
        rejected(call(w=0), "W and H")
        rejected(call(h=0, y1=0), "W and H")
        rejected(call(prec=7), "unknown precision")
        rejected(call(r=16), "radius")
        rejected(call(r=-1), "radius")
        rejected(call(f=6), "patch_radius")
        rejected(call(k=0.0), "k must be")
        rejected(call(k=float("nan")), "k must be")
        for y0, y1 in ((-1, 5), (0, H + 1), (5, 5), (6, 5), (H, H), (H, H + 1)):
            rejected(call(y0=y0, y1=y1), "rows [y0, y1)")
    rejected(colour(params=False), "NULL argument")
    for k in range(4):
        feats = list(fp)
        feats[k] = None
        rejected(feature(feats=feats), "NULL feature buffer")
    rejected(feature(k_f=0.0), "k_f")
    rejected(feature(k_f=float("inf")), "k_f")
    rejected(feature(tau=-1.0), "tau")
    rejected(feature(tau=float("nan")), "tau")
    torch.cuda.synchronize()
    assert (img == SENTINEL).all(), "a rejected call launches nothing"
    assert colour(y0=3, y1=4) == 0 and feature(y0=9, y1=10) == 0
    torch.cuda.synchronize()
    out = img.cpu().numpy()
    assert (out[3:4] != SENTINEL).all() and (out[9:10] != SENTINEL).all()
    assert (out[:3] == SENTINEL).all() and (out[4:9] == SENTINEL).all()
