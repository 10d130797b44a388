"""The variance-guided non-local-means filter of Algorithm B frames (rt_denoise, DESIGN §4.8c).

The oracle is ``nlm_reference`` below: the filter of include/rt_b200.h in NumPy float64.  The kernel computes in FP32,
so its output before the floor differs from the reference's by about 1e-3 levels; where the reference lies more than
1e-2 levels from an integer, the image must sit on exactly the reference's lattice point, and elsewhere within one level.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu

PRECISIONS = ["F32", "F64"]
EPS = 255.0 ** 2 * 1e-10
DEFAULTS = dict(radius=10, patch_radius=3, k=0.45)


@pytest.fixture(scope="module")
def nat(rt):
    from ray_tracer_v1_b200 import _native
    return _native


def nlm_reference(acc, var, radius=10, patch_radius=3, k=0.45):
    """The filter in float64 -> the filtered mean u_hat [H,W,3] in levels, before the floor.  The weighted sum is taken
    about the centre, u_p + sum w (u_q - u_p) / sum w, as the kernel takes it: a window of one colour gives u_p exactly."""
    r, f = radius, patch_radius
    n = acc[..., 3:4].astype(np.float64)
    u = (acc[..., :3].astype(np.float64) / n).astype(np.float32).astype(np.float64)
    V = var.astype(np.float64)
    H, W = u.shape[:2]

    def at(a, ys, xs):                  # reads clamped into the frame
        return a[np.clip(ys, 0, H - 1)][:, np.clip(xs, 0, W - 1)]

    ye, xe = np.arange(-f, H + f), np.arange(-f, W + f)      # every p + t of the frame's patches
    up, vp = at(u, ye, xe), at(V, ye, xe)
    P = 2 * f + 1
    sw, su = np.zeros((H, W, 1)), np.zeros((H, W, 3))
    for oy in range(-r, r + 1):
        for ox in range(-r, r + 1):
            uq, vq = at(u, ye + oy, xe + ox), at(V, ye + oy, xe + ox)
            d = (((up - uq) ** 2 - (vp + np.minimum(vp, vq))) / (EPS + k * k * (vp + vq))).mean(axis=2)
            rows = sum(d[:, t:t + W] for t in range(P))
            D = sum(rows[t:t + H] for t in range(P)) / (P * P)
            w = np.exp(-np.maximum(0.0, D))[..., None]
            sw += w
            su += w * (at(u, np.arange(H) + oy, np.arange(W) + ox) - u)
    return u + su / sw


def lattice(values):
    """rt_resolve's image of per-channel values in levels: min(1, floor(v) / 255) as float32."""
    return np.minimum(1.0, np.floor(values) / 255.0).astype(np.float32)


def check_against_reference(img, u_hat, min_far=None):
    """min_far: the least number of values that must lie far from an integer (default: more than half of them)."""
    far = np.abs(u_hat - np.rint(u_hat)) > 1e-2
    assert (far.mean() > 0.5) if min_far is None else (far.sum() >= min_far), far.sum()
    assert np.array_equal(img[far], lattice(u_hat)[far])
    got = np.rint(img.astype(np.float64) * 255.0)
    assert np.abs(got - np.minimum(255.0, np.floor(u_hat))).max() <= 1


def _ft(nat, prec):
    return np.float64 if prec == nat.F64 else np.float32


def denoise(nat, sc, acc, var, prec, **params):
    """Host arrays in, the filtered image out (device buffers around one rt_denoise)."""
    H, W = acc.shape[:2]
    a, v = nat.DeviceBuffer.from_host(acc, _ft(nat, prec)), nat.DeviceBuffer.from_host(var, np.float32)
    img = nat.DeviceBuffer((H, W, 3), np.float32)
    sc.denoise(a, v, W, H, img, prec, **{**DEFAULTS, **params})
    return img.download()


def uniform(nat, sc, frame, spp, prec, seed):
    """The uniform moments frame -> (accum, variance, resolved image)."""
    cam, W, H, depth, thr = frame
    p = sc.path_params(cam, W, H, spp, depth, thr, seed=seed)
    acc, mom = nat.DeviceBuffer((H, W, 4), _ft(nat, prec)), nat.DeviceBuffer((H, W, 4), np.float64)
    var, img = nat.DeviceBuffer((H, W, 3), np.float32), nat.DeviceBuffer((H, W, 3), np.float32)
    sc.render_path(p, acc, prec, moments=mom)
    sc.resolve_variance(acc, mom, W, H, var, prec)
    sc.resolve(acc, W, H, spp, img, prec)
    return acc.download(), var.download(), img.download()


def golden_frames():
    z, fs = load_golden("path_complex_48x27")
    yield "complex", fs, (z["cam"], int(z["W"]), int(z["H"]), int(z["max_bounces"]), float(z["mirror_threshold"]))
    z, fs = load_golden("path_chandelier_48x27")
    yield "chandelier", fs, (z["cam"], 64, 36, int(z["max_bounces"]), float(z["mirror_threshold"]))


@pytest.mark.parametrize("precision", PRECISIONS)
def test_denoise_matches_reference(nat, precision):
    """The complex golden scene and a small chandelier frame, at the defaults and at (r, f) = (3, 1) and (15, 5)."""
    prec = getattr(nat, precision)
    for name, fs, frame in golden_frames():
        sc = nat.DeviceScene(fs)
        acc, var, _ = uniform(nat, sc, frame, 8, prec, seed=3)
        assert (var > 0).mean() > 0.1, name
        for r, f in ((10, 3), (3, 1), (15, 5)):
            img = denoise(nat, sc, acc, var, prec, radius=r, patch_radius=f)
            check_against_reference(img, nlm_reference(acc, var, r, f))
        sc.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_denoise_frame_smaller_than_the_window(nat, precision):
    """8 x 5 pixels under a 21 x 21 window: both pixels of every pair are read clamped."""
    prec = getattr(nat, precision)
    z, fs = load_golden("path_complex_48x27")
    sc = nat.DeviceScene(fs)
    acc, var, _ = uniform(nat, sc, (z["cam"], 8, 5, int(z["max_bounces"]), float(z["mirror_threshold"])), 16, prec, seed=4)
    for r, f in ((10, 3), (15, 5), (10, 0)):
        check_against_reference(denoise(nat, sc, acc, var, prec, radius=r, patch_radius=f), nlm_reference(acc, var, r, f))
    sc.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_denoise_identity(nat, precision):
    """r = 0 leaves every pixel its own mean on the resolve's lattice; a constant colour with zero variance comes back
    unchanged at any radius."""
    prec = getattr(nat, precision)
    z, fs = load_golden("path_complex_48x27")
    sc = nat.DeviceScene(fs)
    acc, var, img_resolve = uniform(nat, sc, (z["cam"], int(z["W"]), int(z["H"]), int(z["max_bounces"]),
                                              float(z["mirror_threshold"])), 8, prec, seed=6)
    S, n = acc[..., :3].astype(np.float64), acc[..., 3:4].astype(np.float64)
    u32 = (S / n).astype(np.float32).astype(np.float64)
    same_floor = np.floor(u32) == np.floor(S / n)
    for f in (0, 3, 5):
        img = denoise(nat, sc, acc, var, prec, radius=0, patch_radius=f)
        assert np.array_equal(img, lattice(u32))
        assert np.array_equal(img[same_floor], img_resolve[same_floor])
    H, W, spp = 23, 40, 4
    const = np.zeros((H, W, 4))
    const[...] = (17 * spp, 128 * spp, 300 * spp, spp)
    zero = np.zeros((H, W, 3), np.float32)
    for r, f in ((10, 3), (15, 5), (1, 0)):
        img = denoise(nat, sc, const, zero, prec, radius=r, patch_radius=f)
        assert np.array_equal(img, lattice(np.broadcast_to([17.0, 128.0, 300.0], (H, W, 3))))
    sc.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_denoise_adaptive_input(nat, precision):
    """An adaptive frame, whose pixels hold different sample counts, matches the reference taken with those counts."""
    prec = getattr(nat, precision)
    z, fs = load_golden("path_complex_48x27")
    sc = nat.DeviceScene(fs)
    W, H = int(z["W"]), int(z["H"])
    p = sc.path_params(z["cam"], W, H, 16, int(z["max_bounces"]), float(z["mirror_threshold"]), seed=8)
    acc, mom = nat.DeviceBuffer((H, W, 4), _ft(nat, prec)), nat.DeviceBuffer((H, W, 4), np.float64)
    lst, img = nat.DeviceBuffer(H * W + 1, np.uint32), nat.DeviceBuffer((H, W, 3), np.float32)
    var, cnt = nat.DeviceBuffer((H, W, 3), np.float32), nat.DeviceBuffer((H, W), np.int32)
    for tol in (4.0, 2.0, 8.0, 1.0, 16.0):
        sc.render_path_adaptive(p, 2, tol, acc, mom, lst, img, prec, var=var, counts=cnt)
        if len(np.unique(cnt.download())) >= 3:
            break
    counts = cnt.download()
    assert len(np.unique(counts)) >= 3, np.unique(counts)
    out = nat.DeviceBuffer((H, W, 3), np.float32)
    sc.denoise(acc, var, W, H, out, prec)
    a, v = acc.download(), var.download()
    assert np.array_equal(a[..., 3], counts.astype(a.dtype))
    check_against_reference(out.download(), nlm_reference(a, v))
    sc.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_denoise_deterministic(nat, precision):
    """Two calls on the same input give the same bits."""
    prec = getattr(nat, precision)
    z, fs = load_golden("path_complex_48x27")
    sc = nat.DeviceScene(fs)
    W, H = 320, 180
    acc, var, _ = uniform(nat, sc, (z["cam"], W, H, int(z["max_bounces"]), float(z["mirror_threshold"])), 8, prec, seed=9)
    a, v = nat.DeviceBuffer.from_host(acc, _ft(nat, prec)), nat.DeviceBuffer.from_host(var, np.float32)
    outs = []
    for _ in range(2):
        img = nat.DeviceBuffer((H, W, 3), np.float32, zero=False)
        sc.denoise(a, v, W, H, img, prec)
        outs.append(img.download())
    assert outs[0].tobytes() == outs[1].tobytes()
    sc.close()


def test_denoise_validation(nat):
    """Every rejection returns RT_ERR_INVALID and names the cause."""
    L = nat.lib()
    W, H = 16, 8
    frame = np.zeros((H, W, 4), np.float32)
    frame[..., 3] = 1                                               # one sample per pixel: valid input for the calls that run
    acc, var = nat.DeviceBuffer.from_host(frame), nat.DeviceBuffer((H, W, 3), np.float32)
    img = nat.DeviceBuffer((H, W, 3), np.float32)

    def call(prec=nat.F32, w=W, h=H, ptrs=None, params=True, **kw):
        d = nat.DenoiseParams()
        d.radius, d.patch_radius, d.k = kw.get("radius", 10), kw.get("patch_radius", 3), kw.get("k", 0.45)
        a, v, i = ptrs or (acc.ptr, var.ptr, img.ptr)
        rc = L.rt_denoise(0, prec, a, v, w, h, C.byref(d) if params else None, i, None)
        return rc, L.rt_last_error().decode()

    INVALID = 1
    assert call()[0] == 0
    nat.check(L.rt_stream_sync(0, None))
    for ptrs in ((None, var.ptr, img.ptr), (acc.ptr, None, img.ptr), (acc.ptr, var.ptr, None)):
        assert call(ptrs=ptrs) == (INVALID, "NULL argument")
    assert call(params=False) == (INVALID, "NULL argument")
    cases = [(dict(w=0), "W and H must be at least 1"), (dict(h=0), "W and H must be at least 1"),
             (dict(w=-3), "W and H must be at least 1"), (dict(prec=2), "unknown precision"),
             (dict(radius=-1), "radius must be in [0, 15]"), (dict(radius=16), "radius must be in [0, 15]"),
             (dict(patch_radius=-1), "patch_radius must be in [0, 5]"), (dict(patch_radius=6), "patch_radius must be in [0, 5]"),
             (dict(k=0.0), "k must be finite and > 0"), (dict(k=-1.0), "k must be finite and > 0"),
             (dict(k=float("nan")), "k must be finite and > 0"), (dict(k=float("inf")), "k must be finite and > 0")]
    for kw, msg in cases:
        assert call(**kw) == (INVALID, msg), kw
    for kw in (dict(radius=0, patch_radius=0), dict(radius=15, patch_radius=5), dict(k=1e-6)):    # the limits are accepted
        assert call(**kw)[0] == 0, kw
    nat.check(L.rt_stream_sync(0, None))


def _renderer(rt, spec, seed):
    r = rt.ComplexTraditionalRenderer(precision="f32", seed=seed)
    r.scene = spec.spheres
    r.light_sources = [s for s in spec.spheres if s.material.emitive]
    r.camera_position = rt.Vector(*spec.camera)
    r.reuse_output = False
    return r


def test_renderer_denoise(rt, nat):
    """denoise = True returns what render_path + resolve_variance + rt_denoise give, uniform and adaptive, with and
    without track_variance; denoise = False returns the resolved frame."""
    from ray_tracer_v1_b200 import scenes
    spec = scenes.build_complex()
    W, H, spp, seed = 160, 90, 16, 5
    r = _renderer(rt, spec, seed)
    sc = nat.DeviceScene(r.flat_scene())
    p = sc.path_params(spec.camera, W, H, spp, 5, 0.9, seed=seed)
    acc, mom = nat.DeviceBuffer((H, W, 4), np.float32), nat.DeviceBuffer((H, W, 4), np.float64)
    var, img = nat.DeviceBuffer((H, W, 3), np.float32), nat.DeviceBuffer((H, W, 3), np.float32)
    sc.render_path(p, acc, nat.F32, moments=mom)
    sc.resolve(acc, W, H, spp, img, nat.F32)
    resolved = img.download()
    sc.resolve_variance(acc, mom, W, H, var, nat.F32)
    sc.denoise(acc, var, W, H, img, nat.F32)
    denoised, variance = img.download(), var.download()
    assert not np.array_equal(denoised, resolved)

    assert np.array_equal(r.render(W, H, spp, 5), resolved)
    r.denoise = True
    assert np.array_equal(r.render(W, H, spp, 5), denoised)
    r.track_variance = True
    assert np.array_equal(r.render(W, H, spp, 5), denoised) and np.array_equal(r.variance, variance)

    # adaptive: the frame's own per-pixel counts and variance go into the filter
    r.adaptive_tolerance = 2.0
    pa = sc.path_params(spec.camera, W, H, 64, 5, 0.9, seed=seed)
    lst, cnt = nat.DeviceBuffer(H * W + 1, np.uint32), nat.DeviceBuffer((H, W), np.int32)
    sc.render_path_adaptive(pa, r.adaptive_min_spp, 2.0, acc, mom, lst, img, nat.F32, var=var, counts=cnt)
    adaptive_resolved = img.download()
    sc.denoise(acc, var, W, H, img, nat.F32)
    adaptive_denoised = img.download()
    assert np.array_equal(r.render(W, H, 64, 5), adaptive_denoised)
    assert np.array_equal(r.sample_counts, cnt.download()) and np.array_equal(r.variance, var.download())
    assert len(np.unique(r.sample_counts)) > 1
    r.denoise = False
    assert np.array_equal(r.render(W, H, 64, 5), adaptive_resolved)
    sc.close()


def test_frame_context_denoise_needs_the_whole_frame(rt, nat):
    from ray_tracer_v1_b200 import scenes
    from ray_tracer_v1_b200.frames import FrameContext
    import ray_tracer_v1_b200 as rtb
    spec = scenes.build_complex()
    ctx = FrameContext()
    ctx.set_scene(rtb.flatten_scene(spec.spheres, background_colour=spec.background))
    for kw in (dict(rows=(0, 8)), dict(resolve=False)):
        with pytest.raises(ValueError, match="whole frame"):
            ctx.render_path(spec.camera, 64, 36, 4, 5, 0.9, denoise=True, **kw)
    image, stats = ctx.render_path(spec.camera, 64, 36, 4, 5, 0.9, rows=(0, 36), denoise=True)
    assert image.shape == (36, 64, 3) and int(stats[0]) > 0
    ctx.close()


def test_denoise_quality_1080p(rt, nat):
    """Complex scene, 1920 x 1080, seed 1; RMSE of the image in levels against the floored mean of a 4096-spp seed-1000
    frame (as tools/time_adaptive.py measures it):
    the denoised 16-spp frame beats the noisy 64-spp one, and the denoised 64-spp frame is at most 0.6x its RMSE."""
    from ray_tracer_v1_b200 import scenes
    import ray_tracer_v1_b200 as rtb
    spec = scenes.build_complex()
    sc = nat.DeviceScene(rtb.flatten_scene(spec.spheres, background_colour=spec.background))
    W, H = 1920, 1080
    acc, mom = nat.DeviceBuffer((H, W, 4), np.float32), nat.DeviceBuffer((H, W, 4), np.float64)
    var, img = nat.DeviceBuffer((H, W, 3), np.float32), nat.DeviceBuffer((H, W, 3), np.float32)

    def params(spp, seed):
        return sc.path_params(spec.camera, W, H, spp, spec.max_bounces, spec.mirror_threshold, seed=seed)

    sc.render_path(params(4096, 1000), acc, nat.F32)
    ref = np.floor(acc.download()[..., :3].astype(np.float64) / 4096)

    def rmse():
        return float(np.sqrt(np.mean((img.download().astype(np.float64) * 255.0 - ref) ** 2)))

    out = {}
    for spp in (16, 64):
        sc.render_path(params(spp, 1), acc, nat.F32, moments=mom)
        sc.resolve(acc, W, H, spp, img, nat.F32)
        out[f"noisy {spp}"] = rmse()
        sc.resolve_variance(acc, mom, W, H, var, nat.F32)
        sc.denoise(acc, var, W, H, img, nat.F32)
        out[f"denoised {spp}"] = rmse()
    print("RMSE (levels)", out)
    assert out["denoised 16"] < out["noisy 64"], out
    assert out["denoised 64"] <= 0.6 * out["noisy 64"], out
    sc.close()
