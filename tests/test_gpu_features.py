"""First-hit features of Algorithm B frames (rt_render_features) and the feature-guided non-local-means filter
(rt_denoise_features), DESIGN §4.8d.

The AOV oracle is ``aov_reference`` below: the camera rays of the frame from the oracle's Philox stream
(``orc.rng_pair``) and the ``generate_camera_ray`` formula, their nearest hit by Algorithm B's rule (the oracle's
``sphere_discriminant``: nearest by distance, ``trace_path`` in oracle/rt_oracle.c), in NumPy float64.  The filter oracle
is ``nlm_features_reference``: ``nlm_reference`` of test_gpu_denoise.py with the feature term, checked with the same
lattice criterion.
"""
import ctypes as C
import math

import numpy as np
import pytest

from conftest import gate, load_golden
from test_gpu_denoise import check_against_reference, lattice, nlm_reference

pytestmark = pytest.mark.gpu

PRECISIONS = ["F32", "F64"]
EPS = 255.0 ** 2 * 1e-10


@pytest.fixture(scope="module")
def nat(rt):
    from ray_tracer_v1_b200 import _native
    return _native


def _ft(nat, prec):
    return np.float64 if prec == nat.F64 else np.float32


# ------------------------------------------------------------------ AOV reference
def camera_rays(orc, cam, W, H, seed, y0, y1, s, fov=60.0):
    """Directions [y1-y0, W, 3] of sample s: path_camera_ray of the FP64 build (division by W, H; normalised twice)."""
    ys, xs = np.mgrid[y0:y1, 0:W]
    u = np.array([orc.rng_pair(seed, int(y) * W + int(x), s, 0) for y, x in zip(ys.ravel(), xs.ravel())])
    sx, sy = 0.5 + (u[:, 0] - 0.5), 0.5 + (u[:, 1] - 0.5)
    aspect = W / H
    half_h = math.tan((fov * (math.pi / 180.0)) / 2)                 # libm's tan, as the host computes it
    half_w = half_h * aspect
    scx = (2 * ((xs.ravel() + sx) / W) - 1) * aspect * half_w
    scy = (1 - 2 * ((ys.ravel() + sy) / H)) * half_h
    d = np.stack([scx, scy, -np.ones_like(scx)], axis=1)
    for _ in range(2):
        d = d / np.sqrt((d * d).sum(axis=1))[:, None]
    return d.reshape(y1 - y0, W, 3)


def nearest_hits(fs, O, D):
    """Algorithm B's nearest hit (oracle trace_path / sphere_discriminant): -> (index or -1, t) per ray."""
    m = D.shape[0]
    best, bt, bi = np.full(m, np.inf), np.zeros(m), np.full(m, -1)
    C_, R = np.asarray(fs.centre, np.float64), np.asarray(fs.radius, np.float64)
    for i in range(C_.shape[0]):
        L = C_[i] - O
        tca = D @ L
        q = L @ L - tca * tca
        d = np.sqrt(np.maximum(q, 0.0))
        hit = (tca >= 0) & ~(d > R[i])
        with np.errstate(invalid="ignore"):
            t = tca - np.sqrt(R[i] * R[i] - d * d)
        p = O + D * t[:, None]
        dist = np.sqrt(((p - O) ** 2).sum(axis=1))
        better = hit & (dist < best)
        best, bt, bi = np.where(better, dist, best), np.where(better, t, bt), np.where(better, i, bi)
    return bi, bt


def aov_reference(orc, fs, cam, W, H, seed, rows, samples):
    """-> (albedo, normal, depth, fvar) float64 for rows x samples, as rt_render_features defines them."""
    y0, y1 = rows
    O = np.asarray(cam, np.float64)
    C_, R, col = (np.asarray(a, np.float64) for a in (fs.centre, fs.radius, fs.colour))
    s_ = np.zeros((y1 - y0, W, 7))
    q_ = np.zeros((y1 - y0, W, 7))
    for smp in range(*samples):
        D = camera_rays(orc, cam, W, H, seed, y0, y1, smp).reshape(-1, 3)
        idx, t = nearest_hits(fs, O, D)
        f = np.zeros((D.shape[0], 7))
        h = idx >= 0
        f[h, 0:3] = col[idx[h]] / 255.0
        f[h, 3:6] = (O + D[h] * t[h, None] - C_[idx[h]]) * (1.0 / R[idx[h]])[:, None]
        f[h, 6] = t[h]
        f = f.reshape(y1 - y0, W, 7)
        s_ += f
        q_ += f * f
    n = samples[1] - samples[0]
    v = np.zeros_like(s_) if n < 2 else np.maximum(0.0, (q_ - s_ * s_ / n) / (n * (n - 1.0)))
    mean = s_ / n
    fvar = np.stack([(v[..., 0] + v[..., 1] + v[..., 2]) / 3, (v[..., 3] + v[..., 4] + v[..., 5]) / 3, v[..., 6]], -1)
    return mean[..., 0:3], mean[..., 3:6], mean[..., 6], fvar


def render_features(nat, sc, cam, W, H, seed, prec, rows=None, samples=(0, 8), fill=0):
    """Device buffers around one rt_render_features -> (albedo, normal, depth, fvar) host arrays."""
    p = sc.path_params(cam, W, H, samples[1], 1, 0.0, seed=seed, rows=rows, samples=samples)
    bufs = [nat.DeviceBuffer(s, np.float32) for s in ((H, W, 3), (H, W, 3), (H, W), (H, W, 3))]
    if fill:
        for b in bufs:
            b.fill(fill)
    sc.render_features(p, *bufs, precision=prec)
    return [b.download() for b in bufs]


def ulps(a, b):
    """Distance in float32 units in the last place."""
    def key(x):
        i = np.ascontiguousarray(x, np.float32).view(np.int32).astype(np.int64)
        return np.where(i < 0, -(i & 0x7FFFFFFF), i)
    return np.abs(key(a) - key(b))


def feature_frames():
    from ray_tracer_v1_b200 import scenes
    z, fs = load_golden("path_complex_48x27")
    yield "complex", fs, z["cam"], int(z["W"]), int(z["H"]), False
    z, fs = load_golden("path_chandelier_48x27")
    yield "chandelier+lbvh", fs, z["cam"], 64, 36, True
    yield "2000 spheres", scenes.build_many_spheres_flat(2000, seed=2, emissive_fraction=0.05), (0.0, 2.0, 0.0), 40, 24, True
    z, fs = load_golden("path_complex_48x27")
    yield "complex 33x9", fs, z["cam"], 33, 9, False          # one column and one row into a second 32 x 8 CTA
    yield "complex 1x24", fs, z["cam"], 1, 24, False


# FP32 features may differ from the reference only where an FP32 ray flips a hit, at silhouettes: a pixel whose sample
# hits a different sphere (or misses) moves its means by a large step.  The gate bounds the share of such pixels.  On the
# B200 no frame below had one, so the limit is the gate's floor of two pixels per frame.
FP32_FLIP_LIMIT = 0.0


@pytest.mark.parametrize("precision", PRECISIONS)
def test_features_match_reference(nat, orc, precision):
    """Every scene-residency mode (shared, shared + LBVH, global + LBVH), frames one pixel past a CTA in x and y and one
    pixel wide, row bands (one of a single row) and sample ranges (one far from 0)."""
    prec = getattr(nat, precision)
    for name, fs, cam, W, H, lbvh in feature_frames():
        sc = nat.DeviceScene(fs)
        if lbvh:
            sc.build_lbvh()
            assert sc.has_lbvh
        bands = [((0, H), (0, 8)), ((0, H), (2, 3)), ((H // 2, H // 2 + 1), (1000, 1004))]
        for rows, samples in bands + ([((5, H - 7), (3, 7))] if H > 12 else []):
            got = render_features(nat, sc, cam, W, H, 11, prec, rows, samples, fill=0x7F)
            ref = aov_reference(orc, fs, cam, W, H, 11, rows, samples)
            y0, y1 = rows
            for g in got:                                      # rows outside the band are left alone
                assert np.all(g[:y0].view(np.uint8) == 0x7F) and np.all(g[y1:].view(np.uint8) == 0x7F)
            got = [g[y0:y1] for g in got]
            if samples[1] - samples[0] < 2:
                assert np.all(got[3] == 0)
            if prec == nat.F64:
                for j, (g, r) in enumerate(zip(got[:3], ref[:3])):
                    assert ulps(g, r.astype(np.float32)).max() <= 1, (name, j, ulps(g, r.astype(np.float32)).max())
                # a variance is a difference of sums of squares: where it lies far below their rounding error (the
                # depth of a sphere around the camera, t ~ -r, inside one pixel), the last bits of the rays decide it;
                # there it is checked against that error, (1e-13 x the mean square of the feature), elsewhere to 1 ulp
                scale = np.stack([np.ones(ref[2].shape), np.ones(ref[2].shape), np.maximum(1.0, ref[2] ** 2)], -1)
                ok = (ulps(got[3], ref[3].astype(np.float32)) <= 1) | (np.abs(got[3] - ref[3]) <= 1e-13 * scale)
                assert ok.all(), (name, np.abs(got[3] - ref[3])[~ok].max(), ref[3][~ok][:4])
            else:
                bad = np.zeros(got[2].shape, bool)
                for g, r in zip(got, ref):
                    d = np.abs(g.astype(np.float64) - r)
                    tol = 1e-3 * np.maximum(1.0, np.abs(r))
                    d = d if d.ndim == 2 else d.max(axis=-1)
                    bad |= d > (tol if tol.ndim == 2 else tol.max(axis=-1))
                gate(f"features FP32 flipped pixels {name} {rows} {samples}", bad.mean(),
                     max(FP32_FLIP_LIMIT, 2.0 / bad.size))
        sc.close()


# ------------------------------------------------------------------ filter reference
def nlm_features_reference(acc, var, feats, radius=10, patch_radius=3, k=1.0, k_f=1.2, tau=1e-3):
    """nlm_reference (test_gpu_denoise.py) with the feature term, in float64 -> u_hat [H,W,3] before the floor."""
    r, f = radius, patch_radius
    n = acc[..., 3:4].astype(np.float64)
    u = (acc[..., :3].astype(np.float64) / n).astype(np.float32).astype(np.float64)
    V = var.astype(np.float64)
    H, W = u.shape[:2]
    albedo, normal, depth, fvar = (a.astype(np.float64) for a in feats)
    F = [albedo, normal, depth[..., None]]
    FV = [fvar[..., j] for j in range(3)]

    def at(a, ys, xs):
        return a[np.clip(ys, 0, H - 1)][:, np.clip(xs, 0, W - 1)]

    Y, X = np.arange(H), np.arange(W)
    den = []
    for j in range(3):
        gx = (at(F[j], Y, X + 1) - at(F[j], Y, X - 1)) / 2
        gy = (at(F[j], Y + 1, X) - at(F[j], Y - 1, X)) / 2
        G = (gx * gx + gy * gy).mean(axis=2)
        den.append(k_f * k_f * np.maximum(tau, np.maximum(FV[j], G)))
    ye, xe = np.arange(-f, H + f), np.arange(-f, W + f)
    up, vp = at(u, ye, xe), at(V, ye, xe)
    P = 2 * f + 1
    sw, su = np.zeros((H, W, 1)), np.zeros((H, W, 3))
    for oy in range(-r, r + 1):
        for ox in range(-r, r + 1):
            uq, vq = at(u, ye + oy, xe + ox), at(V, ye + oy, xe + ox)
            d = (((up - uq) ** 2 - (vp + np.minimum(vp, vq))) / (EPS + k * k * (vp + vq))).mean(axis=2)
            rows = sum(d[:, t:t + W] for t in range(P))
            e = sum(rows[t:t + H] for t in range(P)) / (P * P)
            with np.errstate(divide="ignore", invalid="ignore"):
                for j in range(3):
                    fq, vfq = at(F[j], Y + oy, X + ox), at(FV[j], Y + oy, X + ox)
                    num = ((F[j] - fq) ** 2).mean(axis=2) - (FV[j] + np.minimum(FV[j], vfq))
                    e = np.fmax(e, num / den[j])
            w = np.exp(-np.maximum(0.0, e))[..., None]
            sw += w
            su += w * (at(u, Y + oy, X + ox) - u)
    return u + su / sw


def uniform(nat, sc, frame, spp, prec, seed):
    """The uniform moments frame and its features -> (accum, variance, features)."""
    cam, W, H, depth, thr = frame
    p = sc.path_params(cam, W, H, spp, depth, thr, seed=seed)
    acc, mom = nat.DeviceBuffer((H, W, 4), _ft(nat, prec)), nat.DeviceBuffer((H, W, 4), np.float64)
    var = nat.DeviceBuffer((H, W, 3), np.float32)
    sc.render_path(p, acc, prec, moments=mom)
    sc.resolve_variance(acc, mom, W, H, var, prec)
    feats = render_features(nat, sc, cam, W, H, seed, prec, samples=(0, min(spp, 8)))
    return acc.download(), var.download(), feats


def denoise_features(nat, sc, acc, var, feats, prec, **params):
    H, W = acc.shape[:2]
    a, v = nat.DeviceBuffer.from_host(acc, _ft(nat, prec)), nat.DeviceBuffer.from_host(var, np.float32)
    fb = [nat.DeviceBuffer.from_host(x, np.float32) for x in feats]
    img = nat.DeviceBuffer((H, W, 3), np.float32)
    sc.denoise(a, v, W, H, img, prec, features=fb, **params)
    return img.download()


def golden_frames():
    z, fs = load_golden("path_complex_48x27")
    yield "complex", fs, (z["cam"], int(z["W"]), int(z["H"]), int(z["max_bounces"]), float(z["mirror_threshold"]))
    z, fs = load_golden("path_chandelier_48x27")
    yield "chandelier", fs, (z["cam"], 64, 36, int(z["max_bounces"]), float(z["mirror_threshold"]))


@pytest.mark.parametrize("precision", PRECISIONS)
def test_denoise_features_matches_reference(nat, precision):
    """Complex and chandelier frames at (r, f) = (10, 3), (3, 1), (15, 5); the features change the image."""
    prec = getattr(nat, precision)
    for name, fs, frame in golden_frames():
        sc = nat.DeviceScene(fs)
        acc, var, feats = uniform(nat, sc, frame, 8, prec, seed=3)
        for r, f in ((10, 3), (3, 1), (15, 5)):
            img = denoise_features(nat, sc, acc, var, feats, prec, radius=r, patch_radius=f)
            u_hat = nlm_features_reference(acc, var, feats, r, f)
            check_against_reference(img, u_hat)
            if name == "complex":       # (on the small chandelier frame the feature term lowers no weight that matters)
                assert np.abs(u_hat - nlm_reference(acc, var, r, f, k=1.0)).max() > 0.1, name
        sc.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_denoise_features_frame_smaller_than_the_window(nat, precision):
    """8 x 5 pixels under a 21 x 21 window: features, gradients and colours are all read clamped."""
    prec = getattr(nat, precision)
    z, fs = load_golden("path_complex_48x27")
    sc = nat.DeviceScene(fs)
    acc, var, feats = uniform(nat, sc, (z["cam"], 8, 5, int(z["max_bounces"]), float(z["mirror_threshold"])), 16, prec, 4)
    for r, f in ((10, 3), (15, 5), (10, 0), (1, 0)):
        check_against_reference(denoise_features(nat, sc, acc, var, feats, prec, radius=r, patch_radius=f),
                                nlm_features_reference(acc, var, feats, r, f))
    sc.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_denoise_features_adaptive_input(nat, precision):
    """An adaptive frame (per-pixel sample counts) with the features of its first 8 samples."""
    prec = getattr(nat, precision)
    z, fs = load_golden("path_complex_48x27")
    sc = nat.DeviceScene(fs)
    W, H = int(z["W"]), int(z["H"])
    p = sc.path_params(z["cam"], W, H, 16, int(z["max_bounces"]), float(z["mirror_threshold"]), seed=8)
    acc, mom = nat.DeviceBuffer((H, W, 4), _ft(nat, prec)), nat.DeviceBuffer((H, W, 4), np.float64)
    lst, img = nat.DeviceBuffer(H * W + 1, np.uint32), nat.DeviceBuffer((H, W, 3), np.float32)
    var, cnt = nat.DeviceBuffer((H, W, 3), np.float32), nat.DeviceBuffer((H, W), np.int32)
    sc.render_path_adaptive(p, 2, 4.0, acc, mom, lst, img, prec, var=var, counts=cnt)
    assert len(np.unique(cnt.download())) >= 2
    feats = render_features(nat, sc, z["cam"], W, H, 8, prec)
    a, v = acc.download(), var.download()
    check_against_reference(denoise_features(nat, sc, a, v, feats, prec), nlm_features_reference(a, v, feats))
    sc.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_denoise_features_identities(nat, precision):
    """k_f = 1e18 gives rt_denoise's image bit for bit (w_f = 1); r = 0 gives floor(float32(S / n)); two calls give the
    same bits."""
    prec = getattr(nat, precision)
    z, fs = load_golden("path_complex_48x27")
    sc = nat.DeviceScene(fs)
    W, H = 160, 90
    acc, var, feats = uniform(nat, sc, (z["cam"], W, H, int(z["max_bounces"]), float(z["mirror_threshold"])), 8, prec, 6)
    a, v = nat.DeviceBuffer.from_host(acc, _ft(nat, prec)), nat.DeviceBuffer.from_host(var, np.float32)
    plain = nat.DeviceBuffer((H, W, 3), np.float32)
    for r, f in ((10, 3), (3, 1), (15, 5)):
        sc.denoise(a, v, W, H, plain, prec, radius=r, patch_radius=f, k=0.45)
        assert np.array_equal(denoise_features(nat, sc, acc, var, feats, prec, radius=r, patch_radius=f, k=0.45, k_f=1e18),
                              plain.download())
    u32 = (acc[..., :3].astype(np.float64) / acc[..., 3:4]).astype(np.float32).astype(np.float64)
    for f in (0, 3):
        assert np.array_equal(denoise_features(nat, sc, acc, var, feats, prec, radius=0, patch_radius=f), lattice(u32))
    outs = [denoise_features(nat, sc, acc, var, feats, prec) for _ in range(2)]
    assert outs[0].tobytes() == outs[1].tobytes()
    again = render_features(nat, sc, z["cam"], W, H, 6, prec)
    assert all(x.tobytes() == y.tobytes() for x, y in zip(again, feats))
    sc.close()


def test_features_validation(nat):
    """Every rejection returns RT_ERR_INVALID and names the cause."""
    L = nat.lib()
    INVALID = 1
    z, fs = load_golden("path_complex_48x27")
    sc = nat.DeviceScene(fs)
    W, H = 16, 8
    bufs = [nat.DeviceBuffer(s, np.float32) for s in ((H, W, 3), (H, W, 3), (H, W), (H, W, 3))]
    ptrs = [b.ptr for b in bufs]

    def render(prec=nat.F32, handle=True, params=True, ptrs_=None, **kw):
        p = sc.path_params(z["cam"], W, H, 4, 1, 0.0, rows=kw.get("rows"), samples=kw.get("samples"))
        rc = L.rt_render_features(sc.handle if handle else None, prec, C.byref(p) if params else None,
                                  *(ptrs_ or ptrs), None)
        return rc, L.rt_last_error().decode()

    assert render()[0] == 0
    nat.check(L.rt_stream_sync(0, None))
    assert render(handle=False) == (INVALID, "NULL argument")
    assert render(params=False) == (INVALID, "NULL argument")
    for k in range(4):
        assert render(ptrs_=[None if i == k else q for i, q in enumerate(ptrs)]) == (INVALID, "NULL argument")
    assert render(rows=(3, 2)) == (INVALID, "row band outside the image")
    assert render(rows=(0, H + 1)) == (INVALID, "row band outside the image")
    assert render(samples=(-1, 4)) == (INVALID, "bad sample range")
    assert render(samples=(4, 4)) == (INVALID, "empty sample range: s1 must be greater than s0")
    assert render(prec=2) == (INVALID, "unknown precision")

    frame = np.zeros((H, W, 4), np.float32)
    frame[..., 3] = 1
    acc, var = nat.DeviceBuffer.from_host(frame), nat.DeviceBuffer((H, W, 3), np.float32)
    img = nat.DeviceBuffer((H, W, 3), np.float32)

    def call(prec=nat.F32, w=W, h=H, base=None, feat=None, params=True, **kw):
        d = nat.DenoiseFeaturesParams()
        d.radius, d.patch_radius, d.k = kw.get("radius", 10), kw.get("patch_radius", 3), kw.get("k", 0.45)
        d.k_f, d.tau = kw.get("k_f", 0.6), kw.get("tau", 1e-3)
        a, v, i = base or (acc.ptr, var.ptr, img.ptr)
        rc = L.rt_denoise_features(0, prec, a, v, *(feat or ptrs), w, h, C.byref(d) if params else None, i, None)
        return rc, L.rt_last_error().decode()

    assert call()[0] == 0
    nat.check(L.rt_stream_sync(0, None))
    for base in ((None, var.ptr, img.ptr), (acc.ptr, None, img.ptr), (acc.ptr, var.ptr, None)):
        assert call(base=base) == (INVALID, "NULL argument")
    assert call(params=False) == (INVALID, "NULL argument")
    for k in range(4):
        assert call(feat=[None if i == k else q for i, q in enumerate(ptrs)]) == (INVALID, "NULL feature buffer")
    cases = [(dict(w=0), "W and H must be at least 1"), (dict(h=-2), "W and H must be at least 1"),
             (dict(prec=2), "unknown precision"), (dict(radius=16), "radius must be in [0, 15]"),
             (dict(radius=-1), "radius must be in [0, 15]"), (dict(patch_radius=6), "patch_radius must be in [0, 5]"),
             (dict(k=0.0), "k must be finite and > 0"), (dict(k=float("nan")), "k must be finite and > 0"),
             (dict(k_f=0.0), "k_f must be finite and > 0"), (dict(k_f=-1.0), "k_f must be finite and > 0"),
             (dict(k_f=float("inf")), "k_f must be finite and > 0"), (dict(k_f=float("nan")), "k_f must be finite and > 0"),
             (dict(tau=-1e-6), "tau must be finite and >= 0"), (dict(tau=float("inf")), "tau must be finite and >= 0"),
             (dict(tau=float("nan")), "tau must be finite and >= 0")]
    for kw, msg in cases:
        assert call(**kw) == (INVALID, msg), kw
    for kw in (dict(radius=0, patch_radius=0), dict(radius=15, patch_radius=5), dict(tau=0.0), dict(k_f=1e18)):
        assert call(**kw)[0] == 0, kw
    nat.check(L.rt_stream_sync(0, None))
    sc.close()


def _renderer(rt, spec, seed):
    r = rt.ComplexTraditionalRenderer(precision="f32", seed=seed)
    r.scene = spec.spheres
    r.light_sources = [s for s in spec.spheres if s.material.emitive]
    r.camera_position = rt.Vector(*spec.camera)
    r.reuse_output = False
    return r


def test_renderer_features(rt, nat):
    """track_features = False changes nothing; True sets albedo / normal / depth (the features of the first
    FEATURE_SPP samples) and makes denoise feature-guided, uniform and adaptive, with and without track_variance."""
    from ray_tracer_v1_b200 import scenes
    from ray_tracer_v1_b200.frames import FrameContext
    spec = scenes.build_complex()
    W, H, spp, seed = 160, 90, 16, 5
    r = _renderer(rt, spec, seed)
    sc = nat.DeviceScene(r.flat_scene())
    nf = min(spp, FrameContext.FEATURE_SPP)
    feats = render_features(nat, sc, spec.camera, W, H, seed, nat.F32, samples=(0, nf))
    p = sc.path_params(spec.camera, W, H, spp, 5, 0.9, seed=seed)
    acc, mom = nat.DeviceBuffer((H, W, 4), np.float32), nat.DeviceBuffer((H, W, 4), np.float64)
    var, img = nat.DeviceBuffer((H, W, 3), np.float32), nat.DeviceBuffer((H, W, 3), np.float32)
    sc.render_path(p, acc, nat.F32, moments=mom)
    sc.resolve(acc, W, H, spp, img, nat.F32)
    resolved = img.download()
    sc.resolve_variance(acc, mom, W, H, var, nat.F32)
    sc.denoise(acc, var, W, H, img, nat.F32)
    denoised = img.download()
    fb = [nat.DeviceBuffer.from_host(x, np.float32) for x in feats]
    sc.denoise(acc, var, W, H, img, nat.F32, features=fb)
    guided = img.download()
    assert not np.array_equal(guided, denoised)

    assert np.array_equal(r.render(W, H, spp, 5), resolved)
    assert r._ctx.features is None and not hasattr(r, "albedo") and r._ctx.launches == 2
    r.track_features = True
    assert np.array_equal(r.render(W, H, spp, 5), resolved) and r._ctx.launches == 3
    assert r.albedo.shape == (H, W, 3) and r.normal.shape == (H, W, 3) and r.depth.shape == (H, W)
    for got, want in zip((r.albedo, r.normal, r.depth), feats):
        assert np.array_equal(got, want)
    r.denoise = True
    assert np.array_equal(r.render(W, H, spp, 5), guided)
    r.track_variance = True
    assert np.array_equal(r.render(W, H, spp, 5), guided) and np.array_equal(r.variance, var.download())
    r.track_features = False
    assert np.array_equal(r.render(W, H, spp, 5), denoised)

    # adaptive: the features of the first FEATURE_SPP samples guide the filter of the adaptive frame
    r.track_features = True
    r.adaptive_tolerance = 2.0
    pa = sc.path_params(spec.camera, W, H, 64, 5, 0.9, seed=seed)
    lst, cnt = nat.DeviceBuffer(H * W + 1, np.uint32), nat.DeviceBuffer((H, W), np.int32)
    sc.render_path_adaptive(pa, r.adaptive_min_spp, 2.0, acc, mom, lst, img, nat.F32, var=var, counts=cnt)
    fa = render_features(nat, sc, spec.camera, W, H, seed, nat.F32, samples=(0, FrameContext.FEATURE_SPP))
    fb = [nat.DeviceBuffer.from_host(x, np.float32) for x in fa]
    sc.denoise(acc, var, W, H, img, nat.F32, features=fb)
    assert np.array_equal(r.render(W, H, 64, 5), img.download())
    assert np.array_equal(r.sample_counts, cnt.download()) and np.array_equal(r.variance, var.download())
    assert all(np.array_equal(g, w) for g, w in zip((r.albedo, r.normal, r.depth), fa))
    sc.close()


def test_frame_context_features(rt, nat):
    """FrameContext: features off allocates nothing; on exposes the feature buffers of the rendered rows; return shapes
    do not change."""
    from ray_tracer_v1_b200 import scenes
    from ray_tracer_v1_b200.frames import FrameContext
    import ray_tracer_v1_b200 as rtb
    spec = scenes.build_complex()
    ctx = FrameContext()
    ctx.set_scene(rtb.flatten_scene(spec.spheres, background_colour=spec.background))
    out = ctx.render_path(spec.camera, 64, 36, 4, 5, 0.9)
    assert len(out) == 2 and ctx.features is None and ctx.albedo is None
    out = ctx.render_path(spec.camera, 64, 36, 4, 5, 0.9, features=True, variance=True, rows=(8, 20))
    assert len(out) == 3
    assert ctx.albedo.shape == (36, 64, 3) and ctx.normal.shape == (36, 64, 3) and ctx.depth.shape == (36, 64)
    assert ctx.feature_var.shape == (36, 64, 3)
    want = render_features(nat, ctx.scene, spec.camera, 64, 36, 0, nat.F32, rows=(8, 20), samples=(0, 4))
    for got, w in zip((ctx.albedo, ctx.normal, ctx.depth, ctx.feature_var), want):
        assert np.array_equal(got[8:20], w[8:20])
    out = ctx.render_path_adaptive(spec.camera, 64, 36, 16, 5, 0.9, 4, 2.0, features=True, denoise=True)
    assert len(out) == 4 and ctx.depth.shape == (36, 64)
    ctx.close()
