"""Adaptive Algorithm B frames (rt_render_path_adaptive): every pixel gets min_spp samples, then doubling rounds for the
pixels whose variance of the mean still exceeds tolerance^2.

The oracle is exact: a pixel that stopped after c samples must equal, bit for bit, the uniform frame rendered with c
samples (accum, moments, variance), because the samples are keyed by (pixel, sample) and the sums are exact.  The
expected sample counts come from replaying the stopping rule on the host over the uniform frames' variances."""
import ctypes as C

import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu

PRECISIONS = ["F32", "F64"]


@pytest.fixture(scope="module")
def nat(rt):
    from ray_tracer_v1_b200 import _native
    return _native


def _ft(nat, prec):
    return np.float64 if prec == nat.F64 else np.float32


def checkpoints(min_spp, max_spp):
    c = [min_spp]
    while c[-1] < max_spp:
        c.append(min(2 * c[-1], max_spp))
    return c


def uniform(nat, sc, frame, spp, prec, **kw):
    """The uniform moments frame with spp samples -> (accum, moments, variance, image, stats)."""
    cam, W, H, depth, thr = frame
    p = sc.path_params(cam, W, H, spp, depth, thr, **kw)
    acc, mom = nat.DeviceBuffer((H, W, 4), _ft(nat, prec)), nat.DeviceBuffer((H, W, 4), np.float64)
    var, img, st = nat.DeviceBuffer((H, W, 3), np.float32), nat.DeviceBuffer((H, W, 3), np.float32), nat.DeviceBuffer(8, np.uint64)
    sc.render_path(p, acc, prec, stats=st, moments=mom)
    sc.resolve_variance(acc, mom, W, H, var, prec)
    sc.resolve(acc, W, H, spp, img, prec)
    return acc.download(), mom.download(), var.download(), img.download(), st.download()


def adaptive(nat, sc, frame, min_spp, max_spp, tol, prec, **kw):
    """-> (accum, moments, variance, image, counts, stats) of the adaptive frame."""
    cam, W, H, depth, thr = frame
    p = sc.path_params(cam, W, H, max_spp, depth, thr, **kw)
    acc, mom = nat.DeviceBuffer((H, W, 4), _ft(nat, prec)), nat.DeviceBuffer((H, W, 4), np.float64)
    lst = nat.DeviceBuffer(H * W + 1, np.uint32)
    var, img = nat.DeviceBuffer((H, W, 3), np.float32), nat.DeviceBuffer((H, W, 3), np.float32)
    cnt, st = nat.DeviceBuffer((H, W), np.int32), nat.DeviceBuffer(8, np.uint64)
    sc.render_path_adaptive(p, min_spp, tol, acc, mom, lst, img, prec, var=var, counts=cnt, stats=st)
    return acc.download(), mom.download(), var.download(), img.download(), cnt.download(), st.download()


def expected_counts(variances, cps, tol):
    """The stopping rule on the host: float32 variances compared in double."""
    thr = -1.0 if tol < 0 else float(tol) ** 2
    n = np.full(variances[0].shape[:2], cps[0], np.int32)
    active = np.ones(n.shape, bool)
    for r in range(len(cps) - 1):
        active &= (variances[r].astype(np.float64) > thr).any(axis=2)
        n[active] = cps[r + 1]
    return n


def pick_tolerance(variances, cps):
    """A tolerance under which pixels stop at every checkpoint and some still reach the last one."""
    v = variances[0].astype(np.float64).max(axis=2)
    for q in (0.5, 0.6, 0.4, 0.7, 0.3, 0.8, 0.2, 0.9):
        tol = float(np.sqrt(np.quantile(v[v > 0], q)))
        n = expected_counts(variances, cps, tol)
        if all((n == c).any() for c in cps):
            return tol, n
    raise AssertionError("no tolerance stops pixels at every checkpoint")


def check_oracle(nat, sc, frame, min_spp, max_spp, prec, **kw):
    cps = checkpoints(min_spp, max_spp)
    U = [uniform(nat, sc, frame, c, prec, **kw) for c in cps]
    tol, n_p = pick_tolerance([u[2] for u in U], cps)
    for c in cps[:-1]:
        assert (n_p == c).any() and (n_p > c).any(), (c, np.bincount(n_p.ravel()))
    acc, mom, var, img, cnt, _ = adaptive(nat, sc, frame, min_spp, max_spp, tol, prec, **kw)
    assert np.array_equal(cnt, n_p)
    assert np.array_equal(acc[..., 3], n_p.astype(acc.dtype)) and np.array_equal(mom[..., 3], n_p.astype(np.float64))
    for r, c in enumerate(cps):
        m = n_p == c
        assert np.array_equal(acc[m], U[r][0][m]), c
        assert np.array_equal(mom[m], U[r][1][m]), c
        assert np.array_equal(var[m], U[r][2][m]), c
        assert np.array_equal(img[m], U[r][3][m]), c
    S, n = acc[..., :3].astype(np.float64), n_p[..., None].astype(np.float64)
    assert np.array_equal(img, np.minimum(1.0, np.floor(S / n) / 255.0).astype(np.float32))
    return n_p


def complex_frame(z):
    return (z["cam"], int(z["W"]), int(z["H"]), int(z["max_bounces"]), float(z["mirror_threshold"]))


@pytest.mark.parametrize("precision", PRECISIONS)
def test_adaptive_exact_complex_schedules_and_ksplit(nat, precision):
    """The complex golden scene: the parameter-block kernel (kMode 3) with its camera-ray candidate lists, without them
    (schedule 2), the shared-memory kernel (schedule 4), and every sample split."""
    prec = getattr(nat, precision)
    z, fs = load_golden("path_complex_48x27")
    sc = nat.DeviceScene(fs)
    frame = complex_frame(z)
    check_oracle(nat, sc, frame, 2, 16, prec, seed=3)
    for schedule in (2, 4):
        check_oracle(nat, sc, frame, 2, 16, prec, seed=3, schedule=schedule)
    for ksplit in (0, 1, 2, 8, 32, -1):
        check_oracle(nat, sc, frame, 4, 24, prec, seed=5, ksplit=ksplit)
    sc.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_adaptive_exact_hierarchy_and_global_memory(nat, precision):
    """The chandelier with the LBVH forced (shared-memory scene + hierarchy) and a 2000-sphere scene (global-memory
    scene + hierarchy)."""
    from ray_tracer_v1_b200 import scenes
    prec = getattr(nat, precision)
    z, fs = load_golden("path_chandelier_48x27")
    sc = nat.DeviceScene(fs)
    sc.build_lbvh()
    assert sc.has_lbvh
    check_oracle(nat, sc, (z["cam"], 64, 36, int(z["max_bounces"]), float(z["mirror_threshold"])), 2, 16, prec, seed=7)
    sc.close()
    sc = nat.DeviceScene(scenes.build_many_spheres_flat(2000, seed=2, emissive_fraction=0.05))
    sc.build_lbvh()
    check_oracle(nat, sc, ((0.0, 2.0, 0.0), 64, 36, 4, 0.0), 2, 8, prec, seed=9)
    sc.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_adaptive_limits(nat, precision):
    """A negative tolerance gives the uniform max_spp frame; a huge one the uniform min_spp frame without a list launch
    (the counters, sphere and AABB tests included, are those of the one uniform launch)."""
    prec = getattr(nat, precision)
    z, fs = load_golden("path_complex_48x27")
    sc = nat.DeviceScene(fs)
    frame = complex_frame(z)
    for tol, spp in ((-1.0, 16), (1e300, 2)):
        acc_u, mom_u, var_u, img_u, st_u = uniform(nat, sc, frame, spp, prec, seed=11)
        acc, mom, var, img, cnt, st = adaptive(nat, sc, frame, 2, 16, tol, prec, seed=11)
        assert np.all(cnt == spp)
        for a, b in ((acc, acc_u), (mom, mom_u), (var, var_u), (img, img_u)):
            assert np.array_equal(a, b)
        if spp == 16:
            assert np.array_equal(st[:5], st_u[:5])            # the cones of the list launches differ: [5], [6] may
        else:
            assert np.array_equal(st, st_u)
    sc.close()


def test_adaptive_list_launch_with_the_fold_table(nat):
    """512 x 512 pixels x 16 samples: the list round of a negative-tolerance frame folds through the per-CTA byte table
    (FP32 kMode 3) and still equals the uniform frame."""
    z, fs = load_golden("path_complex_48x27")
    sc = nat.DeviceScene(fs)
    frame = (z["cam"], 512, 512, 5, float(z["mirror_threshold"]))
    acc_u, mom_u, var_u, img_u, st_u = uniform(nat, sc, frame, 32, nat.F32, seed=3)
    acc, mom, var, img, cnt, st = adaptive(nat, sc, frame, 16, 32, -1.0, nat.F32, seed=3)
    assert np.all(cnt == 32)
    for a, b in ((acc, acc_u), (mom, mom_u), (var, var_u), (img, img_u)):
        assert np.array_equal(a, b)
    assert np.array_equal(st[:5], st_u[:5])
    sc.close()


def test_adaptive_validation(nat):
    """Every rejection returns its code and names the cause."""
    L = nat.lib()
    z, fs = load_golden("path_complex_48x27")
    sc = nat.DeviceScene(fs)
    W, H = int(z["W"]), int(z["H"])
    acc, mom = nat.DeviceBuffer((H, W, 4), np.float32), nat.DeviceBuffer((H, W, 4), np.float64)
    lst, img = nat.DeviceBuffer(H * W + 1, np.uint32), nat.DeviceBuffer((H, W, 3), np.float32)

    def call(scene, prec=nat.F32, min_spp=2, tol=1.0, ptrs=None, **kw):
        p = scene.path_params(z["cam"], W, H, kw.pop("spp", 8), 5, 0.9, **kw)
        a = nat.AdaptiveParams()
        a.min_spp, a.tolerance = min_spp, tol
        acc_p, mom_p, lst_p, img_p = ptrs or (acc.ptr, mom.ptr, lst.ptr, img.ptr)
        rc = L.rt_render_path_adaptive(scene.handle, prec, C.byref(p), C.byref(a), acc_p, mom_p, lst_p, img_p, None, None,
                                       None, None)
        return rc, L.rt_last_error().decode()

    INVALID, UNSUPPORTED = 1, 4
    for ptrs in ((None, mom.ptr, lst.ptr, img.ptr), (acc.ptr, None, lst.ptr, img.ptr), (acc.ptr, mom.ptr, None, img.ptr),
                 (acc.ptr, mom.ptr, lst.ptr, None)):
        rc, msg = call(sc, ptrs=ptrs)
        assert rc == INVALID and "NULL" in msg
    cases = [(dict(samples=(1, 8)), "s0"), (dict(accumulate=True), "accumulate"), (dict(min_spp=1), "min_spp"),
             (dict(min_spp=9), "min_spp"), (dict(tol=float("nan")), "NaN"), (dict(schedule=1), "schedule"),
             (dict(schedule=8), "schedule"), (dict(spp=65537), "65536")]
    for kw, word in cases:
        rc, msg = call(sc, **kw)
        assert rc == INVALID and word in msg, (kw, rc, msg)
    sc.close()
    # non-integer colours
    fs_f = load_golden("path_complex_48x27")[1]
    fs_f.colour = fs_f.colour + 0.37
    sc = nat.DeviceScene(fs_f)
    for prec in (nat.F32, nat.F64):
        rc, msg = call(sc, prec)
        assert rc == UNSUPPORTED and "integer colours" in msg
    sc.close()
    # FP32 sums stop being exact: with colours above 255, 65535 * 257 >= 2^24 while 65535 * 256 < 2^24 (a 255-colour
    # scene stays exact up to the 65536-sample limit: 255 * 65536 < 2^24)
    fs_w = load_golden("path_complex_48x27")[1]
    fs_w.colour = fs_w.colour.copy()
    fs_w.colour[0, 0] = 300.0
    sc = nat.DeviceScene(fs_w)
    rc, msg = call(sc, nat.F32, spp=257)
    assert rc == UNSUPPORTED and "2^24" in msg
    rc, msg = call(sc, nat.F32, spp=256)                              # just below the bound: accepted
    assert rc == 0, msg
    nat.check(L.rt_stream_sync(0, None))
    sc.close()


def _renderer(rt, spec, seed):
    r = rt.ComplexTraditionalRenderer(precision="f32", seed=seed)
    r.scene = spec.spheres
    r.light_sources = [s for s in spec.spheres if s.material.emitive]
    r.camera_position = rt.Vector(*spec.camera)
    return r


def test_renderer_adaptive(rt, nat):
    """ComplexTraditionalRenderer with adaptive_tolerance: the image and counts of FrameContext.render_path_adaptive,
    counts in [min_spp, max_spp]; the variance with track_variance."""
    from ray_tracer_v1_b200 import scenes
    from ray_tracer_v1_b200.frames import FrameContext
    spec = scenes.build_complex()
    W, H, max_spp, tol = 160, 90, 64, 2.0
    r = _renderer(rt, spec, 5)
    r.reuse_output = False
    r.adaptive_tolerance = tol
    r.track_variance = True
    img = r.render(W, H, max_spp, 5)
    ctx = FrameContext()
    ctx.set_scene(r.flat_scene())
    img_c, st_c, var_c, cnt_c = ctx.render_path_adaptive(spec.camera, W, H, max_spp, 5, 0.9, r.adaptive_min_spp, tol, seed=5)
    assert np.array_equal(img, img_c) and np.array_equal(r.sample_counts, cnt_c) and np.array_equal(r.variance, var_c)
    assert r.stats["total_rays"] == int(st_c[0])
    assert r.sample_counts.shape == (H, W) and r.sample_counts.dtype == np.int32
    assert r.sample_counts.min() >= r.adaptive_min_spp and r.sample_counts.max() <= max_spp
    assert r.sample_counts.min() < max_spp                              # some pixels stopped early
    ctx.close()
