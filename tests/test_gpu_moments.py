"""Per-pixel second moments of Algorithm B frames (rt_render_path_moments, rt_wf_finish_moments) and the variance of
each pixel's mean resolved from them (rt_resolve_variance).

The moments are exact: every test compares them bit for bit with the squares of the same samples rendered one sample
per launch (samples=(s, s+1)), or with the FP64 oracle, and checks that the first moments (accum) and the counters do
not change when the moments are asked for."""
import ctypes as C

import numpy as np
import pytest

from conftest import gate, load_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def nat(rt):
    from ray_tracer_v1_b200 import _native
    return _native


def _ft(nat, prec):
    return np.float64 if prec == nat.F64 else np.float32


def render(nat, sc, p, prec, moments):
    """One launch -> (accum [H,W,4], stats u64[8], moments [H,W,4] float64 or None)."""
    acc = nat.DeviceBuffer((p.H, p.W, 4), _ft(nat, prec))
    st = nat.DeviceBuffer(8, np.uint64)
    mom = nat.DeviceBuffer((p.H, p.W, 4), np.float64) if moments else None
    sc.render_path(p, acc, prec, stats=st, moments=mom)
    return acc.download(), st.download(), (mom.download() if moments else None)


def per_sample_squares(nat, sc, args, spp, prec, **kw):
    """sum over s of (colour of sample s)^2, each sample rendered alone; integer-valued, so exact in float64."""
    q = 0.0
    for s in range(spp):
        acc, _, _ = render(nat, sc, sc.path_params(*args, samples=(s, s + 1), **kw), prec, False)
        q = q + acc[..., :3].astype(np.float64) ** 2
    return q


def check_exact(nat, sc, args, spp, prec, **kw):
    """moments == per-sample squares bit for bit, count == spp; accum and stats identical with and without moments."""
    p = sc.path_params(*args, **kw)
    acc_m, st_m, mom = render(nat, sc, p, prec, True)
    acc, st, _ = render(nat, sc, p, prec, False)
    assert np.array_equal(acc_m, acc) and np.array_equal(st_m, st)
    assert np.all(mom[..., 3] == spp)
    q = per_sample_squares(nat, sc, args, spp, prec, **{k: v for k, v in kw.items() if k != "samples"})
    assert np.array_equal(mom[..., :3], q)
    assert mom[..., :3].max() > 0
    return acc, mom


PRECISIONS = ["F32", "F64"]


@pytest.mark.parametrize("precision", PRECISIONS)
def test_moments_exact_complex_schedules_and_ksplit(nat, precision):
    """The complex golden scene (the parameter-block kernel, kMode 3, in FP32): golden size, both diagnostic schedule
    bits and every sample split, each against the squares of its samples rendered one at a time."""
    prec = getattr(nat, precision)
    z, fs = load_golden("path_complex_48x27")
    sc = nat.DeviceScene(fs)
    spp = 8
    args = (z["cam"], int(z["W"]), int(z["H"]), spp, int(z["max_bounces"]), float(z["mirror_threshold"]))
    check_exact(nat, sc, args, spp, prec, seed=3)
    for schedule in (2, 4):
        check_exact(nat, sc, args, spp, prec, seed=3, schedule=schedule)
    for ksplit in (0, 1, 2, 8, 32, -1):
        check_exact(nat, sc, args, spp, prec, seed=5, ksplit=ksplit)
    sc.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_moments_exact_hierarchy_and_global_memory(nat, precision):
    """The chandelier with the LBVH forced (shared-memory scene + hierarchy) and a 2000-sphere scene (global-memory
    scene + hierarchy)."""
    from ray_tracer_v1_b200 import scenes
    prec = getattr(nat, precision)
    z, fs = load_golden("path_chandelier_48x27")
    sc = nat.DeviceScene(fs)
    sc.build_lbvh()
    assert sc.has_lbvh
    spp = 6
    check_exact(nat, sc, (z["cam"], 64, 36, spp, int(z["max_bounces"]), float(z["mirror_threshold"])), spp, prec, seed=7)
    sc.close()
    sc = nat.DeviceScene(scenes.build_many_spheres_flat(2000, seed=2, emissive_fraction=0.05))
    sc.build_lbvh()
    check_exact(nat, sc, ((0.0, 2.0, 0.0), 64, 36, 4, 4, 0.0), 4, prec, seed=9)
    sc.close()


def test_moments_exact_with_the_fold_table(nat):
    """A launch of 4 M pixel-samples folds through the per-CTA byte table (FP32 kMode 3); its moments equal those of the
    same samples rendered one at a time, which fold through the double product."""
    z, fs = load_golden("path_complex_48x27")
    sc = nat.DeviceScene(fs)
    spp = 16
    check_exact(nat, sc, (z["cam"], 512, 512, spp, 5, float(z["mirror_threshold"])), spp, nat.F32, seed=3)
    sc.close()


@pytest.mark.parametrize("name", ["path_complex_48x27", "path_chandelier_48x27"])
def test_moments_fp64_equal_the_oracle(nat, orc, name):
    z, fs = load_golden(name)
    W, H, spp = int(z["W"]), int(z["H"]), 4
    depth, thr = int(z["max_bounces"]), float(z["mirror_threshold"])
    q = 0.0
    for s in range(spp):
        sums, _ = orc.render_path(fs, z["cam"], W, H, spp, depth, thr, seed=13, samples=(s, s + 1))
        q = q + sums ** 2
    sc = nat.DeviceScene(fs)
    _, _, mom = render(nat, sc, sc.path_params(z["cam"], W, H, spp, depth, thr, seed=13), nat.F64, True)
    assert np.array_equal(mom[..., :3], q) and np.all(mom[..., 3] == spp)
    sc.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_moment_shards_compose(nat, precision):
    """Row bands x sample ranges with accumulate give exactly the whole-frame moments (and sums)."""
    prec = getattr(nat, precision)
    z, fs = load_golden("path_complex_48x27")
    W, H, spp = int(z["W"]), int(z["H"]), 6
    sc = nat.DeviceScene(fs)
    args = (z["cam"], W, H, spp, int(z["max_bounces"]), float(z["mirror_threshold"]))
    acc_w, _, mom_w = render(nat, sc, sc.path_params(*args, seed=3), prec, True)
    acc = nat.DeviceBuffer((H, W, 4), _ft(nat, prec))
    mom = nat.DeviceBuffer((H, W, 4), np.float64)
    for rows in ((0, 11), (11, H)):
        for k, smp in enumerate(((0, 2), (2, 3), (3, spp))):
            sc.render_path(sc.path_params(*args, seed=3, rows=rows, samples=smp, accumulate=k > 0), acc, prec, moments=mom)
    assert np.array_equal(acc.download(), acc_w) and np.array_equal(mom.download(), mom_w)
    sc.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_moments_of_the_double_fold(nat, precision):
    """Non-integer colours take the double-division fold: the squares are summed in double, to 1e-12 relative."""
    prec = getattr(nat, precision)
    z, fs = load_golden("path_complex_48x27")
    fs.colour = fs.colour + 0.37
    fs.l_colour = fs.l_colour + 0.37
    W, H, spp = 64, 36, 5
    sc = nat.DeviceScene(fs)
    args = (z["cam"], W, H, spp, 5, 0.9)
    acc_m, st_m, mom = render(nat, sc, sc.path_params(*args, seed=4), prec, True)
    acc, st, _ = render(nat, sc, sc.path_params(*args, seed=4), prec, False)
    assert np.array_equal(acc_m, acc) and np.array_equal(st_m, st)
    q = 0.0
    for s in range(spp):
        a1, _, m1 = render(nat, sc, sc.path_params(*args, seed=4, samples=(s, s + 1)), prec, True)
        if prec == nat.F64:
            assert np.array_equal(m1[..., :3], a1[..., :3] ** 2)          # one sample: its square, c * c in double
        else:                                                             # (accum holds the colour rounded to float)
            np.testing.assert_allclose(m1[..., :3], a1[..., :3].astype(np.float64) ** 2, rtol=2.5e-7)
        q = q + m1[..., :3]
    assert (q != np.rint(q)).any()
    np.testing.assert_allclose(mom[..., :3], q, rtol=1e-12, atol=0)
    assert np.all(mom[..., 3] == spp)
    sc.close()


# ------------------------------------------------------------------ wavefront
def wavefront_moments(nat, sc, p, prec, policy=None, prob=0.0):
    """The rt_wf_* loop of renderers.render_path_wavefront, finished through rt_wf_finish_moments -> (accum, moments)."""
    import torch
    L, dev = nat.lib(), torch.device("cuda", sc.device)
    P = p.W * p.H * (p.s1 - p.s0)
    wf = C.c_void_p()
    nat.check(L.rt_wf_create(sc.handle, prec, P, max(1, p.max_bounces), C.byref(wf)))
    try:
        acc = torch.zeros((p.H, p.W, 4), dtype=torch.float64 if prec == nat.F64 else torch.float32, device=dev)
        mom = torch.zeros((p.H, p.W, 4), dtype=torch.float64, device=dev)
        obs = torch.zeros((P, 22), dtype=torch.float32, device=dev)
        need = torch.zeros(P, dtype=torch.uint8, device=dev)
        actions = torch.zeros((P, 2), dtype=torch.float32, device=dev)
        live = torch.zeros(1, dtype=torch.int32, device=dev)
        nat.check(L.rt_wf_begin(wf, C.byref(p), prob, None, None))
        for _ in range(p.max_bounces):
            nat.check(L.rt_wf_trace(wf, obs.data_ptr(), need.data_ptr(), None, None))
            if prob > 0.0:
                idx = need.nonzero(as_tuple=True)[0]
                if idx.numel():
                    actions[idx] = policy(obs[idx]).to(dtype=torch.float32).reshape(-1, 2)
            live.zero_()
            nat.check(L.rt_wf_bounce(wf, need.data_ptr(), actions.data_ptr(), None, live.data_ptr(), None))
            if int(live.item()) == 0:
                break
        assert L.rt_wf_finish_moments(wf, acc.data_ptr(), None, None) != 0          # NULL moments: rejected
        nat.check(L.rt_wf_finish_moments(wf, acc.data_ptr(), mom.data_ptr(), None))
        torch.cuda.synchronize(dev)
        return acc.cpu().numpy(), mom.cpu().numpy()
    finally:
        nat.load_symbols().rt_wf_destroy(wf)


def _torch_policy(obs):                                  # torch twin of test_oracle_golden.fb_test_policy
    import torch
    a0 = (obs[:, 6] * 0.5 + obs[:, 7] * 0.25 - 0.125).clamp(-1, 1)
    a1 = (obs[:, 8] * 0.5 + obs[:, 3] * 0.25 + obs[:, 16] * 0.5).clamp(-1, 1)
    return torch.stack([a0, a1], dim=1)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_wavefront_moments_equal_the_path_kernel(nat, precision):
    """fb_usage_prob = 0: the wavefront's moments equal the fused path kernel's bit for bit."""
    prec = getattr(nat, precision)
    z, fs = load_golden("path_fb_complex_40x24")
    sc = nat.DeviceScene(fs)
    p = sc.path_params(z["cam"], int(z["W"]), int(z["H"]), 4, int(z["max_bounces"]), float(z["mirror_threshold"]), seed=8)
    acc_k, _, mom_k = render(nat, sc, p, prec, True)
    acc_w, mom_w = wavefront_moments(nat, sc, p, prec)
    assert np.array_equal(acc_w, acc_k) and np.array_equal(mom_w, mom_k)
    sc.close()


def test_wavefront_moments_with_a_policy_equal_the_oracle(nat, orc):
    """With the stand-in policy the FP64 moments equal the squares of the oracle's WorkingFBRenderer samples."""
    from test_oracle_golden import fb_test_policy
    z, fs = load_golden("path_fb_complex_40x24")
    W, H, spp, depth, thr = int(z["W"]), int(z["H"]), 3, int(z["max_bounces"]), float(z["mirror_threshold"])
    q = 0.0
    for s in range(spp):
        sums, st = orc.render_path_fb(fs, z["cam"], W, H, spp, depth, thr, fb_test_policy, 1.0, 17, samples=(s, s + 1))
        assert st["fb_used"] > 0
        q = q + sums ** 2
    sc = nat.DeviceScene(fs)
    _, mom = wavefront_moments(nat, sc, sc.path_params(z["cam"], W, H, spp, depth, thr, seed=17), nat.F64, _torch_policy, 1.0)
    assert np.array_equal(mom[..., :3], q) and np.all(mom[..., 3] == spp)
    sc.close()


# ------------------------------------------------------------------ resolve
def numpy_variance(acc, mom):
    S, Q, n = acc[..., :3].astype(np.float64), mom[..., :3], mom[..., 3:4]
    with np.errstate(divide="ignore", invalid="ignore"):
        v = (Q - S * S / n) / (n * (n - 1))
    return np.where(n >= 2, v, 0.0)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_resolve_variance(nat, precision):
    prec = getattr(nat, precision)
    z, fs = load_golden("path_complex_48x27")
    W, H = int(z["W"]), int(z["H"])
    sc = nat.DeviceScene(fs)
    for spp in (7, 1):
        p = sc.path_params(z["cam"], W, H, spp, int(z["max_bounces"]), float(z["mirror_threshold"]), seed=6)
        acc = nat.DeviceBuffer((H, W, 4), _ft(nat, prec))
        mom = nat.DeviceBuffer((H, W, 4), np.float64)
        sc.render_path(p, acc, prec, moments=mom)
        var = nat.DeviceBuffer((H, W, 3), np.float32)
        var.fill(0xFF)                                               # NaN: rows outside [y0, y1) stay untouched
        sc.resolve_variance(acc, mom, W, H, var, prec, rows=(5, 20))
        v = var.download()
        ref = numpy_variance(acc.download(), mom.download())
        assert np.isnan(v[:5]).all() and np.isnan(v[20:]).all()
        np.testing.assert_allclose(v[5:20], ref[5:20], rtol=1e-6, atol=1e-6 * max(1.0, ref.max()))
        if spp == 1:
            assert not v[5:20].any()
        else:
            assert v[5:20].max() > 0 and v[5:20].min() >= 0
    L = nat.lib()
    for rows in ((-1, 5), (5, H + 1), (6, 5)):
        with pytest.raises(nat.NativeLibraryError, match="row band"):
            sc.resolve_variance(acc, mom, W, H, var, prec, rows=rows)
    assert L.rt_resolve_variance(0, prec, None, mom.ptr, W, H, 0, H, var.ptr, None) != 0
    assert L.rt_resolve_variance(0, prec, acc.ptr, None, W, H, 0, H, var.ptr, None) != 0
    assert L.rt_resolve_variance(0, prec, acc.ptr, mom.ptr, W, H, 0, H, None, None) != 0
    assert L.rt_resolve_variance(0, 7, acc.ptr, mom.ptr, W, H, 0, H, var.ptr, None) != 0
    p = sc.path_params(z["cam"], W, H, 2, 5, 0.9)
    assert L.rt_render_path_moments(sc.handle, prec, C.byref(p), acc.ptr, None, None, None) != 0
    assert L.rt_render_path_moments(sc.handle, prec, C.byref(p), None, mom.ptr, None, None) != 0
    sc.close()


# ------------------------------------------------------------------ renderers
def test_renderers_track_variance(rt, nat):
    """track_variance leaves the image and the counters unchanged, also at a size that takes the banded read-back, and
    the banded variance equals the one-launch variance."""
    from ray_tracer_v1_b200 import scenes, renderers
    spec = scenes.build_complex()
    for (W, H, spp) in ((160, 90, 8), (1920, 1080, 16)):
        r = rt.ComplexTraditionalRenderer(precision="f32", seed=5)
        r.scene = spec.spheres
        r.light_sources = [s for s in spec.spheres if s.material.emitive]
        r.camera_position = rt.Vector(*spec.camera)
        r.reuse_output = False
        img = r.render(W, H, spp, 5)
        st = dict(r.stats)
        assert not hasattr(r, "variance")
        r.track_variance = True
        img_v = r.render(W, H, spp, 5)
        assert np.array_equal(img, img_v)
        assert all(st[k] == r.stats[k] for k in ("total_rays", "total_intersections", "light_hits", "small_light_hits"))
        assert r.variance.shape == (H, W, 3) and r.variance.dtype == np.float32
        assert r._ctx.launches == (6 if W == 1920 else 3)                 # two bands of render + resolve + variance
        fs = r.flat_scene()
        img_f, _, _, var_f = renderers.render_path(fs, spec.camera, W, H, spp, 5, 0.9, seed=5, return_raw=True, variance=True)
        assert np.array_equal(img_f, img) and np.array_equal(var_f, r.variance)
    # the FB renderer on both branches
    z, fs = load_golden("path_fb_complex_40x24")
    for agent in (False, True):
        f = rt.WorkingFBRenderer(camera_position=rt.Vector(*spec.camera), precision="f64", seed=3)
        f.scene, f.light_sources = spec.spheres, [s for s in spec.spheres if s.material.emitive]
        if agent:
            f.fb_agent = type("Agent", (), {"choose_directions": staticmethod(_torch_policy)})()
            f.fb_loaded, f.fb_usage_prob = True, 0.5
        f.reuse_output = False
        a = f.render(40, 24, 4, 5)
        f.track_variance = True
        b = f.render(40, 24, 4, 5)
        assert np.array_equal(a, b) and f.variance.shape == (24, 40, 3) and f.variance.max() > 0


def test_variance_predicts_the_seed_to_seed_error(nat):
    """The estimate predicts the error: for two seeds of the same frame, E[(m1 - m2)^2 / 2] is the variance of one
    pixel mean, so the frame means of (m1 - m2)^2 / 2 and of the predicted variances agree."""
    from ray_tracer_v1_b200 import scenes, flatten_scene
    spec = scenes.build_complex()
    sc = nat.DeviceScene(flatten_scene(spec.spheres, background_colour=spec.background))
    W, H, spp = 160, 90, 16
    means, preds = [], []
    for seed in (1, 2):
        p = sc.path_params(spec.camera, W, H, spp, 5, 0.9, seed=seed)
        acc = nat.DeviceBuffer((H, W, 4), np.float32)
        mom = nat.DeviceBuffer((H, W, 4), np.float64)
        var = nat.DeviceBuffer((H, W, 3), np.float32)
        sc.render_path(p, acc, nat.F32, moments=mom)
        sc.resolve_variance(acc, mom, W, H, var, nat.F32)
        a = acc.download()
        means.append(a[..., :3].astype(np.float64) / spp)
        preds.append(var.download().astype(np.float64))
    observed = float(np.mean((means[0] - means[1]) ** 2 / 2))
    predicted = float(np.mean((preds[0] + preds[1]) / 2))
    print(f"seed-to-seed: observed {observed:.4f} predicted {predicted:.4f} levels^2")
    gate("variance estimate vs seed-to-seed error, |observed / predicted - 1|", abs(observed / predicted - 1), 0.06)
    sc.close()
