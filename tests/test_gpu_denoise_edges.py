"""Both non-local-means filters (rt_denoise, rt_denoise_features; DESIGN §4.8c, §4.8d) on synthetic frames that put the
cases the formulas single out where the 16x16 tiles of the kernels meet: zero variance on both pixels of a pair, a step
between two flat regions, colours above 255, flat features with tau = 0, frames of one pixel in width or height, every
(radius, patch_radius) class on both sides of the 48 KB shared-memory opt-in, and the parameter limits the ABI accepts.

Besides the float64 references (same lattice criterion as test_gpu_denoise.py), three properties need no tolerance:
- range: the output is a convex combination of the window's means, so lattice(min u) <= image <= lattice(max u) over each
  pixel's clamped (2r+1)^2 window;
- locality: a pixel changed outside the (r + f) box of an output pixel (max(r, 1) for features) leaves it bit-identical;
- precision identity: on integer sums the F32 and F64 accum kernels compute the same FP32 arithmetic, so the same bits.
"""
import numpy as np
import pytest
from scipy import ndimage

from conftest import load_golden
from test_gpu_denoise import _ft, check_against_reference, denoise, lattice, nlm_reference
from test_gpu_features import denoise_features, nlm_features_reference

pytestmark = pytest.mark.gpu

FLAT, STEP = (17.0, 200.0, 300.0), (60.0, 120.0, 260.0)     # zero-variance colours: 300 saturates the lattice
TILE = 16


@pytest.fixture(scope="module")
def nat(rt):
    from ray_tracer_v1_b200 import _native
    return _native


@pytest.fixture(scope="module")
def sc(nat):
    _, fs = load_golden("path_complex_48x27")
    s = nat.DeviceScene(fs)          # rt_denoise takes no scene; the handle only carries the device
    yield s
    s.close()


def synthetic(H, W, seed, integer=True):
    """-> (accum [H,W,4] float64, var [H,W,3] float32): noisy texture with per-pixel counts n in [1, 64] and a block
    at n = 4096 (variance 0 where n = 1), and a zero-variance rectangle across the tile seams whose left part has colour
    FLAT and right part STEP.  integer = False adds a fraction to every sum (FP64 accum only)."""
    rng = np.random.default_rng(seed)
    n = rng.integers(1, 65, (H, W)).astype(np.float64)
    n[2 * H // 3:, :W // 3] = 4096
    y, x = np.mgrid[0:H, 0:W]
    mean = 40.0 + 90.0 * (1 + np.sin(x / 5.0)[..., None] * np.cos(y / 7.0)[..., None] * np.array([1.0, -0.7, 0.4]))
    sigma = rng.uniform(2.0, 40.0, (H, W, 3))
    S = np.clip(np.rint((mean + rng.normal(0.0, 1.0, (H, W, 3)) * sigma / np.sqrt(n[..., None])) * n[..., None]), 0, None)
    var = (sigma ** 2 / n[..., None] * rng.uniform(0.5, 1.5, (H, W, 3))).astype(np.float32)
    var[n == 1] = 0
    y0, y1, x0, x1 = H // 5, H - H // 5, W // 5, W - W // 5
    xm = (x0 + x1) // 2
    for (xa, xb), c in (((x0, xm), FLAT), ((xm, x1), STEP)):
        S[y0:y1, xa:xb] = np.array(c) * n[y0:y1, xa:xb, None]
        var[y0:y1, xa:xb] = 0
    if not integer:
        S = S + rng.random(S.shape)
    assert S.max() < 2 ** 24
    return np.concatenate([S, n[..., None]], axis=-1), var


def synthetic_features(H, W, seed):
    """-> (albedo, normal, depth, fvar) float32: noisy hits, misses (all zero) in the top rows, and over the colour
    rectangle of ``synthetic`` a flat zero-variance patch with a depth step across its middle."""
    rng = np.random.default_rng(seed + 1000)
    albedo = rng.uniform(0.1, 0.9, (H, W, 3))
    normal = rng.normal(size=(H, W, 3))
    normal /= np.linalg.norm(normal, axis=-1, keepdims=True)
    depth = rng.uniform(2.0, 8.0, (H, W))
    fvar = rng.uniform(0.0, 1e-2, (H, W, 3))
    miss = slice(0, max(1, H // 6))
    for a in (albedo, normal, depth, fvar):
        a[miss] = 0
    y0, y1, x0, x1 = H // 5, H - H // 5, W // 5, W - W // 5
    ym = (y0 + y1) // 2
    albedo[y0:y1, x0:x1], normal[y0:y1, x0:x1], fvar[y0:y1, x0:x1] = (0.5, 0.6, 0.7), (0.0, 0.0, 1.0), 0
    depth[y0:ym, x0:x1], depth[ym:y1, x0:x1] = 3.0, 5.0
    return [a.astype(np.float32) for a in (albedo, normal, depth, fvar)]


def means(acc):
    """u = float32(S / n) as the kernels stage it, in float64."""
    return (acc[..., :3].astype(np.float64) / acc[..., 3:4]).astype(np.float32).astype(np.float64)


def check_range(img, acc, r):
    """lattice(min u) <= image <= lattice(max u) over each pixel's clamped (2r+1)^2 window, per channel."""
    u = means(acc)
    lo = ndimage.minimum_filter(u, size=(2 * r + 1, 2 * r + 1, 1), mode="nearest")
    hi = ndimage.maximum_filter(u, size=(2 * r + 1, 2 * r + 1, 1), mode="nearest")
    below, above = img < lattice(lo), img > lattice(hi)
    assert not below.any() and not above.any(), (np.argwhere(below)[:5], np.argwhere(above)[:5])


def run(nat, sc, acc, var, feats, prec, **params):
    acc = acc.astype(_ft(nat, prec))
    if feats is None:
        return denoise(nat, sc, acc, var, prec, **params)
    return denoise_features(nat, sc, acc, var, feats, prec, **params)


def reference(acc, var, feats, r, f, **params):
    if feats is None:
        return nlm_reference(acc, var, r, f, **params)
    return nlm_features_reference(acc, var, feats, r, f, **params)


def check_all(nat, sc, acc, var, feats, r, f, **params):
    """Both accum precisions against the reference and the range; the same bits from both on integer sums.  The flat
    regions hold integer means, so only a quarter of the values must lie far from an integer (none of a 1 x 1 frame's)."""
    u_hat = reference(acc, var, feats, r, f, **params)
    imgs = [run(nat, sc, acc, var, feats, getattr(nat, p), radius=r, patch_radius=f, **params) for p in ("F32", "F64")]
    for img in imgs:
        check_against_reference(img, u_hat, u_hat.size // 4)
        check_range(img, acc, r)
    assert imgs[0].tobytes() == imgs[1].tobytes()
    return u_hat, imgs[0]


def denoise_smem(r, f, features):
    """Dynamic shared memory of one CTA (rt_denoise.cu): 6 planes of the colour halo, the patch region's deltas and row
    sums, and with features 10 planes of the (16 + 2r)^2 feature halo."""
    L, R, LF = TILE + 2 * (r + f), TILE + 2 * f, TILE + 2 * r
    return 4 * (6 * L * L + R * R + R * TILE + (10 * LF * LF if features else 0))


GRID = [(r, f) for r in (0, 1, 4, 10, 11, 15) for f in (0, 1, 3, 5)]


def test_grid_straddles_the_shared_memory_opt_in():
    assert denoise_smem(10, 3, False) == 45680 and denoise_smem(15, 5, False) == 79632
    assert denoise_smem(10, 3, True) == 97520 and denoise_smem(15, 5, True) == 164272
    for feats in (False, True):
        sizes = [denoise_smem(r, f, feats) for r, f in GRID]
        assert min(sizes) <= 48 * 1024 < max(sizes), feats
        assert max(sizes) <= 227 * 1024


@pytest.mark.parametrize("kernel", ["colour", "features"])
def test_radius_patch_grid(nat, sc, kernel):
    """47 x 35 (3 x 3 tiles, the last partial in both directions), every (r, f) of GRID."""
    H, W = 35, 47
    acc, var = synthetic(H, W, seed=1)
    feats = synthetic_features(H, W, seed=1) if kernel == "features" else None
    for r, f in GRID:
        check_all(nat, sc, acc, var, feats, r, f)


SHAPES = [(1, 1), (1, 40), (40, 1), (16, 16), (17, 17), (15, 33), (33, 15), (35, 47), (113, 200)]


@pytest.mark.parametrize("shape", SHAPES, ids=[f"{w}x{h}" for h, w in SHAPES])
@pytest.mark.parametrize("kernel", ["colour", "features"])
def test_shapes(nat, sc, kernel, shape):
    """Frames of one pixel, one row or one column (the clamped gradient reads fold onto the pixel itself), one tile, one
    tile and one pixel, partial tiles in x or y, and 13 x 8 tiles; FP64 accum also on non-integer sums."""
    H, W = shape
    acc, var = synthetic(H, W, seed=2)
    feats = synthetic_features(H, W, seed=2) if kernel == "features" else None
    for r, f in ((10, 3), (1, 1)):
        check_all(nat, sc, acc, var, feats, r, f)
    acc, var = synthetic(H, W, seed=3, integer=False)
    img = run(nat, sc, acc, var, feats, nat.F64)
    check_against_reference(img, reference(acc, var, feats, 10, 3), acc[..., :3].size // 4)
    check_range(img, acc, 10)


@pytest.mark.parametrize("k", [1e-6, 0.45, 1e3, 1e19, 1e20, 3e38])
def test_colour_k_limits(nat, sc, k):
    """Every k the ABI accepts.  Above sqrt(FLT_MAX) ~ 1.84e19, k^2 is clamped: a pair of zero-variance pixels still
    gets delta = du^2 / eps, so no weight crosses the step between the two flat regions, while every noisy pair gets
    delta ~ 0."""
    acc, var = synthetic(35, 47, seed=4)
    check_all(nat, sc, acc, var, None, 10, 3, k=k)


@pytest.mark.parametrize("tau", [0.0, 1e-3, 1e6])
@pytest.mark.parametrize("k_f", [1e-3, 1.2, 1e18, 1e20])
def test_features_k_f_tau_limits(nat, sc, k_f, tau):
    """Every (k_f, tau) corner; at tau = 0 the flat patch's denominators are 0, so a pair across its depth step gets
    Phi = +inf and weight 0 however large k_f is."""
    H, W = 35, 47
    acc, var = synthetic(H, W, seed=5)
    feats = synthetic_features(H, W, seed=5)
    check_all(nat, sc, acc, var, feats, 10, 3, k=1.0, k_f=k_f, tau=tau)


def test_features_flat_tau0_is_colour_only(nat, sc):
    """Flat zero-variance features with tau = 0: every Phi is 0 / 0, which the filter ignores, so the image is rt_denoise's
    at the same k, bit for bit, at any k_f."""
    H, W = 35, 47
    acc, var = synthetic(H, W, seed=6)
    flat = [np.full((H, W, 3), 0.5, np.float32), np.full((H, W, 3), (0.0, 0.6, 0.8), np.float32),
            np.full((H, W), 4.0, np.float32), np.zeros((H, W, 3), np.float32)]
    for prec in (nat.F32, nat.F64):
        for k_f in (1.2, 1e20):
            for r, f in ((10, 3), (4, 0)):
                plain = run(nat, sc, acc, var, None, prec, radius=r, patch_radius=f, k=1.0)
                guided = run(nat, sc, acc, var, flat, prec, radius=r, patch_radius=f, k=1.0, k_f=k_f, tau=0.0)
                assert guided.tobytes() == plain.tobytes(), (prec, k_f, r, f)


def test_features_depth_step_tau0(nat, sc):
    """Flat zero-variance features with a depth step across the frame, tau = 0: no weight crosses the step (the
    reference's num / 0 = inf), at k_f = 1.2 and at k_f = 1e20, whose square overflows FP32."""
    H, W = 35, 47
    acc, var = synthetic(H, W, seed=7)
    feats = [np.full((H, W, 3), 0.5, np.float32), np.full((H, W, 3), (0.0, 0.6, 0.8), np.float32),
             np.where(np.arange(H)[:, None] < 18, 3.0, 5.0).astype(np.float32) * np.ones((1, W), np.float32),
             np.zeros((H, W, 3), np.float32)]
    for k_f in (1.2, 1e20):
        u_hat, _ = check_all(nat, sc, acc, var, feats, 10, 3, k=1.0, k_f=k_f, tau=0.0)
        assert np.abs(u_hat - nlm_reference(acc, var, 10, 3, k=1.0)).max() > 1.0     # the step changes the image


@pytest.mark.parametrize("kernel", ["colour", "features"])
def test_locality(nat, sc, kernel):
    """A zero-variance spike (a colour, or a feature vector) on tile seams, at the frame's corners and where the box
    ends one pixel before a tile: only output pixels within r + f (features: max(r, 1)) of it change, every other
    pixel keeps its bits."""
    H, W = 35, 47
    acc, var = synthetic(H, W, seed=8)
    feats = synthetic_features(H, W, seed=8) if kernel == "features" else None
    y, x = np.mgrid[0:H, 0:W]
    for r, f in ((4, 1), (10, 3), (0, 2)):
        base = run(nat, sc, acc, var, feats, nat.F32, radius=r, patch_radius=f)
        reach = (r + f) if feats is None else max(r, 1)
        # the last two: the box ends on the last column (row) of a tile, and starts on the first one of a tile
        for sy, sx in ((15, 16), (16, 15), (0, 0), (H - 1, W - 1), (0, W - 1), (H - 1, 0),
                       (max(0, 15 - reach), 31 - reach), (min(H - 1, 16 + reach), 16 + reach)):
            a, v = acc.copy(), var.copy()
            fs = None if feats is None else [g.copy() for g in feats]
            if fs is None:
                a[sy, sx, :3] = 250.0 * a[sy, sx, 3]
                v[sy, sx] = 0
            else:
                fs[0][sy, sx], fs[1][sy, sx], fs[2][sy, sx], fs[3][sy, sx] = (1.0, 0.0, 0.0), (1.0, 0.0, 0.0), 40.0, 0
            img = run(nat, sc, a, v, fs, nat.F32, radius=r, patch_radius=f)
            outside = (np.abs(y - sy) > reach) | (np.abs(x - sx) > reach)
            assert img[outside].tobytes() == base[outside].tobytes(), (r, f, sy, sx)
            if fs is None:
                assert not np.array_equal(img[sy, sx], base[sy, sx])


def test_range_rendered_frame(nat, sc):
    """The range property on the complex scene, 160 x 90, 8 spp, both filters at their defaults."""
    from test_gpu_features import uniform
    z, fs = load_golden("path_complex_48x27")
    scene = nat.DeviceScene(fs)
    acc, var, feats = uniform(nat, scene, (z["cam"], 160, 90, int(z["max_bounces"]), float(z["mirror_threshold"])), 8,
                              nat.F32, 6)
    check_range(run(nat, sc, acc, var, None, nat.F32), acc, 10)
    check_range(run(nat, sc, acc, var, feats, nat.F32), acc, 10)
    scene.close()
