"""Render entry points of the reference, backed by the CUDA kernels.

* ``TraditionalRenderer``        FB/fb_vs_traditional_chandelier.py:393-554 (Algorithm B; ``mirror_threshold`` 0, the
                                 chandelier flavour) and ``ComplexTraditionalRenderer`` FB/fb_vs_traditional_complex.py:262-422
                                 (threshold 0.9).  Same attribute-injection style (``.scene .light_sources .small_lights
                                 .camera_position``), same ``render(width, height, samples_per_pixel, max_bounces)`` and
                                 ``stats`` keys.
* ``CustomSceneExperiment``      RL/output5.py:264 -- ``render_true_original(scene, path)`` (:416-533) and
                                 ``render_custom_scene(scene, 'traditional', path)`` (:1420-1525) (Algorithm A).
* ``SimplifiedFBRenderer``       FB/output6.py:85-654 in traditional mode (``fb_usage_prob == 0``, the value the reference
                                 ships): ``render_original_style(width, height, output_path)`` and ``trace_ray_simple(ray)``.
* ``render_whitted`` / ``render_path``  the plain functions underneath (flat scene in, numpy image out).

Every call re-flattens the scene (the reference's scenes are mutable lists) and uploads it; frames are rendered and
resolved on the GPU and only the float32 image (plus, on request, the raw sums) comes back to the host.
"""
import ctypes as C
import time
from pathlib import Path

import numpy as np

from . import _native as nat
from .frames import FrameContext
from .colour import Colour
from .light import GlobalLight, PointLight
from .material import Material
from .object import Sphere
from .scene import flatten_scene
from .scenes import custom_scene_grid, notebook_grid
from .vector import Vector

__all__ = ["render_whitted", "render_path", "TraditionalRenderer", "ComplexTraditionalRenderer",
           "CustomSceneExperiment", "SimplifiedFBRenderer", "WorkingFBRenderer", "render_path_wavefront", "save_png"]

_PREC = {"f32": nat.F32, "fp32": nat.F32, "float32": nat.F32, nat.F32: nat.F32,
         "f64": nat.F64, "fp64": nat.F64, "float64": nat.F64, "double": nat.F64}


def _precision(p):
    try:
        return _PREC[p]
    except KeyError:
        raise ValueError(f"unknown precision {p!r}") from None


def _xyz(v):
    return (float(v.x), float(v.y), float(v.z)) if hasattr(v, "x") else tuple(float(c) for c in v)


def save_png(image, path):
    """Raw framebuffer -> 8-bit PNG (the reference saves a matplotlib figure; this writes the pixels themselves)."""
    from PIL import Image
    Image.fromarray((np.clip(image, 0, 1) * 255.0 + 0.5).astype(np.uint8)).save(str(path))


def render_whitted(fs, camera, X, Y, spp=1, max_bounces=1, shadow_max_bounces=0, miss=None, seed=0, prenorm=False,
                   precision="f32", device=0, return_raw=False, context=None):
    """Algorithm A frame over the direction grid (X[i], Y[j], -1) -> float32 image [H,W,3] (``int(sum/spp)/255``).

    return_raw=True also returns (sums [H,W,4], hit [H,W] int32, stats dict).
    context: a ``FrameContext`` to render through -- its scene handle, HBM buffers, pinned host image and resident
    direction grid are reused from frame to frame (the render entries keep one); None = a throw-away scene handle."""
    if context is not None and not return_raw:
        context.set_scene(fs, skip_unchanged=True)      # the same scene list rendered again: nothing to upload
        view, _ = context.render_whitted(_xyz(camera), X, Y, spp=spp, max_bounces=max_bounces,
                                         shadow_max_bounces=shadow_max_bounces, miss=miss, seed=seed, prenorm=prenorm,
                                         precision=_precision(precision))
        return view.copy()
    sc = nat.DeviceScene(fs, device)
    try:
        p = sc.whitted_params(_xyz(camera), X, Y, spp=spp, max_bounces=max_bounces, shadow_max_bounces=shadow_max_bounces,
                              miss=miss, seed=seed, prenorm=prenorm)
        image, sums, hit, st = sc.render_whitted_host(p, _precision(precision), want_accum=return_raw, want_hit=return_raw)
    finally:
        sc.close()
    if return_raw:
        return image, sums, hit, {"primary_rays": int(st[0]), "queries": int(st[4]), "sphere_tests": int(st[5])}
    return image


def _variance_frame(sc, p, prec, W, H):
    """One path-kernel launch with the second moments -> (image [H,W,3], sums [H,W,4], stats u64[8], variance [H,W,3])."""
    ft = np.float64 if prec == nat.F64 else np.float32
    accum, moments = nat.DeviceBuffer((H, W, 4), ft, sc.device), nat.DeviceBuffer((H, W, 4), np.float64, sc.device)
    stats = nat.DeviceBuffer(8, np.uint64, sc.device)
    image, var = nat.DeviceBuffer((H, W, 3), np.float32, sc.device), nat.DeviceBuffer((H, W, 3), np.float32, sc.device)
    sc.render_path(p, accum, prec, stats=stats, moments=moments)
    sc.resolve(accum, W, H, p.s1 - p.s0, image, prec)
    sc.resolve_variance(accum, moments, W, H, var, prec)
    return image.download(), accum.download(), stats.download(), var.download()


def render_path(fs, camera, width, height, spp, max_bounces, mirror_threshold, seed=0, fov=60.0, precision="f32",
                device=0, lbvh=None, return_raw=False, variance=False):
    """Algorithm B frame -> float32 image [H,W,3] (``sum // spp / 255``).  lbvh: None = build the on-device LBVH when
    the scene has more than 256 spheres, True/False to force.  variance=True appends the float32 [H,W,3] variance of
    each pixel's mean in colour levels^2 (0-255 scale), estimated from the same samples in the same launch."""
    sc = nat.DeviceScene(fs, device)
    try:
        if lbvh or (lbvh is None and sc.n > 256):
            sc.build_lbvh()
        p = sc.path_params(_xyz(camera), width, height, spp, max_bounces, mirror_threshold, seed=seed, fov=fov)
        if variance:
            image, sums, st, var = _variance_frame(sc, p, _precision(precision), int(width), int(height))
        else:
            image, sums, st = sc.render_path_host(p, _precision(precision), want_accum=return_raw)
    finally:
        sc.close()
    stats = {"total_rays": int(st[0]), "total_intersections": int(st[1]), "light_hits": int(st[2]),
             "small_light_hits": int(st[3]), "queries": int(st[4]), "sphere_tests": int(st[5]), "aabb_tests": int(st[6])}
    out = (image, sums, stats) if return_raw else (image, stats)
    return out + (var,) if variance else out


class TraditionalRenderer:
    """Drop-in for the reference's ``TraditionalRenderer`` (chandelier flavour: a sphere mirrors when
    ``material.reflective > 0``, FB/fb_vs_traditional_chandelier.py:481).

    The reference draws jitter and bounce directions from the global ``np.random`` stream; here they come from
    Philox4x32-10 keyed (pixel, sample, bounce) with ``self.seed`` (``None`` = a fresh seed per render), so a render is
    reproducible and independent of how it is sharded."""

    mirror_threshold = 0.0
    reuse_output = True
    # True: render() also sets self.variance, the float32 [H,W,3] variance of each pixel's mean in colour levels^2,
    # estimated from the frame's own samples in the same launch (a view of a pinned ring, like the image)
    track_variance = False
    # adaptive sampling: with a tolerance (colour levels, 0-255 scale) render() treats samples_per_pixel as the maximum,
    # gives every pixel adaptive_min_spp samples and doubles the samples of the pixels whose variance of the mean still
    # exceeds tolerance^2 (FrameContext.render_path_adaptive); it then also sets self.sample_counts, int32 [H,W]
    adaptive_tolerance = None
    adaptive_min_spp = 16
    # True: render() returns the frame filtered by the variance-guided non-local-means filter (rt_denoise, library
    # defaults; DESIGN §4.8c), from the frame's own per-pixel variance; combines with track_variance and adaptive_tolerance
    denoise = False
    # True: render() also sets self.albedo [H,W,3], self.normal [H,W,3] and self.depth [H,W] (float32), the first-hit
    # features of the frame's first FrameContext.FEATURE_SPP samples, and a denoised frame uses the feature-guided filter
    # (rt_denoise_features, library defaults; DESIGN §4.8d); combines with track_variance and adaptive_tolerance
    track_features = False

    def __init__(self, device=0, precision="f32", seed=None):
        self.scene = []
        self.camera_position = Vector(0, 2, 0)
        self.camera_angle = None  # unused, as in the reference
        self.global_lights = []
        self.point_lights = []
        self.light_sources = []
        self.small_lights = []
        self.stats = {'total_rays': 0, 'total_intersections': 0, 'light_hits': 0, 'small_light_hits': 0,
                      'render_time': 0, 'rays_per_second': 0}
        self.device, self.precision, self.seed = device, precision, seed
        self._renders = 0
        self._ctx = None            # persistent FrameContext (HBM buffers + pinned host image), created on first render

    def set_render_settings(self, width=200, height=150, max_bounces=3, samples_per_pixel=16):
        self.image_width = width
        self.image_height = height
        self.max_bounces = max_bounces
        self.samples_per_pixel = samples_per_pixel
        self.aspect_ratio = width / height
        self.fov = 60

    def flat_scene(self):
        return flatten_scene(self.scene, background_colour=Colour(2, 2, 5), light_sources=self.light_sources,
                             small_lights=self.small_lights)

    def trace_ray_traditional(self, ray, bounce_count=0, pixel=0, sample=0):
        """One call of the reference's recursive tracer (FB/fb_vs_traditional_chandelier.py:431-521) -> ``Colour``: nearest
        hit, unshadowed direct light from every light sphere, one mirror / cosine-weighted bounce per level, integer
        truncation at every level -- on the GPU, a batch of one through ``rt_trace_paths`` (the frame kernel, fed an
        explicit ray).  The reference draws its bounce directions from global ``np.random``; here they come from the
        Philox stream of (``self.seed``; pixel, sample), the one ``render`` uses for that pixel sample, so
        ``trace_ray_traditional(generate_camera_ray(x, y, .5 + jx, .5 + jy), pixel=y * W + x, sample=s)`` is exactly that
        sample of the frame.  Updates ``stats`` like the reference's counters."""
        seed = self.seed if self.seed is not None else 0
        if self._ctx is None:
            self._ctx = FrameContext(self.device)
        sc = self._ctx.set_scene(self.flat_scene())
        o, d = _xyz(ray.origin), _xyz(ray.D)
        sums, st = sc.trace_paths([[*o, *d]], self.max_bounces, self.mirror_threshold, bounce_count=bounce_count, seed=seed,
                                  ray_ids=[int(pixel)], samples=(int(sample), int(sample) + 1), precision=_precision(self.precision))
        for i, k in enumerate(('total_rays', 'total_intersections', 'light_hits', 'small_light_hits')):
            self.stats[k] = self.stats.get(k, 0) + int(st[i])
        return Colour(float(sums[0, 0]), float(sums[0, 1]), float(sums[0, 2]))

    def generate_camera_ray(self, x, y, sample_x=0.5, sample_y=0.5):
        """The camera ray of pixel (x, y) at sub-pixel position (sample_x, sample_y) as the reference builds it
        (FB/fb_vs_traditional_chandelier.py:417-429: the aspect ratio enters the x coordinate TWICE) -> ``Ray``.
        ``render`` generates the same rays on the device (``path_camera_ray``); needs ``set_render_settings`` first."""
        from .ray import Ray
        half_height = np.tan(np.radians(self.fov) / 2)
        half_width = half_height * self.aspect_ratio
        ndc_x = (x + sample_x) / self.image_width
        ndc_y = (y + sample_y) / self.image_height
        screen_x = (2 * ndc_x - 1) * self.aspect_ratio * half_width
        screen_y = (1 - 2 * ndc_y) * half_height
        return Ray(self.camera_position, Vector(screen_x, screen_y, -1).normalise())

    def render(self, width=200, height=150, samples_per_pixel=4, max_bounces=3):
        self.set_render_settings(width, height, max_bounces, samples_per_pixel)
        self.stats = {k: 0 for k in self.stats}
        start = time.time()
        seed = self.seed if self.seed is not None else (time.time_ns() ^ (self._renders * 0x9E3779B97F4A7C15)) & (2 ** 64 - 1)
        self._renders += 1
        if self._ctx is None:
            self._ctx = FrameContext(self.device)
        self._ctx.set_scene(self.flat_scene())          # re-flattened every render: the scene list is mutable
        if self.adaptive_tolerance is not None:
            out = self._ctx.render_path_adaptive(_xyz(self.camera_position), width, height, samples_per_pixel, max_bounces,
                                                 self.mirror_threshold, min(self.adaptive_min_spp, samples_per_pixel),
                                                 self.adaptive_tolerance, seed=seed, fov=self.fov,
                                                 precision=_precision(self.precision), denoise=self.denoise,
                                                 features=self.track_features)
            self.sample_counts = out[3] if self.reuse_output else out[3].copy()
        else:
            out = self._ctx.render_path(_xyz(self.camera_position), width, height, samples_per_pixel, max_bounces,
                                        self.mirror_threshold, seed=seed, fov=self.fov, precision=_precision(self.precision),
                                        variance=self.track_variance, denoise=self.denoise, features=self.track_features)
        view, st = out[:2]
        if self.track_variance:
            self.variance = out[2] if self.reuse_output else out[2].copy()
        if self.track_features:
            c = self._ctx
            self.albedo, self.normal, self.depth = ((a if self.reuse_output else a.copy()) for a in (c.albedo, c.normal, c.depth))
        # reuse_output (default True): the image is a view of one of the renderer's FrameContext.HOST_RING pinned host
        # buffers -- it stays valid until two more frames have been rendered by THIS renderer, which covers every use
        # in the reference's drivers (plot / save / compare right after render()).  reuse_output = False returns a
        # fresh array per render exactly like the reference, at the price of a 24.9 MB host copy per 1080p frame (~3 ms).
        image = view if self.reuse_output else view.copy()
        for i, k in enumerate(('total_rays', 'total_intersections', 'light_hits', 'small_light_hits')):
            self.stats[k] = int(st[i])
        render_time = time.time() - start
        self.stats['render_time'] = render_time
        if render_time > 0:
            self.stats['rays_per_second'] = self.stats['total_rays'] / render_time
        return image


class ComplexTraditionalRenderer(TraditionalRenderer):
    """The complex-scene flavour (FB/fb_vs_traditional_complex.py:262-422): mirrors only when ``reflective > 0.9`` (:349)."""
    mirror_threshold = 0.9

    def __init__(self, device=0, precision="f32", seed=None):
        super().__init__(device, precision, seed)
        self.camera_position = Vector(0, 0, 12)


class CustomSceneExperiment:
    """The traditional-method render entries of RL/output5.py's ``CustomSceneExperiment``."""

    def __init__(self, output_dir="./custom_scene_results", device=0, precision="f32", seed=0):
        self.output_dir = Path(output_dir)
        self.output_dir.mkdir(parents=True, exist_ok=True)
        self.config = {'max_bounces': 6, 'image_width': 200, 'image_height': 200, 'samples_per_pixel': 16}
        self.timing_data = {'traditional': []}
        self.rendered_images = {}
        self.device, self.precision, self.seed = device, precision, seed
        self._ctx = None            # persistent FrameContext: scene handle, HBM buffers, pinned image, resident grid

    def _context(self):
        if self._ctx is None:
            self._ctx = FrameContext(self.device)
        return self._ctx

    # the constants of RL/output5.py:447-486 / :543-578 (the reference rebuilds them on every call; their values never change)
    _SUN = Sphere(id=0, centre=Vector(-0.6, 0.2, 6), radius=0.1, material=Material(emitive=True), colour=Colour(255, 255, 204))
    _GLOBAL = [GlobalLight(vector=Vector(3, 1, -0.75), colour=Colour(20, 20, 255), strength=1, max_angle=np.radians(90), func=0)]
    _POINT = [PointLight(id=0, position=Vector(-0.6, 0.2, 6), colour=Colour(255, 255, 204), strength=1,
                         max_angle=np.radians(90), func=-1)]
    _BACKGROUND = Colour(2, 2, 5)
    _LIGHTS = None

    @classmethod
    def _as_rendered(cls, scene_spheres):
        """RL/output5.py:447-486 / :543-578: sun id 7 replaced by an id-0 sun appended last, fixed light set."""
        spheres = [s for s in scene_spheres if not (hasattr(s, 'id') and s.id == 7)]
        spheres.append(cls._SUN)
        if cls._LIGHTS is None:               # the constant light set, flattened once
            cls._LIGHTS = flatten_scene([], cls._GLOBAL, cls._POINT, cls._BACKGROUND, path_lights=False)
        return flatten_scene(spheres, path_lights=False, lights_like=cls._LIGHTS)

    def _trace_custom_traditional(self, ray, spheres, scene_id=None):
        """One ray through the traditional path (RL/output5.py:535-607) -> (Colour, stats, strategies): the sun id 7 is
        swapped for the id-0 sun, ``ray.nearestSphereIntersect(all_spheres, max_bounces=config['max_bounces'])`` then
        ``terminalRGB`` with the fixed light set -- both evaluated on the GPU (batches of one through ``rt_trace_rays`` /
        ``rt_terminal_rgb``, FP64 parity build).  The reference's except-branch (a heuristic "enhanced" tracer, SURVEY
        section 2 row 12) is outside the hot path: errors propagate instead."""
        stats = {'reward': 0, 'light_hits': 0, 'steps': 0}
        strategies = ['traditional_mimic']
        sun = Sphere(id=0, centre=Vector(-0.6, 0.2, 6), radius=0.1, material=Material(emitive=True),
                     colour=Colour(255, 255, 204))
        all_spheres = [s for s in spheres if not (hasattr(s, 'id') and s.id == 7)]
        all_spheres.append(sun)
        gl = [GlobalLight(vector=Vector(3, 1, -0.75), colour=Colour(20, 20, 255), strength=1, max_angle=np.radians(90), func=0)]
        pl = [PointLight(id=sun.id, position=sun.centre, colour=sun.colour, strength=1, max_angle=np.radians(90), func=-1)]
        background_colour = Colour(2, 2, 5)
        terminal = ray.nearestSphereIntersect(all_spheres, max_bounces=self.config['max_bounces'])
        if terminal is None:
            return background_colour, stats, strategies
        color = terminal.terminalRGB(spheres=all_spheres, background_colour=background_colour, global_light_sources=gl,
                                     point_light_sources=pl)
        if (color.r + color.g + color.b) / 3 > 10:
            stats['light_hits'] = 1
            stats['reward'] = 10.0
        return color, stats, strategies

    def render_true_original(self, scene_spheres, save_path=None):
        """601x601 notebook grid, depth 5, direction NOT pre-normalised (RL/output5.py:416-533) -> image."""
        X, Y = notebook_grid(300, 0.01 / 3)
        fs = self._as_rendered(scene_spheres)
        image = render_whitted(fs, (0, 0, 1), X, Y, spp=1, max_bounces=5, miss=(2, 2, 5), prenorm=False,
                               precision=self.precision, device=self.device, context=self._context())
        if save_path is not None:
            save_png(image, save_path)
        return image

    def render_custom_scene(self, scene_spheres, method, save_path=None):
        """``render_custom_scene(scene, 'traditional', path)`` (RL/output5.py:1420-1525) -> (render_time, image)."""
        if method != 'traditional':
            raise NotImplementedError("only the traditional method is part of the hot path (SURVEY.md section 2, rows 12-13)")
        width, height = self.config['image_width'], self.config['image_height']
        spp = self.config['samples_per_pixel']
        start = time.time()
        if getattr(self, "_grid_key", None) != (width, height):             # the grid only depends on the frame size
            self._grid_key, self._grid = (width, height), custom_scene_grid(width, height)
        X, Y = self._grid
        fs = self._as_rendered(scene_spheres)
        image = render_whitted(fs, (0, 0, 1), X, Y, spp=spp, max_bounces=self.config['max_bounces'], miss=(2, 2, 5),
                               seed=self.seed, prenorm=True, precision=self.precision, device=self.device,
                               context=self._context())
        render_time = time.time() - start
        self.timing_data['traditional'].append(render_time)
        self.rendered_images[method] = image
        if save_path is not None:
            save_png(image, save_path)
        return render_time, image


class SimplifiedFBRenderer:
    """Drop-in for FB/output6.py ``SimplifiedFBRenderer`` in its traditional mode.

    The reference constructs the scene itself (``create_your_custom_scene()``, output6.py:45-83 = balls_in_space with
    the sun as id 7) and ships ``fb_usage_prob = 0.0`` (:116), i.e. every diffuse bounce is the cosine-weighted
    traditional one; the FB-guided branch needs a trained checkpoint the reference does not include and is out of the
    hot path (SURVEY.md 8f-4): a non-zero ``fb_usage_prob`` raises.  ``np.random.random`` draws (glass 50/50, diffuse
    r1/r2) come from Philox keyed (pixel, bounce) with ``self.seed``."""

    def __init__(self, model_path=None, device=0, precision="f32", seed=None):
        from .scenes import build_balls_in_space
        self.scene = build_balls_in_space(as_rendered=False).spheres
        self.sun_position = Vector(-0.6, 0.2, 6)
        self.sun_radius = 0.1
        self.sun_color = Colour(255, 255, 204)
        self.agent = None
        self.fb_model_loaded = False
        self.max_bounces = 5
        self.samples_per_pixel = 100          # unused by render_original_style, as in the reference (:113)
        self.fb_usage_prob = 0.0
        self.stats = {'total_rays': 0, 'sun_hits': 0, 'fb_used': 0, 'fb_success': 0, 'render_time': 0}
        self.device, self.precision, self.seed = device, precision, seed
        self._renders = 0
        self._sc = None

    def _scene_and_params(self, width, height):
        if self.fb_usage_prob:
            raise NotImplementedError("FB-guided sampling is outside the traditional hot path (fb_usage_prob must be 0)")
        seed = self.seed if self.seed is not None else (time.time_ns() ^ (self._renders * 0x9E3779B97F4A7C15)) & (2 ** 64 - 1)
        self._renders += 1
        fs = flatten_scene(self.scene)                                      # re-flattened: the scene list is mutable
        if self._sc is None:
            self._sc = nat.DeviceScene(fs, self.device)                     # persistent handle
            self._sc._sig = nat.scene_signature(fs)
        else:
            self._sc.update(fs, skip_unchanged=True)                        # re-uploaded when the list was mutated
        sc = self._sc
        p = sc.simple_params(width, height, cam=(0.0, 0.0, 1.0), sun_pos=_xyz(self.sun_position),
                             sun_col=self.sun_color.getList(), sun_id=7, max_bounces=self.max_bounces, seed=seed)
        return sc, p

    def _render_frame(self, sc, p, width, height):
        """One frame through ``rt_render_simple`` into buffers this renderer keeps (HBM rgb / image / stats + pinned host
        copies): no allocation and one synchronisation per frame (``rt_render_simple_host`` allocates and frees four
        device buffers per call, which cost more than the 400x300 frame itself)."""
        L, dev = nat.lib(), self.device
        if getattr(self, "_buf_key", None) != (width, height):
            for b in getattr(self, "_bufs", ()):
                b.free()
            n = width * height
            self._bufs = (nat.DeviceBuffer((n, 4), np.int32, dev), nat.DeviceBuffer((height, width, 3), np.float32, dev),
                          nat.DeviceBuffer(8, np.uint64, dev), nat.PinnedArray((height, width, 3), np.float32),
                          nat.PinnedArray(8, np.uint64))
            self._buf_key = (width, height)
        rgb, img, st, h_img, h_st = self._bufs
        st.fill(0)
        nat.check(L.rt_render_simple(sc.handle, _precision(self.precision), C.byref(p), rgb.ptr, img.ptr, st.ptr, None))
        nat.check(L.rt_memcpy_d2h(dev, h_img.ptr, img.ptr, img.nbytes, None))
        nat.check(L.rt_memcpy_d2h(dev, h_st.ptr, st.ptr, 64, None))
        nat.check(L.rt_stream_sync(dev, None))
        return h_img.array.copy(), h_st.array.copy()

    def trace_ray_simple(self, ray):
        """One ray -> accumulated ``Colour`` (output6.py:434-577); a batch of one through the same kernel."""
        sc, p = self._scene_and_params(1, 1)
        o, d = _xyz(ray.origin), _xyz(ray.D)
        _, rgb, st = sc.render_simple_host(p, _precision(self.precision), rays=np.array([[*o, *d]], np.float64),
                                           want_image=False)
        self.stats['total_rays'] += int(st[0])
        self.stats['sun_hits'] += int(st[1])
        return Colour(int(rgb[0, 0, 0]), int(rgb[0, 0, 1]), int(rgb[0, 0, 2]))

    def calculate_lighting_exact_original(self, intersection):
        """Lighting ``Colour`` at one intersection (output6.py:197-306): the sun's colour on the sun, else
        int(colour * min(255, global + shadowed sun) / 255).  ``intersection`` carries ``object`` (a sphere of
        ``self.scene``), ``point`` and ``normal`` like ``ray.Intersection``; a batch of one through the frame kernel's
        own lighting function (``rt_simple_params.lighting_only``)."""
        sc, p = self._scene_and_params(1, 1)
        obj = intersection.object
        idx = next((k for k, s in enumerate(self.scene) if s is obj), None)
        if idx is None:
            idx = next((k for k, s in enumerate(self.scene) if s.id == obj.id), None)
        if idx is None:
            raise ValueError("intersection.object is not a sphere of this renderer's scene")
        row = np.array([[*_xyz(intersection.point), *_xyz(intersection.normal), float(idx)]], np.float64)
        _, rgb, st = sc.render_simple_host(p, _precision(self.precision), hits=row)
        self.stats['sun_hits'] = self.stats.get('sun_hits', 0) + int(st[1])
        return Colour(int(rgb[0, 0, 0]), int(rgb[0, 0, 1]), int(rgb[0, 0, 2]))

    def render_original_style(self, width=400, height=300, output_path=None):
        """-> (image [H,W,3] float32 in [0,1], output_path) (output6.py:579-654)."""
        if output_path is None:
            output_path = f"./fb_simple_render_{time.strftime('%Y%m%d_%H%M%S')}.png"
        self.stats = {'total_rays': 0, 'sun_hits': 0, 'fb_used': 0, 'fb_success': 0, 'render_time': 0}
        start = time.time()
        sc, p = self._scene_and_params(width, height)
        image, st = self._render_frame(sc, p, width, height)
        self.stats['total_rays'], self.stats['sun_hits'] = int(st[0]), int(st[1])
        self.stats['render_time'] = time.time() - start
        if output_path:
            save_png(image, output_path)
        return image, output_path


# ---- Algorithm B with learned direction sampling (SURVEY.md 8f-4) -----------------------------------------------------
def _batched_policy(agent):
    """``agent.choose_directions(obs [m,22] CUDA tensor) -> [m,2]`` if the agent has it (a torch module evaluated once
    per bounce), else the reference's per-observation ``choose_direction(obs numpy) -> (2,)`` looped on the host."""
    import torch
    if hasattr(agent, "choose_directions"):
        return agent.choose_directions

    def looped(obs):
        rows = obs.cpu().numpy()
        out = np.stack([np.asarray(agent.choose_direction(r), np.float32).reshape(2) for r in rows]) if len(rows) else \
            np.zeros((0, 2), np.float32)
        return torch.as_tensor(out, device=obs.device)
    return looped


def render_path_wavefront(fs, camera, width, height, spp, max_bounces, mirror_threshold, policy=None, fb_usage_prob=1.0,
                          seed=0, fov=60.0, precision="f32", device=0, max_paths=1 << 22, scene=None, variance=False):
    """Algorithm B frame with ``policy(obs [m,22] float32 CUDA tensor) -> actions [m,2]`` choosing the diffuse bounce
    direction with probability ``fb_usage_prob`` (``WorkingFBRenderer.trace_ray_fb``,
    FB/fb_vs_traditional_complex.py:487-601).  Wavefront on the GPU: per bounce one trace kernel, the policy on the
    asking paths, one bounce kernel; sample ranges are processed ``max_paths`` paths at a time.
    -> (image [H,W,3] float32 numpy, sums [H,W,4] numpy, stats dict), plus the float32 [H,W,3] variance of each pixel's
    mean (colour levels^2) when ``variance`` is set."""
    import ctypes as C
    import torch
    prec = _precision(precision)
    own = scene is None
    sc = nat.DeviceScene(fs, device) if own else scene
    wf = C.c_void_p()
    try:
        dev = torch.device("cuda", sc.device)
        per_sample = width * height
        chunk = max(1, min(spp, max_paths // per_sample)) if per_sample <= max_paths else 0
        if chunk == 0:
            raise ValueError("max_paths is smaller than one sample of the frame")
        P = per_sample * chunk
        nat.check(nat.lib().rt_wf_create(sc.handle, prec, P, max(1, int(max_bounces)), C.byref(wf)))
        ft = torch.float64 if prec == nat.F64 else torch.float32
        accum = torch.zeros((height, width, 4), dtype=ft, device=dev)
        moments = torch.zeros((height, width, 4), dtype=torch.float64, device=dev) if variance else None
        obs = torch.zeros((P, 22), dtype=torch.float32, device=dev)
        need = torch.zeros(P, dtype=torch.uint8, device=dev)
        actions = torch.zeros((P, 2), dtype=torch.float32, device=dev)
        live = torch.zeros(1, dtype=torch.int32, device=dev)
        stats = torch.zeros(8, dtype=torch.int64, device=dev)
        prob = float(fb_usage_prob) if policy is not None else 0.0
        for s0 in range(0, spp, chunk):
            s1 = min(spp, s0 + chunk)
            n = per_sample * (s1 - s0)
            p = sc.path_params(camera, width, height, spp, max_bounces, mirror_threshold, seed=seed, fov=fov, samples=(s0, s1))
            nat.check(nat.lib().rt_wf_begin(wf, C.byref(p), prob, stats.data_ptr(), None))
            for _ in range(int(max_bounces)):
                nat.check(nat.lib().rt_wf_trace(wf, obs.data_ptr(), need.data_ptr(), stats.data_ptr(), None))
                if prob > 0.0:
                    idx = need[:n].nonzero(as_tuple=True)[0]
                    if idx.numel():
                        actions[idx] = policy(obs[idx]).to(device=dev, dtype=torch.float32).reshape(-1, 2)
                live.zero_()
                nat.check(nat.lib().rt_wf_bounce(wf, need.data_ptr(), actions.data_ptr(), stats.data_ptr(), live.data_ptr(), None))
                if int(live.item()) == 0:
                    break
            if variance:
                nat.check(nat.lib().rt_wf_finish_moments(wf, accum.data_ptr(), moments.data_ptr(), None))
            else:
                nat.check(nat.lib().rt_wf_finish(wf, accum.data_ptr(), None))
        image = torch.zeros((height, width, 3), dtype=torch.float32, device=dev)
        sc.resolve(accum, width, height, spp, image, prec)
        if variance:
            var = torch.zeros((height, width, 3), dtype=torch.float32, device=dev)
            sc.resolve_variance(accum, moments, width, height, var, prec)
        torch.cuda.synchronize(dev)
        st = stats.cpu().numpy()
        out = {"total_rays": int(st[0]), "total_intersections": int(st[1]), "light_hits": int(st[2]), "small_light_hits": int(st[3]),
               "queries": int(st[4]), "sphere_tests": int(st[5]), "fb_used": int(st[7])}
        if variance:
            return image.cpu().numpy(), accum.cpu().numpy(), out, var.cpu().numpy()
        return image.cpu().numpy(), accum.cpu().numpy(), out
    finally:
        if wf.value:
            nat.load_symbols().rt_wf_destroy(wf)
        if own:
            sc.close()


class WorkingFBRenderer:
    """Drop-in for ``WorkingFBRenderer`` (FB/fb_vs_traditional_complex.py:425-640; the chandelier file's copy differs
    only in the mirror threshold): Algorithm B whose diffuse bounces are steered by ``self.fb_agent`` with probability
    ``self.fb_usage_prob``.  The reference builds the agent from a checkpoint (``TrainedFBAgent(model_path, ...)``);
    the checkpoints and ``fb_ray_tracing`` are not part of the reference, so here the agent is whatever object the
    caller assigns to ``fb_agent``: ``choose_directions(obs [m,22] CUDA tensor) -> [m,2]`` (preferred, one call per
    bounce) or the reference's ``choose_direction(obs) -> (2,)``.  Without an agent it renders like
    ``TraditionalRenderer`` (``fb_usage_prob = 0``, as the reference does when no model is given)."""

    mirror_threshold = 0.9
    reuse_output = True         # agent-less frames: see TraditionalRenderer.render
    track_variance = False      # True: render() also sets self.variance (see TraditionalRenderer), on both branches

    def __init__(self, model_path=None, scene_small_lights=None, camera_position=None, device=0, precision="f32", seed=None):
        if model_path is not None:
            raise NotImplementedError("trained FB checkpoints are not part of the reference: assign an agent to .fb_agent")
        self.scene = []
        self.camera_position = camera_position if camera_position is not None else Vector(0, 2, 0)
        self.camera_angle = None
        self.global_lights, self.point_lights, self.light_sources = [], [], []
        self.small_lights = scene_small_lights if scene_small_lights is not None else []
        self.fb_agent, self.fb_loaded, self.fb_usage_prob = None, False, 0.0
        self.stats = {'total_rays': 0, 'total_intersections': 0, 'light_hits': 0, 'small_light_hits': 0, 'fb_used': 0,
                      'fb_success': 0, 'render_time': 0, 'rays_per_second': 0}
        self.device, self.precision, self.seed = device, precision, seed
        self._renders = 0
        self._ctx = None            # persistent FrameContext of the agent-less frames

    def set_render_settings(self, width=200, height=150, max_bounces=3, samples_per_pixel=4):
        self.image_width, self.image_height = width, height
        self.max_bounces, self.samples_per_pixel = max_bounces, samples_per_pixel
        self.aspect_ratio = width / height
        self.fov = 60

    def render(self, width=200, height=150, samples_per_pixel=4, max_bounces=3):
        self.set_render_settings(width, height, max_bounces, samples_per_pixel)
        self.stats = {k: 0 for k in self.stats}
        start = time.time()
        seed = self.seed if self.seed is not None else (time.time_ns() ^ (self._renders * 0x9E3779B97F4A7C15)) & (2 ** 64 - 1)
        self._renders += 1
        fs = flatten_scene(self.scene, background_colour=Colour(2, 2, 5), light_sources=self.light_sources,
                           small_lights=self.small_lights)
        use = self.fb_loaded and self.fb_agent is not None and self.fb_usage_prob > 0
        if not use:
            # no agent (the state the reference is in without a checkpoint, :436-437) or fb_usage_prob = 0: every bounce is
            # the traditional one and the wavefront's frame equals the fused path kernel's bit for bit
            # (tests/test_gpu_parity.py::test_wavefront_fb_renderer), so the frame goes through that single launch
            if self._ctx is None:
                self._ctx = FrameContext(self.device)
            self._ctx.set_scene(fs)
            out = self._ctx.render_path(_xyz(self.camera_position), width, height, samples_per_pixel, max_bounces,
                                        self.mirror_threshold, seed=seed, fov=self.fov, precision=_precision(self.precision),
                                        variance=self.track_variance)
            view, st = out[:2]
            if self.track_variance:
                self.variance = out[2] if self.reuse_output else out[2].copy()
            for i, k in enumerate(('total_rays', 'total_intersections', 'light_hits', 'small_light_hits')):
                self.stats[k] = int(st[i])
            self.stats['render_time'] = time.time() - start
            if self.stats['render_time'] > 0:
                self.stats['rays_per_second'] = self.stats['total_rays'] / self.stats['render_time']
            return view if self.reuse_output else view.copy()      # as TraditionalRenderer.render: a view of the pinned ring
        res = render_path_wavefront(fs, _xyz(self.camera_position), width, height, samples_per_pixel, max_bounces,
                                    self.mirror_threshold, policy=_batched_policy(self.fb_agent) if use else None,
                                    fb_usage_prob=self.fb_usage_prob if use else 0.0, seed=seed, fov=self.fov,
                                    precision=self.precision, device=self.device, variance=self.track_variance)
        image, _, st = res[:3]
        if self.track_variance:
            self.variance = res[3]
        for k in ('total_rays', 'total_intersections', 'light_hits', 'small_light_hits', 'fb_used'):
            self.stats[k] = st[k]
        self.stats['fb_success'] = st['fb_used']                     # the reference counts both at the same place (:539-544)
        self.stats['render_time'] = time.time() - start
        if self.stats['render_time'] > 0:
            self.stats['rays_per_second'] = self.stats['total_rays'] / self.stats['render_time']
        return image
