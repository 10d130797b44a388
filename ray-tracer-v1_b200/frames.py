"""Persistent frame state on one GPU: scene handle, accumulation / image buffers in HBM and a pinned host image.

``FrameContext`` is what the render entry points and the multi-GPU sharding layer (distributed.py) share.  A frame is
rendered in three stream-ordered launches -- path/whitted kernel -> resolve kernel -> one D2H copy of the float32
image into page-locked memory -- and nothing else crosses PCIe except the few KB of flattened scene.
"""
import ctypes as C

import numpy as np

from . import _native as nat

__all__ = ["FrameContext"]


class FrameContext:
    HOST_RING = 3
    # feature frames trace their first-hit features over the first min(spp, FEATURE_SPP) samples of the frame: geometry
    # converges in a few samples (DESIGN §4.8d)
    FEATURE_SPP = 8

    def __init__(self, device=0):
        self.device = device
        self.scene = None
        self._key = None
        self.accum = self.image = self.stats = self.hit = None
        self.host_image = self.host_stats = None
        self.moments = self.var = None      # variance frames only: [H,W,4] float64 moments, [H,W,3] float32 variance
        self.host_var_ring, self.host_var = [], None
        # adaptive frames only: the active-pixel list ((H*W + 1) uint32) and the [H,W] int32 sample counts
        self.pixel_list = self.counts = None
        self.host_counts_ring, self.host_counts = [], None
        # feature frames only: (albedo [H,W,3], normal [H,W,3], depth [H,W], fvar [H,W,3]) float32 in HBM, their pinned
        # rings, and the host views of the last feature frame read back
        self.features = None
        self.host_features_ring = []
        self.albedo = self.normal = self.depth = self.feature_var = None
        self.h2d_bytes = 0          # bytes of the last scene upload
        self.d2h_bytes = 0          # bytes of the last read-back

    # ---- scene -----------------------------------------------------------------------------------------------
    def set_scene(self, fs, lbvh=None, skip_unchanged=False):
        """(Re)upload the flattened scene; allocations are reused when the census is unchanged.  ``skip_unchanged``: a
        scene whose flattened content equals the resident one is not uploaded again (``h2d_bytes`` = 0 for that frame)."""
        uploaded = True
        if self.scene is None:
            self.scene = nat.DeviceScene(fs, self.device)
            if skip_unchanged:
                self.scene._sig = nat.scene_signature(fs)
        else:
            uploaded = self.scene.update(fs, skip_unchanged=skip_unchanged)
        n, nG, nP, nL = fs.radius.shape[0], fs.g_strength.shape[0], fs.p_strength.shape[0], fs.l_index.shape[0]
        self.h2d_bytes = ((16 + 32) * (3 * n + 2 * (nG + nP + nL)) + 2 * 4 * (n + nG + 2 * nP + nL) + n) if uploaded else 0
        if uploaded and (lbvh or (lbvh is None and self.scene.n > 256)):
            self.scene.build_lbvh()
        return self.scene

    # ---- buffers ---------------------------------------------------------------------------------------------
    def _buffers(self):
        return [self.accum, self.image, self.stats, self.hit, self.host_stats, self.moments, self.var, self.pixel_list,
                self.counts] + list(getattr(self, "host_ring", [])) + list(self.host_var_ring) + \
            list(self.host_counts_ring) + list(self.features or ()) + [b for r in self.host_features_ring for b in r]

    def ensure(self, W, H, precision=nat.F32, want_hit=False, want_variance=False, want_adaptive=False,
               want_features=False):
        key = (int(W), int(H), precision)
        if self._key != key:
            for b in self._buffers():
                if b is not None:
                    b.free()
            ft = np.float64 if precision == nat.F64 else np.float32
            self.accum = nat.DeviceBuffer((H, W, 4), ft, self.device)
            self.image = nat.DeviceBuffer((H, W, 3), np.float32, self.device)
            self.stats = nat.DeviceBuffer(8, np.uint64, self.device)
            # a ring of pinned host images: a frame handed out by read_back stays untouched until HOST_RING - 1 later
            # frames have been read back (TraditionalRenderer.render returns these views without copying them)
            self.host_ring = [nat.PinnedArray((H, W, 3), np.float32) for _ in range(self.HOST_RING)]
            self._ring_at = 0
            self.host_image = self.host_ring[0]
            self.host_stats = nat.PinnedArray(8, np.uint64)
            self.hit = None
            self.moments = self.var = None
            self.host_var_ring = []
            self.pixel_list = self.counts = None
            self.host_counts_ring = []
            self.features = None
            self.host_features_ring = []
            self._key = key
        if want_hit and self.hit is None:
            self.hit = nat.DeviceBuffer((H, W), np.int32, self.device)
        if want_variance and self.moments is None:
            # allocated on the first variance frame: frames without it neither allocate nor write these buffers
            self.moments = nat.DeviceBuffer((H, W, 4), np.float64, self.device)
            self.var = nat.DeviceBuffer((H, W, 3), np.float32, self.device)
            self.host_var_ring = [nat.PinnedArray((H, W, 3), np.float32) for _ in range(self.HOST_RING)]
        if want_adaptive and self.pixel_list is None:
            # allocated on the first adaptive frame
            self.pixel_list = nat.DeviceBuffer(H * W + 1, np.uint32, self.device)
            self.counts = nat.DeviceBuffer((H, W), np.int32, self.device)
            self.host_counts_ring = [nat.PinnedArray((H, W), np.int32) for _ in range(self.HOST_RING)]
        if want_features and self.features is None:
            # allocated on the first feature frame
            shapes = ((H, W, 3), (H, W, 3), (H, W), (H, W, 3))
            self.features = tuple(nat.DeviceBuffer(s, np.float32, self.device) for s in shapes)
            self.host_features_ring = [tuple(nat.PinnedArray(s, np.float32) for s in shapes) for _ in range(self.HOST_RING)]

    def _render_features(self, cam, W, H, spp, seed, fov, precision, rows, s0, stream):
        """The first-hit features of rows over samples [s0, s0 + min(spp, FEATURE_SPP)) into ``self.features``."""
        p = self.scene.path_params(cam, W, H, spp, 1, 0.0, seed=seed, fov=fov, rows=rows,
                                   samples=(s0, s0 + min(int(spp), self.FEATURE_SPP)))
        self.scene.render_features(p, *self.features, precision=precision, stream=stream)

    # ---- frames ----------------------------------------------------------------------------------------------
    def render_path(self, cam, W, H, spp, max_bounces, mirror_threshold, seed=0, fov=60.0, precision=nat.F32, rows=None,
                    samples=None, resolve=True, read_back=True, stream=None, variance=False, denoise=False,
                    features=False):
        """Algorithm B over rows x samples of this rank.  Returns (host image view or None, stats u64[8] or None).

        variance=True: the launch also stores the second moments of every pixel's samples (``self.moments``), and the
        result gains a third item, the float32 [H,W,3] variance of each pixel's mean in colour levels^2 -- a view of a
        pinned host ring like the image (None when not read back; ``self.var`` holds it in HBM when resolved).

        denoise=True: the frame is rendered with its moments, its variance is resolved, and the image is the variance-guided
        non-local-means filter of the frame (``rt_denoise`` with the library defaults) in place of the resolved one; the
        return shape is the one ``variance`` selects.  The filter reads every row, so the whole frame is rendered in one
        launch and read back once after the filter: the banded read-back overlap (``BANDS``) does not apply, and
        ``rows`` must cover the frame.

        features=True: the frame's first-hit features (``rt_render_features`` over its first min(spp, FEATURE_SPP)
        samples) are rendered too and, when read back, exposed as ``self.albedo`` [H,W,3], ``self.normal`` [H,W,3],
        ``self.depth`` [H,W] and ``self.feature_var`` [H,W,3], views of pinned host rings like the image; with denoise,
        the filter is the feature-guided one (``rt_denoise_features``, library defaults).  The return shape does not
        change, and the banded read-back does not apply."""
        if denoise and (not resolve or (rows is not None and (int(rows[0]), int(rows[1])) != (0, int(H)))):
            raise ValueError("denoise filters the whole frame: it needs every row and resolve=True")
        self.ensure(W, H, precision, want_variance=variance or denoise, want_features=features)
        L = nat.lib()
        p = self.scene.path_params(cam, W, H, spp, max_bounces, mirror_threshold, seed=seed, fov=fov, rows=rows,
                                   samples=samples)
        self.stats.fill(0, stream)
        moments = self.moments if (variance or denoise) else None
        bands = self._bands(W, p.y0, p.y1, p.s1 - p.s0) if (resolve and read_back and not denoise and not features) else None
        if bands:
            return self._render_path_banded(p, bands, W, H, precision, stream, variance)
        self.scene.render_path(p, self.accum, precision, stats=self.stats, stream=stream, moments=moments)
        self.launches = 1
        if features:
            self._render_features(cam, W, H, p.s1 - p.s0, seed, fov, precision, (p.y0, p.y1), p.s0, stream)
            self.launches += 1
        if denoise:
            self.scene.resolve_variance(self.accum, self.moments, W, H, self.var, precision, stream=stream)
            self.scene.denoise(self.accum, self.var, W, H, self.image, precision, stream=stream,
                               features=self.features if features else None)
            self.launches += 2
        elif resolve:
            self.scene.resolve(self.accum, W, H, p.s1 - p.s0, self.image, precision, rows=(p.y0, p.y1), stream=stream)
            self.launches += 1
            if variance:
                self.scene.resolve_variance(self.accum, self.moments, W, H, self.var, precision, rows=(p.y0, p.y1),
                                            stream=stream)
                self.launches += 1
        if not read_back:
            return (None, None, None) if variance else (None, None)
        image, stats = self.read_back(W, H, (p.y0, p.y1), stream, variance=variance and resolve, features=features)
        if variance:
            return image, stats, (self.host_var.array if resolve else None)
        return image, stats

    # a frame whose image takes longer to copy out than a launch costs is rendered in row bands: band b is copied to the
    # pinned host image (copy stream) while band b + 1 renders.  Pixels are keyed by (pixel, sample), so the frame is the
    # same bit for bit (tested); every extra launch costs ~30 us of drain, every band hides its share of the copy.  The
    # bands taper (BAND_WEIGHTS): a band's copy hides behind the NEXT band's render, so only the last band's copy is paid.
    # Only the LAST band's copy is exposed and every extra launch costs its drain, so: two bands, the last one 1/16 of the
    # rows.  Measured through ComplexTraditionalRenderer.render(1920, 1080, 64, 5) (tools/debug/bands_ab.py,
    # profiles/bands_ab_r2.txt): one launch 17.53 ms, four equal bands 17.33, (11,10,8,3) 17.25, (6,5,2) 17.23, (7,1) 17.20,
    # (15,1) 17.17, (23,1) 17.16 (kept at 15:1 -- the first band's 23 MB copy still hides at the smallest banded frames).
    BANDS = 2
    BAND_WEIGHTS = (15, 1)
    BAND_MIN_IMAGE_BYTES = 8 << 20
    BAND_MIN_SAMPLES = 24 << 20          # pixel-samples: below ~10 ms of kernel the split is not worth its launches

    def _bands(self, W, y0, y1, ns):
        rows = y1 - y0
        if self.BANDS < 2 or rows * W * 12 < self.BAND_MIN_IMAGE_BYTES or rows * W * ns < self.BAND_MIN_SAMPLES:
            return None
        stripes = (rows + 7) // 8
        w = self.BAND_WEIGHTS if len(self.BAND_WEIGHTS) == self.BANDS else (1,) * self.BANDS
        cuts = [y0 + 8 * ((stripes * sum(w[:k])) // sum(w)) for k in range(self.BANDS)] + [y1]
        return [(a, b) for a, b in zip(cuts[:-1], cuts[1:]) if b > a]

    def _render_path_banded(self, p, bands, W, H, precision, stream, variance=False):
        L = nat.lib()
        if getattr(self, "_copy_stream", None) is None:
            cs = nat.vp()
            nat.check(L.rt_stream_create(self.device, C.byref(cs)))
            self._copy_stream = cs
        cs = self._copy_stream
        self._ring_at = (self._ring_at + 1) % self.HOST_RING
        self.host_image = self.host_ring[self._ring_at]
        if variance:
            self.host_var = self.host_var_ring[self._ring_at]
        ns, y0, y1 = p.s1 - p.s0, p.y0, p.y1
        self.launches = 0
        for (a, b) in bands:
            p.y0, p.y1 = a, b
            self.scene.render_path(p, self.accum, precision, stats=self.stats, stream=stream,
                                   moments=self.moments if variance else None)
            self.scene.resolve(self.accum, W, H, ns, self.image, precision, rows=(a, b), stream=stream)
            self.launches += 2
            if variance:
                self.scene.resolve_variance(self.accum, self.moments, W, H, self.var, precision, rows=(a, b), stream=stream)
                self.launches += 1
            nat.check(L.rt_stream_wait_stream(self.device, cs, stream))
            off, nbytes = a * W * 12, (b - a) * W * 12
            nat.check(L.rt_memcpy_d2h(self.device, self.host_image.ptr + off, self.image.ptr + off, nbytes, cs))
            if variance:
                nat.check(L.rt_memcpy_d2h(self.device, self.host_var.ptr + off, self.var.ptr + off, nbytes, cs))
        p.y0, p.y1 = y0, y1
        nat.check(L.rt_memcpy_d2h(self.device, self.host_stats.ptr, self.stats.ptr, 64, stream))
        nat.check(L.rt_stream_sync(self.device, stream))
        nat.check(L.rt_stream_sync(self.device, cs))
        self.d2h_bytes = (y1 - y0) * W * (24 if variance else 12) + 64
        if variance:
            return self.host_image.array, self.host_stats.array, self.host_var.array
        return self.host_image.array, self.host_stats.array

    def render_path_adaptive(self, cam, W, H, max_spp, max_bounces, mirror_threshold, min_spp, tolerance, seed=0, fov=60.0,
                             precision=nat.F32, stream=None, denoise=False, features=False):
        """Adaptive Algorithm B frame (``rt_render_path_adaptive``): every pixel gets ``min_spp`` samples, then the pixels
        whose variance of the mean still exceeds ``tolerance``^2 (colour levels) get doubling rounds up to ``max_spp``.
        Returns (image [H,W,3] float32, stats u64[8], variance [H,W,3] float32, sample counts [H,W] int32), views of
        pinned host rings like the image of ``render_path``.  The call synchronises the stream once per round.
        denoise=True: the image is the frame filtered by ``rt_denoise`` (library defaults), each pixel's mean and variance
        taken at its own sample count.
        features=True: as for ``render_path``, over the first min(max_spp, FEATURE_SPP) samples."""
        self.ensure(W, H, precision, want_variance=True, want_adaptive=True, want_features=features)
        p = self.scene.path_params(cam, W, H, max_spp, max_bounces, mirror_threshold, seed=seed, fov=fov)
        self.stats.fill(0, stream)
        if features:
            self._render_features(cam, W, H, max_spp, seed, fov, precision, (0, H), 0, stream)
        self.scene.render_path_adaptive(p, min_spp, tolerance, self.accum, self.moments, self.pixel_list, self.image,
                                        precision, var=self.var, counts=self.counts, stats=self.stats, stream=stream)
        if denoise:
            self.scene.denoise(self.accum, self.var, W, H, self.image, precision, stream=stream,
                               features=self.features if features else None)
        image, stats = self.read_back(W, H, (0, H), stream, variance=True, counts=True, features=features)
        return image, stats, self.host_var.array, self.host_counts.array

    def render_whitted(self, cam, X, Y, spp=1, max_bounces=1, shadow_max_bounces=0, miss=None, seed=0, prenorm=False,
                       precision=nat.F32, rows=None, samples=None, read_back=True, stream=None):
        W, H = len(X), len(Y)
        self.ensure(W, H, precision)
        p = self.scene.whitted_params(cam, X, Y, spp=spp, max_bounces=max_bounces, shadow_max_bounces=shadow_max_bounces,
                                      miss=miss, seed=seed, prenorm=prenorm, rows=rows, samples=samples)
        self.stats.fill(0, stream)
        self.scene.render_whitted(p, self.accum, precision, stats=self.stats, stream=stream)
        self.scene.resolve(self.accum, W, H, p.s1 - p.s0, self.image, precision, rows=(p.y0, p.y1), stream=stream)
        self.launches = 2
        if not read_back:
            return None, None
        return self.read_back(W, H, (p.y0, p.y1), stream)

    def read_back(self, W, H, rows, stream=None, variance=False, counts=False, features=False):
        """D2H of the resolved rows (float32) + the stats block into pinned memory; synchronises the stream.  variance:
        the rows of the variance image too, into ``self.host_var`` (the pinned ring slot of this frame); counts: those
        of the int32 sample counts of an adaptive frame, into ``self.host_counts``; features: those of the feature
        buffers, exposed as ``self.albedo``, ``self.normal``, ``self.depth`` and ``self.feature_var``."""
        L = nat.lib()
        y0, y1 = rows
        self._ring_at = (self._ring_at + 1) % self.HOST_RING
        self.host_image = self.host_ring[self._ring_at]
        off, nbytes = y0 * W * 3 * 4, (y1 - y0) * W * 3 * 4
        if nbytes:
            nat.check(L.rt_memcpy_d2h(self.device, self.host_image.ptr + off, self.image.ptr + off, nbytes, stream))
        if variance:
            self.host_var = self.host_var_ring[self._ring_at]
            if nbytes:
                nat.check(L.rt_memcpy_d2h(self.device, self.host_var.ptr + off, self.var.ptr + off, nbytes, stream))
        if counts:
            self.host_counts = self.host_counts_ring[self._ring_at]
            if nbytes:
                nat.check(L.rt_memcpy_d2h(self.device, self.host_counts.ptr + off // 3, self.counts.ptr + off // 3, nbytes // 3,
                                          stream))
        if features:
            host = self.host_features_ring[self._ring_at]
            for h, d in zip(host, self.features):
                k = 1 if h.array.ndim == 2 else 3          # depth has one channel
                if nbytes:
                    nat.check(L.rt_memcpy_d2h(self.device, h.ptr + off // 3 * k, d.ptr + off // 3 * k, nbytes // 3 * k,
                                              stream))
            self.albedo, self.normal, self.depth, self.feature_var = (h.array for h in host)
        nat.check(L.rt_memcpy_d2h(self.device, self.host_stats.ptr, self.stats.ptr, 64, stream))
        nat.check(L.rt_stream_sync(self.device, stream))
        self.d2h_bytes = nbytes * (2 if variance else 1) + (nbytes // 3 if counts else 0) + (nbytes // 3 * 10 if features else 0) + 64
        return self.host_image.array, self.host_stats.array

    def close(self):
        for b in self._buffers():
            if b is not None:
                b.free()
        self.host_ring = []
        self.host_var_ring = []
        self.host_counts_ring = []
        self.host_features_ring = []
        self.moments = self.var = self.pixel_list = self.counts = self.features = None
        self.albedo = self.normal = self.depth = self.feature_var = None
        if getattr(self, "_copy_stream", None) is not None:
            nat.lib().rt_stream_destroy(self.device, self._copy_stream)
            self._copy_stream = None
        self.accum = self.image = self.stats = self.hit = self.host_image = self.host_stats = None
        self._key = None
        if self.scene is not None:
            self.scene.close()
            self.scene = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
