"""Multi-GPU sharding of frames: one process per GPU (torchrun), ``torch.distributed`` for the plumbing.

The path shards three ways (SURVEY.md section 8e); each needs at most ONE collective per frame:

* tiles    -- contiguous row bands, one per rank (C3: complex scene).  Every rank resolves its own band and rank 0
              receives the float32 bands with one NCCL gather straight into the rows of the final image (no staging).
* samples  -- sample ranges of every pixel, one per rank (C4: chandelier at high spp).  One NCCL reduce(sum) of the
              FP32 [H,W,4] accumulation buffers to rank 0, then the ``// spp`` resolve there.  Per-sample colours are
              integers, so FP32 sums are exact below 2^24 and the reduced frame is bit-identical to the unsharded one.
              With ``variance=True`` the float64 second moments are reduced the same way (integer-valued doubles below
              2^53: exact), so the variance image is bit-identical too.
* env      -- environment slices (C5): no collective at all, see ray_tracer_env.BatchedRayTracerEnv.shard.

A denoised frame (``render(..., denoise=True)``, DESIGN §4.8e) is filtered in the same row bands: every rank forms the
final sums of its band (``reduce_row_bands`` in samples mode), receives the ``h`` rows of its neighbours' sums and
variance its filter reads (``halo_plan`` / ``exchange_halos``, one batched point-to-point exchange) and filters its band
with ``rt_denoise_rows``, which reads no row outside that window; rank 0 gathers the bands.

Because the Philox stream is keyed by the GLOBAL (pixel, sample, bounce), a sharded frame equals the unsharded frame
bit for bit for any world size.  The partition/collective helpers take the band renderer as a callable so the
world_size-2 ``gloo`` tests on CPU exercise exactly this code with a stand-in renderer.
"""
import numpy as np

__all__ = ["row_bands", "sample_ranges", "env_slices", "tile_stripes", "gather_row_bands", "reduce_sample_sums",
           "halo_windows", "halo_plan", "exchange_halos", "reduce_row_bands", "PeerFabric", "ShardedPathRenderer"]


def _split(total, world):
    return [(total * r // world, total * (r + 1) // world) for r in range(world)]


def row_bands(height, world):
    """Contiguous [y0, y1) row bands, sizes differing by at most one row."""
    return _split(int(height), int(world))


def sample_ranges(spp, world):
    """Contiguous [s0, s1) sample ranges (a rank may get an empty range when spp < world)."""
    return _split(int(spp), int(world))


def env_slices(n_envs, world):
    """Contiguous [b0, b1) environment slices."""
    return _split(int(n_envs), int(world))


def tile_stripes(height, world, rank, tile_rows=8):
    """Rows of the interleaved 8-row stripes rank ``rank`` renders in the fused tile mode: tiles rank, rank + world, ..."""
    tiles = (int(height) + tile_rows - 1) // tile_rows
    return [(t * tile_rows, min(int(height), (t + 1) * tile_rows)) for t in range(int(rank), tiles, int(world))]


def _dist():
    import torch.distributed as dist
    return dist


def _world(group=None):
    dist = _dist()
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def gather_row_bands(image, bands, group=None, dst=0):
    """``image`` [H,W,C]: each rank has filled its own band ``bands[rank]``; after the call rank ``dst`` holds all rows.

    Equal bands: one gather whose receive buffers are the row slices of ``image`` itself.  Ragged bands: padded to
    the tallest band and copied in."""
    import torch
    dist = _dist()
    rank, world = _world(group)
    if world == 1:
        return image
    sizes = {b[1] - b[0] for b in bands}
    y0, y1 = bands[rank]
    dst_global = dist.get_global_rank(group, dst) if group is not None else dst
    if len(sizes) == 1:
        mine = image[y0:y1]
        if rank == dst:
            recv = [image[a:b] for a, b in bands]
            recv[rank] = torch.empty_like(mine)          # own band is already in place
            dist.gather(mine, recv, dst=dst_global, group=group)
        else:
            dist.gather(mine, None, dst=dst_global, group=group)
        return image
    tallest = max(sizes)
    pad = image.new_zeros((tallest,) + tuple(image.shape[1:]))
    pad[: y1 - y0] = image[y0:y1]
    if rank == dst:
        recv = [torch.empty_like(pad) for _ in bands]
        dist.gather(pad, recv, dst=dst_global, group=group)
        for r, (a, b) in enumerate(bands):
            if r != rank:
                image[a:b] = recv[r][: b - a]
    else:
        dist.gather(pad, None, dst=dst_global, group=group)
    return image


def reduce_sample_sums(accum, group=None, dst=0):
    """Sum the per-rank [H,W,4] accumulation buffers (r,g,b sums + sample count) onto rank ``dst``."""
    dist = _dist()
    rank, world = _world(group)
    if world == 1:
        return accum
    dst_global = dist.get_global_rank(group, dst) if group is not None else dst
    dist.reduce(accum, dst=dst_global, op=dist.ReduceOp.SUM, group=group)
    return accum


def halo_windows(height, world, halo):
    """Each rank's window [y_lo, y_hi) = [max(0, y0 - halo), min(H, y1 + halo)) around its band [y0, y1) of
    ``row_bands``: the rows a stencil of depth ``halo`` reads to compute the band.  An empty band has an empty window."""
    H, h = int(height), int(halo)
    return [(a, a) if a == b else (max(0, a - h), min(H, b + h)) for a, b in row_bands(H, world)]


def halo_plan(height, world, halo):
    """The row copies that give every rank the rows of its ``halo_windows`` window it does not own: a list of
    (src, dst, a, b), rank ``src`` sends rows [a, b) of its band to rank ``dst``.  Every such row is covered exactly
    once, from the rank whose band holds it, so a halo deeper than a neighbour's band takes rows from several ranks."""
    bands = row_bands(height, world)
    plan = []
    for dst, (lo, hi) in enumerate(halo_windows(height, world, halo)):
        for src, (a, b) in enumerate(bands):
            a, b = max(a, lo), min(b, hi)
            if src != dst and a < b:
                plan.append((src, dst, a, b))
    return plan


def exchange_halos(tensors, plan, group=None):
    """Carry out ``halo_plan`` for every [H, ...] tensor of ``tensors`` (each rank's own band already final), with one
    batched point-to-point exchange (``batch_isend_irecv``).  Row slices of a contiguous tensor are contiguous, so the
    rows are sent from and received into the tensors themselves."""
    dist = _dist()
    rank, world = _world(group)
    glob = (lambda r: dist.get_global_rank(group, r)) if group is not None else (lambda r: r)
    ops = []
    for src, dst, a, b in plan:
        if rank == src:
            ops += [dist.P2POp(dist.isend, t[a:b], glob(dst), group) for t in tensors]
        elif rank == dst:
            ops += [dist.P2POp(dist.irecv, t[a:b], glob(src), group) for t in tensors]
    if world > 1 and ops:
        for req in dist.batch_isend_irecv(ops):
            req.wait()
    return tensors


def reduce_row_bands(t, bands, group=None):
    """Sum the per-rank [H, ...] tensors ``t`` so that each rank holds the final sums of its own band ``bands[rank]``:
    one in-place reduce per non-empty band, sent to the band's owner.  The bands do not overlap, so every row is reduced
    once (in all, the traffic of a reduce-scatter); rows outside a rank's own band are left undefined."""
    dist = _dist()
    rank, world = _world(group)
    if world == 1:
        return t
    for owner, (a, b) in enumerate(bands):
        if a < b:
            dst = dist.get_global_rank(group, owner) if group is not None else owner
            dist.reduce(t[a:b], dst=dst, op=dist.ReduceOp.SUM, group=group)
    return t


class _DevArray:
    """Zero-copy view of raw device memory for ``torch.as_tensor`` (CUDA array interface v3)."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 3,
                                         "strides": None}


class PeerFabric:
    """Buffers of every rank of a process group mapped into this process (CUDA IPC, NVLink peer access), plus the
    epoch flags that order writers and readers across ranks.  One instance per rank; collective construction.

    ``alloc(name, nbytes)`` allocates ``nbytes`` on every rank and returns the list of the ``world`` device pointers
    (own buffer at index ``rank``, peer mappings elsewhere).  The handles travel by ``all_gather_object``: this is the
    only use of the process group; the data path is the kernels' own loads/stores/reductions over NVLink."""

    def __init__(self, device, group=None):
        from . import _native as nat
        self.nat, self.device, self.group = nat, int(device), group
        self.rank, self.world = _world(group)
        if self.world > nat.RT_MAX_PEERS:
            raise ValueError(f"at most {nat.RT_MAX_PEERS} ranks")
        self.ptrs, self._own, self._opened = {}, [], []

    def alloc(self, name, nbytes):
        """Collective.  A failure on ANY rank (allocation, IPC export, peer mapping) raises on EVERY rank after the
        exchange, so callers can fall back together instead of leaving peers blocked in a collective."""
        import ctypes as C
        nat, dist = self.nat, _dist()
        own, handle = C.c_void_p(), C.create_string_buffer(nat.IPC_HANDLE_BYTES)
        err = None
        try:
            nat.check(nat.lib().rt_peer_alloc(self.device, int(nbytes), C.byref(own), handle))
            self._own.append(own.value)
        except Exception as e:                      # noqa: BLE001 - reported to every rank below
            err = f"rank {self.rank}: {e}"
        handles = [None] * self.world
        if self.world > 1:
            dist.all_gather_object(handles, None if err else handle.raw, group=self.group)
        ptrs = []
        if err is None and all(h is not None for h in handles if self.world > 1):
            for r in range(self.world):
                if r == self.rank:
                    ptrs.append(own.value)
                    continue
                q = C.c_void_p()
                try:
                    nat.check(nat.lib().rt_peer_open(self.device, handles[r], C.byref(q)))
                except Exception as e:              # noqa: BLE001
                    err = f"rank {self.rank} mapping rank {r}: {e}"
                    break
                self._opened.append(q.value)
                ptrs.append(q.value)
        elif err is None:
            err = f"rank {self.rank}: a peer could not allocate"
        if self.world > 1:
            errs = [None] * self.world
            dist.all_gather_object(errs, err, group=self.group)
            bad = [e for e in errs if e]
            if bad:
                raise nat.NativeLibraryError("peer memory unavailable: " + "; ".join(bad))
        elif err:
            raise nat.NativeLibraryError("peer memory unavailable: " + err)
        self.ptrs[name] = ptrs
        return ptrs

    def signal(self, name, word, targets, epoch, stream=None):
        """Store ``epoch`` into flag word ``word`` of buffer ``name`` on every rank in ``targets`` (after all writes
        this stream issued so far)."""
        import ctypes as C
        nat = self.nat
        tab = (C.c_void_p * len(targets))(*[self.ptrs[name][t] + 4 * int(word) for t in targets])
        nat.check(nat.lib().rt_peer_signal(self.device, tab, len(targets), int(epoch) & 0xFFFFFFFF, stream))

    def wait(self, name, first_word, n, epoch, timed_out=None, timeout_ms=20000, stream=None):
        """Block the stream until the ``n`` local flag words from ``first_word`` have reached ``epoch``."""
        nat = self.nat
        nat.check(nat.lib().rt_peer_wait(self.device, self.ptrs[name][self.rank] + 4 * int(first_word), int(n),
                                         int(epoch) & 0xFFFFFFFF, int(timeout_ms), nat._ptr(timed_out), stream))

    def close(self):
        nat = self.nat
        for q in self._opened:
            nat.load_symbols().rt_peer_close(self.device, q)
        for q in self._own:
            nat.load_symbols().rt_peer_free(self.device, q)
        self._opened, self._own, self.ptrs = [], [], {}


class PendingFrame:
    """A frame on its way to pinned host memory (``to_host="async"``).  ``result()`` waits for the copy and returns the
    numpy view [H,W,3] float32; the view stays valid until the frame after the next one is requested."""

    def __init__(self, host, event):
        self._host, self._event = host, event

    def result(self):
        self._event.synchronize()
        return self._host.numpy()


class ShardedPathRenderer:
    """Algorithm B frames on this rank's GPU, sharded over the process group by tiles or by samples.

    Buffers are torch CUDA tensors (so NCCL can move them); the kernels are launched through the C ABI on torch's
    current stream's device with the tensors' ``data_ptr()``."""

    def __init__(self, device=None, group=None, precision="f32"):
        import torch
        from . import _native as nat
        self.torch, self.nat = torch, nat
        self.group = group
        self.rank, self.world = _world(group)
        self.device = torch.cuda.current_device() if device is None else int(device)
        from .renderers import _precision
        self.precision = _precision(precision)        # 'fp64' / 'float64' / 'double' too; unknown strings raise ValueError
        self.scene = None
        self._key = None
        self.h2d_bytes = self.d2h_bytes = 0
        self.launches = 0

    def set_scene(self, fs, lbvh=None):
        nat = self.nat
        if self.scene is None:
            self.scene = nat.DeviceScene(fs, self.device)
        else:
            self.scene.update(fs)
        n, nG, nP, nL = fs.radius.shape[0], fs.g_strength.shape[0], fs.p_strength.shape[0], fs.l_index.shape[0]
        n_pad, l_pairs = (n + 7) & ~7, (nL + 1) // 2
        # FP32 + FP64 vec4 arrays (sph, sphere pairs, mat, col, lights, light pairs), int arrays, small-light mask
        self.h2d_bytes = ((16 + 32) * (2 * n_pad + 2 * n + 2 * (nG + nP + nL) + 3 * l_pairs)
                          + 2 * 4 * (n + nG + 2 * nP + nL) + n)
        if lbvh or (lbvh is None and self.scene.n > 256):
            self.scene.build_lbvh()

    def _ensure(self, W, H):
        torch = self.torch
        if self._key != (W, H):
            dev = torch.device("cuda", self.device)
            ft = torch.float64 if self.precision == self.nat.F64 else torch.float32
            self.accum = torch.zeros((H, W, 4), dtype=ft, device=dev)
            # device image and pinned host image are double-buffered: with to_host="async" frame f is still being
            # copied out (on the copy stream) while frame f + 1 renders
            self.images = [torch.zeros((H, W, 3), dtype=torch.float32, device=dev) for _ in (0, 1)]
            self.image = self.images[0]
            self.stats = torch.zeros(8, dtype=torch.int64, device=dev)       # uint64 counters, read as int64
            self.host_images = [torch.empty((H, W, 3), dtype=torch.float32, pin_memory=True) for _ in (0, 1)]
            self.host_image = self.host_images[0]
            self._copy_stream = torch.cuda.Stream(device=dev)
            self._copied = [torch.cuda.Event(), torch.cuda.Event()]          # copy of slot k has finished
            self._frame = 0
            self._key = (W, H)

    def _ensure_host_vars(self, W, H):
        """Pinned, double-buffered host slots of the variance image (first variance frame of a size only)."""
        if getattr(self, "_host_var_key", None) != (W, H):
            self.host_vars = [self.torch.empty((H, W, 3), dtype=self.torch.float32, pin_memory=True) for _ in (0, 1)]
            self._host_var_key = (W, H)

    def _ensure_variance(self, W, H):
        """float64 second moments [H,W,4] and double-buffered variance images, allocated by the first variance frame."""
        torch = self.torch
        if getattr(self, "_var_key", None) != (W, H):
            dev = torch.device("cuda", self.device)
            self.moments = torch.zeros((H, W, 4), dtype=torch.float64, device=dev)
            self.vars = [torch.zeros((H, W, 3), dtype=torch.float32, device=dev) for _ in (0, 1)]
            self._var_key = (W, H)
        self._ensure_host_vars(W, H)

    def _ensure_features(self, W, H):
        """First-hit feature buffers (albedo [H,W,3], normal [H,W,3], depth [H,W], fvar [H,W,3] float32), allocated by
        the first feature frame."""
        torch = self.torch
        if getattr(self, "_feat_key", None) != (W, H):
            dev = torch.device("cuda", self.device)
            self.features = tuple(torch.zeros(s, dtype=torch.float32, device=dev)
                                  for s in ((H, W, 3), (H, W, 3), (H, W), (H, W, 3)))
            self._feat_key = (W, H)

    def _to_host(self, src, slot, release=None, var=None):
        """Queue the device->host copy of ``src`` (and of the variance image ``var``, if given) on the copy stream (after
        everything the current stream has queued) into pinned slot ``slot``; ``release`` (optional) runs on the copy
        stream after the copies.  -> (PendingFrame of the image, PendingFrame of the variance or None)."""
        torch = self.torch
        ready = torch.cuda.Event()
        ready.record()
        cs = self._copy_stream
        cs.wait_event(ready)
        with torch.cuda.stream(cs):
            self.host_images[slot].copy_(src, non_blocking=True)
            if var is not None:
                self.host_vars[slot].copy_(var, non_blocking=True)
            # the frame is on the host once the COPY is done: the event must not sit behind the release launch, which
            # (a kernel) cannot start while the next frame's persistent kernel holds every SM -- it would report the
            # frame a whole frame late and stall a caller that reads frame f before it issues frame f + 2
            self._copied[slot].record(cs)
            if release is not None:
                release(cs.cuda_stream)
        self.d2h_bytes = self.host_images[slot].numel() * 4 * (1 if var is None else 2)
        return (PendingFrame(self.host_images[slot], self._copied[slot]),
                None if var is None else PendingFrame(self.host_vars[slot], self._copied[slot]))

    def _deliver(self, image, var, slot, to_host, release=None):
        """Rank 0's (image, variance or None) in the form ``to_host`` asks for."""
        if not to_host:
            return image, var
        pi, pv = self._to_host(image, slot, release, var)
        if to_host == "async":
            return pi, pv
        return pi.result(), (None if pv is None else pv.result())

    def render(self, cam, W, H, spp, max_bounces, mirror_threshold, seed=0, fov=60.0, mode="tiles", to_host=False,
               variance=False, denoise=False, features=False, denoise_params=None):
        """Render one frame cooperatively.  Returns (image, stats) on rank 0 -- image a CUDA tensor [H,W,3] float32, a
        numpy view of pinned host memory when ``to_host`` is True, or a ``PendingFrame`` when ``to_host == "async"``
        (the copy runs on a second stream while the next frame renders) -- and (None, stats) elsewhere.  stats = this
        rank's uint64[8] counter block as a CUDA int64 tensor (not reduced: callers sum what they need).

        ``variance=True`` (the same on every rank of a frame): also the variance of each pixel's mean in colour
        levels^2, [H,W,3] float32, bit-identical to ``render_path(..., variance=True)`` of the unsharded frame.  The
        call then returns (image, stats, var) on rank 0, var of the same kind as image, and (None, stats, None)
        elsewhere.

        ``denoise=True`` (DESIGN §4.8e): the image is the frame filtered by the variance-guided non-local-means filter,
        bit-identical to ``FrameContext.render_path(..., denoise=True)``.  Every rank forms the final sums of its row
        band (samples mode: ``reduce_row_bands`` of the sums and moments in place of the reduce to rank 0), resolves
        its band's variance, exchanges the halo rows of both with its neighbours and filters its band
        (``DeviceScene.denoise(rows=)``); rank 0 gathers the bands.  ``features=True`` (needs ``denoise``): the
        feature-guided filter, each rank rendering the first-hit features of its window rows over the samples
        [0, min(spp, FrameContext.FEATURE_SPP)).  ``denoise_params``: a dict of ``DeviceScene.denoise``'s keywords
        (radius, patch_radius, k, k_f, tau); None: the library defaults.  The return shape does not change."""
        torch, nat, sc = self.torch, self.nat, self.scene
        if features and not denoise:
            raise ValueError("features=True needs denoise=True: the sharded renderer does not gather the feature buffers")
        dparams = dict(denoise_params or {})
        if denoise:
            # the halo depth, from the library; also rejects a bad radius / patch_radius before any collective
            halo = nat.denoise_halo(features=features, **{k: dparams[k] for k in ("radius", "patch_radius") if k in dparams})
        self._ensure(W, H)
        if variance or denoise:
            self._ensure_variance(W, H)
        if features:
            self._ensure_features(W, H)
        self._frame += 1
        slot = self._frame & 1
        self.image = self.images[slot]
        var = self.vars[slot] if (variance or denoise) else None
        moments = self.moments if (variance or denoise) else None
        torch.cuda.current_stream().wait_event(self._copied[slot])         # slot's previous copy-out has finished
        rows = (0, H)
        samples = (0, spp)
        if mode == "tiles":
            bands = row_bands(H, self.world)
            rows = bands[self.rank]
        elif mode == "samples":
            samples = sample_ranges(spp, self.world)[self.rank]
        else:
            raise ValueError("mode must be 'tiles' or 'samples'")
        self.stats.zero_()
        if mode == "samples" and samples[0] == samples[1]:
            self.accum.zero_()
            if moments is not None:
                moments.zero_()
        p = sc.path_params(cam, W, H, spp, max_bounces, mirror_threshold, seed=seed, fov=fov, rows=rows, samples=samples)
        sc.render_path(p, self.accum, self.precision, stats=self.stats, moments=moments)
        self.launches = 1
        if denoise:
            self._denoise_bands(cam, W, H, spp, seed, fov, mode, var, halo, features, dparams)
            gather_row_bands(self.image, row_bands(H, self.world), self.group)
            if variance:
                gather_row_bands(var, row_bands(H, self.world), self.group)
            else:
                var = None
        elif mode == "tiles":
            sc.resolve(self.accum, W, H, spp, self.image, self.precision, rows=rows)
            self.launches += 1
            if variance:
                sc.resolve_variance(self.accum, moments, W, H, var, self.precision, rows=rows)
                self.launches += 1
            gather_row_bands(self.image, bands, self.group)
            if variance:
                gather_row_bands(var, bands, self.group)
        else:
            reduce_sample_sums(self.accum, self.group)
            if variance:
                reduce_sample_sums(moments, self.group)
            if self.rank == 0:
                sc.resolve(self.accum, W, H, spp, self.image, self.precision)
                self.launches += 1
                if variance:
                    sc.resolve_variance(self.accum, moments, W, H, var, self.precision)
                    self.launches += 1
        if self.rank != 0:
            return (None, self.stats, None) if variance else (None, self.stats)
        image, var = self._deliver(self.image, var, slot, to_host)
        return (image, self.stats, var) if variance else (image, self.stats)

    def _denoise_bands(self, cam, W, H, spp, seed, fov, mode, var, halo, features, dparams):
        """The denoised frame's steps after the render: this rank's band sums and variance, the halo exchange, its
        window's features and the band filter into ``self.image``."""
        sc, prec = self.scene, self.precision
        bands = row_bands(H, self.world)
        y0, y1 = bands[self.rank]
        if mode == "samples":
            reduce_row_bands(self.accum, bands, self.group)
            reduce_row_bands(self.moments, bands, self.group)
        if y1 > y0:
            sc.resolve_variance(self.accum, self.moments, W, H, var, prec, rows=(y0, y1))
            self.launches += 1
        exchange_halos([self.accum, var], halo_plan(H, self.world, halo), self.group)
        lo, hi = halo_windows(H, self.world, halo)[self.rank]
        if features and hi > lo:
            # the feature kernel is per pixel: rendering the window rows here equals exchanging them
            from .frames import FrameContext
            p = sc.path_params(cam, W, H, spp, 1, 0.0, seed=seed, fov=fov, rows=(lo, hi),
                               samples=(0, min(int(spp), FrameContext.FEATURE_SPP)))
            sc.render_features(p, *self.features, precision=prec)
            self.launches += 1
        if y1 > y0:
            sc.denoise(self.accum, var, W, H, self.image, prec, rows=(y0, y1),
                       features=self.features if features else None, **dparams)
            self.launches += 1

    # ---- fused sinks over NVLink peer memory ------------------------------------------------------------------
    def _ensure_fabric(self, W, H):
        """Peer-mapped, double-buffered frame storage: the final image on rank 0, one accumulator per rank, flags."""
        torch = self.torch
        if getattr(self, "_fab_key", None) == (W, H):
            return
        if getattr(self, "fabric", None) is not None:
            self.fabric.close()
        fab = self.fabric = PeerFabric(self.device, self.group)
        fab.alloc("image0", H * W * 3 * 4); fab.alloc("image1", H * W * 3 * 4)
        fab.alloc("accum0", H * W * 16); fab.alloc("accum1", H * W * 16)
        fab.alloc("flags", 4 * 64)          # words 0..15 added[rank], 16..31 done[rank], 32 go
        self._epoch = 0
        self._timed_out = torch.zeros(1, dtype=torch.int32, device=torch.device("cuda", self.device))
        self._fused_images = [torch.as_tensor(_DevArray(fab.ptrs[f"image{k}"][self.rank], (H, W, 3), "<f4"),
                                              device=torch.device("cuda", self.device)) for k in (0, 1)]
        if not hasattr(self, "host_image") or self._key != (W, H):
            self._ensure(W, H)
        self._fab_key = (W, H)
        self._fab_var = False

    def _ensure_fabric_variance(self, W, H):
        """Peer-mapped, double-buffered second moments (one [H,W,4] float64 per rank) and variance images (rank 0's),
        allocated by the first variance frame.  Collective, like the frame itself; freshly zeroed, and the epochs and
        flags of the existing buffers are left as they are."""
        if self._fab_var:
            return
        torch, fab = self.torch, self.fabric
        fab.alloc("moments0", H * W * 32); fab.alloc("moments1", H * W * 32)
        fab.alloc("var0", H * W * 3 * 4); fab.alloc("var1", H * W * 3 * 4)
        self._fused_vars = [torch.as_tensor(_DevArray(fab.ptrs[f"var{k}"][self.rank], (H, W, 3), "<f4"),
                                            device=torch.device("cuda", self.device)) for k in (0, 1)]
        self._ensure_host_vars(W, H)
        self._fab_var = True

    def render_fused(self, cam, W, H, spp, max_bounces, mirror_threshold, seed=0, fov=60.0, mode="tiles", to_host=False,
                     kernel_events=None, in_kernel=True, variance=False):
        """The same frame as ``render`` with the collective fused into the path kernel: no NCCL call on the data path.

        tiles    every rank renders interleaved 8-row stripes (tile_stripes) and its path kernel stores the resolved
                 float32 pixels straight into rank 0's image through the NVLink peer mapping.
        samples  every rank renders its sample range of all pixels; the path kernel's epilogue adds each pixel's sums
                 into the accumulators of the rank that owns the pixel's row band (one 16-byte system-scope reduction
                 per pixel: a reduce-scatter), then every rank resolves its band into rank 0's image.
        Ordering across ranks: epoch flags in peer memory.  ``in_kernel=True`` (default): the whole protocol -- wait
        for free buffers, render, publish, resolve the own band, collect on rank 0 -- runs inside ONE launch per rank
        (``rt_path_sink.sync``); ``False``: the round-1 chain of small wait / signal / resolve launches around the
        path kernel (kept for comparison).  Frames are double-buffered so rank 0 can still be reading frame f while
        frame f+1 is written: a returned CUDA image stays valid until the frame after the next one is rendered,
        PROVIDED its consumer is queued on the current stream before the next ``render_fused`` call (the "consumed"
        signal of frame f is published by rank 0's stream at the start of frame f+1, i.e. after everything queued in
        between; with ``to_host`` it follows the copy-out on the copy stream).  kernel_events = (start, end) CUDA
        events recorded around the path kernel alone (bench.py's roofline).

        ``variance=True``: the per-pixel variance travels through the same sinks -- tiles: the path kernel also stores
        each resolved pixel's variance into rank 0's variance image; samples: it also adds the squared colours into the
        owner's float64 moments, which the band resolve turns into rank 0's variance image.  Returns (image, stats,
        var) as ``render`` does.  Like ``mode``, ``variance`` must be the same on every rank for a given frame."""
        nat, sc, torch = self.nat, self.scene, self.torch
        if mode not in ("tiles", "samples"):
            raise ValueError("mode must be 'tiles' or 'samples'")
        self._ensure_fabric(W, H)
        if variance:
            self._ensure_fabric_variance(W, H)
        fab, rank, world = self.fabric, self.rank, self.world
        self._epoch += 1
        e, buf = self._epoch, self._epoch & 1
        everyone = list(range(world))
        self.stats.zero_()
        p = sc.path_params(cam, W, H, spp, max_bounces, mirror_threshold, seed=seed, fov=fov)
        sink = nat.PathSink()
        bands = row_bands(H, world)
        s0, s1 = sample_ranges(spp, world)[rank] if mode == "samples" else (0, spp)
        if mode == "tiles":
            sink.mode, sink.tile_first, sink.tile_step = nat.SINK_IMAGE, rank, world
            # 2-D interleave (one column segment of EVERY stripe) when the width allows it: equal pixel counts per rank
            # whatever the height (1080 rows are 135 stripes: 17 or 16 per rank of 8 = 0.7 % of imbalance)
            sink.col_split = 1 if W % world == 0 else 0      # (the library falls back to stripes if a segment cannot hold its work units)
        else:
            p.s0, p.s1 = s0, s1
            sink.mode = nat.SINK_SCATTER_ADD
            for k in range(world):
                sink.accum[k] = fab.ptrs[f"accum{buf}"][k]
                sink.band_y[k] = bands[k][0]
            sink.band_y[world] = H
        sink.world = world
        sink.image = fab.ptrs[f"image{buf}"][0]
        msink = None
        if variance:
            msink = nat.PathMomentsSink()
            msink.var = fab.ptrs[f"var{buf}"][0]
            if mode == "samples":
                for k in range(world):
                    msink.moments[k] = fab.ptrs[f"moments{buf}"][k]
        pending_go, self._pending_go = getattr(self, "_pending_go", 0), 0
        if in_kernel:
            sink.sync, sink.rank, sink.epoch, sink.spp_total = 1, rank, e, spp
            sink.go_epoch = pending_go if rank == 0 else 0
            for k in range(world):
                sink.flags[k] = fab.ptrs["flags"][k]
            sink.timed_out = self._timed_out.data_ptr()
            if kernel_events:
                kernel_events[0].record()
            sc.render_path_sink(p, sink, stats=self.stats, moments_sink=msink)   # ONE launch: the frame is complete on rank 0 when it ends
            if kernel_events:
                kernel_events[1].record()
            self.launches = 1
        else:
            if rank == 0 and pending_go:
                fab.signal("flags", 32, everyone, pending_go)                  # after whatever the caller queued on frame e - 1
            fab.wait("flags", 32, 1, e - 2, self._timed_out)                  # rank 0 has consumed this image buffer
            if mode == "tiles":
                if kernel_events:
                    kernel_events[0].record()
                sc.render_path_sink(p, sink, stats=self.stats, moments_sink=msink)
                if kernel_events:
                    kernel_events[1].record()
                self.launches = 3 + (2 if rank == 0 else 0)
            else:
                if kernel_events:
                    kernel_events[0].record()
                if s1 > s0:
                    sc.render_path_sink(p, sink, stats=self.stats, moments_sink=msink)
                if kernel_events:
                    kernel_events[1].record()
                fab.signal("flags", rank, everyone, e)                         # my sums have been added everywhere
                fab.wait("flags", 0, world, e, self._timed_out)                # everyone's sums are in my band
                y0, y1 = bands[rank]
                if variance:
                    nat.check(nat.lib().rt_resolve_clear_moments(self.device, fab.ptrs[f"accum{buf}"][rank],
                                                                 fab.ptrs[f"moments{buf}"][rank], W, H, y0, y1, spp,
                                                                 fab.ptrs[f"image{buf}"][0], fab.ptrs[f"var{buf}"][0], 1,
                                                                 None))
                else:
                    nat.check(nat.lib().rt_resolve_clear(self.device, fab.ptrs[f"accum{buf}"][rank], W, H, y0, y1, spp,
                                                         fab.ptrs[f"image{buf}"][0], 1, None))
                self.launches = 6 + (2 if rank == 0 else 0)     # wait, path, signal, wait, resolve, signal (+ wait, signal)
            fab.signal("flags", 16 + rank, [0], e)                             # my part of rank 0's image is written
            if rank == 0:
                fab.wait("flags", 16, world, e, self._timed_out)
        out = var = None
        if rank == 0:
            out, var = self._fused_images[buf], (self._fused_vars[buf] if variance else None)
            if to_host:
                # the copy-out runs on the copy stream; the "consumed" signal follows it there
                out, var = self._deliver(out, var, buf, to_host,
                                         release=lambda st: fab.signal("flags", 32, everyone, e, stream=st))
            else:
                # the caller's consumer of this CUDA image comes AFTER this call: publish "consumed" at the start of the
                # next frame on this stream (in the kernel's own prologue), never right away
                self._pending_go = e
        return (out, self.stats, var) if variance else (out, self.stats)

    def fused_timed_out(self):
        return bool(int(self._timed_out.item())) if getattr(self, "_timed_out", None) is not None else False

    def close(self):
        if getattr(self, "fabric", None) is not None:
            self.fabric.close()
            self.fabric = None
        if self.scene is not None:
            self.scene.close()
            self.scene = None
