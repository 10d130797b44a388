"""ctypes binding of ``csrc/librt_b200.so`` (C ABI: include/rt_b200.h).

This is the only door between the Python scene API and the CUDA kernels.  There is
NO CPU fallback: if the shared library is missing, or no CUDA device is present, every
tracing call raises ``NativeLibraryError``.

Device memory handed across the ABI is either owned by the library helpers below
(``DeviceBuffer``: ``rt_dev_alloc``) or a torch CUDA tensor's ``data_ptr()``
(the batched env hands observations to agents as tensors).
"""
import ctypes as C
import os
import subprocess
import threading

import numpy as np

__all__ = ["NativeLibraryError", "lib", "build", "DeviceBuffer", "PinnedArray", "DeviceScene", "device_count", "device_props",
           "measure_fp32_peak", "F32", "F64", "NO_ID", "REASONS", "LIB_PATH"]

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.environ.get("RT_B200_LIB") or os.path.join(CSRC, "librt_b200.so")      # override: kernel A/B builds

F32, F64 = 0, 1
NO_ID = -(2 ** 31)
REASONS = {0: None, 1: "ray_missed", 2: "ray_escaped", 3: "max_bounces", 4: "hit_sun", 5: "already_on_sun"}
ENV_RL, ENV_FB = 0, 1

c_dp = C.POINTER(C.c_double)
c_ip = C.POINTER(C.c_int32)
c_u8p = C.POINTER(C.c_uint8)
vp = C.c_void_p


class NativeLibraryError(RuntimeError):
    """librt_b200.so is missing / failed to load / reported an error.  Never caught to fall back to the CPU."""


class SceneDesc(C.Structure):
    # the array members are `const double *` / `const int32_t *` / `const uint8_t *` in rt_scene_desc; declared as void
    # pointers here so that make_desc can store raw addresses (a typed ctypes cast costs ~2 us per field, x 20 fields,
    # on every frame of a 30-us render)
    _fields_ = [
        ("n", C.c_int32), ("centre", vp), ("radius", vp), ("material", vp), ("colour", vp), ("ids", vp),
        ("nG", C.c_int32), ("g_vec", vp), ("g_col", vp), ("g_strength", vp), ("g_max_angle", vp), ("g_func", vp),
        ("nP", C.c_int32), ("p_id", vp), ("p_pos", vp), ("p_col", vp), ("p_strength", vp), ("p_max_angle", vp),
        ("p_func", vp),
        ("bg", C.c_double * 3),
        ("nL", C.c_int32), ("l_centre", vp), ("l_colour", vp), ("l_index", vp), ("small", vp),
    ]


class WhittedParams(C.Structure):
    _fields_ = [("cam", C.c_double * 3), ("X", c_dp), ("Y", c_dp), ("W", C.c_int32), ("H", C.c_int32),
                ("y0", C.c_int32), ("y1", C.c_int32), ("s0", C.c_int32), ("s1", C.c_int32), ("spp", C.c_int32),
                ("max_bounces", C.c_int32), ("shadow_max_bounces", C.c_int32), ("miss", C.c_double * 3),
                ("seed", C.c_uint64), ("prenormalise", C.c_int32), ("accumulate", C.c_int32)]


class PathParams(C.Structure):
    _fields_ = [("cam", C.c_double * 3), ("W", C.c_int32), ("H", C.c_int32), ("fov_deg", C.c_double),
                ("y0", C.c_int32), ("y1", C.c_int32), ("s0", C.c_int32), ("s1", C.c_int32), ("max_bounces", C.c_int32),
                ("mirror_threshold", C.c_double), ("seed", C.c_uint64), ("accumulate", C.c_int32),
                ("schedule", C.c_int32), ("ksplit", C.c_int32), ("reserved_", C.c_int32)]


class AdaptiveParams(C.Structure):
    """rt_adaptive_params: samples [0, min_spp) for every pixel, then doubling rounds for the pixels whose variance of the
    mean exceeds ``tolerance``^2 (colour levels, 0-255 scale; negative: every pixel to max_spp)."""
    _fields_ = [("min_spp", C.c_int32), ("reserved_", C.c_int32), ("tolerance", C.c_double)]


class DenoiseParams(C.Structure):
    """rt_denoise_params: the variance-guided non-local-means filter's search radius, patch radius and k."""
    _fields_ = [("radius", C.c_int32), ("patch_radius", C.c_int32), ("k", C.c_float), ("reserved_", C.c_int32)]


class DenoiseFeaturesParams(C.Structure):
    """rt_denoise_features_params: rt_denoise_params plus the feature term's k_f and tau."""
    _fields_ = [("radius", C.c_int32), ("patch_radius", C.c_int32), ("k", C.c_float), ("k_f", C.c_float),
                ("tau", C.c_float), ("reserved_", C.c_int32)]


class SimpleParams(C.Structure):
    _fields_ = [("cam", C.c_double * 3), ("W", C.c_int32), ("H", C.c_int32), ("fov_rad", C.c_double),
                ("sun_pos", C.c_double * 3), ("sun_col", C.c_double * 3), ("sun_id", C.c_int32), ("max_bounces", C.c_int32),
                ("seed", C.c_uint64), ("m", C.c_int32), ("lighting_only", C.c_int32), ("rays_dev", C.c_void_p)]


RT_MAX_PEERS, IPC_HANDLE_BYTES = 16, 64
SINK_ACCUM, SINK_IMAGE, SINK_SCATTER_ADD = 0, 1, 2


class PathSink(C.Structure):
    _fields_ = [("mode", C.c_int32), ("world", C.c_int32), ("tile_first", C.c_int32), ("tile_step", C.c_int32),
                ("image", C.c_void_p), ("accum", C.c_void_p * RT_MAX_PEERS), ("band_y", C.c_int32 * (RT_MAX_PEERS + 1)),
                ("sync", C.c_int32), ("rank", C.c_int32), ("epoch", C.c_uint32), ("go_epoch", C.c_uint32),
                ("flags", C.c_void_p * RT_MAX_PEERS), ("timed_out", C.c_void_p), ("timeout_ms", C.c_int32),
                ("max_ctas", C.c_int32), ("spp_total", C.c_int32), ("col_split", C.c_int32)]


class PathMomentsSink(C.Structure):
    """rt_path_moments_sink: where the fused sinks put the second moments (image sink: ``var``; scatter-add sink:
    ``moments[k]`` of every owner, and ``var`` under ``sync``)."""
    _fields_ = [("moments", C.c_void_p * RT_MAX_PEERS), ("var", C.c_void_p)]


FLAG_WORDS = 64


class EnvDesc(C.Structure):
    _fields_ = [("B", C.c_int32), ("W", C.c_int32), ("H", C.c_int32), ("cam", C.c_double * 3),
                ("cam_angle", C.c_double * 3), ("fov", C.c_double), ("max_bounces", C.c_int32),
                ("flavour", C.c_int32), ("sun_id", C.c_int32), ("reward_mode", C.c_int32), ("light_ids", C.c_int32 * 2),
                ("env_offset", C.c_int32), ("reserved_", C.c_int32)]


# every symbol include/rt_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "rt_last_error": (C.c_char_p, []),
    "rt_version": (C.c_int, []),
    "rt_device_count": (C.c_int, [c_ip]),
    "rt_device_props": (C.c_int, [C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_size_t)]),
    "rt_dev_alloc": (C.c_int, [C.c_int, C.c_size_t, C.POINTER(vp)]),
    "rt_dev_free": (C.c_int, [C.c_int, vp]),
    "rt_host_alloc_pinned": (C.c_int, [C.c_size_t, C.POINTER(vp)]),
    "rt_host_free_pinned": (C.c_int, [vp]),
    "rt_memcpy_h2d": (C.c_int, [C.c_int, vp, vp, C.c_size_t, vp]),
    "rt_memcpy_d2h": (C.c_int, [C.c_int, vp, vp, C.c_size_t, vp]),
    "rt_memset_dev": (C.c_int, [C.c_int, vp, C.c_int, C.c_size_t, vp]),
    "rt_stream_sync": (C.c_int, [C.c_int, vp]),
    "rt_stream_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
    "rt_stream_destroy": (C.c_int, [C.c_int, vp]),
    "rt_stream_wait_stream": (C.c_int, [C.c_int, vp, vp]),
    "rt_measure_fp32_peak": (C.c_int, [C.c_int, C.c_int, c_dp, c_dp]),
    "rt_scene_create": (C.c_int, [C.c_int, C.POINTER(SceneDesc), C.POINTER(vp)]),
    "rt_scene_update": (C.c_int, [vp, C.POINTER(SceneDesc), vp]),
    "rt_scene_destroy": (C.c_int, [vp]),
    "rt_scene_info": (C.c_int, [vp, c_ip, c_ip, c_ip]),
    "rt_lbvh_build": (C.c_int, [vp, C.c_double, vp]),
    "rt_lbvh_drop": (C.c_int, [vp]),
    "rt_sphere_discriminant": (C.c_int, [C.c_int, C.c_int, C.c_int, vp, vp, C.c_int, vp, vp]),
    "rt_trace_rays": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, vp, vp, C.c_int, C.c_int, c_dp, vp, vp, vp]),
    "rt_terminal_rgb": (C.c_int, [vp, C.c_int, C.c_int, vp, C.c_int, vp, vp]),
    "rt_render_whitted": (C.c_int, [vp, C.c_int, C.POINTER(WhittedParams), vp, vp, vp, vp]),
    "rt_render_path": (C.c_int, [vp, C.c_int, C.POINTER(PathParams), vp, vp, vp]),
    "rt_render_path_moments": (C.c_int, [vp, C.c_int, C.POINTER(PathParams), vp, vp, vp, vp]),
    "rt_render_path_adaptive": (C.c_int, [vp, C.c_int, C.POINTER(PathParams), C.POINTER(AdaptiveParams), vp, vp, vp, vp, vp,
                                          vp, vp, vp]),
    "rt_trace_paths": (C.c_int, [vp, C.c_int, C.POINTER(PathParams), C.c_int32, vp, vp, C.c_int32, vp, vp, vp]),
    "rt_resolve": (C.c_int, [C.c_int, C.c_int, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp, vp]),
    "rt_resolve_variance": (C.c_int, [C.c_int, C.c_int, vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp, vp]),
    "rt_denoise": (C.c_int, [C.c_int, C.c_int, vp, vp, C.c_int32, C.c_int32, C.POINTER(DenoiseParams), vp, vp]),
    "rt_render_features": (C.c_int, [vp, C.c_int, C.POINTER(PathParams), vp, vp, vp, vp, vp]),
    "rt_denoise_features": (C.c_int, [C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, C.c_int32, C.c_int32,
                                      C.POINTER(DenoiseFeaturesParams), vp, vp]),
    "rt_denoise_rows": (C.c_int, [C.c_int, C.c_int, vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                  C.POINTER(DenoiseParams), vp, vp]),
    "rt_denoise_features_rows": (C.c_int, [C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, C.c_int32, C.c_int32, C.c_int32,
                                           C.c_int32, C.POINTER(DenoiseFeaturesParams), vp, vp]),
    "rt_denoise_halo": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, c_ip]),
    "rt_wf_create": (C.c_int, [vp, C.c_int, C.c_int32, C.c_int32, C.POINTER(vp)]),
    "rt_wf_destroy": (C.c_int, [vp]),
    "rt_wf_begin": (C.c_int, [vp, C.POINTER(PathParams), C.c_double, vp, vp]),
    "rt_wf_trace": (C.c_int, [vp, vp, vp, vp, vp]),
    "rt_wf_bounce": (C.c_int, [vp, vp, vp, vp, vp, vp]),
    "rt_wf_finish": (C.c_int, [vp, vp, vp]),
    "rt_wf_finish_moments": (C.c_int, [vp, vp, vp, vp]),
    "rt_generate_trajectories": (C.c_int, [vp, C.c_int, C.c_int32, C.c_int32, C.c_int32, C.c_uint64, vp, vp, vp, vp, vp, vp, vp,
                                            vp, vp]),
    "rt_render_simple": (C.c_int, [vp, C.c_int, C.POINTER(SimpleParams), vp, vp, vp, vp]),
    "rt_render_simple_host": (C.c_int, [vp, C.c_int, C.POINTER(SimpleParams), vp, vp, vp, vp]),
    "rt_render_path_sink": (C.c_int, [vp, C.POINTER(PathParams), C.POINTER(PathSink), vp, vp]),
    "rt_resolve_clear": (C.c_int, [C.c_int, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp, C.c_int32, vp]),
    "rt_render_path_sink_moments": (C.c_int, [vp, C.POINTER(PathParams), C.POINTER(PathSink), C.POINTER(PathMomentsSink), vp,
                                              vp]),
    "rt_resolve_clear_moments": (C.c_int, [C.c_int, vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp, vp,
                                           C.c_int32, vp]),
    "rt_peer_alloc": (C.c_int, [C.c_int, C.c_size_t, C.POINTER(vp), C.c_char_p]),
    "rt_peer_open": (C.c_int, [C.c_int, C.c_char_p, C.POINTER(vp)]),
    "rt_peer_close": (C.c_int, [C.c_int, vp]),
    "rt_peer_free": (C.c_int, [C.c_int, vp]),
    "rt_peer_signal": (C.c_int, [C.c_int, C.POINTER(vp), C.c_int32, C.c_uint32, vp]),
    "rt_peer_wait": (C.c_int, [C.c_int, vp, C.c_int32, C.c_uint32, C.c_int32, vp, vp]),
    "rt_render_whitted_host": (C.c_int, [vp, C.c_int, C.POINTER(WhittedParams), vp, vp, vp, vp]),
    "rt_render_path_host": (C.c_int, [vp, C.c_int, C.POINTER(PathParams), vp, vp, vp]),
    "rt_env_create": (C.c_int, [vp, C.c_int, C.POINTER(EnvDesc), C.POINTER(vp)]),
    "rt_env_destroy": (C.c_int, [vp]),
    "rt_env_reset": (C.c_int, [vp, vp, vp, C.c_uint64, vp, vp, vp]),
    "rt_env_step": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "rt_env_step_auto": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_uint64, vp, vp]),
}

_lib = None
_lock = threading.Lock()


def build(force=False, verbose=False):
    """Compile csrc/ for sm_100a with the committed Makefile (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC, "-j4"] + (["-B"] if force else [])
    res = subprocess.run(cmd, capture_output=not verbose, text=True)
    if res.returncode != 0:
        raise NativeLibraryError("building librt_b200.so failed:\n" + (res.stdout or "") + (res.stderr or ""))
    return LIB_PATH


def load_symbols():
    """dlopen the library and bind every declared symbol.  Needs no GPU (used by the CPU-side ABI test)."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise NativeLibraryError(
                    f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                    "(there is no CPU fallback)")
            try:
                handle = C.CDLL(LIB_PATH)
            except OSError as e:
                raise NativeLibraryError(f"cannot load {LIB_PATH}: {e}") from e
            for name, (res, args) in SIGNATURES.items():
                try:
                    fn = getattr(handle, name)
                except AttributeError as e:
                    raise NativeLibraryError(f"{LIB_PATH} does not export {name}") from e
                fn.restype, fn.argtypes = res, args
            _lib = handle
    return _lib


def lib():
    """The loaded library, after checking that a CUDA device is present."""
    h = load_symbols()
    if not getattr(h, "_rt_checked", False):
        n = C.c_int32(0)
        rc = h.rt_device_count(C.byref(n))
        if rc != 0 or n.value <= 0:
            raise NativeLibraryError("no CUDA device: the B200 kernels cannot run here and there is no CPU fallback "
                                     f"({h.rt_last_error().decode()})")
        h._rt_checked = True
    return h


def check(rc):
    if rc != 0:
        raise NativeLibraryError(f"librt_b200 error {rc}: {load_symbols().rt_last_error().decode()}")


def device_count():
    n = C.c_int32(0)
    load_symbols().rt_device_count(C.byref(n))
    return int(n.value)


def device_props(device=0):
    p = (C.c_int64 * 6)()
    mem = C.c_size_t(0)
    check(lib().rt_device_props(device, p, C.byref(mem)))
    return {"sm_count": int(p[0]), "cc": (int(p[1]), int(p[2])), "sm_clock_khz": int(p[3]), "l2_bytes": int(p[4]),
            "smem_optin": int(p[5]), "total_mem": int(mem.value)}


def measure_fp32_peak(device=0, repeats=5):
    """FFMA micro-benchmark -> (TFLOP/s, ms).  The FP32 roofline denominator measured on the box."""
    tf, ms = C.c_double(0), C.c_double(0)
    check(lib().rt_measure_fp32_peak(device, repeats, C.byref(tf), C.byref(ms)))
    return float(tf.value), float(ms.value)


def denoise_halo(radius=10, patch_radius=3, features=False):
    """The halo depth h of the filter (``rt_denoise_halo``): the rows an output row reads lie within h of it, so a row
    band [y0, y1) of ``DeviceScene.denoise(..., rows=)`` reads only rows [y0 - h, y1 + h) of the frame.  Needs no GPU."""
    h = C.c_int32(0)
    check(load_symbols().rt_denoise_halo(int(radius), int(patch_radius), int(bool(features)), C.byref(h)))
    return int(h.value)


def _ptr(x):
    """Device pointer of a DeviceBuffer / torch tensor / int / None."""
    if x is None:
        return None
    if isinstance(x, DeviceBuffer):
        return x.ptr
    if isinstance(x, int):
        return x
    if hasattr(x, "data_ptr"):
        return x.data_ptr()
    raise TypeError(f"not a device buffer: {type(x)!r}")


class DeviceBuffer:
    """A typed block of HBM owned through rt_dev_alloc / rt_dev_free."""

    def __init__(self, shape, dtype, device=0, zero=True):
        self.shape = tuple(int(s) for s in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        self.dtype = np.dtype(dtype)
        self.device = device
        self.nbytes = int(np.prod(self.shape, dtype=np.int64)) * self.dtype.itemsize
        p = vp()
        check(lib().rt_dev_alloc(device, max(self.nbytes, 1), C.byref(p)))
        self.ptr = p.value
        if zero and self.nbytes:
            check(lib().rt_memset_dev(device, self.ptr, 0, self.nbytes, None))

    @classmethod
    def from_host(cls, array, dtype=None, device=0):
        a = np.ascontiguousarray(array, dtype)
        buf = cls(a.shape, a.dtype, device, zero=False)
        buf.upload(a)
        return buf

    def upload(self, array, stream=None):
        a = np.ascontiguousarray(array, self.dtype)
        assert a.nbytes == self.nbytes, (a.shape, self.shape)
        if self.nbytes:
            check(lib().rt_memcpy_h2d(self.device, self.ptr, a.ctypes.data, self.nbytes, stream))
            check(lib().rt_stream_sync(self.device, stream))

    def fill(self, byte=0, stream=None):
        if self.nbytes:
            check(lib().rt_memset_dev(self.device, self.ptr, byte, self.nbytes, stream))

    def download(self, stream=None):
        out = np.empty(self.shape, self.dtype)
        if self.nbytes:
            check(lib().rt_memcpy_d2h(self.device, out.ctypes.data, self.ptr, self.nbytes, stream))
            check(lib().rt_stream_sync(self.device, stream))
        return out

    def free(self):
        if getattr(self, "ptr", None):
            try:
                load_symbols().rt_dev_free(self.device, self.ptr)
            finally:
                self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class PinnedArray:
    """Page-locked host memory (rt_host_alloc_pinned) viewed as a numpy array: the staging end of D2H / H2D copies."""

    def __init__(self, shape, dtype):
        self.shape = tuple(int(s) for s in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        self.dtype = np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape, dtype=np.int64)) * self.dtype.itemsize
        p = vp()
        check(lib().rt_host_alloc_pinned(max(self.nbytes, 1), C.byref(p)))
        self.ptr = p.value
        raw = (C.c_byte * max(self.nbytes, 1)).from_address(self.ptr)
        self.array = np.frombuffer(raw, dtype=self.dtype, count=int(np.prod(self.shape, dtype=np.int64))).reshape(self.shape)

    def free(self):
        if getattr(self, "ptr", None):
            self.array = None
            try:
                load_symbols().rt_host_free_pinned(self.ptr)
            finally:
                self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _d(a, shape=None):
    a = np.ascontiguousarray(a, np.float64)
    return a if shape is None else a.reshape(shape)


def _i(a):
    return np.ascontiguousarray(a, np.int32)


_F64, _I32 = np.dtype(np.float64), np.dtype(np.int32)
_DESC_F = ("centre", "radius", "material", "colour", "g_vec", "g_col", "g_strength", "g_max_angle", "p_pos", "p_col",
           "p_strength", "p_max_angle", "l_centre", "l_colour")
_DESC_I = ("ids", "g_func", "p_id", "p_func", "l_index")


def _as(a, dt):
    """``a`` as a C-contiguous array of dtype ``dt`` (no copy when it already is one: the FlatScene arrays are)."""
    if type(a) is np.ndarray and a.dtype == dt and a.flags.c_contiguous:
        return a
    return np.ascontiguousarray(a, dt)


def make_desc(fs):
    """FlatScene (scene.py) -> (SceneDesc, keep-alive dict).  The float64 arrays travel as ONE packed buffer (and the
    int32 arrays as another): the descriptor's pointers are offsets into it, so marshalling costs two address look-ups
    instead of twenty (this runs on every frame of a 20-us render)."""
    fa = [_as(getattr(fs, name), _F64).reshape(-1) for name in _DESC_F]
    ia = [_as(getattr(fs, name), _I32).reshape(-1) for name in _DESC_I]
    fbuf = np.concatenate(fa) if fa else np.zeros(0, _F64)
    ibuf = np.concatenate(ia) if ia else np.zeros(0, _I32)
    d = SceneDesc()
    at = fbuf.__array_interface__["data"][0]
    for name, a in zip(_DESC_F, fa):
        setattr(d, name, at)
        at += 8 * a.size
    at = ibuf.__array_interface__["data"][0]
    for name, a in zip(_DESC_I, ia):
        setattr(d, name, at)
        at += 4 * a.size
    n = int(fa[1].size)                                   # radius
    small = getattr(fs, "small", None)
    sm = np.ascontiguousarray(small if small is not None else np.zeros(n), np.uint8)
    d.small = sm.__array_interface__["data"][0]
    d.n, d.nG, d.nP, d.nL = n, int(fa[6].size), int(fa[10].size), int(ia[4].size)      # g_strength, p_strength, l_index
    bg = fs.bg
    d.bg[0], d.bg[1], d.bg[2] = float(bg[0]), float(bg[1]), float(bg[2])
    return d, {"f": fbuf, "i": ibuf, "small": sm}


def scene_signature(fs):
    """Content key of a FlatScene: the bytes of every array the device copy is made from.  Two scenes with the same key
    upload the same blob, so a caller that re-flattens an unchanged scene list may skip the upload (``update(...,
    skip_unchanged=True)``: the sub-millisecond frame entries do; the frame / env paths re-upload every time)."""
    small = getattr(fs, "small", None)
    return (tuple(getattr(fs, name).tobytes() for name in _DESC_F), tuple(getattr(fs, name).tobytes() for name in _DESC_I),
            None if small is None else small.tobytes(), fs.bg.tobytes())


class DeviceScene:
    """A flattened scene resident in HBM (``rt_scene``): one per GPU / rank."""

    def __init__(self, fs, device=0):
        self.device = device
        self.handle = None
        d, keep = make_desc(fs)
        h = vp()
        check(lib().rt_scene_create(device, C.byref(d), C.byref(h)))
        self.handle = h.value
        self.n = int(d.n)
        self.flat = fs
        self._sig = None

    def update(self, fs, stream=None, skip_unchanged=False):
        """Re-flatten after the Python scene was mutated (the reference's scenes are mutable lists).  -> True if the scene
        was uploaded; with ``skip_unchanged`` an upload whose content equals the resident one is skipped (False)."""
        if skip_unchanged:
            sig = scene_signature(fs)
            if sig == self._sig:
                return False
            self._sig = sig
        else:
            self._sig = None
        d, keep = make_desc(fs)
        check(lib().rt_scene_update(self.handle, C.byref(d), stream))
        self.n = int(d.n)
        self.flat = fs
        return True

    def build_lbvh(self, huge_radius=50.0, stream=None):
        check(lib().rt_lbvh_build(self.handle, float(huge_radius), stream))

    def drop_lbvh(self):
        check(lib().rt_lbvh_drop(self.handle))

    @property
    def has_lbvh(self):
        n, dev, has = C.c_int32(0), C.c_int32(0), C.c_int32(0)
        check(lib().rt_scene_info(self.handle, C.byref(n), C.byref(dev), C.byref(has)))
        return bool(has.value)

    # ---- frames ----------------------------------------------------------------------------------
    def whitted_params(self, cam, X, Y, spp=1, max_bounces=1, shadow_max_bounces=0, miss=None, seed=0, prenorm=False,
                       rows=None, samples=None, accumulate=False):
        X, Y = _d(X), _d(Y)
        p = WhittedParams()
        p.cam[:] = [float(c) for c in cam]
        p.X, p.Y = X.ctypes.data_as(c_dp), Y.ctypes.data_as(c_dp)
        p.W, p.H = int(X.shape[0]), int(Y.shape[0])
        p.y0, p.y1 = (0, p.H) if rows is None else (int(rows[0]), int(rows[1]))
        p.s0, p.s1 = (0, int(spp)) if samples is None else (int(samples[0]), int(samples[1]))
        p.spp, p.max_bounces, p.shadow_max_bounces = int(spp), int(max_bounces), int(shadow_max_bounces)
        miss = np.asarray(self.flat.bg if miss is None else miss, np.float64).reshape(3)
        p.miss[:] = [float(c) for c in miss]
        p.seed, p.prenormalise, p.accumulate = int(seed), int(bool(prenorm)), int(bool(accumulate))
        p._keep = (X, Y)
        return p

    def path_params(self, cam, W, H, spp, max_bounces, mirror_threshold, seed=0, fov=60.0, rows=None, samples=None,
                    accumulate=False, schedule=0, ksplit=-1):
        p = PathParams()
        p.cam[:] = [float(c) for c in cam]
        p.W, p.H, p.fov_deg = int(W), int(H), float(fov)
        p.y0, p.y1 = (0, p.H) if rows is None else (int(rows[0]), int(rows[1]))
        p.s0, p.s1 = (0, int(spp)) if samples is None else (int(samples[0]), int(samples[1]))
        p.max_bounces, p.mirror_threshold, p.seed = int(max_bounces), float(mirror_threshold), int(seed)
        p.accumulate = int(bool(accumulate))
        p.schedule = int(schedule)
        p.ksplit = int(ksplit)
        return p

    def render_whitted(self, params, accum, precision=F32, hit=None, stats=None, stream=None):
        """Asynchronous launch into device buffers (accum [H,W,4] of the precision's float type)."""
        check(lib().rt_render_whitted(self.handle, precision, C.byref(params), _ptr(accum), _ptr(hit), _ptr(stats), stream))

    def render_path(self, params, accum, precision=F32, stats=None, stream=None, moments=None):
        """Asynchronous launch into device buffers.  ``moments`` (float64 [H,W,4], optional) also receives the sums of
        the squared sample colours and the sample count (``rt_render_path_moments``); accum and stats are the same."""
        if moments is None:
            check(lib().rt_render_path(self.handle, precision, C.byref(params), _ptr(accum), _ptr(stats), stream))
        else:
            check(lib().rt_render_path_moments(self.handle, precision, C.byref(params), _ptr(accum), _ptr(moments),
                                               _ptr(stats), stream))

    def render_path_adaptive(self, params, min_spp, tolerance, accum, moments, pixel_list, image, precision=F32, var=None,
                             counts=None, stats=None, stream=None):
        """Adaptive frame (``rt_render_path_adaptive``): ``params.s1`` is max_spp; every pixel of the band gets
        ``min_spp`` samples, then doubling rounds for the pixels whose variance of the mean exceeds ``tolerance``^2.
        ``pixel_list``: uint32 scratch of (y1 - y0) * W + 1 words.  Resolves into ``image`` (and ``var`` float32
        [H,W,3], ``counts`` int32 [H,W] when given) on the stream; synchronises the stream once per round."""
        a = AdaptiveParams()
        a.min_spp, a.tolerance = int(min_spp), float(tolerance)
        check(lib().rt_render_path_adaptive(self.handle, precision, C.byref(params), C.byref(a), _ptr(accum), _ptr(moments),
                                            _ptr(pixel_list), _ptr(image), _ptr(var), _ptr(counts), _ptr(stats), stream))

    def trace_paths(self, rays, max_bounces, mirror_threshold, bounce_count=0, seed=0, ray_ids=None, samples=(0, 1),
                    precision=F64):
        """``trace_ray_traditional(ray, bounce_count)`` for explicit rays [m,6] (origin, unit direction) ->
        (sums [m,4] = r, g, b summed over the sample range + count, stats u64[8])."""
        rays = _d(rays).reshape(-1, 6)
        m = rays.shape[0]
        r = DeviceBuffer.from_host(rays, np.float64, self.device)
        ids = None if ray_ids is None else DeviceBuffer.from_host(np.asarray(ray_ids).reshape(m), np.int32, self.device)
        ft = np.float64 if precision == F64 else np.float32
        acc = DeviceBuffer((m, 4), ft, self.device)
        st = DeviceBuffer(8, np.uint64, self.device)
        p = self.path_params((0, 0, 0), max(m, 1), 1, samples[1], max_bounces, mirror_threshold, seed=seed, samples=samples)
        check(lib().rt_trace_paths(self.handle, precision, C.byref(p), m, r.ptr, _ptr(ids), int(bounce_count), acc.ptr, st.ptr, None))
        return acc.download(), st.download()

    def render_path_sink(self, params, sink, stats=None, stream=None, moments_sink=None):
        """FP32 path kernel with a fused multi-GPU sink (``PathSink``: image store / scatter-add over peer memory).
        ``moments_sink`` (``PathMomentsSink``, optional) also carries the per-pixel variance through the sink
        (``rt_render_path_sink_moments``); the image and stats are the same."""
        if moments_sink is None:
            check(lib().rt_render_path_sink(self.handle, C.byref(params), C.byref(sink), _ptr(stats), stream))
        else:
            check(lib().rt_render_path_sink_moments(self.handle, C.byref(params), C.byref(sink), C.byref(moments_sink),
                                                    _ptr(stats), stream))

    def resolve(self, accum, W, H, spp, image, precision=F32, rows=None, stream=None):
        y0, y1 = (0, H) if rows is None else rows
        check(lib().rt_resolve(self.device, precision, _ptr(accum), int(W), int(H), int(y0), int(y1), int(spp),
                               _ptr(image), stream))

    def resolve_variance(self, accum, moments, W, H, var, precision=F32, rows=None, stream=None):
        """accum [H,W,4] + moments [H,W,4] float64 -> var [H,W,3] float32: the variance of each pixel's mean in colour
        levels^2 (0 where a pixel has fewer than two samples), rows [y0, y1) only."""
        y0, y1 = (0, H) if rows is None else rows
        check(lib().rt_resolve_variance(self.device, precision, _ptr(accum), _ptr(moments), int(W), int(H), int(y0), int(y1),
                                        _ptr(var), stream))

    def denoise(self, accum, var, W, H, image, precision=F32, radius=10, patch_radius=3, k=None, stream=None,
                features=None, k_f=1.2, tau=1e-3, rows=None):
        """accum [H,W,4] + var [H,W,3] float32 (``resolve_variance``) -> image [H,W,3] float32: the whole frame filtered
        by the variance-guided non-local-means filter (``rt_denoise``), on rt_resolve's lattice.  Per-pixel sample counts
        may differ (adaptive frames).  ``features`` = (albedo, normal, depth, fvar) as ``render_features`` gives them:
        the filter with the feature term (``rt_denoise_features``), with ``k_f`` and ``tau``.  k defaults to 0.45
        without features and 1.0 with them (the defaults measured in DESIGN §4.8c and §4.8d).
        ``rows`` = (y0, y1): only those rows of the image (``rt_denoise_rows`` / ``rt_denoise_features_rows``), equal to
        the same rows of the whole-frame filter; the inputs are read only within ``denoise_halo`` rows of the band."""
        if k is None:
            k = 0.45 if features is None else 1.0
        band = () if rows is None else (int(rows[0]), int(rows[1]))
        if features is None:
            d = DenoiseParams()
            d.radius, d.patch_radius, d.k = int(radius), int(patch_radius), float(k)
            fn = lib().rt_denoise if rows is None else lib().rt_denoise_rows
            check(fn(self.device, precision, _ptr(accum), _ptr(var), int(W), int(H), *band, C.byref(d), _ptr(image),
                     stream))
            return
        albedo, normal, depth, fvar = features
        d = DenoiseFeaturesParams()
        d.radius, d.patch_radius, d.k, d.k_f, d.tau = int(radius), int(patch_radius), float(k), float(k_f), float(tau)
        fn = lib().rt_denoise_features if rows is None else lib().rt_denoise_features_rows
        check(fn(self.device, precision, _ptr(accum), _ptr(var), _ptr(albedo), _ptr(normal), _ptr(depth), _ptr(fvar),
                 int(W), int(H), *band, C.byref(d), _ptr(image), stream))

    def render_features(self, params, albedo, normal, depth, fvar, precision=F32, stream=None):
        """First-hit features of rows [y0, y1) over samples [s0, s1) of ``params`` (``rt_render_features``): the camera
        rays ``render_path`` traces, to their nearest hit.  Means into albedo [H,W,3], normal [H,W,3] and depth [H,W],
        and the variance of the mean of each feature into fvar [H,W,3], all float32; asynchronous."""
        check(lib().rt_render_features(self.handle, precision, C.byref(params), _ptr(albedo), _ptr(normal), _ptr(depth),
                                       _ptr(fvar), stream))

    def render_whitted_host(self, params, precision=F32, want_accum=True, want_hit=True):
        """Host-buffer entry: -> (image [H,W,3] f32, sums [H,W,4], hit [H,W] i32, stats u64[8])."""
        W, H = params.W, params.H
        ft = np.float64 if precision == F64 else np.float32
        image = np.zeros((H, W, 3), np.float32)
        accum = np.zeros((H, W, 4), ft) if want_accum else None
        hit = np.full((H, W), -1, np.int32) if want_hit else None
        stats = np.zeros(8, np.uint64)
        check(lib().rt_render_whitted_host(self.handle, precision, C.byref(params), image.ctypes.data,
                                           None if accum is None else accum.ctypes.data,
                                           None if hit is None else hit.ctypes.data, stats.ctypes.data))
        return image, accum, hit, stats

    def render_path_host(self, params, precision=F32, want_accum=True):
        W, H = params.W, params.H
        ft = np.float64 if precision == F64 else np.float32
        image = np.zeros((H, W, 3), np.float32)
        accum = np.zeros((H, W, 4), ft) if want_accum else None
        stats = np.zeros(8, np.uint64)
        check(lib().rt_render_path_host(self.handle, precision, C.byref(params), image.ctypes.data,
                                        None if accum is None else accum.ctypes.data, stats.ctypes.data))
        return image, accum, stats

    def simple_params(self, W, H, cam=(0.0, 0.0, 1.0), fov=np.pi / 3, sun_pos=(-0.6, 0.2, 6.0), sun_col=(255, 255, 204),
                      sun_id=7, max_bounces=5, seed=0):
        p = SimpleParams()
        p.cam[:] = [float(c) for c in cam]
        p.W, p.H, p.fov_rad = int(W), int(H), float(fov)
        p.sun_pos[:] = [float(c) for c in sun_pos]
        p.sun_col[:] = [float(c) for c in sun_col]
        p.sun_id, p.max_bounces, p.seed = int(sun_id), int(max_bounces), int(seed)
        return p

    def render_simple_host(self, params, precision=F32, rays=None, want_image=True, hits=None):
        """FB/output6.py ``render_original_style`` (or ``trace_ray_simple`` on explicit rays [m,6]) ->
        (image [H,W,3] f32 | None, rgb [H,W,4] int32 = r, g, b, bounce_count, stats u64[8]).
        ``hits`` [m,7] = (point, normal, scene index): ``calculate_lighting_exact_original`` of those intersections
        (output6.py:197-306), rgb [1,m,4]."""
        params.lighting_only = 0
        if hits is not None:
            rays = _d(hits).reshape(-1, 7)
            params.m, params.lighting_only = int(rays.shape[0]), 1
            shape, want_image = (1, params.m), False
        elif rays is not None:
            rays = _d(rays).reshape(-1, 6)
            params.m = int(rays.shape[0])
            shape = (1, params.m)
        else:
            shape = (params.H, params.W)
        rgb = np.zeros(shape + (4,), np.int32)
        image = np.zeros(shape + (3,), np.float32) if want_image else None
        stats = np.zeros(8, np.uint64)
        check(lib().rt_render_simple_host(self.handle, precision, C.byref(params), None if rays is None else rays.ctypes.data,
                                          rgb.ctypes.data, None if image is None else image.ctypes.data, stats.ctypes.data))
        return image, rgb, stats

    # ---- batched primitives ----------------------------------------------------------------------
    def trace_rays(self, rays, suppress=None, bounces0=None, through0=None, max_bounces=1, shadow_max_bounces=0,
                   miss=(0, 0, 0), shade=True, precision=F64):
        """Batch of ``Ray.nearestSphereIntersect`` (+ ``terminalRGB``): rays [m,6] -> (term [m,11], rgb [m,3] | None);
        term = hit, scene index, bounces, through_count, point(3), normal(3), distance."""
        rays = _d(rays).reshape(-1, 6)
        m = rays.shape[0]
        dev = self.device
        r = DeviceBuffer.from_host(rays, np.float64, dev)
        sup = None if suppress is None else DeviceBuffer.from_host(np.asarray(suppress).reshape(m), np.int32, dev)
        b0 = None if bounces0 is None else DeviceBuffer.from_host(np.asarray(bounces0).reshape(m), np.int32, dev)
        t0 = None if through0 is None else DeviceBuffer.from_host(np.asarray(through0).reshape(m), np.int32, dev)
        term = DeviceBuffer((m, 11), np.float64, dev)
        rgb = DeviceBuffer((m, 3), np.float64, dev) if shade else None
        missv = (C.c_double * 3)(*[float(c) for c in miss])
        check(lib().rt_trace_rays(self.handle, precision, m, r.ptr, _ptr(sup), _ptr(b0), _ptr(t0), int(max_bounces),
                                  int(shadow_max_bounces), missv, term.ptr, _ptr(rgb), None))
        return term.download(), (rgb.download() if shade else None)

    def shade_hits(self, hits, shadow_max_bounces=0, precision=F64):
        """Batch of ``Intersection.terminalRGB``: hits [m,7] = scene index, point(3), normal(3) -> rgb [m,3]."""
        hits = _d(hits).reshape(-1, 7)
        m = hits.shape[0]
        h = DeviceBuffer.from_host(hits, np.float64, self.device)
        rgb = DeviceBuffer((m, 3), np.float64, self.device)
        check(lib().rt_terminal_rgb(self.handle, precision, m, h.ptr, int(shadow_max_bounces), rgb.ptr, None))
        return rgb.download()

    def close(self):
        if getattr(self, "handle", None):
            try:
                load_symbols().rt_scene_destroy(self.handle)
            finally:
                self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def sphere_discriminant(rays, spheres, point=0, precision=F64, device=0):
    """Batch of ``Ray.sphereDiscriminant``: rays [m,6], spheres [m,4] -> out [m,8] = hit, t, point(3), normal(3)."""
    rays = _d(rays).reshape(-1, 6)
    sph = _d(spheres).reshape(-1, 4)
    m = rays.shape[0]
    r, s = DeviceBuffer.from_host(rays, np.float64, device), DeviceBuffer.from_host(sph, np.float64, device)
    out = DeviceBuffer((m, 8), np.float64, device)
    check(lib().rt_sphere_discriminant(device, precision, m, r.ptr, s.ptr, int(point), out.ptr, None))
    return out.download()
