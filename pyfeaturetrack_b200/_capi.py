"""ctypes binding of libkltb200.so (include/klt_b200.h).  There is no CPU fallback: if the CUDA library is
missing or no B200 is present, every entry point raises."""
import ctypes as C
import functools
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIBPATH = os.path.join(_HERE, "libkltb200.so")

KLT_MAX_TAPS = 71
PRECISION_FAST, PRECISION_STRICT, PRECISION_FAST_WINDOWED = 0, 1, 2
MIX_COPY, MIX_SMOOTH0, MIX_DOWN2, MIX_LEVEL01 = 0, 1, 2, 3
SELECT_STRICT, SELECT_FAST = 0, 1
KLT_ERR_INVALID, KLT_ERR_CUDA, KLT_ERR_NOMEM, KLT_ERR_UNSUPPORTED, KLT_ERR_ASSERT = -1, -2, -3, -4, -5


class KLTB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libkltb200 error %d: %s" % (code, msg))
        self.code = code


class Kernel1D(C.Structure):
    _fields_ = [("n", C.c_int32), ("reserved", C.c_int32), ("taps", C.c_double * KLT_MAX_TAPS)]

    @classmethod
    def from_taps(cls, taps):
        k = cls()
        taps = [float(t) for t in taps]
        if len(taps) > KLT_MAX_TAPS:
            raise ValueError("kernel longer than %d taps" % KLT_MAX_TAPS)
        k.n = len(taps)
        for i, t in enumerate(taps):
            k.taps[i] = t
        return k


class Taps(C.Structure):
    _fields_ = [("smooth", Kernel1D), ("pyramid", Kernel1D), ("grad_gauss", Kernel1D), ("grad_deriv", Kernel1D)]


class Params(C.Structure):
    _fields_ = [("window_width", C.c_int32), ("window_height", C.c_int32), ("n_levels", C.c_int32),
                ("subsampling", C.c_int32), ("borderx", C.c_double), ("bordery", C.c_double),
                ("mindist", C.c_int32), ("min_eigenvalue", C.c_int32), ("n_skipped_pixels", C.c_int32),
                ("max_iterations", C.c_int32), ("min_determinant", C.c_float), ("min_displacement", C.c_float),
                ("step_factor", C.c_float), ("has_max_residue", C.c_int32), ("max_residue", C.c_float),
                ("retain_trackers", C.c_int32), ("lighting_insensitive", C.c_int32),
                ("affine_consistency_check", C.c_int32), ("affine_window_width", C.c_int32),
                ("affine_window_height", C.c_int32), ("affine_max_iterations", C.c_int32),
                ("affine_max_residue", C.c_float), ("affine_min_displacement", C.c_float),
                ("affine_max_displacement_differ", C.c_float), ("min_eigenvalue_f", C.c_float)]


_lib = None

# The drop-in modules share ONE process-wide context (stream, workspace, scratch pyramids): like the reference under the GIL,
# their entry points run one at a time.  ctypes releases the GIL during the C calls, so the serialisation is explicit.
# Explicit Context objects are not covered: a klt_ctx is single-threaded, distinct contexts may run concurrently.
api_lock = threading.RLock()


def serialized(fn):
    @functools.wraps(fn)
    def wrapper(*a, **kw):
        with api_lock:
            return fn(*a, **kw)
    return wrapper


# name -> (restype, argtypes); every symbol include/klt_b200.h declares
_vp, _i, _sz = C.c_void_p, C.c_int, C.c_size_t
_fp, _dp, _ip, _u8p = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p   # raw addresses: host OR device pointers
SIGNATURES = {
    "klt_abi_version": (_i, []),
    "klt_ctx_create": (_i, [_i, _vp, C.POINTER(_vp)]),
    "klt_ctx_destroy": (_i, [_vp]),
    "klt_last_error": (C.c_char_p, [_vp]),
    "klt_sync": (_i, [_vp]),
    "klt_ctx_stream": (_vp, [_vp]),
    "klt_launch_count": (C.c_int64, [_vp]),
    "klt_host_alloc": (_i, [_sz, C.POINTER(_vp)]),
    "klt_host_free": (_i, [_vp]),
    "klt_device_alloc": (_i, [_vp, _sz, C.POINTER(_vp)]),
    "klt_device_free": (_i, [_vp, _vp]),
    "klt_memcpy": (_i, [_vp, _vp, _vp, _sz]),
    "klt_timer_start": (_i, [_vp]),
    "klt_timer_stop": (_i, [_vp]),
    "klt_timer_elapsed_ms": (_i, [_vp, C.POINTER(C.c_float)]),
    "klt_profile_enable": (_i, [_vp, _i]),
    "klt_profile_reset": (_i, [_vp]),
    "klt_profile_count": (_i, [_vp]),
    "klt_profile_get": (_i, [_vp, _i, C.POINTER(C.c_char_p), C.POINTER(C.c_double), C.POINTER(C.c_int64),
                             C.POINTER(C.c_double)]),
    "klt_probe_traffic_mix": (_i, [_vp, _i, C.c_double, _i, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "klt_convolve_separable_f32": (_i, [_vp, _fp, _i, _i, C.POINTER(Kernel1D), C.POINTER(Kernel1D), _i, _fp]),
    "klt_smooth_f32": (_i, [_vp, _fp, _i, _i, C.POINTER(Kernel1D), _i, _fp]),
    "klt_gradients_f32": (_i, [_vp, _fp, _i, _i, C.POINTER(Kernel1D), C.POINTER(Kernel1D), _i, _fp, _fp]),
    "klt_pyr_create": (_i, [_vp, _i, _i, _i, _i, _i, C.POINTER(_vp)]),
    "klt_pyr_destroy": (_i, [_vp, _vp]),
    "klt_pyr_dims": (_i, [_vp, _i, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]),
    "klt_pyr_bytes": (_sz, [_vp]),
    "klt_pyr_build_u8": (_i, [_vp, _vp, _u8p, _sz, _sz, C.POINTER(Taps), _i]),
    "klt_pyr_build_f32": (_i, [_vp, _vp, _fp, _sz, _sz, C.POINTER(Taps), _i, _i]),
    "klt_pyr_download": (_i, [_vp, _vp, _i, _i, _i, _fp]),
    "klt_pyr_level_ptr": (_i, [_vp, _i, _i, _i, C.POINTER(_vp)]),
    "klt_pyr_ensure_gradients": (_i, [_vp, _vp]),
    "klt_scan_good_features": (_i, [_vp, _fp, _fp, _i, _i, _i, _i, _i, _i, _i, _fp]),
    "klt_select_good_features": (_i, [_vp, C.POINTER(Params), _vp, _i, _fp, _fp, _i, _i, _i, _i, _dp, _dp, _ip,
                                      C.POINTER(C.c_int64)]),
    "klt_select_good_features_batch": (_i, [_vp, C.POINTER(Params), _vp, _i, _i, _i, _dp, _dp, _ip]),
    "klt_eigen_map_batch": (_i, [_vp, C.POINTER(Params), _vp, _i, _fp, C.POINTER(_i), C.POINTER(_i)]),
    "klt_track_features": (_i, [_vp, C.POINTER(Params), _vp, _vp, _i, _dp, _dp, _ip, C.POINTER(C.c_int64)]),
    "klt_track_features_fb": (_i, [_vp, C.POINTER(Params), _vp, _vp, _i, C.c_float, _dp, _dp, _ip, _fp,
                                   C.POINTER(C.c_int64)]),
    "klt_affine_create": (_i, [_vp, _i, _i, _i, C.POINTER(_vp)]),
    "klt_affine_destroy": (_i, [_vp, _vp]),
    "klt_affine_reset": (_i, [_vp, _vp, _ip]),
    "klt_affine_download": (_i, [_vp, _vp, _ip, _fp, _fp, _fp]),
    "klt_affine_download_template": (_i, [_vp, _vp, _i, _fp]),
    "klt_track_features_affine": (_i, [_vp, C.POINTER(Params), _vp, _vp, _i, _dp, _dp, _ip, _vp, C.POINTER(C.c_int64)]),
    "klt_extract_patch": (_i, [_vp, _fp, _i, _i, C.c_float, C.c_float, _i, _i, _fp]),
    "klt_track_iterate": (_i, [_vp, C.POINTER(Params), C.c_float, C.c_float, _fp, _fp, _fp, _fp, _fp, _fp, _i, _i,
                               C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "klt_patch_combine": (_i, [_vp, _fp, _fp, _i, _i, C.c_float, C.c_float, _i, _i, _i, _fp]),
    "klt_enforce_min_distance": (_i, [_vp, _i, _fp, _ip, _ip, _i, _i, _i, C.c_double, _i, _i, _dp, _dp, _ip]),
    "klt_track_pairs_u8": (_i, [_vp, C.POINTER(Params), C.POINTER(Taps), _i, _vp, _vp, _u8p, _u8p, _sz, _sz, _i,
                                _dp, _dp, _ip]),
    "klt_track_pairs_u8_async": (_i, [_vp, C.POINTER(Params), C.POINTER(Taps), _i, _vp, _vp, _u8p, _u8p, _sz, _sz, _i,
                                      _dp, _dp, _ip]),
    "klt_async_result": (_i, [_vp]),
    "klt_async_mark": (_i, [_vp, _i]),
    "klt_async_wait": (_i, [_vp, _i]),
    "klt_sequence_create": (_i, [_vp, C.POINTER(Params), C.POINTER(Taps), _i, _i, _i, _i, _i, _i, C.POINTER(_vp)]),
    "klt_sequence_destroy": (_i, [_vp, _vp]),
    "klt_sequence_start_u8": (_i, [_vp, _vp, _u8p, _sz, _sz, _i]),
    "klt_sequence_set_features": (_i, [_vp, _vp, _dp, _dp, _ip]),
    "klt_sequence_step_u8": (_i, [_vp, _vp, _u8p, _sz, _sz, _i, _dp, _dp, _ip, _ip]),
    "klt_sequence_get_features": (_i, [_vp, _vp, _dp, _dp, _ip, _ip]),
    "klt_sequence_sync": (_i, [_vp, _vp, C.POINTER(C.c_int64)]),
    "klt_sequence_select_stats": (_i, [_vp, _vp, _vp]),
    "klt_sequence_pyramid": (_i, [_vp, C.POINTER(_vp)]),
    "klt_sequence_uses_graph": (_i, [_vp]),
    "klt_sequence_set_fb_check": (_i, [_vp, _vp, C.c_float]),
    "klt_sequence_get_fb_error": (_i, [_vp, _vp, _fp]),
}


def lib():
    """Loads libkltb200.so (built by pyfeaturetrack_b200/build.py).  Raises if it is missing -- never falls back."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIBPATH):
            raise ImportError("%s not found: run `python -m pyfeaturetrack_b200.build` (needs nvcc). "
                              "There is no CPU fallback." % _LIBPATH)
        L = C.CDLL(_LIBPATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


_featlist = False


def featlist():
    """libkltfeatlist.so (csrc/featlist.c: feature list <-> arrays through the CPython C API, host glue only), or None when it
    was not built -- the callers then walk the list in Python."""
    global _featlist
    if _featlist is False:
        path = os.path.join(os.path.dirname(_LIBPATH), "libkltfeatlist.so")
        try:
            L = C.PyDLL(path)
            L.klt_featlist_gather.restype = C.c_int
            L.klt_featlist_gather.argtypes = [C.py_object, C.c_ssize_t, C.c_void_p, C.c_void_p, C.c_void_p]
            L.klt_featlist_scatter_tracked.restype = C.c_int
            L.klt_featlist_scatter_tracked.argtypes = [C.py_object, C.c_ssize_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
            _featlist = L
        except (OSError, AttributeError):
            _featlist = None
    return _featlist


def ptr(a):
    """Address of a numpy array's data, or an int device pointer passed through."""
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return int(a)


class Pyramid:
    """Owns one klt_pyr (a batch of 3-component pyramids in device memory)."""

    def __init__(self, ctx, w, h, n_levels, subsampling, batch=1):
        self.ctx = ctx
        self.w, self.h, self.n_levels, self.subsampling, self.batch = w, h, n_levels, subsampling, batch
        hnd = C.c_void_p()
        ctx.check(lib().klt_pyr_create(ctx.handle, w, h, n_levels, subsampling, batch, C.byref(hnd)))
        self.handle = hnd
        self.dims = []
        for l in range(n_levels):
            a, b, c = C.c_int(), C.c_int(), C.c_int()
            lib().klt_pyr_dims(self.handle, l, C.byref(a), C.byref(b), C.byref(c))
            self.dims.append((a.value, b.value, c.value))

    def build_u8(self, frames, taps, precision, pitch=None, frame_stride=None):
        """frames: uint8 ndarray [batch, h, w] / [h, w] or a raw pointer."""
        if isinstance(frames, np.ndarray):
            assert frames.dtype == np.uint8 and frames.flags.c_contiguous
            pitch = frames.shape[-1] if pitch is None else pitch
            frame_stride = frames.shape[-1] * frames.shape[-2] if frame_stride is None else frame_stride
        self.ctx.check(lib().klt_pyr_build_u8(self.ctx.handle, self.handle, ptr(frames), pitch, frame_stride,
                                              C.byref(taps), precision))
        self._keep = frames   # keep host memory alive until the stream has consumed it

    def build_f32(self, images, taps, precision, already_smoothed, pitch=None, frame_stride=None):
        if isinstance(images, np.ndarray):
            assert images.dtype == np.float32 and images.flags.c_contiguous
            pitch = images.shape[-1] if pitch is None else pitch
            frame_stride = images.shape[-1] * images.shape[-2] if frame_stride is None else frame_stride
        self.ctx.check(lib().klt_pyr_build_f32(self.ctx.handle, self.handle, ptr(images), pitch, frame_stride,
                                               C.byref(taps), precision, 1 if already_smoothed else 0))
        self._keep = images

    def download(self, which, level, image=0):
        w, h, _ = self.dims[level]
        out = np.empty((h, w), np.float32)
        self.ctx.check(lib().klt_pyr_download(self.ctx.handle, self.handle, image, which, level, out.ctypes.data))
        return out

    def level_ptr(self, which, level, image=0):
        p = C.c_void_p()
        lib().klt_pyr_level_ptr(self.handle, image, which, level, C.byref(p))
        return p.value

    def nbytes(self):
        return lib().klt_pyr_bytes(self.handle)

    def close(self):
        if self.handle:
            lib().klt_pyr_destroy(self.ctx.handle, self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class AffineState:
    """Owns one klt_affine: per-feature templates, template centres and 2x2 maps of the affine consistency check."""

    def __init__(self, ctx, n, aw, ah):
        self.ctx, self.n, self.aw, self.ah = ctx, n, aw, ah
        hnd = C.c_void_p()
        ctx.check(lib().klt_affine_create(ctx.handle, n, aw, ah, C.byref(hnd)))
        self.handle = hnd

    def reset(self, mask=None):
        if mask is None:
            self.ctx.check(lib().klt_affine_reset(self.ctx.handle, self.handle, None))
        else:
            m = np.ascontiguousarray(mask, np.int32)
            assert m.shape == (self.n,)
            self.ctx.check(lib().klt_affine_reset(self.ctx.handle, self.handle, m.ctypes.data))
            self.ctx.sync()

    def download(self):
        has = np.empty(self.n, np.int32)
        ax = np.empty(self.n, np.float32)
        ay = np.empty(self.n, np.float32)
        A = np.empty((self.n, 4), np.float32)
        self.ctx.check(lib().klt_affine_download(self.ctx.handle, self.handle, has.ctypes.data, ax.ctypes.data,
                                                 ay.ctypes.data, A.ctypes.data))
        return has, ax, ay, A

    def template(self, slot):
        out = np.empty((3, self.ah + 2, self.aw + 2), np.float32)
        self.ctx.check(lib().klt_affine_download_template(self.ctx.handle, self.handle, slot, out.ctypes.data))
        return out

    def close(self):
        if self.handle:
            lib().klt_affine_destroy(self.ctx.handle, self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Sequence:
    """Owns one klt_sequence: n_sequences lock-stepped sequences (sequentialMode tracking + per-frame replacement)."""

    def __init__(self, ctx, params, taps, w, h, n_sequences, n_features, precision, select_mode):
        self.ctx, self.w, self.h, self.B, self.n = ctx, w, h, n_sequences, n_features
        hnd = C.c_void_p()
        ctx.check(lib().klt_sequence_create(ctx.handle, C.byref(params), C.byref(taps), w, h, n_sequences, n_features,
                                            precision, select_mode, C.byref(hnd)))
        self.handle = hnd
        self._keep = []

    def _frames(self, frames):
        if isinstance(frames, np.ndarray):
            assert frames.dtype == np.uint8 and frames.flags.c_contiguous and frames.shape == (self.B, self.h, self.w)
            self._keep = [frames] + self._keep[:2]       # host memory must outlive the asynchronous upload
            return frames.ctypes.data
        return int(frames)

    def start(self, frames, select=True):
        self.ctx.check(lib().klt_sequence_start_u8(self.ctx.handle, self.handle, self._frames(frames), self.w,
                                                   self.w * self.h, 1 if select else 0))

    def set_features(self, x, y, val):
        x, y = np.ascontiguousarray(x, np.float64), np.ascontiguousarray(y, np.float64)
        val = np.ascontiguousarray(val, np.int32)
        assert x.shape == y.shape == val.shape == (self.B, self.n)
        self.ctx.check(lib().klt_sequence_set_features(self.ctx.handle, self.handle, x.ctypes.data, y.ctypes.data,
                                                       val.ctypes.data))
        self.ctx.sync()

    def step(self, frames, replace=True, out=None):
        """out: None (results stay on the device) or (x, y, val, val_tracked) pinned arrays / device pointers."""
        o = [0, 0, 0, 0] if out is None else [ptr(a) if a is not None else 0 for a in out]
        self.ctx.check(lib().klt_sequence_step_u8(self.ctx.handle, self.handle, self._frames(frames), self.w,
                                                  self.w * self.h, 1 if replace else 0, o[0], o[1], o[2], o[3]))

    def features(self):
        x, y = np.empty((self.B, self.n)), np.empty((self.B, self.n))
        v, vt = np.empty((self.B, self.n), np.int32), np.empty((self.B, self.n), np.int32)
        self.ctx.check(lib().klt_sequence_get_features(self.ctx.handle, self.handle, x.ctypes.data, y.ctypes.data,
                                                       v.ctypes.data, vt.ctypes.data))
        return x, y, v, vt

    def sync(self):
        it = C.c_int64()
        self.ctx.check(lib().klt_sequence_sync(self.ctx.handle, self.handle, C.byref(it)))
        return it.value

    def select_stats(self):
        out = np.zeros((self.B, 4), np.int64)
        self.ctx.check(lib().klt_sequence_select_stats(self.ctx.handle, self.handle, out.ctypes.data))
        return out

    def uses_graph(self):
        return bool(lib().klt_sequence_uses_graph(self.handle))

    def set_fb_check(self, max_fb_error):
        """Forward-backward check inside every following step (max_fb_error > 0, level-0 pixels); 0 or None turns it off."""
        self.ctx.check(lib().klt_sequence_set_fb_check(self.ctx.handle, self.handle,
                                                       0.0 if max_fb_error is None else float(max_fb_error)))

    def fb_error(self):
        """float32 [n_sequences, n_features]: the last step's forward-backward distances (-1 where none was measured)."""
        out = np.empty((self.B, self.n), np.float32)
        self.ctx.check(lib().klt_sequence_get_fb_error(self.ctx.handle, self.handle, out.ctypes.data))
        return out

    def close(self):
        if self.handle:
            lib().klt_sequence_destroy(self.ctx.handle, self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Context:
    """One klt_ctx = one (GPU, stream)."""

    def __init__(self, device=0, stream=None):
        hnd = C.c_void_p()
        rc = lib().klt_ctx_create(device, stream, C.byref(hnd))
        if rc != 0:
            raise KLTB200Error(rc, lib().klt_last_error(None).decode())
        self.handle = hnd
        self.device = device
        self._pyr_cache = {}

    def check(self, rc):
        if rc != 0:
            msg = lib().klt_last_error(self.handle).decode()
            if rc == KLT_ERR_ASSERT:
                raise AssertionError(msg)
            raise KLTB200Error(rc, msg)

    def sync(self):
        self.mark_synced()
        self.check(lib().klt_sync(self.handle))

    def mark_synced(self):
        """A call that waited for the stream has returned: every staging buffer is free again."""
        self.__dict__.setdefault("_busy_stages", set()).clear()

    def launch_count(self):
        return lib().klt_launch_count(self.handle)

    def timer_start(self):
        self.check(lib().klt_timer_start(self.handle))

    def timer_stop(self):
        self.check(lib().klt_timer_stop(self.handle))

    def timer_elapsed_ms(self):
        ms = C.c_float()
        self.check(lib().klt_timer_elapsed_ms(self.handle, C.byref(ms)))
        return ms.value

    def profile(self, on):
        self.check(lib().klt_profile_enable(self.handle, 1 if on else 0))

    def profile_reset(self):
        self.check(lib().klt_profile_reset(self.handle))

    def traffic_mix_probe(self, kind, total_bytes, reps=10):
        """GB/s a trivial linear kernel reaches for the read/write mix `kind` (MIX_*) and launch size `total_bytes`."""
        ms, moved = C.c_double(), C.c_double()
        self.check(lib().klt_probe_traffic_mix(self.handle, kind, float(total_bytes), reps, C.byref(ms), C.byref(moved)))
        return moved.value / (ms.value * 1e-3) / 1e9, ms.value

    def profile_read(self):
        """{kernel name: dict(ms=total, launches=n, bytes=algorithmic bytes)}"""
        out = {}
        for i in range(lib().klt_profile_count(self.handle)):
            name, ms, n, b = C.c_char_p(), C.c_double(), C.c_int64(), C.c_double()
            self.check(lib().klt_profile_get(self.handle, i, C.byref(name), C.byref(ms), C.byref(n), C.byref(b)))
            out[name.value.decode()] = dict(ms=ms.value, launches=n.value, bytes=b.value)
        return out

    def scratch_pyramid(self, w, h, n_levels, subsampling, batch=1, slot=0):
        """Cached scratch pyramids (avoids cudaMalloc per call)."""
        key = (w, h, n_levels, subsampling, batch, slot)
        p = self._pyr_cache.get(key)
        if p is None:
            if len(self._pyr_cache) > 16:
                self._pyr_cache.clear()
            p = self._pyr_cache[key] = Pyramid(self, w, h, n_levels, subsampling, batch)
        return p

    def pinned_stage(self, shape, key):
        """A reusable pinned uint8 staging buffer of the given shape (one per key, e.g. per scratch pyramid).  Buffers that
        are replaced or evicted are handed back to the driver (after a sync: an upload may still be reading them)."""
        st = self.__dict__.setdefault("_stages", {})
        buf = st.get(key)
        if buf is None or buf.shape != tuple(shape):
            stale = [buf] if buf is not None else []
            if len(st) > 8:
                stale += [b for b in st.values() if b is not buf]
                st.clear()
            if stale:
                self.sync()
                for b in stale:
                    self.free_pinned(b)
            buf = st[key] = self.pinned_array(tuple(shape), np.uint8)
        return buf

    def sync_stage(self, key):
        """The previous upload from this staging buffer must have been consumed before it is overwritten: waits only if an
        upload from THIS buffer may still be in flight (none is after any synchronous call), then marks it in use."""
        busy = self.__dict__.setdefault("_busy_stages", set())
        if key in busy:
            self.sync()
        busy.add(key)

    def host_alloc(self, nbytes):
        p = C.c_void_p()
        rc = lib().klt_host_alloc(nbytes, C.byref(p))
        if rc != 0:
            raise KLTB200Error(rc, "klt_host_alloc failed")
        return p.value

    def pinned_array(self, shape, dtype):
        """numpy array over pinned host memory; free_pinned(array) or close() returns it to the driver."""
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        addr = self.host_alloc(max(n, 1))
        buf = (C.c_char * max(n, 1)).from_address(addr)
        arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
        self.__dict__.setdefault("_pinned", {})[arr.ctypes.data] = addr
        return arr

    def free_pinned(self, arr):
        """Hands a pinned_array's memory back (the caller must not touch the array afterwards)."""
        addr = self.__dict__.get("_pinned", {}).pop(arr.ctypes.data, None)
        if addr is not None:
            lib().klt_host_free(addr)

    def device_alloc(self, nbytes):
        p = C.c_void_p()
        self.check(lib().klt_device_alloc(self.handle, nbytes, C.byref(p)))
        return p.value

    def device_free(self, p):
        self.check(lib().klt_device_free(self.handle, p))

    def memcpy(self, dst, src, nbytes):
        self.check(lib().klt_memcpy(self.handle, ptr(dst), ptr(src), nbytes))

    def close(self):
        if self.handle:
            for p in self._pyr_cache.values():
                p.close()
            self._pyr_cache.clear()
            lib().klt_sync(self.handle)
            self.__dict__.get("_stages", {}).clear()
            for addr in self.__dict__.get("_pinned", {}).values():
                lib().klt_host_free(addr)
            self.__dict__.get("_pinned", {}).clear()
            lib().klt_ctx_destroy(self.handle)
            self.handle = None


_default_ctx = None
_default_device = None


def set_device(device):
    """Selects the GPU the drop-in modules use (default: $KLT_B200_DEVICE, else $LOCAL_RANK, else 0)."""
    global _default_ctx, _default_device
    if _default_ctx is not None and _default_ctx.device != device:
        _default_ctx.close()
        _default_ctx = None
    _default_device = device


def default_ctx():
    global _default_ctx, _default_device
    if _default_ctx is None:
        if _default_device is None:
            _default_device = int(os.environ.get("KLT_B200_DEVICE", os.environ.get("LOCAL_RANK", "0")))
        _default_ctx = Context(_default_device)
    return _default_ctx
