"""ctypes binding of librtgrff_b200.so (C ABI: include/rtgrff.h).

There is no CPU fallback: if the shared library has not been built, or no CUDA device is
visible, the first call raises.  Build with ``python -c "import __graft_entry__ as g; g.build()"``
or ``python -m raytracinggrff_b200.build``.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_uint8, c_void_p
from pathlib import Path

import numpy as np

_PKG = Path(__file__).resolve().parent
# RTGRFF_LIB overrides the library path (A/B runs of differently tuned builds; development aid)
LIB_PATH = Path(os.environ["RTGRFF_LIB"]) if os.environ.get("RTGRFF_LIB") else _PKG / "librtgrff_b200.so"

RTGRFF_OK = 0
RTGRFF_EINVAL = -1
RTGRFF_ECUDA = -2
RTGRFF_ENOCUBE = -3
RTGRFF_ENOMEM = -4
RTGRFF_EUNSUPPORTED = -5

S_PER_STEP = 0
S_CUMULATIVE = 1
ORDER_RECORD = 0
ORDER_REVERSED = 1

# every symbol include/rtgrff.h declares (tests check the library exports all of them)
EXPORTS = (
    "rtgrff_version", "rtgrff_last_error", "rtgrff_device_count", "rtgrff_ctx_create", "rtgrff_ctx_destroy",
    "rtgrff_ctx_synchronize", "rtgrff_ctx_launch_count", "rtgrff_ctx_last_kernel_ms", "rtgrff_set_omega_cube", "rtgrff_set_field_cubes",
    "rtgrff_resample_spherical", "rtgrff_compose_cubes", "rtgrff_sample_spherical_los",
    "rtgrff_trace", "rtgrff_sample", "rtgrff_sample_traced", "PyGET_MW", "rtgrff_get_mw_slice",
    "rtgrff_emission_traced", "rtgrff_render_map", "rtgrff_gaussian_beam", "rtgrff_patch_nan",
    "rtgrff_ctx_create_on_stream", "rtgrff_current_device", "rtgrff_get_mw_slice_device", "rtgrff_memcpy",
    "rtgrff_export_cubes", "rtgrff_shard_rows", "rtgrff_comm_unique_id", "rtgrff_comm_init_rank",
    "rtgrff_comm_destroy", "rtgrff_gather_image", "rtgrff_device_alloc", "rtgrff_device_free",
    "rtgrff_ctx_set_pipeline", "rtgrff_ctx_set_grff64", "rtgrff_place_rows", "rtgrff_render_map_diag",
    "rtgrff_set_spherical_model", "rtgrff_render_los_map", "rtgrff_resample_spherical_view",
    "rtgrff_sample_spherical_los_view", "rtgrff_render_los_map_view",
)

# planes of rtgrff_render_map_diag's output (RTGRFF_DIAG_* in include/rtgrff.h), in plane order
DIAG_PLANES = ("em_x", "em_y", "em_z", "em_r", "tau_L", "tau_R", "ray_r_min")


class FreqParams(ctypes.Structure):
    """rtgrff_freq_params."""
    _fields_ = [("freq_hz", c_double), ("dt", c_double), ("n_steps", c_int64), ("record_stride", c_int64)]


_lib = None


def load():
    """Load the shared library (once) and declare the prototypes.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built and this package has no CPU "
            "fallback. Run `python -m raytracinggrff_b200.build` (needs nvcc) first.")
    lib = ctypes.CDLL(str(LIB_PATH))
    dp, fp, ip = POINTER(c_double), POINTER(c_float), POINTER(c_int32)
    lib.rtgrff_version.restype = c_char_p
    lib.rtgrff_last_error.restype = c_char_p
    lib.rtgrff_device_count.restype = c_int
    lib.rtgrff_ctx_create.argtypes = [c_int, c_void_p, POINTER(c_void_p)]
    lib.rtgrff_ctx_create_on_stream.argtypes = [c_int, c_void_p, POINTER(c_void_p)]
    lib.rtgrff_current_device.restype = c_int
    lib.rtgrff_get_mw_slice_device.argtypes = [c_void_p, ip, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.rtgrff_ctx_set_pipeline.argtypes = [c_void_p, c_int]
    lib.rtgrff_ctx_set_grff64.argtypes = [c_void_p, c_int]
    lib.rtgrff_device_alloc.argtypes = [c_void_p, POINTER(c_void_p), ctypes.c_size_t]
    lib.rtgrff_device_free.argtypes = [c_void_p, c_void_p]
    lib.rtgrff_memcpy.argtypes = [c_void_p, c_void_p, c_void_p, ctypes.c_size_t, c_int]
    lib.rtgrff_export_cubes.argtypes = [c_void_p, dp, fp, fp, fp, fp, fp, fp]
    lib.rtgrff_shard_rows.argtypes = [c_int, c_int, c_int, ip, POINTER(c_int), POINTER(c_int)]
    lib.rtgrff_comm_unique_id.argtypes = [ctypes.c_char_p]
    lib.rtgrff_comm_init_rank.argtypes = [c_void_p, c_int, c_int, ctypes.c_char_p]
    lib.rtgrff_comm_destroy.argtypes = [c_void_p]
    lib.rtgrff_place_rows.argtypes = [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]
    lib.rtgrff_gather_image.argtypes = [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int]
    lib.rtgrff_ctx_destroy.argtypes = [c_void_p]
    lib.rtgrff_ctx_synchronize.argtypes = [c_void_p]
    lib.rtgrff_ctx_launch_count.argtypes = [c_void_p]
    lib.rtgrff_ctx_launch_count.restype = c_int64
    lib.rtgrff_ctx_last_kernel_ms.argtypes = [c_void_p]
    lib.rtgrff_ctx_last_kernel_ms.restype = c_double
    lib.rtgrff_set_omega_cube.argtypes = [c_void_p, c_void_p, c_int, c_int, c_int, dp, c_int]
    lib.rtgrff_set_field_cubes.argtypes = [c_void_p, fp, fp, fp, fp, fp, fp, c_int, c_int, c_int, dp]
    lib.rtgrff_resample_spherical.argtypes = [c_void_p, c_int, fp, dp, dp, dp, c_int, c_int, c_int, dp, dp, dp, c_int,
                                              c_int, c_int, dp, c_double, c_double, c_double, c_double, c_int, dp]
    # the _view entry points: the same arguments plus b0_deg, p_deg right after phi0_offset_deg
    a = lib.rtgrff_resample_spherical.argtypes
    lib.rtgrff_resample_spherical_view.argtypes = a[:17] + [c_double, c_double] + a[17:]
    lib.rtgrff_compose_cubes.argtypes = [c_void_p, c_int]
    lib.rtgrff_sample_spherical_los.argtypes = [c_void_p, fp, dp, dp, dp, c_int, c_int, c_int, dp, dp, dp, c_int, c_int,
                                                c_int, c_double, c_double, c_double, c_double, dp]
    a = lib.rtgrff_sample_spherical_los.argtypes
    lib.rtgrff_sample_spherical_los_view.argtypes = a[:15] + [c_double, c_double] + a[15:]
    lib.rtgrff_trace.argtypes = [c_void_p, c_int64, dp, dp, dp, dp, c_double, c_double, c_int64, c_int64, c_int,
                                 c_double, c_int, dp, dp, POINTER(c_int64)]
    lib.rtgrff_sample.argtypes = [c_void_p, c_int64, c_int64, fp, fp, fp, c_double, c_double, c_double, c_double,
                                  fp, fp, fp, fp, POINTER(c_uint8)]
    lib.rtgrff_sample_traced.argtypes = [c_void_p, fp, c_double, c_double, c_double, c_double, fp, fp, fp, fp,
                                         POINTER(c_uint8), fp]
    lib.PyGET_MW.argtypes = [ip, dp, dp, dp, dp, dp, dp]
    lib.PyGET_MW.restype = c_int
    lib.rtgrff_get_mw_slice.argtypes = [c_void_p, ip, dp, dp, dp, dp, dp, dp, ip]
    lib.rtgrff_emission_traced.argtypes = [c_void_p, c_double, c_double, c_int, c_double, c_int, c_int, c_int, dp, dp]
    lib.rtgrff_render_map.argtypes = [c_void_p, c_int64, dp, dp, dp, dp, ip, c_int, POINTER(FreqParams), c_int, c_double,
                                      c_double, c_double, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                      c_int, POINTER(c_int64)]
    lib.rtgrff_render_map_diag.argtypes = lib.rtgrff_render_map.argtypes + [c_void_p]
    lib.rtgrff_set_spherical_model.argtypes = [c_void_p, c_int, fp, dp, dp, dp, c_int, c_int, c_int, c_double]
    lib.rtgrff_render_los_map.argtypes = [c_void_p, c_int, c_int, dp, dp, c_int, dp, dp, c_double, c_double, c_double,
                                          c_int, dp, c_double, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int,
                                          POINTER(c_int64)]
    a = lib.rtgrff_render_los_map.argtypes
    lib.rtgrff_render_los_map_view.argtypes = a[:9] + [c_double, c_double] + a[9:]
    lib.rtgrff_gaussian_beam.argtypes = [c_void_p, dp, c_int, c_int, c_int, c_double, c_double, dp]
    lib.rtgrff_patch_nan.argtypes = [c_void_p, dp, c_int, c_int, c_int, c_int, POINTER(c_int64)]
    for name in EXPORTS:
        getattr(lib, name)          # AttributeError here = the .so is stale; rebuild it
    _lib = lib
    return lib


def check(rc):
    """Map a C return code to the Python exception the reference raises in the same situation."""
    if rc == RTGRFF_OK:
        return
    msg = load().rtgrff_last_error().decode(errors="replace")
    if rc == RTGRFF_EINVAL:
        raise ValueError(msg)
    if rc == RTGRFF_ENOMEM:
        raise MemoryError(msg)
    if rc == RTGRFF_EUNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError(msg)


def ptr(a, ctype):
    return None if a is None else a.ctypes.data_as(POINTER(ctype))


def cuda_array(a):
    """(device pointer, shape, typestr, strides) of an object exposing ``__cuda_array_interface__`` (CuPy
    arrays, torch CUDA tensors, numba device arrays), else None."""
    cai = getattr(a, "__cuda_array_interface__", None)
    if cai is None:
        return None
    return int(cai["data"][0]), tuple(cai["shape"]), cai["typestr"], cai.get("strides")


def is_f_contiguous(shape, strides, itemsize):
    """Fortran-contiguity of a __cuda_array_interface__ array (strides None = C-contiguous)."""
    if strides is None:
        return sum(1 for n in shape if n > 1) <= 1
    expect = itemsize
    for n, st in zip(shape, strides):
        if n > 1 and st != expect:
            return False
        expect *= n
    return True


def f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def check_uniform_grid(grid, name):
    """Grid validation of the reference (raytracingGRFF/gpu_raytrace.py:21-33): 1-D, >= 2 points,
    uniform within max(1e-6*|step|, 1e-7*max(|g0|,|g_last|,1)); returns (g0, mean step)."""
    g = np.asarray(grid, dtype=np.float64)
    if g.ndim != 1 or g.size < 2:
        raise ValueError(f"{name} must be 1D with at least 2 points")
    d = np.diff(g)
    step = float(np.mean(d))
    if not np.isfinite(step) or step <= 0.0:
        raise ValueError(f"{name} has invalid spacing")
    max_dev = float(np.max(np.abs(d - step)))
    tol = max(1e-6 * abs(step), 1e-7 * max(abs(g[0]), abs(g[-1]), 1.0))
    if max_dev > tol:
        raise ValueError(f"{name} must be uniformly spaced")
    return float(g[0]), step


def grid_geom(x_grid, y_grid, z_grid):
    """geom[12] of include/rtgrff.h: per axis {g0, mean step, g_last, g1-g0}."""
    out = np.empty(12, dtype=np.float64)
    for a, (g, name) in enumerate(((x_grid, "x_grid"), (y_grid, "y_grid"), (z_grid, "z_grid"))):
        g0, step = check_uniform_grid(g, name)
        gg = np.asarray(g, dtype=np.float64)
        out[4 * a: 4 * a + 4] = (g0, step, float(gg[-1]), float(gg[1] - gg[0]))
    return out


def current_device():
    """The calling thread's current CUDA device (what torch.cuda.set_device chose)."""
    d = load().rtgrff_current_device()
    if d < 0:
        raise RuntimeError(load().rtgrff_last_error().decode(errors="replace"))
    return d


class Context:
    """One GPU context (rtgrff_ctx).  `stream` is an int cudaStream_t handle — e.g.
    ``torch.cuda.current_stream().cuda_stream``, where 0 is the legacy default stream torch uses by
    default and is honoured as such — or None for a library-owned stream.  `device` None = the
    calling thread's current device."""

    def __init__(self, device=None, stream=None):
        lib = load()
        n = lib.rtgrff_device_count()
        if n <= 0:
            raise RuntimeError("No CUDA device is available to raytracinggrff_b200 "
                               f"({lib.rtgrff_last_error().decode(errors='replace') or 'device count 0'}); "
                               "this package has no CPU path.")
        if device is None:
            device = current_device()
        h = c_void_p()
        if stream is None:
            check(lib.rtgrff_ctx_create(int(device), None, ctypes.byref(h)))
        else:
            check(lib.rtgrff_ctx_create_on_stream(int(device), c_void_p(int(stream)), ctypes.byref(h)))
        self._h = h
        self.device = int(device)
        self.stream = stream
        self._lib = lib

    def close(self):
        if getattr(self, "_h", None):
            self._lib.rtgrff_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    @property
    def handle(self):
        if not self._h:
            raise RuntimeError("context is closed")
        return self._h

    @property
    def launch_count(self):
        return int(self._lib.rtgrff_ctx_launch_count(self.handle))

    @property
    def last_kernel_ms(self):
        return float(self._lib.rtgrff_ctx_last_kernel_ms(self.handle))

    def synchronize(self):
        check(self._lib.rtgrff_ctx_synchronize(self.handle))

    def set_grff64(self, enabled):
        """FP64 voxel evaluation in the per-ray kernels on / off (rtgrff_ctx_set_grff64)."""
        check(self._lib.rtgrff_ctx_set_grff64(self.handle, int(bool(enabled))))

    def set_pipeline(self, enabled):
        """Chunked pinned host pipelines on / off (rtgrff_ctx_set_pipeline)."""
        check(self._lib.rtgrff_ctx_set_pipeline(self.handle, int(bool(enabled))))


_default_ctx = {}


def default_context(device=None):
    """Process-wide context per device, used by the module-level drop-in functions; None = the
    calling thread's current device (a rank working on cuda:k stays on cuda:k)."""
    if device is None:
        device = current_device()
    ctx = _default_ctx.get(device)
    if ctx is None or not ctx._h:
        ctx = _default_ctx[device] = Context(device)
    return ctx
