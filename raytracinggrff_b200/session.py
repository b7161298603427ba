"""RaySession: cubes uploaded once, then any number of trace / sample / emission / render calls
on one GPU.  The drop-in functions of gpu_raytrace.py / build_rays.py / workflow.py are thin
wrappers over this class; every method maps 1:1 to an entry point of include/rtgrff.h."""
from __future__ import annotations

import ctypes
from ctypes import c_double, c_float, c_int64, c_uint8

import numpy as np

from . import _lib
from ._lib import FreqParams, check, f32, f64, ptr


def _s_mode(v):
    """'per_step' / 'cumulative' (or the RTGRFF_S_* integers) -> RTGRFF_S_*."""
    if isinstance(v, str):
        try:
            return {"per_step": _lib.S_PER_STEP, "cumulative": _lib.S_CUMULATIVE}[v.lower()]
        except KeyError:
            raise ValueError(f"Unsupported s_mode '{v}'. Use 'per_step' or 'cumulative'.") from None
    if int(v) not in (_lib.S_PER_STEP, _lib.S_CUMULATIVE):
        raise ValueError(f"Unsupported s_mode {v!r}")
    return int(v)


def _fingerprint(*arrays):
    """Identity + sampled content of host arrays: address, shape, dtype, strides and a hash of ~4096
    evenly spaced elements each.  Used to skip the re-upload of a cube the device already holds when the
    drop-in functions are called again with the same arrays (the reference re-uploads per call,
    gpu_raytrace.py:354, :681).  RTGRFF_CUBE_CACHE=0 turns the shortcut off."""
    import os
    if os.environ.get("RTGRFF_CUBE_CACHE", "1") == "0":
        return None
    key = []
    for a in arrays:
        if a is None:
            key.append(None)
            continue
        a = np.asarray(a)
        flat = a.reshape(-1) if a.flags.c_contiguous else a.ravel()
        step = max(1, flat.size // 4096)
        key.append((a.__array_interface__["data"][0], a.shape, a.dtype.str, a.strides,
                    hash(flat[::step].tobytes()), hash(flat[-1:].tobytes())))
    return tuple(key)


class RaySession:
    def __init__(self, device=None, stream=None, context=None):
        self.ctx = context if context is not None else _lib.Context(device, stream)
        self._lib = _lib.load()
        self.n_rec = 0
        self.n_rays = 0
        self.cube_shape = None
        self.world_size, self.rank = 1, 0
        self.traced_cs = False

    def close(self):
        for ptr_, _ in self.__dict__.pop("_scratch", {}).values():
            try:
                self._lib.rtgrff_device_free(self.ctx.handle, ctypes.c_void_p(ptr_))
            except Exception:      # the context may be gone already
                pass
        self.ctx.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- cubes ---------------------------------------------------------------------------------
    def set_omega_cube(self, omega_pe_3d, x_grid, y_grid, z_grid, reuse=False):
        """build_rays.py:132-143 / gpu_raytrace.py:346-357.  reuse=True: skip the upload when the context
        already holds the cube built from these very arrays (see _fingerprint)."""
        geom = _lib.grid_geom(x_grid, y_grid, z_grid)
        keys = self.ctx.__dict__.setdefault("_cube_keys", {})
        key = _fingerprint(omega_pe_3d, x_grid, y_grid, z_grid) if reuse else None
        if key is not None and keys.get("omega") == key:
            self.cube_shape = tuple(np.shape(omega_pe_3d))
            return
        keys["omega"] = None
        w = f64(omega_pe_3d)
        if w.ndim != 3 or w.shape != (len(x_grid), len(y_grid), len(z_grid)):
            raise ValueError(f"omega_pe_3d shape {w.shape} does not match the grids")
        check(self._lib.rtgrff_set_omega_cube(self.ctx.handle, w.ctypes.data_as(ctypes.c_void_p), *w.shape,
                                              ptr(geom, c_double), 0))
        self.cube_shape = tuple(w.shape)
        keys["omega"] = key

    def set_field_cubes(self, x_grid, y_grid, z_grid, ne_xyz, te_xyz, b_xyz, bx=None, by=None, bz=None, reuse=False):
        """gpu_raytrace.py:638-649 (_as_float32_c of each field, uniform-grid check)."""
        geom = _lib.grid_geom(x_grid, y_grid, z_grid)
        keys = self.ctx.__dict__.setdefault("_cube_keys", {})
        key = _fingerprint(ne_xyz, te_xyz, b_xyz, bx, by, bz, x_grid, y_grid, z_grid) if reuse else None
        if key is not None and keys.get("fields") == key:
            return
        keys["fields"] = None
        ne, te, b = f32(ne_xyz), f32(te_xyz), f32(b_xyz)
        shape = (len(x_grid), len(y_grid), len(z_grid))
        for name, a in (("ne_xyz", ne), ("te_xyz", te), ("b_xyz", b)):
            if a.shape != shape:
                raise ValueError(f"{name} shape {a.shape} does not match the grids {shape}")
        vec = [None, None, None]
        if bx is not None or by is not None or bz is not None:
            if bx is None or by is None or bz is None:
                raise ValueError("bx, by, bz must be given together")
            vec = [f32(bx), f32(by), f32(bz)]
            for a in vec:
                if a.shape != shape:
                    raise ValueError("B-vector cube shape does not match the grids")
        check(self._lib.rtgrff_set_field_cubes(self.ctx.handle, ptr(ne, c_float), ptr(te, c_float), ptr(b, c_float),
                                               ptr(vec[0], c_float), ptr(vec[1], c_float), ptr(vec[2], c_float),
                                               *shape, ptr(geom, c_double)))
        keys["fields"] = key

    def set_model_from_spherical(self, model, x_grid, y_grid, z_grid, phi0_offset=0.0, want_bvec=False, b0_angle=0.0,
                                 p_angle=0.0):
        """Cubes straight from a spherical (phi, latitude, r) model, never visiting the host
        (cubes.set_model_from_spherical; script/resample_with_ray_tracing.py:263-293), seen from the observer view
        b0_angle, p_angle [deg] (include/rtgrff.h, "Observer view")."""
        from . import cubes
        self.ctx.__dict__["_cube_keys"] = {}
        cubes.set_model_from_spherical(self, model, x_grid, y_grid, z_grid, phi0_offset, want_bvec, b0_angle=b0_angle,
                                       p_angle=p_angle)
        self.cube_shape = (len(x_grid), len(y_grid), len(z_grid))

    def set_spherical_model(self, model):
        """rtgrff_set_spherical_model for the five variables of a spherical model (a dict of cubes.SphericalVariable
        with 'rho', 'te' (or 't'), 'br', 'bt', 'bp'): resident on the device for render_los_map.  A variable the
        context already holds from these very arrays is not uploaded again (see _fingerprint)."""
        temp = "te" if "te" in model else "t"
        names = ("rho", temp, "br", "bt", "bp")
        for name in names:
            if name not in model:
                raise ValueError(f"the spherical model has no '{name}' variable")
        keys = self.ctx.__dict__.setdefault("_sph_keys", [None] * len(names))
        for slot, name in enumerate(names):
            var = model[name]
            key = _fingerprint(var.data, var.phi, var.lat, var.r)
            if key is not None:
                key += (float(var.scale),)
                if keys[slot] == key:
                    continue
            keys[slot] = None
            data, phi, lat, r = f32(var.data), f64(var.phi), f64(var.lat), f64(var.r)
            if data.shape != (len(phi), len(lat), len(r)):
                raise ValueError(f"'{name}' data shape {data.shape} does not match its (phi, lat, r) mesh")
            check(self._lib.rtgrff_set_spherical_model(self.ctx.handle, slot, ptr(data, c_float), ptr(phi, c_double),
                                                       ptr(lat, c_double), ptr(r, c_double), *data.shape,
                                                       float(var.scale)))
            keys[slot] = key

    # -- integrator ----------------------------------------------------------------------------
    def trace(self, freq_hz, x_start, y_start, z_start, kvec_in_norm, dt, n_steps, record_stride=10,
              trace_crosssections=False, perturb_ratio=2.0, s_mode=_lib.S_PER_STEP, fetch=True):
        """Integrate rays; returns (r_record (n_rec,n_rays,3) f64, S (n_rec,n_rays) f64 or None,
        active_steps).  With fetch=False the records only stay on the device."""
        xs, ys, zs = f64(x_start).ravel(), f64(y_start).ravel(), f64(z_start).ravel()
        n_rays = xs.shape[0]
        if ys.shape[0] != n_rays or zs.shape[0] != n_rays:
            raise ValueError("x_start, y_start, z_start must have the same length")
        kv = None
        if kvec_in_norm is not None:
            kv = f64(kvec_in_norm)
            if kv.shape != (n_rays, 3):
                raise ValueError(f"kvec_in_norm must have shape ({n_rays}, 3)")
        n_steps, stride = int(n_steps), int(record_stride)
        if stride < 1:
            raise ValueError("record_stride must be >= 1")
        n_rec = (n_steps + stride - 1) // stride if n_steps > 0 else 0
        r_record = np.empty((n_rec, n_rays, 3), dtype=np.float64) if fetch else None
        s_record = np.empty((n_rec, n_rays), dtype=np.float64) if (fetch and trace_crosssections) else None
        active = c_int64(0)
        check(self._lib.rtgrff_trace(self.ctx.handle, n_rays, ptr(xs, c_double), ptr(ys, c_double), ptr(zs, c_double),
                                     ptr(kv, c_double), float(freq_hz), float(dt), n_steps, stride,
                                     int(bool(trace_crosssections)), float(perturb_ratio), _s_mode(s_mode),
                                     ptr(r_record, c_double), ptr(s_record, c_double), ctypes.byref(active)))
        self.n_rec, self.n_rays, self.traced_cs = n_rec, n_rays, bool(trace_crosssections)
        return r_record, s_record, int(active.value)

    # -- sampler -------------------------------------------------------------------------------
    def sample(self, r_record, s_arr, ray_start, r_sun_cm, fill_ne=0.0, fill_te=1e4, fill_b=0.0):
        """gpu_raytrace.py:654-709 on host arrays; returns the reference's dict."""
        pos = f32(np.asarray(r_record))
        s = f32(np.asarray(s_arr))
        rs = f32(np.asarray(ray_start))
        if pos.ndim != 3 or pos.shape[2] != 3:
            raise ValueError("r_record must have shape (n_steps, n_rays, 3)")
        n_rec, n_rays, _ = pos.shape
        if s.shape != (n_rec, n_rays):
            raise ValueError("s_arr must have shape (n_steps, n_rays)")
        if rs.shape != (n_rays, 3):
            raise ValueError("ray_start must have shape (n_rays, 3)")
        out = {k: np.empty((n_rec, n_rays), dtype=np.float32) for k in ("ne", "te", "b", "ds")}
        valid = np.empty((n_rec, n_rays), dtype=np.uint8)
        check(self._lib.rtgrff_sample(self.ctx.handle, n_rec, n_rays, ptr(pos, c_float), ptr(s, c_float),
                                      ptr(rs, c_float), float(r_sun_cm), float(fill_ne), float(fill_te), float(fill_b),
                                      ptr(out["ne"], c_float), ptr(out["te"], c_float), ptr(out["b"], c_float),
                                      ptr(out["ds"], c_float), ptr(valid, c_uint8)))
        out["valid_mask"] = valid.view(np.bool_)      # 0/1 bytes: no copy
        out["s"] = s
        return out

    def sample_traced(self, ray_start, r_sun_cm, fill_ne=0.0, fill_te=1e4, fill_b=0.0, fetch=True):
        """Sampler on the records the last trace() left on the device."""
        rs = f32(np.asarray(ray_start))
        if rs.shape != (self.n_rays, 3):
            raise ValueError("ray_start must have shape (n_rays, 3)")
        shape = (self.n_rec, self.n_rays)
        out = {}
        valid = None
        if fetch:
            out = {k: np.empty(shape, dtype=np.float32) for k in ("ne", "te", "b", "ds", "s")}
            valid = np.empty(shape, dtype=np.uint8)
        check(self._lib.rtgrff_sample_traced(self.ctx.handle, ptr(rs, c_float), float(r_sun_cm), float(fill_ne),
                                             float(fill_te), float(fill_b), ptr(out.get("ne"), c_float),
                                             ptr(out.get("te"), c_float), ptr(out.get("b"), c_float),
                                             ptr(out.get("ds"), c_float), ptr(valid, c_uint8),
                                             ptr(out.get("s"), c_float)))
        if fetch:
            out["valid_mask"] = valid.view(np.bool_)      # 0/1 bytes: no copy
        return out

    # -- GRFF ----------------------------------------------------------------------------------
    def get_mw_slice(self, Lparms_M, Rparms_M, Parms_M, RL_M):
        """fastGRFF get_mw_slice contract (script/resample_with_ray_tracing.py:428-446); RL_M written
        in place (must be Fortran-ordered float64 (7,Nf,Npix)); returns status int32 (Npix).
        With device arrays (anything exposing ``__cuda_array_interface__``: the reference passes CuPy
        arrays) for Rparms_M / Parms_M / RL_M the call runs on them where they are and RL_M is written in
        place on the device; host numpy arrays are staged through the library."""
        dev = [_lib.cuda_array(a) for a in (Rparms_M, Parms_M, RL_M)]
        if any(d is not None for d in dev):
            return self._get_mw_slice_device(Lparms_M, dev, (Rparms_M, Parms_M, RL_M))
        L = self._host_ints(Lparms_M, 6)
        R = np.asfortranarray(Rparms_M, dtype=np.float64)
        P = np.asfortranarray(Parms_M, dtype=np.float64)
        npix, nz, nf = int(L[0]), int(L[1]), int(L[2])
        if P.shape != (15, nz, npix) or R.shape != (3, npix):
            raise ValueError("Parms_M must be (15,Nz,Npix) and Rparms_M (3,Npix)")
        if not (isinstance(RL_M, np.ndarray) and RL_M.dtype == np.float64 and RL_M.flags.f_contiguous
                and RL_M.shape == (7, nf, npix)):
            raise ValueError("RL_M must be a Fortran-ordered float64 array of shape (7,Nf,Npix)")
        status = np.zeros(npix, dtype=np.int32)
        check(self._lib.rtgrff_get_mw_slice(self.ctx.handle, ptr(L, ctypes.c_int32), ptr(R, c_double), ptr(P, c_double),
                                            None, None, None, ptr(RL_M, c_double), ptr(status, ctypes.c_int32)))
        return status

    def _host_ints(self, a, n):
        """n int32 values of a host or device array (Lparms_M is a CuPy array at the reference's call site)."""
        d = _lib.cuda_array(a)
        if d is None:
            return np.asarray(a, dtype=np.int32).ravel()[:n].copy()
        p, shape, typestr, _ = d
        if np.dtype(typestr) != np.int32 or int(np.prod(shape)) < n:
            raise ValueError("Lparms_M must hold at least 6 int32 values")
        out = np.empty(n, dtype=np.int32)
        check(self._lib.rtgrff_memcpy(self.ctx.handle, out.ctypes.data_as(ctypes.c_void_p), ctypes.c_void_p(p), 4 * n, 1))
        return out

    def _get_mw_slice_device(self, Lparms_M, dev, arrays):
        L = self._host_ints(Lparms_M, 6)
        npix, nz, nf = int(L[0]), int(L[1]), int(L[2])
        want = ((3, npix), (15, nz, npix), (7, nf, npix))
        ptrs, keep = [], []
        for name, d, a, shape in zip(("Rparms_M", "Parms_M", "RL_M"), dev, arrays, want):
            if d is None:
                if name == "RL_M":
                    raise TypeError("RL_M must be a device array when Rparms_M / Parms_M are (it is written in place)")
                # a host array next to device ones: stage it on the device for the call
                h = np.asfortranarray(a, dtype=np.float64)
                if h.shape != shape:
                    raise ValueError(f"{name} must have shape {shape}")
                buf = self._device_scratch(name, h.nbytes)
                check(self._lib.rtgrff_memcpy(self.ctx.handle, ctypes.c_void_p(buf), h.ctypes.data_as(ctypes.c_void_p), h.nbytes, 0))
                ptrs.append(buf)
                continue
            p, shp, typestr, strides = d
            if np.dtype(typestr) != np.float64 or tuple(shp) != shape:
                raise ValueError(f"{name} must be float64 with shape {shape}, got {typestr} {tuple(shp)}")
            if not _lib.is_f_contiguous(shp, strides, 8):
                raise ValueError(f"{name} must be Fortran-ordered (order='F'), as the reference builds it")
            ptrs.append(p)
            keep.append(a)
        status_dev = self._device_scratch("status", 4 * max(npix, 1))
        Lh = np.ascontiguousarray(L, dtype=np.int32)
        check(self._lib.rtgrff_get_mw_slice_device(self.ctx.handle, ptr(Lh, ctypes.c_int32), ctypes.c_void_p(ptrs[0]),
                                                   ctypes.c_void_p(ptrs[1]), ctypes.c_void_p(ptrs[2]),
                                                   ctypes.c_void_p(status_dev)))
        status = np.zeros(npix, dtype=np.int32)
        if npix:
            check(self._lib.rtgrff_memcpy(self.ctx.handle, status.ctypes.data_as(ctypes.c_void_p),
                                          ctypes.c_void_p(status_dev), 4 * npix, 1))
        return status

    def _device_scratch(self, key, nbytes):
        """Device scratch buffers owned by this session (rtgrff_device_alloc), grown on demand."""
        cache = self.__dict__.setdefault("_scratch", {})
        ent = cache.get(key)
        if ent is None or ent[1] < nbytes:
            p = ctypes.c_void_p()
            check(self._lib.rtgrff_device_alloc(self.ctx.handle, ctypes.byref(p), int(nbytes)))
            if ent is not None:
                self._lib.rtgrff_device_free(self.ctx.handle, ctypes.c_void_p(ent[0]))
            ent = cache[key] = (p.value, int(nbytes))
        return ent[0]

    def export_cubes(self, omega_pe=True, fields=True, bvec=False):
        """Host copies of the device cubes (rtgrff_export_cubes): the float64 omega_pe exactly as it was
        differenced, n_e / T / |B| and the B vector as stored.  For parity checks of cubes built on the
        device from a spherical model against a CPU implementation."""
        shape = self.cube_shape
        out = {}
        if omega_pe:
            out["omega_pe"] = np.empty(shape, dtype=np.float64)
        if fields:
            for k in ("ne", "te", "b"):
                out[k] = np.empty(shape, dtype=np.float32)
        if bvec:
            for k in ("bx", "by", "bz"):
                out[k] = np.empty(shape, dtype=np.float32)
        check(self._lib.rtgrff_export_cubes(self.ctx.handle, ptr(out.get("omega_pe"), c_double), ptr(out.get("ne"), c_float),
                                            ptr(out.get("te"), c_float), ptr(out.get("b"), c_float),
                                            ptr(out.get("bx"), c_float), ptr(out.get("by"), c_float),
                                            ptr(out.get("bz"), c_float)))
        return out

    # -- multi-GPU -----------------------------------------------------------------------------
    def comm_init(self, world_size, rank, unique_id=None):
        """rtgrff_comm_init_rank: NCCL communicator over the sessions of all ranks (collective)."""
        check(self._lib.rtgrff_comm_init_rank(self.ctx.handle, int(world_size), int(rank), unique_id))
        self.world_size, self.rank = int(world_size), int(rank)

    def comm_destroy(self):
        check(self._lib.rtgrff_comm_destroy(self.ctx.handle))

    def gather_image(self, slab_ptr, n_planes, n_rows, n_cols, root=0, out=None, out_device_ptr=None):
        """rtgrff_gather_image: the ranks' slabs (device float64 (n_planes, max_rows, n_cols)) -> the image
        (n_planes, n_rows, n_cols) on `root`: into `out` (host float64 array, page-locked memory is
        written by DMA directly) or to the device pointer `out_device_ptr`.  Returns `out` on the root."""
        if out_device_ptr is not None:
            dst, on_dev = ctypes.c_void_p(int(out_device_ptr)), 1
        elif out is not None:
            if out.dtype != np.float64 or not out.flags.c_contiguous or out.size != n_planes * n_rows * n_cols:
                raise ValueError("out must be a C-contiguous float64 array of n_planes*n_rows*n_cols elements")
            dst, on_dev = out.ctypes.data_as(ctypes.c_void_p), 0
        else:
            dst, on_dev = None, 0
        check(self._lib.rtgrff_gather_image(self.ctx.handle, ctypes.c_void_p(int(slab_ptr)), int(n_planes), int(n_rows),
                                            int(n_cols), int(root), dst, on_dev))
        return out

    def emission_traced(self, pixel_area_cm2, freq0, n_freq=1, freq_log_step=0.0, em_flag=5, s_max=30,
                        s_input_on=False):
        """script/resample_with_ray_tracing.py:467-530 on the device samples; returns (tb, vi) each
        (n_rays, n_freq) float64."""
        tb = np.empty((self.n_rays, int(n_freq)), dtype=np.float64)
        vi = np.empty_like(tb)
        check(self._lib.rtgrff_emission_traced(self.ctx.handle, float(pixel_area_cm2), float(freq0), int(n_freq),
                                               float(freq_log_step), int(em_flag), int(s_max), int(bool(s_input_on)),
                                               ptr(tb, c_double), ptr(vi, c_double)))
        return tb, vi

    # -- fused map -----------------------------------------------------------------------------
    def render_map(self, x_start, y_start, z_start, freq_params, kvec_in_norm=None, trace_crosssections=True,
                   perturb_ratio=2.0, pixel_area_cm2=1.0, r_sun_cm=6.957e10, em_flag=5, s_max=30, use_bvec=False,
                   voxel_order=_lib.ORDER_RECORD, out_device_ptrs=None, image_shape=None, tile=(4, 8), ray_order=None,
                   s_mode="per_step", s_input_on=False):
        """Fused trace+sample+transfer.  freq_params: sequence of dicts/tuples
        (freq_hz, dt, n_steps, record_stride).  Returns (tb, vi) each (n_freq, n_rays) float64 and
        stats {nominal_ray_steps, active_ray_steps}; with out_device_ptrs=(tb_ptr, vi_ptr) the
        results are written to those device buffers instead and (None, None, stats) is returned.
        image_shape=(n_rows, n_cols): the rays are a row-major image (ray p = i*n_cols + j); threads
        then walk it in `tile` = (width, height) pixel tiles, which keeps a warp's 32 rays in a compact
        patch (-11 % on config 4); results keep the caller's ray numbering.
        s_mode 'per_step' | 'cumulative': the cross-section ratio a record carries (reference CPU / CUDA
        path); s_input_on: that S multiplies the voxel's source term (``--s-input-on``, see include/rtgrff.h)."""
        return self._render(False, x_start, y_start, z_start, freq_params, kvec_in_norm, trace_crosssections,
                            perturb_ratio, pixel_area_cm2, r_sun_cm, em_flag, s_max, use_bvec, voxel_order,
                            out_device_ptrs, image_shape, tile, ray_order, s_mode, s_input_on)

    def render_map_diag(self, x_start, y_start, z_start, freq_params, kvec_in_norm=None, trace_crosssections=True,
                        perturb_ratio=2.0, pixel_area_cm2=1.0, r_sun_cm=6.957e10, em_flag=5, s_max=30, use_bvec=False,
                        voxel_order=_lib.ORDER_RECORD, out_device_ptrs=None, image_shape=None, tile=(4, 8),
                        ray_order=None, s_mode="per_step", s_input_on=False):
        """render_map with the map diagnostics (rtgrff_render_map_diag): where the emission of every (pixel,
        frequency) comes from.  Same keywords and the same tb, vi; returns (tb, vi, stats, diag) with diag a dict of
        (n_freq, n_rays) float64 arrays: em_x, em_y, em_z (emission centroid [R_sun]), em_r (contribution-weighted
        mean heliocentric distance [R_sun]), tau_L, tau_R (total optical depth of the L and R slot), ray_r_min
        (the ray's turning point [R_sun]); definitions in include/rtgrff.h.  With out_device_ptrs=(tb_ptr, vi_ptr,
        diag_ptr) everything goes to device buffers (diag: 7 n_freq planes of n_rays) and (None, None, stats,
        None) is returned."""
        return self._render(True, x_start, y_start, z_start, freq_params, kvec_in_norm, trace_crosssections,
                            perturb_ratio, pixel_area_cm2, r_sun_cm, em_flag, s_max, use_bvec, voxel_order,
                            out_device_ptrs, image_shape, tile, ray_order, s_mode, s_input_on)

    def _render(self, diag, x_start, y_start, z_start, freq_params, kvec_in_norm, trace_crosssections, perturb_ratio,
                pixel_area_cm2, r_sun_cm, em_flag, s_max, use_bvec, voxel_order, out_device_ptrs, image_shape, tile,
                ray_order, s_mode, s_input_on):
        xs, ys, zs = f64(x_start).ravel(), f64(y_start).ravel(), f64(z_start).ravel()
        n_rays = xs.shape[0]
        kv = None
        if kvec_in_norm is not None:
            kv = f64(kvec_in_norm)
            if kv.shape != (n_rays, 3):
                raise ValueError(f"kvec_in_norm must have shape ({n_rays}, 3)")
        order = None
        if ray_order is not None:
            order = np.ascontiguousarray(ray_order, dtype=np.int32)
        elif image_shape is not None and tile is not None:
            n_rows, n_cols = image_shape
            if n_rows * n_cols != n_rays:
                raise ValueError("image_shape does not match the number of rays")
            from .synthetic import tile_order
            order = tile_order(n_cols, n_rows, tile[0], tile[1]).astype(np.int32)
        if order is not None and order.shape != (n_rays,):
            raise ValueError("ray_order must be a permutation of the rays")
        nf = len(freq_params)
        arr = (FreqParams * nf)()
        for i, p in enumerate(freq_params):
            if isinstance(p, dict):
                p = (p["freq_hz"], p["dt"], p["n_steps"], p["record_stride"])
            arr[i] = FreqParams(float(p[0]), float(p[1]), int(p[2]), int(p[3]))
        stats = (c_int64 * 4)()
        dg = None
        if out_device_ptrs is None:
            tb = np.empty((nf, n_rays), dtype=np.float64)
            vi = np.empty_like(tb)
            ptb, pvi, on_dev = tb.ctypes.data_as(ctypes.c_void_p), vi.ctypes.data_as(ctypes.c_void_p), 0
            if diag:
                dg = np.empty((len(_lib.DIAG_PLANES), nf, n_rays), dtype=np.float64)
                pdg = dg.ctypes.data_as(ctypes.c_void_p)
        else:
            if diag and len(out_device_ptrs) != 3:
                raise ValueError("out_device_ptrs must be (tb_ptr, vi_ptr, diag_ptr)")
            tb = vi = None
            ptb, pvi, on_dev = ctypes.c_void_p(out_device_ptrs[0]), ctypes.c_void_p(out_device_ptrs[1]), 1
            if diag:
                pdg = ctypes.c_void_p(out_device_ptrs[2])
        args = (self.ctx.handle, n_rays, ptr(xs, c_double), ptr(ys, c_double), ptr(zs, c_double), ptr(kv, c_double),
                ptr(order, ctypes.c_int32), nf, arr, int(bool(trace_crosssections)), float(perturb_ratio),
                float(pixel_area_cm2), float(r_sun_cm), int(em_flag), int(s_max), int(bool(use_bvec)), int(voxel_order),
                _s_mode(s_mode), int(bool(s_input_on)), ptb, pvi, on_dev, stats)
        if diag:
            check(self._lib.rtgrff_render_map_diag(*args, pdg))
        else:
            check(self._lib.rtgrff_render_map(*args))
        st = {"nominal_ray_steps": int(stats[0]), "active_ray_steps": int(stats[1]),
              "pencil_steps": int(stats[2]), "valid_samples": int(stats[3])}
        if not diag:
            return tb, vi, st
        return tb, vi, st, (None if dg is None else dict(zip(_lib.DIAG_PLANES, dg)))

    # -- fused straight line-of-sight map ---------------------------------------------------------
    def render_los_map(self, x, y, zc, dz_cm, freq_hz, phi0_offset=0.0, r_min=0.9999999, z_eps=1e-6 / 6.957e8,
                       pixel_area_cm2=1.0, em_flag=5, s_max=30, use_bvec=False, diagnostics=False,
                       out_device_ptrs=None, b0_angle=0.0, p_angle=0.0):
        """Straight-LOS map from the model set_spherical_model left on the device (rtgrff_render_los_map): pixel
        (i, j) at (x[j], y[i]) [R_sun], LOS samples at the cumulative offsets zc [R_sun] with segment lengths dz_cm
        [cm], any list of frequencies [Hz].  Returns (tb, vi, stats), tb and vi (n_freq, ny, nx) float64, stats
        {los_samples, valid_samples, voxel_freq_evaluations}; with diagnostics=True (tb, vi, stats, diag), diag a
        dict of (n_freq, ny, nx) planes with render_map_diag's keys.  With out_device_ptrs=(tb_ptr, vi_ptr[,
        diag_ptr]) the results go to those device buffers and the arrays returned are None.  b0_angle, p_angle [deg]:
        the observer's view of the model (include/rtgrff.h, "Observer view"); the diagnostic planes stay in the
        observer frame."""
        from .cubes import check_view
        b0, p = check_view(b0_angle, p_angle)
        xs, ys, z, d = f64(x).ravel(), f64(y).ravel(), f64(zc).ravel(), f64(dz_cm).ravel()
        fr = f64(np.atleast_1d(freq_hz)).ravel()
        if len(d) != len(z):
            raise ValueError("zc and dz_cm must have the same length")
        nf, ny, nx = len(fr), len(ys), len(xs)
        stats = (c_int64 * 3)()
        tb = vi = dg = None
        if out_device_ptrs is None:
            tb = np.empty((nf, ny, nx), dtype=np.float64)
            vi = np.empty_like(tb)
            ptb, pvi, on_dev = tb.ctypes.data_as(ctypes.c_void_p), vi.ctypes.data_as(ctypes.c_void_p), 0
            if diagnostics:
                dg = np.empty((len(_lib.DIAG_PLANES), nf, ny, nx), dtype=np.float64)
            pdg = None if dg is None else dg.ctypes.data_as(ctypes.c_void_p)
        else:
            if len(out_device_ptrs) != (3 if diagnostics else 2):
                raise ValueError("out_device_ptrs must be (tb_ptr, vi_ptr) or, with diagnostics, (tb_ptr, vi_ptr, diag_ptr)")
            ptb, pvi, on_dev = ctypes.c_void_p(out_device_ptrs[0]), ctypes.c_void_p(out_device_ptrs[1]), 1
            pdg = ctypes.c_void_p(out_device_ptrs[2]) if diagnostics else None
        check(self._lib.rtgrff_render_los_map_view(self.ctx.handle, nx, ny, ptr(xs, c_double), ptr(ys, c_double),
                                                   len(z), ptr(z, c_double), ptr(d, c_double), float(phi0_offset), b0, p,
                                                   float(r_min), float(z_eps), nf, ptr(fr, c_double),
                                                   float(pixel_area_cm2), int(em_flag), int(s_max), int(bool(use_bvec)),
                                                   ptb, pvi, pdg, on_dev, stats))
        st = {"los_samples": int(stats[0]), "valid_samples": int(stats[1]), "voxel_freq_evaluations": int(stats[2])}
        if not diagnostics:
            return tb, vi, st
        return tb, vi, st, (None if dg is None else dict(zip(_lib.DIAG_PLANES, dg)))
