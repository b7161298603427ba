"""Cube builder: spherical (phi, latitude, r) model variables -> the xyz cubes of the ray path, on
the GPU (SURVEY.md §8f rank 1).

Drop-in for the resampling helpers of the reference, with the MAS/psipy I/O replaced by in-memory
arrays:

* ``cart_to_sph``               — raytracingGRFF/build_rays.py:35-45
* ``resample_to_xyz_cube``      — raytracingGRFF/build_rays.py:69-125 (and ``resample_var_to_cube``,
                                  script/resample_with_ray_tracing.py:110-151)
* ``RaySession.set_model_from_spherical`` (session.py) — script/resample_with_ray_tracing.py:263-293

Beyond the reference, ``b0_angle`` / ``p_angle`` (degrees) view the model from any observer: the solar B0 angle
tilts the north pole towards the observer, the P angle turns it from image +y towards east (-x).  The conventions
are written out in include/rtgrff.h ("Observer view"); zero angles are the reference's fixed equatorial view.

A model is a mapping ``name -> SphericalVariable``; every variable carries its own mesh (MAS
staggers br, bt, bp) and the factor that converts its stored values to cm^-3 / K / G (what psipy's
unit handling does).
"""
from __future__ import annotations

import ctypes
from ctypes import c_double, c_float
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import check, f32, f64, ptr

R_MIN = 0.9999999      # raytracingGRFF/build_rays.py:26 (the workflow script uses 0.999999, :71)
SLOTS = {"rho": 0, "te": 1, "t": 1, "br": 2, "bt": 3, "bp": 4}


@dataclass
class SphericalVariable:
    data: np.ndarray      # (n_phi, n_lat, n_r), psipy's (phi, theta, r) order
    phi: np.ndarray       # longitude nodes, rad, ascending in [0, 2 pi)
    lat: np.ndarray       # latitude nodes, rad, ascending
    r: np.ndarray         # radius nodes, R_sun, ascending
    scale: float = 1.0    # stored value -> physical unit


def cart_to_sph(x, y, z, phi0_offset=0.0):
    """build_rays.py:35-45."""
    r = np.sqrt(x ** 2 + y ** 2 + z ** 2)
    colat = np.arccos(np.clip(z / r, -1.0, 1.0))
    lon = np.arctan2(y, x)
    lon = lon + phi0_offset * np.pi / 180.0
    lon = np.where(lon < 0, lon + 2 * np.pi, lon)
    return r, colat, lon


def check_view(b0_angle, p_angle):
    """The observer view's angles [deg] as floats: finite, |B0| <= 90, else ValueError (the C library's rule, checked
    here so that a front end fails before any GPU work)."""
    b0, p = float(b0_angle), float(p_angle)
    if not (np.isfinite(b0) and np.isfinite(p)):
        raise ValueError(f"b0_angle and p_angle must be finite (got {b0_angle!r}, {p_angle!r})")
    if abs(b0) > 90.0:
        raise ValueError(f"|b0_angle| must be <= 90 deg (got {b0_angle!r})")
    return b0, p


def load_mas_var_filtered(model, var_name):
    """``raytracingGRFF/build_rays.py:48-66`` reads ``<var>NNN.hdf`` files of a psipy ``MASOutput`` — file I/O
    that is out of scope here (psipy is not available).  For the in-memory models of this package
    (``name -> SphericalVariable``) it returns the variable, so code written against the reference's
    import keeps working on them; anything else raises."""
    if isinstance(model, dict) and var_name in model and isinstance(model[var_name], SphericalVariable):
        return model[var_name]
    raise RuntimeError("load_mas_var_filtered: reading MAS HDF files needs psipy (out of scope); pass a model "
                       "{name: SphericalVariable} (cubes.load_spherical_model) instead")


def _resample(ctx, slot, var, x_grid, y_grid, z_grid, phi0_offset, fill_nan, r_min, fetch, b0_angle=0.0, p_angle=0.0):
    b0, p = check_view(b0_angle, p_angle)
    geom = _lib.grid_geom(x_grid, y_grid, z_grid)
    data = f32(var.data)
    phi, lat, r = f64(var.phi), f64(var.lat), f64(var.r)
    if data.shape != (phi.size, lat.size, r.size):
        raise ValueError(f"data shape {data.shape} does not match the mesh ({phi.size}, {lat.size}, {r.size})")
    shape = (len(x_grid), len(y_grid), len(z_grid))
    xg, yg, zg = f64(x_grid), f64(y_grid), f64(z_grid)
    out = np.empty(shape, dtype=np.float64) if fetch else None
    fill = 0.0 if fill_nan is None else float(fill_nan)
    check(_lib.load().rtgrff_resample_spherical_view(ctx.handle, slot, ptr(data, c_float), ptr(phi, c_double),
                                                     ptr(lat, c_double), ptr(r, c_double), *data.shape, ptr(xg, c_double),
                                                     ptr(yg, c_double), ptr(zg, c_double), *shape,
                                                     ptr(geom, c_double), float(phi0_offset), b0, p, float(r_min),
                                                     float(var.scale), fill, int(fill_nan is not None),
                                                     ptr(out, c_double)))
    return out


def resample_to_xyz_cube(model, var_name, x_grid, y_grid, z_grid, phi0_offset=0.0, fill_nan=0.0, verbose=True,
                         r_min=R_MIN, context=None, b0_angle=0.0, p_angle=0.0):
    """Resample one model variable onto a regular xyz grid (build_rays.py:69-70); returns float64
    (nx, ny, nz) in the variable's physical unit.  b0_angle, p_angle [deg]: the observer's view."""
    check_view(b0_angle, p_angle)
    ctx = context or _lib.default_context()
    slot = SLOTS.get(var_name, 0)
    return _resample(ctx, slot, model[var_name], x_grid, y_grid, z_grid, phi0_offset, fill_nan, r_min, True,
                     b0_angle, p_angle)


def set_model_from_spherical(session, model, x_grid, y_grid, z_grid, phi0_offset=0.0, want_bvec=False,
                             r_min=0.999999, b0_angle=0.0, p_angle=0.0):
    """script/resample_with_ray_tracing.py:263-293 entirely on the device: resample rho, te, br, bt,
    bp with the fills used there (0, NaN, 0, 0, 0), then compose omega_pe (+ gradient), n_e, T, |B|.
    b0_angle, p_angle [deg]: the observer's view; the B vector (want_bvec) is in the observer frame."""
    check_view(b0_angle, p_angle)
    temp = "te" if "te" in model else "t"
    if temp not in model:
        raise ValueError("No electron temperature variable (te or t) found.")
    for k in ("br", "bt", "bp"):
        if k not in model:
            raise ValueError("Magnetic field components (br, bt, bp) not all found.")
    ctx = session.ctx
    for name, fill in (("rho", 0.0), (temp, None), ("br", 0.0), ("bt", 0.0), ("bp", 0.0)):
        _resample(ctx, SLOTS[name], model[name], x_grid, y_grid, z_grid, phi0_offset, fill, r_min, False, b0_angle,
                  p_angle)
    check(_lib.load().rtgrff_compose_cubes(ctx.handle, int(bool(want_bvec))))


def save_spherical_model(path, model):
    """Write a model (name -> SphericalVariable) to one .npz: the in-memory stand-in for a MAS directory
    that the command lines accept (``--model-path``)."""
    arrays = {}
    for name, v in model.items():
        arrays[f"{name}__data"] = np.asarray(v.data, dtype=np.float32)
        arrays[f"{name}__phi"], arrays[f"{name}__lat"], arrays[f"{name}__r"] = f64(v.phi), f64(v.lat), f64(v.r)
        arrays[f"{name}__scale"] = np.float64(v.scale)
    np.savez_compressed(path, **arrays)


def load_spherical_model(path):
    """Inverse of save_spherical_model.  Raises FileNotFoundError like the reference does for a missing
    model directory."""
    with np.load(path) as z:
        names = sorted({k.split("__")[0] for k in z.files})
        return {n: SphericalVariable(z[f"{n}__data"], z[f"{n}__phi"], z[f"{n}__lat"], z[f"{n}__r"],
                                     float(z[f"{n}__scale"])) for n in names}
