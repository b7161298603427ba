"""Straight line-of-sight workflow (BASELINE config 2) on the GPU: the drop-in counterparts of

* ``resample_MAS``  — script/resampling_MAS_LOS.py:100-301 (LOS/resample_MAS_LOS.py is its older copy):
  sample rho, te, br, bt, bp of a spherical model along one straight LOS per pixel on the irregular z
  grid ``dz = dz0 (1 + (5 i/N_z)^2.5)`` and write ``LOS_data.npz``;
* ``SyntheticFF``   — script/synthetic_FF_map_single_thread.py:108-244: per-pixel NaN filter, Parms
  packing (theta = 90, flag 1+4, s_max 30), GET_MW, SFU -> T_b, ``<out>.npz``;
* ``render_los_map`` — both in one fused kernel (rtgrff_render_los_map) with nothing materialised, optionally with
  gyroresonance, theta from the B vector and the emission diagnostics.

The MAS/psipy model is replaced by a mapping of cubes.SphericalVariable (SURVEY.md §8, row 11/12);
everything after the model read keeps the reference's names, array shapes, units and file keys.
"""
from __future__ import annotations

from ctypes import c_double, c_float

import numpy as np

from . import _lib
from ._lib import check, f32, f64, ptr
from .cubes import check_view
from .session import RaySession

R_sun_cm = 6.957e10     # script/resampling_MAS_LOS.py constants
R_sun_m = 6.957e8
R_MIN = 0.9999999
c = 2.998e10            # script/synthetic_FF_map_single_thread.py constants
kb = 1.38065e-16
sfu2cgs = 1e-19


def z_grid(N_z, dz0, variable_spacing_z=True, z_range=None):
    """script/resampling_MAS_LOS.py:141-156: returns (z_coords_Rsun, dz)."""
    if variable_spacing_z:
        idx_z = np.arange(N_z)
        dz = dz0 * (1 + (5 * idx_z / N_z) ** 2.5)
        return np.cumsum(dz), dz
    if z_range is None:
        z_range = [0.0, 4.0]
    z = np.linspace(z_range[0], z_range[1], N_z)
    return z, np.abs(np.diff(z, prepend=z[0]))


def _sample_los(ctx, var, x, y, zc, phi0_offset, r_min, b0_angle, p_angle):
    data = f32(var.data)
    phi, lat, r = f64(var.phi), f64(var.lat), f64(var.r)
    out = np.empty((len(y), len(x), len(zc)), dtype=np.float64)
    check(_lib.load().rtgrff_sample_spherical_los_view(ctx.handle, ptr(data, c_float), ptr(phi, c_double),
                                                       ptr(lat, c_double), ptr(r, c_double), *data.shape,
                                                       ptr(x, c_double), ptr(y, c_double), ptr(zc, c_double), len(x),
                                                       len(y), len(zc), float(phi0_offset), b0_angle, p_angle,
                                                       float(r_min), float(var.scale), 1e-6 / R_sun_m,
                                                       ptr(out, c_double)))
    return out


def _check_model(model, dz0, variable_spacing_z):
    """resample_MAS's argument checks (script/resampling_MAS_LOS.py); returns the temperature key."""
    if variable_spacing_z and dz0 > 1.0:
        raise ValueError(f"dz0={dz0:g} is extremely large in R_sun units. Did you mean something like 7e-4 instead of 7e4?")
    temp = "te" if "te" in model else "t"
    if temp not in model:
        raise ValueError("No electron temperature variable (te or t) found!")
    for k in ("br", "bt", "bp"):
        if k not in model:
            raise ValueError("Magnetic field components (br, bt, bp) not all found!")
    return temp


def resample_MAS(model, N_pix, X_range, Y_range, N_z, dz0, variable_spacing_z=True, z_range=None,
                 out_path="LOS_data.npz", save_plots=False, verbose=True, phi0_offset=0.0, r_min=R_MIN, context=None,
                 b0_angle=0.0, p_angle=0.0):
    """Returns {'Ne_LOS','Te_LOS','B_LOS','ds_LOS' (N_pix,N_pix,N_z) [cm^-3, K, G, cm], 'x_coords',
    'y_coords','z_coords' [m]} and writes them to `out_path` (script/resampling_MAS_LOS.py:288-300).
    b0_angle, p_angle [deg]: the observer's view of the model (include/rtgrff.h, "Observer view")."""
    temp = _check_model(model, dz0, variable_spacing_z)
    b0, p = check_view(b0_angle, p_angle)
    ctx = context or _lib.default_context()
    zc, dz = z_grid(N_z, dz0, variable_spacing_z, z_range)
    xs = np.linspace(X_range[0], X_range[1], N_pix)
    ys = np.linspace(Y_range[0], Y_range[1], N_pix)
    s = {k: _sample_los(ctx, model[k], xs, ys, zc, phi0_offset, r_min, b0, p) for k in ("rho", temp, "br", "bt", "bp")}
    B = np.sqrt(s["br"] ** 2 + s["bt"] ** 2 + s["bp"] ** 2)
    invalid = np.isnan(s["rho"])
    for a in (s[temp], B):
        a[invalid] = np.nan
    if not (np.isfinite(s["rho"]).any() or np.isfinite(s[temp]).any() or np.isfinite(B).any()):
        raise RuntimeError("All sampled LOS values are NaN. Check --dz0 units (R_sun); common mistake is 7e4 vs 7e-4.")
    result = {
        "Ne_LOS": s["rho"], "Te_LOS": s[temp], "B_LOS": B,
        "ds_LOS": np.broadcast_to(dz * R_sun_cm, s["rho"].shape).copy(),
        "x_coords": xs * R_sun_m, "y_coords": ys * R_sun_m, "z_coords": zc * R_sun_m,
    }
    if out_path is not None:
        np.savez_compressed(out_path, **result)
    return result


def SyntheticFF(fname_input, freq0, Nfreq, freq_log_step, fname_output=None, do_inspection_plot=False, session=None):
    """`fname_input`: path of a LOS npz or the dict resample_MAS returns.  Returns (and writes to
    ``fname_output + '.npz'``) emission_cube, emission_polVI_cube (N_pix,N_pix,Nf), frequencies_Hz,
    x_coords, y_coords — script/synthetic_FF_map_single_thread.py:108-244 with one batched GET_MW."""
    data = np.load(fname_input) if isinstance(fname_input, (str, bytes)) or hasattr(fname_input, "__fspath__") else fname_input
    Ne, Te, B, ds = (np.asarray(data[k]) for k in ("Ne_LOS", "Te_LOS", "B_LOS", "ds_LOS"))
    x_coords, y_coords = np.asarray(data["x_coords"]), np.asarray(data["y_coords"])
    n_y, n_x, N_z = Ne.shape
    Nf = int(Nfreq)
    frequencies_Hz = freq0 * (10.0 ** (freq_log_step * np.arange(Nf)))
    pixel_size_Rsun = (x_coords[1] - x_coords[0]) / (R_sun_cm * 1e-2)          # :156-158
    pixel_size_cm = pixel_size_Rsun * R_sun_cm
    area = pixel_size_cm * pixel_size_cm
    npix = n_y * n_x
    valid = ~(np.isnan(Ne) | np.isnan(Te) | np.isnan(B)).reshape(npix, N_z)     # :177
    order = np.argsort(~valid, axis=1, kind="stable")
    keep = np.arange(N_z)[None, :] < valid.sum(axis=1)[:, None]
    P = np.zeros((15, N_z, npix), dtype=np.float64, order="F")                   # :188-200
    P[4], P[6], P[7] = 90.0, 1 + 4, 30
    for m, a in ((0, ds), (1, Te), (2, Ne), (3, B)):
        P[m] = np.where(keep, np.take_along_axis(a.reshape(npix, N_z), order, axis=1), 0.0).T
    L = np.array([npix, N_z, Nf, 1, 0, 0], dtype=np.int32)
    R = np.zeros((3, npix), dtype=np.float64, order="F")
    R[0], R[1], R[2] = area, freq0, freq_log_step
    RL = np.zeros((7, Nf, npix), dtype=np.float64, order="F")
    ses = session or RaySession(context=_lib.default_context())
    status = ses.get_mw_slice(L, R, P, RL)
    inten = (RL[5] + RL[6]).T                                                    # (npix, Nf), :212
    with np.errstate(invalid="ignore", divide="ignore"):
        pol = ((RL[5] - RL[6]) / (RL[5] + RL[6])).T                              # :213 (no epsilon here)
    nu_hz = np.where(RL[0].T > 0, RL[0].T * 1e9, frequencies_Hz[None, :])
    conv = (sfu2cgs * c * c / (2.0 * kb * nu_hz * nu_hz) / area) * (1.49599e13 * 1.49599e13)
    emission = inten * conv
    dead = (status != 0) | (valid.sum(axis=1) == 0)
    emission[dead] = 0.0
    pol[dead] = 0.0
    result = {"emission_cube": emission.reshape(n_y, n_x, Nf), "emission_polVI_cube": pol.reshape(n_y, n_x, Nf),
              "frequencies_Hz": frequencies_Hz, "x_coords": x_coords, "y_coords": y_coords}
    if fname_output is not None:
        np.savez_compressed(str(fname_output) + ".npz", **result)
    return result


def render_los_map(model, N_pix, X_range, Y_range, N_z, dz0, freq0, Nfreq, freq_log_step, variable_spacing_z=True,
                   z_range=None, phi0_offset=0.0, r_min=R_MIN, em_flag=5, s_max=30, use_bvec=False, diagnostics=False,
                   fname_output=None, session=None, b0_angle=0.0, p_angle=0.0):
    """resample_MAS followed by SyntheticFF in one fused kernel: the same LOS geometry and samples, the same packing
    rules and T_b / V/I, with nothing materialised (no LOS arrays, no Parms).  Returns (and writes to
    ``fname_output + '.npz'``) SyntheticFF's dict.  Beyond the reference: em_flag (4 adds gyroresonance), use_bvec
    (theta from the B vector instead of 90 deg) and diagnostics=True, which adds the keys of
    workflow.diagnostic_maps (emission centroid, emission height, optical depths, the LOS's smallest r), and the
    observer's view b0_angle, p_angle [deg] (include/rtgrff.h, "Observer view")."""
    _check_model(model, dz0, variable_spacing_z)
    check_view(b0_angle, p_angle)
    if int(N_pix) < 2:
        raise ValueError("N_pix must be >= 2 (the pixel area comes from the x spacing)")
    if int(Nfreq) < 1:
        raise ValueError("Nfreq must be >= 1")
    zc, dz = z_grid(N_z, dz0, variable_spacing_z, z_range)
    xs = np.linspace(X_range[0], X_range[1], N_pix)
    ys = np.linspace(Y_range[0], Y_range[1], N_pix)
    x_coords, y_coords = xs * R_sun_m, ys * R_sun_m
    Nf = int(Nfreq)
    frequencies_Hz = freq0 * (10.0 ** (freq_log_step * np.arange(Nf)))
    pixel_size_cm = (x_coords[1] - x_coords[0]) / (R_sun_cm * 1e-2) * R_sun_cm
    area = pixel_size_cm * pixel_size_cm
    ses = session or RaySession(context=_lib.default_context())
    ses.set_spherical_model(model)
    out = ses.render_los_map(xs, ys, zc, dz * R_sun_cm, frequencies_Hz, phi0_offset=phi0_offset, r_min=r_min,
                             z_eps=1e-6 / R_sun_m, pixel_area_cm2=area, em_flag=em_flag, s_max=s_max,
                             use_bvec=use_bvec, diagnostics=diagnostics, b0_angle=b0_angle, p_angle=p_angle)
    tb, vi = out[0], out[1]
    result = {"emission_cube": np.ascontiguousarray(np.moveaxis(tb, 0, -1)),
              "emission_polVI_cube": np.ascontiguousarray(np.moveaxis(vi, 0, -1)),
              "frequencies_Hz": frequencies_Hz, "x_coords": x_coords, "y_coords": y_coords}
    if diagnostics:
        from .workflow import diagnostic_maps
        result.update(diagnostic_maps({k: v.reshape(Nf, -1) for k, v in out[3].items()}, N_pix))
    if fname_output is not None:
        np.savez_compressed(str(fname_output) + ".npz", **result)
    return result
