"""ORACLE — TEST INFRASTRUCTURE ONLY: the observer view (solar B0 and P angles) on the CPU.

The cube builder, the LOS sampler and the fused LOS map take the observer's B0 and P angles (include/rtgrff.h,
"Observer view").  This module restates them with plain numpy rotation matrices on top of oracle/oracle_cubes.py and
tests/los_map_oracle.py, which stay the zero-view yardsticks:

* ``view_matrix``: the 3 x 3 matrix M with p_model = M p_observer (undo P about z, then B0 about x);
* ``resample_to_xyz_cube``, ``compose_cubes`` (with the Cartesian B vector bx, by, bz in observer axes),
  ``resample_MAS``, ``los_samples`` and ``bvec_theta_deg`` with ``b0_angle`` / ``p_angle`` keywords [deg];
* ``solar_north``: n = (-sin P cos B0, cos P cos B0, sin B0) in observer axes.
"""
from __future__ import annotations

import numpy as np

from oracle import oracle_cubes as oc
import los_map_oracle as lmo

R_SUN_M = 6.957e8
_zero_view_theta = lmo.bvec_theta_deg     # held here, so that a test may hand los_map_oracle this module's theta


def _sin_cos(deg):
    """sin, cos of an angle in degrees, exact zeros at multiples of 90 deg (a point on an axis stays on it)."""
    a = np.radians(deg)
    s, c = np.sin(a), np.cos(a)
    return (0.0 if abs(s) < 1e-15 else s), (0.0 if abs(c) < 1e-15 else c)


def view_matrix(b0_angle=0.0, p_angle=0.0):
    (sb, cb), (sp, cp) = _sin_cos(b0_angle), _sin_cos(p_angle)
    undo_p = np.array([[cp, sp, 0.0], [-sp, cp, 0.0], [0.0, 0.0, 1.0]])
    undo_b0 = np.array([[1.0, 0.0, 0.0], [0.0, cb, sb], [0.0, -sb, cb]])
    return undo_b0 @ undo_p


def solar_north(b0_angle=0.0, p_angle=0.0):
    (sb, cb), (sp, cp) = _sin_cos(b0_angle), _sin_cos(p_angle)
    return np.array([-sp * cb, cp * cb, sb])


def to_model(x, y, z, b0_angle=0.0, p_angle=0.0):
    """Observer-frame points -> model-aligned points; the points themselves at zero angles."""
    if b0_angle == 0.0 and p_angle == 0.0:
        return x, y, z
    m = view_matrix(b0_angle, p_angle)
    x, y, z = np.broadcast_arrays(np.asarray(x, float), np.asarray(y, float), np.asarray(z, float))
    return (m[0, 0] * x + m[0, 1] * y + m[0, 2] * z, m[1, 0] * x + m[1, 1] * y + m[1, 2] * z,
            m[2, 0] * x + m[2, 1] * y + m[2, 2] * z)


def to_observer(vx, vy, vz, b0_angle=0.0, p_angle=0.0):
    """Model-aligned vectors -> observer frame (the transpose of view_matrix)."""
    if b0_angle == 0.0 and p_angle == 0.0:
        return vx, vy, vz
    m = view_matrix(b0_angle, p_angle).T
    return (m[0, 0] * vx + m[0, 1] * vy + m[0, 2] * vz, m[1, 0] * vx + m[1, 1] * vy + m[1, 2] * vz,
            m[2, 0] * vx + m[2, 1] * vy + m[2, 2] * vz)


def resample_to_xyz_cube(var, x_grid, y_grid, z_grid, phi0_offset=0.0, fill_nan=0.0, r_min=0.9999999, b0_angle=0.0,
                         p_angle=0.0):
    """oracle_cubes.resample_to_xyz_cube with the cube nodes seen from the observer view."""
    X, Y, Z = np.meshgrid(np.asarray(x_grid, float), np.asarray(y_grid, float), np.asarray(z_grid, float),
                          indexing="ij")
    mx, my, mz = to_model(X, Y, Z, b0_angle, p_angle)
    r, colat, lon = oc.cart_to_sph(mx, -mz, my, phi0_offset=phi0_offset)
    lat = np.pi / 2 - colat
    ok = np.isfinite(r) & (r >= r_min)
    out = np.full(r.shape, np.nan)
    if np.any(ok):
        out[ok] = oc.sample_at_coords(var, lon[ok], lat[ok], r[ok])
    if fill_nan is not None:
        out = np.where(np.isfinite(out), out, fill_nan)
    return out


def model_b_vector(x, y, z, br, bt, bp):
    """(br, bt, bp) at model-aligned points -> Cartesian components in the model-aligned cube axes (x, y = rotation
    axis, z), as lmo.bvec_theta_deg rotates them."""
    _, (bx, by, bz) = _zero_view_theta(x, y, z, br, bt, bp)
    return bx, by, bz


def compose_cubes(model, x_grid, y_grid, z_grid, phi0_offset=0.0, r_min=0.999999, b0_angle=0.0, p_angle=0.0):
    """oracle_cubes.compose_cubes from the observer view, plus the Cartesian B vector bx, by, bz in observer axes."""
    temp = "te" if "te" in model else "t"
    kw = dict(phi0_offset=phi0_offset, r_min=r_min, b0_angle=b0_angle, p_angle=p_angle)
    rho = resample_to_xyz_cube(model["rho"], x_grid, y_grid, z_grid, fill_nan=0.0, **kw)
    omega_pe = np.nan_to_num(8.93e3 * np.sqrt(np.maximum(rho, 0.0)) * 2 * np.pi, nan=0.0, posinf=0.0, neginf=0.0)
    te = resample_to_xyz_cube(model[temp], x_grid, y_grid, z_grid, fill_nan=None, **kw)
    te = np.where(np.isfinite(te), te, 1e4)
    br, bt, bp = (resample_to_xyz_cube(model[k], x_grid, y_grid, z_grid, fill_nan=0.0, **kw) for k in ("br", "bt", "bp"))
    X, Y, Z = np.meshgrid(np.asarray(x_grid, float), np.asarray(y_grid, float), np.asarray(z_grid, float),
                          indexing="ij")
    mx, my, mz = to_model(X, Y, Z, b0_angle, p_angle)
    bx, by, bz = to_observer(*model_b_vector(mx, my, mz, br, bt, bp), b0_angle, p_angle)
    return dict(x_grid=x_grid, y_grid=y_grid, z_grid=z_grid, omega_pe=omega_pe, ne=np.maximum(rho, 0.0), te=te,
                b=np.sqrt(br ** 2 + bt ** 2 + bp ** 2), br=br, bt=bt, bp=bp, bx=bx, by=by, bz=bz)


def _los_points(xs, ys, zc):
    X, Y = np.meshgrid(np.asarray(xs, float), np.asarray(ys, float))
    rho2 = X * X + Y * Y
    with np.errstate(invalid="ignore"):
        z0 = np.where(np.sqrt(rho2) < 1.0, np.sqrt(1.0 - rho2), -np.sqrt(rho2 - 1.0)) - 1e-6 / R_SUN_M
    Z = z0[:, :, None] + np.asarray(zc, float)[None, None, :]
    return np.broadcast_to(X[:, :, None], Z.shape), np.broadcast_to(Y[:, :, None], Z.shape), Z


def los_samples(model, xs, ys, zc, phi0_offset=0.0, r_min=0.9999999, b0_angle=0.0, p_angle=0.0):
    """lmo.los_samples from the observer view: the LOS laid out in the observer frame (positions x, y, z stay there),
    each sample point turned to the model before it is sampled."""
    X, Y, Z = _los_points(xs, ys, zc)
    mx, my, mz = to_model(X, Y, Z, b0_angle, p_angle)
    r, colat, lon = oc.cart_to_sph(np.ravel(mx), -np.ravel(mz), np.ravel(my), phi0_offset)
    lat = np.pi / 2 - colat
    ok = r >= r_min
    temp = "te" if "te" in model else "t"
    out = {"x": X, "y": Y, "z": Z}
    for name, key in (("ne", "rho"), ("te", temp), ("br", "br"), ("bt", "bt"), ("bp", "bp")):
        v = np.full(r.shape, np.nan)
        v[ok] = oc.sample_at_coords(model[key], lon[ok], lat[ok], r[ok])
        out[name] = v.reshape(Z.shape)
    out["b"] = np.sqrt(out["br"] ** 2 + out["bt"] ** 2 + out["bp"] ** 2)
    return out


def bvec_theta_deg(x, y, z, br, bt, bp, b0_angle=0.0, p_angle=0.0):
    """Angle [deg] between B and the observer's +z at observer-frame points; 90 where B = 0."""
    mx, my, mz = to_model(x, y, z, b0_angle, p_angle)
    _, _, bz = to_observer(*model_b_vector(mx, my, mz, br, bt, bp), b0_angle, p_angle)
    b = np.sqrt(br * br + bt * bt + bp * bp)
    with np.errstate(invalid="ignore", divide="ignore"):
        cth = np.clip(bz / b, -1.0, 1.0)
    return np.where(b > 0, np.degrees(np.arccos(cth)), lmo.THETA_90)


def resample_MAS(model, N_pix, X_range, Y_range, N_z, dz0, phi0_offset=0.0, r_min=0.9999999, b0_angle=0.0, p_angle=0.0):
    """oracle_cubes.resample_MAS's arrays (in R_sun-based sampling, as the device works) from the observer view:
    Ne_LOS, Te_LOS, B_LOS (N_pix, N_pix, N_z)."""
    idx_z = np.arange(N_z)
    dz = dz0 * (1 + (5 * idx_z / N_z) ** 2.5)
    xs = np.linspace(X_range[0], X_range[1], N_pix)
    ys = np.linspace(Y_range[0], Y_range[1], N_pix)
    s = los_samples(model, xs, ys, np.cumsum(dz), phi0_offset, r_min, b0_angle, p_angle)
    ne, te, b = s["ne"], s["te"], s["b"]
    bad = np.isnan(ne)
    return dict(Ne_LOS=ne, Te_LOS=np.where(bad, np.nan, te), B_LOS=np.where(bad, np.nan, b))


# ---- models for the convention checks -----------------------------------------------------------------------------
def _mesh(n_phi, n_lat, n_r, r_max):
    phi = np.linspace(0.0, 2 * np.pi, n_phi, endpoint=False)
    lat = np.linspace(-np.pi / 2, np.pi / 2, n_lat)
    r = np.concatenate([[0.9995], np.geomspace(1.0, r_max, n_r - 1)])
    return phi, lat, r


def _var(f, phi, lat, r):
    from raytracinggrff_b200.cubes import SphericalVariable
    P, T, R = np.meshgrid(phi, lat, r, indexing="ij")
    return SphericalVariable(np.asarray(f(P, T, R), dtype=np.float32), phi, lat, r, 1.0)


def sin_lat_model(n_phi=8, n_lat=721, n_r=4, r_max=5.0):
    """'rho' = sin(latitude): resampled, it is n . p / |p| with n the solar north of the view."""
    phi, lat, r = _mesh(n_phi, n_lat, n_r, r_max)
    return {"rho": _var(lambda P, T, R: np.sin(T), phi, lat, r)}


def axial_field_model(b=10.0, n_phi=8, n_lat=721, n_r=4, r_max=5.0):
    """A uniform field B along the solar axis (br = B sin lat, bt = -B cos lat, bp = 0) in a uniform plasma: composed,
    the B-vector cube is B n and the |B| cube is B."""
    phi, lat, r = _mesh(n_phi, n_lat, n_r, r_max)
    return {"rho": _var(lambda P, T, R: 1e8 + 0 * R, phi, lat, r), "te": _var(lambda P, T, R: 1e6 + 0 * R, phi, lat, r),
            "br": _var(lambda P, T, R: b * np.sin(T), phi, lat, r), "bt": _var(lambda P, T, R: -b * np.cos(T), phi, lat, r),
            "bp": _var(lambda P, T, R: 0 * R, phi, lat, r)}


def radial_model(n_phi=24, n_lat=33, n_r=96, r_max=8.0):
    """A corona whose every variable depends on r only (the synthetic corona's density and temperature profiles, a
    monopole field): every view of it is the same."""
    phi, lat, r = _mesh(n_phi, n_lat, n_r, r_max)
    rs = lambda R: np.maximum(R, 1e-3)  # noqa: E731
    return {"rho": _var(lambda P, T, R: 4.2e4 * 10.0 ** (4.32 / rs(R)), phi, lat, r),
            "te": _var(lambda P, T, R: 1.0e6 + 0.4e6 * np.tanh(rs(R) - 1.0), phi, lat, r),
            "br": _var(lambda P, T, R: 2.0 / rs(R) ** 2, phi, lat, r),
            "bt": _var(lambda P, T, R: 0 * R, phi, lat, r), "bp": _var(lambda P, T, R: 0 * R, phi, lat, r)}


def symmetric_grid(n, step=2.0 ** -5):
    """An exactly antisymmetric grid: g[n-1-i] == -g[i] bit for bit."""
    return (np.arange(n) - (n - 1) / 2) * step
