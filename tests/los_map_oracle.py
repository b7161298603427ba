"""ORACLE — TEST INFRASTRUCTURE ONLY: a CPU restatement of the fused straight-LOS map (rtgrff_render_los_map).

* ``los_samples``: oracle_cubes.resample_MAS's LOS geometry and sampler (psipy restated), in R_sun units as the
  kernel works, keeping br, bt, bp and every sample's position;
* ``bvec_theta_deg``: theta between the B vector rotated to cube axes and the propagation direction +z;
* ``los_map``: the per-pixel SyntheticFF packing (NaN filter, voxel order kept, Sun side first) with a theta column,
  oracle.get_mw per pixel (or tests/diag_oracle.get_mw_diag with the voxels' float32 positions), SyntheticFF's T_b.
"""
from __future__ import annotations

import numpy as np

from oracle import oracle
from oracle import oracle_cubes as oc

R_SUN_M, R_SUN_CM = 6.957e8, 6.957e10
THETA_90 = 90.0


def bvec_theta_deg(x, y, z, br, bt, bp):
    """Angle [deg] between B and +z at cube points (x, y, z): (br, bt, bp) rotated to cube axes as the cube builder's
    compose step does (model frame (x, -z, y), theta the colatitude from +y), cos theta = B_z / |B|; 90 where B = 0."""
    cx, cy, cz = np.asarray(x, float), -np.asarray(z, float), np.asarray(y, float)
    cx, cy, cz, br, bt, bp = np.broadcast_arrays(cx, cy, cz, br, bt, bp)
    rr, rho_c = np.sqrt(cx * cx + cy * cy + cz * cz), np.sqrt(cx * cx + cy * cy)
    with np.errstate(invalid="ignore", divide="ignore"):
        st, ct, cp, sp = rho_c / rr, cz / rr, cx / rho_c, cy / rho_c
    gen = (rr > 0) & (rho_c > 0)
    mx = np.where(gen, br * st * cp + bt * ct * cp - bp * sp, 0.0)
    my = np.where(gen, br * st * sp + bt * ct * sp + bp * cp, 0.0)
    mz = np.where(gen, br * ct - bt * st, np.where(rr > 0, np.where(cz > 0, br, -br), 0.0))
    bz = -my
    b = np.sqrt(br * br + bt * bt + bp * bp)
    with np.errstate(invalid="ignore", divide="ignore"):
        cth = np.clip(bz / b, -1.0, 1.0)
    return np.where(b > 0, np.degrees(np.arccos(cth)), THETA_90), (mx, mz, bz)


def los_samples(model, xs, ys, zc, phi0_offset=0.0, r_min=0.9999999):
    """Every pixel's LOS (pixel (i, j) at (xs[j], ys[i]) [R_sun]) sampled on the CPU: dict of (ny, nx, nz) arrays
    ne, te, b, br, bt, bp (NaN where r < r_min or outside the mesh) and the positions x, y, z [R_sun]."""
    X, Y = np.meshgrid(np.asarray(xs, float), np.asarray(ys, float))
    rho2 = X * X + Y * Y
    with np.errstate(invalid="ignore"):
        z0 = np.where(np.sqrt(rho2) < 1.0, np.sqrt(1.0 - rho2), -np.sqrt(rho2 - 1.0)) - 1e-6 / R_SUN_M
    Z = z0[:, :, None] + np.asarray(zc, float)[None, None, :]
    Xb, Yb = np.broadcast_to(X[:, :, None], Z.shape), np.broadcast_to(Y[:, :, None], Z.shape)
    r, colat, lon = oc.cart_to_sph(Xb.ravel(), -Z.ravel(), Yb.ravel(), phi0_offset)
    lat = np.pi / 2 - colat
    ok = r >= r_min
    temp = "te" if "te" in model else "t"
    out = {"x": Xb, "y": Yb, "z": Z}
    for name, key in (("ne", "rho"), ("te", temp), ("br", "br"), ("bt", "bt"), ("bp", "bp")):
        v = np.full(r.shape, np.nan)
        v[ok] = oc.sample_at_coords(model[key], lon[ok], lat[ok], r[ok])
        out[name] = v.reshape(Z.shape)
    out["b"] = np.sqrt(out["br"] ** 2 + out["bt"] ** 2 + out["bp"] ** 2)
    return out


def _to_tb(RL, freqs, area):
    inten = RL[5] + RL[6]
    with np.errstate(invalid="ignore", divide="ignore"):
        pol = (RL[5] - RL[6]) / (RL[5] + RL[6])
    nu = np.where(RL[0] > 0, RL[0] * 1e9, freqs)
    conv = (oracle.SFU2CGS * oracle.C_CGS ** 2 / (2.0 * oracle.KB_CGS * nu * nu) / area) * (1.49599e13 * 1.49599e13)
    return inten * conv, pol


def los_map(smp, dz_cm, area, freq0, n_freq, log_step, em_flag=5, s_max=30, use_bvec=False, diagnostics=False):
    """T_b and V/I (ny, nx, n_freq) of the sampled LOS; with diagnostics also a dict of (ny, nx, n_freq) planes
    em_x, em_y, em_z, em_r, tau_L, tau_R from diag_oracle.get_mw_diag (ray_r_min: the LOS's smallest float32 |p|)."""
    import diag_oracle
    ny, nx, nz = smp["ne"].shape
    freqs = freq0 * 10.0 ** (log_step * np.arange(n_freq))
    theta = np.full(smp["ne"].shape, THETA_90)
    if use_bvec:
        theta = bvec_theta_deg(smp["x"], smp["y"], smp["z"], smp["br"], smp["bt"], smp["bp"])[0]
    pos32 = np.stack([smp["x"], smp["y"], smp["z"]], axis=-1).astype(np.float32).astype(np.float64)
    rad = np.sqrt((pos32 ** 2).sum(-1))
    tb, vi = np.zeros((ny, nx, n_freq)), np.zeros((ny, nx, n_freq))
    dg = {k: np.full((ny, nx, n_freq), np.nan) for k in diag_oracle.PLANES}
    R = np.array([area, freq0, log_step])
    for i in range(ny):
        for j in range(nx):
            keep = ~(np.isnan(smp["ne"][i, j]) | np.isnan(smp["te"][i, j]) | np.isnan(smp["b"][i, j]))
            n = int(keep.sum())
            if n == 0:
                for k in ("tau_L", "tau_R"):
                    dg[k][i, j] = 0.0
                continue
            P = np.zeros((15, n), order="F")
            for m, a in ((0, dz_cm[None, None, :]), (1, smp["te"]), (2, smp["ne"]), (3, smp["b"]), (4, theta)):
                P[m] = np.broadcast_to(a, smp["ne"].shape)[i, j][keep]
            P[6], P[7] = em_flag, s_max
            L = np.array([n, n_freq, 0, 0, 0], dtype=np.int32)
            if diagnostics:
                C = np.vstack([pos32[i, j][keep].T, rad[i, j][keep][None]])
                RL, d = diag_oracle.get_mw_diag(L, R, P, C)
                for q, k in enumerate(diag_oracle.PLANES):
                    dg[k][i, j] = d[q]
            else:
                RL = np.zeros((7, n_freq), order="F")
                assert oracle.get_mw(L, R, P, None, None, None, RL) == 0
            tb[i, j], vi[i, j] = _to_tb(RL, freqs, area)
    if not diagnostics:
        return tb, vi
    dg["ray_r_min"] = np.broadcast_to(rad.min(axis=2)[:, :, None], tb.shape).copy()
    return tb, vi, dg
