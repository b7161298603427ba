"""ORACLE — TEST INFRASTRUCTURE ONLY: the CPU side of the map diagnostics (RaySession.render_map_diag).

* ``get_mw_diag``: oracle_get_mw with the diagnostics on one line of sight (tests/native/oracle_diag.c, which
  includes oracle/oracle_grff.c: the same functions compute the transfer, so its RL is oracle_get_mw's).
* ``chain_bvec_diag``: oracle.chain_bvec's stages (ray_trace -> sampler -> Parms with theta from B.d) with every
  compacted voxel's record position next to its Parms, then get_mw_diag per pixel; RAY_RMIN from r_record.
* ``diag_parity``: the GPU diagnostics against that chain on a pixel sub-sample.

The library is compiled with the oracle's flags (oracle/Makefile) into a temporary directory, so that a read-only
checkout works.
"""
from __future__ import annotations

import ctypes
import hashlib
import subprocess
import tempfile
from pathlib import Path

import numpy as np

from oracle import oracle

ROOT = Path(__file__).resolve().parents[1]
SRC = ROOT / "tests" / "native" / "oracle_diag.c"
CFLAGS = ["-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra", "-std=c11", "-D_GNU_SOURCE"]
PLANES = ("em_x", "em_y", "em_z", "em_r", "tau_L", "tau_R")

EM_TOL = 1e-3        # R_sun: ~1/20 of a config-4 cell
TAU_RTOL = 1e-4
RMIN_TOL = 1e-5      # R_sun

_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        key = hashlib.sha256(SRC.read_bytes() + (ROOT / "oracle" / "oracle_grff.c").read_bytes()
                             + " ".join(CFLAGS).encode()).hexdigest()[:16]
        so = Path(tempfile.gettempdir()) / f"rtgrff_oracle_diag_{key}.so"
        if not so.exists():
            tmp = so.with_suffix(f".{np.random.randint(1 << 30)}.tmp")
            subprocess.run(["gcc", *CFLAGS, "-shared", "-o", str(tmp), str(SRC), "-lm"], check=True)
            tmp.replace(so)
        _LIB = ctypes.CDLL(str(so))
        dp = ctypes.POINTER(ctypes.c_double)
        ip = ctypes.POINTER(ctypes.c_int32)
        _LIB.oracle_get_mw_diag.argtypes = [ip, dp, dp, dp, dp, dp]
        _LIB.oracle_get_mw_diag.restype = ctypes.c_int
    return _LIB


def _p(a, ct):
    return a.ctypes.data_as(ctypes.POINTER(ct))


def get_mw_diag(Lparms, Rparms, Parms, coords):
    """Lparms int32[5], Rparms f64[3], Parms f64 (15, Nz) Fortran order as oracle.get_mw; coords f64 (4, Nz)
    {x, y, z, r} per voxel.  Returns (RL (7, Nf), diag (6, Nf): em_x, em_y, em_z, em_r, tau_L, tau_R)."""
    L = np.ascontiguousarray(Lparms, dtype=np.int32)
    R = np.ascontiguousarray(Rparms, dtype=np.float64)
    P = np.asfortranarray(Parms, dtype=np.float64)
    C = np.asfortranarray(coords, dtype=np.float64)
    nz, nf = int(L[0]), int(L[1])
    if P.shape != (15, nz) or C.shape != (4, nz):
        raise ValueError("Parms must be (15, Nz) and coords (4, Nz)")
    RL = np.zeros((7, nf), order="F")
    dg = np.zeros((6, nf), order="F")
    rc = _lib().oracle_get_mw_diag(_p(L, ctypes.c_int32), _p(R, ctypes.c_double), _p(P, ctypes.c_double),
                                   _p(C, ctypes.c_double), _p(RL, ctypes.c_double), _p(dg, ctypes.c_double))
    if rc != 0:
        raise RuntimeError(f"oracle_get_mw_diag returned {rc}")
    return RL, dg


def ray_r_min(r_record):
    """Smallest |p| over each ray's records with a finite position (float32 positions, as the kernel's records);
    NaN if there is none.  r_record (n_rec, n_rays, 3) -> (n_rays,)."""
    pos = np.asarray(r_record).astype(np.float32).astype(np.float64)
    r = np.linalg.norm(pos, axis=2)
    r = np.where(np.all(np.isfinite(pos), axis=2), r, np.inf)
    m = r.min(axis=0, initial=np.inf)
    return np.where(np.isfinite(m), m, np.nan)


def chain_bvec_diag(cube, freq_hz, dt, n_steps, record_stride, xs, ys, zs, area, em_flag=4, s_max=30,
                    perturb_ratio=2, reverse=False, n_threads=0):
    """oracle.chain_bvec with the diagnostics.  reverse=True hands every pixel's voxels to the transfer far end
    first (RTGRFF_ORDER_REVERSED); False in record order (RTGRFF_ORDER_RECORD, the reference's packing).
    Returns (tb, vi, diag, r_record): tb, vi (n_rays,) as chain_bvec, diag a dict of (n_rays,) arrays with the
    keys of RaySession.render_map_diag."""
    kv = np.tile([[0.0, 0.0, -1.0]], (len(xs), 1))
    ray_start = np.column_stack([xs, ys, zs])
    g3 = (cube["x_grid"], cube["y_grid"], cube["z_grid"])
    r_rec, cs = oracle.ray_trace(cube["omega_pe"], *g3, freq_hz, xs, ys, zs, kv, dt, n_steps, record_stride, True,
                                 perturb_ratio=perturb_ratio, n_threads=n_threads, cache_gradient=True)
    s_rec = np.array(cs)
    smp = oracle.sample_model_with_rays_cpu(*g3, cube["ne"], cube["te"], cube["b"], r_rec, s_rec, ray_start,
                                            oracle.R_SUN_CM)
    bv = oracle.sample_model_with_rays_cpu(*g3, cube["bx"], cube["by"], cube["bz"], r_rec, s_rec, ray_start,
                                           oracle.R_SUN_CM, fill_ne=0.0, fill_te=0.0, fill_b=0.0)
    n_rec, n_rays = smp["ne"].shape
    conv = (oracle.SFU2CGS * oracle.C_CGS ** 2 / (2.0 * oracle.KB_CGS * freq_hz ** 2) / area) * oracle.AU_CM ** 2
    # Parms packing as oracle.emission_bvec_from_samples
    valid = smp["valid_mask"]
    pos = r_rec.astype(np.float32).astype(np.float64)
    start = ray_start.astype(np.float32).astype(np.float64)
    idx = np.where(valid, np.arange(n_rec)[:, None], -1)
    last = np.maximum.accumulate(idx, axis=0)
    prev = np.vstack([np.full((1, n_rays), -1, dtype=last.dtype), last[:-1]])
    prev_pos = np.take_along_axis(pos, np.broadcast_to(np.maximum(prev, 0)[:, :, None], pos.shape), axis=0)
    prev_pos = np.where(prev[:, :, None] >= 0, prev_pos, start[None])
    d = pos - prev_pos
    B = np.stack([bv["ne"], bv["te"], bv["b"]], axis=2).astype(np.float64)
    b2 = (B * B).sum(2)
    dn2 = (d * d).sum(2)
    with np.errstate(divide="ignore", invalid="ignore"):
        cth = np.clip(-(B * d).sum(2) / np.sqrt(b2 * dn2), -1.0, 1.0)
    cth = np.where((b2 > 0) & (dn2 > 0), cth, 6.123233995736766e-17)
    theta = np.degrees(np.arccos(cth))
    bmag = np.sqrt(b2)
    keep_src = valid & np.isfinite(smp["ne"]) & np.isfinite(smp["te"]) & np.isfinite(bmag)
    # the record position of each voxel: float32 x, y, z and |p| (the kernel takes |p| of the float32 position)
    pos32 = r_rec.astype(np.float32)
    coord = np.concatenate([pos, np.sqrt((pos32.astype(np.float64) ** 2).sum(2))[:, :, None]], axis=2)
    tb, vi = np.zeros(n_rays), np.zeros(n_rays)
    out = {k: np.full(n_rays, np.nan) for k in PLANES}
    for p in range(n_rays):
        sel = np.nonzero(keep_src[:, p])[0]
        if reverse:
            sel = sel[::-1]
        nz = len(sel)
        P = np.zeros((15, nz), order="F")
        for m, a in ((0, smp["ds"]), (1, smp["te"]), (2, smp["ne"]), (3, bmag), (4, theta)):
            P[m] = np.asarray(a[sel, p], dtype=np.float64)
        P[6], P[7] = em_flag, s_max
        C = np.asfortranarray(coord[sel, p].T)
        RL, dg = get_mw_diag(np.array([nz, 1, 0, 0, 0], np.int32), np.array([area, freq_hz, 0.0]), P, C)
        inten = RL[5, 0] + RL[6, 0]
        tb[p] = inten * conv if nz else 0.0
        vi[p] = (RL[5, 0] - RL[6, 0]) / (inten + 1e-30) if nz else 0.0
        for q, k in enumerate(PLANES):
            out[k][p] = dg[q, 0] if nz else (np.nan if q < 4 else 0.0)
    tb = np.nan_to_num(tb, nan=0.0, posinf=0.0, neginf=0.0)
    out["ray_r_min"] = ray_r_min(r_rec)
    return tb, vi, out, r_rec


def _tau_close(a, b, rtol):
    both_inf = np.isinf(a) & np.isinf(b)
    with np.errstate(invalid="ignore"):
        ok = np.abs(a - b) <= rtol * np.abs(b)
    return both_inf | ok


def diag_parity(cube, freq_params, xs, ys, zs, area, diag_gpu, em_flag=4, s_max=30, reverse=False, n_threads=None,
                cell=None):
    """The GPU diagnostics (dict of (n_freq, n_rays) at the sub-sampled pixels xs, ys, zs) against chain_bvec_diag.
    Pixels whose oracle ray comes within one cell of the r = 1 density discontinuity are chaotic (oracle/parity.py)
    and left out.  Returns a dict of the largest deviations on the others, the counts over tolerance, and how many
    compared pixel-frequencies are optically thick (tau > 1 on both slots) and thin (tau < 0.1 on both)."""
    oracle.set_num_threads(n_threads)
    lo = np.array([cube["x_grid"][0], cube["y_grid"][0], cube["z_grid"][0]])
    hi = np.array([cube["x_grid"][-1], cube["y_grid"][-1], cube["z_grid"][-1]])
    if cell is None:
        cell = float(cube["x_grid"][1] - cube["x_grid"][0])
    res = dict(n_compared=0, n_diving=0, max_d_em=0.0, max_rel_d_tau=0.0, max_d_rmin=0.0, n_em_over=0, n_tau_over=0,
               n_rmin_over=0, n_nan_mismatch=0, n_thick=0, n_thin=0)
    for f, p in enumerate(freq_params):
        _, _, ref, r_rec = chain_bvec_diag(cube, p["freq_hz"], p["dt"], p["n_steps"], p["record_stride"], xs, ys, zs,
                                           area, em_flag, s_max, reverse=reverse)
        inside = np.all((r_rec >= lo) & (r_rec <= hi), axis=2)
        rad = np.where(inside, np.linalg.norm(r_rec, axis=2), np.inf)
        ok = ~(rad.min(axis=0) < 1.0 + cell)
        res["n_diving"] += int((~ok).sum())
        res["n_compared"] += int(ok.sum())
        for k in ("em_x", "em_y", "em_z", "em_r"):
            g, r = np.asarray(diag_gpu[k][f])[ok], ref[k][ok]
            res["n_nan_mismatch"] += int((np.isnan(g) != np.isnan(r)).sum())
            both = ~np.isnan(g) & ~np.isnan(r)
            dd = np.abs(g[both] - r[both])
            res["max_d_em"] = max(res["max_d_em"], float(dd.max(initial=0.0)))
            res["n_em_over"] += int((dd > EM_TOL).sum())
        for k in ("tau_L", "tau_R"):
            g, r = np.asarray(diag_gpu[k][f])[ok], ref[k][ok]
            close = _tau_close(g, r, TAU_RTOL)
            res["n_tau_over"] += int((~close).sum())
            fin = np.isfinite(g) & np.isfinite(r) & (r > 0)
            res["max_rel_d_tau"] = max(res["max_rel_d_tau"], float((np.abs(g[fin] - r[fin]) / r[fin]).max(initial=0.0)))
        g, r = np.asarray(diag_gpu["ray_r_min"][f])[ok], ref["ray_r_min"][ok]
        res["n_nan_mismatch"] += int((np.isnan(g) != np.isnan(r)).sum())
        both = ~np.isnan(g) & ~np.isnan(r)
        dd = np.abs(g[both] - r[both])
        res["max_d_rmin"] = max(res["max_d_rmin"], float(dd.max(initial=0.0)))
        res["n_rmin_over"] += int((dd > RMIN_TOL).sum())
        tl, tr = ref["tau_L"][ok], ref["tau_R"][ok]
        res["n_thick"] += int(((tl > 1) & (tr > 1)).sum())
        res["n_thin"] += int(((tl < 0.1) & (tr < 0.1)).sum())
    return res
