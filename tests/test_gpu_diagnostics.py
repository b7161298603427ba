"""GPU: the map diagnostics of the fused renderer (RaySession.render_map_diag / rtgrff_render_map_diag): emission
centroid and height, optical depths and the ray's turning point per (pixel, frequency).

* T_b and V/I of the diagnostic kernels are the plain kernels' bit for bit, in all 16 variants;
* an analytic uniform cube (straight rays, B = 0) pins the definitions and the voxel-order semantics;
* the bench variant at config 4 and the reversed order on a smaller map against the CPU oracle
  (tests/diag_oracle.py);
* frequency bookkeeping, device output + gather_image, and the --diagnostics files of the workflow and the sweep.
"""
import ctypes
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

import bench  # noqa: E402  (workload definitions: the same tables the benchmark runs)
import diag_oracle  # noqa: E402
from raytracinggrff_b200 import _lib, synthetic  # noqa: E402

pytestmark = pytest.mark.gpu

R_SUN_CM = 6.957e10
PLANES = ("em_x", "em_y", "em_z", "em_r", "tau_L", "tau_R", "ray_r_min")


def _load_cube(session, c):
    g3 = (c["x_grid"], c["y_grid"], c["z_grid"])
    session.set_omega_cube(c["omega_pe"], *g3)
    session.set_field_cubes(*g3, c["ne"], c["te"], c["b"], c["bx"], c["by"], c["bz"])


@pytest.fixture(scope="module")
def c3_cube():
    return synthetic.corona_cube(128, 3.0, active_region=True)


def _c3_rays(n_pix=64):
    xs, ys, zs, kv = synthetic.ray_launch_geometry(n_pix, 1.44, 3.0)
    return xs, ys, zs, (2 * 1.44 / n_pix * R_SUN_CM) ** 2


@pytest.mark.parametrize("cs", [False, True])
@pytest.mark.parametrize("order", [_lib.ORDER_RECORD, _lib.ORDER_REVERSED])
def test_tb_vi_equal_plain_kernels_in_every_variant(session, c3_cube, cs, order):
    """The diagnostic kernels take every operator from the plain kernels' code.  Expected: the same bits; the bound
    is 1e-12 relative on T_b (absolute on V/I, which is O(1) and crosses 0)."""
    _load_cube(session, c3_cube)
    xs, ys, zs, area = _c3_rays()
    fps = [(75e6, 6e-3, 5000, 10), _scaled(1.5e9)]
    report = []
    for bvec in (False, True):
        for em_flag in (4, 5):      # 4: gyroresonance on, 5: free-free only
            kw = dict(trace_crosssections=cs, pixel_area_cm2=area, em_flag=em_flag, use_bvec=bvec, voxel_order=order,
                      image_shape=(64, 64))
            tb, vi, st = session.render_map(xs, ys, zs, fps, **kw)
            tb2, vi2, st2, dg = session.render_map_diag(xs, ys, zs, fps, **kw)
            with np.errstate(divide="ignore", invalid="ignore"):
                rel = np.where(tb != tb2, np.abs(tb2 - tb) / np.abs(tb), 0.0)
            dvi = np.abs(np.nan_to_num(vi2, nan=0.0) - np.nan_to_num(vi, nan=0.0))
            n_diff = int((tb != tb2).sum())
            report.append((bvec, em_flag, n_diff, float(rel.max()), float(dvi.max())))
            assert rel.max() <= 1e-12 and dvi.max() <= 1e-12, report[-1]
            assert np.array_equal(np.isnan(vi), np.isnan(vi2))
            assert st == st2
            assert set(dg) == set(PLANES) and all(dg[k].shape == tb.shape for k in PLANES)
            lit = tb > 0
            assert lit.mean() > 0.3
            assert np.isfinite(dg["em_z"][lit]).all() and (dg["tau_L"][lit] >= 0).all()
    print(f"cs={cs} order={order}: (bvec, em_flag, T_b values not bit-identical, max rel dT_b, max |dV/I|)", report)


def _scaled(f):
    p = synthetic.frequency_scaled_params(f)
    return (f, p["dt"], p["n_steps"], p["record_stride"])


def _uniform_cube(ne, te, extent=1.5, n=33):
    g = np.linspace(-extent, extent, n)
    shape = (n, n, n)
    wpe = 5.64e4 * np.sqrt(ne)
    return dict(x_grid=g, y_grid=g, z_grid=g, omega_pe=np.full(shape, wpe), ne=np.full(shape, ne),
                te=np.full(shape, te), b=np.zeros(shape), bx=np.zeros(shape), by=np.zeros(shape), bz=np.zeros(shape))


def _kappa(ne, te, nu):
    """Free-free opacity at B = 0 (oracle/oracle_grff.c), T, n_e as float32 as the cubes hold them."""
    import grff_checks as gc
    ne, te = float(np.float32(ne)), float(np.float32(te))
    v = gc.E ** 2 * ne / (np.pi * gc.ME) / nu ** 2
    return gc.KFF * ne * ne * gc.ZETA * gc.lnL(te, nu) / (np.sqrt(1 - v) * nu * nu * te * np.sqrt(te))


@pytest.mark.parametrize("order", [_lib.ORDER_RECORD, _lib.ORDER_REVERSED])
def test_uniform_cube_analytic(session, order):
    """Constant omega_pe: straight rays along -z from z0 = 1.2 through the cube's far face at z = -1.5.  B = 0, so
    both slots are the same slab."""
    nu, dt, n_steps, stride, z0 = 300e6, 0.01, 1000, 2, 1.2
    xs = np.array([0.0, 0.3, -0.45, 0.2])
    ys = np.array([0.0, -0.25, 0.1, 0.6])
    zs = np.full(4, z0)
    kv = np.tile([[0.0, 0.0, -1.0]], (4, 1))
    # -- optically thin: n_e = 1e6 cm^-3, T = 1e6 K
    c = _uniform_cube(1e6, 1e6)
    _load_cube(session, c)
    r, _, _ = session.trace(nu, xs, ys, zs, kv, dt, n_steps, stride, False, 2.0)
    inside = np.all(np.abs(r) <= 1.5, axis=2)
    z_last = np.where(inside, r[:, :, 2], np.inf).min(axis=0).astype(np.float32).astype(np.float64)
    h = float(np.abs(np.diff(r[:2, 0, 2])).max())          # record spacing
    assert 0.002 < h < 0.05
    fp = [(nu, dt, n_steps, stride)]
    tb, _, _, dg = session.render_map_diag(xs, ys, zs, fp, kvec_in_norm=kv, trace_crosssections=False, em_flag=5,
                                           voxel_order=order)
    assert (tb > 0).all()
    np.testing.assert_allclose(dg["em_x"][0], xs, atol=1e-6)
    np.testing.assert_allclose(dg["em_y"][0], ys, atol=1e-6)
    # thin: every voxel weighs its ds, and sits at its record position (the far end of its ds)
    pos = r.astype(np.float32).astype(np.float64)
    prev = np.concatenate([np.column_stack([xs, ys, zs])[None].astype(np.float32).astype(np.float64), pos[:-1]])
    ds = np.where(inside, np.linalg.norm(pos - prev, axis=2), 0.0)
    np.testing.assert_allclose(dg["em_z"][0], (ds * pos[:, :, 2]).sum(0) / ds.sum(0), atol=2e-4)
    # ... which puts the centroid half a record spacing beyond the middle of the emitting path
    assert np.all(np.abs(dg["em_z"][0] - 0.5 * (z0 + z_last)) <= h), (dg["em_z"][0], z0, z_last, h)
    L = (np.float32(z0) - z_last) * R_SUN_CM
    tau = _kappa(1e6, 1e6, nu) * L
    assert tau.max() < 1e-2
    np.testing.assert_allclose(dg["tau_L"][0], tau, rtol=1e-5)
    np.testing.assert_allclose(dg["tau_R"][0], tau, rtol=1e-5)
    rho = np.hypot(xs, ys)
    assert np.all(np.abs(dg["ray_r_min"][0] - rho) <= h), (dg["ray_r_min"][0], rho)
    # EM_R: the mean of |p| along the path, not |centroid|
    em_r_ref = np.array([np.mean(np.hypot(rho[p], np.linspace(z0, z_last[p], 2001))) for p in range(4)])
    np.testing.assert_allclose(dg["em_r"][0], em_r_ref, atol=h)
    # -- optically thick: n_e = 3e8 cm^-3 (1/kappa ~ 0.06 R_sun, tau ~ 45)
    c = _uniform_cube(3e8, 1e6)
    _load_cube(session, c)
    kap_rsun = _kappa(3e8, 1e6, nu) * R_SUN_CM
    assert 5 < kap_rsun < 50
    _, _, _, dg = session.render_map_diag(xs, ys, zs, fp, kvec_in_norm=kv, trace_crosssections=False, em_flag=5,
                                          voxel_order=order)
    assert (dg["tau_L"][0] > 20).all()
    np.testing.assert_allclose(dg["em_x"][0], xs, atol=1e-6)
    if order == _lib.ORDER_REVERSED:
        # physical order: the emission comes from within ~1/kappa of the observer-side face
        d = z0 - dg["em_z"][0]
    else:
        # record order: the observer-side record is handed over first, as the far end: the far face shines
        d = dg["em_z"][0] - z_last
    assert np.all((d > 0) & (d < 3.0 / kap_rsun + h)), (d, 1 / kap_rsun, h)


def test_config4_bench_variant_matches_oracle(oracle, session):
    w = bench.workload("c4", 1)
    c = synthetic.corona_cube(w["grid_n"], w["extent"], active_region=True)
    _load_cube(session, c)
    fps = w["freq_params"]
    area = bench.pixel_area(w)
    xs, ys, zs = bench.rays_of(w)
    tb, vi, _, dg = session.render_map_diag(xs, ys, zs, fps, trace_crosssections=True, perturb_ratio=2.0,
                                            pixel_area_cm2=area, r_sun_cm=R_SUN_CM, em_flag=4, s_max=30, use_bvec=True,
                                            image_shape=(w["n_pix_y"], w["n_pix_x"]))
    from oracle import parity
    sel = parity.subsample(512, 512, 16)
    par = diag_oracle.diag_parity(c, fps, xs[sel], ys[sel], zs[sel], area, {k: v[:, sel] for k, v in dg.items()},
                                  em_flag=4)
    print("diag parity c4:", par)
    # rays that come close to r = 1 (at GHz frequencies much of the disc) are left out, as in oracle/parity.py
    assert par["n_compared"] > 0.3 * 1024 * 8
    assert par["n_em_over"] == 0 and par["max_d_em"] <= diag_oracle.EM_TOL, par
    assert par["n_tau_over"] == 0, par
    assert par["n_rmin_over"] == 0 and par["max_d_rmin"] <= diag_oracle.RMIN_TOL, par
    assert par["n_nan_mismatch"] == 0, par
    assert par["n_thick"] > 0 and par["n_thin"] > 0, par


def test_reversed_order_em5_matches_oracle(oracle, session, c3_cube):
    _load_cube(session, c3_cube)
    xs, ys, zs, area = _c3_rays()
    fps = [dict(freq_hz=75e6, dt=6e-3, n_steps=5000, record_stride=10)]
    _, _, _, dg = session.render_map_diag(xs, ys, zs, [tuple(fps[0].values())], trace_crosssections=True,
                                          pixel_area_cm2=area, em_flag=5, use_bvec=True,
                                          voxel_order=_lib.ORDER_REVERSED, image_shape=(64, 64))
    from oracle import parity
    sel = parity.subsample(64, 64, 4)
    par = diag_oracle.diag_parity(c3_cube, fps, xs[sel], ys[sel], zs[sel], area, {k: v[:, sel] for k, v in dg.items()},
                                  em_flag=5, reverse=True)
    print("diag parity reversed:", par)
    assert par["n_compared"] > 128
    assert par["n_em_over"] == 0 and par["n_tau_over"] == 0 and par["n_rmin_over"] == 0, par
    assert par["n_nan_mismatch"] == 0, par


def test_diag_planes_land_on_the_caller_frequency(session, c3_cube):
    """The host launches the frequencies most expensive first; every plane must still land on the caller's index."""
    _load_cube(session, c3_cube)
    xs, ys, zs, area = _c3_rays(32)
    fps = [_scaled(75e6), _scaled(1.2e9), _scaled(300e6)]      # launched as 1.2 GHz, 300 MHz, 75 MHz
    kw = dict(pixel_area_cm2=area, em_flag=4, use_bvec=True)
    tb, vi, _, dg = session.render_map_diag(xs, ys, zs, fps, **kw)
    for f, p in enumerate(fps):
        tb1, vi1, _, d1 = session.render_map_diag(xs, ys, zs, [p], **kw)
        assert np.array_equal(tb[f], tb1[0])
        for k in PLANES:
            assert np.array_equal(dg[k][f], d1[k][0], equal_nan=True), (f, k)
    assert not np.array_equal(dg["em_r"][0], dg["em_r"][1], equal_nan=True)


def test_device_output_through_gather_image(session, c3_cube):
    """tb | vi | diag written by the kernel into one device slab, then gathered as 9 n_freq planes (world size 1)."""
    _load_cube(session, c3_cube)
    n = 32
    xs, ys, zs, area = _c3_rays(n)
    fps = [(75e6, 6e-3, 3000, 10), (150e6, 4e-3, 3000, 10)]
    nf = len(fps)
    kw = dict(pixel_area_cm2=area, em_flag=4, use_bvec=True, image_shape=(n, n))
    tb, vi, _, dg = session.render_map_diag(xs, ys, zs, fps, **kw)
    n_planes = 2 * nf + 7 * nf
    nb = nf * n * n * 8
    base = ctypes.c_void_p()
    lib = _lib.load()
    _lib.check(lib.rtgrff_device_alloc(session.ctx.handle, ctypes.byref(base), n_planes * n * n * 8))
    try:
        session.render_map_diag(xs, ys, zs, fps, out_device_ptrs=(base.value, base.value + nb, base.value + 2 * nb),
                                **kw)
        session.comm_init(1, 0)
        img = np.zeros((n_planes, n, n))
        session.gather_image(base.value, n_planes, n, n, root=0, out=img)
    finally:
        lib.rtgrff_device_free(session.ctx.handle, base)
    want = np.concatenate([tb, vi, np.stack([dg[k] for k in PLANES]).reshape(7 * nf, n * n)]).reshape(n_planes, n, n)
    assert np.array_equal(img, want, equal_nan=True)


def test_diag_needs_an_output(session, c3_cube):
    _load_cube(session, c3_cube)
    lib = _lib.load()
    fp = (_lib.FreqParams * 1)(_lib.FreqParams(75e6, 6e-3, 100, 10))
    x = np.zeros(1)
    p = x.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    out = np.zeros(2)
    rc = lib.rtgrff_render_map_diag(session.ctx.handle, 1, p, p, p, None, None, 1, fp, 1, 2.0, 1.0, R_SUN_CM, 4, 30, 0,
                                    0, 0, 0, out[:1].ctypes.data_as(ctypes.c_void_p),
                                    out[1:].ctypes.data_as(ctypes.c_void_p), 0, None, None)
    assert rc == _lib.RTGRFF_EINVAL


def test_workflow_and_sweep_diagnostics_files(session, tmp_path):
    from raytracinggrff_b200 import sweep
    from raytracinggrff_b200.workflow import run_ray_tracing_emission
    c = synthetic.corona_cube(48, 3.0, active_region=True)
    kw = dict(N_pix=10, X_fov=1.3, freq_hz=90e6, z_observer=3.0, dt=6e-3, n_steps=1500, record_stride=8,
              grff_backend="fused", verbose=False)
    plain = run_ray_tracing_emission(c, out_path=tmp_path / "plain.npz", **kw)
    withd = run_ray_tracing_emission(c, out_path=tmp_path / "diag.npz", diagnostics=True, **kw)
    a, b = np.load(tmp_path / "plain.npz"), np.load(tmp_path / "diag.npz")
    new = {"emission_centroid_xyz", "emission_r_mean", "tau_L", "tau_R", "ray_r_min"}
    assert set(b.files) == set(a.files) | new
    for k in a.files:
        assert np.array_equal(a[k], b[k]), k
        assert np.array_equal(plain[k], withd[k]), k
    assert b["emission_centroid_xyz"].shape == (10, 10, 1, 3)
    for k in new - {"emission_centroid_xyz"}:
        assert b[k].shape == (10, 10, 1), k
    lit = b["emission_cube"][:, :, 0] > 0
    assert np.isfinite(b["emission_r_mean"][:, :, 0][lit]).all() and (b["emission_r_mean"][:, :, 0][lit] >= 1.0).all()
    # the sweep: the emission height against frequency
    model = synthetic.spherical_corona(64, 48, 64, r_max=8.0)
    skw = dict(N_pix=12, fmin_mhz=40.0, fmax_mhz=400.0, n_freq=3, phi0_offset=-140.0, session=session, max_grid_n=64)
    rows = sweep.tb_spectra(model, tmp_path / "plain", **skw)
    rows_d = sweep.tb_spectra(model, tmp_path / "diag", diagnostics=True, **skw)
    heights = []        # median emission height of the central pixels
    for (_, _, p0), (_, _, p1) in zip(rows, rows_d):
        a, b = np.load(p0), np.load(p1)
        assert set(b.files) == set(a.files) | new
        for k in a.files:
            assert np.array_equal(a[k], b[k]), k
        assert b["emission_centroid_xyz"].shape == (12, 12, 1, 3)
        heights.append(np.median(b["emission_r_mean"][5:7, 5:7, 0]))
    # lower frequencies are emitted higher in the corona
    assert heights[0] > heights[-1], heights
