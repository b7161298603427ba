"""GPU: the observer view (solar B0 and P angles) in the cube builder, the LOS sampler and both map renderers.

* zero angles: the _view entry points and keywords give exactly what the fixed-view entry points give;
* parity with the CPU restatement (tests/view_oracle.py) and with the conventions of include/rtgrff.h;
* P = 90 deg is a quarter turn of the image; a model that depends on r only looks the same from every view;
* the renderers at a non-zero view against the staged path, the CPU oracle and oracle-composed cubes.
"""
from ctypes import c_double, c_float

import numpy as np
import pytest

import los_map_oracle as lmo
import view_oracle as vo
from raytracinggrff_b200 import _lib, cubes, los, synthetic
from raytracinggrff_b200._lib import f32, f64, ptr

pytestmark = pytest.mark.gpu

R_SUN_CM = 6.957e10
R_SUN_M = 6.957e8
VIEWS = ((7.25, 0.0), (0.0, 24.0), (-30.0, 115.0))
FOV = (-1.44, 1.44)


@pytest.fixture(scope="module")
def model():
    return synthetic.spherical_corona(64, 48, 64, r_max=8.0, active_region=True)


def _old_set_model(session, model, g, phi0, want_bvec):
    """set_model_from_spherical through the fixed-view entry points rtgrff_resample_spherical + rtgrff_compose_cubes."""
    lib = _lib.load()
    geom = _lib.grid_geom(g, g, g)
    gg = f64(g)
    for slot, (name, fill) in enumerate((("rho", 0.0), ("te", None), ("br", 0.0), ("bt", 0.0), ("bp", 0.0))):
        v = model[name]
        data, phi, lat, r = f32(v.data), f64(v.phi), f64(v.lat), f64(v.r)
        _lib.check(lib.rtgrff_resample_spherical(session.ctx.handle, slot, ptr(data, c_float), ptr(phi, c_double),
                                                 ptr(lat, c_double), ptr(r, c_double), *data.shape, ptr(gg, c_double),
                                                 ptr(gg, c_double), ptr(gg, c_double), len(g), len(g), len(g),
                                                 ptr(geom, c_double), float(phi0), 0.999999, float(v.scale),
                                                 0.0 if fill is None else fill, int(fill is not None), None))
    _lib.check(lib.rtgrff_compose_cubes(session.ctx.handle, int(want_bvec)))
    session.cube_shape = (len(g),) * 3


def _old_los_sample(session, var, xs, ys, zc, phi0):
    data, phi, lat, r = f32(var.data), f64(var.phi), f64(var.lat), f64(var.r)
    x, y, z = f64(xs), f64(ys), f64(zc)
    out = np.empty((len(y), len(x), len(z)))
    _lib.check(_lib.load().rtgrff_sample_spherical_los(session.ctx.handle, ptr(data, c_float), ptr(phi, c_double),
                                                       ptr(lat, c_double), ptr(r, c_double), *data.shape,
                                                       ptr(x, c_double), ptr(y, c_double), ptr(z, c_double), len(x),
                                                       len(y), len(z), float(phi0), 0.9999999, float(var.scale),
                                                       1e-6 / R_SUN_M, ptr(out, c_double)))
    return out


def _old_los_map(session, xs, ys, zc, dz_cm, freqs, phi0, em_flag, use_bvec, diagnostics):
    import ctypes
    x, y, z, d, fr = f64(xs), f64(ys), f64(zc), f64(dz_cm), f64(freqs)
    tb = np.empty((len(fr), len(y), len(x)))
    vi = np.empty_like(tb)
    dg = np.empty((len(_lib.DIAG_PLANES),) + tb.shape) if diagnostics else None
    stats = (ctypes.c_int64 * 3)()
    _lib.check(_lib.load().rtgrff_render_los_map(session.ctx.handle, len(x), len(y), ptr(x, c_double), ptr(y, c_double),
                                                 len(z), ptr(z, c_double), ptr(d, c_double), float(phi0), 0.9999999,
                                                 1e-6 / R_SUN_M, len(fr), ptr(fr, c_double), 1e20, em_flag, 30,
                                                 int(use_bvec), tb.ctypes.data_as(ctypes.c_void_p),
                                                 vi.ctypes.data_as(ctypes.c_void_p),
                                                 None if dg is None else dg.ctypes.data_as(ctypes.c_void_p), 0, stats))
    return tb, vi, dg


def _same(a, b):
    assert np.array_equal(a, b, equal_nan=True)


# ---- 1. zero angles change nothing ---------------------------------------------------------------------------------
def test_zero_view_cubes_are_the_fixed_view_cubes(session, model):
    g = np.linspace(-3.0, 3.0, 40)
    for want_bvec in (False, True):
        _old_set_model(session, model, g, 24.0, want_bvec)
        old = session.export_cubes(bvec=want_bvec)
        session.set_model_from_spherical(model, g, g, g, phi0_offset=24.0, want_bvec=want_bvec, b0_angle=0.0,
                                         p_angle=0.0)
        new = session.export_cubes(bvec=want_bvec)
        for k in old:
            _same(old[k], new[k])
    xg, yg, zg = np.linspace(-3.0, 3.0, 17), np.linspace(-2.0, 2.5, 13), np.linspace(-3.0, 1.0, 15)
    gpu = cubes.resample_to_xyz_cube(model, "bp", xg, yg, zg, phi0_offset=24.0, context=session.ctx)
    ref = cubes.resample_to_xyz_cube(model, "bp", xg, yg, zg, phi0_offset=24.0, context=session.ctx, b0_angle=0.0,
                                     p_angle=0.0)
    _same(gpu, ref)


def test_zero_view_los_is_the_fixed_view_los(session, model):
    kw = dict(N_pix=20, X_range=FOV, Y_range=FOV, N_z=60, dz0=1e-3)
    res = los.resample_MAS(model, out_path=None, phi0_offset=24.0, context=session.ctx, b0_angle=0.0, p_angle=0.0, **kw)
    xs = np.linspace(*FOV, 20)
    zc, _ = los.z_grid(60, 1e-3)
    rho = _old_los_sample(session, model["rho"], xs, xs, zc, 24.0)
    te = _old_los_sample(session, model["te"], xs, xs, zc, 24.0)
    _same(res["Ne_LOS"], rho)
    te[np.isnan(rho)] = np.nan
    _same(res["Te_LOS"], te)
    session.set_spherical_model(model)
    zc, dz = los.z_grid(80, 1e-3)
    freqs = [1e9, 1.7e9, 3e9]
    for em_flag, use_bvec, diagnostics in ((5, False, False), (4, True, False), (5, False, True), (4, True, True)):
        old = _old_los_map(session, xs, xs, zc, dz * R_SUN_CM, freqs, 24.0, em_flag, use_bvec, diagnostics)
        new = session.render_los_map(xs, xs, zc, dz * R_SUN_CM, freqs, phi0_offset=24.0, pixel_area_cm2=1e20,
                                     em_flag=em_flag, use_bvec=use_bvec, diagnostics=diagnostics, b0_angle=0.0,
                                     p_angle=0.0)
        _same(old[0], new[0])
        _same(old[1], new[1])
        if diagnostics:
            for q, k in enumerate(_lib.DIAG_PLANES):
                _same(old[2][q], new[3][k])


# ---- 2. oracle parity --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("b0,p", VIEWS)
def test_resampled_cubes_match_the_oracle(session, b0, p):
    m = synthetic.spherical_corona(48, 40, 50, active_region=True)
    xg = np.linspace(-3.0, 3.0, 37); yg = np.linspace(-2.0, 2.5, 29); zg = np.linspace(-3.0, 1.0, 33)
    for name, fill in (("rho", 0.0), ("te", None), ("br", 0.0), ("bp", -7.0)):
        gpu = cubes.resample_to_xyz_cube(m, name, xg, yg, zg, phi0_offset=24.0, fill_nan=fill, context=session.ctx,
                                         b0_angle=b0, p_angle=p)
        ref = vo.resample_to_xyz_cube(m[name], xg, yg, zg, phi0_offset=24.0, fill_nan=fill, b0_angle=b0, p_angle=p)
        assert np.array_equal(np.isnan(gpu), np.isnan(ref)), name
        assert np.nanmax(np.abs(gpu - ref)) <= 1e-10 * np.nanmax(np.abs(ref)), name


def _f32_close(gpu, ref, floor):
    """float32 cubes against float64 references: the same float32 value or its neighbour; `floor` bounds components
    that cancel to ~0."""
    r32 = ref.astype(np.float32).astype(np.float64)
    d = np.abs(gpu.astype(np.float64) - r32)
    assert np.all(d <= 1.2e-7 * np.abs(r32) + floor), d.max()


@pytest.mark.parametrize("b0,p", VIEWS)
def test_composed_cubes_and_b_vector_match_the_oracle(session, model, b0, p):
    g = np.linspace(-3.0, 3.0, 41)
    session.set_model_from_spherical(model, g, g, g, phi0_offset=24.0, want_bvec=True, b0_angle=b0, p_angle=p)
    gpu = session.export_cubes(bvec=True)
    ref = vo.compose_cubes(model, g, g, g, phi0_offset=24.0, b0_angle=b0, p_angle=p)
    for k in ("ne", "te", "b"):
        _f32_close(gpu[k], ref[k], 0.0)
    for k in ("bx", "by", "bz"):
        _f32_close(gpu[k], ref[k], 1e-12 * ref["b"])
    np.testing.assert_allclose(gpu["omega_pe"], ref["omega_pe"], rtol=1e-12, atol=0)


# ---- 3. conventions, independent of the implementation ----------------------------------------------------------
@pytest.mark.parametrize("b0,p", VIEWS)
def test_conventions_sin_latitude_and_axial_field(session, b0, p):
    g = np.linspace(-2.5, 2.5, 21)
    X, Y, Z = np.meshgrid(g, g, g, indexing="ij")
    r = np.sqrt(X * X + Y * Y + Z * Z)
    ok = (r >= 1.0) & (r <= 5.0)
    n = vo.solar_north(b0, p)
    sl = vo.sin_lat_model()
    gpu = cubes.resample_to_xyz_cube(sl, "rho", g, g, g, phi0_offset=24.0, fill_nan=None, context=session.ctx,
                                     b0_angle=b0, p_angle=p)
    with np.errstate(invalid="ignore"):
        np.testing.assert_allclose(gpu[ok], ((n[0] * X + n[1] * Y + n[2] * Z) / r)[ok], rtol=0, atol=1e-5)
    ax = vo.axial_field_model(b=10.0)
    session.set_model_from_spherical(ax, g, g, g, phi0_offset=24.0, want_bvec=True, b0_angle=b0, p_angle=p)
    c = session.export_cubes(bvec=True)
    np.testing.assert_allclose(c["b"][ok], 10.0, rtol=1e-4)
    for q, k in enumerate(("bx", "by", "bz")):
        np.testing.assert_allclose(c[k][ok], 10.0 * n[q], rtol=0, atol=1e-3, err_msg=k)


# ---- 4. P = 90 deg is a quarter turn -----------------------------------------------------------------------------
def _turn(a):
    """turn(a)[i, j] = a[j, n-1-i] over the first two axes: the value at (x, y) of a map or cube whose (x, y) grids are
    the same antisymmetric grid, read at (y, -x)."""
    return np.swapaxes(np.asarray(a)[:, ::-1], 0, 1)


def test_quarter_turn_of_los_map_and_cubes(session, model):
    xs = vo.symmetric_grid(47)
    zc, dz = los.z_grid(120, 1e-3)
    session.set_spherical_model(model)
    kw = dict(phi0_offset=24.0, pixel_area_cm2=1e20, em_flag=4, use_bvec=True)
    freqs = [450e6, 1e9, 3e9]
    tb0, vi0, _ = session.render_los_map(xs, xs, zc, dz * R_SUN_CM, freqs, **kw)
    tb90, vi90, _ = session.render_los_map(xs, xs, zc, dz * R_SUN_CM, freqs, p_angle=90.0, **kw)
    for f in range(len(freqs)):
        # tb[f] is indexed (row = y, column = x): the map at (x, y) = (x[j], y[i]) is the P = 0 map at (y, -x)
        ref = np.rot90(tb0[f], -1)
        assert (ref > 0).mean() > 0.9
        np.testing.assert_allclose(tb90[f], ref, rtol=1e-9, atol=0)
        np.testing.assert_allclose(vi90[f], np.rot90(vi0[f], -1), rtol=1e-9, atol=1e-12)
    g = vo.symmetric_grid(49, 2.0 ** -3)
    session.set_model_from_spherical(model, g, g, g, phi0_offset=24.0, want_bvec=True)
    c0 = session.export_cubes(bvec=True)
    session.set_model_from_spherical(model, g, g, g, phi0_offset=24.0, want_bvec=True, p_angle=90.0)
    c90 = session.export_cubes(bvec=True)
    for k in ("omega_pe", "ne", "te", "b"):
        np.testing.assert_allclose(c90[k], _turn(c0[k]), rtol=1e-9, atol=0, err_msg=k)
    bmax = float(c0["b"].max())
    np.testing.assert_allclose(c90["bx"], -_turn(c0["by"]), rtol=1e-9, atol=1e-12 * bmax)
    np.testing.assert_allclose(c90["by"], _turn(c0["bx"]), rtol=1e-9, atol=1e-12 * bmax)
    np.testing.assert_allclose(c90["bz"], _turn(c0["bz"]), rtol=1e-9, atol=1e-12 * bmax)


# ---- 5. a model that depends on r only ---------------------------------------------------------------------------
def test_radial_model_looks_the_same_from_every_view(session):
    m = vo.radial_model()
    xs = np.linspace(*FOV, 40)
    zc, dz = los.z_grid(200, 1e-3)
    session.set_spherical_model(m)
    kw = dict(phi0_offset=24.0, pixel_area_cm2=1e20, em_flag=4, use_bvec=True)
    freqs = [75e6, 450e6, 2e9]
    tb0, vi0, _ = session.render_los_map(xs, xs, zc, dz * R_SUN_CM, freqs, **kw)
    assert (tb0 > 0).mean() > 0.9
    g = np.linspace(-3.0, 3.0, 64)
    session.set_model_from_spherical(m, g, g, g, phi0_offset=24.0, want_bvec=True)
    c0 = session.export_cubes(bvec=True)
    xr, yr, zr, kv = synthetic.ray_launch_geometry(16, 1.44, 3.0)
    area = (2 * 1.44 / 16 * R_SUN_CM) ** 2
    rm0 = session.render_map(xr, yr, zr, [(75e6, 6e-3, 2500, 10)], kvec_in_norm=kv, pixel_area_cm2=area)[0]
    assert (rm0 > 1e4).mean() > 0.5
    for b0, p in VIEWS:
        tb, vi, _ = session.render_los_map(xs, xs, zc, dz * R_SUN_CM, freqs, b0_angle=b0, p_angle=p, **kw)
        np.testing.assert_allclose(tb, tb0, rtol=1e-12, atol=0)
        np.testing.assert_allclose(vi, vi0, rtol=1e-12, atol=1e-15)
        session.set_model_from_spherical(m, g, g, g, phi0_offset=24.0, want_bvec=True, b0_angle=b0, p_angle=p)
        c = session.export_cubes(bvec=True)
        for k in ("omega_pe", "ne", "te", "b"):
            np.testing.assert_allclose(c[k], c0[k], rtol=1e-12, atol=0, err_msg=k)
        for k in ("bx", "by", "bz"):
            np.testing.assert_allclose(c[k], c0[k], rtol=0, atol=1e-12 * float(c0["b"].max()), err_msg=k)
        rm = session.render_map(xr, yr, zr, [(75e6, 6e-3, 2500, 10)], kvec_in_norm=kv, pixel_area_cm2=area)[0]
        np.testing.assert_allclose(rm, rm0, rtol=1e-9, atol=0)


# ---- 6. the renderers at a non-zero view -------------------------------------------------------------------------
def test_los_map_matches_staged_path_and_oracle_at_a_view(session, model, oracle, monkeypatch):
    b0, p = -30.0, 115.0
    kw = dict(N_pix=16, X_range=FOV, Y_range=FOV, N_z=120, dz0=1e-3)
    staged = los.SyntheticFF(los.resample_MAS(model, out_path=None, phi0_offset=24.0, context=session.ctx,
                                              b0_angle=b0, p_angle=p, **kw), 450e6, 4, 0.1, session=session)
    fused = los.render_los_map(model, freq0=450e6, Nfreq=4, freq_log_step=0.1, phi0_offset=24.0, session=session,
                               b0_angle=b0, p_angle=p, **kw)
    zero = los.render_los_map(model, freq0=450e6, Nfreq=4, freq_log_step=0.1, phi0_offset=24.0, session=session, **kw)
    tb, ref = fused["emission_cube"], staged["emission_cube"]
    assert np.array_equal(tb == 0, ref == 0)
    nz = ref > 0
    assert nz.mean() > 0.9
    np.testing.assert_allclose(tb[nz], ref[nz], rtol=1e-4)
    assert np.abs(tb[nz] / zero["emission_cube"][nz] - 1).max() > 1e-2          # the view changes the map
    # theta from the rotated B vector with gyroresonance, on the active region, against the CPU restatement
    n_pix, f0, nf, step = 16, 1e9, 3, np.log10(3.0) / 2
    xr, yr = (0.0, 0.6), (-0.1, 0.5)
    b0, p = 7.25, 24.0
    zc, dz = los.z_grid(120, 1e-3)
    smp = vo.los_samples(model, np.linspace(*xr, n_pix), np.linspace(*yr, n_pix), zc, 0.0, b0_angle=b0, p_angle=p)
    kw = dict(N_pix=n_pix, X_range=xr, Y_range=yr, N_z=120, dz0=1e-3, freq0=f0, Nfreq=nf, freq_log_step=step,
              use_bvec=True, session=session)
    gr = los.render_los_map(model, em_flag=4, b0_angle=b0, p_angle=p, **kw)
    gr0 = los.render_los_map(model, em_flag=4, **kw)
    area = ((gr["x_coords"][1] - gr["x_coords"][0]) / (R_SUN_CM * 1e-2) * R_SUN_CM) ** 2
    # los_map_oracle takes theta from its zero-view rotation: hand it the view's
    monkeypatch.setattr(lmo, "bvec_theta_deg",
                        lambda x, y, z, br, bt, bp: (vo.bvec_theta_deg(x, y, z, br, bt, bp, b0, p), None))
    tb_ref, vi_ref = lmo.los_map(smp, dz * R_SUN_CM, area, f0, nf, step, em_flag=4, use_bvec=True)
    tb = gr["emission_cube"]
    nz = tb_ref > 0
    assert nz.mean() > 0.9
    np.testing.assert_allclose(tb[nz], tb_ref[nz], rtol=1e-4)
    fin = np.isfinite(vi_ref) & nz
    np.testing.assert_allclose(gr["emission_polVI_cube"][fin], vi_ref[fin], atol=1e-4, rtol=0)
    assert np.abs(tb[nz] / gr0["emission_cube"][nz] - 1).max() > 1e-2


def test_cubes_composed_at_a_view_drive_the_same_rays(session, model):
    """set_model_from_spherical(view) == uploading the oracle-composed cubes of that view (the tolerances of
    test_cubes.test_cubes_composed_on_device_drive_the_same_rays), θ from the B vector included."""
    b0, p = -30.0, 115.0
    g = np.linspace(-3.0, 3.0, 48)
    c = vo.compose_cubes(model, g, g, g, phi0_offset=24.0, b0_angle=b0, p_angle=p)
    xs, ys, zs, kv = synthetic.ray_launch_geometry(10, 1.3, 3.0)
    start = np.column_stack([xs, ys, zs])
    area = (2 * 1.3 / 10 * R_SUN_CM) ** 2
    session.set_omega_cube(c["omega_pe"], g, g, g)
    session.set_field_cubes(g, g, g, c["ne"], c["te"], c["b"], c["bx"], c["by"], c["bz"])
    r_a, _, _ = session.trace(75e6, xs, ys, zs, kv, 6e-3, 2500, 10, True, 2.0)
    smp_a = session.sample_traced(start, R_SUN_CM)
    tb_a, _ = session.emission_traced(area, 75e6)
    tv_a = session.render_map(xs, ys, zs, [(1e9, 1e-3, 4000, 5)], kvec_in_norm=kv, pixel_area_cm2=area, em_flag=4,
                              use_bvec=True)[0]
    session.set_model_from_spherical(model, g, g, g, phi0_offset=24.0, want_bvec=True, b0_angle=b0, p_angle=p)
    r_b, _, _ = session.trace(75e6, xs, ys, zs, kv, 6e-3, 2500, 10, True, 2.0)
    smp_b = session.sample_traced(start, R_SUN_CM)
    tb_b, _ = session.emission_traced(area, 75e6)
    tv_b = session.render_map(xs, ys, zs, [(1e9, 1e-3, 4000, 5)], kvec_in_norm=kv, pixel_area_cm2=area, em_flag=4,
                              use_bvec=True)[0]
    assert np.nanmax(np.abs(r_a - r_b)) < 1e-7
    assert np.array_equal(smp_a["valid_mask"], smp_b["valid_mask"])
    v = smp_a["valid_mask"]
    for k in ("ne", "te", "b"):
        np.testing.assert_allclose(smp_a[k][v], smp_b[k][v], rtol=2e-6)
    nz = tb_a != 0
    assert nz.any()
    np.testing.assert_allclose(tb_b[nz], tb_a[nz], rtol=1e-5)
    nz = tv_a != 0
    assert nz.mean() > 0.5
    np.testing.assert_allclose(tv_b[nz], tv_a[nz], rtol=1e-5)


# ---- 7. front ends -----------------------------------------------------------------------------------------------
def _quarter_turn_params(freq_hz):
    # exactly antisymmetric grids: linspace(-3, 3, 49) steps by 1/8 and linspace(-1.5, 1.5, 13) by 1/4
    return {"grid_n": 49, "grid_extent": 3.0, "z_observer": 3.0, "x_fov": 1.5, "dt": 6e-3, "n_steps": 2500,
            "record_stride": 10}


def test_workflow_and_sweep_at_p90_are_the_turned_maps(session, model, tmp_path):
    from raytracinggrff_b200 import cubes as cb, sweep, workflow
    kw = dict(N_pix=13, fmin_mhz=75.0, fmax_mhz=75.0, n_freq=1, phi0_offset=24.0, session=session,
              params_fn=_quarter_turn_params)
    rows0 = sweep.tb_spectra(model, tmp_path / "s0", **kw)
    s0 = np.load(rows0[0][2])["emission_cube"][:, :, 0]
    s90 = np.load(sweep.tb_spectra(model, tmp_path / "s90", p_angle=90.0, **kw)[0][2])["emission_cube"][:, :, 0]
    # the sweep's log-spaced frequency (75000000.00000001 Hz): the workflow runs at the same one, so the two front ends
    # must agree bit for bit
    freq = rows0[0][1]
    path = tmp_path / "model.npz"
    cb.save_spherical_model(path, model)
    args = ["--model-path", str(path), "--N-pix", "13", "--X-FOV", "1.5", "--grid-n", "49", "--grid-extent", "3.0",
            "--n-steps", "2500", "--grff-backend", "fused", "--phi0-offset", "24", "--freq", repr(freq), "--quiet"]
    m0 = workflow.main(args + ["--out-path", str(tmp_path / "m0.npz")])["emission_cube"][:, :, 0]
    m90 = workflow.main(args + ["--out-path", str(tmp_path / "m90.npz"), "--p-angle", "90"])["emission_cube"][:, :, 0]
    mb = workflow.main(args + ["--out-path", str(tmp_path / "mb.npz"), "--b0-angle", "7.25"])["emission_cube"][:, :, 0]
    assert (m0 > 1e4).mean() > 0.5
    assert np.abs(mb / m0 - 1)[m0 > 1e4].max() > 1e-3
    assert np.array_equal(s0, m0) and np.array_equal(s90, m90)
    # The view path is exact: the P = 0 cubes turned in numpy and uploaded as a Cartesian model give the P = 90 map bit
    # for bit.  The turned map itself differs from the P = 0 map at float32 rounding (1.5e-7 on a B200), because the
    # tracer's FP32 trilinear weights are not mirror-symmetric ((x - x0) / dx against 1 - that).
    g = np.linspace(-3.0, 3.0, 49)
    session.set_model_from_spherical(model, g, g, g, phi0_offset=24.0)
    c0 = session.export_cubes()
    turned = dict(x_grid=g, y_grid=g, z_grid=g, **{k: np.ascontiguousarray(_turn(v)) for k, v in c0.items()})
    mt = workflow.run_ray_tracing_emission(turned, N_pix=13, X_fov=1.5, freq_hz=freq, n_steps=2500,
                                           grff_backend="fused", session=session, verbose=False)["emission_cube"][:, :, 0]
    assert np.array_equal(m90, mt)
    np.testing.assert_allclose(m90, np.rot90(m0, -1), rtol=1e-6, atol=0)


def test_errors(session, model):
    g = np.linspace(-2.0, 2.0, 9)
    for b0, p in ((np.nan, 0.0), (0.0, -np.inf), (90.01, 0.0)):
        with pytest.raises(ValueError):
            session.set_model_from_spherical(model, g, g, g, b0_angle=b0, p_angle=p)
        with pytest.raises(ValueError):
            session.render_los_map(g, g, [0.1], [1e9], [1e9], b0_angle=b0, p_angle=p)
    # the C library checks the angles too, and composition needs one view for all five slots
    lib = _lib.load()
    v = model["rho"]
    data, phi, lat, r = f32(v.data), f64(v.phi), f64(v.lat), f64(v.r)
    gg, geom = f64(g), _lib.grid_geom(g, g, g)

    def resample(slot, b0, p):
        return lib.rtgrff_resample_spherical_view(session.ctx.handle, slot, ptr(data, c_float), ptr(phi, c_double),
                                                  ptr(lat, c_double), ptr(r, c_double), *data.shape, ptr(gg, c_double),
                                                  ptr(gg, c_double), ptr(gg, c_double), 9, 9, 9, ptr(geom, c_double),
                                                  0.0, b0, p, 0.999999, 1.0, 0.0, 1, None)
    assert resample(0, float("nan"), 0.0) == _lib.RTGRFF_EINVAL
    assert resample(0, -90.5, 0.0) == _lib.RTGRFF_EINVAL
    for slot in range(5):
        assert resample(slot, 7.25 if slot != 3 else 7.0, 24.0) == _lib.RTGRFF_OK
    assert lib.rtgrff_compose_cubes(session.ctx.handle, 1) == _lib.RTGRFF_EINVAL
    assert resample(3, 7.25, 24.0) == _lib.RTGRFF_OK
    assert lib.rtgrff_compose_cubes(session.ctx.handle, 1) == _lib.RTGRFF_OK
    # a Cartesian cube model cannot be re-oriented
    from raytracinggrff_b200.workflow import run_ray_tracing_emission
    with pytest.raises(ValueError):
        run_ray_tracing_emission(synthetic.corona_cube(16, 3.0), N_pix=4, grff_backend="fused", p_angle=10.0,
                                 session=session)
