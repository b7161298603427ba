"""GPU: the fused straight line-of-sight map (los.render_los_map / RaySession.render_los_map / rtgrff_render_los_map).

* parity with the staged drop-ins resample_MAS + SyntheticFF (the same LOS samples and packing rules), with the
  FP64 voxel evaluation too, and with the CPU oracle chain;
* theta from the B vector with gyroresonance against a CPU restatement (tests/los_map_oracle.py);
* the diagnostic planes against tests/diag_oracle.get_mw_diag on the LOS sample positions;
* frequency groups, device output through the image gather, errors and repeatability.
"""
import ctypes

import numpy as np
import pytest

import los_map_oracle as lmo
from raytracinggrff_b200 import _lib, los, synthetic

pytestmark = pytest.mark.gpu

R_SUN_CM = 6.957e10
PLANES = ("em_x", "em_y", "em_z", "em_r", "tau_L", "tau_R", "ray_r_min")
FOV = (-1.44, 1.44)


@pytest.fixture(scope="module")
def model():
    return synthetic.spherical_corona(64, 48, 64, r_max=8.0, active_region=True)


def _kw(n_pix, n_z=120):
    return dict(N_pix=n_pix, X_range=FOV, Y_range=FOV, N_z=n_z, dz0=1e-3)


def _same_patterns(a, b):
    assert np.array_equal(np.isnan(a), np.isnan(b))
    assert np.array_equal(a == 0, b == 0)


@pytest.mark.parametrize("n_pix", [14, 64])
def test_matches_staged_resample_mas_and_synthetic_ff(session, model, n_pix):
    kw = _kw(n_pix)
    staged = los.SyntheticFF(los.resample_MAS(model, out_path=None, phi0_offset=24.0, context=session.ctx, verbose=False,
                                              **kw), 450e6, 4, 0.1, session=session)
    fused = los.render_los_map(model, freq0=450e6, Nfreq=4, freq_log_step=0.1, phi0_offset=24.0, session=session, **kw)
    assert set(fused) == set(staged)
    for k in ("frequencies_Hz", "x_coords", "y_coords"):
        assert np.array_equal(fused[k], staged[k]), k
    tb, tb_ref = fused["emission_cube"], staged["emission_cube"]
    vi, vi_ref = fused["emission_polVI_cube"], staged["emission_polVI_cube"]
    assert tb.shape == tb_ref.shape == (n_pix, n_pix, 4)
    _same_patterns(tb, tb_ref)
    _same_patterns(vi, vi_ref)
    nz = tb_ref > 0
    assert nz.mean() > 0.9
    np.testing.assert_allclose(tb[nz], tb_ref[nz], rtol=1e-4)
    fin = np.isfinite(vi_ref)
    np.testing.assert_allclose(vi[fin], vi_ref[fin], atol=1e-4, rtol=0)
    # the FP64 voxel evaluation: left are the float32 voxel inputs (7 significant digits)
    session.ctx.set_grff64(True)
    try:
        f64 = los.render_los_map(model, freq0=450e6, Nfreq=4, freq_log_step=0.1, phi0_offset=24.0, session=session, **kw)
    finally:
        session.ctx.set_grff64(False)
    _same_patterns(f64["emission_cube"], tb_ref)
    np.testing.assert_allclose(f64["emission_cube"][nz], tb_ref[nz], rtol=1e-6)


def test_stats_count_the_staged_valid_samples(session, model):
    kw = _kw(24)
    smp = los.resample_MAS(model, out_path=None, context=session.ctx, **kw)
    n_valid = int((~(np.isnan(smp["Ne_LOS"]) | np.isnan(smp["Te_LOS"]) | np.isnan(smp["B_LOS"]))).sum())
    zc, dz = los.z_grid(120, 1e-3)
    xs = np.linspace(*FOV, 24)
    session.set_spherical_model(model)
    _, _, st = session.render_los_map(xs, xs, zc, dz * R_SUN_CM, [1e8, 2e8, 3e8])
    assert st == {"los_samples": 24 * 24 * 120, "valid_samples": n_valid, "voxel_freq_evaluations": 3 * n_valid}


def test_matches_cpu_oracle(session, model, oracle):
    from oracle import oracle_cubes as oc
    kw = _kw(14)
    ref = oc.resample_MAS(model, phi0_offset=24.0, **kw)
    area = ((ref["x_coords"][1] - ref["x_coords"][0]) / (R_SUN_CM * 1e-2) * R_SUN_CM) ** 2
    tb_ref, vi_ref, f_ref = oracle.emission_from_los(ref["Ne_LOS"], ref["Te_LOS"], ref["B_LOS"], ref["ds_LOS"], area,
                                                     450e6, 4, 0.1)
    res = los.render_los_map(model, freq0=450e6, Nfreq=4, freq_log_step=0.1, phi0_offset=24.0, session=session, **kw)
    np.testing.assert_array_equal(res["frequencies_Hz"], f_ref)
    nz = tb_ref > 0
    assert nz.mean() > 0.9
    np.testing.assert_allclose(res["emission_cube"][nz], tb_ref[nz], rtol=1e-4)
    np.testing.assert_allclose(res["emission_polVI_cube"][nz], vi_ref[nz], atol=1e-4)


def test_theta_from_b_with_gyroresonance_matches_cpu_restatement(session, model, oracle):
    """A field of view on the active region (up to ~360 G on the LOS): gyroresonance layers at 1 - 3 GHz."""
    n_pix, f0, nf, step = 16, 1e9, 3, np.log10(3.0) / 2          # 1, 1.73, 3 GHz
    xr, yr = (0.1, 0.5), (0.0, 0.4)
    zc, dz = los.z_grid(120, 1e-3)
    smp = lmo.los_samples(model, np.linspace(*xr, n_pix), np.linspace(*yr, n_pix), zc, 0.0)
    dz_cm = dz * R_SUN_CM
    kw = dict(freq0=f0, Nfreq=nf, freq_log_step=step, use_bvec=True, session=session,
              **dict(_kw(n_pix), X_range=xr, Y_range=yr))
    gr = los.render_los_map(model, em_flag=4, **kw)
    ff = los.render_los_map(model, em_flag=5, **kw)
    area = ((gr["x_coords"][1] - gr["x_coords"][0]) / (R_SUN_CM * 1e-2) * R_SUN_CM) ** 2
    tb_ref, vi_ref = lmo.los_map(smp, dz_cm, area, f0, nf, step, em_flag=4, use_bvec=True)
    tb = gr["emission_cube"]
    nz = tb_ref > 0
    assert nz.mean() > 0.9
    np.testing.assert_allclose(tb[nz], tb_ref[nz], rtol=1e-4)
    fin = np.isfinite(vi_ref) & nz
    np.testing.assert_allclose(gr["emission_polVI_cube"][fin], vi_ref[fin], atol=1e-4, rtol=0)
    # gyroresonance really acts on this case
    rel = np.abs(tb[nz] - ff["emission_cube"][nz]) / ff["emission_cube"][nz]
    assert (rel > 0.1).sum() > 0, rel.max()


def test_diagnostics(session, model, oracle):
    import diag_oracle
    n_pix = 12
    base = dict(freq0=450e6, Nfreq=3, freq_log_step=0.3, phi0_offset=24.0, session=session, **_kw(n_pix))
    # theta = 90: T_b and V/I of the diagnostic kernels are the plain kernels' bit for bit
    for em_flag in (4, 5):
        plain = los.render_los_map(model, em_flag=em_flag, **base)
        dg = los.render_los_map(model, em_flag=em_flag, diagnostics=True, **base)
        for k in ("emission_cube", "emission_polVI_cube"):
            assert np.array_equal(plain[k], dg[k], equal_nan=True), (em_flag, k)
    assert dg["emission_centroid_xyz"].shape == (n_pix, n_pix, 3, 3)
    # planes against the CPU diagnostics on the LOS sample positions, theta from B with gyroresonance
    xs = np.linspace(*FOV, n_pix)
    zc, dz = los.z_grid(120, 1e-3)
    session.set_spherical_model(model)
    area = ((xs[1] - xs[0]) * R_SUN_CM) ** 2
    freqs = 450e6 * 10.0 ** (0.3 * np.arange(3))
    tb, vi, _, d = session.render_los_map(xs, xs, zc, dz * R_SUN_CM, freqs, phi0_offset=24.0, pixel_area_cm2=area,
                                          em_flag=4, use_bvec=True, diagnostics=True)
    smp = lmo.los_samples(model, xs, xs, zc, 24.0)
    tb_ref, _, ref = lmo.los_map(smp, dz * R_SUN_CM, area, 450e6, 3, 0.3, em_flag=4, use_bvec=True, diagnostics=True)
    got = {k: np.moveaxis(v, 0, -1) for k, v in d.items()}
    nz = tb_ref > 0
    np.testing.assert_allclose(np.moveaxis(tb, 0, -1)[nz], tb_ref[nz], rtol=1e-4)
    for k in ("em_x", "em_y", "em_z", "em_r"):
        assert np.array_equal(np.isnan(got[k]), np.isnan(ref[k])), k
        ok = ~np.isnan(ref[k])
        assert np.abs(got[k][ok] - ref[k][ok]).max() <= diag_oracle.EM_TOL, k
    for k in ("tau_L", "tau_R"):
        assert diag_oracle._tau_close(got[k], ref[k], diag_oracle.TAU_RTOL).all(), k
    assert np.abs(got["ray_r_min"] - ref["ray_r_min"]).max() <= diag_oracle.RMIN_TOL
    # the centroid lies on its LOS: between the first and the last sample
    z = smp["z"]
    ok = ~np.isnan(got["em_z"])
    assert ok.mean() > 0.9
    lo = np.broadcast_to(z.min(axis=2)[:, :, None], ok.shape)
    hi = np.broadcast_to(z.max(axis=2)[:, :, None], ok.shape)
    assert np.all(got["em_z"][ok] >= lo[ok] - 1e-6) and np.all(got["em_z"][ok] <= hi[ok] + 1e-6)
    assert ((ref["tau_L"] > 1) & (ref["tau_R"] > 1)).any() and ((ref["tau_L"] < 0.1) & (ref["tau_R"] < 0.1)).any()


def _bvec_gr_call(session, xs, ys, freqs, **kw):
    zc, dz = los.z_grid(120, 1e-3)
    return session.render_los_map(xs, ys, zc, dz * R_SUN_CM, freqs, phi0_offset=24.0, pixel_area_cm2=1e18, em_flag=4,
                                  use_bvec=True, **kw)


@pytest.mark.parametrize("n_freq", [1, 3, 8, 17])
def test_every_frequency_row_equals_a_single_frequency_call(session, model, n_freq):
    session.set_spherical_model(model)
    xs, ys = np.linspace(*FOV, 21), np.linspace(-1.2, 1.3, 19)     # partial tiles on both axes
    freqs = np.random.default_rng(n_freq).permutation(np.geomspace(75e6, 3e9, n_freq))
    tb, vi, _, dg = _bvec_gr_call(session, xs, ys, freqs, diagnostics=True)
    assert tb.shape == (n_freq, 19, 21)
    for f in range(n_freq):
        tb1, vi1, _, d1 = _bvec_gr_call(session, xs, ys, [freqs[f]], diagnostics=True)
        assert np.array_equal(tb[f], tb1[0]) and np.array_equal(vi[f], vi1[0], equal_nan=True), f
        for k in PLANES:
            assert np.array_equal(dg[k][f], d1[k][0], equal_nan=True), (f, k)


def test_row_shards_on_device_assemble_to_the_whole_image(session, model):
    """Two ranks' row shards written with out_device_ptrs, placed by rtgrff_place_rows (the root half of
    rtgrff_gather_image), and the whole image through rtgrff_gather_image, against the host call."""
    from raytracinggrff_b200 import dist
    session.set_spherical_model(model)
    n, freqs = 32, [150e6, 600e6]
    nf = len(freqs)
    xs = np.linspace(*FOV, n)
    tb, vi, _, dg = _bvec_gr_call(session, xs, xs, freqs, diagnostics=True)
    want = np.concatenate([tb, vi, np.stack([dg[k] for k in PLANES]).reshape(7 * nf, n, n)])
    n_planes = 9 * nf
    lib = _lib.load()
    shards = [dist.c_shard_rows(n, 2, r) for r in range(2)]
    mr = shards[0][1]
    assert all(len(rows) == mr for rows, _ in shards)
    slab_b = n_planes * mr * n * 8
    gathered, image = ctypes.c_void_p(), ctypes.c_void_p()
    _lib.check(lib.rtgrff_device_alloc(session.ctx.handle, ctypes.byref(gathered), 2 * slab_b))
    _lib.check(lib.rtgrff_device_alloc(session.ctx.handle, ctypes.byref(image), n_planes * n * n * 8))
    try:
        for r, (rows, _) in enumerate(shards):
            base = gathered.value + r * slab_b
            pb = nf * mr * n * 8
            out = _bvec_gr_call(session, xs, xs[rows], freqs, diagnostics=True, out_device_ptrs=(base, base + pb, base + 2 * pb))
            assert out[0] is None and out[3] is None
        _lib.check(lib.rtgrff_place_rows(session.ctx.handle, gathered, 2, n_planes, n, n, image))
        img = np.zeros((n_planes, n, n))
        _lib.check(lib.rtgrff_memcpy(session.ctx.handle, img.ctypes.data_as(ctypes.c_void_p), image, img.nbytes, 1))
        assert np.array_equal(img, want, equal_nan=True)
        # one rank: the whole image on the device, through rtgrff_gather_image
        pb = nf * n * n * 8
        _bvec_gr_call(session, xs, xs, freqs, diagnostics=True, out_device_ptrs=(image.value, image.value + pb,
                                                                                 image.value + 2 * pb))
        session.comm_init(1, 0)
        img = np.zeros((n_planes, n, n))
        session.gather_image(image.value, n_planes, n, n, root=0, out=img)
        assert np.array_equal(img, want, equal_nan=True)
    finally:
        lib.rtgrff_device_free(session.ctx.handle, gathered)
        lib.rtgrff_device_free(session.ctx.handle, image)
        session.comm_destroy()


def _c_call(ses, **over):
    lib = _lib.load()
    x = np.linspace(-1, 1, 4)
    zc, dz = los.z_grid(10, 1e-3)
    f = np.array([1e8])
    tb, vi = np.zeros(16), np.zeros(16)
    dp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))   # noqa: E731
    a = dict(nx=4, ny=4, x=dp(x), y=dp(x), nz=10, zc=dp(zc), dz=dp(dz * R_SUN_CM), n_freq=1, freq=dp(f),
             tb=tb.ctypes.data_as(ctypes.c_void_p), vi=vi.ctypes.data_as(ctypes.c_void_p))
    a.update(over)
    return lib.rtgrff_render_los_map(ses.ctx.handle, a["nx"], a["ny"], a["x"], a["y"], a["nz"], a["zc"], a["dz"], 0.0,
                                     los.R_MIN, 1e-6 / 6.957e8, a["n_freq"], a["freq"], 1e18, 5, 30, 0, a["tb"],
                                     a["vi"], None, 0, None)


def test_errors(model):
    from raytracinggrff_b200 import RaySession
    with RaySession(0) as ses:
        assert _c_call(ses) == _lib.RTGRFF_ENOCUBE            # no slot set
        lib = _lib.load()
        v = model["rho"]
        data = np.ascontiguousarray(v.data, dtype=np.float32)
        phi, lat, r = (np.ascontiguousarray(a, dtype=np.float64) for a in (v.phi, v.lat, v.r))
        fp = ctypes.POINTER(ctypes.c_float)
        dp = ctypes.POINTER(ctypes.c_double)
        args = [data.ctypes.data_as(fp), phi.ctypes.data_as(dp), lat.ctypes.data_as(dp), r.ctypes.data_as(dp),
                *data.shape, 1.0]
        h = ses.ctx.handle
        assert lib.rtgrff_set_spherical_model(h, 5, *args) == _lib.RTGRFF_EINVAL
        assert lib.rtgrff_set_spherical_model(h, 0, None, *args[1:]) == _lib.RTGRFF_EINVAL
        rev = phi[::-1].copy()
        assert lib.rtgrff_set_spherical_model(h, 0, args[0], rev.ctypes.data_as(dp), *args[2:]) == _lib.RTGRFF_EINVAL
        assert lib.rtgrff_set_spherical_model(h, 0, *args[:4], 1, data.shape[1], data.shape[2], 1.0) == _lib.RTGRFF_EINVAL
        for slot in range(4):
            assert lib.rtgrff_set_spherical_model(h, slot, *args) == _lib.RTGRFF_OK
        assert _c_call(ses) == _lib.RTGRFF_ENOCUBE            # bp missing
        ses.set_spherical_model(model)
        assert _c_call(ses) == _lib.RTGRFF_OK
        for bad in (dict(n_freq=0), dict(nx=0), dict(ny=-1), dict(nz=0), dict(x=None), dict(zc=None), dict(dz=None),
                    dict(freq=None), dict(tb=None), dict(vi=None)):
            assert _c_call(ses, **bad) == _lib.RTGRFF_EINVAL, bad
        f0 = np.array([0.0])
        assert _c_call(ses, freq=f0.ctypes.data_as(dp)) == _lib.RTGRFF_EINVAL
        with pytest.raises(ValueError):
            ses.render_los_map(np.zeros(4), np.zeros(4), np.zeros(3), np.zeros(2), [1e8])


def test_large_map_is_repeatable(session, model):
    session.set_spherical_model(model)
    xs = np.linspace(*FOV, 512)
    zc, dz = los.z_grid(400, 3e-4)
    freqs = np.geomspace(75e6, 1.5e9, 8)
    a = session.render_los_map(xs, xs, zc, dz * R_SUN_CM, freqs, pixel_area_cm2=1e18)
    b = session.render_los_map(xs, xs, zc, dz * R_SUN_CM, freqs, pixel_area_cm2=1e18)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1], equal_nan=True)
    assert (a[0] > 0).mean() > 0.5


def test_model_upload_is_skipped_when_repeated(session, model):
    session.set_spherical_model(model)
    keys = list(session.ctx.__dict__["_sph_keys"])
    assert None not in keys
    session.set_spherical_model(model)
    assert session.ctx.__dict__["_sph_keys"] == keys
    other = dict(model, rho=synthetic.spherical_corona(64, 48, 64, r_max=8.0)["rho"])
    session.set_spherical_model(other)
    assert session.ctx.__dict__["_sph_keys"][0] != keys[0] and session.ctx.__dict__["_sph_keys"][1:] == keys[1:]
