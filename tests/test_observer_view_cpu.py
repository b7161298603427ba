"""Observer view (solar B0 and P angles), CPU part: the CPU restatement in tests/view_oracle.py against the zero-view
oracle and against the conventions of include/rtgrff.h, the argument checks and the command lines."""
import numpy as np
import pytest

import los_map_oracle as lmo
import view_oracle as vo
from oracle import oracle_cubes as oc
from raytracinggrff_b200 import cubes, synthetic

VIEWS = ((7.25, 0.0), (0.0, 24.0), (-30.0, 115.0))


def test_view_matrix_is_a_rotation_that_takes_solar_north_to_the_model_axis():
    for b0, p in VIEWS + ((90.0, 0.0), (-90.0, 360.0)):
        m = vo.view_matrix(b0, p)
        np.testing.assert_allclose(m @ m.T, np.eye(3), atol=1e-15)
        assert np.linalg.det(m) == pytest.approx(1.0)
        np.testing.assert_allclose(m @ vo.solar_north(b0, p), [0.0, 1.0, 0.0], atol=1e-15)
    # B0 > 0 tilts north towards the observer (+z), P > 0 turns it towards east (-x)
    assert vo.solar_north(7.25, 0.0)[2] > 0 and vo.solar_north(0.0, 24.0)[0] < 0


def test_zero_view_is_the_zero_view_oracle():
    m = synthetic.spherical_corona(24, 20, 30, active_region=True)
    g = np.linspace(-3.0, 3.0, 11)
    a = vo.compose_cubes(m, g, g, g, phi0_offset=24.0)
    b = oc.compose_cubes(m, g, g, g, phi0_offset=24.0)
    for k in ("omega_pe", "ne", "te", "b", "br", "bt", "bp"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    zc = np.cumsum(np.full(20, 0.05))
    xs = np.linspace(-1.4, 1.4, 6)
    s0, s1 = vo.los_samples(m, xs, xs, zc, 24.0), lmo.los_samples(m, xs, xs, zc, 24.0)
    for k in s1:
        np.testing.assert_array_equal(s0[k], s1[k], err_msg=k)
    np.testing.assert_array_equal(vo.bvec_theta_deg(s0["x"], s0["y"], s0["z"], s0["br"], s0["bt"], s0["bp"]),
                                  lmo.bvec_theta_deg(s1["x"], s1["y"], s1["z"], s1["br"], s1["bt"], s1["bp"])[0])


@pytest.mark.parametrize("b0,p", VIEWS)
def test_sin_latitude_resamples_to_north_dot_unit_vector(b0, p):
    """Independent of the implementation: a variable equal to sin(latitude) is n . p / |p| (n: the view's solar north);
    the tolerance is the linear interpolation error in latitude (dlat^2 / 8 = 5e-6 on a 0.25 deg mesh)."""
    m = vo.sin_lat_model()
    g = np.linspace(-2.5, 2.5, 15)
    out = vo.resample_to_xyz_cube(m["rho"], g, g, g, phi0_offset=24.0, fill_nan=None, b0_angle=b0, p_angle=p)
    X, Y, Z = np.meshgrid(g, g, g, indexing="ij")
    r = np.sqrt(X * X + Y * Y + Z * Z)
    n = vo.solar_north(b0, p)
    ok = (r >= 1.0) & (r <= 5.0)
    assert np.all(np.isfinite(out[ok]))
    np.testing.assert_allclose(out[ok], (n[0] * X + n[1] * Y + n[2] * Z)[ok] / r[ok], rtol=0, atol=1e-5)


@pytest.mark.parametrize("b0,p", VIEWS)
def test_axial_field_composes_to_b_times_north(b0, p):
    m = vo.axial_field_model(b=10.0)
    g = np.linspace(-2.5, 2.5, 15)
    c = vo.compose_cubes(m, g, g, g, phi0_offset=24.0, b0_angle=b0, p_angle=p)
    X, Y, Z = np.meshgrid(g, g, g, indexing="ij")
    r = np.sqrt(X * X + Y * Y + Z * Z)
    ok = (r >= 1.0) & (r <= 5.0)
    n = vo.solar_north(b0, p)
    np.testing.assert_allclose(c["b"][ok], 10.0, rtol=1e-4)
    for q, k in enumerate(("bx", "by", "bz")):
        np.testing.assert_allclose(c[k][ok], 10.0 * n[q], rtol=0, atol=1e-3, err_msg=k)


def test_quarter_turn_permutes_the_oracle_cube():
    """P = 90 deg on an exactly antisymmetric grid: the cube at (x, y) is the P = 0 cube at (y, -x)."""
    m = synthetic.spherical_corona(24, 20, 30, active_region=True)
    g = vo.symmetric_grid(21, 2.0 ** -3)
    c0 = vo.compose_cubes(m, g, g, g, phi0_offset=24.0)
    c90 = vo.compose_cubes(m, g, g, g, phi0_offset=24.0, p_angle=90.0)

    def turn(a):
        return np.transpose(a[:, ::-1, :], (1, 0, 2))       # turn(a)[i, j] = a[j, n-1-i]
    for k in ("ne", "te", "b"):
        np.testing.assert_allclose(c90[k], turn(c0[k]), rtol=1e-9, atol=0, err_msg=k)
    np.testing.assert_allclose(c90["bx"], -turn(c0["by"]), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(c90["by"], turn(c0["bx"]), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(c90["bz"], turn(c0["bz"]), rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("b0,p", [(np.nan, 0.0), (0.0, np.inf), (90.5, 0.0), (-91.0, 10.0)])
def test_bad_angles_raise_before_any_gpu_work(b0, p):
    from raytracinggrff_b200 import los
    m = synthetic.spherical_corona(12, 10, 16)
    g = np.linspace(-2.0, 2.0, 5)
    with pytest.raises(ValueError):
        cubes.check_view(b0, p)
    with pytest.raises(ValueError):
        cubes.resample_to_xyz_cube(m, "rho", g, g, g, b0_angle=b0, p_angle=p)
    with pytest.raises(ValueError):
        los.resample_MAS(m, 4, (-1, 1), (-1, 1), 8, 1e-3, out_path=None, b0_angle=b0, p_angle=p)
    with pytest.raises(ValueError):
        los.render_los_map(m, 4, (-1, 1), (-1, 1), 8, 1e-3, 1e8, 1, 0.0, b0_angle=b0, p_angle=p)
    from raytracinggrff_b200.workflow import run_ray_tracing_emission
    with pytest.raises(ValueError):
        run_ray_tracing_emission(m, N_pix=4, b0_angle=b0, p_angle=p)


def test_cartesian_model_with_a_view_raises_before_any_gpu_work():
    from raytracinggrff_b200.workflow import run_ray_tracing_emission
    c = synthetic.corona_cube(8, 3.0)
    for b0, p in ((7.25, 0.0), (0.0, -3.0)):
        with pytest.raises(ValueError, match="spherical model"):
            run_ray_tracing_emission(c, N_pix=4, grff_backend="fused", b0_angle=b0, p_angle=p)


def test_command_lines_pass_the_view_through(monkeypatch, tmp_path):
    from raytracinggrff_b200 import sweep, workflow
    seen = {}

    def fake_run(model, **kw):
        seen["workflow"] = kw
        return {"emission_cube": np.zeros((2, 2, 1))}

    def fake_sweep(model, out_dir, *args, **kw):
        seen["sweep"] = kw
        return []
    monkeypatch.setattr(workflow, "run_ray_tracing_emission", fake_run)
    monkeypatch.setattr(sweep, "tb_spectra", fake_sweep)
    monkeypatch.setattr(synthetic, "spherical_corona", lambda *a, **k: {})
    workflow.main(["--b0-angle", "7.25", "--p-angle", "-24", "--quiet", "--out-path", str(tmp_path / "m.npz")])
    assert seen["workflow"]["b0_angle"] == 7.25 and seen["workflow"]["p_angle"] == -24.0
    workflow.main(["--quiet", "--out-path", str(tmp_path / "m.npz")])
    assert seen["workflow"]["b0_angle"] == 0.0 and seen["workflow"]["p_angle"] == 0.0
    sweep.main(["--b0-angle", "-3.5", "--p-angle", "115", "--out-dir", str(tmp_path / "s")])
    assert seen["sweep"]["b0_angle"] == -3.5 and seen["sweep"]["p_angle"] == 115.0
