"""GPU: the step loop of the fused map (render_map_kernel) against the staged trace -> sample -> emission path.

The fused kernel steps in record intervals: a step with the cross-section pencil traced (the recorded step of the
per-step S schedule), then the central ray alone up to the next one.  trace_rays_kernel steps every ray with the
same schedule in a plain loop, so on the same rays both kernels move through bit-identical states: the fused map's
counters must equal what the staged path saw, exactly, and T_b must agree within the usual 1e-4.

* valid_samples == the valid records of trace -> sample_traced;
* active_ray_steps == the moved steps trace reports (each ray counts the steps before it froze);
* pencil_steps: every step a ray moved in cumulative mode, every recorded one in per-step mode;
* T_b and V/I within 1e-4 of trace -> sample_traced -> emission_traced.

The cases: stride 1, n_steps not a multiple of the stride, a stride longer than the whole run, rays that leave the
cube (and freeze) inside an interval, rays and a whole warp that start outside the cube, cumulative S, the FP64
stepper (a step longer than 8 cells) and a diagnostic kernel, whose T_b must be the plain kernel's bit for bit.
"""
import numpy as np
import pytest

from raytracinggrff_b200 import synthetic

pytestmark = pytest.mark.gpu

R_SUN_CM = 6.957e10
N_PIX, X_FOV, Z_OBS = 32, 1.44, 3.0


@pytest.fixture(scope="module")
def cube():
    return synthetic.corona_cube(64, 3.0)


def _rays():
    """Config-3 geometry on a 32^2 map; the first warp (rays 0-31) and a few single rays start outside the cube."""
    xs, ys, zs, kv = synthetic.ray_launch_geometry(N_PIX, X_FOV, Z_OBS)
    zs = zs.copy()
    xs = xs.copy()
    zs[:32] = 3.3
    xs[[100, 333, 517, 900]] = 3.2
    return xs, ys, zs, kv


def _both(session, c, freq, dt, n_steps, stride, s_mode="per_step"):
    g = (c["x_grid"], c["y_grid"], c["z_grid"])
    session.set_omega_cube(c["omega_pe"], *g)
    session.set_field_cubes(*g, c["ne"], c["te"], c["b"])
    xs, ys, zs, kv = _rays()
    area = (2 * X_FOV / N_PIX * R_SUN_CM) ** 2
    _, _, active = session.trace(freq, xs, ys, zs, kv, dt, n_steps, stride, True, 2.0, s_mode=s_mode, fetch=False)
    smp = session.sample_traced(np.column_stack([xs, ys, zs]), R_SUN_CM)
    tb_s, vi_s = session.emission_traced(area, freq)
    fp = [(freq, dt, n_steps, stride)]
    tb, vi, st = session.render_map(xs, ys, zs, fp, kvec_in_norm=kv, pixel_area_cm2=area, s_mode=s_mode)
    return dict(active=active, valid=int(smp["valid_mask"].sum()), tb_s=tb_s[:, 0], vi_s=vi_s[:, 0], tb=tb[0],
                vi=vi[0], st=st, rays=(xs, ys, zs, kv), fp=fp, area=area, stride=stride, s_mode=s_mode)


def _check(r, n_steps):
    st = r["st"]
    assert st["nominal_ray_steps"] == n_steps * N_PIX * N_PIX
    assert st["active_ray_steps"] == r["active"]
    assert st["valid_samples"] == r["valid"]
    act, pen = st["active_ray_steps"], st["pencil_steps"]
    assert 0 < act < st["nominal_ray_steps"]
    if r["s_mode"] == "cumulative":
        assert pen == act
    else:       # the sum over the rays of ceil(moved steps / stride)
        assert act / r["stride"] <= pen <= act / r["stride"] + N_PIX * N_PIX
    assert np.array_equal(r["tb"] == 0, r["tb_s"] == 0)
    np.testing.assert_allclose(r["tb"], r["tb_s"], rtol=1e-4)
    np.testing.assert_allclose(r["vi"], r["vi_s"], atol=1e-4)
    # the rays that start outside the cube never move and leave T_b = 0
    assert (r["tb"][:32] == 0).all() and (r["tb"][[100, 333, 517, 900]] == 0).all()
    assert (r["tb"][32:] > 0).mean() > 0.5


@pytest.mark.parametrize("n_steps, stride", [(3000, 1), (3001, 7), (3000, 10), (1200, 5000)],
                         ids=["stride1", "partial_last_interval", "config3_stride", "stride_longer_than_run"])
def test_counters_and_map_equal_the_staged_path(session, cube, n_steps, stride):
    r = _both(session, cube, 75e6, 6e-3, n_steps, stride)
    _check(r, n_steps)
    if stride > n_steps:
        assert r["valid"] <= N_PIX * N_PIX          # one record per ray: step 0
    elif stride > 1:
        # most rays leave the cube inside the run, and so (with stride > 1) mostly inside an interval
        xs, ys, zs, kv = r["rays"]
        rec, _, _ = session.trace(75e6, xs, ys, zs, kv, 6e-3, n_steps, stride, True, 2.0)
        frozen = np.all(rec[-1] == rec[-2], axis=1)
        assert frozen.mean() > 0.3, frozen.mean()


def test_cumulative_s(session, cube):
    _check(_both(session, cube, 75e6, 6e-3, 3001, 7, s_mode="cumulative"), 3001)


def test_fp64_stepper(session, cube):
    """dt = 0.7: a step plus the pencil offset spans 9.5 cells of the 64^3 cube, so both paths run the FP64
    stepper (trace_rays_kernel / render_map_kernel with MODE_F64)."""
    cells = 3 * 0.7 * (2.998e10 / 6.96e10) * (len(cube["x_grid"]) - 1) / 6.0
    assert cells > 8.0
    r = _both(session, cube, 75e6, 0.7, 31, 4)
    _check(r, 31)


def test_diag_kernel_keeps_the_plain_map(session, cube):
    """theta = 90 deg: the diagnostic kernel's T_b and V/I are the plain kernel's bit for bit, with the same counters."""
    r = _both(session, cube, 75e6, 6e-3, 3001, 7)
    xs, ys, zs, kv = r["rays"]
    tb, vi, st, dg = session.render_map_diag(xs, ys, zs, r["fp"], kvec_in_norm=kv, pixel_area_cm2=r["area"])
    assert np.array_equal(tb[0], r["tb"])
    assert np.array_equal(vi[0], r["vi"], equal_nan=True)
    assert st == r["st"]
    lit = tb[0] > 0
    assert np.isfinite(dg["em_z"][0][lit]).all()
