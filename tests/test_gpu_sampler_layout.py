"""The field nodes' two layouts on the device: {n_e, T, |B|, 0} (16 bytes) without a B-vector cube, and
{n_e, T, |B|, 0, B_x, B_y, B_z, 0} (32 bytes, one load per trilinear corner) with one.  The layout is internal to
the context: every reader of n_e / T / |B| must return the same bits from either, `export_cubes` must give back what
was stored, and switching between the layouts must not change what is sampled.  The theta-from-B map, the one
reader of the 32-byte nodes' vector half, is held to the CPU oracle chain as in test_gpu_bench_parity.py.

A config-4-like workload at a small size: 64^3 active-region cube, 48^2 pixels, config 4's lowest and highest
frequency presets."""
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

import bench  # noqa: E402  (config 4's frequency presets)
from raytracinggrff_b200 import RaySession, synthetic  # noqa: E402

pytestmark = pytest.mark.gpu

N_PIX, X_FOV, Z_OBS = 48, 1.44, 3.0
MAP_KW = dict(trace_crosssections=True, perturb_ratio=2.0, r_sun_cm=6.957e10, em_flag=4, s_max=30,
              image_shape=(N_PIX, N_PIX))


@pytest.fixture(scope="module")
def cube():
    return synthetic.corona_cube(64, 3.0, active_region=True)


@pytest.fixture(scope="module")
def rays():
    xs, ys, zs, kv = synthetic.ray_launch_geometry(N_PIX, X_FOV, Z_OBS)
    return xs, ys, zs, kv


@pytest.fixture(scope="module")
def freqs():
    fps = bench.workload("c4", 1)["freq_params"]
    return [fps[0], fps[-1]]


def _grids(c):
    return c["x_grid"], c["y_grid"], c["z_grid"]


def _session(c, bvec):
    s = RaySession(0)
    s.set_omega_cube(c["omega_pe"], *_grids(c))
    vec = (c["bx"], c["by"], c["bz"]) if bvec else ()
    s.set_field_cubes(*_grids(c), c["ne"], c["te"], c["b"], *vec)
    return s


def _area():
    return (2 * X_FOV / N_PIX * 6.957e10) ** 2


def _sample_traced(s, rays, fp):
    xs, ys, zs, kv = rays
    s.trace(fp["freq_hz"], xs, ys, zs, kv, fp["dt"], fp["n_steps"], fp["record_stride"], True, 2.0)
    return s.sample_traced(np.column_stack([xs, ys, zs]), 6.957e10)


def _assert_same_samples(a, b):
    for k in ("ne", "te", "b", "ds", "s", "valid_mask"):
        assert np.array_equal(a[k], b[k], equal_nan=True), k


def test_plain_map_is_the_same_from_16_and_32_byte_nodes(cube, rays, freqs):
    xs, ys, zs, _ = rays
    with _session(cube, bvec=True) as s32, _session(cube, bvec=False) as s16:
        for order in (0, 1):
            tb32, vi32, _ = s32.render_map(xs, ys, zs, freqs, pixel_area_cm2=_area(), use_bvec=False, voxel_order=order,
                                           **MAP_KW)
            tb16, vi16, _ = s16.render_map(xs, ys, zs, freqs, pixel_area_cm2=_area(), use_bvec=False, voxel_order=order,
                                           **MAP_KW)
            assert np.count_nonzero(tb16) > tb16.size // 4
            assert np.array_equal(tb32, tb16) and np.array_equal(vi32, vi16), order


def test_staged_sampler_is_the_same_from_16_and_32_byte_nodes(cube, rays, freqs):
    with _session(cube, bvec=True) as s32, _session(cube, bvec=False) as s16:
        a, b = _sample_traced(s32, rays, freqs[0]), _sample_traced(s16, rays, freqs[0])
        assert a["valid_mask"].any()
        _assert_same_samples(a, b)
        # the host-array sampler (rtgrff_sample) reads the same nodes
        r, sv, _ = s16.trace(freqs[0]["freq_hz"], *rays, freqs[0]["dt"], freqs[0]["n_steps"],
                             freqs[0]["record_stride"], True, 2.0)
        start = np.column_stack(rays[:3])
        _assert_same_samples(s32.sample(r, sv, start, 6.957e10), s16.sample(r, sv, start, 6.957e10))


def test_export_round_trip_and_layout_switch(cube, rays, freqs):
    c = cube
    f32 = {k: np.asarray(c[k], dtype=np.float32) for k in ("ne", "te", "b", "bx", "by", "bz")}
    with _session(c, bvec=True) as s:
        got = s.export_cubes(omega_pe=False, fields=True, bvec=True)
        for k in f32:
            assert np.array_equal(got[k], f32[k]), k
        before = _sample_traced(s, rays, freqs[0])
        # the same fields without the vector: back to 16-byte nodes, the same values sampled
        s.set_field_cubes(*_grids(c), c["ne"], c["te"], c["b"])
        after = _sample_traced(s, rays, freqs[0])
        _assert_same_samples(before, after)
        got = s.export_cubes(omega_pe=False, fields=True, bvec=False)
        for k in ("ne", "te", "b"):
            assert np.array_equal(got[k], f32[k]), k
        with pytest.raises(Exception):
            s.export_cubes(omega_pe=False, fields=False, bvec=True)
        with pytest.raises(Exception):
            s.render_map(*rays[:3], freqs[:1], pixel_area_cm2=_area(), use_bvec=True, **MAP_KW)
        # and to 32-byte nodes again
        s.set_field_cubes(*_grids(c), c["ne"], c["te"], c["b"], c["bx"], c["by"], c["bz"])
        _assert_same_samples(before, _sample_traced(s, rays, freqs[0]))


def test_spherical_model_cubes_round_trip(rays, freqs):
    """compose_cubes_kernel writes the 32-byte nodes; uploading what export_cubes returns through
    set_field_cubes gives the same nodes: the same exported values and the same theta-from-B map, bit for bit."""
    model = synthetic.spherical_corona(60, 40, 48, r_max=6.0, active_region=True)
    g = np.linspace(-3.0, 3.0, 64)
    xs, ys, zs, _ = rays
    with RaySession(0) as sph, RaySession(0) as up, RaySession(0) as plain:
        sph.set_model_from_spherical(model, g, g.copy(), g.copy(), want_bvec=True)
        got = sph.export_cubes(omega_pe=True, fields=True, bvec=True)
        plain.set_model_from_spherical(model, g, g.copy(), g.copy(), want_bvec=False)
        got16 = plain.export_cubes(omega_pe=True, fields=True, bvec=False)
        for k in ("omega_pe", "ne", "te", "b"):
            assert np.array_equal(got[k], got16[k]), k
        assert np.abs(got["bz"]).max() > 0
        up.set_omega_cube(got["omega_pe"], g, g.copy(), g.copy())
        up.set_field_cubes(g, g.copy(), g.copy(), got["ne"], got["te"], got["b"], got["bx"], got["by"], got["bz"])
        again = up.export_cubes(omega_pe=False, fields=True, bvec=True)
        for k in ("ne", "te", "b", "bx", "by", "bz"):
            assert np.array_equal(again[k], got[k]), k
        tb_a, vi_a, _ = sph.render_map(xs, ys, zs, freqs, pixel_area_cm2=_area(), use_bvec=True, **MAP_KW)
        tb_b, vi_b, _ = up.render_map(xs, ys, zs, freqs, pixel_area_cm2=_area(), use_bvec=True, **MAP_KW)
        assert np.array_equal(tb_a, tb_b) and np.array_equal(vi_a, vi_b)


def test_bvec_map_matches_oracle_chain(oracle, cube, rays, freqs):
    from oracle import parity
    xs, ys, zs, _ = rays
    sel = parity.subsample(N_PIX, N_PIX, 6)
    with _session(cube, bvec=True) as s:
        tb, vi, _ = s.render_map(xs, ys, zs, freqs, pixel_area_cm2=_area(), use_bvec=True, **MAP_KW)
        par = parity.map_parity(cube, freqs, xs[sel], ys[sel], zs[sel], _area(), tb[:, sel], vi[:, sel], session=s)
    msg = {k: v for k, v in par.items() if k != "per_freq"}
    assert par["n_pixels"] == 64 and par["n_freq"] == 2
    assert par["n_pixel_freqs_over_tol"] == 0, (msg, par["per_freq"])
    assert par["max_dr_rsun"] <= 1e-5 and par["max_rel_dTb"] <= 1e-4 and par["max_dVI"] <= 1e-4, msg
    assert par["n_diving_over_tol"] <= 0.01 * par["n_pixels"] * par["n_freq"], msg
