"""Parity on the configurations bench.py times (run on the B200 box: ``pytest -m gpu``).

The benchmarked kernel variant — cross-sections on, record order, theta from the B vector, gyroresonance +
free-free (``trace_crosssections=True, em_flag=4, use_bvec=True``) — through exactly the call bench.py makes,
at full image size, against the oracle chain (ray_trace -> sampler -> Parms with theta from B.d -> GET_MW,
``oracle.chain_bvec``) on a pixel sub-sample:

* BASELINE config 4: 512^2 pixels, 256^3 cube, all 8 frequencies 75 MHz - 1.5 GHz, every 16th pixel;
* BASELINE config 5: 2048^2 pixels, 512^3 cube built on the GPU from the spherical model (as bench.py does),
  all 16 frequencies 20 - 300 MHz with the low-band presets, every 64th pixel.

Tolerances: paths <= 1e-5 R_sun, T_b <= 1e-4 relative, V/I <= 1e-4 absolute.  Pixels whose ray grazes the
r = 1 density discontinuity are chaotic (oracle/parity.py): only rays that reach it may breach, and the share
that does is bounded (measured on config 4: 40 of 8192 pixel-frequencies, 0.5 %).
"""
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

import bench  # noqa: E402  (workload definitions: the same tables the benchmark runs)
from raytracinggrff_b200 import synthetic  # noqa: E402

pytestmark = pytest.mark.gpu


def _render_full(session, w, fps, area):
    xs, ys, zs = bench.rays_of(w)
    tb, vi, st = session.render_map(xs, ys, zs, fps, trace_crosssections=True, perturb_ratio=2.0, pixel_area_cm2=area,
                                    r_sun_cm=6.957e10, em_flag=4, s_max=30, use_bvec=True,
                                    image_shape=(w["n_pix_y"], w["n_pix_x"]))
    return xs, ys, zs, tb, vi, st


def _assert_parity(par, max_chaotic_frac):
    """Every pixel whose ray stays clear of the r = 1 density discontinuity is within the tolerances; of the rays
    that reach it (at GHz frequencies: the whole disc) only the grazing ones are chaotic — a small, bounded share."""
    msg = {k: v for k, v in par.items() if k != "per_freq"}
    assert par["n_pixel_freqs_over_tol"] == 0, (msg, par["per_freq"])
    assert par["max_dr_rsun"] <= 1e-5 and par["max_rel_dTb"] <= 1e-4 and par["max_dVI"] <= 1e-4, msg
    assert par["n_diving_over_tol"] <= max_chaotic_frac * par["n_pixels"] * par["n_freq"], msg
    print("parity:", msg)
    for row in par["per_freq"]:
        print("  ", row)


def test_config4_bench_variant_matches_oracle_chain(oracle, session):
    from oracle import parity
    w = bench.workload("c4", 1)
    c = synthetic.corona_cube(w["grid_n"], w["extent"], active_region=True)
    g3 = (c["x_grid"], c["y_grid"], c["z_grid"])
    session.set_omega_cube(c["omega_pe"], *g3)
    session.set_field_cubes(*g3, c["ne"], c["te"], c["b"], c["bx"], c["by"], c["bz"])
    fps = w["freq_params"]
    area = bench.pixel_area(w)
    xs, ys, zs, tb, vi, st = _render_full(session, w, fps, area)
    assert st["nominal_ray_steps"] == 512 * 512 * sum(p["n_steps"] for p in fps)
    sel = parity.subsample(512, 512, 16)
    # the oracle samples the float32 field cubes the device holds (gpu_raytrace.py:647-649 casts them too)
    par = parity.map_parity(c, fps, xs[sel], ys[sel], zs[sel], area, tb[:, sel], vi[:, sel], session=session)
    assert par["n_pixels"] == 1024 and par["n_freq"] == 8
    # gyroresonance must matter somewhere on this cube (active region, GHz frequencies)
    assert max(r["max_abs_vi"] for r in par["per_freq"]) > 1e-3
    _assert_parity(par, max_chaotic_frac=0.01)


def test_bench_dump_outputs_are_the_timed_maps(session, tmp_path):
    """bench.py --dump-outputs writes its last timed step's maps: the T_b and V/I that render_map returns for the
    same workload (config 3, whole map), bit for bit."""
    import subprocess
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--config", "c3", "--steps", "2", "--warmup", "0",
                        "--no-cpu-baseline", "--no-extras", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    w = bench.workload("c3", 1)
    c = bench.host_cube(w)
    g3 = (c["x_grid"], c["y_grid"], c["z_grid"])
    session.set_omega_cube(c["omega_pe"], *g3)
    session.set_field_cubes(*g3, c["ne"], c["te"], c["b"], c["bx"], c["by"], c["bz"])
    _, _, _, tb, vi, _ = _render_full(session, w, w["freq_params"], bench.pixel_area(w))
    assert sorted(f.name for f in tmp_path.iterdir()) == ["tb.npy", "vi.npy"]
    shape = (w["n_freq"], w["n_pix_y"], w["n_pix_x"])
    np.testing.assert_array_equal(np.load(tmp_path / "tb.npy"), tb.reshape(shape))
    np.testing.assert_array_equal(np.load(tmp_path / "vi.npy"), vi.reshape(shape))


def test_config5_bench_variant_matches_oracle_chain(oracle, session):
    from oracle import parity
    w = bench.workload("c5", 8)
    model = synthetic.spherical_corona(200, 140, 160, r_max=1.8 * w["extent"], active_region=True)
    g = np.linspace(-w["extent"], w["extent"], w["grid_n"])
    session.set_model_from_spherical(model, g, g.copy(), g.copy(), phi0_offset=0.0, want_bvec=True)
    c = session.export_cubes(omega_pe=True, fields=True, bvec=True)
    c.update(x_grid=g, y_grid=g.copy(), z_grid=g.copy())
    assert c["omega_pe"].shape == (512, 512, 512) and np.isfinite(c["omega_pe"]).all()
    fps = w["freq_params"]
    area = bench.pixel_area(w)
    xs, ys, zs = bench.rays_of(w)
    sel = parity.subsample(2048, 2048, 64)
    # the full 2048^2 x 16-frequency map on one GPU takes ~7 s; the sub-sampled pixels are rendered through
    # the same kernel variant with the full image's tiling being irrelevant to the result (bit-identical:
    # test_render_map_properties_at_full_config4_size)
    tb, vi, st = session.render_map(xs[sel], ys[sel], zs[sel], fps, trace_crosssections=True, perturb_ratio=2.0,
                                    pixel_area_cm2=area, r_sun_cm=6.957e10, em_flag=4, s_max=30, use_bvec=True)
    par = parity.map_parity(c, fps, xs[sel], ys[sel], zs[sel], area, tb, vi, session=session)
    assert par["n_pixels"] == 1024 and par["n_freq"] == 16
    _assert_parity(par, max_chaotic_frac=0.01)
    # steps longer than a cell at the lowest frequencies (1.1 cells + pencil): still the FP32 stepper
    assert fps[0]["dt"] * (2.998e10 / 6.96e10) * 3 / (g[1] - g[0]) > 1.0
