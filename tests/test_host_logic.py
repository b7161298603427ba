"""CPU: host-side logic, the C-ABI surface and the drop-in error behaviour (no GPU compute)."""
import ctypes
import re
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]


def test_library_loads_and_exports_every_declared_symbol():
    from raytracinggrff_b200 import _lib
    from raytracinggrff_b200.build import build_library
    build_library()
    header = (ROOT / "include" / "rtgrff.h").read_text()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(rtgrff_[a-z_0-9]+|PyGET_MW)\s*\(", header))
    declared -= {"rtgrff_ctx", "rtgrff_freq_params"}
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    lib = ctypes.CDLL(str(_lib.LIB_PATH))
    for name in declared:
        assert hasattr(lib, name), name
    assert b"sm_100a" in _lib.load().rtgrff_version()


def test_sass_is_sm100a_only():
    import subprocess
    from raytracinggrff_b200 import _lib
    from raytracinggrff_b200.build import cuda_tool
    cuobjdump = cuda_tool("cuobjdump")
    if not Path(cuobjdump).exists():
        pytest.skip("cuobjdump not found")
    out = subprocess.run([cuobjdump, "-lelf", str(_lib.LIB_PATH)], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_no_cpu_fallback_and_device_strings():
    import raytracinggrff_b200 as pkg
    from raytracinggrff_b200.workflow import run_ray_tracing_emission
    g = np.linspace(-1, 1, 5)
    w = np.zeros((5, 5, 5))
    z3 = np.zeros(3)
    with pytest.raises(ValueError, match="Unsupported device 'tpu'"):
        pkg.trace_ray("tpu", w, g, g, g, 1e8, z3, z3, z3, np.zeros((3, 3)), 1e-3, 10)
    with pytest.raises(ValueError, match="Unsupported device"):
        pkg.sample_model_with_rays("opencl", g, g, g, w, w, w, np.zeros((2, 3, 3)), np.ones((2, 3)), np.zeros((3, 3)), 1.0)
    with pytest.raises(RuntimeError, match="CUDA-only"):
        pkg.trace_ray("CPU", w, g, g, g, 1e8, z3, z3, z3, np.zeros((3, 3)), 1e-3, 10)
    with pytest.raises(RuntimeError, match="CUDA-only"):
        pkg.sample_model_with_rays("cpu", g, g, g, w, w, w, np.zeros((2, 3, 3)), np.ones((2, 3)), np.zeros((3, 3)), 1.0)
    with pytest.raises(ValueError, match="grff_backend"):
        run_ray_tracing_emission({}, grff_backend="idl")
    with pytest.raises(RuntimeError, match="CUDA-only"):
        run_ray_tracing_emission({}, device="cpu")


def test_product_never_imports_the_oracle():
    for p in (ROOT / "raytracinggrff_b200").rglob("*.py"):
        src = p.read_text()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), p
        assert "liboracle" not in src, p
    for p in (ROOT / "raytracinggrff_b200" / "csrc").glob("*"):
        assert "oracle_" not in p.read_text().replace("oracle/oracle_", ""), p


def test_check_uniform_grid_matches_reference_rules(oracle):
    from raytracinggrff_b200._lib import check_uniform_grid, grid_geom
    g = np.linspace(-3, 3, 128)
    assert check_uniform_grid(g, "x_grid") == oracle.check_uniform_grid(g, "x_grid")
    g32 = np.linspace(-2.0, 2.0, 128, dtype=np.float32)
    assert check_uniform_grid(g32, "x_grid") == oracle.check_uniform_grid(g32, "x_grid")
    for bad, msg in ((np.zeros((2, 2)), "1D"), (np.array([1.0]), "at least 2"), (np.array([0.0, 0.0, 0.0]), "invalid spacing"),
                     (np.array([2.0, 1.0, 0.0]), "invalid spacing"), (np.array([0.0, 1.0, 2.5]), "uniformly spaced")):
        with pytest.raises(ValueError, match=msg):
            check_uniform_grid(bad, "x_grid")
        with pytest.raises(ValueError, match=msg):
            oracle.check_uniform_grid(bad, "x_grid")
    geom = grid_geom(g, g, g32)
    assert geom.shape == (12,) and geom[0] == -3 and geom[2] == 3 and geom[3] == g[1] - g[0]


def test_launch_geometry_and_presets(oracle):
    from raytracinggrff_b200 import synthetic
    a = synthetic.ray_launch_geometry(64, 1.44, 3.0)
    b = oracle.ray_launch_geometry(64, 1.44, 3.0)
    for u, v in zip(a, b):
        np.testing.assert_array_equal(u, v)
    # ray p = i*N_pix + j  <->  x[j], y[i]   (script/resample_with_ray_tracing.py:298-300, :470)
    x = np.linspace(-1.44, 1.44, 64)
    assert a[0][5 * 64 + 7] == x[7] and a[1][5 * 64 + 7] == x[5]
    np.testing.assert_allclose(synthetic.log_frequencies(450e6, 4, 0.1), [450e6, 566.516e6, 713.202e6, 897.868e6], rtol=1e-5)
    p = synthetic.frequency_scaled_params(100e6)
    assert p == {"dt": 6e-3, "n_steps": 4000, "record_stride": 5}
    p = synthetic.frequency_scaled_params(25e6)
    assert p["dt"] == pytest.approx(12e-3) and p["n_steps"] == 2000 and p["record_stride"] == 10
    assert synthetic.frequency_scaled_params(1e6)["n_steps"] == 1200       # floor of the publication presets


def test_synthetic_corona_follows_reference_cube_rules():
    from raytracinggrff_b200 import synthetic
    c = synthetic.corona_cube(33, 3.0, active_region=True)
    r = np.sqrt(sum(np.square(np.meshgrid(c["x_grid"], c["y_grid"], c["z_grid"], indexing="ij"))))
    inside = r < synthetic.R_MIN
    assert inside.any()
    assert np.all(c["ne"][inside] == 0) and np.all(c["b"][inside] == 0) and np.all(c["te"][inside] == 1e4)
    assert np.all(c["omega_pe"][inside] == 0)
    np.testing.assert_allclose(c["omega_pe"], 2 * np.pi * 8.93e3 * np.sqrt(c["ne"]))
    np.testing.assert_allclose(c["b"], np.sqrt(c["bx"] ** 2 + c["by"] ** 2 + c["bz"] ** 2))
    assert np.all(np.isfinite(c["omega_pe"])) and c["ne"][~inside].min() > 1e4
    los = synthetic.straight_los_case(8, 50)
    assert los["Ne_LOS"].shape == (8, 8, 50) and los["ds_LOS"].min() > 0
    assert np.all(np.diff(los["z_coords"]) > 0)


def test_pack_parms_batch_matches_reference_loop(oracle):
    from raytracinggrff_b200.workflow import pack_parms_batch, pixel_area_cm2
    rng = np.random.default_rng(0)
    n_rec, n_rays = 23, 9
    smp = {k: rng.uniform(1, 2, (n_rec, n_rays)).astype(np.float32) for k in ("ne", "te", "b", "ds", "s")}
    smp["valid_mask"] = rng.random((n_rec, n_rays)) > 0.4
    smp["valid_mask"][:, 3] = False
    smp["ne"][2, 1] = np.nan
    area = pixel_area_cm2(1.44, 64)
    np.testing.assert_array_equal(pack_parms_batch(smp, area), oracle.pack_parms_batch(smp, area))
    assert pack_parms_batch(smp, area).flags.f_contiguous


def test_dlogS_ds_diagnostic():
    """script/pub/cross_section_plots.ipynb cell 12, restated inline."""
    from raytracinggrff_b200.util import dlogS_ds
    rng = np.random.default_rng(2)
    r = np.cumsum(rng.random((50, 4, 3)) * 0.01, axis=0)
    S = np.cumprod(1 + 0.01 * rng.standard_normal((50, 4)), axis=0)
    S[10, 1] = 0.001
    S[20:, 3] = np.nan
    got = dlogS_ds(r, S, distance_ray=0)
    Sm = S.copy()
    Sm[Sm < 0.01] = np.nan
    d = np.diff(np.log(Sm), axis=0)
    dist = np.concatenate([[0], np.cumsum(np.sqrt(np.sum(np.diff(r[:, 0, :], axis=0) ** 2, axis=1)))])
    ref = d / np.tile(np.diff(dist), (d.shape[1], 1)).T
    ref[np.isnan(ref)] = 0
    ref[np.isinf(ref)] = 0
    np.testing.assert_allclose(got, ref, rtol=1e-12)
    own = dlogS_ds(r, S)
    assert own.shape == (49, 4) and np.all(own[20:, 3] == 0) and own[9, 1] == 0 and own[10, 1] == 0
