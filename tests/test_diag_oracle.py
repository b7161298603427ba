"""CPU: the oracle of the map diagnostics (tests/native/oracle_diag.c, oracle_get_mw_diag) against hand-computed
lines of sight, its RL against oracle_get_mw bit for bit, and the diagnostics switch of the workflow."""
import numpy as np
import pytest

import diag_oracle
import grff_checks as gc

NU = 150e6


def _kappa_ff_b0(T, ne, nu):
    """Free-free opacity at B = 0 (n^2 = 1 - v) as oracle_grff.c defines it."""
    v = gc.E ** 2 * ne / (np.pi * gc.ME) / nu ** 2
    return gc.KFF * ne * ne * gc.ZETA * gc.lnL(T, nu) / (np.sqrt(1 - v) * nu * nu * T * np.sqrt(T)), 1 - v


def _line(vox, flag=5):
    """vox: list of (dz, T, ne, B, theta, (x, y, z)) from the far end to the observer."""
    nz = len(vox)
    P = np.zeros((15, nz), order="F")
    C = np.zeros((4, nz), order="F")
    for k, (dz, T, ne, B, th, xyz) in enumerate(vox):
        P[0, k], P[1, k], P[2, k], P[3, k], P[4, k] = dz, T, ne, B, th
        C[:3, k] = xyz
        C[3, k] = np.linalg.norm(xyz)
    P[6], P[7] = flag, 30
    return diag_oracle.get_mw_diag(np.array([nz, 1, 0, 0, 0], np.int32), np.array([gc.AREA, NU, 0.0]), P, C)


def test_one_uniform_voxel():
    dz, T, ne, xyz = 3e9, 1.5e6, 3e7, (0.3, -0.2, 1.1)
    RL, d = _line([(dz, T, ne, 0.0, 90.0, xyz)])
    np.testing.assert_allclose(d[:3, 0], xyz, rtol=1e-14)
    np.testing.assert_allclose(d[3, 0], np.linalg.norm(xyz), rtol=1e-14)
    kap, _ = _kappa_ff_b0(T, ne, NU)
    np.testing.assert_allclose(d[4:, 0], [kap * dz, kap * dz], rtol=1e-12)
    assert RL[5, 0] > 0


def test_two_voxels_hand_computed_weights():
    far = (4e9, 2e6, 5e7, 0.0, 90.0, (0.1, 0.2, 0.5))
    near = (2e9, 1e6, 2e7, 0.0, 90.0, (0.1, 0.2, 1.5))
    RL, d = _line([far, near])
    src = []
    tau = []
    for dz, T, ne, *_ in (far, near):
        kap, n2 = _kappa_ff_b0(T, ne, NU)
        tau.append(kap * dz)
        src.append(n2 * NU ** 2 * gc.KB * T / gc.C ** 2)
    w_far = np.exp(-tau[1]) * src[0] * (-np.expm1(-tau[0]))
    w_near = src[1] * (-np.expm1(-tau[1]))
    cf, cn = np.array(far[5]), np.array(near[5])
    np.testing.assert_allclose(d[:3, 0], (w_far * cf + w_near * cn) / (w_far + w_near), rtol=1e-12)
    r = (w_far * np.linalg.norm(cf) + w_near * np.linalg.norm(cn)) / (w_far + w_near)
    np.testing.assert_allclose(d[3, 0], r, rtol=1e-12)
    np.testing.assert_allclose(d[4:, 0], [sum(tau)] * 2, rtol=1e-12)
    # the weights are the contributions to I_L + I_R: their sum is the intensity (two equal slots at B = 0)
    to_sfu = gc.AREA / gc.AU ** 2 / 1e-19
    np.testing.assert_allclose(RL[5, 0] + RL[6, 0], 2 * (w_far + w_near) * to_sfu, rtol=1e-12)


def test_evanescent_mode_is_infinite_depth():
    # the far voxel is above the plasma frequency (v > 1): both modes cut off, the intensity behind it is reset
    ne_cut = 2.0 * np.pi * gc.ME * NU ** 2 / gc.E ** 2
    cut = (1e9, 1e6, ne_cut, 0.0, 90.0, (0.0, 0.0, 1.0))
    emit = (2e9, 1e6, 1e7, 0.0, 90.0, (0.0, 0.0, 2.0))
    _, d = _line([cut, emit])
    assert np.isinf(d[4, 0]) and np.isinf(d[5, 0]) and d[4, 0] > 0
    np.testing.assert_allclose(d[:3, 0], emit[5], rtol=1e-14)
    _, d = _line([cut])
    assert np.isinf(d[4:, 0]).all() and np.isnan(d[:4, 0]).all()


@pytest.mark.parametrize("flag", [4, 5])
def test_rl_bit_identical_to_get_mw(oracle, flag):
    rng = np.random.default_rng(7 + flag)
    npix, nz = 48, 40
    P_M = gc.random_los_batch(rng, npix, nz, with_b=True, flag=flag, theta90=False)
    n_qt = 0
    for p in range(npix):
        P = np.asfortranarray(P_M[:, :, p])
        cnt = int((P[0] > 0).sum())
        C = np.zeros((4, nz), order="F")
        C[:3, :cnt] = rng.uniform(-2, 2, (3, cnt))
        C[3] = np.linalg.norm(C[:3], axis=0)
        L = np.array([nz, 3, 0, 0, 0], np.int32)
        R = np.array([gc.AREA, 1e8, 0.5])
        RL_ref = np.zeros((7, 3), order="F")
        oracle.get_mw(L, R, P, None, None, None, RL_ref)
        RL, d = diag_oracle.get_mw_diag(L, R, P, C)
        assert np.array_equal(RL, RL_ref), p
        th = P[4, :cnt]
        n_qt += int(np.any(np.diff(np.sign(np.cos(np.radians(th)))) != 0))
        if cnt == 0:
            assert np.isnan(d[:4]).all() and (d[4:] == 0).all()
            continue
        assert (d[4:] >= 0).all()
        # the centroid lies in the convex hull of the path's coordinates (here: inside its bounding box)
        for f in range(3):
            if np.isfinite(d[0, f]):
                for q in range(4):
                    assert C[q, :cnt].min() - 1e-12 <= d[q, f] <= C[q, :cnt].max() + 1e-12
    assert n_qt > 0


def test_ray_r_min_skips_non_finite_records():
    r = np.array([[[0.0, 0.0, 3.0], [np.nan, 0, 0]], [[0.0, 1.2, 0.5], [np.nan, 0, 0]]])
    out = diag_oracle.ray_r_min(r)
    np.testing.assert_allclose(out[0], np.float32(np.hypot(1.2, 0.5)), rtol=1e-6)
    assert np.isnan(out[1])


@pytest.mark.parametrize("backend", ["get_mw", "fastgrff", "device"])
def test_diagnostics_need_the_fused_backend(backend):
    from raytracinggrff_b200 import workflow
    with pytest.raises(ValueError, match="fused"):
        workflow.run_ray_tracing_emission({}, grff_backend=backend, diagnostics=True)


def test_diagnostic_maps_layout():
    from raytracinggrff_b200 import workflow
    n, nf = 3, 2
    diag = {k: np.arange(nf * n * n, dtype=float).reshape(nf, n * n) + 100 * q
            for q, k in enumerate(("em_x", "em_y", "em_z", "em_r", "tau_L", "tau_R", "ray_r_min"))}
    m = workflow.diagnostic_maps(diag, n)
    assert m["emission_centroid_xyz"].shape == (n, n, nf, 3)
    for k in ("emission_r_mean", "tau_L", "tau_R", "ray_r_min"):
        assert m[k].shape == (n, n, nf)
    # pixel (i, j) is ray i*n + j, as in emission_cube
    i, j, f = 2, 1, 1
    assert m["emission_centroid_xyz"][i, j, f, 2] == diag["em_z"][f, i * n + j]
    assert m["ray_r_min"][i, j, f] == diag["ray_r_min"][f, i * n + j]
