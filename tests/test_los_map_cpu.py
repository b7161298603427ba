"""CPU: the argument checks of los.render_los_map (raised before any GPU work) and the theta-from-B restatement of
tests/los_map_oracle.py on hand-computed fields."""
import numpy as np
import pytest

import los_map_oracle as lmo
from raytracinggrff_b200 import los, synthetic


@pytest.fixture(scope="module")
def model():
    return synthetic.spherical_corona(16, 12, 16, r_max=4.0)


def _call(model, **kw):
    a = dict(N_pix=8, X_range=(-1.4, 1.4), Y_range=(-1.4, 1.4), N_z=20, dz0=1e-3, freq0=1e8, Nfreq=2, freq_log_step=0.1)
    a.update(kw)
    return los.render_los_map(model, **a)


def test_argument_errors_come_before_the_gpu(model):
    with pytest.raises(ValueError, match="extremely large"):
        _call(model, dz0=7e4)
    with pytest.raises(ValueError, match="electron temperature"):
        _call({k: v for k, v in model.items() if k != "te"})
    for b in ("br", "bt", "bp"):
        with pytest.raises(ValueError, match="Magnetic field components"):
            _call({k: v for k, v in model.items() if k != b})
    with pytest.raises(ValueError, match="N_pix"):
        _call(model, N_pix=1)
    with pytest.raises(ValueError, match="Nfreq"):
        _call(model, Nfreq=0)


def test_theta_from_b_on_hand_computed_fields():
    # on the cube's +x axis the model frame is (x, -z, y) = (2, 0, 0): r along model x, theta (from model z = cube y)
    # points to -cube y, phi to -cube z
    x, y, z = 2.0, 0.0, 0.0
    th, (bx, by, bz) = lmo.bvec_theta_deg(x, y, z, 0.0, 0.0, -1.0)       # B = +z: along the propagation
    assert np.allclose([bx, by, bz], [0, 0, 1]) and th == pytest.approx(0.0)
    th, (bx, by, bz) = lmo.bvec_theta_deg(x, y, z, 0.0, 0.0, 1.0)        # B = -z: against it
    assert np.allclose([bx, by, bz], [0, 0, -1]) and th == pytest.approx(180.0)
    th, (bx, by, bz) = lmo.bvec_theta_deg(x, y, z, 0.0, -1.0, 0.0)       # B = +y: transverse
    assert np.allclose([bx, by, bz], [0, 1, 0]) and th == pytest.approx(90.0)
    th, (bx, by, bz) = lmo.bvec_theta_deg(x, y, z, 1.0, 0.0, -1.0)       # radial + z: 45 deg
    assert np.allclose([bx, by, bz], [1, 0, 1]) and th == pytest.approx(45.0)
    assert lmo.bvec_theta_deg(x, y, z, 0.0, 0.0, 0.0)[0] == 90.0        # no field: the reference's 90 deg
    # a uniform field along +z seen from anywhere: the spherical components of (0, 0, 1) at each point
    rng = np.random.default_rng(1)
    p = rng.uniform(-2, 2, size=(3, 50))
    cx, cy, cz = p[0], -p[2], p[1]
    rr, rho = np.sqrt(cx ** 2 + cy ** 2 + cz ** 2), np.sqrt(cx ** 2 + cy ** 2)
    m = np.array([0.0, -1.0, 0.0])       # cube +z = model -y
    er = np.stack([cx, cy, cz]) / rr
    et = np.stack([cz * cx / rho, cz * cy / rho, -rho]) / rr
    ep = np.stack([-cy, cx, np.zeros_like(cx)]) / rho
    br, bt, bp = (m @ e for e in (er, et, ep))
    th = lmo.bvec_theta_deg(p[0], p[1], p[2], br, bt, bp)[0]
    np.testing.assert_allclose(th, 0.0, atol=1e-5)
