"""Frequency-sweep driver (SURVEY.md §8f rank 2): one ray-traced T_b map per frequency with the
per-frequency grid / field-of-view / integrator presets of the reference's publication driver,
written as the same per-frequency ``.npz`` files and manifest, so the reference's plotting and
spectra scripts read them unchanged.

Reference: script/pub/TbSpectra_gen.py — presets ``select_params`` (:27-88), the loop (:139-192),
file naming (:143-145), manifest (:194-198); npz keys script/resample_with_ray_tracing.py:533-540.
There the cube is re-resampled from the MAS model through psipy for every frequency (the presets
change grid_n / extent per frequency); here that is `RaySession.set_model_from_spherical`
(milliseconds) followed by one fused `render_map` launch.
"""
from __future__ import annotations

import argparse
from pathlib import Path

import numpy as np

from . import synthetic
from .session import RaySession
from .workflow import R_sun_cm, R_sun_m, diagnostic_maps, pixel_area_cm2


def _lowband_params(freq_hz):
    """script/pub/TbSpectra_gen.py:27-44."""
    ref_freq_hz, base_dt, base_n_steps, base_record_stride = 100e6, 6e-3, 4000, 5
    scaling_exp, min_n_steps = 0.5, 1200
    scale = (ref_freq_hz / freq_hz) ** scaling_exp
    return {
        "grid_n": 256, "grid_extent": 4, "z_observer": 4, "x_fov": 2.8,
        "dt": base_dt * scale,
        "n_steps": max(min_n_steps, int(round(base_n_steps / max(scale, 1e-12)))),
        "record_stride": max(1, int(round(base_record_stride * scale))),
    }


def _interp_log_freq_params(freq_hz, f0_hz, p0, f1_hz, p1):
    """script/pub/TbSpectra_gen.py:47-53."""
    t = (np.log(freq_hz) - np.log(f0_hz)) / (np.log(f1_hz) - np.log(f0_hz))
    t = float(np.clip(t, 0.0, 1.0))
    return {k: (1.0 - t) * p0[k] + t * p1[k] for k in p0.keys()}


_HIGHBAND_ANCHORS = {   # script/pub/TbSpectra_gen.py:58-62
    280e6: {"grid_n": 400, "grid_extent": 1.75, "z_observer": 1.75, "x_fov": 1.44, "dt": 1.0e-3, "n_steps": 4500, "record_stride": 10},
    550e6: {"grid_n": 440, "grid_extent": 1.45, "z_observer": 1.45, "x_fov": 1.44, "dt": 0.8e-3, "n_steps": 7500, "record_stride": 5},
    800e6: {"grid_n": 520, "grid_extent": 1.45, "z_observer": 1.44, "x_fov": 1.44, "dt": 0.4e-3, "n_steps": 12000, "record_stride": 5},
}


def _round_ints(p):
    for k in ("grid_n", "n_steps", "record_stride"):
        p[k] = int(round(p[k]))
    return p


def _highband_params(freq_hz):
    """script/pub/TbSpectra_gen.py:56-70."""
    a = _HIGHBAND_ANCHORS
    if freq_hz <= 550e6:
        p = _interp_log_freq_params(freq_hz, 280e6, a[280e6], 550e6, a[550e6])
    else:
        p = _interp_log_freq_params(freq_hz, 550e6, a[550e6], 800e6, a[800e6])
    return _round_ints(p)


def select_params(freq_hz):
    """script/pub/TbSpectra_gen.py:73-88: low band <= 150 MHz, high band >= 280 MHz, log-frequency
    blend in between."""
    if freq_hz <= 150e6:
        return _lowband_params(freq_hz)
    if freq_hz >= 280e6:
        return _highband_params(freq_hz)
    return _round_ints(_interp_log_freq_params(freq_hz, 150e6, _lowband_params(150e6), 280e6, _highband_params(280e6)))


def tb_spectra(model, out_dir, N_pix=128, fmin_mhz=30.0, fmax_mhz=800.0, n_freq=30, start_from_idx=0,
               phi0_offset=-140.0, session=None, quiet=True, params_fn=select_params, use_bvec=False,
               em_flag=5, max_grid_n=None, diagnostics=False, b0_angle=0.0, p_angle=0.0):
    """Run the sweep.  `model` is a spherical model (cubes.SphericalVariable mapping).  Returns the
    manifest rows [(idx, freq_hz, npz_path)].  Existing files of indices < start_from_idx are kept
    (the reference's resume switch, :118-119, :141-142).  diagnostics=True: every npz also holds the keys of
    workflow.diagnostic_maps (emission centroid and height, optical depths, ray turning point), which over the
    sweep give the emission height against frequency.  b0_angle, p_angle [deg]: the observer's view of the model
    (include/rtgrff.h, "Observer view")."""
    from .cubes import check_view
    b0_angle, p_angle = check_view(b0_angle, p_angle)
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    freqs_hz = np.logspace(np.log10(fmin_mhz), np.log10(fmax_mhz), n_freq) * 1e6
    if start_from_idx < 0 or start_from_idx >= len(freqs_hz):
        raise ValueError(f"--start-from-idx must be in [0, {len(freqs_hz)-1}]")
    ses = session or RaySession()
    rows = []
    for i, freq_hz in enumerate(freqs_hz):
        tag = f"{i:02d}_{freq_hz/1e6:08.3f}MHz"
        npz_path = out_dir / f"raytrace_{tag}.npz"
        if i >= start_from_idx:
            p = params_fn(float(freq_hz))
            grid_n = int(p["grid_n"]) if max_grid_n is None else min(int(p["grid_n"]), int(max_grid_n))
            if not quiet:
                print(f"[{i+1:02d}/{len(freqs_hz)}] {freq_hz/1e6:8.3f} MHz | grid_n={grid_n} X_FOV={p['x_fov']:.3f} "
                      f"z_obs={p['z_observer']:.3f} dt={p['dt']:.3g} n_steps={p['n_steps']} stride={p['record_stride']}")
            g = np.linspace(-p["grid_extent"], p["grid_extent"], grid_n)       # script/...:263-265
            ses.set_model_from_spherical(model, g, g, g, phi0_offset=phi0_offset, want_bvec=use_bvec, b0_angle=b0_angle,
                                         p_angle=p_angle)
            xs, ys, zs, kv = synthetic.ray_launch_geometry(N_pix, float(p["x_fov"]), float(p["z_observer"]))
            area = pixel_area_cm2(float(p["x_fov"]), N_pix)
            render = ses.render_map_diag if diagnostics else ses.render_map
            out = render(xs, ys, zs, [(float(freq_hz), float(p["dt"]), int(p["n_steps"]), int(p["record_stride"]))],
                         kvec_in_norm=kv, trace_crosssections=True, perturb_ratio=2.0, pixel_area_cm2=area,
                         r_sun_cm=R_sun_cm, em_flag=em_flag, use_bvec=use_bvec, image_shape=(N_pix, N_pix))
            tb, vi = out[0], out[1]
            extra = diagnostic_maps(out[3], N_pix) if diagnostics else {}
            coords = np.linspace(-p["x_fov"], p["x_fov"], N_pix) * R_sun_m
            np.savez_compressed(npz_path,                                    # script/...:533-540
                                emission_cube=np.nan_to_num(tb[0].reshape(N_pix, N_pix, 1), nan=0.0, posinf=0.0, neginf=0.0),
                                emission_polVI_cube=vi[0].reshape(N_pix, N_pix, 1),
                                frequencies_Hz=np.array([float(freq_hz)]), x_coords=coords, y_coords=coords, **extra)
        if not npz_path.exists():
            raise FileNotFoundError(f"Missing expected npz file: {npz_path}")
        rows.append((i, float(freq_hz), str(npz_path)))
    with open(out_dir / "TbSpectra_manifest.txt", "w", encoding="utf-8") as f:   # :194-198
        f.write("# idx freq_hz npz_path png_path\n")
        for r in rows:
            f.write(f"{r[0]:02d} {r[1]:.6e} {r[2]} -\n")
    return rows


def main(argv=None):
    ap = argparse.ArgumentParser(description="Ray-tracing T_b spectra maps on a synthetic spherical corona.")
    ap.add_argument("--out-dir", default="tb_spectra_out")
    ap.add_argument("--N-pix", "-n", type=int, default=128)
    ap.add_argument("--fmin-mhz", type=float, default=30.0)
    ap.add_argument("--fmax-mhz", type=float, default=800.0)
    ap.add_argument("--n-freq", type=int, default=30)
    ap.add_argument("--start-from-idx", type=int, default=0)
    ap.add_argument("--phi0-offset", type=float, default=-140.0)
    ap.add_argument("--b0-angle", type=float, default=0.0,
                    help="solar B0 angle of the observer [deg], > 0 tilts the north pole towards the observer")
    ap.add_argument("--p-angle", type=float, default=0.0,
                    help="solar P angle of the observer [deg], > 0 turns north from image up towards east (left)")
    ap.add_argument("--device", default="cuda", choices=["cpu", "cuda"])
    ap.add_argument("--raytrace-device", default="cuda", choices=["cpu", "cuda"])
    ap.add_argument("--quiet", "-q", action="store_true")
    ap.add_argument("--diagnostics", action="store_true",
                    help="also save emission centroid and height, optical depths and ray turning point per pixel")
    a = ap.parse_args(argv)
    if a.device != "cuda" or a.raytrace_device != "cuda":
        raise RuntimeError("raytracinggrff_b200 is CUDA-only (no CPU path, no fallback)")
    model = synthetic.spherical_corona(150, 110, 128, r_max=8.0, active_region=True)
    rows = tb_spectra(model, a.out_dir, a.N_pix, a.fmin_mhz, a.fmax_mhz, a.n_freq, a.start_from_idx, a.phi0_offset,
                      quiet=a.quiet, diagnostics=a.diagnostics, b0_angle=a.b0_angle, p_angle=a.p_angle)
    print(f"Saved {len(rows)} maps to {a.out_dir}")


if __name__ == "__main__":
    main()
