"""Ray-traced emission map: the hot-path part of ``run_ray_tracing_emission``
(reference: script/resample_with_ray_tracing.py:154-549) on in-memory cubes.

The reference function starts from a MAS model directory and resamples it through psipy
(:251-293) — out of scope here (SURVEY.md §8 row 13).  Everything after that is kept with the same
keyword names, defaults and result keys: ray launch geometry (:295-303), tracing (:305-352),
GRFF header (:354-365), sampling (:372-398), GRFF per pixel or batched (:400-524), scrubbing and
the npz written at :533-540.  ``model`` is a dict with ``x_grid, y_grid, z_grid, omega_pe, ne,
te, b`` (and optionally ``bx, by, bz``) such as ``synthetic.corona_cube`` returns.

``grff_backend``:
  'get_mw'   per-pixel ``PyGET_MW`` calls with ``Parms (15,N_valid)`` as at :467-524 (drop-in symbol)
  'fastgrff' one batched ``get_mw_slice`` call with ``Parms_M (15,n_rec,n_rays)`` as at :400-466
  'device'   paths and samples stay on the GPU, no Parms is materialised (rtgrff_emission_traced)
  'fused'    single fused kernel per map (rtgrff_render_map)
"""
from __future__ import annotations

import numpy as np

from . import _lib, synthetic
from .grff import initGET_MW
from .session import RaySession

R_sun_cm = 6.957e10      # script/resample_with_ray_tracing.py:68
R_sun_m = 6.957e8
c = 2.998e10             # :91
kb = 1.38065e-16         # :92
sfu2cgs = 1e-19          # :93
AU_cm = 1.49599e13       # :94


def _check_device(name, value):
    v = value.lower()
    if v == "cpu":
        raise RuntimeError(f"{name}='cpu': raytracinggrff_b200 is CUDA-only (no CPU path, no fallback)")
    if v != "cuda":
        raise ValueError(f"Unsupported device '{value}'. Use 'cpu' or 'cuda'.")


def pixel_area_cm2(X_fov, N_pix):
    """script/resample_with_ray_tracing.py:360-363."""
    pixel_size_cm = (2 * X_fov) / N_pix * R_sun_cm
    return pixel_size_cm * pixel_size_cm


def tb_from_rl(RL, frequencies_Hz, area):
    """SFU -> T_b and V/I for one pixel, script/resample_with_ray_tracing.py:513-520."""
    Nf = RL.shape[1]
    tb = np.zeros(Nf)
    vi = np.zeros(Nf)
    for ifreq in range(Nf):
        intensity_sfu = RL[5, ifreq] + RL[6, ifreq]
        vi[ifreq] = (RL[5, ifreq] - RL[6, ifreq]) / (RL[5, ifreq] + RL[6, ifreq] + 1e-30)
        nu_GHz = RL[0, ifreq]
        nu_Hz = frequencies_Hz[ifreq] if nu_GHz <= 0 else nu_GHz * 1e9
        conversion_factor = (sfu2cgs * c * c / (2.0 * kb * nu_Hz * nu_Hz) / area) * (AU_cm * AU_cm)
        tb[ifreq] = intensity_sfu * conversion_factor
    return tb, vi


def pack_parms_batch(sampled, area, s_input_on=False):
    """Parms_M (15, n_rec, n_rays) Fortran order, script/resample_with_ray_tracing.py:404-426:
    theta=90, flag=1+4, s_max=30 everywhere; valid & finite samples compacted to the front."""
    ne_all, te_all, b_all = sampled["ne"], sampled["te"], sampled["b"]
    n_rec, n_rays = ne_all.shape
    valid = sampled["valid_mask"] & np.isfinite(ne_all) & np.isfinite(te_all) & np.isfinite(b_all)
    Parms_M = np.zeros((15, n_rec, n_rays), dtype=np.float64, order="F")
    Parms_M[4] = 90.0
    Parms_M[6] = 1 + 4
    Parms_M[7] = 30
    # stable compaction of the valid samples of every ray, vectorised over rays
    order = np.argsort(~valid, axis=0, kind="stable")
    cnt = valid.sum(axis=0)
    keep = np.arange(n_rec)[:, None] < cnt[None, :]
    for m, key in ((0, "ds"), (1, "te"), (2, "ne"), (3, "b")):
        Parms_M[m] = np.where(keep, np.take_along_axis(sampled[key].astype(np.float64), order, axis=0), 0.0)
    if s_input_on:
        Parms_M[14] = np.where(keep, np.take_along_axis(sampled["s"].astype(np.float64), order, axis=0) * area, 0.0)
    return Parms_M


def _upload_model(ses, model, grid_n, grid_extent, phi0_offset, b0_angle=0.0, p_angle=0.0):
    if "omega_pe" in model:
        xg, yg, zg = model["x_grid"], model["y_grid"], model["z_grid"]
        ses.set_omega_cube(model["omega_pe"], xg, yg, zg)
        ses.set_field_cubes(xg, yg, zg, model["ne"], model["te"], model["b"])
    else:
        # a spherical (phi, latitude, r) model: the cube resampling of :251-293 on the GPU
        xg = yg = zg = np.linspace(-grid_extent, grid_extent, int(grid_n))
        ses.set_model_from_spherical(model, xg, yg, zg, phi0_offset=phi0_offset, b0_angle=b0_angle, p_angle=p_angle)


def diagnostic_maps(diag, N_pix):
    """RaySession.render_map_diag's planes ((n_freq, n_rays) each, ray p = i*N_pix + j) -> the result / npz keys of
    ``diagnostics=True``: emission_centroid_xyz (N_pix, N_pix, n_freq, 3) [R_sun], emission_r_mean, tau_L, tau_R and
    ray_r_min (N_pix, N_pix, n_freq) each, laid out as emission_cube."""
    m = {k: np.moveaxis(np.asarray(v).reshape(-1, N_pix, N_pix), 0, -1) for k, v in diag.items()}
    return {"emission_centroid_xyz": np.stack([m["em_x"], m["em_y"], m["em_z"]], axis=-1),
            "emission_r_mean": m["em_r"], "tau_L": m["tau_L"], "tau_R": m["tau_R"], "ray_r_min": m["ray_r_min"]}


def _emission_of_rays(ses, backend, x_flat, y_flat, z_start, kvec, p, image_shape=None):
    """The hot path for one contiguous range of rays on one GPU: trace -> sample -> GRFF -> T_b.  `p` holds the
    call's scalar settings.  Returns (tb (n_rays, Nf), vi (n_rays, Nf), sampled or None, diag or None); diag is
    render_map_diag's dict of (Nf, n_rays) planes when p["diagnostics"]."""
    n_rays = len(x_flat)
    Nf, freq0, freq_hz, freq_log_step, area = p["Nf"], p["freq0"], p["freq_hz"], p["freq_log_step"], p["area"]
    frequencies_Hz = p["frequencies_Hz"]
    tb_out = np.zeros((n_rays, Nf), dtype="double")
    vi_out = np.zeros((n_rays, Nf), dtype="double")
    ray_start = np.column_stack([x_flat, y_flat, z_start])
    sampled = None
    if backend == "fused":
        render = ses.render_map_diag if p["diagnostics"] else ses.render_map
        out = render(x_flat, y_flat, z_start, [(freq_hz, p["dt"], p["n_steps"], p["record_stride"])],
                     kvec_in_norm=kvec, trace_crosssections=True, perturb_ratio=p["perturb_ratio"],
                     pixel_area_cm2=area, r_sun_cm=R_sun_cm, image_shape=image_shape,
                     s_mode=p["s_mode"], s_input_on=p["s_input_on"])
        tb_out[:, 0], vi_out[:, 0] = out[0][0], out[1][0]
        return tb_out, vi_out, None, (out[3] if p["diagnostics"] else None)
    keep_host = backend in ("get_mw", "fastgrff") or p["return_samples"]
    ses.trace(freq_hz, x_flat, y_flat, z_start, kvec, p["dt"], p["n_steps"], p["record_stride"], True, p["perturb_ratio"],
              s_mode=p["s_mode"], fetch=False)
    sampled = ses.sample_traced(ray_start, R_sun_cm, 0.0, 1e4, 0.0, fetch=keep_host)
    if backend == "device":
        tb, vi = ses.emission_traced(area, freq0, Nf, freq_log_step, s_input_on=p["s_input_on"])
        return tb, vi, sampled, None
    if backend == "fastgrff":
        n_rec = sampled["ne"].shape[0]
        Parms_M = pack_parms_batch(sampled, area, p["s_input_on"])
        Lparms_M = np.array([n_rays, n_rec, Nf, 1, 0, 0], dtype=np.int32)
        Rparms_M = np.zeros((3, n_rays), dtype=np.float64, order="F")
        Rparms_M[0, :], Rparms_M[1, :], Rparms_M[2, :] = area, freq0, freq_log_step
        RL_M = np.zeros((7, Nf, n_rays), dtype=np.float64, order="F")
        status = ses.get_mw_slice(Lparms_M, Rparms_M, Parms_M, RL_M)
        if np.any(status != 0) and p["verbose"]:
            print(f"get_mw_slice: warning {np.count_nonzero(status)} pixels returned non-zero status")
        for q in range(n_rays):
            if status[q] != 0:
                continue
            tb_out[q], vi_out[q] = tb_from_rl(RL_M[:, :, q], frequencies_Hz, area)
        return tb_out, vi_out, sampled, None
    # 'get_mw': the reference's per-pixel loop, script/resample_with_ray_tracing.py:467-524
    GET_MW = initGET_MW(p["grff_lib"])
    Lparms = np.zeros(5, dtype="int32")
    Lparms[1] = Nf
    Rparms = np.array([area, freq0, freq_log_step], dtype="double")
    dummy = np.array(0, dtype="double")
    for q in range(n_rays):
        valid = (sampled["valid_mask"][:, q] & np.isfinite(sampled["ne"][:, q])
                 & np.isfinite(sampled["te"][:, q]) & np.isfinite(sampled["b"][:, q]))
        if not np.any(valid):
            continue
        n_valid = int(np.count_nonzero(valid))
        Parms = np.zeros((15, n_valid), dtype="double", order="F")
        Parms[0] = sampled["ds"][:, q][valid]
        Parms[1] = sampled["te"][:, q][valid]
        Parms[2] = sampled["ne"][:, q][valid]
        Parms[3] = sampled["b"][:, q][valid]
        Parms[4] = 90.0
        Parms[6] = 1 + 4
        Parms[7] = 30
        if p["s_input_on"]:
            Parms[14] = sampled["s"][:, q][valid] * area
        L = Lparms.copy()
        L[0] = n_valid
        RL = np.zeros((7, Nf), dtype="double", order="F")
        if GET_MW(L, Rparms, Parms, dummy, dummy, dummy, RL) != 0:
            continue
        tb_out[q], vi_out[q] = tb_from_rl(RL, frequencies_Hz, area)
    return tb_out, vi_out, sampled, None


def run_ray_tracing_emission(model, N_pix=64, X_fov=1.44, freq_hz=75e6, z_observer=3.0, dt=6e-3, n_steps=5000,
                             record_stride=10, n_workers=1, s_input_on=False, out_path=None, grff_lib=None, Nfreq=1,
                             freq0=None, freq_log_step=0.0, save_plots=False, verbose=True, device="cuda",
                             fallback_to_cpu=False, raytrace_device="cuda", grff_backend="get_mw",
                             perturb_ratio=2, session=None, return_samples=False, s_mode="per_step",
                             grid_n=128, grid_extent=3.0, phi0_offset=0.0, consider_beam=False, beam_fwhm=0.2,
                             diagnostics=False, b0_angle=0.0, p_angle=0.0):
    """``n_workers`` (the reference's ``--workers``, script/resample_with_ray_tracing.py:333-352: contiguous ray
    chunks over a process pool, concatenated on the ray axis) maps to GPUs here: the rays are split into
    ``n_workers`` contiguous chunks exactly as there, chunk k runs on GPU k mod (number of visible GPUs) from its
    own host thread (the library calls release the GIL) with its own context and a replica of the cubes, and the
    chunks' maps are concatenated.  Rays never interact, so the result does not depend on the split.
    ``diagnostics`` (fused backend only): the result and the npz also hold where each pixel's emission comes from,
    the keys of diagnostic_maps (RaySession.render_map_diag); every other key is the same as without.
    ``b0_angle``, ``p_angle`` [deg]: the observer's view of a spherical model (include/rtgrff.h, "Observer view"); a
    Cartesian cube model (one with ``omega_pe``) cannot be re-oriented and takes zero angles only."""
    from .cubes import check_view
    b0_angle, p_angle = check_view(b0_angle, p_angle)
    if "omega_pe" in model and (b0_angle != 0.0 or p_angle != 0.0):
        raise ValueError("b0_angle / p_angle need a spherical model: a Cartesian cube model (omega_pe) cannot be "
                         "re-oriented")
    if freq0 is None:
        freq0 = freq_hz
    backend = grff_backend.lower()
    if backend not in ("get_mw", "fastgrff", "device", "fused"):
        raise ValueError(f"Unsupported grff_backend '{grff_backend}'. Use 'get_mw', 'fastgrff', 'device' or 'fused'.")
    if diagnostics and backend != "fused":
        raise ValueError(f"diagnostics need the fused backend (grff_backend='fused'), not '{grff_backend}'")
    _check_device("device", device)
    _check_device("raytrace_device", raytrace_device)
    # s_input_on (script/resample_with_ray_tracing.py:501): Parms[14] = S * area.  The reference leaves the
    # meaning of that slot to a private GRFF build; here the voxel's source term is multiplied by
    # Parms[14] / area = S (include/rtgrff.h).  s_mode picks the S of the reference's CPU path (per step,
    # ~1) or of its CUDA path (cumulative since the start of the ray: the pencil's magnification).
    x_flat, y_flat, z_start, kvec = synthetic.ray_launch_geometry(N_pix, X_fov, z_observer)
    n_rays = len(x_flat)
    Nf = int(Nfreq)
    frequencies_Hz = synthetic.log_frequencies(freq0, Nf, freq_log_step)
    area = pixel_area_cm2(X_fov, N_pix)
    x_coords = np.linspace(-X_fov, X_fov, N_pix) * R_sun_m
    y_coords = np.linspace(-X_fov, X_fov, N_pix) * R_sun_m
    if backend == "fused" and (Nf != 1 or abs(freq0 - freq_hz) > 0):
        raise ValueError("the fused backend traces and emits at the same frequency: use Nfreq=1, freq0=freq_hz "
                         "(or RaySession.render_map for a list of frequencies)")
    p = dict(Nf=Nf, freq0=freq0, freq_hz=freq_hz, freq_log_step=freq_log_step, area=area, frequencies_Hz=frequencies_Hz,
             dt=dt, n_steps=n_steps, record_stride=record_stride, perturb_ratio=perturb_ratio, s_mode=s_mode,
             s_input_on=s_input_on, return_samples=return_samples, verbose=verbose, grff_lib=grff_lib,
             diagnostics=bool(diagnostics))

    n_workers = max(1, int(n_workers))
    if n_workers == 1 or n_rays < 2:
        ses = session or RaySession(context=_lib.default_context())
        _upload_model(ses, model, grid_n, grid_extent, phi0_offset, b0_angle, p_angle)
        tb, vi, sampled, diag = _emission_of_rays(ses, backend, x_flat, y_flat, z_start, kvec, p,
                                                  image_shape=(N_pix, N_pix))
    else:
        from concurrent.futures import ThreadPoolExecutor
        n_dev = _lib.load().rtgrff_device_count()
        if n_dev <= 0:
            raise RuntimeError("No CUDA device is available to raytracinggrff_b200 (no CPU path).")
        chunk_size = (n_rays + n_workers - 1) // n_workers                       # script/...:336
        chunks = [(s, min(s + chunk_size, n_rays)) for s in range(0, n_rays, chunk_size)]

        def work(k):
            s, e = chunks[k]
            ses_k = RaySession(device=k % n_dev)                                  # its own context, stream and cube replica
            try:
                _upload_model(ses_k, model, grid_n, grid_extent, phi0_offset, b0_angle, p_angle)
                return _emission_of_rays(ses_k, backend, x_flat[s:e], y_flat[s:e], z_start[s:e], kvec[s:e], p)
            finally:
                ses_k.close()
        with ThreadPoolExecutor(max_workers=min(len(chunks), n_dev)) as ex:
            parts = list(ex.map(work, range(len(chunks))))
        tb = np.concatenate([q[0] for q in parts], axis=0)                        # script/...:351-352 (ray axis)
        vi = np.concatenate([q[1] for q in parts], axis=0)
        sampled = None
        if parts[0][2]:
            sampled = {k: np.concatenate([q[2][k] for q in parts], axis=1) for k in parts[0][2]}
        diag = None
        if parts[0][3]:
            diag = {k: np.concatenate([q[3][k] for q in parts], axis=1) for k in parts[0][3]}

    emission_cube = tb.reshape(N_pix, N_pix, Nf)
    emission_polVI_cube = vi.reshape(N_pix, N_pix, Nf)
    emission_cube = np.nan_to_num(emission_cube, nan=0.0, posinf=0.0, neginf=0.0)
    result = {
        "emission_cube": emission_cube,
        "emission_polVI_cube": emission_polVI_cube,
        "frequencies_Hz": frequencies_Hz,
        "x_coords": x_coords,
        "y_coords": y_coords,
    }
    if consider_beam:
        # --consider-beam (:618-624): the reference convolves the plotted map only; here the convolved
        # map is returned (and saved) next to the raw cube
        from .util import convolve_beam
        beam = emission_cube[:, :, 0].copy()
        beam[beam == 0] = np.nan
        result["emission_map_beam"] = convolve_beam(beam, beam_fwhm, [-X_fov, X_fov], N_pix)
    if diag is not None:
        result.update(diagnostic_maps(diag, N_pix))
    if out_path is not None:
        np.savez_compressed(out_path, **result)
    if return_samples and sampled:
        result["sampled"] = sampled
    return result


def main(argv=None):
    """Command line of script/resample_with_ray_tracing.py:652-730 with the same flags.  ``--model-path``
    is an .npz of spherical variables (raytracinggrff_b200.cubes.save_spherical_model) or 'synthetic'
    (the analytic corona) instead of a MAS directory: reading MAS HDF files needs psipy (out of scope)."""
    import argparse
    parser = argparse.ArgumentParser(description="Ray-tracing emission map on the GPU (librtgrff_b200).")
    parser.add_argument("--model-path", "-m", type=str, default="synthetic")
    parser.add_argument("--N-pix", "-n", type=int, default=32)
    parser.add_argument("--X-FOV", "-f", type=float, default=1.44)
    parser.add_argument("--freq", type=float, default=75e6)
    parser.add_argument("--grid-n", type=int, default=128)
    parser.add_argument("--grid-extent", type=float, default=3.0)
    parser.add_argument("--z-observer", type=float, default=3.0)
    parser.add_argument("--dt", type=float, default=6e-3)
    parser.add_argument("--n-steps", type=int, default=5000)
    parser.add_argument("--record-stride", type=int, default=10)
    parser.add_argument("--workers", "-w", type=int, default=1, help="ray chunks, spread over the visible GPUs (chunk k on GPU k mod n_gpus)")
    parser.add_argument("--out-path", "-o", type=str, default="ray_tracing_emission.npz")
    parser.add_argument("--grff-lib", type=str, default=None, help="library exporting PyGET_MW (default: librtgrff_b200.so)")
    parser.add_argument("--grff-backend", type=str, default="get_mw", choices=["get_mw", "fastgrff", "device", "fused"])
    parser.add_argument("--s-input-on", action="store_true")
    parser.add_argument("--s-mode", type=str, default="per_step", choices=["per_step", "cumulative"])
    parser.add_argument("--device", type=str, default="cuda", choices=["cpu", "cuda"])
    parser.add_argument("--raytrace-device", type=str, default="cuda", choices=["cpu", "cuda"])
    parser.add_argument("--consider-beam", action="store_true")
    parser.add_argument("--beam-fwhm", type=float, default=0.2)
    parser.add_argument("--phi0-offset", type=float, default=0)
    parser.add_argument("--b0-angle", type=float, default=0.0,
                        help="solar B0 angle of the observer [deg], > 0 tilts the north pole towards the observer")
    parser.add_argument("--p-angle", type=float, default=0.0,
                        help="solar P angle of the observer [deg], > 0 turns north from image up towards east (left)")
    parser.add_argument("--no-fallback", action="store_true", help="accepted for compatibility; there is no CPU path to fall back to")
    parser.add_argument("--no-plots", action="store_true", help="accepted for compatibility; no plots are made")
    parser.add_argument("--quiet", "-q", action="store_true")
    parser.add_argument("--diagnostics", action="store_true",
                        help="also save emission centroid, emission height, optical depths and ray turning point "
                             "per pixel (fused backend only)")
    args = parser.parse_args(argv)
    if args.model_path == "synthetic":
        model = synthetic.spherical_corona()
    else:
        from .cubes import load_spherical_model
        model = load_spherical_model(args.model_path)
    res = run_ray_tracing_emission(
        model, N_pix=args.N_pix, X_fov=args.X_FOV, freq_hz=args.freq, grid_n=args.grid_n, grid_extent=args.grid_extent,
        z_observer=args.z_observer, dt=args.dt, n_steps=args.n_steps, record_stride=args.record_stride,
        n_workers=args.workers, s_input_on=args.s_input_on, out_path=args.out_path, grff_lib=args.grff_lib, Nfreq=1,
        freq0=args.freq, freq_log_step=0.0, save_plots=False, verbose=not args.quiet, device=args.device,
        fallback_to_cpu=not args.no_fallback, raytrace_device=args.raytrace_device, grff_backend=args.grff_backend,
        consider_beam=args.consider_beam, beam_fwhm=args.beam_fwhm, phi0_offset=args.phi0_offset, s_mode=args.s_mode,
        diagnostics=args.diagnostics, b0_angle=args.b0_angle, p_angle=args.p_angle)
    if not args.quiet:
        tb = res["emission_cube"]
        print(f"T_b map {tb.shape} at {args.freq / 1e6:.1f} MHz: max {tb.max():.3e} K -> {args.out_path}")
    return res


if __name__ == "__main__":
    main()
