"""Straight line-of-sight maps on one GPU: the staged drop-ins (los.resample_MAS + los.SyntheticFF) against the fused
kernel (los.render_los_map), and the fused kernel alone at larger sizes.

    python scripts/los_bench.py [--reps 5] [--warmup 1] [--out result.json] [--quick]

* config-2 shape: 256^2 pixels, N_z 400 (dz0 3e-4), 4 frequencies from 450 MHz in log steps of 0.1, on
  synthetic.spherical_corona(150, 110, 128, r_max=8, active_region=True); both paths end to end from the model
  (host clock around calls that end in a device synchronise), alternated, warmed; the largest relative T_b
  difference between them;
* render_los_map alone at 512^2 x 400 x 8 frequencies (75 MHz - 1.5 GHz) and 2048^2 x 400 x 16 frequencies
  (20 - 300 MHz), each plain (theta = 90, free-free), with diagnostics, and with theta from B + gyroresonance
  (em_flag 4): kernel time (CUDA events), LOS samples/s and voxel-frequency evaluations/s over the kernel time.

Medians of --reps runs.  Prints the card's name and power limit, read in the same run.  Writes nothing unless --out
is given.  --quick: small sizes and one rep, to rehearse the script.
"""
from __future__ import annotations

import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "scripts"))

from diag_bench import card  # noqa: E402
from raytracinggrff_b200 import RaySession, los, synthetic  # noqa: E402

R_SUN_CM = 6.957e10
FOV = (-1.44, 1.44)


def _timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return out, time.perf_counter() - t0


def config2(ses, model, reps, warmup, n_pix):
    kw = dict(N_pix=n_pix, X_range=FOV, Y_range=FOV, N_z=400, dz0=3e-4)
    calls = {
        "staged": lambda: los.SyntheticFF(los.resample_MAS(model, out_path=None, context=ses.ctx, **kw), 450e6, 4, 0.1,
                                          session=ses),
        "fused": lambda: los.render_los_map(model, freq0=450e6, Nfreq=4, freq_log_step=0.1, session=ses, **kw),
    }
    for _ in range(warmup):
        for f in calls.values():
            f()
    times = {k: [] for k in calls}
    outs = {}
    for rep in range(reps):
        for name in (list(calls) if rep % 2 == 0 else list(calls)[::-1]):
            outs[name], dt = _timed(calls[name])
            times[name].append(dt)
    tb, ref = outs["fused"]["emission_cube"], outs["staged"]["emission_cube"]
    nz = ref > 0
    med = {k: float(np.median(v)) for k, v in times.items()}
    return dict(n_pix=n_pix, n_z=400, n_freq=4, staged_s=med["staged"], fused_s=med["fused"],
                speedup=med["staged"] / med["fused"], staged_all_s=times["staged"], fused_all_s=times["fused"],
                max_rel_d_tb=float((np.abs(tb[nz] - ref[nz]) / ref[nz]).max()),
                zero_nan_patterns_equal=bool(np.array_equal(np.isnan(tb), np.isnan(ref))
                                             and np.array_equal(tb == 0, ref == 0)))


def sized(ses, n_pix, n_z, freqs, reps, warmup):
    xs = np.linspace(*FOV, n_pix)
    zc, dz = los.z_grid(n_z, 3e-4)
    area = ((xs[1] - xs[0]) * R_SUN_CM) ** 2
    variants = {"plain": dict(em_flag=5), "diagnostics": dict(em_flag=5, diagnostics=True),
                "bvec_gr": dict(em_flag=4, use_bvec=True)}
    out = []
    for name, v in variants.items():
        call = lambda: ses.render_los_map(xs, xs, zc, dz * R_SUN_CM, freqs, pixel_area_cm2=area, **v)  # noqa: E731
        for _ in range(warmup):
            call()
        k_ms, wall = [], []
        for _ in range(reps):
            res, dt = _timed(call)
            wall.append(dt)
            k_ms.append(ses.ctx.last_kernel_ms)
        st = res[2]
        k = float(np.median(k_ms)) / 1e3
        out.append(dict(variant=name, n_pix=n_pix, n_z=n_z, n_freq=len(freqs), kernel_ms=k * 1e3, kernel_ms_all=k_ms,
                        call_s=float(np.median(wall)), los_samples=st["los_samples"], valid_samples=st["valid_samples"],
                        voxel_freq_evaluations=st["voxel_freq_evaluations"],
                        los_samples_per_s=st["los_samples"] / k, voxel_freq_evals_per_s=st["voxel_freq_evaluations"] / k))
        print(f"{n_pix}^2 x {n_z} x {len(freqs)} {name:12s} kernel {k * 1e3:9.2f} ms  "
              f"{st['los_samples'] / k:.3e} LOS samples/s  {st['voxel_freq_evaluations'] / k:.3e} voxel-freq evals/s")
        del res
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None, help="also write the result as JSON to this path")
    ap.add_argument("--quick", action="store_true", help="small sizes, one rep (rehearsal)")
    a = ap.parse_args(argv)
    if a.reps < 1:
        raise SystemExit("--reps must be >= 1")
    reps = 1 if a.quick else a.reps
    model = synthetic.spherical_corona(150, 110, 128, r_max=8.0, active_region=True)
    res = dict(reps=reps, warmup=a.warmup, card=card())
    with RaySession(0) as ses:
        res["config2"] = config2(ses, model, reps, a.warmup, 32 if a.quick else 256)
        c2 = res["config2"]
        print(f"config-2 shape {c2['n_pix']}^2: staged {c2['staged_s']:.3f} s, fused {c2['fused_s']:.3f} s "
              f"(x{c2['speedup']:.1f}), max rel dT_b {c2['max_rel_d_tb']:.2e}")
        ses.set_spherical_model(model)
        res["sizes"] = (sized(ses, 64 if a.quick else 512, 400, np.geomspace(75e6, 1.5e9, 8), reps, a.warmup)
                        + sized(ses, 128 if a.quick else 2048, 400, np.geomspace(20e6, 300e6, 16), reps, a.warmup))
    print(f"card {res['card']}")
    print(json.dumps(res))
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
