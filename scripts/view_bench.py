"""Cost of the observer view (solar B0 / P) on one GPU: the same work at B0 = P = 0 and at a non-zero view, alternated.

    python scripts/view_bench.py [--reps 5] [--warmup 1] [--b0 7.25] [--p 24] [--out result.json] [--quick]

* render_los_map at 512^2 x 400 x 8 frequencies (75 MHz - 1.5 GHz), plain (theta = 90, free-free) and with theta from
  the B vector + gyroresonance (em_flag 4): kernel time (CUDA events);
* set_model_from_spherical at 512^3 (config 5's model and cube, want_bvec=True): host clock around the call, which ends
  in a device synchronise (the five uploads of the model included).

Medians of --reps runs and the ratio view / zero view.  Prints the card's name and power limit, read in the same run.
Writes nothing unless --out is given.  --quick: small sizes and one rep, to rehearse the script.
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


def _alternate(calls, reps, warmup, measure):
    """calls: {name: fn}; each rep runs every call once, in alternating order; returns {name: [measure(...)]}."""
    for _ in range(warmup):
        for f in calls.values():
            f()
    out = {k: [] for k in calls}
    for rep in range(reps):
        for name in (list(calls) if rep % 2 == 0 else list(calls)[::-1]):
            out[name].append(measure(calls[name]))
    return out


def los_map(ses, n_pix, view, reps, warmup):
    xs = np.linspace(-1.44, 1.44, n_pix)
    zc, dz = los.z_grid(400, 3e-4)
    freqs = np.geomspace(75e6, 1.5e9, 8)
    area = ((xs[1] - xs[0]) * R_SUN_CM) ** 2
    res = []
    for variant, kw in (("plain", dict(em_flag=5)), ("bvec_gr", dict(em_flag=4, use_bvec=True))):
        calls = {name: (lambda b0=b0, p=p: ses.render_los_map(xs, xs, zc, dz * R_SUN_CM, freqs, pixel_area_cm2=area,
                                                              b0_angle=b0, p_angle=p, **kw))
                 for name, (b0, p) in (("zero", (0.0, 0.0)), ("view", view))}

        def kernel_ms(f):
            f()
            return ses.ctx.last_kernel_ms
        t = _alternate(calls, reps, warmup, kernel_ms)
        med = {k: float(np.median(v)) for k, v in t.items()}
        res.append(dict(variant=variant, n_pix=n_pix, n_z=400, n_freq=8, zero_ms=med["zero"], view_ms=med["view"],
                        ratio=med["view"] / med["zero"], zero_all_ms=t["zero"], view_all_ms=t["view"]))
        print(f"render_los_map {n_pix}^2 x 400 x 8 {variant:8s} zero {med['zero']:8.2f} ms  view {med['view']:8.2f} ms  "
              f"ratio {med['view'] / med['zero']:.4f}")
    return res


def cube(ses, model, grid_n, view, reps, warmup):
    g = np.linspace(-4.0, 4.0, grid_n)
    calls = {name: (lambda b0=b0, p=p: ses.set_model_from_spherical(model, g, g, g, want_bvec=True, b0_angle=b0,
                                                                    p_angle=p))
             for name, (b0, p) in (("zero", (0.0, 0.0)), ("view", view))}

    def wall(f):
        t0 = time.perf_counter()
        f()
        return time.perf_counter() - t0
    t = _alternate(calls, reps, warmup, wall)
    med = {k: float(np.median(v)) for k, v in t.items()}
    print(f"set_model_from_spherical {grid_n}^3 zero {med['zero'] * 1e3:8.1f} ms  view {med['view'] * 1e3:8.1f} ms  "
          f"ratio {med['view'] / med['zero']:.4f}")
    return dict(grid_n=grid_n, zero_s=med["zero"], view_s=med["view"], ratio=med["view"] / med["zero"],
                zero_all_s=t["zero"], view_all_s=t["view"])


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--b0", type=float, default=7.25, help="B0 of the non-zero view [deg]")
    ap.add_argument("--p", type=float, default=24.0, help="P of the non-zero view [deg]")
    ap.add_argument("--out", default=None, help="also write the result as JSON to this path")
    ap.add_argument("--quick", action="store_true", help="small sizes, one rep (rehearsal)")
    a = ap.parse_args(argv)
    if a.reps < 1:
        raise SystemExit("--reps must be >= 1")
    reps = 1 if a.quick else a.reps
    view = (a.b0, a.p)
    model = synthetic.spherical_corona(200, 140, 160, r_max=7.2, active_region=True)   # bench.py config 5's model
    res = dict(reps=reps, warmup=a.warmup, view_deg=dict(b0=a.b0, p=a.p), card=card())
    with RaySession(0) as ses:
        ses.set_spherical_model(model)
        res["los_map"] = los_map(ses, 64 if a.quick else 512, view, reps, a.warmup)
        res["set_model_from_spherical"] = cube(ses, model, 64 if a.quick else 512, view, reps, a.warmup)
    print(f"card {res['card']}")
    print(json.dumps(res))
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
