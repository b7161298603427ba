#!/usr/bin/env python
"""Device time of each config-4 frequency rendered alone: where a change to render_map_kernel gains or loses.

    python scripts/freq_bench.py [--reps N] [--json PATH]

bench.py's workload (512^2 pixels, 256^3 cube, GR+FF, theta from the B vector, cross-sections traced, 4x8 tiles),
one render_map call per frequency: one launch, timed by the library's events around it (ctx.last_kernel_ms).
Each frequency is warmed once and timed N times; the median is printed.  The record stride of a frequency's preset
sets how many of its steps carry a record (and trace the cross-section pencil): 1 in 6 at 75 MHz, every one at
1.5 GHz.  The library is the package's, or RTGRFF_LIB's; compare two builds by running this once with each.
"""
import argparse
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402  (the workload tables the benchmark runs)
from raytracinggrff_b200 import RaySession, _lib  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--json", help="also write the table to this file")
    args = ap.parse_args()
    w = bench.workload("c4", 1)
    c = bench.host_cube(w)
    xs, ys, zs = bench.rays_of(w)
    g = (c["x_grid"], c["y_grid"], c["z_grid"])
    rows = []
    with RaySession(0) as ses:
        ses.set_omega_cube(c["omega_pe"], *g)
        ses.set_field_cubes(*g, c["ne"], c["te"], c["b"], c["bx"], c["by"], c["bz"])
        kw = dict(trace_crosssections=True, perturb_ratio=2.0, pixel_area_cm2=bench.pixel_area(w), r_sun_cm=bench.R_SUN_CM,
                  em_flag=4, s_max=30, use_bvec=True, image_shape=(w["n_pix_y"], w["n_pix_x"]))
        for p in w["freq_params"]:
            fp = [p]
            _, _, st = ses.render_map(xs, ys, zs, fp, **kw)
            ms = []
            for _ in range(args.reps):
                ses.render_map(xs, ys, zs, fp, **kw)
                ms.append(ses.ctx.last_kernel_ms)
            med = float(np.median(ms))
            rows.append(dict(freq_hz=p["freq_hz"], n_steps=p["n_steps"], stride=p["record_stride"], ms=ms, median_ms=med,
                             active_ray_steps=st["active_ray_steps"], nominal_ray_steps=st["nominal_ray_steps"]))
            print(f"GR+FF bvec f={p['freq_hz'] / 1e6:7.1f} MHz T={p['n_steps']:6d} stride={p['record_stride']}: {med:7.2f} ms  "
                  f"active {st['active_ray_steps'] / med / 1e6:.2f} G ray-steps/s  "
                  f"({st['active_ray_steps'] / st['nominal_ray_steps']:.2f} active)  [{' '.join(f'{m:.2f}' for m in ms)}]",
                  flush=True)
    total = sum(r["median_ms"] for r in rows)
    print(f"GR+FF bvec total {total:.1f} ms  lib {_lib.LIB_PATH}")
    if args.json:
        Path(args.json).write_text(json.dumps(dict(lib=str(_lib.LIB_PATH), reps=args.reps, rows=rows, total_ms=total),
                                              indent=1))


if __name__ == "__main__":
    main()
