"""Cost of the map diagnostics: render_map against render_map_diag on BASELINE config 4 (the bench workload: 512^2
pixels, 256^3 cube with the active region, 8 frequencies 75 MHz - 1.5 GHz, cross-sections on, theta from the B
vector, gyroresonance + free-free), in one process, warmed, alternating the two calls.

    python scripts/diag_bench.py [--reps 5] [--warmup 1] [--out result.json]

Prints the median wall time of each call (host clock around the call, which ends in a device synchronise), their
ratio, and the card's name and power limit, which belong to the numbers.  Writes nothing unless --out is given.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import bench  # noqa: E402
from raytracinggrff_b200 import RaySession, synthetic  # noqa: E402


def card():
    """Name and power limit of GPU 0 (nvidia-smi query, read only)."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # noqa: BLE001
        return dict(name="unknown", error=str(e))


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None, help="also write the result as JSON to this path")
    a = ap.parse_args(argv)
    if a.reps < 1:
        raise SystemExit("--reps must be >= 1")
    w = bench.workload("c4", 1)
    c = synthetic.corona_cube(w["grid_n"], w["extent"], active_region=True)
    xs, ys, zs = bench.rays_of(w)
    kw = dict(trace_crosssections=True, perturb_ratio=2.0, pixel_area_cm2=bench.pixel_area(w), r_sun_cm=6.957e10,
              em_flag=4, s_max=30, use_bvec=True, image_shape=(w["n_pix_y"], w["n_pix_x"]))
    fps = w["freq_params"]
    times = {"render_map": [], "render_map_diag": []}
    with RaySession(0) as ses:
        g3 = (c["x_grid"], c["y_grid"], c["z_grid"])
        ses.set_omega_cube(c["omega_pe"], *g3)
        ses.set_field_cubes(*g3, c["ne"], c["te"], c["b"], c["bx"], c["by"], c["bz"])
        calls = {"render_map": lambda: ses.render_map(xs, ys, zs, fps, **kw),
                 "render_map_diag": lambda: ses.render_map_diag(xs, ys, zs, fps, **kw)}
        for _ in range(a.warmup):
            for f in calls.values():
                f()
        same = None
        for rep in range(a.reps):
            order = list(calls) if rep % 2 == 0 else list(calls)[::-1]
            outs = {}
            for name in order:
                t0 = time.perf_counter()
                outs[name] = calls[name]()
                times[name].append(time.perf_counter() - t0)
            if same is None:
                same = bool(np.array_equal(outs["render_map"][0], outs["render_map_diag"][0]))
    med = {k: float(np.median(v)) for k, v in times.items()}
    res = dict(workload="config4 bench variant", reps=a.reps, warmup=a.warmup,
               render_map_s=med["render_map"], render_map_diag_s=med["render_map_diag"],
               ratio=med["render_map_diag"] / med["render_map"],
               render_map_all_s=times["render_map"], render_map_diag_all_s=times["render_map_diag"],
               tb_bit_identical=same, card=card())
    print(f"render_map      {med['render_map']:.4f} s  (median of {a.reps})")
    print(f"render_map_diag {med['render_map_diag']:.4f} s")
    print(f"ratio           {res['ratio']:.3f}")
    print(f"card            {res['card']}")
    print(json.dumps(res))
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
