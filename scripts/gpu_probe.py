#!/usr/bin/env python
"""Quick GPU probe: parity numbers and raw kernel timings of each stage (development aid)."""
import os
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))     # cases.los_sampler_case: the reference benchmark's fixture
import cases  # noqa: E402
from raytracinggrff_b200 import RaySession, synthetic  # noqa: E402
from oracle import oracle  # noqa: E402


def timeit(fn, n=3):
    fn()
    best = 1e9
    for _ in range(n):
        t0 = time.perf_counter()
        fn()
        best = min(best, time.perf_counter() - t0)
    return best


def main():
    which = sys.argv[1] if len(sys.argv) > 1 else "all"
    ses = RaySession(0)
    if which in ("all", "c3"):
        c = synthetic.corona_cube(128, 3.0)
        ses.set_omega_cube(c["omega_pe"], c["x_grid"], c["y_grid"], c["z_grid"])
        xs, ys, zs, kv = synthetic.ray_launch_geometry(64, 1.44, 3.0)
        r, s, act = ses.trace(75e6, xs, ys, zs, kv, 6e-3, 5000, 10, True, 2.0)
        t0 = time.perf_counter()
        r_ref, cs_ref, act_ref = oracle.ray_trace(c["omega_pe"], c["x_grid"], c["y_grid"], c["z_grid"], 75e6, xs, ys, zs,
                                                  kv, 6e-3, 5000, 10, True, perturb_ratio=2, return_active=True)
        t_cpu = time.perf_counter() - t0
        s_ref = np.array(cs_ref)
        ok = np.isfinite(s_ref)
        print(f"C3 parity: max|dr|={np.nanmax(np.abs(r - r_ref)):.3e}  max rel dS={np.max(np.abs(s[ok]-s_ref[ok])/s_ref[ok]):.3e} "
              f"active gpu/cpu={act}/{act_ref}  oracle {t_cpu:.2f}s ({os.cpu_count()} threads)")
        t = timeit(lambda: ses.trace(75e6, xs, ys, zs, kv, 6e-3, 5000, 10, True, 2.0, fetch=False))
        print(f"C3 trace (cs): {t*1e3:.1f} ms  nominal {4096*5000/t:.3e} ray-steps/s  active {act/t:.3e}")
        t = timeit(lambda: ses.trace(75e6, xs, ys, zs, kv, 6e-3, 5000, 10, False, 2.0, fetch=False))
        print(f"C3 trace (no cs): {t*1e3:.1f} ms  nominal {4096*5000/t:.3e} ray-steps/s")
    if which in ("all", "c4"):
        c = synthetic.corona_cube(256, 3.0)
        ses.set_omega_cube(c["omega_pe"], c["x_grid"], c["y_grid"], c["z_grid"])
        ses.set_field_cubes(c["x_grid"], c["y_grid"], c["z_grid"], c["ne"], c["te"], c["b"])
        xs, ys, zs, kv = synthetic.ray_launch_geometry(512, 1.44, 3.0)
        for f in (75e6, 300e6):
            p = synthetic.frequency_scaled_params(f)
            _, _, act = ses.trace(f, xs, ys, zs, kv, p["dt"], p["n_steps"], max(p["record_stride"], 50), True, 2.0, fetch=False)
            t = timeit(lambda: ses.trace(f, xs, ys, zs, kv, p["dt"], p["n_steps"], max(p["record_stride"], 50), True, 2.0, fetch=False), n=2)
            nom = xs.size * p["n_steps"]
            print(f"C4 trace f={f/1e6:.0f}MHz T={p['n_steps']}: {t*1e3:.1f} ms nominal {nom/t:.3e} active {act/t:.3e} ray-steps/s "
                  f"(alg {act*1536/t/1e9:.0f} GB/s)")
            area = (2 * 1.44 / 512 * 6.957e10) ** 2
            fp = [(f, p["dt"], p["n_steps"], p["record_stride"])]
            _, _, st = ses.render_map(xs, ys, zs, fp, kvec_in_norm=kv, pixel_area_cm2=area)
            t = timeit(lambda: ses.render_map(xs, ys, zs, fp, kvec_in_norm=kv, pixel_area_cm2=area), n=2)
            print(f"C4 fused f={f/1e6:.0f}MHz: {t*1e3:.1f} ms nominal {st['nominal_ray_steps']/t:.3e} active {st['active_ray_steps']/t:.3e} ray-steps/s")
    if which == "c4freq":
        c = synthetic.corona_cube(int(os.environ.get("RTGRFF_G", "256")), 3.0, active_region=True)
        ses.set_omega_cube(c["omega_pe"], c["x_grid"], c["y_grid"], c["z_grid"])
        ses.set_field_cubes(c["x_grid"], c["y_grid"], c["z_grid"], c["ne"], c["te"], c["b"], c["bx"], c["by"], c["bz"])
        xs, ys, zs, kv = synthetic.ray_launch_geometry(512, 1.44, 3.0)
        tile = os.environ.get("RTGRFF_TILE")
        if tile:
            tw, th = (int(t) for t in tile.split("x"))
            perm = synthetic.tile_order(512, 512, tw, th)
            xs, ys, zs = xs[perm], ys[perm], zs[perm]
            print("tile order", tile)
        area = (2 * 1.44 / 512 * 6.957e10) ** 2
        freqs = synthetic.log_frequencies(75e6, 8, np.log10(20.0) / 7)
        combos = (("GR+FF bvec", dict(em_flag=4, use_bvec=True)), ("FF theta90", dict(em_flag=5, use_bvec=False)))
        if os.environ.get("RTGRFF_ALL_VARIANTS"):
            combos += (("FF bvec", dict(em_flag=5, use_bvec=True)), ("GR+FF theta90", dict(em_flag=4, use_bvec=False)),
                       ("GR+FF bvec no-cs", dict(em_flag=4, use_bvec=True, trace_crosssections=False)))
        for label, kw in combos:
            tot = 0.0
            for f in freqs:
                p = synthetic.frequency_scaled_params(float(f))
                fp = [(float(f), p["dt"], p["n_steps"], p["record_stride"])]
                _, _, st = ses.render_map(xs, ys, zs, fp, pixel_area_cm2=area, **kw)
                ms = ses.ctx.last_kernel_ms
                tot += ms
                print(f"{label} f={f/1e6:7.1f} MHz T={p['n_steps']:6d} stride={p['record_stride']}: {ms:7.1f} ms  "
                      f"active {st['active_ray_steps']/ms/1e6:.2f} G ray-steps/s  ({st['active_ray_steps']/st['nominal_ray_steps']:.2f} active)")
            print(f"{label} total {tot:.1f} ms")
    if which == "c4all":
        # the bench call itself: one render_map with all 8 frequencies, 4x8 tiles; device time of the whole call
        c = synthetic.corona_cube(256, 3.0, active_region=True)
        ses.set_omega_cube(c["omega_pe"], c["x_grid"], c["y_grid"], c["z_grid"])
        ses.set_field_cubes(c["x_grid"], c["y_grid"], c["z_grid"], c["ne"], c["te"], c["b"], c["bx"], c["by"], c["bz"])
        xs, ys, zs, kv = synthetic.ray_launch_geometry(512, 1.44, 3.0)
        area = (2 * 1.44 / 512 * 6.957e10) ** 2
        freqs = synthetic.log_frequencies(75e6, 8, np.log10(20.0) / 7)
        fps = [dict(freq_hz=float(f), **synthetic.frequency_scaled_params(float(f))) for f in freqs]
        ms = []
        tile = tuple(int(t) for t in os.environ.get("RTGRFF_TILE", "4x8").split("x"))
        for _ in range(5):
            tb, vi, st = ses.render_map(xs, ys, zs, fps, pixel_area_cm2=area, em_flag=4, use_bvec=True, image_shape=(512, 512),
                                        tile=tile)
            ms.append(ses.ctx.last_kernel_ms)
        print("c4all ms:", " ".join(f"{m:.1f}" for m in ms), " best", min(ms), " checksum", float(tb.sum()), float(np.abs(vi).sum()))
    if which == "ncu_c4f":
        # one fused launch of the bench configuration at one frequency (RTGRFF_FIDX) for ncu
        c = synthetic.corona_cube(256, 3.0, active_region=True)
        ses.set_omega_cube(c["omega_pe"], c["x_grid"], c["y_grid"], c["z_grid"])
        ses.set_field_cubes(c["x_grid"], c["y_grid"], c["z_grid"], c["ne"], c["te"], c["b"], c["bx"], c["by"], c["bz"])
        xs, ys, zs, kv = synthetic.ray_launch_geometry(512, 1.44, 3.0)
        area = (2 * 1.44 / 512 * 6.957e10) ** 2
        f = float(synthetic.log_frequencies(75e6, 8, np.log10(20.0) / 7)[int(os.environ.get("RTGRFF_FIDX", "7"))])
        p = synthetic.frequency_scaled_params(f)
        _, _, st = ses.render_map(xs, ys, zs, [(f, p["dt"], p["n_steps"], p["record_stride"])], pixel_area_cm2=area,
                                  em_flag=4, use_bvec=True)
        print(f, p, st, ses.ctx.last_kernel_ms)
    if which == "tile":
        c = synthetic.corona_cube(256, 3.0)
        ses.set_omega_cube(c["omega_pe"], c["x_grid"], c["y_grid"], c["z_grid"])
        xs, ys, zs, kv = synthetic.ray_launch_geometry(512, 1.44, 3.0)
        p = synthetic.frequency_scaled_params(75e6)
        for tw, th in ((32, 1), (16, 2), (8, 4), (4, 8)):
            perm = synthetic.tile_order(512, 512, tw, th)
            a, b, cz = xs[perm], ys[perm], zs[perm]
            _, _, act = ses.trace(75e6, a, b, cz, None, p["dt"], p["n_steps"], 50, True, 2.0, fetch=False)
            t = timeit(lambda: ses.trace(75e6, a, b, cz, None, p["dt"], p["n_steps"], 50, True, 2.0, fetch=False), n=2)
            print(f"tile {tw}x{th}: {t*1e3:.1f} ms (kernel {ses.ctx.last_kernel_ms:.1f} ms) active {act/t:.3e} ray-steps/s")
    if which in ("ncu_trace", "ncu_fused"):
        c = synthetic.corona_cube(256, 3.0)
        ses.set_omega_cube(c["omega_pe"], c["x_grid"], c["y_grid"], c["z_grid"])
        ses.set_field_cubes(c["x_grid"], c["y_grid"], c["z_grid"], c["ne"], c["te"], c["b"])
        xs, ys, zs, kv = synthetic.ray_launch_geometry(512, 1.44, 3.0)
        f = 75e6
        p = synthetic.frequency_scaled_params(f)
        if which == "ncu_trace":
            _, _, act = ses.trace(f, xs, ys, zs, kv, p["dt"], p["n_steps"], p["record_stride"], True, 2.0, fetch=False)
            print("active", act)
        else:
            area = (2 * 1.44 / 512 * 6.957e10) ** 2
            _, _, st = ses.render_map(xs, ys, zs, [(f, p["dt"], p["n_steps"], p["record_stride"])], kvec_in_norm=kv, pixel_area_cm2=area)
            print(st)
    if which in ("all", "c1"):
        args = cases.los_sampler_case(256, 256, 128, seed=0)
        ses.set_field_cubes(args[0], args[1], args[2], args[3], args[4], args[5])
        t = timeit(lambda: ses.sample(args[6], args[7], args[8], 6.957e10))
        print(f"C1 sampler e2e (H2D+kernel+D2H): {t*1e3:.1f} ms  {256*256*256/t:.3e} samples/s")
    print("launches", ses.ctx.launch_count)


if __name__ == "__main__":
    main()
