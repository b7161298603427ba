#!/usr/bin/env python
"""Benchmark of the per-ray hot path (BASELINE.json: ray-steps/s and full-map wall time incl. GRFF at
1/2/4/8 B200 next to the host CPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   # this repo's CUDA path
    python bench.py --impl reference [...]                       # the reference's CPU algorithm (oracle port)

A "step" is one full ray-traced GR+FF map through the fused kernel (trace + sample + transfer, theta from the
B vector, cross-sections traced, rays re-traced per frequency with the publication drivers' presets):

  N = 1   BASELINE config 4: 512^2 pixels, 256^3 cube {n_e, T, B vector}, 8 log-spaced frequencies 75 MHz-1.5 GHz.
  N > 1   BASELINE config 5, STRONG scaling: 2048^2 pixels, 512^3 cube built on the GPU from a spherical model,
          16 frequencies 20-300 MHz; one process per GPU (torchrun), cube replicated, image rows dealt to the
          ranks (rtgrff_shard_rows), the slabs gathered on rank 0 through the library's NCCL entry
          (rtgrff_gather_image) every step.
  `--config c4|c5|c3` overrides (c4 / c3 at N > 1 = weak scaling: 512 x 512N pixels over the same field of view).

value    nominal ray-steps (n_rays x sum_f n_steps_f; one ray-step = one RK4 advance of a central ray, its two
         cross-section rays ride along) / device time, inputs resident in HBM; render + image gather.
e2e      the same through the public API with HOST inputs: H2D of the cubes (config 4: pinned numpy cubes;
         config 5: the spherical model, resampled on the GPU) and ray starts, and the D2H of the T_b / V/I
         maps into page-locked host memory on rank 0, inside the timed region every step.
parity   max |dr| [R_sun], max rel dT_b, max |d(V/I)| of this very run's map against the CPU oracle chain on a
         pixel sub-sample (oracle/parity.py; BASELINE.md 4.4).
roofline bound = "issue": executed warp-instructions per second against the SM issue peak (4 schedulers x 148
         SMs x 1 instruction / cycle at the sampled SM clock); see DESIGN.md 4.1 for why no memory level binds.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

from raytracinggrff_b200 import synthetic  # noqa: E402

R_SUN_CM = 6.957e10
BYTES_PER_RAY_STEP_CS = 1536      # SURVEY.md §8d: 3 RK4 x 4 RHS x 8 corners x 16 B
BYTES_PER_RAY_STEP_NOCS = 512
N_SM = 148


def workload(config: str, n_gpus: int):
    if config == "auto":
        config = "c4" if n_gpus == 1 else "c5"
    if config == "c4":
        w = dict(name="config4", grid_n=256, extent=3.0, n_pix_x=512, n_pix_y=512 * n_gpus, x_fov=1.44,
                 z_obs=3.0, f0=75e6, f1=1.5e9, n_freq=8, scaling="weak")
    elif config == "c5":
        w = dict(name="config5", grid_n=512, extent=4.0, n_pix_x=2048, n_pix_y=2048, x_fov=2.8, z_obs=4.0,
                 f0=20e6, f1=300e6, n_freq=16, scaling="strong")
    elif config == "c3":
        w = dict(name="config3", grid_n=128, extent=3.0, n_pix_x=64, n_pix_y=64 * n_gpus, x_fov=1.44, z_obs=3.0,
                 f0=75e6, f1=75e6, n_freq=1, scaling="weak")
    else:
        raise SystemExit(f"unknown --config {config}")
    step = np.log10(w["f1"] / w["f0"]) / max(w["n_freq"] - 1, 1)
    freqs = synthetic.log_frequencies(w["f0"], w["n_freq"], step)
    if config == "c3":
        fps = [dict(freq_hz=75e6, dt=6e-3, n_steps=5000, record_stride=10)]
    else:
        fps = [dict(freq_hz=float(f), **synthetic.frequency_scaled_params(float(f))) for f in freqs]
    w["freq_params"] = fps
    w["log_step"] = step
    w["key"] = config
    return w


def rays_of(w, idx=None):
    xs, ys, zs, _ = synthetic.ray_launch_geometry(w["n_pix_x"], w["x_fov"], w["z_obs"], N_pix_y=w["n_pix_y"])
    if idx is not None:
        xs, ys, zs = xs[idx], ys[idx], zs[idx]
    return xs, ys, zs


def pixel_area(w):
    # pixel area (script/resample_with_ray_tracing.py:360-363); a weak-scaled N>1 map samples the same field of
    # view more finely in y
    dx = 2 * w["x_fov"] / w["n_pix_x"] * R_SUN_CM
    dy = 2 * w["x_fov"] / w["n_pix_y"] * R_SUN_CM
    return dx * dy


def host_cube(w):
    """The analytic corona on the workload's grid as host arrays (float64 omega_pe, float32 fields), built in
    x-slabs so that a 512^3 cube needs 5 GB instead of 20."""
    n, e = w["grid_n"], w["extent"]
    if n <= 256:
        c = synthetic.corona_cube(n, e, active_region=True)
        for k in ("ne", "te", "b", "bx", "by", "bz"):
            c[k] = c[k].astype(np.float32)
        return c
    out = None
    for i0 in range(0, n, 32):
        part = synthetic.corona_cube(n, e, active_region=True, x_slice=slice(i0, min(n, i0 + 32)))
        if out is None:
            out = {k: (np.empty((n, n, n), dtype=np.float64 if k == "omega_pe" else np.float32)
                       if np.ndim(v) == 3 else v) for k, v in part.items()}
        for k, v in part.items():
            if np.ndim(v) == 3:
                out[k][i0:i0 + v.shape[0]] = v
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        try:
            for line in open(self.path):
                p = [t.strip() for t in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1])); smax.append(float(p[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(smax)), reasons=sorted(reasons), samples=len(sm))
        return out


# ----------------------------------------------------------------------------------------- CPU legs ----
def cpu_chain_step(w, cube, sel, n_threads=None):
    """The reference's CPU algorithm (oracle port) for the SAME physics as the GPU arm on a pixel sub-sample:
    ray_trace -> sampler -> Parms with theta from B -> GET_MW per frequency.  Returns (nominal ray-steps, seconds)."""
    from oracle import oracle
    oracle.set_num_threads(n_threads)
    xs, ys, zs = rays_of(w, sel)
    area = pixel_area(w)
    nominal = 0
    t0 = time.perf_counter()
    for p in w["freq_params"]:
        oracle.chain_bvec(cube, p["freq_hz"], p["dt"], p["n_steps"], p["record_stride"], xs, ys, zs, area, 4, 30,
                          cache_gradient=True)
        nominal += len(xs) * p["n_steps"]
    return nominal, time.perf_counter() - t0


def reference_numpy_timing(cube, w, budget_rays=4096, n_steps=150):
    """The UNMODIFIED reference package (baseline/_ref, installed by baseline/install_ref.sh) on the host cores:
    ray_trace (build_rays.py:128-248) single-process on config 3's ray count, and its own parallel mode — contiguous
    ray chunks over a ProcessPoolExecutor with the cube pickled to every worker
    (script/resample_with_ray_tracing.py:42-61, :333-352) — plus sample_model_with_rays('cpu').  Bounded: n_steps steps."""
    ref = ROOT / "baseline" / "_ref"
    if not (ref / "raytracingGRFF").is_dir():
        return {"unavailable": "baseline/_ref is not installed (sh baseline/install_ref.sh <raytracingGRFF checkout>)"}
    code = r"""
import json, os, sys, time
import numpy as np
from concurrent.futures import ProcessPoolExecutor
sys.path[:0] = [%r, %r, %r]
from raytracingGRFF.build_rays import ray_trace
from raytracingGRFF.gpu_raytrace import sample_model_with_rays
from raytracinggrff_b200 import synthetic
n_rays, n_steps, grid_n, extent = %d, %d, %d, %r
c = synthetic.corona_cube(grid_n, extent, active_region=True)
n_side = int(round(n_rays ** 0.5))
xs, ys, zs, kv = synthetic.ray_launch_geometry(n_side, 1.44, 3.0)
args = (c["omega_pe"], c["x_grid"], c["y_grid"], c["z_grid"], 75e6)
def chunk(a):
    s, e = a
    return ray_trace(*args, xs[s:e], ys[s:e], zs[s:e], kv[s:e], 6e-3, n_steps, 10, trace_crosssections=True, perturb_ratio=2)
def main():
    out = {"rays": len(xs), "n_steps": n_steps, "cube": grid_n}
    t0 = time.perf_counter(); r, cs = chunk((0, len(xs))); t1 = time.perf_counter() - t0
    out["ray_trace_single_process_ray_steps_per_s"] = len(xs) * n_steps / t1
    nw = os.cpu_count() or 1
    size = (len(xs) + nw - 1) // nw
    chunks = [(s, min(s + size, len(xs))) for s in range(0, len(xs), size)]
    t0 = time.perf_counter()
    with ProcessPoolExecutor(max_workers=nw) as ex:
        res = list(ex.map(chunk, chunks))
    r2 = np.concatenate([q[0] for q in res], axis=1)
    t2 = time.perf_counter() - t0
    assert np.array_equal(r, r2)
    out["ray_trace_process_pool_ray_steps_per_s"] = len(xs) * n_steps / t2
    out["process_pool_workers"] = nw
    t0 = time.perf_counter()
    smp = sample_model_with_rays("cpu", c["x_grid"], c["y_grid"], c["z_grid"], c["ne"], c["te"], c["b"], r, np.array(cs),
                                 np.column_stack([xs, ys, zs]), 6.957e10, verbose=False)
    out["sampler_samples_per_s"] = smp["ne"].size / (time.perf_counter() - t0)
    print(json.dumps(out))
if __name__ == "__main__":
    main()
""" % (str(ref), str(ROOT / "baseline" / "mpl_stub"), str(ROOT), budget_rays, n_steps, w["grid_n"], w["extent"])
    try:
        with tempfile.NamedTemporaryFile("w", suffix=".py", delete=False) as f:
            f.write(code)
        env = dict(os.environ)
        env.pop("OMP_NUM_THREADS", None)
        p = subprocess.run([sys.executable, f.name], capture_output=True, text=True, timeout=240, env=env)
        os.unlink(f.name)
        if p.returncode != 0:
            return {"unavailable": "reference run failed: " + p.stderr.strip().splitlines()[-1][:200]}
        d = json.loads(p.stdout.strip().splitlines()[-1])
        d["what"] = ("unmodified raytracingGRFF.build_rays.ray_trace (numpy/scipy, cross-sections on, 75 MHz, dt 6e-3) and "
                     "gpu_raytrace.sample_model_with_rays('cpu'); GRFF itself is an absent third-party binary")
        return d
    except Exception as e:  # noqa: BLE001
        return {"unavailable": f"{type(e).__name__}: {e}"[:200]}


def run_reference(args, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle, parity
    oracle.build()
    cores = oracle.set_num_threads(None)          # all host cores, whatever the launcher put in OMP_NUM_THREADS
    w1 = workload(w["key"], 1) if w["scaling"] == "weak" else w   # the CPU sample is taken from the square N=1 image
    cube = host_cube(w1)
    stride = args.cpu_sample_stride or (16 if w1["name"] != "config5" else 128)
    sel = parity.subsample(w1["n_pix_x"], w1["n_pix_y"], stride)
    for _ in range(args.warmup):
        cpu_chain_step(w1, cube, sel[:: 8])
    tot_steps, tot_t = 0, 0.0
    for _ in range(args.steps):
        n, t = cpu_chain_step(w1, cube, sel)
        tot_steps += n
        tot_t += t
    value = tot_steps / tot_t
    sample = (f"{len(sel)} rays (every {stride}th pixel in x and y of the {w1['n_pix_x']}x{w1['n_pix_y']} image) x "
              f"{w1['n_freq']} freqs, full n_steps; oracle ray_trace + sampler + GET_MW with theta from B (GR+FF): the GPU "
              f"arm's physics; cube preparation (np.gradient) amortised as over a full map")
    line = {
        "impl": "reference", "metric": "ray_steps_per_s", "value": value, "unit": "ray-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(args.steps, 1), "higher_is_better": True,
        "scaling": w["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(w, args),
        "cpu_baseline": {"value": value, "unit": "ray-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "ray-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def config_dict(w, args):
    spherical = w["name"] == "config5" or getattr(args, "spherical", False)
    return {
        "workload": f"BASELINE {w['name']}: {w['n_pix_x']}x{w['n_pix_y']} px, {w['grid_n']}^3 cube, {w['n_freq']} freqs "
                    f"{w['f0'] / 1e6:g}-{w['f1'] / 1e6:g} MHz, GR+FF, cross-sections on, fused trace+sample+transfer",
        "per_freq": [[p["freq_hz"], p["dt"], p["n_steps"], p["record_stride"]] for p in w["freq_params"]],
        "sharding": "rows dealt round-robin to the ranks in groups of 8 (rtgrff_shard_rows), cube replicated, slabs "
                    "gathered on rank 0 over NCCL (rtgrff_gather_image)",
        "thread_order": "4x8-pixel tiles per warp (ray_order), results in row-major ray order",
        "l2": f"cubes (3 x {16 * w['grid_n'] ** 3 / 1e6:.0f} MB float4 + {128 * w['grid_n'] ** 3 / 1e6:.0f} MB cell-major polynomial "
              "cube) exceed the 126 MB L2; no flush between steps",
        "cubes": "built on the GPU from a spherical (phi,lat,r) model" if spherical
                 else "analytic corona, uploaded from pinned host memory",
        "precision": "FP64 ray state and intensity accumulation, FP32 cube storage, cell-relative RHS and voxel opacities "
                     "(FP64 fallback near the mode cut-offs), FP32 angle to B",
        "cross_sections": "pencil rays traced on recorded steps only (the reference computes S at every step but "
                          "outputs only recorded steps, build_rays.py:241-244); RTGRFF_CS_EVERY_STEP=1 restores it",
    }


DUMP_BYTES = 64_000_000
NPY_HEADER_ROOM = 4096       # for the (at most three) .npy headers, so that the files on disk stay within the budget


def dump_outputs(image, n_freq, out_dir, max_bytes=DUMP_BYTES):
    """Write a rendered map as the caller of render_map receives it: tb.npy (T_b [K]) and vi.npy (V/I), float64,
    one plane per frequency, from `image` = [tb planes | vi planes][row][col] (a torch tensor, any device).  A map
    whose files would exceed max_bytes is replaced by the same fixed, seeded sample of pixels from every plane;
    pixel_index.npy then holds their row-major indices into the image.  Returns the names written."""
    import torch
    planes, ny, nx = image.shape
    out = {}
    data_bytes = max_bytes - NPY_HEADER_ROOM
    if image.numel() * 8 > data_bytes:
        m = data_bytes // (planes * 8 + 8)
        idx = np.sort(np.random.default_rng(0).choice(ny * nx, m, replace=False))
        image = image.reshape(planes, ny * nx)[:, torch.from_numpy(idx).to(image.device)]
        out["pixel_index"] = idx.astype(np.float64)
    host = image.cpu().numpy()
    out["tb"], out["vi"] = host[:n_freq], host[n_freq:]
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in out.items():
        np.save(out_dir / f"{name}.npy", a)
    return sorted(out)


def lib_fingerprint():
    """sha1 of the kernel sources (csrc/*.cuh; the .cu file is host staging): ties a bench line to the ncu captures
    under profiles/."""
    h = hashlib.sha1()
    for p in sorted((ROOT / "raytracinggrff_b200" / "csrc").glob("*.cuh")):
        h.update(p.read_bytes())
    return h.hexdigest()[:12]


# ----------------------------------------------------------------------------------------- CUDA arm ----
class MapRunner:
    """One workload on this rank: inputs, upload, render (+ gather), timing helpers."""

    def __init__(self, w, args, ses, torch, dist, rdist, world, rank, dev):
        self.w, self.ses, self.torch, self.dist, self.world, self.rank, self.dev = w, ses, torch, dist, world, rank, dev
        self.spherical = w["name"] == "config5" or args.spherical
        self.rows, self.mr = rdist.c_shard_rows(w["n_pix_y"], world, rank)
        idx = (self.rows[:, None] * w["n_pix_x"] + np.arange(w["n_pix_x"])[None, :]).ravel()
        self.xs, self.ys, self.zs = rays_of(w, idx)
        self.nf = w["n_freq"]
        self.area = pixel_area(w)
        self.fps = w["freq_params"]
        self.n_local = len(self.xs)
        self.nominal_total = w["n_pix_x"] * w["n_pix_y"] * sum(p["n_steps"] for p in self.fps)
        self.cube = None
        if self.spherical:
            self.model = synthetic.spherical_corona(200, 140, 160, r_max=1.8 * w["extent"], active_region=True)
            g = np.linspace(-w["extent"], w["extent"], w["grid_n"])
            self.grids = (g, g.copy(), g.copy())
            self.h2d_cubes = sum(v.data.nbytes + v.phi.nbytes + v.lat.nbytes + v.r.nbytes for v in self.model.values())
        else:
            self.cube = host_cube(w)

            def pinned(a):
                t = torch.empty(a.shape, dtype=torch.float64 if a.dtype == np.float64 else torch.float32, pin_memory=True)
                t.copy_(torch.from_numpy(np.ascontiguousarray(a)))
                return t.numpy()
            self.h_w = pinned(self.cube["omega_pe"])
            self.h_f = {k: pinned(self.cube[k]) for k in ("ne", "te", "b", "bx", "by", "bz")}
            self.grids = (self.cube["x_grid"], self.cube["y_grid"], self.cube["z_grid"])
            self.h2d_cubes = self.h_w.nbytes + sum(a.nbytes for a in self.h_f.values())
        nx, ny = w["n_pix_x"], w["n_pix_y"]
        self.slab = torch.zeros((2 * self.nf, self.mr, nx), dtype=torch.float64, device=dev)
        self.image = torch.zeros((2 * self.nf, ny, nx), dtype=torch.float64, device=dev) if rank == 0 else None
        self.host_image = torch.empty((2 * self.nf, ny, nx), dtype=torch.float64, pin_memory=True) if rank == 0 else None
        self.stats = {}
        self.h2d = self.h2d_cubes + 3 * 8 * self.n_local
        self.d2h = 2 * self.nf * nx * ny * 8 if rank == 0 else 0

    def upload(self):
        if self.spherical:
            self.ses.set_model_from_spherical(self.model, *self.grids, phi0_offset=0.0, want_bvec=True)
        else:
            self.ses.set_omega_cube(self.h_w, *self.grids)
            f = self.h_f
            self.ses.set_field_cubes(*self.grids, f["ne"], f["te"], f["b"], f["bx"], f["by"], f["bz"])

    def render(self, to_host=False):
        """The rank's rows into its slab, then the gather on rank 0 (device image, or the pinned host image)."""
        nx = self.w["n_pix_x"]
        kw = dict(trace_crosssections=True, perturb_ratio=2.0, pixel_area_cm2=self.area, r_sun_cm=R_SUN_CM, em_flag=4,
                  s_max=30, use_bvec=True, image_shape=(len(self.rows), nx))
        if len(self.rows) == self.mr:
            tgt = self.slab
        else:    # ragged share: the kernel writes planes of len(rows) rows; place them into the padded slab
            tgt = self.torch.empty((2 * self.nf, len(self.rows), nx), dtype=self.torch.float64, device=self.dev)
        _, _, st = self.ses.render_map(self.xs, self.ys, self.zs, self.fps,
                                       out_device_ptrs=(tgt[:self.nf].data_ptr(), tgt[self.nf:].data_ptr()), **kw)
        if tgt is not self.slab:
            self.slab[:, :len(self.rows)] = tgt
        self.stats = dict(st, kernel_ms=self.ses.ctx.last_kernel_ms)
        ny = self.w["n_pix_y"]
        if to_host:
            self.ses.gather_image(self.slab.data_ptr(), 2 * self.nf, ny, nx, root=0,
                                  out=self.host_image.numpy() if self.rank == 0 else None)
        else:
            self.ses.gather_image(self.slab.data_ptr(), 2 * self.nf, ny, nx, root=0,
                                  out_device_ptr=self.image.data_ptr() if self.rank == 0 else None)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, steps, to_host=False, reupload=False):
        """(ms per step on the device, max over ranks; wall s per step, max over ranks; mean kernel ms, max over ranks)"""
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        kms = []
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            if reupload:
                self.upload()
            self.render(to_host=to_host)
            kms.append(self.stats["kernel_ms"])
        e1.record()
        self.barrier()
        wall = (time.perf_counter() - t0) / steps
        t = torch.tensor([e0.elapsed_time(e1) / steps, wall * 1e3, float(np.mean(kms))], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]) * 1e-3, float(t[2])

    def totals(self):
        torch = self.torch
        t = torch.tensor([float(self.stats["active_ray_steps"]), float(self.stats["pencil_steps"]),
                          float(self.stats["valid_samples"])], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t[0]), float(t[1]), float(t[2])

    def host_cube_for_oracle(self):
        """The very cubes the device holds, on the host, for the oracle."""
        if self.cube is not None:
            return self.cube
        c = self.ses.export_cubes(omega_pe=True, fields=True, bvec=True)
        c.update(x_grid=self.grids[0], y_grid=self.grids[1], z_grid=self.grids[2])
        return c


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="auto", choices=["auto", "c3", "c4", "c5"])
    ap.add_argument("--cpu-sample-stride", type=int, default=0, help="pixel stride of the CPU / parity sub-sample (0: per workload)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the oracle run (then no parity block either)")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary workloads (configs 1-3, the other scaling mode, the numpy reference)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--spherical", action="store_true", help="build the cubes on the GPU from a spherical model")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's T_b and V/I maps to DIR/*.npy "
                    "(float64, at most 64 MB: a larger map is a fixed pixel sample) to compare builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the CUDA arm's maps; the reference arm keeps none")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    w = workload(args.config, args.gpus)
    if args.impl == "reference":
        return run_reference(args, w)

    # keep stdout clean for the single JSON line: anything libraries print there (NCCL's version banner
    # among others) goes to stderr until the result is ready
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    from raytracinggrff_b200 import RaySession, _lib
    from raytracinggrff_b200 import dist as rdist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    # the library works on torch's current stream (handle 0 = the legacy default stream, honoured as such)
    ses = RaySession(context=_lib.Context(local_rank, torch.cuda.current_stream().cuda_stream))
    if world > 1:
        rdist.init_comm(ses)
    else:
        ses.comm_init(1, 0)

    run = MapRunner(w, args, ses, torch, dist, rdist, world, rank, dev)
    run.upload()
    for _ in range(args.warmup):
        run.render()
    # ---- timed region: device-resident inputs ----
    clocks = ClockSampler(local_rank)
    run.barrier()
    clocks.start()
    launches0 = ses.ctx.launch_count
    ms_per_step, _, kernel_ms = run.timed(args.steps)
    clk = clocks.stop()
    launches = ses.ctx.launch_count - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(run.image, run.nf, args.dump_outputs)
    active_total, pencil_total, samples_total = run.totals()
    value = run.nominal_total / (ms_per_step * 1e-3)

    # ---- end to end: host inputs in, host maps out, every step ----
    run.upload(); run.render(to_host=True)
    e2e_ms, e2e_wall, _ = run.timed(args.e2e_steps, to_host=True, reupload=True)
    e2e_t = max(e2e_ms * 1e-3, e2e_wall)
    e2e_value = run.nominal_total / e2e_t
    gpu_map = run.host_image.numpy().copy() if rank == 0 else None      # [tb planes | vi planes][row][col]

    line = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(ROOT / "MEASURED_PEAKS.json"))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        hbm_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
        # ---- the roofline that binds: instruction issue ----
        counters = {}
        try:
            counters = json.load(open(ROOT / "profiles" / "roofline_counters.json")).get(f"{w['key']}", {})
        except Exception:
            pass
        nominal_max_rank = run.mr * w["n_pix_x"] * sum(p["n_steps"] for p in run.fps)
        warp_inst = None
        if counters.get("warp_inst_per_nominal_ray_step"):
            warp_inst = counters["warp_inst_per_nominal_ray_step"] * nominal_max_rank
        sm_mhz = clk.get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0
        issue_peak = 4 * N_SM * sm_mhz * 1e6            # warp-instructions / s: 4 schedulers per SM, 1 per cycle
        achieved = warp_inst / (kernel_ms * 1e-3) if warp_inst else None
        # algorithmic HBM bytes per launch (SURVEY 8d per-unit figures x the units processed): NOT the binding bound
        alg_bytes = (active_total * BYTES_PER_RAY_STEP_NOCS + pencil_total * (BYTES_PER_RAY_STEP_CS - BYTES_PER_RAY_STEP_NOCS)
                     + samples_total * (2 * 128 + 16)) / world
        alg_gbs = alg_bytes / (kernel_ms * 1e-3) / 1e9
        roof = {
            "bound": "issue", "achieved": achieved, "peak": issue_peak, "unit": "warp-inst/s",
            "frac": (achieved / issue_peak) if achieved else None, "traffic": counters.get("dram_bytes_per_launch"),
            "kernel": "render_map_kernel", "kernel_ms": kernel_ms,
            "peak_source": f"4 schedulers x {N_SM} SMs x 1 warp-instruction/cycle x {sm_mhz:.0f} MHz (SM clock sampled during the "
                           "timed region); microbenchmarked issue / FP32 / FP64 / L1 / L2 ceilings: profiles/r2_microbench.json",
            "warp_inst_per_launch": warp_inst,
            "thread_inst_per_active_ray_step": (counters.get("thread_inst_per_nominal_ray_step", 0) * run.nominal_total / active_total)
                                               if counters.get("thread_inst_per_nominal_ray_step") and active_total else None,
            "min_rhs_floor_thread_inst_per_active_ray_step": 55.0 * (4.0 * active_total + 8.0 * pencil_total) / active_total
                                                             if active_total else None,
            "counters_source": counters.get("source"), "counters_lib": counters.get("lib"), "lib": lib_fingerprint(),
            "hbm_algorithmic": {"achieved_gbs": alg_gbs, "peak_gbs": hbm_peak, "frac": alg_gbs / hbm_peak, "binding": False,
                                "peak_source": hbm_src,
                                "note": "512 B x active central steps + 1024 B x pencil steps + 272 B x valid samples per launch / kernel "
                                        "time; served by registers / L1 / L2 (DRAM traffic ~ cube size), so it exceeds the HBM copy peak: "
                                        "not a bound of this kernel"},
        }
        line = {
            "metric": "ray_steps_per_s", "value": value, "unit": "ray-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": w["scaling"],
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_dict(w, args),
            "full_map_wall_s": ms_per_step * 1e-3,
            "nominal_ray_steps_per_step": run.nominal_total, "active_ray_steps_per_step": active_total,
            "active_ray_steps_per_s": active_total / (ms_per_step * 1e-3),
            "pencil_steps_per_step": pencil_total, "valid_samples_per_step": samples_total,
            "clocks": clk,
            "e2e": {"value": e2e_value, "unit": "ray-steps/s", "h2d_bytes_per_step": int(run.h2d),
                    "d2h_bytes_per_step": int(run.d2h), "full_map_wall_s": e2e_t},
            "gpu_launches": int(launches),
            "roofline": roof,
        }

    # ---- parity of this run's map + the CPU baseline (rank 0; the other ranks wait at the next collective) ----
    if rank == 0 and not args.no_cpu_baseline:
        try:
            from oracle import oracle, parity
            oracle.build()
            cores = oracle.set_num_threads(None)
            stride = args.cpu_sample_stride or (16 if w["name"] != "config5" else 128)
            nx, ny = w["n_pix_x"], w["n_pix_y"]
            sel = parity.subsample(nx, ny, stride)
            xs, ys, zs = rays_of(w, sel)
            cube = run.host_cube_for_oracle()
            tb_gpu = gpu_map[:run.nf].reshape(run.nf, -1)[:, sel]
            vi_gpu = gpu_map[run.nf:].reshape(run.nf, -1)[:, sel]
            t0 = time.perf_counter()
            par = parity.map_parity(cube, run.fps, xs, ys, zs, run.area, tb_gpu, vi_gpu, session=ses)
            par["seconds"] = time.perf_counter() - t0
            par["sample"] = f"every {stride}th pixel in x and y ({len(sel)} pixels) x {run.nf} freqs of this run's e2e map"
            line["parity"] = par
            if world == 1:
                # the oracle run that produced the parity numbers IS the CPU baseline: same pixels, same physics
                n, tcpu = par["oracle_nominal_ray_steps"], par["oracle_seconds"]
                line["cpu_baseline"] = {
                    "value": n / tcpu, "unit": "ray-steps/s", "cores": cores, "kind": "port",
                    "sample": f"{len(sel)} rays (every {stride}th pixel in x and y) x {run.nf} freqs, full n_steps; oracle ray_trace + "
                              f"sampler + GET_MW with theta from B (the GPU arm's physics; cube preparation amortised as over a "
                              f"full map), {tcpu:.1f} s"}
        except Exception as e:  # noqa: BLE001  (the other ranks wait at the next collective: never die here)
            line["parity"] = {"error": f"{type(e).__name__}: {e}"[:300]}

    # ---- secondary workloads ----
    if not args.no_extras:
        extras = {}
        other_key = "c5" if w["key"] == "c4" else ("c4" if w["key"] == "c5" else None)
        if other_key:
            try:
                w2 = workload(other_key, world)
                del run.slab, run.image, run.host_image
                run2 = MapRunner(w2, args, ses, torch, dist, rdist, world, rank, dev)
                run2.upload()
                run2.render()
                ms2, _, k2 = run2.timed(2)
                e2e2_ms, e2e2_wall, _ = run2.timed(1, to_host=True, reupload=True)
                act2, _, _ = run2.totals()
                extras[f"{w2['name']}_{w2['scaling']}"] = {
                    "workload": config_dict(w2, args)["workload"], "n_gpus": world, "scaling": w2["scaling"], "steps": 2,
                    "value": run2.nominal_total / (ms2 * 1e-3), "unit": "ray-steps/s", "full_map_wall_s": ms2 * 1e-3,
                    "kernel_ms": k2, "e2e_full_map_wall_s": max(e2e2_ms * 1e-3, e2e2_wall),
                    "active_ray_steps_per_step": act2, "nominal_ray_steps_per_step": run2.nominal_total}
                del run2
            except Exception as e:  # noqa: BLE001  (a secondary number must not take the headline down)
                extras["other_config_error"] = f"{type(e).__name__}: {e}"[:300]
        if rank == 0 and world == 1:
            try:
                sys.path.insert(0, str(ROOT / "scripts"))
                import stage_bench
                extras["stages_configs_1_to_3"] = stage_bench.run_all(ses, quick=True)
            except Exception as e:  # noqa: BLE001
                extras["stages_error"] = f"{type(e).__name__}: {e}"[:300]
            if not args.no_cpu_baseline:
                extras["reference_numpy"] = reference_numpy_timing(None, workload("c3", 1))
        if rank == 0:
            line["extras"] = extras

    if rank == 0:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        ses.comm_destroy()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
