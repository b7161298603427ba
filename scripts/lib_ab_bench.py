"""Two or more builds of the library on the same workloads in one run, alternated: is a kernel change faster, and does
it compute the same maps?

    python scripts/lib_ab_bench.py --lib old=build/libs/lib_old.so --lib new=raytracinggrff_b200/librtgrff_b200.so
        [--rounds 3] [--steps 3] [--warmup 3] [--c5] [--stage] [--freq] [--out result.json] [--work DIR]

Each round runs `bench.py --config c4` (one GPU, no extras, no oracle) once per build, in alternating order, each in a
process of its own with RTGRFF_LIB naming the build.  Per build: the per-map times (`ms_per_step`) of every round and
their median, and whether its `--dump-outputs` T_b and V/I maps are np.array_equal to the first build's.
--c5: config 5 on one GPU once per build (a fixed pixel sample of its maps is compared).  --stage:
scripts/stage_bench.py (configs 1-3 stage by stage) once per build.  --freq: scripts/freq_bench.py (each config-4
frequency alone) once per build.  The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "scripts"))

from diag_bench import card  # noqa: E402


def run(cmd, lib, timeout):
    env = dict(os.environ, RTGRFF_LIB=str(Path(lib).resolve()))
    res = subprocess.run([sys.executable, *cmd], cwd=ROOT, env=env, capture_output=True, text=True, timeout=timeout)
    if res.returncode != 0:
        raise RuntimeError(f"{' '.join(cmd)} with {lib} exited {res.returncode}:\n{res.stderr[-4000:]}")
    return res.stdout


def bench_line(stdout):
    return json.loads([ln for ln in stdout.splitlines() if ln.startswith("{")][-1])


def same_maps(a: Path, b: Path):
    out = {}
    for name in ("tb", "vi", "pixel_index"):
        fa, fb = a / f"{name}.npy", b / f"{name}.npy"
        if fa.exists() or fb.exists():
            out[name] = bool(fa.exists() and fb.exists() and np.array_equal(np.load(fa), np.load(fb), equal_nan=True))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", required=True, metavar="NAME=PATH")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--c5", action="store_true")
    ap.add_argument("--stage", action="store_true")
    ap.add_argument("--freq", action="store_true")
    ap.add_argument("--out")
    ap.add_argument("--work", help="directory for the dumped maps (default: a temporary one)")
    args = ap.parse_args()
    libs = dict(s.split("=", 1) for s in args.lib)
    work = Path(args.work or tempfile.mkdtemp(prefix="lib_ab_"))
    res = dict(card=card(), libs=libs, rounds=args.rounds, steps=args.steps, warmup=args.warmup,
               c4={k: dict(ms_per_map=[]) for k in libs})
    print(json.dumps(res["card"]), flush=True)
    names = list(libs)
    first = names[0]
    for r in range(args.rounds):
        for name in (names if r % 2 == 0 else names[::-1]):
            d = work / f"c4_{name}"
            line = bench_line(run(["bench.py", "--gpus", "1", "--config", "c4", "--steps", str(args.steps), "--warmup",
                                   str(args.warmup), "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(d)],
                                  libs[name], 900))
            res["c4"][name]["ms_per_map"].append(line["ms_per_step"])
            print(f"round {r} {name}: config 4 {line['ms_per_step']:.2f} ms per map", flush=True)
    for name in names:
        c = res["c4"][name]
        c["median_ms"] = float(np.median(c["ms_per_map"]))
        c["same_maps_as_" + first] = same_maps(work / f"c4_{first}", work / f"c4_{name}")
        c["ratio_to_" + first] = c["median_ms"] / res["c4"][first]["median_ms"]
    if args.c5:
        res["c5"] = {}
        for name in names:
            d = work / f"c5_{name}"
            line = bench_line(run(["bench.py", "--gpus", "1", "--config", "c5", "--steps", "1", "--warmup", "3",
                                   "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(d)], libs[name], 1800))
            res["c5"][name] = dict(ms_per_map=line["ms_per_step"], **{"same_maps_as_" + first: same_maps(work / f"c5_{first}", d)})
            print(f"{name}: config 5 {line['ms_per_step']:.1f} ms per map", flush=True)
    if args.stage:
        res["stage"] = {name: json.loads(run(["scripts/stage_bench.py"], libs[name], 900)) for name in names}
    if args.freq:
        res["freq"] = {}
        for name in names:
            f = work / f"freq_{name}.json"
            run(["scripts/freq_bench.py", "--reps", "3", "--json", str(f)], libs[name], 900)
            res["freq"][name] = dict(json.loads(f.read_text()), lib=libs[name])
    summary = {k: dict(median_ms=v["median_ms"], ratio=v["ratio_to_" + first], same=v["same_maps_as_" + first])
               for k, v in res["c4"].items()}
    print(json.dumps(summary), flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
