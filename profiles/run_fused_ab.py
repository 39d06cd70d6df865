#!/usr/bin/env python
"""A/B of builds of the library on the flagship workload, alternated in one run.

    --lib NAME=PATH, repeated: the first is the reference (e.g. the parent commit's libdcd_b200.so, built from that commit's
    tree); default for the last one: this tree's dcd_b200/libdcd_b200.so as "new"

Each repetition runs `python bench.py --config kitti_val <bench args>` once per build, in the order given, with DCD_B200_LIB
set, and keeps its JSON line: objects/s (`value`), `roofline.avg_launch_ms` and `roofline.frac`.  Then, once per build: the
other configs (--configs), `--dump-outputs` of kitti_val compared array for array with the reference's (numpy.array_equal),
and with --trace NAME=PATH (trace builds, `python -m dcd_b200.build --trace`) the in-kernel timeline of CTA 0
(profiles/trace_fused.py): median cycles of a converter step (warp 0, step start to step start inside a layer: tags x100 ->
x100) and of a tile on the MMA warp (operand ready to operand ready: tags 200 + t), each over all steps of the traced launch.

    python profiles/run_fused_ab.py --lib parent=A.so [--lib new=B.so ...] [--reps 3] [--configs kitti_val_full sweep1m]
                                    [--trace parent=A_trace.so --trace new=B_trace.so] [--out FILE.json] [-- bench args]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")
LIB = os.path.join(ROOT, "dcd_b200", "libdcd_b200.so")


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return "unavailable: %s" % e


def run(cmd, lib):
    env = dict(os.environ, DCD_B200_LIB=os.path.abspath(lib))
    res = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=ROOT)
    if res.returncode != 0:
        raise RuntimeError("%s failed (%d):\n%s\n%s" % (" ".join(cmd), res.returncode, res.stdout[-4000:], res.stderr[-4000:]))
    return res.stdout


def bench(lib, args):
    out = run([sys.executable, BENCH] + args, lib)
    line = [ln for ln in out.splitlines() if ln.startswith("{")][-1]
    r = json.loads(line)
    roof = r.get("roofline", {})
    return {"value": r["value"], "avg_launch_ms": roof.get("avg_launch_ms"), "frac": roof.get("frac")}


def trace_summary(lib):
    out = run([sys.executable, os.path.join(ROOT, "profiles", "trace_fused.py")], lib)
    ev = {0: [], 1: []}
    for ln in out.splitlines():
        p = ln.split()
        if len(p) == 4 and p[0] in ("0", "1"):
            ev[int(p[0])].append((int(p[1]), int(p[3])))
    conv = [t1 - t0 for (a0, t0), (a1, t1) in zip(ev[0], ev[0][1:])
            if a0 % 1000 // 100 == 1 and a1 % 1000 // 100 == 1 and a0 < 3000 and a1 < 3000 and a1 // 1000 == a0 // 1000 and a1 == a0 + 1]
    tiles = [e for e in ev[1] if 200 <= e[0] < 300]
    mma = [t1 - t0 for (a0, t0), (a1, t1) in zip(tiles, tiles[1:]) if a1 == a0 + 1]
    return {"converter_step_cycles_median": statistics.median(conv) if conv else None, "converter_steps": len(conv),
            "mma_tile_cycles_median": statistics.median(mma) if mma else None, "mma_tiles": len(mma)}


def pairs(items):
    out = {}
    for it in items:
        name, _, path = it.partition("=")
        out[name] = path
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], help="NAME=PATH; the first is the reference")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--configs", nargs="*", default=[])
    ap.add_argument("--trace", action="append", default=[], help="NAME=PATH of a trace build")
    ap.add_argument("--out")
    ap.add_argument("bench_args", nargs=argparse.REMAINDER)
    args = ap.parse_args()
    extra = [a for a in args.bench_args if a != "--"]
    libs = pairs(args.lib)
    if len(libs) < 2:
        libs.setdefault("new", LIB)
    names = list(libs)
    ref = names[0]
    rep = {"card": card(), "libs": libs, "bench_args": extra, "kitti_val": {k: [] for k in names}}
    for i in range(args.reps):
        for k in names:
            r = bench(libs[k], ["--config", "kitti_val"] + extra)
            rep["kitti_val"][k].append(r)
            print("rep %d %s kitti_val %.1f objects/s  launch %.3f ms  frac %.4f" % (i, k, r["value"], r["avg_launch_ms"], r["frac"]),
                  flush=True)
    if args.reps > 0:
        v = {k: [r["value"] for r in rep["kitti_val"][k]] for k in names}
        rep["summary"] = {k: {"median": statistics.median(v[k]), "gain": statistics.median(v[k]) / statistics.median(v[ref]) - 1.0,
                              "min_over_ref_max": min(v[k]) / max(v[ref])} for k in names}
        print(json.dumps(rep["summary"]), flush=True)
    for cfg in args.configs:
        rep[cfg] = {}
        for k in names:
            rep[cfg][k] = bench(libs[k], ["--config", cfg] + extra)
            print("%s %s %.1f objects/s" % (cfg, k, rep[cfg][k]["value"]), flush=True)
    with tempfile.TemporaryDirectory() as tmp:
        dumps = {}
        for k in names:
            d = os.path.join(tmp, k)
            bench(libs[k], ["--config", "kitti_val", "--dump-outputs", d] + extra)
            dumps[k] = {f: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d)) if f.endswith(".npy")}
        rep["outputs_equal"] = {k: {f: bool(np.array_equal(dumps[ref][f], dumps[k].get(f))) for f in dumps[ref]} for k in names[1:]}
        print("outputs equal to %s:" % ref, rep["outputs_equal"], flush=True)
    traces = pairs(args.trace)
    if traces:
        rep["trace"] = {k: trace_summary(lib) for k, lib in traces.items()}
        print("trace:", json.dumps(rep["trace"]), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rep, f, indent=1)


if __name__ == "__main__":
    main()
