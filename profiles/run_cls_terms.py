#!/usr/bin/env python
"""The correspondence loss through the plan (edge_P) vs through its two sums (GMW.transport_terms), GMW/main.py:453-465.

One training step = compute_z -> GMW (depth 12) -> w_cls * correspondence loss + w_reg * reg loss -> backward, on two paths:
    dense  GMW.forward with with_edge_P = True, correspondenceLoss((1 - 2 eye) * P) as the reference writes it
    terms  GMW.transport_terms + dcd_b200.correspondence_loss (no E x E tensor but K)
each eager, and the terms step also replayed from a CUDA graph (GraphedGmwStep), for
    cls        w_cls = 1.0, w_reg = 0.0 (GMW's first 50 epochs, GMW/main.py:313-315)
    cls+reg    w_cls = 0.1, w_reg = 1.0
at n = 73 and b = 8, 64.  The three step kinds of a (b, weights) cell are alternated step by step in one process and timed
with CUDA events around each whole step (it ends in a device synchronise), after warm-up steps of every kind.
Peak memory: torch.cuda.max_memory_allocated of one eager step above what was allocated before it, after empty_cache and
reset_peak_memory_stats.  n = 256, b = 1: one cls step of each path (time and peak); the batch each path's measured
per-object peak allows on the card is total memory // peak (computed, not found by allocation).

    python profiles/run_cls_terms.py [--steps 20] [--warmup 5] [--out FILE.json]
"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import dcd_b200  # noqa: E402
from dcd_b200 import synth  # noqa: E402
from run_kpts_grad import card  # noqa: E402

WEIGHTS = {"cls": (1.0, 0.0), "cls+reg": (0.1, 1.0)}
BATCHES = (8, 64)


def eager_step(model, data, w_cls, w_reg, plan_free):
    k2, k3, rot, gt = data
    model.zero_grad(set_to_none=True)
    Z, idx = dcd_b200.compute_z(k2, k3, rot)
    if plan_free:
        w, terms = model.transport_terms(k2, k3)
        cls = dcd_b200.correspondence_loss(terms)
    else:
        model.with_edge_P = True
        try:
            w, P = model(k2, k3, rot, None)
        finally:
            model.with_edge_P = False
        eye = torch.eye(P.shape[1], device=P.device).expand_as(P)
        cls = ((1.0 - 2.0 * eye) * P).sum(dim=(-2, -1)).mean()
    reg, _ = dcd_b200.compute_reg_loss(Z, w, gt, idx)
    (w_reg * reg + w_cls * cls).backward()


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def peak_bytes(fn):
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def stats(t):
    return {"median": statistics.median(t), "min": min(t), "max": max(t)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert args.steps >= 10 and args.warmup >= 3
    torch.backends.cuda.matmul.allow_tf32 = False
    sd = synth.random_state_dict(7)
    model = dcd_b200.GMW(depth=12).cuda().load_reference_state_dict(sd)
    total = torch.cuda.get_device_properties(0).total_memory
    result = {"card": card(), "total_memory_bytes": total, "steps": args.steps, "warmup": args.warmup, "depth": 12, "n": 73,
              "cells": []}
    for b in BATCHES:
        ob = synth.make_objects(N=b, n=73, seed=11)
        data = (ob.kps_norm.cuda(), ob.kps_3d.cuda(), ob.rot_y.cuda().reshape(-1, 1), ob.gt_depth.cuda())
        for wname, (w_cls, w_reg) in WEIGHTS.items():
            peaks = {path: peak_bytes(lambda: eager_step(model, data, w_cls, w_reg, path == "terms"))
                     for path in ("dense", "terms")}
            graph = dcd_b200.GraphedGmwStep(dcd_b200.GMW(depth=12).cuda().load_reference_state_dict(sd), batch=b, n=73,
                                            cls_weight=w_cls, reg_weight=w_reg)
            kinds = {
                "dense_eager": lambda: eager_step(model, data, w_cls, w_reg, False),
                "terms_eager": lambda: eager_step(model, data, w_cls, w_reg, True),
                "terms_graph": lambda: graph(*data),
            }
            for _ in range(args.warmup):
                for fn in kinds.values():
                    timed(fn)
            times = {k: [] for k in kinds}
            for _ in range(args.steps):
                for k, fn in kinds.items():
                    times[k].append(timed(fn))
            cell = {"b": b, "loss": wname, "w_cls": w_cls, "w_reg": w_reg, "ms": {k: stats(t) for k, t in times.items()},
                    "peak_bytes": peaks}
            cell["ms"]["saved_eager_ms"] = cell["ms"]["dense_eager"]["median"] - cell["ms"]["terms_eager"]["median"]
            cell["peak_saved_bytes"] = peaks["dense"] - peaks["terms"]
            cell["peak_saved_in_bEE_tensors"] = cell["peak_saved_bytes"] / (b * 4 * 2628 * 2628)
            result["cells"].append(cell)
            print("n=73 b=%2d %-7s " % (b, wname) + "  ".join("%s %.3f ms" % (k, cell["ms"][k]["median"]) for k in kinds)
                  + "  peak dense %.0f MB terms %.0f MB (%.2f [b,E,E] tensors less)"
                  % (peaks["dense"] / 1e6, peaks["terms"] / 1e6, cell["peak_saved_in_bEE_tensors"]), flush=True)
            del graph, kinds
    # n = 256, b = 1, cls only: one step of each path (after one warm-up step each), time and peak
    ob = synth.make_objects(N=1, n=256, seed=12)
    data = (ob.kps_norm.cuda(), ob.kps_3d.cuda(), ob.rot_y.cuda().reshape(-1, 1), ob.gt_depth.cuda())
    big = {"n": 256, "b": 1, "loss": "cls"}
    for path in ("dense", "terms"):
        fn = lambda: eager_step(model, data, 1.0, 0.0, path == "terms")  # noqa: E731
        peak = peak_bytes(fn)
        ms = [timed(fn) for _ in range(3)]
        big[path] = {"peak_bytes": peak, "ms": stats(ms), "batch_allowed_by_peak": total // peak}
        print("n=256 b=1 cls %s: %.1f ms, peak %.2f GB -> batch %d on %.0f GB" % (path, statistics.median(ms), peak / 1e9,
                                                                               total // peak, total / 1e9), flush=True)
    result["n256"] = big
    print(json.dumps(result["card"]))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
