#!/usr/bin/env python
"""Cost of the keypoint gradients in the GMW training step (GMW/main.py:453-465, reg loss only, depth 12).

One step = compute_z -> GMW.forward -> compute_reg_loss -> backward, in three variants:
    params       trainable parameters, keypoints without grad (the reference's training loop)
    params+kpts  trainable parameters and keypoints that require grad (gradient through compute_z and the MLP)
    kpts         frozen parameters, keypoints that require grad (a trained GMW as a differentiable refiner)
The variants are alternated step by step in one process and timed with CUDA events around each whole step (the backward
ends in a device synchronise), after warm-up steps of every variant.

    python profiles/run_kpts_grad.py [--steps 30] [--warmup 6] [--out FILE.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import dcd_b200  # noqa: E402
from dcd_b200 import synth  # noqa: E402

SHAPES = [(73, 8), (73, 64), (256, 2)]          # (n, b): the reference's keypoints at its batch (-b 8) and at 64; the stress n
VARIANTS = ("params", "params+kpts", "kpts")


def card():
    out = {"device": torch.cuda.get_device_name()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60).stdout.strip()
        out["nvidia_smi"] = q
    except (OSError, subprocess.SubprocessError) as e:
        out["nvidia_smi"] = "unavailable: %s" % e
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert args.steps >= 20 and args.warmup >= 5
    torch.backends.cuda.matmul.allow_tf32 = False
    model = dcd_b200.GMW(depth=12).cuda().load_reference_state_dict(synth.random_state_dict(7))
    result = {"card": card(), "steps": args.steps, "warmup": args.warmup, "depth": 12, "shapes": []}
    for n, b in SHAPES:
        ob = synth.make_objects(N=b, n=n, seed=11)
        k2, k3, rot, gt = ob.kps_norm.cuda(), ob.kps_3d.cuda(), ob.rot_y.cuda(), ob.gt_depth.cuda()
        num_k = min(1500, n * (n - 1) // 2)

        def step(variant):
            frozen = variant == "kpts"
            for p in model.parameters():
                p.requires_grad_(not frozen)
            model.zero_grad(set_to_none=True)
            kg = variant != "params"
            a, c = k2.clone().requires_grad_(kg), k3.clone().requires_grad_(kg)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            Z, idx = dcd_b200.compute_z(a, c, rot, num_k=num_k)
            w, _ = model(a, c, rot, None)
            loss, _ = dcd_b200.compute_reg_loss(Z, w, gt, idx)
            loss.backward()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1)

        for _ in range(args.warmup):
            for v in VARIANTS:
                step(v)
        times = {v: [] for v in VARIANTS}
        for _ in range(args.steps):
            for v in VARIANTS:
                times[v].append(step(v))
        row = {"n": n, "b": b, "ms": {v: {"median": statistics.median(t), "min": min(t), "max": max(t)} for v, t in times.items()}}
        base = row["ms"]["params"]["median"]
        for v in VARIANTS[1:]:
            row["ms"][v]["extra_vs_params_ms"] = row["ms"][v]["median"] - base
        result["shapes"].append(row)
        print("n=%3d b=%2d  " % (n, b) + "  ".join("%s %.3f ms [%.3f, %.3f]" % (v, s["median"], s["min"], s["max"])
                                                    for v, s in row["ms"].items()), flush=True)
    for p in model.parameters():
        p.requires_grad_(True)
    print(json.dumps(result["card"]))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
