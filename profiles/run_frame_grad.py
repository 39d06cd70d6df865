#!/usr/bin/env python
"""Forward + backward of the DGDE frame epilogue from the regression map, two routes alternated in one process:

    fused        frame_depths_from_map (dcd_dgde_frame_fwd + dcd_dgde_frame_bwd)
    composition  select_point_of_interest per image -> channel slices -> (off + centre) * 4 - pad ->
                 decode_pairs_kpts_depth(training=False)[0].mean(1) -> decode_location_flatten -> + h/2 (the unfused
                 differentiable calls)

Loss: a random linear function of depth and location.  Shapes: 8 images with ~186 detections in all on a [8,415,96,320] FP32
map (384 x 1280 input / 4), and 1 image with 5, 20 and 50 detections; 73 keypoints, the DGDE channel table.  Reported per
shape and route: median step time (CUDA events around forward + backward, after warm-up), and the dense map gradient's
bytes over the fused step time.  The map (and its gradient) is larger than the 126 MB L2 at the 8-image shape.

    python profiles/run_frame_grad.py [--steps 30] [--warmup 5] [--out FILE.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import dcd_b200  # noqa: E402
from dcd_b200 import synth  # noqa: E402

C, H, W, n = 415, 96, 320, 73
CH = dcd_b200.ops.DGDE_CHANNELS


def card():
    out = {"device": torch.cuda.get_device_name()}
    try:
        out["nvidia_smi"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True,
                                           timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["nvidia_smi"] = "unavailable: %s" % e
    return out


def make_inputs(counts, seed, dev):
    g = torch.Generator().manual_seed(seed)
    B = len(counts)
    ob = synth.make_objects(n=n, seed=seed, counts=torch.tensor(counts), jitter_fx=0.02)
    N, bi = ob.N, ob.frame_id
    fm = torch.randn(B, C, H, W, generator=g) * 0.1
    pos = torch.empty(N, dtype=torch.int64)
    for b in range(B):
        sel = (bi == b).nonzero().reshape(-1)
        pos[sel] = torch.randperm(H * W, generator=g)[:len(sel)]
    pad_b = torch.rand(B, 2, generator=g) * 20
    pad = pad_b[bi]
    pts = torch.stack(((pos % W).float(), (pos // W).float()), 1)
    ofs = torch.rand(N, 2, generator=g) - 0.5
    off = (ob.kps + pad.unsqueeze(1)) / 4 - (pts + ofs).unsqueeze(1)
    flat = fm.view(B, C, -1)
    for first, vals in ((CH["extra_kpts_2d"], off.reshape(N, -1)), (CH["extra_kpts_3d"], ob.kps_3d.reshape(N, -1)),
                        (CH["3d_offset"], ofs)):
        c = first + torch.arange(vals.shape[1])
        flat.index_put_((bi[:, None], c[None, :], pos[:, None]), vals)
    P = np.stack([ob.K[(bi == b).nonzero()[0, 0]].double().numpy() for b in range(B)])
    dims = torch.stack((torch.full((N,), 3.9), -ob.kps_3d[:, -1, 1], torch.full((N,), 1.6)), dim=1)
    return dict(fm=fm.to(dev), pos=pos.to(dev), bi=bi.to(dev), rot=ob.rot_y.reshape(-1).to(dev), P=torch.from_numpy(P).to(dev),
                pad=pad_b.to(dev), dims=dims.to(dev), pts=pts.to(dev), B=B, N=N,
                g_depth=torch.randn(N, generator=g).to(dev), g_loc=torch.randn(N, 3, generator=g).to(dev))


def step(x, fm, dims, route):
    bi = x["bi"]
    if route == "fused":
        depth, loc = dcd_b200.frame_depths_from_map(fm, x["pos"], x["rot"], x["P"], x["pad"], dims=dims, batch_idxs=bi)
    else:
        parts = []
        for b in range(x["B"]):
            sel = (bi == b).nonzero().reshape(-1)
            parts.append((sel, dcd_b200.select_point_of_interest(1, x["pos"][sel].reshape(1, -1), fm[b:b + 1]).reshape(-1, C)))
        rows = torch.cat([p for _, p in parts])[torch.argsort(torch.cat([s for s, _ in parts]))]
        off = rows[:, CH["extra_kpts_2d"]:CH["extra_kpts_2d"] + 2 * n].reshape(-1, n, 2)
        k3 = rows[:, CH["extra_kpts_3d"]:CH["extra_kpts_3d"] + 3 * n].reshape(-1, n, 3)
        ofs = rows[:, CH["3d_offset"]:CH["3d_offset"] + 2]
        K = x["P"][bi]
        kimg = (off + (x["pts"] + ofs).unsqueeze(1)) * 4 - x["pad"][bi].unsqueeze(1)
        depth = dcd_b200.decode_pairs_kpts_depth(kimg, k3, x["rot"], K, training=False)[0].mean(1)
        loc = dcd_b200.decode_location_flatten(x["pts"], ofs, depth, K, x["pad"], bi)
        loc = torch.cat((loc[:, :1], loc[:, 1:2] + dims[:, 1:2] / 2, loc[:, 2:]), 1)
    L = (depth * x["g_depth"]).sum() + (loc * x["g_loc"]).sum()
    return torch.autograd.grad(L, [fm, dims])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda")
    shapes = {"8 images": [23, 25, 21, 24, 22, 26, 20, 25], "1 image, 5": [5], "1 image, 20": [20], "1 image, 50": [50]}
    res = {"card": card(), "steps": a.steps, "shapes": {}}
    for name, counts in shapes.items():
        x = make_inputs(counts, seed=len(counts) * 100 + sum(counts), dev=dev)
        fm = x["fm"].requires_grad_()
        dims = x["dims"].requires_grad_()
        ref = step(x, fm, dims, "composition")
        got = step(x, fm, dims, "fused")
        err = float((got[0] - ref[0]).abs().max() / ref[0].abs().max())
        for _ in range(a.warmup):
            for route in ("fused", "composition"):
                step(x, fm, dims, route)
        times = {"fused": [], "composition": []}
        for _ in range(a.steps):
            for route in ("fused", "composition"):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                step(x, fm, dims, route)
                e1.record()
                e1.synchronize()
                times[route].append(e0.elapsed_time(e1))
        med = {r: statistics.median(t) for r, t in times.items()}
        grad_bytes = fm.numel() * 4
        res["shapes"][name] = {"map": list(fm.shape), "detections": x["N"], "median_ms": med,
                               "speedup": med["composition"] / med["fused"], "map_grad_MB": grad_bytes / 1e6,
                               "map_grad_written_GBs_over_fused_step": grad_bytes / (med["fused"] * 1e-3) / 1e9,
                               "map_grad_rel_diff_vs_composition": err}
        print(name, json.dumps(res["shapes"][name]), flush=True)
    print(json.dumps(res["card"]))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
