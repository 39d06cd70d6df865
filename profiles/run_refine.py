#!/usr/bin/env python
"""DGDE detections refined by GMW, two routes alternated in one run:

    refine    dcd_b200.refine_detections: regression map -> GMW-rescaled locations, one library call
    hand      frame_depths_from_map -> FP32 normalisation (torch) -> gmw_weighted_depth -> ray_rescale

Batched: 8 images per [8, 440, 96, 320] FP32 regression map (384 x 1280 input / 4), U{1..50} detections per image, 73
keypoints; objects/s of each route (CUDA events around `--steps` calls, median over `--reps` alternated repetitions) and
whether their outputs are equal.  Per frame: one image with 5, 20 and 50 detections, median wall time of one call ending in
a device synchronise.  Hand-off the call removes: host time of wire.from_detector + the reference's indent=4 JSON write +
wire.load_reference_json of the same records (gen_data_infer.json, DGDE/engine/inference.py:59-84 -> GMW/main.py:524).
The map (8 x 440 x 96 x 320 x 4 B = 433 MB) is larger than the 126 MB L2; the routes read only the detections' columns.

    python profiles/run_refine.py [--steps 20] [--reps 5] [--warmup 3] [--out FILE.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import dcd_b200  # noqa: E402
from dcd_b200 import synth, wire  # noqa: E402
from oracle import dcd_oracle as O  # noqa: E402

C, H, W, n = 440, 96, 320, 73
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
    """Geometry-consistent detections planted in a [B,440,96,320] map (image keypoints of synth objects through KITTI's P2,
    per-image pad), the head's dims (l, h, w) and decoded yaw."""
    B = len(counts)
    g = torch.Generator().manual_seed(seed)
    ob = synth.make_objects(n=n, seed=seed, counts=torch.tensor(counts), jitter_fx=0.02)
    N, bi = ob.N, ob.frame_id
    fmap = torch.randn(B, C, H, W, generator=g) * 0.1
    pos = torch.empty(N, dtype=torch.int64)
    for b in range(B):
        sel = (bi == b).nonzero().reshape(-1)
        pos[sel] = torch.randperm(H * W, generator=g)[:len(sel)]
    pad_b = torch.rand(B, 2, generator=g) * 20
    pts = torch.stack(((pos % W).float(), (pos // W).float()), 1)
    ofs = torch.rand(N, 2, generator=g) - 0.5
    off = (ob.kps + pad_b[bi].unsqueeze(1)) / 4 - (pts + ofs).unsqueeze(1)
    for d in range(N):
        b, p = int(bi[d]), int(pos[d])
        fmap[b, CH["3d_offset"]:CH["3d_offset"] + 2].view(2, -1)[:, p] = ofs[d]
        fmap[b, CH["extra_kpts_2d"]:CH["extra_kpts_2d"] + 2 * n].view(2 * n, -1)[:, p] = off[d].reshape(-1)
        fmap[b, CH["extra_kpts_3d"]:CH["extra_kpts_3d"] + 3 * n].view(3 * n, -1)[:, p] = ob.kps_3d[d].reshape(-1)
    dims = torch.stack((torch.full((N,), 3.9), -ob.kps_3d[:, -1, 1], torch.full((N,), 1.6)), dim=1)
    P = torch.stack([ob.K[(bi == b).nonzero()[0, 0]] for b in range(B)]).to(dev)        # [B,3,4] float64 per image
    return {"fm": fmap.to(dev), "pos": pos.to(dev), "rot": ob.rot_y.reshape(-1).to(dev), "dims": dims.to(dev), "P": P,
            "pad": pad_b.to(dev), "bi": bi.to(dev) if B > 1 else None, "N": N, "B": B}


def route_refine(x, model):
    r = dcd_b200.refine_detections(x["fm"], x["pos"], x["rot"], x["P"] if x["B"] > 1 else x["P"][0],
                                   x["pad"] if x["B"] > 1 else x["pad"][0], x["dims"], model, batch_idxs=x["bi"])
    return r["gmw_depth"], r["location"]


def route_hand(x, model):
    P = x["P"] if x["B"] > 1 else x["P"][0]
    _, loc, kimg, k3 = dcd_b200.frame_depths_from_map(x["fm"], x["pos"], x["rot"], P, x["pad"] if x["B"] > 1 else x["pad"][0],
                                                      dims=x["dims"], batch_idxs=x["bi"], return_keypoints=True)
    K = (x["P"][x["bi"].long()] if x["bi"] is not None else x["P"][0].expand(x["N"], 3, 4)).float()
    k2 = torch.stack(((kimg[..., 0] - K[:, None, 0, 2]) / K[:, None, 0, 0], (kimg[..., 1] - K[:, None, 1, 2]) / K[:, None, 1, 1]), -1)
    z = dcd_b200.gmw_weighted_depth(k2, k3, x["rot"], model)
    return z, dcd_b200.ray_rescale(loc, z, x["dims"][:, [1, 2, 0]])


ROUTES = {"refine": route_refine, "hand": route_hand}


def event_ms(fn, steps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps


def wall_ms(fn, calls):
    ts = []
    for _ in range(calls):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts)


def handoff_ms(x, model, reps):
    """Host side of the file hand-off on the records of one batch: records to the host, the reference's JSON, parse back."""
    _, loc, kimg, k3 = dcd_b200.frame_depths_from_map(x["fm"], x["pos"], x["rot"], x["P"], x["pad"], dims=x["dims"],
                                                      batch_idxs=x["bi"], return_keypoints=True)
    Pobj = x["P"][x["bi"].long()]
    bi = x["bi"].cpu().numpy()
    ts = {"from_detector": [], "json_write": [], "load_reference_json": []}
    json_bytes = 0
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "gen_data_infer.json")
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            rec = wire.from_detector(kimg, k3, x["rot"], loc, Pobj, dim=x["dims"][:, [1, 2, 0]])
            t1 = time.perf_counter()
            data = {}
            for m in range(x["N"]):
                data.setdefault("%06d" % bi[m], []).append({
                    "kpts_2d": rec["kpts_2d"][m].reshape(-1).tolist(), "kpts_3d": rec["kpts_3d"][m].reshape(-1).tolist(),
                    "pred_rot": rec["pred_rot"][m].tolist(), "dim": rec["dim"][m].tolist(),
                    "pred_location": rec["gt_location"][m].tolist()})
            with open(path, "w") as f:
                json.dump(data, f, indent=4)
            t2 = time.perf_counter()
            back = wire.load_reference_json(path, "valid")
            t3 = time.perf_counter()
            assert back["kpts_2d"].shape == (x["N"], n, 2)
            json_bytes = os.path.getsize(path)
            ts["from_detector"].append((t1 - t0) * 1e3)
            ts["json_write"].append((t2 - t1) * 1e3)
            ts["load_reference_json"].append((t3 - t2) * 1e3)
    out = {k + "_ms": statistics.median(v) for k, v in ts.items()}
    out["total_ms"] = sum(out.values())
    out["json_bytes"] = json_bytes
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("run_refine.py measures on the GPU: no CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda")
    model = dcd_b200.GMW().to(dev).load_reference_state_dict(O.random_state_dict(7))
    result = {"card": card(), "steps": a.steps, "reps": a.reps}
    torch.set_grad_enabled(False)

    g = torch.Generator().manual_seed(5)
    counts = torch.randint(1, 51, (8,), generator=g).tolist()
    x = make_inputs(counts, 21, dev)
    for fn in ROUTES.values():                                     # warm every shape of both routes
        for _ in range(a.warmup):
            fn(x, model)
    torch.cuda.synchronize()
    outs = {k: fn(x, model) for k, fn in ROUTES.items()}
    equal = all(torch.equal(p, q) for p, q in zip(outs["refine"], outs["hand"]))
    ms = {k: [] for k in ROUTES}
    for _ in range(a.reps):
        for k, fn in ROUTES.items():
            ms[k].append(event_ms(lambda: fn(x, model), a.steps))
    result["batched"] = {"images": 8, "map": [8, C, H, W], "detections_per_image": counts, "objects": x["N"],
                         "outputs_equal": equal,
                         **{k: {"ms_per_call": statistics.median(v), "ms_all_reps": v,
                                "objects_per_s": x["N"] / (statistics.median(v) * 1e-3)} for k, v in ms.items()}}
    result["handoff_host"] = handoff_ms(x, model, max(3, a.reps))
    del x

    per = {}
    for N in (5, 20, 50):
        y = make_inputs([N], 30 + N, dev)
        for fn in ROUTES.values():
            for _ in range(a.warmup):
                fn(y, model)
        med = {k: [] for k in ROUTES}
        for _ in range(a.reps):
            for k, fn in ROUTES.items():
                med[k].append(wall_ms(lambda: fn(y, model), a.steps))
        per[str(N)] = {k + "_ms": statistics.median(v) for k, v in med.items()}
        per[str(N)]["outputs_equal"] = all(torch.equal(p, q) for p, q in zip(route_refine(y, model), route_hand(y, model)))
    result["per_frame_latency"] = per
    js = json.dumps(result, indent=1)
    print(js)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(js + "\n")


if __name__ == "__main__":
    main()
