#!/usr/bin/env python
"""Forward + backward of a DGDE-loss-shaped chain through the detector-head functions, eager, two routes alternated:

    dcd_b200  select_point_of_interest -> image keypoints (torch) -> edge_depth_mean(training=True) -> decode_location_flatten,
              decode_depth_from_keypoints_batch + depth_ensemble on other channel slices; L1 losses (torch)
    oracle    the same chain through oracle/dcd_oracle.py (the reference's torch ops) on the same GPU

Shape: 8 images, a [8, 440, 96, 320] FP32 regression map (384 x 1280 input / 4), 40 target slots per image of which
U{15..40} are objects and the rest padding on position 0 (as the reference's targets), 73 keypoints.  Reported: median step
time and peak memory per route, and the map-gradient kernels (dcd_poi_gather_bwd) alone: bytes of the dense gradient
written, achieved GB/s against the HBM3e data-sheet figure, and the split between the fill and the sparse pass.

    python profiles/run_dgde_head_grad.py [--steps 30] [--warmup 5] [--out FILE.json]
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
from dcd_b200 import _lib, synth  # noqa: E402
from oracle import dcd_oracle as O  # noqa: E402

B, C, H, W, SLOTS, n = 8, 440, 96, 320, 40, 73
CH = {"off3d": 0, "kp10": 2, "dims": 22, "direct": 25, "lud": 26, "luk": 27, "kpts2d": 30, "kpts3d": 176}
HBM_DATASHEET_GBS = 7700.0       # NVIDIA HGX B200 data sheet, one GPU: 7.7 TB/s HBM3e


def card():
    out = {"device": torch.cuda.get_device_name()}
    try:
        out["nvidia_smi"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True,
                                           timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["nvidia_smi"] = "unavailable: %s" % e
    return out


def make_inputs(dev):
    g = torch.Generator().manual_seed(12)
    counts = torch.randint(15, SLOTS + 1, (B,), generator=g)
    ob = synth.make_objects(n=n, seed=13, counts=counts, jitter_fx=0.02)
    N = ob.N
    fmap = torch.randn(B, C, H, W, generator=g) * 0.1
    idx = torch.zeros(B, SLOTS, dtype=torch.int64)
    mask = torch.zeros(B, SLOTS, dtype=torch.bool)
    pos = torch.empty(N, dtype=torch.int64)
    for b in range(B):
        sel = (ob.frame_id == b).nonzero().reshape(-1)
        p = torch.randperm(H * W - 1, generator=g)[:len(sel)] + 1
        pos[sel], idx[b, :len(sel)], mask[b, :len(sel)] = p, p, True
    pts = torch.stack(((pos % W).float(), (pos // W).float()), 1)
    pad_b = torch.rand(B, 2, generator=g) * 20
    pad = pad_b[ob.frame_id]
    ofs = torch.rand(N, 2, generator=g) - 0.5
    centre = pts + ofs
    off = (ob.kps + pad.unsqueeze(1)) / 4 - centre.unsqueeze(1)
    kp10 = (ob.kps[:, -10:] + pad.unsqueeze(1)) / 4 - centre.unsqueeze(1)
    dims = torch.stack((torch.full((N,), 3.9), -ob.kps_3d[:, -1, 1], torch.full((N,), 1.6)), dim=1)
    for o in range(N):
        col = fmap[int(ob.frame_id[o])].view(C, -1)[:, int(pos[o])]
        col[0:2] = ofs[o]
        col[2:22] = kp10[o].reshape(-1)
        col[22:25] = dims[o]
        col[25] = ob.gt_depth[o]
        col[26:30] = torch.rand(4, generator=g) - 0.5
        col[30:176] = off[o].reshape(-1)
        col[176:395] = ob.kps_3d[o].reshape(-1)
    P = [ob.K[(ob.frame_id == f).nonzero()[0, 0]].double().numpy() for f in range(B)]
    return dict(fmap=fmap.to(dev), idx=idx.to(dev), mask=mask.to(dev), pts=pts.to(dev), pad=pad_b.to(dev), bi=ob.frame_id.to(dev),
                K=ob.K.to(dev), rot=ob.rot_y.to(dev), gt=ob.gt_depth.to(dev), P=P, f_us=[float(p[0, 0]) for p in P], N=N)


def step(x, fm, route):
    N = x["N"]
    pois = (dcd_b200.select_point_of_interest if route == "dcd_b200" else O.select_point_of_interest)(B, x["idx"], fm)
    v = pois[x["mask"]]
    ofs = v[:, 0:2]
    kimg = (v[:, 30:176].reshape(N, n, 2) + (x["pts"] + ofs).unsqueeze(1)) * 4 - x["pad"][x["bi"]].unsqueeze(1)
    k3 = v[:, 176:395].reshape(N, n, 3)
    kp10, dims, direct, lud, luk = v[:, 2:22].reshape(N, 10, 2), v[:, 22:25], v[:, 25], v[:, 26], v[:, 27:30]
    if route == "dcd_b200":
        depth = dcd_b200.edge_depth_mean(kimg, k3, x["rot"], x["K"], training=True)
        loc = dcd_b200.decode_location_flatten(x["pts"], ofs, depth, x["K"], x["pad"], x["bi"])
        kd = dcd_b200.decode_depth_from_keypoints_batch(kp10, dims, x["K"])
        out = dcd_b200.depth_ensemble(kp10, dims, x["K"], luk, direct_depths=direct, direct_log_uncertainty=lud)
        ens, err = out["depth"], out["depth_error"]
    else:
        depth = O.decode_pairs_kpts_depth(kimg, k3, x["rot"], x["K"], training=True)[0].mean(1)
        loc = O.decode_location_flatten(x["pts"], ofs, depth, x["P"], x["pad"], x["bi"])
        kd = O.decode_depth_from_keypoints_batch(kp10, dims, x["f_us"], x["bi"])
        ens, err, _ = O.depth_ensemble(direct, kd, lud, luk)
    L = (loc[:, 2] - x["gt"]).abs().mean() + (kd - x["gt"].unsqueeze(1)).abs().mean() + (ens - x["gt"]).abs().mean() + 0.1 * err.mean()
    L.backward()


def time_route(x, route):
    fm = x["fmap"].clone().requires_grad_()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    step(x, fm, route)
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e), (torch.cuda.max_memory_allocated() - base) / 2 ** 20


def time_map_gradient(x, reps=50):
    """dcd_poi_gather_bwd alone (fill + sparse pass) and its fill alone (K = 0), CUDA events over `reps` launches each."""
    L = _lib.lib()
    g = torch.randn(B, SLOTS, C, device="cuda")
    out = torch.empty(B, C, H, W, device="cuda")
    st = torch.cuda.current_stream().cuda_stream

    def run(K):
        for _ in range(5):
            _lib.check(L.dcd_poi_gather_bwd(g.data_ptr(), x["idx"].data_ptr(), B, K, C, H * W, out.data_ptr(), st), "bwd")
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(reps):
            L.dcd_poi_gather_bwd(g.data_ptr(), x["idx"].data_ptr(), B, K, C, H * W, out.data_ptr(), st)
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e) / reps * 1e3

    full_us, fill_us = run(SLOTS), run(0)
    nbytes = B * C * H * W * 4
    return {"dense_gradient_bytes": nbytes, "fill_plus_sparse_us": round(full_us, 2), "fill_only_us": round(fill_us, 2),
            "sparse_pass_us": round(full_us - fill_us, 2), "achieved_GBs": round(nbytes / full_us / 1e3, 1),
            "share_of_datasheet_HBM": round(nbytes / full_us / 1e3 / HBM_DATASHEET_GBS, 3),
            "torch_route_bytes_lower_bound": 3 * nbytes,
            "note": "working set 432 MB > 126 MB L2; torch route: zeros NHWC + scatter_add + permute back to NCHW (>= 3 passes)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    x = make_inputs("cuda")
    routes = ("dcd_b200", "oracle")
    for _ in range(args.warmup):
        for r in routes:
            time_route(x, r)
    t = {r: [] for r in routes}
    mem = {r: 0.0 for r in routes}
    for _ in range(args.steps):
        for r in routes:
            ms, mb = time_route(x, r)
            t[r].append(ms)
            mem[r] = max(mem[r], mb)
    result = {"card": card(), "shape": {"images": B, "map": [B, C, H, W], "slots_per_image": SLOTS, "objects": x["N"],
                                        "keypoints": n, "padding": "unused slots on position 0"},
              "steps": args.steps, "warmup": args.warmup,
              "routes": {r: {"median_step_ms": round(statistics.median(t[r]), 3), "min_step_ms": round(min(t[r]), 3),
                             "peak_mem_MiB": round(mem[r], 1)} for r in routes},
              "map_gradient": time_map_gradient(x)}
    result["speedup"] = round(result["routes"]["oracle"]["median_step_ms"] / result["routes"]["dcd_b200"]["median_step_ms"], 2)
    js = json.dumps(result, indent=1)
    print(js)
    if args.out:
        with open(args.out, "w") as f:
            f.write(js + "\n")


if __name__ == "__main__":
    main()
