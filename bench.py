#!/usr/bin/env python
"""Benchmark of the densely-constrained-depth hot path (BASELINE.json metric: objects/sec, edge solve +
GMW aggregate).

    python bench.py [--gpus N] [--steps K] [--warmup W]          # this repo's CUDA path, BASELINE configs[1]
    python bench.py --impl reference [...]                       # the reference algorithm on the host CPU
    python bench.py --config sweep1m   [--gpus N]                # BASELINE configs[3]: 2^20 objects, STRONG scaling, all-gather
    python bench.py --config stress256 [--gpus N]                # BASELINE configs[4]: 256 keypoints, forward + backward
    python bench.py [...] --dump-outputs DIR                     # also save the outputs of the last timed step as DIR/*.npy

Default (`--config kitti_val`): a *step* is one forward pass of the GMW pipeline (compute_z -> edge-weight MLP ->
softmax-weighted depth, GMW/main.py:524-533) over one KITTI-val-shaped synthetic batch (BASELINE configs[1]:
3769 frames, <= 50 objects per frame, 73 keypoints).  With N GPUs every rank owns a contiguous shard of
N x 3769 frames (weak scaling) and the step ends with the all-gather of the per-object depths.  One JSON line is
printed by rank 0; see DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "objects/sec (edge solve + GMW aggregate)"
UNIT = "objects/s"
N_KPTS = 73
EDGES = N_KPTS * (N_KPTS - 1) // 2
K_SEL = 1500
DEPTH = 12
FRAMES = 3769
WEIGHT_SEED = 7
C = 128


# algorithmic work per object (SURVEY.md section 8d / BASELINE.md section 4)
def edges_of(n):
    return n * (n - 1) // 2


def f_solve(n):                     # 29 346 FLOP at n = 73
    return 6 * n + 11 * edges_of(n)


def f_solve_bwd(n):                 # 22 E + 12 n
    return 22 * edges_of(n) + 12 * n


def b_solve(n):                     # 1516 B in + mean out at n = 73
    return 20 * n + 56


def f_mlp_ref(n):                   # the reference's 36 GEMM layers per net: 6.207 GFLOP at n = 73
    return edges_of(n) * (2 * C * (4 + 6) + 36 * 2 * 2 * C * C)


def f_mlp(n):                       # preconv.conv1 folded (no non-linearity between them): 24 GEMM layers per net are executed,
    return edges_of(n) * (2 * C * (4 + 6) + 24 * 2 * 2 * C * C)   # and only those are counted (SURVEY 8d): 4.140 GFLOP


F_SOLVE, B_SOLVE, F_MLP, F_MLP_REF = f_solve(N_KPTS), b_solve(N_KPTS), f_mlp(N_KPTS), f_mlp_ref(N_KPTS)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="dcd_b200", choices=["dcd_b200", "reference"])
    ap.add_argument("--config", default="kitti_val", choices=["kitti_val", "kitti_val_full", "sweep1m", "stress256"],
                    help="kitti_val = BASELINE configs[1] ragged (default, the metric's config); kitti_val_full = 50 objects in "
                         "every frame; sweep1m = configs[3]; stress256 = configs[4]")
    ap.add_argument("--frames", type=int, default=FRAMES, help="frames per GPU (default: the KITTI val split)")
    ap.add_argument("--chunk", type=int, default=2048, help="objects per MLP workspace chunk")
    ap.add_argument("--cpu-sample", type=int, default=512, help="objects of the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--objects", type=int, default=1 << 20, help="sweep1m: total objects")
    ap.add_argument("--quick", action="store_true", help="skip the per-stage breakdown (multi-rank scaling runs)")
    ap.add_argument("--graph-collective", action="store_true", help="sweep1m: also time solve + all-gather replayed from a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the timed path returned in its last step as DIR/<name>.npy "
                         "(inputs are seeded, so two builds can be compared output for output)")
    return ap.parse_args()


DUMP_BYTES = 64 * 10**6


def dump_outputs(args, arrays):
    """--dump-outputs: every (float32) array as DIR/<name>.npy, at most DUMP_BYTES in all.  An array larger than its
    share of the budget is stored as a fixed seeded sample of its flattened elements, in order; the sampled positions
    depend only on the array's size, so the dumps of two builds stay comparable element for element."""
    if not args.dump_outputs:
        return
    import numpy as np
    os.makedirs(args.dump_outputs, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().float().cpu()
        cap = DUMP_BYTES // len(arrays) // 4
        if a.numel() > cap:
            g = torch.Generator().manual_seed(WEIGHT_SEED)
            a = a.reshape(-1)[torch.randperm(a.numel(), generator=g)[:cap].sort().values]
        np.save(os.path.join(args.dump_outputs, name + ".npy"), a.numpy())


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def measured_traffic(kernel: str):
    """DRAM bytes (read + write) per launch of `kernel` from the committed ncu --set full capture of this build
    (profiles/traffic.json, written by profiles/summarise.py); None when no capture has been recorded."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(path) as f:
            return json.load(f).get(kernel)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        try:
            with open(self.path) as f:
                for line in f:
                    c = [x.strip() for x in line.split(",")]
                    if len(c) < 9:
                        continue
                    try:
                        sm.append(float(c[1]))
                        smax.append(float(c[2]))
                    except ValueError:
                        continue
                    for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                        if val.lower().startswith("active"):
                            reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            busy = sorted(sm)[len(sm) // 2:]          # upper half = samples under load
            out = {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(smax), "reasons": sorted(reasons),
                   "samples": len(sm)}
        return out


class CpuReference:
    """The reference's algorithm for this path on the host CPU (oracle port, `faithful` mode: the per-pair
    Python loops of get_up and the E x E distance matrix, i.e. what the reference executes; the Sinkhorn
    branch is outside the path), batch 8 like the reference's `-b 8`, all host threads."""

    def __init__(self, n: int = N_KPTS):
        from oracle import dcd_oracle as O
        self.O = O
        self.n = n
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        self.sd = O.random_state_dict(WEIGHT_SEED)

    def run(self, objects: int, seed: int) -> float:
        """Process `objects` synthetic objects; returns seconds and keeps their depths in `self.depth`."""
        from dcd_b200 import synth
        ob = synth.make_objects(N=objects, n=self.n, seed=seed)
        t0 = time.perf_counter()
        with torch.no_grad():
            depths = [self.O.gmw_pipeline(ob.kps_norm[lo:lo + 8], ob.kps_3d[lo:lo + 8], ob.rot_y[lo:lo + 8], self.sd, faithful=True)
                      for lo in range(0, objects, 8)]
        secs = time.perf_counter() - t0
        self.depth = torch.cat(depths)
        return secs


def cpu_reference_rate(sample_objects: int, seed: int):
    ref = CpuReference()
    ref.run(8, seed + 1)                      # warm-up (thread pools, oneDNN primitives)
    secs = ref.run(sample_objects, seed)
    return sample_objects / secs, secs, ref.cores


WORKLOAD_TEXT = {
    "kitti_val": "configs[1]: KITTI-val-shaped synthetic batch (3769 frames x U{1..50} objects/frame, 73 keypoints): "
                 "compute_z + GMW.forward reg branch + weighted depth, forward only",
    "kitti_val_full": "configs[1] (full variant): KITTI-val-shaped synthetic batch (3769 frames x 50 objects/frame, 73 keypoints): "
                      "compute_z + GMW.forward reg branch + weighted depth, forward only",
    "sweep1m": "configs[3]: 1M-object synthetic sweep (73 keypoints): compute_z + GMW.forward reg branch + weighted depth, forward only",
    "stress256": "configs[4]: dense keypoint stress, 256 keypoints/object (32 640 edges): compute_z + GMW.forward + reg loss, "
                 "forward + backward",
}


def run_reference(args):
    """`--impl reference`: rank 0 times the CPU reference arm; other ranks exit without work."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    ref = CpuReference()
    sample = max(8, args.cpu_sample // 2)
    for w in range(args.warmup):
        ref.run(8, 1 + w)
    secs = sum(ref.run(sample, 100 + s) for s in range(args.steps))
    dump_outputs(args, {"depth": ref.depth})
    rate = sample * args.steps / secs
    line = {
        "metric": METRIC, "value": rate, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD_TEXT["kitti_val"] + "; each step is a bounded sample of %d objects in batches of 8" % sample},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": ref.cores, "kind": "port",
                         "sample": "%d objects per step in batches of 8, torch %s CPU, oracle port in faithful mode "
                                   "(Python get_up loops + E x E distance matrix; Sinkhorn branch excluded)" % (sample, torch.__version__)},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------------------
# shared plumbing of the CUDA arms
# --------------------------------------------------------------------------------------------------------------
class Ctx:
    def __init__(self, args):
        import torch.distributed as dist
        import dcd_b200
        from dcd_b200 import _lib
        self.args = args
        self.dist = dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise RuntimeError("bench.py needs a CUDA device (dcd_b200 has no CPU path); use --impl reference for the CPU arm")
        # the CPU baseline leg runs BEFORE the process group exists and only in single-GPU runs, so that no rank ever
        # spins in a collective while rank 0 times the host (r01: 297 s and a bogus figure at N = 8)
        self.cpu_baseline = None
        if self.world == 1 and not args.no_cpu_baseline and args.config in ("kitti_val", "kitti_val_full"):
            rate, secs, cores = cpu_reference_rate(args.cpu_sample, 99)
            self.cpu_baseline = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                                 "sample": "%d objects in batches of 8 (%.1f s), oracle port in faithful mode on the host CPU"
                                           % (args.cpu_sample, secs)}
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            import datetime
            # a short collective timeout: a rank that dies must not keep the others (and the box) waiting for 10 minutes
            dist.init_process_group("nccl", device_id=self.dev, timeout=datetime.timedelta(seconds=240))
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
        self.L = _lib.lib()
        self.peaks = measured_peaks()
        self.dcd = dcd_b200

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, values):
        t = torch.tensor(values, dtype=torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def fp32_peak(self, clocks):
        props = torch.cuda.get_device_properties(self.dev)
        sm_max_mhz = (clocks or {}).get("sm_max_mhz") or 1965.0
        return props.multi_processor_count * 128 * 2 * sm_max_mhz * 1e6 / 1e12            # TFLOP/s

    def finish(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def time_kernel(fn, reps=10, warm=3):
    for _ in range(warm):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def shard_objects(ctx, counts, n, seed):
    """Contiguous frame shard of this rank (dist.shard_bounds) -> (Objects, bounds, N_total)."""
    from dcd_b200 import dist as ddist, synth
    bounds = ddist.shard_bounds(counts.tolist(), ctx.world)
    cum = torch.cat([torch.zeros(1, dtype=torch.int64), counts.cumsum(0)])
    ob = synth.make_objects(n=n, seed=seed + 1000 * ctx.rank, counts=frames_of_shard(counts, cum, bounds[ctx.rank]))
    assert ob.N == bounds[ctx.rank][1] - bounds[ctx.rank][0]
    return ob, bounds, int(cum[-1])


def frames_of_shard(counts, cum, bound):
    lo_obj, hi_obj = bound
    f_lo = int((cum == lo_obj).nonzero()[0]) if lo_obj < int(cum[-1]) else len(counts)
    f_hi = int((cum == hi_obj).nonzero()[-1])
    return counts[f_lo:f_hi]


def make_objects_chunked(counts, n, seed, chunk_frames=1024):
    """synth.make_objects over a long frame list in bounded pieces (the generator works in float64)."""
    from dcd_b200 import synth
    parts = []
    for f0 in range(0, counts.numel(), chunk_frames):
        parts.append(synth.make_objects(n=n, seed=seed + 7919 * (f0 // chunk_frames), counts=counts[f0:f0 + chunk_frames]))
    cat = lambda name: torch.cat([getattr(p, name) for p in parts])   # noqa: E731
    return synth.Objects(kps=cat("kps"), kps_norm=cat("kps_norm"), kps_3d=cat("kps_3d"), rot_y=cat("rot_y"), K=cat("K"),
                         mask=cat("mask"), gt_depth=cat("gt_depth"), frame_id=cat("frame_id"), counts=counts)


class GmwForward:
    """select -> edge-weight MLP -> aggregate per chunk of objects, through the C ABI on the current stream."""

    def __init__(self, ctx, N, n, chunk, p4, p6):
        from dcd_b200._lib import check, ptr, stream_ptr
        self.ctx, self.N, self.n, self.E = ctx, N, n, edges_of(n)
        self.check, self.ptr, self.stream_ptr = check, ptr, stream_ptr
        L, dev = ctx.L, ctx.dev
        self.chunk = max(1, min(chunk, N))
        self.ws = torch.empty((L.dcd_gmw_workspace_bytes(self.chunk, n, DEPTH, 0) // 4 + 64,), dtype=torch.float32, device=dev)
        self.idx = torch.empty((self.chunk, K_SEL), dtype=torch.int64, device=dev)
        self.zsel = torch.empty((self.chunk, K_SEL), dtype=torch.float32, device=dev)
        self.regw = torch.empty((self.chunk, self.E), dtype=torch.float32, device=dev)
        self.depth_out = torch.empty((N,), dtype=torch.float32, device=dev)
        self.p4, self.p6 = p4, p6
        self.launches = 0
        self.mlp_events = []

    def step(self, k2, k3, rot, record_mlp: bool):
        L, check, ptr = self.ctx.L, self.check, self.ptr
        st = self.stream_ptr()
        n, E = self.n, self.E
        for c0 in range(0, self.N, self.chunk):
            nc = min(self.chunk, self.N - c0)
            a2, a3, ar = k2[c0:c0 + nc], k3[c0:c0 + nc], rot[c0:c0 + nc]
            check(L.dcd_edge_select_fwd(ptr(a2), ptr(a3), ptr(ar), 0, 0, nc, n, K_SEL, 0.1, 80.0, 0,
                                        ptr(self.idx), ptr(self.zsel), 0, 0, st), "select")
            if record_mlp:
                e0 = torch.cuda.Event(enable_timing=True)
                e1 = torch.cuda.Event(enable_timing=True)
                e0.record()
            check(L.dcd_gmw_weights_fwd(ptr(a2), ptr(a3), ptr(self.p4), ptr(self.p6), nc, n, DEPTH, 0, ptr(self.regw), 0, 0,
                                        ptr(self.ws), self.ws.numel() * 4, st), "mlp")
            if record_mlp:
                e1.record()
                self.mlp_events.append((e0, e1, nc))
            check(L.dcd_gmw_aggregate_fwd(ptr(self.regw), ptr(self.zsel), ptr(self.idx), nc, E, K_SEL, 1,
                                          ptr(self.depth_out[c0:]), 0, st), "aggregate")
            # select | layer folding, weight image, fused MLP (all layers of both nets), edge weights | aggregate
            self.launches += 1 + 4 + 1


def check_shard_bit_equality(ctx, full, bounds, recompute):
    """SURVEY 8e correctness check: the depths gathered from ANOTHER rank must equal, bit for bit, a recomputation of
    that rank's shard on rank 0 (same kernels, same per-object arithmetic).  Returns a small report (rank 0)."""
    if ctx.world == 1 or ctx.rank != 0:
        return None
    other = 1
    lo, hi = bounds[other]
    mine = recompute(other)
    same = bool(torch.equal(mine, full[lo:hi]))
    if not same:
        raise AssertionError("depths of rank %d differ from their single-rank recomputation" % other)
    return {"rank_checked": other, "objects": hi - lo, "bit_identical": same}


# --------------------------------------------------------------------------------------------------------------
# configs[1]: KITTI-val-shaped batch, GMW pipeline forward (the metric's config)
# --------------------------------------------------------------------------------------------------------------
def run_kitti_val(args):
    ctx = Ctx(args)
    dcd_b200, L, dev, world, rank = ctx.dcd, ctx.L, ctx.dev, ctx.world, ctx.rank
    from dcd_b200 import synth
    from dcd_b200 import dist as ddist
    from dcd_b200._lib import check, ptr, stream_ptr
    peaks = ctx.peaks
    ragged = args.config == "kitti_val"

    # ---- workload: world x FRAMES frames, sharded contiguously by frame (weak scaling)
    seed = synth.BASE_SEED + 1
    counts = synth.frame_counts(args.frames * world, 50, ragged, seed)
    ob, bounds, N_total = shard_objects(ctx, counts, N_KPTS, seed)
    N = ob.N
    lo_obj, hi_obj = bounds[rank]
    model = dcd_b200.GMW().to(dev).load_reference_state_dict(synth.random_state_dict(WEIGHT_SEED))
    p4, p6 = model.params4.detach(), model.params6.detach()

    # host (pinned) and device copies of the inputs
    h_k2, h_k3, h_rot = ob.kps_norm.pin_memory(), ob.kps_3d.pin_memory(), ob.rot_y.reshape(-1).contiguous().pin_memory()
    d_k2, d_k3, d_rot = h_k2.to(dev), h_k3.to(dev), h_rot.to(dev)
    h2d_bytes = (h_k2.numel() + h_k3.numel() + h_rot.numel()) * 4
    fw = GmwForward(ctx, N, N_KPTS, args.chunk, p4, p6)
    chunk = fw.chunk
    h_out = torch.empty((N,), dtype=torch.float32).pin_memory()

    def gather():
        if world > 1:
            return ddist.all_gather_depths(fw.depth_out, bounds)
        return fw.depth_out

    # ---- device-resident timing (value)
    for _ in range(args.warmup):
        fw.step(d_k2, d_k3, d_rot, False)
        gather()
    fw.launches = 0
    sampler = ClockSampler(ctx.local_rank)
    ctx.barrier()
    if rank == 0:
        sampler.start()
    t_beg, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_beg.record()
    for _ in range(args.steps):
        fw.step(d_k2, d_k3, d_rot, True)
        full = gather()
    t_end.record()
    ctx.barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms = t_beg.elapsed_time(t_end)
    timed_launches = fw.launches
    mlp_ms = sum(a.elapsed_time(b) for a, b, _ in fw.mlp_events)
    mlp_objs = sum(nc for _, _, nc in fw.mlp_events)
    assert full.numel() == N_total
    full = full.clone()
    if rank == 0:
        dump_outputs(args, {"depth": full})

    def recompute(other):
        ob2 = synth.make_objects(n=N_KPTS, seed=seed + 1000 * other,
                                 counts=frames_of_shard(counts, torch.cat([torch.zeros(1, dtype=torch.int64), counts.cumsum(0)]), bounds[other]))
        f2 = GmwForward(ctx, ob2.N, N_KPTS, args.chunk, p4, p6)
        f2.step(ob2.kps_norm.to(dev), ob2.kps_3d.to(dev), ob2.rot_y.reshape(-1).contiguous().to(dev), False)
        torch.cuda.synchronize()
        return f2.depth_out
    shard_check = check_shard_bit_equality(ctx, full, bounds, recompute)

    # ---- end-to-end timing through the public API with HOST buffers (e2e)
    def e2e_step():
        k2 = h_k2.to(dev, non_blocking=True)
        k3 = h_k3.to(dev, non_blocking=True)
        rot = h_rot.to(dev, non_blocking=True)
        out = dcd_b200.gmw_weighted_depth(k2, k3, rot, model, chunk=chunk)
        if world > 1:
            out = ddist.all_gather_depths(out, bounds)[lo_obj:hi_obj]
        h_out.copy_(out, non_blocking=True)
    e2e_step()
    ctx.barrier()
    e_beg, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e_beg.record()
    for _ in range(args.steps):
        e2e_step()
    e_end.record()
    ctx.barrier()
    e2e_ms = e_beg.elapsed_time(e_end)
    assert torch.isfinite(h_out).all()

    stages = {}
    if not args.quick:
        stages = kitti_val_stages(ctx, ob, d_k2, d_k3, d_rot, model)

    # ---- reduce over ranks (max time) and report
    ms, e2e_ms, mlp_ms_max = ctx.max_over_ranks([ms, e2e_ms, mlp_ms])
    if rank == 0:
        fp32_peak = ctx.fp32_peak(clocks)
        value = N_total * args.steps / (ms * 1e-3)
        e2e_value = N_total * args.steps / (e2e_ms * 1e-3)
        mlp_tflops = F_MLP * mlp_objs / (mlp_ms * 1e-3) / 1e12
        n_mlp_launches = len(fw.mlp_events)
        out_bytes = EDGES * 4 + N_KPTS * 20                               # per object: keypoints in, edge weights out (paired schedule)
        traffic = measured_traffic("mlp_fused_kernel") if chunk == 2048 else None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[1]%s: KITTI-val-shaped synthetic batch, %d frames x %s objects/frame "
                                   "(%d objects per GPU), 73 keypoints, 2628 edges: compute_z + edge-weight MLP + "
                                   "softmax-weighted depth, forward only%s" % ("" if ragged else " (full variant)", args.frames,
                                                                              "U{1..50}" if ragged else "50", N,
                                                                              ", + all-gather of depths" if world > 1 else ""),
                       "objects_per_gpu": N, "objects_total": N_total, "chunk_objects": chunk, "net_depth": DEPTH,
                       "l2_policy": "inputs larger than L2: a step reads %.0f MB of keypoints and writes %.0f MB of edge weights + depths per "
                                    "GPU against 126 MB of L2; per chunk the kernel also parks 25 MB of 4-d features in L2" % (
                                        N * (N_KPTS * 20 + 4) / 1e6, N * (EDGES * 4 + 4) / 1e6),
                       "weights": "random init, seed %d, reference state_dict layout" % WEIGHT_SEED},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": N * 4,
                    "api": "dcd_b200.gmw_weighted_depth on pinned host tensors"},
            "gpu_launches": timed_launches,
            "roofline": {"kernel": "mlp_fused_kernel (edge-feature MLP, the whole net in one launch: groups of 24 co-resident CTAs work on three objects "
                                   "at a time, activations stay in shared/tensor memory, one object's context-norm exchange runs behind the other two's "
                                   "tiles; preconv.conv1 folded: 24 GEMM layers x 2 nets on tcgen05, FP16x3 split, FP32 accumulate in TMEM; the "
                                   "edge weights come out of the kernel's own epilogue)",
                         "bound": "tensor",
                         "achieved": mlp_tflops, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                         "frac": mlp_tflops / peaks["bf16_tflops_sustained"],
                         # ncu dram__bytes_read+write of ONE mlp_fused_kernel launch on a 2048-object chunk, from the committed
                         # capture of this build (profiles/traffic.json); algorithmic: 2048 x 12 KB (keypoints in, edge weights out)
                         "traffic": traffic,
                         "peak_source": "%s dense bf16 (sustained, of measured); `achieved` counts the algorithmic FP32 GEMM FLOPs, the "
                                        "tensor pipe executes 3 FP16 MMAs per FP32 product (x3 = %.1f TFLOP/s issued); vs the FP32 "
                                        "CUDA-core roofline (%.1f TFLOP/s) the same number is %.2fx. The events bracket dcd_gmw_weights_fwd "
                                        "(layer folding + weight image, fused MLP, edge weights; the fused kernel is ~96%% of it)" % (
                                            peaks["source"], 3 * mlp_tflops, fp32_peak, mlp_tflops / fp32_peak),
                         "hbm_gbs": out_bytes * mlp_objs / (mlp_ms * 1e-3) / 1e9,
                         "frac_hbm": out_bytes * mlp_objs / (mlp_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                         "hbm_bytes_per_object": out_bytes, "hbm_bytes_per_object_layerwise": 198.0e6,
                         "frac_fp32_roofline": mlp_tflops / fp32_peak,
                         "flops_per_object": F_MLP, "flops_per_object_unfolded_reference": F_MLP_REF,
                         "avg_launch_ms": mlp_ms / max(n_mlp_launches, 1),
                         "share_of_step": mlp_ms_max / ms},
            "stages": dict(stages, fp32_peak_tflops=fp32_peak),
            "clocks": clocks,
        }
        if shard_check is not None:
            line["shard_check"] = shard_check
        for st in line["stages"].values():
            if isinstance(st, dict) and "fp32_tflops" in st:
                st["frac_fp32_roofline"] = st["fp32_tflops"] / fp32_peak
        if ctx.cpu_baseline is not None:
            line["cpu_baseline"] = ctx.cpu_baseline
        print(json.dumps(line), flush=True)
    ctx.finish()


def kitti_val_stages(ctx, ob, d_k2, d_k3, d_rot, model):
    """Per-stage breakdown on this rank's objects, kernel-only (CUDA events), next to the headline."""
    dcd_b200, L, dev, world = ctx.dcd, ctx.L, ctx.dev, ctx.world
    from dcd_b200 import synth
    from dcd_b200 import dist as ddist
    from dcd_b200._lib import check, ptr, stream_ptr
    N = ob.N
    peaks = ctx.peaks
    d_kps, d_K = ob.kps.to(dev), ob.K.to(dev)
    mean = torch.empty((N,), dtype=torch.float32, device=dev)
    edges = torch.empty((N, EDGES), dtype=torch.float32, device=dev)
    st = stream_ptr()
    ms_mean = time_kernel(lambda: check(L.dcd_edge_solve_fwd(ptr(d_kps), ptr(d_k3), ptr(d_rot), ptr(d_K), N, N_KPTS, 2.0, 80.0, 3,
                                                             0, ptr(mean), st), "solve"))
    ms_fast = time_kernel(lambda: check(L.dcd_edge_solve_fwd(ptr(d_kps), ptr(d_k3), ptr(d_rot), ptr(d_K), N, N_KPTS, 2.0, 80.0, 3 | 4,
                                                             0, ptr(mean), st), "solve"))
    ms_edges = time_kernel(lambda: check(L.dcd_edge_solve_fwd(ptr(d_kps), ptr(d_k3), ptr(d_rot), ptr(d_K), N, N_KPTS, 2.0, 80.0, 3,
                                                              ptr(edges), 0, st), "solve"))
    del edges
    # DGDE training pattern (detector_loss.py:378-381): top-1500 selection + depths, then the backward of the solve
    sel_n = min(N, 16384)
    idx_b = torch.empty((sel_n, K_SEL), dtype=torch.int64, device=dev)
    z_b = torch.empty((sel_n, K_SEL), dtype=torch.float32, device=dev)
    ms_sel = time_kernel(lambda: check(L.dcd_edge_select_fwd(ptr(d_kps), ptr(d_k3), ptr(d_rot), ptr(d_K), 0, sel_n, N_KPTS, K_SEL,
                                                             2.0, 80.0, 3, ptr(idx_b), ptr(z_b), 0, 0, st), "select"), reps=5)
    g_sel = torch.randn((sel_n, K_SEL), device=dev)
    g_kps = torch.empty((sel_n, N_KPTS, 2), device=dev)
    g_k3 = torch.empty((sel_n, N_KPTS, 3), device=dev)
    ms_bwd = time_kernel(lambda: check(L.dcd_edge_solve_bwd(ptr(d_kps), ptr(d_k3), ptr(d_rot), ptr(d_K), sel_n, N_KPTS, 2.0, 80.0, 3,
                                                            ptr(idx_b), K_SEL, ptr(g_sel), 0, ptr(g_kps), ptr(g_k3), st), "bwd"), reps=5)
    # frame epilogue (SURVEY 8f N2/N4): image-space keypoints -> edge solve + mean -> 3D location, one launch
    pad_o = torch.tensor([19.0, 5.0], device=dev).expand(N, 2).contiguous()
    ctr = (d_kps.mean(1) + pad_o) / 4
    pts_o = ctr.floor()
    ofs_o = (ctr - pts_o).contiguous()
    off_o = ((d_kps + pad_o.unsqueeze(1)) / 4 - ctr.unsqueeze(1)).contiguous()
    dims_o = torch.stack((torch.full((N,), 3.9, device=dev), -d_k3[:, -1, 1], torch.full((N,), 1.6, device=dev)), dim=1).contiguous()
    loc_o = torch.empty((N, 3), dtype=torch.float32, device=dev)
    ms_loc = time_kernel(lambda: check(L.dcd_dgde_locate_fwd(ptr(off_o), ptr(d_k3), ptr(d_rot), ptr(d_K), ptr(pts_o), ptr(ofs_o),
                                                             ptr(pad_o), ptr(dims_o), 0, N, N_KPTS, 2.0, 80.0, 3, 4.0, ptr(mean),
                                                             ptr(loc_o), st), "locate"))

    # one frame of the detector head (50 detections) through the public API: POI gather on a [1,440,96,320] regression map,
    # fused keypoints -> edge solve -> location, depth ensemble (SURVEY 8f N2/N4): latency, launch overheads included
    fr = 50
    fmap = torch.randn((1, 440, 96, 320), device=dev)
    fidx = torch.randint(0, 96 * 320, (1, fr), device=dev)
    P_np = ob.K[0].double().numpy()
    lu_k = torch.zeros((fr, 3), device=dev)

    def frame_epilogue():
        with torch.no_grad():
            dcd_b200.select_point_of_interest(1, fidx, fmap)
            d, _ = dcd_b200.compute_pairs_kpts_depth(off_o[:fr], pts_o[:fr], ofs_o[:fr], pad_o[:1], d_k3[:fr], d_rot[:fr], P_np,
                                                     dims=dims_o[:fr], return_locations=True)
            dcd_b200.depth_ensemble(off_o[:fr, -10:], dims_o[:fr], P_np, lu_k, direct_depths=d, direct_log_uncertainty=lu_k[:, 0])
    ms_frame = time_kernel(frame_epilogue, reps=20)
    # the same frame in ONE launch straight from the regression map (row N2 fused into the load stage), eager and replayed
    # from a CUDA graph (device-resident calibration / pad, as a detector loop would hold them)
    fmap415 = torch.randn((1, 415, 96, 320), device=dev) * 0.1
    K_fr, pad_fr, rot_fr, dims_fr = d_K[:fr].contiguous(), pad_o[:fr].contiguous(), d_rot[:fr].contiguous(), dims_o[:fr].contiguous()
    fidx1 = fidx.reshape(-1).contiguous()

    def frame_from_map():
        with torch.no_grad():
            return dcd_b200.frame_depths_from_map(fmap415, fidx1, rot_fr, K_fr, pad_fr, dims=dims_fr)
    ms_frame_map = time_kernel(frame_from_map, reps=50)
    ms_frame_graph = None
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            frame_from_map()
        torch.cuda.current_stream().wait_stream(side)
        gfr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gfr):
            frame_from_map()
        ms_frame_graph = time_kernel(gfr.replay, reps=200)
    except Exception as e:
        sys.stderr.write("frame graph capture failed: %r\n" % (e,))

    # ---- GMW training step, batch 8 per GPU (BASELINE configs[2]): compute_z + forward (saved) + loss + backward
    def make_train_step(tb):
        t_k2, t_k3, t_rot = d_k2[:tb].contiguous(), d_k3[:tb].contiguous(), d_rot[:tb].reshape(-1, 1).contiguous()
        t_gt = ob.gt_depth[:tb].to(dev)
        train_model = dcd_b200.GMW().to(dev).load_reference_state_dict(synth.random_state_dict(WEIGHT_SEED))

        def train_step():
            train_model.zero_grad(set_to_none=True)
            Zt, idxt = dcd_b200.compute_z(t_k2, t_k3, t_rot)
            wt, _ = train_model(t_k2, t_k3, t_rot, None)
            loss, _ = dcd_b200.compute_reg_loss(Zt, wt, t_gt, idxt)
            loss.backward()
            if world > 1:
                ddist.allreduce_gradients(train_model)
        return train_step, train_model, (t_k2, t_k3, t_rot, t_gt)
    train8, train_model, (t_k2, t_k3, t_rot8, t_gt8) = make_train_step(8)
    ms_train = time_kernel(train8, reps=5)
    # the same step replayed from a CUDA graph (one launch instead of ~80)
    graph_model = dcd_b200.GMW().to(dev).load_reference_state_dict(synth.random_state_dict(WEIGHT_SEED))
    gstep = dcd_b200.GraphedGmwStep(graph_model, batch=8, n=N_KPTS)

    def train8_graph():
        gstep(t_k2, t_k3, t_rot8, t_gt8)
        if world > 1:
            ddist.allreduce_gradients(graph_model)
    ms_train_graph = time_kernel(train8_graph, reps=10)
    train64, _, _ = make_train_step(64)
    ms_train64 = time_kernel(train64, reps=3, warm=2)
    # correspondence branch, forward (SURVEY 8f N1): E x E distances + Sinkhorn for the same 8 objects, P not materialised
    ms_cls = time_kernel(lambda: train_model.edge_transport(t_k2, t_k3, materialise=False), reps=3)

    # context: the same pipeline as plain torch ops (the oracle, diagonal form) on THIS GPU, cuBLAS FP32 with TF32 off -
    # what a DCD user runs today on a B200 (test infrastructure, timed beside the product like the CPU port)
    torch_ctx = None
    if ctx.rank == 0:
        from oracle import dcd_oracle as O
        sd_dev = {k: v.to(dev) for k, v in synth.random_state_dict(WEIGHT_SEED).items()}
        tn = 64
        o_k2, o_k3, o_rot = d_k2[:tn], d_k3[:tn], d_rot[:tn].reshape(-1, 1)

        def torch_oracle():
            with torch.no_grad():
                for lo in range(0, tn, 8):
                    O.gmw_pipeline(o_k2[lo:lo + 8], o_k3[lo:lo + 8], o_rot[lo:lo + 8], sd_dev)
        ms_t = time_kernel(torch_oracle, reps=2, warm=1)
        torch_ctx = {"objects_per_s": tn / (ms_t * 1e-3), "ms": ms_t, "objects": tn,
                     "what": "oracle (plain torch ops, diagonal form of the distance, vectorised get_up) on the same B200 in batches "
                             "of 8, cuBLAS/cuDNN FP32 with TF32 off; context only"}

    stages = {
        "dgde_solve_mean": {"objects_per_s": N / (ms_mean * 1e-3), "ms": ms_mean,
                            "fp32_tflops": F_SOLVE * N / (ms_mean * 1e-3) / 1e12,
                            "hbm_gbs": B_SOLVE * N / (ms_mean * 1e-3) / 1e9,
                            "issue_slot_ceiling": "12 issue slots per edge in the SASS of the inner loop (3 LDS + 5.5 packed FP32 + "
                                                  "3 FMNMX + 1 MUFU, minus rounding) for 11 counted FLOP: at most 11 / (2 x 12) = 46 % "
                                                  "of the FP32-FMA roofline"},
        "dgde_solve_mean_fast": {"objects_per_s": N / (ms_fast * 1e-3), "ms": ms_fast,
                                 "fp32_tflops": F_SOLVE * N / (ms_fast * 1e-3) / 1e12,
                                 "what": "opt-in DCD_FAST_QUOTIENT: hardware reciprocal instead of the IEEE division (per-object depth within "
                                         "1e-6 of the default; per-edge values not bit-faithful)"},
        "dgde_solve_edges": {"objects_per_s": N / (ms_edges * 1e-3), "ms": ms_edges,
                             "hbm_gbs": (B_SOLVE + 4 * EDGES) * N / (ms_edges * 1e-3) / 1e9,
                             "frac_hbm": (B_SOLVE + 4 * EDGES) * N / (ms_edges * 1e-3) / 1e9 / peaks["hbm_gbs"]},
        "dgde_frame_epilogue": {"objects_per_s": N / (ms_loc * 1e-3), "ms": ms_loc,
                                "fp32_tflops": F_SOLVE * N / (ms_loc * 1e-3) / 1e12,
                                "hbm_gbs": (B_SOLVE + 52) * N / (ms_loc * 1e-3) / 1e9,
                                "what": "keypoint offsets -> image keypoints -> edge solve + mean -> 3D location "
                                        "(detector_infer.py:215-227,186-188), one launch"},
        "dgde_frame_latency": {"us": ms_frame * 1e3, "objects": fr,
                               "what": "one frame, 50 detections, python API: select_point_of_interest + compute_pairs_kpts_depth "
                                       "(with locations) + depth_ensemble; three launches, host overheads included"},
        "dgde_frame_from_map": {"us_eager": ms_frame_map * 1e3, "us_cuda_graph": None if ms_frame_graph is None else ms_frame_graph * 1e3,
                                "objects": fr,
                                "what": "dcd_b200.frame_depths_from_map: POI gather + image keypoints + edge solve + mean + 3D location "
                                        "for 50 detections in ONE launch reading the [1,415,96,320] regression map (detector_infer.py:107,"
                                        "181-188); eager through the Python wrapper, and the launch alone replayed from a CUDA graph"},
        "edge_select_top1500": {"objects_per_s": sel_n / (ms_sel * 1e-3), "ms": ms_sel, "objects": sel_n,
                                "hbm_gbs": (B_SOLVE + 12 * K_SEL) * sel_n / (ms_sel * 1e-3) / 1e9,
                                "what": "a1 training branch: radix select + register bitonic sort of the 1500 winners + their depths"},
        "edge_solve_bwd_top1500": {"objects_per_s": sel_n / (ms_bwd * 1e-3), "ms": ms_bwd, "objects": sel_n,
                                   "fp32_tflops": f_solve_bwd(N_KPTS) * sel_n / (ms_bwd * 1e-3) / 1e12,
                                   "what": "a9: backward of the selected depths into kps / kps_3d (per-keypoint gather, no atomics)"},
        "gmw_train_step_b8": {"ms": ms_train, "objects_per_s": 8 * world / (ms_train * 1e-3),
                              "what": "configs[2]: compute_z + edge MLP fwd + softmax aggregate + L1 loss + full backward (all GEMMs on "
                                      "tcgen05) for 8 objects per GPU%s; optimizer step excluded" % (" + gradient all-reduce" if world > 1 else "")},
        "gmw_train_step_b8_cuda_graph": {"ms": ms_train_graph, "objects_per_s": 8 * world / (ms_train_graph * 1e-3),
                                         "what": "the same step captured once in a CUDA graph (dcd_b200.GraphedGmwStep) and replayed; inputs "
                                                 "copied into the static buffers inside the timed region"},
        "gmw_train_step_b64": {"ms": ms_train64, "objects_per_s": 64 * world / (ms_train64 * 1e-3),
                               "mlp_tflops": 3 * F_MLP * 64 / (ms_train64 * 1e-3) / 1e12,
                               "what": "the same step at 64 objects per GPU (fwd + bwd = 3 x the folded forward GEMM FLOPs)"},
        "gmw_cls_forward_b8": {"ms": ms_cls, "objects_per_s": 8 / (ms_cls * 1e-3),
                               "what": "edge MLP + E x E feature distances + Sinkhorn (lambda 10, <= 100 iterations, "
                                       "GMW/model/model.py:170-192) -> sum P, trace P for 8 objects; forward only"},
    }
    if torch_ctx is not None:
        stages["torch_cuda_oracle"] = torch_ctx
    return stages


# --------------------------------------------------------------------------------------------------------------
# configs[3]: 2^20 objects, STRONG scaling, both pipelines, all-gather of the depths inside the timed region
# --------------------------------------------------------------------------------------------------------------
def run_sweep1m(args):
    ctx = Ctx(args)
    dcd_b200, L, dev, world, rank = ctx.dcd, ctx.L, ctx.dev, ctx.world, ctx.rank
    from dcd_b200 import synth
    from dcd_b200 import dist as ddist
    from dcd_b200._lib import check, ptr, stream_ptr
    peaks = ctx.peaks
    seed = synth.BASE_SEED + 3
    frames = (args.objects + 49) // 50
    counts = torch.full((frames,), 50, dtype=torch.int64)
    if frames * 50 != args.objects:
        counts[-1] = args.objects - (frames - 1) * 50
    bounds = ddist.shard_bounds(counts.tolist(), world)
    cum = torch.cat([torch.zeros(1, dtype=torch.int64), counts.cumsum(0)])

    def shard(r):
        return make_objects_chunked(frames_of_shard(counts, cum, bounds[r]), N_KPTS, seed + 1000 * r)
    ob = shard(rank)
    N, N_total = ob.N, int(cum[-1])
    lo_obj, hi_obj = bounds[rank]
    model = dcd_b200.GMW().to(dev).load_reference_state_dict(synth.random_state_dict(WEIGHT_SEED))
    p4, p6 = model.params4.detach(), model.params6.detach()
    d_k2, d_k3 = ob.kps_norm.to(dev), ob.kps_3d.to(dev)
    d_rot = ob.rot_y.reshape(-1).contiguous().to(dev)
    d_kps, d_K = ob.kps.to(dev), ob.K.to(dev)

    # ---- pipeline (i): DGDE inference, a1 + a3 (edge solve + mean), then the all-gather
    sizes = [hi - lo for lo, hi in bounds]
    m = max(sizes)
    equal = all(s == m for s in sizes)
    send = torch.zeros((m,), dtype=torch.float32, device=dev)
    recv = torch.empty((world * m,), dtype=torch.float32, device=dev)

    def dgde_step():
        check(L.dcd_edge_solve_fwd(ptr(d_kps), ptr(d_k3), ptr(d_rot), ptr(d_K), N, N_KPTS, 2.0, 80.0, 3, 0, ptr(send), stream_ptr()), "solve")
        if world > 1:
            ctx.dist.all_gather_into_tensor(recv, send)

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        ctx.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        ctx.barrier()
        return a.elapsed_time(b) / steps
    dg_steps = max(args.steps, 20)
    ms_dgde = timed(dgde_step, dg_steps, max(args.warmup, 5))
    # the same step replayed from a CUDA graph (kernel + collective captured together: one launch per step instead of two
    # host round trips — SURVEY 7-H6: at 8 GPUs the solve is ~0.1 ms, comparable to the collective's launch latency)
    ms_dgde_graph = None
    try:
        if world > 1 and not args.graph_collective:          # capturing an NCCL collective is opt-in: a failed capture on one
            raise RuntimeError("skipped (pass --graph-collective)")   # rank would leave the others waiting in the collective
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(3):
                dgde_step()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        with torch.cuda.graph(g):
            dgde_step()
        ms_dgde_graph = timed(g.replay, dg_steps, 5)
    except Exception as e:                                   # graph capture of the collective unsupported here: report the eager figure only
        ms_dgde_graph = None
        if rank == 0 and "skipped" not in str(e):
            sys.stderr.write("CUDA-graph capture of solve + all-gather failed: %r\n" % (e,))
        torch.cuda.synchronize()
    # two half-shards: the all-gather of the first half runs on NCCL's stream while the second half is being solved
    ms_dgde_overlap = None
    if world > 1:
        h = (N + 1) // 2
        mh = (m + 1) // 2
        send2 = torch.zeros((2, mh), dtype=torch.float32, device=dev)
        recv2 = torch.empty((2, world * mh), dtype=torch.float32, device=dev)
        halves = [(0, h), (h, N)]

        def dgde_step_overlap():
            works = []
            for i, (a0, a1) in enumerate(halves):
                if a1 > a0:
                    check(L.dcd_edge_solve_fwd(ptr(d_kps[a0:]), ptr(d_k3[a0:]), ptr(d_rot[a0:]), ptr(d_K[a0:]), a1 - a0, N_KPTS, 2.0, 80.0, 3,
                                               0, ptr(send2[i]), stream_ptr()), "solve")
                works.append(ctx.dist.all_gather_into_tensor(recv2[i], send2[i], async_op=True))
            for w in works:
                w.wait()
        ms_dgde_overlap = timed(dgde_step_overlap, dg_steps, 5)
    ms_solve_only = time_kernel(lambda: check(L.dcd_edge_solve_fwd(ptr(d_kps), ptr(d_k3), ptr(d_rot), ptr(d_K), N, N_KPTS, 2.0, 80.0, 3,
                                                                   0, ptr(send), stream_ptr()), "solve"), reps=20)
    dgde_full = recv.view(world, m)                          # [rank][padded shard]
    dgde_local = send[:N].clone()

    # ---- pipeline (ii): GMW, a4 - a8 forward, then the all-gather (the metric)
    fw = GmwForward(ctx, N, N_KPTS, args.chunk, p4, p6)

    def gather():
        if world > 1:
            return ddist.all_gather_depths(fw.depth_out, bounds)
        return fw.depth_out
    for _ in range(args.warmup):
        fw.step(d_k2, d_k3, d_rot, False)
        gather()
    fw.launches = 0
    sampler = ClockSampler(ctx.local_rank)
    ctx.barrier()
    if rank == 0:
        sampler.start()
    t_beg, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_beg.record()
    for _ in range(args.steps):
        fw.step(d_k2, d_k3, d_rot, True)
        full = gather()
    t_end.record()
    ctx.barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms = t_beg.elapsed_time(t_end)
    mlp_ms = sum(a.elapsed_time(b) for a, b, _ in fw.mlp_events)
    mlp_objs = sum(nc for _, _, nc in fw.mlp_events)
    assert full.numel() == N_total
    full = full.clone()
    if rank == 0:
        dump_outputs(args, {"depth": full})

    def recompute(other):
        ob2 = shard(other)
        f2 = GmwForward(ctx, ob2.N, N_KPTS, args.chunk, p4, p6)
        f2.step(ob2.kps_norm.to(dev), ob2.kps_3d.to(dev), ob2.rot_y.reshape(-1).contiguous().to(dev), False)
        torch.cuda.synchronize()
        return f2.depth_out
    shard_check = check_shard_bit_equality(ctx, full, bounds, recompute)
    dgde_check = None
    if world > 1 and rank == 0:
        ob2 = shard(1)
        out2 = torch.empty((ob2.N,), dtype=torch.float32, device=dev)
        o_kps, o_k3, o_rot, o_K = ob2.kps.to(dev), ob2.kps_3d.to(dev), ob2.rot_y.reshape(-1).contiguous().to(dev), ob2.K.to(dev)
        check(L.dcd_edge_solve_fwd(ptr(o_kps), ptr(o_k3), ptr(o_rot), ptr(o_K), ob2.N, N_KPTS, 2.0, 80.0, 3, 0, ptr(out2),
                                   stream_ptr()), "solve")
        torch.cuda.synchronize()
        dgde_check = bool(torch.equal(out2, dgde_full[1][: ob2.N]))
        if not dgde_check:
            raise AssertionError("DGDE depths of rank 1 differ from their single-rank recomputation")

    # ---- e2e: host buffers in, host depths out, through the public API
    h_k2, h_k3, h_rot = ob.kps_norm.pin_memory(), ob.kps_3d.pin_memory(), ob.rot_y.reshape(-1).contiguous().pin_memory()
    h_out = torch.empty((N,), dtype=torch.float32).pin_memory()

    def e2e_step():
        out = dcd_b200.gmw_weighted_depth(h_k2.to(dev, non_blocking=True), h_k3.to(dev, non_blocking=True),
                                          h_rot.to(dev, non_blocking=True), model, chunk=fw.chunk)
        if world > 1:
            out = ddist.all_gather_depths(out, bounds)[lo_obj:hi_obj]
        h_out.copy_(out, non_blocking=True)
    e2e_ms = timed(e2e_step, args.steps, 1) * args.steps

    ms, e2e_ms, mlp_ms_max, ms_dgde, ms_solve_only = ctx.max_over_ranks([ms, e2e_ms, mlp_ms, ms_dgde, ms_solve_only])
    if ms_dgde_graph is not None:
        ms_dgde_graph = ctx.max_over_ranks([ms_dgde_graph])[0]
    if ms_dgde_overlap is not None:
        ms_dgde_overlap = ctx.max_over_ranks([ms_dgde_overlap])[0]
    if rank == 0:
        fp32_peak = ctx.fp32_peak(clocks)
        value = N_total * args.steps / (ms * 1e-3)
        mlp_tflops = F_MLP * mlp_objs / (mlp_ms * 1e-3) / 1e12
        best_dgde = min(x for x in (ms_dgde, ms_dgde_graph, ms_dgde_overlap) if x is not None)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[3]: %d-object synthetic sweep (%d frames of 50, 73 keypoints) sharded by frame over %d GPU(s): "
                                   "compute_z + edge-weight MLP + softmax-weighted depth, forward only, + all-gather of the per-object "
                                   "depths; total work fixed (strong scaling)" % (N_total, frames, world),
                       "objects_per_gpu": N, "objects_total": N_total, "chunk_objects": fw.chunk, "net_depth": DEPTH,
                       "l2_policy": "inputs (%.0f MB per GPU) and the per-chunk feature stream exceed L2" % (N * 1464 / 1e6)},
            "e2e": {"value": N_total * args.steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": N * (N_KPTS * 20 + 4),
                    "d2h_bytes_per_step": N * 4, "api": "dcd_b200.gmw_weighted_depth on pinned host tensors"},
            "gpu_launches": fw.launches,
            "roofline": {"kernel": "mlp_fused_kernel", "bound": "tensor", "achieved": mlp_tflops, "peak": peaks["bf16_tflops_sustained"],
                         "unit": "TFLOP/s", "frac": mlp_tflops / peaks["bf16_tflops_sustained"],
                         "traffic": measured_traffic("mlp_fused_kernel") if fw.chunk == 2048 else None,
                         "flops_per_object": F_MLP, "share_of_step": mlp_ms_max / ms},
            "stages": {
                "dgde_pipeline": {"what": "pipeline (i): DGDE inference edge solve + mean (a1 + a3) on the same %d objects, then ONE all-gather "
                                          "of the [N] depths; strong scaling" % N_total,
                                  "objects_per_s": N_total / (best_dgde * 1e-3), "ms_per_step": best_dgde,
                                  "ms_eager": ms_dgde, "ms_cuda_graph": ms_dgde_graph, "ms_two_chunks_overlapped": ms_dgde_overlap,
                                  "ms_solve_kernel_only": ms_solve_only,
                                  "fp32_tflops_per_gpu": F_SOLVE * N / (ms_solve_only * 1e-3) / 1e12,
                                  "frac_fp32_roofline_kernel": F_SOLVE * N / (ms_solve_only * 1e-3) / 1e12 / fp32_peak,
                                  "allgather_and_launch_ms": best_dgde - ms_solve_only,
                                  "bit_identical_to_single_rank": dgde_check},
            },
            "clocks": clocks,
        }
        if shard_check is not None:
            line["shard_check"] = shard_check
        print(json.dumps(line), flush=True)
    ctx.finish()


# --------------------------------------------------------------------------------------------------------------
# configs[4]: 256 keypoints (32 640 edges), forward + backward
# --------------------------------------------------------------------------------------------------------------
def run_stress256(args):
    ctx = Ctx(args)
    dcd_b200, L, dev, world, rank = ctx.dcd, ctx.L, ctx.dev, ctx.world, ctx.rank
    from dcd_b200 import synth
    from dcd_b200 import dist as ddist
    from dcd_b200._lib import check, ptr, stream_ptr
    peaks = ctx.peaks
    n, E = 256, edges_of(256)
    N_solve, N_mlp = 4096, 64                                # per GPU (SURVEY 8d cfg 5), weak scaling
    seed = synth.BASE_SEED + 4
    ob = synth.make_objects(N=N_solve, n=n, seed=seed + 1000 * rank)
    d_kps, d_k3, d_K = ob.kps.to(dev), ob.kps_3d.to(dev), ob.K.to(dev)
    d_rot = ob.rot_y.reshape(-1).contiguous().to(dev)
    d_k2 = ob.kps_norm.to(dev)
    st = stream_ptr()

    # ---- (a) DGDE training pattern a1(train) + a9 on 4096 objects: top-1500 selection + depths, backward into the keypoints
    idx = torch.empty((N_solve, K_SEL), dtype=torch.int64, device=dev)
    zsel = torch.empty((N_solve, K_SEL), dtype=torch.float32, device=dev)
    g_sel = torch.randn((N_solve, K_SEL), device=dev)
    g_kps = torch.empty((N_solve, n, 2), device=dev)
    g_k3 = torch.empty((N_solve, n, 3), device=dev)
    mean = torch.empty((N_solve,), device=dev)

    def dgde_train():
        check(L.dcd_edge_select_fwd(ptr(d_kps), ptr(d_k3), ptr(d_rot), ptr(d_K), 0, N_solve, n, K_SEL, 2.0, 80.0, 3, ptr(idx), ptr(zsel),
                                    0, 0, st), "select")
        check(L.dcd_edge_solve_bwd(ptr(d_kps), ptr(d_k3), ptr(d_rot), ptr(d_K), N_solve, n, 2.0, 80.0, 3, ptr(idx), K_SEL, ptr(g_sel), 0,
                                   ptr(g_kps), ptr(g_k3), st), "bwd")
    ms_dgde = time_kernel(dgde_train, reps=5)
    ms_sel = time_kernel(lambda: check(L.dcd_edge_select_fwd(ptr(d_kps), ptr(d_k3), ptr(d_rot), ptr(d_K), 0, N_solve, n, K_SEL, 2.0, 80.0, 3,
                                                             ptr(idx), ptr(zsel), 0, 0, st), "select"), reps=5)
    ms_mean = time_kernel(lambda: check(L.dcd_edge_solve_fwd(ptr(d_kps), ptr(d_k3), ptr(d_rot), ptr(d_K), N_solve, n, 2.0, 80.0, 3, 0,
                                                             ptr(mean), st), "solve"), reps=10)

    # ---- (b) GMW training step a4 - a8 + a10 on 64 objects per GPU (the step of this config)
    t_k2, t_k3 = d_k2[:N_mlp].contiguous(), d_k3[:N_mlp].contiguous()
    t_rot, t_gt = d_rot[:N_mlp].reshape(-1, 1).contiguous(), ob.gt_depth[:N_mlp].to(dev)
    model = dcd_b200.GMW().to(dev).load_reference_state_dict(synth.random_state_dict(WEIGHT_SEED))
    fwd_ev = []

    def train_step(record=False):
        model.zero_grad(set_to_none=True)
        Zt, idxt = dcd_b200.compute_z(t_k2, t_k3, t_rot)
        if record:
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record()
        wt, _ = model(t_k2, t_k3, t_rot, None)
        if record:
            e1.record()
        loss, depth = dcd_b200.compute_reg_loss(Zt, wt, t_gt, idxt)
        loss.backward()
        if record:
            e2.record()
            fwd_ev.append((e0, e1, e2))
        if world > 1:
            ddist.allreduce_gradients(model)
        return loss, depth
    for _ in range(max(args.warmup, 3)):
        train_step()
    sampler = ClockSampler(ctx.local_rank)
    ctx.barrier()
    if rank == 0:
        sampler.start()
    t_beg, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_beg.record()
    for _ in range(args.steps):
        loss, depth = train_step(True)
    t_end.record()
    ctx.barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms = t_beg.elapsed_time(t_end)
    fwd_ms = sum(a.elapsed_time(b) for a, b, _ in fwd_ev)
    bwd_ms = sum(b.elapsed_time(c) for _, b, c in fwd_ev)
    assert torch.isfinite(loss).all() and torch.isfinite(model.params4.grad).all()
    if rank == 0:
        dump_outputs(args, {"loss": loss, "depth": depth, "grad_params4": model.params4.grad, "grad_params6": model.params6.grad})

    # e2e: host inputs, host loss, through the public API
    h_k2, h_k3, h_rot, h_gt = t_k2.cpu().pin_memory(), t_k3.cpu().pin_memory(), t_rot.cpu().pin_memory(), t_gt.cpu().pin_memory()
    h_loss = torch.empty((), dtype=torch.float32).pin_memory()

    def e2e_step():
        k2, k3 = h_k2.to(dev, non_blocking=True), h_k3.to(dev, non_blocking=True)
        rot, gt = h_rot.to(dev, non_blocking=True), h_gt.to(dev, non_blocking=True)
        model.zero_grad(set_to_none=True)
        Zt, idxt = dcd_b200.compute_z(k2, k3, rot)
        wt, _ = model(k2, k3, rot, None)
        lo_, _ = dcd_b200.compute_reg_loss(Zt, wt, gt, idxt)
        lo_.backward()
        if world > 1:
            ddist.allreduce_gradients(model)
        h_loss.copy_(lo_.detach(), non_blocking=True)
    e2e_step()
    ctx.barrier()
    e_beg, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e_beg.record()
    for _ in range(args.steps):
        e2e_step()
    e_end.record()
    ctx.barrier()
    e2e_ms = e_beg.elapsed_time(e_end)

    ms, e2e_ms, fwd_ms, bwd_ms, ms_dgde, ms_sel, ms_mean = ctx.max_over_ranks([ms, e2e_ms, fwd_ms, bwd_ms, ms_dgde, ms_sel, ms_mean])
    if rank == 0:
        fp32_peak = ctx.fp32_peak(clocks)
        EP = 128 * ((E + 127) // 128)
        # layer-wise schedule: per block and net the forward writes / reads X, Y1, Y2 (+ saves them for the backward)
        fwd_bytes = 24 * 128 * EP * DEPTH * 2                    # B per object: the 198 MB / object model of n = 73 scaled by EP
        hbm_fwd = fwd_bytes * N_mlp * args.steps / (fwd_ms * 1e-3) / 1e9
        mlp_tflops = 3 * f_mlp(n) * N_mlp * args.steps / ((fwd_ms + bwd_ms) * 1e-3) / 1e12
        line = {
            "metric": METRIC, "value": N_mlp * world * args.steps / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[4]: dense keypoint stress, 256 keypoints / 32 640 edges per object: GMW training step (compute_z + "
                                   "edge MLP forward with saved activations + softmax aggregate + L1 loss + full backward%s) on %d objects per "
                                   "GPU; the DGDE pattern a1(train) + a9 on %d objects per GPU is reported under stages"
                                   % (" + gradient all-reduce" if world > 1 else "", N_mlp, N_solve),
                       "objects_per_gpu": N_mlp, "objects_total": N_mlp * world, "net_depth": DEPTH,
                       "l2_policy": "the activations of one step (%.1f GB) exceed L2 many times over" % (fwd_bytes * N_mlp / 1e9)},
            "e2e": {"value": N_mlp * world * args.steps / (e2e_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": N_mlp * (n * 20 + 8), "d2h_bytes_per_step": 4,
                    "api": "dcd_b200.compute_z + GMW.forward + compute_reg_loss + backward on pinned host tensors, loss read back"},
            "gpu_launches": args.steps * (2 + 4 + 1 + 2 * DEPTH + 1 + 1 + 3 + 5 * DEPTH + 2),
            "roofline": {"kernel": "mlp_tc_kernel<FIRST|B|CA> (layer-wise edge MLP forward, one persistent tcgen05 launch per segment between "
                                   "context norms; n = 256 does not fit the on-chip schedule)",
                         "bound": "hbm", "achieved": hbm_fwd, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": hbm_fwd / peaks["hbm_gbs"],
                         "traffic": measured_traffic("mlp_tc_kernel_n256"),
                         "bytes_per_object_forward": fwd_bytes, "forward_ms_per_step": fwd_ms / args.steps,
                         "backward_ms_per_step": bwd_ms / args.steps,
                         "mlp_tflops_fwd_bwd": mlp_tflops, "frac_tensor_peak": mlp_tflops / peaks["bf16_tflops_sustained"],
                         "peak_source": "%s STREAM-style copy bandwidth (of measured)" % peaks["source"]},
            "stages": {
                "dgde_train_pattern_n256": {"objects_per_s": N_solve / (ms_dgde * 1e-3), "ms": ms_dgde, "objects": N_solve,
                                            "what": "a1(train) + a9: top-1500 of 32 640 edges by |V| + depths, then the backward into kps / kps_3d"},
                "edge_select_top1500_n256": {"objects_per_s": N_solve / (ms_sel * 1e-3), "ms": ms_sel},
                "edge_solve_bwd_n256": {"objects_per_s": N_solve / ((ms_dgde - ms_sel) * 1e-3), "ms": ms_dgde - ms_sel,
                                        "fp32_tflops": f_solve_bwd(n) * N_solve / ((ms_dgde - ms_sel) * 1e-3) / 1e12},
                "dgde_solve_mean_n256": {"objects_per_s": N_solve / (ms_mean * 1e-3), "ms": ms_mean,
                                         "fp32_tflops": f_solve(n) * N_solve / (ms_mean * 1e-3) / 1e12,
                                         "frac_fp32_roofline": f_solve(n) * N_solve / (ms_mean * 1e-3) / 1e12 / fp32_peak},
                "fp32_peak_tflops": fp32_peak,
            },
            "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    ctx.finish()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.config in ("kitti_val", "kitti_val_full"):
        run_kitti_val(args)
    elif args.config == "sweep1m":
        run_sweep1m(args)
    else:
        run_stress256(args)


if __name__ == "__main__":
    main()
