"""CPU-only checks: the C-ABI library loads and exports every symbol of include/dcd_b200.h, argument
validation, host-side logic (weight blobs, synthetic generator, sharding, patching).  No compute call
is made (there is no GPU here and the product has no CPU path)."""
import ctypes
import os
import re
import types

import pytest
import torch

import dcd_b200
from dcd_b200 import _lib, dist as ddist, patch, synth, weights
from oracle import dcd_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from dcd_b200.build import build_library
    return _lib.load_library(build_library())


def header_functions():
    src = open(os.path.join(ROOT, "include", "dcd_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(dcd_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(lib):
    names = header_functions()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), "symbol %s declared in include/dcd_b200.h is not exported" % n
    assert set(names) == set(_lib.SIGNATURES), "ctypes prototypes out of sync with the header"


def test_library_has_no_torch_dependency():
    out = os.popen("ldd %s" % _lib.LIB_PATH).read()
    assert "torch" not in out and "c10" not in out


def test_version_strerror_and_size_queries(lib):
    assert lib.dcd_version() == 2
    assert lib.dcd_strerror(0) == b"ok"
    assert b"workspace" in lib.dcd_strerror(-2)
    assert lib.dcd_gmw_param_count(4, 12) == 595072 and lib.dcd_gmw_param_count(6, 12) == 595328
    assert lib.dcd_gmw_param_count(4, 12) + lib.dcd_gmw_param_count(6, 12) == 1190400     # SURVEY fact 8
    E, T = 2628, 21
    acts_and_stats = 4 * (2 * 3 * 128 * T * 128 + 2 * 12 * 2 * T * 128 * 2)
    scales = 768                                         # 72 per-matrix (scale, 1/scale) pairs, 256-byte aligned
    # tail of the fused forward: 48 matrices (folded preconv.conv1 and conv2 per block and net): scales, biases, pre-split
    # FP16 hi/lo weight image; then the statistics exchange buffer [group][object][slot][rank][128] float2
    image = 512 + 48 * 128 * 4 + 48 * 128 * 128 * 4 + 10 * 3 * 2 * 24 * 128 * 8
    image += 24 * (128 * 128 + 128) * 4 + 256            # folded preconv.conv1 layers (Wf^T, bf) + their running maxima
    assert lib.dcd_gmw_workspace_bytes(1, 73, 12, 0) == acts_and_stats + scales + image
    assert lib.dcd_gmw_workspace_bytes(0, 73, 12, 0) == 0
    assert lib.dcd_gmw_workspace_bytes(8, 73, 12, 1) > lib.dcd_gmw_workspace_bytes(8, 73, 12, 0)
    assert lib.dcd_gmw_bwd_scratch_bytes(8, 73, 12) > 0
    assert lib.dcd_gmw_depth_workspace_bytes(100000, 73, 12, 1024) == lib.dcd_gmw_depth_workspace_bytes(2000, 73, 12, 1024)


def test_argument_validation_without_a_gpu(lib):
    """Invalid arguments are rejected before any CUDA call (so this runs on a CPU-only box)."""
    assert lib.dcd_edge_solve_fwd(0, 0, 0, 0, 5, 73, 2.0, 80.0, 3, 0, 0, 0) == -1        # null pointers
    assert lib.dcd_edge_solve_fwd(8, 8, 8, 8, 5, 1, 2.0, 80.0, 3, 8, 8, 0) == -1          # n < 2
    assert lib.dcd_edge_solve_fwd(8, 8, 8, 8, 5, 257, 2.0, 80.0, 3, 8, 8, 0) == -1        # n > 256
    assert lib.dcd_edge_solve_fwd(8, 8, 8, 0, 5, 73, 2.0, 80.0, 3, 8, 8, 0) == -1         # flags need K
    assert lib.dcd_edge_solve_fwd(8, 8, 8, 8, 0, 73, 2.0, 80.0, 3, 8, 8, 0) == 0          # N = 0 is a no-op
    assert lib.dcd_edge_select_fwd(8, 8, 8, 8, 0, 5, 8, 1500, 2.0, 80.0, 3, 8, 8, 0, 0, 0) == -1   # k > E (28 edges)
    assert lib.dcd_gmw_aggregate_fwd(8, 8, 8, 4, 100, 200, 0, 8, 0, 0) == -1               # k > E
    assert lib.dcd_gmw_weights_fwd(8, 8, 16, 16, 4, 73, 12, 0, 8, 0, 0, 256, 16, 0) == -2  # workspace too small
    # frame epilogue entries (SURVEY 8f N2/N4)
    assert lib.dcd_dgde_locate_fwd(8, 8, 8, 0, 8, 8, 8, 0, 0, 5, 73, 2.0, 80.0, 3, 4.0, 8, 8, 0) == -1       # K is required
    assert lib.dcd_dgde_locate_fwd(8, 8, 8, 8, 8, 8, 8, 0, 0, 5, 73, 2.0, 80.0, 3, 4.0, 0, 0, 0) == -1       # no output
    assert lib.dcd_dgde_locate_fwd(0, 0, 0, 8, 8, 8, 8, 0, 0, 5, 73, 2.0, 80.0, 3, 4.0, 0, 8, 0) == -1       # no solve: depth_in
    assert lib.dcd_dgde_locate_fwd(8, 8, 8, 8, 8, 8, 8, 0, 0, 5, 300, 2.0, 80.0, 3, 4.0, 8, 8, 0) == -1      # n > 256
    assert lib.dcd_dgde_locate_fwd(8, 8, 8, 8, 8, 8, 8, 0, 0, 0, 73, 2.0, 80.0, 3, 4.0, 8, 8, 0) == 0        # N = 0
    assert lib.dcd_dgde_depth_ensemble_fwd(8, 8, 8, 8, 0, 8, 0, 5, 4.0, 1e-3, 0.1, 100.0, 8, 8, 8, 0, 0, 0) == -1   # direct without its uncertainty
    assert lib.dcd_dgde_depth_ensemble_fwd(8, 8, 8, 0, 0, 8, 0, 5, 4.0, 1e-3, 0.1, 100.0, 0, 0, 0, 0, 8, 0) == -1   # scores_out without scores
    assert lib.dcd_dgde_depth_ensemble_fwd(8, 8, 8, 0, 0, 0, 0, 5, 4.0, 1e-3, 0.1, 100.0, 0, 0, 0, 0, 0, 0) == -1   # nothing to compute
    assert lib.dcd_poi_gather_fwd(8, 8, 2, 50, 0, 100, 8, 0) == -1 and lib.dcd_poi_gather_fwd(8, 8, 0, 50, 4, 100, 8, 0) == 0
    assert lib.dcd_gmw_ray_rescale_fwd(8, 8, 0, 5, 8, 0) == -1 and lib.dcd_gmw_ray_rescale_fwd(8, 8, 8, 0, 8, 0) == 0


def test_ops_reject_cpu_tensors():
    ob = synth.make_objects(N=2, n=73, seed=1)
    with pytest.raises(RuntimeError, match="CUDA"):
        dcd_b200.decode_pairs_kpts_depth(ob.kps, ob.kps_3d, ob.rot_y, ob.K)
    with pytest.raises(RuntimeError, match="CUDA"):
        dcd_b200.compute_z(ob.kps_norm, ob.kps_3d, ob.rot_y)
    with pytest.raises(RuntimeError, match="CUDA"):
        dcd_b200.GMW()(ob.kps_norm, ob.kps_3d, ob.rot_y, None)


def test_product_never_imports_the_oracle():
    for root, _, files in os.walk(os.path.join(ROOT, "dcd_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(root, f)).read()
                assert "oracle" not in src, "%s references the oracle" % f


def test_weight_blob_round_trip():
    sd = O.random_state_dict(5)
    for name, cin in weights.NET_NAMES:
        blob = weights.pack_state_dict(sd, name, cin)
        assert blob.numel() == weights.blob_size(cin) and blob.dtype == torch.float32
        back = weights.unpack_blob(blob, name, cin)
        for k, v in back.items():
            assert torch.equal(v, sd[k]) and v.shape == sd[k].shape
        # conv_in is stored transposed [in][out] at the start of the blob
        w = sd[name + ".conv_in.0.weight"][:, :, 0]
        assert torch.equal(blob[: cin * 128].reshape(cin, 128), w.t())
    m = dcd_b200.GMW().load_reference_state_dict({"module." + k: v for k, v in sd.items()})   # DDP prefix (main.py:286)
    back = m.reference_state_dict()
    assert all(torch.equal(back[k], sd[k]) for k in sd)
    assert sum(p.numel() for p in m.parameters()) == 1190400


def test_synthetic_generator_is_seeded_and_kitti_shaped():
    a = synth.make_objects(N=60, n=73, seed=3)
    b = synth.make_objects(N=60, n=73, seed=3)
    assert torch.equal(a.kps, b.kps) and torch.equal(a.kps_3d, b.kps_3d) and torch.equal(a.mask, b.mask)
    assert a.kps.shape == (60, 73, 2) and a.kps_3d.shape == (60, 73, 3) and a.K.shape == (60, 3, 4)
    assert a.counts.tolist() == [50, 10] and a.frame_id[49] == 0 and a.frame_id[50] == 1
    assert float(a.K[0, 1, 1]) == pytest.approx(721.5377) and float(a.K[0, 2, 3]) == pytest.approx(0.002745884)
    # last ten keypoints: 8 corners then bottom / top centre of the box (kitti_utils.py:136-147)
    assert torch.allclose(a.kps_3d[:, -2], torch.zeros(60, 3)) and bool((a.kps_3d[:, -1, 1] < 0).all())
    # geometry-consistent: the mean edge depth lands near the generating depth
    d = O.dgde_pipeline(a.kps, a.kps_3d, a.rot_y, a.K)
    assert float(((d - a.gt_depth).abs() / a.gt_depth).median()) < 0.05
    val = synth.frame_counts(3769, 50, True, synth.BASE_SEED + 1)
    assert val.numel() == 3769 and int(val.min()) >= 1 and int(val.max()) <= 50


def test_shard_bounds_cover_and_balance():
    counts = synth.frame_counts(3769, 50, True, 7).tolist()
    total = sum(counts)
    for world in (1, 2, 4, 8):
        b = ddist.shard_bounds(counts, world)
        assert b[0][0] == 0 and b[-1][1] == total
        assert all(b[r][1] == b[r + 1][0] for r in range(world - 1))
        sizes = [hi - lo for lo, hi in b]
        assert max(sizes) - min(sizes) <= 100            # within two frames of each other
        cum, cuts = 0, {0}
        for c in counts:
            cum += c
            cuts.add(cum)
        assert all(lo in cuts and hi in cuts for lo, hi in b)   # shards end on frame boundaries
    assert ddist.shard_bounds([5], 4) == [(0, 5), (5, 5), (5, 5), (5, 5)]
    # frames without detections (common in KITTI), also trailing ones
    assert ddist.shard_bounds([3, 0], 1) == [(0, 3)]
    assert ddist.shard_bounds([3, 2, 0], 2) == [(0, 3), (3, 5)]
    assert ddist.shard_bounds([0, 0], 2) == [(0, 0), (0, 0)]
    assert ddist.shard_bounds([0, 3, 0, 0, 2, 0], 3) == [(0, 3), (3, 5), (5, 5)]
    assert ddist.shard_bounds([], 2) == [(0, 0), (0, 0)]


def test_patch_install_and_uninstall():
    class FakeEncoder:
        def decode_pairs_kpts_depth(self, *a, **k):
            return "reference"

    main = types.ModuleType("main")
    main.compute_z = lambda *a: "ref_z"
    main.compute_reg_loss = lambda *a: "ref_loss"
    patch.install(anno_encoder_cls=FakeEncoder, gmw_main=main)
    assert main.compute_z is dcd_b200.compute_z and main.compute_reg_loss is dcd_b200.compute_reg_loss
    ob = synth.make_objects(N=1, n=73, seed=1)
    with pytest.raises(RuntimeError, match="CUDA"):          # routed into the CUDA op (which refuses CPU tensors)
        FakeEncoder().decode_pairs_kpts_depth(ob.kps, ob.kps_3d, ob.rot_y, ob.K)
    patch.uninstall()
    assert FakeEncoder().decode_pairs_kpts_depth() == "reference" and main.compute_z() == "ref_z"


def test_bench_reference_arm_runs_on_cpu(tmp_path):
    import json
    import subprocess
    import sys
    import numpy as np
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "0", "--cpu-sample", "16", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0 and line["unit"] == "objects/s"
    assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0
    # --dump-outputs: the depths of the last timed step (8 objects of seed 101)
    assert sorted(os.listdir(tmp_path)) == ["depth.npy"]
    depth = np.load(tmp_path / "depth.npy")
    assert depth.dtype == np.float32 and depth.shape == (8,)
    ob = synth.make_objects(N=8, n=73, seed=101)
    with torch.no_grad():
        want = O.gmw_pipeline(ob.kps_norm, ob.kps_3d, ob.rot_y, O.random_state_dict(7))
    assert float(((torch.from_numpy(depth) - want).abs() / want.abs()).max()) < 1e-5


def test_patch_against_reference_shaped_objects():
    """install() on stand-ins of the reference objects: an Anno_Encoder class whose decode_pairs_kpts_depth is the oracle's,
    a GMW/main.py module with the oracle's compute_z / compute_reg_loss, and an nn.Module with the reference GMW's
    parameter tree; weights copied bit-exactly, uninstall() restores everything."""
    from test_gpu_patch import reference_shaped_gmw

    class Anno_Encoder:
        def decode_pairs_kpts_depth(self, kps, kps_3d, rot_y, K, training=False, kpts_2d_mask=None, gt_depth=None, weight=None):
            return O.decode_pairs_kpts_depth(kps, kps_3d, rot_y, K, training=training, kpts_2d_mask=kpts_2d_mask)

    enc = Anno_Encoder()
    ref_main = types.ModuleType("main")
    ref_main.compute_z, ref_main.compute_reg_loss = O.compute_z, O.compute_reg_loss
    model = reference_shaped_gmw(O.random_state_dict(3), 12).eval()
    orig_decode = type(enc).decode_pairs_kpts_depth
    orig_cz, orig_forward = ref_main.compute_z, model.forward
    n_keys = len(model.state_dict())
    patch.install(anno_encoder_cls=type(enc), gmw_main=ref_main, gmw_model=model)
    try:
        assert ref_main.compute_z is dcd_b200.compute_z
        assert len(model.state_dict()) == n_keys                     # the fast module is not registered as a sub-module
        assert model._dcd_b200.depth == 12 and model._dcd_b200.with_edge_P
        live = model._dcd_b200_blobs
        with torch.no_grad():
            p4, p6 = live.get()
        for (name, cin), blob in zip(weights.NET_NAMES, (p4, p6)):
            back = weights.unpack_blob(blob, name, cin)
            for k, v in back.items():
                assert torch.equal(v, model.state_dict()[k]), k
        # the blobs follow the live parameters: an optimizer step or a load_state_dict is seen by the next forward
        with torch.no_grad():
            assert live.get()[0] is p4                                   # cached while nothing changed
            first = next(model.parameters())
            first.add_(1.0)
            q4, _ = live.get()
            assert q4 is not p4 and not torch.equal(q4, p4)
            sd2 = {k: v + 0.5 for k, v in model.state_dict().items()}
            model.load_state_dict(sd2)
            r4, r6 = live.get()
            for (name, cin), blob in zip(weights.NET_NAMES, (r4, r6)):
                for k, v in weights.unpack_blob(blob, name, cin).items():
                    assert torch.equal(v, sd2[k]), k
        # under autograd the pack is differentiable: blob gradients land in the reference parameters' .grad
        b4, b6 = live.get()
        assert b4.requires_grad and b6.requires_grad
        g = torch.Generator().manual_seed(0)
        c4, c6 = torch.randn(b4.shape, generator=g), torch.randn(b6.shape, generator=g)
        ((b4 * c4).sum() + (b6 * c6).sum()).backward()
        for (name, cin), coef in zip(weights.NET_NAMES, (c4, c6)):
            expect = weights.unpack_blob(coef, name, cin)
            for k, p in model.named_parameters():
                if k.startswith(name):
                    assert torch.equal(p.grad, expect[k]), k
        model.zero_grad()
        ob = synth.make_objects(N=2, n=73, seed=2)
        with pytest.raises(RuntimeError, match="CUDA"):
            enc.decode_pairs_kpts_depth(ob.kps, ob.kps_3d, ob.rot_y, ob.K)
        with pytest.raises(RuntimeError, match="CUDA"):
            model(ob.kps_norm, ob.kps_3d, ob.rot_y, None)
    finally:
        patch.uninstall()
    assert type(enc).decode_pairs_kpts_depth is orig_decode and ref_main.compute_z is orig_cz
    assert model.forward == orig_forward and not hasattr(model, "_dcd_b200") and not hasattr(model, "_dcd_b200_blobs")
    d, _ = enc.decode_pairs_kpts_depth(ob.kps, ob.kps_3d, ob.rot_y, ob.K)        # the reference path works again
    assert d.shape == (2, 2628)
