"""dcd_b200.refine_detections (dcd_dgde_gmw_refine_fwd): the DGDE regression map to GMW-rescaled 3D locations in one
stream-ordered call.  Bit-identical to the hand composition frame_depths_from_map -> FP32 normalisation ->
gmw_weighted_depth -> ray_rescale on the same GPU, to wire.from_detector's keypoints, and within the GMW / location bars of
the oracle (FP32 on CUDA and FP64)."""
import numpy as np
import pytest
import torch

import dcd_b200
from dcd_b200 import synth, wire
from oracle import dcd_oracle as O
from conftest import rel_err

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
C, H, W, NK = 415, 96, 320, 73
CH = dcd_b200.ops.DGDE_CHANNELS


def image_P(b):
    """KITTI's P2 moved a little per image (focal lengths, principal point, 4th column); f_v != f_u, so that a u normalised
    with f_v cannot pass."""
    P = np.array(synth.P2, dtype=np.float64)
    P[0, 0] *= 1 + 0.02 * b
    P[1, 1] *= 1 + 0.02 * b + 1e-3
    P[0, 2] += 4.0 * b
    P[1, 2] -= 2.0 * b
    P[0, 3] += 0.5 * b
    return P


def make_frames(counts, seed):
    """B = len(counts) images with their own P and pad; geometry-consistent keypoint offsets, template points and sub-pixel
    offsets planted in a [B,415,96,320] map at distinct positions per image (as tests/test_gpu_locate.py)."""
    B = len(counts)
    g = torch.Generator().manual_seed(seed)
    ob = synth.make_objects(n=NK, seed=seed, counts=torch.tensor(counts))
    N = ob.N
    bi = ob.frame_id.clone()
    fmap = torch.randn(B, C, H, W, generator=g) * 0.1
    pos = torch.empty(N, dtype=torch.int64)
    for b in range(B):
        sel = (bi == b).nonzero().reshape(-1)
        pos[sel] = torch.randperm(H * W, generator=g)[:sel.numel()]
    pad_b = torch.tensor([[19.0, 5.0], [3.0, 7.0], [0.0, 0.0], [11.0, 2.0]])[:B]
    pad = pad_b[bi]
    pts = torch.stack(((pos % W).float(), (pos // W).float()), dim=1)
    ofs = torch.rand(N, 2, generator=g) - 0.5
    off = (ob.kps + pad.unsqueeze(1)) / 4 - (pts + ofs).unsqueeze(1)
    for d in range(N):
        b, p = int(bi[d]), int(pos[d])
        fmap[b, CH["3d_offset"]:CH["3d_offset"] + 2].view(2, -1)[:, p] = ofs[d]
        fmap[b, CH["extra_kpts_2d"]:CH["extra_kpts_2d"] + 2 * NK].view(2 * NK, -1)[:, p] = off[d].reshape(-1)
        fmap[b, CH["extra_kpts_3d"]:CH["extra_kpts_3d"] + 3 * NK].view(3 * NK, -1)[:, p] = ob.kps_3d[d].reshape(-1)
    dims = torch.stack((torch.full((N,), 3.9), -ob.kps_3d[:, -1, 1], torch.full((N,), 1.6)), dim=1)    # (l, h, w)
    P = np.stack([image_P(b) for b in range(B)])
    f = {"fm": fmap.to(DEV), "pos": pos.to(DEV), "rot": ob.rot_y.to(DEV), "dims": dims.to(DEV), "N": N, "B": B,
         "cpu": {"off": off, "pts": pts, "ofs": ofs, "k3": ob.kps_3d, "rot": ob.rot_y, "dims": dims, "bi": bi, "pad_b": pad_b}}
    if B == 1:                      # one image: the reference's [3,4] calibration and [2] pad, no batch index
        f.update(P=P[0], pad=pad_b[0].to(DEV), bi=None, P_obj=np.broadcast_to(P[0], (N, 3, 4)))
    else:
        f.update(P=P, pad=pad_b.to(DEV), bi=bi.to(DEV), P_obj=P[bi.numpy()])
    return f


@pytest.fixture(scope="module")
def model():
    return dcd_b200.GMW().to(DEV).load_reference_state_dict(O.random_state_dict(7))


def refine(f, model, **kw):
    with torch.no_grad():
        return dcd_b200.refine_detections(f["fm"], f["pos"], f["rot"], f["P"], f["pad"], f["dims"], model, batch_idxs=f["bi"],
                                          **kw)


def hand_composition(f, model, chunk):
    """What a caller chains by hand today: frame_depths_from_map -> normalisation -> gmw_weighted_depth -> ray_rescale."""
    with torch.no_grad():
        d, loc, kimg, k3 = dcd_b200.frame_depths_from_map(f["fm"], f["pos"], f["rot"], f["P"], f["pad"], dims=f["dims"],
                                                          batch_idxs=f["bi"], return_keypoints=True)
        Kd = torch.as_tensor(np.ascontiguousarray(f["P_obj"]), dtype=torch.float32).to(DEV)
        kimg, k3 = kimg[:, :NK], k3[:, :NK].contiguous()
        k2 = torch.stack(((kimg[..., 0] - Kd[:, None, 0, 2]) / Kd[:, None, 0, 0],
                          (kimg[..., 1] - Kd[:, None, 1, 2]) / Kd[:, None, 1, 1]), dim=-1)
        z, gidx = dcd_b200.gmw_weighted_depth(k2, k3, f["rot"], model, chunk=chunk, return_idx=True)
        out = dcd_b200.ray_rescale(loc, z, f["dims"][:, [1, 2, 0]])
    return {"dgde_depth": d, "dgde_location": loc, "gmw_depth": z, "location": out, "kpts_2d": k2, "kpts_3d": k3,
            "good_idx": gidx, "kimg": kimg}


FRAMES = {5: ([5], 11), 17: ([9, 8], 12), 40: ([12, 7, 11, 10], 13), 301: ([80, 75, 70, 76], 14)}
_cache = {}


def frames(N):
    if N not in _cache:
        _cache.clear()
        _cache[N] = make_frames(*FRAMES[N])
    return _cache[N]


@pytest.mark.parametrize("N", [5, 17, 40, 301])
@pytest.mark.parametrize("chunk", [1, 7, None])
def test_refine_equals_hand_composition_bit_for_bit(model, N, chunk):
    """N = 5, 17: unpaired MLP schedule; 40, 301: paired, ragged last triple; 1, 2 and 4 images with their own P and pad."""
    f = frames(N)
    chunk = chunk or N
    r = refine(f, model, chunk=chunk, return_inputs=True)
    h = hand_composition(f, model, chunk)
    for key in ("dgde_depth", "dgde_location", "gmw_depth", "location", "kpts_2d", "kpts_3d", "good_idx"):
        assert r[key].shape == h[key].shape and torch.equal(r[key], h[key]), key
    assert r["good_idx"].shape == (N, 1500) and bool(torch.isfinite(r["location"]).all())
    # the records of the binary / JSON hand-off: the same normalised keypoints as wire.from_detector, bit for bit
    rec = wire.from_detector(h["kimg"], h["kpts_3d"], f["rot"], h["dgde_location"], f["P_obj"], dim=f["dims"])
    assert np.array_equal(rec["kpts_2d"], r["kpts_2d"].cpu().numpy())
    assert np.array_equal(rec["kpts_3d"], r["kpts_3d"].cpu().numpy())
    # the GMW-rescaled location sits at the GMW depth (z * (z_gmw / z): one rounding of each)
    assert rel_err(r["location"][:, 2], r["gmw_depth"]) < 1e-6


def frame_locations(args, P, dims):
    """O.frame_locations in the inputs' precision (the oracle's decode_location_flatten allocates FP32 locations): edge
    depths -> mean -> project_image_to_rect((points + offsets) * 4 - pad, depth) -> y += h / 2."""
    if args[0].dtype == torch.float32:
        return O.frame_locations(*args, P, dims)[1]
    off, pts, ofs, pad, k3, rot = args
    K = torch.from_numpy(np.asarray(P)).unsqueeze(0).expand(off.shape[0], -1, -1)
    depth = O.compute_pairs_kpts_depth(off, pts, ofs, pad.reshape(-1), k3, rot, K)
    uv = (pts + ofs) * O.DOWN_RATIO - pad.reshape(1, 2)
    loc = O.project_image_to_rect(torch.cat((uv, depth[:, None]), dim=1), P)
    loc[:, 1] += dims[:, 1] / 2
    return loc


def test_refine_vs_oracle_fp32_and_fp64(model):
    """Per image: O.frame_locations -> normalisation -> O.gmw_pipeline -> O.ray_rescale, FP32 on CUDA (TF32 off) and FP64."""
    f = frames(40)
    r = refine(f, model)
    c = f["cpu"]
    sd = O.random_state_dict(7)
    for dt in (torch.float32, torch.float64):
        sd_d = {k: v.to(DEV, dt) for k, v in sd.items()}
        for b in range(f["B"]):
            sel = (c["bi"] == b).nonzero().reshape(-1)
            P = f["P_obj"][int(sel[0])]
            args = [c["off"][sel], c["pts"][sel], c["ofs"][sel], c["pad_b"][b:b + 1], c["k3"][sel], c["rot"][sel]]
            args = [a.to(dt) for a in args]
            dims = c["dims"][sel].to(dt)
            loc_o = frame_locations(args, P, dims)
            kimg = O.decode_kpts_2d_img(args[0], args[1], args[2], args[3].reshape(-1))[:, :NK]
            Pt = torch.as_tensor(P, dtype=dt)
            k2 = torch.stack(((kimg[..., 0] - Pt[0, 2]) / Pt[0, 0], (kimg[..., 1] - Pt[1, 2]) / Pt[1, 1]), dim=-1)
            with torch.no_grad():
                z_o = O.gmw_pipeline(k2.to(DEV), args[4][:, :NK].to(DEV), args[5].to(DEV), sd_d).cpu()
            loc_r = O.ray_rescale(loc_o, z_o, dims[:, [1, 2, 0]])
            sd_idx = sel.to(DEV)
            assert rel_err(r["gmw_depth"][sd_idx].cpu(), z_o) < 1e-5, (dt, b)
            got = r["location"][sd_idx].cpu().double()
            assert bool(((got - loc_r.double()).abs() <= 1e-4 + 1e-5 * loc_r.double().abs()).all()), (dt, b)


def test_refine_index_outside_the_map_is_nan_for_that_object_only(model):
    f = frames(40)
    r = refine(f, model, return_inputs=True)
    bad = dict(f)
    bad["pos"] = f["pos"].clone()
    bad["pos"][3] = H * W + 5
    rb = refine(bad, model, return_inputs=True)
    keep = torch.arange(f["N"], device=DEV) != 3
    for key in ("dgde_depth", "dgde_location", "gmw_depth", "location", "kpts_2d"):
        assert bool(torch.isnan(rb[key][3]).all()), key
        assert torch.equal(rb[key][keep], r[key][keep]), key
    assert torch.equal(rb["good_idx"][keep], r["good_idx"][keep])


def test_refine_empty_graph_capture_and_params_route(model):
    f = frames(40)
    empty = dict(f, pos=f["pos"][:0], rot=f["rot"][:0], dims=f["dims"][:0], bi=f["bi"][:0])
    e = refine(empty, model, return_inputs=True)
    shapes = {"dgde_depth": (0,), "dgde_location": (0, 3), "gmw_depth": (0,), "location": (0, 3), "kpts_2d": (0, NK, 2),
              "kpts_3d": (0, NK, 3), "good_idx": (0, 1500)}
    assert {k: tuple(v.shape) for k, v in e.items()} == shapes
    # CUDA-graph capture and replay == eager (calibration and pad already on the device: nothing crosses from the host)
    g_in = dict(f, P=torch.as_tensor(f["P"]).to(DEV), pad=f["pad"].to(DEV))
    eager = refine(g_in, model, chunk=16, return_inputs=True)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        refine(g_in, model, chunk=16)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = refine(g_in, model, chunk=16, return_inputs=True)
    graph.replay()
    torch.cuda.synchronize()
    for key in eager:
        assert torch.equal(captured[key], eager[key]), key
    # explicit parameter blobs (a patched reference module's route) == the module's own blobs
    blobs = (model.params4.detach().clone(), model.params6.detach().clone())
    via = refine(f, dcd_b200.GMW(depth=model.depth), chunk=16, params=blobs, return_inputs=True)
    for key in eager:
        assert torch.equal(via[key], eager[key]), key
