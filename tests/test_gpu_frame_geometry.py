"""The DGDE frame epilogue (csrc/dgde_locate.cu) at every launch layout it accepts: `dgde_locate_warp_kernel` (256 threads,
8 warps: compute_pairs_kpts_depth) and `dgde_frame_warp_kernel` (128 threads, 4 warps: frame_depths_from_map, and its GMW
instantiation in refine_detections).

Each keypoint count n is here for a reason:
    2, 3           fewer edges than lanes
    32, 33, 64, 65 the per-lane keypoint staging loop (t = lane, lane + 32, ...) wraps
    73             the product shape
    74, 100        refine_detections with n > 73 (its 73-keypoint GMW outputs have a row stride != n)
    128, 129       the locate kernel's 2n^2 + 126n bytes of shared memory pass 48 KB (opt-in) at n = 129
    142, 143       the frame kernel's 2n^2 + 62n bytes pass 48 KB at n = 143
    256            the largest pair table, the (i*16) | (j*16) << 16 packing at its widest
and each batch size N: 1, NWARP - 1, NWARP, NWARP + 1 (first CTA) at every n; cap - 1, cap, cap + 1, 2 cap + 3 (the grid-stride
loop once N exceeds the grid cap = SMs x 8 CTAs x NWARP) of both kernels at n = 3, 73, 256.

Checks: FP64 oracle on slices (first CTA, both sides of each grid-stride pass boundary, last object) with the bars of
tests/test_gpu_locate.py (depth rel <= 1e-5, location abs <= 1e-4 + rel 1e-5); saturated inputs whose mean is exact in FP32
(bit for bit: catches a missing, duplicated or mispaired edge and stale or foreign keypoints in shared memory); bit-identities
between the two kernels, across warp slots and passes, and of refine_detections with its hand composition.
"""
import numpy as np
import pytest
import torch

import dcd_b200
from dcd_b200 import synth
from oracle import dcd_oracle as O
from conftest import rel_err

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
NW_FRAME, NW_LOCATE = 4, 8
GEOMETRY_N = (2, 3, 32, 33, 64, 65, 73, 74, 100, 128, 129, 142, 143, 256)
LARGE_N_AT = (3, 73, 256)
SMALL = ("1", "NWF-1", "NWF", "NWF+1", "NWL-1", "NWL", "NWL+1")
LARGE = ("capF-1", "capF", "capF+1", "2capF+3", "capL-1", "capL", "capL+1", "2capL+3")
CASES = [(n, s) for n in GEOMETRY_N for s in SMALL + (LARGE if n in LARGE_N_AT else ())]
P_FRAME = np.array(synth.P2, dtype=np.float64)
PAD_B = torch.tensor([[19.0, 5.0], [3.0, 7.0]])
B = 2


def caps():
    sm = torch.cuda.get_device_properties(DEV).multi_processor_count
    return sm * 8 * NW_FRAME, sm * 8 * NW_LOCATE


def batch_size(label):
    """`label` of SMALL / LARGE: F = the frame kernel (NWF warps, grid cap capF), L = the locate kernel."""
    capF, capL = caps()
    sizes = {"1": 1}
    for k, nw, cap in (("F", NW_FRAME, capF), ("L", NW_LOCATE, capL)):
        sizes.update({"NW%s-1" % k: nw - 1, "NW%s" % k: nw, "NW%s+1" % k: nw + 1,
                      "cap%s-1" % k: cap - 1, "cap%s" % k: cap, "cap%s+1" % k: cap + 1, "2cap%s+3" % k: 2 * cap + 3})
    return sizes[label]


def boundary_objects(N):
    """First CTA of either kernel, both sides of every grid-stride pass boundary, the last object."""
    capF, capL = caps()
    picks = set(range(NW_LOCATE)) | {N - 1}
    for cap in (capF, capL):
        for p in (cap, 2 * cap):
            picks |= {p - 1, p}
    return sorted(i for i in picks if 0 <= i < N)


def channels(n):
    """A non-default channel table: keypoint groups first, the sub-pixel offset last (one spare channel after it)."""
    ch = {"extra_kpts_2d": 1, "extra_kpts_3d": 2 + 2 * n, "3d_offset": 3 + 5 * n}
    return ch, ch["3d_offset"] + 3


def layout(N, n, seed):
    """A random [B,C,H,W] map and distinct positions per image for N detections (alternating between the B images)."""
    ch, C = channels(n)
    W = 160
    H = max(4, -(-(-(-N // B)) // W))               # ceil(ceil(N / B) / W) rows
    g = torch.Generator(device=DEV).manual_seed(seed)
    fmap = torch.randn(B, C, H, W, device=DEV, generator=g) * 0.1
    bi = torch.arange(N, device=DEV) % B
    pos = torch.empty(N, dtype=torch.int64, device=DEV)
    for b in range(B):
        sel = (bi == b).nonzero().reshape(-1)
        pos[sel] = torch.randperm(H * W, device=DEV, generator=g)[:sel.numel()]
    pts = torch.stack(((pos % W).float(), (pos // W).float()), dim=1).cpu()
    return dict(fm=fmap, pos=pos, bi=bi, ch=ch), pts


def plant(f, off, k3, ofs):
    """Keypoint offsets [N,n,2], template points [N,n,3] and sub-pixel offsets [N,2] into the map at each detection's
    position: one vectorised index_put per channel group."""
    fm, N = f["fm"], off.shape[0]
    flat = fm.view(fm.shape[0], fm.shape[1], -1)
    for first, vals in ((f["ch"]["extra_kpts_2d"], off.reshape(N, -1)), (f["ch"]["extra_kpts_3d"], k3.reshape(N, -1)),
                        (f["ch"]["3d_offset"], ofs)):
        c = first + torch.arange(vals.shape[1], device=DEV)
        flat.index_put_((f["bi"][:, None], c[None, :], f["pos"][:, None]), vals.to(DEV))


_pool = {}


def objects(n, N):
    """Geometry-consistent objects (synth), one pool per n so that every batch size takes a prefix of the same objects."""
    key = (n, N > 64)
    if key not in _pool:
        _pool.clear()
        nmax = 2 * caps()[1] + 3 if N > 64 else 64
        ob = synth.make_objects(n=n, seed=500 + n, counts=torch.tensor([nmax]))
        _pool[key] = (ob.kps, ob.kps_3d, ob.rot_y)
    kps, k3, rot = (t[:N] for t in _pool[key])
    return kps, k3, rot


def geometric_frame(n, N, seed):
    kps, k3, rot = objects(n, N)
    g = torch.Generator().manual_seed(seed)
    ofs = torch.rand(N, 2, generator=g) - 0.5
    f, pts = layout(N, n, seed)
    pad = PAD_B[f["bi"].cpu()]
    off = (kps + pad.unsqueeze(1)) / 4 - (pts + ofs).unsqueeze(1)     # image keypoints (off + pts + ofs) * 4 - pad = synth's
    plant(f, off, k3, ofs)
    dims = torch.stack((torch.full((N,), 3.9), -k3[:, -1, 1], torch.full((N,), 1.6)), dim=1)
    f.update(rot=rot.to(DEV), dims=dims.to(DEV), P=P_FRAME, cpu=dict(off=off, pts=pts, ofs=ofs, pad=pad, k3=k3, rot=rot, dims=dims))
    return f


def frame(f, n, sel=None, **kw):
    s = slice(None) if sel is None else sel
    with torch.no_grad():
        return dcd_b200.frame_depths_from_map(f["fm"], f["pos"][s], f["rot"][s], f["P"], PAD_B.to(DEV), dims=f["dims"][s],
                                              batch_idxs=f["bi"][s], n=n, channels=f["ch"], **kw)


def locate(f, off, ofs, k3, sel=None):
    s = slice(None) if sel is None else sel
    pts = torch.stack(((f["pos"] % f["fm"].shape[3]).float(), (f["pos"] // f["fm"].shape[3]).float()), dim=1)
    with torch.no_grad():
        return dcd_b200.compute_pairs_kpts_depth(off[s], pts[s], ofs[s], PAD_B.to(DEV), k3[s], f["rot"][s], f["P"],
                                                 batch_idxs=f["bi"][s], dims=f["dims"][s], return_locations=True)


def oracle_f64(c, idx, P):
    """O.frame_locations' operations in float64 with a per-object pad (objects of both images at once)."""
    off, pts, ofs, pad, k3, rot, dims = (c[k][idx].double() for k in ("off", "pts", "ofs", "pad", "k3", "rot", "dims"))
    K = torch.from_numpy(P).unsqueeze(0).expand(len(idx), -1, -1)
    real = O.decode_kpts_2d_img(off, pts, ofs, pad)
    depth = O.decode_pairs_kpts_depth(real, k3, rot, K)[0].mean(1)
    uv = (pts + ofs) * O.DOWN_RATIO - pad
    loc = O.project_image_to_rect(torch.cat((uv, depth[:, None]), dim=1), P)
    loc[:, 1] += dims[:, 1] / 2
    return depth, loc


def gather_route(f, n):
    """select_point_of_interest per image, then the channel slices: the [N,C] values the frame kernel reads itself."""
    C = f["fm"].shape[1]
    pois = torch.empty((f["pos"].shape[0], C), device=DEV)
    for b in range(B):
        sel = (f["bi"] == b).nonzero().reshape(-1)
        pois[sel] = dcd_b200.select_point_of_interest(1, f["pos"][sel].reshape(1, -1), f["fm"][b:b + 1]).reshape(-1, C)
    ch = f["ch"]
    return (pois[:, ch["extra_kpts_2d"]:ch["extra_kpts_2d"] + 2 * n].reshape(-1, n, 2),
            pois[:, ch["3d_offset"]:ch["3d_offset"] + 2],
            pois[:, ch["extra_kpts_3d"]:ch["extra_kpts_3d"] + 3 * n].reshape(-1, n, 3))


@pytest.mark.parametrize("n,size", CASES)
def test_frame_kernels_vs_fp64_and_bit_identities(n, size):
    N = batch_size(size)
    f = geometric_frame(n, N, seed=n * 7 + N)
    c = f["cpu"]
    depth, loc, kimg, k3o = frame(f, n, return_keypoints=True)
    # staged keypoints: the image keypoints are the oracle's FP32 expression bit for bit, the template points the planted ones
    assert torch.equal(kimg.cpu(), O.decode_kpts_2d_img(c["off"], c["pts"], c["ofs"], c["pad"]))
    assert torch.equal(k3o.cpu(), c["k3"])
    # FP64 on the slices where a layout changes
    idx = boundary_objects(N)
    d64, l64 = oracle_f64(c, idx, f["P"])
    assert rel_err(depth.cpu()[idx], d64) < 1e-5
    got = loc.cpu()[idx].double()
    assert bool(((got - l64).abs() <= 1e-4 + 1e-5 * l64.abs()).all())
    assert torch.equal(loc[:, 2], depth) and bool(torch.isfinite(loc).all())
    # frame kernel == select_point_of_interest + the locate kernel (same arithmetic on the same values)
    o2, of, o3 = gather_route(f, n)
    d2, l2 = locate(f, o2, of, o3)
    assert torch.equal(d2, depth) and torch.equal(l2, loc)
    # an object's outputs depend neither on its warp slot nor on its grid-stride pass: the batch shifted by one, and a slice
    # around the last pass boundary on its own
    shifted = dict(f, pos=torch.cat((f["pos"][-1:], f["pos"])), rot=torch.cat((f["rot"][-1:], f["rot"])),
                   dims=torch.cat((f["dims"][-1:], f["dims"])), bi=torch.cat((f["bi"][-1:], f["bi"])))
    ds, ls = frame(shifted, n)
    assert torch.equal(ds[1:], depth) and torch.equal(ls[1:], loc)
    d2s, l2s = locate(shifted, torch.cat((o2[-1:], o2)), torch.cat((of[-1:], of)), torch.cat((o3[-1:], o3)))
    assert torch.equal(d2s[1:], depth) and torch.equal(l2s[1:], loc)
    part = slice(max(0, idx[-2] - 5) if len(idx) > 1 else 0, N)
    dp, lp = frame(f, n, sel=part)
    assert torch.equal(dp, depth[part]) and torch.equal(lp, loc[part])
    dq, lq = locate(f, o2, of, o3, sel=part)
    assert torch.equal(dq, depth[part]) and torch.equal(lq, loc[part])


def saturated_objects(n, N, seed):
    """Keypoints whose every edge clamps exactly: yaw 0 and Z = 0 make C = X sin - Z cos = 0, so H = Y_i - Y_j with Y in
    {0, 1}; the vertical offset puts each keypoint in one of two rows 800 px apart.  An edge within a row has V = 0 and depth
    80 when its Y differ (|H| / 1e-10), 2 when they agree (0 / 1e-10); an edge across rows has |V| ~ 1.1 >= |H|, depth 2.
    With b3 = 0 every partial sum is an integer below 2^24, so the FP32 mean is the correctly rounded (80 a + 2 (E - a)) / E.
    The row and Y probabilities change from object to object, so neighbours have different patterns."""
    g = torch.Generator().manual_seed(seed)
    p = 0.05 + 0.9 * torch.rand(N, 2, 1, generator=g)
    row = (torch.rand(N, n, generator=g) < p[:, 0]).float()
    ybit = (torch.rand(N, n, generator=g) < p[:, 1]).float()
    off = torch.stack((torch.randn(N, n, generator=g), 200 * row - 100), dim=-1)
    k3 = torch.stack((torch.randn(N, n, generator=g), ybit, torch.zeros(N, n)), dim=-1)
    cnt = [((row == r) & (ybit == y)).sum(1) for r in (0, 1) for y in (0, 1)]
    a = cnt[0] * cnt[1] + cnt[2] * cnt[3]
    E = n * (n - 1) // 2
    total = (80 * a + 2 * (E - a)).to(torch.float32)
    assert int(total.max()) < 1 << 24
    return off, k3, total / torch.tensor(float(E))


@pytest.mark.parametrize("n,size", CASES)
def test_frame_kernels_saturated_mean_is_exact(n, size):
    N = batch_size(size)
    off, k3, want = saturated_objects(n, N, seed=n * 11 + N)
    g = torch.Generator().manual_seed(N)
    ofs = torch.rand(N, 2, generator=g) - 0.5
    f, _ = layout(N, n, seed=n + N)
    plant(f, off, k3, ofs)
    P = P_FRAME.copy()
    P[2, 3] = 0.0                                    # b3 = 0: the depths stay integers
    f.update(rot=torch.zeros(N, 1, device=DEV), dims=torch.ones(N, 3, device=DEV), P=P)
    depth, loc = frame(f, n)
    assert torch.equal(depth.cpu(), want)
    assert torch.equal(loc[:, 2], depth)
    d2, l2 = locate(f, off.to(DEV), ofs.to(DEV), k3.to(DEV))
    assert torch.equal(d2.cpu(), want)
    assert torch.equal(l2, loc)


@pytest.fixture(scope="module")
def model():
    return dcd_b200.GMW().to(DEV).load_reference_state_dict(O.random_state_dict(7))


def refine(f, model, n, chunk, **kw):
    with torch.no_grad():
        return dcd_b200.refine_detections(f["fm"], f["pos"], f["rot"], f["P"], PAD_B.to(DEV), f["dims"], model,
                                          batch_idxs=f["bi"], n=n, channels=f["ch"], chunk=chunk, **kw)


def hand_composition(f, model, n, chunk):
    """frame_depths_from_map -> FP32 normalisation of keypoints 0 .. 72 -> gmw_weighted_depth -> ray_rescale
    (as tests/test_gpu_refine.py)."""
    NK = dcd_b200.ops.GMW_KPTS
    d, loc, kimg, k3 = frame(f, n, return_keypoints=True)
    with torch.no_grad():
        Kd = torch.as_tensor(f["P"], dtype=torch.float32).to(DEV)
        kimg, k3 = kimg[:, :NK], k3[:, :NK].contiguous()
        k2 = torch.stack(((kimg[..., 0] - Kd[0, 2]) / Kd[0, 0], (kimg[..., 1] - Kd[1, 2]) / Kd[1, 1]), dim=-1)
        z, gidx = dcd_b200.gmw_weighted_depth(k2, k3, f["rot"], model, chunk=chunk, return_idx=True)
        out = dcd_b200.ray_rescale(loc, z, f["dims"][:, [1, 2, 0]])
    return {"dgde_depth": d, "dgde_location": loc, "gmw_depth": z, "location": out, "kpts_2d": k2, "kpts_3d": k3,
            "good_idx": gidx}


@pytest.mark.parametrize("n,size", [(74, "NWL+1"), (100, "NWL+1"), (256, "NWL+1"), (256, "capF+1")])
def test_refine_above_73_keypoints_equals_hand_composition(model, n, size):
    """The GMW instantiation of the frame kernel at n > 73: GMW's inputs are keypoints 0 .. 72 with a row stride of 73."""
    N = batch_size(size)
    f = geometric_frame(n, N, seed=3 * n + N)
    chunk = max(1, N // 2)
    r = refine(f, model, n, chunk, return_inputs=True)
    h = hand_composition(f, model, n, chunk)
    for key in h:
        assert r[key].shape == h[key].shape and torch.equal(r[key], h[key]), key
    assert bool(torch.isfinite(r["location"]).all())


def test_position_outside_the_map_at_256_keypoints(model):
    """One detection outside the map: NaN for that object only, in both instantiations of the frame kernel."""
    n, N = 256, 2 * NW_LOCATE + 1
    f = geometric_frame(n, N, seed=99)
    H, W = f["fm"].shape[2:]
    bad = dict(f, pos=f["pos"].clone())
    bad["pos"][5] = H * W + 5
    keep = torch.arange(N, device=DEV) != 5
    good = frame(f, n, return_keypoints=True)
    worse = frame(bad, n, return_keypoints=True)
    for a, b in zip(good, worse):
        assert bool(torch.isnan(b[5]).all()) and torch.equal(b[keep], a[keep])
    r = refine(f, model, n, N, return_inputs=True)
    rb = refine(bad, model, n, N, return_inputs=True)
    for key in ("dgde_depth", "dgde_location", "gmw_depth", "location", "kpts_2d"):
        assert bool(torch.isnan(rb[key][5]).all()), key
        assert torch.equal(rb[key][keep], r[key][keep]), key
    assert torch.equal(rb["good_idx"][keep], r["good_idx"][keep])
