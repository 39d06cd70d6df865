"""Gradients of the DGDE detector-head functions around the edge solve (select_point_of_interest, decode_location_flatten,
decode_depth_from_keypoints_batch, depth_ensemble) against the autograd of the oracle restatement (oracle/dcd_oracle.py, whose
forward tests/golden pins to the unmodified reference).

Numeric bar, per gradient tensor: with every relu and clamp input at least 1e-3 (relative) away from its threshold,
    max|ours - f64| <= max(2 max|FP32 oracle - f64|, 1e-6 max|f64|)
where "f64" is the oracle's autograd in float64 on the same FP32 inputs and "FP32 oracle" its autograd on CUDA in FP32; the
pattern of exact zeros equals the FP32 oracle's.  The end-to-end chain (map -> gather -> edge solve -> locations, and the
depth ensemble on other channels) holds the map gradient to 1e-4 max|f64| as well.  The measured errors are printed.
"""
import numpy as np
import pytest
import torch

import dcd_b200
from dcd_b200 import synth
from oracle import dcd_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
COUNTS = torch.tensor([3, 50, 1, 17], dtype=torch.int64)      # ragged objects per image
PAD_B = torch.tensor([[19.0, 5.0], [0.0, 0.0], [7.0, 3.0], [12.0, 8.0]])


def check_grad(name, ours, o32, o64, extra_bar=None):
    """The bar of the module docstring; returns (our error, FP32 oracle error)."""
    ours, o32, o64 = ours.detach().double().cpu(), o32.detach().double().cpu(), o64.detach().double().cpu()
    scale = float(o64.abs().max()) if o64.numel() else 0.0
    e_ours = float((ours - o64).abs().max()) if o64.numel() else 0.0
    e_32 = float((o32 - o64).abs().max()) if o64.numel() else 0.0
    print("%-28s max|f64| %.3e  ours %.3e  FP32 oracle %.3e" % (name, scale, e_ours, e_32))
    assert e_ours <= max(2 * e_32, 1e-6 * scale), name
    if extra_bar is not None:
        assert e_ours <= extra_bar * scale, name
    assert torch.equal(ours == 0, o32 == 0), name + ": zero pattern"
    return e_ours, e_32


# ---------------------------------------------------------------------------------------------------------------------
# data: synth frames, several images with their own P and pad
# ---------------------------------------------------------------------------------------------------------------------
def frames(seed=77):
    ob = synth.make_objects(n=73, seed=seed, counts=COUNTS, jitter_fx=0.02)
    g = torch.Generator().manual_seed(seed + 1)
    N = ob.N
    pad = PAD_B[ob.frame_id]
    centre = (ob.kps.mean(1) + pad) / 4
    pts = centre.floor()
    ofs = centre - pts + 0.05 * (torch.rand(centre.shape, generator=g) - 0.5)
    kp10 = (ob.kps[:, -10:] + pad.unsqueeze(1)) / 4 - (pts + ofs).unsqueeze(1)      # box keypoints, feature-map units
    dims = torch.stack((torch.full((N,), 3.9), -ob.kps_3d[:, -1, 1], torch.full((N,), 1.6)), dim=1)
    direct = ob.gt_depth * (1 + 0.05 * torch.randn(N, generator=g))
    lud = torch.rand(N, generator=g) * 2 - 1.5
    luk = torch.rand(N, 3, generator=g) * 2 - 1.5
    scores = torch.rand(N, generator=g) * 0.9 + 0.05
    # keep the clamp of depth_error (0.01, 1) out of reach of 1e-3: shift the log uncertainties of an object near it
    for _ in range(4):
        u = torch.cat((lud.double().exp().unsqueeze(1), luk.double().exp()), 1)
        near = torch.zeros(N, dtype=torch.bool)
        for err in (4 / (1 / u).sum(1), 3 / (1 / u[:, 1:]).sum(1)):     # with and without the direct depth
            near |= ((err - 1).abs() < 2e-3) | ((err - 0.01).abs() < 2e-5)
        lud[near] += 0.01
        luk[near] += 0.01
    P = [ob.K[(ob.frame_id == f).nonzero()[0, 0]].double().numpy() for f in range(len(COUNTS))]
    return dict(ob=ob, pts=pts, ofs=ofs, kp10=kp10.contiguous(), dims=dims, direct=direct, lud=lud, luk=luk, scores=scores, P=P,
                bi=ob.frame_id, K=ob.K)


def oracle_ensemble(d, inputs, dtype, dev, grads, with_direct=True, with_scores=True):
    """Oracle chain of depth_ensemble; inputs: dict of leaf tensors (already of `dtype` on `dev`) -> outputs."""
    f_us = [float(p[0, 0]) for p in d["P"]]
    bi = d["bi"].to(dev)
    kd = O.decode_depth_from_keypoints_batch(inputs["kp10"], inputs["dims"], f_us, bi)
    depth, err, amax = O.depth_ensemble(inputs["direct"] if with_direct else None, kd, inputs["lud"] if with_direct else None,
                                        inputs["luk"])
    so = O.uncertainty_scores(inputs["scores"].view(-1, 1), err) if with_scores else None
    return kd, depth, err, amax, so


def oracle_locations(points, offsets, depths, Ps, pad_b, bi):
    """O.decode_location_flatten; in float64 its per-image steps (O.project_image_to_rect) gathered in the input's dtype (the
    oracle's own result tensor is float32, like the reference's)."""
    if points.dtype == torch.float32:
        return O.decode_location_flatten(points, offsets, depths, Ps, pad_b, bi)
    pts = (points + offsets) * O.DOWN_RATIO - pad_b[bi]
    parts = []
    for b in torch.unique(bi, sorted=True).tolist():           # objects are sorted by image
        sel = torch.nonzero(bi == b).squeeze(-1)
        parts.append(O.project_image_to_rect(torch.cat((pts[sel], depths[sel, None]), dim=1), Ps[b]))
    return torch.cat(parts)


def upstream(N, seed=3):
    g = torch.Generator().manual_seed(seed)
    return dict(kd=torch.randn(N, 3, generator=g), depth=torch.randn(N, generator=g), err=torch.randn(N, generator=g),
                so=torch.randn(N, 1, generator=g))


def ensemble_loss(out, up, dev, dtype):
    kd, depth, err, so = out
    L = (kd * up["kd"].to(dev, dtype)).sum() + (depth * up["depth"].to(dev, dtype)).sum()
    L = L + (err * up["err"].to(dev, dtype)).sum()
    if so is not None:
        L = L + (so * up["so"].to(dev, dtype)).sum()
    return L


ENS_INPUTS = ("kp10", "dims", "direct", "lud", "luk", "scores")


def oracle_ensemble_grads(d, dtype, dev, up, with_direct=True, with_scores=True):
    leaves = {k: d[k].to(dev, dtype).requires_grad_() for k in ENS_INPUTS}
    kd, depth, err, _, so = oracle_ensemble(d, leaves, dtype, dev, None, with_direct, with_scores)
    L = ensemble_loss((kd, depth, err, so), up, dev, dtype)
    names = [k for k in ENS_INPUTS if (with_direct or k not in ("direct", "lud")) and (with_scores or k != "scores")]
    gs = torch.autograd.grad(L, [leaves[k] for k in names])
    return dict(zip(names, gs))


def ours_ensemble(d, up, with_direct=True, with_scores=True, dtype=torch.float32):
    leaves = {k: d[k].to(DEV, dtype).requires_grad_() for k in ENS_INPUTS}
    K = d["K"].to(DEV)
    out = dcd_b200.depth_ensemble(leaves["kp10"], leaves["dims"], K, leaves["luk"],
                                  direct_depths=leaves["direct"] if with_direct else None,
                                  direct_log_uncertainty=leaves["lud"] if with_direct else None,
                                  scores=leaves["scores"] if with_scores else None)
    L = ensemble_loss((out["keypoint_depths"], out["depth"], out["depth_error"], out["scores"]), up, DEV, torch.float32)
    names = [k for k in ENS_INPUTS if (with_direct or k not in ("direct", "lud")) and (with_scores or k != "scores")]
    gs = torch.autograd.grad(L, [leaves[k] for k in names])
    return dict(zip(names, gs)), out


# ---------------------------------------------------------------------------------------------------------------------
# depth ensemble + keypoint depths
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("with_direct,with_scores", [(True, True), (False, True), (True, False)])
def test_depth_ensemble_grad_vs_oracle(with_direct, with_scores):
    d = frames()
    # the margins the bar assumes: heights, keypoint depths and depth_error away from their thresholds
    v = d["kp10"][:, :, 1].double()
    hts = torch.stack((v[:, 8] - v[:, 9], v[:, 0] - v[:, 4], v[:, 2] - v[:, 6], v[:, 1] - v[:, 5], v[:, 3] - v[:, 7]), 1)
    assert float(hts.min()) > 1e-3
    kd64 = O.decode_depth_from_keypoints_batch(d["kp10"].double(), d["dims"].double(), [float(p[0, 0]) for p in d["P"]], d["bi"])
    assert float(kd64.min()) > 0.1 * 1.001 and float(kd64.max()) < 100 * 0.999
    up = upstream(d["ob"].N)
    g64 = oracle_ensemble_grads(d, torch.float64, "cpu", up, with_direct, with_scores)
    g32 = oracle_ensemble_grads(d, torch.float32, DEV, up, with_direct, with_scores)
    ours, _ = ours_ensemble(d, up, with_direct, with_scores)
    for k in g64:
        check_grad("ensemble %s" % k, ours[k], g32[k], g64[k])
    assert bool((ours["kp10"][:, :, 0] == 0).all()) and bool((ours["dims"][:, [0, 2]] == 0).all())


def test_depth_ensemble_boundaries_follow_the_oracle_zero_pattern():
    """Zero heights (relu at 0), negative heights, keypoint depths clamped at 0.1 and at 100: exactly the oracle's zeros."""
    d = frames(seed=91)
    kp = d["kp10"]
    N = kp.shape[0]
    kp[0, 9, 1] = kp[0, 8, 1]                        # centre height exactly 0 -> f_u h / eps, clamped at 100
    kp[1, 4, 1] = kp[1, 0, 1]                        # one corner_02 height exactly 0
    kp[2, 5, 1] = kp[2, 1, 1] + 3.0                  # negative corner_13 height
    kp[3, 9, 1] = kp[3, 8, 1] + 1.0                  # negative centre height
    kp[4, :, 1] *= 1e4                               # huge heights: depths below 0.1
    kp[5, 8, 1] = kp[5, 9, 1] + 1e-6                 # tiny positive height: above 100
    d["dims"][6, 1] = -d["dims"][6, 1]               # negative 3D height: negative depths clamped at 0.1
    kp[7, 9, 1] = kp[7, 8, 1]                        # zero centre height with a tiny 3D height: f_u h / eps inside the clamp,
    d["dims"][7, 1] = 1e-4                           # so only the relu decides the keypoints' gradient
    d["dims"][8, 1], kp[8, 8, 1] = exact_depth_pair(float(d["K"][8, 0, 0]), 100.0)     # centre depth exactly 100: the
    kp[8, 9, 1] = 0.0                                                                    # clamp is inclusive
    up = upstream(N, seed=4)
    g64 = oracle_ensemble_grads(d, torch.float64, "cpu", up)
    g32 = oracle_ensemble_grads(d, torch.float32, DEV, up)
    ours, out = ours_ensemble(d, up)
    kd = out["keypoint_depths"]
    assert bool((kd == 100).any()) and bool((kd == 0.1).any())
    for k in g64:
        assert torch.equal(ours[k].cpu() == 0, g32[k].cpu() == 0), k
    # rows 0..6 have a boundary in their keypoint depths; their zeros are there, and nowhere else
    assert bool((ours["kp10"][0, 8:10, 1] == 0).all()) and bool((ours["kp10"][1, [0, 4], 1] == 0).all())
    assert bool((ours["kp10"][2, [1, 5], 1] == 0).all()) and bool((ours["kp10"][3, 8:10, 1] == 0).all())
    assert bool((ours["kp10"][7, 8:10, 1] == 0).all()) and float(ours["dims"][7, 1]) != 0
    assert float(kd[8, 0]) == 100.0 and bool((ours["kp10"][8, 8:10, 1] != 0).all())
    assert bool((ours["kp10"][9:, :, 1] != 0).all())


def exact_depth_pair(f_u, depth):
    """(3D height h, 2D height ht) with f_u * h / (relu(ht) * 4 + eps) == depth exactly in FP32 (the kernel's and torch's
    rounding), searched over neighbouring floats of both."""
    f32 = torch.float32
    h0 = torch.tensor(1.5, dtype=f32)
    ht0 = ((torch.tensor(f_u, dtype=f32) * h0) / torch.tensor(depth, dtype=f32) - torch.tensor(1e-3, dtype=f32)) / 4
    h = h0 + torch.arange(-64, 64, dtype=f32) * 2 ** -22
    ht = ht0 + torch.arange(-64, 64, dtype=f32) * 2 ** -21
    q = (torch.tensor(f_u, dtype=f32) * h)[:, None] / (ht[None, :].clamp_min(0) * 4 + torch.tensor(1e-3, dtype=f32))
    hit = (q == depth).nonzero()
    assert hit.shape[0] > 0, "no exact pair found"
    return float(h[hit[0, 0]]), float(ht[hit[0, 1]])


def test_depth_ensemble_non_finite_inputs_follow_the_oracle():
    """exp overflow, NaN log uncertainties and NaN / inf scores: the NaN / inf / zero pattern of the oracle's autograd on CUDA
    (incl. `out[isnan(out)] = 0` of uncertainty_scores), and no other object's gradient changes."""
    d = frames(seed=93)
    clean = {k: v.clone() if torch.is_tensor(v) else v for k, v in d.items()}
    d["luk"][0, 1] = 200.0                          # exp -> inf
    d["lud"][1] = float("nan")
    d["scores"][2] = float("nan")
    d["scores"][3] = float("inf")
    d["luk"][4, :] = -200.0                         # exp -> 0: 1/u = inf
    d["direct"][5] = float("inf")
    up = upstream(d["ob"].N, seed=5)
    g32 = oracle_ensemble_grads(d, torch.float32, DEV, up)
    ours, _ = ours_ensemble(d, up)
    ref, _ = ours_ensemble(clean, up)
    for k in g32:
        a, b = ours[k].cpu(), g32[k].cpu()
        assert torch.equal(torch.isnan(a), torch.isnan(b)), k
        assert torch.equal(torch.isinf(a), torch.isinf(b)), k
        assert torch.equal(a == 0, b == 0), k
        assert torch.equal(ours[k][6:], ref[k][6:]), k            # other objects untouched


def test_keypoint_depth_gradients_are_one_kernel_for_both_functions():
    d = frames()
    K = d["K"].to(DEV)
    g = torch.randn(d["ob"].N, 3, device=DEV)
    kp1, dm1 = d["kp10"].to(DEV).requires_grad_(), d["dims"].to(DEV).requires_grad_()
    kd = dcd_b200.decode_depth_from_keypoints_batch(kp1, dm1, K)
    a = torch.autograd.grad(kd, [kp1, dm1], g)
    kp2, dm2 = d["kp10"].to(DEV).requires_grad_(), d["dims"].to(DEV).requires_grad_()
    out = dcd_b200.depth_ensemble(kp2, dm2, K, d["luk"].to(DEV), direct_depths=d["direct"].to(DEV),
                                  direct_log_uncertainty=d["lud"].to(DEV), scores=d["scores"].to(DEV))
    b = torch.autograd.grad(out["keypoint_depths"], [kp2, dm2], g)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    # per image P with batch_idxs, as the reference passes it
    Pb = torch.stack([torch.from_numpy(p) for p in d["P"]]).to(DEV)
    kp3 = d["kp10"].to(DEV).requires_grad_()
    kd3 = dcd_b200.decode_depth_from_keypoints_batch(kp3, d["dims"].to(DEV), Pb, batch_idxs=d["bi"].to(DEV))
    assert torch.equal(torch.autograd.grad(kd3, kp3, g)[0], a[0])


# ---------------------------------------------------------------------------------------------------------------------
# decode_location_flatten
# ---------------------------------------------------------------------------------------------------------------------
def test_decode_location_flatten_grad_vs_oracle():
    d = frames()
    N = d["ob"].N
    depth = d["ob"].gt_depth.clone()
    gl = torch.randn(N, 3, generator=torch.Generator().manual_seed(8))

    def oracle(dtype, dev):
        pts, ofs, dep = (t.to(dev, dtype).requires_grad_() for t in (d["pts"], d["ofs"], depth))
        loc = oracle_locations(pts, ofs, dep, d["P"], PAD_B.to(dev, dtype), d["bi"].to(dev))
        return torch.autograd.grad((loc * gl.to(dev, loc.dtype)).sum(), [pts, ofs, dep])

    g64, g32 = oracle(torch.float64, "cpu"), oracle(torch.float32, DEV)
    pts, ofs, dep = (t.to(DEV).requires_grad_() for t in (d["pts"], d["ofs"], depth))
    loc = dcd_b200.decode_location_flatten(pts, ofs, dep, d["K"].to(DEV), PAD_B.to(DEV), d["bi"].to(DEV))
    ours = torch.autograd.grad((loc * gl.to(DEV)).sum(), [pts, ofs, dep])
    for name, a, b, c in zip(("points", "offsets", "depths"), ours, g32, g64):
        check_grad("locate %s" % name, a, b, c)
    # integer target centres (the reference's training call): no gradient to them, the others unchanged
    pti = d["pts"].to(DEV).long()
    ofs2, dep2 = d["ofs"].to(DEV).requires_grad_(), depth.to(DEV).requires_grad_()
    loc2 = dcd_b200.decode_location_flatten(pti, ofs2, dep2, d["K"].to(DEV), PAD_B.to(DEV), d["bi"].to(DEV))
    o2 = torch.autograd.grad((loc2 * gl.to(DEV)).sum(), [ofs2, dep2])
    assert torch.equal(o2[0], ours[1]) and torch.equal(o2[1], ours[2])


# ---------------------------------------------------------------------------------------------------------------------
# select_point_of_interest
# ---------------------------------------------------------------------------------------------------------------------
def sequential_scatter(idx, g, B, C, HW):
    """CPU reference: FP32 sum in ascending slot order, out-of-range slots dropped."""
    out = torch.zeros(B, HW, C)
    for b in range(B):
        for k in range(idx.shape[1]):
            p = int(idx[b, k])
            if 0 <= p < HW:
                out[b, p] = out[b, p] + g[b, k]
    return out.permute(0, 2, 1).reshape(B, C, HW)


def test_poi_gather_grad_unique_positions_equal_the_oracle():
    B, C, H, W, K = 3, 440, 96, 320, 50
    gen = torch.Generator().manual_seed(1)
    fm = torch.randn(B, C, H, W, generator=gen).to(DEV).requires_grad_()
    idx = torch.stack([torch.randperm(H * W, generator=gen)[:K] for _ in range(B)]).to(DEV)
    g = torch.randn(B, K, C, device=DEV)
    ours = torch.autograd.grad(dcd_b200.select_point_of_interest(B, idx, fm), fm, g)[0]
    ref = torch.autograd.grad(O.select_point_of_interest(B, idx, fm), fm, g)[0]
    assert torch.equal(ours, ref)
    # [B,K,2] (x, y) point form
    pts = torch.stack((idx % W, idx // W), dim=-1)
    assert torch.equal(torch.autograd.grad(dcd_b200.select_point_of_interest(B, pts, fm), fm, g)[0], ref)


def test_poi_gather_grad_duplicates_are_summed_in_slot_order():
    B, C, H, W, K = 4, 64, 24, 40, 48
    gen = torch.Generator().manual_seed(2)
    fm = torch.randn(B, C, H, W, generator=gen).to(DEV).requires_grad_()
    idx = torch.randint(0, 12, (B, K), generator=gen)                 # many repeats
    idx[0, 10:] = 7                                                   # padded slots of a training batch: one position
    idx[1, :] = 3                                                     # every slot on one position
    g = torch.randn(B, K, C, generator=gen) * torch.logspace(-3, 3, K).view(1, K, 1)    # order matters at these scales
    out = dcd_b200.select_point_of_interest(B, idx.to(DEV), fm)
    ours = torch.autograd.grad(out, fm, g.to(DEV))[0]
    ref = sequential_scatter(idx, g, B, C, H * W).reshape(B, C, H, W)
    assert torch.equal(ours.cpu(), ref)
    again = torch.autograd.grad(dcd_b200.select_point_of_interest(B, idx.to(DEV), fm), fm, g.to(DEV))[0]
    assert torch.equal(again, ours)                                   # bit-identical rerun
    # a reversed or partial sum would differ: the reference is not order-insensitive at these scales
    rev = sequential_scatter(idx.flip(1), g.flip(1), B, C, H * W).reshape(B, C, H, W)
    assert not torch.equal(rev, ref)


def test_poi_gather_grad_out_of_range_and_empty():
    B, C, H, W, K = 2, 32, 16, 20, 12
    gen = torch.Generator().manual_seed(4)
    fm = torch.randn(B, C, H, W, generator=gen).to(DEV).requires_grad_()
    idx = torch.randint(0, H * W, (B, K), generator=gen)
    idx[0, 3] = H * W
    idx[1, 0] = -1
    idx[1, 5] = 1 << 40
    g = torch.randn(B, K, C, generator=gen)
    out = dcd_b200.select_point_of_interest(B, idx.to(DEV), fm)
    assert bool(torch.isnan(out[0, 3]).all()) and bool(torch.isnan(out[1, 0]).all())
    ours = torch.autograd.grad(out, fm, g.to(DEV))[0]
    torch.cuda.synchronize()                                          # a fault would surface here
    assert torch.equal(ours.cpu(), sequential_scatter(idx, g, B, C, H * W).reshape(B, C, H, W))
    # K = 0: an all-zero map gradient
    e = dcd_b200.select_point_of_interest(B, idx[:, :0].to(DEV), fm)
    assert e.shape == (B, 0, C)
    z = torch.autograd.grad(e, fm, torch.zeros_like(e))[0]
    assert z.shape == fm.shape and not bool(z.any())
    with pytest.raises(RuntimeError):                                 # the bound of the duplicate scan
        big = dcd_b200.select_point_of_interest(1, torch.zeros((1, 1025), dtype=torch.int64, device=DEV), fm[:1])
        big.sum().backward()


def test_no_objects():
    """N = 0 through the location decode, the keypoint depths and the ensemble: empty gradients, no launch."""
    z2, z1 = torch.zeros((0, 2), device=DEV, requires_grad=True), torch.zeros((0,), device=DEV, requires_grad=True)
    K = torch.zeros((0, 3, 4), device=DEV)
    loc = dcd_b200.decode_location_flatten(z2, z2, z1, K, torch.zeros(2, device=DEV))
    g = torch.autograd.grad(loc.sum(), [z2, z1])
    assert g[0].shape == (0, 2) and g[1].shape == (0,)
    kp, dm, lu = (torch.zeros(s, device=DEV, requires_grad=True) for s in ((0, 10, 2), (0, 3), (0, 3)))
    out = dcd_b200.depth_ensemble(kp, dm, K, lu, direct_depths=z1, direct_log_uncertainty=z1, scores=z1)
    L = out["keypoint_depths"].sum() + out["depth"].sum() + out["depth_error"].sum() + out["scores"].sum()
    assert [t.shape for t in torch.autograd.grad(L, [kp, dm, lu, z1])] == [(0, 10, 2), (0, 3), (0, 3), (0,)]


# ---------------------------------------------------------------------------------------------------------------------
# bit-level properties
# ---------------------------------------------------------------------------------------------------------------------
def test_forward_bits_with_and_without_autograd_and_frozen_inputs():
    d = frames()
    K, bi = d["K"].to(DEV), d["bi"].to(DEV)
    up = upstream(d["ob"].N)
    with torch.no_grad():
        ref = dcd_b200.depth_ensemble(*(d[k].to(DEV) for k in ("kp10", "dims")), K, d["luk"].to(DEV),
                                      direct_depths=d["direct"].to(DEV), direct_log_uncertainty=d["lud"].to(DEV),
                                      scores=d["scores"].to(DEV))
        loc_ref = dcd_b200.decode_location_flatten(d["pts"].to(DEV), d["ofs"].to(DEV), d["direct"].to(DEV), K, PAD_B.to(DEV), bi)
    full, out = ours_ensemble(d, up)
    for k in ("keypoint_depths", "depth", "depth_error", "min_uncertainty", "scores"):
        assert torch.equal(out[k], ref[k]), k
    ofs = d["ofs"].to(DEV).requires_grad_()
    assert torch.equal(dcd_b200.decode_location_flatten(d["pts"].to(DEV), ofs, d["direct"].to(DEV), K, PAD_B.to(DEV), bi), loc_ref)
    # one frozen input at a time: it receives nothing, every other gradient keeps its bits
    for frozen in ENS_INPUTS:
        leaves = {k: d[k].to(DEV).requires_grad_(k != frozen) for k in ENS_INPUTS}
        o = dcd_b200.depth_ensemble(leaves["kp10"], leaves["dims"], K, leaves["luk"], direct_depths=leaves["direct"],
                                    direct_log_uncertainty=leaves["lud"], scores=leaves["scores"])
        L = ensemble_loss((o["keypoint_depths"], o["depth"], o["depth_error"], o["scores"]), up, DEV, torch.float32)
        L.backward()
        assert leaves[frozen].grad is None, frozen
        for k in ENS_INPUTS:
            if k != frozen:
                assert torch.equal(leaves[k].grad, full[k]), (frozen, k)
    # an output the loss does not use passes no gradient: a depth-only loss equals the oracle's depth-only gradient pattern
    leaves = {k: d[k].to(DEV).requires_grad_() for k in ENS_INPUTS}
    o = dcd_b200.depth_ensemble(leaves["kp10"], leaves["dims"], K, leaves["luk"], direct_depths=leaves["direct"],
                                direct_log_uncertainty=leaves["lud"], scores=leaves["scores"])
    o["depth"].sum().backward()
    assert not bool(leaves["scores"].grad.any())
    # constants that require grad fail loudly
    Kg = K.clone().requires_grad_()
    with pytest.raises(RuntimeError):
        dcd_b200.depth_ensemble(leaves["kp10"], leaves["dims"], Kg, leaves["luk"])
    with pytest.raises(RuntimeError):
        dcd_b200.decode_depth_from_keypoints_batch(leaves["kp10"], leaves["dims"], Kg)
    with pytest.raises(RuntimeError):
        dcd_b200.decode_location_flatten(d["pts"].to(DEV), ofs, d["direct"].to(DEV), Kg, PAD_B.to(DEV), bi)
    with pytest.raises(RuntimeError):
        dcd_b200.decode_location_flatten(d["pts"].to(DEV), ofs, d["direct"].to(DEV), K, PAD_B.to(DEV).requires_grad_(), bi)


def test_float64_inputs_get_float64_gradients():
    d = frames()
    up = upstream(d["ob"].N)
    g32, _ = ours_ensemble(d, up)
    g64, _ = ours_ensemble(d, up, dtype=torch.float64)
    for k in ENS_INPUTS:
        assert g64[k].dtype == torch.float64 and torch.equal(g64[k].float(), g32[k]), k
    fm = torch.randn(2, 16, 8, 8, device=DEV, dtype=torch.float64, requires_grad=True)
    idx = torch.tensor([[1, 5, 5], [0, 63, 2]], device=DEV)
    g = torch.randn(2, 3, 16, device=DEV)
    gm = torch.autograd.grad(dcd_b200.select_point_of_interest(2, idx, fm), fm, g)[0]
    fm32 = fm.detach().float().requires_grad_()
    g32m = torch.autograd.grad(dcd_b200.select_point_of_interest(2, idx, fm32), fm32, g)[0]
    assert gm.dtype == torch.float64 and torch.equal(gm.float(), g32m)


# ---------------------------------------------------------------------------------------------------------------------
# end to end: a DGDE-loss-shaped chain from the regression map
# ---------------------------------------------------------------------------------------------------------------------
CH = {"off3d": 0, "kp10": 2, "dims": 22, "direct": 25, "lud": 26, "luk": 27, "kpts2d": 30, "kpts3d": 176}
C_MAP, H_MAP, W_MAP, SLOTS = 395, 24, 80, 56


def e2e_inputs(seed=31):
    d = frames(seed)
    ob = d["ob"]
    N, B = ob.N, len(COUNTS)
    g = torch.Generator().manual_seed(seed)
    fmap = torch.randn(B, C_MAP, H_MAP, W_MAP, generator=g) * 0.1
    idx = torch.zeros(B, SLOTS, dtype=torch.int64)                   # padded slots all point at position 0
    mask = torch.zeros(B, SLOTS, dtype=torch.bool)
    pos = torch.empty(N, dtype=torch.int64)
    for b in range(B):
        sel = (ob.frame_id == b).nonzero().reshape(-1)
        p = torch.randperm(H_MAP * W_MAP - 1, generator=g)[:len(sel)] + 1
        pos[sel] = p
        idx[b, :len(sel)] = p
        mask[b, :len(sel)] = True
    pts = torch.stack(((pos % W_MAP).float(), (pos // W_MAP).float()), 1)
    pad = PAD_B[ob.frame_id]
    ofs = torch.rand(N, 2, generator=g) - 0.5
    centre = pts + ofs
    off = (ob.kps + pad.unsqueeze(1)) / 4 - centre.unsqueeze(1)
    kp10 = (ob.kps[:, -10:] + pad.unsqueeze(1)) / 4 - centre.unsqueeze(1)
    for o in range(N):
        b, p = int(ob.frame_id[o]), int(pos[o])
        col = fmap[b].view(C_MAP, -1)[:, p]
        col[CH["off3d"]:CH["off3d"] + 2] = ofs[o]
        col[CH["kp10"]:CH["kp10"] + 20] = kp10[o].reshape(-1)
        col[CH["dims"]:CH["dims"] + 3] = d["dims"][o]
        col[CH["direct"]] = d["direct"][o]
        col[CH["lud"]] = d["lud"][o]
        col[CH["luk"]:CH["luk"] + 3] = d["luk"][o]
        col[CH["kpts2d"]:CH["kpts2d"] + 146] = off[o].reshape(-1)
        col[CH["kpts3d"]:CH["kpts3d"] + 219] = ob.kps_3d[o].reshape(-1)
    # the ground truth the losses compare against: a little off the planted geometry
    gt_loc = torch.stack((torch.zeros(N), torch.zeros(N), ob.gt_depth), 1) + torch.randn(N, 3, generator=g)
    gt_depth = ob.gt_depth + torch.randn(N, generator=g)
    return d, fmap, idx, mask, pts, gt_loc, gt_depth


def e2e_chain(d, fmap, idx, mask, pts, gt_loc, gt_depth, impl, dev):
    """DGDE-loss-shaped chain; impl "ours" (dcd_b200) or "oracle"; all other steps plain torch."""
    ob = d["ob"]
    N, n, B = ob.N, 73, len(COUNTS)
    dtype = fmap.dtype
    bi = d["bi"].to(dev)
    pad = PAD_B.to(dev, dtype)
    K = d["K"].to(dev, dtype)
    if impl == "ours":
        pois = dcd_b200.select_point_of_interest(B, idx.to(dev), fmap)
    else:
        pois = O.select_point_of_interest(B, idx.to(dev), fmap)
    v = pois[mask.to(dev)]                                            # [N,C] valid target slots, image order
    ofs = v[:, CH["off3d"]:CH["off3d"] + 2]
    ptsd = pts.to(dev, dtype)
    kimg = (v[:, CH["kpts2d"]:CH["kpts2d"] + 146].reshape(N, n, 2) + (ptsd + ofs).unsqueeze(1)) * 4 - pad[bi].unsqueeze(1)
    k3 = v[:, CH["kpts3d"]:CH["kpts3d"] + 219].reshape(N, n, 3)
    rot = ob.rot_y.to(dev, dtype)
    if impl == "ours":
        depth = dcd_b200.edge_depth_mean(kimg, k3, rot, K, training=True)
        loc = dcd_b200.decode_location_flatten(ptsd, ofs, depth, K, pad, bi)
    else:
        depth = O.decode_pairs_kpts_depth(kimg, k3, rot, K, training=True)[0].mean(1)
        loc = oracle_locations(ptsd, ofs, depth, d["P"], pad, bi)
    L = (loc - gt_loc.to(dev, loc.dtype)).abs().mean()
    kp10 = v[:, CH["kp10"]:CH["kp10"] + 20].reshape(N, 10, 2)
    dims = v[:, CH["dims"]:CH["dims"] + 3]
    direct, lud = v[:, CH["direct"]], v[:, CH["lud"]]
    luk = v[:, CH["luk"]:CH["luk"] + 3]
    if impl == "ours":
        kd = dcd_b200.decode_depth_from_keypoints_batch(kp10, dims, K)
        out = dcd_b200.depth_ensemble(kp10, dims, K, luk, direct_depths=direct, direct_log_uncertainty=lud)
        ens, err = out["depth"], out["depth_error"]
    else:
        f_us = [float(p[0, 0]) for p in d["P"]]
        kd = O.decode_depth_from_keypoints_batch(kp10, dims, f_us, bi)
        ens, err, _ = O.depth_ensemble(direct, kd, lud, luk)
    gtd = gt_depth.to(dev, dtype)
    L = L + (kd - gtd.unsqueeze(1)).abs().mean() + (ens - gtd).abs().mean() + 0.1 * err.mean()
    return L


def test_end_to_end_map_gradient_vs_oracle():
    d, fmap, idx, mask, pts, gt_loc, gt_depth = e2e_inputs()
    grads = {}
    for impl, dtype, dev in (("ours", torch.float32, DEV), ("oracle", torch.float32, DEV), ("oracle", torch.float64, "cpu")):
        fm = fmap.to(dev, dtype).requires_grad_()
        L = e2e_chain(d, fm, idx, mask, pts, gt_loc, gt_depth, impl, dev)
        grads[(impl, dtype)] = torch.autograd.grad(L, fm)[0]
    ours, o32, o64 = grads[("ours", torch.float32)], grads[("oracle", torch.float32)], grads[("oracle", torch.float64)]
    assert float(o64.abs().max()) > 0
    check_grad("end-to-end map", ours, o32, o64, extra_bar=1e-4)
