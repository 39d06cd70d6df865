"""Gradients of the fused DGDE frame epilogue (frame_depths_from_map, compute_pairs_kpts_depth) and of the GMW ray rescale.

Bars: against the hand composition of the unfused differentiable calls (select_point_of_interest -> channel slices ->
(off + centre) * 4 - pad -> decode_pairs_kpts_depth(training=False)[0].mean(1) -> decode_location_flatten -> + h/2), which
runs the same FP32 operations summed in another order, max|ours - composition| <= 1e-5 max|composition| per gradient tensor;
against the FP64 autograd of the oracle's frame_locations steps (oracle/dcd_oracle.py), the project's gradient bar
max|ours - f64| <= max(2 max|FP32 composition - f64|, 1e-4 max|f64|).
"""
import numpy as np
import pytest
import torch

import dcd_b200
from dcd_b200 import synth
from oracle import dcd_oracle as O

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
GEOMETRY_N = (2, 3, 32, 33, 73, 142, 143, 256)
SIZES_N = (0, 1, 5, 50, 301)
IMAGES = (1, 2, 4)
PAD_B = torch.tensor([[19.0, 5.0], [3.0, 7.0], [0.0, 0.0], [12.0, 8.0]])
UPSTREAM = ("depth", "loc", "kimg", "k3")


def channels(n):
    ch = {"extra_kpts_2d": 1, "extra_kpts_3d": 2 + 2 * n, "3d_offset": 3 + 5 * n}
    return ch, ch["3d_offset"] + 3


def make_frame(n, N, B, seed, W=64, bi=None, pos=None):
    """N detections spread over B images (each with its own P and pad), planted at distinct positions of each image (or at
    the given `pos` of images `bi`; detections sharing a position read the column planted last there)."""
    ch, C = channels(n)
    g = torch.Generator().manual_seed(seed)
    H = max(4, -(-N // W) + 1)
    if pos is None:
        bi = torch.sort(torch.randint(0, B, (N,), generator=g)).values
        pos = torch.empty(N, dtype=torch.int64)
        for b in range(B):
            sel = (bi == b).nonzero().reshape(-1)
            pos[sel] = torch.randperm(H * W, generator=g)[:sel.numel()]
    ob = synth.make_objects(n=n, seed=seed, counts=torch.tensor([max(N, 1)]))
    kps, k3, rot = ob.kps[:N], ob.kps_3d[:N], ob.rot_y[:N].reshape(-1)
    P = np.stack([np.array(synth.P2, dtype=np.float64) for _ in range(B)])
    P[:, 0, 0] *= 1 + 0.02 * np.arange(B)
    P[:, 1, 1] *= 1 + 0.02 * np.arange(B)
    pad = PAD_B[bi]
    pts = torch.stack(((pos % W).float(), (pos // W).float()), 1)
    ofs = torch.rand(N, 2, generator=g) - 0.5
    off = (kps + pad.unsqueeze(1)) / 4 - (pts + ofs).unsqueeze(1)
    fm = torch.randn(B, C, H, W, generator=g) * 0.1
    flat = fm.view(B, C, -1)
    for first, vals in ((ch["extra_kpts_2d"], off.reshape(N, 2 * n)), (ch["extra_kpts_3d"], k3.reshape(N, 3 * n)), (ch["3d_offset"], ofs)):
        c = first + torch.arange(vals.shape[1])
        flat.index_put_((bi[:, None], c[None, :], pos[:, None]), vals)
    dims = torch.stack((torch.full((N,), 3.9), 1.5 + torch.rand(N, generator=g), torch.full((N,), 1.6)), 1)
    return dict(fm=fm, pos=pos, bi=bi, rot=rot, P=P, pad=PAD_B[:B].clone(), dims=dims, ch=ch, n=n, B=B, W=W)


def upstream(N, n, seed=5, which=UPSTREAM):
    g = torch.Generator().manual_seed(seed)
    up = dict(depth=torch.randn(N, generator=g), loc=torch.randn(N, 3, generator=g), kimg=torch.randn(N, n, 2, generator=g) * 0.01,
              k3=torch.randn(N, n, 3, generator=g))
    return {k: (v if k in which else None) for k, v in up.items()}


def loss(outs, up, dev, dtype):
    L = 0
    for o, k in zip(outs, UPSTREAM):
        if o is not None and up[k] is not None:
            L = L + (o * up[k].to(dev, dtype)).sum()
    return L


def ours(f, up, return_keypoints=True, dtype=torch.float32):
    fm = f["fm"].to(DEV, dtype).requires_grad_()
    dims = f["dims"].to(DEV, dtype).requires_grad_()
    out = dcd_b200.frame_depths_from_map(fm, f["pos"].to(DEV), f["rot"].to(DEV), torch.from_numpy(f["P"]).to(DEV), f["pad"].to(DEV),
                                         dims=dims, batch_idxs=f["bi"].to(DEV), n=f["n"], channels=f["ch"],
                                         return_keypoints=return_keypoints)
    outs = tuple(out) + (None,) * (4 - len(out))
    return grads(loss(outs, up, DEV, torch.float32), [fm, dims]), outs


def grads(L, leaves):
    """Gradients of L, zeros for a leaf it does not reach."""
    gs = torch.autograd.grad(L, leaves, allow_unused=True)
    return tuple(torch.zeros_like(t) if g is None else g for g, t in zip(gs, leaves))


def gather(fm, f, impl):
    """select_point_of_interest per image, stitched in detection order -> [N,C]."""
    N, C = f["pos"].shape[0], fm.shape[1]
    rows = [None] * N
    for b in range(f["B"]):
        sel = (f["bi"] == b).nonzero().reshape(-1)
        if sel.numel() == 0:
            continue
        idx = f["pos"][sel].reshape(1, -1).to(fm.device)
        g = (dcd_b200.select_point_of_interest(1, idx, fm[b:b + 1]) if impl == "ours" else
             O.select_point_of_interest(1, idx, fm[b:b + 1])).reshape(-1, C)
        for r, i in enumerate(sel.tolist()):
            rows[i] = g[r]
    return torch.stack(rows) if N else fm.new_zeros((0, C))


def slices(v, f):
    n, ch, N = f["n"], f["ch"], v.shape[0]
    return (v[:, ch["extra_kpts_2d"]:ch["extra_kpts_2d"] + 2 * n].reshape(N, n, 2), v[:, ch["3d_offset"]:ch["3d_offset"] + 2],
            v[:, ch["extra_kpts_3d"]:ch["extra_kpts_3d"] + 3 * n].reshape(N, n, 3))


def composition(f, up, impl, dtype, dev):
    """impl "ours": the unfused dcd_b200 calls (FP32); "oracle": the oracle's steps in `dtype` (float64 on the CPU)."""
    fm = f["fm"].to(dev, dtype).requires_grad_()
    dims = f["dims"].to(dev, dtype).requires_grad_()
    N = f["pos"].shape[0]
    bi = f["bi"].to(dev)
    off, ofs, k3 = slices(gather(fm, f, impl), f)
    pts = torch.stack(((f["pos"] % f["W"]).to(dev, dtype), (f["pos"] // f["W"]).to(dev, dtype)), 1)
    pad = f["pad"].to(dev, dtype)
    Kt = torch.from_numpy(f["P"]).to(dev)[bi]
    kimg = (off + (pts + ofs).unsqueeze(1)) * 4 - pad[bi].unsqueeze(1)
    if impl == "ours":
        depth = dcd_b200.decode_pairs_kpts_depth(kimg, k3, f["rot"].to(dev), Kt, training=False)[0].mean(1)
        loc = dcd_b200.decode_location_flatten(pts, ofs, depth, Kt, pad, bi)
    else:
        depth = O.decode_pairs_kpts_depth(kimg, k3, f["rot"].to(dev, dtype).reshape(-1, 1), Kt.to(dtype), training=False)[0].mean(1)
        uv = (pts + ofs) * O.DOWN_RATIO - pad[bi]
        parts = [O.project_image_to_rect(torch.cat((uv[bi == b], depth[bi == b, None]), 1), f["P"][b]) for b in range(f["B"])]
        loc = torch.cat(parts) if N else uv.new_zeros((0, 3))
    loc = torch.cat((loc[:, :1], loc[:, 1:2] + dims[:, 1:2] / 2, loc[:, 2:]), 1)
    return grads(loss((depth, loc, kimg, k3), up, dev, dtype), [fm, dims]), (depth, loc, kimg, k3)


def close(a, b, bar, name):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    scale = float(b.abs().max()) if b.numel() else 0.0
    err = float((a - b).abs().max()) if b.numel() else 0.0
    assert err <= bar * scale, "%s: max err %.3e vs max|ref| %.3e" % (name, err, scale)


def check_against_references(f, up, fp64=True, return_keypoints=True):
    g, _ = ours(f, up, return_keypoints)
    gc, _ = composition(f, up, "ours", torch.float32, DEV)
    assert bool(torch.isfinite(g[0]).all())
    close(g[0], gc[0], 1e-5, "map vs composition")
    close(g[1], gc[1], 1e-5, "dims vs composition")
    if fp64:
        g64, _ = composition(f, up, "oracle", torch.float64, "cpu")
        for name, a, c, b in (("map", g[0], gc[0], g64[0]), ("dims", g[1], gc[1], g64[1])):
            # FP32 itself is off FP64 where |V| is small or an edge sits at a clamp: the bar allows twice the FP32 composition's
            # own error, and 1e-4 max|f64| in any case (the project's gradient bar, tests/test_gpu_dgde_head_grad.py)
            b = b.double()
            e32 = float((c.detach().double().cpu() - b).abs().max())
            err = float((a.detach().double().cpu() - b).abs().max())
            assert err <= max(2 * e32, 1e-4 * float(b.abs().max())), "%s vs FP64: %.3e, FP32 composition %.3e" % (name, err, e32)
    # nothing outside the three channel groups at the detections' positions
    mask = torch.zeros_like(f["fm"], dtype=torch.bool)
    ch, n = f["ch"], f["n"]
    groups = torch.cat([torch.arange(ch[k], ch[k] + w) for k, w in (("extra_kpts_2d", 2 * n), ("extra_kpts_3d", 3 * n),
                                                                       ("3d_offset", 2))])
    mask.view(f["B"], mask.shape[1], -1)[f["bi"][:, None], groups[None, :], f["pos"][:, None]] = True
    assert not bool(g[0].cpu()[~mask].any())
    assert not bool(g[1][:, [0, 2]].any())
    return g


CASES = [(n, N, IMAGES[(i + j) % 3]) for i, n in enumerate(GEOMETRY_N) for j, N in enumerate(SIZES_N)]


@pytest.mark.parametrize("n,N,B", CASES)
def test_frame_grad_vs_composition_and_fp64(n, N, B):
    f = make_frame(n, N, B, seed=10 * n + N + B)
    up = upstream(N, n)
    if N == 0:
        g, _ = ours(f, up)
        assert g[0].shape == f["fm"].shape and not bool(g[0].any()) and g[1].shape == (0, 3)
        return
    check_against_references(f, up)


@pytest.mark.parametrize("which", [(k,) for k in UPSTREAM] + [UPSTREAM, "no_keypoints"])
def test_each_upstream_gradient(which):
    n, N, B = 73, 50, 2
    f = make_frame(n, N, B, seed=123)
    if which == "no_keypoints":
        check_against_references(f, upstream(N, n, which=("depth", "loc")), return_keypoints=False)
    else:
        check_against_references(f, upstream(N, n, which=which))


def test_forward_is_unchanged_by_autograd():
    f = make_frame(73, 50, 2, seed=7)
    args = (f["pos"].to(DEV), f["rot"].to(DEV), torch.from_numpy(f["P"]).to(DEV), f["pad"].to(DEV))
    kw = dict(batch_idxs=f["bi"].to(DEV), n=73, channels=f["ch"], return_keypoints=True)
    with torch.no_grad():
        ref = dcd_b200.frame_depths_from_map(f["fm"].to(DEV), *args, dims=f["dims"].to(DEV), **kw)
    got = dcd_b200.frame_depths_from_map(f["fm"].to(DEV).requires_grad_(), *args, dims=f["dims"].to(DEV).requires_grad_(), **kw)
    for a, b in zip(got, ref):
        assert a.requires_grad and torch.equal(a.detach(), b)
    # the gathered form and the ray rescale
    off, ofs, k3g = (t.detach() for t in slices(gather(f["fm"].to(DEV), f, "ours"), f))
    pts = torch.stack(((f["pos"] % f["W"]).float(), (f["pos"] // f["W"]).float()), 1).to(DEV)
    Kt = torch.from_numpy(f["P"]).to(DEV)[f["bi"].to(DEV)]
    cargs = (pts, ofs, f["pad"].to(DEV), k3g, f["rot"].to(DEV), Kt)
    with torch.no_grad():
        rd, rl = dcd_b200.compute_pairs_kpts_depth(off, *cargs[:3], *cargs[3:], batch_idxs=f["bi"].to(DEV), dims=f["dims"].to(DEV),
                                                   return_locations=True)
    gd, gl = dcd_b200.compute_pairs_kpts_depth(off.clone().requires_grad_(), *cargs[:3], *cargs[3:], batch_idxs=f["bi"].to(DEV),
                                               dims=f["dims"].to(DEV), return_locations=True)
    assert torch.equal(gd.detach(), rd) and torch.equal(gl.detach(), rl) and torch.equal(rd, ref[0]) and torch.equal(rl, ref[1])
    z = ref[0] * 1.1
    with torch.no_grad():
        rr = dcd_b200.ray_rescale(ref[1], z, f["dims"].to(DEV))
    assert torch.equal(dcd_b200.ray_rescale(ref[1].clone().requires_grad_(), z, f["dims"].to(DEV)).detach(), rr)


def test_duplicates_are_summed_in_slot_order_like_poi_gather_bwd():
    """B images x K slots, several slots on one position: the map gradient is bit for bit dcd_poi_gather_bwd of the per-slot
    gradients (from the gathered form's backward), which sums in ascending slot order."""
    n, B, K, W = 33, 2, 12, 16
    pos = torch.randint(0, 40, (B, K), generator=torch.Generator().manual_seed(3))
    pos[0, 2:7] = 9                                                   # five slots on one position
    pos[1, :] = 17                                                    # every slot of image 1 on one position
    f = make_frame(n, B * K, B, seed=31, W=W, bi=torch.arange(B).repeat_interleave(K), pos=pos.reshape(-1))
    g = torch.Generator().manual_seed(4)
    scale = torch.logspace(-3, 3, B * K)[torch.randperm(B * K, generator=g)]
    up = upstream(B * K, n, which=("depth", "loc"))
    up = {k: (v * scale.view(-1, *([1] * (v.dim() - 1))) if v is not None else None) for k, v in up.items()}
    gm, _ = ours(f, up)
    # per-slot gradients of the same values through compute_pairs_kpts_depth's backward
    fm = f["fm"].to(DEV)
    off, ofs, k3 = (t.detach().clone().requires_grad_() for t in slices(gather(fm, f, "ours"), f))
    pts = torch.stack(((f["pos"] % W).float(), (f["pos"] // W).float()), 1).to(DEV)
    bi = f["bi"].to(DEV)
    d, l = dcd_b200.compute_pairs_kpts_depth(off, pts, ofs, f["pad"].to(DEV), k3, f["rot"].to(DEV),
                                             torch.from_numpy(f["P"]).to(DEV)[bi], batch_idxs=bi, dims=f["dims"].to(DEV),
                                             return_locations=True)
    go, gof, gk3 = grads(loss((d, l, None, None), up, DEV, torch.float32), [off, ofs, k3])
    C = fm.shape[1]
    per_slot = torch.zeros(B * K, C, device=DEV)
    ch = f["ch"]
    per_slot[:, ch["extra_kpts_2d"]:ch["extra_kpts_2d"] + 2 * n] = go.reshape(B * K, -1)
    per_slot[:, ch["extra_kpts_3d"]:ch["extra_kpts_3d"] + 3 * n] = gk3.reshape(B * K, -1)
    per_slot[:, ch["3d_offset"]:ch["3d_offset"] + 2] = gof
    fm2 = fm.clone().requires_grad_()
    ref = torch.autograd.grad(dcd_b200.select_point_of_interest(B, f["pos"].reshape(B, K).to(DEV), fm2), fm2,
                              per_slot.reshape(B, K, C))[0]
    assert torch.equal(gm[0], ref)
    # the order is visible at these scales: the reversed sum differs
    rev = torch.autograd.grad(dcd_b200.select_point_of_interest(B, f["pos"].reshape(B, K).flip(1).to(DEV), fm2), fm2,
                              per_slot.reshape(B, K, C).flip(1))[0]
    assert not torch.equal(rev, ref)


def test_position_outside_the_map_drops_only_its_own_gradient():
    n, N, B = 73, 9, 2
    f = make_frame(n, N, B, seed=41)
    up = upstream(N, n)
    H, W = f["fm"].shape[2:]
    bad = dict(f, pos=f["pos"].clone())
    bad["pos"][4] = H * W + 5
    gb, outs = ours(bad, up)
    torch.cuda.synchronize()
    assert bool(torch.isnan(outs[0][4])) and bool(torch.isfinite(gb[0]).all())
    keep = torch.arange(N) != 4
    sub = dict(f, pos=f["pos"][keep], bi=f["bi"][keep], rot=f["rot"][keep], dims=f["dims"][keep])
    gs, _ = ours(sub, {k: v[keep] for k, v in up.items()})
    assert torch.equal(gb[0], gs[0])
    assert torch.equal(gb[1][keep], gs[1]) and float(gb[1][4, 1]) == float(up["loc"][4, 1]) / 2


def saturated_frame(n, N, seed):
    """Every edge clamps (yaw 0, Z = 0, Y in {0, 1}, keypoints in two rows 800 px apart; see test_gpu_frame_geometry.py)."""
    f = make_frame(n, N, 1, seed)
    g = torch.Generator().manual_seed(seed)
    row = (torch.rand(N, n, generator=g) < 0.5).float()
    off = torch.stack((torch.randn(N, n, generator=g), 200 * row - 100), -1)
    k3 = torch.stack((torch.randn(N, n, generator=g), (torch.rand(N, n, generator=g) < 0.5).float(), torch.zeros(N, n)), -1)
    ch = f["ch"]
    flat = f["fm"].view(1, f["fm"].shape[1], -1)
    for first, vals in ((ch["extra_kpts_2d"], off.reshape(N, -1)), (ch["extra_kpts_3d"], k3.reshape(N, -1))):
        c = first + torch.arange(vals.shape[1])
        flat.index_put_((f["bi"][:, None], c[None, :], f["pos"][:, None]), vals)
    f["rot"] = torch.zeros(N)
    return f


def test_saturated_edges_pass_no_gradient():
    n, N = 33, 20
    f = saturated_frame(n, N, seed=51)
    up = upstream(N, n, which=("depth",))
    g, _ = ours(f, up)
    assert not bool(g[0].any())                                       # the depth alone reaches nothing through clamped edges
    gc, _ = composition(f, up, "ours", torch.float32, DEV)
    assert not bool(gc[0].any())
    check_against_references(f, upstream(N, n), fp64=False)


def test_gathered_form_vs_composition():
    n, N, B = 73, 50, 2
    f = make_frame(n, N, B, seed=61)
    fm = f["fm"].to(DEV)
    vals = [t.detach() for t in slices(gather(fm, f, "ours"), f)]
    pts0 = torch.stack(((f["pos"] % f["W"]).float(), (f["pos"] // f["W"]).float()), 1).to(DEV)
    bi = f["bi"].to(DEV)
    Kt = torch.from_numpy(f["P"]).to(DEV)[bi]
    up = upstream(N, n)
    res = {}
    for impl in ("fused", "composition"):
        off, ofs, k3 = (t.clone().requires_grad_() for t in vals)
        pts, dims = pts0.clone().requires_grad_(), f["dims"].to(DEV).requires_grad_()
        if impl == "fused":
            d, l = dcd_b200.compute_pairs_kpts_depth(off, pts, ofs, f["pad"].to(DEV), k3, f["rot"].to(DEV), Kt, batch_idxs=bi,
                                                     dims=dims, return_locations=True)
        else:
            kimg = (off + (pts + ofs).unsqueeze(1)) * 4 - f["pad"].to(DEV)[bi].unsqueeze(1)
            d = dcd_b200.decode_pairs_kpts_depth(kimg, k3, f["rot"].to(DEV), Kt, training=False)[0].mean(1)
            l = dcd_b200.decode_location_flatten(pts, ofs, d, Kt, f["pad"].to(DEV), bi)
            l = torch.cat((l[:, :1], l[:, 1:2] + dims[:, 1:2] / 2, l[:, 2:]), 1)
        res[impl] = torch.autograd.grad(loss((d, l, None, None), up, DEV, torch.float32), [off, k3, ofs, pts, dims])
    for name, a, b in zip(("kpts_off", "kps3d", "offsets", "points", "dims"), res["fused"], res["composition"]):
        close(a, b, 1e-5, name)
    assert not bool(res["fused"][0][:, :, 0].any())                  # the solve reads no u; no kimg upstream here
    assert torch.equal(res["fused"][2], res["fused"][3])


def ray_rescale_out_of_place(raw_location, pred_depth, dim):
    """oracle.ray_rescale's operations without its in-place updates (which autograd cannot differentiate)."""
    scale = pred_depth / raw_location[:, 2]
    h = dim[:, 0]
    y = raw_location[:, 1] - h / 2
    loc = scale.unsqueeze(-1) * torch.stack((raw_location[:, 0], y, raw_location[:, 2]), 1)
    return torch.stack((loc[:, 0], loc[:, 1] + h / 2, loc[:, 2]), 1)


def test_ray_rescale_grad_vs_fp64():
    N = 301
    g = torch.Generator().manual_seed(71)
    raw = torch.randn(N, 3, generator=g) * 5
    raw[:, 2] = 5 + 40 * torch.rand(N, generator=g)
    z = raw[:, 2] * (1 + 0.1 * torch.randn(N, generator=g))
    dim = torch.rand(N, 3, generator=g) + 1
    up = torch.randn(N, 3, generator=g)
    with torch.no_grad():
        assert torch.equal(ray_rescale_out_of_place(raw.double(), z.double(), dim.double()), O.ray_rescale(raw.double(), z.double(), dim.double()))
    leaves64 = [t.double().requires_grad_() for t in (raw, z, dim)]
    g64 = torch.autograd.grad((ray_rescale_out_of_place(*leaves64) * up.double()).sum(), leaves64)
    leaves = [t.to(DEV).requires_grad_() for t in (raw, z, dim)]
    ours_g = torch.autograd.grad((dcd_b200.ray_rescale(*leaves) * up.to(DEV)).sum(), leaves)
    for name, a, b in zip(("raw_location", "pred_depth", "dim"), ours_g, g64):
        close(a, b, 1e-5, name)
    assert not bool(ours_g[2][:, 1:].any())
    leaves = [t.to(DEV, torch.float64).requires_grad_() for t in (raw, z, dim)]
    g64d = torch.autograd.grad((dcd_b200.ray_rescale(*leaves) * up.to(DEV, torch.float64)).sum(), leaves)
    assert all(a.dtype == torch.float64 and torch.equal(a.float(), b) for a, b in zip(g64d, ours_g))


def test_float64_map_gets_float64_gradients():
    f = make_frame(33, 20, 2, seed=81)
    up = upstream(20, 33)
    g32, _ = ours(f, up)
    g64, _ = ours(f, up, dtype=torch.float64)
    assert g64[0].dtype == torch.float64 and torch.equal(g64[0].float(), g32[0]) and torch.equal(g64[1].float(), g32[1])


def test_cuda_graph_replays_forward_and_backward():
    f = make_frame(73, 50, 2, seed=91)
    up = {k: v.to(DEV) for k, v in upstream(50, 73).items()}
    fm = f["fm"].to(DEV).requires_grad_()
    dims = f["dims"].to(DEV).requires_grad_()
    args = (f["pos"].to(DEV), f["rot"].to(DEV), torch.from_numpy(f["P"]).float().to(DEV)[f["bi"].to(DEV)], f["pad"].to(DEV))
    kw = dict(dims=dims, batch_idxs=f["bi"].to(DEV), n=73, channels=f["ch"], return_keypoints=True)

    def step():
        outs = dcd_b200.frame_depths_from_map(fm, *args, **kw)
        return torch.autograd.grad(loss(outs, up, DEV, torch.float32), [fm, dims])

    eager = step()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = step()
    with torch.no_grad():
        static[0].fill_(float("nan"))
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(static[0], eager[0]) and torch.equal(static[1], eager[1])


def test_frozen_gmw_chain_from_the_map():
    """frame_depths_from_map(return_keypoints) -> normalisation -> compute_z + GMW.forward + compute_reg_loss -> ray_rescale ->
    loss, with a frozen GMW: the map gradient equals the same chain on the unfused calls; GMW's parameters get none."""
    n, N, B = 73, 20, 2
    f = make_frame(n, N, B, seed=101)
    model = dcd_b200.GMW().to(DEV).load_reference_state_dict(O.random_state_dict(7))
    model.params4.requires_grad_(False)
    model.params6.requires_grad_(False)
    bi = f["bi"].to(DEV)
    Kd = torch.from_numpy(f["P"]).float().to(DEV)[bi]
    rot = f["rot"].to(DEV)
    g = torch.Generator().manual_seed(5)
    gt_depth = (torch.rand(N, generator=g) * 30 + 10).to(DEV)
    gt_loc = (torch.randn(N, 3, generator=g) * 3).to(DEV)

    def chain(loc, kimg, k3, dims):
        k2 = torch.stack(((kimg[..., 0] - Kd[:, None, 0, 2]) / Kd[:, None, 0, 0], (kimg[..., 1] - Kd[:, None, 1, 2]) / Kd[:, None, 1, 1]), -1)
        Z, gidx = dcd_b200.compute_z(k2, k3, rot)
        w, _ = model(k2, k3, rot, None)
        reg, z = dcd_b200.compute_reg_loss(Z, w, gt_depth, gidx)
        out = dcd_b200.ray_rescale(loc, z, dims[:, [1, 2, 0]])
        return reg + (out - gt_loc).abs().mean()

    grads = {}
    for impl in ("fused", "composition"):
        fm = f["fm"].to(DEV).requires_grad_()
        dims = f["dims"].to(DEV).requires_grad_()
        if impl == "fused":
            _, loc, kimg, k3 = dcd_b200.frame_depths_from_map(fm, f["pos"].to(DEV), rot, torch.from_numpy(f["P"]).to(DEV),
                                                              f["pad"].to(DEV), dims=dims, batch_idxs=bi, n=n, channels=f["ch"],
                                                              return_keypoints=True)
        else:
            off, ofs, k3 = slices(gather(fm, f, "ours"), f)
            pts = torch.stack(((f["pos"] % f["W"]).float(), (f["pos"] // f["W"]).float()), 1).to(DEV)
            pad = f["pad"].to(DEV)
            kimg = (off + (pts + ofs).unsqueeze(1)) * 4 - pad[bi].unsqueeze(1)
            d = dcd_b200.decode_pairs_kpts_depth(kimg, k3, rot, Kd, training=False)[0].mean(1)
            loc = dcd_b200.decode_location_flatten(pts, ofs, d, Kd, pad, bi)
            loc = torch.cat((loc[:, :1], loc[:, 1:2] + dims[:, 1:2] / 2, loc[:, 2:]), 1)
        chain(loc, kimg[:, :73], k3[:, :73].contiguous(), dims).backward()
        grads[impl] = (fm.grad, dims.grad)
    assert float(grads["fused"][0].abs().max()) > 0
    close(grads["fused"][0], grads["composition"][0], 1e-5, "map")
    close(grads["fused"][1], grads["composition"][1], 1e-5, "dims")
    assert model.params4.grad is None and model.params6.grad is None
