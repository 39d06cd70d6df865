"""GMW softmax aggregation (csrc/gmw_aggregate.cu) against FP64: compute_reg_loss's gather -> softmax -> weighted sum and its
backward (GMW/main.py:364-371), and the C ABI's two depth layouts and its `probs` output, at the shapes, weight ranges and
index patterns where a warp-per-object gather / softmax / scatter goes wrong.

The reference is the same torch code evaluated in float64 on the GPU, with autograd (torch.gather's backward is a
scatter_add: a repeated index receives the SUM of its slots' gradients).  Bar, per tensor, as `_anchored` in
tests/test_gpu_gmw.py: |ours - f64| <= max(4 |ref32 - f64|, floor max|f64|) in max-norm, ref32 = the same torch code in FP32 on
the GPU; floor 1e-6 for the forward (depth, probs), 1e-5 for the gradients.
"""
import pytest
import torch

import dcd_b200
from dcd_b200 import _lib
from dcd_b200._lib import check, ptr, stream_ptr

pytestmark = pytest.mark.gpu
DEV = "cuda"
FLOOR_FWD, FLOOR_GRAD = 1e-6, 1e-5

# E = n(n-1)/2 for n = 2, 3, 20, 73, 256; k around the warp width, the reference's 1500 and k = E
EDGES = (1, 3, 190, 2628, 32640)
KS = (1, 31, 32, 33, 1500)
SHAPES = [(E, k) for E in EDGES for k in sorted({k for k in KS if k < E} | {E})]
# one object, one CTA minus / exactly / plus one warp (8 objects per CTA), and a ragged last CTA
NS = (1, 7, 8, 9, 1003)
PATTERNS = ("equal", "narrow", "wide", "dominant")


def weights(pattern, N, E, idx, g):
    """[N,E] edge weights.  wide: span 120, so that exp(w - max) of most selected edges is denormal or 0 in FP32;
    dominant: one selected edge (a different slot per object) 30 above the rest."""
    if pattern == "equal":
        return torch.full((N, E), 1.7, device=DEV)
    if pattern == "wide":
        return 120 * torch.rand(N, E, device=DEV, generator=g) - 60
    w = 1.5 + torch.rand(N, E, device=DEV, generator=g)
    if pattern == "dominant":
        slot = torch.randint(0, idx.shape[1], (N, 1), device=DEV, generator=g)
        w.scatter_(1, idx.gather(1, slot), 32.0)
    return w


def unique_idx(N, E, k, g):
    return torch.rand(N, E, device=DEV, generator=g).argsort(dim=1)[:, :k].contiguous()


def reference(w, z, idx, gout, sel, dtype):
    """(depth [N], probs [N,k], grad_w [N,E], grad_z) of the torch expression in `dtype`; z is [N,k] when sel else [N,E]."""
    w = w.detach().to(dtype).clone().requires_grad_(True)
    z = z.detach().to(dtype).clone().requires_grad_(True)
    p = w.gather(-1, idx).softmax(dim=-1)
    zs = z if sel else z.gather(-1, idx)
    out = (zs * p).sum(-1)
    gw, gz = torch.autograd.grad(out, (w, z), gout.to(dtype))
    return out.detach(), p.detach(), gw, gz


def anchored(name, mine, r32, r64, floor, log=None):
    e_o = float((mine.double() - r64).abs().max())
    e_r = float((r32.double() - r64).abs().max())
    amax = float(r64.abs().max())
    bound = max(4 * e_r, floor * amax)
    assert e_o <= bound, "%s: |ours - f64| = %.3g > %.3g (|ref32 - f64| = %.3g, max|f64| = %.3g)" % (name, e_o, bound, e_r, amax)
    if log is not None:
        log.append((name, e_o / max(amax, 1e-300), e_r / max(amax, 1e-300)))


def abi_forward(w, z, idx, sel):
    N, E = w.shape
    k = idx.shape[1]
    out = torch.full((N,), float("nan"), device=DEV)
    probs = torch.full((N, k), float("nan"), device=DEV)
    check(_lib.lib().dcd_gmw_aggregate_fwd(ptr(w), ptr(z), ptr(idx), N, E, k, int(sel), ptr(out), ptr(probs), stream_ptr()),
          "dcd_gmw_aggregate_fwd")
    return out, probs


def abi_backward(w, z, idx, sel, gout):
    """Outputs pre-filled with NaN: the kernel must write every element (dense grad_w: zero outside idx)."""
    N, E = w.shape
    k = idx.shape[1]
    gw = torch.full((N, E), float("nan"), device=DEV)
    gz = torch.full(tuple(z.shape), float("nan"), device=DEV)
    check(_lib.lib().dcd_gmw_aggregate_bwd(ptr(w), ptr(z), ptr(idx), N, E, k, int(sel), ptr(gout), ptr(gw), ptr(gz),
                                           stream_ptr()), "dcd_gmw_aggregate_bwd")
    return gw, gz


def check_all_paths(w, z, idx, gout, ref_idx=None, log=None, tag=""):
    """compute_reg_loss (ABI mode 0 with autograd) and both ABI modes with probs, against FP64 / FP32 references built from
    `ref_idx` (the clamped index when `idx` holds out-of-range entries).  Returns every output for determinism checks."""
    ref_idx = idx if ref_idx is None else ref_idx
    N, E = w.shape
    # mode 0 through the autograd wrapper: dense [N,E] depths gathered through idx
    wa, za = w.clone().requires_grad_(True), z.clone().requires_grad_(True)
    gt = torch.zeros(N, device=DEV)
    _, Z = dcd_b200.compute_reg_loss(za, wa, gt, idx)
    Z.backward(gout)
    d64, p64, gw64, gz64 = reference(w, z, ref_idx, gout, False, torch.float64)
    d32, p32, gw32, gz32 = reference(w, z, ref_idx, gout, False, torch.float32)
    anchored(tag + "depth", Z.detach(), d32, d64, FLOOR_FWD, log)
    anchored(tag + "grad_w", wa.grad, gw32, gw64, FLOOR_GRAD, log)
    anchored(tag + "grad_z", za.grad, gz32, gz64, FLOOR_GRAD, log)
    outs = [Z.detach(), wa.grad, za.grad]
    # mode 0 through the ABI with probs, and mode 1 (already-selected [N,k] depths)
    d0, pr0 = abi_forward(w, z, idx, False)
    assert torch.equal(d0, Z.detach())
    anchored(tag + "probs", pr0, p32, p64, FLOOR_FWD, log)
    zsel = z.gather(-1, ref_idx).contiguous()
    d1, pr1 = abi_forward(w, zsel, idx, True)
    s64, sp64, sgw64, sgz64 = reference(w, zsel, ref_idx, gout, True, torch.float64)
    s32, sp32, sgw32, sgz32 = reference(w, zsel, ref_idx, gout, True, torch.float32)
    anchored(tag + "depth sel", d1, s32, s64, FLOOR_FWD, log)
    assert torch.equal(pr1, pr0)
    gw1, gz1 = abi_backward(w, zsel, idx, True, gout)
    anchored(tag + "grad_w sel", gw1, sgw32, sgw64, FLOOR_GRAD, log)
    anchored(tag + "grad_z sel", gz1, sgz32, sgz64, FLOOR_GRAD, log)
    return outs + [pr0, d1, gw1, gz1]


@pytest.mark.parametrize("N", NS)
@pytest.mark.parametrize("E,k", SHAPES)
def test_aggregate_vs_fp64(E, k, N):
    g = torch.Generator(device=DEV).manual_seed(1000 * E + 10 * k + N)
    idx = unique_idx(N, E, k, g)
    z = 5 + 50 * torch.rand(N, E, device=DEV, generator=g)
    gout = torch.randn(N, device=DEV, generator=g)
    log = []
    for pattern in PATTERNS:
        check_all_paths(weights(pattern, N, E, idx, g), z, idx, gout, log=log, tag=pattern + " ")
    worst = max(log, key=lambda t: t[1] - 4 * t[2])
    print("E=%d k=%d N=%d: worst %s ours %.3g, ref32 %.3g (relative to max|f64|)" % (E, k, N, *worst))


def repeated_idx(N, E, k, g):
    """Unique rows with one edge planted at several slots: 2 copies in one lane chunk and across chunks, 3 copies in lanes
    0 / 31 / 0 of consecutive chunks, 33 consecutive copies (all lanes of a chunk + one), 33 copies at stride 45, several
    repeated edges in one chunk, 33 copies ending at the ragged last chunk; the last row has no repeat."""
    idx = unique_idx(N, E, k, g)
    plans = [[5, 17], [5, 1000], [0, 31, 32], list(range(100, 133)), [7 + 45 * t for t in range(33)],
             [[64, 66, 90], [65, 95], [70, 71, 72, 73]], list(range(k - 33, k))]
    for row, plan in enumerate(plans[:N - 1]):
        for slots in (plan if isinstance(plan[0], list) else [plan]):
            idx[row, slots] = idx[row, slots[-1]].clone()
    return idx


@pytest.mark.parametrize("k", [33, 1500])
def test_aggregate_repeated_indices_sum_like_scatter_add(k):
    """A repeated entry of good_idx: its gradients are the SUM over its slots (torch.gather's scatter_add backward), in both
    layouts; two runs are bit-identical."""
    N, E = 9, 2628
    g = torch.Generator(device=DEV).manual_seed(77 + k)
    idx = repeated_idx(N, E, 1500, g)[:, :k].contiguous() if k == 1500 else None
    if idx is None:         # k = 33: two chunks, the second of one lane
        idx = unique_idx(N, E, k, g)
        for row, slots in enumerate(([0, 1], [0, 32], [3, 20, 32], list(range(33)))):
            idx[row, slots] = idx[row, slots[0]].clone()
    assert any(int(torch.unique(r).numel()) < k for r in idx)
    z = 5 + 50 * torch.rand(N, E, device=DEV, generator=g)
    gout = torch.randn(N, device=DEV, generator=g)
    for pattern in PATTERNS:
        w = weights(pattern, N, E, idx, g)
        a = check_all_paths(w, z, idx, gout, tag=pattern + " ")
        b = check_all_paths(w, z, idx, gout, tag=pattern + " ")
        for x, y in zip(a, b):
            assert torch.equal(x, y)


def test_aggregate_out_of_range_indices_are_clamped():
    """An index below 0 reads edge 0 and one >= E edge E - 1 (the kernels clamp instead of faulting; validate=True raises).
    The reference is built from the clamped index only: a raw out-of-range index never reaches a torch op on the GPU.  The
    clamped slots land on edges that other slots also select, so the gradients there are sums."""
    N, E, k = 9, 2628, 1500
    g = torch.Generator(device=DEV).manual_seed(5)
    idx = unique_idx(N, E, k, g)
    idx[0, 0], idx[1, 7] = 0, E - 1                  # the clamp target is a real index of that row as well
    bad = torch.tensor([-1, -5, E, E + 100, -(1 << 40), 1 << 40], device=DEV)
    for row in range(N - 1):
        slots = 8 + torch.randperm(k - 8, device=DEV, generator=g)[:row + 1]
        idx[row, slots] = bad[torch.arange(row + 1, device=DEV) % bad.numel()]
    clamped = idx.clamp(0, E - 1)
    z = 5 + 50 * torch.rand(N, E, device=DEV, generator=g)
    gout = torch.randn(N, device=DEV, generator=g)
    for pattern in PATTERNS:
        w = weights(pattern, N, E, clamped, g)
        a = check_all_paths(w, z, idx, gout, ref_idx=clamped, tag=pattern + " ")
        b = check_all_paths(w, z, clamped, gout, tag=pattern + " ")
        for x, y in zip(a, b):
            assert torch.equal(x, y)
    with pytest.raises(RuntimeError):
        dcd_b200.compute_reg_loss(z, w, torch.zeros(N, device=DEV), idx, validate=True)


@pytest.mark.parametrize("E,k", [(190, 190), (2628, 1500), (32640, 1500)])
def test_aggregate_deterministic(E, k):
    N = 1003
    g = torch.Generator(device=DEV).manual_seed(E + k)
    idx = unique_idx(N, E, k, g)
    z = 5 + 50 * torch.rand(N, E, device=DEV, generator=g)
    w = weights("narrow", N, E, idx, g)
    gout = torch.randn(N, device=DEV, generator=g)
    runs = [(abi_forward(w, z, idx, False), abi_backward(w, z, idx, False, gout)) for _ in range(2)]
    for x, y in zip(runs[0], runs[1]):
        assert all(torch.equal(a, b) for a, b in zip(x, y))
