"""Host-side mirror of the reference's call surface for the densely-constrained-depth path.

Same names, argument meaning and return values as the reference functions they replace
(SURVEY.md section 8b); the arithmetic runs in libdcd_b200.so (CUDA, sm_100a).  There is no
CPU path: non-CUDA tensors raise.

    decode_pairs_kpts_depth   <- Anno_Encoder.decode_pairs_kpts_depth   DGDE/model/anno_encoder.py:326
    compute_z                 <- compute_z                              GMW/main.py:373
    GMW.forward               <- GMW.forward                            GMW/model/model.py:195
    compute_reg_loss          <- compute_reg_loss                       GMW/main.py:364
plus fused fast paths for callers that do not need the per-edge intermediates:
    edge_depth_mean           decode_pairs_kpts_depth(...)[0].mean(1)   detector_infer.py:222-225, detector_loss.py:388
    gmw_weighted_depth        compute_z -> GMW.forward -> weighted sum  GMW/main.py:524-533
"""
from __future__ import annotations

import os
from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn

from . import _lib
from ._lib import check, f32c, ptr, require_cuda, stream_ptr
from .weights import NET_DEPTH, NET_NAMES, blob_size, pack_state_dict, unpack_blob

_CHECK_FINITE = os.environ.get("DCD_B200_CHECK_FINITE", "0") == "1"   # debug: synchronising range check of the GMW edge weights
K_SEL = 1500                 # anno_encoder.py:378, GMW/main.py:413
DGDE_CLAMP = (2.0, 80.0)     # anno_encoder.py:375
GMW_CLAMP = (0.1, 80.0)      # GMW/main.py:410
FLAG_NORMALISE_2D = 1
FLAG_SUB_B3 = 2
FLAG_FAST_QUOTIENT = 4
MAX_KPTS = 256


def _num_edges(n: int) -> int:
    return n * (n - 1) // 2


def _inference_only(name: str, *tensors) -> None:
    """Inference-only ops (refine_detections) have no backward: fail loudly instead of silently cutting the autograd graph."""
    if torch.is_grad_enabled() and any(t is not None and torch.is_tensor(t) and t.requires_grad for t in tensors):
        raise RuntimeError("dcd_b200.%s is inference-only (no backward is implemented): call it under torch.no_grad() "
                           "or detach its inputs" % name)


def _constant_inputs(name: str, **inputs) -> None:
    """Inputs that are constants in the reference (calibration, padding) get no gradient: fail loudly instead of silently
    cutting the graph when one requires grad."""
    for arg, t in inputs.items():
        if torch.is_grad_enabled() and torch.is_tensor(t) and t.requires_grad:
            raise RuntimeError("dcd_b200.%s: `%s` receives no gradient (a constant in the reference): detach it" % (name, arg))


def _check_shapes(kps, kps_3d, rot, K=None):
    if kps.dim() != 3 or kps.shape[-1] != 2:
        raise ValueError("kps must be [N,n,2], got %s" % (tuple(kps.shape),))
    N, n = kps.shape[0], kps.shape[1]
    if tuple(kps_3d.shape) != (N, n, 3):
        raise ValueError("kps_3d must be [N,n,3] matching kps, got %s" % (tuple(kps_3d.shape),))
    if rot.numel() != N:
        raise ValueError("rot_y must hold one yaw per object ([N,1] or [N])")
    if K is not None and tuple(K.shape) != (N, 3, 4):
        raise ValueError("K must be [N,3,4], got %s" % (tuple(K.shape),))
    if not 2 <= n <= MAX_KPTS:
        raise ValueError("keypoints per object must be in [2, %d]" % MAX_KPTS)
    return N, n


# ---------------------------------------------------------------------------------------------
# edge solve
# ---------------------------------------------------------------------------------------------
class _EdgeSolve(torch.autograd.Function):
    """All E edge depths (+ optional fused mean).  Gradients flow to kps and kps_3d only."""

    @staticmethod
    def forward(ctx, kps, kps_3d, rot, K, lo, hi, flags, want_edges, want_mean):
        N, n = kps.shape[0], kps.shape[1]
        E = _num_edges(n)
        dev = kps.device
        edges = torch.empty((N, E), dtype=torch.float32, device=dev) if want_edges else None
        mean = torch.empty((N,), dtype=torch.float32, device=dev) if want_mean else None
        if N:
            check(_lib.lib().dcd_edge_solve_fwd(ptr(kps), ptr(kps_3d), ptr(rot), ptr(K), N, n, lo, hi, flags,
                                                ptr(edges), ptr(mean), stream_ptr()), "dcd_edge_solve_fwd")
        ctx.save_for_backward(kps, kps_3d, rot, K)
        ctx.cfg = (lo, hi, flags)
        ctx.set_materialize_grads(False)
        if edges is None:
            edges = torch.empty((0,), dtype=torch.float32, device=dev)
            ctx.mark_non_differentiable(edges)
        if mean is None:
            mean = torch.empty((0,), dtype=torch.float32, device=dev)
            ctx.mark_non_differentiable(mean)
        return edges, mean

    @staticmethod
    def backward(ctx, g_edges, g_mean):
        kps, kps_3d, rot, K = ctx.saved_tensors
        lo, hi, flags = ctx.cfg
        N, n = kps.shape[0], kps.shape[1]
        g_kps = torch.zeros_like(kps)
        g_k3 = torch.zeros_like(kps_3d)
        if N and (g_edges is not None or g_mean is not None):
            ge = f32c(g_edges) if g_edges is not None else None
            gm = f32c(g_mean) if g_mean is not None else None
            check(_lib.lib().dcd_edge_solve_bwd(ptr(kps), ptr(kps_3d), ptr(rot), ptr(K), N, n, lo, hi, flags,
                                                0, 0, ptr(ge), ptr(gm), ptr(g_kps), ptr(g_k3), stream_ptr()),
                  "dcd_edge_solve_bwd")
        return g_kps, g_k3, None, None, None, None, None, None, None


class _EdgeSelectSolve(torch.autograd.Function):
    """Top-k edges by |V| (canonical order) with their depths, pair mask and mean."""

    @staticmethod
    def forward(ctx, kps, kps_3d, rot, K, mask_u8, lo, hi, flags, k, want_mean):
        N, n = kps.shape[0], kps.shape[1]
        dev = kps.device
        idx = torch.empty((N, k), dtype=torch.int64, device=dev)
        depth = torch.empty((N, k), dtype=torch.float32, device=dev)
        msel = torch.empty((N, k), dtype=torch.float32, device=dev) if mask_u8 is not None else None
        mean = torch.empty((N,), dtype=torch.float32, device=dev) if want_mean else None
        if N:
            check(_lib.lib().dcd_edge_select_fwd(ptr(kps), ptr(kps_3d), ptr(rot), ptr(K), ptr(mask_u8), N, n, k,
                                                 lo, hi, flags, ptr(idx), ptr(depth), ptr(msel), ptr(mean),
                                                 stream_ptr()), "dcd_edge_select_fwd")
        ctx.save_for_backward(kps, kps_3d, rot, K, idx)
        ctx.cfg = (lo, hi, flags, k)
        ctx.set_materialize_grads(False)
        ctx.mark_non_differentiable(idx)
        if msel is None:
            msel = torch.empty((0,), dtype=torch.float32, device=dev)
        ctx.mark_non_differentiable(msel)
        if mean is None:
            mean = torch.empty((0,), dtype=torch.float32, device=dev)
            ctx.mark_non_differentiable(mean)
        return depth, msel, idx, mean

    @staticmethod
    def backward(ctx, g_depth, _g_mask, _g_idx, g_mean):
        kps, kps_3d, rot, K, idx = ctx.saved_tensors
        lo, hi, flags, k = ctx.cfg
        N, n = kps.shape[0], kps.shape[1]
        g_kps = torch.zeros_like(kps)
        g_k3 = torch.zeros_like(kps_3d)
        if N and (g_depth is not None or g_mean is not None):
            gd = f32c(g_depth) if g_depth is not None else None
            gm = f32c(g_mean) if g_mean is not None else None
            check(_lib.lib().dcd_edge_solve_bwd(ptr(kps), ptr(kps_3d), ptr(rot), ptr(K), N, n, lo, hi, flags,
                                                ptr(idx), k, ptr(gd), ptr(gm), ptr(g_kps), ptr(g_k3), stream_ptr()),
                  "dcd_edge_solve_bwd")
        return g_kps, g_k3, None, None, None, None, None, None, None, None


def _prep_dgde(kps, kps_3d, rot_y, K):
    require_cuda(kps, kps_3d, rot_y, K)
    kps, kps_3d = f32c(kps), f32c(kps_3d)
    rot = f32c(rot_y).reshape(-1)
    K = f32c(K)                       # float64 stride-0 calibration at inference (detector_infer.py:221)
    _check_shapes(kps, kps_3d, rot, K)
    return kps, kps_3d, rot, K


def decode_pairs_kpts_depth(kps, kps_3d, rot_y, K, training=False, kpts_2d_mask=None, gt_depth=None, weight=None,
                            num_k: int = K_SEL, return_idx: bool = False):
    """Drop-in for Anno_Encoder.decode_pairs_kpts_depth (DGDE/model/anno_encoder.py:326-390).

    Returns (depth_all, depth_mask): depth_all is [N,E] (all edges, row-major i<j order) when not
    training, else the [N,1500] depths of the edges with the largest |v_i - v_j| sorted descending
    (ties by ascending edge id); depth_mask is the float32 0/1 product of the keypoint masks of the
    selected pairs, or None when kpts_2d_mask is None.  `gt_depth` and `weight` are accepted and
    unused, as in the reference.  Differentiable w.r.t. kps (v column) and kps_3d.
    """
    kps, kps_3d, rot, K = _prep_dgde(kps, kps_3d, rot_y, K)
    n = kps.shape[1]
    flags = FLAG_NORMALISE_2D | FLAG_SUB_B3
    lo, hi = DGDE_CLAMP
    if not training:
        depth, _ = _EdgeSolve.apply(kps, kps_3d, rot, K, lo, hi, flags, True, False)
        mask = None
        if kpts_2d_mask is not None:   # the reference still returns the (un-gathered) pair mask in this case
            m = kpts_2d_mask.to(torch.float32)
            ii, jj = torch.triu_indices(n, n, 1, device=kps.device)
            mask = m[:, ii] * m[:, jj]
        return (depth, mask, None) if return_idx else (depth, mask)
    if _num_edges(n) < num_k:
        raise RuntimeError("selected index k out of range: %d edges < k=%d (n=%d keypoints)" % (_num_edges(n), num_k, n))
    mask_u8 = None
    if kpts_2d_mask is not None:
        require_cuda(kpts_2d_mask)
        mask_u8 = (kpts_2d_mask != 0).to(torch.uint8).contiguous()
    depth, msel, idx, _ = _EdgeSelectSolve.apply(kps, kps_3d, rot, K, mask_u8, lo, hi, flags, num_k, False)
    mask = msel if kpts_2d_mask is not None else None
    return (depth, mask, idx) if return_idx else (depth, mask)


def edge_depth_mean(kps, kps_3d, rot_y, K, training=False, num_k: int = K_SEL, fast: bool = False) -> torch.Tensor:
    """Fused `decode_pairs_kpts_depth(...)[0].mean(1)` (detector_infer.py:222-225, detector_loss.py:388):
    per-object depth [N] without materialising the per-edge depths.  `fast=True` (inference, large batches) trades the
    IEEE division for the hardware reciprocal: per-object depth within 1e-6 (relative) of the default, see DCD_FAST_QUOTIENT."""
    kps, kps_3d, rot, K = _prep_dgde(kps, kps_3d, rot_y, K)
    flags = FLAG_NORMALISE_2D | FLAG_SUB_B3 | (FLAG_FAST_QUOTIENT if fast and not training else 0)
    lo, hi = DGDE_CLAMP
    if not training:
        return _EdgeSolve.apply(kps, kps_3d, rot, K, lo, hi, flags, False, True)[1]
    if _num_edges(kps.shape[1]) < num_k:
        raise RuntimeError("selected index k out of range")
    return _EdgeSelectSolve.apply(kps, kps_3d, rot, K, None, lo, hi, flags, num_k, True)[3]


DOWN_RATIO = 4.0    # MODEL.BACKBONE.DOWN_RATIO of the reference; hard-coded `*4` at detector_infer.py:217


def _calib_per_object(P, N, dev):
    """[3,4] / [N,3,4] torch or numpy projection matrix (float64 in the reference) -> contiguous FP32 [N,3,4]."""
    P = torch.as_tensor(P)
    if P.dim() == 2:
        P = P.unsqueeze(0).expand(N, -1, -1)
    return f32c(P.to(dev))


def _pad_per_object(pad_size, batch_idxs, N, dev):
    pad = torch.as_tensor(pad_size, dtype=torch.float32, device=dev)
    if pad.dim() == 1:
        return pad.reshape(1, 2).expand(N, 2).contiguous()
    if batch_idxs is not None:
        return pad[batch_idxs.to(dev).long()].contiguous()
    if pad.shape[0] == 1:
        return pad.expand(N, 2).contiguous()
    return f32c(pad)


class _LocateSolve(torch.autograd.Function):
    """compute_pairs_kpts_depth through dcd_dgde_locate_fwd (solve form); backward dcd_dgde_locate_solve_bwd -> keypoint offsets,
    template points, points (when floating), sub-pixel offsets, dims (h column)."""

    @staticmethod
    def forward(ctx, off, k3, pts, ofs, d3, rot, K, pad, want_loc):
        depth, loc = _locate_solve_fwd(off, k3, pts, ofs, d3, rot, K, pad, want_loc)
        ctx.save_for_backward(off, k3, pts, ofs, d3, rot, K, pad)
        ctx.set_materialize_grads(False)
        return (depth, loc) if want_loc else depth

    @staticmethod
    def backward(ctx, g_depth, g_loc=None):
        off, k3, pts, ofs, d3, rot, K, pad = ctx.saved_tensors
        need = ctx.needs_input_grad
        outs = [torch.empty_like(t) if t is not None and need[i] else None for i, t in ((0, off), (1, k3), (3, ofs), (2, pts), (4, d3))]
        N, n = off.shape[0], off.shape[1]
        if g_depth is None and g_loc is None or all(o is None for o in outs):
            return (None,) * 9
        if N:
            lo, hi = DGDE_CLAMP
            gd, gl = (f32c(g) if g is not None else None for g in (g_depth, g_loc))
            check(_lib.lib().dcd_dgde_locate_solve_bwd(ptr(off), ptr(k3), ptr(rot), ptr(K), ptr(pts), ptr(ofs), ptr(pad), ptr(d3), N, n,
                                                       lo, hi, FLAG_NORMALISE_2D | FLAG_SUB_B3, DOWN_RATIO, ptr(gd), ptr(gl),
                                                       *(ptr(o) for o in outs), stream_ptr()), "dcd_dgde_locate_solve_bwd")
        g_off, g_k3, g_ofs, g_pts, g_d3 = outs
        return g_off, g_k3, g_pts, g_ofs, g_d3, None, None, None, None


def _locate_solve_fwd(off, k3, pts, ofs, d3, rot, K, pad, want_loc):
    N, n = off.shape[0], off.shape[1]
    depth = torch.empty((N,), dtype=torch.float32, device=off.device)
    loc = torch.empty((N, 3), dtype=torch.float32, device=off.device) if want_loc else None
    lo, hi = DGDE_CLAMP
    if N:
        check(_lib.lib().dcd_dgde_locate_fwd(ptr(off), ptr(k3), ptr(rot), ptr(K), ptr(pts), ptr(ofs), ptr(pad),
                                             ptr(d3) if d3 is not None else 0, 0, N, n, lo, hi,
                                             FLAG_NORMALISE_2D | FLAG_SUB_B3, DOWN_RATIO, ptr(depth),
                                             ptr(loc) if loc is not None else 0, stream_ptr()), "dcd_dgde_locate_fwd")
    return depth, loc


def _needs_grad(*tensors) -> bool:
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors)


def compute_pairs_kpts_depth(pred_extra_kpts_2d, pred_bbox_points, pred_offset_3D, pad_size, pred_extra_kpts_3d, pred_rots, P,
                             batch_idxs=None, dims=None, return_locations: bool = False):
    """Fused form of PostProcessor.compute_pairs_kpts_depth (DGDE/model/head/detector_infer.py:215-227): the image-space
    keypoints `(kpts + (points + offsets)) * 4 - pad_size` are formed on the fly, solved over all keypoint pairs and
    averaged -> depth [N].  With `return_locations` also the object's 3D location (decode_location_flatten,
    anno_encoder.py:147-161, and `+ h / 2` on y when `dims` [N,3] is given, detector_infer.py:186-188) from the same launch.
    P: the image's 3x4 projection matrix (or one per object), pad_size: [2], [1,2], or [B,2] with batch_idxs.
    Differentiable (dcd_dgde_locate_solve_bwd) w.r.t. pred_extra_kpts_2d (the u column's gradient is exactly 0),
    pred_extra_kpts_3d, pred_offset_3D, pred_bbox_points when floating, and dims (h column); pred_rots, P and pad_size
    receive none (raise when they require grad).  float64 inputs get float64 gradients (the arithmetic is FP32)."""
    _constant_inputs("compute_pairs_kpts_depth", pred_rots=pred_rots, P=P, pad_size=pad_size)
    require_cuda(pred_extra_kpts_2d, pred_extra_kpts_3d, pred_rots, pred_bbox_points, pred_offset_3D)
    off, k3 = f32c(pred_extra_kpts_2d), f32c(pred_extra_kpts_3d)
    rot = f32c(pred_rots).reshape(-1)
    N, n = off.shape[0], off.shape[1]
    dev = off.device
    K = _calib_per_object(P, N, dev)
    _check_shapes(off, k3, rot, K)
    pts, ofs = f32c(pred_bbox_points), f32c(pred_offset_3D)
    pad = _pad_per_object(pad_size, batch_idxs, N, dev)
    d3 = f32c(dims) if dims is not None else None
    if _needs_grad(off, k3, pts, ofs, d3):
        return _LocateSolve.apply(off, k3, pts, ofs, d3, rot, K, pad, return_locations)
    depth, loc = _locate_solve_fwd(off, k3, pts, ofs, d3, rot, K, pad, return_locations)
    return (depth, loc) if return_locations else depth


# first channel of each regression group in the head's channel table of the reference configuration
# (DGDE/runs/DGDE.yaml:27-28: [4],[2],[20],[3],[3],[8,8],[1],[1],[146],[219]; layers/utils.py:22-38 Converter_key2channel)
DGDE_CHANNELS = {"3d_offset": 4, "extra_kpts_2d": 50, "extra_kpts_3d": 196}


def _frame_inputs(pred_regression, indexs, pred_rots, P, pad_size, batch_idxs, channels):
    """Arguments of the regression-map entry points -> (map [B,C,H,W], index [N] int64, batch index [N] int32 or None,
    yaw [N], calibration [N,3,4], pad [N,2] (all FP32 contiguous), channel table)."""
    fm = f32c(pred_regression)
    B = fm.shape[0]
    ch = dict(DGDE_CHANNELS)
    if channels:
        ch.update(channels)
    idx = indexs.reshape(-1).long().contiguous()
    N, dev = idx.shape[0], fm.device
    rot = f32c(pred_rots).reshape(-1)
    if rot.shape[0] != N:
        raise ValueError("pred_rots must hold one yaw per detection")
    bi = batch_idxs.to(dev).to(torch.int32).contiguous() if batch_idxs is not None else None
    if B > 1 and bi is None:
        raise ValueError("batch_idxs is required for a multi-image map")
    Pt = torch.as_tensor(P)
    if Pt.dim() == 3 and Pt.shape[0] != N and batch_idxs is not None:
        Pt = Pt.to(dev)[batch_idxs.to(dev).long()]
    K = _calib_per_object(Pt, N, dev)
    pad = _pad_per_object(pad_size, batch_idxs, N, dev)
    return fm, idx, bi, rot, K, pad, ch


def _frame_fwd(fm, idx, bi, rot, K, pad, d3, ch, n, return_keypoints):
    B, C, H, W = fm.shape
    N, dev = idx.shape[0], fm.device
    depth = torch.empty((N,), dtype=torch.float32, device=dev)
    loc = torch.empty((N, 3), dtype=torch.float32, device=dev)
    kimg = torch.empty((N, n, 2), dtype=torch.float32, device=dev) if return_keypoints else None
    k3 = torch.empty((N, n, 3), dtype=torch.float32, device=dev) if return_keypoints else None
    lo, hi = DGDE_CLAMP
    if N:
        check(_lib.lib().dcd_dgde_frame_fwd(ptr(fm), ptr(idx), ptr(bi), B, C, H, W, ch["extra_kpts_2d"], ch["extra_kpts_3d"],
                                            ch["3d_offset"], ptr(rot), ptr(K), ptr(pad), ptr(d3), N, n, lo, hi,
                                            FLAG_NORMALISE_2D | FLAG_SUB_B3, DOWN_RATIO, ptr(depth), ptr(loc), ptr(kimg), ptr(k3),
                                            stream_ptr()), "dcd_dgde_frame_fwd")
    return (depth, loc, kimg, k3) if return_keypoints else (depth, loc)


class _FrameDepths(torch.autograd.Function):
    """frame_depths_from_map through dcd_dgde_frame_fwd; backward dcd_dgde_frame_bwd -> the dense map gradient and dims (h
    column).  An output the loss does not use passes no gradient."""

    @staticmethod
    def forward(ctx, fm, d3, idx, bi, rot, K, pad, ch, n, return_keypoints):
        out = _frame_fwd(fm, idx, bi, rot, K, pad, d3, ch, n, return_keypoints)
        ctx.save_for_backward(fm, d3, idx, bi, rot, K, pad)
        ctx.cfg = (ch, n)
        ctx.set_materialize_grads(False)
        return out

    @staticmethod
    def backward(ctx, g_depth, g_loc, g_kimg=None, g_k3=None):
        fm, d3, idx, bi, rot, K, pad = ctx.saved_tensors
        ch, n = ctx.cfg
        up = [f32c(g) if g is not None else None for g in (g_depth, g_loc, g_kimg, g_k3)]
        if all(g is None for g in up):
            return (None,) * 10
        B, C, H, W = fm.shape
        N = idx.shape[0]
        g_map = torch.empty_like(fm) if N else torch.zeros_like(fm)
        g_d3 = torch.empty_like(d3) if d3 is not None and ctx.needs_input_grad[1] else None
        if N:
            lo, hi = DGDE_CLAMP
            check(_lib.lib().dcd_dgde_frame_bwd(ptr(fm), ptr(idx), ptr(bi), B, C, H, W, ch["extra_kpts_2d"], ch["extra_kpts_3d"],
                                                ch["3d_offset"], ptr(rot), ptr(K), ptr(pad), ptr(d3), N, n, lo, hi,
                                                FLAG_NORMALISE_2D | FLAG_SUB_B3, DOWN_RATIO, *(ptr(g) for g in up), ptr(g_map),
                                                ptr(g_d3), stream_ptr()), "dcd_dgde_frame_bwd")
        return (g_map if ctx.needs_input_grad[0] else None), g_d3, None, None, None, None, None, None, None, None


def frame_depths_from_map(pred_regression, indexs, pred_rots, P, pad_size, dims=None, batch_idxs=None, n: int = 73,
                          channels=None, return_keypoints: bool = False):
    """POI gather + image keypoints + edge solve + mean + 3D location in ONE launch, reading the regression map itself
    (detector_infer.py:107 select_point_of_interest, :133 / :216-219 channel slices, :215-227 compute_pairs_kpts_depth,
    :186-188 decode_location_flatten): pred_regression [B,C,H,W], indexs [N] int64 heat-map positions y * W + x of the kept
    detections (select_topk), pred_rots [N] decoded yaw, P the 3x4 calibration ([3,4], per image [B,3,4] with batch_idxs, or
    per object), pad_size [2] / [B,2], dims [N,3] or None -> (depth [N], locations [N,3]) and, with return_keypoints, the
    image-space 2D keypoints [N,n,2] and template points [N,n,3] that generate_infer_data dumps (:228-236).
    Every output is differentiable w.r.t. pred_regression and dims (h column) (dcd_dgde_frame_bwd: one dense map gradient,
    non-zero only in the three channel groups at the detections' positions; detections on one position summed in ascending
    order; a position outside the map passes none).  pred_rots, P and pad_size receive no gradient (raise when they require
    grad); float64 inputs get float64 gradients (the arithmetic is FP32).  The channel groups must not overlap."""
    _constant_inputs("frame_depths_from_map", pred_rots=pred_rots, P=P, pad_size=pad_size)
    require_cuda(pred_regression, indexs, pred_rots)
    fm, idx, bi, rot, K, pad, ch = _frame_inputs(pred_regression, indexs, pred_rots, P, pad_size, batch_idxs, channels)
    d3 = f32c(dims) if dims is not None else None
    if _needs_grad(fm, d3):
        return _FrameDepths.apply(fm, d3, idx, bi, rot, K, pad, ch, n, return_keypoints)
    return _frame_fwd(fm, idx, bi, rot, K, pad, d3, ch, n, return_keypoints)


class _LocateFlatten(torch.autograd.Function):
    """decode_location_flatten through dcd_dgde_locate_fwd (no solve); backward dcd_dgde_locate_bwd -> points (when floating
    and requiring grad), offsets, depths."""

    @staticmethod
    def forward(ctx, pts, ofs, dep, K, pad):
        N = pts.shape[0]
        loc = torch.empty((N, 3), dtype=torch.float32, device=pts.device)
        if N:
            check(_lib.lib().dcd_dgde_locate_fwd(0, 0, 0, ptr(K), ptr(pts), ptr(ofs), ptr(pad), 0, ptr(dep), N, 2, 0.0, 0.0, 0,
                                                 DOWN_RATIO, 0, ptr(loc), stream_ptr()), "dcd_dgde_locate_fwd")
        ctx.save_for_backward(pts, ofs, dep, K, pad)
        ctx.set_materialize_grads(False)
        return loc

    @staticmethod
    def backward(ctx, g_loc):
        pts, ofs, dep, K, pad = ctx.saved_tensors
        need = ctx.needs_input_grad
        if g_loc is None:
            return None, None, None, None, None
        N = pts.shape[0]
        g_pts = torch.empty_like(pts) if need[0] else None
        g_ofs = torch.empty_like(ofs) if need[1] else None
        g_dep = torch.empty_like(dep) if need[2] else None
        if N and (need[0] or need[1] or need[2]):
            check(_lib.lib().dcd_dgde_locate_bwd(ptr(K), ptr(pts), ptr(ofs), ptr(pad), ptr(dep), ptr(f32c(g_loc)), N, DOWN_RATIO,
                                                 ptr(g_ofs), ptr(g_pts), ptr(g_dep), stream_ptr()), "dcd_dgde_locate_bwd")
        return g_pts, g_ofs, g_dep, None, None


def decode_location_flatten(points, offsets, depths, P, pad_size, batch_idxs=None):
    """Anno_Encoder.decode_location_flatten (DGDE/model/anno_encoder.py:147-161) with the calibration given as the
    3x4 matrix of the image ([3,4]) or per object ([N,3,4]) instead of Calibration objects -> locations [N,3].
    Differentiable w.r.t. offsets, depths and (floating) points; P and pad_size are constants (raise when they require
    grad).  float64 inputs get float64 gradients (the arithmetic is FP32)."""
    require_cuda(points, offsets, depths)
    _constant_inputs("decode_location_flatten", P=P, pad_size=pad_size)
    pts, ofs, dep = f32c(points), f32c(offsets), f32c(depths).reshape(-1)
    N, dev = pts.shape[0], pts.device
    K = _calib_per_object(P, N, dev)
    pad = _pad_per_object(pad_size, batch_idxs, N, dev)
    return _LocateFlatten.apply(pts, ofs, dep, K, pad)


class _PoiGather(torch.autograd.Function):
    """select_point_of_interest through dcd_poi_gather_fwd; backward dcd_poi_gather_bwd (dense map gradient, duplicates summed
    in ascending slot order, no atomics)."""

    @staticmethod
    def forward(ctx, fm, idx):
        B, C, H, W = fm.shape
        out = torch.empty((B, idx.shape[1], C), dtype=torch.float32, device=fm.device)
        if out.numel():
            check(_lib.lib().dcd_poi_gather_fwd(ptr(fm), ptr(idx), B, idx.shape[1], C, H * W, ptr(out), stream_ptr()),
                  "dcd_poi_gather_fwd")
        ctx.save_for_backward(idx)
        ctx.shape = (B, C, H, W)
        ctx.set_materialize_grads(False)
        return out

    @staticmethod
    def backward(ctx, g_out):
        if g_out is None:
            return None, None
        (idx,) = ctx.saved_tensors
        B, C, H, W = ctx.shape
        g_map = torch.empty((B, C, H, W), dtype=torch.float32, device=idx.device)
        g = f32c(g_out)
        check(_lib.lib().dcd_poi_gather_bwd(ptr(g), ptr(idx), B, idx.shape[1], C, H * W, ptr(g_map), stream_ptr()),
              "dcd_poi_gather_bwd")
        return g_map, None


def select_point_of_interest(batch, index, feature_maps, validate: bool = False):
    """Drop-in for DGDE/model/layers/utils.py:120-145: feature_maps [B,C,H,W], index [B,K] flattened positions (or
    [B,K,2] (x, y) points) -> [B,K,C], reading only the selected values (no NHWC copy of the map).  An index outside the
    map yields NaN; `validate=True` checks the range first (a host synchronisation) and raises like torch.gather.
    Differentiable w.r.t. feature_maps: the [B,C,H,W] gradient is written densely by the library (no NHWC copy, no
    scatter_add), positions selected by several slots receive the sum of their gradients in ascending slot order, an index
    outside the map passes none; at most DCD_POI_BWD_MAX_K (1024) slots per image."""
    require_cuda(feature_maps, index)
    fm = f32c(feature_maps)
    B, C, H, W = fm.shape
    if index.dim() == 3:
        index = index[:, :, 1] * W + index[:, :, 0]
    idx = index.reshape(batch, -1).long().contiguous()
    if validate and idx.numel() and (int(idx.min()) < 0 or int(idx.max()) >= H * W):
        raise RuntimeError("index out of range")
    return _PoiGather.apply(fm, idx)


DEPTH_RANGE = (0.1, 100.0)   # MODEL.HEAD.DEPTH_RANGE (DGDE/config/defaults.py:196)
KP_DEPTH_EPS = 1e-3          # Anno_Encoder.EPS (anno_encoder.py:17)


class _DepthEnsemble(torch.autograd.Function):
    """dcd_dgde_depth_ensemble_fwd: keypoint depths only (`ensemble` False, decode_depth_from_keypoints_batch) or the whole
    ensemble (depth_ensemble).  Backward dcd_dgde_depth_ensemble_bwd: one launch for every output's gradient; an output the
    loss does not use passes none, so the keypoint-depth gradient alone is the same launch for both functions."""

    @staticmethod
    def forward(ctx, kp, dm, K, luk, dd, lud, sc, ensemble):
        N, dev = kp.shape[0], kp.device
        kd = torch.empty((N, 3), dtype=torch.float32, device=dev)
        depth = err = amax = so = None
        if ensemble:
            depth = torch.empty((N,), dtype=torch.float32, device=dev)
            err = torch.empty((N,), dtype=torch.float32, device=dev)
            amax = torch.empty((N,), dtype=torch.int64, device=dev)
            so = torch.empty((N,), dtype=torch.float32, device=dev) if sc is not None else None
        if N:
            check(_lib.lib().dcd_dgde_depth_ensemble_fwd(ptr(kp), ptr(dm), ptr(K), ptr(dd), ptr(lud), ptr(luk), ptr(sc), N,
                                                         DOWN_RATIO, KP_DEPTH_EPS, DEPTH_RANGE[0], DEPTH_RANGE[1], ptr(kd),
                                                         ptr(depth), ptr(err), ptr(amax), ptr(so), stream_ptr()),
                  "dcd_dgde_depth_ensemble_fwd")
        ctx.save_for_backward(kp, dm, K, luk, dd, lud, sc)
        ctx.set_materialize_grads(False)
        if not ensemble:
            return kd
        if amax is not None:
            ctx.mark_non_differentiable(amax)
        if so is None:
            so = torch.empty((0,), dtype=torch.float32, device=dev)
            ctx.mark_non_differentiable(so)
        return kd, depth, err, amax, so

    @staticmethod
    def backward(ctx, g_kd, g_depth=None, g_err=None, _g_amax=None, g_so=None):
        kp, dm, K, luk, dd, lud, sc = ctx.saved_tensors
        need = ctx.needs_input_grad
        N = kp.shape[0]
        if sc is None:
            g_so = None
        g_up = [f32c(g).reshape(-1) if g is not None else None for g in (g_kd, g_depth, g_err, g_so)]
        outs = [torch.empty_like(t) if t is not None and need[i] else None
                for i, t in ((0, kp), (1, dm), (4, dd), (5, lud), (3, luk), (6, sc))]
        if N and any(g is not None for g in g_up) and any(o is not None for o in outs):
            check(_lib.lib().dcd_dgde_depth_ensemble_bwd(ptr(kp), ptr(dm), ptr(K), ptr(dd), ptr(lud), ptr(luk), ptr(sc), N,
                                                         DOWN_RATIO, KP_DEPTH_EPS, DEPTH_RANGE[0], DEPTH_RANGE[1],
                                                         *(ptr(g) for g in g_up), *(ptr(o) for o in outs), stream_ptr()),
                  "dcd_dgde_depth_ensemble_bwd")
        else:
            outs = [o.zero_() if o is not None else None for o in outs]
        g_kp, g_dm, g_dd, g_lud, g_luk, g_sc = outs
        return g_kp, g_dm, None, g_luk, g_dd, g_lud, g_sc, None


def decode_depth_from_keypoints_batch(pred_keypoints, pred_dimensions, P, batch_idxs=None):
    """Anno_Encoder.decode_depth_from_keypoints_batch (DGDE/model/anno_encoder.py:193-224) with the calibration as the
    image's 3x4 matrix ([3,4]; [B,3,4] with batch_idxs; or per object [N,3,4]) -> [N,3] (centre, corner_02, corner_13).
    Differentiable w.r.t. pred_keypoints (v column; the u column's gradient is exactly 0) and pred_dimensions (h column);
    P is a constant (raises when it requires grad)."""
    require_cuda(pred_keypoints, pred_dimensions)
    _constant_inputs("decode_depth_from_keypoints_batch", P=P)
    kp, dm = f32c(pred_keypoints).reshape(-1, 10, 2), f32c(pred_dimensions)
    N, dev = kp.shape[0], kp.device
    P = torch.as_tensor(P)
    if P.dim() == 3 and batch_idxs is not None and P.shape[0] != N:
        P = P.to(dev)[batch_idxs.to(dev).long()]
    K = _calib_per_object(P, N, dev)
    return _DepthEnsemble.apply(kp, dm, K, None, None, None, None, False)


def depth_ensemble(pred_keypoints, pred_dimensions, P, keypoint_log_uncertainty, direct_depths=None,
                   direct_log_uncertainty=None, scores=None):
    """Fused detector_infer.py:141-171,197-203: keypoint depths, uncertainties = exp(channels), inverse-uncertainty soft
    ensemble -> dict(keypoint_depths [N,3], depth [N], depth_error [N], min_uncertainty [N] int64, scores [N,1] or None).
    Differentiable (like the reference's autograd) w.r.t. pred_keypoints (v column), pred_dimensions (h column), the log
    uncertainties, direct_depths and scores; min_uncertainty is not differentiable and P is a constant (raises when it
    requires grad)."""
    require_cuda(pred_keypoints, pred_dimensions, keypoint_log_uncertainty)
    _constant_inputs("depth_ensemble", P=P)
    kp, dm = f32c(pred_keypoints).reshape(-1, 10, 2), f32c(pred_dimensions)
    N, dev = kp.shape[0], kp.device
    K = _calib_per_object(P, N, dev)
    luk = f32c(keypoint_log_uncertainty).reshape(N, 3)
    dd = f32c(direct_depths).reshape(-1) if direct_depths is not None else None
    lud = f32c(direct_log_uncertainty).reshape(-1) if direct_log_uncertainty is not None else None
    if (dd is None) != (lud is None):
        raise RuntimeError("direct depth and its uncertainty channel go together")
    sc = f32c(scores).reshape(-1) if scores is not None else None
    kd, depth, err, amax, so = _DepthEnsemble.apply(kp, dm, K, luk, dd, lud, sc, True)
    return {"keypoint_depths": kd, "depth": depth, "depth_error": err, "min_uncertainty": amax,
            "scores": so.reshape(-1, 1) if sc is not None else None}


class _RayRescale(torch.autograd.Function):
    """dcd_gmw_ray_rescale_fwd; backward dcd_gmw_ray_rescale_bwd -> raw location, GMW depth, dim (h column)."""

    @staticmethod
    def forward(ctx, rl, pd, dm):
        out = _ray_rescale_fwd(rl, pd, dm)
        ctx.save_for_backward(rl, pd, dm)
        ctx.set_materialize_grads(False)
        return out

    @staticmethod
    def backward(ctx, g_out):
        if g_out is None:
            return None, None, None
        rl, pd, dm = ctx.saved_tensors
        outs = [torch.empty_like(t) if ctx.needs_input_grad[i] else None for i, t in enumerate((rl, pd, dm))]
        if rl.shape[0]:
            check(_lib.lib().dcd_gmw_ray_rescale_bwd(ptr(rl), ptr(pd), ptr(dm), ptr(f32c(g_out)), rl.shape[0],
                                                     *(ptr(o) for o in outs), stream_ptr()), "dcd_gmw_ray_rescale_bwd")
        return tuple(outs)


def _ray_rescale_fwd(rl, pd, dm):
    out = torch.empty_like(rl)
    if rl.shape[0]:
        check(_lib.lib().dcd_gmw_ray_rescale_fwd(ptr(rl), ptr(pd), ptr(dm), rl.shape[0], ptr(out), stream_ptr()),
              "dcd_gmw_ray_rescale_fwd")
    return out


def ray_rescale(raw_location, pred_depth, dim):
    """GMW/main.py:542-547: detector location [N,3] moved along its viewing ray to the GMW depth (dim [N,3] = (h,w,l)).
    Differentiable w.r.t. all three inputs (dim: h column only); float64 inputs get float64 gradients."""
    require_cuda(raw_location, pred_depth, dim)
    rl, pd, dm = f32c(raw_location), f32c(pred_depth).reshape(-1), f32c(dim)
    if _needs_grad(rl, pd, dm):
        return _RayRescale.apply(rl, pd, dm)
    return _ray_rescale_fwd(rl, pd, dm)


def compute_z(kpts_2d, kpts_3d, pred_rot, num_k: int = K_SEL) -> Tuple[torch.Tensor, torch.Tensor]:
    """Drop-in for GMW/main.py:373-416: (Z_v_raw [b,E] clamped to [0.1,80], good_idx [b,1500] int64).

    Z_v_raw is differentiable w.r.t. kpts_2d (v column; the u column's gradient is exactly 0, the solve does not read it)
    and kpts_3d, like the reference's.  pred_rot receives no gradient (as in decode_pairs_kpts_depth)."""
    require_cuda(kpts_2d, kpts_3d, pred_rot)
    kps, kps_3d = f32c(kpts_2d), f32c(kpts_3d)
    rot = f32c(pred_rot).reshape(-1)
    N, n = _check_shapes(kps, kps_3d, rot)
    if _num_edges(n) < num_k:
        raise RuntimeError("selected index k out of range")
    lo, hi = GMW_CLAMP
    Z, _ = _EdgeSolve.apply(kps, kps_3d, rot, None, lo, hi, 0, True, False)
    with torch.no_grad():
        idx = torch.empty((N, num_k), dtype=torch.int64, device=kps.device)
        if N:
            check(_lib.lib().dcd_edge_select_fwd(ptr(kps), ptr(kps_3d), ptr(rot), 0, 0, N, n, num_k, lo, hi, 0,
                                                 ptr(idx), 0, 0, 0, stream_ptr()), "dcd_edge_select_fwd")
    return Z, idx


# ---------------------------------------------------------------------------------------------
# GMW edge weights + aggregation
# ---------------------------------------------------------------------------------------------
POISON_WORKSPACES = os.environ.get("DCD_B200_POISON", "0") == "1"   # debug/tests: NaN-fill every workspace first


def _alloc_bytes(nbytes: int, dev) -> torch.Tensor:
    t = torch.empty(((nbytes + 255) // 256 * 64,), dtype=torch.float32, device=dev)
    if POISON_WORKSPACES:
        t.fill_(float("nan"))       # the kernels must never read what they did not write
    return t


def _mlp_backward(ctx, kpts_2d, kpts_3d, params4, params6, depth, g_reg_w, gn4, gn6):
    """dcd_gmw_weights_bwd over the activations the forward saved in ctx.ws, then dcd_gmw_kpts_bwd from the same scratch
    when a keypoint tensor needs a gradient -> (d kpts_2d, d kpts_3d, d params4, d params6), None where not needed.
    Frozen parameters still take the parameter backward (it fills the scratch the keypoint gradient is read from): its
    blobs are thrown away."""
    N, n = kpts_2d.shape[0], kpts_2d.shape[1]
    need = ctx.needs_input_grad
    g4 = torch.zeros_like(params4)
    g6 = torch.zeros_like(params6)
    gk2 = torch.zeros_like(kpts_2d) if need[0] else None
    gk3 = torch.zeros_like(kpts_3d) if need[1] else None
    if N and (g_reg_w is not None or gn4 is not None or gn6 is not None):
        L = _lib.lib()
        scratch = _alloc_bytes(L.dcd_gmw_bwd_scratch_bytes(N, n, depth), kpts_2d.device)
        check(L.dcd_gmw_weights_bwd(ptr(kpts_2d), ptr(kpts_3d), ptr(params4), ptr(params6), N, n, depth,
                                    ptr(g_reg_w), ptr(gn4), ptr(gn6), ptr(g4), ptr(g6), ptr(ctx.ws), ctx.ws.numel() * 4,
                                    ptr(scratch), scratch.numel() * 4, stream_ptr()), "dcd_gmw_weights_bwd")
        if gk2 is not None or gk3 is not None:
            check(L.dcd_gmw_kpts_bwd(ptr(params4), ptr(params6), N, n, depth, ptr(scratch), scratch.numel() * 4,
                                     ptr(gk2), ptr(gk3), stream_ptr()), "dcd_gmw_kpts_bwd")
    return gk2, gk3, (g4 if need[2] else None), (g6 if need[3] else None)


SINKHORN_CG_ITERATIONS, SINKHORN_CG_TOLERANCE = 32, 1e-7


def _gmw_forward(kpts_2d, kpts_3d, params4, params6, depth, save, plan, sums, lam, tol, iters):
    """Edge MLP (dcd_gmw_weights_fwd), then the Sinkhorn correspondence branch (dcd_gmw_transport_fwd, GMW/model/model.py:
    170-192) when `plan` or `sums` asks for it -> (reg_weights [N,E], edge_P [N,E,E] or None, (sum P, trace P) [N,2] or
    None, kept).  kept = (MLP workspace, f4, f6, u, v, Sinkhorn workspace whose first block is K) holds what a backward
    reads; with save=False (no backward will run) the MLP workspace is released before the Sinkhorn workspace is allocated
    and u, v are not written."""
    N, n = kpts_2d.shape[0], kpts_2d.shape[1]
    E = _num_edges(n)
    dev = kpts_2d.device
    L = _lib.lib()
    transport = plan or sums
    reg_w = torch.empty((N, E), dtype=torch.float32, device=dev)
    P = torch.empty((N, E, E), dtype=torch.float32, device=dev) if plan else None
    terms = torch.empty((N, 2), dtype=torch.float32, device=dev) if sums else None
    ws = f4 = f6 = u = v = tws = None
    if N:
        if transport:
            f4 = torch.empty((N, 128, E), dtype=torch.float32, device=dev)
            f6 = torch.empty((N, 128, E), dtype=torch.float32, device=dev)
        ws = _alloc_bytes(L.dcd_gmw_workspace_bytes(N, n, depth, int(save)), dev)
        check(L.dcd_gmw_weights_fwd(ptr(kpts_2d), ptr(kpts_3d), ptr(params4), ptr(params6), N, n, depth, int(save),
                                    ptr(reg_w), ptr(f4), ptr(f6), ptr(ws), ws.numel() * 4, stream_ptr()), "dcd_gmw_weights_fwd")
        if _CHECK_FINITE and not bool(torch.isfinite(reg_w).all()):
            # the tensor-core path carries activations as FP16 hi+lo pairs: |activation| must stay below 65504
            raise FloatingPointError("dcd_b200.GMW: non-finite edge weights (activation outside the FP16 hi/lo range?)")
        if not save:
            ws = None
        if transport:
            if save:
                u = torch.empty((N, E), dtype=torch.float32, device=dev)
                v = torch.empty((N, E), dtype=torch.float32, device=dev)
            tws = _alloc_bytes(L.dcd_gmw_transport_workspace_bytes(N, n), dev)
            check(L.dcd_gmw_transport_fwd(ptr(f4), ptr(f6), N, n, lam, tol, iters, ptr(P), ptr(u), ptr(v), ptr(terms),
                                          ptr(tws), tws.numel() * 4, stream_ptr()), "dcd_gmw_transport_fwd")
    return reg_w, P, terms, (ws, f4, f6, u, v, tws)


class _GmwEdgeBranch(torch.autograd.Function):
    """GMW.forward like the reference (GMW/model/model.py:195-207): reg_weights [b,E] and, by `branch`, no second output
    (None), the Sinkhorn transport plan edge_P [b,E,E] ("plan") or its two sums terms [b,2] = (sum P, trace P) ("terms"),
    all differentiable w.r.t. the parameter blobs and the keypoints.  Backward = implicit gradient of the Sinkhorn fixed
    point (optimal_transport.py:75-128 as one conjugate-gradient solve) -> feature gradients -> MLP backward.  For "terms"
    dL/dP = alpha 11^T + beta I with (alpha, beta) = dL/dterms: the backward rebuilds P from the forward's K, u and v inside
    the kernels (dcd_gmw_transport_terms_bwd), so K is the only E x E tensor kept between forward and backward, and the
    gradients equal the "plan" branch's for a dL/dP of that form.  An output the loss does not use passes no gradient
    (set_materialize_grads(False)): a reg_weights-only loss runs no transport backward on either branch."""

    @staticmethod
    def forward(ctx, kpts_2d, kpts_3d, params4, params6, depth, need_grad, branch, lam, tol, iters):
        ctx.set_materialize_grads(False)
        reg_w, P, terms, (ws, f4, f6, u, v, tws) = _gmw_forward(kpts_2d, kpts_3d, params4, params6, depth, need_grad,
                                                                branch == "plan", branch == "terms", lam, tol, iters)
        if need_grad:
            ctx.save_for_backward(kpts_2d, kpts_3d, params4, params6, f4, f6, u, v, P)
            ctx.ws, ctx.tws = ws, (tws if branch == "terms" else None)
            ctx.cfg = (depth, branch, lam)
        return reg_w, (P if branch == "plan" else terms)

    @staticmethod
    def backward(ctx, g_reg_w, g_second):
        kpts_2d, kpts_3d, params4, params6, f4, f6, u, v, P = ctx.saved_tensors
        depth, branch, lam = ctx.cfg
        N, n = kpts_2d.shape[0], kpts_2d.shape[1]
        L = _lib.lib()
        gn4 = gn6 = None
        if N and g_second is not None:
            g = f32c(g_second)
            gn4, gn6 = torch.empty_like(f4), torch.empty_like(f6)
            bws = _alloc_bytes(L.dcd_gmw_transport_bwd_workspace_bytes(N, n), g.device)
            if branch == "plan":
                check(L.dcd_gmw_transport_bwd(ptr(f4), ptr(f6), ptr(P), ptr(u), ptr(v), ptr(g), N, n, lam,
                                              SINKHORN_CG_ITERATIONS, SINKHORN_CG_TOLERANCE, ptr(gn4), ptr(gn6), 0,
                                              ptr(bws), bws.numel() * 4, stream_ptr()), "dcd_gmw_transport_bwd")
            else:
                check(L.dcd_gmw_transport_terms_bwd(ptr(f4), ptr(f6), ptr(ctx.tws), ctx.tws.numel() * 4, ptr(u), ptr(v),
                                                    ptr(g), N, n, lam, SINKHORN_CG_ITERATIONS, SINKHORN_CG_TOLERANCE,
                                                    ptr(gn4), ptr(gn6), 0, ptr(bws), bws.numel() * 4, stream_ptr()),
                      "dcd_gmw_transport_terms_bwd")
        ctx.tws = None
        g = f32c(g_reg_w) if g_reg_w is not None else None
        grads = _mlp_backward(ctx, kpts_2d, kpts_3d, params4, params6, depth, g, gn4, gn6)
        ctx.ws = None
        return grads + (None,) * 6


def correspondence_loss(terms: torch.Tensor) -> torch.Tensor:
    """correspondenceLoss(edge_P, eye) of GMW/main.py:456-457 (lib/losses.py:22-26,115-119) from GMW.transport_terms's
    terms [b,2] = (sum P, trace P): mean over objects of sum - 2 trace."""
    return (terms[:, 0] - 2 * terms[:, 1]).mean()


class _GmwAggregate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, reg_w, depths, idx):
        N, E = reg_w.shape
        k = idx.shape[1]
        out = torch.empty((N,), dtype=torch.float32, device=reg_w.device)
        if N:
            check(_lib.lib().dcd_gmw_aggregate_fwd(ptr(reg_w), ptr(depths), ptr(idx), N, E, k, 0, ptr(out), 0,
                                                   stream_ptr()), "dcd_gmw_aggregate_fwd")
        ctx.save_for_backward(reg_w, depths, idx)
        return out

    @staticmethod
    def backward(ctx, g_out):
        reg_w, depths, idx = ctx.saved_tensors
        N, E = reg_w.shape
        k = idx.shape[1]
        g_w = torch.empty_like(reg_w)
        g_z = torch.empty_like(depths) if ctx.needs_input_grad[1] else None
        if N:
            check(_lib.lib().dcd_gmw_aggregate_bwd(ptr(reg_w), ptr(depths), ptr(idx), N, E, k, 0, ptr(f32c(g_out)),
                                                   ptr(g_w), ptr(g_z), stream_ptr()), "dcd_gmw_aggregate_bwd")
        return g_w, g_z, None


class GMW(nn.Module):
    """Drop-in for the reference `GMW` module's regression branch (GMW/model/model.py:103-207).

    forward(kpts_2d, kpts_3d, pred_rot, args) -> (reg_weights [b,E], edge_P); `pred_rot` and `args`
    are ignored as in the reference (SURVEY fact 9).  edge_P (the Sinkhorn correspondence matrix
    of the classification branch, SURVEY 8f row N1) is None unless the module attribute `with_edge_P`
    is set (dcd_b200.patch.install sets it: both loops of GMW/main.py consume edge_P, :456 and :526); then it
    is the [b,E,E] transport plan, differentiable like the reference's (implicit Sinkhorn gradient,
    optimal_transport.py:75-128).  Both outputs are differentiable w.r.t. kpts_2d and kpts_3d as well (frozen parameters
    and keypoints that require grad: a trained GMW as a differentiable refiner of upstream keypoints).
    `edge_transport` gives the plan's (sum, trace) without materialising it; `transport_terms` gives them differentiably
    (with `correspondence_loss`, the correspondence loss at the memory cost of K alone).
    Parameters live in two flat blobs; `load_state_dict`/`state_dict` of the *reference* format
    are available through `load_reference_state_dict` / `reference_state_dict`.
    """

    def __init__(self, args=None, depth: int = NET_DEPTH):
        super().__init__()
        self.depth = depth
        self.params4 = nn.Parameter(torch.zeros(blob_size(4, depth)))
        self.params6 = nn.Parameter(torch.zeros(blob_size(6, depth)))
        self.with_edge_P = False

    def load_reference_state_dict(self, sd: Dict[str, torch.Tensor]) -> "GMW":
        sd = {k[len("module."):] if k.startswith("module.") else k: v for k, v in sd.items()}   # main.py:286-289
        with torch.no_grad():
            for (name, cin), p in zip(NET_NAMES, (self.params4, self.params6)):
                p.copy_(pack_state_dict(sd, name, cin, self.depth).to(p.device))
        return self

    def reference_state_dict(self) -> Dict[str, torch.Tensor]:
        out = {}
        for (name, cin), p in zip(NET_NAMES, (self.params4, self.params6)):
            out.update({k: v.detach().clone() for k, v in unpack_blob(p.data, name, cin, self.depth).items()})
        return out

    def reference_grads(self) -> Dict[str, torch.Tensor]:
        out = {}
        for (name, cin), p in zip(NET_NAMES, (self.params4, self.params6)):
            out.update({k: v.clone() for k, v in unpack_blob(p.grad, name, cin, self.depth).items()})
        return out

    SINKHORN_LAMBDA, SINKHORN_TOLERANCE, SINKHORN_ITERATIONS = 10.0, 1e-9, 100     # GMW/model/model.py:117-119

    @torch.no_grad()
    def edge_transport(self, kpts_2d, kpts_3d, materialise: bool = True, params=None):
        """Correspondence branch, forward only (SURVEY 8f row N1; GMW/model/model.py:170-192): returns
        (reg_weights [b,E], edge_P [b,E,E] or None, cls_terms [b,2] = (sum P, trace P)).
        correspondenceLoss(edge_P, eye) of GMW/main.py:456-457 is `(cls_terms[:, 0] - 2 * cls_terms[:, 1]).mean()`;
        with materialise=False the 4 E^2 bytes per object of edge_P are never written.  No gradient."""
        p4, p6 = params if params is not None else (self.params4, self.params6)
        k2, k3, _ = self._prepare(kpts_2d, kpts_3d, p4, p6)
        return _gmw_forward(k2, k3, p4, p6, self.depth, False, materialise, True, self.SINKHORN_LAMBDA,
                            self.SINKHORN_TOLERANCE, self.SINKHORN_ITERATIONS)[:3]

    def transport_terms(self, kpts_2d, kpts_3d, params=None):
        """Differentiable correspondence branch without the plan: (reg_weights [b,E], terms [b,2] = (sum P, trace P)).
        correspondenceLoss(edge_P, eye) of GMW/main.py:456-457 is `dcd_b200.correspondence_loss(terms)`.  Both outputs are
        differentiable w.r.t. the parameter blobs and the keypoints like forward()'s; the gradient of the plan goes through
        the same implicit Sinkhorn backward as edge_P's, rebuilding P from the forward's K (dcd_gmw_transport_terms_bwd),
        so the E x E tensors of edge_P, of the loss and of dL/dP are never formed: K (4 E^2 bytes per object) is the only one
        kept for the backward.  Under torch.no_grad() this is edge_transport(materialise=False) without the plan."""
        p4, p6 = params if params is not None else (self.params4, self.params6)
        return self._edge_branch("terms", kpts_2d, kpts_3d, p4, p6)

    def forward(self, kpts_2d, kpts_3d, pred_rot=None, args=None):
        return self.forward_blobs(kpts_2d, kpts_3d, self.params4, self.params6)

    @staticmethod
    def _prepare(kpts_2d, kpts_3d, params4, params6):
        require_cuda(kpts_2d, kpts_3d, params4, params6)
        k2, k3 = f32c(kpts_2d), f32c(kpts_3d)
        if k2.dim() != 3 or k2.shape[-1] != 2 or tuple(k3.shape) != (k2.shape[0], k2.shape[1], 3):
            raise ValueError("kpts_2d must be [b,n,2] and kpts_3d [b,n,3]")
        # the layer-wise forward that saves its activations runs whenever autograd will call the backward; otherwise
        # (torch.no_grad(), or nothing requires grad) the on-chip inference forward
        need_grad = torch.is_grad_enabled() and any(t.requires_grad for t in (k2, k3, params4, params6))
        return k2, k3, need_grad

    def forward_blobs(self, kpts_2d, kpts_3d, params4, params6):
        """forward() on explicit parameter blobs (dcd_b200.patch passes blobs packed from the LIVE reference parameters,
        so that their optimizer, checkpoints and DDP hooks keep working unchanged)."""
        return self._edge_branch("plan" if self.with_edge_P else None, kpts_2d, kpts_3d, params4, params6)

    def _edge_branch(self, branch, kpts_2d, kpts_3d, params4, params6):
        k2, k3, need_grad = self._prepare(kpts_2d, kpts_3d, params4, params6)
        return _GmwEdgeBranch.apply(k2, k3, params4, params6, self.depth, need_grad, branch, self.SINKHORN_LAMBDA,
                                    self.SINKHORN_TOLERANCE, self.SINKHORN_ITERATIONS)


def compute_reg_loss(pre_depths, edge_weight, gt_depth, good_idx=None, validate: bool = False):
    """Drop-in for GMW/main.py:364-371 -> (reg_loss, Z_select_weighted).  Shapes are checked; `validate=True` also checks
    the index range (a host synchronisation; the kernels clamp an out-of-range index to 0 or E - 1 instead of faulting).
    good_idx may repeat an edge: as with torch.gather, every slot counts in the softmax and the edge's gradients are the sum
    over its slots (in ascending slot order, deterministic)."""
    if good_idx is None:
        raise UnboundLocalError("compute_reg_loss needs good_idx (the reference fails without it too)")
    require_cuda(pre_depths, edge_weight, good_idx)
    if edge_weight.dim() != 2 or tuple(pre_depths.shape) != tuple(edge_weight.shape):
        raise RuntimeError("compute_reg_loss: pre_depths %s and edge_weight %s must both be [b,E]"
                           % (tuple(pre_depths.shape), tuple(edge_weight.shape)))
    if good_idx.dim() != 2 or good_idx.shape[0] != edge_weight.shape[0] or good_idx.shape[1] > edge_weight.shape[1]:
        raise RuntimeError("compute_reg_loss: good_idx must be [b,k] with k <= E, got %s" % (tuple(good_idx.shape),))
    idx = good_idx.to(torch.int64).contiguous()
    if validate and idx.numel() and (int(idx.min()) < 0 or int(idx.max()) >= edge_weight.shape[1]):
        raise RuntimeError("index out of range in compute_reg_loss (torch.gather raises here too)")
    Z = _GmwAggregate.apply(f32c(edge_weight), f32c(pre_depths), idx)
    reg_loss = (Z - gt_depth).abs().mean()
    return reg_loss, Z


def gmw_weighted_depth(kpts_2d, kpts_3d, pred_rot, model: GMW, chunk: int = 1024, num_k: int = K_SEL,
                       return_idx: bool = False):
    """Fused GMW inference (GMW/main.py:524-533): per-object softmax-weighted depth [b]."""
    require_cuda(kpts_2d, kpts_3d, pred_rot, model.params4)
    k2, k3 = f32c(kpts_2d), f32c(kpts_3d)
    rot = f32c(pred_rot).reshape(-1)
    N, n = _check_shapes(k2, k3, rot)
    if _num_edges(n) < num_k:
        raise RuntimeError("selected index k out of range")
    L = _lib.lib()
    out = torch.empty((N,), dtype=torch.float32, device=k2.device)
    idx = torch.empty((N, num_k), dtype=torch.int64, device=k2.device) if return_idx else None
    if N:
        chunk = max(1, min(chunk, N))
        ws = _alloc_bytes(L.dcd_gmw_depth_workspace_bytes(N, n, model.depth, chunk), k2.device)
        lo, hi = GMW_CLAMP
        with torch.no_grad():
            check(L.dcd_gmw_depth_fwd(ptr(k2), ptr(k3), ptr(rot), ptr(model.params4), ptr(model.params6), N, n,
                                      model.depth, num_k, lo, hi, chunk, ptr(out), ptr(idx), 0, ptr(ws),
                                      ws.numel() * 4, stream_ptr()), "dcd_gmw_depth_fwd")
    return (out, idx) if return_idx else out


GMW_KPTS = 73                # GMW reads the first 73 keypoints of every object (DCD_GMW_KPTS, wire.NUM_KPTS)


def refine_detections(pred_regression, indexs, pred_rots, P, pad_size, dims, gmw: GMW, batch_idxs=None, n: int = 73,
                      channels=None, chunk: int = 1024, params=None, return_inputs: bool = False) -> Dict[str, torch.Tensor]:
    """DGDE detections refined by GMW in one stream-ordered library call (dcd_dgde_gmw_refine_fwd): the regression map to
    the GMW-rescaled 3D locations with no host round trip (the reference writes gen_data_infer.json in
    DGDE/engine/inference.py:59-84 and reads it back in GMW/main.py:524-547).

    pred_regression, indexs, pred_rots, P, pad_size, batch_idxs, n, channels: as frame_depths_from_map (P [3,4], per image
    [B,3,4] with batch_idxs, or per object [N,3,4]).  dims [N,3]: the head's pred_dimensions in ITS order (l, h, w); h =
    dims[:, 1] is the `+ h/2` of the DGDE location and the h of the GMW ray rescale (GMW itself orders dim (h, w, l)).
    GMW's compute_z gets the same decoded yaw `pred_rots` as the DGDE solve (what wire.from_detector(pred_rot=...) records
    too).  gmw: a dcd_b200.GMW (its depth, and its parameter blobs unless `params` = (params4, params6) is given, e.g.
    `model._dcd_b200_blobs.get()` of a reference module patched by dcd_b200.patch.install, with gmw=`model._dcd_b200`).
    chunk: objects per GMW launch sequence (bounds the workspace, as gmw_weighted_depth's).

    Returns a dict: dgde_depth [N], dgde_location [N,3] (== frame_depths_from_map(..., dims)), gmw_depth [N] and location
    [N,3] (the GMW-rescaled location); with return_inputs also kpts_2d [N,73,2] (the normalised keypoints
    ((u - c_u) / f_u, (v - c_v) / f_v) of wire.from_detector, bit for bit), kpts_3d [N,73,3] and good_idx [N,1500] int64.
    Every output equals frame_depths_from_map -> normalisation -> gmw_weighted_depth (same chunk) -> ray_rescale(loc, z,
    dims[:, [1, 2, 0]]) bit for bit.  Inference-only (raises when an input requires grad; no gradient reaches the GMW
    parameters); a detection index outside the map gives NaN outputs for that object only."""
    if dims is None:
        raise ValueError("refine_detections needs dims [N,3] (l, h, w): h places the box centre for the ray rescale")
    if n < GMW_KPTS:
        raise ValueError("refine_detections needs n >= %d keypoints per object (GMW reads keypoints 0..%d), got %d"
                         % (GMW_KPTS, GMW_KPTS - 1, n))
    _inference_only("refine_detections", pred_regression, pred_rots, dims)
    p4, p6 = params if params is not None else (gmw.params4, gmw.params6)
    require_cuda(pred_regression, indexs, pred_rots, dims, p4, p6)
    fm, idx, bi, rot, K, pad, ch = _frame_inputs(pred_regression, indexs, pred_rots, P, pad_size, batch_idxs, channels)
    B, C, H, W = fm.shape
    N, dev = idx.shape[0], fm.device
    d3 = f32c(dims)
    if tuple(d3.shape) != (N, 3):
        raise ValueError("dims must be [N,3] (l, h, w), got %s" % (tuple(d3.shape),))
    p4, p6 = f32c(p4.detach()), f32c(p6.detach())
    f32 = dict(dtype=torch.float32, device=dev)
    out = {"dgde_depth": torch.empty((N,), **f32), "dgde_location": torch.empty((N, 3), **f32),
           "gmw_depth": torch.empty((N,), **f32), "location": torch.empty((N, 3), **f32)}
    k2 = k3 = gidx = None
    if return_inputs:
        k2 = torch.empty((N, GMW_KPTS, 2), **f32)
        k3 = torch.empty((N, GMW_KPTS, 3), **f32)
        gidx = torch.empty((N, K_SEL), dtype=torch.int64, device=dev)
        out.update(kpts_2d=k2, kpts_3d=k3, good_idx=gidx)
    if N:
        L = _lib.lib()
        chunk = max(1, min(chunk, N))
        ws = _alloc_bytes(L.dcd_dgde_gmw_refine_workspace_bytes(N, n, gmw.depth, chunk), dev)
        check(L.dcd_dgde_gmw_refine_fwd(ptr(fm), ptr(idx), ptr(bi), B, C, H, W, ch["extra_kpts_2d"], ch["extra_kpts_3d"],
                                        ch["3d_offset"], ptr(rot), ptr(K), ptr(pad), ptr(d3), ptr(p4), ptr(p6), N, n, gmw.depth,
                                        K_SEL, chunk, ptr(out["dgde_depth"]), ptr(out["dgde_location"]), ptr(out["gmw_depth"]),
                                        ptr(out["location"]), ptr(k2), ptr(k3), ptr(gidx), ptr(ws), ws.numel() * 4,
                                        stream_ptr()), "dcd_dgde_gmw_refine_fwd")
    return out
