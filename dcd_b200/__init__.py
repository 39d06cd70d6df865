"""dcd_b200 — B200-native (sm_100a) implementation of DCD's densely-constrained-depth hot path.

Public API (mirrors the reference's call surface, see dcd_b200/ops.py):
    decode_pairs_kpts_depth, edge_depth_mean, compute_z, GMW, compute_reg_loss, correspondence_loss, gmw_weighted_depth,
    compute_pairs_kpts_depth, decode_location_flatten, decode_depth_from_keypoints_batch, depth_ensemble, ray_rescale
    (detector-head frame epilogue), refine_detections (regression map -> GMW-rescaled locations in one call)
Host-side helpers: patch (attribute-patch the reference), dist (frame sharding + collectives),
weights (state_dict <-> parameter blob), synth (seeded KITTI-shaped objects), build (nvcc).
"""
from .ops import (GMW, K_SEL, compute_pairs_kpts_depth, compute_reg_loss, compute_z, correspondence_loss, decode_depth_from_keypoints_batch,
                  decode_location_flatten, decode_pairs_kpts_depth, depth_ensemble, edge_depth_mean, frame_depths_from_map,
                  gmw_weighted_depth, ray_rescale, refine_detections, select_point_of_interest)

__all__ = ["GMW", "K_SEL", "compute_pairs_kpts_depth", "compute_reg_loss", "compute_z", "correspondence_loss",
           "decode_depth_from_keypoints_batch",
           "decode_location_flatten", "decode_pairs_kpts_depth", "depth_ensemble", "edge_depth_mean", "frame_depths_from_map",
           "gmw_weighted_depth",
           "ray_rescale", "refine_detections", "select_point_of_interest"]
from .graphs import GraphedGmwStep  # noqa: E402

__all__.append("GraphedGmwStep")
__version__ = "0.2.0"
