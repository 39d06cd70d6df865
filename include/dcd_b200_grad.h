/*
 * dcd_b200_grad.h — backward of the fused frame-epilogue entry points of include/dcd_b200.h.
 *
 * Exported by the same library (libdcd_b200.so) with the same conventions as include/dcd_b200.h: extern "C", plain
 * device pointers and sizes, asynchronous on the given stream of the current device, allocation-free, capture-safe,
 * deterministic (no atomics), arguments checked before any CUDA call, N == 0 a no-op, outputs OVERWRITTEN, status
 * DCD_OK or DCD_E_*.  These are the training-side companions of dcd_dgde_frame_fwd, dcd_dgde_locate_fwd (solve form) and
 * dcd_gmw_ray_rescale_fwd; the gradients are those of the reference's unfused autograd (select_point_of_interest ->
 * channel slices -> image keypoints -> decode_pairs_kpts_depth(training=False).mean(1) -> decode_location_flatten -> + h/2,
 * and GMW/main.py:542-547) up to summation order.
 * 3 exported functions.
 */
#ifndef DCD_B200_GRAD_H_
#define DCD_B200_GRAD_H_

#include "dcd_b200.h"

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)   /* the library is built with -fvisibility=hidden */
#endif

/* Backward of dcd_dgde_frame_fwd, same inputs and scalars (the DGDE head's loss on the depth and location it reports, and on
 * the keypoints it hands to GMW).  Upstream gradients grad_depth [N], grad_locations [N,3], grad_kpts_img [N,n,2], grad_kps3d
 * [N,n,3]: each may be NULL (no gradient from that output), not all four.  Per detection the forward's reads are recomputed
 * from the map; the location's gradient (as dcd_dgde_locate_bwd, on the recomputed depth) and dL/d(depth) / E on every edge
 * of the mean (as dcd_edge_solve_bwd: the u column of the solve is exactly 0, clamp masks inclusive) go back through
 * (kpts_off + centre) * down_ratio - pad.  Outputs: grad_maps [B,C,H,W], dense, every element written: non-zero only in the
 * channel groups '3d_offset', 'extra_kpts_2d', 'extra_kpts_3d' at the detections' positions (keypoint channels down_ratio x
 * d/d(image keypoint); offset channels the sum of those over the keypoints plus the location's term); grad_dims [N,3] or NULL
 * (needs dims; only the h column is non-zero: grad_locations[:, 1] / 2).  Conventions of dcd_poi_gather_bwd: detections on
 * one position of one image are summed in ascending slot order (no atomics), a position outside the map passes no gradient to
 * it.  The three channel groups must not overlap.  No gradient flows to rot, K or pad. */
int dcd_dgde_frame_bwd(const float* feature_maps, const int64_t* index, const int32_t* batch_idx, int64_t B, int C, int H, int W,
                       int ch_kpts2d, int ch_kpts3d, int ch_offset3d, const float* rot, const float* K, const float* pad,
                       const float* dims, int64_t N, int n, float lo, float hi, int flags, float down_ratio,
                       const float* grad_depth, const float* grad_locations, const float* grad_kpts_img, const float* grad_kps3d,
                       float* grad_maps, float* grad_dims, void* stream);

/* Backward of dcd_dgde_locate_fwd's solve form (kpts_off != NULL), same inputs and scalars, with the per-object arithmetic of
 * dcd_dgde_frame_bwd.  grad_depth [N] and/or grad_locations [N,3] (not both NULL).  Outputs, each may be NULL, not all:
 * grad_kpts_off [N,n,2], grad_kps3d [N,n,3], grad_offsets [N,2], grad_points [N,2] (the same values: both enter as points +
 * offsets), grad_dims [N,3] (needs dims; h column only).  No gradient flows to rot, K or pad. */
int dcd_dgde_locate_solve_bwd(const float* kpts_off, const float* kps3d, const float* rot, const float* K, const float* points,
                              const float* offsets, const float* pad, const float* dims, int64_t N, int n, float lo, float hi,
                              int flags, float down_ratio, const float* grad_depth, const float* grad_locations,
                              float* grad_kpts_off, float* grad_kps3d, float* grad_offsets, float* grad_points, float* grad_dims,
                              void* stream);

/* Backward of dcd_gmw_ray_rescale_fwd (torch's autograd of GMW/main.py:542-547): grad_pred_location [N,3] -> grad_raw_location
 * [N,3], grad_pred_depth [N], grad_dim [N,3] (h = dim[:, 0] only; the other columns exactly 0); each output may be NULL, not
 * all three. */
int dcd_gmw_ray_rescale_bwd(const float* raw_location, const float* pred_depth, const float* dim, const float* grad_pred_location,
                            int64_t N, float* grad_raw_location, float* grad_pred_depth, float* grad_dim, void* stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* DCD_B200_GRAD_H_ */
