/*
 * dcd_b200.h — C ABI of the B200-native densely-constrained-depth hot path.
 *
 * One shared library (libdcd_b200.so, CUDA sm_100a only).  Every entry point is
 *   - extern "C", plain pointers and sizes (no torch / C++ types),
 *   - asynchronous on the given CUDA stream (cudaStream_t passed as void*), on the CURRENT device,
 *   - allocation-free and free of global mutable state (scratch comes from the caller as `workspace`,
 *     sized by the matching *_workspace_bytes query); safe under CUDA-graph capture,
 *   - returns 0 (DCD_OK) or a negative DCD_E_* code, never throws or aborts; dcd_strerror() names it.
 * All tensor pointers are DEVICE pointers to contiguous row-major FP32 unless stated otherwise.
 *
 * Notation: N objects, n keypoints per object, E = n(n-1)/2 edges in row-major strict-upper-triangle
 * order (edge e <-> (i,j), i<j; identical to torch.triu_indices(n,n,1)), k selected edges (1500 in
 * the reference).  Reference citations are relative to the BraveGroup/DCD repository.
 * 31 exported functions.
 */
#ifndef DCD_B200_H_
#define DCD_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)   /* the library is built with -fvisibility=hidden */
#endif

#define DCD_ABI_VERSION 2

/* status codes */
#define DCD_OK              0
#define DCD_E_INVALID      -1   /* bad argument (null pointer, n out of range, k > E, ...) */
#define DCD_E_WORKSPACE    -2   /* workspace too small / misaligned */
#define DCD_E_LAUNCH       -3   /* CUDA launch failure (cudaGetLastError) */
#define DCD_E_UNSUPPORTED  -4   /* shape outside what the kernels were built for */
#define DCD_E_DEVICE       -5   /* not an sm_100 device */

/* flags of the edge solve */
#define DCD_NORMALISE_2D    1   /* v = (kps_v - K[1][2]) / K[1][1]   (DGDE form, anno_encoder.py:331-334) */
#define DCD_SUB_B3          2   /* subtract K[2][3] after the clamp   (DGDE form, anno_encoder.py:385)     */
#define DCD_FAST_QUOTIENT   4   /* fused mean only (depth_edges == NULL, large N): |H| * rcp(|V|) with the 1-ulp hardware
                                   reciprocal instead of the IEEE division; per-object mean within 1e-6 (relative) of the
                                   exact one, per-edge values not bit-faithful.  Opt-in; ignored otherwise. */

#define DCD_MAX_KPTS      256   /* pair ids are packed in 16 bits */
#define DCD_NET_CH        128   /* channels of the edge MLP (yi2018cvpr/config.py:72) */
#define DCD_GMW_KPTS       73   /* GMW reads the first 73 keypoints of every object (GMW/utilities/dataset_utilities.py:45-46) */

int         dcd_version(void);
const char* dcd_strerror(int rc);

/* ------------------------------------------------------------------------------------------------
 * Edge-depth solve, forward.  Replaces Anno_Encoder.decode_pairs_kpts_depth(training=False)
 * (DGDE/model/anno_encoder.py:326-390) incl. get_up (:313-324), and the depth half of GMW's compute_z
 * (GMW/main.py:373-411).  Per edge (i<j):
 *     C = X*sin(rot) - Z*cos(rot);  H = (Y_i - Y_j) + (v_i*C_i - v_j*C_j);  V = v_i - v_j
 *     z = min(max(|H| / max(|V|, 1e-10), lo), hi)  [- K[2][3] if DCD_SUB_B3]
 * with every product/sum rounded separately and an IEEE division, i.e. the reference's FP32 rounding
 * sequence.  kps [N,n,2] (u,v), kps3d [N,n,3], rot [N], K [N,3,4] (may be NULL when neither flag is set).
 * depth_edges [N,E] and/or depth_mean [N] (mean over all E edges, detector_infer.py:225) may be NULL.
 */
int dcd_edge_solve_fwd(const float* kps, const float* kps3d, const float* rot, const float* K,
                       int64_t N, int n, float lo, float hi, int flags,
                       float* depth_edges, float* depth_mean, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Edge selection + solve.  Replaces the training branch of decode_pairs_kpts_depth
 * (anno_encoder.py:377-382: torch.topk of |V|, gather of depths and of the pair mask) and the index
 * half of compute_z (GMW/main.py:413-414).  idx_out [N,k] int64: the k edges with the largest |V|,
 * sorted by (|V| descending, edge id ascending) — the canonical tie rule.  depth_sel [N,k] depths of
 * those edges (same arithmetic as dcd_edge_solve_fwd), mask_sel [N,k] = mask[i]*mask[j] as 0/1 float
 * (kpt_mask [N,n] uint8, may be NULL together with mask_sel), depth_mean [N] = mean of depth_sel
 * (detector_loss.py:388).  Outputs other than idx_out may be NULL.
 */
size_t dcd_edge_select_workspace_bytes(int64_t N, int n);
int dcd_edge_select_fwd(const float* kps, const float* kps3d, const float* rot, const float* K,
                        const uint8_t* kpt_mask, int64_t N, int n, int k, float lo, float hi, int flags,
                        int64_t* idx_out, float* depth_sel, float* mask_sel, float* depth_mean,
                        void* stream);

/* ------------------------------------------------------------------------------------------------
 * Frame epilogue of the detector head around the edge solve (SURVEY 8f rows N2 / N4), fused:
 *   image-space keypoints  (kpts_off + (points + offsets)) * down_ratio - pad     DGDE/model/head/detector_infer.py:216-217
 *   edge solve + mean over the edges (inference form of decode_pairs_kpts_depth)  DGDE/model/anno_encoder.py:326-390, detector_infer.py:225
 *   location = project_image_to_rect((points + offsets) * down_ratio - pad, depth) anno_encoder.py:147-161, kitti_utils.py:239-244,399-417
 *   location.y += dims[:, 1] / 2 when dims != NULL                                 detector_infer.py:188
 * kpts_off [N,n,2] keypoint regression offsets (feature-map units), points / offsets [N,2] (heat-map peak and its
 * sub-pixel offset), pad [N,2] (pad_size[batch_idxs]), K [N,3,4] (required), dims [N,3] (l,h,w) or NULL.
 * kpts_off == NULL: no solve, the depths are read from depth_in [N] (the reference's first decode_location_flatten
 * call with the ensemble depth, detector_infer.py:175-176).  Outputs: depth_out [N] and/or locations [N,3].
 */
int dcd_dgde_locate_fwd(const float* kpts_off, const float* kps3d, const float* rot, const float* K,
                        const float* points, const float* offsets, const float* pad, const float* dims,
                        const float* depth_in, int64_t N, int n, float lo, float hi, int flags, float down_ratio,
                        float* depth_out, float* locations, void* stream);

/* The frame epilogue straight from the detector's regression map (row N2 fused into the load stage): ONE launch for
 *   select_point_of_interest                                        DGDE/model/layers/utils.py:120-145, detector_infer.py:107
 *   the key2channel slices '3d_offset', 'extra_kpts_2d', 'extra_kpts_3d'   detector_infer.py:133,216,219 (layers/utils.py:22-38)
 *   image keypoints -> edge solve -> mean -> location (+ h/2)          as dcd_dgde_locate_fwd
 * feature_maps [B,C,H,W]; index [N] int64 = y * W + x of each kept detection (select_topk's indices after the score
 * threshold), batch_idx [N] int32 (NULL when B == 1); ch_*: first channel of each group in the head's channel table
 * (DGDE.yaml: 4, 50, 196 for '3d_offset', 'extra_kpts_2d', 'extra_kpts_3d'); points = (index % W, index / W) as in
 * select_topk (layers/utils.py:61-93).  rot [N] (decoded yaw), K [N,3,4], pad [N,2], dims [N,3] or NULL.
 * Outputs (NULL to skip): depth_out [N], locations [N,3], kpts_img_out [N,n,2] / kps3d_out [N,n,3] (what
 * generate_infer_data dumps for GMW, detector_infer.py:228-236).  A position outside the map yields NaN, never a fault. */
int dcd_dgde_frame_fwd(const float* feature_maps, const int64_t* index, const int32_t* batch_idx, int64_t B, int C, int H, int W,
                       int ch_kpts2d, int ch_kpts3d, int ch_offset3d, const float* rot, const float* K, const float* pad,
                       const float* dims, int64_t N, int n, float lo, float hi, int flags, float down_ratio, float* depth_out,
                       float* locations, float* kpts_img_out, float* kps3d_out, void* stream);

/* Depth ensemble of the detector head (rest of row N4).  kp10 [N,10,2]: the regressed box keypoints (8 corners, bottom
 * centre, top centre; feature-map units), dims [N,3] (l,h,w), K [N,3,4] (f_u = K[0][0]).
 *   keypoint depths [N,3] = clamp(f_u * h / (relu(height) * down_ratio + eps), lo, hi) for the centre line and the two
 *   diagonal corner pairs (mean of two each)                           DGDE/model/anno_encoder.py:193-224
 *   uncertainties = exp(log_unc_*); weights = (1/u) / sum(1/u); depth = sum(w d); depth_error = sum(w u)
 *   over {direct, 3 keypoint depths} (direct == NULL: the 3 keypoint depths)      detector_infer.py:141,154,158-171
 *   scores_out = scores * (1 - clamp(depth_error, 0.01, 1)), NaN -> 0             detector_infer.py:197-203
 * Every output may be NULL; argmax is torch.argmax of the weights (int64). */
int dcd_dgde_depth_ensemble_fwd(const float* kp10, const float* dims, const float* K, const float* direct,
                                const float* log_unc_direct, const float* log_unc_kp, const float* scores, int64_t N,
                                float down_ratio, float eps, float lo, float hi, float* kp_depths, float* depth,
                                float* depth_error, int64_t* argmax, float* scores_out, void* stream);

/* Upstream gather (row N2): select_point_of_interest (DGDE/model/layers/utils.py:120-145).  feature_maps [B,C,H,W],
 * index [B,K] int64 flattened positions y * W + x, out [B,K,C] = feature_maps[b, :, index[b,k]] (NaN for an index outside
 * [0, H*W): no memory fault, no device-side assert).
 * The reference permutes the whole map to NHWC first; this reads only the K*C selected values. */
int dcd_poi_gather_fwd(const float* feature_maps, const int64_t* index, int64_t B, int64_t K, int C, int64_t HW,
                       float* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Backward of the frame-epilogue functions around the edge solve (the autograd of the reference's DGDE loss,
 * detector_loss.py:391).  Same conventions as the forwards: outputs OVERWRITTEN, N == 0 (B == 0) a no-op, deterministic, no
 * atomics, arguments checked before any CUDA call.
 *
 * Backward of dcd_poi_gather_fwd.  grad_out [B,K,C] -> grad_maps [B,C,HW] (dense, every element written):
 * grad_maps[b,c,p] = sum of grad_out[b,k,c] over the k with index[b,k] == p, summed in ascending k, +0.0 elsewhere.
 * Duplicate positions (padded target slots) are the normal case.  An index outside [0, HW) drops its gradient.  Each slot
 * scans the image's K indices for duplicates: K > DCD_POI_BWD_MAX_K returns DCD_E_UNSUPPORTED.  grad_out and index may be
 * NULL when K == 0 (grad_maps is then filled with zeros). */
#define DCD_POI_BWD_MAX_K 1024
int dcd_poi_gather_bwd(const float* grad_out, const int64_t* index, int64_t B, int64_t K, int C, int64_t HW, float* grad_maps,
                       void* stream);

/* Backward of dcd_dgde_locate_fwd's no-solve form (decode_location_flatten, anno_encoder.py:147-161; kpts_off == NULL, dims
 * == NULL): grad_loc [N,3] -> grad_offsets [N,2], grad_points [N,2] (the same values: both enter as points + offsets) and
 * grad_depth [N].  K, points, offsets, pad, depth: the forward's inputs (depth = its depth_in).  Each output may be NULL, not
 * all three.  No gradient flows to K or pad (the calibration and the padding are constants in the reference). */
int dcd_dgde_locate_bwd(const float* K, const float* points, const float* offsets, const float* pad, const float* depth,
                        const float* grad_loc, int64_t N, float down_ratio, float* grad_offsets, float* grad_points,
                        float* grad_depth, void* stream);

/* Backward of dcd_dgde_depth_ensemble_fwd, same inputs and scalars.  Upstream gradients grad_kp_depths [N,3], grad_depth [N],
 * grad_depth_error [N], grad_scores_out [N]: each may be NULL (no gradient from that output), not all four; any of the last
 * three needs log_unc_kp (and log_unc_direct when direct != NULL), grad_scores_out needs scores.  Outputs, each may be NULL,
 * not all: grad_kp10 [N,10,2] (v column; the u column is exactly 0), grad_dims [N,3] (h column; l and w exactly 0),
 * grad_direct [N], grad_log_unc_direct [N] (both need direct != NULL), grad_log_unc_kp [N,3], grad_scores [N].  argmax has no
 * gradient, K none (calibration).  Masks as torch: relu passes where height > 0, clamps are inclusive; a NaN score product
 * (zeroed by the forward) passes no gradient.  Height NaNs are outside the contract (the forward's relu maps them to 0). */
int dcd_dgde_depth_ensemble_bwd(const float* kp10, const float* dims, const float* K, const float* direct,
                                const float* log_unc_direct, const float* log_unc_kp, const float* scores, int64_t N,
                                float down_ratio, float eps, float lo, float hi, const float* grad_kp_depths,
                                const float* grad_depth, const float* grad_depth_error, const float* grad_scores_out,
                                float* grad_kp10, float* grad_dims, float* grad_direct, float* grad_log_unc_direct,
                                float* grad_log_unc_kp, float* grad_scores, void* stream);

/* GMW validation (GMW/main.py:542-547): move a detector location [N,3] along its viewing ray through the box centre to
 * the GMW depth: scale = pred_depth / z; y -= h/2; loc *= scale; y += h/2  (dim [N,3] = (h,w,l) there). */
int dcd_gmw_ray_rescale_fwd(const float* raw_location, const float* pred_depth, const float* dim, int64_t N,
                            float* pred_location, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Edge solve, backward (the autograd of decode_pairs_kpts_depth, consumers detector_loss.py:188-214,
 * :388-396).  grad_depth is [N,k] when idx != NULL (gradient of the selected depths) or [N,E] when
 * idx == NULL; grad_mean [N] (may be NULL) is the gradient of depth_mean and is spread as g/k (or g/E).
 * At least one of grad_depth / grad_mean must be given.  Outputs: grad_kps [N,n,2] (the u column is
 * exactly 0: only the vertical constraint is used), grad_kps3d [N,n,3].  Clamp masks are inclusive like
 * torch.clamp; no gradient flows to rot or K (GT yaw / calibration in the reference).  Deterministic
 * (per-keypoint gather, no atomics).
 */
int dcd_edge_solve_bwd(const float* kps, const float* kps3d, const float* rot, const float* K,
                       int64_t N, int n, float lo, float hi, int flags,
                       const int64_t* idx, int k, const float* grad_depth, const float* grad_mean,
                       float* grad_kps, float* grad_kps3d, void* stream);

/* ------------------------------------------------------------------------------------------------
 * GMW edge weights.  Replaces GMW.forward's reg_weights (GMW/model/model.py:195-207): edge_expand
 * (:153-163), the two edge-feature nets (yi2018cvpr/model.py:63-67, ops.py:7-19,125-131), L2
 * normalisation (:176-177), the DIAGONAL of pairwiseL2Dist (:28-35, same expansion and association)
 * and graph_extract (:165-168):  reg_weights[N,E] = 1 / sqrt(max((|c|^2 - 2 a.c) + |a|^2, 1e-30)).
 *
 * params4 / params6: packed FP32 parameter blobs of FeatureExtractor4d / 6d, layout (Cin = 4 or 6):
 *     W_in^T [Cin][128], b_in [128], then per block k<depth: Wp^T [128][128], bp [128], W1^T, b1, W2^T, b2
 * (transposed = [in][out]; dcd_b200.weights.pack_state_dict builds it from the reference state_dict).
 * kpts2d [N,n,2] normalised image coordinates, kpts3d [N,n,3].
 * save != 0 keeps the per-block activations in the workspace for dcd_gmw_weights_bwd (layer-wise kernels, one
 * launch per segment between context norms).  save == 0 and n <= 73 (E <= 2688): the whole network runs in ONE
 * persistent kernel with the activations held on chip (groups of 8 co-resident CTAs per object; cooperative launch,
 * so the device must not be oversubscribed by kernels that wait on this stream); larger n fall back to the
 * layer-wise kernels.  Results of the two forms agree to FP32 rounding (the context-norm partial statistics are
 * merged in a different order).  Environment: DCD_B200_LAYERWISE=1 forces the layer-wise kernels.
 * feat4 / feat6 (may be NULL): final un-normalised edge features, [N,128,E] channel-major.
 */
size_t dcd_gmw_param_count(int cin, int depth);
size_t dcd_gmw_workspace_bytes(int64_t N, int n, int depth, int save);
int dcd_gmw_weights_fwd(const float* kpts2d, const float* kpts3d, const float* params4, const float* params6,
                        int64_t N, int n, int depth, int save, float* reg_weights,
                        float* feat4, float* feat6, void* workspace, size_t workspace_bytes, void* stream);

/* Correspondence branch of GMW, forward only (SURVEY 8f row N1): from the final features feat4 / feat6 [N,128,E] of
 * dcd_gmw_weights_fwd:  M = pairwiseL2Dist(normalise(f4), normalise(f6)) (GMW/model/model.py:17-36,176-180),
 * P = Sinkhorn(M; r = c = 1/E, lambda, tolerance, max_iterations) (GMW/lib/optimal_transport.py:52-72, model.py:186-191).
 * Outputs (each may be NULL): P [N,E,E], u / v [N,E] (P = diag(u) K diag(v), K = exp(-lambda min(M,5))),
 * sums [N,2] = (sum P, trace P) — correspondenceLoss(P, eye) = mean over objects of sum - 2 trace (lib/losses.py:22-26,
 * 115-119; GMW/main.py:456-457,526-527).  The workspace holds K (4 E^2 bytes per object); N <= 65535. */
size_t dcd_gmw_transport_workspace_bytes(int64_t N, int n);
int dcd_gmw_transport_fwd(const float* feat4, const float* feat6, int64_t N, int n, float lambda, float tolerance,
                          int max_iterations, float* P, float* u, float* v, float* sums, void* workspace,
                          size_t workspace_bytes, void* stream);

/* Backward of dcd_gmw_transport_fwd (RegularisedTransportFn.backward, GMW/lib/optimal_transport.py:75-128,184-222, then
 * the autograd of pairwiseL2Dist, GMW/model/model.py:17-36): from grad_P [N,E,E] = dL/dP to the gradient w.r.t. the
 * L2-NORMALISED features, grad_nfeat4 / grad_nfeat6 [N,128,E] (feed them to dcd_gmw_weights_bwd).  P, u, v: outputs of the
 * forward call; feat4 / feat6: its inputs.  The reference's E x E Cholesky + inverse + three E^3 products are replaced by
 * ONE matrix-free conjugate-gradient solve of the same SPD system (two passes over P per iteration; relative residual
 * cg_tolerance, at most max_cg_iterations, typically 6-20) — see csrc/gmw_transport_bwd.cu.  cg_info (may be NULL) [N,8]:
 * (final |r|^2, initial |r|^2, converged flag, iterations, -, -, -, -) per object. */
size_t dcd_gmw_transport_bwd_workspace_bytes(int64_t N, int n);
int dcd_gmw_transport_bwd(const float* feat4, const float* feat6, const float* P, const float* u, const float* v,
                          const float* grad_P, int64_t N, int n, float lambda, int max_cg_iterations, float cg_tolerance,
                          float* grad_nfeat4, float* grad_nfeat6, float* cg_info, void* workspace, size_t workspace_bytes,
                          void* stream);

/* The same backward for a loss on the plan's two sums only, L(sum P, trace P) (correspondenceLoss, lib/losses.py:115-119),
 * without any E x E tensor besides the forward's K.  dL/dP is then alpha 11^T + beta I per object, with grad_terms [N,2] =
 * (alpha, beta) = (dL/d sum P, dL/d trace P), formed in registers; the plan is rebuilt entry by entry from K, u and v as
 * (u_i K_ij) v_j, the forward's own two roundings.  With the same plan and the same dL/dP values this gives grad_nfeat4 /
 * grad_nfeat6 and cg_info bit-identical to dcd_gmw_transport_bwd with a dense grad_P.
 * fwd_workspace: the workspace of the dcd_gmw_transport_fwd call (same N, n, lambda; P may have been NULL there), which holds
 * K; nothing may be written to it in between.  u, v: that call's u / v outputs; feat4 / feat6: its inputs.  The workspace is
 * sized by dcd_gmw_transport_bwd_workspace_bytes.  N >= 1. */
int dcd_gmw_transport_terms_bwd(const float* feat4, const float* feat6, const void* fwd_workspace, size_t fwd_workspace_bytes,
                                const float* u, const float* v, const float* grad_terms, int64_t N, int n, float lambda,
                                int max_cg_iterations, float cg_tolerance, float* grad_nfeat4, float* grad_nfeat6, float* cg_info,
                                void* workspace, size_t workspace_bytes, void* stream);

/* Backward of dcd_gmw_weights_fwd w.r.t. the parameters (autograd of GMW/main.py:465).
 * workspace: the one filled by the forward call with save=1 (same N, n, depth).  grad_reg_weights [N,E] (reg path) and/or
 * grad_nfeat4 / grad_nfeat6 [N,128,E] (gradient w.r.t. the normalised final features, from dcd_gmw_transport_bwd: cls path);
 * each may be NULL, not all three.
 * grad_params4 / grad_params6: same layout as the parameter blobs, OVERWRITTEN with the sum over the N
 * objects.  Deterministic (per-CTA partial sums reduced in a fixed order).
 */
size_t dcd_gmw_bwd_scratch_bytes(int64_t N, int n, int depth);
int dcd_gmw_weights_bwd(const float* kpts2d, const float* kpts3d, const float* params4, const float* params6,
                        int64_t N, int n, int depth, const float* grad_reg_weights,
                        const float* grad_nfeat4, const float* grad_nfeat6,
                        float* grad_params4, float* grad_params6,
                        void* workspace, size_t workspace_bytes, void* scratch, size_t scratch_bytes,
                        void* stream);

/* Backward of dcd_gmw_weights_fwd w.r.t. the keypoints, from the scratch that dcd_gmw_weights_bwd just filled
 * (same N, n, depth, params; same stream; nothing written to the scratch in between).  grad_kpts2d [N,n,2],
 * grad_kpts3d [N,n,3], each may be NULL (not both), OVERWRITTEN.  Deterministic.
 * The chain below the first residual block is linear: dF = W_in^T-contraction of dL/d(conv_in output) per edge
 * (GMW/model/yi2018cvpr/model.py:63), then the backward of edge_expand (GMW/model/model.py:153-163) as a per-keypoint
 * gather over the n-1 incident edges (fixed order, no atomics).  dcd_gmw_weights_bwd's own outputs do not change. */
int dcd_gmw_kpts_bwd(const float* params4, const float* params6, int64_t N, int n, int depth,
                     void* scratch, size_t scratch_bytes, float* grad_kpts2d, float* grad_kpts3d, void* stream);

/* ------------------------------------------------------------------------------------------------
 * GMW weighted aggregation.  Replaces the forward of compute_reg_loss (GMW/main.py:364-371):
 * depth_out[N] = sum_r softmax_r(reg_weights[idx[r]]) * depths[idx[r]].  depths is [N,E] when
 * depths_are_selected == 0 (gathered through idx) or already-gathered [N,k] otherwise.
 * probs [N,k] (may be NULL) receives the softmax for the backward.
 */
int dcd_gmw_aggregate_fwd(const float* reg_weights, const float* depths, const int64_t* idx,
                          int64_t N, int64_t E, int k, int depths_are_selected,
                          float* depth_out, float* probs, void* stream);

/* Backward: grad_reg_weights [N,E] (dense, zero outside idx; OVERWRITTEN) = g * p_r * (z_r - depth_out),
 * grad_depths (may be NULL; [N,E] dense or [N,k] as in the forward) = g * p_r.  An edge that idx selects at several slots
 * receives the sum over those slots (torch.gather's scatter_add backward), summed in ascending slot order: deterministic, no
 * floating-point atomics; with distinct indices each edge's value is its one slot's.  An index outside [0, E) is clamped to
 * 0 or E - 1 like the forward (and adds to that edge).  k > DCD_AGG_BWD_MAX_K returns DCD_E_UNSUPPORTED.
 */
#define DCD_AGG_BWD_MAX_K (1 << 22)
int dcd_gmw_aggregate_bwd(const float* reg_weights, const float* depths, const int64_t* idx,
                          int64_t N, int64_t E, int k, int depths_are_selected,
                          const float* grad_depth_out, float* grad_reg_weights, float* grad_depths,
                          void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused GMW inference: compute_z -> GMW.forward -> softmax-weighted depth (GMW/main.py:524-533) for N
 * objects, processed in chunks so that the workspace stays bounded: depth_out [N].
 * lo/hi are compute_z's clamp (0.1, 80), k its 1500.  idx_out [N,k] int64 and reg_weights [N,E] may be NULL.
 */
size_t dcd_gmw_depth_workspace_bytes(int64_t N, int n, int depth, int64_t chunk);
int dcd_gmw_depth_fwd(const float* kpts2d, const float* kpts3d, const float* rot,
                      const float* params4, const float* params6,
                      int64_t N, int n, int depth, int k, float lo, float hi, int64_t chunk,
                      float* depth_out, int64_t* idx_out, float* reg_weights,
                      void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * DGDE detections refined by GMW in one stream-ordered chain (SURVEY 8f row N3, on-GPU half): the regression map to the
 * GMW-rescaled 3D locations, replacing the gen_data_infer.json hand-off (DGDE/engine/inference.py:59-84 -> GMW/main.py:
 * 524-547).  Launches, no host synchronisation, no allocation:
 *   1. the dcd_dgde_frame_fwd kernel over all N objects with its fixed scalars (lo, hi = 2, 80; DCD_NORMALISE_2D |
 *      DCD_SUB_B3; down_ratio 4) -> dgde_depth [N], dgde_location [N,3] (with + h/2), and GMW's inputs for keypoints
 *      0 .. 72: gmw_kpts [N,73,2] = ((u - K[0][2]) / K[0][0], (v - K[1][2]) / K[1][1]) (FP32, one rounding each) and
 *      kps3d [N,73,3];
 *   2. per chunk of <= `chunk` objects, dcd_gmw_depth_fwd's sequence on those inputs with lo, hi = 0.1, 80, no flags and
 *      the DGDE yaw `rot` -> gmw_depth [N]; its aggregate also writes location [N,3] = the GMW ray rescale
 *      (dcd_gmw_ray_rescale_fwd's operations) of dgde_location to gmw_depth with h = dims[:, 1].
 * Every output is bit-identical to dcd_dgde_frame_fwd -> normalisation -> dcd_gmw_depth_fwd (same chunk) ->
 * dcd_gmw_ray_rescale_fwd(dim = dims[:, (1,2,0)]).  Arguments as dcd_dgde_frame_fwd and dcd_gmw_depth_fwd; dims [N,3] (l,h,w)
 * is required; n >= DCD_GMW_KPTS; 1 <= k <= 2628.  gmw_kpts, kps3d, idx_out [N,k] int64 (the selected edges) may be NULL
 * (the workspace holds them then).  A position outside the map yields NaN outputs for that object only. */
size_t dcd_dgde_gmw_refine_workspace_bytes(int64_t N, int n, int depth, int64_t chunk);
int dcd_dgde_gmw_refine_fwd(const float* feature_maps, const int64_t* index, const int32_t* batch_idx, int64_t B, int C, int H,
                            int W, int ch_kpts2d, int ch_kpts3d, int ch_offset3d, const float* rot, const float* K, const float* pad,
                            const float* dims, const float* params4, const float* params6, int64_t N, int n, int depth, int k,
                            int64_t chunk, float* dgde_depth, float* dgde_location, float* gmw_depth, float* location,
                            float* gmw_kpts, float* kps3d, int64_t* idx_out, void* workspace, size_t workspace_bytes,
                            void* stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* DCD_B200_H_ */
