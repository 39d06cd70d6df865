// extern "C" entry points of libdcd_b200.so: argument validation, workspace carving, kernel launches.
// See include/dcd_b200.h for the contract of every function.
#include "gmw_mlp.cuh"

namespace dcd {
int launch_edge_solve_fwd(const float*, const float*, const float*, const float*, int64_t, int, float, float, int,
                          float*, float*, cudaStream_t);
int launch_edge_select(const float*, const float*, const float*, const float*, const uint8_t*, int64_t, int, int,
                       float, float, int, int64_t*, float*, float*, float*, cudaStream_t);
int launch_edge_solve_bwd(const float*, const float*, const float*, const float*, int64_t, int, float, float, int,
                          const int64_t*, int, const float*, const float*, float*, float*, cudaStream_t);
int launch_gmw_aggregate_fwd(const float*, const float*, const int64_t*, int64_t, int64_t, int, int, float*, float*,
                             cudaStream_t);
int launch_gmw_aggregate_bwd(const float*, const float*, const int64_t*, int64_t, int64_t, int, int, const float*,
                             float*, float*, cudaStream_t);
int launch_gmw_weights_fwd(const float*, const float*, const float*, const float*, int64_t, int, int, int, float*,
                           float*, float*, float*, cudaStream_t);
int launch_dgde_locate(const float*, const float*, const float*, const float*, const float*, const float*, const float*,
                       const float*, const float*, int64_t, int, float, float, int, float, float*, float*, cudaStream_t);
int launch_dgde_frame(const float*, const int64_t*, const int32_t*, int, int, int, int, int, int, const float*, const float*,
                      const float*, const float*, int64_t, int, float, float, int, float, float*, float*, float*, float*, float*, float*,
                      cudaStream_t);
int launch_gmw_aggregate_rescale_fwd(const float*, const float*, const int64_t*, int64_t, int64_t, int, int, float*, const float*,
                                     const float*, float*, cudaStream_t);
int launch_dgde_depth_ensemble(const float*, const float*, const float*, const float*, const float*, const float*, const float*,
                               int64_t, float, float, float, float, float*, float*, float*, int64_t*, float*, cudaStream_t);
int launch_gmw_ray_rescale(const float*, const float*, const float*, int64_t, float*, cudaStream_t);
int launch_poi_gather(const float*, const int64_t*, int64_t, int64_t, int, int64_t, float*, cudaStream_t);
int launch_poi_gather_bwd(const float*, const int64_t*, int64_t, int64_t, int, int64_t, float*, cudaStream_t);
int launch_dgde_locate_bwd(const float*, const float*, const float*, const float*, const float*, const float*, int64_t, float, float*,
                           float*, float*, cudaStream_t);
int launch_dgde_depth_ensemble_bwd(const float*, const float*, const float*, const float*, const float*, const float*, const float*,
                                   int64_t, float, float, float, float, const float*, const float*, const float*, const float*, float*,
                                   float*, float*, float*, float*, float*, cudaStream_t);
size_t gmw_transport_workspace_bytes(int64_t N, int E);
int launch_gmw_transport_fwd(const float*, const float*, int64_t, int, float, float, int, float*, float*, float*, float*, void*,
                             cudaStream_t);
size_t gmw_bwd_scratch_floats(int64_t N, int n, int depth);
size_t tc_weight_image_bytes(int depth);
int launch_gmw_weights_bwd(const float*, const float*, const float*, const float*, int64_t, int, int, const float*,
                           const float*, const float*, float*, float*, float*, float*, cudaStream_t);
int launch_gmw_kpts_bwd(const float*, const float*, int64_t, int, int, float*, float*, float*, cudaStream_t);
size_t gmw_transport_bwd_workspace_bytes(int64_t N, int E);
int launch_gmw_transport_bwd(const float*, const float*, const float*, const float*, const float*, const float*, int64_t, int, float,
                             int, float, float*, float*, float*, void*, cudaStream_t);
const float* gmw_transport_workspace_k(const void*);
int launch_gmw_transport_terms_bwd(const float*, const float*, const float*, const float*, const float*, const float*, int64_t, int,
                                   float, int, float, float*, float*, float*, void*, cudaStream_t);
}  // namespace dcd

using namespace dcd;

namespace {
inline bool bad_n(int n) { return n < 2 || n > DCD_MAX_KPTS; }
inline bool misaligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) != 0; }
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// The chunk loop of dcd_gmw_depth_fwd (workspace laid out by dcd_gmw_depth_workspace_bytes for `chunk` <= N objects): per
// chunk the top-k edge selection, the edge MLP and the softmax aggregate.  raw_loc != NULL (with dims, loc_out; all [N,3]):
// the aggregate also moves raw_loc along its viewing ray to the weighted depth (dcd_dgde_gmw_refine_fwd).
int gmw_depth_chunks(const float* kpts2d, const float* kpts3d, const float* rot, const float* params4, const float* params6,
                     int64_t N, int n, int depth, int k, float lo, float hi, int64_t chunk, float* depth_out, int64_t* idx_out,
                     float* reg_weights, void* workspace, const float* raw_loc, const float* dims, float* loc_out,
                     cudaStream_t st) {
    const int64_t E = num_edges(n);
    unsigned char* p = static_cast<unsigned char*>(workspace);
    const size_t mlp_bytes = align_up(dcd_gmw_workspace_bytes(chunk, n, depth, 0), 256);
    float* mlp_ws = reinterpret_cast<float*>(p);
    p += mlp_bytes;
    int64_t* idx_ws = reinterpret_cast<int64_t*>(p);
    p += align_up((size_t)chunk * E * sizeof(int64_t), 256);
    float* zsel_ws = reinterpret_cast<float*>(p);
    p += align_up((size_t)chunk * E * sizeof(float), 256);
    float* regw_ws = reinterpret_cast<float*>(p);
    for (int64_t c0 = 0; c0 < N; c0 += chunk) {
        const int64_t nc = (N - c0 < chunk) ? N - c0 : chunk;
        const float* k2 = kpts2d + c0 * n * 2;
        const float* k3 = kpts3d + c0 * n * 3;
        int64_t* idx = idx_out ? idx_out + c0 * k : idx_ws;
        float* rw = reg_weights ? reg_weights + c0 * E : regw_ws;
        int rc = launch_edge_select(k2, k3, rot + c0, nullptr, nullptr, nc, n, k, lo, hi, 0, idx, zsel_ws, nullptr,
                                    nullptr, st);
        if (rc != DCD_OK) return rc;
        rc = launch_gmw_weights_fwd(k2, k3, params4, params6, nc, n, depth, 0, rw, nullptr, nullptr, mlp_ws, st);
        if (rc != DCD_OK) return rc;
        rc = raw_loc ? launch_gmw_aggregate_rescale_fwd(rw, zsel_ws, idx, nc, E, k, 1, depth_out + c0, raw_loc + c0 * 3,
                                                        dims + c0 * 3, loc_out + c0 * 3, st)
                     : launch_gmw_aggregate_fwd(rw, zsel_ws, idx, nc, E, k, 1, depth_out + c0, nullptr, st);
        if (rc != DCD_OK) return rc;
    }
    return DCD_OK;
}

// fixed scalars of the detector head's frame epilogue (frame_depths_from_map) and of compute_z inside the refine chain
constexpr float kDgdeLo = 2.f, kDgdeHi = 80.f, kDownRatio = 4.f, kGmwLo = 0.1f, kGmwHi = 80.f;
}  // namespace

extern "C" {

int dcd_version(void) { return DCD_ABI_VERSION; }

const char* dcd_strerror(int rc) {
    switch (rc) {
        case DCD_OK: return "ok";
        case DCD_E_INVALID: return "invalid argument";
        case DCD_E_WORKSPACE: return "workspace too small or misaligned";
        case DCD_E_LAUNCH: return "CUDA kernel launch failed";
        case DCD_E_UNSUPPORTED: return "shape not supported by the sm_100a kernels";
        case DCD_E_DEVICE: return "device is not sm_100";
        default: return "unknown dcd error";
    }
}

int dcd_edge_solve_fwd(const float* kps, const float* kps3d, const float* rot, const float* K, int64_t N, int n,
                       float lo, float hi, int flags, float* depth_edges, float* depth_mean, void* stream) {
    if (N < 0 || bad_n(n)) return DCD_E_INVALID;
    if (N == 0) return DCD_OK;
    if (!kps || !kps3d || !rot || (!depth_edges && !depth_mean)) return DCD_E_INVALID;
    if ((flags & (DCD_NORMALISE_2D | DCD_SUB_B3)) && !K) return DCD_E_INVALID;
    if (misaligned(kps, 8)) return DCD_E_INVALID;
    return launch_edge_solve_fwd(kps, kps3d, rot, K, N, n, lo, hi, flags, depth_edges, depth_mean, (cudaStream_t)stream);
}

size_t dcd_edge_select_workspace_bytes(int64_t, int) { return 0; }

int dcd_edge_select_fwd(const float* kps, const float* kps3d, const float* rot, const float* K,
                        const uint8_t* kpt_mask, int64_t N, int n, int k, float lo, float hi, int flags,
                        int64_t* idx_out, float* depth_sel, float* mask_sel, float* depth_mean, void* stream) {
    if (N < 0 || bad_n(n)) return DCD_E_INVALID;
    const int64_t E = num_edges(n);
    if (k < 1 || k > E) return DCD_E_INVALID;
    if (N == 0) return DCD_OK;
    if (!kps || !kps3d || !rot || !idx_out) return DCD_E_INVALID;
    if ((flags & (DCD_NORMALISE_2D | DCD_SUB_B3)) && !K) return DCD_E_INVALID;
    if (mask_sel && !kpt_mask) return DCD_E_INVALID;
    if (misaligned(kps, 8)) return DCD_E_INVALID;
    return launch_edge_select(kps, kps3d, rot, K, kpt_mask, N, n, k, lo, hi, flags, idx_out, depth_sel, mask_sel,
                              depth_mean, (cudaStream_t)stream);
}

int dcd_edge_solve_bwd(const float* kps, const float* kps3d, const float* rot, const float* K, int64_t N, int n,
                       float lo, float hi, int flags, const int64_t* idx, int k, const float* grad_depth,
                       const float* grad_mean, float* grad_kps, float* grad_kps3d, void* stream) {
    if (N < 0 || bad_n(n)) return DCD_E_INVALID;
    const int64_t E = num_edges(n);
    if (idx && (k < 1 || k > E)) return DCD_E_INVALID;
    if (N == 0) return DCD_OK;
    if (!kps || !kps3d || !rot || !grad_kps || !grad_kps3d || (!grad_depth && !grad_mean)) return DCD_E_INVALID;
    if ((flags & (DCD_NORMALISE_2D | DCD_SUB_B3)) && !K) return DCD_E_INVALID;
    if (misaligned(kps, 8) || misaligned(grad_kps, 8)) return DCD_E_INVALID;
    return launch_edge_solve_bwd(kps, kps3d, rot, K, N, n, lo, hi, flags, idx, k, grad_depth, grad_mean, grad_kps,
                                 grad_kps3d, (cudaStream_t)stream);
}

int dcd_dgde_locate_fwd(const float* kpts_off, const float* kps3d, const float* rot, const float* K, const float* points,
                        const float* offsets, const float* pad, const float* dims, const float* depth_in, int64_t N, int n,
                        float lo, float hi, int flags, float down_ratio, float* depth_out, float* locations, void* stream) {
    if (N < 0) return DCD_E_INVALID;
    if (kpts_off && bad_n(n)) return DCD_E_INVALID;
    if (N == 0) return DCD_OK;
    if (!K || !points || !offsets || !pad || (!depth_out && !locations)) return DCD_E_INVALID;
    if (kpts_off ? (!kps3d || !rot) : !depth_in) return DCD_E_INVALID;
    return launch_dgde_locate(kpts_off, kps3d, rot, K, points, offsets, pad, dims, depth_in, N, kpts_off ? n : 2, lo, hi, flags,
                              down_ratio, depth_out, locations, (cudaStream_t)stream);
}

int dcd_dgde_frame_fwd(const float* feature_maps, const int64_t* index, const int32_t* batch_idx, int64_t B, int C, int H, int W,
                       int ch_kpts2d, int ch_kpts3d, int ch_offset3d, const float* rot, const float* K, const float* pad,
                       const float* dims, int64_t N, int n, float lo, float hi, int flags, float down_ratio, float* depth_out,
                       float* locations, float* kpts_img_out, float* kps3d_out, void* stream) {
    if (N < 0 || B < 1 || C < 1 || H < 1 || W < 1 || bad_n(n)) return DCD_E_INVALID;
    if (ch_kpts2d < 0 || ch_kpts2d + 2 * n > C || ch_kpts3d < 0 || ch_kpts3d + 3 * n > C || ch_offset3d < 0 || ch_offset3d + 2 > C)
        return DCD_E_INVALID;
    if (N == 0) return DCD_OK;
    if (!feature_maps || !index || !rot || !K || !pad || (!depth_out && !locations)) return DCD_E_INVALID;
    if (B > 1 && !batch_idx) return DCD_E_INVALID;
    return launch_dgde_frame(feature_maps, index, batch_idx, C, H, W, ch_kpts2d, ch_kpts3d, ch_offset3d, rot, K, pad, dims, N, n, lo,
                             hi, flags, down_ratio, depth_out, locations, kpts_img_out, kps3d_out, nullptr, nullptr,
                             (cudaStream_t)stream);
}

int dcd_dgde_depth_ensemble_fwd(const float* kp10, const float* dims, const float* K, const float* direct,
                                const float* log_unc_direct, const float* log_unc_kp, const float* scores, int64_t N,
                                float down_ratio, float eps, float lo, float hi, float* kp_depths, float* depth,
                                float* depth_error, int64_t* argmax, float* scores_out, void* stream) {
    if (N < 0) return DCD_E_INVALID;
    if (N == 0) return DCD_OK;
    if (!kp10 || !dims || !K) return DCD_E_INVALID;
    const bool ensemble = depth || depth_error || argmax || scores_out;
    if (!ensemble && !kp_depths) return DCD_E_INVALID;
    if (ensemble && (!log_unc_kp || (direct && !log_unc_direct))) return DCD_E_INVALID;
    if (scores_out && !scores) return DCD_E_INVALID;
    return launch_dgde_depth_ensemble(kp10, dims, K, direct, log_unc_direct, log_unc_kp, scores, N, down_ratio, eps, lo, hi,
                                      kp_depths, depth, depth_error, argmax, scores_out, (cudaStream_t)stream);
}

int dcd_poi_gather_fwd(const float* feature_maps, const int64_t* index, int64_t B, int64_t K, int C, int64_t HW, float* out,
                       void* stream) {
    if (B < 0 || K < 0 || C < 1 || HW < 1) return DCD_E_INVALID;
    if (B == 0 || K == 0) return DCD_OK;
    if (!feature_maps || !index || !out) return DCD_E_INVALID;
    return launch_poi_gather(feature_maps, index, B, K, C, HW, out, (cudaStream_t)stream);
}

int dcd_poi_gather_bwd(const float* grad_out, const int64_t* index, int64_t B, int64_t K, int C, int64_t HW, float* grad_maps,
                       void* stream) {
    if (B < 0 || K < 0 || C < 1 || HW < 1) return DCD_E_INVALID;
    if (K > DCD_POI_BWD_MAX_K) return DCD_E_UNSUPPORTED;
    if (B == 0) return DCD_OK;
    if (!grad_maps || (K > 0 && (!grad_out || !index))) return DCD_E_INVALID;
    return launch_poi_gather_bwd(grad_out, index, B, K, C, HW, grad_maps, (cudaStream_t)stream);
}

int dcd_dgde_locate_bwd(const float* K, const float* points, const float* offsets, const float* pad, const float* depth,
                        const float* grad_loc, int64_t N, float down_ratio, float* grad_offsets, float* grad_points,
                        float* grad_depth, void* stream) {
    if (N < 0) return DCD_E_INVALID;
    if (N == 0) return DCD_OK;
    if (!K || !points || !offsets || !pad || !depth || !grad_loc) return DCD_E_INVALID;
    if (!grad_offsets && !grad_points && !grad_depth) return DCD_E_INVALID;
    return launch_dgde_locate_bwd(K, points, offsets, pad, depth, grad_loc, N, down_ratio, grad_offsets, grad_points, grad_depth,
                                  (cudaStream_t)stream);
}

int dcd_dgde_depth_ensemble_bwd(const float* kp10, const float* dims, const float* K, const float* direct,
                                const float* log_unc_direct, const float* log_unc_kp, const float* scores, int64_t N,
                                float down_ratio, float eps, float lo, float hi, const float* grad_kp_depths,
                                const float* grad_depth, const float* grad_depth_error, const float* grad_scores_out,
                                float* grad_kp10, float* grad_dims, float* grad_direct, float* grad_log_unc_direct,
                                float* grad_log_unc_kp, float* grad_scores, void* stream) {
    if (N < 0) return DCD_E_INVALID;
    if (N == 0) return DCD_OK;
    if (!kp10 || !dims || !K) return DCD_E_INVALID;
    const bool ensemble = grad_depth || grad_depth_error || grad_scores_out;
    if (!ensemble && !grad_kp_depths) return DCD_E_INVALID;
    if (!grad_kp10 && !grad_dims && !grad_direct && !grad_log_unc_direct && !grad_log_unc_kp && !grad_scores) return DCD_E_INVALID;
    if (ensemble && (!log_unc_kp || (direct && !log_unc_direct))) return DCD_E_INVALID;
    if (grad_scores_out && !scores) return DCD_E_INVALID;
    if ((grad_direct || grad_log_unc_direct) && !direct) return DCD_E_INVALID;
    return launch_dgde_depth_ensemble_bwd(kp10, dims, K, direct, log_unc_direct, log_unc_kp, scores, N, down_ratio, eps, lo, hi,
                                          grad_kp_depths, grad_depth, grad_depth_error, grad_scores_out, grad_kp10, grad_dims,
                                          grad_direct, grad_log_unc_direct, grad_log_unc_kp, grad_scores, (cudaStream_t)stream);
}

int dcd_gmw_ray_rescale_fwd(const float* raw_location, const float* pred_depth, const float* dim, int64_t N,
                            float* pred_location, void* stream) {
    if (N < 0) return DCD_E_INVALID;
    if (N == 0) return DCD_OK;
    if (!raw_location || !pred_depth || !dim || !pred_location) return DCD_E_INVALID;
    return launch_gmw_ray_rescale(raw_location, pred_depth, dim, N, pred_location, (cudaStream_t)stream);
}

size_t dcd_gmw_transport_workspace_bytes(int64_t N, int n) {
    if (N <= 0 || bad_n(n)) return 0;
    return gmw_transport_workspace_bytes(N, (int)num_edges(n));
}

int dcd_gmw_transport_fwd(const float* feat4, const float* feat6, int64_t N, int n, float lambda, float tolerance,
                          int max_iterations, float* P, float* u, float* v, float* sums, void* workspace,
                          size_t workspace_bytes, void* stream) {
    if (N < 0 || bad_n(n) || max_iterations < 0 || !(lambda > 0.f)) return DCD_E_INVALID;
    if (N == 0) return DCD_OK;
    if (!feat4 || !feat6 || (!P && !u && !v && !sums)) return DCD_E_INVALID;
    if (N > 65535) return DCD_E_UNSUPPORTED;                  // objects map to gridDim.y / .z; K alone is 27.6 MB per object
    if (misaligned(workspace, 256) || workspace_bytes < dcd_gmw_transport_workspace_bytes(N, n)) return DCD_E_WORKSPACE;
    return launch_gmw_transport_fwd(feat4, feat6, N, (int)num_edges(n), lambda, tolerance, max_iterations, P, u, v, sums, workspace,
                                    (cudaStream_t)stream);
}

size_t dcd_gmw_transport_bwd_workspace_bytes(int64_t N, int n) {
    if (N <= 0 || bad_n(n)) return 0;
    return gmw_transport_bwd_workspace_bytes(N, (int)num_edges(n));
}

int dcd_gmw_transport_bwd(const float* feat4, const float* feat6, const float* P, const float* u, const float* v,
                          const float* grad_P, int64_t N, int n, float lambda, int max_cg_iterations, float cg_tolerance,
                          float* grad_nfeat4, float* grad_nfeat6, float* cg_info, void* workspace, size_t workspace_bytes,
                          void* stream) {
    if (N < 0 || bad_n(n) || max_cg_iterations < 1 || !(lambda > 0.f) || !(cg_tolerance >= 0.f)) return DCD_E_INVALID;
    if (N == 0) return DCD_OK;
    if (!feat4 || !feat6 || !P || !u || !v || !grad_P || !grad_nfeat4 || !grad_nfeat6) return DCD_E_INVALID;
    if (N > 65535) return DCD_E_UNSUPPORTED;
    if (misaligned(P, 16) || misaligned(grad_P, 16)) return DCD_E_INVALID;
    if (misaligned(workspace, 256) || workspace_bytes < dcd_gmw_transport_bwd_workspace_bytes(N, n)) return DCD_E_WORKSPACE;
    return launch_gmw_transport_bwd(feat4, feat6, P, u, v, grad_P, N, (int)num_edges(n), lambda, max_cg_iterations, cg_tolerance,
                                    grad_nfeat4, grad_nfeat6, cg_info, workspace, (cudaStream_t)stream);
}

int dcd_gmw_transport_terms_bwd(const float* feat4, const float* feat6, const void* fwd_workspace, size_t fwd_workspace_bytes,
                                const float* u, const float* v, const float* grad_terms, int64_t N, int n, float lambda,
                                int max_cg_iterations, float cg_tolerance, float* grad_nfeat4, float* grad_nfeat6, float* cg_info,
                                void* workspace, size_t workspace_bytes, void* stream) {
    if (N < 1 || bad_n(n) || max_cg_iterations < 1 || !(lambda > 0.f) || !(cg_tolerance >= 0.f)) return DCD_E_INVALID;
    if (!feat4 || !feat6 || !fwd_workspace || !u || !v || !grad_terms || !grad_nfeat4 || !grad_nfeat6 || !workspace)
        return DCD_E_INVALID;
    if (N > 65535) return DCD_E_UNSUPPORTED;
    if (misaligned(fwd_workspace, 256) || fwd_workspace_bytes < dcd_gmw_transport_workspace_bytes(N, n)) return DCD_E_WORKSPACE;
    if (misaligned(workspace, 256) || workspace_bytes < dcd_gmw_transport_bwd_workspace_bytes(N, n)) return DCD_E_WORKSPACE;
    return launch_gmw_transport_terms_bwd(feat4, feat6, gmw_transport_workspace_k(fwd_workspace), u, v, grad_terms, N,
                                          (int)num_edges(n), lambda, max_cg_iterations, cg_tolerance, grad_nfeat4, grad_nfeat6,
                                          cg_info, workspace, (cudaStream_t)stream);
}

size_t dcd_gmw_param_count(int cin, int depth) { return (size_t)blob_size(cin, depth); }

size_t dcd_gmw_workspace_bytes(int64_t N, int n, int depth, int save) {
    if (N <= 0 || bad_n(n) || depth < 1) return 0;
    // activations + context-norm statistics, then the FP16 hi/lo tensor-core image of the weights
    return align_up((size_t)make_layout(N, n, depth, save).total * sizeof(float), 256) + tc_weight_image_bytes(depth);
}

int dcd_gmw_weights_fwd(const float* kpts2d, const float* kpts3d, const float* params4, const float* params6,
                        int64_t N, int n, int depth, int save, float* reg_weights, float* feat4, float* feat6,
                        void* workspace, size_t workspace_bytes, void* stream) {
    if (N < 0 || bad_n(n) || depth < 1) return DCD_E_INVALID;
    if (N == 0) return DCD_OK;
    if (!kpts2d || !kpts3d || !params4 || !params6 || !reg_weights || !workspace) return DCD_E_INVALID;
    if (misaligned(kpts2d, 8) || misaligned(params4, 16) || misaligned(params6, 16)) return DCD_E_INVALID;
    if (misaligned(workspace, 256) || workspace_bytes < dcd_gmw_workspace_bytes(N, n, depth, save)) return DCD_E_WORKSPACE;
    return launch_gmw_weights_fwd(kpts2d, kpts3d, params4, params6, N, n, depth, save, reg_weights, feat4, feat6,
                                  static_cast<float*>(workspace), (cudaStream_t)stream);
}

size_t dcd_gmw_bwd_scratch_bytes(int64_t N, int n, int depth) {
    if (N <= 0 || bad_n(n) || depth < 1) return 0;
    return gmw_bwd_scratch_floats(N, n, depth) * sizeof(float);
}

int dcd_gmw_weights_bwd(const float* kpts2d, const float* kpts3d, const float* params4, const float* params6,
                        int64_t N, int n, int depth, const float* grad_reg_weights, const float* grad_nfeat4,
                        const float* grad_nfeat6, float* grad_params4,
                        float* grad_params6, void* workspace, size_t workspace_bytes, void* scratch,
                        size_t scratch_bytes, void* stream) {
    if (N <= 0 || bad_n(n) || depth < 1) return DCD_E_INVALID;
    if (!kpts2d || !kpts3d || !params4 || !params6 || !grad_params4 || !grad_params6) return DCD_E_INVALID;
    if (!grad_reg_weights && !grad_nfeat4 && !grad_nfeat6) return DCD_E_INVALID;
    if (!workspace || !scratch) return DCD_E_INVALID;
    if (misaligned(workspace, 256) || workspace_bytes < dcd_gmw_workspace_bytes(N, n, depth, 1)) return DCD_E_WORKSPACE;
    if (misaligned(scratch, 256) || scratch_bytes < dcd_gmw_bwd_scratch_bytes(N, n, depth)) return DCD_E_WORKSPACE;
    return launch_gmw_weights_bwd(kpts2d, kpts3d, params4, params6, N, n, depth, grad_reg_weights, grad_nfeat4, grad_nfeat6,
                                  grad_params4, grad_params6, static_cast<float*>(workspace), static_cast<float*>(scratch),
                                  (cudaStream_t)stream);
}

int dcd_gmw_kpts_bwd(const float* params4, const float* params6, int64_t N, int n, int depth, void* scratch,
                     size_t scratch_bytes, float* grad_kpts2d, float* grad_kpts3d, void* stream) {
    if (N <= 0 || bad_n(n) || depth < 1) return DCD_E_INVALID;
    if (!params4 || !params6 || !scratch || (!grad_kpts2d && !grad_kpts3d)) return DCD_E_INVALID;
    if (misaligned(scratch, 256) || scratch_bytes < dcd_gmw_bwd_scratch_bytes(N, n, depth)) return DCD_E_WORKSPACE;
    return launch_gmw_kpts_bwd(params4, params6, N, n, depth, static_cast<float*>(scratch), grad_kpts2d, grad_kpts3d,
                               (cudaStream_t)stream);
}

int dcd_gmw_aggregate_fwd(const float* reg_weights, const float* depths, const int64_t* idx, int64_t N, int64_t E,
                          int k, int depths_are_selected, float* depth_out, float* probs, void* stream) {
    if (N < 0 || E < 1 || k < 1 || k > E) return DCD_E_INVALID;
    if (N == 0) return DCD_OK;
    if (!reg_weights || !depths || !idx || !depth_out) return DCD_E_INVALID;
    return launch_gmw_aggregate_fwd(reg_weights, depths, idx, N, E, k, depths_are_selected, depth_out, probs,
                                    (cudaStream_t)stream);
}

int dcd_gmw_aggregate_bwd(const float* reg_weights, const float* depths, const int64_t* idx, int64_t N, int64_t E,
                          int k, int depths_are_selected, const float* grad_depth_out, float* grad_reg_weights,
                          float* grad_depths, void* stream) {
    if (N < 0 || E < 1 || k < 1 || k > E) return DCD_E_INVALID;
    if (k > DCD_AGG_BWD_MAX_K) return DCD_E_UNSUPPORTED;
    if (N == 0) return DCD_OK;
    if (!reg_weights || !depths || !idx || !grad_depth_out || !grad_reg_weights) return DCD_E_INVALID;
    return launch_gmw_aggregate_bwd(reg_weights, depths, idx, N, E, k, depths_are_selected, grad_depth_out,
                                    grad_reg_weights, grad_depths, (cudaStream_t)stream);
}

// workspace of the fused call: [mlp workspace for `chunk` objects][idx chunk*k i64][depth_sel chunk*k][reg_w chunk*E]
size_t dcd_gmw_depth_workspace_bytes(int64_t N, int n, int depth, int64_t chunk) {
    if (N <= 0 || bad_n(n) || depth < 1 || chunk < 1) return 0;
    if (chunk > N) chunk = N;
    const int64_t E = num_edges(n);
    size_t b = align_up(dcd_gmw_workspace_bytes(chunk, n, depth, 0), 256);
    b += align_up((size_t)chunk * E * sizeof(int64_t), 256);      // idx (k <= E)
    b += align_up((size_t)chunk * E * sizeof(float), 256);        // selected depths
    b += align_up((size_t)chunk * E * sizeof(float), 256);        // reg_weights
    return b;
}

int dcd_gmw_depth_fwd(const float* kpts2d, const float* kpts3d, const float* rot, const float* params4,
                      const float* params6, int64_t N, int n, int depth, int k, float lo, float hi, int64_t chunk,
                      float* depth_out, int64_t* idx_out, float* reg_weights, void* workspace,
                      size_t workspace_bytes, void* stream) {
    if (N < 0 || bad_n(n) || depth < 1 || chunk < 1) return DCD_E_INVALID;
    const int64_t E = num_edges(n);
    if (k < 1 || k > E) return DCD_E_INVALID;
    if (N == 0) return DCD_OK;
    if (!kpts2d || !kpts3d || !rot || !params4 || !params6 || !depth_out || !workspace) return DCD_E_INVALID;
    if (chunk > N) chunk = N;
    if (misaligned(workspace, 256) || workspace_bytes < dcd_gmw_depth_workspace_bytes(N, n, depth, chunk))
        return DCD_E_WORKSPACE;
    return gmw_depth_chunks(kpts2d, kpts3d, rot, params4, params6, N, n, depth, k, lo, hi, chunk, depth_out, idx_out, reg_weights,
                            workspace, nullptr, nullptr, nullptr, (cudaStream_t)stream);
}

// workspace of the refine chain: [GMW 2D keypoints N*73*2][template points N*73*3][dcd_gmw_depth_fwd workspace for 73 keypoints]
size_t dcd_dgde_gmw_refine_workspace_bytes(int64_t N, int n, int depth, int64_t chunk) {
    if (N <= 0 || bad_n(n) || n < DCD_GMW_KPTS || depth < 1 || chunk < 1) return 0;
    size_t b = align_up((size_t)N * DCD_GMW_KPTS * 2 * sizeof(float), 256);
    b += align_up((size_t)N * DCD_GMW_KPTS * 3 * sizeof(float), 256);
    return b + dcd_gmw_depth_workspace_bytes(N, DCD_GMW_KPTS, depth, chunk);
}

int dcd_dgde_gmw_refine_fwd(const float* feature_maps, const int64_t* index, const int32_t* batch_idx, int64_t B, int C, int H,
                            int W, int ch_kpts2d, int ch_kpts3d, int ch_offset3d, const float* rot, const float* K, const float* pad,
                            const float* dims, const float* params4, const float* params6, int64_t N, int n, int depth, int k,
                            int64_t chunk, float* dgde_depth, float* dgde_location, float* gmw_depth, float* location,
                            float* gmw_kpts, float* kps3d, int64_t* idx_out, void* workspace, size_t workspace_bytes,
                            void* stream) {
    if (N < 0 || B < 1 || C < 1 || H < 1 || W < 1 || bad_n(n) || n < DCD_GMW_KPTS || depth < 1 || chunk < 1)
        return DCD_E_INVALID;
    if (ch_kpts2d < 0 || ch_kpts2d + 2 * n > C || ch_kpts3d < 0 || ch_kpts3d + 3 * n > C || ch_offset3d < 0 || ch_offset3d + 2 > C)
        return DCD_E_INVALID;
    if (k < 1 || k > num_edges(DCD_GMW_KPTS)) return DCD_E_INVALID;
    if (N == 0) return DCD_OK;
    if (!feature_maps || !index || !rot || !K || !pad || !dims || !params4 || !params6) return DCD_E_INVALID;
    if (!dgde_depth || !dgde_location || !gmw_depth || !location || !workspace) return DCD_E_INVALID;
    if (B > 1 && !batch_idx) return DCD_E_INVALID;
    if (misaligned(gmw_kpts, 8) || misaligned(params4, 16) || misaligned(params6, 16)) return DCD_E_INVALID;
    if (chunk > N) chunk = N;
    if (misaligned(workspace, 256) || workspace_bytes < dcd_dgde_gmw_refine_workspace_bytes(N, n, depth, chunk))
        return DCD_E_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char* p = static_cast<unsigned char*>(workspace);
    float* k2 = reinterpret_cast<float*>(p);
    p += align_up((size_t)N * DCD_GMW_KPTS * 2 * sizeof(float), 256);
    float* k3 = reinterpret_cast<float*>(p);
    p += align_up((size_t)N * DCD_GMW_KPTS * 3 * sizeof(float), 256);
    if (gmw_kpts) k2 = gmw_kpts;
    if (kps3d) k3 = kps3d;
    int rc = launch_dgde_frame(feature_maps, index, batch_idx, C, H, W, ch_kpts2d, ch_kpts3d, ch_offset3d, rot, K, pad, dims, N, n,
                               kDgdeLo, kDgdeHi, DCD_NORMALISE_2D | DCD_SUB_B3, kDownRatio, dgde_depth, dgde_location, nullptr,
                               nullptr, k2, k3, st);
    if (rc != DCD_OK) return rc;
    return gmw_depth_chunks(k2, k3, rot, params4, params6, N, DCD_GMW_KPTS, depth, k, kGmwLo, kGmwHi, chunk, gmw_depth, idx_out,
                            nullptr, p, dgde_location, dims, location, st);
}

}  // extern "C"
