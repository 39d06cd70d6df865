// Frame epilogue of the DGDE detector head around the edge solve (SURVEY 8f rows N2 / N4), one kernel:
//   image-space keypoints   real_2d = (kpts_off + (points + offsets)) * down_ratio - pad       detector_infer.py:216-217
//   edge solve + mean       depth   = mean_e clamp(|H| / max(|V|, 1e-10), lo, hi) - b3          anno_encoder.py:326-390, :225
//   3D location             (u, v)  = (points + offsets) * down_ratio - pad                      anno_encoder.py:147-161
//                           x = ((u - c_u) * depth) / f_u + b_x,  y likewise,  z = depth         kitti_utils.py:239-244, 399-417
//                           y += h / 2                                                           detector_infer.py:188
// so the 2D keypoints never exist in global memory and the location needs no second launch.
// One warp per object, same staging as the throughput edge-solve kernel (edge_solve.cu): 16-byte per-keypoint
// terms in shared memory, (i, j) byte offsets from a CTA-shared pair table, per-lane strided accumulation.
// Every operation is rounded like the reference's FP32 torch sequence; the calibration scalars b_x, b_y are formed
// in FP32 from the FP32 matrix (the reference forms them in float64 numpy: a 1-ulp difference of a 0.06 m offset).
#include "dcd_common.cuh"

namespace dcd {
namespace {

template <int THREADS>
__global__ void __launch_bounds__(THREADS)
dgde_locate_warp_kernel(const float* __restrict__ kpts_off, const float* __restrict__ kps3d, const float* __restrict__ rot,
                        const float* __restrict__ K, const float* __restrict__ points, const float* __restrict__ offsets,
                        const float* __restrict__ pad, const float* __restrict__ dims, const float* __restrict__ depth_in,
                        int64_t N, int n, float lo, float hi, int flags, float down_ratio,
                        float* __restrict__ depth_out, float* __restrict__ loc_out) {
    constexpr int NWARP = THREADS / 32;
    const int E = n * (n - 1) / 2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float4* kp_all = reinterpret_cast<float4*>(smem_raw);                     // [NWARP][n]
    uint32_t* tab_s = reinterpret_cast<uint32_t*>(kp_all + NWARP * n);        // [E] byte offsets (i*16) | (j*16) << 16
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool solve = kpts_off != nullptr;
    if (solve) {
        for (int e = tid; e < E; e += THREADS) {
            int i, j;
            decode_edge(e, n, i, j);
            tab_s[e] = (uint32_t)(i * 16) | ((uint32_t)(j * 16) << 16);
        }
    }
    __syncthreads();
    float4* kp = kp_all + warp * n;
    const unsigned char* kpb = reinterpret_cast<const unsigned char*>(kp);
    const bool normalise = (flags & DCD_NORMALISE_2D) != 0;
    for (int64_t obj = (int64_t)blockIdx.x * NWARP + warp; obj < N; obj += (int64_t)gridDim.x * NWARP) {
        const float* Ko = K + obj * 12;
        const float f_u = __ldg(Ko + 0), c_u = __ldg(Ko + 2), f_v = __ldg(Ko + 5), c_v = __ldg(Ko + 6);
        const float cx = __fadd_rn(__ldg(points + obj * 2), __ldg(offsets + obj * 2));
        const float cyy = __fadd_rn(__ldg(points + obj * 2 + 1), __ldg(offsets + obj * 2 + 1));
        const float pad_u = __ldg(pad + obj * 2), pad_v = __ldg(pad + obj * 2 + 1);
        float depth;
        if (solve) {
            const float b3 = (flags & DCD_SUB_B3) ? __ldg(Ko + 11) : 0.f;
            const float r = __ldg(rot + obj);
            const float sn = sinf(r), cs = cosf(r);
            for (int t = lane; t < n; t += 32) {
                const float off_v = __ldg(kpts_off + (obj * n + t) * 2 + 1);
                const float v_img = __fsub_rn(__fmul_rn(__fadd_rn(off_v, cyy), down_ratio), pad_v);
                const float* p3 = kps3d + (obj * n + t) * 3;
                kp[t] = keypoint_terms(v_img, __ldg(p3), __ldg(p3 + 1), __ldg(p3 + 2), sn, cs, normalise, c_v, f_v);
            }
            __syncwarp();
            float acc = 0.f;
            for (int e = lane; e < E; e += 32) {
                const uint32_t p = tab_s[e];
                const float4 a = *reinterpret_cast<const float4*>(kpb + (p & 0xffffu));
                const float4 b = *reinterpret_cast<const float4*>(kpb + (p >> 16));
                acc += edge_depth(a, b, lo, hi, b3);
            }
            acc = warp_sum(acc);
            depth = __fdiv_rn(acc, (float)E);
            __syncwarp();                                    // all lanes done with kp before it is restaged
        } else {
            depth = __ldg(depth_in + obj);
        }
        if (lane == 0) {
            if (depth_out != nullptr) depth_out[obj] = depth;
            if (loc_out != nullptr) {
                const float u = __fsub_rn(__fmul_rn(cx, down_ratio), pad_u);
                const float v = __fsub_rn(__fmul_rn(cyy, down_ratio), pad_v);
                const float b_x = __fdiv_rn(__ldg(Ko + 3), -f_u), b_y = __fdiv_rn(__ldg(Ko + 7), -f_v);
                float x = __fadd_rn(__fdiv_rn(__fmul_rn(__fsub_rn(u, c_u), depth), f_u), b_x);
                float y = __fadd_rn(__fdiv_rn(__fmul_rn(__fsub_rn(v, c_v), depth), f_v), b_y);
                if (dims != nullptr) y = __fadd_rn(y, __fmul_rn(__ldg(dims + obj * 3 + 1), 0.5f));
                loc_out[obj * 3 + 0] = x;
                loc_out[obj * 3 + 1] = y;
                loc_out[obj * 3 + 2] = depth;
            }
        }
    }
}

// The same epilogue reading the detector's regression map directly (row N2 fused into the load stage): for detection d at
// heat-map position index[d] of image batch_idx[d] the keypoint offsets, 3D template points and the sub-pixel offset are
// the values of their channel groups at that position of the [B,C,H,W] map (select_point_of_interest,
// DGDE/model/layers/utils.py:120-145, + the key2channel slices of detector_infer.py:133,216,219), so POI gather ->
// image keypoints -> edge solve -> mean -> location is ONE launch and the [B,K,C] gather never exists in memory.
// GMW = true (dcd_dgde_gmw_refine_fwd) also writes GMW's inputs for keypoints 0 .. DCD_GMW_KPTS-1: the normalised 2D keypoints
// ((u - K[0][2]) / K[0][0], (v - K[1][2]) / K[1][1]; the two FP32 roundings of wire.from_detector) and the template points,
// both with a row stride of DCD_GMW_KPTS.  GMW = false is the kernel of dcd_dgde_frame_fwd, unchanged.
template <int THREADS, bool GMW>
__global__ void __launch_bounds__(THREADS)
dgde_frame_warp_kernel(const float* __restrict__ fmap, const int64_t* __restrict__ index, const int32_t* __restrict__ batch_idx,
                       int C, int H, int W, int ch_k2, int ch_k3, int ch_off,
                       const float* __restrict__ rot, const float* __restrict__ K, const float* __restrict__ pad,
                       const float* __restrict__ dims, int64_t N, int n, float lo, float hi, int flags, float down_ratio,
                       float* __restrict__ depth_out, float* __restrict__ loc_out, float* __restrict__ kimg_out,
                       float* __restrict__ k3_out, float* __restrict__ gmw_k2_out, float* __restrict__ gmw_k3_out) {
    constexpr int NWARP = THREADS / 32;
    const int E = n * (n - 1) / 2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float4* kp_all = reinterpret_cast<float4*>(smem_raw);                     // [NWARP][n]
    uint32_t* tab_s = reinterpret_cast<uint32_t*>(kp_all + NWARP * n);        // [E]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int e = tid; e < E; e += THREADS) {
        int i, j;
        decode_edge(e, n, i, j);
        tab_s[e] = (uint32_t)(i * 16) | ((uint32_t)(j * 16) << 16);
    }
    __syncthreads();
    float4* kp = kp_all + warp * n;
    const unsigned char* kpb = reinterpret_cast<const unsigned char*>(kp);
    const bool normalise = (flags & DCD_NORMALISE_2D) != 0;
    const int64_t HW = (int64_t)H * W;
    const float qnan = __int_as_float(0x7fc00000);
    for (int64_t obj = (int64_t)blockIdx.x * NWARP + warp; obj < N; obj += (int64_t)gridDim.x * NWARP) {
        const int64_t pos = index[obj];
        const bool inside = pos >= 0 && pos < HW;             // like dcd_poi_gather_fwd: NaN instead of a fault
        const float* base = fmap + (int64_t)(batch_idx != nullptr ? batch_idx[obj] : 0) * C * HW + (inside ? pos : 0);
        auto chan = [&](int c) { return inside ? __ldg(base + (int64_t)c * HW) : qnan; };
        const float* Ko = K + obj * 12;
        const float f_u = __ldg(Ko + 0), c_u = __ldg(Ko + 2), f_v = __ldg(Ko + 5), c_v = __ldg(Ko + 6);
        const float px = (float)(pos % W), py = (float)(pos / W);             // select_topk: xs = ind % W, ys = ind // W
        const float cx = __fadd_rn(px, chan(ch_off)), cyy = __fadd_rn(py, chan(ch_off + 1));
        const float pad_u = __ldg(pad + obj * 2), pad_v = __ldg(pad + obj * 2 + 1);
        const float b3 = (flags & DCD_SUB_B3) ? __ldg(Ko + 11) : 0.f;
        const float r = __ldg(rot + obj);
        const float sn = sinf(r), cs = cosf(r);
        for (int t = lane; t < n; t += 32) {
            const float off_v = chan(ch_k2 + 2 * t + 1);
            const float v_img = __fsub_rn(__fmul_rn(__fadd_rn(off_v, cyy), down_ratio), pad_v);
            const float X = chan(ch_k3 + 3 * t), Y = chan(ch_k3 + 3 * t + 1), Z = chan(ch_k3 + 3 * t + 2);
            kp[t] = keypoint_terms(v_img, X, Y, Z, sn, cs, normalise, c_v, f_v);
            if (kimg_out != nullptr) {
                const float u_img = __fsub_rn(__fmul_rn(__fadd_rn(chan(ch_k2 + 2 * t), cx), down_ratio), pad_u);
                kimg_out[(obj * n + t) * 2] = u_img;
                kimg_out[(obj * n + t) * 2 + 1] = v_img;
            }
            if (k3_out != nullptr) {
                float* o = k3_out + (obj * n + t) * 3;
                o[0] = X; o[1] = Y; o[2] = Z;
            }
            if constexpr (GMW) {
                if (t < DCD_GMW_KPTS) {
                    const float u_img = __fsub_rn(__fmul_rn(__fadd_rn(chan(ch_k2 + 2 * t), cx), down_ratio), pad_u);
                    float* g2 = gmw_k2_out + (obj * DCD_GMW_KPTS + t) * 2;
                    g2[0] = __fdiv_rn(__fsub_rn(u_img, c_u), f_u);
                    g2[1] = __fdiv_rn(__fsub_rn(v_img, c_v), f_v);
                    float* g3 = gmw_k3_out + (obj * DCD_GMW_KPTS + t) * 3;
                    g3[0] = X; g3[1] = Y; g3[2] = Z;
                }
            }
        }
        __syncwarp();
        float acc = 0.f;
        for (int e = lane; e < E; e += 32) {
            const uint32_t p = tab_s[e];
            const float4 a = *reinterpret_cast<const float4*>(kpb + (p & 0xffffu));
            const float4 b = *reinterpret_cast<const float4*>(kpb + (p >> 16));
            acc += edge_depth(a, b, lo, hi, b3);
        }
        acc = warp_sum(acc);
        const float depth = __fdiv_rn(acc, (float)E);
        __syncwarp();
        if (lane == 0) {
            if (depth_out != nullptr) depth_out[obj] = depth;
            if (loc_out != nullptr) {
                const float u = __fsub_rn(__fmul_rn(cx, down_ratio), pad_u);
                const float v = __fsub_rn(__fmul_rn(cyy, down_ratio), pad_v);
                const float b_x = __fdiv_rn(__ldg(Ko + 3), -f_u), b_y = __fdiv_rn(__ldg(Ko + 7), -f_v);
                float x = __fadd_rn(__fdiv_rn(__fmul_rn(__fsub_rn(u, c_u), depth), f_u), b_x);
                float y = __fadd_rn(__fdiv_rn(__fmul_rn(__fsub_rn(v, c_v), depth), f_v), b_y);
                if (dims != nullptr) y = __fadd_rn(y, __fmul_rn(__ldg(dims + obj * 3 + 1), 0.5f));
                loc_out[obj * 3 + 0] = x;
                loc_out[obj * 3 + 1] = y;
                loc_out[obj * 3 + 2] = depth;
            }
        }
    }
}

}  // namespace

// gmw_k2_out == NULL: the dcd_dgde_frame_fwd kernel; otherwise (with gmw_k3_out, both [N,DCD_GMW_KPTS,.], n >= DCD_GMW_KPTS) the
// GMW = true instantiation that also writes GMW's inputs.
int launch_dgde_frame(const float* fmap, const int64_t* index, const int32_t* batch_idx, int C, int H, int W, int ch_k2, int ch_k3,
                      int ch_off, const float* rot, const float* K, const float* pad, const float* dims, int64_t N, int n, float lo,
                      float hi, int flags, float down_ratio, float* depth_out, float* loc_out, float* kimg_out, float* k3_out,
                      float* gmw_k2_out, float* gmw_k3_out, cudaStream_t st) {
    constexpr int T = 128;                                  // a frame has <= 50 detections: more, smaller CTAs
    const int E = n * (n - 1) / 2;
    const size_t smem = (size_t)(T / 32) * n * sizeof(float4) + (size_t)E * sizeof(uint32_t);
    if (smem > 227 * 1024) return DCD_E_UNSUPPORTED;
    auto kernel = gmw_k2_out != nullptr ? dgde_frame_warp_kernel<T, true> : dgde_frame_warp_kernel<T, false>;
    if (smem > 48 * 1024) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int64_t want = (N + T / 32 - 1) / (T / 32);
    const int64_t cap = (int64_t)device_sm_count() * 8;
    const int grid = (int)(want < cap ? want : cap);
    kernel<<<grid, T, smem, st>>>(fmap, index, batch_idx, C, H, W, ch_k2, ch_k3, ch_off, rot, K, pad, dims, N, n, lo, hi, flags,
                                  down_ratio, depth_out, loc_out, kimg_out, k3_out, gmw_k2_out, gmw_k3_out);
    DCD_CHECK_LAUNCH();
    return DCD_OK;
}

namespace {

// Backward of the no-solve form of dgde_locate_warp_kernel (decode_location_flatten, anno_encoder.py:147-161), one thread per
// object, in the order torch's autograd forms it for x = ((u - c_u) * d) / f_u + b_x, u = (p + o) * down_ratio - pad:
//   d/du: (g_x / f_u) * d,  d/d(p + o) = that * down_ratio,  d/dd: (g_x / f_u) * (u - c_u) + (y likewise) + g_z.
__global__ void __launch_bounds__(256)
dgde_locate_bwd_kernel(const float* __restrict__ K, const float* __restrict__ points, const float* __restrict__ offsets,
                       const float* __restrict__ pad, const float* __restrict__ depth, const float* __restrict__ grad_loc, int64_t N,
                       float down_ratio, float* __restrict__ grad_offsets, float* __restrict__ grad_points,
                       float* __restrict__ grad_depth) {
    const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= N) return;
    const float* Ko = K + o * 12;
    const float f_u = __ldg(Ko + 0), c_u = __ldg(Ko + 2), f_v = __ldg(Ko + 5), c_v = __ldg(Ko + 6);
    const float d = __ldg(depth + o);
    const float gx = __ldg(grad_loc + o * 3), gy = __ldg(grad_loc + o * 3 + 1), gz = __ldg(grad_loc + o * 3 + 2);
    const float ax = __fdiv_rn(gx, f_u), ay = __fdiv_rn(gy, f_v);
    const float g_u = __fmul_rn(__fmul_rn(ax, d), down_ratio), g_v = __fmul_rn(__fmul_rn(ay, d), down_ratio);
    if (grad_offsets != nullptr) { grad_offsets[o * 2] = g_u; grad_offsets[o * 2 + 1] = g_v; }
    if (grad_points != nullptr) { grad_points[o * 2] = g_u; grad_points[o * 2 + 1] = g_v; }
    if (grad_depth != nullptr) {
        const float u = __fsub_rn(__fmul_rn(__fadd_rn(__ldg(points + o * 2), __ldg(offsets + o * 2)), down_ratio), __ldg(pad + o * 2));
        const float v = __fsub_rn(__fmul_rn(__fadd_rn(__ldg(points + o * 2 + 1), __ldg(offsets + o * 2 + 1)), down_ratio),
                                  __ldg(pad + o * 2 + 1));
        grad_depth[o] = __fadd_rn(__fadd_rn(__fmul_rn(ax, __fsub_rn(u, c_u)), __fmul_rn(ay, __fsub_rn(v, c_v))), gz);
    }
}

}  // namespace

int launch_dgde_locate_bwd(const float* K, const float* points, const float* offsets, const float* pad, const float* depth,
                           const float* grad_loc, int64_t N, float down_ratio, float* grad_offsets, float* grad_points,
                           float* grad_depth, cudaStream_t st) {
    dgde_locate_bwd_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(K, points, offsets, pad, depth, grad_loc, N, down_ratio,
                                                                         grad_offsets, grad_points, grad_depth);
    DCD_CHECK_LAUNCH();
    return DCD_OK;
}

int launch_dgde_locate(const float* kpts_off, const float* kps3d, const float* rot, const float* K, const float* points,
                       const float* offsets, const float* pad, const float* dims, const float* depth_in, int64_t N, int n,
                       float lo, float hi, int flags, float down_ratio, float* depth_out, float* loc_out, cudaStream_t st) {
    constexpr int T = 256;
    const int E = n * (n - 1) / 2;
    const size_t smem = (size_t)(T / 32) * n * sizeof(float4) + (size_t)E * sizeof(uint32_t);
    if (smem > 227 * 1024) return DCD_E_UNSUPPORTED;
    if (smem > 48 * 1024)
        cudaFuncSetAttribute(dgde_locate_warp_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int64_t want = (N + T / 32 - 1) / (T / 32);
    const int64_t cap = (int64_t)device_sm_count() * 8;
    const int grid = (int)(want < cap ? want : cap);
    dgde_locate_warp_kernel<T><<<grid, T, smem, st>>>(kpts_off, kps3d, rot, K, points, offsets, pad, dims, depth_in, N, n, lo, hi,
                                                      flags, down_ratio, depth_out, loc_out);
    DCD_CHECK_LAUNCH();
    return DCD_OK;
}

}  // namespace dcd

// ---------------------------------------------------------------------------------------------
// Rest of row N4: per-object depth ensemble of the detector head and the GMW-validation ray rescale.
// One thread per object; every operation rounded like the reference's FP32 torch sequence.
// ---------------------------------------------------------------------------------------------
namespace dcd {
namespace {

// depth of one projected height: f_u * h3d / (relu(height) * down_ratio + eps)          anno_encoder.py:209-211
__device__ __forceinline__ float height_depth(float fh, float height, float down_ratio, float eps) {
    return __fdiv_rn(fh, __fadd_rn(__fmul_rn(fmaxf(height, 0.f), down_ratio), eps));
}

__global__ void __launch_bounds__(256)
dgde_depth_ensemble_kernel(const float* __restrict__ kp10, const float* __restrict__ dims, const float* __restrict__ K,
                           const float* __restrict__ direct, const float* __restrict__ log_unc_direct,
                           const float* __restrict__ log_unc_kp, const float* __restrict__ scores, int64_t N, float down_ratio,
                           float eps, float lo, float hi, float* __restrict__ kp_depths, float* __restrict__ depth,
                           float* __restrict__ depth_error, int64_t* __restrict__ argmax, float* __restrict__ scores_out) {
    const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= N) return;
    const float* kp = kp10 + o * 20;
    float v[10];
#pragma unroll
    for (int t = 0; t < 10; ++t) v[t] = __ldg(kp + 2 * t + 1);
    const float fh = __fmul_rn(__ldg(K + o * 12), __ldg(dims + o * 3 + 1));          // calib.f_u * pred_height_3D
    // anno_encoder.py:199-201, 209-214, 221: centre line, corner pairs (0,4),(2,6) and (1,5),(3,7); mean of two; clamp
    float d[4];
    d[1] = height_depth(fh, __fsub_rn(v[8], v[9]), down_ratio, eps);
    d[2] = __fmul_rn(__fadd_rn(height_depth(fh, __fsub_rn(v[0], v[4]), down_ratio, eps),
                               height_depth(fh, __fsub_rn(v[2], v[6]), down_ratio, eps)), 0.5f);
    d[3] = __fmul_rn(__fadd_rn(height_depth(fh, __fsub_rn(v[1], v[5]), down_ratio, eps),
                               height_depth(fh, __fsub_rn(v[3], v[7]), down_ratio, eps)), 0.5f);
#pragma unroll
    for (int j = 1; j < 4; ++j) d[j] = fminf(fmaxf(d[j], lo), hi);
    if (kp_depths != nullptr) {
        kp_depths[o * 3 + 0] = d[1]; kp_depths[o * 3 + 1] = d[2]; kp_depths[o * 3 + 2] = d[3];
    }
    if (depth == nullptr && depth_error == nullptr && argmax == nullptr && scores_out == nullptr) return;
    // detector_infer.py:141,154,158-171: uncertainties = exp(channel); weights = (1/u) / sum(1/u)
    const int first = direct != nullptr ? 0 : 1;
    float u[4], w[4];
    if (first == 0) {
        d[0] = __ldg(direct + o);
        u[0] = expf(__ldg(log_unc_direct + o));
    }
#pragma unroll
    for (int j = 1; j < 4; ++j) u[j] = expf(__ldg(log_unc_kp + o * 3 + j - 1));
    float wsum = 0.f;
    int best = first;
    for (int j = first; j < 4; ++j) {
        w[j] = __fdiv_rn(1.f, u[j]);
        wsum = __fadd_rn(wsum, w[j]);
        if (w[j] > w[best]) best = j;                       // first maximum, like torch.argmax
    }
    float dsum = 0.f, esum = 0.f;
    for (int j = first; j < 4; ++j) {
        const float wn = __fdiv_rn(w[j], wsum);
        dsum = __fadd_rn(dsum, __fmul_rn(d[j], wn));
        esum = __fadd_rn(esum, __fmul_rn(wn, u[j]));
    }
    if (depth != nullptr) depth[o] = dsum;
    if (depth_error != nullptr) depth_error[o] = esum;
    if (argmax != nullptr) argmax[o] = best - first;
    if (scores_out != nullptr) {                             // detector_infer.py:197-203
        const float conf = __fsub_rn(1.f, fminf(fmaxf(esum, 0.01f), 1.f));
        const float s = __fmul_rn(__ldg(scores + o), conf);
        scores_out[o] = (esum != esum || s != s) ? 0.f : s;       // torch.clamp keeps NaN (fmaxf drops it): NaN -> 0
    }
}

// Backward of dgde_depth_ensemble_kernel: the forward is recomputed in its own operation order, then every backward formula is
// torch's for the reference's op (div: g / b and -g * ((a / b) / b); 1 / u = reciprocal: -g * (r * r); exp: g * e; mean of two:
// g / 2; relu: g where height > 0; clamp: g where lo <= x <= hi), with a term skipped (not multiplied by 0) when its upstream
// gradient is absent, so that infinities and NaNs reach the same gradients as in the reference's autograd.  The NaN -> 0 of
// the scores (detector_infer.py:202) zeroes their upstream gradient there.  One thread per object: nothing crosses objects.
__global__ void __launch_bounds__(256)
dgde_depth_ensemble_bwd_kernel(const float* __restrict__ kp10, const float* __restrict__ dims, const float* __restrict__ K,
                               const float* __restrict__ direct, const float* __restrict__ log_unc_direct,
                               const float* __restrict__ log_unc_kp, const float* __restrict__ scores, int64_t N, float down_ratio,
                               float eps, float lo, float hi, const float* __restrict__ g_kp_depths, const float* __restrict__ g_depth,
                               const float* __restrict__ g_depth_error, const float* __restrict__ g_scores_out,
                               float* __restrict__ grad_kp10, float* __restrict__ grad_dims, float* __restrict__ grad_direct,
                               float* __restrict__ grad_lud, float* __restrict__ grad_luk, float* __restrict__ grad_scores) {
    const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= N) return;
    const float* kp = kp10 + o * 20;
    float v[10];
#pragma unroll
    for (int t = 0; t < 10; ++t) v[t] = __ldg(kp + 2 * t + 1);
    const float f_u = __ldg(K + o * 12);
    const float fh = __fmul_rn(f_u, __ldg(dims + o * 3 + 1));
    // heights in the forward's order: centre (8, 9), corner_02 (0, 4), (2, 6), corner_13 (1, 5), (3, 7)
    constexpr int PA[5] = {8, 0, 2, 1, 3}, PB[5] = {9, 4, 6, 5, 7};
    float ht[5], q[5];
#pragma unroll
    for (int e = 0; e < 5; ++e) {
        ht[e] = __fsub_rn(v[PA[e]], v[PB[e]]);
        q[e] = height_depth(fh, ht[e], down_ratio, eps);
    }
    float draw[4], d[4];
    draw[1] = q[0];
    draw[2] = __fmul_rn(__fadd_rn(q[1], q[2]), 0.5f);
    draw[3] = __fmul_rn(__fadd_rn(q[3], q[4]), 0.5f);
#pragma unroll
    for (int j = 1; j < 4; ++j) d[j] = fminf(fmaxf(draw[j], lo), hi);

    // gradients of the keypoint depths (after the clamp); has[j]: some upstream gradient reached d[j]
    float gd[4] = {0.f, 0.f, 0.f, 0.f};
    bool has[4] = {false, false, false, false};
    if (g_kp_depths != nullptr) {
#pragma unroll
        for (int j = 1; j < 4; ++j) { gd[j] = __ldg(g_kp_depths + o * 3 + j - 1); has[j] = true; }
    }
    const bool want_depth = g_depth != nullptr;
    const bool want_err = g_depth_error != nullptr || g_scores_out != nullptr;
    float g_sc = 0.f;
    if (want_depth || want_err) {
        const int first = direct != nullptr ? 0 : 1;
        float u[4], r[4], wn[4];
        if (first == 0) {
            d[0] = __ldg(direct + o);
            u[0] = expf(__ldg(log_unc_direct + o));
        }
#pragma unroll
        for (int j = 1; j < 4; ++j) u[j] = expf(__ldg(log_unc_kp + o * 3 + j - 1));
        float S = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j < first) continue;
            r[j] = __fdiv_rn(1.f, u[j]);
            S = __fadd_rn(S, r[j]);
        }
        float esum = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j < first) continue;
            wn[j] = __fdiv_rn(r[j], S);
            esum = __fadd_rn(esum, __fmul_rn(wn[j], u[j]));
        }
        // depth_error's gradient: its own, plus the score path  out = scores * (1 - clamp(err, 0.01, 1)); out[isnan(out)] = 0
        float ge = g_depth_error != nullptr ? __ldg(g_depth_error + o) : 0.f;
        if (g_scores_out != nullptr) {
            const float qnan = __int_as_float(0x7fc00000);
            const float cl = esum != esum ? qnan : fminf(fmaxf(esum, 0.01f), 1.f);    // torch.clamp keeps NaN
            const float conf = __fsub_rn(1.f, cl);
            const float sc = __ldg(scores + o);
            const float s = __fmul_rn(sc, conf);
            const float go = s != s ? 0.f : __ldg(g_scores_out + o);
            g_sc = __fmul_rn(go, conf);
            const float gconf = __fmul_rn(go, sc);
            const float gcl = (esum >= 0.01f && esum <= 1.f) ? -gconf : 0.f;
            ge = g_depth_error != nullptr ? __fadd_rn(ge, gcl) : gcl;
        }
        const float gdep = want_depth ? __ldg(g_depth + o) : 0.f;
        // depth = sum(d * wn), err = sum(wn * u), wn = r / S, r = 1 / u, u = exp(l)
        float gwn[4], gu[4], gS = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j < first) continue;
            if (want_depth && want_err) gwn[j] = __fadd_rn(__fmul_rn(gdep, d[j]), __fmul_rn(ge, u[j]));
            else gwn[j] = want_depth ? __fmul_rn(gdep, d[j]) : __fmul_rn(ge, u[j]);
            gS = __fsub_rn(gS, __fmul_rn(gwn[j], __fdiv_rn(__fdiv_rn(r[j], S), S)));
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j < first) continue;
            const float gr = __fadd_rn(__fdiv_rn(gwn[j], S), gS);
            const float grec = __fmul_rn(-gr, __fmul_rn(r[j], r[j]));
            gu[j] = want_err ? __fadd_rn(__fmul_rn(ge, wn[j]), grec) : grec;
            if (want_depth) {
                const float g = __fmul_rn(gdep, wn[j]);
                gd[j] = has[j] ? __fadd_rn(gd[j], g) : g;
                has[j] = true;
            }
        }
        if (grad_direct != nullptr) grad_direct[o] = first == 0 && want_depth ? gd[0] : 0.f;
        if (grad_lud != nullptr) grad_lud[o] = first == 0 ? __fmul_rn(gu[0], u[0]) : 0.f;
        if (grad_luk != nullptr) {
#pragma unroll
            for (int j = 1; j < 4; ++j) grad_luk[o * 3 + j - 1] = __fmul_rn(gu[j], u[j]);
        }
    } else {
        if (grad_direct != nullptr) grad_direct[o] = 0.f;
        if (grad_lud != nullptr) grad_lud[o] = 0.f;
        if (grad_luk != nullptr) grad_luk[o * 3] = grad_luk[o * 3 + 1] = grad_luk[o * 3 + 2] = 0.f;
    }
    if (grad_scores != nullptr) grad_scores[o] = g_sc;

    // back through the clamps, the means of two, the divisions and the relus
    float gq[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    bool hq[5] = {false, false, false, false, false};
#pragma unroll
    for (int j = 1; j < 4; ++j) {
        if (!has[j]) continue;
        const float g = (draw[j] >= lo && draw[j] <= hi) ? gd[j] : 0.f;
        if (j == 1) { gq[0] = g; hq[0] = true; }
        else {
            const float gh = __fdiv_rn(g, 2.f);
            gq[2 * j - 3] = gh; gq[2 * j - 2] = gh; hq[2 * j - 3] = hq[2 * j - 2] = true;
        }
    }
    float gfh[3] = {0.f, 0.f, 0.f}, gv[10];
#pragma unroll
    for (int t = 0; t < 10; ++t) gv[t] = 0.f;
#pragma unroll
    for (int e = 0; e < 5; ++e) {
        if (!hq[e]) continue;
        const float den = __fadd_rn(__fmul_rn(fmaxf(ht[e], 0.f), down_ratio), eps);
        const float gf = __fdiv_rn(gq[e], den);
        const int grp = e == 0 ? 0 : (e + 1) / 2;
        gfh[grp] = __fadd_rn(gfh[grp], gf);
        const float gden = __fmul_rn(-gq[e], __fdiv_rn(q[e], den));
        const float gh = ht[e] > 0.f ? __fmul_rn(gden, down_ratio) : 0.f;
        gv[PA[e]] = gh;
        gv[PB[e]] = -gh;
    }
    if (grad_kp10 != nullptr) {
        float* gk = grad_kp10 + o * 20;
#pragma unroll
        for (int t = 0; t < 10; ++t) { gk[2 * t] = 0.f; gk[2 * t + 1] = gv[t]; }
    }
    if (grad_dims != nullptr) {
        float gh = 0.f;
        bool any = false;
#pragma unroll
        for (int grp = 0; grp < 3; ++grp) {
            if (!hq[grp == 0 ? 0 : 2 * grp - 1]) continue;
            const float t = __fmul_rn(gfh[grp], f_u);
            gh = any ? __fadd_rn(gh, t) : t;
            any = true;
        }
        grad_dims[o * 3] = 0.f; grad_dims[o * 3 + 1] = gh; grad_dims[o * 3 + 2] = 0.f;
    }
}

// GMW/main.py:542-547
__global__ void __launch_bounds__(256)
gmw_ray_rescale_kernel(const float* __restrict__ raw_location, const float* __restrict__ pred_depth, const float* __restrict__ dim,
                       int64_t N, float* __restrict__ out) {
    const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= N) return;
    ray_rescale_one(__ldg(raw_location + o * 3), __ldg(raw_location + o * 3 + 1), __ldg(raw_location + o * 3 + 2),
                    __ldg(pred_depth + o), __ldg(dim + o * 3), out + o * 3);
}

}  // namespace

int launch_dgde_depth_ensemble(const float* kp10, const float* dims, const float* K, const float* direct, const float* lud,
                               const float* luk, const float* scores, int64_t N, float down_ratio, float eps, float lo, float hi,
                               float* kp_depths, float* depth, float* depth_error, int64_t* argmax, float* scores_out,
                               cudaStream_t st) {
    dgde_depth_ensemble_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(kp10, dims, K, direct, lud, luk, scores, N, down_ratio, eps,
                                                                             lo, hi, kp_depths, depth, depth_error, argmax, scores_out);
    DCD_CHECK_LAUNCH();
    return DCD_OK;
}

int launch_dgde_depth_ensemble_bwd(const float* kp10, const float* dims, const float* K, const float* direct, const float* lud,
                                   const float* luk, const float* scores, int64_t N, float down_ratio, float eps, float lo, float hi,
                                   const float* g_kd, const float* g_depth, const float* g_err, const float* g_so, float* grad_kp10,
                                   float* grad_dims, float* grad_direct, float* grad_lud, float* grad_luk, float* grad_scores,
                                   cudaStream_t st) {
    dgde_depth_ensemble_bwd_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(
        kp10, dims, K, direct, lud, luk, scores, N, down_ratio, eps, lo, hi, g_kd, g_depth, g_err, g_so, grad_kp10, grad_dims,
        grad_direct, grad_lud, grad_luk, grad_scores);
    DCD_CHECK_LAUNCH();
    return DCD_OK;
}

int launch_gmw_ray_rescale(const float* raw_location, const float* pred_depth, const float* dim, int64_t N, float* out,
                           cudaStream_t st) {
    gmw_ray_rescale_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(raw_location, pred_depth, dim, N, out);
    DCD_CHECK_LAUNCH();
    return DCD_OK;
}

}  // namespace dcd

// ---------------------------------------------------------------------------------------------
// Row N2, upstream gather: select_point_of_interest (DGDE/model/layers/utils.py:120-145) without the NCHW -> NHWC copy of
// the whole regression map the reference makes to pick <= 50 points per image:  out[b, k, c] = feat[b, c, index[b, k]].
// ---------------------------------------------------------------------------------------------
namespace dcd {
namespace {

__global__ void __launch_bounds__(256)
poi_gather_kernel(const float* __restrict__ feat, const int64_t* __restrict__ index, int64_t B, int64_t Kp, int C, int64_t HW,
                  float* __restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= B * Kp * C) return;
    const int c = (int)(t % C);
    const int64_t bk = t / C, b = bk / Kp;
    const int64_t p = index[bk];
    out[t] = (p >= 0 && p < HW) ? __ldg(feat + (b * C + c) * HW + p) : __int_as_float(0x7fc00000);   // out of range: NaN, no fault
}

// Backward, pass 1: the dense [B,C,H,W] gradient is zero except at <= B*K positions per channel, so it is filled at full store
// bandwidth (16-byte stores, grid-stride) and pass 2 overwrites the selected positions.
__global__ void __launch_bounds__(256)
poi_fill_zero_kernel(float* __restrict__ out, int64_t total, bool vec) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t done = 0;
    if (vec) {
        float4* o4 = reinterpret_cast<float4*>(out);
        const int64_t n4 = total / 4;
        for (int64_t i = t; i < n4; i += stride) o4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        done = n4 * 4;
    }
    for (int64_t i = done + t; i < total; i += stride) out[i] = 0.f;
}

// Backward, pass 2: one CTA per target slot (b, k).  The slot writes its position only if no earlier slot of the image holds
// the same position; it then sums, per channel, grad_out over every slot k' >= k with that position in ascending k', so each
// selected element is written once, deterministically, without atomics.  The duplicate scan is O(K) per slot
// (K <= DCD_POI_BWD_MAX_K).  An index outside [0, HW) drops its gradient (the forward gave NaN there).
__global__ void __launch_bounds__(128)
poi_scatter_kernel(const float* __restrict__ grad_out, const int64_t* __restrict__ index, int64_t B, int Kp, int C, int64_t HW,
                   float* __restrict__ grad_maps) {
    __shared__ int list[DCD_POI_BWD_MAX_K];
    __shared__ int count;
    const int tid = threadIdx.x, lane = tid & 31;
    for (int64_t slot = blockIdx.x; slot < B * Kp; slot += gridDim.x) {
        const int64_t b = slot / Kp;
        const int k = (int)(slot - b * Kp);
        const int64_t* ib = index + b * Kp;
        const int64_t p = ib[k];
        if (p < 0 || p >= HW) continue;                                   // uniform over the CTA
        bool earlier = false;
        for (int j = tid; j < k; j += blockDim.x) earlier |= ib[j] == p;
        if (__syncthreads_or(earlier)) continue;
        if (tid < 32) {                                                   // warp 0: ascending list of the slots >= k at p
            int cnt = 0;
            for (int base = k; base < Kp; base += 32) {
                const int j = base + lane;
                const bool m = j < Kp && ib[j] == p;
                const unsigned bal = __ballot_sync(0xffffffffu, m);
                if (m) list[cnt + __popc(bal & ((1u << lane) - 1u))] = j;
                cnt += __popc(bal);
            }
            if (lane == 0) count = cnt;
        }
        __syncthreads();
        const int cnt = count;
        const float* gb = grad_out + b * (int64_t)Kp * C;
        for (int c = tid; c < C; c += blockDim.x) {
            float acc = 0.f;
            for (int i = 0; i < cnt; ++i) acc += __ldg(gb + (int64_t)list[i] * C + c);
            grad_maps[(b * C + c) * HW + p] = acc;
        }
        __syncthreads();                                                  // list / count are rebuilt for the next slot
    }
}

}  // namespace

int launch_poi_gather_bwd(const float* grad_out, const int64_t* index, int64_t B, int64_t Kp, int C, int64_t HW, float* grad_maps,
                          cudaStream_t st) {
    const int64_t total = B * C * HW;
    const int64_t cap = (int64_t)device_sm_count() * 8;
    int64_t want = (total / 4 + 255) / 256;
    poi_fill_zero_kernel<<<(unsigned)(want < cap ? (want > 0 ? want : 1) : cap), 256, 0, st>>>(
        grad_maps, total, (reinterpret_cast<uintptr_t>(grad_maps) & 15) == 0);
    DCD_CHECK_LAUNCH();
    if (Kp == 0) return DCD_OK;
    want = B * Kp;
    poi_scatter_kernel<<<(unsigned)(want < cap * 4 ? want : cap * 4), 128, 0, st>>>(grad_out, index, B, (int)Kp, C, HW, grad_maps);
    DCD_CHECK_LAUNCH();
    return DCD_OK;
}

int launch_poi_gather(const float* feat, const int64_t* index, int64_t B, int64_t Kp, int C, int64_t HW, float* out, cudaStream_t st) {
    const int64_t total = B * Kp * C;
    poi_gather_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(feat, index, B, Kp, C, HW, out);
    DCD_CHECK_LAUNCH();
    return DCD_OK;
}

}  // namespace dcd
