// Edge-depth solve (forward, top-k selection, backward) for sm_100a.
//
// Replaces DGDE/model/anno_encoder.py:313-390 (decode_pairs_kpts_depth + get_up) and the solve/top-k of
// GMW/main.py:351-416 (compute_z).  Design (see DESIGN.md):
//   * the object's keypoints (2D v, 3D X/Y/Z, yaw, intrinsics: ~1.5 KB) are read from HBM once, reduced
//     to 16 B of per-keypoint terms {v, Y, v*C, C} and staged in shared memory; edges are enumerated by
//     index (never materialised as an n x n matrix) and every per-edge operation is rounded like the
//     reference's FP32 torch ops;
//   * throughput regime (N >= 16 x SMs): ONE WARP PER OBJECT, no block barrier in the object loop, the
//     (i,j) byte offsets come from a pair table shared by the CTA, next object's inputs prefetched in
//     registers, per-object mean by warp shuffles;
//   * latency regime (a frame's worth of objects): ONE CTA PER OBJECT, every thread owns a fixed set of
//     edges whose (i,j) offsets live in registers (n = 73), double-buffered staging with one
//     __syncthreads per object, fixed-order cross-warp sum (deterministic).
#include <cstdlib>
#include "dcd_common.cuh"

namespace dcd {

namespace {

// Stage one object's per-keypoint terms into shared memory.
template <int THREADS>
__device__ __forceinline__ float stage_object(const float* __restrict__ kps, const float* __restrict__ kps3d,
                                              const float* __restrict__ rot, const float* __restrict__ K,
                                              int64_t obj, int n, int flags, float4* kp_s) {
    const bool normalise = (flags & DCD_NORMALISE_2D) != 0;
    float cy = 0.f, fy = 1.f, b3 = 0.f;
    if (K != nullptr) {
        const float* Ko = K + obj * 12;
        if (normalise) { cy = __ldg(Ko + 6); fy = __ldg(Ko + 5); }
        if (flags & DCD_SUB_B3) b3 = __ldg(Ko + 11);
    }
    if ((int)threadIdx.x < ((n + 31) & ~31)) {   // only the warps that own keypoints evaluate sin/cos
        const float r = __ldg(rot + obj);
        const float s = sinf(r), c = cosf(r);
        for (int t = threadIdx.x; t < n; t += THREADS) {
            const float2 uv = __ldg(reinterpret_cast<const float2*>(kps + (obj * n + t) * 2));
            const float* p3 = kps3d + (obj * n + t) * 3;
            kp_s[t] = keypoint_terms(uv.y, __ldg(p3), __ldg(p3 + 1), __ldg(p3 + 2), s, c, normalise, cy, fy);
        }
    }
    return b3;
}

// ---------------------------------------------------------------------------------------------
// forward: per-edge depths and/or per-object mean
// NK > 0: compile-time keypoint count, (i,j) of the thread's edges held in registers.
// NK == 0: any n <= 256, (i,j) from a shared-memory table built once per CTA.
// ---------------------------------------------------------------------------------------------
template <int NK, int THREADS, bool WRITE_EDGES>
__global__ void __launch_bounds__(THREADS)
edge_solve_fwd_kernel(const float* __restrict__ kps, const float* __restrict__ kps3d,
                      const float* __restrict__ rot, const float* __restrict__ K,
                      int64_t N, int n_rt, float lo, float hi, int flags,
                      float* __restrict__ depth_edges, float* __restrict__ depth_mean) {
    constexpr int NWARP = THREADS / 32;
    const int n = NK > 0 ? NK : n_rt;
    const int E = n * (n - 1) / 2;
    constexpr int EPT = NK > 0 ? (NK * (NK - 1) / 2 + THREADS - 1) / THREADS : 1;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    float4* kp_s = reinterpret_cast<float4*>(smem_raw);                       // [2][n]
    float* part_s = reinterpret_cast<float*>(kp_s + 2 * n);                   // [2][NWARP]
    uint16_t* tab_s = reinterpret_cast<uint16_t*>(part_s + 2 * NWARP);        // [E] (generic only)

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    uint32_t pr[EPT];     // byte offsets (i*16) | (j*16) << 16 of this thread's edges
    if (NK > 0) {
#pragma unroll
        for (int m = 0; m < EPT; ++m) {
            const int e = tid + m * THREADS;
            int i = 0, j = 1;
            if (e < E) decode_edge(e, n, i, j);
            pr[m] = (uint32_t)(i * 16) | ((uint32_t)(j * 16) << 16);
        }
    } else {
        for (int e = tid; e < E; e += THREADS) {
            int i, j;
            decode_edge(e, n, i, j);
            tab_s[e] = (uint16_t)((i << 8) | j);
        }
        // visibility is ordered by the first __syncthreads of the object loop
    }

    int buf = 0;
    int64_t prev = -1;
    float prev_b3 = 0.f;
    (void)prev_b3;
    for (int64_t obj = blockIdx.x; obj < N; obj += gridDim.x) {
        float4* kp = kp_s + buf * n;
        const float b3 = stage_object<THREADS>(kps, kps3d, rot, K, obj, n, flags, kp);
        __syncthreads();
        if (depth_mean != nullptr && tid == 0 && prev >= 0) {
            float t = 0.f;
#pragma unroll
            for (int w = 0; w < NWARP; ++w) t += part_s[(buf ^ 1) * NWARP + w];
            depth_mean[prev] = __fdiv_rn(t, (float)E);
        }
        float acc = 0.f;
        const unsigned char* kpb = reinterpret_cast<const unsigned char*>(kp);
        float* out = WRITE_EDGES ? depth_edges + obj * (int64_t)E : nullptr;
        if (NK > 0) {
#pragma unroll
            for (int m = 0; m < EPT; ++m) {
                const int e = tid + m * THREADS;
                if (m < EPT - 1 || e < E) {
                    const float4 a = *reinterpret_cast<const float4*>(kpb + (pr[m] & 0xffffu));
                    const float4 b = *reinterpret_cast<const float4*>(kpb + (pr[m] >> 16));
                    const float z = edge_depth(a, b, lo, hi, b3);
                    if (WRITE_EDGES) __stcs(out + e, z);
                    acc += z;
                }
            }
        } else {
            for (int e = tid; e < E; e += THREADS) {
                const uint32_t p = tab_s[e];
                const float4 a = kp[p >> 8];
                const float4 b = kp[p & 0xffu];
                const float z = edge_depth(a, b, lo, hi, b3);
                if (WRITE_EDGES) __stcs(out + e, z);
                acc += z;
            }
        }
        if (depth_mean != nullptr) {
            acc = warp_sum(acc);
            if (lane == 0) part_s[buf * NWARP + warp] = acc;
        }
        prev = obj;
        buf ^= 1;
    }
    if (depth_mean != nullptr) {
        __syncthreads();
        if (tid == 0 && prev >= 0) {
            float t = 0.f;
#pragma unroll
            for (int w = 0; w < NWARP; ++w) t += part_s[(buf ^ 1) * NWARP + w];
            depth_mean[prev] = __fdiv_rn(t, (float)E);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// forward, throughput variant: ONE WARP PER OBJECT (used for large N).  No block barrier in the object loop
// (the per-object barrier of the CTA-per-object kernel is what bounds it at large N): a warp stages its
// object's keypoint terms in a private shared-memory slice, walks the E edges 32 at a time through a pair
// table shared by the CTA (coalesced 128-byte stores of the per-edge depths), and reduces the mean with
// shuffles.  The next object's raw inputs are prefetched into registers (n = 73: 3 keypoints per lane).
// ---------------------------------------------------------------------------------------------
template <int NK, int THREADS, bool WRITE_EDGES>
__global__ void __launch_bounds__(THREADS)
edge_solve_fwd_warp_kernel(const float* __restrict__ kps, const float* __restrict__ kps3d,
                           const float* __restrict__ rot, const float* __restrict__ K,
                           int64_t N, int n_rt, float lo, float hi, int flags,
                           float* __restrict__ depth_edges, float* __restrict__ depth_mean) {
    constexpr int NWARP = THREADS / 32;
    const int n = NK > 0 ? NK : n_rt;
    const int E = n * (n - 1) / 2;
    constexpr int KPL = NK > 0 ? (NK + 31) / 32 : 1;         // keypoints per lane held in registers (NK > 0)
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float4* kp_all = reinterpret_cast<float4*>(smem_raw);                     // [NWARP][n]
    uint32_t* tab_s = reinterpret_cast<uint32_t*>(kp_all + NWARP * n);        // [E] byte offsets (i*16) | (j*16) << 16
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
    const int64_t stride = (int64_t)gridDim.x * NWARP;

    float2 nx_uv[KPL];
    float nx_p[KPL][3];
    auto load_raw = [&](int64_t o) {
        if (NK == 0 || o >= N) return;
#pragma unroll
        for (int q = 0; q < KPL; ++q) {
            const int t = lane + q * 32;
            if (t < n) {
                nx_uv[q] = __ldg(reinterpret_cast<const float2*>(kps + (o * n + t) * 2));
                const float* p3 = kps3d + (o * n + t) * 3;
                nx_p[q][0] = __ldg(p3); nx_p[q][1] = __ldg(p3 + 1); nx_p[q][2] = __ldg(p3 + 2);
            }
        }
    };
    int64_t obj = (int64_t)blockIdx.x * NWARP + warp;
    load_raw(obj);
    for (; obj < N; obj += stride) {
        float cy = 0.f, fy = 1.f, b3 = 0.f;
        if (K != nullptr) {
            const float* Ko = K + obj * 12;
            if (normalise) { cy = __ldg(Ko + 6); fy = __ldg(Ko + 5); }
            if (flags & DCD_SUB_B3) b3 = __ldg(Ko + 11);
        }
        const float r = __ldg(rot + obj);
        const float sn = sinf(r), cs = cosf(r);
        if (NK > 0) {
#pragma unroll
            for (int q = 0; q < KPL; ++q) {
                const int t = lane + q * 32;
                if (t < n) kp[t] = keypoint_terms(nx_uv[q].y, nx_p[q][0], nx_p[q][1], nx_p[q][2], sn, cs, normalise, cy, fy);
            }
        } else {
            for (int t = lane; t < n; t += 32) {
                const float2 uv = __ldg(reinterpret_cast<const float2*>(kps + (obj * n + t) * 2));
                const float* p3 = kps3d + (obj * n + t) * 3;
                kp[t] = keypoint_terms(uv.y, __ldg(p3), __ldg(p3 + 1), __ldg(p3 + 2), sn, cs, normalise, cy, fy);
            }
        }
        __syncwarp();
        load_raw(obj + stride);                              // in flight during the edge loop
        float acc = 0.f;
        float* out = WRITE_EDGES ? depth_edges + obj * (int64_t)E : nullptr;
        int e = lane;
#pragma unroll 4
        for (; e + 96 < E; e += 128) {
            float z[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const uint32_t p = tab_s[e + 32 * u];
                const float4 a = *reinterpret_cast<const float4*>(kpb + (p & 0xffffu));
                const float4 b = *reinterpret_cast<const float4*>(kpb + (p >> 16));
                z[u] = edge_depth(a, b, lo, hi, b3);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (WRITE_EDGES) __stcs(out + e + 32 * u, z[u]);
                acc += z[u];
            }
        }
        for (; e < E; e += 32) {
            const uint32_t p = tab_s[e];
            const float4 a = *reinterpret_cast<const float4*>(kpb + (p & 0xffffu));
            const float4 b = *reinterpret_cast<const float4*>(kpb + (p >> 16));
            const float z = edge_depth(a, b, lo, hi, b3);
            if (WRITE_EDGES) __stcs(out + e, z);
            acc += z;
        }
        if (depth_mean != nullptr) {
            acc = warp_sum(acc);
            if (lane == 0) depth_mean[obj] = __fdiv_rn(acc, (float)E);
        }
        __syncwarp();                                        // all lanes done with kp before it is restaged
    }
}

// ---------------------------------------------------------------------------------------------
// forward, mean only, throughput variant (large N): a warp owns a GROUP of G consecutive objects.
//
// The edge loop is issue-bound (an IEEE-exact quotient costs 6 of the ~16 instructions of an edge), so this kernel
// removes everything else from it:
//   * per-keypoint terms as three separate arrays {v, Y, v*C} (12 B per keypoint; C itself is not needed forward);
//   * lane = one (object, keypoint i) SLOT; the G objects of a group are chosen so that G*n fills whole warps
//     (n = 73: G = 7, 511 of 512 slots busy), the slot's own terms sit in registers;
//   * circulant enumeration: every unordered pair is {i, (i + d) mod n} for exactly one d in 1..n/2, so the slot
//     walks d = 1 .. n/2 and reads its partner's terms at [i + d] of arrays whose first n/2 entries are repeated
//     after the n-th (no modulo).  Consecutive lanes read consecutive words (the per-object stride is congruent
//     to n modulo 32 so this also holds across objects of the group): 3 conflict-free LDS.32 per edge, offsets
//     are immediates, no pair table, no index arithmetic;
//   * |H| and |V| are symmetric in the endpoints (IEEE subtraction is antisymmetric), so every edge value is the
//     one of the reference's (i < j) evaluation, bit for bit; only the order of the sum differs (mean: 1e-6 bar);
//   * objects with a non-finite term take a separate loop with torch's NaN-propagating clamps.
// ---------------------------------------------------------------------------------------------
constexpr int GRP_WARPS = 4;
#ifndef BLK_PPS
#define BLK_PPS 4          // partner pairs per software-pipeline step of the blocked kernel (16 interleaved chains; 1 / 2 / 4 -> 0.164 / 0.165 / 0.157 ms)
#endif
__host__ __device__ constexpr int grp_stride(int n) { return n + 32 * ((n / 2 + 31) / 32); }   // == n (mod 32), >= n + n/2
__host__ __device__ constexpr int grp_warp_floats(int n, int G) { return 3 * G * grp_stride(n) + ((G * n + 31) & ~31) + 8 * G; }   // v, Y, vC | per-slot sums | 5 per-object scalars

template <int NK, int GC, bool FAST>
__global__ void __launch_bounds__(GRP_WARPS * 32)
edge_mean_group_kernel(const float* __restrict__ kps, const float* __restrict__ kps3d,
                       const float* __restrict__ rot, const float* __restrict__ K,
                       int64_t N, int n_rt, int G_rt, float lo, float hi, int flags,
                       float* __restrict__ depth_mean) {
    const int n = NK > 0 ? NK : n_rt;
    const int G = NK > 0 ? GC : G_rt;
    const int S = grp_stride(n);
    const int D = n / 2;                                     // offsets 1 .. D; for even n the last one covers i < n/2 only
    const int Dfull = (n - 1) / 2;
    const int E = n * (n - 1) / 2;
    extern __shared__ __align__(16) float grp_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* v_s = grp_smem + (size_t)warp * grp_warp_floats(n, G);
    float* Y_s = v_s + G * S;
    float* c_s = Y_s + G * S;
    float* part_s = c_s + G * S;                             // [G * n] per-slot sums
    float* sc_s = part_s + ((G * n + 31) & ~31);             // [5][G]: sin, cos, cy, fy, b3 of the group's objects
    const bool normalise = (flags & DCD_NORMALISE_2D) != 0;
    const int64_t ngroups = (N + G - 1) / G;

    for (int64_t grp = (int64_t)blockIdx.x * GRP_WARPS + warp; grp < ngroups; grp += (int64_t)gridDim.x * GRP_WARPS) {
        const int64_t obj0 = grp * G;
        const int gcount = (int)((N - obj0 < G) ? N - obj0 : G);
        const int slots = gcount * n;
        if (lane < gcount) {
            const int64_t obj = obj0 + lane;
            float cy = 0.f, fy = 1.f, b3 = 0.f;
            if (K != nullptr) {
                const float* Ko = K + obj * 12;
                if (normalise) { cy = __ldg(Ko + 6); fy = __ldg(Ko + 5); }
                if (flags & DCD_SUB_B3) b3 = __ldg(Ko + 11);
            }
            const float r = __ldg(rot + obj);
            sc_s[lane] = sinf(r);
            sc_s[G + lane] = cosf(r);
            sc_s[2 * G + lane] = cy;
            sc_s[3 * G + lane] = fy;
            sc_s[4 * G + lane] = b3;
        }
        __syncwarp();
        // ---- stage the group's keypoint terms: global keypoint index = obj0 * n + slot (coalesced)
        bool bad = false;
        const float* kv = kps + obj0 * n * 2 + 1;
        const float* k3 = kps3d + obj0 * n * 3;
#pragma unroll 4
        for (int s0 = 0; s0 < slots; s0 += 32) {
            const int s = s0 + lane;
            if (s < slots) {
                const int g = s / n, i = s - g * n;
                const float4 t = keypoint_terms(__ldg(kv + 2 * s), __ldg(k3 + 3 * s), __ldg(k3 + 3 * s + 1), __ldg(k3 + 3 * s + 2),
                                                sc_s[g], sc_s[G + g], normalise, sc_s[2 * G + g], sc_s[3 * G + g]);
                const int base = g * S + i;
                v_s[base] = t.x; Y_s[base] = t.y; c_s[base] = t.z;
                if (i < D) { v_s[base + n] = t.x; Y_s[base + n] = t.y; c_s[base + n] = t.z; }
                bad |= !(fabsf(t.x) + fabsf(t.y) + fabsf(t.z) <= 3.0e38f);
            }
        }
        bad = __any_sync(0xffffffffu, bad);
        __syncwarp();
        // ---- edges
        for (int s0 = 0; s0 < slots; s0 += 32) {
            const int s = s0 + lane;
            const bool active = s < slots;
            const int g = active ? s / n : 0, i = active ? s - g * n : 0;
            const float* pv = v_s + g * S + i;
            const float* pY = pv + G * S;
            const float* pc = pY + G * S;
            const float vi = pv[0], Yi = pY[0], ci = pc[0];
            float acc0 = 0.f, acc1 = 0.f;
            if (!bad) {
                // two partners per step on packed FP32 pairs (FADD2 / FMUL2 / FFMA2): 12 issue slots per edge instead of 17
                const float2 vi2 = make_float2(vi, vi), Yi2 = make_float2(Yi, Yi), ci2 = make_float2(ci, ci);
                float2 acc = make_float2(0.f, 0.f);
                int d = 1;
                if (NK > 0) {
#pragma unroll
                    for (; d + 1 <= Dfull; d += 2) {
                        const float2 vj = make_float2(pv[d], pv[d + 1]), Yj = make_float2(pY[d], pY[d + 1]), cj = make_float2(pc[d], pc[d + 1]);
                        acc = add2_rn(acc, FAST ? edge_quotient_fast2(vi2, Yi2, ci2, vj, Yj, cj, lo, hi)
                                                : edge_quotient_finite2(vi2, Yi2, ci2, vj, Yj, cj, lo, hi));
                    }
                } else {
#pragma unroll 2
                    for (; d + 1 <= Dfull; d += 2) {
                        const float2 vj = make_float2(pv[d], pv[d + 1]), Yj = make_float2(pY[d], pY[d + 1]), cj = make_float2(pc[d], pc[d + 1]);
                        acc = add2_rn(acc, FAST ? edge_quotient_fast2(vi2, Yi2, ci2, vj, Yj, cj, lo, hi)
                                                : edge_quotient_finite2(vi2, Yi2, ci2, vj, Yj, cj, lo, hi));
                    }
                }
                acc0 = acc.x;
                acc1 = acc.y;
                if (d <= Dfull) acc0 += FAST ? edge_quotient_fast(vi, Yi, ci, pv[d], pY[d], pc[d], lo, hi)
                                             : edge_quotient_finite(vi, Yi, ci, pv[d], pY[d], pc[d], lo, hi);
                if (D > Dfull && i < D) acc1 += FAST ? edge_quotient_fast(vi, Yi, ci, pv[D], pY[D], pc[D], lo, hi)
                                                     : edge_quotient_finite(vi, Yi, ci, pv[D], pY[D], pc[D], lo, hi);
            } else {
#pragma unroll 1
                for (int d = 1; d <= Dfull; ++d) acc0 += edge_quotient_ieee(vi, Yi, ci, pv[d], pY[d], pc[d], lo, hi);
                if (D > Dfull && i < D) acc1 += edge_quotient_ieee(vi, Yi, ci, pv[D], pY[D], pc[D], lo, hi);
            }
            if (active) part_s[s] = acc0 + acc1;
        }
        __syncwarp();
        // ---- per-object mean (fixed order: deterministic and independent of the group an object falls into)
        for (int g = 0; g < gcount; ++g) {
            float t = 0.f;
            for (int i = lane; i < n; i += 32) t += part_s[g * n + i];
            t = warp_sum(t);
            if (lane == 0) depth_mean[obj0 + g] = __fsub_rn(__fdiv_rn(t, (float)E), sc_s[4 * G + g]);
        }
        __syncwarp();                                        // all lanes done with the group's arrays before restaging
    }
}

// ---------------------------------------------------------------------------------------------
// forward, mean only, throughput variant for n = 1 (mod 4) keypoints (the reference's n = 73): register blocking on
// top of the circulant enumeration.  ncu on the kernel above (profiles/r02_edge_mean.md): 3 LDS.32 per edge keep the
// LSU at 55-66 % and, with ~4 warps per scheduler and one dependent chain per edge pair, the warps mostly wait on
// fixed-latency dependencies.  Here a lane OWNS 4 CONSECUTIVE keypoints i0 .. i0+3 (12 terms in registers) and walks
// the 39 partners i0+1 .. i0+39: every loaded partner serves up to four edges (0.8 LDS.32 per edge instead of 3) and
// the four edges are independent chains (4x the instruction-level parallelism).  Which (own, partner) combinations
// are circulant pairs (1 <= offset <= (n-1)/2) is a compile-time pattern, the same for every lane, so nothing is
// masked at run time: per lane 70 packed pairs + 4 single edges.  The (n-1)/4 lanes of an object cover keypoints
// 0 .. n-2; the last keypoint's (n-1)/2 edges (partners 0 .. (n-1)/2-1) are dealt two per lane.  Keypoint terms are
// stored interleaved by (index mod 4) so that consecutive lanes read consecutive words for every partner, and the
// per-object stride is congruent to the lanes per object modulo 32: conflict-free across the objects of a group.
// Every edge value is still bit-identical to the reference's; sum order per object is fixed (deterministic,
// independent of the group an object falls into).
// ---------------------------------------------------------------------------------------------
template <int NK>
struct BlkGeom {
    static_assert(NK % 4 == 1 && NK >= 9, "the blocked kernel needs n = 1 (mod 4)");
    static constexpr int LPO = (NK - 1) / 4;                 // lanes per object (18)
    static constexpr int D = (NK - 1) / 2;                   // circulant offsets 1 .. D (36)
    static constexpr int NPART = D + 3;                      // partners i0+1 .. i0+NPART of a lane's four keypoints (39)
    static constexpr int S4 = (4 * (LPO - 1) + NPART) / 4 + 1;                        // entries per residue class (27)
    static constexpr int OS = 4 * S4 + ((LPO - 4 * S4) % 32 + 32) % 32;               // object stride == LPO (mod 32) (114)
    static constexpr int NDUP = 4 * (LPO - 1) + NPART - NK + 1;                       // keypoints repeated after the n-th (35)
};
// per warp: terms v, Y, vC [G][OS] | per-lane sums | 5 per-object scalars | raw inputs of the NEXT group (v pixel row, X Y Z)
template <int NK, int G>
__host__ __device__ constexpr int blk_warp_floats() {
    return 3 * G * BlkGeom<NK>::OS + ((G * BlkGeom<NK>::LPO + 31) & ~31) + 8 * G + 4 * G * NK;
}
__device__ __forceinline__ void cp_async4(float* dst_smem, const float* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit_wait_all() {
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}

template <int NK, int G, bool FAST>
__global__ void __launch_bounds__(GRP_WARPS * 32)
edge_mean_block_kernel(const float* __restrict__ kps, const float* __restrict__ kps3d,
                       const float* __restrict__ rot, const float* __restrict__ K,
                       int64_t N, float lo, float hi, int flags, float* __restrict__ depth_mean) {
    using Gm = BlkGeom<NK>;
    constexpr int LPO = Gm::LPO, D = Gm::D, NPART = Gm::NPART, S4 = Gm::S4, OS = Gm::OS;
    constexpr int E = NK * (NK - 1) / 2;
    extern __shared__ __align__(16) float blk_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* v_s = blk_smem + (size_t)warp * blk_warp_floats<NK, G>();
    float* Y_s = v_s + G * OS;
    float* c_s = Y_s + G * OS;
    float* part_s = c_s + G * OS;                            // [G * LPO] per-lane sums
    float* sc_s = part_s + ((G * LPO + 31) & ~31);           // [5][G]: sin, cos, cy, fy, b3
    float* rawv_s = sc_s + 8 * G;                            // [G * NK] pixel row of every keypoint of the next group
    float* raw3_s = rawv_s + G * NK;                         // [G * NK * 3] its template points
    const bool normalise = (flags & DCD_NORMALISE_2D) != 0;
    const int64_t ngroups = (N + G - 1) / G;
    const int64_t gstride = (int64_t)gridDim.x * GRP_WARPS;
    auto pos = [](int e) { return (e & 3) * S4 + (e >> 2); };   // interleaved position of element e inside an object
    // asynchronous copy of a group's raw inputs (LDGSTS, 4 bytes per lane and instruction, fully coalesced): issued one group
    // ahead, so the DRAM latency is covered by the previous group's edge loop instead of stalling the warp
    auto prefetch = [&](int64_t g0) {
        if (g0 >= ngroups) return;
        const int64_t o0 = g0 * G;
        const int cnt = (int)((N - o0 < G) ? N - o0 : G) * NK;
        const float* kv = kps + o0 * NK * 2 + 1;
        const float* k3 = kps3d + o0 * NK * 3;
        for (int s = lane; s < cnt; s += 32) cp_async4(rawv_s + s, kv + 2 * s);
        for (int s = lane; s < 3 * cnt; s += 32) cp_async4(raw3_s + s, k3 + s);
    };
    prefetch((int64_t)blockIdx.x * GRP_WARPS + warp);

    for (int64_t grp = (int64_t)blockIdx.x * GRP_WARPS + warp; grp < ngroups; grp += gstride) {
        const int64_t obj0 = grp * G;
        const int gcount = (int)((N - obj0 < G) ? N - obj0 : G);
        if (lane < gcount) {
            const int64_t obj = obj0 + lane;
            float cy = 0.f, fy = 1.f, b3 = 0.f;
            if (K != nullptr) {
                const float* Ko = K + obj * 12;
                if (normalise) { cy = __ldg(Ko + 6); fy = __ldg(Ko + 5); }
                if (flags & DCD_SUB_B3) b3 = __ldg(Ko + 11);
            }
            const float r = __ldg(rot + obj);
            sc_s[lane] = sinf(r);
            sc_s[G + lane] = cosf(r);
            sc_s[2 * G + lane] = cy;
            sc_s[3 * G + lane] = fy;
            sc_s[4 * G + lane] = b3;
        }
        __syncwarp();
        cp_async_commit_wait_all();                          // this group's raw inputs have landed
        __syncwarp();
        // ---- keypoint terms of the group from the raw staging buffer
        bool bad = false;
        const int slots = gcount * NK;
#pragma unroll 4
        for (int s0 = 0; s0 < slots; s0 += 32) {
            const int s = s0 + lane;
            if (s < slots) {
                const int g = s / NK, i = s - g * NK;
                const float4 t = keypoint_terms(rawv_s[s], raw3_s[3 * s], raw3_s[3 * s + 1], raw3_s[3 * s + 2],
                                                sc_s[g], sc_s[G + g], normalise, sc_s[2 * G + g], sc_s[3 * G + g]);
                const int p = g * OS + pos(i);
                v_s[p] = t.x; Y_s[p] = t.y; c_s[p] = t.z;
                if (i < Gm::NDUP) {
                    const int p2 = g * OS + pos(i + NK);
                    v_s[p2] = t.x; Y_s[p2] = t.y; c_s[p2] = t.z;
                }
                bad |= !(fabsf(t.x) + fabsf(t.y) + fabsf(t.z) <= 3.0e38f);
            }
        }
        bad = __any_sync(0xffffffffu, bad);
        __syncwarp();
        prefetch(grp + gstride);                             // the raw buffer is free again: fetch the next group behind the edge loop
        // ---- edges: lane = (object g, quad q), keypoints 4q .. 4q+3
        const int lanes = gcount * LPO;
        for (int L0 = 0; L0 < lanes; L0 += 32) {
            const int L = L0 + lane;
            const bool active = L < lanes;
            const int g = active ? L / LPO : 0, q = active ? L - g * LPO : 0;
            const float* pv = v_s + g * OS + q;              // element 4q + t sits at pv[(t & 3) * S4 + (t >> 2)]
            const float* pY = pv + G * OS;
            const float* pc = pY + G * OS;
            float total;
            if (!bad) {
                float2 ov[4], oY[4], oc[4];                  // own terms, duplicated into both halves of a packed pair
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                    const float x = pv[a * S4], y = pY[a * S4], z = pc[a * S4];
                    ov[a] = make_float2(x, x); oY[a] = make_float2(y, y); oc[a] = make_float2(z, z);
                }
                float2 acc0 = make_float2(0.f, 0.f), acc1 = make_float2(0.f, 0.f);
                float accs = 0.f;
                auto partner_pair = [&](int tp, float2& vj, float2& Yj, float2& cj) {      // partners tp, tp + 1 (tp + 1 <= NPART)
                    const int o0 = (tp & 3) * S4 + (tp >> 2), o1 = ((tp + 1) & 3) * S4 + ((tp + 1) >> 2);
                    vj = make_float2(pv[o0], pv[o1]); Yj = make_float2(pY[o0], pY[o1]); cj = make_float2(pc[o0], pc[o1]);
                };
                // partner pairs (tp, tp + 1) with tp = TP0, TP0 + 2, ..., TP1 pair with all four own keypoints: software-
                // pipelined, the reciprocals of step k + 1 are issued before step k is refined and accumulated
                constexpr int TP0 = 5, TP1 = (D - 1) | 1;                               // odd tp, tp >= 4 and tp + 1 <= D
                constexpr int PPS = BLK_PPS;                                              // partner pairs per pipeline step
                constexpr int NSTEP = ((TP1 - TP0) / 2 + 1) / PPS;                      // full steps; leftover pairs go with the ends
                constexpr int TPE = TP0 + 2 * PPS * NSTEP;                               // first tp not covered by the pipeline
                {
                    EdgeStage<4 * PPS> cur, nxt;
                    float2 vj[PPS], Yj[PPS], cj[PPS];
#pragma unroll
                    for (int p = 0; p < PPS; ++p) partner_pair(TP0 + 2 * p, vj[p], Yj[p], cj[p]);
                    edge_stage_a<4 * PPS>(ov, oY, oc, vj, Yj, cj, cur);
#pragma unroll
                    for (int st = 0; st < NSTEP; ++st) {
                        if (st + 1 < NSTEP) {
#pragma unroll
                            for (int p = 0; p < PPS; ++p) partner_pair(TP0 + 2 * PPS * (st + 1) + 2 * p, vj[p], Yj[p], cj[p]);
                            edge_stage_a<4 * PPS>(ov, oY, oc, vj, Yj, cj, nxt);
                        }
                        float2 z[4 * PPS];
                        edge_stage_b<FAST, 4 * PPS>(cur, lo, hi, z);
#pragma unroll
                        for (int w = 0; w < 4 * PPS; w += 2) {
                            acc0 = add2_rn(acc0, z[w]);
                            acc1 = add2_rn(acc1, z[w + 1]);
                        }
                        if (st + 1 < NSTEP) cur = nxt;
                    }
                }
                // the partial partner pairs at both ends of the window
#pragma unroll
                for (int tp = 1; tp <= NPART; tp += 2) {
                    if (tp >= TP0 && tp < TPE) continue;
                    const bool has1 = tp + 1 <= NPART;
                    const int o0 = (tp & 3) * S4 + (tp >> 2), o1 = has1 ? ((tp + 1) & 3) * S4 + ((tp + 1) >> 2) : o0;
                    const float2 vj = make_float2(pv[o0], pv[o1]), Yj = make_float2(pY[o0], pY[o1]), cj = make_float2(pc[o0], pc[o1]);
#pragma unroll
                    for (int a = 0; a < 4; ++a) {
                        const int d0 = tp - a, d1 = tp + 1 - a;
                        const bool ok0 = d0 >= 1 && d0 <= D, ok1 = has1 && d1 >= 1 && d1 <= D;
                        if (ok0 && ok1) {
                            const float2 z = FAST ? edge_quotient_fast2(ov[a], oY[a], oc[a], vj, Yj, cj, lo, hi)
                                                  : edge_quotient_finite2(ov[a], oY[a], oc[a], vj, Yj, cj, lo, hi);
                            if (a & 1) acc1 = add2_rn(acc1, z); else acc0 = add2_rn(acc0, z);
                        } else if (ok0) {
                            accs += FAST ? edge_quotient_fast(ov[a].x, oY[a].x, oc[a].x, vj.x, Yj.x, cj.x, lo, hi)
                                         : edge_quotient_finite(ov[a].x, oY[a].x, oc[a].x, vj.x, Yj.x, cj.x, lo, hi);
                        } else if (ok1) {
                            accs += FAST ? edge_quotient_fast(ov[a].x, oY[a].x, oc[a].x, vj.y, Yj.y, cj.y, lo, hi)
                                         : edge_quotient_finite(ov[a].x, oY[a].x, oc[a].x, vj.y, Yj.y, cj.y, lo, hi);
                        }
                    }
                }
                // the last keypoint (NK - 1) against partners 2q, 2q + 1
                {
                    const float* bv = v_s + g * OS;
                    const float* bY = bv + G * OS;
                    const float* bc = bY + G * OS;
                    constexpr int pl = ((NK - 1) & 3) * S4 + ((NK - 1) >> 2);
                    const int e0 = 2 * q, e1 = 2 * q + 1;
                    const int p0 = (e0 & 3) * S4 + (e0 >> 2), p1 = (e1 & 3) * S4 + (e1 >> 2);
                    const float xl = bv[pl], yl = bY[pl], zl = bc[pl];
                    const float2 z = FAST ? edge_quotient_fast2(make_float2(xl, xl), make_float2(yl, yl), make_float2(zl, zl),
                                                                make_float2(bv[p0], bv[p1]), make_float2(bY[p0], bY[p1]),
                                                                make_float2(bc[p0], bc[p1]), lo, hi)
                                          : edge_quotient_finite2(make_float2(xl, xl), make_float2(yl, yl), make_float2(zl, zl),
                                                                  make_float2(bv[p0], bv[p1]), make_float2(bY[p0], bY[p1]),
                                                                  make_float2(bc[p0], bc[p1]), lo, hi);
                    acc0 = add2_rn(acc0, z);
                }
                total = ((acc0.x + acc0.y) + (acc1.x + acc1.y)) + accs;
            } else {
                // non-finite terms somewhere in the group: the same edges with torch's NaN-propagating clamps
                const float* bv = v_s + g * OS;
                const float* bY = bv + G * OS;
                const float* bc = bY + G * OS;
                float acc = 0.f;
#pragma unroll 1
                for (int a = 0; a < 4; ++a) {
                    const int pa = pos(4 * q + a);
#pragma unroll 1
                    for (int d = 1; d <= D; ++d) {
                        const int pb = pos(4 * q + a + d);
                        acc += edge_quotient_ieee(bv[pa], bY[pa], bc[pa], bv[pb], bY[pb], bc[pb], lo, hi);
                    }
                }
                const int pl = pos(NK - 1);
#pragma unroll 1
                for (int k = 0; k < 2; ++k) {
                    const int pb = pos(2 * q + k);
                    acc += edge_quotient_ieee(bv[pl], bY[pl], bc[pl], bv[pb], bY[pb], bc[pb], lo, hi);
                }
                total = acc;
            }
            if (active) part_s[L] = total;
        }
        __syncwarp();
        // ---- per-object mean: the LPO lane sums of an object in fixed order
        if (lane < gcount) {
            float t = 0.f;
#pragma unroll
            for (int k = 0; k < LPO; ++k) t += part_s[lane * LPO + k];
            depth_mean[obj0 + lane] = __fsub_rn(__fdiv_rn(t, (float)E), sc_s[4 * G + lane]);
        }
        __syncwarp();                                        // all lanes done with the group's arrays before restaging
    }
}

// objects per group: the G in 1..8 that fills the warps of a group best within ~12 KB of shared memory per warp
int grp_pick_G(int n) {
    int best = 1;
    double best_eff = 0.0;
    for (int G = 1; G <= 8; ++G) {
        if (G > 1 && (size_t)grp_warp_floats(n, G) * sizeof(float) > 14 * 1024) break;
        const int slots = G * n, rounds = (slots + 31) / 32;
        const double eff = (double)slots / (32.0 * rounds);
        if (eff > best_eff + 1e-9) { best_eff = eff; best = G; }
    }
    return best;
}

// ---------------------------------------------------------------------------------------------
// selection, general k (k > 2048; the reference's k = 1500 runs edge_select.cu): top-k edges by |V| sorted
// (|V| desc, edge id asc) + their depths / pair masks / mean.  One CTA per object; bitonic sort of all (key, id)
// pairs in shared memory.
// ---------------------------------------------------------------------------------------------
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
edge_select_kernel(const float* __restrict__ kps, const float* __restrict__ kps3d,
                   const float* __restrict__ rot, const float* __restrict__ K,
                   const uint8_t* __restrict__ kpt_mask, int64_t N, int n, int P, int k,
                   float lo, float hi, int flags,
                   int64_t* __restrict__ idx_out, float* __restrict__ depth_sel,
                   float* __restrict__ mask_sel, float* __restrict__ depth_mean) {
    constexpr int NWARP = THREADS / 32;
    const int E = n * (n - 1) / 2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint32_t* key_s = reinterpret_cast<uint32_t*>(smem_raw);                  // [P]
    float4* kp_s = reinterpret_cast<float4*>(key_s + P);                      // [n]
    float* red_s = reinterpret_cast<float*>(kp_s + n);                        // [NWARP]
    uint16_t* id_s = reinterpret_cast<uint16_t*>(red_s + NWARP);              // [P]
    uint8_t* m_s = reinterpret_cast<uint8_t*>(id_s + P);                      // [n]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    for (int64_t obj = blockIdx.x; obj < N; obj += gridDim.x) {
        __syncthreads();   // previous object's readers are done with shared memory
        const float b3 = stage_object<THREADS>(kps, kps3d, rot, K, obj, n, flags, kp_s);
        if (kpt_mask != nullptr)
            for (int t = tid; t < n; t += THREADS) m_s[t] = kpt_mask[obj * n + t];
        __syncthreads();
        // keys: bit pattern of |v_i - v_j| (non-negative floats order like unsigned integers)
        for (int e = tid; e < P; e += THREADS) {
            uint32_t key = 0u;
            uint16_t id = 0xffffu;
            if (e < E) {
                int i, j;
                decode_edge(e, n, i, j);
                key = __float_as_uint(fabsf(__fsub_rn(kp_s[i].x, kp_s[j].x)));
                id = (uint16_t)e;
            }
            key_s[e] = key;
            id_s[e] = id;
        }
        // bitonic sort, descending by (key, -id)
        for (int size = 2; size <= P; size <<= 1) {
            for (int stride = size >> 1; stride > 0; stride >>= 1) {
                __syncthreads();
                for (int t = tid; t < (P >> 1); t += THREADS) {
                    const int a = 2 * t - (t & (stride - 1));
                    const int b = a + stride;
                    const uint32_t ka = key_s[a], kb = key_s[b];
                    const uint16_t ia = id_s[a], ib = id_s[b];
                    const bool a_first = (ka > kb) || (ka == kb && ia < ib);
                    const bool desc = (a & size) == 0;
                    if (a_first != desc) {
                        key_s[a] = kb; key_s[b] = ka;
                        id_s[a] = ib; id_s[b] = ia;
                    }
                }
            }
        }
        __syncthreads();
        float acc = 0.f;
        for (int r = tid; r < k; r += THREADS) {
            const int e = id_s[r];
            int i, j;
            decode_edge(e, n, i, j);
            const float z = edge_depth(kp_s[i], kp_s[j], lo, hi, b3);
            idx_out[obj * k + r] = (int64_t)e;
            if (depth_sel != nullptr) depth_sel[obj * k + r] = z;
            if (mask_sel != nullptr) mask_sel[obj * k + r] = (m_s[i] != 0 && m_s[j] != 0) ? 1.f : 0.f;
            acc += z;
        }
        if (depth_mean != nullptr) {
            acc = warp_sum(acc);
            if (lane == 0) red_s[warp] = acc;
            __syncthreads();
            if (tid == 0) {
                float t = 0.f;
#pragma unroll
                for (int w = 0; w < NWARP; ++w) t += red_s[w];
                depth_mean[obj] = __fdiv_rn(t, (float)k);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// backward: per-keypoint gather over the n-1 incident edges (deterministic, no atomics)
// ---------------------------------------------------------------------------------------------
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
edge_solve_bwd_kernel(const float* __restrict__ kps, const float* __restrict__ kps3d,
                      const float* __restrict__ rot, const float* __restrict__ K,
                      int64_t N, int n, float lo, float hi, int flags,
                      const int64_t* __restrict__ idx, int k,
                      const float* __restrict__ grad_depth, const float* __restrict__ grad_mean,
                      float* __restrict__ grad_kps, float* __restrict__ grad_kps3d) {
    constexpr int NWARP = THREADS / 32;
    const int E = n * (n - 1) / 2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float4* kp_s = reinterpret_cast<float4*>(smem_raw);                       // [n]
    float* g_s = reinterpret_cast<float*>(kp_s + n);                          // [E] (only when idx != null)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool normalise = (flags & DCD_NORMALISE_2D) != 0;

    for (int64_t obj = blockIdx.x; obj < N; obj += gridDim.x) {
        __syncthreads();
        stage_object<THREADS>(kps, kps3d, rot, K, obj, n, flags, kp_s);
        const float r = __ldg(rot + obj);
        const float sn = sinf(r), cs = cosf(r);
        const float fy = (normalise && K != nullptr) ? __ldg(K + obj * 12 + 5) : 1.f;
        const float gm = grad_mean != nullptr ? __fdiv_rn(__ldg(grad_mean + obj), (float)(idx != nullptr ? k : E)) : 0.f;
        if (idx != nullptr) {
            for (int e = tid; e < E; e += THREADS) g_s[e] = 0.f;
            __syncthreads();
            for (int q = tid; q < k; q += THREADS) {
                const float g = grad_depth != nullptr ? __ldg(grad_depth + obj * k + q) : 0.f;
                g_s[(int)idx[obj * k + q]] = g + gm;
            }
        }
        __syncthreads();
        const float* gd = (idx == nullptr && grad_depth != nullptr) ? grad_depth + obj * (int64_t)E : nullptr;
        for (int kk = warp; kk < n; kk += NWARP) {
            const float4 me = kp_s[kk];
            float gH, gV;
            keypoint_edge_grad(kp_s, me, kk, n, lane, lo, hi, [&](int e) {
                if (idx != nullptr) return g_s[e];
                return (gd != nullptr ? __ldg(gd + e) : 0.f) + gm;
            }, gH, gV);
            if (lane == 0) {
                const float gv = gV + gH * me.w;          // d/dv: V and the v*C term of H
                const float gC = gH * me.x;               // d/dC
                float2 o2 = make_float2(0.f, normalise ? __fdiv_rn(gv, fy) : gv);
                *reinterpret_cast<float2*>(grad_kps + (obj * n + kk) * 2) = o2;
                float* o3 = grad_kps3d + (obj * n + kk) * 3;
                o3[0] = gC * sn;
                o3[1] = gH;
                o3[2] = -gC * cs;
            }
        }
    }
}

int next_pow2(int x) {
    int p = 1;
    while (p < x) p <<= 1;
    return p;
}

}  // namespace

int device_sm_count() {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms > 0 ? sms : 148;
}

int launch_edge_solve_fwd(const float* kps, const float* kps3d, const float* rot, const float* K,
                          int64_t N, int n, float lo, float hi, int flags,
                          float* depth_edges, float* depth_mean, cudaStream_t st) {
    constexpr int T = 256;
    const int E = n * (n - 1) / 2;
    const int sms = device_sm_count();
    // throughput regime, mean only: groups of objects per warp, circulant edge enumeration (edge_mean_group_kernel)
    if (N >= (int64_t)sms * 16 && depth_edges == nullptr) {
        const int G = n == 73 ? 7 : grp_pick_G(n);
        const size_t gsmem = (size_t)GRP_WARPS * grp_warp_floats(n, G) * sizeof(float);
        const int64_t ngroups = (N + G - 1) / G;
        const int64_t want = (ngroups + GRP_WARPS - 1) / GRP_WARPS;
        int per_sm = (int)((227 * 1024) / (gsmem + 1024));
        if (per_sm > 8) per_sm = 8;
        if (per_sm < 1) return DCD_E_UNSUPPORTED;
        const int64_t cap = (int64_t)sms * per_sm;
        const int grid = (int)(want < cap ? want : cap);
        const bool fast = (flags & DCD_FAST_QUOTIENT) != 0;
#define DCD_LAUNCH_GRP(NKV, GCV, FASTV)                                                                                       \
    do {                                                                                                                      \
        if (gsmem > 48 * 1024)                                                                                                \
            cudaFuncSetAttribute(edge_mean_group_kernel<NKV, GCV, FASTV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gsmem); \
        edge_mean_group_kernel<NKV, GCV, FASTV><<<grid, GRP_WARPS * 32, gsmem, st>>>(kps, kps3d, rot, K, N, n, G, lo, hi, flags, \
                                                                                      depth_mean);                           \
    } while (0)
        if (n == 73) {
            // n = 1 (mod 4): the register-blocked kernel; G objects (18 G lanes) per warp group.  More objects fill the last
            // round's lanes better (G = 7: 126 of 128 lanes, G = 5: 90 of 96), fewer leave shared memory for more resident
            // warps; measured on B200 (96 406 objects): G = 3 / 5 / 7 -> 0.179 / 0.164 / 0.167 ms.
            int BG = 5;
            if (const char* e = getenv("DCD_B200_BLOCK_G")) BG = atoi(e);      // tuning aid (profiles/): 3, 5 or 7
#define DCD_LAUNCH_BLK(GV)                                                                                                  \
    do {                                                                                                                    \
        const size_t bsmem = (size_t)GRP_WARPS * blk_warp_floats<73, GV>() * sizeof(float);                                 \
        const int64_t bgroups = (N + GV - 1) / GV, bwant = (bgroups + GRP_WARPS - 1) / GRP_WARPS;                           \
        int bper = (int)((227 * 1024) / (bsmem + 1024));                                                                    \
        if (bper > 8) bper = 8;                                                                                             \
        const int64_t bcap = (int64_t)sms * bper;                                                                           \
        const int bgrid = (int)(bwant < bcap ? bwant : bcap);                                                               \
        if (fast) {                                                                                                         \
            cudaFuncSetAttribute(edge_mean_block_kernel<73, GV, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bsmem);  \
            edge_mean_block_kernel<73, GV, true><<<bgrid, GRP_WARPS * 32, bsmem, st>>>(kps, kps3d, rot, K, N, lo, hi, flags, depth_mean); \
        } else {                                                                                                            \
            cudaFuncSetAttribute(edge_mean_block_kernel<73, GV, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bsmem); \
            edge_mean_block_kernel<73, GV, false><<<bgrid, GRP_WARPS * 32, bsmem, st>>>(kps, kps3d, rot, K, N, lo, hi, flags, depth_mean); \
        }                                                                                                                   \
    } while (0)
            if (BG == 3) DCD_LAUNCH_BLK(3); else if (BG == 5) DCD_LAUNCH_BLK(5); else DCD_LAUNCH_BLK(7);
#undef DCD_LAUNCH_BLK
        } else if (false) {
            if (fast) DCD_LAUNCH_GRP(73, 7, true); else DCD_LAUNCH_GRP(73, 7, false);
        } else {
            if (fast) DCD_LAUNCH_GRP(0, 0, true); else DCD_LAUNCH_GRP(0, 0, false);
        }
#undef DCD_LAUNCH_GRP
        DCD_CHECK_LAUNCH();
        return DCD_OK;
    }
    // throughput regime with per-edge output: one warp per object (no per-object block barrier)
    const size_t wsmem = (size_t)(T / 32) * n * sizeof(float4) + (size_t)E * sizeof(uint32_t);
    if (N >= (int64_t)sms * 16 && wsmem <= 100 * 1024) {
        const int64_t want = (N + T / 32 - 1) / (T / 32), cap = (int64_t)sms * 6;
        const int grid = (int)(want < cap ? want : cap);
#define DCD_LAUNCH_WARP(NKV, WE)                                                                                   \
    do {                                                                                                           \
        if (wsmem > 48 * 1024)                                                                                     \
            cudaFuncSetAttribute(edge_solve_fwd_warp_kernel<NKV, T, WE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem); \
        edge_solve_fwd_warp_kernel<NKV, T, WE><<<grid, T, wsmem, st>>>(kps, kps3d, rot, K, N, n, lo, hi, flags,    \
                                                                       depth_edges, depth_mean);                   \
    } while (0)
        if (n == 73) {
            if (depth_edges) DCD_LAUNCH_WARP(73, true); else DCD_LAUNCH_WARP(73, false);
        } else {
            if (depth_edges) DCD_LAUNCH_WARP(0, true); else DCD_LAUNCH_WARP(0, false);
        }
#undef DCD_LAUNCH_WARP
        DCD_CHECK_LAUNCH();
        return DCD_OK;
    }
    // latency regime (a frame's worth of objects): one CTA per object
    const int64_t max_grid = (int64_t)sms * 8;
    const int grid = (int)(N < max_grid ? N : max_grid);
    size_t smem = (size_t)2 * n * sizeof(float4) + 2 * (T / 32) * sizeof(float);
    if (n == 73) {
        if (depth_edges)
            edge_solve_fwd_kernel<73, T, true><<<grid, T, smem, st>>>(kps, kps3d, rot, K, N, n, lo, hi, flags, depth_edges, depth_mean);
        else
            edge_solve_fwd_kernel<73, T, false><<<grid, T, smem, st>>>(kps, kps3d, rot, K, N, n, lo, hi, flags, depth_edges, depth_mean);
    } else {
        smem += (size_t)E * sizeof(uint16_t);
        if (depth_edges) {
            if (smem > 48 * 1024) cudaFuncSetAttribute(edge_solve_fwd_kernel<0, T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            edge_solve_fwd_kernel<0, T, true><<<grid, T, smem, st>>>(kps, kps3d, rot, K, N, n, lo, hi, flags, depth_edges, depth_mean);
        } else {
            if (smem > 48 * 1024) cudaFuncSetAttribute(edge_solve_fwd_kernel<0, T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            edge_solve_fwd_kernel<0, T, false><<<grid, T, smem, st>>>(kps, kps3d, rot, K, N, n, lo, hi, flags, depth_edges, depth_mean);
        }
    }
    DCD_CHECK_LAUNCH();
    return DCD_OK;
}

int launch_edge_select_bitonic(const float* kps, const float* kps3d, const float* rot, const float* K,
                       const uint8_t* kpt_mask, int64_t N, int n, int k, float lo, float hi, int flags,
                       int64_t* idx_out, float* depth_sel, float* mask_sel, float* depth_mean, cudaStream_t st) {
    constexpr int T = 256;
    const int E = n * (n - 1) / 2;
    const int P = next_pow2(E < 2 ? 2 : E);
    size_t smem = (size_t)P * 4 + (size_t)n * 16 + (T / 32) * 4 + (size_t)P * 2 + (size_t)((n + 15) & ~15);
    if (smem > 227 * 1024) return DCD_E_UNSUPPORTED;
    if (smem > 48 * 1024) cudaFuncSetAttribute(edge_select_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int64_t max_grid = (int64_t)device_sm_count() * 8;
    const int grid = (int)(N < max_grid ? N : max_grid);
    edge_select_kernel<T><<<grid, T, smem, st>>>(kps, kps3d, rot, K, kpt_mask, N, n, P, k, lo, hi, flags,
                                                 idx_out, depth_sel, mask_sel, depth_mean);
    DCD_CHECK_LAUNCH();
    return DCD_OK;
}

int launch_edge_solve_bwd(const float* kps, const float* kps3d, const float* rot, const float* K,
                          int64_t N, int n, float lo, float hi, int flags, const int64_t* idx, int k,
                          const float* grad_depth, const float* grad_mean, float* grad_kps, float* grad_kps3d,
                          cudaStream_t st) {
    constexpr int T = 256;
    const int E = n * (n - 1) / 2;
    size_t smem = (size_t)n * 16 + (idx != nullptr ? (size_t)E * 4 : 0);
    if (smem > 227 * 1024) return DCD_E_UNSUPPORTED;
    if (smem > 48 * 1024) cudaFuncSetAttribute(edge_solve_bwd_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int64_t max_grid = (int64_t)device_sm_count() * 8;
    const int grid = (int)(N < max_grid ? N : max_grid);
    edge_solve_bwd_kernel<T><<<grid, T, smem, st>>>(kps, kps3d, rot, K, N, n, lo, hi, flags, idx, k,
                                                    grad_depth, grad_mean, grad_kps, grad_kps3d);
    DCD_CHECK_LAUNCH();
    return DCD_OK;
}

}  // namespace dcd
