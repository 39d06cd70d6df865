// Correspondence branch of GMW, forward (SURVEY 8f row N1): pairwise feature distances + entropy-regularised transport.
//   f4n, f6n  = L2-normalised final edge features of the two nets                      GMW/model/model.py:176-177
//   M[i][j]   = sqrt(max((|c_j|^2 - 2 a_i.c_j) + |a_i|^2, 1e-30))                      model.py:17-36 (pairwiseL2Dist)
//   K         = exp(-lambda * min(M, 5));  u = r;  repeat <= max_iter:                  GMW/lib/optimal_transport.py:52-72
//                   stop when |u - u_prev| <= tol everywhere (whole batch);  u = r / (K (c / (K^T u)))
//   v = c / (K^T u);  P = (u * K) * v^T          with r = 1/E, c = 1/E                  model.py:186-191
// Both training and validation loops consume P only through correspondenceLoss(P, eye) = sum(P) - 2 trace(P)
// (GMW/main.py:456-457,526-527, lib/losses.py:22-26,115-119), so the kernels also return those two sums per object and
// P itself is optional.  The backward lives in gmw_transport_bwd.cu.
//
// K is built on the tensor cores (transport_k_tc_kernel) and kept as E x E FP32 (27.6 MB per object at n = 73) in the caller's
// workspace; every Sinkhorn iteration streams it twice
// (column pass K^T u with the rows split over 16 partial sums, row pass K w with a warp per row), deterministic: no
// atomics on floating-point data.  The convergence test is a device flag, later iterations become no-ops.
#include <cstdlib>
#include "gmw_tc_common.cuh"

namespace dcd {
namespace {

constexpr int TP_CHUNKS = 16;       // row chunks of the column pass

// per-edge norms of the final features and the squared norms of the normalised vectors (model.py:176-177, :27-28)
__global__ void __launch_bounds__(256) transport_norm_kernel(const float* __restrict__ feat4, const float* __restrict__ feat6,
                                                             int64_t N, int E, float* __restrict__ nrm /* [N][4][E] */) {
    const int64_t obj = blockIdx.y;
    const int e = blockIdx.x * 256 + threadIdx.x;
    if (e >= E) return;
    const float* X4 = feat4 + obj * (int64_t)CH * E + e;
    const float* X6 = feat6 + obj * (int64_t)CH * E + e;
    float n4 = 0.f, n6 = 0.f;
    for (int c = 0; c < CH; ++c) {
        const float x4 = X4[(int64_t)c * E], x6 = X6[(int64_t)c * E];
        n4 = fmaf(x4, x4, n4);
        n6 = fmaf(x6, x6, n6);
    }
    n4 = fmaxf(sqrtf(n4), 1e-12f);
    n6 = fmaxf(sqrtf(n6), 1e-12f);
    float a2 = 0.f, c2 = 0.f;
    for (int c = 0; c < CH; ++c) {
        const float av = __fdiv_rn(X4[(int64_t)c * E], n4), cv = __fdiv_rn(X6[(int64_t)c * E], n6);
        a2 = fmaf(av, av, a2);
        c2 = fmaf(cv, cv, c2);
    }
    float* o = nrm + obj * 4 * (int64_t)E;
    o[e] = n4; o[E + e] = n6; o[2 * (int64_t)E + e] = a2; o[3 * (int64_t)E + e] = c2;
}

// K tile on the CUDA cores (any E; the tensor-core kernel below needs E % 4 == 0): 64 x 64 outputs, 128-deep dot products of
// the normalised features, 4 x 4 outputs per thread
__global__ void __launch_bounds__(256) transport_k_kernel(const float* __restrict__ feat4, const float* __restrict__ feat6,
                                                          const float* __restrict__ nrm, int E, float lambda, float max_distance,
                                                          float* __restrict__ Kmat) {
    extern __shared__ float sm[];                           // A[128][64], B[128][64]
    float* As = sm;
    float* Bs = sm + CH * 64;
    const int64_t obj = blockIdx.z;
    const int i0 = blockIdx.y * 64, j0 = blockIdx.x * 64;
    const float* nr = nrm + obj * 4 * (int64_t)E;
    const int tid = threadIdx.x;
    for (int idx = tid; idx < CH * 64; idx += 256) {
        const int c = idx >> 6, t = idx & 63;
        const int i = i0 + t, j = j0 + t;
        As[idx] = i < E ? __fdiv_rn(feat4[(obj * CH + c) * (int64_t)E + i], nr[i]) : 0.f;
        Bs[idx] = j < E ? __fdiv_rn(feat6[(obj * CH + c) * (int64_t)E + j], nr[E + j]) : 0.f;
    }
    __syncthreads();
    const int ti = (tid >> 4) * 4, tj = (tid & 15) * 4;
    float acc[4][4] = {};
#pragma unroll 4
    for (int c = 0; c < CH; ++c) {
        const float4 a = *reinterpret_cast<const float4*>(As + c * 64 + ti);
        const float4 b = *reinterpret_cast<const float4*>(Bs + c * 64 + tj);
        const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int p = 0; p < 4; ++p)
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[p][q] = fmaf(av[p], bv[q], acc[p][q]);
    }
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        const int i = i0 + ti + p;
        if (i >= E) continue;
        const float a2 = nr[2 * (int64_t)E + i];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int j = j0 + tj + q;
            if (j >= E) continue;
            const float c2 = nr[3 * (int64_t)E + j];
            const float m = sqrtf(fmaxf(__fadd_rn(__fadd_rn(c2, -2.f * acc[p][q]), a2), 1e-30f));
            Kmat[(obj * E + i) * (int64_t)E + j] = expf(-lambda * fminf(m, max_distance));
        }
    }
}

// The same K tile on the tensor cores (tcgen05 + TMEM), 128 x 128 outputs per step: the 2628 x 2628 x 128 contraction of an
// object (1.77 GFLOP) is the second dense contraction of GMW.  A CTA owns a 128-row block of net-4 edges: their L2-normalised
// features are written once as FP16 hi/lo images in the MN-major 128B-swizzled UMMA layout (the layout of the MLP kernels'
// activation operand: 8 consecutive edges of one channel are one 16-byte chunk, which is how the features lie in memory,
// [128 channels][E]); it then walks the 128-column blocks of net-6 edges, building that operand the
// same way, issuing D[i][j] = sum_c A[i][c] B[c][j] as 3 x 8 MMAs (FP16x3 split, both operands MN-major from shared memory,
// FP32 accumulators in tensor memory) and turning the accumulators into K = exp(-lambda min(sqrt((c2 - 2 a.c) + a2), 5)) in
// the epilogue (thread = row, all 8 warps).  Features are scaled by 2^8 before the split so that the low parts stay normal
// FP16 numbers; the product carries 2^16, removed exactly.  Used when E is a multiple of 4 (16-byte row alignment).
constexpr int KT = 128;                                 // tile edge
constexpr size_t kKtcSmem = 4 * B_PART_BYTES + 2 * KT * sizeof(float) * 2 + 64;      // A hi/lo, B hi/lo, (a2, 1/n) x 2, barrier
constexpr float kKtcScale = 256.f, kKtcUnscale = 1.f / 65536.f;
constexpr uint32_t kIdescMnMn = kIdesc | (1u << 15);    // A MN-major as well (bit 15), B MN-major (bit 16), M = N = 128, F16 -> F32

// one 128-edge block of one net -> FP16 hi/lo operand image; also the block's per-edge 1/norm and |normalised|^2
__device__ __forceinline__ void ktc_build_operand(const float* __restrict__ feat, const float* __restrict__ nrm_n, const float* __restrict__ nrm_2,
                                                  int E, int e0, unsigned char* hi, unsigned char* lo, float* sq_s, int tid) {
    // 128 channels x 16 chunks of 8 edges = 2048 chunks, 256 threads: 8 chunks per thread; lanes run along the edge chunks
#pragma unroll 2
    for (int it = 0; it < 8; ++it) {
        const int id = it * 256 + tid;
        const int c = id >> 4, eblk = id & 15;
        const int e = e0 + eblk * 8;
        float v[8];
        const float* src = feat + (int64_t)c * E + e;
        if (e + 8 <= E) {
            const float4 x0 = *reinterpret_cast<const float4*>(src), x1 = *reinterpret_cast<const float4*>(src + 4);
            const float4 n0 = *reinterpret_cast<const float4*>(nrm_n + e), n1 = *reinterpret_cast<const float4*>(nrm_n + e + 4);
            v[0] = __fdiv_rn(x0.x, n0.x); v[1] = __fdiv_rn(x0.y, n0.y); v[2] = __fdiv_rn(x0.z, n0.z); v[3] = __fdiv_rn(x0.w, n0.w);
            v[4] = __fdiv_rn(x1.x, n1.x); v[5] = __fdiv_rn(x1.y, n1.y); v[6] = __fdiv_rn(x1.z, n1.z); v[7] = __fdiv_rn(x1.w, n1.w);
        } else {
#pragma unroll
            for (int q = 0; q < 8; ++q) v[q] = (e + q < E) ? __fdiv_rn(src[q], nrm_n[e + q]) : 0.f;
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) v[q] *= kKtcScale;
        store_b8(hi, lo, c, eblk, v);
    }
    if (tid < KT) sq_s[tid] = (e0 + tid < E) ? nrm_2[e0 + tid] : 0.f;
}

__global__ void __launch_bounds__(256, 1) transport_k_tc_kernel(const float* __restrict__ feat4, const float* __restrict__ feat6,
                                                                const float* __restrict__ nrm, int E, float lambda, float max_distance,
                                                                float* __restrict__ Kmat) {
    extern __shared__ __align__(1024) unsigned char ksm[];
    unsigned char* A_hi = ksm;
    unsigned char* A_lo = A_hi + B_PART_BYTES;
    unsigned char* B_hi = A_lo + B_PART_BYTES;
    unsigned char* B_lo = B_hi + B_PART_BYTES;
    float* a2_s = reinterpret_cast<float*>(B_lo + B_PART_BYTES);       // [128] |a_i|^2 of the row block
    float* c2_s = a2_s + KT;                                            // [128] |c_j|^2 of the current column block
    uint64_t* bar = reinterpret_cast<uint64_t*>(ksm + 4 * B_PART_BYTES + 2 * KT * sizeof(float) * 2);
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bar + 2);
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int64_t obj = blockIdx.y;
    const int i0 = blockIdx.x * KT;
    const float* nr = nrm + obj * 4 * (int64_t)E;           // [4][E]: |f4|, |f6|, |a|^2, |c|^2 (transport_norm_kernel)
    const float* f4 = feat4 + obj * (int64_t)CH * E;
    const float* f6 = feat6 + obj * (int64_t)CH * E;
    float* Kobj = Kmat + obj * (int64_t)E * E;
    if (tid == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) tmem_alloc(tmem_ptr, 128);
    ktc_build_operand(f4, nr, nr + 2 * (int64_t)E, E, i0, A_hi, A_lo, a2_s, tid);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = __shfl_sync(0xffffffffu, *tmem_ptr, 0);
    const int quarter = warp & 3, half = warp >> 2;          // TMEM lane quarter (rows), column half
    const int row = 32 * quarter + lane;                     // this thread's row of the tile
    const int i = i0 + row;
    const float a2 = a2_s[row];
    uint32_t phase = 0;
    for (int j0 = 0; j0 < E; j0 += KT) {
        ktc_build_operand(f6, nr + (int64_t)E, nr + 3 * (int64_t)E, E, j0, B_hi, B_lo, c2_s, tid);
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (warp == 0 && elect_one()) {
            tc_fence_after();
            uint32_t acc = 0;
#pragma unroll
            for (int term = 0; term < 3; ++term) {          // Ah.Bl + Al.Bh + Ah.Bh
                const uint32_t pa = smem_u32(term == 1 ? A_lo : A_hi);
                const uint32_t pb = smem_u32(term == 0 ? B_lo : B_hi);
#pragma unroll
                for (int ks = 0; ks < CH / 16; ++ks) {
                    umma_f16_ss(tmem_d, smem_desc(pa + ks * B_KSTEP, B_LBO, B_SBO), smem_desc(pb + ks * B_KSTEP, B_LBO, B_SBO), kIdescMnMn, acc);
                    acc = 1;
                }
            }
            umma_commit(bar);
        }
        mbar_wait(bar, phase);
        phase ^= 1;
        tc_fence_after();
        // epilogue: thread = row i, 64 columns of this warp's half
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
            float v[32];
            const int col0 = half * 64 + cc * 32;
            tmem_ld32(tmem_d + ((uint32_t)(32 * quarter) << 16) + (uint32_t)col0, v);
            if (i < E) {
                float* dst = Kobj + (int64_t)i * E + j0 + col0;
#pragma unroll
                for (int q = 0; q < 32; q += 4) {
                    float o[4];
#pragma unroll
                    for (int t = 0; t < 4; ++t) {
                        const float dot = v[q + t] * kKtcUnscale;
                        const float m = sqrtf(fmaxf(__fadd_rn(__fadd_rn(c2_s[col0 + q + t], -2.f * dot), a2), 1e-30f));
                        o[t] = expf(-lambda * fminf(m, max_distance));
                    }
                    const int j = j0 + col0 + q;
                    if (j + 4 <= E) *reinterpret_cast<float4*>(dst + q) = make_float4(o[0], o[1], o[2], o[3]);
                    else
#pragma unroll
                        for (int t = 0; t < 4; ++t)
                            if (j + t < E) dst[q + t] = o[t];
                }
            }
        }
        tc_fence_before();
        __syncthreads();                                     // accumulators read, B operand and c2_s free for the next block
        tc_fence_after();
    }
    if (warp == 0) tmem_dealloc(tmem_d, 128);
}

// column pass: partial[obj][chunk][j] = sum over the chunk's rows i of K[i][j] * u[i]
__global__ void __launch_bounds__(256) transport_col_kernel(const float* __restrict__ Kmat, const float* __restrict__ u, int E,
                                                            const int* __restrict__ stop, float* __restrict__ partial) {
    if (stop != nullptr && *stop) return;
    const int64_t obj = blockIdx.z;
    const int j = blockIdx.x * 256 + threadIdx.x;
    const int rows = (E + TP_CHUNKS - 1) / TP_CHUNKS;
    const int ib = blockIdx.y * rows, ie = min(E, ib + rows);
    if (j >= E) return;
    const float* Kp = Kmat + obj * (int64_t)E * E + j;
    const float* up = u + obj * (int64_t)E;
    float acc = 0.f;
#pragma unroll 4
    for (int i = ib; i < ie; ++i) acc = fmaf(Kp[(int64_t)i * E], up[i], acc);
    partial[(obj * TP_CHUNKS + blockIdx.y) * (int64_t)E + j] = acc;
}

// w[j] = c / (K^T u)[j]   (partials summed in chunk order)
__global__ void __launch_bounds__(256) transport_w_kernel(const float* __restrict__ partial, int E, float cval, const int* __restrict__ stop,
                                                          float* __restrict__ w) {
    if (stop != nullptr && *stop) return;
    const int64_t obj = blockIdx.y;
    const int j = blockIdx.x * 256 + threadIdx.x;
    if (j >= E) return;
    float t = 0.f;
    for (int k = 0; k < TP_CHUNKS; ++k) t += partial[(obj * TP_CHUNKS + k) * (int64_t)E + j];
    w[obj * (int64_t)E + j] = __fdiv_rn(cval, t);
}

// row pass (a warp per row): u[i] = r / (K w)[i]; raises *changed when |u - u_old| > tol anywhere
__global__ void __launch_bounds__(256) transport_row_kernel(const float* __restrict__ Kmat, const float* __restrict__ w, int E, float rval,
                                                            float tol, const int* __restrict__ stop, float* __restrict__ u,
                                                            int* __restrict__ changed) {
    if (stop != nullptr && *stop) return;
    const int64_t obj = blockIdx.y;
    const int i = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= E) return;
    const float* Kp = Kmat + (obj * E + i) * (int64_t)E;
    const float* wp = w + obj * (int64_t)E;
    // rows are 16-byte aligned when E % 4 == 0 (E = 2628): 512 bytes per warp and load, four loads in flight
    float acc = 0.f;
    if ((E & 3) == 0) {
        const float4* K4 = reinterpret_cast<const float4*>(Kp);
        const float4* w4 = reinterpret_cast<const float4*>(wp);
        const int E4 = E >> 2;
        float a4[4] = {0.f, 0.f, 0.f, 0.f};
        int j = lane;
        for (; j + 96 < E4; j += 128) {
            float4 k[4], x[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) { k[q] = __ldcs(K4 + j + 32 * q); x[q] = w4[j + 32 * q]; }
#pragma unroll
            for (int q = 0; q < 4; ++q)
                a4[q] = fmaf(k[q].w, x[q].w, fmaf(k[q].z, x[q].z, fmaf(k[q].y, x[q].y, fmaf(k[q].x, x[q].x, a4[q]))));
        }
        for (; j < E4; j += 32) {
            const float4 k = __ldcs(K4 + j), x = w4[j];
            a4[0] = fmaf(k.w, x.w, fmaf(k.z, x.z, fmaf(k.y, x.y, fmaf(k.x, x.x, a4[0]))));
        }
        acc = (a4[0] + a4[1]) + (a4[2] + a4[3]);
    } else {
        for (int j = lane; j < E; j += 32) acc = fmaf(Kp[j], wp[j], acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) {
        const float un = __fdiv_rn(rval, acc);
        const float uo = u[obj * (int64_t)E + i];
        u[obj * (int64_t)E + i] = un;
        if (!(fabsf(un - uo) <= tol)) atomicOr(changed, 1);
    }
}

// stop[k] = !changed[k]: the iteration after a converged one (and all later ones) does nothing.  Also seeds u = r.
__global__ void transport_flag_kernel(int* __restrict__ flags, int it) {
    // flags[0] = stop, flags[1] = changed of the iteration that just ran
    if (it > 0 && flags[1] == 0) flags[0] = 1;
    flags[1] = 0;
}
__global__ void __launch_bounds__(256) transport_fill_kernel(float* __restrict__ p, int64_t n, float v) {
    const int64_t t = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (t < n) p[t] = v;
}

// P = (u * K) * v^T (optional), sums[obj] = (sum P, trace P)   — a warp per row, per-row partials reduced by a second kernel
__global__ void __launch_bounds__(256) transport_p_kernel(const float* __restrict__ Kmat, const float* __restrict__ u,
                                                          const float* __restrict__ v, int E, float* __restrict__ P,
                                                          float* __restrict__ rowsum /* [N][2][E] */) {
    const int64_t obj = blockIdx.y;
    const int i = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= E) return;
    const float* Kp = Kmat + (obj * E + i) * (int64_t)E;
    const float* vp = v + obj * (int64_t)E;
    const float ui = u[obj * (int64_t)E + i];
    float acc = 0.f, diag = 0.f;
    for (int j = lane; j < E; j += 32) {
        const float p = __fmul_rn(__fmul_rn(ui, Kp[j]), vp[j]);
        if (P != nullptr) P[(obj * E + i) * (int64_t)E + j] = p;
        acc += p;
        if (j == i) diag = p;
    }
    acc = warp_sum(acc);
    diag = warp_sum(diag);
    if (lane == 0) {
        rowsum[(obj * 2) * (int64_t)E + i] = acc;
        rowsum[(obj * 2 + 1) * (int64_t)E + i] = diag;
    }
}
__global__ void __launch_bounds__(256) transport_sum_kernel(const float* __restrict__ rowsum, int E, float* __restrict__ sums) {
    __shared__ float red[2][8];
    const int64_t obj = blockIdx.x;
    float a = 0.f, d = 0.f;
    for (int i = threadIdx.x; i < E; i += 256) {
        a += rowsum[(obj * 2) * (int64_t)E + i];
        d += rowsum[(obj * 2 + 1) * (int64_t)E + i];
    }
    a = warp_sum(a);
    d = warp_sum(d);
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = a; red[1][threadIdx.x >> 5] = d; }
    __syncthreads();
    if (threadIdx.x == 0) {
        a = 0.f; d = 0.f;
        for (int k = 0; k < 8; ++k) { a += red[0][k]; d += red[1][k]; }
        sums[obj * 2] = a;
        sums[obj * 2 + 1] = d;
    }
}

inline size_t al(size_t x) { return (x + 255) / 256 * 256; }

}  // namespace

// workspace: K [N][E][E] | norms [N][4][E] | u, w (v) [N][E] each | partial [N][16][E] | row sums [N][2][E] | flags
size_t gmw_transport_workspace_bytes(int64_t N, int E) {
    const size_t e = (size_t)E;
    return al((size_t)N * e * e * 4) + al((size_t)N * 4 * e * 4) + 2 * al((size_t)N * e * 4) + al((size_t)N * TP_CHUNKS * e * 4) +
           al((size_t)N * 2 * e * 4) + 256;
}

// K inside a workspace filled by launch_gmw_transport_fwd (its first block, [N][E][E]): the plan source of the terms backward
const float* gmw_transport_workspace_k(const void* workspace) { return reinterpret_cast<const float*>(workspace); }

int launch_gmw_transport_fwd(const float* feat4, const float* feat6, int64_t N, int E, float lambda, float tol, int max_iter,
                             float* P, float* u_out, float* v_out, float* sums, void* workspace, cudaStream_t st) {
    const size_t e = (size_t)E;
    unsigned char* p = reinterpret_cast<unsigned char*>(workspace);
    float* Kmat = reinterpret_cast<float*>(p); p += al((size_t)N * e * e * 4);
    float* nrm = reinterpret_cast<float*>(p); p += al((size_t)N * 4 * e * 4);
    float* u = reinterpret_cast<float*>(p); p += al((size_t)N * e * 4);
    float* w = reinterpret_cast<float*>(p); p += al((size_t)N * e * 4);
    float* partial = reinterpret_cast<float*>(p); p += al((size_t)N * TP_CHUNKS * e * 4);
    float* rowsum = reinterpret_cast<float*>(p); p += al((size_t)N * 2 * e * 4);
    int* flags = reinterpret_cast<int*>(p);
    const unsigned eb = (unsigned)((E + 255) / 256), rb = (unsigned)((E + 7) / 8), tb = (unsigned)((E + 63) / 64);
    const float rc = 1.0f / (float)E;                        // r = c = 1 / E (model.py:186-190)
    cudaMemsetAsync(flags, 0, 2 * sizeof(int), st);
    transport_norm_kernel<<<dim3(eb, (unsigned)N), 256, 0, st>>>(feat4, feat6, N, E, nrm);
    const char* ktc_env = getenv("DCD_B200_KTC");          // DCD_B200_KTC=0: the FP32 CUDA-core tiles (A/B measurements, cross-checks)
    if ((E & 3) == 0 && !(ktc_env != nullptr && ktc_env[0] == '0')) {
        // tensor-core tiles (rows of K 16-byte aligned): cls forward at 8 objects 4.44 -> 4.04 ms, same loss to 6 digits
        cudaFuncSetAttribute(transport_k_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kKtcSmem);
        transport_k_tc_kernel<<<dim3((unsigned)((E + KT - 1) / KT), (unsigned)N), 256, kKtcSmem, st>>>(feat4, feat6, nrm, E, lambda, 5.0f, Kmat);
    } else {
        constexpr int kSmem = 2 * CH * 64 * sizeof(float);
        cudaFuncSetAttribute(transport_k_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
        transport_k_kernel<<<dim3(tb, tb, (unsigned)N), 256, kSmem, st>>>(feat4, feat6, nrm, E, lambda, 5.0f, Kmat);
    }
    transport_fill_kernel<<<(unsigned)((N * e + 255) / 256), 256, 0, st>>>(u, (int64_t)(N * e), rc);
    DCD_CHECK_LAUNCH();
    // optimal_transport.py:63-69: the test at the top of iteration 0 compares u = r with u_prev = 1 (never close), so
    // iteration 0 always runs; iteration k > 0 runs iff iteration k-1 changed u by more than tol somewhere in the batch
    for (int it = 0; it < max_iter; ++it) {
        transport_flag_kernel<<<1, 1, 0, st>>>(flags, it);
        transport_col_kernel<<<dim3(eb, TP_CHUNKS, (unsigned)N), 256, 0, st>>>(Kmat, u, E, flags, partial);
        transport_w_kernel<<<dim3(eb, (unsigned)N), 256, 0, st>>>(partial, E, rc, flags, w);
        transport_row_kernel<<<dim3(rb, (unsigned)N), 256, 0, st>>>(Kmat, w, E, rc, tol, flags, u, flags + 1);
    }
    DCD_CHECK_LAUNCH();
    // v = c / (K^T u), P = (u * K) * v^T
    transport_col_kernel<<<dim3(eb, TP_CHUNKS, (unsigned)N), 256, 0, st>>>(Kmat, u, E, nullptr, partial);
    transport_w_kernel<<<dim3(eb, (unsigned)N), 256, 0, st>>>(partial, E, rc, nullptr, w);
    transport_p_kernel<<<dim3(rb, (unsigned)N), 256, 0, st>>>(Kmat, u, w, E, P, rowsum);
    if (sums != nullptr) transport_sum_kernel<<<(unsigned)N, 256, 0, st>>>(rowsum, E, sums);
    if (u_out != nullptr) cudaMemcpyAsync(u_out, u, (size_t)N * e * 4, cudaMemcpyDeviceToDevice, st);
    if (v_out != nullptr) cudaMemcpyAsync(v_out, w, (size_t)N * e * 4, cudaMemcpyDeviceToDevice, st);
    DCD_CHECK_LAUNCH();
    return DCD_OK;
}

}  // namespace dcd
