// GMW edge-feature MLP, backward w.r.t. the parameters on the tensor cores (tcgen05 + TMEM), sm_100a.
//
// Autograd of GMW/main.py:465 restricted to the regression path, over the activations saved by the forward
// (block input x, preconv output P, pre-norm outputs Y1, Y2 + context-norm statistics).  Per residual block,
// last to first, two launches of ONE templated kernel (plus the small sums kernel of the second norm):
//     R2 :  dy2 = CN'(G * relu')          dW2 += dy2 . yhat1^T     d yhat1 = W2^T dy2   (+ sums for CN1')
//     R3F:  dy1 = CN'(d yhat1)            dWf += dy1 . x^T         G       = Wf^T dy1 + G   (folded preconv.conv1, residual path)
// followed by the chain rule through the fold (fold_wgrad_kernel: dWp, dW1 from dWf).  What the block loop leaves in G,
// dL/d(conv_in output), also gives the keypoint gradient (dcd_gmw_kpts_bwd: kpts_feat_bwd_kernel, kpts_gather_bwd_kernel).
// Every launch is the same dataflow on a 128-edge tile:
//   * the gradient operand A1 (128 channels x 128 edges) and the activation operand A2 are written ONCE into
//     shared memory as FP16 hi/lo images in the 128B-swizzled layout of the forward; the same A1 image is the
//     MN-major B operand of the data-gradient GEMM (A = W^T resident in tensor memory) and the K-major A operand
//     of the weight-gradient GEMM (B = A2 image, K = edges) — only the descriptors differ;
//   * FP32 fidelity: FP16x3 split (3 MMAs per product) as in the forward; the gradient image is scaled by a
//     power of two derived from the running maximum of the object's upstream gradient (tracked per object with one
//     atomicMax per warp in the producing epilogue), so hi/lo stay inside FP16's normal range whatever the other
//     objects' gradients are (a batch-wide maximum left an object 2^-12 below it with a subnormal lo part);
//   * the 128x128 weight gradient ACCUMULATES IN TENSOR MEMORY across the tiles of one object within the CTA; at each
//     object change and at the end it is unscaled into the CTA's partial (written by the first object, added to by the
//     next), reduced over the CTAs in a fixed order afterwards (deterministic, no float atomics);
//   * block conv biases receive exact zeros: they are cancelled by the mean subtraction that follows each of
//     them (SURVEY 7-H5; the reference's own values there are rounding noise around 1e-8).
#include "gmw_tc_common.cuh"

namespace dcd {

struct BwdTcArgs {
    const float* kpts2d;
    const float* kpts3d;
    const float* params[2];
    float* ws;              // forward workspace (save = 1)
    WsLayout L;
    const float2* scales;   // per-matrix (scale, 1/scale) written by the forward
    const float* fold;      // folded layers Wf^T, bf per (net, block) written by the forward (FOLD_STRIDE floats each)
    float* dwf;             // [2][128*128] gradient of the folded layer, blob layout [in][out]
    float* G;               // [2][N][128][EP] gradient w.r.t. the current block output
    float* D1;              // [2][N][128][EP] gradient w.r.t. yhat1
    float2* bstat;          // [2][2][N][T][128] partial sums of the context-norm backward
    float* wpart;           // [3][2 * ctas][128*128] per-CTA partial weight gradients
    float* inpart;          // [2*N*T][128][8] partial conv_in gradients
    float* gmax;            // [2][N][3*depth + 1] running |gradient| maxima per object (float bits, >= 0)
};

size_t tc_fold_offset_bytes(int depth);

namespace {

// R2: dy2, dW2, dyhat1.  R3F: dy1 (context-norm backward), dWf, dx + residual for the folded preconv.conv1 layer.
enum { MODE_R2 = 0, MODE_R3F = 3 };
constexpr int BT_THREADS = 512;
constexpr uint32_t TMB_W_HI = 0, TMB_W_LO = 64, TMB_DW = 128, TMB_D = 256;
constexpr size_t SMB_A1 = 0;                                       // gradient image  {hi, lo} 64 KB (also the output staging)
constexpr size_t SMB_A2 = SMB_A1 + 2 * B_PART_BYTES;               // activation image {hi, lo} 64 KB
constexpr size_t SMB_ST1 = SMB_A2 + 2 * B_PART_BYTES;              // [128] (mean1, inv1)
constexpr size_t SMB_ST2 = SMB_ST1 + CH * sizeof(float2);          // [128] (mean2, inv2)
constexpr size_t SMB_SB = SMB_ST2 + CH * sizeof(float2);           // [128] (S1/E, S2/(E-1)) of the norm being inverted
constexpr size_t SMB_RED = SMB_SB + CH * sizeof(float2);           // [4][128] float2 partial sums of the epilogue
constexpr size_t SMB_BAR = SMB_RED + 4 * CH * sizeof(float2);
constexpr size_t kBwdTcSmem = SMB_BAR + 64;

__device__ __forceinline__ int64_t gmax_slot(const WsLayout& L, int net, int64_t obj, int blk, int stage) {
    return ((int64_t)net * L.N + obj) * (3 * L.depth + 1) + blk * 3 + stage;
}

__device__ __forceinline__ void atomic_max_abs(float* slot, float v) {
    v = warp_max(v);
    if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int*>(slot), __float_as_int(v));
}
// power-of-two scale that maps `m` to about 2^target
__device__ __forceinline__ float pow2_scale(float m, int target) {
    if (!(m > 0.f)) return 1.f;
    int e;
    frexpf(m, &e);
    return ldexpf(1.f, target - e);
}
// reconstruct the 8 FP32 values of one operand chunk from its FP16 hi/lo parts
__device__ __forceinline__ void load_chunk(const unsigned char* hi, const unsigned char* lo, int ch, int eblk, float (&v)[8]) {
    const uint32_t krow = (uint32_t)ch & 7u;
    const uint32_t off = (uint32_t)(ch >> 3) * B_SBO + (uint32_t)(eblk >> 3) * B_LBO + krow * 128u + ((((uint32_t)eblk & 7u) ^ krow) << 4);
    const uint4 h = *reinterpret_cast<const uint4*>(hi + off), l = *reinterpret_cast<const uint4*>(lo + off);
    const __half2* hh = reinterpret_cast<const __half2*>(&h);
    const __half2* ll = reinterpret_cast<const __half2*>(&l);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float2 a = __half22float2(hh[q]), b = __half22float2(ll[q]);
        v[2 * q] = a.x + b.x;
        v[2 * q + 1] = a.y + b.y;
    }
}

__global__ void bwd_tc_init_kernel(float* gmax, int64_t n) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) gmax[i] = 0.f;
}

// BW0: d reg_weights (+ optionally the gradient w.r.t. the NORMALISED features coming from the correspondence branch,
// gn4 / gn6 [N][128][E]) -> d final features (mirrors gmw_edge_weight_kernel) + running max of |G|
__global__ void __launch_bounds__(256) edge_weight_bwd_tc_kernel(BwdTcArgs a, const float* __restrict__ grad_w,
                                                                 const float* __restrict__ gn4, const float* __restrict__ gn6) {
    const WsLayout& L = a.L;
    const int E = L.E, EP = L.EP, last = L.depth - 1;
    const int nb = (E + 255) / 256;
    const int64_t obj = blockIdx.x / nb;
    const int e = (blockIdx.x % nb) * 256 + threadIdx.x;
    __shared__ float2 stat_s[2][CH];
    {
        const int net = threadIdx.x >> 7, c = threadIdx.x & 127;
        stat_s[net][c] = merge_cn_stats(stat_ptr(a.ws, L, net, last, 1) + obj * (int64_t)L.T * CH, c, L.T, E);
    }
    __syncthreads();
    float m4 = 0.f, m6 = 0.f;
    if (e < E) {
        const int64_t off = obj * (int64_t)CH * EP + e;
        const float* Y4 = act_ptr(a.ws, L, 0, last, SLOT_Y2) + off;
        const float* X4 = act_ptr(a.ws, L, 0, last, SLOT_X) + off;
        const float* Y6 = act_ptr(a.ws, L, 1, last, SLOT_Y2) + off;
        const float* X6 = act_ptr(a.ws, L, 1, last, SLOT_X) + off;
        float n4 = 0.f, n6 = 0.f;
        for (int c = 0; c < CH; ++c) {
            const float2 s4 = stat_s[0][c], s6 = stat_s[1][c];
            const float x4 = fmaxf((Y4[(int64_t)c * EP] - s4.x) * s4.y, 0.f) + X4[(int64_t)c * EP];
            const float x6 = fmaxf((Y6[(int64_t)c * EP] - s6.x) * s6.y, 0.f) + X6[(int64_t)c * EP];
            n4 = fmaf(x4, x4, n4);
            n6 = fmaf(x6, x6, n6);
        }
        const float r4 = sqrtf(n4), r6 = sqrtf(n6);
        n4 = fmaxf(r4, 1e-12f);
        n6 = fmaxf(r6, 1e-12f);
        float a2 = 0.f, c2 = 0.f, ac = 0.f, ag = 0.f, cg = 0.f;
        const float* N4 = gn4 != nullptr ? gn4 + obj * (int64_t)CH * E + e : nullptr;
        const float* N6 = gn6 != nullptr ? gn6 + obj * (int64_t)CH * E + e : nullptr;
        for (int c = 0; c < CH; ++c) {
            const float2 s4 = stat_s[0][c], s6 = stat_s[1][c];
            const float x4 = fmaxf((Y4[(int64_t)c * EP] - s4.x) * s4.y, 0.f) + X4[(int64_t)c * EP];
            const float x6 = fmaxf((Y6[(int64_t)c * EP] - s6.x) * s6.y, 0.f) + X6[(int64_t)c * EP];
            const float av = __fdiv_rn(x4, n4), cv = __fdiv_rn(x6, n6);
            a2 = fmaf(av, av, a2);
            c2 = fmaf(cv, cv, c2);
            ac = fmaf(av, cv, ac);
            if (N4 != nullptr) ag = fmaf(av, N4[(int64_t)c * E], ag);
            if (N6 != nullptr) cg = fmaf(cv, N6[(int64_t)c * E], cg);
        }
        const float s = __fadd_rn(__fadd_rn(c2, -2.f * ac), a2);
        const float w = __fdiv_rn(1.f, sqrtf(fmaxf(s, 1e-30f)));
        const float gw = grad_w != nullptr ? __ldg(grad_w + obj * (int64_t)E + e) : 0.f;
        const float q = (s > 1e-30f) ? -0.5f * gw * w * w * w : 0.f;      // dL/ds, w = s^(-1/2)
        const float ada = q * (2.f * a2 - 2.f * ac) + ag, cdc = q * (2.f * c2 - 2.f * ac) + cg;
        float* G4 = a.G + (obj * (int64_t)CH) * EP + e;
        float* G6 = a.G + ((L.N + obj) * (int64_t)CH) * EP + e;
        const bool live4 = r4 > 1e-12f, live6 = r6 > 1e-12f;
        for (int c = 0; c < CH; ++c) {
            const float2 s4 = stat_s[0][c], s6 = stat_s[1][c];
            const float x4 = fmaxf((Y4[(int64_t)c * EP] - s4.x) * s4.y, 0.f) + X4[(int64_t)c * EP];
            const float x6 = fmaxf((Y6[(int64_t)c * EP] - s6.x) * s6.y, 0.f) + X6[(int64_t)c * EP];
            const float av = __fdiv_rn(x4, n4), cv = __fdiv_rn(x6, n6);
            const float da = q * (2.f * av - 2.f * cv) + (N4 != nullptr ? N4[(int64_t)c * E] : 0.f);
            const float dc = q * (2.f * cv - 2.f * av) + (N6 != nullptr ? N6[(int64_t)c * E] : 0.f);
            const float g4 = live4 ? (da - av * ada) / n4 : da / n4;
            const float g6 = live6 ? (dc - cv * cdc) / n6 : dc / n6;
            G4[(int64_t)c * EP] = g4;
            G6[(int64_t)c * EP] = g6;
            m4 = fmaxf(m4, fabsf(g4));
            m6 = fmaxf(m6, fabsf(g6));
        }
    }
    atomic_max_abs(a.gmax + gmax_slot(L, 0, obj, last, 0), m4);
    atomic_max_abs(a.gmax + gmax_slot(L, 1, obj, last, 0), m6);
}

// partial sums (sum dyh, sum dyh*yh) of the second context norm's backward, dyh = G * (yh > 0)
__global__ void __launch_bounds__(256) cn2_bwd_sums_tc_kernel(BwdTcArgs a, int blk) {
    const WsLayout& L = a.L;
    const int tile = blockIdx.x % L.T;
    const int64_t obj = blockIdx.x / L.T;
    const int net = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int E = L.E, EP = L.EP;
    __shared__ float2 stat_s[CH];
    if (threadIdx.x < CH)
        stat_s[threadIdx.x] = merge_cn_stats(stat_ptr(a.ws, L, net, blk, 1) + obj * (int64_t)L.T * CH, threadIdx.x, L.T, E);
    __syncthreads();
    const float* Y2 = act_ptr(a.ws, L, net, blk, SLOT_Y2) + obj * (int64_t)CH * EP;
    const float* G = a.G + ((int64_t)net * L.N + obj) * CH * EP;
    float2* out = a.bstat + (((int64_t)net * 2 + 0) * L.N + obj) * L.T * CH + (int64_t)tile * CH;
    const int e0 = tile * TE + lane * 4;
    for (int row = warp * 16; row < warp * 16 + 16; ++row) {
        const float2 st = stat_s[row];
        const float4 y = *reinterpret_cast<const float4*>(Y2 + (int64_t)row * EP + e0);
        const float4 g = *reinterpret_cast<const float4*>(G + (int64_t)row * EP + e0);
        const float yv[4] = {y.x, y.y, y.z, y.w}, gv[4] = {g.x, g.y, g.z, g.w};
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float yh = (yv[q] - st.x) * st.y;
            if (e0 + q < E && yh > 0.f) {
                s1 += gv[q];
                s2 = fmaf(gv[q], yh, s2);
            }
        }
        s1 = warp_sum(s1);
        s2 = warp_sum(s2);
        if (lane == 0) out[row] = make_float2(s1, s2);
    }
}

template <int MODE>
__global__ void __launch_bounds__(BT_THREADS, 1) mlp_bwd_tc_kernel(BwdTcArgs a, int blk) {
    const WsLayout& L = a.L;
    const int net = blockIdx.y;
    const int cin = net == 0 ? 4 : 6;
    const float* __restrict__ prm = a.params[net];
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform for the compiler (MMA issue on the uniform datapath)
    const int quarter = warp & 3, cq = warp >> 2;           // TMEM lane quarter / column quarter (32 edges) in epilogues
    const int E = L.E, EP = L.EP, T = L.T;

    extern __shared__ __align__(1024) unsigned char smem[];
    unsigned char* A1_hi = smem + SMB_A1;
    unsigned char* A1_lo = A1_hi + B_PART_BYTES;
    unsigned char* A2_hi = smem + SMB_A2;
    unsigned char* A2_lo = A2_hi + B_PART_BYTES;
    float2* st1_s = reinterpret_cast<float2*>(smem + SMB_ST1);
    float2* st2_s = reinterpret_cast<float2*>(smem + SMB_ST2);
    float2* sb_s = reinterpret_cast<float2*>(smem + SMB_SB);
    float2* red_s = reinterpret_cast<float2*>(smem + SMB_RED);
    uint64_t* bar_mma = reinterpret_cast<uint64_t*>(smem + SMB_BAR);
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + SMB_BAR + 16);

    // ---- setup: barrier, tensor memory, W^T resident as the A operand of the data-gradient GEMM
    const int which = (MODE == MODE_R2) ? 2 : 1;
    constexpr bool kResidual = MODE == MODE_R3F;      // output = dx of the block: add the skip gradient
    constexpr bool kCnBackward = MODE == MODE_R3F;    // gradient image = context-norm backward of y1
    const int mat = (net * L.depth + blk) * 3 + which;
    if (tid == 0) {
        mbar_init(bar_mma, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) tmem_alloc(tmem_ptr, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_ptr, 0);
    const int ch = 32 * quarter + lane;
    const uint32_t lane_off = (uint32_t)(32 * quarter) << 16;
    const float2 wsc = __ldg(a.scales + mat);
    if (warp < 8)
        load_weight_row_to_tmem_T(MODE == MODE_R3F ? a.fold + ((int64_t)net * L.depth + blk) * FOLD_STRIDE : prm + blob_w(cin, blk, which),
                                  wsc.x, ch, tmem_base + lane_off + TMB_W_HI, tmem_base + lane_off + TMB_W_LO, cq & 1);
    // the stage's slots of the per-object maxima: read (what feeds the gradient image) and written (this launch's output)
    const int in_blk = blk, in_stage = MODE == MODE_R3F ? 1 : MODE;
    const int out_blk = kResidual ? (blk > 0 ? blk - 1 : L.depth) : blk, out_stage = kResidual ? 0 : MODE + 1;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    const int64_t ntiles = L.N * (int64_t)T;
    const int64_t t_begin = ntiles * blockIdx.x / gridDim.x, t_end = ntiles * (blockIdx.x + 1) / gridDim.x;
    const int eblk = lane & 15;
    uint32_t mma_phase = 0;
    int64_t stat_obj = -1;
    float omax = 0.f;
    float gs = 1.f, un_d = 0.f;       // the current object's image scale and data-gradient unscale
    float* part = a.wpart + (((int64_t)which * 2 + net) * gridDim.x + blockIdx.x) * (CH * CH) + (int64_t)ch * CH + cq * 32;
    bool part_written = false;
    // the weight gradient accumulated in tensor memory for one object -> (unscaled) into this CTA's partial
    auto flush_wgrad = [&]() {
        float v[32];
        tmem_ld32(tmem_base + TMB_DW + lane_off + (uint32_t)(cq * 32), v);
        const float un_w = 1.f / gs;
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
            float4 w = make_float4(v[i] * un_w, v[i + 1] * un_w, v[i + 2] * un_w, v[i + 3] * un_w);
            if (part_written) {
                const float4 p = *reinterpret_cast<const float4*>(part + i);
                w.x += p.x; w.y += p.y; w.z += p.z; w.w += p.w;
            }
            *reinterpret_cast<float4*>(part + i) = w;
        }
        part_written = true;
    };

    for (int64_t t = t_begin; t < t_end; ++t) {
        const int64_t obj = t / T;
        const int tile = (int)(t - obj * T);
        const int64_t obj_off = obj * (int64_t)CH * EP;
        const int valid = min(TE, E - tile * TE);
        const int64_t gobj = ((int64_t)net * L.N + obj) * CH * EP;
        const bool new_obj = stat_obj != obj;          // CTA-uniform

        if (new_obj) {
            if (stat_obj >= 0) {                       // leave the previous object: its output maximum and weight gradient
                atomic_max_abs(a.gmax + gmax_slot(L, net, stat_obj, out_blk, out_stage), omax);
                omax = 0.f;
                flush_wgrad();
            }
            // scale of the gradient image from the running maximum of what feeds it, for this object
            gs = pow2_scale(a.gmax[gmax_slot(L, net, obj, in_blk, in_stage)], 4);   // |dy| <= ~1700 x the tracked maximum
            un_d = wsc.y / gs;                                                     // data-gradient accumulator -> FP32
            if (tid < CH) {
                st1_s[tid] = merge_cn_stats(stat_ptr(a.ws, L, net, blk, 0) + obj * (int64_t)T * CH, tid, T, E);
                if (MODE == MODE_R2)
                    st2_s[tid] = merge_cn_stats(stat_ptr(a.ws, L, net, blk, 1) + obj * (int64_t)T * CH, tid, T, E);
                const float2 sb = merge_sums(a.bstat + (((int64_t)net * 2 + (MODE == MODE_R2 ? 0 : 1)) * L.N + obj) * T * CH, tid, T);
                sb_s[tid] = make_float2(sb.x / (float)E, sb.y / (float)(E - 1));
            }
            __syncthreads();
            stat_obj = obj;
        }

        // ---- operand images: a warp owns 8 channels = 4 row pairs, lanes 0-15 / 16-31 take the two rows,
        //      each lane one 256-bit load per array and one 16-byte chunk per image part
        {
            const float* S1p;   // first array feeding A1
            const float* S2p;   // second array feeding A1 (R2: G, R3F: Y1)
            const float* S3p;   // array feeding A2
            if (MODE == MODE_R2) {
                S1p = act_ptr(a.ws, L, net, blk, SLOT_Y2) + obj_off;
                S2p = a.G + gobj;
                S3p = act_ptr(a.ws, L, net, blk, SLOT_Y1) + obj_off;
            } else {
                S1p = a.D1 + gobj;
                S2p = act_ptr(a.ws, L, net, blk, SLOT_Y1) + obj_off;
                S3p = act_ptr(a.ws, L, net, blk, SLOT_X) + obj_off;
            }
            const int64_t eoff = tile * TE + eblk * 8;
#pragma unroll 1
            for (int it0 = 0; it0 < 4; it0 += 2) {
                F8 b1[2], b2[2], b3[2];
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int c = warp * 8 + (it0 + u) * 2 + (lane >> 4);
                    b1[u] = ld256(S1p + (int64_t)c * EP + eoff);
                    b2[u] = ld256(S2p + (int64_t)c * EP + eoff);
                    b3[u] = ld256(S3p + (int64_t)c * EP + eoff);
                }
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int c = warp * 8 + (it0 + u) * 2 + (lane >> 4);
                    float g[8], h[8];
                    if (MODE == MODE_R2) {
                        const float2 s2 = st2_s[c], s1 = st1_s[c], sb = sb_s[c];
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const float yh = (b1[u].v[q] - s2.x) * s2.y;
                            const float dyh = yh > 0.f ? b2[u].v[q] : 0.f;
                            g[q] = s2.y * (dyh - sb.x - yh * sb.y);
                            h[q] = (b3[u].v[q] - s1.x) * s1.y;
                        }
                    } else {
                        const float2 s1 = st1_s[c], sb = sb_s[c];
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const float yh = (b2[u].v[q] - s1.x) * s1.y;
                            g[q] = s1.y * (b1[u].v[q] - sb.x - yh * sb.y);
                            h[q] = b3[u].v[q];
                        }
                    }
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const bool ok = eblk * 8 + q < valid;       // invalid edges must not reach the K = edges sum
                        g[q] = ok ? g[q] * gs : 0.f;
                        h[q] = ok ? h[q] : 0.f;
                    }
                    store_b8(A1_hi, A1_lo, c, eblk, g);
                    store_b8(A2_hi, A2_lo, c, eblk, h);
                }
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (warp == 0 && elect_one()) {
            tc_fence_after();
            // weight gradient: D_w[o][i] += sum_e A1[o][e] A2[i][e]   (both K-major views, accumulates over the object's tiles)
            uint32_t acc = new_obj ? 0u : 1u;
#pragma unroll
            for (int term = 0; term < 3; ++term) {
                const uint32_t pa = smem_u32(term == 1 ? A1_lo : A1_hi);
                const uint32_t pb = smem_u32(term == 0 ? A2_lo : A2_hi);
#pragma unroll
                for (int ks = 0; ks < TE / 16; ++ks) {
                    umma_f16_ss(tmem_base + TMB_DW, smem_desc(pa + kmajor_koff(ks), 16, B_SBO), smem_desc(pb + kmajor_koff(ks), 16, B_SBO),
                                kIdescKK, acc);
                    acc = 1u;
                }
            }
            // data gradient: D[i][e] = sum_o W[o][i] A1[o][e]
            issue_layer_gemm(tmem_base + TMB_D, tmem_base + TMB_W_HI, tmem_base + TMB_W_LO, smem_u32(A1_hi), smem_u32(A1_lo));
            umma_commit(bar_mma);
        }
        mbar_wait(bar_mma, mma_phase);
        mma_phase ^= 1;
        tc_fence_after();

        // ---- epilogue: thread = channel `ch`, 32 edges of column quarter `cq`
        {
            float v[32];
            tmem_ld32(tmem_base + TMB_D + lane_off + (uint32_t)(cq * 32), v);
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] *= un_d;
            if (MODE == MODE_R2) {
                float s1 = 0.f, s2 = 0.f;                    // sums for the first context norm's backward
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float yh[8];
                    load_chunk(A2_hi, A2_lo, ch, cq * 4 + j, yh);
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        s1 += v[j * 8 + q];
                        s2 = fmaf(v[j * 8 + q], yh[q], s2);
                    }
                }
                red_s[cq * CH + ch] = make_float2(s1, s2);
            }
            float4* stage = reinterpret_cast<float4*>(A1_hi);   // the gradient image is consumed: reuse it as staging
#pragma unroll
            for (int q = 0; q < 8; ++q)
                stage[ch * 32 + ((cq * 8 + q) ^ (ch & 31))] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
            tc_fence_before();
            __syncthreads();
            if (MODE == MODE_R2 && tid < CH) {
                const float2 p0 = red_s[tid], p1 = red_s[CH + tid], p2 = red_s[2 * CH + tid], p3 = red_s[3 * CH + tid];
                a.bstat[(((int64_t)net * 2 + 1) * L.N + obj) * T * CH + (int64_t)tile * CH + tid] =
                    make_float2((p0.x + p1.x) + (p2.x + p3.x), (p0.y + p1.y) + (p2.y + p3.y));
            }
            float* Out = (MODE == MODE_R2 ? a.D1 : a.G) + gobj + tile * TE;
#pragma unroll 4
            for (int i = 0; i < 8; ++i) {
                const int r = warp * 8 + i;
                float4 val = stage[r * 32 + (lane ^ (r & 31))];
                float* dst = Out + (int64_t)r * EP + lane * 4;
                if (kResidual) {                             // residual path: dx = W^T dy + G
                    const float4 g = *reinterpret_cast<const float4*>(dst);
                    val.x += g.x; val.y += g.y; val.z += g.z; val.w += g.w;
                }
                // padded columns (edge >= E) hold no data: keep them zero and out of the running maximum
                const int c0 = lane * 4;
                if (c0 + 0 >= valid) val.x = 0.f;
                if (c0 + 1 >= valid) val.y = 0.f;
                if (c0 + 2 >= valid) val.z = 0.f;
                if (c0 + 3 >= valid) val.w = 0.f;
                *reinterpret_cast<float4*>(dst) = val;
                omax = fmaxf(omax, fmaxf(fmaxf(fabsf(val.x), fabsf(val.y)), fmaxf(fabsf(val.z), fabsf(val.w))));
            }
            __syncthreads();                                 // images free for the next tile
        }
    }
    // ---- the last object of this CTA's tiles: output maximum, weight gradient -> the CTA's partial
    if (stat_obj >= 0) {
        atomic_max_abs(a.gmax + gmax_slot(L, net, stat_obj, out_blk, out_stage), omax);
        flush_wgrad();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 512);
}

// BW4: conv_in gradient partials.  Warp w owns channels 16w..16w+15, lanes own 4 edges of the tile each.
__global__ void __launch_bounds__(256) conv_in_bwd_tc_kernel(BwdTcArgs a) {
    const WsLayout& L = a.L;
    const int tile = blockIdx.x % L.T;
    const int64_t obj = blockIdx.x / L.T;
    const int net = blockIdx.y;
    const int cin = net == 0 ? 4 : 6;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int E = L.E, EP = L.EP;
    const int64_t cta = ((int64_t)net * L.N + obj) * L.T + tile;
    float f[4][6];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int e = tile * TE + lane * 4 + q;
        int i, j;
        decode_edge(e < E ? e : E - 1, L.n, i, j);
        if (net == 0) {
            const float* pi = a.kpts2d + (obj * L.n + i) * 2;
            const float* pj = a.kpts2d + (obj * L.n + j) * 2;
            f[q][0] = __ldg(pi); f[q][1] = __ldg(pi + 1); f[q][2] = __ldg(pj); f[q][3] = __ldg(pj + 1);
            f[q][4] = 0.f; f[q][5] = 0.f;
        } else {
            const float* pi = a.kpts3d + (obj * L.n + i) * 3;
            const float* pj = a.kpts3d + (obj * L.n + j) * 3;
            f[q][0] = __ldg(pi); f[q][1] = __ldg(pi + 1); f[q][2] = __ldg(pi + 2);
            f[q][3] = __ldg(pj); f[q][4] = __ldg(pj + 1); f[q][5] = __ldg(pj + 2);
        }
    }
    const float* G = a.G + ((int64_t)net * L.N + obj) * CH * EP;
    float* out = a.inpart + cta * (CH * 8);
    const int e0 = tile * TE + lane * 4;
    for (int c = warp * 16; c < warp * 16 + 16; ++c) {
        const float4 g4 = *reinterpret_cast<const float4*>(G + (int64_t)c * EP + e0);
        const float g[4] = {e0 + 0 < E ? g4.x : 0.f, e0 + 1 < E ? g4.y : 0.f, e0 + 2 < E ? g4.z : 0.f, e0 + 3 < E ? g4.w : 0.f};
        float s[7];
#pragma unroll
        for (int k = 0; k < 7; ++k) s[k] = 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
#pragma unroll
            for (int k = 0; k < 6; ++k) s[k] = fmaf(g[q], f[q][k], s[k]);
            s[6] += g[q];
        }
#pragma unroll
        for (int k = 0; k < 7; ++k) s[k] = warp_sum(s[k]);
        if (lane == 0) {
#pragma unroll
            for (int k = 0; k < 6; ++k) out[c * 8 + k] = (k < cin) ? s[k] : 0.f;
            out[c * 8 + 6] = s[6];
            out[c * 8 + 7] = 0.f;
        }
    }
}

// Sum the per-CTA partials of one (matrix, net) in CTA order into the gradient blob (transposed back to the
// blob's [in][out] layout); the block's conv biases get exact zeros.
// blockIdx.y = 0: conv2 (which = 2) into the blob; blockIdx.y = 1: the folded layer (partials of slot 1) into a.dwf.
__global__ void __launch_bounds__(256) reduce_wgrad_tc_kernel(BwdTcArgs a, int blk, int ctas, float* __restrict__ g4, float* __restrict__ g6) {
    const int which = blockIdx.y == 0 ? 2 : 1, net = blockIdx.z;
    const int t = blockIdx.x * 256 + threadIdx.x;          // t = o * 128 + i
    const int cin = net == 0 ? 4 : 6;
    float* g = net == 0 ? g4 : g6;
    if (t < CH) {                                           // the block's three conv biases: exact zeros
        if (which == 2) g[blob_b(cin, blk, 2) + t] = 0.f;
        else { g[blob_b(cin, blk, 0) + t] = 0.f; g[blob_b(cin, blk, 1) + t] = 0.f; }
    }
    if (t >= CH * CH) return;
    const float* p = a.wpart + (((int64_t)which * 2 + net) * ctas) * (CH * CH) + t;
    float s0 = 0.f, s1 = 0.f;
    int i = 0;
    for (; i + 2 <= ctas; i += 2) {
        s0 += p[(int64_t)i * CH * CH];
        s1 += p[(int64_t)(i + 1) * CH * CH];
    }
    if (i < ctas) s0 += p[(int64_t)i * CH * CH];
    const int o = t / CH, in = t % CH;
    if (which == 2) g[blob_w(cin, blk, 2) + (int64_t)in * CH + o] = s0 + s1;
    else a.dwf[(int64_t)net * CH * CH + (int64_t)in * CH + o] = s0 + s1;
}

// Chain rule through the fold Wf^T = Wp^T . W1^T (blob layouts [in][mid], [mid][out]):
//   dWp^T = dWf^T . W1^T^T,   dW1^T = Wp^T^T . dWf^T        blockIdx.y: 0 -> dWp, 1 -> dW1
// (the bias term of dW1, (sum_e dy1) bp^T, vanishes with the context norm that follows: sum_e dy1 = 0.)
__global__ void __launch_bounds__(256) fold_wgrad_kernel(BwdTcArgs a, int blk, float* __restrict__ g4, float* __restrict__ g6) {
    // 32 x 32 output tile per block, 32-deep chunks of the contraction staged in shared memory (both products read their
    // operands along the contiguous index; the A . B^T one is transposed on the way in)
    __shared__ float As[32][33], Bs[32][33];
    const int net = blockIdx.z, cin = net == 0 ? 4 : 6;
    const float* prm = a.params[net];
    const float* Wp = prm + blob_w(cin, blk, 0);            // [in][mid]
    const float* W1 = prm + blob_w(cin, blk, 1);            // [mid][out]
    const float* dWf = a.dwf + (int64_t)net * CH * CH;      // [in][out]
    float* g = net == 0 ? g4 : g6;
    const bool first = blockIdx.y == 0;                     // dWp^T[in r][mid c] = sum_o dWf^T[r][o] W1^T[c][o]
    const int r0 = (blockIdx.x >> 2) * 32, c0 = (blockIdx.x & 3) * 32;   // else dW1^T[mid r][out c] = sum_i Wp^T[i][r] dWf^T[i][c]
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5; // 8 rows of 32 threads
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int k0 = 0; k0 < CH; k0 += 32) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int y = ty + 8 * q;
            if (first) {
                As[y][tx] = dWf[(r0 + y) * CH + k0 + tx];    // As[r][k]
                Bs[y][tx] = W1[(c0 + y) * CH + k0 + tx];     // Bs[c][k]
            } else {
                As[y][tx] = Wp[(k0 + y) * CH + r0 + tx];     // As[k][r]
                Bs[y][tx] = dWf[(k0 + y) * CH + c0 + tx];    // Bs[k][c]
            }
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 32; ++k) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int y = ty + 8 * q;
                acc[q] = first ? fmaf(As[y][k], Bs[tx][k], acc[q]) : fmaf(As[k][y], Bs[k][tx], acc[q]);
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) g[blob_w(cin, blk, first ? 0 : 1) + (r0 + ty + 8 * q) * CH + c0 + tx] = acc[q];
}

__global__ void __launch_bounds__(128) reduce_conv_in_tc_kernel(BwdTcArgs a, float* __restrict__ g4, float* __restrict__ g6) {
    const WsLayout& L = a.L;
    const int net = blockIdx.y, k = blockIdx.x, c = threadIdx.x;     // k in 0..6
    const int cin = net == 0 ? 4 : 6;
    if (k < 6 && k >= cin) return;
    const int64_t per_net = L.N * L.T;
    const float* p = a.inpart + (int64_t)net * per_net * (CH * 8) + c * 8 + k;
    float s = 0.f;
    for (int64_t i = 0; i < per_net; ++i) s += p[i * (CH * 8)];
    float* g = net == 0 ? g4 : g6;
    if (k == 6) g[blob_in_b(cin) + c] = s;
    else g[blob_in_w() + (int64_t)k * CH + c] = s;
}

// ---- keypoint gradient (dcd_gmw_kpts_bwd), from G = dL/dx0 left by the block loop.  conv_in and edge_expand are linear:
//   KA: dF[e][k] = sum_c W_in^T[k][c] G[c][e]   one thread per (net, object, edge), channels in a fixed order
//   KB: d kpt[i]  = sum_{j>i} dF_(i,j)[0:h] + sum_{h'<i} dF_(h',i)[h:2h]   one warp per (net, object, keypoint), h = cin / 2
// dF [net][N][E][cin] lives in the D1 region of the scratch (dead after the block loop, >= 2 N E 128 floats).
template <int CIN>
__device__ __forceinline__ void kpts_feat_bwd_edge(const float* __restrict__ G, const float* __restrict__ w_s, int EP, int e,
                                                   float* __restrict__ out) {
    float acc[CIN];
#pragma unroll
    for (int k = 0; k < CIN; ++k) acc[k] = 0.f;
#pragma unroll 4
    for (int c = 0; c < CH; ++c) {
        const float g = G[(int64_t)c * EP + e];
#pragma unroll
        for (int k = 0; k < CIN; ++k) acc[k] = fmaf(w_s[k * CH + c], g, acc[k]);
    }
#pragma unroll
    for (int k = 0; k < CIN; ++k) out[k] = acc[k];
}

__global__ void __launch_bounds__(256) kpts_feat_bwd_kernel(const float* __restrict__ params4, const float* __restrict__ params6,
                                                            const float* __restrict__ Gs, float* __restrict__ dF, int64_t N,
                                                            int E, int EP, int net0) {
    const int net = net0 + blockIdx.y, cin = net == 0 ? 4 : 6;
    const int nb = (E + 255) / 256;
    const int64_t obj = blockIdx.x / nb;
    const int e = (blockIdx.x % nb) * 256 + threadIdx.x;
    __shared__ float w_s[6 * CH];
    const float* prm = (net == 0 ? params4 : params6) + blob_in_w();
    for (int t = threadIdx.x; t < cin * CH; t += 256) w_s[t] = __ldg(prm + t);
    __syncthreads();
    if (e >= E) return;                                   // padded columns e >= E contribute nothing
    const float* G = Gs + ((int64_t)net * N + obj) * CH * EP;
    float* out = dF + (net == 0 ? 0 : N * (int64_t)E * 4) + (obj * E + e) * cin;
    if (net == 0) kpts_feat_bwd_edge<4>(G, w_s, EP, e, out);
    else kpts_feat_bwd_edge<6>(G, w_s, EP, e, out);
}

__global__ void __launch_bounds__(256) kpts_gather_bwd_kernel(const float* __restrict__ dF, int64_t N, int n, int net0,
                                                              float* __restrict__ grad2, float* __restrict__ grad3) {
    const int net = net0 + blockIdx.y, cin = net == 0 ? 4 : 6, h = cin / 2;
    const int E = n * (n - 1) / 2;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nb = (n + 7) / 8;
    const int64_t obj = blockIdx.x / nb;
    const int kk = (blockIdx.x % nb) * 8 + warp;
    if (kk >= n) return;
    const float* F = dF + (net == 0 ? 0 : N * (int64_t)E * 4) + obj * E * (int64_t)cin;
    float s[3] = {0.f, 0.f, 0.f};
    for (int m = lane; m < n; m += 32) {                  // the n - 1 incident edges, lane-strided in partner order
        if (m == kk) continue;
        const int i = min(kk, m), j = max(kk, m);
        const float* f = F + (int64_t)(row_offset(i, n) + j - i - 1) * cin + (kk == i ? 0 : h);
#pragma unroll
        for (int q = 0; q < 3; ++q)
            if (q < h) s[q] += f[q];
    }
#pragma unroll
    for (int q = 0; q < 3; ++q) s[q] = warp_sum(s[q]);
    if (lane == 0) {
        float* o = (net == 0 ? grad2 : grad3) + (obj * n + kk) * h;
#pragma unroll
        for (int q = 0; q < 3; ++q)
            if (q < h) o[q] = s[q];
    }
}

struct BwdTcScratch {
    int64_t G, D1, bstat, wpart, inpart, gmax, dwf, total;   // float offsets
};

BwdTcScratch bwd_tc_layout(const WsLayout& L, int ctas) {
    BwdTcScratch s;
    int64_t o = 0;
    auto take = [&](int64_t n) { int64_t r = o; o += (n + 63) & ~(int64_t)63; return r; };
    s.G = take(2 * L.act);
    s.D1 = take(2 * L.act);
    s.bstat = take((int64_t)2 * 2 * L.stat * 2);
    s.wpart = take((int64_t)3 * 2 * ctas * CH * CH);
    s.inpart = take((int64_t)2 * L.N * L.T * CH * 8);
    s.gmax = take((int64_t)2 * L.N * (3 * L.depth + 1));
    s.dwf = take((int64_t)2 * CH * CH);
    s.total = o;
    return s;
}

int bwd_tc_ctas(const WsLayout& L) {
    const int64_t ntiles = L.N * (int64_t)L.T;
    const int per_net = max(1, device_sm_count() / 2);
    return (int)(ntiles < per_net ? ntiles : per_net);
}

}  // namespace

size_t gmw_bwd_scratch_floats(int64_t N, int n, int depth) {
    const WsLayout L = make_layout(N, n, depth, 1);
    // sized for the largest grid any device can ask for (independent of the current device)
    const int64_t ntiles = L.N * (int64_t)L.T;
    const int ctas = (int)(ntiles < 128 ? ntiles : 128);
    return (size_t)bwd_tc_layout(L, ctas).total;
}

int launch_gmw_weights_bwd(const float* kpts2d, const float* kpts3d, const float* params4, const float* params6,
                           int64_t N, int n, int depth, const float* grad_reg_w, const float* grad_nfeat4,
                           const float* grad_nfeat6, float* grad4, float* grad6,
                           float* ws, float* scratch, cudaStream_t st) {
    BwdTcArgs a;
    a.kpts2d = kpts2d; a.kpts3d = kpts3d;
    a.params[0] = params4; a.params[1] = params6;
    a.ws = ws;
    a.L = make_layout(N, n, depth, 1);
    if ((int64_t)a.L.T * N > 0x7fffffffLL) return DCD_E_UNSUPPORTED;
    int ctas = bwd_tc_ctas(a.L);
    if (ctas > 128) ctas = 128;
    const BwdTcScratch S = bwd_tc_layout(a.L, ctas);
    a.scales = reinterpret_cast<const float2*>(reinterpret_cast<unsigned char*>(ws) +
                                               (((size_t)a.L.total * sizeof(float) + 255) / 256) * 256);
    a.G = scratch + S.G;
    a.D1 = scratch + S.D1;
    a.bstat = reinterpret_cast<float2*>(scratch + S.bstat);
    a.wpart = scratch + S.wpart;
    a.inpart = scratch + S.inpart;
    a.gmax = scratch + S.gmax;
    a.dwf = scratch + S.dwf;
    a.fold = reinterpret_cast<const float*>(reinterpret_cast<const unsigned char*>(a.scales) + tc_fold_offset_bytes(depth));
    cudaFuncSetAttribute(mlp_bwd_tc_kernel<MODE_R2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBwdTcSmem);
    cudaFuncSetAttribute(mlp_bwd_tc_kernel<MODE_R3F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBwdTcSmem);

    const int64_t ng = 2 * N * (3 * depth + 1);
    bwd_tc_init_kernel<<<(unsigned)((ng + 127) / 128), 128, 0, st>>>(a.gmax, ng);
    const unsigned g0 = (unsigned)(((a.L.E + 255) / 256) * N);
    edge_weight_bwd_tc_kernel<<<g0, 256, 0, st>>>(a, grad_reg_w, grad_nfeat4, grad_nfeat6);
    const dim3 tgrid((unsigned)(a.L.T * N), 2);
    const dim3 grid((unsigned)ctas, 2);
    const dim3 rgrid((CH * CH + 255) / 256, 2, 2);
    for (int blk = depth - 1; blk >= 0; --blk) {
        cn2_bwd_sums_tc_kernel<<<tgrid, 256, 0, st>>>(a, blk);
        mlp_bwd_tc_kernel<MODE_R2><<<grid, BT_THREADS, kBwdTcSmem, st>>>(a, blk);
        mlp_bwd_tc_kernel<MODE_R3F><<<grid, BT_THREADS, kBwdTcSmem, st>>>(a, blk);
        reduce_wgrad_tc_kernel<<<rgrid, 256, 0, st>>>(a, blk, ctas, grad4, grad6);
        fold_wgrad_kernel<<<dim3(16, 2, 2), 256, 0, st>>>(a, blk, grad4, grad6);
    }
    conv_in_bwd_tc_kernel<<<tgrid, 256, 0, st>>>(a);
    reduce_conv_in_tc_kernel<<<dim3(7, 2), 128, 0, st>>>(a, grad4, grad6);
    DCD_CHECK_LAUNCH();
    return DCD_OK;
}

int launch_gmw_kpts_bwd(const float* params4, const float* params6, int64_t N, int n, int depth, float* scratch,
                        float* grad_kpts2d, float* grad_kpts3d, cudaStream_t st) {
    const WsLayout L = make_layout(N, n, depth, 1);
    if ((int64_t)L.T * N > 0x7fffffffLL) return DCD_E_UNSUPPORTED;
    const BwdTcScratch S = bwd_tc_layout(L, 1);          // the G and D1 offsets do not depend on the CTA count
    const int net0 = grad_kpts2d != nullptr ? 0 : 1;
    const unsigned nets = (grad_kpts2d != nullptr && grad_kpts3d != nullptr) ? 2 : 1;
    const int64_t ga = (int64_t)((L.E + 255) / 256) * N, gb = (int64_t)((n + 7) / 8) * N;
    if (ga > 0x7fffffffLL) return DCD_E_UNSUPPORTED;
    kpts_feat_bwd_kernel<<<dim3((unsigned)ga, nets), 256, 0, st>>>(params4, params6, scratch + S.G, scratch + S.D1, N, L.E,
                                                                    L.EP, net0);
    kpts_gather_bwd_kernel<<<dim3((unsigned)gb, nets), 256, 0, st>>>(scratch + S.D1, N, n, net0, grad_kpts2d, grad_kpts3d);
    DCD_CHECK_LAUNCH();
    return DCD_OK;
}

}  // namespace dcd
