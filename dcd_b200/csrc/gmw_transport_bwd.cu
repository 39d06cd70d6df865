// Correspondence branch of GMW, backward (SURVEY 8f row N1): gradient of a loss on the transport plan P w.r.t. the
// L2-normalised edge features of the two nets.
//
// Reference: RegularisedTransportFn.backward / gradientFn (GMW/lib/optimal_transport.py:75-128, 184-222), the
// implicit-function gradient of the Sinkhorn fixed point, followed by autograd through pairwiseL2Dist
// (GMW/model/model.py:17-36).  The reference forms S = diag(colsum B) - B'^T diag(1/rowsum B') B'  (B = lambda P, B' = B
// without its first row), factorises it (E x E Cholesky), inverts it and builds R, Q (three more E^3 products).  Every
// one of those matrices is only ever applied to ONE vector, so with  u1 = rowsum(V*B)[1:], u2 = colsum(V*B)  (V = dL/dP)
//     x   = S^-1 (u2 - B'^T (u1 / r1))            r1 = rowsum(B)[1:]
//     u3  = (u1 - B' x) / r1                      (0 for the removed first row)
//     dL/dM[i][j] = B[i][j] * (u3[i] + x[j] - V[i][j])
// is the same gradient (u4 = x, u3 as in the reference) with a single SPD solve.  S is (lambda/E)(I - Pn'^T Pn') for
// the nearly doubly-stochastic Pn = E P: one eigenvalue ~1/E (the constant vector), the rest clustered — conjugate
// gradients converge in 6-20 iterations (matrix-free: two passes over P per iteration, nothing E x E is formed) and in
// FP32 are 100-1000x closer to the FP64 gradient than the reference's own FP32 Cholesky (DESIGN.md section 2,
// tests/test_gpu_transport.py).
// Then, with M recovered from P = u K v, K = exp(-lambda M):  W = (dL/dM) / M  and
//     dL/da_i = (sum_j W_ij) a_i - sum_j W_ij c_j,      dL/dc_j = (sum_i W_ij) c_j - sum_i W_ij a_i
// (a, c the normalised features) as two tiled FP32 products that never materialise W.
// Deterministic: fixed-order partial sums, no floating-point atomics.
// Two instantiations of the same passes: the dense one (P and V read from [N][E][E] tensors, dcd_gmw_transport_bwd) and the
// terms one for a loss on (sum P, trace P) only (dcd_gmw_transport_terms_bwd): P rebuilt from the forward's K, u, v and
// V = alpha 11^T + beta I formed in registers, so that only K is E x E; same results bit for bit on the same P and V values.
#include "gmw_mlp.cuh"

namespace dcd {
namespace {

constexpr int TB_CHUNKS = 16;           // row chunks of the column passes
enum { ROW_INIT = 0, ROW_MATVEC = 1, ROW_U3 = 2 };
enum { CG_INIT = 0, CG_RHS = 1, CG_UPDATE = 2 };

struct TbWs {                           // per-object vectors of length E unless noted
    float* r1;      // lambda * rowsum(P)
    float* c2;      // lambda * colsum(P)
    float* u1;      // lambda * rowsum(V * P)
    float* u2;      // lambda * colsum(V * P)
    float* x;       // CG solution
    float* r;       // CG residual
    float* p;       // CG direction
    float* y;       // row-pass result (already divided by r1, 0 for row 0)
    float* u3;
    float* part;    // [2][TB_CHUNKS][E] column-pass partials
    float* scal;    // [8]: rr, rr0, done, iterations
    float* nrm;     // [4][E]: |f4|, |f6| (clamped), then unused
};

// Sources of the two E x E operands of the passes below, the plan P and V = dL/dP.  A kernel binds a source to its object
// (`bind`) and reads row i through `row(i)`: at(j) one entry, at4(j) the four entries j..j+3 (j % 4 == 0, 16-byte aligned).
//   PlanDense  the P that dcd_gmw_transport_fwd wrote.
//   PlanFromK  P rebuilt from that call's K, u and v as (u_i K_ij) v_j: the two roundings of transport_p_kernel, so every
//              entry is bit-identical to the written plan and nothing E x E but K is read.
//   GradDense  a dense V [N][E][E] (streamed: read once per pass).
//   GradTerms  V = alpha 11^T + beta I, the gradient of a loss on (sum P, trace P), from terms [N][2] = (alpha, beta) in
//              registers; alpha + beta is rounded once per object.
// With the same P and V values the two instantiations run the same loads-to-arithmetic sequence: same results, bit for bit.
struct PlanDense {
    const float* P;
    struct Row {
        const float* p;
        __device__ __forceinline__ float at(int j) const { return __ldg(p + j); }
        __device__ __forceinline__ float4 at4(int j) const { return __ldg(reinterpret_cast<const float4*>(p + j)); }
    };
    struct Obj {
        const float* P;
        int E;
        __device__ __forceinline__ Row row(int i) const { return {P + (int64_t)i * E}; }
    };
    __device__ __forceinline__ Obj bind(int64_t obj, int E) const { return {P + obj * (int64_t)E * E, E}; }
};

struct PlanFromK {
    const float* K;
    const float* u;
    const float* v;
    struct Row {
        const float* k;
        float ui;
        const float* v;
        __device__ __forceinline__ float at(int j) const { return __fmul_rn(__fmul_rn(ui, __ldg(k + j)), __ldg(v + j)); }
        __device__ __forceinline__ float4 at4(int j) const {
            const float4 kk = __ldg(reinterpret_cast<const float4*>(k + j));
            return make_float4(__fmul_rn(__fmul_rn(ui, kk.x), __ldg(v + j)), __fmul_rn(__fmul_rn(ui, kk.y), __ldg(v + j + 1)),
                               __fmul_rn(__fmul_rn(ui, kk.z), __ldg(v + j + 2)), __fmul_rn(__fmul_rn(ui, kk.w), __ldg(v + j + 3)));
        }
    };
    struct Obj {
        const float* K;
        const float* u;
        const float* v;
        int E;
        __device__ __forceinline__ Row row(int i) const { return {K + (int64_t)i * E, __ldg(u + i), v}; }
    };
    __device__ __forceinline__ Obj bind(int64_t obj, int E) const {
        return {K + obj * (int64_t)E * E, u + obj * (int64_t)E, v + obj * (int64_t)E, E};
    }
};

struct GradDense {
    const float* V;
    struct Row {
        const float* p;
        __device__ __forceinline__ float at(int j) const { return __ldcs(p + j); }
        __device__ __forceinline__ float4 at4(int j) const { return __ldcs(reinterpret_cast<const float4*>(p + j)); }
    };
    struct Obj {
        const float* V;
        int E;
        __device__ __forceinline__ Row row(int i) const { return {V + (int64_t)i * E}; }
    };
    __device__ __forceinline__ Obj bind(int64_t obj, int E) const { return {V + obj * (int64_t)E * E, E}; }
};

struct GradTerms {
    const float* terms;
    struct Row {
        float off, diag;
        int i;
        __device__ __forceinline__ float at(int j) const { return j == i ? diag : off; }
        __device__ __forceinline__ float4 at4(int j) const { return make_float4(at(j), at(j + 1), at(j + 2), at(j + 3)); }
    };
    struct Obj {
        float off, diag;
        __device__ __forceinline__ Row row(int i) const { return {off, diag, i}; }
    };
    __device__ __forceinline__ Obj bind(int64_t obj, int) const {
        const float alpha = __ldg(terms + 2 * obj);
        return {alpha, __fadd_rn(alpha, __ldg(terms + 2 * obj + 1))};
    }
};

// warp per row i of P
template <int MODE, class Plan, class Grad>
__global__ void __launch_bounds__(256) tb_row_kernel(Plan plan, Grad grad, int E, float lambda,
                                                     const float* __restrict__ vec, const float* __restrict__ r1, const float* __restrict__ u1,
                                                     const float* __restrict__ scal, float* __restrict__ out0, float* __restrict__ out1,
                                                     int64_t stride_scal) {
    const int64_t obj = blockIdx.y;
    if (MODE == ROW_MATVEC && scal[obj * stride_scal + 2] != 0.f) return;         // this object's CG has converged
    const int i = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= E) return;
    const auto Pp = plan.bind(obj, E).row(i);
    const auto Vp = grad.bind(obj, E).row(i);                                      // read by ROW_INIT only
    const float* xp = MODE == ROW_INIT ? nullptr : vec + obj * (int64_t)E;
    float a = 0.f, b = 0.f;
    if ((E & 3) == 0) {
        const float4* x4 = reinterpret_cast<const float4*>(xp);
        const int E4 = E >> 2;
#pragma unroll 4
        for (int j = lane; j < E4; j += 32) {
            const float4 p = Pp.at4(4 * j);
            if constexpr (MODE == ROW_INIT) {
                const float4 v = Vp.at4(4 * j);
                a += (p.x + p.y) + (p.z + p.w);
                b = fmaf(p.w, v.w, fmaf(p.z, v.z, fmaf(p.y, v.y, fmaf(p.x, v.x, b))));
            } else {
                const float4 x = x4[j];
                a = fmaf(p.w, x.w, fmaf(p.z, x.z, fmaf(p.y, x.y, fmaf(p.x, x.x, a))));
            }
        }
    } else {
        for (int j = lane; j < E; j += 32) {
            const float p = Pp.at(j);
            if constexpr (MODE == ROW_INIT) { a += p; b = fmaf(p, Vp.at(j), b); }
            else a = fmaf(p, xp[j], a);
        }
    }
    a = warp_sum(a);
    if (MODE == ROW_INIT) b = warp_sum(b);
    if (lane != 0) return;
    const int64_t o = obj * (int64_t)E + i;
    if (MODE == ROW_INIT) {
        const float rr = lambda * a, uu = lambda * b;
        out0[o] = rr;                                        // r1
        out1[o] = uu;                                        // u1
    } else if (MODE == ROW_MATVEC) {
        out0[o] = i >= 1 ? __fdiv_rn(lambda * a, r1[o]) : 0.f;                      // y = (B' p) / r1
    } else {
        out0[o] = i >= 1 ? __fdiv_rn(u1[o] - lambda * a, r1[o]) : 0.f;              // u3
    }
}

// y0 = u1 / r1 (0 for row 0): the weights of the column pass that forms the right-hand side
__global__ void __launch_bounds__(256) tb_y0_kernel(const float* __restrict__ u1, const float* __restrict__ r1, int E, float* __restrict__ y) {
    const int64_t obj = blockIdx.y;
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= E) return;
    const int64_t o = obj * (int64_t)E + i;
    y[o] = i >= 1 ? __fdiv_rn(u1[o], r1[o]) : 0.f;
}

// thread per column j, rows split into TB_CHUNKS chunks: part[0][chunk][j] = sum_i P_ij t_i  (INIT: t = 1 and
// part[1] = sum_i P_ij V_ij)
template <bool INIT, class Plan, class Grad>
__global__ void __launch_bounds__(256) tb_col_kernel(Plan plan, Grad grad, int E,
                                                     const float* __restrict__ t, const float* __restrict__ scal, int64_t stride_scal,
                                                     float* __restrict__ part) {
    const int64_t obj = blockIdx.z;
    if (!INIT && scal != nullptr && scal[obj * stride_scal + 2] != 0.f) return;
    const int j = blockIdx.x * 256 + threadIdx.x;
    const int rows = (E + TB_CHUNKS - 1) / TB_CHUNKS;
    const int ib = blockIdx.y * rows, ie = min(E, ib + rows);
    if (j >= E) return;
    const auto Pm = plan.bind(obj, E);
    const auto Vm = grad.bind(obj, E);                                             // read by INIT only
    const float* tp = INIT ? nullptr : t + obj * (int64_t)E;
    float a = 0.f, b = 0.f;
#pragma unroll 4
    for (int i = ib; i < ie; ++i) {
        const float p = Pm.row(i).at(j);
        if constexpr (INIT) { a += p; b = fmaf(p, Vm.row(i).at(j), b); }
        else a = fmaf(p, tp[i], a);
    }
    float* o = part + (obj * 2 * TB_CHUNKS + blockIdx.y) * (int64_t)E + j;
    o[0] = a;
    if (INIT) o[(int64_t)TB_CHUNKS * E] = b;
}

__device__ __forceinline__ float block_sum_256(float v, float* red) {
    v = warp_sum(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += red[w];
    return t;
}

// vector stage of the conjugate-gradient solve, one CTA per object (E <= 256 * TB_EPT)
constexpr int TB_EPT = 128;             // E <= 32 768
template <int STAGE>
__global__ void __launch_bounds__(256) tb_cg_kernel(TbWs w, int E, float lambda, float tol2, int64_t stride_vec) {
    __shared__ float red[8];
    const int64_t obj = blockIdx.x;
    const int64_t o = obj * stride_vec;
    float* scal = w.scal + obj * 8;
    const float* part = w.part + obj * 2 * TB_CHUNKS * (int64_t)E;
    if (STAGE == CG_UPDATE && scal[2] != 0.f) return;
    auto colsum = [&](int which, int j) {
        float t = 0.f;
#pragma unroll
        for (int k = 0; k < TB_CHUNKS; ++k) t += part[((int64_t)which * TB_CHUNKS + k) * E + j];
        return lambda * t;
    };
    if (STAGE == CG_INIT) {
        for (int j = threadIdx.x; j < E; j += 256) {
            w.c2[o + j] = colsum(0, j);
            w.u2[o + j] = colsum(1, j);
        }
        return;
    }
    if (STAGE == CG_RHS) {
        float rr = 0.f;
        for (int j = threadIdx.x; j < E; j += 256) {
            const float rhs = w.u2[o + j] - colsum(0, j);
            w.x[o + j] = 0.f;
            w.r[o + j] = rhs;
            w.p[o + j] = rhs;
            rr = fmaf(rhs, rhs, rr);
        }
        rr = block_sum_256(rr, red);
        if (threadIdx.x == 0) {
            scal[0] = rr;
            scal[1] = rr;
            scal[2] = (rr > 0.f) ? 0.f : 1.f;                // a zero right-hand side: x = 0
            scal[3] = 0.f;
        }
        return;
    }
    // CG_UPDATE:  Ap = c2 * p - lambda * B'^T y
    const float rr = scal[0], rr0 = scal[1];
    float pAp = 0.f;
    for (int j = threadIdx.x; j < E; j += 256) {
        const float p = w.p[o + j];
        const float Ap = fmaf(w.c2[o + j], p, -colsum(0, j));
        pAp = fmaf(p, Ap, pAp);
    }
    pAp = block_sum_256(pAp, red);
    if (!(pAp > 0.f)) {                                      // breakdown (S is SPD: only by rounding at convergence)
        if (threadIdx.x == 0) scal[2] = 1.f;
        return;
    }
    const float alpha = rr / pAp;
    float rn = 0.f;
    for (int j = threadIdx.x; j < E; j += 256) {
        const float p = w.p[o + j];
        const float Ap = fmaf(w.c2[o + j], p, -colsum(0, j));
        w.x[o + j] = fmaf(alpha, p, w.x[o + j]);
        const float r = fmaf(-alpha, Ap, w.r[o + j]);
        w.r[o + j] = r;
        rn = fmaf(r, r, rn);
    }
    rn = block_sum_256(rn, red);
    const float beta = rn / rr;
    for (int j = threadIdx.x; j < E; j += 256) w.p[o + j] = fmaf(beta, w.p[o + j], w.r[o + j]);
    if (threadIdx.x == 0) {
        scal[0] = rn;
        scal[3] += 1.f;
        if (!(rn > tol2 * rr0)) scal[2] = 1.f;
    }
}

// per-edge norms of the final features (clamped like F.normalize, model.py:176-177)
__global__ void __launch_bounds__(256) tb_norm_kernel(const float* __restrict__ feat4, const float* __restrict__ feat6, int E,
                                                      float* __restrict__ nrm, int64_t stride_nrm) {
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
    nrm[obj * stride_nrm + e] = fmaxf(sqrtf(n4), 1e-12f);
    nrm[obj * stride_nrm + E + e] = fmaxf(sqrtf(n6), 1e-12f);
}

// W_ij = lambda P_ij (u3_i + x_j - V_ij) / M_ij,   M_ij = (ln u_i + ln v_j - ln P_ij) / lambda   (P = u K v, K = exp(-lambda M))
__device__ __forceinline__ float w_entry(float p, float v, float u3i, float xj, float lnu_i, float lnv_j, float lambda, float inv_lambda) {
    if (!(p > 0.f)) return 0.f;
    const float m = (lnu_i + lnv_j - logf(p)) * inv_lambda;
    if (!(m > 1e-15f)) return 0.f;                           // the reference's clamp_min(1e-30) on M^2 passes no gradient there
    return __fdiv_rn(lambda * p * (u3i + xj - v), m);
}

// Tiled product with the features of the OTHER net, never materialising W.
// TRANS == false: the CTA owns 64 rows i (edges of net 4):  out[c][i] = rsW_i a_i[c] - sum_j W_ij c_j[c]
// TRANS == true : the CTA owns 64 columns j (edges of net 6): out[c][j] = csW_j c_j[c] - sum_i W_ij a_i[c]
// 256 threads: tile loads 64 x 64 of P and V per step; accumulators 4 own-edges x 8 channels per thread.
constexpr int FT = 64;
constexpr int FT_WS = FT + 4;           // WsT[k][own] row stride (floats; keeps 16-byte alignment)
constexpr size_t kFeatSmem = ((size_t)FT * FT_WS + (size_t)FT * CH + 4 * FT + 2 * FT) * sizeof(float);

template <bool TRANS, class Plan, class Grad>
__global__ void __launch_bounds__(256) tb_feat_kernel(Plan plan, Grad grad, const float* __restrict__ feat_own, const float* __restrict__ feat_oth,
                                                      const float* __restrict__ nrm, int64_t stride_nrm,
                                                      const float* __restrict__ uvec, const float* __restrict__ vvec,
                                                      const float* __restrict__ u3, const float* __restrict__ x,
                                                      int E, float lambda, float* __restrict__ out) {
    extern __shared__ __align__(16) float fsm[];
    float* WsT = fsm;                                        // [FT k][FT_WS own]
    float* FsT = WsT + FT * FT_WS;                           // [FT k][CH]
    float* red_s = FsT + FT * CH;                            // [4][FT]
    float* kvec_s = red_s + 4 * FT;                          // [2][FT]: per-k (other index) vectors of the current step
    const int64_t obj = blockIdx.y;
    const int own0 = blockIdx.x * FT;
    const int tid = threadIdx.x;
    const float inv_lambda = 1.0f / lambda;
    const int64_t vo = obj * (int64_t)E;
    const float* n_own = nrm + obj * stride_nrm + (TRANS ? E : 0);
    const float* n_oth = nrm + obj * stride_nrm + (TRANS ? 0 : E);
    const auto Pm = plan.bind(obj, E);
    const auto Vm = grad.bind(obj, E);

    // tile-load mapping: `lo` = own index inside the tile, `seg` = 16 consecutive k
    const int lo = tid & 63, seg = tid >> 6;
    const int own = own0 + lo;
    const bool own_ok = own < E;
    // per-own vectors: rows need (u3_i, ln u_i); columns need (x_j, ln v_j)
    const float own_a = own_ok ? (TRANS ? x[vo + own] : u3[vo + own]) : 0.f;
    const float own_ln = own_ok ? logf(TRANS ? vvec[vo + own] : uvec[vo + own]) : 0.f;
    float wsum = 0.f;                                        // this thread's share of rsW / csW

    // accumulator mapping: 4 own edges x 8 channels
    const int to = (tid & 15) * 4, tc = (tid >> 4) * 8;
    float acc[4][8];                                         // sum over all steps; each step's 64 terms are summed separately
#pragma unroll                                               // first (two-level summation: W has both signs and the products cancel)
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) acc[a][b] = 0.f;

    for (int k0 = 0; k0 < E; k0 += FT) {
        __syncthreads();                                     // previous step's readers are done
        if (tid < FT) {
            const int k = k0 + tid;
            const bool ok = k < E;
            kvec_s[tid] = ok ? (TRANS ? u3[vo + k] : x[vo + k]) : 0.f;
            kvec_s[FT + tid] = ok ? logf(TRANS ? uvec[vo + k] : vvec[vo + k]) : 0.f;
        }
        // other net's normalised features of the step's 64 edges: FsT[k][c]
        // (a warp moves 8 consecutive edges of 4 channels: full 32-byte sectors in, 32 distinct banks out; the 16-byte
        //  channel chunks of a row are XOR-swizzled by the edge so that the float4 reads below stay aligned)
        for (int idx = tid; idx < FT * CH; idx += 256) {
            const int rest = idx >> 5;
            const int kk = (rest & 7) * 8 + (idx & 7), c = (rest >> 3) * 4 + ((idx >> 3) & 3);
            const int k = k0 + kk;
            FsT[kk * CH + ((((c >> 2) ^ (kk & 7)) << 2) | (c & 3))] =
                k < E ? __fdiv_rn(feat_oth[(obj * CH + c) * (int64_t)E + k], n_oth[k]) : 0.f;
        }
        __syncthreads();
        // W tile -> WsT[k][own]
        if (!TRANS && (E & 3) == 0) {                        // rows of P: four 16-byte loads per thread
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
                const int kk = seg * 16 + q4 * 4, k = k0 + kk;
                float4 p = make_float4(0.f, 0.f, 0.f, 0.f), v = p;
                const bool ok = own_ok && k < E;             // E % 4 == 0: the four columns are valid together
                if (ok) {
                    p = Pm.row(own).at4(k);
                    v = Vm.row(own).at4(k);
                }
                const float pp[4] = {p.x, p.y, p.z, p.w}, vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float wv = ok ? w_entry(pp[q], vv[q], own_a, kvec_s[kk + q], own_ln, kvec_s[FT + kk + q], lambda, inv_lambda) : 0.f;
                    WsT[(kk + q) * FT_WS + lo] = wv;
                    wsum += wv;
                }
            }
        } else {
#pragma unroll 4
            for (int q = 0; q < 16; ++q) {
                const int kk = seg * 16 + q, k = k0 + kk;
                float wv = 0.f;
                if (own_ok && k < E) {
                    const int r = TRANS ? k : own, c = TRANS ? own : k;
                    const float p = Pm.row(r).at(c), v = Vm.row(r).at(c);
                    wv = TRANS ? w_entry(p, v, kvec_s[kk], own_a, kvec_s[FT + kk], own_ln, lambda, inv_lambda)
                               : w_entry(p, v, own_a, kvec_s[kk], own_ln, kvec_s[FT + kk], lambda, inv_lambda);
                }
                WsT[kk * FT_WS + lo] = wv;
                wsum += wv;
            }
        }
        __syncthreads();
        float blk[4][8];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 8; ++b) blk[a][b] = 0.f;
#pragma unroll 8
        for (int kk = 0; kk < FT; ++kk) {
            const float4 wv = *reinterpret_cast<const float4*>(WsT + kk * FT_WS + to);
            const float4 f0 = *reinterpret_cast<const float4*>(FsT + kk * CH + (((tc >> 2) ^ (kk & 7)) << 2));
            const float4 f1 = *reinterpret_cast<const float4*>(FsT + kk * CH + ((((tc >> 2) + 1) ^ (kk & 7)) << 2));
            const float wa[4] = {wv.x, wv.y, wv.z, wv.w};
            const float fb[8] = {f0.x, f0.y, f0.z, f0.w, f1.x, f1.y, f1.z, f1.w};
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 8; ++b) blk[a][b] = fmaf(wa[a], fb[b], blk[a][b]);
        }
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 8; ++b) acc[a][b] += blk[a][b];
    }
    // rsW / csW of the tile's own edges (fixed order over the 4 segments)
    red_s[seg * FT + lo] = wsum;
    __syncthreads();
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int e = own0 + to + a;
        if (e >= E) continue;
        const float sw = (red_s[to + a] + red_s[FT + to + a]) + (red_s[2 * FT + to + a] + red_s[3 * FT + to + a]);
        const float inv_n = 1.0f / n_own[e];
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            const int64_t off = (obj * CH + tc + b) * (int64_t)E + e;
            const float f = feat_own[off] * inv_n;           // normalised own feature
            out[off] = fmaf(sw, f, -acc[a][b]);
        }
    }
}

inline size_t al(size_t x) { return (x + 255) / 256 * 256; }

}  // namespace

// workspace: 9 vectors [N][E] | partials [N][2][16][E] | norms [N][2][E] | scalars [N][8]
size_t gmw_transport_bwd_workspace_bytes(int64_t N, int E) {
    const size_t e = (size_t)E;
    return 9 * al((size_t)N * e * 4) + al((size_t)N * 2 * TB_CHUNKS * e * 4) + al((size_t)N * 2 * e * 4) + al((size_t)N * 8 * 4);
}

namespace {

// the whole backward on one pair of operand sources (see PlanDense ... GradTerms)
template <class Plan, class Grad>
int run_transport_bwd(Plan P, Grad gradP, const float* feat4, const float* feat6, const float* u, const float* v, int64_t N, int E,
                      float lambda, int max_iter, float tol, float* gn4, float* gn6, float* cg_info, void* workspace, cudaStream_t st) {
    if (E > 256 * TB_EPT) return DCD_E_UNSUPPORTED;
    const size_t e = (size_t)E;
    unsigned char* p = reinterpret_cast<unsigned char*>(workspace);
    auto take = [&](size_t bytes) { float* r = reinterpret_cast<float*>(p); p += al(bytes); return r; };
    TbWs w;
    w.r1 = take(N * e * 4); w.c2 = take(N * e * 4); w.u1 = take(N * e * 4); w.u2 = take(N * e * 4);
    w.x = take(N * e * 4); w.r = take(N * e * 4); w.p = take(N * e * 4); w.y = take(N * e * 4);
    w.u3 = take(N * e * 4);
    w.part = take((size_t)N * 2 * TB_CHUNKS * e * 4);
    w.nrm = take((size_t)N * 2 * e * 4);
    w.scal = take((size_t)N * 8 * 4);
    const unsigned eb = (unsigned)((E + 255) / 256), rb = (unsigned)((E + 7) / 8);
    const dim3 rgrid(rb, (unsigned)N), cgrid(eb, TB_CHUNKS, (unsigned)N), vgrid(eb, (unsigned)N);
    const int64_t sv = (int64_t)E;

    // r1, u1 (rows) and c2, u2 (columns) of B = lambda P and V * B
    tb_row_kernel<ROW_INIT><<<rgrid, 256, 0, st>>>(P, gradP, E, lambda, nullptr, nullptr, nullptr, nullptr, w.r1, w.u1, 8);
    tb_col_kernel<true><<<cgrid, 256, 0, st>>>(P, gradP, E, nullptr, nullptr, 8, w.part);
    tb_cg_kernel<CG_INIT><<<(unsigned)N, 256, 0, st>>>(w, E, lambda, 0.f, sv);
    // rhs = u2 - B'^T (u1 / r1)
    tb_y0_kernel<<<vgrid, 256, 0, st>>>(w.u1, w.r1, E, w.y);
    tb_col_kernel<false><<<cgrid, 256, 0, st>>>(P, gradP, E, w.y, nullptr, 8, w.part);
    tb_cg_kernel<CG_RHS><<<(unsigned)N, 256, 0, st>>>(w, E, lambda, 0.f, sv);
    DCD_CHECK_LAUNCH();
    // conjugate gradients on S x = rhs, S p = c2 * p - B'^T ((B' p) / r1); converged objects skip their passes
    for (int it = 0; it < max_iter; ++it) {
        tb_row_kernel<ROW_MATVEC><<<rgrid, 256, 0, st>>>(P, gradP, E, lambda, w.p, w.r1, nullptr, w.scal, w.y, nullptr, 8);
        tb_col_kernel<false><<<cgrid, 256, 0, st>>>(P, gradP, E, w.y, w.scal, 8, w.part);
        tb_cg_kernel<CG_UPDATE><<<(unsigned)N, 256, 0, st>>>(w, E, lambda, tol * tol, sv);
    }
    DCD_CHECK_LAUNCH();
    // u3 = (u1 - B' x) / r1
    tb_row_kernel<ROW_U3><<<rgrid, 256, 0, st>>>(P, gradP, E, lambda, w.x, w.r1, w.u1, nullptr, w.u3, nullptr, 8);
    // gradients of the normalised features
    tb_norm_kernel<<<vgrid, 256, 0, st>>>(feat4, feat6, E, w.nrm, 2 * sv);
    cudaFuncSetAttribute(tb_feat_kernel<false, Plan, Grad>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFeatSmem);
    cudaFuncSetAttribute(tb_feat_kernel<true, Plan, Grad>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFeatSmem);
    const dim3 fgrid((unsigned)((E + FT - 1) / FT), (unsigned)N);
    tb_feat_kernel<false><<<fgrid, 256, kFeatSmem, st>>>(P, gradP, feat4, feat6, w.nrm, 2 * sv, u, v, w.u3, w.x, E, lambda, gn4);
    tb_feat_kernel<true><<<fgrid, 256, kFeatSmem, st>>>(P, gradP, feat6, feat4, w.nrm, 2 * sv, u, v, w.u3, w.x, E, lambda, gn6);
    if (cg_info != nullptr) cudaMemcpyAsync(cg_info, w.scal, (size_t)N * 8 * sizeof(float), cudaMemcpyDeviceToDevice, st);
    DCD_CHECK_LAUNCH();
    return DCD_OK;
}

}  // namespace

int launch_gmw_transport_bwd(const float* feat4, const float* feat6, const float* P, const float* u, const float* v,
                             const float* gradP, int64_t N, int E, float lambda, int max_iter, float tol,
                             float* gn4, float* gn6, float* cg_info, void* workspace, cudaStream_t st) {
    return run_transport_bwd(PlanDense{P}, GradDense{gradP}, feat4, feat6, u, v, N, E, lambda, max_iter, tol, gn4, gn6, cg_info,
                             workspace, st);
}

// the plan from the forward's K (+ u, v), dL/dP = alpha 11^T + beta I from grad_terms [N][2]
int launch_gmw_transport_terms_bwd(const float* feat4, const float* feat6, const float* K, const float* u, const float* v,
                                   const float* grad_terms, int64_t N, int E, float lambda, int max_iter, float tol,
                                   float* gn4, float* gn6, float* cg_info, void* workspace, cudaStream_t st) {
    return run_transport_bwd(PlanFromK{K, u, v}, GradTerms{grad_terms}, feat4, feat6, u, v, N, E, lambda, max_iter, tol, gn4, gn6,
                             cg_info, workspace, st);
}

}  // namespace dcd
