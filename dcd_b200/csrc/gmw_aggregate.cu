// GMW weighted depth aggregation (forward + backward) for sm_100a.
//
// Replaces compute_reg_loss's gather + softmax + weighted sum (GMW/main.py:364-371) and its autograd.
// One warp per object: k (=1500) selected edges are gathered through idx, the softmax follows torch's
// three passes (max, sum of exp(x-max), exp(x-max)/sum) and every reduction is a warp-shuffle tree.
#include "dcd_common.cuh"

namespace dcd {
namespace {

constexpr int AGG_THREADS = 256;

struct Softmax {
    float mx, sum;
};

// an index outside [0, E) must not fault (torch.gather raises there; the Python wrapper validates on request)
__device__ __forceinline__ int64_t edge_id(const int64_t* __restrict__ id_row, int r, int64_t E) {
    const int64_t id = id_row[r];
    return id < 0 ? 0 : (id >= E ? E - 1 : id);
}

__device__ __forceinline__ Softmax warp_softmax_stats(const float* __restrict__ w_row,
                                                      const int64_t* __restrict__ id_row, int k, int64_t E, int lane) {
    float mx = -INFINITY;
    for (int r = lane; r < k; r += 32) mx = fmaxf(mx, __ldg(w_row + edge_id(id_row, r, E)));
    mx = warp_max(mx);
    float s = 0.f;
    for (int r = lane; r < k; r += 32) s += expf(__ldg(w_row + edge_id(id_row, r, E)) - mx);
    s = warp_sum(s);
    return {mx, s};
}

// RESCALE (dcd_dgde_gmw_refine_fwd): lane 0 also moves the detector location raw_loc [N,3] to the weighted depth it just
// wrote (ray_rescale_one with h = dims[:, 1], dims (l,h,w)) -> loc_out [N,3]: the values of gmw_ray_rescale_kernel on depth_out.
template <bool RESCALE>
__global__ void __launch_bounds__(AGG_THREADS)
gmw_aggregate_fwd_kernel(const float* __restrict__ reg_w, const float* __restrict__ depths,
                         const int64_t* __restrict__ idx, int64_t N, int64_t E, int k, int sel,
                         float* __restrict__ depth_out, float* __restrict__ probs, const float* __restrict__ raw_loc,
                         const float* __restrict__ dims, float* __restrict__ loc_out) {
    const int lane = threadIdx.x & 31;
    const int64_t obj = (int64_t)blockIdx.x * (AGG_THREADS / 32) + (threadIdx.x >> 5);
    if (obj >= N) return;
    const float* w_row = reg_w + obj * E;
    const int64_t* id_row = idx + obj * k;
    const float* z_row = depths + obj * (sel ? (int64_t)k : E);
    const Softmax sm = warp_softmax_stats(w_row, id_row, k, E, lane);
    float acc = 0.f;
    for (int r = lane; r < k; r += 32) {
        const int64_t id = edge_id(id_row, r, E);
        const float p = __fdiv_rn(expf(__ldg(w_row + id) - sm.mx), sm.sum);
        const float z = sel ? __ldg(z_row + r) : __ldg(z_row + id);
        if (probs != nullptr) probs[obj * k + r] = p;
        acc += z * p;
    }
    acc = warp_sum(acc);
    if (lane == 0) {
        depth_out[obj] = acc;
        if constexpr (RESCALE)
            ray_rescale_one(__ldg(raw_loc + obj * 3), __ldg(raw_loc + obj * 3 + 1), __ldg(raw_loc + obj * 3 + 2), acc,
                            __ldg(dims + obj * 3 + 1), loc_out + obj * 3);
    }
}

// Claim of slot r on its edge, stored in the grad_w row as the bits of a positive NaN whose payload k - r is largest for the
// first slot.  A computed gradient is never such a NaN: the GPU's float arithmetic returns the canonical NaN 0x7fffffff, and
// k - r <= k <= DCD_AGG_BWD_MAX_K = 2^22 stays below that payload.
__device__ __forceinline__ int slot_claim(int r, int k) { return 0x7f800000 | (k - r); }

// The backward of the gather is torch's scatter_add: a repeated index receives the SUM of its slots' gradients.  Every slot
// claims its edge with an integer atomicMax (the first slot wins); if no slot lost its claim (all indices distinct, the case of
// compute_z's top-k) each slot writes its value as a plain store.  Otherwise the warp walks the slots in ascending chunks of
// 32: the lanes of a chunk that share an edge are summed by the lowest of them in lane order, onto the edge's running sum
// from earlier chunks (the first slot starts it), so repeated edges are summed in ascending slot order, deterministically,
// without floating-point atomics.
__global__ void __launch_bounds__(AGG_THREADS)
gmw_aggregate_bwd_kernel(const float* __restrict__ reg_w, const float* __restrict__ depths,
                         const int64_t* __restrict__ idx, int64_t N, int64_t E, int k, int sel,
                         const float* __restrict__ grad_out, float* __restrict__ grad_w,
                         float* __restrict__ grad_z) {
    const int lane = threadIdx.x & 31;
    const int64_t obj = (int64_t)blockIdx.x * (AGG_THREADS / 32) + (threadIdx.x >> 5);
    if (obj >= N) return;
    const float* w_row = reg_w + obj * E;
    const int64_t* id_row = idx + obj * k;
    const float* z_row = depths + obj * (sel ? (int64_t)k : E);
    float* gw_row = grad_w + obj * E;
    int* claim_row = reinterpret_cast<int*>(gw_row);
    float* gz_dense = grad_z != nullptr && !sel ? grad_z + obj * E : nullptr;
    for (int64_t e = lane; e < E; e += 32) gw_row[e] = 0.f;
    if (gz_dense != nullptr)
        for (int64_t e = lane; e < E; e += 32) gz_dense[e] = 0.f;
    const Softmax sm = warp_softmax_stats(w_row, id_row, k, E, lane);
    float acc = 0.f;
    for (int r = lane; r < k; r += 32) {
        const int64_t id = edge_id(id_row, r, E);
        const float p = __fdiv_rn(expf(__ldg(w_row + id) - sm.mx), sm.sum);
        const float z = sel ? __ldg(z_row + r) : __ldg(z_row + id);
        acc += z * p;
    }
    const float Zbar = warp_sum(acc);
    const float g = __ldg(grad_out + obj);
    __syncwarp();   // orders the zero fill before the claims
    for (int r = lane; r < k; r += 32) atomicMax(claim_row + edge_id(id_row, r, E), slot_claim(r, k));
    __syncwarp();
    bool lost = false;
    for (int r = lane; r < k; r += 32) lost |= __ldcg(claim_row + edge_id(id_row, r, E)) != slot_claim(r, k);
    const bool repeated = __any_sync(0xffffffffu, lost);
    __syncwarp();   // every claim is read before a value overwrites one
    if (!repeated) {
        for (int r = lane; r < k; r += 32) {
            const int64_t id = edge_id(id_row, r, E);
            const float p = __fdiv_rn(expf(__ldg(w_row + id) - sm.mx), sm.sum);
            const float z = sel ? __ldg(z_row + r) : __ldg(z_row + id);
            gw_row[id] = g * p * (z - Zbar);
            if (grad_z != nullptr) {
                if (sel) grad_z[obj * k + r] = g * p;
                else gz_dense[id] = g * p;
            }
        }
        return;
    }
    for (int base = 0; base < k; base += 32) {
        const int r = base + lane;
        int64_t id = -1;
        float vw = 0.f, vz = 0.f;
        if (r < k) {
            id = edge_id(id_row, r, E);
            const float p = __fdiv_rn(expf(__ldg(w_row + id) - sm.mx), sm.sum);
            const float z = sel ? __ldg(z_row + r) : __ldg(z_row + id);
            vw = g * p * (z - Zbar);
            vz = g * p;
            if (grad_z != nullptr && sel) grad_z[obj * k + r] = vz;
        }
        const unsigned grp = __match_any_sync(0xffffffffu, (unsigned long long)id);
        if (r < k) {
            const bool lead = lane == __ffs(grp) - 1;
            float sw = vw, sz = vz;
            if (lead) {
                const int cur = __ldcg(claim_row + id);
                if (cur != slot_claim(r, k)) {                       // not the edge's first slot: continue its sum
                    sw = __fadd_rn(__int_as_float(cur), vw);
                    if (gz_dense != nullptr) sz = __fadd_rn(__ldcg(gz_dense + id), vz);
                }
            }
            for (unsigned m = grp & (grp - 1u); m != 0u; m &= m - 1u) {   // the group's other lanes, ascending
                const int j = __ffs(m) - 1;
                const float aw = __shfl_sync(grp, vw, j), az = __shfl_sync(grp, vz, j);
                if (lead) {
                    sw = __fadd_rn(sw, aw);
                    sz = __fadd_rn(sz, az);
                }
            }
            if (lead) {
                gw_row[id] = sw;
                if (gz_dense != nullptr) gz_dense[id] = sz;
            }
        }
        __syncwarp();   // this chunk's sums are stored before the next chunk reads them
    }
}

}  // namespace

int launch_gmw_aggregate_fwd(const float* reg_w, const float* depths, const int64_t* idx, int64_t N, int64_t E,
                             int k, int sel, float* depth_out, float* probs, cudaStream_t st) {
    const int64_t per = AGG_THREADS / 32;
    const unsigned grid = (unsigned)((N + per - 1) / per);
    gmw_aggregate_fwd_kernel<false><<<grid, AGG_THREADS, 0, st>>>(reg_w, depths, idx, N, E, k, sel, depth_out, probs, nullptr,
                                                                  nullptr, nullptr);
    DCD_CHECK_LAUNCH();
    return DCD_OK;
}

int launch_gmw_aggregate_rescale_fwd(const float* reg_w, const float* depths, const int64_t* idx, int64_t N, int64_t E, int k,
                                     int sel, float* depth_out, const float* raw_loc, const float* dims, float* loc_out,
                                     cudaStream_t st) {
    const int64_t per = AGG_THREADS / 32;
    const unsigned grid = (unsigned)((N + per - 1) / per);
    gmw_aggregate_fwd_kernel<true><<<grid, AGG_THREADS, 0, st>>>(reg_w, depths, idx, N, E, k, sel, depth_out, nullptr, raw_loc,
                                                                 dims, loc_out);
    DCD_CHECK_LAUNCH();
    return DCD_OK;
}

int launch_gmw_aggregate_bwd(const float* reg_w, const float* depths, const int64_t* idx, int64_t N, int64_t E,
                             int k, int sel, const float* grad_out, float* grad_w, float* grad_z, cudaStream_t st) {
    const int64_t per = AGG_THREADS / 32;
    const unsigned grid = (unsigned)((N + per - 1) / per);
    gmw_aggregate_bwd_kernel<<<grid, AGG_THREADS, 0, st>>>(reg_w, depths, idx, N, E, k, sel, grad_out, grad_w, grad_z);
    DCD_CHECK_LAUNCH();
    return DCD_OK;
}

}  // namespace dcd
