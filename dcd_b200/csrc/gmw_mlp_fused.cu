// GMW edge-feature MLP forward, inference form: ONE kernel for the whole net (conv_in + 12 blocks; each block's
// preconv and conv1 folded into one layer: 1 + 24 layers instead of 1 + 36), the objects' activations never leave
// the chip (sm_100a: tcgen05 + TMEM, persistent co-resident CTA groups).
//
// The layer-wise kernels (gmw_mlp_tc.cu) are bound by HBM: every context norm needs the statistics of the
// whole object, so each of the 24 normalised layers writes its output and reads it back (198 MB / object).
// Here a group of 24 CTAs works on THREE objects of one net at a time: CTA r holds the edge slice [r*ES, (r+1)*ES)
// of each of them (ES <= 112) for ALL 128 channels on chip for the whole network, the three slices side by side
// (3 ES = 336 columns = 7 MMA tiles of 48 edges per layer).  The only thing the CTAs exchange per context norm is
// the per-channel (mean, M2) partial of a slice (1 KB per CTA and object, through L2 with self-validating words:
// no fences, no barriers) — and because the three objects follow each other through every layer, one object's
// exchange (the drain of its last MMAs, the L2 round trip between 24 CTAs, the merge) runs behind the other two
// objects' tiles instead of idling the tensor pipe at the end of every layer; the layer weights are fetched once
// for three objects.  Groups are plain consecutive CTAs of a cooperative launch (all CTAs resident, one per SM):
// 6 groups use 144 of the 148 SMs.
// Per CTA (E <= 2688, i.e. up to the reference's n = 73 keypoints; at least 3 units of 16 edges per slice, n >= 40):
//   * residual stream X        : FP32 in shared memory, [3 ES/4][128 ch] float4          (172 KB)
//   * layer output (P, Y1, Y2) : FP32 accumulators in tensor memory, columns [0, 3 ES)   (336 of 512 columns);
//                                every GEMM overwrites its own input tile in place
//   * weights                  : FP16 hi/lo pairs as the A operand in tensor memory, columns [384, 512),
//                                reloaded per layer from an L2-resident pre-split image (64 KB / layer)
//   * B operand                : two 24 KB buffers (hi + lo of a 48-edge tile, MN-major, no swizzle),
//                                written by the threads that produce the values (thread = channel)
// Warp roles: 12 converter warps (thread = channel, a warp converts one 16-edge unit per tile: accumulators ->
// context norm / ReLU / residual -> FP16 hi/lo operand; statistics of the layer output two tiles behind), the MMA
// warp (weights of its lane quarter -> tensor memory; tcgen05.mma from an elected lane), 3 statistics warps (weights
// of their lane quarters; publish / collect / merge the slices' statistics and hand the three rank-subset results back:
// the converter threads finish (mean, rstd) of their channel themselves when they pick them up).  Hand-offs
// are mbarriers and named barriers; there is no CTA-wide barrier per tile.  Waits that would spin against the
// warps being waited for back off (nanosleep): the statistics warps are the shortest resource of the kernel.
// Arithmetic is the one of the layer-wise kernels (FP16x3 split, power-of-two weight scaling, FP32 statistics) up to
// the folded layer (Wf = W1.Wp formed in FP64, rounded once), the shifted-sum form of the slice statistics, rsqrtf for
// the reciprocal standard deviation and the order in which the partials are merged (fixed: results are bit-identical
// whichever place of a triple, chunk or schedule an object takes).
// HBM traffic: keypoints in, edge weights out (paired schedule) or final features out (2.75 MB / object).
#include <type_traits>
#include "gmw_tc_common.cuh"

// back-off (ns) of the waits whose spinning competes with the warps being waited for; 0 = spin on the test
#ifndef DCD_FUSED_STAT_SLEEP
#define DCD_FUSED_STAT_SLEEP 40      // converters waiting for a layer's statistics
#endif
#ifndef DCD_FUSED_CONV_FINAL
#define DCD_FUSED_CONV_FINAL 1       // 1: the last merge of a context norm's statistics runs on the converter threads
#endif
#ifndef DCD_FUSED_POLL_GRACE
#define DCD_FUSED_POLL_GRACE 500    // statistics warps: pause between publishing a slice and the first look at the others'
#endif
#ifndef DCD_FUSED_DONE_SLEEP
#define DCD_FUSED_DONE_SLEEP 20      // converters waiting for an operand buffer
#endif
#ifndef DCD_FUSED_STAT_NBAR
#define DCD_FUSED_STAT_NBAR 0        // 1: converters wait for a layer's statistics on a hardware named barrier, 0: on an mbarrier
#endif
#ifndef DCD_FUSED_STEP_UNROLL
#define DCD_FUSED_STEP_UNROLL 2      // unroll depth of the converters' step loop (1: 0.5 % slower, DESIGN.md §5)
#endif

namespace dcd {
// Optional in-kernel timeline (build with -DDCD_FUSED_TRACE, see profiles/trace_fused.py): lane 0 of converter warp 0
// and of the MMA warp and the first statistics warp of CTA 0 record (tag, clock64) pairs; read back with dcd_debug_fused_trace().
// -DDCD_FUSED_TRACE=2 adds the fine-grained tags (each costs ~100 clk: the coarse level keeps the timeline honest).
#ifdef DCD_FUSED_TRACE
__device__ long long g_trace[12288];
__device__ int g_trace_n[3];
#ifndef DCD_FUSED_TRACE_CTA
#define DCD_FUSED_TRACE_CTA 0
#endif
#ifndef DCD_FUSED_TRACE_WARP
#define DCD_FUSED_TRACE_WARP 0
#endif
#define TR_DECL const bool trace_on = blockIdx.x == DCD_FUSED_TRACE_CTA && (warp == DCD_FUSED_TRACE_WARP || warp == FCONV_WARPS || warp == FCONV_WARPS + 1); int tr_k = 0;
#define TR(slot, tag)                                                       \
    do {                                                                    \
        if (trace_on && lane == 0 && tr_k < 2048) {                         \
            g_trace[(slot) * 4096 + 2 * tr_k] = (tag);                      \
            g_trace[(slot) * 4096 + 2 * tr_k + 1] = clock64();              \
            ++tr_k;                                                         \
            g_trace_n[slot] = tr_k;                                         \
        }                                                                   \
    } while (0)
#else
#define TR_DECL
#define TR(slot, tag) do { } while (0)
#endif
#if defined(DCD_FUSED_TRACE) && DCD_FUSED_TRACE + 0 >= 2
#define TRF(slot, tag) TR(slot, tag)     // fine-grained tags (they cost ~100 clk each: the coarse level keeps the timeline honest)
#else
#define TRF(slot, tag) do { } while (0)
#endif
namespace {

constexpr int kStepUnroll = DCD_FUSED_STEP_UNROLL;
constexpr int FCS = 24;             // CTAs per group = edge slices per object
constexpr int FOBJ = 3;             // a group works on THREE objects at a time (same net, same layer weights)
constexpr int FCONV_WARPS = 12;     // converter warps: 4 TMEM lane quarters x 3 units (16 edges) of a 48-edge sub-tile
constexpr int FCONV_THREADS = 32 * FCONV_WARPS;
constexpr int FTHREADS = FCONV_THREADS + 128;   // + 4 service warps: weight loads (all 4), MMA issue (the first)
constexpr int FSUB = 48;            // edges per MMA sub-tile
constexpr int FES_MAX = 112;        // edges per CTA and object (FOBJ * FES_MAX = 336 = 7 sub-tiles)
constexpr uint32_t FT_W = 384;      // tensor-memory columns: D = [0, 336) (three objects side by side), weights hi = [384, 448), lo = [448, 512)
constexpr uint32_t FB_SBO = 128;    // B operand: bytes between 8-edge blocks of one 8-channel block
constexpr uint32_t FB_LBO = 768;    //            bytes between 8-channel blocks (6 edge blocks)
constexpr uint32_t FB_PART = 16 * FB_LBO;   // 12 KB: hi or lo part of one sub-tile

constexpr size_t SMF_X = 0;
constexpr size_t SMF_B = SMF_X + (size_t)FOBJ * FES_MAX * CH * sizeof(float);   // [2 buffers]{hi, lo}
constexpr size_t SMF_PART = SMF_B + 4 * FB_PART;                                // [3][3][128] float2 (mean, M2) / (mean, rstd) + count tables
constexpr size_t SMF_BAR = SMF_PART + (FOBJ * 3 * CH + 64) * sizeof(float2);
constexpr size_t kFusedSmem = SMF_BAR + 128;
static_assert(kFusedSmem <= 232448, "shared memory budget");
static_assert(FOBJ * 6 * FES_MAX * sizeof(float) <= 4 * FB_PART, "edge features are staged in the operand buffers");
static_assert(FOBJ * FES_MAX <= FCONV_THREADS, "one converter thread per staged edge");
// mbarriers (8 bytes each, at SMF_BAR)
enum { BAR_FULL0 = 0, BAR_FULL1 = 1, BAR_DONE0 = 2, BAR_DONE1 = 3, BAR_PDONE = 4, BAR_WREADY = 5, BAR_STAT0 = 6, BAR_COUNT = 9 };
// hardware named barriers (a blocked warp takes no issue slots): 0 = CTA, 1 = converters, 2..4 = the units of the epilogue,
// 5..7 = partial statistics of object 0..2 posted: the converters (12 warps) arrive, the statistics warps (3 warps) wait;
// 8 = the statistics warps among themselves; 9..11 = (mean, rstd) of object 0..2 handed back: the statistics warps arrive,
// the converters wait (DCD_FUSED_STAT_NBAR)
enum { NB_PART0 = 5, NB_STATW = 8, NB_STAT0 = 9 };
constexpr int FSTAT_THREADS = 96;
constexpr int NB_THREADS = FCONV_THREADS + FSTAT_THREADS;

// Statistics exchange between the 24 CTAs of a group through global memory (L2): every published 8-byte word carries
// its own "ready" flag in the sign bit of its second float (an M2 is never negative), so there are no fences, no
// barriers and no ordering requirements: a reader re-reads a word until the flag matches the expected use count.
__device__ __forceinline__ void st_flagged(float2* dst, float a, float b, uint32_t flag) {
    const uint32_t bits = (__float_as_uint(b) & 0x7fffffffu) | (flag << 31);
    // one 64-bit access at GPU scope (the words never leave this device; `volatile` would be system scope)
    const unsigned long long w = ((unsigned long long)bits << 32) | (unsigned long long)__float_as_uint(a);
    asm volatile("st.relaxed.gpu.global.b64 [%0], %1;" ::"l"(dst), "l"(w) : "memory");
}
__device__ __forceinline__ float2 ld_volatile_f2(const float2* p) {
    float2 v;
    unsigned long long w;
    asm volatile("ld.relaxed.gpu.global.b64 %0, [%1];" : "=l"(w) : "l"(p) : "memory");
    v.x = __uint_as_float((uint32_t)w);
    v.y = __uint_as_float((uint32_t)(w >> 32));
    return v;
}
// weight image: read-only, re-read by every CTA for every layer -> keep it in L2 against the streamed outputs
__device__ __forceinline__ void ld_weights8(const uint32_t* p, uint32_t* r) {
    asm volatile("ld.global.nc.L2::evict_last.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "l"(p));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// mbarrier wait that backs off between tests (ptxas drops try_wait's suspend-time hint on sm_100a: the default time-out is
// short and a spinning warp takes issue slots from the warps it is waiting for)
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity, uint32_t ns) {
    uint32_t done;
    for (;;) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (done) break;
        if (ns) __nanosleep(ns);
    }
}
__device__ __forceinline__ void nbar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void nbar_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void conv_sync() { asm volatile("bar.sync 1, %0;" ::"n"(FCONV_THREADS) : "memory"); }

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// the same load split into issue and wait, so that its latency can be covered by independent work
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld16_wait(uint32_t (&r)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                   "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
                 :
                 : "memory");
}

// packed FP32 pair arithmetic (sm_100 FFMA2 / FADD2, crt/sm_100_rt.hpp): one issue slot for two elements.  The operands are
// float2 values that ptxas places in register pairs itself; the broadcast pairs are built once per layer or object.
__device__ __forceinline__ float2 f2_of(uint32_t a, uint32_t b) { return make_float2(__uint_as_float(a), __uint_as_float(b)); }
__device__ __forceinline__ float2 bcast2(float a) { return make_float2(a, a); }

// no-swizzle (interleaved) shared-memory matrix descriptor
__device__ __forceinline__ uint64_t smem_desc_ns(uint32_t addr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((addr & 0x3ffffu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46);
}

// (v0, v1) -> packed FP16 pair hp = rn(v) and lp = rn(hp - v) = MINUS the low part (the MMA that consumes the
// low parts negates B): F2FP + 2 x FHADD (mixed f16/f32 add) + F2FP for two values.
__device__ __forceinline__ void split2_neg(float v0, float v1, uint32_t& hp, uint32_t& lp) {
    asm("{\n\t.reg .f16 h0, h1;\n\t.reg .f32 l0, l1;\n\t"
        "cvt.rn.f16x2.f32 %0, %3, %2;\n\t"
        "mov.b32 {h0, h1}, %0;\n\t"
        "sub.rn.f32.f16 l0, h0, %2;\n\t"
        "sub.rn.f32.f16 l1, h1, %3;\n\t"
        "cvt.rn.f16x2.f32 %1, l1, l0;\n\t}"
        : "=&r"(hp), "=r"(lp)
        : "f"(v0), "f"(v1));
}

// byte offset of a converter thread's 16 edges (edge blocks 2u, 2u+1 of the sub-tile) of input channel ch in an operand part
__device__ __forceinline__ uint32_t unit_offset(int ch, int u) {
    return (uint32_t)(2 * u) * FB_SBO + (uint32_t)(ch >> 3) * FB_LBO + (uint32_t)(ch & 7) * 16u;
}
// 16 edges of one input channel -> FP16 hi / -lo, two 16-byte stores each (b_hi: the unit's place in the hi part)
__device__ __forceinline__ void store_unit(unsigned char* b_hi, const float2 (&v)[8]) {
    uint32_t hp[8], lp[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) split2_neg(v[q].x, v[q].y, hp[q], lp[q]);
    *reinterpret_cast<uint4*>(b_hi) = make_uint4(hp[0], hp[1], hp[2], hp[3]);
    *reinterpret_cast<uint4*>(b_hi + FB_SBO) = make_uint4(hp[4], hp[5], hp[6], hp[7]);
    *reinterpret_cast<uint4*>(b_hi + FB_PART) = make_uint4(lp[0], lp[1], lp[2], lp[3]);
    *reinterpret_cast<uint4*>(b_hi + FB_PART + FB_SBO) = make_uint4(lp[4], lp[5], lp[6], lp[7]);
}

// one sub-tile GEMM D[128 x N] = W[128 x 128] . B[128 x N] as 3 x 8 MMAs: Wh.(-(-Bl)), Wl.Bh, Wh.Bh
__device__ __forceinline__ void issue_sub_gemm(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo, int N) {
    const uint32_t idesc = (1u << 4) | (1u << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(CH >> 4) << 24);
    const uint64_t d_hi = smem_desc_ns(b_hi, FB_LBO, FB_SBO), d_lo = smem_desc_ns(b_lo, FB_LBO, FB_SBO);
    uint32_t acc = 0;
#pragma unroll
    for (int term = 0; term < 3; ++term) {
        const uint32_t a = (term == 1) ? a_lo : a_hi;
        const uint64_t d = (term == 0) ? d_lo : d_hi;
        const uint32_t id = (term == 0) ? (idesc | (1u << 14)) : idesc;      // bit 14: negate B
#pragma unroll
        for (int ks = 0; ks < CH / 16; ++ks) {
            umma_f16_ts(tmem_d, a + ks * 8, d + (uint64_t)((ks * 2 * FB_LBO) >> 4), id, acc);
            acc = 1;
        }
    }
}

}  // namespace

// Layer matrices of the fused forward.  There is no non-linearity between a block's preconv and conv1
// (ops.py:125-131: x = preconv(x); x = conv1(x) -> context norm), so the two 128x128 layers are folded into one:
//     Wf = W1 . Wp,   bf = W1 . bp + b1        (FP64 accumulation, rounded once to FP32; tc_fold_prep_kernel)
// which removes a third of the GEMM layers (24 instead of 36 per net; SURVEY 8d: report F_m with 24).
// Per matrix m = (net, block, j) with j = 0: Wf, j = 1: W2 this kernel writes the power-of-two FP16 scale, the bias
// and the pre-split weight image: per row (= out channel) 128 x u32, columns 0-63 the FP16 pairs (k = 2c, 2c+1) of
// scale*W (hi part), columns 64-127 the lo parts — the tensor-memory image of the A operand — stored as
// [half][chunk of 8 columns][row][8] so that the 32 rows a warp loads lie next to each other.
__global__ void __launch_bounds__(1024) fused_prep_kernel(const float* __restrict__ p4, const float* __restrict__ p6, int depth,
                                                         const float* __restrict__ fold, float2* __restrict__ scales2,
                                                         float* __restrict__ bias2, uint32_t* __restrict__ img) {
    extern __shared__ float wf_s[];                           // [in][out] FP32, 64 KB
    __shared__ float red[32];
    __shared__ float scale_s;
    const int m = blockIdx.x;
    const int j = m & 1, blk = (m >> 1) % depth, net = m / (2 * depth);
    const int cin = net == 0 ? 4 : 6;
    const float* prm = net == 0 ? p4 : p6;
    const int tid = threadIdx.x;
    if (j == 0) {                                            // folded layer, formed by tc_fold_prep_kernel (gmw_mlp_tc.cu)
        const float* F = fold + ((int64_t)net * depth + blk) * FOLD_STRIDE;
        for (int i = tid; i < CH * CH; i += 1024) wf_s[i] = F[i];
        if (tid < CH) bias2[m * CH + tid] = F[CH * CH + tid];
    } else {
        const float* W2 = prm + blob_w(cin, blk, 2);
        for (int i = tid; i < CH * CH; i += 1024) wf_s[i] = W2[i];
        if (tid < CH) bias2[m * CH + tid] = prm[blob_b(cin, blk, 2) + tid];
    }
    __syncthreads();
    // per-matrix power-of-two scale that puts max|W| in [512, 1024): FP16 hi/lo both stay normal
    float mx = 0.f;
    for (int i = tid; i < CH * CH; i += 1024) mx = fmaxf(mx, fabsf(wf_s[i]));
    mx = warp_max(mx);
    if ((tid & 31) == 0) red[tid >> 5] = mx;
    __syncthreads();
    if (tid == 0) {
        mx = 0.f;
        for (int w = 0; w < 32; ++w) mx = fmaxf(mx, red[w]);
        int e = 0;
        if (mx > 0.f) frexpf(mx, &e);
        scales2[m] = make_float2(ldexpf(1.f, 10 - e), ldexpf(1.f, e - 10));
        scale_s = ldexpf(1.f, 10 - e);
    }
    __syncthreads();
    const float scale = scale_s;
    uint32_t* out = img + (size_t)m * CH * CH;
    for (int idx = tid; idx < CH * 64; idx += 1024) {
        const int row = idx & 127, c = idx >> 7;
        const float w0 = wf_s[(2 * c) * CH + row] * scale, w1 = wf_s[(2 * c + 1) * CH + row] * scale;
        const __half h0 = __float2half_rn(w0), h1 = __float2half_rn(w1);
        const __half l0 = __float2half_rn(w0 - __half2float(h0)), l1 = __float2half_rn(w1 - __half2float(h1));
        // [half][chunk of 8 columns][row][8]: a warp (32 rows) fetches one chunk as 1 KB of consecutive bytes
        out[(((c >> 3)) * CH + row) * 8 + (c & 7)] = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
        out[((8 + (c >> 3)) * CH + row) * 8 + (c & 7)] = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
    }
}

namespace {

template <int V> struct IntC { static constexpr int value = V; };   // compile-time step variant (converters' generic lambdas)

// UPO = 16-edge units per object in a CTA = 48-column tiles per layer (FOBJ * ES == 48 * UPO): the slice geometry is a
// compile-time constant, so the converters' object boundaries, unit streams and operand offsets are too.
template <int UPO>
__global__ void __launch_bounds__(FTHREADS, 1)
mlp_fused_kernel(MlpArgs a, const float2* __restrict__ scales, const float* __restrict__ bias2, const uint32_t* __restrict__ wimg,
                 float2* xg, float* __restrict__ reg_w, float4* park) {
    static_assert(UPO >= 3 && 16 * UPO <= FES_MAX, "slice geometry");
    const WsLayout& L = a.L;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);  // warp-uniform for the compiler (uniform datapath)
    const int quarter = warp & 3;                            // TMEM lane quarter this warp may access
    TR_DECL
    const int ch = 32 * quarter + lane;                      // this thread's channel = TMEM lane = weight row
    const uint32_t rank = blockIdx.x % FCS, group = blockIdx.x / FCS;   // 24 consecutive CTAs form a group (co-resident: cooperative launch)
    const int E = L.E, EP = L.EP, depth = L.depth;
    constexpr int upo = UPO;                                 // 16-edge units per object in this CTA
    constexpr int ES = 16 * upo;                             // edges per CTA and object
    constexpr int ntile = upo;                               // 48-column tiles of the CTA
    const int nphase = 2 * depth;                            // per block: folded preconv.conv1, conv2
#if DCD_FUSED_CONV_FINAL
    // (slices of 4 units: a converter warp's next post could overtake another warp's read of the shared partial slots)
    constexpr bool conv_final = upo != 4;
#endif

    extern __shared__ __align__(1024) unsigned char smem[];
    float4* Xs = reinterpret_cast<float4*>(smem + SMF_X);
    unsigned char* Bbuf = smem + SMF_B;
    float2* pbuf = reinterpret_cast<float2*>(smem + SMF_PART);               // [3 objects][3 unit streams][128]: (mean, M2) posted by the
                                                                             // converters, overwritten with (mean, rstd) by the statistics warps
    float2* tab_s = pbuf + FOBJ * 3 * CH;                                    // count tables, see below
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + SMF_BAR);
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + SMF_BAR + 8 * BAR_COUNT);

    if (tid == 0) {
        mbar_init(bar + BAR_FULL0, FCONV_WARPS);
        mbar_init(bar + BAR_FULL1, FCONV_WARPS);
        mbar_init(bar + BAR_DONE0, 1);
        mbar_init(bar + BAR_DONE1, 1);
        mbar_init(bar + BAR_PDONE, 1);
        mbar_init(bar + BAR_WREADY, 4);
        for (int o = 0; o < FOBJ; ++o) mbar_init(bar + BAR_STAT0 + o, 3);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // Columns of the CTA: unit u (16 columns) = object u / upo, its edges [16 (u % upo), +16) of the slice; unit u is converted by
    // the converter warps with warp / 4 == u % 3.  The partial statistics of an object are kept per "unit stream" k = (unit index
    // inside the object) % 3 — one converter warp per lane quarter each — so that the merge order does not depend on which of
    // the three places an object takes.  Statistics merge weights:
    //   tab_s[3 o + k]      = (n_ok, n_ok / n_cta)  valid edges of object o in unit stream k (the same for every o)
    //   tab_s[9 + 3 o + k]  = (1 / n_ok or 0, -)
    //   tab_s[32 + r]       = (n_r, n_r / N_s)      valid edges of the slice of rank r; s = r / 8: the three rank subsets the
    //   tab_s[56 + s]       = (N_s, N_s / E)        statistics warps merge first
    if (tid < 9) {
        const int o = tid / 3, k = tid % 3;
        const int vld = max(0, min(ES, E - (int)rank * ES));
        int nq = 0;
        for (int u = o * upo; u < (o + 1) * upo; ++u)
            if ((u - o * upo) % 3 == k) nq += max(0, min(16, vld - 16 * (u - o * upo)));
        tab_s[tid] = make_float2((float)nq, vld > 0 ? (float)nq / (float)vld : 0.f);
        tab_s[9 + tid] = make_float2(nq > 0 ? 1.0f / (float)nq : 0.f, 0.f);
    } else if (tid >= 32 && tid < 32 + FCS) {
        const int r = tid - 32, sb = r / 8;
        const int nr = max(0, min(ES, E - r * ES));
        const int ns = max(0, min(E, (sb + 1) * 8 * ES) - min(E, sb * 8 * ES));
        tab_s[tid] = make_float2((float)nr, ns > 0 ? (float)nr / (float)ns : 0.f);
    } else if (tid >= 56 && tid < 59) {
        const int sb = tid - 56;
        const int ns = max(0, min(E, (sb + 1) * 8 * ES) - min(E, sb * 8 * ES));
        tab_s[tid] = make_float2((float)ns, (float)ns / (float)E);
    }
    if (warp == 0) tmem_alloc(tmem_ptr, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_ptr, 0);
    const uint32_t t_lane = tmem_base + ((uint32_t)(32 * quarter) << 16);
    // Work list of a group: "rounds" = (net, object triple 3p, 3p + 1, 3p + 2) — the three objects share the layer weights and
    // follow each other through every layer, so the statistics exchange of one object's layer (drain of its last MMAs, L2
    // round trip between the 24 CTAs) is hidden behind the other two objects' tiles.  PAIRED (reg_w != nullptr): triples
    // group, group + G, ... with both nets of a triple back to back (net 0 then net 1), so that the second net's final pass
    // finds the first net's features parked by the very same threads and emits the edge weights itself (see the epilogue).
    // Otherwise (features requested, or too few objects): rounds 2 p + net dealt round-robin, final features to global memory.
    // A last, incomplete triple repeats its last object (one output).
    const int64_t ngroups = gridDim.x / FCS;
    const bool paired = reg_w != nullptr;
    const int64_t ntrip = (L.N + FOBJ - 1) / FOBJ;
    const int64_t nlist = paired ? ntrip : 2 * ntrip;        // entries dealt round-robin: triples (paired) or rounds
    const int64_t nmine = nlist > (int64_t)group ? (nlist - 1 - group) / ngroups + 1 : 0;
    const int64_t nd = paired ? 2 * nmine : nmine;           // rounds of this group
    auto round_trip = [&](int64_t d) { return paired ? (int64_t)group + (d >> 1) * ngroups : ((int64_t)group + d * ngroups) >> 1; };
    auto round_net = [&](int64_t d) { return paired ? (int)(d & 1) : (int)(((int64_t)group + d * ngroups) & 1); };

    if (warp >= FCONV_WARPS) {
        // =====================================================================================================
        // service warps: stream the layers' weight images into tensor memory; the first one issues the MMAs,
        // the other three run the context-norm statistics exchange
        // =====================================================================================================
        uint32_t wr[64];
        // weight image of a matrix: [half (hi, lo)][chunk of 8 columns][row][8 x u32] — a warp's load of one chunk is 1 KB contiguous
        auto w_load = [&](int mat, int half) {
            const uint32_t* src = wimg + (size_t)mat * CH * CH + ((size_t)(half * 8) * CH + ch) * 8;
#pragma unroll
            for (int i = 0; i < 8; ++i) ld_weights8(src + (size_t)i * CH * 8, wr + 8 * i);
        };
        auto w_store = [&](int half) {
            uint32_t t[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) t[i] = wr[i];
            tmem_st32(t_lane + FT_W + 64 * half, t);
#pragma unroll
            for (int i = 0; i < 32; ++i) t[i] = wr[32 + i];
            tmem_st32(t_lane + FT_W + 64 * half + 32, t);
        };
        auto w_publish = [&]() {
            tc_wait_st();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar + BAR_WREADY);
        };
        uint32_t g = 0;                                       // running tile step: operand buffer = g & 1
        uint32_t fpar = 0, wpar = 0, ppar = 0;                // parities: full[2] (bits), wready, pdone
        // ---- context-norm statistics (service warps 1..3; the MMA warp takes no part).  Every converter warp posts one (mean, M2)
        //      per object and layer for its unit stream (NB_PART0 + object).  A statistics thread owns a channel (the first warp
        //      two): it merges the 3 unit streams, publishes the slice's (mean, M2) in global memory for the 23 other CTAs of the
        //      group (flagged words, see st_flagged), collects theirs, merges in rank order and hands (mean, rstd) of the layer
        //      back through the converters' own partial slots (BAR_STAT0 + object).  All counts are constants of the launch: no
        //      divisions.  The converters wait for an exchange only if it takes longer than the other two objects' tiles.
        const int nrep = warp == FCONV_WARPS + 1 ? 2 : 1;
        const float inv_em1 = 1.0f / (float)(E - 1);
        uint32_t sxc = 0;                                     // exchanges done per object, mod 4 (2 bits each): slot = count & 1, flag = (count >> 1) & 1
        auto ev_row = [&](int o) {
            const uint32_t xc = (sxc >> (2 * o)) & 3u;
            return xg + ((size_t)((group * FOBJ + o) * 2 + (xc & 1u)) * FCS) * CH;        // [rank][128] of this group, object and slot
        };
        auto ev_flag = [&](int o) { return (sxc >> (2 * o + 1)) & 1u; };
        // the 12 partial posts of (object, layer) are in: merge the unit streams, publish the slice
        auto ev_publish = [&](int o) {
            TR(2, 700 + o);
            nbar_sync(NB_PART0 + o, NB_THREADS);
            TR(2, 710 + o);
            float2* xrow0 = ev_row(o);
            const uint32_t flag = ev_flag(o);
            float2 tb[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) tb[k] = tab_s[o * 3 + k];
            const int c0 = 32 * (warp - FCONV_WARPS - 1) + lane, c1 = 96 + lane;       // (the second channel: first statistics warp only)
            float2 q[2][3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                q[0][k] = pbuf[(o * 3 + k) * CH + c0];
                q[1][k] = pbuf[(o * 3 + k) * CH + c1];
            }
#pragma unroll
            for (int rep = 0; rep < 2; ++rep) {
                float m = 0.f, M2 = 0.f;
#pragma unroll
                for (int k = 0; k < 3; ++k) m = fmaf(tb[k].y, q[rep][k].x, m);
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const float dd = q[rep][k].x - m;
                    if (tb[k].x > 0.f) M2 += fmaf(tb[k].x * dd, dd, q[rep][k].y);
                }
                if (rep < nrep) st_flagged(xrow0 + rank * CH + (rep ? c1 : c0), m, M2, flag);
            }
            // every post of this (object, layer) is consumed before any statistics warp reuses the partial slots (ev_finish)
            nbar_sync(NB_STATW, FSTAT_THREADS);
            TR(2, 720 + o);
        };
        // (mean, rstd) or the rank-subset results of object o are in the partial slots: release the converters waiting for them
        auto stat_handback = [&](int o) {
#if DCD_FUSED_STAT_NBAR
            nbar_arrive(NB_STAT0 + o, NB_THREADS);     // (a hardware barrier: the waiting converter warps take no issue slots)
#else
            __syncwarp();
            if (lane == 0) mbar_arrive(bar + BAR_STAT0 + o);
#endif
        };
        // Collect the 24 slices (the own one included) and hand (mean, rstd) to the converters.  Each statistics warp takes 8
        // ranks for all 128 channels (a lane: 4 channels x 8 flagged words in flight at once, re-read until every word carries
        // this exchange's flag) and merges them; the three subset results meet in the object's partial slots, then every channel
        // is finished by one thread (rank subsets in order: the same operations in every CTA of the group).
        auto ev_finish = [&](int o, bool fresh) {
            const int sb = warp - FCONV_WARPS - 1;            // rank subset of this warp: ranks 8 sb .. 8 sb + 7
            const float2* xrow0 = ev_row(o) + (size_t)(8 * sb) * CH + lane;
            const uint32_t flag = ev_flag(o);
            // (right after this CTA's own publication the other slices cannot be visible yet: a first look would be wasted)
            if (fresh) __nanosleep(DCD_FUSED_POLL_GRACE);
            float2 v[4][8];
            for (;;) {
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int r = 0; r < 8; ++r) v[q][r] = ld_volatile_f2(xrow0 + r * CH + 32 * q);
                uint32_t bad = 0;
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int r = 0; r < 8; ++r) bad |= (__float_as_uint(v[q][r].y) >> 31) ^ flag;
                if (!bad) break;
                __nanosleep(64);                                                  // (slices still missing: poll at a low rate)
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                float mu = 0.f, M2 = 0.f;
#pragma unroll
                for (int r = 0; r < 8; ++r) mu = fmaf(tab_s[32 + 8 * sb + r].y, v[q][r].x, mu);
#pragma unroll
                for (int r = 0; r < 8; ++r) {
                    const float dd = v[q][r].x - mu;
                    M2 += fmaf(tab_s[32 + 8 * sb + r].x * dd, dd, __uint_as_float(__float_as_uint(v[q][r].y) & 0x7fffffffu));
                }
                pbuf[(o * 3 + sb) * CH + 32 * q + lane] = make_float2(mu, M2);
            }
#if DCD_FUSED_CONV_FINAL
            if (conv_final) {                                 // the converter threads finish their channel themselves (see `collect`)
                stat_handback(o);
                TR(2, 730 + o);
                sxc = (sxc & ~(3u << (2 * o))) | (((((sxc >> (2 * o)) & 3u) + 1u) & 3u) << (2 * o));
                return;
            }
#endif
            nbar_sync(NB_STATW, FSTAT_THREADS);
            for (int rep = 0; rep < nrep; ++rep) {
                const int c = rep ? 96 + lane : 32 * sb + lane;
                float2 q[3];
#pragma unroll
                for (int k = 0; k < 3; ++k) q[k] = pbuf[(o * 3 + k) * CH + c];
                float m = 0.f, M2 = 0.f;
#pragma unroll
                for (int k = 0; k < 3; ++k) m = fmaf(tab_s[56 + k].y, q[k].x, m);
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const float dd = q[k].x - m;
                    M2 += fmaf(tab_s[56 + k].x * dd, dd, q[k].y);
                }
                const float var = M2 * inv_em1;
                const float2 st = make_float2(m, rsqrtf(var + 1e-3f));
#pragma unroll
                for (int k = 0; k < 3; ++k) pbuf[(o * 3 + k) * CH + c] = st;
            }
            stat_handback(o);
            TR(2, 730 + o);
            sxc = (sxc & ~(3u << (2 * o))) | (((((sxc >> (2 * o)) & 3u) + 1u) & 3u) << (2 * o));
        };
        if (nd > 0) {
            const int mat = round_net(0) * nphase;
            w_load(mat, 0);
            w_store(0);
            w_load(mat, 1);
            w_store(1);
            w_publish();
        }
        for (int64_t d = 0; d < nd; ++d) {
            const int mat_base = round_net(d) * nphase;
            for (int ph = 0; ph <= nphase; ++ph) {            // (ph == nphase: only the last layer's last statistics event)
                if (warp == FCONV_WARPS) {
                    if (ph == nphase) break;
                    TR(1, 10);
                    mbar_wait(bar + BAR_WREADY, wpar);
                    tc_fence_after();
                    TR(1, 11);
                    for (int t = 0; t < ntile; ++t, ++g) {
                        const uint32_t b = g & 1u;
                        TRF(1, 100 + t);
                        mbar_wait(bar + BAR_FULL0 + b, (fpar >> b) & 1u);
                        fpar ^= 1u << b;
                        tc_fence_after();
                        TR(1, 200 + t);
                        if (elect_one()) {
                            const uint32_t b_hi = smem_u32(Bbuf) + b * 2 * FB_PART;
                            issue_sub_gemm(tmem_base + FSUB * t, tmem_base + FT_W, tmem_base + FT_W + 64, b_hi, b_hi + FB_PART, FSUB);
                            umma_commit(bar + BAR_DONE0 + b);
                            if (t == ntile - 1) umma_commit(bar + BAR_PDONE);
                        }
                        __syncwarp();
                    }
                } else {
                    // layer outputs in the order the converters complete them: object 2 of the previous layer during this layer's
                    // first tiles, then objects 0 and 1 of this layer.  Object 1's exchange overlaps the end of the layer, where
                    // the next weights are due: they go first, the slices are collected afterwards.
                    if (ph > 0) {
                        ev_publish(2);
                        ev_finish(2, true);
                    }
                    if (ph == nphase) break;
                    ev_publish(0);
                    ev_finish(0, true);
                    ev_publish(1);
                }
                wpar ^= 1u;
                // next layer's weights: first half fetched while this layer's last MMAs drain
                const bool last_ph = ph + 1 == nphase;
                const bool more = !last_ph || d + 1 < nd;
                if (more) {
                    const int mat = last_ph ? round_net(d + 1) * nphase : mat_base + ph + 1;
#ifdef DCD_EXP_NO_WRELOAD
                    (void)mat;
                    mbar_wait(bar + BAR_PDONE, ppar);
                    tc_fence_after();
                    w_publish();
#else
                    w_load(mat, 0);
                    TR(warp == FCONV_WARPS ? 1 : 2, 20);
                    mbar_wait(bar + BAR_PDONE, ppar);
                    tc_fence_after();
                    TR(warp == FCONV_WARPS ? 1 : 2, 21);
                    w_store(0);
                    w_load(mat, 1);
                    w_store(1);
                    w_publish();
#endif
                    TR(warp == FCONV_WARPS ? 1 : 2, 22);
                } else {
                    mbar_wait(bar + BAR_PDONE, ppar);
                }
                ppar ^= 1u;
                if (warp != FCONV_WARPS) ev_finish(1, false);
            }
        }
    } else {
        // =====================================================================================================
        // converter warps: thread = channel; units of 16 edges; produce the B operands, consume the accumulators
        // =====================================================================================================
        const int wg = warp >> 2;                             // unit stream: this warp converts the units u with u % 3 == wg
        const int e_base = (int)rank * ES;
        const int valid = max(0, min(ES, E - e_base));        // valid edges of this CTA's slice (the same for the three objects)
        uint32_t g = 0;                                       // running tile step (same sequence as the MMA warp)
        uint32_t par = 0, pend = 0;                           // per operand buffer: next wait parity, MMA in flight
        auto wait_buf = [&](uint32_t b) {
            if ((pend >> b) & 1u) {
                mbar_wait_backoff(bar + BAR_DONE0 + b, (par >> b) & 1u, DCD_FUSED_DONE_SLEEP);
                par ^= 1u << b;
                pend &= ~(1u << b);
                tc_fence_after();
            }
        };
        auto obj_of = [&](int u) { return (u >= upo ? 1 : 0) + (u >= 2 * upo ? 1 : 0); };
#if !DCD_FUSED_STAT_NBAR
        uint32_t spar = 0;                                    // wait parities of the three statistics barriers (this warp's view)
#endif
#if DCD_FUSED_CONV_FINAL
        const float inv_em1_c = 1.0f / (float)(E - 1);
#endif
        // tiles where this warp's unit is the first / the last one it has of an object (upo >= 3: every warp has units of all three)
        uint32_t firstmask = 0, lastmask = 0;
        for (int t = 0; t < ntile; ++t) {
            const int u = 3 * t + wg;
            if (t == 0 || obj_of(u) != obj_of(u - 3)) firstmask |= 1u << t;
            if (t == ntile - 1 || obj_of(u + 3) != obj_of(u)) lastmask |= 1u << t;
        }
        // unit stream of this warp's units of object o: (wg - o * upo) mod 3
        auto stream_of = [&](int o) { return (wg + 3 * o * upo - o * upo) % 3; };

        for (int64_t d = 0; d < nd; ++d) {
            const int64_t trip = round_trip(d);
            const int net = round_net(d);
            const int64_t obj0 = FOBJ * trip;                 // objects obj0 + o, clamped to the last one
            const int cin = net == 0 ? 4 : 6;
            const float* __restrict__ prm = a.params[net];
            const int mat_base = net * nphase;

            // ---- edge features of the three slices, staged in the (idle) operand buffers: f_s[3][6][ES]
            TR(0, 900);
            wait_buf(0);
            wait_buf(1);
            conv_sync();
            float* f_s = reinterpret_cast<float*>(Bbuf);
            if (tid < FOBJ * ES) {
                const int o = obj_of(tid >> 4);
                const int el = tid - o * ES;
                const int e = e_base + el;
                const int64_t obj = min(obj0 + o, L.N - 1);
                int i, j;
                decode_edge(e < E ? e : E - 1, L.n, i, j);
                float f[6];
                if (net == 0) {
                    const float2 pi = __ldg(reinterpret_cast<const float2*>(a.kpts2d + (obj * L.n + i) * 2));
                    const float2 pj = __ldg(reinterpret_cast<const float2*>(a.kpts2d + (obj * L.n + j) * 2));
                    f[0] = pi.x; f[1] = pi.y; f[2] = pj.x; f[3] = pj.y; f[4] = 0.f; f[5] = 0.f;
                } else {
                    const float* pi = a.kpts3d + (obj * L.n + i) * 3;
                    const float* pj = a.kpts3d + (obj * L.n + j) * 3;
                    f[0] = __ldg(pi); f[1] = __ldg(pi + 1); f[2] = __ldg(pi + 2);
                    f[3] = __ldg(pj); f[4] = __ldg(pj + 1); f[5] = __ldg(pj + 2);
                }
#pragma unroll
                for (int r = 0; r < 6; ++r) f_s[(o * 6 + r) * ES + el] = f[r];
            }
            conv_sync();
            // ---- conv_in: X0 = W_in . f + b_in   (the features are warp-wide broadcasts)
            {
                float wq[6];
#pragma unroll
                for (int q = 0; q < 6; ++q) wq[q] = (q < cin) ? __ldg(prm + blob_in_w() + q * CH + ch) : 0.f;
                const float b = __ldg(prm + blob_in_b(cin) + ch);
                for (int u = wg; u < FOBJ * upo; u += 3) {
                    const int o = obj_of(u);
                    const int lc = 16 * (u - o * upo);
                    const float* fo = f_s + o * 6 * ES + lc;
#pragma unroll
                    for (int q4 = 0; q4 < 4; ++q4) {
                        float x[4];
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const int e = 4 * q4 + i;
                            float acc = b;
#pragma unroll
                            for (int r = 0; r < 6; ++r) acc = fmaf(wq[r], fo[r * ES + e], acc);
                            x[i] = (lc + e < valid) ? acc : 0.f;
                        }
                        Xs[(4 * u + q4) * CH + ch] = make_float4(x[0], x[1], x[2], x[3]);
                    }
                }
            }
            conv_sync();                                      // the features are consumed: operand buffers free
            TR(0, 901);

            // ---- the layers: a stream of steps (layer, tile).  This warp converts unit 3 t + wg of tile t; the units of an object are
            //      consecutive, so the object and the offset inside its slice are running values (firstmask / lastmask: the tiles
            //      where this warp's unit is its first / last of an object).
            float un_out = 0.f, b_out = 0.f, un_prev = 0.f, b_prev = 0.f;   // scale / bias of the matrices of this and the previous layer
            float2 un2_out = make_float2(0.f, 0.f), un2_prev = un2_out;     // (the scales as broadcast pairs)
            float un_next = __ldg(scales + mat_base).y, b_next = __ldg(bias2 + mat_base * CH + ch);       // (fetched one layer ahead)
            // the tile whose statistics are due next (two steps behind the conversion): tile, object, object's first column
            int npend = 0, t_e = 0, o_e = 0, ob_e = 0;
            float K = 0.f, s1 = 0.f, s2 = 0.f;                // shifted sums of the layer output being accumulated (one object at a time)
            float2 bK2 = make_float2(0.f, 0.f);               // bias - K of that object, both halves
            bool have_K = false;
            uint32_t cv[16], sv[16];

            // statistics of one unit from its raw accumulators (un2, bb: scale and bias of the producing matrix), as sums shifted
            // by K = the object's first value seen by this thread
            auto stats_math = [&](const uint32_t (&raw)[16], int nv, float2 un2, float bb) {
                if (!have_K) {
                    K = fmaf(__uint_as_float(raw[0]), un2.x, bb);
                    bK2 = bcast2(bb - K);
                    have_K = true;
                }
                if (nv >= 16) {
                    float2 t1a = make_float2(0.f, 0.f), t1b = t1a, t2a = t1a, t2b = t1a;
#pragma unroll
                    for (int i = 0; i < 16; i += 4) {
                        const float2 d01 = __ffma2_rn(f2_of(raw[i], raw[i + 1]), un2, bK2);
                        const float2 d23 = __ffma2_rn(f2_of(raw[i + 2], raw[i + 3]), un2, bK2);
                        t1a = __fadd2_rn(t1a, d01);
                        t1b = __fadd2_rn(t1b, d23);
                        t2a = __ffma2_rn(d01, d01, t2a);
                        t2b = __ffma2_rn(d23, d23, t2b);
                    }
                    s1 += (t1a.x + t1a.y) + (t1b.x + t1b.y);
                    s2 += (t2a.x + t2a.y) + (t2b.x + t2b.y);
                } else {
#pragma unroll
                    for (int i = 0; i < 16; ++i)
                        if (i < nv) {
                            const float dd = fmaf(__uint_as_float(raw[i]), un2.x, bK2.x);
                            s1 += dd;
                            s2 = fmaf(dd, dd, s2);
                        }
                }
            };
            // this unit stream's part of object o's layer output is complete: post its (mean, M2) for the statistics warps
            auto post = [&](int o) {
                const int k = stream_of(o);
                const float ic = tab_s[9 + o * 3 + k].x;
                const float m = K + s1 * ic;
                const float M2 = fmaxf(fmaf(-s1 * ic, s1, s2), 0.f);
                pbuf[(o * 3 + k) * CH + ch] = make_float2(m, M2);
                nbar_arrive(NB_PART0 + o, NB_THREADS);
                TR(0, 603);
                K = 0.f; s1 = 0.f; s2 = 0.f; bK2 = make_float2(0.f, 0.f);
                have_K = false;
            };
            // (mean, rstd) of object o's latest layer, handed back by the statistics warps in this warp's partial slot
            auto collect = [&](int o) {
                TR(0, 606);
#if DCD_FUSED_STAT_NBAR
                nbar_sync(NB_STAT0 + o, NB_THREADS);
#else
                mbar_wait_backoff(bar + BAR_STAT0 + o, (spar >> o) & 1u, DCD_FUSED_STAT_SLEEP);
                spar ^= 1u << o;
#endif
                TR(0, 608);
#if DCD_FUSED_CONV_FINAL
                if (conv_final) {
                    // the three rank-subset results of this channel -> (mean, rstd): the very operations of the statistics
                    // warps' last stage, done by the 384 converter threads instead of 96 statistics threads one after the other
                    float2 q[3];
#pragma unroll
                    for (int k = 0; k < 3; ++k) q[k] = pbuf[(o * 3 + k) * CH + ch];
                    float m = 0.f, M2 = 0.f;
#pragma unroll
                    for (int k = 0; k < 3; ++k) m = fmaf(tab_s[56 + k].y, q[k].x, m);
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        const float dd = q[k].x - m;
                        M2 += fmaf(tab_s[56 + k].x * dd, dd, q[k].y);
                    }
                    return make_float2(m, rsqrtf(M2 * inv_em1_c + 1e-3f));
                }
#endif
                return pbuf[(o * 3 + stream_of(o)) * CH + ch];
            };
            // statistics of the due tile (its MMA is complete; `loaded`: its accumulators are already in sv; `cur`: it belongs to
            // the layer being converted, else to the previous one).  FULL: every edge of the slice is valid.
            auto process_due = [&](auto full_c, bool loaded, bool cur) {
                constexpr bool FULL = decltype(full_c)::value != 0;
                const int cb = FSUB * t_e + 16 * wg;          // first column of the unit
                const int nv = FULL ? 16 : valid - (cb - ob_e);   // valid edges from the unit's first on
                if (nv > 0) {
                    if (!loaded) {
                        tmem_ld16_issue(t_lane + cb, sv);
                        tmem_ld16_wait(sv);
                    }
                    stats_math(sv, nv, cur ? un2_out : un2_prev, cur ? b_out : b_prev);
                }
                if ((lastmask >> t_e) & 1u) post(o_e);
                if (++t_e == ntile) {
                    t_e = 0; o_e = 0; ob_e = 0;
                } else if ((firstmask >> t_e) & 1u) {
                    ++o_e; ob_e += ES;
                }
            };

            // input transform of the current object as one FMA on the raw accumulator, both halves: the context norm of the
            // producing layer folded in ((d*un + b - mean) * rstd)
            float2 a_in2 = make_float2(0.f, 0.f), c_in2 = a_in2;
            auto take_stats = [&](int o) {
                const float2 st = collect(o);
                a_in2 = bcast2(un_prev * st.y);
                c_in2 = bcast2((b_prev - st.x) * st.y);
            };
            const bool full = valid == ES;                    // no edge of the slice masked (all CTAs of a group but the last ones)
            const uint32_t uoff = unit_offset(ch, wg);        // this thread's place in an operand part

            // One layer, specialised by kind — 0: residual update, then the folded preconv.conv1; 1: the same for the net's first
            // layer (no accumulators to read, X is the input); 2: conv2 — and by FULL (no tail masks).  Software pipeline over the
            // steps: the accumulators of the NEXT unit to convert (cv, issued at the end of the previous step) and of the unit whose
            // statistics are due (sv, two steps behind: its MMA is known complete when its operand buffer comes free) are in flight
            // from tensor memory while the current unit is being processed.
            auto layer = [&](auto kind_c, auto full_c, int ph) {
                constexpr int KIND = decltype(kind_c)::value;
                constexpr bool FULL = decltype(full_c)::value != 0;
                constexpr bool reads_d = KIND != 1;
                constexpr int KTAG = KIND == 2 ? 2 : 0;       // (trace tags: the kind of the layer's matrix)
                (void)KTAG;
                int o = 0, ob = 0;
                if (reads_d) take_stats(0);
#pragma unroll (UPO == 4 ? 1 : kStepUnroll)        // (UPO = 4 spills when unrolled)
                for (int t = 0; t < ntile; ++t, ++g) {
                    const int cb = FSUB * t + 16 * wg;        // this warp's unit: columns [cb, cb + 16) of the CTA
                    if (t > 0 && ((firstmask >> t) & 1u)) {
                        ++o; ob += ES;
                        if (reads_d) take_stats(o);
                    }
                    const int lc = cb - ob;                   // first edge of the unit inside the object's slice
                    (void)lc;
                    const uint32_t b = g & 1u;
                    TR(0, 1000 * KTAG + 100 + t);
                    if (reads_d) {                            // (both buffers are in use from the round's third step on)
                        mbar_wait_backoff(bar + BAR_DONE0 + b, (par >> b) & 1u, DCD_FUSED_DONE_SLEEP);
                        par ^= 1u << b;
                        tc_fence_after();
                    } else {
                        wait_buf(b);
                    }
                    TRF(0, 1000 * KTAG + 200 + t);
                    // the tile of two steps ago (same operand buffer: its MMA is complete) is due for its statistics (the first two
                    // steps of a round have none)
                    const bool due = KIND != 1 || t >= 2;
                    const int cb_e = FSUB * t_e + 16 * wg;
                    const bool st_load = due && (FULL || valid > cb_e - ob_e);
                    float2 v[8];
                    float4* Xp = Xs + (cb >> 2) * CH + ch;
                    float4 x4[4];
                    if (KIND != 2) {
#pragma unroll
                        for (int q4 = 0; q4 < 4; ++q4) x4[q4] = Xp[q4 * CH];
                    }
                    if (reads_d) tmem_ld16_wait(cv);
                    TRF(0, 1000 * KTAG + 300 + t);
                    if (st_load) tmem_ld16_issue(t_lane + cb_e, sv);
                    if (KIND == 0) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            v[i] = __ffma2_rn(f2_of(cv[2 * i], cv[2 * i + 1]), a_in2, c_in2);
                            v[i].x = fmaxf(v[i].x, 0.f);
                            v[i].y = fmaxf(v[i].y, 0.f);
                        }
#pragma unroll
                        for (int q4 = 0; q4 < 4; ++q4) {
                            v[2 * q4] = __fadd2_rn(v[2 * q4], make_float2(x4[q4].x, x4[q4].y));
                            v[2 * q4 + 1] = __fadd2_rn(v[2 * q4 + 1], make_float2(x4[q4].z, x4[q4].w));
                        }
                        if (!FULL && lc + 16 > valid) {
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                if (lc + 2 * i >= valid) v[i].x = 0.f;
                                if (lc + 2 * i + 1 >= valid) v[i].y = 0.f;
                            }
                        }
#pragma unroll
                        for (int q4 = 0; q4 < 4; ++q4) Xp[q4 * CH] = make_float4(v[2 * q4].x, v[2 * q4].y, v[2 * q4 + 1].x, v[2 * q4 + 1].y);
                    } else if (KIND == 1) {
#pragma unroll
                        for (int q4 = 0; q4 < 4; ++q4) {
                            v[2 * q4] = make_float2(x4[q4].x, x4[q4].y);
                            v[2 * q4 + 1] = make_float2(x4[q4].z, x4[q4].w);
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < 8; ++i) v[i] = __ffma2_rn(f2_of(cv[2 * i], cv[2 * i + 1]), a_in2, c_in2);
                    }
                    store_unit(Bbuf + (size_t)b * 2 * FB_PART + uoff, v);
                    TRF(0, 1000 * KTAG + 400 + t);
                    fence_async_smem();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar + BAR_FULL0 + b);
                    pend |= 1u << b;
                    TRF(0, 1000 * KTAG + 500 + t);
                    if (st_load) tmem_ld16_wait(sv);              // (before the next load is issued: the wait covers all loads in flight)
                    // the next unit to convert: the next tile's, else the next layer's first (whose producing MMA is long complete)
                    if (t + 1 < ntile) {
                        if (reads_d) tmem_ld16_issue(t_lane + cb + FSUB, cv);
                    } else if (ph + 1 < nphase) {
                        tmem_ld16_issue(t_lane + 16 * wg, cv);
                    }
                    if (due) process_due(full_c, true, t >= 2); else ++npend;
                }
            };

            for (int ph = 0; ph < nphase; ++ph) {
                un_prev = un_out;
                b_prev = b_out;
                un_out = un_next;
                b_out = b_next;
                un2_prev = un2_out;
                un2_out = bcast2(un_out);
                if (ph + 1 < nphase) {
                    un_next = __ldg(scales + mat_base + ph + 1).y;
                    b_next = __ldg(bias2 + (mat_base + ph + 1) * CH + ch);
                }
                if (full) {
                    if (ph & 1) layer(IntC<2>(), IntC<1>(), ph);
                    else if (ph > 0) layer(IntC<0>(), IntC<1>(), ph);
                    else layer(IntC<1>(), IntC<1>(), ph);
                } else {
                    if (ph & 1) layer(IntC<2>(), IntC<0>(), ph);
                    else if (ph > 0) layer(IntC<0>(), IntC<0>(), ph);
                    else layer(IntC<1>(), IntC<0>(), ph);
                }
            }
            TR(0, 600);

            // ---- final features x = relu(cn(Y2)) + X of the three objects.  First the statistics still due (their MMAs are then
            //      complete and the operand buffers free for the epilogue's scratch).
            wait_buf(0);
            wait_buf(1);
            un_prev = un_out;
            b_prev = b_out;
            un2_prev = un2_out;
            while (npend > 0) {
                process_due(IntC<0>(), false, false);
                --npend;
            }
            TR(0, 601);
            int o_cur = -1;
            float a_fin = 0.f, c_fin = 0.f;
            int itn = 0;
            for (int u = wg; u < FOBJ * upo; u += 3, ++itn) {
                const int o = obj_of(u);
                const int lc = 16 * (u - o * upo);
                if (o != o_cur) {
                    const float2 st = collect(o);
                    a_fin = un_out * st.y;
                    c_fin = (b_out - st.x) * st.y;
                    o_cur = o;
                }
                const bool emit = obj0 + o < L.N;
                const int64_t obj = min(obj0 + o, L.N - 1);
                float v[16];
                {
                    const float4* Xp = Xs + (4 * u) * CH + ch;
                    float4 x4[4];
#pragma unroll
                    for (int q4 = 0; q4 < 4; ++q4) x4[q4] = Xp[q4 * CH];
                    tmem_ld16(t_lane + 16 * u, v);
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] = fmaxf(fmaf(v[i], a_fin, c_fin), 0.f);
#pragma unroll
                    for (int q4 = 0; q4 < 4; ++q4) {
                        v[4 * q4] += x4[q4].x; v[4 * q4 + 1] += x4[q4].y; v[4 * q4 + 2] += x4[q4].z; v[4 * q4 + 3] += x4[q4].w;
                    }
                    if (lc + 16 > valid) {
#pragma unroll
                        for (int i = 0; i < 16; ++i)
                            if (lc + i >= valid) v[i] = 0.f;
                    }
                }
                if (!paired) {
                    // -> global, channel-major [obj][128][EP] (consumed by gmw_edge_weight_kernel / the correspondence branch)
                    float* G = act_ptr(a.ws, L, net, 0, SLOT_X) + obj * (int64_t)CH * EP + (int64_t)ch * EP;
#pragma unroll
                    for (int q4 = 0; q4 < 4; ++q4)
                        if (emit && e_base + lc + 4 * q4 < EP)
                            __stcs(reinterpret_cast<float4*>(G + e_base + lc + 4 * q4), make_float4(v[4 * q4], v[4 * q4 + 1], v[4 * q4 + 2], v[4 * q4 + 3]));   // streamed: keep the weight image in L2
                } else if (net == 0) {
                    // park the 4-d net's features in this CTA's slice of an L2-resident scratch ([3 ES / 4][128] float4 like Xs):
                    // the thread that writes a word is the one that reads it back after the 6-d net, so no fence or barrier is needed
                    float4* Pk = park + ((size_t)blockIdx.x * (4 * FOBJ * upo) + 4 * u) * CH + ch;
#pragma unroll
                    for (int q4 = 0; q4 < 4; ++q4) Pk[q4 * CH] = make_float4(v[4 * q4], v[4 * q4 + 1], v[4 * q4 + 2], v[4 * q4 + 3]);
                } else {
                    // edge weights straight from the two nets' final features (GMW/model/model.py:176-181, diagonal of pairwiseL2Dist):
                    // per edge the three channel sums |a|^2, |c|^2, a.c — 32 channels by a halving shuffle tree, the 4 lane quarters
                    // through shared memory (the operand buffers are idle here) — then
                    //   w = 1 / sqrt(max((|c^|^2 - 2 a^.c^) + |a^|^2, 1e-30)),  a^ = a / max(|a|, 1e-12)
                    const float4* Pk = park + ((size_t)blockIdx.x * (4 * FOBJ * upo) + 4 * u) * CH + ch;
                    float* red = reinterpret_cast<float*>(Bbuf) + wg * (2 * 4 * 48);      // [2 buffers][4 quarters][16 edges][3]
                    float* W = reg_w + obj * (int64_t)E + e_base + lc;
                    float aa[16], cc[16], ac[16];
#pragma unroll
                    for (int q4 = 0; q4 < 4; ++q4) {
                        const float4 p = Pk[q4 * CH];
                        const float av[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const float c = v[4 * q4 + i];
                            aa[4 * q4 + i] = __fmul_rn(av[i], av[i]);          // (explicit roundings: gmw_edge_weight_kernel<true>
                            cc[4 * q4 + i] = __fmul_rn(c, c);                  //  replays this exact sequence)
                            ac[4 * q4 + i] = __fmul_rn(av[i], c);
                        }
                    }
                    // halving tree over the 32 lanes: afterwards lane l holds the sums of edge l >> 1
#pragma unroll
                    for (int h = 8; h >= 1; h >>= 1) {
                        const bool up = (lane & (2 * h)) != 0;
#pragma unroll
                        for (int k = 0; k < h; ++k) {
                            const float sa = up ? aa[k] : aa[k + h], sc = up ? cc[k] : cc[k + h], sx = up ? ac[k] : ac[k + h];
                            const float ka = up ? aa[k + h] : aa[k], kc = up ? cc[k + h] : cc[k], kx = up ? ac[k + h] : ac[k];
                            aa[k] = __fadd_rn(ka, __shfl_xor_sync(0xffffffffu, sa, 2 * h));
                            cc[k] = __fadd_rn(kc, __shfl_xor_sync(0xffffffffu, sc, 2 * h));
                            ac[k] = __fadd_rn(kx, __shfl_xor_sync(0xffffffffu, sx, 2 * h));
                        }
                    }
                    aa[0] = __fadd_rn(aa[0], __shfl_xor_sync(0xffffffffu, aa[0], 1));
                    cc[0] = __fadd_rn(cc[0], __shfl_xor_sync(0xffffffffu, cc[0], 1));
                    ac[0] = __fadd_rn(ac[0], __shfl_xor_sync(0xffffffffu, ac[0], 1));
                    float* rb = red + (itn & 1) * (4 * 48);
                    if ((lane & 1) == 0) {
                        float* op = rb + quarter * 48 + (lane >> 1) * 3;
                        op[0] = aa[0]; op[1] = cc[0]; op[2] = ac[0];
                    }
                    asm volatile("bar.sync %0, 128;" ::"r"(2 + wg) : "memory");       // the 4 warps (lane quarters) of this unit
                    if (quarter == 0 && lane < 16) {
                        if (lc + lane < valid && emit) {
                            const float* op = rb + lane * 3;
                            const float saa = __fadd_rn(__fadd_rn(op[0], op[48]), __fadd_rn(op[96], op[144]));
                            const float scc = __fadd_rn(__fadd_rn(op[1], op[49]), __fadd_rn(op[97], op[145]));
                            const float sac = __fadd_rn(__fadd_rn(op[2], op[50]), __fadd_rn(op[98], op[146]));
                            const float n4 = fmaxf(sqrtf(saa), 1e-12f), n6 = fmaxf(sqrtf(scc), 1e-12f);
                            const float a2 = __fdiv_rn(saa, __fmul_rn(n4, n4)), c2 = __fdiv_rn(scc, __fmul_rn(n6, n6));
                            const float acn = __fdiv_rn(sac, __fmul_rn(n4, n6));
                            const float s2w = __fadd_rn(__fadd_rn(c2, -2.f * acn), a2);
                            W[lane] = __fdiv_rn(1.f, sqrtf(fmaxf(s2w, 1e-30f)));
                        }
                    }
                }
            }
            TR(0, 610);
            tc_fence_before();                                // the next round's MMAs overwrite these columns
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 512);
}

}  // namespace

#ifdef DCD_FUSED_TRACE
}  // namespace dcd
extern "C" __attribute__((visibility("default"))) int dcd_debug_fused_trace(long long* dst, int* n) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(dst, dcd::g_trace, sizeof(long long) * 12288);
    cudaMemcpyFromSymbol(n, dcd::g_trace_n, sizeof(int) * 3);
    return 0;
}
namespace dcd {
#endif

bool gmw_fused_supported(int n) {
    const int E = n * (n - 1) / 2;
    const int upo = (E + 16 * FCS - 1) / (16 * FCS);          // 16-edge units per object and CTA
    return upo >= 3 && 16 * upo <= FES_MAX;                  // (below 3 a converter warp would not see every object: layer-wise kernels)
}

constexpr int FMAX_GROUPS = 10;                               // exchange buffer sized for up to 256 SMs
constexpr size_t kExchangeBytes = (size_t)FMAX_GROUPS * FOBJ * 2 * FCS * CH * sizeof(float2);    // [group][object][slot][rank][128]

// Tail of the workspace used by the fused forward, per matrix m = (net, block, {folded preconv.conv1, conv2}):
//   scales2 [4*depth] float2 (256-byte padded) | bias2 [4*depth][128] | weight image [4*depth][128][128] u32 | exchange buffer
static size_t fused_scales_bytes(int depth) { return (((size_t)4 * depth * sizeof(float2)) + 255) / 256 * 256; }
static size_t fused_bias_bytes(int depth) { return (size_t)4 * depth * CH * sizeof(float); }
static size_t fused_image_only_bytes(int depth) { return (size_t)4 * depth * CH * CH * sizeof(uint32_t); }
size_t gmw_fused_image_bytes(int depth) {
    return fused_scales_bytes(depth) + fused_bias_bytes(depth) + fused_image_only_bytes(depth) + kExchangeBytes;
}

// Runs both nets of all objects.  reg_w != nullptr and at least three objects per group: PAIRED schedule, the kernel emits
// the edge weights itself (*emitted = true; nothing but reg_w is written to HBM; the first net's features are parked in the
// otherwise unused SLOT_Y1 area of the inference workspace, three slices per CTA, which stays in L2).  Otherwise the
// final features land in SLOT_X of the workspace (*emitted = false) for gmw_edge_weight_kernel / the correspondence branch.
// `tail` points to gmw_fused_image_bytes(depth) bytes (256-byte aligned).
int launch_gmw_fused_fwd(const MlpArgs& a, const float* params4, const float* params6, void* tail, float* reg_w, bool* emitted,
                         cudaStream_t st) {
    const int depth = a.L.depth;
    unsigned char* base = reinterpret_cast<unsigned char*>(tail);
    float2* scales2 = reinterpret_cast<float2*>(base);
    float* bias2 = reinterpret_cast<float*>(base + fused_scales_bytes(depth));
    uint32_t* wimg = reinterpret_cast<uint32_t*>(base + fused_scales_bytes(depth) + fused_bias_bytes(depth));
    float2* xg = reinterpret_cast<float2*>(base + fused_scales_bytes(depth) + fused_bias_bytes(depth) + fused_image_only_bytes(depth));
    // The CTAs of a group wait for each other, so all of them must be resident: cooperative launch, one CTA per SM.
    // (queried on every call: the library keeps no state between calls; these are host-side lookups, no device work)
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return DCD_E_DEVICE;
    // one instantiation per slice geometry (16-edge units per object and CTA, the range gmw_fused_supported accepts)
    using FusedKernel = void (*)(MlpArgs, const float2*, const float*, const uint32_t*, float2*, float*, float4*);
    static const FusedKernel kernels[] = {mlp_fused_kernel<3>, mlp_fused_kernel<4>, mlp_fused_kernel<5>, mlp_fused_kernel<6>,
                                          mlp_fused_kernel<7>};
    const int upo = (a.L.E + 16 * FCS - 1) / (16 * FCS);
    if (upo < 3 || upo > 7) return DCD_E_UNSUPPORTED;
    const FusedKernel kernel = kernels[upo - 3];
    cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFusedSmem);
    cudaFuncSetAttribute(fused_prep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(CH * CH * sizeof(float)));
    int coop = 0, per_sm = 0;
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, FTHREADS, kFusedSmem);
    if (!coop || per_sm < 1) return DCD_E_UNSUPPORTED;
    int max_groups = device_sm_count() * per_sm / FCS;
    if (max_groups > FMAX_GROUPS) max_groups = FMAX_GROUPS;
    if (max_groups < 1) return DCD_E_UNSUPPORTED;
    fused_prep_kernel<<<4 * depth, 1024, CH * CH * sizeof(float), st>>>(params4, params6, depth, a.fold, scales2, bias2, wimg);
    cudaMemsetAsync(xg, 0x80, kExchangeBytes, st);            // every word starts with the flag its first use does not expect
    // work is dealt to the groups as object triples (paired schedule: both nets of a triple back to back; the first net's
    // features are parked in one activation slot, FOBJ * FCS * ES columns per group) or as (triple, net) rounds
    const int64_t es = 16 * upo;
    const bool paired = reg_w != nullptr && a.L.N >= FOBJ * (int64_t)max_groups &&
                        a.L.N * (int64_t)a.L.EP >= (int64_t)max_groups * FOBJ * FCS * es;
    const int64_t npairs = (a.L.N + FOBJ - 1) / FOBJ;
    const int64_t nitems = paired ? npairs : npairs * 2;
    const int ngroups = (int)(nitems < max_groups ? nitems : max_groups);
    MlpArgs args = a;
    const float2* scales_arg = scales2;
    const float* bias_arg = bias2;
    const uint32_t* wimg_arg = wimg;
    float* regw_arg = paired ? reg_w : nullptr;
    float4* park_arg = reinterpret_cast<float4*>(act_ptr(a.ws, a.L, 0, 0, SLOT_Y1));
    void* kargs[] = {&args, &scales_arg, &bias_arg, &wimg_arg, &xg, &regw_arg, &park_arg};
    if (cudaLaunchCooperativeKernel(reinterpret_cast<void*>(kernel), dim3(FCS * ngroups), dim3(FTHREADS), kargs, kFusedSmem,
                                    st) != cudaSuccess) {
        cudaGetLastError();
        return DCD_E_LAUNCH;
    }
    *emitted = paired;
    return DCD_OK;
}

}  // namespace dcd
