// stack_tc.cu -- whole-model fused inference kernels on the 5th-gen tensor cores (tcgen05 + TMEM), fp32-accurate:
//   nf_spline_stack_tc_forward     L x SplineCouplingLayer (+ between-layer BatchNorm affine), hidden_dim <= 64
//   nf_coupling_stack_tc_forward   L x CouplingLayer in eval mode (conditioner BatchNorm folded at pack time)
// (spline_coupling_layer.py:96-309, coupling_layer.py:40-96, normalizing_flow_model.py:25-128)
//
// Mapping.  Warpgroup = 128 threads (one per CTA; two independent ones in the spline stack kernel, see there); thread t
// owns row t of a 128-row sub-tile and keeps its x / log-det in registers for
// the whole stack (a row is 8..32 bytes: HBM traffic is 4D in + 4D+4 out).  Per layer and sub-tile:
//   (a) layer 1 (K = data_dim <= 8) on the FP32 pipe, ReLU, 3xTF32 split, written by the owning thread straight
//       into TMEM as the A operand (lane = row, column = k) with tcgen05.st          -- no activation in smem
//   (b) layer 2: D2[128x64] = A1 * W2^T on tcgen05 (kind::tf32, M=128, N=64, 8 k-steps x 3 split passes),
//       W2 hi/lo images resident in shared memory (K-major SWIZZLE_128B, packed on the host)
//   (c) bias + ReLU + split of D2 (tcgen05.ld -> registers -> tcgen05.st) = A operand of the head
//   (d) head: D3[128 x 32*Dt] = A2 * W3^T on tcgen05 (every transformed dim's 3K-1 parameters padded to 32 columns)
//   (e) tcgen05.ld of the thread's own parameters, rational-quadratic spline / affine transform, row log-det.
// One elected thread issues the MMAs; completion comes back through an mbarrier (tcgen05.commit).  Layer weights
// (~50 KB) are double-buffered in shared memory with cp.async and shared by T sub-tiles; two CTAs per SM overlap
// one CTA's tensor phase with the other's FP32 phase.  TMEM: A_hi | A_lo | D2 | D3 = 64+64+64+<=64 columns.
#include <stdio.h>
#include "nf_common.cuh"
#include "nf_rng.cuh"
#include "stack_small.cuh"
#include "tc_common.cuh"

namespace nf {

constexpr int kTcThreads = 128;
constexpr int kTcSub = 4;            // sub-tiles (of 128 rows) per weight staging
constexpr int kColAhi = 0, kColAlo = 64, kColD2 = 128, kColD3 = 192;
constexpr int kTmemCols = 256;

__device__ __forceinline__ float relu_keepnan(float x) {      // torch.relu: NaN stays NaN
    float r;
    asm("max.NaN.f32 %0, %1, 0f00000000;" : "=f"(r) : "f"(x));
    return r;
}

// Row state of a tile in shared memory, sx [kTcSub][DM+1][128]: thread t of sub-tile s keeps its row's DM values and
// then its log-det slot, from the row load through every layer to the row store.
template <int DM>
__device__ __forceinline__ float slab_load(const float* sx, int s, int t, float (&xv)[DM]) {
#pragma unroll
    for (int d = 0; d < DM; ++d) xv[d] = sx[(s * (DM + 1) + d) * kTcThreads + t];
    return sx[(s * (DM + 1) + DM) * kTcThreads + t];
}

template <int DM>
__device__ __forceinline__ void slab_store(float* sx, int s, int t, const float (&xv)[DM], float tot) {
#pragma unroll
    for (int d = 0; d < DM; ++d) sx[(s * (DM + 1) + d) * kTcThreads + t] = xv[d];
    sx[(s * (DM + 1) + DM) * kTcThreads + t] = tot;
}

// SAMPLE variants of the stack kernels (nf_*_sample): the row is the N(0, I) draw of nf_rng.cuh instead of a load, and
// its log-det slot starts at -log N(z) -- the epilogue stores the negated sum, log N(z) - log_det (sample_and_log_prob).
// rng_state != NULL (nf_*_sample_state): the key comes from the device-resident state, taken by every CTA before the
// setup barrier into two words after the barriers (the launch adds 16 bytes of shared memory for them) and advanced by
// the launch; otherwise from the seed / offset arguments.  Non-SAMPLE kernels ignore it.  The coupling and MADE kernels
// read the key where they draw (it then holds no registers across the kernel), the spline kernel once after its setup
// barrier: each is the form with the lower register and spill counts.
// rng_key: the key slot of nf_rng_state_take when the launch has a device-resident state, NULL otherwise
template <int DM>
__device__ __forceinline__ void draw_row_tc(float* srow, int64_t r, int64_t B, int D, uint64_t seed, uint64_t offset,
                                            const unsigned long long* rng_key) {
    if (rng_key) { seed = rng_key[0]; offset = rng_key[1]; }
    float z[DM];
    const float lz = nf_std_normal_row<DM>(seed, offset, (uint32_t)r, D, z);
#pragma unroll
    for (int d = 0; d < DM; ++d) srow[d * kTcThreads] = (r < B) ? z[d] : 0.f;
    srow[DM * kTcThreads] = -lz;
}

// One CTA-wide round of the coupling and MADE kernels: every thread's TMEM stores are done, warp 0 issues the MMAs
// (`issue`, completing on `bar`), and every thread waits for them.
template <typename Issue>
__device__ __forceinline__ void cta_mma_round(int warp, uint64_t* bar, uint32_t& phase, Issue issue) {
    tc::wait_st();
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) { tc::fence_after_sync(); issue(); }
    tc::mbar_wait(bar, phase); phase ^= 1;
    tc::fence_after_sync();
}

// Layer 1 for data_dim <= 3 (W1S == 4), two hidden units per packed-fp32 FMA.  The host stores the units in pairs:
// [w0a w0b | w1a w1b | w2a w2b | ba bb] (packing._tc_net_block), i.e. two LDS.128 per pair like the unit-major layout, and
// every FFMA2 operand pair sits in adjacent registers.  Returns relu(W1 x + b1) of units 2p, 2p+1.
template <int DM>
__device__ __forceinline__ float2 layer1_pair(const float* __restrict__ sW1k, int p, const float (&xa)[DM]) {
    const float4 wa = *reinterpret_cast<const float4*>(sW1k + p * 8);          // w0a w0b w1a w1b
    const float4 wb = *reinterpret_cast<const float4*>(sW1k + p * 8 + 4);      // w2a w2b ba  bb
    float2 t = make_float2(wb.z, wb.w);
    t = __ffma2_rn(make_float2(wa.x, wa.y), make_float2(xa[0], xa[0]), t);
    if constexpr (DM > 1) t = __ffma2_rn(make_float2(wa.z, wa.w), make_float2(xa[1], xa[1]), t);
    if constexpr (DM > 2) t = __ffma2_rn(make_float2(wb.x, wb.y), make_float2(xa[2], xa[2]), t);
    return make_float2(relu_keepnan(t.x), relu_keepnan(t.y));
}

// (c): D2 + b2 -> ReLU -> split -> A operand.  Four 16-column loads are issued before each wait (64 columns at a time).
template <int HP = 64>
__device__ __forceinline__ void hidden2_to_tmem(const float* __restrict__ sb2, uint32_t lane_addr) {
    constexpr int kColAhi = 0, kColAlo = HP, kColD2 = 2 * HP;
#pragma unroll
    for (int cg = 0; cg < HP / 64; ++cg) {
        uint32_t v[4][16];
#pragma unroll
        for (int c = 0; c < 4; ++c) tc::tmem_ld16(lane_addr + kColD2 + (cg * 4 + c) * 16, v[c]);
        tc::wait_ld();
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            uint32_t hi[16], lo[16];
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
                const float4 b = *reinterpret_cast<const float4*>(sb2 + (cg * 4 + c) * 16 + j4 * 4);
                const float2 s0 = __fadd2_rn(make_float2(__uint_as_float(v[c][j4 * 4 + 0]), __uint_as_float(v[c][j4 * 4 + 1])), make_float2(b.x, b.y));
                const float2 s1 = __fadd2_rn(make_float2(__uint_as_float(v[c][j4 * 4 + 2]), __uint_as_float(v[c][j4 * 4 + 3])), make_float2(b.z, b.w));
                tc::split_tf32_x2(relu_keepnan(s0.x), relu_keepnan(s0.y), hi[j4 * 4 + 0], hi[j4 * 4 + 1], lo[j4 * 4 + 0], lo[j4 * 4 + 1]);
                tc::split_tf32_x2(relu_keepnan(s1.x), relu_keepnan(s1.y), hi[j4 * 4 + 2], hi[j4 * 4 + 3], lo[j4 * 4 + 2], lo[j4 * 4 + 3]);
            }
            tc::tmem_st16(lane_addr + kColAhi + (cg * 4 + c) * 16, hi);
            tc::tmem_st16(lane_addr + kColAlo + (cg * 4 + c) * 16, lo);
        }
    }
}

// named barriers (ids 1..15; id 0 is __syncthreads): sub-block synchronisation of the two-warpgroup kernel
__device__ __forceinline__ void named_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
__device__ __forceinline__ void named_arrive(int id, int nthreads) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// layout of one layer block in shared memory (words)
struct BlkOff { int w1k, b2, b3, wc, w2hi, w2lo, w3hi, w3lo, net_words; };
__host__ __device__ inline int pad256(int x) { return (x + 255) & ~255; }
// nets conditioner blocks follow the 80-word layer header; every block is a multiple of 256 words so that the
// weight images stay 1024-byte aligned
// HP: hidden units padded to 64 (every kernel here) or 128 (the affine coupling stack with hidden_dim in (64, 128])
// CW: context columns of the conditional layouts ('NFC2' spline, 'NFD2' affine: Wc[HP/2][CW][2] after b3), 0 in every other
// layout
__host__ __device__ inline BlkOff blk_offsets(int W1S, int NO3, int HP = 64, int CW = 0) {
    BlkOff o;
    o.w1k = 0; o.b2 = HP * W1S; o.b3 = o.b2 + HP;
    o.w2hi = pad256(NF_LAYER_HDR + o.b3 + NO3 + HP * CW) - NF_LAYER_HDR;   // first net: header shares the leading pad
    o.wc = o.b3 + NO3;
    o.w2lo = o.w2hi + HP * HP; o.w3hi = o.w2lo + HP * HP; o.w3lo = o.w3hi + NO3 * HP;
    o.net_words = o.w3lo + NO3 * HP;
    return o;
}

// ------------------------------------------------------------------------------------------------
// spline stack: two independent warpgroups per CTA (256 threads), half-K staging.
// Each warpgroup owns 128 TMEM columns: A_hi 32 | A_lo 32 | D 64.  A K=64 contraction is fed in two halves of 32
// (st half 1 -> 12 MMAs -> st half 2 -> 12 accumulating MMAs), the second half being computed on the FP32 pipe while
// the first half's MMAs run; the head accumulator aliases D2 (read out to registers first).  Halving the A footprint
// doubles the number of concurrent tensor windows per SM: 2 CTAs x 2 warpgroups = 4 windows, 16 resident warps.
// ------------------------------------------------------------------------------------------------
constexpr int kTc2Threads = 256;
constexpr int kWgCols = 128, kWgAhi = 0, kWgAlo = 32, kWgD = 64;

// 16 hidden-layer-1 outputs (units u0..u0+15) of this thread's row: relu, split
template <int DM>
__device__ __forceinline__ void layer1_chunk(const float* __restrict__ sW1k, int W1S, const float (&xa)[DM], int u0,
                                             uint32_t (&hi)[16], uint32_t (&lo)[16]) {
    if constexpr (DM <= 4) {
#pragma unroll
        for (int j = 0; j < 16; j += 2) {
            const float2 t = layer1_pair<DM>(sW1k, (u0 + j) >> 1, xa);
            tc::split_tf32_x2(t.x, t.y, hi[j], hi[j + 1], lo[j], lo[j + 1]);
        }
    } else {
        float t16[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const float* w1 = sW1k + (u0 + j) * W1S;
            const float4 v0 = *reinterpret_cast<const float4*>(w1);
            const float4 v1 = *reinterpret_cast<const float4*>(w1 + 4);
            float t = w1[W1S - 1];
            t = fmaf(v0.x, xa[0], t); t = fmaf(v0.y, xa[1], t); t = fmaf(v0.z, xa[2], t); t = fmaf(v0.w, xa[3], t);
            t = fmaf(v1.x, xa[4], t); t = fmaf(v1.y, xa[5], t); t = fmaf(v1.z, xa[6], t); t = fmaf(v1.w, xa[7], t);
            t16[j] = relu_keepnan(t);
        }
#pragma unroll
        for (int j = 0; j < 16; j += 2) tc::split_tf32_x2(t16[j], t16[j + 1], hi[j], hi[j + 1], lo[j], lo[j + 1]);
    }
}

// Conditional twin of layer1_chunk: the same x FMAs in the same order, then the C context FMAs of each unit, in column
// order, before the ReLU.  Wc holds the units in pairs, [c0a c0b | c1a c1b | ..] with CM column slots per pair
// (packing._tc_wc), so every FFMA2 finds both units' weights in adjacent registers.  The loop runs column by column over
// the chunk's 8 unit pairs, reading one context value (through L1) at a time: holding the row's CM values beside the
// chunk's accumulators pushes the DM = 2 kernels into spills.  Columns at or beyond the runtime C are skipped, as
// KS == 0 skips the bins beyond num_bins.
template <int DM, int CM>
__device__ __forceinline__ void layer1_chunk_ctx(const float* __restrict__ sW1k, int W1S, const float* __restrict__ sWc,
                                                 const float (&xa)[DM], const float* __restrict__ crow, int C, int u0,
                                                 uint32_t (&hi)[16], uint32_t (&lo)[16]) {
    float2 t[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        if constexpr (DM <= 4) {
            const int p = (u0 >> 1) + q;
            const float4 wa = *reinterpret_cast<const float4*>(sW1k + p * 8);
            const float4 wb = *reinterpret_cast<const float4*>(sW1k + p * 8 + 4);
            t[q] = make_float2(wb.z, wb.w);
            t[q] = __ffma2_rn(make_float2(wa.x, wa.y), make_float2(xa[0], xa[0]), t[q]);
            if constexpr (DM > 1) t[q] = __ffma2_rn(make_float2(wa.z, wa.w), make_float2(xa[1], xa[1]), t[q]);
            if constexpr (DM > 2) t[q] = __ffma2_rn(make_float2(wb.x, wb.y), make_float2(xa[2], xa[2]), t[q]);
        } else {
            float u[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const float* w1 = sW1k + (u0 + 2 * q + e) * W1S;
                const float4 v0 = *reinterpret_cast<const float4*>(w1);
                const float4 v1 = *reinterpret_cast<const float4*>(w1 + 4);
                float a = w1[W1S - 1];
                a = fmaf(v0.x, xa[0], a); a = fmaf(v0.y, xa[1], a); a = fmaf(v0.z, xa[2], a); a = fmaf(v0.w, xa[3], a);
                a = fmaf(v1.x, xa[4], a); a = fmaf(v1.y, xa[5], a); a = fmaf(v1.z, xa[6], a); a = fmaf(v1.w, xa[7], a);
                u[e] = a;
            }
            t[q] = make_float2(u[0], u[1]);
        }
    }
    const float* wc = sWc + (u0 >> 1) * (2 * CM);
#pragma unroll 1
    for (int c = 0; c < C; ++c) {
        const float v = __ldg(crow + c);
#pragma unroll
        for (int q = 0; q < 8; ++q)
            t[q] = __ffma2_rn(*reinterpret_cast<const float2*>(wc + q * 2 * CM + 2 * c), make_float2(v, v), t[q]);
    }
#pragma unroll
    for (int q = 0; q < 8; ++q)
        tc::split_tf32_x2(relu_keepnan(t[q].x), relu_keepnan(t[q].y), hi[2 * q], hi[2 * q + 1], lo[2 * q], lo[2 * q + 1]);
}

// (a): hidden layer 1 of one conditioner for this thread's row -> TMEM A operand (hi at kColAhi, lo at kColAlo).
// CM > 0 (the conditional affine layout 'NFD2'): each 16-unit chunk goes through layer1_chunk_ctx, which adds the C
// context columns of row `crow` (Wc at sWc) after the x FMAs of every unit, before the ReLU.
template <int DM, int HP = 64, int CM = 0>
__device__ __forceinline__ void layer1_to_tmem(const float* __restrict__ sW1k, int W1S, const float (&xa)[DM], uint32_t lane_addr,
                                               const float* __restrict__ sWc = nullptr, const float* __restrict__ crow = nullptr,
                                               int C = 0) {
    constexpr int kColAhi = 0, kColAlo = HP;        // TMEM columns of an HP-wide conditioner: A hi | A lo | D2 | D3
#pragma unroll
    for (int c = 0; c < HP / 16; ++c) {
        uint32_t hi[16], lo[16];
        if constexpr (CM > 0) {
            layer1_chunk_ctx<DM, CM>(sW1k, W1S, sWc, xa, crow, C, c * 16, hi, lo);
        } else if constexpr (DM <= 4) {
#pragma unroll
            for (int j = 0; j < 16; j += 2) {
                const float2 t = layer1_pair<DM>(sW1k, (c * 16 + j) >> 1, xa);
                tc::split_tf32_x2(t.x, t.y, hi[j], hi[j + 1], lo[j], lo[j + 1]);
            }
        } else {
            float t16[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const float* w1 = sW1k + (c * 16 + j) * W1S;
                const float4 v0 = *reinterpret_cast<const float4*>(w1);
                const float4 v1 = *reinterpret_cast<const float4*>(w1 + 4);
                float t = w1[W1S - 1];
                t = fmaf(v0.x, xa[0], t); t = fmaf(v0.y, xa[1], t); t = fmaf(v0.z, xa[2], t); t = fmaf(v0.w, xa[3], t);
                t = fmaf(v1.x, xa[4], t); t = fmaf(v1.y, xa[5], t); t = fmaf(v1.z, xa[6], t); t = fmaf(v1.w, xa[7], t);
                t16[j] = relu_keepnan(t);
            }
#pragma unroll
            for (int j = 0; j < 16; j += 2) tc::split_tf32_x2(t16[j], t16[j + 1], hi[j], hi[j + 1], lo[j], lo[j + 1]);
        }
        tc::tmem_st16(lane_addr + kColAhi + c * 16, hi);
        tc::tmem_st16(lane_addr + kColAlo + c * 16, lo);
    }
}

// 16 raw layer-2 accumulators + bias -> relu -> split
__device__ __forceinline__ void hidden2_chunk(const uint32_t (&v)[16], const float* __restrict__ sb2, uint32_t (&hi)[16], uint32_t (&lo)[16]) {
#pragma unroll
    for (int j4 = 0; j4 < 4; ++j4) {
        const float4 b = *reinterpret_cast<const float4*>(sb2 + j4 * 4);
        // packed fp32 (FADD2 / FMUL2 / FFMA2): bias add and the hi/lo split two values per instruction
        const float2 s0 = __fadd2_rn(make_float2(__uint_as_float(v[j4 * 4 + 0]), __uint_as_float(v[j4 * 4 + 1])), make_float2(b.x, b.y));
        const float2 s1 = __fadd2_rn(make_float2(__uint_as_float(v[j4 * 4 + 2]), __uint_as_float(v[j4 * 4 + 3])), make_float2(b.z, b.w));
        tc::split_tf32_x2(relu_keepnan(s0.x), relu_keepnan(s0.y), hi[j4 * 4 + 0], hi[j4 * 4 + 1], lo[j4 * 4 + 0], lo[j4 * 4 + 1]);
        tc::split_tf32_x2(relu_keepnan(s1.x), relu_keepnan(s1.y), hi[j4 * 4 + 2], hi[j4 * 4 + 3], lo[j4 * 4 + 2], lo[j4 * 4 + 3]);
    }
}

// KS > 0: num_bins known at compile time (== KMAX), every per-bin guard folds away; KS == 0: runtime num_bins <= KMAX.
// CM > 0: the conditional layout ('NFC2'): layer 1 also reads C <= CM context columns of row r / ctx_div of `ctx`,
// fetched through L1 at every layer (see DESIGN.md §3); CM == 0 is the unconditional kernel, the context arguments unused.
// tid: threadIdx.x read in the __global__ wrapper, where the compiler knows its range from __launch_bounds__ (read here,
// it would not, and the CM == 0 code would differ from the kernel's before the body moved here).
template <int DM, int KMAX, int KS, bool SAMPLE, int CM>
__device__ __forceinline__ void
spline_stack_tc2_body(int tid, const float* __restrict__ packed, const float* __restrict__ x, float* __restrict__ y,
                      float* __restrict__ ld, int64_t B, int flags, uint64_t seed, uint64_t offset,
                      unsigned long long* rng_state, const float* __restrict__ ctx, int64_t ctx_div, int C) {
    const int inverse = flags & NF_STACK_INVERSE;
    extern __shared__ __align__(1024) float sbuf[];
    const StackHdr hd = nf_stack_hdr_device(packed);
    const int D = hd.D, K = (KS > 0) ? KS : hd.K, L = hd.L, W1S = hd.W1S, NO3 = hd.NO, BW = hd.layer_stride;
    float* sx = sbuf + (size_t)2 * BW;                         // [kTcSub][DM+1][128] row state
    uint64_t* bars = reinterpret_cast<uint64_t*>(sx + kTcSub * (DM + 1) * kTcThreads);
    uint64_t* mbar = bars;                                     // [2] MMA completion, one per warpgroup
    uint64_t* wbar = bars + 2;                                 // [2] weight-block arrival
    uint32_t& tmem_base_s = *reinterpret_cast<uint32_t*>(bars + 4);
    const BlkOff off = blk_offsets(W1S, NO3, 64, CM);

    RqsCfg<float> cfg;
    cfg.lo = -hd.bound; cfg.hi = hd.bound; cfg.span = 2.0f * hd.bound; cfg.eps = 1e-8f;
    cfg.min_w = hd.min_w; cfg.min_h = hd.min_h; cfg.min_d = hd.min_d; cfg.scale_w = hd.scale_w; cfg.scale_h = hd.scale_h;

    const int warp = tid >> 5, wg = tid >> 7, wtid = tid & 127, wwarp = warp & 3;
    const int bar_local = 1 + wg;
    if (warp == 0) tc::tmem_alloc(&tmem_base_s, kTmemCols);
    unsigned long long* rng_key = reinterpret_cast<unsigned long long*>(bars + 5);   // SAMPLE + device state: every
    if constexpr (SAMPLE) if (rng_state) nf_rng_state_take(rng_state, rng_key);   // CTA, before the role split / tiles
    if (tid == 0) {
        tc::mbar_init(&mbar[0], 1); tc::mbar_init(&mbar[1], 1); tc::mbar_init(&wbar[0], 1); tc::mbar_init(&wbar[1], 1);
        tc::fence_mbar_init();
    }
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    // this kernel takes the key into the seed / offset registers once (reading it at each draw, as the coupling and MADE
    // kernels do, makes ptxas spill in the DM = 4 twins); the draw below is then the host-key code unchanged
    if constexpr (SAMPLE) if (rng_state) { seed = rng_key[0]; offset = rng_key[1]; }
    const uint32_t tb = tmem_base_s + (uint32_t)(wg * kWgCols);           // this warpgroup's 128 columns
    const uint32_t lane_addr = tb + ((uint32_t)(wwarp * 32) << 16);
    uint64_t* mb = &mbar[wg];
    uint32_t phase = 0, wphase = 0u;

    constexpr int ROWS = kTcThreads * kTcSub;
    const int64_t ntiles = (B + ROWS - 1) / ROWS;
    const float* layers = packed + NF_STACK_HDR;
    int buf = 0;
    if (tid == 0 && (int64_t)blockIdx.x < ntiles) {
        tc::mbar_arrive_expect_tx(&wbar[0], (uint32_t)BW * 4u);
        tc::bulk_g2s(sbuf, layers + (size_t)(inverse ? L - 1 : 0) * BW, (uint32_t)BW * 4u, &wbar[0]);
    }
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        for (int s = wg; s < kTcSub; s += 2) {
            const int64_t r = tile * ROWS + s * kTcThreads + wtid;
            if constexpr (SAMPLE) {
                draw_row_tc<DM>(sx + s * (DM + 1) * kTcThreads + wtid, r, B, D, seed, offset, nullptr);
                continue;
            }
#pragma unroll
            for (int d = 0; d < DM; ++d) sx[(s * (DM + 1) + d) * kTcThreads + wtid] = (d < D && r < B) ? ld_stream(x + r * D + d) : 0.f;
            sx[(s * (DM + 1) + DM) * kTcThreads + wtid] = 0.f;
        }
        for (int li = 0; li < L; ++li) {
            tc::fence_proxy_async_smem();
            __syncthreads();                                    // both warpgroups are done with the other buffer
            if (tid == 0) {
                const bool last = (li == L - 1);
                if (!last || (tile + gridDim.x < ntiles)) {
                    const int nli = last ? 0 : li + 1;
                    tc::mbar_arrive_expect_tx(&wbar[buf ^ 1], (uint32_t)BW * 4u);
                    tc::bulk_g2s(sbuf + (size_t)(buf ^ 1) * BW, layers + (size_t)(inverse ? L - 1 - nli : nli) * BW,
                                 (uint32_t)BW * 4u, &wbar[buf ^ 1]);
                }
            }
            tc::mbar_wait(&wbar[buf], (wphase >> buf) & 1u);
            wphase ^= (1u << buf);
            const float* sL = sbuf + (size_t)buf * BW;
            const float* net = sL + NF_LAYER_HDR;
            const LayerHdr lh{sL};
            const bool rescale = lh.rescale(), bn_on = lh.bn_on();
            const float* mask = lh.mask();
            const uint32_t w2hi = tc::smem_u32(net + off.w2hi), w2lo = tc::smem_u32(net + off.w2lo);
            const uint32_t w3hi = tc::smem_u32(net + off.w3hi), w3lo = tc::smem_u32(net + off.w3lo);
            const float* sW1k = net + off.w1k;
            const float* sb2 = net + off.b2;

#pragma unroll 1
            for (int s = wg; s < kTcSub; s += 2) {
                float xv[DM];
                float tot = slab_load<DM>(sx, s, wtid, xv);
                if (inverse && bn_on) nf_stack_bn_between<DM>(lh, D, true, xv, tot);
                float xs[DM], xa[DM];
#pragma unroll
                for (int d = 0; d < DM; ++d) {
                    float v = xv[d];
                    if (rescale && d < D) v = lh.to_spline(v, d, hd.bound);
                    xs[d] = v;
                    xa[d] = (d < D) ? v * mask[d] : 0.f;
                }
                uint32_t hi[16], lo[16];
                uint32_t crow = 0;                              // the row's context row (conditional kernel)
                if constexpr (CM > 0) {
                    const int64_t r = tile * ROWS + s * kTcThreads + wtid;     // < 2^31, as ctx_div (the launcher)
                    crow = r < B ? (uint32_t)r / (uint32_t)ctx_div : 0u;
                }
                // ---- layer 2, K half 1: hidden units 0..31 ----
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    if constexpr (CM > 0) layer1_chunk_ctx<DM, CM>(sW1k, W1S, net + off.wc, xa, ctx + (size_t)crow * C, C, c * 16, hi, lo);
                    else layer1_chunk<DM>(sW1k, W1S, xa, c * 16, hi, lo);
                    tc::tmem_st16(lane_addr + kWgAhi + c * 16, hi);
                    tc::tmem_st16(lane_addr + kWgAlo + c * 16, lo);
                }
                tc::wait_st();
                tc::fence_before_sync();
                named_sync(bar_local, kTcThreads);
                if (wwarp == 0) { tc::fence_after_sync(); tc::warp_issue_gemm_krange_3xtf32(tb, kWgD, kWgAhi, kWgAlo, w2hi, w2lo, 64u, 0, 4, 0u, mb); }
                // ---- K half 2: hidden units 32..63, computed while half 1 multiplies ----
                uint32_t hi2[16], lo2[16];
                if constexpr (CM > 0) {
                    layer1_chunk_ctx<DM, CM>(sW1k, W1S, net + off.wc, xa, ctx + (size_t)crow * C, C, 32, hi, lo);
                    layer1_chunk_ctx<DM, CM>(sW1k, W1S, net + off.wc, xa, ctx + (size_t)crow * C, C, 48, hi2, lo2);
                } else {
                    layer1_chunk<DM>(sW1k, W1S, xa, 32, hi, lo);
                    layer1_chunk<DM>(sW1k, W1S, xa, 48, hi2, lo2);
                }
                tc::mbar_wait(mb, phase); phase ^= 1;           // half-1 MMAs done: the A columns are free
                tc::fence_after_sync();
                tc::tmem_st16(lane_addr + kWgAhi, hi);   tc::tmem_st16(lane_addr + kWgAlo, lo);
                tc::tmem_st16(lane_addr + kWgAhi + 16, hi2); tc::tmem_st16(lane_addr + kWgAlo + 16, lo2);
                tc::wait_st();
                tc::fence_before_sync();
                named_sync(bar_local, kTcThreads);
                if (wwarp == 0) { tc::fence_after_sync(); tc::warp_issue_gemm_krange_3xtf32(tb, kWgD, kWgAhi, kWgAlo, w2hi, w2lo, 64u, 4, 4, 1u, mb); }
                tc::mbar_wait(mb, phase); phase ^= 1;
                tc::fence_after_sync();
                // ---- head: D2 -> registers (the head accumulator aliases it), two K halves again ----
                uint32_t v0[16], v1[16], v2[16], v3[16];
                tc::tmem_ld16(lane_addr + kWgD, v0);      tc::tmem_ld16(lane_addr + kWgD + 16, v1);
                tc::tmem_ld16(lane_addr + kWgD + 32, v2); tc::tmem_ld16(lane_addr + kWgD + 48, v3);
                tc::wait_ld();
                hidden2_chunk(v0, sb2, hi, lo);
                tc::tmem_st16(lane_addr + kWgAhi, hi); tc::tmem_st16(lane_addr + kWgAlo, lo);
                hidden2_chunk(v1, sb2 + 16, hi, lo);
                tc::tmem_st16(lane_addr + kWgAhi + 16, hi); tc::tmem_st16(lane_addr + kWgAlo + 16, lo);
                tc::wait_st();
                tc::fence_before_sync();
                named_sync(bar_local, kTcThreads);
                if (wwarp == 0) { tc::fence_after_sync(); tc::warp_issue_gemm_krange_3xtf32(tb, kWgD, kWgAhi, kWgAlo, w3hi, w3lo, (uint32_t)NO3, 0, 4, 0u, mb); }
                hidden2_chunk(v2, sb2 + 32, hi, lo);
                hidden2_chunk(v3, sb2 + 48, hi2, lo2);
                tc::mbar_wait(mb, phase); phase ^= 1;
                tc::fence_after_sync();
                tc::tmem_st16(lane_addr + kWgAhi, hi);   tc::tmem_st16(lane_addr + kWgAlo, lo);
                tc::tmem_st16(lane_addr + kWgAhi + 16, hi2); tc::tmem_st16(lane_addr + kWgAlo + 16, lo2);
                tc::wait_st();
                tc::fence_before_sync();
                named_sync(bar_local, kTcThreads);
                if (wwarp == 0) { tc::fence_after_sync(); tc::warp_issue_gemm_krange_3xtf32(tb, kWgD, kWgAhi, kWgAlo, w3hi, w3lo, (uint32_t)NO3, 4, 4, 1u, mb); }
                tc::mbar_wait(mb, phase); phase ^= 1;
                tc::fence_after_sync();

                // ---- spline parameters of this row: 32 columns per transformed dim ----
                float lsum = 0.f;
                int t = 0;
#pragma unroll
                for (int d = 0; d < DM; ++d) {
                    if (d < D && mask[d] == 0.f) {
                        uint32_t p0[16], p1[16];
                        tc::tmem_ld16(lane_addr + kWgD + t * 32, p0);
                        if constexpr (3 * KMAX - 1 <= 24) {
                            uint32_t q[8];
                            tc::tmem_ld8(lane_addr + kWgD + t * 32 + 16, q);
#pragma unroll
                            for (int j = 0; j < 8; ++j) p1[j] = q[j];
#pragma unroll
                            for (int j = 8; j < 16; ++j) p1[j] = 0u;
                        } else {
                            tc::tmem_ld16(lane_addr + kWgD + t * 32 + 16, p1);
                        }
                        tc::wait_ld();
                        const float* b3 = net + off.b3 + t * 32;
                        float prm[32];
#pragma unroll
                        for (int j = 0; j < 16; j += 4) {             // packed fp32 bias adds (FADD2), bias fetched 16 bytes at a time
                            const float4 ba = *reinterpret_cast<const float4*>(b3 + j), bb = *reinterpret_cast<const float4*>(b3 + 16 + j);
                            const float2 s0 = __fadd2_rn(make_float2(__uint_as_float(p0[j]), __uint_as_float(p0[j + 1])), make_float2(ba.x, ba.y));
                            const float2 s1 = __fadd2_rn(make_float2(__uint_as_float(p0[j + 2]), __uint_as_float(p0[j + 3])), make_float2(ba.z, ba.w));
                            const float2 s2 = __fadd2_rn(make_float2(__uint_as_float(p1[j]), __uint_as_float(p1[j + 1])), make_float2(bb.x, bb.y));
                            const float2 s3 = __fadd2_rn(make_float2(__uint_as_float(p1[j + 2]), __uint_as_float(p1[j + 3])), make_float2(bb.z, bb.w));
                            prm[j] = s0.x; prm[j + 1] = s0.y; prm[j + 2] = s1.x; prm[j + 3] = s1.y;
                            prm[16 + j] = s2.x; prm[16 + j + 1] = s2.y; prm[16 + j + 2] = s3.x; prm[16 + j + 3] = s3.y;
                        }
                        float uw[KMAX], uh[KMAX], ud[KMAX];
#pragma unroll
                        for (int j = 0; j < KMAX; ++j) {
                            uw[j] = prm[j];
                            uh[j] = prm[KMAX + j];
                            ud[j] = (j < KMAX - 1) ? prm[2 * KMAX + j] : 0.f;
                        }
                        float out, lad;
                        rqs_eval<float, KMAX, true>(xs[d], uw, uh, ud, K, inverse != 0, cfg, out, lad);
                        if (rescale) out = lh.from_spline(out, d, hd.bound);
                        xv[d] = out;
                        lsum += lad;
                        ++t;
                    }
                }
                tc::fence_before_sync();                        // D3 reads precede the next sub-tile's MMA writes
#pragma unroll
                for (int d = 0; d < DM; ++d) xv[d] = scrub0(xv[d]);
                tot += scrub0(lsum);
                if (!inverse && bn_on) nf_stack_bn_between<DM>(lh, D, false, xv, tot);
                slab_store<DM>(sx, s, wtid, xv, tot);
            }
            buf ^= 1;
        }
        for (int s = wg; s < kTcSub; s += 2) {
            const int64_t r = tile * ROWS + s * kTcThreads + wtid;
            if (r < B) {
                float zr[DM];
#pragma unroll
                for (int d = 0; d < DM; ++d) zr[d] = sx[(s * (DM + 1) + d) * kTcThreads + wtid];
                if (!(flags & NF_STACK_SKIP_Y)) {
#pragma unroll
                    for (int d = 0; d < DM; ++d) if (d < D) st_stream(y + r * D + d, zr[d]);
                }
                const float tot = sx[(s * (DM + 1) + DM) * kTcThreads + wtid];
                st_stream(ld + r, SAMPLE ? -tot : (flags & NF_STACK_LOG_PROB_HEAD) ? nf_stack_row_head<DM>(zr, D, tot) : tot);
            }
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc(tmem_base_s, kTmemCols);
}

template <int DM, int KMAX, int KS, bool SAMPLE = false>
__global__ void __launch_bounds__(kTc2Threads, 2)
spline_stack_tc2_kernel(const float* __restrict__ packed, const float* __restrict__ x, float* __restrict__ y,
                        float* __restrict__ ld, int64_t B, int flags, uint64_t seed, uint64_t offset,
                        unsigned long long* rng_state) {
    spline_stack_tc2_body<DM, KMAX, KS, SAMPLE, 0>(threadIdx.x, packed, x, y, ld, B, flags, seed, offset, rng_state, nullptr, 1, 0);
}

// conditional spline stack ('NFC2'): C <= kCtxMax context columns of row r / ctx_div enter every layer's first Linear
constexpr int kCtxMax = 8;
template <int DM, int KMAX, int KS, bool SAMPLE = false>
__global__ void __launch_bounds__(kTc2Threads, 2)
spline_stack_ctx_tc2_kernel(const float* __restrict__ packed, const float* __restrict__ x, float* __restrict__ y,
                            float* __restrict__ ld, int64_t B, int flags, uint64_t seed, uint64_t offset,
                            unsigned long long* rng_state, const float* __restrict__ ctx, int64_t ctx_div, int C) {
    spline_stack_tc2_body<DM, KMAX, KS, SAMPLE, kCtxMax>(threadIdx.x, packed, x, y, ld, B, flags, seed, offset, rng_state, ctx, ctx_div,
                                                         C);
}

// ------------------------------------------------------------------------------------------------
// affine coupling stack (eval mode; conditioner BatchNorm folded into the Linears at pack time)
//   per layer two conditioner nets (s_net, b_net: coupling_layer.py:18-35) run one after the other through the same
//   TMEM regions; the staging unit is one NET block (header lead + W1k | b2 | b3 | W2 hi/lo | W3 hi/lo, ~43 KB), double
//   buffered: while net b computes, the next layer's net s arrives.  Head: D outputs padded to 16 columns.
// ------------------------------------------------------------------------------------------------
// HP = 128 (hidden_dim in (64, 128], e.g. the reference's published RealNVP(2, 10, 128)): A hi / lo 2 x 128 TMEM columns,
//   D2 128, D3 16 = all 512 columns of the SM, so ONE CTA per SM; a net block is ~151 KB (W2 hi / lo images alone 128 KB)
//   and is single buffered -- the next block is requested when every thread is done with the current one (~1 us of a
//   ~16 us net pass per tile).  Same code otherwise: K = 128 is 16 k-steps per pass, the head reads 4 K atoms.
// CM > 0: the conditional layout ('NFD2'): layer 1 of both nets also reads C <= CM context columns of row r / ctx_div
// of `ctx`, through L1 at every use, as the conditional spline kernel; CM == 0 is the unconditional kernel.  tid: see
// spline_stack_tc2_body.
template <int DM, int HP, bool SAMPLE, int CM>
__device__ __forceinline__ void
coupling_stack_tc_body(int tid, const float* __restrict__ packed, const float* __restrict__ x, float* __restrict__ y,
                       float* __restrict__ ld, int64_t B, int flags, int nsub, uint64_t seed, uint64_t offset,
                       unsigned long long* rng_state, const float* __restrict__ ctx, int64_t ctx_div, int C) {
    constexpr int NBUF = (HP == 64) ? 2 : 1;
    constexpr int kColAhi = 0, kColAlo = HP, kColD2 = 2 * HP, kColD3 = 3 * HP;
    constexpr int kTmemCols = (HP == 64) ? 256 : 512;
    const int inverse = flags & NF_STACK_INVERSE;
    extern __shared__ __align__(1024) float sbuf[];
    const StackHdr hd = nf_stack_hdr_device(packed);
    const int D = hd.D, L = hd.L, W1S = hd.W1S, NO3 = hd.NO, NBW = hd.layer_stride;     // NBW: words per net block
    float* sx = sbuf + (size_t)NBUF * NBW;                       // [kTcSub][DM+1][128] row state
    float* sraw = sx + kTcSub * (DM + 1) * kTcThreads;           // [kTcSub][DM][128] raw s_net outputs
    float* shdr = sraw + kTcSub * DM * kTcThreads;               // [80] layer header (outlives the net-s buffer)
    uint64_t* bars = reinterpret_cast<uint64_t*>(shdr + NF_LAYER_HDR);
    uint64_t& bar = bars[0];
    uint64_t* wbar = bars + 1;
    uint32_t& tmem_base_s = *reinterpret_cast<uint32_t*>(bars + 3);
    const BlkOff off = blk_offsets(W1S, NO3, HP, CM);

    const int warp = tid >> 5;
    if (warp == 0) tc::tmem_alloc(&tmem_base_s, kTmemCols);
    unsigned long long* rng_key = reinterpret_cast<unsigned long long*>(bars + 4);   // SAMPLE + device state: every
    if constexpr (SAMPLE) if (rng_state) nf_rng_state_take(rng_state, rng_key);   // CTA, before the role split / tiles
    if (tid == 0) { tc::mbar_init(&bar, 1); tc::mbar_init(&wbar[0], 1); tc::mbar_init(&wbar[1], 1); tc::fence_mbar_init(); }
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tb = tmem_base_s;
    const uint32_t lane_addr = tb + ((uint32_t)(warp * 32) << 16);
    uint32_t phase = 0, wphase = 0u;

    const int ROWS = kTcThreads * nsub;
    const int64_t ntiles = (B + ROWS - 1) / ROWS;
    const float* blocks = packed + NF_STACK_HDR;
    const int NQ = 2 * L;                                         // net blocks per pass, order: layer (direction-aware), net
    auto block_of = [&](int q) { const int li = q >> 1; return (size_t)(2 * (inverse ? L - 1 - li : li) + (q & 1)) * NBW; };

    int buf = 0;
    if (NBUF == 2 && tid == 0 && (int64_t)blockIdx.x < ntiles) {
        tc::mbar_arrive_expect_tx(&wbar[0], (uint32_t)NBW * 4u);
        tc::bulk_g2s(sbuf, blocks + block_of(0), (uint32_t)NBW * 4u, &wbar[0]);
    }
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        for (int s = 0; s < nsub; ++s) {
            const int64_t r = tile * ROWS + s * kTcThreads + tid;
            if constexpr (SAMPLE) {
                draw_row_tc<DM>(sx + s * (DM + 1) * kTcThreads + tid, r, B, D, seed, offset, rng_state ? rng_key : nullptr);
                continue;
            }
#pragma unroll
            for (int d = 0; d < DM; ++d) sx[(s * (DM + 1) + d) * kTcThreads + tid] = (d < D && r < B) ? ld_stream(x + r * D + d) : 0.f;
            sx[(s * (DM + 1) + DM) * kTcThreads + tid] = 0.f;
        }
        for (int q = 0; q < NQ; ++q) {
            const int net = q & 1;
            tc::fence_proxy_async_smem();
            __syncthreads();                                      // everyone is done with the other buffer
            if (tid == 0) {
                if (NBUF == 2) {
                    const bool last = (q == NQ - 1);
                    if (!last || (tile + gridDim.x < ntiles)) {
                        tc::mbar_arrive_expect_tx(&wbar[buf ^ 1], (uint32_t)NBW * 4u);
                        tc::bulk_g2s(sbuf + (size_t)(buf ^ 1) * NBW, blocks + block_of(last ? 0 : q + 1), (uint32_t)NBW * 4u, &wbar[buf ^ 1]);
                    }
                } else {                                          // single buffer: this net's block, now that everyone left the last one
                    tc::mbar_arrive_expect_tx(&wbar[0], (uint32_t)NBW * 4u);
                    tc::bulk_g2s(sbuf, blocks + block_of(q), (uint32_t)NBW * 4u, &wbar[0]);
                }
            }
            tc::mbar_wait(&wbar[buf], (wphase >> buf) & 1u);
            wphase ^= (1u << buf);
            const float* sN = sbuf + (size_t)buf * NBW;
            if (net == 0) {
                if (tid < NF_LAYER_HDR) shdr[tid] = sN[tid];
                __syncthreads();
            }
            const float* nb = sN + NF_LAYER_HDR;
            const LayerHdr lh{shdr};
            const bool bn_on = lh.bn_on();
            const float* mask = lh.mask();
            const uint32_t w2hi = tc::smem_u32(nb + off.w2hi), w2lo = tc::smem_u32(nb + off.w2lo);
            const uint32_t w3hi = tc::smem_u32(nb + off.w3hi), w3lo = tc::smem_u32(nb + off.w3lo);
#pragma unroll 1
            for (int s = 0; s < nsub; ++s) {
                float xv[DM];
                float tot = slab_load<DM>(sx, s, tid, xv);
                if (net == 0 && inverse && bn_on) {
                    nf_stack_bn_between<DM>(lh, D, true, xv, tot);
                    slab_store<DM>(sx, s, tid, xv, tot);
                }
                float xa[DM];
#pragma unroll
                for (int d = 0; d < DM; ++d) xa[d] = (d < D) ? xv[d] * mask[d] : 0.f;
                if constexpr (CM > 0) {
                    const int64_t r = tile * ROWS + s * kTcThreads + tid;     // < 2^31, as ctx_div (the launcher)
                    const uint32_t crow = r < B ? (uint32_t)r / (uint32_t)ctx_div : 0u;
                    layer1_to_tmem<DM, HP, CM>(nb + off.w1k, W1S, xa, lane_addr, nb + off.wc, ctx + (size_t)crow * C, C);
                } else {
                    layer1_to_tmem<DM, HP>(nb + off.w1k, W1S, xa, lane_addr);
                }
                cta_mma_round(warp, &bar, phase, [&] {
                    if (HP == 64) tc::warp_issue_gemm_k64_3xtf32(tb, kColD2, kColAhi, kColAlo, w2hi, w2lo, 64u, &bar);
                    else tc::warp_issue_gemm_krange_3xtf32(tb, kColD2, kColAhi, kColAlo, w2hi, w2lo, (uint32_t)HP, 0, HP / 8, 0u, &bar);
                });
                hidden2_to_tmem<HP>(nb + off.b2, lane_addr);
                cta_mma_round(warp, &bar, phase, [&] {
                    if (HP == 64) tc::warp_issue_gemm_k64_3xtf32(tb, kColD3, kColAhi, kColAlo, w3hi, w3lo, (uint32_t)NO3, &bar);
                    else tc::warp_issue_gemm_krange_3xtf32(tb, kColD3, kColAhi, kColAlo, w3hi, w3lo, (uint32_t)NO3, 0, HP / 8, 0u, &bar);
                });
                uint32_t p[8];
                tc::tmem_ld8(lane_addr + kColD3, p);
                tc::wait_ld();
                float raw[DM];
#pragma unroll
                for (int d = 0; d < DM; ++d) raw[d] = __uint_as_float(p[d]) + nb[off.b3 + d];
                if (net == 0) {
#pragma unroll
                    for (int d = 0; d < DM; ++d) sraw[(s * DM + d) * kTcThreads + tid] = raw[d];
                } else {
                    float lsum = 0.f;
#pragma unroll
                    for (int d = 0; d < DM; ++d) if (d < D) {
                        float out, t;
                        affine_coupling_elem<float>(xv[d], mask[d], sraw[(s * DM + d) * kTcThreads + tid], raw[d], inverse != 0, out, t);
                        xv[d] = scrub0(out);
                        lsum += t;
                    }
                    tot += scrub0(lsum);
                    if (!inverse && bn_on) nf_stack_bn_between<DM>(lh, D, false, xv, tot);
                    slab_store<DM>(sx, s, tid, xv, tot);
                }
            }
            if (NBUF == 2) buf ^= 1;
        }
        for (int s = 0; s < nsub; ++s) {
            const int64_t r = tile * ROWS + s * kTcThreads + tid;
            if (r < B) {
                float zr[DM];
#pragma unroll
                for (int d = 0; d < DM; ++d) zr[d] = sx[(s * (DM + 1) + d) * kTcThreads + tid];
                if (!(flags & NF_STACK_SKIP_Y)) {
#pragma unroll
                    for (int d = 0; d < DM; ++d) if (d < D) st_stream(y + r * D + d, zr[d]);
                }
                const float tot = sx[(s * (DM + 1) + DM) * kTcThreads + tid];
                st_stream(ld + r, SAMPLE ? -tot : (flags & NF_STACK_LOG_PROB_HEAD) ? nf_stack_row_head<DM>(zr, D, tot) : tot);
            }
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc(tb, kTmemCols);
}

template <int DM, int HP, bool SAMPLE = false>
__global__ void __launch_bounds__(kTcThreads, HP == 64 ? 2 : 1)
coupling_stack_tc_kernel(const float* __restrict__ packed, const float* __restrict__ x, float* __restrict__ y,
                         float* __restrict__ ld, int64_t B, int flags, int nsub, uint64_t seed, uint64_t offset,
                         unsigned long long* rng_state) {     // nsub <= kTcSub sub-tiles per weight staging
    coupling_stack_tc_body<DM, HP, SAMPLE, 0>(threadIdx.x, packed, x, y, ld, B, flags, nsub, seed, offset, rng_state, nullptr, 1, 0);
}

// conditional affine coupling stack ('NFD2'): C <= kCtxMax context columns of row r / ctx_div enter the first Linear of
// both conditioner nets of every layer
template <int DM, int HP, bool SAMPLE = false>
__global__ void __launch_bounds__(kTcThreads, HP == 64 ? 2 : 1)
coupling_stack_ctx_tc_kernel(const float* __restrict__ packed, const float* __restrict__ x, float* __restrict__ y,
                             float* __restrict__ ld, int64_t B, int flags, int nsub, uint64_t seed, uint64_t offset,
                             unsigned long long* rng_state, const float* __restrict__ ctx, int64_t ctx_div, int C) {
    coupling_stack_tc_body<DM, HP, SAMPLE, kCtxMax>(threadIdx.x, packed, x, y, ld, B, flags, nsub, seed, offset, rng_state, ctx,
                                                    ctx_div, C);
}

// ------------------------------------------------------------------------------------------------
// MADE / MAF / IAF stack (eval mode, hidden_dim <= 64, data_dim <= 8; masks and eval-mode BatchNorm folded at pack time)
//   One block per layer: lead (80-word layer header) | W1k | b2 | b3 | b4[16] | pad | W2 hi/lo | W3 hi/lo | W4 hi/lo images
//   (73 KB, single buffered: two CTAs per SM keep their 2 x 256 TMEM columns).  The conditioner of made.py:81-140 is
//   in -> H (FP32 pipe, K = data_dim) -> H -> H (two 64 x 64 tensor-core layers through the same TMEM regions) -> 2 D
//   (head, 16 columns: [mu_0.. | alpha_0..]).  PARALLEL modes (MAF.inverse, IAF.forward: masked_autoregressive_flow.py:
//   18-44, inverse_autoregressive_flow.py:30-63): one conditioner pass on the row, then the affine transform of every
//   dim.  SEQUENTIAL modes for data_dim == 2 (MAF.forward, IAF.inverse: :46-78 / :65-103): the reference's loop evaluates
//   MADE twice; on zeros the outputs of dim 0 are exactly its output biases (their masked weight rows are all zero), so
//   dim 0 comes from b4 and the ONE conditioner pass on (out_0, 0) yields dim 1 -- NaN / Inf in out_0 reaches dim 1
//   through the dense layers as in the reference.  Per-layer scrubs and log-det clamps as nf_affine_ar_forward /
//   nf_ar_finish_forward.  The reference's published 6 x MAF(2, 64) / 6 x IAF(2, 64) (plots/_common.py:165-167) are one
//   launch per direction.
// ------------------------------------------------------------------------------------------------
struct MadeBlkOff { int w1k, b2, b3, b4, w2hi, w2lo, w3hi, w3lo, w4hi, w4lo, words; };
__host__ __device__ inline MadeBlkOff made_blk_offsets(int W1S) {
    MadeBlkOff o;
    o.w1k = 0; o.b2 = 64 * W1S; o.b3 = o.b2 + 64; o.b4 = o.b3 + 64;
    o.w2hi = pad256(NF_LAYER_HDR + o.b4 + 16) - NF_LAYER_HDR;
    o.w2lo = o.w2hi + 4096; o.w3hi = o.w2lo + 4096; o.w3lo = o.w3hi + 4096; o.w4hi = o.w3lo + 4096; o.w4lo = o.w4hi + 16 * 64;
    o.words = o.w4lo + 16 * 64;
    return o;
}

template <int DM, bool SAMPLE = false>
__global__ void __launch_bounds__(kTcThreads, 2)
made_stack_tc_kernel(const float* __restrict__ packed, const float* __restrict__ x, float* __restrict__ y,
                     float* __restrict__ ld, int64_t B, int flags, int nsub, int mode, uint64_t seed, uint64_t offset,
                     unsigned long long* rng_state) {
    const int inverse = flags & NF_STACK_INVERSE;
    extern __shared__ __align__(1024) float sbuf[];
    const StackHdr hd = nf_stack_hdr_device(packed);
    const int D = hd.D, L = hd.L, W1S = hd.W1S, NBW = hd.layer_stride;
    float* sx = sbuf + (size_t)NBW;                              // [kTcSub][DM+1][128] row state
    uint64_t* bars = reinterpret_cast<uint64_t*>(sx + kTcSub * (DM + 1) * kTcThreads);
    uint64_t& bar = bars[0];
    uint64_t& wbar = bars[1];
    uint32_t& tmem_base_s = *reinterpret_cast<uint32_t*>(bars + 2);
    const MadeBlkOff off = made_blk_offsets(W1S);
    const bool sequential = (mode == AR_MAF_FWD || mode == AR_IAF_INV);
    const bool iaf = (mode == AR_IAF_FWD || mode == AR_IAF_INV);
    const float lim = iaf ? 50.f : 100.f;

    const int tid = threadIdx.x, warp = tid >> 5;
    if (warp == 0) tc::tmem_alloc(&tmem_base_s, kTmemCols);
    unsigned long long* rng_key = reinterpret_cast<unsigned long long*>(bars + 3);   // SAMPLE + device state: every
    if constexpr (SAMPLE) if (rng_state) nf_rng_state_take(rng_state, rng_key);   // CTA, before the role split / tiles
    if (tid == 0) { tc::mbar_init(&bar, 1); tc::mbar_init(&wbar, 1); tc::fence_mbar_init(); }
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tb = tmem_base_s;
    const uint32_t lane_addr = tb + ((uint32_t)(warp * 32) << 16);
    uint32_t phase = 0, wphase = 0u;

    const int ROWS = kTcThreads * nsub;
    const int64_t ntiles = (B + ROWS - 1) / ROWS;
    const float* blocks = packed + NF_STACK_HDR;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        for (int s = 0; s < nsub; ++s) {
            const int64_t r = tile * ROWS + s * kTcThreads + tid;
            if constexpr (SAMPLE) {
                draw_row_tc<DM>(sx + s * (DM + 1) * kTcThreads + tid, r, B, D, seed, offset, rng_state ? rng_key : nullptr);
                continue;
            }
#pragma unroll
            for (int d = 0; d < DM; ++d) sx[(s * (DM + 1) + d) * kTcThreads + tid] = (d < D && r < B) ? ld_stream(x + r * D + d) : 0.f;
            sx[(s * (DM + 1) + DM) * kTcThreads + tid] = 0.f;
        }
        for (int li = 0; li < L; ++li) {
            const int layer = inverse ? L - 1 - li : li;
            tc::fence_proxy_async_smem();
            __syncthreads();                                      // everyone is done with the previous layer's block
            if (tid == 0) {
                tc::mbar_arrive_expect_tx(&wbar, (uint32_t)NBW * 4u);
                tc::bulk_g2s(sbuf, blocks + (size_t)layer * NBW, (uint32_t)NBW * 4u, &wbar);
            }
            tc::mbar_wait(&wbar, wphase); wphase ^= 1u;
            const LayerHdr lh{sbuf};
            const float* nb = sbuf + NF_LAYER_HDR;
            const bool bn_on = lh.bn_on();
            const uint32_t w2hi = tc::smem_u32(nb + off.w2hi), w2lo = tc::smem_u32(nb + off.w2lo);
            const uint32_t w3hi = tc::smem_u32(nb + off.w3hi), w3lo = tc::smem_u32(nb + off.w3lo);
            const uint32_t w4hi = tc::smem_u32(nb + off.w4hi), w4lo = tc::smem_u32(nb + off.w4lo);
            const float* b4 = nb + off.b4;
#pragma unroll 1
            for (int s = 0; s < nsub; ++s) {
                float xv[DM];
                float tot = slab_load<DM>(sx, s, tid, xv);
                if (inverse && bn_on) nf_stack_bn_between<DM>(lh, D, true, xv, tot);
                // conditioner input: the row itself (parallel), or (out_0, 0) with out_0 from the output biases (sequential, D == 2)
                float xa[DM], c0 = 0.f, t0 = 0.f;
#pragma unroll
                for (int d = 0; d < DM; ++d) xa[d] = (d < D) ? xv[d] : 0.f;
                if (sequential) {
                    affine_ar_elem<float>(mode, xv[0], b4[0], b4[D], c0, t0);
#pragma unroll
                    for (int d = 0; d < DM; ++d) xa[d] = 0.f;
                    xa[0] = c0;
                }
                layer1_to_tmem<DM, 64>(nb + off.w1k, W1S, xa, lane_addr);
                cta_mma_round(warp, &bar, phase, [&] { tc::warp_issue_gemm_k64_3xtf32(tb, kColD2, kColAhi, kColAlo, w2hi, w2lo, 64u, &bar); });
                hidden2_to_tmem<64>(nb + off.b2, lane_addr);
                cta_mma_round(warp, &bar, phase, [&] { tc::warp_issue_gemm_k64_3xtf32(tb, kColD2, kColAhi, kColAlo, w3hi, w3lo, 64u, &bar); });
                hidden2_to_tmem<64>(nb + off.b3, lane_addr);
                cta_mma_round(warp, &bar, phase, [&] { tc::warp_issue_gemm_k64_3xtf32(tb, kColD3, kColAhi, kColAlo, w4hi, w4lo, 16u, &bar); });
                uint32_t p[16];
                tc::tmem_ld16(lane_addr + kColD3, p);
                tc::wait_ld();
                tc::fence_before_sync();                          // D3 / A reads precede the next sub-tile's writes
                float lsum = 0.f;
                if (!sequential) {
#pragma unroll
                    for (int d = 0; d < DM; ++d) if (d < D) {
                        float mu = 0.f, al = 0.f;
#pragma unroll
                        for (int q = 0; q < 16; ++q) { if (q == d) mu = __uint_as_float(p[q]) + b4[q]; if (q == D + d) al = __uint_as_float(p[q]) + b4[q]; }
                        float o, t;
                        affine_ar_elem<float>(mode, xv[d], mu, al, o, t);
                        if (!is_finite(o)) o = iaf ? xv[d] : 0.f;
                        xv[d] = o;
                        lsum += t;
                    }
                } else {
                    float mu = 0.f, al = 0.f;
#pragma unroll
                    for (int q = 0; q < 16; ++q) { if (q == 1) mu = __uint_as_float(p[q]) + b4[q]; if (q == D + 1) al = __uint_as_float(p[q]) + b4[q]; }
                    float c1, t1;
                    affine_ar_elem<float>(mode, xv[1], mu, al, c1, t1);
                    lsum = t0 + t1;
                    xv[0] = is_finite(c0) ? c0 : (iaf ? xv[0] : 0.f);
                    xv[1] = is_finite(c1) ? c1 : (iaf ? xv[1] : 0.f);
                }
                tot += clamp_mm(scrub0(lsum), -lim, lim);
                if (!inverse && bn_on) nf_stack_bn_between<DM>(lh, D, false, xv, tot);
                slab_store<DM>(sx, s, tid, xv, tot);
            }
        }
        for (int s = 0; s < nsub; ++s) {
            const int64_t r = tile * ROWS + s * kTcThreads + tid;
            if (r < B) {
                float zr[DM];
#pragma unroll
                for (int d = 0; d < DM; ++d) zr[d] = sx[(s * (DM + 1) + d) * kTcThreads + tid];
                if (!(flags & NF_STACK_SKIP_Y)) {
#pragma unroll
                    for (int d = 0; d < DM; ++d) if (d < D) st_stream(y + r * D + d, zr[d]);
                }
                const float tot = sx[(s * (DM + 1) + DM) * kTcThreads + tid];
                st_stream(ld + r, SAMPLE ? -tot : (flags & NF_STACK_LOG_PROB_HEAD) ? nf_stack_row_head<DM>(zr, D, tot) : tot);
            }
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc(tb, kTmemCols);
}

// CTAs per SM that shared memory (1 KB reserved per CTA) and the SM's 512 TMEM columns allow, times the SMs; 0: none fits
static int64_t tc_resident_ctas(size_t smem, int tmem_cols) {
    int per_sm = (int)((227 * 1024) / (smem + 1024));
    if (per_sm > 512 / tmem_cols) per_sm = 512 / tmem_cols;
    return (int64_t)kNumSMs * per_sm;
}

// small batches: fewer sub-tiles per weight staging so that every SM gets rows (4 000 rows on eight 512-row tiles left
// 140 SMs idle); from kTcSub sub-tiles per resident CTA on, the staging is shared by kTcSub sub-tiles
static int tc_nsub(int64_t B, int64_t res_ctas) {
    const int nsub = (int)cdiv(cdiv(B, kTcThreads), res_ctas);
    return nsub < 1 ? 1 : (nsub > kTcSub ? kTcSub : nsub);
}

// CTX: the conditional layout ('NFC2'; header word 3 = context width C) and spline_stack_ctx_tc2_kernel
template <bool CTX>
static int spline_stack_tc_launch(const StackCall& c, const StackHdr& h) {
    const int D = h.D, K = h.K, W1S = h.W1S, NO3 = h.NO, BW = h.layer_stride;
    if (CTX) {
        if (c.cx.ctx == nullptr) return NF_ERR_NULL;
        if (c.cx.div < 1 || c.cx.rows < cdiv(c.B, c.cx.div)) return NF_ERR_BAD_SHAPE;
        if (h.HP < 1 || h.HP > kCtxMax) return NF_ERR_UNSUPPORTED;
        if (c.B > 0x7FFFFFFF || c.cx.div > 0x7FFFFFFF) return NF_ERR_UNSUPPORTED;     // 32-bit row / context-row indices
    }
    if (D < 1 || D > NF_STACK_DMAX || h.H < 1 || h.H > 64 || h.L < 1 || K < 2 || K > 10) return NF_ERR_UNSUPPORTED;
    if (NO3 != 32 && NO3 != 64) return NF_ERR_UNSUPPORTED;
    if (W1S != nf_stack_w1s(D) || BW != NF_LAYER_HDR + blk_offsets(W1S, NO3, 64, CTX ? kCtxMax : 0).net_words)
        return NF_ERR_BAD_SHAPE;
    if (!c.holds(NF_STACK_HDR + (int64_t)h.L * BW)) return NF_ERR_WORKSPACE;
    const int DMh = D <= 2 ? 2 : (D <= 3 ? 4 : 8);
    const size_t smem = sizeof(float) * ((size_t)2 * BW + (size_t)kTcSub * (DMh + 1) * kTcThreads + 12 + (c.rng_state ? 4 : 0));
    if (smem > 227 * 1024) return NF_ERR_UNSUPPORTED;
    const int64_t ntiles = cdiv(c.B, kTcThreads * kTcSub);
    const int64_t cap = tc_resident_ctas(smem, kTmemCols);
    if (cap < 1) return NF_ERR_UNSUPPORTED;
    const int grid = (int)(ntiles < cap ? ntiles : cap);
#define NF_TC(DMv, KMv, KSv)                                                                                         \
    do {                                                                                                             \
        if constexpr (CTX) {                                                                                         \
            auto kern = c.sample ? spline_stack_ctx_tc2_kernel<DMv, KMv, KSv, true>                                  \
                                 : spline_stack_ctx_tc2_kernel<DMv, KMv, KSv>;                                       \
            const int rc = stack_smem_attributes(kern, smem);                                                        \
            if (rc != NF_OK) return rc;                                                                              \
            kern<<<grid, kTc2Threads, smem, c.st>>>((const float*)c.packed, (const float*)c.x, (float*)c.y,          \
                                                    (float*)c.ld, c.B, c.flags, c.seed, c.offset, c.rng_state,       \
                                                    (const float*)c.cx.ctx, c.cx.div, h.HP);                         \
        } else {                                                                                                     \
            auto kern = c.sample ? spline_stack_tc2_kernel<DMv, KMv, KSv, true> : spline_stack_tc2_kernel<DMv, KMv, KSv>; \
            const int rc = stack_smem_attributes(kern, smem);                                                        \
            if (rc != NF_OK) return rc;                                                                              \
            kern<<<grid, kTc2Threads, smem, c.st>>>((const float*)c.packed, (const float*)c.x, (float*)c.y,          \
                                                    (float*)c.ld, c.B, c.flags, c.seed, c.offset, c.rng_state);      \
        }                                                                                                            \
    } while (0)
#define NF_TC_K(DMv)                                      \
    do {                                                  \
        if (K == 8) NF_TC(DMv, 8, 8);                     \
        else if (K == 10) NF_TC(DMv, 10, 10);             \
        else if (K < 8) NF_TC(DMv, 8, 0);                 \
        else NF_TC(DMv, 10, 0);                           \
    } while (0)
    if (D <= 2) NF_TC_K(2);
    else if (D <= 3) NF_TC_K(4);
    else NF_TC_K(8);
#undef NF_TC_K
#undef NF_TC
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

// CTX: the conditional layout ('NFD2'; header word 3 = context width C) and coupling_stack_ctx_tc_kernel, with the
// refusals of spline_stack_tc_launch<true>
template <bool CTX>
static int coupling_stack_tc_launch(const StackCall& c, const StackHdr& h) {
    const int D = h.D, H = h.H, W1S = h.W1S, NO3 = h.NO, NBW = h.layer_stride;
    if (CTX) {
        if (c.cx.ctx == nullptr) return NF_ERR_NULL;
        if (c.cx.div < 1 || c.cx.rows < cdiv(c.B, c.cx.div)) return NF_ERR_BAD_SHAPE;
        if (h.HP < 1 || h.HP > kCtxMax) return NF_ERR_UNSUPPORTED;
        if (c.B > 0x7FFFFFFF || c.cx.div > 0x7FFFFFFF) return NF_ERR_UNSUPPORTED;     // 32-bit row / context-row indices
    }
    if (D < 1 || D > NF_STACK_DMAX || H < 1 || H > 128 || h.L < 1 || NO3 != 16) return NF_ERR_UNSUPPORTED;
    const int HP = H <= 64 ? 64 : 128;
    if (W1S != nf_stack_w1s(D) || NBW != NF_LAYER_HDR + blk_offsets(W1S, NO3, HP, CTX ? kCtxMax : 0).net_words)
        return NF_ERR_BAD_SHAPE;
    if (!c.holds(NF_STACK_HDR + (int64_t)2 * h.L * NBW)) return NF_ERR_WORKSPACE;
    const int DMh = D <= 2 ? 2 : (D <= 3 ? 4 : 8);
    const int nbuf = HP == 64 ? 2 : 1, tmem_cols = HP == 64 ? 256 : 512;
    const size_t smem = sizeof(float) * ((size_t)nbuf * NBW + (size_t)kTcSub * (2 * DMh + 1) * kTcThreads + NF_LAYER_HDR + 8 +
                                         (c.rng_state ? 4 : 0));
    if (smem > 227 * 1024) return NF_ERR_UNSUPPORTED;
    const int nsub = tc_nsub(c.B, kNumSMs * (512 / tmem_cols));
    const int64_t ntiles = cdiv(c.B, kTcThreads * nsub);
    const int64_t cap = tc_resident_ctas(smem, tmem_cols);
    if (cap < 1) return NF_ERR_UNSUPPORTED;
    const int grid = (int)(ntiles < cap ? ntiles : cap);
#define NF_CTC(DMv, HPv)                                                                                              \
    do {                                                                                                             \
        if constexpr (CTX) {                                                                                         \
            auto kern = c.sample ? coupling_stack_ctx_tc_kernel<DMv, HPv, true> : coupling_stack_ctx_tc_kernel<DMv, HPv>; \
            const int rc = stack_smem_attributes(kern, smem);                                                        \
            if (rc != NF_OK) return rc;                                                                              \
            kern<<<grid, kTcThreads, smem, c.st>>>((const float*)c.packed, (const float*)c.x, (float*)c.y,           \
                                                   (float*)c.ld, c.B, c.flags, nsub, c.seed, c.offset, c.rng_state,  \
                                                   (const float*)c.cx.ctx, c.cx.div, h.HP);                          \
        } else {                                                                                                     \
            auto kern = c.sample ? coupling_stack_tc_kernel<DMv, HPv, true> : coupling_stack_tc_kernel<DMv, HPv>;      \
            const int rc = stack_smem_attributes(kern, smem);                                                        \
            if (rc != NF_OK) return rc;                                                                              \
            kern<<<grid, kTcThreads, smem, c.st>>>((const float*)c.packed, (const float*)c.x, (float*)c.y,           \
                                                   (float*)c.ld, c.B, c.flags, nsub, c.seed, c.offset, c.rng_state); \
        }                                                                                                            \
    } while (0)
    if (HP == 64) { if (D <= 2) NF_CTC(2, 64); else if (D <= 3) NF_CTC(4, 64); else NF_CTC(8, 64); }
    else          { if (D <= 2) NF_CTC(2, 128); else if (D <= 3) NF_CTC(4, 128); else NF_CTC(8, 128); }
#undef NF_CTC
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

static int made_stack_tc_launch(const StackCall& c, const StackHdr& h) {
    const int D = h.D, W1S = h.W1S, NBW = h.layer_stride, mode = c.mode;
    if (D < 1 || D > NF_STACK_DMAX || h.H < 1 || h.H > 64 || h.L < 1) return NF_ERR_UNSUPPORTED;
    if (mode < NF_AR_MAF_INVERSE || mode > NF_AR_IAF_INVERSE) return NF_ERR_UNSUPPORTED;
    if ((mode == NF_AR_MAF_FORWARD || mode == NF_AR_IAF_INVERSE) && D != 2) return NF_ERR_UNSUPPORTED;   // sequential: 2-D only
    if (W1S != nf_stack_w1s(D) || NBW != NF_LAYER_HDR + made_blk_offsets(W1S).words) return NF_ERR_BAD_SHAPE;
    if (!c.holds(NF_STACK_HDR + (int64_t)h.L * NBW)) return NF_ERR_WORKSPACE;
    const int DMh = D <= 2 ? 2 : (D <= 3 ? 4 : 8);
    const size_t smem = sizeof(float) * ((size_t)NBW + (size_t)kTcSub * (DMh + 1) * kTcThreads + 8 + (c.rng_state ? 4 : 0));
    if (smem > 113 * 1024) return NF_ERR_UNSUPPORTED;             // two CTAs per SM
    const int res_ctas = kNumSMs * 2;
    const int nsub = tc_nsub(c.B, res_ctas);
    const int64_t ntiles = cdiv(c.B, kTcThreads * nsub);
    const int grid = (int)(ntiles < res_ctas ? ntiles : res_ctas);
#define NF_MTC(DMv)                                                                                                  \
    do {                                                                                                             \
        auto kern = c.sample ? made_stack_tc_kernel<DMv, true> : made_stack_tc_kernel<DMv>;                          \
        const int rc = stack_smem_attributes(kern, smem);                                                            \
        if (rc != NF_OK) return rc;                                                                                  \
        kern<<<grid, kTcThreads, smem, c.st>>>((const float*)c.packed, (const float*)c.x, (float*)c.y, (float*)c.ld,  \
                                               c.B, c.flags, nsub, mode, c.seed, c.offset, c.rng_state);             \
    } while (0)
    if (D <= 2) NF_MTC(2); else if (D <= 3) NF_MTC(4); else NF_MTC(8);
#undef NF_MTC
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

static const StackFamily kSplineTc = {NF_STACK_MAGIC_SPLINE_TC, spline_stack_tc_launch<false>};
static const StackFamily kSplineCtxTc = {NF_STACK_MAGIC_SPLINE_CTX_TC, spline_stack_tc_launch<true>};
static const StackFamily kCouplingTc = {NF_STACK_MAGIC_AFFINE_TC, coupling_stack_tc_launch<false>};
static const StackFamily kCouplingCtxTc = {NF_STACK_MAGIC_AFFINE_CTX_TC, coupling_stack_tc_launch<true>};
static const StackFamily kMadeTc = {NF_STACK_MAGIC_MADE_TC, made_stack_tc_launch};

}  // namespace nf

using namespace nf;

extern "C" int64_t nf_spline_stack_tc_block_words(int D, int K, int max_dt) {
    if (D < 1 || D > NF_STACK_DMAX || K < 2 || K > 10 || max_dt < 1 || max_dt > 2) return -1;
    const int W1S = nf_stack_w1s(D), NO3 = 32 * max_dt;
    return NF_LAYER_HDR + blk_offsets(W1S, NO3).net_words;
}

extern "C" int nf_spline_stack_tc_forward(const void* packed, const void* hdr_host, int64_t packed_bytes, const void* x,
                                          void* y, void* ld, int64_t B, int inverse, nf_stream_t stream) {
    return stack_forward(kSplineTc, packed, hdr_host, packed_bytes, x, y, ld, B, inverse, 0, stream);
}

extern "C" int nf_spline_stack_tc_sample(const void* packed, const void* hdr_host, int64_t packed_bytes, uint64_t seed,
                                         uint64_t offset, void* x, void* log_q, int64_t B, nf_stream_t stream) {
    return stack_sample(kSplineTc, packed, hdr_host, packed_bytes, 0, seed, offset, x, log_q, B, stream);
}

extern "C" int nf_spline_stack_tc_sample_state(const void* packed, const void* hdr_host, int64_t packed_bytes,
                                               void* rng_state, void* x, void* log_q, int64_t B, nf_stream_t stream) {
    return stack_sample_state(kSplineTc, packed, hdr_host, packed_bytes, 0, rng_state, x, log_q, B, stream);
}

extern "C" int nf_spline_stack_ctx_tc_forward(const void* packed, const void* hdr_host, int64_t packed_bytes, const void* x,
                                              const void* context, int64_t ctx_rows, int64_t ctx_div, void* y, void* ld,
                                              int64_t B, int flags, nf_stream_t stream) {
    return stack_forward(kSplineCtxTc, packed, hdr_host, packed_bytes, x, y, ld, B, flags, 0, stream,
                         {context, ctx_rows, ctx_div});
}

extern "C" int nf_spline_stack_ctx_tc_sample(const void* packed, const void* hdr_host, int64_t packed_bytes,
                                             const void* context, int64_t ctx_rows, int64_t ctx_div, uint64_t seed,
                                             uint64_t offset, void* x, void* log_q, int64_t B, nf_stream_t stream) {
    return stack_sample(kSplineCtxTc, packed, hdr_host, packed_bytes, 0, seed, offset, x, log_q, B, stream,
                        {context, ctx_rows, ctx_div});
}

extern "C" int nf_spline_stack_ctx_tc_sample_state(const void* packed, const void* hdr_host, int64_t packed_bytes,
                                                   const void* context, int64_t ctx_rows, int64_t ctx_div, void* rng_state,
                                                   void* x, void* log_q, int64_t B, nf_stream_t stream) {
    return stack_sample_state(kSplineCtxTc, packed, hdr_host, packed_bytes, 0, rng_state, x, log_q, B, stream,
                              {context, ctx_rows, ctx_div});
}

extern "C" int64_t nf_coupling_stack_tc_block_words(int D) {
    if (D < 1 || D > NF_STACK_DMAX) return -1;
    return NF_LAYER_HDR + blk_offsets(nf_stack_w1s(D), 16).net_words;      // words per NET block (2 per layer)
}
extern "C" int64_t nf_coupling_stack_tc_block_words_hidden(int D, int H) {  // hidden units padded to 64 or 128
    if (D < 1 || D > NF_STACK_DMAX || H < 1 || H > 128) return -1;
    return NF_LAYER_HDR + blk_offsets(nf_stack_w1s(D), 16, H <= 64 ? 64 : 128).net_words;
}

extern "C" int nf_coupling_stack_tc_forward(const void* packed, const void* hdr_host, int64_t packed_bytes, const void* x,
                                            void* y, void* ld, int64_t B, int inverse, nf_stream_t stream) {
    return stack_forward(kCouplingTc, packed, hdr_host, packed_bytes, x, y, ld, B, inverse, 0, stream);
}

extern "C" int nf_coupling_stack_tc_sample(const void* packed, const void* hdr_host, int64_t packed_bytes, uint64_t seed,
                                           uint64_t offset, void* x, void* log_q, int64_t B, nf_stream_t stream) {
    return stack_sample(kCouplingTc, packed, hdr_host, packed_bytes, 0, seed, offset, x, log_q, B, stream);
}

extern "C" int nf_coupling_stack_tc_sample_state(const void* packed, const void* hdr_host, int64_t packed_bytes,
                                                 void* rng_state, void* x, void* log_q, int64_t B, nf_stream_t stream) {
    return stack_sample_state(kCouplingTc, packed, hdr_host, packed_bytes, 0, rng_state, x, log_q, B, stream);
}

extern "C" int64_t nf_coupling_stack_ctx_tc_block_words_hidden(int D, int H) {   // 'NFD2': with the Wc section
    if (D < 1 || D > NF_STACK_DMAX || H < 1 || H > 128) return -1;
    return NF_LAYER_HDR + blk_offsets(nf_stack_w1s(D), 16, H <= 64 ? 64 : 128, kCtxMax).net_words;
}

extern "C" int nf_coupling_stack_ctx_tc_forward(const void* packed, const void* hdr_host, int64_t packed_bytes, const void* x,
                                                const void* context, int64_t ctx_rows, int64_t ctx_div, void* y, void* ld,
                                                int64_t B, int flags, nf_stream_t stream) {
    return stack_forward(kCouplingCtxTc, packed, hdr_host, packed_bytes, x, y, ld, B, flags, 0, stream,
                         {context, ctx_rows, ctx_div});
}

extern "C" int nf_coupling_stack_ctx_tc_sample(const void* packed, const void* hdr_host, int64_t packed_bytes,
                                               const void* context, int64_t ctx_rows, int64_t ctx_div, uint64_t seed,
                                               uint64_t offset, void* x, void* log_q, int64_t B, nf_stream_t stream) {
    return stack_sample(kCouplingCtxTc, packed, hdr_host, packed_bytes, 0, seed, offset, x, log_q, B, stream,
                        {context, ctx_rows, ctx_div});
}

extern "C" int nf_coupling_stack_ctx_tc_sample_state(const void* packed, const void* hdr_host, int64_t packed_bytes,
                                                     const void* context, int64_t ctx_rows, int64_t ctx_div, void* rng_state,
                                                     void* x, void* log_q, int64_t B, nf_stream_t stream) {
    return stack_sample_state(kCouplingCtxTc, packed, hdr_host, packed_bytes, 0, rng_state, x, log_q, B, stream,
                              {context, ctx_rows, ctx_div});
}

extern "C" int64_t nf_made_stack_tc_block_words(int D) {
    if (D < 1 || D > NF_STACK_DMAX) return -1;
    return NF_LAYER_HDR + made_blk_offsets(nf_stack_w1s(D)).words;           // words per layer block
}

extern "C" int nf_made_stack_tc_forward(const void* packed, const void* hdr_host, int64_t packed_bytes, const void* x,
                                        void* y, void* ld, int64_t B, int flags, int mode, nf_stream_t stream) {
    return stack_forward(kMadeTc, packed, hdr_host, packed_bytes, x, y, ld, B, flags, mode, stream);
}

// the sampling directions only: IAF.forward (parallel) and MAF.forward (sequential, data_dim 2)
static bool made_samples(int mode) { return mode == NF_AR_IAF_FORWARD || mode == NF_AR_MAF_FORWARD; }

extern "C" int nf_made_stack_tc_sample(const void* packed, const void* hdr_host, int64_t packed_bytes, int mode, uint64_t seed,
                                       uint64_t offset, void* x, void* log_q, int64_t B, nf_stream_t stream) {
    if (!made_samples(mode)) return NF_ERR_UNSUPPORTED;
    return stack_sample(kMadeTc, packed, hdr_host, packed_bytes, mode, seed, offset, x, log_q, B, stream);
}

extern "C" int nf_made_stack_tc_sample_state(const void* packed, const void* hdr_host, int64_t packed_bytes, int mode,
                                             void* rng_state, void* x, void* log_q, int64_t B, nf_stream_t stream) {
    if (!made_samples(mode)) return NF_ERR_UNSUPPORTED;
    return stack_sample_state(kMadeTc, packed, hdr_host, packed_bytes, mode, rng_state, x, log_q, B, stream);
}
