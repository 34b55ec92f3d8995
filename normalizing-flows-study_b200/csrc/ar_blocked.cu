// ar_blocked.cu -- sequential directions of the affine autoregressive flows (MAF.forward / IAF.inverse,
// masked_autoregressive_flow.py:46-78 / inverse_autoregressive_flow.py:65-103) as a *blocked* triangular evaluation.
//
// The reference re-evaluates the whole MADE D times (D x 4 dense GEMMs).  Hidden units sorted by degree make every
// masked weight block-lower-triangular, so the D dependent steps are grouped into blocks of `gb` consecutive degrees:
//   * contributions of all PREVIOUS blocks to the block's pre-activations are plain dense products over the whole
//     batch -> nf_linear_tc (tcgen05, 3xTF32, TMA) on column slices of the activation buffers:
//         pre_l[:, blk] = act_{l-1}[:, :u0] * W_l[blk, :u0]^T        (l = 1..3),   preo[:, dims] = act3[:, :u0] * W3[dims, :u0]^T
//   * the IN-BLOCK part (gb dependent steps over <= ~72 units per layer) runs in ar_block_mma_kernel (third version, below:
//     the steps as register-level mma.sync m16n8k8 3xTF32 products, a warp owns 16 rows for the whole block, no CTA
//     barrier); ar_block_warp_kernel is the second version (FP32 pipe, a warp owns 32 rows), the fallback where the unit
//     layout does not give whole 8-unit tiles per degree; ar_block_kernel is the first version (32 rows per CTA, four
//     __syncthreads per degree), kept for blocks whose weights do not fit in shared memory.
// Every hidden unit is still evaluated exactly once (total work = one masked MADE pass), ~75 % of it on the tensor pipe.
#include "nf_common.cuh"

extern "C" int nf_linear_tc(const void*, const void*, const void*, const void*, void*, int64_t, int64_t, int64_t, int64_t,
                            int64_t, int64_t, int, const int32_t*, nf_stream_t);
extern "C" int nf_ar_finish_forward(const void*, const void*, const void*, void*, void*, int64_t, int, int, int, nf_stream_t);

namespace nf {

int gemm_tc2_launch(const void* x, const void* w_hi, const void* w_lo, const void* bias, void* y, int64_t M, int64_t N, int64_t K,
                    int64_t ldx, int64_t ldw, int64_t ldy, int relu, const int32_t* k_begin, const int32_t* k_extent,
                    cudaStream_t st, int accumulate);

// Y[M,N] (+)= X[M,K] W[N,K]^T for K <= 128 through the persistent direct-epilogue kernel of gemm_tc2.cu
static int linear_tc_push(const float* x, const float* w_hi, const float* w_lo, float* y, int64_t M, int64_t N, int64_t K,
                          int64_t ldx, int64_t ldw, int64_t ldy, int accumulate, cudaStream_t st) {
    if (!aligned16(x) || !aligned16(w_hi) || !aligned16(w_lo) || (ldx % 4) != 0 || (ldw % 4) != 0) return NF_ERR_UNSUPPORTED;
    const int rc = gemm_tc2_launch(x, w_hi, w_lo, nullptr, y, M, N, K, ldx, ldw, ldy, 0, nullptr, nullptr, st, accumulate);
    if (rc != NF_OK) return rc;
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

constexpr int kBlkRows = 32;
constexpr int kBlkWarps = 4;
constexpr int kBlkPad = 33;          // [unit][row] tiles padded to 33 rows: conflict-free transposed fills and lane reads

// dot over v in [0,n) of w[v] * act[v][lane]; w warp-uniform (global, read-only path), act [*][kBlkPad] in shared memory
__device__ __forceinline__ float dot_tile(const float* __restrict__ w, const float* __restrict__ act, int n, int lane) {
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    int v = 0;
    for (; v + 4 <= n; v += 4) {
        s0 = fmaf(__ldg(w + v + 0), act[(v + 0) * kBlkPad + lane], s0);
        s1 = fmaf(__ldg(w + v + 1), act[(v + 1) * kBlkPad + lane], s1);
        s2 = fmaf(__ldg(w + v + 2), act[(v + 2) * kBlkPad + lane], s2);
        s3 = fmaf(__ldg(w + v + 3), act[(v + 3) * kBlkPad + lane], s3);
    }
    for (; v < n; ++v) s0 = fmaf(__ldg(w + v), act[v * kBlkPad + lane], s0);
    return (s0 + s1) + (s2 + s3);
}

// coalesced [rows x n] slice of a row-major [B, ld] array -> transposed shared tile [n][kBlkPad] (zeros when src == nullptr)
__device__ __forceinline__ void fill_tile(float* tile, const float* __restrict__ src, int64_t r0, int nrow, int ld, int c0, int n) {
    for (int i = threadIdx.x; i < kBlkRows * n; i += blockDim.x) {
        const int r = i / n, c = i - r * n;
        tile[c * kBlkPad + r] = (src && r < nrow) ? src[(r0 + r) * ld + c0 + c] : 0.f;
    }
}
__device__ __forceinline__ void drain_tile(const float* tile, float* __restrict__ dst, int64_t r0, int nrow, int ld, int c0, int n) {
    for (int i = threadIdx.x; i < nrow * n; i += blockDim.x) {
        const int r = i / n, c = i - r * n;
        dst[(r0 + r) * ld + c0 + c] = tile[c * kBlkPad + r];
    }
}

// dims [g0,g1), hidden units [u0,u1) (= degrees g0..g1-1).  pre*/preo: partial sums from previous blocks (nullptr for
// the first block).  xcur: outputs so far, unscrubbed (NaN/Inf must keep poisoning later dims like the dense reference).
__global__ void __launch_bounds__(kBlkRows * kBlkWarps)
ar_block_kernel(const float* __restrict__ vin, float* __restrict__ xcur, const float* __restrict__ pre1,
                const float* __restrict__ pre2, const float* __restrict__ pre3, const float* __restrict__ preo,
                float* __restrict__ act1, float* __restrict__ act2, float* __restrict__ act3,
                const float* __restrict__ w0, const float* __restrict__ b0, const float* __restrict__ w1,
                const float* __restrict__ b1, const float* __restrict__ w2, const float* __restrict__ b2,
                const float* __restrict__ w3, const float* __restrict__ b3, const int32_t* __restrict__ gstart,
                float* __restrict__ ldacc, int* __restrict__ bad, int64_t B, int D, int H, int g0, int g1, int u0, int u1,
                int mode) {
    extern __shared__ __align__(16) float sm[];
    const int nd = g1 - g0, nu = u1 - u0;
    float* sx = sm;                              // [nd][pad] inputs of the block's dims, replaced by outputs
    float* a1 = sx + nd * kBlkPad;               // [nu][pad] layer-1 pre-activation partials -> activations
    float* a2 = a1 + nu * kBlkPad;
    float* a3 = a2 + nu * kBlkPad;
    float* sld = a3 + nu * kBlkPad;              // [32] running log-det
    int* sbad = reinterpret_cast<int*>(sld + kBlkRows);   // [32] poison flag
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t r0 = (int64_t)blockIdx.x * kBlkRows;
    const int nrow = (int)((B - r0) < kBlkRows ? (B - r0) : kBlkRows);
    const bool first = (g0 == 0);

    fill_tile(sx, vin, r0, nrow, D, g0, nd);
    fill_tile(a1, pre1, r0, nrow, H, u0, nu);
    fill_tile(a2, pre2, r0, nrow, H, u0, nu);
    fill_tile(a3, pre3, r0, nrow, H, u0, nu);
    if (threadIdx.x < kBlkRows) {
        const bool ok = threadIdx.x < nrow;
        sld[threadIdx.x] = (!first && ok) ? ldacc[r0 + threadIdx.x] : 0.f;
        sbad[threadIdx.x] = (!first && ok) ? bad[r0 + threadIdx.x] : 0;
    }
    __syncthreads();

    for (int g = g0; g < g1; ++g) {
        const int ub0 = gstart[g] - u0, ub1 = gstart[g + 1] - u0;     // in-block units of degree g
        // (A) parameters of dim g: previous blocks (preo) + in-block layer-3 units of degree < g
        if (warp == 0) {
            float mu = __ldg(b3 + g) + dot_tile(w3 + (size_t)g * H + u0, a3, ub0, lane);
            float al = __ldg(b3 + D + g) + dot_tile(w3 + (size_t)(D + g) * H + u0, a3, ub0, lane);
            if (preo && lane < nrow) { mu += preo[(r0 + lane) * 2 * D + 2 * g]; al += preo[(r0 + lane) * 2 * D + 2 * g + 1]; }
            float o, t;
            affine_ar_elem<float>(mode, sx[(g - g0) * kBlkPad + lane], mu, al, o, t);
            if (sbad[lane]) { o = __int_as_float(0x7fc00000); t = o; }
            if (!is_finite(o)) sbad[lane] = 1;      // 0*NaN of the dense reference poisons every later dim
            sx[(g - g0) * kBlkPad + lane] = o;
            sld[lane] += t;
        }
        __syncthreads();
        if (g == D - 1) break;
        // (B) hidden units of degree g, layer by layer
        for (int u = ub0 + warp; u < ub1; u += kBlkWarps) {
            float s = a1[u * kBlkPad + lane] + __ldg(b0 + u0 + u);
            s += dot_tile(w0 + (size_t)(u0 + u) * D + g0, sx, g - g0 + 1, lane);
            a1[u * kBlkPad + lane] = relu_nan(s);
        }
        __syncthreads();
        for (int u = ub0 + warp; u < ub1; u += kBlkWarps) {
            const float s = a2[u * kBlkPad + lane] + __ldg(b1 + u0 + u) + dot_tile(w1 + (size_t)(u0 + u) * H + u0, a1, ub1, lane);
            a2[u * kBlkPad + lane] = relu_nan(s);
        }
        __syncthreads();
        for (int u = ub0 + warp; u < ub1; u += kBlkWarps) {
            const float s = a3[u * kBlkPad + lane] + __ldg(b2 + u0 + u) + dot_tile(w2 + (size_t)(u0 + u) * H + u0, a2, ub1, lane);
            a3[u * kBlkPad + lane] = relu_nan(s);
        }
        __syncthreads();
    }
    drain_tile(sx, xcur, r0, nrow, D, g0, nd);
    if (g1 < D) {
        drain_tile(a1, act1, r0, nrow, H, u0, nu);
        drain_tile(a2, act2, r0, nrow, H, u0, nu);
        drain_tile(a3, act3, r0, nrow, H, u0, nu);
    }
    if (threadIdx.x < nrow) { ldacc[r0 + threadIdx.x] = sld[threadIdx.x]; bad[r0 + threadIdx.x] = sbad[threadIdx.x]; }
}


// ------------------------------------------------------------------------------------------------------------------
// Second version of the in-block kernel.  Every tile access above is [unit][lane]: a lane only ever touches its own
// row, so nothing in the step loop needs a CTA barrier -- the first version still split the units of a degree across
// four warps and paid four __syncthreads per degree (plus two loads per FMA in dot_tile): 0.83 ms per block at
// 262 144 rows.  Here a warp owns 32 rows for the whole block (no barrier after the weight staging), the in-block
// weights sit in shared memory TRANSPOSED ([v][unit]) so that the weights of four consecutive units are one
// broadcast LDS.128, and up to three 4-unit chunks share every activation load: 1 LDS.32 + 3 LDS.128 per 12 FMAs.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kWarpChunks = 3;       // 4-unit chunks evaluated together (12 independent FMA chains per lane)

// [32 rows x n] slice of a row-major [B, ld] array -> transposed tile [n][kBlkPad] of the calling warp.  4-byte cp.async:
// every element of the slice is in flight at once (the warp is alone on its scheduler: a register-staged loop would
// expose the full global-memory latency per element); rows are walked in the outer loop, so no integer division.
__device__ __forceinline__ void warp_fill_tile(float* tile, const float* __restrict__ src, int64_t r0, int nrow, int ld, int c0,
                                               int n, int lane) {
    if (!src) {
        for (int c = 0; c < n; ++c) tile[c * kBlkPad + lane] = 0.f;
        return;
    }
    // lanes along the columns (coalesced 128-byte row segments), rows in the unrolled inner loop: one LDGSTS and one
    // pointer bump per element (the first version recomputed both addresses per element: 25 instructions per copy)
    for (int c = lane; c < n; c += 32) {
        const float* gp = src + r0 * (int64_t)ld + c0 + c;
        const unsigned sa = static_cast<unsigned>(__cvta_generic_to_shared(tile + c * kBlkPad));
        if (nrow == kBlkRows) {
#pragma unroll 8
            for (int r = 0; r < kBlkRows; ++r, gp += ld)
                asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(sa + 4u * r), "l"(gp));
        } else {
            for (int r = 0; r < kBlkRows; ++r, gp += ld) {
                if (r < nrow) asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(sa + 4u * r), "l"(gp));
                else tile[c * kBlkPad + r] = 0.f;
            }
        }
    }
}
__device__ __forceinline__ void warp_drain_tile(const float* tile, float* __restrict__ dst, int64_t r0, int nrow, int ld, int c0,
                                                int n, int lane) {
    for (int c = lane; c < n; c += 32) {
        float* gp = dst + r0 * (int64_t)ld + c0 + c;
        const float* sp = tile + c * kBlkPad;
        if (nrow == kBlkRows) {
#pragma unroll 8
            for (int r = 0; r < kBlkRows; ++r, gp += ld) *gp = sp[r];
        } else {
            for (int r = 0; r < nrow; ++r, gp += ld) *gp = sp[r];
        }
    }
}

template <int NCH, int NUP>
__device__ __forceinline__ void warp_units_chunk(const float* __restrict__ wt, const float* __restrict__ bias,
                                                 const float* __restrict__ in, int nv, float* __restrict__ out, int cu, int ub0,
                                                 int ub1, int lane) {
    // accumulators as register pairs: packed fp32 FMAs (FFMA2), two units per instruction -- the weights of a pair are
    // adjacent in the broadcast LDS.128, the lane's activation is duplicated into a pair; same operations and order
    float2 acc2[NCH][2];
#pragma unroll
    for (int c = 0; c < NCH; ++c) { acc2[c][0] = make_float2(0.f, 0.f); acc2[c][1] = make_float2(0.f, 0.f); }
    // compile-time row pitches (NUP, kBlkPad): the unrolled body addresses everything with immediate offsets
    const float* ap = in + lane;
    const float* wp = wt + cu;
    // groups of four inputs, software-pipelined by hand: the operands of group i+1 are requested before the FMAs of group
    // i issue.  A warp shares its scheduler with at most one other warp here (shared memory bounds the CTA at 5-6 warps),
    // so nothing else covers the ~30-cycle LDS latency: the straight loop sat on the short scoreboard for 40 % of its
    // samples (profiles/r02l_c3_ar_block_warp_ncu.txt).  Same FMAs in the same order.
    auto load = [&](int grp, float (&a)[4], float4 (&w)[4][NCH]) {
        const float* a_ = ap + grp * 4 * kBlkPad;
        const float* w_ = wp + grp * 4 * NUP;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            a[k] = a_[k * kBlkPad];
#pragma unroll
            for (int c = 0; c < NCH; ++c) w[k][c] = *reinterpret_cast<const float4*>(w_ + k * NUP + 4 * c);   // rows padded by 4*kWarpChunks floats
        }
    };
    auto fma = [&](const float (&a)[4], const float4 (&w)[4][NCH]) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float2 aa = make_float2(a[k], a[k]);
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
                acc2[c][0] = __ffma2_rn(make_float2(w[k][c].x, w[k][c].y), aa, acc2[c][0]);
                acc2[c][1] = __ffma2_rn(make_float2(w[k][c].z, w[k][c].w), aa, acc2[c][1]);
            }
        }
    };
    const int ngrp = nv >> 2;
    if (ngrp > 0) {
        float aA[4], aB[4];
        float4 wA[4][NCH], wB[4][NCH];
        load(0, aA, wA);
        int g = 0;
        for (; g + 2 <= ngrp; g += 2) {
            load(g + 1, aB, wB);
            fma(aA, wA);
            if (g + 2 < ngrp) load(g + 2, aA, wA);
            fma(aB, wB);
        }
        if (g < ngrp) fma(aA, wA);
    }
    ap += ngrp * 4 * kBlkPad; wp += ngrp * 4 * NUP;
    for (int v = ngrp * 4; v < nv; ++v, ap += kBlkPad, wp += NUP) {
        const float a = *ap;
        const float2 aa = make_float2(a, a);
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            const float4 w = *reinterpret_cast<const float4*>(wp + 4 * c);
            acc2[c][0] = __ffma2_rn(make_float2(w.x, w.y), aa, acc2[c][0]);
            acc2[c][1] = __ffma2_rn(make_float2(w.z, w.w), aa, acc2[c][1]);
        }
    }
    float acc[NCH][4];
#pragma unroll
    for (int c = 0; c < NCH; ++c) { acc[c][0] = acc2[c][0].x; acc[c][1] = acc2[c][0].y; acc[c][2] = acc2[c][1].x; acc[c][3] = acc2[c][1].y; }
    float* op = out + cu * kBlkPad + lane;
    const float* bp = bias + cu;
#pragma unroll
    for (int c = 0; c < NCH; ++c)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int u = cu + 4 * c + j;
            if (u >= ub0 && u < ub1) op[(4 * c + j) * kBlkPad] = relu_nan(op[(4 * c + j) * kBlkPad] + bp[4 * c + j] + acc[c][j]);
        }
}

template <int NUP>
__device__ __forceinline__ void warp_units(const float* __restrict__ wt, const float* __restrict__ bias,
                                           const float* __restrict__ in, int nv, float* __restrict__ out, int ub0, int ub1,
                                           int lane) {
    int cu = ub0 & ~3;
    while (cu < ub1) {
        const int left = (ub1 - cu + 3) >> 2;          // 4-unit chunks still to do (warp-uniform)
        if (left >= 3) { warp_units_chunk<3, NUP>(wt, bias, in, nv, out, cu, ub0, ub1, lane); cu += 12; }
        else if (left == 2) { warp_units_chunk<2, NUP>(wt, bias, in, nv, out, cu, ub0, ub1, lane); cu += 8; }
        else { warp_units_chunk<1, NUP>(wt, bias, in, nv, out, cu, ub0, ub1, lane); cu += 4; }
    }
}

constexpr int kBlkMaxDeg = 8;        // degrees per block the warp kernel takes (compile-time pitch of its W3 tile)

// Layer 3 of the in-block step: the units [ub0, ub1) of the current degree, evaluated like warp_units_chunk (inputs: the
// layer-2 tile), but their values never go to shared memory.  Nothing in the block reads a layer-3 activation except the
// output layer, so each finished unit is PUSHED straight into the (mu, alpha) partial sums of the block's dims, held in
// registers (par[d]; the output weights of dims the unit does not feed are exact zeros of the folded mask), and written
// to the global activation buffer for the later blocks' pull / push products.  The partial pre-activation (previous
// blocks' pull product) comes straight from global memory -- requested before the contraction loop, used after it.
// Without the layer-3 tile a warp's tile is a third smaller: eight warps per SM instead of five or six.
template <int NCH, int NUP>
__device__ __forceinline__ void warp_units_l3_chunk(const float* __restrict__ wt, const float* __restrict__ bias,
                                                    const float* __restrict__ in, int nv, const float* __restrict__ pre_row,
                                                    float* __restrict__ act_row, const float* __restrict__ w3t,
                                                    float2 (&par)[kBlkMaxDeg], int cu, int ub0, int ub1, int lane) {
    float4 pre[NCH];
#pragma unroll
    for (int c = 0; c < NCH; ++c)
        pre[c] = pre_row ? *reinterpret_cast<const float4*>(pre_row + cu + 4 * c) : make_float4(0.f, 0.f, 0.f, 0.f);
    float2 acc2[NCH][2];
#pragma unroll
    for (int c = 0; c < NCH; ++c) { acc2[c][0] = make_float2(0.f, 0.f); acc2[c][1] = make_float2(0.f, 0.f); }
    const float* ap = in + lane;
    const float* wp = wt + cu;
    auto load = [&](int grp, float (&a)[4], float4 (&w)[4][NCH]) {
        const float* a_ = ap + grp * 4 * kBlkPad;
        const float* w_ = wp + grp * 4 * NUP;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            a[k] = a_[k * kBlkPad];
#pragma unroll
            for (int c = 0; c < NCH; ++c) w[k][c] = *reinterpret_cast<const float4*>(w_ + k * NUP + 4 * c);
        }
    };
    auto fma = [&](const float (&a)[4], const float4 (&w)[4][NCH]) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float2 aa = make_float2(a[k], a[k]);
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
                acc2[c][0] = __ffma2_rn(make_float2(w[k][c].x, w[k][c].y), aa, acc2[c][0]);
                acc2[c][1] = __ffma2_rn(make_float2(w[k][c].z, w[k][c].w), aa, acc2[c][1]);
            }
        }
    };
    const int ngrp = nv >> 2;
    if (ngrp > 0) {
        float aA[4], aB[4];
        float4 wA[4][NCH], wB[4][NCH];
        load(0, aA, wA);
        int g = 0;
        for (; g + 2 <= ngrp; g += 2) {
            load(g + 1, aB, wB);
            fma(aA, wA);
            if (g + 2 < ngrp) load(g + 2, aA, wA);
            fma(aB, wB);
        }
        if (g < ngrp) fma(aA, wA);
    }
    ap += ngrp * 4 * kBlkPad; wp += ngrp * 4 * NUP;
    for (int v = ngrp * 4; v < nv; ++v, ap += kBlkPad, wp += NUP) {
        const float a = *ap;
        const float2 aa = make_float2(a, a);
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            const float4 w = *reinterpret_cast<const float4*>(wp + 4 * c);
            acc2[c][0] = __ffma2_rn(make_float2(w.x, w.y), aa, acc2[c][0]);
            acc2[c][1] = __ffma2_rn(make_float2(w.z, w.w), aa, acc2[c][1]);
        }
    }
    const float* bp = bias + cu;
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
        const float accv[4] = {acc2[c][0].x, acc2[c][0].y, acc2[c][1].x, acc2[c][1].y};
        const float prev[4] = {pre[c].x, pre[c].y, pre[c].z, pre[c].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int u = cu + 4 * c + j;
            if (u >= ub0 && u < ub1) {                               // warp-uniform
                const float h = relu_nan(prev[j] + bp[4 * c + j] + accv[j]);
                if (act_row) act_row[u] = h;
                const float2 hh = make_float2(h, h);
                const float4* wr = reinterpret_cast<const float4*>(w3t + u * (2 * kBlkMaxDeg));
#pragma unroll
                for (int q = 0; q < kBlkMaxDeg / 2; ++q) {
                    const float4 w = wr[q];                           // (mu, alpha) weights of dims 2q, 2q + 1
                    par[2 * q] = __ffma2_rn(make_float2(w.x, w.y), hh, par[2 * q]);
                    par[2 * q + 1] = __ffma2_rn(make_float2(w.z, w.w), hh, par[2 * q + 1]);
                }
            }
        }
    }
}

template <int NUP>
__device__ __forceinline__ void warp_units_l3(const float* __restrict__ wt, const float* __restrict__ bias,
                                              const float* __restrict__ in, int nv, const float* __restrict__ pre_row,
                                              float* __restrict__ act_row, const float* __restrict__ w3t,
                                              float2 (&par)[kBlkMaxDeg], int ub0, int ub1, int lane) {
    int cu = ub0 & ~3;
    while (cu < ub1) {
        const int left = (ub1 - cu + 3) >> 2;
        if (left >= 3) { warp_units_l3_chunk<3, NUP>(wt, bias, in, nv, pre_row, act_row, w3t, par, cu, ub0, ub1, lane); cu += 12; }
        else if (left == 2) { warp_units_l3_chunk<2, NUP>(wt, bias, in, nv, pre_row, act_row, w3t, par, cu, ub0, ub1, lane); cu += 8; }
        else { warp_units_l3_chunk<1, NUP>(wt, bias, in, nv, pre_row, act_row, w3t, par, cu, ub0, ub1, lane); cu += 4; }
    }
}

// PERSISTENT: the block's weights are staged once per CTA (one CTA per SM) and every warp then walks over row tiles on
// its own -- no CTA barrier after the staging, so one warp's tile fill / drain overlaps the other warps' step loops.  (As
// one CTA per 6 row tiles, each of the ~9 CTAs an SM ran in turn re-staged ~58 KB of weights and sat alone on the SM
// while they and the tiles arrived: a third of the kernel's stall samples, profiles/r02l_c3_ar_block_warp_ncu.txt.)
// preo: [B, 2D] with (mu, alpha) of a dim adjacent -- the layout the push GEMMs of nf_ar_blocked_forward accumulate into.
template <int NUP>
__global__ void __launch_bounds__(256)
ar_block_warp_kernel(const float* __restrict__ vin, float* __restrict__ xcur, const float* __restrict__ pre1,
                     const float* __restrict__ pre2, const float* __restrict__ pre3, const float* __restrict__ preo,
                     float* __restrict__ act1, float* __restrict__ act2, float* __restrict__ act3,
                     const float* __restrict__ w0, const float* __restrict__ b0, const float* __restrict__ w1,
                     const float* __restrict__ b1, const float* __restrict__ w2, const float* __restrict__ b2,
                     const float* __restrict__ w3, const float* __restrict__ b3, const int32_t* __restrict__ gstart,
                     float* __restrict__ ldacc, int* __restrict__ bad, int64_t B, int D, int H, int g0, int g1, int u0, int u1,
                     int mode) {
    extern __shared__ __align__(16) float sm[];
    const int nd = g1 - g0, nu = u1 - u0;
    constexpr int nup = NUP;                                     // padded row length of the transposed weight tiles
    constexpr int p3 = 2 * kBlkMaxDeg;                           // row pitch of the W3 tile
    const int nwarps = blockDim.x >> 5;
    // shared weights: W0t [nd][nup], W1t / W2t [nu][nup], W3t [nu][p3] (mu, alpha interleaved per dim), biases [3][nu],
    // output biases [p3] (mu, alpha interleaved), in-block unit boundaries of the block's degrees [kBlkMaxDeg + 2]
    float* W0t = sm;
    float* W1t = W0t + nd * nup;
    float* W2t = W1t + nu * nup;
    float* W3t = W2t + nu * nup;
    float* bs = W3t + nu * p3;
    float* b3s = bs + ((3 * nu + 3) & ~3);
    int* gsm = reinterpret_cast<int*>(b3s + p3);
    float* tiles = b3s + p3 + 16;
    const int tile_floats = (nd + 2 * nu) * kBlkPad;             // inputs/outputs of the dims, layer-1 and layer-2 units
    for (int i = threadIdx.x; i < (nd + 2 * nu) * nup + nu * p3; i += blockDim.x) W0t[i] = 0.f;      // padding columns must be finite
    __syncthreads();
    {
        const int lane_ = threadIdx.x & 31, warp_ = threadIdx.x >> 5, nw_ = blockDim.x >> 5;
#define NF_CPA4(dst, srcp) asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(static_cast<unsigned>(__cvta_generic_to_shared(dst))), "l"(srcp))
        for (int u = warp_; u < nu; u += nw_) {                   // one unit (weight row) per warp, lanes along v; all copies in flight
            const float* r0p = w0 + (size_t)(u0 + u) * D + g0;
            for (int d = lane_; d < nd; d += 32) NF_CPA4(W0t + d * nup + u, r0p + d);
            const float* r1p = w1 + (size_t)(u0 + u) * H + u0;
            const float* r2p = w2 + (size_t)(u0 + u) * H + u0;
            for (int v = lane_; v < nu; v += 32) { NF_CPA4(W1t + v * nup + u, r1p + v); NF_CPA4(W2t + v * nup + u, r2p + v); }
        }
        for (int d = warp_; d < nd; d += nw_) {
            const float* rm = w3 + (size_t)(g0 + d) * H + u0;
            const float* ra = w3 + (size_t)(D + g0 + d) * H + u0;
            for (int v = lane_; v < nu; v += 32) { NF_CPA4(W3t + v * p3 + 2 * d, rm + v); NF_CPA4(W3t + v * p3 + 2 * d + 1, ra + v); }
        }
#undef NF_CPA4
    }
    for (int i = threadIdx.x; i < nu; i += blockDim.x) { bs[i] = b0[u0 + i]; bs[nu + i] = b1[u0 + i]; bs[2 * nu + i] = b2[u0 + i]; }
    if (threadIdx.x < nd) { b3s[2 * threadIdx.x] = b3[g0 + threadIdx.x]; b3s[2 * threadIdx.x + 1] = b3[D + g0 + threadIdx.x]; }
    if (threadIdx.x <= nd + 1) gsm[threadIdx.x] = (g0 + (int)threadIdx.x <= D ? gstart[g0 + threadIdx.x] : gstart[D]) - u0;
    asm volatile("cp.async.commit_group;\n" ::);
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
    __syncthreads();                                 // the weights (all warps' copies) have landed; no CTA barrier below

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool first = (g0 == 0);
    float* sx = tiles + (size_t)warp * tile_floats;
    float* a1 = sx + nd * kBlkPad;
    float* a2 = a1 + nu * kBlkPad;
    const int64_t ntiles = (B + kBlkRows - 1) / kBlkRows;
    for (int64_t tile = (int64_t)blockIdx.x * nwarps + warp; tile < ntiles; tile += (int64_t)gridDim.x * nwarps) {
        const int64_t r0 = tile * kBlkRows;
        const int nrow = (int)((B - r0) < kBlkRows ? (B - r0) : kBlkRows);
        warp_fill_tile(sx, vin, r0, nrow, D, g0, nd, lane);
        warp_fill_tile(a1, pre1, r0, nrow, H, u0, nu, lane);
        warp_fill_tile(a2, pre2, r0, nrow, H, u0, nu, lane);
        asm volatile("cp.async.commit_group;\n" ::);
        const bool ok = lane < nrow;
        float ld = (!first && ok) ? ldacc[r0 + lane] : 0.f;
        int poisoned = (!first && ok) ? bad[r0 + lane] : 0;
        // previous blocks' contributions to the parameters of this block's dims, up front: inside the step loop every
        // global load would sit on the critical path of a warp that is nearly alone on its scheduler
        const float4* prow = (preo && ok) ? reinterpret_cast<const float4*>(preo + (r0 + lane) * 2 * D + 2 * g0) : nullptr;
        float2 par[kBlkMaxDeg];                      // (mu, alpha) partial sums of the block's dims
#pragma unroll
        for (int q = 0; q < kBlkMaxDeg / 2; ++q) {
            const float4 pv = (prow && 2 * q < nd) ? prow[q] : make_float4(0.f, 0.f, 0.f, 0.f);      // nd is a multiple of 4
            par[2 * q] = make_float2(pv.x, pv.y); par[2 * q + 1] = make_float2(pv.z, pv.w);
        }
        const float* pre3_row = (pre3 && ok) ? pre3 + (r0 + lane) * (int64_t)H + u0 : nullptr;
        float* act3_row = (g1 < D && ok) ? act3 + (r0 + lane) * (int64_t)H + u0 : nullptr;
        asm volatile("cp.async.wait_group 0;\n" ::: "memory");
        __syncwarp();

        for (int g = g0; g < g1; ++g) {
            const int gi = g - g0;
            const int ub0 = gsm[gi], ub1 = gsm[gi + 1];                       // in-block units of degree g
            // (A) parameters of dim g: bias + previous blocks (preo) + the in-block layer-3 units of degree < g, all
            //     already folded into par[gi] by the pushes of the earlier steps
            {
                float2 pq = par[0];
#pragma unroll
                for (int d = 1; d < kBlkMaxDeg; ++d) if (gi == d) pq = par[d];
                const float2 bq = *reinterpret_cast<const float2*>(b3s + 2 * gi);
                const float mu = bq.x + pq.x, al = bq.y + pq.y;
                float o, t;
                affine_ar_elem<float>(mode, sx[gi * kBlkPad + lane], mu, al, o, t);
                if (poisoned) { o = __int_as_float(0x7fc00000); t = o; }
                if (!is_finite(o)) poisoned = 1;        // 0*NaN of the dense reference poisons every later dim
                sx[gi * kBlkPad + lane] = o;
                ld += t;
            }
            if (g == D - 1) break;
            // (B) hidden units of degree g, layer by layer (all lane-private: no synchronisation)
            warp_units<NUP>(W0t, bs, sx, gi + 1, a1, ub0, ub1, lane);
            warp_units<NUP>(W1t, bs + nu, a1, ub1, a2, ub0, ub1, lane);
            warp_units_l3<NUP>(W2t, bs + 2 * nu, a2, ub1, pre3_row, act3_row, W3t, par, ub0, ub1, lane);
        }
        __syncwarp();
        warp_drain_tile(sx, xcur, r0, nrow, D, g0, nd, lane);
        if (g1 < D) {
            warp_drain_tile(a1, act1, r0, nrow, H, u0, nu, lane);
            warp_drain_tile(a2, act2, r0, nrow, H, u0, nu, lane);
        }
        if (ok) { ldacc[r0 + lane] = ld; bad[r0 + lane] = poisoned; }
        __syncwarp();                                // the drain's reads of the tile are done before the next fill lands
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Third version of the in-block kernel: the dependent in-block steps on the tensor cores.
//   The step of degree g multiplies a [rows x K] activation slice (K = the block's units of degree <= g: 8..80) into the
//   8 or 9 units of that degree -- M x 8 x K products on a dependent chain.  tcgen05 wants M = 128 tiles, operands in
//   shared memory / TMEM and an mbarrier round trip per dependent product; the register-level mma.sync.m16n8k8 (TF32,
//   measured here at a 20-cycle dependent latency and 0.5 MMA / clk / SM, profiles/r02ap_mma_sync_probe.txt) takes the
//   accumulator fragment straight back as the next epilogue's input, so this kernel uses it: a warp owns 32 rows (two
//   m16 tiles) for the whole block, as in the second version, with no CTA barrier after the weight staging.
//   * fp32 parity as everywhere else: 3xTF32 (a_lo b_hi + a_hi b_lo into a correction accumulator, a_hi b_hi into the main
//     one; both operands split on the fly with cvt.rna, two ALU operations per element).
//   * activation tiles are ROW-major [32][pitch], pitch = 4 (mod 8): the four k columns x eight rows of an A fragment
//     load hit 32 different banks, fills / drains are 16-byte cp.async / stores of row-contiguous global segments.
//   * every degree occupies whole 8-unit tiles in shared memory (a 9-unit degree: two tiles); dead slots hold zeros.  The
//     weights are staged once per CTA as B fragments ([pair][lane] float2: the lane's two k rows of its n column), one
//     LDS.64 per (k-tile, n-tile) pair and warp -- against one LDS.128 per four FMAs-per-lane in the FP32 version, which
//     kept that kernel at the shared-memory wavefront limit (one per clock and SM) rather than at the FMA rate.
//   * layer-3 units go straight to global memory (later blocks' pulls) and through a 2-tile scratch into the output
//     layer's PUSH products, accumulated in C fragments (`par`: (mu, alpha) of the block's dims, 16 columns).
//   * the affine step of dim g runs in the lane quad's owner of that column pair (lane % 4 == g % 4); NaN / Inf poison
//     flags are shared over the quad with one shuffle per step; log-det terms are summed per owner lane and reduced over
//     the quad in a fixed order at the end.  The MADE input of a step is x with zeros in the dims not yet produced (the
//     reference's loop, masked_autoregressive_flow.py:46-78), so the noise v stays in registers and the x tile starts at 0.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kMmaMaxTiles = 16;     // 8-unit tiles per block (8 degrees of <= 16 units)
constexpr int kMmaRows = 16;         // rows per warp: one m16 tile
constexpr int kMmaMaxWarps = 16;
constexpr int kSxPitch = 12;         // x tile: 8 dims + 4
constexpr int kH3Pitch = 20;         // layer-3 scratch: 2 tiles + 4

// hi = x rounded to TF32 (nearest, ties away: add half an ulp of the 10-bit mantissa to the magnitude and clear the low 13
// bits -- two integer operations; cvt.rna.tf32.f32 compiles to a ~6-instruction sequence on sm_100a and was a third of
// this kernel's instruction stream), lo = x - hi exactly; the tensor core ignores lo's low 13 bits (<= 2^-21 |x|).
__device__ __forceinline__ void split_tf32_reg(float x, uint32_t& hi, uint32_t& lo) {
    hi = (__float_as_uint(x) + 0x1000u) & 0xffffe000u;
    lo = __float_as_uint(x - __uint_as_float(hi));
}
__device__ __forceinline__ void mma_tf32_16x8x8(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

struct MmaBlockGeom { int NT, P; };
// tiles / (k-tile, n-tile) pairs of the block [g0, g1): every degree takes ceil(count / 8) tiles; the n-tiles of degree g
// see the k-tiles of all degrees <= g of the block
static inline MmaBlockGeom mma_block_geom(const int32_t* gstart, int g0, int g1) {
    MmaBlockGeom m{0, 0};
    for (int g = g0; g < g1; ++g) {
        const int ntl = (gstart[g + 1] - gstart[g] + 7) / 8;
        m.NT += ntl;
        m.P += ntl * m.NT;
    }
    return m;
}

// A fragment of the warp's m16 tile from a row-major tile, split hi / lo: p0 = the lane's element (row rq, column q) in
// the k-tile, p8 = 8 * pitch
__device__ __forceinline__ void mma_load_a(const float* __restrict__ p0, int p8, uint32_t (&ah)[4], uint32_t (&al)[4]) {
    float x[4];
    x[0] = p0[0]; x[1] = p0[p8]; x[2] = p0[4]; x[3] = p0[p8 + 4];
#pragma unroll
    for (int i = 0; i < 4; ++i) split_tf32_reg(x[i], ah[i], al[i]);
}
// acc (main / correction) += A (k-tile) x B fragment, 3xTF32
__device__ __forceinline__ void mma_step(float (&am)[4], float (&ac)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4], float2 b) {
    uint32_t bh0, bl0, bh1, bl1;
    split_tf32_reg(b.x, bh0, bl0);
    split_tf32_reg(b.y, bh1, bl1);
    mma_tf32_16x8x8(ac, al, bh0, bh1);
    mma_tf32_16x8x8(am, ah, bh0, bh1);
    mma_tf32_16x8x8(ac, ah, bl0, bl1);
}

__global__ void __launch_bounds__(32 * kMmaMaxWarps)
ar_block_mma_kernel(const float* __restrict__ vin, float* __restrict__ xcur, const float* __restrict__ pre1,
                    const float* __restrict__ pre2, const float* __restrict__ pre3, const float* __restrict__ preo,
                    float* __restrict__ act1, float* __restrict__ act2, float* __restrict__ act3,
                    const float* __restrict__ w0, const float* __restrict__ b0, const float* __restrict__ w1,
                    const float* __restrict__ b1, const float* __restrict__ w2, const float* __restrict__ b2,
                    const float* __restrict__ w3, const float* __restrict__ b3, const int32_t* __restrict__ gstart,
                    float* __restrict__ ldacc, int* __restrict__ bad, int64_t B, int D, int H, int g0, int g1, int u0,
                    int mode, int NT, int P) {
    extern __shared__ __align__(16) float sm[];
    constexpr int R = kMmaRows;                                  // rows per warp
    const int nd = g1 - g0, NU8 = NT * 8, AP = NU8 + 4;
    float2* Bf0 = reinterpret_cast<float2*>(sm);                 // [NT][32]       input layer: k-tile = the block's dims
    float2* Bf1 = Bf0 + NT * 32;                                 // [P][32]        hidden -> hidden
    float2* Bf2 = Bf1 + P * 32;                                  // [P][32]
    float2* Bf3 = Bf2 + P * 32;                                  // [NT][2][32]    output layer: 16 columns (mu, alpha) x 8 dims
    float* bs = reinterpret_cast<float*>(Bf3 + NT * 64);         // [3][NU8]       biases by shared-memory slot
    float* b3s = bs + 3 * NU8;                                   // [16]
    int* Tt = reinterpret_cast<int*>(b3s + 16);                  // [12]  first tile of the block's degree gi
    int* kmax = Tt + 12;                                         // [16]  k-tiles an n-tile sees
    int* pb = kmax + 16;                                         // [16]  first pair of an n-tile
    int* gsl = pb + 16;                                          // [8]   first unit of degree gi, relative to u0
    int* cnt = gsl + 8;                                          // [8]   units of degree gi (padded layout: multiple of 4)
    int* gmap = cnt + 8;                                         // [NU8] global unit of a slot, -1 for dead slots
    int* ctab = gmap + NU8;                                      // [NU8 / 2]  16-byte chunks of a tile row: (global column - u0, slot)
    float* tiles = reinterpret_cast<float*>(ctab + NU8 / 2);
    __shared__ int nch_s;
    if (threadIdx.x == 0) {
        int t = 0, nch = 0, pairs = 0;
        for (int gi = 0; gi < nd; ++gi) {
            const int gs = gstart[g0 + gi] - u0, c = gstart[g0 + gi + 1] - gstart[g0 + gi];
            const int ntl = (c + 7) >> 3;
            Tt[gi] = t; gsl[gi] = gs; cnt[gi] = c;
            for (int j = 0; j < ntl; ++j) { kmax[t + j] = t + ntl; pb[t + j] = pairs; pairs += t + ntl; }
            for (int s = 0; s < ntl * 8; ++s) gmap[t * 8 + s] = s < c ? u0 + gs + s : -1;
            for (int c4 = 0; c4 < c; c4 += 4) { ctab[2 * nch] = gs + c4; ctab[2 * nch + 1] = t * 8 + c4; ++nch; }
            t += ntl;
        }
        Tt[nd] = t;
        nch_s = nch;
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < NT * 32; idx += blockDim.x) {
        const int nt = idx >> 5, l = idx & 31, n = gmap[nt * 8 + (l >> 2)], k0 = l & 3, k1 = k0 + 4;
        Bf0[idx] = make_float2((n >= 0 && k0 < nd) ? w0[(size_t)n * D + g0 + k0] : 0.f, (n >= 0 && k1 < nd) ? w0[(size_t)n * D + g0 + k1] : 0.f);
    }
    for (int nt = 0; nt < NT; ++nt) {
        const int base = pb[nt] * 32;
        for (int i = threadIdx.x; i < kmax[nt] * 32; i += blockDim.x) {
            const int kt = i >> 5, l = i & 31, n = gmap[nt * 8 + (l >> 2)], ka = gmap[kt * 8 + (l & 3)], kb = gmap[kt * 8 + (l & 3) + 4];
            Bf1[base + i] = make_float2((n >= 0 && ka >= 0) ? w1[(size_t)n * H + ka] : 0.f, (n >= 0 && kb >= 0) ? w1[(size_t)n * H + kb] : 0.f);
            Bf2[base + i] = make_float2((n >= 0 && ka >= 0) ? w2[(size_t)n * H + ka] : 0.f, (n >= 0 && kb >= 0) ? w2[(size_t)n * H + kb] : 0.f);
        }
    }
    for (int idx = threadIdx.x; idx < NT * 64; idx += blockDim.x) {
        const int kt = idx >> 6, n2 = (idx >> 5) & 1, l = idx & 31, col = n2 * 8 + (l >> 2), d = col >> 1, e = col & 1;
        const int ka = gmap[kt * 8 + (l & 3)], kb = gmap[kt * 8 + (l & 3) + 4];
        const float* wr = w3 + (size_t)(e * D + g0 + d) * H;
        Bf3[idx] = make_float2((d < nd && ka >= 0) ? wr[ka] : 0.f, (d < nd && kb >= 0) ? wr[kb] : 0.f);
    }
    for (int s = threadIdx.x; s < NU8; s += blockDim.x) {
        const int n = gmap[s];
        bs[s] = n >= 0 ? b0[n] : 0.f; bs[NU8 + s] = n >= 0 ? b1[n] : 0.f; bs[2 * NU8 + s] = n >= 0 ? b2[n] : 0.f;
    }
    if (threadIdx.x < 16) {
        const int d = threadIdx.x >> 1, e = threadIdx.x & 1;
        b3s[threadIdx.x] = d < nd ? b3[e * D + g0 + d] : 0.f;
    }
    __syncthreads();                                 // tables and fragments staged; no CTA barrier below

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int q = lane & 3, rq = lane >> 2, nch = nch_s;
    const bool first = (g0 == 0);
    const int tile_floats = R * (kSxPitch + 2 * AP + kH3Pitch);
    float* sx = tiles + (size_t)warp * tile_floats;
    float* a1 = sx + R * kSxPitch;
    float* a2 = a1 + R * AP;
    float* h3s = a2 + R * AP;
    // the lane's A-fragment origins (row rq, column q) in the m16 tile of each tile array
    const float* sx0 = sx + rq * kSxPitch + q;
    const float* a10 = a1 + rq * AP + q;
    const float* a20 = a2 + rq * AP + q;
    const float* h30 = h3s + rq * kH3Pitch + q;
    // 16-byte chunk of a tile row this lane moves in the fills / drains (a row has nch <= 32 chunks)
    const bool has_chunk = lane < nch;
    const int gc = has_chunk ? ctab[2 * lane] : 0, sc = has_chunk ? ctab[2 * lane + 1] : 0;
    const int64_t ntiles = (B + R - 1) / R;
    for (int64_t tile = (int64_t)blockIdx.x * nwarps + warp; tile < ntiles; tile += (int64_t)gridDim.x * nwarps) {
        const int64_t r0 = tile * R;
        const int nrow = (int)((B - r0) < R ? (B - r0) : R);
        // ---- fill: x tile zeroed, pre1 / pre2 slices of the block's units by 16-byte cp.async (zeros without a previous block)
        for (int i = lane; i < R * kSxPitch / 4; i += 32) reinterpret_cast<float4*>(sx)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (!pre1 || nrow < R) for (int i = lane; i < R * AP / 4; i += 32) reinterpret_cast<float4*>(a1)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (!pre2 || nrow < R) for (int i = lane; i < R * AP / 4; i += 32) reinterpret_cast<float4*>(a2)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        __syncwarp();
        if (has_chunk && (pre1 || pre2)) {
            const int64_t gofs = r0 * (int64_t)H + u0 + gc;
            const unsigned s1 = static_cast<unsigned>(__cvta_generic_to_shared(a1 + sc)), s2 = static_cast<unsigned>(__cvta_generic_to_shared(a2 + sc));
            const float* g1p = pre1 ? pre1 + gofs : nullptr;
            const float* g2p = pre2 ? pre2 + gofs : nullptr;
#pragma unroll 4
            for (int r = 0; r < nrow; ++r) {
                if (g1p) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s1 + 4u * (unsigned)(r * AP)), "l"(g1p + (int64_t)r * H));
                if (g2p) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s2 + 4u * (unsigned)(r * AP)), "l"(g2p + (int64_t)r * H));
            }
        }
        asm volatile("cp.async.commit_group;\n" ::);
        // ---- per-lane row state: rows rq + 8 * h; the quad's lane q owns dims q and q + 4 of the block
        float vreg[2][2], par[2][4], ldv[2];
        int pois[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int r = rq + 8 * h;
            const bool ok = r < nrow;
            const float* vr = vin + (r0 + r) * (int64_t)D + g0;
            vreg[h][0] = (ok && q < nd) ? vr[q] : 0.f;
            vreg[h][1] = (ok && q + 4 < nd) ? vr[q + 4] : 0.f;
            const float* prow = preo + (r0 + r) * 2 * (int64_t)D + 2 * g0;
#pragma unroll
            for (int n2 = 0; n2 < 2; ++n2) {
                const float2 pv = (preo && ok && n2 * 4 + q < nd) ? *reinterpret_cast<const float2*>(prow + 2 * (n2 * 4 + q)) : make_float2(0.f, 0.f);
                par[n2][2 * h] = pv.x; par[n2][2 * h + 1] = pv.y;
            }
            ldv[h] = (!first && ok && q == 0) ? ldacc[r0 + r] : 0.f;
            pois[h] = (!first && ok) ? bad[r0 + r] : 0;
        }
        asm volatile("cp.async.wait_group 0;\n" ::: "memory");
        __syncwarp();

        for (int g = g0; g < g1; ++g) {
            const int gi = g - g0;
            // (A) dim g: parameters = bias + previous blocks (preo) + pushes of the in-block layer-3 units of lower degree
            {
                const bool owner = (q == (gi & 3));
                const float bmu = b3s[2 * gi], bal = b3s[2 * gi + 1];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const float pm = (gi & 4) ? par[1][2 * h] : par[0][2 * h];
                    const float pa = (gi & 4) ? par[1][2 * h + 1] : par[0][2 * h + 1];
                    const float xv = (gi & 4) ? vreg[h][1] : vreg[h][0];
                    float o, t;
                    affine_ar_elem<float>(mode, xv, bmu + pm, bal + pa, o, t);
                    if (pois[h]) { o = __int_as_float(0x7fc00000); t = o; }
                    int nb = is_finite(o) ? 0 : 1;
                    nb = __shfl_sync(0xffffffffu, nb, (lane & ~3) | (gi & 3));
                    if (owner) { sx[(rq + 8 * h) * kSxPitch + gi] = o; ldv[h] += t; }
                    pois[h] |= nb;           // 0 * NaN of the dense reference poisons every later dim
                }
            }
            if (g == D - 1) break;
            __syncwarp();
            const int t0 = Tt[gi], t1 = Tt[gi + 1], cg = cnt[gi];
            uint32_t ah[4], al[4];
            // previous blocks' share of this degree's layer-3 pre-activations: requested now, used two layers later (in the
            // layer-3 loop the load sat on the critical path of every step: 6 % of the stall samples, profiles/r02as)
            float2 pv3[2][2];
#pragma unroll
            for (int tt = 0; tt < 2; ++tt)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int r = rq + 8 * h, j = tt * 8 + 2 * q;
                    pv3[tt][h] = (pre3 && (tt == 0 || t1 - t0 > 1) && j < cg && r < nrow) ? *reinterpret_cast<const float2*>(pre3 + (r0 + r) * (int64_t)H + u0 + gsl[gi] + j)
                                                                   : make_float2(0.f, 0.f);
                }
            // (B) hidden units of degree g, layer by layer
            for (int nt = t0; nt < t1; ++nt) {               // layer 1: one k-tile (the block's dims; later dims are still zero)
                float am[4] = {}, ac[4] = {};
                mma_load_a(sx0, 8 * kSxPitch, ah, al);
                mma_step(am, ac, ah, al, Bf0[nt * 32 + lane]);
                const int j = (nt - t0) * 8 + 2 * q;
                const bool live = j < cg;
                const float2 bb = *reinterpret_cast<const float2*>(bs + nt * 8 + 2 * q);
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    float2* dst = reinterpret_cast<float2*>(a1 + (rq + 8 * h) * AP + nt * 8 + 2 * q);
                    const float2 pv = *dst;
                    *dst = live ? make_float2(relu_nan(pv.x + bb.x + (am[2 * h] + ac[2 * h])),
                                              relu_nan(pv.y + bb.y + (am[2 * h + 1] + ac[2 * h + 1]))) : make_float2(0.f, 0.f);
                }
            }
            __syncwarp();
            for (int nt = t0; nt < t1; ++nt) {               // layer 2
                float am[4] = {}, ac[4] = {};
                const float2* bp = Bf1 + pb[nt] * 32 + lane;
                const int nk = kmax[nt];
                for (int kt = 0; kt < nk; ++kt) {
                    mma_load_a(a10 + kt * 8, 8 * AP, ah, al);
                    mma_step(am, ac, ah, al, bp[kt * 32]);
                }
                const int j = (nt - t0) * 8 + 2 * q;
                const bool live = j < cg;
                const float2 bb = *reinterpret_cast<const float2*>(bs + NU8 + nt * 8 + 2 * q);
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    float2* dst = reinterpret_cast<float2*>(a2 + (rq + 8 * h) * AP + nt * 8 + 2 * q);
                    const float2 pv = *dst;
                    *dst = live ? make_float2(relu_nan(pv.x + bb.x + (am[2 * h] + ac[2 * h])),
                                              relu_nan(pv.y + bb.y + (am[2 * h + 1] + ac[2 * h + 1]))) : make_float2(0.f, 0.f);
                }
            }
            __syncwarp();
            for (int nt = t0; nt < t1; ++nt) {               // layer 3: to global memory and the push scratch, never to a tile
                const int j = (nt - t0) * 8 + 2 * q;
                const bool live = j < cg;
                float am[4] = {}, ac[4] = {};
                const float2* bp = Bf2 + pb[nt] * 32 + lane;
                const int nk = kmax[nt];
                for (int kt = 0; kt < nk; ++kt) {
                    mma_load_a(a20 + kt * 8, 8 * AP, ah, al);
                    mma_step(am, ac, ah, al, bp[kt * 32]);
                }
                const float2 bb = *reinterpret_cast<const float2*>(bs + 2 * NU8 + nt * 8 + 2 * q);
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int r = rq + 8 * h;
                    const float2 pvv = (nt == t0) ? pv3[0][h] : pv3[1][h];
                    const float2 hv = live ? make_float2(relu_nan(pvv.x + bb.x + (am[2 * h] + ac[2 * h])),
                                                         relu_nan(pvv.y + bb.y + (am[2 * h + 1] + ac[2 * h + 1]))) : make_float2(0.f, 0.f);
                    *reinterpret_cast<float2*>(h3s + r * kH3Pitch + j) = hv;
                    if (g1 < D && live && r < nrow) *reinterpret_cast<float2*>(act3 + (r0 + r) * (int64_t)H + u0 + gsl[gi] + j) = hv;
                }
            }
            __syncwarp();
            if (gi + 1 < nd) {                               // push into the parameters of the block's later dims
                for (int kt = 0; kt < t1 - t0; ++kt) {
                    mma_load_a(h30 + kt * 8, 8 * kH3Pitch, ah, al);
#pragma unroll
                    for (int n2 = 0; n2 < 2; ++n2) {
                        if (n2 * 4 + 3 <= gi || n2 * 4 >= nd) continue;          // all four dims of this half are done / beyond the block
                        const float2 b = Bf3[((t0 + kt) * 2 + n2) * 32 + lane];
                        uint32_t bh0, bl0, bh1, bl1;
                        split_tf32_reg(b.x, bh0, bl0);
                        split_tf32_reg(b.y, bh1, bl1);
                        mma_tf32_16x8x8(par[n2], al, bh0, bh1);
                        mma_tf32_16x8x8(par[n2], ah, bl0, bl1);
                        mma_tf32_16x8x8(par[n2], ah, bh0, bh1);
                    }
                }
                __syncwarp();                                // the scratch is rewritten by the next step's layer 3
            }
        }
        __syncwarp();
        // ---- drain: x, layer-1 / layer-2 activations (for the later blocks' pulls), log-det sums and poison flags
        if (lane < nrow)
            for (int c = 0; c < nd; c += 4)
                *reinterpret_cast<float4*>(xcur + (r0 + lane) * (int64_t)D + g0 + c) = *reinterpret_cast<const float4*>(sx + lane * kSxPitch + c);
        if (g1 < D && has_chunk) {
            float* d1 = act1 + r0 * (int64_t)H + u0 + gc;
            float* d2 = act2 + r0 * (int64_t)H + u0 + gc;
#pragma unroll 4
            for (int r = 0; r < nrow; ++r) {
                *reinterpret_cast<float4*>(d1 + (int64_t)r * H) = *reinterpret_cast<const float4*>(a1 + r * AP + sc);
                *reinterpret_cast<float4*>(d2 + (int64_t)r * H) = *reinterpret_cast<const float4*>(a2 + r * AP + sc);
            }
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            float s = ldv[h];
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            const int r = rq + 8 * h;
            if (q == 0 && r < nrow) { ldacc[r0 + r] = s; bad[r0 + r] = pois[h]; }
        }
        __syncwarp();                                // the drain's reads of the tiles are done before the next fill lands
    }
}

}  // namespace nf

using namespace nf;
#define NF_REQ(p) do { if ((p) == nullptr) return NF_ERR_NULL; } while (0)

extern "C" int64_t nf_ar_blocked_workspace_floats(int64_t B, int D, int H) {
    // act1..3, pre1..3: 6*B*H; preo: 2*B*D; xcur: B*D; ldacc: B; bad: B (ints)
    return 6 * B * H + 3 * B * D + 2 * B;
}

extern "C" int nf_ar_blocked_forward(const void* v, const void* const* w, const void* const* w_hi, const void* const* w_lo,
                                     const void* const* b, const int32_t* gstart_dev, const int32_t* gstart_host,
                                     void* workspace, void* out, void* ld, int64_t B, int D, int H, int mode,
                                     int block_degrees, nf_stream_t stream) {
    if (B < 0 || D < 1 || H < 1 || block_degrees < 1) return NF_ERR_BAD_SHAPE;
    if (mode != NF_AR_MAF_FORWARD && mode != NF_AR_IAF_INVERSE) return NF_ERR_UNSUPPORTED;
    if (B == 0) return NF_OK;
    NF_REQ(v); NF_REQ(w); NF_REQ(w_hi); NF_REQ(w_lo); NF_REQ(b); NF_REQ(gstart_dev); NF_REQ(gstart_host);
    NF_REQ(workspace); NF_REQ(out); NF_REQ(ld);
    if ((D % 4) != 0 || (H % 4) != 0 || (block_degrees % 4) != 0) return NF_ERR_UNSUPPORTED;      // TMA row pitches of the slice GEMMs
    // every block of hidden units starts at a multiple of 4 (packing.blocked_made_pack pads the blocks with dead units):
    // 16-byte TMA bases of the push products' column slices, 128-bit row stores of the pull products.  (Multiples of 8
    // would allow 256-bit stores, but a 65-unit block padded to 72 costs the in-block kernel one of its six warps.)
    for (int g0 = 0; g0 < D; g0 += block_degrees)
        if (gstart_host[g0] % 4) return NF_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    float* ws = (float*)workspace;
    const size_t BH = (size_t)B * H, BD = (size_t)B * D;
    float* act1 = ws; float* act2 = act1 + BH; float* act3 = act2 + BH;
    float* pre1 = act3 + BH; float* pre2 = pre1 + BH; float* pre3 = pre2 + BH;
    float* preo = pre3 + BH; float* xcur = preo + 2 * BD; float* ldacc = xcur + BD;
    int* bad = reinterpret_cast<int*>(ldacc + B);
    const float* w0 = (const float*)w[0]; const float* w1 = (const float*)w[1];
    const float* w2 = (const float*)w[2]; const float* w3 = (const float*)w[3];
    const int grid = (int)cdiv(B, kBlkRows);
    bool pushed = false;
    for (int g0 = 0; g0 < D; g0 += block_degrees) {
        const int g1 = (g0 + block_degrees < D) ? g0 + block_degrees : D;
        const int u0 = gstart_host[g0], u1 = gstart_host[g1];
        const int nd = g1 - g0, nu = u1 - u0;
        const size_t smem = sizeof(float) * ((size_t)(nd + 3 * nu) * kBlkPad + 2 * kBlkRows);
        if (smem > 160 * 1024) return NF_ERR_UNSUPPORTED;
        const bool prev = g0 > 0;
        int rc;
        if (prev && nu > 0) {
            // PULL: contributions of dims < g0 / units < u0 (all final) to the block's hidden pre-activations, dense over
            // the whole batch (the output layer's share arrives by PUSH, below)
            rc = nf_linear_tc(xcur, (const float*)w_hi[0] + (size_t)u0 * D, (const float*)w_lo[0] + (size_t)u0 * D, nullptr,
                              pre1 + u0, B, nu, g0, D, D, H, 0, nullptr, stream);
            if (rc) return rc;
            if (u0 > 0) {
                rc = nf_linear_tc(act1, (const float*)w_hi[1] + (size_t)u0 * H, (const float*)w_lo[1] + (size_t)u0 * H, nullptr,
                                  pre2 + u0, B, nu, u0, H, H, H, 0, nullptr, stream);
                if (rc) return rc;
                rc = nf_linear_tc(act2, (const float*)w_hi[2] + (size_t)u0 * H, (const float*)w_lo[2] + (size_t)u0 * H, nullptr,
                                  pre3 + u0, B, nu, u0, H, H, H, 0, nullptr, stream);
                if (rc) return rc;
            }
        }
        const bool hp = prev && u0 > 0;
        const bool have_preo = pushed;               // some earlier block pushed into preo (it covers every later dim)
        bool launched = false;
        if (nu > 0 && nd <= kBlkMaxDeg && (nd % 4) == 0) {
            // tensor-core kernel (mma.sync): every degree of the block 4-aligned (per-degree padded layout) and <= 16 units
            bool ok = true;
            for (int g = g0; g < g1; ++g)
                if ((gstart_host[g] % 4) != 0 || gstart_host[g + 1] - gstart_host[g] > 16) ok = false;
            const MmaBlockGeom mg = mma_block_geom(gstart_host, g0, g1);
            const int NU8 = mg.NT * 8, AP = NU8 + 4;
            const size_t wfl = (size_t)mg.NT * 64 + 2 * (size_t)mg.P * 64 + (size_t)mg.NT * 128 + 3 * (size_t)NU8 + 16 + 60 + NU8 + NU8 / 2;
            const size_t tfl = (size_t)kMmaRows * (size_t)(kSxPitch + 2 * AP + kH3Pitch);
            int nw = (ok && mg.NT >= 1 && mg.NT <= kMmaMaxTiles && wfl * sizeof(float) < 180 * 1024)
                         ? (int)((226 * 1024 / sizeof(float) - wfl) / tfl) : 0;
            if (nw > kMmaMaxWarps) nw = kMmaMaxWarps;
            if (nw >= 2) {
                const size_t smem2 = sizeof(float) * (wfl + (size_t)nw * tfl);
                const int64_t ctas = cdiv(cdiv(B, (int64_t)kMmaRows), (int64_t)nw);
                const int grid2 = (int)(ctas < kNumSMs ? ctas : kNumSMs);              // persistent: one CTA per SM
                NF_CUDA(cudaFuncSetAttribute(ar_block_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
                ar_block_mma_kernel<<<grid2, 32 * nw, smem2, st>>>(
                    (const float*)v, xcur, prev ? pre1 : nullptr, hp ? pre2 : nullptr, hp ? pre3 : nullptr,
                    have_preo ? preo : nullptr, act1, act2, act3, w0, (const float*)b[0], w1, (const float*)b[1], w2,
                    (const float*)b[2], w3, (const float*)b[3], gstart_dev, ldacc, bad, B, D, H, g0, g1, u0, mode, mg.NT, mg.P);
                count_launch();
                NF_LAUNCH_CHECK();
                launched = true;
            }
        }
        if (!launched) {
            // warp-private kernel (FP32 pipe): shared transposed weights + one tile per warp; as many warps as fit in 220 KB
            const int need = ((nu + 3) & ~3) + 4 * kWarpChunks;
            const int nup = need <= 48 ? 48 : (need <= 80 ? 80 : (need <= 96 ? 96 : 160));   // compile-time pitches of ar_block_warp_kernel
            const size_t wfl = (size_t)(nd + 2 * nu) * nup + (size_t)nu * 2 * kBlkMaxDeg + ((3 * nu + 3) & ~3) + 2 * kBlkMaxDeg + 16;
            const size_t tfl = (size_t)(nd + 2 * nu) * kBlkPad;
            int nw = wfl * sizeof(float) < 200 * 1024 ? (int)((220 * 1024 / sizeof(float) - wfl) / tfl) : 0;
            if (nw > 8) nw = 8;
            if (nw >= 2 && need <= 160 && nd <= kBlkMaxDeg && (nd % 4) == 0) {
                const size_t smem2 = sizeof(float) * (wfl + (size_t)nw * tfl);
                const int64_t ctas = cdiv(cdiv(B, (int64_t)kBlkRows), (int64_t)nw);
                const int grid2 = (int)(ctas < kNumSMs ? ctas : kNumSMs);              // persistent: one CTA per SM
#define NF_ABW(NUPV)                                                                                                          \
                do {                                                                                                          \
                    NF_CUDA(cudaFuncSetAttribute(ar_block_warp_kernel<NUPV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2)); \
                    ar_block_warp_kernel<NUPV><<<grid2, 32 * nw, smem2, st>>>(                                                 \
                        (const float*)v, xcur, prev ? pre1 : nullptr, hp ? pre2 : nullptr, hp ? pre3 : nullptr,                \
                        have_preo ? preo : nullptr, act1, act2, act3, w0, (const float*)b[0], w1, (const float*)b[1], w2,      \
                        (const float*)b[2], w3, (const float*)b[3], gstart_dev, ldacc, bad, B, D, H, g0, g1, u0, u1, mode);    \
                } while (0)
                if (nup == 48) NF_ABW(48); else if (nup == 80) NF_ABW(80); else if (nup == 96) NF_ABW(96); else NF_ABW(160);
#undef NF_ABW
                count_launch();
                NF_LAUNCH_CHECK();
                launched = true;
            }
        }
        if (!launched) {
            if (smem > 48 * 1024)
                NF_CUDA(cudaFuncSetAttribute(ar_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            ar_block_kernel<<<grid, kBlkRows * kBlkWarps, smem, st>>>(
                (const float*)v, xcur, prev ? pre1 : nullptr, hp ? pre2 : nullptr, hp ? pre3 : nullptr, have_preo ? preo : nullptr,
                act1, act2, act3, w0, (const float*)b[0], w1, (const float*)b[1], w2, (const float*)b[2], w3, (const float*)b[3],
                gstart_dev, ldacc, bad, B, D, H, g0, g1, u0, u1, mode);
            count_launch();
            NF_LAUNCH_CHECK();
        }
        // PUSH: the block's layer-3 units are final -> their share of the output-layer pre-activations of ALL later dims in
        // one narrow-K product, accumulated into preo ([B, 2D], (mu, alpha) of a dim adjacent; w_hi[3] / w_lo[3] hold the
        // output layer's rows in that order).  Pulling per block instead re-read act3[:, :u0] for 2 x 8 outputs every time:
        // 1.85 ms of the 8.3 ms pass at [262144, 64] x 512 (profiles/r01z_c3_launches.csv).
        if (g1 < D && nu > 0) {
            rc = linear_tc_push(act3 + u0, (const float*)w_hi[3] + (size_t)2 * g1 * H + u0, (const float*)w_lo[3] + (size_t)2 * g1 * H + u0,
                                preo + 2 * g1, B, 2 * (D - g1), nu, H, H, 2 * D, pushed ? 1 : 0, st);
            if (rc) return rc;
            pushed = true;
        }
    }
    return nf_ar_finish_forward(xcur, v, ldacc, out, ld, B, D, mode, NF_F32, stream);
}
