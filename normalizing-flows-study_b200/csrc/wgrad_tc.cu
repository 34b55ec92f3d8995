// wgrad_tc.cu -- fp32-accurate weight gradient of a dense layer on the 5th-gen tensor cores:
//     dW[N,K] = sum_b dY[b,N] * X[b,K]            (the reduction runs over the batch rows)
//   (autograd of F.linear in MaskedLinear / MADE, masked_linear.py:14-18, made.py:136-140, and of the coupling /
//    spline conditioner MLPs, coupling_layer.py:18-35, spline_coupling_layer.py:55-62)
//
// Both operands are row-major [B, *]: the reduction dimension is the strided one, i.e. both are "MN-major" in UMMA
// terms.  No transposed copies are made:
//   * dY tile [32 b x 128 n] lands in shared memory through TMA (four 32-float-wide SWIZZLE_128B boxes); converter
//     thread n reads its column (conflict-free: a warp reads 32 consecutive floats of one row), splits it hi/lo and
//     stores it into TMEM as the MMA A operand (lane = n, column = b);
//   * X tile [32 b x 128 k] lands through TMA in SWIZZLE_128B_ATOM_32B mode and is the MMA B operand *in place* as an
//     MN-major SWIZZLE_128B_BASE32B image (LBO = 4096 B between 32-float column chunks, 8 b-rows = 1024 B = one k-step);
//     the converters round it to TF32 in place (hi) and write the residual image (lo) beside it.
// 3xTF32: D += A_hi*B_hi + A_lo*B_hi + A_hi*B_lo with fp32 accumulation in TMEM.
// Few output tiles, very long reduction => split over the batch: grid = tiles x splits, every split writes its
// partial tile to the caller's workspace and wgrad_reduce_kernel sums the partials in a fixed order (deterministic,
// no atomics).  Warp roles: warp 0 TMA producer, warp 1 MMA issuer, warps 2-5 converters + epilogue.
#include <cuda.h>
#include "nf_common.cuh"
#include "tc_common.cuh"

namespace nf {

constexpr int kWgBM = 128, kWgBN = 128, kWgBK = 32;    // dW rows (dY columns) x dW columns (X columns) x batch rows per stage
constexpr int kWgStages = 2;
constexpr int kWgThreads = 192;
constexpr int kWgTmemCols = 256;                       // D: 128 | A stage 0: hi 32 + lo 32 | A stage 1: hi 32 + lo 32
constexpr int kWgColD = 0, kWgColA = 128;
constexpr uint32_t kWgChunkBytes = kWgBK * 128;        // one 32-float-wide box: 32 rows x 128 B
constexpr uint32_t kWgTileBytes = 4 * kWgChunkBytes;   // 128 columns
constexpr uint32_t kWgStageBytes = 3 * kWgTileBytes;   // dY | X hi (in place) | X lo

__device__ __forceinline__ void wg_tma_load_2d(void* smem_dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(tc::smem_u32(smem_dst)), "l"(map), "r"(c0), "r"(c1), "r"(tc::smem_u32(bar)) : "memory");
}

// shared-memory descriptor of an MN-major tf32 operand.  The only MN-major layout the tensor core accepts for 32-bit
// operands is SWIZZLE_128B_BASE32B (layout type 1; plain SWIZZLE_128B silently multiplies by zero -- measured with
// scripts/dbg/umma_probe.cu): rows of 128 B = 32 floats along N, one row per k; the four 32-byte atoms of a row are
// XOR-swizzled with (row % 4) (address bits [5,7) ^= bits [7,9)) -- what TMA's SWIZZLE_128B_ATOM_32B mode writes.
// LBO = distance between 32-float chunks along N, SBO = distance between groups of four k rows (512 B).
__device__ __forceinline__ uint64_t smem_desc_mn_sw128_32b(uint32_t smem_byte_addr, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_byte_addr >> 4) & 0x3fffu);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16;
    d |= (uint64_t)(512u >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)1 << 61;
    return d;
}

__global__ void __launch_bounds__(kWgThreads, 2)
wgrad_tc_kernel(const __grid_constant__ CUtensorMap tm_g, const __grid_constant__ CUtensorMap tm_x, float* __restrict__ out,
                int N, int K, int nkb, int kb_per_split, int64_t ld_out, int64_t split_stride,
                const uint8_t* __restrict__ tile_live, const float* __restrict__ dy_direct, int64_t ld_dy, int64_t B,
                int passes, int vec) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kWgStages * kWgStageBytes);
    uint64_t* full = bars;                       // [S] TMA landed
    uint64_t* empty = bars + kWgStages;          // [S] MMAs consumed the stage and its TMEM A stage
    uint64_t* ready = bars + 2 * kWgStages;      // [S] converters wrote the TMEM A stage and the X hi / lo images
    uint64_t* d_full = ready + kWgStages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(d_full + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int k_tiles = (K + kWgBN - 1) / kWgBN;
    const int n0 = (int)(blockIdx.x / k_tiles) * kWgBM;          // dW row block = dY column block
    const int k0 = (int)(blockIdx.x % k_tiles) * kWgBN;          // dW column block = X column block
    const int kb0 = (int)blockIdx.y * kb_per_split;
    const int kb1 = min(nkb, kb0 + kb_per_split);
    // tile_live[tile] == 0: the weight mask is zero on this whole 128 x 128 tile (MADE): nothing to accumulate, zeros out
    const int nloc = (tile_live && !tile_live[blockIdx.x]) ? 0 : max(0, kb1 - kb0);

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < kWgStages; ++i) { tc::mbar_init(&full[i], 1); tc::mbar_init(&empty[i], 1); tc::mbar_init(&ready[i], 128); }
        tc::mbar_init(d_full, 1);
        tc::fence_mbar_init();
    }
    if (warp == 1) tc::tmem_alloc(tmem_slot, kWgTmemCols);
    // 32-float-wide boxes that hold live columns of dY / X.  Boxes entirely past N / K are never requested (narrow layers:
    // the 64-wide conditioners of the 2-D flows had half of their TMA boxes filled with out-of-bounds zeros, and
    // out-of-bounds fill is slow, profiles/r02az_slice_gemm.jsonl); their shared-memory chunks are zeroed once here.
    const int ng = min(4, (N - n0 + 31) / 32), nx = min(4, (K - k0 + 31) / 32);
    if (nloc > 0) {
        for (int s = 0; s < kWgStages; ++s) {
            uint8_t* st = smem + s * kWgStageBytes;
            for (int j = ng; j < 4; ++j)
                for (int i = tid; i < (int)(kWgChunkBytes / 16); i += kWgThreads) reinterpret_cast<uint4*>(st + j * kWgChunkBytes)[i] = make_uint4(0u, 0u, 0u, 0u);
            for (int j = nx; j < 4; ++j)
                for (int i = tid; i < (int)(kWgChunkBytes / 16); i += kWgThreads) reinterpret_cast<uint4*>(st + kWgTileBytes + j * kWgChunkBytes)[i] = make_uint4(0u, 0u, 0u, 0u);
        }
        tc::fence_proxy_async_smem();
    }
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tb = *tmem_slot;

    if (warp == 0) {
        // ---------------- TMA producer ----------------
        if (lane == 0) {
            const uint32_t tx_bytes = (uint32_t)((dy_direct ? 0 : ng) + nx) * kWgChunkBytes;
            for (int i = 0; i < nloc; ++i) {
                const int s = i % kWgStages;
                if (i >= kWgStages) tc::mbar_wait(&empty[s], ((i / kWgStages) - 1) & 1);
                uint8_t* st = smem + s * kWgStageBytes;
                const int b0 = (kb0 + i) * kWgBK;
                tc::mbar_arrive_expect_tx(&full[s], tx_bytes);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (!dy_direct && j < ng) wg_tma_load_2d(st + j * kWgChunkBytes, &tm_g, n0 + 32 * j, b0, &full[s]);
                    if (j < nx) wg_tma_load_2d(st + kWgTileBytes + j * kWgChunkBytes, &tm_x, k0 + 32 * j, b0, &full[s]);
                }
            }
        }
    } else if (warp == 1) {
        // ---------------- MMA issuer (whole warp, convergent; one elected lane issues) ----------------
        const uint32_t idesc = tc::idesc_tf32_m128((uint32_t)(nx * 32)) | (1u << 16);   // B operand MN-major; only the live X columns
        const bool leader = tc::elect_one();
        for (int i = 0; i < nloc; ++i) {
            const int s = i % kWgStages;
            tc::mbar_wait(&ready[s], (i / kWgStages) & 1);
            tc::fence_after_sync();
            const uint32_t st = tc::smem_u32(smem + s * kWgStageBytes);
            const uint64_t d_hi = smem_desc_mn_sw128_32b(st + kWgTileBytes, kWgChunkBytes);
            const uint64_t d_lo = smem_desc_mn_sw128_32b(st + 2 * kWgTileBytes, kWgChunkBytes);
            const uint32_t a_hi = tb + kWgColA + s * 64, a_lo = a_hi + 32;
#pragma unroll
            for (int pass = 0; pass < 3; ++pass) {
                if (pass >= passes) break;                    // passes == 1: one TF32 pass (nf_set_option(7, .), gemm_tc2.cu)
                const uint32_t ac = (pass == 1) ? a_lo : a_hi;
                const uint64_t wd = (pass == 2) ? d_lo : d_hi;
#pragma unroll
                for (int k = 0; k < 4; ++k) {                 // 8 batch rows per MMA = 1024 B
                    if (leader) tc::mma_tf32_ts(tb + kWgColD, ac + k * 8, wd + (uint64_t)(k * (1024 >> 4)), idesc, (i | pass | k) != 0 ? 1u : 0u);
                }
            }
            if (leader) tc::mma_commit(&empty[s]);
            __syncwarp();
        }
        if (leader) tc::mma_commit(d_full);
        __syncwarp();
    } else {
        // ---------------- converters, then epilogue (warps 2..5; TMEM lane quadrant = warp % 4) ----------------
        const int q = warp & 3;
        const int ct = (warp - 2) * 32 + lane;               // 0..127: slice of the X tile handled by this thread
        const uint32_t lane_addr = tb + ((uint32_t)(q * 32) << 16);
        for (int i = 0; i < nloc; ++i) {
            const int s = i % kWgStages;
            // full[s] of round i also implies empty[s] of round i-2 (the producer waited for it): the TMEM A stage is free
            tc::mbar_wait(&full[s], (i / kWgStages) & 1);
            tc::fence_after_sync();
            uint8_t* st = smem + s * kWgStageBytes;
            // dY column n = 32q + lane: element (b, n) sits at chunk q, row b, 16-byte slot ((lane/4) ^ (b%8))
            const uint8_t* gcol = st + q * kWgChunkBytes + (lane & 3) * 4;
            uint32_t hi[32], lo[32];
            const bool dy_live = dy_direct != nullptr || q < ng;       // warp-uniform: this quadrant's 32 dY columns exist
            if (!dy_live) {
                // dW rows past N: never stored, their A rows may hold anything
            } else if (dy_direct) {
                // dY rows whose pitch TMA cannot take (N % 4 != 0, e.g. the 3K-1 = 23 / 29 wide spline heads): the converter
                // thread fetches its column straight from global memory (a warp reads 32 consecutive floats per row)
                const int n = n0 + q * 32 + lane;
                const int64_t b0 = (int64_t)(kb0 + i) * kWgBK;
                const float* gp = dy_direct + b0 * ld_dy + (n < N ? n : 0);
                float v[32];
#pragma unroll
                for (int b = 0; b < 32; ++b) v[b] = (n < N && b0 + b < B) ? __ldg(gp + b * ld_dy) : 0.f;
#pragma unroll
                for (int b = 0; b < 32; ++b) tc::split_tf32(v[b], hi[b], lo[b]);
            } else {
#pragma unroll
                for (int b = 0; b < 32; ++b) {
                    const float v = *reinterpret_cast<const float*>(gcol + b * 128 + ((((uint32_t)lane >> 2) ^ (uint32_t)(b & 7)) << 4));
                    tc::split_tf32(v, hi[b], lo[b]);
                }
            }
            const uint32_t a_hi = lane_addr + kWgColA + s * 64, a_lo = a_hi + 32;
            if (dy_live) {
                uint32_t t0[16], t1[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) { t0[j] = hi[j]; t1[j] = hi[16 + j]; }
                tc::tmem_st16(a_hi, t0); tc::tmem_st16(a_hi + 16, t1);
                if (passes != 1) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) { t0[j] = lo[j]; t1[j] = lo[16 + j]; }
                    tc::tmem_st16(a_lo, t0); tc::tmem_st16(a_lo + 16, t1);
                }
            }
            // X tile: elementwise hi (in place) / lo (second image, same offsets)
            uint8_t* xh = st + kWgTileBytes;
            uint8_t* xl = st + 2 * kWgTileBytes;
#pragma unroll
            for (int j = 0; j < (int)(kWgTileBytes / 16 / 128); ++j) {
                if (j >= 2 * nx) break;                          // two 2 KB slabs per 32-column chunk; dead chunks stay zero
                const uint32_t off = (uint32_t)(j * 128 + ct) * 16u;
                const float4 v = *reinterpret_cast<const float4*>(xh + off);
                uint4 h, l;
                tc::split_tf32_weight(v.x, h.x, l.x);
                tc::split_tf32_weight(v.y, h.y, l.y);
                tc::split_tf32_weight(v.z, h.z, l.z);
                tc::split_tf32_weight(v.w, h.w, l.w);
                *reinterpret_cast<uint4*>(xh + off) = h;
                if (passes != 1) *reinterpret_cast<uint4*>(xl + off) = l;
            }
            tc::fence_proxy_async_smem();
            tc::wait_st();
            tc::fence_before_sync();
            tc::mbar_arrive(&ready[s]);
        }
        // epilogue once every MMA has completed
        tc::mbar_wait(d_full, 0);
        tc::fence_after_sync();
        // the thread owns dW row n0 + 32q + lane: one 256-bit store per 8 columns (tc::epilogue_store8)
        float* dst = out + (int64_t)blockIdx.y * split_stride;
        const int row = n0 + q * 32 + lane;
        float* yrow = dst + (int64_t)row * ld_out;
        float* tbuf = reinterpret_cast<float*>(smem) + (size_t)q * 32 * 33;      // stage memory is free once d_full has fired
#pragma unroll
        for (int c = 0; c < kWgBN / 32; ++c) {
            if (c >= nx) break;                                  // columns past K: neither accumulated nor stored
            uint32_t v0[16], v1[16];
            if (nloc > 0) {
                tc::tmem_ld16(lane_addr + kWgColD + c * 32, v0);
                tc::tmem_ld16(lane_addr + kWgColD + c * 32 + 16, v1);
                tc::wait_ld();
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) { v0[j] = 0u; v1[j] = 0u; }
            }
            if (vec) {
                if (row < N) tc::epilogue_store32(yrow, k0 + c * 32, K, v0, v1, nullptr, 0, true);
            } else {
                tc::epilogue_store32_transposed(dst, ld_out, n0 + q * 32, N, k0 + c * 32, K, v0, v1, nullptr, 0, tbuf, lane);
            }
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 1) tc::tmem_dealloc(tb, kWgTmemCols);
}

// dW[r, c] = sum_s partial[s][r][c]  (fixed order => deterministic); splits == 0 writes zeros
__global__ void wgrad_reduce_kernel(const float* __restrict__ part, float* __restrict__ dw, int N, int K, int64_t ld_dw,
                                    int splits, int64_t split_stride) {
    const int64_t total = (int64_t)N * K, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        float acc = 0.f;
        for (int s = 0; s < splits; ++s) acc += part[s * split_stride + i];
        dw[(i / K) * ld_dw + (i % K)] = acc;
    }
}

// Small outputs with many splits (the 64 x 64 layers of the 2-D flows at 2^20 rows: 296 partial tiles for 4096 sums): the
// kernel above leaves 4096 threads walking 296 strided values each (40 us).  Here a block owns 32 consecutive outputs, warp
// w sums the splits w, w + 8, ... (coalesced 128-byte rows, four loads in flight) and the eight partial sums are added in
// warp order -- still a fixed order, so still deterministic.
__global__ void __launch_bounds__(256)
wgrad_reduce_wide_kernel(const float* __restrict__ part, float* __restrict__ dw, int N, int K, int64_t ld_dw, int splits,
                         int64_t split_stride) {
    __shared__ float red[8][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t total = (int64_t)N * K;
    for (int64_t base = (int64_t)blockIdx.x * 32; base < total; base += (int64_t)gridDim.x * 32) {
        const int64_t i = base + lane;
        float acc = 0.f;
        if (i < total) {
            const float* p = part + i;
            int sp = warp;
            for (; sp + 24 < splits; sp += 32) {
                const float v0 = p[sp * split_stride], v1 = p[(sp + 8) * split_stride], v2 = p[(sp + 16) * split_stride],
                            v3 = p[(sp + 24) * split_stride];
                acc += v0; acc += v1; acc += v2; acc += v3;
            }
            for (; sp < splits; sp += 8) acc += p[sp * split_stride];
        }
        red[warp][lane] = acc;
        __syncthreads();
        if (warp == 0 && i < total) {
            float t = red[0][lane];
#pragma unroll
            for (int w = 1; w < 8; ++w) t += red[w][lane];
            dw[(i / K) * ld_dw + (i % K)] = t;
        }
        __syncthreads();
    }
}

// row-major fp32 [rows, cols] with pitch ld: box = 32 rows x 32 floats (one 128-byte swizzle span wide), zero OOB fill
static bool wg_make_map(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int64_t ld, CUtensorMapSwizzle swz) {
    const tc::EncodeTiledFn fn = tc::encode_tiled_fn();
    if (!fn) return false;
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    cuuint32_t box[2] = {32u, (cuuint32_t)kWgBK};
    cuuint32_t estr[2] = {1, 1};
    return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

constexpr int kWgradMaxKB = 64;    // K blocks per TMEM accumulation chain at most (see wg_plan)
extern int g_tc_passes;             // nf_set_option(7, v)

// Number of batch splits.  (1) Fill two CTAs per SM, with at least 8 K blocks (256 rows) per split.  (2) The tensor
// core's fp32 accumulation truncates (measured: the error of a TMEM accumulation chain grows linearly, ~2^-24 of the
// running sum per MMA, 12 MMAs per K block), so a chain is at most kWgradMaxKB K blocks long; the partials are then
// summed with round-to-nearest fp32 adds by wgrad_reduce_kernel.
static void wg_plan(int64_t B, int64_t N, int64_t K, int* splits, int* kb_per_split, int* nkb_out) {
    const int64_t tiles = cdiv(N, kWgBM) * cdiv(K, kWgBN);
    const int64_t nkb = cdiv(B, kWgBK);
    int64_t s = (2 * (int64_t)kNumSMs) / tiles;
    if (s < 1) s = 1;
    const int64_t smax = nkb / 8 > 1 ? nkb / 8 : 1;
    if (s > smax) s = smax;
    const int64_t smin = cdiv(nkb, (int64_t)kWgradMaxKB);
    if (s < smin) s = smin;
    const int64_t per = cdiv(nkb, s);
    s = cdiv(nkb, per);
    *splits = (int)s; *kb_per_split = (int)per; *nkb_out = (int)nkb;
}

}  // namespace nf

using namespace nf;
#define NF_REQ(p) do { if ((p) == nullptr) return NF_ERR_NULL; } while (0)

extern "C" int64_t nf_linear_wgrad_tc_workspace(int64_t B, int64_t N, int64_t K) {
    if (B < 1 || N < 1 || K < 1 || B > 2147483647LL - 64) return 0;
    int splits, per, nkb;
    wg_plan(B, N, K, &splits, &per, &nkb);
    return splits > 1 ? (int64_t)splits * N * K * 4 : 0;
}

extern "C" int nf_linear_wgrad_tc_masked(const void* dy, const void* x, void* dw, int64_t B, int64_t N, int64_t K, int64_t ld_dy,
                                         int64_t ld_x, int64_t ld_dw, void* workspace, int64_t ws_bytes,
                                         const uint8_t* tile_live, nf_stream_t stream);

extern "C" int nf_linear_wgrad_tc(const void* dy, const void* x, void* dw, int64_t B, int64_t N, int64_t K, int64_t ld_dy,
                                  int64_t ld_x, int64_t ld_dw, void* workspace, int64_t ws_bytes, nf_stream_t stream) {
    return nf_linear_wgrad_tc_masked(dy, x, dw, B, N, K, ld_dy, ld_x, ld_dw, workspace, ws_bytes, nullptr, stream);
}

extern "C" int nf_linear_wgrad_tc_masked(const void* dy, const void* x, void* dw, int64_t B, int64_t N, int64_t K, int64_t ld_dy,
                                         int64_t ld_x, int64_t ld_dw, void* workspace, int64_t ws_bytes,
                                         const uint8_t* tile_live, nf_stream_t stream) {
    if (B < 0 || N < 1 || K < 1 || ld_dy < N || ld_x < K || ld_dw < K) return NF_ERR_BAD_SHAPE;
    if (B > 2147483647LL - 64 || N > 2147483647LL - 128 || K > 2147483647LL - 128) return NF_ERR_BAD_SHAPE;
    NF_REQ(dw);
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t rblocks = cdiv(N * K, 256);
    const int rgrid = (int)(rblocks < (int64_t)kNumSMs * 8 ? rblocks : (int64_t)kNumSMs * 8);
    if (B == 0) {
        wgrad_reduce_kernel<<<rgrid, 256, 0, st>>>(nullptr, (float*)dw, (int)N, (int)K, ld_dw, 0, 0);
        count_launch();
        NF_LAUNCH_CHECK();
        return NF_OK;
    }
    NF_REQ(dy); NF_REQ(x);
    if (!aligned16(x) || (ld_x % 4) != 0) return NF_ERR_UNSUPPORTED;
    const bool direct = !aligned16(dy) || (ld_dy % 4) != 0;          // dY through plain loads instead of TMA
    int splits, per, nkb;
    wg_plan(B, N, K, &splits, &per, &nkb);
    if (splits > 1) {
        NF_REQ(workspace);
        if (ws_bytes < (int64_t)splits * N * K * 4) return NF_ERR_WORKSPACE;
    }
    alignas(64) CUtensorMap tg, tx;
    if (!wg_make_map(&tx, x, B, K, ld_x, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) return NF_ERR_UNSUPPORTED;
    if (direct) tg = tx;                                              // unused by the kernel in direct mode
    else if (!wg_make_map(&tg, dy, B, N, ld_dy, CU_TENSOR_MAP_SWIZZLE_128B)) return NF_ERR_UNSUPPORTED;
    const size_t smem = (size_t)kWgStages * kWgStageBytes + 256;
    NF_CUDA(cudaFuncSetAttribute(wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    NF_CUDA(cudaFuncSetAttribute(wgrad_tc_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    const int64_t tiles = cdiv(N, kWgBM) * cdiv(K, kWgBN);
    if (tiles > 2147483647LL) return NF_ERR_BAD_SHAPE;
    float* out = splits > 1 ? (float*)workspace : (float*)dw;
    const int64_t ld_out = splits > 1 ? K : ld_dw;
    wgrad_tc_kernel<<<dim3((unsigned)tiles, (unsigned)splits), kWgThreads, smem, st>>>(tg, tx, out, (int)N, (int)K, nkb, per, ld_out,
                                                                                         (int64_t)N * K, tile_live, direct ? (const float*)dy : nullptr, ld_dy, B, g_tc_passes,
                                                                                         (aligned32(out) && (ld_out % 8) == 0 && (((int64_t)N * K) % 8) == 0) ? 1 : 0);
    count_launch();
    NF_LAUNCH_CHECK();
    if (splits > 1) {
        if (splits >= 16 && N * K <= 65536)
            wgrad_reduce_wide_kernel<<<(unsigned)cdiv(N * K, 32), 256, 0, st>>>((const float*)workspace, (float*)dw, (int)N, (int)K, ld_dw, splits, (int64_t)N * K);
        else
        wgrad_reduce_kernel<<<rgrid, 256, 0, st>>>((const float*)workspace, (float*)dw, (int)N, (int)K, ld_dw, splits, (int64_t)N * K);
        count_launch();
        NF_LAUNCH_CHECK();
    }
    return NF_OK;
}
