// gemm_tc2.cu -- dense layer on the 5th-gen tensor cores:  Y[M,N] = act(X[M,K] * W[N,K]^T + bias), 3xTF32 on tcgen05
// with SHORT accumulation chains (nf_linear_tc / nf_linear_tc_range; W pre-split into W_hi / W_lo by nf_split_tf32).
//   (F.linear of MaskedLinear / MADE, masked_linear.py:14-18, made.py:136-140, and of the coupling / spline
//    conditioner MLPs, coupling_layer.py:18-35, spline_coupling_layer.py:55-62)
//
// Why: the tensor core truncates its fp32 accumulator on every MMA, so the error of a TMEM accumulation chain grows
// linearly with its length (DESIGN.md: K = 1024 -> 384 MMAs -> rms 7e-6 of rms(y), 12x an FFMA GEMM, and a coherent
// log-det bias of 4e-4 over a 784-dim spline layer).  Here a chain is at most kChainKB = 2 K-blocks (24 MMAs, the
// K = 64 error class) whatever K is: the MMA warp rotates over three TMEM accumulators, and four *drainer* warps
// fold every finished chain into fp32 registers with round-to-nearest adds -- thread r keeps row r's 128 running sums
// in registers for the whole tile, so the epilogue (bias, ReLU, store) comes straight from registers.
//
// One persistent CTA per SM (the 512 TMEM columns hold three 128-column chain accumulators and two A stages), 10 warps:
//   warp 0      TMA producer: X tile [128x32] and W_hi / W_lo tiles [128x32] per stage, 4 stages, running across tiles
//   warp 1      MMA issuer: 12 tcgen05.mma per K block (A from TMEM, B from shared memory), commits stage / A-stage /
//               chain barriers
//   warps 2-5   converters: split the X tile into hi / lo and store it into the TMEM A stage (lane = row)
//   warps 6-9   drainers: stage the tile's bias in shared memory and start the row's 128 running sums from it;
//               tcgen05.ld every finished chain accumulator, add it into the registers, release it; after the tile's
//               last chain: ReLU + sixteen 256-bit stores into the thread's own output row (no transpose, no loads),
//               overlapping the next tile's main loop
// passes == 1 (nf_set_option(7, 1), the reduced-precision mode): one TF32 pass, no W_lo loads, 6 stages of 32 KB,
// chains of 6 K blocks.
#include <cuda.h>
#include "nf_common.cuh"
#include "tc_common.cuh"

namespace nf {

constexpr int k2BM = 128, k2BN = 128, k2BK = 32;
constexpr int k2Stages = 4;                   // 3xTF32: 4 stages of X | W_hi | W_lo (48 KB)
constexpr int k2StagesFast = 6;               // one pass: 6 stages of X | W_hi (32 KB) in the same 192 KB
constexpr int k2MaxStages = 6;
constexpr int k2Threads = 320;
constexpr int k2ThreadsDirect = 448;          // two drainer groups
constexpr int k2ChainKB = 2;                  // K blocks per TMEM accumulation chain
constexpr int k2NAcc = 3;                     // chain accumulators in flight (drain latency hides behind two chains)
constexpr int k2AStages = 2;                  // TMEM A stages (hi 32 + lo 32 columns each)
constexpr int k2TmemCols = 512;               // D0: 0 | D1: 128 | D2: 256 | A stage 0: 384 (hi 32 + lo 32) | A stage 1: 448
constexpr int k2ColA = k2NAcc * 128;
static_assert(k2ColA + k2AStages * 64 == k2TmemCols, "TMEM split");
// nf_set_option(10, 1), one-pass mode only: feed the X tile to the MMA straight from shared memory (SS form; the tensor
// core then TRUNCATES x to TF32 instead of the converters' round-to-nearest) -- no converter work at all.
int g_gemm_tc2_ss = 0;
constexpr uint32_t k2XBytes = k2BM * k2BK * 4, k2WBytes = k2BN * k2BK * 4;
constexpr uint32_t k2StageBytes = k2XBytes + 2 * k2WBytes;
// per drainer group: two 128-float bias tiles (aligned outputs) OR four per-warp [32][33] transpose buffers (unaligned ones)
constexpr uint32_t k2TbufBytes = 4 * 32 * 33 * 4;

// nf_set_option(7, v): tensor-core passes per product.  3 = 3xTF32 (fp32 parity, default); 1 = one TF32 pass (operands
// rounded to nearest TF32, 10-bit mantissa: the documented reduced-precision mode for the conditioner GEMMs -- three
// more mantissa bits than bf16, no W_lo traffic, no lo conversions; chains of k2ChainKBFast K blocks = the same 24 MMAs)
int g_tc_passes = 3;
constexpr int k2ChainKBFast = 6;

__device__ __forceinline__ void tma2_load_2d(void* smem_dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(tc::smem_u32(smem_dst)), "l"(map), "r"(c0), "r"(c1), "r"(tc::smem_u32(bar)) : "memory");
}

// tile t -> (column block, row block).  Column blocks rotate with the row block: with k_extent (block-triangular MADE
// weights) the K length depends on the column block, and a CTA's tiles t, t + gridDim.x, ... would otherwise all fall on
// the same column block whenever gridDim.x is a multiple of n_tiles (148 = 4 * 37: measured +23 % on the C3 chain).
// Consecutive tiles still share their X row block (L2 reuse).
__device__ __forceinline__ void tile_decode(int t, int n_tiles, int& n0, int& m0) {
    const int mt = t / n_tiles;
    const int nt = (t - mt * n_tiles + mt) % n_tiles;
    n0 = nt * k2BN; m0 = mt * k2BM;
}

// K-block range [kb_first, kb_first + nkb) of the output tile starting at column n0
__device__ __forceinline__ void tile_k_range(int n0, int N, int K, const int32_t* __restrict__ k_extent,
                                             const int32_t* __restrict__ k_begin, int& kb_first, int& nkb) {
    int k_end = K;
    if (k_extent) {
        int e = 0;
        for (int c = n0 / 64; c <= (n0 + k2BN - 1) / 64 && c * 64 < N; ++c) e = max(e, k_extent[c]);
        k_end = min(K, e);
    }
    kb_first = 0;
    if (k_begin) {
        int b = K;
        for (int c = n0 / 64; c <= (n0 + k2BN - 1) / 64 && c * 64 < N; ++c) b = min(b, k_begin[c]);
        kb_first = max(0, min(b, k_end)) / k2BK;
    }
    nkb = max(0, (k_end + k2BK - 1) / k2BK - kb_first);
}

// DIRECT = true: contractions of at most 128 (<= 4 K blocks = one short chain per tile).  No register accumulation is
// needed, so the drainers write each tile straight from TMEM and there are two drainer groups (warps 6-9 and 10-13)
// taking alternate tiles: for small K the tile's epilogue (64 KB of output) is longer than its main loop, and a
// non-persistent kernel pays launch, TMEM allocation and pipeline fill per tile (measured with the first, one-chain-per-
// tile kernel at 2^20 x 64 x 64: 0.22 ms = 2.4 TB/s of a 0.08 ms HBM floor).
template <bool DIRECT>
__global__ void __launch_bounds__(DIRECT ? k2ThreadsDirect : k2Threads, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_wh,
                const __grid_constant__ CUtensorMap tm_wl, float* __restrict__ Y, const float* __restrict__ bias,
                int M, int N, int K, int64_t ldc, int relu, const int32_t* __restrict__ k_extent,
                const int32_t* __restrict__ k_begin, int num_tiles, int passes, int vec, int ss, int accumulate, int w_box_rows) {
    // accumulate (DIRECT + vec only, checked on the host): Y += X W^T instead of Y = ... (the blocked sampler's push of a
    // finished block of layer-3 units into the output-layer pre-activations of all later dims)
    extern __shared__ __align__(1024) uint8_t smem[];
    const int chain_kb = passes == 1 ? k2ChainKBFast : k2ChainKB;
    const int n_stages = passes == 1 ? k2StagesFast : k2Stages;
    const uint32_t stage_bytes = passes == 1 ? k2XBytes + k2WBytes : k2StageBytes;
    uint8_t* tbuf_base = smem + k2Stages * k2StageBytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(tbuf_base + (DIRECT ? 2 : 1) * k2TbufBytes);
    uint64_t* full = bars;                         // [S] TMA landed
    uint64_t* empty = full + k2MaxStages;          // [S] stage consumed (MMA commit)
    uint64_t* a_full = empty + k2MaxStages;        // [A] converters wrote the TMEM A stage
    uint64_t* a_empty = a_full + k2AStages;        // [A] MMAs consumed the TMEM A stage
    uint64_t* d_full = a_empty + k2AStages;        // [NAcc] chain accumulator complete
    uint64_t* d_empty = d_full + k2NAcc;           // [NAcc] drainers read the chain accumulator
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(d_empty + k2NAcc);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_tiles = (N + k2BN - 1) / k2BN;

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < k2MaxStages; ++i) { tc::mbar_init(&full[i], 1); tc::mbar_init(&empty[i], 1); }
        for (int i = 0; i < k2AStages; ++i) { tc::mbar_init(&a_full[i], 128); tc::mbar_init(&a_empty[i], 1); }
        for (int i = 0; i < k2NAcc; ++i) { tc::mbar_init(&d_full[i], 1); tc::mbar_init(&d_empty[i], 128); }
        tc::fence_mbar_init();
    }
    if (warp == 1) tc::tmem_alloc(tmem_slot, k2TmemCols);
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tb = *tmem_slot;

    if (warp == 0) {
        // ---------------- TMA producer ----------------
        if (lane == 0) {
            // stage index / round parity kept incrementally (n_stages is a run-time value: no div / mod per K block)
            // narrow outputs (N < 128, one column tile): the W boxes hold only the live rows (w_box_rows), see gemm_tc2_launch
            const uint32_t tx_bytes = k2XBytes + (passes == 1 ? 1u : 2u) * (uint32_t)w_box_rows * (k2BK * 4);
            int s = 0;
            uint32_t ph = 0;
            bool first_round = true;
            for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
                int n0, m0;
                tile_decode(t, n_tiles, n0, m0);
                int kb_first, nkb;
                tile_k_range(n0, N, K, k_extent, k_begin, kb_first, nkb);
                for (int kb = 0; kb < nkb; ++kb) {
                    if (!first_round) tc::mbar_wait(&empty[s], ph ^ 1u);
                    uint8_t* st = smem + s * stage_bytes;
                    tc::mbar_arrive_expect_tx(&full[s], tx_bytes);
                    tma2_load_2d(st, &tm_x, (kb_first + kb) * k2BK, m0, &full[s]);
                    tma2_load_2d(st + k2XBytes, &tm_wh, (kb_first + kb) * k2BK, n0, &full[s]);
                    if (passes != 1) tma2_load_2d(st + k2XBytes + k2WBytes, &tm_wl, (kb_first + kb) * k2BK, n0, &full[s]);
                    if (++s == n_stages) { s = 0; ph ^= 1u; first_round = false; }
                }
            }
        }
    } else if (warp == 1) {
        // ---------------- MMA issuer (whole warp, convergent; one elected lane issues) ----------------
        const bool leader = tc::elect_one();
        int it = 0, s = 0, ic = 0, cb = 0;               // K-block counter, stage, position in the chain, accumulator
        uint32_t ph = 0, dph = 0;                        // parity of the stage round / of the accumulator round
        bool first_acc_round = true;
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
            int n0, m0;
            tile_decode(t, n_tiles, n0, m0);
            (void)m0;
            int kb_first, nkb;
            tile_k_range(n0, N, K, k_extent, k_begin, kb_first, nkb);
            // narrow tiles (column slices of the blocked sampler, 2*D-wide heads): the MMA covers only the live columns,
            // rounded up to the instruction's N granularity of 16 -- its cost is proportional to N
            const uint32_t idesc = tc::idesc_tf32_m128((uint32_t)((min(k2BN, N - n0) + 15) & ~15));
            for (int kb = 0; kb < nkb; ++kb, ++it) {
                const int a = it & (k2AStages - 1);
                if (ic == 0 && !first_acc_round) tc::mbar_wait(&d_empty[cb], dph ^ 1u);
                tc::mbar_wait(&full[s], ph);
                if (!ss) tc::mbar_wait(&a_full[a], (it >> 1) & 1);
                tc::fence_after_sync();
                const uint32_t st = tc::smem_u32(smem + s * stage_bytes);
                const uint64_t d_hi = tc::smem_desc_k_sw128(st + k2XBytes), d_lo = tc::smem_desc_k_sw128(st + k2XBytes + k2WBytes);
                const uint32_t a_hi = tb + k2ColA + a * 64, a_lo = a_hi + 32;
                const uint32_t dcol = tb + cb * 128;
                if (ss) {
                    const uint64_t d_x = tc::smem_desc_k_sw128(st);          // the X tile as landed by TMA: K-major SWIZZLE_128B
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        if (leader) tc::mma_tf32_ss(dcol, d_x + (uint64_t)(k * 2), d_hi + (uint64_t)(k * 2), idesc, (ic | k) != 0 ? 1u : 0u);
                    }
                } else {
#pragma unroll
                    for (int pass = 0; pass < 3; ++pass) {
                        if (pass >= passes) break;
                        const uint32_t ac = (pass == 1) ? a_lo : a_hi;
                        const uint64_t wd = (pass == 2) ? d_lo : d_hi;
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            if (leader) tc::mma_tf32_ts(dcol, ac + k * 8, wd + (uint64_t)(k * 2), idesc, (ic | pass | k) != 0 ? 1u : 0u);
                        }
                    }
                }
                const bool chain_end = (!DIRECT && ic == chain_kb - 1) || (kb == nkb - 1);
                if (leader) {
                    tc::mma_commit(&empty[s]);
                    if (!ss) tc::mma_commit(&a_empty[a]);
                    if (chain_end) tc::mma_commit(&d_full[cb]);
                }
                __syncwarp();
                if (++s == n_stages) { s = 0; ph ^= 1u; }
                if (chain_end) {
                    ic = 0;
                    if (++cb == k2NAcc) { cb = 0; dph ^= 1u; first_acc_round = false; }
                } else {
                    ++ic;
                }
            }
        }
    } else if (warp < 6) {
        // ---------------- converters (warps 2..5; TMEM lane quadrant = warp % 4) ----------------
        const int q = warp & 3;
        const int r = q * 32 + lane;
        const uint32_t lane_addr = tb + ((uint32_t)(q * 32) << 16);
        int it = 0, s = 0;
        uint32_t ph = 0;
        for (int t = blockIdx.x; t < (ss ? 0 : num_tiles); t += gridDim.x) {       // SS form: no converter work
            int n0, m0;
            tile_decode(t, n_tiles, n0, m0);
            (void)m0;
            int kb_first, nkb;
            tile_k_range(n0, N, K, k_extent, k_begin, kb_first, nkb);
            for (int kb = 0; kb < nkb; ++kb, ++it) {
                const int a = it & (k2AStages - 1);
                tc::mbar_wait(&full[s], ph);
                if (it >= k2AStages) tc::mbar_wait(&a_empty[a], ((it >> 1) - 1) & 1);
                tc::fence_after_sync();
                const uint8_t* xrow = smem + s * stage_bytes + (r >> 3) * 1024 + (r & 7) * 128;
                uint32_t hi[32], lo[32];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const float4 v = *reinterpret_cast<const float4*>(xrow + ((c ^ (r & 7)) << 4));
                    tc::split_tf32(v.x, hi[4 * c + 0], lo[4 * c + 0]);
                    tc::split_tf32(v.y, hi[4 * c + 1], lo[4 * c + 1]);
                    tc::split_tf32(v.z, hi[4 * c + 2], lo[4 * c + 2]);
                    tc::split_tf32(v.w, hi[4 * c + 3], lo[4 * c + 3]);
                }
                const uint32_t a_hi = lane_addr + k2ColA + a * 64, a_lo = a_hi + 32;
                {
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
                tc::wait_st();
                tc::fence_before_sync();
                tc::mbar_arrive(&a_full[a]);
                if (++s == n_stages) { s = 0; ph ^= 1u; }
            }
        }
    } else if constexpr (DIRECT) {
        // ---------------- two drainer groups (warps 6..9, 10..13), alternate tiles, straight from TMEM ----------------
        const int q = warp & 3, grp = (warp - 6) >> 2;
        const uint32_t lane_addr = tb + ((uint32_t)(q * 32) << 16);
        int cc = 0, ti = 0;
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++ti) {
            int n0, m0;
            tile_decode(t, n_tiles, n0, m0);
            int kb_first, nkb;
            tile_k_range(n0, N, K, k_extent, k_begin, kb_first, nkb);
            const int my_cc = cc;
            if (nkb > 0) ++cc;                                   // one chain per non-empty tile, counted by both groups
            if ((ti & 1) != grp) continue;
            const int cb = my_cc % k2NAcc;
            // aligned outputs: bias tile -> shared memory (two buffers per group, alternating with the group's tiles);
            // unaligned outputs: the same memory is the warps' transpose buffers
            float* grp_mem = reinterpret_cast<float*>(tbuf_base) + grp * (k2TbufBytes / 4);
            float* bias_s = grp_mem + ((ti >> 1) & 1) * 128;
            float* tbuf = grp_mem + (size_t)(warp - 6 - 4 * grp) * 32 * 33;
            if (vec) tc::stage_bias_tile(bias_s, bias, n0, N, (warp - 6 - 4 * grp) * 32 + lane, 1 + grp);
            if (nkb > 0) {
                tc::mbar_wait(&d_full[cb], (my_cc / k2NAcc) & 1);
                tc::fence_after_sync();
            }
            const int row = m0 + q * 32 + lane;
            float* yrow = Y + (int64_t)row * ldc;
            const int n_live = min(k2BN, N - n0);                 // columns past it are neither multiplied nor stored
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const bool live = c * 32 < n_live;                // CTA-uniform
                uint32_t v0[16], v1[16];
                float old[32];
                if (live && accumulate) {
                    // requested ahead of the accumulator wait; rows past M / columns past N read as zero
#pragma unroll
                    for (int h = 0; h < 4; ++h) {
                        const int col = n0 + c * 32 + 8 * h;
                        if (row < M && col + 8 <= N) {
                            const float4 o0 = *reinterpret_cast<const float4*>(yrow + col);
                            const float4 o1 = *reinterpret_cast<const float4*>(yrow + col + 4);
                            old[8 * h + 0] = o0.x; old[8 * h + 1] = o0.y; old[8 * h + 2] = o0.z; old[8 * h + 3] = o0.w;
                            old[8 * h + 4] = o1.x; old[8 * h + 5] = o1.y; old[8 * h + 6] = o1.z; old[8 * h + 7] = o1.w;
                        } else {
#pragma unroll
                            for (int i = 0; i < 8; ++i) old[8 * h + i] = (row < M && col + i < N) ? yrow[col + i] : 0.f;
                        }
                    }
                }
                if (nkb > 0) {
                    if (live) {
                        tc::tmem_ld16(lane_addr + cb * 128 + c * 32, v0);
                        tc::tmem_ld16(lane_addr + cb * 128 + c * 32 + 16, v1);
                        tc::wait_ld();
                    }
                    if (c == 3) { tc::fence_before_sync(); tc::mbar_arrive(&d_empty[cb]); }     // accumulator free again
                } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j) { v0[j] = 0u; v1[j] = 0u; }
                }
                if (!live) continue;
                if (accumulate) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        v0[j] = __float_as_uint(__uint_as_float(v0[j]) + old[j]);
                        v1[j] = __float_as_uint(__uint_as_float(v1[j]) + old[16 + j]);
                    }
                }
                if (vec) {
                    if (row < M) tc::epilogue_store32(yrow, n0 + c * 32, N, v0, v1, bias_s + c * 32, relu, vec);
                } else {
                    tc::epilogue_store32_transposed(Y, ldc, m0 + q * 32, M, n0 + c * 32, N, v0, v1, bias, relu, tbuf, lane);
                }
            }
        }
    } else {
        // ---------------- drainers (warps 6..9; TMEM lane quadrant = warp % 4), then the tile epilogue ----------------
        const int q = warp & 3;
        const uint32_t lane_addr = tb + ((uint32_t)(q * 32) << 16);
        int cb = 0, ti = 0;
        uint32_t dph = 0;
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++ti) {
            int n0, m0;
            tile_decode(t, n_tiles, n0, m0);
            int kb_first, nkb;
            tile_k_range(n0, N, K, k_extent, k_begin, kb_first, nkb);
            const int nchains = (nkb + chain_kb - 1) / chain_kb;
            // aligned outputs: bias tile -> shared memory while the first chain is still accumulating (two buffers,
            // alternating tiles) and the running sums START from the bias, so the epilogue has no loads at all;
            // unaligned outputs: sums start from zero and the same memory is the warps' transpose buffers
            float* bias_s = reinterpret_cast<float*>(tbuf_base) + (ti & 1) * 128;
            float* tbuf = reinterpret_cast<float*>(tbuf_base) + (size_t)(warp - 6) * 32 * 33;
            float acc[128];
            if (vec) {
                tc::stage_bias_tile(bias_s, bias, n0, N, (warp - 6) * 32 + lane, 1);
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float4 b = *reinterpret_cast<const float4*>(bias_s + 4 * j);
                    acc[4 * j + 0] = b.x; acc[4 * j + 1] = b.y; acc[4 * j + 2] = b.z; acc[4 * j + 3] = b.w;
                }
            } else {
#pragma unroll
                for (int j = 0; j < 128; ++j) acc[j] = 0.f;
            }
            const int n_live = min(k2BN, N - n0);                 // columns past it are neither multiplied nor stored
            for (int c = 0; c < nchains; ++c) {
                tc::mbar_wait(&d_full[cb], dph);
                tc::fence_after_sync();
#pragma unroll
                for (int ch = 0; ch < 8; ++ch) {
                    if (ch * 16 >= n_live) break;
                    uint32_t v[16];
                    tc::tmem_ld16(lane_addr + cb * 128 + ch * 16, v);
                    tc::wait_ld();
#pragma unroll
                    for (int j = 0; j < 16; ++j) acc[ch * 16 + j] += __uint_as_float(v[j]);      // round-to-nearest fp32 adds
                }
                tc::fence_before_sync();
                tc::mbar_arrive(&d_empty[cb]);
                if (++cb == k2NAcc) { cb = 0; dph ^= 1u; }
            }
            // epilogue from registers: the thread owns row m0 + 32q + lane; ReLU + one 256-bit store per 8 columns
            const int row = m0 + q * 32 + lane;
            if (vec) {
                if (row < M) {
                    float* yrow = Y + (int64_t)row * ldc;
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        float a[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) a[i] = acc[j * 8 + i];
                        tc::epilogue_store8(yrow, n0 + j * 8, N, a, relu, vec);
                    }
                }
            } else {
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    uint32_t v0[16], v1[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) { v0[j] = __float_as_uint(acc[c * 32 + j]); v1[j] = __float_as_uint(acc[c * 32 + 16 + j]); }
                    tc::epilogue_store32_transposed(Y, ldc, m0 + q * 32, M, n0 + c * 32, N, v0, v1, bias, relu, tbuf, lane);
                }
            }
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 1) tc::tmem_dealloc(tb, k2TmemCols);
}

// W ~= hi + lo: hi = W rounded to the nearest TF32, lo = (W - hi) rounded to the nearest TF32 (|W - hi - lo| <= 2^-24 |W|)
__global__ void split_tf32_kernel(const float* __restrict__ w, float* __restrict__ hi, float* __restrict__ lo, int64_t n) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        uint32_t h, l;
        tc::split_tf32_weight(w[i], h, l);
        hi[i] = __uint_as_float(h);
        lo[i] = __uint_as_float(l);
    }
}

static bool make_map2(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
    const tc::EncodeTiledFn fn = tc::encode_tiled_fn();
    if (!fn) return false;
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    cuuint32_t box[2] = {(cuuint32_t)k2BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// returns NF_OK when launched; NF_ERR_UNSUPPORTED when a tensor map cannot be encoded or `accumulate` is asked for
// outside its conditions
int gemm_tc2_launch(const void* x, const void* w_hi, const void* w_lo, const void* bias, void* y, int64_t M, int64_t N, int64_t K,
                    int64_t ldx, int64_t ldw, int64_t ldy, int relu, const int32_t* k_begin, const int32_t* k_extent,
                    cudaStream_t st, int accumulate) {
    alignas(64) CUtensorMap tx, twh, twl;
    // W boxes: 128 rows, or only the live rows of a narrow output (rounded up to the MMA's N granularity).  A 128-row box
    // over a tensor of fewer than 64 rows -- more than half of it out-of-bounds fill -- cost the column-slice GEMMs of the
    // blocked sampler 35-40 % (K = 448: N = 56 / 60 167 / 171 us against 124 us at N = 64, profiles/r02aw_slice_gemm.jsonl)
    const int wbox = N >= k2BN ? k2BN : (int)((N + 15) & ~15);
    if (!make_map2(&tx, x, M, K, ldx, k2BM) || !make_map2(&twh, w_hi, N, K, ldw, wbox) || !make_map2(&twl, w_lo, N, K, ldw, wbox))
        return NF_ERR_UNSUPPORTED;
    const int64_t tiles = cdiv(N, k2BN) * cdiv(M, k2BM);
    if (tiles > 2147483647LL) return NF_ERR_BAD_SHAPE;
    const int grid = (int)(tiles < kNumSMs ? tiles : kNumSMs);
    // row stores in the epilogue: 256-bit for 32-byte aligned rows of Y, 2 x 128-bit for 16-byte aligned ones
    const int vec = (aligned32(y) && (ldy % 8) == 0) ? 1 : ((aligned16(y) && (ldy % 4) == 0) ? 2 : 0);
    const int ss = (g_tc_passes == 1 && g_gemm_tc2_ss) ? 1 : 0;
    if (accumulate && (K > 4 * k2BK || !vec || bias != nullptr || relu)) return NF_ERR_UNSUPPORTED;
    if (K <= 4 * k2BK) {
        const size_t smem = (size_t)k2Stages * k2StageBytes + 2 * k2TbufBytes + 256;
        NF_CUDA(cudaFuncSetAttribute(gemm_tc2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        gemm_tc2_kernel<true><<<grid, k2ThreadsDirect, smem, st>>>(tx, twh, twl, (float*)y, (const float*)bias, (int)M, (int)N, (int)K,
                                                           ldy, relu, k_extent, k_begin, (int)tiles, g_tc_passes, vec, ss, accumulate, wbox);
    } else {
        const size_t smem = (size_t)k2Stages * k2StageBytes + k2TbufBytes + 256;
        NF_CUDA(cudaFuncSetAttribute(gemm_tc2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        gemm_tc2_kernel<false><<<grid, k2Threads, smem, st>>>(tx, twh, twl, (float*)y, (const float*)bias, (int)M, (int)N, (int)K, ldy,
                                                              relu, k_extent, k_begin, (int)tiles, g_tc_passes, vec, ss, accumulate, wbox);
    }
    return NF_OK;
}

}  // namespace nf

using namespace nf;
#define NF_REQ(p) do { if ((p) == nullptr) return NF_ERR_NULL; } while (0)

extern "C" int nf_split_tf32(const void* w, void* w_hi, void* w_lo, int64_t n, nf_stream_t stream) {
    if (n < 0) return NF_ERR_BAD_SHAPE;
    if (n == 0) return NF_OK;
    NF_REQ(w); NF_REQ(w_hi); NF_REQ(w_lo);
    int64_t need = cdiv(n, 256), cap = (int64_t)kNumSMs * 8;
    split_tf32_kernel<<<(int)(need < cap ? need : cap), 256, 0, (cudaStream_t)stream>>>((const float*)w, (float*)w_hi, (float*)w_lo, n);
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

extern "C" int nf_linear_tc_range(const void* x, const void* w_hi, const void* w_lo, const void* bias, void* y, int64_t M,
                                  int64_t N, int64_t K, int64_t ldx, int64_t ldw, int64_t ldy, int relu,
                                  const int32_t* k_begin, const int32_t* k_extent, nf_stream_t stream) {
    if (M < 0 || N < 1 || K < 1 || ldx < K || ldw < K || ldy < N) return NF_ERR_BAD_SHAPE;
    if (M == 0) return NF_OK;
    NF_REQ(x); NF_REQ(w_hi); NF_REQ(w_lo); NF_REQ(y);
    // TMA: 16-byte aligned bases and row pitches
    if (!aligned16(x) || !aligned16(w_hi) || !aligned16(w_lo) || (ldx % 4) != 0 || (ldw % 4) != 0) return NF_ERR_UNSUPPORTED;
    if (M > 2147483647LL - 128 || N > 2147483647LL - 128 || K > 2147483647LL - 64) return NF_ERR_BAD_SHAPE;
    const int rc = gemm_tc2_launch(x, w_hi, w_lo, bias, y, M, N, K, ldx, ldw, ldy, relu, k_begin, k_extent, (cudaStream_t)stream, 0);
    if (rc != NF_OK) return rc;
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

extern "C" int nf_linear_tc(const void* x, const void* w_hi, const void* w_lo, const void* bias, void* y, int64_t M,
                            int64_t N, int64_t K, int64_t ldx, int64_t ldw, int64_t ldy, int relu,
                            const int32_t* k_extent, nf_stream_t stream) {
    return nf_linear_tc_range(x, w_hi, w_lo, bias, y, M, N, K, ldx, ldw, ldy, relu, nullptr, k_extent, stream);
}
