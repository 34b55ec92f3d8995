// made_chain_bf16.cu -- the whole parallel direction of an affine autoregressive flow in ONE persistent launch, bf16
// operands on tcgen05 (kind::f16, fp32 accumulation in TMEM):
//     MAF.inverse / IAF.forward  =  MADE (4 masked linears, 3 ReLU; made.py:136-140) + affine-AR transform + row log-det
//     (masked_autoregressive_flow.py:18-44, inverse_autoregressive_flow.py:30-63) [+ the N(0,I) log-prob head, flow.py:56-73]
// This is the reduced-precision ("bf16 conditioner GEMMs") mode; the fp32-parity default stays the 3xTF32 GEMM chain.
//
// Why one kernel: unfused, the chain moves the [B, H] activations through HBM between every pair of GEMMs (~12.8 KB per
// row against 516 B of compulsory traffic at MAF(64, 512)).  Here a CTA owns 128 rows for the whole chain and the
// activations never leave the SM:
//     TMEM accumulator (fp32) -> tcgen05.ld -> +bias, ReLU, -> bf16 -> shared memory (K-major SWIZZLE_128B) = A operand
//     of the next layer's MMAs;
// only x (fp32, read once) and z / log-det (written once) touch HBM.  Weights (bf16, mask folded, hidden units sorted by
// degree so that every masked weight is block lower-triangular) stream from L2 through a TMA ring.
//
// Activation buffer: KA + 2 slots of one K atom each ([128 rows x 64 bf16] = 16 KB), addressed through a ROTATING map
//     slot(l, a) = (o + a + 2 l) mod (KA + 2)          (l = layer whose INPUT the atom is, a = atom, o = tile offset)
// Output blocks (128 columns = 2 atoms) of a layer are produced in DESCENDING order and written two slots "ahead" of the
// input atoms: block j's output lands where input atoms 2j+2, 2j+3 lived -- inputs that only output blocks >= j (+ the
// few "spill" columns of degree groups that straddle a block boundary, read by block j itself) still need, and those
// MMAs have completed when block j's accumulator is drained.  So the epilogue of block j overlaps the MMAs of block
// j-1, and the NEXT layer's first (widest) block can start on atoms 7, 6, ... as soon as they are written: the MMA warp
// issues one continuous stream of MMAs across layers and tiles.  The next tile's x goes to a slot that is free during the
// last layer (o' = o + 4).
//
// Warp roles (576 threads, one CTA per SM, all 512 TMEM columns = four 128-column accumulators):
//   warp 0      TMA producer: weight tiles [128 x 64] bf16, 3-stage ring, in (tile, layer, block desc., atom desc.) order
//   warp 1      MMA issuer (whole warp convergent, one elected lane): waits x / block-ready / stage-full / accumulator-empty
//   warps 2-17  epilogue: warp w drains TMEM lane quadrant w % 4, column quarter (w - 2) / 4 of each accumulator
#include <cuda.h>
#include <cuda_bf16.h>
#include "nf_common.cuh"
#include "stack_small.cuh"
#include "tc_common.cuh"

namespace nf {

constexpr int kMcRows = 128;                 // rows per CTA tile (UMMA M)
constexpr int kMcBN = 128;                   // output block width (UMMA N)
constexpr int kMcAtom = 64;                  // bf16 elements per K atom (128 bytes: one swizzle span)
constexpr int kMcAtomBytes = kMcRows * kMcAtom * 2;      // 16 KB: one activation slot = one weight stage
constexpr int kMcStages = 3;                 // 3 x 16 KB weight stages: the 4th stage's room holds the biases (see below)
constexpr int kMcMaxKA = 8;                  // hidden_dim <= 512
constexpr int kMcEpiWarps = 16;
constexpr int kMcThreads = 64 + 32 * kMcEpiWarps;
constexpr int kMcTmemCols = 512;

#ifdef NF_MC_PROFILE
// debug builds only (-DNF_MC_PROFILE): cycles CTA 0 spends waiting, per role and barrier
__device__ long long g_mc_prof[16];
#define MC_PROF_DECL long long pf_[8] = {0, 0, 0, 0, 0, 0, 0, 0}; const long long pf_start_ = clock64();
#define MC_WAIT(i, stmt) do { const long long t__ = clock64(); stmt; pf_[i] += clock64() - t__; } while (0)
#define MC_PROF_STORE(base, n) do { if (blockIdx.x == 0 && lane == 0) { for (int i__ = 0; i__ < (n); ++i__) g_mc_prof[(base) + i__] = pf_[i__]; \
                                                                      g_mc_prof[(base) + (n)] = clock64() - pf_start_; } } while (0)
#else
#define MC_PROF_DECL
#define MC_WAIT(i, stmt) do { stmt; } while (0)
#define MC_PROF_STORE(base, n) do { } while (0)
#endif

struct McParams {
    int kext16[4][4];       // [layer][block]: 16-wide k-steps the block's outputs depend on (monotone in block)
    int NB;                 // 128-column blocks of the hidden layers (H / 128)
    int KA;                 // K atoms of the hidden layers (H / 64)
    int D;                  // data_dim (<= 64, multiple of 4)
    int mode;               // NF_AR_MAF_INVERSE / NF_AR_IAF_FORWARD
    int flags;              // NF_STACK_LOG_PROB_HEAD | NF_STACK_SKIP_Y | NF_STACK_SAMPLE_LOG_Q semantics (bits 1, 2, 3)
    int64_t B;
    int num_tiles;
};

__device__ __forceinline__ void mc_tma_load_2d(void* smem_dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(tc::smem_u32(smem_dst)), "l"(map), "r"(c0), "r"(c1), "r"(tc::smem_u32(bar)) : "memory");
}
// instruction descriptor: kind::f16, A = B = bf16, fp32 accumulate, both K-major, M = 128
__host__ __device__ constexpr uint32_t mc_idesc_bf16(uint32_t N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((N >> 3) << 17) | ((128u >> 4) << 24);
}
__device__ __forceinline__ void mc_mma_bf16_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ uint32_t mc_pack_bf16(float lo, float hi) {
    const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);          // .x = lo (low 16 bits), .y = hi
    return *reinterpret_cast<const uint32_t*>(&v);
}
// max(x, 0) with NaN kept (torch.relu) and round-to-nearest bf16, two values per instruction (F2FP.RELU.BF16.F32.PACK_AB;
// cvt's .relu maps NaN to the canonical NaN and -0 / negatives to +0)
__device__ __forceinline__ uint32_t mc_pack_relu_bf16(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
// one 16-byte chunk (8 bf16) of row r of a K-major SWIZZLE_128B atom: chunk c sits at position c ^ (r % 8)
__device__ __forceinline__ void mc_store_chunk(uint8_t* atom, int r, int c, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3) {
    uint8_t* p = atom + (r >> 3) * 1024 + (r & 7) * 128 + ((c ^ (r & 7)) << 4);
    *reinterpret_cast<uint4*>(p) = make_uint4(w0, w1, w2, w3);
}

// (o + k) mod nslot for o < nslot, k <= 3 * nslot: conditional subtractions (a run-time `%` is a ~25-instruction division)
__device__ __forceinline__ int mc_slot(int o, int k, int nslot) {
    int s = o + k;
    if (s >= 2 * nslot) s -= 2 * nslot;
    if (s >= nslot) s -= nslot;
    if (s >= nslot) s -= nslot;
    return s;
}
__device__ __forceinline__ float mc_relu_keepnan(float x) {      // torch.relu: NaN stays NaN
    float r;
    asm("max.NaN.f32 %0, %1, 0f00000000;" : "=f"(r) : "f"(x));
    return r;
}

__global__ void __launch_bounds__(kMcThreads, 1)
made_chain_bf16_kernel(const __grid_constant__ CUtensorMap tm_w0, const __grid_constant__ CUtensorMap tm_w1,
                       const __grid_constant__ CUtensorMap tm_w2, const __grid_constant__ CUtensorMap tm_w3,
                       const float* __restrict__ x, const float* __restrict__ b0, const float* __restrict__ b1,
                       const float* __restrict__ b2, const float* __restrict__ b3, float* __restrict__ out,
                       float* __restrict__ ld_out, const __grid_constant__ McParams P) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int NSLOT = P.KA + 2;
    uint8_t* act = smem;                                           // NSLOT activation slots
    uint8_t* wst = smem + (size_t)NSLOT * kMcAtomBytes;            // kMcStages weight stages
    // all biases (b0 | b1 | b2 | b3: 3 H + 128 floats) staged once: the first version fetched them with __ldg in front of
    // every use -- two 16-byte loads at a time for want of registers -- and the epilogue warps, the critical path of the
    // kernel, spent a quarter of their samples waiting on those loads (profiles/r02b_made_chain_bf16_ncu.txt)
    float* bias_s = reinterpret_cast<float*>(wst + (size_t)kMcStages * kMcAtomBytes);
    const int H = P.KA * kMcAtom;
    uint64_t* bars = reinterpret_cast<uint64_t*>(bias_s + 3 * H + 128);
    uint64_t* w_full = bars;                    // [kMcStages]
    uint64_t* w_empty = w_full + kMcStages;     // [kMcStages]
    uint64_t* acc_full = w_empty + kMcStages;   // [4]
    uint64_t* acc_empty = acc_full + 4;         // [4]
    uint64_t* blk_ready = acc_empty + 4;        // [4] block jb of the current layer's input activations written
    uint64_t* x_ready = blk_ready + 4;          // [1]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(x_ready + 1);
    float* row_part = reinterpret_cast<float*>(tmem_slot + 2);     // [2 tile parities][3 column quarters][2 values][128 rows]
    int* kext_s = reinterpret_cast<int*>(row_part + 2 * 3 * 256);  // [4 layers][4 blocks]: P.kext16 (dynamic indexing of a
                                                                   // __grid_constant__ struct member goes through local memory)

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int NB = P.NB;

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < kMcStages; ++i) { tc::mbar_init(&w_full[i], 1); tc::mbar_init(&w_empty[i], 1); }
        for (int i = 0; i < 4; ++i) {
            tc::mbar_init(&acc_full[i], 1); tc::mbar_init(&acc_empty[i], kMcEpiWarps); tc::mbar_init(&blk_ready[i], kMcEpiWarps);
        }
        tc::mbar_init(x_ready, kMcEpiWarps);
        tc::fence_mbar_init();
    }
    if (warp == 1) tc::tmem_alloc(tmem_slot, kMcTmemCols);
    if (tid < 16) kext_s[tid] = P.kext16[tid >> 2][tid & 3];
    for (int i = tid; i < 3 * H + 128; i += kMcThreads)
        bias_s[i] = i < H ? __ldg(b0 + i) : (i < 2 * H ? __ldg(b1 + i - H) : (i < 3 * H ? __ldg(b2 + i - 2 * H) : __ldg(b3 + i - 3 * H)));
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tb = *tmem_slot;

    if (warp == 0) {
        // ---------------- weight producer ----------------
        if (lane == 0) {
            MC_PROF_DECL
            int s = 0;
            uint32_t ph = 0;
            bool first_round = true;
            for (int t = blockIdx.x; t < P.num_tiles; t += gridDim.x) {
                for (int l = 0; l < 4; ++l) {
                    const CUtensorMap* map = l == 0 ? &tm_w0 : (l == 1 ? &tm_w1 : (l == 2 ? &tm_w2 : &tm_w3));
                    const int nblk = (l == 3) ? 1 : NB;
                    for (int j = nblk - 1; j >= 0; --j) {
                        const int na = (kext_s[l * 4 + j] + 3) >> 2;
                        for (int a = na - 1; a >= 0; --a) {
                            if (!first_round) MC_WAIT(0, tc::mbar_wait(&w_empty[s], ph ^ 1u));
                            tc::mbar_arrive_expect_tx(&w_full[s], (uint32_t)kMcAtomBytes);
                            mc_tma_load_2d(wst + (size_t)s * kMcAtomBytes, map, a * kMcAtom, j * kMcBN, &w_full[s]);
                            if (++s == kMcStages) { s = 0; ph ^= 1u; first_round = false; }
                        }
                    }
                }
            }
            MC_PROF_STORE(0, 1);           // [0] producer waits for a free stage, [1] producer total
        }
    } else if (warp == 1) {
        // ---------------- MMA issuer ----------------
        const uint32_t idesc = mc_idesc_bf16((uint32_t)kMcBN);
        const bool leader = tc::elect_one();
        MC_PROF_DECL
        int s = 0, u = 0, it = 0, o = 0;                   // weight stage, unit counter (accumulator ring), tile iteration, slot offset
        uint32_t ph = 0;
        for (int t = blockIdx.x; t < P.num_tiles; t += gridDim.x, ++it) {
            for (int l = 0; l < 4; ++l) {
                const int nblk = (l == 3) ? 1 : NB;
                uint32_t ready = 0;                            // input blocks of this layer already waited for
                if (l == 0) MC_WAIT(0, tc::mbar_wait(x_ready, (uint32_t)(it & 1)));
                for (int j = nblk - 1; j >= 0; --j, ++u) {
                    const int acc = u & 3;
                    if (u >= 4) MC_WAIT(1, tc::mbar_wait(&acc_empty[acc], (uint32_t)(((u >> 2) & 1) ^ 1)));
                    const int k16 = kext_s[l * 4 + j];
                    const int na = (k16 + 3) >> 2;
                    const uint32_t dcol = tb + (uint32_t)(acc * kMcBN);
                    bool first = true;
                    for (int a = na - 1; a >= 0; --a) {
                        if (l > 0) {
                            const int jb = a >> 1;
                            if (!(ready & (1u << jb))) {
                                // h_l block jb: completion number 3*it + (l-1) of blk_ready[jb]
                                MC_WAIT(2, tc::mbar_wait(&blk_ready[jb], (uint32_t)((3 * it + (l - 1)) & 1)));
                                ready |= 1u << jb;
                            }
                        }
                        MC_WAIT(3, tc::mbar_wait(&w_full[s], ph));
                        tc::fence_after_sync();
                        const int slot = mc_slot(o, a + 2 * l, NSLOT);
                        const uint64_t da = tc::smem_desc_k_sw128(tc::smem_u32(act + (size_t)slot * kMcAtomBytes));
                        const uint64_t db = tc::smem_desc_k_sw128(tc::smem_u32(wst + (size_t)s * kMcAtomBytes));
                        const int nk = min(4, k16 - 4 * a);
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            if (k < nk && leader)
                                mc_mma_bf16_ss(dcol, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (first && k == 0) ? 0u : 1u);
                        }
                        first = false;
                        if (leader) tc::mma_commit(&w_empty[s]);
                        __syncwarp();
                        if (++s == kMcStages) { s = 0; ph ^= 1u; }
                    }
                    if (leader) tc::mma_commit(&acc_full[acc]);      // na == 0 (all-zero block): completes at once, accumulator unread
                    __syncwarp();
                }
            }
            o = mc_slot(o, 4, NSLOT);
        }
        MC_PROF_STORE(2, 4);               // [2] x ready, [3] accumulator empty, [4] input block ready, [5] weight stage full, [6] MMA warp total
    } else {
        // ---------------- epilogue warps ----------------
        // 16 warps: warp w drains TMEM lane quadrant w % 4, column quarter cq = (w - 2) / 4 (32 of a block's 128 columns).
        // The first version had 8 warps with 64 columns each: ~220 dependent instructions per unit at two warps per
        // scheduler took ~2 400 clk per unit against ~1 000 clk of MMAs -- the MMA warp spent a third of its time waiting
        // for a free accumulator (profiles/r02d_chain_phase.log).
        const int q = warp & 3, cq = (warp - 2) >> 2;
        const int r = q * 32 + lane;                                   // row inside the tile = TMEM lane
        const uint32_t lane_addr = tb + ((uint32_t)(q * 32) << 16);
        const int D = P.D;
        const bool iaf = (P.mode == AR_IAF_FWD);
        const float lim = iaf ? 50.f : 100.f;
        const int c0 = cq * 16;                                        // this thread's 16 data columns
        float xc[16], xn[16];
        // byte offsets of this thread's row and of its four 16-byte chunks inside a SWIZZLE_128B atom (constant per thread)
        const uint32_t row_off = (uint32_t)((r >> 3) * 1024 + (r & 7) * 128);
        uint32_t chunk_off[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) chunk_off[c] = (uint32_t)((((cq & 1) * 4 + c) ^ (r & 7)) << 4);

        auto load_x = [&](int tile, float (&v)[16]) {
            const int64_t row = (int64_t)tile * kMcRows + r;
            const bool ok = tile < P.num_tiles && row < P.B;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
                if (ok && c0 + 4 * i < D) f = __ldcs(reinterpret_cast<const float4*>(x + row * D + c0 + 4 * i));
                v[4 * i + 0] = f.x; v[4 * i + 1] = f.y; v[4 * i + 2] = f.z; v[4 * i + 3] = f.w;
            }
        };
        auto write_x = [&](const float (&v)[16], int slot) {
            uint8_t* atom = act + (size_t)slot * kMcAtomBytes;
#pragma unroll
            for (int c = 0; c < 2; ++c)
                mc_store_chunk(atom, r, cq * 2 + c, mc_pack_bf16(v[8 * c + 0], v[8 * c + 1]), mc_pack_bf16(v[8 * c + 2], v[8 * c + 3]),
                               mc_pack_bf16(v[8 * c + 4], v[8 * c + 5]), mc_pack_bf16(v[8 * c + 6], v[8 * c + 7]));
            tc::fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(x_ready);
        };

        MC_PROF_DECL
        int u = 0, it = 0, o = 0;
        load_x(blockIdx.x, xc);
        if ((int)blockIdx.x < P.num_tiles) write_x(xc, 0);
        for (int t = blockIdx.x; t < P.num_tiles; t += gridDim.x, ++it) {
            load_x(t + gridDim.x, xn);                                  // in flight during layers 0..2
            for (int l = 0; l < 3; ++l) {
                const float* bias = bias_s + l * H;
                for (int j = NB - 1; j >= 0; --j, ++u) {
                    const int acc = u & 3;
                    // The epilogue is the critical path (13 units x ~2 000 clk per tile against ~1 000 clk of MMAs per unit,
                    // profiles/r02e_chain_phase.log) and it is ISSUE-bound: 16 warps x ~180 instructions per unit over four
                    // schedulers.  So the unit body is pared down: per-thread store offsets precomputed, bias added with
                    // packed f32x2 adds (FADD2), ReLU folded into the bf16 pack (F2FP.RELU), no zero-fill path (the host
                    // guarantees at least one k-step per block).
                    MC_WAIT(0, tc::mbar_wait(&acc_full[acc], (uint32_t)((u >> 2) & 1)));
                    tc::fence_after_sync();
                    uint32_t v[2][16];
                    tc::tmem_ld16(lane_addr + (uint32_t)(acc * kMcBN + cq * 32), v[0]);
                    tc::tmem_ld16(lane_addr + (uint32_t)(acc * kMcBN + cq * 32 + 16), v[1]);
                    tc::wait_ld();
                    tc::fence_before_sync();
                    __syncwarp();
                    if (lane == 0) tc::mbar_arrive(&acc_empty[acc]);
                    // columns [32 cq, 32 cq + 32) of h_{l+1} block j = chunks 4 (cq & 1) .. + 3 of atom 2j + cq / 2
                    uint8_t* dst = act + (size_t)mc_slot(o, (2 * j + (cq >> 1)) + 2 * (l + 1), NSLOT) * kMcAtomBytes + row_off;
                    const float4* bp = reinterpret_cast<const float4*>(bias + j * kMcBN + cq * 32);
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const float4 b0 = bp[2 * c], b1 = bp[2 * c + 1];
                        const uint32_t* vv = &v[c >> 1][(c & 1) * 8];
                        const float2 f0 = __fadd2_rn(make_float2(__uint_as_float(vv[0]), __uint_as_float(vv[1])), make_float2(b0.x, b0.y));
                        const float2 f1 = __fadd2_rn(make_float2(__uint_as_float(vv[2]), __uint_as_float(vv[3])), make_float2(b0.z, b0.w));
                        const float2 f2 = __fadd2_rn(make_float2(__uint_as_float(vv[4]), __uint_as_float(vv[5])), make_float2(b1.x, b1.y));
                        const float2 f3 = __fadd2_rn(make_float2(__uint_as_float(vv[6]), __uint_as_float(vv[7])), make_float2(b1.z, b1.w));
                        *reinterpret_cast<uint4*>(dst + chunk_off[c]) =
                            make_uint4(mc_pack_relu_bf16(f0.x, f0.y), mc_pack_relu_bf16(f1.x, f1.y), mc_pack_relu_bf16(f2.x, f2.y),
                                       mc_pack_relu_bf16(f3.x, f3.y));
                    }
                    tc::fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) tc::mbar_arrive(&blk_ready[j]);
                }
            }
            // every MMA of layers 0..2 has completed: the next tile's x may take the slot that is free during layer 3
            const int o_next = mc_slot(o, 4, NSLOT);
            if (t + (int)gridDim.x < P.num_tiles) write_x(xn, o_next);
            // ---- layer 3: [mu | alpha] -> affine autoregressive transform, row log-det (+ head) ----
            {
                const int acc = u & 3;
                MC_WAIT(1, tc::mbar_wait(&acc_full[acc], (uint32_t)((u >> 2) & 1)));
                tc::fence_after_sync();
                uint32_t vm[16], va[16];
                tc::tmem_ld16(lane_addr + (uint32_t)(acc * kMcBN + c0), vm);
                tc::tmem_ld16(lane_addr + (uint32_t)(acc * kMcBN + 64 + c0), va);
                tc::wait_ld();
                tc::fence_before_sync();
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(&acc_empty[acc]);
                ++u;
                const int64_t row = (int64_t)t * kMcRows + r;
                float lsum = 0.f, sq = 0.f, o16[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int d = c0 + i;
                    float ov = 0.f;
                    if (d < D) {
                        const float mu = __uint_as_float(vm[i]) + bias_s[3 * H + d];
                        const float al = __uint_as_float(va[i]) + bias_s[3 * H + 64 + d];
                        float tt;
                        affine_ar_elem<float>(P.mode, xc[i], mu, al, ov, tt);
                        if (!is_finite(ov)) ov = iaf ? xc[i] : 0.f;          // IAF scrubs to the input (:53)
                        lsum += tt;
                        const float hv = (P.flags & NF_STACK_SAMPLE_LOG_Q) ? xc[i] : ov;     // head on the input row
                        sq += -0.5f * hv * hv;
                    }
                    o16[i] = ov;
                }
                if (row < P.B && !(P.flags & NF_STACK_SKIP_Y)) {
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        if (c0 + 4 * i < D)
                            __stcs(reinterpret_cast<float4*>(out + row * D + c0 + 4 * i),
                                   make_float4(o16[4 * i], o16[4 * i + 1], o16[4 * i + 2], o16[4 * i + 3]));
                }
                // the four column quarters of a row live in four warps: combine through shared memory in a fixed order
                float* part = row_part + (it & 1) * (3 * 256);
                if (cq > 0) { part[(cq - 1) * 256 + r] = lsum; part[(cq - 1) * 256 + 128 + r] = sq; }
                asm volatile("bar.sync 1, 512;" ::: "memory");
                if (cq == 0 && row < P.B) {
                    const float tot = clamp_mm(scrub0(((lsum + part[r]) + part[256 + r]) + part[512 + r]), -lim, lim);
                    float res = tot;
                    if (P.flags & (NF_STACK_LOG_PROB_HEAD | NF_STACK_SAMPLE_LOG_Q)) {
                        const float lz = (((sq + part[128 + r]) + part[256 + 128 + r]) + part[512 + 128 + r]) -
                                         (float)(0.5 * (double)D * 1.8378770664093453);
                        res = (P.flags & NF_STACK_SAMPLE_LOG_Q) ? lz - tot : lz + tot;
                    }
                    __stcs(ld_out + row, res);
                }
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) xc[i] = xn[i];
            o = o_next;
        }
        if (warp == 2) MC_PROF_STORE(8, 2);    // [8] hidden-layer accumulator full, [9] last-layer accumulator full, [10] epilogue warp total
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 1) tc::tmem_dealloc(tb, kMcTmemCols);
}

// bf16 weight [rows, K] row-major (K % 64 == 0, rows % 128 == 0): boxes of [128 rows x 64 k] = one SWIZZLE_128B atom block
static bool mc_make_map(CUtensorMap* m, const void* base, int64_t rows, int64_t K) {
    const tc::EncodeTiledFn fn = tc::encode_tiled_fn();
    if (!fn) return false;
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)K * 2};
    cuuint32_t box[2] = {(cuuint32_t)kMcAtom, (cuuint32_t)kMcBN};
    cuuint32_t estr[2] = {1, 1};
    return fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace nf

using namespace nf;
#define NF_REQ(p) do { if ((p) == nullptr) return NF_ERR_NULL; } while (0)

#ifdef NF_MC_PROFILE
extern "C" __attribute__((visibility("default"))) int nf_debug_mc_profile(long long* out) {
    return cudaMemcpyFromSymbol(out, nf::g_mc_prof, sizeof(long long) * 16) == cudaSuccess ? 0 : -4;
}
#endif

extern "C" int nf_made_chain_bf16_forward(const void* x, const void* w0, const void* w1, const void* w2, const void* w3,
                                          const void* b0, const void* b1, const void* b2, const void* b3,
                                          const int32_t* kext16_host, void* out, void* ld, int64_t B, int D, int H, int mode,
                                          int flags, nf_stream_t stream) {
    if (B < 0 || D < 1 || H < 1) return NF_ERR_BAD_SHAPE;
    if (mode != NF_AR_MAF_INVERSE && mode != NF_AR_IAF_FORWARD) return NF_ERR_UNSUPPORTED;
    if ((flags & NF_STACK_SAMPLE_LOG_Q) && (mode != NF_AR_IAF_FORWARD || (flags & NF_STACK_LOG_PROB_HEAD))) return NF_ERR_UNSUPPORTED;
    if (D > 64 || (D % 4) != 0 || (H % 128) != 0 || H > kMcMaxKA * kMcAtom) return NF_ERR_UNSUPPORTED;
    NF_REQ(kext16_host);
    if (B == 0) return NF_OK;
    NF_REQ(x); NF_REQ(w0); NF_REQ(w1); NF_REQ(w2); NF_REQ(w3); NF_REQ(b0); NF_REQ(b1); NF_REQ(b2); NF_REQ(b3); NF_REQ(ld);
    if (!(flags & NF_STACK_SKIP_Y)) NF_REQ(out);
    if (!aligned16(x) || (out && !aligned16(out)) || !aligned16(b0) || !aligned16(b1) || !aligned16(b2)) return NF_ERR_MISALIGNED;
    McParams P;
    P.NB = H / kMcBN; P.KA = H / kMcAtom; P.D = D; P.mode = mode; P.flags = flags; P.B = B;
    const int64_t tiles = cdiv(B, kMcRows);
    if (tiles > 2147483647LL) return NF_ERR_BAD_SHAPE;
    P.num_tiles = (int)tiles;
    for (int l = 0; l < 4; ++l) {
        const int kmax = (l == 0 ? kMcAtom : H) / 16;
        int prev = 0;
        for (int j = 0; j < 4; ++j) {
            int v = kext16_host[l * 4 + j];
            if (v < 0 || v > kmax) return NF_ERR_BAD_SHAPE;
            if (j >= (l == 3 ? 1 : P.NB)) v = 0;
            else { v = v > prev ? v : prev; v = v < 1 ? 1 : v; prev = v; }   // monotone in the block index (block-triangular
                                                                   // weights); >= 1: every accumulator is written by an MMA
            P.kext16[l][j] = v;
        }
    }
    alignas(64) CUtensorMap t0, t1, t2, t3;
    if (!mc_make_map(&t0, w0, H, kMcAtom) || !mc_make_map(&t1, w1, H, H) || !mc_make_map(&t2, w2, H, H) ||
        !mc_make_map(&t3, w3, kMcBN, H))
        return NF_ERR_UNSUPPORTED;
    const size_t smem = (size_t)(P.KA + 2 + kMcStages) * kMcAtomBytes + (size_t)(3 * H + 128) * sizeof(float) + 256 +
                        (2 * 3 * 256 + 16) * sizeof(float);
    if (smem > 227 * 1024) return NF_ERR_UNSUPPORTED;
    NF_CUDA(cudaFuncSetAttribute(made_chain_bf16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int grid = (int)(tiles < kNumSMs ? tiles : kNumSMs);
    made_chain_bf16_kernel<<<grid, kMcThreads, smem, (cudaStream_t)stream>>>(
        t0, t1, t2, t3, (const float*)x, (const float*)b0, (const float*)b1, (const float*)b2, (const float*)b3, (float*)out,
        (float*)ld, P);
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}
