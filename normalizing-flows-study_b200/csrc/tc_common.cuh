// tc_common.cuh -- sm_100a tensor-core plumbing shared by the tcgen05 kernels: mbarrier, TMEM allocation,
// tcgen05.mma (kind::tf32, A from TMEM or shared memory, B from shared memory), tcgen05.ld/st, descriptors, and
// the host-side lookup of the TMA tensor-map encoder.
//
// Conventions used by every kernel here:
//   * operands are fp32 containers read as TF32 by the tensor core; fp32 accuracy comes from the 3xTF32 split
//       a*b ~= a_hi*b_hi + a_lo*b_hi + a_hi*b_lo,   x_hi = x rounded to TF32, x_lo = x - x_hi (exact in fp32)
//     (the dropped a_lo*b_lo term and the truncation of a_lo are O(2^-23) relative);
//   * B (weights, [N][K] row-major = K-major) lives in shared memory in the canonical UMMA K-major SWIZZLE_128B
//     layout: K is cut into atoms of 32 floats (128 B); inside an atom block row n occupies 128 B at
//     (n/8)*1024 + (n%8)*128 and its eight 16-byte chunks are XOR-swizzled with (n%8); the host packs that image;
//   * A (activations) is written by its owning thread into TMEM: lane = tile row, column = k (M = 128).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace nf {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ---------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t a = smem_u32(bar);
    uint32_t ok;
    do {
        // (a suspend-time hint on the try_wait makes no difference: profiles/r02z_mbar_hint_ab.txt)
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(a), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// generic-proxy writes to shared memory (st.shared / cp.async) -> visible to the async proxy (tcgen05.mma, TMA)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// 1-D bulk copy global -> shared through the TMA unit (async proxy), completion on an mbarrier
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ---- TMEM -----------------------------------------------------------------------------------------------
// one full warp; writes the base address (lane 0, column c0) to *dst_smem
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(ncols) : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// MMA completion -> mbarrier (implies tcgen05.fence::before_thread_sync)
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// warp-collective: thread (lane l of warp w) reads / writes 16 consecutive columns of TMEM lane 32*(w%4)+l
__device__ __forceinline__ void tmem_ld16(uint32_t addr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(addr) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t addr, const uint32_t (&v)[16]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
                 ::"r"(addr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
                   "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t addr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(addr) : "memory");
}

// ---- descriptors --------------------------------------------------------------------------------------
// shared-memory matrix descriptor, K-major SWIZZLE_128B (sm_100 version 1): start address >> 4 in bits [0,14),
// LBO (unused for swizzled K-major) bits [16,30), SBO = 1024 B (8 rows x 128 B) >> 4 in bits [32,46),
// version = 1 at bit 46, layout type SWIZZLE_128B = 2 at bits [61,64).  The tile base must be 1024-byte aligned;
// advancing K inside an atom adds the byte offset to the start address.
__device__ __forceinline__ uint64_t smem_desc_k_sw128(uint32_t smem_byte_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_byte_addr >> 4) & 0x3fffu);
    d |= (uint64_t)(1024u >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// instruction descriptor for kind::tf32, fp32 accumulate, A and B K-major, M = 128
__host__ __device__ constexpr uint32_t idesc_tf32_m128(uint32_t N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((N >> 3) << 17) | ((128u >> 4) << 24);
}
// D[tmem] (+)= A[tmem] * B[smem]^T : one elected thread
__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T
__device__ __forceinline__ void mma_tf32_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}

// warp-convergent election of one lane (the MMA issuer); the whole warp must execute this
__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}

// 3xTF32 GEMM over K = 64 of the CTA's TMEM-resident A operand (hi columns a_hi_col.., lo columns a_lo_col..) with a
// [N][64] weight whose hi / lo SWIZZLE_128B images sit at shared-memory byte addresses w_hi / w_lo; result (overwritten)
// in TMEM columns d_col.. .  Must be executed by ONE WHOLE WARP with convergent control flow: descriptors are then
// computed once in uniform registers and the 24 tcgen05.mma issue back to back from the elected lane (issuing from a
// divergent `if (tid == 0)` costs ~70 cycles per MMA in R2UR transfers).  Ends with tcgen05.commit -> bar.
__device__ __forceinline__ void warp_issue_gemm_k64_3xtf32(uint32_t tmem_base, uint32_t d_col, uint32_t a_hi_col, uint32_t a_lo_col,
                                                           uint32_t w_hi, uint32_t w_lo, uint32_t N, uint64_t* bar) {
    const uint32_t idesc = idesc_tf32_m128(N);
    const uint32_t atom16 = (N * 128u) >> 4;                  // K-atom block stride in 16-byte units
    const uint64_t d_hi = smem_desc_k_sw128(w_hi), d_lo = smem_desc_k_sw128(w_lo);
    const bool leader = elect_one();
#pragma unroll
    for (int pass = 0; pass < 3; ++pass) {
        const uint32_t a_col = (pass == 1) ? a_lo_col : a_hi_col;
        const uint64_t wd = (pass == 2) ? d_lo : d_hi;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const uint64_t bd = wd + (uint64_t)((uint32_t)(k >> 2) * atom16 + (uint32_t)(k & 3) * 2u);
            if (leader) mma_tf32_ts(tmem_base + d_col, tmem_base + a_col + k * 8, bd, idesc, (pass | k) != 0 ? 1u : 0u);
        }
    }
    if (leader) mma_commit(bar);
    __syncwarp();
}

// Same for a K range: k-steps [k0, k0+nk) of the weight images against nk*8 A columns starting at a_hi_col / a_lo_col
// (the A operand of those k-steps only); acc_first = 0 overwrites the accumulator with the first MMA.
__device__ __forceinline__ void warp_issue_gemm_krange_3xtf32(uint32_t tmem_base, uint32_t d_col, uint32_t a_hi_col, uint32_t a_lo_col,
                                                              uint32_t w_hi, uint32_t w_lo, uint32_t N, int k0, int nk,
                                                              uint32_t acc_first, uint64_t* bar) {
    const uint32_t idesc = idesc_tf32_m128(N);
    const uint32_t atom16 = (N * 128u) >> 4;
    const uint64_t d_hi = smem_desc_k_sw128(w_hi), d_lo = smem_desc_k_sw128(w_lo);
    const bool leader = elect_one();
#pragma unroll
    for (int pass = 0; pass < 3; ++pass) {
        const uint32_t a_col = (pass == 1) ? a_lo_col : a_hi_col;
        const uint64_t wd = (pass == 2) ? d_lo : d_hi;
#pragma unroll 4
        for (int kk = 0; kk < nk; ++kk) {
            const int k = k0 + kk;
            const uint64_t bd = wd + (uint64_t)((uint32_t)(k >> 2) * atom16 + (uint32_t)(k & 3) * 2u);
            if (leader) mma_tf32_ts(tmem_base + d_col, tmem_base + a_col + kk * 8, bd, idesc, (pass | kk) != 0 ? 1u : acc_first);
        }
    }
    if (leader) mma_commit(bar);
    __syncwarp();
}

// ---- 3xTF32 split -----------------------------------------------------------------------------------
// hi = a rounded to the nearest TF32 (add half an ulp of the 13 dropped bits, then clear them; the carry walks into
// the exponent correctly, Inf stays Inf), lo = a - hi exactly, |lo| <= 2^-12 |a|.  The tensor core truncates lo to
// TF32 (error <= 2^-23 |a|); with the dropped lo*lo term the 3-pass product is within ~2.4e-7 of sum |a||b|.
__device__ __forceinline__ void split_tf32(float a, uint32_t& hi, uint32_t& lo) {
    hi = (__float_as_uint(a) + 0x1000u) & 0xffffe000u;
    lo = __float_as_uint(a - __uint_as_float(hi));
}
// Two values at once on the packed fp32 pipe (Blackwell FMUL2 / FFMA2: 3 instructions per PAIR instead of the 6 integer / FP
// ones above -- the fused stack kernels are issue-bound and split 128 activations per row and layer).  Veltkamp's split
// with C = 2^13 + 1:  c = fl(C a);  hi = c - 2^13 a  (2^13 a is exact and the difference has at most 11 significant bits,
// so the FMA does not round: hi = a rounded to the nearest TF32);  lo = a - hi exactly.  Same guarantees as split_tf32
// (ties may round the other way, which lo absorbs); |a| > 2^114 overflows c, Inf / NaN give NaN in both as before the MMA.
__device__ __forceinline__ void split_tf32_x2(float a0, float a1, uint32_t& hi0, uint32_t& hi1, uint32_t& lo0, uint32_t& lo1) {
    const float2 a = make_float2(a0, a1);
    const float2 c = __fmul2_rn(a, make_float2(8193.0f, 8193.0f));
    const float2 h = __ffma2_rn(a, make_float2(-8192.0f, -8192.0f), c);
    const float2 l = __ffma2_rn(h, make_float2(-1.0f, -1.0f), a);
    hi0 = __float_as_uint(h.x); hi1 = __float_as_uint(h.y);
    lo0 = __float_as_uint(l.x); lo1 = __float_as_uint(l.y);
}
// weights (split once per weight version): lo is additionally rounded to TF32 so that the hardware truncation is exact
__device__ __forceinline__ void split_tf32_weight(float a, uint32_t& hi, uint32_t& lo) {
    split_tf32(a, hi, lo);
    lo = (lo + 0x1000u) & 0xffffe000u;
}

// ---- epilogue stores ------------------------------------------------------------------------------------
// After tcgen05.ld a thread owns one output ROW (TMEM lane = row) and a run of consecutive columns, so it can write its
// own row directly: one 256-bit store (STG.E.256, sm_100) per 8 columns = one full 32-byte sector, no shared-memory
// transpose, no LDS.  (The first epilogue transposed through shared memory and issued one 4-byte store per element:
// 128 x (LDS + STG) per thread and tile, measured at ~12 000 clk per 128 x 128 tile in gemm_tc2 -- longer than the three
// accumulation chains the MMA warp can run ahead -- so the tensor pipe idled half of the time.)
__device__ __forceinline__ void st_global_v8(float* p, const float (&o)[8]) {
    // no "memory" clobber: the compiler may batch the bias loads of later stores ahead of this one
    asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"l"(p), "f"(o[0]), "f"(o[1]), "f"(o[2]), "f"(o[3]), "f"(o[4]), "f"(o[5]), "f"(o[6]), "f"(o[7]));
}
// 8 consecutive outputs of one row starting at column col (col % 8 == 0), bias already added: ReLU + store.  No loads
// in here: the callers fetch the bias (from the shared-memory tile staged by stage_bias_tile) in one batch BEFORE the
// stores -- a bias load in front of every store waited ~370 clk each behind the queued 1 KB stores (measured).
// vec (checked on the host): 1 = &yrow[col] is 32-byte aligned (one 256-bit store), 2 = only 16-byte aligned (two 128-bit
// stores: column slices that start at a multiple of 4 units); ragged column tails take the scalar path.
__device__ __forceinline__ void epilogue_store8(float* __restrict__ yrow, int col, int N, const float (&a)[8], int relu, int vec) {
    float o[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = (relu && a[i] < 0.f) ? 0.f : a[i];          // NaN stays NaN (torch.relu)
    if (vec == 1 && col + 8 <= N) {
        st_global_v8(yrow + col, o);
    } else if (vec == 2 && col + 8 <= N) {
        asm volatile("st.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(yrow + col), "f"(o[0]), "f"(o[1]), "f"(o[2]), "f"(o[3]));
        asm volatile("st.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(yrow + col + 4), "f"(o[4]), "f"(o[5]), "f"(o[6]), "f"(o[7]));
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (col + i < N) yrow[col + i] = o[i];
    }
}
// 32 columns [c0, c0 + 32) of one row held as the raw tcgen05.ld words v0 (first 16) / v1 (last 16); bias32 = the 32 bias
// values of these columns in shared memory (16-byte aligned), read in one batch ahead of the stores
__device__ __forceinline__ void epilogue_store32(float* __restrict__ yrow, int c0, int N, const uint32_t (&v0)[16],
                                                 const uint32_t (&v1)[16], const float* __restrict__ bias32, int relu, int vec) {
    float o[32];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float4 b = bias32 ? *reinterpret_cast<const float4*>(bias32 + 4 * j) : make_float4(0.f, 0.f, 0.f, 0.f);
        const uint32_t* v = (j < 4) ? &v0[4 * j] : &v1[4 * (j - 4)];
        o[4 * j + 0] = __uint_as_float(v[0]) + b.x; o[4 * j + 1] = __uint_as_float(v[1]) + b.y;
        o[4 * j + 2] = __uint_as_float(v[2]) + b.z; o[4 * j + 3] = __uint_as_float(v[3]) + b.w;
    }
#pragma unroll
    for (int h = 0; h < 4; ++h) {
        float a8[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) a8[i] = o[8 * h + i];
        epilogue_store8(yrow, c0 + 8 * h, N, a8, relu, vec);
    }
}
// Fallback for outputs the 256-bit row stores cannot take (base or pitch not 32-byte aligned: column slices starting at
// an arbitrary unit, 23 / 29-wide heads): lane = row holds o[32] = 32 consecutive columns [c0, c0 + 32) (bias NOT yet
// added); transposed through the warp's [32][33] shared-memory buffer so that a warp writes 128 contiguous bytes of one
// row per store.  All 32 lanes must call it.  (Per-thread scalar stores into the own row were 2.2x slower on the
// [262144, 64] slice products of the blocked sequential direction: 32 sectors per 128 bytes.)
__device__ __forceinline__ void epilogue_store32_transposed(float* __restrict__ Y, int64_t ldc, int row0, int M, int c0, int N,
                                                            const uint32_t (&v0)[16], const uint32_t (&v1)[16],
                                                            const float* __restrict__ bias, int relu, float* tbuf, int lane) {
#pragma unroll
    for (int j = 0; j < 16; ++j) { tbuf[lane * 33 + j] = __uint_as_float(v0[j]); tbuf[lane * 33 + 16 + j] = __uint_as_float(v1[j]); }
    __syncwarp();
    const int col = c0 + lane;
    if (col < N) {
        const float bv = bias ? __ldg(bias + col) : 0.f;
#pragma unroll 4
        for (int rr = 0; rr < 32; ++rr) {
            const int row = row0 + rr;
            if (row < M) {
                float o = tbuf[rr * 33 + lane] + bv;
                if (relu) o = (o < 0.f) ? 0.f : o;          // NaN stays NaN (torch.relu)
                Y[(int64_t)row * ldc + col] = o;
            }
        }
    }
    __syncwarp();
}
// 128 epilogue threads (four warps) stage the tile's 128 bias values (zeros past N or without a bias) in shared memory;
// named barrier `bar_id` (1..15) makes them visible to the four warps
__device__ __forceinline__ void stage_bias_tile(float* bias_s, const float* __restrict__ bias, int n0, int N, int t128, int bar_id) {
    bias_s[t128] = (bias && n0 + t128 < N) ? __ldg(bias + n0 + t128) : 0.f;
    asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
}

// byte offset of element (n, k) inside a K-major SWIZZLE_128B image of an [rows][K] fp32 matrix (K % 32 == 0, rows % 8 == 0)
__host__ __device__ constexpr uint32_t sw128_offset(uint32_t n, uint32_t k, uint32_t rows) {
    return (k >> 5) * (rows * 128u) + (n >> 3) * 1024u + (n & 7u) * 128u + ((((k & 31u) >> 2) ^ (n & 7u)) << 4) + (k & 3u) * 4u;
}

// ---- host: TMA tensor maps -----------------------------------------------------------------------------
// cuTensorMapEncodeTiled through the runtime's driver entry point (the library does not link libcuda); nullptr when
// the driver does not provide it.  Each caller builds its own maps: box, swizzle and element type differ per kernel.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_tiled_fn() {
    static const EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        const bool ok = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
                        qres == cudaDriverEntryPointSuccess;
        return ok ? reinterpret_cast<EncodeTiledFn>(p) : nullptr;
    }();
    return fn;
}

}  // namespace tc
}  // namespace nf
