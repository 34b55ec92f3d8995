// nf_rng.cuh -- the N(0, I) base draw of sample_and_log_prob: one fixed, counter-based stream shared by every route
// (the standalone nf_std_normal_draw and the in-kernel draw of the fused stacks), so that the same (seed, offset) gives
// bit-identical z whichever kernel draws it.  Host + device, like nf_math.cuh (the host side is compiled by the CPU
// tests; the library only draws on the device).
//
//   generator  Philox4x32-10 with the constants of curand_philox4x32_x.h
//   key        (lo32(seed) ^ 0x6E666232, hi32(seed)): the xor keeps this stream apart from torch's Philox streams of the
//              same generator seed
//   counter    (j, row, lo32(offset / 4), hi32(offset / 4)) for dims 4j .. 4j+3 of `row`
//   normals    Box-Muller on the pairs (u0, u1), (u2, u3): a = u * 2^-32 + 2^-33 (curand's uniform), r = sqrt(-2 log a),
//              z = (r cos(2 pi b), r sin(2 pi b)); dims >= D are discarded
// A row's values depend on (seed, offset, row) only, so a draw of n1 rows is a bit-exact prefix of a draw of n2 > n1.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define NF_RNG_HD __host__ __device__ __forceinline__
#else
#include <cmath>
#define NF_RNG_HD inline
#endif

namespace nf {

constexpr uint32_t kPhiloxW0 = 0x9E3779B9u, kPhiloxW1 = 0xBB67AE85u;   // key schedule (PHILOX_W32_0 / _1)
constexpr uint32_t kPhiloxM0 = 0xD2511F53u, kPhiloxM1 = 0xCD9E8D57u;   // round multipliers (PHILOX_M4x32_0 / _1)
constexpr uint32_t kNfRngKeyXor = 0x6E666232u;                           // 'nfb2'

NF_RNG_HD uint32_t nf_mulhi32(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}

// Philox4x32-10: c[4] (counter) -> c[4] (four 32-bit outputs) under key (k0, k1)
NF_RNG_HD void nf_philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = nf_mulhi32(kPhiloxM0, c[0]), lo0 = kPhiloxM0 * c[0];
        const uint32_t hi1 = nf_mulhi32(kPhiloxM1, c[2]), lo1 = kPhiloxM1 * c[2];
        const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
        c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
        k0 += kPhiloxW0; k1 += kPhiloxW1;
    }
}

NF_RNG_HD float nf_u32_to_unit(uint32_t u) {           // (0, 1]: curand's _curand_uniform
    return (float)u * 2.3283064365386963e-10f + 1.1641532182693481e-10f;    // 2^-32, 2^-33
}

// one Box-Muller pair from two 32-bit words
NF_RNG_HD void nf_box_muller(uint32_t ua, uint32_t ub, float& z0, float& z1) {
    const float a = nf_u32_to_unit(ua), b = nf_u32_to_unit(ub);
#ifdef __CUDA_ARCH__
    const float r = sqrtf(-2.0f * logf(a));
    float s, c;
    sincospif(2.0f * b, &s, &c);
#else
    // host twin for the CPU tests: the same fp32 uniforms, log / sin / cos rounded from double
    const float r = std::sqrt(-2.0f * (float)std::log((double)a));
    const double t = 3.141592653589793 * (double)(2.0f * b);
    const float s = (float)std::sin(t), c = (float)std::cos(t);
#endif
    z0 = r * c;
    z1 = r * s;
}

// the four normals of dims 4j .. 4j+3 of `row`
NF_RNG_HD void nf_std_normal4(uint64_t seed, uint64_t offset, uint32_t row, uint32_t j, float (&z)[4]) {
    const uint64_t o4 = offset >> 2;
    uint32_t c[4] = {j, row, (uint32_t)o4, (uint32_t)(o4 >> 32)};
    nf_philox4x32_10(c, (uint32_t)seed ^ kNfRngKeyXor, (uint32_t)(seed >> 32));
    nf_box_muller(c[0], c[1], z[0], z[1]);
    nf_box_muller(c[2], c[3], z[2], z[3]);
}

// z[0..D) of `row` (z[d >= D] = 0); returns log N(z; 0, I) with the arithmetic of nf_stack_row_head
template <int DM>
NF_RNG_HD float nf_std_normal_row(uint64_t seed, uint64_t offset, uint32_t row, int D, float (&z)[DM]) {
#pragma unroll
    for (int j = 0; j < (DM + 3) / 4; ++j) {
        float q[4] = {0.f, 0.f, 0.f, 0.f};
        if (4 * j < D) nf_std_normal4(seed, offset, row, (uint32_t)j, q);
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (4 * j + k < DM) z[4 * j + k] = (4 * j + k < D) ? q[k] : 0.f;
    }
    float acc = 0.f;
#pragma unroll
    for (int d = 0; d < DM; ++d) if (d < D) acc += -0.5f * z[d] * z[d];
    return acc - (float)(0.5 * (double)D * 1.8378770664093453);
}

#ifdef __CUDACC__
// Device-resident generator state (nf_*_sample_state, nf_std_normal_draw_state): uint64[4] = {seed, offset, ticket,
// reserved} in caller memory, ticket 0 between calls.  A launch draws with the key (seed, offset) it reads there and
// moves offset on by 4 in the same launch, so a CUDA-graph replay draws new samples.  Ticket protocol: every CTA of the
// grid calls this exactly once, before any early exit or role split; thread 0 reads (seed, offset) into key[0..1]
// (shared memory), fences, and takes a ticket.  The CTA that takes ticket gridDim.x - 1 knows every CTA has read the
// key, so it stores offset + 4 and ticket = 0.  key[] is valid for the CTA after the caller's next __syncthreads(); the
// kernels read it where they draw, so the key costs no registers across the kernel.
__device__ __forceinline__ void nf_rng_state_take(unsigned long long* state, unsigned long long* key) {
    if (threadIdx.x == 0) {
        const unsigned long long seed = __ldcg(state), offset = __ldcg(state + 1);
        key[0] = seed;
        key[1] = offset;
        __threadfence();
        if (atomicAdd(state + 2, 1ull) == (unsigned long long)gridDim.x - 1) {
            __threadfence();
            state[1] = offset + 4;
            state[2] = 0;
        }
    }
}

// the key slot of kernels without a spare dynamic shared-memory word (one per kernel: a function-scope static)
__device__ __forceinline__ unsigned long long* nf_rng_key_static() {
    __shared__ unsigned long long key[2];
    return key;
}

// entry-point check of a caller's state pointer (64-bit atomics need 8-byte alignment)
inline int nf_rng_state_check(const void* state) {
    if (state == nullptr) return NF_ERR_NULL;
    return (reinterpret_cast<uintptr_t>(state) & 7) ? NF_ERR_MISALIGNED : NF_OK;
}

// B == 0: the sampling entry points launch nothing else, but a call still advances the state (aux_kernels.cu)
int nf_rng_state_advance(unsigned long long* state, cudaStream_t st);
#endif

}  // namespace nf

#undef NF_RNG_HD
