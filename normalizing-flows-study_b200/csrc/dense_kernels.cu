// dense_kernels.cu -- dense building blocks of the general / training path:
//   nf_gemm              strided SIMT GEMM with bias/ReLU epilogue, zero-tile skipping (k_extent) and split-K
//                        (F.linear of the conditioners and of MaskedLinear, masked_linear.py:14-18, + its backward)
//   nf_mul_rows, nf_relu_backward, nf_col_sum     small elementwise / reduction helpers
//   nf_batchnorm_*       nn.BatchNorm1d (+ReLU) of the coupling conditioners (coupling_layer.py:20-24)
// fp32 accumulate in fp32 FFMA (bit-level parity class of the reference's sgemm); fp64 for gradcheck.
// The tcgen05 GEMMs for the large shapes live in gemm_tc2.cu / wgrad_tc.cu, the streaming kernels for
// shapes with one tiny dimension in skinny_kernels.cu; this kernel is the exact-fp32 fallback
// for every shape and the only path for fp64.
#include "nf_common.cuh"

namespace nf {

// ------------------------------------------------------------------------------------------------
// GEMM: C[M,N] (+)= A[M,K] * B[K,N], element strides (sam,sak) / (sbk,sbn).
//   float : 128x128x16 tile, 256 threads, 8x8 micro-tile split as 2x2 blocks of 4x4 (conflict-free LDS.128)
//   double:  64x64x16 tile, 256 threads, 4x4 micro-tile
// ------------------------------------------------------------------------------------------------
template <typename T> struct GemmCfg;
template <> struct GemmCfg<float>  { static constexpr int BM = 128, BN = 128, BK = 16, TM = 8, TN = 8; };
template <> struct GemmCfg<double> { static constexpr int BM = 64,  BN = 64,  BK = 16, TM = 4, TN = 4; };

template <typename T>
__global__ void __launch_bounds__(256, 2)
gemm_kernel(const T* __restrict__ A, const T* __restrict__ Bm, T* __restrict__ C, const T* __restrict__ bias,
            int64_t M, int64_t N, int64_t K, int64_t sam, int64_t sak, int64_t sbk, int64_t sbn, int64_t ldc,
            int relu, int accumulate, const int32_t* __restrict__ k_extent, int ksplit_len) {
    using Cfg = GemmCfg<T>;
    constexpr int BM = Cfg::BM, BN = Cfg::BN, BK = Cfg::BK, TM = Cfg::TM, TN = Cfg::TN;
    constexpr int PADM = BM + 4, PADN = BN + 4;
    constexpr int NT = 256;
    constexpr int LA = BM * BK / NT, LB = BN * BK / NT;
    __shared__ __align__(16) T As[BK][PADM];
    __shared__ __align__(16) T Bs[BK][PADN];

    const int tid = threadIdx.x;
    const int64_t m0 = (int64_t)blockIdx.x * BM, n0 = (int64_t)blockIdx.y * BN;   // M tiles on x (2^31 limit)
    int64_t k_begin = 0, k_end = K;
    if (k_extent) {                         // entries are per 64 output columns
        int e = 0;
        for (int64_t c = n0 / 64; c <= (n0 + BN - 1) / 64 && c * 64 < N; ++c) e = max(e, k_extent[c]);
        k_end = (K < (int64_t)e) ? K : (int64_t)e;
    }
    if (ksplit_len > 0) {
        k_begin = (int64_t)blockIdx.z * ksplit_len;
        k_end = (k_end < k_begin + ksplit_len) ? k_end : k_begin + ksplit_len;
    }
    const bool a_kfast = (sak == 1);
    const bool b_nfast = (sbn == 1);
    const int ty = tid / (BN / TN), tx = tid % (BN / TN);

    T acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = T(0);

    T ra[LA], rb[LB];
    auto load_tile = [&](int64_t kt) {
#pragma unroll
        for (int i = 0; i < LA; ++i) {
            const int idx = tid + i * NT;
            const int kk = a_kfast ? idx % BK : idx / BM;
            const int mm = a_kfast ? idx / BK : idx % BM;
            const int64_t gm = m0 + mm, gk = kt + kk;
            ra[i] = (gm < M && gk < k_end) ? A[gm * sam + gk * sak] : T(0);
        }
#pragma unroll
        for (int i = 0; i < LB; ++i) {
            const int idx = tid + i * NT;
            const int nn = b_nfast ? idx % BN : idx / BK;
            const int kk = b_nfast ? idx / BN : idx % BK;
            const int64_t gn = n0 + nn, gk = kt + kk;
            rb[i] = (gn < N && gk < k_end) ? Bm[gk * sbk + gn * sbn] : T(0);
        }
    };
    auto store_tile = [&]() {
#pragma unroll
        for (int i = 0; i < LA; ++i) {
            const int idx = tid + i * NT;
            const int kk = a_kfast ? idx % BK : idx / BM;
            const int mm = a_kfast ? idx / BK : idx % BM;
            As[kk][mm] = ra[i];
        }
#pragma unroll
        for (int i = 0; i < LB; ++i) {
            const int idx = tid + i * NT;
            const int nn = b_nfast ? idx % BN : idx / BK;
            const int kk = b_nfast ? idx / BN : idx % BK;
            Bs[kk][nn] = rb[i];
        }
    };

    if (k_begin < k_end) load_tile(k_begin);
    for (int64_t kt = k_begin; kt < k_end; kt += BK) {
        __syncthreads();
        store_tile();
        __syncthreads();
        if (kt + BK < k_end) load_tile(kt + BK);       // prefetch next tile into registers
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            T a[TM], b[TN];
            if constexpr (sizeof(T) == 4) {
                float4 v0 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
                float4 v1 = *reinterpret_cast<const float4*>(&As[kk][BM / 2 + ty * 4]);
                a[0] = v0.x; a[1] = v0.y; a[2] = v0.z; a[3] = v0.w; a[4] = v1.x; a[5] = v1.y; a[6] = v1.z; a[7] = v1.w;
                float4 w0 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
                float4 w1 = *reinterpret_cast<const float4*>(&Bs[kk][BN / 2 + tx * 4]);
                b[0] = w0.x; b[1] = w0.y; b[2] = w0.z; b[3] = w0.w; b[4] = w1.x; b[5] = w1.y; b[6] = w1.z; b[7] = w1.w;
            } else {
#pragma unroll
                for (int i = 0; i < TM; ++i) a[i] = As[kk][ty * TM + i];
#pragma unroll
                for (int j = 0; j < TN; ++j) b[j] = Bs[kk][tx * TN + j];
            }
            if constexpr (sizeof(T) == 4) {
                // packed fp32 FMAs (Blackwell FFMA2): two output columns per instruction, a[i] duplicated into a pair; the
                // accumulators of a column pair are adjacent registers.  Same operations per element, bit-identical.
#pragma unroll
                for (int i = 0; i < TM; ++i) {
                    const float2 aa = make_float2((float)a[i], (float)a[i]);
#pragma unroll
                    for (int j = 0; j < TN; j += 2) {
                        const float2 r = __ffma2_rn(aa, make_float2((float)b[j], (float)b[j + 1]),
                                                    make_float2((float)acc[i][j], (float)acc[i][j + 1]));
                        acc[i][j] = (T)r.x; acc[i][j + 1] = (T)r.y;
                    }
                }
            } else {
#pragma unroll
                for (int i = 0; i < TM; ++i)
#pragma unroll
                    for (int j = 0; j < TN; ++j) acc[i][j] += a[i] * b[j];
            }
        }
    }

    // epilogue
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        int64_t gm;
        if constexpr (sizeof(T) == 4) gm = m0 + (i < 4 ? ty * 4 + i : BM / 2 + ty * 4 + (i - 4));
        else gm = m0 + ty * TM + i;
        if (gm >= M) continue;
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            int64_t gn;
            if constexpr (sizeof(T) == 4) gn = n0 + (j < 4 ? tx * 4 + j : BN / 2 + tx * 4 + (j - 4));
            else gn = n0 + tx * TN + j;
            if (gn >= N) continue;
            T v = acc[i][j];
            T* cp = C + gm * ldc + gn;
            if (ksplit_len > 0) { atomicAdd(cp, v); continue; }
            if (bias) v += bias[gn];
            if (accumulate) v += *cp;
            if (relu) v = relu_nan(v);
            *cp = v;
        }
    }
}

// skinny_kernels.cu: products with one dimension <= 8 (data_dim of the low-dimensional flows)
template <typename T>
int skinny_gemm_try(const void* A, const void* Bm, void* C, const void* bias, int64_t M, int64_t N, int64_t K, int64_t sam,
                    int64_t sak, int64_t sbk, int64_t sbn, int64_t ldc, int relu, int accumulate, const int32_t* k_extent,
                    cudaStream_t st);
template <typename T>
int col_sum_small_launch(const void* a, void* out, int64_t rows, int cols, cudaStream_t st);

template <typename T>
static int gemm_launch(const void* A, const void* Bm, void* C, const void* bias, int64_t M, int64_t N, int64_t K,
                       int64_t sam, int64_t sak, int64_t sbk, int64_t sbn, int64_t ldc, int relu, int accumulate,
                       const int32_t* k_extent, cudaStream_t st) {
    using Cfg = GemmCfg<T>;
    {
        const int rc = skinny_gemm_try<T>(A, Bm, C, bias, M, N, K, sam, sak, sbk, sbn, ldc, relu, accumulate, k_extent, st);
        if (rc < 0) return rc;
        if (rc == 1) { count_launch(); NF_LAUNCH_CHECK(); return NF_OK; }
    }
    const int64_t tm = cdiv(M, Cfg::BM), tn = cdiv(N, Cfg::BN);
    if (tn > 65535 || tm > 2147483647LL) return NF_ERR_BAD_SHAPE;
    int splits = 1;
    if (!bias && !relu && !k_extent && tm * tn < kNumSMs && K >= 4096) {   // weight-gradient shape: split K
        { int64_t a_ = cdiv(2 * kNumSMs, tm * tn), b_ = K / 1024; splits = (int)(a_ < b_ ? a_ : b_); }
        if (splits < 1) splits = 1;
    }
    int ksplit_len = 0;
    if (splits > 1) {
        ksplit_len = (int)(cdiv(cdiv(K, splits), Cfg::BK) * Cfg::BK);
        splits = (int)cdiv(K, ksplit_len);
        if (!accumulate) {
            if (ldc == N) NF_CUDA(cudaMemsetAsync(C, 0, sizeof(T) * M * N, st));
            else NF_CUDA(cudaMemset2DAsync(C, sizeof(T) * ldc, 0, sizeof(T) * N, M, st));
        }
    }
    dim3 grid((unsigned)tm, (unsigned)tn, (unsigned)splits);
    gemm_kernel<T><<<grid, 256, 0, st>>>((const T*)A, (const T*)Bm, (T*)C, (const T*)bias, M, N, K, sam, sak, sbk, sbn,
                                         ldc, relu, accumulate, k_extent, ksplit_len);
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

// ------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void mul_rows_kernel(const T* __restrict__ a, const T* __restrict__ b, T* __restrict__ out, int64_t rows,
                                int64_t cols, int64_t b_rows) {
    const int64_t n = rows * cols, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        out[i] = a[i] * (b_rows == 1 ? b[i % cols] : b[i]);
}

template <typename T>
__global__ void relu_bwd_kernel(const T* __restrict__ y, const T* __restrict__ gy, T* __restrict__ gx, int64_t n) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        gx[i] = (y[i] > T(0)) ? gy[i] : T(0);
}

// column sums of a[rows, cols]: block = 32 columns x 8 row-lanes; grid.y row chunks combine with atomics
template <typename T>
__global__ void __launch_bounds__(256)
col_sum_kernel(const T* __restrict__ a, T* __restrict__ out, int64_t rows, int64_t cols, int64_t rows_per_chunk) {
    __shared__ double red[8][33];
    const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
    const int64_t col = (int64_t)blockIdx.x * 32 + cx;
    const int64_t r0 = (int64_t)blockIdx.y * rows_per_chunk;
    const int64_t r1 = (rows < r0 + rows_per_chunk) ? rows : r0 + rows_per_chunk;
    double s = 0.0;
    if (col < cols)
        for (int64_t r = r0 + ry; r < r1; r += 8) s += (double)a[r * cols + col];
    red[ry][cx] = s;
    __syncthreads();
    if (ry == 0 && col < cols) {
        double t = 0.0;
#pragma unroll
        for (int i = 0; i < 8; ++i) t += red[i][cx];
        if (gridDim.y == 1) out[col] = (T)t; else atomicAdd(out + col, (T)t);
    }
}

// float32, cols % 4 == 0, 16-byte aligned: block = 32 lanes x 4 columns (one 512-byte row segment per warp load) x 8
// row-lanes, four independent 128-bit loads in flight per thread; grid.y row chunks fill the machine (HBM-bound:
// the first version moved 4 bytes per thread per dependent iteration and reached 1.2 TB/s)
__global__ void __launch_bounds__(256)
col_sum_vec4_kernel(const float* __restrict__ a, float* __restrict__ out, int64_t rows, int64_t cols, int64_t rows_per_chunk) {
    __shared__ float4 red[8][33];
    const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
    const int64_t col = ((int64_t)blockIdx.x * 32 + cx) * 4;
    const int64_t r0 = (int64_t)blockIdx.y * rows_per_chunk;
    const int64_t r1 = (rows < r0 + rows_per_chunk) ? rows : r0 + rows_per_chunk;
    float4 s0 = make_float4(0.f, 0.f, 0.f, 0.f), s1 = s0, s2 = s0, s3 = s0;
    if (col < cols) {
        const float* p = a + col;
        int64_t r = r0 + ry;
        for (; r + 24 < r1; r += 32) {
            const float4 v0 = __ldcs(reinterpret_cast<const float4*>(p + r * cols));
            const float4 v1 = __ldcs(reinterpret_cast<const float4*>(p + (r + 8) * cols));
            const float4 v2 = __ldcs(reinterpret_cast<const float4*>(p + (r + 16) * cols));
            const float4 v3 = __ldcs(reinterpret_cast<const float4*>(p + (r + 24) * cols));
            s0.x += v0.x; s0.y += v0.y; s0.z += v0.z; s0.w += v0.w;
            s1.x += v1.x; s1.y += v1.y; s1.z += v1.z; s1.w += v1.w;
            s2.x += v2.x; s2.y += v2.y; s2.z += v2.z; s2.w += v2.w;
            s3.x += v3.x; s3.y += v3.y; s3.z += v3.z; s3.w += v3.w;
        }
        for (; r < r1; r += 8) {
            const float4 v0 = __ldcs(reinterpret_cast<const float4*>(p + r * cols));
            s0.x += v0.x; s0.y += v0.y; s0.z += v0.z; s0.w += v0.w;
        }
    }
    red[ry][cx] = make_float4((s0.x + s1.x) + (s2.x + s3.x), (s0.y + s1.y) + (s2.y + s3.y), (s0.z + s1.z) + (s2.z + s3.z),
                              (s0.w + s1.w) + (s2.w + s3.w));
    __syncthreads();
    if (ry == 0 && col < cols) {
        double t0 = 0.0, t1 = 0.0, t2 = 0.0, t3 = 0.0;
#pragma unroll
        for (int i = 0; i < 8; ++i) { const float4 v = red[i][cx]; t0 += v.x; t1 += v.y; t2 += v.z; t3 += v.w; }
        if (gridDim.y == 1) { out[col] = (float)t0; out[col + 1] = (float)t1; out[col + 2] = (float)t2; out[col + 3] = (float)t3; }
        else { atomicAdd(out + col, (float)t0); atomicAdd(out + col + 1, (float)t1); atomicAdd(out + col + 2, (float)t2); atomicAdd(out + col + 3, (float)t3); }
    }
}

// ------------------------------------------------------------------------------------------------
// BatchNorm1d (+ReLU).  Batch statistics: every CTA owns 32 columns x one chunk of rows, accumulates in double and
// combines with double atomics into the caller's workspace acc[2H] (sum, sum of squares); a second tiny kernel turns
// the sums into mean / rstd and moves the running statistics.  The grid covers all SMs for any H (the first version
// used ceil(H/32) CTAs only: 2 CTAs for H = 64).
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
bn_partial_sums_kernel(const T* __restrict__ x, double* __restrict__ acc, int64_t B, int H, int64_t rows_per_chunk) {
    __shared__ double s1[8][33], s2[8][33];
    const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
    const int col = blockIdx.x * 32 + cx;
    const int64_t r0 = (int64_t)blockIdx.y * rows_per_chunk;
    const int64_t r1 = (B < r0 + rows_per_chunk) ? B : r0 + rows_per_chunk;
    double a = 0.0, b = 0.0;
    if (col < H) {
        int64_t r = r0 + ry;
        for (; r + 24 < r1; r += 32) {             // 4 independent loads in flight per thread
            const double v0 = (double)x[r * H + col], v1 = (double)x[(r + 8) * H + col];
            const double v2 = (double)x[(r + 16) * H + col], v3 = (double)x[(r + 24) * H + col];
            a += (v0 + v1) + (v2 + v3);
            b += (v0 * v0 + v1 * v1) + (v2 * v2 + v3 * v3);
        }
        for (; r < r1; r += 8) { const double v = (double)x[r * H + col]; a += v; b += v * v; }
    }
    s1[ry][cx] = a; s2[ry][cx] = b;
    __syncthreads();
    if (ry == 0 && col < H) {
        double ta = 0.0, tb = 0.0;
#pragma unroll
        for (int i = 0; i < 8; ++i) { ta += s1[i][cx]; tb += s2[i][cx]; }
        atomicAdd(acc + col, ta);
        atomicAdd(acc + H + col, tb);
    }
}

template <typename T>
__global__ void bn_finish_stats_kernel(const double* __restrict__ acc, T* __restrict__ running_mean, T* __restrict__ running_var,
                                       T* __restrict__ save_mean, T* __restrict__ save_rstd, int64_t B, int H,
                                       double momentum, double eps, const double* __restrict__ count_dev) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= H) return;
    if (count_dev) B = (int64_t)(*count_dev + 0.5);          // synchronised statistics: the global row count, all-reduced with the sums
    const double mean = acc[col] / (double)B;
    double var = acc[H + col] / (double)B - mean * mean;
    if (var < 0.0) var = 0.0;
    save_mean[col] = (T)mean;
    save_rstd[col] = (T)(1.0 / sqrt(var + eps));
    if (running_mean) {
        const double unb = (B > 1) ? var * (double)B / (double)(B - 1) : var;
        running_mean[col] = (T)((1.0 - momentum) * (double)running_mean[col] + momentum * mean);
        running_var[col] = (T)((1.0 - momentum) * (double)running_var[col] + momentum * unb);
    }
}

static inline void bn_chunking(int64_t B, int H, int& chunks, int64_t& rpc) {
    const int64_t col_blocks = (H + 31) / 32;
    int64_t c = (4 * (int64_t)kNumSMs + col_blocks - 1) / col_blocks;      // ~4 CTAs per SM in total
    const int64_t maxc = (B + 255) / 256;                                  // at least 256 rows per chunk
    if (c > maxc) c = maxc;
    if (c < 1) c = 1;
    rpc = (B + c - 1) / c;
    rpc = (rpc + 7) / 8 * 8;
    chunks = (int)((B + rpc - 1) / rpc);
}

template <typename T>
__global__ void bn_eval_stats_kernel(const T* __restrict__ running_mean, const T* __restrict__ running_var,
                                     T* __restrict__ save_mean, T* __restrict__ save_rstd, int H, double eps) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < H) { save_mean[c] = running_mean[c]; save_rstd[c] = (T)(1.0 / sqrt((double)running_var[c] + eps)); }
}

// y = (x - mean) * rstd * gamma + beta with a fixed operation order (no compiler-chosen contraction): the 128-bit backward
// kernels re-derive the ReLU mask from x with this same function instead of reading y, so it has to be bit-identical in
// every forward variant
__device__ __forceinline__ float bn_affine(float x, float mu, float rs, float ga, float be) {
    return __fmaf_rn(__fmul_rn(__fsub_rn(x, mu), rs), ga, be);
}
__device__ __forceinline__ double bn_affine(double x, double mu, double rs, double ga, double be) {
    return (x - mu) * rs * ga + be;
}

template <typename T>
__global__ void bn_apply_kernel(const T* __restrict__ x, const T* __restrict__ gamma, const T* __restrict__ beta,
                                const T* __restrict__ mean, const T* __restrict__ rstd, T* __restrict__ y, int64_t B,
                                int H, int relu) {
    const int64_t n = B * H, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int c = (int)(i % H);
        T v = bn_affine(x[i], mean[c], rstd[c], gamma[c], beta[c]);
        y[i] = relu ? relu_nan(v) : v;
    }
}

// partial sums of ggamma = sum gy_eff*xhat and gbeta = sum gy_eff (gy_eff = gy * (y>0) when relu) into acc[2H]
template <typename T>
__global__ void __launch_bounds__(256)
bn_bwd_partial_kernel(const T* __restrict__ x, const T* __restrict__ y, const T* __restrict__ mean,
                      const T* __restrict__ rstd, const T* __restrict__ gy, double* __restrict__ acc, int64_t B, int H,
                      int relu, int64_t rows_per_chunk) {
    __shared__ double s1[8][33], s2[8][33];
    const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
    const int col = blockIdx.x * 32 + cx;
    const int64_t r0 = (int64_t)blockIdx.y * rows_per_chunk;
    const int64_t r1 = (B < r0 + rows_per_chunk) ? B : r0 + rows_per_chunk;
    double a = 0.0, b = 0.0;
    if (col < H) {
        const double mu = (double)mean[col], rs = (double)rstd[col];
        for (int64_t r = r0 + ry; r < r1; r += 8) {
            const int64_t o = r * H + col;
            double g = (double)gy[o];
            if (relu && !(y[o] > T(0))) g = 0.0;
            a += g * ((double)x[o] - mu) * rs;
            b += g;
        }
    }
    s1[ry][cx] = a; s2[ry][cx] = b;
    __syncthreads();
    if (ry == 0 && col < H) {
        double ta = 0.0, tb = 0.0;
#pragma unroll
        for (int i = 0; i < 8; ++i) { ta += s1[i][cx]; tb += s2[i][cx]; }
        atomicAdd(acc + col, ta);
        atomicAdd(acc + H + col, tb);
    }
}

template <typename T>
__global__ void bn_bwd_finish_kernel(const double* __restrict__ acc, T* __restrict__ ggamma, T* __restrict__ gbeta, int H) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col < H) { ggamma[col] = (T)acc[col]; gbeta[col] = (T)acc[H + col]; }
}

template <typename T>
__global__ void bn_bwd_apply_kernel(const T* __restrict__ x, const T* __restrict__ y, const T* __restrict__ gamma,
                                    const T* __restrict__ mean, const T* __restrict__ rstd, const T* __restrict__ gy,
                                    const T* __restrict__ ggamma, const T* __restrict__ gbeta, T* __restrict__ gx,
                                    int64_t B, int H, int relu, int training, int64_t count,
                                    const double* __restrict__ count_dev) {
    const int64_t n = B * H, stride = (int64_t)gridDim.x * blockDim.x;
    // rows behind the statistics: B, or the global count with synchronised statistics (host value or all-reduced on the device)
    const T invB = count_dev ? (T)(1.0 / *count_dev) : T(1) / (T)count;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int c = (int)(i % H);
        T g = gy[i];
        if (relu && !(y[i] > T(0))) g = T(0);
        if (training) {
            const T xhat = (x[i] - mean[c]) * rstd[c];
            gx[i] = gamma[c] * rstd[c] * (g - invB * (gbeta[c] + xhat * ggamma[c]));
        } else {
            gx[i] = gamma[c] * rstd[c] * g;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// float32, H % 4 == 0, 16-byte aligned: 128-bit versions of the four BatchNorm passes.  A block is TX column groups
// (4 columns each) x TY row lanes; a thread keeps its columns' statistics in registers and streams rows with four
// independent LDG.128 in flight.  (The scalar kernels above take `i % H` of a 64-bit index per element and move
// 4 bytes per load: 45 % of HBM; they remain the float64 / odd-H path.)  Same operation order per element.
// ------------------------------------------------------------------------------------------------
struct BnVecGeom { int tx, ty, col_blocks, chunks; int64_t rpc; };

static inline BnVecGeom bn_vec_geom(int64_t B, int H) {
    BnVecGeom g;
    const int q = H / 4;
    g.tx = 1;
    while (g.tx < q && g.tx < 256) g.tx <<= 1;
    g.ty = 256 / g.tx;
    g.col_blocks = (q + g.tx - 1) / g.tx;
    int64_t c = ((int64_t)kNumSMs * 6 + g.col_blocks - 1) / g.col_blocks;
    const int64_t maxc = (B + (int64_t)g.ty * 8 - 1) / ((int64_t)g.ty * 8);     // at least 8 rows per row lane
    if (c > maxc) c = maxc;
    if (c < 1) c = 1;
    g.rpc = (B + c - 1) / c;
    g.chunks = (int)((B + g.rpc - 1) / g.rpc);
    return g;
}

__device__ __forceinline__ float4 ld4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

__global__ void __launch_bounds__(256)
bn_partial_sums_vec4_kernel(const float* __restrict__ x, double* __restrict__ acc, int64_t B, int H, int64_t rpc, int tx) {
    extern __shared__ double bn_red[];                          // [ty][tx][8]
    const int ty = 256 / tx, cx = threadIdx.x & (tx - 1), ry = threadIdx.x / tx;
    const int col = (blockIdx.x * tx + cx) * 4;
    const int64_t r0 = (int64_t)blockIdx.y * rpc, r1 = (B < r0 + rpc) ? B : r0 + rpc;
    double a[4] = {0, 0, 0, 0}, b[4] = {0, 0, 0, 0};
    if (col < H) {
        const float* p = x + col;
        int64_t r = r0 + ry;
        for (; r + 3 * ty < r1; r += 4 * ty) {
            const float4 v0 = ld4(p + r * H), v1 = ld4(p + (r + ty) * H), v2 = ld4(p + (r + 2 * ty) * H), v3 = ld4(p + (r + 3 * ty) * H);
            a[0] += ((double)v0.x + v1.x) + ((double)v2.x + v3.x); b[0] += ((double)v0.x * v0.x + (double)v1.x * v1.x) + ((double)v2.x * v2.x + (double)v3.x * v3.x);
            a[1] += ((double)v0.y + v1.y) + ((double)v2.y + v3.y); b[1] += ((double)v0.y * v0.y + (double)v1.y * v1.y) + ((double)v2.y * v2.y + (double)v3.y * v3.y);
            a[2] += ((double)v0.z + v1.z) + ((double)v2.z + v3.z); b[2] += ((double)v0.z * v0.z + (double)v1.z * v1.z) + ((double)v2.z * v2.z + (double)v3.z * v3.z);
            a[3] += ((double)v0.w + v1.w) + ((double)v2.w + v3.w); b[3] += ((double)v0.w * v0.w + (double)v1.w * v1.w) + ((double)v2.w * v2.w + (double)v3.w * v3.w);
        }
        for (; r < r1; r += ty) {
            const float4 v = ld4(p + r * H);
            a[0] += v.x; b[0] += (double)v.x * v.x; a[1] += v.y; b[1] += (double)v.y * v.y;
            a[2] += v.z; b[2] += (double)v.z * v.z; a[3] += v.w; b[3] += (double)v.w * v.w;
        }
    }
    double* mine = bn_red + ((size_t)ry * tx + cx) * 8;
#pragma unroll
    for (int j = 0; j < 4; ++j) { mine[j] = a[j]; mine[4 + j] = b[j]; }
    __syncthreads();
    if (ry == 0 && col < H) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double ta = 0.0, tb = 0.0;
            for (int i = 0; i < ty; ++i) { ta += bn_red[((size_t)i * tx + cx) * 8 + j]; tb += bn_red[((size_t)i * tx + cx) * 8 + 4 + j]; }
            atomicAdd(acc + col + j, ta);
            atomicAdd(acc + H + col + j, tb);
        }
    }
}

__global__ void __launch_bounds__(256)
bn_apply_vec4_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                     const float* __restrict__ mean, const float* __restrict__ rstd, float* __restrict__ y, int64_t B, int H,
                     int relu, int64_t rpc, int tx) {
    const int ty = 256 / tx, cx = threadIdx.x & (tx - 1), ry = threadIdx.x / tx;
    const int col = (blockIdx.x * tx + cx) * 4;
    if (col >= H) return;
    const float4 mu = ld4(mean + col), rs = ld4(rstd + col), ga = ld4(gamma + col), be = ld4(beta + col);
    const int64_t r0 = (int64_t)blockIdx.y * rpc, r1 = (B < r0 + rpc) ? B : r0 + rpc;
    const float* p = x + col;
    float* o = y + col;
#pragma unroll 4
    for (int64_t r = r0 + ry; r < r1; r += ty) {
        const float4 v = __ldcs(reinterpret_cast<const float4*>(p + r * H));
        float4 w;
        w.x = bn_affine(v.x, mu.x, rs.x, ga.x, be.x); w.y = bn_affine(v.y, mu.y, rs.y, ga.y, be.y);
        w.z = bn_affine(v.z, mu.z, rs.z, ga.z, be.z); w.w = bn_affine(v.w, mu.w, rs.w, ga.w, be.w);
        if (relu) { w.x = relu_nan(w.x); w.y = relu_nan(w.y); w.z = relu_nan(w.z); w.w = relu_nan(w.w); }
        *reinterpret_cast<float4*>(o + r * H) = w;
    }
}

__global__ void __launch_bounds__(256)
bn_bwd_partial_vec4_kernel(const float* __restrict__ x, const float* __restrict__ y, const float* __restrict__ mean,
                           const float* __restrict__ rstd, const float* __restrict__ gy, double* __restrict__ acc, int64_t B,
                           int H, int relu, int64_t rpc, int tx, const float* __restrict__ gamma_m,
                           const float* __restrict__ beta_m) {
    // gamma_m / beta_m != nullptr: the ReLU mask comes from bn_affine(x) (what the forward computed before its ReLU), y is
    // not read -- a third less traffic for this pass
    extern __shared__ double bn_red[];
    const int ty = 256 / tx, cx = threadIdx.x & (tx - 1), ry = threadIdx.x / tx;
    const int col = (blockIdx.x * tx + cx) * 4;
    const int64_t r0 = (int64_t)blockIdx.y * rpc, r1 = (B < r0 + rpc) ? B : r0 + rpc;
    double a[4] = {0, 0, 0, 0}, b[4] = {0, 0, 0, 0};
    if (col < H) {
        const float4 mu4 = ld4(mean + col), rs4 = ld4(rstd + col);
        const double mu[4] = {mu4.x, mu4.y, mu4.z, mu4.w}, rs[4] = {rs4.x, rs4.y, rs4.z, rs4.w};
        const bool remask = relu && gamma_m != nullptr;
        const float4 ga4 = remask ? ld4(gamma_m + col) : make_float4(0.f, 0.f, 0.f, 0.f), be4 = remask ? ld4(beta_m + col) : ga4;
        const float muf[4] = {mu4.x, mu4.y, mu4.z, mu4.w}, rsf[4] = {rs4.x, rs4.y, rs4.z, rs4.w};
        const float gaf[4] = {ga4.x, ga4.y, ga4.z, ga4.w}, bef[4] = {be4.x, be4.y, be4.z, be4.w};
#pragma unroll 2
        for (int64_t r = r0 + ry; r < r1; r += ty) {
            const int64_t off = r * H + col;
            const float4 g4 = ld4(gy + off), x4 = ld4(x + off);
            float g[4] = {g4.x, g4.y, g4.z, g4.w};
            const float xv[4] = {x4.x, x4.y, x4.z, x4.w};
            if (remask) {
#pragma unroll
                for (int j = 0; j < 4; ++j) if (!(bn_affine(xv[j], muf[j], rsf[j], gaf[j], bef[j]) > 0.f)) g[j] = 0.f;
            } else if (relu) {
                const float4 y4 = ld4(y + off);
                if (!(y4.x > 0.f)) g[0] = 0.f;
                if (!(y4.y > 0.f)) g[1] = 0.f;
                if (!(y4.z > 0.f)) g[2] = 0.f;
                if (!(y4.w > 0.f)) g[3] = 0.f;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) { a[j] += (double)g[j] * ((double)xv[j] - mu[j]) * rs[j]; b[j] += (double)g[j]; }
        }
    }
    double* mine = bn_red + ((size_t)ry * tx + cx) * 8;
#pragma unroll
    for (int j = 0; j < 4; ++j) { mine[j] = a[j]; mine[4 + j] = b[j]; }
    __syncthreads();
    if (ry == 0 && col < H) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double ta = 0.0, tb = 0.0;
            for (int i = 0; i < ty; ++i) { ta += bn_red[((size_t)i * tx + cx) * 8 + j]; tb += bn_red[((size_t)i * tx + cx) * 8 + 4 + j]; }
            atomicAdd(acc + col + j, ta);
            atomicAdd(acc + H + col + j, tb);
        }
    }
}

__global__ void __launch_bounds__(256)
bn_bwd_apply_vec4_kernel(const float* __restrict__ x, const float* __restrict__ y, const float* __restrict__ gamma,
                         const float* __restrict__ mean, const float* __restrict__ rstd, const float* __restrict__ gy,
                         const float* __restrict__ ggamma, const float* __restrict__ gbeta, float* __restrict__ gx, int64_t B,
                         int H, int relu, int training, int64_t rpc, int tx, int64_t count, const double* __restrict__ count_dev,
                         const float* __restrict__ beta_m) {
    const int ty = 256 / tx, cx = threadIdx.x & (tx - 1), ry = threadIdx.x / tx;
    const int col = (blockIdx.x * tx + cx) * 4;
    if (col >= H) return;
    const float4 mu4 = ld4(mean + col), rs4 = ld4(rstd + col), ga4 = ld4(gamma + col), gg4 = ld4(ggamma + col), gb4 = ld4(gbeta + col);
    const float mu[4] = {mu4.x, mu4.y, mu4.z, mu4.w}, rs[4] = {rs4.x, rs4.y, rs4.z, rs4.w}, ga[4] = {ga4.x, ga4.y, ga4.z, ga4.w};
    const float gg[4] = {gg4.x, gg4.y, gg4.z, gg4.w}, gb[4] = {gb4.x, gb4.y, gb4.z, gb4.w};
    const float invB = count_dev ? (float)(1.0 / *count_dev) : 1.0f / (float)count;
    const int64_t r0 = (int64_t)blockIdx.y * rpc, r1 = (B < r0 + rpc) ? B : r0 + rpc;
    const bool remask = relu && beta_m != nullptr;            // ReLU mask from bn_affine(x) instead of y (see the partial kernel)
    const float4 be4 = remask ? ld4(beta_m + col) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float be[4] = {be4.x, be4.y, be4.z, be4.w};
#pragma unroll 2
    for (int64_t r = r0 + ry; r < r1; r += ty) {
        const int64_t off = r * H + col;
        const float4 g4 = __ldcs(reinterpret_cast<const float4*>(gy + off));
        float g[4] = {g4.x, g4.y, g4.z, g4.w};
        float4 x4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (training || remask) x4 = __ldcs(reinterpret_cast<const float4*>(x + off));
        const float xv[4] = {x4.x, x4.y, x4.z, x4.w};
        if (remask) {
#pragma unroll
            for (int j = 0; j < 4; ++j) if (!(bn_affine(xv[j], mu[j], rs[j], ga[j], be[j]) > 0.f)) g[j] = 0.f;
        } else if (relu) {
            const float4 y4 = __ldcs(reinterpret_cast<const float4*>(y + off));
            if (!(y4.x > 0.f)) g[0] = 0.f;
            if (!(y4.y > 0.f)) g[1] = 0.f;
            if (!(y4.z > 0.f)) g[2] = 0.f;
            if (!(y4.w > 0.f)) g[3] = 0.f;
        }
        float o[4];
        if (training) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float xhat = (xv[j] - mu[j]) * rs[j];
                o[j] = ga[j] * rs[j] * (g[j] - invB * (gb[j] + xhat * gg[j]));
            }
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) o[j] = ga[j] * rs[j] * g[j];
        }
        *reinterpret_cast<float4*>(gx + off) = make_float4(o[0], o[1], o[2], o[3]);
    }
}

static inline bool bn_vec_ok(int H, const void* a, const void* b, const void* c, const void* d) {
    return H % 4 == 0 && H >= 16 && aligned16(a) && aligned16(b) && (!c || aligned16(c)) && (!d || aligned16(d));
}

// ReLU backward fused with the column sums of its result (the bias gradient of the Linear the ReLU belongs to): gx = gy
// where y > 0, out[c] += sum_rows gx[:, c].  As two kernels the [B, H] gradient was written by relu_bwd_kernel and read
// again by col_sum_vec4_kernel (16 x 62 us per training step of the 2-D spline stack at 2^20 rows).  float32, H % 4 == 0,
// 16-byte aligned; `out` must be zero on entry; per-thread float sums, chunk sums in double, one float atomic per column and
// chunk (like col_sum_vec4_kernel).
__global__ void __launch_bounds__(256)
relu_bwd_colsum_vec4_kernel(const float* __restrict__ y, const float* __restrict__ gy, float* __restrict__ gx,
                            float* __restrict__ out, int64_t B, int H, int64_t rpc, int tx) {
    extern __shared__ double bn_red[];                          // [ty][tx][4]
    const int ty = 256 / tx, cx = threadIdx.x & (tx - 1), ry = threadIdx.x / tx;
    const int col = (blockIdx.x * tx + cx) * 4;
    const int64_t r0 = (int64_t)blockIdx.y * rpc, r1 = (B < r0 + rpc) ? B : r0 + rpc;
    float4 s0 = make_float4(0.f, 0.f, 0.f, 0.f), s1 = s0;
    if (col < H) {
        int64_t r = r0 + ry;
        for (; r + ty < r1; r += 2 * ty) {
            const int64_t o0 = r * H + col, o1 = (r + ty) * H + col;
            const float4 ga = __ldcs(reinterpret_cast<const float4*>(gy + o0)), ya = __ldcs(reinterpret_cast<const float4*>(y + o0));
            const float4 gb = __ldcs(reinterpret_cast<const float4*>(gy + o1)), yb = __ldcs(reinterpret_cast<const float4*>(y + o1));
            const float4 a = make_float4(ya.x > 0.f ? ga.x : 0.f, ya.y > 0.f ? ga.y : 0.f, ya.z > 0.f ? ga.z : 0.f, ya.w > 0.f ? ga.w : 0.f);
            const float4 b = make_float4(yb.x > 0.f ? gb.x : 0.f, yb.y > 0.f ? gb.y : 0.f, yb.z > 0.f ? gb.z : 0.f, yb.w > 0.f ? gb.w : 0.f);
            *reinterpret_cast<float4*>(gx + o0) = a;
            *reinterpret_cast<float4*>(gx + o1) = b;
            s0.x += a.x; s0.y += a.y; s0.z += a.z; s0.w += a.w;
            s1.x += b.x; s1.y += b.y; s1.z += b.z; s1.w += b.w;
        }
        for (; r < r1; r += ty) {
            const int64_t o0 = r * H + col;
            const float4 ga = __ldcs(reinterpret_cast<const float4*>(gy + o0)), ya = __ldcs(reinterpret_cast<const float4*>(y + o0));
            const float4 a = make_float4(ya.x > 0.f ? ga.x : 0.f, ya.y > 0.f ? ga.y : 0.f, ya.z > 0.f ? ga.z : 0.f, ya.w > 0.f ? ga.w : 0.f);
            *reinterpret_cast<float4*>(gx + o0) = a;
            s0.x += a.x; s0.y += a.y; s0.z += a.z; s0.w += a.w;
        }
    }
    double* mine = bn_red + ((size_t)ry * tx + cx) * 4;
    mine[0] = (double)s0.x + s1.x; mine[1] = (double)s0.y + s1.y; mine[2] = (double)s0.z + s1.z; mine[3] = (double)s0.w + s1.w;
    __syncthreads();
    if (ry == 0 && col < H) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double t = 0.0;
            for (int i = 0; i < ty; ++i) t += bn_red[((size_t)i * tx + cx) * 4 + j];
            atomicAdd(out + col + j, (float)t);
        }
    }
}

static inline int ew_grid(int64_t n) {
    int64_t need = cdiv(n, 256);
    int64_t cap = (int64_t)kNumSMs * 16;
    return (int)(need < 1 ? 1 : (need < cap ? need : cap));
}

template <typename T>
// stage 0: the whole pass.  Synchronised statistics (data-parallel training, SURVEY 8e: exact N-GPU == 1-GPU equivalence
// of CouplingLayer's train-mode BatchNorm needs the (sum x, sum x^2, n) triples all-reduced): stage 1 = this shard's sums
// into ws and return; the caller all-reduces ws; stage 2 = statistics from ws over `count` rows, running-stat update,
// apply to this shard's B rows.
static int bn_forward(const void* x, const void* gamma, const void* beta, void* rm, void* rv, void* y, void* sm,
                      void* sr, void* ws, int64_t B, int H, int training, double momentum, double eps, int relu,
                      cudaStream_t st, int stage = 0, int64_t count = 0) {
    const bool vec = sizeof(T) == 4 && bn_vec_ok(H, x, y ? y : x, gamma ? gamma : x, beta ? beta : x) &&
                     (sm == nullptr || aligned16(sm)) && (sr == nullptr || aligned16(sr));
    const BnVecGeom vg = bn_vec_geom(B, H);
    const bool count_on_device = (stage == 2 && count < 0);     // workspace[2H] holds the all-reduced row count (no host read)
    if (count <= 0) count = B;
    if (training) {
        if (stage != 2) {
            NF_CUDA(cudaMemsetAsync(ws, 0, sizeof(double) * 2 * H, st));
            int chunks; int64_t rpc;
            bn_chunking(B, H, chunks, rpc);
            dim3 grid((unsigned)((H + 31) / 32), (unsigned)chunks);
            if (vec)
                bn_partial_sums_vec4_kernel<<<dim3((unsigned)vg.col_blocks, (unsigned)vg.chunks), 256, sizeof(double) * 256 * 8, st>>>(
                    (const float*)x, (double*)ws, B, H, vg.rpc, vg.tx);
            else
                bn_partial_sums_kernel<T><<<grid, 256, 0, st>>>((const T*)x, (double*)ws, B, H, rpc);
            count_launch();
            NF_LAUNCH_CHECK();
            if (stage == 1) return NF_OK;
        }
        bn_finish_stats_kernel<T><<<(H + 127) / 128, 128, 0, st>>>((const double*)ws, (T*)rm, (T*)rv, (T*)sm, (T*)sr, count, H,
                                                                  momentum, eps, count_on_device ? (const double*)ws + 2 * H : nullptr);
    } else {
        bn_eval_stats_kernel<T><<<(H + 255) / 256, 256, 0, st>>>((const T*)rm, (const T*)rv, (T*)sm, (T*)sr, H, eps);
    }
    count_launch();
    NF_LAUNCH_CHECK();
    if (B == 0) return NF_OK;                    // empty shard of a synchronised pass: statistics only
    if (vec)
        bn_apply_vec4_kernel<<<dim3((unsigned)vg.col_blocks, (unsigned)vg.chunks), 256, 0, st>>>(
            (const float*)x, (const float*)gamma, (const float*)beta, (const float*)sm, (const float*)sr, (float*)y, B, H, relu, vg.rpc, vg.tx);
    else
    bn_apply_kernel<T><<<ew_grid(B * H), 256, 0, st>>>((const T*)x, (const T*)gamma, (const T*)beta, (const T*)sm,
                                                       (const T*)sr, (T*)y, B, H, relu);
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

template <typename T>
// stage 0: the whole pass.  Synchronised statistics: stage 1 = this shard's (sum g*xhat, sum g) into ws and return (they
// are also this shard's ggamma / gbeta); the caller all-reduces a copy; stage 2 = gx of this shard's rows from the
// all-reduced sums in ws over `count` rows (gg / gb receive the GLOBAL sums as a by-product).
static int bn_backward(const void* x, const void* y, const void* gamma, const void* sm, const void* sr, const void* gy,
                       void* gx, void* gg, void* gb, void* ws, int64_t B, int H, int relu, int training, cudaStream_t st,
                       int stage = 0, int64_t count = 0, const void* beta = nullptr) {
    int chunks; int64_t rpc;
    bn_chunking(B, H, chunks, rpc);
    dim3 grid((unsigned)((H + 31) / 32), (unsigned)chunks);
    const bool vec = sizeof(T) == 4 && bn_vec_ok(H, x, gy, y, gx ? gx : x) && aligned16(sm) && aligned16(sr) &&
                     (gamma == nullptr || aligned16(gamma)) && (gg == nullptr || aligned16(gg)) && (gb == nullptr || aligned16(gb));
    // mask parameters of the 128-bit kernels (nullptr: read y)
    const float* gamma_m = (relu && gamma && beta && aligned16(beta) && aligned16(gamma)) ? (const float*)gamma : nullptr;
    const float* beta_m = gamma_m ? (const float*)beta : nullptr;
    const BnVecGeom vg = bn_vec_geom(B, H);
    const double* count_dev = (stage == 2 && count < 0) ? (const double*)ws + 2 * H : nullptr;
    if (count <= 0) count = B;
    if (stage != 2) {
        NF_CUDA(cudaMemsetAsync(ws, 0, sizeof(double) * 2 * H, st));
        if (vec)
            bn_bwd_partial_vec4_kernel<<<dim3((unsigned)vg.col_blocks, (unsigned)vg.chunks), 256, sizeof(double) * 256 * 8, st>>>(
                (const float*)x, (const float*)y, (const float*)sm, (const float*)sr, (const float*)gy, (double*)ws, B, H, relu, vg.rpc, vg.tx, gamma_m, beta_m);
        else
            bn_bwd_partial_kernel<T><<<grid, 256, 0, st>>>((const T*)x, (const T*)y, (const T*)sm, (const T*)sr, (const T*)gy,
                                                           (double*)ws, B, H, relu, rpc);
        count_launch();
        NF_LAUNCH_CHECK();
        if (stage == 1) return NF_OK;
    }
    bn_bwd_finish_kernel<T><<<(H + 127) / 128, 128, 0, st>>>((const double*)ws, (T*)gg, (T*)gb, H);
    count_launch();
    NF_LAUNCH_CHECK();
    if (vec)
        bn_bwd_apply_vec4_kernel<<<dim3((unsigned)vg.col_blocks, (unsigned)vg.chunks), 256, 0, st>>>(
            (const float*)x, (const float*)y, (const float*)gamma, (const float*)sm, (const float*)sr, (const float*)gy,
            (const float*)gg, (const float*)gb, (float*)gx, B, H, relu, training, vg.rpc, vg.tx, count, count_dev, beta_m);
    else
    bn_bwd_apply_kernel<T><<<ew_grid(B * H), 256, 0, st>>>((const T*)x, (const T*)y, (const T*)gamma, (const T*)sm,
                                                           (const T*)sr, (const T*)gy, (const T*)gg, (const T*)gb,
                                                           (T*)gx, B, H, relu, training, count, count_dev);
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

}  // namespace nf

using namespace nf;
#define NF_REQ(p) do { if ((p) == nullptr) return NF_ERR_NULL; } while (0)

extern "C" int nf_gemm(const void* A, const void* Bm, void* C, const void* bias, int64_t M, int64_t N, int64_t K,
                       int64_t sam, int64_t sak, int64_t sbk, int64_t sbn, int64_t ldc, int relu, int accumulate,
                       const int32_t* k_extent, int dtype, nf_stream_t stream) {
    if (M < 0 || N < 0 || K < 0 || ldc < N) return NF_ERR_BAD_SHAPE;
    if (M == 0 || N == 0) return NF_OK;
    NF_REQ(C);
    if (K > 0) { NF_REQ(A); NF_REQ(Bm); }
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == NF_F32)
        return gemm_launch<float>(A, Bm, C, bias, M, N, K, sam, sak, sbk, sbn, ldc, relu, accumulate, k_extent, st);
    if (dtype == NF_F64)
        return gemm_launch<double>(A, Bm, C, bias, M, N, K, sam, sak, sbk, sbn, ldc, relu, accumulate, k_extent, st);
    return NF_ERR_UNSUPPORTED;
}

extern "C" int nf_mul_rows(const void* a, const void* b, void* out, int64_t rows, int64_t cols, int64_t b_rows,
                           int dtype, nf_stream_t stream) {
    if (rows < 0 || cols < 0 || (b_rows != 1 && b_rows != rows)) return NF_ERR_BAD_SHAPE;
    if (rows * cols == 0) return NF_OK;
    NF_REQ(a); NF_REQ(b); NF_REQ(out);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == NF_F32)
        mul_rows_kernel<float><<<ew_grid(rows * cols), 256, 0, st>>>((const float*)a, (const float*)b, (float*)out, rows, cols, b_rows);
    else if (dtype == NF_F64)
        mul_rows_kernel<double><<<ew_grid(rows * cols), 256, 0, st>>>((const double*)a, (const double*)b, (double*)out, rows, cols, b_rows);
    else return NF_ERR_UNSUPPORTED;
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

extern "C" int nf_col_sum(const void* a, void* out, int64_t rows, int64_t cols, int dtype, nf_stream_t stream);
extern "C" int nf_relu_backward(const void* y, const void* gy, void* gx, int64_t n, int dtype, nf_stream_t stream);

// gx = gy * (y > 0) and colsum[c] = sum_rows gx[:, c] (the ReLU backward of a Linear(+ReLU) and its bias gradient) in one pass
extern "C" int nf_relu_backward_colsum(const void* y, const void* gy, void* gx, void* colsum, int64_t rows, int64_t cols,
                                       int dtype, nf_stream_t stream) {
    if (rows < 0 || cols < 0) return NF_ERR_BAD_SHAPE;
    if (cols == 0) return NF_OK;
    NF_REQ(colsum);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == NF_F32 && rows >= 1024 && cols >= 16 && cols <= 2147483647LL && bn_vec_ok((int)cols, y, gy, gx, colsum)) {
        NF_REQ(y); NF_REQ(gy); NF_REQ(gx);
        const BnVecGeom vg = bn_vec_geom(rows, (int)cols);
        NF_CUDA(cudaMemsetAsync(colsum, 0, sizeof(float) * cols, st));
        relu_bwd_colsum_vec4_kernel<<<dim3((unsigned)vg.col_blocks, (unsigned)vg.chunks), 256, sizeof(double) * 256 * 4, st>>>(
            (const float*)y, (const float*)gy, (float*)gx, (float*)colsum, rows, (int)cols, vg.rpc, vg.tx);
        count_launch();
        NF_LAUNCH_CHECK();
        return NF_OK;
    }
    const int rc = nf_relu_backward(y, gy, gx, rows * cols, dtype, stream);
    if (rc != NF_OK) return rc;
    return nf_col_sum(gx, colsum, rows, cols, dtype, stream);
}

extern "C" int nf_relu_backward(const void* y, const void* gy, void* gx, int64_t n, int dtype, nf_stream_t stream) {
    if (n < 0) return NF_ERR_BAD_SHAPE;
    if (n == 0) return NF_OK;
    NF_REQ(y); NF_REQ(gy); NF_REQ(gx);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == NF_F32) relu_bwd_kernel<float><<<ew_grid(n), 256, 0, st>>>((const float*)y, (const float*)gy, (float*)gx, n);
    else if (dtype == NF_F64) relu_bwd_kernel<double><<<ew_grid(n), 256, 0, st>>>((const double*)y, (const double*)gy, (double*)gx, n);
    else return NF_ERR_UNSUPPORTED;
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

extern "C" int nf_col_sum(const void* a, void* out, int64_t rows, int64_t cols, int dtype, nf_stream_t stream) {
    if (rows < 0 || cols < 0) return NF_ERR_BAD_SHAPE;
    if (cols == 0) return NF_OK;
    NF_REQ(out);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t es = dtype == NF_F64 ? 8 : 4;
    const int64_t rows1 = rows > 1 ? rows : 1;
    if (dtype == NF_F32 && rows >= 1024 && cols % 4 == 0 && a && aligned16(a)) {
        const int64_t cblocks = cdiv(cols, 128);
        int64_t ch = cdiv((int64_t)kNumSMs * 6, cblocks);               // ~6 CTAs of 256 threads per SM
        const int64_t chmax = rows / 256;                                // at least 256 rows (32 per row-lane) per chunk
        if (ch > chmax) ch = chmax;
        if (ch < 1) ch = 1;
        const int64_t rpc4 = cdiv(rows, ch);
        ch = cdiv(rows, rpc4);
        if (ch > 65535) return NF_ERR_BAD_SHAPE;
        if (ch > 1) NF_CUDA(cudaMemsetAsync(out, 0, es * cols, st));
        col_sum_vec4_kernel<<<dim3((unsigned)cblocks, (unsigned)ch), 256, 0, st>>>((const float*)a, (float*)out, rows, cols, rpc4);
        count_launch();
        NF_LAUNCH_CHECK();
        return NF_OK;
    }
    if ((cols <= 8 || (cols <= 32 && cols % 4 != 0)) && rows >= 1 && a) {
        int rc = dtype == NF_F32 ? col_sum_small_launch<float>(a, out, rows, (int)cols, st)
               : dtype == NF_F64 ? col_sum_small_launch<double>(a, out, rows, (int)cols, st) : NF_ERR_UNSUPPORTED;
        if (rc) return rc;
        count_launch();
        NF_LAUNCH_CHECK();
        return NF_OK;
    }
    int chunks = (int)(rows / 4096 < 1 ? 1 : (rows / 4096 > 64 ? 64 : rows / 4096));
    const int64_t rpc = cdiv(rows1, chunks);
    chunks = (int)cdiv(rows1, rpc);
    if (chunks > 1 || rows == 0) NF_CUDA(cudaMemsetAsync(out, 0, es * cols, st));
    if (rows == 0) return NF_OK;
    NF_REQ(a);
    dim3 grid((unsigned)cdiv(cols, 32), (unsigned)chunks);
    if (dtype == NF_F32) col_sum_kernel<float><<<grid, 256, 0, st>>>((const float*)a, (float*)out, rows, cols, rpc);
    else if (dtype == NF_F64) col_sum_kernel<double><<<grid, 256, 0, st>>>((const double*)a, (double*)out, rows, cols, rpc);
    else return NF_ERR_UNSUPPORTED;
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

extern "C" int nf_batchnorm_forward(const void* x, const void* gamma, const void* beta, void* running_mean,
                                    void* running_var, void* y, void* save_mean, void* save_rstd, void* workspace,
                                    int64_t B, int H, int training, double momentum, double eps, int relu, int dtype,
                                    nf_stream_t stream) {
    if (B < 0 || H < 1) return NF_ERR_BAD_SHAPE;
    if (B == 0) return NF_OK;
    NF_REQ(x); NF_REQ(gamma); NF_REQ(beta); NF_REQ(y); NF_REQ(save_mean); NF_REQ(save_rstd);
    if (!training) { NF_REQ(running_mean); NF_REQ(running_var); } else { NF_REQ(workspace); }
    if ((running_mean == nullptr) != (running_var == nullptr)) return NF_ERR_NULL;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == NF_F32)
        return bn_forward<float>(x, gamma, beta, running_mean, running_var, y, save_mean, save_rstd, workspace, B, H, training, momentum, eps, relu, st);
    if (dtype == NF_F64)
        return bn_forward<double>(x, gamma, beta, running_mean, running_var, y, save_mean, save_rstd, workspace, B, H, training, momentum, eps, relu, st);
    return NF_ERR_UNSUPPORTED;
}

extern "C" int nf_batchnorm_forward_staged(const void* x, const void* gamma, const void* beta, void* running_mean,
                                           void* running_var, void* y, void* save_mean, void* save_rstd, void* workspace,
                                           int64_t B, int H, double momentum, double eps, int relu, int stage, int64_t count,
                                           int dtype, nf_stream_t stream) {
    if (B < 0 || H < 1 || (stage != 1 && stage != 2)) return NF_ERR_BAD_SHAPE;
    NF_REQ(workspace);
    if (stage == 2) {
        if (count < 1 && count != -1) return NF_ERR_BAD_SHAPE;
        NF_REQ(gamma); NF_REQ(beta); NF_REQ(save_mean); NF_REQ(save_rstd);
        if (B > 0) { NF_REQ(x); NF_REQ(y); }
    } else if (B > 0) {
        NF_REQ(x);
    }
    if ((running_mean == nullptr) != (running_var == nullptr)) return NF_ERR_NULL;
    cudaStream_t st = (cudaStream_t)stream;
    if (B == 0 && stage == 1) return cudaMemsetAsync(workspace, 0, sizeof(double) * 2 * H, st) == cudaSuccess ? NF_OK : NF_ERR_CUDA;
    if (dtype == NF_F32)
        return bn_forward<float>(x, gamma, beta, running_mean, running_var, y, save_mean, save_rstd, workspace, B, H, 1, momentum, eps, relu, st, stage, count);
    if (dtype == NF_F64)
        return bn_forward<double>(x, gamma, beta, running_mean, running_var, y, save_mean, save_rstd, workspace, B, H, 1, momentum, eps, relu, st, stage, count);
    return NF_ERR_UNSUPPORTED;
}

extern "C" int nf_batchnorm_backward_staged(const void* x, const void* y, const void* gamma, const void* save_mean,
                                            const void* save_rstd, const void* gy, void* gx, void* ggamma, void* gbeta,
                                            void* workspace, int64_t B, int H, int relu, int stage, int64_t count, int dtype,
                                            const void* beta, nf_stream_t stream) {
    if (B < 0 || H < 1 || (stage != 1 && stage != 2)) return NF_ERR_BAD_SHAPE;
    NF_REQ(workspace); NF_REQ(save_mean); NF_REQ(save_rstd);
    cudaStream_t st = (cudaStream_t)stream;
    if (stage == 2) {
        if (count < 1 && count != -1) return NF_ERR_BAD_SHAPE;
        NF_REQ(gamma); NF_REQ(ggamma); NF_REQ(gbeta);
    }
    if (B == 0) {
        if (stage == 1) return cudaMemsetAsync(workspace, 0, sizeof(double) * 2 * H, st) == cudaSuccess ? NF_OK : NF_ERR_CUDA;
        return NF_OK;
    }
    NF_REQ(x); NF_REQ(y); NF_REQ(gy);
    if (stage == 2) NF_REQ(gx);
    if (dtype == NF_F32)
        return bn_backward<float>(x, y, gamma, save_mean, save_rstd, gy, gx, ggamma, gbeta, workspace, B, H, relu, 1, st, stage, count, beta);
    if (dtype == NF_F64)
        return bn_backward<double>(x, y, gamma, save_mean, save_rstd, gy, gx, ggamma, gbeta, workspace, B, H, relu, 1, st, stage, count);
    return NF_ERR_UNSUPPORTED;
}

extern "C" int nf_batchnorm_backward(const void* x, const void* y, const void* gamma, const void* save_mean,
                                     const void* save_rstd, const void* gy, void* gx, void* ggamma, void* gbeta,
                                     void* workspace, int64_t B, int H, int relu, int training, int dtype,
                                     const void* beta, nf_stream_t stream) {
    if (B < 0 || H < 1) return NF_ERR_BAD_SHAPE;
    if (B == 0) return NF_OK;
    NF_REQ(x); NF_REQ(y); NF_REQ(gamma); NF_REQ(save_mean); NF_REQ(save_rstd); NF_REQ(gy); NF_REQ(gx); NF_REQ(ggamma); NF_REQ(gbeta); NF_REQ(workspace);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == NF_F32)
        return bn_backward<float>(x, y, gamma, save_mean, save_rstd, gy, gx, ggamma, gbeta, workspace, B, H, relu, training, st, 0, 0, beta);
    if (dtype == NF_F64)
        return bn_backward<double>(x, y, gamma, save_mean, save_rstd, gy, gx, ggamma, gbeta, workspace, B, H, relu, training, st);
    return NF_ERR_UNSUPPORTED;
}
