// aux_kernels.cu -- the remaining [B,D]-sized pieces of the layered (training / float64) route:
//   nf_feature_affine_*   per-feature affine  y = (x - sub[d]) / div[d] * mul[d] + add[d]
//                         = between-layer BatchNorm on running statistics and its inverse
//                           (normalizing_flow_model.py:67-85, :110-128) and the spline layer's
//                           data_min/data_max rescale of the conditioner input (spline_coupling_layer.py:78-94)
//   nf_col_stats          per-feature batch mean / biased variance (running-stat update, normalizing_flow_model.py:74-79)
//   nf_ar_step_*          one step of the sequential autoregressive loop
//                         (masked_autoregressive_flow.py:55-67, inverse_autoregressive_flow.py:76-91)
//   nf_ar_finish_*        the NaN/Inf scrubs and log-det clamp that close that loop (:69-76 / :93-101)
// All are streaming, HBM-bound kernels; reductions over rows accumulate in double.
#include "nf_common.cuh"
#include "nf_rng.cuh"

namespace nf {

static inline int ew_grid(int64_t n) {
    int64_t need = cdiv(n, 256);
    int64_t cap = (int64_t)kNumSMs * 16;
    return (int)(need < 1 ? 1 : (need < cap ? need : cap));
}

template <typename T>
__global__ void __launch_bounds__(256)
feature_affine_fwd_kernel(const T* __restrict__ x, const T* __restrict__ sub, const T* __restrict__ div,
                          const T* __restrict__ mul, const T* __restrict__ add, T add_scalar, T* __restrict__ y,
                          int64_t B, int D) {
    const int64_t n = B * D, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int d = (int)(i % D);
        T v = x[i];
        if (sub) v = v - sub[d];
        if (div) v = v / div[d];
        if (mul) v = v * mul[d];
        v = v + (add ? add[d] : add_scalar);
        y[i] = v;
    }
}

// float32, 16-byte aligned x / y, D % 4 == 0 or D in {1, 2}: 128-bit loads / stores, two chunks in flight per thread, the
// per-column constants of a chunk fetched as one float4 (the scalar kernel above takes a 64-bit `i % D` and an IEEE
// division per 4-byte access: 40 % of HBM).  PERIOD = 4 (D % 4 == 0: the chunk's columns are col..col+3), 2 (D == 2:
// columns 0,1,0,1), 1 (D == 1).  Same operation order per element: ((x - sub) / div) * mul + add.
template <int PERIOD>
__global__ void __launch_bounds__(256)
feature_affine_fwd_vec4_kernel(const float* __restrict__ x, const float* __restrict__ sub, const float* __restrict__ div,
                               const float* __restrict__ mul, const float* __restrict__ add, float add_scalar,
                               float* __restrict__ y, int64_t nchunks, int D) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t c0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    auto col_of = [&](int64_t c) -> int { return PERIOD == 4 ? (int)((c * 4) % D) : 0; };
    auto params = [&](const float* p, int col, float dflt, float (&o)[4]) {
        if (!p) { o[0] = o[1] = o[2] = o[3] = dflt; return; }
        if (PERIOD == 4) { const float4 v = __ldg(reinterpret_cast<const float4*>(p + col)); o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w; }
        else if (PERIOD == 2) { o[0] = o[2] = __ldg(p); o[1] = o[3] = __ldg(p + 1); }
        else { o[0] = o[1] = o[2] = o[3] = __ldg(p); }
    };
    auto apply = [&](const float4 v, int col) -> float4 {
        float s4[4], d4[4], m4[4], a4[4], e[4] = {v.x, v.y, v.z, v.w};
        params(sub, col, 0.f, s4); params(div, col, 1.f, d4); params(mul, col, 1.f, m4); params(add, col, add_scalar, a4);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float t = e[j];
            if (sub) t = t - s4[j];
            if (div) t = t / d4[j];
            if (mul) t = t * m4[j];
            e[j] = t + a4[j];
        }
        return make_float4(e[0], e[1], e[2], e[3]);
    };
    int64_t c = c0;
    for (; c + stride < nchunks; c += 2 * stride) {
        const float4 v0 = __ldcs(reinterpret_cast<const float4*>(x) + c);
        const float4 v1 = __ldcs(reinterpret_cast<const float4*>(x) + c + stride);
        __stcs(reinterpret_cast<float4*>(y) + c, apply(v0, col_of(c)));
        __stcs(reinterpret_cast<float4*>(y) + c + stride, apply(v1, col_of(c + stride)));
    }
    if (c < nchunks) __stcs(reinterpret_cast<float4*>(y) + c, apply(__ldcs(reinterpret_cast<const float4*>(x) + c), col_of(c)));
}

template <typename T>
__global__ void __launch_bounds__(256)
feature_affine_bwd_x_kernel(const T* __restrict__ div, const T* __restrict__ mul, const T* __restrict__ gy,
                            T* __restrict__ gx, int64_t B, int D) {
    const int64_t n = B * D, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int d = (int)(i % D);
        T g = gy[i];
        if (mul) g = g * mul[d];
        if (div) g = g / div[d];
        gx[i] = g;
    }
}

// partial column sums S1[d] = sum_b w[b,d], S2[d] = sum_b w[b,d]*(x[b,d]-sub[d]); w = gy (or 1 for statistics).
// block = 32 columns x 8 row lanes; grid.y row chunks combine with double atomics into acc[2*D].
template <typename T>
__global__ void __launch_bounds__(256)
col_moments_kernel(const T* __restrict__ x, const T* __restrict__ sub, const T* __restrict__ w, double* __restrict__ acc,
                   int64_t B, int D, int64_t rows_per_chunk, int square) {
    __shared__ double s1[8][33], s2[8][33];
    const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
    const int col = blockIdx.x * 32 + cx;
    const int64_t r0 = (int64_t)blockIdx.y * rows_per_chunk;
    const int64_t r1 = (B < r0 + rows_per_chunk) ? B : r0 + rows_per_chunk;
    double a = 0.0, b = 0.0;
    if (col < D) {
        const double sb = sub ? (double)sub[col] : 0.0;
        for (int64_t r = r0 + ry; r < r1; r += 8) {
            const double xv = (double)x[r * D + col] - sb;
            const double wv = w ? (double)w[r * D + col] : 1.0;
            if (square) { a += xv; b += xv * xv; }      // statistics mode: sum x, sum x^2
            else        { a += wv; b += wv * xv; }
        }
    }
    s1[ry][cx] = a; s2[ry][cx] = b;
    __syncthreads();
    if (ry == 0 && col < D) {
        double ta = 0.0, tb = 0.0;
#pragma unroll
        for (int i = 0; i < 8; ++i) { ta += s1[i][cx]; tb += s2[i][cx]; }
        atomicAdd(acc + col, ta);
        atomicAdd(acc + D + col, tb);
    }
}

// Column moments for narrow matrices (D <= 8): the 32-column x 8-row block above keeps D of its 32 column lanes busy
// (D = 2: 6.7 % of HBM).  Here a thread owns whole rows -- 16 / 32-byte row loads, D running sums in registers, four
// rows in flight -- and a block combines through warp shuffles and one double atomic per column.  Same sums as
// col_moments_kernel (double accumulation; the order of the additions differs).
template <int DM>
__global__ void __launch_bounds__(256)
col_moments_rows_kernel(const float* __restrict__ x, const float* __restrict__ sub, const float* __restrict__ w,
                        double* __restrict__ acc, int64_t B, int D, int square) {
    double a[DM], b[DM];
    float sb[DM];
#pragma unroll
    for (int d = 0; d < DM; ++d) { a[d] = 0.0; b[d] = 0.0; sb[d] = (sub && d < D) ? __ldg(sub + d) : 0.f; }
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const bool vec = (D == DM) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0) && (!w || (reinterpret_cast<uintptr_t>(w) & 15) == 0) && DM >= 2;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < B; r += stride) {
        float xv[DM], wv[DM];
        if (vec) {
            if (DM == 2) {
                const float2 t = __ldcs(reinterpret_cast<const float2*>(x) + r); xv[0] = t.x; xv[1] = t.y;
                if (w) { const float2 u = __ldcs(reinterpret_cast<const float2*>(w) + r); wv[0] = u.x; wv[1] = u.y; }
            } else {
#pragma unroll
                for (int q = 0; q < DM / 4; ++q) {
                    const float4 t = __ldcs(reinterpret_cast<const float4*>(x) + r * (DM / 4) + q);
                    xv[4 * q] = t.x; xv[4 * q + 1] = t.y; xv[4 * q + 2] = t.z; xv[4 * q + 3] = t.w;
                    if (w) {
                        const float4 u = __ldcs(reinterpret_cast<const float4*>(w) + r * (DM / 4) + q);
                        wv[4 * q] = u.x; wv[4 * q + 1] = u.y; wv[4 * q + 2] = u.z; wv[4 * q + 3] = u.w;
                    }
                }
            }
        } else {
#pragma unroll
            for (int d = 0; d < DM; ++d) {
                xv[d] = d < D ? x[r * D + d] : 0.f;
                wv[d] = (w && d < D) ? w[r * D + d] : 0.f;
            }
        }
#pragma unroll
        for (int d = 0; d < DM; ++d) {
            const double xd = (double)xv[d] - (double)sb[d];
            const double wd = w ? (double)wv[d] : 1.0;
            if (square) { a[d] += xd; b[d] += xd * xd; }
            else        { a[d] += wd; b[d] += wd * xd; }
        }
    }
    __shared__ double red[8][2 * DM];
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
#pragma unroll
    for (int d = 0; d < DM; ++d) {
        double ta = a[d], tb = b[d];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { ta += __shfl_xor_sync(0xffffffffu, ta, o); tb += __shfl_xor_sync(0xffffffffu, tb, o); }
        if (lane == 0) { red[wp][d] = ta; red[wp][DM + d] = tb; }
    }
    __syncthreads();
    if (threadIdx.x < 2 * DM) {
        const int d = threadIdx.x % DM, which = threadIdx.x / DM;
        if (d < D) {
            double t = 0.0;
#pragma unroll
            for (int i = 0; i < 8; ++i) t += red[i][which * DM + d];
            atomicAdd(acc + which * D + d, t);
        }
    }
}

// returns true when the narrow-matrix kernel took the launch
static bool col_moments_rows_launch(const float* x, const float* sub, const float* w, double* acc, int64_t B, int D, int square,
                                    cudaStream_t st) {
    if (D > 8) return false;
    int64_t need = cdiv(B, 256 * 4);
    const int64_t cap = (int64_t)kNumSMs * 8;
    const int grid = (int)(need < 1 ? 1 : (need < cap ? need : cap));
    if (D <= 2) col_moments_rows_kernel<2><<<grid, 256, 0, st>>>(x, sub, w, acc, B, D, square);
    else if (D <= 4) col_moments_rows_kernel<4><<<grid, 256, 0, st>>>(x, sub, w, acc, B, D, square);
    else col_moments_rows_kernel<8><<<grid, 256, 0, st>>>(x, sub, w, acc, B, D, square);
    return true;
}

template <typename T>
__global__ void feature_affine_bwd_finish_kernel(const double* __restrict__ acc, const T* __restrict__ div,
                                                 const T* __restrict__ mul, T* __restrict__ gsub, T* __restrict__ gdiv,
                                                 T* __restrict__ gmul, T* __restrict__ gadd, int D) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= D) return;
    const double S1 = acc[d], S2 = acc[D + d];
    const double dv = div ? (double)div[d] : 1.0, ml = mul ? (double)mul[d] : 1.0;
    if (gadd) gadd[d] = (T)S1;
    if (gmul) gmul[d] = (T)(S2 / dv);
    if (gsub) gsub[d] = (T)(-S1 * ml / dv);
    if (gdiv) gdiv[d] = (T)(-S2 * ml / (dv * dv));
}

template <typename T>
__global__ void col_stats_finish_kernel(const double* __restrict__ acc, T* __restrict__ mean, T* __restrict__ var,
                                        int64_t B, int D) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= D) return;
    const double m = acc[d] / (double)B;
    double v = acc[D + d] / (double)B - m * m;
    if (v < 0.0) v = 0.0;
    mean[d] = (T)m;
    var[d] = (T)v;
}

static inline void chunking(int64_t B, int& chunks, int64_t& rpc) {
    int64_t c = B / 2048;
    if (c < 1) c = 1;
    if (c > 4 * kNumSMs) c = 4 * kNumSMs;
    rpc = cdiv(B, c);
    chunks = (int)cdiv(B, rpc);
}

// ------------------------------------------------------------------------------------------------
// sequential autoregressive loop body and epilogue
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
ar_step_fwd_kernel(const T* __restrict__ cur, const T* __restrict__ v, const T* __restrict__ params,
                   const T* __restrict__ ld_in, T* __restrict__ out, T* __restrict__ ld_out, int64_t B, int D, int col,
                   int mode) {
    const int64_t n = B * D, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int64_t row = i / D;
        const int d = (int)(i - row * D);
        if (d != col) { out[i] = cur[i]; continue; }
        T o, t;
        affine_ar_elem<T>(mode, v[i], params[row * 2 * D + d], params[row * 2 * D + D + d], o, t);
        out[i] = o;
        ld_out[row] = (ld_in ? ld_in[row] : T(0)) + t;
    }
}

template <typename T>
__global__ void __launch_bounds__(256)
ar_step_bwd_kernel(const T* __restrict__ v, const T* __restrict__ params, const T* __restrict__ gout,
                   const T* __restrict__ gld, T* __restrict__ gcur, T* __restrict__ gv, T* __restrict__ gparams,
                   int64_t B, int D, int col, int mode) {
    const int64_t n = B * D, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int64_t row = i / D;
        const int d = (int)(i - row * D);
        T a = T(0), c = T(0), e = T(0);
        if (d == col) {
            affine_ar_elem_bwd<T>(mode, v[i], params[row * 2 * D + d], params[row * 2 * D + D + d], gout[i], gld[row],
                                  a, c, e);
            gcur[i] = T(0);
        } else {
            gcur[i] = gout[i];
        }
        gv[i] = a;
        gparams[row * 2 * D + d] = c;
        gparams[row * 2 * D + D + d] = e;
    }
}

template <typename T>
__global__ void __launch_bounds__(256)
ar_finish_fwd_kernel(const T* __restrict__ cur, const T* __restrict__ v, const T* __restrict__ ld_sum,
                     T* __restrict__ out, T* __restrict__ ld, int64_t B, int D, int mode) {
    const int64_t n = B * D, stride = (int64_t)gridDim.x * blockDim.x;
    const T lim = (mode == AR_IAF_INV) ? T(50) : T(100);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const T c = cur[i];
        out[i] = is_finite(c) ? c : ((mode == AR_IAF_INV) ? v[i] : T(0));
        if (i < B) ld[i] = clamp_mm(scrub0(ld_sum[i]), -lim, lim);
    }
}

template <typename T>
__global__ void __launch_bounds__(256)
ar_finish_bwd_kernel(const T* __restrict__ cur, const T* __restrict__ ld_sum, const T* __restrict__ gout,
                     const T* __restrict__ gld, T* __restrict__ gcur, T* __restrict__ gv, T* __restrict__ gld_sum,
                     int64_t B, int D, int mode) {
    const int64_t n = B * D, stride = (int64_t)gridDim.x * blockDim.x;
    const T lim = (mode == AR_IAF_INV) ? T(50) : T(100);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const bool fin = is_finite(cur[i]);
        gcur[i] = fin ? gout[i] : T(0);
        gv[i] = (!fin && mode == AR_IAF_INV) ? gout[i] : T(0);
        if (i < B) {
            const T s = ld_sum[i];
            gld_sum[i] = (is_finite(s) && pass_mm(s, -lim, lim)) ? gld[i] : T(0);
        }
    }
}


// ------------------------------------------------------------------------------------------------
// Flow.log_prob head for a standard-normal base (flow.py:56-73): lp = sum_d(-z^2/2) - D/2 log(2 pi) + log_det
// ------------------------------------------------------------------------------------------------
// LOG_Q: the sample_and_log_prob head log N(z; 0, I) - ld instead (ld required)
template <typename T, int G, bool LOG_Q = false>
__global__ void __launch_bounds__(256)
std_normal_log_prob_fwd_kernel(const T* __restrict__ z, const T* __restrict__ ld, T* __restrict__ lp, int64_t B, int D,
                               T norm_const) {
    constexpr int RPW = 32 / G;
    const int lane = threadIdx.x & 31, g = lane % G;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t nblk = (B + RPW - 1) / RPW;
    for (int64_t blk = warp; blk < nblk; blk += nwarps) {
        const int64_t row = blk * RPW + lane / G;
        const bool valid = row < B;
        T acc = T(0);
        if (valid)
            for (int d = g; d < D; d += G) { const T v = ld_stream(z + row * D + d); acc += T(-0.5) * v * v; }
        acc = group_sum<T, G>(acc);
        if (valid && g == 0) lp[row] = LOG_Q ? acc - norm_const - ld[row] : acc - norm_const + (ld ? ld[row] : T(0));
    }
}

// float32, 16-byte aligned z: D % 4 == 0 -> G lanes per row (G = pow2 >= D/4, <= 32), each lane sums float4 chunks, four
// row groups in flight; D == 2 -> one thread per PAIR of rows (one float4).  (The scalar kernel keeps one 4-byte load in
// flight per lane: 28-31 % of HBM at D <= 64.)  Same per-element arithmetic; the order of the D additions differs.
template <int G>
__global__ void __launch_bounds__(256)
std_normal_log_prob_vec4_kernel(const float* __restrict__ z, const float* __restrict__ ld, float* __restrict__ lp, int64_t B,
                                int D, float norm_const) {
    constexpr int RPW = 32 / G;
    const int lane = threadIdx.x & 31, g = lane % G, sub = lane / G;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t nblk = (B + RPW - 1) / RPW;
    const int nch = D >> 2;
    auto row_sum = [&](int64_t row) -> float {
        float acc = 0.f;
        if (row < B) {
            const float4* p = reinterpret_cast<const float4*>(z + row * D);
            for (int c = g; c < nch; c += G) {
                const float4 v = __ldcs(p + c);
                acc += -0.5f * v.x * v.x; acc += -0.5f * v.y * v.y; acc += -0.5f * v.z * v.z; acc += -0.5f * v.w * v.w;
            }
        }
        return acc;
    };
    constexpr int U = 4;                                   // row groups in flight per warp
    for (int64_t blk = warp; blk < nblk; blk += U * nwarps) {
        int64_t rr[U];
        float a[U];
#pragma unroll
        for (int k = 0; k < U; ++k) {
            rr[k] = (blk + k * nwarps) * RPW + sub;
            a[k] = (blk + k * nwarps < nblk) ? row_sum(rr[k]) : 0.f;
        }
#pragma unroll
        for (int k = 0; k < U; ++k) {
            a[k] = group_sum<float, G>(a[k]);
            if (g == 0 && blk + k * nwarps < nblk && rr[k] < B) lp[rr[k]] = a[k] - norm_const + (ld ? ld[rr[k]] : 0.f);
        }
    }
}

__global__ void __launch_bounds__(256)
std_normal_log_prob_d2_kernel(const float* __restrict__ z, const float* __restrict__ ld, float* __restrict__ lp, int64_t B,
                              float norm_const) {
    const int64_t npair = B >> 1, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < npair; p += stride) {
        const float4 v = __ldcs(reinterpret_cast<const float4*>(z) + p);
        float a = 0.f, b = 0.f;
        a += -0.5f * v.x * v.x; a += -0.5f * v.y * v.y;
        b += -0.5f * v.z * v.z; b += -0.5f * v.w * v.w;
        lp[2 * p] = a - norm_const + (ld ? ld[2 * p] : 0.f);
        lp[2 * p + 1] = b - norm_const + (ld ? ld[2 * p + 1] : 0.f);
    }
    if ((B & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
        const int64_t r = B - 1;
        float a = 0.f;
        a += -0.5f * z[2 * r] * z[2 * r]; a += -0.5f * z[2 * r + 1] * z[2 * r + 1];
        lp[r] = a - norm_const + (ld ? ld[r] : 0.f);
    }
}

// backward of log N(z; 0, I) - ld: gz = -z * g (skipped when gz is NULL: a drawn z is a constant), gld = -g
template <typename T>
__global__ void __launch_bounds__(256)
std_normal_log_q_bwd_kernel(const T* __restrict__ z, const T* __restrict__ g, T* __restrict__ gz, T* __restrict__ gld,
                            int64_t B, int D) {
    const int64_t n = gz ? B * D : B, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        if (gz) gz[i] = -z[i] * g[i / D];
        if (gld && i < B) gld[i] = -g[i];
    }
}

// the N(0, I) base draw of nf_rng.cuh: one thread per group of four dims of a row; float64 widens the fp32 normals.
// rng_state != NULL: the key is read from, and advanced in, the device-resident state (nf_rng_state_take)
template <typename T>
__global__ void __launch_bounds__(256)
std_normal_draw_kernel(uint64_t seed, uint64_t offset, unsigned long long* rng_state, T* __restrict__ z, int64_t B, int D) {
    if (rng_state) {
        const unsigned long long* key = nf_rng_key_static();
        nf_rng_state_take(rng_state, nf_rng_key_static());
        __syncthreads();
        seed = key[0];
        offset = key[1];
    }
    const int J = (D + 3) >> 2;
    const int64_t n = B * J, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int64_t r = i / J;
        const int j = (int)(i - r * J);
        float q[4];
        nf_std_normal4(seed, offset, (uint32_t)r, (uint32_t)j, q);
        T* p = z + r * D + 4 * j;
        if (sizeof(T) == 4 && (D & 3) == 0) {
            __stcs(reinterpret_cast<float4*>(p), make_float4(q[0], q[1], q[2], q[3]));
        } else {
            const int m = D - 4 * j < 4 ? D - 4 * j : 4;
#pragma unroll
            for (int k = 0; k < 4; ++k) if (k < m) st_stream(p + k, (T)q[k]);
        }
    }
}

// B == 0 under a device-resident state: the call draws nothing but still moves the offset on by 4
__global__ void __launch_bounds__(1) rng_state_advance_kernel(unsigned long long* rng_state) {
    nf_rng_state_take(rng_state, nf_rng_key_static());
}

int nf_rng_state_advance(unsigned long long* state, cudaStream_t st) {
    rng_state_advance_kernel<<<1, 1, 0, st>>>(state);
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

template <typename T>
__global__ void __launch_bounds__(256)
std_normal_log_prob_bwd_kernel(const T* __restrict__ z, const T* __restrict__ glp, T* __restrict__ gz, int64_t B, int D) {
    const int64_t n = B * D, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) gz[i] = -z[i] * glp[i / D];
}

template <typename T>
static int feature_affine_bwd(const void* x, const void* sub, const void* div, const void* mul, const void* gy, void* gx,
                              void* gsub, void* gdiv, void* gmul, void* gadd, void* ws, int64_t B, int D,
                              cudaStream_t st) {
    feature_affine_bwd_x_kernel<T><<<ew_grid(B * D), 256, 0, st>>>((const T*)div, (const T*)mul, (const T*)gy, (T*)gx, B, D);
    count_launch();
    NF_LAUNCH_CHECK();
    if (!gsub && !gdiv && !gmul && !gadd) return NF_OK;
    NF_CUDA(cudaMemsetAsync(ws, 0, sizeof(double) * 2 * D, st));
    int chunks; int64_t rpc;
    chunking(B, chunks, rpc);
    dim3 grid((unsigned)cdiv(D, 32), (unsigned)chunks);
    if (!(sizeof(T) == 4 && col_moments_rows_launch((const float*)x, (const float*)sub, (const float*)gy, (double*)ws, B, D, 0, st)))
    col_moments_kernel<T><<<grid, 256, 0, st>>>((const T*)x, (const T*)sub, (const T*)gy, (double*)ws, B, D, rpc, 0);
    count_launch();
    NF_LAUNCH_CHECK();
    feature_affine_bwd_finish_kernel<T><<<(D + 127) / 128, 128, 0, st>>>((const double*)ws, (const T*)div, (const T*)mul,
                                                                        (T*)gsub, (T*)gdiv, (T*)gmul, (T*)gadd, D);
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

template <typename T>
static int col_stats(const void* x, void* mean, void* var, void* ws, int64_t B, int D, cudaStream_t st) {
    NF_CUDA(cudaMemsetAsync(ws, 0, sizeof(double) * 2 * D, st));
    int chunks; int64_t rpc;
    chunking(B, chunks, rpc);
    dim3 grid((unsigned)cdiv(D, 32), (unsigned)chunks);
    if (!(sizeof(T) == 4 && col_moments_rows_launch((const float*)x, nullptr, nullptr, (double*)ws, B, D, 1, st)))
    col_moments_kernel<T><<<grid, 256, 0, st>>>((const T*)x, nullptr, nullptr, (double*)ws, B, D, rpc, 1);
    count_launch();
    NF_LAUNCH_CHECK();
    col_stats_finish_kernel<T><<<(D + 127) / 128, 128, 0, st>>>((const double*)ws, (T*)mean, (T*)var, B, D);
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

}  // namespace nf

using namespace nf;
#define NF_REQ(p) do { if ((p) == nullptr) return NF_ERR_NULL; } while (0)
#define NF_DISPATCH(expr_f, expr_d)                         \
    do {                                                    \
        if (dtype == NF_F32) { expr_f; }                    \
        else if (dtype == NF_F64) { expr_d; }               \
        else return NF_ERR_UNSUPPORTED;                     \
    } while (0)

extern "C" int nf_feature_affine_forward(const void* x, const void* sub, const void* div, const void* mul,
                                         const void* add, double add_scalar, void* y, int64_t B, int D, int dtype,
                                         nf_stream_t stream) {
    if (B < 0 || D < 1) return NF_ERR_BAD_SHAPE;
    if (B == 0) return NF_OK;
    NF_REQ(x); NF_REQ(y);
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = ew_grid(B * D);
    const int64_t n = B * D;
    const bool pal = (D % 4 != 0) || ((!sub || aligned16(sub)) && (!div || aligned16(div)) && (!mul || aligned16(mul)) && (!add || aligned16(add)));
    if (dtype == NF_F32 && (n % 4) == 0 && aligned16(x) && aligned16(y) && pal && (D % 4 == 0 || D == 2 || D == 1)) {
        const int64_t nch = n / 4;
        int64_t need = cdiv(nch, 256 * 2);
        const int64_t cap = (int64_t)kNumSMs * 16;
        const int g4 = (int)(need < 1 ? 1 : (need < cap ? need : cap));
#define NF_FA(PER) feature_affine_fwd_vec4_kernel<PER><<<g4, 256, 0, st>>>((const float*)x, (const float*)sub, (const float*)div, \
            (const float*)mul, (const float*)add, (float)add_scalar, (float*)y, nch, D)
        if (D % 4 == 0) NF_FA(4); else if (D == 2) NF_FA(2); else NF_FA(1);
#undef NF_FA
        count_launch();
        NF_LAUNCH_CHECK();
        return NF_OK;
    }
    NF_DISPATCH(
        (feature_affine_fwd_kernel<float><<<grid, 256, 0, st>>>((const float*)x, (const float*)sub, (const float*)div,
            (const float*)mul, (const float*)add, (float)add_scalar, (float*)y, B, D)),
        (feature_affine_fwd_kernel<double><<<grid, 256, 0, st>>>((const double*)x, (const double*)sub, (const double*)div,
            (const double*)mul, (const double*)add, add_scalar, (double*)y, B, D)));
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

extern "C" int nf_feature_affine_backward(const void* x, const void* sub, const void* div, const void* mul,
                                          const void* gy, void* gx, void* gsub, void* gdiv, void* gmul, void* gadd,
                                          void* workspace, int64_t B, int D, int dtype, nf_stream_t stream) {
    if (B < 0 || D < 1) return NF_ERR_BAD_SHAPE;
    const bool need_red = gsub || gdiv || gmul || gadd;
    if (need_red) NF_REQ(workspace);
    if (B == 0) {
        if (need_red) {
            const size_t es = dtype == NF_F64 ? 8 : 4;
            cudaStream_t st0 = (cudaStream_t)stream;
            if (gsub) NF_CUDA(cudaMemsetAsync(gsub, 0, es * D, st0));
            if (gdiv) NF_CUDA(cudaMemsetAsync(gdiv, 0, es * D, st0));
            if (gmul) NF_CUDA(cudaMemsetAsync(gmul, 0, es * D, st0));
            if (gadd) NF_CUDA(cudaMemsetAsync(gadd, 0, es * D, st0));
        }
        return NF_OK;
    }
    NF_REQ(x); NF_REQ(gy); NF_REQ(gx);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == NF_F32) return feature_affine_bwd<float>(x, sub, div, mul, gy, gx, gsub, gdiv, gmul, gadd, workspace, B, D, st);
    if (dtype == NF_F64) return feature_affine_bwd<double>(x, sub, div, mul, gy, gx, gsub, gdiv, gmul, gadd, workspace, B, D, st);
    return NF_ERR_UNSUPPORTED;
}

extern "C" int nf_col_stats(const void* x, void* mean, void* var, void* workspace, int64_t B, int D, int dtype,
                            nf_stream_t stream) {
    if (B < 1 || D < 1) return NF_ERR_BAD_SHAPE;
    NF_REQ(x); NF_REQ(mean); NF_REQ(var); NF_REQ(workspace);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == NF_F32) return col_stats<float>(x, mean, var, workspace, B, D, st);
    if (dtype == NF_F64) return col_stats<double>(x, mean, var, workspace, B, D, st);
    return NF_ERR_UNSUPPORTED;
}

extern "C" int nf_ar_step_forward(const void* cur, const void* v, const void* params, const void* ld_in, void* out,
                                  void* ld_out, int64_t B, int D, int col, int mode, int dtype, nf_stream_t stream) {
    if (B < 0 || D < 1 || col < 0 || col >= D) return NF_ERR_BAD_SHAPE;
    if (mode != NF_AR_MAF_FORWARD && mode != NF_AR_IAF_INVERSE) return NF_ERR_UNSUPPORTED;
    if (B == 0) return NF_OK;
    NF_REQ(cur); NF_REQ(v); NF_REQ(params); NF_REQ(out); NF_REQ(ld_out);
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = ew_grid(B * D);
    NF_DISPATCH(
        (ar_step_fwd_kernel<float><<<grid, 256, 0, st>>>((const float*)cur, (const float*)v, (const float*)params,
            (const float*)ld_in, (float*)out, (float*)ld_out, B, D, col, mode)),
        (ar_step_fwd_kernel<double><<<grid, 256, 0, st>>>((const double*)cur, (const double*)v, (const double*)params,
            (const double*)ld_in, (double*)out, (double*)ld_out, B, D, col, mode)));
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

extern "C" int nf_ar_step_backward(const void* v, const void* params, const void* gout, const void* gld, void* gcur,
                                   void* gv, void* gparams, int64_t B, int D, int col, int mode, int dtype,
                                   nf_stream_t stream) {
    if (B < 0 || D < 1 || col < 0 || col >= D) return NF_ERR_BAD_SHAPE;
    if (mode != NF_AR_MAF_FORWARD && mode != NF_AR_IAF_INVERSE) return NF_ERR_UNSUPPORTED;
    if (B == 0) return NF_OK;
    NF_REQ(v); NF_REQ(params); NF_REQ(gout); NF_REQ(gld); NF_REQ(gcur); NF_REQ(gv); NF_REQ(gparams);
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = ew_grid(B * D);
    NF_DISPATCH(
        (ar_step_bwd_kernel<float><<<grid, 256, 0, st>>>((const float*)v, (const float*)params, (const float*)gout,
            (const float*)gld, (float*)gcur, (float*)gv, (float*)gparams, B, D, col, mode)),
        (ar_step_bwd_kernel<double><<<grid, 256, 0, st>>>((const double*)v, (const double*)params, (const double*)gout,
            (const double*)gld, (double*)gcur, (double*)gv, (double*)gparams, B, D, col, mode)));
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

extern "C" int nf_ar_finish_forward(const void* cur, const void* v, const void* ld_sum, void* out, void* ld, int64_t B,
                                    int D, int mode, int dtype, nf_stream_t stream) {
    if (B < 0 || D < 1) return NF_ERR_BAD_SHAPE;
    if (mode != NF_AR_MAF_FORWARD && mode != NF_AR_IAF_INVERSE) return NF_ERR_UNSUPPORTED;
    if (B == 0) return NF_OK;
    NF_REQ(cur); NF_REQ(v); NF_REQ(ld_sum); NF_REQ(out); NF_REQ(ld);
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = ew_grid(B * D);
    NF_DISPATCH(
        (ar_finish_fwd_kernel<float><<<grid, 256, 0, st>>>((const float*)cur, (const float*)v, (const float*)ld_sum,
            (float*)out, (float*)ld, B, D, mode)),
        (ar_finish_fwd_kernel<double><<<grid, 256, 0, st>>>((const double*)cur, (const double*)v, (const double*)ld_sum,
            (double*)out, (double*)ld, B, D, mode)));
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

extern "C" int nf_ar_finish_backward(const void* cur, const void* ld_sum, const void* gout, const void* gld, void* gcur,
                                     void* gv, void* gld_sum, int64_t B, int D, int mode, int dtype,
                                     nf_stream_t stream) {
    if (B < 0 || D < 1) return NF_ERR_BAD_SHAPE;
    if (mode != NF_AR_MAF_FORWARD && mode != NF_AR_IAF_INVERSE) return NF_ERR_UNSUPPORTED;
    if (B == 0) return NF_OK;
    NF_REQ(cur); NF_REQ(ld_sum); NF_REQ(gout); NF_REQ(gld); NF_REQ(gcur); NF_REQ(gv); NF_REQ(gld_sum);
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = ew_grid(B * D);
    NF_DISPATCH(
        (ar_finish_bwd_kernel<float><<<grid, 256, 0, st>>>((const float*)cur, (const float*)ld_sum, (const float*)gout,
            (const float*)gld, (float*)gcur, (float*)gv, (float*)gld_sum, B, D, mode)),
        (ar_finish_bwd_kernel<double><<<grid, 256, 0, st>>>((const double*)cur, (const double*)ld_sum, (const double*)gout,
            (const double*)gld, (double*)gcur, (double*)gv, (double*)gld_sum, B, D, mode)));
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

extern "C" int nf_std_normal_log_prob_forward(const void* z, const void* ld, void* lp, int64_t B, int D, int dtype,
                                              nf_stream_t stream) {
    if (B < 0 || D < 1) return NF_ERR_BAD_SHAPE;
    if (B == 0) return NF_OK;
    NF_REQ(z); NF_REQ(lp);
    cudaStream_t st = (cudaStream_t)stream;
    const double nc = 0.5 * (double)D * 1.8378770664093453;   // D/2 * log(2 pi)
    if (dtype == NF_F32 && aligned16(z) && (D == 2 || (D % 4 == 0))) {
        const int64_t cap4 = (int64_t)kNumSMs * 16;
        if (D == 2) {
            int64_t need4 = cdiv(B / 2 + 1, 256);
            const int g4 = (int)(need4 < 1 ? 1 : (need4 < cap4 ? need4 : cap4));
            std_normal_log_prob_d2_kernel<<<g4, 256, 0, st>>>((const float*)z, (const float*)ld, (float*)lp, B, (float)nc);
        } else {
            int G4 = 1; while (G4 < D / 4 && G4 < 32) G4 <<= 1;
            int64_t need4 = cdiv(cdiv(B, 32 / G4), 8 * 4);
            const int g4 = (int)(need4 < 1 ? 1 : (need4 < cap4 ? need4 : cap4));
#define NF_LP4(GG) std_normal_log_prob_vec4_kernel<GG><<<g4, 256, 0, st>>>((const float*)z, (const float*)ld, (float*)lp, B, D, (float)nc)
            switch (G4) { case 1: NF_LP4(1); break; case 2: NF_LP4(2); break; case 4: NF_LP4(4); break; case 8: NF_LP4(8); break;
                          case 16: NF_LP4(16); break; default: NF_LP4(32); break; }
#undef NF_LP4
        }
        count_launch();
        NF_LAUNCH_CHECK();
        return NF_OK;
    }
    int G = 1; while (G < D && G < 32) G <<= 1;
    int64_t need = cdiv(cdiv(B, 32 / G), 8), cap = (int64_t)kNumSMs * 32;
    const int grid = (int)(need < 1 ? 1 : (need < cap ? need : cap));
#define NF_LP(T, GG) std_normal_log_prob_fwd_kernel<T, GG><<<grid, 256, 0, st>>>((const T*)z, (const T*)ld, (T*)lp, B, D, (T)nc)
#define NF_LP_G(T) switch (G) { case 1: NF_LP(T, 1); break; case 2: NF_LP(T, 2); break; case 4: NF_LP(T, 4); break; \
                                case 8: NF_LP(T, 8); break; case 16: NF_LP(T, 16); break; default: NF_LP(T, 32); break; }
    NF_DISPATCH(NF_LP_G(float), NF_LP_G(double));
#undef NF_LP_G
#undef NF_LP
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

extern "C" int nf_std_normal_log_prob_backward(const void* z, const void* glp, void* gz, int64_t B, int D, int dtype,
                                               nf_stream_t stream) {
    if (B < 0 || D < 1) return NF_ERR_BAD_SHAPE;
    if (B == 0) return NF_OK;
    NF_REQ(z); NF_REQ(glp); NF_REQ(gz);
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = ew_grid(B * D);
    NF_DISPATCH(
        (std_normal_log_prob_bwd_kernel<float><<<grid, 256, 0, st>>>((const float*)z, (const float*)glp, (float*)gz, B, D)),
        (std_normal_log_prob_bwd_kernel<double><<<grid, 256, 0, st>>>((const double*)z, (const double*)glp, (double*)gz, B, D)));
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

// rng_state == NULL: the key (seed, offset) given by the caller; otherwise the device-resident state
static int std_normal_draw_launch(uint64_t seed, uint64_t offset, unsigned long long* rng_state, void* z, int64_t B,
                                  int D, int dtype, nf_stream_t stream) {
    if (B < 0 || B > (int64_t)0xFFFFFFFFLL || D < 1) return NF_ERR_BAD_SHAPE;
    if (rng_state && dtype != NF_F32 && dtype != NF_F64) return NF_ERR_UNSUPPORTED;    // refused: the state stays put
    cudaStream_t st = (cudaStream_t)stream;
    if (B == 0) return rng_state ? nf_rng_state_advance(rng_state, st) : NF_OK;
    NF_REQ(z);
    if (dtype == NF_F32 && (D & 3) == 0 && !aligned16(z)) return NF_ERR_MISALIGNED;
    const int grid = ew_grid(B * ((D + 3) / 4));
    NF_DISPATCH(
        (std_normal_draw_kernel<float><<<grid, 256, 0, st>>>(seed, offset, rng_state, (float*)z, B, D)),
        (std_normal_draw_kernel<double><<<grid, 256, 0, st>>>(seed, offset, rng_state, (double*)z, B, D)));
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

extern "C" int nf_std_normal_draw(uint64_t seed, uint64_t offset, void* z, int64_t B, int D, int dtype, nf_stream_t stream) {
    return std_normal_draw_launch(seed, offset, nullptr, z, B, D, dtype, stream);
}

extern "C" int nf_std_normal_draw_state(void* rng_state, void* z, int64_t B, int D, int dtype, nf_stream_t stream) {
    const int rc = nf_rng_state_check(rng_state);
    if (rc != NF_OK) return rc;
    return std_normal_draw_launch(0, 0, (unsigned long long*)rng_state, z, B, D, dtype, stream);
}

extern "C" int nf_std_normal_log_q_forward(const void* z, const void* ld, void* lq, int64_t B, int D, int dtype,
                                           nf_stream_t stream) {
    if (B < 0 || D < 1) return NF_ERR_BAD_SHAPE;
    if (B == 0) return NF_OK;
    NF_REQ(z); NF_REQ(ld); NF_REQ(lq);
    cudaStream_t st = (cudaStream_t)stream;
    const double nc = 0.5 * (double)D * 1.8378770664093453;   // D/2 * log(2 pi)
    int G = 1; while (G < D && G < 32) G <<= 1;
    int64_t need = cdiv(cdiv(B, 32 / G), 8), cap = (int64_t)kNumSMs * 32;
    const int grid = (int)(need < 1 ? 1 : (need < cap ? need : cap));
#define NF_LQ(T, GG) std_normal_log_prob_fwd_kernel<T, GG, true><<<grid, 256, 0, st>>>((const T*)z, (const T*)ld, (T*)lq, B, D, (T)nc)
#define NF_LQ_G(T) switch (G) { case 1: NF_LQ(T, 1); break; case 2: NF_LQ(T, 2); break; case 4: NF_LQ(T, 4); break; \
                                case 8: NF_LQ(T, 8); break; case 16: NF_LQ(T, 16); break; default: NF_LQ(T, 32); break; }
    NF_DISPATCH(NF_LQ_G(float), NF_LQ_G(double));
#undef NF_LQ_G
#undef NF_LQ
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}

extern "C" int nf_std_normal_log_q_backward(const void* z, const void* glq, void* gz, void* gld, int64_t B, int D, int dtype,
                                            nf_stream_t stream) {
    if (B < 0 || D < 1) return NF_ERR_BAD_SHAPE;
    if (B == 0 || (!gz && !gld)) return NF_OK;
    NF_REQ(glq);
    if (gz) NF_REQ(z);
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = ew_grid(gz ? B * D : B);
    NF_DISPATCH(
        (std_normal_log_q_bwd_kernel<float><<<grid, 256, 0, st>>>((const float*)z, (const float*)glq, (float*)gz, (float*)gld, B, D)),
        (std_normal_log_q_bwd_kernel<double><<<grid, 256, 0, st>>>((const double*)z, (const double*)glq, (double*)gz, (double*)gld, B, D)));
    count_launch();
    NF_LAUNCH_CHECK();
    return NF_OK;
}
