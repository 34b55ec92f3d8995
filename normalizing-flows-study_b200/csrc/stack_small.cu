// stack_small.cu -- whole-model fused inference kernels for small data_dim (<=8) and hidden_dim<=128:
//   nf_spline_stack_forward    L x SplineCouplingLayer (+ between-layer BatchNorm affine)
//                              spline_coupling_layer.py:96-309 + normalizing_flow_model.py:25-128
//   nf_coupling_stack_forward  L x CouplingLayer in eval mode (conditioner BatchNorm folded at pack time)
//                              coupling_layer.py:40-96 + normalizing_flow_model.py:25-128
//
// One launch evaluates the whole stack: a row is 8..32 bytes, so HBM traffic is 4D in + 4D+4 out and the
// kernel is bound by the FP32 pipe (conditioner MLPs, ~11-17 kFLOP per row and layer).  Mapping:
//   * one thread owns R rows; CTA = 128 threads = 128*R rows per tile; tiles are walked grid-stride;
//   * per layer the packed weights (stack_small.cuh) are staged into shared memory with cp.async;
//   * layer 1 is recomputed on the fly inside the k-loop of layer 2 (K=D is tiny), layer-2 accumulators
//     live in registers (R x HP), weights are read as warp-uniform LDS.128 broadcasts (4R FFMA per LDS);
//   * the head (layer 3) runs in chunks of 4 outputs; spline parameters go through a per-thread column of
//     shared memory, then the rational-quadratic spline / affine transform and the row log-det finish in
//     registers.  No activation ever touches HBM.
#include "nf_common.cuh"
#include "stack_small.cuh"
#include "nf_rng.cuh"

namespace nf {

constexpr int kStackThreads = 128;

// cooperative global->shared copy of n words (n % 4 == 0, both 16B aligned)
__device__ __forceinline__ void stage_words(float* dst, const float* __restrict__ src, int n) {
    for (int i = threadIdx.x * 4; i < n; i += kStackThreads * 4) cp_async16(dst + i, src + i);
}

// hidden layers 1+2 of one conditioner for R rows: acc[i][j] = relu(b2[j] + sum_k W2[j][k] relu(b1[k] + W1[k].xa_i))
template <int HP, int R, int DM>
__device__ __forceinline__ void mlp_hidden(const float* __restrict__ sW1k, const float* __restrict__ sW2t,
                                           const float* __restrict__ sb2, int W1S, const float (&xa)[R][DM],
                                           float (&acc)[R][HP]) {
    // layer-2 accumulators as register PAIRS: the inner product runs on the packed fp32 pipe (FFMA2: two outputs per
    // instruction, the weights of a pair adjacent in the LDS.128, h broadcast into a pair) -- 64 FFMA2 + 32 LDS.128 per k
    // at HP = 128 instead of 128 FFMA + 32 LDS.128; same operations, bit-identical results
    float2 a2[R][HP / 2];
#pragma unroll
    for (int j4 = 0; j4 < HP / 4; ++j4) {
        const float4 b = *reinterpret_cast<const float4*>(sb2 + 4 * j4);
#pragma unroll
        for (int i = 0; i < R; ++i) { a2[i][2 * j4] = make_float2(b.x, b.y); a2[i][2 * j4 + 1] = make_float2(b.z, b.w); }
    }
#pragma unroll 2
    for (int k = 0; k < HP; ++k) {
        const float* w1 = sW1k + k * W1S;
        float2 h[R];
        if constexpr (DM <= 4) {       // D<=3 (W1S=4): one LDS.128 {w0,w1,w2,b1}
            const float4 v = *reinterpret_cast<const float4*>(w1);
#pragma unroll
            for (int i = 0; i < R; ++i) {
                float t = v.w;
                t = fmaf(v.x, xa[i][0], t);
                if (DM > 1) t = fmaf(v.y, xa[i][1], t);
                if (DM > 2) t = fmaf(v.z, xa[i][2], t);
                t = relu_nan(t);
                h[i] = make_float2(t, t);
            }
        } else {                        // 4<=D<=8 (W1S=12): {w0..w7, 0, 0, 0, b1}
            const float4 v0 = *reinterpret_cast<const float4*>(w1);
            const float4 v1 = *reinterpret_cast<const float4*>(w1 + 4);
            const float bb = w1[W1S - 1];
#pragma unroll
            for (int i = 0; i < R; ++i) {
                float t = bb;
                t = fmaf(v0.x, xa[i][0], t); t = fmaf(v0.y, xa[i][1], t); t = fmaf(v0.z, xa[i][2], t); t = fmaf(v0.w, xa[i][3], t);
                t = fmaf(v1.x, xa[i][4], t); t = fmaf(v1.y, xa[i][5], t); t = fmaf(v1.z, xa[i][6], t); t = fmaf(v1.w, xa[i][7], t);
                t = relu_nan(t);
                h[i] = make_float2(t, t);
            }
        }
        const float4* w2 = reinterpret_cast<const float4*>(sW2t + k * HP);
#pragma unroll
        for (int j4 = 0; j4 < HP / 4; ++j4) {
            const float4 w = w2[j4];
#pragma unroll
            for (int i = 0; i < R; ++i) {
                a2[i][2 * j4]     = __ffma2_rn(make_float2(w.x, w.y), h[i], a2[i][2 * j4]);
                a2[i][2 * j4 + 1] = __ffma2_rn(make_float2(w.z, w.w), h[i], a2[i][2 * j4 + 1]);
            }
        }
    }
#pragma unroll
    for (int i = 0; i < R; ++i)
#pragma unroll
        for (int j = 0; j < HP / 2; ++j) { acc[i][2 * j] = relu_nan(a2[i][j].x); acc[i][2 * j + 1] = relu_nan(a2[i][j].y); }
}

// one chunk of 4 head outputs: o[i][q] = b3[4c+q] + sum_j W3[4c+q][j] * h2[i][j]
template <int HP, int R>
__device__ __forceinline__ void head_chunk(const float* __restrict__ sW3c, const float* __restrict__ sb3, int c,
                                           const float (&h2)[R][HP], float (&o)[R][4]) {
    const float4 b = *reinterpret_cast<const float4*>(sb3 + 4 * c);
    float2 o01[R], o23[R];
#pragma unroll
    for (int i = 0; i < R; ++i) { o01[i] = make_float2(b.x, b.y); o23[i] = make_float2(b.z, b.w); }
    const float4* w3 = reinterpret_cast<const float4*>(sW3c) + (size_t)c * HP;
#pragma unroll
    for (int j = 0; j < HP; ++j) {
        const float4 w = w3[j];
#pragma unroll
        for (int i = 0; i < R; ++i) {                     // packed fp32: two head outputs per FFMA2
            const float2 hh = make_float2(h2[i][j], h2[i][j]);
            o01[i] = __ffma2_rn(make_float2(w.x, w.y), hh, o01[i]);
            o23[i] = __ffma2_rn(make_float2(w.z, w.w), hh, o23[i]);
        }
    }
#pragma unroll
    for (int i = 0; i < R; ++i) { o[i][0] = o01[i].x; o[i][1] = o01[i].y; o[i][2] = o23[i].x; o[i][3] = o23[i].y; }
}

// R rows of one thread through the between-layer BatchNorm
template <int R, int DM>
__device__ __forceinline__ void bn_between(LayerHdr lh, int D, bool inverse, float (&xv)[R][DM], float (&tot)[R]) {
#pragma unroll
    for (int i = 0; i < R; ++i) nf_stack_bn_between<DM>(lh, D, inverse, xv[i], tot[i]);
}

// ------------------------------------------------------------------------------------------------
// spline stack
// ------------------------------------------------------------------------------------------------
// SAMPLE (both kernels, nf_*_stack_sample): the row is the N(0, I) draw of nf_rng.cuh instead of a load, tot starts at
// -log N(z) and the epilogue stores -tot = log N(z) - log_det (sample_and_log_prob).  rng_state != NULL
// (nf_*_stack_sample_state): the key comes from the device-resident state, which the launch advances; otherwise from
// the seed / offset arguments.  Non-SAMPLE instantiations ignore all three.
template <int HP, int R, int DM, int KMAX, bool SAMPLE = false>
__global__ void __launch_bounds__(kStackThreads)
spline_stack_kernel(const float* __restrict__ packed, const float* __restrict__ x, float* __restrict__ y,
                    float* __restrict__ ld, int64_t B, int flags, int layer_words_pad, uint64_t seed, uint64_t offset,
                    unsigned long long* rng_state) {
    const int inverse = flags & NF_STACK_INVERSE;
    extern __shared__ __align__(16) float smem[];
    const StackHdr hd = nf_stack_hdr_device(packed);
    const int D = hd.D, K = hd.K, L = hd.L, W1S = hd.W1S, NO = hd.NO, P = 3 * hd.K - 1;
    constexpr int ROWS = kStackThreads * R;
    float* sL = smem;                          // staged layer block
    float* sP = smem + layer_words_pad;        // head outputs: [NO][ROWS], one column per (thread,row)
    const float* sW1k = sL + NF_LAYER_HDR;
    const float* sW2t = sW1k + HP * W1S;
    const float* sb2 = sW2t + HP * HP;
    const float* sW3c = sb2 + HP;
    const float* sb3 = sW3c + (size_t)NO * HP;

    RqsCfg<float> cfg;
    cfg.lo = -hd.bound; cfg.hi = hd.bound; cfg.span = 2.0f * hd.bound; cfg.eps = 1e-8f;
    cfg.min_w = hd.min_w; cfg.min_h = hd.min_h; cfg.min_d = hd.min_d; cfg.scale_w = hd.scale_w; cfg.scale_h = hd.scale_h;

    const int tid = threadIdx.x;
    if constexpr (SAMPLE) {
        if (rng_state) {                        // every CTA, before the tile loop (a CTA may find no tile)
            nf_rng_state_take(rng_state, nf_rng_key_static());
            __syncthreads();
        }
    }
    const int64_t ntiles = (B + ROWS - 1) / ROWS;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        float xv[R][DM], tot[R];
        int64_t row[R];
#pragma unroll
        for (int i = 0; i < R; ++i) {
            row[i] = tile * ROWS + i * kStackThreads + tid;
            if constexpr (SAMPLE) {
                const unsigned long long* key = nf_rng_key_static();
                tot[i] = -nf_std_normal_row<DM>(rng_state ? key[0] : seed, rng_state ? key[1] : offset, (uint32_t)row[i],
                                                D, xv[i]);
                continue;
            }
            tot[i] = 0.f;
#pragma unroll
            for (int d = 0; d < DM; ++d) xv[i][d] = (d < D && row[i] < B) ? ld_stream(x + row[i] * D + d) : 0.f;
        }
        for (int li = 0; li < L; ++li) {
            const int layer = inverse ? L - 1 - li : li;
            __syncthreads();                                   // everyone is done with the previous block
            stage_words(sL, packed + NF_STACK_HDR + (size_t)layer * hd.layer_stride, hd.layer_stride);
            cp_async_commit();
            cp_async_wait<0>();
            __syncthreads();
            const LayerHdr lh{sL};
            const bool rescale = lh.rescale(), bn_on = lh.bn_on();
            const float* mask = lh.mask();
            if (inverse && bn_on) bn_between<R, DM>(lh, D, true, xv, tot);

            float xs[R][DM];                                  // value in spline coordinates
            {
                float xa[R][DM];
#pragma unroll
                for (int i = 0; i < R; ++i)
#pragma unroll
                    for (int d = 0; d < DM; ++d) {
                        float v = xv[i][d];
                        if (rescale && d < D) v = lh.to_spline(v, d, hd.bound);
                        xs[i][d] = v;
                        xa[i][d] = (d < D) ? v * mask[d] : 0.f;
                    }
                float h2[R][HP];
                mlp_hidden<HP, R, DM>(sW1k, sW2t, sb2, W1S, xa, h2);
                for (int c = 0; c < NO / 4; ++c) {
                    float o[R][4];
                    head_chunk<HP, R>(sW3c, sb3, c, h2, o);
#pragma unroll
                    for (int i = 0; i < R; ++i)
#pragma unroll
                        for (int q = 0; q < 4; ++q) sP[(size_t)(4 * c + q) * ROWS + i * kStackThreads + tid] = o[i][q];
                }
            }
            // transform (each thread reads back only its own columns: no barrier needed)
            float lsum[R];
#pragma unroll
            for (int i = 0; i < R; ++i) lsum[i] = 0.f;
            int t = 0;
#pragma unroll
            for (int d = 0; d < DM; ++d) {
                if (d < D && mask[d] == 0.f) {
#pragma unroll
                    for (int i = 0; i < R; ++i) {
                        const float* col = sP + (size_t)(t * P) * ROWS + i * kStackThreads + tid;
                        float uw[KMAX], uh[KMAX], ud[KMAX];
#pragma unroll
                        for (int j = 0; j < KMAX; ++j) {
                            uw[j] = (j < K) ? col[(size_t)j * ROWS] : 0.f;
                            uh[j] = (j < K) ? col[(size_t)(K + j) * ROWS] : 0.f;
                            ud[j] = (j < K - 1) ? col[(size_t)(2 * K + j) * ROWS] : 0.f;
                        }
                        float out, lad;
                        rqs_eval<float, KMAX, true>(xs[i][d], uw, uh, ud, K, inverse != 0, cfg, out, lad);
                        if (rescale) out = lh.from_spline(out, d, hd.bound);
                        xv[i][d] = out;
                        lsum[i] += lad;
                    }
                    ++t;
                }
            }
#pragma unroll
            for (int i = 0; i < R; ++i) {
#pragma unroll
                for (int d = 0; d < DM; ++d) xv[i][d] = scrub0(xv[i][d]);      // layer-level scrub (:130-135)
                tot[i] += scrub0(lsum[i]);
            }
            if (!inverse && bn_on) bn_between<R, DM>(lh, D, false, xv, tot);
        }
#pragma unroll
        for (int i = 0; i < R; ++i)
            if (row[i] < B) nf_stack_row_store<DM, SAMPLE>(y, ld, row[i], D, flags, xv[i], tot[i]);
    }
}

// ------------------------------------------------------------------------------------------------
// affine coupling stack (eval mode)
// ------------------------------------------------------------------------------------------------
template <int HP, int R, int DM, bool SAMPLE = false>
__global__ void __launch_bounds__(kStackThreads)
coupling_stack_kernel(const float* __restrict__ packed, const float* __restrict__ x, float* __restrict__ y,
                      float* __restrict__ ld, int64_t B, int flags, uint64_t seed, uint64_t offset,
                      unsigned long long* rng_state) {
    const int inverse = flags & NF_STACK_INVERSE;
    extern __shared__ __align__(16) float smem[];
    const StackHdr hd = nf_stack_hdr_device(packed);
    const int D = hd.D, L = hd.L, W1S = hd.W1S;
    constexpr int NO = DM;                      // head outputs padded to DM (4 or 8)
    constexpr int ROWS = kStackThreads * R;
    float* sL = smem;
    const int net_words = HP * W1S + HP * HP + HP + NO * HP + NO;

    const int tid = threadIdx.x;
    if constexpr (SAMPLE) {
        if (rng_state) {                        // every CTA, before the tile loop (a CTA may find no tile)
            nf_rng_state_take(rng_state, nf_rng_key_static());
            __syncthreads();
        }
    }
    const int64_t ntiles = (B + ROWS - 1) / ROWS;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        float xv[R][DM], tot[R];
        int64_t row[R];
#pragma unroll
        for (int i = 0; i < R; ++i) {
            row[i] = tile * ROWS + i * kStackThreads + tid;
            if constexpr (SAMPLE) {
                const unsigned long long* key = nf_rng_key_static();
                tot[i] = -nf_std_normal_row<DM>(rng_state ? key[0] : seed, rng_state ? key[1] : offset, (uint32_t)row[i],
                                                D, xv[i]);
                continue;
            }
            tot[i] = 0.f;
#pragma unroll
            for (int d = 0; d < DM; ++d) xv[i][d] = (d < D && row[i] < B) ? ld_stream(x + row[i] * D + d) : 0.f;
        }
        for (int li = 0; li < L; ++li) {
            const int layer = inverse ? L - 1 - li : li;
            __syncthreads();
            stage_words(sL, packed + NF_STACK_HDR + (size_t)layer * hd.layer_stride, hd.layer_stride);
            cp_async_commit();
            cp_async_wait<0>();
            __syncthreads();
            const LayerHdr lh{sL};
            const bool bn_on = lh.bn_on();
            const float* mask = lh.mask();
            if (inverse && bn_on) bn_between<R, DM>(lh, D, true, xv, tot);

            float xa[R][DM];
#pragma unroll
            for (int i = 0; i < R; ++i)
#pragma unroll
                for (int d = 0; d < DM; ++d) xa[i][d] = (d < D) ? xv[i][d] * mask[d] : 0.f;
            float sb[2][R][DM];                  // raw s_net / b_net outputs
#pragma unroll
            for (int net = 0; net < 2; ++net) {
                const float* sW1k = sL + NF_LAYER_HDR + net * net_words;
                const float* sW2t = sW1k + HP * W1S;
                const float* sb2 = sW2t + HP * HP;
                const float* sW3c = sb2 + HP;
                const float* sb3 = sW3c + NO * HP;
                float h2[R][HP];
                mlp_hidden<HP, R, DM>(sW1k, sW2t, sb2, W1S, xa, h2);
#pragma unroll
                for (int c = 0; c < NO / 4; ++c) {
                    float o[R][4];
                    head_chunk<HP, R>(sW3c, sb3, c, h2, o);
#pragma unroll
                    for (int i = 0; i < R; ++i)
#pragma unroll
                        for (int q = 0; q < 4; ++q) sb[net][i][4 * c + q] = o[i][q];
                }
            }
#pragma unroll
            for (int i = 0; i < R; ++i) {
                float lsum = 0.f;
#pragma unroll
                for (int d = 0; d < DM; ++d) if (d < D) {
                    float out, t;
                    affine_coupling_elem<float>(xv[i][d], mask[d], sb[0][i][d], sb[1][i][d], inverse != 0, out, t);
                    xv[i][d] = scrub0(out);
                    lsum += t;
                }
                tot[i] += scrub0(lsum);
            }
            if (!inverse && bn_on) bn_between<R, DM>(lh, D, false, xv, tot);
        }
#pragma unroll
        for (int i = 0; i < R; ++i)
            if (row[i] < B) nf_stack_row_store<DM, SAMPLE>(y, ld, row[i], D, flags, xv[i], tot[i]);
    }
}

// ------------------------------------------------------------------------------------------------
// host
// ------------------------------------------------------------------------------------------------
#define NF_REQ(p) do { if ((p) == nullptr) return NF_ERR_NULL; } while (0)

// The checks every family shares, in this order, then the family's launcher.  The header lives in device memory; the
// caller passes a host copy of its 16 words beside it (cheap, and keeps the library free of hidden device->host syncs).
static int run_stack(const StackFamily& f, const StackCall& c) {
    if (c.B < 0 || (c.sample && c.B > (int64_t)0xFFFFFFFFLL)) return NF_ERR_BAD_SHAPE;
    NF_REQ(c.hdr_host);
    if (c.B == 0) return c.rng_state ? nf_rng_state_advance(c.rng_state, c.st) : NF_OK;
    NF_REQ(c.packed); NF_REQ(c.ld);
    if (!c.sample) NF_REQ(c.x);
    if (!(c.flags & NF_STACK_SKIP_Y)) NF_REQ(c.y);
    if (!aligned16(c.packed)) return NF_ERR_MISALIGNED;
    const StackHdr h = nf_stack_hdr(c.hdr_host);
    if (h.magic != f.magic) return NF_ERR_BAD_SHAPE;
    return f.launch(c, h);
}

int stack_forward(const StackFamily& f, const void* packed, const void* hdr_host, int64_t packed_bytes, const void* x,
                  void* y, void* ld, int64_t B, int flags, int mode, nf_stream_t stream, StackCtx cx) {
    return run_stack(f, {packed, hdr_host, packed_bytes, x, y, ld, B, flags, mode, false, 0, 0, nullptr,
                         (cudaStream_t)stream, cx});
}

int stack_sample(const StackFamily& f, const void* packed, const void* hdr_host, int64_t packed_bytes, int mode,
                 uint64_t seed, uint64_t offset, void* x, void* log_q, int64_t B, nf_stream_t stream, StackCtx cx) {
    return run_stack(f, {packed, hdr_host, packed_bytes, nullptr, x, log_q, B, x ? 0 : NF_STACK_SKIP_Y, mode, true, seed,
                         offset, nullptr, (cudaStream_t)stream, cx});
}

int stack_sample_state(const StackFamily& f, const void* packed, const void* hdr_host, int64_t packed_bytes, int mode,
                       void* rng_state, void* x, void* log_q, int64_t B, nf_stream_t stream, StackCtx cx) {
    const int rc = nf_rng_state_check(rng_state);
    if (rc != NF_OK) return rc;
    return run_stack(f, {packed, hdr_host, packed_bytes, nullptr, x, log_q, B, x ? 0 : NF_STACK_SKIP_Y, mode, true, 0, 0,
                         (unsigned long long*)rng_state, (cudaStream_t)stream, cx});
}

template <typename Kern>
static int launch_stack(Kern kern, size_t smem_bytes, int rows_per_cta, const StackCall& c, int extra, bool has_extra) {
    // the SAMPLE twins hold the 16-byte key of nf_rng_state_take in static shared memory
    if (smem_bytes + (c.sample ? 16 : 0) > 227 * 1024) return NF_ERR_UNSUPPORTED;
    const int rc = stack_smem_attributes(kern, smem_bytes);
    if (rc != NF_OK) return rc;
    int per_sm = 0;
    NF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kStackThreads, smem_bytes));
    if (per_sm < 1) return NF_ERR_UNSUPPORTED;
    const int64_t ntiles = cdiv(c.B, rows_per_cta);
    const int64_t cap = (int64_t)kNumSMs * per_sm;
    const int grid = (int)(ntiles < cap ? ntiles : cap);
    void* args_s[] = {(void*)&c.packed, (void*)&c.x, (void*)&c.y, (void*)&c.ld, (void*)&c.B, (void*)&c.flags, (void*)&extra,
                      (void*)&c.seed, (void*)&c.offset, (void*)&c.rng_state};
    void* args_n[] = {(void*)&c.packed, (void*)&c.x, (void*)&c.y, (void*)&c.ld, (void*)&c.B, (void*)&c.flags,
                      (void*)&c.seed, (void*)&c.offset, (void*)&c.rng_state};
    NF_CUDA(cudaLaunchKernel((const void*)kern, dim3(grid), dim3(kStackThreads), has_extra ? args_s : args_n, smem_bytes,
                             c.st));
    count_launch();
    return NF_OK;
}

// the FP32-pipe layouts' header checks after the magic
static int check_hdr(const StackHdr& h) {
    if (h.D < 1 || h.D > NF_STACK_DMAX || h.L < 1) return NF_ERR_BAD_SHAPE;
    if (h.HP != 64 && h.HP != 128) return NF_ERR_BAD_SHAPE;
    if (h.layer_stride % 4 != 0) return NF_ERR_MISALIGNED;
    return NF_OK;
}

static int spline_stack_launch(const StackCall& c, const StackHdr& h) {
    const int rc = check_hdr(h);
    if (rc != NF_OK) return rc;
    const int D = h.D, HP = h.HP, K = h.K, NO = h.NO, stride = h.layer_stride;
    if (K < 2 || K > 16 || NO % 4 != 0) return NF_ERR_BAD_SHAPE;
    if (!c.holds(NF_STACK_HDR + (int64_t)h.L * stride)) return NF_ERR_WORKSPACE;
    const int R = (HP == 64) ? 2 : 1;
    const int rows = kStackThreads * R;
    const size_t smem = sizeof(float) * ((size_t)stride + (size_t)NO * rows);
#define NF_SS(HPv, Rv, DMv, KMv)                                                                                     \
    return launch_stack(c.sample ? spline_stack_kernel<HPv, Rv, DMv, KMv, true> : spline_stack_kernel<HPv, Rv, DMv, KMv>, \
                        smem, rows, c, stride, true)
    if (HP == 64) {
        if (D <= 3) { if (K <= 8) NF_SS(64, 2, 4, 8); else NF_SS(64, 2, 4, 16); }
        else        { if (K <= 8) NF_SS(64, 2, 8, 8); else NF_SS(64, 2, 8, 16); }
    } else {
        if (D <= 3) { if (K <= 8) NF_SS(128, 1, 4, 8); else NF_SS(128, 1, 4, 16); }
        else        { if (K <= 8) NF_SS(128, 1, 8, 8); else NF_SS(128, 1, 8, 16); }
    }
#undef NF_SS
}

static int coupling_stack_launch(const StackCall& c, const StackHdr& h) {
    const int rc = check_hdr(h);
    if (rc != NF_OK) return rc;
    const int D = h.D, HP = h.HP, stride = h.layer_stride;
    if (h.NO != (D <= 3 ? 4 : 8)) return NF_ERR_BAD_SHAPE;
    if (!c.holds(NF_STACK_HDR + (int64_t)h.L * stride)) return NF_ERR_WORKSPACE;
    const int R = (HP == 64) ? 2 : 1;
    const int rows = kStackThreads * R;
    const size_t smem = sizeof(float) * (size_t)stride;
#define NF_CS(HPv, Rv, DMv)                                                                                          \
    return launch_stack(c.sample ? coupling_stack_kernel<HPv, Rv, DMv, true> : coupling_stack_kernel<HPv, Rv, DMv>,   \
                        smem, rows, c, 0, false)
    if (HP == 64) { if (D <= 3) NF_CS(64, 2, 4); else NF_CS(64, 2, 8); }
    else          { if (D <= 3) NF_CS(128, 1, 4); else NF_CS(128, 1, 8); }
#undef NF_CS
}

static const StackFamily kSpline = {NF_STACK_MAGIC_SPLINE, spline_stack_launch};
static const StackFamily kCoupling = {NF_STACK_MAGIC_AFFINE, coupling_stack_launch};

}  // namespace nf

using namespace nf;

extern "C" int64_t nf_spline_stack_packed_floats(int D, int H, int K, int L) {
    if (D < 1 || D > NF_STACK_DMAX || H < 1 || H > 128 || K < 2 || K > 16 || L < 1) return -1;
    const int HP = nf_stack_hp(H), W1S = nf_stack_w1s(D), P = 3 * K - 1;
    const int NO = 4 * ((D * P + 3) / 4);   // upper bound: the host packs with NO = 4*ceil(max_layers(Dt)*P/4) <= this
    return NF_STACK_HDR + (int64_t)L * (NF_LAYER_HDR + nf_stack_net_words(HP, W1S, NO));
}

extern "C" int64_t nf_coupling_stack_packed_floats(int D, int H, int L) {
    if (D < 1 || D > NF_STACK_DMAX || H < 1 || H > 128 || L < 1) return -1;
    const int HP = nf_stack_hp(H), W1S = nf_stack_w1s(D), NO = D <= 3 ? 4 : 8;
    return NF_STACK_HDR + (int64_t)L * (NF_LAYER_HDR + 2 * nf_stack_net_words(HP, W1S, NO));
}

extern "C" int nf_spline_stack_forward(const void* packed, const void* hdr_host, int64_t packed_bytes, const void* x,
                                       void* y, void* ld, int64_t B, int inverse, nf_stream_t stream) {
    return stack_forward(kSpline, packed, hdr_host, packed_bytes, x, y, ld, B, inverse, 0, stream);
}

extern "C" int nf_spline_stack_sample(const void* packed, const void* hdr_host, int64_t packed_bytes, uint64_t seed,
                                      uint64_t offset, void* x, void* log_q, int64_t B, nf_stream_t stream) {
    return stack_sample(kSpline, packed, hdr_host, packed_bytes, 0, seed, offset, x, log_q, B, stream);
}

extern "C" int nf_spline_stack_sample_state(const void* packed, const void* hdr_host, int64_t packed_bytes,
                                            void* rng_state, void* x, void* log_q, int64_t B, nf_stream_t stream) {
    return stack_sample_state(kSpline, packed, hdr_host, packed_bytes, 0, rng_state, x, log_q, B, stream);
}

extern "C" int nf_coupling_stack_forward(const void* packed, const void* hdr_host, int64_t packed_bytes,
                                         const void* x, void* y, void* ld, int64_t B, int inverse,
                                         nf_stream_t stream) {
    return stack_forward(kCoupling, packed, hdr_host, packed_bytes, x, y, ld, B, inverse, 0, stream);
}

extern "C" int nf_coupling_stack_sample(const void* packed, const void* hdr_host, int64_t packed_bytes, uint64_t seed,
                                        uint64_t offset, void* x, void* log_q, int64_t B, nf_stream_t stream) {
    return stack_sample(kCoupling, packed, hdr_host, packed_bytes, 0, seed, offset, x, log_q, B, stream);
}

extern "C" int nf_coupling_stack_sample_state(const void* packed, const void* hdr_host, int64_t packed_bytes,
                                              void* rng_state, void* x, void* log_q, int64_t B, nf_stream_t stream) {
    return stack_sample_state(kCoupling, packed, hdr_host, packed_bytes, 0, rng_state, x, log_q, B, stream);
}
