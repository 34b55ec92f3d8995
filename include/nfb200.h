/* nfb200.h -- C ABI of libnfb200.so, the B200 (sm_100a) implementation of the
 * itxtx/normalizing-flows-study transform hot path.
 *
 * The reference has no FFI/plugin boundary of its own: its hot path is nn.Module code calling ATen
 * eager ops (SURVEY 8b).  This header is therefore the boundary *we* define underneath the
 * reference's Python class surface; each entry point names the reference function whose arithmetic
 * it replaces (paths relative to the reference repository root).
 *
 * Conventions (every function):
 *   - plain device pointers + sizes; no torch types.  All tensors are dense, row-major, contiguous.
 *   - the caller owns every buffer (outputs and workspaces included); the library never allocates
 *     device memory, never synchronises, keeps no per-call global state and launches on `stream`
 *     (a cudaStream_t passed as void*).  Calls on distinct streams may run concurrently.
 *   - `dtype` selects the arithmetic type of all floating buffers of the call (NF_F32 / NF_F64).
 *   - returns NF_OK (0) or a negative nf_status; nothing is launched when an argument check fails.
 *   - built for sm_100a only; there is no CPU path.
 */
#ifndef NFB200_H
#define NFB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* nf_stream_t; /* cudaStream_t */

#if defined(__GNUC__)
#define NF_API __attribute__((visibility("default")))
#else
#define NF_API
#endif

enum nf_status {
    NF_OK = 0,
    NF_ERR_BAD_SHAPE = -1,   /* negative / inconsistent sizes, unsupported bin count, ... */
    NF_ERR_UNSUPPORTED = -2, /* dtype or configuration without a kernel */
    NF_ERR_MISALIGNED = -3,  /* a pointer that must be 16-byte aligned is not */
    NF_ERR_CUDA = -4,        /* a CUDA runtime call failed: see nf_last_cuda_error() */
    NF_ERR_NULL = -5,        /* required pointer is NULL */
    NF_ERR_WORKSPACE = -6    /* workspace / packed-weight buffer too small */
};
enum nf_dtype { NF_F32 = 0, NF_F64 = 1 };

/* affine autoregressive modes (nf_affine_ar_*, nf_ar_sequential_*) */
enum nf_ar_mode {
    NF_AR_MAF_INVERSE = 0, /* masked_autoregressive_flow.py:18-44  (parallel, density) */
    NF_AR_IAF_FORWARD = 1, /* inverse_autoregressive_flow.py:30-63 (parallel, sampling) */
    NF_AR_MAF_FORWARD = 2, /* masked_autoregressive_flow.py:46-78  (sequential, sampling) */
    NF_AR_IAF_INVERSE = 3  /* inverse_autoregressive_flow.py:65-103 (sequential, density) */
};

NF_API int nf_abi_version(void);
NF_API const char* nf_status_string(int status);
NF_API const char* nf_last_cuda_error(void);
/* number of kernel launches issued by this library since load (bench.py's gpu_launches) */
NF_API int64_t nf_launch_count(void);
/* library options (0 = accepted; any other key than 7, 10 and 11 is refused with NF_ERR_UNSUPPORTED):
 * key 7 = nf_linear_tc* and nf_linear_wgrad_tc*: tensor-core passes per product.  3 = 3xTF32 (fp32 parity, default);
 *         1 = one TF32 pass, operands rounded to the nearest TF32 (the reduced-precision conditioner-GEMM mode the
 *         reference reaches with autocast, optimization/mixed_precision.py:89-105; w_lo is not read);
 * key 10 = nf_linear_tc* in the one-pass mode: 1 = A operand straight from shared memory (x truncated to TF32 by the tensor
 *         core instead of rounded by the converter warps); default 0;
 * key 11 = nf_spline_transform_* (float32, compact layout, 8 / 10 bins): 1 = TMA-staged kernels (spline_stream.cu,
 *         default), 0 = the first-version cp.async kernels */
NF_API int nf_set_option(int key, int value);

/* ---- a7: rational_quadratic_spline(inputs, widths, heights, derivatives, inverse, ...) ----------
 * src/flows/spline/rational_quadratic_spline.py:4-104.  x,y,ld: [n]; w,h: [n,K]; d: [n,K-1].
 * Per-element outputs and per-element log|dy/dx| (no row sum), domain [0,1], epsilon 1e-6. */
NF_API int nf_rqs_unit_forward(const void* x, const void* w, const void* h, const void* d, void* y, void* ld, int64_t n,
                        int num_bins, int inverse, double min_bin_width, double min_bin_height, double min_derivative,
                        int dtype, nf_stream_t stream);
/* reverse mode of the above: gx [n], gw/gh [n,K], gd [n,K-1] are overwritten. */
NF_API int nf_rqs_unit_backward(const void* x, const void* w, const void* h, const void* d, const void* gy, const void* gld,
                         void* gx, void* gw, void* gh, void* gd, int64_t n, int num_bins, int inverse,
                         double min_bin_width, double min_bin_height, double min_derivative, int dtype,
                         nf_stream_t stream);

/* ---- a5/a6: SplineCouplingLayer.forward/.inverse minus the conditioner ------------------------------
 * src/flows/spline/spline_coupling_layer.py:96-309.  x,y: [B,D]; params: [B, D*(3K-1)] = param_net output
 * (row d*P+j = parameter j of dim d, :71); mask: [D] float {0,1}; tidx: [Dt] int32 indices with mask==0;
 * ld: [B] = row sum over transformed dims, NaN/Inf scrubbed (:130-135).  rescale_in/rescale_lo/rescale_out:
 * NULL, or [D] arrays a,lo,c with x_spline = a*(x-lo)-bound and x_out = (y+bound)*c+lo (:78-94). */
NF_API int nf_spline_transform_forward(const void* x, const void* params, const void* mask, const int32_t* tidx, void* y,
                                void* ld, int64_t B, int D, int Dt, int num_bins, int inverse, double bound,
                                double min_bin_width, double min_bin_height, double min_derivative,
                                const void* rescale_in, const void* rescale_lo, const void* rescale_out,
                                int params_compact, int dtype, nf_stream_t stream);
/* params_compact != 0: params is [B, Dt*(3K-1)], block t = parameters of dim tidx[t] (the conditioner's last layer
 * restricted to the transformed dims: the reference computes and discards the other half, SURVEY D9).
 * gx: [B,D] overwritten; gparams: same layout as params -- only the transformed dims' entries are written, the
 * caller zero-fills the buffer beforehand in the non-compact layout. */
NF_API int nf_spline_transform_backward(const void* x, const void* params, const void* mask, const int32_t* tidx,
                                 const void* gy, const void* gld, void* gx, void* gparams, int64_t B, int D, int Dt,
                                 int num_bins, int inverse, double bound, double min_bin_width, double min_bin_height,
                                 double min_derivative, const void* rescale_in, const void* rescale_lo,
                                 const void* rescale_out, int params_compact, int dtype, nf_stream_t stream);

/* ---- a1/a2: CouplingLayer.forward/.inverse minus the conditioners ---------------------------------
 * src/flows/coupling/coupling_layer.py:47-66 / :76-94.  s_raw,b_raw: [B,D] un-clamped s_net/b_net outputs. */
NF_API int nf_affine_coupling_forward(const void* x, const void* s_raw, const void* b_raw, const void* mask, void* y,
                               void* ld, int64_t B, int D, int inverse, int dtype, nf_stream_t stream);
NF_API int nf_affine_coupling_backward(const void* x, const void* s_raw, const void* b_raw, const void* mask, const void* gy,
                                const void* gld, void* gx, void* gs, void* gb, int64_t B, int D, int inverse,
                                int dtype, nf_stream_t stream);

/* ---- a11/a13 (parallel directions): MAF.inverse / IAF.forward minus MADE ----------------------------
 * params: [B,2D] = [mu_0..mu_{D-1}, alpha_0..alpha_{D-1}] (made.py:67-78).  ld clamped to +-100 / +-50. */
NF_API int nf_affine_ar_forward(const void* v, const void* params, void* out, void* ld, int64_t B, int D, int mode,
                         int dtype, nf_stream_t stream);
/* ld_saved: the forward's ld output (decides whether the +-100/+-50 clamp passes gradient). */
NF_API int nf_affine_ar_backward(const void* v, const void* params, const void* ld_saved, const void* gout, const void* gld,
                          void* gv, void* gparams, int64_t B, int D, int mode, int dtype, nf_stream_t stream);

/* ---- a8/a10 and the conditioner MLPs: dense building block ---------------------------------------------
 * C[M,N] (+)= A[M,K] * Bm[K,N] (+ bias[N]) (ReLU), with element strides for A and Bm so that
 *   Y = X W^T + b   (F.linear, masked_linear.py:18)      : sam=K, sak=1, sbk=1, sbn=K
 *   dX = dY W       (backward wrt input)                    : A=dY, Bm=W  -> sbk=K_w, sbn=1
 *   dW = dY^T X     (backward wrt weight)                   : A=dY^T      -> sam=1, sak=N_dy
 * k_extent: NULL, or int32[ceil(N/64)]: output columns [64t, 64t+64) only accumulate k < k_extent[t]
 * (zero-tile skipping for mask-folded, degree-sorted MADE weights, whose masks are block lower-triangular).
 * Weight-gradient shapes (few output tiles, K>=4096) are split along K and combined with atomics. */
NF_API int nf_gemm(const void* A, const void* Bm, void* C, const void* bias, int64_t M, int64_t N, int64_t K, int64_t sam,
            int64_t sak, int64_t sbk, int64_t sbn, int64_t ldc, int relu, int accumulate, const int32_t* k_extent,
            int dtype, nf_stream_t stream);

/* elementwise helpers of the training path (so that it never leaves this library):
 *   out = a * b (broadcast b over rows if b_rows==1): mask folding W*mask (masked_linear.py:17-18)
 *   relu backward: gx = gy * (y > 0);  column sum: out[N] = sum_m a[m,n] (bias gradient) */
NF_API int nf_mul_rows(const void* a, const void* b, void* out, int64_t rows, int64_t cols, int64_t b_rows, int dtype,
                nf_stream_t stream);
NF_API int nf_relu_backward(const void* y, const void* gy, void* gx, int64_t n, int dtype, nf_stream_t stream);
/* ReLU backward of a Linear(+ReLU) fused with that Linear's bias gradient (torch.relu's backward followed by the
 * grad_output.sum(0) of F.linear): gx[rows, cols] = gy where y > 0 else 0, colsum[cols] = column sums of gx; one pass
 * over y and gy instead of writing gx and reading it again.  colsum is overwritten. */
NF_API int nf_relu_backward_colsum(const void* y, const void* gy, void* gx, void* colsum, int64_t rows, int64_t cols,
                            int dtype, nf_stream_t stream);
NF_API int nf_col_sum(const void* a, void* out, int64_t rows, int64_t cols, int dtype, nf_stream_t stream);

/* nn.BatchNorm1d inside the coupling conditioners (coupling_layer.py:20,23), fused with the following ReLU.
 * training!=0: batch statistics normalise (biased variance), running stats are updated in place with
 * `momentum` (unbiased variance), save_mean/save_rstd [H] receive the batch statistics for backward.
 * training==0: running statistics normalise.  y = relu?(gamma*(x-mean)*rstd+beta).
 * workspace: 2*H doubles (batch-statistic partial sums; may be NULL when training==0). */
NF_API int nf_batchnorm_forward(const void* x, const void* gamma, const void* beta, void* running_mean, void* running_var,
                         void* y, void* save_mean, void* save_rstd, void* workspace, int64_t B, int H, int training,
                         double momentum, double eps, int relu, int dtype, nf_stream_t stream);
/* y is the forward output (post-ReLU when relu!=0).  gx [B,H], ggamma/gbeta [H] overwritten.  training
 * selects the batch-statistics Jacobian (training!=0) or the plain affine one (eval).  workspace: 2*H doubles.
 * beta (optional, may be NULL): the forward's beta.  With relu!=0 and beta given, the float32 128-bit kernels re-derive
 * the ReLU mask from x with the forward's own expression (bit-identical) instead of reading y -- a third / a quarter less
 * traffic for the two passes; y must still be valid (the other kernel variants read it). */
NF_API int nf_batchnorm_backward(const void* x, const void* y, const void* gamma, const void* save_mean,
                          const void* save_rstd, const void* gy, void* gx, void* ggamma, void* gbeta, void* workspace,
                          int64_t B, int H, int relu, int training, int dtype, const void* beta, nf_stream_t stream);

/* BatchNorm1d with statistics synchronised over data-parallel ranks (SURVEY 8e: CouplingLayer's train-mode BatchNorm,
 * coupling_layer.py:18-35, is the one cross-row reduction of the path; per-shard statistics make N GPUs != 1 GPU).
 * forward  stage 1: workspace[2H] doubles <- this shard's (sum x, sum x^2); nothing else is touched.  The caller all-reduces
 *          the workspace (and the row count) over the ranks.
 *          stage 2: statistics from the workspace over `count` rows (= all ranks' rows), running-stat update (unbiased
 *          variance with `count`), normalisation of this shard's B rows.
 * backward stage 1: workspace[2H] doubles <- this shard's (sum g*xhat, sum g) = its ggamma / gbeta (g = gy masked by ReLU).
 *          stage 2: gx of this shard's rows from the all-reduced sums in the workspace over `count` rows; ggamma / gbeta
 *          receive the GLOBAL sums (the caller keeps the local ones from stage 1 as the parameter gradients).
 * backward: beta as in nf_batchnorm_backward (stage 1 then also takes gamma for the mask; both optional).
 * count = -1 in stage 2: the row count is read from workspace[2H] on the device (the caller all-reduces [2H + 1] doubles:
 * the sums and its row count), so the pass needs no host read.  B may be 0 (empty shard). */
NF_API int nf_batchnorm_forward_staged(const void* x, const void* gamma, const void* beta, void* running_mean,
                                void* running_var, void* y, void* save_mean, void* save_rstd, void* workspace, int64_t B,
                                int H, double momentum, double eps, int relu, int stage, int64_t count, int dtype,
                                nf_stream_t stream);
NF_API int nf_batchnorm_backward_staged(const void* x, const void* y, const void* gamma, const void* save_mean,
                                 const void* save_rstd, const void* gy, void* gx, void* ggamma, void* gbeta,
                                 void* workspace, int64_t B, int H, int relu, int stage, int64_t count, int dtype,
                                 const void* beta, nf_stream_t stream);

/* ---- fused inference stacks (small data_dim): whole NormalizingFlowModel in one launch --------------------
 * a4-a6 + a14/a15: L SplineCouplingLayers (+ optional between-layer BatchNorm affine using running stats,
 * normalizing_flow_model.py:25-128) for data_dim<=8, hidden_dim<=128, num_bins<=16; fp32 only.
 * `packed` is the float32 device buffer laid out by the host side (csrc/stack_small.cuh documents the layout);
 * `hdr_host` is a HOST copy of its first 16 words (so the library never reads device memory on the host).
 * Returns NF_ERR_UNSUPPORTED when the configuration does not fit one SM's shared memory (caller uses the
 * layer-wise path: nf_gemm + nf_spline_transform_forward).
 * `inverse` of all four fused-stack entry points is a flag word: bit 0 = direction (1: x -> z); bit 1
 * (NF_STACK_LOG_PROB_HEAD = 2) = `ld` receives log N(z; 0, I) + log_det, the Flow.log_prob head for a standard-normal
 * base (flow.py:56-73), evaluated on the row while it is still in registers; bit 2 (NF_STACK_SKIP_Y = 4) = the
 * transformed rows are not stored (y may be NULL). */
NF_API int nf_spline_stack_forward(const void* packed, const void* hdr_host, int64_t packed_bytes, const void* x, void* y,
                            void* ld, int64_t B, int inverse, nf_stream_t stream);
/* a1/a2 + a14/a15: L CouplingLayers in eval mode (conditioner BatchNorm folded into the Linears at pack time). */
NF_API int nf_coupling_stack_forward(const void* packed, const void* hdr_host, int64_t packed_bytes, const void* x, void* y,
                              void* ld, int64_t B, int inverse, nf_stream_t stream);
/* upper bound (in 32-bit words) of the packed buffer for a configuration; -1 if the fused path cannot take it */
NF_API int64_t nf_spline_stack_packed_floats(int D, int H, int K, int L);
NF_API int64_t nf_coupling_stack_packed_floats(int D, int H, int L);

/* ---- a10-a13 fused: MADE chain + affine autoregressive transform --------------------------------------
 * Parallel directions (MAF.inverse, IAF.forward).  w0..w3: mask-folded weights W*mask ([H,D],[H,H],[H,H],[2D,H]),
 * b0..b3 biases; kext1/kext2/kext3: optional int32 k-extent arrays for layers 1..3 (see nf_gemm).
 * workspace: 2*B*max(H,2D) elements of `dtype`.  fp32/fp64. */
NF_API int nf_made_affine_forward(const void* v, const void* w0, const void* b0, const void* w1, const void* b1,
                           const void* w2, const void* b2, const void* w3, const void* b3, const int32_t* kext1,
                           const int32_t* kext2, const int32_t* kext3, void* workspace, void* out, void* ld, int64_t B,
                           int D, int H, int mode, int dtype, nf_stream_t stream);
/* Sequential directions (MAF.forward, IAF.inverse) computed incrementally: one masked MADE evaluation in
 * total instead of D (masked_autoregressive_flow.py:55-67 re-evaluates MADE D times).  Hidden units must be
 * ordered by non-decreasing degree (made.py:25-41; the host permutes them for D==2); gstart: int32[D+1],
 * gstart[g] = index of the first hidden unit with degree >= g.  fp32 only.  NF_ERR_UNSUPPORTED when the
 * (D+3H)*32 activation tile does not fit shared memory. */
NF_API int nf_ar_sequential_forward(const void* v, const void* w0, const void* b0, const void* w1, const void* b1,
                             const void* w2, const void* b2, const void* w3, const void* b3, const int32_t* gstart,
                             void* out, void* ld, int64_t B, int D, int H, int mode, nf_stream_t stream);

/* ---- a14: between-layer BatchNorm as an invertible per-feature affine, and the spline layer's rescale -------
 * y[b,d] = (x[b,d] - sub[d]) / div[d] * mul[d] + add[d]; sub/div/mul/add are [D] arrays or NULL (0, 1, 1,
 * add_scalar).  normalizing_flow_model.py:67-85 is (sub,div,mul,add) = (running_mean, sqrt(var+eps), gamma, beta);
 * its inverse :110-128 is (beta, gamma, sqrt(var+eps), running_mean); spline_coupling_layer.py:78-94 is
 * (data_min, NULL, scale, -bound). */
NF_API int nf_feature_affine_forward(const void* x, const void* sub, const void* div, const void* mul, const void* add,
                              double add_scalar, void* y, int64_t B, int D, int dtype, nf_stream_t stream);
/* gx [B,D] overwritten; gsub/gdiv/gmul/gadd: [D] outputs or NULL (skipped); workspace: 2*D doubles. */
NF_API int nf_feature_affine_backward(const void* x, const void* sub, const void* div, const void* mul, const void* gy,
                               void* gx, void* gsub, void* gdiv, void* gmul, void* gadd, void* workspace, int64_t B,
                               int D, int dtype, nf_stream_t stream);
/* per-feature batch mean and biased variance (running-stat update of normalizing_flow_model.py:74-79).
 * workspace: 2*D doubles. */
NF_API int nf_col_stats(const void* x, void* mean, void* var, void* workspace, int64_t B, int D, int dtype,
                 nf_stream_t stream);

/* ---- a12/a13 sequential directions, layered route (autograd / float64 / configurations the incremental kernel
 * does not take): loop body of masked_autoregressive_flow.py:55-67 / inverse_autoregressive_flow.py:76-91.
 * out = cur with column `col` replaced by the transform of v[:,col] under params[:, col], params[:, D+col];
 * ld_out = ld_in (NULL = 0) +- alpha.  mode: NF_AR_MAF_FORWARD or NF_AR_IAF_INVERSE. */
NF_API int nf_ar_step_forward(const void* cur, const void* v, const void* params, const void* ld_in, void* out,
                       void* ld_out, int64_t B, int D, int col, int mode, int dtype, nf_stream_t stream);
NF_API int nf_ar_step_backward(const void* v, const void* params, const void* gout, const void* gld, void* gcur, void* gv,
                        void* gparams, int64_t B, int D, int col, int mode, int dtype, nf_stream_t stream);
/* closing scrubs + log-det clamp of the loop (:69-76 / :93-101) */
NF_API int nf_ar_finish_forward(const void* cur, const void* v, const void* ld_sum, void* out, void* ld, int64_t B, int D,
                         int mode, int dtype, nf_stream_t stream);
NF_API int nf_ar_finish_backward(const void* cur, const void* ld_sum, const void* gout, const void* gld, void* gcur,
                          void* gv, void* gld_sum, int64_t B, int D, int mode, int dtype, nf_stream_t stream);

/* ---- a16: Flow.log_prob head for a standard-normal base (flow.py:56-73) ---------------------------------
 * lp[b] = sum_d(-z[b,d]^2/2) - D/2*log(2*pi) + ld[b]   (ld may be NULL).  backward: gz = -z*glp[b]; gld = glp. */
NF_API int nf_std_normal_log_prob_forward(const void* z, const void* ld, void* lp, int64_t B, int D, int dtype,
                                   nf_stream_t stream);
NF_API int nf_std_normal_log_prob_backward(const void* z, const void* glp, void* gz, int64_t B, int D, int dtype,
                                    nf_stream_t stream);

/* ---- sample_and_log_prob with a standard-normal base: z ~ N(0, I), (x, log_det) = forward(z), log_q = log N(z) - log_det
 * The base stream (csrc/nf_rng.cuh) is Philox4x32-10 keyed by (lo32(seed) ^ 0x6E666232, hi32(seed)), counter
 * (j, row, lo32(offset/4), hi32(offset/4)) for dims 4j..4j+3 of a row, Box-Muller on the two word pairs; every route draws
 * the same bits for the same (seed, offset), and a row does not depend on B.  B >= 2^32 is refused (NF_ERR_BAD_SHAPE).
 * nf_std_normal_draw: z [B,D] <- the draw (NF_F64 widens the float32 normals; float32 with D % 4 == 0 needs a 16-byte
 * aligned z).  log-q head: lq[b] = sum_d(-z[b,d]^2/2) - D/2*log(2*pi) - ld[b]; backward: gz = -z*glq[b] and
 * gld = -glq (either output may be NULL, then it is not written). */
NF_API int nf_std_normal_draw(uint64_t seed, uint64_t offset, void* z, int64_t B, int D, int dtype, nf_stream_t stream);
NF_API int nf_std_normal_log_q_forward(const void* z, const void* ld, void* lq, int64_t B, int D, int dtype,
                                       nf_stream_t stream);
NF_API int nf_std_normal_log_q_backward(const void* z, const void* glq, void* gz, void* gld, int64_t B, int D, int dtype,
                                        nf_stream_t stream);
/* The fused stacks with the draw in the kernel: the row load of nf_*_stack*_forward becomes the draw above, the stack runs
 * in the sampling direction, x (may be NULL) receives the rows and log_q the per-row log N(z) - log_det; one launch, no
 * input tensor.  Same packed layouts, headers and NF_ERR_UNSUPPORTED envelopes as the forward entry points. */
NF_API int nf_spline_stack_sample(const void* packed, const void* hdr_host, int64_t packed_bytes, uint64_t seed,
                                  uint64_t offset, void* x, void* log_q, int64_t B, nf_stream_t stream);
NF_API int nf_spline_stack_tc_sample(const void* packed, const void* hdr_host, int64_t packed_bytes, uint64_t seed,
                                     uint64_t offset, void* x, void* log_q, int64_t B, nf_stream_t stream);
NF_API int nf_coupling_stack_sample(const void* packed, const void* hdr_host, int64_t packed_bytes, uint64_t seed,
                                    uint64_t offset, void* x, void* log_q, int64_t B, nf_stream_t stream);
NF_API int nf_coupling_stack_tc_sample(const void* packed, const void* hdr_host, int64_t packed_bytes, uint64_t seed,
                                       uint64_t offset, void* x, void* log_q, int64_t B, nf_stream_t stream);
/* mode: NF_AR_IAF_FORWARD (any data_dim <= 8) or NF_AR_MAF_FORWARD (data_dim == 2) */
NF_API int nf_made_stack_tc_sample(const void* packed, const void* hdr_host, int64_t packed_bytes, int mode, uint64_t seed,
                                   uint64_t offset, void* x, void* log_q, int64_t B, nf_stream_t stream);
/* Device-resident generator state (CUDA-graph safe drawing): the *_state twins of nf_std_normal_draw and the five
 * nf_*_sample entry points take `rng_state`, caller-owned device memory holding uint64[4] = {seed, offset, ticket,
 * reserved} (8-byte aligned), ticket 0 between calls.  The call draws with the key (seed, offset) it reads from the state,
 * the same bits as the entry point above with that seed and offset, and the same launch advances the state: once the
 * call completes, offset has moved on by 4 and ticket is 0 (the last CTA to read the key stores them).  Nothing is read
 * or advanced on the host, so a captured call draws new samples on every replay.  B == 0 launches a one-thread kernel
 * that only advances the state; a refused call (any error code) launches nothing and leaves the state as it was.
 * A device-state launch of a tcgen05 stack needs 16 bytes more shared memory (the key) and the FP32-pipe sampling kernels
 * hold it in both forms; no configuration inside the envelopes comes within 16 bytes of a shared-memory limit (the closest
 * leaves 1.8 KB), so both forms accept the same configurations and the bit equality holds wherever either runs.
 * Stream-ordered: one state must not be used by two streams at once.  The library neither allocates nor synchronises;
 * the state is caller memory. */
NF_API int nf_std_normal_draw_state(void* rng_state, void* z, int64_t B, int D, int dtype, nf_stream_t stream);
NF_API int nf_spline_stack_sample_state(const void* packed, const void* hdr_host, int64_t packed_bytes, void* rng_state,
                                        void* x, void* log_q, int64_t B, nf_stream_t stream);
NF_API int nf_spline_stack_tc_sample_state(const void* packed, const void* hdr_host, int64_t packed_bytes, void* rng_state,
                                           void* x, void* log_q, int64_t B, nf_stream_t stream);
NF_API int nf_coupling_stack_sample_state(const void* packed, const void* hdr_host, int64_t packed_bytes, void* rng_state,
                                          void* x, void* log_q, int64_t B, nf_stream_t stream);
NF_API int nf_coupling_stack_tc_sample_state(const void* packed, const void* hdr_host, int64_t packed_bytes,
                                             void* rng_state, void* x, void* log_q, int64_t B, nf_stream_t stream);
NF_API int nf_made_stack_tc_sample_state(const void* packed, const void* hdr_host, int64_t packed_bytes, int mode,
                                         void* rng_state, void* x, void* log_q, int64_t B, nf_stream_t stream);

/* ---- fused inference stacks on the tensor cores (tcgen05 + TMEM, 3xTF32 = fp32-accurate): same contract as
 * nf_spline_stack_forward, for hidden_dim <= 64, num_bins <= 10 and at most 2 transformed dims per layer; `packed`
 * follows the tensor-core layout (csrc/stack_tc.cu; magic 'NFS2').  NF_ERR_UNSUPPORTED otherwise. */
NF_API int nf_spline_stack_tc_forward(const void* packed, const void* hdr_host, int64_t packed_bytes, const void* x, void* y,
                               void* ld, int64_t B, int inverse, nf_stream_t stream);
/* affine coupling stack (eval mode) on the tensor cores: same contract as nf_coupling_stack_forward for hidden_dim <= 128
 * (hidden units padded to 64, two CTAs per SM, or to 128, one CTA per SM with all 512 TMEM columns);
 * `packed` in the tensor-core layout (magic 'NFA2': two net blocks per layer, csrc/stack_tc.cu). */
NF_API int nf_coupling_stack_tc_forward(const void* packed, const void* hdr_host, int64_t packed_bytes, const void* x,
                                 void* y, void* ld, int64_t B, int inverse, nf_stream_t stream);
NF_API int64_t nf_coupling_stack_tc_block_words(int D);
/* words per NET block of that layout for hidden_dim H (<= 64: same as above; <= 128: the 128-wide layout); -1 = unsupported */
NF_API int64_t nf_coupling_stack_tc_block_words_hidden(int D, int H);
/* words per layer block of that layout (-1 if the configuration is not supported) */
NF_API int64_t nf_spline_stack_tc_block_words(int D, int K, int max_dt);
/* eval-mode stack of MaskedAutoregressiveFlow / InverseAutoregressiveFlow layers on the tensor cores (hidden_dim <= 64,
 * data_dim <= 8; masked_autoregressive_flow.py:18-78, inverse_autoregressive_flow.py:30-103 around made.py:81-140) in ONE
 * launch: `packed` = magic 'NFM2', one block per layer of mask-folded weights (csrc/stack_tc.cu).  flags: the stack flag
 * word (NF_STACK_INVERSE walks the layers backwards, NF_STACK_LOG_PROB_HEAD / NF_STACK_SKIP_Y as above); mode: the
 * per-layer transform, NF_AR_MAF_INVERSE / NF_AR_IAF_FORWARD (parallel) for any data_dim, NF_AR_MAF_FORWARD /
 * NF_AR_IAF_INVERSE (the sequential directions) for data_dim == 2 only. */
NF_API int nf_made_stack_tc_forward(const void* packed, const void* hdr_host, int64_t packed_bytes, const void* x, void* y,
                             void* ld, int64_t B, int flags, int mode, nf_stream_t stream);
NF_API int64_t nf_made_stack_tc_block_words(int D);
/* ---- conditional spline stack on the tensor cores: L x SplineCouplingLayer with context_dim = C (1 <= C <= 8), whose
 * first Linear reads [x_rescaled * mask, c].  Same contract, flags and envelope as nf_spline_stack_tc_forward / _sample /
 * _sample_state, with `packed` in the conditional layout (magic 'NFC2', header word 3 = C; csrc/stack_small.cuh).
 * context: float32 [ctx_rows][C], row-major; row r of the batch reads context row r / ctx_div (ctx_div = 1: one context
 * row per row; ctx_div = B: one row broadcast to all; ctx_div = n: n consecutive sampled rows per context row).
 * Refused before any CUDA call, after the checks of the other stacks (B == 0 returns first, advancing a device state):
 * context == NULL -> NF_ERR_NULL; ctx_div < 1 or ctx_rows < ceil(B / ctx_div) -> NF_ERR_BAD_SHAPE; C outside 1..8 ->
 * NF_ERR_UNSUPPORTED.  An unconditional pack has another magic (NF_ERR_BAD_SHAPE), and so has an 'NFC2' pack passed to
 * the unconditional entry points.  The context does not enter the N(0, I) draw: the same (seed, offset) draws the same
 * rows as nf_spline_stack_tc_sample. */
NF_API int nf_spline_stack_ctx_tc_forward(const void* packed, const void* hdr_host, int64_t packed_bytes, const void* x,
                                          const void* context, int64_t ctx_rows, int64_t ctx_div, void* y, void* ld,
                                          int64_t B, int flags, nf_stream_t stream);
NF_API int nf_spline_stack_ctx_tc_sample(const void* packed, const void* hdr_host, int64_t packed_bytes,
                                         const void* context, int64_t ctx_rows, int64_t ctx_div, uint64_t seed,
                                         uint64_t offset, void* x, void* log_q, int64_t B, nf_stream_t stream);
NF_API int nf_spline_stack_ctx_tc_sample_state(const void* packed, const void* hdr_host, int64_t packed_bytes,
                                               const void* context, int64_t ctx_rows, int64_t ctx_div, void* rng_state,
                                               void* x, void* log_q, int64_t B, nf_stream_t stream);
/* ---- conditional affine coupling stack on the tensor cores: L x CouplingLayer with context_dim = C (1 <= C <= 8), whose
 * s_net and b_net both read [x * mask, c] in their first Linear.  Same contract, flags and envelope as
 * nf_coupling_stack_tc_forward / _sample / _sample_state, with `packed` in the conditional layout (magic 'NFD2', header
 * word 3 = C; csrc/stack_small.cuh).
 * context: float32 [ctx_rows][C], row-major; row r of the batch reads context row r / ctx_div (ctx_div = 1: one context
 * row per row; ctx_div = B: one row broadcast to all; ctx_div = n: n consecutive sampled rows per context row).
 * Refused before any CUDA call, after the checks of the other stacks (B == 0 returns first, advancing a device state):
 * context == NULL -> NF_ERR_NULL; ctx_div < 1 or ctx_rows < ceil(B / ctx_div) -> NF_ERR_BAD_SHAPE; C outside 1..8, or B
 * or ctx_div beyond 2^31 - 1 -> NF_ERR_UNSUPPORTED.  An unconditional pack has another magic (NF_ERR_BAD_SHAPE), and so
 * has an 'NFD2' pack passed to the unconditional entry points.  The context does not enter the N(0, I) draw: the same
 * (seed, offset) draws the same rows as nf_coupling_stack_tc_sample. */
NF_API int nf_coupling_stack_ctx_tc_forward(const void* packed, const void* hdr_host, int64_t packed_bytes, const void* x,
                                            const void* context, int64_t ctx_rows, int64_t ctx_div, void* y, void* ld,
                                            int64_t B, int flags, nf_stream_t stream);
NF_API int nf_coupling_stack_ctx_tc_sample(const void* packed, const void* hdr_host, int64_t packed_bytes,
                                           const void* context, int64_t ctx_rows, int64_t ctx_div, uint64_t seed,
                                           uint64_t offset, void* x, void* log_q, int64_t B, nf_stream_t stream);
NF_API int nf_coupling_stack_ctx_tc_sample_state(const void* packed, const void* hdr_host, int64_t packed_bytes,
                                                 const void* context, int64_t ctx_rows, int64_t ctx_div, void* rng_state,
                                                 void* x, void* log_q, int64_t B, nf_stream_t stream);
/* words per NET block of the 'NFD2' layout for data_dim D and hidden_dim H (<= 128); -1 = unsupported */
NF_API int64_t nf_coupling_stack_ctx_tc_block_words_hidden(int D, int H);

/* ---- a8/a10 and the conditioner MLPs on the tensor cores: y[M,N] = relu?(x[M,K] * W[N,K]^T + bias) ---------
 * fp32 in / fp32 out, 3xTF32 on tcgen05 (fp32-accurate), TMA-fed, accumulators in TMEM (csrc/gemm_tc2.cu).
 * w_hi / w_lo: the split of W produced by nf_split_tf32 (K contiguous).  ldx / ldw / ldy: row pitches in elements
 * (sub-matrices of larger arrays are addressed by pointer offset + pitch).  k_extent as in nf_gemm.  Requires
 * 16-byte aligned x / w_hi / w_lo and ldx % 4 == 0, ldw % 4 == 0 (NF_ERR_UNSUPPORTED otherwise: use nf_gemm). */
NF_API int nf_linear_tc(const void* x, const void* w_hi, const void* w_lo, const void* bias, void* y, int64_t M, int64_t N,
                 int64_t K, int64_t ldx, int64_t ldw, int64_t ldy, int relu, const int32_t* k_extent,
                 nf_stream_t stream);
/* same, with a per-64-output-columns lower bound of the K loop: columns k < k_begin[n/64] of those outputs' weights
 * are exact zeros (the transposed, block-lower-triangular MADE weights of the input-gradient product) */
NF_API int nf_linear_tc_range(const void* x, const void* w_hi, const void* w_lo, const void* bias, void* y, int64_t M,
                       int64_t N, int64_t K, int64_t ldx, int64_t ldw, int64_t ldy, int relu, const int32_t* k_begin,
                       const int32_t* k_extent, nf_stream_t stream);
/* hi = w rounded to the nearest TF32, lo = (w - hi) rounded to the nearest TF32; n elements, fp32 */
NF_API int nf_split_tf32(const void* w, void* w_hi, void* w_lo, int64_t n, nf_stream_t stream);

/* ---- weight gradient of those layers on the tensor cores: dw[N,K] = sum_b dy[b,N] * x[b,K] -----------------
 * (autograd of F.linear, masked_linear.py:18; fp32, 3xTF32 on tcgen05, both operands consumed in their row-major
 * layout: dy through TMEM as the A operand, x as an MN-major shared-memory B operand; csrc/wgrad_tc.cu).
 * The reduction over the batch is split across CTAs; partial tiles go to `workspace`
 * (nf_linear_wgrad_tc_workspace(B,N,K) bytes, 0 when no split is needed) and are summed in a fixed order
 * (deterministic).  Requires 16-byte aligned x and ld_x % 4 == 0 (NF_ERR_UNSUPPORTED otherwise: use nf_gemm); a dy
 * whose pitch TMA cannot take (ld_dy % 4 != 0: the 3K-1 wide spline heads) is read with plain loads.  B == 0 writes zeros. */
NF_API int64_t nf_linear_wgrad_tc_workspace(int64_t B, int64_t N, int64_t K);
NF_API int nf_linear_wgrad_tc(const void* dy, const void* x, void* dw, int64_t B, int64_t N, int64_t K, int64_t ld_dy,
                       int64_t ld_x, int64_t ld_dw, void* workspace, int64_t ws_bytes, nf_stream_t stream);
/* tile_live: NULL, or uint8[ceil(N/128) * ceil(K/128)] (K tiles fastest): 0 marks a 128 x 128 tile of dw on which the
 * layer's weight mask is entirely zero (MaskedLinear, masked_linear.py:17) -- it is written as zeros without being computed */
NF_API int nf_linear_wgrad_tc_masked(const void* dy, const void* x, void* dw, int64_t B, int64_t N, int64_t K, int64_t ld_dy,
                              int64_t ld_x, int64_t ld_dw, void* workspace, int64_t ws_bytes, const uint8_t* tile_live,
                              nf_stream_t stream);

/* ---- (f2) ARQS, one step of either sequential loop (src/flows/spline/arqs.py:53-76 / :93-116) ------------------
 * out[B,D] = cur with column `col` replaced by rational_quadratic_spline(v[:, col]; params[row]) on [0,1]
 * (rational_quadratic_spline.py:4-104), ld_out = ld_in + log|dy/dx| (ld_in NULL = zeros).  params: the [B, 3K-1]
 * conditioner outputs of dimension `col` (row pitch ldp elements).  ld_in / ld_out / gld are float32 for every
 * dtype (the reference accumulates into torch.zeros(B), arqs.py:52).  out may alias cur.  num_bins <= 16. */
NF_API int nf_arqs_step_forward(const void* cur, const void* v, const void* params, int64_t ldp, const void* ld_in,
                         void* out, void* ld_out, int64_t B, int D, int col, int num_bins, int inverse,
                         double min_bin_width, double min_bin_height, double min_derivative, int dtype,
                         nf_stream_t stream);
/* gcur = gout with column col zeroed; gv [B,D] zero outside col; gparams [B, 3K-1] dense; gld may be NULL */
NF_API int nf_arqs_step_backward(const void* v, const void* params, int64_t ldp, const void* gout, const void* gld,
                          void* gcur, void* gv, void* gparams, int64_t B, int D, int col, int num_bins, int inverse,
                          double min_bin_width, double min_bin_height, double min_derivative, int dtype,
                          nf_stream_t stream);

/* ---- a12/a13 sequential directions, blocked (csrc/ar_blocked.cu): hidden pre-activations of a block of degrees PULL
 * the contributions of all previous blocks as dense products on tcgen05 (column slices of the activation buffers),
 * the in-block dependent steps run in a persistent small-footprint kernel, and every finished block PUSHES its
 * layer-3 units into the output-layer pre-activations of all later dims (one narrow-K product, accumulated).
 * w / b: arrays of 4 device pointers, mask-folded degree-sorted weights and biases of the 4 MADE layers (output layer
 * as made.py:136-140 lays it out, [mu rows | alpha rows]); w_hi / w_lo: their TF32 splits, the output layer's rows
 * INTERLEAVED (row 2g = mu_g, row 2g+1 = alpha_g).  gstart: int32[D+1], first unit of degree >= g (device and host
 * copies); every block of `block_degrees` degrees must start at a multiple of 4 units (pad the blocks with dead units:
 * zero weights and biases -- packing.blocked_made_pack does), H is that padded width.  workspace:
 * nf_ar_blocked_workspace_floats() floats.  float32; D % 4 == 0, H % 4 == 0, block_degrees % 4 == 0 (8). */
NF_API int nf_ar_blocked_forward(const void* v, const void* const* w, const void* const* w_hi, const void* const* w_lo,
                          const void* const* b, const int32_t* gstart_dev, const int32_t* gstart_host, void* workspace,
                          void* out, void* ld, int64_t B, int D, int H, int mode, int block_degrees, nf_stream_t stream);
NF_API int64_t nf_ar_blocked_workspace_floats(int64_t B, int D, int H);

/* ---- a10 + a11 / a13 in ONE launch, bf16 tensor-core mode (csrc/made_chain_bf16.cu): MADE.forward (made.py:136-140, 4 masked
 * linears + 3 ReLU) + MAF.inverse (masked_autoregressive_flow.py:18-44) / IAF.forward (inverse_autoregressive_flow.py:30-63)
 * + row log-det; activations stay on the SM in bf16 (kind::f16 MMAs, fp32 accumulation), only x [B,D] fp32 is read and
 * out [B,D] / ld [B] fp32 are written.  Reduced precision: bf16 operands (documented bounds in DESIGN.md) -- the fp32-parity
 * path is nf_linear_tc x4 + nf_affine_ar_forward.
 * w0 [H,64] (input layer, K zero-padded to 64), w1 / w2 [H,H], w3 [128,H] (rows 0..D-1 = mu rows, rows 64..64+D-1 = alpha
 * rows, others zero): bf16, row-major, mask folded, hidden units sorted by degree; b0..b2 [H], b3 [128] (same row layout
 * as w3): fp32.  kext16_host: HOST int32[16] = [layer][128-column block] number of 16-wide k-steps holding non-zero
 * weights (the rest is skipped).  flags: bit 1 (2) = ld receives log N(out; 0, I) + log_det (Flow.log_prob head, flow.py:56-73);
 * bit 2 (4) = out is not stored (may be NULL); bit 3 (NF_STACK_SAMPLE_LOG_Q = 8, NF_AR_IAF_FORWARD only) = ld receives
 * log N(x; 0, I) - log_det of the INPUT row, the sample_and_log_prob head when x is the N(0, I) draw.  mode: NF_AR_MAF_INVERSE or NF_AR_IAF_FORWARD.
 * NF_ERR_UNSUPPORTED unless D <= 64, D % 4 == 0, H % 128 == 0, H <= 512. */
NF_API int nf_made_chain_bf16_forward(const void* x, const void* w0, const void* w1, const void* w2, const void* w3,
                               const void* b0, const void* b1, const void* b2, const void* b3, const int32_t* kext16_host,
                               void* out, void* ld, int64_t B, int D, int H, int mode, int flags, nf_stream_t stream);

/* ---- unit-test hook of the tcgen05 tile primitive (csrc/tc_common.cuh): D[128,N] = A[128,64] * W[N,64]^T.
 * w_images: the hi then the lo K-major SWIZZLE_128B image of W (packing.umma_sw128_images); N % 16 == 0, <= 128;
 * passes: 3 = 3xTF32 (fp32-accurate), 1 = single TF32 pass; > 3 and nacc > 1 (independent accumulators) are for
 * timing only.  timing: NULL or 2 x int64 device words receiving (issue cycles, issue-to-completion cycles). */
NF_API int nf_debug_tc_gemm128(const void* a, const void* w_images, void* d, int N, int passes, void* timing, int nacc,
                        nf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* NFB200_H */
