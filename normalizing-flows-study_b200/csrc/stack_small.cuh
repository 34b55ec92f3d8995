// stack_small.cuh -- packed-weight layout of the fused small-data_dim inference stacks.
// Shared by stack_small.cu (device) and mirrored by the Python packer (nfb200/packing.py), which asks
// nf_*_stack_packed_floats() for sizes and fills the buffer following the offsets documented here.
//
// All words are 32-bit; integers are stored as int32 bit patterns inside the float buffer.
//
//   header (NF_STACK_HDR words, read on the host through StackHdr below):
//     [0] magic   [1] D   [2] H (true hidden_dim)   [3] HP (padded: 64 or 128; the tcgen05 layouts of stack_tc.cu
//     store the number of conditioner nets per layer here instead: 1 spline / MADE, 2 affine; 'NFC2' / 'NFD2' the context width C)   [4] K (spline) / 0 (affine)
//     [5] L       [6] W1S (words per hidden unit in W1k: 4 if D<=3 else 12)      [7] NO (padded #outputs of the head)
//     [8] layer_stride (words)   [9] bn_between (0/1)   [10] bound   [11] min_w  [12] min_h  [13] min_d
//     [14] scale_w = 1-min_w*K   [15] scale_h
//   per layer (layer_stride words, 16-byte aligned sections):
//     the 80-word layer header (NF_LAYER_HDR, see LayerHdr below)
//     then `nets` conditioner blocks (1 for spline: param_net; 2 for affine: s_net, b_net), each:
//       W1k [HP][W1S]   : {W1[k][0..D-1], zero pad.., b1[k] at slot W1S-1}
//       W2t [HP][HP]    : W2t[k][j] = W2[j][k]
//       b2  [HP]
//       W3c [NO/4][HP][4]: W3c[c][j][q] = W3[out(c*4+q)][j]
//       b3  [NO]
//   spline head outputs are ordered t*P + p for transformed dim t (P = 3K-1); affine head outputs are d.
//
// The tcgen05 spline layout 'NFS2' (stack_tc.cu: blk_offsets, packing._tc_net_block) has per layer the 80-word header,
// then W1k [64][W1S] | b2 [64] | b3 [NO] | pad to 256 words | W2 hi / lo images | W3 hi / lo images.  Its conditional
// twin 'NFC2' (SplineCouplingLayer with context_dim = C, 1 <= C <= 8) stores C in header word [3] and inserts the
// context columns of the first Linear after b3:
//       Wc  [32][8][2]  : unit pairs (2p, 2p+1), 8 context slots each: Wc[p][c][e] = W1[2p+e][D+c], zero for c >= C
// W1k keeps the x columns W1[k][0..D-1] exactly as in 'NFS2', so a pack whose context columns are zero computes what
// the 'NFS2' pack of the remaining weights computes.
// The tcgen05 affine layout 'NFA2' has two such net blocks per layer (s_net, b_net; HP = 64 or 128 hidden units, each
// block led by 80 words: the layer header for s_net, zeros for b_net).  Its conditional twin 'NFD2' (CouplingLayer with
// context_dim = C, 1 <= C <= 8) stores C in header word [3] and gives EACH net block a Wc [HP/2][8][2] section after b3,
// laid out as above, from the first Linear with its BatchNorm folded in: the fold scales whole rows of the [H, D + C]
// weight, context columns included, before they are split into W1k and Wc.
#pragma once
#include <stdint.h>
#include <string.h>
#include "nf_common.cuh"

#define NF_STACK_MAGIC_SPLINE 0x4e465331  /* 'NFS1' */
#define NF_STACK_MAGIC_AFFINE 0x4e464131  /* 'NFA1' */
#define NF_STACK_MAGIC_SPLINE_TC 0x4e465332  /* 'NFS2': tensor-core layout, see stack_tc.cu */
#define NF_STACK_MAGIC_AFFINE_TC 0x4e464132  /* 'NFA2' */
#define NF_STACK_MAGIC_MADE_TC 0x4e464d32    /* 'NFM2': MADE / MAF / IAF stack on the tensor cores, see stack_tc.cu */
#define NF_STACK_MAGIC_SPLINE_CTX_TC 0x4e464332  /* 'NFC2': conditional spline stack on the tensor cores, see below */
#define NF_STACK_MAGIC_AFFINE_CTX_TC 0x4e464432  /* 'NFD2': conditional affine coupling stack on the tensor cores */
#define NF_STACK_HDR 16
#define NF_LAYER_HDR 80
#define NF_STACK_DMAX 8
// `inverse` argument of the fused stack entry points is a flag word:
//   bit 0  direction (1 = inverse, x -> z)
//   bit 1  log-prob head: the per-row output is log N(z; 0, I) + log_det (Flow.log_prob, flow.py:56-73) instead of
//          log_det -- the standard-normal head evaluated on the row while it is still in registers
//   bit 2  do not store the transformed rows (y may be NULL): Flow.log_prob only returns the per-row value
//   bit 3  (nf_made_chain_bf16_forward, IAF.forward only) the per-row output is log N(x_in; 0, I) - log_det of the INPUT
//          row: the sample_and_log_prob head when the input is the N(0, I) draw
#define NF_STACK_INVERSE 1
#define NF_STACK_LOG_PROB_HEAD 2
#define NF_STACK_SKIP_Y 4
#define NF_STACK_SAMPLE_LOG_Q 8

// the 16 header words; HP is word 3 (nets per layer in the tcgen05 layouts)
struct StackHdr {
    int magic, D, H, HP, K, L, W1S, NO, layer_stride, bn_between;
    float bound, min_w, min_h, min_d, scale_w, scale_h;
};
static_assert(sizeof(StackHdr) == 4 * NF_STACK_HDR, "StackHdr mirrors the 16 header words");

// host copy of the header that the caller passes beside the device buffer (hdr_host of the entry points)
static inline StackHdr nf_stack_hdr(const void* hdr_host) {
    StackHdr h;
    memcpy(&h, hdr_host, sizeof(int32_t) * NF_STACK_HDR);
    return h;
}

#ifdef __CUDACC__
// the kernels' read of the same words at the start of the packed buffer
__device__ __forceinline__ StackHdr nf_stack_hdr_device(const float* __restrict__ p) {
    const int* q = reinterpret_cast<const int*>(p);
    StackHdr h;
    h.magic = q[0]; h.D = q[1]; h.H = q[2]; h.HP = q[3]; h.K = q[4]; h.L = q[5]; h.W1S = q[6]; h.NO = q[7];
    h.layer_stride = q[8]; h.bn_between = q[9];
    h.bound = p[10]; h.min_w = p[11]; h.min_h = p[12]; h.min_d = p[13]; h.scale_w = p[14]; h.scale_h = p[15];
    return h;
}
#endif

static inline int nf_stack_hp(int H) { return H <= 64 ? 64 : 128; }
static inline int nf_stack_w1s(int D) { return D <= 3 ? 4 : 12; }
static inline int64_t nf_stack_net_words(int HP, int W1S, int NO) {
    return (int64_t)HP * W1S + (int64_t)HP * HP + HP + (int64_t)NO * HP + NO;
}

#ifdef __CUDACC__
namespace nf {

// One call of a fused-stack entry point.  sample: the SAMPLE kernel draws the rows from (seed, offset), or from the
// device-resident state when rng_state is not NULL; x is not read.  mode: MADE only.
// The context of a conditional stack: row r of the batch reads row r / div of ctx [rows][C] (div = 1: one context row
// per row; div = B: one row broadcast; div = n: n samples per context row).  ctx == NULL in the unconditional families.
struct StackCtx { const void* ctx = nullptr; int64_t rows = 0, div = 1; };

struct StackCall {
    const void* packed; const void* hdr_host; int64_t packed_bytes;
    const void* x; void* y; void* ld; int64_t B; int flags; int mode;
    bool sample; uint64_t seed, offset; unsigned long long* rng_state; cudaStream_t st;
    StackCtx cx = {};
    bool holds(int64_t words) const { return packed_bytes >= (int64_t)sizeof(float) * words; }   // packed_bytes suffices
};

// A family's launcher: its envelope checks, shared-memory sizing and instantiation switch, called with the header
// after the checks every family shares (stack_small.cu: run_stack).
struct StackFamily {
    int magic;
    int (*launch)(const StackCall& c, const StackHdr& h);
};

// bodies of the nf_*_forward / nf_*_sample / nf_*_sample_state entry points
int stack_forward(const StackFamily& f, const void* packed, const void* hdr_host, int64_t packed_bytes, const void* x,
                  void* y, void* ld, int64_t B, int flags, int mode, nf_stream_t stream, StackCtx cx = {});
int stack_sample(const StackFamily& f, const void* packed, const void* hdr_host, int64_t packed_bytes, int mode,
                 uint64_t seed, uint64_t offset, void* x, void* log_q, int64_t B, nf_stream_t stream, StackCtx cx = {});
int stack_sample_state(const StackFamily& f, const void* packed, const void* hdr_host, int64_t packed_bytes, int mode,
                       void* rng_state, void* x, void* log_q, int64_t B, nf_stream_t stream, StackCtx cx = {});

// dynamic shared memory beyond 48 KB, and the largest shared-memory carveout: with the default preference the driver
// sizes the SM for ONE CTA of the kernel and a second co-resident CTA never arrives
template <typename Kern>
inline int stack_smem_attributes(Kern kern, size_t smem) {
    NF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    NF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    return NF_OK;
}

// The 80-word header at the start of every layer block, as packing._layer_header writes it (ints as int32 bit
// patterns, one 8-word section per field):
//   mask | tdim (int) | meta: {Dt, rescale, bn_on (int), bn_ld (float)} | r_in | r_lo | r_out | bn_mean | bn_sd | bn_gamma
//   | bn_beta
// A view of it in shared memory.
struct LayerHdr {
    enum : int { kMask = 0, kTdim = 8, kMeta = 16, kRin = 24, kRlo = 32, kRout = 40,
                 kBnMean = 48, kBnSd = 56, kBnGamma = 64, kBnBeta = 72 };
    const float* p;
    __device__ __forceinline__ const float* mask() const { return p + kMask; }
    __device__ __forceinline__ bool rescale() const { return reinterpret_cast<const int*>(p + kMeta)[1] != 0; }
    __device__ __forceinline__ bool bn_on() const { return reinterpret_cast<const int*>(p + kMeta)[2] != 0; }
    // data_min / data_max rescale of a spline layer (spline_coupling_layer.py:101-102): dim d into spline coordinates
    // [-bound, bound] and back
    __device__ __forceinline__ float to_spline(float v, int d, float bound) const {
        return p[kRin + d] * (v - p[kRlo + d]) - bound;
    }
    __device__ __forceinline__ float from_spline(float v, int d, float bound) const {
        return (v + bound) * p[kRout + d] + p[kRlo + d];
    }
};
static_assert(LayerHdr::kBnBeta + 8 == NF_LAYER_HDR, "LayerHdr covers the layer header");

// between-layer BatchNorm as an invertible affine on running stats (normalizing_flow_model.py:67-128), one row
template <int DM>
__device__ __forceinline__ void nf_stack_bn_between(LayerHdr lh, int D, bool inverse, float (&xv)[DM], float& tot) {
    const float* mean = lh.p + LayerHdr::kBnMean; const float* sd = lh.p + LayerHdr::kBnSd;
    const float* gm = lh.p + LayerHdr::kBnGamma; const float* bt = lh.p + LayerHdr::kBnBeta;
    const float bn_ld = lh.p[LayerHdr::kMeta + 3];
#pragma unroll
    for (int d = 0; d < DM; ++d) if (d < D) {
        if (!inverse) xv[d] = (xv[d] - mean[d]) / sd[d] * gm[d] + bt[d];
        else          xv[d] = (xv[d] - bt[d]) / gm[d] * sd[d] + mean[d];
    }
    tot = inverse ? tot - bn_ld : tot + bn_ld;
}

// log N(z; 0, I) + log_det for one row held in registers (same arithmetic as std_normal_log_prob_fwd_kernel)
template <int DM>
__device__ __forceinline__ float nf_stack_row_head(const float (&z)[DM], int D, float log_det) {
    float acc = 0.f;
#pragma unroll
    for (int d = 0; d < DM; ++d) if (d < D) acc += -0.5f * z[d] * z[d];
    return acc - (float)(0.5 * (double)D * 1.8378770664093453) + log_det;
}

// Row epilogue (r < B): the row into y unless NF_STACK_SKIP_Y, then the per-row value into ld:
// -tot when sampling, the log-prob head under NF_STACK_LOG_PROB_HEAD, tot otherwise
template <int DM, bool SAMPLE>
__device__ __forceinline__ void nf_stack_row_store(float* __restrict__ y, float* __restrict__ ld, int64_t r, int D, int flags,
                                                   const float (&z)[DM], float tot) {
    if (!(flags & NF_STACK_SKIP_Y)) {
#pragma unroll
        for (int d = 0; d < DM; ++d) if (d < D) st_stream(y + r * D + d, z[d]);
    }
    st_stream(ld + r, SAMPLE ? -tot : (flags & NF_STACK_LOG_PROB_HEAD) ? nf_stack_row_head<DM>(z, D, tot) : tot);
}

}  // namespace nf
#endif
