// capi_core.cu -- library-wide C-ABI helpers (status strings, last CUDA error, launch counter, options).
#include <atomic>
#include <mutex>
#include <string>
#include "nf_common.cuh"

namespace nf {

static std::atomic<int64_t> g_launches{0};
static std::mutex g_err_mu;
static std::string g_last_cuda_error;

void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
void count_launches(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

int nf_set_cuda_error(cudaError_t e) {
    std::lock_guard<std::mutex> lk(g_err_mu);
    g_last_cuda_error = cudaGetErrorString(e);
    return NF_ERR_CUDA;
}

}  // namespace nf

extern "C" int nf_abi_version(void) { return 1; }

extern "C" const char* nf_status_string(int status) {
    switch (status) {
        case NF_OK: return "ok";
        case NF_ERR_BAD_SHAPE: return "bad shape or size argument";
        case NF_ERR_UNSUPPORTED: return "unsupported dtype or configuration";
        case NF_ERR_MISALIGNED: return "pointer not 16-byte aligned";
        case NF_ERR_CUDA: return "CUDA runtime error";
        case NF_ERR_NULL: return "required pointer is NULL";
        case NF_ERR_WORKSPACE: return "workspace or packed buffer too small";
        default: return "unknown status";
    }
}

extern "C" const char* nf_last_cuda_error(void) {
    static thread_local std::string copy;
    std::lock_guard<std::mutex> lk(nf::g_err_mu);
    copy = nf::g_last_cuda_error;
    return copy.c_str();
}

extern "C" int64_t nf_launch_count(void) { return nf::g_launches.load(std::memory_order_relaxed); }

// library options: key 7 = tensor-core passes per product of the dense-layer and weight-gradient kernels: 3 = 3xTF32
// (fp32 parity, default), 1 = one TF32 pass (reduced-precision mode, set_gemm_precision("tf32"));
// key 10 = one-pass mode only: the dense layer reads its X operand straight from shared memory (SS form, gemm_tc2.cu;
// set_gemm_precision("bf16") turns it on); key 11 = compact spline transform: 1 = TMA-staged kernels of spline_stream.cu
// (default), 0 = first-version kernels (the bit-identical reference).  Any other key is refused.
namespace nf { extern int g_tc_passes; extern int g_gemm_tc2_ss; extern int g_spline_stream; }
extern "C" int nf_set_option(int key, int value) {
    if (key == 7) { if (value != 1 && value != 3) return NF_ERR_BAD_SHAPE; nf::g_tc_passes = value; return NF_OK; }
    if (key == 10) { nf::g_gemm_tc2_ss = value != 0; return NF_OK; }
    if (key == 11) { nf::g_spline_stream = value != 0; return NF_OK; }
    return NF_ERR_UNSUPPORTED;
}
