// Host build of csrc/nf_rng.cuh for tests/test_hostcheck_rng.py (g++, no CUDA).
#include "nf_rng.cuh"

extern "C" {

// n counter / key sets -> n x 4 outputs
void hc_philox(const uint32_t* ctr, const uint32_t* key, uint32_t* out, long n) {
    for (long i = 0; i < n; ++i) {
        uint32_t c[4] = {ctr[4 * i], ctr[4 * i + 1], ctr[4 * i + 2], ctr[4 * i + 3]};
        nf::nf_philox4x32_10(c, key[2 * i], key[2 * i + 1]);
        for (int k = 0; k < 4; ++k) out[4 * i + k] = c[k];
    }
}

// n pairs of 32-bit words -> n pairs of normals
void hc_box_muller(const uint32_t* u, float* z, long n) {
    for (long i = 0; i < n; ++i) nf::nf_box_muller(u[2 * i], u[2 * i + 1], z[2 * i], z[2 * i + 1]);
}

// rows [0, B) of the draw at (seed, offset), D <= 8; lp[b] = log N(z_b; 0, I)
void hc_std_normal_rows(uint64_t seed, uint64_t offset, long B, int D, float* z, float* lp) {
    for (long r = 0; r < B; ++r) {
        float row[8];
        lp[r] = nf::nf_std_normal_row<8>(seed, offset, (uint32_t)r, D, row);
        for (int d = 0; d < D; ++d) z[r * D + d] = row[d];
    }
}
}
