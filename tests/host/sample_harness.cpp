// tests/host/sample_harness.cpp — host instantiation of the sample(state, n; replace) pieces of csrc/ws_math.cuh
// (ws_sample_q / ws_sample_target / ws_sample_key), TEST INFRASTRUCTURE ONLY.  The same source the device kernels
// compile, built here with g++, so tests/sample_spec.py regenerates the device's integer weights and keys bit for bit.
#include <stdint.h>
#include "../../weightedsampling.jl_b200/csrc/ws_math.cuh"

extern "C" {

void hh_sample_q(const double* logw, int64_t n, double m, uint64_t* out) {
    for (int64_t i = 0; i < n; ++i) out[i] = ws_sample_q(logw[i], m);
}
void hh_sample_targets(int64_t n_draws, uint64_t stream, uint64_t seed, uint64_t T_hi, uint64_t T_lo, uint64_t* out_hi_lo) {
    const ws_u128 T{T_hi, T_lo};
    for (int64_t k = 0; k < n_draws; ++k) {
        const ws_u128 t = ws_sample_target((uint64_t)k, stream, seed, T);
        out_hi_lo[2 * k] = t.hi;
        out_hi_lo[2 * k + 1] = t.lo;
    }
}
void hh_sample_keys(const double* logw, int64_t n, uint64_t first, uint64_t stream, uint64_t seed, uint64_t* out) {
    for (int64_t i = 0; i < n; ++i) out[i] = ws_sample_key(logw[i], first + (uint64_t)i, stream, seed);
}

}  // extern "C"
