// ws_stats.h — describe(state) on the device (ws_kernels_stats.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "ws_internal.h"

struct WsPlaneStats {
    double mean, median, std, min, max;
    double hist[8];
};

cudaError_t ws_stats_init(int device);
// q[i] = rint(w_i 2^61), w = exp_norm(logw) (or 1/N when the log-weights are uniform)
cudaError_t ws_stats_weights(const double* logw, const WsReduceOut* red, int uniform, int64_t n, int64_t n_global,
                             unsigned long long* q, cudaStream_t s);
size_t ws_stats_scratch_bytes(int64_t n);
// Cross-rank hooks of describe on a sharded state (nullptr: one GPU).  The statistics are sums / minima / maxima of
// per-shard partials and the median's radix select works on histograms, so a sharded describe is the single-GPU
// algorithm with these three reductions in between; every rank ends with the same numbers.
struct WsStatsComm {
    void* ctx;
    int nranks;
    int (*allgather_words)(void* ctx, const unsigned long long* in, size_t words, unsigned long long* out);  // host -> host, rank order
    int (*allreduce_doubles)(void* ctx, double* v, int n);                      // sum, in place, host
    int (*allreduce_u64_device)(void* ctx, unsigned long long* d, size_t n);    // sum, in place, device buffer, stream-ordered
    int rank;
};
cudaError_t ws_stats_plane(const double* x, const unsigned long long* q, int64_t n, void* d_scratch, void* h_scratch,
                           cudaStream_t s, WsPlaneStats* out, int* n_launches, const WsStatsComm* comm = nullptr);

// sample(state, n; replace): the n_draws 0-based GLOBAL indices of the draw include/wsb200.h defines (collective on a
// sharded state: every rank gets the same indices).  m = the global maximum log-weight (finite); d_scratch holds
// ws_sample_scratch_bytes(n, n_draws, replace).  Only the draws (8 B each, 16 without replacement) come to the host.
size_t ws_sample_scratch_bytes(int64_t n, int64_t n_draws, int replace);
cudaError_t ws_sample_draw(const double* logw, int64_t n, int64_t offset, int64_t n_global, double m, uint64_t seed, uint64_t stream,
                           int64_t n_draws, int replace, void* d_scratch, cudaStream_t s, int64_t* out, int* n_launches,
                           int64_t* d2h_bytes, const WsStatsComm* comm = nullptr);
// dst[pos[j]] = src[j] for j < n
cudaError_t ws_sample_scatter_rows(const double* src, const int64_t* pos, int64_t n, double* dst, cudaStream_t s);

// multinomial resampling: sorted iid uniforms (Philox draws when `in` is nullptr)

