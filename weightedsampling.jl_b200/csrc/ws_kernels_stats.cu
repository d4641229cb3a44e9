// ws_kernels_stats.cu — device side of describe(state) (src/utils.jl:183-289): weighted mean / std / min / max,
// 8-bin weighted histogram and the weighted median of StatsBase.quantile(v, Weights(w), 0.5) for one plane.
//
// The reference sorts all (value, weight) pairs on the host.  Here the median is found by a radix SELECT
// over the order-preserving 64-bit image of the doubles: eight passes of 8 bits, each a weighted histogram
// of the keys that share the prefix chosen so far.  Weights are the resampler's 2^61 fixed-point integers,
// so the histogram sums are exact and the selected element does not depend on the summation order.
//   pass W   w_i = exp(l_i - m)/S -> fixed point q_i (once per describe call, shared by all planes)
//   pass 1   sum w x, min, max, NaN flag, (smallest value with non-zero weight, its smallest weight)
//   pass 2   sum w (x - mean)^2, histogram over [min, max]
//   8 x (histogram of the next key byte | pick the byte where the running mass first exceeds h)
//   pass F   neighbours of the selected value: largest smaller value, smallest weight at the value
// All of it is HBM streaming work: 8 (x) + 8 (q) bytes per particle and pass.
//
// The second half of the file is sample(state, n; replace) (src/utils.jl:102-118), the draw include/wsb200.h defines
// above ws_sample_indices.  It reuses the pick step of the radix select and the same cross-rank hooks.
#include <algorithm>
#include <vector>
#include <string.h>
#include "ws_internal.h"
#include "ws_stats.h"

static int g_stats_sms = 148;

__device__ __forceinline__ unsigned long long ws_key_of(double x) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(x);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double ws_value_of_key(unsigned long long k) {
    const unsigned long long b = (k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k;
    return __longlong_as_double((long long)b);
}

// ---- pass W: fixed-point weights ------------------------------------------------------------------
__global__ void __launch_bounds__(256) ws_stats_weights_kernel(const double* __restrict__ logw, const WsReduceOut* __restrict__ red,
                                                                int uniform, int64_t n, int64_t n_global,
                                                                unsigned long long* __restrict__ q) {
    double m = 0.0, S = 1.0;
    if (!uniform) {
        m = red->m;
        S = red->S;
    }
    const double rS = 1.0 / S;
    const double wu = 1.0 / (double)n_global;
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) {
        const double w = uniform ? wu : ws_div_pos(ws_exp_nonpos(logw[i] - m), S, rS);
        unsigned long long v = 0ull;
        if (w > 0.0) v = (w >= 1.0) ? (1ull << 61) : __double2ull_rn(w * 2305843009213693952.0);
        q[i] = v;
    }
}

// ---- pass 1 -------------------------------------------------------------------------------------------
struct WsStat1 {
    double swx, sw, mn, mx, minv_nz, minw_nz;
    int has_nan, pad;
};

__device__ __forceinline__ void stat1_merge(WsStat1& a, const WsStat1& b) {
    a.swx += b.swx;
    a.sw += b.sw;
    a.mn = fmin(a.mn, b.mn);
    a.mx = fmax(a.mx, b.mx);
    a.has_nan |= b.has_nan;
    if (b.minv_nz < a.minv_nz || (b.minv_nz == a.minv_nz && b.minw_nz < a.minw_nz)) {
        a.minv_nz = b.minv_nz;
        a.minw_nz = b.minw_nz;
    }
}

__global__ void __launch_bounds__(256) ws_stats_pass1_kernel(const double* __restrict__ x, const unsigned long long* __restrict__ q,
                                                              int64_t n, WsStat1* __restrict__ partials) {
    __shared__ WsStat1 sm[8];
    WsStat1 a;
    a.swx = 0.0;
    a.sw = 0.0;
    a.mn = INFINITY;
    a.mx = -INFINITY;
    a.minv_nz = INFINITY;
    a.minw_nz = INFINITY;
    a.has_nan = 0;
    a.pad = 0;
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) {
        const double v = x[i];
        const double w = (double)q[i] * (1.0 / 2305843009213693952.0);
        if (v != v) a.has_nan = 1;
        a.swx += w * v;
        a.sw += w;
        a.mn = fmin(a.mn, v);
        a.mx = fmax(a.mx, v);
        if (w > 0.0 && (v < a.minv_nz || (v == a.minv_nz && w < a.minw_nz))) {
            a.minv_nz = v;
            a.minw_nz = w;
        }
    }
    for (int d = 16; d > 0; d >>= 1) {
        WsStat1 b;
        b.swx = __shfl_down_sync(0xffffffffu, a.swx, d);
        b.sw = __shfl_down_sync(0xffffffffu, a.sw, d);
        b.mn = __shfl_down_sync(0xffffffffu, a.mn, d);
        b.mx = __shfl_down_sync(0xffffffffu, a.mx, d);
        b.minv_nz = __shfl_down_sync(0xffffffffu, a.minv_nz, d);
        b.minw_nz = __shfl_down_sync(0xffffffffu, a.minw_nz, d);
        b.has_nan = __shfl_down_sync(0xffffffffu, a.has_nan, d);
        stat1_merge(a, b);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) sm[warp] = a;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) stat1_merge(a, sm[w]);
        partials[blockIdx.x] = a;
    }
}

// ---- pass 2 -------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ws_stats_pass2_kernel(const double* __restrict__ x, const unsigned long long* __restrict__ q,
                                                              int64_t n, double mean, double lo, double hi,
                                                              double* __restrict__ partials /* [grid][1 + 8] */) {
    __shared__ double sm[8][9];
    double acc[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) acc[k] = 0.0;
    const double scale = (hi > lo) ? 8.0 / (hi - lo) : 0.0;
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) {
        const double v = x[i];
        const double w = (double)q[i] * (1.0 / 2305843009213693952.0);
        const double d = v - mean;
        acc[0] += w * d * d;
        int b = (int)((v - lo) * scale);  // clamp(searchsortedlast(range(lo, hi, 9), v), 1, 8) - 1
        b = b < 0 ? 0 : (b > 7 ? 7 : b);
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (k == b) acc[1 + k] += w;
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        double v = acc[k];
        for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
        if (lane == 0) sm[warp][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < 9) {
        double v = 0.0;
        for (int w = 0; w < 8; ++w) v += sm[w][threadIdx.x];
        partials[(size_t)blockIdx.x * 9 + threadIdx.x] = v;
    }
}

// ---- radix select -------------------------------------------------------------------------------------
// state[0] = key prefix chosen so far (left-aligned), state[1] = fixed-point mass of all keys below the
// prefix range, state[2] = h (the fixed-point mass the running sum has to exceed), state[3] = mass of the
// selected byte's bin (after the last pass: total mass of the selected value), state[4] = 1 if the mass
// never exceeds h (the answer is the maximum)
__global__ void __launch_bounds__(256) ws_stats_hist_kernel(const double* __restrict__ x, const unsigned long long* __restrict__ q,
                                                             int64_t n, int pass, const unsigned long long* __restrict__ state,
                                                             unsigned long long* __restrict__ hist /* [256] */) {
    __shared__ unsigned long long h[8][256];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int k = lane; k < 256; k += 32) h[warp][k] = 0ull;
    __syncwarp();
    const unsigned long long prefix = state[0];
    const int shift = 56 - 8 * pass;
    const unsigned long long himask = pass == 0 ? 0ull : (~0ull << (shift + 8));
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) {
        const unsigned long long key = ws_key_of(x[i]);
        const unsigned long long w = q[i];
        if ((key & himask) == prefix && w != 0ull) atomicAdd(&h[warp][(key >> shift) & 0xFFull], w);
    }
    __syncthreads();
    {
        unsigned long long s = 0ull;
        for (int w = 0; w < 8; ++w) s += h[w][threadIdx.x];
        if (s != 0ull) atomicAdd(hist + threadIdx.x, s);
    }
}

// the bin b where the running mass `below` + hist[0..b] first exceeds hh (-1: never); `below` is advanced to the mass
// of the bins before it and *mass gets the bin's own mass
__device__ __forceinline__ int ws_radix_pick(unsigned long long& below, unsigned long long hh, const unsigned long long* hist,
                                             unsigned long long* mass) {
    int pick = -1;
    for (int b = 0; b < 256; ++b) {
        const unsigned long long c = hist[b];
        if (pick < 0 && c != 0ull && below + c > hh) {
            pick = b;
            *mass = c;
        }
        if (pick < 0) below += c;
    }
    return pick;
}

__global__ void ws_stats_pick_kernel(int pass, unsigned long long* __restrict__ state, unsigned long long* __restrict__ hist) {
    if (threadIdx.x != 0) return;
    unsigned long long below = state[1];
    int pick = ws_radix_pick(below, state[2], hist, &state[3]);
    if (pick < 0) {
        state[4] = 1ull;  // the running mass never exceeds h: quantile() returns the maximum
        pick = 255;
    }
    state[0] |= (unsigned long long)pick << (56 - 8 * pass);
    state[1] = below;
    for (int b = 0; b < 256; ++b) hist[b] = 0ull;
}

// ---- pass F: neighbours of the selected value -----------------------------------------------------------
struct WsStatF {
    unsigned long long prev_key;  // largest key below the selected one among non-zero weights (0: none)
    unsigned long long minq_eq;   // smallest non-zero fixed-point weight at the selected value
};
__global__ void __launch_bounds__(256) ws_stats_final_kernel(const double* __restrict__ x, const unsigned long long* __restrict__ q,
                                                              int64_t n, const unsigned long long* __restrict__ state,
                                                              WsStatF* __restrict__ partials) {
    __shared__ WsStatF sm[8];
    const unsigned long long sel = state[0];
    unsigned long long pk = 0ull, mq = ~0ull;
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) {
        const unsigned long long w = q[i];
        if (w == 0ull) continue;
        const unsigned long long key = ws_key_of(x[i]);
        if (key < sel) pk = key > pk ? key : pk;
        else if (key == sel) mq = w < mq ? w : mq;
    }
    for (int d = 16; d > 0; d >>= 1) {
        const unsigned long long a = __shfl_down_sync(0xffffffffu, pk, d), b = __shfl_down_sync(0xffffffffu, mq, d);
        pk = a > pk ? a : pk;
        mq = b < mq ? b : mq;
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) {
        sm[warp].prev_key = pk;
        sm[warp].minq_eq = mq;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) {
            pk = sm[w].prev_key > pk ? sm[w].prev_key : pk;
            mq = sm[w].minq_eq < mq ? sm[w].minq_eq : mq;
        }
        partials[blockIdx.x].prev_key = pk;
        partials[blockIdx.x].minq_eq = mq;
    }
}

// ---- host-side driver (called by ws_describe in ws_runtime.cu) -------------------------------------------
static int stats_grid(int64_t n) {
    int64_t g = (n + 255) / 256;
    const int64_t cap = (int64_t)g_stats_sms * 8;
    if (g > cap) g = cap;
    return (int)(g < 1 ? 1 : g);
}

cudaError_t ws_stats_init(int device) {
    cudaDeviceProp prop;
    cudaError_t e = cudaGetDeviceProperties(&prop, device);
    if (e == cudaSuccess) g_stats_sms = prop.multiProcessorCount;
    return e;
}

cudaError_t ws_stats_weights(const double* logw, const WsReduceOut* red, int uniform, int64_t n, int64_t n_global,
                             unsigned long long* q, cudaStream_t s) {
    ws_stats_weights_kernel<<<stats_grid(n), 256, 0, s>>>(logw, red, uniform, n, n_global, q);
    return cudaGetLastError();
}

// scratch: device buffer of at least ws_stats_scratch_bytes(n); h_scratch: pinned host buffer of the same size
size_t ws_stats_scratch_bytes(int64_t n) {
    const size_t g = (size_t)stats_grid(n);
    return g * sizeof(WsStat1) + g * 9 * sizeof(double) + g * sizeof(WsStatF) + 256 * 8 + 8 * 8 + 256;
}

static void stat1_merge_host(WsStat1& a, const WsStat1& b) {
    a.swx += b.swx;
    a.sw += b.sw;
    a.mn = fmin(a.mn, b.mn);
    a.mx = fmax(a.mx, b.mx);
    a.has_nan |= b.has_nan;
    if (b.minv_nz < a.minv_nz || (b.minv_nz == a.minv_nz && b.minw_nz < a.minw_nz)) {
        a.minv_nz = b.minv_nz;
        a.minw_nz = b.minw_nz;
    }
}

cudaError_t ws_stats_plane(const double* x, const unsigned long long* q, int64_t n, void* d_scratch, void* h_scratch,
                           cudaStream_t s, WsPlaneStats* out, int* n_launches, const WsStatsComm* comm) {
    static_assert(sizeof(WsStat1) % 8 == 0, "WsStat1 travels as 64-bit words");
    const int g = stats_grid(n);
    char* dp = (char*)d_scratch;
    char* hp = (char*)h_scratch;
    WsStat1* d1 = (WsStat1*)dp;
    double* d2 = (double*)(dp + (size_t)g * sizeof(WsStat1));
    WsStatF* dF = (WsStatF*)((char*)d2 + (size_t)g * 9 * sizeof(double));
    unsigned long long* d_hist = (unsigned long long*)((char*)dF + (size_t)g * sizeof(WsStatF));
    unsigned long long* d_state = d_hist + 256;
    WsStat1* h1 = (WsStat1*)hp;
    double* h2 = (double*)(hp + (size_t)g * sizeof(WsStat1));
    WsStatF* hF = (WsStatF*)((char*)h2 + (size_t)g * 9 * sizeof(double));
    unsigned long long* h_state = (unsigned long long*)((char*)hF + (size_t)g * sizeof(WsStatF)) + 256;
    cudaError_t e;
    const double FX = 2305843009213693952.0;

    ws_stats_pass1_kernel<<<g, 256, 0, s>>>(x, q, n, d1);
    if ((e = cudaMemcpyAsync(h1, d1, sizeof(WsStat1) * g, cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return e;
    WsStat1 a = h1[0];
    for (int k = 1; k < g; ++k) stat1_merge_host(a, h1[k]);
    if (comm != nullptr) {  // shard partials -> global, merged in rank order on every rank
        const size_t words = sizeof(WsStat1) / 8;
        std::vector<unsigned long long> all(words * (size_t)comm->nranks);
        if (comm->allgather_words(comm->ctx, reinterpret_cast<const unsigned long long*>(&a), words, all.data()) != 0) return cudaErrorUnknown;
        memcpy(&a, all.data(), sizeof(WsStat1));
        for (int r = 1; r < comm->nranks; ++r) {
            WsStat1 b;
            memcpy(&b, all.data() + words * (size_t)r, sizeof(WsStat1));
            stat1_merge_host(a, b);
        }
    }
    *n_launches = 1;
    out->min = a.mn;
    out->max = a.mx;
    out->mean = a.swx / a.sw;
    if (a.has_nan) {
        out->min = out->max = out->mean = out->std = out->median = NAN;
        for (int k = 0; k < 8; ++k) out->hist[k] = NAN;
        return cudaSuccess;
    }

    ws_stats_pass2_kernel<<<g, 256, 0, s>>>(x, q, n, out->mean, a.mn, a.mx, d2);
    if ((e = cudaMemcpyAsync(h2, d2, sizeof(double) * 9 * g, cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;

    // weighted median: StatsBase.quantile(v, Weights(w), 0.5): h = p (wsum - w1) + w1, first k with S_k > h
    const double h = 0.5 * (a.sw - a.minw_nz) + a.minw_nz;
    unsigned long long st0[8] = {0ull, 0ull, (unsigned long long)floor(h * FX), 0ull, 0ull, 0ull, 0ull, 0ull};
    if ((e = cudaMemcpyAsync(d_state, st0, sizeof(st0), cudaMemcpyHostToDevice, s)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(d_hist, 0, 256 * 8, s)) != cudaSuccess) return e;
    for (int pass = 0; pass < 8; ++pass) {
        ws_stats_hist_kernel<<<g, 256, 0, s>>>(x, q, n, pass, d_state, d_hist);
        if (comm != nullptr && comm->allreduce_u64_device(comm->ctx, d_hist, 256) != 0) return cudaErrorUnknown;  // exact integer sums
        ws_stats_pick_kernel<<<1, 32, 0, s>>>(pass, d_state, d_hist);
    }
    ws_stats_final_kernel<<<g, 256, 0, s>>>(x, q, n, d_state, dF);
    if ((e = cudaMemcpyAsync(hF, dF, sizeof(WsStatF) * g, cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(h_state, d_state, 8 * 8, cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return e;
    *n_launches += 1 + 16 + 1;

    double ss = 0.0;
    for (int k = 0; k < 8; ++k) out->hist[k] = 0.0;
    for (int b = 0; b < g; ++b) {
        ss += h2[(size_t)b * 9];
        for (int k = 0; k < 8; ++k) out->hist[k] += h2[(size_t)b * 9 + 1 + k];
    }
    if (comm != nullptr) {
        double v[9] = {ss};
        for (int k = 0; k < 8; ++k) v[1 + k] = out->hist[k];
        if (comm->allreduce_doubles(comm->ctx, v, 9) != 0) return cudaErrorUnknown;
        ss = v[0];
        for (int k = 0; k < 8; ++k) out->hist[k] = v[1 + k];
    }
    out->std = sqrt(ss / a.sw);

    unsigned long long pk = 0ull, mq = ~0ull;
    for (int b = 0; b < g; ++b) {
        pk = hF[b].prev_key > pk ? hF[b].prev_key : pk;
        mq = hF[b].minq_eq < mq ? hF[b].minq_eq : mq;
    }
    if (comm != nullptr) {
        const unsigned long long mine[2] = {pk, mq};
        std::vector<unsigned long long> all(2 * (size_t)comm->nranks);
        if (comm->allgather_words(comm->ctx, mine, 2, all.data()) != 0) return cudaErrorUnknown;
        for (int r = 0; r < comm->nranks; ++r) {
            pk = all[2 * r] > pk ? all[2 * r] : pk;
            mq = all[2 * r + 1] < mq ? all[2 * r + 1] : mq;
        }
    }
    const unsigned long long sel = h_state[0], below = h_state[1];
    auto val = [](unsigned long long k) {
        const unsigned long long b = (k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k;
        double v;
        memcpy(&v, &b, 8);
        return v;
    };
    const double vsel = val(sel);
    if (h_state[4] != 0ull) {
        out->median = a.mx;  // "out was initialized with maximum v"
    } else if (pk != 0ull && mq != ~0ull && below + mq > h_state[2]) {
        // the running mass crosses h at the FIRST element of the selected value's group: interpolate from the
        // previous element,  v_{k-1} + (h - S_{k-1}) / (S_k - S_{k-1}) (v_k - v_{k-1})
        const double Skold = (double)below / FX, wk = (double)mq / FX, vprev = val(pk);
        out->median = vprev + (h - Skold) / wk * (vsel - vprev);
    } else {
        out->median = vsel;
    }
    return cudaSuccess;
}

// =========================================================================================================
// sample(state, n; replace) on the device
//
// With replacement (exact inversion of the integer CDF of q_i = ws_sample_q(l_i, m)):
//   ws_sample_cdf_tiles_kernel   q -> tile-local inclusive prefix P (8 B per particle) and one sum per tile of 2048
//   ws_sample_offsets_kernel     one CTA: exclusive 128-bit scan of the tile sums, the shard's mass T_r at the end
//   ws_sample_draw_kernel        one thread per draw: Philox -> t_k; skip unless t_k falls in [O_r, O_r + T_r);
//                                binary search over the tile offsets, then inside the tile -> global index + 1
//   sharded: the T_r travel with one allgather, the draws with one integer all-reduce (each draw has one owner)
// Without replacement (the n largest Gumbel keys, ties to the lower global index):
//   ws_sample_keys_kernel        64-bit key image per particle
//   8 x (ws_sample_hist_kernel | ws_sample_pick_kernel)   radix select over COUNT histograms: the n-th largest key
//   4 x (the same over the index bytes of the particles at that key)  the lowest-index ones taken at a tie
//   ws_sample_compact_kernel     the n winners (key, global index); the host sorts them (n log n, n << N)
// Every count and mass is an integer, so the result does not depend on the grid or on the number of ranks.
// =========================================================================================================
#define WS_SMP_TILE 2048      // particles per CDF tile: a tile sum <= 2048 (2^52 + 1) stays below 2^63
#define WS_SMP_PER_THREAD 8   // consecutive particles per thread (256 threads)
typedef unsigned __int128 ws_smp_u128;

__global__ void __launch_bounds__(256) ws_sample_cdf_tiles_kernel(const double* __restrict__ logw, int64_t n, double m,
                                                                   unsigned long long* __restrict__ P,
                                                                   unsigned long long* __restrict__ tile_sum) {
    __shared__ unsigned long long warp_tot[8];
    const int64_t base = (int64_t)blockIdx.x * WS_SMP_TILE + (int64_t)threadIdx.x * WS_SMP_PER_THREAD;
    unsigned long long pre[WS_SMP_PER_THREAD];
    unsigned long long s = 0ull;
#pragma unroll
    for (int j = 0; j < WS_SMP_PER_THREAD; ++j) {
        const int64_t i = base + j;
        s += i < n ? ws_sample_q(logw[i], m) : 0ull;
        pre[j] = s;
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long x = s;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= d) x += y;
    }
    if (lane == 31) warp_tot[warp] = x;
    __syncthreads();
    unsigned long long before = x - s;
    for (int w = 0; w < warp; ++w) before += warp_tot[w];
#pragma unroll
    for (int j = 0; j < WS_SMP_PER_THREAD; ++j)
        if (base + j < n) P[base + j] = before + pre[j];
    if (threadIdx.x == 255) tile_sum[blockIdx.x] = before + s;
}

// off[b] = sum of the tile sums before b (128-bit), off[n_tiles] = the shard's total T_r
__global__ void __launch_bounds__(1024) ws_sample_offsets_kernel(const unsigned long long* __restrict__ tile_sum, int64_t n_tiles,
                                                                  ws_smp_u128* __restrict__ off) {
    __shared__ ws_smp_u128 sm[1024];
    const int t = threadIdx.x;
    const int64_t per = (n_tiles + 1023) / 1024;
    const int64_t b0 = (int64_t)t * per, b1 = b0 + per < n_tiles ? b0 + per : n_tiles;
    ws_smp_u128 s = 0;
    for (int64_t b = b0; b < b1; ++b) s += tile_sum[b];
    sm[t] = s;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
        const ws_smp_u128 v = t >= d ? sm[t - d] : (ws_smp_u128)0;
        __syncthreads();
        sm[t] += v;
        __syncthreads();
    }
    ws_smp_u128 run = sm[t] - s;
    for (int64_t b = b0; b < b1; ++b) {
        off[b] = run;
        run += tile_sum[b];
    }
    if (t == 1023) off[n_tiles] = sm[1023];
}

__global__ void __launch_bounds__(256) ws_sample_draw_kernel(const unsigned long long* __restrict__ P, const ws_smp_u128* __restrict__ off,
                                                              int64_t n_tiles, int64_t n, int64_t offset, ws_u128 T, ws_u128 O,
                                                              int64_t n_draws, uint64_t stream, uint64_t seed,
                                                              unsigned long long* __restrict__ out) {
    const int64_t k = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (k >= n_draws) return;
    const ws_u128 t = ws_sample_target((uint64_t)k, stream, seed, T);
    const ws_smp_u128 tt = ((ws_smp_u128)t.hi << 64) | t.lo, o = ((ws_smp_u128)O.hi << 64) | O.lo;
    if (tt < o || tt - o >= off[n_tiles]) {  // another rank's particle
        out[k] = 0ull;
        return;
    }
    const ws_smp_u128 loc = tt - o;
    int64_t lo = 0, hi = n_tiles - 1;  // the last tile whose offset is <= loc (it has a non-zero sum)
    while (lo < hi) {
        const int64_t mid = (lo + hi + 1) >> 1;
        if (off[mid] <= loc) lo = mid; else hi = mid - 1;
    }
    const unsigned long long w = (unsigned long long)(loc - off[lo]);
    int64_t a = lo * WS_SMP_TILE, e = (a + WS_SMP_TILE < n ? a + WS_SMP_TILE : n) - 1;  // the first j with P[j] > w
    while (a < e) {
        const int64_t mid = (a + e) >> 1;
        if (P[mid] > w) e = mid; else a = mid + 1;
    }
    out[k] = (unsigned long long)(offset + a + 1);
}

__global__ void __launch_bounds__(256) ws_sample_keys_kernel(const double* __restrict__ logw, int64_t n, int64_t offset, uint64_t stream,
                                                              uint64_t seed, unsigned long long* __restrict__ keys) {
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += stride)
        keys[i] = ws_sample_key(logw[i], (uint64_t)(offset + i), stream, seed);
}

// state: [0] key prefix (left-aligned; after pass 7 the selected key), [1] count below the prefix range, [2] the rank h
// to select (ascending), [3] count in the selected bin, [5] index prefix (passes 8..11), [6] 1: every particle at the
// selected key is taken (the index passes are skipped), [7] 1: a histogram never crossed h (cannot happen)
#define WS_SMP_KEY_PASSES 8
#define WS_SMP_PASSES 12   // + 4 bytes of the global index (N < 2^31)
__global__ void __launch_bounds__(256) ws_sample_hist_kernel(const unsigned long long* __restrict__ keys, int64_t n, int64_t offset, int pass,
                                                              const unsigned long long* __restrict__ state,
                                                              unsigned long long* __restrict__ hist /* [256] */) {
    __shared__ unsigned int h[8][256];
    if (pass >= WS_SMP_KEY_PASSES && state[6] != 0ull) return;
    for (int k = threadIdx.x; k < 8 * 256; k += 256) (&h[0][0])[k] = 0u;
    __syncthreads();
    const int warp = threadIdx.x >> 5;
    const int64_t stride = (int64_t)gridDim.x * 256;
    if (pass < WS_SMP_KEY_PASSES) {
        const unsigned long long prefix = state[0];
        const int shift = 56 - 8 * pass;
        const unsigned long long himask = pass == 0 ? 0ull : (~0ull << (shift + 8));
        for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) {
            const unsigned long long key = keys[i];
            if ((key & himask) == prefix) atomicAdd(&h[warp][(key >> shift) & 0xFFull], 1u);
        }
    } else {
        const unsigned long long sel = state[0], prefix = state[5];
        const int shift = 24 - 8 * (pass - WS_SMP_KEY_PASSES);
        const unsigned long long himask = ~0ull << (shift + 8);
        for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) {
            if (keys[i] != sel) continue;
            const unsigned long long g = (unsigned long long)(offset + i);
            if ((g & himask) == prefix) atomicAdd(&h[warp][(g >> shift) & 0xFFull], 1u);
        }
    }
    __syncthreads();
    unsigned long long s = 0ull;
    for (int w = 0; w < 8; ++w) s += h[w][threadIdx.x];
    if (s != 0ull) atomicAdd(hist + threadIdx.x, s);
}

__global__ void ws_sample_pick_kernel(int pass, unsigned long long* __restrict__ state, unsigned long long* __restrict__ hist) {
    if (threadIdx.x != 0) return;
    if (pass >= WS_SMP_KEY_PASSES && state[6] != 0ull) return;  // nothing was counted
    unsigned long long below = state[1], mass = 0ull;
    int pick = ws_radix_pick(below, state[2], hist, &mass);
    if (pick < 0) {  // the counts sum to the number of candidates, which always exceeds h
        state[7] = 1ull;
        pick = 0;
    }
    if (pass < WS_SMP_KEY_PASSES) {
        state[0] |= (unsigned long long)pick << (56 - 8 * pass);
        state[1] = below;
        state[3] = mass;
        if (pass == WS_SMP_KEY_PASSES - 1) {
            // the particles at the selected key hold ascending ranks [below, below + mass); ranks >= h are taken
            const unsigned long long h = state[2];
            if (below == h) {
                state[6] = 1ull;
            } else {  // take the (below + mass - h) lowest global indices among them: select the last one
                state[2] = below + mass - h - 1ull;
                state[1] = 0ull;
            }
        }
    } else {
        state[5] |= (unsigned long long)pick << (24 - 8 * (pass - WS_SMP_KEY_PASSES));
        state[1] = below;
    }
    for (int b = 0; b < 256; ++b) hist[b] = 0ull;
}

__global__ void __launch_bounds__(256) ws_sample_compact_kernel(const unsigned long long* __restrict__ keys, int64_t n, int64_t offset,
                                                                 const unsigned long long* __restrict__ state,
                                                                 unsigned long long* __restrict__ count,
                                                                 unsigned long long* __restrict__ pairs, int64_t cap) {
    const unsigned long long sel = state[0], gmax = state[6] != 0ull ? ~0ull : state[5];
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) {
        const unsigned long long key = keys[i], g = (unsigned long long)(offset + i);
        if (key > sel || (key == sel && g <= gmax)) {
            const unsigned long long pos = atomicAdd(count, 1ull);
            if (pos < (unsigned long long)cap) {
                pairs[2 * pos] = key;
                pairs[2 * pos + 1] = g;
            }
        }
    }
}

__global__ void __launch_bounds__(256) ws_sample_scatter_kernel(const double* __restrict__ src, const int64_t* __restrict__ pos, int64_t n,
                                                                 double* __restrict__ dst) {
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (j < n) dst[pos[j]] = src[j];
}

static size_t smp_up(size_t b) { return (b + 255) & ~(size_t)255; }
static int64_t smp_tiles(int64_t n) { return (n + WS_SMP_TILE - 1) / WS_SMP_TILE; }

size_t ws_sample_scratch_bytes(int64_t n, int64_t n_draws, int replace) {
    const int64_t t = smp_tiles(n);
    if (replace)
        return smp_up(8 * (size_t)n) + smp_up(8 * (size_t)t) + smp_up(16 * (size_t)(t + 1)) + smp_up(8 * (size_t)n_draws);
    return smp_up(8 * (size_t)n) + smp_up(8 * 256) + smp_up(8 * 8) + smp_up(8) + smp_up(16 * (size_t)n_draws);
}

static cudaError_t sample_with_replacement(const double* logw, int64_t n, int64_t offset, double m, uint64_t seed, uint64_t stream,
                                           int64_t n_draws, char* dp, cudaStream_t s, int64_t* out, int* n_launches,
                                           int64_t* d2h_bytes, const WsStatsComm* comm) {
    const int64_t tiles = smp_tiles(n);
    unsigned long long* P = (unsigned long long*)dp;
    unsigned long long* tsum = (unsigned long long*)(dp + smp_up(8 * (size_t)n));
    ws_smp_u128* off = (ws_smp_u128*)((char*)tsum + smp_up(8 * (size_t)tiles));
    unsigned long long* d_out = (unsigned long long*)((char*)off + smp_up(16 * (size_t)(tiles + 1)));
    cudaError_t e;
    ws_sample_cdf_tiles_kernel<<<(unsigned)tiles, 256, 0, s>>>(logw, n, m, P, tsum);
    ws_sample_offsets_kernel<<<1, 1024, 0, s>>>(tsum, tiles, off);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    ws_smp_u128 Tr = 0;
    if ((e = cudaMemcpyAsync(&Tr, off + tiles, 16, cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return e;
    *d2h_bytes += 16;
    ws_smp_u128 O = 0, T = Tr;
    if (comm != nullptr) {  // the ranks' masses in rank order: this rank's draws are the t in [O, O + T_r)
        const unsigned long long mine[2] = {(unsigned long long)(Tr >> 64), (unsigned long long)Tr};
        std::vector<unsigned long long> all(2 * (size_t)comm->nranks);
        if (comm->allgather_words(comm->ctx, mine, 2, all.data()) != 0) return cudaErrorUnknown;
        *d2h_bytes += 16 * comm->nranks;
        T = 0;
        for (int r = 0; r < comm->nranks; ++r) {
            const ws_smp_u128 v = ((ws_smp_u128)all[2 * r] << 64) | all[2 * r + 1];
            if (r < comm->rank) O += v;
            T += v;
        }
    }
    ws_u128 T2, O2;
    T2.hi = (uint64_t)(T >> 64);
    T2.lo = (uint64_t)T;
    O2.hi = (uint64_t)(O >> 64);
    O2.lo = (uint64_t)O;
    ws_sample_draw_kernel<<<(unsigned)((n_draws + 255) / 256), 256, 0, s>>>(P, off, tiles, n, offset, T2, O2, n_draws, stream, seed, d_out);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    *n_launches += 3;
    if (comm != nullptr && comm->allreduce_u64_device(comm->ctx, d_out, (size_t)n_draws) != 0) return cudaErrorUnknown;
    if ((e = cudaMemcpyAsync(out, d_out, 8 * (size_t)n_draws, cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return e;
    *d2h_bytes += 8 * n_draws;
    for (int64_t k = 0; k < n_draws; ++k) {
        if (out[k] <= 0) return cudaErrorInvalidValue;  // no rank owned the draw
        out[k] -= 1;
    }
    return cudaSuccess;
}

static cudaError_t sample_without_replacement(const double* logw, int64_t n, int64_t offset, int64_t n_global, uint64_t seed,
                                              uint64_t stream, int64_t n_draws, char* dp, cudaStream_t s, int64_t* out,
                                              int* n_launches, int64_t* d2h_bytes, const WsStatsComm* comm) {
    unsigned long long* keys = (unsigned long long*)dp;
    unsigned long long* d_hist = (unsigned long long*)(dp + smp_up(8 * (size_t)n));
    unsigned long long* d_state = (unsigned long long*)((char*)d_hist + smp_up(8 * 256));
    unsigned long long* d_count = (unsigned long long*)((char*)d_state + smp_up(8 * 8));
    unsigned long long* d_pairs = (unsigned long long*)((char*)d_count + smp_up(8));
    const int g = stats_grid(n);
    cudaError_t e;
    ws_sample_keys_kernel<<<g, 256, 0, s>>>(logw, n, offset, stream, seed, keys);
    const unsigned long long st0[8] = {0ull, 0ull, (unsigned long long)(n_global - n_draws), 0ull, 0ull, 0ull, 0ull, 0ull};
    if ((e = cudaMemcpyAsync(d_state, st0, sizeof(st0), cudaMemcpyHostToDevice, s)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(d_hist, 0, 8 * 256, s)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(d_count, 0, 8, s)) != cudaSuccess) return e;
    for (int pass = 0; pass < WS_SMP_PASSES; ++pass) {
        ws_sample_hist_kernel<<<g, 256, 0, s>>>(keys, n, offset, pass, d_state, d_hist);
        if (comm != nullptr && comm->allreduce_u64_device(comm->ctx, d_hist, 256) != 0) return cudaErrorUnknown;  // exact counts
        ws_sample_pick_kernel<<<1, 32, 0, s>>>(pass, d_state, d_hist);
    }
    ws_sample_compact_kernel<<<g, 256, 0, s>>>(keys, n, offset, d_state, d_count, d_pairs, n_draws);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    *n_launches += 2 + 2 * WS_SMP_PASSES;
    unsigned long long h_state[8], cnt = 0ull;
    if ((e = cudaMemcpyAsync(h_state, d_state, sizeof(h_state), cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(&cnt, d_count, 8, cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return e;
    *d2h_bytes += sizeof(h_state) + 8;
    if (h_state[7] != 0ull || cnt > (unsigned long long)n_draws) return cudaErrorInvalidValue;
    std::vector<unsigned long long> pairs(2 * (size_t)cnt);
    if (cnt > 0ull) {
        if ((e = cudaMemcpyAsync(pairs.data(), d_pairs, 16 * (size_t)cnt, cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
        if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return e;
        *d2h_bytes += 16 * (int64_t)cnt;
    }
    if (comm != nullptr) {  // every rank's winners, in rank order
        std::vector<unsigned long long> counts((size_t)comm->nranks);
        if (comm->allgather_words(comm->ctx, &cnt, 1, counts.data()) != 0) return cudaErrorUnknown;
        const unsigned long long mx = *std::max_element(counts.begin(), counts.end());
        std::vector<unsigned long long> mine(2 * (size_t)mx, 0ull), all(2 * (size_t)mx * comm->nranks);
        std::copy(pairs.begin(), pairs.end(), mine.begin());
        if (mx > 0ull && comm->allgather_words(comm->ctx, mine.data(), 2 * (size_t)mx, all.data()) != 0) return cudaErrorUnknown;
        *d2h_bytes += 8 * comm->nranks * (1 + 2 * (int64_t)mx);
        pairs.clear();
        for (int r = 0; r < comm->nranks; ++r)
            pairs.insert(pairs.end(), all.begin() + 2 * (size_t)mx * r, all.begin() + 2 * (size_t)mx * r + 2 * (size_t)counts[r]);
    }
    if ((int64_t)(pairs.size() / 2) != n_draws) return cudaErrorInvalidValue;
    std::vector<std::pair<unsigned long long, unsigned long long>> kv((size_t)n_draws);
    for (int64_t k = 0; k < n_draws; ++k) kv[(size_t)k] = {pairs[2 * (size_t)k], pairs[2 * (size_t)k + 1]};
    std::sort(kv.begin(), kv.end(), [](const std::pair<unsigned long long, unsigned long long>& a,
                                       const std::pair<unsigned long long, unsigned long long>& b) {
        return a.first != b.first ? a.first > b.first : a.second < b.second;  // descending key, then lower index
    });
    for (int64_t k = 0; k < n_draws; ++k) out[k] = (int64_t)kv[(size_t)k].second;
    return cudaSuccess;
}

cudaError_t ws_sample_draw(const double* logw, int64_t n, int64_t offset, int64_t n_global, double m, uint64_t seed, uint64_t stream,
                           int64_t n_draws, int replace, void* d_scratch, cudaStream_t s, int64_t* out, int* n_launches,
                           int64_t* d2h_bytes, const WsStatsComm* comm) {
    *n_launches = 0;
    if (replace)
        return sample_with_replacement(logw, n, offset, m, seed, stream, n_draws, (char*)d_scratch, s, out, n_launches, d2h_bytes, comm);
    return sample_without_replacement(logw, n, offset, n_global, seed, stream, n_draws, (char*)d_scratch, s, out, n_launches, d2h_bytes,
                                      comm);
}

cudaError_t ws_sample_scatter_rows(const double* src, const int64_t* pos, int64_t n, double* dst, cudaStream_t s) {
    ws_sample_scatter_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, pos, n, dst);
    return cudaGetLastError();
}
