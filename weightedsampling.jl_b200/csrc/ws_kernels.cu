// ws_kernels.cu — hand-written sm_100a kernels of the particle hot path.
//
//   ws_vm_kernel          fused elementwise window (Assign / Sample / Observe / Weight) with the
//                         (m, S, Q) log-weight reduction folded into its epilogue
//   ws_reduce_logw_kernel stand-alone (m, S, Q) partials (after an upload)
//   ws_finalize_kernel    combines partials -> logsumexp, ESS%, resample decision
//   ws_cdf_tiles_kernel   w = exp_norm(logw) in 2^61 fixed point, tile-local inclusive prefix sums
//   ws_cdf_offsets_kernel exclusive scan of the tile aggregates (one CTA)
//   ws_search_kernel      per-particle slot counts F(C) on the stratified / systematic grid, offspring
//                         expansion (ws_expand_heavy_kernel for one-hot weights), ancestors out
//   ws_gather_kernel      ancestor gather of all planes (resample!)
//   sharded states        ws_finalize_mbox_kernel, ws_offsets_bounds_mbox_kernel, ws_barrier_mbox_kernel: the small exchanges
//                         of a step made by the kernels through peer-mapped mailboxes (ws_mailbox.cuh);
//                         ws_trace_rows_kernel, ws_push_traced_kernel: migrating offspring of planes that are behind
//   small helpers         fill, exp_norm write, row gather, ancestor compose
//
// None of these is a dense contraction: they are HBM-bound streaming kernels (and FP64-ALU work
// for exp / log / Philox), so the design rules are coalescing, enough bytes in flight per SM and
// persistent grids sized in multiples of the SM count.  Tensor cores are not used.
#include "ws_internal.h"

static int g_sm_count = 148;

// ------------------------------------------------------------------------------------------
// (m, S, Q) helpers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void lse_push(WsLse& a, double l) {
    if (l == -INFINITY) return;  // contributes exp(-inf) = 0
    if (l > a.m) {
        double sc = ws_exp_nonpos(a.m - l);  // a.m == -inf -> 0
        a.S = a.S * sc + 1.0;
        a.Q = a.Q * sc * sc + 1.0;
        a.m = l;
    } else {
        double e = ws_exp_nonpos(l - a.m);
        a.S += e;
        a.Q += e * e;
    }
}

// K values at once: raise the running maximum first (one rescale, rarely taken once a thread has seen a
// few tiles), then K independent exps.  `skip[j]` marks values that do not exist (tail of the last tile).
template <int K>
__device__ __forceinline__ void lse_push_many(WsLse& a, const double (&l)[K], const bool (&live)[K]) {
    double mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < K; ++j)
        if (live[j]) mx = fmax(mx, l[j]);  // fmax drops NaN here; the NaN still reaches S below
    if (mx > a.m) {
        const double sc = ws_exp_nonpos(a.m - mx);  // a.m == -inf -> 0
        a.S *= sc;
        a.Q *= sc * sc;
        a.m = mx;
    }
#pragma unroll
    for (int j = 0; j < K; ++j) {
        if (live[j] && l[j] != -INFINITY) {
            const double e = ws_exp_nonpos(l[j] - a.m);
            a.S += e;
            a.Q += e * e;
        }
    }
}

__device__ __forceinline__ WsLse lse_combine(const WsLse& a, const WsLse& b) {
    if (b.m == -INFINITY) return a;
    if (a.m == -INFINITY) return b;
    WsLse r;
    r.m = fmax(a.m, b.m);
    double ea = ws_exp_nonpos(a.m - r.m), eb = ws_exp_nonpos(b.m - r.m);
    r.S = a.S * ea + b.S * eb;
    r.Q = a.Q * ea * ea + b.Q * eb * eb;
    return r;
}

__device__ __forceinline__ WsLse lse_shfl_down(const WsLse& a, int delta) {
    WsLse r;
    r.m = __shfl_down_sync(0xffffffffu, a.m, delta);
    r.S = __shfl_down_sync(0xffffffffu, a.S, delta);
    r.Q = __shfl_down_sync(0xffffffffu, a.Q, delta);
    return r;
}

// Block-wide combine in a fixed (deterministic) order; result valid in thread 0.
template <int BLOCK>
__device__ __forceinline__ WsLse lse_block_reduce(WsLse v, WsLse* warp_scratch /* BLOCK/32 */) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v = lse_combine(v, lse_shfl_down(v, d));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) warp_scratch[warp] = v;
    __syncthreads();
    if (warp == 0) {
        WsLse t;
        if (lane < BLOCK / 32) {
            t = warp_scratch[lane];
        } else {
            t.m = -INFINITY;
            t.S = 0.0;
            t.Q = 0.0;
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) t = lse_combine(t, lse_shfl_down(t, d));
        v = t;
    }
    return v;
}

// (m, S, Q) of n_partials partials, combined in a fixed order; result valid in thread 0.
template <int BLOCK>
__device__ __forceinline__ WsLse lse_block_combine(const WsLse* __restrict__ partials, int n_partials, WsLse* warp_scratch /* BLOCK/32 */) {
    WsLse part;
    part.m = -INFINITY;
    part.S = 0.0;
    part.Q = 0.0;
    for (int i = threadIdx.x; i < n_partials; i += BLOCK) part = lse_combine(part, partials[i]);
    return lse_block_reduce<BLOCK>(part, warp_scratch);
}

// Sharded state: the ranks' (m, S, Q) triples (msq[3 r ..]) combined in rank order.  Every rank runs this on identical
// inputs in identical order, so the ESS decision and the normalisation constants are bit-identical on all ranks.
__device__ __forceinline__ WsLse lse_combine_ranks(const double* msq, int n_ranks) {
    WsLse tot;
    tot.m = -INFINITY;
    tot.S = 0.0;
    tot.Q = 0.0;
    for (int r = 0; r < n_ranks; ++r) {
        WsLse v;
        v.m = msq[3 * r + 0];
        v.S = msq[3 * r + 1];
        v.Q = msq[3 * r + 2];
        tot = lse_combine(tot, v);
    }
    return tot;
}

// The Resample decision (transformers.jl:474-498) from the combined (m, S, Q) of all n_global particles.
// ESS% == ess_perc_min to within a few ulp: the reference's 1 / (N sum w^2) and this S^2 / (N Q) round differently
// there (for exactly equal weights and ess_perc_min = 1.0 the reference fires for some N and not for others), so the
// decision of such a step is rounding noise on both sides; they are counted into *ties (ws_get_ess_ties) when it is set.
__device__ __forceinline__ void ws_decide(const WsLse& tot, int64_t n_global, double ess_perc_min, WsReduceOut* out,
                                          unsigned long long* ties) {
    out->m = tot.m;
    out->S = tot.S;
    out->Q = tot.Q;
    const double lse = tot.m + log(tot.S);
    out->lse = lse;
    const double nn = (double)n_global;
    out->ess_perc = (tot.S * tot.S) / (nn * tot.Q);  // 1 / (N * sum w^2), w = e / S
    out->log_mean_w = lse - log(nn);
    out->do_resample = (out->ess_perc < ess_perc_min) ? 1 : 0;  // NaN compares false, as in Julia
    if (ties != nullptr && fabs(out->ess_perc - ess_perc_min) <= 8.0 * 2.220446049250313e-16 * fabs(ess_perc_min)) atomicAdd(ties, 1ull);
}

// ------------------------------------------------------------------------------------------
// Fused elementwise window
// ------------------------------------------------------------------------------------------
// Persistent grid; a CTA of WS_VM_BLOCK threads works on tiles of WS_VM_BLOCK * WS_VM_P particles,
// thread t owning particles tile + t + j*WS_VM_BLOCK (j < WS_VM_P: every global access is coalesced).
// The register file is a [n_regs][WS_VM_P][WS_VM_BLOCK] array in shared memory: a thread only ever
// touches its own column, so the pass needs no barrier and shared-memory accesses are conflict-free
// 64-bit lanes.  Each micro-op is decoded once per thread and applied to its WS_VM_P particles, which
// amortises the interpreter overhead and gives WS_VM_P independent dependency chains.
//
// STAGED = true (whenever the staging rows fit next to the register file): the plane loads of the NEXT
// tile are issued as cp.async (LDGSTS, 8 B per particle and plane: the gather through the ancestors is
// per element, so there is no bulk/TMA shape to use) into [n_loads] staging rows behind the register file
// while the current tile runs its program, and the ancestors are fetched two tiles ahead.  A thread only
// reads what it copied itself, so cp.async.wait_group is all the synchronisation there is.  Without this
// a warp spent a third of its time waiting on ancestor -> plane load chains (profiles/r1_ncu_*_r1e).
__device__ __forceinline__ void ws_cp_async8(double* smem_dst, const double* gsrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void ws_cp_async16(void* smem_dst, const void* gsrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void ws_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void ws_cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

template <bool STAGED, bool CKPT = false>
__global__ void __launch_bounds__(WS_VM_BLOCK, WS_VM_MINB) ws_vm_kernel(const __grid_constant__ WsVmProgram P) {
    extern __shared__ __align__(16) double ws_vm_smem[];
    __shared__ WsLse warp_scratch[WS_VM_BLOCK / 32];
    double* R = ws_vm_smem + threadIdx.x;
    constexpr int RS = WS_VM_P * WS_VM_BLOCK;  // doubles between two registers of the file
    double* const stage = R + P.n_regs * RS;   // [n_loads][WS_VM_P][WS_VM_BLOCK]   (STAGED only)
    // the program, unpacked once per CTA (ws_vm.cuh: WsDop) behind the register file and the staging rows
    WsDop* const dops = reinterpret_cast<WsDop*>(ws_vm_smem + (P.n_regs + (STAGED ? P.n_loads : 0)) * RS);
    for (int t = threadIdx.x; t < P.n_ops; t += WS_VM_BLOCK) dops[t] = ws_decode_op<WS_VM_BLOCK, WS_VM_P>(P.ops[t]);
    // per-thread (m, S, Q) states of the checkpoints: [n_ckpt][3][WS_VM_BLOCK] behind the decoded program
    double* const ck = reinterpret_cast<double*>(dops + P.n_ops) + threadIdx.x;
    for (int c = 0; CKPT && c < P.n_ckpt; ++c) {
        ck[(c * 3 + 0) * WS_VM_BLOCK] = -INFINITY;
        ck[(c * 3 + 1) * WS_VM_BLOCK] = 0.0;
        ck[(c * 3 + 2) * WS_VM_BLOCK] = 0.0;
    }
    __syncthreads();

    WsLse part;
    part.m = -INFINITY;
    part.S = 0.0;
    part.Q = 0.0;
    double esum[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) esum[k] = 0.0;
    double red_m = 0.0, red_invS = 0.0;
    if (P.n_expect > 0) {
        red_m = P.red->m;
        red_invS = 1.0 / P.red->S;
    }

    // local particle indices fit 32 bits (ws_create: n < 2^31 - 65536), which halves the address arithmetic
    constexpr int TILE = WS_VM_BLOCK * WS_VM_P;
    const int n = (int)P.n;
    const int n_tiles = (n + TILE - 1) / TILE;
    // logw_mode 3: the Resample step in front of this pass is still pending on the host; its flag decides
    const bool fired = (P.logw_mode != 3) || P.red->do_resample != 0;
    const int lmode = (P.logw_mode == 3) ? (fired ? 2 : 1) : P.logw_mode;
    const double lbase = (P.logw_mode == 3) ? P.red->log_mean_w : P.logw_base;
    const bool any_gather = P.load_gather != 0u && fired;  // not fired: the ancestors are the identity

    // clamped index of the thread's j-th particle in a tile (always a valid address)
    auto tile_index = [&](int tile, int j) -> int {
        const int i = tile * TILE + (int)threadIdx.x + j * WS_VM_BLOCK;
        return i < n ? i : n - 1;
    };
    // issue the staged loads of `tile` (source rows anc[] for gathered planes)
    auto issue_stage = [&](int tile, const int (&anc)[WS_VM_P]) {
        for (int k = 0; k < P.n_loads; ++k) {
            const bool g = any_gather && ((P.load_gather >> k) & 1u);
            const double* __restrict__ ptr = P.load_ptr[k];
            double* dst = stage + k * RS;
#pragma unroll
            for (int j = 0; j < WS_VM_P; ++j)
                ws_cp_async8(dst + j * WS_VM_BLOCK, ptr + (unsigned)(g ? anc[j] : tile_index(tile, j)));
        }
        ws_cp_async_commit();
    };

    int anc_next[WS_VM_P];  // STAGED: ancestors of the tile after the one whose loads are in flight
    if (STAGED) {
        const int t0 = blockIdx.x, t1 = blockIdx.x + gridDim.x;
        if (t0 < n_tiles) {
            int a0[WS_VM_P];
#pragma unroll
            for (int j = 0; j < WS_VM_P; ++j) a0[j] = any_gather ? __ldg(P.ancestors + tile_index(t0, j)) : 0;
            issue_stage(t0, a0);
        }
#pragma unroll
        for (int j = 0; j < WS_VM_P; ++j) anc_next[j] = (any_gather && t1 < n_tiles) ? __ldg(P.ancestors + tile_index(t1, j)) : 0;
    }

    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        int idx[WS_VM_P];   // clamped (always valid) index of the thread's j-th particle
        bool live[WS_VM_P];
        uint64_t particle[WS_VM_P];
        const int first = tile * TILE + (int)threadIdx.x;
#pragma unroll
        for (int j = 0; j < WS_VM_P; ++j) {
            const int i = first + j * WS_VM_BLOCK;
            live[j] = i < n;
            idx[j] = live[j] ? i : n - 1;
            particle[j] = (uint64_t)(P.particle_offset + (int64_t)idx[j]);
        }
        // ---- loads ------------------------------------------------------------------------------
        if (STAGED) {
            ws_cp_async_wait_all();
            for (int k = 0; k < P.n_loads; ++k) {
                const double* srcs = stage + k * RS;
                double* dst = R + (int)P.load_reg[k] * RS;
                double t[WS_VM_P];
#pragma unroll
                for (int j = 0; j < WS_VM_P; ++j) t[j] = srcs[j * WS_VM_BLOCK];
#pragma unroll
                for (int j = 0; j < WS_VM_P; ++j) dst[j * WS_VM_BLOCK] = t[j];
            }
            const int tn = tile + gridDim.x, tnn = tn + gridDim.x;
            if (tn < n_tiles) issue_stage(tn, anc_next);
            if (any_gather && tnn < n_tiles) {
#pragma unroll
                for (int j = 0; j < WS_VM_P; ++j) anc_next[j] = __ldg(P.ancestors + tile_index(tnn, j));
            }
        } else {
            int src[WS_VM_P];
#pragma unroll
            for (int j = 0; j < WS_VM_P; ++j) src[j] = idx[j];
            if (any_gather) {
#pragma unroll
                for (int j = 0; j < WS_VM_P; ++j) src[j] = __ldg(P.ancestors + idx[j]);
            }
            for (int k0 = 0; k0 < P.n_loads; k0 += 4) {
                double tmp[4][WS_VM_P];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (k0 + k < P.n_loads) {
                        const bool g = any_gather && ((P.load_gather >> (k0 + k)) & 1u);
                        const double* __restrict__ ptr = P.load_ptr[k0 + k];
#pragma unroll
                        for (int j = 0; j < WS_VM_P; ++j) tmp[k][j] = __ldg(ptr + (unsigned)(g ? src[j] : idx[j]));
                    }
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (k0 + k < P.n_loads) {
                        double* dst = R + (int)P.load_reg[k0 + k] * RS;
#pragma unroll
                        for (int j = 0; j < WS_VM_P; ++j) dst[j * WS_VM_BLOCK] = tmp[k][j];
                    }
                }
            }
        }
        double lw_old[WS_VM_P];
#pragma unroll
        for (int j = 0; j < WS_VM_P; ++j) lw_old[j] = 0.0;
        if (lmode == 1 || P.n_expect > 0) {
#pragma unroll
            for (int j = 0; j < WS_VM_P; ++j) lw_old[j] = P.logw[(unsigned)idx[j]];
        }

        // ---- program ------------------------------------------------------------------------------
        double acc[WS_VM_P];
        double lw_run[WS_VM_P];   // CKPT: log-weight the window started from (+ the terms folded in at checkpoints)
#pragma unroll
        for (int j = 0; j < WS_VM_P; ++j) {
            acc[j] = 0.0;
            lw_run[j] = lmode == 1 ? lw_old[j] : lbase;
        }
        if (!CKPT) {
            for (int pc = 0; pc < P.n_ops; ++pc) {
                ws_vm_exec_d<WS_VM_BLOCK, WS_VM_P>(dops[pc], R, acc, P.rng, particle);
            }
        } else {
            int next = 0;
            for (int pc = 0; pc < P.n_ops; ++pc) {
                ws_vm_exec_d<WS_VM_BLOCK, WS_VM_P>(dops[pc], R, acc, P.rng, particle);
                if (next < P.n_ckpt && pc == (int)P.ckpt_pc[next]) {
#pragma unroll
                    for (int j = 0; j < WS_VM_P; ++j) {
                        lw_run[j] += acc[j];
                        acc[j] = 0.0;
                    }
                    WsLse st;
                    st.m = ck[(next * 3 + 0) * WS_VM_BLOCK];
                    st.S = ck[(next * 3 + 1) * WS_VM_BLOCK];
                    st.Q = ck[(next * 3 + 2) * WS_VM_BLOCK];
                    lse_push_many<WS_VM_P>(st, lw_run, live);
                    ck[(next * 3 + 0) * WS_VM_BLOCK] = st.m;
                    ck[(next * 3 + 1) * WS_VM_BLOCK] = st.S;
                    ck[(next * 3 + 2) * WS_VM_BLOCK] = st.Q;
                    ++next;
                }
            }
        }

        // ---- stores ---------------------------------------------------------------------------------
        for (int k = 0; k < P.n_stores; ++k) {
            const double* srcr = R + (int)P.store_reg[k] * RS;
            double* __restrict__ ptr = P.store_ptr[k];
#pragma unroll
            for (int j = 0; j < WS_VM_P; ++j)
                if (live[j]) ptr[(unsigned)idx[j]] = srcr[j * WS_VM_BLOCK];
        }
        if (P.logw_mode != 0) {
            double lw[WS_VM_P];
#pragma unroll
            for (int j = 0; j < WS_VM_P; ++j) {
                lw[j] = (CKPT ? lw_run[j] : (lmode == 1 ? lw_old[j] : lbase)) + acc[j];
                if (live[j]) (CKPT && P.logw_out != nullptr ? P.logw_out : P.logw)[(unsigned)idx[j]] = lw[j];
            }
            lse_push_many<WS_VM_P>(part, lw, live);
        }
        if (P.n_expect > 0) {
#pragma unroll
            for (int j = 0; j < WS_VM_P; ++j) {
                if (live[j]) {
                    const double w = ws_exp_nonpos(lw_old[j] - red_m) * red_invS;
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        if (k < P.n_expect) esum[k] += w * R[(int)P.expect_reg[k] * RS + j * WS_VM_BLOCK];
                    }
                }
            }
        }
    }

    if (P.logw_mode != 0 && P.partials != nullptr) {
        WsLse tot = lse_block_reduce<WS_VM_BLOCK>(part, warp_scratch);
        if (threadIdx.x == 0) P.partials[blockIdx.x] = tot;
    }
    for (int c = 0; CKPT && c < P.n_ckpt; ++c) {
        WsLse st;
        st.m = ck[(c * 3 + 0) * WS_VM_BLOCK];
        st.S = ck[(c * 3 + 1) * WS_VM_BLOCK];
        st.Q = ck[(c * 3 + 2) * WS_VM_BLOCK];
        __syncthreads();  // warp_scratch of the previous reduction has been read
        WsLse tot = lse_block_reduce<WS_VM_BLOCK>(st, warp_scratch);
        if (threadIdx.x == 0) P.ckpt_partials[(size_t)c * gridDim.x + blockIdx.x] = tot;
    }
    if (P.n_expect > 0) {
        __shared__ double esc[WS_VM_BLOCK / 32][8];
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            double v = esum[k];
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
            if (lane == 0) esc[warp][k] = v;
        }
        __syncthreads();
        if (threadIdx.x < 8 && threadIdx.x < P.n_expect) {
            double v = 0.0;
            for (int w = 0; w < WS_VM_BLOCK / 32; ++w) v += esc[w][threadIdx.x];
            P.expect_partials[(size_t)blockIdx.x * P.n_expect + threadIdx.x] = v;
        }
    }
}

// ------------------------------------------------------------------------------------------
// Straight-line form of the fused window (ws_vm_sl.cuh): same tiling, staging and epilogue as
// ws_vm_kernel<true>, but the window is a compile-time signature and its register file lives in registers.
// Shared memory holds only the staging rows of the next tile's plane loads ([n_loads][PP][WS_VM_BLOCK]).
// ------------------------------------------------------------------------------------------
#include "ws_vm_sl.cuh"
#ifndef WS_SL_P
#define WS_SL_P 4      // particles per thread (measured on B200, profiles/r2n_sl_shape_sweep.txt: 2x6 1.72 ms, 3x4 1.58, 3x5 1.72, 4x4 1.70, 4x3 1.51)
#endif
#ifndef WS_SL_MINB
#define WS_SL_MINB 3   // resident CTAs per SM the kernels are compiled for
#endif
template <class Sig, int PP>
__global__ void __launch_bounds__(WS_VM_BLOCK, WS_SL_MINB) ws_vm_sl_kernel(const __grid_constant__ WsVmProgram P) {
    extern __shared__ __align__(16) double ws_vm_smem[];
    __shared__ WsLse warp_scratch[WS_VM_BLOCK / 32];
    constexpr int RS = PP * WS_VM_BLOCK;
    constexpr int TILE = WS_VM_BLOCK * PP;
    constexpr int NL = Sig::n_loads, NS = Sig::n_stores;
    double* const stage = ws_vm_smem + threadIdx.x;  // [NL][PP][WS_VM_BLOCK]

    WsLse part;
    part.m = -INFINITY;
    part.S = 0.0;
    part.Q = 0.0;
    const int n = (int)P.n;
    const int n_tiles = (n + TILE - 1) / TILE;
    // logw_mode 3: the Resample step in front of this pass is still pending on the host; its flag decides
    const bool fired = (P.logw_mode != 3) || P.red->do_resample != 0;
    const int lmode = (P.logw_mode == 3) ? (fired ? 2 : 1) : P.logw_mode;
    const double lbase = (P.logw_mode == 3) ? P.red->log_mean_w : P.logw_base;
    const bool any_gather = P.load_gather != 0u && fired;  // not fired: the ancestors are the identity

    auto tile_index = [&](int tile, int j) -> int {
        const int i = tile * TILE + (int)threadIdx.x + j * WS_VM_BLOCK;
        return i < n ? i : n - 1;
    };
    auto issue_stage = [&](int tile, const int (&anc)[PP]) {
#pragma unroll
        for (int k = 0; k < NL; ++k) {
            const bool g = any_gather && ((P.load_gather >> k) & 1u);
            const double* __restrict__ ptr = P.load_ptr[k];
#pragma unroll
            for (int j = 0; j < PP; ++j)
                ws_cp_async8(stage + k * RS + j * WS_VM_BLOCK, ptr + (unsigned)(g ? anc[j] : tile_index(tile, j)));
        }
        ws_cp_async_commit();
    };

    WsSlConsts<Sig> K;
    ws_sl_load_consts<Sig>(K, P, std::make_integer_sequence<int, Sig::n_ops>{});
    const bool replay = P.rng.replay_n != nullptr || P.rng.replay_u != nullptr || P.rng.replay_e != nullptr;

    int anc_next[PP];
    {
        const int t0 = blockIdx.x, t1 = blockIdx.x + gridDim.x;
        if (t0 < n_tiles) {
            int a0[PP];
#pragma unroll
            for (int j = 0; j < PP; ++j) a0[j] = any_gather ? __ldg(P.ancestors + tile_index(t0, j)) : 0;
            issue_stage(t0, a0);
        }
#pragma unroll
        for (int j = 0; j < PP; ++j) anc_next[j] = (any_gather && t1 < n_tiles) ? __ldg(P.ancestors + tile_index(t1, j)) : 0;
    }

    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        int idx[PP];
        bool live[PP];
        uint64_t particle[PP];
        const int first = tile * TILE + (int)threadIdx.x;
#pragma unroll
        for (int j = 0; j < PP; ++j) {
            const int i = first + j * WS_VM_BLOCK;
            live[j] = i < n;
            idx[j] = live[j] ? i : n - 1;
            particle[j] = (uint64_t)(P.particle_offset + (int64_t)idx[j]);
        }
        double R[Sig::n_regs * PP];
        if (NL > 0) {
            ws_cp_async_wait_all();
            ws_sl_loads<Sig, PP, WS_VM_BLOCK>(R, stage, std::make_integer_sequence<int, NL>{});
            const int tn = tile + gridDim.x, tnn = tn + gridDim.x;
            if (tn < n_tiles) issue_stage(tn, anc_next);
            if (any_gather && tnn < n_tiles) {
#pragma unroll
                for (int j = 0; j < PP; ++j) anc_next[j] = __ldg(P.ancestors + tile_index(tnn, j));
            }
        }
        double lw_old[PP];
#pragma unroll
        for (int j = 0; j < PP; ++j) lw_old[j] = 0.0;
        if (lmode == 1) {
#pragma unroll
            for (int j = 0; j < PP; ++j) lw_old[j] = P.logw[(unsigned)idx[j]];
        }

        double acc[PP];
#pragma unroll
        for (int j = 0; j < PP; ++j) acc[j] = 0.0;
        ws_sl_run<Sig, PP>(R, acc, P, K, replay, particle, std::make_integer_sequence<int, Sig::n_ops>{});

        ws_sl_stores<Sig, PP, WS_VM_BLOCK>(R, P, (unsigned)first, live, std::make_integer_sequence<int, NS>{});
        if (P.logw_mode != 0) {
            double lw[PP];
#pragma unroll
            for (int j = 0; j < PP; ++j) {
                lw[j] = (lmode == 1 ? lw_old[j] : lbase) + acc[j];
                if (live[j]) P.logw[(unsigned)first + j * WS_VM_BLOCK] = lw[j];
            }
            lse_push_many<PP>(part, lw, live);
        }
    }
    if (P.logw_mode != 0 && P.partials != nullptr) {
        WsLse tot = lse_block_reduce<WS_VM_BLOCK>(part, warp_scratch);
        if (threadIdx.x == 0) P.partials[blockIdx.x] = tot;
    }
}

// ---- straight-line form of a checkpointed window (speculative blocks, ws_exec_spec) ------------------------------
// The window is a signature's window repeated n_ckpt <= NCK times with other constants (the K observations of a block
// of examples/linear_regression.jl's loop), a checkpoint behind every repetition.  The planes are loaded once, every
// repetition runs the signature's micro-ops (the interpreter's own arithmetic, as in ws_vm_sl_kernel), folds its
// terms into the running log-weight and pushes it into that repetition's (m, S, Q) state — NCK states in registers.
// The interpreter's checkpoints (ws_vm_kernel<., true>) keep their states in shared memory, which costs it its
// occupancy: 65 us per observation at N = 1e7 against 20 here.
#ifndef WS_SLCK_N
#define WS_SLCK_N 8      // checkpoints per pass
#endif
#ifndef WS_SLCK_P
#define WS_SLCK_P 2      // particles per thread
#endif
#ifndef WS_SLCK_MINB
#define WS_SLCK_MINB 4
#endif
template <class Sig, int PP, int NCK>
__global__ void __launch_bounds__(WS_VM_BLOCK, WS_SLCK_MINB) ws_vm_sl_ckpt_kernel(const __grid_constant__ WsVmProgram P) {
    extern __shared__ __align__(16) double ws_vm_smem[];
    __shared__ WsLse warp_scratch[WS_VM_BLOCK / 32];
    __shared__ double kc[NCK][Sig::n_ops][3];   // constants of the repetitions
    constexpr int RS = PP * WS_VM_BLOCK;
    constexpr int TILE = WS_VM_BLOCK * PP;
    constexpr int NL = Sig::n_loads;
    double* const stage = ws_vm_smem + threadIdx.x;  // [NL][PP][WS_VM_BLOCK]
    const int reps = P.n_ckpt;
    for (int t = threadIdx.x; t < reps * Sig::n_ops; t += WS_VM_BLOCK) {
        kc[t / Sig::n_ops][t % Sig::n_ops][0] = P.ops[t].k0;
        kc[t / Sig::n_ops][t % Sig::n_ops][1] = P.ops[t].k1;
        kc[t / Sig::n_ops][t % Sig::n_ops][2] = P.ops[t].k2;
    }
    __syncthreads();
    WsLse st[NCK];
#pragma unroll
    for (int c = 0; c < NCK; ++c) {
        st[c].m = -INFINITY;
        st[c].S = 0.0;
        st[c].Q = 0.0;
    }
    const int n = (int)P.n;
    const int n_tiles = (n + TILE - 1) / TILE;
    const int lmode = P.logw_mode;          // 1 or 2 (a block starts from resolved log-weights)
    const double lbase = P.logw_base;
    const bool any_gather = P.load_gather != 0u;
    auto tile_index = [&](int tile, int j) -> int {
        const int i = tile * TILE + (int)threadIdx.x + j * WS_VM_BLOCK;
        return i < n ? i : n - 1;
    };
    auto issue_stage = [&](int tile) {
#pragma unroll
        for (int k = 0; k < NL; ++k) {
            const bool g = any_gather && ((P.load_gather >> k) & 1u);
            const double* __restrict__ ptr = P.load_ptr[k];
#pragma unroll
            for (int j = 0; j < PP; ++j) {
                const int i = tile_index(tile, j);
                ws_cp_async8(stage + k * RS + j * WS_VM_BLOCK, ptr + (unsigned)(g ? __ldg(P.ancestors + i) : i));
            }
        }
        ws_cp_async_commit();
    };
    if ((int)blockIdx.x < n_tiles) issue_stage(blockIdx.x);
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        bool live[PP];
        uint64_t particle[PP];
        const int first = tile * TILE + (int)threadIdx.x;
#pragma unroll
        for (int j = 0; j < PP; ++j) {
            const int i = first + j * WS_VM_BLOCK;
            live[j] = i < n;
            particle[j] = (uint64_t)(P.particle_offset + (int64_t)(live[j] ? i : n - 1));
        }
        double R[Sig::n_regs * PP];
        ws_cp_async_wait_all();
        ws_sl_loads<Sig, PP, WS_VM_BLOCK>(R, stage, std::make_integer_sequence<int, NL>{});
        if (tile + (int)gridDim.x < n_tiles) issue_stage(tile + gridDim.x);
        double lw[PP];
#pragma unroll
        for (int j = 0; j < PP; ++j) lw[j] = lmode == 1 ? P.logw[(unsigned)tile_index(tile, j)] : lbase;
#pragma unroll
        for (int c = 0; c < NCK; ++c) {
            if (c < reps) {
                WsSlConsts<Sig> K;
#pragma unroll
                for (int i = 0; i < Sig::n_ops; ++i) {
                    K.k[i][0] = kc[c][i][0];
                    K.k[i][1] = kc[c][i][1];
                    K.k[i][2] = kc[c][i][2];
                }
                double acc[PP];
#pragma unroll
                for (int j = 0; j < PP; ++j) acc[j] = 0.0;
                ws_sl_run_at<Sig, PP>(R, acc, P, P.ops + c * Sig::n_ops, K, particle, std::make_integer_sequence<int, Sig::n_ops>{});
#pragma unroll
                for (int j = 0; j < PP; ++j) lw[j] += acc[j];
                lse_push_many<PP>(st[c], lw, live);
            }
        }
        double* const lout = P.logw_out != nullptr ? P.logw_out : P.logw;
#pragma unroll
        for (int j = 0; j < PP; ++j)
            if (live[j]) lout[(unsigned)first + j * WS_VM_BLOCK] = lw[j];
    }
#pragma unroll
    for (int c = 0; c < NCK; ++c) {
        if (c < reps) {
            __syncthreads();  // warp_scratch of the previous reduction has been read
            WsLse tot = lse_block_reduce<WS_VM_BLOCK>(st[c], warp_scratch);
            if (threadIdx.x == 0) {
                P.ckpt_partials[(size_t)c * gridDim.x + blockIdx.x] = tot;
                if (c == reps - 1 && P.partials != nullptr) P.partials[blockIdx.x] = tot;   // the log-weights the pass leaves behind
            }
        }
    }
}
static bool ws_slck_ok(const WsVmProgram& P) {
    return P.n_ckpt > 0 && P.n_expect == 0 && (P.logw_mode == 1 || P.logw_mode == 2) && ws_sl_matches_repeated<WsSigLinregObs>(P, WS_SLCK_N);
}
static int ws_slck_grid(const WsVmProgram& P) {
    constexpr int TILE = WS_VM_BLOCK * WS_SLCK_P;
    const int64_t tiles = (P.n + TILE - 1) / TILE;
    const int grid = (int)(tiles < (int64_t)g_sm_count * WS_SLCK_MINB ? tiles : (int64_t)g_sm_count * WS_SLCK_MINB);
    return grid < 1 ? 1 : grid;
}

static bool g_vm_interp_only = false;  // env WSB200_VM=interp: every window on the interpreter (A/B, tests)
template <class Sig>
static cudaError_t ws_launch_vm_sl(const WsVmProgram& P, cudaStream_t s) {
    constexpr int TILE = WS_VM_BLOCK * WS_SL_P;
    const int64_t tiles = (P.n + TILE - 1) / TILE;
    int grid = (int)(tiles < (int64_t)g_sm_count * WS_SL_MINB ? tiles : (int64_t)g_sm_count * WS_SL_MINB);
    if (grid < 1) grid = 1;
    const int smem = (Sig::n_loads > 0 ? Sig::n_loads : 1) * TILE * (int)sizeof(double);
    ws_vm_sl_kernel<Sig, WS_SL_P><<<grid, WS_VM_BLOCK, smem, s>>>(P);
    return cudaGetLastError();
}
// (m, S, Q) partials a straight-line launch of this window would write (the runtime sizes n_partials with it)
int ws_vm_sl_grid(const WsVmProgram& P) {
    if (!g_vm_interp_only && P.n_ckpt != 0 && ws_slck_ok(P)) return ws_slck_grid(P);
    if (g_vm_interp_only || P.n_ckpt != 0 || ws_sl_find(P) < 0) return 0;
    constexpr int TILE = WS_VM_BLOCK * WS_SL_P;
    const int64_t tiles = (P.n + TILE - 1) / TILE;
    int grid = (int)(tiles < (int64_t)g_sm_count * WS_SL_MINB ? tiles : (int64_t)g_sm_count * WS_SL_MINB);
    return grid < 1 ? 1 : grid;
}

// rows of the shared-memory register file: n_regs registers (+ n_loads staging rows when they fit)
static bool ws_vm_staged(int n_regs, int n_loads) {
    return n_loads > 0 && (size_t)(n_regs + n_loads) * WS_VM_BLOCK * WS_VM_P * sizeof(double) <= (size_t)200 * 1024;
}
int ws_vm_smem_bytes(int n_regs, int n_loads, int n_ops, int n_ckpt) {
    const int rows = (n_regs < 1 ? 1 : n_regs) + (ws_vm_staged(n_regs < 1 ? 1 : n_regs, n_loads) ? n_loads : 0);
    return rows * WS_VM_BLOCK * WS_VM_P * (int)sizeof(double) + n_ops * (int)sizeof(WsDop) + n_ckpt * 3 * WS_VM_BLOCK * (int)sizeof(double);
}

int ws_vm_max_grid(int n_regs, int n_loads, int n_ops, int sm_count, int n_ckpt) {
    // resident CTAs per SM limited by the shared-memory register file and 2048 threads / SM
    const int smem = ws_vm_smem_bytes(n_regs, n_loads, n_ops, n_ckpt) + 1024;
    int per_sm = (227 * 1024) / smem;
    if (per_sm > WS_VM_MINB) per_sm = WS_VM_MINB;  // __launch_bounds__(WS_VM_BLOCK, WS_VM_MINB)
    if (per_sm < 1) per_sm = 1;
    return per_sm * sm_count;
}

cudaError_t ws_launch_vm(const WsVmProgram& P, int grid, cudaStream_t s) {
    if (!g_vm_interp_only && P.n_ckpt == 0) {
        switch (ws_sl_find(P)) {
#define WS_SL_CASE(idx, Sig) \
    case idx: return ws_launch_vm_sl<Sig>(P, s);
            WS_SL_SIGS(WS_SL_CASE)
#undef WS_SL_CASE
            default: break;
        }
    }
    if (!g_vm_interp_only && P.n_ckpt != 0 && ws_slck_ok(P)) {
        constexpr int smem_ck = WsSigLinregObs::n_loads * WS_VM_BLOCK * WS_SLCK_P * (int)sizeof(double);
        ws_vm_sl_ckpt_kernel<WsSigLinregObs, WS_SLCK_P, WS_SLCK_N><<<ws_slck_grid(P), WS_VM_BLOCK, smem_ck, s>>>(P);
        return cudaGetLastError();
    }
    const int smem = ws_vm_smem_bytes(P.n_regs, P.n_loads, P.n_ops, P.n_ckpt);
    if (P.n_ckpt > 0) {
        if (ws_vm_staged(P.n_regs, P.n_loads)) ws_vm_kernel<true, true><<<grid, WS_VM_BLOCK, smem, s>>>(P);
        else ws_vm_kernel<false, true><<<grid, WS_VM_BLOCK, smem, s>>>(P);
    } else if (ws_vm_staged(P.n_regs, P.n_loads)) ws_vm_kernel<true><<<grid, WS_VM_BLOCK, smem, s>>>(P);
    else ws_vm_kernel<false><<<grid, WS_VM_BLOCK, smem, s>>>(P);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// Stand-alone (m, S, Q) partials + finalize
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ws_reduce_logw_kernel(const double* __restrict__ logw, int64_t n,
                                                             WsLse* __restrict__ partials) {
    __shared__ WsLse warp_scratch[8];
    WsLse part;
    part.m = -INFINITY;
    part.S = 0.0;
    part.Q = 0.0;
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) lse_push(part, __ldg(logw + i));
    WsLse tot = lse_block_reduce<256>(part, warp_scratch);
    if (threadIdx.x == 0) partials[blockIdx.x] = tot;
}

cudaError_t ws_launch_reduce_logw(const double* logw, int64_t n, WsLse* partials, int grid, cudaStream_t s) {
    ws_reduce_logw_kernel<<<grid, 256, 0, s>>>(logw, n, partials);
    return cudaGetLastError();
}

// CTA j combines partials[j * n_partials ..] into out[j]: one CTA for a Resample step, K for the checkpoints of a
// speculative block.  Fixed combination order => the decision is deterministic for a given number of partials.
__global__ void __launch_bounds__(256) ws_finalize_kernel(const WsLse* __restrict__ partials, int n_partials,
                                                          int64_t n_global, double ess_perc_min,
                                                          WsReduceOut* __restrict__ out, unsigned long long* ties) {
    __shared__ WsLse warp_scratch[8];
    const WsLse tot = lse_block_combine<256>(partials + (size_t)blockIdx.x * n_partials, n_partials, warp_scratch);
    if (threadIdx.x == 0) ws_decide(tot, n_global, ess_perc_min, out + blockIdx.x, ties);
}

cudaError_t ws_launch_finalize(const WsLse* partials, int n_partials, int k, int64_t n_global, double ess_perc_min,
                               WsReduceOut* out, unsigned long long* ties, cudaStream_t s) {
    ws_finalize_kernel<<<k, 256, 0, s>>>(partials, n_partials, n_global, ess_perc_min, out, ties);
    return cudaGetLastError();
}

// Sharded state: combine the ranks' (m, S, Q) triples (allgathered, rank order) into the global reduction.
__global__ void ws_finalize_global_kernel(const double* __restrict__ all_msq, int n_ranks, int64_t n_global,
                                          double ess_perc_min, WsReduceOut* __restrict__ out, unsigned long long* ties) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    ws_decide(lse_combine_ranks(all_msq, n_ranks), n_global, ess_perc_min, out, ties);
}

cudaError_t ws_launch_finalize_global(const double* all_msq, int n_ranks, int64_t n_global, double ess_perc_min,
                                      WsReduceOut* out, cudaStream_t s, unsigned long long* ties) {
    ws_finalize_global_kernel<<<1, 32, 0, s>>>(all_msq, n_ranks, n_global, ess_perc_min, out, ties);
    return cudaGetLastError();
}

// Sharded state, mailbox form (ws_mailbox.cuh): the shard's partials are reduced, the (m, S, Q) triple is stored into
// every rank's mailbox, and as soon as all R triples are here they are combined in rank order — ws_finalize_kernel,
// ncclAllGather and ws_finalize_global_kernel in one launch, same operations in the same order (bit-identical result).
__global__ void __launch_bounds__(WS_MBOX_THREADS) ws_finalize_mbox_kernel(const WsLse* __restrict__ partials, int n_partials, int64_t n_global,
                                                                           double ess_perc_min, WsReduceOut* __restrict__ out,
                                                                           double* __restrict__ all_msq, unsigned long long* ties,
                                                                           const __grid_constant__ WsMailbox M) {
    __shared__ WsLse warp_scratch[WS_MBOX_THREADS / 32];
    __shared__ unsigned long long mine[3];
    __shared__ unsigned long long all[3 * WS_MBOX_MAX_RANKS];
    const WsLse loc = lse_block_combine<WS_MBOX_THREADS>(partials, n_partials, warp_scratch);
    if (threadIdx.x == 0) {
        mine[0] = (unsigned long long)__double_as_longlong(loc.m);
        mine[1] = (unsigned long long)__double_as_longlong(loc.S);
        mine[2] = (unsigned long long)__double_as_longlong(loc.Q);
    }
    __syncthreads();
    ws_mbox_allgather(M, M.seq, mine, 3, all);
    if (threadIdx.x != 0) return;
    const double* msq = reinterpret_cast<const double*>(all);   // the triples' bits, as they were sent
    for (int k = 0; k < 3 * M.nranks; ++k) all_msq[k] = msq[k];
    ws_decide(lse_combine_ranks(msq, M.nranks), n_global, ess_perc_min, out, ties);
}
cudaError_t ws_launch_finalize_mbox(const WsLse* partials, int n_partials, int64_t n_global, double ess_perc_min, WsReduceOut* out,
                                    double* all_msq, unsigned long long* ties, const WsMailbox& M, cudaStream_t s) {
    ws_finalize_mbox_kernel<<<1, WS_MBOX_THREADS, 0, s>>>(partials, n_partials, n_global, ess_perc_min, out, all_msq, ties, M);
    return cudaGetLastError();
}

// The barrier behind the offspring pushed into the peers' planes by earlier kernels of the stream.
__global__ void __launch_bounds__(64) ws_barrier_mbox_kernel(const __grid_constant__ WsMailbox M) {
    __shared__ unsigned long long got[WS_MBOX_MAX_RANKS];
    ws_mbox_barrier(M, M.seq, got);
}
cudaError_t ws_launch_barrier_mbox(const WsMailbox& M, cudaStream_t s) {
    ws_barrier_mbox_kernel<<<1, 64, 0, s>>>(M);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// CDF scan fused with the ancestor search
// ------------------------------------------------------------------------------------------
#define WS_FXS_SCALE 2305843009213693952.0 /* 2^61: two top bits of the tile word carry the status */
#define WS_FXS_MASK 0x3FFFFFFFFFFFFFFFull
#define WS_TILE_AGG 1ull
#define WS_TILE_INCL 2ull

// Fixed-point weights: q = rint(w * scale), scale <= 2^61 (ws_scan_set_scale): 2^61 for the floating-point slot
// grid (replayed / caller uniforms), N * 2^S for the integer slot grid of the Philox path, where the slot index of a
// CDF value is then simply its high bits.
__device__ __forceinline__ unsigned long long ws_w_to_fxs(double w, double scale) {
    if (!(w > 0.0)) return 0ull;
    if (w >= 1.0) return (unsigned long long)scale;
    return __double2ull_rn(w * scale);
}
__device__ __forceinline__ double ws_fxs_to_double(unsigned long long c, double scale) { return (double)c / scale; }

__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// slot -> uniform provider.  Philox mode: one Philox block serves two neighbouring slots
// (slot k uses words (2(k&1), 2(k&1)+1) of block k>>1); the last block is cached because
// consecutive particles ask for the same or neighbouring slots.
struct SlotUniform {
    int scheme;  // 0 stratified, 1 systematic
    uint64_t seed, stream;
    const double* replay;
    double r0;
    int64_t cached_blk;
    ws_u32x4 cached;
    __device__ __forceinline__ double operator()(int64_t k) {
        if (scheme == 1) return r0;
        if (replay != nullptr) return replay[k];
        const int64_t blk = k >> 1;
        if (blk != cached_blk) {
            cached = ws_philox4x32_10((uint64_t)blk, stream, seed);
            cached_blk = blk;
        }
        return (k & 1) ? ws_u01(cached.z, cached.w) : ws_u01(cached.x, cached.y);
    }
};

// F(C) for an arbitrary ascending uniform array: #{n : u_n <= C}  (icdf with caller uniforms, multinomial)
__device__ __forceinline__ int64_t ws_count_sorted_le(const double* __restrict__ us, int64_t n, double C) {
    int64_t lo = 0, hi = n;  // first index with us[idx] > C
    while (lo < hi) {
        int64_t mid = (lo + hi) >> 1;
        if (__ldg(us + mid) <= C) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ int64_t ws_F(const WsScanParams& P, double C, double inv_n, SlotUniform& su) {
    if (P.sorted_u != nullptr) return ws_count_sorted_le(P.sorted_u, P.n_slots, C);
    return ws_count_slots_le(C, P.n_slots, inv_n, su);
}

// ---- CDF + search in three dependency-free passes ------------------------------------------------
//   ws_cdf_tiles_kernel    w_i = exp(l_i - m)/S -> fixed point q_i; CTA tile of WS_CDF_TILE particles:
//                          tile-local inclusive prefix sums (8 B / particle) + one aggregate per tile
//   ws_cdf_offsets_kernel  one CTA: exclusive scan of the tile aggregates (n / 2048 values)
//   ws_search_kernel       warp-granular: C_m = offset[tile] + local prefix -> F(C_m) -> offspring slots
// A single-pass decoupled look-back was measured first (profiles/r1_scan_lookback_*): with thousands of
// small tiles in flight every tile walks back through all tiles that are still unfinished, and the
// kernel spent most of its time spinning on predecessor flags.  Materialising the tile-local CDF costs
// 16 B of extra traffic per particle but removes every inter-tile dependency; the fixed-point sums
// make the result independent of the summation order either way.
//
// Two ways to evaluate F(C) = #{slots n : u_n <= C}:
//   EXACT_FP = true   the reference's floating-point slot uniforms u_n = (n-1)*invN + r_n*invN
//                     (src/resampling.jl:39-41) with caller-supplied r (replay / icdf / multinomial):
//                     bit-compatible with the oracle for identical uniforms.
//   EXACT_FP = false  (Philox draws, the production path) the same stratified grid in exact integer
//                     arithmetic: with the CDF as a 2^61 fixed-point integer C and r_k a 61-bit Philox
//                     integer,  u_k <= C  <=>  k*2^61 + r_k <= C*N, so F = k + [r_k <= frac] with
//                     (k, frac) = divmod(C*N, 2^61) from one 64x32-bit product.  One Philox block and
//                     no loop per particle; the test-suite checks it against exact big-integer arithmetic.
#define WS_TILE_GROUP 32       // CDF tiles per group of the two-level tile offsets
#define WS_EXPAND_CHUNK 512    // output slots a warp stages in shared memory per round
#ifndef WS_EXPAND_LANE
#define WS_EXPAND_LANE 12      // staged slots a lane resolves per round of the running maximum (a multiple of 4)
#endif
#define WS_DIRECT_MAX 8        // offspring a lane writes itself; larger families are filled by the warp
#define WS_WARPS_PER_CTA (WS_SCAN_BLOCK / 32)
#define WS_MN_MAX_WINDOWS 64   // multinomial: windows of WS_RBUF_SLOTS slots a warp works through before the tile counts as heavy
#define WS_RBUF_SLOTS 512      // 8-byte words of a warp's window: slot uniforms of the tile's slot range (stratified), running spacing
                               // sums of two blocks of slots (multinomial), then the staged offspring

// The integer slot grid (Philox path).  The CDF is an integer C in units of 2^-S slots (scale = N * 2^S), slot k's
// uniform is u_k = (k + (r_k + 1/2) / 2^32) / N with r_k a 32-bit Philox word (slot k: word k & 3 of block k >> 2;
// systematic: one word for all slots), so with T = C * 2^(32 - S)
//      F(C) = #{k : u_k <= C} = hi32(T) + [ r'_k <= lo32(T) ],     r' = r masked to the bits lo32(T) can carry (S < 32)
// — two shifts, no multiplication.  `sh` = S - 32 (may be negative for N > 2^29), `rmask` = the mask of r'.
__device__ __forceinline__ void ws_slot_split(unsigned long long C, unsigned int n, int sh, unsigned int& k, unsigned int& frac) {
    const unsigned long long T = sh >= 0 ? (C >> sh) : (C << (-sh));
    const unsigned long long k64 = T >> 32;
    k = (k64 >= (unsigned long long)n) ? n : (unsigned int)k64;
    frac = (unsigned int)T;
}
__device__ __forceinline__ unsigned int ws_slot_word(const ws_u32x4& b, unsigned int k) {
    const unsigned int j = k & 3u;
    return j == 0u ? b.x : (j == 1u ? b.y : (j == 2u ? b.z : b.w));
}
__device__ __forceinline__ int ws_F_int(unsigned long long C, unsigned int n, int sh, unsigned int rmask, int scheme, unsigned int r0,
                                        uint64_t seed, uint64_t stream) {
    unsigned int k, frac;
    ws_slot_split(C, n, sh, k, frac);
    if (k >= n) return (int)n;
    unsigned int r;
    if (scheme == 1) {
        r = r0;
    } else {
        r = ws_slot_word(ws_philox4x32_10((uint64_t)(k >> 2), stream, seed), k);
    }
    return (int)k + ((r & rmask) <= frac ? 1 : 0);
}

#ifndef WS_CDF_ASYNC
#define WS_CDF_ASYNC 0   // (measured, profiles/r2o_scan_variants.txt: registers 0.74 ms, cp.async 0.81 ms for scan + search at N = 1e8) next tile's log-weights by cp.async into shared memory (1) or by plain loads into registers (0)
#endif
#ifndef WS_CDF_MINB
#define WS_CDF_MINB 4   // <= 64 registers, four CTAs per SM: no spills (at five CTAs, 48 registers, the prefetched tile spilled)
#endif
#ifndef WS_CDF_GRID
#define WS_CDF_GRID 4
#endif
__global__ void __launch_bounds__(WS_SCAN_BLOCK, WS_CDF_MINB) ws_cdf_tiles_kernel(const __grid_constant__ WsScanParams P) {
    if (P.gate != 0 && P.red->do_resample == 0) return;
    __shared__ unsigned long long warp_tot[2][WS_SCAN_BLOCK / 32];
    int parity = 0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = (int)P.n;
    const int n_tiles = (n + WS_CDF_TILE - 1) / WS_CDF_TILE;
    double m = 0.0, Sden = 1.0;
    if (P.mode == 0) {
        m = P.red->m;
        Sden = P.red->S;  // w = e / S as exp_norm does (correctly rounded quotient, see ws_div_pos)
    }
    const double rS = 1.0 / Sden;
    const double uniform_w = 1.0 / (double)P.n_slots;
#if WS_CDF_ASYNC
    // the log-weights of the NEXT tile are requested before the current tile is processed (the kernel was waiting on
    // its loads, not on the arithmetic: profiles/r1i_ncu_ws_cdf_tiles_kernel_20M.txt) — by cp.async into thread-private
    // slots of shared memory rather than into registers, which the FP64 part needs (ptxas spilled them)
    __shared__ __align__(16) double2 lbuf_all[WS_SCAN_ITEMS / 2][WS_SCAN_BLOCK];
    double2* const lbuf = &lbuf_all[0][threadIdx.x];
    auto request = [&](int tile) {
        if (P.mode != 2 && (tile + 1) * WS_CDF_TILE <= n) {
            const double2* p2 = reinterpret_cast<const double2*>(P.logw + (size_t)tile * WS_CDF_TILE + threadIdx.x * WS_SCAN_ITEMS);
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS / 2; ++k) ws_cp_async16(lbuf + k * WS_SCAN_BLOCK, p2 + k);
        }
        ws_cp_async_commit();
    };
    if ((int)blockIdx.x < n_tiles) request(blockIdx.x);
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int item0 = tile * WS_CDF_TILE + threadIdx.x * WS_SCAN_ITEMS;
        unsigned long long q[WS_SCAN_ITEMS];
        if (P.mode == 2) {
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS; ++k) q[k] = (item0 + k < n) ? ws_w_to_fxs(uniform_w, P.fx_scale) : 0ull;
        } else {
            double l[WS_SCAN_ITEMS];
            ws_cp_async_wait_all();
            if ((tile + 1) * WS_CDF_TILE <= n) {
#pragma unroll
                for (int k = 0; k < WS_SCAN_ITEMS / 2; ++k) {
                    const double2 v = lbuf[k * WS_SCAN_BLOCK];
                    l[2 * k] = v.x;
                    l[2 * k + 1] = v.y;
                }
            } else {
#pragma unroll
                for (int k = 0; k < WS_SCAN_ITEMS; ++k) l[k] = (item0 + k < n) ? __ldg(P.logw + item0 + k) : -INFINITY;
            }
            if (tile + (int)gridDim.x < n_tiles) request(tile + gridDim.x);   // (the thread's slots of lbuf were read above)
            if (P.mode == 0) {
                // items beyond the shard were loaded as -inf: e = 0.  e <= 1 and S >= 1, so w is in [0, 1] or NaN and the
                // saturating conversion (NaN -> 0) is ws_w_to_fxs without its two compares
#pragma unroll
                for (int k = 0; k < WS_SCAN_ITEMS; ++k)
                    q[k] = __double2ull_rn(ws_div_pos(ws_exp_nonpos_or0(l[k] - m), Sden, rS) * P.fx_scale);
            } else {
#pragma unroll
                for (int k = 0; k < WS_SCAN_ITEMS; ++k) q[k] = (item0 + k < n) ? ws_w_to_fxs(l[k], P.fx_scale) : 0ull;
            }
        }
#else
    // the log-weights of the NEXT tile are requested before the current tile is processed: the kernel was waiting on
    // its loads (long-scoreboard stalls, profiles/r1i_ncu_ws_cdf_tiles_kernel_20M.txt), not on the arithmetic
    auto load_tile = [&](int tile, double (&l)[WS_SCAN_ITEMS]) {
        const int item0 = tile * WS_CDF_TILE + threadIdx.x * WS_SCAN_ITEMS;
        if (item0 + WS_SCAN_ITEMS <= n) {
            const double2* p2 = reinterpret_cast<const double2*>(P.logw + item0);
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS / 2; ++k) {
                double2 v = __ldg(p2 + k);
                l[2 * k] = v.x;
                l[2 * k + 1] = v.y;
            }
        } else {
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS; ++k) l[k] = (item0 + k < n) ? __ldg(P.logw + item0 + k) : -INFINITY;
        }
    };
    // A landed tile is converted to fixed point before the next one is requested, so that only one set of eight
    // 64-bit values (the loads in flight, then q) is live besides the other: holding l, l_next and q together spilled
    // under the five-CTA register cap.
    double l[WS_SCAN_ITEMS];
#pragma unroll
    for (int k = 0; k < WS_SCAN_ITEMS; ++k) l[k] = -INFINITY;
    if (P.mode != 2 && (int)blockIdx.x < n_tiles) load_tile(blockIdx.x, l);
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int item0 = tile * WS_CDF_TILE + threadIdx.x * WS_SCAN_ITEMS;
        unsigned long long q[WS_SCAN_ITEMS];
        if (P.mode == 2) {
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS; ++k) q[k] = (item0 + k < n) ? ws_w_to_fxs(uniform_w, P.fx_scale) : 0ull;
        } else {
            if (P.mode == 0) {
                // items beyond the shard were loaded as -inf: e = 0.  e <= 1 and S >= 1, so w is in [0, 1] and the
                // conversion is ws_w_to_fxs without its two compares; NaN, -inf and d < -708 all give e = 0, q = 0
#pragma unroll
                for (int k = 0; k < WS_SCAN_ITEMS; ++k)
                    q[k] = __double2ull_rn(ws_div_pos(ws_exp_nonpos_or0(l[k] - m), Sden, rS) * P.fx_scale);
            } else {
#pragma unroll
                for (int k = 0; k < WS_SCAN_ITEMS; ++k) q[k] = (item0 + k < n) ? ws_w_to_fxs(l[k], P.fx_scale) : 0ull;
            }
            if (tile + (int)gridDim.x < n_tiles) load_tile(tile + gridDim.x, l);
        }
#endif
#pragma unroll
        for (int k = 1; k < WS_SCAN_ITEMS; ++k) q[k] += q[k - 1];
        const unsigned long long thread_total = q[WS_SCAN_ITEMS - 1];
        unsigned long long incl = thread_total;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            unsigned long long t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += t;
        }
        // two sets of warp totals, alternating with the tile: a warp writes set p only after the barrier of the tile in
        // between, which every warp passes after it has read set p, so one barrier per tile suffices
        unsigned long long* const wt = warp_tot[parity];
        parity ^= 1;
        if (lane == 31) wt[warp] = incl;
        __syncthreads();
        // lanes 0..7 take one warp total each: a shuffle scan over them gives the warp's exclusive prefix and the tile's sum
        unsigned long long t8 = lane < WS_SCAN_BLOCK / 32 ? wt[lane] : 0ull;
#pragma unroll
        for (int d = 1; d < WS_SCAN_BLOCK / 32; d <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, t8, d);
            if (lane >= d) t8 += t;
        }
        const unsigned long long tile_agg = __shfl_sync(0xffffffffu, t8, WS_SCAN_BLOCK / 32 - 1);
        unsigned long long warp_excl = __shfl_sync(0xffffffffu, t8, (warp + 31) & 31);
        if (warp == 0) warp_excl = 0ull;
        const unsigned long long thread_excl = warp_excl + (incl - thread_total);
        if (item0 + WS_SCAN_ITEMS <= n) {
            ulonglong2* dst = reinterpret_cast<ulonglong2*>(P.cdf_local + item0);
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS / 2; ++k) dst[k] = make_ulonglong2(thread_excl + q[2 * k], thread_excl + q[2 * k + 1]);
        } else {
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS; ++k)
                if (item0 + k < n) P.cdf_local[item0 + k] = thread_excl + q[k];
        }
        // the tile's aggregate: the offsets pass sums them per group of WS_TILE_GROUP tiles and scans the group sums
        // (n / 65 536 words); the search adds the <= 31 tile words in front of its tile to its group's prefix
        if (threadIdx.x == 0) P.tile_words[tile] = tile_agg;
    }
}

// exclusive scan of `count` words, in place, by one CTA of 1024 threads (fixed order); every thread
// takes WS_OFF_ITEMS consecutive words per round so that the loads of a round are all in flight together
#define WS_OFF_ITEMS 8
__device__ __forceinline__ void ws_scan_words_cta(unsigned long long* __restrict__ words, const int n_tiles, unsigned long long* total_out) {
    __shared__ unsigned long long warp_tot[32];
    __shared__ unsigned long long s_carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0ull;
    __syncthreads();
    for (int base = 0; base < n_tiles; base += 1024 * WS_OFF_ITEMS) {
        const int i0 = base + threadIdx.x * WS_OFF_ITEMS;
        unsigned long long v[WS_OFF_ITEMS];
#pragma unroll
        for (int k = 0; k < WS_OFF_ITEMS; ++k) v[k] = (i0 + k < n_tiles) ? words[i0 + k] : 0ull;
        unsigned long long thread_total = 0ull;
#pragma unroll
        for (int k = 0; k < WS_OFF_ITEMS; ++k) thread_total += v[k];
        unsigned long long incl = thread_total;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            unsigned long long t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += t;
        }
        if (lane == 31) warp_tot[warp] = incl;
        __syncthreads();
        unsigned long long warp_excl = 0ull, total = 0ull;
#pragma unroll
        for (int w = 0; w < 32; ++w) {
            const unsigned long long t = warp_tot[w];
            if (w < warp) warp_excl += t;
            total += t;
        }
        const unsigned long long carry = s_carry;
        unsigned long long run = carry + warp_excl + (incl - thread_total);
#pragma unroll
        for (int k = 0; k < WS_OFF_ITEMS; ++k) {
            if (i0 + k < n_tiles) words[i0 + k] = run;
            run += v[k];
        }
        __syncthreads();
        if (threadIdx.x == 0) s_carry = carry + total;
        __syncthreads();
    }
    if (threadIdx.x == 0 && total_out != nullptr) *total_out = s_carry;
}
// multinomial: the tile sums of the exponential spacings
__global__ void __launch_bounds__(1024) ws_cdf_offsets_kernel(const __grid_constant__ WsScanParams P) {
    if (P.gate != 0 && P.red->do_resample == 0) return;
    ws_scan_words_cta(P.tile_words, (int)((P.n + WS_CDF_TILE - 1) / WS_CDF_TILE), P.total);
}
// the CDF: the group sums behind the tile words (see ws_cdf_tiles_kernel), and the shard's total mass
__device__ __forceinline__ void ws_cdf_group_offsets_body(const WsScanParams& P) {   // one CTA of 1024 threads
    if (threadIdx.x == 0 && P.heavy_count != nullptr) *P.heavy_count = 0u;   // (the search that follows counts its heavy tiles here)
    if (P.gate != 0 && P.red->do_resample == 0) return;
    const int n_tiles = (int)((P.n + WS_CDF_TILE - 1) / WS_CDF_TILE);
    const int n_groups = (n_tiles + WS_TILE_GROUP - 1) / WS_TILE_GROUP;
    unsigned long long* const grp = P.tile_words + n_tiles;
    // group sums: a warp per group, a tile word per lane (coalesced 256-byte reads out of L2)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int g = warp; g < n_groups; g += 32) {
        const int idx = g * WS_TILE_GROUP + lane;
        unsigned long long v = idx < n_tiles ? P.tile_words[idx] : 0ull;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
        if (lane == 0) grp[g] = v;
    }
    __syncthreads();
    ws_scan_words_cta(grp, n_groups, P.total);
}
__global__ void __launch_bounds__(1024) ws_cdf_group_offsets_kernel(const __grid_constant__ WsScanParams P) { ws_cdf_group_offsets_body(P); }
// exclusive prefix of CDF tile `ct` (all lanes of a warp call; every lane gets the result)
__device__ __forceinline__ unsigned long long ws_tile_offset(const WsScanParams& P, const int n_tiles, const int ct, const int lane) {
    const int g = ct / WS_TILE_GROUP, idx = g * WS_TILE_GROUP + lane;
    unsigned long long v = idx < ct ? __ldg(P.tile_words + idx) : 0ull;
    if (lane == 31) v = __ldg(P.tile_words + n_tiles + g);   // (idx = 32 g + 31 >= ct always: the lane is free for the group's prefix)
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    return v;
}

// ---- multinomial without a sort: exponential spacings ------------------------------------------------------------
// T = floor(C * S_total / 2^61): the threshold of a CDF value in the units of the spacing sums
__device__ __forceinline__ unsigned long long ws_mn_threshold(unsigned long long C, unsigned long long S_total) {
    const unsigned long long lo = C * S_total, hi = __umul64hi(C, S_total);
    return (hi << 3) | (lo >> 61);
}
// global exclusive prefix of block b (WS_SCAN_TILE slots)
__device__ __forceinline__ unsigned long long ws_mn_block_prefix(const WsScanParams& P, int b) {
    return __ldg(P.mn_tile_off + b / (WS_CDF_TILE / WS_SCAN_TILE)) + __ldg(P.mn_block_local + b);
}
// the block whose slots contain the first running sum > T: largest b with prefix(b) <= T (two-level binary search)
__device__ __forceinline__ int ws_mn_find_block(const WsScanParams& P, unsigned long long T) {
    constexpr int BPT = WS_CDF_TILE / WS_SCAN_TILE;
    const int n_all = (int)P.n_slots + 1;
    const int n_tiles = (n_all + WS_CDF_TILE - 1) / WS_CDF_TILE, n_blocks = (n_all + WS_SCAN_TILE - 1) / WS_SCAN_TILE;
    int lo = 0, hi = n_tiles - 1;  // largest tile with tile_off <= T
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(P.mn_tile_off + mid) <= T) lo = mid; else hi = mid - 1;
    }
    const unsigned long long base = __ldg(P.mn_tile_off + lo);
    int b = lo * BPT;
    const int b_end = min(b + BPT, n_blocks);
    for (int j = b + 1; j < b_end; ++j)
        if (base + __ldg(P.mn_block_local + j) <= T) b = j;
    return b;
}
// F(C) = #{slots k < n_slots : S_k <= T} by one thread (rank edges, heavy tiles): find the block, walk its spacings
__device__ __forceinline__ int ws_F_mn(const WsScanParams& P, unsigned long long C) {
    const int ns = (int)P.n_slots;
    const unsigned long long T = ws_mn_threshold(C, *P.mn_total);
    const int b = ws_mn_find_block(P, T);
    unsigned long long S = ws_mn_block_prefix(P, b);
    int k = b * WS_SCAN_TILE;
    const int k_end = min(k + WS_SCAN_TILE, ns);
    while (k < k_end) {
        S += ws_spacing_of_slot((uint64_t)k, P.mn_shift, P.seed, P.stream);
        if (S > T) break;
        ++k;
    }
    return k;
}

// spacing prefixes of all n_slots + 1 global slots: one CTA tile of WS_CDF_TILE slots, one warp per block
__global__ void __launch_bounds__(WS_SCAN_BLOCK) ws_spacing_tiles_kernel(const __grid_constant__ WsScanParams P) {
    if (P.gate != 0 && P.red->do_resample == 0) return;
    __shared__ unsigned long long warp_tot[WS_SCAN_BLOCK / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_all = (int)P.n_slots + 1;
    const int n_tiles = (n_all + WS_CDF_TILE - 1) / WS_CDF_TILE;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int k0 = tile * WS_CDF_TILE + threadIdx.x * WS_SCAN_ITEMS;   // 8 consecutive slots = 4 Philox blocks
        unsigned long long sum = 0ull;
#pragma unroll
        for (int j = 0; j < WS_SCAN_ITEMS / 2; ++j) {
            const int k = k0 + 2 * j;
            if (k < n_all) {
                const ws_u32x4 r = ws_philox4x32_10((uint64_t)(k >> 1), P.stream, P.seed);
                sum += ws_spacing_fx(r.x, r.y, P.mn_shift);
                if (k + 1 < n_all) sum += ws_spacing_fx(r.z, r.w, P.mn_shift);
            }
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
        __syncthreads();
        if (lane == 0) warp_tot[warp] = sum;
        __syncthreads();
        unsigned long long excl = 0ull, agg = 0ull;
#pragma unroll
        for (int w = 0; w < WS_SCAN_BLOCK / 32; ++w) {
            const unsigned long long t = warp_tot[w];
            if (w < warp) excl += t;
            agg += t;
        }
        const int b = tile * (WS_CDF_TILE / WS_SCAN_TILE) + warp;
        if (lane == 0 && b * WS_SCAN_TILE < n_all) P.mn_block_local[b] = excl;
        if (threadIdx.x == 0) P.mn_tile_off[tile] = agg;
    }
}

// fixed-point mass below this rank's shard: given by value, or summed from the allgathered per-rank masses
// (sharded runs: saves the host a device round trip between the CDF pass and the search)
__device__ __forceinline__ unsigned long long ws_cdf_offset(const WsScanParams& P) {
    if (P.all_tot == nullptr) return P.cdf_offset;
    unsigned long long off = 0ull;
    for (int q = 0; q < P.rank; ++q) off += P.all_tot[q];
    return off;
}

// first / end global slot produced by this rank: F at the rank's left and right CDF edge
template <bool EXACT_FP>
__device__ __forceinline__ void ws_bounds_body(const WsScanParams& P) {   // one thread
    const int ns = (int)P.n_slots;
    const double inv_n = 1.0 / (double)ns;
    SlotUniform su;
    su.scheme = (P.scheme == 1) ? 1 : 0;
    su.seed = P.seed;
    su.stream = P.stream;
    su.replay = P.replay_u;
    su.r0 = 0.0;
    su.cached_blk = -1;
    unsigned int r0_int = 0u;
    if (P.scheme == 1 && P.sorted_u == nullptr) {
        if (P.replay_u != nullptr) {
            su.r0 = P.replay_u[0];
        } else {
            ws_u32x4 r = ws_philox4x32_10(0ull, P.stream, P.seed);
            su.r0 = ws_u01(r.x, r.y);
            r0_int = r.x;
        }
    }
    const int sh = P.fx_shift - 32;
    const unsigned int rmask = sh >= 0 ? 0xFFFFFFFFu : ~((1u << (-sh)) - 1u);
    const unsigned long long cdf_offset = ws_cdf_offset(P);
    const unsigned long long lo = cdf_offset, hi = cdf_offset + *P.total;
    int fs, fe;
    if (!EXACT_FP && P.scheme == 2) {
        fs = ws_F_mn(P, lo);
        fe = ws_F_mn(P, hi);
    } else if (EXACT_FP) {
        fs = (int)ws_F(P, ws_fxs_to_double(lo, P.fx_scale), inv_n, su);
        fe = (int)ws_F(P, ws_fxs_to_double(hi, P.fx_scale), inv_n, su);
    } else {
        fs = ws_F_int(lo, (unsigned int)ns, sh, rmask, su.scheme, r0_int, P.seed, P.stream);
        fe = ws_F_int(hi, (unsigned int)ns, sh, rmask, su.scheme, r0_int, P.seed, P.stream);
    }
    if (cdf_offset == 0ull) fs = 0;  // F(C_0) is 0 by definition for the very first particle
    if (P.last_rank) fe = ns;
    P.bounds[0] = fs;
    P.bounds[1] = fe;
}
template <bool EXACT_FP>
__global__ void ws_bounds_kernel(const __grid_constant__ WsScanParams P) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (P.gate != 0 && P.red->do_resample == 0) return;   // queued before the decision was read (sharded steps): nothing to bound
    ws_bounds_body<EXACT_FP>(P);
}
// Mailbox form of a sharded step's middle part (ws_mailbox.cuh), one launch instead of two kernels and two collectives:
// group offsets of the tile CDF and the shard's mass -> the masses of all ranks (exchange 1) -> this rank's slot bounds
// -> everybody's bounds + plane addresses, the exchange plan's input (exchange 2; P.bounds is word 0 of `xmine`).
template <bool EXACT_FP>
__global__ void __launch_bounds__(1024) ws_offsets_bounds_mbox_kernel(const __grid_constant__ WsScanParams P, const __grid_constant__ WsMailbox M,
                                                                      unsigned long long* all_tot, const unsigned long long* xmine, int xw,
                                                                      unsigned long long* xall) {
    ws_cdf_group_offsets_body(P);
    if (P.gate != 0 && P.red->do_resample == 0) return;   // (every rank reads the same decision: nobody sends, nobody waits)
    __syncthreads();   // *P.total
    ws_mbox_allgather(M, M.seq, P.total, 1, all_tot);
    if (threadIdx.x == 0) ws_bounds_body<EXACT_FP>(P);
    __syncthreads();
    ws_mbox_allgather(M, M.seq + 1u, xmine, xw, xall);
}

// What every warp of a search needs besides the CDF: the slot-uniform provider and the slot grid.
struct WsSearchCtx {
    SlotUniform su;
    unsigned int r0_int, rmask;
    int n, ns, slot_base, sh;
    double inv_n, fx_scale;
};
__device__ __forceinline__ void ws_search_setup(const WsScanParams& P, WsSearchCtx& X) {
    X.n = (int)P.n;          // local particles
    X.ns = (int)P.n_slots;   // global slots
    X.inv_n = 1.0 / (double)X.ns;
    X.slot_base = P.slot_base;
    X.su.scheme = (P.scheme == 1) ? 1 : 0;
    X.su.seed = P.seed;
    X.su.stream = P.stream;
    X.su.replay = P.replay_u;
    X.su.r0 = 0.0;
    X.su.cached_blk = -1;
    X.r0_int = 0u;
    X.sh = P.fx_shift - 32;
    X.rmask = X.sh >= 0 ? 0xFFFFFFFFu : ~((1u << (-X.sh)) - 1u);
    X.fx_scale = P.fx_scale;
    if (P.scheme == 1 && P.sorted_u == nullptr) {
        if (P.replay_u != nullptr) {
            X.su.r0 = P.replay_u[0];
        } else {
            ws_u32x4 r = ws_philox4x32_10(0ull, P.stream, P.seed);
            X.su.r0 = ws_u01(r.x, r.y);
            X.r0_int = r.x;
        }
    }
}

#ifndef WS_INTERIOR_FAST
#define WS_INTERIOR_FAST 1   // 0: every tile takes the range-checked search (A/B)
#endif
#define WS_RING_BLOCKS 128u   // Philox blocks (16 B each) a warp keeps from one tile to the next (power of two)
// A warp's Philox blocks carried from tile to tile (Philox-stratified interior tiles): blocks [lo, hi) are valid, block
// b is buf[b % WS_RING_BLOCKS], its words masked with rmask.  Every lane holds the same lo and hi.
struct WsRing {
    uint4* buf;
    unsigned int lo, hi;
};
// One warp, one tile of WS_SCAN_TILE consecutive particles starting at `tile_base`, lane L holding the global
// fixed-point CDF C[k] of particles tile_base + 8 L + k: per-particle slot counts F(C_m), then the offspring slots
// [F(C_{m-1}), F(C_m)) of every particle are written to P.ancestors.  `Cp` (lane 0; valid iff has_prev) is the CDF of
// the particle in front of the tile.  `rbuf`: the warp's shared-memory window (WS_RBUF_SLOTS words).  SHR: the slot
// split's shift X.sh is known to be >= 0 (N <= 2^29 without WSB200_FX_EXTRA_BITS).  `ring` (optional): the warp's
// Philox ring, for a warp that searches consecutive tiles.
template <bool EXACT_FP, bool MN, bool SHR = false>
__device__ __forceinline__ void ws_search_warp_tile(const WsScanParams& P, WsSearchCtx& X, unsigned long long* const rbuf,
                                                    const int lane, const int tile_base,
                                                    const unsigned long long (&C)[WS_SCAN_ITEMS], const unsigned long long Cp,
                                                    const bool has_prev, const bool interior = false, WsRing* const ring = nullptr) {
    int32_t* const out_s = reinterpret_cast<int32_t*>(rbuf);
    unsigned int* const rbuf32 = reinterpret_cast<unsigned int*>(rbuf);
    SlotUniform& su = X.su;
    const unsigned int r0_int = X.r0_int, rmask = X.rmask;
    const int n = X.n, ns = X.ns, slot_base = X.slot_base, sh = X.sh;
    const double inv_n = X.inv_n;
    const int item0 = tile_base + lane * WS_SCAN_ITEMS;
    // ---- per-particle F(C_m) -----------------------------------------------------------------------
    // F at the left edge of the particle set is by definition 0 (a slot with u = 0 belongs to
    // particle 1, as in icdf); elsewhere it is the previous particle's F.
    int f[WS_SCAN_ITEMS];
    int fstart = slot_base;
    bool coop = false, ringed = false;
    if (!EXACT_FP && MN) {
        // Multinomial: thresholds T_m of the lane's particles in the units of the spacing sums; the warp finds the
        // blocks of slots the tile can reach, regenerates their spacings once (running sums in the shared window)
        // and every lane counts the sums below its thresholds by binary search.
        const unsigned long long S_total = *P.mn_total;
        unsigned long long T[WS_SCAN_ITEMS];
#pragma unroll
        for (int k = 0; k < WS_SCAN_ITEMS; ++k) T[k] = ws_mn_threshold(C[k], S_total);
        unsigned long long Tp = has_prev ? ws_mn_threshold(Cp, S_total) : 0ull;
        Tp = __shfl_sync(0xffffffffu, Tp, 0);
        // the last particle of the shard present in this tile bounds the range from above
        const int n_in_tile = min(WS_SCAN_TILE, n - tile_base);
        const int last_lane = (n_in_tile - 1) / WS_SCAN_ITEMS, last_k = (n_in_tile - 1) % WS_SCAN_ITEMS;
        unsigned long long Tmax = 0ull;
#pragma unroll
        for (int k = 0; k < WS_SCAN_ITEMS; ++k)
            if (k == last_k) Tmax = T[k];
        Tmax = __shfl_sync(0xffffffffu, Tmax, last_lane);
        int b_lo = 0, b_hi = 0;
        if (lane == 0) b_lo = ws_mn_find_block(P, has_prev ? Tp : 0ull);
        if (lane == 1) b_hi = ws_mn_find_block(P, Tmax);
        b_lo = __shfl_sync(0xffffffffu, b_lo, 0);
        b_hi = __shfl_sync(0xffffffffu, b_hi, 1);
        const int k_lo = b_lo * WS_SCAN_TILE;
        const int k_hi = min((b_hi + 1) * WS_SCAN_TILE, ns);       // slots [k_lo, k_hi) are regenerated
        // the range is worked through in windows of WS_RBUF_SLOTS slots (two blocks): a tile with more offspring than one
        // window — any tile of skewed weights — used to fall back to one block walk per PARTICLE (44 ms at N = 1e8)
        coop = (k_hi - k_lo) <= WS_RBUF_SLOTS * WS_MN_MAX_WINDOWS;
        if (coop) {
            constexpr int PER = WS_RBUF_SLOTS / 32;                 // consecutive slots per lane
            int cnt[WS_SCAN_ITEMS];
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS; ++k) cnt[k] = 0;
            int cnt_p = 0;
            unsigned long long carry = ws_mn_block_prefix(P, b_lo);
            for (int k_win = k_lo; k_win < k_hi; k_win += WS_RBUF_SLOTS) {
                const int n_win = min(WS_RBUF_SLOTS, k_hi - k_win);
                unsigned long long lane_sum = 0ull;
                for (int j = 0; j < PER; j += 2) {                      // spacings into the window, lane totals in registers
                    const int k = k_win + lane * PER + j;
                    unsigned long long e0 = 0ull, e1 = 0ull;
                    if (k < k_hi) {
                        const ws_u32x4 r = ws_philox4x32_10((uint64_t)(k >> 1), P.stream, P.seed);
                        e0 = ws_spacing_fx(r.x, r.y, P.mn_shift);
                        if (k + 1 < k_hi) e1 = ws_spacing_fx(r.z, r.w, P.mn_shift);
                    }
                    rbuf[lane * PER + j] = e0;
                    rbuf[lane * PER + j + 1] = e1;
                    lane_sum += e0 + e1;
                }
                unsigned long long incl = lane_sum;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += t;
                }
                unsigned long long run = carry + (incl - lane_sum);
                for (int j = 0; j < PER; ++j) {                         // ... and in place into running sums
                    run += rbuf[lane * PER + j];
                    const int k = k_win + lane * PER + j;
                    rbuf[lane * PER + j] = (k < k_hi) ? run : ~0ull;    // beyond the range: larger than any threshold
                }
                carry += __shfl_sync(0xffffffffu, incl, 31);
                __syncwarp();
                const unsigned long long s_first = rbuf[0], s_last = rbuf[n_win - 1];
                auto count_le = [&](unsigned long long t) -> int {     // #{j < n_win : rbuf[j] <= t}
                    if (t < s_first) return 0;
                    if (t >= s_last) return n_win;
                    int lo = 0, hi = n_win;
                    while (lo < hi) {
                        const int mid = (lo + hi) >> 1;
                        if (rbuf[mid] <= t) lo = mid + 1; else hi = mid;
                    }
                    return lo;
                };
#pragma unroll
                for (int k = 0; k < WS_SCAN_ITEMS; ++k) cnt[k] += count_le(T[k]);
                if (lane == 0 && has_prev) cnt_p += count_le(Tp);
                __syncwarp();  // the window is refilled (and finally reused for the offspring below)
            }
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS; ++k) {
                int fk;
                if (item0 + k >= n) {
                    fk = -1;  // patched below
                } else {
                    fk = k_lo + cnt[k];
                    if (item0 + k == n - 1 && P.last_rank) {
                        if (fk < ns) atomicAdd(P.n_clamped, (unsigned long long)(ns - fk));
                        fk = ns;
                    }
                }
                f[k] = fk;
            }
            if (lane == 0 && has_prev) fstart = k_lo + cnt_p;
        }
    }
    if (!EXACT_FP && !MN && su.scheme == 0 && interior) {
        // The same as the branch below for a tile that lies inside the particle set and does not hold its last
        // particle (warp-uniform, said by the caller): no per-item range checks, and — the CDF being
        // non-decreasing — the slot range comes from the two ends of the tile instead of a min / max over all items.
        // A CDF value at or beyond the scale (zero-weight tail behind a total that rounded up) owns every slot: it is
        // looked up as the last slot with an always-true comparison.
        unsigned int kk[WS_SCAN_ITEMS];
        unsigned int fr[WS_SCAN_ITEMS];
        const unsigned int last = (unsigned int)ns - 1u;
#pragma unroll
        for (int k = 0; k < WS_SCAN_ITEMS; ++k) {
            const unsigned long long T = (SHR || sh >= 0) ? (C[k] >> sh) : (C[k] << (-sh));
            kk[k] = (unsigned int)(T >> 32);
            fr[k] = (unsigned int)T;
            if (kk[k] > last) {
                kk[k] = last;
                fr[k] = 0xFFFFFFFFu;
            }
        }
        unsigned int kp = kk[0], frp = 0u;
        if (lane == 0 && has_prev) {
            const unsigned long long T = (SHR || sh >= 0) ? (Cp >> sh) : (Cp << (-sh));
            kp = (unsigned int)(T >> 32);
            frp = (unsigned int)T;
            if (kp > last) {
                kp = last;
                frp = 0xFFFFFFFFu;
            }
        }
        const unsigned int blk0 = __shfl_sync(0xffffffffu, kp, 0) >> 2;
        const unsigned int blk1 = __shfl_sync(0xffffffffu, kk[WS_SCAN_ITEMS - 1], 31) >> 2;
        const unsigned int nblk = blk1 - blk0 + 1u;
        coop = nblk <= (unsigned int)(WS_RBUF_SLOTS / 2);
        if (ring != nullptr && nblk <= WS_RING_BLOCKS - 32u) {
            // The ring keeps the blocks a warp generated for its previous tiles: consecutive tiles share their boundary
            // block, and a round of 32 blocks that overshoots the tile serves the next one.  A round writes blocks
            // [hi, hi + 32) over [hi - WS_RING_BLOCKS, ...), which lie below blk0 as long as nblk <= WS_RING_BLOCKS - 32.
            if (blk0 < ring->lo || blk0 >= ring->hi) ring->lo = ring->hi = blk0;
            __syncwarp();   // every lane is done reading the blocks this round replaces
            for (; ring->hi <= blk1; ring->hi += 32u) {
                const unsigned int b = ring->hi + (unsigned int)lane;
                const ws_u32x4 r = ws_philox4x32_10((uint64_t)b, P.stream, P.seed);
                ring->buf[b & (WS_RING_BLOCKS - 1u)] = make_uint4(r.x & rmask, r.y & rmask, r.z & rmask, r.w & rmask);
            }
            if (ring->hi - ring->lo > WS_RING_BLOCKS) ring->lo = ring->hi - WS_RING_BLOCKS;
            __syncwarp();
            const unsigned int* const rb = reinterpret_cast<const unsigned int*>(ring->buf);
            constexpr unsigned int RMASK = 4u * WS_RING_BLOCKS - 1u;
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS; ++k) f[k] = (int)kk[k] + (rb[kk[k] & RMASK] <= fr[k] ? 1 : 0);
            if (lane == 0 && has_prev) fstart = (int)kp + (rb[kp & RMASK] <= frp ? 1 : 0);
            coop = ringed = true;
        } else if (coop) {
            for (unsigned int b = lane; b < nblk; b += 32u) {
                const ws_u32x4 r = ws_philox4x32_10((uint64_t)(blk0 + b), P.stream, P.seed);
                reinterpret_cast<uint4*>(rbuf32)[b] = make_uint4(r.x & rmask, r.y & rmask, r.z & rmask, r.w & rmask);
            }
            __syncwarp();
            const unsigned int* const rb = rbuf32 - 4u * blk0;
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS; ++k) f[k] = (int)kk[k] + (rb[kk[k]] <= fr[k] ? 1 : 0);
            if (lane == 0 && has_prev) fstart = (int)kp + (rb[kp] <= frp ? 1 : 0);
            __syncwarp();  // the window is reused for the offspring below
        }
    } else if (!EXACT_FP && !MN && su.scheme == 0) {
        // Philox-stratified: neighbouring particles ask for neighbouring slots, and one Philox block
        // serves four slots, so the warp generates the uniforms of the tile's whole slot range once
        // (a quarter of a Philox block per particle instead of one) and every lane looks its slots up.
        unsigned int kk[WS_SCAN_ITEMS];
        unsigned int fr[WS_SCAN_ITEMS];
        unsigned int kmax = 0u, kmin = 0xFFFFFFFFu;
#pragma unroll
        for (int k = 0; k < WS_SCAN_ITEMS; ++k) {
            ws_slot_split(C[k], (unsigned int)ns, sh, kk[k], fr[k]);
            if (item0 + k >= n) kk[k] = 0xFFFFFFFFu;  // beyond the shard: patched below
            if (kk[k] < (unsigned int)ns) {
                kmax = max(kmax, kk[k]);
                kmin = min(kmin, kk[k]);
            }
        }
        unsigned int kp = 0u;
        unsigned int frp = 0u;
        if (lane == 0 && has_prev) {
            ws_slot_split(Cp, (unsigned int)ns, sh, kp, frp);
            if (kp < (unsigned int)ns) {
                kmax = max(kmax, kp);
                kmin = min(kmin, kp);
            }
        }
        kmax = __reduce_max_sync(0xffffffffu, kmax);
        kmin = __reduce_min_sync(0xffffffffu, kmin);
        const unsigned int blk0 = kmin >> 2;
        coop = (kmin == 0xFFFFFFFFu) || ((kmax >> 2) - blk0 < (unsigned int)(WS_RBUF_SLOTS / 2));
        if (coop) {
            if (kmin != 0xFFFFFFFFu) {
                const unsigned int nblk = (kmax >> 2) - blk0 + 1u;
                for (unsigned int b = lane; b < nblk; b += 32u) {
                    const ws_u32x4 r = ws_philox4x32_10((uint64_t)(blk0 + b), P.stream, P.seed);
                    reinterpret_cast<uint4*>(rbuf32)[b] = make_uint4(r.x & rmask, r.y & rmask, r.z & rmask, r.w & rmask);
                }
            }
            __syncwarp();
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS; ++k) {
                int fk;
                if (kk[k] == 0xFFFFFFFFu) fk = -1;
                else if (kk[k] >= (unsigned int)ns) fk = ns;
                else fk = (int)kk[k] + (rbuf32[kk[k] - 4u * blk0] <= fr[k] ? 1 : 0);
                if (item0 + k == n - 1 && P.last_rank) {
                    if (fk < ns) atomicAdd(P.n_clamped, (unsigned long long)(ns - fk));
                    fk = ns;
                }
                f[k] = fk;
            }
            if (lane == 0 && has_prev)
                fstart = (kp >= (unsigned int)ns) ? ns : (int)kp + (rbuf32[kp - 4u * blk0] <= frp ? 1 : 0);
            __syncwarp();  // the window is reused for the offspring below
        }
    }
    if (!coop) {
#pragma unroll
        for (int k = 0; k < WS_SCAN_ITEMS; ++k) {
            const int gi = item0 + k;
            int fk;
            if (gi >= n) {
                fk = -1;  // patched below
            } else {
                if (EXACT_FP) fk = (int)ws_F(P, ws_fxs_to_double(C[k], X.fx_scale), inv_n, su);
                else if (MN) fk = ws_F_mn(P, C[k]);
                else fk = ws_F_int(C[k], (unsigned int)ns, sh, rmask, su.scheme, r0_int, P.seed, P.stream);
                if (gi == n - 1 && P.last_rank) {
                    if (fk < ns) atomicAdd(P.n_clamped, (unsigned long long)(ns - fk));
                    fk = ns;  // leftover slots go to the last particle (the reference would throw BoundsError)
                }
            }
            f[k] = fk;
        }
        if (lane == 0 && has_prev) {
            if (EXACT_FP) fstart = (int)ws_F(P, ws_fxs_to_double(Cp, X.fx_scale), inv_n, su);
            else if (MN) fstart = ws_F_mn(P, Cp);
            else fstart = ws_F_int(Cp, (unsigned int)ns, sh, rmask, su.scheme, r0_int, P.seed, P.stream);
        }
    }
    // the other paths use the whole window for their slot uniforms, the ring's half included
    if (ring != nullptr && !ringed) ring->lo = ring->hi = 0u;
    // items beyond the shard produce nothing: they repeat the F of the shard's last particle
    if (!interior) {
        const int rank_end = P.bounds != nullptr ? P.bounds[1] : ns;
#pragma unroll
        for (int k = 0; k < WS_SCAN_ITEMS; ++k)
            if (f[k] < 0) f[k] = rank_end;
    }
    fstart = __shfl_sync(0xffffffffu, fstart, 0);
    int f_prev = __shfl_up_sync(0xffffffffu, f[WS_SCAN_ITEMS - 1], 1);
    if (lane == 0) f_prev = fstart;
    const int fend = __shfl_sync(0xffffffffu, f[WS_SCAN_ITEMS - 1], 31);

    if (fend - fstart > WS_HEAVY_TILE_SLOTS) {
        // a few particles own a huge share of the offspring: publish the tile's F table and let
        // ws_expand_heavy_kernel fill its slots with the whole grid
        unsigned int slot = 0;
        if (lane == 0) slot = atomicAdd(P.heavy_count, 1u);
        slot = __shfl_sync(0xffffffffu, slot, 0);
        int32_t* dst = P.heavy_F + (size_t)slot * (WS_SCAN_TILE + 2);
#pragma unroll
        for (int k = 0; k < WS_SCAN_ITEMS; ++k) dst[lane * WS_SCAN_ITEMS + k] = f[k];
        if (lane == 0) {
            dst[WS_SCAN_TILE] = fstart;
            dst[WS_SCAN_TILE + 1] = tile_base / WS_SCAN_TILE;
        }
        return;
    }

    // ---- expand: offspring slots [F(C_{m-1}), F(C_m)) of particle m ---------------------------------
    constexpr int PL = WS_EXPAND_LANE, PR = 32 * PL, Q = PL / 4;
    if (fend - fstart + 3 <= PR) {
        // the common case (a tile of near-uniform weights has ~256 slots): the tile's slots, behind up to 3 slots of
        // padding, fit one round of PL consecutive slots per lane.  Every particle with offspring marks the FIRST of its
        // slots with its index (one predicated store, no divergence on the family size); the other slots take the last
        // mark before them (a running maximum: marks increase with the slot, -1 = no mark), written as 16-byte stores.
        int32_t* const gdst = P.ancestors + (fstart - slot_base);
        const int pad = (int)((reinterpret_cast<uintptr_t>(gdst) >> 2) & 3u);  // window starts 16-byte aligned in global memory
        const int W = fend - fstart + pad;
        int4* const w4 = reinterpret_cast<int4*>(out_s);
#pragma unroll
        for (int j = 0; j < Q; ++j) w4[j * 32 + lane] = make_int4(-1, -1, -1, -1);
        __syncwarp();
        {
            int lo = f_prev;
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS; ++k) {
                const int hi = f[k];
                if (hi > lo) out_s[lo - fstart + pad] = item0 + k;
                lo = hi;
            }
        }
        __syncwarp();
        int32_t* const dst = gdst - pad;
        {
            int mk[PL];
#pragma unroll
            for (int j = 0; j < Q; ++j) {
                const int4 v = w4[lane * Q + j];
                mk[4 * j] = v.x;
                mk[4 * j + 1] = v.y;
                mk[4 * j + 2] = v.z;
                mk[4 * j + 3] = v.w;
            }
#pragma unroll
            for (int j = 1; j < PL; ++j) mk[j] = max(mk[j], mk[j - 1]);
            int incl = mk[PL - 1];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl = max(incl, t);
            }
            int excl = __shfl_up_sync(0xffffffffu, incl, 1);
            if (lane == 0) excl = -1;
#pragma unroll
            for (int j = 0; j < PL; ++j) mk[j] = max(mk[j], excl);
            const int p0 = lane * PL;
            if (p0 >= pad && p0 + PL <= W) {
#pragma unroll
                for (int j = 0; j < Q; ++j)
                    *reinterpret_cast<int4*>(dst + p0 + 4 * j) = make_int4(mk[4 * j], mk[4 * j + 1], mk[4 * j + 2], mk[4 * j + 3]);
            } else {
#pragma unroll
                for (int j = 0; j < PL; ++j)
                    if (p0 + j >= pad && p0 + j < W) dst[p0 + j] = mk[j];
            }
        }
        __syncwarp();
        return;
    }
    // does this lane own a family too large for one lane?
    bool has_big = false;
    {
        int lo = f_prev;
#pragma unroll
        for (int k = 0; k < WS_SCAN_ITEMS; ++k) {
            if (f[k] - lo > WS_DIRECT_MAX) has_big = true;
            lo = f[k];
        }
    }
    const unsigned big_mask = __ballot_sync(0xffffffffu, has_big);
    for (int chunk = fstart; chunk < fend; chunk += WS_EXPAND_CHUNK) {
        const int chunk_end = min(chunk + WS_EXPAND_CHUNK, fend);
        {
            int lo = f_prev;
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS; ++k) {
                const int hi = f[k];
                if (hi - lo <= WS_DIRECT_MAX) {
                    const int a = max(lo, chunk), e = min(hi, chunk_end);
                    for (int pos = a; pos < e; ++pos) out_s[pos - chunk] = item0 + k;
                }
                lo = hi;
            }
        }
        unsigned bm = big_mask;
        while (bm != 0u) {
            const int src = __ffs(bm) - 1;
            bm &= bm - 1u;
            int lo = __shfl_sync(0xffffffffu, f_prev, src);
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS; ++k) {
                const int hi = __shfl_sync(0xffffffffu, f[k], src);
                if (hi - lo > WS_DIRECT_MAX) {
                    const int a = max(lo, chunk), e = min(hi, chunk_end);
                    const int anc = tile_base + src * WS_SCAN_ITEMS + k;
                    for (int pos = a + lane; pos < e; pos += 32) out_s[pos - chunk] = anc;
                }
                lo = hi;
            }
        }
        __syncwarp();
        for (int pos = chunk + lane; pos < chunk_end; pos += 32) P.ancestors[pos - slot_base] = out_s[pos - chunk];
        __syncwarp();
    }
}

#ifndef WS_SEARCH_ASYNC
#define WS_SEARCH_ASYNC 1   // next tile's CDF by cp.async into shared memory while this one is searched (1) or loaded when needed (0)
#endif
#ifndef WS_SEARCH_MINB
#define WS_SEARCH_MINB 3   // (4 CTAs per SM fit the 48 KB of shared memory, but at 64 registers the kernel spills and measured slower)
#endif
#ifndef WS_SEARCH_GRID
#define WS_SEARCH_GRID 3   // CTAs per SM launched: persistent warps, each pipelining its tiles (next tile requested while this one is searched)
#endif
// A gated step that does not fire (ws_resample_async): the search-type kernels leave the identity in the ancestor
// vector themselves (single-GPU states: slot i <- particle i) instead of a separate launch.
__device__ __forceinline__ bool ws_gate_closed_identity(const WsScanParams& P) {
    if (P.gate == 0 || P.red->do_resample != 0) return false;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < P.n; i += stride) P.ancestors[i] = (int32_t)i;
    return true;
}
#define WS_SEARCH_SMEM_BYTES ((WS_WARPS_PER_CTA * WS_RBUF_SLOTS + WS_CDF_TILE) * 8)
template <bool EXACT_FP, bool MN, bool SHR>
__global__ void __launch_bounds__(WS_SCAN_BLOCK, WS_SEARCH_MINB) ws_search_kernel(const __grid_constant__ WsScanParams P) {
    if (ws_gate_closed_identity(P)) return;

    // per-warp window: first the slot uniforms of the tile's slot range (Philox mode), then the staged offspring;
    // behind the windows, per warp, the tile-local CDF of the warp's NEXT tile, copied asynchronously while the current
    // one is searched (the kernel was waiting on these loads: profiles/r2m_ncu_ws_search_kernel_20M.txt).  The upper half
    // of a window, above the offspring staging, holds the warp's Philox ring (WsRing) while the ring is in use.
    extern __shared__ __align__(16) unsigned long long search_smem[];
    static_assert(WS_RBUF_SLOTS * 8 >= (WS_EXPAND_CHUNK + 128) * 4 && (WS_RBUF_SLOTS * 8) % 16 == 0, "window too small for the offspring staging");
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long* const rbuf = search_smem + warp * WS_RBUF_SLOTS;
    ulonglong2* const cbuf = reinterpret_cast<ulonglong2*>(search_smem + WS_WARPS_PER_CTA * WS_RBUF_SLOTS + warp * WS_SCAN_TILE) + lane;

    const unsigned long long cdf_offset = ws_cdf_offset(P);
    WsSearchCtx X;
    ws_search_setup(P, X);
    const int n = X.n;
    const int n_tiles = (n + WS_SCAN_TILE - 1) / WS_SCAN_TILE;
    const int n_ctiles = (n + WS_CDF_TILE - 1) / WS_CDF_TILE;
    const int warps_total = gridDim.x * WS_WARPS_PER_CTA;

#if WS_SEARCH_ASYNC
    // what a tile needs from memory besides its CDF values: the lane's word of the tile-offset sum (ws_tile_offset) and
    // the local CDF of the particle in front of the tile (lane 0; zero when that particle closes the previous CDF tile:
    // its global CDF is then exactly this tile's offset)
    unsigned long long ow = 0ull, pw = 0ull;
    auto request = [&](int tile) {
        const int tile_base = tile * WS_SCAN_TILE;
        const int ct = tile_base / WS_CDF_TILE;
        if (tile_base + WS_SCAN_TILE <= n) {
            const ulonglong2* p2 = reinterpret_cast<const ulonglong2*>(P.cdf_local + tile_base + lane * WS_SCAN_ITEMS);
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS / 2; ++k) ws_cp_async16(cbuf + k * 32, p2 + k);
        }
        ws_cp_async_commit();
        const int idx = (ct / WS_TILE_GROUP) * WS_TILE_GROUP + lane;
        ow = idx < ct ? __ldg(P.tile_words + idx) : 0ull;
        if (lane == 31) ow = __ldg(P.tile_words + n_ctiles + ct / WS_TILE_GROUP);   // (32 g + 31 >= ct: the lane is free for the group's prefix)
        pw = (lane == 0 && tile_base % WS_CDF_TILE != 0) ? __ldg(P.cdf_local + tile_base - 1) : 0ull;
    };
    // every warp searches a run of consecutive tiles, so that the Philox blocks at the end of one tile's slot range are
    // still in the warp's ring when the next tile starts
    static_assert(WS_EXPAND_CHUNK * 4 + WS_RING_BLOCKS * 16 <= WS_RBUF_SLOTS * 8 && 32 * WS_EXPAND_LANE <= WS_EXPAND_CHUNK,
                  "the ring and the offspring staging share a window");
    WsRing ring{reinterpret_cast<uint4*>(rbuf + WS_EXPAND_CHUNK / 2), 0u, 0u};
    const int per_warp = (n_tiles + warps_total - 1) / warps_total;
    int tile = (blockIdx.x * WS_WARPS_PER_CTA + warp) * per_warp;
    const int tile_end = min(tile + per_warp, n_tiles);
    if (tile < tile_end) request(tile);
    for (; tile < tile_end; ++tile) {
        const int tile_base = tile * WS_SCAN_TILE;
        const int item0 = tile_base + lane * WS_SCAN_ITEMS;
        // global fixed-point CDF of the lane's 8 consecutive particles
        unsigned long long C[WS_SCAN_ITEMS];
        ws_cp_async_wait_all();
        if (tile_base + WS_SCAN_TILE <= n) {
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS / 2; ++k) {
                const ulonglong2 v = cbuf[k * 32];
                C[2 * k] = v.x;
                C[2 * k + 1] = v.y;
            }
        } else {
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS; ++k) C[k] = (item0 + k < n) ? __ldg(P.cdf_local + item0 + k) : 0ull;
        }
        unsigned long long off = ow;
        const unsigned long long pl = pw;
        if (tile + 1 < tile_end) request(tile + 1);   // (the lane's slots of cbuf were read above)
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) off += __shfl_xor_sync(0xffffffffu, off, d);
        off += cdf_offset;
        if (tile_base + WS_SCAN_TILE <= n) {
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS; ++k) C[k] += off;
        } else {
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS; ++k) C[k] = (item0 + k < n) ? off + C[k] : 0ull;
        }
        ws_search_warp_tile<EXACT_FP, MN, SHR>(P, X, rbuf, lane, tile_base, C, off + pl, tile != 0,
                                               WS_INTERIOR_FAST && tile_base + WS_SCAN_TILE < n, &ring);
    }
#else
    for (int tile = blockIdx.x * WS_WARPS_PER_CTA + warp; tile < n_tiles; tile += warps_total) {
        const int tile_base = tile * WS_SCAN_TILE;
        const int item0 = tile_base + lane * WS_SCAN_ITEMS;
        const int ct = tile_base / WS_CDF_TILE;
        const unsigned long long offset = cdf_offset + ws_tile_offset(P, n_ctiles, ct, lane);

        // global fixed-point CDF of the lane's 8 consecutive particles
        unsigned long long C[WS_SCAN_ITEMS];
        if (item0 + WS_SCAN_ITEMS <= n) {
            const ulonglong2* p2 = reinterpret_cast<const ulonglong2*>(P.cdf_local + item0);
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS / 2; ++k) {
                ulonglong2 v = __ldg(p2 + k);
                C[2 * k] = offset + v.x;
                C[2 * k + 1] = offset + v.y;
            }
        } else {
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS; ++k) C[k] = (item0 + k < n) ? offset + __ldg(P.cdf_local + item0 + k) : 0ull;
        }
        unsigned long long Cp = 0ull;
        if (lane == 0 && tile != 0) {
            const int p = tile_base - 1;
            // (the particle in front of the first warp tile of a CDF tile lies in the previous CDF tile)
            Cp = (p / WS_CDF_TILE == ct ? offset : offset - __ldg(P.tile_words + ct - 1)) + __ldg(P.cdf_local + p);
        }
        ws_search_warp_tile<EXACT_FP, MN, SHR>(P, X, rbuf, lane, tile_base, C, Cp, tile != 0,
                                               WS_INTERIOR_FAST && tile_base + WS_SCAN_TILE < n);
    }
#endif
}

// ---- CDF + search in ONE pass (single-GPU states) ---------------------------------------------------
// A CTA takes the next tile of WS_CDF_TILE particles from an atomic ticket (tiles start in ticket order, so every
// predecessor of a running tile is running or done: the look-back below cannot wait on a tile that has not been
// scheduled), forms the tile's fixed-point weights and their local prefix sums in registers, publishes the tile
// aggregate, obtains its exclusive prefix by a decoupled look-back over the predecessors' status words (one warp,
// 32 predecessors per poll; flag and value travel in the same 64-bit word, so no fence is needed) and goes straight
// on to the search / offspring expansion of its eight warp tiles.  Nothing but the log-weights is read (8 B) and
// nothing but the ancestors written (4 B): the three-pass form's 16 B round trip through cdf_local is gone, and
// the CDF — integer sums — is bit-identical to it.
#ifndef WS_FUSED_MINB
#define WS_FUSED_MINB 3
#endif
template <bool EXACT_FP>
__global__ void __launch_bounds__(WS_SCAN_BLOCK, WS_FUSED_MINB) ws_scan_search_kernel(const __grid_constant__ WsScanParams P) {
    if (ws_gate_closed_identity(P)) return;
    __shared__ __align__(16) unsigned long long win_all[WS_WARPS_PER_CTA][WS_RBUF_SLOTS];
    __shared__ unsigned long long warp_tot[WS_WARPS_PER_CTA];
    __shared__ unsigned long long s_prefix;
    __shared__ unsigned long long lb_sum[WS_WARPS_PER_CTA];
    __shared__ int lb_found[WS_WARPS_PER_CTA];
    __shared__ int s_tile;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_tile = (int)atomicAdd(P.tile_counter, 1u);
    WsSearchCtx X;
    ws_search_setup(P, X);
    const int n = X.n;
    double m = 0.0, Sden = 1.0;
    if (P.mode == 0) {
        m = P.red->m;
        Sden = P.red->S;  // w = e / S as exp_norm does (correctly rounded quotient, see ws_div_pos)
    }
    const double rS = 1.0 / Sden;
    __syncthreads();
    const int tile = s_tile;
    const int item0 = tile * WS_CDF_TILE + threadIdx.x * WS_SCAN_ITEMS;

    // ---- fixed-point weights of the thread's 8 consecutive particles, inclusive sums ----
    unsigned long long q[WS_SCAN_ITEMS];
    if (P.mode == 2) {
        const unsigned long long qu = ws_w_to_fxs(1.0 / (double)P.n_slots, P.fx_scale);
#pragma unroll
        for (int k = 0; k < WS_SCAN_ITEMS; ++k) q[k] = (item0 + k < n) ? qu : 0ull;
    } else {
        double l[WS_SCAN_ITEMS];
        if (item0 + WS_SCAN_ITEMS <= n) {
            const double2* p2 = reinterpret_cast<const double2*>(P.logw + item0);
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS / 2; ++k) {
                const double2 v = __ldg(p2 + k);
                l[2 * k] = v.x;
                l[2 * k + 1] = v.y;
            }
        } else {
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS; ++k) l[k] = (item0 + k < n) ? __ldg(P.logw + item0 + k) : -INFINITY;
        }
#pragma unroll
        for (int k = 0; k < WS_SCAN_ITEMS; ++k) {
            double w;
            if (P.mode == 0) w = ws_div_pos(ws_exp_nonpos(l[k] - m), Sden, rS);
            else w = (item0 + k < n) ? l[k] : 0.0;
            q[k] = (item0 + k < n) ? ws_w_to_fxs(w, P.fx_scale) : 0ull;
        }
    }
#pragma unroll
    for (int k = 1; k < WS_SCAN_ITEMS; ++k) q[k] += q[k - 1];
    const unsigned long long thread_total = q[WS_SCAN_ITEMS - 1];
    unsigned long long incl = thread_total;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += t;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    unsigned long long warp_excl = 0ull, tile_agg = 0ull;
#pragma unroll
    for (int w = 0; w < WS_WARPS_PER_CTA; ++w) {
        const unsigned long long t = warp_tot[w];
        if (w < warp) warp_excl += t;
        tile_agg += t;
    }

    // ---- decoupled look-back, by the whole CTA: thread t inspects predecessor tile - 1 - t, so one round covers
    // 256 predecessors (with one warp, a tile walked back through up to ~450 tiles in flight, 32 per ~1 us round,
    // while the other seven warps waited at the barrier) ----
    if (tile == 0) {
        if (threadIdx.x == 0) {
            st_relaxed_u64(P.tile_words, (WS_TILE_INCL << 62) | tile_agg);
            s_prefix = 0ull;
        }
    } else {
        if (threadIdx.x == 0) st_relaxed_u64(P.tile_words + tile, (WS_TILE_AGG << 62) | tile_agg);
        unsigned long long excl = 0ull;  // CTA-uniform
        int look = tile - 1;
        while (true) {
            const int idx = look - (int)threadIdx.x;
            unsigned long long word;
            do {
                word = (idx >= 0) ? ld_relaxed_u64(P.tile_words + idx) : (WS_TILE_INCL << 62);
            } while (__any_sync(0xffffffffu, (word >> 62) == 0ull));
            const unsigned incl_mask = __ballot_sync(0xffffffffu, (word >> 62) == WS_TILE_INCL);
            const int first = incl_mask != 0u ? __ffs(incl_mask) - 1 : 31;
            unsigned long long v = (lane <= first) ? (word & WS_FXS_MASK) : 0ull;
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
            __syncthreads();  // lb_* of the previous round (and warp_tot) have been consumed
            if (lane == 0) {
                lb_sum[warp] = v;
                lb_found[warp] = incl_mask != 0u ? 1 : 0;
            }
            __syncthreads();
            bool found = false;
#pragma unroll
            for (int w = 0; w < WS_WARPS_PER_CTA; ++w) {
                if (!found) {
                    excl += lb_sum[w];
                    found = lb_found[w] != 0;
                }
            }
            if (found) break;
            look -= WS_SCAN_BLOCK;
        }
        if (threadIdx.x == 0) {
            st_relaxed_u64(P.tile_words + tile, (WS_TILE_INCL << 62) | (excl + tile_agg));
            s_prefix = excl;
        }
    }
    __syncthreads();
    const unsigned long long prefix = P.cdf_offset + s_prefix;

    // ---- search: the thread's CDF values are exactly what ws_search_kernel would have read back ----
    unsigned long long C[WS_SCAN_ITEMS];
    const unsigned long long thread_excl = prefix + warp_excl + (incl - thread_total);
#pragma unroll
    for (int k = 0; k < WS_SCAN_ITEMS; ++k) C[k] = (item0 + k < n) ? thread_excl + q[k] : 0ull;
    const int warp_base = tile * WS_CDF_TILE + warp * WS_SCAN_TILE;
    if (warp_base < n) ws_search_warp_tile<EXACT_FP, false>(P, X, win_all[warp], lane, warp_base, C, prefix + warp_excl, warp_base != 0);
}

// ---- CDF + search in ONE pass, look-back deferred by one tile ("chain") ------------------------------------------
// The single-pass kernel above loses to the three passes because a tile looks back right after publishing its own
// aggregate, i.e. while the ~40 predecessors that started together with it are still forming theirs.  Here a CTA is
// persistent and keeps TWO tiles in flight: it forms the fixed-point weights and local sums of tile t1 (phase 1,
// FP64), publishes t1's aggregate, and only then looks back for the tile t0 it took one round earlier and runs t0's
// search / expansion (phase 2, integer) from sums parked in shared memory.  By then every predecessor of t0 —
// ticketed before t0, published one phase earlier — is visible, so the look-back is one poll, not a spin.  Depth is
// bounded by a second level: tiles form groups of WS_CHAIN_GROUP; a tile adds its aggregate to its group's two
// accumulators (low / high 31 bits, each with a tile count in its top bits: one fire-and-forget atomic each, no fence,
// no return value), the first tile of a group publishes the group's exclusive prefix, and a look-back reads at most
// 31 tile words (warp 0) and a few group words (warp 1).  Integer sums: ancestors are bit-identical to the other forms.
#define WS_CHAIN_GROUP WS_TILE_GROUP
#ifndef WS_CHAIN_MINB
#define WS_CHAIN_MINB 3
#endif
#ifndef WS_CHAIN_MAXREG
#define WS_CHAIN_MAXREG 80    // 65 536 / (WS_CHAIN_MINB x 256 threads) = 85, whatever the CTA size (ptxas does not derive it from small CTAs)
#endif
#define WS_CHAIN_CNT_SHIFT 40
#define WS_CHAIN_PART_MASK ((1ull << WS_CHAIN_CNT_SHIFT) - 1ull)
#define WS_CHAIN_SMEM_BYTES(BLOCK) ((((BLOCK) / 32) * WS_RBUF_SLOTS + 2 * (BLOCK) * WS_SCAN_ITEMS) * 8)
#define WS_CHAIN_MIN_TILE (32 * WS_SCAN_ITEMS)   // smallest chain tile (one warp per CTA): sizes the tile words

size_t ws_scan_words(int64_t n) {
    const int64_t n_tiles = (n + WS_CHAIN_MIN_TILE - 1) / WS_CHAIN_MIN_TILE;
    const int64_t n_groups = (n_tiles + WS_CHAIN_GROUP - 1) / WS_CHAIN_GROUP;
    return (size_t)(n_tiles + 3 * n_groups + 2);
}

template <bool EXACT_FP, int BLOCK>
__global__ void __maxnreg__(WS_CHAIN_MAXREG) ws_chain_kernel(const __grid_constant__ WsScanParams P) {
    constexpr int TILE = BLOCK * WS_SCAN_ITEMS;   // particles per chain tile
    constexpr int WARPS = BLOCK / 32;
    constexpr int GRP_WARP = WARPS > 1 ? 1 : 0;    // the warp that looks back over the groups (warp 0: the tiles of its own group)
    if (ws_gate_closed_identity(P)) return;
    extern __shared__ __align__(16) unsigned long long chain_smem[];
    __shared__ unsigned long long warp_tot[WARPS];
    __shared__ unsigned long long s_wexcl[WARPS];
    __shared__ unsigned long long lb_part[2];
    __shared__ int s_tile;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned long long* const win = chain_smem + warp * WS_RBUF_SLOTS;
    // parked tile-local CDF of the deferred tile: [WS_SCAN_ITEMS / 2][BLOCK] 16-byte words, thread-private slots
    ulonglong2* const stash = reinterpret_cast<ulonglong2*>(chain_smem + WARPS * WS_RBUF_SLOTS) + tid;
    // log-weights of the tile after next, copied asynchronously while this round computes (same layout, thread-private)
    double2* const lbuf = reinterpret_cast<double2*>(chain_smem + WARPS * WS_RBUF_SLOTS + TILE) + tid;
    const int n = (int)P.n;
    const int n_tiles = (n + TILE - 1) / TILE;
    const int n_groups = (n_tiles + WS_CHAIN_GROUP - 1) / WS_CHAIN_GROUP;
    unsigned long long* const grp_lo = P.tile_words + n_tiles;
    unsigned long long* const grp_hi = grp_lo + n_groups;
    unsigned long long* const grp_incl = grp_hi + n_groups;
    WsSearchCtx X;
    ws_search_setup(P, X);
    double m = 0.0, Sden = 1.0;
    if (P.mode == 0) {
        m = P.red->m;
        Sden = P.red->S;
    }
    const double rS = 1.0 / Sden;
    const double uniform_w = 1.0 / (double)P.n_slots;
    // a full tile's log-weights are prefetched; the ragged last tile is loaded with guards when its turn comes
    auto prefetch = [&](int tile) {
        if (P.mode != 2 && tile < n_tiles && (tile + 1) * TILE <= n) {
            const double2* p2 = reinterpret_cast<const double2*>(P.logw + (size_t)tile * TILE + tid * WS_SCAN_ITEMS);
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS / 2; ++k) ws_cp_async16(lbuf + k * BLOCK, p2 + k);
        }
        ws_cp_async_commit();
    };
    if (tid == 0) s_tile = (int)atomicAdd(P.tile_counter, 1u);
    __syncthreads();
    int t1 = s_tile;
    prefetch(t1);
    __syncthreads();  // s_tile has been read by everybody
    int t0 = -1;
    while (true) {
        const bool have1 = t1 < n_tiles;
        if (tid == 0) s_tile = (int)atomicAdd(P.tile_counter, 1u);  // the tile after t1: known to all after the next barrier
        // the look-back words of t0 are requested now and looked at after phase 1 of t1: their latency is off the
        // path between the two barriers (they are polled again there if a predecessor was late)
        unsigned long long lbt = 0ull, lbw0 = 0ull, lbw1 = 0ull, lbw2 = 0ull;
        if (t0 >= 0) {
            const int g0 = t0 / WS_CHAIN_GROUP;
            if (warp == 0) {
                const int idx = g0 * WS_CHAIN_GROUP + lane;
                if (idx < t0) lbt = ld_relaxed_u64(P.tile_words + idx);
            }
            if (warp == GRP_WARP) {
                const int gi = g0 - 1 - lane;
                if (gi >= 0) {
                    lbw0 = ld_relaxed_u64(grp_incl + gi);
                    lbw1 = ld_relaxed_u64(grp_lo + gi);
                    lbw2 = ld_relaxed_u64(grp_hi + gi);
                }
            }
        }
        // ---- phase 1 of t1: fixed-point weights, inclusive sums within the thread, then within the warp ----
        unsigned long long q[WS_SCAN_ITEMS];
        unsigned long long incl = 0ull, thread_total = 0ull;
        if (have1) {
            const int base = t1 * TILE;
            const int item0 = base + tid * WS_SCAN_ITEMS;
            if (P.mode == 2) {
                const unsigned long long qu = ws_w_to_fxs(uniform_w, P.fx_scale);
#pragma unroll
                for (int k = 0; k < WS_SCAN_ITEMS; ++k) q[k] = (item0 + k < n) ? qu : 0ull;
            } else {
                double l[WS_SCAN_ITEMS];
                if (base + TILE <= n) {
                    ws_cp_async_wait_all();
#pragma unroll
                    for (int k = 0; k < WS_SCAN_ITEMS / 2; ++k) {
                        const double2 v = lbuf[k * BLOCK];
                        l[2 * k] = v.x;
                        l[2 * k + 1] = v.y;
                    }
                } else {
                    const double pad = (P.mode == 0) ? -INFINITY : 0.0;
#pragma unroll
                    for (int k = 0; k < WS_SCAN_ITEMS; ++k) l[k] = (item0 + k < n) ? __ldg(P.logw + item0 + k) : pad;
                }
                if (P.mode == 0) {
                    // e <= 1 and S >= 1, so w in [0, 1] or NaN: the saturating conversion (NaN -> 0) is ws_w_to_fxs
                    // without its two compares
#pragma unroll
                    for (int k = 0; k < WS_SCAN_ITEMS; ++k)
                        q[k] = __double2ull_rn(ws_div_pos(ws_exp_nonpos(l[k] - m), Sden, rS) * P.fx_scale);
                } else {
#pragma unroll
                    for (int k = 0; k < WS_SCAN_ITEMS; ++k) q[k] = ws_w_to_fxs(l[k], P.fx_scale);
                }
            }
#pragma unroll
            for (int k = 1; k < WS_SCAN_ITEMS; ++k) q[k] += q[k - 1];
            thread_total = q[WS_SCAN_ITEMS - 1];
            incl = thread_total;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl += t;
            }
            if (lane == 31) warp_tot[warp] = incl;
        }
        __syncthreads();
        const int t2 = s_tile;
        prefetch(t2);  // (the thread's parking slots in lbuf were consumed above)
        // ---- swap: take the deferred tile's sums out of the parking slots, park t1's ----
        unsigned long long C0[WS_SCAN_ITEMS];
        unsigned long long wexcl0 = 0ull;
        if (t0 >= 0) {
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS / 2; ++k) {
                const ulonglong2 v = stash[k * BLOCK];
                C0[2 * k] = v.x;
                C0[2 * k + 1] = v.y;
            }
            wexcl0 = s_wexcl[warp];
        }
        __syncwarp();
        if (have1) {
            unsigned long long warp_excl = 0ull, tile_agg = 0ull;
#pragma unroll
            for (int w = 0; w < WARPS; ++w) {
                const unsigned long long t = warp_tot[w];
                if (w < warp) warp_excl += t;
                tile_agg += t;
            }
            if (tid == 0) {
                st_relaxed_u64(P.tile_words + t1, (WS_TILE_AGG << 62) | tile_agg);
                const int g = t1 / WS_CHAIN_GROUP;
                atomicAdd(grp_lo + g, (1ull << WS_CHAIN_CNT_SHIFT) | (tile_agg & 0x7FFFFFFFull));
                atomicAdd(grp_hi + g, (1ull << WS_CHAIN_CNT_SHIFT) | (tile_agg >> 31));
            }
            const unsigned long long thread_excl = warp_excl + (incl - thread_total);
#pragma unroll
            for (int k = 0; k < WS_SCAN_ITEMS / 2; ++k)
                stash[k * BLOCK] = make_ulonglong2(thread_excl + q[2 * k], thread_excl + q[2 * k + 1]);
            if (lane == 0) s_wexcl[warp] = warp_excl;
        }
        if (t0 >= 0) {
            // ---- look-back for t0: tiles of its own group (warp 0), whole groups before it (warp 1) ----
            const int g0 = t0 / WS_CHAIN_GROUP;
            if (warp == 0) {
                const int idx = g0 * WS_CHAIN_GROUP + lane;
                unsigned long long v = 0ull;
                if (idx < t0) {
                    unsigned long long word = lbt;
                    while ((word >> 62) == 0ull) word = ld_relaxed_u64(P.tile_words + idx);
                    v = word & WS_FXS_MASK;
                }
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
                if (lane == 0) lb_part[0] = v;
            }
            if (warp == GRP_WARP) {
                unsigned long long acc = 0ull;
                int look = g0 - 1;
                bool fresh = true;   // first round, first look: the words requested at the top of the iteration
                while (true) {
                    const int gi = look - lane;
                    unsigned long long v;
                    bool has_incl;
                    unsigned int first;
                    while (true) {
                        bool ready = true;
                        has_incl = true;
                        v = 0ull;
                        if (gi >= 0) {
                            const unsigned long long inc = fresh ? lbw0 : ld_relaxed_u64(grp_incl + gi);
                            const unsigned long long lo = fresh ? lbw1 : ld_relaxed_u64(grp_lo + gi);
                            const unsigned long long hi = fresh ? lbw2 : ld_relaxed_u64(grp_hi + gi);
                            has_incl = (inc >> 62) == WS_TILE_INCL;
                            if (has_incl) {
                                v = inc & WS_FXS_MASK;
                            } else {
                                ready = (lo >> WS_CHAIN_CNT_SHIFT) == WS_CHAIN_GROUP && (hi >> WS_CHAIN_CNT_SHIFT) == WS_CHAIN_GROUP;
                                v = ((hi & WS_CHAIN_PART_MASK) << 31) + (lo & WS_CHAIN_PART_MASK);
                            }
                        }
                        fresh = false;
                        const unsigned int incl_mask = __ballot_sync(0xffffffffu, has_incl);
                        const unsigned int wait_mask = __ballot_sync(0xffffffffu, !ready);
                        first = incl_mask != 0u ? (unsigned int)(__ffs(incl_mask) - 1) : 32u;
                        const unsigned int need = first >= 31u ? 0xFFFFFFFFu : ((2u << first) - 1u);
                        if ((wait_mask & need) == 0u) break;
                    }
                    if ((unsigned int)lane > first) v = 0ull;
#pragma unroll
                    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
                    acc += v;
                    if (first < 32u) break;
                    look -= 32;
                }
                if (lane == 0) {
                    lb_part[1] = acc;
                    // the first tile of a group hands the group's exclusive prefix to everybody behind it
                    if (g0 > 0 && t0 == g0 * WS_CHAIN_GROUP) st_relaxed_u64(grp_incl + (g0 - 1), (WS_TILE_INCL << 62) | acc);
                }
            }
        }
        __syncthreads();  // look-back result; s_tile and warp_tot have been read by everybody
        if (t0 >= 0) {
            // ---- phase 2 of t0: search + offspring expansion, one warp tile per warp ----
            const unsigned long long prefix = P.cdf_offset + lb_part[0] + lb_part[1];
            {
                const int item0 = t0 * TILE + tid * WS_SCAN_ITEMS;
#pragma unroll
                for (int k = 0; k < WS_SCAN_ITEMS; ++k) C0[k] = (item0 + k < n) ? prefix + C0[k] : 0ull;
            }
            const int warp_base = t0 * TILE + warp * WS_SCAN_TILE;
            if (warp_base < n)
                ws_search_warp_tile<EXACT_FP, false>(P, X, win, lane, warp_base, C0, prefix + wexcl0, warp_base != 0,
                                                     WS_INTERIOR_FAST && warp_base + WS_SCAN_TILE < n);
        }
        if (!have1) break;
        t0 = t1;
        t1 = t2;
    }
    ws_cp_async_wait_all();
}

// ---- small particle sets: the whole Resample step in ONE kernel --------------------------------------------------
// Below WS_SMALL_N particles a step is launch-latency bound: finalize, two memsets, tile CDF, offsets, search, heavy
// expansion and the identity fill are eight stream operations of a few microseconds each.  One CTA does all of it:
// the (m, S, Q) combination and the decision (those of ws_finalize_kernel: same order, same bits), the
// fixed-point CDF in chunks with a running carry, F(C_m) per particle through the same ws_F_int, and the expansion by a
// binary search of every slot in the F table.  Ancestors are bit-identical to the large-N kernels (integer sums).
__global__ void __launch_bounds__(256) ws_resample_small_kernel(const __grid_constant__ WsScanParams P, const WsLse* __restrict__ partials,
                                                                int n_partials, double ess_perc_min, WsReduceOut* __restrict__ out,
                                                                unsigned long long* ties, int do_finalize, int32_t* __restrict__ Ftab) {
    __shared__ WsLse warp_scratch[8];
    __shared__ unsigned long long warp_tot[8];
    __shared__ unsigned long long s_carry;
    __shared__ int s_fire;
    __shared__ int32_t Fs[WS_SMALL_N];   // F(C_m) of every particle: the expansion searches it 12 steps per slot
    (void)Ftab;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (do_finalize) {
        const WsLse tot = lse_block_combine<256>(partials, n_partials, warp_scratch);
        if (threadIdx.x == 0) {
            ws_decide(tot, P.n_slots, ess_perc_min, out, ties);
            __threadfence_block();
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        s_fire = (P.gate == 0 || out->do_resample != 0) ? 1 : 0;
        s_carry = 0ull;
    }
    __syncthreads();
    const int n = (int)P.n, ns = (int)P.n_slots;
    if (!s_fire) {
        for (int i = threadIdx.x; i < n; i += 256) P.ancestors[i] = i;   // a step that does not fire: the identity
        return;
    }
    const double m = out->m, Sden = out->S, rS = 1.0 / out->S;
    const int sh = P.fx_shift - 32;
    const unsigned int rmask = sh >= 0 ? 0xFFFFFFFFu : ~((1u << (-sh)) - 1u);
    unsigned int r0 = 0u;
    if (P.scheme == 1) r0 = ws_philox4x32_10(0ull, P.stream, P.seed).x;
    for (int base = 0; base < n; base += 256 * WS_SCAN_ITEMS) {
        const int item0 = base + threadIdx.x * WS_SCAN_ITEMS;
        unsigned long long q[WS_SCAN_ITEMS];
#pragma unroll
        for (int k = 0; k < WS_SCAN_ITEMS; ++k) {
            const int i = item0 + k;
            q[k] = (i < n) ? ws_w_to_fxs(ws_div_pos(ws_exp_nonpos(P.logw[i] - m), Sden, rS), P.fx_scale) : 0ull;
        }
#pragma unroll
        for (int k = 1; k < WS_SCAN_ITEMS; ++k) q[k] += q[k - 1];
        const unsigned long long thread_total = q[WS_SCAN_ITEMS - 1];
        unsigned long long incl = thread_total;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += t;
        }
        __syncthreads();   // warp_tot / s_carry of the previous chunk have been consumed
        if (lane == 31) warp_tot[warp] = incl;
        __syncthreads();
        unsigned long long warp_excl = 0ull, chunk_tot = 0ull;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            const unsigned long long t = warp_tot[w];
            if (w < warp) warp_excl += t;
            chunk_tot += t;
        }
        const unsigned long long excl = s_carry + warp_excl + (incl - thread_total);
#pragma unroll
        for (int k = 0; k < WS_SCAN_ITEMS; ++k) {
            const int i = item0 + k;
            if (i < n) {
                int fk = ws_F_int(excl + q[k], (unsigned int)ns, sh, rmask, P.scheme == 1 ? 1 : 0, r0, P.seed, P.stream);
                if (i == n - 1) {
                    if (fk < ns) atomicAdd(P.n_clamped, (unsigned long long)(ns - fk));
                    fk = ns;   // leftover slots go to the last particle
                }
                Fs[i] = fk;
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) s_carry += chunk_tot;
    }
    __syncthreads();
    // slot j belongs to the first particle m with F(C_m) > j
    for (int j = threadIdx.x; j < ns; j += 256) {
        int lo = 0, hi = n - 1;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (Fs[mid] > j) hi = mid; else lo = mid + 1;
        }
        P.ancestors[j] = lo;
    }
}

cudaError_t ws_launch_resample_small(const WsScanParams& P, const WsLse* partials, int n_partials, double ess_perc_min, WsReduceOut* out,
                                     unsigned long long* ties, int do_finalize, cudaStream_t s) {
    ws_resample_small_kernel<<<1, 256, 0, s>>>(P, partials, n_partials, ess_perc_min, out, ties, do_finalize,
                                               reinterpret_cast<int32_t*>(P.cdf_local));
    return cudaGetLastError();
}

// Slots of the heavy tiles (see above): every CTA takes an equal slice of each heavy tile's output
// window and finds the ancestors by binary search in the tile's F table.
__global__ void __launch_bounds__(256) ws_expand_heavy_kernel(const __grid_constant__ WsScanParams P) {
    if (P.gate != 0 && P.red->do_resample == 0) return;
    __shared__ int32_t Fs[WS_SCAN_TILE];
    const unsigned int n_heavy = *P.heavy_count;
    for (unsigned int h = 0; h < n_heavy; ++h) {
        const int32_t* src = P.heavy_F + (size_t)h * (WS_SCAN_TILE + 2);
        __syncthreads();
        for (int k = threadIdx.x; k < WS_SCAN_TILE; k += 256) Fs[k] = src[k];
        __syncthreads();
        const int64_t fstart = (int64_t)src[WS_SCAN_TILE];
        const int64_t tile_base = (int64_t)src[WS_SCAN_TILE + 1] * WS_SCAN_TILE;
        const int64_t fend = (int64_t)Fs[WS_SCAN_TILE - 1];
        const int64_t len = fend - fstart;
        const int64_t per = (len + gridDim.x - 1) / gridDim.x;
        const int64_t a = fstart + (int64_t)blockIdx.x * per;
        const int64_t e = (a + per < fend) ? a + per : fend;
        for (int64_t j = a + threadIdx.x; j < e; j += 256) {
            int lo = 0, hi = WS_SCAN_TILE - 1;  // smallest k with Fs[k] > j
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if ((int64_t)Fs[mid] > j) hi = mid; else lo = mid + 1;
            }
            P.ancestors[j - P.slot_base] = (int32_t)(tile_base + lo);
        }
    }
}

// env WSB200_FX_EXTRA_BITS (tests): shrink the fixed-point scale by that many bits, so that the S < 32 arithmetic of
// ws_slot_split (normally only reached by N > 2^29 particles) can be exercised at small N
static int g_fx_extra_bits = 0;
// scale of the fixed-point CDF (see ws_w_to_fxs / ws_slot_split); call after n_slots, replay_u, sorted_u are set
void ws_scan_set_scale(WsScanParams& P) {
    const bool exact_fp = P.replay_u != nullptr || P.sorted_u != nullptr;
    int shift = 61;
    {   // multinomial: spacings of mean 2^mn_shift, so that the sum of n_slots + 1 of them stays below 2^61
        int bits = 0;
        while (((int64_t)1 << bits) < P.n_slots + 1) ++bits;
        P.mn_shift = 60 - bits;
    }
    if (!exact_fp && P.scheme != 2) {
        int bits = 0;
        while (((int64_t)1 << bits) < P.n_slots) ++bits;
        shift = 61 - bits - g_fx_extra_bits;
        if (shift < 24) shift = 24;
    }
    P.fx_shift = shift;
    P.fx_scale = (exact_fp || P.scheme == 2) ? 2305843009213693952.0 : ldexp((double)P.n_slots, shift);   // multinomial: 2^61 (ws_mn_threshold)
}

// multinomial (Philox): tile / block prefixes of the exponential spacings of ALL global slots and their total.
// On a sharded state every rank computes the same table (counter-based draws: no exchange needed).
cudaError_t ws_launch_spacings(const WsScanParams& P, cudaStream_t s) {
    const int64_t n_all = P.n_slots + 1;
    const int64_t tiles = (n_all + WS_CDF_TILE - 1) / WS_CDF_TILE;
    int g = (int)(tiles < (int64_t)g_sm_count * 8 ? tiles : (int64_t)g_sm_count * 8);
    ws_spacing_tiles_kernel<<<g < 1 ? 1 : g, WS_SCAN_BLOCK, 0, s>>>(P);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    WsScanParams Q = P;   // exclusive scan of the tile sums, in place, with the existing single-CTA kernel
    Q.n = n_all;
    Q.tile_words = P.mn_tile_off;
    Q.total = P.mn_total;
    ws_cdf_offsets_kernel<<<1, 1024, 0, s>>>(Q);
    return cudaGetLastError();
}

cudaError_t ws_launch_cdf(const WsScanParams& P, cudaStream_t s) {
    const int64_t cdf_tiles = (P.n + WS_CDF_TILE - 1) / WS_CDF_TILE;
    int g1 = (int)(cdf_tiles < (int64_t)g_sm_count * WS_CDF_GRID ? cdf_tiles : (int64_t)g_sm_count * WS_CDF_GRID);
    if (g1 < 1) g1 = 1;
    ws_cdf_tiles_kernel<<<g1, WS_SCAN_BLOCK, 0, s>>>(P);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    ws_cdf_group_offsets_kernel<<<1, 1024, 0, s>>>(P);
    return cudaGetLastError();
}

cudaError_t ws_launch_bounds(const WsScanParams& P, cudaStream_t s) {
    const bool exact_fp = P.replay_u != nullptr || P.sorted_u != nullptr;
    if (exact_fp) ws_bounds_kernel<true><<<1, 32, 0, s>>>(P);
    else ws_bounds_kernel<false><<<1, 32, 0, s>>>(P);
    return cudaGetLastError();
}

cudaError_t ws_launch_cdf_tiles(const WsScanParams& P, cudaStream_t s) {   // the tile CDF alone (its offsets: ws_launch_offsets_bounds_mbox)
    const int64_t cdf_tiles = (P.n + WS_CDF_TILE - 1) / WS_CDF_TILE;
    int g1 = (int)(cdf_tiles < (int64_t)g_sm_count * WS_CDF_GRID ? cdf_tiles : (int64_t)g_sm_count * WS_CDF_GRID);
    if (g1 < 1) g1 = 1;
    ws_cdf_tiles_kernel<<<g1, WS_SCAN_BLOCK, 0, s>>>(P);
    return cudaGetLastError();
}
cudaError_t ws_launch_offsets_bounds_mbox(const WsScanParams& P, const WsMailbox& M, unsigned long long* all_tot, const unsigned long long* xmine,
                                          int xw, unsigned long long* xall, cudaStream_t s) {
    const bool exact_fp = P.replay_u != nullptr || P.sorted_u != nullptr;
    if (exact_fp) ws_offsets_bounds_mbox_kernel<true><<<1, 1024, 0, s>>>(P, M, all_tot, xmine, xw, xall);
    else ws_offsets_bounds_mbox_kernel<false><<<1, 1024, 0, s>>>(P, M, all_tot, xmine, xw, xall);
    return cudaGetLastError();
}

cudaError_t ws_launch_search(const WsScanParams& P, cudaStream_t s) {
    const int64_t warp_tiles = (P.n + WS_SCAN_TILE - 1) / WS_SCAN_TILE;
    const int64_t ctas = (warp_tiles + WS_WARPS_PER_CTA - 1) / WS_WARPS_PER_CTA;
    int g3 = (int)(ctas < (int64_t)g_sm_count * WS_SEARCH_GRID ? ctas : (int64_t)g_sm_count * WS_SEARCH_GRID);
    if (g3 < 1) g3 = 1;
    const bool exact_fp = P.replay_u != nullptr || P.sorted_u != nullptr;
    if (exact_fp) ws_search_kernel<true, false, false><<<g3, WS_SCAN_BLOCK, WS_SEARCH_SMEM_BYTES, s>>>(P);
    else if (P.scheme == 2) ws_search_kernel<false, true, false><<<g3, WS_SCAN_BLOCK, WS_SEARCH_SMEM_BYTES, s>>>(P);
    else if (P.fx_shift >= 32) ws_search_kernel<false, false, true><<<g3, WS_SCAN_BLOCK, WS_SEARCH_SMEM_BYTES, s>>>(P);   // N <= 2^29
    else ws_search_kernel<false, false, false><<<g3, WS_SCAN_BLOCK, WS_SEARCH_SMEM_BYTES, s>>>(P);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    ws_expand_heavy_kernel<<<g_sm_count * 4, 256, 0, s>>>(P);
    return cudaGetLastError();
}

// Three forms of CDF + search on a single-GPU state (env WSB200_SCAN = 3pass | 1pass | chain):
//   3pass  tile CDF -> offsets -> search through cdf_local (also what sharded runs use: the ranks' masses are exchanged
//          between the CDF and the search)
//   1pass  one CTA per ticketed tile, look-back right after the tile's own aggregate: saves the 16 B round trip but, as
//          measured on B200 (profiles/r2b_*), loses more than that waiting in the look-back
//   chain  persistent CTAs, look-back deferred by one tile, two-level aggregates (ws_chain_kernel)
#ifndef WS_SCAN_DEFAULT_FORM
#define WS_SCAN_DEFAULT_FORM 0
#endif
static int g_scan_form = WS_SCAN_DEFAULT_FORM;  // 0 three passes, 1 single pass, 2 chain
#ifndef WS_CHAIN_DEFAULT_BLOCK
#define WS_CHAIN_DEFAULT_BLOCK WS_SCAN_BLOCK
#endif
static int g_chain_block = WS_CHAIN_DEFAULT_BLOCK;   // threads per CTA of the chain form (env WSB200_CHAIN_BLOCK = 32 | 64 | 256): tile = 8 x that
template <int BLOCK>
static cudaError_t ws_launch_chain(const WsScanParams& P, bool exact_fp, cudaStream_t s) {
    const int64_t tiles = (P.n + BLOCK * WS_SCAN_ITEMS - 1) / (BLOCK * WS_SCAN_ITEMS);
    const int64_t resident = (int64_t)g_sm_count * WS_CHAIN_MINB * (WS_SCAN_BLOCK / BLOCK);
    int g = (int)(tiles < resident ? tiles : resident);
    if (g < 1) g = 1;
    if (exact_fp) ws_chain_kernel<true, BLOCK><<<g, BLOCK, WS_CHAIN_SMEM_BYTES(BLOCK), s>>>(P);
    else ws_chain_kernel<false, BLOCK><<<g, BLOCK, WS_CHAIN_SMEM_BYTES(BLOCK), s>>>(P);
    return cudaGetLastError();
}
cudaError_t ws_launch_scan_search(const WsScanParams& P, int grid, cudaStream_t s) {
    (void)grid;
    if (g_scan_form != 0 && P.all_tot == nullptr && P.total == nullptr && P.bounds == nullptr && P.scheme != 2) {
        // single-GPU state: one pass (the caller has zeroed the ticket / heavy-tile counters)
        const int64_t cdf_tiles = (P.n + WS_CDF_TILE - 1) / WS_CDF_TILE;
        const bool exact_fp = P.replay_u != nullptr || P.sorted_u != nullptr;
        cudaError_t e = cudaMemsetAsync(P.tile_counter, 0, sizeof(unsigned int) * 2, s);   // ticket, heavy-tile count
        if (e != cudaSuccess) return e;
        if (g_scan_form == 2) {
            const int64_t ch_tiles = (P.n + g_chain_block * WS_SCAN_ITEMS - 1) / (g_chain_block * WS_SCAN_ITEMS);
            e = cudaMemsetAsync(P.tile_words, 0, sizeof(unsigned long long) * (size_t)(ch_tiles + 3 * ((ch_tiles + WS_CHAIN_GROUP - 1) / WS_CHAIN_GROUP)), s);
            if (e != cudaSuccess) return e;
            e = g_chain_block == 32 ? ws_launch_chain<32>(P, exact_fp, s) : (g_chain_block == 64 ? ws_launch_chain<64>(P, exact_fp, s) : ws_launch_chain<WS_SCAN_BLOCK>(P, exact_fp, s));
            if (e != cudaSuccess) return e;
        } else {
            e = cudaMemsetAsync(P.tile_words, 0, sizeof(unsigned long long) * (size_t)cdf_tiles, s);
            if (e != cudaSuccess) return e;
            if (exact_fp) ws_scan_search_kernel<true><<<(unsigned)cdf_tiles, WS_SCAN_BLOCK, 0, s>>>(P);
            else ws_scan_search_kernel<false><<<(unsigned)cdf_tiles, WS_SCAN_BLOCK, 0, s>>>(P);
        }
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        ws_expand_heavy_kernel<<<g_sm_count * 4, 256, 0, s>>>(P);
        return cudaGetLastError();
    }
    cudaError_t e = ws_launch_cdf(P, s);
    if (e != cudaSuccess) return e;
    return ws_launch_search(P, s);
}

// ------------------------------------------------------------------------------------------
// Ancestor gather (resample!)
// ------------------------------------------------------------------------------------------
// dst[p][i] = src[p][a_i].  Ancestors are non-decreasing, so neighbouring threads read the same or
// neighbouring sectors: the reads coalesce in L1/L2 and DRAM sees each live source sector once.
__global__ void __launch_bounds__(256) ws_gather_kernel(const __grid_constant__ WsGatherParams P) {
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < P.n; i += stride) {
        const int64_t a = (int64_t)__ldg(P.ancestors + i);
        for (int p0 = 0; p0 < P.n_planes; p0 += 8) {
            double v[8];
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (p0 + k < P.n_planes) v[k] = __ldg(P.src[p0 + k] + a);
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (p0 + k < P.n_planes) P.dst[p0 + k][i] = v[k];
        }
    }
}

cudaError_t ws_launch_gather(const WsGatherParams& P, int grid, cudaStream_t s) {
    ws_gather_kernel<<<grid, 256, 0, s>>>(P);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// helpers
// ------------------------------------------------------------------------------------------
// ancestors of a Resample step that turned out not to fire: the identity (see ws_resample_async)
__global__ void ws_fill_kernel(double* __restrict__ dst, double v, int64_t n) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = v;
}
cudaError_t ws_launch_fill(double* dst, double v, int64_t n, int grid, cudaStream_t s) {
    ws_fill_kernel<<<grid, 256, 0, s>>>(dst, v, n);
    return cudaGetLastError();
}

// exp_norm: w_i = exp(l_i - m) / S  (src/resampling.jl:72-77)
__global__ void ws_exp_norm_kernel(const double* __restrict__ logw, const WsReduceOut* __restrict__ red,
                                   double* __restrict__ w, int64_t n) {
    const double m = red->m, S = red->S;
    const double rS = 1.0 / S;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) w[i] = ws_div_pos(ws_exp_nonpos(logw[i] - m), S, rS);
}
cudaError_t ws_launch_exp_norm(const double* logw, const WsReduceOut* red, double* w, int64_t n, int grid,
                               cudaStream_t s) {
    ws_exp_norm_kernel<<<grid, 256, 0, s>>>(logw, red, w, n);
    return cudaGetLastError();
}

// sum of squares partials (ess_perc on a caller-supplied weight vector; src/resampling.jl:51-54)
__global__ void __launch_bounds__(256) ws_sumsq_kernel(const double* __restrict__ w, int64_t n,
                                                       double* __restrict__ partials) {
    __shared__ double sc[8];
    double acc = 0.0;
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) {
        const double v = w[i];
        acc += v * v;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, d);
    if ((threadIdx.x & 31) == 0) sc[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int k = 0; k < 8; ++k) t += sc[k];
        partials[blockIdx.x] = t;
    }
}
cudaError_t ws_launch_sumsq(const double* w, int64_t n, double* partials, int grid, cudaStream_t s) {
    ws_sumsq_kernel<<<grid, 256, 0, s>>>(w, n, partials);
    return cudaGetLastError();
}

// Sharded deferred gather: ancestor of local slot i.  Slots [self_lo, self_hi) are filled by this rank's
// own offspring (anc_self, slot order); the slots below / above were received from lower / higher ranks
// and sit, in slot order, in the spare rows n, n+1, ... behind every plane.
// (`spare_base`: first spare row of this event's received offspring — spare rows are handed out event by event while
// older planes still read the rows of earlier events, see SpareRing in ws_runtime.cu)
__global__ void ws_local_ancestors_kernel(int32_t* __restrict__ anc, int64_t n, const int32_t* __restrict__ anc_self,
                                          int64_t self_lo, int64_t self_hi, int64_t spare_base) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        int32_t a;
        if (i < self_lo) a = (int32_t)(n + spare_base + i);
        else if (i >= self_hi) a = (int32_t)(n + spare_base + self_lo + (i - self_hi));
        else a = anc_self[i - self_lo];
        anc[i] = a;
    }
}
cudaError_t ws_launch_local_ancestors(int32_t* anc, int64_t n, const int32_t* anc_self, int64_t self_lo, int64_t self_hi,
                                      int64_t spare_base, int grid, cudaStream_t s) {
    ws_local_ancestors_kernel<<<grid, 256, 0, s>>>(anc, n, anc_self, self_lo, self_hi, spare_base);
    return cudaGetLastError();
}

// the same for ancestors that the search already wrote in place: only the received slots are patched
__global__ void ws_patch_ancestors_kernel(int32_t* __restrict__ anc, int64_t n, int64_t self_lo, int64_t self_hi, int64_t spare_base) {
    const int64_t n_patch = self_lo + (n - self_hi);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n_patch; k += stride) {
        if (k < self_lo) anc[k] = (int32_t)(n + spare_base + k);
        else anc[self_hi + (k - self_lo)] = (int32_t)(n + spare_base + k);
    }
}
cudaError_t ws_launch_patch_ancestors(int32_t* anc, int64_t n, int64_t self_lo, int64_t self_hi, int64_t spare_base, cudaStream_t s) {
    const int64_t n_patch = self_lo + (n - self_hi);
    if (n_patch <= 0) return cudaSuccess;
    int grid = (int)((n_patch + 255) / 256);
    if (grid > g_sm_count * 8) grid = g_sm_count * 8;
    ws_patch_ancestors_kernel<<<grid, 256, 0, s>>>(anc, n, self_lo, self_hi, spare_base);
    return cudaGetLastError();
}

// ---- sharded genealogy: migrating offspring of planes that are still in an older particle order -----------------------
// A plane that is `level` resampling events behind stores the value of current slot a at row chain_{level-1}[ ... chain_0[a]]
// (chain_t = the ancestors of event E - t, nullptr for a queued step that did not fire; the walk ends at a spare row, see
// ws_compose_kernel).  For the m offspring a rank produces for another rank, ws_trace_rows_kernel walks the chain ONCE per
// offspring and keeps the row at every level; ws_push_traced_kernel then writes all planes of all levels into the peer's
// spare rows in one launch — m chains instead of gathering every stale plane over all n particles before every event.
__global__ void __launch_bounds__(256) ws_trace_rows_kernel(const int32_t* __restrict__ anc, int64_t m, const int32_t* const* __restrict__ chain,
                                                            int n_levels, int64_t n_rows, int32_t* __restrict__ rows /* [n_levels + 1][m] */) {
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x; j < m; j += stride) {
        int64_t idx = (int64_t)__ldg(anc + j);
        rows[j] = (int32_t)idx;
        for (int t = 0; t < n_levels; ++t) {
            const int32_t* a = chain[t];
            if (a != nullptr && idx < n_rows) idx = (int64_t)__ldg(a + idx);
            rows[(size_t)(t + 1) * (size_t)m + j] = (int32_t)idx;
        }
    }
}
__global__ void __launch_bounds__(256) ws_push_traced_kernel(const WsTracedPlane* __restrict__ planes, int64_t m, const int32_t* __restrict__ rows) {
    const WsTracedPlane pl = planes[blockIdx.y];
    const int32_t* const r = rows + (size_t)pl.level * (size_t)m;
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x; j < m; j += stride) pl.dst[j] = __ldg(pl.src + __ldg(r + j));
}
cudaError_t ws_launch_trace_rows(const int32_t* anc, int64_t m, const int32_t* const* chain, int n_levels, int64_t n_rows, int32_t* rows,
                                 cudaStream_t s) {
    if (m <= 0) return cudaSuccess;
    int grid = (int)((m + 255) / 256);
    if (grid > g_sm_count * 8) grid = g_sm_count * 8;
    ws_trace_rows_kernel<<<grid, 256, 0, s>>>(anc, m, chain, n_levels, n_rows, rows);
    return cudaGetLastError();
}
cudaError_t ws_launch_push_traced(const WsTracedPlane* planes, int n_planes, int64_t m, const int32_t* rows, cudaStream_t s) {
    if (m <= 0 || n_planes <= 0) return cudaSuccess;
    int gx = (int)((m + 255) / 256);
    if (gx > g_sm_count * 2) gx = g_sm_count * 2;
    for (int p0 = 0; p0 < n_planes; p0 += 32768) {   // (gridDim.y <= 65535)
        const int np = n_planes - p0 < 32768 ? n_planes - p0 : 32768;
        ws_push_traced_kernel<<<dim3((unsigned)gx, (unsigned)np), 256, 0, s>>>(planes + p0, m, rows);
    }
    return cudaGetLastError();
}

__global__ void ws_gather_rows_kernel(const double* __restrict__ src, const int64_t* __restrict__ idx, int64_t n_idx,
                                      double* __restrict__ dst) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_idx; i += stride) dst[i] = src[idx[i]];
}
cudaError_t ws_launch_gather_rows(const double* src, const int64_t* idx, int64_t n_idx, double* dst, cudaStream_t s) {
    int grid = (int)((n_idx + 255) / 256);
    if (grid > g_sm_count * 8) grid = g_sm_count * 8;
    if (grid < 1) grid = 1;
    ws_gather_rows_kernel<<<grid, 256, 0, s>>>(src, idx, n_idx, dst);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// Genealogy: composition of ancestor vectors
// ------------------------------------------------------------------------------------------
// A plane that has not been touched for several resampling events is stored in the order of the event
// after which it was last written; its current content is plane[a_{e+1}[a_{e+2}[... a_E[i]]]].  The chain
// is applied innermost-last: chain[0] = a_E, chain[1] = a_{E-1}, ...; `start` (optional) continues from a
// map composed earlier.  One dependent 4-byte load per event and particle, instead of gathering every
// column at every event as the reference's resample! does (src/stores.jl:105-121).
template <class I>
__global__ void __launch_bounds__(256) ws_compose_kernel(const WsComposeParams P, I* out, const I* start) {  // (out may alias start: element-wise)
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < P.n; i += stride) {
        int64_t idx = start != nullptr ? (int64_t)start[i] : i;
        // a row >= n_rows is a spare row (sharded states): an offspring received from another rank, whose value the
        // sender traced through ITS genealogy when it pushed it — the chain ends there
        for (int t = 0; t < P.n_chain; ++t)
            if (idx < P.n_rows) idx = (int64_t)__ldg(P.chain[t] + idx);
        out[i] = (I)idx;
    }
}
cudaError_t ws_launch_compose(const WsComposeParams& P, int32_t* out, const int32_t* start, cudaStream_t s) {
    int grid = (int)((P.n + 255) / 256);
    if (grid > g_sm_count * 8) grid = g_sm_count * 8;
    if (grid < 1) grid = 1;
    ws_compose_kernel<int32_t><<<grid, 256, 0, s>>>(P, out, start);
    return cudaGetLastError();
}
cudaError_t ws_launch_compose_rows(const WsComposeParams& P, int64_t* out, const int64_t* start, cudaStream_t s) {
    int grid = (int)((P.n + 255) / 256);
    if (grid > g_sm_count * 8) grid = g_sm_count * 8;
    if (grid < 1) grid = 1;
    ws_compose_kernel<int64_t><<<grid, 256, 0, s>>>(P, out, start);
    return cudaGetLastError();
}

cudaError_t ws_kernels_init(int device) {
    cudaDeviceProp prop;
    cudaError_t e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) return e;
    g_sm_count = prop.multiProcessorCount;
    {
        const char* v = getenv("WSB200_SCAN");
        if (v != nullptr) g_scan_form = strcmp(v, "1pass") == 0 ? 1 : (strcmp(v, "chain") == 0 ? 2 : (strcmp(v, "3pass") == 0 ? 0 : WS_SCAN_DEFAULT_FORM));
        else g_scan_form = WS_SCAN_DEFAULT_FORM;
        v = getenv("WSB200_CHAIN_BLOCK");
        g_chain_block = v != nullptr ? atoi(v) : WS_CHAIN_DEFAULT_BLOCK;
        if (g_chain_block != 32 && g_chain_block != 64) g_chain_block = WS_SCAN_BLOCK;
        v = getenv("WSB200_FX_EXTRA_BITS");
        g_fx_extra_bits = v != nullptr ? atoi(v) : 0;
        v = getenv("WSB200_VM");
        g_vm_interp_only = v != nullptr && strcmp(v, "interp") == 0;
    }
    // the register file of the fused pass can take most of the SM's shared memory
    e = cudaFuncSetAttribute(ws_search_kernel<true, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, WS_SEARCH_SMEM_BYTES);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(ws_search_kernel<false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, WS_SEARCH_SMEM_BYTES);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(ws_search_kernel<false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, WS_SEARCH_SMEM_BYTES);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(ws_search_kernel<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, WS_SEARCH_SMEM_BYTES);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(ws_chain_kernel<true, WS_SCAN_BLOCK>, cudaFuncAttributeMaxDynamicSharedMemorySize, WS_CHAIN_SMEM_BYTES(WS_SCAN_BLOCK));
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(ws_chain_kernel<false, WS_SCAN_BLOCK>, cudaFuncAttributeMaxDynamicSharedMemorySize, WS_CHAIN_SMEM_BYTES(WS_SCAN_BLOCK));
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(ws_vm_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 208 * 1024);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(ws_vm_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 208 * 1024);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(ws_vm_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 208 * 1024);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(ws_vm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 208 * 1024);
    return e;
}
