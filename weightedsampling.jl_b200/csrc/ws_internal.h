// ws_internal.h — structs shared between the host runtime (ws_runtime.cu) and the kernel
// translation units, plus the launcher prototypes.  Not part of the public ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "ws_vm.cuh"
#include "ws_mailbox.cuh"

#ifndef WS_VM_BLOCK
#define WS_VM_BLOCK 128       // threads per CTA of the fused elementwise pass
#endif
#ifndef WS_VM_P
#define WS_VM_P 3             // particles per thread: one decoded micro-op is applied to all of them
#endif
#ifndef WS_VM_MINB
#define WS_VM_MINB 5          // resident CTAs per SM the kernel is compiled for (register cap 65536/(128*MINB))
#endif
#define WS_VM_MAX_IO 24       // planes loaded / stored per fused pass
#define WS_VM_MAX_CKPT 16     // checkpoints per fused pass (speculative blocks)
#define WS_VM_MAX_OPS 96      // micro-ops per fused pass (program travels in kernel params)
#define WS_VM_MAX_REGS ((192 * 1024) / (WS_VM_BLOCK * WS_VM_P * 8))  // register-file rows per pass (<= 192 KB of smem)
#define WS_SCAN_BLOCK 256
#define WS_SCAN_ITEMS 8
#define WS_SCAN_TILE (32 * WS_SCAN_ITEMS)  // particles per warp-granular search tile
#define WS_CDF_TILE (WS_SCAN_BLOCK * WS_SCAN_ITEMS)  // particles per CTA tile of the CDF pass
#define WS_GATHER_MAX_PLANES 32
#define WS_HEAVY_TILE_SLOTS 32768  // a tile with more offspring than this is expanded by the whole grid
#define WS_MAX_PARTIALS 4096  // upper bound on CTAs that write (m,S,Q) partials

// (m, S, Q) = (max l, sum exp(l-m), sum exp(2(l-m))) — everything exp_norm / ess_perc /
// logsumexp need (src/resampling.jl:51-77), in one pass.
struct WsLse {
    double m, S, Q;
};

// Result of the reduction + resampling decision, device resident and mirrored to pinned host.
struct WsReduceOut {
    double m, S, Q;
    double lse;         // m + log S
    double ess_perc;    // S^2 / (N Q)
    double log_mean_w;  // lse - log N
    int32_t do_resample;
    int32_t pad;
};

struct WsVmProgram {
    int64_t n;                // local particles
    int64_t particle_offset;  // global index of local particle 0 (RNG counters, replay offsets)
    int32_t n_ops, n_loads, n_stores, n_regs;
    const double* load_ptr[WS_VM_MAX_IO];
    double* store_ptr[WS_VM_MAX_IO];
    uint8_t load_reg[WS_VM_MAX_IO];
    uint8_t store_reg[WS_VM_MAX_IO];
    // pending ancestor gather folded into the loads (lazy resample!): bit k of load_gather set
    // => plane k is read through ancestors[i]
    const int32_t* ancestors;
    uint32_t load_gather;
    // log-weight accumulation of the window's Observe / Weight / weighter terms
    int32_t logw_mode;  // 0: window has no weight term; 1: logw[i] += acc; 2: logw[i] = logw_base + acc;
                        // 3: decided by red->do_resample (a Resample step still pending on the host): 2 with
                        //    logw_base = red->log_mean_w if it fired, else 1 — and the gathered loads read straight
    double* logw;
    double logw_base;
    WsLse* partials;  // per-CTA (m,S,Q) of the NEW log-weights (nullptr: skip)
    // expectation mode (ws_expectation): sum_i w_i * r[expect_reg[k]], w_i = exp(logw_i - m)/S
    int32_t n_expect;
    uint8_t expect_reg[8];
    const WsReduceOut* red;  // (m,S) for expectation mode
    double* expect_partials; // [gridDim.x][n_expect]
    // Checkpoints (speculative blocks of weighting statements, ws_exec_spec): after micro-op ckpt_pc[j] the weight
    // terms accumulated so far are folded into the running log-weight — the log-weight the statement-by-statement
    // passes would have stored at that point, same association — and pushed into the j-th (m, S, Q) state, so ONE
    // pass yields the ESS after each of its statements.  Interpreter only (ws_vm_kernel).
    int32_t n_ckpt;
    uint8_t ckpt_pc[WS_VM_MAX_CKPT];
    WsLse* ckpt_partials;    // [n_ckpt][gridDim.x]
    double* logw_out;        // checkpointed windows write the new log-weights here (the old array is the roll-back copy); nullptr: in place
    WsRng rng;
    WsOp ops[WS_VM_MAX_OPS];
};

struct WsScanParams {
    const double* logw;        // log-weights (mode 0) or normalised weights (mode 1)
    int32_t mode;              // 0: w_i = exp(l_i - m)/S from *red ; 1: w_i given ; 2: uniform weights 1/N
    int32_t scheme;            // WS_RESAMPLER_*
    const WsReduceOut* red;    // mode 0; also carries do_resample (checked when gate != 0)
    int32_t gate;              // 1: return immediately unless red->do_resample
    int32_t pad;
    int64_t n;                 // local particles (this rank's shard)
    int64_t n_slots;           // output slots == GLOBAL particle count (== n on one GPU)
    unsigned long long cdf_offset;  // fixed-point mass of all lower ranks (0 on one GPU) ...
    const unsigned long long* all_tot;  // ... or, if set, the allgathered per-rank masses: offset = sum of all_tot[0..rank)
    int32_t rank;
    int32_t pad2;
    int32_t slot_base;         // global index of the first slot this rank produces; ancestors[slot - slot_base]
    int32_t last_rank;         // the last particle of the last rank takes the clamped slots
    int32_t* bounds;           // [2] ws_bounds_kernel: first / end global slot produced by this rank
    unsigned long long* total; // [1] ws_cdf_offsets_kernel: this rank's fixed-point mass
    uint64_t seed, stream;     // Philox stream for the slot uniforms
    const double* replay_u;    // n uniforms (stratified) / 1 uniform (systematic) or nullptr
    const double* sorted_u;    // multinomial: n sorted uniforms (device)
    int32_t* ancestors;        // out, 0-based
    unsigned long long* tile_words;  // [n / WS_CDF_TILE]: tile aggregates, then their exclusive scan
    unsigned long long* cdf_local;   // [n]: tile-local inclusive fixed-point CDF
    unsigned int* tile_counter;      // single-pass kernel: the tile ticket, zeroed before launch
    double fx_scale;                 // fixed-point scale of the CDF and log2 of the units per slot (ws_scan_set_scale)
    int32_t fx_shift;
    int32_t mn_shift;                // multinomial: fixed-point scale 2^mn_shift of the exponential spacings
    // Multinomial resampling without a sort (scheme 2, Philox draws): the order statistics of n_slots iid uniforms are
    // u_k = S_k / S_total with S_k the running sum of n_slots + 1 iid exponential spacings (slot k's spacing is
    // Philox(k)); only coarse prefixes are stored — per tile of WS_CDF_TILE slots (exclusive, scanned) and per block
    // of WS_SCAN_TILE slots (tile-local, exclusive) — and the search regenerates the spacings of the blocks it needs.
    unsigned long long* mn_tile_off;     // [ceil((n_slots + 1) / WS_CDF_TILE)]
    unsigned long long* mn_block_local;  // [ceil((n_slots + 1) / WS_SCAN_TILE)]
    unsigned long long* mn_total;        // [1] S_total
    unsigned long long* n_clamped;  // += slots beyond the last CDF entry (clamped to the last particle)
    unsigned int* heavy_count;       // number of heavy tiles, zeroed before launch
    int32_t* heavy_F;                // [n/WS_HEAVY_TILE_SLOTS + 2][WS_SCAN_TILE + 2]: F table, fstart, tile id
};

struct WsGatherParams {
    int64_t n;
    const int32_t* ancestors;
    int32_t n_planes;
    int32_t pad;
    const double* src[WS_GATHER_MAX_PLANES];
    double* dst[WS_GATHER_MAX_PLANES];
};

#define WS_COMPOSE_MAX_CHAIN 24
struct WsComposeParams {
    int64_t n;
    int64_t n_rows;   // rows >= n_rows end a chain (spare rows of a sharded state); the shard size
    int32_t n_chain;
    int32_t pad;
    const int32_t* chain[WS_COMPOSE_MAX_CHAIN];  // applied in this order: idx = chain[t][idx]
};

// launchers (ws_kernels.cu)
cudaError_t ws_launch_vm(const WsVmProgram& P, int grid, cudaStream_t s);
cudaError_t ws_launch_reduce_logw(const double* logw, int64_t n, WsLse* partials, int grid, cudaStream_t s);
// k reductions of n_partials partials each (partials[j * n_partials ..] -> out[j]); ties: knife-edge decisions, or nullptr
cudaError_t ws_launch_finalize(const WsLse* partials, int n_partials, int k, int64_t n_global, double ess_perc_min,
                               WsReduceOut* out, unsigned long long* ties, cudaStream_t s);
#define WS_SMALL_N 4096   // up to this many particles (single-GPU, Philox stratified / systematic) a Resample step is one kernel
                          // (one CTA: its time grows with N — 75 us at N = 1e4 against 45 us for the four launches of the tiled form)
cudaError_t ws_launch_resample_small(const WsScanParams& P, const WsLse* partials, int n_partials, double ess_perc_min, WsReduceOut* out,
                                     unsigned long long* ties, int do_finalize, cudaStream_t s);
void ws_scan_set_scale(WsScanParams& P);
size_t ws_scan_words(int64_t n);  // 8-byte words of WsScanParams::tile_words for n particles (tile words + the chain form's group words)
cudaError_t ws_launch_scan_search(const WsScanParams& P, int grid, cudaStream_t s);
// sharded resampling runs the same passes in two halves with collectives in between
cudaError_t ws_launch_spacings(const WsScanParams& P, cudaStream_t s);  // multinomial: spacing prefixes of all global slots
cudaError_t ws_launch_cdf(const WsScanParams& P, cudaStream_t s);     // tile CDF + offsets (+ total)
cudaError_t ws_launch_bounds(const WsScanParams& P, cudaStream_t s);  // first / end slot of this rank
cudaError_t ws_launch_search(const WsScanParams& P, cudaStream_t s);  // F(C_m) + expansion (+ heavy tiles)
cudaError_t ws_launch_finalize_global(const double* all_msq, int n_ranks, int64_t n_global, double ess_perc_min,
                                      WsReduceOut* out, cudaStream_t s, unsigned long long* ties = nullptr);
// mailbox forms (ws_mailbox.cuh): the small exchanges of a sharded step done by the kernels themselves over peer memory
cudaError_t ws_launch_finalize_mbox(const WsLse* partials, int n_partials, int64_t n_global, double ess_perc_min, WsReduceOut* out,
                                    double* all_msq, unsigned long long* ties, const WsMailbox& M, cudaStream_t s);
cudaError_t ws_launch_cdf_tiles(const WsScanParams& P, cudaStream_t s);
cudaError_t ws_launch_offsets_bounds_mbox(const WsScanParams& P, const WsMailbox& M, unsigned long long* all_tot, const unsigned long long* xmine,
                                          int xw, unsigned long long* xall, cudaStream_t s);
cudaError_t ws_launch_barrier_mbox(const WsMailbox& M, cudaStream_t s);
cudaError_t ws_launch_gather(const WsGatherParams& P, int grid, cudaStream_t s);
cudaError_t ws_launch_fill(double* dst, double v, int64_t n, int grid, cudaStream_t s);
cudaError_t ws_launch_exp_norm(const double* logw, const WsReduceOut* red, double* w, int64_t n, int grid,
                               cudaStream_t s);
cudaError_t ws_launch_sumsq(const double* w, int64_t n, double* partials, int grid, cudaStream_t s);
cudaError_t ws_launch_local_ancestors(int32_t* anc, int64_t n, const int32_t* anc_self, int64_t self_lo, int64_t self_hi,
                                      int64_t spare_base, int grid, cudaStream_t s);
cudaError_t ws_launch_patch_ancestors(int32_t* anc, int64_t n, int64_t self_lo, int64_t self_hi, int64_t spare_base, cudaStream_t s);
// sharded genealogy: offspring pushed to a peer for planes that are `level` events behind (ws_kernels.cu)
struct WsTracedPlane {
    const double* src;   // the plane's front buffer (its own, older, particle order)
    double* dst;         // first row of the piece in the peer's plane
    int64_t level;       // resampling events the plane is behind
};
cudaError_t ws_launch_trace_rows(const int32_t* anc, int64_t m, const int32_t* const* chain, int n_levels, int64_t n_rows, int32_t* rows,
                                 cudaStream_t s);
cudaError_t ws_launch_push_traced(const WsTracedPlane* planes, int n_planes, int64_t m, const int32_t* rows, cudaStream_t s);
cudaError_t ws_launch_gather_rows(const double* src, const int64_t* idx, int64_t n_idx, double* dst, cudaStream_t s);
cudaError_t ws_launch_compose(const WsComposeParams& P, int32_t* out, const int32_t* start, cudaStream_t s);
cudaError_t ws_launch_compose_rows(const WsComposeParams& P, int64_t* out, const int64_t* start, cudaStream_t s);
int ws_vm_sl_grid(const WsVmProgram& P);  // > 0: the window runs on a straight-line executor with this grid
int ws_vm_max_grid(int n_regs, int n_loads, int n_ops, int sm_count, int n_ckpt = 0);
int ws_vm_smem_bytes(int n_regs, int n_loads, int n_ops, int n_ckpt = 0);
cudaError_t ws_kernels_init(int device);
