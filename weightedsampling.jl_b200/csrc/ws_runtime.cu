// ws_runtime.cu — the C ABI of include/wsb200.h: device-resident SMCState + ColumnStore, the
// statement fusion queue, the Resample state machine and the analysis reductions.
//
// Reference map (all under /root/reference/src):
//   ws_ctx                      SMCState + ColumnStore                 types.jl:48-78, stores.jl:70-111
//   statement calls             apply!(::Assign/Sample/Observe/Weight) transformers.jl:28-32,172-182,228-235,283-289
//   ws_resample                 apply!(::Resample)                     transformers.jl:474-498
//   ws_exp_norm/ws_log_evidence exp_norm, logsumexp, ess_perc          resampling.jl:51-77, utils.jl:21
//   ws_move                     apply!(::Move), RW, autoRW             transformers.jl:588-623, move_kernels.jl:189-253
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <algorithm>
#include <functional>
#include <memory>
#include <deque>
#include <map>
#include <string>
#include <vector>

#include <dlfcn.h>
#include <unistd.h>
#include <chrono>

#include "../../include/wsb200.h"
#include "ws_internal.h"
#include "ws_lowering.h"
#include "ws_move.h"
#include "ws_stats.h"
#include "ws_exchange.h"

using wsl::Plane;
using wsl::Program;
using wsl::Val;

static thread_local std::string g_create_error;

// ------------------------------------------------------------------------------------------
// NCCL, bound at run time (dlopen) so that the library loads on machines without NCCL and shares the
// process's NCCL instance (e.g. the one PyTorch bundles) instead of linking a second copy.
// ------------------------------------------------------------------------------------------
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
enum { WS_NCCL_INT8 = 0, WS_NCCL_UINT8 = 1, WS_NCCL_INT32 = 2, WS_NCCL_UINT32 = 3, WS_NCCL_INT64 = 4, WS_NCCL_UINT64 = 5,
       WS_NCCL_FLOAT64 = 8 };
enum { WS_NCCL_SUM = 0 };
struct NcclApi {
    void* handle = nullptr;
    int (*GetUniqueId)(ncclUniqueId*) = nullptr;
    int (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*Send)(const void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*Recv)(void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;
static bool load_nccl(std::string& err) {
    if (g_nccl.handle != nullptr) return true;
    std::vector<std::string> cand;
    if (const char* e = getenv("WSB200_NCCL_LIB")) cand.push_back(e);
    cand.push_back("libnccl.so.2");
    cand.push_back("libnccl.so");
    void* h = nullptr;
    for (auto& c : cand) {
        h = dlopen(c.c_str(), RTLD_NOW | RTLD_GLOBAL);
        if (h) break;
    }
    if (!h) {
        err = std::string("cannot load NCCL (set WSB200_NCCL_LIB): ") + (dlerror() ? dlerror() : "");
        return false;
    }
#define WS_SYM(field, name)                                                  \
    *(void**)(&g_nccl.field) = dlsym(h, name);                               \
    if (!g_nccl.field) {                                                     \
        err = std::string("NCCL symbol missing: ") + name;                   \
        return false;                                                        \
    }
    WS_SYM(GetUniqueId, "ncclGetUniqueId")
    WS_SYM(CommInitRank, "ncclCommInitRank")
    WS_SYM(CommDestroy, "ncclCommDestroy")
    WS_SYM(AllGather, "ncclAllGather")
    WS_SYM(AllReduce, "ncclAllReduce")
    WS_SYM(Send, "ncclSend")
    WS_SYM(Recv, "ncclRecv")
    WS_SYM(GroupStart, "ncclGroupStart")
    WS_SYM(GroupEnd, "ncclGroupEnd")
    WS_SYM(GetErrorString, "ncclGetErrorString")
#undef WS_SYM
    g_nccl.handle = h;
    return true;
}

enum WsKernelClass { KC_VM = 0, KC_REDUCE, KC_FINALIZE, KC_SCAN, KC_GATHER, KC_FILL, KC_MOVE, KC_OTHER, KC_COUNT };

struct Column {
    std::string name;
    int32_t width;
    std::vector<double*> front, back;
    // Lazy resample!: after a resampling step the gather of a plane is deferred until the plane is
    // next read.  stale[k] means "front[k] still holds the pre-resample order; element i of the
    // current particle set is front[k][d_anc[i]]".
    std::vector<uint8_t> stale;
    // Genealogy: ep[k] = number of resampling events after which front[k] was last written / gathered.
    // stale[k] <=> ep[k] < ctx.epoch; the current content is front[k][a_{ep+1}[... a_epoch[i]]].
    std::vector<int64_t> ep;
};

struct TimedEvent {
    int kclass;
    cudaEvent_t a, b;
};

struct TapeEntry {
    int64_t depth;   // state.depth before the statement ran (it is scored iff depth < target_depth)
    int32_t op_end;  // score_prog.ops[0 .. op_end) covers the tape up to and including this entry
    int32_t cache_ops;  // leading ops of this entry that are a sigma-cache prologue (needed by later entries too)
    double konst_end;  // particle-independent part of the log-densities up to and including this entry (Program::acc_const)
    std::function<void(Program&)> lower;  // re-lowers the statement's log-density (owns its expressions)
    std::vector<Plane> refs;              // planes the log-density reads
};

// deep copy of caller expressions, so that a tape entry can be lowered again later
struct OwnedExprs {
    std::vector<std::vector<ws_tok>> toks;
    std::vector<ws_expr> ex;
    explicit OwnedExprs(std::initializer_list<std::pair<const ws_expr*, int>> groups) {
        for (auto& g : groups)
            for (int i = 0; i < g.second; ++i) toks.emplace_back(g.first[i].toks, g.first[i].toks + g.first[i].n);
        for (auto& t : toks) ex.push_back(ws_expr{t.data(), (int32_t)t.size(), 0});
    }
    void planes(std::vector<Plane>& out) const {
        for (auto& t : toks)
            for (auto& k : t)
                if (k.op == WS_TOK_PLANE) out.push_back(Plane{k.col, k.comp});
    }
};

struct ws_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    int64_t n = 0;         // local particles
    int64_t spare = 0;     // extra rows behind every plane: offspring received from other ranks land here
    int64_t n_global = 0;
    int64_t offset = 0;    // global index of local particle 0
    int rank = 0, nranks = 1;
    uint64_t seed = 0;
    uint64_t next_stream = 1;
    double ess_perc_min = 0.5;
    int resampler = WS_RESAMPLER_STRATIFIED;

    // SMCState scalars
    bool resampled = false, weights_changed = false;
    int64_t depth = 0;

    // store
    std::vector<Column> cols;
    std::map<std::string, int32_t> col_index;

    // log-weights
    double* logw = nullptr;
    bool logw_uniform = true;  // every entry equals logw_base (the array itself may be stale)
    double logw_base = 0.0;
    bool partials_valid = false;
    int n_partials = 0;
    WsLse* d_partials = nullptr;
    WsReduceOut* d_red = nullptr;
    WsReduceOut* h_red = nullptr;  // pinned
    bool red_valid = false;        // h_red/d_red describe the current log-weights
    // Resample steps whose decision the host has not looked at yet (ws_resample_async): the (m, S, Q, ESS, decision)
    // record of each is copied, stream-ordered, into a pinned ring; the scan / search kernels run gated on the device
    // flag, the host books the event as if it had fired (if it did not, the ancestors are the identity) and learns the
    // truth when somebody asks (resolve_spec).  logw_spec: the LAST such step has not been followed by a weighting pass
    // yet, i.e. the log-weights are "all equal to d_red->log_mean_w if it fired, else the array as it is".
    static constexpr int SPEC_RING = 512;
    WsReduceOut* h_ring = nullptr;  // pinned [SPEC_RING]
    int64_t ring_event[SPEC_RING] = {0};  // resampling event booked for each record
    int64_t spec_head = 0;          // records [spec_head - spec_pending, spec_head) are unresolved
    int spec_pending = 0;
    bool logw_spec = false;
    bool async_resample = true;     // env WSB200_ASYNC_RESAMPLE=0: ws_resample_async behaves like ws_resample
    bool merged_decision_wait = true;  // sharded steps: the decision is read with the slot bounds (env WSB200_MERGED_WAIT=0: two waits)
    bool small_resample = true;     // env WSB200_SMALL_RESAMPLE=0: small particle sets use the multi-kernel resampler too
    ws_resample_info last_info{};   // outcome of the most recent Resample step (ws_last_resample)
    bool last_info_pending = false; // ... which is the newest unresolved record
    // A model that reads `resampled` after every step (`if resampled ... end`, examples/linear_regression.jl:22)
    // waits for each decision anyway; queueing the step then only adds the gated launches and a resampling event
    // per non-firing step.  Two steps in a row resolved before anything else was queued switch the run to ws_resample.
    int spec_immediate = 0;
    // Speculative block (ws_exec_spec): K consecutive (weighting statements, Resample) steps issued as ONE pass whose
    // checkpoints give the ESS after each step; spec_block is set while the steps are being queued.
    struct SpecStep {
        size_t tape_size;           // tape / score program right after the step's statements
        Program::Mark score_mark;
        int64_t depth;
        uint64_t stream_before;     // next_stream before the step's Resample took its Philox stream
        int32_t ckpt_pc;            // last micro-op of the step in the window
    };
    bool spec_block = false, spec_flushing = false;
    std::vector<SpecStep> spec_steps;
    double* d_logw_bak = nullptr;       // log-weights before the block (restored when a step fires)
    WsLse* d_ck_partials = nullptr;     // [WS_VM_MAX_CKPT][WS_MAX_PARTIALS]
    WsReduceOut* d_ck_red = nullptr;    // [WS_VM_MAX_CKPT]
    WsReduceOut* h_ck_red = nullptr;    // pinned

    // resampling scratch
    int32_t* d_anc = nullptr;  // ancestors of the latest resampling event (== anc_live.back().ptr)
    bool anc_pending = false;  // some plane is stale
    // Genealogy (SURVEY §8f.2): a resampling event no longer forces the gather of the planes that are still
    // in an older order; their ancestor vectors are kept instead and composed when such a plane is read.
    struct AncVec {
        int64_t event;  // maps slots of epoch `event` to slots of epoch `event - 1`
        int32_t* ptr;
        bool identity = false;  // a queued step that turned out not to fire (resolve_spec): the map is the identity
    };
    int64_t epoch = 0;                // resampling events so far
    std::deque<AncVec> anc_live;      // vectors some plane may still need, ascending events
    std::vector<int32_t*> anc_pool;   // recycled vectors
    bool genealogy = true;
    size_t genealogy_budget = 0;      // bytes of retained ancestor vectors before old planes are gathered anyway
    // Sharded genealogy: planes that are not read keep their order over the events of a sharded run too.  The offspring a
    // plane receives at an event stay in spare rows handed out event by event (ws_exchange.h: WsSpareRing, one ring per
    // rank, all of them kept on every rank), and what a rank pushes to a peer for a plane that is behind is found by
    // tracing the migrating offspring — not the whole shard — through the retained ancestor vectors.
    std::vector<WsSpareRing> spare_rings;  // [rank]
    bool event_keeps = false;         // the resampling event being prepared keeps stale planes (prepare_resample_event)
    void* d_gen = nullptr;            // scratch of the traced push: [chain pointers | plane table | rows per level]
    size_t gen_bytes = 0;
    int64_t traced_rows = 0;          // offspring pushed for planes that were behind (rows x planes), for the tests
    int64_t trace_forced_planes = 0, trace_full_gathers = 0, trace_ipc_rounds = 0;  // WSB200_TRACE: planes brought up to date to free
                                      // ancestor vectors / spare rows, events that had to bring everything up to date, IPC mapping rounds
    // planes and ancestor vectors are carved out of slabs: a cudaMalloc per new column costs milliseconds
    // (models that create a column per time step: x{t}), and nothing is ever freed before ws_destroy
    struct Slab {
        char* base;
        size_t size, used;
    };
    std::vector<Slab> slabs;
    int32_t* d_map = nullptr;         // cached composition: slot of epoch map_E -> row in the order of epoch map_ep
    int64_t map_ep = -1, map_E = -1;
    bool lazy_gather = true;
    unsigned long long* d_tile_words = nullptr;
    unsigned long long* d_cdf_local = nullptr;  // [n] tile-local fixed-point CDF (scratch of the resampler)
    unsigned int* d_tile_counter = nullptr;  // [0] dynamic tile id, [1] heavy-tile count
    int32_t* d_heavy_F = nullptr;
    // multinomial without a sort: coarse prefixes of the exponential spacings of all global slots (ws_launch_spacings)
    unsigned long long* d_mn = nullptr;       // [tile offsets | block-local prefixes | total]
    int64_t mn_cap_slots = 0;
    int64_t heavy_cap_n = 0;                  // particle count d_heavy_F is sized for
    int64_t n_tiles = 0;
    unsigned long long* d_counters = nullptr;  // [0] clamped slots (cumulative), [1] clamped (host-array calls), [2] MH accepts

    // fusion window + score tape
    Program win;
    Program score;
    std::vector<TapeEntry> tape;
    WsOp* d_score_ops = nullptr;
    size_t d_score_cap = 0, d_score_uploaded = 0;
    WsOp* d_seg_ops = nullptr;  // micro-ops of the tape segment being folded (wide tapes)
    size_t d_seg_cap = 0;
    bool record_only = false;
    bool tape_enabled = true;
    bool score_wide = false;  // the tape reads more planes than one register file holds: fold it in segments

    // replay buffers
    double* d_replay_n = nullptr;
    double* d_replay_u = nullptr;
    double* d_replay_e = nullptr;
    double* d_replay_v = nullptr;
    int64_t replay_v_len = 0, cur_v = 0;
    int64_t replay_n_len = 0, replay_u_len = 0, replay_e_len = 0;
    int64_t cur_n = 0, cur_u = 0, cur_e = 0;

    // scratch for MH / analysis
    double* d_scratch = nullptr;
    void* d_scratch2 = nullptr;  // second grow-only scratch (sharded distinct count: receive buffer + owner table)
    size_t scratch2_bytes = 0;
    size_t scratch_bytes = 0;
    double* h_scratch = nullptr;  // pinned
    size_t h_scratch_bytes = 0;

    // sharded state (one rank per GPU): NCCL communicator + exchange scratch
    ncclComm_t comm = nullptr;
    double* d_all_msq = nullptr;             // [nranks][3] allgathered (m, S, Q)
    unsigned long long* d_all_tot = nullptr; // [nranks] allgathered fixed-point masses; [nranks] own total staged at the end
    int32_t* d_all_bounds = nullptr;         // [nranks][2] allgathered (first, end) produced slot; own pair staged at the end
    int32_t* d_anc_src = nullptr;            // ancestors (local indices) of the slots this rank produces
    int64_t anc_src_cap = 0;
    double* d_send = nullptr;                // staging of outgoing offspring, one plane batch at a time
    int64_t send_cap = 0;
    int64_t migrated_total = 0;              // particles received from other ranks so far
    // direct exchange: migrating offspring are gathered STRAIGHT into the destination rank's planes over NVLink
    // (peer mappings of the other ranks' slabs, cudaIpc), one kernel per destination instead of stage + ncclSend/Recv
    bool push_exchange = true;               // env WSB200_EXCHANGE=nccl: always stage + ncclSend / ncclRecv
    int64_t push_min = 0;                    // migrants over all ranks from which the direct path is used (env WSB200_PUSH_MIN)
    size_t slabs_published = 0;              // how many of my slabs the other ranks have mapped
    std::vector<std::vector<char*>> peer_slabs;  // [rank][slab index]: that rank's slabs in this process's address space
    unsigned long long* d_barrier = nullptr; // 8 bytes all-reduced after the pushes: a stream-ordered barrier over the ranks
    // per-step message of a rank, all-gathered once: [(first, end) produced slot | slab count | pid | per plane:
    // (slab, offset) of the front and of the back buffer].  The bounds are written by ws_bounds_kernel, the rest
    // by the host; the plane addresses ride along so that the direct exchange needs no round trip of its own.
    int64_t* d_xmsg = nullptr;
    size_t xmsg_words = 0;                   // words per rank the buffer was sized for
    int64_t pushed_total = 0;                // particles written directly into peers so far
    // mailbox exchanges (ws_mailbox.cuh): the small all-to-all messages of a sharded step are stored by the producing
    // kernel straight into the peers' mailboxes (mapped once, here) instead of travelling as NCCL collectives
    bool mbox_on = false;                    // every rank mapped every mailbox and the trial exchange went through (env WSB200_MAILBOX=0: off)
    unsigned long long* d_mbox = nullptr;    // my mailbox: [2 parities][nranks sources][mbox_cap] 8-byte words
    std::vector<unsigned long long*> mbox_peer;  // rank q's mailbox in this process's address space ([rank] = d_mbox)
    int32_t mbox_cap = 0;
    uint32_t mbox_seq = 0;                   // sequence number of the last exchange (the same on every rank)
    unsigned int* h_mbox_err = nullptr;      // mapped host word: an exchange timed out
    unsigned int* d_mbox_err = nullptr;      // its device address
    int64_t mbox_exchanges = 0;
    double phase_ms[8] = {0};                // WSB200_TRACE=1: host wall time per phase of resample_sharded
    int64_t phase_n = 0;

    // stats / timing
    ws_stats stats{};
    bool timing = false;
    std::vector<TimedEvent> pending_events;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> event_pool;
    double kc_ms[KC_COUNT] = {0};
    int64_t kc_count[KC_COUNT] = {0};

    std::string err;
};

static int materialize_planes(ws_ctx* c, const std::vector<Plane>* only = nullptr);
static int materialize_deep(ws_ctx* c, const std::vector<Plane>& planes);
static int map_for_epoch(ws_ctx* c, int64_t ep, const int32_t** out);
static const int32_t* anc_of_event(const ws_ctx* c, int64_t event);
static int materialize_tape_planes(ws_ctx* c, int32_t n_extra, const int32_t* col, const int32_t* comp);
static int resolve_spec(ws_ctx* c);
static int mbox_setup(ws_ctx* c);
static WsMailbox mbox_next(ws_ctx* c, int n_exchanges);
static int mbox_check(ws_ctx* c);

// ------------------------------------------------------------------------------------------
// error helpers
// ------------------------------------------------------------------------------------------
static int fail(ws_ctx* c, int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (c != nullptr) c->err = buf; else g_create_error = buf;
    return code;
}
#define CK(c, call)                                                                                     \
    do {                                                                                                \
        cudaError_t e__ = (call);                                                                       \
        if (e__ != cudaSuccess)                                                                         \
            return fail((c), e__ == cudaErrorMemoryAllocation ? WS_ENOMEM : WS_ECUDA, "%s failed: %s (%s:%d)", #call, \
                        cudaGetErrorString(e__), __FILE__, __LINE__);                                   \
    } while (0)
#define TRY(expr)                 \
    do {                          \
        int rc__ = (expr);        \
        if (rc__ != WS_OK) return rc__; \
    } while (0)
#define NCK(c, call)                                                                                       \
    do {                                                                                                   \
        int r__ = (call);                                                                                  \
        if (r__ != 0) return fail((c), WS_ENCCL, "%s failed: %s", #call, g_nccl.GetErrorString(r__));      \
    } while (0)

// ------------------------------------------------------------------------------------------
// timing
// ------------------------------------------------------------------------------------------
static void timed_begin(ws_ctx* c, int kclass, TimedEvent& te) {
    te.kclass = kclass;
    te.a = te.b = nullptr;
    c->stats.kernel_launches++;
    c->kc_count[kclass]++;
    if (!c->timing) return;
    if (c->event_pool.empty()) {
        cudaEventCreate(&te.a);
        cudaEventCreate(&te.b);
    } else {
        te.a = c->event_pool.back().first;
        te.b = c->event_pool.back().second;
        c->event_pool.pop_back();
    }
    cudaEventRecord(te.a, c->stream);
}
static void timed_end(ws_ctx* c, TimedEvent& te) {
    if (!c->timing || te.a == nullptr) return;
    cudaEventRecord(te.b, c->stream);
    c->pending_events.push_back(te);
}
static void resolve_events(ws_ctx* c) {
    if (c->pending_events.empty()) return;
    cudaStreamSynchronize(c->stream);
    for (auto& te : c->pending_events) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, te.a, te.b) == cudaSuccess) c->kc_ms[te.kclass] += (double)ms;
        c->event_pool.push_back({te.a, te.b});
    }
    c->pending_events.clear();
}

static int pool_alloc(ws_ctx* c, void** out, size_t bytes) {
    bytes = (bytes + 255) & ~(size_t)255;
    for (auto& sl : c->slabs) {
        if (sl.size - sl.used >= bytes) {
            *out = sl.base + sl.used;
            sl.used += bytes;
            return WS_OK;
        }
    }
    // 32 requests of this size per slab, between 8 MB and 256 MB (never less than the request itself).  Sharded states
    // grow geometrically on top (a new slab is as large as all slabs so far, up to 8 GB): every new slab has to be
    // mapped into the other ranks (cudaIpcGetMemHandle / cudaIpcOpenMemHandle + two host exchanges, ~3 ms a round,
    // measured), and a model that creates a column per time step (x{t}) would otherwise pay that every few steps
    size_t slab = std::max(bytes, std::min((size_t)256 << 20, std::max((size_t)8 << 20, 32 * bytes)));
    if (c->nranks > 1) {
        size_t total = 0;
        for (auto& sl : c->slabs) total += sl.size;
        slab = std::max(slab, std::min((size_t)8 << 30, total));
    }
    char* base = nullptr;
    cudaError_t e = cudaMalloc(&base, slab);
    size_t got = slab;
    if (e != cudaSuccess && slab > bytes) {
        cudaGetLastError();
        e = cudaMalloc(&base, bytes);
        got = bytes;
    }
    if (e != cudaSuccess) {
        c->err = std::string("device allocation failed: ") + cudaGetErrorString(e);
        return e == cudaErrorMemoryAllocation ? WS_ENOMEM : WS_ECUDA;
    }
    c->slabs.push_back({base, got, bytes});
    *out = base;
    return WS_OK;
}

static int grid_for(const ws_ctx* c, int64_t n, int block, int per_sm) {
    int64_t g = (n + block - 1) / block;
    int64_t cap = (int64_t)c->sm_count * per_sm;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}

static int ensure_scratch(ws_ctx* c, size_t bytes) {
    if (c->scratch_bytes >= bytes) return WS_OK;
    if (c->d_scratch != nullptr) {
        CK(c, cudaStreamSynchronize(c->stream));
        CK(c, cudaFree(c->d_scratch));
        c->d_scratch = nullptr;
        c->scratch_bytes = 0;
    }
    CK(c, cudaMalloc(&c->d_scratch, bytes));
    c->scratch_bytes = bytes;
    return WS_OK;
}
static int ensure_scratch2(ws_ctx* c, size_t bytes) {
    if (c->scratch2_bytes >= bytes) return WS_OK;
    if (c->d_scratch2 != nullptr) {
        CK(c, cudaStreamSynchronize(c->stream));
        CK(c, cudaFree(c->d_scratch2));
        c->d_scratch2 = nullptr;
        c->scratch2_bytes = 0;
    }
    bytes += bytes / 4;  // head room: the receive count varies a little from call to call
    CK(c, cudaMalloc(&c->d_scratch2, bytes));
    c->scratch2_bytes = bytes;
    return WS_OK;
}
static int ensure_h_scratch(ws_ctx* c, size_t bytes) {
    if (c->h_scratch_bytes >= bytes) return WS_OK;
    if (c->h_scratch != nullptr) {
        CK(c, cudaStreamSynchronize(c->stream));
        CK(c, cudaFreeHost(c->h_scratch));
        c->h_scratch = nullptr;
        c->h_scratch_bytes = 0;
    }
    CK(c, cudaMallocHost(&c->h_scratch, bytes));
    c->h_scratch_bytes = bytes;
    return WS_OK;
}

// ------------------------------------------------------------------------------------------
// lifecycle
// ------------------------------------------------------------------------------------------
static void reset_window(ws_ctx* c) {
    c->win = Program();
    c->win.max_regs = WS_VM_MAX_REGS;
    c->win.max_ops = WS_VM_MAX_OPS;
    c->win.max_io = WS_VM_MAX_IO;
}
static void reset_score(ws_ctx* c) {
    c->score = Program();
    c->score.score_mode = true;
    c->score.temp_base = 0;
    c->score.n_temp_slots = WS_SCORE_TEMPS;
    c->score.max_regs = WS_SCORE_MAX_REGS;
    c->score.max_ops = 1 << 30;
    c->score.max_io = 1 << 30;
    c->tape.clear();
    c->d_score_uploaded = 0;
    c->score_wide = false;
}

extern "C" int ws_abi_version(void) { return WSB200_ABI_VERSION; }

extern "C" int ws_device_count(int* out) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        if (out) *out = 0;
        return fail(nullptr, WS_ENODEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    }
    if (out) *out = n;
    return WS_OK;
}

extern "C" const char* ws_last_error(const ws_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

extern "C" int ws_create_sharded(ws_ctx** out, int64_t n_global, int rank, int nranks, const void* nccl_unique_id,
                                 int device, uint64_t seed, double ess_perc_min, int resampler) {
    if (out == nullptr) return fail(nullptr, WS_EINVAL, "ws_create: out is NULL");
    *out = nullptr;
    if (n_global <= 0) return fail(nullptr, WS_EINVAL, "ws_create: n_particles must be positive (got %lld)", (long long)n_global);
    if (n_global >= (int64_t)2147483647 - 65536) return fail(nullptr, WS_EINVAL, "ws_create: n_particles must be < 2^31 - 65536 (Int32 ancestors)");
    if (nranks < 1 || rank < 0 || rank >= nranks) return fail(nullptr, WS_EINVAL, "ws_create: bad rank %d of %d", rank, nranks);
    if (nranks > 1 && nccl_unique_id == nullptr) return fail(nullptr, WS_EINVAL, "ws_create_sharded: nccl_unique_id is NULL");
    if (nranks > 1) {
        std::string err;
        if (!load_nccl(err)) return fail(nullptr, WS_ENCCL, "%s", err.c_str());
    }
    if (resampler < 0 || resampler > 2) return fail(nullptr, WS_EINVAL, "ws_create: unknown resampler %d", resampler);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, WS_ENODEVICE, "no CUDA device available (%s); wsb200 has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    if (device < 0 || device >= ndev) return fail(nullptr, WS_EINVAL, "ws_create: device %d out of range (0..%d)", device, ndev - 1);

    ws_ctx* c = new ws_ctx();
    c->device = device;
    c->rank = rank;
    c->nranks = nranks;
    c->n_global = n_global;
    const int64_t lo = (n_global * rank) / nranks, hi = (n_global * (rank + 1)) / nranks;
    c->n = hi - lo;
    c->offset = lo;
    c->seed = seed;
    c->ess_perc_min = ess_perc_min;
    c->resampler = resampler;
    reset_window(c);
    reset_score(c);

#define CKC(call)                                                                                   \
    do {                                                                                            \
        cudaError_t e__ = (call);                                                                   \
        if (e__ != cudaSuccess) {                                                                   \
            int rc__ = fail(nullptr, e__ == cudaErrorMemoryAllocation ? WS_ENOMEM : WS_ECUDA, "%s failed: %s", #call, \
                            cudaGetErrorString(e__));                                               \
            ws_destroy(c);                                                                          \
            return rc__;                                                                            \
        }                                                                                           \
    } while (0)
    CKC(cudaSetDevice(device));
    cudaDeviceProp prop;
    CKC(cudaGetDeviceProperties(&prop, device));
    c->sm_count = prop.multiProcessorCount;
    CKC(ws_kernels_init(device));
    CKC(ws_move_kernels_init(device));
    CKC(ws_stats_init(device));
    CKC(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CKC(cudaMalloc(&c->logw, sizeof(double) * (size_t)c->n));
    CKC(cudaMalloc(&c->d_partials, sizeof(WsLse) * WS_MAX_PARTIALS));
    CKC(cudaMalloc(&c->d_red, sizeof(WsReduceOut)));
    CKC(cudaMemsetAsync(c->d_red, 0, sizeof(WsReduceOut), c->stream));
    CKC(cudaMallocHost(&c->h_red, sizeof(WsReduceOut)));
    memset(c->h_red, 0, sizeof(WsReduceOut));
    CKC(cudaMallocHost(&c->h_ring, sizeof(WsReduceOut) * ws_ctx::SPEC_RING));
    {
        const char* v = getenv("WSB200_ASYNC_RESAMPLE");
        c->async_resample = !(v != nullptr && strcmp(v, "0") == 0);
        v = getenv("WSB200_MERGED_WAIT");
        c->merged_decision_wait = !(v != nullptr && strcmp(v, "0") == 0);
        v = getenv("WSB200_SMALL_RESAMPLE");
        c->small_resample = !(v != nullptr && strcmp(v, "0") == 0);
    }
    if (nranks > 1) c->spare = std::max<int64_t>(4096, c->n / 32);
    // sharded: a margin of `spare` entries on BOTH sides, so that the search can write the ancestors of the slots
    // this rank produces for its neighbours in place, next to those of its own slots (resample_sharded)
    if (pool_alloc(c, (void**)&c->d_anc, sizeof(int32_t) * (size_t)(c->n + 2 * c->spare)) != WS_OK) {
        int rc__ = fail(nullptr, WS_ENOMEM, "%s", c->err.c_str());
        ws_destroy(c);
        return rc__;
    }
    c->d_anc += c->spare;
    {
        // genealogy budget: WSB200_GENEALOGY_BYTES, default a quarter of the device memory
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        c->genealogy_budget = total_b / 4;
        if (const char* e = getenv("WSB200_GENEALOGY_BYTES")) c->genealogy_budget = (size_t)strtoull(e, nullptr, 10);
        if (const char* e = getenv("WSB200_GENEALOGY")) c->genealogy = atoi(e) != 0;
    }
    c->n_tiles = (c->n + WS_CDF_TILE - 1) / WS_CDF_TILE;
    CKC(cudaMalloc(&c->d_tile_words, sizeof(unsigned long long) * ws_scan_words(c->n)));
    CKC(cudaMalloc(&c->d_cdf_local, sizeof(unsigned long long) * (size_t)c->n));
    CKC(cudaMalloc(&c->d_tile_counter, sizeof(unsigned int) * 2));
    CKC(cudaMalloc(&c->d_counters, sizeof(unsigned long long) * 4));
    CKC(cudaMemsetAsync(c->d_counters, 0, sizeof(unsigned long long) * 4, c->stream));
    CKC(cudaMalloc(&c->d_all_msq, sizeof(double) * 3 * (size_t)(nranks + 1)));
    CKC(cudaMalloc(&c->d_all_tot, sizeof(unsigned long long) * (size_t)(nranks + 1)));
    CKC(cudaMalloc(&c->d_all_bounds, sizeof(int32_t) * 2 * (size_t)(nranks + 1)));
#undef CKC
    if (nranks > 1) {
        ncclUniqueId id;
        memcpy(&id, nccl_unique_id, sizeof(id));
        int r = g_nccl.CommInitRank(&c->comm, nranks, id, rank);
        if (r != 0) {
            int rc = fail(nullptr, WS_ENCCL, "ncclCommInitRank failed: %s", g_nccl.GetErrorString(r));
            ws_destroy(c);
            return rc;
        }
        c->peer_slabs.resize((size_t)nranks);
        c->spare_rings.assign((size_t)nranks, WsSpareRing());
        if (const char* e = getenv("WSB200_EXCHANGE")) c->push_exchange = strcmp(e, "nccl") != 0;
        if (const char* e = getenv("WSB200_PUSH_MIN")) c->push_min = strtoll(e, nullptr, 10);
        if (cudaMalloc(&c->d_barrier, 64) != cudaSuccess || cudaMemset(c->d_barrier, 0, 64) != cudaSuccess) {
            int rc = fail(nullptr, WS_ECUDA, "cudaMalloc failed (barrier word)");
            ws_destroy(c);
            return rc;
        }
        // NCCL sets up its peer-to-peer channels on first use (hundreds of ms); do that here, not in
        // the first resampling steps: one 3-double message to and from every peer + the collectives used
        {
            bool ok = g_nccl.GroupStart() == 0;
            for (int d = 0; d < nranks && ok; ++d) {
                if (d == rank) continue;
                ok = ok && g_nccl.Send(c->d_all_msq + 3 * nranks, 3, WS_NCCL_FLOAT64, d, c->comm, c->stream) == 0;
                ok = ok && g_nccl.Recv(c->d_all_msq + 3 * d, 3, WS_NCCL_FLOAT64, d, c->comm, c->stream) == 0;
            }
            ok = ok && g_nccl.GroupEnd() == 0;
            ok = ok && g_nccl.AllGather(c->d_all_tot + nranks, c->d_all_tot, 1, WS_NCCL_UINT64, c->comm, c->stream) == 0;
            ok = ok && g_nccl.AllReduce(c->d_all_msq, c->d_all_msq, 3, WS_NCCL_FLOAT64, WS_NCCL_SUM, c->comm, c->stream) == 0;
            if (!ok || cudaStreamSynchronize(c->stream) != cudaSuccess) {
                int rc = fail(nullptr, WS_ENCCL, "NCCL warm-up exchange failed");
                ws_destroy(c);
                return rc;
            }
        }
        if (mbox_setup(c) != WS_OK) {
            int rc = fail(nullptr, WS_ENCCL, "%s", c->err.c_str());
            ws_destroy(c);
            return rc;
        }
    }
    c->logw_uniform = true;
    c->logw_base = 0.0;
    *out = c;
    return WS_OK;
}

extern "C" int ws_create(ws_ctx** out, int64_t n_particles, int device, uint64_t seed, double ess_perc_min, int resampler) {
    return ws_create_sharded(out, n_particles, 0, 1, nullptr, device, seed, ess_perc_min, resampler);
}

extern "C" int ws_nccl_unique_id(void* out128) {
    if (out128 == nullptr) return fail(nullptr, WS_EINVAL, "ws_nccl_unique_id: out is NULL");
    std::string err;
    if (!load_nccl(err)) return fail(nullptr, WS_ENCCL, "%s", err.c_str());
    ncclUniqueId id;
    int r = g_nccl.GetUniqueId(&id);
    if (r != 0) return fail(nullptr, WS_ENCCL, "ncclGetUniqueId failed: %s", g_nccl.GetErrorString(r));
    memcpy(out128, &id, sizeof(id));
    return WS_OK;
}

extern "C" int ws_destroy(ws_ctx* c) {
    if (c == nullptr) return WS_OK;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (getenv("WSB200_TRACE") && c->phase_n > 0)
        fprintf(stderr, "[wsb200 rank %d] sharded resample host ms/step: cdf+exchanges+sync %.3f | (of the exchange: peer addresses %.3f) | "
                        "search launch %.3f | exchange %.3f (steady %.3f) | (of the exchange: traced push %.3f) | of the first: plane addresses %.3f | prepare %.3f  (n=%lld)\n",
                c->rank, c->phase_ms[0] / c->phase_n, c->phase_ms[1] / c->phase_n, c->phase_ms[2] / c->phase_n,
                c->phase_ms[3] / c->phase_n, c->phase_ms[5] / std::max<int64_t>(1, c->phase_n - 6), c->phase_ms[4] / c->phase_n,
                c->phase_ms[6] / c->phase_n, c->phase_ms[7] / c->phase_n, (long long)c->phase_n);
    if (getenv("WSB200_TRACE") && c->phase_n > 0)
        fprintf(stderr, "[wsb200 rank %d] genealogy: %lld planes brought up to date to free vectors / spare rows, %lld events gathered everything, "
                        "%lld IPC mapping rounds, %zu slabs, traced values %lld\n",
                c->rank, (long long)c->trace_forced_planes, (long long)c->trace_full_gathers, (long long)c->trace_ipc_rounds, c->slabs.size(),
                (long long)c->traced_rows);
    if (c->d_scratch2) cudaFree(c->d_scratch2);
    for (auto& sl : c->slabs) cudaFree(sl.base);  // planes and ancestor vectors
    cudaFree(c->logw);
    cudaFree(c->d_partials);
    cudaFree(c->d_red);
    if (c->h_red) cudaFreeHost(c->h_red);
    if (c->h_ring) cudaFreeHost(c->h_ring);
    cudaFree(c->d_map);
    cudaFree(c->d_tile_words);
    cudaFree(c->d_logw_bak);
    cudaFree(c->d_ck_partials);
    cudaFree(c->d_ck_red);
    if (c->h_ck_red) cudaFreeHost(c->h_ck_red);
    cudaFree(c->d_cdf_local);
    cudaFree(c->d_tile_counter);
    cudaFree(c->d_heavy_F);
    cudaFree(c->d_counters);
    cudaFree(c->d_all_msq);
    cudaFree(c->d_all_tot);
    cudaFree(c->d_all_bounds);
    cudaFree(c->d_anc_src);
    cudaFree(c->d_send);
    for (auto& ps : c->peer_slabs)
        for (char* b : ps)
            if (b) cudaIpcCloseMemHandle(b);
    if (c->d_barrier) cudaFree(c->d_barrier);
    if (c->d_xmsg) cudaFree(c->d_xmsg);
    if (c->d_gen) cudaFree(c->d_gen);
    for (size_t q = 0; q < c->mbox_peer.size(); ++q)
        if ((int)q != c->rank && c->mbox_peer[q]) cudaIpcCloseMemHandle(c->mbox_peer[q]);
    if (c->d_mbox) cudaFree(c->d_mbox);
    if (c->h_mbox_err) cudaFreeHost(c->h_mbox_err);
    if (c->comm) g_nccl.CommDestroy(c->comm);
    cudaFree(c->d_score_ops);
    cudaFree(c->d_seg_ops);
    cudaFree(c->d_replay_n);
    cudaFree(c->d_replay_u);
    cudaFree(c->d_replay_e);
    cudaFree(c->d_mn);
    cudaFree(c->d_replay_v);
    cudaFree(c->d_scratch);
    if (c->h_scratch) cudaFreeHost(c->h_scratch);
    for (auto& te : c->pending_events) {
        cudaEventDestroy(te.a);
        cudaEventDestroy(te.b);
    }
    for (auto& ev : c->event_pool) {
        cudaEventDestroy(ev.first);
        cudaEventDestroy(ev.second);
    }
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return WS_OK;
}

// ------------------------------------------------------------------------------------------
// fusion window
// ------------------------------------------------------------------------------------------
static double* plane_ptr(ws_ctx* c, Plane p) { return c->cols[p.col].front[p.comp]; }

static int check_plane(ws_ctx* c, int32_t col, int32_t comp) {
    if (col < 0 || col >= (int32_t)c->cols.size()) return fail(c, WS_EINVAL, "unknown column id %d", col);
    if (comp < 0 || comp >= c->cols[col].width)
        return fail(c, WS_EINVAL, "component %d out of range for column %s (width %d)", comp, c->cols[col].name.c_str(),
                    c->cols[col].width);
    return WS_OK;
}
static int check_expr(ws_ctx* c, const ws_expr* e, const char* what) {
    if (e == nullptr || e->toks == nullptr || e->n <= 0) return fail(c, WS_EINVAL, "%s: empty expression", what);
    for (int i = 0; i < e->n; ++i)
        if (e->toks[i].op == WS_TOK_PLANE) TRY(check_plane(c, e->toks[i].col, e->toks[i].comp));
    return WS_OK;
}

static int flush_window(ws_ctx* c) {
    Program& w = c->win;
    if (w.ops.empty() && w.dirty.empty()) {
        reset_window(c);
        return WS_OK;
    }
    if (c->spec_block && !c->spec_flushing)
        return fail(c, WS_EUNSUPPORTED, "a speculative block was interrupted by a flush of the statement window");
    CK(c, cudaSetDevice(c->device));
    WsVmProgram P;
    memset(&P, 0, sizeof(P));
    P.n = c->n;
    P.particle_offset = c->offset;
    P.n_ops = (int)w.ops.size();
    P.n_loads = (int)w.loads.size();
    P.n_stores = (int)w.dirty.size();
    P.n_regs = std::max(1, w.high_water);
    // Deferred resample!: a stale plane is read through the ancestors; if the window also writes it,
    // the new values go to the back buffer (other threads still read the old order) and the buffers
    // are swapped afterwards.  A stale plane that is only written never needs its gather at all.
    {
        std::vector<Plane> loaded;
        for (auto& ld : w.loads) loaded.push_back(ld.first);
        TRY(materialize_deep(c, loaded));  // planes older than the latest event are gathered first
    }
    P.ancestors = c->d_anc;
    P.load_gather = 0u;
    std::vector<Plane> swap_after;
    for (int k = 0; k < P.n_loads; ++k) {
        const Plane pl = w.loads[k].first;
        P.load_ptr[k] = plane_ptr(c, pl);
        P.load_reg[k] = (uint8_t)w.loads[k].second;
        if (c->cols[pl.col].stale[pl.comp]) P.load_gather |= (1u << k);
    }
    for (int k = 0; k < P.n_stores; ++k) {
        const Plane pl = w.dirty[k];
        Column& col = c->cols[pl.col];
        P.store_reg[k] = (uint8_t)w.plane_reg[pl];
        bool loaded = false;
        for (auto& ld : w.loads)
            if (ld.first == pl) loaded = true;
        if (col.stale[pl.comp] && loaded) {
            if (col.back[pl.comp] == nullptr) TRY(pool_alloc(c, (void**)&col.back[pl.comp], sizeof(double) * (size_t)(c->n + c->spare)));
            P.store_ptr[k] = col.back[pl.comp];
            swap_after.push_back(pl);
        } else {
            P.store_ptr[k] = col.front[pl.comp];
        }
    }
    if (w.has_acc) {
        P.logw = c->logw;
        if (c->logw_spec) {
            P.logw_mode = 3;  // decided on the device: base = red->log_mean_w if the pending Resample fired, else read logw
            P.red = c->d_red;
        } else if (c->logw_uniform) {
            P.logw_mode = 2;
            P.logw_base = c->logw_base;
        } else {
            P.logw_mode = 1;
        }
    } else {
        P.logw_mode = 0;
    }
    if (c->spec_flushing) {
        P.n_ckpt = (int32_t)c->spec_steps.size();
        for (int32_t j = 0; j < P.n_ckpt; ++j) P.ckpt_pc[j] = (uint8_t)c->spec_steps[j].ckpt_pc;
        P.ckpt_partials = c->d_ck_partials;
        P.logw_out = c->d_logw_bak;   // ping-pong: the array the block started from stays intact (ws_exec_spec swaps the two)
    }
    const int64_t vm_tile = (int64_t)WS_VM_BLOCK * WS_VM_P;
    const int grid = (int)std::min<int64_t>(ws_vm_max_grid(P.n_regs, P.n_loads, P.n_ops, c->sm_count, P.n_ckpt), (c->n + vm_tile - 1) / vm_tile);
    P.partials = w.has_acc ? c->d_partials : nullptr;
    P.n_expect = 0;
    P.rng.seed = c->seed;
    P.rng.replay_n = c->d_replay_n;
    P.rng.replay_u = c->d_replay_u;
    P.rng.replay_e = c->d_replay_e;
    P.rng.replay_v = c->d_replay_v;
    memcpy(P.ops, w.ops.data(), sizeof(WsOp) * w.ops.size());

    const int sl_grid = ws_vm_sl_grid(P);  // straight-line executor (ws_vm_sl.cuh): it sizes its own grid
    TimedEvent te;
    timed_begin(c, KC_VM, te);
    CK(c, ws_launch_vm(P, std::max(1, grid), c->stream));
    timed_end(c, te);
    if (sl_grid > 0) c->stats.sl_passes++;
    for (auto& pl : swap_after) std::swap(c->cols[pl.col].front[pl.comp], c->cols[pl.col].back[pl.comp]);
    for (auto& pl : w.dirty) {  // written planes are in the current order
        c->cols[pl.col].stale[pl.comp] = 0;
        c->cols[pl.col].ep[pl.comp] = c->epoch;
    }
    c->stats.fused_passes++;
    c->stats.fused_statements += w.n_statements;
    if (w.has_acc) {
        c->logw_uniform = false;
        c->logw_spec = false;
        c->partials_valid = true;
        c->n_partials = sl_grid > 0 ? sl_grid : std::max(1, grid);
        c->red_valid = false;
    }
    reset_window(c);
    return WS_OK;
}

extern "C" int ws_flush(ws_ctx* c) {
    if (!c) return WS_EINVAL;
    return flush_window(c);
}
extern "C" int ws_sync(ws_ctx* c) {
    if (!c) return WS_EINVAL;
    TRY(flush_window(c));
    CK(c, cudaStreamSynchronize(c->stream));
    TRY(resolve_spec(c));
    return WS_OK;
}

// Run `body` against the fusion window; if the window overflows, flush it and lower the statement
// again into an empty window.
template <class F>
static int lower_statement(ws_ctx* c, F body) {
    for (int attempt = 0; attempt < 2; ++attempt) {
        Program snapshot = c->win;
        const uint64_t s_stream = c->next_stream;
        const int64_t s_n = c->cur_n, s_u = c->cur_u, s_e = c->cur_e, s_v = c->cur_v;
        body(c->win);
        if (!c->win.error.empty()) {
            std::string m = c->win.error;
            c->win = snapshot;
            c->next_stream = s_stream;
            c->cur_n = s_n;
            c->cur_u = s_u;
            c->cur_e = s_e;
            c->cur_v = s_v;
            return fail(c, WS_EINVAL, "%s", m.c_str());
        }
        if (!c->win.overflow) {
            c->win.end_statement();
            return WS_OK;
        }
        c->win = snapshot;
        c->next_stream = s_stream;
        c->cur_n = s_n;
        c->cur_u = s_u;
        c->cur_e = s_e;
        c->cur_v = s_v;
        if (attempt == 1 || (snapshot.ops.empty() && snapshot.dirty.empty()))
            return fail(c, WS_EUNSUPPORTED, "statement does not fit one device pass (more than %d micro-ops, %d planes or %d registers)",
                        WS_VM_MAX_OPS, WS_VM_MAX_IO, WS_VM_MAX_REGS);
        TRY(flush_window(c));
    }
    return WS_OK;
}

// Append the log-density of a statement to the score tape (device form of score!).  `lower` owns copies of
// the statement's expressions; it is lowered now into the incremental score program and kept so that
// wide tapes can be re-lowered segment by segment.
static int tape_statement(ws_ctx* c, std::function<void(Program&)> lower, std::vector<Plane> refs) {
    if (!c->tape_enabled) return WS_OK;
    if (!c->score_wide) {
        // roll-back point: sizes only (copying the program per statement is quadratic in the tape length)
        const Program::Mark mark = c->score.mark();
        lower(c->score);
        if (!c->score.error.empty()) {
            std::string m = c->score.error;
            c->score.rollback(mark);
            return fail(c, WS_EINVAL, "%s", m.c_str());
        }
        if (c->score.overflow || (int)c->score.loads.size() > WS_SCORE_MAX_LOADS) {
            // too many distinct planes for one register file: from now on the tape is folded in segments
            c->score_wide = true;
            c->score = Program();
        }
    }
    const int32_t cache_ops = c->score_wide ? 0 : (int32_t)c->score.stmt_cache_ops;
    if (!c->score_wide) c->score.end_statement();
    c->tape.push_back(TapeEntry{c->depth, c->score_wide ? 0 : (int32_t)c->score.ops.size(), cache_ops,
                                c->score_wide ? 0.0 : c->score.acc_const, std::move(lower), std::move(refs)});
    return WS_OK;
}

// sum a few host doubles over all ranks (NCCL allreduce on a small device buffer)
static int allreduce_host_doubles(ws_ctx* c, double* v, int n) {
    if (c->nranks <= 1) return WS_OK;
    TRY(ensure_scratch(c, sizeof(double) * (size_t)n));
    CK(c, cudaMemcpyAsync(c->d_scratch, v, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
    NCK(c, g_nccl.AllReduce(c->d_scratch, c->d_scratch, (size_t)n, WS_NCCL_FLOAT64, WS_NCCL_SUM, c->comm, c->stream));
    CK(c, cudaMemcpyAsync(v, c->d_scratch, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return WS_OK;
}

static wsl::RngCursor rng_cursor(ws_ctx* c) {
    return wsl::RngCursor{&c->next_stream, &c->cur_n, &c->cur_u, &c->cur_e, c->n_global, &c->cur_v};
}

static int check_replay(ws_ctx* c) {
    if (c->d_replay_n != nullptr && c->cur_n > c->replay_n_len)
        return fail(c, WS_EREPLAY, "replay normals exhausted (%lld needed, %lld installed)", (long long)c->cur_n, (long long)c->replay_n_len);
    if (c->d_replay_e != nullptr && c->cur_e > c->replay_e_len)
        return fail(c, WS_EREPLAY, "replay exponentials exhausted (%lld needed, %lld installed)", (long long)c->cur_e, (long long)c->replay_e_len);
    if (c->d_replay_v != nullptr && c->cur_v > c->replay_v_len)
        return fail(c, WS_EREPLAY, "replay variates exhausted (%lld needed, %lld installed)", (long long)c->cur_v, (long long)c->replay_v_len);
    if (c->d_replay_u != nullptr && c->cur_u > c->replay_u_len)
        return fail(c, WS_EREPLAY, "replay uniforms exhausted (%lld needed, %lld installed)", (long long)c->cur_u, (long long)c->replay_u_len);
    return WS_OK;
}

// ------------------------------------------------------------------------------------------
// state scalars
// ------------------------------------------------------------------------------------------
extern "C" int ws_n_particles(const ws_ctx* c, int64_t* n_local, int64_t* n_global) {
    if (!c) return WS_EINVAL;
    if (n_local) *n_local = c->n;
    if (n_global) *n_global = c->n_global;
    return WS_OK;
}
extern "C" int ws_get_flags(ws_ctx* c, int* resampled, int* weights_changed, int64_t* depth) {
    if (!c) return WS_EINVAL;
    if (resampled) TRY(resolve_spec(c));   // `if resampled` is host control flow: this is where a pending decision is awaited
    if (resampled) *resampled = c->resampled ? 1 : 0;
    if (weights_changed) *weights_changed = c->weights_changed ? 1 : 0;
    if (depth) *depth = c->depth;
    return WS_OK;
}
extern "C" int ws_set_flags(ws_ctx* c, int resampled, int weights_changed) {
    if (!c) return WS_EINVAL;
    TRY(resolve_spec(c));
    c->resampled = resampled != 0;
    c->weights_changed = weights_changed != 0;
    return WS_OK;
}
extern "C" int ws_set_depth(ws_ctx* c, int64_t depth) {
    if (!c) return WS_EINVAL;
    c->depth = depth;
    return WS_OK;
}
extern "C" int ws_set_ess_perc_min(ws_ctx* c, double v) {
    if (!c) return WS_EINVAL;
    c->ess_perc_min = v;
    c->red_valid = false;  // the cached resampling decision depended on the old threshold
    return WS_OK;
}
extern "C" int ws_get_ess_perc_min(const ws_ctx* c, double* out) {
    if (!c || !out) return WS_EINVAL;
    *out = c->ess_perc_min;
    return WS_OK;
}
extern "C" int ws_begin_run(ws_ctx* c) {
    if (!c) return WS_EINVAL;
    TRY(flush_window(c));
    c->depth = 0;
    c->spec_immediate = 0;
    reset_score(c);
    return WS_OK;
}

// ------------------------------------------------------------------------------------------
// store
// ------------------------------------------------------------------------------------------
extern "C" int ws_col_ensure(ws_ctx* c, const char* name, int32_t width, int32_t* id_out) {
    if (!c || !name) return WS_EINVAL;
    if (width < 1 || width > 4096) return fail(c, WS_EINVAL, "column %s: width %d out of range", name, width);
    auto it = c->col_index.find(name);
    if (it != c->col_index.end()) {
        if (c->cols[it->second].width != width)
            return fail(c, WS_EINVAL, "column %s already exists with width %d (requested %d)", name, c->cols[it->second].width, width);
        if (id_out) *id_out = it->second;
        return WS_OK;
    }
    CK(c, cudaSetDevice(c->device));
    Column col;
    col.name = name;
    col.width = width;
    col.stale.assign((size_t)width, 0);
    col.ep.assign((size_t)width, c->epoch);
    for (int k = 0; k < width; ++k) {
        double *f = nullptr, *b = nullptr;
        TRY(pool_alloc(c, (void**)&f, sizeof(double) * (size_t)(c->n + c->spare)));
        // the back buffer (target of a gather) is created on first use, except in sharded runs whose
        // exchange writes straight into it
        if (c->nranks > 1) TRY(pool_alloc(c, (void**)&b, sizeof(double) * (size_t)(c->n + c->spare)));
        CK(c, cudaMemsetAsync(f, 0, sizeof(double) * (size_t)c->n, c->stream));
        col.front.push_back(f);
        col.back.push_back(b);
    }
    c->cols.push_back(col);
    const int32_t id = (int32_t)c->cols.size() - 1;
    c->col_index[name] = id;
    if (id_out) *id_out = id;
    return WS_OK;
}
extern "C" int ws_col_lookup(const ws_ctx* c, const char* name, int32_t* id_out, int32_t* width_out) {
    if (!c || !name) return WS_EINVAL;
    auto it = c->col_index.find(name);
    if (it == c->col_index.end()) {
        if (id_out) *id_out = -1;
        if (width_out) *width_out = 0;
        return WS_OK;
    }
    if (id_out) *id_out = it->second;
    if (width_out) *width_out = c->cols[it->second].width;
    return WS_OK;
}
extern "C" int ws_col_count(const ws_ctx* c, int32_t* out) {
    if (!c || !out) return WS_EINVAL;
    *out = (int32_t)c->cols.size();
    return WS_OK;
}
extern "C" int ws_col_info(const ws_ctx* c, int32_t id, char* name_buf, int32_t name_buf_len, int32_t* width_out) {
    if (!c) return WS_EINVAL;
    if (id < 0 || id >= (int32_t)c->cols.size()) return WS_EINVAL;
    if (name_buf && name_buf_len > 0) {
        strncpy(name_buf, c->cols[id].name.c_str(), (size_t)name_buf_len - 1);
        name_buf[name_buf_len - 1] = 0;
    }
    if (width_out) *width_out = c->cols[id].width;
    return WS_OK;
}
extern "C" int ws_col_download(ws_ctx* c, int32_t id, double* host_out) {
    if (!c || !host_out) return WS_EINVAL;
    if (id < 0 || id >= (int32_t)c->cols.size()) return fail(c, WS_EINVAL, "unknown column id %d", id);
    TRY(flush_window(c));
    CK(c, cudaSetDevice(c->device));
    const Column& col = c->cols[id];
    for (int k = 0; k < col.width; ++k) {
        const double* src = col.front[k];
        const int32_t* map = nullptr;
        if (col.stale[k]) TRY(map_for_epoch(c, col.ep[k], &map));   // nullptr: only identity events in between
        if (map != nullptr) {
            // read through the (composed) ancestors into scratch: the plane itself stays in its old order,
            // so exporting a long history costs one 4-byte chain step per event, not a gather of everything
            TRY(ensure_scratch(c, sizeof(double) * (size_t)c->n));
            WsGatherParams G;
            memset(&G, 0, sizeof(G));
            G.n = c->n;
            G.ancestors = map;
            G.n_planes = 1;
            G.src[0] = col.front[k];
            G.dst[0] = c->d_scratch;
            TimedEvent te;
            timed_begin(c, KC_GATHER, te);
            CK(c, ws_launch_gather(G, grid_for(c, c->n, 256, 8), c->stream));
            timed_end(c, te);
            src = c->d_scratch;
        }
        CK(c, cudaMemcpyAsync(host_out + (size_t)k * c->n, src, sizeof(double) * (size_t)c->n, cudaMemcpyDeviceToHost, c->stream));
        if (map != nullptr) CK(c, cudaStreamSynchronize(c->stream));  // scratch is reused by the next plane
    }
    CK(c, cudaStreamSynchronize(c->stream));
    c->stats.d2h_bytes += (int64_t)sizeof(double) * c->n * col.width;
    return WS_OK;
}
extern "C" int ws_col_upload(ws_ctx* c, int32_t id, const double* host_in) {
    if (!c || !host_in) return WS_EINVAL;
    if (id < 0 || id >= (int32_t)c->cols.size()) return fail(c, WS_EINVAL, "unknown column id %d", id);
    TRY(flush_window(c));
    Column& col = c->cols[id];
    for (auto& st : col.stale) st = 0;  // the whole column is overwritten: its deferred gather is moot
    for (auto& e : col.ep) e = c->epoch;
    for (int k = 0; k < col.width; ++k)
        CK(c, cudaMemcpyAsync(col.front[k], host_in + (size_t)k * c->n, sizeof(double) * (size_t)c->n, cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    c->stats.h2d_bytes += (int64_t)sizeof(double) * c->n * col.width;
    return WS_OK;
}

static int materialize_logw(ws_ctx* c) {
    TRY(resolve_spec(c));
    if (!c->logw_uniform) return WS_OK;
    TimedEvent te;
    timed_begin(c, KC_FILL, te);
    CK(c, ws_launch_fill(c->logw, c->logw_base, c->n, grid_for(c, c->n, 256, 8), c->stream));
    timed_end(c, te);
    c->logw_uniform = false;
    c->partials_valid = false;
    return WS_OK;
}

extern "C" int ws_weights_download(ws_ctx* c, double* host_out) {
    if (!c || !host_out) return WS_EINVAL;
    TRY(flush_window(c));
    TRY(materialize_logw(c));
    CK(c, cudaMemcpyAsync(host_out, c->logw, sizeof(double) * (size_t)c->n, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    c->stats.d2h_bytes += (int64_t)sizeof(double) * c->n;
    return WS_OK;
}
extern "C" int ws_weights_upload(ws_ctx* c, const double* host_in, int mark_changed) {
    if (!c || !host_in) return WS_EINVAL;
    TRY(flush_window(c));
    TRY(resolve_spec(c));
    CK(c, cudaMemcpyAsync(c->logw, host_in, sizeof(double) * (size_t)c->n, cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    c->stats.h2d_bytes += (int64_t)sizeof(double) * c->n;
    c->logw_uniform = false;
    c->partials_valid = false;
    c->red_valid = false;
    if (mark_changed) c->weights_changed = true;
    return WS_OK;
}

// ------------------------------------------------------------------------------------------
// statements
// ------------------------------------------------------------------------------------------
extern "C" int ws_assign(ws_ctx* c, int32_t col, int32_t comp, const ws_expr* rhs) {
    if (!c) return WS_EINVAL;
    TRY(check_plane(c, col, comp));
    TRY(check_expr(c, rhs, "ws_assign"));
    if (!c->record_only) {
        TRY(lower_statement(c, [&](Program& p) { wsl::stmt_assign(p, Plane{col, comp}, *rhs); }));
    }
    c->depth++;
    return WS_OK;
}

extern "C" int ws_assign_vec(ws_ctx* c, int32_t col, int32_t d, const ws_expr* rhs) {
    if (!c || !rhs) return WS_EINVAL;
    if (col < 0 || col >= (int32_t)c->cols.size()) return fail(c, WS_EINVAL, "unknown column id %d", col);
    if (d != c->cols[col].width) return fail(c, WS_EINVAL, "ws_assign_vec: %d expressions for column %s of width %d", d, c->cols[col].name.c_str(), c->cols[col].width);
    for (int j = 0; j < d; ++j) TRY(check_expr(c, &rhs[j], "ws_assign_vec"));
    if (!c->record_only) {
        bool hazard = false;
        for (int j = 0; j < d; ++j)
            for (int i = 0; i < rhs[j].n; ++i)
                if (rhs[j].toks[i].op == WS_TOK_PLANE && rhs[j].toks[i].col == col && rhs[j].toks[i].comp != j) hazard = true;
        if (hazard || d <= 8) {
            TRY(lower_statement(c, [&](Program& p) { wsl::stmt_assign_vec(p, col, d, rhs); }));
        } else {
            // wide vectors (theta .= zeros(J)): independent components, lowered one by one so that the
            // fusion window can be flushed in between
            for (int j = 0; j < d; ++j)
                TRY(lower_statement(c, [&](Program& p) { wsl::stmt_assign(p, Plane{col, j}, rhs[j]); }));
        }
    }
    c->depth++;
    return WS_OK;
}

extern "C" int ws_sample_normal(ws_ctx* c, int32_t col, int32_t comp, const ws_expr* mu, const ws_expr* sigma) {
    if (!c) return WS_EINVAL;
    TRY(check_plane(c, col, comp));
    TRY(check_expr(c, mu, "ws_sample_normal(mu)"));
    TRY(check_expr(c, sigma, "ws_sample_normal(sigma)"));
    if (!c->record_only) {
        wsl::RngCursor rc = rng_cursor(c);
        TRY(lower_statement(c, [&](Program& p) { wsl::stmt_sample_normal(p, rc, Plane{col, comp}, *mu, *sigma); }));
        TRY(check_replay(c));
    }
    {
        auto ox = std::make_shared<OwnedExprs>(std::initializer_list<std::pair<const ws_expr*, int>>{{mu, 1}, {sigma, 1}});
        std::vector<Plane> refs{Plane{col, comp}};
        ox->planes(refs);
        TRY(tape_statement(c, [ox, col, comp](Program& p) { wsl::score_sample_normal(p, Plane{col, comp}, ox->ex[0], ox->ex[1]); }, refs));
    }
    c->depth++;
    return WS_OK;
}

extern "C" int ws_sample_exponential(ws_ctx* c, int32_t col, int32_t comp, const ws_expr* theta) {
    if (!c) return WS_EINVAL;
    TRY(check_plane(c, col, comp));
    TRY(check_expr(c, theta, "ws_sample_exponential(theta)"));
    if (!c->record_only) {
        wsl::RngCursor rc = rng_cursor(c);
        TRY(lower_statement(c, [&](Program& p) { wsl::stmt_sample_exponential(p, rc, Plane{col, comp}, *theta); }));
        TRY(check_replay(c));
    }
    {
        auto ox = std::make_shared<OwnedExprs>(std::initializer_list<std::pair<const ws_expr*, int>>{{theta, 1}});
        std::vector<Plane> refs{Plane{col, comp}};
        ox->planes(refs);
        TRY(tape_statement(c, [ox, col, comp](Program& p) { wsl::score_sample_exponential(p, Plane{col, comp}, ox->ex[0]); }, refs));
    }
    c->depth++;
    return WS_OK;
}

static int mvn_factors(ws_ctx* c, int d, const double* cov, std::vector<double>& L, std::vector<double>& Linv, double& c0) {
    if (d < 1 || d > 16) return fail(c, WS_EUNSUPPORTED, "MvNormal dimension %d outside 1..16", d);
    if (cov == nullptr) return fail(c, WS_EINVAL, "MvNormal: covariance is NULL");
    if (!wsl::mvnormal_factors(d, cov, L, Linv, c0)) return fail(c, WS_ENUMERIC, "MvNormal: covariance is not positive definite");
    return WS_OK;
}

extern "C" int ws_sample_mvnormal(ws_ctx* c, int32_t col, int32_t d, const ws_expr* mu, const double* cov) {
    if (!c || !mu) return WS_EINVAL;
    if (col < 0 || col >= (int32_t)c->cols.size()) return fail(c, WS_EINVAL, "unknown column id %d", col);
    if (d != c->cols[col].width) return fail(c, WS_EINVAL, "ws_sample_mvnormal: dimension %d but column %s has width %d", d, c->cols[col].name.c_str(), c->cols[col].width);
    for (int j = 0; j < d; ++j) TRY(check_expr(c, &mu[j], "ws_sample_mvnormal(mu)"));
    std::vector<double> L, Linv;
    double c0;
    TRY(mvn_factors(c, d, cov, L, Linv, c0));
    if (!c->record_only) {
        wsl::RngCursor rc = rng_cursor(c);
        TRY(lower_statement(c, [&](Program& p) { wsl::stmt_sample_mvnormal(p, rc, col, d, mu, L); }));
        TRY(check_replay(c));
    }
    {
        auto ox = std::make_shared<OwnedExprs>(std::initializer_list<std::pair<const ws_expr*, int>>{{mu, d}});
        std::vector<Plane> refs;
        for (int j = 0; j < d; ++j) refs.push_back(Plane{col, j});
        ox->planes(refs);
        TRY(tape_statement(c, [ox, col, d, Linv, c0](Program& p) { wsl::score_sample_mvnormal(p, col, d, ox->ex.data(), Linv, c0); }, refs));
    }
    c->depth++;
    return WS_OK;
}

extern "C" int ws_observe_normal(ws_ctx* c, const ws_expr* obs, const ws_expr* mu, const ws_expr* sigma) {
    if (!c) return WS_EINVAL;
    TRY(check_expr(c, obs, "ws_observe_normal(obs)"));
    TRY(check_expr(c, mu, "ws_observe_normal(mu)"));
    TRY(check_expr(c, sigma, "ws_observe_normal(sigma)"));
    auto body = [&](Program& p) { wsl::stmt_observe_normal(p, *obs, *mu, *sigma); };
    if (!c->record_only) {
        TRY(lower_statement(c, body));
        c->weights_changed = true;
    }
    {
        auto ox = std::make_shared<OwnedExprs>(std::initializer_list<std::pair<const ws_expr*, int>>{{obs, 1}, {mu, 1}, {sigma, 1}});
        std::vector<Plane> refs;
        ox->planes(refs);
        TRY(tape_statement(c, [ox](Program& p) { wsl::stmt_observe_normal(p, ox->ex[0], ox->ex[1], ox->ex[2]); }, refs));
    }
    c->depth++;
    return WS_OK;
}

extern "C" int ws_observe_exponential(ws_ctx* c, const ws_expr* obs, const ws_expr* theta) {
    if (!c) return WS_EINVAL;
    TRY(check_expr(c, obs, "ws_observe_exponential(obs)"));
    TRY(check_expr(c, theta, "ws_observe_exponential(theta)"));
    auto body = [&](Program& p) { wsl::stmt_observe_exponential(p, *obs, *theta); };
    if (!c->record_only) {
        TRY(lower_statement(c, body));
        c->weights_changed = true;
    }
    {
        auto ox = std::make_shared<OwnedExprs>(std::initializer_list<std::pair<const ws_expr*, int>>{{obs, 1}, {theta, 1}});
        std::vector<Plane> refs;
        ox->planes(refs);
        TRY(tape_statement(c, [ox](Program& p) { wsl::stmt_observe_exponential(p, ox->ex[0], ox->ex[1]); }, refs));
    }
    c->depth++;
    return WS_OK;
}

extern "C" int ws_observe_mvnormal(ws_ctx* c, int32_t d, const ws_expr* obs, const ws_expr* mu, const double* cov) {
    if (!c || !obs || !mu) return WS_EINVAL;
    std::vector<double> L, Linv;
    double c0;
    TRY(mvn_factors(c, d, cov, L, Linv, c0));
    for (int j = 0; j < d; ++j) {
        TRY(check_expr(c, &obs[j], "ws_observe_mvnormal(obs)"));
        TRY(check_expr(c, &mu[j], "ws_observe_mvnormal(mu)"));
    }
    auto body = [&](Program& p) { wsl::stmt_observe_mvnormal(p, d, obs, mu, Linv, c0); };
    if (!c->record_only) {
        TRY(lower_statement(c, body));
        c->weights_changed = true;
    }
    {
        auto ox = std::make_shared<OwnedExprs>(std::initializer_list<std::pair<const ws_expr*, int>>{{obs, d}, {mu, d}});
        std::vector<Plane> refs;
        ox->planes(refs);
        TRY(tape_statement(c, [ox, d, Linv, c0](Program& p) { wsl::stmt_observe_mvnormal(p, d, ox->ex.data(), ox->ex.data() + d, Linv, c0); }, refs));
    }
    c->depth++;
    return WS_OK;
}

extern "C" int ws_weight_expr(ws_ctx* c, const ws_expr* term) {
    if (!c) return WS_EINVAL;
    TRY(check_expr(c, term, "ws_weight_expr"));
    auto body = [&](Program& p) { wsl::stmt_weight_expr(p, *term); };
    if (!c->record_only) {
        TRY(lower_statement(c, body));
        c->weights_changed = true;
    }
    {
        auto ox = std::make_shared<OwnedExprs>(std::initializer_list<std::pair<const ws_expr*, int>>{{term, 1}});
        std::vector<Plane> refs;
        ox->planes(refs);
        TRY(tape_statement(c, [ox](Program& p) { wsl::stmt_weight_expr(p, ox->ex[0]); }, refs));
    }
    c->depth++;
    return WS_OK;
}

extern "C" int ws_sample_expr(ws_ctx* c, int32_t col, int32_t comp, const ws_expr* sampler, const ws_expr* weighter,
                              const ws_expr* logpdf) {
    if (!c) return WS_EINVAL;
    TRY(check_plane(c, col, comp));
    TRY(check_expr(c, sampler, "ws_sample_expr(sampler)"));
    if (weighter) TRY(check_expr(c, weighter, "ws_sample_expr(weighter)"));
    if (logpdf) TRY(check_expr(c, logpdf, "ws_sample_expr(logpdf)"));
    if (!c->record_only) {
        wsl::RngCursor rc = rng_cursor(c);
        TRY(lower_statement(c, [&](Program& p) { wsl::stmt_sample_expr(p, rc, Plane{col, comp}, *sampler, weighter); }));
        TRY(check_replay(c));
        if (weighter) c->weights_changed = true;
    }
    if (logpdf) {
        auto ox = std::make_shared<OwnedExprs>(std::initializer_list<std::pair<const ws_expr*, int>>{{logpdf, 1}});
        std::vector<Plane> refs{Plane{col, comp}};
        ox->planes(refs);
        TRY(tape_statement(c, [ox](Program& p) { wsl::stmt_weight_expr(p, ox->ex[0]); }, refs));
    }
    c->depth++;
    return WS_OK;
}

extern "C" int ws_sample_importance_normal(ws_ctx* c, int32_t col, int32_t comp, double pm, double ps, double tm, double ts) {
    if (!c) return WS_EINVAL;
    TRY(check_plane(c, col, comp));
    if (!(ps > 0.0) || !(ts > 0.0)) return fail(c, WS_EINVAL, "importance_kernel: standard deviations must be positive");
    if (!c->record_only) {
        wsl::RngCursor rc = rng_cursor(c);
        TRY(lower_statement(c, [&](Program& p) { wsl::stmt_importance_normal(p, rc, Plane{col, comp}, pm, ps, tm, ts); }));
        TRY(check_replay(c));
        c->weights_changed = true;
    }
    TRY(tape_statement(c, [col, comp, tm, ts](Program& p) {
        p.acc_normal_logpdf(Val::lin(0.0, 1.0, p.reg_for_read(Plane{col, comp})), Val::constant(tm), Val::constant(ts));
    }, std::vector<Plane>{Plane{col, comp}}));
    c->depth++;
    return WS_OK;
}

// ------------------------------------------------------------------------------------------
// reductions / resampling
// ------------------------------------------------------------------------------------------
// Bring the host's view up to date with the Resample steps it issued without looking at their outcome
// (ws_resample_async): wait for the stream, read their records from the pinned ring in order.
static int resolve_spec(ws_ctx* c) {
    if (c->spec_pending == 0) return WS_OK;
    c->spec_immediate = (c->spec_pending == 1 && c->logw_spec) ? c->spec_immediate + 1 : 0;
    CK(c, cudaSetDevice(c->device));
    CK(c, cudaStreamSynchronize(c->stream));
    c->stats.d2h_bytes += (int64_t)sizeof(WsReduceOut) * c->spec_pending;
    WsReduceOut last{};
    for (int64_t k = c->spec_head - c->spec_pending; k < c->spec_head; ++k) {
        last = c->h_ring[k % ws_ctx::SPEC_RING];
        if (last.do_resample) {
            c->resampled = true;
            c->stats.resamples_done++;
        } else {
            c->resampled = false;
            for (auto& v : c->anc_live)  // reads of planes that are behind this event skip it from now on
                if (v.event == c->ring_event[k % ws_ctx::SPEC_RING]) v.identity = true;
        }
    }
    c->spec_pending = 0;
    if (c->last_info_pending) {
        c->last_info.fired = 1;
        c->last_info.resampled = last.do_resample ? 1 : 0;
        c->last_info.ess_perc = last.ess_perc;
        c->last_info.log_mean_w = last.log_mean_w;
        c->last_info.n_clamped = -1;
        c->last_info_pending = false;
    }
    if (c->logw_spec) {
        // no weighting pass has run since the last of them: its outcome decides what the log-weights are
        c->logw_spec = false;
        if (last.do_resample) {
            c->logw_uniform = true;   // fill!(weights, mean_logW), kept symbolic
            c->logw_base = last.log_mean_w;
            c->partials_valid = false;
            c->red_valid = false;
        } else {
            c->logw_uniform = false;  // the array and the reduction of it that decided are both still current
            *c->h_red = last;
            c->partials_valid = true;
            c->red_valid = true;
        }
    }
    return WS_OK;
}

// Make d_red / h_red describe the current log-weights (m, S, Q, lse, ESS%, decision).
static int ensure_reduced(ws_ctx* c, bool for_resample = false, bool wait = true) {
    TRY(flush_window(c));
    TRY(resolve_spec(c));
    if (c->red_valid) return WS_OK;
    CK(c, cudaSetDevice(c->device));
    if (c->logw_uniform) TRY(materialize_logw(c));
    if (!c->partials_valid) {
        const int grid = std::min(grid_for(c, c->n, 256, 8), WS_MAX_PARTIALS);
        TimedEvent te;
        timed_begin(c, KC_REDUCE, te);
        CK(c, ws_launch_reduce_logw(c->logw, c->n, c->d_partials, grid, c->stream));
        timed_end(c, te);
        c->n_partials = grid;
        c->partials_valid = true;
    }
    TimedEvent te;
    unsigned long long* ties = for_resample ? c->d_counters + 3 : nullptr;   // knife-edge decisions (ws_get_ess_ties)
    if (c->nranks > 1 && c->mbox_on) {
        // shard reduction, exchange of the (m, S, Q) triples and their combination in ONE kernel (ws_finalize_mbox_kernel)
        const WsMailbox M = mbox_next(c, 1);
        timed_begin(c, KC_FINALIZE, te);
        CK(c, ws_launch_finalize_mbox(c->d_partials, c->n_partials, c->n_global, c->ess_perc_min, c->d_red, c->d_all_msq, ties, M, c->stream));
        timed_end(c, te);
    } else {
        timed_begin(c, KC_FINALIZE, te);
        CK(c, ws_launch_finalize(c->d_partials, c->n_partials, c->n_global, c->ess_perc_min, c->d_red, c->stream, c->nranks > 1 ? nullptr : ties));
        timed_end(c, te);
        if (c->nranks > 1) {
            // every rank reduces its shard; the (m, S, Q) triples are allgathered and combined in rank order
            NCK(c, g_nccl.AllGather(c->d_red, c->d_all_msq, 3, WS_NCCL_FLOAT64, c->comm, c->stream));
            timed_begin(c, KC_FINALIZE, te);
            CK(c, ws_launch_finalize_global(c->d_all_msq, c->nranks, c->n_global, c->ess_perc_min, c->d_red, c->stream, ties));
            timed_end(c, te);
        }
    }
    CK(c, cudaMemcpyAsync(c->h_red, c->d_red, sizeof(WsReduceOut), cudaMemcpyDeviceToHost, c->stream));
    c->stats.d2h_bytes += (int64_t)sizeof(WsReduceOut);
    if (!wait) return WS_OK;   // the caller's next wait on the stream delivers *h_red (it then sets red_valid)
    CK(c, cudaStreamSynchronize(c->stream));
    TRY(mbox_check(c));
    c->red_valid = true;
    return WS_OK;
}

static int gather_planes(ws_ctx* c, const int32_t* d_anc, const std::vector<Plane>& which) {
    // resample!(store, indices) for the given planes: front -> back through the ancestors, then swap
    for (size_t p0 = 0; p0 < which.size(); p0 += WS_GATHER_MAX_PLANES) {
        WsGatherParams G;
        memset(&G, 0, sizeof(G));
        G.n = c->n;
        G.ancestors = d_anc;
        G.n_planes = (int)std::min((size_t)WS_GATHER_MAX_PLANES, which.size() - p0);
        for (int k = 0; k < G.n_planes; ++k) {
            const Plane pl = which[p0 + k];
            Column& col = c->cols[pl.col];
            if (col.back[pl.comp] == nullptr)  // back buffers are created on first use
                TRY(pool_alloc(c, (void**)&col.back[pl.comp], sizeof(double) * (size_t)(c->n + c->spare)));
            G.src[k] = col.front[pl.comp];
            G.dst[k] = col.back[pl.comp];
        }
        TimedEvent te;
        timed_begin(c, KC_GATHER, te);
        CK(c, ws_launch_gather(G, grid_for(c, c->n, 256, 8), c->stream));
        timed_end(c, te);
    }
    for (auto& pl : which) {
        std::swap(c->cols[pl.col].front[pl.comp], c->cols[pl.col].back[pl.comp]);
        c->cols[pl.col].stale[pl.comp] = 0;
        c->cols[pl.col].ep[pl.comp] = c->epoch;
    }
    return WS_OK;
}

// ---- genealogy ---------------------------------------------------------------------------------------
static const int32_t* anc_of_event(const ws_ctx* c, int64_t event) {
    for (auto& v : c->anc_live)
        if (v.event == event) return v.ptr;
    return nullptr;
}

// Device map "slot of the current epoch -> row of a plane stored in the order of epoch `ep`":
// nullptr for ep == epoch (identity), the latest ancestors for ep == epoch - 1, otherwise the composition
// a_{ep+1}[... a_epoch[i]], continued from the cached map when that was composed for a later epoch.
static int map_for_epoch(ws_ctx* c, int64_t ep, const int32_t** out) {
    *out = nullptr;
    if (ep >= c->epoch) return WS_OK;
    auto is_identity = [&](int64_t event) {
        for (auto& v : c->anc_live)
            if (v.event == event) return v.identity;
        return false;
    };
    while (ep < c->epoch && is_identity(ep + 1)) ++ep;  // leading identity events: the plane is effectively newer
    if (ep >= c->epoch) return WS_OK;
    if (ep == c->epoch - 1) {
        // (d_anc itself is the vector of the NEXT event while a resampling step is between its commit and its end)
        const int32_t* a = anc_of_event(c, c->epoch);
        *out = a != nullptr ? a : c->d_anc;
        return WS_OK;
    }
    if (c->map_E == c->epoch && c->map_ep == ep) {
        *out = c->d_map;
        return WS_OK;
    }
    if (c->d_map == nullptr) CK(c, cudaMalloc(&c->d_map, sizeof(int32_t) * (size_t)c->n));
    int64_t from = c->epoch;  // events still to apply: from, from-1, ..., ep+1
    const int32_t* start = nullptr;
    if (c->map_E == c->epoch && c->map_ep > ep && c->map_ep < c->epoch) {
        from = c->map_ep;
        start = c->d_map;
    }
    while (from > ep) {
        WsComposeParams P;
        memset(&P, 0, sizeof(P));
        P.n = c->n;
        P.n_rows = c->n;
        while (from > ep && P.n_chain < WS_COMPOSE_MAX_CHAIN) {
            const int32_t* a = anc_of_event(c, from);
            if (a == nullptr) return fail(c, WS_EINVAL, "genealogy: ancestors of event %lld were released", (long long)from);
            if (!is_identity(from)) P.chain[P.n_chain++] = a;
            --from;
        }
        if (P.n_chain == 0 && start == nullptr) {  // nothing but identities so far: keep walking, or the map is the identity
            if (from > ep) continue;
            c->map_E = -1;
            return WS_OK;
        }
        CK(c, ws_launch_compose(P, c->d_map, start, c->stream));
        c->stats.kernel_launches++;
        start = c->d_map;
    }
    c->map_E = c->epoch;
    c->map_ep = ep;
    *out = c->d_map;
    return WS_OK;
}

// Apply the deferred gather to every plane (or to the given ones) that is still in an older order.
static int materialize_planes(ws_ctx* c, const std::vector<Plane>* only) {
    if (!c->anc_pending) return WS_OK;
    std::map<int64_t, std::vector<Plane>, std::greater<int64_t>> by_ep;  // newest first: the map cache continues downwards
    auto take = [&](Plane pl) {
        Column& col = c->cols[pl.col];
        if (col.stale[pl.comp]) {
            auto& v = by_ep[col.ep[pl.comp]];
            if (std::find(v.begin(), v.end(), pl) == v.end()) v.push_back(pl);
        }
    };
    if (only) {
        for (auto& pl : *only) take(pl);
    } else {
        for (int32_t ci = 0; ci < (int32_t)c->cols.size(); ++ci)
            for (int32_t k = 0; k < c->cols[ci].width; ++k) take(Plane{ci, k});
    }
    for (auto& g : by_ep) {
        const int32_t* map = nullptr;
        TRY(map_for_epoch(c, g.first, &map));
        if (map == nullptr) {
            // every event these planes are behind was a queued step that did not fire (identity): nothing to move
            for (auto& pl : g.second) {
                c->cols[pl.col].stale[pl.comp] = 0;
                c->cols[pl.col].ep[pl.comp] = c->epoch;
            }
            continue;
        }
        TRY(gather_planes(c, map, g.second));
    }
    if (!only) c->anc_pending = false;
    return WS_OK;
}

// Score folds and moves read the planes of the score tape (and the move targets), nothing else: a long
// history of untouched columns stays untouched.
static int materialize_tape_planes(ws_ctx* c, int32_t n_extra, const int32_t* col, const int32_t* comp) {
    std::vector<Plane> need;
    for (auto& ld : c->score.loads) need.push_back(ld.first);
    for (auto& te : c->tape)
        for (auto& pl : te.refs) need.push_back(pl);
    for (int32_t t = 0; t < n_extra; ++t) need.push_back(Plane{col[t], comp[t]});
    std::vector<Plane> ok;
    for (auto& pl : need)
        if (pl.col >= 0 && pl.col < (int32_t)c->cols.size() && pl.comp >= 0 && pl.comp < c->cols[pl.col].width) ok.push_back(pl);
    return materialize_planes(c, &ok);
}

// Planes older than the latest event cannot be read through d_anc by the fused pass: gather those first.
static int materialize_deep(ws_ctx* c, const std::vector<Plane>& planes) {
    std::vector<Plane> deep;
    for (auto& pl : planes) {
        const Column& col = c->cols[pl.col];
        if (col.stale[pl.comp] && col.ep[pl.comp] < c->epoch - 1) deep.push_back(pl);
    }
    if (deep.empty()) return WS_OK;
    return materialize_planes(c, &deep);
}

// Called before a resampling event writes a new ancestor vector.  Without genealogy (eager mode, sharded runs whose
// exchange cannot carry stale planes) every stale plane is gathered and the single vector is reused.  With it, vectors
// no plane needs any more are recycled, the retained ones are capped by the byte budget (oldest planes gathered first),
// and a fresh vector becomes d_anc.  Two halves: `prepare` does everything that may MOVE planes (a sharded step
// announces its plane addresses to the other ranks afterwards, and may do this before it knows whether the step fires);
// `commit` takes the vector.  Every decision in here depends only on what all ranks of a sharded state know alike.
static bool shard_genealogy_ok(const ws_ctx* c) { return c->push_exchange && c->push_min == 0; }
static int64_t spare_ring_cap(const ws_ctx* c, int q) {
    return ws_spare_rows(ws_rank_lo(c->n_global, c->nranks, q + 1) - ws_rank_lo(c->n_global, c->nranks, q));
}
static int prepare_resample_event(ws_ctx* c) {
    c->event_keeps = c->genealogy && c->lazy_gather && (c->nranks == 1 || shard_genealogy_ok(c));
    if (!c->event_keeps) {
        TRY(materialize_planes(c));
        for (auto& rg : c->spare_rings) rg.clear();
        return WS_OK;
    }
    auto min_ep = [&]() {
        int64_t m = c->epoch;
        for (auto& col : c->cols)
            for (int k = 0; k < col.width; ++k)
                if (col.stale[k]) m = std::min(m, col.ep[k]);
        return m;
    };
    auto gc = [&]() {
        const int64_t m = min_ep();  // events <= m are not needed by anybody
        while (!c->anc_live.empty() && c->anc_live.front().event <= m) {
            c->anc_pool.push_back(c->anc_live.front().ptr);
            c->anc_live.pop_front();
        }
        for (auto& rg : c->spare_rings) ws_spare_ring_release(rg, m);
    };
    auto gather_oldest = [&](bool* any) {
        const int64_t m = min_ep();
        std::vector<Plane> oldest;
        for (int32_t ci = 0; ci < (int32_t)c->cols.size(); ++ci)
            for (int32_t k = 0; k < c->cols[ci].width; ++k)
                if (c->cols[ci].stale[k] && c->cols[ci].ep[k] == m) oldest.push_back(Plane{ci, k});
        *any = !oldest.empty();
        if (!*any) return (int)WS_OK;
        c->trace_forced_planes += (int64_t)oldest.size();
        return materialize_planes(c, &oldest);
    };
    gc();
    const size_t n_ref = c->nranks > 1 ? (size_t)(c->n_global / c->nranks + 1) : (size_t)c->n;  // (shards differ by one particle)
    while (!c->anc_live.empty() && (c->anc_live.size() + 1) * sizeof(int32_t) * n_ref > c->genealogy_budget) {
        // over budget: bring the oldest planes up to date, which releases the oldest vectors
        bool any = false;
        TRY(gather_oldest(&any));
        if (!any) break;
        gc();
    }
    // sharded: keep a quarter of every rank's spare rows free for the offspring of this event (if more arrive the step
    // brings everything up to date and starts the rings afresh, resample_sharded)
    for (;;) {
        bool low = false;
        for (int q = 0; q < (int)c->spare_rings.size(); ++q)
            if (ws_spare_ring_peek(c->spare_rings[(size_t)q], spare_ring_cap(c, q), spare_ring_cap(c, q) / 4) < 0) low = true;
        if (!low) break;
        bool any = false;
        TRY(gather_oldest(&any));
        if (!any) break;
        gc();
    }
    return WS_OK;
}
static int commit_resample_event(ws_ctx* c) {
    if (!c->event_keeps) {
        c->anc_live.clear();
        c->anc_live.push_back({c->epoch + 1, c->d_anc});
        return WS_OK;
    }
    if (c->anc_live.empty() && c->anc_pool.empty() && c->d_anc != nullptr) c->anc_pool.push_back(c->d_anc);  // the vector made by ws_create
    int32_t* fresh = nullptr;
    if (!c->anc_pool.empty()) {
        fresh = c->anc_pool.back();
        c->anc_pool.pop_back();
    } else {
        // (sharded: a margin of `spare` entries on both sides, as for the vector made by ws_create_sharded)
        const int64_t margin = c->nranks > 1 ? c->spare : 0;
        TRY(pool_alloc(c, (void**)&fresh, sizeof(int32_t) * (size_t)(c->n + c->spare + margin)));
        fresh += margin;
    }
    c->anc_live.push_back({c->epoch + 1, fresh});
    c->d_anc = fresh;
    return WS_OK;
}
static int begin_resample_event(ws_ctx* c) {
    TRY(prepare_resample_event(c));
    return commit_resample_event(c);
}

// after the ancestors of the new event are in d_anc
static void end_resample_event(ws_ctx* c) {
    c->epoch++;
    for (auto& col : c->cols)
        for (auto& st : col.stale) st = 1;
    c->anc_pending = !c->cols.empty();
}

static int gather_all(ws_ctx* c, const int32_t* d_anc) {
    std::vector<Plane> which;
    for (int32_t ci = 0; ci < (int32_t)c->cols.size(); ++ci)
        for (int32_t k = 0; k < c->cols[ci].width; ++k) which.push_back(Plane{ci, k});
    return gather_planes(c, d_anc, which);
}

// Small particle sets: reduce-finalize (optional), CDF, search and expansion of a Resample step in one kernel.
static bool small_resample_ok(const ws_ctx* c, const double* d_ru) {
    return c->small_resample && c->nranks == 1 && c->n <= WS_SMALL_N && d_ru == nullptr && c->resampler != WS_RESAMPLER_MULTINOMIAL;
}
static int run_small_resample(ws_ctx* c, uint64_t stream_id, int gate, int do_finalize) {
    WsScanParams S;
    memset(&S, 0, sizeof(S));
    S.logw = c->logw;
    S.mode = 0;
    S.scheme = c->resampler;
    S.red = c->d_red;
    S.gate = gate;
    S.n = c->n;
    S.n_slots = c->n;
    S.last_rank = 1;
    S.seed = c->seed;
    S.stream = stream_id;
    S.ancestors = c->d_anc;
    S.cdf_local = c->d_cdf_local;
    S.n_clamped = c->d_counters + 0;
    ws_scan_set_scale(S);
    TimedEvent te;
    timed_begin(c, KC_SCAN, te);
    CK(c, ws_launch_resample_small(S, c->d_partials, c->n_partials, c->ess_perc_min, c->d_red, c->d_counters + 3, do_finalize, c->stream));
    timed_end(c, te);
    return WS_OK;
}

// Multinomial resampling with Philox draws: point S at the spacing tables (sized for S.n_slots) and fill them.
static int prepare_multinomial(ws_ctx* c, WsScanParams& S) {
    const int64_t n_all = S.n_slots + 1;
    const int64_t tiles = (n_all + WS_CDF_TILE - 1) / WS_CDF_TILE, blocks = (n_all + WS_SCAN_TILE - 1) / WS_SCAN_TILE;
    if (c->d_mn == nullptr || c->mn_cap_slots < n_all) {
        if (c->d_mn) {
            CK(c, cudaStreamSynchronize(c->stream));
            CK(c, cudaFree(c->d_mn));
            c->d_mn = nullptr;
        }
        CK(c, cudaMalloc(&c->d_mn, sizeof(unsigned long long) * (size_t)(tiles + blocks + 2)));
        c->mn_cap_slots = n_all;
    }
    S.mn_tile_off = c->d_mn;
    S.mn_block_local = c->d_mn + tiles;
    S.mn_total = c->d_mn + tiles + blocks;
    TimedEvent te;
    timed_begin(c, KC_SCAN, te);
    CK(c, ws_launch_spacings(S, c->stream));
    timed_end(c, te);
    c->stats.kernel_launches += 1;
    return WS_OK;
}

// Multinomial resampling with REPLAYED uniforms (parity tests): u = sort(N iid uniforms) (SURVEY Appendix B), sorted
// on the host — a test path; production draws need no sort (prepare_multinomial).
static int sorted_replay_uniforms(ws_ctx* c, const double* d_ru, int64_t n, const double** d_sorted) {
    std::vector<double> u((size_t)n);
    CK(c, cudaMemcpyAsync(u.data(), d_ru, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    std::sort(u.begin(), u.end());
    TRY(ensure_scratch(c, sizeof(double) * (size_t)n));
    CK(c, cudaMemcpyAsync(c->d_scratch, u.data(), sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    *d_sorted = c->d_scratch;
    return WS_OK;
}

static int run_scan_search(ws_ctx* c, const double* d_w, int mode, int scheme, int64_t n, const double* d_replay_u,
                           const double* d_sorted_u, int32_t* d_anc, unsigned long long* d_words,
                           unsigned long long* d_cdf_local, uint64_t stream_id, unsigned long long* d_clamped, int gate = 0) {
    const int64_t n_tiles = (n + WS_CDF_TILE - 1) / WS_CDF_TILE;
    if (c->d_heavy_F == nullptr || c->heavy_cap_n < n) {
        // at most n / WS_HEAVY_TILE_SLOTS families can own more than WS_HEAVY_TILE_SLOTS offspring each
        if (c->d_heavy_F) {
            CK(c, cudaStreamSynchronize(c->stream));
            CK(c, cudaFree(c->d_heavy_F));
            c->d_heavy_F = nullptr;
        }
        const size_t slots = (size_t)(n / WS_HEAVY_TILE_SLOTS) + 2;
        CK(c, cudaMalloc(&c->d_heavy_F, sizeof(int32_t) * slots * (WS_SCAN_TILE + 2)));
        c->heavy_cap_n = n;
    }
    (void)n_tiles;
    WsScanParams S;   // (the ticket / heavy-tile counters are zeroed by the launch itself)
    memset(&S, 0, sizeof(S));
    S.logw = d_w;
    S.mode = mode;
    S.scheme = scheme;
    S.red = c->d_red;
    S.gate = gate;
    S.n = n;
    S.n_slots = n;
    S.cdf_offset = 0ull;
    S.slot_base = 0;
    S.last_rank = 1;
    S.bounds = nullptr;
    S.total = nullptr;
    S.seed = c->seed;
    S.stream = stream_id;
    S.replay_u = d_replay_u;
    S.sorted_u = d_sorted_u;
    S.ancestors = d_anc;
    S.tile_words = d_words;
    S.cdf_local = d_cdf_local;
    S.tile_counter = c->d_tile_counter;
    S.n_clamped = d_clamped;
    S.heavy_count = c->d_tile_counter + 1;
    S.heavy_F = c->d_heavy_F;
    ws_scan_set_scale(S);
    if (scheme == WS_RESAMPLER_MULTINOMIAL && d_sorted_u == nullptr && d_replay_u == nullptr) TRY(prepare_multinomial(c, S));
    TimedEvent te;
    timed_begin(c, KC_SCAN, te);
    CK(c, ws_launch_scan_search(S, 0, c->stream));
    c->stats.kernel_launches += 3;  // cdf tiles, offsets, search, heavy expansion
    // (a gated step that does not fire: the search kernel itself leaves the identity in the ancestor vector)
    timed_end(c, te);
    return WS_OK;
}

// Exact GLOBAL stratified resampling of a sharded particle set (SURVEY.md §8e).
//   1. tile CDF of the shard with the global (m, S)  ->  this rank's fixed-point mass T_r
//   2. allgather T_r  ->  CDF offset O_r = sum_{q<r} T_q   (integers: identical on every rank)
//   3. first / end global slot produced by this rank (F at the shard's CDF edges), allgathered
//   4. search: ancestors (local indices) of the produced slots [fs_r, fe_r)
//   5. per plane: gather the offspring in slot order; the part that falls into rank d's slot range
//      [d N/R, (d+1) N/R) is sent to d (NCCL send/recv = all-to-all-v over NVLink); the part that stays
//      is gathered straight into the back buffer.  Slot order makes every (source, destination) piece
//      contiguous on both sides.
// ---- direct (peer-memory) exchange ---------------------------------------------------------------------------
// host bytes of every rank, in rank order (bytes % 8 == 0)
static int allgather_host_bytes(ws_ctx* c, const void* mine, size_t bytes, std::vector<char>& all) {
    const size_t R = (size_t)c->nranks, words = bytes / 8;
    TRY(ensure_scratch2(c, bytes * (R + 1)));
    char* d = (char*)c->d_scratch2;
    CK(c, cudaMemcpyAsync(d + bytes * R, mine, bytes, cudaMemcpyHostToDevice, c->stream));
    NCK(c, g_nccl.AllGather(d + bytes * R, d, words, WS_NCCL_UINT64, c->comm, c->stream));
    all.resize(bytes * R);
    CK(c, cudaMemcpyAsync(all.data(), d, bytes * R, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return WS_OK;
}

// ---- mailboxes (ws_mailbox.cuh) --------------------------------------------------------------------------------
// the descriptor of the next `n_exchanges` exchanges (one kernel): every rank calls this at the same points
static WsMailbox mbox_next(ws_ctx* c, int n_exchanges) {
    WsMailbox M;
    memset(&M, 0, sizeof(M));
    for (int q = 0; q < c->nranks; ++q) M.box[q] = c->mbox_peer[(size_t)q];
    M.rank = c->rank;
    M.nranks = c->nranks;
    M.seq = c->mbox_seq + 1u;
    M.cap = c->mbox_cap;
    M.err = c->d_mbox_err;
    M.timeout_ns = 60000000000ull;   // (a rank that is merely slow — a long host-side pause between two steps — must not fail the job)
    if (const char* e = getenv("WSB200_MAILBOX_TIMEOUT_MS")) M.timeout_ns = strtoull(e, nullptr, 10) * 1000000ull;
    c->mbox_seq += (uint32_t)n_exchanges;
    c->mbox_exchanges += n_exchanges;
    return M;
}
// after a host wait on the stream: did an exchange give up?
static int mbox_check(ws_ctx* c) {
    if (c->h_mbox_err != nullptr && *reinterpret_cast<volatile unsigned int*>(c->h_mbox_err) != 0u)
        return fail(c, WS_ENCCL, "mailbox exchange timed out: a rank died or the ranks left lock-step");
    return WS_OK;
}
static void mbox_release(ws_ctx* c) {
    for (size_t q = 0; q < c->mbox_peer.size(); ++q)
        if ((int)q != c->rank && c->mbox_peer[q]) cudaIpcCloseMemHandle(c->mbox_peer[q]);
    c->mbox_peer.clear();
    if (c->d_mbox) cudaFree(c->d_mbox);
    c->d_mbox = nullptr;
    c->mbox_on = false;
    cudaGetLastError();
}
// Allocate this rank's mailbox, map everybody else's (cudaIpc), and prove the path with one barrier exchange.  Any
// failure on any rank — ranks sharing a process, no IPC / peer access, a trial that times out — is agreed on over
// NCCL and leaves the whole job on the NCCL collectives (mbox_on = false everywhere).
static int mbox_setup(ws_ctx* c) {
    const int R = c->nranks, r = c->rank;
    if (const char* e = getenv("WSB200_MAILBOX"))
        if (strcmp(e, "0") == 0) return WS_OK;
    if (R > WS_MBOX_MAX_RANKS) return WS_OK;
    CK(c, cudaSetDevice(c->device));
    struct Msg {
        int64_t pid, ok;
        cudaIpcMemHandle_t h;
    };
    static_assert(sizeof(Msg) % 8 == 0, "Msg travels as 64-bit words");
    Msg mine;
    memset(&mine, 0, sizeof(mine));
    mine.pid = (int64_t)getpid();
    c->mbox_cap = 16384;
    const size_t bytes = sizeof(unsigned long long) * 2 * (size_t)R * (size_t)c->mbox_cap;
    bool ok = cudaMalloc(&c->d_mbox, bytes) == cudaSuccess && cudaMemset(c->d_mbox, 0, bytes) == cudaSuccess;
    if (ok && c->h_mbox_err == nullptr) {
        ok = cudaHostAlloc(&c->h_mbox_err, 64, cudaHostAllocMapped) == cudaSuccess;
        if (ok) {
            memset(c->h_mbox_err, 0, 64);
            ok = cudaHostGetDevicePointer((void**)&c->d_mbox_err, c->h_mbox_err, 0) == cudaSuccess;
        }
    }
    ok = ok && cudaIpcGetMemHandle(&mine.h, c->d_mbox) == cudaSuccess;
    ok = ok && cudaDeviceSynchronize() == cudaSuccess;   // the mailbox is zero before anybody can learn its handle
    cudaGetLastError();
    mine.ok = ok ? 1 : 0;
    std::vector<char> all;
    TRY(allgather_host_bytes(c, &mine, sizeof(mine), all));
    const Msg* msgs = reinterpret_cast<const Msg*>(all.data());
    bool usable = true;
    for (int q = 0; q < R; ++q) {
        if (!msgs[q].ok) usable = false;
        for (int q2 = q + 1; q2 < R; ++q2)
            if (msgs[q].pid == msgs[q2].pid) usable = false;   // IPC mappings need separate processes
    }
    if (!usable) {
        mbox_release(c);
        return WS_OK;
    }
    c->mbox_peer.assign((size_t)R, nullptr);
    c->mbox_peer[(size_t)r] = c->d_mbox;
    int64_t bad = 0;
    for (int q = 0; q < R; ++q) {
        if (q == r) continue;
        void* base = nullptr;
        if (cudaIpcOpenMemHandle(&base, msgs[q].h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
            cudaGetLastError();
            bad = 1;
            base = nullptr;
        }
        c->mbox_peer[(size_t)q] = (unsigned long long*)base;
    }
    std::vector<char> flags;
    TRY(allgather_host_bytes(c, &bad, sizeof(bad), flags));
    for (int q = 0; q < R; ++q)
        if (reinterpret_cast<const int64_t*>(flags.data())[q] != 0) usable = false;
    if (usable) {
        // trial: one barrier exchange with a short limit
        WsMailbox M = mbox_next(c, 1);
        M.timeout_ns = 10000000000ull;
        bad = (ws_launch_barrier_mbox(M, c->stream) != cudaSuccess || cudaStreamSynchronize(c->stream) != cudaSuccess || *c->h_mbox_err != 0u) ? 1 : 0;
        cudaGetLastError();
        TRY(allgather_host_bytes(c, &bad, sizeof(bad), flags));
        for (int q = 0; q < R; ++q)
            if (reinterpret_cast<const int64_t*>(flags.data())[q] != 0) usable = false;
    }
    if (!usable) {
        mbox_release(c);
        if (c->h_mbox_err) *c->h_mbox_err = 0u;
        return WS_OK;
    }
    c->mbox_on = true;
    return WS_OK;
}

// (slab index, byte offset) of a device pointer inside this rank's slabs; slab = -1 for nullptr
static int locate_in_slabs(ws_ctx* c, const void* ptr, int64_t* slab, int64_t* off) {
    *slab = -1;
    *off = 0;
    if (ptr == nullptr) return WS_OK;
    for (size_t k = 0; k < c->slabs.size(); ++k) {
        const char* b = c->slabs[k].base;
        if ((const char*)ptr >= b && (const char*)ptr < b + c->slabs[k].size) {
            *slab = (int64_t)k;
            *off = (int64_t)((const char*)ptr - b);
            return WS_OK;
        }
    }
    return fail(c, WS_ECUDA, "direct exchange: a plane buffer is not inside a slab");
}

#define WS_XMSG_HEAD 3  // words before the plane table: packed bounds, slab count, pid
static size_t xmsg_words(size_t n_planes) { return WS_XMSG_HEAD + 4 * n_planes; }

// host part of this rank's message (words 1 ..): slab count, pid, (slab, offset) of every plane's front and back buffer
static int fill_xmsg(ws_ctx* c, const std::vector<Plane>& planes, std::vector<int64_t>& w) {
    w.assign(xmsg_words(planes.size()), 0);
    w[1] = (int64_t)c->slabs.size();
    w[2] = (int64_t)getpid();
    for (size_t p = 0; p < planes.size(); ++p) {
        const Column& col = c->cols[planes[p].col];
        TRY(locate_in_slabs(c, col.front[planes[p].comp], &w[WS_XMSG_HEAD + 4 * p], &w[WS_XMSG_HEAD + 4 * p + 1]));
        TRY(locate_in_slabs(c, col.back[planes[p].comp], &w[WS_XMSG_HEAD + 4 * p + 2], &w[WS_XMSG_HEAD + 4 * p + 3]));
    }
    return WS_OK;
}

// From the all-gathered messages: map the slabs that are new since the last exchange (cudaIpcGetMemHandle /
// cudaIpcOpenMemHandle, rounds of up to 32 handles per rank, the same rounds on every rank) and resolve
// peer[q][p] = rank q's front (lazy) or back (eager) buffer of plane p as a pointer valid in THIS process.
// *usable = false (on every rank alike) when two ranks share a process: IPC mappings need separate processes.
static int resolve_peer_planes(ws_ctx* c, const std::vector<int64_t>& all, size_t words, size_t P, bool lazy,
                               std::vector<std::vector<double*>>& peer, bool* usable) {
    const int R = c->nranks, r = c->rank;
    auto row = [&](int q) { return all.data() + words * (size_t)q; };
    *usable = true;
    for (int q = 0; q < R; ++q)
        for (int q2 = q + 1; q2 < R; ++q2)
            if (row(q)[2] == row(q2)[2]) *usable = false;
    if (!*usable) return WS_OK;
    const int H = 32;
    struct Block {
        int64_t count;
        cudaIpcMemHandle_t h[H];
    };
    static_assert(sizeof(Block) % 8 == 0, "Block travels as 64-bit words");
    bool map_failed = false;
    int rounds = 0;
    for (;;) {
        bool need = false;
        for (int q = 0; q < R; ++q) {
            const size_t known = (q == r) ? c->slabs_published : c->peer_slabs[q].size();
            if ((size_t)row(q)[1] > known) need = true;
        }
        if (!need) break;
        Block b;
        memset(&b, 0, sizeof(b));
        const size_t target = (size_t)row(r)[1];  // the slab count announced in the message (nothing is allocated in between)
        while (c->slabs_published + (size_t)b.count < target && b.count < H) {
            if (cudaIpcGetMemHandle(&b.h[b.count], c->slabs[c->slabs_published + (size_t)b.count].base) != cudaSuccess) {
                cudaGetLastError();  // memory that cannot be exported: agreed on below
                map_failed = true;
                memset(&b.h[b.count], 0, sizeof(cudaIpcMemHandle_t));
            }
            b.count++;
        }
        c->slabs_published += (size_t)b.count;
        std::vector<char> hall;
        TRY(allgather_host_bytes(c, &b, sizeof(b), hall));
        for (int q = 0; q < R; ++q) {
            if (q == r) continue;
            const Block* pb = reinterpret_cast<const Block*>(hall.data() + sizeof(Block) * (size_t)q);
            for (int64_t k = 0; k < pb->count; ++k) {
                void* base = nullptr;
                cudaError_t e = cudaIpcOpenMemHandle(&base, pb->h[k], cudaIpcMemLazyEnablePeerAccess);
                if (e != cudaSuccess) {
                    cudaGetLastError();  // no peer access / IPC between these two processes: agreed on below
                    map_failed = true;
                    base = nullptr;
                }
                c->peer_slabs[q].push_back((char*)base);
            }
        }
        rounds++;
        c->trace_ipc_rounds++;
    }
    if (rounds > 0) {
        // a rank that could not map a peer's memory must not be written to blindly by the others either: everybody
        // learns of any failure and the whole job stays on ncclSend / ncclRecv (the caller clears push_exchange)
        const int64_t mine = map_failed ? 1 : 0;
        std::vector<char> flags;
        TRY(allgather_host_bytes(c, &mine, sizeof(mine), flags));
        for (int q = 0; q < R; ++q)
            if (reinterpret_cast<const int64_t*>(flags.data())[q] != 0) *usable = false;
        if (!*usable) return WS_OK;
    }
    peer.assign((size_t)R, std::vector<double*>(P, nullptr));
    for (int q = 0; q < R; ++q) {
        if (q == r) continue;
        for (size_t p = 0; p < P; ++p) {
            const int64_t slab = row(q)[WS_XMSG_HEAD + 4 * p + (lazy ? 0 : 2)], off = row(q)[WS_XMSG_HEAD + 4 * p + (lazy ? 1 : 3)];
            if (slab < 0 || (size_t)slab >= c->peer_slabs[q].size()) return fail(c, WS_ECUDA, "direct exchange: unknown peer buffer");
            peer[q][p] = reinterpret_cast<double*>(c->peer_slabs[q][(size_t)slab] + off);
        }
    }
    return WS_OK;
}

// `fired` != nullptr: the decision of this step has not been read yet (ensure_reduced(.., wait = false)): the kernels in
// front of the one host wait this function needs anyway (for the slot bounds) run gated on the device flag, the wait
// delivers the decision together with the bounds, and a step that does not fire returns there (*fired = 0).
static int resample_sharded(ws_ctx* c, const double* d_ru, uint64_t stream_id, int* fired = nullptr) {
    const int R = c->nranks, r = c->rank;
    auto t_now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double t0 = t_now();
    c->phase_n++;
    WsScanParams S;
    memset(&S, 0, sizeof(S));
    S.logw = c->logw;
    S.mode = 0;
    S.scheme = c->resampler;
    S.red = c->d_red;
    S.gate = fired != nullptr ? 1 : 0;
    S.n = c->n;
    S.n_slots = c->n_global;
    S.seed = c->seed;
    S.stream = stream_id;
    S.replay_u = d_ru;
    ws_scan_set_scale(S);
    if (c->resampler == WS_RESAMPLER_MULTINOMIAL) TRY(prepare_multinomial(c, S));   // every rank: the same table of all global slots
    S.ancestors = nullptr;
    S.tile_words = c->d_tile_words;
    S.cdf_local = c->d_cdf_local;
    S.tile_counter = c->d_tile_counter;
    S.n_clamped = c->d_counters + 0;
    S.heavy_count = c->d_tile_counter + 1;
    S.last_rank = (r == R - 1) ? 1 : 0;
    S.total = c->d_all_tot + R;           // own total staged behind the allgather buffer
    // this rank's message of the step (bounds + plane addresses, see d_xmsg), staged behind the allgather buffer
    std::vector<Plane> planes;
    for (int32_t ci = 0; ci < (int32_t)c->cols.size(); ++ci)
        for (int32_t k = 0; k < c->cols[ci].width; ++k) planes.push_back(Plane{ci, k});
    const size_t xw = xmsg_words(planes.size());
    if (xw > c->xmsg_words) {
        if (c->d_xmsg) {
            CK(c, cudaStreamSynchronize(c->stream));
            CK(c, cudaFree(c->d_xmsg));
            c->d_xmsg = nullptr;
        }
        c->xmsg_words = xw + 64;
        CK(c, cudaMalloc(&c->d_xmsg, sizeof(int64_t) * c->xmsg_words * (size_t)(R + 1)));
    }
    int64_t* const d_xmine = c->d_xmsg + xw * (size_t)R;
    S.bounds = reinterpret_cast<int32_t*>(d_xmine);   // word 0: (first, end) produced slot, written by ws_bounds_kernel
    std::vector<int64_t> xmine;
    {
        const double tf = t_now();
        TRY(fill_xmsg(c, planes, xmine));
        c->phase_ms[6] += t_now() - tf;
    }
    CK(c, cudaMemcpyAsync(d_xmine + 1, xmine.data() + 1, sizeof(int64_t) * (xw - 1), cudaMemcpyHostToDevice, c->stream));
    TimedEvent te;
    const bool mbox = c->mbox_on && 2 * xw <= (size_t)c->mbox_cap;   // (the same on every rank: same planes, same capacity)
    if (mbox) {
        // tile CDF, then ONE kernel: group offsets + mass -> masses of all ranks -> my slot bounds -> everybody's message
        timed_begin(c, KC_SCAN, te);
        CK(c, ws_launch_cdf_tiles(S, c->stream));
        S.all_tot = c->d_all_tot;
        S.rank = r;
        const WsMailbox M = mbox_next(c, 2);
        CK(c, ws_launch_offsets_bounds_mbox(S, M, c->d_all_tot, reinterpret_cast<const unsigned long long*>(d_xmine), (int)xw,
                                            reinterpret_cast<unsigned long long*>(c->d_xmsg), c->stream));
        timed_end(c, te);
    } else {
        timed_begin(c, KC_SCAN, te);
        CK(c, ws_launch_cdf(S, c->stream));
        timed_end(c, te);
        NCK(c, g_nccl.AllGather(c->d_all_tot + R, c->d_all_tot, 1, WS_NCCL_UINT64, c->comm, c->stream));
        // the CDF offset of this rank (sum of the lower ranks' masses) is formed on the device from the
        // allgathered masses, so the host does not have to wait for them
        S.all_tot = c->d_all_tot;
        S.rank = r;
        CK(c, ws_launch_bounds(S, c->stream));
        NCK(c, g_nccl.AllGather(d_xmine, c->d_xmsg, xw, WS_NCCL_UINT64, c->comm, c->stream));
    }
    std::vector<int64_t> xall(xw * (size_t)R);
    CK(c, cudaMemcpyAsync(xall.data(), c->d_xmsg, sizeof(int64_t) * xw * (size_t)R, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    TRY(mbox_check(c));
    c->stats.d2h_bytes += (int64_t)(sizeof(int64_t) * xw * (size_t)R);
    if (fired != nullptr) {
        c->red_valid = true;              // *h_red arrived with the same wait
        *fired = c->h_red->do_resample ? 1 : 0;
        if (!*fired) return WS_OK;        // (the gated kernels did nothing; every rank reads the same decision)
        TRY(commit_resample_event(c));    // the rest of begin_resample_event
        S.gate = 0;
    }
    std::vector<int32_t> bnd(2 * R);
    for (int q = 0; q < R; ++q) memcpy(&bnd[2 * q], &xall[xw * (size_t)q], 2 * sizeof(int32_t));
    c->phase_ms[0] += t_now() - t0;
    t0 = t_now();
    const int64_t fs = bnd[2 * r], fe = bnd[2 * r + 1];
    const int64_t produced = fe - fs;
    if (produced > c->anc_src_cap) {
        if (c->d_anc_src) CK(c, cudaFree(c->d_anc_src));
        c->d_anc_src = nullptr;
        c->anc_src_cap = produced + produced / 4 + c->spare + 1024;
        CK(c, cudaMalloc(&c->d_anc_src, sizeof(int32_t) * (size_t)c->anc_src_cap));
    }
    // heavy-tile tables are sized for the slots this rank can produce (at most n_global)
    if (c->d_heavy_F == nullptr || c->heavy_cap_n < c->n_global) {
        if (c->d_heavy_F) CK(c, cudaFree(c->d_heavy_F));
        const size_t slots = (size_t)(c->n_global / WS_HEAVY_TILE_SLOTS) + 2;
        CK(c, cudaMalloc(&c->d_heavy_F, sizeof(int32_t) * slots * (WS_SCAN_TILE + 2)));
        c->heavy_cap_n = c->n_global;
    }
    S.heavy_F = c->d_heavy_F;
    CK(c, cudaMemsetAsync(c->d_tile_counter, 0, sizeof(unsigned int) * 2, c->stream));
    // Deferred gather + few migrants (the usual case): the search writes the ancestors of global slot s straight to
    // d_anc[s - my_lo] — own slots in place, the slots produced for the neighbours into the margins on either side —
    // instead of a staging vector that a second pass copies into place (8 B per particle saved).
    // (ws_exchange.h: every rank derives the whole plan from the all-gathered bounds)
    auto rank_lo = [&](int d) { return ws_rank_lo(c->n_global, R, d); };
    const WsExchangePlan plan = ws_exchange_plan(bnd.data(), R, r, c->n_global);
    const bool fits_all = plan.fits;
    const int64_t lo_r = (c->n_global * (int64_t)r) / R, hi_r = (c->n_global * (int64_t)(r + 1)) / R;
    const bool inplace = c->lazy_gather && fits_all && (lo_r - fs) <= c->spare && (fe - hi_r) <= c->spare;
    int32_t* const anc_src = inplace ? c->d_anc + (fs - lo_r) : c->d_anc_src;
    S.ancestors = anc_src;
    S.slot_base = (int32_t)fs;
    timed_begin(c, KC_SCAN, te);
    CK(c, ws_launch_search(S, c->stream));
    timed_end(c, te);
    c->stats.kernel_launches += 4;

    c->phase_ms[2] += t_now() - t0;
    t0 = t_now();
    // ---- exchange plan (slot ranges) ------------------------------------------------------------
    const std::vector<int64_t>&send_off = plan.send_off, &send_cnt = plan.send_cnt, &recv_off = plan.recv_off, &recv_cnt = plan.recv_cnt;
    const int64_t remote_send = plan.remote_send, remote_recv = plan.remote_recv;
    c->migrated_total += remote_recv;
    // Spare rows of this event on every rank (ws_exchange.h: rings kept alike on all ranks), and whether planes that
    // are behind can follow the exchange through the genealogy.  Every rank takes the same branches: the plan, the
    // rings and the bookkeeping of the planes are the same everywhere.
    std::vector<int64_t> incoming((size_t)R, 0), starts((size_t)R, 0);
    for (int d = 0; d < R; ++d)
        incoming[(size_t)d] = (rank_lo(d + 1) - rank_lo(d)) - ws_piece(bnd.data(), c->n_global, R, d, d);
    auto ring_try = [&]() {
        bool ok = true;
        for (int q = 0; q < R; ++q) {
            starts[(size_t)q] = ws_spare_ring_peek(c->spare_rings[(size_t)q], spare_ring_cap(c, q), incoming[(size_t)q]);
            if (starts[(size_t)q] < 0) {
                ok = false;
                starts[(size_t)q] = 0;
            }
        }
        return ok;
    };
    bool any_stale = false;
    for (auto& pl : planes)
        if (c->cols[pl.col].stale[pl.comp]) any_stale = true;
    const bool push_wanted = c->push_exchange && plan.total_remote > 0 && plan.total_remote >= c->push_min && !planes.empty();
    bool ring_ok = ring_try();
    bool readdress = false;
    if (any_stale && (!ring_ok || (!push_wanted && plan.total_remote > 0))) {
        // more offspring than the rings hold, or an exchange that cannot trace stale planes: bring every plane up to
        // date (the eager and the staged paths below assume that) and start the rings afresh
        TRY(materialize_planes(c));
        c->trace_full_gathers++;
        for (auto& rg : c->spare_rings) rg.clear();
        ring_ok = ring_try();
        any_stale = false;
        readdress = push_wanted;   // front / back buffers were swapped: the peers need the new addresses
    }
    if (readdress) {
        TRY(fill_xmsg(c, planes, xmine));
        CK(c, cudaMemcpyAsync(d_xmine + 1, xmine.data() + 1, sizeof(int64_t) * (xw - 1), cudaMemcpyHostToDevice, c->stream));
        NCK(c, g_nccl.AllGather(d_xmine, c->d_xmsg, xw, WS_NCCL_UINT64, c->comm, c->stream));
        CK(c, cudaMemcpyAsync(xall.data(), c->d_xmsg, sizeof(int64_t) * xw * (size_t)R, cudaMemcpyDeviceToHost, c->stream));
        CK(c, cudaStreamSynchronize(c->stream));
    }
    const bool fits = plan.fits && ring_ok;
    const bool lazy = c->lazy_gather && fits;
    if (lazy) {
        for (int q = 0; q < R; ++q)
            c->spare_rings[(size_t)q].push_back(WsSpareRegion{c->epoch + 1, starts[(size_t)q], incoming[(size_t)q]});
    } else {
        for (auto& rg : c->spare_rings) rg.clear();   // eager: every plane ends up in the new order, nothing stays in spare rows
        std::fill(starts.begin(), starts.end(), 0);
    }

    const int BATCH = 8;
    // Direct exchange: the gather kernel that would stage a
    // destination's offspring writes them straight into that rank's planes over NVLink — into the spare rows behind
    // its front planes (lazy) or at their final slots of its back planes (eager) — so gather and transfer are ONE
    // kernel per destination and nothing is staged or received.  Safe without a barrier in front: every rank has
    // passed the allgather of the bounds, i.e. finished all earlier kernels that touch its planes, and what it
    // runs meanwhile (search, its own gathers) reads front rows [0, n) and writes its OWN slots only.  A
    // stream-ordered all-reduce of one word afterwards is the barrier that tells a rank its incoming rows are complete.
    bool push = push_wanted;
    std::vector<std::vector<double*>> peer;
    if (push) {
        bool usable = false;
        const double tr0 = t_now();
        TRY(resolve_peer_planes(c, xall, xw, planes.size(), lazy, peer, &usable));
        c->phase_ms[1] += t_now() - tr0;
        if (!usable) {
            push = false;
            c->push_exchange = false;  // ranks share a process, or no IPC / peer access: stay on ncclSend / ncclRecv (every rank decides alike)
            if (any_stale) {           // the staged path reads the planes in the current order
                TRY(materialize_planes(c));
                any_stale = false;
            }
        }
    }
    // the migrating offspring are the produced slots outside my own range: a prefix [0, pre) (to lower
    // ranks) and a suffix [suf0, produced) (to higher ranks) of the produced range
    const int64_t pre = send_off[r] > 0 || send_cnt[r] > 0 ? send_off[r] : produced;
    const int64_t suf0 = send_cnt[r] > 0 ? send_off[r] + send_cnt[r] : produced;
    const int64_t n_pre = std::min(pre, produced), n_suf = produced - suf0;
    if (!push && remote_send * BATCH > c->send_cap) {
        // grow geometrically (a cudaFree / cudaMalloc pair synchronises the device and costs milliseconds)
        if (c->d_send) CK(c, cudaFree(c->d_send));
        c->d_send = nullptr;
        c->send_cap = std::max<int64_t>(2 * remote_send * BATCH, 2 * c->spare * BATCH);
        CK(c, cudaMalloc(&c->d_send, sizeof(double) * (size_t)c->send_cap));
    }
    // position of destination d's piece inside one staged plane (prefix pieces first, then suffix pieces)
    auto stage_pos = [&](int d) { return d < r ? send_off[d] : n_pre + (send_off[d] - suf0); };
    // where rank q's offspring land on my side: lazily in the spare rows behind the FRONT planes
    // (lower ranks first), eagerly at their final slots in the BACK planes
    const std::vector<int64_t>& spare_pos = plan.spare_pos;
    const double tt0 = t_now();
    if (push && any_stale) {
        // Planes that are behind (sharded genealogy; lazy by construction): the offspring produced for rank d are traced
        // through the retained ancestor vectors, once per offspring, and ONE kernel writes every plane — from the row
        // it has the offspring's value at — into d's spare rows.
        int64_t n_levels = 0;
        for (auto& pl : planes)
            if (c->cols[pl.col].stale[pl.comp]) n_levels = std::max(n_levels, c->epoch - c->cols[pl.col].ep[pl.comp]);
        std::vector<const int32_t*> chain((size_t)n_levels, nullptr);
        for (int64_t t = 0; t < n_levels; ++t) {
            const int64_t ev = c->epoch - t;
            bool found = false;
            for (auto& v : c->anc_live)
                if (v.event == ev) {
                    found = true;
                    chain[(size_t)t] = v.identity ? nullptr : v.ptr;
                }
            if (!found) return fail(c, WS_EINVAL, "genealogy: ancestors of event %lld were released", (long long)ev);
        }
        int64_t m_max = 0;
        for (int d = 0; d < R; ++d)
            if (d != r) m_max = std::max(m_max, send_cnt[d]);
        const size_t chain_b = ((size_t)n_levels * sizeof(void*) + 255) & ~(size_t)255;
        const size_t table_b = (planes.size() * sizeof(WsTracedPlane) + 255) & ~(size_t)255;
        const size_t rows_b = (size_t)(n_levels + 1) * (size_t)m_max * sizeof(int32_t);
        if (chain_b + table_b + rows_b > c->gen_bytes) {
            CK(c, cudaStreamSynchronize(c->stream));
            if (c->d_gen) CK(c, cudaFree(c->d_gen));
            c->d_gen = nullptr;
            c->gen_bytes = 2 * (chain_b + table_b + rows_b);
            CK(c, cudaMalloc(&c->d_gen, c->gen_bytes));
        }
        const int32_t** d_chain = reinterpret_cast<const int32_t**>(c->d_gen);
        WsTracedPlane* d_table = reinterpret_cast<WsTracedPlane*>((char*)c->d_gen + chain_b);
        int32_t* d_rows = reinterpret_cast<int32_t*>((char*)c->d_gen + chain_b + table_b);
        if (n_levels > 0) CK(c, cudaMemcpyAsync(d_chain, chain.data(), (size_t)n_levels * sizeof(void*), cudaMemcpyHostToDevice, c->stream));
        std::vector<WsTracedPlane> table(planes.size());
        for (int d = 0; d < R; ++d) {
            if (d == r || send_cnt[d] <= 0) continue;
            const int64_t at = ws_push_offset(bnd.data(), R, r, d, c->n_global, true) + starts[(size_t)d];
            for (size_t p = 0; p < planes.size(); ++p) {
                const Column& col = c->cols[planes[p].col];
                table[p].src = col.front[planes[p].comp];
                table[p].dst = peer[d][p] + at;
                table[p].level = col.stale[planes[p].comp] ? c->epoch - col.ep[planes[p].comp] : 0;
            }
            CK(c, cudaMemcpyAsync(d_table, table.data(), table.size() * sizeof(WsTracedPlane), cudaMemcpyHostToDevice, c->stream));
            timed_begin(c, KC_GATHER, te);
            CK(c, ws_launch_trace_rows(anc_src + send_off[d], send_cnt[d], d_chain, (int)n_levels, c->n, d_rows, c->stream));
            CK(c, ws_launch_push_traced(d_table, (int)planes.size(), send_cnt[d], d_rows, c->stream));
            timed_end(c, te);
            c->stats.kernel_launches += 2;
            c->traced_rows += send_cnt[d] * (int64_t)planes.size();
        }
        c->phase_ms[4] += t_now() - tt0;
    }
    for (size_t p0 = 0; p0 < planes.size() && !(push && any_stale); p0 += BATCH) {
        const int nb = (int)std::min<size_t>(BATCH, planes.size() - p0);
        if (!lazy && send_cnt[r] > 0) {
            // offspring that stay: gather straight into the back buffers
            WsGatherParams G;
            memset(&G, 0, sizeof(G));
            G.n = send_cnt[r];
            G.ancestors = anc_src + send_off[r];
            G.n_planes = nb;
            for (int k = 0; k < nb; ++k) {
                const Plane pl = planes[p0 + k];
                G.src[k] = c->cols[pl.col].front[pl.comp];
                G.dst[k] = c->cols[pl.col].back[pl.comp] + recv_off[r];
            }
            timed_begin(c, KC_GATHER, te);
            CK(c, ws_launch_gather(G, grid_for(c, G.n, 256, 8), c->stream));
            timed_end(c, te);
        }
        if (push) {
            for (int d = 0; d < R; ++d) {
                if (d == r || send_cnt[d] <= 0) continue;
                WsGatherParams G;
                memset(&G, 0, sizeof(G));
                G.n = send_cnt[d];
                G.ancestors = anc_src + send_off[d];
                G.n_planes = nb;
                const int64_t at = ws_push_offset(bnd.data(), R, r, d, c->n_global, lazy) + starts[(size_t)d];
                for (int k = 0; k < nb; ++k) {
                    const Plane pl = planes[p0 + k];
                    G.src[k] = c->cols[pl.col].front[pl.comp];
                    G.dst[k] = peer[d][p0 + k] + at;
                }
                timed_begin(c, KC_GATHER, te);
                CK(c, ws_launch_gather(G, grid_for(c, G.n, 256, 8), c->stream));
                timed_end(c, te);
            }
            continue;
        }
        // stage the migrating offspring of this batch (slot order)
        const int64_t seg_start[2] = {0, suf0}, seg_len[2] = {n_pre, n_suf}, seg_dst[2] = {0, n_pre};
        for (int sgi = 0; sgi < 2; ++sgi) {
            if (seg_len[sgi] <= 0 || remote_send == 0) continue;
            WsGatherParams G;
            memset(&G, 0, sizeof(G));
            G.n = seg_len[sgi];
            G.ancestors = anc_src + seg_start[sgi];
            G.n_planes = nb;
            for (int k = 0; k < nb; ++k) {
                const Plane pl = planes[p0 + k];
                G.src[k] = c->cols[pl.col].front[pl.comp];
                G.dst[k] = c->d_send + (size_t)k * remote_send + seg_dst[sgi];
            }
            timed_begin(c, KC_GATHER, te);
            CK(c, ws_launch_gather(G, grid_for(c, G.n, 256, 8), c->stream));
            timed_end(c, te);
        }
        NCK(c, g_nccl.GroupStart());
        for (int k = 0; k < nb; ++k) {
            const Plane pl = planes[p0 + k];
            for (int d = 0; d < R; ++d) {
                if (d == r) continue;
                if (send_cnt[d] > 0)
                    NCK(c, g_nccl.Send(c->d_send + (size_t)k * remote_send + stage_pos(d), (size_t)send_cnt[d], WS_NCCL_FLOAT64, d, c->comm, c->stream));
                if (recv_cnt[d] > 0) {
                    double* dst = lazy ? c->cols[pl.col].front[pl.comp] + c->n + starts[(size_t)r] + spare_pos[d]
                                       : c->cols[pl.col].back[pl.comp] + recv_off[d];
                    NCK(c, g_nccl.Recv(dst, (size_t)recv_cnt[d], WS_NCCL_FLOAT64, d, c->comm, c->stream));
                }
            }
        }
        NCK(c, g_nccl.GroupEnd());
    }
    if (push) {
        if (c->mbox_on) CK(c, ws_launch_barrier_mbox(mbox_next(c, 1), c->stream));
        else NCK(c, g_nccl.AllReduce(c->d_barrier, c->d_barrier, 1, WS_NCCL_UINT64, WS_NCCL_SUM, c->comm, c->stream));
        c->pushed_total += remote_send;
    }
    if (c->phase_n > 6) c->phase_ms[5] += t_now() - t0;  // exchange without the communicator's first-use set-up
    c->phase_ms[3] += t_now() - t0;
    t0 = t_now();
    if (lazy) {
        // ancestors of my slots: local offspring point at their parent, received offspring at the spare
        // row they were written to; every plane is now in pre-resample order (+ spare rows) and is
        // gathered by its next reader, exactly as on one GPU
        const int64_t self_lo = recv_off[r], self_hi = recv_off[r] + send_cnt[r];
        if (inplace) {
            // own slots are already in place: only the slots received from other ranks get their spare-row index
            CK(c, ws_launch_patch_ancestors(c->d_anc, c->n, send_cnt[r] > 0 ? self_lo : c->n, send_cnt[r] > 0 ? self_hi : c->n,
                                             starts[(size_t)r], c->stream));
        } else {
            CK(c, ws_launch_local_ancestors(c->d_anc, c->n, anc_src + send_off[r], send_cnt[r] > 0 ? self_lo : c->n,
                                             send_cnt[r] > 0 ? self_hi : c->n, starts[(size_t)r], grid_for(c, c->n, 256, 8), c->stream));
        }
        c->stats.kernel_launches++;
        end_resample_event(c);
        return WS_OK;
    }
    for (auto& col : c->cols) std::swap(col.front, col.back);
    c->epoch++;
    for (auto& col : c->cols)
        for (auto& e : col.ep) e = c->epoch;
    return WS_OK;
}

static int spec_checkpoint(ws_ctx* c);

extern "C" int ws_resample(ws_ctx* c, ws_resample_info* info) {
    if (!c) return WS_EINVAL;
    if (c->spec_block && !c->spec_flushing) return info ? fail(c, WS_EUNSUPPORTED, "ws_resample with an outcome inside a speculative block") : spec_checkpoint(c);
    if (info) {
        TRY(resolve_spec(c));  // the caller wants the outcome, including the current value of `resampled`
        info->fired = 0;
        info->resampled = c->resampled ? 1 : 0;
        info->ess_perc = NAN;
        info->log_mean_w = NAN;
        info->n_clamped = -1;  // cumulative count is reported by ws_get_clamped (needs a sync)
    }
    if (!c->weights_changed) {  // `resampled` keeps its previous value (transformers.jl:475-477)
        c->last_info = ws_resample_info{0, -1, NAN, NAN, -1};  // resampled: filled in by ws_last_resample
        c->last_info_pending = false;
        return WS_OK;
    }
    if (c->resampler == WS_RESAMPLER_MULTINOMIAL && c->nranks > 1 && c->d_replay_u != nullptr)
        return fail(c, WS_EUNSUPPORTED, "multinomial resampling of a sharded state with replayed uniforms (Philox draws are supported)");
    if (c->nranks > 1 && c->d_replay_u == nullptr && c->merged_decision_wait) {
        // Sharded step: the decision travels with the slot bounds (one host wait per step instead of two).
        TRY(ensure_reduced(c, true, /*wait=*/false));
        c->stats.resamples_fired++;
        const uint64_t step_stream = c->next_stream++;
        int fired = 0;
        if (c->red_valid) {   // (nothing was weighted on the device since the last reduction: *h_red is current)
            fired = c->h_red->do_resample ? 1 : 0;
            if (fired) {
                TRY(begin_resample_event(c));
                TRY(resample_sharded(c, nullptr, step_stream));
            }
        } else {
            const auto tp0 = std::chrono::steady_clock::now();
            TRY(prepare_resample_event(c));   // the half of begin_resample_event that moves planes (harmless if the step does not fire)
            c->phase_ms[7] += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tp0).count();
            TRY(resample_sharded(c, nullptr, step_stream, &fired));
        }
        const WsReduceOut r = *c->h_red;
        if (fired) {
            c->logw_uniform = true;
            c->logw_base = r.log_mean_w;
            c->partials_valid = false;
            c->red_valid = false;
            c->resampled = true;
            c->stats.resamples_done++;
        } else {
            c->resampled = false;
        }
        c->weights_changed = false;
        c->last_info = ws_resample_info{1, fired, r.ess_perc, r.log_mean_w, -1};
        c->last_info_pending = false;
        if (info) *info = c->last_info;
        return WS_OK;
    }
    TRY(ensure_reduced(c, true));
    c->stats.resamples_fired++;
    const WsReduceOut r = *c->h_red;
    // the Philox stream of this step's slot uniforms is taken whether or not the step fires, so that the streams of
    // everything that follows do not depend on how (or when) the decision is learnt
    const uint64_t step_stream = c->next_stream++;
    if (r.do_resample) {
        // slot uniforms: one per slot (stratified) or one in total (systematic), in replay order
        const double* d_ru = nullptr;
        if (c->d_replay_u != nullptr) {
            const int64_t need = (c->resampler == WS_RESAMPLER_SYSTEMATIC) ? 1 : c->n_global;
            if (c->cur_u + need > c->replay_u_len)
                return fail(c, WS_EREPLAY, "replay uniforms exhausted in Resample (%lld needed, %lld installed)",
                            (long long)(c->cur_u + need), (long long)c->replay_u_len);
            d_ru = c->d_replay_u + c->cur_u;
            c->cur_u += need;
        }
        if (c->nranks > 1) {
            TRY(begin_resample_event(c));
            TRY(resample_sharded(c, d_ru, step_stream));
            c->logw_uniform = true;
            c->logw_base = r.log_mean_w;
            c->partials_valid = false;
            c->red_valid = false;
            c->resampled = true;
            c->stats.resamples_done++;
            c->weights_changed = false;
            c->last_info = ws_resample_info{1, 1, r.ess_perc, r.log_mean_w, -1};
            c->last_info_pending = false;
            if (info) *info = c->last_info;
            return WS_OK;
        }
        const uint64_t stream_id = step_stream;
        // planes still in an older order keep their ancestor vectors (genealogy) or are gathered now
        TRY(begin_resample_event(c));
        const double* d_sorted = nullptr;
        if (c->resampler == WS_RESAMPLER_MULTINOMIAL && d_ru != nullptr) {
            TRY(sorted_replay_uniforms(c, d_ru, c->n, &d_sorted));   // replayed draws (tests): sorted on the host
            d_ru = nullptr;
        }
        if (small_resample_ok(c, d_ru) && d_sorted == nullptr) {
            TRY(run_small_resample(c, stream_id, 0, 0));
        } else {
            TRY(run_scan_search(c, c->logw, 0, c->resampler, c->n, d_ru, d_sorted, c->d_anc, c->d_tile_words, c->d_cdf_local, stream_id, c->d_counters + 0));
        }
        // resample!(store, indices) is deferred: each plane is gathered when it is next read
        end_resample_event(c);
        if (!c->lazy_gather) TRY(materialize_planes(c));
        // fill!(state.weights, mean_logW): kept symbolic until somebody reads the array
        c->logw_uniform = true;
        c->logw_base = r.log_mean_w;
        c->partials_valid = false;
        c->red_valid = false;
        c->resampled = true;
        c->stats.resamples_done++;
    } else {
        c->resampled = false;
    }
    c->weights_changed = false;
    c->last_info = ws_resample_info{1, c->resampled ? 1 : 0, r.ess_perc, r.log_mean_w, -1};
    c->last_info_pending = false;
    if (info) *info = c->last_info;
    return WS_OK;
}

// Resample.apply! without waiting for its outcome.  The reference's state machine (transformers.jl:474-498) needs
// ESS% < ess_perc_min on the host only to decide what to launch; here everything that depends on the decision runs
// on the device behind the decision flag, so the host issues the step and goes on:
//   * (m, S, Q) partials -> ws_finalize_kernel -> d_red (+ a stream-ordered copy into the pinned ring);
//   * CDF + ancestor search gated on d_red->do_resample; if the step does not fire the same kernel writes the
//     identity into the ancestor vector;
//   * the host books the event as fired (new ancestor vector, every plane one event behind): the deferred gather
//     of the next pass reads through the ancestors either way, and that pass takes its old log-weights from
//     d_red->log_mean_w or from the array according to the same flag (logw_mode 3).
// `state.resampled`, the counters and anything that reads the log-weights resolve the pending records first
// (resolve_spec), which is the only place the host waits.  Not taken (falls back to ws_resample): replayed
// uniforms (the cursor advances only on a firing step), sharded states, multinomial, eager gather.
extern "C" int ws_resample_async(ws_ctx* c) {
    if (!c) return WS_EINVAL;
    if (c->spec_block && !c->spec_flushing) return spec_checkpoint(c);
    if (!c->weights_changed) {
        c->last_info = ws_resample_info{0, -1, NAN, NAN, -1};
        c->last_info_pending = false;
        return WS_OK;
    }
    if (!c->async_resample || c->d_replay_u != nullptr || c->nranks > 1 || c->resampler == WS_RESAMPLER_MULTINOMIAL ||
        !c->lazy_gather || c->cols.empty() || c->spec_immediate >= 2)
        return ws_resample(c, nullptr);
    TRY(flush_window(c));
    if (c->red_valid || c->logw_uniform || c->logw_spec) return ws_resample(c, nullptr);  // nothing new was weighted on the device
    CK(c, cudaSetDevice(c->device));
    if (c->spec_pending >= ws_ctx::SPEC_RING - 1) TRY(resolve_spec(c));
    if (!c->partials_valid) {
        const int grid = std::min(grid_for(c, c->n, 256, 8), WS_MAX_PARTIALS);
        TimedEvent te;
        timed_begin(c, KC_REDUCE, te);
        CK(c, ws_launch_reduce_logw(c->logw, c->n, c->d_partials, grid, c->stream));
        timed_end(c, te);
        c->n_partials = grid;
        c->partials_valid = true;
    }
    const uint64_t stream_id = c->next_stream++;
    if (small_resample_ok(c, nullptr)) {
        // one kernel: finalize + decision + CDF + search + expansion (or the identity); then the record for the host
        TRY(begin_resample_event(c));
        TRY(run_small_resample(c, stream_id, /*gate=*/1, /*do_finalize=*/1));
        CK(c, cudaMemcpyAsync(&c->h_ring[c->spec_head % ws_ctx::SPEC_RING], c->d_red, sizeof(WsReduceOut), cudaMemcpyDeviceToHost, c->stream));
        c->ring_event[c->spec_head % ws_ctx::SPEC_RING] = c->epoch + 1;
        end_resample_event(c);
    } else {
        TimedEvent te;
        timed_begin(c, KC_FINALIZE, te);
        CK(c, ws_launch_finalize(c->d_partials, c->n_partials, c->n_global, c->ess_perc_min, c->d_red, c->stream, c->d_counters + 3));
        timed_end(c, te);
        CK(c, cudaMemcpyAsync(&c->h_ring[c->spec_head % ws_ctx::SPEC_RING], c->d_red, sizeof(WsReduceOut), cudaMemcpyDeviceToHost, c->stream));
        c->ring_event[c->spec_head % ws_ctx::SPEC_RING] = c->epoch + 1;
        TRY(begin_resample_event(c));
        TRY(run_scan_search(c, c->logw, 0, c->resampler, c->n, nullptr, nullptr, c->d_anc, c->d_tile_words, c->d_cdf_local, stream_id,
                            c->d_counters + 0, /*gate=*/1));
        end_resample_event(c);
    }
    c->spec_head++;
    c->spec_pending++;
    c->stats.resamples_fired++;
    c->logw_uniform = false;
    c->logw_spec = true;
    c->partials_valid = false;
    c->red_valid = false;
    c->weights_changed = false;
    c->last_info_pending = true;
    return WS_OK;
}

// A statement list with parameters (Loop bodies): substitute, then issue each statement through its own entry point.
extern "C" int ws_exec(ws_ctx* c, const ws_cmd* cmds, int32_t n_cmds, const double* params, int32_t n_params) {
    if (!c || (!cmds && n_cmds > 0) || n_cmds < 0) return WS_EINVAL;
    std::vector<ws_tok> toks;
    std::vector<ws_expr> ex;
    for (int32_t k = 0; k < n_cmds; ++k) {
        const ws_cmd& cm = cmds[k];
        // copy the command's expressions with the parameters filled in (offsets first: the pool may reallocate)
        toks.clear();
        ex.clear();
        size_t first[3] = {0, 0, 0};
        std::vector<size_t> off;
        for (int a = 0; a < 3; ++a) {
            first[a] = ex.size();
            if (cm.n_e[a] < 0 || (cm.n_e[a] > 0 && cm.e[a] == nullptr)) return fail(c, WS_EINVAL, "ws_exec: command %d has a bad expression list", k);
            for (int32_t j = 0; j < cm.n_e[a]; ++j) {
                const ws_expr& src = cm.e[a][j];
                if (src.toks == nullptr || src.n <= 0) return fail(c, WS_EINVAL, "ws_exec: command %d has an empty expression", k);
                off.push_back(toks.size());
                for (int32_t i = 0; i < src.n; ++i) {
                    ws_tok t = src.toks[i];
                    if (t.op == WS_TOK_PARAM) {
                        if (t.col < 0 || t.col >= n_params || params == nullptr)
                            return fail(c, WS_EINVAL, "ws_exec: parameter %d of %d", t.col, n_params);
                        t.op = WS_TOK_CONST;
                        t.val = params[t.col];
                        t.col = 0;
                    }
                    toks.push_back(t);
                }
                ex.push_back(ws_expr{nullptr, src.n, 0});
            }
        }
        for (size_t j = 0; j < ex.size(); ++j) ex[j].toks = toks.data() + off[j];
        const ws_expr* e0 = cm.n_e[0] > 0 ? &ex[first[0]] : nullptr;
        const ws_expr* e1 = cm.n_e[1] > 0 ? &ex[first[1]] : nullptr;
        const ws_expr* e2 = cm.n_e[2] > 0 ? &ex[first[2]] : nullptr;
        switch (cm.fn) {
            case WS_CMD_ASSIGN: TRY(ws_assign(c, cm.i0, cm.i1, e0)); break;
            case WS_CMD_ASSIGN_VEC: TRY(ws_assign_vec(c, cm.i0, cm.i1, e0)); break;
            case WS_CMD_SAMPLE_NORMAL: TRY(ws_sample_normal(c, cm.i0, cm.i1, e0, e1)); break;
            case WS_CMD_SAMPLE_EXPONENTIAL: TRY(ws_sample_exponential(c, cm.i0, cm.i1, e0)); break;
            case WS_CMD_SAMPLE_MVNORMAL: TRY(ws_sample_mvnormal(c, cm.i0, cm.i1, e0, cm.mat)); break;
            case WS_CMD_OBSERVE_NORMAL: TRY(ws_observe_normal(c, e0, e1, e2)); break;
            case WS_CMD_OBSERVE_EXPONENTIAL: TRY(ws_observe_exponential(c, e0, e1)); break;
            case WS_CMD_OBSERVE_MVNORMAL: TRY(ws_observe_mvnormal(c, cm.i0, e0, e1, cm.mat)); break;
            case WS_CMD_WEIGHT_EXPR: TRY(ws_weight_expr(c, e0)); break;
            case WS_CMD_SAMPLE_EXPR: TRY(ws_sample_expr(c, cm.i0, cm.i1, e0, e1, e2)); break;
            case WS_CMD_RESAMPLE: TRY(ws_resample_async(c)); break;
            default: return fail(c, WS_EINVAL, "ws_exec: unknown command %d", cm.fn);
        }
    }
    return WS_OK;
}

// the list once per element, for n_elems consecutive elements (params[e][n_params]): one call per block of loop elements
extern "C" int ws_exec_n(ws_ctx* c, const ws_cmd* cmds, int32_t n_cmds, const double* params, int32_t n_params, int32_t n_elems) {
    if (!c || n_elems < 0 || (n_params > 0 && n_elems > 0 && !params)) return WS_EINVAL;
    for (int32_t e = 0; e < n_elems; ++e) TRY(ws_exec(c, cmds, n_cmds, params + (size_t)e * (size_t)n_params, n_params));
    return WS_OK;
}

// ---- speculative blocks of (weighting statements, Resample) steps --------------------------------------------------
// A model that only observes between resampling events (examples/linear_regression.jl: y => Normal(alpha + beta x_i, 1)
// and `if resampled` moves, 12 events in 10 000 steps) pays, statement by statement, one pass over the particles and
// one host round trip per observation, because Resample.apply! needs the ESS after every one.  Here K steps are issued
// as ONE pass: the Resample of each step becomes a checkpoint of the window (ws_vm_kernel<.., true>: the terms so far
// are folded into the running log-weight — same association as the separate passes — and pushed into that step's
// (m, S, Q) state), K finalize kernels give the K decisions, and the host looks at them once.
//   * none fires: the K steps are done (log-weights, tape, depth, Philox stream numbering as if run one by one);
//   * step k is the first to fire: everything after step k is rolled back (log-weights from the copy taken before the
//     block, tape / score program / depth / stream numbering from the marks of step k), the first k + 1 steps are run
//     again as a plain window, and the Resample of step k goes through ws_resample itself.
// Statements that write planes or draw variates are refused (nothing but log-weights may change inside a block).
static int spec_checkpoint(ws_ctx* c) {
    if (!c->weights_changed) return WS_OK;   // Resample is a no-op (transformers.jl:475-477): no decision to record
    if (c->win.ops.empty() || !c->win.has_acc) return fail(c, WS_EUNSUPPORTED, "speculative block: a step without a weighting term");
    if (!c->win.dirty.empty()) return fail(c, WS_EUNSUPPORTED, "speculative block: a statement writes a column");
    if (c->spec_steps.size() >= WS_VM_MAX_CKPT) return fail(c, WS_EUNSUPPORTED, "speculative block: more than %d steps", WS_VM_MAX_CKPT);
    if (c->win.ops.size() > 255) return fail(c, WS_EUNSUPPORTED, "speculative block: window too long");
    ws_ctx::SpecStep st;
    st.tape_size = c->tape.size();
    st.score_mark = c->score.mark();
    st.depth = c->depth;
    st.stream_before = c->next_stream;
    st.ckpt_pc = (int32_t)c->win.ops.size() - 1;
    c->spec_steps.push_back(st);
    c->next_stream++;            // the step's Philox stream is taken whether or not it fires (ws_resample)
    c->weights_changed = false;
    return WS_OK;
}

extern "C" int ws_exec_spec(ws_ctx* c, const ws_cmd* cmds, int32_t n_cmds, const double* params, int32_t n_params, int32_t n_steps,
                            int32_t* n_done, int32_t* fired) {
    if (!c || !n_done || !fired || n_steps < 1 || (n_params > 0 && !params)) return WS_EINVAL;
    *n_done = 0;
    *fired = 0;
    if (c->nranks > 1 || c->d_replay_u != nullptr || c->d_replay_n != nullptr || !c->lazy_gather || c->cols.empty() || !c->async_resample)
        return fail(c, WS_EUNSUPPORTED, "speculative blocks need a single-GPU state without replayed streams");
    TRY(flush_window(c));
    TRY(resolve_spec(c));
    CK(c, cudaSetDevice(c->device));
    if (c->d_ck_partials == nullptr) {
        CK(c, cudaMalloc(&c->d_ck_partials, sizeof(WsLse) * WS_MAX_PARTIALS * WS_VM_MAX_CKPT));
        CK(c, cudaMalloc(&c->d_ck_red, sizeof(WsReduceOut) * WS_VM_MAX_CKPT));
        CK(c, cudaMallocHost(&c->h_ck_red, sizeof(WsReduceOut) * WS_VM_MAX_CKPT));
        CK(c, cudaMalloc(&c->d_logw_bak, sizeof(double) * (size_t)c->n));
    }
    // ---- snapshot ----
    const bool s_uniform = c->logw_uniform, s_partials = c->partials_valid, s_red = c->red_valid, s_resampled = c->resampled,
               s_changed = c->weights_changed, s_wide = c->score_wide;
    const double s_base = c->logw_base;
    const int s_npart = c->n_partials;
    const size_t s_tape = c->tape.size();
    const Program::Mark s_score = c->score.mark();
    const int64_t s_depth = c->depth;
    const uint64_t s_stream = c->next_stream;
    const ws_stats s_stats = c->stats;
    auto restore = [&](size_t tape_size, const Program::Mark& score_mark, int64_t depth, uint64_t stream) {
        reset_window(c);
        c->tape.resize(tape_size);
        if (c->score_wide != s_wide) {
            c->score = Program();   // the tape went wide inside the block: it is folded from its entries anyway
        } else if (!c->score_wide) {
            c->score.rollback(score_mark);
            c->d_score_uploaded = std::min(c->d_score_uploaded, c->score.ops.size());
        }
        c->depth = depth;
        c->next_stream = stream;
    };
    // ---- queue the steps ----
    c->spec_block = true;
    c->spec_steps.clear();
    int rc = WS_OK;
    int32_t issued = 0;
    for (; issued < n_steps; ++issued) {
        // room for one more step?  (every step of a block lowers to the same number of micro-ops)
        if (issued > 0) {
            const size_t per = (size_t)c->spec_steps[0].ckpt_pc + 1;
            if (c->win.ops.size() + per > (size_t)std::min(WS_VM_MAX_OPS, 255) || (int)c->spec_steps.size() >= WS_VM_MAX_CKPT) break;
        }
        const size_t before = c->spec_steps.size();
        rc = ws_exec(c, cmds, n_cmds, params + (size_t)issued * (size_t)n_params, n_params);
        if (rc != WS_OK) break;
        if (c->spec_steps.size() != before + 1) {
            rc = fail(c, WS_EUNSUPPORTED, "speculative block: a step must end in exactly one Resample that has something to decide");
            break;
        }
    }
    if (rc != WS_OK) {
        const std::string msg = c->err;
        c->spec_block = false;
        c->spec_steps.clear();
        restore(s_tape, s_score, s_depth, s_stream);
        c->weights_changed = s_changed;
        c->stats = s_stats;
        c->err = msg;
        return rc;
    }
    // ---- one pass, K decisions ----
    const int32_t K = (int32_t)c->spec_steps.size();
    Program saved = c->win;
    c->spec_flushing = true;
    rc = flush_window(c);
    c->spec_flushing = false;
    c->spec_block = false;
    if (rc != WS_OK) return rc;
    std::swap(c->logw, c->d_logw_bak);   // the pass wrote the other array: c->logw = after the block, d_logw_bak = before it
    const int grid = c->n_partials;
    CK(c, ws_launch_finalize_multi(c->d_ck_partials, grid, K, c->n_global, c->ess_perc_min, c->d_ck_red, c->stream));
    CK(c, cudaMemcpyAsync(c->h_ck_red, c->d_ck_red, sizeof(WsReduceOut) * (size_t)K, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    c->stats.kernel_launches += 1;
    c->stats.d2h_bytes += (int64_t)sizeof(WsReduceOut) * K;
    int32_t first = K;
    for (int32_t j = 0; j < K; ++j)
        if (c->h_ck_red[j].do_resample) {
            first = j;
            break;
        }
    if (first == K) {
        // nothing fired: the block is done
        const WsReduceOut& last = c->h_ck_red[K - 1];
        *c->h_red = last;
        CK(c, cudaMemcpyAsync(c->d_red, c->d_ck_red + (K - 1), sizeof(WsReduceOut), cudaMemcpyDeviceToDevice, c->stream));
        c->red_valid = true;
        c->resampled = false;
        c->weights_changed = false;
        c->stats.resamples_fired += K;
        c->last_info = ws_resample_info{1, 0, last.ess_perc, last.log_mean_w, -1};
        c->last_info_pending = false;
        c->spec_steps.clear();
        *n_done = K;
        *fired = 0;
        return WS_OK;
    }
    // ---- step `first` fires: back to the state before the block, the first `first + 1` steps again as a plain window ----
    const ws_ctx::SpecStep st = c->spec_steps[first];
    std::swap(c->logw, c->d_logw_bak);   // back to the array the block started from
    c->logw_uniform = s_uniform;
    c->logw_base = s_base;
    c->logw_spec = false;
    c->partials_valid = false;
    c->red_valid = false;
    (void)s_partials; (void)s_red; (void)s_npart;
    c->resampled = s_resampled;
    restore(st.tape_size, st.score_mark, st.depth, st.stream_before);
    // steps 0 .. first again, as the same kind of pass (its checkpoints are simply not looked at)
    saved.ops.resize((size_t)st.ckpt_pc + 1);
    c->win = saved;
    c->spec_steps.resize((size_t)first + 1);
    c->spec_flushing = true;
    rc = flush_window(c);
    c->spec_flushing = false;
    c->spec_steps.clear();
    if (rc != WS_OK) return rc;
    std::swap(c->logw, c->d_logw_bak);
    c->stats.resamples_fired += first;   // the steps before it were evaluated and did not fire
    c->weights_changed = true;
    ws_resample_info info{};
    TRY(ws_resample(c, &info));
    *n_done = first + 1;
    *fired = info.resampled;
    return WS_OK;
}

extern "C" int ws_last_resample(ws_ctx* c, ws_resample_info* info) {
    if (!c || !info) return WS_EINVAL;
    if (c->last_info_pending) TRY(resolve_spec(c));
    if (c->last_info.resampled < 0) {  // a no-op step: `resampled` is whatever the steps before it left
        TRY(resolve_spec(c));
        c->last_info.resampled = c->resampled ? 1 : 0;
    }
    *info = c->last_info;
    return WS_OK;
}

extern "C" int ws_gather(ws_ctx* c, const int32_t* ancestors_host) {
    if (!c || !ancestors_host) return WS_EINVAL;
    TRY(flush_window(c));
    TRY(materialize_planes(c));
    CK(c, cudaMemcpyAsync(c->d_anc, ancestors_host, sizeof(int32_t) * (size_t)c->n, cudaMemcpyHostToDevice, c->stream));
    c->stats.h2d_bytes += (int64_t)sizeof(int32_t) * c->n;
    TRY(gather_all(c, c->d_anc));
    CK(c, cudaStreamSynchronize(c->stream));
    return WS_OK;
}

extern "C" int ws_ancestors_download(ws_ctx* c, int32_t* host_out) {
    if (!c || !host_out) return WS_EINVAL;
    TRY(flush_window(c));
    CK(c, cudaMemcpyAsync(host_out, c->d_anc, sizeof(int32_t) * (size_t)c->n, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    c->stats.d2h_bytes += (int64_t)sizeof(int32_t) * c->n;
    return WS_OK;
}

extern "C" int ws_log_evidence(ws_ctx* c, double* log_evidence, double* ess_perc) {
    if (!c) return WS_EINVAL;
    TRY(flush_window(c));
    TRY(resolve_spec(c));
    if (c->logw_uniform) {  // logsumexp(fill(c, N)) - log N = c ; ESS% = 1
        if (log_evidence) *log_evidence = c->logw_base;
        if (ess_perc) *ess_perc = 1.0;
        return WS_OK;
    }
    TRY(ensure_reduced(c));
    if (log_evidence) *log_evidence = c->h_red->log_mean_w;
    if (ess_perc) *ess_perc = c->h_red->ess_perc;
    return WS_OK;
}

extern "C" int ws_exp_norm(ws_ctx* c, double* host_out) {
    if (!c || !host_out) return WS_EINVAL;
    TRY(ensure_reduced(c));
    TRY(ensure_scratch(c, sizeof(double) * (size_t)c->n));
    TimedEvent te;
    timed_begin(c, KC_OTHER, te);
    CK(c, ws_launch_exp_norm(c->logw, c->d_red, c->d_scratch, c->n, grid_for(c, c->n, 256, 8), c->stream));
    timed_end(c, te);
    CK(c, cudaMemcpyAsync(host_out, c->d_scratch, sizeof(double) * (size_t)c->n, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    c->stats.d2h_bytes += (int64_t)sizeof(double) * c->n;
    return WS_OK;
}

// ---- pure functions on caller arrays ------------------------------------------------------------
struct TempBuf {
    void* p = nullptr;
    ~TempBuf() {
        if (p) cudaFree(p);
    }
};

static int reduce_host_array(ws_ctx* c, const double* d_logw, int64_t n) {
    TRY(resolve_spec(c));  // d_partials / d_red are reused as scratch below
    const int grid = std::min(grid_for(c, n, 256, 8), WS_MAX_PARTIALS);
    TimedEvent te;
    timed_begin(c, KC_REDUCE, te);
    CK(c, ws_launch_reduce_logw(d_logw, n, c->d_partials, grid, c->stream));
    timed_end(c, te);
    timed_begin(c, KC_FINALIZE, te);
    CK(c, ws_launch_finalize(c->d_partials, grid, n, c->ess_perc_min, c->d_red, c->stream));
    timed_end(c, te);
    CK(c, cudaMemcpyAsync(c->h_red, c->d_red, sizeof(WsReduceOut), cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    // the state's own reduction is no longer what d_red / d_partials hold
    c->red_valid = false;
    c->partials_valid = false;
    return WS_OK;
}

extern "C" int ws_exp_norm_host(ws_ctx* c, const double* logw, int64_t n, double* w_out) {
    if (!c || !logw || !w_out || n <= 0) return c ? fail(c, WS_EINVAL, "ws_exp_norm_host: bad arguments") : WS_EINVAL;
    TRY(flush_window(c));
    CK(c, cudaSetDevice(c->device));
    TempBuf in, out;
    CK(c, cudaMalloc(&in.p, sizeof(double) * (size_t)n));
    CK(c, cudaMalloc(&out.p, sizeof(double) * (size_t)n));
    CK(c, cudaMemcpyAsync(in.p, logw, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    TRY(reduce_host_array(c, (const double*)in.p, n));
    CK(c, ws_launch_exp_norm((const double*)in.p, c->d_red, (double*)out.p, n, grid_for(c, n, 256, 8), c->stream));
    c->stats.kernel_launches++;
    CK(c, cudaMemcpyAsync(w_out, out.p, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    c->stats.h2d_bytes += (int64_t)sizeof(double) * n;
    c->stats.d2h_bytes += (int64_t)sizeof(double) * n;
    return WS_OK;
}

extern "C" int ws_logsumexp_host(ws_ctx* c, const double* logw, int64_t n, double* out) {
    if (!c || !logw || !out || n <= 0) return c ? fail(c, WS_EINVAL, "ws_logsumexp_host: bad arguments") : WS_EINVAL;
    TRY(flush_window(c));
    CK(c, cudaSetDevice(c->device));
    TempBuf in;
    CK(c, cudaMalloc(&in.p, sizeof(double) * (size_t)n));
    CK(c, cudaMemcpyAsync(in.p, logw, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    TRY(reduce_host_array(c, (const double*)in.p, n));
    *out = c->h_red->lse;
    c->stats.h2d_bytes += (int64_t)sizeof(double) * n;
    return WS_OK;
}

extern "C" int ws_ess_perc_host(ws_ctx* c, const double* w, int64_t n, double* out) {
    if (!c || !w || !out || n <= 0) return c ? fail(c, WS_EINVAL, "ws_ess_perc_host: bad arguments") : WS_EINVAL;
    TRY(flush_window(c));
    CK(c, cudaSetDevice(c->device));
    TempBuf in, part;
    const int grid = std::min(grid_for(c, n, 256, 8), WS_MAX_PARTIALS);
    CK(c, cudaMalloc(&in.p, sizeof(double) * (size_t)n));
    CK(c, cudaMalloc(&part.p, sizeof(double) * (size_t)grid));
    CK(c, cudaMemcpyAsync(in.p, w, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CK(c, ws_launch_sumsq((const double*)in.p, n, (double*)part.p, grid, c->stream));
    c->stats.kernel_launches++;
    std::vector<double> hp(grid);
    CK(c, cudaMemcpyAsync(hp.data(), part.p, sizeof(double) * (size_t)grid, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    double s = 0.0;
    for (int i = 0; i < grid; ++i) s += hp[i];
    *out = 1.0 / ((double)n * s);
    c->stats.h2d_bytes += (int64_t)sizeof(double) * n;
    return WS_OK;
}

static int resample_host_impl(ws_ctx* c, const double* weights, int64_t n, int scheme, const double* uniforms,
                              int64_t n_uniforms, bool sorted_mode, int32_t* indices_out, int64_t* n_clamped) {
    TRY(flush_window(c));
    TRY(resolve_spec(c));
    CK(c, cudaSetDevice(c->device));
    if (n >= (int64_t)2147483647 - 65536) return fail(c, WS_EINVAL, "n must be < 2^31 - 65536");
    TempBuf w, u, anc, words, cdf;
    const int64_t n_tiles = (n + WS_CDF_TILE - 1) / WS_CDF_TILE;
    CK(c, cudaMalloc(&w.p, sizeof(double) * (size_t)n));
    CK(c, cudaMalloc(&anc.p, sizeof(int32_t) * (size_t)n));
    CK(c, cudaMalloc(&words.p, sizeof(unsigned long long) * ws_scan_words(n)));
    CK(c, cudaMalloc(&cdf.p, sizeof(unsigned long long) * (size_t)n));
    CK(c, cudaMemcpyAsync(w.p, weights, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    if (uniforms != nullptr) {
        CK(c, cudaMalloc(&u.p, sizeof(double) * (size_t)n_uniforms));
        CK(c, cudaMemcpyAsync(u.p, uniforms, sizeof(double) * (size_t)n_uniforms, cudaMemcpyHostToDevice, c->stream));
    }
    CK(c, cudaMemsetAsync(c->d_counters + 1, 0, sizeof(unsigned long long), c->stream));
    const uint64_t stream_id = c->next_stream++;
    TRY(run_scan_search(c, (const double*)w.p, 1, scheme, n, sorted_mode ? nullptr : (const double*)u.p,
                        sorted_mode ? (const double*)u.p : nullptr, (int32_t*)anc.p, (unsigned long long*)words.p,
                        (unsigned long long*)cdf.p, stream_id, c->d_counters + 1));
    CK(c, cudaMemcpyAsync(indices_out, anc.p, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    unsigned long long h_clamped = 0;
    CK(c, cudaMemcpyAsync(&h_clamped, c->d_counters + 1, sizeof(h_clamped), cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    if (n_clamped) *n_clamped = (int64_t)h_clamped;
    c->stats.h2d_bytes += (int64_t)sizeof(double) * (n + (uniforms ? n_uniforms : 0));
    c->stats.d2h_bytes += (int64_t)sizeof(int32_t) * n;
    return WS_OK;
}

extern "C" int ws_icdf_host(ws_ctx* c, const double* weights, const double* us, int64_t n, int32_t* indices_out, int64_t* n_clamped) {
    if (!c || !weights || !us || !indices_out || n <= 0) return c ? fail(c, WS_EINVAL, "ws_icdf_host: bad arguments") : WS_EINVAL;
    return resample_host_impl(c, weights, n, WS_RESAMPLER_STRATIFIED, us, n, true, indices_out, n_clamped);
}

extern "C" int ws_resample_host(ws_ctx* c, const double* weights, int64_t n, int scheme, const double* uniforms,
                                int32_t* indices_out, int64_t* n_clamped) {
    if (!c || !weights || !indices_out || n <= 0) return c ? fail(c, WS_EINVAL, "ws_resample_host: bad arguments") : WS_EINVAL;
    if (scheme == WS_RESAMPLER_STRATIFIED) return resample_host_impl(c, weights, n, scheme, uniforms, n, false, indices_out, n_clamped);
    if (scheme == WS_RESAMPLER_SYSTEMATIC) return resample_host_impl(c, weights, n, scheme, uniforms, 1, false, indices_out, n_clamped);
    if (scheme == WS_RESAMPLER_MULTINOMIAL) {
        if (uniforms == nullptr) return resample_host_impl(c, weights, n, scheme, nullptr, 0, false, indices_out, n_clamped);  // Philox: no sort
        std::vector<double> su(uniforms, uniforms + n);
        std::sort(su.begin(), su.end());
        return resample_host_impl(c, weights, n, scheme, su.data(), n, true, indices_out, n_clamped);
    }
    return fail(c, WS_EINVAL, "unknown resampling scheme %d", scheme);
}

// ------------------------------------------------------------------------------------------
// analysis
// ------------------------------------------------------------------------------------------
extern "C" int ws_expectation(ws_ctx* c, const ws_expr* f, int32_t n_exprs, double* out) {
    if (!c || !f || !out) return WS_EINVAL;
    if (n_exprs < 1 || n_exprs > 8) return fail(c, WS_EINVAL, "ws_expectation: 1..8 expressions per call");
    for (int k = 0; k < n_exprs; ++k) TRY(check_expr(c, &f[k], "ws_expectation"));
    TRY(ensure_reduced(c));
    Program p;
    p.max_regs = WS_VM_MAX_REGS;
    p.max_ops = WS_VM_MAX_OPS;
    p.max_io = WS_VM_MAX_IO;
    int regs[8];
    for (int k = 0; k < n_exprs; ++k) {
        Val v = p.compile(f[k]);
        // keep the result in a register that later expressions cannot recycle
        int t = p.alloc_plane_reg();
        if (v.is_const)
            p.emit(ws_make_op(WS_OP_LIN2, t, WS_REG_NONE, WS_REG_NONE, WS_REG_NONE, 0, v.c0, 0, 0));
        else
            p.emit(ws_make_op(WS_OP_LIN2, t, v.reg, WS_REG_NONE, WS_REG_NONE, 0, v.c0, v.c1, 0));
        regs[k] = t;
        p.end_statement();
    }
    if (!p.error.empty()) return fail(c, WS_EINVAL, "%s", p.error.c_str());
    if (p.overflow) return fail(c, WS_EUNSUPPORTED, "ws_expectation: expressions do not fit one device pass");
    WsVmProgram P;
    memset(&P, 0, sizeof(P));
    P.n = c->n;
    P.particle_offset = c->offset;
    P.n_ops = (int)p.ops.size();
    P.n_loads = (int)p.loads.size();
    P.n_stores = 0;
    P.n_regs = std::max(1, p.high_water);
    {
        std::vector<Plane> loaded;
        for (auto& ld : p.loads) loaded.push_back(ld.first);
        TRY(materialize_deep(c, loaded));
    }
    P.ancestors = c->d_anc;
    for (int k = 0; k < P.n_loads; ++k) {
        const Plane pl = p.loads[k].first;
        P.load_ptr[k] = plane_ptr(c, pl);
        P.load_reg[k] = (uint8_t)p.loads[k].second;
        if (c->cols[pl.col].stale[pl.comp]) P.load_gather |= (1u << k);
    }
    P.logw_mode = 0;
    P.logw = c->logw;
    P.n_expect = n_exprs;
    for (int k = 0; k < n_exprs; ++k) P.expect_reg[k] = (uint8_t)regs[k];
    P.red = c->d_red;
    const int64_t vm_tile = (int64_t)WS_VM_BLOCK * WS_VM_P;
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(ws_vm_max_grid(P.n_regs, P.n_loads, P.n_ops, c->sm_count), (c->n + vm_tile - 1) / vm_tile));
    TRY(ensure_scratch(c, sizeof(double) * (size_t)grid * 8));
    TRY(ensure_h_scratch(c, sizeof(double) * (size_t)grid * 8));
    P.expect_partials = c->d_scratch;
    P.rng.seed = c->seed;
    memcpy(P.ops, p.ops.data(), sizeof(WsOp) * p.ops.size());
    TimedEvent te;
    timed_begin(c, KC_VM, te);
    CK(c, ws_launch_vm(P, grid, c->stream));
    timed_end(c, te);
    CK(c, cudaMemcpyAsync(c->h_scratch, c->d_scratch, sizeof(double) * (size_t)grid * n_exprs, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    for (int k = 0; k < n_exprs; ++k) {
        double s = 0.0;
        for (int b = 0; b < grid; ++b) s += c->h_scratch[(size_t)b * n_exprs + k];
        out[k] = s;
    }
    if (c->nranks > 1) TRY(allreduce_host_doubles(c, out, n_exprs));
    return WS_OK;
}

// rows `d_idx` (n_idx local row indices on the device) of plane k of column `col` -> d_out: the requested rows are traced
// back through the genealogy when the plane is behind (n_idx chains, not n); `rows` is scratch for the traced indices
static int gather_rows_traced(ws_ctx* c, const Column& col, int k, const int64_t* d_idx, int64_t n_idx, TempBuf& rows, double* d_out) {
    const int64_t* use = d_idx;
    if (col.stale[k]) {
        if (rows.p == nullptr) CK(c, cudaMalloc(&rows.p, sizeof(int64_t) * (size_t)n_idx));
        const int64_t* start = d_idx;
        int64_t from = c->epoch;
        while (from > col.ep[k]) {
            WsComposeParams P;
            memset(&P, 0, sizeof(P));
            P.n = n_idx;
            P.n_rows = c->n;
            while (from > col.ep[k] && P.n_chain < WS_COMPOSE_MAX_CHAIN) {
                const int32_t* a = anc_of_event(c, from);
                if (a == nullptr) return fail(c, WS_EINVAL, "genealogy: ancestors of event %lld were released", (long long)from);
                P.chain[P.n_chain++] = a;
                --from;
            }
            CK(c, ws_launch_compose_rows(P, (int64_t*)rows.p, start, c->stream));
            c->stats.kernel_launches++;
            start = (const int64_t*)rows.p;
        }
        use = (const int64_t*)rows.p;
    }
    CK(c, ws_launch_gather_rows(col.front[k], use, n_idx, d_out, c->stream));
    c->stats.kernel_launches++;
    return WS_OK;
}

extern "C" int ws_col_download_rows(ws_ctx* c, int32_t id, const int64_t* indices, int64_t n_idx, double* host_out) {
    if (!c || !indices || !host_out || n_idx <= 0) return c ? fail(c, WS_EINVAL, "ws_col_download_rows: bad arguments") : WS_EINVAL;
    if (id < 0 || id >= (int32_t)c->cols.size()) return fail(c, WS_EINVAL, "unknown column id %d", id);
    for (int64_t i = 0; i < n_idx; ++i)
        if (indices[i] < 0 || indices[i] >= c->n) return fail(c, WS_EINVAL, "row index %lld out of range", (long long)indices[i]);
    TRY(flush_window(c));
    CK(c, cudaSetDevice(c->device));
    TempBuf idx, out, rows;
    CK(c, cudaMalloc(&idx.p, sizeof(int64_t) * (size_t)n_idx));
    CK(c, cudaMalloc(&out.p, sizeof(double) * (size_t)n_idx));
    CK(c, cudaMemcpyAsync(idx.p, indices, sizeof(int64_t) * (size_t)n_idx, cudaMemcpyHostToDevice, c->stream));
    const Column& col = c->cols[id];
    for (int k = 0; k < col.width; ++k) {
        TRY(gather_rows_traced(c, col, k, (const int64_t*)idx.p, n_idx, rows, (double*)out.p));
        CK(c, cudaMemcpyAsync(host_out + (size_t)k * n_idx, out.p, sizeof(double) * (size_t)n_idx, cudaMemcpyDeviceToHost, c->stream));
    }
    CK(c, cudaStreamSynchronize(c->stream));
    return WS_OK;
}

// cross-rank hooks of a sharded describe / sample (ws_stats.h: WsStatsComm)
static int stats_allgather_words(void* ctx, const unsigned long long* in, size_t words, unsigned long long* out);
static int stats_allreduce_doubles(void* ctx, double* v, int n);
static int stats_allreduce_u64_device(void* ctx, unsigned long long* d, size_t n);

// Rows of GLOBAL particle indices.  Every rank reads the rows it owns into a zeroed n_idx x width buffer of bit patterns;
// on a sharded state the buffers are summed as 64-bit integers, which is exact (one rank contributes each row) and
// keeps -0.0 and NaN payloads.
extern "C" int ws_col_download_global_rows(ws_ctx* c, int32_t id, const int64_t* global_indices, int64_t n_idx, double* host_out) {
    if (!c || !global_indices || !host_out || n_idx <= 0)
        return c ? fail(c, WS_EINVAL, "ws_col_download_global_rows: bad arguments") : WS_EINVAL;
    if (id < 0 || id >= (int32_t)c->cols.size()) return fail(c, WS_EINVAL, "unknown column id %d", id);
    for (int64_t i = 0; i < n_idx; ++i)
        if (global_indices[i] < 0 || global_indices[i] >= c->n_global)
            return fail(c, WS_EINVAL, "particle index %lld out of range", (long long)global_indices[i]);
    TRY(flush_window(c));
    const Column& col = c->cols[id];
    if (c->nranks > 1) {  // sharded states have no genealogy: bring the planes into the current particle order first
        std::vector<Plane> pl;
        for (int k = 0; k < col.width; ++k) pl.push_back(Plane{id, k});
        TRY(materialize_planes(c, &pl));
    }
    CK(c, cudaSetDevice(c->device));
    std::vector<int64_t> loc, pos;  // local row and place in the output of the rows this rank owns
    for (int64_t i = 0; i < n_idx; ++i) {
        const int64_t r = global_indices[i] - c->offset;
        if (r >= 0 && r < c->n) {
            loc.push_back(r);
            pos.push_back(i);
        }
    }
    const int64_t n_own = (int64_t)loc.size();
    const size_t total = (size_t)n_idx * (size_t)col.width;
    TempBuf d_loc, d_pos, tmp, out, rows;
    CK(c, cudaMalloc(&out.p, sizeof(double) * total));
    CK(c, cudaMemsetAsync(out.p, 0, sizeof(double) * total, c->stream));
    if (n_own > 0) {
        CK(c, cudaMalloc(&d_loc.p, sizeof(int64_t) * (size_t)n_own));
        CK(c, cudaMalloc(&d_pos.p, sizeof(int64_t) * (size_t)n_own));
        CK(c, cudaMalloc(&tmp.p, sizeof(double) * (size_t)n_own));
        CK(c, cudaMemcpyAsync(d_loc.p, loc.data(), sizeof(int64_t) * (size_t)n_own, cudaMemcpyHostToDevice, c->stream));
        CK(c, cudaMemcpyAsync(d_pos.p, pos.data(), sizeof(int64_t) * (size_t)n_own, cudaMemcpyHostToDevice, c->stream));
        c->stats.h2d_bytes += (int64_t)(2 * sizeof(int64_t)) * n_own;
        for (int k = 0; k < col.width; ++k) {
            TRY(gather_rows_traced(c, col, k, (const int64_t*)d_loc.p, n_own, rows, (double*)tmp.p));
            CK(c, ws_sample_scatter_rows((const double*)tmp.p, (const int64_t*)d_pos.p, n_own, (double*)out.p + (size_t)k * n_idx, c->stream));
            c->stats.kernel_launches++;
        }
    }
    if (c->nranks > 1) TRY(stats_allreduce_u64_device(c, (unsigned long long*)out.p, total));
    CK(c, cudaMemcpyAsync(host_out, out.p, sizeof(double) * total, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    c->stats.d2h_bytes += (int64_t)(sizeof(double) * total);
    return WS_OK;
}

// sample(state, n; replace) (src/utils.jl:102-118): the draw include/wsb200.h defines, made on the device
// (csrc/ws_kernels_stats.cu).  Nothing of size N leaves the device: only the n indices (and, without replacement, their
// keys) come to the host.  Collective on a sharded state.
extern "C" int ws_sample_indices(ws_ctx* c, int64_t n_draws, int replace, int64_t* indices_out) {
    if (!c || !indices_out) return WS_EINVAL;
    if (n_draws <= 0) return fail(c, WS_EINVAL, "Number of samples must be positive");
    if (!replace && n_draws > c->n_global)
        return fail(c, WS_EINVAL, "Cannot sample %lld particles without replacement from %lld particles", (long long)n_draws, (long long)c->n_global);
    TRY(ensure_reduced(c));  // flushes the window; m is the global maximum on a sharded state
    const double m = c->h_red->m;
    if (!std::isfinite(m)) return fail(c, WS_ENUMERIC, "sample(state, n): the largest log-weight is %g, so the weights cannot be normalised", m);
    CK(c, cudaSetDevice(c->device));
    const uint64_t stream_id = c->next_stream++;
    TRY(ensure_scratch(c, ws_sample_scratch_bytes(c->n, n_draws, replace)));
    WsStatsComm comm{c, c->nranks, stats_allgather_words, stats_allreduce_doubles, stats_allreduce_u64_device, c->rank};
    int launches = 0;
    const cudaError_t e = ws_sample_draw(c->logw, c->n, c->offset, c->n_global, m, c->seed, stream_id, n_draws, replace, c->d_scratch,
                                         c->stream, indices_out, &launches, &c->stats.d2h_bytes, c->nranks > 1 ? &comm : nullptr);
    c->stats.kernel_launches += launches;
    if (e == cudaErrorInvalidValue) return fail(c, WS_EINVAL, "sample(state, n): the draw is inconsistent across the ranks");
    CK(c, e);
    return WS_OK;
}

// ------------------------------------------------------------------------------------------
// replay
// ------------------------------------------------------------------------------------------
static int set_replay(ws_ctx* c, double** dptr, int64_t* dlen, int64_t* cursor, const double* host, int64_t len) {
    TRY(flush_window(c));
    TRY(resolve_spec(c));
    CK(c, cudaSetDevice(c->device));
    CK(c, cudaStreamSynchronize(c->stream));
    if (*dptr) {
        CK(c, cudaFree(*dptr));
        *dptr = nullptr;
    }
    *dlen = 0;
    *cursor = 0;
    if (host == nullptr || len <= 0) return WS_OK;
    CK(c, cudaMalloc(dptr, sizeof(double) * (size_t)len));
    CK(c, cudaMemcpy(*dptr, host, sizeof(double) * (size_t)len, cudaMemcpyHostToDevice));
    *dlen = len;
    c->stats.h2d_bytes += (int64_t)sizeof(double) * len;
    return WS_OK;
}
extern "C" int ws_set_replay_normals(ws_ctx* c, const double* host, int64_t len) {
    if (!c) return WS_EINVAL;
    return set_replay(c, &c->d_replay_n, &c->replay_n_len, &c->cur_n, host, len);
}
extern "C" int ws_set_replay_uniforms(ws_ctx* c, const double* host, int64_t len) {
    if (!c) return WS_EINVAL;
    return set_replay(c, &c->d_replay_u, &c->replay_u_len, &c->cur_u, host, len);
}
extern "C" int ws_set_replay_variates(ws_ctx* c, const double* host, int64_t len) {
    if (!c) return WS_EINVAL;
    return set_replay(c, &c->d_replay_v, &c->replay_v_len, &c->cur_v, host, len);
}
extern "C" int ws_set_replay_exponentials(ws_ctx* c, const double* host, int64_t len) {
    if (!c) return WS_EINVAL;
    return set_replay(c, &c->d_replay_e, &c->replay_e_len, &c->cur_e, host, len);
}

// ------------------------------------------------------------------------------------------
// tape control / scoring / moves
// ------------------------------------------------------------------------------------------
extern "C" int ws_tape_clear(ws_ctx* c) {
    if (!c) return WS_EINVAL;
    reset_score(c);
    return WS_OK;
}
extern "C" int ws_tape_record_only(ws_ctx* c, int on) {
    if (!c) return WS_EINVAL;
    if (on) TRY(flush_window(c));
    c->record_only = on != 0;
    return WS_OK;
}
extern "C" int ws_tape_enable(ws_ctx* c, int on) {
    if (!c) return WS_EINVAL;
    c->tape_enabled = on != 0;
    return WS_OK;
}
extern "C" int ws_tape_length(const ws_ctx* c, int64_t* n) {
    if (!c || !n) return WS_EINVAL;
    *n = (int64_t)c->tape.size();
    return WS_OK;
}

// number of score micro-ops belonging to entries with depth < target_depth (a prefix: depth is
// non-decreasing along the tape)
static int score_prefix_ops(ws_ctx* c, int64_t target_depth) {
    int n_ops = 0;
    for (auto& e : c->tape) {
        if (e.depth < target_depth) n_ops = e.op_end; else break;
    }
    return n_ops;
}

static double score_prefix_const(ws_ctx* c, int64_t target_depth) {
    double k = 0.0;
    for (auto& e : c->tape) {
        if (e.depth < target_depth) k = e.konst_end; else break;
    }
    return k;
}

static int upload_score_program(ws_ctx* c) {
    const size_t n_ops = c->score.ops.size();
    if (n_ops == 0) return WS_OK;
    if (n_ops > c->d_score_cap) {
        size_t cap = std::max<size_t>(1024, c->d_score_cap * 2);
        while (cap < n_ops) cap *= 2;
        WsOp* nd = nullptr;
        CK(c, cudaMalloc(&nd, sizeof(WsOp) * cap));
        CK(c, cudaStreamSynchronize(c->stream));
        if (c->d_score_ops) CK(c, cudaFree(c->d_score_ops));
        c->d_score_ops = nd;
        c->d_score_cap = cap;
        c->d_score_uploaded = 0;
    }
    if (c->d_score_uploaded < n_ops) {
        // pageable source: the copy is staged before the call returns, so the vector may grow later
        CK(c, cudaMemcpyAsync(c->d_score_ops + c->d_score_uploaded, c->score.ops.data() + c->d_score_uploaded,
                              sizeof(WsOp) * (n_ops - c->d_score_uploaded), cudaMemcpyHostToDevice, c->stream));
        c->stats.h2d_bytes += (int64_t)(sizeof(WsOp) * (n_ops - c->d_score_uploaded));
        c->d_score_uploaded = n_ops;
    }
    return WS_OK;
}

// Wide tapes: lower the scored prefix of the tape into segments that each fit one register file and hand
// every segment to `run`.  `only` (may be null) keeps just the entries that read one of those planes:
// for a move, factors that do not involve a target cancel in s_new - s_old.
template <class F>
static int for_each_tape_segment(ws_ctx* c, int64_t target_depth, const std::vector<Plane>* only, F run) {
    static const int seg_regs = [] {
        const char* e = getenv("WSB200_SEG_REGS");
        const int v = e ? atoi(e) : WS_SCORE_SEG_REGS;
        return std::min(WS_SCORE_MAX_REGS, std::max(WS_SCORE_TEMPS + 4, v));
    }();
    auto fresh = [] {
        Program p;
        p.score_mode = true;
        p.temp_base = 0;
        p.n_temp_slots = WS_SCORE_TEMPS;
        p.max_regs = seg_regs;
        p.max_ops = 1 << 30;
        p.max_io = WS_SCORE_MAX_LOADS;
        return p;
    };
    auto launch = [&](Program& seg) -> int {
        if (seg.ops.empty()) return WS_OK;
        if (seg.ops.size() > c->d_seg_cap) {
            if (c->d_seg_ops) {
                CK(c, cudaStreamSynchronize(c->stream));
                CK(c, cudaFree(c->d_seg_ops));
                c->d_seg_ops = nullptr;
            }
            c->d_seg_cap = std::max<size_t>(4096, seg.ops.size() * 2);
            CK(c, cudaMalloc(&c->d_seg_ops, sizeof(WsOp) * c->d_seg_cap));
        }
        // the previous segment's kernel may still be reading the buffer: stream order protects it, and the
        // source vector is pageable (copied before the call returns)
        CK(c, cudaMemcpyAsync(c->d_seg_ops, seg.ops.data(), sizeof(WsOp) * seg.ops.size(), cudaMemcpyHostToDevice, c->stream));
        c->stats.h2d_bytes += (int64_t)(sizeof(WsOp) * seg.ops.size());
        return run(seg);
    };
    Program seg = fresh();
    for (auto& e : c->tape) {
        if (!(e.depth < target_depth)) break;
        if (only != nullptr) {
            bool dep = false;
            for (auto& r : e.refs)
                for (auto& t : *only)
                    if (r == t) dep = true;
            if (!dep) continue;
        }
        const Program::Mark mk = seg.mark();   // (sizes only: copying the segment per entry made a move's host side quadratic)
        e.lower(seg);
        if (!seg.error.empty()) return fail(c, WS_EINVAL, "%s", seg.error.c_str());
        if (seg.overflow) {
            seg.rollback(mk);
            TRY(launch(seg));
            seg = fresh();
            e.lower(seg);
            if (seg.overflow) return fail(c, WS_EUNSUPPORTED, "one statement reads more than %d planes", WS_SCORE_MAX_LOADS);
        }
        seg.end_statement();
    }
    return launch(seg);
}

// A launch folds a prefix / a selection of the tape: keep only the register-file rows those entries touch
// (a tape reserves WS_SCORE_TEMPS temporaries and one register per plane it ever read; fewer rows = more
// particles per thread and more CTAs per SM in the fold kernels).  The ops stay as they are on the device;
// the kernels renumber while unpacking them (ws_decode_op).
static void compact_score_regs(WsScoreParams& S, const WsOp* ops, size_t n_ops, uint8_t* target_reg, int d) {
    std::vector<uint8_t> keep;
    for (int k = 0; k < S.n_loads; ++k) keep.push_back(S.load_reg[k]);
    for (int t = 0; t < d; ++t) keep.push_back(target_reg[t]);
    S.n_regs = std::max(1, ws_compact_regs(ops, n_ops, keep.data(), (int)keep.size(), S.reg_map));
    for (int k = 0; k < S.n_loads; ++k) S.load_reg[k] = S.reg_map[S.load_reg[k]];
    for (int t = 0; t < d; ++t) target_reg[t] = S.reg_map[target_reg[t]];
}
static void identity_reg_map(WsScoreParams& S) {
    for (int r = 0; r < 256; ++r) S.reg_map[r] = (uint8_t)r;
}

static void fill_segment_launch(ws_ctx* c, WsScoreParams& S, Program& seg) {
    memset(&S, 0, sizeof(S));
    identity_reg_map(S);
    S.n = c->n;
    S.particle_offset = c->offset;
    S.ops = c->d_seg_ops;
    S.n_ops = (int)seg.ops.size();
    S.n_regs = std::max(1, seg.high_water);
    S.n_loads = (int)seg.loads.size();
    S.konst = seg.acc_const;
    for (int k = 0; k < S.n_loads; ++k) {
        S.load_ptr[k] = plane_ptr(c, seg.loads[k].first);
        S.load_reg[k] = (uint8_t)seg.loads[k].second;
    }
}

static int fill_score_launch(ws_ctx* c, WsScoreParams& S, int n_ops) {
    memset(&S, 0, sizeof(S));
    identity_reg_map(S);
    S.n = c->n;
    S.particle_offset = c->offset;
    S.ops = c->d_score_ops;
    S.n_ops = n_ops;
    S.n_regs = std::max(1, c->score.high_water);
    // planes the tape reads: a plane register loaded only if the scored prefix can reference it is
    // not tracked; loading all tape planes is always correct
    S.n_loads = (int)c->score.loads.size();
    if (S.n_loads > WS_SCORE_MAX_LOADS) return fail(c, WS_EUNSUPPORTED, "score tape references more than %d planes", WS_SCORE_MAX_LOADS);
    for (int k = 0; k < S.n_loads; ++k) {
        S.load_ptr[k] = plane_ptr(c, c->score.loads[k].first);
        S.load_reg[k] = (uint8_t)c->score.loads[k].second;
    }
    return WS_OK;
}

extern "C" int ws_score_logpdf(ws_ctx* c, int64_t target_depth, double* host_out) {
    if (!c || !host_out) return WS_EINVAL;
    TRY(flush_window(c));
    TRY(materialize_tape_planes(c, 0, nullptr, nullptr));
    CK(c, cudaSetDevice(c->device));
    TRY(ensure_scratch(c, sizeof(double) * (size_t)c->n));
    if (c->score_wide) {
        CK(c, cudaMemsetAsync(c->d_scratch, 0, sizeof(double) * (size_t)c->n, c->stream));
        WsMoveParams M;
        memset(&M, 0, sizeof(M));
        TRY(for_each_tape_segment(c, target_depth, nullptr, [&](Program& seg) -> int {
            fill_segment_launch(c, M.score, seg);
            TimedEvent te;
            timed_begin(c, KC_MOVE, te);
            CK(c, ws_launch_move_delta(M, 0, nullptr, c->d_scratch, c->sm_count, c->stream));
            timed_end(c, te);
            return WS_OK;
        }));
    } else {
        const int n_ops = score_prefix_ops(c, target_depth);
        TRY(upload_score_program(c));
        WsScoreParams S;
        TRY(fill_score_launch(c, S, n_ops));
        S.konst = score_prefix_const(c, target_depth);
        S.score_out = c->d_scratch;
        compact_score_regs(S, c->score.ops.data(), (size_t)n_ops, nullptr, 0);
        TimedEvent te;
        timed_begin(c, KC_MOVE, te);
        CK(c, ws_launch_score(S, c->sm_count, c->stream));
        timed_end(c, te);
    }
    CK(c, cudaMemcpyAsync(host_out, c->d_scratch, sizeof(double) * (size_t)c->n, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    c->stats.d2h_bytes += (int64_t)sizeof(double) * c->n;
    return WS_OK;
}

extern "C" int ws_marginal_diversity(ws_ctx* c, int32_t n_targets, const int32_t* col, const int32_t* comp, double* out) {
    if (!c || !col || !comp || !out || n_targets < 1) return c ? fail(c, WS_EINVAL, "ws_marginal_diversity: bad arguments") : WS_EINVAL;
    TRY(flush_window(c));
    for (int t = 0; t < n_targets; ++t) TRY(check_plane(c, col[t], comp[t]));
    {
        std::vector<Plane> tg;
        for (int t = 0; t < n_targets; ++t) tg.push_back(Plane{col[t], comp[t]});
        TRY(materialize_planes(c, &tg));
    }
    CK(c, cudaSetDevice(c->device));
    double best = INFINITY;
    for (int t = 0; t < n_targets; ++t) {
        TRY(check_plane(c, col[t], comp[t]));
        // open-addressing table with 2N slots (power of two)
        size_t slots = 1;
        while (slots < (size_t)std::max<int64_t>(c->n, 1) * 2) slots <<= 1;
        const int R = c->nranks;
        // sharded: [table | counter | per-owner counts | per-owner key lists]
        const size_t part_cap = (R > 1) ? (size_t)c->n : 0;
        const size_t words = slots + 8 + (size_t)R + (size_t)R * part_cap;
        TRY(ensure_scratch(c, sizeof(unsigned long long) * words));
        unsigned long long* table = (unsigned long long*)c->d_scratch;
        unsigned long long* counter = table + slots;
        unsigned long long* part_count = counter + 8;
        unsigned long long* part_base = part_count + R;
        TimedEvent te;
        timed_begin(c, KC_OTHER, te);
        CK(c, ws_launch_unique_count(plane_ptr(c, Plane{col[t], comp[t]}), c->n, table, slots, counter, c->sm_count, c->stream, 0,
                                     R > 1 ? part_base : nullptr, (int64_t)part_cap, R > 1 ? part_count : nullptr, R));
        timed_end(c, te);
        unsigned long long distinct = 0;
        if (R == 1) {
            CK(c, cudaMemcpyAsync(&distinct, counter, sizeof(distinct), cudaMemcpyDeviceToHost, c->stream));
            CK(c, cudaStreamSynchronize(c->stream));
        } else {
            // Exact distinct count over all ranks: every locally-new key goes to the rank that owns its
            // hash range (all-to-all-v over NVLink), owners count distinct keys, counts are all-reduced.
            std::vector<unsigned long long> cnt(R), all((size_t)R * R);
            CK(c, cudaMemcpyAsync(cnt.data(), part_count, sizeof(unsigned long long) * R, cudaMemcpyDeviceToHost, c->stream));
            CK(c, cudaStreamSynchronize(c->stream));
            // [counts R x (R+1) | received keys | owner table]: one grow-only buffer (a cudaMalloc / cudaFree per
            // diversity check cost milliseconds each, more than the count itself)
            const size_t cnt_words = ((size_t)R * (R + 1) + 31) & ~(size_t)31;
            TRY(ensure_scratch2(c, sizeof(unsigned long long) * cnt_words));
            unsigned long long* d_cnt = (unsigned long long*)c->d_scratch2;
            CK(c, cudaMemcpyAsync(d_cnt + (size_t)R * R, cnt.data(), sizeof(unsigned long long) * R, cudaMemcpyHostToDevice, c->stream));
            NCK(c, g_nccl.AllGather(d_cnt + (size_t)R * R, d_cnt, (size_t)R, WS_NCCL_UINT64, c->comm, c->stream));
            CK(c, cudaMemcpyAsync(all.data(), d_cnt, sizeof(unsigned long long) * (size_t)R * R, cudaMemcpyDeviceToHost, c->stream));
            CK(c, cudaStreamSynchronize(c->stream));
            size_t n_recv = 0;
            std::vector<size_t> roff(R);
            for (int q = 0; q < R; ++q) {
                roff[q] = n_recv;
                n_recv += (size_t)all[(size_t)q * R + c->rank];  // what q holds for me
            }
            size_t slots2 = 1;
            while (slots2 < std::max<size_t>(n_recv, 1) * 2) slots2 <<= 1;
            const size_t recv_words = (std::max<size_t>(n_recv, 1) + 31) & ~(size_t)31;
            TRY(ensure_scratch2(c, sizeof(unsigned long long) * (cnt_words + recv_words + slots2 + 8)));  // nothing in flight uses it yet
            unsigned long long* d_recv = (unsigned long long*)c->d_scratch2 + cnt_words;
            NCK(c, g_nccl.GroupStart());
            for (int d = 0; d < R; ++d) {
                if (cnt[d] > 0) NCK(c, g_nccl.Send(part_base + (size_t)d * part_cap, (size_t)cnt[d], WS_NCCL_UINT64, d, c->comm, c->stream));
                const size_t rc = (size_t)all[(size_t)d * R + c->rank];
                if (rc > 0) NCK(c, g_nccl.Recv(d_recv + roff[d], rc, WS_NCCL_UINT64, d, c->comm, c->stream));
            }
            NCK(c, g_nccl.GroupEnd());
            unsigned long long* t2 = d_recv + recv_words;
            CK(c, ws_launch_unique_count((const double*)d_recv, (int64_t)n_recv, t2, slots2, t2 + slots2, c->sm_count, c->stream, 1));
            c->stats.kernel_launches++;
            unsigned long long mine = 0;
            CK(c, cudaMemcpyAsync(&mine, t2 + slots2, sizeof(mine), cudaMemcpyDeviceToHost, c->stream));
            CK(c, cudaStreamSynchronize(c->stream));
            double tot = (double)mine;
            TRY(allreduce_host_doubles(c, &tot, 1));
            distinct = (unsigned long long)(tot + 0.5);
        }
        const double frac = (double)distinct / (double)c->n_global;
        if (frac < best) best = frac;
    }
    *out = best;
    return WS_OK;
}

extern "C" int ws_move(ws_ctx* c, const ws_move_spec* spec, ws_move_info* info) {
    if (!c || !spec) return WS_EINVAL;
    const int d = spec->n_targets;
    if (d < 1 || d > WS_MOVE_MAX_D) return fail(c, WS_EUNSUPPORTED, "Move with %d targets (supported: 1..%d)", d, WS_MOVE_MAX_D);
    if (!spec->col || !spec->comp) return fail(c, WS_EINVAL, "ws_move: targets missing");
    for (int t = 0; t < d; ++t) TRY(check_plane(c, spec->col[t], spec->comp[t]));
    if (spec->proposal != WS_PROPOSAL_RW && spec->proposal != WS_PROPOSAL_AUTORW) return fail(c, WS_EINVAL, "ws_move: unknown proposal %d", spec->proposal);
    if (spec->has_bounds && (!spec->lo || !spec->hi)) return fail(c, WS_EINVAL, "ws_move: bounds missing");
    TRY(flush_window(c));
    TRY(resolve_spec(c));
    TRY(materialize_tape_planes(c, d, spec->col, spec->comp));
    CK(c, cudaSetDevice(c->device));
    if (info) {
        info->ran = 0;
        info->diversity = NAN;
        info->n_accepted = 0;
    }
    // diversity gate (transformers.jl:592-594)
    if (!isnan(spec->diversity)) {
        double div = 0.0;
        TRY(ws_marginal_diversity(c, d, spec->col, spec->comp, &div));
        if (info) info->diversity = div;
        if (div >= spec->diversity) return WS_OK;
    }
    const int64_t target_depth = spec->target_depth < 0 ? c->depth : spec->target_depth;

    WsMoveParams M;
    memset(&M, 0, sizeof(M));
    M.d = d;
    for (int t = 0; t < d; ++t) {
        M.target_ptr[t] = plane_ptr(c, Plane{spec->col[t], spec->comp[t]});
        M.lo[t] = spec->has_bounds ? spec->lo[t] : -INFINITY;
        M.hi[t] = spec->has_bounds ? spec->hi[t] : INFINITY;
        M.bound_kind[t] = ws_bound_kind(M.lo[t], M.hi[t]);
    }
    // target registers inside the score program (a target the tape never mentions gets none)
    for (int t = 0; t < d; ++t) {
        auto it = c->score.plane_reg.find(Plane{spec->col[t], spec->comp[t]});
        M.target_reg[t] = (it == c->score.plane_reg.end()) ? 0xFF : (uint8_t)it->second;
    }

    // proposal covariance factor L (d x d lower, row-major): z' = z + L xi
    std::vector<double> L((size_t)d * d, 0.0);
    if (spec->proposal == WS_PROPOSAL_RW) {
        // RW: std = step_size per target (move_kernels.jl:189-212)
        for (int t = 0; t < d; ++t) L[t * d + t] = spec->step;
        // unbounded RW draws target-major (for each target N normals); bounded RW and autoRW draw
        // particle-major d x N (move_kernels.jl:200-202 vs :150,209)
        M.normals_target_major = spec->has_bounds ? 0 : 1;
    } else {
        // autoRW: lambda * weighted covariance of the (unconstrained) targets (move_kernels.jl:144-151)
        if (c->logw_uniform) {
            M.w_uniform = 1;
        } else {
            TRY(ensure_reduced(c));
            M.w_uniform = 0;
        }
        const int n_mom = 1 + d + d * (d + 1) / 2;
        const int grid = std::min(c->sm_count * 4, (int)((c->n + 255) / 256));
        TRY(ensure_scratch(c, sizeof(double) * (size_t)std::max(1, grid) * n_mom * 2));
        TRY(ensure_h_scratch(c, sizeof(double) * (size_t)std::max(1, grid) * n_mom * 2));
        M.logw = c->logw;
        M.red = c->d_red;
        // two passes (mean, then centred second moments), like StatsBase.cov
        std::vector<double> mean(d, 0.0), cov((size_t)d * d, 0.0);
        double wsum = 0.0;
        for (int pass = 0; pass < 2; ++pass) {
            for (int t = 0; t < d; ++t) M.mean[t] = mean[t];
            TimedEvent te;
            timed_begin(c, KC_MOVE, te);
            CK(c, ws_launch_move_moments(M, c->n, pass, c->d_scratch, std::max(1, grid), c->stream));
            timed_end(c, te);
            CK(c, cudaMemcpyAsync(c->h_scratch, c->d_scratch, sizeof(double) * (size_t)std::max(1, grid) * n_mom, cudaMemcpyDeviceToHost, c->stream));
            CK(c, cudaStreamSynchronize(c->stream));
            std::vector<double> tot(n_mom, 0.0);
            for (int b = 0; b < std::max(1, grid); ++b)
                for (int k = 0; k < n_mom; ++k) tot[k] += c->h_scratch[(size_t)b * n_mom + k];
            TRY(allreduce_host_doubles(c, tot.data(), n_mom));  // sharded: moments of the GLOBAL particle set
            if (pass == 0) {
                wsum = tot[0];
                for (int t = 0; t < d; ++t) mean[t] = tot[1 + t] / wsum;
            } else {
                int k = 1 + d;
                for (int i = 0; i < d; ++i)
                    for (int j = 0; j <= i; ++j) {
                        cov[i * d + j] = cov[j * d + i] = tot[k] / wsum;
                        ++k;
                    }
            }
        }
        const double lambda = 2.38 / sqrt((double)d);
        std::vector<double> S((size_t)d * d);
        for (int i = 0; i < d * d; ++i) {
            double v = cov[i];
            if (v == 0.0) v = spec->step;  // Sigma[Sigma .== 0] .= min_step
            S[i] = lambda * v;
        }
        if (!wsl::cholesky_lower(d, S.data(), L))
            return fail(c, WS_ENUMERIC, "autoRW: proposal covariance is not positive definite (rank-deficient particle cloud)");
        M.normals_target_major = 0;
    }
    for (int i = 0; i < d * d; ++i) M.L[i] = L[i];

    // random streams
    M.rng.seed = c->seed;
    M.rng.replay_n = c->d_replay_n;
    M.rng.replay_u = c->d_replay_u;
    M.rng.replay_e = nullptr;
    M.rng.replay_v = nullptr;
    M.stream_normals = c->next_stream;
    c->next_stream += (uint64_t)((d + 1) / 2);
    M.stream_uniform = c->next_stream++;
    M.replay_n_base = c->cur_n;
    M.replay_u_base = c->cur_u;
    M.n_global = c->n_global;
    if (c->d_replay_n != nullptr) {
        c->cur_n += c->n_global * d;
        if (c->cur_n > c->replay_n_len) return fail(c, WS_EREPLAY, "replay normals exhausted in Move");
    }
    if (c->d_replay_u != nullptr) {
        c->cur_u += c->n_global;
        if (c->cur_u > c->replay_u_len) return fail(c, WS_EREPLAY, "replay uniforms exhausted in Move");
    }

    CK(c, cudaMemsetAsync(c->d_counters + 2, 0, sizeof(unsigned long long), c->stream));
    M.n_accept = c->d_counters + 2;
    if (c->score_wide) {
        // propose -> (delta per tape segment) -> accept
        TRY(ensure_scratch(c, sizeof(double) * (size_t)c->n * (size_t)(d + 2)));
        double* x_new = c->d_scratch;
        double* lpr = x_new + (size_t)d * c->n;
        double* delta = lpr + c->n;
        M.score.n = c->n;
        M.score.particle_offset = c->offset;
        TimedEvent te;
        timed_begin(c, KC_MOVE, te);
        CK(c, ws_launch_move_propose(M, x_new, lpr, delta, c->sm_count, c->stream));
        timed_end(c, te);
        std::vector<Plane> targets;
        for (int t = 0; t < d; ++t) targets.push_back(Plane{spec->col[t], spec->comp[t]});
        TRY(for_each_tape_segment(c, target_depth, &targets, [&](Program& seg) -> int {
            fill_segment_launch(c, M.score, seg);
            for (int t = 0; t < d; ++t) {
                auto it = seg.plane_reg.find(targets[t]);
                M.target_reg[t] = (it == seg.plane_reg.end()) ? 0xFF : (uint8_t)it->second;
            }
            TimedEvent te2;
            timed_begin(c, KC_MOVE, te2);
            CK(c, ws_launch_move_delta(M, 1, x_new, delta, c->sm_count, c->stream));
            timed_end(c, te2);
            return WS_OK;
        }));
        M.score.n = c->n;
        M.score.particle_offset = c->offset;
        timed_begin(c, KC_MOVE, te);
        CK(c, ws_launch_move_accept(M, x_new, lpr, delta, c->sm_count, c->stream));
        timed_end(c, te);
    } else {
        const int n_ops = score_prefix_ops(c, target_depth);
        TRY(upload_score_program(c));
        TRY(fill_score_launch(c, M.score, n_ops));
        // Terms that do not involve a target cancel in s_new - s_old: fold only the entries that read a target
        // (plus the sigma-cache prologues later entries rely on), and load only the planes those read.
        {
            std::vector<WsOp> sel;
            std::vector<Plane> need;
            int begin = 0;
            for (auto& e : c->tape) {
                if (!(e.depth < target_depth)) break;
                const int b = begin, pe = b + e.cache_ops, en = e.op_end;
                begin = en;
                bool dep = false;
                for (auto& r : e.refs)
                    for (int t = 0; t < d; ++t)
                        if (r.col == spec->col[t] && r.comp == spec->comp[t]) dep = true;
                if (e.cache_ops > 0 || dep)
                    for (auto& r : e.refs) need.push_back(r);
                if (e.cache_ops > 0) sel.insert(sel.end(), c->score.ops.begin() + b, c->score.ops.begin() + pe);
                if (dep) sel.insert(sel.end(), c->score.ops.begin() + pe, c->score.ops.begin() + en);
            }
            if ((int)sel.size() < n_ops) {
                if (sel.size() > c->d_seg_cap) {
                    if (c->d_seg_ops) {
                        CK(c, cudaStreamSynchronize(c->stream));
                        CK(c, cudaFree(c->d_seg_ops));
                        c->d_seg_ops = nullptr;
                    }
                    c->d_seg_cap = std::max<size_t>(4096, sel.size() * 2);
                    CK(c, cudaMalloc(&c->d_seg_ops, sizeof(WsOp) * c->d_seg_cap));
                }
                if (!sel.empty()) {
                    CK(c, cudaMemcpyAsync(c->d_seg_ops, sel.data(), sizeof(WsOp) * sel.size(), cudaMemcpyHostToDevice, c->stream));
                    c->stats.h2d_bytes += (int64_t)(sizeof(WsOp) * sel.size());
                }
                M.score.ops = c->d_seg_ops;
                M.score.n_ops = (int)sel.size();
                int k2 = 0;
                for (int k = 0; k < (int)c->score.loads.size(); ++k) {
                    const Plane pl = c->score.loads[k].first;
                    if (std::find(need.begin(), need.end(), pl) == need.end()) continue;
                    M.score.load_ptr[k2] = plane_ptr(c, pl);
                    M.score.load_reg[k2] = (uint8_t)c->score.loads[k].second;
                    ++k2;
                }
                M.score.n_loads = k2;
                compact_score_regs(M.score, sel.data(), sel.size(), M.target_reg, d);
            } else {
                compact_score_regs(M.score, c->score.ops.data(), (size_t)n_ops, M.target_reg, d);
            }
        }
        TimedEvent te;
        timed_begin(c, KC_MOVE, te);
        CK(c, ws_launch_move(M, c->sm_count, c->stream));
        timed_end(c, te);
    }
    c->stats.moves_run++;
    if (info) {
        info->ran = 1;
        unsigned long long acc = 0;
        CK(c, cudaMemcpyAsync(&acc, c->d_counters + 2, sizeof(acc), cudaMemcpyDeviceToHost, c->stream));
        CK(c, cudaStreamSynchronize(c->stream));
        info->n_accepted = (int64_t)acc;
    }
    return WS_OK;
}

// ------------------------------------------------------------------------------------------
// instrumentation
// ------------------------------------------------------------------------------------------
extern "C" int ws_get_clamped(ws_ctx* c, int64_t* out) {
    if (!c || !out) return WS_EINVAL;
    unsigned long long h = 0;
    CK(c, cudaMemcpyAsync(&h, c->d_counters + 0, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    *out = (int64_t)h;
    return WS_OK;
}

extern "C" int ws_get_ess_ties(ws_ctx* c, int64_t* out) {
    if (!c || !out) return WS_EINVAL;
    TRY(flush_window(c));
    unsigned long long v = 0;
    CK(c, cudaMemcpyAsync(&v, c->d_counters + 3, sizeof(v), cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    *out = (int64_t)v;
    return WS_OK;
}
extern "C" int ws_get_stats(ws_ctx* c, ws_stats* out) {
    if (!c || !out) return WS_EINVAL;
    TRY(resolve_spec(c));
    resolve_events(c);
    c->stats.last_pass_ms = c->kc_ms[KC_VM];
    c->stats.last_resample_ms = c->kc_ms[KC_SCAN] + c->kc_ms[KC_GATHER];
    *out = c->stats;
    return WS_OK;
}
extern "C" int ws_kernel_times(ws_ctx* c, double* ms_out, int64_t* count_out, int32_t n_classes) {
    if (!c) return WS_EINVAL;
    resolve_events(c);
    for (int k = 0; k < n_classes && k < KC_COUNT; ++k) {
        if (ms_out) ms_out[k] = c->kc_ms[k];
        if (count_out) count_out[k] = c->kc_count[k];
    }
    return WS_OK;
}
extern "C" int ws_reset_kernel_times(ws_ctx* c) {
    if (!c) return WS_EINVAL;
    resolve_events(c);
    for (int k = 0; k < KC_COUNT; ++k) {
        c->kc_ms[k] = 0.0;
        c->kc_count[k] = 0;
    }
    return WS_OK;
}
extern "C" int ws_set_timing(ws_ctx* c, int on) {
    if (!c) return WS_EINVAL;
    resolve_events(c);
    c->timing = on != 0;
    return WS_OK;
}
extern "C" int ws_set_lazy_gather(ws_ctx* c, int on) {
    if (!c) return WS_EINVAL;
    TRY(flush_window(c));
    TRY(resolve_spec(c));
    TRY(materialize_planes(c));
    c->lazy_gather = on != 0;
    return WS_OK;
}
static int stats_allgather_words(void* ctx, const unsigned long long* in, size_t words, unsigned long long* out) {
    ws_ctx* c = (ws_ctx*)ctx;
    const size_t R = (size_t)c->nranks;
    TRY(ensure_scratch2(c, sizeof(unsigned long long) * words * (R + 1)));
    unsigned long long* d = (unsigned long long*)c->d_scratch2;
    CK(c, cudaMemcpyAsync(d + words * R, in, sizeof(unsigned long long) * words, cudaMemcpyHostToDevice, c->stream));
    NCK(c, g_nccl.AllGather(d + words * R, d, words, WS_NCCL_UINT64, c->comm, c->stream));
    CK(c, cudaMemcpyAsync(out, d, sizeof(unsigned long long) * words * R, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return WS_OK;
}
static int stats_allreduce_doubles(void* ctx, double* v, int n) {
    ws_ctx* c = (ws_ctx*)ctx;
    TRY(ensure_scratch2(c, sizeof(double) * (size_t)n));
    CK(c, cudaMemcpyAsync(c->d_scratch2, v, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
    NCK(c, g_nccl.AllReduce(c->d_scratch2, c->d_scratch2, (size_t)n, WS_NCCL_FLOAT64, WS_NCCL_SUM, c->comm, c->stream));
    CK(c, cudaMemcpyAsync(v, c->d_scratch2, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return WS_OK;
}
static int stats_allreduce_u64_device(void* ctx, unsigned long long* d, size_t n) {
    ws_ctx* c = (ws_ctx*)ctx;
    NCK(c, g_nccl.AllReduce(d, d, n, WS_NCCL_UINT64, WS_NCCL_SUM, c->comm, c->stream));
    return WS_OK;
}

extern "C" int ws_describe(ws_ctx* c, int32_t n_planes, const int32_t* col, const int32_t* comp, ws_plane_stats* out, double* ess) {
    if (!c || !col || !comp || !out || n_planes < 1) return c ? fail(c, WS_EINVAL, "ws_describe: bad arguments") : WS_EINVAL;
    for (int t = 0; t < n_planes; ++t) TRY(check_plane(c, col[t], comp[t]));
    TRY(ensure_reduced(c));  // flushes the window; (m, S, Q) of the current log-weights (global on a sharded state)
    WsStatsComm comm{c, c->nranks, stats_allgather_words, stats_allreduce_doubles, stats_allreduce_u64_device, c->rank};
    if (c->nranks > 1) {  // sharded states have no genealogy: bring the planes into the current particle order first
        std::vector<Plane> pl;
        for (int t = 0; t < n_planes; ++t) pl.push_back(Plane{col[t], comp[t]});
        TRY(materialize_planes(c, &pl));
    }
    CK(c, cudaSetDevice(c->device));
    static_assert(sizeof(ws_plane_stats) == sizeof(WsPlaneStats), "ws_plane_stats layout");
    const size_t sb = ws_stats_scratch_bytes(c->n);
    // scratch: [stats partials | q (8 n) | x through the genealogy (8 n)]
    const size_t q_off = (sb + 255) & ~(size_t)255;
    TRY(ensure_scratch(c, q_off + 16 * (size_t)c->n));
    TRY(ensure_h_scratch(c, sb));
    unsigned long long* d_q = (unsigned long long*)((char*)c->d_scratch + q_off);
    double* d_x = (double*)(d_q + c->n);
    CK(c, ws_stats_weights(c->logw, c->d_red, c->logw_uniform ? 1 : 0, c->n, c->n_global, d_q, c->stream));
    c->stats.kernel_launches++;
    for (int t = 0; t < n_planes; ++t) {
        const Column& cl = c->cols[col[t]];
        const double* x = cl.front[comp[t]];
        const int32_t* map = nullptr;
        if (cl.stale[comp[t]]) TRY(map_for_epoch(c, cl.ep[comp[t]], &map));
        if (map != nullptr) {
            WsGatherParams G;
            memset(&G, 0, sizeof(G));
            G.n = c->n;
            G.ancestors = map;
            G.n_planes = 1;
            G.src[0] = x;
            G.dst[0] = d_x;
            TimedEvent te;
            timed_begin(c, KC_GATHER, te);
            CK(c, ws_launch_gather(G, grid_for(c, c->n, 256, 8), c->stream));
            timed_end(c, te);
            x = d_x;
        }
        int launches = 0;
        WsPlaneStats ps;
        CK(c, ws_stats_plane(x, d_q, c->n, c->d_scratch, c->h_scratch, c->stream, &ps, &launches, c->nranks > 1 ? &comm : nullptr));
        c->stats.kernel_launches += launches;
        memcpy(&out[t], &ps, sizeof(ps));
    }
    if (ess) *ess = (double)c->n_global * c->h_red->ess_perc;
    return WS_OK;
}

extern "C" int ws_set_genealogy(ws_ctx* c, int on, int64_t budget_bytes) {
    if (!c) return WS_EINVAL;
    TRY(flush_window(c));
    if (!on) TRY(materialize_planes(c));
    c->genealogy = on != 0;
    if (budget_bytes > 0) c->genealogy_budget = (size_t)budget_bytes;
    return WS_OK;
}
extern "C" int ws_genealogy_info(ws_ctx* c, int64_t* n_vectors, int64_t* bytes, int64_t* events) {
    if (!c) return WS_EINVAL;
    if (n_vectors) *n_vectors = (int64_t)c->anc_live.size();
    if (bytes) *bytes = (int64_t)(c->anc_live.size() * sizeof(int32_t) * (size_t)(c->n + c->spare));
    if (events) *events = c->epoch;
    return WS_OK;
}
extern "C" int ws_col_events_behind(ws_ctx* c, int32_t id, int64_t* out) {
    if (!c || !out) return WS_EINVAL;
    if (id < 0 || id >= (int32_t)c->cols.size()) return fail(c, WS_EINVAL, "unknown column id %d", id);
    int64_t b = 0;
    for (int k = 0; k < c->cols[id].width; ++k)
        if (c->cols[id].stale[k]) b = std::max(b, c->epoch - c->cols[id].ep[k]);
    *out = b;
    return WS_OK;
}
extern "C" int ws_next_philox_stream(ws_ctx* c, uint64_t* stream_out, uint64_t* seed_out) {
    if (!c) return WS_EINVAL;
    if (stream_out) *stream_out = c->next_stream;
    if (seed_out) *seed_out = c->seed;
    return WS_OK;
}
extern "C" int ws_get_traced_pushes(ws_ctx* c, int64_t* out) {
    if (!c || !out) return WS_EINVAL;
    *out = c->traced_rows;
    return WS_OK;
}
extern "C" int ws_get_mailbox_exchanges(ws_ctx* c, int64_t* out) {
    if (!c || !out) return WS_EINVAL;
    *out = c->mbox_on ? c->mbox_exchanges : 0;
    return WS_OK;
}
extern "C" int ws_get_pushed(ws_ctx* c, int64_t* out) {
    if (!c || !out) return WS_EINVAL;
    *out = c->pushed_total;
    return WS_OK;
}
extern "C" int ws_get_migrated(ws_ctx* c, int64_t* out) {
    if (!c || !out) return WS_EINVAL;
    *out = c->migrated_total;
    return WS_OK;
}
extern "C" int ws_stream(ws_ctx* c, void** stream_out) {
    if (!c || !stream_out) return WS_EINVAL;
    *stream_out = (void*)c->stream;
    return WS_OK;
}
