/* wsb200.h — C ABI of the B200-native particle hot path behind WeightedSampling.jl's API.
 *
 * This is the drop-in boundary: everything `run!(model, state)` does per statement in the
 * reference (sample / weight / exp_norm + ESS / stratified resample / gather / MH move) is one
 * call below.  The reference is pure Julia (no FFI of its own), so each entry point cites the
 * Julia function whose `apply!` body / numeric helper it replaces; a Julia host binds them with
 * `ccall` (see INTEGRATION.md), and the Python host in `weightedsampling.jl_b200/` binds the
 * same symbols with ctypes.  All citations are into /root/reference.
 *
 * Conventions
 *   - every function returns 0 on success, a negative WS_E* code otherwise;
 *     `ws_last_error(ctx)` gives the message (Julia side: rethrow as ErrorException /
 *     ArgumentError, matching the reference's exceptions);
 *   - the caller owns host buffers, the library owns device buffers;
 *   - particle data are Float64 planes (struct of arrays): a column of width d is d planes of
 *     n doubles; host transfers are plane-major (`host[p*n + i]`);
 *   - ops are stream-ordered on the context's stream and FUSED: elementwise statements are
 *     queued and compiled into one device pass at the next flush point (resample, move,
 *     download, ws_flush).  Host-blocking happens only where a value is returned;
 *   - one host thread per context (the reference is single-threaded: TODO.md:28);
 *   - there is NO CPU fallback: without a CUDA device every call fails with WS_ENODEVICE.
 */
#ifndef WSB200_H
#define WSB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WSB200_ABI_VERSION 2

/* ---- status codes ---------------------------------------------------------------------- */
#define WS_OK 0
#define WS_EINVAL (-1)     /* bad argument (reference: ArgumentError / error(...))            */
#define WS_ENODEVICE (-2)  /* no CUDA device / driver                                        */
#define WS_ECUDA (-3)      /* CUDA runtime failure, message has the cudaError string         */
#define WS_ENOMEM (-4)     /* device allocation failed                                       */
#define WS_EUNSUPPORTED (-5) /* outside the fixed device-op set (rejected, never run on CPU) */
#define WS_EREPLAY (-6)    /* replay stream exhausted                                        */
#define WS_ENUMERIC (-7)   /* e.g. autoRW covariance not positive definite (TODO.md:4)       */
#define WS_ENCCL (-8)      /* NCCL failure                                                   */

typedef struct ws_ctx ws_ctx;

/* ---- resampling schemes ------------------------------------------------------------------
 * STRATIFIED is the reference's only scheme (src/resampling.jl:35-43).  SYSTEMATIC and
 * MULTINOMIAL are the two extra schemes BASELINE.json's microbenchmark names; they have no
 * reference implementation and follow SURVEY.md Appendix B.                                  */
#define WS_RESAMPLER_STRATIFIED 0
#define WS_RESAMPLER_SYSTEMATIC 1
#define WS_RESAMPLER_MULTINOMIAL 2

/* ---- expressions ---------------------------------------------------------------------------
 * Statement arguments are per-particle scalar expressions in postfix (RPN) form.  This is what
 * `vectorize` (src/rewrites.jl:146-219) produces as a fused broadcast in the reference; here the
 * host serialises the same expression tree as tokens and the runtime compiles it to device
 * micro-ops.  Anything that cannot be written with these tokens is outside the device-op set
 * and must be rejected by the host at model-construction time.                                */
enum ws_tok_op {
    WS_TOK_CONST = 0, /* push val                                   */
    WS_TOK_PLANE = 1, /* push column `col`, component `comp`        */
    WS_TOK_ADD = 2,
    WS_TOK_SUB = 3,
    WS_TOK_MUL = 4,
    WS_TOK_DIV = 5,
    WS_TOK_NEG = 6,
    WS_TOK_EXP = 7,
    WS_TOK_LOG = 8,
    WS_TOK_SQRT = 9,
    WS_TOK_SQUARE = 10,
    WS_TOK_SIN = 11,
    WS_TOK_COS = 12,
    WS_TOK_ABS = 13,
    WS_TOK_POW = 14, /* binary: base exponent                        */
    /* fresh standard variates, one per particle and token (only inside ws_sample_expr's sampler) */
    WS_TOK_RANDN = 15,
    WS_TOK_RANDU = 16,
    WS_TOK_RANDEXP = 17,
    /* comparisons give 1.0 / 0.0 (the device form of Bool columns); SELECT pops (cond, a, b) */
    WS_TOK_LT = 18,
    WS_TOK_LE = 19,
    WS_TOK_EQ = 20,
    WS_TOK_SELECT = 21,
    WS_TOK_MIN = 22,
    WS_TOK_MAX = 23,
    WS_TOK_NOT = 24, /* x == 0 ? 1 : 0 */
    WS_TOK_LGAMMA = 25,
    WS_TOK_LOG1P = 26,
    WS_TOK_EXPM1 = 27,
    WS_TOK_TAN = 28,
    WS_TOK_ATAN = 29,
    WS_TOK_TANH = 30,
    WS_TOK_FLOOR = 31,
    /* variates with a parameter (unary: pop the parameter, push the draw), sampler expressions only:
     * standard Gamma(shape) (Marsaglia-Tsang) and Poisson(rate) (inversion / PTRS) — the building blocks of the
     * reference's Gamma, Beta, TDist, Chisq, InverseGamma, Poisson kernels (src/default_kernels.jl:83-102) */
    WS_TOK_RANDGAMMA = 32,
    WS_TOK_RANDPOISSON = 33,
    /* a constant supplied later: only inside the expressions of a ws_exec command list, where it is replaced by
     * params[col] before the statement is issued */
    WS_TOK_PARAM = 34,
    /* build-time constant tables (ws_table below); `col` is the table id, the operands are popped:
     * TABLE pops (row, column) and pushes T[row, column]; comp = 1 pushes log T[row, column] instead, with a column
     * outside 1..n_cols giving -Inf without a fault (the log-probability of a Categorical value).
     * RANDCAT pops the row and pushes a draw of Categorical(T[row, :]) (sampler expressions only). */
    WS_TOK_TABLE = 35,
    WS_TOK_RANDCAT = 36
};

typedef struct ws_tok {
    int32_t op;   /* enum ws_tok_op */
    int32_t col;  /* WS_TOK_PLANE: column id from ws_col_ensure / ws_col_lookup */
    int32_t comp; /* WS_TOK_PLANE: component (plane) inside the column, 0-based */
    int32_t reserved;
    double val; /* WS_TOK_CONST */
} ws_tok;

typedef struct ws_expr {
    const ws_tok* toks;
    int32_t n;
    int32_t reserved;
} ws_expr;

/* ---- build-time constant tables ------------------------------------------------------------
 * `vectorize` broadcasts `mu[s]` / `P[s, k]` like any getindex (src/rewrites.jl:146-219); here a Julia array that is a
 * build-time constant and is indexed by a particle value becomes a table:
 *   - A table is an n_rows x n_cols array of Float64, row-major; a vector is one row.  ws_table uploads it once per
 *     context (deduplicated by content: the same values give the same id) and ws_destroy frees it.  Rows longer than
 *     2^16 entries are WS_EUNSUPPORTED.
 *   - Indices are Julia values, so 1-based: an index must be an integer-valued double in [1, n].  Any other index
 *     (non-integer, out of range, NaN) gives NaN and never reads outside the table, and each such read adds one to
 *     a sticky device counter of the context (ws_get_index_faults).  The reference throws BoundsError at the
 *     statement; a host checks the counter when a run ends (DESIGN.md §7).
 *   - Categorical(p), p a row of a table (a constant vector is a one-row table), with C_k = p_1 + ... + p_k summed
 *     sequentially in Float64 on the host: the draw at one uniform u per particle (Philox, or the replayed uniform
 *     stream, one per particle and draw in statement order, as for Uniform) is x = 1 + #{k < K : C_k <= u}:
 *     Distributions 0.25's `while cp <= draw && i < n` walk over DiscreteNonParametric, found by a binary search.
 *     logpdf(x) = log p_x for integer x in 1..K (log 0 = -Inf), -Inf for any other x.  Whether p is a probability
 *     vector is the host's check (the Python front-end raises ValueError when the model is built).                */
int ws_table(ws_ctx* ctx, const double* values, int64_t n_rows, int32_t n_cols, int32_t* id_out);
/* out-of-range / non-integer / NaN table indices met so far by this context's kernels (flushes and waits) */
int ws_get_index_faults(ws_ctx* ctx, int64_t* out);

/* ---- lifecycle ---------------------------------------------------------------------------
 * SMCState(n; ess_perc_min = 0.5)  (src/types.jl:48-78): creates the device-resident state:
 * log-weights (zeros), flags resampled = weights_changed = false, depth = 0, empty store.   */
int ws_create(ws_ctx** out, int64_t n_particles, int device, uint64_t seed, double ess_perc_min,
              int resampler);
/* Sharded state: this rank owns global particle slots [rank*n/nranks, (rank+1)*n/nranks).
 * `nccl_unique_id` is the 128-byte ncclUniqueId created by rank 0 and distributed by the host
 * (torch.distributed / MPI / Julia Distributed); NULL with nranks == 1.                       */
int ws_create_sharded(ws_ctx** out, int64_t n_particles_global, int rank, int nranks,
                      const void* nccl_unique_id, int device, uint64_t seed, double ess_perc_min,
                      int resampler);
int ws_nccl_unique_id(void* out128);
int ws_destroy(ws_ctx* ctx);
const char* ws_last_error(const ws_ctx* ctx); /* ctx may be NULL: error of the last failed create */
int ws_abi_version(void);
int ws_device_count(int* out);
int ws_sync(ws_ctx* ctx);  /* flush the fusion queue and wait for the stream */
int ws_flush(ws_ctx* ctx); /* flush the fusion queue, do not wait            */

/* ---- state scalars (src/types.jl:48-60) ---------------------------------------------------- */
int ws_n_particles(const ws_ctx* ctx, int64_t* n_local, int64_t* n_global);
int ws_get_flags(ws_ctx* ctx, int* resampled, int* weights_changed, int64_t* depth);
int ws_set_flags(ws_ctx* ctx, int resampled, int weights_changed);
int ws_set_depth(ws_ctx* ctx, int64_t depth);
int ws_set_ess_perc_min(ws_ctx* ctx, double ess_perc_min);
int ws_get_ess_perc_min(const ws_ctx* ctx, double* out);
/* run!(root, state) prologue (src/types.jl:120-126): depth = 0 and the score tape restarts.  */
int ws_begin_run(ws_ctx* ctx);

/* ---- particle store (src/stores.jl:28-35, 70-111) ------------------------------------------
 * ColumnStore: named columns, created on first write, ping-pong front/back planes.           */
int ws_col_ensure(ws_ctx* ctx, const char* name, int32_t width, int32_t* id_out);
int ws_col_lookup(const ws_ctx* ctx, const char* name, int32_t* id_out, int32_t* width_out);
int ws_col_count(const ws_ctx* ctx, int32_t* out);
int ws_col_info(const ws_ctx* ctx, int32_t id, char* name_buf, int32_t name_buf_len, int32_t* width_out);
/* getcol(store, name) (src/stores.jl:82): host copy, plane-major, local shard.               */
int ws_col_download(ws_ctx* ctx, int32_t id, double* host_out);
int ws_col_upload(ws_ctx* ctx, int32_t id, const double* host_in);
int ws_weights_download(ws_ctx* ctx, double* host_out); /* state.weights */
int ws_weights_upload(ws_ctx* ctx, const double* host_in, int mark_changed);
/* resample!(store, indices) (src/stores.jl:105-121) with caller-supplied 0-based ancestors.   */
int ws_gather(ws_ctx* ctx, const int32_t* ancestors_host);
int ws_ancestors_download(ws_ctx* ctx, int32_t* host_out); /* ancestors of the last firing resample, 0-based */

/* ---- statements ----------------------------------------------------------------------------
 * Each counted statement advances `depth` by one exactly like advance!(state)
 * (src/types.jl:162-166) and, for Sample/Observe/Weight, appends its log-density to the score
 * tape that ws_move folds (the device form of score!; src/transformers.jl:39,77,139,193,243,297). */

/* Assign.apply! / AccessorAssign.apply!  `x .= expr`, `x[j] .= expr`
 * (src/transformers.jl:28-32, 67-71; src/stores.jl:85-96). */
int ws_assign(ws_ctx* ctx, int32_t col, int32_t comp, const ws_expr* rhs);
/* Same for a whole width-d column (one expression per component), e.g. `x .= [0.0, 0.0]`. */
int ws_assign_vec(ws_ctx* ctx, int32_t col, int32_t d, const ws_expr* rhs);

/* Sample.apply! / AccessorSample.apply! with the default kernels
 * (src/transformers.jl:118-131,172-182; src/default_kernels.jl:87,93,94). */
int ws_sample_normal(ws_ctx* ctx, int32_t col, int32_t comp, const ws_expr* mu, const ws_expr* sigma);
int ws_sample_exponential(ws_ctx* ctx, int32_t col, int32_t comp, const ws_expr* theta);
/* MvNormal(mu, Sigma): mu is d per-particle expressions, Sigma a constant d x d covariance
 * (row-major); the lower Cholesky factor is taken once on the host. */
int ws_sample_mvnormal(ws_ctx* ctx, int32_t col, int32_t d, const ws_expr* mu, const double* cov);

/* Observe.apply! / Weight.apply!: weights .+= logpdf.(D(args...), obs); weights_changed = true
 * (src/transformers.jl:228-235, 283-289). */
int ws_observe_normal(ws_ctx* ctx, const ws_expr* obs, const ws_expr* mu, const ws_expr* sigma);
int ws_observe_exponential(ws_ctx* ctx, const ws_expr* obs, const ws_expr* theta);
int ws_observe_mvnormal(ws_ctx* ctx, int32_t d, const ws_expr* obs, const ws_expr* mu, const double* cov);
/* Weight with an arbitrary log-weight expression: weights .+= expr. */
int ws_weight_expr(ws_ctx* ctx, const ws_expr* logw_term);
/* importance_kernel(Normal(pm,ps), Normal(tm,ts)) as a Sample with weighter
 * (src/default_kernels.jl:69-73): draw from the proposal, add logpdf(target)-logpdf(proposal)
 * to the weights, score with the target's logpdf. */
int ws_sample_importance_normal(ws_ctx* ctx, int32_t col, int32_t comp, double prop_mu, double prop_sigma,
                                double targ_mu, double targ_sigma);

/* A WeightedKernel(sampler, weighter, logpdf) whose three parts are device expressions
 * (src/types.jl:226-230; src/transformers.jl:172-182):  x = sampler(args...) with WS_TOK_RAND* variates,
 * weights += weighter(args..., x) (NULL: uniform weights), and logpdf(args..., x) is what score! adds
 * (NULL: the statement is not scored).  weighter / logpdf read x through WS_TOK_PLANE (col, comp). */
int ws_sample_expr(ws_ctx* ctx, int32_t col, int32_t comp, const ws_expr* sampler, const ws_expr* weighter,
                   const ws_expr* logpdf);

/* ---- statement lists -----------------------------------------------------------------------
 * Loop.apply! (src/transformers.jl:378-383) rebuilds and applies the loop body once per element; in a filter the
 * bodies differ only in constants (the observation).  A host can describe the body ONCE as a list of the statement
 * calls above, with WS_TOK_PARAM tokens where the element's values go, and replay it per element with one call:
 * ws_exec substitutes params[] and issues the statements exactly as the individual calls would (same fusion, same
 * depth and tape bookkeeping, same results).  `i0, i1` are the call's integer arguments in order, `e[k]` its
 * expression arguments in order with `n_e[k]` expressions behind each (0: the argument is NULL), `mat` the constant
 * covariance of the MvNormal calls. */
enum ws_cmd_fn {
    WS_CMD_ASSIGN = 0,            /* ws_assign(i0 = col, i1 = comp, e[0])                         */
    WS_CMD_ASSIGN_VEC = 1,        /* ws_assign_vec(i0 = col, i1 = d, e[0][d])                     */
    WS_CMD_SAMPLE_NORMAL = 2,     /* ws_sample_normal(i0 = col, i1 = comp, e[0], e[1])            */
    WS_CMD_SAMPLE_EXPONENTIAL = 3,/* ws_sample_exponential(i0 = col, i1 = comp, e[0])             */
    WS_CMD_SAMPLE_MVNORMAL = 4,   /* ws_sample_mvnormal(i0 = col, i1 = d, e[0][d], mat)           */
    WS_CMD_OBSERVE_NORMAL = 5,    /* ws_observe_normal(e[0], e[1], e[2])                          */
    WS_CMD_OBSERVE_EXPONENTIAL = 6,/* ws_observe_exponential(e[0], e[1])                          */
    WS_CMD_OBSERVE_MVNORMAL = 7,  /* ws_observe_mvnormal(i0 = d, e[0][d], e[1][d], mat)           */
    WS_CMD_WEIGHT_EXPR = 8,       /* ws_weight_expr(e[0])                                         */
    WS_CMD_SAMPLE_EXPR = 9,       /* ws_sample_expr(i0 = col, i1 = comp, e[0], e[1] | NULL, e[2] | NULL) */
    WS_CMD_RESAMPLE = 10          /* ws_resample_async()                                          */
};
typedef struct ws_cmd {
    int32_t fn; /* enum ws_cmd_fn */
    int32_t i0, i1;
    int32_t n_e[3];
    const ws_expr* e[3];
    const double* mat;
} ws_cmd;
int ws_exec(ws_ctx* ctx, const ws_cmd* cmds, int32_t n_cmds, const double* params, int32_t n_params);
/* ws_exec once per element for n_elems consecutive loop elements (params[e][n_params]): the host's loop over a block of
 * elements moved behind the boundary (one foreign call instead of n_elems). */
int ws_exec_n(ws_ctx* ctx, const ws_cmd* cmds, int32_t n_cmds, const double* params, int32_t n_params, int32_t n_elems);
/* The same list run for up to n_steps consecutive loop elements (params[step][n_params]) as ONE device pass, for
 * bodies of the form "weighting statements, Resample(), if resampled ... end" (examples/linear_regression.jl:20-26:
 * the reference's Resample.apply!, src/transformers.jl:474-498, needs the ESS after every observation, i.e. one pass
 * and one host round trip per statement).  The pass records the (m, S, Q) of the log-weights after each step; if no
 * step's ESS falls below the threshold all of them are done (*n_done = steps issued — possibly fewer than n_steps, a
 * pass holds a bounded number — *fired = 0); otherwise the steps behind the first firing one are rolled back, that
 * step's Resample runs as ws_resample would have, and *n_done counts the steps up to and including it, *fired = 1:
 * the caller applies the `if resampled` body and goes on with the next element.  Log-weights, tape, depth and Philox
 * stream numbering are those of the statement-by-statement run; the (m, S, Q) sums are grouped differently, so an
 * ESS within an ulp of the threshold may decide differently (as between any two kernel shapes; ws_get_ess_ties).
 * WS_EUNSUPPORTED (nothing changed): sharded or replayed states, statements that write columns or draw variates. */
int ws_exec_spec(ws_ctx* ctx, const ws_cmd* cmds, int32_t n_cmds, const double* params, int32_t n_params, int32_t n_steps,
                 int32_t* n_done, int32_t* fired);

/* Resample.apply! (src/transformers.jl:474-498) — the exact state machine:
 * no-op if !weights_changed; else exp_norm -> ess_perc -> if ess < ess_perc_min: stratified
 * ancestors, gather every column, weights .= logsumexp - log N, resampled = true; else
 * resampled = false; weights_changed = false.  Outputs may be NULL.
 * `fired` = 0 when the call was a no-op because nothing was weighted.                         */
typedef struct ws_resample_info {
    int32_t fired;      /* weights_changed was set                                   */
    int32_t resampled;  /* state.resampled after the call                             */
    double ess_perc;    /* ESS / N computed by this call (NaN if !fired)              */
    double log_mean_w;  /* logsumexp(weights) - log N at the time of the call        */
    int64_t n_clamped;  /* slots whose uniform exceeded the last CDF entry (reference would throw BoundsError; SURVEY §7) */
} ws_resample_info;
int ws_resample(ws_ctx* ctx, ws_resample_info* info);
/* The same step without waiting for its outcome: what depends on the decision (CDF, ancestor search, the weight
 * reset) runs on the device behind the decision flag, the host only queues it.  `state.resampled` (ws_get_flags with
 * a non-NULL `resampled`), ws_get_stats, ws_last_resample and every call that reads the log-weights wait for the
 * pending steps first; a model without `if resampled` never does.  Falls back to ws_resample(ctx, NULL) for replayed
 * uniforms, sharded states, multinomial resampling and eager gather.  Results are identical to ws_resample's.
 * (transformers.jl:474-498; env WSB200_ASYNC_RESAMPLE=0 disables it) */
int ws_resample_async(ws_ctx* ctx);
/* outcome of the most recent ws_resample / ws_resample_async (waits for it if it is still pending) */
int ws_last_resample(ws_ctx* ctx, ws_resample_info* info);

/* ---- resampling numerics on their own (src/resampling.jl) -------------------------------- */
/* exp_norm(state.weights) -> host (src/resampling.jl:72-77). */
int ws_exp_norm(ws_ctx* ctx, double* host_out);
/* log_evidence(state) = logsumexp(weights) - log N (src/utils.jl:21); also returns ess_perc. */
int ws_log_evidence(ws_ctx* ctx, double* log_evidence, double* ess_perc);
/* Pure functions on caller arrays of length n (any n; independent of the state's particles):
 *   ws_exp_norm_host      exp_norm(logw)                     src/resampling.jl:72-77
 *   ws_logsumexp_host     logsumexp(logw)                    src/resampling.jl:61-64
 *   ws_ess_perc_host      ess_perc(w)                        src/resampling.jl:51-54
 *   ws_icdf_host          icdf(weights, us) 0-based          src/resampling.jl:13-26
 *   ws_resample_host      stratified_resample(weights) etc.  src/resampling.jl:35-43
 * `uniforms` for ws_resample_host: n values (stratified), 1 value (systematic), n values
 * (multinomial, sorted by the library), or NULL to draw them from Philox.                    */
int ws_exp_norm_host(ws_ctx* ctx, const double* logw, int64_t n, double* w_out);
int ws_logsumexp_host(ws_ctx* ctx, const double* logw, int64_t n, double* out);
int ws_ess_perc_host(ws_ctx* ctx, const double* w, int64_t n, double* out);
int ws_icdf_host(ws_ctx* ctx, const double* weights, const double* us, int64_t n, int32_t* indices_out,
                 int64_t* n_clamped);
int ws_resample_host(ws_ctx* ctx, const double* weights, int64_t n, int scheme, const double* uniforms,
                     int32_t* indices_out, int64_t* n_clamped);

/* ---- analysis (src/utils.jl) ------------------------------------------------------------- */
/* @E(f, state) / expectation(values, weights): sum_i f_i * exp_norm(weights)_i
 * (src/utils.jl:11,45-68).  n_exprs expectations in one pass. */
int ws_expectation(ws_ctx* ctx, const ws_expr* f, int32_t n_exprs, double* out);
/* sample(state, n; replace) index draw (src/utils.jl:102-118): n 0-based GLOBAL particle indices drawn with
 * probability exp_norm(weights), made on the device.  On one GPU global and local indices are the same.  Collective on
 * a sharded state: every rank calls it and gets the same n indices.  The draw does not depend on the number of GPUs:
 * l_i is the current log-weight of global particle i, m = max_i l_i (exact in any reduction order), and the Philox
 * stream is the context's next stream (one per call, so the ranks stay in lockstep).
 *   With replacement:  q_i = rint(exp(l_i - m) 2^52) (0 for NaN or -inf l_i),  Q_j = sum_{i<=j} q_i and T = Q_{N-1}
 *     in exact integers (128-bit);  r_k = the 128-bit integer of Philox block (k, stream, seed),
 *     t_k = floor(r_k T / 2^128),  index_k = min{ j : Q_j > t_k }.  Every draw lands on a particle with q_j > 0.
 *     A particle whose weight is below 2^-53 of the largest is never drawn.
 *   Without replacement (n <= N):  key_i = l_i - log(E_i), E_i the standard exponential of Philox block
 *     (i, stream, seed) (ws_randexp).  The n largest keys in descending order, equal keys to the lower index;
 *     particles with a NaN or -inf log-weight rank below every finite key, ordered by index.
 * WS_ENUMERIC if the largest log-weight is not finite (all -inf or NaN, or +inf); WS_EINVAL for n <= 0 and for
 * n > N without replacement.  Only the n draws cross PCIe.  (csrc/ws_math.cuh: ws_sample_q, ws_sample_target,
 * ws_sample_key; csrc/ws_kernels_stats.cu) */
int ws_sample_indices(ws_ctx* ctx, int64_t n_draws, int replace, int64_t* indices_out);
/* rows `indices` of column id -> host (plane-major, n_idx per plane). */
int ws_col_download_rows(ws_ctx* ctx, int32_t id, const int64_t* indices, int64_t n_idx, double* host_out);
/* rows of GLOBAL particle indices (0 <= index < N) of column id -> host (plane-major, n_idx per plane).  Collective on
 * a sharded state: each rank reads the rows it owns and every rank gets all n_idx rows, bit for bit.  On one GPU the
 * same as ws_col_download_rows. */
int ws_col_download_global_rows(ws_ctx* ctx, int32_t id, const int64_t* global_indices, int64_t n_idx, double* host_out);

/* ---- MH moves (src/transformers.jl:588-623, src/move_kernels.jl:189-253) ------------------ */
#define WS_PROPOSAL_RW 0
#define WS_PROPOSAL_AUTORW 1
typedef struct ws_move_spec {
    int32_t n_targets;      /* d                                                        */
    const int32_t* col;     /* target planes: column ids ...                            */
    const int32_t* comp;    /* ... and components                                       */
    int32_t proposal;       /* WS_PROPOSAL_RW | WS_PROPOSAL_AUTORW                      */
    int32_t has_bounds;     /* 0: bounds === nothing                                    */
    const double* lo;       /* d lower bounds (-Inf = none), when has_bounds            */
    const double* hi;       /* d upper bounds (+Inf = none), when has_bounds            */
    double step;            /* RW: step_size (a standard deviation); autoRW: min_step   */
    double diversity;       /* diversity threshold, NaN = nothing (always move)         */
    int64_t target_depth;   /* score cut-off; -1 = state.depth (what Move.apply! uses)  */
} ws_move_spec;
typedef struct ws_move_info {
    int32_t ran;            /* 0: skipped by the diversity gate                         */
    int32_t reserved;
    double diversity;       /* marginal_diversity (NaN if not computed)                 */
    int64_t n_accepted;     /* accepted proposals on this rank                          */
} ws_move_info;
int ws_move(ws_ctx* ctx, const ws_move_spec* spec, ws_move_info* info);
/* marginal_diversity(store, targets) (src/transformers.jl:560-565). */
int ws_marginal_diversity(ws_ctx* ctx, int32_t n_targets, const int32_t* col, const int32_t* comp, double* out);
/* score_logpdf(state, targets, target_depth) (src/types.jl:183-206): fold of the recorded tape
 * entries with depth < target_depth, into a host vector. */
int ws_score_logpdf(ws_ctx* ctx, int64_t target_depth, double* host_out);
/* Explicit tape control for hosts that re-walk their own program tree (score! fold):
 * ws_tape_clear drops the recorded tape; statements executed between ws_tape_record_only(1)
 * and ws_tape_record_only(0) are appended to the tape WITHOUT being executed. */
int ws_tape_clear(ws_ctx* ctx);
int ws_tape_record_only(ws_ctx* ctx, int on);
int ws_tape_length(const ws_ctx* ctx, int64_t* n_entries);
/* Models without `<<` never fold the tape: a host that knows this (the @model front-end does)
 * switches recording off so that long filters do not accumulate one entry per statement. */
int ws_tape_enable(ws_ctx* ctx, int on);

/* ---- replay hooks (parity tests; SURVEY §8c "stream consumption order") --------------------
 * When a replay buffer is installed, every draw of that kind is taken from it in the
 * reference's consumption order instead of from Philox; running past the end is WS_EREPLAY.
 * Passing NULL/0 removes the buffer. */
int ws_set_replay_normals(ws_ctx* ctx, const double* host, int64_t len);
int ws_set_replay_uniforms(ws_ctx* ctx, const double* host, int64_t len);
int ws_set_replay_exponentials(ws_ctx* ctx, const double* host, int64_t len);
/* already-accepted variates of WS_TOK_RANDGAMMA / WS_TOK_RANDPOISSON draws (one per particle and draw, in statement
 * order): standard Gamma(a_i) / Poisson(lam_i) values produced by the caller with the particle's own parameter */
int ws_set_replay_variates(ws_ctx* ctx, const double* host, int64_t len);

/* ---- instrumentation ---------------------------------------------------------------------- */
typedef struct ws_stats {
    int64_t kernel_launches;   /* kernels of this library launched so far                */
    int64_t fused_passes;      /* elementwise fusion windows flushed                     */
    int64_t fused_statements;  /* statements that went into them                         */
    int64_t resamples_fired;   /* Resample calls that had weights_changed                */
    int64_t resamples_done;    /* ... of which actually resampled                        */
    int64_t moves_run;
    int64_t h2d_bytes;
    int64_t d2h_bytes;
    double last_resample_ms;   /* device time of the last scan+gather (CUDA events), when timing is on */
    double last_pass_ms;       /* device time of the last fused elementwise pass                     */
    int64_t sl_passes;         /* ... fusion windows that ran on a straight-line executor (csrc/ws_vm_sl.cuh)  */
} ws_stats;
int ws_get_stats(ws_ctx* ctx, ws_stats* out);
/* cumulative number of output slots whose uniform lay beyond the last CDF entry (clamped to the
 * last particle; the reference's icdf would throw BoundsError there, SURVEY.md §7) */
int ws_get_clamped(ws_ctx* ctx, int64_t* out);
/* Resample steps whose ESS% equalled ess_perc_min to within 8 ulp.  The reference computes 1 / (N sum w^2)
 * (src/resampling.jl:51-54, src/transformers.jl:484), the device S^2 / (N Q): for such a step (exactly equal weights
 * with ess_perc_min = 1.0 is the one that occurs) the two can fall on different sides of the threshold, so whether it
 * fires is rounding noise in both; the count makes the deviation visible. */
int ws_get_ess_ties(ws_ctx* ctx, int64_t* out);
/* per kernel class device time (ms, CUDA events on the context's stream; needs ws_set_timing(1)) and
 * launch counts.  Classes: 0 fused elementwise pass, 1 stand-alone reduce, 2 finalize, 3 scan+search,
 * 4 gather, 5 fill, 6 MH / score, 7 other. */
#define WS_N_KERNEL_CLASSES 8
int ws_kernel_times(ws_ctx* ctx, double* ms_out, int64_t* count_out, int32_t n_classes);
int ws_reset_kernel_times(ws_ctx* ctx);
/* resample!(store, indices) is deferred by default: after a resampling step each plane is gathered
 * through the ancestors by the next kernel that reads it (and never, if it is overwritten first).
 * on = 0 restores the reference's eager gather of every column inside ws_resample (stores.jl:105-111);
 * results are identical either way. */
int ws_set_lazy_gather(ws_ctx* ctx, int on);
/* describe(state) (src/utils.jl:183-289) for one plane: weighted mean, StatsBase weighted median
 * (quantile(v, Weights(w), 0.5): sort by (value, weight), h = (wsum - w1)/2 + w1, first k with S_k > h,
 * linear interpolation from the previous element), uncorrected weighted std, min, max and the weights of the
 * 8 equal-width bins of [min, max]; weights are exp_norm(state.weights).  The median is found on the device
 * by an 8-pass radix select over fixed-point weight histograms (no sort, nothing but the 13 numbers comes
 * back).  Any NaN in the plane makes mean / median / std / min / max NaN, as in the reference. */
typedef struct ws_plane_stats {
    double mean, median, std, min, max;
    double hist[8];
} ws_plane_stats;
int ws_describe(ws_ctx* ctx, int32_t n_planes, const int32_t* col, const int32_t* comp, ws_plane_stats* out, double* ess);

/* Genealogy (SURVEY.md §8f.2).  The reference's resample! gathers EVERY column at every resampling step
 * (src/stores.jl:105-121), so a model that keeps its history (x{t}, examples/1D_ssm.jl, 2D_ssm.jl) pays
 * O(t) per step.  Here a plane that is not read keeps the order of the event after which it was written;
 * the per-event ancestor vectors (4 B per particle and event) are kept instead, and a read composes them
 * (one dependent 4-byte load per event).  on = 0: gather stale planes at the next event, as before.
 * budget_bytes > 0: retained ancestor vectors above this are released by gathering the oldest planes
 * (default: a quarter of the device memory; WSB200_GENEALOGY_BYTES).  Single-GPU states only. */
int ws_set_genealogy(ws_ctx* ctx, int on, int64_t budget_bytes);
/* retained ancestor vectors, their bytes, and the number of resampling events so far */
int ws_genealogy_info(ws_ctx* ctx, int64_t* n_vectors, int64_t* bytes, int64_t* events);
/* how many resampling events a column's oldest plane is behind (0: stored in the current order) */
int ws_col_events_behind(ws_ctx* ctx, int32_t id, int64_t* out);
int ws_set_timing(ws_ctx* ctx, int on); /* record per-phase CUDA events (adds syncs; for profiling only) */
/* sharded state: particles this rank has received from other ranks in all resampling steps so far */
int ws_get_migrated(ws_ctx* ctx, int64_t* out);
/* offspring this rank has written DIRECTLY into other ranks' planes over NVLink (peer mappings; the exchange falls back to
 * stage + ncclSend / ncclRecv with WSB200_EXCHANGE=nccl or when ranks share a process) */
int ws_get_pushed(ws_ctx* ctx, int64_t* out);
/* small exchanges of sharded steps ((m, S, Q) triples, masses, slot bounds, barriers) that the kernels made themselves by
 * storing into the other ranks' mailboxes over NVLink instead of going through an NCCL collective (0: ranks share a
 * process, no peer mappings, or WSB200_MAILBOX=0) */
int ws_get_mailbox_exchanges(ws_ctx* ctx, int64_t* out);
/* sharded genealogy: values (offspring x planes) this rank pushed to other ranks for planes that were one or more resampling
 * events behind, found by tracing the migrating offspring through the retained ancestor vectors (src/stores.jl:105-121
 * gathers every column at every event instead) */
int ws_get_traced_pushes(ws_ctx* ctx, int64_t* out);
/* the Philox stream id the next random statement / resample will use, and the key (tests reproduce draws) */
int ws_next_philox_stream(ws_ctx* ctx, uint64_t* stream_out, uint64_t* seed_out);
/* raw cudaStream_t of the context (as void*), so a host can bracket calls with its own events */
int ws_stream(ws_ctx* ctx, void** stream_out);

#ifdef __cplusplus
}
#endif
#endif /* WSB200_H */
