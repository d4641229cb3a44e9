// ws_lowering.h — host-side lowering of statements to device micro-ops (the "fixed set of device
// ops" the @model front-end targets).  Header-only and CUDA-free so that tests can compile it
// with g++ and check the generated programs against the oracle on the CPU.
//
// What is lowered (reference semantics in parentheses):
//   assign            Assign.apply! / AccessorAssign.apply!   (src/transformers.jl:28-32, 67-71)
//   sample_*          Sample.apply! / AccessorSample.apply!   (src/transformers.jl:118-131, 172-182)
//   observe_* / weight Observe.apply! / Weight.apply!          (src/transformers.jl:228-235, 283-289)
// Expressions arrive as postfix tokens (include/wsb200.h: ws_tok), i.e. the serialised form of the
// fused broadcast that `vectorize` builds (src/rewrites.jl:146-219).
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>
#include <map>
#include <string>
#include <utility>
#include <vector>
#include "../../include/wsb200.h"
#include "ws_vm.cuh"

namespace wsl {

struct Plane {
    int32_t col, comp;
    bool operator<(const Plane& o) const { return col < o.col || (col == o.col && comp < o.comp); }
    bool operator==(const Plane& o) const { return col == o.col && comp == o.comp; }
};

// A value on the expression stack: either a constant or the unmaterialised affine form
// c0 + c1 * r[reg].  Keeping the affine form symbolic lets `a*x`, `x + v`, `alpha + beta*x`
// collapse into a single LIN2 micro-op.
struct Val {
    bool is_const;
    double c0, c1;
    int reg;
    static Val constant(double v) { return Val{true, v, 0.0, -1}; }
    static Val lin(double c0, double c1, int reg) { return Val{false, c0, c1, reg}; }
    bool pure() const { return !is_const && c0 == 0.0 && c1 == 1.0; }
};

struct RngCursor {
    uint64_t* stream;     // next Philox stream id
    int64_t* normals;     // replay cursors (elements consumed so far)
    int64_t* uniforms;
    int64_t* exponentials;
    int64_t n_global;     // particles (global): one statement consumes n_global * d variates
    int64_t* variates = nullptr;  // replay cursor of the WS_OP_RANDV ops (accepted Gamma / Poisson variates)
};

// A build-time constant table as the lowering sees it (include/wsb200.h: ws_table): the addresses of its values, of
// their logarithms and of its row-wise sequential partial sums, each array behind its own WsTableHdr.  Device
// addresses in the runtime, host addresses in tests/host/.
struct TableRef {
    uint64_t values, logv, cdf;
    int64_t n_rows;
    int32_t n_cols;
};

// The memory image of a table (ws_table): three arrays, each [WsTableHdr | n_rows * n_cols doubles] — the values, their
// logarithms, and the sequential Float64 partial sums of each row (cp += p[i], the order Distributions sums in).  The
// runtime uploads it as it is; tests/host/ uses it in place.  TableRef addresses point at image + table_offset(k).
inline size_t table_segment(int64_t n_rows, int32_t n_cols) { return 2 + (size_t)n_rows * (size_t)n_cols; }
inline std::vector<double> table_image(const double* values, int64_t n_rows, int32_t n_cols) {
    static_assert(sizeof(WsTableHdr) == 2 * sizeof(double), "a table header is two doubles");
    const size_t seg = table_segment(n_rows, n_cols), ne = seg - 2;
    std::vector<double> h(3 * seg, 0.0);
    for (int k = 0; k < 3; ++k) {
        const WsTableHdr hdr{0ull, n_rows};
        memcpy(&h[k * seg], &hdr, sizeof hdr);
    }
    double* hv = &h[2];
    double* hl = &h[seg + 2];
    double* hc = &h[2 * seg + 2];
    for (size_t i = 0; i < ne; ++i) {
        hv[i] = values[i];
        hl[i] = log(values[i]);
    }
    for (int64_t r = 0; r < n_rows; ++r) {
        double cp = 0.0;
        for (int32_t k = 0; k < n_cols; ++k) {
            cp += values[(size_t)r * n_cols + k];
            hc[(size_t)r * n_cols + k] = cp;
        }
    }
    return h;
}
inline TableRef table_ref_at(const double* image, int64_t n_rows, int32_t n_cols) {
    const size_t seg = table_segment(n_rows, n_cols);
    return TableRef{(uint64_t)(uintptr_t)(image + 2), (uint64_t)(uintptr_t)(image + seg + 2), (uint64_t)(uintptr_t)(image + 2 * seg + 2),
                    n_rows, n_cols};
}

// One fusion window (or the persistent score program): micro-ops + register allocation.
struct Program {
    int max_regs = 64, max_ops = 96, max_io = 24;
    int temp_base = 0;       // registers [temp_base, temp_base + n_temp_slots) are statement temporaries
    int n_temp_slots = 0;    // 0: temporaries share the plane register space (forward windows)
    bool score_mode = false; // score programs never write planes or draw random numbers

    std::vector<WsOp> ops;
    std::map<Plane, int> plane_reg;
    std::vector<std::pair<Plane, int>> loads;  // planes read before being written in this window
    std::vector<Plane> dirty;                  // planes written in this window
    std::vector<int> free_regs;                // recycled temporaries
    std::vector<int> stmt_temps;               // temporaries of the statement being lowered
    int next_reg = 0;
    int next_temp = 0;  // score mode
    int high_water = 0; // registers actually used
    bool has_acc = false;
    // score programs: particle-independent part of the log-densities lowered so far (kept out of the
    // micro-ops: it is one scalar per tape prefix, and it cancels in a Metropolis-Hastings ratio)
    double acc_const = 0.0;
    // score programs: (1/sigma, log sigma) of a plane used as a Normal's sigma, computed once per fold in
    // persistent registers (a hierarchical model scores hundreds of terms with the same per-particle sigma)
    std::map<int, std::pair<int, int>> sigma_cache;
    std::vector<int> sigma_log;
    size_t stmt_begin_ops = 0;  // ops.size() when the current statement started
    int stmt_cache_ops = 0;     // sigma-cache prologue ops of the current statement (kept at its very start)
    RngCursor* rng = nullptr;  // set while a sampler expression is being lowered (WS_TOK_RAND*)
    const std::vector<TableRef>* tables = nullptr;  // the context's tables, by id (WS_TOK_TABLE, WS_TOK_RANDCAT)
    int n_statements = 0;
    bool overflow = false;
    std::string error;

    void fail(const std::string& m) {
        if (error.empty()) error = m;
    }
    // cheap roll-back point for score programs (they only grow: ops, loads and their plane registers)
    struct Mark {
        size_t n_ops, n_loads, n_sigma;
        int next_reg, next_temp, high_water;
        bool has_acc, overflow;
        double acc_const;
    };
    Mark mark() const { return Mark{ops.size(), loads.size(), sigma_log.size(), next_reg, next_temp, high_water, has_acc, overflow, acc_const}; }
    void rollback(const Mark& m) {
        ops.resize(m.n_ops);
        while (loads.size() > m.n_loads) {
            plane_reg.erase(loads.back().first);
            loads.pop_back();
        }
        while (sigma_log.size() > m.n_sigma) {
            sigma_cache.erase(sigma_log.back());
            sigma_log.pop_back();
        }
        next_reg = m.next_reg;
        next_temp = m.next_temp;
        high_water = m.high_water;
        has_acc = m.has_acc;
        overflow = m.overflow;
        acc_const = m.acc_const;
        stmt_begin_ops = m.n_ops;
        stmt_cache_ops = 0;
        stmt_temps.clear();
        error.clear();
    }
    void note_reg(int r) {
        if (r + 1 > high_water) high_water = r + 1;
        if (r >= max_regs) overflow = true;
    }
    int alloc_plane_reg() {
        int r;
        if (!score_mode && !free_regs.empty()) {
            r = free_regs.back();
            free_regs.pop_back();
        } else {
            if (score_mode && next_reg < temp_base + n_temp_slots) next_reg = temp_base + n_temp_slots;
            r = next_reg++;
        }
        note_reg(r);
        return r;
    }
    int alloc_temp() {
        int r;
        if (score_mode) {
            r = temp_base + next_temp++;
            if (next_temp > n_temp_slots) overflow = true;
        } else if (!free_regs.empty()) {
            r = free_regs.back();
            free_regs.pop_back();
        } else {
            r = next_reg++;
        }
        note_reg(r);
        stmt_temps.push_back(r);
        return r;
    }
    void end_statement() {
        stmt_begin_ops = ops.size();
        stmt_cache_ops = 0;
        if (score_mode) {
            next_temp = 0;
        } else {
            for (int r : stmt_temps) free_regs.push_back(r);
        }
        stmt_temps.clear();
        ++n_statements;
    }
    // A plane that is READ gets a register nobody has touched in this window: all loads are hoisted
    // to the start of the pass, so a recycled temporary would be clobbered before the read.
    int alloc_fresh_reg() {
        if (score_mode && next_reg < temp_base + n_temp_slots) next_reg = temp_base + n_temp_slots;
        int r = next_reg++;
        note_reg(r);
        return r;
    }
    int reg_for_read(Plane p) {
        auto it = plane_reg.find(p);
        if (it != plane_reg.end()) return it->second;
        int r = alloc_fresh_reg();
        plane_reg[p] = r;
        loads.push_back({p, r});
        if ((int)loads.size() > max_io) overflow = true;
        return r;
    }
    int reg_for_write(Plane p) {
        if (score_mode) {
            fail("internal: plane write in a score program");
            return 0;
        }
        auto it = plane_reg.find(p);
        int r;
        if (it != plane_reg.end()) {
            r = it->second;
        } else {
            r = alloc_plane_reg();
            plane_reg[p] = r;
        }
        bool found = false;
        for (auto& d : dirty)
            if (d == p) found = true;
        if (!found) {
            dirty.push_back(p);
            if ((int)dirty.size() > max_io) overflow = true;
        }
        return r;
    }
    void emit(const WsOp& o) {
        ops.push_back(o);
        if ((int)ops.size() > max_ops) overflow = true;
    }
    bool is_temp(int r) const {
        for (int t : stmt_temps)
            if (t == r) return true;
        return false;
    }

    // ---- value algebra ----------------------------------------------------------------------
    int materialize(const Val& v) {
        if (v.is_const) {
            int t = alloc_temp();
            emit(ws_make_op(WS_OP_LIN2, t, WS_REG_NONE, WS_REG_NONE, WS_REG_NONE, 0, v.c0, 0, 0));
            return t;
        }
        if (v.pure()) return v.reg;
        int t = alloc_temp();
        emit(ws_make_op(WS_OP_LIN2, t, v.reg, WS_REG_NONE, WS_REG_NONE, 0, v.c0, v.c1, 0));
        return t;
    }
    Val add(const Val& a, const Val& b, double sb = 1.0) {  // a + sb*b
        if (a.is_const && b.is_const) return Val::constant(a.c0 + sb * b.c0);
        if (a.is_const) return Val::lin(a.c0 + sb * b.c0, sb * b.c1, b.reg);
        if (b.is_const) return Val::lin(a.c0 + sb * b.c0, a.c1, a.reg);
        int t = alloc_temp();
        emit(ws_make_op(WS_OP_LIN2, t, a.reg, b.reg, WS_REG_NONE, 0, a.c0 + sb * b.c0, a.c1, sb * b.c1));
        return Val::lin(0.0, 1.0, t);
    }
    Val scale(const Val& a, double s) {
        if (a.is_const) return Val::constant(a.c0 * s);
        return Val::lin(a.c0 * s, a.c1 * s, a.reg);
    }
    Val mul(const Val& a, const Val& b) {
        if (a.is_const) return scale(b, a.c0);
        if (b.is_const) return scale(a, b.c0);
        int ra = a.reg, rb = b.reg;
        double k = 1.0;
        if (a.c0 != 0.0) ra = materialize(a); else k *= a.c1;
        if (b.c0 != 0.0) rb = materialize(b); else k *= b.c1;
        int t = alloc_temp();
        emit(ws_make_op(WS_OP_MUL, t, ra, rb, WS_REG_NONE, 0, k, 0, 0));
        return Val::lin(0.0, 1.0, t);
    }
    Val div(const Val& a, const Val& b) {
        if (a.is_const && b.is_const) return Val::constant(a.c0 / b.c0);
        int t;
        if (b.is_const) {
            // keep a true division (x / c), not x * (1/c), to follow the reference's rounding
            if (a.c0 == 0.0) {
                t = alloc_temp();
                emit(ws_make_op(WS_OP_DIV, t, a.reg, WS_REG_NONE, WS_REG_NONE, 0, a.c1, 0, b.c0));
            } else {
                int ra = materialize(a);
                t = alloc_temp();
                emit(ws_make_op(WS_OP_DIV, t, ra, WS_REG_NONE, WS_REG_NONE, 0, 1.0, 0, b.c0));
            }
            return Val::lin(0.0, 1.0, t);
        }
        int rb = materialize(b);
        if (a.is_const) {
            t = alloc_temp();
            emit(ws_make_op(WS_OP_DIV, t, WS_REG_NONE, rb, WS_REG_NONE, 0, 1.0, a.c0, 0));
        } else if (a.c0 == 0.0) {
            t = alloc_temp();
            emit(ws_make_op(WS_OP_DIV, t, a.reg, rb, WS_REG_NONE, 0, a.c1, 0, 0));
        } else {
            int ra = materialize(a);
            t = alloc_temp();
            emit(ws_make_op(WS_OP_DIV, t, ra, rb, WS_REG_NONE, 0, 1.0, 0, 0));
        }
        return Val::lin(0.0, 1.0, t);
    }
    static double host_unary(uint32_t f, double x) {
        switch (f) {
            case WS_UN_EXP: return exp(x);
            case WS_UN_LOG: return log(x);
            case WS_UN_SQRT: return sqrt(x);
            case WS_UN_SIN: return sin(x);
            case WS_UN_COS: return cos(x);
            case WS_UN_ABS: return fabs(x);
            case WS_UN_NOT: return x == 0.0 ? 1.0 : 0.0;
            case WS_UN_LGAMMA: return lgamma(x);
            case WS_UN_LOG1P: return log1p(x);
            case WS_UN_EXPM1: return expm1(x);
            case WS_UN_TAN: return tan(x);
            case WS_UN_ATAN: return atan(x);
            case WS_UN_TANH: return tanh(x);
            case WS_UN_FLOOR: return floor(x);
            default: return x * x;
        }
    }
    Val unary(uint32_t f, const Val& a) {
        if (a.is_const) return Val::constant(host_unary(f, a.c0));
        if (f == WS_UN_SQUARE) return mul(a, a);
        int ra = materialize(a);
        int t = alloc_temp();
        emit(ws_make_op(WS_OP_UNARY, t, ra, WS_REG_NONE, WS_REG_NONE, f, 0, 0, 0));
        return Val::lin(0.0, 1.0, t);
    }
    Val power(const Val& a, const Val& b) {
        if (a.is_const && b.is_const) return Val::constant(pow(a.c0, b.c0));
        if (b.is_const && b.c0 == 2.0) return mul(a, a);
        if (b.is_const && b.c0 == 1.0) return a;
        int ra = a.is_const ? (int)WS_REG_NONE : materialize(a);
        int rb = b.is_const ? (int)WS_REG_NONE : materialize(b);
        int t = alloc_temp();
        emit(ws_make_op(WS_OP_POW, t, ra, rb, WS_REG_NONE, 0, 0, a.is_const ? a.c0 : 0.0, b.is_const ? b.c0 : 0.0));
        return Val::lin(0.0, 1.0, t);
    }

    Val compare(uint32_t kind, const Val& a, const Val& b) {  // 0 <, 1 <=, 2 ==
        if (a.is_const && b.is_const) {
            const bool t = kind == 0 ? (a.c0 < b.c0) : (kind == 1 ? (a.c0 <= b.c0) : (a.c0 == b.c0));
            return Val::constant(t ? 1.0 : 0.0);
        }
        const int ra = a.is_const ? (int)WS_REG_NONE : materialize(a);
        const int rb = b.is_const ? (int)WS_REG_NONE : materialize(b);
        int t = alloc_temp();
        emit(ws_make_op(WS_OP_CMP, t, ra, rb, WS_REG_NONE, kind, 0, a.is_const ? a.c0 : 0.0, b.is_const ? b.c0 : 0.0));
        return Val::lin(0.0, 1.0, t);
    }
    Val minmax(uint32_t is_max, const Val& a, const Val& b) {
        if (a.is_const && b.is_const) return Val::constant(is_max ? fmax(a.c0, b.c0) : fmin(a.c0, b.c0));
        const int ra = a.is_const ? (int)WS_REG_NONE : materialize(a);
        const int rb = b.is_const ? (int)WS_REG_NONE : materialize(b);
        int t = alloc_temp();
        emit(ws_make_op(WS_OP_MINMAX, t, ra, rb, WS_REG_NONE, is_max, 0, a.is_const ? a.c0 : 0.0, b.is_const ? b.c0 : 0.0));
        return Val::lin(0.0, 1.0, t);
    }
    Val select(const Val& cnd, const Val& a, const Val& b) {
        if (cnd.is_const) return cnd.c0 != 0.0 ? a : b;
        const int rc = materialize(cnd);
        const int ra = a.is_const ? (int)WS_REG_NONE : materialize(a);
        const int rb = b.is_const ? (int)WS_REG_NONE : materialize(b);
        int t = alloc_temp();
        emit(ws_make_op(WS_OP_SELECT, t, ra, rb, rc, 0, 0, a.is_const ? a.c0 : 0.0, b.is_const ? b.c0 : 0.0));
        return Val::lin(0.0, 1.0, t);
    }
    Val variate(int32_t tok) {
        if (score_mode || rng == nullptr) {
            fail("random variates are only allowed in a sampler expression");
            return Val::constant(NAN);
        }
        int t = alloc_temp();
        const uint64_t stream = (*rng->stream)++;
        double sbits;
        memcpy(&sbits, &stream, 8);
        if (tok == WS_TOK_RANDN) {
            emit(ws_make_op(WS_OP_RANDN2, t, WS_REG_NONE, WS_REG_NONE, WS_REG_NONE, 0, sbits, (double)*rng->normals, 1.0));
            *rng->normals += rng->n_global;
        } else if (tok == WS_TOK_RANDU) {
            emit(ws_make_op(WS_OP_RANDU, t, WS_REG_NONE, WS_REG_NONE, WS_REG_NONE, 0, sbits, (double)*rng->uniforms, 1.0));
            *rng->uniforms += rng->n_global;
        } else {
            emit(ws_make_op(WS_OP_RANDEXP, t, WS_REG_NONE, WS_REG_NONE, WS_REG_NONE, 0, sbits, (double)*rng->exponentials, 1.0));
            *rng->exponentials += rng->n_global;
        }
        return Val::lin(0.0, 1.0, t);
    }

    // Gamma(shape) / Poisson(rate) variate with a per-particle or constant parameter (WS_OP_RANDV)
    Val variate_param(uint32_t kind, const Val& a) {
        if (score_mode || rng == nullptr) {
            fail("random variates are only allowed in a sampler expression");
            return Val::constant(NAN);
        }
        const int ra = a.is_const ? (int)WS_REG_NONE : materialize(a);
        int t = alloc_temp();
        const uint64_t stream = (*rng->stream)++;
        double sbits;
        memcpy(&sbits, &stream, 8);
        int64_t base = 0;
        if (rng->variates != nullptr) {
            base = *rng->variates;
            *rng->variates += rng->n_global;
        }
        emit(ws_make_op(WS_OP_RANDV, t, ra, WS_REG_NONE, WS_REG_NONE, kind, sbits, (double)base, a.is_const ? a.c0 : 0.0));
        return Val::lin(0.0, 1.0, t);
    }

    // ---- tables ---------------------------------------------------------------------------------
    const TableRef* table_ref(int32_t id) {
        if (tables == nullptr || id < 0 || id >= (int32_t)tables->size()) {
            fail("unknown table id");
            return nullptr;
        }
        return &(*tables)[(size_t)id];
    }
    static double addr_bits(uint64_t addr) {
        double b;
        memcpy(&b, &addr, 8);
        return b;
    }
    // T[row, col] (logp: log T[row, col] with a column outside 1..n_cols giving -Inf, the log-probability of a Categorical)
    Val table_read(const TableRef& t, const Val& row, const Val& col, bool logp) {
        const int ra = row.is_const ? (int)WS_REG_NONE : materialize(row);
        const int rb = col.is_const ? (int)WS_REG_NONE : materialize(col);
        const int d = alloc_temp();
        emit(ws_make_op(WS_OP_TABLE, d, ra, rb, WS_REG_NONE, (uint32_t)t.n_cols | (logp ? WS_TABLE_LOGP : 0u),
                        addr_bits(logp ? t.logv : t.values), row.is_const ? row.c0 : 0.0, col.is_const ? col.c0 : 0.0));
        return Val::lin(0.0, 1.0, d);
    }
    // Categorical(T[row, :]): one uniform per particle (an ordinary WS_OP_RANDU: replay and Philox as for Uniform), then
    // the search of that row's partial sums
    Val categorical(const TableRef& t, const Val& row) {
        const int rb = row.is_const ? (int)WS_REG_NONE : materialize(row);
        const Val u = variate(WS_TOK_RANDU);
        if (!error.empty()) return Val::constant(NAN);
        const int d = alloc_temp();
        emit(ws_make_op(WS_OP_CAT, d, u.reg, rb, WS_REG_NONE, (uint32_t)t.n_cols, addr_bits(t.cdf), row.is_const ? row.c0 : 0.0, 0.0));
        return Val::lin(0.0, 1.0, d);
    }

    // postfix tokens -> Val
    Val compile(const ws_expr& e) {
        std::vector<Val> st;
        if (e.toks == nullptr || e.n <= 0) {
            fail("empty expression");
            return Val::constant(NAN);
        }
        for (int i = 0; i < e.n; ++i) {
            const ws_tok& t = e.toks[i];
            switch (t.op) {
                case WS_TOK_CONST: st.push_back(Val::constant(t.val)); break;
                case WS_TOK_PLANE: st.push_back(Val::lin(0.0, 1.0, reg_for_read(Plane{t.col, t.comp}))); break;
                case WS_TOK_RANDN:
                case WS_TOK_RANDU:
                case WS_TOK_RANDEXP: st.push_back(variate(t.op)); break;
                case WS_TOK_SELECT: {
                    if (st.size() < 3) {
                        fail("malformed expression (select needs three operands)");
                        return Val::constant(NAN);
                    }
                    Val b = st.back(); st.pop_back();
                    Val a = st.back(); st.pop_back();
                    Val cnd = st.back(); st.pop_back();
                    st.push_back(select(cnd, a, b));
                } break;
                case WS_TOK_ADD:
                case WS_TOK_SUB:
                case WS_TOK_MUL:
                case WS_TOK_DIV:
                case WS_TOK_LT:
                case WS_TOK_LE:
                case WS_TOK_EQ:
                case WS_TOK_MIN:
                case WS_TOK_MAX:
                case WS_TOK_POW: {
                    if (st.size() < 2) {
                        fail("malformed expression (binary operator needs two operands)");
                        return Val::constant(NAN);
                    }
                    Val b = st.back();
                    st.pop_back();
                    Val a = st.back();
                    st.pop_back();
                    Val r = Val::constant(NAN);
                    if (t.op == WS_TOK_ADD) r = add(a, b, 1.0);
                    else if (t.op == WS_TOK_SUB) r = add(a, b, -1.0);
                    else if (t.op == WS_TOK_MUL) r = mul(a, b);
                    else if (t.op == WS_TOK_DIV) r = div(a, b);
                    else if (t.op == WS_TOK_LT) r = compare(0, a, b);
                    else if (t.op == WS_TOK_LE) r = compare(1, a, b);
                    else if (t.op == WS_TOK_EQ) r = compare(2, a, b);
                    else if (t.op == WS_TOK_MIN) r = minmax(0, a, b);
                    else if (t.op == WS_TOK_MAX) r = minmax(1, a, b);
                    else r = power(a, b);
                    st.push_back(r);
                } break;
                case WS_TOK_TABLE: {
                    if (st.size() < 2) {
                        fail("malformed expression (a table read needs a row and a column)");
                        return Val::constant(NAN);
                    }
                    const TableRef* tr = table_ref(t.col);
                    if (tr == nullptr) return Val::constant(NAN);
                    Val cl = st.back();
                    st.pop_back();
                    Val rw = st.back();
                    st.pop_back();
                    st.push_back(table_read(*tr, rw, cl, t.comp == 1));
                } break;
                case WS_TOK_RANDCAT: {
                    if (st.empty()) {
                        fail("malformed expression (a Categorical draw needs its row)");
                        return Val::constant(NAN);
                    }
                    const TableRef* tr = table_ref(t.col);
                    if (tr == nullptr) return Val::constant(NAN);
                    Val rw = st.back();
                    st.pop_back();
                    st.push_back(categorical(*tr, rw));
                } break;
                case WS_TOK_RANDGAMMA:
                case WS_TOK_RANDPOISSON: {
                    if (st.empty()) {
                        fail("malformed expression (variate needs its parameter)");
                        return Val::constant(NAN);
                    }
                    Val a = st.back();
                    st.pop_back();
                    st.push_back(variate_param(t.op == WS_TOK_RANDGAMMA ? 0u : 1u, a));
                } break;
                case WS_TOK_NEG:
                case WS_TOK_EXP:
                case WS_TOK_LOG:
                case WS_TOK_SQRT:
                case WS_TOK_SQUARE:
                case WS_TOK_SIN:
                case WS_TOK_COS:
                case WS_TOK_NOT:
                case WS_TOK_LGAMMA:
                case WS_TOK_LOG1P:
                case WS_TOK_EXPM1:
                case WS_TOK_TAN:
                case WS_TOK_ATAN:
                case WS_TOK_TANH:
                case WS_TOK_FLOOR:
                case WS_TOK_ABS: {
                    if (st.empty()) {
                        fail("malformed expression (unary operator needs an operand)");
                        return Val::constant(NAN);
                    }
                    Val a = st.back();
                    st.pop_back();
                    Val r = Val::constant(NAN);
                    switch (t.op) {
                        case WS_TOK_NEG: r = scale(a, -1.0); break;
                        case WS_TOK_EXP: r = unary(WS_UN_EXP, a); break;
                        case WS_TOK_LOG: r = unary(WS_UN_LOG, a); break;
                        case WS_TOK_SQRT: r = unary(WS_UN_SQRT, a); break;
                        case WS_TOK_SQUARE: r = unary(WS_UN_SQUARE, a); break;
                        case WS_TOK_SIN: r = unary(WS_UN_SIN, a); break;
                        case WS_TOK_COS: r = unary(WS_UN_COS, a); break;
                        case WS_TOK_NOT: r = unary(WS_UN_NOT, a); break;
                        case WS_TOK_LGAMMA: r = unary(WS_UN_LGAMMA, a); break;
                        case WS_TOK_LOG1P: r = unary(WS_UN_LOG1P, a); break;
                        case WS_TOK_EXPM1: r = unary(WS_UN_EXPM1, a); break;
                        case WS_TOK_TAN: r = unary(WS_UN_TAN, a); break;
                        case WS_TOK_ATAN: r = unary(WS_UN_ATAN, a); break;
                        case WS_TOK_TANH: r = unary(WS_UN_TANH, a); break;
                        case WS_TOK_FLOOR: r = unary(WS_UN_FLOOR, a); break;
                        default: r = unary(WS_UN_ABS, a); break;
                    }
                    st.push_back(r);
                } break;
                default:
                    fail("unknown expression token");
                    return Val::constant(NAN);
            }
        }
        if (st.size() != 1) {
            fail("malformed expression (stack does not reduce to one value)");
            return Val::constant(NAN);
        }
        return st.back();
    }

    // write `v` into plane p.  If v is the result of the op just emitted into a temporary, that op
    // is retargeted at the plane's register (its sources are read before the write, so in-place
    // updates such as `x .= x + v` or `x ~ Normal(a*x, q)` are safe).
    void store_val(Plane p, const Val& v) {
        int dst = reg_for_write(p);
        if (v.is_const) {
            emit(ws_make_op(WS_OP_LIN2, dst, WS_REG_NONE, WS_REG_NONE, WS_REG_NONE, 0, v.c0, 0, 0));
            return;
        }
        if (v.pure() && is_temp(v.reg) && !ops.empty()) {
            WsOp& last = ops.back();
            const uint32_t lop = last.w0 & 0xFFu;
            const uint32_t ldst = (last.w0 >> 8) & 0xFFu;
            if ((int)ldst == v.reg && (lop <= WS_OP_POW || (lop >= WS_OP_CMP && lop <= WS_OP_MINMAX) || lop == WS_OP_TABLE ||
                                       lop == WS_OP_CAT)) {
                last.w0 = (last.w0 & ~0xFF00u) | ((uint32_t)dst << 8);
                return;
            }
        }
        emit(ws_make_op(WS_OP_LIN2, dst, v.reg, WS_REG_NONE, WS_REG_NONE, 0, v.c0, v.c1, 0));
    }

    // ---- random draws ------------------------------------------------------------------------
    // d standard normals for one statement; replay layout: buf[base + particle*d + j]
    std::vector<int> draw_normals(int d, RngCursor& rc) {
        std::vector<int> regs(d);
        for (int j = 0; j < d; ++j) regs[j] = alloc_temp();
        const int64_t base = *rc.normals;
        for (int j = 0; j < d; j += 2) {
            const uint64_t stream = (*rc.stream)++;
            double sbits;
            static_assert(sizeof(double) == sizeof(uint64_t), "");
            memcpy(&sbits, &stream, 8);
            const int second = (j + 1 < d) ? regs[j + 1] : (int)WS_REG_NONE;
            emit(ws_make_op(WS_OP_RANDN2, regs[j], second, WS_REG_NONE, WS_REG_NONE, (uint32_t)j, sbits, (double)base,
                            (double)d));
        }
        *rc.normals += rc.n_global * (int64_t)d;
        return regs;
    }
    int draw_exponential(RngCursor& rc) {
        int t = alloc_temp();
        const uint64_t stream = (*rc.stream)++;
        double sbits;
        memcpy(&sbits, &stream, 8);
        emit(ws_make_op(WS_OP_RANDEXP, t, WS_REG_NONE, WS_REG_NONE, WS_REG_NONE, 0, sbits, (double)*rc.exponentials, 1.0));
        *rc.exponentials += rc.n_global;
        return t;
    }

    // ---- log densities into acc ----------------------------------------------------------------
    void acc_normal_logpdf(const Val& x, const Val& mu, const Val& sigma) {
        has_acc = true;
        if (sigma.is_const && sigma.c0 > 0.0 && isfinite(sigma.c0)) {
            const double s = sigma.c0;
            const double K = -0.5 * WS_LOG2PI - log(s);
            if (score_mode && !(x.is_const && mu.is_const)) {
                // Score tapes are folded twice per particle and move (k terms each): z = (x - mu)/s is kept
                // as ONE affine form of at most two registers — the LIN2 that produced an affine mean such
                // as alpha + beta*x_i is absorbed — and the constant goes to acc_const.
                const double is = 1.0 / s;
                double k0 = 0.0, kk[2] = {0.0, 0.0};
                int rr[2] = {(int)WS_REG_NONE, (int)WS_REG_NONE};
                int nr = 0;
                auto absorb = [&](const Val& v, double sign) {  // adds sign * v / s to the form
                    if (v.is_const) {
                        k0 += sign * v.c0 * is;
                        return;
                    }
                    if (nr == 0 && !ops.empty() && is_temp(v.reg)) {
                        const WsOp& last = ops.back();
                        const uint32_t lop = last.w0 & 0xFFu, ldst = (last.w0 >> 8) & 0xFFu;
                        if (lop == WS_OP_LIN2 && (int)ldst == v.reg) {
                            const int la = (int)((last.w0 >> 16) & 0xFFu), lb = (int)((last.w0 >> 24) & 0xFFu);
                            const double f = sign * v.c1 * is;
                            k0 += sign * v.c0 * is + f * last.k0;
                            if (la != (int)WS_REG_NONE) {
                                rr[nr] = la;
                                kk[nr++] = f * last.k1;
                            }
                            if (lb != (int)WS_REG_NONE) {
                                rr[nr] = lb;
                                kk[nr++] = f * last.k2;
                            }
                            ops.pop_back();
                            return;
                        }
                    }
                    k0 += sign * v.c0 * is;
                    rr[nr] = v.reg;
                    kk[nr++] = sign * v.c1 * is;
                };
                // the side that may be a freshly computed affine temporary first (only the LAST op can be absorbed)
                if (x.is_const) {
                    absorb(mu, -1.0);
                    absorb(x, 1.0);
                } else if (mu.is_const) {
                    absorb(x, 1.0);
                    absorb(mu, -1.0);
                } else {
                    k0 = (x.c0 - mu.c0) * is;
                    rr[0] = x.reg;
                    kk[0] = x.c1 * is;
                    rr[1] = mu.reg;
                    kk[1] = -mu.c1 * is;
                }
                emit(ws_make_op(WS_OP_ACC_SQLIN2, 0, rr[0], rr[1], WS_REG_NONE, 0, k0, kk[0], kk[1]));
                acc_const += K;
                return;
            }
            if (x.is_const && mu.is_const) {
                const double z = (x.c0 - mu.c0) / s;
                emit(ws_make_op(WS_OP_ACC_LIN2, 0, WS_REG_NONE, WS_REG_NONE, WS_REG_NONE, 0, -(z * z + WS_LOG2PI) / 2.0 - log(s), 0, 0));
                return;
            }
            // (x - mu)^2 is symmetric: put whichever side is per-particle into the MU register slot
            if (mu.is_const) {
                int rx = materialize(x);
                emit(ws_make_op(WS_OP_LOGPDF_NORMAL_CS, 0, WS_REG_NONE, rx, WS_REG_NONE, 0, mu.c0, 1.0 / s, K));
            } else if (x.is_const) {
                int rm = materialize(mu);
                emit(ws_make_op(WS_OP_LOGPDF_NORMAL_CS, 0, WS_REG_NONE, rm, WS_REG_NONE, 0, x.c0, 1.0 / s, K));
            } else {
                int rx = materialize(x);
                int rm = materialize(mu);
                emit(ws_make_op(WS_OP_LOGPDF_NORMAL_CS, 0, rx, rm, WS_REG_NONE, 0, 0.0, 1.0 / s, K));
            }
            return;
        }
        if (score_mode && sigma.pure() && !is_temp(sigma.reg) && !(x.is_const && mu.is_const)) {
            // per-particle sigma that is a plane: z = (x - mu) / sigma as an affine form times the cached 1/sigma,
            // minus the cached log sigma; the LIN2 that produced an affine mean is absorbed as above
            auto it = sigma_cache.find(sigma.reg);
            if (it == sigma_cache.end()) {
                const int ris = alloc_fresh_reg(), rls = alloc_fresh_reg();
                // the prologue goes to the very start of the statement's ops, so that a move can keep it while
                // dropping the terms that do not involve its targets
                const WsOp pro[2] = {ws_make_op(WS_OP_DIV, ris, WS_REG_NONE, sigma.reg, WS_REG_NONE, 0, 1.0, 1.0, 0.0),
                                     ws_make_op(WS_OP_UNARY, rls, sigma.reg, WS_REG_NONE, WS_REG_NONE, WS_UN_LOG, 0, 0, 0)};
                ops.insert(ops.begin() + (std::ptrdiff_t)(stmt_begin_ops + (size_t)stmt_cache_ops), pro, pro + 2);
                stmt_cache_ops += 2;
                if ((int)ops.size() > max_ops) overflow = true;
                it = sigma_cache.emplace(sigma.reg, std::make_pair(ris, rls)).first;
                sigma_log.push_back(sigma.reg);
            }
            double k0 = 0.0, kk[2] = {0.0, 0.0};
            int rr[2] = {(int)WS_REG_NONE, (int)WS_REG_NONE};
            int nr = 0;
            if (!x.is_const && !mu.is_const) {
                // x and mu both per-particle (theta_j ~ Normal(mu, tau)): two registers, nothing to absorb
                emit(ws_make_op(WS_OP_ACC_SQLIN2_S, it->second.second, x.reg, mu.reg, it->second.first, 0, x.c0 - mu.c0, x.c1, -mu.c1));
                acc_const += -0.5 * WS_LOG2PI;
                return;
            }
            const Val& v = x.is_const ? mu : x;
            const double sign = x.is_const ? -1.0 : 1.0;
            const Val& cst = x.is_const ? x : mu;
            bool absorbed = false;
            if (!v.is_const && !ops.empty() && is_temp(v.reg)) {
                const WsOp& last = ops.back();
                const uint32_t lop = last.w0 & 0xFFu, ldst = (last.w0 >> 8) & 0xFFu;
                if (lop == WS_OP_LIN2 && (int)ldst == v.reg) {
                    const int la = (int)((last.w0 >> 16) & 0xFFu), lb = (int)((last.w0 >> 24) & 0xFFu);
                    const double f = sign * v.c1;
                    k0 = sign * v.c0 + f * last.k0;
                    if (la != (int)WS_REG_NONE) {
                        rr[nr] = la;
                        kk[nr++] = f * last.k1;
                    }
                    if (lb != (int)WS_REG_NONE) {
                        rr[nr] = lb;
                        kk[nr++] = f * last.k2;
                    }
                    ops.pop_back();
                    absorbed = true;
                }
            }
            if (!absorbed) {
                k0 = sign * v.c0;
                rr[0] = v.reg;
                kk[0] = sign * v.c1;
            }
            k0 += -sign * cst.c0;
            emit(ws_make_op(WS_OP_ACC_SQLIN2_S, it->second.second, rr[0], rr[1], it->second.first, 0, k0, kk[0], kk[1]));
            acc_const += -0.5 * WS_LOG2PI;
            return;
        }
        const int rx = x.is_const ? (int)WS_REG_NONE : materialize(x);
        const int rm = mu.is_const ? (int)WS_REG_NONE : materialize(mu);
        const int rs = sigma.is_const ? (int)WS_REG_NONE : materialize(sigma);
        emit(ws_make_op(WS_OP_LOGPDF_NORMAL, 0, rx, rm, rs, 0, x.is_const ? x.c0 : 0.0, mu.is_const ? mu.c0 : 0.0,
                        sigma.is_const ? sigma.c0 : 0.0));
    }
    void acc_exponential_logpdf(const Val& x, const Val& theta) {
        has_acc = true;
        const int rx = x.is_const ? (int)WS_REG_NONE : materialize(x);
        const int rt = theta.is_const ? (int)WS_REG_NONE : materialize(theta);
        emit(ws_make_op(WS_OP_LOGPDF_EXPON, 0, rx, rt, WS_REG_NONE, 0, x.is_const ? x.c0 : 0.0,
                        theta.is_const ? theta.c0 : 0.0, 0));
    }
    // acc += c0 - 1/2 * || Linv (x - mu) ||^2    (MvNormal logpdf; Linv lower triangular, row-major d x d)
    void acc_mvnormal_logpdf(int d, const std::vector<Val>& x, const std::vector<Val>& mu, const std::vector<double>& Linv,
                             double c0) {
        has_acc = true;
        std::vector<Val> diff(d, Val::constant(0.0));
        for (int j = 0; j < d; ++j) diff[j] = add(x[j], mu[j], -1.0);
        double konst = c0;
        std::vector<int> yregs;
        for (int j = 0; j < d; ++j) {
            Val y = Val::constant(0.0);
            for (int k = 0; k <= j; ++k) {
                const double l = Linv[j * d + k];
                if (l == 0.0) continue;
                y = add(y, scale(diff[k], l));
            }
            if (y.is_const) {
                konst += -0.5 * y.c0 * y.c0;
            } else {
                yregs.push_back(materialize(y));
            }
        }
        if (yregs.empty()) {
            emit(ws_make_op(WS_OP_ACC_LIN2, 0, WS_REG_NONE, WS_REG_NONE, WS_REG_NONE, 0, konst, 0, 0));
            return;
        }
        for (size_t j = 0; j < yregs.size(); j += 2) {
            const int a = yregs[j];
            const int b = (j + 1 < yregs.size()) ? yregs[j + 1] : (int)WS_REG_NONE;
            emit(ws_make_op(WS_OP_ACC_QUAD2, 0, a, b, WS_REG_NONE, 0, j == 0 ? konst : 0.0, -0.5, -0.5));
        }
    }
    void acc_val(const Val& v, double s = 1.0) {
        has_acc = true;
        if (v.is_const) {
            emit(ws_make_op(WS_OP_ACC_LIN2, 0, WS_REG_NONE, WS_REG_NONE, WS_REG_NONE, 0, s * v.c0, 0, 0));
        } else {
            emit(ws_make_op(WS_OP_ACC_LIN2, 0, v.reg, WS_REG_NONE, WS_REG_NONE, 0, s * v.c0, s * v.c1, 0));
        }
    }
};

// lower Cholesky factor of a symmetric positive definite d x d matrix (row-major); false if not PD
inline bool cholesky_lower(int d, const double* A, std::vector<double>& L) {
    L.assign((size_t)d * d, 0.0);
    for (int j = 0; j < d; ++j) {
        double s = A[j * d + j];
        for (int k = 0; k < j; ++k) s -= L[j * d + k] * L[j * d + k];
        if (!(s > 0.0)) return false;
        const double ljj = sqrt(s);
        L[j * d + j] = ljj;
        for (int i = j + 1; i < d; ++i) {
            double t = A[i * d + j];
            for (int k = 0; k < j; ++k) t -= L[i * d + k] * L[j * d + k];
            L[i * d + j] = t / ljj;
        }
    }
    return true;
}
inline void lower_inverse(int d, const std::vector<double>& L, std::vector<double>& Li) {
    Li.assign((size_t)d * d, 0.0);
    for (int i = 0; i < d; ++i) {
        Li[i * d + i] = 1.0 / L[i * d + i];
        for (int j = 0; j < i; ++j) {
            double s = 0.0;
            for (int k = j; k < i; ++k) s += L[i * d + k] * Li[k * d + j];
            Li[i * d + j] = -s / L[i * d + i];
        }
    }
}


// ---------------------------------------------------------------------------------------------
// Statements.  `stmt_*` lower the forward (apply!) form into a fusion window, `score_*` append the
// statement's log-density to a score program (score!).  Both the CUDA runtime and the CPU test
// harness (tests/host/) call exactly these.
// ---------------------------------------------------------------------------------------------
inline void stmt_assign(Program& p, Plane dst, const ws_expr& rhs) { p.store_val(dst, p.compile(rhs)); }

inline void stmt_assign_vec(Program& p, int32_t col, int32_t d, const ws_expr* rhs) {
    // does any component read another component of the destination?  then evaluate all right-hand
    // sides before the first write (Julia evaluates the whole RHS broadcast first)
    bool hazard = false;
    for (int j = 0; j < d; ++j)
        for (int i = 0; i < rhs[j].n; ++i)
            if (rhs[j].toks[i].op == WS_TOK_PLANE && rhs[j].toks[i].col == col && rhs[j].toks[i].comp != j) hazard = true;
    if (!hazard) {
        for (int j = 0; j < d; ++j) p.store_val(Plane{col, j}, p.compile(rhs[j]));
        return;
    }
    std::vector<Val> vals;
    for (int j = 0; j < d; ++j) {
        Val v = p.compile(rhs[j]);
        if (!v.is_const) {
            int r = p.materialize(v);
            if (!p.is_temp(r)) {  // a plane register: copy, the plane may be overwritten below
                int t = p.alloc_temp();
                p.emit(ws_make_op(WS_OP_LIN2, t, r, WS_REG_NONE, WS_REG_NONE, 0, 0.0, 1.0, 0));
                r = t;
            }
            v = Val::lin(0.0, 1.0, r);
        }
        vals.push_back(v);
    }
    for (int j = 0; j < d; ++j) {
        int dst = p.reg_for_write(Plane{col, j});
        if (vals[j].is_const)
            p.emit(ws_make_op(WS_OP_LIN2, dst, WS_REG_NONE, WS_REG_NONE, WS_REG_NONE, 0, vals[j].c0, 0, 0));
        else
            p.emit(ws_make_op(WS_OP_LIN2, dst, vals[j].reg, WS_REG_NONE, WS_REG_NONE, 0, 0.0, 1.0, 0));
    }
}

// x = mu + sigma * z   (rand(Normal(mu, sigma)))
inline void stmt_sample_normal(Program& p, RngCursor& rc, Plane dst, const ws_expr& mu, const ws_expr& sigma) {
    Val vm = p.compile(mu), vs = p.compile(sigma);
    std::vector<int> z = p.draw_normals(1, rc);
    p.store_val(dst, p.add(vm, p.mul(vs, Val::lin(0.0, 1.0, z[0]))));
}
inline void score_sample_normal(Program& p, Plane x, const ws_expr& mu, const ws_expr& sigma) {
    Val vm = p.compile(mu), vs = p.compile(sigma);
    p.acc_normal_logpdf(Val::lin(0.0, 1.0, p.reg_for_read(x)), vm, vs);
}

// x = theta * e   (rand(Exponential(theta)))
inline void stmt_sample_exponential(Program& p, RngCursor& rc, Plane dst, const ws_expr& theta) {
    Val vt = p.compile(theta);
    int e = p.draw_exponential(rc);
    p.store_val(dst, p.mul(vt, Val::lin(0.0, 1.0, e)));
}
inline void score_sample_exponential(Program& p, Plane x, const ws_expr& theta) {
    Val vt = p.compile(theta);
    p.acc_exponential_logpdf(Val::lin(0.0, 1.0, p.reg_for_read(x)), vt);
}

// x = mu + L z   (rand(MvNormal): unwhiten, then add the mean)
inline void stmt_sample_mvnormal(Program& p, RngCursor& rc, int32_t col, int32_t d, const ws_expr* mu,
                                 const std::vector<double>& L) {
    std::vector<Val> vm;
    for (int j = 0; j < d; ++j) vm.push_back(p.compile(mu[j]));
    std::vector<int> z = p.draw_normals(d, rc);
    for (int j = 0; j < d; ++j) {
        Val t = Val::constant(0.0);
        for (int k = 0; k <= j; ++k) {
            if (L[j * d + k] == 0.0) continue;
            t = p.add(t, Val::lin(0.0, L[j * d + k], z[k]));
        }
        p.store_val(Plane{col, j}, p.add(t, vm[j]));
    }
}
inline void score_sample_mvnormal(Program& p, int32_t col, int32_t d, const ws_expr* mu, const std::vector<double>& Linv,
                                  double c0) {
    std::vector<Val> vm, vx;
    for (int j = 0; j < d; ++j) vm.push_back(p.compile(mu[j]));
    for (int j = 0; j < d; ++j) vx.push_back(Val::lin(0.0, 1.0, p.reg_for_read(Plane{col, j})));
    p.acc_mvnormal_logpdf(d, vx, vm, Linv, c0);
}

// weights .+= logpdf.(D(args...), obs)  — identical in the forward window and on the tape
inline void stmt_observe_normal(Program& p, const ws_expr& obs, const ws_expr& mu, const ws_expr& sigma) {
    Val vo = p.compile(obs), vm = p.compile(mu), vs = p.compile(sigma);
    p.acc_normal_logpdf(vo, vm, vs);
}
inline void stmt_observe_exponential(Program& p, const ws_expr& obs, const ws_expr& theta) {
    Val vo = p.compile(obs), vt = p.compile(theta);
    p.acc_exponential_logpdf(vo, vt);
}
inline void stmt_observe_mvnormal(Program& p, int32_t d, const ws_expr* obs, const ws_expr* mu, const std::vector<double>& Linv,
                                  double c0) {
    std::vector<Val> vo, vm;
    for (int j = 0; j < d; ++j) vo.push_back(p.compile(obs[j]));
    for (int j = 0; j < d; ++j) vm.push_back(p.compile(mu[j]));
    p.acc_mvnormal_logpdf(d, vo, vm, Linv, c0);
}
inline void stmt_weight_expr(Program& p, const ws_expr& term) { p.acc_val(p.compile(term)); }

// importance_kernel(Normal(pm, ps), Normal(tm, ts)) (src/default_kernels.jl:69-73): x from the
// proposal, weights += logpdf(target, x) - logpdf(proposal, x)
inline void stmt_importance_normal(Program& p, RngCursor& rc, Plane dst, double pm, double ps, double tm, double ts) {
    std::vector<int> z = p.draw_normals(1, rc);
    p.store_val(dst, Val::lin(pm, ps, z[0]));
    Val xr = Val::lin(0.0, 1.0, p.plane_reg[dst]);
    Val zt = p.scale(p.add(xr, Val::constant(tm), -1.0), 1.0 / ts);
    Val zp = p.scale(p.add(xr, Val::constant(pm), -1.0), 1.0 / ps);
    Val st = p.mul(zt, zt), sp = p.mul(zp, zp);
    const double K = (-0.5 * WS_LOG2PI - log(ts)) - (-0.5 * WS_LOG2PI - log(ps));
    p.has_acc = true;
    p.emit(ws_make_op(WS_OP_ACC_LIN2, 0, st.reg, sp.reg, WS_REG_NONE, 0, K, -0.5, 0.5));
}

// x = sampler(args...) with fresh variates; weights += weighter(args..., x)
inline void stmt_sample_expr(Program& p, RngCursor& rc, Plane dst, const ws_expr& sampler, const ws_expr* weighter) {
    p.rng = &rc;
    Val x = p.compile(sampler);
    p.rng = nullptr;
    p.store_val(dst, x);
    if (weighter != nullptr) p.acc_val(p.compile(*weighter));
}

// MvNormal(mu, Sigma) constants: L = chol(Sigma).L, Linv, c0 = -(d log 2pi + logdet Sigma)/2
inline bool mvnormal_factors(int d, const double* cov, std::vector<double>& L, std::vector<double>& Linv, double& c0) {
    if (!cholesky_lower(d, cov, L)) return false;
    lower_inverse(d, L, Linv);
    double logdet = 0.0;
    for (int j = 0; j < d; ++j) logdet += log(L[j * d + j]);
    logdet *= 2.0;
    c0 = -((double)d * WS_LOG2PI + logdet) / 2.0;
    return true;
}

}  // namespace wsl
