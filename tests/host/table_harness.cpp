// tests/host/table_harness.cpp — CPU harness for table reads and Categorical draws (TEST INFRASTRUCTURE ONLY).
//
// Like harness.cpp it runs the product's statement lowering (csrc/ws_lowering.h) and micro-op interpreter
// (csrc/ws_vm.cuh, host instantiation) over host arrays, here with host tables: the memory image is the one
// ws_table uploads (wsl::table_image), used in place, so WS_OP_TABLE / WS_OP_CAT read it and count their index
// faults in its headers exactly as the kernels do on the device.
#include <stdint.h>
#include <string.h>
#include <map>
#include <string>
#include <vector>
#include "../../weightedsampling.jl_b200/csrc/ws_lowering.h"

using wsl::Plane;
using wsl::Program;

struct TH {
    int64_t n;
    uint64_t seed, next_stream = 1;
    int64_t cur_n = 0, cur_u = 0, cur_e = 0, cur_v = 0;
    std::vector<std::vector<std::vector<double>>> cols;  // [col][comp][i]
    std::vector<double> logw, ru;
    std::vector<std::vector<double>> images;              // one table image per id
    std::vector<wsl::TableRef> tables;
    std::map<std::string, int32_t> table_ids;
    Program win, score;
    std::string err;
};

static void reset(TH* h) {
    h->win = Program();
    h->win.tables = &h->tables;
}

static void run_program(TH* h, const Program& p, std::vector<double>* acc_out) {
    WsRng rng;
    rng.seed = h->seed;
    rng.replay_n = nullptr;
    rng.replay_u = h->ru.empty() ? nullptr : h->ru.data();
    rng.replay_e = nullptr;
    rng.replay_v = nullptr;
    std::vector<double> R((size_t)std::max(1, p.high_water));
    for (int64_t i = 0; i < h->n; ++i) {
        for (auto& ld : p.loads) R[ld.second] = h->cols[ld.first.col][ld.first.comp][(size_t)i];
        double acc[1] = {0.0};
        const uint64_t pid[1] = {(uint64_t)i};
        for (const WsOp& o : p.ops) ws_vm_exec<1, 1>(o, R.data(), acc, rng, pid);
        for (auto& d : p.dirty) h->cols[d.col][d.comp][(size_t)i] = R[p.plane_reg.at(d)];
        if (acc_out) (*acc_out)[(size_t)i] += acc[0];
    }
}

static int finish(TH* h, Program& p) {
    if (!p.error.empty()) {
        h->err = p.error;
        return -1;
    }
    p.end_statement();
    return 0;
}

extern "C" {

TH* th_new(int64_t n, uint64_t seed) {
    TH* h = new TH();
    h->n = n;
    h->seed = seed;
    h->logw.assign((size_t)n, 0.0);
    reset(h);
    h->score.tables = &h->tables;
    h->score.score_mode = true;
    h->score.n_temp_slots = 12;
    h->score.max_regs = 200;
    h->score.max_ops = 1 << 30;
    h->score.max_io = 1 << 30;
    return h;
}
void th_free(TH* h) { delete h; }
const char* th_error(TH* h) { return h->err.c_str(); }
int th_col(TH* h, int width) {
    h->cols.push_back(std::vector<std::vector<double>>(width, std::vector<double>((size_t)h->n, 0.0)));
    return (int)h->cols.size() - 1;
}
void th_set_plane(TH* h, int col, int comp, const double* v) { memcpy(h->cols[col][comp].data(), v, sizeof(double) * h->n); }
void th_set_replay_uniforms(TH* h, const double* u, int64_t nu) { h->ru.assign(u, u + nu); }
int th_table(TH* h, const double* values, int64_t n_rows, int32_t n_cols, int32_t* id_out) {
    if (n_rows < 1 || n_cols < 1 || n_cols > WS_TABLE_MAX_COLS) return -5;
    std::string key((const char*)&n_cols, sizeof n_cols);
    key.append((const char*)values, sizeof(double) * (size_t)n_rows * (size_t)n_cols);
    auto it = h->table_ids.find(key);
    if (it != h->table_ids.end()) {
        *id_out = it->second;
        return 0;
    }
    h->images.push_back(wsl::table_image(values, n_rows, n_cols));
    h->tables.push_back(wsl::table_ref_at(h->images.back().data(), n_rows, n_cols));
    *id_out = (int32_t)h->tables.size() - 1;
    h->table_ids.emplace(key, *id_out);
    return 0;
}
int th_flush(TH* h) {
    if (h->win.ops.empty() && h->win.dirty.empty()) return 0;
    run_program(h, h->win, h->win.has_acc ? &h->logw : nullptr);
    reset(h);
    return 0;
}
int64_t th_index_faults(TH* h) {
    th_flush(h);
    int64_t s = 0;
    for (size_t t = 0; t < h->images.size(); ++t) {
        const size_t seg = wsl::table_segment(h->tables[t].n_rows, h->tables[t].n_cols);
        for (int k = 0; k < 3; ++k) s += (int64_t)reinterpret_cast<const WsTableHdr*>(h->images[t].data() + k * seg)->faults;
    }
    return s;
}
void th_get_plane(TH* h, int col, int comp, double* out) {
    th_flush(h);
    memcpy(out, h->cols[col][comp].data(), sizeof(double) * h->n);
}
void th_get_logw(TH* h, double* out) {
    th_flush(h);
    memcpy(out, h->logw.data(), sizeof(double) * h->n);
}
int th_window_ops(TH* h) { return (int)h->win.ops.size(); }

int th_assign(TH* h, int col, int comp, const ws_expr* rhs) {
    wsl::stmt_assign(h->win, Plane{col, comp}, *rhs);
    return finish(h, h->win);
}
int th_observe_normal(TH* h, const ws_expr* obs, const ws_expr* mu, const ws_expr* sigma) {
    wsl::stmt_observe_normal(h->win, *obs, *mu, *sigma);
    wsl::stmt_observe_normal(h->score, *obs, *mu, *sigma);
    if (finish(h, h->score) != 0) return -1;
    return finish(h, h->win);
}
int th_weight_expr(TH* h, const ws_expr* term) {
    wsl::stmt_weight_expr(h->win, *term);
    wsl::stmt_weight_expr(h->score, *term);
    if (finish(h, h->score) != 0) return -1;
    return finish(h, h->win);
}
int th_sample_expr(TH* h, int col, int comp, const ws_expr* sampler, const ws_expr* weighter, const ws_expr* logpdf) {
    wsl::RngCursor rc{&h->next_stream, &h->cur_n, &h->cur_u, &h->cur_e, h->n, &h->cur_v};
    wsl::stmt_sample_expr(h->win, rc, Plane{col, comp}, *sampler, weighter);
    if (logpdf) {
        wsl::stmt_weight_expr(h->score, *logpdf);
        if (finish(h, h->score) != 0) return -1;
    }
    return finish(h, h->win);
}
// the score tape folded at the current column values (every recorded entry)
int th_score(TH* h, double* out) {
    th_flush(h);
    std::vector<double> acc((size_t)h->n, 0.0);
    run_program(h, h->score, &acc);
    memcpy(out, acc.data(), sizeof(double) * h->n);
    return 0;
}
int th_score_ops(TH* h) { return (int)h->score.ops.size(); }

}  // extern "C"
