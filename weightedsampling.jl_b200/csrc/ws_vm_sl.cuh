// ws_vm_sl.cuh — straight-line executors of the fused elementwise window.
//
// ws_vm_kernel (ws_kernels.cu) interprets ANY lowered window: its per-particle register file lives in shared
// memory and every micro-op is fetched, decoded and dispatched at run time — ~14 instructions of overhead per
// op and two shared-memory accesses per operand (profiles/r1z_ncu_ws_vm_kernel_20M.txt: 81 M shared wavefronts,
// issue-bound at 528 instructions per particle for the 2-D SSM step).  The windows that carry the benchmarks are
// a handful of fixed op patterns (the step of examples/2D_ssm.jl, of benchmarks/ssm/.../lgssm1d.jl, of
// examples/1D_ssm.jl, the observe of examples/linear_regression.jl).  For those the pattern — op codes and
// register numbers, NOT the constants — is a compile-time signature: the register file is a local array whose
// every index is a constant after unrolling, i.e. it lives in registers, there is no decode and no dispatch, and
// the arithmetic is the interpreter's own (the very same ws_vm_exec_d, inlined with a constant op), so results
// are bit-identical to the interpreted window (tests/test_gpu_parity.py::test_straight_line_equals_interpreter).
// Constants (k0, k1, k2), plane pointers, ancestors and the RNG description still come from the WsVmProgram of
// the launch.  A window that matches no signature runs on the interpreter as before.
#pragma once
#include <cmath>
#include <utility>
#include "ws_vm.cuh"
#if defined(__CUDACC__)
#include "ws_internal.h"
#endif

// one op of a signature, registers in CANONICAL numbering: registers are numbered in order of first appearance,
// scanning the window's loads first and then each op's (dst, a, b, c); fields an op does not use are WS_REG_NONE
#if defined(__CUDACC__)
#define WS_SL_CX __host__ __device__ constexpr
#else
#define WS_SL_CX constexpr
#endif
struct WsSlOp {
    uint8_t op, dst, a, b, c;
    uint32_t imm;
    uint8_t kflags;   // WS_SL_K*: constants whose VALUE is part of the signature (0 or 1), see ws_sl_step
};
// `x .= x + v` lowers to LIN2 with (k0, k1, k2) = (0, 1, 1) and `dv = L z` to (0, L, -): when the signature pins those
// values the executor sees literal 0.0 / 1.0 and the op is one DADD / DMUL instead of two DFMAs whose constants are
// fetched from the launch parameters every tile (IEEE-identical: 1*a and fma(k, a, 0) are exact)
#define WS_SL_K0Z 1u     // k0 == 0.0
#define WS_SL_K1ONE 2u   // k1 == 1.0
#define WS_SL_K2ONE 4u   // k2 == 1.0
#define WS_SL_ADD (WS_SL_K0Z | WS_SL_K1ONE | WS_SL_K2ONE)

WS_SL_CX bool ws_sl_dst_is_reg(uint32_t op) {
    return !(op == WS_OP_LOGPDF_NORMAL || op == WS_OP_LOGPDF_EXPON || op == WS_OP_ACC_LIN2 || op == WS_OP_ACC_QUAD2 ||
             op == WS_OP_ACC_SCALE || op == WS_OP_LOGPDF_NORMAL_CS || op == WS_OP_ACC_SQLIN2);
}
// does the random-number op take its `imm` from the launch (replay component index)?  imm is then not part of the signature
WS_SL_CX bool ws_sl_imm_is_runtime(uint32_t op) { return op == WS_OP_RANDN2 || op == WS_OP_RANDEXP || op == WS_OP_RANDU; }

#define WS_SL_N 0xFFu

// ---- the signatures -------------------------------------------------------------------------------------------
// examples/2D_ssm.jl:11-16, filter-only form:  x .= x + v ; dv ~ MvNormal(0, s I) ; v .= v + dv ; o => MvNormal(x, r I)
struct WsSigSsm2d {
    static constexpr int n_loads = 4, n_stores = 6, n_regs = 8, n_ops = 10;
    static constexpr uint8_t load_reg[4] = {0, 1, 2, 3};            // x1 v1 x2 v2
    static constexpr uint8_t store_reg[6] = {0, 2, 6, 7, 1, 3};     // x1 x2 dv1 dv2 v1 v2
    static constexpr WsSlOp ops[10] = {
        {WS_OP_LIN2, 0, 0, 1, WS_SL_N, 0, WS_SL_ADD},        // x1 += v1
        {WS_OP_LIN2, 2, 2, 3, WS_SL_N, 0, WS_SL_ADD},        // x2 += v2
        {WS_OP_RANDN2, 4, 5, WS_SL_N, WS_SL_N, 0},  // z1, z2
        {WS_OP_LIN2, 6, 4, WS_SL_N, WS_SL_N, 0, WS_SL_K0Z},  // dv1 = L11 z1
        {WS_OP_LIN2, 7, 5, WS_SL_N, WS_SL_N, 0, WS_SL_K0Z},  // dv2 = L22 z2
        {WS_OP_LIN2, 1, 1, 6, WS_SL_N, 0, WS_SL_ADD},        // v1 += dv1
        {WS_OP_LIN2, 3, 3, 7, WS_SL_N, 0, WS_SL_ADD},        // v2 += dv2
        {WS_OP_LIN2, 4, 0, WS_SL_N, WS_SL_N, 0},  // whitened residual 1
        {WS_OP_LIN2, 5, 2, WS_SL_N, WS_SL_N, 0},  // whitened residual 2
        {WS_OP_ACC_QUAD2, WS_SL_N, 4, 5, WS_SL_N, 0},
    };
};
// examples/2D_ssm.jl:11-16 verbatim (history kept):  x{t+1} .= x{t} + v ; dv ~ ... ; v .= v + dv ; o => MvNormal(x{t+1}, r I)
struct WsSigSsm2dHist {
    static constexpr int n_loads = 4, n_stores = 6, n_regs = 10, n_ops = 10;
    static constexpr uint8_t load_reg[4] = {0, 1, 2, 3};            // x{t}1 v1 x{t}2 v2
    static constexpr uint8_t store_reg[6] = {4, 5, 8, 9, 1, 3};     // x{t+1}1 x{t+1}2 dv1 dv2 v1 v2
    static constexpr WsSlOp ops[10] = {
        {WS_OP_LIN2, 4, 0, 1, WS_SL_N, 0, WS_SL_ADD},
        {WS_OP_LIN2, 5, 2, 3, WS_SL_N, 0, WS_SL_ADD},
        {WS_OP_RANDN2, 6, 7, WS_SL_N, WS_SL_N, 0},
        {WS_OP_LIN2, 8, 6, WS_SL_N, WS_SL_N, 0, WS_SL_K0Z},
        {WS_OP_LIN2, 9, 7, WS_SL_N, WS_SL_N, 0, WS_SL_K0Z},
        {WS_OP_LIN2, 1, 1, 8, WS_SL_N, 0, WS_SL_ADD},
        {WS_OP_LIN2, 3, 3, 9, WS_SL_N, 0, WS_SL_ADD},
        {WS_OP_LIN2, 6, 4, WS_SL_N, WS_SL_N, 0},
        {WS_OP_LIN2, 7, 5, WS_SL_N, WS_SL_N, 0},
        {WS_OP_ACC_QUAD2, WS_SL_N, 6, 7, WS_SL_N, 0},
    };
};
// benchmarks/ssm/WeightedSampling/lgssm1d.jl:20-23:  x ~ Normal(a x, q) ; y => Normal(x, r)
struct WsSigLgssm1d {
    static constexpr int n_loads = 1, n_stores = 1, n_regs = 2, n_ops = 3;
    static constexpr uint8_t load_reg[1] = {0};
    static constexpr uint8_t store_reg[1] = {0};
    static constexpr WsSlOp ops[3] = {
        {WS_OP_RANDN2, 1, WS_SL_N, WS_SL_N, WS_SL_N, 0},
        {WS_OP_LIN2, 0, 0, 1, WS_SL_N, 0, WS_SL_K0Z},
        {WS_OP_LOGPDF_NORMAL_CS, WS_SL_N, WS_SL_N, 0, WS_SL_N, 0},
    };
};
// examples/1D_ssm.jl:10-15, filter-only form:  x .= x + v ; dv ~ Normal(0, s) ; v .= v + dv ; o => Normal(x, r)
struct WsSigSsm1d {
    static constexpr int n_loads = 2, n_stores = 3, n_regs = 4, n_ops = 5;
    static constexpr uint8_t load_reg[2] = {0, 1};
    static constexpr uint8_t store_reg[3] = {0, 3, 1};
    static constexpr WsSlOp ops[5] = {
        {WS_OP_LIN2, 0, 0, 1, WS_SL_N, 0, WS_SL_ADD},
        {WS_OP_RANDN2, 2, WS_SL_N, WS_SL_N, WS_SL_N, 0},
        {WS_OP_LIN2, 3, 2, WS_SL_N, WS_SL_N, 0, WS_SL_K0Z},
        {WS_OP_LIN2, 1, 1, 3, WS_SL_N, 0, WS_SL_ADD},
        {WS_OP_LOGPDF_NORMAL_CS, WS_SL_N, WS_SL_N, 0, WS_SL_N, 0},
    };
};
// examples/linear_regression.jl:21:  y => Normal(alpha + beta * x_i, sigma)   (observe only: nothing is stored)
struct WsSigLinregObs {
    static constexpr int n_loads = 2, n_stores = 0, n_regs = 3, n_ops = 2;
    static constexpr uint8_t load_reg[2] = {0, 1};
    static constexpr uint8_t store_reg[1] = {0};
    static constexpr WsSlOp ops[2] = {
        {WS_OP_LIN2, 2, 0, 1, WS_SL_N, 0, WS_SL_K0Z | WS_SL_K1ONE},
        {WS_OP_LOGPDF_NORMAL_CS, WS_SL_N, WS_SL_N, 2, WS_SL_N, 0},
    };
};

// the table: index = what ws_sl_find returns
#define WS_SL_SIGS(X) X(0, WsSigSsm2d) X(1, WsSigSsm2dHist) X(2, WsSigLgssm1d) X(3, WsSigSsm1d) X(4, WsSigLinregObs)

// ---- matching (host) ------------------------------------------------------------------------------------------
// canonical renumbering of a launch's registers.  `Prog` is WsVmProgram (or the CPU test harness's view of a
// queued window with the same fields: n_ops, n_loads, n_stores, n_expect, load_reg, store_reg, ops)
template <class Prog>
inline void ws_sl_canonical(const Prog& P, uint8_t (&map)[256]) {
    for (int i = 0; i < 256; ++i) map[i] = WS_SL_N;
    int next = 0;
    auto see = [&](uint32_t r) {
        if (r != WS_REG_NONE && map[r] == WS_SL_N) map[r] = (uint8_t)next++;
    };
    for (int k = 0; k < P.n_loads; ++k) see(P.load_reg[k]);
    for (int i = 0; i < P.n_ops; ++i) {
        const WsOp& o = P.ops[i];
        const uint32_t op = o.w0 & 0xFFu;
        if (ws_sl_dst_is_reg(op)) see((o.w0 >> 8) & 0xFFu);
        see((o.w0 >> 16) & 0xFFu);
        see((o.w0 >> 24) & 0xFFu);
        see(o.w1 & 0xFFu);
    }
}

// Table reads and Categorical draws (WS_OP_TABLE, WS_OP_CAT) dereference a table address and may count index faults:
// no signature has them, and a window that contains one always runs on the interpreter
template <class Prog>
inline bool ws_sl_has_table_ops(const Prog& P, int n_ops) {
    for (int i = 0; i < n_ops; ++i) {
        const uint32_t op = P.ops[i].w0 & 0xFFu;
        if (op == WS_OP_TABLE || op == WS_OP_CAT) return true;
    }
    return false;
}

template <class Sig, class Prog>
inline bool ws_sl_matches(const Prog& P, const uint8_t (&map)[256]) {
    if (P.n_expect != 0 || P.n_ops != Sig::n_ops || P.n_loads != Sig::n_loads || P.n_stores != Sig::n_stores) return false;
    for (int k = 0; k < Sig::n_loads; ++k)
        if (map[P.load_reg[k]] != Sig::load_reg[k]) return false;
    for (int k = 0; k < Sig::n_stores; ++k)
        if (map[P.store_reg[k]] != Sig::store_reg[k]) return false;
    auto canon = [&](uint32_t r) -> uint8_t { return r == WS_REG_NONE ? (uint8_t)WS_SL_N : map[r]; };
    for (int i = 0; i < Sig::n_ops; ++i) {
        const WsOp& o = P.ops[i];
        const WsSlOp s = Sig::ops[i];
        const uint32_t op = o.w0 & 0xFFu;
        if (op != s.op) return false;
        if (ws_sl_dst_is_reg(op) && canon((o.w0 >> 8) & 0xFFu) != s.dst) return false;
        if (canon((o.w0 >> 16) & 0xFFu) != s.a || canon((o.w0 >> 24) & 0xFFu) != s.b || canon(o.w1 & 0xFFu) != s.c) return false;
        if (!ws_sl_imm_is_runtime(op) && (o.w1 >> 8) != s.imm) return false;
        if ((s.kflags & WS_SL_K0Z) && !(o.k0 == 0.0 && !std::signbit(o.k0))) return false;
        if ((s.kflags & WS_SL_K1ONE) && o.k1 != 1.0) return false;
        if ((s.kflags & WS_SL_K2ONE) && o.k2 != 1.0) return false;
    }
    return true;
}

// A checkpointed window (speculative block) that is the signature's window repeated n_ckpt times, a checkpoint behind
// every repetition: each repetition is matched on its own under the register numbering of the first.
template <class Sig, class Prog>
inline bool ws_sl_matches_repeated(const Prog& P, int max_reps) {
    struct View {
        int n_ops, n_loads, n_stores, n_expect;
        const uint8_t* load_reg;
        const uint8_t* store_reg;
        const WsOp* ops;
    };
    const int r = P.n_ckpt;
    if (r < 1 || r > max_reps || Sig::n_stores != 0 || P.n_stores != 0 || P.n_ops != r * Sig::n_ops) return false;
    if (ws_sl_has_table_ops(P, P.n_ops)) return false;
    for (int j = 0; j < r; ++j)
        if ((int)P.ckpt_pc[j] != (j + 1) * Sig::n_ops - 1) return false;
    View v{Sig::n_ops, P.n_loads, 0, P.n_expect, P.load_reg, P.store_reg, P.ops};
    uint8_t map[256];
    ws_sl_canonical(v, map);
    for (int j = 0; j < r; ++j) {
        v.ops = P.ops + j * Sig::n_ops;
        if (!ws_sl_matches<Sig>(v, map)) return false;
    }
    return true;
}

template <class Prog>
inline int ws_sl_find(const Prog& P) {
    if (ws_sl_has_table_ops(P, P.n_ops)) return -1;
    uint8_t map[256];
    ws_sl_canonical(P, map);
#define WS_SL_TRY(idx, Sig) \
    if (ws_sl_matches<Sig>(P, map)) return idx;
    WS_SL_SIGS(WS_SL_TRY)
#undef WS_SL_TRY
    return -1;
}

#if defined(__CUDACC__)
// ---- execution (device) -----------------------------------------------------------------------------------------
// op I of the signature applied to the thread's PP particles; R = [n_regs][PP] doubles, all indices constant
// Does op `s` read constant k_j (0, 1, 2) at run time?  (not pinned by a value flag, and actually used by the op's form)
WS_SL_CX bool ws_sl_uses_k(const WsSlOp& s, int j) {
    const bool has_a = s.a != WS_SL_N, has_b = s.b != WS_SL_N;
    switch (s.op) {
        case WS_OP_LIN2:
            if (j == 0) return !(s.kflags & WS_SL_K0Z);
            if (j == 1) return (has_a && !(s.kflags & WS_SL_K1ONE));
            return has_b && !(s.kflags & WS_SL_K2ONE);       // (k2 of a b-only LIN2 is read as k1 after the swap)
        case WS_OP_RANDN2:
        case WS_OP_RANDEXP:
        case WS_OP_RANDU: return j == 0;                      // the Philox stream; replay offsets (k1, k2) stay in the parameters
        case WS_OP_LOGPDF_NORMAL_CS: return j != 0 || !has_a;
        case WS_OP_ACC_QUAD2:
        case WS_OP_ACC_LIN2:
        case WS_OP_ACC_SQLIN2: return j == 0 || (j == 1 && has_a) || (j == 2 && has_b);
        default: return true;
    }
}
// The constants of the window, read from the launch parameters ONCE per thread and pinned in registers: inside the tile
// loop the compiler otherwise re-fetches them from the (3.6 KB) parameter block every tile, and the constant-cache
// miss of one such fetch was the largest single stall of the kernel (profiles/r2d_ncu_ws_vm_sl_kernel_20M.txt:
// LDCU.64 -> DFMA, 29 % of the samples).
template <class Sig>
struct WsSlConsts {
    double k[Sig::n_ops][3];
};
template <class Sig, int I>
__device__ __forceinline__ void ws_sl_load_const1(WsSlConsts<Sig>& K, const WsVmProgram& P) {
    constexpr WsSlOp s = Sig::ops[I];
    constexpr bool u0 = ws_sl_uses_k(s, 0), u1 = ws_sl_uses_k(s, 1), u2 = ws_sl_uses_k(s, 2);
    K.k[I][0] = u0 ? P.ops[I].k0 : 0.0;
    K.k[I][1] = u1 ? P.ops[I].k1 : 0.0;
    K.k[I][2] = u2 ? P.ops[I].k2 : 0.0;
#ifndef WS_SL_NOPIN   // (A/B switch)
    if (u0) asm volatile("" : "+d"(K.k[I][0]));   // opaque from here on: cannot be rematerialised from constant memory
    if (u1) asm volatile("" : "+d"(K.k[I][1]));
    if (u2) asm volatile("" : "+d"(K.k[I][2]));
#endif
}
template <class Sig, int... I>
__device__ __forceinline__ void ws_sl_load_consts(WsSlConsts<Sig>& K, const WsVmProgram& P, std::integer_sequence<int, I...>) {
    (ws_sl_load_const1<Sig, I>(K, P), ...);
}

template <class Sig, int I, int PP>
__device__ __forceinline__ void ws_sl_step(double* __restrict__ R, double (&acc)[PP], const WsOp& o, const double (&kk)[3],
                                           const bool replay, const WsRng& rng, const uint64_t (&particle)[PP]) {
    constexpr WsSlOp s = Sig::ops[I];
    constexpr bool lin2 = s.op == WS_OP_LIN2;
    constexpr bool swap = lin2 && s.a == WS_SL_N && s.b != WS_SL_N;  // k0 + k2*r[b]: executed as k0 + k1'*r[a'] (ws_decode_op)
    constexpr uint8_t ra = swap ? s.b : s.a, rb = swap ? (uint8_t)WS_SL_N : s.b;
    WsDop d;
    d.op = !lin2 ? (uint32_t)s.op
                 : (ra == WS_SL_N ? (uint32_t)WS_DOP_LIN2_K : (rb == WS_SL_N ? (uint32_t)WS_DOP_LIN2_A : (uint32_t)WS_DOP_LIN2_AB));
    d.dst = (s.dst == WS_SL_N) ? WS_OFF_NONE : (uint32_t)s.dst * PP;
    d.a = (ra == WS_SL_N) ? WS_OFF_NONE : (uint32_t)ra * PP;
    d.b = (rb == WS_SL_N) ? WS_OFF_NONE : (uint32_t)rb * PP;
    d.c = (s.c == WS_SL_N) ? WS_OFF_NONE : (uint32_t)s.c * PP;
    constexpr bool rt_imm = ws_sl_imm_is_runtime(s.op);
    d.imm = rt_imm ? (o.w1 >> 8) : s.imm;
    // (a swapped LIN2 carries no value flags in any signature)
    constexpr bool rnd = ws_sl_imm_is_runtime(s.op);
    d.k0 = (s.kflags & WS_SL_K0Z) ? 0.0 : kk[0];
    d.k1 = (s.kflags & WS_SL_K1ONE) ? 1.0 : (swap ? kk[2] : kk[1]);
    d.k2 = (s.kflags & WS_SL_K2ONE) ? 1.0 : kk[2];
    if (rnd && replay) {          // replayed draws (tests): offsets of the draw in the replay buffers
        d.k1 = o.k1;
        d.k2 = o.k2;
    }
    ws_vm_exec_d<1, PP>(d, R, acc, rng, particle);
}
// register <- staging row K (the plane loads of this tile), and plane <- register for store K: the register numbers
// are read in constant expressions (a signature's tables do not exist in device memory)
template <class Sig, int PP, int BLOCK, int K>
__device__ __forceinline__ void ws_sl_load1(double* __restrict__ R, const double* __restrict__ stage) {
    constexpr int r = Sig::load_reg[K];
#pragma unroll
    for (int j = 0; j < PP; ++j) R[r * PP + j] = stage[(K * PP + j) * BLOCK];
}
template <class Sig, int PP, int BLOCK, int... K>
__device__ __forceinline__ void ws_sl_loads(double* __restrict__ R, const double* __restrict__ stage, std::integer_sequence<int, K...>) {
    (ws_sl_load1<Sig, PP, BLOCK, K>(R, stage), ...);
}
// plane K <- register: the thread's particles sit BLOCK apart, so one address per plane and constant offsets
template <class Sig, int PP, int BLOCK, int K>
__device__ __forceinline__ void ws_sl_store1(const double* __restrict__ R, const WsVmProgram& P, const unsigned first, const bool (&live)[PP]) {
    constexpr int r = Sig::store_reg[K];
    double* __restrict__ ptr = P.store_ptr[K] + first;
#pragma unroll
    for (int j = 0; j < PP; ++j)
        if (live[j]) ptr[j * BLOCK] = R[r * PP + j];
}
template <class Sig, int PP, int BLOCK, int... K>
__device__ __forceinline__ void ws_sl_stores(const double* __restrict__ R, const WsVmProgram& P, const unsigned first, const bool (&live)[PP],
                                             std::integer_sequence<int, K...>) {
    (ws_sl_store1<Sig, PP, BLOCK, K>(R, P, first, live), ...);
}
template <class Sig, int PP, int... I>
__device__ __forceinline__ void ws_sl_run(double* __restrict__ R, double (&acc)[PP], const WsVmProgram& P, const WsSlConsts<Sig>& K,
                                          const bool replay, const uint64_t (&particle)[PP], std::integer_sequence<int, I...>) {
    (ws_sl_step<Sig, I, PP>(R, acc, P.ops[I], K.k[I], replay, P.rng, particle), ...);
}
// the same for one repetition of a repeated window: its micro-ops start at `ops`
template <class Sig, int PP, int... I>
__device__ __forceinline__ void ws_sl_run_at(double* __restrict__ R, double (&acc)[PP], const WsVmProgram& P, const WsOp* ops,
                                             const WsSlConsts<Sig>& K, const uint64_t (&particle)[PP], std::integer_sequence<int, I...>) {
    (ws_sl_step<Sig, I, PP>(R, acc, ops[I], K.k[I], false, P.rng, particle), ...);
}
#endif
