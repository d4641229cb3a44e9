// ws_vm.cuh — the fixed device-op set ("micro-ops") and its in-kernel interpreter.
//
// The reference runs every model statement as one fused Julia broadcast over all particles
// (src/transformers.jl: Assign :28-32, Sample :172-182, Observe :228-235, Weight :283-289,
// AccessorSample :118-131).  Here a window of consecutive statements is lowered by the host
// runtime (ws_runtime.cu: Lowering) to a short program of the micro-ops below and executed
// in ONE pass over the particles: plane values live in a per-thread register file in shared
// memory for the whole window, so each plane is read and written at most once per window.
//
// The same interpreter folds the score tape inside the MH kernel (ws_kernels_move.cu), which
// is the device form of the reference's score! walk (src/transformers.jl:39,77,139,193,243,297).
#pragma once
#include <string.h>
#include "ws_math.cuh"

#define WS_REG_NONE 0xFFu

enum WsOpCode : uint32_t {
    WS_OP_LIN2 = 0,         // r[dst] = k0 + k1*r[a] + k2*r[b]        (a / b == NONE: term absent)
    WS_OP_MUL = 1,          // r[dst] = k0 * A * B       A = a==NONE ? k1 : r[a];  B = b==NONE ? k2 : r[b]
    WS_OP_DIV = 2,          // r[dst] = k0 * A / B
    WS_OP_UNARY = 3,        // r[dst] = f_imm(A)
    WS_OP_POW = 4,          // r[dst] = pow(A, B)
    WS_OP_RANDN2 = 5,       // r[dst] (, r[a]) = standard normals
    WS_OP_RANDEXP = 6,      // r[dst] = standard exponential
    WS_OP_RANDU = 7,        // r[dst] = uniform [0,1)
    WS_OP_LOGPDF_NORMAL = 8,  // acc += logN(X; MU, SIGMA)   X = a==NONE?k0:r[a]; MU = b==NONE?k1:r[b]; SIGMA = c==NONE?k2:r[c]
    WS_OP_LOGPDF_EXPON = 9,   // acc += logExp(X; THETA)     X = a==NONE?k0:r[a]; THETA = b==NONE?k1:r[b]
    WS_OP_ACC_LIN2 = 10,      // acc += k0 + k1*r[a] + k2*r[b]
    WS_OP_ACC_QUAD2 = 11,     // acc += k0 + k1*r[a]^2 + k2*r[b]^2
    WS_OP_ACC_SCALE = 12,     // acc = k0 * acc   (used to negate a proposal log-density)
    WS_OP_LOGPDF_NORMAL_CS = 13,  // constant sigma: acc += k2 - 0.5*((X - r[b])*k1)^2,  X = a==NONE?k0:r[a]
    WS_OP_CMP = 14,      // r[dst] = (A op B) ? 1 : 0     imm: 0 <, 1 <=, 2 ==      A = a==NONE?k1:r[a]; B = b==NONE?k2:r[b]
    WS_OP_SELECT = 15,   // r[dst] = (r[c] != 0) ? A : B
    WS_OP_MINMAX = 16,   // r[dst] = imm ? max(A,B) : min(A,B)
    WS_OP_ACC_SQLIN2 = 17  // acc -= (k0 + k1*r[a] + k2*r[b])^2 / 2   (a / b == NONE: term absent).  A Normal log-density
                           // with constant sigma and an affine mean, minus its constant, in ONE op (score tapes)
    ,
    WS_OP_ACC_SQLIN2_S = 18  // acc -= ((k0 + k1*r[a] + k2*r[b]) * r[c])^2 / 2 + r[dst]: the same with a per-particle sigma
                             // whose reciprocal r[c] and logarithm r[dst] were computed once per fold (score tapes)
    ,
    WS_OP_RANDV = 19  // r[dst] = variate with a parameter A = a==NONE ? k2 : r[a];  imm: 0 standard Gamma(shape A),
                      // 1 Poisson(A).  k0 = Philox stream; replay: r[dst] = replay_v[(int64)k1 + particle]
    ,
    WS_OP_TABLE = 20  // r[dst] = T[(ROW-1)*n_cols + (COL-1)]   ROW = a==NONE ? k1 : r[a];  COL = b==NONE ? k2 : r[b];
                      // k0 = the table's device address (bit-cast), imm = n_cols | WS_TABLE_LOGP (see ws_table_read)
    ,
    WS_OP_CAT = 21  // r[dst] = 1 + #{k < K : C[(ROW-1)*K + k-1] <= U}   U = r[a];  ROW = b==NONE ? k1 : r[b];
                    // k0 = the address of the table's row-wise partial sums C (bit-cast), imm = K (ws_cat_draw)
};

enum WsUnary : uint32_t {
    WS_UN_EXP = 0,
    WS_UN_LOG = 1,
    WS_UN_SQRT = 2,
    WS_UN_SIN = 3,
    WS_UN_COS = 4,
    WS_UN_ABS = 5,
    WS_UN_SQUARE = 6,
    WS_UN_NOT = 7,
    WS_UN_LGAMMA = 8,
    WS_UN_LOG1P = 9,
    WS_UN_EXPM1 = 10,
    WS_UN_TAN = 11,
    WS_UN_ATAN = 12,
    WS_UN_TANH = 13,
    WS_UN_FLOOR = 14
};

// 32-byte micro-op; two 16-byte words so one uniform 128-bit load pair fetches it.
struct alignas(16) WsOp {
    uint32_t w0;  // op | dst<<8 | a<<16 | b<<24
    uint32_t w1;  // c | imm<<8 (24 bits)
    double k0, k1, k2;
};
static_assert(sizeof(WsOp) == 32, "WsOp must be 32 bytes");

// does the op use its dst field as a register?  (the pure accumulate ops leave it unused)
WS_HD bool ws_op_dst_is_reg(uint32_t op) {
    return !(op == WS_OP_LOGPDF_NORMAL || op == WS_OP_LOGPDF_EXPON || op == WS_OP_ACC_LIN2 || op == WS_OP_ACC_QUAD2 ||
             op == WS_OP_ACC_SCALE || op == WS_OP_LOGPDF_NORMAL_CS || op == WS_OP_ACC_SQLIN2);
}

WS_HD WsOp ws_make_op(uint32_t op, uint32_t dst, uint32_t a, uint32_t b, uint32_t c, uint32_t imm, double k0,
                      double k1, double k2) {
    WsOp o;
    o.w0 = (op & 0xFFu) | ((dst & 0xFFu) << 8) | ((a & 0xFFu) << 16) | ((b & 0xFFu) << 24);
    o.w1 = (c & 0xFFu) | ((imm & 0xFFFFFFu) << 8);
    o.k0 = k0;
    o.k1 = k1;
    o.k2 = k2;
    return o;
}

// Random-source description shared by every particle of a launch.
//   Philox mode : counter = (global particle index, stream id), key = seed.
//   replay mode : value = buf[base + particle*stride + j]  (reference consumption order,
//                 SURVEY.md §8c), base/stride/j come from the op.
struct WsRng {
    uint64_t seed;
    const double* replay_n;  // standard normals or nullptr
    const double* replay_u;  // uniforms or nullptr
    const double* replay_e;  // standard exponentials or nullptr
    const double* replay_v;  // already-accepted variates of the WS_OP_RANDV ops (standard Gamma(a_i) / Poisson(lam_i)) or nullptr
};

WS_HD uint64_t ws_double_bits(double v) {
#if defined(__CUDA_ARCH__)
    return (uint64_t)__double_as_longlong(v);
#else
    uint64_t b;
    memcpy(&b, &v, 8);
    return b;
#endif
}

// ---- build-time constant tables (WS_OP_TABLE, WS_OP_CAT; include/wsb200.h: ws_table) ------------------------------
// A device table is [WsTableHdr | n_rows * n_cols doubles, row-major]; the ops carry the address of the data, so the
// header is found just below it.  Indices are Julia's: 1-based integer-valued doubles.  Any other index (non-integer,
// out of range, NaN) reads nothing, gives NaN and counts one fault in the header (ws_get_index_faults sums them).
struct alignas(16) WsTableHdr {
    unsigned long long faults;
    int64_t n_rows;
};
#define WS_TABLE_MAX_COLS 65536
#define WS_TABLE_COLS_MASK 0x1FFFFu
// the column is the value of a Categorical: outside 1..n_cols it is outside the support, log-probability -Inf, no fault
#define WS_TABLE_LOGP (1u << 23)

WS_HD const double* ws_table_ptr(double k0) { return reinterpret_cast<const double*>((uintptr_t)ws_double_bits(k0)); }
WS_HD void ws_table_fault(const double* T) {
    unsigned long long* f = &(reinterpret_cast<WsTableHdr*>(const_cast<double*>(T)) - 1)->faults;
#if defined(__CUDA_ARCH__)
    atomicAdd(f, 1ull);
#else
    ++*f;
#endif
}
WS_HD bool ws_table_index_ok(double x, int64_t n) { return x >= 1.0 && x <= (double)n && x == floor(x); }
WS_HD double ws_table_read(const double* T, uint32_t imm, double row, double col) {
    const int64_t n_cols = (int64_t)(imm & WS_TABLE_COLS_MASK);
    const int64_t n_rows = (reinterpret_cast<const WsTableHdr*>(T) - 1)->n_rows;
    const bool row_ok = ws_table_index_ok(row, n_rows);
    if (row_ok && ws_table_index_ok(col, n_cols)) return T[((int64_t)row - 1) * n_cols + ((int64_t)col - 1)];
    if (row_ok && (imm & WS_TABLE_LOGP)) return -INFINITY;
    ws_table_fault(T);
    return NAN;
}
// Categorical(C's row) at uniform u: Distributions' `while cp <= u && i < K` walk over the sequential partial sums,
// i.e. 1 + the number of C_1 .. C_{K-1} that are <= u, found by a binary search (C is non-decreasing)
WS_HD double ws_cat_draw(const double* C, uint32_t K, double row, double u) {
    const int64_t n_rows = (reinterpret_cast<const WsTableHdr*>(C) - 1)->n_rows;
    if (!ws_table_index_ok(row, n_rows)) {
        ws_table_fault(C);
        return NAN;
    }
    const double* c = C + ((int64_t)row - 1) * (int64_t)K;
    uint32_t lo = 0, hi = K - 1;  // count of c[0 .. K-2] that are <= u lies in [lo, hi]
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (c[mid] <= u) lo = mid + 1;
        else hi = mid;
    }
    return (double)(lo + 1);
}

// Decoded micro-op: what the interpreter executes.  The 32-byte WsOp is what the lowering emits and what
// travels (kernel parameters, the device score tape); unpacking it cost ~25 of the ~40 instructions a
// thread spent per micro-op outside the arithmetic (shifts, masks, register-row multiplies, the walk down
// the LIN2 sub-cases), so a CTA unpacks each op ONCE into shared memory (ws_decode_op) and its threads
// fetch the decoded form with three 16-byte loads:
//   * dst / a / b / c are element offsets into the thread's register-file column (reg * P * STRIDE),
//     WS_OFF_NONE where the operand is absent;
//   * LIN2 is split by operand pattern (constant / one term / two terms) so the hot op is one compare away.
#define WS_OFF_NONE 0xFFFFFFFFu
enum WsDopCode : uint32_t {
    WS_DOP_LIN2_K = 32,   // r[dst] = k0
    WS_DOP_LIN2_A = 33,   // r[dst] = k0 + k1*r[a]              (a LIN2 with only b present is stored swapped)
    WS_DOP_LIN2_AB = 34   // r[dst] = (k0 + k1*r[a]) + k2*r[b]
};
struct alignas(16) WsDop {
    uint32_t op, dst, a, b;
    uint32_t c, imm;
    double k0;
    double k1, k2;
};
static_assert(sizeof(WsDop) == 48, "WsDop must be 48 bytes");

// `reg_map` (optional): renumbering of the registers, so that a launch that folds part of a tape keeps only
// the register-file rows that part touches (ws_runtime.cu: compact_score_regs)
template <int STRIDE, int P>
WS_HD WsDop ws_decode_op(const WsOp& o, const uint8_t* reg_map = nullptr) {
    WsDop d;
    const uint32_t op = o.w0 & 0xFFu;
    const uint32_t r[4] = {(o.w0 >> 8) & 0xFFu, (o.w0 >> 16) & 0xFFu, (o.w0 >> 24) & 0xFFu, o.w1 & 0xFFu};
    uint32_t off[4];
    for (int k = 0; k < 4; ++k)
        off[k] = (r[k] == WS_REG_NONE) ? WS_OFF_NONE : (uint32_t)(reg_map ? reg_map[r[k]] : r[k]) * (uint32_t)(P * STRIDE);
    d.op = op;
    d.dst = off[0];
    d.a = off[1];
    d.b = off[2];
    d.c = off[3];
    d.imm = o.w1 >> 8;
    d.k0 = o.k0;
    d.k1 = o.k1;
    d.k2 = o.k2;
    if (op == WS_OP_LIN2) {
        if (d.a == WS_OFF_NONE && d.b == WS_OFF_NONE) {
            d.op = WS_DOP_LIN2_K;
        } else if (d.a == WS_OFF_NONE) {  // k0 + k2*r[b]: the same arithmetic with the operands renamed
            d.op = WS_DOP_LIN2_A;
            d.a = d.b;
            d.k1 = o.k2;
            d.b = WS_OFF_NONE;
        } else if (d.b == WS_OFF_NONE) {
            d.op = WS_DOP_LIN2_A;
        } else {
            d.op = WS_DOP_LIN2_AB;
        }
    }
    return d;
}

// Register file layout: register r of the thread's j-th particle lives at R[(r*P + j)*STRIDE], where R
// points at this thread's column of the shared-memory register file.  One decoded micro-op is applied
// to all P particles of the thread, which amortises the (warp-uniform) decode over P particles and
// gives P independent dependency chains per thread.  P = 1, STRIDE = 1 is the plain scalar form.
// (WS_HD: the host instantiation exists only for tests/host/, which runs lowered programs through
// this very interpreter on the CPU to check the lowering without a GPU.)
template <int STRIDE, int P>
WS_HD void ws_vm_exec_d(const WsDop& o, double* __restrict__ R, double (&acc)[P], const WsRng& rng,
                        const uint64_t (&particle)[P]) {
    const uint32_t op = o.op & 0xFFu;          // (bits 8.. : run length, see ws_vm_exec_sqlin2_run)
    const uint32_t a = o.a, b = o.b, c = o.c;  // element offsets (WS_OFF_NONE: operand absent, pointer unused)
    const uint32_t imm = o.imm;
    double* const Rd = R + o.dst;
    const double* const Ra = R + a;
    const double* const Rb = R + b;
    const double* const Rc = R + c;
    const double k0 = o.k0, k1 = o.k1, k2 = o.k2;
    // r = k0 + k1 a + k2 b is most of every program (sums, affine means, Cholesky rows, residuals)
    if (op >= WS_DOP_LIN2_K) {
        if (op == WS_DOP_LIN2_AB) {
#pragma unroll
            for (int j = 0; j < P; ++j) {
                double v = k0 + k1 * Ra[j * STRIDE];
                Rd[j * STRIDE] = v + k2 * Rb[j * STRIDE];
            }
        } else if (op == WS_DOP_LIN2_A) {
#pragma unroll
            for (int j = 0; j < P; ++j) Rd[j * STRIDE] = k0 + k1 * Ra[j * STRIDE];
        } else {
#pragma unroll
            for (int j = 0; j < P; ++j) Rd[j * STRIDE] = k0;
        }
        return;
    }
    switch (op) {
        case WS_OP_MUL: {
#pragma unroll
            for (int j = 0; j < P; ++j) {
                const double A = (a == WS_OFF_NONE) ? k1 : Ra[j * STRIDE];
                const double B = (b == WS_OFF_NONE) ? k2 : Rb[j * STRIDE];
                Rd[j * STRIDE] = k0 * A * B;
            }
        } break;
        case WS_OP_DIV: {
#pragma unroll
            for (int j = 0; j < P; ++j) {
                const double A = (a == WS_OFF_NONE) ? k1 : Ra[j * STRIDE];
                const double B = (b == WS_OFF_NONE) ? k2 : Rb[j * STRIDE];
                Rd[j * STRIDE] = k0 * A / B;
            }
        } break;
        case WS_OP_UNARY: {
#pragma unroll
            for (int j = 0; j < P; ++j) {
                const double A = (a == WS_OFF_NONE) ? k1 : Ra[j * STRIDE];
                double v;
                switch (imm) {
                    case WS_UN_EXP: v = exp(A); break;
                    case WS_UN_LOG: v = log(A); break;
                    case WS_UN_SQRT: v = sqrt(A); break;
                    case WS_UN_SIN: v = sin(A); break;
                    case WS_UN_COS: v = cos(A); break;
                    case WS_UN_ABS: v = fabs(A); break;
                    case WS_UN_NOT: v = (A == 0.0) ? 1.0 : 0.0; break;
                    case WS_UN_LGAMMA: v = lgamma(A); break;
                    case WS_UN_LOG1P: v = log1p(A); break;
                    case WS_UN_EXPM1: v = expm1(A); break;
                    case WS_UN_TAN: v = tan(A); break;
                    case WS_UN_ATAN: v = atan(A); break;
                    case WS_UN_TANH: v = tanh(A); break;
                    case WS_UN_FLOOR: v = floor(A); break;
                    default: v = A * A; break;
                }
                Rd[j * STRIDE] = v;
            }
        } break;
        case WS_OP_POW: {
#pragma unroll
            for (int j = 0; j < P; ++j) {
                const double A = (a == WS_OFF_NONE) ? k1 : Ra[j * STRIDE];
                const double B = (b == WS_OFF_NONE) ? k2 : Rb[j * STRIDE];
                Rd[j * STRIDE] = pow(A, B);
            }
        } break;
        case WS_OP_RANDN2: {
            if (rng.replay_n != nullptr) {
                // k1 = base offset, k2 = stride (both exact integers), imm = component j
#pragma unroll
                for (int j = 0; j < P; ++j) {
                    const int64_t base = (int64_t)k1 + (int64_t)particle[j] * (int64_t)k2 + (int64_t)imm;
                    Rd[j * STRIDE] = rng.replay_n[base];
                    if (a != WS_OFF_NONE) const_cast<double*>(Ra)[j * STRIDE] = rng.replay_n[base + 1];
                }
            } else {
                const uint64_t stream = ws_double_bits(k0);
#pragma unroll
                for (int j = 0; j < P; ++j) {
                    double z0, z1;
                    ws_randn2(particle[j], stream, rng.seed, z0, z1);
                    Rd[j * STRIDE] = z0;
                    if (a != WS_OFF_NONE) const_cast<double*>(Ra)[j * STRIDE] = z1;
                }
            }
        } break;
        case WS_OP_RANDEXP: {
#pragma unroll
            for (int j = 0; j < P; ++j) {
                double e;
                if (rng.replay_e != nullptr) {
                    e = rng.replay_e[(int64_t)k1 + (int64_t)particle[j] * (int64_t)k2 + (int64_t)imm];
                } else {
                    e = ws_randexp(particle[j], ws_double_bits(k0), rng.seed);
                }
                Rd[j * STRIDE] = e;
            }
        } break;
        case WS_OP_RANDU: {
#pragma unroll
            for (int j = 0; j < P; ++j) {
                double u;
                if (rng.replay_u != nullptr) {
                    u = rng.replay_u[(int64_t)k1 + (int64_t)particle[j] * (int64_t)k2 + (int64_t)imm];
                } else {
                    double u1;
                    ws_randu2(particle[j], ws_double_bits(k0), rng.seed, u, u1);
                }
                Rd[j * STRIDE] = u;
            }
        } break;
        case WS_OP_RANDV: {
#pragma unroll 1
            for (int j = 0; j < P; ++j) {
                double v;
                if (rng.replay_v != nullptr) {
                    v = rng.replay_v[(int64_t)k1 + (int64_t)particle[j]];
                } else {
                    const double A = (a == WS_OFF_NONE) ? k2 : Ra[j * STRIDE];
                    v = (imm == 0u) ? ws_rand_gamma(A, particle[j], ws_double_bits(k0), rng.seed)
                                    : ws_rand_poisson(A, particle[j], ws_double_bits(k0), rng.seed);
                }
                Rd[j * STRIDE] = v;
            }
        } break;
        case WS_OP_TABLE: {
            const double* T = ws_table_ptr(k0);
#pragma unroll
            for (int j = 0; j < P; ++j) {
                const double row = (a == WS_OFF_NONE) ? k1 : Ra[j * STRIDE];
                const double col = (b == WS_OFF_NONE) ? k2 : Rb[j * STRIDE];
                Rd[j * STRIDE] = ws_table_read(T, imm, row, col);
            }
        } break;
        case WS_OP_CAT: {
            const double* Ct = ws_table_ptr(k0);
#pragma unroll
            for (int j = 0; j < P; ++j) {
                const double row = (b == WS_OFF_NONE) ? k1 : Rb[j * STRIDE];
                Rd[j * STRIDE] = ws_cat_draw(Ct, imm, row, Ra[j * STRIDE]);
            }
        } break;
        case WS_OP_LOGPDF_NORMAL: {
#pragma unroll
            for (int j = 0; j < P; ++j) {
                const double X = (a == WS_OFF_NONE) ? k0 : Ra[j * STRIDE];
                const double MU = (b == WS_OFF_NONE) ? k1 : Rb[j * STRIDE];
                const double SG = (c == WS_OFF_NONE) ? k2 : Rc[j * STRIDE];
                acc[j] += ws_normal_logpdf(X, MU, SG);
            }
        } break;
        case WS_OP_LOGPDF_NORMAL_CS: {
            // constant sigma > 0, hoisted by the host: k1 = 1/sigma, k2 = -log(2pi)/2 - log(sigma).
            // D = X - MU with MU = r[b] (always a register) and X = r[a] or the constant k0.
#pragma unroll
            for (int j = 0; j < P; ++j) {
                const double X = (a == WS_OFF_NONE) ? k0 : Ra[j * STRIDE];
                const double z = (X - Rb[j * STRIDE]) * k1;
                acc[j] += k2 - 0.5 * (z * z);
            }
        } break;
        case WS_OP_LOGPDF_EXPON: {
#pragma unroll
            for (int j = 0; j < P; ++j) {
                const double X = (a == WS_OFF_NONE) ? k0 : Ra[j * STRIDE];
                const double TH = (b == WS_OFF_NONE) ? k1 : Rb[j * STRIDE];
                acc[j] += ws_exponential_logpdf(X, TH);
            }
        } break;
        case WS_OP_ACC_LIN2: {
#pragma unroll
            for (int j = 0; j < P; ++j) {
                double v = k0;
                if (a != WS_OFF_NONE) v += k1 * Ra[j * STRIDE];
                if (b != WS_OFF_NONE) v += k2 * Rb[j * STRIDE];
                acc[j] += v;
            }
        } break;
        case WS_OP_ACC_QUAD2: {
#pragma unroll
            for (int j = 0; j < P; ++j) {
                double v = k0;
                if (a != WS_OFF_NONE) {
                    const double t = Ra[j * STRIDE];
                    v += k1 * t * t;
                }
                if (b != WS_OFF_NONE) {
                    const double t = Rb[j * STRIDE];
                    v += k2 * t * t;
                }
                acc[j] += v;
            }
        } break;
        case WS_OP_CMP: {
#pragma unroll
            for (int j = 0; j < P; ++j) {
                const double A = (a == WS_OFF_NONE) ? k1 : Ra[j * STRIDE];
                const double B = (b == WS_OFF_NONE) ? k2 : Rb[j * STRIDE];
                const bool t = (imm == 0) ? (A < B) : ((imm == 1) ? (A <= B) : (A == B));
                Rd[j * STRIDE] = t ? 1.0 : 0.0;
            }
        } break;
        case WS_OP_SELECT: {
#pragma unroll
            for (int j = 0; j < P; ++j) {
                const double A = (a == WS_OFF_NONE) ? k1 : Ra[j * STRIDE];
                const double B = (b == WS_OFF_NONE) ? k2 : Rb[j * STRIDE];
                Rd[j * STRIDE] = (Rc[j * STRIDE] != 0.0) ? A : B;
            }
        } break;
        case WS_OP_MINMAX: {
#pragma unroll
            for (int j = 0; j < P; ++j) {
                const double A = (a == WS_OFF_NONE) ? k1 : Ra[j * STRIDE];
                const double B = (b == WS_OFF_NONE) ? k2 : Rb[j * STRIDE];
                Rd[j * STRIDE] = imm ? fmax(A, B) : fmin(A, B);
            }
        } break;
        case WS_OP_ACC_SQLIN2: {
#pragma unroll
            for (int j = 0; j < P; ++j) {
                double z = k0;
                if (a != WS_OFF_NONE) z += k1 * Ra[j * STRIDE];
                if (b != WS_OFF_NONE) z += k2 * Rb[j * STRIDE];
                acc[j] -= 0.5 * (z * z);
            }
        } break;
        case WS_OP_ACC_SQLIN2_S: {
#pragma unroll
            for (int j = 0; j < P; ++j) {
                double z = k0;
                if (a != WS_OFF_NONE) z += k1 * Ra[j * STRIDE];
                if (b != WS_OFF_NONE) z += k2 * Rb[j * STRIDE];
                z *= Rc[j * STRIDE];
                acc[j] -= 0.5 * (z * z) + Rd[j * STRIDE];
            }
        } break;
        case WS_OP_ACC_SCALE: {
#pragma unroll
            for (int j = 0; j < P; ++j) acc[j] = k0 * acc[j];
        } break;
        default: break;
    }
}

// Renumber the registers that `ops` (and `keep`: load / target registers) touch into 0 .. n-1, ascending; map[r] is the
// new number of register r (WS_REG_NONE stays).  Returns n.  A score tape reserves temporaries and one register per
// plane it ever read; a launch that folds part of it keeps only these rows of the register file.
inline int ws_compact_regs(const WsOp* ops, size_t n_ops, const uint8_t* keep, int n_keep, uint8_t* map /* [256] */) {
    bool used[256] = {false};
    for (size_t i = 0; i < n_ops; ++i) {
        const WsOp& o = ops[i];
        const uint32_t op = o.w0 & 0xFFu;
        const uint32_t r[4] = {(o.w0 >> 8) & 0xFFu, (o.w0 >> 16) & 0xFFu, (o.w0 >> 24) & 0xFFu, o.w1 & 0xFFu};
        if (ws_op_dst_is_reg(op)) used[r[0]] = true;
        used[r[1]] = used[r[2]] = used[r[3]] = true;
    }
    for (int k = 0; k < n_keep; ++k) used[keep[k]] = true;
    used[WS_REG_NONE] = false;
    int next = 0;
    for (int r = 0; r < 256; ++r) map[r] = used[r] ? (uint8_t)next++ : (uint8_t)0;
    map[WS_REG_NONE] = WS_REG_NONE;
    return next;
}

// Is entry i of a tape the continuation of a run (a squared-residual entry over the same registers as entry i-1)?
WS_HD bool ws_run_continues(const WsOp& prev, const WsOp& cur) {
    const uint32_t op = cur.w0 & 0xFFu;
    return (op == WS_OP_ACC_SQLIN2 || op == WS_OP_ACC_SQLIN2_S) && prev.w0 == cur.w0 && (prev.w1 & 0xFFu) == (cur.w1 & 0xFFu);
}

// A run of `len` consecutive ACC_SQLIN2 (or ACC_SQLIN2_S) entries over the SAME registers, e.g. the likelihood
// of a regression, sum_i logN(y_i; alpha + beta x_i, sigma): the operands are read from the register file once
// and each entry costs its three coefficients and four FP64 operations per particle, in the same order and
// with the same roundings as entry-by-entry execution (score-tape folds; run[0].op >> 8 == len).
template <int STRIDE, int P>
WS_HD void ws_vm_exec_sqlin2_run(const WsDop* __restrict__ run, int len, const double* __restrict__ R, double (&acc)[P]) {
    const WsDop& h = run[0];
    const bool scaled = (h.op & 0xFFu) == WS_OP_ACC_SQLIN2_S;
    const bool ha = h.a != WS_OFF_NONE, hb = h.b != WS_OFF_NONE;
    double A[P], B[P], C[P], D[P];
#pragma unroll
    for (int j = 0; j < P; ++j) {
        A[j] = ha ? R[h.a + j * STRIDE] : 0.0;
        B[j] = hb ? R[h.b + j * STRIDE] : 0.0;
        C[j] = scaled ? R[h.c + j * STRIDE] : 1.0;
        D[j] = scaled ? R[h.dst + j * STRIDE] : 0.0;
    }
    if (ha && hb && !scaled) {
        for (int i = 0; i < len; ++i) {
            const double k0 = run[i].k0, k1 = run[i].k1, k2 = run[i].k2;
#pragma unroll
            for (int j = 0; j < P; ++j) {
                double z = k0;
                z += k1 * A[j];
                z += k2 * B[j];
                acc[j] -= 0.5 * (z * z);
            }
        }
    } else if (ha && hb) {
        for (int i = 0; i < len; ++i) {
            const double k0 = run[i].k0, k1 = run[i].k1, k2 = run[i].k2;
#pragma unroll
            for (int j = 0; j < P; ++j) {
                double z = k0;
                z += k1 * A[j];
                z += k2 * B[j];
                z *= C[j];
                acc[j] -= 0.5 * (z * z) + D[j];
            }
        }
    } else {
        for (int i = 0; i < len; ++i) {
            const double k0 = run[i].k0, k1 = run[i].k1, k2 = run[i].k2;
#pragma unroll
            for (int j = 0; j < P; ++j) {
                double z = k0;
                if (ha) z += k1 * A[j];
                if (hb) z += k2 * B[j];
                if (scaled) {
                    z *= C[j];
                    acc[j] -= 0.5 * (z * z) + D[j];
                } else {
                    acc[j] -= 0.5 * (z * z);
                }
            }
        }
    }
}

// undecoded form (host harness, kernels that fetch ops per thread)
template <int STRIDE, int P>
WS_HD void ws_vm_exec(const WsOp& o, double* __restrict__ R, double (&acc)[P], const WsRng& rng,
                      const uint64_t (&particle)[P]) {
    ws_vm_exec_d<STRIDE, P>(ws_decode_op<STRIDE, P>(o), R, acc, rng, particle);
}
