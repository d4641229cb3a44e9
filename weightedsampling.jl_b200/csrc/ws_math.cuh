// ws_math.cuh — scalar building blocks shared by every wsb200 kernel.
//
// Everything here is a pure function of its arguments, marked WS_HD so that
//   * nvcc compiles it into the sm_100a kernels (the product path), and
//   * tests/host_math_check.cpp can compile the very same source with g++ and
//     compare it against the oracle without a GPU (test infrastructure only;
//     nothing in the shipped library runs these on the host).
//
// Reference formulas restated here (third-party, un-vendored; SURVEY.md §8c):
//   Normal      rand = mu + sigma*z ; logpdf = -(zv^2 + log2pi)/2 - log(sigma)
//               (StatsFuns normlogpdf, used through src/default_kernels.jl:12-23,94)
//   Exponential rand = theta*e ; logpdf = log(1/theta) - x/theta, -Inf for x<0
//               (src/default_kernels.jl:87)
//   bound transforms / Jacobians: src/move_kernels.jl:37-85
#pragma once
#include <stdint.h>
#include <math.h>
#include <string.h>

#if defined(__CUDACC__)
#define WS_HD __host__ __device__ __forceinline__
#else
#define WS_HD inline
#endif

#define WS_LOG2PI 1.8378770664093453
#define WS_TWO_M53 1.1102230246251565e-16 /* 2^-53 */

// ---------------------------------------------------------------------------
// Philox4x32-10 counter-based RNG (Salmon et al., SC'11).  Counter layout used
// everywhere in wsb200:  (particle_lo, particle_hi, stream_lo, stream_hi),
// key = (seed_lo, seed_hi).  `particle` is the GLOBAL particle / slot index, so
// draws do not depend on grid shape, fusion window or the number of ranks.
// ---------------------------------------------------------------------------
struct ws_u32x4 {
    uint32_t x, y, z, w;
};

WS_HD void ws_mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
#if defined(__CUDA_ARCH__)
    lo = a * b;
    hi = __umulhi(a, b);
#else
    uint64_t p = (uint64_t)a * (uint64_t)b;
    lo = (uint32_t)p;
    hi = (uint32_t)(p >> 32);
#endif
}

WS_HD ws_u32x4 ws_philox4x32_10(uint64_t particle, uint64_t stream, uint64_t seed) {
    uint32_t c0 = (uint32_t)particle, c1 = (uint32_t)(particle >> 32);
    uint32_t c2 = (uint32_t)stream, c3 = (uint32_t)(stream >> 32);
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0, lo0, hi1, lo1;
        ws_mulhilo(0xD2511F53u, c0, hi0, lo0);
        ws_mulhilo(0xCD9E8D57u, c2, hi1, lo1);
        uint32_t n0 = hi1 ^ c1 ^ k0;
        uint32_t n2 = hi0 ^ c3 ^ k1;
        c0 = n0;
        c1 = lo1;
        c2 = n2;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    ws_u32x4 out;
    out.x = c0;
    out.y = c1;
    out.z = c2;
    out.w = c3;
    return out;
}

// 53-bit uniform in [0,1) from two 32-bit words (same support as Julia's rand()).
WS_HD double ws_u01(uint32_t hi, uint32_t lo) {
    uint64_t v = (((uint64_t)hi << 32) | (uint64_t)lo) >> 11;
    return (double)v * WS_TWO_M53;
}
// 53-bit uniform in (0,1] (safe argument for log).
WS_HD double ws_u01_open0(uint32_t hi, uint32_t lo) {
    uint64_t v = ((((uint64_t)hi << 32) | (uint64_t)lo) >> 11) + 1ull;
    return (double)v * WS_TWO_M53;
}

// ---------------------------------------------------------------------------
// FP64 elementary functions specialised to the arguments this library feeds them.
// The general-purpose libdevice routines spend half their instructions on special cases and
// range checks that cannot occur here (profiles/r1_ncu_lines_*: log + sqrt + sincospi + exp were
// 285 of the 600 instructions per particle of the fused pass).  Coefficients: scripts/fit_math_polys.py
// (Chebyshev-node interpolation in 60-digit arithmetic); every routine is accurate to ~2 ulp and is
// checked against mpmath / libm in tests/test_device_math.py through the host instantiation.
// ---------------------------------------------------------------------------
WS_HD double ws_bits_to_double(uint64_t b) {
#if defined(__CUDA_ARCH__)
    return __longlong_as_double((long long)b);
#else
    double v;
    memcpy(&v, &b, 8);
    return v;
#endif
}
WS_HD uint64_t ws_double_to_bits(double v) {
#if defined(__CUDA_ARCH__)
    return (uint64_t)__double_as_longlong(v);
#else
    uint64_t b;
    memcpy(&b, &v, 8);
    return b;
#endif
}
WS_HD double ws_fma(double a, double b, double c) {
#if defined(__CUDA_ARCH__)
    return __fma_rn(a, b, c);
#else
    return fma(a, b, c);
#endif
}
// ~2^-21-accurate starting values (MUFU.RCP64H / MUFU.RSQ64H on the device)
WS_HD double ws_rcp_seed(double x) {
#if defined(__CUDA_ARCH__)
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    return y;
#else
    return (double)(float)(1.0 / x);
#endif
}
WS_HD double ws_rsqrt_seed(double x) {
#if defined(__CUDA_ARCH__)
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    return y;
#else
    return (double)(float)(1.0 / sqrt(x));
#endif
}

// Polynomial coefficients and reduction constants of the routines below.  On the device they live in constant
// memory and are consumed as constant-bank operands of the DFMAs: as 64-bit immediates the compiler built each one
// with two UMOVs in front of its DFMA — ~70 of the ~410 instructions per particle of the fused 2-D SSM step
// (profiles/r2b_ncu_ws_vm_sl_kernel_20M.txt).
#define WS_MATH_COEFS(X) \
    X(EXP_LOG2E, 1.4426950408889634) \
    X(EXP_NLN2HI, -6.93147180369123816490e-01) \
    X(EXP_NLN2LO, -1.90821492927058770002e-10) \
    X(EXP_P0, 0x1.af631d0059becp-26) \
    X(EXP_P1, 0x1.28b4057f44145p-22) \
    X(EXP_P2, 0x1.71ddf5749d126p-19) \
    X(EXP_P3, 0x1.a01991ac8730ap-16) \
    X(EXP_P4, 0x1.a01a01b14378fp-13) \
    X(EXP_P5, 0x1.6c16c187fbe02p-10) \
    X(EXP_P6, 0x1.111111110f225p-7) \
    X(EXP_P7, 0x1.555555554f0cfp-5) \
    X(EXP_P8, 0x1.555555555555ap-3) \
    X(EXP_P9, 0x1.0000000000011p-1) \
    X(LOG_A0, 0x1.2be6c99b32a48p-4) \
    X(LOG_A1, 0x1.39f2bba043e06p-4) \
    X(LOG_A2, 0x1.74630f3e18fa7p-4) \
    X(LOG_A3, 0x1.c71c61a40ddfbp-4) \
    X(LOG_A4, 0x1.2492492eefe17p-3) \
    X(LOG_A5, 0x1.99999999949d0p-3) \
    X(LOG_A6, 0x1.5555555555558p-2) \
    X(LOG_LN2LO, 1.90821492927058770002e-10) \
    X(LOG_LN2HI, 6.93147180369123816490e-01) \
    X(SIN_P0, 0x1.e3f38399551bfp-38) \
    X(SIN_P1, -0x1.e30071afc3e59p-30) \
    X(SIN_P2, 0x1.50782fda12d96p-22) \
    X(SIN_P3, -0x1.32d2cce2e5b19p-15) \
    X(SIN_P4, 0x1.466bc677587f8p-9) \
    X(SIN_P5, -0x1.4abbce625be41p-4) \
    X(SIN_P6, 0x1.921fb54442d18p-1) \
    X(COS_Q0, -0x1.b264ba152378ap-42) \
    X(COS_Q1, 0x1.f9cc41140bb60p-34) \
    X(COS_Q2, -0x1.a6d1ec7906c20p-26) \
    X(COS_Q3, 0x1.e1f5068355e15p-19) \
    X(COS_Q4, -0x1.55d3c7e3c90f8p-12) \
    X(COS_Q5, 0x1.03c1f081b5aacp-6) \
    X(COS_Q6, -0x1.3bd3cc9be45dep-2)
enum WsCoefIndex {
#define WS_COEF_ENUM(name, value) WS_CI_##name,
    WS_MATH_COEFS(WS_COEF_ENUM)
#undef WS_COEF_ENUM
    WS_CI_COUNT
};
#define WS_COEF_VALUE(name, value) value,
#if defined(__CUDACC__)
static __constant__ double ws_coef_dev[WS_CI_COUNT] = {WS_MATH_COEFS(WS_COEF_VALUE)};
#endif
static const double ws_coef_host[WS_CI_COUNT] = {WS_MATH_COEFS(WS_COEF_VALUE)};
#undef WS_COEF_VALUE
#if defined(WS_COEF_IMM)   // A/B switch: the coefficients as immediates again
#define WS_KV_EXP_LOG2E 1.4426950408889634
#define WS_KV_EXP_NLN2HI -6.93147180369123816490e-01
#define WS_KV_EXP_NLN2LO -1.90821492927058770002e-10
#define WS_KV_EXP_P0 0x1.af631d0059becp-26
#define WS_KV_EXP_P1 0x1.28b4057f44145p-22
#define WS_KV_EXP_P2 0x1.71ddf5749d126p-19
#define WS_KV_EXP_P3 0x1.a01991ac8730ap-16
#define WS_KV_EXP_P4 0x1.a01a01b14378fp-13
#define WS_KV_EXP_P5 0x1.6c16c187fbe02p-10
#define WS_KV_EXP_P6 0x1.111111110f225p-7
#define WS_KV_EXP_P7 0x1.555555554f0cfp-5
#define WS_KV_EXP_P8 0x1.555555555555ap-3
#define WS_KV_EXP_P9 0x1.0000000000011p-1
#define WS_KV_LOG_A0 0x1.2be6c99b32a48p-4
#define WS_KV_LOG_A1 0x1.39f2bba043e06p-4
#define WS_KV_LOG_A2 0x1.74630f3e18fa7p-4
#define WS_KV_LOG_A3 0x1.c71c61a40ddfbp-4
#define WS_KV_LOG_A4 0x1.2492492eefe17p-3
#define WS_KV_LOG_A5 0x1.99999999949d0p-3
#define WS_KV_LOG_A6 0x1.5555555555558p-2
#define WS_KV_LOG_LN2LO 1.90821492927058770002e-10
#define WS_KV_LOG_LN2HI 6.93147180369123816490e-01
#define WS_KV_SIN_P0 0x1.e3f38399551bfp-38
#define WS_KV_SIN_P1 -0x1.e30071afc3e59p-30
#define WS_KV_SIN_P2 0x1.50782fda12d96p-22
#define WS_KV_SIN_P3 -0x1.32d2cce2e5b19p-15
#define WS_KV_SIN_P4 0x1.466bc677587f8p-9
#define WS_KV_SIN_P5 -0x1.4abbce625be41p-4
#define WS_KV_SIN_P6 0x1.921fb54442d18p-1
#define WS_KV_COS_Q0 -0x1.b264ba152378ap-42
#define WS_KV_COS_Q1 0x1.f9cc41140bb60p-34
#define WS_KV_COS_Q2 -0x1.a6d1ec7906c20p-26
#define WS_KV_COS_Q3 0x1.e1f5068355e15p-19
#define WS_KV_COS_Q4 -0x1.55d3c7e3c90f8p-12
#define WS_KV_COS_Q5 0x1.03c1f081b5aacp-6
#define WS_KV_COS_Q6 -0x1.3bd3cc9be45dep-2
#define WS_K(name) WS_KV_##name
#elif defined(__CUDA_ARCH__)
#define WS_K(name) ws_coef_dev[WS_CI_##name]
#else
#define WS_K(name) ws_coef_host[WS_CI_##name]
#endif

// exp(d) for -708 < d <= 0: Cody-Waite reduction, degree-11 polynomial.  Outside that range the result is garbage.
WS_HD double ws_exp_nonpos_core(double d) {
    const double MAGIC = 6755399441055744.0;  // 1.5 * 2^52: fma(d, log2e, MAGIC) holds rint(d*log2e) in its low word
    const double t = ws_fma(d, WS_K(EXP_LOG2E), MAGIC);
    const double kd = t - MAGIC;
    double r = ws_fma(kd, WS_K(EXP_NLN2HI), d);   // ln2 hi (32 trailing zero bits)
    r = ws_fma(kd, WS_K(EXP_NLN2LO), r);          // ln2 lo
    double p = WS_K(EXP_P0);
    p = ws_fma(p, r, WS_K(EXP_P1));
    p = ws_fma(p, r, WS_K(EXP_P2));
    p = ws_fma(p, r, WS_K(EXP_P3));
    p = ws_fma(p, r, WS_K(EXP_P4));
    p = ws_fma(p, r, WS_K(EXP_P5));
    p = ws_fma(p, r, WS_K(EXP_P6));
    p = ws_fma(p, r, WS_K(EXP_P7));
    p = ws_fma(p, r, WS_K(EXP_P8));
    p = ws_fma(p, r, WS_K(EXP_P9));
    p = ws_fma(p, r, 1.0);
    p = ws_fma(p, r, 1.0);
    const uint64_t k = (uint64_t)(uint32_t)ws_double_to_bits(t);  // low word of t = k as a two's-complement int32
    return ws_bits_to_double(ws_double_to_bits(p) + (k << 52));
}

// exp(d) for d <= 0 (log-weight minus its maximum).
// d < -708 (result below the normal range) and d = -inf give 0; NaN gives NaN.
WS_HD double ws_exp_nonpos(double d) {
    const double v = ws_exp_nonpos_core(d);
    return (d > -708.0) ? v : ((d != d) ? d : 0.0);
}

// ws_exp_nonpos with NaN sent to 0 as well (one compare instead of two), for callers that convert the result
// with a saturating NaN -> 0 conversion anyway: d < -708, -inf and NaN give 0.
WS_HD double ws_exp_nonpos_or0(double d) {
    const double v = ws_exp_nonpos_core(d);
    return (d > -708.0) ? v : 0.0;
}

// a / b for finite a >= 0, b > 0 with rb = RN(1 / b) hoisted by the caller: product, exact residual, one
// correction (Markstein) — the IEEE quotient without the division subroutine's ~25 instructions.
WS_HD double ws_div_pos(double a, double b, double rb) {
    const double q = a * rb;
    return ws_fma(ws_fma(-q, b, a), rb, q);
}

// log(x * 2^kbias) for a positive, finite, normal x, without libdevice's special-case paths:
// x = 2^k z, z in [0.707, 1.414), log z = 2 atanh(s), s = (z-1)/(z+1).  (kbias keeps the result
// relatively accurate when x * 2^kbias is close to 1, as for a uniform close to 1.)
WS_HD double ws_log_pos(double x, int kbias = 0) {
    const uint64_t ix = ws_double_to_bits(x);
    const uint32_t hi = (uint32_t)(ix >> 32);
    const uint32_t th = hi - 0x3FE6A09Eu;                   // exponent of x / (sqrt(1/2) .. sqrt(2)) lands in the top bits
    const int k = (int)th >> 20;
    const double z = ws_bits_to_double(((uint64_t)(hi - ((uint32_t)k << 20)) << 32) | (ix & 0xFFFFFFFFull));
    const double f = z - 1.0;                               // exact
    const double g = z + 1.0;
    double y = ws_rcp_seed(g);
    double e = ws_fma(-g, y, 1.0);
    y = ws_fma(y, e, y);
    e = ws_fma(-g, y, 1.0);
    y = ws_fma(y, e, y);                                    // 1/g to ~1 ulp
    double s = f * y;
    s = ws_fma(ws_fma(-s, g, f), y, s);                     // f/g correctly rounded (Markstein)
    const double s2 = s * s;
    double a = WS_K(LOG_A0);
    a = ws_fma(a, s2, WS_K(LOG_A1));
    a = ws_fma(a, s2, WS_K(LOG_A2));
    a = ws_fma(a, s2, WS_K(LOG_A3));
    a = ws_fma(a, s2, WS_K(LOG_A4));
    a = ws_fma(a, s2, WS_K(LOG_A5));
    a = ws_fma(a, s2, WS_K(LOG_A6));
    const double kd = (double)(k + kbias);
    const double s3a = (s * s2) * a;
    // k ln2 + 2 s + 2 s^3 A(s^2), small terms first
    const double lo = ws_fma(kd, WS_K(LOG_LN2LO), s3a + s3a);
    return ws_fma(kd, WS_K(LOG_LN2HI), (s + s) + lo);
}

// sqrt(t) for a positive, finite, normal t: MUFU seed, two Newton steps on 1/sqrt, one residual correction.
WS_HD double ws_sqrt_pos(double t) {
    double y = ws_rsqrt_seed(t);
    const double h = 0.5 * t;
    double e = ws_fma(-(h * y), y, 0.5);
    y = ws_fma(y, e, y);
    e = ws_fma(-(h * y), y, 0.5);
    y = ws_fma(y, e, y);
    double r = t * y;
    r = ws_fma(ws_fma(-r, r, t), 0.5 * y, r);
    return r;
}

// (sin, cos) of (pi/4) f for f in [0, 1]
WS_HD void ws_sincos_octant(double f, double& sn, double& cs) {
    const double f2 = f * f;
    double p = WS_K(SIN_P0);
    p = ws_fma(p, f2, WS_K(SIN_P1));
    p = ws_fma(p, f2, WS_K(SIN_P2));
    p = ws_fma(p, f2, WS_K(SIN_P3));
    p = ws_fma(p, f2, WS_K(SIN_P4));
    p = ws_fma(p, f2, WS_K(SIN_P5));
    p = ws_fma(p, f2, WS_K(SIN_P6));
    sn = p * f;
    double q = WS_K(COS_Q0);
    q = ws_fma(q, f2, WS_K(COS_Q1));
    q = ws_fma(q, f2, WS_K(COS_Q2));
    q = ws_fma(q, f2, WS_K(COS_Q3));
    q = ws_fma(q, f2, WS_K(COS_Q4));
    q = ws_fma(q, f2, WS_K(COS_Q5));
    q = ws_fma(q, f2, WS_K(COS_Q6));
    cs = ws_fma(q, f2, 1.0);
}

// Box-Muller from two 64-bit words:
//   u1 = (2 k + 1) 2^-53, k = top 52 bits of w1  (open interval: log and sqrt never see 0 or 1)
//   angle: bits 0..51 of w2 give f in [0,1) (position inside an octant), bits 52..54 pick the octant as
//   (swap sin/cos, sign of the first, sign of the second) — the eight sign/swap images of the arc
//   (pi/4) f tile the circle exactly once, so the pair is uniform on the circle.
WS_HD void ws_box_muller(uint64_t w1, uint64_t w2, double& z0, double& z1) {
    const double v = ws_bits_to_double(0x4340000000000000ull | (w1 >> 12)) - 9007199254740991.0;  // 2k+1, exact
    const double t = -2.0 * ws_log_pos(v, -53);  // -2 log u1 in [2^-52, 73.5]
    const double rad = ws_sqrt_pos(t);
    const double f = ws_bits_to_double(0x3FF0000000000000ull | (w2 & 0x000FFFFFFFFFFFFFull)) - 1.0;
    double sn, cs;
    ws_sincos_octant(f, sn, cs);
    const bool swap = (w2 >> 52) & 1ull;
    const double a = swap ? sn : cs, b = swap ? cs : sn;
    const uint64_t sa = ((w2 >> 53) & 1ull) << 63, sb = ((w2 >> 54) & 1ull) << 63;
    z0 = ws_bits_to_double(ws_double_to_bits(rad * a) ^ sa);
    z1 = ws_bits_to_double(ws_double_to_bits(rad * b) ^ sb);
}

// One Philox block -> two independent standard normals (Box-Muller, FP64).
WS_HD void ws_randn2(uint64_t particle, uint64_t stream, uint64_t seed, double& z0, double& z1) {
    ws_u32x4 r = ws_philox4x32_10(particle, stream, seed);
    ws_box_muller(((uint64_t)r.x << 32) | r.y, ((uint64_t)r.z << 32) | r.w, z0, z1);
}

// One Philox block -> two uniforms in [0,1).
WS_HD void ws_randu2(uint64_t particle, uint64_t stream, uint64_t seed, double& u0, double& u1) {
    ws_u32x4 r = ws_philox4x32_10(particle, stream, seed);
    u0 = ws_u01(r.x, r.y);
    u1 = ws_u01(r.z, r.w);
}

// Standard exponential variate e = -log(u), u in (0,1].
WS_HD double ws_randexp(uint64_t particle, uint64_t stream, uint64_t seed) {
    ws_u32x4 r = ws_philox4x32_10(particle, stream, seed);
    const uint64_t v = ((((uint64_t)r.x << 32) | (uint64_t)r.y) >> 11) + 1ull;  // u = v 2^-53 in (0, 1]
    return -ws_log_pos((double)v, -53);
}


// ---------------------------------------------------------------------------
// Variates that need a rejection loop (the reference draws them with Distributions.jl's samplers,
// src/default_kernels.jl:83-102: Gamma, and through it Beta, TDist, Chisq, InverseGamma; Poisson).  Trial t of a
// particle takes Philox blocks (particle, stream | (2t) << 40) and (particle, stream | (2t+1) << 40): counters, not
// state, so a draw does not depend on what other threads do, and stream ids stay below 2^40.
// ---------------------------------------------------------------------------
#define WS_TRIAL_SHIFT 40
#define WS_MAX_TRIALS 64
WS_HD uint64_t ws_trial_stream(uint64_t stream, uint32_t k) { return stream | ((uint64_t)(k + 1u) << WS_TRIAL_SHIFT); }

// Standard Gamma(shape a > 0, scale 1): Marsaglia & Tsang (2000): d = a - 1/3, c = 1/sqrt(9 d), v = (1 + c z)^3,
// accept if log u < z^2/2 + d - d v + d log v; a < 1 through Gamma(a + 1) U^(1/a).  a <= 0 or NaN gives NaN.
WS_HD double ws_rand_gamma(double a, uint64_t particle, uint64_t stream, uint64_t seed) {
    if (!(a > 0.0)) return NAN;
    const bool boost = a < 1.0;
    const double aa = boost ? a + 1.0 : a;
    const double d = aa - 1.0 / 3.0;
    const double c = 1.0 / sqrt(9.0 * d);
    double g = d;  // (returned only if WS_MAX_TRIALS trials in a row are rejected: probability < 1e-80)
    double u_boost = 0.5;
    for (uint32_t t = 0; t < WS_MAX_TRIALS; ++t) {
        double z, z1, u, u1;
        ws_randn2(particle, ws_trial_stream(stream, 2u * t), seed, z, z1);
        const ws_u32x4 r = ws_philox4x32_10(particle, ws_trial_stream(stream, 2u * t + 1u), seed);
        u = ws_u01_open0(r.x, r.y);
        u1 = ws_u01_open0(r.z, r.w);
        const double w = 1.0 + c * z;
        if (w <= 0.0) continue;
        const double v = w * w * w;
        if (log(u) < 0.5 * z * z + d - d * v + d * log(v)) {
            g = d * v;
            u_boost = u1;
            break;
        }
    }
    return boost ? g * pow(u_boost, 1.0 / a) : g;
}

// Poisson(lam >= 0): inversion by sequential search for lam < 10, PTRS (Hormann 1993, "The transformed rejection
// method for generating Poisson random variables") otherwise.  lam < 0 or NaN gives NaN.
WS_HD double ws_rand_poisson(double lam, uint64_t particle, uint64_t stream, uint64_t seed) {
    if (!(lam >= 0.0)) return NAN;
    if (lam == 0.0) return 0.0;
    if (lam < 10.0) {
        const ws_u32x4 r = ws_philox4x32_10(particle, ws_trial_stream(stream, 0u), seed);
        const double u = ws_u01(r.x, r.y);
        double p = exp(-lam), F = p;
        int k = 0;
        while (u > F && k < 200) {
            ++k;
            p *= lam / (double)k;
            F += p;
        }
        return (double)k;
    }
    const double slam = sqrt(lam), loglam = log(lam);
    const double b = 0.931 + 2.53 * slam;
    const double a = -0.059 + 0.02483 * b;
    const double inv_alpha = 1.1239 + 1.1328 / (b - 3.4);
    const double vr = 0.9277 - 3.6224 / (b - 2.0);
    double k = floor(lam);
    for (uint32_t t = 0; t < WS_MAX_TRIALS; ++t) {
        const ws_u32x4 r = ws_philox4x32_10(particle, ws_trial_stream(stream, t), seed);
        const double U = ws_u01(r.x, r.y) - 0.5;
        const double V = ws_u01_open0(r.z, r.w);
        const double us = 0.5 - fabs(U);
        k = floor((2.0 * a / us + b) * U + lam + 0.43);
        if (us >= 0.07 && V <= vr) break;
        if (k < 0.0 || (us < 0.013 && V > us)) continue;
        if (log(V) + log(inv_alpha) - log(a / (us * us) + b) <= -lam + k * loglam - lgamma(k + 1.0)) break;
    }
    return k < 0.0 ? 0.0 : k;
}

// Multinomial resampling without a sort (csrc/ws_kernels.cu): the order statistics of N iid uniforms are running sums
// of N + 1 iid exponential spacings divided by their total.  Slot k's spacing in fixed point:
// e_k = max(1, rint(Exp(1) * 2^mn_shift)), the exponential from words (2(k&1), 2(k&1)+1) of Philox block k >> 1.
// Host and device evaluate the same code (ws_log_pos is built from explicit fmas), so the tests regenerate the
// spacings bit for bit through the CPU harness.
WS_HD unsigned long long ws_spacing_fx(uint32_t hi, uint32_t lo, int mn_shift) {
    const uint64_t v = ((((uint64_t)hi << 32) | (uint64_t)lo) >> 11) + 1ull;  // u = v 2^-53 in (0, 1]
    const double e = -ws_log_pos((double)v, -53);
    const unsigned long long q = (unsigned long long)llrint(ldexp(e, mn_shift));
    return q < 1ull ? 1ull : q;
}
WS_HD unsigned long long ws_spacing_of_slot(uint64_t k, int mn_shift, uint64_t seed, uint64_t stream) {
    const ws_u32x4 r = ws_philox4x32_10(k >> 1, stream, seed);
    return (k & 1ull) ? ws_spacing_fx(r.z, r.w, mn_shift) : ws_spacing_fx(r.x, r.y, mn_shift);
}

// ---------------------------------------------------------------------------
// sample(state, n; replace) (src/utils.jl:102-118), drawn on the device (csrc/ws_kernels_stats.cu).  Every piece is a
// function of the particle's GLOBAL index, its log-weight and the global maximum m only, so the draw does not depend
// on the number of ranks; the CPU harness evaluates the same code to regenerate the device values bit for bit.
// ---------------------------------------------------------------------------
#define WS_SAMPLE_Q_SCALE 4503599627370496.0 /* 2^52, relative to the largest weight */
struct ws_u128 {
    uint64_t hi, lo;
};
// with replacement: integer weight q_i = rint(exp(l_i - m) 2^52); NaN, -inf and l_i - m < -708 give 0
WS_HD uint64_t ws_sample_q(double l, double m) {
    const double v = ws_exp_nonpos_or0(l - m) * WS_SAMPLE_Q_SCALE;
#if defined(__CUDA_ARCH__)
    return __double2ull_rn(v);
#else
    return (uint64_t)llrint(v);
#endif
}
WS_HD void ws_mul64(uint64_t a, uint64_t b, uint64_t& hi, uint64_t& lo) {
#if defined(__CUDA_ARCH__)
    lo = a * b;
    hi = __umul64hi(a, b);
#else
    const unsigned __int128 p = (unsigned __int128)a * b;
    lo = (uint64_t)p;
    hi = (uint64_t)(p >> 64);
#endif
}
// draw k's target t_k = floor(r_k T / 2^128), r_k = the 128-bit integer (x, y, z, w) of Philox block (k, stream, seed);
// t_k < T, and the draw is index_k = min{ j : Q_j > t_k } over the exact integer CDF Q of the q_i
WS_HD ws_u128 ws_sample_target(uint64_t k, uint64_t stream, uint64_t seed, ws_u128 T) {
    const ws_u32x4 r = ws_philox4x32_10(k, stream, seed);
    const uint64_t a1 = ((uint64_t)r.x << 32) | r.y, a0 = ((uint64_t)r.z << 32) | r.w;
    uint64_t h11, l11, h10, l10, h01, l01, h00, l00;
    ws_mul64(a1, T.hi, h11, l11);
    ws_mul64(a1, T.lo, h10, l10);
    ws_mul64(a0, T.hi, h01, l01);
    ws_mul64(a0, T.lo, h00, l00);
    (void)l00;
    // bits 64..127 of the product: h00 + l10 + l01, whose carries (0..2) go to bits 128..
    uint64_t mid = h00 + l10;
    uint64_t carry = mid < l10 ? 1ull : 0ull;
    mid += l01;
    carry += mid < l01 ? 1ull : 0ull;
    ws_u128 t;
    t.lo = l11 + h10;
    uint64_t c2 = t.lo < h10 ? 1ull : 0ull;
    t.lo += h01;
    c2 += t.lo < h01 ? 1ull : 0ull;
    t.lo += carry;
    c2 += t.lo < carry ? 1ull : 0ull;
    t.hi = h11 + c2;
    return t;
}
// without replacement: the Gumbel / Efraimidis-Spirakis key  key_i = l_i - log(E_i),  E_i = ws_randexp(i, stream, seed);
// the n largest keys are an exact weighted draw without replacement, in descending order distributed like successive
// draws.  E_i = 0 (u = 1, probability 2^-53) is read as 2^-54, half the smallest positive value, to stay in the domain
// of ws_log_pos.  Returned as its order-preserving 64-bit image; a NaN or infinite l_i gives 0, below every finite key.
WS_HD uint64_t ws_sample_key(double l, uint64_t i, uint64_t stream, uint64_t seed) {
    if (!(fabs(l) <= 1.7976931348623157e308)) return 0ull;
    double e = ws_randexp(i, stream, seed);
    if (!(e > 0.0)) e = 5.551115123125783e-17;  // 2^-54
    const uint64_t b = ws_double_to_bits(l - ws_log_pos(e));
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

// ---------------------------------------------------------------------------
// log densities
// ---------------------------------------------------------------------------
WS_HD double ws_normal_logpdf(double x, double mu, double sigma) {
    double z;
    if (sigma == 0.0) {
        if (x == mu) {
            z = 0.0;  // zval(mu, 1, x)
        } else {
            z = (x - mu) / sigma;  // +-Inf
            sigma = 1.0;
        }
    } else {
        z = (x - mu) / sigma;
    }
    return -(z * z + WS_LOG2PI) / 2.0 - log(sigma);
}

WS_HD double ws_exponential_logpdf(double x, double theta) {
    double lam = 1.0 / theta;
    double z = log(lam) - lam * x;
    return x < 0.0 ? -INFINITY : z;
}

// ---------------------------------------------------------------------------
// MH bound transforms (src/move_kernels.jl:37-85).  kind: 0 none, 1 lower only,
// 2 upper only, 3 both.
// ---------------------------------------------------------------------------
WS_HD int ws_bound_kind(double lo, double hi) {
    bool flo = isfinite(lo), fhi = isfinite(hi);
    return (flo && fhi) ? 3 : (flo ? 1 : (fhi ? 2 : 0));
}
WS_HD double ws_to_unconstrained(double x, double lo, double hi, int kind) {
    switch (kind) {
        case 3: return log(x - lo) - log(hi - x);
        case 1: return log(x - lo);
        case 2: return log(hi - x);
        default: return x;
    }
}
WS_HD double ws_from_unconstrained(double z, double lo, double hi, int kind) {
    switch (kind) {
        case 3: return lo + (hi - lo) / (1.0 + exp(-z));
        case 1: return lo + exp(z);
        case 2: return hi - exp(z);
        default: return z;
    }
}
WS_HD double ws_log1pexp(double z) { return z > 0.0 ? z + log1p(exp(-z)) : log1p(exp(z)); }
WS_HD double ws_log_abs_jacobian(double z, double lo, double hi, int kind) {
    switch (kind) {
        case 3: return log(hi - lo) - ws_log1pexp(z) - ws_log1pexp(-z);
        case 1:
        case 2: return z;
        default: return 0.0;
    }
}

// ---------------------------------------------------------------------------
// Stratified / systematic slot uniforms in the reference's exact FP order
// (src/resampling.jl:39-41):  u_n = (n-1)*invN + r_n*invN,  n = 1..N.
// `n0` is the 0-based slot index (n-1).
// ---------------------------------------------------------------------------
// The explicit _rn intrinsics stop nvcc from contracting the expression into an
// FMA (Julia does not contract), so u_n is bit-identical to the reference's.
template <class I>
WS_HD double ws_slot_u(I n0, double r, double inv_n) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(__dmul_rn((double)n0, inv_n), __dmul_rn(r, inv_n));
#else
    volatile double a = (double)n0 * inv_n;
    volatile double b = r * inv_n;
    return a + b;
#endif
}

// Fixed-point CDF: weights are accumulated as unsigned 64-bit integers with
// scale 2^63 so that prefix sums are exactly associative (deterministic for any
// scan order, tile shape or rank count).  See DESIGN.md "CDF arithmetic".
#define WS_FX_SCALE 9223372036854775808.0 /* 2^63 */
WS_HD uint64_t ws_weight_to_fx(double w) {
    // w in [0,1]; NaN / negative -> 0
    if (!(w > 0.0)) return 0ull;
    if (w >= 1.0) return 1ull << 63;
    double s = w * WS_FX_SCALE;
#if defined(__CUDA_ARCH__)
    return __double2ull_rn(s);
#else
    return (uint64_t)llrint(s);
#endif
}
WS_HD double ws_fx_to_double(uint64_t c) { return (double)c * (1.0 / WS_FX_SCALE); }

// Number of output slots whose uniform is <= C, i.e. F(C) = #{n0 in [0,N) : u(n0) <= C}
// for the (monotone) stratified / systematic grid u(n0) = n0*invN + r(n0)*invN.
// Offspring of particle m are exactly the slots  F(C_{m-1}) <= n0 < F(C_m), which
// restates icdf's  a_n = min{ m : C_m >= u_n }  (src/resampling.jl:13-26) per particle
// instead of per slot.  `r` is any callable slot -> uniform in [0,1).
template <class RFn>
WS_HD int64_t ws_count_slots_le(double C, int64_t N, double inv_n, RFn& r) {
    // Invariant wanted on exit: u(k-1) <= C (or k == 0) and u(k) > C (or k == N).  A uniform is only
    // drawn when the cheap bounds  fl(k*invN) <= u(k) <= fl(fl(k*invN) + invN)  cannot decide, which
    // leaves about one draw per call.  N < 2^31 (Int32 ancestors), so k fits an int.
    const double t = C * (double)N;
    int k = (t >= (double)N) ? (int)N : (t > 0.0 ? (int)t : 0);
    const int n = (int)N;
    bool advanced = false;
    while (k < n) {
        if (C < ws_slot_u(k, 0.0, inv_n)) break;  // u(k) >= fl(k*invN) > C
        if (ws_slot_u(k, r((int64_t)k), inv_n) <= C) {
            ++k;
            advanced = true;
        } else {
            break;
        }
    }
    if (!advanced) {
        while (k > 0) {
            if (C >= ws_slot_u(k - 1, 1.0, inv_n)) break;  // u(k-1) <= fl(fl((k-1)*invN) + invN) <= C
            if (ws_slot_u(k - 1, r((int64_t)(k - 1)), inv_n) > C) --k; else break;
        }
    }
    return (int64_t)k;
}
