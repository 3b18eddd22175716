// sin / exp / log for the render path (Expr::Sin/Exp/Ln, reference src/lib.rs:648-650).
//
// exp and log: glibc's algorithms, restated in device_libm_glibc.cuh -- the reference's bits, and cheaper than the
// polynomial versions they replaced.  sin: a fast version here (reduction by pi, one odd polynomial; <= 1.8 ULP measured
// on the host rendition against 80-bit libm, tools/libm_check.c, 2e6 samples per range), or glibc's own in exact mode
// (MR_LIBM_GLIBC).  Why not CUDA's libdevice: its routines are accurate, but each call costs ~25 instructions that are not
// FP64 work (constants rebuilt with two 32-bit moves each, special-case branches, address arithmetic); here every constant
// is a constant-bank operand and arguments outside the fast range take one rarely taken branch to an out-of-line routine.
//
// The same text compiles for the host when MR_LIBM_HOST is defined (fma() for __fma_rn), which is how the accuracy numbers
// and the bit-for-bit comparison with glibc (tools/glibc_libm_check.c) are produced without a GPU.
#ifndef MARAY_DEVICE_LIBM_CUH
#define MARAY_DEVICE_LIBM_CUH

#ifdef MR_LIBM_PLAIN
// A/B switch and host-side text checks: the platform's own sin/exp/log (libdevice on the GPU).
#ifndef MR_PLAIN_FN
#define MR_PLAIN_FN __device__ __forceinline__
#endif
MR_PLAIN_FN double mr_sin(double x) { return sin(x); }
MR_PLAIN_FN double mr_exp(double x) { return exp(x); }
MR_PLAIN_FN double mr_log(double x) { return log(x); }
MR_PLAIN_FN int mr_sin_ge0(double x) { return sin(x) >= 0.0; }
MR_PLAIN_FN double mr_sin_call(double a) { return mr_sin(a); }
MR_PLAIN_FN double mr_exp_call(double a) { return mr_exp(a); }
MR_PLAIN_FN double mr_log_call(double a) { return mr_log(a); }
#ifdef MR_SCR_STRIDE
#ifndef MR_DYN_DECL
#define MR_DYN_DECL extern __shared__ double mr_dyn_f64[];
#endif
MR_DYN_DECL
#define MR_S(k) mr_dyn_f64[(k) * MR_SCR_STRIDE + threadIdx.x]
#define MR_R(k) MR_S(8 + (k))
#define MR_DEFINE_SCRATCH_BATCH_S(fn, SUF)                                                                  \
    MR_PLAIN_FN unsigned int mr_##fn##_batch##SUF(const unsigned int n) {                                   \
        for (unsigned int k = 0; k < n; k++) MR_R(k) = mr_##fn(MR_S(k));                               \
        return 0u;                                                                                     \
    }                                                                                                  \
    MR_PLAIN_FN void mr_##fn##_fix##SUF(unsigned int) {}
#define MR_BATCH_HELPERS(SUF) MR_DEFINE_SCRATCH_BATCH_S(sin, SUF) MR_DEFINE_SCRATCH_BATCH_S(exp, SUF) MR_DEFINE_SCRATCH_BATCH_S(log, SUF)
#ifndef MR_NO_DEFAULT_BATCH_HELPERS
MR_BATCH_HELPERS()
#endif
MR_PLAIN_FN void mr_scratch_tables_init() {}   // the platform's own exp and log bring their own tables
#endif
#else

// The out-of-range branch is cold: saying so lets the compiler place its block out of line, so the
// fast path falls through.  In MBs of straight-line code a TAKEN branch restarts the sequential
// instruction prefetch, and one per sin/exp/ln is what made inlined transcendental-heavy programs
// instruction-fetch bound (DESIGN.md 3.1).
#define MR_UNLIKELY(c) __builtin_expect(!!(c), 0)

#ifdef MR_LIBM_HOST
#include <math.h>
#include <stdint.h>
#include <string.h>
#define MR_FN static inline
#define MR_TABLE static const
#define MR_FMA(a, b, c) fma((a), (b), (c))
static inline int mr_lo32(double d) { uint64_t u; memcpy(&u, &d, 8); return (int)(uint32_t)u; }
static inline int mr_hi32(double d) { uint64_t u; memcpy(&u, &d, 8); return (int)(uint32_t)(u >> 32); }
static inline double mr_hilo(int hi, int lo) {
    uint64_t u = ((uint64_t)(uint32_t)hi << 32) | (uint32_t)lo; double d; memcpy(&d, &u, 8); return d;
}
#define MR_SLOW_SIN_F(x) sin(x)
#define MR_LDG2(p, lo, hi) do { (lo) = (p)[0]; (hi) = (p)[1]; } while (0)
#else
#define MR_FN __device__ __forceinline__
#define MR_TABLE static __constant__
#define MR_FMA(a, b, c) __fma_rn((a), (b), (c))
__device__ __forceinline__ int mr_lo32(double d) { return __double2loint(d); }
__device__ __forceinline__ int mr_hi32(double d) { return __double2hiint(d); }
__device__ __forceinline__ double mr_hilo(int hi, int lo) { return __hiloint2double(hi, lo); }
// Out-of-range arguments of the fast sine go to libdevice, out of line so the call sites stay small.
static __device__ __noinline__ double mr_slow_sin(double x) { return sin(x); }
#define MR_SLOW_SIN_F(x) mr_slow_sin(x)
#define MR_LDG2(p, lo, hi) do { double2 v2_ = __ldg(reinterpret_cast<const double2*>(p)); (lo) = v2_.x; (hi) = v2_.y; } while (0)
#endif

#include "device_libm_glibc.cuh"   // glibc's routines: mr_*_inrange_g, mr_*_fast_g, mr_*_slow_g (exp and log ARE these)

// Constants, read as constant-bank operands.  The compiler fetches two neighbours that share a 16-byte line with one
// LDCU.128, so where the entries sit relative to those lines shapes the code: entry 1 is unused and keeps 1/pi and the
// pi parts in the pairs they were measured in, and an odd entry count keeps the scene's constant table (MRK_BITS, next
// in the bank) on the same alignment.  Dropping entry 1 doubled chess's per-thread constant loads (LDC.64).
MR_TABLE double MR_LK[] = {
    /* 0 */ 0x1.8p52,                    // round-to-integer magic (1.5 * 2^52)
    /* 1 */ 0.0,                         // unused: alignment (above)
    // reduction by pi: 160 bits of pi in three parts, the first product exact (pi middle is one ulp short, so the tail
    // is positive: all three products of a +0 quotient are -0 and sin(-0) stays -0)
    /* 2 */ 0x1.45f306dc9c883p-2,        // 1/pi
    /* 3 */ 0x1.921fb54442d18p+1,        // pi high
    /* 4 */ 0x1.1a62633145c06p-53,       // pi middle
    /* 5 */ 0x1.c1cd129024e09p-106,      // pi low
    // sin(r) = r + r*s*S(s), s = r*r, |r| <= pi/2: S of degree 8, lowest first (relative error 2^-58.7; tools/gen_libm_coeffs.py)
    /* 6 */ -0x1.5555555555555p-3, 0x1.11111111110a9p-7, -0x1.a01a01a010c5cp-13, 0x1.71de3a4f8ab99p-19,
    /* 10 */ -0x1.ae64528659a2dp-26, 0x1.6122db98108c0p-33, -0x1.add52c09d1f58p-41, 0x1.6dc19ddd0cdfbp-49,
    /* 14 */ 0x1.4b52654981457p-56,
};

// Fast range of the sine: |x| < 2^22.  Everything else (incl. NaN, infinity) goes to libdevice.
// The range tests look at the high word only (integer pipe, not the FP64 pipe); NaN and infinity
// have a high word above every bound, so they always take the libdevice branch.
MR_FN int mr_sin_inrange_f(double x) { return (unsigned int)(mr_hi32(x) & 0x7fffffff) < 0x41500000u; }   // |x| < 2^22
// exp and log are glibc's algorithms in every mode (device_libm_glibc.cuh): fewer FP64 instructions than the
// polynomial versions they replaced (12 and 15 against 17 and 30), dependency chains half as long -- which is what
// bounds the batched helpers -- and the reference's bits.  exp: |x| < 512; tiny arguments need no special case here
// (for |x| < 2^-54 the main path rounds 1 + x + x^2/2.. to exactly what glibc's early `1.0 + x` returns).
MR_FN int mr_exp_inrange_f(double x) { return (unsigned int)((mr_hi32(x) >> 20) & 0x7ff) < 0x408u; }
MR_FN int mr_log_inrange_f(double x) { return mr_log_inrange_g(x); }

// Straight-line fast paths: safe (no traps, no loops) for ANY argument, meaningful inside the range.
// sin(x), fast version: x = k*pi + r, |r| <= pi/2 (three FMAs over 160 bits of pi, the first product exact),
// sin(x) = (-1)^k (r + r*s*S(s)).  One polynomial for every argument -- no parity-dependent coefficient rows, hence no
// table loads and no selects --, evaluated by Estrin's scheme: eight FMAs in four dependent steps.  More FP64 instructions
// than the quadrant version it replaced (20 against 15) but a chain of 12 instead of 16 and a third fewer instructions
// overall, which is what counts in the batched helpers (latency-bound: DESIGN.md 3.1).  sin(-0) = -0: S*s is made +0 by
// an explicit +0.0 addend, so the last FMA adds (-0) to (-0).
MR_FN double mr_sin_fast_f(double x) {
    const double t = MR_FMA(x, MR_LK[2], MR_LK[0]);
    const double k = t - MR_LK[0];
    double r = MR_FMA(k, -MR_LK[3], x);
    r = MR_FMA(k, -MR_LK[4], r);
    r = MR_FMA(k, -MR_LK[5], r);
    const double s = r * r;
    // the six high coefficients by Estrin's scheme (three independent FMAs, then two steps), the three low ones by
    // Horner's: the low end decides the rounding error, the high end the length of the chain
    const double p34 = MR_FMA(MR_LK[10], s, MR_LK[9]);
    const double p56 = MR_FMA(MR_LK[12], s, MR_LK[11]);
    const double p78 = MR_FMA(MR_LK[14], s, MR_LK[13]);
    const double s2 = s * s;
    double S = MR_FMA(p56, s2, p34);
    S = MR_FMA(p78, s2 * s2, S);
    S = MR_FMA(S, s, MR_LK[8]);
    S = MR_FMA(S, s, MR_LK[7]);
    S = MR_FMA(S, s, MR_LK[6]);
    const double v = MR_FMA(MR_FMA(S, s, 0.0), r, r);
    return mr_hilo((int)((unsigned int)mr_hi32(v) ^ ((unsigned int)mr_lo32(t) << 31)), mr_lo32(v));   // odd k: negate
}

MR_FN double mr_exp_fast_f(double x) { return mr_exp_fast_g(x); }
MR_FN double mr_log_fast_f(double x) { return mr_log_fast_g(x); }

// Which implementation the names below mean.  Default: the fast versions above.  MR_LIBM_GLIBC (MARAY_LIBM=glibc):
// the exact mode of device_libm_glibc.cuh.  MR_LIBM_BOTH (the interpreter kernel, which is compiled ahead of time and
// switches at run time): fast under the plain names, exact as mr_sin_g / mr_exp_g / mr_log_g.
#ifdef MR_LIBM_GLIBC
#define MR_SEL(name) name##_g
#define MR_SLOW_SIN(x) mr_sin_slow_g(x)
#else
#define MR_SEL(name) name##_f
#define MR_SLOW_SIN(x) MR_SLOW_SIN_F(x)
#endif
#define MR_SLOW_EXP(x) mr_exp_slow_g(x)
#define MR_SLOW_LOG(x) mr_log_slow_g(x)
#define MR_DEFINE_SELECTED(fn)                                                          \
    MR_FN int mr_##fn##_inrange(double x) { return MR_SEL(mr_##fn##_inrange)(x); }      \
    MR_FN double mr_##fn##_fast(double x) { return MR_SEL(mr_##fn##_fast)(x); }
MR_DEFINE_SELECTED(sin)
MR_DEFINE_SELECTED(exp)
MR_DEFINE_SELECTED(log)
#if defined(MR_LIBM_GLIBC) || defined(MR_LIBM_BOTH) || defined(MR_LIBM_HOST)
MR_FN double mr_sin_g(double x) { return mr_sin_inrange_g(x) ? mr_sin_fast_g(x) : mr_sin_slow_g(x); }
MR_FN double mr_exp_g(double x) { return mr_exp_inrange_g(x) ? mr_exp_fast_g(x) : mr_exp_slow_g(x); }
MR_FN double mr_log_g(double x) { return mr_log_inrange_g(x) ? mr_log_fast_g(x) : mr_log_slow_g(x); }
#endif

// Two shapes, measured: inlined into straight-line code the "compute, then repair" form is faster
// (chess_4k 7.80 vs 8.19 ms); inside the out-of-line batched helpers the early-out form is
// (deep scene 20.0 vs 23.6 ms: nothing but x is live across the libdevice call).
MR_FN double mr_sin(double x) {
#ifdef MR_LIBM_GLIBC
    if (MR_UNLIKELY(!mr_sin_inrange(x))) return MR_SLOW_SIN(x);
    return mr_sin_fast(x);
#else
    double r = mr_sin_fast(x);
    if (MR_UNLIKELY(!mr_sin_inrange(x))) r = MR_SLOW_SIN(x);
    return r;
#endif
}
MR_FN double mr_sin_eo(double x) {
    if (!mr_sin_inrange(x)) return MR_SLOW_SIN(x);
    return mr_sin_fast(x);
}

MR_FN double mr_exp(double x) {
#ifdef MR_LIBM_GLIBC
    if (MR_UNLIKELY(!mr_exp_inrange(x))) return MR_SLOW_EXP(x);
    return mr_exp_fast(x);
#else
    double r = mr_exp_fast(x);
    if (MR_UNLIKELY(!mr_exp_inrange(x))) r = MR_SLOW_EXP(x);
    return r;
#endif
}
MR_FN double mr_exp_eo(double x) {
    if (!mr_exp_inrange(x)) return MR_SLOW_EXP(x);
    return mr_exp_fast(x);
}
MR_FN double mr_log(double x) {
#ifdef MR_LIBM_GLIBC
    if (MR_UNLIKELY(!mr_log_inrange(x))) return MR_SLOW_LOG(x);
    return mr_log_fast(x);
#else
    double r = mr_log_fast(x);
    if (MR_UNLIKELY(!mr_log_inrange(x))) r = MR_SLOW_LOG(x);
    return r;
#endif
}
MR_FN double mr_log_eo(double x) {
    if (!mr_log_inrange(x)) return MR_SLOW_LOG(x);
    return mr_log_fast(x);
}

// mr_sin(x) >= 0.0 without the sine: what `step(sin(u))` needs (Maray's `chess`, reference src/lib.rs:969-973).
// x = k*pi + r with |r| <= pi/2 (the Cody-Waite reduction of mr_sin_fast_f: 160 bits of pi, first product exact): sin(x) = (-1)^k sin(r), and sin(r) has the sign of r and is +-0 exactly when r is.  The
// reduced argument of a nonzero double is never closer to zero than ~2^-60 while r is good to ~2^-100 absolute here, so
// the sign of r IS the sign of the true sine -- which every sine with a relative error bound returns, the fast one
// above, libdevice's and glibc's (exact mode) alike.  Checked against both on the host (tools/glibc_libm_check.c, all
// ranges and the neighbourhoods of 8 000 multiples of pi/2).  Outside |x| < 2^22: the full routine.
MR_FN int mr_sin_ge0_fast(double x) {
    const double t = MR_FMA(x, MR_LK[2], MR_LK[0]);
    const double k = t - MR_LK[0];
    double r = MR_FMA(k, -MR_LK[3], x);
    r = MR_FMA(k, -MR_LK[4], r);
    r = MR_FMA(k, -MR_LK[5], r);
    // r, or -r for odd k; -0 >= 0 holds, as step(-0.0) = 1 requires
    return mr_hilo((int)((unsigned int)mr_hi32(r) ^ ((unsigned int)mr_lo32(t) << 31)), mr_lo32(r)) >= 0.0;
}
#ifdef MR_LIBM_HOST
static int mr_sin_ge0_slow(double x) { return mr_sin_eo(x) >= 0.0; }
#else
static __device__ __noinline__ int mr_sin_ge0_slow(double x) { return mr_sin_eo(x) >= 0.0; }   // one copy, not one per sine
#endif
MR_FN int mr_sin_ge0(double x) {
    int ge = mr_sin_ge0_fast(x);                 // safe for any argument; repaired below (the cold block goes out of line)
    if (MR_UNLIKELY(!mr_sin_inrange_f(x))) ge = mr_sin_ge0_slow(x);
    return ge;
}

#ifndef MR_LIBM_HOST
// One out-of-line evaluation: what the NVRTC back end emits for a transcendental that is not in a batch.
static __device__ __noinline__ double mr_sin_call(double a) { return mr_sin_eo(a); }
static __device__ __noinline__ double mr_exp_call(double a) { return mr_exp_eo(a); }
static __device__ __noinline__ double mr_log_call(double a) { return mr_log_eo(a); }

// Scratch-batched form (the NVRTC back end's default for transcendental-heavy programs).  Arguments
// and results travel through a per-thread column of dynamic shared memory, MR_S(k) = row k of this
// thread, instead of the call ABI's fixed registers: one STS + one LDS per value replaces four moves,
// and the helper is a LEAF with a four-wide loop -- no nested call, so nothing has to survive one, no
// callee-saved registers are touched and nothing is spilled (helpers that took four arguments and
// returned four results in the call ABI's registers spent 4/5 of their instructions on exactly that).
// The loop body is a few hundred bytes and stays in the instruction cache, which is what bounds
// straight-line code of this size (DESIGN.md 3.1).
// Out-of-range arguments are left in place and reported in the returned mask; the caller hands the
// mask to mr_*_fix (libdevice), a call that is practically never executed.
#ifdef MR_SCR_STRIDE
extern __shared__ double mr_dyn_f64[];
#define MR_S(k) mr_dyn_f64[(k) * MR_SCR_STRIDE + threadIdx.x]
// Independent evaluations per loop iteration (the scratch has 8 rows).  4 since the sine lost its table loads and
// selects (measured, deep scene at 20 000 values: 13.4 ms against 13.8 with 2; with round 1's sine 4 did not pay: the
// helper has the ~38 registers its caller leaves).
#define MR_W 4
#define MR_EACH _Pragma("unroll") for (int i = 0; i < MR_W; i++)
// glibc's exp and log tables (2 KB each) sit in shared memory behind the 16 scratch rows, copied there once per block
// by mr_scratch_tables_init().  A lookup is then one LDS.128 at a 32-bit offset instead of a 64-bit address computation
// (IADD3 + IMAD.X) and an LDG whose latency is the long scoreboard's (measured, deep scene at 20 000 values: 12.87 ms
// against 13.35 with the tables in global memory).
#define MR_TAB_EXP (reinterpret_cast<const unsigned long long*>(mr_dyn_f64 + 16 * MR_SCR_STRIDE))
#define MR_TAB_LOG (mr_dyn_f64 + 16 * MR_SCR_STRIDE + 256)
#define MR_TAB_LD2U(p, a, b) do { const ulonglong2 v2_ = *reinterpret_cast<const ulonglong2*>(p); (a) = v2_.x; (b) = v2_.y; } while (0)
#define MR_TAB_LD2(p, a, b) do { const double2 v2_ = *reinterpret_cast<const double2*>(p); (a) = v2_.x; (b) = v2_.y; } while (0)
__device__ __forceinline__ void mr_scratch_tables_init() {
    for (unsigned int i = threadIdx.x; i < 256u; i += blockDim.x) {
        reinterpret_cast<unsigned long long*>(mr_dyn_f64 + 16 * MR_SCR_STRIDE)[i] = MRG_EXP_TAB[i];
        mr_dyn_f64[16 * MR_SCR_STRIDE + 256 + i] = MRG_LOG_TAB[i];
    }
    __syncthreads();
}
// The fast paths again, MR_W evaluations at a time and written STEP-MAJOR: every step is applied to
// all lanes before the next one, so the lanes' dependent DFMA chains are interleaved in program order.
// (Left to itself the compiler emits one whole chain after the other -- measured: 47 % of the helpers'
// cycles were fixed-latency waits on the previous DFMA with 4 warps per scheduler.)  Same operations in
// the same order per lane as mr_sin_fast / mr_exp_fast / mr_log_fast: bit-identical results.
__device__ __forceinline__ void mr_sin_fast_w_f(const double* x, double* out) {
    double t[MR_W], k[MR_W], r[MR_W], s[MR_W], p34[MR_W], p56[MR_W], p78[MR_W], s2[MR_W], S[MR_W];
    MR_EACH t[i] = MR_FMA(x[i], MR_LK[2], MR_LK[0]);
    MR_EACH k[i] = t[i] - MR_LK[0];
    MR_EACH r[i] = MR_FMA(k[i], -MR_LK[3], x[i]);
    MR_EACH r[i] = MR_FMA(k[i], -MR_LK[4], r[i]);
    MR_EACH r[i] = MR_FMA(k[i], -MR_LK[5], r[i]);
    MR_EACH s[i] = r[i] * r[i];
    MR_EACH p34[i] = MR_FMA(MR_LK[10], s[i], MR_LK[9]);
    MR_EACH p56[i] = MR_FMA(MR_LK[12], s[i], MR_LK[11]);
    MR_EACH p78[i] = MR_FMA(MR_LK[14], s[i], MR_LK[13]);
    MR_EACH s2[i] = s[i] * s[i];
    MR_EACH S[i] = MR_FMA(p56[i], s2[i], p34[i]);
    MR_EACH S[i] = MR_FMA(p78[i], s2[i] * s2[i], S[i]);
    MR_EACH S[i] = MR_FMA(S[i], s[i], MR_LK[8]);
    MR_EACH S[i] = MR_FMA(S[i], s[i], MR_LK[7]);
    MR_EACH S[i] = MR_FMA(S[i], s[i], MR_LK[6]);
    MR_EACH {
        const double v = MR_FMA(MR_FMA(S[i], s[i], 0.0), r[i], r[i]);
        out[i] = mr_hilo((int)((unsigned int)mr_hi32(v) ^ ((unsigned int)mr_lo32(t[i]) << 31)), mr_lo32(v));
    }
}
// glibc's exp, MR_W evaluations step-major: same operations per lane as mr_exp_fast_g.
__device__ __forceinline__ void mr_exp_fast_w_f(const double* x, double* out) {
    double kd0[MR_W], kd[MR_W], r[MR_W], tail[MR_W], p23[MR_W], tr[MR_W], r2[MR_W], p45[MR_W], t1[MR_W], scale[MR_W];
    MR_EACH kd0[i] = MR_FMA(x[i], MRG_EXP_K[0], MRG_EXP_K[1]);
    MR_EACH kd[i] = kd0[i] - MRG_EXP_K[1];
    MR_EACH r[i] = MR_FMA(kd[i], MRG_EXP_K[2], x[i]);
    MR_EACH r[i] = MR_FMA(kd[i], MRG_EXP_K[3], r[i]);
    MR_EACH {
        const unsigned int ki = (unsigned int)mr_lo32(kd0[i]);
        unsigned long long tb, sb;
        MR_TAB_LD2U(MR_TAB_EXP + 2 * (ki & 127u), tb, sb);
        sb += (unsigned long long)ki << 45;
        tail[i] = mr_hilo((int)(tb >> 32), (int)(unsigned int)tb);
        scale[i] = mr_hilo((int)(sb >> 32), (int)(unsigned int)sb);
    }
    MR_EACH p23[i] = MR_FMA(r[i], MRG_EXP_K[5], MRG_EXP_K[4]);
    MR_EACH tr[i] = r[i] + tail[i];
    MR_EACH r2[i] = r[i] * r[i];
    MR_EACH p45[i] = MR_FMA(r[i], MRG_EXP_K[7], MRG_EXP_K[6]);
    MR_EACH t1[i] = MR_FMA(p23[i], r2[i], tr[i]);
    MR_EACH r2[i] = r2[i] * r2[i];
    MR_EACH t1[i] = MR_FMA(r2[i], p45[i], t1[i]);
    MR_EACH out[i] = MR_FMA(scale[i], t1[i], scale[i]);
}
// glibc's log: the table path for all lanes step-major, then the lanes close to 1 (a different polynomial) again.
__device__ __forceinline__ void mr_log_fast_w_f(const double* x, double* out) {
    double z[MR_W], invc[MR_W], logc[MR_W], kd[MR_W], w[MR_W], r[MR_W], a12[MR_W], hi[MR_W], r2[MR_W], lo[MR_W], r3[MR_W], a34[MR_W];
    MR_EACH {
        const int hx = mr_hi32(x[i]);
        const int th = hx - 0x3fe60000;
        z[i] = mr_hilo(hx - (int)((unsigned int)th & 0xfff00000u), mr_lo32(x[i]));
        MR_TAB_LD2(MR_TAB_LOG + 2 * ((th >> 13) & 127), invc[i], logc[i]);
        kd[i] = (double)(th >> 20);
    }
    MR_EACH w[i] = MR_FMA(kd[i], MRG_LOG_K[0], logc[i]);
    MR_EACH r[i] = MR_FMA(z[i], invc[i], -1.0);
    MR_EACH a12[i] = MR_FMA(r[i], MRG_LOG_K[4], MRG_LOG_K[3]);
    MR_EACH hi[i] = r[i] + w[i];
    MR_EACH r2[i] = r[i] * r[i];
    MR_EACH lo[i] = (w[i] - hi[i]) + r[i];
    MR_EACH lo[i] = MR_FMA(kd[i], MRG_LOG_K[1], lo[i]);
    MR_EACH r3[i] = r[i] * r2[i];
    MR_EACH a34[i] = MR_FMA(r[i], MRG_LOG_K[6], MRG_LOG_K[5]);
    MR_EACH lo[i] = MR_FMA(r2[i], MRG_LOG_K[2], lo[i]);
    MR_EACH a34[i] = MR_FMA(a34[i], r2[i], a12[i]);
    MR_EACH out[i] = MR_FMA(r3[i], a34[i], lo[i]) + hi[i];
    MR_EACH if ((unsigned int)(mr_hi32(x[i]) - 0x3fee0000) < 0x30900u) out[i] = mr_log_fast_g(x[i]);
}
#ifdef MR_LIBM_GLIBC
// The exact mode branches inside an evaluation (ranges of sin, the near-1 path of log), so it is not written step-major.
#define MR_DEFINE_FAST_W(fn) __device__ __forceinline__ void mr_##fn##_fast_w(const double* x, double* out) { MR_EACH out[i] = mr_##fn##_fast_g(x[i]); }
#else
#define MR_DEFINE_FAST_W(fn) __device__ __forceinline__ void mr_##fn##_fast_w(const double* x, double* out) { mr_##fn##_fast_w_f(x, out); }
#endif
MR_DEFINE_FAST_W(sin)
MR_DEFINE_FAST_W(exp)
MR_DEFINE_FAST_W(log)
// Rows 0..7 of the scratch hold the arguments and are left intact; results go to rows 8..15
// (MR_R(k)).  The helper returns one flag, "some argument was outside the fast range", and mr_*_fix
// then recomputes exactly those rows with libdevice: no per-lane mask, no selects on the stores.
#define MR_R(k) MR_S(8 + (k))
#define MR_DEFINE_SCRATCH_BATCH_S(fn, SLOW, SUF)                                                              \
    static __device__ __noinline__ unsigned int mr_##fn##_batch##SUF(const unsigned int n) {                \
        bool all_ok = true;                                                                            \
        double* s = mr_dyn_f64 + threadIdx.x;                                                          \
        for (unsigned int k = 0; k < n; k += MR_W, s += MR_W * MR_SCR_STRIDE) {                        \
            double x[MR_W], r[MR_W];                                                                   \
            MR_EACH x[i] = s[i * MR_SCR_STRIDE];   /* rows past n: stale but in bounds, results unused */ \
            mr_##fn##_fast_w(x, r);                                                                    \
            MR_EACH s[(8 + i) * MR_SCR_STRIDE] = r[i];                                                 \
            MR_EACH all_ok &= mr_##fn##_inrange(x[i]);   /* rows past n included: a stale row can only */ \
                                                         /* raise the flag, and mr_*_fix looks at rows < n */ \
        }                                                                                              \
        return all_ok ? 0u : 1u;                                                                       \
    }                                                                                                  \
    static __device__ __noinline__ void mr_##fn##_fix##SUF(const unsigned int n) {                          \
        for (unsigned int k = 0; k < n; k++)                                                           \
            if (!mr_##fn##_inrange(MR_S(k))) MR_R(k) = SLOW(MR_S(k));                                  \
    }
// One instance per segment function (MR_BATCH_HELPERS(_s3)): in a large single unit, helpers shared by
// every segment are compiled against the generic call ABI and spill; private copies keep the
// compiler's per-caller register coordination (measured, DESIGN.md 3.1).
#define MR_BATCH_HELPERS(SUF)                                  \
    MR_DEFINE_SCRATCH_BATCH_S(sin, MR_SLOW_SIN, SUF)           \
    MR_DEFINE_SCRATCH_BATCH_S(exp, MR_SLOW_EXP, SUF)           \
    MR_DEFINE_SCRATCH_BATCH_S(log, MR_SLOW_LOG, SUF)
#ifndef MR_NO_DEFAULT_BATCH_HELPERS
MR_BATCH_HELPERS()
#endif
#endif  // MR_SCR_STRIDE
#endif

#endif  // MR_LIBM_PLAIN
#endif  // MARAY_DEVICE_LIBM_CUH
