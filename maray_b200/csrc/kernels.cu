// Hand-written sm_100a kernels of the render path:
//   maray_interp<P>   -- the bytecode interpreter (MARAY_BACKEND_INTERP), P pixels per thread
//   fp64_issue_rate   -- FP64-pipe issue-rate microbenchmark (the roofline denominator)
//   band_signal/wait  -- the completion signal of the one-process-per-GPU band render (counters behind the shared frame)
// The NVRTC back end's kernel is generated at run time (codegen.cpp) from the same device_sem.cuh.
//
// Compiled with --fmad=false: the reference never fuses a*b+c (SURVEY.md Appendix B).
#include <cuda_runtime.h>

#include <cstdint>

#include "bytecode.hpp"
#define MR_LIBM_BOTH 1   // fast libm under the plain names, the exact mode (glibc's bits) as mr_*_g: chosen at run time
#include "device_sem.cuh"
#include "interp_dispatch.inc"   // generated: tools/gen_interp_dispatch.py (jump-table dispatch + hot bodies, inline PTX)
#include "kernels.hpp"

namespace maray {

// ------------------------------------------------------------------------------------------------
// Bytecode interpreter (bytecode.hpp, version 3).
//
// Mapping: a block of B threads renders B*P consecutive pixels of ONE image row (thread t: columns
// xs + k*B + t, k < P); the grid is (blocks per row) x (rows).  Values that depend on x are WIDE: P per
// thread, in registers while they are the accumulator, otherwise in the per-thread slot file in shared
// memory (16-byte words per thread for P >= 2, so one LDS.128 moves two pixels and a warp's accesses are
// conflict-free).  Values that do not depend on x are SCALARS: one per block, kept with the constants
// in a small scalar file every lane reads as a broadcast, computed with one FP64 instruction per warp.
// Every warp computes and stores every scalar itself (same bits), and scalar slots are never recycled,
// so a warp only ever reads what it wrote: no barrier.  The instruction stream is warp-uniform: staged
// from global memory in double-buffered chunks with cp.async, every lane reads the same word.
//
// Dispatch: the handler id in the low byte selects, with ONE indexed branch, a body specialised on the
// operation AND on where both operands come from (accumulator / slot / scalar file / scalar
// accumulator), so a body is just its loads, P FP64 instructions and nothing else; the store (a flag)
// follows the switch.  Rare forms (texture fetch, everything in the scalar shape) take generic bodies
// that read the operand kinds from the flags.

constexpr int kChunk = kBcChunk;   // instruction words per staged chunk (2 KiB); the stream is a whole number of chunks

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    unsigned int s = (unsigned int)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

// The per-thread view of the two files.  Wide slot operands arrive PRE-SCALED by the host (the launch
// shape is fixed when the program is uploaded): field = slot * (P * B) / 2, the slot's offset in 16-byte
// units (P * B is even for every shape), so an address is one shift-add.
template <int P>
struct Files {
    unsigned char* wide;        // this thread's first byte of wide slot 0
    unsigned int half_stride;   // P == 4: bytes between the two 16-byte halves of a slot (16 * B)
    const double* scal;         // scalar file (constants, then row-uniform slots)

    __device__ __forceinline__ void load(unsigned int s16, double (&v)[P]) const {
        const unsigned char* q = wide + ((size_t)s16 << 4);
        if constexpr (P == 1) {
            v[0] = *reinterpret_cast<const double*>(q);
        } else {
#pragma unroll
            for (int hlf = 0; hlf < P / 2; hlf++) {
                const double2 t = *reinterpret_cast<const double2*>(q + hlf * half_stride);
                v[2 * hlf] = t.x; v[2 * hlf + 1] = t.y;
            }
        }
    }
    __device__ __forceinline__ void store(unsigned int s16, const double (&v)[P]) const {
        unsigned char* q = wide + ((size_t)s16 << 4);
        if constexpr (P == 1) {
            *reinterpret_cast<double*>(q) = v[0];
        } else {
#pragma unroll
            for (int hlf = 0; hlf < P / 2; hlf++)
                *reinterpret_cast<double2*>(q + hlf * half_stride) = make_double2(v[2 * hlf], v[2 * hlf + 1]);
        }
    }
};

template <int P, int K>
__device__ __forceinline__ void mr_fetch(const Files<P>& f, const double (&acc)[P], double sacc, unsigned int idx, double (&v)[P]) {
    if constexpr (K == BC_K_A) {
#pragma unroll
        for (int k = 0; k < P; k++) v[k] = acc[k];
    } else if constexpr (K == BC_K_W) {
        f.load(idx, v);
    } else if constexpr (K == BC_K_S) {
        const double s = f.scal[idx];
#pragma unroll
        for (int k = 0; k < P; k++) v[k] = s;
    } else {
#pragma unroll
        for (int k = 0; k < P; k++) v[k] = sacc;
    }
}
template <int P>
__device__ __forceinline__ void mr_fetch_rt(const Files<P>& f, const double (&acc)[P], double sacc, unsigned int kind, unsigned int idx,
                                            double (&v)[P]) {
    switch (kind) {
    case BC_K_A: mr_fetch<P, BC_K_A>(f, acc, sacc, idx, v); break;
    case BC_K_W: mr_fetch<P, BC_K_W>(f, acc, sacc, idx, v); break;
    case BC_K_S: mr_fetch<P, BC_K_S>(f, acc, sacc, idx, v); break;
    default: mr_fetch<P, BC_K_T>(f, acc, sacc, idx, v); break;
    }
}

struct OpAdd { static __device__ __forceinline__ double f(double x, double y) { return x + y; } };
struct OpMul { static __device__ __forceinline__ double f(double x, double y) { return x * y; } };
struct OpMax { static __device__ __forceinline__ double f(double x, double y) { return mr_max(x, y); } };
struct OpMin { static __device__ __forceinline__ double f(double x, double y) { return mr_min(x, y); } };
struct OpMov { static __device__ __forceinline__ double f(double x) { return x; } };
struct OpNeg { static __device__ __forceinline__ double f(double x) { return -x; } };
struct OpAbs { static __device__ __forceinline__ double f(double x) { return fabs(x); } };
struct OpRecip { static __device__ __forceinline__ double f(double x) { return mr_recip(x); } };
struct OpSqrt { static __device__ __forceinline__ double f(double x) { return mr_sqrt(x); } };
struct OpStep { static __device__ __forceinline__ double f(double x) { return mr_step(x); } };
struct OpSin { static __device__ __forceinline__ double f(double x) { return mr_sin(x); } };
struct OpExp { static __device__ __forceinline__ double f(double x) { return mr_exp(x); } };
struct OpLn { static __device__ __forceinline__ double f(double x) { return mr_log(x); } };
// Exact mode (MrTileParams::libm_exact, device_libm_glibc.cuh): out of line, so the default path's code and
// registers are what they were.
static __device__ __noinline__ double mr_sin_exact(double x) { return mr_sin_g(x); }
static __device__ __noinline__ double mr_exp_exact(double x) { return mr_exp_g(x); }
static __device__ __noinline__ double mr_log_exact(double x) { return mr_log_g(x); }
struct OpSinX { static __device__ __forceinline__ double f(double x) { return mr_sin_exact(x); } };
struct OpExpX { static __device__ __forceinline__ double f(double x) { return mr_exp_exact(x); } };
struct OpLnX { static __device__ __forceinline__ double f(double x) { return mr_log_exact(x); } };

template <int P, int KA, int KB, class Op>
__device__ __forceinline__ void mr_bin(const Files<P>& f, double (&acc)[P], double sacc, unsigned int a, unsigned int b) {
    double x[P], y[P];
    mr_fetch<P, KA>(f, acc, sacc, a, x);
    mr_fetch<P, KB>(f, acc, sacc, b, y);
#pragma unroll
    for (int k = 0; k < P; k++) acc[k] = Op::f(x[k], y[k]);
}
template <int P, int KA, class Op>
__device__ __forceinline__ void mr_un(const Files<P>& f, double (&acc)[P], double sacc, unsigned int a) {
    double x[P];
    mr_fetch<P, KA>(f, acc, sacc, a, x);
    if constexpr (KA == BC_K_S || KA == BC_K_T) {
        const double r = Op::f(x[0]);       // a scalar operand: one evaluation serves the P pixels
#pragma unroll
        for (int k = 0; k < P; k++) acc[k] = r;
    } else {
#pragma unroll
        for (int k = 0; k < P; k++) acc[k] = Op::f(x[k]);
    }
}

#define MR_BIN_ROW(OPI, OP, KA)                                                                              \
    case BC_H_BIN + (OPI) * 16 + (KA) * 4 + 0: mr_bin<P, KA, 0, OP>(F, acc, sacc, a, b); break;              \
    case BC_H_BIN + (OPI) * 16 + (KA) * 4 + 1: mr_bin<P, KA, 1, OP>(F, acc, sacc, a, b); break;              \
    case BC_H_BIN + (OPI) * 16 + (KA) * 4 + 2: mr_bin<P, KA, 2, OP>(F, acc, sacc, a, b); break;              \
    case BC_H_BIN + (OPI) * 16 + (KA) * 4 + 3: mr_bin<P, KA, 3, OP>(F, acc, sacc, a, b); break;
#define MR_BIN_CASES(OPI, OP) MR_BIN_ROW(OPI, OP, 0) MR_BIN_ROW(OPI, OP, 1) MR_BIN_ROW(OPI, OP, 2) MR_BIN_ROW(OPI, OP, 3)
#define MR_UN_CASES(U, OP)                                                                                   \
    case BC_H_UN + (U) * 4 + 0: mr_un<P, 0, OP>(F, acc, sacc, a); break;                                      \
    case BC_H_UN + (U) * 4 + 1: mr_un<P, 1, OP>(F, acc, sacc, a); break;                                      \
    case BC_H_UN + (U) * 4 + 2: mr_un<P, 2, OP>(F, acc, sacc, a); break;                                      \
    case BC_H_UN + (U) * 4 + 3: mr_un<P, 3, OP>(F, acc, sacc, a); break;
#define MR_UN_CASES_LIBM(U, OP, OPX)                                                                         \
    case BC_H_UN + (U) * 4 + 0: if (exact) mr_un<P, 0, OPX>(F, acc, sacc, a); else mr_un<P, 0, OP>(F, acc, sacc, a); break; \
    case BC_H_UN + (U) * 4 + 1: if (exact) mr_un<P, 1, OPX>(F, acc, sacc, a); else mr_un<P, 1, OP>(F, acc, sacc, a); break; \
    case BC_H_UN + (U) * 4 + 2: if (exact) mr_un<P, 2, OPX>(F, acc, sacc, a); else mr_un<P, 2, OP>(F, acc, sacc, a); break; \
    case BC_H_UN + (U) * 4 + 3: if (exact) mr_un<P, 3, OPX>(F, acc, sacc, a); else mr_un<P, 3, OP>(F, acc, sacc, a); break;
#define MR_OUT_CASES(C)                                                                                      \
    case BC_H_OUT + (C) * 4 + 0: { double x[P]; mr_fetch<P, 0>(F, acc, sacc, a, x); F.store(out16 + (C) * slot16, x); } break; \
    case BC_H_OUT + (C) * 4 + 1: { double x[P]; mr_fetch<P, 1>(F, acc, sacc, a, x); F.store(out16 + (C) * slot16, x); } break; \
    case BC_H_OUT + (C) * 4 + 2: { double x[P]; mr_fetch<P, 2>(F, acc, sacc, a, x); F.store(out16 + (C) * slot16, x); } break; \
    case BC_H_OUT + (C) * 4 + 3: { double x[P]; mr_fetch<P, 3>(F, acc, sacc, a, x); F.store(out16 + (C) * slot16, x); } break;

template <int P>
__global__ void __launch_bounds__(512) maray_interp(const MrTileParams p, const uint64_t* __restrict__ code, unsigned int n_instr,
                                                    const double* __restrict__ consts, unsigned int n_consts, unsigned int n_scal,
                                                    unsigned int n_wide, unsigned int all_wide) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // layout: [2][kChunk] instruction words | staging tile (3*B*P bytes, 16-aligned) | scalar file | wide slots (+3 channel slots)
    uint64_t* code_s = reinterpret_cast<uint64_t*>(smem_raw);
    unsigned char* stage = smem_raw + 2 * kChunk * sizeof(uint64_t);
    const unsigned int B = blockDim.x;
    const unsigned int tid = threadIdx.x;
    double* scal = reinterpret_cast<double*>(stage + ((3u * B * P + 15u) & ~15u));
    double* wide = scal + ((n_scal + 1u) & ~1u);

    Files<P> F;
    F.wide = reinterpret_cast<unsigned char*>(wide + (P == 1 ? tid : 2u * tid));
    F.half_stride = 16u * B;
    F.scal = scal;
    const unsigned int wbase_s = (unsigned int)__cvta_generic_to_shared(F.wide);   // the same, as shared-window addresses
    const unsigned int sbase_s = (unsigned int)__cvta_generic_to_shared(scal);
    const unsigned int slot16 = P * B / 2u;              // one wide slot in 16-byte units
    const unsigned int out16 = n_wide * slot16;          // the three channel slots follow the program's slots

    const bool exact = p.libm_exact != 0u;

    const unsigned int row = blockIdx.x / p.nxb;
    const unsigned int xb = blockIdx.x - row * p.nxb;
    const unsigned int yi = p.y0 + row;
    const unsigned int xs = p.x0 + xb * B * P;          // first column of this block
    double acc[P];
    double sacc = 0.0;
    {
        double xv[P], yv[P];
#pragma unroll
        for (int k = 0; k < P; k++) {
            const unsigned int xi = xs + k * B + tid;
            // idle lanes redo the row's last pixel; `x as f64` (reference src/render.rs:25) plus the pass's offset
            xv[k] = (double)(xi < p.x1 ? xi : p.x1 - 1u) + p.ox;
            yv[k] = (double)yi + p.oy;
            acc[k] = 0.0;
        }
        F.store(0, xv);
        if (all_wide) F.store(slot16, yv);
    }
    for (unsigned int i = tid; i < n_consts; i += B) scal[i] = consts[i];
    if (!all_wide && tid == 0) scal[n_consts] = (double)yi + p.oy;   // Y stays uniform along the row in every pass

    // The stream is a whole number of chunks (bytecode_for_launch): all but the last end with YIELD, the last
    // is padded with END.
    const unsigned int n_chunks = n_instr / kChunk;
    for (unsigned int i = tid; i < kChunk / 2; i += B) cp_async16(code_s + 2 * i, code + 2 * i);   // prefetch chunk 0
    cp_async_commit();

    for (unsigned int c = 0; c < n_chunks; c++) {
        cp_async_wait_all();
        __syncthreads();   // chunk c (and, first time, the scalar file and X/Y) landed; chunk c-1 is done
        if (c + 1 < n_chunks) {
            uint64_t* dst = code_s + ((c + 1) & 1) * kChunk;
            const uint64_t* src = code + (size_t)(c + 1) * kChunk;
            for (unsigned int i = tid; i < kChunk / 2; i += B) cp_async16(dst + 2 * i, src + 2 * i);
            cp_async_commit();
        }
        const uint64_t* cs = code_s + (c & 1) * kChunk;
        const unsigned int cs_s = (unsigned int)__cvta_generic_to_shared(cs);
        unsigned int pc = cs_s;                            // shared-window address of the current instruction word
        for (;;) {
            // Inner loop (inline PTX, interp_dispatch.inc): fetch, indexed branch into a body specialised on
            // operation and operand kinds, store, next -- until an instruction it has no body for.
            if constexpr (P == 1) MR_INTERP_LOOP_P1(acc[0], sacc, pc, wbase_s, sbase_s, F.half_stride);
            else if constexpr (P == 2) MR_INTERP_LOOP_P2(acc[0], acc[1], sacc, pc, wbase_s, sbase_s, F.half_stride);
            else MR_INTERP_LOOP_P4(acc[0], acc[1], acc[2], acc[3], sacc, pc, wbase_s, sbase_s, F.half_stride);
            // The instruction it stopped at goes through the C++ switch, which implements EVERY handler.
            const uint64_t w = cs[(pc - cs_s) >> 3];
            pc += 8u;
            const unsigned int lo = (unsigned int)w, hi = (unsigned int)(w >> 32);
            const unsigned int h = lo & 0xffu;
            const unsigned int a = hi & 0xffffu, b = hi >> 16;   // wide indices pre-scaled by the host: see Files
            if (h <= BC_H_YIELD) break;                          // YIELD: next chunk; END: the last chunk is done
            if (h < BC_H_SCALAR || h >= BC_H_BINN) {
                switch (h) {
                    MR_BIN_CASES(0, OpAdd)
                    MR_BIN_CASES(1, OpMul)
                    MR_BIN_CASES(2, OpMax)
                    MR_BIN_CASES(3, OpMin)
                    MR_UN_CASES(0, OpNeg)
                    MR_UN_CASES(1, OpAbs)
                    MR_UN_CASES(2, OpRecip)
                    MR_UN_CASES(3, OpSqrt)
                    MR_UN_CASES(4, OpStep)
                    MR_UN_CASES_LIBM(5, OpSin, OpSinX)
                    MR_UN_CASES_LIBM(6, OpExp, OpExpX)
                    MR_UN_CASES_LIBM(7, OpLn, OpLnX)
                    MR_UN_CASES(8, OpMov)
                    MR_OUT_CASES(0)
                    MR_OUT_CASES(1)
                    MR_OUT_CASES(2)
                case BC_H_TEX: {
                    double x[P], y[P];
                    mr_fetch_rt<P>(F, acc, sacc, (lo >> (8 + BC_F_KA_SHIFT)) & 3u, a, x);
                    mr_fetch_rt<P>(F, acc, sacc, (lo >> (8 + BC_F_KB_SHIFT)) & 3u, b, y);
                    const unsigned int imm = lo >> 16;
                    const MrTexture t = p.tex[imm >> 2];
#pragma unroll
                    for (int k = 0; k < P; k++) acc[k] = mr_tex(t.data, t.w, t.h, imm & 3u, x[k], y[k]);
                } break;
                default:
                    if (h >= BC_H_BINN) {
                        // binary operation whose accumulator operand is negated first (a `neg` fused into its consumer)
                        const unsigned int ka = (lo >> (8 + BC_F_KA_SHIFT)) & 3u, kb = (lo >> (8 + BC_F_KB_SHIFT)) & 3u;
                        double x[P], y[P];
                        mr_fetch_rt<P>(F, acc, sacc, ka, a, x);
                        mr_fetch_rt<P>(F, acc, sacc, kb, b, y);
#pragma unroll
                        for (int k = 0; k < P; k++) {
                            if (ka == BC_K_A) x[k] = -x[k]; else y[k] = -y[k];
                            switch ((h - BC_H_BINN) / 6u) {
                            case 0: acc[k] = x[k] + y[k]; break;
                            case 1: acc[k] = x[k] * y[k]; break;
                            case 2: acc[k] = mr_max(x[k], y[k]); break;
                            default: acc[k] = mr_min(x[k], y[k]); break;
                            }
                        }
                    }
                    break;
                }
                if ((lo & (BC_F_STORE << 8)) && h != BC_H_TEX) F.store(lo >> 16, acc);
            } else {
                // scalar shape: one value per block, operands from the scalar file or the scalar accumulator
                const double x = ((lo >> (8 + BC_F_KA_SHIFT)) & 3u) == BC_K_T ? sacc : scal[a];
                const double y = ((lo >> (8 + BC_F_KB_SHIFT)) & 3u) == BC_K_T ? sacc : scal[b];
                const unsigned int op = h < BC_H_SUN ? BC_ADD + ((h - BC_H_SBIN) >> 2)
                                      : h < BC_H_STEX ? (((h - BC_H_SUN) >> 1) == 8u ? (unsigned)BC_MOV : BC_NEG + ((h - BC_H_SUN) >> 1))
                                                      : (unsigned)BC_TEX;
                switch (op) {
                case BC_MOV: sacc = x; break;
                case BC_ADD: sacc = x + y; break;
                case BC_MUL: sacc = x * y; break;
                case BC_MAX: sacc = mr_max(x, y); break;
                case BC_MIN: sacc = mr_min(x, y); break;
                case BC_NEG: sacc = -x; break;
                case BC_ABS: sacc = fabs(x); break;
                case BC_RECIP: sacc = mr_recip(x); break;
                case BC_SQRT: sacc = mr_sqrt(x); break;
                case BC_STEP: sacc = mr_step(x); break;
                case BC_SIN: sacc = exact ? mr_sin_exact(x) : mr_sin(x); break;
                case BC_EXP: sacc = exact ? mr_exp_exact(x) : mr_exp(x); break;
                case BC_LN: sacc = exact ? mr_log_exact(x) : mr_log(x); break;
                case BC_TEX: {
                    const unsigned int imm = lo >> 16;
                    const MrTexture t = p.tex[imm >> 2];
                    sacc = mr_tex(t.data, t.w, t.h, imm & 3u, x, y);
                } break;
                default: break;
                }
                if ((lo & (BC_F_STORE << 8)) && op != BC_TEX) scal[lo >> 16] = sacc;   // same bits from every lane
            }
        }
    }

    // `as u8` + RGB pack through the staging tile, then coalesced 16-byte stores.  A supersampling pass first adds its
    // samples to the accumulator; only the last pass stores (the pass index is uniform, so the whole block returns).
    const unsigned int ww = p.x1 - p.x0;
    const size_t row_first = (size_t)row * ww + (xs - p.x0);     // index of this block's first pixel in the output
    {
        double o_r[P], o_g[P], o_b[P];
        F.load(out16, o_r);
        F.load(out16 + slot16, o_g);
        F.load(out16 + 2u * slot16, o_b);
        MrSampling sp;
        sp.acc = p.acc; sp.pass = p.pass; sp.count = p.count;
        bool store = true;
#pragma unroll
        for (int k = 0; k < P; k++) {
            const unsigned int l = k * B + tid;                  // pixel within the block
            unsigned int r8 = mr_as_u8(o_r[k]), g8 = mr_as_u8(o_g[k]), b8 = mr_as_u8(o_b[k]);
            if (p.acc != nullptr) store = mr_accumulate(sp, row_first + l, xs + l < p.x1, r8, g8, b8);
            stage[3u * l + 0u] = (unsigned char)r8;
            stage[3u * l + 1u] = (unsigned char)g8;
            stage[3u * l + 2u] = (unsigned char)b8;
            if (p.f64_out != nullptr && xs + l < p.x1) {
                p.f64_out[row_first + l] = o_r[k];
                p.f64_out[(size_t)p.f64_plane + row_first + l] = o_g[k];
                p.f64_out[2u * (size_t)p.f64_plane + row_first + l] = o_b[k];
            }
        }
        if (!store) return;
    }
    __syncthreads();
    const unsigned int span = B * P;
    const unsigned int valid = (p.x1 - xs < span) ? (p.x1 - xs) : span;
    unsigned char* dst = p.out + 3u * row_first;
    if (p.out_aligned && valid == span && (span & 15u) == 0u && ((3u * row_first) & 15u) == 0u) {
        for (unsigned int i = tid; i < 3u * span / 16u; i += B)
            reinterpret_cast<uint4*>(dst)[i] = reinterpret_cast<const uint4*>(stage)[i];
    } else {
        for (unsigned int i = tid; i < 3u * valid; i += B) dst[i] = stage[i];
    }
}

size_t interp_smem_bytes(unsigned int block, unsigned int pixels_per_thread, unsigned int n_wide, unsigned int n_scal) {
    size_t stage = (3u * (size_t)block * pixels_per_thread + 15u) & ~size_t(15);
    return 2 * kChunk * sizeof(uint64_t) + stage + (size_t)((n_scal + 1u) & ~1u) * sizeof(double) +
           (size_t)(n_wide + 3u) * pixels_per_thread * block * sizeof(double);   // + 3 channel-output slots
}

template <int P>
static cudaError_t launch_interp_as(const MrTileParams& p, const uint64_t* d_code, unsigned int n_instr, const double* d_consts,
                                    unsigned int n_consts, unsigned int n_scal, unsigned int n_wide, bool all_wide,
                                    unsigned int block, unsigned int grid, size_t smem, cudaStream_t stream) {
    cudaError_t e = cudaFuncSetAttribute(maray_interp<P>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    maray_interp<P><<<grid, block, smem, stream>>>(p, d_code, n_instr, d_consts, n_consts, n_scal, n_wide, all_wide ? 1u : 0u);
    return cudaGetLastError();
}

cudaError_t launch_interp(MrTileParams p, const uint64_t* d_code, unsigned int n_instr, const double* d_consts,
                          unsigned int n_consts, unsigned int n_uniform, unsigned int n_wide, bool all_wide, unsigned int block,
                          unsigned int pixels_per_thread, cudaStream_t stream) {
    if (p.rows == 0 || p.x1 <= p.x0) return cudaSuccess;
    const unsigned int n_scal = n_consts + n_uniform;
    const size_t smem = interp_smem_bytes(block, pixels_per_thread, n_wide, n_scal);
    const unsigned int span = block * pixels_per_thread;
    p.nxb = (p.x1 - p.x0 + span - 1) / span;
    if ((uint64_t)p.nxb * p.rows > 0x7fffffffull) return cudaErrorInvalidValue;
    const unsigned int grid = p.nxb * p.rows;
#define MR_LAUNCH(PP) launch_interp_as<PP>(p, d_code, n_instr, d_consts, n_consts, n_scal, n_wide, all_wide, block, grid, smem, stream)
    switch (pixels_per_thread) {
    case 1: return MR_LAUNCH(1);
    case 2: return MR_LAUNCH(2);
    case 4: return MR_LAUNCH(4);
    default: return cudaErrorInvalidValue;
    }
#undef MR_LAUNCH
}

// ------------------------------------------------------------------------------------------------
// FP64 issue-rate microbenchmark: 8 independent DADD/DMUL chains per thread (no FMA: the render
// path has none), or 8 DFMA chains for the nominal figure.  Counts warp-instructions * 32.
template <bool FMA>
__global__ void __launch_bounds__(256) fp64_issue_rate(double* sink, int iters, double m, double a) {
    double v0 = threadIdx.x * 1e-9, v1 = v0 + 1, v2 = v0 + 2, v3 = v0 + 3, v4 = v0 + 4, v5 = v0 + 5, v6 = v0 + 6, v7 = v0 + 7;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 8; u++) {
            if (FMA) {
                v0 = __fma_rn(v0, m, a); v1 = __fma_rn(v1, m, a); v2 = __fma_rn(v2, m, a); v3 = __fma_rn(v3, m, a);
                v4 = __fma_rn(v4, m, a); v5 = __fma_rn(v5, m, a); v6 = __fma_rn(v6, m, a); v7 = __fma_rn(v7, m, a);
            } else {
                v0 = __dmul_rn(v0, m); v1 = __dadd_rn(v1, a); v2 = __dmul_rn(v2, m); v3 = __dadd_rn(v3, a);
                v4 = __dmul_rn(v4, m); v5 = __dadd_rn(v5, a); v6 = __dmul_rn(v6, m); v7 = __dadd_rn(v7, a);
            }
        }
    }
    double s = v0 + v1 + v2 + v3 + v4 + v5 + v6 + v7;
    if (s == 123.456) sink[0] = s;   // never true; keeps the chains alive
}

cudaError_t launch_fp64_issue_rate(bool fma, double* d_sink, int iters, int blocks, cudaStream_t stream) {
    if (fma) fp64_issue_rate<true><<<blocks, 256, 0, stream>>>(d_sink, iters, 1.0000001, 1e-9);
    else fp64_issue_rate<false><<<blocks, 256, 0, stream>>>(d_sink, iters, 1.0000001, 1e-9);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Completion signal between the processes that render row bands into one frame (api.cu: maray_cuda_band_signal /
// maray_cuda_band_wait).  A band kernel's stores into the frame of GPU 0 travel over NVLink; the kernel boundary
// orders them before this one 4-byte write, and the write is a system-scope release, so a reader that has seen the
// counter reach `value` (system-scope acquire) sees the band.  Both sides are atomics, performed at the home L2 of the
// counter (the exporting GPU), like every atomic over NVLink: polled with loads instead (acquire.sys or volatile), the
// exporting GPU saw a peer's write 1-50 ms late, with the atomic poll in 6-8 us (measured at N = 2,
// profiles/r02c_band_completion_signal_n2.md).  The wait is bounded: after ~2 s of polling it records a time-out and
// ends, so a lost peer can never hang the GPU.
__global__ void band_signal(unsigned int* counter, unsigned int value) {
    __threadfence_system();
    unsigned int old;
    asm volatile("atom.exch.release.sys.global.b32 %0, [%1], %2;" : "=r"(old) : "l"(counter), "r"(value) : "memory");
    (void)old;
    __threadfence_system();
}

__global__ void band_wait(unsigned int* counters, unsigned int stride, unsigned int n, unsigned int value, unsigned int* timed_out,
                          long long max_cycles) {
    const unsigned int i = threadIdx.x;
    if (i >= n) return;
    unsigned int* c = counters + size_t(i) * stride;
    const long long t0 = clock64();
    for (;;) {
        unsigned int seen;
        asm volatile("atom.add.acquire.sys.global.u32 %0, [%1], 0;" : "=r"(seen) : "l"(c) : "memory");
        if (int(seen - value) >= 0) break;               // counters only grow; wrapping compare
        if (clock64() - t0 > max_cycles) { *timed_out = 1u; break; }
        __nanosleep(64);
    }
    __threadfence_system();
}

cudaError_t launch_band_signal(unsigned int* counter, unsigned int value, cudaStream_t stream) {
    band_signal<<<1, 1, 0, stream>>>(counter, value);
    return cudaGetLastError();
}

cudaError_t launch_band_wait(unsigned int* counters, unsigned int stride, unsigned int n, unsigned int value, unsigned int* timed_out,
                             long long max_cycles, cudaStream_t stream) {
    band_wait<<<1, ((n + 31) / 32) * 32, 0, stream>>>(counters, stride, n, value, timed_out, max_cycles);
    return cudaGetLastError();
}

}  // namespace maray
