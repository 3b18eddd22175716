"""Test-side checkers of the HOST logic (lowering, code generation, bytecode), runnable without a GPU.

Nothing here is part of the product and nothing in the product can reach it:
  * host_jit_run   compiles the CUDA source the NVRTC back end generated as plain C++ with g++
                   (-ffp-contract=off) behind a shim of the few CUDA intrinsics it uses, and runs the
                   kernel body thread by thread.  It checks the generated program text, not the GPU.
  * bytecode_run   a numpy reading of the interpreter's bytecode (csrc/bytecode.hpp).
Both are compared with the oracle in tests/test_host_lowering.py.
"""
from __future__ import annotations

import ctypes
import hashlib
import math
import os
import subprocess
import tempfile

import numpy as np

HOST_SHIM = r"""
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <cstring>
#define __device__
#define __global__
#define __forceinline__ inline
#define __noinline__
#define __restrict__
#define __shared__ static
#define __constant__ static
#define __launch_bounds__(...)
#define MR_LIBM_PLAIN 1          /* the host check uses the host libm, like the oracle */
#define MR_PLAIN_FN static inline
#define MR_HOST_TEXT 1
#define MR_DYN_DECL static double mr_dyn_f64[32 * 256];   /* the scratch rows of the batched sin/exp/ln calls */
struct uint3_ { unsigned int x, y, z; };
static uint3_ threadIdx, blockIdx, blockDim;
struct uint4 { unsigned int x, y, z, w; };
static inline double __drcp_rn(double v) { return 1.0 / v; }
static inline double __dsqrt_rn(double v) { return std::sqrt(v); }
static inline unsigned int __double2uint_rz(double v) {
    if (v != v) return 0xffffffffu;   // pessimistic: generated code must not rely on NaN -> 0
    if (!(v > 0.0)) return 0u;
    if (v >= 4294967295.0) return 4294967295u;
    return (unsigned int)v;
}
static inline unsigned char __ldg(const unsigned char* p) { return *p; }
static inline double __ldg(const double* p) { return *p; }
static inline double __longlong_as_double(long long b) { double d; std::memcpy(&d, &b, 8); return d; }
static inline void __syncthreads() {}
using std::fabs; using std::fmax; using std::fmin;
#ifdef MR_HOST_PERTURB_LIBM
// Conditioning probe: every sin/exp/log result is moved by -1, 0 or +1 unit in the last place (chosen by a
// hash of the argument).  A scene whose bytes survive this is insensitive to which libm evaluates it.
static inline double mr_nudge(double v, double x) {
    if (!(v - v == 0.0) || v == 0.0) return v;
    unsigned long long b, hsh; std::memcpy(&b, &v, 8); std::memcpy(&hsh, &x, 8);
    hsh *= 0x9E3779B97F4A7C15ull; hsh ^= hsh >> 29;
    b += (unsigned long long)((long long)(hsh % 3) - 1);
    std::memcpy(&v, &b, 8); return v;
}
static inline double mr_host_sin(double x) { return mr_nudge(std::sin(x), x); }
static inline double mr_host_exp(double x) { return mr_nudge(std::exp(x), x); }
static inline double mr_host_log(double x) { return mr_nudge(std::log(x), x); }
#define sin mr_host_sin
#define exp mr_host_exp
#define log mr_host_log
#else
using std::sin; using std::exp; using std::log;
#endif
"""

HOST_DRIVER = r"""
extern "C" void host_run(unsigned char* out, double* f64_out, unsigned long long plane, const MrTexture* tex,
                         unsigned int p0, unsigned int n, unsigned int W) {
    MrParams p;
    p.out = out; p.f64_out = f64_out; p.f64_plane = plane; p.tex = tex; p.p0 = p0; p.n = n; p.W = W;
    p.out_aligned = 0;
    blockDim.x = 256; blockDim.y = blockDim.z = 1;
    unsigned int blocks = (n + 255) / 256;
    for (unsigned int b = 0; b < blocks; b++) {
        blockIdx.x = b;
        // two passes: after the first every thread's bytes are in the staging tile, so the second
        // pass's cooperative copy-out sees a complete tile (sequential stand-in for __syncthreads)
        for (int pass = 0; pass < 2; pass++)
            for (unsigned int t = 0; t < 256; t++) { threadIdx.x = t; maray_jit(p); }
    }
}
"""


# Chain form (one kernel per segment, values crossing a cut in a global frame F[slot * FS + pixel]): each
# translation unit becomes its own shared object; they run in order over one frame buffer.
HOST_DRIVER_CHAIN = r"""
extern "C" void host_run(unsigned char* out, double* f64_out, unsigned long long plane, const MrTexture* tex,
                         unsigned int p0, unsigned int n, unsigned int W, double* F, unsigned long long FS) {
    MrParams p;
    p.out = out; p.f64_out = f64_out; p.f64_plane = plane; p.tex = tex; p.p0 = p0; p.n = n; p.W = W;
    p.out_aligned = 0;
    blockDim.x = 256; blockDim.y = blockDim.z = 1;
    unsigned int blocks = (n + 255) / 256;
    for (unsigned int b = 0; b < blocks; b++) {
        blockIdx.x = b;
        for (int pass = 0; pass < 2; pass++)          // see HOST_DRIVER: second pass = after the barrier
            for (unsigned int t = 0; t < 256; t++) { threadIdx.x = t; maray_jit(p, F, FS); }
    }
}
"""


class _Tex(ctypes.Structure):
    _fields_ = [("data", ctypes.c_void_p), ("w", ctypes.c_uint32), ("h", ctypes.c_uint32)]


_CACHE = {}


def host_jit_run(source: str, w: int, p0: int, n: int, textures=(), perturb_libm: bool = False):
    """Runs the generated kernel text on the CPU.  Returns (rgb uint8 (n,3), planes float64 (3,n)).
    perturb_libm: every sin/exp/log result is moved by up to one unit in the last place (conditioning probe)."""
    key = hashlib.sha256(source.encode()).hexdigest() + ("p" if perturb_libm else "")
    lib = _CACHE.get(key)
    if lib is None:
        d = tempfile.mkdtemp(prefix="maray_hostjit_")
        src = os.path.join(d, "k.cpp")
        with open(src, "w") as f:
            if perturb_libm:
                f.write("#define MR_HOST_PERTURB_LIBM 1\n")
            f.write(HOST_SHIM)
            f.write(source.replace('extern "C" __global__', "static"))
            f.write(HOST_DRIVER)
        so = os.path.join(d, "k.so")
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC",
                               "-w", "-o", so, src])
        lib = ctypes.CDLL(so)
        lib.host_run.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_ulonglong, ctypes.c_void_p,
                                 ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32]
        _CACHE[key] = lib
    rgb = np.zeros((n, 3), dtype=np.uint8)
    planes = np.zeros((3, n), dtype=np.float64)
    arrs = [np.ascontiguousarray(t, dtype=np.uint8) for t in textures]
    tab = (_Tex * max(1, len(arrs)))()
    for i, a in enumerate(arrs):
        tab[i].data = a.ctypes.data
        tab[i].w, tab[i].h = a.shape[1], a.shape[0]
    lib.host_run(rgb.ctypes.data, planes.ctypes.data, n, ctypes.addressof(tab), p0, n, w)
    return rgb, planes


def host_chain_run(modules, w: int, p0: int, n: int, frame_slots: int, textures=()):
    """Runs the chain form of a program (CudaRenderer.modules(): one kernel per segment) on the CPU: every unit
    is compiled on its own and they run in order over one frame.  Returns (rgb uint8 (n,3), planes float64 (3,n))."""
    rgb = np.zeros((n, 3), dtype=np.uint8)
    planes = np.zeros((3, n), dtype=np.float64)
    arrs = [np.ascontiguousarray(t, dtype=np.uint8) for t in textures]
    tab = (_Tex * max(1, len(arrs)))()
    for i, a in enumerate(arrs):
        tab[i].data = a.ctypes.data
        tab[i].w, tab[i].h = a.shape[1], a.shape[0]
    fs = ((n + 255) // 256) * 256
    frame = np.full(max(1, frame_slots) * fs, np.nan, dtype=np.float64)     # a read of a never-written slot shows up as NaN
    for source in modules:
        key = hashlib.sha256(source.encode()).hexdigest() + "chain"
        lib = _CACHE.get(key)
        if lib is None:
            d = tempfile.mkdtemp(prefix="maray_hostjit_")
            src = os.path.join(d, "k.cpp")
            with open(src, "w") as f:
                f.write(HOST_SHIM)
                f.write(source.replace('extern "C" __global__', "static"))
                f.write(HOST_DRIVER_CHAIN)
            so = os.path.join(d, "k.so")
            subprocess.check_call(["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC",
                                   "-w", "-o", so, src])
            lib = ctypes.CDLL(so)
            lib.host_run.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_ulonglong, ctypes.c_void_p,
                                     ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_ulonglong]
            _CACHE[key] = lib
        lib.host_run(rgb.ctypes.data, planes.ctypes.data, n, ctypes.addressof(tab), p0, n, w, frame.ctypes.data, fs)
    return rgb, planes


# ---- bytecode (csrc/bytecode.hpp, version 3) -------------------------------------------------------
(BC_END, BC_MOV, BC_ADD, BC_MUL, BC_MAX, BC_MIN, BC_NEG, BC_ABS, BC_RECIP, BC_SQRT, BC_STEP, BC_SIN, BC_EXP, BC_LN,
 BC_TEX, BC_OUT_R, BC_OUT_G, BC_OUT_B) = range(18)
K_A, K_W, K_S, K_T = 0, 1, 2, 3
H_END, H_BIN, H_UN, H_OUT, H_TEX, H_SCALAR, H_SBIN, H_SUN, H_STEX, H_BINN, H_COUNT = 0, 16, 80, 116, 128, 144, 144, 160, 178, 179, 203
F_STORE, F_NEG_ACC, F_KA_SHIFT, F_KB_SHIFT = 1, 2, 2, 4


def bc_decode(w):
    """(shape_is_scalar, op, ka, kb, store, dst, a, b) of one instruction word; checks that the handler id
    and the flags agree on the operand kinds (the kernel's specialised bodies read the id, its generic
    bodies the flags).  op + 100: the accumulator operand is negated first (BC_H_BINN)."""
    w = int(w)
    h, fl, dst, a, b = w & 0xFF, (w >> 8) & 0xFF, (w >> 16) & 0xFFFF, (w >> 32) & 0xFFFF, (w >> 48) & 0xFFFF
    ka, kb = (fl >> F_KA_SHIFT) & 3, (fl >> F_KB_SHIFT) & 3
    store = bool(fl & F_STORE)
    if h == H_END:
        return False, BC_END, 0, 0, False, 0, 0, 0
    if h >= H_BINN:
        assert h < H_COUNT and (fl & F_NEG_ACC) and (ka == K_A) != (kb == K_A)
        c = (h - H_BINN) % 6
        assert c == (kb - 1 if ka == K_A else 3 + ka - 1), "handler id and flags disagree on the operand kinds"
        return False, 100 + BC_ADD + (h - H_BINN) // 6, ka, kb, store, dst, a, b
    assert not (fl & F_NEG_ACC)
    if h >= H_SCALAR:
        assert h < H_BINN and ka in (K_S, K_T), "scalar instruction with a wide operand"
        if h < H_SUN:
            op = BC_ADD + (h - H_SBIN) // 4
            assert kb in (K_S, K_T) and (h - H_SBIN) % 4 == (ka == K_T) * 2 + (kb == K_T), "handler id and flags disagree"
        elif h < H_STEX:
            u = (h - H_SUN) // 2
            op = BC_MOV if u == 8 else BC_NEG + u
            assert (h - H_SUN) % 2 == (ka == K_T), "handler id and flags disagree"
        else:
            op = BC_TEX
            assert kb in (K_S, K_T)
        return True, op, ka, kb, store, dst, a, b
    if H_BIN <= h < H_UN:
        op = BC_ADD + (h - H_BIN) // 16
        assert ((h - H_BIN) % 16) == ka * 4 + kb, "handler id and flags disagree on the operand kinds"
    elif H_UN <= h < H_OUT:
        u = (h - H_UN) // 4
        op = BC_MOV if u == 8 else BC_NEG + u
        assert (h - H_UN) % 4 == ka
    elif H_OUT <= h < H_TEX:
        op = BC_OUT_R + (h - H_OUT) // 4
        assert (h - H_OUT) % 4 == ka
    else:
        assert h == H_TEX, f"bad handler id {h}"
        op = BC_TEX
    return False, op, ka, kb, store, dst, a, b


def _vec(fn):
    def safe(v):
        try:
            return fn(v)
        except (ValueError, OverflowError):
            if fn is math.log:
                return -math.inf if v == 0 else math.nan
            if fn is math.exp:
                return math.inf
            return math.nan
    uf = np.frompyfunc(safe, 1, 1)
    return lambda a: uf(a).astype(np.float64)


_sin, _exp, _log = _vec(math.sin), _vec(math.exp), _vec(math.log)      # the host libm, like the oracle


def sem_max(a, b):
    """f64::max as the reference compiles it: NaN ignored, tie returns the first operand."""
    return np.where((b > a) | np.isnan(a), b, a)


def sem_min(a, b):
    return np.where((b < a) | np.isnan(a), b, a)


def as_u8(v):
    v = np.where(np.isnan(v), 0.0, v)
    return np.clip(np.trunc(v), 0, 255).astype(np.uint8)


def _as_u32(v):
    v = np.where(np.isnan(v), 0.0, v)
    return np.clip(np.trunc(v), 0, 4294967295).astype(np.uint64)


def tex_fetch(tex, ch, x, y):
    h, w = tex.shape[0], tex.shape[1]
    xi, yi = _as_u32(x), _as_u32(y)
    ok = ~((x < 0.0) | (y < 0.0)) & (xi < w) & (yi < h)
    out = np.zeros(x.shape, dtype=np.float64)
    out[ok] = tex[yi[ok], xi[ok], ch].astype(np.float64)
    return out


def bytecode_run(code, consts, xs, ys, textures=(), row_uniform=True):
    """Executes the bytecode for the pixels (xs[i], ys[i]) the way the kernel does: a wide accumulator and
    wide slots (one value per pixel), a scalar accumulator and the scalar file (constants, then row-uniform
    slots; ONE value for all pixels, which must therefore share one y).  Every scalar result is computed
    from pixel 0 and asserted to be what every other pixel would have computed -- a value wrongly classified
    as row-uniform fails here -- and row-uniform slots are never recycled.  Returns planes float64 (3, n)."""
    xs = np.asarray(xs, dtype=np.float64)
    ys = np.asarray(ys, dtype=np.float64)
    n = xs.shape[0]
    consts = np.asarray(consts, dtype=np.float64)
    nk = consts.shape[0]
    wide = {0: xs}
    scal = {i: float(consts[i]) for i in range(nk)}
    if row_uniform:
        assert np.unique(ys).size == 1, "row-uniform bytecode must be run one row at a time"
        scal[nk] = float(ys[0])
    else:
        wide[1] = ys
    acc = np.zeros(n)
    sacc = 0.0
    out = np.zeros((3, n))

    def wide_operand(kind, idx):
        if kind == K_A: return acc
        if kind == K_W: return wide[idx]
        if kind == K_S: return np.full(n, scal[idx])
        return np.full(n, sacc)

    def apply(op, x, y, dst):
        if op == BC_MOV: return x
        if op == BC_ADD: return x + y
        if op == BC_MUL: return x * y
        if op == BC_MAX: return sem_max(x, y)
        if op == BC_MIN: return sem_min(x, y)
        if op == BC_NEG: return -x
        if op == BC_ABS: return np.abs(x)
        if op == BC_RECIP: return 1.0 / x
        if op == BC_SQRT: return np.sqrt(x)
        if op == BC_STEP: return np.where(x >= 0.0, 1.0, 0.0)
        if op == BC_SIN: return _sin(x)
        if op == BC_EXP: return _exp(x)
        if op == BC_LN: return _log(x)
        if op == BC_TEX: return tex_fetch(textures[dst >> 2], dst & 3, x, y)
        raise ValueError(f"bad opcode {op}")

    with np.errstate(all="ignore"):
        for w in code:
            is_scalar, op, ka, kb, store, dst, a, b = bc_decode(w)
            if op == BC_END:
                break
            if is_scalar:
                assert row_uniform
                x = np.array([sacc if ka == K_T else scal[a]])
                y = np.array([sacc if kb == K_T else scal[b]]) if (BC_ADD <= op <= BC_MIN or op == BC_TEX) else x
                sacc = float(apply(op, x, y, dst)[0])
                if store:
                    assert op != BC_TEX, "TEX keeps its texture id in the dst field and must not store"
                    assert dst >= nk and dst not in scal, "row-uniform slots are never recycled"
                    scal[dst] = sacc
                continue
            if op >= 100:                         # the accumulator operand is negated first
                op -= 100
                x = -acc if ka == K_A else wide_operand(ka, a)
                y = -acc if kb == K_A else wide_operand(kb, b)
                acc = apply(op, x, y, dst)
                if store:
                    wide[dst] = acc
                continue
            x = wide_operand(ka, a)
            if BC_OUT_R <= op <= BC_OUT_B:
                out[op - BC_OUT_R] = x
                assert not store
                continue
            y = wide_operand(kb, b) if (BC_ADD <= op <= BC_MIN or op == BC_TEX) else x
            acc = apply(op, x, y, dst)
            if store:
                assert op != BC_TEX, "TEX keeps its texture id in the dst field and must not store"
                wide[dst] = acc
    return out


def bits_equal(a, b):
    """Bit-identical float64 arrays, any NaN matching any NaN."""
    a = np.ascontiguousarray(a, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    return (a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b))


def sign_rewrite_scene(w):
    """Steps whose operand is only asked for its sign: step(sin(u)) over zero, tiny, ordinary, huge (beyond the fast
    range), infinite and NaN arguments; step(v + c) with v = +-inf, NaN, -0 and values equal to -c; and the same
    operands with a second reader, which must NOT be rewritten."""
    from maray_b200 import expr as E
    X, Y = E.x(), E.y()
    rat = lambda p, q: E.div(E.nat(p), E.nat(q))
    inf = E.recip(E.sub(X, E.nat(3)))                       # +-inf at x = 3 ... finite elsewhere
    nan = E.mul(inf, E.sub(X, E.nat(3)))                    # NaN at x = 3 (inf * 0)
    u_small = E.mul(E.sub(X, E.nat(8)), rat(1, 7))          # crosses zero at x = 8 (+0 there)
    u_neg0 = E.mul(E.neg(E.sub(X, E.nat(8))), E.nat(0))     # -0 / +0
    u_big = E.mul(E.mul(X, X), E.mul(X, E.nat(4000000)))    # up to ~1e11: out of the fast range
    s1 = E.step(E.sin(E.mul(u_small, E.add(Y, E.nat(1)))))
    s2 = E.step(E.sin(u_neg0))
    s3 = E.step(E.sin(u_big))
    s4 = E.step(E.sin(E.add(inf, nan)))
    sv = E.sin(E.mul(X, rat(5, 3)))
    s5 = E.add(E.step(sv), sv)                              # the sine has a second reader
    c1 = E.step(E.add(E.mul(X, rat(1, 4)), E.neg(E.nat(2))))            # zero sum at x = 8
    c2 = E.step(E.add(E.nat(5), inf))
    c3 = E.step(E.add(nan, rat(1, 3)))
    c4 = E.step(E.add(u_neg0, E.nat(0)))
    sm = E.add(E.mul(X, rat(1, 8)), E.neg(E.nat(1)))
    c5 = E.mul(E.step(sm), sm)                              # the sum has a second reader
    r = E.add(E.add(E.add(s1, E.mul(s2, E.nat(2))), E.add(E.mul(s3, E.nat(4)), E.mul(s4, E.nat(8)))), E.mul(s5, E.nat(16)))
    g = E.add(E.add(E.add(c1, E.mul(c2, E.nat(2))), E.add(E.mul(c3, E.nat(4)), E.mul(c4, E.nat(8)))), E.mul(c5, E.nat(16)))
    return E.to_bytes([w, 4], [r, g, E.add(r, g)])


