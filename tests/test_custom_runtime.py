"""Custom runtimes (maray_cuda_set_functions / maray_cuda_set_context, DESIGN.md 3.7): App(id, a, b) calls a
user-supplied `maray_app` over a context buffer, on every generated-kernel path.

The reference side is the oracle's interpreter (oracle/maray_oracle.c) with a custom runtime: this file builds a copy of
that C text in which `App` calls a C callback with maray_app's own signature, in the place where the oracle calls its
texture runtime (reference src/lib.rs:664-668: functions[id](&ctx, id, a, b); an id past n keeps the panic flag).  The
callback is the very user source, compiled by g++ with -ffp-contract=off behind the `__device__`-stripping shim of
tests/helpers.py after the library's device prelude.  Device and host then run the same arithmetic, and frames are
compared bit for bit.  On the host, the generated units run under this file's own
driver, which also sets the two context constants the units declare."""
import ctypes
import hashlib
import os
import struct
import subprocess
import tempfile

import numpy as np
import pytest

from maray_b200 import (CudaFunctions, CudaRenderer, MarayCudaError, RenderMethod, Runtime, Textures, _lib, gen_to_image,
                        scenes)
from maray_b200 import expr as E
from oracle.oracle import OracleScene

from helpers import HOST_SHIM, bits_equal
from test_supersample import box_mean, shifted_scene

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "maray_b200", "csrc")

# A context of two doubles, a small RGB image (w, h as u32 at byte 16, the bytes from byte 24), and five functions:
# 0 doubles from the context, 1 an RGB channel through mr_tex, 2 integer hashing of the argument bits, 3 glibc's exp and
# log (bit-exact in every libm mode), 4 sin (glibc's bits only in exact mode).
SRC = r"""
__device__ double maray_app(const unsigned char* ctx, unsigned long long ctx_bytes, unsigned int id, double a, double b) {
    const double* k = reinterpret_cast<const double*>(ctx);
    if (id == 0u) return a * k[0] + b * k[1];
    if (id == 1u) {
        const unsigned int w = *reinterpret_cast<const unsigned int*>(ctx + 16);
        const unsigned int h = *reinterpret_cast<const unsigned int*>(ctx + 20);
        return mr_tex(ctx + 24, w, h, 1u, a, b) + (double)(ctx_bytes & 1u);
    }
    if (id == 2u) {
        unsigned long long ua = (unsigned long long)__double_as_longlong(a);
        unsigned long long ub = (unsigned long long)__double_as_longlong(b);
        unsigned long long x = ua * 0x9E3779B97F4A7C15ull ^ (ub + 0x7F4A7C15ull);
        x ^= x >> 29;
        x *= 0xBF58476D1CE4E5B9ull;
        x ^= x >> 32;
        return (double)(x & 0xFFull);
    }
    if (id == 3u) return mr_exp(a * 0.01) + mr_log(b);
    return mr_sin(a) * b;
}
"""
N_FUNCTIONS = 5
# the host twin of the one intrinsic the user source uses that tests/helpers.py's shim lacks
EXTRA_SHIM = """
static inline long long __double_as_longlong(double d) { long long b; std::memcpy(&b, &d, 8); return b; }
"""


def make_ctx(k0=1.5, k1=-0.25, w=13, h=9, seed=3):
    img = np.random.default_rng(seed).integers(0, 256, size=(h, w, 3), dtype=np.uint8)
    return struct.pack("<ddII", k0, k1, w, h) + img.tobytes()


def app_scene(w=96, h=40, with_sin=False):
    """Every function of SRC, over ordinary, NaN, +-inf and -0 arguments."""
    X, Y = E.x(), E.y()
    A = lambda i, a, b: E.app(i, a, b)
    inf = E.recip(E.sub(X, E.nat(3)))                          # +-inf at x = 3
    nan = E.mul(inf, E.sub(X, E.nat(3)))                       # NaN at x = 3
    neg0 = E.neg(E.mul(X, E.nat(0)))                           # -0
    r = E.add(A(0, X, Y), A(1, E.sub(E.div(X, E.nat(4)), E.nat(2)), E.sub(E.div(Y, E.nat(3)), E.nat(1))))
    g = E.add(E.mul(A(2, X, Y), E.nat(1)), A(3, E.sub(X, E.nat(40)), E.add(Y, E.div(E.nat(1), E.nat(2)))))
    b = E.add(E.add(A(2, inf, nan), A(0, neg0, inf)), E.add(A(3, nan, neg0), A(2, neg0, E.nat(0))))
    b = E.add(b, A(1, nan, E.neg(inf)))
    if with_sin:
        r = E.add(r, A(4, E.mul(X, E.div(E.nat(7), E.nat(3))), E.add(Y, E.nat(10))))
    return E.to_bytes([w, h], [r, g, b])


def guarded_scene(w=96, h=40):
    """A boolean AND whose heavy body calls maray_app: a guarded region (pixel pairs follow)."""
    X, Y = E.x(), E.y()
    guard = E.range(E.nat(20), E.nat(60), X)
    body = E.step(E.sub(E.add(E.app(2, X, Y), E.app(0, E.mul(X, Y), Y)), E.nat(128)))
    inner = E.mul(guard, body)
    r = E.mul(inner, E.nat(255))
    g = E.add(E.mul(E.app(2, Y, X), E.nat(1)), r)
    return E.to_bytes([w, h], [r, g, E.app(0, X, E.nat(1))])


def long_scene(w=64, h=8, terms=90):
    """More than one chain segment's worth of values (with MARAY_JIT_SEGMENT_VALUES), every part calling maray_app."""
    X, Y = E.x(), E.y()
    acc = E.nat(0)
    for k in range(terms):
        acc = E.add(acc, E.mul(E.app(k % 4, E.add(X, E.nat(k)), E.add(Y, E.nat(2 * k + 1))), E.recip(E.nat(k + 3))))
    return E.to_bytes([w, h], [acc, E.mul(acc, E.nat(2)), E.app(2, acc, X)])


# ---- the g++-built callback of the oracle ------------------------------------------------------------------------
_LIBS = {}


def _gxx(text, prefix):
    d = tempfile.mkdtemp(prefix=prefix)
    src = os.path.join(d, "k.cpp")
    with open(src, "w") as f:
        f.write(text)
    so = os.path.join(d, "k.so")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-w",
                           "-I", CSRC, "-o", so, src])
    return ctypes.CDLL(so)


def host_app(source):
    """maray_app of `source` compiled for the host: the oracle's callback."""
    key = ("app", source)
    if key not in _LIBS:
        _LIBS[key] = _gxx(HOST_SHIM + EXTRA_SHIM + '#include "device_sem.cuh"\n' + source + r"""
extern "C" double host_app(const unsigned char* c, unsigned long long n, unsigned int id, double a, double b) {
    return maray_app(c, n, id, a, b);
}
""", "maray_app_")
    return _LIBS[key].host_app


# The oracle's interpreter with a custom runtime: the text of oracle/maray_oracle.c, edited at the anchors below (each
# must occur exactly once), built with the oracle's own flags (oracle/Makefile).
ORACLE_C = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "maray_oracle.c")
APP_FN = ctypes.CFUNCTYPE(ctypes.c_double, ctypes.c_void_p, ctypes.c_ulonglong, ctypes.c_uint32, ctypes.c_double,
                          ctypes.c_double)
_ORACLE_EDITS = [
    ("/* Cache: src/cache.rs:6-42",
     "typedef double (*mo_app_fn)(const unsigned char *, unsigned long long, uint32_t, double, double);\n"
     "static mo_app_fn g_app_fn; static uint32_t g_app_n; static unsigned char *g_app_ctx; static size_t g_app_bytes;\n"
     "/* Cache: src/cache.rs:6-42"),
    ("        return texture_fn(rt->tex, e->app_id, a, b);",
     "        return g_app_fn(g_app_ctx, g_app_bytes, (uint32_t)e->app_id, a, b);   /* functions[id](&ctx, id, a, b) */"),
    ("Rt rt = {&s->tex, s->tex.n * ALIGN, 0, NULL};", "Rt rt = {&s->tex, g_app_n, 0, NULL};"),
    ("/* Whole image of size w x h",
     "void mo_set_functions(mo_app_fn fn, uint32_t n, const void *ctx, size_t bytes) {\n"
     "    free(g_app_ctx); g_app_ctx = (unsigned char *)malloc(bytes ? bytes : 1); memcpy(g_app_ctx, ctx, bytes);\n"
     "    g_app_fn = fn; g_app_n = n; g_app_bytes = bytes;\n}\n"
     "/* Whole image of size w x h"),
]


def _custom_oracle_lib():
    if "oracle" not in _LIBS:
        text = open(ORACLE_C).read()
        for anchor, new in _ORACLE_EDITS:
            assert text.count(anchor) == 1, anchor
            text = text.replace(anchor, new)
        d = tempfile.mkdtemp(prefix="maray_oracle_app_")
        src, so = os.path.join(d, "o.c"), os.path.join(d, "o.so")
        with open(src, "w") as f:
            f.write(text)
        subprocess.check_call(["gcc", "-O2", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-w", "-pthread",
                               "-shared", "-o", so, src, "-lm", "-lpthread"])
        L = ctypes.CDLL(so)
        L.mo_open.restype = ctypes.c_void_p
        L.mo_open.argtypes = [ctypes.c_char_p, ctypes.c_size_t]
        L.mo_close.argtypes = [ctypes.c_void_p]
        L.mo_set_functions.argtypes = [APP_FN, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_size_t]
        L.mo_render_window.argtypes = [ctypes.c_void_p] + [ctypes.c_uint32] * 4 + [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
        _LIBS["oracle"] = L
    return _LIBS["oracle"]


class oracle:
    """The oracle's render_window (oracle/oracle.py) under the custom runtime (source, n, ctx).  The runtime is process
    state of the built copy, so it is set again by every render."""

    def __init__(self, scene, ctx, source=SRC, n=N_FUNCTIONS):
        self.scene, self.ctx, self.n = bytes(scene), bytes(ctx), n
        self.fn = ctypes.cast(host_app(source), APP_FN)

    def render_window(self, x0, x1, y0, y1, want_f64=False):
        L = _custom_oracle_lib()
        L.mo_set_functions(self.fn, self.n, self.ctx, len(self.ctx))
        h = L.mo_open(self.scene, len(self.scene))
        assert h, "oracle: not a .maray file"
        try:
            rgb = np.zeros((y1 - y0, x1 - x0, 3), dtype=np.uint8)
            planes = np.zeros((3, y1 - y0, x1 - x0), dtype=np.float64)
            rc = L.mo_render_window(h, x0, x1, y0, y1, os.cpu_count() or 1, rgb.ctypes.data, planes.ctypes.data)
            if rc == -1:
                raise IndexError("oracle: App id outside Runtime::functions (the reference panics here)")
            assert rc == 0, rc
        finally:
            L.mo_close(h)
        return (rgb, planes) if want_f64 else rgb


# ---- the generated units on the host ----------------------------------------------------------------------------
def _driver(unit):
    chain = "double* __restrict__ F" in unit
    set_ctx = "mr_app_ctx = ctx; mr_app_ctx_bytes = ctx_bytes;" if "mr_app_ctx" in unit else "(void)ctx; (void)ctx_bytes;"
    return r"""
extern "C" void host_run(unsigned char* out, double* f64_out, unsigned long long plane, unsigned int p0, unsigned int n,
                         unsigned int W, unsigned int threads, unsigned int grid_ppt, const unsigned char* ctx,
                         unsigned long long ctx_bytes, double* F, unsigned long long FS) {
    %s
    MrParams p;
    p.out = out; p.f64_out = f64_out; p.f64_plane = plane; p.tex = nullptr; p.p0 = p0; p.n = n; p.W = W;
    p.out_aligned = 0;
    blockDim.x = threads; blockDim.y = blockDim.z = 1;
    const unsigned int span = grid_ppt * threads, blocks = (n + span - 1) / span;
    for (unsigned int b = 0; b < blocks; b++) {
        blockIdx.x = b;
        for (int sweep = 0; sweep < 2; sweep++)   // the second sweep sees a complete staging tile (tests/helpers.py)
            for (unsigned int t = 0; t < threads; t++) { threadIdx.x = t; maray_jit(p%s); }
    }
}
""" % (set_ctx, ", F, FS" if chain else "")


def host_run(units, w, p0, n, ctx, threads=256, grid_ppt=1, frame_slots=0):
    """Runs the units (one, or a chain in order over one frame) for pixels p0 .. p0+n-1.  Returns (rgb (n,3), planes (3,n))."""
    rgb = np.zeros((n, 3), dtype=np.uint8)
    planes = np.zeros((3, n), dtype=np.float64)
    fs = ((n + threads - 1) // threads) * threads
    frame = np.full(max(1, frame_slots) * fs, np.nan, dtype=np.float64)
    cbuf = ctypes.create_string_buffer(ctx, len(ctx) + 8)
    for unit in units:
        key = ("unit", hashlib.sha256(unit.encode()).hexdigest())
        if key not in _LIBS:
            lib = _gxx(HOST_SHIM + EXTRA_SHIM + unit.replace('extern "C" __global__', "static") + _driver(unit), "maray_unit_")
            lib.host_run.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_ulonglong] + [ctypes.c_uint32] * 5 + \
                                    [ctypes.c_void_p, ctypes.c_ulonglong, ctypes.c_void_p, ctypes.c_ulonglong]
            _LIBS[key] = lib
        _LIBS[key].host_run(rgb.ctypes.data, planes.ctypes.data, n, p0, n, w, threads, grid_ppt, cbuf, len(ctx),
                            frame.ctypes.data, fs)
    return rgb, planes


def compile_units(scene, source=SRC, n=N_FUNCTIONS, backend="nvrtc", ctx=None):
    """(modules, stats) of the NVRTC back end on a host-only handle."""
    with CudaRenderer(gpus=0) as r:
        r.set_functions(source, n)
        if ctx is not None:
            r.set_context(ctx)
        r.load(scene)
        st = r.compile(backend)
        return r.modules(), st


def assert_matches_oracle(units, scene, ctx, window, **kw):
    x0, x1, y0, y1 = window
    w = E_size(scene)[0]
    assert x0 == 0 and x1 == w
    want_rgb, want_f64 = oracle(scene, ctx).render_window(x0, x1, y0, y1, want_f64=True)
    rgb, planes = host_run(units, w, y0 * w, (y1 - y0) * w, ctx, **kw)
    assert bits_equal(planes, want_f64.reshape(3, -1)).all()
    assert np.array_equal(rgb, want_rgb.reshape(-1, 3))


def E_size(scene):
    return OracleScene(scene).size


# ---- CPU: refusals and errors -----------------------------------------------------------------------------------
def test_app_id_past_n_functions_is_a_scene_error():
    scene = E.to_bytes([8, 8], [E.app(5, E.x(), E.y()), E.x(), E.y()])
    with CudaRenderer(gpus=0) as r:
        r.set_functions(SRC, N_FUNCTIONS)
        r.load(scene)
        with pytest.raises(MarayCudaError) as ei:
            r.compile("nvrtc")
        assert ei.value.code == _lib.E_SCENE and "custom runtime" in ei.value.message


def test_interpreter_refuses_a_custom_app():
    with CudaRenderer(gpus=0) as r:
        r.set_functions(SRC, N_FUNCTIONS)
        r.load(app_scene())
        with pytest.raises(MarayCudaError) as ei:
            r.compile("interp")
        assert ei.value.code == _lib.E_UNSUPPORTED and "interpreter" in ei.value.message


def test_syntax_error_in_the_user_source_is_a_compile_error_with_the_nvrtc_log(monkeypatch, tmp_path):
    monkeypatch.setenv("MARAY_JIT_CACHE", str(tmp_path))
    bad = SRC.replace("return mr_sin(a) * b;", "return mr_sin(a) * b +;")
    with CudaRenderer(gpus=0) as r:
        r.set_functions(bad, N_FUNCTIONS)
        r.load(app_scene())
        with pytest.raises(MarayCudaError) as ei:
            r.compile("nvrtc")
        assert ei.value.code == _lib.E_COMPILE
        assert "expected an expression" in ei.value.message


@pytest.mark.parametrize("back", ["set_textures", "set_functions_null"])
def test_texture_runtime_replaces_the_custom_one(back, monkeypatch):
    scene = E.to_bytes([8, 8], [E.app(2, E.x(), E.y()), E.x(), E.y()])
    with CudaRenderer(gpus=0) as r:
        r.set_functions(SRC, N_FUNCTIONS)
        r.set_context(make_ctx())
        r.load(scene)
        monkeypatch.setenv("MARAY_JIT_SOURCE_ONLY", "1")
        with pytest.raises(MarayCudaError) as ei:
            r.compile("nvrtc")
        assert ei.value.code == _lib.E_COMPILE     # source generated: the id was valid for the custom runtime
        monkeypatch.delenv("MARAY_JIT_SOURCE_ONLY")
        if back == "set_textures":
            r.set_textures([])
        else:
            r.set_functions(None)
        with pytest.raises(MarayCudaError) as ei:
            r.compile("nvrtc")
        assert ei.value.code == _lib.E_SCENE and "texture runtime" in ei.value.message


def test_runtime_from_parts_accepts_cuda_functions():
    rt = Runtime.from_parts(make_ctx(), CudaFunctions(SRC, N_FUNCTIONS))
    assert rt.functions.n == N_FUNCTIONS
    with pytest.raises(MarayCudaError) as ei:
        Runtime.from_parts(Textures([]), [lambda *a: 0.0])
    assert ei.value.code == _lib.E_UNSUPPORTED


# ---- CPU: generated text ----------------------------------------------------------------------------------------
def _source_only(scene, textures=(), custom=False, monkeypatch=None):
    monkeypatch.setenv("MARAY_JIT_SOURCE_ONLY", "1")
    with CudaRenderer(gpus=0) as r:
        if custom:
            r.set_functions(SRC, N_FUNCTIONS)
        else:
            r.set_textures(list(textures))
        r.load(scene)
        with pytest.raises(MarayCudaError):
            r.compile("nvrtc")
        return r.modules()


def test_user_source_once_in_every_unit_that_calls_it(monkeypatch):
    (unit,) = _source_only(app_scene(), custom=True, monkeypatch=monkeypatch)
    assert unit.count(SRC) == 1 and "maray_app(mr_app_ctx, mr_app_ctx_bytes, 4u, " not in unit
    monkeypatch.setenv("MARAY_JIT_SEGMENT_VALUES", "64")
    units = _source_only(long_scene(), custom=True, monkeypatch=monkeypatch)
    assert len(units) > 1
    for u in units:
        calls = "maray_app(mr_app_ctx" in u
        assert u.count(SRC) == (1 if calls else 0)
        assert ("__constant__ const unsigned char* mr_app_ctx;" in u) == calls


@pytest.mark.parametrize("name", ["chess_1k", "sdf", "textured", "deep"])
def test_texture_runtime_units_never_mention_the_custom_runtime(name, monkeypatch):
    if name == "deep":
        scene, textures = scenes.deep(w=256, h=64, n_values=3000), []
    else:
        scene, textures, _ = scenes.by_name(name)
    for u in _source_only(scene, textures, monkeypatch=monkeypatch):
        assert "maray_app" not in u and "mr_app_ctx" not in u


# ---- CPU: bit-exact on the host ---------------------------------------------------------------------------------
def test_functions_bit_exact_on_the_host():
    scene, ctx = app_scene(with_sin=True), make_ctx()
    (unit,), _ = compile_units(scene)
    assert_matches_oracle([unit], scene, ctx, (0, 96, 0, 40))


def test_odd_context_size_reaches_the_function():
    scene, ctx = app_scene(), make_ctx() + b"\x07"    # id 1 adds ctx_bytes & 1
    (unit,), _ = compile_units(scene)
    assert_matches_oracle([unit], scene, ctx, (0, 96, 0, 40))


@pytest.mark.parametrize("vote", ["lane", "always"])
def test_app_inside_a_guarded_region_on_both_grids(vote):
    scene, ctx = guarded_scene(), make_ctx()
    (unit,), st = compile_units(scene)
    assert "if (mr_warp_any(" in unit and st["jit_pixels_per_thread"] == 2
    if vote == "always":
        unit = "#define MR_HOST_GUARDS_ALWAYS 1\n" + unit
    assert_matches_oracle([unit], scene, ctx, (0, 96, 0, 40))                                   # the suite's grid
    assert_matches_oracle([unit], scene, ctx, (0, 96, 3, 17), threads=st["jit_block"], grid_ppt=2)   # the library's
    assert_matches_oracle([unit], scene, ctx, (0, 96, 5, 6), threads=32, grid_ppt=2)           # a ragged last block


def test_chain_form_bit_exact_on_the_host(monkeypatch):
    monkeypatch.setenv("MARAY_JIT_SEGMENT_VALUES", "64")
    scene, ctx = long_scene(), make_ctx()
    units, st = compile_units(scene)
    assert len(units) > 1 and st["jit_frame_slots"] > 0
    assert_matches_oracle(units, scene, ctx, (0, 64, 0, 8), frame_slots=st["jit_frame_slots"])


# ---- CPU: cubin cache -------------------------------------------------------------------------------------------
def test_cache_hits_on_the_same_source_and_misses_on_a_changed_one(monkeypatch, tmp_path):
    monkeypatch.setenv("MARAY_JIT_CACHE", str(tmp_path))
    scene = app_scene()
    _, st = compile_units(scene)
    assert st["jit_cache_hit"] == 0
    _, st = compile_units(scene)
    assert st["jit_cache_hit"] == 1
    _, st = compile_units(scene, source=SRC.replace("k[0]", "k[0] * 2.0"))
    assert st["jit_cache_hit"] == 0
    with CudaRenderer(gpus=0) as r:
        r.set_functions(SRC, N_FUNCTIONS)
        r.load(scene)
        before = r.compile("nvrtc")
        files = sorted(os.listdir(tmp_path))
        r.set_context(make_ctx(k0=7.0))
        assert r.stats() == {**before, "jit_active": r.stats()["jit_active"]}
        assert sorted(os.listdir(tmp_path)) == files


# ---- GPU ---------------------------------------------------------------------------------------------------------
def _gpu(scene, ctx, source=SRC, n=N_FUNCTIONS, backend="nvrtc", libm=None, **kw):
    r = CudaRenderer(**kw) if kw else CudaRenderer(device_ids=[0])
    r.set_functions(source, n)
    r.set_context(ctx)
    r.load(scene)
    r.compile(backend, libm=libm)
    return r


@pytest.mark.gpu
def test_gpu_frames_match_the_oracle():
    ctx = make_ctx()
    for (w, h) in [(1920, 1080), (1001, 37)]:
        scene = app_scene(w, h)
        want_rgb, want_f64 = oracle(scene, ctx).render_window(0, w, 0, h, want_f64=True)
        with _gpu(scene, ctx) as r:
            assert np.array_equal(r.render(w, h), want_rgb)
            planes, rgb = r.render_window_f64(w, h, 0, w, h // 3, h // 3 + 5)
            assert bits_equal(planes, want_f64[:, h // 3:h // 3 + 5]).all()
            if w == 1920:
                import torch
                frame = torch.zeros(h * w * 3, dtype=torch.uint8, device="cuda")
                for (y0, y1) in [(0, 333), (333, 334), (334, 701), (701, h)]:
                    r.render_band(w, h, y0, y1, frame.data_ptr() + y0 * w * 3, torch.cuda.current_stream().cuda_stream)
                torch.cuda.synchronize()
                assert np.array_equal(frame.cpu().numpy().reshape(h, w, 3), want_rgb)
                d = r.render_device(w, h)
                out = np.zeros((h, w, 3), dtype=np.uint8)
                r.copy_to_host(d, out)
                assert np.array_equal(out, want_rgb)


@pytest.mark.gpu
def test_gpu_exact_mode_sin_matches_the_oracle():
    w, h = 640, 200
    scene, ctx = app_scene(w, h, with_sin=True), make_ctx()
    want = oracle(scene, ctx).render_window(0, w, 0, h, want_f64=True)[1]
    with _gpu(scene, ctx, libm="glibc") as r:
        assert bits_equal(r.render_window_f64(w, h, 0, w, 0, h)[0], want).all()


@pytest.mark.gpu
def test_gpu_guarded_supersampled_and_chain_forms(monkeypatch):
    w, h = 1920, 1080
    ctx = make_ctx()
    scene = guarded_scene(w, h)
    with _gpu(scene, ctx) as r:
        assert r.stats()["jit_pixels_per_thread"] == 2
        assert np.array_equal(r.render(w, h), oracle(scene, ctx).render_window(0, w, 0, h))
        r.set_samples(2)
        want = box_mean([oracle(shifted_scene(scene, i, j, 2), ctx).render_window(0, w, 0, h)
                         for j in range(2) for i in range(2)], 2)
        assert np.array_equal(r.render(w, h), want)
    monkeypatch.setenv("MARAY_JIT_SEGMENT_VALUES", "64")
    scene = long_scene(w, 270)
    with _gpu(scene, ctx) as r:
        assert r.stats()["jit_units"] > 1
        assert np.array_equal(r.render(w, 270), oracle(scene, ctx).render_window(0, w, 0, 270))


@pytest.mark.gpu
def test_gpu_multi_gpu_bands():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs")
    w, h = 1920, 1080
    scene, ctx = app_scene(w, h), make_ctx()
    with _gpu(scene, ctx, device_ids=[0, 1]) as r:
        want = oracle(scene, ctx).render_window(0, w, 0, h)
        assert np.array_equal(r.render(w, h), want)
        d = r.render_device(w, h)
        out = np.zeros((h, w, 3), dtype=np.uint8)
        r.copy_to_host(d, out)
        assert np.array_equal(out, want)


@pytest.mark.gpu
def test_gpu_set_context_after_compile_recompiles_nothing():
    w, h = 800, 300
    scene = app_scene(w, h)
    ctx_a, ctx_b = make_ctx(), make_ctx(k0=-3.0, k1=0.125, w=5, h=21, seed=9)
    with _gpu(scene, ctx_a) as r:
        st = r.stats()
        assert np.array_equal(r.render(w, h), oracle(scene, ctx_a).render_window(0, w, 0, h))
        r.set_context(ctx_b)
        got = r.render(w, h)
        assert np.array_equal(got, oracle(scene, ctx_b).render_window(0, w, 0, h))
        assert not np.array_equal(got, oracle(scene, ctx_a).render_window(0, w, 0, h))
        st2 = r.stats()
        assert st2["nvrtc_ms"] == st["nvrtc_ms"] and st2["jit_units"] == st["jit_units"]
        assert st2["jit_cache_hit"] == st["jit_cache_hit"]


@pytest.mark.gpu
def test_gpu_auto_gives_the_nvrtc_bytes_cold_and_cached(monkeypatch, tmp_path):
    monkeypatch.setenv("MARAY_JIT_CACHE", str(tmp_path))
    w, h = 1024, 256
    scene, ctx = app_scene(w, h), make_ctx()
    with _gpu(scene, ctx, backend="nvrtc") as r:
        want = r.render(w, h)
    for hit in (0, 1):
        if hit == 0:
            for f in os.listdir(tmp_path):
                os.remove(os.path.join(tmp_path, f))
        with _gpu(scene, ctx, backend="auto") as r:
            st = r.stats()
            assert st["jit_active"] == 1 and st["jit_cache_hit"] == hit
            assert np.array_equal(r.render(w, h), want)


@pytest.mark.gpu
def test_gpu_restated_texture_runtime_is_byte_identical_at_4k():
    scene, textures, (w, h) = scenes.by_name("textured")
    with CudaRenderer(device_ids=[0]) as r:
        r.set_textures(textures)
        r.load(scene)
        r.compile("nvrtc")
        want = r.render(w, h)
    img = np.zeros((h, w, 3), dtype=np.uint8)
    rt = Runtime.from_parts(scenes.pack_textures(textures), CudaFunctions(scenes.TEXTURE_RUNTIME_SOURCE, 5 * len(textures)))
    gen_to_image(RenderMethod.Cuda(backend="nvrtc"), rt, scene, img)
    assert np.array_equal(img, want)
    assert want.std() > 1.0
