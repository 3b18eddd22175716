"""Supersampled anti-aliasing (maray_cuda_set_samples): s x s samples per pixel, box-filtered to RGB8.

Sample (i, j) of pixel (x, y) is the scene at (x + o_i, y + o_j), o_k = (2k + 1 - s) * (1 / (2s)); the pixel is
(sum of the s*s u8 samples + s*s/2) // (s*s) per channel.  So sample (i, j) is pixel (x, y) of the reference's frame of
the scene with x -> x + K_i, y -> y + K_j substituted everywhere, and every supersampled frame is pinned to the oracle
(or to s = 1 frames of the substituted scenes) bit for bit."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import pytest

from maray_b200 import CudaRenderer, MarayCudaError, scenes
from maray_b200 import _lib
from maray_b200 import expr as E
from oracle.oracle import OracleScene

from helpers import HOST_SHIM

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- the definition, restated ---------------------------------------------------------------------------------
def offsets(s):
    return [float(2 * k + 1 - s) * (1.0 / (2.0 * s)) for k in range(s)]


def offset_expr(k, s):
    """K_k: an expression whose host constant folding gives exactly the bits of offsets(s)[k]."""
    c = 2 * k + 1 - s
    if c == 0:
        return E.nat(0)
    if c > 0:
        return E.mul(E.nat(c), E.recip(E.nat(2 * s)))
    return E.neg(E.mul(E.nat(-c), E.recip(E.nat(2 * s))))


def shifted_scene(scene, i, j, s):
    """The scene with x -> x + K_i, y -> y + K_j everywhere (Let definitions included)."""
    size, color, _legacy = E.from_bytes(scene)
    return E.to_bytes(size, E.map_xy(color, E.add(E.x(), offset_expr(i, s)), E.add(E.y(), offset_expr(j, s))))


def box_mean(samples, s):
    """samples: the s*s u8 frames; the rounded integer mean per channel."""
    total = np.zeros(samples[0].shape, dtype=np.uint32)
    for f in samples:
        total += f
    n = s * s
    return ((total + n // 2) // n).astype(np.uint8)


def oracle_box_window(scene, s, window, textures=()):
    x0, x1, y0, y1 = window
    return box_mean([OracleScene(shifted_scene(scene, i, j, s), list(textures)).render_window(x0, x1, y0, y1)
                     for j in range(s) for i in range(s)], s)


def test_offsets_are_the_grid_centres():
    for s in range(1, 17):
        o = offsets(s)
        assert o == sorted(o) and o == [-v for v in reversed(o)] and all(-0.5 < v < 0.5 for v in o)
    assert offsets(1) == [0.0] and offsets(3)[1] == 0.0 and offsets(2) == [-0.25, 0.25]


# ---- C ABI on a handle without a GPU ------------------------------------------------------------------------------
def test_set_samples_range_on_host_only_handle():
    scene = scenes.sdf(64, 48, 6, seed=4)
    with CudaRenderer(gpus=0) as r:
        r.load(scene)
        r.compile("nvrtc")
        src, st = r.source(), r.stats()
        for s in range(1, 17):
            r.set_samples(s)
        for bad in (0, 17, 1000):
            with pytest.raises(MarayCudaError) as ei:
                r.set_samples(bad)
            assert ei.value.code == _lib.E_INVALID and "1..16" in ei.value.message
        # nothing was recompiled, and the kernels do not depend on s
        assert r.source() == src and r.stats()["nvrtc_ms"] == st["nvrtc_ms"]
        r.compile("nvrtc")
        assert r.source() == src


# ---- the generated kernels, compiled for the host -------------------------------------------------------------------
# A driver of this file's own: it passes the sampling argument the library passes on the GPU.  Threads run one after
# the other, each block twice (the second sweep sees a complete staging tile, as after __syncthreads; see
# tests/helpers.py HOST_DRIVER); the block's accumulator words are put back before the second sweep so that each
# pass adds its samples once.
_SS_DRIVER = r"""
extern "C" void host_run_ss(unsigned char* out, const MrTexture* tex, unsigned int p0, unsigned int n, unsigned int W,
                            double ox, double oy, unsigned short* acc, unsigned int pass, unsigned int count
                            MR_CHAIN_ARGS) {
    MrParams p;
    p.out = out; p.f64_out = nullptr; p.f64_plane = 0; p.tex = tex; p.p0 = p0; p.n = n; p.W = W;
    p.out_aligned = 0;
    MrSampling sp;
    sp.ox = ox; sp.oy = oy; sp.acc = acc; sp.pass = pass; sp.count = count;
    blockDim.x = 256; blockDim.y = blockDim.z = 1;
    static unsigned short saved[3 * 256];
    unsigned int blocks = (n + 255) / 256;
    for (unsigned int b = 0; b < blocks; b++) {
        blockIdx.x = b;
        const unsigned int first = b * 256, cnt = (n - first < 256) ? n - first : 256;
        if (acc) std::memcpy(saved, acc + 3 * (size_t)first, 6 * cnt);
        for (int sweep = 0; sweep < 2; sweep++) {
            if (acc) std::memcpy(acc + 3 * (size_t)first, saved, 6 * cnt);
            for (unsigned int t = 0; t < 256; t++) { threadIdx.x = t; maray_jit(p MR_CHAIN_CALL, sp); }
        }
    }
}
"""

_SO = {}


def _host_module(source, chain):
    key = hashlib.sha256(source.encode()).hexdigest() + ("c" if chain else "s")
    lib = _SO.get(key)
    if lib is None:
        d = tempfile.mkdtemp(prefix="maray_ss_")
        src = os.path.join(d, "k.cpp")
        with open(src, "w") as f:
            f.write(HOST_SHIM)
            f.write(source.replace('extern "C" __global__', "static"))
            if chain:
                f.write("#define MR_CHAIN_ARGS , double* F, unsigned long long FS\n#define MR_CHAIN_CALL , F, FS\n")
            else:
                f.write("#define MR_CHAIN_ARGS\n#define MR_CHAIN_CALL\n")
            f.write(_SS_DRIVER)
        so = os.path.join(d, "k.so")
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-w",
                               "-o", so, src])
        lib = ctypes.CDLL(so)
        args = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_double,
                ctypes.c_double, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32]
        lib.host_run_ss.argtypes = args + ([ctypes.c_void_p, ctypes.c_ulonglong] if chain else [])
        _SO[key] = lib
    return lib


def host_pass(modules, frame_slots, w, p0, n, ox, oy, acc=None, pass_=0, count=1):
    """One pass of the generated kernel(s) over pixels p0 .. p0+n-1 on the CPU; returns the RGB8 output (n, 3)."""
    rgb = np.zeros((n, 3), dtype=np.uint8)
    tab = (ctypes.c_void_p * 2)()
    chain = len(modules) > 1
    fs = ((n + 255) // 256) * 256
    frame = np.full(max(1, frame_slots) * fs, np.nan, dtype=np.float64)
    acc_p = acc.ctypes.data if acc is not None else None
    for m in modules:
        extra = [frame.ctypes.data, fs] if chain else []
        _host_module(m, chain).host_run_ss(rgb.ctypes.data, ctypes.addressof(tab), p0, n, w, ox, oy, acc_p, pass_, count, *extra)
    return rgb


def _generated(scene, chain_env, monkeypatch):
    if chain_env:
        monkeypatch.setenv("MARAY_JIT_SEGMENT_VALUES", str(chain_env))
        monkeypatch.setenv("MARAY_JIT_CHAIN_SEGMENT_VALUES", str(chain_env))
    with CudaRenderer(gpus=0) as r:
        r.load(scene)
        st = r.compile("nvrtc")
        modules = r.modules()
    assert (len(modules) > 1) == bool(chain_env)
    return modules, st["jit_frame_slots"]


@pytest.mark.parametrize("form", ["single", "chain"])
@pytest.mark.parametrize("which", ["sdf", "chess"])
def test_generated_passes_match_the_oracle(monkeypatch, chess_bytes, which, form):
    if which == "sdf":
        scene, w, window = scenes.sdf(320, 200, 40, seed=2), 320, (0, 320, 57, 59)          # two whole rows
        chain_env = 256
    else:
        scene, w, window = chess_bytes, 1024, (384, 640, 512, 513)                          # across the top edge
        chain_env = 1500
    modules, slots = _generated(scene, chain_env if form == "chain" else 0, monkeypatch)
    x0, x1, y0, y1 = window
    assert y1 - y0 == 1 or (x0, x1) == (0, w)                      # a linear pixel range
    p0, n = y0 * w + x0, (y1 - y0) * (x1 - x0)
    # one pass at an offset (no accumulator): the oracle's frame of the substituted scene
    o = offsets(3)
    got = host_pass(modules, slots, w, p0, n, o[0], o[2])
    want = OracleScene(shifted_scene(scene, 0, 2, 3)).render_window(x0, x1, y0, y1).reshape(n, 3)
    assert np.array_equal(got, want)
    # s*s passes with accumulation and resolve: the box mean of the oracle's frames
    for s in (2, 3):
        o = offsets(s)
        acc = np.full(3 * n, 0xABCD, dtype=np.uint16)            # pass 0 must overwrite, not add
        out = None
        for j in range(s):
            for i in range(s):
                rgb = host_pass(modules, slots, w, p0, n, o[i], o[j], acc, j * s + i, s * s)
                if j * s + i + 1 < s * s:
                    assert not rgb.any(), "a pass before the last stored pixels"
                out = rgb
        want = oracle_box_window(scene, s, window).reshape(n, 3)
        assert np.array_equal(out, want), (s, int((out != want).any(axis=1).sum()))
        assert len(np.unique(want)) > 2                       # the edge pixels really are mixed


# ---- on the GPU -----------------------------------------------------------------------------------------------------
def _renderer(scene, backend, textures=(), gpus=1, libm=None):
    r = CudaRenderer(gpus=gpus)
    r.set_textures(list(textures))
    r.load(scene)
    r.compile(backend, libm=libm)
    return r


_FRAME_REF = {}


def _frame_reference(scene, s, w, h):
    """Box mean of the s*s full s = 1 frames of the substituted scenes, rendered by the interpreter (cheap compiles)."""
    key = (hashlib.sha256(scene).hexdigest(), s, w, h)
    if key not in _FRAME_REF:
        frames = []
        for j in range(s):
            for i in range(s):
                with _renderer(shifted_scene(scene, i, j, s), "interp") as r:
                    frames.append(r.render(w, h))
        _FRAME_REF[key] = box_mean(frames, s)
    return _FRAME_REF[key]


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["nvrtc", "interp"])
@pytest.mark.parametrize("s", [2, 3, 4])
def test_sdf_full_frame_is_the_box_mean(backend, s):
    w, h = 1920, 1080
    scene = scenes.sdf(w, h)
    want = _frame_reference(scene, s, w, h)
    with _renderer(scene, backend) as r:
        r.set_samples(s)
        got = r.render(w, h)
        one = r.render(w, h)
    assert np.array_equal(got, want) and np.array_equal(one, want)      # the accumulator is reset by pass 0
    # the anti-aliased frame differs from the one-sample frame only near edges
    with _renderer(scene, backend) as r:
        plain = r.render(w, h)
    changed = (got != plain).any(axis=2).mean()
    assert 0.0 < changed < 0.5


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["nvrtc", "interp"])
def test_chess_exact_libm_windows_against_oracle(backend):
    scene = scenes.chess_1k()
    with _renderer(scene, backend, libm="glibc") as r:
        r.set_samples(4)
        frame = r.render(1024, 1024)
    for window in ((384, 640, 500, 532), (0, 1024, 800, 804)):
        x0, x1, y0, y1 = window
        want = oracle_box_window(scene, 4, window)
        assert np.array_equal(frame[y0:y1, x0:x1], want), window


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["nvrtc", "interp"])
def test_textured_scene_against_oracle(backend):
    tex = scenes.synthetic_textures(4, 64)
    scene = scenes.textured(256, 128)
    with _renderer(scene, backend, tex) as r:
        r.set_samples(2)
        frame = r.render(256, 128)
    for window in ((0, 256, 0, 8), (100, 180, 60, 128)):
        x0, x1, y0, y1 = window
        assert np.array_equal(frame[y0:y1, x0:x1], oracle_box_window(scene, 2, window, tex)), window


@pytest.mark.gpu
def test_chain_form_matches_the_interpreter(monkeypatch):
    w, h = 512, 256
    scene = scenes.deep(w, h, n_values=9000, seed=3)
    with _renderer(scene, "interp") as r:
        r.set_samples(2)
        want = r.render(w, h)
    monkeypatch.setenv("MARAY_JIT_SEGMENT_VALUES", "3000")            # cut into a chain of kernels
    monkeypatch.setenv("MARAY_JIT_CHAIN_SEGMENT_VALUES", "3000")
    with _renderer(scene, "nvrtc") as r:
        assert r.stats()["jit_units"] >= 3
        r.set_samples(2)
        got = r.render(w, h)
    assert np.array_equal(got, want)


@pytest.mark.gpu
def test_auto_backend_cold_first_frame(monkeypatch, tmp_path):
    import time
    scene = scenes.chess_1k()
    with _renderer(scene, "nvrtc") as r:
        r.set_samples(2)
        want = r.render(1024, 1024)
    monkeypatch.setenv("MARAY_JIT_CACHE", str(tmp_path))
    with CudaRenderer(gpus=1) as r:
        r.load(scene)
        r.compile("auto")
        r.set_samples(2)
        first = r.render(1024, 1024)
        assert r.stats()["tier_rows_interp"] > 0
        assert np.array_equal(first, want)
        deadline = time.perf_counter() + 120
        while not r.stats()["jit_active"] and time.perf_counter() < deadline:
            time.sleep(0.2)
            assert np.array_equal(r.render(1024, 1024), want)
        assert r.stats()["jit_active"] == 1
        assert np.array_equal(r.render(1024, 1024), want)


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["nvrtc", "interp"])
def test_render_paths_agree(backend):
    import torch
    w, h = 1920, 1080                        # 6 MB: render_into takes the pipelined host path
    scene = scenes.sdf(w, h, 24, seed=7)
    with _renderer(scene, backend) as r:
        r.set_samples(2)
        img = np.zeros((h, w, 3), dtype=np.uint8)
        r.render_into(img)
        dev = np.zeros((h, w, 3), dtype=np.uint8)
        r.copy_to_host(r.render_device(w, h), dev)
        y0, y1 = 301, 517
        band = torch.zeros((y1 - y0) * w * 3, dtype=torch.uint8, device="cuda")
        r.render_band(w, h, y0, y1, band.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        band = band.cpu().numpy().reshape(y1 - y0, w, 3)
    assert np.array_equal(img, dev)
    assert np.array_equal(band, img[y0:y1])
    assert np.array_equal(img, _frame_reference(scene, 2, w, h))
    if torch.cuda.device_count() >= 2:                              # in-process bands over two GPUs
        with _renderer(scene, backend, gpus=2) as r2:
            r2.set_samples(2)
            assert np.array_equal(r2.render(w, h), img)
            dev2 = np.zeros((h, w, 3), dtype=np.uint8)
            r2.copy_to_host(r2.render_device(w, h), dev2)
            assert np.array_equal(dev2, img)


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["nvrtc", "interp"])
def test_switching_back_to_one_sample(backend):
    scene = scenes.chess_1k()
    with _renderer(scene, backend) as fresh:
        want = fresh.render(1024, 1024)
    with _renderer(scene, backend) as r:
        r.set_samples(4)
        aa = r.render(1024, 1024)
        r.set_samples(1)
        assert np.array_equal(r.render(1024, 1024), want)
    assert not np.array_equal(aa, want)


@pytest.mark.gpu
def test_window_f64_refuses_supersampling():
    scene = scenes.sdf(64, 48, 6, seed=4)
    with _renderer(scene, "nvrtc") as r:
        r.set_samples(2)
        with pytest.raises(MarayCudaError) as ei:
            r.render_window_f64(64, 48, 0, 64, 0, 48)
        assert ei.value.code == _lib.E_INVALID and "one sample" in ei.value.message
        r.set_samples(1)
        r.render_window_f64(64, 48, 0, 64, 0, 48)


@pytest.mark.gpu
def test_cli_samples_flag(tmp_path):
    from PIL import Image
    scene = scenes.sdf(320, 200, 12, seed=3)
    path = tmp_path / "s.maray"
    path.write_bytes(scene)
    out = str(tmp_path / "o.png")
    cli = os.path.join(ROOT, "maray_b200", "maray_cuda")
    res = subprocess.run([cli, "-i", str(path), "-o", out, "-s", "4"], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    with _renderer(scene, "nvrtc") as r:
        r.set_samples(4)
        want = r.render(320, 200)
    assert np.array_equal(np.array(Image.open(out).convert("RGB")), want)
    bad = subprocess.run([cli, "-i", str(path), "-o", out, "-s", "17"], capture_output=True, text=True)
    assert bad.returncode == 2
