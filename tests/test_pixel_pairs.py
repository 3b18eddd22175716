"""Pixel pairs (codegen.cpp, DESIGN.md 3.1): a straight-line kernel with guarded regions evaluates two pixels per thread.
A block of B threads covers the 2B launch pixels from blockIdx.x * 2B; thread t evaluates pixels t and B + t of them,
every statement once for each, and one warp vote on `guard || guard_b` covers both.

On the host the paired text runs under two drivers: the suite's own (tests/helpers.py: 256 threads, a grid sized for one
pixel per thread, so the blocks past the frame must store nothing) and the library's grid for pairs, ceil(n / 2B) blocks
of B threads.  Both must give the oracle's bits, in both host vote modes; so must s = 2 supersampling through the paired
store.  Other programs generate the same text as without pairs."""
import ctypes
import hashlib
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from maray_b200 import CudaRenderer, scenes
from oracle.oracle import OracleScene

from helpers import HOST_SHIM, bits_equal, host_jit_run
from test_guard_regions import ALWAYS, VOTE, _edge_scene, _modules, _source
from test_supersample import offsets, oracle_box_window

# The library's launch for pixel pairs, restated: ceil(n / 2B) blocks of B threads.  Threads run one after the other,
# each block twice (the second sweep sees a complete staging tile, as after __syncthreads; see tests/helpers.py
# HOST_DRIVER); the block's accumulator words are put back before the second sweep so that each pass adds its samples once.
PAIR_DRIVER = r"""
extern "C" void host_run_pairs(unsigned char* out, double* f64_out, unsigned long long plane, unsigned int p0,
                               unsigned int n, unsigned int W, unsigned int threads, double ox, double oy,
                               unsigned short* acc, unsigned int pass, unsigned int count) {
    MrParams p;
    p.out = out; p.f64_out = f64_out; p.f64_plane = plane; p.tex = nullptr; p.p0 = p0; p.n = n; p.W = W;
    p.out_aligned = 0;
    MrSampling sp;
    sp.ox = ox; sp.oy = oy; sp.acc = acc; sp.pass = pass; sp.count = count;
    blockDim.x = threads; blockDim.y = blockDim.z = 1;
    static unsigned short saved[3 * 2048];
    const unsigned int span = 2 * threads, blocks = (n + span - 1) / span;
    for (unsigned int b = 0; b < blocks; b++) {
        blockIdx.x = b;
        const unsigned int first = b * span, cnt = (n - first < span) ? n - first : span;
        if (acc) std::memcpy(saved, acc + 3 * (size_t)first, 6 * cnt);
        for (int sweep = 0; sweep < 2; sweep++) {
            if (acc) std::memcpy(acc + 3 * (size_t)first, saved, 6 * cnt);
            for (unsigned int t = 0; t < threads; t++) { threadIdx.x = t; maray_jit(p, sp); }
        }
    }
}
"""

_SO = {}


def _pair_lib(source):
    key = hashlib.sha256(source.encode()).hexdigest()
    lib = _SO.get(key)
    if lib is None:
        d = tempfile.mkdtemp(prefix="maray_pairs_")
        src = os.path.join(d, "k.cpp")
        with open(src, "w") as f:
            f.write(HOST_SHIM)
            f.write(source.replace('extern "C" __global__', "static"))
            f.write(PAIR_DRIVER)
        so = os.path.join(d, "k.so")
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-w",
                               "-o", so, src])
        lib = ctypes.CDLL(so)
        lib.host_run_pairs.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_ulonglong, ctypes.c_uint32,
                                       ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_double, ctypes.c_double,
                                       ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32]
        _SO[key] = lib
    return lib


def pair_run(source, w, p0, n, threads, ox=0.0, oy=0.0, acc=None, pass_=0, count=1):
    """One pass of the paired kernel over pixels p0 .. p0+n-1 on the library's grid.  Returns (rgb (n,3), planes (3,n))."""
    rgb = np.zeros((n, 3), dtype=np.uint8)
    planes = np.zeros((3, n), dtype=np.float64)
    acc_p = acc.ctypes.data if acc is not None else None
    _pair_lib(source).host_run_pairs(rgb.ctypes.data, planes.ctypes.data, n, p0, n, w, threads, ox, oy, acc_p, pass_, count)
    return rgb, planes


def _oracle_range(oracle, w, p0, n):
    """The oracle's RGB8 and f64 planes of the linear pixel range p0 .. p0+n-1, row piece by row piece."""
    rgbs, planes = [], []
    p, end = p0, p0 + n
    while p < end:
        y, x0 = divmod(p, w)
        x1 = min(w, x0 + end - p)
        rgb, f64 = oracle.render_window(x0, x1, y, y + 1, want_f64=True)
        rgbs.append(rgb.reshape(-1, 3))
        planes.append(f64.reshape(3, -1))
        p += x1 - x0
    return np.concatenate(rgbs), np.concatenate(planes, axis=1)


def _kernel(src):
    return src[src.index('extern "C" __global__'):]


# ---- which programs are paired --------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["chess_1k", "chess_4k"])
def test_chess_is_paired(monkeypatch, name):
    sc, _tex, _size = scenes.by_name(name)
    k = _kernel(_source(sc, monkeypatch))
    assert "const unsigned int j_b = j + blockDim.x;" in k and "mr_store_block_pair(p, stage," in k
    votes = re.findall(r"if \(mr_warp_any\((b\d+) \|\| (b\d+)_b\)\)", k)
    assert len(votes) == k.count(VOTE) == 128 and all(a == b for a, b in votes)     # one vote per region, both pixels
    monkeypatch.setenv("MARAY_JIT_PAIRS", "0")
    single = _kernel(_source(sc, monkeypatch))
    assert "j_b" not in single and "_pair(" not in single and single.count(VOTE) == 128
    # every statement of the single-pixel kernel is in the paired one, and once more for the second pixel
    decl = re.compile(r"^  (?:const )?(?:bool|double) ([bv]\d+)(_b)? = ", re.M)
    assert sorted(m[0] for m in decl.findall(k) if not m[1]) == sorted(m[0] for m in decl.findall(k) if m[1]) \
        == sorted(m[0] for m in decl.findall(single))


@pytest.mark.parametrize("name", ["sdf", "textured", "deep"])
def test_other_workloads_generate_the_same_text(monkeypatch, name):
    sc, tex, _size = scenes.by_name(name)
    paired = _modules(sc, monkeypatch, tex)
    monkeypatch.setenv("MARAY_JIT_PAIRS", "0")
    assert _modules(sc, monkeypatch, tex) == paired
    for unit in paired:
        assert "_pair(" not in _kernel(unit) and "j_b" not in _kernel(unit)


# ---- the host text against the oracle -------------------------------------------------------------------------------
# (p0, n) on the 1024-wide chess frame: whole rows; an odd piece of one row, not a multiple of 2B; a range that starts
# mid-block, mid-warp and crosses a row
RANGES = [(512 * 1024, 2048), (600 * 1024 + 300, 701), (700 * 1024 + 1000, 1024 + 77)]


def test_chess_ranges_in_both_host_modes_and_grids(monkeypatch, chess_bytes):
    src = _source(chess_bytes, monkeypatch)
    oracle = OracleScene(chess_bytes)
    for p0, n in RANGES:
        want_rgb, want = _oracle_range(oracle, 1024, p0, n)
        for text in (src, ALWAYS + src):
            runs = [host_jit_run(text, 1024, p0, n)] + [pair_run(text, 1024, p0, n, threads) for threads in (64, 640)]
            for rgb, planes in runs:
                assert bits_equal(planes, want).all(), (p0, n, text is src)
                assert np.array_equal(rgb, want_rgb), (p0, n, text is src)


def test_edge_cases_on_the_pair_grid(monkeypatch):
    w, h = 40, 8
    sc = _edge_scene(w, h)
    src = _source(sc, monkeypatch)
    assert "mr_store_block_pair(p, stage," in src
    want_rgb, want = _oracle_range(OracleScene(sc), w, 0, w * h)
    for text in (src, ALWAYS + src):
        for threads in (32, 96):                              # 2B = 64 (five blocks, the last partial), 192 (two)
            rgb, planes = pair_run(text, w, 0, w * h, threads)
            assert bits_equal(planes, want).all(), (threads, text is src)
            assert np.array_equal(rgb, want_rgb), (threads, text is src)


def test_supersampling_through_the_paired_store(monkeypatch, chess_bytes):
    """s = 2: four passes accumulate and the last resolves, for both pixels of every pair, on a range whose blocks are
    full, partial and (under the suite's grid) empty."""
    src = _source(chess_bytes, monkeypatch)
    x0, x1, y = 101, 1000, 512                                  # across the top edge of the trapezoid
    n, s = x1 - x0, 2
    o = offsets(s)
    for threads in (64, 256):
        acc = np.full(3 * n, 0xABCD, dtype=np.uint16)          # pass 0 must overwrite, not add
        for j in range(s):
            for i in range(s):
                rgb, _ = pair_run(src, 1024, y * 1024 + x0, n, threads, o[i], o[j], acc, j * s + i, s * s)
                if j * s + i + 1 < s * s:
                    assert not rgb.any(), "a pass before the last stored pixels"
        want = oracle_box_window(chess_bytes, s, (x0, x1, y, y + 1)).reshape(n, 3)
        assert np.array_equal(rgb, want), (threads, int((rgb != want).any(axis=1).sum()))
        assert len(np.unique(want)) > 2


# ---- on the GPU -----------------------------------------------------------------------------------------------------
def _renderer(scene, backend="nvrtc", gpus=1):
    r = CudaRenderer(gpus=gpus)
    r.load(scene)
    r.compile(backend)
    return r


@pytest.mark.gpu
def test_chess_4k_stats_and_frame_equal_the_single_pixel_kernel(monkeypatch):
    import torch
    sc = scenes.chess_4k()
    with _renderer(sc) as r:
        st = r.stats()
        got = r.render(3840, 2160)
    assert st["jit_block"] == 640 and st["jit_pixels_per_thread"] == 2
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert st["jit_round_pixels"] == sms * 640 * 2                 # 148 * 640 * 2 on a B200
    monkeypatch.setenv("MARAY_JIT_PAIRS", "0")
    with _renderer(sc) as r:
        assert r.stats()["jit_pixels_per_thread"] == 1
        assert np.array_equal(r.render(3840, 2160), got)


@pytest.mark.gpu
def test_render_paths_agree():
    """render, render_into, render_device, render_band (a band starting mid-block) and, with two GPUs, in-process bands:
    the same bytes, and those of the interpreter."""
    import torch
    w, h = 1001, 1024
    sc = scenes.chess_1k()
    with _renderer(sc, "interp") as r:
        want = r.render(w, h)
    with _renderer(sc) as r:
        assert r.stats()["jit_pixels_per_thread"] == 2
        assert np.array_equal(r.render(w, h), want)
        img = np.zeros((h, w, 3), dtype=np.uint8)
        r.render_into(img)
        assert np.array_equal(img, want)
        dev = np.zeros((h, w, 3), dtype=np.uint8)
        r.copy_to_host(r.render_device(w, h), dev)
        assert np.array_equal(dev, want)
        y0, y1 = 301, 517
        band = torch.zeros((y1 - y0) * w * 3, dtype=torch.uint8, device="cuda")
        r.render_band(w, h, y0, y1, band.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert np.array_equal(band.cpu().numpy().reshape(y1 - y0, w, 3), want[y0:y1])
        r.set_samples(2)
        ss = r.render(w, h)
    with _renderer(sc, "interp") as r:
        r.set_samples(2)
        assert np.array_equal(ss, r.render(w, h))
    if torch.cuda.device_count() >= 2:
        with _renderer(sc, gpus=2) as r2:
            assert np.array_equal(r2.render(w, h), want)
            dev2 = np.zeros((h, w, 3), dtype=np.uint8)
            r2.copy_to_host(r2.render_device(w, h), dev2)
            assert np.array_equal(dev2, want)
