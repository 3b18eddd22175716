"""The exact mode of the device libm (csrc/device_libm_glibc.cuh, MARAY_LIBM_GLIBC): sin/exp/ln with the bits of the
host libm the reference calls (reference src/lib.rs:648-650, src/wasm.rs:11-13).

CPU: the header's host rendition against this host's glibc, bit for bit (tools/glibc_libm_check.c), and on any host
against glibc 2.39's results stored under tests/golden; the committed tables against the host library; the exact mode
compiles through NVRTC without a GPU.
GPU (`-m gpu`): f64 channel values of sin/exp/ln scenes and of the deep scene are BIT-IDENTICAL to the oracle's in
exact mode, with both back ends -- the class of scenes that is only "within 1 LSB" with the default libm."""
import os
import platform
import subprocess
import sys

import numpy as np
import pytest

from maray_b200 import CudaRenderer, scenes
from maray_b200 import expr as E

from conftest import ROOT
from helpers import bits_equal, sign_rewrite_scene

GLIBC = platform.libc_ver()
needs_glibc_239 = pytest.mark.skipif(GLIBC[0] != "glibc" or GLIBC[1] != "2.39" or platform.machine() != "x86_64",
                                     reason="the exact mode restates glibc 2.39's x86-64 FMA variants")


def _cpu_has_fma():
    try:
        flags = open("/proc/cpuinfo").read()
    except OSError:
        return False
    return " fma " in flags and " avx2 " in flags


@needs_glibc_239
@pytest.mark.skipif(not _cpu_has_fma(), reason="glibc selects its FMA variants only on AVX2+FMA hosts")
def test_exact_mode_returns_the_host_libms_bits(tmp_path):
    """Exact mode: sin, exp, log and the sign of the sine.  Default mode (-DFAST_MODE): exp and log are the same routines
    (only the sine differs), and the sign of the sine equals glibc's there too."""
    for flags in ([], ["-DFAST_MODE"]):
        exe = tmp_path / ("glibc_libm_check" + "_fast" * bool(flags))
        subprocess.check_call(["gcc", "-O2", "-mfma", "-ffp-contract=off", "-fno-builtin-sin", "-fno-builtin-exp",
                               "-fno-builtin-log", *flags, "-o", str(exe), os.path.join(ROOT, "tools", "glibc_libm_check.c"), "-lm"])
        out = subprocess.run([str(exe), "2000000"], capture_output=True, text=True)
        assert "total differing: 0" in out.stdout and out.returncode == 0, out.stdout[-3000:]
        assert out.stdout.count(" 0 differ") >= 25          # every (function, range) line


LIBM_DRIVER = r"""
#define MR_LIBM_HOST 1
#ifndef FAST_MODE
#define MR_LIBM_GLIBC 1
#endif
#include "device_libm.cuh"
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
/* argv: function (sin, exp, log, sgn), n, input file of n doubles, output file */
int main(int argc, char** argv) {
    if (argc != 5) return 2;
    const long n = atol(argv[2]);
    double* x = malloc(n * sizeof *x);
    FILE* f = fopen(argv[3], "rb");
    if (!f || fread(x, sizeof *x, n, f) != (size_t)n) return 3;
    fclose(f);
    for (long i = 0; i < n; i++) {
        if (!strcmp(argv[1], "sin")) x[i] = mr_sin_g(x[i]);
        else if (!strcmp(argv[1], "exp")) x[i] = mr_exp(x[i]);        /* the names the kernels call, in the mode compiled */
        else if (!strcmp(argv[1], "log")) x[i] = mr_log(x[i]);
        else x[i] = mr_sin_ge0(x[i]);
    }
    f = fopen(argv[4], "wb");
    return !f || fwrite(x, sizeof *x, n, f) != (size_t)n || fclose(f);
}
"""


def test_exact_mode_returns_the_stored_glibc_bits(tmp_path):
    """The host rendition of the exact mode against results of glibc 2.39 kept under tests/golden (make_libm_golden.py):
    the check of test_exact_mode_returns_the_host_libms_bits on a sample of its arguments, on any host.  Default mode
    (-DFAST_MODE): exp and log are the same routines, and the sign of the sine is glibc's too."""
    golden = os.path.join(ROOT, "tests", "golden")
    (tmp_path / "driver.c").write_text(LIBM_DRIVER)
    for flags in ([], ["-DFAST_MODE"]):
        exe = tmp_path / ("driver" + "_fast" * bool(flags))
        subprocess.check_call(["gcc", "-O2", "-std=gnu11", "-ffp-contract=off", "-fno-builtin", *flags,
                               "-I", os.path.join(ROOT, "maray_b200", "csrc"), "-o", str(exe), str(tmp_path / "driver.c"), "-lm"])
        for name in ("sin", "exp", "log"):
            pairs = np.load(os.path.join(golden, f"glibc_239_{name}.npy"))
            x, want = pairs[:, 0].view(np.float64), pairs[:, 1].view(np.float64)
            checks = [("sgn", (want >= 0.0).astype(np.float64))] if name == "sin" else []
            if not (flags and name == "sin"):
                checks.append((name, want))
            for fn, expect in checks:
                np.ascontiguousarray(x).tofile(tmp_path / "x.bin")
                subprocess.check_call([str(exe), fn, str(x.size), str(tmp_path / "x.bin"), str(tmp_path / "y.bin")])
                got = np.fromfile(tmp_path / "y.bin", dtype=np.float64)
                same = bits_equal(got, expect)
                assert same.all(), (flags, fn, int((~same).sum()), x[~same][:4], got[~same][:4], expect[~same][:4])


@needs_glibc_239
def test_committed_tables_are_the_host_librarys():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "extract_glibc_libm.py")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert out.stdout == open(os.path.join(ROOT, "maray_b200", "csrc", "glibc_libm_tables.inc")).read()


def _trans_scene(w, h):
    """Three channels that put sin, exp and ln through their ranges: small and large arguments of either sign, the
    table points, the near-1 path of log, overflow/underflow of exp, the out-of-range branches."""
    X, Y = E.x(), E.y()
    cx = E.sub(X, E.nat(w // 2))                                   # -w/2 .. w/2
    rat = lambda p, q: E.div(E.nat(p), E.nat(q))
    s_arg = E.add(E.mul(cx, E.mul(Y, rat(37, 1000))), E.mul(Y, rat(1, 128)))         # |arg| up to ~0.037*w/2*h
    e_arg = E.add(E.mul(cx, rat(3, 2)), E.neg(E.mul(Y, rat(5, 3))))           # from underflow (< -745) to overflow (> 709.78)
    l_arg = E.add(E.nat(1), E.mul(cx, E.mul(E.sub(Y, E.nat(3)), rat(1, 4096))))     # around 1, negative at the edges
    return E.to_bytes([w, h], [E.sin(s_arg), E.exp(e_arg), E.ln(l_arg)])


@pytest.mark.gpu
@needs_glibc_239
@pytest.mark.parametrize("backend", ["nvrtc", "interp"])
def test_transcendental_values_are_bit_exact_in_exact_mode(backend):
    from oracle.oracle import OracleScene
    w, h = 1024, 512
    scene = _trans_scene(w, h)
    want_rgb, want = OracleScene(scene).render_window(0, w, 0, h, want_f64=True)
    with CudaRenderer(gpus=1) as r:
        r.load(scene)
        r.compile(backend, libm="glibc")
        planes, rgb = r.render_window_f64(w, h, 0, w, 0, h)
    for c, name in enumerate(("sin", "exp", "ln")):
        same = bits_equal(planes[c], want[c])
        assert same.all(), (name, int((~same).sum()), planes[c][~same][:4], want[c][~same][:4])
    assert np.array_equal(rgb, want_rgb)
    # and the default libm is NOT bit-exact on this scene: the test distinguishes the two modes
    with CudaRenderer(gpus=1) as r:
        r.load(scene)
        r.compile(backend)
        fast, _ = r.render_window_f64(w, h, 0, w, 0, h)
    assert not bits_equal(fast, want).all()
    assert np.max(np.abs(fast[0] - want[0])) < 2.0 ** -40                                    # sin: absolute
    for c in (1, 2):                                                                          # exp, ln: a few ULP
        ok = np.isfinite(want[c]) & (np.abs(want[c]) > 1e-300)
        assert np.max(np.abs(fast[c][ok] - want[c][ok]) / np.abs(want[c][ok])) < 4e-15


@pytest.mark.gpu
@needs_glibc_239
@pytest.mark.parametrize("backend", ["nvrtc", "interp"])
def test_deep_scene_is_bit_exact_in_exact_mode(backend):
    """Config 5's generator at 20 000 values (the segmented / batched NVRTC form; the interpreter's all-wide form):
    every f64 channel value equals the oracle's."""
    from oracle.oracle import OracleScene
    w, h = 512, 256
    scene = scenes.deep(w, h, n_values=20000, seed=5)
    oracle = OracleScene(scene)
    with CudaRenderer(gpus=1) as r:
        r.load(scene)
        r.compile(backend, libm="glibc")
        for (x0, y0) in [(0, 0), (240, 120), (480, 240)]:
            planes, rgb = r.render_window_f64(w, h, x0, x0 + 32, y0, y0 + 16)
            want_rgb, want = oracle.render_window(x0, x0 + 32, y0, y0 + 16, want_f64=True)
            assert bits_equal(planes, want).all()
            assert np.array_equal(rgb, want_rgb)


@pytest.mark.gpu
@needs_glibc_239
@pytest.mark.parametrize("backend", ["nvrtc", "interp"])
def test_sign_only_rewrites_on_device(backend):
    """step(sin(u)) as the sign of the sine and step(v + c) as a comparison (codegen.cpp find_sign_only_sines) over zero,
    -0, tiny, huge, infinite and NaN operands: exact mode reproduces the oracle's f64 values bit for bit, the default mode
    its bytes; the interpreter (which evaluates the full sine) agrees with the generated kernels."""
    from oracle.oracle import OracleScene
    w, h = 32, 4
    scene = sign_rewrite_scene(w)
    want_rgb, want = OracleScene(scene).render_window(0, w, 0, h, want_f64=True)
    for libm in ("glibc", "fast"):
        with CudaRenderer(gpus=1) as r:
            r.load(scene)
            r.compile(backend, libm=libm)
            planes, rgb = r.render_window_f64(w, h, 0, w, 0, h)
        assert np.array_equal(rgb, want_rgb), libm
        if libm == "glibc":
            assert bits_equal(planes, want).all()


@needs_glibc_239
def test_exact_mode_compiles_without_a_gpu():
    with CudaRenderer(gpus=0) as r:
        r.load(_trans_scene(64, 64))
        st = r.compile("nvrtc", libm="glibc")
        assert st["jit_registers"] > 0
        assert "mr_sin_call(" in r.source()             # exact mode: always out of line
    with CudaRenderer(gpus=0) as r:
        with pytest.raises(Exception):
            r.set_libm("no such libm")
