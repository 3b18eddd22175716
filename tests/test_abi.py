"""The C-ABI boundary without a GPU: the library loads, exports every symbol include/maray_cuda.h
declares, and its host side (load, validate, lower, generate, NVRTC-compile) behaves -- including
the error behaviour the header promises.  No compute is launched here."""
import ctypes
import os
import re

import numpy as np
import pytest

from maray_b200 import CudaRenderer, MarayCudaError, _lib, scenes
from maray_b200 import expr as E
from maray_b200.roofline import fp64_ops_per_pixel

from conftest import ROOT


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "maray_cuda.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(maray_cuda_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 17
    L = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(L, name), f"{name} is declared in include/maray_cuda.h but not exported"
    assert declared == {n for n, _, _ in _lib.SYMBOLS}, "ctypes binding and header disagree"
    assert b"sm_100a" in _lib.load().maray_cuda_version()


def test_no_torch_or_oracle_in_the_product():
    """The product path must not route through the oracle, numpy evaluation or torch."""
    for fn in ("render.py", "_lib.py", "expr.py", "scenes.py", "bands.py", "roofline.py", "__init__.py"):
        src = open(os.path.join(ROOT, "maray_b200", fn)).read()
        assert "oracle" not in src.replace("oracle/", "").lower() or fn == "roofline.py" or "import oracle" not in src
        assert "from oracle" not in src and "import oracle" not in src
    out = os.popen(f"ldd {_lib.LIB_PATH}").read()
    assert "libtorch" not in out and "maray_oracle" not in out
    # NVRTC is linked statically: which compiler builds the kernels must not depend on what else is in the process
    # (PyTorch brings its own libnvrtc.so.12, an older one; DESIGN.md section 10 has the miscompile that exposed this).
    assert "nvrtc" not in out and "libcudart" not in out


def test_host_only_handle_compiles_but_cannot_render(chess_bytes):
    with CudaRenderer(gpus=0) as r:
        assert r.load(chess_bytes) == (1024, 1024)
        st = r.compile("interp")
        # program facts pinned by SURVEY.md section 8(a1) / BASELINE.md section 4
        assert st["legacy_layout"] == 1 and st["tree_nodes"] == 3 * 29314
        assert st["n_y_only"] == 845 and st["n_sin"] == 256 and st["n_step"] == 1482
        assert st["n_min"] == 768 and st["n_max"] == 256 and st["n_recip"] == 0 and st["n_sqrt"] == 0
        assert st["dag_nodes"] == st["n_const"] + st["n_x_only"] + st["n_y_only"] + st["n_xy"] + 0
        assert st["interp_instructions"] > st["n_xy"] and 2 < st["interp_slots"] < 400
        assert fp64_ops_per_pixel(st) == st["n_add"] + st["n_mul"] + st["n_step"] + 2 * 1024 + 18 * 256
        with pytest.raises(MarayCudaError) as ei:
            r.render(64, 64)
        assert ei.value.code == _lib.E_CUDA and "no CPU fallback" in ei.value.message


def test_nvrtc_backend_compiles_for_sm_100a_without_a_gpu():
    with CudaRenderer(gpus=0) as r:
        r.load(scenes.sdf(320, 200, 8))
        st = r.compile("nvrtc")
        assert st["jit_cubin_bytes"] > 1000 and st["jit_registers"] > 0 and st["nvrtc_ms"] > 0
        src = r.source()
        assert "maray_jit" in src and "--fmad=false" in src and "mr_sqrt(" in src
        # user arithmetic is never fused: no fma in the generated statements (the libm prelude has its own)
        body = src[src.index('extern "C" __global__'):]
        assert "fma" not in body and " + " in body and " * " in body


def test_error_behaviour():
    with CudaRenderer(gpus=0) as r:
        with pytest.raises(MarayCudaError) as ei:
            r.load(b"\x01\x02\x03")
        assert ei.value.code == _lib.E_PARSE
        with pytest.raises(MarayCudaError) as ei:
            r.load(b"\x00" * 8 + b"\xff\xff\xff\xff" * 3)
        assert ei.value.code == _lib.E_PARSE
        with pytest.raises(MarayCudaError) as ei:
            r.compile("nvrtc")                       # nothing loaded
        assert ei.value.code == _lib.E_INVALID
        # App id outside the runtime's table: the reference panics on the index (src/lib.rs:665)
        r.load(E.to_bytes([8, 8], [E.app(E.channel(1, 0), E.x(), E.y())] * 3))
        r.set_textures([np.zeros((4, 4, 3), np.uint8)])
        with pytest.raises(MarayCudaError) as ei:
            r.compile("interp")
        assert ei.value.code == _lib.E_SCENE and "App id 5" in ei.value.message
        # cyclic Let
        cyc = E.let_([(0, E.add(E.var_id(1), E.nat(1))), (1, E.var_id(0))], E.var_id(0))
        r.load(E.to_bytes([8, 8], [cyc] * 3))
        with pytest.raises(MarayCudaError) as ei:
            r.compile("interp")
        assert ei.value.code == _lib.E_SCENE and "cyclic" in ei.value.message
        # a stray unbound variable is already refused by the loader (the reference yields NaN,
        # src/cache.rs:40).  App keeps the bytes from also decoding under the legacy numbering.
        with pytest.raises(MarayCudaError) as ei:
            r.load(E.to_bytes([8, 8], [E.app(0, E.var_id(3), E.x())] * 3))
        assert ei.value.code == _lib.E_PARSE and "unbound variable" in ei.value.message


def test_texture_dimensions_fold_to_constants():
    e = E.add(E.app(E.image_width(0), E.x(), E.y()), E.app(E.image_height(0), E.nat(0), E.nat(0)))
    with CudaRenderer(gpus=0) as r:
        r.set_textures([np.zeros((7, 13, 3), np.uint8)])
        r.load(E.to_bytes([4, 4], [e, e, e]))
        st = r.compile("interp")
        assert st["dag_nodes"] == 1 and st["n_const"] == 1 and st["n_tex"] == 0
        code, consts = r.bytecode()
        assert 20.0 in consts.tolist()


def test_auto_backend_builds_in_the_background(monkeypatch, tmp_path):
    """MARAY_BACKEND_AUTO on a host-only handle: with an empty cubin cache the compile call returns with the
    bytecode ready (milliseconds) while NVRTC works on another thread -- destroy joins it, and the finished cubin
    lands in the cache --; with the cubin in the cache the generated kernels are installed at once."""
    import time
    monkeypatch.setenv("MARAY_JIT_CACHE", str(tmp_path))
    scene = scenes.sdf(64, 48, 6, seed=4)
    with CudaRenderer(gpus=0) as r:
        r.load(scene)
        t0 = time.perf_counter()
        st = r.compile("auto")
        dt = time.perf_counter() - t0
        assert st["interp_instructions"] > 0 and st["jit_units"] == 0 and r.stats()["jit_active"] == 0
        assert dt < 5.0
    # close() joined the background build; its cubin is in the cache now
    assert any(f.endswith(".mrcubin") for f in os.listdir(tmp_path))
    with CudaRenderer(gpus=0) as r:
        r.load(scene)
        st = r.compile("auto")
        assert st["jit_cache_hit"] == 1 and st["jit_units"] == 1 and r.stats()["jit_active"] == 1
        assert "maray_jit" in r.source()


def test_launch_shape_follows_the_program(monkeypatch, chess_bytes):
    """Large straight-line programs are generated for one 640-thread block per SM (their warps share instruction
    fetches, DESIGN.md 3.1), small ones and programs with batched sin/exp/ln helpers for 256 x 2; MARAY_JIT_BLOCK /
    MARAY_JIT_MIN_BLOCKS set the shape by hand.  (MARAY_JIT_SOURCE_ONLY: the text is generated, NVRTC is not run; the
    stats of a compiled program carry the shape as jit_block / jit_round_pixels, checked on the GPU.)"""
    import re
    monkeypatch.setenv("MARAY_JIT_SOURCE_ONLY", "1")

    def shape(scene, **env):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        with CudaRenderer(gpus=0) as r:
            r.load(scene)
            with pytest.raises(Exception):
                r.compile("nvrtc")
            src = r.source()
        for k in env:
            monkeypatch.delenv(k)
        return int(re.search(r"__launch_bounds__\((\d+)", src).group(1)), src

    # the shipped scene declares 1024 x 1024: 6.92 rounds of 1 024-thread blocks on 148 SMs against 11.07 of 640
    block, src = shape(chess_bytes)
    assert block == 1024 and "__launch_bounds__(1024, 1) maray_jit" in src and "for (unsigned int blk" not in src
    block, src = shape(scenes.chess_4k())             # the same program declared at 3840 x 2160: 87.6 rounds of 640
    assert block == 640 and "__launch_bounds__(640, 1) maray_jit" in src
    block, src = shape(chess_bytes, MARAY_JIT_BLOCK="256")
    assert block == 256 and "__launch_bounds__(256, 2) maray_jit" in src
    block, src = shape(scenes.sdf(64, 48, 6, seed=4))
    assert block == 256 and "__launch_bounds__(256, 2) maray_jit" in src
    block, src = shape(scenes.deep(64, 64, n_values=9000, seed=3))          # batched helpers: scratch rows sized for 256 threads
    assert block == 256 and "#define MR_SCR_STRIDE 256" in src and "mr_scratch_tables_init();" in src
