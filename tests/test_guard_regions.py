"""Guarded regions of the straight-line kernel (codegen.cpp find_guard_regions): the operand of a boolean AND that only
that AND reads is evaluated only when the other operand is true on some lane of the warp (`false && x == false`).

On the host the generated text runs one pixel at a time, in two modes that bracket what a warp does: the vote is the
pixel's own guard (MR_HOST_TEXT), or it is always true (MR_HOST_GUARDS_ALWAYS: every body at every pixel).  Both must
give the oracle's bits.  On the GPU the frames must equal the interpreter's, which has no regions."""
import os

import numpy as np
import pytest

from maray_b200 import CudaRenderer, scenes
from maray_b200 import expr as E
from oracle.oracle import OracleScene

from helpers import bits_equal, host_jit_run

ALWAYS = "#define MR_HOST_GUARDS_ALWAYS 1\n"
VOTE = "if (mr_warp_any("


def _source(scene, monkeypatch, textures=()):
    monkeypatch.setenv("MARAY_JIT_SOURCE_ONLY", "1")
    with CudaRenderer(gpus=0) as r:
        r.set_textures(list(textures))
        r.load(scene)
        with pytest.raises(Exception):
            r.compile("nvrtc")
        return r.source()


def _modules(scene, monkeypatch, textures=()):
    monkeypatch.setenv("MARAY_JIT_SOURCE_ONLY", "1")
    with CudaRenderer(gpus=0) as r:
        r.set_textures(list(textures))
        r.load(scene)
        with pytest.raises(Exception):
            r.compile("nvrtc")
        return r.modules()


def _regions(src):
    """(votes, deepest nesting, values declared inside a region but named outside every region) of the kernel text."""
    import re
    depth = deepest = votes = 0
    inside, outside = set(), set()
    for line in src[src.index('extern "C" __global__'):].splitlines():
        if line.startswith("  " + VOTE):
            votes += 1
            depth += 1
            deepest = max(deepest, depth)
            continue
        if line == "  }":
            depth -= 1
            continue
        decl = re.match(r"\s+(?:const )?(?:bool|double) ([bv]\d+) = (.*)", line)
        names = set(re.findall(r"\b[bv]\d+\b", decl.group(2) if decl else line))
        if depth:
            if decl:
                inside.add(decl.group(1)[1:])
        else:
            outside |= {n[1:] for n in names}
    assert depth == 0
    return votes, deepest, inside & outside


def _check_rows(scene, w, rows, src, textures=()):
    """Both host modes against the oracle's f64 planes, bit for bit, on whole rows."""
    oracle = OracleScene(scene, list(textures))
    for y in rows:
        want_rgb, want = oracle.render_window(0, w, y, y + 1, want_f64=True)
        for text in (src, ALWAYS + src):
            rgb, planes = host_jit_run(text, w, y * w, w, textures)
            assert bits_equal(planes, want.reshape(3, w)).all(), (y, text is src)
            assert np.array_equal(rgb, want_rgb.reshape(w, 3)), (y, text is src)


# ---- which programs get regions ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["chess_1k", "chess_4k"])
def test_chess_has_one_region_per_triangle_texture(monkeypatch, name):
    """64 cells x 2 triangles, each `inside_triangle * texture`: one region per triangle around its texture.  The ANDs
    inside the textures are too light for regions of their own."""
    sc, _tex, _size = scenes.by_name(name)
    src = _source(sc, monkeypatch)
    assert _regions(src) == (128, 1, set())


@pytest.mark.parametrize("name", ["sdf", "textured", "deep"])
def test_other_workloads_have_no_region(monkeypatch, name):
    sc, tex, _size = scenes.by_name(name)
    for unit in _modules(sc, monkeypatch, tex):
        assert VOTE not in unit


# ---- the host text against the oracle ---------------------------------------------------------------------------------
def test_chess_rows_in_both_host_modes(monkeypatch, chess_bytes):
    src = _source(chess_bytes, monkeypatch)
    assert src.count(VOTE) == 128
    _check_rows(chess_bytes, 1024, [512, 600, 700], src)


def test_chess_4k_row_in_both_host_modes(monkeypatch):
    sc = scenes.chess_4k()
    src = _source(sc, monkeypatch)
    _check_rows(sc, 3840, [1485], src)


def _heavy(e, k):
    """e put through k dependent additions and multiplications: a body that weighs about 2k."""
    for i in range(k):
        e = E.mul(E.add(e, E.div(E.nat(i + 3), E.nat(7))), E.div(E.nat(5), E.nat(6)))
    return e


def _edge_scene(w, h):
    x, y = E.x(), E.y()
    inf = E.recip(E.sub(x, E.nat(9)))                                   # +-inf at x = 9
    g1 = E.step(E.sub(x, E.nat(12)))                                    # guards: false left of x = 12 ...
    g2 = E.step(E.sub(y, E.nat(3)))                                     # ... above y = 3
    # 1. a plain region; its body holds NaN (inf * 0 at x = 9) and +-inf, read through a step
    b1 = E.step(_heavy(E.mul(E.add(inf, E.mul(inf, E.sub(x, E.nat(9)))), E.nat(3)), 20))
    r1 = E.mul(g1, b1)
    # 2. the dearer operand is also read by a channel root: no region around it
    shared = E.step(E.sub(_heavy(E.sin(E.mul(x, E.div(E.nat(1), E.nat(3)))), 14), E.nat(1)))
    r2 = E.min(g2, shared)
    # 3. a body value also read by a value outside the AND: it stays outside, the rest of the body is guarded
    inner = _heavy(E.mul(x, y), 6)
    b3 = E.step(E.sub(_heavy(inner, 20), E.nat(40)))
    r3 = E.mul(g2, b3)
    outside = E.mul(inner, E.div(E.nat(1), E.nat(1000)))
    # 4. a body read through the NOT form (1 - b, emitted as !b)
    b4 = E.set_inv(E.step(_heavy(E.sub(y, x), 20)))
    r4 = E.min(g1, b4)
    # 5. nested ANDs: the outer body contains a heavy AND of its own
    inner_and = E.mul(E.step(E.sub(E.mul(x, x), E.nat(300))), E.step(_heavy(E.add(x, E.mul(y, E.nat(2))), 20)))
    b5 = E.max(inner_and, E.step(_heavy(E.sub(x, y), 12)))
    r5 = E.mul(E.step(E.sub(E.nat(30), x)), b5)
    # 6. a boolean times an ordinary value: not an AND, no region
    r6 = E.mul(g1, _heavy(E.add(x, y), 16))
    # 7. a boolean inside a body that is also read through the NOT form outside the AND (`1 + -(b)` reads b itself):
    # it stays outside, the rest of the body is guarded
    c7 = E.step(_heavy(E.sub(E.mul(y, E.nat(3)), x), 8))
    b7 = E.max(c7, E.step(_heavy(E.add(E.mul(x, E.nat(2)), y), 20)))
    r7 = E.mul(g2, b7)
    not_c7 = E.set_inv(c7)
    red = E.add(E.add(E.mul(r1, E.nat(100)), E.mul(r2, E.nat(50))), E.add(E.mul(r3, E.nat(25)), outside))
    green = E.add(E.add(E.mul(r4, E.nat(120)), E.mul(r5, E.nat(60))), shared)
    blue = E.add(E.add(r6, E.mul(E.max(r1, r4), E.nat(7))), E.add(E.mul(r7, E.nat(90)), E.mul(not_c7, E.nat(30))))
    return E.to_bytes([w, h], [red, green, blue])


def test_edge_cases_in_both_host_modes(monkeypatch):
    w, h = 40, 8
    sc = _edge_scene(w, h)
    src = _source(sc, monkeypatch)
    # regions 1, 3, 4, 7 and 5 with 5's inner AND inside it; not 2 (a root reads its body) nor 6 (not boolean); no value
    # declared in a region is named outside it
    assert _regions(src) == (6, 2, set())
    not_reads = {m for m in __import__("re").findall(r"= !b(\d+);", src)}
    assert len(not_reads) >= 2                                  # case 4's NOT inside its body, case 7's outside
    _check_rows(sc, w, list(range(h)), src)


# ---- on the GPU ------------------------------------------------------------------------------------------------------
def _renderer(scene, backend):
    r = CudaRenderer(gpus=1)
    r.load(scene)
    r.compile(backend)
    return r


@pytest.mark.gpu
def test_chess_4k_full_frame_equals_the_interpreter():
    sc = scenes.chess_4k()
    with _renderer(sc, "nvrtc") as r:
        assert r.source().count(VOTE) == 128
        got = r.render(3840, 2160)
    with _renderer(sc, "interp") as r:
        want = r.render(3840, 2160)
    assert np.array_equal(got, want)


@pytest.mark.gpu
def test_chess_1k_against_the_oracle_golden():
    from PIL import Image

    from conftest import GOLDEN
    gold = np.array(Image.open(os.path.join(GOLDEN, "chess_oracle_1024.png")).convert("RGB"))
    with _renderer(scenes.chess_1k(), "nvrtc") as r:
        frame = r.render(1024, 1024)
    with _renderer(scenes.chess_1k(), "interp") as r:
        assert np.array_equal(frame, r.render(1024, 1024))
    assert int((frame != gold).any(axis=2).sum()) <= 1024 * 1024 // 10000


@pytest.mark.gpu
def test_ragged_frame_and_mid_block_bands():
    """1001 x 1024 (warps straddle rows) and bands starting at rows whose first pixel is mid-block, mid-warp."""
    import torch
    sc = scenes.chess_1k()
    w, h = 1001, 1024
    with _renderer(sc, "interp") as r:
        want = r.render(w, h)
    with _renderer(sc, "nvrtc") as r:
        assert np.array_equal(r.render(w, h), want)
        assert np.array_equal(r.render(1001, 77), want[:77])
        frame = torch.zeros(h * w * 3, dtype=torch.uint8, device="cuda")
        for (y0, y1) in [(0, 333), (333, 517), (517, 518), (518, 1024)]:
            r.render_band(w, h, y0, y1, frame.data_ptr() + y0 * w * 3, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert np.array_equal(frame.cpu().numpy().reshape(h, w, 3), want)


@pytest.mark.gpu
def test_supersampled_frame_is_the_box_mean():
    from test_supersample import oracle_box_window
    sc = scenes.chess_1k()
    with _renderer(sc, "nvrtc") as r:
        r.set_samples(2)
        got = r.render(1024, 1024)
    with _renderer(sc, "interp") as r:
        r.set_samples(2)
        assert np.array_equal(got, r.render(1024, 1024))
    window = (384, 640, 500, 532)
    x0, x1, y0, y1 = window
    want = oracle_box_window(sc, 2, window)
    assert int((got[y0:y1, x0:x1] != want).any(axis=2).sum()) <= (x1 - x0) * (y1 - y0) // 1000
