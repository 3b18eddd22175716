"""Lowering, code generation and bytecode compilation checked on the CPU against the oracle.

The generated CUDA text is compiled as plain C++ with g++ behind a small intrinsic shim and the
bytecode is read by a numpy executor (tests/helpers.py); both must reproduce the oracle's f64
channel values bit for bit.  This proves the host logic before any GPU time is spent; the kernels
themselves are covered by the -m gpu tests."""
import numpy as np
import pytest

from maray_b200 import CudaRenderer, scenes
from maray_b200 import expr as E
from oracle.oracle import OracleScene

from helpers import as_u8, bits_equal, bytecode_run, host_chain_run, host_jit_run, sign_rewrite_scene


def _oracle_window(scene, textures, x0, x1, y0, y1):
    rgb, planes = OracleScene(scene, textures).render_window(x0, x1, y0, y1, want_f64=True)
    return rgb, planes


def _check_scene(scene, w, rows, textures=(), exact_rgb=True):
    with CudaRenderer(gpus=0) as r:
        r.set_textures(list(textures))
        r.load(scene)
        r.compile("interp")
        code, consts = r.bytecode()
        r.compile("nvrtc")
        src = r.source()
    for y in rows:
        want_rgb, want = _oracle_window(scene, list(textures), 0, w, y, y + 1)
        want = want.reshape(3, w)
        rgb, planes = host_jit_run(src, w, y * w, w, textures)
        assert bits_equal(planes, want).all(), f"generated source differs from the oracle on row {y}"
        assert np.array_equal(rgb, want_rgb.reshape(w, 3))
        bc = bytecode_run(code, consts, np.arange(w), np.full(w, y), textures)
        assert bits_equal(bc, want).all(), f"bytecode differs from the oracle on row {y}"
        assert np.array_equal(as_u8(bc).T, want_rgb.reshape(w, 3))


def test_sdf_scene_bit_exact():
    _check_scene(scenes.sdf(320, 200, 16, seed=2), 320, [0, 57, 199])


def test_chess_rows_bit_exact(chess_bytes):
    # the host libm serves both sides here, so even the sin-dependent rows must agree exactly
    _check_scene(chess_bytes, 1024, [512, 700])


def test_textured_scene_bit_exact():
    tex = scenes.synthetic_textures(4, 64)
    _check_scene(scenes.textured(256, 128), 256, [0, 64, 127], tex)


def test_texture_fetch_at_constant_coordinates():
    """App(channel, const, const) -- both coordinates literal.  The bytecode must not route one of them
    through a slot (the kernel fetches operands one instruction ahead of the store)."""
    tex = scenes.synthetic_textures(2, 16)
    x, y = E.x(), E.y()
    t57 = E.app(E.channel(0, 1), E.nat(5), E.nat(7))
    color = [E.add(t57, x), E.mul(E.sin(E.add(E.app(E.channel(1, 2), E.nat(3), E.nat(2)), x)), y),
             E.add(E.mul(t57, y), E.app(E.channel(1, 0), E.nat(15), E.nat(0)))]
    scene = E.to_bytes([24, 6], color)
    _check_scene(scene, 24, [0, 5], tex)


def test_deep_scene_bit_exact():
    _check_scene(scenes.deep(96, 64, n_values=600, seed=4), 96, [0, 33])


def test_deep_scene_is_well_conditioned(monkeypatch):
    """The deep benchmark scene must not amplify last-bit differences between libms: with every sin/exp/log
    result nudged by up to one unit in the last place (tests/helpers.py, perturb_libm) the bytes stay the same
    and the channel values move by less than 1e-9 of a grey level.  (Round 1's generator failed this badly: its
    sin(k*p + c) with k up to 4.5 doubled the sensitivity every few levels -- 8e-11 relative at 12 000 values,
    1e-5 at 40 000, whole grey levels at 100 000 -- so no two libms could agree on its image.)"""
    monkeypatch.setenv("MARAY_JIT_SOURCE_ONLY", "1")
    scene = scenes.deep(64, 64, n_values=12000, seed=5)
    with CudaRenderer(gpus=0) as r:
        r.load(scene)
        with pytest.raises(Exception):
            r.compile("nvrtc")              # MARAY_JIT_SOURCE_ONLY: the text is generated, NVRTC is not run
        src, st = r.source(), r.stats()
    assert st["dag_depth"] > 250 and (st["n_sin"] + st["n_exp"] + st["n_ln"]) / (st["dag_nodes"] - st["n_const"]) >= 0.28
    rgb, planes = host_jit_run(src, 64, 64 * 10, 64)
    rgb_n, planes_n = host_jit_run(src, 64, 64 * 10, 64, perturb_libm=True)
    assert np.array_equal(rgb, rgb_n)
    assert np.abs(planes - planes_n).max() < 1e-9
    assert rgb.std() > 20                                   # and it is an image, not a grey card


def test_segmented_source_matches_unsegmented(monkeypatch):
    scene = scenes.deep(64, 64, n_values=900, seed=11)
    srcs = []
    for seg, inl in (("100000", "100000"), ("64", "0")):
        monkeypatch.setenv("MARAY_JIT_SEGMENT_VALUES", seg)
        monkeypatch.setenv("MARAY_JIT_INLINE_TRANS_BELOW", inl)
        with CudaRenderer(gpus=0) as r:
            r.load(scene)
            st = r.compile("nvrtc")
            srcs.append(r.source())
        assert (st["jit_segments"] > 1) == (seg == "64")
    a = host_jit_run(srcs[0], 64, 64 * 10, 64)
    b = host_jit_run(srcs[1], 64, 64 * 10, 64)
    assert "mr_seg3(" in srcs[1] and "mr_sin_call" in srcs[1]
    assert bits_equal(a[1], b[1]).all() and np.array_equal(a[0], b[0])


def test_boolean_logic_is_value_preserving(monkeypatch, chess_bytes):
    """0/1-valued values (step, products / min / max of them, 1 - b) are emitted as `bool` logic with a
    double shadow (codegen.cpp find_booleans).  The text must evaluate to the oracle's bits: with the
    logic on and off, in one function and cut into segments (booleans crossing a cut travel through the
    frame as doubles and are re-derived), and on constructions that LOOK boolean but are not: -0.0 as a
    constant, step of NaN, a product of a boolean with an ordinary value, 1 - x for a non-boolean x."""
    x, y = E.x(), E.y()
    inf = E.recip(E.nat(0))
    nan = E.mul(E.mul(inf, E.nat(0)), E.add(x, E.nat(1)))
    b1, b2 = E.step(E.sub(x, E.nat(5))), E.step(E.sub(y, E.nat(2)))
    negzero = E.neg(E.nat(0))
    tricky = [
        E.mul(E.add(E.set_xor(b1, b2), E.mul(E.set_inv(b1), E.nat(3))), E.nat(60)),        # NOT feeding arithmetic
        E.recip(E.add(E.mul(E.min(b1, negzero), E.nat(1)), E.mul(b2, negzero))),            # -0.0 is not a boolean: 1/(+-0)
        E.add(E.mul(E.max(E.step(nan), E.mul(b1, E.mul(x, E.recip(E.nat(8))))), E.nat(100)),   # step(NaN) = 0; b * value
              E.mul(E.set_inv(E.mul(x, E.recip(E.nat(16)))), E.nat(50))),                   # 1 - x with x not boolean
    ]
    tricky_scene = E.to_bytes([16, 6], tricky)
    for seg in ("100000", "1500"):
        for on in ("1", "0"):
            monkeypatch.setenv("MARAY_JIT_SEGMENT_VALUES", seg)
            monkeypatch.setenv("MARAY_JIT_BOOLEAN", on)
            cases = [(tricky_scene, 16, [0, 2, 5])]
            if on == "1":                            # the shipped scene without the logic: test_chess_rows_bit_exact's job
                cases.append((chess_bytes, 1024, [511, 512]))
            for scene, w, rows in cases:
                with CudaRenderer(gpus=0) as r:
                    r.load(scene)
                    st = r.compile("nvrtc")
                    src = r.source()
                body = src[src.index("mr_seg0") if "mr_seg0" in src else src.index('extern "C" __global__'):]
                assert ("const bool b" in body) == (on == "1")
                if scene is chess_bytes:
                    assert (st["jit_segments"] > 1) == (seg == "1500")
                for yrow in rows:
                    want_rgb, want = _oracle_window(scene, [], 0, w, yrow, yrow + 1)
                    rgb, planes = host_jit_run(src, w, yrow * w, w)
                    assert bits_equal(planes, want.reshape(3, w)).all(), (seg, on, yrow)
                    assert np.array_equal(rgb, want_rgb.reshape(w, 3))


def test_row_uniform_and_all_wide_bytecode_forms(monkeypatch, chess_bytes):
    """The bytecode's default form keeps values that do not depend on x in the per-block scalar file (the
    GPU counterpart of the reference's row cache, src/cache.rs:18-20); MARAY_INTERP_UNIFORM=0 compiles the
    all-wide form.  Both must evaluate to the oracle's bits (numpy reader, one row at a time, which also
    checks that every scalar really is the same along the row and that scalar slots are never recycled),
    and the per-pixel slot file must shrink -- chess keeps 59 y-only values live at its peak."""
    monkeypatch.setenv("MARAY_INTERP_UNIFORM", "0")
    with CudaRenderer(gpus=0) as r:
        r.load(chess_bytes)
        plain = r.compile("interp")
        code0, consts0 = r.bytecode()
    assert plain["interp_uniform_slots"] == 0 and 60 <= plain["interp_slots"] <= 100
    _rgb, want = _oracle_window(chess_bytes, [], 0, 1024, 700, 701)
    assert bits_equal(bytecode_run(code0, consts0, np.arange(1024), np.full(1024, 700), row_uniform=False), want.reshape(3, 1024)).all()
    monkeypatch.delenv("MARAY_INTERP_UNIFORM")
    tex = scenes.synthetic_textures(1, 32)
    x, y = E.x(), E.y()
    mixed = E.to_bytes([40, 6], [E.add(E.mul(E.sin(E.mul(y, E.nat(3))), x), E.app(E.channel(0, 1), x, E.mul(y, E.nat(2)))),
                                 E.max(E.step(E.sub(y, E.nat(2))), E.mul(E.sqrt(y), E.recip(E.add(x, E.nat(1))))),
                                 E.mul(E.exp(E.neg(y)), E.nat(200))])                  # third channel: y-only root
    for scene, textures, w, rows in ((chess_bytes, [], 1024, [0, 512, 704]), (scenes.sdf(320, 200, 12, seed=3), [], 320, [7, 150]),
                                     (mixed, tex, 40, [0, 3, 5])):
        with CudaRenderer(gpus=0) as r:
            r.set_textures(textures)
            r.load(scene)
            st = r.compile("interp")
            code, consts = r.bytecode()
        handlers = code & np.uint64(0xFF)
        assert st["interp_uniform_slots"] >= 1 and (handlers >= np.uint64(144)).any()
        assert st["interp_block"] % 32 == 0 and st["interp_pixels_per_thread"] in (1, 2, 4)
        if scene is chess_bytes:
            assert st["interp_slots"] <= 40 and st["interp_slots"] < plain["interp_slots"] // 2
        for yrow in rows:
            _rgb, want = _oracle_window(scene, textures, 0, w, yrow, yrow + 1)
            got = bytecode_run(code, consts, np.arange(w), np.full(w, yrow), textures)
            assert bits_equal(got, want.reshape(3, w)).all(), yrow


def test_reference_example_programs():
    """The reference's examples/test.rs, test6.rs and test7.rs re-authored with the DSL mirror (test.rs goes
    through the restated simplify + compress): both back ends' host-checkable forms must evaluate to the
    oracle's bits, and test.rs must come out as the four-definition formula the compressor finds."""
    from maray_b200 import compress as C
    scene = scenes.example_test_rs()
    _size, color, _ = E.from_bytes(scene)
    shape = color[0].a
    assert shape.tag == E.LET and len(shape.vars) == 4
    assert C.fmt(shape.a) == "max(min($2,1-$3),min($3,1-$2))"
    assert C.fmt(shape.vars[3][1]) == "step(1/3-sqrt((x/512-1/2)^2+(y/512-1/2)^2))"
    _check_scene(scene, 512, [0, 100, 256, 400])
    rgb = OracleScene(scene).render_rows([256], 512)[0]
    # the centre row: outside both shapes, inside the circle only, inside both (XOR = 0)
    assert set(int(v) for v in np.unique(rgb)) == {0, 255} and rgb[10, 0] == 0 and rgb[100, 0] == 255 and rgb[256, 0] == 0
    tex = scenes.synthetic_textures(1, 64)
    _check_scene(scenes.example_test6_rs(), 1024, [0, 33, 1023], tex)
    _check_scene(scenes.example_test7_rs(), 128, [0, 127])


def test_let_scoping_and_sharing():
    x, y = E.x(), E.y()
    # Same Let on every channel with different bodies: the canonical compress shape (SURVEY.md F6).
    # $0 refers FORWARD to $2: the interpreter looks names up lazily (reference src/cache.rs:30-38).
    ctx = [(0, E.add(E.var_id(2), x)), (1, E.mul(E.var_id(0), E.var_id(0))), (2, E.mul(y, E.nat(3)))]
    color = [E.let_(ctx, E.var_id(1)), E.let_(ctx, E.sqrt(E.var_id(1))), E.let_(ctx, E.add(E.var_id(2), E.var_id(0)))]
    scene = E.to_bytes([16, 8], color)
    _check_scene(scene, 16, [0, 5])
    # constant operands of App are materialised by the bytecode compiler
    tex = scenes.synthetic_textures(1, 32)
    e = E.app(E.channel(0, 1), E.nat(5), y)
    e2 = E.app(E.channel(0, 2), x, E.nat(7))
    nan_at_9 = E.mul(E.recip(E.nat(0)), E.sub(x, E.nat(9)))            # NaN at x == 9
    e3 = E.app(E.channel(0, 0), E.min(x, nan_at_9), y)                  # NaN coordinate -> column 0
    _check_scene(E.to_bytes([16, 8], [e, e2, E.add(e3, e2)]), 16, [0, 7], tex)


def test_nan_inf_and_zero_sign_semantics():
    x = E.x()
    inf = E.recip(E.nat(0))
    nan = E.add(inf, E.neg(inf))
    negzero = E.neg(E.nat(0))
    xm = E.add(x, E.neg(E.nat(4)))                   # crosses zero inside the row
    color = [
        E.max(E.mul(xm, nan), xm),                   # max(NaN, v) = v
        E.recip(E.min(E.mul(xm, negzero), E.mul(xm, E.nat(0)))),   # +-0 ties, made visible by 1/x
        E.mul(E.step(E.mul(xm, negzero)), E.add(E.mul(inf, xm), E.nat(300))),   # step(-0)=1, inf*0=NaN
    ]
    _check_scene(E.to_bytes([9, 2], color), 9, [0, 1])


def test_sign_only_rewrites_keep_every_value(monkeypatch):
    """codegen.cpp find_sign_only_sines: step(sin(u)) -> mr_sin_ge0(u), step(v + c) -> -v <= c.  The generated text
    (host-compiled) must reproduce the oracle bit for bit with the rewrites and without."""
    scene = sign_rewrite_scene(32)
    with CudaRenderer(gpus=0) as r:
        r.load(scene)
        r.compile("nvrtc")
        src = r.source()
    assert src.count("mr_sin_ge0(") >= 4 + 1 and src.count(") <= ") >= 4      # (+1: the definition in the prelude)
    assert "mr_sin(" in src[src.index('extern "C" __global__'):]               # the sine with two readers stays a sine
    _check_scene(scene, 32, [0, 1, 3])
    monkeypatch.setenv("MARAY_JIT_SIGN_OF_SINE", "0")
    with CudaRenderer(gpus=0) as r:
        r.load(scene)
        r.compile("nvrtc")
        assert "mr_sin_ge0(" not in r.source()[r.source().index('extern "C" __global__'):]
    _check_scene(scene, 32, [0, 1, 3])


@pytest.mark.parametrize("form", ["scratch", "chain", "functions"])
def test_transcendental_batching_keeps_values(monkeypatch, form):
    """Programs with >= 2048 sin/exp/ln values get their schedule batched and call out-of-line helpers
    through the per-thread shared-memory scratch.  Above the segment size a program is cut: into a CHAIN of kernels, one translation unit each, values crossing a cut
    in a global frame (default), or into segment functions inside one unit (MARAY_JIT_CHAIN=0)."""
    monkeypatch.setenv("MARAY_JIT_SEGMENT_VALUES", "3000" if form in ("chain", "functions") else "100000")
    if form in ("chain", "functions"):
        monkeypatch.setenv("MARAY_JIT_CACHE", "off")          # the compile statistics below are those of a real compile
    if form == "functions":
        monkeypatch.setenv("MARAY_JIT_CHAIN", "0")
    scene = scenes.deep(48, 32, n_values=9000, seed=3)
    with CudaRenderer(gpus=0) as r:
        r.load(scene)
        st = r.compile("nvrtc")
        src = r.source()
        modules = r.modules()
        r.compile("interp")
        code, consts = r.bytecode()
    assert st["n_sin"] + st["n_exp"] + st["n_ln"] >= 2048
    body = src[src.index("mr_seg0") if "mr_seg0" in src else src.index('extern "C" __global__'):]
    assert "_batch" in body and "MR_R(" in body
    want_rgb, want = _oracle_window(scene, [], 0, 48, 7, 8)
    if form == "chain":
        assert st["jit_segments"] >= 3 and st["jit_units"] == st["jit_segments"] == len(modules) and st["jit_compile_threads"] >= 1
        assert st["jit_frame_slots"] > 0 and st["jit_cubin_bytes"] > 1000
        assert all("double* __restrict__ F, const unsigned long long FS" in m for m in modules) and "mr_store_block" in modules[-1]
        assert all("mr_store_block(p" not in m for m in modules[:-1])
        rgb, planes = host_chain_run(modules, 48, 7 * 48, 48, st["jit_frame_slots"])
        assert bits_equal(planes, want.reshape(3, 48)).all() and np.array_equal(rgb, want_rgb.reshape(48, 3))
    else:
        assert st["jit_units"] == 1 and len(modules) == 1 and modules[0] == src
        assert (st["jit_segments"] >= 3) == (form == "functions")
    rgb, planes = host_jit_run(src, 48, 7 * 48, 48)
    assert bits_equal(planes, want.reshape(3, 48)).all() and np.array_equal(rgb, want_rgb.reshape(48, 3))
    bc = bytecode_run(code, consts, np.arange(48), np.full(48, 7))
    assert bits_equal(bc, want.reshape(3, 48)).all()


def test_cubin_cache_round_trip(monkeypatch, tmp_path):
    """MARAY_JIT_CACHE: the second compile of the same scene with the same options loads the cubin
    from the directory (no NVRTC run); a different option misses."""
    monkeypatch.setenv("MARAY_JIT_CACHE", str(tmp_path))
    scene = scenes.sdf(64, 48, 6, seed=4)
    stats = []
    for _ in range(2):
        with CudaRenderer(gpus=0) as r:
            r.load(scene)
            stats.append(r.compile("nvrtc"))
    assert stats[0]["jit_cache_hit"] == 0 and stats[1]["jit_cache_hit"] == 1
    assert stats[0]["jit_cubin_bytes"] == stats[1]["jit_cubin_bytes"] and stats[1]["jit_registers"] == stats[0]["jit_registers"]
    assert len(list(tmp_path.glob("*.mrcubin"))) == 1
    monkeypatch.setenv("MARAY_JIT_MIN_BLOCKS", "1")
    with CudaRenderer(gpus=0) as r:
        r.load(scene)
        assert r.compile("nvrtc")["jit_cache_hit"] == 0
    assert len(list(tmp_path.glob("*.mrcubin"))) == 2


def _random_scene(seed: int, w: int, h: int, n_values: int):
    """Seeded random DAG over every non-transcendental operation, rich in the shapes the boolean logic and
    the segment cuts care about: steps, 1 - b, products / min / max of booleans and of ordinary values,
    negated booleans, +-0, infinities and NaN (1/0, inf - inf), values shared across channels."""
    rng = scenes.Lcg(seed)
    x, y = E.x(), E.y()
    pool = [x, y, E.div(x, E.nat(w)), E.div(y, E.nat(h)), E.sub(x, E.nat(rng.between(1, w - 1))),
            E.sub(y, E.nat(rng.between(0, h - 1))), E.nat(0), E.nat(1), E.neg(E.nat(0)), E.recip(E.nat(0))]
    bools = []
    for _ in range(n_values):
        k = rng.below(100)
        a = pool[rng.below(len(pool))]
        b = pool[rng.below(len(pool))]
        if k < 18:
            v = E.step(a); bools.append(v)
        elif k < 30 and bools:
            p, q = bools[rng.below(len(bools))], bools[rng.below(len(bools))]
            v = [E.set_and(p, q), E.set_or(p, q), E.mul(p, q), E.set_inv(p), E.set_xor(p, q), E.neg(p)][rng.below(6)]
            if v.tag != E.NEG:
                bools.append(v)
        elif k < 45:
            v = E.add(a, b)
        elif k < 60:
            v = E.mul(a, b)
        elif k < 68:
            v = E.max(a, b)
        elif k < 76:
            v = E.min(a, b)
        elif k < 82:
            v = E.neg(a)
        elif k < 87:
            v = E.abs(a)
        elif k < 92:
            v = E.recip(a)
        elif k < 96:
            v = E.sqrt(E.abs(a))
        else:
            v = E.sub(E.nat(1), a)                      # 1 - a with a NOT necessarily boolean
        pool.append(v)
    chans = []
    for c in range(3):
        acc = pool[-1 - c]
        for _ in range(6):
            acc = E.add(acc, E.mul(pool[rng.below(len(pool))], E.nat(rng.between(1, 9))))
        chans.append(E.mul(E.min(E.max(acc, E.neg(E.nat(2))), E.nat(3)), E.nat(50)))
    return E.to_bytes([w, h], E.share_let(chans))


@pytest.mark.parametrize("seed", range(8))
def test_random_scenes_bit_exact(monkeypatch, seed):
    """Property test of lowering + both code generators against the oracle on seeded random programs
    (no transcendentals: every bit must match), unsegmented and cut into small segments."""
    w, h = 24, 5
    scene = _random_scene(seed + 100, w, h, 260)
    for seg in ("100000", "64"):
        monkeypatch.setenv("MARAY_JIT_SEGMENT_VALUES", seg)
        _check_scene(scene, w, [0, 2, 4])
