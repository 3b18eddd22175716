"""Parity of the CUDA path with the oracle, through the C ABI, on a real B200 (`-m gpu`).

Bars (BASELINE.json north_star):
  * scenes made of + * neg 1/ sqrt abs min max step: bit-exact f64 channel values and RGB8 bytes;
  * transcendental scenes: RGB8 equal to the oracle on >= 99.99 % of pixels; a differing channel is
    either within 1 LSB (CUDA libm vs glibc in the last bits) or a `step` flip, which is attributed by
    showing that the step argument is within a few ULP of zero (SURVEY.md F5).
Full-size frames are additionally checked through size-independent properties: the two back ends
(independent kernels) agree, bands reassemble the frame, windows equal the frame."""
import os

import numpy as np
import pytest
from PIL import Image

from maray_b200 import CudaRenderer, RenderMethod, Report, Runtime, Textures, gen_to_image, scenes
from maray_b200 import expr as E
from maray_b200.render import MarayCudaError
from oracle.oracle import OracleScene

from conftest import GOLDEN
from helpers import bits_equal

pytestmark = pytest.mark.gpu
BACKENDS = ["nvrtc", "interp"]


def _renderer(scene, backend, textures=(), gpus=1):
    r = CudaRenderer(gpus=gpus)
    r.set_textures(list(textures))
    r.load(scene)
    r.compile(backend)
    return r


@pytest.mark.parametrize("backend", BACKENDS)
def test_known_answers_on_device(backend):
    """The reference's `it_works` vectors (src/lib.rs:1241-1285), evaluated at pixel (x, 0)."""
    X = E.x()
    half = E.div(X, E.nat(2))                        # pixel coordinates are integers: x/2 reaches .5 values
    cases = [
        (E.mul(X, X), {2: 4.0}),
        (E.neg(E.nat(1)), {0: -1.0}),
        (E.div(E.nat(1), E.nat(2)), {0: 0.5}),
        (E.pi(), {0: 3.141592653589793}),
        (E.lerp(E.neg(E.nat(1)), E.nat(1), X), {0: -1.0, 1: 1.0}),
        (E.cos(X), {0: 1.0}),
        (E.step(E.sub(X, E.nat(1))), {0: 0.0, 1: 1.0, 2: 1.0}),
        (E.step_at(E.nat(2), X), {1: 0.0, 2: 1.0}),
        (E.range(E.nat(1), E.nat(2), half), {1: 0.0, 3: 1.0, 5: 0.0}),
        (E.p2_len([X, X]), {0: 0.0, 1: 2.0 ** 0.5}),
        (E.clamp(E.nat(1), E.nat(5), X), {0: 1.0, 1: 1.0, 5: 5.0, 6: 5.0}),
    ]
    for e, want in cases:
        with _renderer(E.to_bytes([8, 1], [e, e, e]), backend) as r:
            planes, _ = r.render_window_f64(8, 1, 0, 8, 0, 1)
        for x, v in want.items():
            assert planes[0, 0, x] == v, (e, x, v, planes[0, 0, x])


@pytest.mark.parametrize("backend", BACKENDS)
def test_sdf_bit_exact(backend):
    """Config 2 at full size: 1920x1080, f64 planes of 64x64 tiles and sampled rows vs the oracle."""
    scene = scenes.sdf()
    w, h = 1920, 1080
    oracle = OracleScene(scene)
    with _renderer(scene, backend) as r:
        frame = r.render(w, h)
        for (x0, y0) in [(0, 0), (928, 508), (1856, 1016)]:
            planes, rgb = r.render_window_f64(w, h, x0, x0 + 64, y0, y0 + 64)
            want_rgb, want = oracle.render_window(x0, x0 + 64, y0, y0 + 64, want_f64=True)
            assert bits_equal(planes, want).all()
            assert np.array_equal(rgb, want_rgb)
            assert np.array_equal(frame[y0:y0 + 64, x0:x0 + 64], want_rgb)
    rows = [0, 137, 540, 1079]
    want_rows = oracle.render_rows(rows, w)
    for i, y in enumerate(rows):
        assert np.array_equal(frame[y], want_rows[i])


def test_backends_agree_on_full_frames():
    """Two independent kernels (generated straight-line code, bytecode interpreter) must produce the
    same bytes on whole frames -- a size-independent check at BASELINE sizes."""
    for scene, (w, h), tex in [(scenes.sdf(), (1920, 1080), ()),
                               (scenes.chess_1k(), (1024, 1024), ()),
                               (scenes.textured(1920, 1080), (1920, 1080), scenes.synthetic_textures(4, 512))]:
        frames = []
        for backend in BACKENDS:
            with _renderer(scene, backend, tex) as r:
                frames.append(r.render(w, h))
        assert np.array_equal(frames[0], frames[1])


def _attribute_mismatches(scene, got, want, max_report=50):
    """Every differing pixel must be a <=1 LSB difference or a 0<->255-style step flip."""
    diff = (got.astype(np.int16) - want.astype(np.int16))
    bad = np.abs(diff) > 1
    return int((diff != 0).any(axis=2).sum()), int(bad.any(axis=2).sum())


STEP_FLIP_ULP = 64.0


def _assert_flips_are_step_boundaries(oracle, got, want, x0=0, y0=0, textures=None):
    """SURVEY.md F5: a channel that differs by more than 1 LSB must be a `step` flip.  For every such
    pixel the oracle re-evaluates the scene and reports how close the nearest step argument is to zero
    (in ULP of the larger term of the sum it comes from): a flip is legitimate only if some step sits
    within a few ULP of its threshold, where the last bits of sin/exp/ln decide."""
    diff = np.abs(got.astype(np.int16) - want.astype(np.int16)).max(axis=2)
    ys, xs = np.nonzero(diff > 1)
    for y, x in zip(ys.tolist(), xs.tolist()):
        m = oracle.step_margin(float(x0 + x), float(y0 + y))
        assert m <= STEP_FLIP_ULP, f"pixel ({x0 + x},{y0 + y}) differs by {diff[y, x]} but no step argument is near zero (margin {m:.3g} ULP)"
    return len(ys)


@pytest.mark.parametrize("backend", BACKENDS)
def test_chess_against_oracle_golden(backend):
    """Config 1: the shipped scene at its stored size vs the committed full oracle render."""
    gold = np.array(Image.open(os.path.join(GOLDEN, "chess_oracle_1024.png")).convert("RGB"))
    ref_png = np.array(Image.open(os.path.join(GOLDEN, "chess_reference.png")).convert("RGB"))
    with _renderer(scenes.chess_1k(), backend) as r:
        frame = r.render(1024, 1024)
        mism = (frame != gold).any(axis=2)
        n_mism = int(mism.sum())
        assert n_mism <= 1024 * 1024 // 10000, f"{n_mism} pixels differ from the oracle (> 0.01 %)"
        # attribute: every mismatch is a step flip (0 <-> 255 on all three channels) whose step argument
        # the oracle finds within a few ULP of zero (SURVEY.md F5) ...
        if n_mism:
            ys, xs = np.nonzero(mism)
            assert set(np.unique(np.abs(frame[ys, xs].astype(int) - gold[ys, xs].astype(int)))) <= {255}
            assert _assert_flips_are_step_boundaries(OracleScene(scenes.chess_1k()), frame, gold) == n_mism
        # ... and the reference's own PNG differs from us only where it differs from the oracle
        # (rows 512 and 704, SURVEY.md F4) or on those flips
        d_png = (frame != ref_png).any(axis=2)
        rows = set(np.nonzero(d_png & ~mism)[0].tolist())
        assert rows <= {512, 704}


@pytest.mark.parametrize("backend", BACKENDS)
def test_textured_scene(backend):
    """Config 4 shape (smaller frame and textures): texture lookups incl. the out-of-range branches."""
    tex = scenes.synthetic_textures(4, 256)
    scene = scenes.textured(960, 540)
    oracle = OracleScene(scene, tex)
    with _renderer(scene, backend, tex) as r:
        frame = r.render(960, 540)
        for (x0, y0) in [(0, 0), (448, 238), (896, 476)]:
            planes, rgb = r.render_window_f64(960, 540, x0, x0 + 64, y0, y0 + 64)
            want_rgb, want = oracle.render_window(x0, x0 + 64, y0, y0 + 64, want_f64=True)
            assert bits_equal(planes, want).all()
            assert np.array_equal(rgb, want_rgb)
    rows = [0, 270, 539]
    want_rows = oracle.render_rows(rows, 960)
    for i, y in enumerate(rows):
        assert np.array_equal(frame[y], want_rows[i])


@pytest.mark.parametrize("backend", BACKENDS)
def test_texture_edges_and_out_of_range(backend):
    """fun_color_channel's early returns (reference src/textures.rs:30,34): negative coordinates,
    coordinates at and beyond the texture edge, and the truncation of fractional coordinates."""
    tex = scenes.synthetic_textures(2, 16)
    x, y = E.x(), E.y()
    u = E.div(E.sub(x, E.nat(6)), E.nat(2))          # -3.0 .. 12.5 in steps of .5
    v = E.sub(y, E.nat(3))
    nan_at_9 = E.mul(E.recip(E.nat(0)), E.sub(x, E.nat(9)))   # inf*(x-9): NaN at x == 9, +-inf elsewhere
    color = [E.app(E.channel(0, 0), u, v), E.app(E.channel(1, 1), v, u),
             E.app(E.channel(1, 2), E.min(u, nan_at_9), E.mul(v, v))]   # NaN coordinate -> texel column 0
    scene = E.to_bytes([40, 24], color)
    want_rgb, want = OracleScene(scene, tex).render_window(0, 40, 0, 24, want_f64=True)
    with _renderer(scene, backend, tex) as r:
        planes, rgb = r.render_window_f64(40, 24, 0, 40, 0, 24)
    assert bits_equal(planes, want).all() and np.array_equal(rgb, want_rgb)
    assert (want[0][:, :6] == 0).all() and (want[0][:3] == 0).all() and (want[0][3:19, 6:38] != 0).any()


@pytest.mark.parametrize("backend", BACKENDS)
def test_deep_transcendental_scene_within_tolerance(backend):
    """Config 5 shape at a size the oracle finishes: >= 99.99 % identical bytes, rest within 1 LSB;
    f64 channel values within 1e-10 of the oracle's on the 0..255 scale (the device sin/exp/log are <= 1.5/0.9/0.6
    ULP; the generator's maps never expand a difference, the final 127.5*sin(40*mean) scales it by ~5000)."""
    scene = scenes.deep(192, 128, n_values=500, seed=7)
    w, h = 192, 128
    want_rgb, want = OracleScene(scene).render_window(0, w, 0, h, want_f64=True)
    with _renderer(scene, backend) as r:
        planes, rgb = r.render_window_f64(w, h, 0, w, 0, h)
        frame = r.render(w, h)
    assert np.array_equal(frame, rgb)
    n_diff, n_bad = _attribute_mismatches(scene, rgb, want_rgb)
    assert n_bad == 0, "a channel differs from the oracle by more than 1 LSB"
    assert n_diff <= max(1, w * h // 10000)
    assert np.nanmax(np.abs(planes - want)) < 1e-10


def _heavy_scene_with_out_of_range_arguments(w, h):
    """>= 2048 sin/exp/ln values (so the NVRTC back end batches them through out-of-line helpers) plus
    arguments outside every fast range: sin of ~1e9 and of inf (NaN), exp beyond 709 (inf) and below
    -745 (0), ln of a negative (NaN), of 0 (-inf) and of a subnormal."""
    _size, color, _ = E.from_bytes(scenes.deep(w, h, n_values=9000, seed=3))
    x, y = E.x(), E.y()
    inf = E.recip(E.nat(0))
    tiny = E.exp(E.neg(E.nat(740)))                                   # subnormal constant, folded on the host
    odd = [
        E.sin(E.mul(E.add(x, E.nat(3)), E.nat(123456789))),            # huge: Payne-Hanek territory
        E.sin(E.mul(inf, E.add(x, E.nat(1)))),                          # sin(inf) = NaN
        E.exp(E.mul(E.add(y, E.nat(1)), E.nat(400))),                   # overflow to inf
        E.exp(E.neg(E.mul(E.add(y, E.nat(2)), E.nat(400)))),            # underflow to 0
        E.ln(E.add(x, E.neg(E.nat(5)))),                                # negative -> NaN, 0 -> -inf
        E.ln(E.mul(tiny, E.add(x, E.nat(1)))),                          # subnormal argument
    ]
    # f64::max/min ignore NaN (reference src/lib.rs:652-655), so every channel stays defined
    extra = [E.mul(E.max(E.nat(0), E.min(E.nat(1), E.mul(t, t))), E.nat(40)) for t in odd]
    def inner(c):
        return c.a if c.tag == E.LET else c
    assert all(c.tag == E.LET for c in color)
    out = []
    for i, c in enumerate(color):
        body = E.add(E.add(c.a, extra[2 * i]), extra[2 * i + 1])
        out.append(E.let_(c.vars, body))
    return E.to_bytes([w, h], out)


@pytest.mark.parametrize("form", ["scratch", "chain", "functions"])
def test_batched_transcendentals_and_their_repair_path(monkeypatch, form):
    """The out-of-line sin/exp/ln forms of the NVRTC back end on a program above the batching threshold,
    with arguments that must take the libdevice repair path, and both ways of cutting a large program (a chain
    of kernels over a global frame -- rendered in several chunks here --, segment functions in one unit).  All
    forms run the same device routines, so their f64 planes must be bit-identical to each other; against the
    oracle the usual tolerance."""
    w, h = 96, 64
    scene = _heavy_scene_with_out_of_range_arguments(w, h)
    want_rgb, want = OracleScene(scene).render_window(0, w, 0, h, want_f64=True)
    monkeypatch.setenv("MARAY_JIT_SEGMENT_VALUES", "3000" if form in ("chain", "functions") else "100000")
    if form == "functions":
        monkeypatch.setenv("MARAY_JIT_CHAIN", "0")
    if form == "chain":
        monkeypatch.setenv("MARAY_JIT_FRAME_MB", "1")        # 1 MiB of frame: the 96x64 image takes several chunks
    with _renderer(scene, "nvrtc") as r:
        st = r.stats()
        planes, rgb = r.render_window_f64(w, h, 0, w, 0, h)
        frame = r.render(w, h)
    if form == "chain":
        assert st["jit_units"] == st["jit_segments"] >= 3
    if form == "functions":
        assert st["jit_units"] == 1 and st["jit_segments"] >= 3
    assert np.array_equal(frame, rgb)
    for k in ("MARAY_JIT_CHAIN", "MARAY_JIT_SEGMENT_VALUES", "MARAY_JIT_FRAME_MB"):
        monkeypatch.delenv(k, raising=False)
    # yardstick: the interpreter kernel, whose handlers inline the scalar routines
    with _renderer(scene, "interp") as r:
        ref_planes, ref_rgb = r.render_window_f64(w, h, 0, w, 0, h)
    assert bits_equal(planes, ref_planes).all(), "batched and inlined sin/exp/ln disagree"
    assert np.array_equal(rgb, ref_rgb)
    n_diff, n_bad = _attribute_mismatches(scene, rgb, want_rgb)
    assert n_bad == 0 and n_diff <= max(1, w * h // 10000)


@pytest.mark.parametrize("backend", BACKENDS)
def test_nan_inf_zero_semantics_on_device(backend):
    x = E.x()
    inf = E.recip(E.nat(0))
    nan = E.add(inf, E.neg(inf))
    negzero = E.neg(E.nat(0))
    xm = E.add(x, E.neg(E.nat(4)))
    color = [
        E.max(E.mul(xm, nan), xm),
        E.recip(E.min(E.mul(xm, negzero), E.mul(xm, E.nat(0)))),
        E.mul(E.step(E.mul(xm, negzero)), E.add(E.mul(inf, xm), E.nat(300))),
    ]
    scene = E.to_bytes([9, 2], color)
    want_rgb, want = OracleScene(scene).render_window(0, 9, 0, 2, want_f64=True)
    with _renderer(scene, backend) as r:
        planes, rgb = r.render_window_f64(9, 2, 0, 9, 0, 2)
    assert bits_equal(planes, want).all()
    assert np.array_equal(rgb, want_rgb)


@pytest.mark.parametrize("backend", BACKENDS)
def test_clamp_of_nan_with_literal_bounds(backend):
    """max(0, min(1, t)) with literal bounds and t = NaN must be 1 (f64::min ignores the NaN, reference
    src/lib.rs:655-658); the compiler's own min/max pattern turns the pair into min(1, max(0, t)) = 0
    (device_sem.cuh, mr_pick).  Also the mirrored clamp, and bounds on the other side."""
    x = E.x()
    inf = E.recip(E.nat(0))
    t_nan = E.mul(E.mul(inf, E.nat(0)), E.add(x, E.nat(1)))           # NaN at every pixel, not foldable
    t_mixed = E.ln(E.add(x, E.neg(E.nat(3))))                         # NaN for x < 3, -inf at 3, numbers after
    def clamp(t): return E.max(E.nat(0), E.min(E.nat(1), t))
    def clamp_rev(t): return E.min(E.nat(1), E.max(E.nat(0), t))
    color = [E.mul(clamp(t_nan), E.nat(200)),
             E.mul(clamp(E.mul(t_mixed, t_mixed)), E.nat(200)),
             E.mul(E.add(clamp_rev(t_mixed), E.max(E.min(t_mixed, E.nat(1)), E.nat(0))), E.nat(100))]
    scene = E.to_bytes([8, 1], color)
    want_rgb, want = OracleScene(scene).render_window(0, 8, 0, 1, want_f64=True)
    assert want[0, 0, 0] == 200.0 and want[1, 0, 0] == 200.0          # the NaN is ignored: min gives the bound 1
    with _renderer(scene, backend) as r:
        planes, rgb = r.render_window_f64(8, 1, 0, 8, 0, 1)
    assert np.array_equal(rgb, want_rgb)
    assert (np.abs(planes - want) <= 1e-13 * np.abs(want)).all()      # ln differs from glibc in the last bits only


@pytest.mark.parametrize("backend", BACKENDS)
def test_ragged_sizes_bands_and_windows(backend):
    """Odd widths (unaligned row starts), a 1x1 image, bands that do not divide the height."""
    scene = scenes.sdf(333, 77, 5, seed=8)
    want = OracleScene(scene).render(333, 77)
    with _renderer(scene, backend) as r:
        assert np.array_equal(r.render(333, 77), want)
        assert np.array_equal(r.render(1, 1), want[:1, :1])
        assert np.array_equal(r.render(2, 77), want[:, :2])
        # bands through the one-process-per-GPU entry point, into one device frame
        import torch
        frame = torch.zeros(77 * 333 * 3, dtype=torch.uint8, device="cuda")
        for (y0, y1) in [(0, 26), (26, 51), (51, 77)]:
            r.render_band(333, 77, y0, y1, frame.data_ptr() + y0 * 333 * 3, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert np.array_equal(frame.cpu().numpy().reshape(77, 333, 3), want)


def test_gen_to_image_entry_point_and_report():
    """The reference-shaped call (src/lib.rs:1177-1195) incl. the progress callback (Report::Row)."""
    scene = scenes.sdf(256, 128, 6, seed=5)
    size, color, _ = E.from_bytes(scene)
    img = np.zeros((128, 256, 3), dtype=np.uint8)
    ticks = []
    gen_to_image(RenderMethod.Cuda(gpus=1, report=Report.row(32)), Runtime.new(), color, img,
                 lambda partial, p: ticks.append((p, int(partial[:int(p * 128)].any()))))
    assert np.array_equal(img, OracleScene(scene).render())
    assert [p for p, _ in ticks] == [0.25, 0.5, 0.75]


# ---- BASELINE.json configs 3, 4, 5 at their stated sizes -------------------------------------------
def _windows_and_rows_vs_oracle(r, oracle, w, h, windows, rows, exact, frame=None):
    """f64 windows + full rows of a w x h render against the oracle.  exact: bit-identical planes and
    bytes; otherwise >= 99.99 % identical bytes, the rest <= 1 LSB or an attributed step flip."""
    frame = r.render(w, h) if frame is None else frame
    n_px = n_diff = 0
    for (x0, y0, ww, hh) in windows:
        planes, rgb = r.render_window_f64(w, h, x0, x0 + ww, y0, y0 + hh)
        want_rgb, want = oracle.render_window(x0, x0 + ww, y0, y0 + hh, want_f64=True)
        assert np.array_equal(frame[y0:y0 + hh, x0:x0 + ww], rgb), "window render differs from the same region of the frame"
        if exact:
            assert bits_equal(planes, want).all(), f"f64 planes differ from the oracle in window {(x0, y0)}"
            assert np.array_equal(rgb, want_rgb)
        else:
            _assert_flips_are_step_boundaries(oracle, rgb, want_rgb, x0, y0)
            n_diff += int((rgb != want_rgb).any(axis=2).sum())
            close = (np.abs(rgb.astype(np.int16) - want_rgb.astype(np.int16)) <= 1).transpose(2, 0, 1)   # not a step flip
            ok = np.isfinite(want) & close
            assert np.nanmax(np.abs(planes[ok] - want[ok]) / np.maximum(np.abs(want[ok]), 1.0), initial=0.0) < 1e-9
        n_px += ww * hh
    if rows:
        want_rows = oracle.render_rows(rows, w)
        for i, y in enumerate(rows):
            if exact:
                assert np.array_equal(frame[y], want_rows[i]), f"row {y} differs from the oracle"
            else:
                _assert_flips_are_step_boundaries(oracle, frame[y][None], want_rows[i][None], 0, y)
                n_diff += int((frame[y] != want_rows[i]).any(axis=1).sum())
        n_px += len(rows) * w
    if not exact:
        assert n_diff <= max(1, n_px // 10000), f"{n_diff} of {n_px} sampled pixels differ from the oracle"
    return frame


def test_chess_4k_benchmark_workload_against_oracle():
    """Config 3 as benchmarked (bench.py's default workload): three 64x64 f64 windows and four full rows
    of the 3840x2160 frame against the oracle, the interpreter kernel on the same rows."""
    scene = scenes.chess_4k()
    w, h = 3840, 2160
    oracle = OracleScene(scene)
    with _renderer(scene, "nvrtc") as r:
        frame = _windows_and_rows_vs_oracle(r, oracle, w, h, [(1888, 1048, 64, 64), (760, 1060, 64, 64), (3000, 1700, 64, 64)],
                                            [0, 1080, 1485, 2159], exact=False)
    assert frame.any() and not frame.all()
    with _renderer(scene, "interp") as r:
        import torch
        band = torch.zeros(8 * w * 3, dtype=torch.uint8, device="cuda")
        r.render_band(w, h, 1480, 1488, band.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert np.array_equal(band.cpu().numpy().reshape(8, w, 3), frame[1480:1488])


def test_chess_regenerated_from_the_example_at_4k():
    """Config 3 literally: examples/chess.rs re-run through the builder at [3840, 2160] (without
    simplify/compress, which HEAD cannot run on this scene: DESIGN.md section 11)."""
    scene = scenes.chess_dsl(3840, 2160)
    w, h = 3840, 2160
    with _renderer(scene, "nvrtc") as r:
        frame = _windows_and_rows_vs_oracle(r, OracleScene(scene), w, h, [(1888, 1048, 64, 64), (700, 1100, 64, 64), (3100, 1690, 64, 64)],
                                            [1081, 1500, 1727], exact=False)
    assert frame.any() and not frame.all()


@pytest.mark.parametrize("backend", BACKENDS)
def test_textured_scene_at_stated_size(backend):
    """Config 4 at its stated size: 3840x2160 over four 2048x2048 textures; windows in all four corners
    (where the rotated/offset footprints leave the textures on both sides) and in the middle."""
    tex = scenes.synthetic_textures(4, 2048)
    scene = scenes.textured(3840, 2160)
    w, h = 3840, 2160
    oracle = OracleScene(scene, tex)
    windows = [(0, 0, 64, 64), (3776, 0, 64, 64), (0, 2096, 64, 64), (3776, 2096, 64, 64), (1900, 1000, 64, 64)]
    # the corner windows do reach both zero-return branches of fun_color_channel (src/textures.rs:30,34):
    # texture 2's v = (5x + 12y)/13 * 2048/3840 - 400 is negative at the top, texture 1's
    # v = (3x + 4y)/5 * 2048/3840 + 200 exceeds 2047 at the bottom right
    assert (5 * 63 + 12 * 63) / 13 * 2048 / 3840 - 400 < 0 and (3 * 3776 + 4 * 2096) / 5 * 2048 / 3840 + 200 >= 2048
    with _renderer(scene, backend, tex) as r:
        _windows_and_rows_vs_oracle(r, oracle, w, h, windows, [0, 1079, 2159], exact=True)


def test_deep_scene_at_stated_size_default_path():
    """Config 5 at its stated size: ~1e5 values, 8192x8192, through the DEFAULT form of the NVRTC back end
    for a program of this size (a chain of segment kernels over a global frame).  Small windows -- the
    oracle's by-name Let lookup makes one pixel of this scene cost ~0.2 s of CPU -- spread over the frame,
    and size-independent properties of the full frame: bands reassemble it, windows equal it."""
    scene = scenes.deep()
    w, h = 8192, 8192
    oracle = OracleScene(scene)
    with _renderer(scene, "nvrtc") as r:
        st = r.stats()
        assert st["dag_nodes"] > 90000 and st["jit_segments"] > 1 and st["jit_units"] == st["jit_segments"]   # a chain of kernels
        windows = [(0, 0, 16, 8), (4088, 4090, 16, 8), (8176, 8184, 16, 8), (1000, 7000, 16, 8)]
        frame = _windows_and_rows_vs_oracle(r, oracle, w, h, windows, [], exact=False)
        import torch
        bands_buf = torch.zeros(64 * w * 3, dtype=torch.uint8, device="cuda")
        for (y0, y1) in [(5000, 5021), (5021, 5064)]:
            r.render_band(w, h, y0, y1, bands_buf.data_ptr() + (y0 - 5000) * w * 3, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert np.array_equal(bands_buf.cpu().numpy().reshape(64, w, 3), frame[5000:5064])
    assert frame.std() > 1.0


# ---- optional forms of both back ends: same bytes as the default forms ------------------------------
def test_interpreter_row_uniform_form(monkeypatch):
    """MARAY_INTERP_UNIFORM=1: y-only values in per-block words.  Whole frames against the default form
    and oracle rows, on widths where every block lies inside one row (and one where it does not, which
    must fall back to the per-pixel form)."""
    cases = [(scenes.chess_1k(), 1024, 1024, [512, 700], False), (scenes.sdf(2048, 96, 24, seed=6), 2048, 96, [0, 95], True),
             (scenes.sdf(333, 77, 5, seed=8), 333, 77, [3], True)]
    for scene, w, h, rows, exact in cases:
        with _renderer(scene, "interp") as r:
            base = r.render(w, h)
        monkeypatch.setenv("MARAY_INTERP_UNIFORM", "1")
        with _renderer(scene, "interp") as r:
            st = r.stats()
            got = r.render(w, h)
        monkeypatch.delenv("MARAY_INTERP_UNIFORM")
        assert st["interp_uniform_slots"] > 0
        assert np.array_equal(got, base)
        want_rows = OracleScene(scene).render_rows(rows, w)
        for i, y in enumerate(rows):
            if exact:
                assert np.array_equal(got[y], want_rows[i])
            else:
                assert (got[y] != want_rows[i]).any(axis=1).sum() <= 1


def test_pipelined_host_render(monkeypatch):
    """Host-bound frames of 4 MiB and more are rendered in row chunks whose device->host copies overlap the
    next chunks (the default; MARAY_PIPELINE=0 is the plain render): same bytes either way, on a frame above
    the threshold and an odd-sized one."""
    for scene, w, h in [(scenes.sdf(), 1920, 1080), (scenes.sdf(1501, 1203, 9, seed=2), 1501, 1203)]:
        with _renderer(scene, "nvrtc") as r:
            monkeypatch.setenv("MARAY_PIPELINE", "0")
            base = r.render(w, h)
            monkeypatch.delenv("MARAY_PIPELINE")
            got = r.render(w, h)
            got2 = r.render(w, h)
        assert np.array_equal(got, base) and np.array_equal(got2, base)
        want_rows = OracleScene(scene).render_rows([0, h // 2, h - 1], w)
        for i, y in enumerate([0, h // 2, h - 1]):
            assert np.array_equal(got[y], want_rows[i])


@pytest.mark.parametrize("backend", BACKENDS)
def test_texture_fetch_at_constant_coordinates_on_device(backend):
    """App(channel, const, const): both coordinates literal (the advisor's round-1 finding for the bytecode)."""
    tex = scenes.synthetic_textures(2, 16)
    x, y = E.x(), E.y()
    t57 = E.app(E.channel(0, 1), E.nat(5), E.nat(7))
    color = [E.add(t57, x), E.mul(E.sin(E.add(E.app(E.channel(1, 2), E.nat(3), E.nat(2)), x)), y),
             E.add(E.mul(t57, y), E.app(E.channel(1, 0), E.nat(15), E.nat(0)))]
    scene = E.to_bytes([24, 6], color)
    want_rgb, want = OracleScene(scene, tex).render_window(0, 24, 0, 6, want_f64=True)
    with _renderer(scene, backend, tex) as r:
        planes, rgb = r.render_window_f64(24, 6, 0, 24, 0, 6)
    assert np.array_equal(rgb, want_rgb)
    assert bits_equal(planes[[0, 2]], want[[0, 2]]).all()                   # channels without sin: exact
    assert (np.abs(planes[1] - want[1]) <= 1e-13 * np.abs(want[1])).all()


def test_auto_backend_first_frame_and_switch(monkeypatch, tmp_path):
    """MARAY_BACKEND_AUTO (time to first frame): with an empty cubin cache the first frame comes from the
    interpreter while NVRTC compiles on another thread; later frames come from the generated kernels.  Same
    bytes throughout, equal to the plain NVRTC render; a second handle finds the cubin in the cache."""
    import time
    scene = scenes.chess_1k()
    with _renderer(scene, "nvrtc") as r:
        want = r.render(1024, 1024)
    monkeypatch.setenv("MARAY_JIT_CACHE", str(tmp_path))
    with CudaRenderer(gpus=1) as r:
        r.load(scene)
        t0 = time.perf_counter()
        r.compile("auto")
        first = r.render(1024, 1024)
        first_s = time.perf_counter() - t0
        st = r.stats()
        assert np.array_equal(first, want)
        assert st["tier_rows_interp"] == 1024 and st["jit_active"] == 0, "the first frame should not have waited for NVRTC"
        assert first_s < 1.5
        deadline = time.perf_counter() + 120
        while not r.stats()["jit_active"] and time.perf_counter() < deadline:
            time.sleep(0.2)
            frame = r.render(1024, 1024)
            assert np.array_equal(frame, want)
        assert r.stats()["jit_active"] == 1
        assert np.array_equal(r.render(1024, 1024), want)
    with CudaRenderer(gpus=1) as r:
        r.load(scene)
        st = r.compile("auto")
        assert st["jit_cache_hit"] == 1 and r.stats()["jit_active"] == 1
        assert np.array_equal(r.render(1024, 1024), want)


def test_frame_shared_between_processes_over_cuda_ipc(tmp_path):
    """One process per GPU without a gather: the first process exports its device frame (CUDA IPC), a second
    process opens it and renders its band straight into that memory.  (Both processes share the one GPU of the
    test box; on the 8-GPU node the stores travel over NVLink -- bench.py --gpus N.)"""
    import subprocess
    import sys
    scene = scenes.sdf(640, 360, 16, seed=2)
    w, h, cut = 640, 360, 131
    scene_path = tmp_path / "s.maray"
    scene_path.write_bytes(scene)
    with _renderer(scene, "nvrtc") as r:
        want = r.render(w, h)
        handle, frame = r.frame_export(w, h)
        r.render_band(w, h, 0, cut, frame, 0)
        r.band_signal(frame, w, h, 0, 1, 0)            # completion counters behind the frame: rank 0's band of step 1
        child = (
            "import sys; sys.path.insert(0, %r)\n"
            "import numpy as np\n"
            "from maray_b200 import CudaRenderer\n"
            "r = CudaRenderer(gpus=1); r.load(open(%r, 'rb').read()); r.compile('nvrtc')\n"
            "p = r.frame_import(bytes.fromhex(%r))\n"
            "r.render_band(%d, %d, %d, %d, p + %d, 0)\n"
            "r.band_signal(p, %d, %d, 1, 1, 0)                           # rank 1's band of step 1 has landed\n"
            "probe = np.zeros(1, np.uint8); r.copy_to_host(p, probe)   # default-stream copy: the band kernel is done\n"
            "r.close()\n" % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), str(scene_path), handle.hex(), w, h, cut, h, cut * w * 3, w, h))
        res = subprocess.run([sys.executable, "-c", child], capture_output=True, text=True, timeout=300)
        assert res.returncode == 0, res.stderr[-2000:]
        r.band_wait(frame, w, h, 2, 1, 0)              # both counters are at 1: returns at once
        got = np.zeros((h, w, 3), dtype=np.uint8)
        r.copy_to_host(frame, got)
        assert np.array_equal(got, want)
        # nobody signals step 2: the wait is bounded, and the next copy reports the time-out
        import time
        t0 = time.perf_counter()
        r.band_wait(frame, w, h, 2, 2, 0)
        with pytest.raises(MarayCudaError, match="timed out"):
            r.copy_to_host(frame, got)
        assert 1.0 < time.perf_counter() - t0 < 10.0
        r.copy_to_host(frame, got)                     # the flag is cleared: the handle stays usable
    assert np.array_equal(got, want)


def test_multi_gpu_in_process_matches_single():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    scene = scenes.chess_1k()
    with _renderer(scene, "nvrtc", gpus=1) as a, _renderer(scene, "nvrtc", gpus=2) as b:
        assert np.array_equal(a.render(1024, 1024), b.render(1024, 1024))


def test_fp64_peak_microbenchmark_is_sane():
    with CudaRenderer(gpus=1) as r:
        nofma, fma = r.fp64_peak(0)
    # nominal: 148 SMs x 64 lanes x <=1.965 GHz = 18.6e12 lane-ops/s
    assert 5e12 < nofma < 25e12 and 5e12 < fma < 25e12


def test_chain_segmentations_render_the_same_frame(monkeypatch):
    """Regression (round 2): the 7-kernel chain of the 20 000-value deep scene, built by the NVRTC 12.8 that PyTorch had
    put into the process, rendered a different image (a miscompiled 2-wide sine helper); the generated text was right
    (CPU-checked) and NVRTC 12.9 builds it correctly.  NVRTC is now linked statically; this pins the frames of three
    segmentations to each other and to the oracle, with torch imported first as in bench.py."""
    import torch  # noqa: F401  (what used to swap the compiler)
    w = h = 512
    scene = scenes.deep(w, h, n_values=20000, seed=1)
    frames, segments = [], []
    for seg in ("6144", "3072", "1536"):
        monkeypatch.setenv("MARAY_JIT_CHAIN_SEGMENT_VALUES", seg)
        with _renderer(scene, "nvrtc") as r:
            segments.append(r.stats()["jit_segments"])
            frames.append(r.render(w, h))
    assert segments[0] >= 3 and segments[0] < segments[1] < segments[2]
    assert np.array_equal(frames[0], frames[1]) and np.array_equal(frames[0], frames[2])
    want_rgb, _ = OracleScene(scene).render_window(100, 132, 200, 208, want_f64=True)
    assert np.abs(frames[1][200:208, 100:132].astype(int) - want_rgb.astype(int)).max() <= 1


def test_code_generation_knobs_render_the_same_frame(monkeypatch):
    """The forms the code generator can take for a transcendental-heavy program (literal or banked constants, segment
    functions instead of a chain, other chain cuts, no boolean logic) must all render the bytes of the default form: the
    class of fault the NVRTC 12.8 miscompile belonged to (DESIGN.md 10.7)."""
    w, h = 384, 256
    scene = scenes.deep(w, h, n_values=12000, seed=2)
    with _renderer(scene, "nvrtc") as r:
        want = r.render(w, h)
    variants = [{"MARAY_JIT_CONST_BANK": "0"},
                {"MARAY_JIT_CHAIN": "0", "MARAY_JIT_SEGMENT_VALUES": "4096"}, {"MARAY_JIT_CHAIN_SEGMENT_VALUES": "2000", "MARAY_JIT_SEGMENT_VALUES": "4096"},
                {"MARAY_JIT_BOOLEAN": "0"}, {"MARAY_JIT_LINEINFO": "0"}, {"MARAY_JIT_CARVEOUT": "-2"}]
    for env in variants:
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        with _renderer(scene, "nvrtc") as r:
            got = r.render(w, h)
        for k in env:
            monkeypatch.delenv(k)
        assert np.array_equal(got, want), env


LAUNCH_SHAPE_VARIANTS = [{"MARAY_JIT_BLOCK": "256"}, {"MARAY_JIT_BLOCK": "640", "MARAY_JIT_MIN_BLOCKS": "1"},
                         {"MARAY_JIT_BLOCK": "128", "MARAY_JIT_MIN_BLOCKS": "5"}]


def test_launch_shapes_render_the_same_frame(monkeypatch):
    """A large straight-line program runs as one 640-thread block per SM by default (DESIGN.md 3.1 "launch shape").
    The frame must not depend on that choice: ragged sizes (the last block is partial, rows straddle blocks), the old
    256 x 2 shape and hand-set shapes render the same bytes, and
    the default form matches the oracle."""
    scene = scenes.chess_1k()
    w, h = 1001, 77                       # 77 077 pixels: not a multiple of 640, 256, 1024 or 128
    with _renderer(scene, "nvrtc") as r:
        st = r.stats()
        auto_block = st["jit_block"]        # 1 024 for this scene (it declares 1024 x 1024: 6.92 rounds), 640 for a 4K frame
        assert auto_block in (640, 768, 1024) and st["jit_registers"] * auto_block <= 65536
        assert st["jit_round_pixels"] % auto_block == 0 and st["jit_round_pixels"] >= 100 * auto_block
        want = r.render(w, h)
        band = np.zeros((20, w, 3), dtype=np.uint8)
        # a band that starts inside a block of the frame's own partition
        import torch
        d = torch.empty(20 * w * 3, dtype=torch.uint8, device="cuda")
        r.render_band(w, h, 31, 51, d.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        band[:] = d.cpu().numpy().reshape(20, w, 3)
    assert np.array_equal(band, want[31:51])
    want_rgb, _ = OracleScene(scene).render_window(0, w, 40, 44, want_f64=True)
    assert np.array_equal(want[40:44], want_rgb)
    for env in LAUNCH_SHAPE_VARIANTS:
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        with _renderer(scene, "nvrtc") as r:
            assert r.stats()["jit_block"] == int(env.get("MARAY_JIT_BLOCK", auto_block))
            got = r.render(w, h)
        for k in env:
            monkeypatch.delenv(k)
        assert np.array_equal(got, want), env
