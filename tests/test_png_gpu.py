"""PNG encoding on the GPU (maray_cuda_render_png) and its CPU twin.

The twin (maray_cuda_png_encode_host) runs the encoder's per-position, per-token and per-segment functions serially;
its files are checked here with zlib, a numpy unfilter and a small inflate that reads the deflate tokens.  On the GPU
the file must decode to the rendered frame and be byte-identical to the twin's file for that frame."""
import ctypes
import io
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

from maray_b200 import CudaRenderer, Report, _lib, scenes
from maray_b200 import expr as E

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "maray_b200", "maray_cuda")
IDAT_BYTES = 1 << 30


# ---- the twin ---------------------------------------------------------------------------------------------------
def twin(img, idat_bytes=IDAT_BYTES):
    """(file bytes, segments, stored segments) of the CPU twin for an (h, w, 3) uint8 frame."""
    L = _lib.load()
    fn = L.maray_cuda_png_encode_host
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_size_t,
                   ctypes.POINTER(ctypes.c_size_t), ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_uint32)]
    img = np.ascontiguousarray(img, dtype=np.uint8)
    h, w = img.shape[:2]
    n = h * (3 * w + 1)
    cap = 2 * n + 12 * (n // idat_bytes + 2) + 4096
    out = np.zeros(cap, np.uint8)
    ln, segs, stored = ctypes.c_size_t(), ctypes.c_uint32(), ctypes.c_uint32()
    rc = fn(img.ctypes.data, w, h, idat_bytes, out.ctypes.data, cap, ctypes.byref(ln), ctypes.byref(segs), ctypes.byref(stored))
    assert rc == _lib.OK
    return out[:ln.value].tobytes(), segs.value, stored.value


# ---- reading a PNG ----------------------------------------------------------------------------------------------
def chunks(png):
    """[(type, data)], every CRC checked."""
    assert png[:8] == b"\x89PNG\r\n\x1a\n"
    pos, out = 8, []
    while pos < len(png):
        n, t = struct.unpack(">I4s", png[pos:pos + 8])
        d = png[pos + 8:pos + 8 + n]
        assert struct.unpack(">I", png[pos + 8 + n:pos + 12 + n])[0] == zlib.crc32(t + d), f"bad CRC of {t}"
        out.append((t, d))
        pos += 12 + n
    assert pos == len(png)
    return out


def unfilter(raw, w, h):
    stride = 3 * w
    rows = np.frombuffer(raw, np.uint8).reshape(h, stride + 1)
    out = np.zeros((h, stride), np.uint8)
    prev = np.zeros(stride, np.int32)
    for y in range(h):
        ft, x = rows[y, 0], rows[y, 1:].astype(np.int32)
        if ft == 0:
            cur = x
        elif ft == 2:
            cur = (x + prev) & 255
        else:   # Sub, Average, Paeth depend on the left neighbour: byte by byte
            cur = np.zeros(stride, np.int32)
            for i in range(stride):
                a = cur[i - 3] if i >= 3 else 0
                b = prev[i]
                c = prev[i - 3] if i >= 3 else 0
                if ft == 1:
                    p = a
                elif ft == 3:
                    p = (a + b) // 2
                else:
                    q = a + b - c
                    pa, pb, pc = abs(q - a), abs(q - b), abs(q - c)
                    p = a if pa <= pb and pa <= pc else (b if pb <= pc else c)
                cur[i] = (x[i] + p) & 255
        out[y] = cur
        prev = cur.astype(np.int32)
    return out.reshape(h, w, 3)


def decode(png):
    """(frame, zlib stream, IDAT count): IHDR fields, FCHECK and CRCs checked."""
    cs = chunks(png)
    assert cs[0][0] == b"IHDR" and cs[-1] == (b"IEND", b"")
    w, h, depth, ctype, comp, filt, interlace = struct.unpack(">IIBBBBB", cs[0][1])
    assert (depth, ctype, comp, filt, interlace) == (8, 2, 0, 0, 0)
    idats = [d for t, d in cs if t == b"IDAT"]
    assert len(idats) == len(cs) - 2 and all(0 < len(d) < 2 ** 31 for d in idats)
    z = b"".join(idats)
    assert z[0] == 0x78 and (z[0] * 256 + z[1]) % 31 == 0
    return unfilter(zlib.decompress(z), w, h), z, len(idats)


class Bits:
    def __init__(self, data):
        self.v = int.from_bytes(data, "little")
        self.pos = 0

    def get(self, n):
        r = (self.v >> self.pos) & ((1 << n) - 1)
        self.pos += n
        return r


def _decoder(lens):
    count = [0] * 16
    for l in lens:
        if l:
            count[l] += 1
    code, nxt = 0, [0] * 16
    for b in range(1, 16):
        code = (code + count[b - 1]) << 1
        nxt[b] = code
    table = {}
    for s, l in enumerate(lens):
        if l:
            table[(l, nxt[l])] = s
            nxt[l] += 1
    return table


def _sym(bits, table):
    code, l = 0, 0
    while True:
        code = (code << 1) | bits.get(1)
        l += 1
        if (l, code) in table:
            return table[(l, code)]
        assert l < 16


LBASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
DBASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
         6145, 8193, 12289, 16385, 24577]
DEXTRA = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]
ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]


def blocks(z):
    """The deflate blocks of a zlib stream: [{"type", "final", "matches": [(length, distance)], "max_code"}]."""
    bits = Bits(z[2:-4])
    out = []
    while True:
        final, btype = bits.get(1), bits.get(2)
        blk = {"type": btype, "final": final, "matches": [], "max_code": 0}
        out.append(blk)
        if btype == 0:
            bits.pos = (bits.pos + 7) & ~7
            n, nn = bits.get(16), bits.get(16)
            assert n ^ nn == 0xFFFF
            bits.pos += 8 * n
        else:
            assert btype == 2, "the encoder writes dynamic and stored blocks only"
            hlit, hdist, hclen = bits.get(5) + 257, bits.get(5) + 1, bits.get(4) + 4
            cl = [0] * 19
            for i in range(hclen):
                cl[ORDER[i]] = bits.get(3)
            assert max(cl) <= 7
            clt, lens = _decoder(cl), []
            while len(lens) < hlit + hdist:
                s = _sym(bits, clt)
                if s < 16:
                    lens.append(s)
                elif s == 16:
                    lens += [lens[-1]] * (3 + bits.get(2))
                elif s == 17:
                    lens += [0] * (3 + bits.get(3))
                else:
                    lens += [0] * (11 + bits.get(7))
            blk["max_code"] = max(lens)
            lt, dt = _decoder(lens[:hlit]), _decoder(lens[hlit:])
            while True:
                s = _sym(bits, lt)
                if s == 256:
                    break
                if s > 256:
                    ln = LBASE[s - 257] + bits.get(LEXTRA[s - 257])
                    d = _sym(bits, dt)
                    blk["matches"].append((ln, DBASE[d] + bits.get(DEXTRA[d])))
        if final:
            return out


def check(img, idat_bytes=IDAT_BYTES):
    png, segs, stored = twin(img, idat_bytes)
    got, z, n_idat = decode(png)
    assert np.array_equal(got, np.asarray(img, np.uint8))
    return png, segs, stored, z, n_idat


# ---- CPU --------------------------------------------------------------------------------------------------------
def test_noise_goes_through_stored_blocks():
    img = np.random.default_rng(1).integers(0, 256, (300, 257, 3), dtype=np.uint8)
    png, segs, stored, z, _ = check(img)
    assert segs > 1 and stored == segs
    assert {b["type"] for b in blocks(z)} == {0}


def test_constant_frame_is_runs_of_258():
    img = np.full((64, 500, 3), 200, np.uint8)
    png, segs, stored, z, _ = check(img)
    assert stored == 0
    lengths = [m[0] for b in blocks(z) for m in b["matches"]]
    # rows of 1501 bytes, each one filter byte and zeros (Up): five or six matches per row, most of them 258 long
    assert lengths.count(258) > len(lengths) // 2 and len(png) < 2000


def test_matches_exactly_32768_back():
    """Rows of 3w+1 = 16384 bytes repeating A B A B A B, one row per segment: a row with the same row above as the row
    two before has the same filtered bytes, and can only match them, 32768 bytes back."""
    rng = np.random.default_rng(2)
    a, b = rng.integers(0, 256, (2, 1, 5461, 3), dtype=np.uint8)
    img = np.concatenate([a, b] * 3)
    png, segs, stored, z, _ = check(img)
    assert segs == 6 and stored == 3   # rows 0, 1, 2; rows 3 (same row above as row 1), 4 and 5 match
    dists = [m[1] for blk in blocks(z) for m in blk["matches"]]
    assert dists and max(dists) == 32768 and sum(m[0] for blk in blocks(z) for m in blk["matches"]) > 32000


@pytest.mark.parametrize("w,h", [(1, 1), (1, 700), (700, 1), (2, 3)])
def test_tiny_frames(w, h):
    img = np.random.default_rng(w * 1000 + h).integers(0, 256, (h, w, 3), dtype=np.uint8)
    check(img)


@pytest.mark.parametrize("w", [5, 1365, 1366, 5462])
def test_rows_straddle_segment_boundaries(w):
    """3w+1 does not divide the segment size: rows start anywhere in a segment."""
    rng = np.random.default_rng(w)
    h = max(40, 40000 // w)
    y, x = np.mgrid[0:h, 0:w]
    img = np.stack([(x * 3 + y) & 255, (x * y) & 255, rng.integers(0, 4, (h, w))], axis=2).astype(np.uint8)
    png, segs, _, _, _ = check(img)
    assert segs >= 2


def test_many_segments_with_matches_across_boundaries():
    tile = np.random.default_rng(3).integers(0, 256, (1, 97, 3), dtype=np.uint8)
    img = np.tile(tile, (400, 40, 1))
    png, segs, stored, z, _ = check(img)
    bl = blocks(z)
    assert segs >= 20 and stored == 0 and len(bl) == 2 * segs - 1   # a coded block + an empty stored block, last: one
    assert all(b["matches"] for b in bl if b["type"] == 2)
    assert len(png) < img.size // 50


def first_block_code_lengths(z):
    """The lit/len and distance code lengths declared by the first (dynamic) block of a zlib stream."""
    bits = Bits(z[2:4098])
    assert bits.get(1) == 0 and bits.get(2) == 2
    hlit, hdist, hclen = bits.get(5) + 257, bits.get(5) + 1, bits.get(4) + 4
    cl = [0] * 19
    for i in range(hclen):
        cl[ORDER[i]] = bits.get(3)
    clt, lens = _decoder(cl), []
    while len(lens) < hlit + hdist:
        s = _sym(bits, clt)
        if s < 16:
            lens.append(s)
        elif s == 16:
            lens += [lens[-1]] * (3 + bits.get(2))
        else:
            lens += [0] * ((3 + bits.get(3)) if s == 17 else (11 + bits.get(7)))
    return lens


def test_skewed_histogram_stays_within_15_bits():
    """17 byte values with counts 2^16 .. 1 fill the first 128 KiB segment (row 0, filter None because the values sit
    next to 0).  Matches take part of the frequent values, so the code need not reach 15 bits; it must stay within."""
    k = 17
    near0 = [0] + [(j + 1) // 2 if j % 2 else 256 - j // 2 for j in range(1, k)]
    vals = np.concatenate([np.full(2 ** (k - 1 - j), near0[j], np.uint8) for j in range(k)])
    np.random.default_rng(4).shuffle(vals)
    img = np.zeros((313, (len(vals) + 2) // 3, 3), np.uint8)
    img[0].reshape(-1)[:len(vals)] = vals
    png, segs, stored = twin(img)
    z = b"".join(d for t, d in chunks(png) if t == b"IDAT")
    assert 13 <= max(first_block_code_lengths(z)) <= 15
    got = zlib.decompress(z)
    assert got[0] == 0 and got[1:1 + len(vals)] == vals.tobytes()


def test_several_idat_chunks():
    img = np.random.default_rng(5).integers(0, 16, (60, 301, 3), dtype=np.uint8)
    png, _, _, _, n_idat = check(img, idat_bytes=1000)
    assert n_idat > 5
    one, _, _ = twin(img)
    assert decode(one)[0].tobytes() == decode(png)[0].tobytes()


def test_render_png_refuses_what_png_cannot_hold():
    r = CudaRenderer(gpus=0)
    r.load(E.to_bytes([4, 4], [E.x(), E.y(), E.nat(0)]))
    r.compile("nvrtc")
    p, n = ctypes.c_void_p(), ctypes.c_size_t()
    L = _lib.load()
    assert L.maray_cuda_render_png(r._h, 2 ** 31, 1, None, ctypes.byref(p), ctypes.byref(n), None, None) == _lib.E_INVALID
    assert L.maray_cuda_render_png(r._h, 4, 4, None, None, ctypes.byref(n), None, None) == _lib.E_INVALID
    assert L.maray_cuda_render_png(r._h, 4, 4, None, ctypes.byref(p), ctypes.byref(n), None, None) == _lib.E_CUDA
    r.close()


# ---- GPU --------------------------------------------------------------------------------------------------------
def level6_bytes(img):
    """What the host writer (filter None, zlib level 6) produces for this frame."""
    h, w = img.shape[:2]
    raw = np.concatenate([np.zeros((h, 1), np.uint8), img.reshape(h, 3 * w)], axis=1).tobytes()
    return 8 + 25 + 12 + len(zlib.compress(raw, 6)) + 12


def renderer(scene, textures=(), backend="nvrtc", samples=1, gpus=1, custom=False):
    r = CudaRenderer(gpus=gpus)
    if custom:
        r.set_functions(scenes.TEXTURE_RUNTIME_SOURCE, 5 * len(textures))
        r.set_context(scenes.pack_textures(textures))
    else:
        r.set_textures(list(textures))
    r.load(scene)
    r.compile(backend)
    r.set_samples(samples)
    return r


def assert_png_of(r, w, h):
    png, st, ps = r.render_png(w, h)
    frame = r.render(w, h)
    got, _, _ = decode(png)
    assert np.array_equal(got, frame)
    from PIL import Image
    assert np.array_equal(np.array(Image.open(io.BytesIO(png)).convert("RGB")), frame)
    assert png == twin(frame)[0], "GPU file differs from the CPU twin's"
    assert ps["png_bytes"] == len(png) and ps["scanline_bytes"] == h * (3 * w + 1) and ps["encode_ms"] > 0
    return png, ps, frame


SMALL_TEX = None


def small_textures():
    global SMALL_TEX
    if SMALL_TEX is None:
        SMALL_TEX = scenes.synthetic_textures(2, 256)
    return SMALL_TEX


CASES = {
    "sdf": lambda: (scenes.sdf(640, 360, n_circles=16, seed=3), (), (640, 360)),
    "textured": lambda: (scenes.textured(640, 360, n_tex=2), small_textures(), (640, 360)),
    "chess_1k": lambda: (scenes.chess_1k(), (), (1024, 1024)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["nvrtc", "interp", "auto"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_render_png_decodes_to_the_frame(name, backend):
    scene, tex, (w, h) = CASES[name]()
    r = renderer(scene, tex, backend)
    png, ps, frame = assert_png_of(r, w, h)
    assert r.render_png(w, h)[0] == png, "two calls give different files"
    r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["chess_1k", "sdf", "textured"])
def test_png_bytes_against_the_host_writer(name):
    """The workloads at their benchmark sizes: at most 1.5x what write_png_rgb8 (filter None, level 6) writes."""
    from PIL import Image
    scene, tex, (w, h) = scenes.by_name(name)
    r = renderer(scene, tex)
    img = np.zeros((h, w, 3), np.uint8)
    png, _, ps = r.render_png(img=img)
    r.close()
    assert np.array_equal(np.array(Image.open(io.BytesIO(png)).convert("RGB")), img)
    assert len(png) <= 1.5 * level6_bytes(img), (len(png), level6_bytes(img))


@pytest.mark.gpu
def test_backends_and_samples_give_the_same_file():
    scene, tex, (w, h) = CASES["sdf"]()
    files = {}
    for backend in ("nvrtc", "interp"):
        r = renderer(scene, tex, backend, samples=2)
        files[backend] = assert_png_of(r, w, h)[0]
        r.close()
    assert files["nvrtc"] == files["interp"]


@pytest.mark.gpu
def test_custom_runtime_frame():
    scene, tex, (w, h) = CASES["textured"]()
    r = renderer(scene, tex, "nvrtc", custom=True)
    png, _, frame = assert_png_of(r, w, h)
    r2 = renderer(scene, tex, "nvrtc")
    assert r2.render_png(w, h)[0] == png
    r.close(); r2.close()


@pytest.mark.gpu
def test_noise_texture_goes_through_stored_blocks_on_the_device():
    noise = np.random.default_rng(7).integers(0, 256, (2048, 2048, 3), dtype=np.uint8)
    x, y = E.x(), E.y()
    scene = E.to_bytes([2048, 2048], [E.app(E.channel(0, c), x, y) for c in range(3)])
    r = renderer(scene, [noise])
    png, ps, frame = assert_png_of(r, 2048, 2048)
    assert np.array_equal(frame, noise)
    assert ps["stored_segments"] == ps["segments"] > 1
    r.close()


@pytest.mark.gpu
def test_host_image_and_progress_as_render():
    scene, tex, (w, h) = CASES["sdf"]()
    r = renderer(scene, tex)
    calls = []
    r.set_report(Report.row(64), lambda img, p: calls.append(p))
    img = np.zeros((h, w, 3), np.uint8)
    png, _, _ = r.render_png(img=img)
    assert calls and all(0 < p < 1 for p in calls)
    assert np.array_equal(decode(png)[0], img)
    n = len(calls)
    want = np.zeros_like(img)
    r.render_into(want)
    assert len(calls) == 2 * n and np.array_equal(img, want)
    r.close()


@pytest.mark.gpu
def test_one_and_two_gpus_give_the_same_file():
    try:
        r2 = renderer(scenes.chess_1k(), (), gpus=2)
    except Exception:
        pytest.skip("needs two GPUs")
    r1 = renderer(scenes.chess_1k(), ())
    img = np.zeros((1024, 1024, 3), np.uint8)
    a = r2.render_png(img=img)[0]
    assert a == r1.render_png(1024, 1024)[0] and np.array_equal(decode(a)[0], img)
    r1.close(); r2.close()


@pytest.mark.gpu
def test_cli_file_decodes_to_the_oracle_frame(tmp_path):
    from PIL import Image
    scene = tmp_path / "chess.maray"
    scene.write_bytes(scenes.chess_1k())
    out = tmp_path / "chess.png"
    r = subprocess.run([CLI, "-i", str(scene), "-o", str(out)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = decode(out.read_bytes())[0]
    want = np.array(Image.open(os.path.join(ROOT, "tests", "golden", "chess_oracle_1024.png")).convert("RGB"))
    assert got.shape == want.shape
    assert int((got != want).any(axis=2).sum()) <= got.shape[0] * got.shape[1] // 10000
