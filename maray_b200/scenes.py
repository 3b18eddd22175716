"""The benchmark / parity scenes of BASELINE.json `configs`, made concrete as in SURVEY.md section 8(d).

Every generator returns `.maray` bytes (current layout) plus, where needed, its textures; all are
deterministic (seeded 64-bit LCG, no use of Python's `random`).  These are inputs only -- nothing
here evaluates an expression.

  config 1  chess_1k()        data/chess.maray as shipped (legacy layout, 1024x1024)
  config 2  sdf(1920, 1080)   64 circles via sqrt/min/max/step/abs/recip, no transcendentals
  config 3  chess_4k()        the shipped chess DAG resampled to 3840x2160 (documented stand-in)
            chess_dsl(w, h)   examples/chess.rs re-run through the builder (no simplify/compress)
  config 4  textured(...)     4 synthetic 2048x2048 textures sampled through `app`
  config 5  deep(...)         seeded random DAG, ~1e5 values, sin/exp/ln heavy
"""
from __future__ import annotations

import os
import struct
from typing import List, Sequence, Tuple

import numpy as np

from . import expr as E

_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data")


class Lcg:
    """Knuth's MMIX 64-bit LCG; the high 32 bits are the output."""

    def __init__(self, seed: int):
        self.s = (seed * 0x9E3779B97F4A7C15 + 1) & 0xFFFFFFFFFFFFFFFF

    def next(self) -> int:
        self.s = (self.s * 6364136223846793005 + 1442695040888963407) & 0xFFFFFFFFFFFFFFFF
        return self.s >> 32

    def below(self, n: int) -> int:
        return self.next() % n

    def between(self, lo: int, hi: int) -> int:
        """inclusive"""
        return lo + self.below(hi - lo + 1)


# ---- config 1 -------------------------------------------------------------------------------------
def chess_1k() -> bytes:
    """The reference's shipped scene, byte for byte (data/chess.maray; sha256 b1ad82f4...baaba4): a bench
    and test INPUT owned by the package (maray_b200/data/), not an oracle."""
    with open(os.path.join(_DATA, "chess.maray"), "rb") as f:
        return f.read()


# ---- config 2 -------------------------------------------------------------------------------------
def sdf(w: int = 1920, h: int = 1080, n_circles: int = 64, seed: int = 1) -> bytes:
    """2-D signed-distance scene restricted to + * neg 1/ sqrt abs min max step (bit-exact class).

    Circle i: d_i = Sd2::Circle{r}.to_expr().translate([cx, cy])  (reference src/sd.rs:32,
    src/lib.rs:799-801), i.e. sqrt((x + -cx)^2 + (y + -cy)^2) + -r with integer cx, cy, r.
    Two halves are unioned with `min`; the halves are intersected with `max`.
      R = step(-d_union) * 255                      (Sd2::inside, reference src/sd.rs:51-53)
      G = max(16, min(255, |d_union| * 3))          (distance bands)
      B = 255 * 1/(1 + |d_intersection|)            (one reciprocal per pixel)
    Three different Let-free channels.
    """
    rng = Lcg(seed)
    ds = []
    for _ in range(n_circles):
        cx, cy, r = rng.below(w), rng.below(h), rng.between(20, 200)
        ds.append(E.sd_circle(E.nat(r)).translate([E.nat(cx), E.nat(cy)]))
    half = max(1, n_circles // 2)

    def fold(fn, items):
        acc = items[0]
        for it in items[1:]:
            acc = fn(acc, it)
        return acc

    d_a, d_b = fold(E.min, ds[:half]), fold(E.min, ds[half:] or ds[:1])
    d_union, d_inter = E.min(d_a, d_b), E.max(d_a, d_b)
    r_ch = E.mul(E.sd_inside(d_union), E.nat(255))
    g_ch = E.max(E.nat(16), E.min(E.nat(255), E.mul(E.abs(d_union), E.nat(3))))
    b_ch = E.mul(E.nat(255), E.recip(E.add(E.nat(1), E.abs(d_inter))))
    return E.to_bytes([w, h], [r_ch, g_ch, b_ch])


# ---- config 3 -------------------------------------------------------------------------------------
def chess_resampled(w: int, h: int) -> bytes:
    """The shipped chess DAG with x -> x*(1024/w), y -> y*(1024/h) substituted everywhere (also inside
    the Let definitions).  SURVEY.md 8(d) config 3 names this the acceptable stand-in for
    "regenerated from examples/chess.rs at 3840x2160" until simplify+compress are restated."""
    size, color, _legacy = E.from_bytes(chess_1k())
    sx = E.mul(E.x(), E.mul(E.nat(size[0]), E.recip(E.nat(w))))
    sy = E.mul(E.y(), E.mul(E.nat(size[1]), E.recip(E.nat(h))))
    return E.to_bytes([w, h], E.map_xy(color, sx, sy))


def chess_4k() -> bytes:
    return chess_resampled(3840, 2160)


def chess_shape(w: int = 1024, h: int = 1024, cells: int = 8) -> E.Expr:
    """The `shape` expression of examples/chess.rs at size [w, h], as built by lines 8-39 of that file
    (before `simplify`/`compress`)."""
    fx, fy = E.div(E.x(), E.nat(w)), E.div(E.y(), E.nat(h))
    p = [fx, fy]
    texture = E.set_unit_square(E.chess(8))
    p1 = [E.recip(E.nat(5)), E.recip(E.nat(2))]
    p2 = [E.sub(E.nat(1), E.recip(E.nat(5))), E.recip(E.nat(2))]
    p3 = [E.nat(0), E.sub(E.nat(1), E.recip(E.nat(5)))]
    p4 = [E.nat(1), E.sub(E.nat(1), E.recip(E.nat(5)))]
    shape = E.nat(0)
    xy = [E.x(), E.y()]
    for i in range(cells):
        for j in range(cells):
            quad, uv = E.grid_cell([cells, cells], [i, j], [p1, p2, p3, p4])
            (tri, uv1), (tri2, uv2) = E.quad_to_tri(quad, uv)
            get_uv = texture.subst2(E.to_uv(tri, uv1, xy))
            shape1 = E.mul(E.inside_triangle(tri, xy), get_uv).subst2(p)
            get_uv2 = texture.subst2(E.to_uv(tri2, uv2, xy))
            shape2 = E.mul(E.inside_triangle(tri2, xy), get_uv2).subst2(p)
            shape = E.set_or(shape, E.set_or(shape1, shape2))
    return shape


def chess_dsl(w: int = 1024, h: int = 1024, cells: int = 8) -> bytes:
    """examples/chess.rs re-run through the builder at size [w, h] (reference examples/chess.rs:5-50),
    WITHOUT `simplify`/`compress`: HEAD's `simplify` does not terminate on this scene
    (maray_b200/simplify.py `SimplifyDiverges`, tests/test_simplify.py), so the shipped file cannot be
    regenerated from HEAD; sharing is put on the wire with `share_let`."""
    ch = E.mul(chess_shape(w, h, cells), E.nat(255))
    return E.to_bytes([w, h], E.share_let([ch, ch, ch]))


# ---- config 4 -------------------------------------------------------------------------------------
def synthetic_textures(n: int = 4, size: int = 2048) -> List[np.ndarray]:
    """texel (x, y, c) of texture t = (x*7 + y*13 + c*31 + t*101 + ((x ^ y) & 0xFF)) & 0xFF."""
    ys, xs = np.meshgrid(np.arange(size, dtype=np.uint32), np.arange(size, dtype=np.uint32), indexing="ij")
    out = []
    for t in range(n):
        img = np.empty((size, size, 3), dtype=np.uint8)
        for c in range(3):
            img[:, :, c] = ((xs * 7 + ys * 13 + c * 31 + t * 101 + ((xs ^ ys) & 0xFF)) & 0xFF).astype(np.uint8)
        out.append(img)
    return out


def textured(w: int = 3840, h: int = 2160, n_tex: int = 4) -> bytes:
    """Per channel c: mean over t of app(channel(t,c), u_t, v_t).

    (u_t, v_t) = rotate_t(x, y) * W_t / w + offset_t, with W_t = app(image_width(t), 0, 0) and
    H_t = app(image_height(t), 0, 0) (reference src/textures.rs:17-23).  Rotations use Pythagorean
    triples so every coefficient is an exact small rational; offsets push part of each footprint
    below 0 and beyond the texture edge to exercise the zero-return branches
    (reference src/textures.rs:30,34)."""
    rots = [(1, 0, 1), (4, 3, 5), (12, 5, 13), (15, 8, 17)]          # (cos*d, sin*d, d)
    offs = [(0, 0), (-300, 200), (150, -400), (-700, -100)]
    x, y = E.x(), E.y()
    zero = E.nat(0)
    chans = []
    for c in range(3):
        acc = None
        for t in range(n_tex):
            ca, sa, d = rots[t % len(rots)]
            ox, oy = offs[t % len(offs)]
            wt = E.app(E.image_width(t), zero, zero)
            ht = E.app(E.image_height(t), zero, zero)
            rx = E.div(E.sub(E.mul(E.nat(ca), x), E.mul(E.nat(sa), y)), E.nat(d))
            ry = E.div(E.add(E.mul(E.nat(sa), x), E.mul(E.nat(ca), y)), E.nat(d))
            off_x = E.nat(ox) if ox >= 0 else E.neg(E.nat(-ox))
            off_y = E.nat(oy) if oy >= 0 else E.neg(E.nat(-oy))
            u = E.add(E.div(E.mul(rx, wt), E.nat(w)), off_x)
            v = E.add(E.div(E.mul(ry, ht), E.nat(w)), off_y)
            s = E.app(E.channel(t, c), u, v)
            acc = s if acc is None else E.add(acc, s)
        chans.append(E.div(acc, E.nat(n_tex)))
    return E.to_bytes([w, h], E.share_let(chans))


# ---- config 5 -------------------------------------------------------------------------------------
def deep(w: int = 8192, h: int = 8192, n_values: int = 100_000, seed: int = 5, window: int = 192) -> bytes:
    """Seeded random DAG of about `n_values` non-constant values, >= 30 % of them sin/exp/ln.

    Leaves u = x/w, v = y/h and 16 "phase fields" L_i = a_i*u + b_i*v + c_j (4 directions x 4 offsets, shared by
    the whole program -- and live through all of it, which is why there are not more of them).  Every new value combines one or two
    earlier values p, q taken from a sliding window (so the DAG is deep, and the number of simultaneously
    live values stays near `window`):
        sin(k*p + L_i)              k  in {1/8 .. 8/8}
        sin(k1*p + k2*q + L_i)      k1, k2 in {1/16 .. 8/16}
        exp(-(p*p))    ln(1 + p*p)    p*q    (p+q)/2
    All of them map [-1,1] into [-1,1], and -- the point of this generator -- none of them EXPANDS: the
    derivative with respect to an earlier value is at most 1 in magnitude (|k| <= 1, k1 + k2 <= 1,
    |2p exp(-p^2)| <= 0.86, |2p/(1+p^2)| <= 1), so a last-bit difference in one sin/exp/ln result stays a
    last-bit difference thousands of levels later.  (Round 1's generator used sin(k*p + c) with k up to 4.5: its
    values double their sensitivity every few levels, at 1e5 values a 1-ULP nudge of the libm results moves the
    channels by whole grey levels, and no two libms -- glibc versions included -- agree on such an image; see
    tests/test_host_lowering.py::test_deep_scene_is_well_conditioned.)  Position enters every sine through L_i,
    so deep values still vary over the image.
    Values nobody consumed by the time they leave the window are added to one of three running channel sums;
    channel = 127.5 + 127.5 * clamp(sin(40 * mean), -1, 1) via min/max (the mean of thousands of values varies
    little; the sine spreads it over the grey range without saturating).
    """
    rng = Lcg(seed)
    u, v = E.div(E.x(), E.nat(w)), E.div(E.y(), E.nat(h))

    def rat(lo: int, hi: int, den: int) -> E.Expr:
        n = rng.between(lo, hi)
        return E.div(E.nat(n), E.nat(den)) if n >= 0 else E.neg(E.div(E.nat(-n), E.nat(den)))

    dirs = [E.add(E.mul(rat(1, 40, 1), u), E.mul(rat(1, 40, 1), v)) for _ in range(4)]
    offs = [rat(0, 628, 100) for _ in range(4)]
    phases = [E.add(d, c) for d in dirs for c in offs]
    pool: List[E.Expr] = []
    uses: List[int] = []
    count = 4 * 3 + 16
    for _ in range(16):
        f = E.sin(E.add(E.add(E.mul(rat(1, 40, 1), u), E.mul(rat(1, 40, 1), v)), rat(0, 628, 100)))
        pool.append(f); uses.append(0); count += 6

    def pick() -> int:
        lo = max(0, len(pool) - window)
        # prefer values nobody has consumed yet, so (almost) everything stays reachable
        for _try in range(4):
            i = lo + rng.below(len(pool) - lo)
            if uses[i] == 0:
                return i
        return lo + rng.below(len(pool) - lo)

    sums: List = [None, None, None]      # running per-channel sums of the values nobody consumed
    n_summed = [0, 0, 0]
    retired = 0                          # pool[:retired] has left the window

    named: List[E.Expr] = []             # the running sums are bound to Let variables where they arise

    def fold(val: E.Expr) -> None:
        c = sum(n_summed) % 3
        sums[c] = val if sums[c] is None else E.add(sums[c], val)
        n_summed[c] += 1
        named.append(sums[c])

    while count < n_values:
        kind = rng.below(100)
        i = pick(); p = pool[i]; uses[i] += 1
        if kind < 32:
            ph = phases[rng.below(len(phases))]
            nv = E.sin(E.add(E.mul(rat(1, 8, 8), p), ph)); count += 3
        elif kind < 58:
            nv = E.exp(E.neg(E.mul(p, p))); count += 3
        elif kind < 84:
            nv = E.ln(E.add(E.nat(1), E.mul(p, p))); count += 3
        elif kind < 92:
            j = pick(); q = pool[j]; uses[j] += 1
            ph = phases[rng.below(len(phases))]
            nv = E.sin(E.add(E.add(E.mul(rat(1, 8, 16), p), E.mul(rat(1, 8, 16), q)), ph)); count += 5
        elif kind < 96:
            j = pick(); q = pool[j]; uses[j] += 1
            nv = E.mul(p, q); count += 1
        else:
            j = pick(); q = pool[j]; uses[j] += 1
            nv = E.mul(E.add(p, q), E.half()); count += 2
        pool.append(nv); uses.append(0)
        # values that leave the window unconsumed join a channel sum right away (keeps few values live)
        while retired < len(pool) - window:
            if uses[retired] == 0:
                fold(pool[retired]); count += 1
            retired += 1
    for i in range(retired, len(pool)):
        if uses[i] == 0:
            fold(pool[i])
    chans = []
    for c in range(3):
        acc = sums[c] if sums[c] is not None else pool[-1 - c]
        mean = E.div(acc, E.nat(max(1, n_summed[c])))
        cl = E.max(E.neg(E.nat(1)), E.min(E.nat(1), E.sin(E.mul(E.nat(40), mean))))
        half255 = E.div(E.nat(255), E.nat(2))
        chans.append(E.add(half255, E.mul(half255, cl)))
    return E.to_bytes([w, h], E.share_let(chans, bind=named))


# ---- the reference's example programs, re-run through the restated tooling -------------------------
def example_test_rs() -> bytes:
    """examples/test.rs:7-31: a rounded box XOR a circle at 512x512, `simplify` then `compressor::compress`,
    every channel `shape * 255` -- built with the DSL mirror and the restated simplify/compress."""
    from . import compress as C
    from . import simplify as S

    size = [512, 512]
    p = [E.div(E.x(), E.nat(size[0])), E.div(E.y(), E.nat(size[1]))]
    center = [E.half(), E.half()]
    tenth = E.div(E.nat(1), E.nat(10))
    box = E.sd_inside(E.sd_rounded_box([E.div(E.half(), E.nat(2)), E.half()], E.p4_same(tenth))).translate(center)
    circle = E.sd_inside(E.sd_circle(E.recip(E.nat(3)))).translate(center)
    shape = C.compress(S.simplify(E.set_xor(box, circle).subst2(p)))
    ch = E.mul(shape, E.nat(255))
    return E.to_bytes(size, [ch, ch, ch])


def example_test6_rs() -> bytes:
    """examples/test6.rs: the three channels of texture 0, the blue one flipped with `nat(1024) - y()`."""
    color = [E.app(E.channel(0, 0), E.x(), E.y()), E.app(E.channel(0, 1), E.x(), E.y()),
             E.app(E.channel(0, 2), E.x(), E.nat(1024) - E.y())]
    return E.to_bytes([1024, 1024], color)


def example_test7_rs() -> bytes:
    """examples/test7.rs: `nat(255) * x() / nat(128)` on every channel, 128x128."""
    e = E.nat(255) * E.x() / E.nat(128)
    return E.to_bytes([128, 128], [e, e, e])


# The default texture runtime (reference src/textures.rs:27-50) restated as a custom runtime (maray_cuda_set_functions):
# the context packs the images as a u32 count, then (w u32, h u32, byte offset u64) per image, then the RGB8 data.
TEXTURE_RUNTIME_SOURCE = r"""
__device__ double maray_app(const unsigned char* ctx, unsigned long long ctx_bytes, unsigned int id, double a, double b) {
    const unsigned int img = id / 5u, k = id % 5u;
    const unsigned char* e = ctx + 8u + 16u * img;
    const unsigned int w = *reinterpret_cast<const unsigned int*>(e);
    const unsigned int h = *reinterpret_cast<const unsigned int*>(e + 4);
    if (k == 3u) return (double)w;                           // fun_image_width
    if (k == 4u) return (double)h;                           // fun_image_height
    const unsigned long long off = *reinterpret_cast<const unsigned long long*>(e + 8);
    return mr_tex(ctx + off, w, h, k, a, b);                 // fun_color_channel
}
"""


def pack_textures(images: Sequence[np.ndarray]) -> bytes:
    """The context of TEXTURE_RUNTIME_SOURCE for these (h, w, 3) uint8 images; 5 functions per image."""
    head = struct.pack("<II", len(images), 0)
    off = 8 + 16 * len(images)
    data = b""
    for im in images:
        head += struct.pack("<IIQ", im.shape[1], im.shape[0], off + len(data))
        data += np.ascontiguousarray(im, dtype=np.uint8).tobytes()
    return head + data


def by_name(name: str) -> Tuple[bytes, List[np.ndarray], Tuple[int, int]]:
    """(maray bytes, textures, (w, h)) for a workload name used by bench.py and the tests."""
    if name == "chess_1k":
        return chess_1k(), [], (1024, 1024)
    if name == "sdf":
        return sdf(), [], (1920, 1080)
    if name == "chess_4k":
        return chess_4k(), [], (3840, 2160)
    if name == "textured":
        return textured(), synthetic_textures(), (3840, 2160)
    if name == "chess_dsl":
        return chess_dsl(3840, 2160), [], (3840, 2160)
    if name == "deep":
        # MARAY_DEEP_VALUES shrinks the program for quick experiments (the benchmark config is 100 000)
        return deep(n_values=int(os.environ.get("MARAY_DEEP_VALUES", "100000"))), [], (8192, 8192)
    raise KeyError(name)
