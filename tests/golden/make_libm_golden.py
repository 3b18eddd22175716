"""Writes glibc_239_{sin,exp,log}.npy: arguments and results of glibc 2.39's sin, exp and log (x86-64, the FMA variants
an AVX2+FMA host selects), as uint64 bit patterns, shape (n, 2).  They pin the exact mode of the device libm
(csrc/device_libm_glibc.cuh) on hosts whose libm is another one (tests/test_glibc_libm.py).

The arguments follow tools/glibc_libm_check.c at a smaller scale: uniform and bit-uniform samples of every range it
tries, a few doubles on either side of its thresholds and table points, and the specials.  Seeded: a rerun on the
same glibc writes the same files.

usage (on an x86-64 host with glibc 2.39 and AVX2+FMA): python tests/golden/make_libm_golden.py
"""
import ctypes
import os
import platform

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PER_RANGE = 400
AROUND = 2


def _bits(v):
    return np.asarray(v, dtype=np.float64).view(np.uint64)


def _uniform(rng, lo, hi, both):
    x = lo + (hi - lo) * rng.random(PER_RANGE)
    return np.where(rng.random(PER_RANGE) < 0.5, -x, x) if both else x


def _bit_uniform(rng, lo, hi, both, n=PER_RANGE):
    a, b = int(_bits(lo)), int(_bits(hi))
    x = (np.uint64(a) + rng.integers(0, b - a, n, dtype=np.uint64)).view(np.float64)
    return np.where(rng.random(n) < 0.5, -x, x) if both else x


def _around(values, signs=(1.0, -1.0)):
    u = _bits(np.abs(np.asarray(values, dtype=np.float64)))
    out = [(u.astype(np.int64) + d).astype(np.uint64).view(np.float64) * s
           for d in range(-AROUND, AROUND + 1) for s in signs]
    return np.concatenate(out)


def arguments():
    rng = np.random.default_rng(239)
    inf = np.inf
    pi2 = float.fromhex("0x1.921fb54442d18p+0")
    sin_th = [2.0 ** -26, 0.126, 0.855469, 2.426265, 105414350.0, pi2, 2 * pi2, float.fromhex("0x1.2d97c7f3321d2p+1"),
              4 * pi2, 2.0 ** -1022, 1.0, 0.5, 710.0] + [k / 128 for k in range(1, 113)] + [k * pi2 for k in range(1, 65)]
    sin = [_uniform(rng, lo, hi, True) for lo, hi in [(2.0 ** -26, 0.126), (0.126, 0.855469), (0.855469, 2.426265),
                                                     (2.426265, 64.0), (64.0, 1e5), (1e5, 105414350.0)]]
    sin += [_bit_uniform(rng, 2.0 ** -1074, 105414350.0, True), _around(sin_th),
            np.array([0.0, -0.0, inf, -inf, np.nan, 2.0 ** -1074, 2.0 ** -27])]
    sin = np.concatenate(sin)
    sin = sin[~(np.abs(sin) >= 105414350.0) | ~np.isfinite(sin)]     # beyond: the documented gap (libdevice's sine)
    exp = [_uniform(rng, lo, hi, True) for lo, hi in [(0.0, 1.0), (0.0, 64.0), (0.0, 512.0), (512.0, 760.0)]]
    exp += [_bit_uniform(rng, 2.0 ** -1074, 2000.0, True),
            _around([2.0 ** -54, 512.0, 1024.0, 709.782712893384, 708.3964185322641, 745.1332191019411,
                     0.0054152123481245725, 1.0, float.fromhex("0x1.62e42fefa39efp-1"), float.fromhex("0x1.62e42fefa39efp-8"),
                     2.0 ** -1022]),
            np.array([0.0, -0.0, inf, -inf, np.nan, 2.0 ** -1074, 1e308, -1e308])]
    log = [_uniform(rng, lo, hi, False) for lo, hi in [(2.0 ** -20, 2.0), (0.9375, 1.0647), (1.0, 65.0), (1.0, 1e6)]]
    log += [_bit_uniform(rng, 2.0 ** -1074, float.fromhex("0x1.fffffffffffffp+1023"), False),
            _bit_uniform(rng, 2.0 ** -1074, 2.0 ** -1022, False, PER_RANGE // 10),
            _around([1.0, 0.9375, 1.0 + float.fromhex("0x1.09p-4"), 2.0 ** -1022, 0.5, 2.0, float.fromhex("0x1.6p-1"),
                     float.fromhex("0x1.6p+0")], signs=(1.0,)),
            np.array([0.0, -0.0, inf, -inf, np.nan, 2.0 ** -1074, -1.0, -(2.0 ** -1074), float.fromhex("0x1.fffffffffffffp+1023")])]
    return {"sin": sin, "exp": np.concatenate(exp), "log": np.concatenate(log)}


def main() -> None:
    assert platform.libc_ver() == ("glibc", "2.39") and platform.machine() == "x86_64", platform.libc_ver()
    libm = ctypes.CDLL("libm.so.6")
    for name, xs in arguments().items():
        fn = getattr(libm, name)
        fn.restype, fn.argtypes = ctypes.c_double, [ctypes.c_double]
        ys = np.array([fn(float(x)) for x in xs], dtype=np.float64)
        np.save(os.path.join(HERE, f"glibc_239_{name}.npy"), np.stack([_bits(xs), _bits(ys)], axis=1))
        print(name, xs.size)


if __name__ == "__main__":
    main()
