"""ctypes binding of libmaray_cuda.so (include/maray_cuda.h).  No fallback: if the library is not
built, importing this module raises with the build command."""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmaray_cuda.so")

OK, E_INVALID, E_PARSE, E_SCENE, E_COMPILE, E_CUDA, E_UNSUPPORTED = 0, -1, -2, -3, -4, -5, -6
BACKEND_INTERP, BACKEND_NVRTC, BACKEND_AUTO = 0, 1, 2
REPORT_NONE, REPORT_ROW, REPORT_DURATION_MS = 0, 1, 2
IPC_HANDLE_BYTES = 64
LIBM_FAST, LIBM_GLIBC, LIBM_CUDA = 0, 1, 2

REPORT_FN = ctypes.CFUNCTYPE(None, ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint8), ctypes.c_uint32, ctypes.c_uint32,
                             ctypes.c_double)


class Stats(ctypes.Structure):
    _fields_ = (
        [(n, ctypes.c_uint64) for n in (
            "tree_nodes", "dag_nodes", "n_const", "n_x_only", "n_y_only", "n_xy",
            "n_add", "n_mul", "n_neg", "n_abs", "n_recip", "n_sqrt", "n_step", "n_min", "n_max",
            "n_sin", "n_exp", "n_ln", "n_tex")]
        + [(n, ctypes.c_uint32) for n in (
            "dag_depth", "legacy_layout", "backend", "interp_instructions", "interp_slots",
            "jit_segments", "jit_frame_slots", "jit_registers", "jit_source_bytes", "jit_cubin_bytes",
            "jit_units", "jit_compile_threads", "jit_cache_hit", "interp_uniform_slots", "interp_block",
            "interp_pixels_per_thread", "tier_rows_interp", "jit_active", "jit_block", "jit_round_pixels")]
        + [("lower_ms", ctypes.c_double), ("codegen_ms", ctypes.c_double), ("nvrtc_ms", ctypes.c_double),
           ("load_ms", ctypes.c_double), ("kernel_ms", ctypes.c_double * 8), ("gather_ms", ctypes.c_double),
           ("d2h_ms", ctypes.c_double), ("render_ms", ctypes.c_double)]
    )

    def as_dict(self) -> dict:
        d = {}
        for name, _ in self._fields_:
            v = getattr(self, name)
            d[name] = list(v) if name == "kernel_ms" else v
        return d


# every symbol include/maray_cuda.h declares: (name, restype, argtypes)
_P = ctypes.c_void_p
SYMBOLS = [
    ("maray_cuda_create", ctypes.c_int, [ctypes.c_int, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(_P)]),
    ("maray_cuda_destroy", None, [_P]),
    ("maray_cuda_last_error", ctypes.c_char_p, [_P]),
    ("maray_cuda_set_textures", ctypes.c_int, [_P, ctypes.c_uint32, ctypes.POINTER(_P), ctypes.POINTER(ctypes.c_uint32),
                                               ctypes.POINTER(ctypes.c_uint32)]),
    ("maray_cuda_load_maray", ctypes.c_int, [_P, ctypes.c_char_p, ctypes.c_size_t]),
    ("maray_cuda_scene_size", ctypes.c_int, [_P, ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_uint32)]),
    ("maray_cuda_set_libm", ctypes.c_int, [_P, ctypes.c_int]),
    ("maray_cuda_set_samples", ctypes.c_int, [_P, ctypes.c_uint32]),
    ("maray_cuda_compile", ctypes.c_int, [_P, ctypes.c_int, ctypes.POINTER(Stats)]),
    ("maray_cuda_set_report", ctypes.c_int, [_P, ctypes.c_int, ctypes.c_uint32, REPORT_FN, _P]),
    ("maray_cuda_render", ctypes.c_int, [_P, ctypes.c_uint32, ctypes.c_uint32, _P, ctypes.POINTER(Stats)]),
    ("maray_cuda_render_device", ctypes.c_int, [_P, ctypes.c_uint32, ctypes.c_uint32, ctypes.POINTER(_P),
                                                ctypes.POINTER(Stats)]),
    ("maray_cuda_render_band", ctypes.c_int, [_P, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, _P, _P]),
    ("maray_cuda_frame_export", ctypes.c_int, [_P, ctypes.c_uint32, ctypes.c_uint32, _P, ctypes.POINTER(_P)]),
    ("maray_cuda_frame_import", ctypes.c_int, [_P, _P, ctypes.POINTER(_P)]),
    ("maray_cuda_band_signal", ctypes.c_int, [_P, _P] + [ctypes.c_uint32] * 4 + [_P]),
    ("maray_cuda_band_wait", ctypes.c_int, [_P, _P] + [ctypes.c_uint32] * 4 + [_P]),
    ("maray_cuda_copy_to_host", ctypes.c_int, [_P, _P, _P, ctypes.c_size_t]),
    ("maray_cuda_render_window_f64", ctypes.c_int, [_P] + [ctypes.c_uint32] * 6 + [_P, _P]),
    ("maray_cuda_get_stats", ctypes.c_int, [_P, ctypes.POINTER(Stats)]),
    ("maray_cuda_get_source", ctypes.c_int, [_P, ctypes.c_char_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t)]),
    ("maray_cuda_get_module", ctypes.c_int, [_P, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t)]),
    ("maray_cuda_get_cubin", ctypes.c_int, [_P, ctypes.c_uint32, _P, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t)]),
    ("maray_cuda_get_bytecode", ctypes.c_int, [_P, _P, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t), _P,
                                               ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t)]),
    ("maray_cuda_fp64_peak", ctypes.c_int, [_P, ctypes.c_int, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]),
    ("maray_cuda_version", ctypes.c_char_p, []),
]

_lib = None


def load():
    """Loads libmaray_cuda.so.  Raises if it is missing -- the render path has no other implementation."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is not built. Build it with `make -C maray_b200/csrc` "
                "(or `python -c 'import __graft_entry__ as g; g.build()'`); maray_b200 has no CPU or PyTorch fallback.")
        L = ctypes.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib
