"""Host-side mirror of the reference's render entry points, on top of the C ABI.

  reference                                   here
  ------------------------------------------  ---------------------------------------------
  RenderMethod::{..}   src/lib.rs:1154-1173   RenderMethod.Cuda(gpus, report, backend, samples)  (new arm)
  Report               src/report.rs:19-27    Report.none() / Report.row(n) / Report.duration(ms)
  Runtime<Textures>    src/lib.rs:72-98       Runtime(Textures(images))  (functions = textures.functions(n))
  Runtime<T>           src/lib.rs:72-98       Runtime.from_parts(ctx_bytes, CudaFunctions(source, n))
  gen_to_image         src/lib.rs:1177-1195   gen_to_image(method, rt, color, img, report)
  gen                  src/lib.rs:1199-1213   gen(method, rt, color, file, size)
  open / save          src/lib.rs:1216-1235   open_ / save  (maray_b200.expr)

The CPU render methods of the reference (SingleInterpreted, ParallelInterpreted, JIT) are not
offered: this package is the GPU path only and has no CPU fallback.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass, field
from typing import Callable, List, Optional, Sequence, Union

import numpy as np

from . import _lib
from . import expr as _expr


class MarayCudaError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"maray_cuda error {code}: {message}")
        self.code = code
        self.message = message


@dataclass(frozen=True)
class Report:
    """reference src/report.rs:19-27"""
    kind: int = _lib.REPORT_NONE
    every: int = 0

    @staticmethod
    def none() -> "Report": return Report(_lib.REPORT_NONE, 0)
    @staticmethod
    def row(n: int) -> "Report": return Report(_lib.REPORT_ROW, int(n))
    @staticmethod
    def duration(ms: int) -> "Report": return Report(_lib.REPORT_DURATION_MS, int(ms))


class RenderMethod:
    """The new arm of the reference's `RenderMethod` (src/lib.rs:1154-1173)."""

    @dataclass(frozen=True)
    class Cuda:
        gpus: int = 1
        report: Report = field(default_factory=Report.none)
        # "auto": renders at once (cached cubins, else the bytecode kernel) while NVRTC compiles in the background;
        # "nvrtc": the JIT sibling of wasm.rs, compiled before the first render; "interp": the bytecode kernel only
        backend: str = "auto"
        device_ids: Optional[Sequence[int]] = None
        # anti-aliasing: samples x samples per pixel, box-filtered (CudaRenderer.set_samples); 1 is the reference's frame
        samples: int = 1


@dataclass
class Textures:
    """reference src/textures.rs:9-12 -- images are uint8 arrays shaped (h, w, 3)."""
    images: List[np.ndarray] = field(default_factory=list)


@dataclass(frozen=True)
class CudaFunctions:
    """The device twin of a `Runtime<T>`'s `functions` (reference src/lib.rs:72-98): CUDA source defining
    `__device__ double maray_app(const unsigned char* ctx, unsigned long long ctx_bytes, unsigned int id, double a,
    double b)`, and n = functions.len().  App(id, a, b) evaluates to maray_app(ctx, ctx_bytes, id, a, b) for id < n
    (include/maray_cuda.h, maray_cuda_set_functions, states what the function may and may not do)."""
    source: str
    n: int


@dataclass
class Runtime:
    """reference src/lib.rs:72-98.  The default texture runtime (`textures::functions(n)`, reference
    src/textures.rs:54-65), whose `functions` are implied, or a custom runtime: `functions` a CudaFunctions and `ctx`
    its context bytes."""
    ctx: Union[Textures, bytes, np.ndarray] = field(default_factory=Textures)
    functions: Optional[CudaFunctions] = None

    @staticmethod
    def new() -> "Runtime": return Runtime(Textures([]))
    @staticmethod
    def from_parts(ctx, functions=None) -> "Runtime":
        if isinstance(functions, CudaFunctions):
            return Runtime(ctx, functions)
        if functions is not None and len(functions) != 5 * len(ctx.images):
            raise MarayCudaError(_lib.E_UNSUPPORTED, "only the default texture runtime (5 functions per image) or "
                                                     "CudaFunctions can run on the device")
        return Runtime(ctx)


_BACKENDS = {"interp": _lib.BACKEND_INTERP, "nvrtc": _lib.BACKEND_NVRTC, "auto": _lib.BACKEND_AUTO}


class CudaRenderer:
    """Thin object wrapper over one `maray_cuda_t` handle."""

    def __init__(self, gpus: int = 1, device_ids: Optional[Sequence[int]] = None):
        self._L = _lib.load()
        self._h = ctypes.c_void_p()
        ids = None
        if device_ids is not None:
            ids = (ctypes.c_int * len(device_ids))(*device_ids)
            gpus = len(device_ids)
        rc = self._L.maray_cuda_create(gpus, ids, ctypes.byref(self._h))
        if rc != _lib.OK:
            raise MarayCudaError(rc, (self._L.maray_cuda_last_error(None) or b"").decode())
        self.gpus = gpus
        self._report_cb = None
        self._keep = []

    # -- plumbing ---------------------------------------------------------------------------
    def _check(self, rc: int) -> None:
        if rc != _lib.OK:
            raise MarayCudaError(rc, (self._L.maray_cuda_last_error(self._h) or b"").decode())

    def close(self) -> None:
        if getattr(self, "_h", None) and self._h.value:
            self._L.maray_cuda_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self): return self
    def __exit__(self, *a): self.close()

    # -- scene ------------------------------------------------------------------------------
    def set_textures(self, images: Sequence[np.ndarray]) -> None:
        arrs = [np.ascontiguousarray(a, dtype=np.uint8) for a in images]
        for a in arrs:
            if a.ndim != 3 or a.shape[2] != 3:
                raise ValueError("textures must be uint8 arrays shaped (h, w, 3)")
        n = len(arrs)
        ptrs = (ctypes.c_void_p * max(n, 1))(*[a.ctypes.data for a in arrs])
        ws = (ctypes.c_uint32 * max(n, 1))(*[a.shape[1] for a in arrs])
        hs = (ctypes.c_uint32 * max(n, 1))(*[a.shape[0] for a in arrs])
        self._check(self._L.maray_cuda_set_textures(self._h, n, ptrs, ws, hs))

    def set_functions(self, source: Optional[str], n: int = 0) -> None:
        """A custom runtime (maray_cuda_set_functions): `source` defines maray_app, App ids below n call it.  None
        returns to the default texture runtime with no textures.  Takes effect at the next compile."""
        self._check(self._L.maray_cuda_set_functions(self._h, None if source is None else source.encode(), int(n)))

    def set_context(self, buf) -> None:
        """The custom runtime's context bytes (maray_cuda_set_context): bytes-like or a C-contiguous numpy array.
        Takes effect at the next render; nothing is recompiled."""
        if isinstance(buf, np.ndarray):
            if not buf.flags.c_contiguous:
                raise ValueError("the context array must be C-contiguous")
            data = buf.view(np.uint8).reshape(-1)
        else:
            data = np.frombuffer(bytes(buf), dtype=np.uint8)
        self._check(self._L.maray_cuda_set_context(self._h, data.ctypes.data if data.size else None, data.size))

    def load(self, scene: Union[bytes, tuple]) -> tuple:
        """scene: `.maray` bytes, or (size, color) as returned by maray_b200.expr.open_."""
        if not isinstance(scene, (bytes, bytearray)):
            size, color = scene
            scene = _expr.to_bytes(size, color)
        scene = bytes(scene)
        self._check(self._L.maray_cuda_load_maray(self._h, scene, len(scene)))
        w, h = ctypes.c_uint32(), ctypes.c_uint32()
        self._check(self._L.maray_cuda_scene_size(self._h, ctypes.byref(w), ctypes.byref(h)))
        self.size = (w.value, h.value)
        return self.size

    def set_libm(self, libm: str) -> None:
        """"fast" (default), "glibc" (exact mode: the bits of the host libm the reference calls, reference
        src/lib.rs:648-650) or "cuda" (libdevice).  Takes effect at the next compile."""
        self._check(self._L.maray_cuda_set_libm(self._h, {"fast": _lib.LIBM_FAST, "glibc": _lib.LIBM_GLIBC, "cuda": _lib.LIBM_CUDA}[libm]))

    def set_samples(self, s: int) -> None:
        """Supersampled anti-aliasing: s x s samples per pixel (1 <= s <= 16), box-filtered to RGB8 (maray_cuda_set_samples).
        Sample (i, j) of pixel (x, y) is the scene at (x + o_i, y + o_j), o_k = (2k + 1 - s) * (1 / (2s)); the pixel is
        the rounded integer mean of the samples' u8 values.  1, the default, is the reference's frame.  Takes effect at
        the next render; nothing is recompiled."""
        self._check(self._L.maray_cuda_set_samples(self._h, int(s)))

    def compile(self, backend: str = "nvrtc", libm: Optional[str] = None) -> dict:
        if libm is not None:
            self.set_libm(libm)
        st = _lib.Stats()
        self._check(self._L.maray_cuda_compile(self._h, _BACKENDS[backend], ctypes.byref(st)))
        return st.as_dict()

    def stats(self) -> dict:
        st = _lib.Stats()
        self._check(self._L.maray_cuda_get_stats(self._h, ctypes.byref(st)))
        return st.as_dict()

    def source(self) -> str:
        n = ctypes.c_size_t()
        self._check(self._L.maray_cuda_get_source(self._h, None, 0, ctypes.byref(n)))
        buf = ctypes.create_string_buffer(n.value + 1)
        self._check(self._L.maray_cuda_get_source(self._h, buf, n.value + 1, None))
        return buf.value.decode()

    def modules(self) -> list:
        """The translation units NVRTC compiled for the last scene (one, or one kernel per segment)."""
        out = []
        n = ctypes.c_size_t()
        i = 0
        while self._L.maray_cuda_get_module(self._h, i, None, 0, ctypes.byref(n)) == _lib.OK:
            buf = ctypes.create_string_buffer(n.value + 1)
            self._check(self._L.maray_cuda_get_module(self._h, i, buf, n.value + 1, None))
            out.append(buf.value.decode())
            i += 1
        return out

    def cubin(self, index: int = 0) -> bytes:
        """The cubin of translation unit `index` of the NVRTC back end."""
        n = ctypes.c_size_t()
        self._check(self._L.maray_cuda_get_cubin(self._h, index, None, 0, ctypes.byref(n)))
        buf = ctypes.create_string_buffer(n.value)
        self._check(self._L.maray_cuda_get_cubin(self._h, index, buf, n.value, ctypes.byref(n)))
        return buf.raw

    def bytecode(self):
        ni, nk = ctypes.c_size_t(), ctypes.c_size_t()
        self._check(self._L.maray_cuda_get_bytecode(self._h, None, 0, ctypes.byref(ni), None, 0, ctypes.byref(nk)))
        code = np.zeros(ni.value, dtype=np.uint64)
        consts = np.zeros(nk.value, dtype=np.float64)
        self._check(self._L.maray_cuda_get_bytecode(self._h, code.ctypes.data, ni.value, None, consts.ctypes.data, nk.value, None))
        return code, consts

    # -- render -----------------------------------------------------------------------------
    def set_report(self, report: Report, fn: Optional[Callable[[np.ndarray, float], None]]) -> None:
        if fn is None or report.kind == _lib.REPORT_NONE:
            self._report_cb = _lib.REPORT_FN(0)
            self._check(self._L.maray_cuda_set_report(self._h, _lib.REPORT_NONE, 0, self._report_cb, None))
            return

        def tramp(_user, rgb, w, h, progress):
            img = np.ctypeslib.as_array(rgb, shape=(h, w, 3))
            fn(img, progress)

        self._report_cb = _lib.REPORT_FN(tramp)
        self._check(self._L.maray_cuda_set_report(self._h, report.kind, report.every, self._report_cb, None))

    def render_into(self, img: np.ndarray) -> dict:
        """img: writable C-contiguous uint8 (h, w, 3) -- the RgbImage raw layout."""
        if img.dtype != np.uint8 or img.ndim != 3 or img.shape[2] != 3 or not img.flags.c_contiguous or not img.flags.writeable:
            raise ValueError("img must be a writable C-contiguous uint8 array shaped (h, w, 3)")
        st = _lib.Stats()
        self._check(self._L.maray_cuda_render(self._h, img.shape[1], img.shape[0], img.ctypes.data, ctypes.byref(st)))
        return st.as_dict()

    def render(self, w: Optional[int] = None, h: Optional[int] = None) -> np.ndarray:
        w = self.size[0] if w is None else w
        h = self.size[1] if h is None else h
        img = np.zeros((h, w, 3), dtype=np.uint8)
        self.render_into(img)
        return img

    def render_png(self, w: Optional[int] = None, h: Optional[int] = None, img: Optional[np.ndarray] = None):
        """Renders a frame and encodes it as a PNG on the first GPU (maray_cuda_render_png).  Returns (file bytes,
        stats, png_stats).  With `img` (a writable C-contiguous uint8 (h, w, 3) array) the frame also lands there and
        progress reports fire as in render_into; without it the frame stays on the device."""
        if img is not None:
            if img.dtype != np.uint8 or img.ndim != 3 or img.shape[2] != 3 or not img.flags.c_contiguous or not img.flags.writeable:
                raise ValueError("img must be a writable C-contiguous uint8 array shaped (h, w, 3)")
            h, w = img.shape[0], img.shape[1]
        w = self.size[0] if w is None else w
        h = self.size[1] if h is None else h
        p, n = ctypes.c_void_p(), ctypes.c_size_t()
        st, ps = _lib.Stats(), _lib.PngStats()
        self._check(self._L.maray_cuda_render_png(self._h, w, h, None if img is None else img.ctypes.data, ctypes.byref(p),
                                                  ctypes.byref(n), ctypes.byref(st), ctypes.byref(ps)))
        return ctypes.string_at(p.value, n.value), st.as_dict(), ps.as_dict()

    def render_device(self, w: int, h: int) -> int:
        """Renders and leaves the frame on the first GPU; returns the device pointer."""
        p = ctypes.c_void_p()
        self._check(self._L.maray_cuda_render_device(self._h, w, h, ctypes.byref(p), None))
        return p.value

    def render_band(self, w: int, h: int, y0: int, y1: int, d_band: int, stream: int = 0) -> None:
        self._check(self._L.maray_cuda_render_band(self._h, w, h, y0, y1, ctypes.c_void_p(d_band), ctypes.c_void_p(stream)))

    def frame_export(self, w: int, h: int):
        """(handle bytes, device pointer) of this handle's frame buffer on its first GPU, for other processes to
        open with frame_import and render their bands into (maray_cuda_frame_export)."""
        buf = ctypes.create_string_buffer(_lib.IPC_HANDLE_BYTES)
        p = ctypes.c_void_p()
        self._check(self._L.maray_cuda_frame_export(self._h, w, h, buf, ctypes.byref(p)))
        return buf.raw, p.value

    def frame_import(self, handle: bytes) -> int:
        p = ctypes.c_void_p()
        self._check(self._L.maray_cuda_frame_import(self._h, ctypes.c_char_p(handle), ctypes.byref(p)))
        return p.value

    def band_signal(self, d_frame: int, w: int, h: int, rank: int, value: int, stream: int = 0) -> None:
        """Counter `rank` behind the shared frame := value, stream-ordered after this process's band kernel."""
        self._check(self._L.maray_cuda_band_signal(self._h, d_frame, w, h, rank, value, stream))

    def band_wait(self, d_frame: int, w: int, h: int, n_ranks: int, value: int, stream: int = 0) -> None:
        """Exporting process: `stream` waits until every rank's counter has reached `value` (bounded, ~2 s)."""
        self._check(self._L.maray_cuda_band_wait(self._h, d_frame, w, h, n_ranks, value, stream))

    def copy_to_host(self, d_src: int, out: np.ndarray) -> None:
        self._check(self._L.maray_cuda_copy_to_host(self._h, ctypes.c_void_p(d_src), out.ctypes.data, out.nbytes))

    def render_window_f64(self, w: int, h: int, x0: int, x1: int, y0: int, y1: int):
        """(planes float64 (3, y1-y0, x1-x0), rgb uint8 (y1-y0, x1-x0, 3)) of that window."""
        planes = np.zeros((3, y1 - y0, x1 - x0), dtype=np.float64)
        rgb = np.zeros((y1 - y0, x1 - x0, 3), dtype=np.uint8)
        self._check(self._L.maray_cuda_render_window_f64(self._h, w, h, x0, x1, y0, y1, planes.ctypes.data, rgb.ctypes.data))
        return planes, rgb

    def fp64_peak(self, gpu_index: int = 0):
        a, b = ctypes.c_double(), ctypes.c_double()
        self._check(self._L.maray_cuda_fp64_peak(self._h, gpu_index, ctypes.byref(a), ctypes.byref(b)))
        return a.value, b.value


def gen_to_image(method: "RenderMethod.Cuda", rt: Runtime, color, img: np.ndarray,
                 report: Optional[Callable[[np.ndarray, float], None]] = None) -> dict:
    """reference src/lib.rs:1177-1195.  `color` is [r, g, b] Exprs (maray_b200.expr) or `.maray` bytes
    (whose stored size is ignored, as the reference renders at the image's dimensions)."""
    if not isinstance(method, RenderMethod.Cuda):
        raise MarayCudaError(_lib.E_UNSUPPORTED, "only RenderMethod.Cuda is available (no CPU fallback)")
    h, w = img.shape[0], img.shape[1]
    with CudaRenderer(method.gpus, method.device_ids) as r:
        stats = _setup(r, method, rt, color, w, h, report)
        stats.update({k: v for k, v in r.render_into(img).items() if k.endswith("_ms")})
        return stats


def _setup(r: CudaRenderer, method: "RenderMethod.Cuda", rt: Runtime, color, w: int, h: int, report) -> dict:
    """Runtime, scene, back end, samples and progress of a gen_to_image / gen call; returns the compile stats."""
    if rt.functions is not None:
        r.set_functions(rt.functions.source, rt.functions.n)
        r.set_context(rt.ctx)
    else:
        r.set_textures(rt.ctx.images)
    r.load(color if isinstance(color, (bytes, bytearray)) else ([w, h], list(color)))
    stats = r.compile(method.backend)
    r.set_samples(method.samples)
    r.set_report(method.report, report)
    return stats


def gen(method: "RenderMethod.Cuda", rt: Runtime, color, file: str, size: Sequence[int]) -> dict:
    """reference src/lib.rs:1199-1213: render and save a PNG.  Progress ticks re-save the partial image on the host;
    the final file is encoded on the GPU (CudaRenderer.render_png)."""
    import os
    import sys

    from PIL import Image

    img = np.zeros((size[1], size[0], 3), dtype=np.uint8)

    def progress(partial: np.ndarray, p: float) -> None:
        print(f"{100.0 * p:.2f} %", file=sys.stderr, flush=True)
        Image.fromarray(partial).save(file)

    if not isinstance(method, RenderMethod.Cuda):
        raise MarayCudaError(_lib.E_UNSUPPORTED, "only RenderMethod.Cuda is available (no CPU fallback)")
    with CudaRenderer(method.gpus, method.device_ids) as r:
        _setup(r, method, rt, color, size[0], size[1], progress)
        png, stats, png_stats = r.render_png(img=img)
    tmp = file + ".tmp"
    with open(tmp, "wb") as f:
        f.write(png)
    os.replace(tmp, file)
    stats.update({"png_" + k: v for k, v in png_stats.items()})
    return stats
