/*
 * maray_cuda.h -- C ABI of the B200 (sm_100a) render path for Maray scenes.
 *
 * The reference (advancedresearch/maray v0.3.8, Rust) has no FFI: its render back ends are Rust
 * functions behind `gen_to_image` (reference src/lib.rs:1177-1195).  This ABI is what a new
 * `RenderMethod::Cuda` arm / `render::cuda_gen_to_image` would bind through `extern "C"`; each
 * entry point names the reference interface it stands in for.  INTEGRATION.md shows the Rust side.
 *
 * Conventions
 *   - every function returns MARAY_OK (0) or a negative MARAY_E_* code; the message for the last
 *     failure on a handle is maray_cuda_last_error(h) (for a failed create: last_error(NULL));
 *   - no exception or panic crosses this boundary; invalid scenes are rejected at load/compile
 *     time, never by a device fault;
 *   - the caller owns every host buffer it passes; the library copies what it keeps;
 *   - a handle may be used from one thread at a time; calls block until their work is complete
 *     unless they take a stream;
 *   - there is NO CPU fallback: render calls fail with MARAY_E_CUDA when no usable GPU exists.
 */
#ifndef MARAY_CUDA_H
#define MARAY_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct maray_cuda maray_cuda_t;

enum {
    MARAY_OK = 0,
    MARAY_E_INVALID = -1,      /* bad argument / call order                                   */
    MARAY_E_PARSE = -2,        /* not a .maray file (either layout)                           */
    MARAY_E_SCENE = -3,        /* scene rejected: unbound variable, cyclic Let, App id out of the
                                  runtime's function table (the reference yields NaN / panics)  */
    MARAY_E_COMPILE = -4,      /* NVRTC / code generation failure                             */
    MARAY_E_CUDA = -5,         /* CUDA runtime failure or no usable device                    */
    MARAY_E_UNSUPPORTED = -6   /* e.g. the interpreter asked to run a custom runtime's App     */
};

/* Back ends (siblings of the reference's WAT code generator, reference src/wasm.rs). */
enum {
    MARAY_BACKEND_INTERP = 0,  /* flat register bytecode run by the hand-written interpreter kernel */
    MARAY_BACKEND_NVRTC = 1,   /* straight-line CUDA compiled at run time for sm_100a, --fmad=false  */
    MARAY_BACKEND_AUTO = 2     /* time to first frame: cubins from the cache if they are there; otherwise the
                                  interpreter renders at once while NVRTC compiles on another thread, and renders
                                  switch to the generated kernels (between row chunks) when they are built.  Both
                                  back ends produce the same bytes. */
};

/* Progress reporting, the counterpart of `Report` (reference src/report.rs:19-27).  The callback is
 * the counterpart of the `report: F` closure of gen_to_image (reference src/lib.rs:1183):
 * it receives the caller's image buffer with the rows finished so far filled in, and progress in
 * [0,1].  It is invoked on the calling thread, between row bands. */
enum { MARAY_REPORT_NONE = 0, MARAY_REPORT_ROW = 1, MARAY_REPORT_DURATION_MS = 2 };
typedef void (*maray_report_fn)(void* user, uint8_t* rgb, uint32_t w, uint32_t h, double progress);

/* What the lowering found and what the last compile/render cost. */
typedef struct maray_cuda_stats {
    /* program */
    uint64_t tree_nodes;          /* nodes of the three channel trees as stored on the wire          */
    uint64_t dag_nodes;           /* values after hash-consing across the channels                   */
    uint64_t n_const, n_x_only, n_y_only, n_xy;
    uint64_t n_add, n_mul, n_neg, n_abs, n_recip, n_sqrt, n_step, n_min, n_max, n_sin, n_exp, n_ln, n_tex;
    uint32_t dag_depth;
    uint32_t legacy_layout;       /* 1 when the file used the pre-`Arc` variant numbering            */
    /* back end */
    uint32_t backend;
    uint32_t interp_instructions; /* bytecode length (interpreter back end)                          */
    uint32_t interp_slots;        /* per-pixel (wide) value slots the bytecode needs                 */
    uint32_t jit_segments;        /* parts the generated program was cut into (chain form: kernels)  */
    uint32_t jit_frame_slots;     /* doubles per pixel that cross a cut (0 when not segmented)       */
    uint32_t jit_registers;       /* registers per thread of the generated kernel (0 = unknown)      */
    uint32_t jit_source_bytes;
    uint32_t jit_cubin_bytes;
    uint32_t jit_units;           /* translation units compiled (1, or one per segment kernel)       */
    uint32_t jit_compile_threads; /* host threads that ran NVRTC concurrently (0 on a cache hit)     */
    uint32_t jit_cache_hit;       /* 1 when every cubin came from the cache directory                */
    uint32_t interp_uniform_slots;/* per-block row-uniform scalar slots (interpreter; 0 in the all-wide form) */
    uint32_t interp_block;        /* interpreter launch shape: threads per block ...                 */
    uint32_t interp_pixels_per_thread; /* ... and pixels per thread (a block spans block*ppt pixels of one row) */
    uint32_t tier_rows_interp;    /* MARAY_BACKEND_AUTO, last render: rows the interpreter rendered before the
                                     generated kernels took over (0 once they are installed)               */
    uint32_t jit_active;          /* 1 when launches go to the generated kernels                           */
    uint32_t jit_block;           /* generated kernels: threads per block                                  */
    uint32_t jit_round_pixels;    /* generated kernels: pixels one round of resident blocks covers on the first GPU
                                     (SMs x resident blocks x jit_block x jit_pixels_per_thread; 0 without a GPU).  A
                                     band or row chunk that is a whole number of rounds long pays no tail: hosts that
                                     cut a frame can cut there */
    uint32_t jit_pixels_per_thread; /* generated kernels: pixels per thread (2 with pixel pairs; a block covers
                                     jit_block x jit_pixels_per_thread consecutive pixels)                    */
    /* timings, milliseconds */
    double lower_ms;              /* Expr -> SSA                                                     */
    double codegen_ms;            /* SSA -> source / bytecode                                        */
    double nvrtc_ms;              /* NVRTC compile, all units (reported separately from render time) */
    double load_ms;               /* cubin load + uploads                                            */
    double kernel_ms[8];          /* last render: device time of the band kernel, per GPU            */
    double gather_ms;             /* last render: band gather to GPU 0 (peer copies)                 */
    double d2h_ms;                /* last render: device -> caller buffer                            */
    double render_ms;             /* last render: wall time of the call                              */
} maray_cuda_stats;

/* ---- lifetime ---------------------------------------------------------------------------------- */

/* Creates a render handle over `n_gpus` devices (`device_ids` NULL = devices 0..n_gpus-1).
 * n_gpus == 0 creates a host-only handle: it can load, validate, lower and compile scenes (NVRTC
 * needs no GPU) but every render call fails with MARAY_E_CUDA.
 * Stands in for: choosing `RenderMethod::JIT{threads,..}` (reference src/lib.rs:1166-1172). */
int maray_cuda_create(int n_gpus, const int* device_ids, maray_cuda_t** out);
void maray_cuda_destroy(maray_cuda_t* h);
const char* maray_cuda_last_error(const maray_cuda_t* h);

/* ---- scene ------------------------------------------------------------------------------------- */

/* The default texture runtime: `Runtime::<Textures>::from_parts(Textures{images}, functions(n))`
 * (reference examples/maray.rs:58-69, src/textures.rs:54-65).  rgb8[i] is w[i]*h[i]*3 bytes,
 * row-major R,G,B (image::RgbImage).  Copied to every GPU of the handle.  Must precede compile. */
int maray_cuda_set_textures(maray_cuda_t* h, uint32_t n, const uint8_t* const* rgb8,
                            const uint32_t* w, const uint32_t* hgt);

/* A Runtime<T> other than the default texture runtime (reference src/lib.rs:72-98).  `cuda_source` defines
 *     __device__ double maray_app(const unsigned char* ctx, unsigned long long ctx_bytes,
 *                                 unsigned int id, double a, double b);
 * and the scene's App(id, a, b) evaluates to maray_app(ctx, ctx_bytes, id, a, b) for id < n_functions (the reference's
 * functions[id](&ctx, id, a, b), src/lib.rs:664-668).  Replaces the texture runtime, and set_textures replaces it: one
 * runtime per handle, the last call of set_textures / set_functions wins.  NULL returns the handle to the default
 * texture runtime with no textures.  Takes effect at the next compile.
 *   - App id >= n_functions is MARAY_E_SCENE at compile time (the reference's index panic, as for textures).
 *   - maray_app must be a pure function of its arguments and the context bytes: the code generator may evaluate it
 *     once for equal arguments, skip it inside a guarded region whose guard is false across a warp, evaluate it twice
 *     per thread (pixel pairs), and evaluate it for idle lanes that redo a launch's first pixel.  It must not write
 *     memory, use shared memory, barriers or warp intrinsics.
 *   - The source is compiled after the library's device prelude with the same NVRTC options (sm_100a, --fmad=false):
 *     it may call mr_sin, mr_exp, mr_log (in the handle's libm mode, exact mode included), mr_tex and
 *     mr_as_u32_nonneg.  A compile error in it is MARAY_E_COMPILE; last_error carries the NVRTC log.
 *   - Only the NVRTC back end can call it.  MARAY_BACKEND_INTERP returns MARAY_E_UNSUPPORTED for a scene that calls
 *     App under a custom runtime; MARAY_BACKEND_AUTO uses cached cubins at once and otherwise compiles with NVRTC
 *     before it returns, so on a cold cache the first frame waits for NVRTC.
 *   - A fault inside maray_app (e.g. a read past ctx_bytes) is a bug of the caller's code: it is the one case in which
 *     this library's "never a device fault" does not hold. */
int maray_cuda_set_functions(maray_cuda_t* h, const char* cuda_source, uint32_t n_functions);
/* The context bytes of the custom runtime (`rt.ctx`), copied to every GPU of the handle.  Valid before or after
 * compile.  Takes effect at the next render and recompiles nothing.  Waits for the handle's in-flight work on its GPUs
 * (including bands rendered on a caller's stream) before it replaces the buffer. */
int maray_cuda_set_context(maray_cuda_t* h, const void* ctx, size_t bytes);

/* `maray::open` on an in-memory file (reference src/lib.rs:1227-1235): bincode
 * ([u32;2],[Expr;3]), current or legacy variant numbering. */
int maray_cuda_load_maray(maray_cuda_t* h, const uint8_t* bytes, size_t len);
/* The [u32;2] size stored in the file. */
int maray_cuda_scene_size(const maray_cuda_t* h, uint32_t* w, uint32_t* hgt);

/* Which sin/exp/ln the device evaluates `Expr::Sin/Exp/Ln` with (reference src/lib.rs:648-650 calls the platform
 * libm; src/wasm.rs:11-13 imports the same functions).  Takes effect at the next maray_cuda_compile.
 *   MARAY_LIBM_FAST   the default: exp and ln are glibc's algorithms (bit-exact); sin is a fast version, 18 FP64
 *                     instructions, <= 1.8 ULP, equal to glibc's result in ~80 % of arguments and one ULP away otherwise;
 *   MARAY_LIBM_GLIBC  exact mode: glibc 2.39's own algorithms (x86-64 FMA variants) operation for operation, so every
 *                     value has the bits the reference computes on such a host (|x| >= 105414350 in sin excepted);
 *   MARAY_LIBM_CUDA   libdevice's sin/exp/log (A/B).
 * The environment variable MARAY_LIBM=fast|glibc|cuda sets the default of new handles. */
enum { MARAY_LIBM_FAST = 0, MARAY_LIBM_GLIBC = 1, MARAY_LIBM_CUDA = 2 };
int maray_cuda_set_libm(maray_cuda_t* h, int libm);

/* Lowers the scene (lexical Let, hash-consing across channels, host constant folding) and builds
 * the chosen back end.  Stands in for `var_fixer::fix_color` + `Wasm::from_expr` x3
 * (reference src/render.rs:117,163-165; src/wasm.rs:136-158).  `stats` may be NULL. */
int maray_cuda_compile(maray_cuda_t* h, int backend, maray_cuda_stats* stats);

/* ---- render ------------------------------------------------------------------------------------ */

/* Progress settings for maray_cuda_render (default: MARAY_REPORT_NONE). */
int maray_cuda_set_report(maray_cuda_t* h, int kind, uint32_t every, maray_report_fn fn, void* user);

/* Supersampled anti-aliasing: s x s samples per pixel (1 <= s <= 16, else MARAY_E_INVALID), box-filtered to RGB8.
 * Every handle starts at s = 1, which is exactly the reference's frame (one sample at the integer coordinate).
 *   sample offsets   o_k = (double)(2k + 1 - s) * (1.0 / (2.0 * s)), k in [0, s): the centres of an s x s grid over the
 *                    pixel footprint [xi - 1/2, xi + 1/2), which is centred on the reference's sample point;
 *   sample (i, j)    of pixel (xi, yi) is the scene evaluated at X = (double)xi + o_i, Y = (double)yi + o_j (one IEEE
 *                    addition each), each channel converted with the reference's saturating `as u8`;
 *   pixel            per channel (sum over the s*s u8 samples + s*s/2) / (s*s), integer division: the box filter of the
 *                    reference's own frame rendered at s x the resolution.
 * Sample (i, j) is therefore pixel (xi, yi) of the reference's frame of the scene with x -> x + o_i, y -> y + o_j
 * substituted everywhere.  The frame is rendered as s*s passes of the compiled kernels, so it costs about s*s frames;
 * each GPU of the handle keeps a 6-byte-per-pixel accumulator, allocated at the first supersampled render.  Takes
 * effect at the next render (nothing is recompiled), on every render call; maray_cuda_render_window_f64 returns
 * MARAY_E_INVALID while s > 1.  Valid on a host-only handle. */
int maray_cuda_set_samples(maray_cuda_t* h, uint32_t s);

/* `gen_to_image(method, rt, color, &mut img, report)` (reference src/lib.rs:1177-1195):
 * renders a w x h image into the caller's HOST buffer `rgb` (w*h*3 bytes, the raw RgbImage layout,
 * so Rust passes img.as_mut_ptr(); a pageable Vec<u8> is the expected case).  One GPU: the frame is rendered
 * in row chunks whose device->host copies overlap the chunks still rendering.  Several GPUs: rows are split
 * into contiguous bands, every GPU renders its band and copies it into `rgb` over its own PCIe link. */
int maray_cuda_render(maray_cuda_t* h, uint32_t w, uint32_t hgt, uint8_t* rgb, maray_cuda_stats* stats);

/* What maray_cuda_render_png's encoder did. */
typedef struct maray_cuda_png_stats {
    uint64_t scanline_bytes;   /* hgt * (3*w + 1): the PNG's uncompressed image data                  */
    uint64_t png_bytes;        /* the whole file                                                      */
    uint32_t segments;         /* deflate segments encoded in parallel                                */
    uint32_t stored_segments;  /* segments emitted as stored blocks because Huffman coding did not pay */
    double   encode_ms;        /* device time from the filter kernel to the assembled file, first GPU  */
    double   d2h_ms;           /* copy of the file to the host                                        */
} maray_cuda_png_stats;

/* `gen(method, rt, color, file, size)` without the file (reference src/lib.rs:1199-1213): renders a w x hgt frame and
 * encodes it as a PNG (8-bit RGB, not interlaced) on the handle's first GPU.  With `rgb` not NULL the call renders
 * exactly as maray_cuda_render does (the frame lands in `rgb`, progress reports fire); with `rgb` NULL it renders as
 * maray_cuda_render_device does.  *png receives a pointer to the file's *len bytes in a pinned host buffer owned by
 * the handle, valid until the next maray_cuda_render_png or destroy.  The file's bytes are a function of the frame
 * alone (not of the GPU, the back end or the number of GPUs); decoded, it is the frame.  `stats` and `png_stats` may
 * be NULL.  Errors as maray_cuda_render; w or hgt above 2^31-1 is MARAY_E_INVALID (PNG fields are 31-bit); a failed
 * scratch allocation is MARAY_E_CUDA.  The encoder's scratch (about 7 bytes per scanline byte) stays allocated on the
 * first GPU until destroy. */
int maray_cuda_render_png(maray_cuda_t* h, uint32_t w, uint32_t hgt, uint8_t* rgb, const uint8_t** png, size_t* len,
                          maray_cuda_stats* stats, maray_cuda_png_stats* png_stats);

/* Same, but the finished frame stays in device memory on the handle's first GPU (bands of the other GPUs
 * are gathered there by peer copy over NVLink -- the only exchange step of the path):
 * *d_rgb receives a device pointer (owned by the handle, valid until the next render/destroy). */
int maray_cuda_render_device(maray_cuda_t* h, uint32_t w, uint32_t hgt, void** d_rgb, maray_cuda_stats* stats);

/* One band, for one-process-per-GPU hosts: renders rows [y0, y1) of the w x hgt image on the
 * handle's first GPU into the DEVICE buffer d_band ((y1-y0)*w*3 bytes), asynchronously on `stream`
 * (a cudaStream_t; NULL = the default stream).  The caller orders and gathers bands itself. */
int maray_cuda_render_band(maray_cuda_t* h, uint32_t w, uint32_t hgt, uint32_t y0, uint32_t y1,
                           void* d_band, void* stream);

/* One process per GPU, frame to be assembled in the first process's GPU memory: that process exports its frame
 * buffer once (CUDA IPC), the others open it and pass `frame + y0 * w * 3` to maray_cuda_render_band -- their band
 * kernels then store straight into that memory over NVLink, and no gather step remains.  The exporting handle
 * keeps the buffer until it renders a larger frame or is destroyed; importers must not outlive it. */
#define MARAY_IPC_HANDLE_BYTES 64
int maray_cuda_frame_export(maray_cuda_t* h, uint32_t w, uint32_t hgt, void* handle64, void** d_frame);
int maray_cuda_frame_import(maray_cuda_t* h, const void* handle64, void** d_frame);
/* The completion signal of that arrangement -- its only exchange, and not a collective: 64 counters live behind the
 * exported frame (same allocation, so every importer has them mapped).  maray_cuda_band_signal, enqueued on `stream`
 * after the band kernel, writes `value` into counter `rank` (one 4-byte atomic exchange over NVLink, system-scope
 * release: whoever sees the counter sees the band; each counter has a 128-byte line of its own).  maray_cuda_band_wait, on the exporting process, enqueues a wait until counters
 * [0, n_ranks) have all reached `value` (counters only grow: pass the step number).  The wait is bounded (~2 s); a
 * time-out is reported by the next maray_cuda_copy_to_host on that handle.  Pass the pointer frame_export /
 * frame_import returned, and the same w, hgt.  The poll is an atomic too: polled with loads, B200 shows a peer's
 * store tens of milliseconds late (DESIGN.md 6).  For hosts without a collective library; bench.py keeps NCCL's
 * one-element reduce as its default signal (measured next to each other: `bench.py --completion counters`). */
int maray_cuda_band_signal(maray_cuda_t* h, void* d_frame, uint32_t w, uint32_t hgt, uint32_t rank, uint32_t value, void* stream);
int maray_cuda_band_wait(maray_cuda_t* h, void* d_frame, uint32_t w, uint32_t hgt, uint32_t n_ranks, uint32_t value, void* stream);
/* Synchronous device -> host copy on the handle's first GPU (reads back a frame held by maray_cuda_frame_export /
 * maray_cuda_render_device without the caller needing a CUDA binding of its own). */
int maray_cuda_copy_to_host(maray_cuda_t* h, const void* d_src, void* host_dst, size_t bytes);

/* Parity instrumentation: the raw f64 channel values of the window [x0,x1) x [y0,y1) of the
 * w x hgt image, as 3 planes of (y1-y0)*(x1-x0) doubles (R, G, B), plus optionally its RGB8. */
int maray_cuda_render_window_f64(maray_cuda_t* h, uint32_t w, uint32_t hgt, uint32_t x0, uint32_t x1,
                                 uint32_t y0, uint32_t y1, double* planes, uint8_t* rgb);

/* ---- introspection ----------------------------------------------------------------------------- */

int maray_cuda_get_stats(const maray_cuda_t* h, maray_cuda_stats* stats);
/* Generated CUDA source of the NVRTC back end (after compile).  Returns its length in *len; copies
 * at most cap bytes (NUL-terminated when cap > 0). */
int maray_cuda_get_source(const maray_cuda_t* h, char* buf, size_t cap, size_t* len);
/* The translation units NVRTC actually compiled for the last scene (stats.jit_units of them; for a program
 * above the segment size one kernel per segment, launched in order -- see stats.jit_segments).  Same calling
 * convention as maray_cuda_get_source; MARAY_E_INVALID when `index` is out of range. */
int maray_cuda_get_module(const maray_cuda_t* h, uint32_t index, char* buf, size_t cap, size_t* len);
/* The sm_100a cubin NVRTC produced for translation unit `index` (tooling: `cuobjdump -sass` of it is how the FP64-pipe
 * instruction counts behind the roofline are read).  *len receives its size; at most cap bytes are copied. */
int maray_cuda_get_cubin(const maray_cuda_t* h, uint32_t index, void* buf, size_t cap, size_t* len);
/* Bytecode of the interpreter back end: 8-byte instructions, then the constant pool. */
int maray_cuda_get_bytecode(const maray_cuda_t* h, uint64_t* code, size_t cap_instr, size_t* n_instr,
                            double* consts, size_t cap_consts, size_t* n_consts);

/* Measures the FP64 pipe on GPU `gpu_index` of the handle with a DADD/DMUL (no FMA) issue-rate
 * kernel: *lane_ops_per_s = warp instructions * 32 / s.  The roofline denominator of bench.py. */
int maray_cuda_fp64_peak(maray_cuda_t* h, int gpu_index, double* lane_ops_per_s, double* dfma_lane_ops_per_s);

/* Library version string. */
const char* maray_cuda_version(void);

#ifdef __cplusplus
}
#endif
#endif /* MARAY_CUDA_H */
