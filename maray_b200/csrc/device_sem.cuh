// Device-side operation semantics of the render path.  This text is BOTH #included by the
// bytecode-interpreter kernel (interp_kernel.cu) and prepended to every NVRTC-generated kernel
// (embedded as a string by the build), so the two back ends cannot disagree on an operation.
//
// Each function restates one arm of the reference interpreter, reference src/lib.rs:632-669, and
// the `as u8` cast of reference src/render.rs:26-28 (table: SURVEY.md Appendix B).  All code that
// includes this is compiled with --fmad=false: the reference never fuses a*b+c.
#ifndef MARAY_DEVICE_SEM_CUH
#define MARAY_DEVICE_SEM_CUH

#include "device_libm.cuh"   // mr_sin / mr_exp / mr_log  (the build inlines this text for NVRTC)

// Step(a): `if v >= 0.0 {1.0} else {0.0}`  (NaN -> 0, -0.0 -> 1).  reference src/lib.rs:644-647
__device__ __forceinline__ double mr_step(double v) { return (v >= 0.0) ? 1.0 : 0.0; }

// f64::max / f64::min as compiled for x86-64: NaN operands are ignored, and on an equal-compare
// tie (incl. +0/-0) the FIRST operand is returned.  reference src/lib.rs:655-658; DESIGN.md
// "Semantics".  (CUDA's fmax/fmin would return +0 for max(-0,+0) regardless of order.)
// Written as one select on (b > a || isnan(a)): 2 DSETP + 2 FSEL in SASS.
//
// The select itself is inline PTX on purpose.  Written as `cond ? b : a`, NVVM recognises the pattern
// (whenever `a` is a literal, so `a != a` folds away) and emits PTX min.f64 / max.f64, and ptxas then
// re-associates a max(0, min(1, t)) pair into min(1, max(0, t)) -- equal for numbers, but for t = NaN
// the first form is 1 (NaN ignored, then max(0,1)) and the second is 0.  Measured on sm_100a with
// CUDA 12.9: `max(0, min(1, ln(x-5)^2))` rendered 0 instead of 1 wherever the logarithm was NaN
// (tests/test_gpu_parity.py::test_batched_transcendentals_and_their_repair_path).  An opaque selp keeps
// the compare-and-select exactly as written; the cost is the same 2 DSETP + 2 FSEL (1 + 2 for a literal).
#ifdef MR_HOST_TEXT   /* tests/helpers.py compiles the generated text as plain C++ */
static inline double mr_pick(bool take_b, double a, double b) { return take_b ? b : a; }
#else
__device__ __forceinline__ double mr_pick(bool take_b, double a, double b) {
    double r;
    asm("{ .reg .pred p; setp.ne.s32 p, %3, 0; selp.f64 %0, %2, %1, p; }" : "=d"(r) : "d"(a), "d"(b), "r"((int)take_b));
    return r;
}
#endif
__device__ __forceinline__ double mr_max(double a, double b) { return mr_pick((b > a) || (a != a), a, b); }
__device__ __forceinline__ double mr_min(double a, double b) { return mr_pick((b < a) || (a != a), a, b); }

// The vote in front of a guarded region of a generated kernel (codegen.cpp find_guard_regions): is the guard true on
// some lane of this warp?  Every lane of the warp reaches every vote.  The host builds of the text run one thread at a
// time: there the guard decides alone, or, with MR_HOST_GUARDS_ALWAYS, every region is evaluated at every pixel -- the
// two extremes between which the GPU lies, warp by warp.
#if defined(MR_HOST_GUARDS_ALWAYS)
static inline bool mr_warp_any(bool) { return true; }
#elif defined(MR_HOST_TEXT)
static inline bool mr_warp_any(bool b) { return b; }
#else
__device__ __forceinline__ bool mr_warp_any(bool b) { return __any_sync(0xffffffffu, b); }
#endif

// Recip(a) = 1.0 / a, IEEE round-to-nearest.  reference src/lib.rs:642
__device__ __forceinline__ double mr_recip(double v) { return __drcp_rn(v); }
// Sqrt(a), IEEE round-to-nearest.  reference src/lib.rs:643
__device__ __forceinline__ double mr_sqrt(double v) { return __dsqrt_rn(v); }

// `f64 as u8`: truncate toward zero, saturate to [0,255], NaN -> 0.  reference src/render.rs:26-28
// fmax(v, 0) maps NaN and negatives to 0 (CUDA fmax returns the non-NaN operand), fmin clamps the
// top; the conversion then only ever sees [0, 255].  (The conversion is NOT relied on for NaN:
// measured on sm_100a, cvt.rzi.u32.f64 of the NaN produced by inf*0 is not 0.)
__device__ __forceinline__ unsigned int mr_as_u8(double v) {
    return __double2uint_rz(fmin(fmax(v, 0.0), 255.0));
}
// `f64 as u32` for a value already known not to be negative: saturating, NaN -> 0.
__device__ __forceinline__ unsigned int mr_as_u32_nonneg(double v) {
    return __double2uint_rz(fmax(v, 0.0));
}

// fun_color_channel.  reference src/textures.rs:27-36
//   if x < 0.0 || y < 0.0 -> 0.0 (NaN passes this test); x as u32, y as u32 (saturating, NaN -> 0);
//   if x >= w || y >= h -> 0.0; else data[(y*w + x)*3 + k] as f64.
__device__ __forceinline__ double mr_tex(const unsigned char* __restrict__ data, unsigned int w, unsigned int h,
                                         unsigned int k, double x, double y) {
    if (x < 0.0 || y < 0.0) return 0.0;
    unsigned int xi = mr_as_u32_nonneg(x);
    unsigned int yi = mr_as_u32_nonneg(y);
    if (xi >= w || yi >= h) return 0.0;
    return (double)__ldg(data + ((size_t)yi * w + xi) * 3u + k);
}

// One texture as the kernels see it (device-resident RGB8, row-major, no padding).
struct MrTexture {
    const unsigned char* data;
    unsigned int w, h;
};

// Launch parameters shared by both back ends.  A launch renders the n pixels with linear index
// p0 .. p0+n-1 (index = y*W + x, the RgbImage order of reference src/render.rs:19-31) and writes
// pixel p0+j to out[3*j .. 3*j+2].
struct MrParams {
    unsigned char* out;        // RGB8 band buffer
    double* f64_out;           // optional (parity checks): raw channel values, 3 planes; pixel p0+j
                               // goes to f64_out[c*f64_plane + j]
    unsigned long long f64_plane;
    const MrTexture* tex;      // device texture table (may be null when the program has no App)
    unsigned int p0, n, W;
    unsigned int out_aligned;  // out is 16-byte aligned: full blocks store uint4
    // Unused by the generated kernels.  Kept so that host code written against this struct -- drivers that compile the
    // text maray_cuda_get_source returns, like the test suite's -- still compiles, and so that the chain kernels' frame
    // arguments (F, FS), which follow it, keep their parameter offsets: without these 24 bytes F sits at another 16-byte
    // offset, ptxas loads it per thread (LDC.64) instead of uniformly (LDCU.64), and the deep scene ran 0.3 % slower
    // (B200, 1000 W).
    const double* colv;
    const double* rowv;
    unsigned int row_base, rows;
};

// Supersampling (maray_cuda_set_samples): a frame of s x s samples per pixel is rendered as s*s passes of the same
// kernel, each with one uniform sub-pixel offset; the kernel evaluates the scene at X = xi + ox, Y = yi + oy.  The u8
// samples are summed in a uint16 x 3 accumulator (pixel p0+j of the launch at acc[3*j .. 3*j+2]) and the last pass
// writes the box mean (sum + count/2) / count as RGB8.  A separate kernel parameter, not a field of MrParams: host
// code that builds an MrParams and calls the kernel with it alone still gets the zero value, one sample per pixel.
struct MrSampling {
    double ox, oy;             // this pass's sub-pixel offset
    unsigned short* acc;       // null: one sample per pixel, the epilogue stores RGB8 directly
    unsigned int pass, count;  // pass in [0, count); count = s*s
};

// Adds this pass's u8 samples to the accumulator.  Returns true on the last pass, with (r8, g8, b8) resolved to the
// pixel's RGB8; false otherwise (nothing to store yet).  `pass` and `count` are uniform, so is the result.
__device__ __forceinline__ bool mr_accumulate(const MrSampling& sp, size_t idx, bool active, unsigned int& r8,
                                              unsigned int& g8, unsigned int& b8) {
    unsigned short* a = sp.acc + 3u * idx;
    if (active && sp.pass != 0u) { r8 += a[0]; g8 += a[1]; b8 += a[2]; }
    if (sp.pass + 1u < sp.count) {
        if (active) { a[0] = (unsigned short)r8; a[1] = (unsigned short)g8; a[2] = (unsigned short)b8; }
        return false;
    }
    const unsigned int half = sp.count >> 1;
    r8 = (r8 + half) / sp.count; g8 = (g8 + half) / sp.count; b8 = (b8 + half) / sp.count;
    return true;
}

// Packs one pixel's RGB8 into the block's staging tile and writes the tile with coalesced 16-byte
// stores (768 B per 256 pixels).  Every thread of the block must call this.
__device__ __forceinline__ void mr_store_rgb8(const MrParams& p, unsigned int* stage, unsigned int r8, unsigned int g8,
                                              unsigned int b8, double r, double g, double b, bool active, unsigned int j) {
    const unsigned int tid = threadIdx.x;
    const unsigned int first = blockIdx.x * blockDim.x;
    unsigned char* sb = reinterpret_cast<unsigned char*>(stage);
    sb[3u * tid + 0u] = (unsigned char)r8;
    sb[3u * tid + 1u] = (unsigned char)g8;
    sb[3u * tid + 2u] = (unsigned char)b8;
    if (p.f64_out != nullptr && active) {
        p.f64_out[j] = r;
        p.f64_out[(size_t)p.f64_plane + j] = g;
        p.f64_out[2u * (size_t)p.f64_plane + j] = b;
    }
    __syncthreads();
    const unsigned int valid = (p.n - first < blockDim.x) ? (p.n - first) : blockDim.x;
    unsigned char* dst = p.out + 3u * (size_t)first;
    if (p.out_aligned && valid == blockDim.x && (blockDim.x & 15u) == 0u) {
        const unsigned int vecs = 3u * blockDim.x / 16u;
        if (tid < vecs) reinterpret_cast<uint4*>(dst)[tid] = reinterpret_cast<const uint4*>(stage)[tid];
    } else {
        for (unsigned int i = tid; i < 3u * valid; i += blockDim.x) dst[i] = sb[i];
    }
}

// The epilogue of a generated kernel: `as u8` of the three channels, then mr_store_rgb8.  (Its arguments stay as they
// are: host code compiled against the generated text, like the oracle's JIT stand-in, puts its own store in its place.)
__device__ __forceinline__ void mr_store_block(const MrParams& p, unsigned int* stage, double r, double g, double b,
                                               bool active, unsigned int j) {
    mr_store_rgb8(p, stage, mr_as_u8(r), mr_as_u8(g), mr_as_u8(b), r, g, b, active, j);
}

// The epilogue of a supersampling pass (sp.acc != null): adds the u8 samples to the accumulator; the last pass stores
// the resolved pixels.  Every thread of the block must call this; before the last pass the whole block returns.
__device__ __forceinline__ void mr_store_sampled(const MrParams& p, const MrSampling& sp, unsigned int* stage, double r,
                                                 double g, double b, bool active, unsigned int j) {
    unsigned int r8 = mr_as_u8(r), g8 = mr_as_u8(g), b8 = mr_as_u8(b);
    if (!mr_accumulate(sp, j, active, r8, g8, b8)) return;
    mr_store_rgb8(p, stage, r8, g8, b8, r, g, b, active, j);
}

#endif  // MARAY_DEVICE_SEM_CUH
