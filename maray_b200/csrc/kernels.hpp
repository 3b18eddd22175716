// Host-side launchers of the kernels in kernels.cu.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

struct MrTexture;

// One launch of the interpreter kernel renders the window [x0, x1) x [y0, y0 + rows) of the image; pixel
// (x, y) goes to out[3 * ((y - y0) * (x1 - x0) + (x - x0))] (for whole rows of a frame: the RgbImage
// order of reference src/render.rs:19-31) and, optionally, its raw channel values to three f64 planes
// at the same pixel index.  Every block lies inside one row.
struct MrTileParams {
    unsigned char* out;
    double* f64_out;               // optional (parity checks); plane c starts at f64_out + c * f64_plane
    unsigned long long f64_plane;
    const MrTexture* tex;          // device texture table (may be null when the program has no App)
    unsigned int x0, x1, y0, rows;
    unsigned int nxb;              // blocks per row (set by launch_interp)
    unsigned int out_aligned;      // out is 16-byte aligned: full, aligned blocks store uint4
    unsigned int libm_exact;       // 1: sin/exp/ln return glibc's bits (device_libm_glibc.cuh, MARAY_LIBM=glibc)
    // Supersampling pass (device_sem.cuh MrSampling): pixel (x, y) is evaluated at (x + ox, y + oy); with acc set its
    // u8 samples are summed at acc[3 * i ..], i indexed like `out`, and the last of `count` passes stores the mean.
    double ox, oy;
    unsigned short* acc;           // null: one sample per pixel
    unsigned int pass, count;
};

namespace maray {

// Dynamic shared memory the interpreter needs for a launch configuration (n_scal = constants + row-uniform slots).
size_t interp_smem_bytes(unsigned int block, unsigned int pixels_per_thread, unsigned int n_wide, unsigned int n_scal);

// d_code / n_instr: the stream made by bytecode_for_launch (a whole number of kBcChunk-word chunks).
cudaError_t launch_interp(MrTileParams p, const uint64_t* d_code, unsigned int n_instr, const double* d_consts,
                          unsigned int n_consts, unsigned int n_uniform, unsigned int n_wide, bool all_wide, unsigned int block,
                          unsigned int pixels_per_thread, cudaStream_t stream);

cudaError_t launch_fp64_issue_rate(bool fma, double* d_sink, int iters, int blocks, cudaStream_t stream);

// Completion counters of a frame shared by band processes (kernels.cu, "band_signal/wait").
cudaError_t launch_band_signal(unsigned int* counter, unsigned int value, cudaStream_t stream);
cudaError_t launch_band_wait(unsigned int* counters, unsigned int stride, unsigned int n, unsigned int value, unsigned int* timed_out,
                             long long max_cycles, cudaStream_t stream);

}  // namespace maray
