// PNG encoder on the GPU (DESIGN.md 3.8): RGB8 frame in device memory -> one PNG file in pinned host memory.
// Adaptive filters, deflate in independent segments (one thread block each), device checksums and framing.
// png_gpu.cu also holds the encoder's CPU twin, which runs the same per-position, per-token and per-segment code
// serially; the GPU's file is byte-identical to the twin's.
#pragma once

#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>
#include <string>

namespace maray {

// Scratch of the encoder on one GPU, allocated at first use and grown, never shrunk (like the supersampling
// accumulator).  png_release frees it.
struct PngScratch {
    uint8_t* d_scan = nullptr; size_t scan_cap = 0;       // filtered scanlines, hgt * (3w + 1) bytes
    uint32_t* d_tokens = nullptr; size_t tokens_cap = 0;  // LZ77 tokens, at most one per scanline byte
    uint8_t* d_slots = nullptr; size_t slots_cap = 0;     // each segment's deflate bytes, slot_bytes(S) apart
    uint32_t* d_seg = nullptr; size_t seg_cap = 0;        // per segment: bytes, Adler-32 sums A and B, stored flag
    uint64_t* d_zoff = nullptr; size_t zoff_cap = 0;      // per segment: offset in the zlib stream
    uint8_t* d_file = nullptr; size_t file_cap = 0;       // the assembled file
    uint32_t* d_crc = nullptr; size_t crc_cap = 0;        // CRC-32 of each piece of each IDAT
    uint64_t* d_info = nullptr;                           // file bytes, stored segments
    uint8_t* h_file = nullptr; size_t h_cap = 0;          // pinned copy of the file
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
};

struct PngResult {
    const uint8_t* file = nullptr;
    uint64_t file_bytes = 0, scanline_bytes = 0;
    uint32_t segments = 0, stored_segments = 0;
    double encode_ms = 0.0, d2h_ms = 0.0;
};

// Encodes the w x hgt RGB8 frame at d_rgb (device memory of the current device) on `stream` and copies the file to
// sc.h_file.  w and hgt are at most 2^31 - 1.  Returns a CUDA error (message in *err) or cudaSuccess.
cudaError_t png_encode_device(PngScratch& sc, const uint8_t* d_rgb, uint32_t w, uint32_t hgt, cudaStream_t stream,
                              PngResult* out, std::string* err);
void png_release(PngScratch& sc);

}  // namespace maray
