// Straight-line CUDA source from the SSA program: the GPU sibling of the reference's WAT code
// generator (reference src/wasm.rs:77-124).  Differences that are deliberate (SURVEY.md F9):
// the source is emitted from the hash-consed SSA program, not from the tree text, so every value
// is computed once, all three channels share one kernel, and declarations never collide.
#pragma once
#include <string>
#include <vector>

#include "program.hpp"

namespace maray {

struct CodegenOptions {
    // Programs with more values than this are cut into segments of at most this many values (see `chain`).
    // Bounds ptxas time, which is super-linear in basic-block size, and sets how many units can compile
    // concurrently.
    uint32_t segment_values = 16384;
    // sin/exp/ln are inlined below this many transcendental values, called out-of-line above it
    // (their inlined bodies dominate code size and compile time in transcendental-heavy scenes).
    uint32_t inline_transcendentals_below = kOutOfLineTranscendentals;
    // Launch shape chosen from the program (see `block`, `min_blocks_per_sm`): a LARGE straight-line program -- one
    // kernel, sin/exp/ln inlined, at least kOneBlockPerSmValues values: hundreds of KB of code that no warp re-uses --
    // runs as ONE 640-thread block per SM (96 registers, 20 warps).  Warps that start together stay within the
    // instruction caches' reach of each other and share fetches; separately scheduled small blocks each stream the
    // code on their own.  Measured, chess_4k (profiles/r02c_variants_chess4k_launch_shape.jsonl): 256 x 2 3.86 ms,
    // 640 x 1 3.48 ms -- and 128 x 5, the same registers and warps in five blocks, 4.75 ms.  Sizes that are not a
    // multiple of 128 (uneven warps per scheduler) lose 8 %.  Everything else keeps 256 x 2.  false = `block` and
    // `min_blocks_per_sm` as given (set by MARAY_JIT_BLOCK / MARAY_JIT_MIN_BLOCKS).
    bool auto_shape = true;
    // The scene's declared frame size and the GPU's SM count, when known: a frame of few rounds pays for its last,
    // partial round of blocks, so among the one-block-per-SM shapes that measured within 2 % of each other on a
    // large frame (640 threads / 96 registers 1.00, 768 / 80 1.015, 1 024 / 64 1.02) the one whose rounds fit the
    // frame best is taken: 1 024 x 1 024 pixels are 11.07 rounds of 640 (12 paid) but 6.92 rounds of 1 024.
    uint64_t frame_pixels_hint = 0;
    uint32_t sm_count_hint = 148;
    // Threads per block of the generated kernel (a multiple of 32; one pixel per thread).
    uint32_t block = 256;
    // __launch_bounds__ second argument: resident blocks per SM the register allocation must allow
    // (0 = leave it to ptxas).  2 x 256 threads caps the kernel at 128 registers = 16 resident warps
    // per SM, the best point of the sweep in profiles/ (ptxas left alone lands anywhere in 128..190).
    uint32_t min_blocks_per_sm = 2;
    // Scene constants live in a __constant__ table and are read as c[bank][offset] operands of the
    // FP64 instructions instead of being materialised with two 32-bit moves each.
    bool constants_in_bank = true;
    // step(sin(u)) with no other reader of the sine evaluates only the sign of the sine (mr_sin_ge0): exact, and on
    // chess.maray a quarter of all instructions (MARAY_JIT_SIGN_OF_SINE=0 for A/B).
    bool sign_of_sine = true;
    // Programs above segment_values: one KERNEL per segment, each its own translation unit, values that cross
    // a cut in a global-memory frame F[slot * FS + pixel].  The units share nothing: NVRTC compiles them
    // concurrently, nothing is linked, no segment pays a call ABI.  false = __noinline__ segment functions in
    // one unit with a per-thread local-memory frame (round 1's form: generate_cuda_source, MARAY_JIT_CHAIN=0).
    bool chain = true;
    // Size of a chain segment.  Smaller than segment_values on purpose: the cut-off decides WHETHER a program is
    // cut (below it one kernel is fastest), this decides how many units compile concurrently once it is.
    uint32_t chain_segment_values = 6144;
    // Evaluate values that are exactly 0.0 or 1.0 at every pixel (step, products/min/max of such
    // values, 1 - b) as boolean logic instead of FP64 arithmetic.  Exact: no channel bit changes.
    bool boolean_logic = true;
};

struct CodegenInfo {
    uint32_t segments = 0;
    bool chain = false;             // one kernel per segment (modules.size() == segments), launched in order
    uint32_t frame_slots = 0;       // doubles per pixel of the frame that carries values across cuts (0 when not segmented)
    bool transcendentals_inlined = true;
    uint32_t block = 256;           // threads per block the kernel must be launched with
    uint32_t dynamic_smem_bytes = 0; // dynamic shared memory the kernel must be launched with (batch scratch + tables)
};

// Names of the generated kernels (extern "C").
extern const char* const kJitKernelName;
constexpr uint32_t kOneBlockPerSmValues = 4096;   // CodegenOptions::auto_shape
// Guarded regions (codegen.cpp find_guard_regions): a boolean AND whose dearer operand is read by nothing else
// evaluates that operand only when the other one is true on some lane of the warp.  A region is made when the skipped
// operand weighs at least this much (one per value, 7 per sign-only sine, 16 per inlined sin/exp/ln).  Chess's texture
// operands weigh 40-51 and get a region each; the ANDs inside them (23-25) and beside them (11) do not pay: measured,
// chess_4k on one B200, profiles/r04_guard_threshold_sweep.jsonl: 3.517 ms without regions, 2.939 ms with the
// 128 texture regions, 2.943 / 2.982 / 3.058 ms when the 15 / 128 / 207 smaller ANDs get regions too.  sdf, textured
// and deep have no AND this heavy.
constexpr uint32_t kGuardBodyMinWeight = 32;

// One translation unit (segment functions, if any, as __noinline__ functions of the same unit).
std::string generate_cuda_source(const Program& prog, const CodegenOptions& opt, CodegenInfo* info);
// The translation units to compile: one, or -- opt.chain and a program above opt.segment_values -- one per
// segment, each holding a kernel named kJitKernelName with the extra arguments (double* F, unsigned long long FS).
std::vector<std::string> generate_cuda_modules(const Program& prog, const CodegenOptions& opt, CodegenInfo* info);

}  // namespace maray
