// C ABI of the render path (include/maray_cuda.h): handle, texture upload, compile, render.
//
// Shape of the work per render call (the counterpart of reference src/render.rs:102-192):
//   rows are cut into contiguous bands, one per GPU of the handle; each GPU runs the band kernel
//   on its own stream; GPU 0 renders straight into the frame buffer, the other GPUs render into a
//   local band buffer and push it into GPU 0's frame with one peer copy (the only exchange step);
//   one device->host copy hands the frame to the caller.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <sys/stat.h>
#include <unistd.h>
#include <nvrtc.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "../../include/maray_cuda.h"
#include "bytecode.hpp"
#include "codegen.hpp"
#include "device_sem.cuh"
#include "expr.hpp"
#include "kernels.hpp"
#include "program.hpp"

using namespace maray;

namespace {

thread_local std::string g_create_error;

double now_ms() {
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

struct HostTexture { uint32_t w, h; std::vector<uint8_t> rgb; };

struct Gpu {
    int device = 0;
    int sms = 148;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // pipelined host renders (render_frame_pipelined): one stream + event per row chunk, one copy stream
    static constexpr int kChunks = 4;
    cudaStream_t chunk_stream[kChunks] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t chunk_done[kChunks] = {nullptr, nullptr, nullptr, nullptr};
    cudaStream_t copy_stream = nullptr;
    // band / frame buffer
    uint8_t* d_out = nullptr; size_t out_cap = 0;
    double* d_f64 = nullptr; size_t f64_cap = 0;
    // supersampling: uint16 x 3 sums per pixel, indexed by the pixel's index in the frame (maray_cuda_set_samples)
    uint16_t* d_acc = nullptr; size_t acc_cap = 0;
    // textures
    std::vector<uint8_t*> d_tex;
    MrTexture* d_textab = nullptr;
    // back ends
    std::vector<cudaLibrary_t> libs;                   // one per translation unit (chain form: one per segment)
    std::vector<cudaKernel_t> jit_kernels;             // the kernel of each unit, in launch order
    double* d_frame = nullptr; size_t frame_cap = 0;   // chain form: values crossing segment cuts, F[slot * FS + pixel]
    cudaEvent_t frame_done = nullptr;                  // last chain launch that used d_frame (one per GPU, not per stream)
    uint64_t* d_code = nullptr;
    double* d_consts = nullptr;
    double* d_sink = nullptr;
    bool peer_to_0 = false;
};

}  // namespace

// What the NVRTC back end builds from a program.  It does not touch the handle or a device, so it can be
// made on another thread while the interpreter renders (MARAY_BACKEND_AUTO).
struct JitBuild {
    std::vector<std::string> modules;         // every translation unit
    std::string source;                       // the same statements as ONE unit (tooling, host-side tests)
    std::vector<std::vector<char>> cubins;    // one per unit
    CodegenInfo info;
    unsigned maxreg = 0;
    int libm = MARAY_LIBM_FAST;               // which sin/exp/ln the units are compiled against (maray_cuda_set_libm)
    uint64_t frame_pixels = 0;                // the scene's declared size (a hint for the launch shape), 0 = unknown
    uint32_t sms = 148;                       // SMs of the first GPU (148 without one)
    double codegen_ms = 0.0, nvrtc_ms = 0.0;
    uint32_t registers = 0, compile_threads = 0, cache_hit = 0;
    std::string error;
};

struct JitJob {
    std::thread th;
    std::atomic<int> state{0};                // 0 running, 1 built, 2 failed
    std::atomic<bool> cancel{false};          // set by the handle when the result is no longer wanted
    Program prog;                             // the job's own copy
    JitBuild build;
    int rc = 0;
};

struct maray_cuda {
    std::vector<Gpu> gpus;
    std::string error;
    Scene scene;
    bool have_scene = false;
    std::vector<HostTexture> textures;
    bool textures_uploaded = false;
    Program prog;
    bool compiled = false;
    int backend = -1;                   // as asked for: MARAY_BACKEND_*
    bool use_jit = false;               // launches go to the generated kernels (else: to the interpreter)
    bool have_interp = false;           // bytecode compiled (and uploaded when there are GPUs)
    std::vector<void*> imported;        // frames of other processes opened with maray_cuda_frame_import
    std::unique_ptr<JitJob> job;        // MARAY_BACKEND_AUTO: the NVRTC build in flight, or finished and not yet installed
    JitBuild jit;                       // the installed build
    Bytecode bc;
    std::vector<uint64_t> bc_device;                   // bc.code with operand fields scaled for the launch shape
    unsigned interp_block = 128, interp_ppt = 2;       // launch shape: threads per block, pixels per thread
    int libm = MARAY_LIBM_FAST;                        // maray_cuda_set_libm / MARAY_LIBM
    uint32_t samples = 1;                              // maray_cuda_set_samples: s x s samples per pixel
    unsigned jit_block = 256;
    unsigned jit_dyn_smem = 0;                         // dynamic shared memory of the generated kernel
    unsigned jit_maxreg = 0;
    bool jit_chain = false;                            // one kernel per segment, launched in order over a global frame
    unsigned jit_frame_slots = 0;
    maray_cuda_stats stats{};
    int report_kind = MARAY_REPORT_NONE;
    uint32_t report_every = 0;
    maray_report_fn report_fn = nullptr;
    void* report_user = nullptr;
};

namespace {

int fail(maray_cuda* h, int code, const std::string& msg) {
    if (h) h->error = msg; else g_create_error = msg;
    return code;
}

int jit_build(const Program& prog, JitBuild* jb, bool cached_only, const std::atomic<bool>* cancel);
int jit_install(maray_cuda* h, JitBuild&& jb);
int interp_build_and_install(maray_cuda* h);
void fill_jit_stats(maray_cuda* h);

#define CU_TRY(h, expr)                                                                                   \
    do {                                                                                                  \
        cudaError_t e_ = (expr);                                                                          \
        if (e_ != cudaSuccess)                                                                            \
            return fail(h, MARAY_E_CUDA, std::string(#expr) + ": " + cudaGetErrorName(e_) + " (" +       \
                                             cudaGetErrorString(e_) + ")");                               \
    } while (0)

// cancel: the result is no longer wanted (another scene, another back end) -- units not started yet are skipped,
// a unit inside NVRTC runs to its end.  Without cancel (destroy) the build is left to finish, so that its cubins
// reach the cache and the next process starts on the generated kernels.
void stop_job(maray_cuda* h, bool cancel) {
    if (!h->job) return;
    if (cancel) h->job->cancel = true;
    if (h->job->th.joinable()) h->job->th.join();
    h->job.reset();
}

void release_backend(maray_cuda* h, bool cancel_job = true) {
    stop_job(h, cancel_job);
    h->use_jit = false;
    h->have_interp = false;
    for (Gpu& g : h->gpus) {
        cudaSetDevice(g.device);
        for (cudaLibrary_t l : g.libs) cudaLibraryUnload(l);
        g.libs.clear(); g.jit_kernels.clear();
        if (g.d_frame) { cudaFree(g.d_frame); g.d_frame = nullptr; g.frame_cap = 0; }
        if (g.d_code) { cudaFree(g.d_code); g.d_code = nullptr; }
        if (g.d_consts) { cudaFree(g.d_consts); g.d_consts = nullptr; }
    }
    h->compiled = false;
}

void release_textures(maray_cuda* h) {
    for (Gpu& g : h->gpus) {
        cudaSetDevice(g.device);
        for (uint8_t* p : g.d_tex) if (p) cudaFree(p);
        g.d_tex.clear();
        if (g.d_textab) { cudaFree(g.d_textab); g.d_textab = nullptr; }
    }
    h->textures_uploaded = false;
}

int upload_textures(maray_cuda* h) {
    if (h->textures_uploaded || h->gpus.empty()) return MARAY_OK;
    for (Gpu& g : h->gpus) {
        CU_TRY(h, cudaSetDevice(g.device));
        std::vector<MrTexture> tab(h->textures.size());
        g.d_tex.assign(h->textures.size(), nullptr);
        for (size_t i = 0; i < h->textures.size(); i++) {
            const HostTexture& t = h->textures[i];
            size_t bytes = std::max<size_t>(t.rgb.size(), 16);
            CU_TRY(h, cudaMalloc(&g.d_tex[i], bytes));
            if (!t.rgb.empty()) CU_TRY(h, cudaMemcpy(g.d_tex[i], t.rgb.data(), t.rgb.size(), cudaMemcpyHostToDevice));
            tab[i] = MrTexture{g.d_tex[i], t.w, t.h};
        }
        if (!tab.empty()) {
            CU_TRY(h, cudaMalloc(&g.d_textab, tab.size() * sizeof(MrTexture)));
            CU_TRY(h, cudaMemcpy(g.d_textab, tab.data(), tab.size() * sizeof(MrTexture), cudaMemcpyHostToDevice));
        }
    }
    h->textures_uploaded = true;
    return MARAY_OK;
}

// Completion counters of a frame shared between band processes: one 32-bit counter per rank, in the same allocation
// as the frame (the importers have it mapped already), behind the pixels.
constexpr uint32_t kBandCounters = 64;
constexpr uint32_t kBandCounterStride = 32;    // 32-bit words between two counters: one 128-byte line each
inline size_t band_counters_offset(uint32_t w, uint32_t hgt) { return (size_t(w) * hgt * 3 + 255) & ~size_t(255); }
inline unsigned int* band_timeout_word(Gpu& g) { return reinterpret_cast<unsigned int*>(reinterpret_cast<uint8_t*>(g.d_sink) + 128); }

int ensure_out(maray_cuda* h, Gpu& g, size_t bytes) {
    if (g.out_cap >= bytes) return MARAY_OK;
    CU_TRY(h, cudaSetDevice(g.device));
    if (g.d_out) cudaFree(g.d_out);
    g.d_out = nullptr; g.out_cap = 0;
    CU_TRY(h, cudaMalloc(&g.d_out, std::max<size_t>(bytes, 256)));
    g.out_cap = bytes;
    return MARAY_OK;
}

void fill_program_stats(maray_cuda* h) {
    maray_cuda_stats& s = h->stats;
    const ProgramStats& p = h->prog.stats;
    s.tree_nodes = p.tree_nodes; s.dag_nodes = p.dag_nodes;
    s.n_const = p.n_const; s.n_x_only = p.n_x; s.n_y_only = p.n_y; s.n_xy = p.n_xy;
    s.n_add = p.op_count[OP_ADD]; s.n_mul = p.op_count[OP_MUL]; s.n_neg = p.op_count[OP_NEG];
    s.n_abs = p.op_count[OP_ABS]; s.n_recip = p.op_count[OP_RECIP]; s.n_sqrt = p.op_count[OP_SQRT];
    s.n_step = p.op_count[OP_STEP]; s.n_min = p.op_count[OP_MIN]; s.n_max = p.op_count[OP_MAX];
    s.n_sin = p.op_count[OP_SIN]; s.n_exp = p.op_count[OP_EXP]; s.n_ln = p.op_count[OP_LN];
    s.n_tex = p.op_count[OP_TEX];
    s.dag_depth = p.depth;
    s.legacy_layout = h->scene.legacy_layout ? 1 : 0;
}

// ---- NVRTC: source -> sm_100a cubin.  Works without a GPU. ----------------------------------------
//
// Every translation unit is compiled straight to its own cubin; several (the chain form of a large program:
// one kernel per segment) are compiled concurrently, one NVRTC program per host thread, and nothing is
// linked.  Finished cubins are kept in a directory (jit_cache_dir) keyed by the unit's text and the options.

struct UnitResult {
    nvrtcResult rc = NVRTC_SUCCESS;
    std::vector<char> cubin;
    std::string log;
    uint32_t max_registers = 0;   // largest "Used N registers" in the ptxas -v log of the unit
};

void compile_unit(const std::string& source, const std::vector<std::string>& options, UnitResult* out) {
    nvrtcProgram prog;
    out->rc = nvrtcCreateProgram(&prog, source.c_str(), "maray_jit.cu", 0, nullptr, nullptr);
    if (out->rc != NVRTC_SUCCESS) return;
    std::vector<const char*> opts;
    for (const std::string& o : options) opts.push_back(o.c_str());
    out->rc = nvrtcCompileProgram(prog, int(opts.size()), opts.data());
    size_t log_size = 0;
    nvrtcGetProgramLogSize(prog, &log_size);
    out->log.assign(log_size, '\0');
    if (log_size > 1) nvrtcGetProgramLog(prog, &out->log[0]);
    if (out->rc == NVRTC_SUCCESS) {
        size_t n = 0;
        if (nvrtcGetCUBINSize(prog, &n) == NVRTC_SUCCESS && n) {
            out->cubin.resize(n);
            nvrtcGetCUBIN(prog, out->cubin.data());
        } else {
            out->rc = NVRTC_ERROR_INTERNAL_ERROR;
        }
    }
    nvrtcDestroyProgram(&prog);
    for (size_t at = out->log.find("Used "); at != std::string::npos; at = out->log.find("Used ", at + 5)) {
        uint32_t r = uint32_t(std::atoi(out->log.c_str() + at + 5));
        if (out->log.compare(at + 5 + std::to_string(r).size(), 10, " registers") == 0 && r > out->max_registers)
            out->max_registers = r;
    }
}

// 128-bit FNV-1a style key over the generated text and the compile options.
std::string cache_key(const std::string& module, const std::vector<std::string>& options) {
    uint64_t a = 0xcbf29ce484222325ull, b = 0x84222325cbf29ce4ull;
    auto mix = [&](const std::string& t) {
        for (unsigned char c : t) {
            a = (a ^ c) * 0x100000001b3ull;
            b = (b ^ (c + 0x9e)) * 0x00000100000001b5ull;
        }
        a = (a ^ 0xff) * 0x100000001b3ull;
        b = (b ^ 0xfe) * 0x00000100000001b5ull;
    };
    mix(module);
    for (const std::string& o : options) mix(o);
    int major = 0, minor = 0;
    nvrtcVersion(&major, &minor);
    mix("nvrtc " + std::to_string(major) + "." + std::to_string(minor) + " " + maray_cuda_version());
    char buf[40];
    std::snprintf(buf, sizeof buf, "%016llx%016llx", (unsigned long long)a, (unsigned long long)b);
    return buf;
}

struct CacheHeader { char magic[8]; uint32_t registers; uint32_t units; uint64_t cubin_bytes; };
const char kCacheMagic[8] = {'M', 'R', 'C', 'U', 'B', 'I', 'N', '1'};

bool cache_load(const std::string& path, std::vector<char>* cubin, uint32_t* registers) {
    FILE* f = std::fopen(path.c_str(), "rb");
    if (!f) return false;
    CacheHeader hd;
    bool ok = std::fread(&hd, sizeof hd, 1, f) == 1 && std::memcmp(hd.magic, kCacheMagic, 8) == 0 &&
              hd.cubin_bytes > 0 && hd.cubin_bytes < (1ull << 32);
    if (ok) {
        cubin->resize(size_t(hd.cubin_bytes));
        ok = std::fread(cubin->data(), 1, cubin->size(), f) == cubin->size();
        *registers = hd.registers;
    }
    std::fclose(f);
    return ok;
}

void cache_store(const std::string& path, const std::vector<char>& cubin, uint32_t registers, uint32_t units) {
    // several processes may finish the same scene at the same time (one rank per GPU): private temporary names
    std::string tmp = path + ".tmp" + std::to_string((unsigned long long)getpid()) + "_" + std::to_string((unsigned long long)now_ms());
    FILE* f = std::fopen(tmp.c_str(), "wb");
    if (!f) return;
    CacheHeader hd;
    std::memcpy(hd.magic, kCacheMagic, 8);
    hd.registers = registers; hd.units = units; hd.cubin_bytes = cubin.size();
    bool ok = std::fwrite(&hd, sizeof hd, 1, f) == 1 && std::fwrite(cubin.data(), 1, cubin.size(), f) == cubin.size();
    ok = (std::fclose(f) == 0) && ok;
    if (ok) ok = std::rename(tmp.c_str(), path.c_str()) == 0;   // atomic: readers never see a partial file
    if (!ok) std::remove(tmp.c_str());
}

// Where finished cubins are kept.  On by default (the reference compiles per render, src/wasm.rs:136-158,
// and NVRTC is ~1 ms per value): $MARAY_JIT_CACHE, else $XDG_CACHE_HOME/maray_b200, else ~/.cache/maray_b200.
// MARAY_JIT_CACHE set to "", "0" or "off" turns it off.  Returns "" when there is no usable directory.
std::string jit_cache_dir() {
    std::string dir;
    if (const char* e = std::getenv("MARAY_JIT_CACHE")) {
        dir = e;
        if (dir.empty() || dir == "0" || dir == "off") return "";
    } else if (const char* x = std::getenv("XDG_CACHE_HOME"); x && *x) {
        dir = std::string(x) + "/maray_b200";
    } else if (const char* hm = std::getenv("HOME"); hm && *hm) {
        dir = std::string(hm) + "/.cache/maray_b200";
    } else {
        return "";
    }
    // mkdir -p (the last two levels are enough for the defaults)
    for (size_t at = dir.find('/', 1); ; at = dir.find('/', at + 1)) {
        std::string part = at == std::string::npos ? dir : dir.substr(0, at);
        if (!part.empty()) ::mkdir(part.c_str(), 0755);
        if (at == std::string::npos) break;
    }
    struct stat sb;
    if (::stat(dir.c_str(), &sb) != 0 || !S_ISDIR(sb.st_mode) || ::access(dir.c_str(), W_OK) != 0) return "";
    return dir;
}

int nvrtc_compile(JitBuild* jb, const std::atomic<bool>* cancel, bool cached_only) {
    const size_t n_units = jb->modules.size();
    std::vector<std::string> options = {
        "--gpu-architecture=sm_100a",
        "--fmad=false",               // the reference never fuses a*b+c
        "--std=c++17",
        "--ptxas-options=-v",
        "--diag-suppress=177",        // unused double shadows of boolean values: dead code by design
    };
    // Line tables map SASS to the generated text (ncu source page).
    bool lineinfo = true;
    if (const char* e = std::getenv("MARAY_JIT_LINEINFO")) lineinfo = std::strtoul(e, nullptr, 10) != 0;
    if (lineinfo) options.push_back("-lineinfo");
    if (jb->maxreg) options.push_back("--maxrregcount=" + std::to_string(jb->maxreg));
    if (jb->libm == MARAY_LIBM_CUDA) options.push_back("-DMR_LIBM_PLAIN=1");    // A/B: libdevice's sin/exp/log
    if (jb->libm == MARAY_LIBM_GLIBC) options.push_back("-DMR_LIBM_GLIBC=1");   // exact mode (device_libm_glibc.cuh)

    jb->registers = 0;
    jb->compile_threads = 0;
    jb->cache_hit = 0;
    jb->cubins.assign(n_units, {});

    // cache: per unit, so an edit that changes one segment recompiles one segment
    const std::string cache_dir = jit_cache_dir();
    std::vector<std::string> cache_path(n_units);
    std::vector<size_t> todo;
    for (size_t i = 0; i < n_units; i++) {
        uint32_t regs = 0;
        if (!cache_dir.empty()) {
            cache_path[i] = cache_dir + "/" + cache_key(jb->modules[i], options) + ".mrcubin";
            if (cache_load(cache_path[i], &jb->cubins[i], &regs)) {
                jb->registers = std::max(jb->registers, regs);
                continue;
            }
        }
        todo.push_back(i);
    }
    if (todo.empty()) { jb->cache_hit = 1; return MARAY_OK; }
    if (cached_only) { jb->error = "not every unit is in the cubin cache"; return MARAY_E_COMPILE; }

    std::vector<UnitResult> res(n_units);
    unsigned n_threads = std::thread::hardware_concurrency();
    if (const char* e = std::getenv("MARAY_JIT_THREADS")) n_threads = unsigned(std::strtoul(e, nullptr, 10));
    n_threads = std::max(1u, std::min<unsigned>(n_threads, unsigned(todo.size())));
    jb->compile_threads = n_threads;
    if (n_threads == 1) {
        for (size_t i : todo) {
            if (cancel && *cancel) { jb->error = "compile cancelled"; return MARAY_E_COMPILE; }
            compile_unit(jb->modules[i], options, &res[i]);
        }
    } else {
        std::atomic<size_t> next{0};
        std::vector<std::thread> pool;
        for (unsigned t = 0; t < n_threads; t++)
            pool.emplace_back([&] {
                for (size_t k = next.fetch_add(1); k < todo.size(); k = next.fetch_add(1)) {
                    if (cancel && *cancel) { res[todo[k]].rc = NVRTC_ERROR_INTERNAL_ERROR; res[todo[k]].log = "error: compile cancelled"; continue; }
                    compile_unit(jb->modules[todo[k]], options, &res[todo[k]]);
                }
            });
        for (std::thread& t : pool) t.join();
    }
    for (size_t i : todo) {
        if (res[i].rc != NVRTC_SUCCESS) {
            // the diagnostics that matter first: a long log of warnings must not push the errors out of the message
            std::string log, rest;
            size_t pos = 0;
            int keep = 0;
            while (pos < res[i].log.size()) {
                size_t nl = res[i].log.find('\n', pos);
                if (nl == std::string::npos) nl = res[i].log.size();
                std::string line = res[i].log.substr(pos, nl - pos);
                if (line.find("error") != std::string::npos) keep = 3;      // the line and the source excerpt after it
                ((keep > 0) ? log : rest) += line + "\n";
                if (keep > 0) keep--;
                pos = nl + 1;
            }
            log += rest;
            if (log.size() > 4000) log.resize(4000);
            jb->error = "NVRTC (unit " + std::to_string(i) + "): " + nvrtcGetErrorString(res[i].rc) + "\n" + log;
            return MARAY_E_COMPILE;
        }
        if (std::getenv("MARAY_JIT_VERBOSE")) std::fprintf(stderr, "%s\n", res[i].log.c_str());
        // registers of the kernel from the ptxas -v log: "Function properties for maray_jit" ... "Used N registers"
        uint32_t regs = res[i].max_registers;
        const std::string& log = res[i].log;
        size_t at = log.find(std::string("Function properties for ") + kJitKernelName);
        if (at != std::string::npos) {
            size_t u = log.find("Used ", at);
            if (u != std::string::npos) regs = uint32_t(std::atoi(log.c_str() + u + 5));
        }
        jb->registers = std::max(jb->registers, regs);
        jb->cubins[i] = std::move(res[i].cubin);
        if (!cache_path[i].empty()) cache_store(cache_path[i], jb->cubins[i], regs, 1);
    }
    return MARAY_OK;
}

// Interpreter launch shape.  The per-thread slot file (n_wide * P * 8 bytes) bounds how many warps an SM
// holds, and one bytecode instruction is a chain of dependent shared-memory, branch and FP64 latencies, so
// throughput follows the number of pixels in flight per SM: resident warps x P, with diminishing returns
// on both (measured sweeps: profiles/r02_interp_sweeps.md).  Blocks of any multiple of 32 threads are
// considered: fewer, larger blocks spend less shared memory on the per-block parts (instruction chunks,
// scalar file, staging tile) and so hold more warps.
void choose_interp_shape(maray_cuda* h) {
    const unsigned n_scal = unsigned(h->bc.consts.size()) + h->bc.n_uniform;
    auto fits = [&](unsigned b, unsigned p) {
        return interp_smem_bytes(b, p, h->bc.n_wide, n_scal) <= 227 * 1024 && uint64_t(h->bc.n_wide + 3) * (p * b / 2) <= 0xffff;
    };
    if (const char* e = std::getenv("MARAY_INTERP_SHAPE")) {   // "block,pixels_per_thread" (tuning)
        unsigned b = 0, p = 0;
        if (std::sscanf(e, "%u,%u", &b, &p) == 2 && b % 32 == 0 && b >= 32 && b <= 512 && (p == 1 || p == 2 || p == 4) && fits(b, p)) {
            h->interp_block = b; h->interp_ppt = p;
            return;
        }
    }
    h->interp_block = 0;   // does not fit
    double best = -1.0;
    const unsigned ppts[] = {2, 4, 1};
    for (unsigned p : ppts)
        for (unsigned b = 32; b <= 512; b += 32) {
            if (!fits(b, p)) continue;
            const size_t per_block = interp_smem_bytes(b, p, h->bc.n_wide, n_scal) + 1024;   // + the per-block reservation
            const unsigned resident = unsigned(std::min<size_t>(size_t(228) * 1024 / per_block, std::min<size_t>(32, 2048 / b)));
            const double warps = double(resident) * b / 32.0;
            // lanes past the end of a row idle: count the row width the scene was authored for
            const unsigned span = b * p, sw = std::max<unsigned>(h->scene.size[0], 1);
            const double row_fill = double(sw) / (double((sw + span - 1) / span) * span);
            // measured (profiles/r02_interp_sweeps.md): throughput follows resident warps up to ~24 per SM, and
            // P pixels per thread amortise the dispatch a little less than linearly
            const double score = std::min(warps, 24.0) * std::pow(double(p), 0.85) * row_fill - 0.001 * b;
            if (score > best) { best = score; h->interp_block = b; h->interp_ppt = p; }
        }
}

// ---- building and installing the two back ends ------------------------------------------------------

// Code generation + NVRTC for `prog` (tuning knobs from the environment, DESIGN.md "Knobs").  cached_only: succeed
// only if every unit's cubin is already in the cache directory (nothing is compiled).
int jit_build(const Program& prog, JitBuild* jb, bool cached_only, const std::atomic<bool>* cancel) {
    double t1 = now_ms();
    CodegenOptions copt;
    // Exact mode: the routines branch on ranges and read tables -- always out of line (inlined, chess.maray's 256 sines
    // are 5.7 MB of code and 53 s of NVRTC here instead of 1.7 MB / 11 s).
    if (jb->libm == MARAY_LIBM_GLIBC) copt.inline_transcendentals_below = 0;
    copt.frame_pixels_hint = jb->frame_pixels;
    copt.sm_count_hint = jb->sms ? jb->sms : 148;
    if (const char* e = std::getenv("MARAY_JIT_SEGMENT_VALUES")) copt.segment_values = uint32_t(std::strtoul(e, nullptr, 10));
    if (const char* e = std::getenv("MARAY_JIT_INLINE_TRANS_BELOW")) copt.inline_transcendentals_below = uint32_t(std::strtoul(e, nullptr, 10));
    if (const char* e = std::getenv("MARAY_JIT_CONST_BANK")) copt.constants_in_bank = std::strtoul(e, nullptr, 10) != 0;
    if (const char* e = std::getenv("MARAY_JIT_BOOLEAN")) copt.boolean_logic = std::strtoul(e, nullptr, 10) != 0;
    if (const char* e = std::getenv("MARAY_JIT_SIGN_OF_SINE")) copt.sign_of_sine = std::strtoul(e, nullptr, 10) != 0;
    if (const char* e = std::getenv("MARAY_JIT_BLOCK")) { copt.block = uint32_t(std::strtoul(e, nullptr, 10)); copt.auto_shape = false; }
    if (const char* e = std::getenv("MARAY_JIT_MIN_BLOCKS")) { copt.min_blocks_per_sm = uint32_t(std::strtoul(e, nullptr, 10)); copt.auto_shape = false; }
    jb->maxreg = 0;
    if (const char* e = std::getenv("MARAY_JIT_MAXREG")) jb->maxreg = unsigned(std::strtoul(e, nullptr, 10));
    // Programs above the segment size compile as a CHAIN of kernels, one translation unit each (codegen.hpp):
    // the units compile concurrently on all host cores and nothing is linked.  MARAY_JIT_CHAIN=0 gives round
    // 1's form (segment functions in one unit).  sin/exp/ln stay out of line above the threshold:
    // inlined, the code of a transcendental-heavy program is several MB of instructions no warp ever re-uses
    // and the kernel becomes instruction-fetch bound (measured: 33.8 ms inlined vs 18.7 ms out of line on the
    // 20 000-value deep scene, no_instruction stalls 9.1 per issued instruction; profiles/).
    if (const char* e = std::getenv("MARAY_JIT_CHAIN")) copt.chain = std::strtoul(e, nullptr, 10) != 0;
    if (const char* e = std::getenv("MARAY_JIT_CHAIN_SEGMENT_VALUES")) copt.chain_segment_values = uint32_t(std::strtoul(e, nullptr, 10));
    jb->modules = generate_cuda_modules(prog, copt, &jb->info);
    if (jb->modules.size() > 1) {
        CodegenInfo unused;
        jb->source = generate_cuda_source(prog, copt, &unused);   // the same statements as ONE unit (tooling, tests)
    } else {
        jb->source = jb->modules[0];
    }
    jb->codegen_ms = now_ms() - t1;
    if (std::getenv("MARAY_JIT_SOURCE_ONLY")) {   // tooling: inspect the generated text without paying for NVRTC
        jb->error = "MARAY_JIT_SOURCE_ONLY is set: source generated, not compiled";
        return MARAY_E_COMPILE;
    }
    double t2 = now_ms();
    int rc = nvrtc_compile(jb, cancel, cached_only);
    jb->nvrtc_ms = now_ms() - t2;
    return rc;
}

void fill_jit_stats(maray_cuda* h) {
    const JitBuild& jb = h->jit;
    h->stats.codegen_ms = jb.codegen_ms;
    h->stats.nvrtc_ms = jb.nvrtc_ms;
    h->stats.jit_segments = jb.info.segments;
    h->stats.jit_frame_slots = jb.info.frame_slots;
    h->stats.jit_source_bytes = uint32_t(jb.source.size());
    h->stats.jit_units = uint32_t(jb.modules.size());
    h->stats.jit_compile_threads = jb.compile_threads;
    h->stats.jit_cache_hit = jb.cache_hit;
    h->stats.jit_registers = jb.registers;
    h->stats.jit_block = jb.info.block;
    h->stats.jit_round_pixels = 0;
    h->stats.jit_cubin_bytes = 0;
    for (const std::vector<char>& c : jb.cubins) h->stats.jit_cubin_bytes += uint32_t(c.size());
}

// Makes a finished build the handle's: loads the cubins on every GPU and routes launches to the kernels.
int jit_install(maray_cuda* h, JitBuild&& jb) {
    h->jit = std::move(jb);
    h->jit_block = h->jit.info.block;
    h->jit_dyn_smem = h->jit.info.dynamic_smem_bytes;
    h->jit_chain = h->jit.info.chain;
    h->jit_frame_slots = h->jit.info.frame_slots;
    fill_jit_stats(h);
    double t3 = now_ms();
    for (Gpu& g : h->gpus) {
        CU_TRY(h, cudaSetDevice(g.device));
        h->stats.jit_registers = 0;
        for (const std::vector<char>& cubin : h->jit.cubins) {
            cudaLibrary_t lib = nullptr;
            cudaKernel_t kern = nullptr;
            CU_TRY(h, cudaLibraryLoadData(&lib, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0));
            g.libs.push_back(lib);
            CU_TRY(h, cudaLibraryGetKernel(&kern, lib, kJitKernelName));
            g.jit_kernels.push_back(kern);
            cudaFuncAttributes fa;
            if (cudaFuncGetAttributes(&fa, reinterpret_cast<const void*>(kern)) == cudaSuccess) {
                h->stats.jit_registers = std::max(h->stats.jit_registers, uint32_t(fa.numRegs));
                // Shared-memory carve-out: no more than the resident blocks use, the rest of the 256 KB is L1.  Left to
                // itself the driver sizes it for the shared-memory occupancy limit (132 KB for the 33 KB scratch kernels,
                // whose registers allow two blocks), and the spilled values of a large program then miss in a 121 KB L1.
                const unsigned regs = std::max(1, fa.numRegs), blk = std::max(1u, h->jit_block);
                const size_t smem_per_block = h->jit_dyn_smem + fa.sharedSizeBytes + 1024;
                unsigned blocks = std::min(std::min(65536u / ((regs + 7) / 8 * 8 * blk), 2048u / blk), 32u);
                blocks = std::max(1u, std::min<unsigned>(blocks, unsigned(233472 / smem_per_block)));      // resident blocks per SM
                if (&g == &h->gpus[0] && &cubin == &h->jit.cubins[0]) h->stats.jit_round_pixels = uint32_t(g.sms) * blocks * blk;
                int pct = -1;
                if (const char* e = std::getenv("MARAY_JIT_CARVEOUT")) pct = int(std::strtol(e, nullptr, 10));   // percent; -1 = computed, -2 = driver's choice
                if (pct == -1) {
                    const size_t need = size_t(blocks) * smem_per_block;
                    static const unsigned kConfigKb[] = {0, 8, 16, 32, 64, 100, 132, 164, 196, 228};   // sm_100 carve-outs
                    size_t cfg = 228;
                    for (unsigned kb : kConfigKb) if (size_t(kb) * 1024 >= need) { cfg = kb; break; }
                    pct = int(std::min<size_t>(100, (cfg * 1024 * 100 + 233471) / 233472));   // rounded up: never below the configuration that holds the blocks
                }
                if (pct >= 0 && cudaFuncSetAttribute(reinterpret_cast<const void*>(kern), cudaFuncAttributePreferredSharedMemoryCarveout, pct) != cudaSuccess)
                    cudaGetLastError();
            } else cudaGetLastError();
        }
    }
    if (!h->gpus.empty()) cudaSetDevice(h->gpus[0].device);
    h->stats.load_ms += now_ms() - t3;
    h->use_jit = true;
    return MARAY_OK;
}

// Bytecode + launch shape + upload: the interpreter back end is ready when this returns.
int interp_build_and_install(maray_cuda* h) {
    double t1 = now_ms();
    std::string err;
    // Row-uniform form by default; the all-wide form when the scalar file would crowd out the slot file
    // (or MARAY_INTERP_UNIFORM=0, for A/B).
    bool uniform = true;
    if (const char* e = std::getenv("MARAY_INTERP_UNIFORM")) uniform = std::strtoul(e, nullptr, 10) != 0;
    if (!compile_bytecode(h->prog, &h->bc, &err, uniform)) return fail(h, MARAY_E_COMPILE, err);
    if (uniform && h->bc.n_uniform > 4096 && !compile_bytecode(h->prog, &h->bc, &err, false)) return fail(h, MARAY_E_COMPILE, err);
    choose_interp_shape(h);
    if (!h->interp_block)
        return fail(h, MARAY_E_UNSUPPORTED, "program needs " + std::to_string(h->bc.n_wide) +
                                                " live values per pixel, more than the interpreter's shared-memory slot file holds");
    h->bc_device = bytecode_for_launch(h->bc, h->interp_block * h->interp_ppt / 2, &err);
    if (h->bc_device.empty()) return fail(h, MARAY_E_UNSUPPORTED, err);
    if (h->backend == MARAY_BACKEND_INTERP) h->stats.codegen_ms = now_ms() - t1;
    h->stats.interp_instructions = uint32_t(h->bc.code.size());
    h->stats.interp_slots = h->bc.n_wide;
    h->stats.interp_uniform_slots = h->bc.n_uniform;
    h->stats.interp_block = h->interp_block;
    h->stats.interp_pixels_per_thread = h->interp_ppt;
    double t3 = now_ms();
    for (Gpu& g : h->gpus) {
        CU_TRY(h, cudaSetDevice(g.device));
        CU_TRY(h, cudaMalloc(&g.d_code, h->bc_device.size() * sizeof(uint64_t)));
        CU_TRY(h, cudaMemcpy(g.d_code, h->bc_device.data(), h->bc_device.size() * sizeof(uint64_t), cudaMemcpyHostToDevice));
        CU_TRY(h, cudaMalloc(&g.d_consts, h->bc.consts.size() * sizeof(double)));
        CU_TRY(h, cudaMemcpy(g.d_consts, h->bc.consts.data(), h->bc.consts.size() * sizeof(double), cudaMemcpyHostToDevice));
    }
    if (!h->gpus.empty()) cudaSetDevice(h->gpus[0].device);
    h->stats.load_ms += now_ms() - t3;
    h->have_interp = true;
    return MARAY_OK;
}

// MARAY_BACKEND_AUTO: if the background build has finished, make it the handle's.  Called between row chunks.
int adopt_finished_job(maray_cuda* h) {
    if (!h->job || h->job->state.load() == 0) return MARAY_OK;
    if (h->job->th.joinable()) h->job->th.join();
    std::unique_ptr<JitJob> job = std::move(h->job);
    if (job->state.load() != 1) return MARAY_OK;          // the build failed: stay on the interpreter (its error is in stats' absence)
    return jit_install(h, std::move(job->build));
}

// One pass of the kernels over pixels p0 .. p0+n-1.  sp: the pass's sampling state (zero: one sample per pixel), its
// accumulator, if any, already offset to pixel p0.
int launch_pass(maray_cuda* h, Gpu& g, uint32_t w, uint32_t p0, uint32_t n, uint8_t* d_out, double* d_f64,
                size_t f64_plane, cudaStream_t stream, const MrSampling& sp) {
    MrParams p{};
    p.out = d_out; p.f64_out = d_f64; p.f64_plane = f64_plane; p.tex = g.d_textab;
    p.p0 = p0; p.n = n; p.W = w;
    p.out_aligned = (reinterpret_cast<uintptr_t>(d_out) % 16 == 0) ? 1u : 0u;
    if (n == 0) return MARAY_OK;
    if (h->use_jit) {
        if (!h->jit_chain) {
            MrSampling a = sp;
            void* args[] = {&p, &a};
            const unsigned grid = (n + h->jit_block - 1) / h->jit_block;
            CU_TRY(h, cudaLaunchKernel(reinterpret_cast<const void*>(g.jit_kernels[0]), dim3(grid), dim3(h->jit_block), args, h->jit_dyn_smem, stream));
        } else {
            // Chain form: the segment kernels run in order over a chunk of pixels whose frame (values that cross
            // a cut, F[slot * FS + pixel]) fits the budget; chunks follow each other on the stream.
            size_t budget = size_t(2) << 30;
            if (const char* e = std::getenv("MARAY_JIT_FRAME_MB")) budget = std::max<size_t>(1, std::strtoull(e, nullptr, 10)) << 20;
            const size_t per_px = std::max<size_t>(h->jit_frame_slots, 1) * sizeof(double);
            size_t chunk = std::max<size_t>(budget / per_px, h->jit_block);
            chunk = std::min<size_t>(chunk / h->jit_block * h->jit_block, (size_t(n) + h->jit_block - 1) / h->jit_block * h->jit_block);
            // One frame per GPU: a band issued on another stream must not overwrite it while the previous band's
            // kernels still use it (maray_cuda_render_band takes any stream), so launches that use it are serialised.
            if (!g.frame_done) CU_TRY(h, cudaEventCreateWithFlags(&g.frame_done, cudaEventDisableTiming));
            else CU_TRY(h, cudaStreamWaitEvent(stream, g.frame_done, 0));
            if (g.frame_cap < chunk * per_px) {
                if (g.d_frame) cudaFree(g.d_frame);
                g.d_frame = nullptr; g.frame_cap = 0;
                CU_TRY(h, cudaMalloc(&g.d_frame, chunk * per_px));
                g.frame_cap = chunk * per_px;
            }
            unsigned long long fs = chunk;
            static const bool poison = std::getenv("MARAY_JIT_FRAME_POISON") != nullptr;   // debugging: a value read before it is written is a NaN
            for (size_t done = 0; done < n; done += chunk) {
                if (poison) CU_TRY(h, cudaMemsetAsync(g.d_frame, 0xff, g.frame_cap, stream));
                MrParams q = p;
                q.p0 = p0 + uint32_t(done);
                q.n = uint32_t(std::min<size_t>(chunk, n - done));
                q.out = d_out + 3 * done;
                q.out_aligned = (reinterpret_cast<uintptr_t>(q.out) % 16 == 0) ? 1u : 0u;
                if (d_f64) q.f64_out = d_f64 + done;
                MrSampling a = sp;
                if (a.acc) a.acc += 3 * done;
                void* args[] = {&q, &g.d_frame, &fs, &a};
                unsigned grid = (q.n + h->jit_block - 1) / h->jit_block;
                for (cudaKernel_t k : g.jit_kernels)
                    CU_TRY(h, cudaLaunchKernel(reinterpret_cast<const void*>(k), dim3(grid), dim3(h->jit_block), args, h->jit_dyn_smem, stream));
            }
            CU_TRY(h, cudaEventRecord(g.frame_done, stream));
        }
    } else {
        // The interpreter renders windows [x0,x1) x rows with every block inside one row: a linear pixel range
        // is at most a partial first row, whole rows, and a partial last row.
        uint32_t left = n, pix = p0;
        size_t done = 0;
        while (left) {
            const uint32_t y = pix / w, x = pix - y * w;
            uint32_t cols, rows;
            if (x != 0 || left < w) { cols = std::min(left, w - x); rows = 1; }
            else { cols = w; rows = left / w; }
            MrTileParams t;
            t.out = d_out + 3 * done;
            t.f64_out = d_f64 ? d_f64 + done : nullptr;
            t.f64_plane = f64_plane;
            t.tex = g.d_textab;
            t.x0 = x; t.x1 = x + cols; t.y0 = y; t.rows = rows; t.nxb = 0;
            t.out_aligned = (reinterpret_cast<uintptr_t>(t.out) % 16 == 0) ? 1u : 0u;
            t.libm_exact = h->libm == MARAY_LIBM_GLIBC ? 1u : 0u;
            t.ox = sp.ox; t.oy = sp.oy;
            t.acc = sp.acc ? sp.acc + 3 * done : nullptr;
            t.pass = sp.pass; t.count = sp.count;
            CU_TRY(h, launch_interp(t, g.d_code, unsigned(h->bc_device.size()), g.d_consts, unsigned(h->bc.consts.size()),
                                    h->bc.n_uniform, h->bc.n_wide, !h->bc.row_uniform, h->interp_block, h->interp_ppt, stream));
            const uint32_t count = cols * rows;
            done += count; pix += count; left -= count;
        }
    }
    return MARAY_OK;
}

// Offset of sample k of s along one axis: the centres of an s x s grid over the pixel footprint [xi - 1/2, xi + 1/2).
double sample_offset(uint32_t k, uint32_t s) { return double(int(2 * k + 1) - int(s)) * (1.0 / (2.0 * double(s))); }

int ensure_acc(maray_cuda* h, Gpu& g, size_t pixels) {
    if (g.acc_cap >= pixels) return MARAY_OK;
    CU_TRY(h, cudaSetDevice(g.device));
    if (g.d_acc) cudaFree(g.d_acc);   // synchronises: no pass that still uses the old buffer is left running
    g.d_acc = nullptr; g.acc_cap = 0;
    CU_TRY(h, cudaMalloc(&g.d_acc, pixels * 3 * sizeof(uint16_t)));
    g.acc_cap = pixels;
    return MARAY_OK;
}

// Renders pixels p0 .. p0+n-1 of a w-wide frame into d_out: every render path comes through here.  With s x s samples
// per pixel (maray_cuda_set_samples) that is s*s passes in order on `stream`, each at one sub-pixel offset; the last
// resolves the accumulator into RGB8.  The accumulator is indexed by the pixel's index in the frame, so launches on
// disjoint pixel ranges (row chunks on several streams, bands) never share a word.
int launch_band(maray_cuda* h, Gpu& g, uint32_t w, uint32_t p0, uint32_t n, uint8_t* d_out, double* d_f64,
                size_t f64_plane, cudaStream_t stream) {
    const uint32_t s = h->samples;
    if (s <= 1 || n == 0) return launch_pass(h, g, w, p0, n, d_out, d_f64, f64_plane, stream, MrSampling{});
    int rc = ensure_acc(h, g, size_t(p0) + n);
    if (rc) return rc;
    MrSampling sp{};
    sp.acc = g.d_acc + 3 * size_t(p0);
    sp.count = s * s;
    for (uint32_t jy = 0; jy < s; jy++)
        for (uint32_t ix = 0; ix < s; ix++) {
            sp.ox = sample_offset(ix, s);
            sp.oy = sample_offset(jy, s);
            sp.pass = jy * s + ix;
            rc = launch_pass(h, g, w, p0, n, d_out, d_f64, f64_plane, stream, sp);
            if (rc) return rc;
        }
    return MARAY_OK;
}

int check_renderable(maray_cuda* h, uint32_t w, uint32_t hgt) {
    if (!h) return MARAY_E_INVALID;
    if (!h->compiled) return fail(h, MARAY_E_INVALID, "render called before maray_cuda_compile");
    if (h->gpus.empty()) return fail(h, MARAY_E_CUDA, "host-only handle (created with 0 GPUs): there is no CPU fallback");
    if (w == 0 || hgt == 0) return fail(h, MARAY_E_INVALID, "empty image");
    if (uint64_t(w) * hgt > 0xffffffffull) return fail(h, MARAY_E_INVALID, "image has more than 2^32-1 pixels");
    return MARAY_OK;
}

// Renders rows [ya, yb) of the w x hgt frame into GPU 0's frame buffer (device), banded over GPUs.
int render_rows_to_frame(maray_cuda* h, uint32_t w, uint32_t hgt, uint32_t ya, uint32_t yb) {
    (void)hgt;
    const size_t G = h->gpus.size();
    const uint32_t rows = yb - ya;
    Gpu& g0 = h->gpus[0];
    std::vector<uint32_t> b0(G + 1);
    for (size_t g = 0; g <= G; g++) b0[g] = ya + uint32_t(uint64_t(rows) * g / G);
    for (size_t gi = 0; gi < G; gi++) {
        Gpu& g = h->gpus[gi];
        uint32_t y0 = b0[gi], y1 = b0[gi + 1];
        size_t bytes = size_t(y1 - y0) * w * 3;
        CU_TRY(h, cudaSetDevice(g.device));
        uint8_t* dst;
        if (gi == 0) dst = g0.d_out + size_t(y0) * w * 3;
        else {
            int rc = ensure_out(h, g, bytes);
            if (rc) return rc;
            dst = g.d_out;
        }
        CU_TRY(h, cudaEventRecord(g.ev0, g.stream));
        int rc = launch_band(h, g, w, y0 * w, (y1 - y0) * w, dst, nullptr, 0, g.stream);
        if (rc) return rc;
        CU_TRY(h, cudaEventRecord(g.ev1, g.stream));
        if (gi != 0 && bytes)
            CU_TRY(h, cudaMemcpyPeerAsync(g0.d_out + size_t(y0) * w * 3, g0.device, g.d_out, g.device, bytes, g.stream));
    }
    double t_gather0 = now_ms();
    for (size_t gi = 0; gi < G; gi++) {
        Gpu& g = h->gpus[gi];
        CU_TRY(h, cudaSetDevice(g.device));
        CU_TRY(h, cudaStreamSynchronize(g.stream));
        float ms = 0.f;
        CU_TRY(h, cudaEventElapsedTime(&ms, g.ev0, g.ev1));
        if (gi < 8) h->stats.kernel_ms[gi] += ms;
    }
    (void)t_gather0;
    CU_TRY(h, cudaSetDevice(g0.device));
    return MARAY_OK;
}

// One GPU, frame wanted in host memory, no progress callback: the rows are rendered in kChunks launches
// on kChunks streams (the tail of one chunk's grid overlaps the head of the next, so cutting the frame
// costs no wave quantisation) and every chunk is copied out on a separate stream as soon as it is done,
// while later chunks still render.  What remains exposed of the device->host copy is the last chunk.
int render_frame_pipelined(maray_cuda* h, uint32_t w, uint32_t hgt, uint8_t* host_rgb) {
    Gpu& g = h->gpus[0];
    CU_TRY(h, cudaSetDevice(g.device));
    if (!g.copy_stream) {
        CU_TRY(h, cudaStreamCreateWithFlags(&g.copy_stream, cudaStreamNonBlocking));
        for (int c = 0; c < Gpu::kChunks; c++) {
            CU_TRY(h, cudaStreamCreateWithFlags(&g.chunk_stream[c], cudaStreamNonBlocking));
            CU_TRY(h, cudaEventCreateWithFlags(&g.chunk_done[c], cudaEventDisableTiming));
        }
    }
    // chunk boundaries on multiples of 16 rows: every chunk starts 16-byte aligned in the frame
    uint32_t y[Gpu::kChunks + 1];
    for (int c = 0; c <= Gpu::kChunks; c++) y[c] = std::min<uint32_t>(hgt, ((uint64_t(hgt) * c / Gpu::kChunks) + 15u) & ~15u);
    y[0] = 0; y[Gpu::kChunks] = hgt;
    CU_TRY(h, cudaEventRecord(g.ev0, g.stream));
    for (int c = 0; c < Gpu::kChunks; c++) {
        if (y[c + 1] <= y[c]) continue;
        CU_TRY(h, cudaStreamWaitEvent(g.chunk_stream[c], g.ev0, 0));
        int rc = launch_band(h, g, w, y[c] * w, (y[c + 1] - y[c]) * w, g.d_out + size_t(y[c]) * w * 3, nullptr, 0, g.chunk_stream[c]);
        if (rc) return rc;
        CU_TRY(h, cudaEventRecord(g.chunk_done[c], g.chunk_stream[c]));
        CU_TRY(h, cudaStreamWaitEvent(g.stream, g.chunk_done[c], 0));
    }
    CU_TRY(h, cudaEventRecord(g.ev1, g.stream));          // all chunks rendered
    double t1 = now_ms();
    for (int c = 0; c < Gpu::kChunks; c++) {
        if (y[c + 1] <= y[c]) continue;
        CU_TRY(h, cudaStreamWaitEvent(g.copy_stream, g.chunk_done[c], 0));
        CU_TRY(h, cudaMemcpyAsync(host_rgb + size_t(y[c]) * w * 3, g.d_out + size_t(y[c]) * w * 3,
                                  size_t(y[c + 1] - y[c]) * w * 3, cudaMemcpyDeviceToHost, g.copy_stream));
    }
    CU_TRY(h, cudaStreamSynchronize(g.copy_stream));
    CU_TRY(h, cudaStreamSynchronize(g.stream));
    float ms = 0.f;
    CU_TRY(h, cudaEventElapsedTime(&ms, g.ev0, g.ev1));
    h->stats.kernel_ms[0] = ms;
    h->stats.d2h_ms = std::max(0.0, (now_ms() - t1) - double(ms));   // what the copies added after the last kernel
    return MARAY_OK;
}

// MARAY_BACKEND_AUTO while NVRTC is still at work: the interpreter renders row chunks of ~30 ms; between
// chunks the finished build is adopted, and the rest of the frame goes to the generated kernels in one piece.
int render_frame_tiered(maray_cuda* h, uint32_t w, uint32_t hgt) {
    uint32_t ya = 0, rows = 8;
    h->stats.tier_rows_interp = 0;
    while (ya < hgt) {
        int rc = adopt_finished_job(h);
        if (rc) return rc;
        if (h->use_jit) return render_rows_to_frame(h, w, hgt, ya, hgt);
        const uint32_t yb = std::min(hgt, ya + rows);
        double t0 = now_ms();
        rc = render_rows_to_frame(h, w, hgt, ya, yb);     // synchronises
        if (rc) return rc;
        const double ms = std::max(now_ms() - t0, 0.01);
        h->stats.tier_rows_interp += yb - ya;
        rows = uint32_t(std::min<double>(std::max<double>(double(yb - ya) * 30.0 / ms, 1.0), 4096.0));
        ya = yb;
    }
    return MARAY_OK;
}

// Several GPUs, frame wanted in host memory: every GPU renders its row band into its own buffer and copies it
// straight into the caller's image over its own PCIe link, one host thread per GPU (a pageable destination
// makes the copy call synchronous, so the threads are what lets the copies overlap).  No gather: bands only
// have to meet in GPU 0's memory when the frame is to stay on the device (render_rows_to_frame).
int render_frame_bands_to_host(maray_cuda* h, uint32_t w, uint32_t hgt, uint8_t* host_rgb) {
    const size_t G = h->gpus.size();
    std::vector<int> rcs(G, MARAY_OK);
    std::vector<float> kms(G, 0.f);
    std::vector<double> copy_ms(G, 0.0);
    std::vector<std::thread> pool;
    for (size_t gi = 0; gi < G; gi++)
        pool.emplace_back([&, gi] {
            Gpu& g = h->gpus[gi];
            const uint32_t y0 = uint32_t(uint64_t(hgt) * gi / G), y1 = uint32_t(uint64_t(hgt) * (gi + 1) / G);
            const size_t bytes = size_t(y1 - y0) * w * 3;
            if (!bytes) return;
            auto body = [&]() -> int {
                CU_TRY(h, cudaSetDevice(g.device));
                int rc = ensure_out(h, g, gi == 0 ? size_t(w) * hgt * 3 : bytes);
                if (rc) return rc;
                uint8_t* dst = gi == 0 ? g.d_out + size_t(y0) * w * 3 : g.d_out;
                CU_TRY(h, cudaEventRecord(g.ev0, g.stream));
                rc = launch_band(h, g, w, y0 * w, (y1 - y0) * w, dst, nullptr, 0, g.stream);
                if (rc) return rc;
                CU_TRY(h, cudaEventRecord(g.ev1, g.stream));
                CU_TRY(h, cudaStreamSynchronize(g.stream));
                double t1 = now_ms();
                CU_TRY(h, cudaMemcpy(host_rgb + size_t(y0) * w * 3, dst, bytes, cudaMemcpyDeviceToHost));
                copy_ms[gi] = now_ms() - t1;
                CU_TRY(h, cudaEventElapsedTime(&kms[gi], g.ev0, g.ev1));
                return MARAY_OK;
            };
            rcs[gi] = body();
        });
    for (std::thread& t : pool) t.join();
    cudaSetDevice(h->gpus[0].device);
    for (size_t gi = 0; gi < G; gi++) {
        if (rcs[gi]) return rcs[gi];
        if (gi < 8) h->stats.kernel_ms[gi] = kms[gi];
        h->stats.d2h_ms = std::max(h->stats.d2h_ms, copy_ms[gi]);
    }
    return MARAY_OK;
}

int render_frame(maray_cuda* h, uint32_t w, uint32_t hgt, uint8_t* host_rgb) {
    int rc = check_renderable(h, w, hgt);
    if (rc) return rc;
    double t0 = now_ms();
    Gpu& g0 = h->gpus[0];
    rc = ensure_out(h, g0, size_t(w) * hgt * 3);
    if (rc) return rc;
    for (Gpu& g : h->gpus) {   // the accumulators before any pass is in flight (a larger one replaces the old)
        if (h->samples > 1 && (rc = ensure_acc(h, g, size_t(w) * hgt)) != MARAY_OK) return rc;
    }
    for (double& k : h->stats.kernel_ms) k = 0.0;
    h->stats.gather_ms = 0.0; h->stats.d2h_ms = 0.0;
    rc = adopt_finished_job(h);
    if (rc) return rc;
    if (h->job && (h->report_kind == MARAY_REPORT_NONE || !h->report_fn)) {
        rc = render_frame_tiered(h, w, hgt);
        if (rc) return rc;
        if (host_rgb) {
            double t1 = now_ms();
            CU_TRY(h, cudaMemcpy(host_rgb, g0.d_out, size_t(w) * hgt * 3, cudaMemcpyDeviceToHost));
            h->stats.d2h_ms = now_ms() - t1;
        }
        h->stats.render_ms = now_ms() - t0;
        return MARAY_OK;
    }

    // Host-bound frames of 4 MiB and more are rendered in row chunks whose device->host copies overlap the
    // chunks still rendering (render_frame_pipelined).  Measured on chess_4k into a pageable buffer: 1 075 ->
    // 1 245 Mpixel/s end to end (profiles/r02_calls.md).  MARAY_PIPELINE=0 turns it off (A/B).
    bool pipelined = true;
    if (const char* e = std::getenv("MARAY_PIPELINE")) pipelined = std::strtoul(e, nullptr, 10) != 0;
    if (host_rgb && h->gpus.size() == 1 && pipelined &&
        (h->report_kind == MARAY_REPORT_NONE || !h->report_fn) && size_t(w) * hgt * 3 >= (size_t(4) << 20)) {
        rc = render_frame_pipelined(h, w, hgt, host_rgb);
        if (rc) return rc;
    } else if (host_rgb && h->gpus.size() > 1 && hgt >= h->gpus.size() && (h->report_kind == MARAY_REPORT_NONE || !h->report_fn)) {
        rc = render_frame_bands_to_host(h, w, hgt, host_rgb);
        if (rc) return rc;
    } else if (h->report_kind == MARAY_REPORT_NONE || !h->report_fn || !host_rgb) {
        rc = render_rows_to_frame(h, w, hgt, 0, hgt);
        if (rc) return rc;
        if (host_rgb) {
            double t1 = now_ms();
            CU_TRY(h, cudaMemcpy(host_rgb, g0.d_out, size_t(w) * hgt * 3, cudaMemcpyDeviceToHost));
            h->stats.d2h_ms = now_ms() - t1;
        }
    } else {
        // Progress reporting (reference src/report.rs:37-56): the frame is rendered in row chunks;
        // after a chunk the finished rows are copied out and the callback sees the partial image.
        uint32_t chunk = (h->report_kind == MARAY_REPORT_ROW) ? std::max<uint32_t>(1, h->report_every)
                                                              : std::max<uint32_t>(1, hgt / 64);
        double last = now_ms();
        uint32_t last_row = 0;
        for (uint32_t ya = 0; ya < hgt; ya += chunk) {
            uint32_t yb = std::min(hgt, ya + chunk);
            rc = render_rows_to_frame(h, w, hgt, ya, yb);
            if (rc) return rc;
            double t1 = now_ms();
            CU_TRY(h, cudaMemcpy(host_rgb + size_t(ya) * w * 3, g0.d_out + size_t(ya) * w * 3, size_t(yb - ya) * w * 3,
                                 cudaMemcpyDeviceToHost));
            h->stats.d2h_ms += now_ms() - t1;
            if (yb == hgt) break;
            bool fire;
            if (h->report_kind == MARAY_REPORT_ROW) {
                fire = yb >= last_row + h->report_every;
                if (fire) last_row += h->report_every;
            } else {
                fire = now_ms() - last >= double(h->report_every);
                if (fire) last = now_ms();
            }
            if (fire) h->report_fn(h->report_user, host_rgb, w, hgt, double(yb) / double(hgt));
        }
    }
    h->stats.render_ms = now_ms() - t0;
    return MARAY_OK;
}

}  // namespace

// ================================================================================================
extern "C" {

const char* maray_cuda_version(void) { return "maray_b200 0.1 (sm_100a)"; }

const char* maray_cuda_last_error(const maray_cuda_t* h) { return h ? h->error.c_str() : g_create_error.c_str(); }

int maray_cuda_create(int n_gpus, const int* device_ids, maray_cuda_t** out) {
    if (!out || n_gpus < 0) return fail(nullptr, MARAY_E_INVALID, "maray_cuda_create: bad arguments");
    *out = nullptr;
    std::unique_ptr<maray_cuda> h(new maray_cuda());
    if (const char* e = std::getenv("MARAY_LIBM")) {
        const std::string v(e);
        h->libm = v == "glibc" ? MARAY_LIBM_GLIBC : v == "cuda" ? MARAY_LIBM_CUDA : MARAY_LIBM_FAST;
    }
    if (n_gpus > 0) {
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || count == 0)
            return fail(nullptr, MARAY_E_CUDA, std::string("no usable CUDA device: ") + cudaGetErrorString(e) +
                                                   " (this render path has no CPU fallback)");
        for (int i = 0; i < n_gpus; i++) {
            int dev = device_ids ? device_ids[i] : i;
            if (dev < 0 || dev >= count)
                return fail(nullptr, MARAY_E_CUDA, "device " + std::to_string(dev) + " requested but only " +
                                                       std::to_string(count) + " visible");
            Gpu g;
            g.device = dev;
            h->gpus.push_back(g);
        }
        maray_cuda* hp = nullptr;   // errors during create go to the thread-local message
        for (size_t i = 0; i < h->gpus.size(); i++) {
            Gpu& g = h->gpus[i];
            CU_TRY(hp, cudaSetDevice(g.device));
            CU_TRY(hp, cudaStreamCreateWithFlags(&g.stream, cudaStreamNonBlocking));
            if (cudaDeviceGetAttribute(&g.sms, cudaDevAttrMultiProcessorCount, g.device) != cudaSuccess || g.sms <= 0) { g.sms = 148; cudaGetLastError(); }
            CU_TRY(hp, cudaEventCreate(&g.ev0));
            CU_TRY(hp, cudaEventCreate(&g.ev1));
            CU_TRY(hp, cudaMalloc(&g.d_sink, 256));
            CU_TRY(hp, cudaMemset(g.d_sink, 0, 256));
            if (i > 0) {
                int can = 0;
                cudaDeviceCanAccessPeer(&can, g.device, h->gpus[0].device);
                if (can) {
                    cudaError_t pe = cudaDeviceEnablePeerAccess(h->gpus[0].device, 0);
                    if (pe == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); pe = cudaSuccess; }
                    g.peer_to_0 = (pe == cudaSuccess);
                }
            }
        }
        cudaSetDevice(h->gpus[0].device);
    }
    *out = h.release();
    return MARAY_OK;
}

void maray_cuda_destroy(maray_cuda_t* h) {
    if (!h) return;
    release_backend(h, /*cancel_job=*/false);
    release_textures(h);
    if (!h->gpus.empty() && !h->imported.empty()) {
        cudaSetDevice(h->gpus[0].device);
        for (void* p : h->imported) cudaIpcCloseMemHandle(p);
    }
    for (Gpu& g : h->gpus) {
        cudaSetDevice(g.device);
        if (g.d_out) cudaFree(g.d_out);
        if (g.d_f64) cudaFree(g.d_f64);
        if (g.d_acc) cudaFree(g.d_acc);
        if (g.d_sink) cudaFree(g.d_sink);
        if (g.frame_done) cudaEventDestroy(g.frame_done);
        if (g.ev0) cudaEventDestroy(g.ev0);
        if (g.ev1) cudaEventDestroy(g.ev1);
        if (g.stream) cudaStreamDestroy(g.stream);
        if (g.copy_stream) cudaStreamDestroy(g.copy_stream);
        for (int c = 0; c < Gpu::kChunks; c++) {
            if (g.chunk_stream[c]) cudaStreamDestroy(g.chunk_stream[c]);
            if (g.chunk_done[c]) cudaEventDestroy(g.chunk_done[c]);
        }
    }
    delete h;
}

int maray_cuda_set_textures(maray_cuda_t* h, uint32_t n, const uint8_t* const* rgb8, const uint32_t* w, const uint32_t* hgt) {
    if (!h || (n && (!rgb8 || !w || !hgt))) return fail(h, MARAY_E_INVALID, "maray_cuda_set_textures: bad arguments");
    release_textures(h);
    h->textures.clear();
    h->textures.resize(n);
    for (uint32_t i = 0; i < n; i++) {
        HostTexture& t = h->textures[i];
        t.w = w[i]; t.h = hgt[i];
        size_t bytes = size_t(w[i]) * hgt[i] * 3;
        if (bytes && !rgb8[i]) return fail(h, MARAY_E_INVALID, "maray_cuda_set_textures: null texture data");
        t.rgb.assign(rgb8[i], rgb8[i] + bytes);
    }
    h->compiled = false;   // width/height constants are folded into the program
    return MARAY_OK;
}

int maray_cuda_load_maray(maray_cuda_t* h, const uint8_t* bytes, size_t len) {
    if (!h || !bytes) return fail(h, MARAY_E_INVALID, "maray_cuda_load_maray: bad arguments");
    release_backend(h);
    h->have_scene = false;
    Scene sc;
    std::string err;
    if (!parse_maray(bytes, len, &sc, &err)) return fail(h, MARAY_E_PARSE, err);
    h->scene = std::move(sc);
    h->have_scene = true;
    return MARAY_OK;
}

int maray_cuda_scene_size(const maray_cuda_t* h, uint32_t* w, uint32_t* hgt) {
    if (!h || !h->have_scene || !w || !hgt) return MARAY_E_INVALID;
    *w = h->scene.size[0]; *hgt = h->scene.size[1];
    return MARAY_OK;
}

int maray_cuda_compile(maray_cuda_t* h, int backend, maray_cuda_stats* stats) {
    if (!h) return MARAY_E_INVALID;
    if (!h->have_scene) return fail(h, MARAY_E_INVALID, "maray_cuda_compile called before maray_cuda_load_maray");
    if (backend != MARAY_BACKEND_INTERP && backend != MARAY_BACKEND_NVRTC && backend != MARAY_BACKEND_AUTO)
        return fail(h, MARAY_E_INVALID, "unknown back end");
    release_backend(h);
    h->stats = maray_cuda_stats{};
    h->stats.backend = uint32_t(backend);
    h->backend = backend;

    double t0 = now_ms();
    std::vector<TextureDim> dims;
    for (const HostTexture& t : h->textures) dims.push_back(TextureDim{t.w, t.h});
    std::string err;
    Program prog;
    if (!lower_scene(h->scene, dims, &prog, &err)) return fail(h, MARAY_E_SCENE, err);
    h->prog = std::move(prog);
    h->stats.lower_ms = now_ms() - t0;
    fill_program_stats(h);
    if (!h->gpus.empty()) {
        int rc = upload_textures(h);
        if (rc) return rc;
    }

    int rc = MARAY_OK;
    if (backend == MARAY_BACKEND_INTERP) {
        rc = interp_build_and_install(h);
    } else if (backend == MARAY_BACKEND_NVRTC) {
        JitBuild jb;
        jb.libm = h->libm; jb.frame_pixels = uint64_t(h->scene.size[0]) * h->scene.size[1]; jb.sms = h->gpus.empty() ? 148u : uint32_t(h->gpus[0].sms);
        rc = jit_build(h->prog, &jb, /*cached_only=*/false, nullptr);
        if (rc) { h->jit = std::move(jb); fill_jit_stats(h); return fail(h, rc, h->jit.error); }   // the generated text stays inspectable
        rc = jit_install(h, std::move(jb));
    } else {
        // AUTO (time to first frame): cubins already in the cache are used at once.  Otherwise the interpreter --
        // ready in milliseconds -- renders while NVRTC works on another thread; renders switch to the generated
        // kernels, between row chunks, as soon as they are built.  Both back ends produce the same bytes.
        JitBuild jb;
        jb.libm = h->libm; jb.frame_pixels = uint64_t(h->scene.size[0]) * h->scene.size[1]; jb.sms = h->gpus.empty() ? 148u : uint32_t(h->gpus[0].sms);
        rc = jit_build(h->prog, &jb, /*cached_only=*/true, nullptr);
        if (rc == MARAY_OK) {
            rc = jit_install(h, std::move(jb));
        } else {
            rc = interp_build_and_install(h);
            if (rc == MARAY_E_UNSUPPORTED) {
                // the slot file does not fit: compile now, there is nothing to render with meanwhile
                JitBuild now;
                now.libm = h->libm; now.frame_pixels = uint64_t(h->scene.size[0]) * h->scene.size[1]; now.sms = h->gpus.empty() ? 148u : uint32_t(h->gpus[0].sms);
                rc = jit_build(h->prog, &now, false, nullptr);
                if (rc) return fail(h, rc, now.error);
                rc = jit_install(h, std::move(now));
            } else if (rc == MARAY_OK && !std::getenv("MARAY_JIT_SOURCE_ONLY")) {
                h->job.reset(new JitJob());
                JitJob* job = h->job.get();
                job->prog = h->prog;
                job->build.libm = h->libm; job->build.frame_pixels = uint64_t(h->scene.size[0]) * h->scene.size[1]; job->build.sms = h->gpus.empty() ? 148u : uint32_t(h->gpus[0].sms);
                job->th = std::thread([job] {
                    job->rc = jit_build(job->prog, &job->build, false, &job->cancel);
                    job->state = job->rc == MARAY_OK ? 1 : 2;
                });
            }
        }
    }
    if (rc) return rc;
    h->compiled = true;
    if (stats) *stats = h->stats;
    return MARAY_OK;
}

int maray_cuda_set_libm(maray_cuda_t* h, int libm) {
    if (!h || libm < MARAY_LIBM_FAST || libm > MARAY_LIBM_CUDA) return fail(h, MARAY_E_INVALID, "maray_cuda_set_libm: bad libm");
    h->libm = libm;
    return MARAY_OK;
}

int maray_cuda_set_samples(maray_cuda_t* h, uint32_t s) {
    if (!h) return MARAY_E_INVALID;
    if (s < 1 || s > 16) return fail(h, MARAY_E_INVALID, "maray_cuda_set_samples: samples per axis must be 1..16, got " + std::to_string(s));
    h->samples = s;
    return MARAY_OK;
}

int maray_cuda_set_report(maray_cuda_t* h, int kind, uint32_t every, maray_report_fn fn, void* user) {
    if (!h || kind < MARAY_REPORT_NONE || kind > MARAY_REPORT_DURATION_MS) return fail(h, MARAY_E_INVALID, "bad report kind");
    h->report_kind = kind; h->report_every = every; h->report_fn = fn; h->report_user = user;
    return MARAY_OK;
}

int maray_cuda_render(maray_cuda_t* h, uint32_t w, uint32_t hgt, uint8_t* rgb, maray_cuda_stats* stats) {
    if (!h) return MARAY_E_INVALID;
    if (!rgb) return fail(h, MARAY_E_INVALID, "maray_cuda_render: null output buffer");
    int rc = render_frame(h, w, hgt, rgb);
    if (rc == MARAY_OK && stats) *stats = h->stats;
    return rc;
}

int maray_cuda_render_device(maray_cuda_t* h, uint32_t w, uint32_t hgt, void** d_rgb, maray_cuda_stats* stats) {
    if (!h) return MARAY_E_INVALID;
    if (!d_rgb) return fail(h, MARAY_E_INVALID, "maray_cuda_render_device: null output pointer");
    int rc = render_frame(h, w, hgt, nullptr);
    if (rc) return rc;
    *d_rgb = h->gpus[0].d_out;
    if (stats) *stats = h->stats;
    return MARAY_OK;
}

int maray_cuda_render_band(maray_cuda_t* h, uint32_t w, uint32_t hgt, uint32_t y0, uint32_t y1, void* d_band, void* stream) {
    int rc = check_renderable(h, w, hgt);
    if (rc) return rc;
    if (y0 > y1 || y1 > hgt || !d_band) return fail(h, MARAY_E_INVALID, "maray_cuda_render_band: bad band");
    rc = adopt_finished_job(h);               // MARAY_BACKEND_AUTO: switch to the generated kernels once they are built
    if (rc) return rc;
    Gpu& g = h->gpus[0];
    CU_TRY(h, cudaSetDevice(g.device));
    return launch_band(h, g, w, y0 * w, (y1 - y0) * w, static_cast<uint8_t*>(d_band), nullptr, 0,
                       static_cast<cudaStream_t>(stream));
}

int maray_cuda_frame_export(maray_cuda_t* h, uint32_t w, uint32_t hgt, void* handle64, void** d_frame) {
    int rc = check_renderable(h, w, hgt);
    if (rc) return rc;
    if (!handle64 || !d_frame) return fail(h, MARAY_E_INVALID, "maray_cuda_frame_export: null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == MARAY_IPC_HANDLE_BYTES, "CUDA IPC handle size");
    Gpu& g = h->gpus[0];
    CU_TRY(h, cudaSetDevice(g.device));
    rc = ensure_out(h, g, band_counters_offset(w, hgt) + kBandCounters * kBandCounterStride * sizeof(uint32_t));   // frame + completion counters
    if (rc) return rc;
    CU_TRY(h, cudaMemset(g.d_out + band_counters_offset(w, hgt), 0, kBandCounters * kBandCounterStride * sizeof(uint32_t)));
    cudaIpcMemHandle_t hd;
    CU_TRY(h, cudaIpcGetMemHandle(&hd, g.d_out));
    std::memcpy(handle64, &hd, sizeof hd);
    *d_frame = g.d_out;
    return MARAY_OK;
}

int maray_cuda_frame_import(maray_cuda_t* h, const void* handle64, void** d_frame) {
    if (!h || !handle64 || !d_frame) return fail(h, MARAY_E_INVALID, "maray_cuda_frame_import: null argument");
    if (h->gpus.empty()) return fail(h, MARAY_E_CUDA, "host-only handle");
    CU_TRY(h, cudaSetDevice(h->gpus[0].device));
    cudaIpcMemHandle_t hd;
    std::memcpy(&hd, handle64, sizeof hd);
    void* p = nullptr;
    CU_TRY(h, cudaIpcOpenMemHandle(&p, hd, cudaIpcMemLazyEnablePeerAccess));
    h->imported.push_back(p);
    *d_frame = p;
    return MARAY_OK;
}

int maray_cuda_band_signal(maray_cuda_t* h, void* d_frame, uint32_t w, uint32_t hgt, uint32_t rank, uint32_t value, void* stream) {
    if (!h || !d_frame || rank >= kBandCounters) return fail(h, MARAY_E_INVALID, "maray_cuda_band_signal: bad argument");
    if (h->gpus.empty()) return fail(h, MARAY_E_CUDA, "host-only handle");
    CU_TRY(h, cudaSetDevice(h->gpus[0].device));
    auto* counters = reinterpret_cast<uint32_t*>(static_cast<uint8_t*>(d_frame) + band_counters_offset(w, hgt));
    CU_TRY(h, launch_band_signal(counters + size_t(rank) * kBandCounterStride, value, static_cast<cudaStream_t>(stream)));
    return MARAY_OK;
}

int maray_cuda_band_wait(maray_cuda_t* h, void* d_frame, uint32_t w, uint32_t hgt, uint32_t n_ranks, uint32_t value, void* stream) {
    if (!h || !d_frame || n_ranks == 0 || n_ranks > kBandCounters) return fail(h, MARAY_E_INVALID, "maray_cuda_band_wait: bad argument");
    if (h->gpus.empty()) return fail(h, MARAY_E_CUDA, "host-only handle");
    Gpu& g = h->gpus[0];
    CU_TRY(h, cudaSetDevice(g.device));
    auto* counters = reinterpret_cast<uint32_t*>(static_cast<uint8_t*>(d_frame) + band_counters_offset(w, hgt));
    int khz = 0;
    if (cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, g.device) != cudaSuccess || khz <= 0) { khz = 2000000; cudaGetLastError(); }
    CU_TRY(h, launch_band_wait(counters, kBandCounterStride, n_ranks, value, band_timeout_word(g), 2000ll * khz,
                               static_cast<cudaStream_t>(stream)));   // ~2 s
    return MARAY_OK;
}

int maray_cuda_copy_to_host(maray_cuda_t* h, const void* d_src, void* host_dst, size_t bytes) {
    if (!h || !d_src || !host_dst) return fail(h, MARAY_E_INVALID, "maray_cuda_copy_to_host: null argument");
    if (h->gpus.empty()) return fail(h, MARAY_E_CUDA, "host-only handle");
    Gpu& g = h->gpus[0];
    CU_TRY(h, cudaSetDevice(g.device));
    CU_TRY(h, cudaMemcpy(host_dst, d_src, bytes, cudaMemcpyDeviceToHost));
    uint32_t timed_out = 0;                       // a band wait that gave up: the frame may be incomplete
    CU_TRY(h, cudaMemcpy(&timed_out, band_timeout_word(g), sizeof timed_out, cudaMemcpyDeviceToHost));
    if (timed_out) {
        CU_TRY(h, cudaMemset(band_timeout_word(g), 0, sizeof timed_out));
        return fail(h, MARAY_E_CUDA, "maray_cuda_band_wait timed out: a band process never signalled");
    }
    return MARAY_OK;
}

int maray_cuda_render_window_f64(maray_cuda_t* h, uint32_t w, uint32_t hgt, uint32_t x0, uint32_t x1, uint32_t y0,
                                 uint32_t y1, double* planes, uint8_t* rgb) {
    int rc = check_renderable(h, w, hgt);
    if (rc) return rc;
    if (x0 > x1 || x1 > w || y0 > y1 || y1 > hgt) return fail(h, MARAY_E_INVALID, "window outside the image");
    if (h->samples > 1)   // the f64 planes are the values of single samples
        return fail(h, MARAY_E_INVALID, "maray_cuda_render_window_f64 renders one sample per pixel; call maray_cuda_set_samples(h, 1) first");
    const uint32_t ww = x1 - x0, hh = y1 - y0;
    const size_t npx = size_t(ww) * hh;
    if (npx == 0) return MARAY_OK;
    Gpu& g = h->gpus[0];
    CU_TRY(h, cudaSetDevice(g.device));
    rc = ensure_out(h, g, npx * 3 + 16 * size_t(hh));
    if (rc) return rc;
    if (g.f64_cap < npx * 3) {
        if (g.d_f64) cudaFree(g.d_f64);
        g.d_f64 = nullptr; g.f64_cap = 0;
        CU_TRY(h, cudaMalloc(&g.d_f64, npx * 3 * sizeof(double)));
        g.f64_cap = npx * 3;
    }
    // one launch per window row (instrumentation path, not a fast path)
    for (uint32_t r = 0; r < hh; r++) {
        rc = launch_band(h, g, w, (y0 + r) * w + x0, ww, g.d_out + size_t(r) * ww * 3,
                         planes ? g.d_f64 + size_t(r) * ww : nullptr, npx, g.stream);
        if (rc) return rc;
    }
    CU_TRY(h, cudaStreamSynchronize(g.stream));
    if (planes) CU_TRY(h, cudaMemcpy(planes, g.d_f64, npx * 3 * sizeof(double), cudaMemcpyDeviceToHost));
    if (rgb) CU_TRY(h, cudaMemcpy(rgb, g.d_out, npx * 3, cudaMemcpyDeviceToHost));
    return MARAY_OK;
}

int maray_cuda_get_stats(const maray_cuda_t* h, maray_cuda_stats* stats) {
    if (!h || !stats) return MARAY_E_INVALID;
    *stats = h->stats;
    stats->jit_active = h->use_jit ? 1u : 0u;
    return MARAY_OK;
}

int maray_cuda_get_source(const maray_cuda_t* h, char* buf, size_t cap, size_t* len) {
    if (!h) return MARAY_E_INVALID;
    if (len) *len = h->jit.source.size();
    if (buf && cap) {
        size_t n = std::min(cap - 1, h->jit.source.size());
        std::memcpy(buf, h->jit.source.data(), n);
        buf[n] = '\0';
    }
    return MARAY_OK;
}

int maray_cuda_get_module(const maray_cuda_t* h, uint32_t index, char* buf, size_t cap, size_t* len) {
    if (!h || index >= h->jit.modules.size()) return MARAY_E_INVALID;
    const std::string& m = h->jit.modules[index];
    if (len) *len = m.size();
    if (buf && cap) {
        size_t n = std::min(cap - 1, m.size());
        std::memcpy(buf, m.data(), n);
        buf[n] = '\0';
    }
    return MARAY_OK;
}

int maray_cuda_get_cubin(const maray_cuda_t* h, uint32_t index, void* buf, size_t cap, size_t* len) {
    if (!h || index >= h->jit.cubins.size()) return MARAY_E_INVALID;
    const std::vector<char>& c = h->jit.cubins[index];
    if (len) *len = c.size();
    if (buf && cap) std::memcpy(buf, c.data(), std::min(cap, c.size()));
    return MARAY_OK;
}

int maray_cuda_get_bytecode(const maray_cuda_t* h, uint64_t* code, size_t cap_instr, size_t* n_instr, double* consts,
                            size_t cap_consts, size_t* n_consts) {
    if (!h) return MARAY_E_INVALID;
    const Bytecode& bc = h->bc;
    if (n_instr) *n_instr = bc.code.size();
    if (n_consts) *n_consts = bc.consts.size();
    if (code) std::memcpy(code, bc.code.data(), std::min(cap_instr, bc.code.size()) * sizeof(uint64_t));
    if (consts) std::memcpy(consts, bc.consts.data(), std::min(cap_consts, bc.consts.size()) * sizeof(double));
    return MARAY_OK;
}

int maray_cuda_fp64_peak(maray_cuda_t* h, int gpu_index, double* lane_ops_per_s, double* dfma_lane_ops_per_s) {
    if (!h) return MARAY_E_INVALID;
    if (gpu_index < 0 || size_t(gpu_index) >= h->gpus.size()) return fail(h, MARAY_E_CUDA, "no such GPU in this handle");
    Gpu& g = h->gpus[gpu_index];
    CU_TRY(h, cudaSetDevice(g.device));
    cudaDeviceProp prop;
    CU_TRY(h, cudaGetDeviceProperties(&prop, g.device));
    const int blocks = prop.multiProcessorCount * 8;   // 8 x 256 threads = 2048 threads per SM
    const int iters = 4096;
    for (int fma = 0; fma < 2; fma++) {
        double best = 0.0;
        for (int rep = 0; rep < 4; rep++) {
            CU_TRY(h, cudaEventRecord(g.ev0, g.stream));
            CU_TRY(h, launch_fp64_issue_rate(fma != 0, g.d_sink, iters, blocks, g.stream));
            CU_TRY(h, cudaEventRecord(g.ev1, g.stream));
            CU_TRY(h, cudaStreamSynchronize(g.stream));
            float ms = 0.f;
            CU_TRY(h, cudaEventElapsedTime(&ms, g.ev0, g.ev1));
            double ops = double(blocks) * 256.0 * double(iters) * 64.0;   // 8 chains x 8 unrolled per iteration
            if (rep > 0) best = std::max(best, ops / (double(ms) * 1e-3));
        }
        if (fma == 0 && lane_ops_per_s) *lane_ops_per_s = best;
        if (fma == 1 && dfma_lane_ops_per_s) *dfma_lane_ops_per_s = best;
    }
    return MARAY_OK;
}

}  // extern "C"
