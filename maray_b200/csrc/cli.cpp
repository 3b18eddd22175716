// maray_cuda -- command-line front end of the CUDA render path, shaped like the reference's CLI
// (reference examples/maray.rs:9-47):
//     maray_cuda -i scene.maray -o out.png [-t tex0.png tex1.png ...] [-c N] [-g GPUS] [-b nvrtc|interp] [-s N]
// -s/--samples N renders N x N samples per pixel, box-filtered (maray_cuda_set_samples; 1, the default, is the
// reference's frame).
// -c/--cpus is accepted for command-line compatibility and ignored, exactly as the reference ignores
// it at HEAD (reference examples/maray.rs:55: parsed into `_cpus`).  Progress is reported every
// 500 ms the way `gen` does (reference src/lib.rs:1203-1208, examples/maray.rs:77-79): percentage on
// stderr and the partial image re-saved.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/maray_cuda.h"
#include "png.hpp"

namespace {

struct ProgressCtx { std::string out; };

void on_progress(void* user, uint8_t* rgb, uint32_t w, uint32_t h, double progress) {
    ProgressCtx* c = static_cast<ProgressCtx*>(user);
    std::fprintf(stderr, "%.2f %%\n", 100.0 * progress);
    std::string err;
    maray::write_png_rgb8(c->out, w, h, rgb, &err);
}

int usage() {
    std::fprintf(stderr,
                 "Maray (CUDA render path)\n"
                 "usage: maray_cuda -i <file.maray> -o <file.png> [-t <texture.png>...] [-c <cpus, ignored>]\n"
                 "                  [-g <gpus>] [-b nvrtc|interp] [-s <samples per axis, 1..16>]\n");
    return 2;
}

}  // namespace

int main(int argc, char** argv) {
    std::string input, output, backend = "nvrtc";
    std::vector<std::string> textures;
    int gpus = 1, samples = 1;
    for (int i = 1; i < argc; i++) {
        std::string a = argv[i];
        auto value = [&]() -> const char* { return i + 1 < argc ? argv[++i] : nullptr; };
        if (a == "-i" || a == "--input") { const char* v = value(); if (!v) return usage(); input = v; }
        else if (a == "-o" || a == "--output") { const char* v = value(); if (!v) return usage(); output = v; }
        else if (a == "-c" || a == "--cpus") { if (!value()) return usage(); }
        else if (a == "-g" || a == "--gpus") { const char* v = value(); if (!v) return usage(); gpus = std::atoi(v); }
        else if (a == "-s" || a == "--samples") { const char* v = value(); if (!v) return usage(); samples = std::atoi(v); }
        else if (a == "-b" || a == "--backend") { const char* v = value(); if (!v) return usage(); backend = v; }
        else if (a == "-t" || a == "--textures") {
            while (i + 1 < argc && argv[i + 1][0] != '-') textures.push_back(argv[++i]);
        } else return usage();
    }
    if (input.empty() || output.empty() || gpus < 1 || samples < 1 || samples > 16 || (backend != "nvrtc" && backend != "interp")) return usage();

    // open(file)  (reference src/lib.rs:1227-1235)
    std::vector<uint8_t> scene;
    {
        FILE* f = std::fopen(input.c_str(), "rb");
        if (!f) { std::fprintf(stderr, "error: cannot open %s\n", input.c_str()); return 1; }
        uint8_t buf[65536];
        size_t n;
        while ((n = std::fread(buf, 1, sizeof buf, f)) > 0) scene.insert(scene.end(), buf, buf + n);
        std::fclose(f);
    }
    // textures -> Runtime<Textures>  (reference examples/maray.rs:58-69)
    std::vector<std::vector<uint8_t>> tex(textures.size());
    std::vector<const uint8_t*> tex_ptr;
    std::vector<uint32_t> tw(textures.size()), th(textures.size());
    for (size_t i = 0; i < textures.size(); i++) {
        std::string err;
        if (!maray::read_png_rgb8(textures[i], &tw[i], &th[i], &tex[i], &err)) { std::fprintf(stderr, "error: %s\n", err.c_str()); return 1; }
        tex_ptr.push_back(tex[i].data());
    }

    maray_cuda_t* h = nullptr;
    if (maray_cuda_create(gpus, nullptr, &h) != MARAY_OK) { std::fprintf(stderr, "error: %s\n", maray_cuda_last_error(nullptr)); return 1; }
    auto die = [&](const char* what) {
        std::fprintf(stderr, "error: %s: %s\n", what, maray_cuda_last_error(h));
        maray_cuda_destroy(h);
        return 1;
    };
    if (maray_cuda_set_textures(h, uint32_t(tex.size()), tex_ptr.data(), tw.data(), th.data()) != MARAY_OK) return die("textures");
    if (maray_cuda_load_maray(h, scene.data(), scene.size()) != MARAY_OK) return die("open");
    uint32_t w = 0, hgt = 0;
    maray_cuda_scene_size(h, &w, &hgt);
    if (maray_cuda_set_samples(h, uint32_t(samples)) != MARAY_OK) return die("samples");
    maray_cuda_stats st;
    if (maray_cuda_compile(h, backend == "nvrtc" ? MARAY_BACKEND_NVRTC : MARAY_BACKEND_INTERP, &st) != MARAY_OK) return die("compile");
    std::vector<uint8_t> img(size_t(w) * hgt * 3);
    ProgressCtx ctx{output};
    maray_cuda_set_report(h, MARAY_REPORT_DURATION_MS, 500, on_progress, &ctx);
    if (maray_cuda_render(h, w, hgt, img.data(), &st) != MARAY_OK) return die("render");
    std::string err;
    if (!maray::write_png_rgb8(output, w, hgt, img.data(), &err)) { std::fprintf(stderr, "error: %s\n", err.c_str()); maray_cuda_destroy(h); return 1; }
    std::fprintf(stderr, "%ux%u, %llu values, lower %.1f ms, compile %.1f ms, render %.2f ms (kernel %.2f ms on GPU 0)\n", w, hgt,
                 (unsigned long long)st.dag_nodes, st.lower_ms, st.codegen_ms + st.nvrtc_ms + st.load_ms, st.render_ms, st.kernel_ms[0]);
    maray_cuda_destroy(h);
    return 0;
}
