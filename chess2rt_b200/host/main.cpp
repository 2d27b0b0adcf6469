// Headless mode of the renderer (north star: "the renderer gains a headless mode"; SURVEY.md §8f-1).
// The reference's only entry is `chess2rt --file=<scene>` opening the SDL GUI
// (/root/reference/source/app.d:9-22); this executable takes the same --file and renders one or more
// frames through renderSceneAsync -> libc2rt.so without a window, then writes the image.
//
//   chess2rt_headless --file scenes/lecture5.sdl --out out.bmp [--pfm out.pfm] [--width W --height H]
//                     [--gpus N] [--no-dof] [--no-aa] [--seed S] [--repeat K] [--pad-rows] [--orbit K]
//                     [--depth d.pfm] [--ids ids.pgm]
// --out writes the BMP the reference's Bitmap.saveImage would (bitmap.d:84-103 -> bmp.d:195-237, rows unpadded: only
// widths with 3 W % 4 == 0 give a file other readers accept); --pad-rows writes the valid file for any width.
// --orbit K: the interactive loop without a window — K frames, the camera turned by 360 / K degrees of yaw before each
// (Camera.rotate, camera.d:211-229, what the arrow keys do: raytracer_demo.d:268-340), scene resident on the GPU, only the
// camera / settings blocks go down and only the packed ARGB plane comes back (what SDL2Gui.draw blits, sdl2_gui.d:139-155).
// --depth / --ids: renderPixel's hit distance / node of every pixel (one c2rt_render_hits call after the last frame), as a
// one-channel PFM (bottom row first, +inf for a miss) / a 16-bit binary PGM (node + 1, 0 for a miss).
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>

#include "renderer.hpp"

using namespace rt;

static void usage() {
    fprintf(stderr,
            "usage: chess2rt_headless --file <scene.sdl|scene.json> [--out img.bmp] [--pfm img.pfm]\n"
            "                         [--width W --height H] [--gpus N] [--no-dof] [--no-aa] [--seed S] [--repeat K]\n"
            "                         [--pad-rows] [--orbit K] [--depth d.pfm] [--ids ids.pgm]\n");
}

int main(int argc, char** argv) {
    std::string file, out, pfm, depth, ids;
    uint32_t width = 0, height = 0;
    int gpus = 1, repeat = 1, orbit = 0;
    bool noDof = false, noAA = false, padRows = false;
    uint64_t seed = 0;
    for (int i = 1; i < argc; i++) {
        std::string a = argv[i];
        auto val = [&](const char* name) -> const char* {
            size_t n = strlen(name);
            if (a.compare(0, n, name) == 0 && a.size() > n && a[n] == '=') return argv[i] + n + 1;
            if (a == name && i + 1 < argc) return argv[++i];
            return nullptr;
        };
        const char* v;
        if ((v = val("--file"))) file = v;
        else if ((v = val("--out"))) out = v;
        else if ((v = val("--pfm"))) pfm = v;
        else if ((v = val("--depth"))) depth = v;
        else if ((v = val("--ids"))) ids = v;
        else if ((v = val("--width"))) width = (uint32_t)atoi(v);
        else if ((v = val("--height"))) height = (uint32_t)atoi(v);
        else if ((v = val("--gpus"))) gpus = atoi(v);
        else if ((v = val("--seed"))) seed = strtoull(v, nullptr, 0);
        else if ((v = val("--repeat"))) repeat = atoi(v);
        else if ((v = val("--orbit"))) orbit = atoi(v);
        else if (a == "--pad-rows") padRows = true;
        else if (a == "--no-dof") noDof = true;
        else if (a == "--no-aa") noAA = true;
        else if (a == "--headless") {}
        else { usage(); return 2; }
    }
    if (file.empty() || gpus < 1 || repeat < 1 || orbit < 0) { usage(); return 2; }
    try {
        auto scene = parseSceneFromFile(file);   // (load errors are reported before any device is touched)
        setRenderDevices(gpus);
        if (width && height) {
            scene->settings.frameWidth = width;
            scene->settings.frameHeight = height;
            scene->camera.setFrameSize(width, height);
        }
        if (noDof) scene->camera.dof = false;
        if (noAA) scene->settings.AAEnabled = false;
        const uint32_t W = scene->settings.frameWidth, H = scene->settings.frameHeight;
        Image<Color> screen(W, H);
        Image<uint32_t> argb(W, H);
        // page-lock the output planes: the per-frame device->host copies then overlap with rendering
        c2rt_pin_host_buffer(screen.pixels.data(), screen.pixels.size() * sizeof(Color));
        c2rt_pin_host_buffer(argb.pixels.data(), argb.pixels.size() * sizeof(uint32_t));
        RenderOptions opt;
        opt.rngSeed = seed;
        opt.countRays = true;
        opt.argb = &argb;
        c2rt_stats stats{};
        for (int k = 0; k < repeat; k++) {
            std::atomic<bool> isRendering{true}, needsRendering{false};
            auto t0 = std::chrono::steady_clock::now();
            scene->beginFrame();
            Renderer renderer(*scene, screen, &isRendering, &needsRendering);
            renderer.options = opt;
            renderer.renderRT();
            double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
            stats = renderer.lastStats;
            printf("frame %d: %ux%u on %u GPU(s): kernel %.3f ms, end-to-end %.3f ms, %.2f Mrays/s (%.0f primary + %.0f shadow rays)\n", k, W,
                   H, stats.n_gpus, stats.kernel_ms, ms, (stats.primary_rays + stats.shadow_rays) / (stats.kernel_ms * 1e3),
                   (double)stats.primary_rays, (double)stats.shadow_rays);
        }
        if (!out.empty()) {
            auto bytes = saveBmp(argb, padRows);
            std::ofstream f(out, std::ios::binary);
            f.write((const char*)bytes.data(), (std::streamsize)bytes.size());
            printf("wrote %s\n", out.c_str());
        }
        if (!pfm.empty()) {  // float RGB, bottom row first (PFM convention), little endian
            std::ofstream f(pfm, std::ios::binary);
            f << "PF\n" << W << " " << H << "\n-1.0\n";
            for (uint32_t y = H; y-- > 0;) f.write((const char*)&screen.pixels[(size_t)W * y], (std::streamsize)W * sizeof(Color));
            printf("wrote %s\n", pfm.c_str());
        }
        if (!depth.empty() || !ids.empty()) {
            HitPlanes hits;
            if (!depth.empty()) hits.dist.resize((size_t)W * H);
            if (!ids.empty()) hits.node.resize((size_t)W * H);
            Renderer renderer(*scene, screen);
            renderer.options = opt;
            renderer.renderHits(hits);
            if (!depth.empty()) {  // one-channel float, bottom row first (PFM convention), little endian
                std::ofstream f(depth, std::ios::binary);
                f << "Pf\n" << W << " " << H << "\n-1.0\n";
                for (uint32_t y = H; y-- > 0;) f.write((const char*)&hits.dist[(size_t)W * y], (std::streamsize)W * sizeof(float));
                printf("wrote %s\n", depth.c_str());
            }
            if (!ids.empty()) {  // 16-bit binary PGM: most significant byte first, top row first
                std::ofstream f(ids, std::ios::binary);
                f << "P5\n" << W << " " << H << "\n65535\n";
                std::vector<uint8_t> row((size_t)W * 2);
                for (uint32_t y = 0; y < H; y++) {
                    for (uint32_t x = 0; x < W; x++) {
                        const uint32_t v = (uint32_t)(hits.node[(size_t)W * y + x] + 1);
                        row[2 * x] = (uint8_t)(v >> 8);
                        row[2 * x + 1] = (uint8_t)v;
                    }
                    f.write((const char*)row.data(), (std::streamsize)row.size());
                }
                printf("wrote %s\n", ids.c_str());
            }
        }
        if (orbit > 0) {
            RenderOptions io = opt;
            io.countRays = false;
            io.argbOnly = true;
            double total_ms = 0, kernel_ms = 0;
            for (int k = 0; k < orbit; k++) {
                scene->camera.rotate(360.0 / orbit, 0, 0);
                std::atomic<bool> isRendering{true}, needsRendering{false};
                auto t0 = std::chrono::steady_clock::now();
                scene->beginFrame();
                Renderer renderer(*scene, screen, &isRendering, &needsRendering);
                renderer.options = io;
                renderer.renderRT();
                total_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
                kernel_ms += renderer.lastStats.kernel_ms;
            }
            printf("orbit: %d frames of %ux%u, ARGB-only delivery: %.3f ms per frame end to end (%.1f fps), kernel %.3f ms\n", orbit, W, H,
                   total_ms / orbit, 1e3 * orbit / total_ms, kernel_ms / orbit);
        }
        c2rt_unpin_host_buffer(screen.pixels.data());
        c2rt_unpin_host_buffer(argb.pixels.data());
    } catch (const std::exception& e) {
        fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    c2rt_shutdown();
    return 0;
}
