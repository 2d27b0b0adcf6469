// The renderer seam, re-pointed at libc2rt.so.  Same entry points and argument meaning as
// /root/reference/source/rt/renderer.d:
//   renderSceneAsync :23-44   scene.beginFrame(); render on a spawned thread; clears *isRendering when done
//   renderPixel      :46-57   one un-antialiased sample + TraceResult for the debug pixel pick
//   Renderer         :59-189  Renderer(scene, output[, isRendering, isStopRequested]).renderRT()
// The body of renderRT (bucket list, prepass, 1-spp pass, AA pass over a CPU TaskPool) is replaced
// by one call of c2rt_render; the prepass and the dead needsAA mask have no pixel effect and are
// dropped (SURVEY.md §7 "dead work").  Errors from the backend surface as rt::BackendException;
// there is no CPU fallback.
#pragma once
#include <atomic>
#include <thread>
#include <tuple>

#include "flatten.hpp"
#include "rt.hpp"

namespace rt {

struct TraceResult {  // renderer.d:14-21 (closestNode as an index into scene.nodes, -1 = miss)
    int closestNode = -1;
    double dist = 1e99;
    Vector p, normal;
    double u = NAN, v = NAN;
    bool hitLight = false;
    Color hitLightColor;
};

struct RenderOptions {        // knobs the reference does not have
    uint64_t rngSeed = 0;     // seed of the pinned DOF generator (SURVEY.md F4)
    bool countRays = false;   // fill lastStats.primary_rays / shadow_rays
    Image<uint32_t>* argb = nullptr;  // optional Color.toRGB32 plane produced on the GPU
    bool argbOnly = false;    // interactive hosts that only blit `argb` (sdl2_gui.d:139-155): the float frame is neither written nor copied
};

// renderPixel's hit record for every pixel of the frame (c2rt_render_hits): structure of arrays, row-major, top row first.
// renderHits fills the planes that are not empty; a non-empty plane must hold exactly W * H records.
struct HitPlanes {
    std::vector<int32_t> node;   // [W*H] closestNode, -1 = miss
    std::vector<float> dist;     // [W*H] hit distance, +inf for a miss
    std::vector<float> normal;   // [W*H*3] unit geometric normal, 0 for a miss
    std::vector<float> uv;       // [W*H*2] u, v, 0 for a miss
};

// The closest-hit records of caller-supplied rays (c2rt_trace_rays): one entry per ray, structure of arrays.  traceRays fills
// the planes that are not empty; a non-empty plane must hold exactly as many records as there are rays.
struct RayHits {
    std::vector<int32_t> node;   // [n] closestNode, -1 = miss
    std::vector<double> dist;    // [n] distance along the unit direction, +inf for a miss
    std::vector<double> p;       // [n*3] world-space hit point, 0 for a miss
    std::vector<double> normal;  // [n*3] unit geometric normal, 0 for a miss
    std::vector<double> uv;      // [n*2] u, v, 0 for a miss
};

struct Renderer {
    Renderer(const Scene& scene, Image<Color>& output, std::atomic<bool>* isRendering = nullptr,
             const std::atomic<bool>* isStopRequested = nullptr);

    void renderRT();                               // renderer.d:83-189
    // renderRT's frame, bit for bit, re-rendering only the tiles the scene's edits since the last renderUpdate can have changed
    // (c2rt_render_update with the scene's frameCache).  The output image and options.argb must be the buffers the last
    // renderUpdate of this scene wrote, unchanged since; lastUpdate tells how many tiles were rendered.
    void renderUpdate();
    void renderHits(HitPlanes& planes);            // no counterpart: renderPixelNoAA's hit record for every pixel, no colour
    Color renderPixelNoAA(int x, int y);           // renderer.d:223-228 (also records lastTracingResult)
    // renderer.d:325-376's closest-hit loop on (orig[i], normalize(dir[i])) for every i (c2rt_trace_rays)
    void traceRays(const std::vector<Vector>& orig, const std::vector<Vector>& dir, RayHits& hits);
    // scene.d:62-78 testVisibility(from[i], to[i]) for every i: visible[i] = 1 or 0 (c2rt_test_visibility)
    void testVisibility(const std::vector<Vector>& from, const std::vector<Vector>& to, std::vector<uint8_t>& visible);
    // renderer.d:325-376 trace((orig[i], normalize(dir[i]))) at depth 0 for every i, with the scene's ambientLightColor
    // (c2rt_shade_rays): out[i] is the colour; argb (optional) gets Color.toRGB32 of it
    void shadeRays(const std::vector<Vector>& orig, const std::vector<Vector>& dir, std::vector<Color>& out,
                   std::vector<uint32_t>* argb = nullptr);

    TraceResult lastTracingResult;
    c2rt_stats lastStats{};
    c2rt_update_info lastUpdate{};                 // the last renderUpdate's tiles
    RenderOptions options;
    bool cancelled = false;                        // the last renderRT ended early on a stop request (the frame is partial)

private:
    void frame(bool update);
    const Scene& scene_;
    Image<Color>& output_;
    std::atomic<bool>* isRendering_;
    const std::atomic<bool>* isStopRequested_;
};

// Spawns the render thread like the reference does; `worker` (optional) receives the thread so a
// headless caller can join it instead of polling *isRendering.
void renderSceneAsync(Scene& scene, Image<Color>& output, std::atomic<bool>* isRendering,
                      const std::atomic<bool>* needsRendering, std::thread* worker = nullptr,
                      const RenderOptions& options = RenderOptions());

std::tuple<Color, TraceResult> renderPixel(Scene& scene, Image<Color>& output, int x, int y);

// The stop request of the reference (raytracer_demo.d:102-124 sets needsRendering; renderer.d:93-97,129,147,180 polls it between
// passes) for a frame that is already on the GPU: sets *isStopRequested like the GUI does and tells the backend, which skips
// every tile that has not started.  Callable from the GUI thread while the render thread is inside renderRT.
void requestStop(std::atomic<bool>* isStopRequested);

// c2rt_init wrapper: selects the GPUs the next frames are banded over (default: device 0 only).
void setRenderDevices(int nGpus, const int* deviceIds = nullptr);

// The scene's uploaded copy (Scene::deviceScene), which every frame and query renders through: created from flatten(scene) on
// first use, under the GPUs setRenderDevices selected, and kept until the scene drops it.  Throws BackendException on a library
// error (InvalidSceneException on a dangling reference).
c2rt_scene* uploadedScene(const Scene& scene);
// The scene's frame cache (Scene::frameCache) for c2rt_render_update, created on first use and kept with the scene.
c2rt_frame_cache* frameCache(const Scene& scene);

}  // namespace rt
