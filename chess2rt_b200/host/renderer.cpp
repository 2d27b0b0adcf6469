#include "renderer.hpp"

#include <cstring>

namespace rt {
namespace {

[[noreturn]] void raise(int status) { throw BackendException(status, c2rt_last_error()); }

struct DeviceSceneHolder {
    c2rt_scene* handle = nullptr;
    ~DeviceSceneHolder() { c2rt_scene_destroy(handle); }
};

struct FrameCacheHolder {
    c2rt_frame_cache* handle = nullptr;
    ~FrameCacheHolder() { c2rt_frame_cache_destroy(handle); }
};

}  // namespace

void setRenderDevices(int nGpus, const int* deviceIds) {
    int rc = c2rt_init(nGpus, deviceIds);
    if (rc != C2RT_OK) raise(rc);
}

Renderer::Renderer(const Scene& scene, Image<Color>& output, std::atomic<bool>* isRendering, const std::atomic<bool>* isStopRequested)
    : scene_(scene), output_(output), isRendering_(isRendering), isStopRequested_(isStopRequested) {}

c2rt_scene* uploadedScene(const Scene& scene) {
    if (!scene.deviceScene) {
        FlatScene flat = flatten(scene);
        c2rt_scene_desc d = flat.desc();
        auto holder = std::make_shared<DeviceSceneHolder>();
        int rc = c2rt_scene_create(&d, &holder->handle);
        if (rc != C2RT_OK) raise(rc);
        scene.deviceScene = holder;
    }
    return static_cast<DeviceSceneHolder*>(scene.deviceScene.get())->handle;
}

c2rt_frame_cache* frameCache(const Scene& scene) {
    if (!scene.frameCache) {
        auto holder = std::make_shared<FrameCacheHolder>();
        int rc = c2rt_frame_cache_create(&holder->handle);
        if (rc != C2RT_OK) raise(rc);
        scene.frameCache = holder;
    }
    return static_cast<FrameCacheHolder*>(scene.frameCache.get())->handle;
}

namespace {

// An edit of the uploaded scene (when there is one) through `set` (flatten.hpp setShaders, ...)
template <class Set>
void editDeviceScene(Scene& scene, const std::vector<int>& indices, Set set) {
    if (!scene.deviceScene || indices.empty()) return;   // (no uploaded scene: the next frame flattens the whole scene)
    int rc = set(static_cast<DeviceSceneHolder*>(scene.deviceScene.get())->handle, scene, indices);
    if (rc != C2RT_OK) {
        scene.invalidateDeviceScene();   // the next frame re-creates it from the edited scene
        raise(rc);
    }
}

}  // namespace

void Scene::nodesEdited(const std::vector<int>& indices) { editDeviceScene(*this, indices, setNodes); }
void Scene::nodeShadersEdited(const std::vector<int>& indices) { editDeviceScene(*this, indices, setNodeShaders); }
void Scene::shadersEdited(const std::vector<int>& indices) { editDeviceScene(*this, indices, setShaders); }
void Scene::texturesEdited(const std::vector<int>& indices) { editDeviceScene(*this, indices, setTextures); }
void Scene::lightsEdited(const std::vector<int>& indices) { editDeviceScene(*this, indices, setLights); }

void Renderer::renderRT() { frame(false); }
void Renderer::renderUpdate() { frame(true); }

void Renderer::frame(bool update) {
    struct Done {  // renderer.d:87-91 end()
        std::atomic<bool>* flag;
        ~Done() { if (flag) flag->store(false); }
    } done{isRendering_};

    const uint32_t W = scene_.settings.frameWidth, H = scene_.settings.frameHeight;
    if (output_.width != W || output_.height != H || output_.pixels.size() < (size_t)W * H)
        throw RTException("output image size does not match settings.frameWidth x frameHeight");
    if (isStopRequested_ && isStopRequested_->load()) return;  // renderer.d:93-97,129

    c2rt_camera cam = flattenCamera(scene_.camera);
    c2rt_settings set = flattenSettings(scene_.settings, options.rngSeed, options.countRays);
    uint32_t* argb = nullptr;
    if (options.argb) {
        options.argb->alloc(W, H);
        argb = options.argb->pixels.data();
    }
    static_assert(sizeof(Color) == 3 * sizeof(float), "Color must be three packed floats (color.d:27-35)");
    if (options.argbOnly && !argb) throw RTException("argbOnly needs RenderOptions::argb");
    float* rgb = options.argbOnly ? nullptr : reinterpret_cast<float*>(output_.pixels.data());
    int rc = update ? c2rt_render_update(uploadedScene(scene_), &cam, &set, frameCache(scene_), rgb, argb, &lastStats, &lastUpdate)
                    : c2rt_render(uploadedScene(scene_), &cam, &set, rgb, argb, &lastStats);
    cancelled = rc == C2RT_CANCELLED;   // a stop request reached the frame in flight: return like the reference's `return end()`
    if (rc != C2RT_OK && !cancelled) raise(rc);
}

void Renderer::renderHits(HitPlanes& planes) {
    const size_t n = (size_t)scene_.settings.frameWidth * scene_.settings.frameHeight;
    if ((!planes.node.empty() && planes.node.size() != n) || (!planes.dist.empty() && planes.dist.size() != n) ||
        (!planes.normal.empty() && planes.normal.size() != 3 * n) || (!planes.uv.empty() && planes.uv.size() != 2 * n))
        throw RTException("hit plane size does not match settings.frameWidth x frameHeight");
    c2rt_camera cam = flattenCamera(scene_.camera);
    c2rt_settings set = flattenSettings(scene_.settings, options.rngSeed, false);
    c2rt_hit_planes p;
    p.node = planes.node.empty() ? nullptr : planes.node.data();
    p.dist = planes.dist.empty() ? nullptr : planes.dist.data();
    p.normal = planes.normal.empty() ? nullptr : planes.normal.data();
    p.uv = planes.uv.empty() ? nullptr : planes.uv.data();
    int rc = c2rt_render_hits(uploadedScene(scene_), &cam, &set, &p, &lastStats);
    if (rc != C2RT_OK) raise(rc);
}

namespace {
std::vector<double> flattenVectors(const std::vector<Vector>& v) {
    std::vector<double> out(v.size() * 3);
    for (size_t i = 0; i < v.size(); i++) { out[3 * i] = v[i].x; out[3 * i + 1] = v[i].y; out[3 * i + 2] = v[i].z; }
    return out;
}
}  // namespace

void Renderer::traceRays(const std::vector<Vector>& orig, const std::vector<Vector>& dir, RayHits& hits) {
    const size_t n = orig.size();
    if (dir.size() != n) throw RTException("traceRays: as many directions as origins are needed");
    if ((!hits.node.empty() && hits.node.size() != n) || (!hits.dist.empty() && hits.dist.size() != n) ||
        (!hits.p.empty() && hits.p.size() != 3 * n) || (!hits.normal.empty() && hits.normal.size() != 3 * n) ||
        (!hits.uv.empty() && hits.uv.size() != 2 * n))
        throw RTException("ray hit plane size does not match the number of rays");
    const std::vector<double> o = flattenVectors(orig), d = flattenVectors(dir);
    c2rt_ray_hits p;
    p.node = hits.node.empty() ? nullptr : hits.node.data();
    p.dist = hits.dist.empty() ? nullptr : hits.dist.data();
    p.p = hits.p.empty() ? nullptr : hits.p.data();
    p.normal = hits.normal.empty() ? nullptr : hits.normal.data();
    p.uv = hits.uv.empty() ? nullptr : hits.uv.data();
    int rc = c2rt_trace_rays(uploadedScene(scene_), n, o.data(), d.data(), &p, &lastStats);
    if (rc != C2RT_OK) raise(rc);
}

void Renderer::testVisibility(const std::vector<Vector>& from, const std::vector<Vector>& to, std::vector<uint8_t>& visible) {
    if (to.size() != from.size()) throw RTException("testVisibility: as many `to` points as `from` points are needed");
    const std::vector<double> f = flattenVectors(from), t = flattenVectors(to);
    visible.resize(from.size());
    int rc = c2rt_test_visibility(uploadedScene(scene_), from.size(), f.data(), t.data(), visible.data(), &lastStats);
    if (rc != C2RT_OK) raise(rc);
}

void Renderer::shadeRays(const std::vector<Vector>& orig, const std::vector<Vector>& dir, std::vector<Color>& out,
                         std::vector<uint32_t>* argb) {
    static_assert(sizeof(Color) == 3 * sizeof(float), "a Color[] is the rgb plane of c2rt_shade_rays");
    const size_t n = orig.size();
    if (dir.size() != n) throw RTException("shadeRays: as many directions as origins are needed");
    const std::vector<double> o = flattenVectors(orig), d = flattenVectors(dir);
    const Color& amb = scene_.settings.ambientLightColor;
    const float ambient[3] = {amb.r, amb.g, amb.b};
    out.resize(n);
    if (argb) argb->resize(n);
    int rc = c2rt_shade_rays(uploadedScene(scene_), ambient, n, o.data(), d.data(), reinterpret_cast<float*>(out.data()),
                             argb ? argb->data() : nullptr, &lastStats);
    if (rc != C2RT_OK) raise(rc);
}

void requestStop(std::atomic<bool>* isStopRequested) {
    if (isStopRequested) isStopRequested->store(true);
    c2rt_cancel();
}

Color Renderer::renderPixelNoAA(int x, int y) {
    c2rt_camera cam = flattenCamera(scene_.camera);
    c2rt_settings set = flattenSettings(scene_.settings, options.rngSeed, false);
    float rgb[3];
    c2rt_hit hit;
    int rc = c2rt_render_pixel(uploadedScene(scene_), &cam, &set, x, y, rgb, &hit);
    if (rc != C2RT_OK) raise(rc);
    Color c(rgb[0], rgb[1], rgb[2]);
    output_(x, y) = c;  // renderer.d:226
    lastTracingResult = TraceResult();
    lastTracingResult.closestNode = hit.node;
    lastTracingResult.dist = hit.dist;
    if (hit.node >= 0) {
        lastTracingResult.p = Vector(hit.p[0], hit.p[1], hit.p[2]);
        lastTracingResult.normal = Vector(hit.normal[0], hit.normal[1], hit.normal[2]);
        lastTracingResult.u = hit.u;
        lastTracingResult.v = hit.v;
    }
    return c;
}

void renderSceneAsync(Scene& scene, Image<Color>& output, std::atomic<bool>* isRendering, const std::atomic<bool>* needsRendering,
                      std::thread* worker, const RenderOptions& options) {
    scene.beginFrame();  // renderer.d:31
    std::thread t([&scene, &output, isRendering, needsRendering, options]() {
        Renderer renderer(scene, output, isRendering, needsRendering);
        renderer.options = options;
        try {
            renderer.renderRT();
        } catch (const std::exception& e) {
            // the reference's render thread has nowhere to report to either; keep the message visible
            fprintf(stderr, "render thread: %s\n", e.what());
        }
    });
    if (worker) *worker = std::move(t);
    else t.detach();
}

std::tuple<Color, TraceResult> renderPixel(Scene& scene, Image<Color>& output, int x, int y) {
    scene.beginFrame();  // renderer.d:50
    Renderer renderer(scene, output);
    Color color = renderer.renderPixelNoAA(x, y);
    return std::make_tuple(color, renderer.lastTracingResult);
}

}  // namespace rt
