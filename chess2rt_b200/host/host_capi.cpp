// C entry points over the C++ host mirror, for the Python harness (tests/, bench.py) — the same
// calls the headless executable makes: load a scene file with the reference-compatible loader,
// flatten it, render through libc2rt.so.  No torch types, no CPU rendering.
#include <cstring>
#include <string>

#include "flatten.hpp"
#include "renderer.hpp"

using namespace rt;

struct c2rt_host_scene {
    std::unique_ptr<Scene> scene;
    FlatScene flat;          // kept alive: c2rt_host_scene_desc() hands out pointers into it
    c2rt_scene_desc desc;
    bool flat_valid = false;
};

static thread_local std::string g_host_err;

extern "C" {

const char* c2rt_host_last_error(void) { return g_host_err.c_str(); }

c2rt_host_scene* c2rt_host_scene_load(const char* path) {
    try {
        auto h = new c2rt_host_scene;
        h->scene = parseSceneFromFile(path);
        return h;
    } catch (const std::exception& e) {
        g_host_err = e.what();
        return nullptr;
    }
}

void c2rt_host_scene_free(c2rt_host_scene* h) { delete h; }

// as if the scene file had been edited: settings.frameWidth/Height + camera.setFrameSize (camera.d:254)
void c2rt_host_scene_set_frame_size(c2rt_host_scene* h, uint32_t w, uint32_t hgt) {
    h->scene->settings.frameWidth = w;
    h->scene->settings.frameHeight = hgt;
    h->scene->camera.setFrameSize(w, hgt);
}
void c2rt_host_scene_get_frame_size(const c2rt_host_scene* h, uint32_t* w, uint32_t* hgt) {
    *w = h->scene->settings.frameWidth;
    *hgt = h->scene->settings.frameHeight;
}
// -1 keeps the scene-file value
void c2rt_host_scene_override(c2rt_host_scene* h, int aa, int dof, int prepass, int num_samples) {
    if (aa >= 0) h->scene->settings.AAEnabled = aa != 0;
    if (dof >= 0) h->scene->camera.dof = dof != 0;
    if (prepass >= 0) h->scene->settings.prepassEnabled = prepass != 0;
    if (num_samples >= 0) h->scene->camera.numSamples = (size_t)num_samples;
}

// flattened description (valid until the scene is freed)
const c2rt_scene_desc* c2rt_host_scene_desc(c2rt_host_scene* h) {
    try {
        if (!h->flat_valid) {
            h->flat = flatten(*h->scene);
            h->desc = h->flat.desc();
            h->flat_valid = true;
        }
        return &h->desc;
    } catch (const std::exception& e) {
        g_host_err = e.what();
        return nullptr;
    }
}
// The uploaded scene (Scene::deviceScene) every c2rt_host_* call renders through, created on first use under the current
// c2rt_init; the edits below change it in place.  NULL on an error.
c2rt_scene* c2rt_host_device_scene(c2rt_host_scene* h) {
    try {
        return uploadedScene(*h->scene);
    } catch (const std::exception& e) {
        g_host_err = e.what();
        return nullptr;
    }
}

}  // extern "C"

namespace {

int refuse(const std::string& message) {
    g_host_err = message;
    return C2RT_ERR_INVALID_ARG;
}

// An edit of the host scene, `edit` (which checks every argument before it changes anything), under the error handling of the
// entry points: a library error is its c2rt status, any other exception C2RT_ERR_INVALID_ARG.  An edit ends with its
// Scene::*Edited hook, which edits the uploaded scene in place or, on a library error, drops it (the next use re-creates it
// from the edited scene) and throws.
template <class F>
int guarded(F edit) {
    try {
        return edit();
    } catch (const BackendException& e) {
        g_host_err = e.what();
        return e.status;
    } catch (const std::exception& e) {
        g_host_err = e.what();
        return C2RT_ERR_INVALID_ARG;
    }
}

// `call` (a libc2rt call) on the uploaded scene: C2RT_ERR_CUDA when there is none, else the call's status, with the library's
// message for any status but C2RT_OK (C2RT_CANCELLED included)
template <class F>
int onDevice(c2rt_host_scene* h, F call) {
    c2rt_scene* dev = c2rt_host_device_scene(h);
    if (!dev) return C2RT_ERR_CUDA;
    int rc = call(dev);
    if (rc != C2RT_OK) g_host_err = std::string("libc2rt: ") + c2rt_last_error();
    return rc;
}

template <class T>
int indexIn(const std::vector<std::unique_ptr<T>>& v, const std::map<std::string, T*>& names, const char* name) {
    auto it = name ? names.find(name) : names.end();
    if (it == names.end()) return -1;
    for (size_t i = 0; i < v.size(); i++)
        if (v[i].get() == it->second) return (int)i;
    return -1;
}

template <class T>
const char* nameOf(const std::vector<std::unique_ptr<T>>& v, const std::map<std::string, T*>& names, int index) {
    if (index < 0 || (size_t)index >= v.size()) return nullptr;
    for (auto& named : names)
        if (named.second == v[index].get()) return named.first.c_str();
    return nullptr;
}

bool inRange(int i, size_t n, const char* what, const char* call) {
    if (i >= 0 && (size_t)i < n) return true;
    refuse(std::string(call) + ": " + what + " index " + std::to_string(i) + " out of range (" + std::to_string(n) + " " + what + "s)");
    return false;
}

const Texture*& shaderTexture(Shader& s) {
    if (auto* la = dynamic_cast<Lambert*>(&s)) return la->texture;
    return dynamic_cast<Phong&>(s).texture;
}

}  // namespace

extern "C" {

// index of the entity of `section` ("nodes", "shaders", "textures" or "lights") the scene file names `name` (its place in
// c2rt_scene_desc's arrays), -1 if there is none
int c2rt_host_scene_index(const c2rt_host_scene* h, const char* section, const char* name) {
    const Scene& s = *h->scene;
    const std::string sec = section ? section : "";
    if (sec == "nodes") return indexIn(s.nodes, s.namedEntities.nodes, name);
    if (sec == "shaders") return indexIn(s.shaders, s.namedEntities.shaders, name);
    if (sec == "textures") return indexIn(s.textures, s.namedEntities.textures, name);
    if (sec == "lights") return indexIn(s.lights, s.namedEntities.lights, name);
    return -1;
}

// the name the scene file gives entity `index` of `section` ("nodes", "shaders", "textures" or "lights"), NULL if it has none
const char* c2rt_host_scene_name(const c2rt_host_scene* h, const char* section, int index) {
    const Scene& s = *h->scene;
    const std::string sec = section ? section : "";
    if (sec == "nodes") return nameOf(s.nodes, s.namedEntities.nodes, index);
    if (sec == "shaders") return nameOf(s.shaders, s.namedEntities.shaders, index);
    if (sec == "textures") return nameOf(s.textures, s.namedEntities.textures, index);
    if (sec == "lights") return nameOf(s.lights, s.namedEntities.lights, index);
    return nullptr;
}

// As if the scene file's entry of node `node` had been edited: its geometry becomes the one named `geometry` (NULL: kept), its
// Transform is reset and the given keys are applied the way the loader applies them (makeNode: scale, then rotate through
// scale as the reference does, then translate; NULL: key absent).  The flat description and the uploaded scene follow
// (Scene::nodesEdited).  A bad node index or geometry name changes nothing.
int c2rt_host_scene_place_node(c2rt_host_scene* h, int node, const char* geometry, const double* scale, const double* rotate,
                               const double* translate) {
    return guarded([&]() -> int {
        Scene& sc = *h->scene;
        if (!inRange(node, sc.nodes.size(), "node", "place_node")) return C2RT_ERR_INVALID_ARG;
        const Geometry* g = nullptr;
        if (geometry) {
            auto it = sc.namedEntities.geometries.find(geometry);
            if (it == sc.namedEntities.geometries.end()) return refuse(std::string("place_node: no geometry named \"") + geometry + "\"");
            g = it->second;
        }
        Node& nd = *sc.nodes[node];
        if (g) nd.geom = g;
        nd.transform.reset();
        if (scale) nd.transform.scale(scale[0], scale[1], scale[2]);
        if (rotate) nd.transform.scale(rotate[0], rotate[1], rotate[2]);   // sic: scene_loader.cpp makeNode, node.d:89-90
        if (translate) nd.transform.translate(Vector(translate[0], translate[1], translate[2]));
        if (h->flat_valid) h->flat.put(node, flattenNode(sc, nd));   // in place: handed-out pointers stay valid
        sc.nodesEdited({node});
        return 0;
    });
}

// As if node `node`'s `shader` key in the scene file named `shader`.  The flat description and the uploaded scene follow
// (Scene::nodeShadersEdited).  A bad index or name changes nothing.
int c2rt_host_scene_set_node_shader(c2rt_host_scene* h, int node, const char* shader) {
    return guarded([&]() -> int {
        Scene& sc = *h->scene;
        if (!inRange(node, sc.nodes.size(), "node", "set_node_shader")) return C2RT_ERR_INVALID_ARG;
        auto it = shader ? sc.namedEntities.shaders.find(shader) : sc.namedEntities.shaders.end();
        if (it == sc.namedEntities.shaders.end()) return refuse(std::string("set_node_shader: no shader named \"") + (shader ? shader : "") + "\"");
        Node& nd = *sc.nodes[node];
        nd.shader = it->second;
        if (h->flat_valid) h->flat.put(node, flattenNode(sc, nd));
        sc.nodeShadersEdited({node});
        return 0;
    });
}

// As if shader `shader`'s entry in the scene file had been edited: `kind` ("Lambert" or "Phong"; NULL keeps the object)
// replaces it with a fresh object of that kind, with that kind's defaults, under the same name and index; then the given keys
// apply as the loader applies them (Phong's exponent and strength clamped).  texture: a texture name, "" for none, NULL keeps
// it; exponent and strength are Phong keys.  The flat description and the uploaded scene follow (Scene::shadersEdited).  A bad
// index, kind, texture name or key changes nothing.
int c2rt_host_scene_set_shader(c2rt_host_scene* h, int shader, const char* kind, const float* color, const char* texture,
                               const double* exponent, const float* strength) {
    return guarded([&]() -> int {
        Scene& sc = *h->scene;
        if (!inRange(shader, sc.shaders.size(), "shader", "set_shader")) return C2RT_ERR_INVALID_ARG;
        const std::string k = kind ? kind : "";
        if (kind && k != "Lambert" && k != "Phong") return refuse("set_shader: unknown shader kind \"" + k + "\"");
        const Texture* tex = nullptr;
        if (texture && texture[0]) {
            auto it = sc.namedEntities.textures.find(texture);
            if (it == sc.namedEntities.textures.end()) return refuse(std::string("set_shader: no texture named \"") + texture + "\"");
            tex = it->second;
        }
        const bool phong = kind ? k == "Phong" : dynamic_cast<const Phong*>(sc.shaders[shader].get()) != nullptr;
        if (!phong && (exponent || strength)) return refuse("set_shader: exponent and strength are Phong keys; the shader is a Lambert");
        if (kind) {   // a fresh object in the same slot: the nodes and the name that referred to the old one refer to it
            std::unique_ptr<Shader> fresh;
            if (phong) fresh = std::make_unique<Phong>();
            else fresh = std::make_unique<Lambert>();
            const Shader* old = sc.shaders[shader].get();
            for (auto& nd : sc.nodes)
                if (nd->shader == old) nd->shader = fresh.get();
            for (auto& named : sc.namedEntities.shaders)
                if (named.second == old) named.second = fresh.get();
            sc.shaders[shader] = std::move(fresh);
        }
        Shader& s = *sc.shaders[shader];
        if (color) s.color = Color(color[0], color[1], color[2]);
        if (texture) shaderTexture(s) = tex;
        if (exponent) static_cast<Phong&>(s).exponent = Phong::clampExponent(*exponent);
        if (strength) static_cast<Phong&>(s).strength = Phong::clampStrength(*strength);
        if (h->flat_valid) h->flat.put(shader, flattenShader(sc, s));
        sc.shadersEdited({shader});
        return 0;
    });
}

// As if texture `texture`'s entry in the scene file had its given keys replaced (NULL: kept).  Checker: color1, color2 [3],
// size; Procedure2: colorU, colorV [9] (three colours), freqU, freqV [3]; BitmapTexture: scaling.  A texture keeps its kind,
// file and gamma.  The flat description and the uploaded scene follow (Scene::texturesEdited).  A bad index
// or a key of another kind changes nothing.
int c2rt_host_scene_set_texture(c2rt_host_scene* h, int texture, const float* color1, const float* color2, const double* size,
                                const float* colorU, const float* colorV, const double* freqU, const double* freqV,
                                const float* scaling) {
    return guarded([&]() -> int {
        Scene& sc = *h->scene;
        if (!inRange(texture, sc.textures.size(), "texture", "set_texture")) return C2RT_ERR_INVALID_ARG;
        Texture& t = *sc.textures[texture];
        auto* ch = dynamic_cast<Checker*>(&t);
        auto* pr = dynamic_cast<Procedure2*>(&t);
        auto* bm = dynamic_cast<BitmapTexture*>(&t);
        if (!ch && (color1 || color2 || size)) return refuse("set_texture: color1, color2 and size are Checker keys");
        if (!pr && (colorU || colorV || freqU || freqV)) return refuse("set_texture: colorU, colorV, freqU and freqV are Procedure2 keys");
        if (!bm && scaling) return refuse("set_texture: scaling is a BitmapTexture key");
        auto colors3 = [](const float* c) { return std::vector<Color>{Color(c[0], c[1], c[2]), Color(c[3], c[4], c[5]), Color(c[6], c[7], c[8])}; };
        if (color1) ch->color1 = Color(color1[0], color1[1], color1[2]);
        if (color2) ch->color2 = Color(color2[0], color2[1], color2[2]);
        if (size) ch->size = *size;
        if (colorU) pr->colorU = colors3(colorU);
        if (colorV) pr->colorV = colors3(colorV);
        if (freqU) pr->freqU.assign(freqU, freqU + 3);
        if (freqV) pr->freqV.assign(freqV, freqV + 3);
        if (scaling) bm->scaling = *scaling;
        if (h->flat_valid) h->flat.put(texture, flattenTexture(t));
        sc.texturesEdited({texture});
        return 0;
    });
}

// As if light `light`'s entry in the scene file had its given keys (pos [3], color [3], power) replaced (NULL: kept).  The flat
// description and the uploaded scene follow (Scene::lightsEdited).  A bad index changes nothing.
int c2rt_host_scene_set_light(c2rt_host_scene* h, int light, const double* pos, const float* color, const float* power) {
    return guarded([&]() -> int {
        Scene& sc = *h->scene;
        if (!inRange(light, sc.lights.size(), "light", "set_light")) return C2RT_ERR_INVALID_ARG;
        auto& l = dynamic_cast<PointLight&>(*sc.lights[light]);
        if (pos) l.pos = Vector(pos[0], pos[1], pos[2]);
        if (color) l.lightColor = Color(color[0], color[1], color[2]);
        if (power) l.lightPower = *power;
        if (h->flat_valid) h->flat.put(light, flattenLight(l));
        sc.lightsEdited({light});
        return 0;
    });
}

// per-frame blocks: runs scene.beginFrame() first, like renderSceneAsync (renderer.d:31)
void c2rt_host_frame_blocks(c2rt_host_scene* h, uint64_t seed, int count_rays, c2rt_camera* cam, c2rt_settings* set) {
    h->scene->beginFrame();
    *cam = flattenCamera(h->scene->camera);
    *set = flattenSettings(h->scene->settings, seed, count_rays != 0);
}
// Renderer(scene, output).renderRT() with HOST buffers (rgb: W*H*3 floats, argb nullable)
int c2rt_host_render(c2rt_host_scene* h, float* rgb, uint32_t* argb, uint64_t seed, int count_rays, c2rt_stats* stats) {
    Scene& sc = *h->scene;
    sc.beginFrame();
    const c2rt_camera cam = flattenCamera(sc.camera);
    const c2rt_settings set = flattenSettings(sc.settings, seed, count_rays != 0);
    return onDevice(h, [&](c2rt_scene* dev) { return c2rt_render(dev, &cam, &set, rgb, argb, stats); });
}

// c2rt_host_render's frame through the scene's frame cache (c2rt_render_update): rgb / argb must be what the last
// c2rt_host_render_update of this scene wrote into them
int c2rt_host_render_update(c2rt_host_scene* h, float* rgb, uint32_t* argb, uint64_t seed, int count_rays, c2rt_stats* stats,
                            c2rt_update_info* info) {
    Scene& sc = *h->scene;
    sc.beginFrame();
    const c2rt_camera cam = flattenCamera(sc.camera);
    const c2rt_settings set = flattenSettings(sc.settings, seed, count_rays != 0);
    return onDevice(h, [&](c2rt_scene* dev) { return c2rt_render_update(dev, &cam, &set, frameCache(sc), rgb, argb, stats, info); });
}

// renderPixel's hit record for every pixel into caller-owned HOST planes (c2rt_render_hits; `seed`: DOF / stereo frames)
int c2rt_host_render_hits(c2rt_host_scene* h, const c2rt_hit_planes* planes, uint64_t seed, c2rt_stats* stats) {
    Scene& sc = *h->scene;
    sc.beginFrame();
    const c2rt_camera cam = flattenCamera(sc.camera);
    const c2rt_settings set = flattenSettings(sc.settings, seed, false);
    return onDevice(h, [&](c2rt_scene* dev) { return c2rt_render_hits(dev, &cam, &set, planes, stats); });
}

// the closest hit of n caller-supplied rays into caller-owned HOST arrays (c2rt_trace_rays)
int c2rt_host_trace_rays(c2rt_host_scene* h, size_t n, const double* origins, const double* dirs, const c2rt_ray_hits* out,
                         c2rt_stats* stats) {
    return onDevice(h, [&](c2rt_scene* dev) { return c2rt_trace_rays(dev, n, origins, dirs, out, stats); });
}

// testVisibility(from[i], to[i]) for n pairs into a caller-owned HOST array (c2rt_test_visibility)
int c2rt_host_test_visibility(c2rt_host_scene* h, size_t n, const double* from, const double* to, uint8_t* visible, c2rt_stats* stats) {
    return onDevice(h, [&](c2rt_scene* dev) { return c2rt_test_visibility(dev, n, from, to, visible, stats); });
}

// trace(ray) at depth 0 for n caller-supplied rays into caller-owned HOST arrays (c2rt_shade_rays; rgb / argb nullable), with
// the scene file's ambientLightColor
int c2rt_host_shade_rays(c2rt_host_scene* h, size_t n, const double* origins, const double* dirs, float* rgb, uint32_t* argb,
                         c2rt_stats* stats) {
    const Color& amb = h->scene->settings.ambientLightColor;
    const float ambient[3] = {amb.r, amb.g, amb.b};
    return onDevice(h, [&](c2rt_scene* dev) { return c2rt_shade_rays(dev, ambient, n, origins, dirs, rgb, argb, stats); });
}

// renderPixel(scene, output, x, y) (renderer.d:46-57)
int c2rt_host_render_pixel(c2rt_host_scene* h, int x, int y, float rgb[3], c2rt_hit* hit) {
    Scene& sc = *h->scene;
    sc.beginFrame();
    const c2rt_camera cam = flattenCamera(sc.camera);
    const c2rt_settings set = flattenSettings(sc.settings, 0, false);
    return onDevice(h, [&](c2rt_scene* dev) { return c2rt_render_pixel(dev, &cam, &set, x, y, rgb, hit); });
}

// camera.d:211-229 rotate / :181-204 move — what the GUI's key handlers call between frames (raytracer_demo.d:268-340)
void c2rt_host_camera_rotate(c2rt_host_scene* h, double dYaw, double dRoll, double dPitch) { h->scene->camera.rotate(dYaw, dRoll, dPitch); }
void c2rt_host_camera_move(c2rt_host_scene* h, double dx, double dy, double dz) { h->scene->camera.move(dx, dy, dz); }

// saveBmp (imageio/bmp.d:195-237) of a packed Color.toRGB32 plane; returns the byte count (0 if `cap` is too small)
size_t c2rt_host_save_bmp(const uint32_t* argb, uint32_t w, uint32_t hgt, int pad_rows, uint8_t* out, size_t cap) {
    Image<uint32_t> img(w, hgt);
    memcpy(img.pixels.data(), argb, (size_t)w * hgt * sizeof(uint32_t));
    std::vector<uint8_t> bytes = saveBmp(img, pad_rows != 0);
    if (bytes.size() > cap) return 0;
    memcpy(out, bytes.data(), bytes.size());
    return bytes.size();
}

// scene summary for tests: nodes, geoms, shaders, textures, lights, AA, dof, numSamples
void c2rt_host_scene_info(const c2rt_host_scene* h, int32_t out[8]) {
    const Scene& s = *h->scene;
    out[0] = (int32_t)s.nodes.size();
    out[1] = (int32_t)s.geometries.size();
    out[2] = (int32_t)s.shaders.size();
    out[3] = (int32_t)s.textures.size();
    out[4] = (int32_t)s.lights.size();
    out[5] = s.settings.AAEnabled;
    out[6] = s.camera.dof;
    out[7] = (int32_t)s.camera.numSamples;
}

// BMP decode through the host loader (for the reference's BMP known-answer tests): packed 0x00RRGGBB
int c2rt_host_decode_bmp(const uint8_t* bytes, size_t n, uint32_t* w, uint32_t* hgt, uint32_t* out, size_t cap) {
    try {
        Image<Color> img = loadBmpImage(std::vector<uint8_t>(bytes, bytes + n));
        *w = (uint32_t)img.width;
        *hgt = (uint32_t)img.height;
        if (img.width * img.height > cap) { g_host_err = "output too small"; return C2RT_ERR_INVALID_ARG; }
        for (size_t i = 0; i < img.width * img.height; i++) {
            const Color& c = img.pixels[i];
            out[i] = ((uint32_t)lrintf(c.r * 255.f) << 16) | ((uint32_t)lrintf(c.g * 255.f) << 8) | (uint32_t)lrintf(c.b * 255.f);
        }
        return 0;
    } catch (const std::exception& e) {
        g_host_err = e.what();
        return C2RT_ERR_INVALID_ARG;
    }
}

}  // extern "C"
