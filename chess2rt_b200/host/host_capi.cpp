// C entry points over the C++ host mirror, for the Python harness (tests/, bench.py) — the same
// calls the headless executable makes: load a scene file with the reference-compatible loader,
// flatten it, render through libc2rt.so.  No torch types, no CPU rendering.
#include <algorithm>
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
    c2rt_scene* device = nullptr;  // for the render_device path
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

void c2rt_host_scene_free(c2rt_host_scene* h) {
    if (!h) return;
    if (h->device) c2rt_scene_destroy(h->device);
    delete h;
}

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
// index of the node the scene file names `name` (its place in c2rt_scene_desc's node arrays), -1 if there is none
int c2rt_host_scene_node_index(const c2rt_host_scene* h, const char* name) {
    const Scene& s = *h->scene;
    auto it = name ? s.namedEntities.nodes.find(name) : s.namedEntities.nodes.end();
    if (it == s.namedEntities.nodes.end()) return -1;
    for (size_t i = 0; i < s.nodes.size(); i++)
        if (s.nodes[i].get() == it->second) return (int)i;
    return -1;
}

// As if the scene file's entry of node `node` had been edited: its geometry becomes the one named `geometry` (NULL: kept), its
// Transform is reset and the given keys are applied the way the loader applies them (makeNode: scale, then rotate through
// scale as the reference does, then translate; NULL: key absent).  The flat description and both uploaded scenes (the
// render_device one and the Renderer's) follow with c2rt_scene_set_nodes.  A bad node index or geometry name changes nothing.
int c2rt_host_scene_place_node(c2rt_host_scene* h, int node, const char* geometry, const double* scale, const double* rotate,
                               const double* translate) {
    try {
        Scene& sc = *h->scene;
        if (node < 0 || (size_t)node >= sc.nodes.size()) {
            g_host_err = "place_node: node index " + std::to_string(node) + " out of range (" + std::to_string(sc.nodes.size()) + " nodes)";
            return C2RT_ERR_INVALID_ARG;
        }
        const Geometry* g = nullptr;
        if (geometry) {
            auto it = sc.namedEntities.geometries.find(geometry);
            if (it == sc.namedEntities.geometries.end()) {
                g_host_err = std::string("place_node: no geometry named \"") + geometry + "\"";
                return C2RT_ERR_INVALID_ARG;
            }
            g = it->second;
        }
        Node& nd = *sc.nodes[node];
        if (g) nd.geom = g;
        nd.transform.reset();
        if (scale) nd.transform.scale(scale[0], scale[1], scale[2]);
        if (rotate) nd.transform.scale(rotate[0], rotate[1], rotate[2]);   // sic: scene_loader.cpp makeNode, node.d:89-90
        if (translate) nd.transform.translate(Vector(translate[0], translate[1], translate[2]));
        const FlatNode f = flattenNode(sc, nd);
        if (h->flat_valid) {   // in place: the pointers c2rt_host_scene_desc handed out stay valid
            FlatScene& fl = h->flat;
            fl.node_geom[node] = f.geom;
            std::copy(f.transform, f.transform + 9, fl.node_transform.begin() + 9 * node);
            std::copy(f.inverse, f.inverse + 9, fl.node_inverse.begin() + 9 * node);
            std::copy(f.inverse_t, f.inverse_t + 9, fl.node_inverse_t.begin() + 9 * node);
            std::copy(f.offset, f.offset + 3, fl.node_offset.begin() + 3 * node);
        }
        sc.nodesEdited({node});
        if (h->device) {
            const uint32_t id = (uint32_t)node;
            int rc = c2rt_scene_set_nodes(h->device, 1, &id, &f.geom, f.transform, f.inverse, f.inverse_t, f.offset);
            if (rc != C2RT_OK) {
                g_host_err = std::string("libc2rt: ") + c2rt_last_error();
                c2rt_scene_destroy(h->device);   // the next use re-creates it from the edited scene
                h->device = nullptr;
                return rc;
            }
        }
        return 0;
    } catch (const BackendException& e) {
        g_host_err = e.what();
        return e.status;
    } catch (const std::exception& e) {
        g_host_err = e.what();
        return C2RT_ERR_INVALID_ARG;
    }
}

}  // extern "C"

namespace {

int refuse(const std::string& message) {
    g_host_err = message;
    return C2RT_ERR_INVALID_ARG;
}

// An edit of the host scene, `edit` (which checks every argument before it changes anything), under the error handling of the
// entry points: a library error is its c2rt status, any other exception C2RT_ERR_INVALID_ARG
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

// The render_device scene follows an edit of entity `index` through `set` (flatten.hpp setShaders, ...); on a library error it
// is dropped, and the next use re-creates it from the edited scene
template <class Set>
int followDevice(c2rt_host_scene* h, int index, Set set) {
    if (!h->device) return 0;
    int rc = set(h->device, *h->scene, {index});
    if (rc != C2RT_OK) {
        g_host_err = std::string("libc2rt: ") + c2rt_last_error();
        c2rt_scene_destroy(h->device);
        h->device = nullptr;
    }
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

// As if node `node`'s `shader` key in the scene file named `shader`.  The flat description and both uploaded scenes (the
// render_device one and the Renderer's) follow with c2rt_scene_set_node_shaders.  A bad index or name changes nothing.
int c2rt_host_scene_set_node_shader(c2rt_host_scene* h, int node, const char* shader) {
    return guarded([&]() -> int {
        Scene& sc = *h->scene;
        if (!inRange(node, sc.nodes.size(), "node", "set_node_shader")) return C2RT_ERR_INVALID_ARG;
        auto it = shader ? sc.namedEntities.shaders.find(shader) : sc.namedEntities.shaders.end();
        if (it == sc.namedEntities.shaders.end()) return refuse(std::string("set_node_shader: no shader named \"") + (shader ? shader : "") + "\"");
        Node& nd = *sc.nodes[node];
        nd.shader = it->second;
        if (h->flat_valid) h->flat.node_shader[node] = flattenNode(sc, nd).shader;   // in place: handed-out pointers stay valid
        sc.nodeShadersEdited({node});
        return followDevice(h, node, setNodeShaders);
    });
}

// As if shader `shader`'s entry in the scene file had been edited: `kind` ("Lambert" or "Phong"; NULL keeps the object)
// replaces it with a fresh object of that kind, with that kind's defaults, under the same name and index; then the given keys
// apply as the loader applies them (Phong's exponent and strength clamped).  texture: a texture name, "" for none, NULL keeps
// it; exponent and strength are Phong keys.  The flat description and both uploaded scenes follow with c2rt_scene_set_shaders.
// A bad index, kind, texture name or key changes nothing.
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
        if (h->flat_valid) {
            const FlatShader f = flattenShader(sc, s);
            FlatScene& fl = h->flat;
            fl.shader_type[shader] = f.type;
            fl.shader_texture[shader] = f.texture;
            std::copy(f.color, f.color + 3, fl.shader_color.begin() + 3 * shader);
            fl.shader_exponent[shader] = f.exponent;
            fl.shader_strength[shader] = f.strength;
        }
        sc.shadersEdited({shader});
        return followDevice(h, shader, setShaders);
    });
}

// As if texture `texture`'s entry in the scene file had its given keys replaced (NULL: kept).  Checker: color1, color2 [3],
// size; Procedure2: colorU, colorV [9] (three colours), freqU, freqV [3]; BitmapTexture: scaling.  A texture keeps its kind,
// file and gamma.  The flat description and both uploaded scenes follow with c2rt_scene_set_textures.  A bad index or a key
// of another kind changes nothing.
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
        if (h->flat_valid) {
            const FlatTexture f = flattenTexture(t);
            std::copy(f.colors, f.colors + 18, h->flat.tex_colors.begin() + 18 * texture);
            std::copy(f.params, f.params + 6, h->flat.tex_params.begin() + 6 * texture);
        }
        sc.texturesEdited({texture});
        return followDevice(h, texture, setTextures);
    });
}

// As if light `light`'s entry in the scene file had its given keys (pos [3], color [3], power) replaced (NULL: kept).  The flat
// description and both uploaded scenes follow with c2rt_scene_set_lights.  A bad index changes nothing.
int c2rt_host_scene_set_light(c2rt_host_scene* h, int light, const double* pos, const float* color, const float* power) {
    return guarded([&]() -> int {
        Scene& sc = *h->scene;
        if (!inRange(light, sc.lights.size(), "light", "set_light")) return C2RT_ERR_INVALID_ARG;
        auto& l = dynamic_cast<PointLight&>(*sc.lights[light]);
        if (pos) l.pos = Vector(pos[0], pos[1], pos[2]);
        if (color) l.lightColor = Color(color[0], color[1], color[2]);
        if (power) l.lightPower = *power;
        if (h->flat_valid) {
            const FlatLight f = flattenLight(l);
            std::copy(f.pos, f.pos + 3, h->flat.light_pos.begin() + 3 * light);
            std::copy(f.color, f.color + 3, h->flat.light_color.begin() + 3 * light);
            h->flat.light_power[light] = f.power;
        }
        sc.lightsEdited({light});
        return followDevice(h, light, setLights);
    });
}

// per-frame blocks: runs scene.beginFrame() first, like renderSceneAsync (renderer.d:31)
void c2rt_host_frame_blocks(c2rt_host_scene* h, uint64_t seed, int count_rays, c2rt_camera* cam, c2rt_settings* set) {
    h->scene->beginFrame();
    *cam = flattenCamera(h->scene->camera);
    *set = flattenSettings(h->scene->settings, seed, count_rays != 0);
}
// uploaded scene for c2rt_render_device (created on first use under the current c2rt_init)
c2rt_scene* c2rt_host_device_scene(c2rt_host_scene* h) {
    if (h->device) return h->device;
    const c2rt_scene_desc* d = c2rt_host_scene_desc(h);
    if (!d) return nullptr;
    int rc = c2rt_scene_create(d, &h->device);
    if (rc != C2RT_OK) {
        g_host_err = std::string("libc2rt: ") + c2rt_last_error();
        h->device = nullptr;
    }
    return h->device;
}

// Renderer(scene, output).renderRT() with HOST buffers (rgb: W*H*3 floats, argb nullable)
int c2rt_host_render(c2rt_host_scene* h, float* rgb, uint32_t* argb, uint64_t seed, int count_rays, c2rt_stats* stats) {
    try {
        Scene& sc = *h->scene;
        const uint32_t W = sc.settings.frameWidth, H = sc.settings.frameHeight;
        sc.beginFrame();
        // render straight into the caller's buffer: borrow it as the Image's storage
        c2rt_camera cam = flattenCamera(sc.camera);
        c2rt_settings set = flattenSettings(sc.settings, seed, count_rays != 0);
        c2rt_scene* dev = c2rt_host_device_scene(h);
        if (!dev) return C2RT_ERR_CUDA;
        (void)W; (void)H;
        int rc = c2rt_render(dev, &cam, &set, rgb, argb, stats);
        if (rc != C2RT_OK) g_host_err = std::string("libc2rt: ") + c2rt_last_error();
        return rc;
    } catch (const std::exception& e) {
        g_host_err = e.what();
        return C2RT_ERR_INVALID_ARG;
    }
}

// renderPixel's hit record for every pixel into caller-owned HOST planes (c2rt_render_hits; `seed`: DOF / stereo frames)
int c2rt_host_render_hits(c2rt_host_scene* h, const c2rt_hit_planes* planes, uint64_t seed, c2rt_stats* stats) {
    try {
        Scene& sc = *h->scene;
        sc.beginFrame();
        c2rt_camera cam = flattenCamera(sc.camera);
        c2rt_settings set = flattenSettings(sc.settings, seed, false);
        c2rt_scene* dev = c2rt_host_device_scene(h);
        if (!dev) return C2RT_ERR_CUDA;
        int rc = c2rt_render_hits(dev, &cam, &set, planes, stats);
        if (rc != C2RT_OK) g_host_err = std::string("libc2rt: ") + c2rt_last_error();
        return rc;
    } catch (const std::exception& e) {
        g_host_err = e.what();
        return C2RT_ERR_INVALID_ARG;
    }
}

// the closest hit of n caller-supplied rays into caller-owned HOST arrays (c2rt_trace_rays)
int c2rt_host_trace_rays(c2rt_host_scene* h, size_t n, const double* origins, const double* dirs, const c2rt_ray_hits* out,
                         c2rt_stats* stats) {
    try {
        c2rt_scene* dev = c2rt_host_device_scene(h);
        if (!dev) return C2RT_ERR_CUDA;
        int rc = c2rt_trace_rays(dev, n, origins, dirs, out, stats);
        if (rc != C2RT_OK) g_host_err = std::string("libc2rt: ") + c2rt_last_error();
        return rc;
    } catch (const std::exception& e) {
        g_host_err = e.what();
        return C2RT_ERR_INVALID_ARG;
    }
}

// testVisibility(from[i], to[i]) for n pairs into a caller-owned HOST array (c2rt_test_visibility)
int c2rt_host_test_visibility(c2rt_host_scene* h, size_t n, const double* from, const double* to, uint8_t* visible, c2rt_stats* stats) {
    try {
        c2rt_scene* dev = c2rt_host_device_scene(h);
        if (!dev) return C2RT_ERR_CUDA;
        int rc = c2rt_test_visibility(dev, n, from, to, visible, stats);
        if (rc != C2RT_OK) g_host_err = std::string("libc2rt: ") + c2rt_last_error();
        return rc;
    } catch (const std::exception& e) {
        g_host_err = e.what();
        return C2RT_ERR_INVALID_ARG;
    }
}

// trace(ray) at depth 0 for n caller-supplied rays into caller-owned HOST arrays (c2rt_shade_rays; rgb / argb nullable), with
// the scene file's ambientLightColor
int c2rt_host_shade_rays(c2rt_host_scene* h, size_t n, const double* origins, const double* dirs, float* rgb, uint32_t* argb,
                         c2rt_stats* stats) {
    try {
        const Color& amb = h->scene->settings.ambientLightColor;
        const float ambient[3] = {amb.r, amb.g, amb.b};
        c2rt_scene* dev = c2rt_host_device_scene(h);
        if (!dev) return C2RT_ERR_CUDA;
        int rc = c2rt_shade_rays(dev, ambient, n, origins, dirs, rgb, argb, stats);
        if (rc != C2RT_OK) g_host_err = std::string("libc2rt: ") + c2rt_last_error();
        return rc;
    } catch (const std::exception& e) {
        g_host_err = e.what();
        return C2RT_ERR_INVALID_ARG;
    }
}

// renderPixel(scene, output, x, y) (renderer.d:46-57)
int c2rt_host_render_pixel(c2rt_host_scene* h, int x, int y, float rgb[3], c2rt_hit* hit) {
    try {
        Scene& sc = *h->scene;
        sc.beginFrame();
        c2rt_camera cam = flattenCamera(sc.camera);
        c2rt_settings set = flattenSettings(sc.settings, 0, false);
        c2rt_scene* dev = c2rt_host_device_scene(h);
        if (!dev) return C2RT_ERR_CUDA;
        int rc = c2rt_render_pixel(dev, &cam, &set, x, y, rgb, hit);
        if (rc != C2RT_OK) g_host_err = std::string("libc2rt: ") + c2rt_last_error();
        return rc;
    } catch (const std::exception& e) {
        g_host_err = e.what();
        return C2RT_ERR_INVALID_ARG;
    }
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
