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
