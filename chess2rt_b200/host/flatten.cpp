#include "flatten.hpp"

#include <algorithm>
#include <cstring>
#include <string>

namespace rt {
namespace {

template <class T>
int indexOf(const std::vector<std::unique_ptr<T>>& v, const T* p) {
    for (size_t i = 0; i < v.size(); i++)
        if (v[i].get() == p) return (int)i;
    return -1;
}

void putMatrix(double dst[9], const Matrix& m) {
    for (int r = 0; r < 3; r++)
        for (int c = 0; c < 3; c++) dst[3 * r + c] = m.c[r][c];
}

// entry i of an array whose entries are N values each
template <class T, size_t N>
void putEntry(std::vector<T>& v, size_t i, const T (&entry)[N]) {
    std::copy(entry, entry + N, v.begin() + N * i);
}

}  // namespace

void FlatScene::resize(size_t nodes, size_t shaders, size_t textures, size_t lights) {
    node_geom.resize(nodes);
    node_shader.resize(nodes);
    node_transform.resize(9 * nodes);
    node_inverse.resize(9 * nodes);
    node_inverse_t.resize(9 * nodes);
    node_offset.resize(3 * nodes);
    shader_type.resize(shaders);
    shader_texture.resize(shaders);
    shader_color.resize(3 * shaders);
    shader_exponent.resize(shaders);
    shader_strength.resize(shaders);
    tex_type.resize(textures);
    tex_width.resize(textures);
    tex_height.resize(textures);
    tex_texel_offset.resize(textures);
    tex_colors.resize(18 * textures);
    tex_params.resize(6 * textures);
    light_pos.resize(3 * lights);
    light_color.resize(3 * lights);
    light_power.resize(lights);
}

void FlatScene::put(size_t i, const FlatNode& n) {
    node_geom[i] = n.geom;
    node_shader[i] = n.shader;
    putEntry(node_transform, i, n.transform);
    putEntry(node_inverse, i, n.inverse);
    putEntry(node_inverse_t, i, n.inverse_t);
    putEntry(node_offset, i, n.offset);
}

void FlatScene::put(size_t i, const FlatShader& s) {
    shader_type[i] = s.type;
    shader_texture[i] = s.texture;
    putEntry(shader_color, i, s.color);
    shader_exponent[i] = s.exponent;
    shader_strength[i] = s.strength;
}

void FlatScene::put(size_t i, const FlatTexture& t) {
    tex_type[i] = t.type;
    tex_width[i] = t.width;
    tex_height[i] = t.height;
    putEntry(tex_colors, i, t.colors);
    putEntry(tex_params, i, t.params);
}

void FlatScene::put(size_t i, const FlatLight& l) {
    putEntry(light_pos, i, l.pos);
    putEntry(light_color, i, l.color);
    light_power[i] = l.power;
}

FlatScene flatten(const Scene& scene) {
    FlatScene f;
    f.resize(scene.nodes.size(), scene.shaders.size(), scene.textures.size(), scene.lights.size());

    // geometries, in declaration order (CSG children are always earlier: geometry.d:343-347)
    for (size_t i = 0; i < scene.geometries.size(); i++) {
        const Geometry* g = scene.geometries[i].get();
        double p[4] = {0, 0, 0, 0};
        int type, left = -1, right = -1;
        if (auto* pl = dynamic_cast<const Plane*>(g)) {
            type = C2RT_GEOM_PLANE;
            p[0] = pl->y;
            p[1] = pl->limit;
        } else if (auto* sp = dynamic_cast<const Sphere*>(g)) {
            type = C2RT_GEOM_SPHERE;
            p[0] = sp->center.x; p[1] = sp->center.y; p[2] = sp->center.z; p[3] = sp->R;
        } else if (auto* cu = dynamic_cast<const Cube*>(g)) {
            type = C2RT_GEOM_CUBE;
            p[0] = cu->center.x; p[1] = cu->center.y; p[2] = cu->center.z; p[3] = cu->side;
        } else if (auto* op = dynamic_cast<const CsgOp*>(g)) {
            type = dynamic_cast<const CsgUnion*>(g) ? C2RT_GEOM_CSG_UNION : dynamic_cast<const CsgInter*>(g) ? C2RT_GEOM_CSG_INTER : C2RT_GEOM_CSG_DIFF;
            left = indexOf(scene.geometries, op->left);
            right = indexOf(scene.geometries, op->right);
            if (left < 0 || right < 0) throw InvalidSceneException("CSG geometry refers to a geometry outside the scene");
        } else {
            throw InvalidSceneException("unknown Geometry subclass");
        }
        f.geom_type.push_back(type);
        f.geom_left.push_back(left);
        f.geom_right.push_back(right);
        f.geom_params.insert(f.geom_params.end(), p, p + 4);
    }

    // textures; a bitmap's texels are appended to `texels`
    for (size_t i = 0; i < scene.textures.size(); i++) {
        const Texture* t = scene.textures[i].get();
        f.put(i, flattenTexture(*t));
        if (auto* bm = dynamic_cast<const BitmapTexture*>(t)) {
            f.tex_texel_offset[i] = f.texels.size() / 3;
            for (const Color& c : bm->bmp.data.pixels) {
                f.texels.push_back(c.r);
                f.texels.push_back(c.g);
                f.texels.push_back(c.b);
            }
        }
    }

    for (size_t i = 0; i < scene.shaders.size(); i++) f.put(i, flattenShader(scene, *scene.shaders[i]));
    for (size_t i = 0; i < scene.lights.size(); i++) f.put(i, flattenLight(*scene.lights[i]));

    // environment (cubemap extension: rt.hpp Environment): the six faces follow the bitmap textures' texels
    if (scene.environment.cubemap) {
        f.env_type = C2RT_ENV_CUBEMAP;
        for (int k = 0; k < 6; k++) {
            const Bitmap& b = scene.environment.faces[k];
            f.env_face_width[k] = (int32_t)b.width();
            f.env_face_height[k] = (int32_t)b.height();
            f.env_face_texel_offset[k] = f.texels.size() / 3;
            for (const Color& c : b.data.pixels) {
                f.texels.push_back(c.r);
                f.texels.push_back(c.g);
                f.texels.push_back(c.b);
            }
        }
    }

    for (size_t i = 0; i < scene.nodes.size(); i++) f.put(i, flattenNode(scene, *scene.nodes[i]));
    return f;
}

FlatNode flattenNode(const Scene& scene, const Node& n) {
    FlatNode f;
    f.geom = indexOf(scene.geometries, n.geom);
    f.shader = indexOf(scene.shaders, n.shader);
    if (f.geom < 0 || f.shader < 0) throw InvalidSceneException("node refers to a geometry / shader outside the scene");
    putMatrix(f.transform, n.transform.transform);
    putMatrix(f.inverse, n.transform.inverseTransform);
    putMatrix(f.inverse_t, n.transform.transposedInverse);
    f.offset[0] = n.transform.offset.x;
    f.offset[1] = n.transform.offset.y;
    f.offset[2] = n.transform.offset.z;
    return f;
}

FlatShader flattenShader(const Scene& scene, const Shader& s) {
    FlatShader f;
    f.texture = -1;
    f.exponent = 0;
    f.strength = 0;
    if (auto* la = dynamic_cast<const Lambert*>(&s)) {
        f.type = C2RT_SHADER_LAMBERT;
        if (la->texture) f.texture = indexOf(scene.textures, la->texture);
    } else if (auto* ph = dynamic_cast<const Phong*>(&s)) {
        f.type = C2RT_SHADER_PHONG;
        if (ph->texture) f.texture = indexOf(scene.textures, ph->texture);
        f.exponent = ph->exponent;
        f.strength = ph->strength;
    } else {
        throw InvalidSceneException("unknown Shader subclass");
    }
    f.color[0] = s.color.r; f.color[1] = s.color.g; f.color[2] = s.color.b;
    return f;
}

FlatTexture flattenTexture(const Texture& t) {
    FlatTexture f{};
    if (auto* ch = dynamic_cast<const Checker*>(&t)) {
        f.type = C2RT_TEX_CHECKER;
        f.colors[0] = ch->color1.r; f.colors[1] = ch->color1.g; f.colors[2] = ch->color1.b;
        f.colors[3] = ch->color2.r; f.colors[4] = ch->color2.g; f.colors[5] = ch->color2.b;
        f.params[0] = ch->size;
    } else if (auto* pr = dynamic_cast<const Procedure2*>(&t)) {
        f.type = C2RT_TEX_PROCEDURE2;
        // texture.d:81 reads exactly three entries of each array (a D RangeError otherwise)
        if (pr->colorU.size() < 3 || pr->colorV.size() < 3 || pr->freqU.size() < 3 || pr->freqV.size() < 3)
            throw InvalidSceneException("Procedure2 needs three colorU / colorV / freqU / freqV entries");
        for (int k = 0; k < 3; k++) {
            f.colors[3 * k + 0] = pr->colorU[k].r; f.colors[3 * k + 1] = pr->colorU[k].g; f.colors[3 * k + 2] = pr->colorU[k].b;
            f.colors[9 + 3 * k + 0] = pr->colorV[k].r; f.colors[9 + 3 * k + 1] = pr->colorV[k].g; f.colors[9 + 3 * k + 2] = pr->colorV[k].b;
            f.params[k] = pr->freqU[k];
            f.params[3 + k] = pr->freqV[k];
        }
    } else if (auto* bm = dynamic_cast<const BitmapTexture*>(&t)) {
        f.type = C2RT_TEX_BITMAP;
        f.width = (int)bm->bmp.width();
        f.height = (int)bm->bmp.height();
        f.params[0] = (double)bm->scaling;  // `u *= scaling` widens the float (texture.d:118)
    } else {
        throw InvalidSceneException("unknown Texture subclass");
    }
    return f;
}

FlatLight flattenLight(const Light& l) {
    // PointLight is the only Light subclass the reference has: light.d:52
    auto* pl = dynamic_cast<const PointLight*>(&l);
    if (!pl) throw InvalidSceneException("unknown Light subclass");
    FlatLight f;
    f.pos[0] = pl->pos.x; f.pos[1] = pl->pos.y; f.pos[2] = pl->pos.z;
    f.color[0] = pl->lightColor.r; f.color[1] = pl->lightColor.g; f.color[2] = pl->lightColor.b;
    f.power = pl->lightPower;
    return f;
}

namespace {

std::vector<uint32_t> editIds(const std::vector<int>& indices, size_t count, const char* what) {
    std::vector<uint32_t> ids;
    for (int i : indices) {
        if (i < 0 || (size_t)i >= count) throw RTException(std::string(what) + " index " + std::to_string(i) + " out of range");
        ids.push_back((uint32_t)i);
    }
    return ids;
}

}  // namespace

int setNodes(c2rt_scene* device, const Scene& scene, const std::vector<int>& nodes) {
    const std::vector<uint32_t> ids = editIds(nodes, scene.nodes.size(), "node");
    FlatScene f;
    f.resize(ids.size(), 0, 0, 0);
    for (size_t k = 0; k < ids.size(); k++) f.put(k, flattenNode(scene, *scene.nodes[ids[k]]));
    return c2rt_scene_set_nodes(device, ids.size(), ids.data(), f.node_geom.data(), f.node_transform.data(), f.node_inverse.data(),
                                f.node_inverse_t.data(), f.node_offset.data());
}

int setNodeShaders(c2rt_scene* device, const Scene& scene, const std::vector<int>& nodes) {
    const std::vector<uint32_t> ids = editIds(nodes, scene.nodes.size(), "node");
    FlatScene f;
    f.resize(ids.size(), 0, 0, 0);
    for (size_t k = 0; k < ids.size(); k++) f.put(k, flattenNode(scene, *scene.nodes[ids[k]]));
    return c2rt_scene_set_node_shaders(device, ids.size(), ids.data(), f.node_shader.data());
}

int setShaders(c2rt_scene* device, const Scene& scene, const std::vector<int>& shaders) {
    const std::vector<uint32_t> ids = editIds(shaders, scene.shaders.size(), "shader");
    FlatScene f;
    f.resize(0, ids.size(), 0, 0);
    for (size_t k = 0; k < ids.size(); k++) f.put(k, flattenShader(scene, *scene.shaders[ids[k]]));
    return c2rt_scene_set_shaders(device, ids.size(), ids.data(), f.shader_type.data(), f.shader_color.data(), f.shader_texture.data(),
                                  f.shader_exponent.data(), f.shader_strength.data());
}

int setTextures(c2rt_scene* device, const Scene& scene, const std::vector<int>& textures) {
    const std::vector<uint32_t> ids = editIds(textures, scene.textures.size(), "texture");
    FlatScene f;
    f.resize(0, 0, ids.size(), 0);
    for (size_t k = 0; k < ids.size(); k++) f.put(k, flattenTexture(*scene.textures[ids[k]]));
    return c2rt_scene_set_textures(device, ids.size(), ids.data(), f.tex_colors.data(), f.tex_params.data());
}

int setLights(c2rt_scene* device, const Scene& scene, const std::vector<int>& lights) {
    const std::vector<uint32_t> ids = editIds(lights, scene.lights.size(), "light");
    FlatScene f;
    f.resize(0, 0, 0, ids.size());
    for (size_t k = 0; k < ids.size(); k++) f.put(k, flattenLight(*scene.lights[ids[k]]));
    return c2rt_scene_set_lights(device, ids.size(), ids.data(), f.light_pos.data(), f.light_color.data(), f.light_power.data());
}

c2rt_scene_desc FlatScene::desc() const {
    c2rt_scene_desc d;
    memset(&d, 0, sizeof d);
    d.struct_size = sizeof d;
    d.abi_version = C2RT_ABI_VERSION;
    d.n_nodes = (uint32_t)node_geom.size();
    d.node_geom = node_geom.data();
    d.node_shader = node_shader.data();
    d.node_transform = node_transform.data();
    d.node_inverse = node_inverse.data();
    d.node_inverse_t = node_inverse_t.data();
    d.node_offset = node_offset.data();
    d.n_geoms = (uint32_t)geom_type.size();
    d.geom_type = geom_type.data();
    d.geom_params = geom_params.data();
    d.geom_left = geom_left.data();
    d.geom_right = geom_right.data();
    d.n_shaders = (uint32_t)shader_type.size();
    d.shader_type = shader_type.data();
    d.shader_color = shader_color.data();
    d.shader_texture = shader_texture.data();
    d.shader_exponent = shader_exponent.data();
    d.shader_strength = shader_strength.data();
    d.n_textures = (uint32_t)tex_type.size();
    d.tex_type = tex_type.data();
    d.tex_colors = tex_colors.data();
    d.tex_params = tex_params.data();
    d.tex_width = tex_width.data();
    d.tex_height = tex_height.data();
    d.tex_texel_offset = tex_texel_offset.data();
    d.texels = texels.data();
    d.n_texels = texels.size() / 3;
    d.n_lights = (uint32_t)light_power.size();
    d.light_pos = light_pos.data();
    d.light_color = light_color.data();
    d.light_power = light_power.data();
    d.env_type = env_type;
    for (int k = 0; k < 6; k++) {
        d.env_face_width[k] = env_face_width[k];
        d.env_face_height[k] = env_face_height[k];
        d.env_face_texel_offset[k] = env_face_texel_offset[k];
    }
    return d;
}

c2rt_camera flattenCamera(const Camera& cam) {
    c2rt_camera c;
    memset(&c, 0, sizeof c);
    auto put = [](double dst[3], const Vector& v) { dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; };
    put(c.pos, cam.pos);
    put(c.up_left, cam.upLeft());
    put(c.up_right, cam.upRight());
    put(c.down_left, cam.downLeft());
    put(c.right_dir, cam.rightDir());
    put(c.up_dir, cam.upDir());
    put(c.front_dir, cam.frontDir());
    c.frame_width = (uint32_t)cam.frameWidth;
    c.frame_height = (uint32_t)cam.frameHeight;
    c.dof = cam.dof;
    c.num_samples = (uint32_t)cam.numSamples;
    c.focal_plane_dist = cam.focalPlaneDist;
    c.disc_multiplier = cam.discMultiplier;
    c.stereo_separation = cam.stereoSeparation;
    return c;
}

c2rt_settings flattenSettings(const GlobalSettings& s, uint64_t rngSeed, bool countRays) {
    c2rt_settings o;
    memset(&o, 0, sizeof o);
    o.frame_width = s.frameWidth;
    o.frame_height = s.frameHeight;
    o.aa_enabled = s.AAEnabled;
    o.gi_enabled = s.GIEnabled;
    o.prepass_enabled = s.prepassEnabled;
    o.prepass_only = s.prepassOnly;
    o.max_trace_depth = s.maxTraceDepth;
    o.ambient_light[0] = s.ambientLightColor.r;
    o.ambient_light[1] = s.ambientLightColor.g;
    o.ambient_light[2] = s.ambientLightColor.b;
    o.rng_seed = rngSeed;
    o.count_rays = countRays;
    o.bucket_size = s.bucketSize;
    o.paths_per_pixel = s.pathsPerPixel;
    return o;
}

}  // namespace rt
