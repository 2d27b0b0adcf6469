// Scene flattener: lowers the host object graph (rt::Scene and the CSG trees hanging off its
// geometries) into the structure-of-arrays description of include/c2rt.h.  This is subsystem (1)
// of the north star; field map in SURVEY.md Appendix B.  Object references become indices;
// objects shared by several nodes keep a single entry; CSG children keep their identity as an index
// (the reference's `current.g is left` test, /root/reference/source/rt/geometry.d:314).
// Runs once per scene (load time); the camera / settings blocks are refreshed per frame.
#pragma once
#include <map>
#include <vector>

#include "../../include/c2rt.h"
#include "rt.hpp"

namespace rt {

// One node's entries of the node arrays (c2rt_scene_desc, c2rt_scene_set_nodes): geometry and shader index, the three
// matrices row-major, the offset
struct FlatNode {
    int32_t geom, shader;
    double transform[9], inverse[9], inverse_t[9], offset[3];
};

// One shader's entries of the shader arrays (c2rt_scene_desc, c2rt_scene_set_shaders)
struct FlatShader {
    int32_t type, texture;
    float color[3];
    double exponent;
    float strength;
};

// One texture's entries of the texture arrays (c2rt_scene_desc, c2rt_scene_set_textures); a bitmap's texels are not among them
struct FlatTexture {
    int32_t type, width, height;
    float colors[18];
    double params[6];
};

// One light's entries of the light arrays (c2rt_scene_desc, c2rt_scene_set_lights)
struct FlatLight {
    double pos[3];
    float color[3];
    float power;
};

struct FlatScene {
    std::vector<int32_t> node_geom, node_shader;
    std::vector<double> node_transform, node_inverse, node_inverse_t, node_offset;
    std::vector<int32_t> geom_type, geom_left, geom_right;
    std::vector<double> geom_params;
    std::vector<int32_t> shader_type, shader_texture;
    std::vector<float> shader_color, shader_strength;
    std::vector<double> shader_exponent;
    std::vector<int32_t> tex_type, tex_width, tex_height;
    std::vector<float> tex_colors;
    std::vector<double> tex_params;
    std::vector<uint64_t> tex_texel_offset;
    std::vector<float> texels;
    std::vector<double> light_pos;
    std::vector<float> light_color, light_power;
    int32_t env_type = C2RT_ENV_BLACK;
    int32_t env_face_width[6] = {0}, env_face_height[6] = {0};
    uint64_t env_face_texel_offset[6] = {0};

    // Sizes the node, shader, texture and light arrays for that many entries of each (new entries are zero)
    void resize(size_t nodes, size_t shaders, size_t textures, size_t lights);
    // Entry i of one kind's arrays; the texture writer leaves tex_texel_offset alone
    void put(size_t i, const FlatNode& node);
    void put(size_t i, const FlatShader& shader);
    void put(size_t i, const FlatTexture& texture);
    void put(size_t i, const FlatLight& light);
    c2rt_scene_desc desc() const;  // borrows the vectors above
};

FlatScene flatten(const Scene& scene);                        // throws InvalidSceneException on dangling references
FlatNode flattenNode(const Scene& scene, const Node& node);   // the same for one node
FlatShader flattenShader(const Scene& scene, const Shader& shader);
FlatTexture flattenTexture(const Texture& texture);
FlatLight flattenLight(const Light& light);

// c2rt_scene_set_nodes / _set_node_shaders / _set_shaders / _set_textures / _set_lights of the listed entities of `scene`
// (indices into its vectors), re-flattened through the routines above, on the uploaded scene `device`: the c2rt status.
// setNodes sets each node's geometry and transform.  Throws RTException on an index out of range, before any call.
int setNodes(c2rt_scene* device, const Scene& scene, const std::vector<int>& nodes);
int setNodeShaders(c2rt_scene* device, const Scene& scene, const std::vector<int>& nodes);
int setShaders(c2rt_scene* device, const Scene& scene, const std::vector<int>& shaders);
int setTextures(c2rt_scene* device, const Scene& scene, const std::vector<int>& textures);
int setLights(c2rt_scene* device, const Scene& scene, const std::vector<int>& lights);
c2rt_camera flattenCamera(const Camera& cam);                 // call after Camera.beginFrame
c2rt_settings flattenSettings(const GlobalSettings& s, uint64_t rngSeed = 0, bool countRays = false);

}  // namespace rt
