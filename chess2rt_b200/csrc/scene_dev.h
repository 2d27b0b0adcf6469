// Device-side scene block and per-frame parameter block (plain PODs shared by host and device code).
//
// The whole flattened scene lives in constant memory: the reference tests every ray against every
// node linearly (/root/reference/source/rt/renderer.d:336-338, scene.d:73-75), the node loop is
// warp-uniform, so every record read is a constant-cache broadcast.  Bitmap texels are the only
// scene data in global memory (float4 per texel, one 16-byte load each).
#pragma once
#include <stdint.h>

#include "../../include/c2rt.h"

namespace c2rt {

enum : int {
    NODE_IDENTITY = 1,     // transform == identity (offset may be non-zero): skip the six mat-vecs of node.d:27-47
    NODE_UNBOUNDED = 2,    // no finite bounding sphere (planes)
};

// Per-node fast paths chosen at scene-create time: identity-transform primitive nodes are tested
// directly in world space against pre-offset parameters (`wp`).
enum : int { KIND_PLANE_W = 0, KIND_SPHERE_W = 1, KIND_CUBE_W = 2, KIND_GENERIC = 3 };

struct DevNode {
    double Minv[9];   // Transform.inverseTransform
    double M[9];      // Transform.transform
    double MinvT[9];  // Transform.transposedInverse
    double off[3];    // Transform.offset
    double wp[4];     // KIND_*_W: plane y + off.y | sphere/cube centre + off, R / side
    float bcf[3];     // world-space bounding sphere centre (FP32 copy for the conservative cull)
    float brf;        // radius, inflated
    float br2f;       // radius squared
    float bclen;      // |centre|, for the cull's rounding-error margin
    int geom, shader, flags, kind;
    int pad0, pad1;
};

struct DevGeom {
    double p[4];      // plane: y, limit | sphere: c.xyz, R | cube: c.xyz, side
    int type, left, right;
    int depth;        // CSG depth: 0 primitive, 1 CSG of primitives, >1 nested (or forced literal: -1)
};

struct DevShader {
    double exponent;
    float color[3];
    float strength;
    int type, tex;
};

struct DevTex {
    double d[6];      // checker: size, 1/size | procedure2: freqU[3], freqV[3] in 2^-32 revolutions per unit (freq / 2pi * 2^32) | bitmap: scaling
    float c[18];      // checker: color1, color2 | procedure2: colorU[3][3], colorV[3][3]
    // bitmap: width, height | procedure2: w / h = high word of the |u| / |v| below which every phase stays under 2^19 revolutions
    // (render_kernel.cu sin_phase)
    int type, w, h, pad;
    const float4* texels;    // bitmap, general form: one float4 per texel (post-gamma values, exactly the host's Image!Color)
    // bitmap with <= 256 distinct texel colours (every 8-bit-palette BMP; the load-time gamma maps equal inputs to equal
    // outputs): `quads` holds, per texel, the palette indices of the four texels a bilinear lookup at that texel reads —
    // (x, y), (x+1, y), (x, y+1), (x+1, y+1) with the wrap of bitmap.d:55-56, one byte each, low byte first — so a lookup is ONE
    // 4-byte load plus four reads of the 4 KB palette instead of four 16-byte gathers.  Bit-identical to the general form.
    const uint32_t* quads;
    const float4* palette;
};

struct DevLight {
    double pos[3];
    float color[3];   // lightColor * lightPower, the FP32 product of light.d:11-14
    int lit;          // color.intensity() != 0 (shader.d:88,219)
    float posf[3];    // FP32 copy of pos (plane-only scene classes take the horizontal light vector in FP32)
    float near2;      // (0.24 |pos|)^2: closer than this to the light, that FP32 difference cancels and FP64 is used (render_kernel.cu shade)
};

struct DevScene {
    int n_nodes, n_geoms, n_shaders, n_textures, n_lights, env_type, n_lit, pad2;
    int lit[C2RT_MAX_LIGHTS];   // indices of the lights with intensity != 0, in scene order (the others shoot no shadow ray: shader.d:88,219)
    // MODE_BIG (a scene beyond C2RT_MAX_NODES / GEOMS / SHADERS / TEXTURES): the record arrays live in global memory instead
    const DevNode* g_nodes;
    const DevGeom* g_geoms;
    const DevShader* g_shaders;
    const DevTex* g_textures;
    DevTex env_faces[6];   // C2RT_ENV_CUBEMAP: +x, -x, +y, -y, +z, -z as bitmap records (render_kernel.cu env_lookup)
    DevNode nodes[C2RT_MAX_NODES];
    DevGeom geoms[C2RT_MAX_GEOMS];
    DevShader shaders[C2RT_MAX_SHADERS];
    DevTex textures[C2RT_MAX_TEXTURES];
    DevLight lights[C2RT_MAX_LIGHTS];
};

struct FrameParams {
    // camera.d:123-147 with the frame invariants hoisted: ul_rel = upLeft - pos, du = upRight - upLeft,
    // dv = downLeft - upLeft, inv_w / inv_h = 1 / camera.frameWidth, 1 / camera.frameHeight
    double pos[3], ul_rel[3], du[3], dv[3];
    float posf[3], posf_len;          // FP32 copy of pos and its length (the cull's ray shadow, render_kernel.cu set_shadow)
    double right_dir[3], up_dir[3], front_dir[3];
    double inv_w, inv_h;
    double tap_d[5][3];               // ray-direction offset of AA tap k: du * kx/W + dv * ky/H (renderer.d:235-247)
    double focal_plane_dist, disc_multiplier;
    double stereo_sep;                // camera.stereoSeparation (0 = off)
    unsigned long long seed;
    uint32_t W, H;                    // output size
    int aa, dof;
    uint32_t num_samples;
    // frame number of the done_flags signalling (below).  It sits here so that every 4-byte field keeps its offset mod 8:
    // ptxas reads adjacent 8-byte-aligned pairs of them with one 64-bit constant load (LDC.64 / LDCU.64)
    uint32_t frame_no;
    float ambient[3];
    int count_rays;
    uint32_t prepass_bucket;          // > 0: prepassOnly frame (16x16-block preview inside buckets of this size)
    int gi;                           // GI frame: every pixel is gi_fill (see c2rt_api.cu fill_params)
    float gi_fill;
    // interleaved row bands
    uint32_t rank, n_ranks, tiles_per_band, compact;
    uint32_t tile_row0;               // first local tile row of this launch (one launch per band, c2rt_api.cu render_bands)
    // per-node bounding spheres (x, y, z, radius; radius < 0: unbounded) in GLOBAL memory for the per-warp node masks, whose
    // lanes each test a different node (render_kernel.cu camera_mask / shadow_mask)
    const float4* bounds;
    // frame-complete signalling folded into the kernel (render_frame_kernel epilogue); done_flags == nullptr: off
    uint32_t* done_flags;             // in rank 0's memory: [r] = last frame number rank r completed, [n_ranks] = wait time-outs
    uint32_t* done_counter;           // this device: CTAs of the current launch that have finished
    // MODE_SOLO frames (render_kernel.cu solo_plane_test): solo_fast = the frame is regular (camera — the whole lens under
    // DOF / stereo — off the plane, light on the camera's side, moderate magnitudes: c2rt_api.cu fill_params); the kernels
    // without the sampling loop only run such frames, the sampling kernels branch on it.  Then: side of the plane the camera is
    // on (+1 above, -1 below), the sign bit a ray's d.y must NOT have xor'ed in (0x80000000 above the plane: d.y must be
    // negative), the camera position's height above the plane (pos.y - y), and 1e-18 max|d|^2 over the frame's camera rays.
    // solo_rows: a regular frame with du.y == 0 (no camera roll): a camera ray's d.y depends on its row and AA tap only, and
    // render_solo_kernel takes the plane hit and light height from a per-row table (render_kernel.cu row_tap)
    int solo_fast, solo_side;
    uint32_t solo_sign, solo_rows;
    double solo_h, graze_dy2;
    const int* cancel;                // device flag raised by c2rt_cancel: CTAs that start after it skip their tile (nullptr: off)
    // outputs (rgb == nullptr: only the ARGB plane is wanted)
    float* rgb;
    uint32_t* argb;
    unsigned long long* counters;     // [0] primary, [1] shadow
    const uint8_t* lut;               // 4097-entry sRGB table
    // solo_zrows: a solo_rows frame with du.z == 0 as well (no yaw): a camera ray's d.z, its hit point's z and what depends on
    // it alone are constants of the (row, AA tap) too (render_kernel.cu RowZ).  Last, so that every other field keeps its offset.
    uint32_t solo_zrows;
};

// Kernel specialisations by scene class (chosen at scene-create time, c2rt_api.cu):
//   MODE_BOUNDED  some node has a finite bounding sphere -> FP32 ray shadow + conservative cull
//   MODE_GENERIC  some node needs the object-space path (non-identity transform, CSG, bounded plane)
//   MODE_NESTED   some CSG has a CSG child -> literal emulation of the reference's recursive walk
//                 (bit 8 was MODE_CLUSTERS, the two-level cull of round 1: replaced by the per-warp node masks, render_kernel.cu)
//   MODE_SAMPLING the CAMERA asks for depth of field and/or stereo: several rays per sample (chosen per frame)
//   MODE_SOLO     one world-space plane node and one light (lecture4*, zaphod): node / shader / texture / light records
//                 sit at index 0 (c2rt_api.cu moves them there), so every scene constant is read through a static
//                 c[3][imm] operand instead of an indexed LDC, no loop survives, and the texture kind
//                 (MODE_TEX_SHIFT: 0 none, 1 + C2RT_TEX_*) and shader kind (MODE_PHONG) are compile-time
constexpr int MODE_BOUNDED = 1, MODE_GENERIC = 2, MODE_NESTED = 4, MODE_SAMPLING = 16;
constexpr int MODE_SOLO = 32, MODE_TEX_SHIFT = 6, MODE_TEX_MASK = 3 << MODE_TEX_SHIFT, MODE_PHONG = 256;
//   MODE_BIG      the scene exceeds the constant block: node / geometry / shader / texture records in global memory
//                 (DevScene::g_*), node masks of one 64-bit word per 64 nodes in shared memory (render_kernel.cu NodeMask)
constexpr int MODE_BIG = 512;
// every node is a world-space plane (KIND_PLANE_W): no bounded and no generic node exists
#ifdef __CUDACC__
__host__ __device__
#endif
constexpr bool plane_only(int mode) { return (mode & (MODE_BOUNDED | MODE_GENERIC | MODE_NESTED)) == 0; }

// Scene classes whose rays go through per-warp node masks (render_kernel.cu camera_mask / shadow_mask): every scene class
// but the plane-only ones.  Camera rays get a mask only when they all start at the camera position (no DOF / stereo
// sampling loop); shadow rays always do.
#ifdef __CUDACC__
__host__ __device__
#endif
constexpr bool camera_masked(int mode) { return !plane_only(mode) && !(mode & MODE_SAMPLING); }

// CTA tile: 4 warps of 8x4 pixels each, 2x2 warps (32x4 was measured and not kept: profiles/r2_tile_shape.log)
constexpr int TILE_W = 16;
constexpr int TILE_H = 8;
static_assert(TILE_W % 8 == 0 && TILE_H % 4 == 0 && TILE_W * TILE_H == 128, "a CTA tile is four 8x4 warp patches");
constexpr int BLOCK_THREADS = TILE_W * TILE_H;

// The pinned RNG of DOF sampling (c2rt.h c2rt_rng_u31): the kernel's lens samples and the exported function are this one
// definition; the oracle keeps an independent copy (oracle/orc_scene.hpp rng_u31) that the tests compare it with.
// Counter-based: four rounds of the 32-bit "lowbias32" finaliser over (seed, pixel) / (tap, sample) / draw.
// The pixel and sample rounds do not depend on `draw`, so a compiler hoists them out of the draw sequence.
#ifdef __CUDACC__
__host__ __device__ __forceinline__
#endif
constexpr uint32_t rng_u31(uint64_t seed, uint32_t px, uint32_t py, uint32_t tap, uint32_t sample, uint32_t draw) {
    uint32_t h = (uint32_t)seed ^ ((uint32_t)(seed >> 32) * 0x9E3779B9u) ^ (px * 0x85EBCA6Bu);
    h ^= h >> 16; h *= 0x7FEB352Du; h ^= h >> 15; h *= 0x846CA68Bu; h ^= h >> 16;
    h ^= py * 0xC2B2AE35u;
    h ^= h >> 16; h *= 0x7FEB352Du; h ^= h >> 15; h *= 0x846CA68Bu; h ^= h >> 16;
    h ^= tap * 0x27D4EB2Fu + sample * 0x165667B1u;
    h ^= h >> 16; h *= 0x7FEB352Du; h ^= h >> 15; h *= 0x846CA68Bu; h ^= h >> 16;
    h += draw * 0x9E3779B9u;
    h ^= h >> 16; h *= 0x7FEB352Du; h ^= h >> 15; h *= 0x846CA68Bu; h ^= h >> 16;
    return h >> 1;
}

// renderer.d:46-57 renderPixel: what render_pixel_kernel writes for c2rt_render_pixel
struct PixelOut {
    float rgb[3];
    int node;
    double dist, p[3], n[3], u, v;
};

}  // namespace c2rt
