/* c2rt.h — C ABI of libc2rt.so, the B200 (sm_100a) implementation of Chess2RT's per-pixel
 * render loop.  Plain C, no exceptions, no torch/C++ types in any signature.
 *
 * This is the drop-in boundary for the reference's renderer seam:
 *   /root/reference/source/rt/renderer.d:23-44   renderSceneAsync(Scene, Image!Color, isRendering*, needsRendering*)
 *   /root/reference/source/rt/renderer.d:46-57   renderPixel(Scene, Image!Color, x, y) -> (Color, TraceResult)
 *   /root/reference/source/rt/renderer.d:72-189  Renderer(scene, output).renderRT()
 * The D host keeps its loaders and object model; a scene flattener lowers `Scene`
 * (/root/reference/source/rt/scene.d:38-51) into the structure-of-arrays description below
 * (field map: SURVEY.md Appendix B; D-side binding: INTEGRATION.md), and the calls below replace
 * the body of renderRT / renderPixel.  The C++ mirror of that host side lives in
 * chess2rt_b200/host/ (this image has no D toolchain).
 *
 * Conventions
 *   - every function returns C2RT_OK (0) or a negative c2rt_status; c2rt_last_error() gives the
 *     message for the calling thread.  Nothing unwinds across this boundary.
 *   - all pointers in a description are borrowed for the duration of the call only; the library
 *     deep-copies what it keeps.  Output buffers are caller-owned and never retained.
 *   - geometry quantities are FP64, colour quantities FP32, as in the reference
 *     (imported_types.d:10-11 `Vector = vec3d`; color.d:27-35 `Color{float r,g,b}`).
 *   - matrices are 3x3 row-major `m[3*row+col]`, used as row-vector x matrix
 *     (imported_types.d:13-20 `mul`).
 *   - there is no CPU fallback: every entry point that renders fails with C2RT_ERR_CUDA when no
 *     sm_100-class device / driver is usable.
 */
#ifndef C2RT_H
#define C2RT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define C2RT_ABI_VERSION 2

typedef enum c2rt_status {
    C2RT_CANCELLED = 1,          /* not an error: c2rt_render ended early because c2rt_cancel was called (the frame is partial) */
    C2RT_OK = 0,
    C2RT_ERR_INVALID_ARG = -1,   /* null pointer, bad index, inconsistent sizes */
    C2RT_ERR_UNSUPPORTED = -2,   /* input the path cannot honour (GI on a Phong-shaded scene, CSG nesting beyond the limit) */
    C2RT_ERR_CUDA = -3,          /* CUDA runtime error or no usable device */
    C2RT_ERR_NOT_INITIALISED = -4,
    C2RT_ERR_LIMIT = -5          /* scene exceeds a compiled-in capacity (C2RT_MAX_*) */
} c2rt_status;

/* Capacities of the on-chip (constant memory) scene block.  A scene within them renders from constant memory; a larger one
 * (the reference's scene.nodes is unbounded: scene.d:38-51, renderer.d:336-338) keeps its node / geometry / shader / texture
 * records in global memory, up to the *_GLOBAL limits below; beyond those c2rt_scene_create returns C2RT_ERR_LIMIT. */
#define C2RT_MAX_NODES_GLOBAL 4096
#define C2RT_MAX_GEOMS_GLOBAL 16384
#define C2RT_MAX_SHADERS_GLOBAL 4096
#define C2RT_MAX_TEXTURES_GLOBAL 1024
#define C2RT_MAX_NODES 64
#define C2RT_MAX_GEOMS 128
#define C2RT_MAX_SHADERS 64
#define C2RT_MAX_TEXTURES 32
#define C2RT_MAX_LIGHTS 8
#define C2RT_MAX_GPUS 8

/* Geometry kinds — geometry.d:15 Plane, :73 Sphere, :149 Cube, :357 CsgUnion, :367 CsgInter, :377 CsgDiff */
enum { C2RT_GEOM_PLANE = 0, C2RT_GEOM_SPHERE = 1, C2RT_GEOM_CUBE = 2, C2RT_GEOM_CSG_UNION = 3, C2RT_GEOM_CSG_INTER = 4, C2RT_GEOM_CSG_DIFF = 5 };
/* Shader kinds — shader.d:54 Lambert, :177 Phong */
enum { C2RT_SHADER_LAMBERT = 0, C2RT_SHADER_PHONG = 1 };
/* Texture kinds — texture.d:20 Checker, :70 Procedure2, :103 BitmapTexture */
enum { C2RT_TEX_CHECKER = 0, C2RT_TEX_PROCEDURE2 = 1, C2RT_TEX_BITMAP = 2 };
/* Environment kinds — environment.d:5-15: the reference has the black stub only.  CUBEMAP is an EXTENSION (no counterpart in the
 * reference, parity unpinned; DESIGN.md "Cubemap environment"): six bitmap faces, looked up by the ray direction of a miss. */
enum { C2RT_ENV_BLACK = 0, C2RT_ENV_CUBEMAP = 1 };

/* Flattened scene: structure of arrays, indices instead of object references.
 * One D object -> one index; objects shared by several nodes keep one entry (lecture5.sdl's
 * sphere "S" is used by three nodes).  CSG children are geometry indices that must be smaller
 * than the CSG's own index (the loader only resolves names defined above, geometry.d:343-347),
 * so the `current.g is left` identity test (geometry.d:314) becomes an index comparison. */
typedef struct c2rt_scene_desc {
    uint32_t struct_size;          /* sizeof(c2rt_scene_desc), for ABI checking */
    uint32_t abi_version;          /* C2RT_ABI_VERSION */

    /* nodes — node.d:7-10 + transform.d:11-14 */
    uint32_t n_nodes;
    const int32_t* node_geom;      /* [n_nodes] geometry index */
    const int32_t* node_shader;    /* [n_nodes] shader index */
    const double* node_transform;  /* [n_nodes*9] Transform.transform */
    const double* node_inverse;    /* [n_nodes*9] Transform.inverseTransform */
    const double* node_inverse_t;  /* [n_nodes*9] Transform.transposedInverse */
    const double* node_offset;     /* [n_nodes*3] Transform.offset */

    /* geometries — geometry.d */
    uint32_t n_geoms;
    const int32_t* geom_type;      /* [n_geoms] C2RT_GEOM_* */
    const double* geom_params;     /* [n_geoms*4] plane: y, limit (NaN = unbounded, geometry.d:19,46), -, -
                                                   sphere: center xyz, R;  cube: center xyz, side;  csg: unused */
    const int32_t* geom_left;      /* [n_geoms] CSG left child index, -1 otherwise */
    const int32_t* geom_right;     /* [n_geoms] CSG right child index, -1 otherwise */

    /* shaders — shader.d:26,57,179-181 */
    uint32_t n_shaders;
    const int32_t* shader_type;    /* [n_shaders] C2RT_SHADER_* */
    const float* shader_color;     /* [n_shaders*3] */
    const int32_t* shader_texture; /* [n_shaders] texture index or -1 */
    const double* shader_exponent; /* [n_shaders] Phong.exponent (already clamped, shader.d:268) */
    const float* shader_strength;  /* [n_shaders] Phong.strength (already clamped, shader.d:271) */

    /* textures — texture.d:22-23,72-73,151-161 */
    uint32_t n_textures;
    const int32_t* tex_type;       /* [n_textures] C2RT_TEX_* */
    const float* tex_colors;       /* [n_textures*18] checker: color1[3], color2[3];
                                                      procedure2: colorU[3][3] then colorV[3][3]; bitmap: unused */
    const double* tex_params;      /* [n_textures*6]  checker: size; procedure2: freqU[3], freqV[3];
                                                      bitmap: scaling (the D field is a float; widen it exactly) */
    const int32_t* tex_width;      /* [n_textures] bitmap width, 0 otherwise */
    const int32_t* tex_height;     /* [n_textures] bitmap height, 0 otherwise */
    const uint64_t* tex_texel_offset; /* [n_textures] offset, in texels, of this bitmap inside `texels` */
    const float* texels;           /* all bitmaps back to back: r,g,b per texel, row-major, row 0 first —
                                      exactly Image!Color.pixels after the load-time gamma pass
                                      (imageio/image.d:18-54, texture.d:137-141) */
    uint64_t n_texels;

    /* lights — light.d:8-9,54 (PointLight only) */
    uint32_t n_lights;
    const double* light_pos;       /* [n_lights*3] */
    const float* light_color;      /* [n_lights*3] lightColor (NOT premultiplied) */
    const float* light_power;      /* [n_lights]   lightPower */

    /* environment — environment.d:5-15 (what `scene.environment.getEnvironment(ray.dir)` returns for a miss, renderer.d:366-368) */
    int32_t env_type;              /* C2RT_ENV_* */
    int32_t env_reserved;
    int32_t env_face_width[6];     /* CUBEMAP: faces in the order +x, -x, +y, -y, +z, -z */
    int32_t env_face_height[6];
    uint64_t env_face_texel_offset[6]; /* offset, in texels, of each face inside `texels` (post-gamma values like the bitmaps) */
} c2rt_scene_desc;

/* Camera state AFTER Camera.beginFrame (camera.d:77-117) and setFrameSize (camera.d:231-236). */
typedef struct c2rt_camera {
    double pos[3];
    double up_left[3], up_right[3], down_left[3];   /* camera.d:51, world space (pos already added) */
    double right_dir[3], up_dir[3], front_dir[3];   /* camera.d:52 */
    uint32_t frame_width, frame_height;             /* camera.d:29-30: the divisors in getScreenRay */
    int32_t dof;                                    /* camera.d:43 */
    uint32_t num_samples;                           /* camera.d:44 */
    double focal_plane_dist;                        /* camera.d:40 */
    double disc_multiplier;                         /* camera.d:42,252 = 10 / fNumber */
    double stereo_separation;                       /* camera.d:45; 0 = off, otherwise every sample traces a left and a right
                                                       eye ray and combines them (combineStereo, color.d:10-15) */
} c2rt_camera;

/* GlobalSettings fields the render path reads (global_settings.d:8-35) + the pinned-RNG seed. */
typedef struct c2rt_settings {
    uint32_t frame_width, frame_height;   /* output size */
    int32_t aa_enabled;                   /* AAEnabled: 5 samples per pixel for ALL pixels (renderer.d:183-186) */
    int32_t gi_enabled;                   /* GIEnabled: path tracing when the camera has no DOF (renderer.d:256-263).  With the only light
                                             type of the reference (PointLight, solidAngle 0: light.d:72-75) every path returns exactly
                                             black, so the frame is black; a Phong-shaded node makes the reference halt (shader.d:252-262)
                                             and is refused with C2RT_ERR_UNSUPPORTED (DESIGN.md section 0, row f-4) */
    int32_t prepass_enabled;              /* accepted and ignored: the prepass is fully overwritten (renderer.d:110-142) */
    int32_t prepass_only;                 /* prepassOnly: with prepass_enabled, the frame is the 16x16-block preview of renderer.d:110-130
                                             (one sample per block, replicated); without it nothing is rendered, like the reference */
    uint32_t max_trace_depth;             /* renderer.d:330 (primary rays have depth 0) */
    float ambient_light[3];               /* ambientLightColor */
    uint64_t rng_seed;                    /* DOF only: seed of the pinned counter-based generator (c2rt_rng_u31) */
    int32_t count_rays;                   /* non-zero: fill c2rt_stats.primary_rays / shadow_rays (slightly slower) */
    uint32_t bucket_size;                 /* bucketSize (global_settings.d:16); only the prepass block grid depends on it; 0 = 48 */
    uint32_t paths_per_pixel;             /* pathsPerPixel (renderer.d:293-300): GI frames only; 0 makes the mean 0/0 = NaN like the reference */
    uint32_t reserved;
} c2rt_settings;

/* Interleaved row bands (multi-GPU): row y belongs to rank ((y / band_rows) % n_ranks).
 * band_rows must be a multiple of 8 (the CUDA block tile height). */
typedef struct c2rt_band {
    uint32_t rank, n_ranks, band_rows;
    uint32_t compact;   /* 0: outputs are full frames (row y at y*W); 1: outputs hold only this rank's rows, in order */
    /* Frame-complete signalling for one process per GPU (bands stored into rank 0's frame through a c2rt_frame_import
     * mapping).  NULL: off.  Otherwise uint32 flags[n_ranks + 1] in RANK 0's frame allocation, zero at start: [0] is the
     * start gate's counter (c2rt_gate), [r] the last frame_no rank r > 0 completed, [n_ranks] counts time-outs.  A peer's
     * c2rt_render_device enqueues a one-thread kernel behind its render kernel that stores frame_no into flags[rank]
     * (st.release.sys; the kernel boundary has performed the band stores at system scope).  The last CTA of RANK 0's render
     * kernel waits for flags[1..n_ranks-1] >= frame_no, so rank 0's kernel ends when the whole frame is in its memory — no
     * wait launch on its critical path.  The wait gives up after ~2 s and bumps flags[n_ranks] instead of hanging the device:
     * read that word back before trusting a frame.  frame_no must grow by one per frame (1, 2, ...); one such launch in
     * flight per device. */
    void* done_flags;
    uint32_t frame_no;
    uint32_t reserved;
} c2rt_band;

typedef struct c2rt_stats {
    double kernel_ms;        /* device time of the render kernel(s), CUDA events (max over devices) */
    double total_ms;         /* host wall time of the call, copies included */
    uint64_t primary_rays;   /* only when settings.count_rays */
    uint64_t shadow_rays;
    uint32_t n_gpus;
    uint32_t launches;       /* kernels launched by the call */
} c2rt_stats;

/* renderer.d:14-21 TraceResult, the part a caller can use */
typedef struct c2rt_hit {
    int32_t node;            /* index of closestNode, -1 = miss */
    int32_t reserved;
    double dist;
    double p[3];
    double normal[3];
    double u, v;
} c2rt_hit;

typedef struct c2rt_scene c2rt_scene;

/* Library lifetime.  device_ids == NULL -> devices 0..n_gpus-1.  With n_gpus > 1 c2rt_render splits
 * the frame into interleaved row bands; every device copies its bands to the caller's host frame over
 * its own PCIe link.  The library then owns n_gpus - 1 helper threads (one per extra device, idle
 * between frames; joined by c2rt_shutdown or the next c2rt_init).  Calling c2rt_init again
 * re-initialises. */
int c2rt_init(int n_gpus, const int* device_ids);
void c2rt_shutdown(void);
int c2rt_abi_version(void);
int c2rt_device_count(void);
const char* c2rt_last_error(void);

/* Scene upload: validates, deep-copies, builds the device scene block + bounding volumes. */
int c2rt_scene_create(const c2rt_scene_desc* desc, c2rt_scene** out);
void c2rt_scene_destroy(c2rt_scene* scene);

/* Node edits in place: moves a piece (its transform), captures it (moves it off the board), promotes it (its geometry index)
 * without re-creating the scene.  Entry i edits node nodes[i]; the arrays have the layout of c2rt_scene_desc's node arrays
 * ([n], [n*9], [n*9], [n*9], [n*3]).  geom == NULL keeps every edited node's geometry; the four transform arrays are given
 * together, or all NULL to keep every edited node's transform; at least one of the two must be given.  Entries apply in array
 * order, so a later entry for the same node wins.  Node shaders, shaders, textures and lights have edits of their own (below);
 * the environment, the node count and the node order stay as created.
 * Afterwards every call on the scene (frames, _device frames, hit frames, the pixel pick, ray queries, visibility, shaded rays)
 * gives the same result, bit for bit, as on a scene c2rt_scene_create built from the edited description, on every device.
 * Errors: a null scene, nodes == NULL with n > 0, a node index >= n_nodes, a geometry index outside 0..n_geoms-1 or a partial
 * set of transform arrays is C2RT_ERR_INVALID_ARG.  Every check runs before anything changes: on any of these errors the scene
 * is unchanged.  n == 0 is a no-op.  A C2RT_ERR_CUDA leaves the scene fit only for c2rt_scene_destroy.
 * Blocking: takes the library lock (so it waits for a c2rt_render running on another thread) and waits for all work on every
 * context device, since kernels in flight read the scene.  The first frame after an edit, like a scene's first frame on a
 * device, must be issued outside any CUDA stream capture, and a graph captured before the edit must not be replayed after it. */
int c2rt_scene_set_nodes(c2rt_scene* scene, size_t n, const uint32_t* nodes, const int32_t* geom,
                         const double* transform, const double* inverse, const double* inverse_t, const double* offset);

/* Shading and light edits in place: point nodes at other shaders (highlight a piece and back), replace shaders (colour, kind,
 * Phong exponent / strength, texture), textures (Checker colours and size, Procedure2 colours and frequencies, a bitmap's
 * scaling) and lights (position, colour, power) without re-creating the scene.  Entry i replaces the whole entry the description
 * gave for index nodes[i] / shaders[i] / textures[i] / lights[i]; every index is a description index (a position in the
 * c2rt_scene_desc arrays the scene was created from), and the arrays have the layout of the matching c2rt_scene_desc arrays for
 * n entries.  A shader's texture index < 0 means none.  A texture keeps its kind, and a bitmap its texels and size: a bitmap
 * entry reads params[0] (scaling) only, a Checker or Procedure2 entry all of colors [18] and params [6].  Values
 * c2rt_scene_create accepts are accepted here (non-finite colours, zero power).  Entries apply in array order, so a later
 * entry for the same index wins.  The environment and the counts and kinds stay as created.
 * Afterwards every call on the scene gives the same result, bit for bit, as on a scene c2rt_scene_create built from the
 * edited description, on every device; a GI frame's refusal of Phong-shaded nodes follows the edited shaders.
 * Errors: a null scene, a null array with n > 0, an index out of range, a node's shader outside 0..n_shaders-1, an unknown
 * shader type or a shader texture >= n_textures is C2RT_ERR_INVALID_ARG.  Every check runs before anything changes: on any of
 * these errors the scene is unchanged.  n == 0 is a no-op.  A C2RT_ERR_CUDA leaves the scene fit only for c2rt_scene_destroy.
 * Blocking, locking and stream capture: as c2rt_scene_set_nodes. */
int c2rt_scene_set_node_shaders(c2rt_scene* scene, size_t n, const uint32_t* nodes, const int32_t* shader);
int c2rt_scene_set_shaders(c2rt_scene* scene, size_t n, const uint32_t* shaders, const int32_t* type, const float* color,
                           const int32_t* texture, const double* exponent, const float* strength);
int c2rt_scene_set_textures(c2rt_scene* scene, size_t n, const uint32_t* textures, const float* colors, const double* params);
int c2rt_scene_set_lights(c2rt_scene* scene, size_t n, const uint32_t* lights, const double* pos, const float* color,
                          const float* power);

/* Replaces Renderer.renderRT (renderer.d:83-189): blocking, one frame into caller-owned HOST
 * memory.  rgb: frame_width*frame_height*3 floats laid out as Image!Color.pixels
 * (row-major, top row first, imageio/image.d:45-54).  argb (nullable): one uint32 per pixel,
 * Color.toRGB32 packing (color.d:154-162: r<<16 | g<<8 | b through the sRGB table). */
int c2rt_render(c2rt_scene* scene, const c2rt_camera* camera, const c2rt_settings* settings,
                float* rgb, uint32_t* argb, c2rt_stats* stats);
/* rgb may be NULL when argb is not: ARGB-only delivery for an interactive host that only blits the packed plane
 * (sdl2_gui.d:139-155) — no float frame is written or copied, a 1080p frame is 8.3 MB over PCIe instead of 33 MB. */

/* Replaces the stop request the reference polls between its passes (renderer.d:93-97,129,147,180): callable from ANY thread
 * while another thread is inside c2rt_render.  Raises a flag on every device; tiles whose CTA has not started yet are skipped,
 * tiles in flight finish, and that c2rt_render returns C2RT_CANCELLED with a partially rendered frame (a frame the GUI is about
 * to replace anyway: raytracer_demo.d:102-124).  A cancel that arrives while no frame is in progress cancels nothing. */
int c2rt_cancel(void);

/* Partial frames after edits: c2rt_render's frame, bit for bit, re-rendering only the CTA tiles (16x8 pixels) an edit since the
 * previous frame can have changed.  A c2rt_frame_cache remembers the frame the last c2rt_render_update with it delivered: the
 * scene records it was rendered from, its camera, settings and output pointers, and per 8x4 pixel patch a bound of the points
 * its camera rays hit.  It owns device buffers on the devices of the c2rt_init it was filled under.  create touches no device;
 * destroy frees the buffers (NULL is a no-op).  One cache serves one stream of frames into one pair of host buffers. */
typedef struct c2rt_frame_cache c2rt_frame_cache;
int c2rt_frame_cache_create(c2rt_frame_cache** out);
void c2rt_frame_cache_destroy(c2rt_frame_cache* cache);

typedef struct c2rt_update_info {
    uint32_t tiles_total;     /* CTA tiles (16x8) of the frame */
    uint32_t tiles_rendered;  /* tiles traced by this call (== tiles_total for a full frame) */
    uint32_t full;            /* 1: the call rendered the whole frame (first frame, or a condition below did not hold) */
    uint32_t reserved;
} c2rt_update_info;

/* Caller contract: on entry rgb / argb (HOST buffers, layout and nullability as c2rt_render) hold what the previous
 * c2rt_render_update with this cache wrote into them; on return they hold exactly what c2rt_render writes for the scene's
 * current state, camera and settings.  The call renders only the tiles that can differ from that previous frame when all of
 * these hold, and the whole frame (refilling the cache) otherwise:
 *   - the cache holds a frame of this scene (the same c2rt_scene_create; the scene's edits since are found by comparing its
 *     records with the cache's copy, so any sequence of c2rt_scene_set_* calls, an edit and its undo included, is handled);
 *   - camera and settings are byte-equal to that frame's, the same output pointers are given (and so the same planes), and the
 *     c2rt_init configuration is the same;
 *   - the scene class is the same and camera-masked: not plane-only (every node an unbounded world plane, a one-plane scene
 *     included), no DOF or stereo camera, not a GI or prepass frame;
 *   - the previous c2rt_render_update with this cache was not cancelled;
 *   - only node records changed (transform, geometry, shader index), and every changed node has a finite bounding sphere
 *     before and after; a shader, texture or light edit renders the whole frame.
 * A tile is re-rendered when a changed node, in its old or its new place, can be reached by one of its camera rays or by a
 * shadow ray from one of its camera hits (DESIGN.md §4.9); its rows are then copied to the host planes.  Every other tile of
 * the host planes is left as it is.
 * Errors, locking and cancellation as c2rt_render; a null cache is C2RT_ERR_INVALID_ARG.  A cancelled call returns
 * C2RT_CANCELLED and empties the cache, so the next call renders the whole frame.  prepass_only without prepass_enabled draws
 * nothing and leaves the cache as it is, as c2rt_render leaves the image.
 * stats as c2rt_render (kernel_ms covers the dirty test and the gather of a partial frame); with count_rays, primary_rays /
 * shadow_rays count the rays this call traced, only in the tiles it rendered.  info (nullable) reports the tiles. */
int c2rt_render_update(c2rt_scene* scene, const c2rt_camera* camera, const c2rt_settings* settings, c2rt_frame_cache* cache,
                       float* rgb, uint32_t* argb, c2rt_stats* stats, c2rt_update_info* info);

/* Same frame, outputs in DEVICE memory of the CURRENT device, launched on `stream`
 * (a cudaStream_t, NULL = default stream) and NOT synchronised.  One process per GPU uses this
 * with its own band; a single-GPU caller passes band == NULL.  d_argb may be NULL.
 * stats (nullable) gets launches only; timing belongs to the caller's events.
 * d_rgb must be 16-byte aligned when frame_width is a multiple of 4 (bands are written with float4 stores).
 * A device holds ONE scene block at a time: rendering a different scene than the previous call on this device first waits
 * for all work on the device and re-uploads the block, so (i) frames of two scenes never overlap on one device and
 * (ii) the first frame of a scene on a device must be issued outside any CUDA stream capture (later ones may be captured).
 * The same holds for the first frame after a c2rt_scene_set_* edit: the edit re-uploads the block, and a frame captured into a
 * graph before the edit is not valid after it. */
int c2rt_render_device(c2rt_scene* scene, const c2rt_camera* camera, const c2rt_settings* settings,
                       const c2rt_band* band, float* d_rgb, uint32_t* d_argb, void* stream, c2rt_stats* stats);

/* Ray counters accumulated by c2rt_render_device calls with settings.count_rays since the last
 * read on the current device (synchronises `stream`), then reset. */
int c2rt_read_ray_counters(c2rt_scene* scene, void* stream, uint64_t* primary, uint64_t* shadow);

/* Rank 0 side of the band gather: `gathered` holds n_ranks compact band buffers back to back
 * (rank-major, each padded to `rows_per_rank_padded` rows); scatter them into the full frame.
 * elem_floats = 3 for RGB float frames, 1 for ARGB words (reinterpreted). Device pointers, async on `stream`. */
int c2rt_deinterleave(const void* gathered, void* frame, uint32_t width, uint32_t height, uint32_t elem_words,
                      uint32_t n_ranks, uint32_t band_rows, uint32_t rows_per_rank_padded, void* stream);

/* Replaces renderPixel (renderer.d:46-57): one un-antialiased sample at the pixel corner. */
int c2rt_render_pixel(c2rt_scene* scene, const c2rt_camera* camera, const c2rt_settings* settings,
                      int x, int y, float rgb[3], c2rt_hit* hit);

/* Hit buffers: for every pixel of the frame, the hit record that the renderPixel replacement above returns for that pixel
 * (the un-antialiased ray at the pixel corner; on DOF / stereo frames sample 0 of the left eye with the pinned generator),
 * floating-point fields rounded to FP32.  Structure of arrays, row-major, top row first; every plane may be NULL.
 * No colour is computed.  aa_enabled, prepass_only and count_rays are ignored; the ray counters and the cancel flag are
 * neither read nor changed.  GI frames are refused with C2RT_ERR_UNSUPPORTED, as the pixel pick refuses them. */
typedef struct c2rt_hit_planes {
    int32_t* node;     /* [W*H] closestNode, -1 = miss */
    float* dist;       /* [W*H] hit distance, +inf for a miss */
    float* normal;     /* [W*H*3] unit geometric normal, 0 for a miss */
    float* uv;         /* [W*H*2] u, v, 0 for a miss */
} c2rt_hit_planes;

/* Blocking, into caller-owned HOST planes.  With n_gpus > 1 the frame is split into the same interleaved row bands as the
 * colour frame, and every device copies its own rows.  stats (nullable): kernel_ms, total_ms, n_gpus, launches. */
int c2rt_render_hits(c2rt_scene* scene, const c2rt_camera* camera, const c2rt_settings* settings,
                     const c2rt_hit_planes* host_planes, c2rt_stats* stats);
/* The same into DEVICE planes of the current device, async on `stream`, with the band and scene-residency rules of the
 * colour frame's device call (band NULL = the whole frame; compact 0 or 1).  band->done_flags must be NULL: hit frames
 * have no frame-complete signalling.  stats (nullable) gets launches only. */
int c2rt_render_hits_device(c2rt_scene* scene, const c2rt_camera* camera, const c2rt_settings* settings,
                            const c2rt_band* band, const c2rt_hit_planes* device_planes, void* stream, c2rt_stats* stats);

/* Ray queries: the reference's two scene queries for rays the caller chooses, n queries per call, one thread each.
 *   c2rt_trace_rays       the closest-hit loop of trace / renderPixel (renderer.d:325-376) on the ray (origin, normalize(dir)):
 *                         the walk starts at dist = 1e99, visits the nodes in scene order, and the last node that reports a hit
 *                         wins.  The direction is normalised on the device in FP64, as camera rays are.
 *   c2rt_test_visibility  Scene.testVisibility(from, to) (scene.d:62-78): the ray from `from` towards normalize(to - from) is
 *                         occluded iff some node, planes included, hits it at a distance <= |to - from|.
 * A query is traced only when its six coordinates are finite and the squared length of its direction (dir, or to - from) is
 * positive and finite in FP64.  Any other query (a zero direction, from == to, a NaN or an infinity) is a miss, or visible = 1.
 * Each result depends on the scene and that one query only: not on the other queries, their order, n or the devices.
 * No camera, settings or GI rule applies; the ray counters and the cancel flag are neither read nor changed; the scene is
 * made resident on the device by the residency rule of the frame calls.
 * n == 0 is a no-op.  A null scene, all outputs null, or a null input with n > 0 is C2RT_ERR_INVALID_ARG; n > 2^31 - 1 is
 * C2RT_ERR_LIMIT.  These checks come before any device is touched.
 * Speed: the 32 consecutive queries of a warp share one node mask, so batches whose runs of 32 queries are close in origin
 * and direction (e.g. 8x4 pixel patches of a camera) skip most nodes; incoherent batches walk every node. */
typedef struct c2rt_ray_hits {   /* every pointer may be NULL; at least one must not be */
    int32_t* node;     /* [n]   closest node, -1 = miss */
    double* dist;      /* [n]   distance along the unit direction, +inf for a miss */
    double* p;         /* [n*3] world-space hit point, 0 for a miss */
    double* normal;    /* [n*3] unit geometric normal as c2rt_hit reports it (CsgDiff flip applied, not face-forwarded), 0 for a miss */
    double* uv;        /* [n*2] u, v, 0 for a miss */
} c2rt_ray_hits;

/* Blocking, HOST arrays ([n*3] doubles each in, host_out planes out).  With n_gpus > 1 the queries are split into n_gpus
 * contiguous chunks of whole CTAs; every device uploads its chunk, runs it and copies its results back over its own link.
 * stats (nullable): kernel_ms, total_ms, n_gpus, launches. */
int c2rt_trace_rays(c2rt_scene* scene, size_t n, const double* origins, const double* dirs, const c2rt_ray_hits* host_out,
                    c2rt_stats* stats);
/* The same on DEVICE arrays of the current device, async on `stream`.  stats (nullable) gets launches only. */
int c2rt_trace_rays_device(c2rt_scene* scene, size_t n, const double* d_origins, const double* d_dirs,
                           const c2rt_ray_hits* device_out, void* stream, c2rt_stats* stats);
/* visible[i] = 1 when nothing occludes the segment from[i] -> to[i], 0 when something does.  Host / device forms as above. */
int c2rt_test_visibility(c2rt_scene* scene, size_t n, const double* from, const double* to, uint8_t* visible, c2rt_stats* stats);
int c2rt_test_visibility_device(c2rt_scene* scene, size_t n, const double* d_from, const double* d_to, uint8_t* d_visible,
                                void* stream, c2rt_stats* stats);

/* Shaded ray queries: the colour Renderer.trace returns (renderer.d:325-376) for the ray (origin, normalize(dir)), depth 0 —
 * the closest hit shaded by its Lambert or Phong shader with one shadow ray per lit light and the ambient term, or
 * env_lookup(dir) for a miss (black, or the C2RT_ENV_CUBEMAP extension).  The shading is the colour frames' own code.
 *   rgb   [n*3] FP32, laid out like Color[n] (nullable)
 *   argb  [n]   Color.toRGB32 through the sRGB table (c2rt_srgb_table), bit-exact as in frames (nullable; not both null)
 *   ambient  GlobalSettings.ambientLightColor, a HOST pointer in both forms: the only setting trace reads at depth 0.  GI does
 *            not apply: this is trace, not pathtrace.
 * A query is traced under the rule of c2rt_trace_rays; an untraced query gives rgb (0, 0, 0) and argb 0.  Each result depends
 * on the scene, ambient and that one query only: not on the other queries, their order, n or the devices.  No camera, AA,
 * DOF or stereo applies (the caller supplies the rays); the ray counters and the cancel flag are neither read nor changed; the
 * scene is made resident by the residency rule of the frame calls.
 * n == 0 is a no-op that zeroes stats.  A null scene, a null ambient, both outputs null, or a null input with n > 0 is
 * C2RT_ERR_INVALID_ARG; n > 2^31 - 1 is C2RT_ERR_LIMIT.  These checks come before any device is touched.
 * Speed: as for c2rt_trace_rays, runs of 32 queries close in origin and direction (a camera's 8x4 pixel patches, rows of a
 * panorama) skip most nodes for the camera ray; shadow rays get their own per-warp node mask. */
/* Blocking, HOST arrays; with n_gpus > 1 the queries are split into contiguous chunks of whole CTAs, as c2rt_trace_rays does.
 * stats (nullable): kernel_ms, total_ms, n_gpus, launches. */
int c2rt_shade_rays(c2rt_scene* scene, const float ambient[3], size_t n, const double* origins, const double* dirs, float* rgb,
                    uint32_t* argb, c2rt_stats* stats);
/* The same on DEVICE arrays of the current device, async on `stream`.  stats (nullable) gets launches only. */
int c2rt_shade_rays_device(c2rt_scene* scene, const float ambient[3], size_t n, const double* d_origins, const double* d_dirs,
                           float* d_rgb, uint32_t* d_argb, void* stream, c2rt_stats* stats);

/* Number of rows rank `rank` owns in a frame of `height` rows. */
uint32_t c2rt_band_rows_owned(uint32_t height, uint32_t rank, uint32_t n_ranks, uint32_t band_rows);

/* The pinned generator that stands in for util/random.d's libc rand() (SURVEY.md F4): 31 bits keyed
 * by (seed, pixel, AA tap, DOF sample, draw index); uniform(0,1) = value / 2147483647.0 . */
uint32_t c2rt_rng_u31(uint64_t seed, uint32_t px, uint32_t py, uint32_t tap, uint32_t sample, uint32_t draw);

/* The 4097-entry sRGB compression table (color.d:209-229) used for ARGB output. */
void c2rt_srgb_table(uint8_t out[4097]);

/* Peer-visible device buffers for the one-process-per-GPU path: rank 0 allocates the frame and
 * exports a 64-byte handle; the other ranks import it and pass the mapped pointer as d_rgb so their
 * kernels store bands directly into rank 0's memory over NVLink. */
int c2rt_frame_alloc(size_t bytes, void** d_ptr);   /* zero-filled */
int c2rt_frame_free(void* d_ptr);
int c2rt_frame_export(void* d_ptr, uint8_t handle[64]);
int c2rt_frame_import(const uint8_t handle[64], void** d_ptr);
int c2rt_frame_unimport(void* d_ptr);
/* asynchronous byte fill of (part of) such a frame on `stream` (e.g. 0xFF = NaN pixels before a checked frame, so that a band
 * that never arrived cannot pass for one left over from the previous frame) */
int c2rt_frame_memset(void* d_ptr, int byte_value, size_t bytes, void* stream);
/* asynchronous device->host copy of (part of) such a frame on `stream` (host memory should be pinned) */
int c2rt_frame_download(void* host_dst, const void* d_src, size_t bytes, void* stream);

/* Device-side start gate for the one-process-per-GPU path: every rank enqueues c2rt_gate(flags, n_ranks, round, stream) in
 * front of a frame, with round = 1, 2, 3, ... counted per flags allocation; the one-thread kernel adds 1 to flags[0] (rank 0's
 * memory, over NVLink for the peers) and waits until it reaches round * n_ranks, i.e. until every rank arrived.  The ranks'
 * render kernels then start together without a host round trip, and no peer can store bands of frame k + 1 while rank 0's
 * stream still works on (renders, copies out, clears) frame k.  Same ~2 s time-out rule and error word (flags[n_ranks]) as
 * c2rt_band.done_flags. */
int c2rt_gate(void* d_flags, uint32_t n_ranks, uint32_t round, void* stream);

/* Page-locks a caller-owned host buffer (e.g. the D host's Image!Color.pixels, which is ordinary GC memory) so
 * that c2rt_render's device->host copies run asynchronously at full PCIe rate and overlap with rendering.
 * Optional: without it the copies still work, through the driver's staging path.  Unpin before freeing. */
int c2rt_pin_host_buffer(void* ptr, size_t bytes);
int c2rt_unpin_host_buffer(void* ptr);

/* Micro-benchmarks used by bench.py to measure the roofline denominators on the box:
 * dependent-free FFMA / DFMA throughput in TFLOP/s on the current device. */
int c2rt_measure_fma_peak(int fp64, double* tflops, double* sm_clock_mhz_est);

/* Test hook (no GPU needed): drives the helper-thread pool c2rt_render uses after c2rt_init(N > 1) through
 * `rounds` frames of dummy work on `workers` threads, with the spin and the sleep hand-off paths both
 * exercised, restarting the pool in between.  Returns the number of work items executed
 * (== workers * rounds when nothing was lost or duplicated), negative on bad arguments. */
long long c2rt_selftest_device_pool(int workers, int rounds);

/* Test hook (no GPU needed): validates `desc` as c2rt_scene_create does and returns the kernel specialisation the scene
 * would get (>= 0: the MODE_* bits of chess2rt_b200/csrc/scene_dev.h), or a negative C2RT_ERR_* code.  Nothing is uploaded. */
int c2rt_selftest_scene_class(const c2rt_scene_desc* desc);

#ifdef __cplusplus
}
#endif
#endif /* C2RT_H */
