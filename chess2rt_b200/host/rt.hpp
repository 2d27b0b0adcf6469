// Host-side mirror of the reference's scene API for the render path, in C++ because this image has
// no D toolchain (SURVEY.md F2).  Same names, fields, defaults and error behaviour as the D classes:
//   Scene            /root/reference/source/rt/scene.d:38-58
//   GlobalSettings   rt/global_settings.d:8-35
//   Camera           rt/camera.d:12-117,181-255
//   Transform, Node  rt/transform.d:9-55, rt/node.d:7-21,70-94
//   Plane/Sphere/Cube/Csg*  rt/geometry.d:15-23,73-90,149-163,250-267,357-403
//   Checker/Procedure2/BitmapTexture  rt/texture.d:20-34,70-75,103-161; Bitmap rt/bitmap.d:11-136
//   Lambert/Phong    rt/shader.d:24-65,177-195,263-280
//   PointLight       rt/light.d:6-14,52-82
//   Image<C>         imageio/image.d:18-60
//   exceptions       rt/exception.d:5-69, imageio/exception.d:3-31
// The per-ray methods of these classes (intersect / shade / getTexColor / getScreenRay) are NOT
// here: that work runs in libc2rt.so's CUDA kernels.  What is here is what the D host keeps —
// the object model and loaders — plus the new pieces the north star asks for: the scene flattener
// (flatten.hpp) and the renderer entry points re-pointed at the C ABI (renderer.hpp).
#pragma once
#include <cmath>
#include <cstdint>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

namespace rt {

// ------------------------------------------------------------------ exceptions (rt/exception.d)
struct RTException : std::runtime_error {
    using std::runtime_error::runtime_error;
};
struct SceneNotFoundException : RTException {
    SceneNotFoundException() : RTException("Scene file not found!") {}
};
struct InvalidSceneException : RTException {
    using RTException::RTException;
};
struct EntityWithDuplicateName : RTException {
    explicit EntityWithDuplicateName(const std::string& n) : RTException("Entity with duplicate name: " + n) {}
};
struct PropertyNotFoundException : RTException {
    explicit PropertyNotFoundException(const std::string& n) : RTException("Property not found: " + n) {}
};
struct ImageIOException : std::runtime_error {
    using std::runtime_error::runtime_error;
};
struct ErrorLoadingImageException : ImageIOException {
    using ImageIOException::ImageIOException;
};
struct UnknownImageTypeException : ImageIOException {
    UnknownImageTypeException() : ImageIOException("Unknown image type") {}
};
// raised when libc2rt.so reports an error (negative c2rt_status); never swallowed, never a CPU fallback
struct BackendException : RTException {
    int status;
    BackendException(int st, const std::string& m) : RTException("libc2rt: " + m), status(st) {}
};

// ------------------------------------------------------------------ basic types
struct Color {  // rt/color.d:27-35: components default to 0
    float r = 0.f, g = 0.f, b = 0.f;
    Color() = default;
    Color(float r_, float g_, float b_) : r(r_), g(g_), b(b_) {}
    explicit Color(uint32_t rgb) {  // color.d:60-66
        const float divider = 1.0f / 255.0f;
        r = float((rgb >> 16) & 0xff) * divider;
        g = float((rgb >> 8) & 0xff) * divider;
        b = float(rgb & 0xff) * divider;
    }
};

struct Vector {  // gfm vec3d: default-initialised to NaN like every D double
    double x = NAN, y = NAN, z = NAN;
    Vector() = default;
    Vector(double x_, double y_, double z_) : x(x_), y(y_), z(z_) {}
};

struct Matrix {  // gfm mat3d, row-major c[row][col]
    double c[3][3];
    static Matrix identity();
    static Matrix scaledIdentity(double x, double y, double z);  // imported_types.d:22-29
    static Matrix rotateX(double a);
    static Matrix rotateY(double a);
    static Matrix rotateZ(double a);
    Matrix operator*(const Matrix& o) const;
    Matrix inverse() const;
    Matrix transposed() const;
};
Vector mul(const Vector& v, const Matrix& m);  // imported_types.d:13-20
double radians(double deg);

template <class C>
struct Image {  // imageio/image.d:18-60
    size_t width = 0, height = 0;
    std::vector<C> pixels;
    Image() = default;
    Image(size_t w, size_t h) { alloc(w, h); }
    void alloc(size_t w, size_t h) {
        width = w;
        height = h;
        if (pixels.size() < w * h) pixels.resize(w * h);
    }
    C& operator()(size_t x, size_t y) { return pixels[width * y + x]; }
    const C& operator()(size_t x, size_t y) const { return pixels[width * y + x]; }
    bool empty() const { return pixels.empty(); }
};

// ------------------------------------------------------------------ settings / camera
struct GlobalSettings {
    uint32_t frameWidth = 640, frameHeight = 480;
    bool fullscreen = false, allowResize = false, dynamicAspectRatio = false, interactive = false;
    uint32_t bucketSize = 48, threadCount = 0;
    bool prepassEnabled = true, prepassOnly = false, GIEnabled = false, AAEnabled = true;
    double AAThreshold = 0.1;
    uint32_t pathsPerPixel = 40, maxTraceDepth = 4;
    Color ambientLightColor;
    bool debugEnabled = true;
};

class Camera {
public:
    size_t frameWidth = 0, frameHeight = 0;
    double aspect = 1.0;
    Vector pos;
    double yaw = 0, pitch = 0, roll = 0;
    double fov = 0;
    double focalPlaneDist = 1.0, fNumber = 1.0, discMultiplier = NAN;
    bool dof = false;
    size_t numSamples = 25;
    double stereoSeparation = 0.0;

    void beginFrame();                             // camera.d:77-117
    void setFrameSize(uint32_t w, uint32_t h);     // camera.d:231-236
    void move(double dx, double dy, double dz);    // camera.d:181-204
    void rotate(double dYaw, double dRoll, double dPitch);  // camera.d:211-229

    // accessors for the flattener (module-private in D: camera.d:47-53)
    const Vector& upLeft() const { return upLeft_; }
    const Vector& upRight() const { return upRight_; }
    const Vector& downLeft() const { return downLeft_; }
    const Vector& frontDir() const { return frontDir_; }
    const Vector& rightDir() const { return rightDir_; }
    const Vector& upDir() const { return upDir_; }

private:
    Vector upLeft_, upRight_, downLeft_, frontDir_, rightDir_, upDir_;
};


// ------------------------------------------------------------------ geometry
struct Geometry {
    virtual ~Geometry() = default;
};
struct Plane : Geometry {
    double y = NAN, limit = NAN;  // geometry.d:18-19 (limit is not loadable -> NaN -> unbounded)
};
struct Sphere : Geometry {
    Vector center{0, 0, 0};
    double R = 1;
};
struct Cube : Geometry {
    Vector center{0, 0, 0};
    double side = 1;
};
struct CsgOp : Geometry {
    const Geometry* left = nullptr;
    const Geometry* right = nullptr;
};
struct CsgUnion : CsgOp {};
struct CsgInter : CsgOp {};
struct CsgDiff : CsgOp {};

// ------------------------------------------------------------------ textures
struct Texture {
    virtual ~Texture() = default;
};
struct Checker : Texture {
    Color color1{0, 0, 0}, color2{1, 1, 1};
    double size = 1.0;
};
struct Procedure2 : Texture {
    std::vector<Color> colorU, colorV;
    std::vector<double> freqU, freqV;
};
struct Bitmap {  // rt/bitmap.d:11-136 (load + gamma only; filtering runs on the GPU)
    Image<Color> data;
    size_t width() const { return data.width; }
    size_t height() const { return data.height; }
    void loadImage(const std::string& filename);
    void decompressGamma_sRGB();
    void decompressGamma(float gamma);
};
struct BitmapTexture : Texture {
    Bitmap bmp;
    float scaling = 1;
    float assumedGamma = 2.2f;
};

// rt/environment.d:5-15 is a stub that always returns black and reads no keys.  EXTENSION (no counterpart in the reference,
// DESIGN.md "Cubemap environment"): an optional `folder` key names a directory holding posx/negx/posy/negy/posz/negz .bmp;
// `assumedGamma` is applied at load time exactly like BitmapTexture's (texture.d:137-141).  The lookup runs on the GPU.
struct Environment {
    Bitmap faces[6];   // +x, -x, +y, -y, +z, -z
    bool cubemap = false;
    float assumedGamma = 2.2f;
};

// ------------------------------------------------------------------ shaders / lights / nodes
struct Shader {
    Color color;
    virtual ~Shader() = default;
};
struct Lambert : Shader {
    const Texture* texture = nullptr;
    Lambert() { color = Color(1, 1, 1); }
};
struct Phong : Shader {
    const Texture* texture = nullptr;
    double exponent = 16.0;
    float strength = 1.0f;
    Phong() { color = Color(1, 1, 1); }
    // the ranges shader.d:263-280 clamps a loaded exponent and strength to
    static double clampExponent(double e) { return e < 1e-6 ? 1e-6 : (e > 1e6 ? 1e6 : e); }
    static float clampStrength(float s) { return s < 0.f ? 0.f : (s > 1e6f ? 1e6f : s); }
};

struct Light {
    Color lightColor;
    float lightPower = NAN;
    virtual ~Light() = default;
};
struct PointLight : Light {
    Vector pos;
};

struct Transform {  // rt/transform.d:9-55
    Matrix transform, inverseTransform, transposedInverse;
    Vector offset;
    Transform() { reset(); }
    void reset();
    void scale(double x, double y, double z);
    void rotate(double yaw, double pitch, double roll);
    void translate(const Vector& v);
};

struct Node {  // rt/node.d:7-21
    const Geometry* geom = nullptr;
    const Shader* shader = nullptr;
    const Texture* bumpmap = nullptr;
    Transform transform;
};

struct NamedEntities {  // rt/scene.d:9-36
    std::map<std::string, Light*> lights;
    std::map<std::string, Geometry*> geometries;
    std::map<std::string, Texture*> textures;
    std::map<std::string, Shader*> shaders;
    std::map<std::string, Node*> nodes;
};

class Scene {  // rt/scene.d:38-58
public:
    std::string name;
    GlobalSettings settings;
    Environment environment;
    Camera camera;
    std::vector<std::unique_ptr<Light>> lights;
    std::vector<std::unique_ptr<Geometry>> geometries;
    std::vector<std::unique_ptr<Texture>> textures;
    std::vector<std::unique_ptr<Shader>> shaders;
    std::vector<std::unique_ptr<Node>> nodes;
    NamedEntities namedEntities;

    void beginFrame() { camera.beginFrame(); }

    // New with the CUDA backend: the uploaded (flattened) scene, created on first use by
    // uploadedScene (renderer.hpp) and reused by every later frame and query, the Renderer's and
    // the C entry points' (host_capi.cpp) alike.  Call invalidateDeviceScene() after
    // editing geometry or the environment, adding / removing entities, changing a texture's kind
    // or a bitmap's pixels (camera and settings are per-frame).  After changing only existing
    // entities' properties, call the matching hook instead: it re-flattens the listed entities
    // (indices into the vectors above) and edits the uploaded scene in place rather than
    // re-creating it.  nodesEdited: a node's geom or transform (c2rt_scene_set_nodes);
    // nodeShadersEdited: a node's shader (c2rt_scene_set_node_shaders); shadersEdited: a shader's
    // properties, or a shader replaced by another object in the same slot (c2rt_scene_set_shaders);
    // texturesEdited: a texture's colours, size, frequencies or scaling (c2rt_scene_set_textures);
    // lightsEdited: a light's pos, colour or power (c2rt_scene_set_lights).  They throw
    // BackendException on a library error, after dropping the uploaded scene.
    mutable std::shared_ptr<void> deviceScene;
    void invalidateDeviceScene() { deviceScene.reset(); }
    // The c2rt_frame_cache of Renderer::renderUpdate / c2rt_host_render_update (renderer.hpp frameCache): the last partial-or-full
    // frame delivered from this scene.  It compares the uploaded scene's records itself, so edits need not tell it anything.
    mutable std::shared_ptr<void> frameCache;
    void nodesEdited(const std::vector<int>& indices);
    void nodeShadersEdited(const std::vector<int>& indices);
    void shadersEdited(const std::vector<int>& indices);
    void texturesEdited(const std::vector<int>& indices);
    void lightsEdited(const std::vector<int>& indices);
};

// rt/scene_loader.d:20-41
std::unique_ptr<Scene> parseSceneFromFile(const std::string& filename);

// imageio/bmp.d:31-34 loadBmpImage!Color, :195-237 saveBmp (24 bpp)
Image<Color> loadBmpImage(const std::vector<uint8_t>& bytes);
// saveBmp writes what the reference writes, byte for byte: 14-byte file header, 40-byte BITMAPINFOHEADER (72 dpi = 2835 px/m),
// rows bottom-up, b g r per pixel — and, like the reference, NO padding of the rows to 4 bytes, so a width with 3 W % 4 != 0
// gives a file other readers (and the reference's own loader, bmp.d:136-188) misread.  padRows = true writes the valid file.
std::vector<uint8_t> saveBmp(const Image<uint32_t>& rgb32, bool padRows = false);

}  // namespace rt
