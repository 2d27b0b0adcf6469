// parseSceneFromFile: .sdl / .json -> rt::Scene.  Mirrors the reference loader's observable behaviour
// (/root/reference/source/rt/scene_loader.d:20-83 entry + fixed section order, :100-133 set/setTo with
// "missing property keeps the default", :142-203 value extraction, class factory by type name, named
// entities with duplicate detection) and each class's `deserialize`.  Load-time only.
#include <functional>

#include "rt.hpp"
#include "scene_text.hpp"

namespace rt {
namespace {

using c2rt_text::DscNode;

class SceneLoadContext {  // scene_loader.d:87-204
public:
    Scene* scene;
    std::string filePath;
    NamedEntities& named() { return scene->namedEntities; }

    template <class T>
    bool set(T& property, const DscNode& val, const char* name) {
        if (!val.isSpecified(name)) return false;
        extract(property, *val.getChild(name));
        return true;
    }
    std::string resolveRelativePath(const std::string& p) const {
        if (!p.empty() && p[0] == '/') return p;
        return c2rt_text::Document::dirName(filePath) + "/" + p;
    }

private:
    static void extract(bool& out, const DscNode& n) { out = n.getBool(); }
    static void extract(double& out, const DscNode& n) { out = n.getFloat(); }
    static void extract(float& out, const DscNode& n) { out = (float)n.getFloat(); }
    static void extract(std::string& out, const DscNode& n) { out = n.getString(); }
    static void extract(uint32_t& out, const DscNode& n) {
        long long v = n.getInt();
        if (v < 0 || v > 0xffffffffll) throw InvalidSceneException("integer value out of range");  // std.conv.to!uint throws
        out = (uint32_t)v;
    }
    static void extract(size_t& out, const DscNode& n) {
        long long v = n.getInt();
        if (v < 0) throw InvalidSceneException("integer value out of range");
        out = (size_t)v;
    }
    static void triple(const DscNode& n, double v[3]) {  // scene_loader.d:152-157
        auto vals = n.getValues();
        if (vals.size() < 3) throw InvalidSceneException("a Vector / Color needs three values");
        for (int i = 0; i < 3; i++) v[i] = vals[i].asDouble();
    }
    static void extract(Vector& out, const DscNode& n) {
        double v[3];
        triple(n, v);
        out = Vector(v[0], v[1], v[2]);
    }
    static void extract(Color& out, const DscNode& n) {
        double v[3];
        triple(n, v);
        out = Color((float)v[0], (float)v[1], (float)v[2]);
    }
    static void extract(std::vector<double>& out, const DscNode& n) {  // scalar arrays: the tag's values (:169-171)
        out.clear();
        for (auto& v : n.getValues()) out.push_back(v.asDouble());
    }
    static void extract(std::vector<Color>& out, const DscNode& n) {  // arrays of Color: one child per element (:173-174)
        out.clear();
        for (auto& ch : n.getChildren()) {
            Color c;
            extract(c, *ch);
            out.push_back(c);
        }
    }
};

template <class M>
typename M::mapped_type byName(M& m, const std::string& key, const char* what) {
    auto it = m.find(key);
    if (it == m.end()) throw InvalidSceneException(std::string("Unknown ") + what + " name: '" + key + "'");  // D: RangeError on the AA lookup
    return it->second;
}

template <class T, class M>
void store(const DscNode& n, T* obj, M& m) {  // scene_loader.d:195-200
    if (!n.hasName()) return;
    const std::string name = n.getName();
    if (m.count(name)) throw EntityWithDuplicateName(name);
    m[name] = obj;
}

void deserialize(GlobalSettings& s, const DscNode& v, SceneLoadContext& c) {  // global_settings.d:47-71
    c.set(s.frameWidth, v, "frameWidth");
    c.set(s.frameHeight, v, "frameHeight");
    c.set(s.fullscreen, v, "fullscreen");
    c.set(s.allowResize, v, "allowResize");
    c.set(s.dynamicAspectRatio, v, "dynamicAspectRatio");
    c.set(s.interactive, v, "interactive");
    c.set(s.bucketSize, v, "bucketSize");
    c.set(s.threadCount, v, "threadCount");
    c.set(s.prepassEnabled, v, "prepassEnabled");
    c.set(s.prepassOnly, v, "prepassOnly");
    c.set(s.GIEnabled, v, "GIEnabled");
    c.set(s.AAEnabled, v, "AAEnabled");
    c.set(s.AAThreshold, v, "AAThreshold");
    c.set(s.maxTraceDepth, v, "maxTraceDepth");
    c.set(s.pathsPerPixel, v, "pathsPerPixel");
    c.set(s.ambientLightColor, v, "ambientLightColor");
    c.set(s.debugEnabled, v, "debugEnabled");
}

void deserialize(Camera& cam, const DscNode& v, SceneLoadContext& c) {  // camera.d:238-255
    c.set(cam.pos, v, "pos");
    c.set(cam.yaw, v, "yaw");
    c.set(cam.pitch, v, "pitch");
    c.set(cam.roll, v, "roll");
    c.set(cam.fov, v, "fov");
    c.set(cam.focalPlaneDist, v, "focalPlaneDist");
    c.set(cam.fNumber, v, "fNumber");
    c.set(cam.dof, v, "dof");
    c.set(cam.numSamples, v, "numSamples");
    c.set(cam.stereoSeparation, v, "stereoSeparation");
    cam.discMultiplier = 10.0 / cam.fNumber;
    cam.setFrameSize(c.scene->settings.frameWidth, c.scene->settings.frameHeight);
}

const Texture* optionalTexture(const DscNode& v, SceneLoadContext& c, const char* key) {
    std::string t;
    c.set(t, v, key);
    auto it = c.named().textures.find(t);
    return it == c.named().textures.end() ? nullptr : it->second;
}

// util/factory2.d:5-23 makeInstanceOf: class by name
std::unique_ptr<Light> makeLight(const DscNode& n, SceneLoadContext& c) {
    if (n.getType() != "PointLight") throw InvalidSceneException("Unknown object type (or not yet supported): " + n.getType());
    auto l = std::make_unique<PointLight>();
    c.set(l->lightColor, n, "color");  // light.d:39-43
    c.set(l->lightPower, n, "power");
    c.set(l->pos, n, "pos");           // light.d:77-82
    return l;
}

std::unique_ptr<Geometry> makeGeometry(const DscNode& n, SceneLoadContext& c) {
    const std::string type = n.getType();
    if (type == "Plane") {
        auto g = std::make_unique<Plane>();
        c.set(g->y, n, "y");  // geometry.d:61-64
        return g;
    }
    if (type == "Sphere") {
        auto g = std::make_unique<Sphere>();
        if (!c.set(g->center, n, "center")) g->center = Vector(0, 0, 0);  // geometry.d:132-140
        c.set(g->R, n, "R");
        return g;
    }
    if (type == "Cube") {
        auto g = std::make_unique<Cube>();
        c.set(g->center, n, "center");  // geometry.d:237-241
        c.set(g->side, n, "side");
        return g;
    }
    if (type == "CsgUnion" || type == "CsgInter" || type == "CsgDiff") {
        std::unique_ptr<CsgOp> g;
        if (type == "CsgUnion") g = std::make_unique<CsgUnion>();
        else if (type == "CsgInter") g = std::make_unique<CsgInter>();
        else g = std::make_unique<CsgDiff>();
        std::string geomName;  // geometry.d:339-348
        c.set(geomName, n, "left");
        g->left = byName(c.named().geometries, geomName, "geometry");
        c.set(geomName, n, "right");
        g->right = byName(c.named().geometries, geomName, "geometry");
        return g;
    }
    throw InvalidSceneException("Unknown object type (or not yet supported): " + type);
}

std::unique_ptr<Texture> makeTexture(const DscNode& n, SceneLoadContext& c) {
    const std::string type = n.getType();
    if (type == "Checker") {
        auto t = std::make_unique<Checker>();
        c.set(t->color1, n, "color1");  // texture.d:56-61
        c.set(t->color2, n, "color2");
        c.set(t->size, n, "size");
        return t;
    }
    if (type == "Procedure2") {
        auto t = std::make_unique<Procedure2>();
        c.set(t->colorU, n, "colorU");  // texture.d:88-94
        c.set(t->colorV, n, "colorV");
        c.set(t->freqU, n, "freqU");
        c.set(t->freqV, n, "freqV");
        return t;
    }
    if (type == "BitmapTexture") {
        auto t = std::make_unique<BitmapTexture>();
        c.set(t->scaling, n, "scaling");  // texture.d:128-142
        c.set(t->assumedGamma, n, "assumedGamma");
        std::string file;
        c.set(file, n, "file");
        t->bmp.loadImage(c.resolveRelativePath(file));
        if (t->assumedGamma == 2.2f) t->bmp.decompressGamma_sRGB();
        else if (t->assumedGamma != 1 && t->assumedGamma > 0 && t->assumedGamma < 10) t->bmp.decompressGamma(t->assumedGamma);
        return t;
    }
    throw InvalidSceneException("Unknown object type (or not yet supported): " + type);
}

std::unique_ptr<Shader> makeShader(const DscNode& n, SceneLoadContext& c) {
    const std::string type = n.getType();
    if (type == "Lambert") {
        auto s = std::make_unique<Lambert>();
        c.set(s->color, n, "color");  // shader.d:40-44
        s->texture = optionalTexture(n, c, "texture");  // shader.d:137-147
        return s;
    }
    if (type == "Phong") {
        auto s = std::make_unique<Phong>();
        c.set(s->color, n, "color");
        c.set(s->exponent, n, "exponent");  // shader.d:263-280
        s->exponent = Phong::clampExponent(s->exponent);
        c.set(s->strength, n, "strength");
        s->strength = Phong::clampStrength(s->strength);
        s->texture = optionalTexture(n, c, "texture");
        return s;
    }
    throw InvalidSceneException("Unknown object type (or not yet supported): " + type);
}

std::unique_ptr<Node> makeNode(const DscNode& n, SceneLoadContext& c) {  // node.d:70-94
    if (n.getType() != "Node") throw InvalidSceneException("Unknown object type (or not yet supported): " + n.getType());
    auto node = std::make_unique<Node>();
    std::string geom, shad;
    c.set(geom, n, "geometry");
    c.set(shad, n, "shader");
    node->geom = byName(c.named().geometries, geom, "geometry");
    node->shader = byName(c.named().shaders, shad, "shader");
    node->bumpmap = optionalTexture(n, c, "bump");
    Vector v;
    if (c.set(v, n, "scale")) node->transform.scale(v.x, v.y, v.z);
    if (c.set(v, n, "rotate")) node->transform.scale(v.x, v.y, v.z);  // sic: the reference calls scale here (node.d:89-90)
    if (c.set(v, n, "translate")) node->transform.translate(v);
    return node;
}

template <class T, class M, class F>
void loadArray(const DscNode& root, const char* section, std::vector<std::unique_ptr<T>>& dst, M& names, SceneLoadContext& c, F make) {
    if (!root.isSpecified(section)) return;
    for (auto& child : root.getChild(section)->getChildren()) {
        std::unique_ptr<T> obj = make(*child, c);
        store(*child, obj.get(), names);
        dst.push_back(std::move(obj));
    }
}

}  // namespace

std::unique_ptr<Scene> parseSceneFromFile(const std::string& filename) {
    std::unique_ptr<c2rt_text::Document> doc;
    try {
        doc = std::make_unique<c2rt_text::Document>(filename);
    } catch (const c2rt_text::ParseError& e) {
        const std::string what = e.what();
        if (what.rfind("cannot open", 0) == 0) throw SceneNotFoundException();
        if (what.find("unknown file type") != std::string::npos) throw InvalidSceneException(what);
        throw InvalidSceneException(std::string(c2rt_text::Document::lowerExt(filename) == ".json" ? "Invalid JSON in scene file! " : "Invalid SDL in scene file! ") + what);
    }
    auto scene = std::make_unique<Scene>();
    SceneLoadContext ctx;
    ctx.scene = scene.get();
    ctx.filePath = filename;
    try {
        auto root = doc->root();
        ctx.set(scene->name, *root, "Name");
        if (root->isSpecified("GlobalSettings")) deserialize(scene->settings, *root->getChild("GlobalSettings"), ctx);
        if (root->isSpecified("Camera")) deserialize(scene->camera, *root->getChild("Camera"), ctx);
        // environment.d:12-14 reads no keys; the cubemap extension reads `folder` / `assumedGamma` (rt.hpp Environment)
        if (root->isSpecified("Environment")) {
            const auto enp = root->getChild("Environment");   // (keep the node alive: getChild returns it by value)
            const DscNode& en = *enp;
            std::string folder;
            ctx.set(folder, en, "folder");
            if (!folder.empty()) {
                static const char* names[6] = {"posx", "negx", "posy", "negy", "posz", "negz"};
                Environment& e = scene->environment;
                ctx.set(e.assumedGamma, en, "assumedGamma");
                for (int f = 0; f < 6; f++) {
                    e.faces[f].loadImage(ctx.resolveRelativePath(folder + "/" + names[f] + ".bmp"));
                    if (e.assumedGamma == 2.2f) e.faces[f].decompressGamma_sRGB();
                    else if (e.assumedGamma != 1 && e.assumedGamma > 0 && e.assumedGamma < 10) e.faces[f].decompressGamma(e.assumedGamma);
                }
                e.cubemap = true;
            }
        }
        loadArray(*root, "Lights", scene->lights, scene->namedEntities.lights, ctx, makeLight);
        loadArray(*root, "Geometries", scene->geometries, scene->namedEntities.geometries, ctx, makeGeometry);
        loadArray(*root, "Textures", scene->textures, scene->namedEntities.textures, ctx, makeTexture);
        loadArray(*root, "Shaders", scene->shaders, scene->namedEntities.shaders, ctx, makeShader);
        loadArray(*root, "Nodes", scene->nodes, scene->namedEntities.nodes, ctx, makeNode);
    } catch (const c2rt_text::ParseError& e) {
        throw InvalidSceneException(std::string("Invalid scene description: ") + e.what());
    }
    return scene;
}

}  // namespace rt
