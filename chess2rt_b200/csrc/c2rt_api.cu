// C ABI of libc2rt.so (include/c2rt.h): scene validation + upload (scene class, bounding spheres, node runs), frame
// launches on 1..8 devices (one helper thread per extra device: DevicePool), band copies to the host frame, error
// reporting.  No CPU fallback anywhere:
// every rendering entry point fails with C2RT_ERR_CUDA if the CUDA runtime cannot run the kernel.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <atomic>
#include <condition_variable>
#include <cstring>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "scene_dev.h"

namespace c2rt {
cudaError_t upload_scene(const DevScene& s, cudaStream_t st);
cudaError_t launch_frame(const FrameParams& fp, int mode, uint32_t local_tile_rows, cudaStream_t st);
cudaError_t launch_pixel(const FrameParams& fp, int mode, int x, int y, PixelOut* d_out, cudaStream_t st);
cudaError_t launch_hits(const FrameParams& fp, int mode, uint32_t local_tile_rows, const c2rt_hit_planes& out, cudaStream_t st);
cudaError_t launch_deinterleave(const void* src, void* dst, uint32_t row_words, uint32_t height, uint32_t n_ranks,
                                uint32_t band_rows, uint32_t rows_pad, cudaStream_t st);
cudaError_t launch_fma_peak(bool fp64, int blocks, int threads, int iters, void* d_out, cudaStream_t st);
cudaError_t launch_gate(void* gate, uint32_t round, uint32_t n_ranks, void* err, cudaStream_t st);
cudaError_t launch_signal(void* flag, uint32_t frame_no, cudaStream_t st);
}  // namespace c2rt

using namespace c2rt;

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) return fail(C2RT_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

struct DeviceCtx {
    int dev = -1;
    cudaStream_t stream = nullptr, copy_stream = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    std::vector<cudaEvent_t> band_done;
    uint64_t uploaded_scene = 0;   // id of the scene currently in this device's constant memory
    unsigned long long* d_counters = nullptr;
    uint32_t* d_done_counter = nullptr;   // CTAs of the current launch that finished (in-kernel completion)
    int* d_cancel = nullptr;       // raised by c2rt_cancel, cleared at the start of every c2rt_render
    cudaStream_t cancel_stream = nullptr;
    uint8_t* d_lut = nullptr;
    PixelOut* d_pixel = nullptr;
    float* d_rgb = nullptr;
    uint32_t* d_argb = nullptr;
    uint32_t* d_hits = nullptr;   // the four planes of a c2rt_render_hits frame, one after the other
    size_t rgb_cap = 0, argb_cap = 0, hits_cap = 0;
};

struct Context {
    bool inited = false;
    int n = 0;
    DeviceCtx d[C2RT_MAX_GPUS];
    uint64_t next_scene_id = 1;
    uint8_t lut[4097];
};

Context g_ctx;
std::mutex g_mu;
std::atomic<bool> g_cancel_requested{false};   // c2rt_cancel -> the c2rt_render in progress (c2rt_cancel takes no lock)

// One host thread per extra device (c2rt_init(N > 1)): c2rt_render hands every device's launch / copy sequence to its
// own thread, so the ~10 driver calls per device are issued in parallel instead of one after the other (at 1080p the
// serial submission of 8 devices cost more than rendering and copying the frame).  Workers spin for a short while after
// a frame — an interactive loop or a benchmark asks for the next one immediately — and then sleep on a condition variable.
class DevicePool {
public:
    void start(int n_workers) {
        stop();
        stop_ = false;
        const uint64_t g0 = gen_.load(std::memory_order_acquire);
        for (int w = 0; w < n_workers; w++) th_.emplace_back([this, w, g0] { loop(w, g0); });
    }
    void stop() {
        {
            std::lock_guard<std::mutex> lk(m_);
            stop_ = true;
            gen_.fetch_add(1, std::memory_order_release);
        }
        cv_work_.notify_all();
        for (auto& t : th_) t.join();
        th_.clear();
    }
    // runs fn(w) on every worker w = 0..n_workers-1; returns immediately, wait() joins the round
    void run(std::function<void(int)> fn) {
        fn_ = std::move(fn);
        pending_.store((int)th_.size(), std::memory_order_relaxed);
        {
            std::lock_guard<std::mutex> lk(m_);
            gen_.fetch_add(1, std::memory_order_release);
        }
        cv_work_.notify_all();
    }
    void wait() {
        for (int k = 0; k < 200000 && pending_.load(std::memory_order_acquire) != 0; k++) relax();
        if (pending_.load(std::memory_order_acquire) == 0) return;
        std::unique_lock<std::mutex> lk(m_);
        cv_done_.wait(lk, [this] { return pending_.load(std::memory_order_acquire) == 0; });
    }
    ~DevicePool() { stop(); }

private:
    static void relax() {
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#endif
    }
    void loop(int w, uint64_t seen) {
        for (;;) {
            bool got = false;
            for (int k = 0; k < 100000; k++) {
                if (gen_.load(std::memory_order_acquire) != seen) { got = true; break; }
                relax();
            }
            if (!got) {
                std::unique_lock<std::mutex> lk(m_);
                cv_work_.wait(lk, [&] { return gen_.load(std::memory_order_acquire) != seen; });
            }
            seen = gen_.load(std::memory_order_acquire);
            if (stop_) return;
            fn_(w);
            if (pending_.fetch_sub(1, std::memory_order_acq_rel) == 1) {
                std::lock_guard<std::mutex> lk(m_);
                cv_done_.notify_one();
            }
        }
    }
    std::vector<std::thread> th_;
    std::mutex m_;
    std::condition_variable cv_work_, cv_done_;
    std::function<void(int)> fn_;
    std::atomic<uint64_t> gen_{0};
    std::atomic<int> pending_{0};
    bool stop_ = false;
};
DevicePool g_pool;

// color.d:194-207 convertTo8bit_sRGB, quirks kept: 12.02 linear slope, floor instead of round
uint8_t srgb8(float x) {
    if (x <= 0) return 0;
    if (x >= 1) return 255;
    if (x <= 0.0031308f) x = x * 12.02f;
    else x = (float)(1.055 * pow((double)x, 1 / 2.4) - 0.055);
    return (uint8_t)floorf(x * 255.0f);
}

void destroy_device(DeviceCtx& c) {
    if (c.dev < 0) return;
    cudaSetDevice(c.dev);
    if (c.stream) cudaStreamDestroy(c.stream);
    if (c.copy_stream) cudaStreamDestroy(c.copy_stream);
    for (auto& e : c.band_done) cudaEventDestroy(e);
    if (c.e0) cudaEventDestroy(c.e0);
    if (c.e1) cudaEventDestroy(c.e1);
    cudaFree(c.d_counters);
    cudaFree(c.d_done_counter);
    cudaFree(c.d_cancel);
    if (c.cancel_stream) cudaStreamDestroy(c.cancel_stream);
    cudaFree(c.d_lut);
    cudaFree(c.d_pixel);
    cudaFree(c.d_rgb);
    cudaFree(c.d_argb);
    cudaFree(c.d_hits);
    c = DeviceCtx();
}

int init_locked(int n_gpus, const int* ids) {
    if (n_gpus < 1 || n_gpus > C2RT_MAX_GPUS) return fail(C2RT_ERR_INVALID_ARG, "n_gpus must be in 1..%d", C2RT_MAX_GPUS);
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(C2RT_ERR_CUDA, "no CUDA device available (%s); libc2rt has no CPU fallback", cudaGetErrorString(e));
    g_pool.stop();
    for (int i = 0; i < g_ctx.n; i++) destroy_device(g_ctx.d[i]);
    g_ctx.n = 0;
    g_ctx.inited = false;
    for (int i = 0; i < 4097; i++) g_ctx.lut[i] = srgb8((float)i / 4096.f);
    for (int i = 0; i < n_gpus; i++) {
        int dev = ids ? ids[i] : i;
        if (dev < 0 || dev >= count) return fail(C2RT_ERR_INVALID_ARG, "device id %d out of range (have %d)", dev, count);
        DeviceCtx& c = g_ctx.d[i];
        c.dev = dev;
        CU(cudaSetDevice(dev));
        CU(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&c.copy_stream, cudaStreamNonBlocking));
        CU(cudaEventCreate(&c.e0));
        CU(cudaEventCreate(&c.e1));
        CU(cudaMalloc(&c.d_counters, 2 * sizeof(unsigned long long)));
        CU(cudaMemset(c.d_counters, 0, 2 * sizeof(unsigned long long)));
        CU(cudaMalloc(&c.d_done_counter, sizeof(uint32_t)));
        CU(cudaMemset(c.d_done_counter, 0, sizeof(uint32_t)));
        CU(cudaMalloc(&c.d_cancel, sizeof(int)));
        CU(cudaMemset(c.d_cancel, 0, sizeof(int)));
        CU(cudaStreamCreateWithFlags(&c.cancel_stream, cudaStreamNonBlocking));
        CU(cudaMalloc(&c.d_lut, 4097));
        CU(cudaMemcpy(c.d_lut, g_ctx.lut, 4097, cudaMemcpyHostToDevice));
        CU(cudaMalloc(&c.d_pixel, sizeof(PixelOut)));
        g_ctx.n = i + 1;
    }
    cudaSetDevice(g_ctx.d[0].dev);
    g_ctx.inited = true;
    if (n_gpus > 1) g_pool.start(n_gpus - 1);   // worker w drives device w + 1; the caller's thread drives device 0
    return C2RT_OK;
}

int ensure_init_locked() {
    if (g_ctx.inited) return C2RT_OK;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) {
        cudaGetLastError();
        return fail(C2RT_ERR_CUDA, "no CUDA device available; libc2rt has no CPU fallback");
    }
    return init_locked(1, &dev);
}

DeviceCtx* find_device(int dev) {
    for (int i = 0; i < g_ctx.n; i++)
        if (g_ctx.d[i].dev == dev) return &g_ctx.d[i];
    return nullptr;
}

}  // namespace

struct c2rt_scene {
    uint64_t id;
    DevScene host;                       // constant block; record arrays copied in from the vectors below when they fit
    std::vector<DevNode> nodes;          // the scene's records (texel pointers patched per device at upload)
    std::vector<DevGeom> geoms;
    std::vector<DevShader> shaders;
    std::vector<DevTex> textures;
    bool big = false;                    // beyond the constant block: the records go to global memory (MODE_BIG)
    void* d_records[C2RT_MAX_GPUS][4];   // big scenes, per context device: nodes, geoms, shaders, textures
    std::vector<float4> texels;          // bitmaps in the general form, float4 per texel
    std::vector<size_t> tex_offset;      // per texture, in texels (general-form bitmaps only)
    float4* d_texels[C2RT_MAX_GPUS];     // per context device
    // bitmaps with <= 256 distinct colours (scene_dev.h DevTex::quads): index quads + 256-entry palettes
    std::vector<uint32_t> quads;
    std::vector<float4> palettes;
    std::vector<long long> quad_offset, pal_offset;   // per texture; -1 = general form
    uint32_t* d_quads[C2RT_MAX_GPUS];
    float4* d_palettes[C2RT_MAX_GPUS];
    float4* d_bounds[C2RT_MAX_GPUS];     // per context device: node bounding spheres for the per-warp masks (FrameParams.bounds)
    int n_dev;
    int mode;                            // kernel specialisation (render_kernel.cu MODE_*)
};

namespace {

struct Bound {
    bool finite;
    double c[3], r;
};

Bound union_bound(const Bound& l, const Bound& r) {
    Bound b{};
    if (!l.finite || !r.finite) { b.finite = false; return b; }
    double dx = r.c[0] - l.c[0], dy = r.c[1] - l.c[1], dz = r.c[2] - l.c[2];
    double dist = sqrt(dx * dx + dy * dy + dz * dz);
    if (dist + r.r <= l.r) return l;
    if (dist + l.r <= r.r) return r;
    b.finite = true;
    b.r = (dist + l.r + r.r) * 0.5;
    double t = (b.r - l.r) / dist;
    b.c[0] = l.c[0] + dx * t; b.c[1] = l.c[1] + dy * t; b.c[2] = l.c[2] + dz * t;
    return b;
}

// Bounding sphere of everything a geometry can report a hit on.  For a CSG of two primitives the boolean
// is evaluated faithfully, so diff is bounded by its left child and inter by the smaller child.  Once a
// child is itself a CSG the reference's walk is quirky (a nested child's crossings toggle the wrong flag,
// entry-only crossing lists flip the initial parity: tests/scenes/nested.sdl) and a hit may be reported on
// ANY leaf surface: the bound is then the union over all leaves.
Bound bound_of(const c2rt_scene_desc* d, int gi) {
    Bound b{};
    const double* p = d->geom_params + 4 * gi;
    const int type = d->geom_type[gi];
    if (type == C2RT_GEOM_SPHERE) {
        b.finite = std::isfinite(p[3]);
        b.c[0] = p[0]; b.c[1] = p[1]; b.c[2] = p[2];
        b.r = fabs(p[3]);
    } else if (type == C2RT_GEOM_CUBE) {
        b.finite = std::isfinite(p[3]);
        b.c[0] = p[0]; b.c[1] = p[1]; b.c[2] = p[2];
        b.r = fabs(p[3]) * 0.5 * sqrt(3.0);
    } else if (type >= C2RT_GEOM_CSG_UNION) {
        const int li = d->geom_left[gi], ri = d->geom_right[gi];
        Bound l = bound_of(d, li), r = bound_of(d, ri);
        const bool nested = d->geom_type[li] >= C2RT_GEOM_CSG_UNION || d->geom_type[ri] >= C2RT_GEOM_CSG_UNION;
        if (nested || type == C2RT_GEOM_CSG_UNION) b = union_bound(l, r);
        else if (type == C2RT_GEOM_CSG_INTER) {
            if (l.finite && r.finite) b = l.r <= r.r ? l : r;
            else if (l.finite) b = l;
            else if (r.finite) b = r;
            else b.finite = false;
        } else b = l;  // diff
    } else {
        b.finite = false;  // plane
    }
    if (b.finite && !(std::isfinite(b.c[0]) && std::isfinite(b.c[1]) && std::isfinite(b.c[2]) && std::isfinite(b.r))) b.finite = false;
    return b;
}

bool is_identity(const double* m) {
    for (int i = 0; i < 9; i++)
        if (m[i] != ((i % 4 == 0) ? 1.0 : 0.0)) return false;
    return true;
}

// Device form of one bitmap (a texture or an environment face): palette-index quads when it has <= 256 distinct texel
// colours (scene_dev.h DevTex::quads), float4 texels otherwise.  `slot` indexes the scene's offset tables.
void build_bitmap(c2rt_scene* s, const DevTex& t, const float* src, int slot) {
    const uint64_t n = (uint64_t)t.w * t.h;
    const int i = slot;
    // <= 256 distinct texel colours -> palette form (C2RT_NO_PALETTE=1: test hook, keep the general form)
    const char* no_pal = getenv("C2RT_NO_PALETTE");
    std::vector<uint8_t> idx;
    std::vector<float4> pal;
    if (!(no_pal && no_pal[0] == '1')) {
        struct Key { uint32_t r, g, b; bool operator==(const Key& o) const { return r == o.r && g == o.g && b == o.b; } };
        struct KeyHash { size_t operator()(const Key& k) const { return (size_t)k.r * 0x9E3779B1u ^ (size_t)k.g * 0x85EBCA77u ^ (size_t)k.b * 0xC2B2AE3Du; } };
        std::unordered_map<Key, int, KeyHash> seen;
        idx.resize(n);
        for (uint64_t k = 0; k < n; k++) {
            Key key;
            memcpy(&key, src + 3 * k, 12);   // bit patterns: -0 / NaN payloads stay distinct, the palette returns the same bits
            auto it = seen.find(key);
            if (it == seen.end()) {
                if (seen.size() == 256) { idx.clear(); break; }
                it = seen.emplace(key, (int)seen.size()).first;
                pal.push_back(make_float4(src[3 * k], src[3 * k + 1], src[3 * k + 2], 0.f));
            }
            idx[k] = (uint8_t)it->second;
        }
    }
    if (!idx.empty()) {
        s->quad_offset[i] = (long long)s->quads.size();
        s->pal_offset[i] = (long long)s->palettes.size();
        pal.resize(256, make_float4(0.f, 0.f, 0.f, 0.f));
        s->palettes.insert(s->palettes.end(), pal.begin(), pal.end());
        s->quads.resize(s->quads.size() + n);
        uint32_t* q = s->quads.data() + s->quad_offset[i];
        for (int y = 0; y < t.h; y++) {
            const int yn = y + 1 == t.h ? 0 : y + 1;
            for (int x = 0; x < t.w; x++) {
                const int xn = x + 1 == t.w ? 0 : x + 1;
                q[(size_t)y * t.w + x] = (uint32_t)idx[(size_t)y * t.w + x] | ((uint32_t)idx[(size_t)y * t.w + xn] << 8) |
                                         ((uint32_t)idx[(size_t)yn * t.w + x] << 16) | ((uint32_t)idx[(size_t)yn * t.w + xn] << 24);
            }
        }
    } else {
        s->tex_offset[i] = s->texels.size();
        s->texels.resize(s->texels.size() + n);
        float4* dst = s->texels.data() + s->tex_offset[i];
        for (uint64_t k = 0; k < n; k++) dst[k] = make_float4(src[3 * k], src[3 * k + 1], src[3 * k + 2], 0.f);
    }
}

int validate_and_build(const c2rt_scene_desc* d, c2rt_scene* s) {
    if (!d) return fail(C2RT_ERR_INVALID_ARG, "scene description is null");
    if (d->struct_size != sizeof(c2rt_scene_desc) || d->abi_version != C2RT_ABI_VERSION)
        return fail(C2RT_ERR_INVALID_ARG, "scene description ABI mismatch (size %u/%zu, version %u/%d)", d->struct_size,
                    sizeof(c2rt_scene_desc), d->abi_version, C2RT_ABI_VERSION);
    if (d->n_nodes > C2RT_MAX_NODES_GLOBAL) return fail(C2RT_ERR_LIMIT, "too many nodes (%u > %d)", d->n_nodes, C2RT_MAX_NODES_GLOBAL);
    if (d->n_geoms > C2RT_MAX_GEOMS_GLOBAL) return fail(C2RT_ERR_LIMIT, "too many geometries (%u > %d)", d->n_geoms, C2RT_MAX_GEOMS_GLOBAL);
    if (d->n_shaders > C2RT_MAX_SHADERS_GLOBAL) return fail(C2RT_ERR_LIMIT, "too many shaders (%u > %d)", d->n_shaders, C2RT_MAX_SHADERS_GLOBAL);
    if (d->n_textures > C2RT_MAX_TEXTURES_GLOBAL) return fail(C2RT_ERR_LIMIT, "too many textures (%u > %d)", d->n_textures, C2RT_MAX_TEXTURES_GLOBAL);
    if (d->n_lights > C2RT_MAX_LIGHTS) return fail(C2RT_ERR_LIMIT, "too many lights (%u > %d)", d->n_lights, C2RT_MAX_LIGHTS);
    // a scene beyond the constant block keeps its records in global memory (C2RT_FORCE_GLOBAL=1: test hook, any scene does)
    const char* force_big = getenv("C2RT_FORCE_GLOBAL");
    s->big = d->n_nodes > C2RT_MAX_NODES || d->n_geoms > C2RT_MAX_GEOMS || d->n_shaders > C2RT_MAX_SHADERS ||
             d->n_textures > C2RT_MAX_TEXTURES || (force_big && force_big[0] == '1');
    if (d->n_nodes && !(d->node_geom && d->node_shader && d->node_transform && d->node_inverse && d->node_inverse_t && d->node_offset))
        return fail(C2RT_ERR_INVALID_ARG, "node arrays missing");
    if (d->n_geoms && !(d->geom_type && d->geom_params && d->geom_left && d->geom_right))
        return fail(C2RT_ERR_INVALID_ARG, "geometry arrays missing");
    if (d->n_shaders && !(d->shader_type && d->shader_color && d->shader_texture && d->shader_exponent && d->shader_strength))
        return fail(C2RT_ERR_INVALID_ARG, "shader arrays missing");
    if (d->n_textures && !(d->tex_type && d->tex_colors && d->tex_params && d->tex_width && d->tex_height && d->tex_texel_offset))
        return fail(C2RT_ERR_INVALID_ARG, "texture arrays missing");
    if (d->n_lights && !(d->light_pos && d->light_color && d->light_power)) return fail(C2RT_ERR_INVALID_ARG, "light arrays missing");

    DevScene& h = s->host;
    memset(&h, 0, sizeof h);
    DevNode zn; DevGeom zg; DevShader zs; DevTex zt;
    memset(&zn, 0, sizeof zn); memset(&zg, 0, sizeof zg); memset(&zs, 0, sizeof zs); memset(&zt, 0, sizeof zt);
    s->nodes.assign(d->n_nodes, zn);
    s->geoms.assign(d->n_geoms, zg);
    s->shaders.assign(d->n_shaders, zs);
    s->textures.assign(d->n_textures, zt);
    h.n_nodes = d->n_nodes; h.n_geoms = d->n_geoms; h.n_shaders = d->n_shaders; h.n_textures = d->n_textures; h.n_lights = d->n_lights;

    for (uint32_t i = 0; i < d->n_geoms; i++) {
        int t = d->geom_type[i];
        DevGeom& g = s->geoms[i];
        g.type = t; g.left = -1; g.right = -1;
        memcpy(g.p, d->geom_params + 4 * i, 4 * sizeof(double));
        if (t < C2RT_GEOM_PLANE || t > C2RT_GEOM_CSG_DIFF) return fail(C2RT_ERR_INVALID_ARG, "geometry %u: unknown type %d", i, t);
        if (t >= C2RT_GEOM_CSG_UNION) {
            int l = d->geom_left[i], r = d->geom_right[i];
            if (l < 0 || r < 0 || l >= (int)i || r >= (int)i)
                return fail(C2RT_ERR_INVALID_ARG, "geometry %u: CSG children must be earlier geometries (left %d, right %d)", i, l, r);
            g.left = l; g.right = r;
            const int dl = abs(s->geoms[l].depth), dr = abs(s->geoms[r].depth);
            g.depth = 1 + (dl > dr ? dl : dr);
            if (g.depth > 3)
                return fail(C2RT_ERR_UNSUPPORTED, "geometry %u: CSG nesting deeper than 3 levels is not supported", i);
            // tuning / testing aid: C2RT_CSG_LITERAL=1 routes every CSG through the literal emulation
            const char* lit = getenv("C2RT_CSG_LITERAL");
            if (lit && lit[0] == '1' && g.depth == 1) g.depth = -1;
        }
    }
    s->tex_offset.assign(d->n_textures + 6, 0);     // + 6: the environment faces
    s->quad_offset.assign(d->n_textures + 6, -1);
    s->pal_offset.assign(d->n_textures + 6, -1);
    for (uint32_t i = 0; i < d->n_textures; i++) {
        DevTex& t = s->textures[i];
        t.type = d->tex_type[i];
        if (t.type < C2RT_TEX_CHECKER || t.type > C2RT_TEX_BITMAP) return fail(C2RT_ERR_INVALID_ARG, "texture %u: unknown type %d", i, t.type);
        memcpy(t.c, d->tex_colors + 18 * i, 18 * sizeof(float));
        memcpy(t.d, d->tex_params + 6 * i, 6 * sizeof(double));
        if (t.type == C2RT_TEX_CHECKER) t.d[1] = 1.0 / t.d[0];
        if (t.type == C2RT_TEX_PROCEDURE2) {
            // frequencies in 2^-32 revolutions per unit (render_kernel.cu sin_phase / sin_rev), and the |u|, |v| up to which every
            // phase stays below 2^18 revolutions, as the high word of a double (compared against the coordinate's high word)
            for (int a = 0; a < 2; a++) {
                double fmax = 0.0;
                for (int k = 0; k < 3; k++) {
                    double& f = t.d[3 * a + k];
                    f = f / 6.283185307179586476925 * 4294967296.0;
                    fmax = std::isfinite(f) ? std::max(fmax, std::fabs(f)) : INFINITY;
                }
                const double lim = fmax > 0 ? 262144.0 * 4294967296.0 / fmax : INFINITY;   // (fmax = inf: 0, always the two-step path)
                uint64_t bits;
                memcpy(&bits, &lim, 8);
                (a ? t.h : t.w) = (int)(uint32_t)(bits >> 32);
            }
        }
        if (t.type == C2RT_TEX_BITMAP) {
            t.w = d->tex_width[i]; t.h = d->tex_height[i];
            if (t.w <= 0 || t.h <= 0) return fail(C2RT_ERR_INVALID_ARG, "texture %u: empty bitmap", i);
            uint64_t off = d->tex_texel_offset[i], n = (uint64_t)t.w * t.h;
            if (!d->texels || off + n > d->n_texels) return fail(C2RT_ERR_INVALID_ARG, "texture %u: texel range outside `texels`", i);
            build_bitmap(s, t, d->texels + 3 * off, (int)i);
        }
    }
    // environment (c2rt.h C2RT_ENV_CUBEMAP): six more bitmap records, slots n_textures .. n_textures + 5 of the offset tables
    h.env_type = d->env_type;
    if (d->env_type != C2RT_ENV_BLACK && d->env_type != C2RT_ENV_CUBEMAP) return fail(C2RT_ERR_INVALID_ARG, "unknown environment type %d", d->env_type);
    if (d->env_type == C2RT_ENV_CUBEMAP)
        for (int f = 0; f < 6; f++) {
            DevTex& t = h.env_faces[f];
            t.type = C2RT_TEX_BITMAP;
            t.w = d->env_face_width[f]; t.h = d->env_face_height[f];
            if (t.w <= 0 || t.h <= 0) return fail(C2RT_ERR_INVALID_ARG, "environment face %d: empty bitmap", f);
            uint64_t off = d->env_face_texel_offset[f], n = (uint64_t)t.w * t.h;
            if (!d->texels || off + n > d->n_texels) return fail(C2RT_ERR_INVALID_ARG, "environment face %d: texel range outside `texels`", f);
            build_bitmap(s, t, d->texels + 3 * off, (int)d->n_textures + f);
        }
    for (uint32_t i = 0; i < d->n_shaders; i++) {
        DevShader& sh = s->shaders[i];
        sh.type = d->shader_type[i];
        if (sh.type != C2RT_SHADER_LAMBERT && sh.type != C2RT_SHADER_PHONG) return fail(C2RT_ERR_INVALID_ARG, "shader %u: unknown type %d", i, sh.type);
        sh.tex = d->shader_texture[i];
        if (sh.tex >= (int)d->n_textures) return fail(C2RT_ERR_INVALID_ARG, "shader %u: texture index %d out of range", i, sh.tex);
        if (sh.tex < 0) sh.tex = -1;
        memcpy(sh.color, d->shader_color + 3 * i, 3 * sizeof(float));
        sh.exponent = d->shader_exponent[i];
        sh.strength = d->shader_strength[i];
    }
    for (uint32_t i = 0; i < d->n_lights; i++) {
        DevLight& L = h.lights[i];
        memcpy(L.pos, d->light_pos + 3 * i, 3 * sizeof(double));
        // light.d:11-14: Color * float in FP32
        float pw = d->light_power[i];
        for (int k = 0; k < 3; k++) L.color[k] = d->light_color[3 * i + k] * pw;
        float intensity = (L.color[0] + L.color[1] + L.color[2]) / 3;  // color.d:141-144
        L.lit = intensity != 0;
        for (int k = 0; k < 3; k++) L.posf[k] = (float)L.pos[k];
        L.near2 = (float)(0.0576 * (L.pos[0] * L.pos[0] + L.pos[1] * L.pos[1] + L.pos[2] * L.pos[2]));
        if (L.lit) h.lit[h.n_lit++] = (int)i;
    }
    for (uint32_t i = 0; i < d->n_nodes; i++) {
        DevNode& nd = s->nodes[i];
        nd.geom = d->node_geom[i];
        nd.shader = d->node_shader[i];
        if (nd.geom < 0 || nd.geom >= (int)d->n_geoms) return fail(C2RT_ERR_INVALID_ARG, "node %u: geometry index %d out of range", i, nd.geom);
        if (nd.shader < 0 || nd.shader >= (int)d->n_shaders) return fail(C2RT_ERR_INVALID_ARG, "node %u: shader index %d out of range", i, nd.shader);
        memcpy(nd.M, d->node_transform + 9 * i, 9 * sizeof(double));
        memcpy(nd.Minv, d->node_inverse + 9 * i, 9 * sizeof(double));
        memcpy(nd.MinvT, d->node_inverse_t + 9 * i, 9 * sizeof(double));
        memcpy(nd.off, d->node_offset + 3 * i, 3 * sizeof(double));
        nd.flags = 0;
        if (is_identity(nd.M) && is_identity(nd.Minv) && is_identity(nd.MinvT)) nd.flags |= NODE_IDENTITY;
        Bound b = bound_of(d, nd.geom);
        if (b.finite) {
            // world centre = c*M + offset; radius scaled by an upper bound of |M|_2
            double cx = b.c[0] * nd.M[0] + b.c[1] * nd.M[3] + b.c[2] * nd.M[6] + nd.off[0];
            double cy = b.c[0] * nd.M[1] + b.c[1] * nd.M[4] + b.c[2] * nd.M[7] + nd.off[1];
            double cz = b.c[0] * nd.M[2] + b.c[1] * nd.M[5] + b.c[2] * nd.M[8] + nd.off[2];
            double fro = 0, n1 = 0, ninf = 0;
            for (int r = 0; r < 3; r++) {
                double rs = 0, cs = 0;
                for (int c = 0; c < 3; c++) {
                    fro += nd.M[3 * r + c] * nd.M[3 * r + c];
                    rs += fabs(nd.M[3 * r + c]);
                    cs += fabs(nd.M[3 * c + r]);
                }
                ninf = fmax(ninf, rs);
                n1 = fmax(n1, cs);
            }
            double scale = fmin(sqrt(fro), sqrt(n1 * ninf));
            // inflate: covers the 1e-6 restarts/probes of the CSG walk and rounding in the test itself
            double r = b.r * scale * (1.0 + 1e-6) + 1e-4 * fmax(1.0, scale);
            // the cull runs in FP32: round the centre, grow the radius by the rounding it introduces
            float fx = (float)cx, fy = (float)cy, fz = (float)cz;
            double shift = sqrt((cx - fx) * (cx - fx) + (cy - fy) * (cy - fy) + (cz - fz) * (cz - fz));
            r = (r + shift) * (1.0 + 1e-6);
            float rf = (float)r;
            if ((double)rf < r) rf = nextafterf(rf, INFINITY);
            if (std::isfinite(cx) && std::isfinite(cy) && std::isfinite(cz) && std::isfinite(r) && std::isfinite(rf) &&
                std::isfinite(rf * rf)) {
                nd.bcf[0] = fx; nd.bcf[1] = fy; nd.bcf[2] = fz;
                nd.brf = rf;
                nd.br2f = nextafterf(rf * rf, INFINITY);
                nd.bclen = nextafterf(sqrtf(fx * fx + fy * fy + fz * fz), INFINITY);
            } else {
                nd.flags |= NODE_UNBOUNDED;
            }
        } else {
            nd.flags |= NODE_UNBOUNDED;
        }
        // world-space fast path for identity-transform primitives, and for unbounded planes under a positive
        // diagonal scale (Node "scale", zaphod.sdl): such a plane is the world plane y = y0 * sy + off.y, its
        // object-space uv (geometry.d:54-55) are the world offsets times 1/sx, 1/sz
        nd.kind = KIND_GENERIC;
        const DevGeom& g = s->geoms[nd.geom];
        nd.wp[1] = 1.0; nd.wp[2] = 1.0;
        if (g.type == C2RT_GEOM_PLANE && std::isnan(g.p[1])) {   // bounded planes (limit set) keep the generic path
            bool diag = nd.M[0] > 0 && nd.M[4] > 0 && nd.M[8] > 0;
            for (int k = 0; k < 9; k++)
                if (k % 4 != 0 && (nd.M[k] != 0.0 || nd.Minv[k] != 0.0)) diag = false;
            if (diag) {
                nd.kind = KIND_PLANE_W;
                nd.wp[0] = g.p[0] * nd.M[4] + nd.off[1];
                nd.wp[1] = nd.Minv[0];
                nd.wp[2] = nd.Minv[8];
            }
        } else if ((nd.flags & NODE_IDENTITY) && !(nd.flags & NODE_UNBOUNDED) && (g.type == C2RT_GEOM_SPHERE || g.type == C2RT_GEOM_CUBE)) {
            // (a sphere / cube whose bound was rejected — non-finite or overflowing radius — stays KIND_GENERIC: the
            // plane-only and bounded kernel classes assume every KIND_*_W sphere / cube carries a finite bound)
            nd.kind = g.type == C2RT_GEOM_SPHERE ? KIND_SPHERE_W : KIND_CUBE_W;
            nd.wp[0] = g.p[0] + nd.off[0]; nd.wp[1] = g.p[1] + nd.off[1]; nd.wp[2] = g.p[2] + nd.off[2];
            nd.wp[3] = g.p[3];
        }
    }
    s->mode = 0;
    for (uint32_t i = 0; i < d->n_nodes; i++) {
        if (!(s->nodes[i].flags & NODE_UNBOUNDED)) s->mode |= MODE_BOUNDED;
        if (s->nodes[i].kind == KIND_GENERIC) s->mode |= MODE_GENERIC;
        const DevGeom& ng = s->geoms[s->nodes[i].geom];
        // (MODE_NESTED implies the generic, bounded kernel)
        if (ng.type >= C2RT_GEOM_CSG_UNION && ng.depth != 1) s->mode |= MODE_NESTED | MODE_GENERIC | MODE_BOUNDED;
    }
    // MODE_SOLO: exactly one node, a world-space plane, and exactly one light.  The node's shader and that shader's
    // texture are swapped into record 0 so the kernel addresses every scene constant statically.
    const char* no_solo = getenv("C2RT_NO_SOLO");   // test hook: keep such scenes on the general plane-only kernel
    if (!s->big && s->mode == 0 && h.n_nodes == 1 && h.n_lights == 1 && s->nodes[0].kind == KIND_PLANE_W && !(no_solo && no_solo[0] == '1')) {
        const int si = s->nodes[0].shader;
        std::swap(s->shaders[0], s->shaders[si]);
        s->nodes[0].shader = 0;
        const int ti = s->shaders[0].tex;
        if (ti >= 0) {
            std::swap(s->textures[0], s->textures[ti]);
            std::swap(s->tex_offset[0], s->tex_offset[ti]);
            std::swap(s->quad_offset[0], s->quad_offset[ti]);
            std::swap(s->pal_offset[0], s->pal_offset[ti]);
            for (int k = 0; k < h.n_shaders; k++) {
                if (s->shaders[k].tex == 0) s->shaders[k].tex = ti;
                else if (s->shaders[k].tex == ti) s->shaders[k].tex = 0;
            }
        }
        s->mode = MODE_SOLO | ((s->shaders[0].tex >= 0 ? 1 + s->textures[0].type : 0) << MODE_TEX_SHIFT) |
                  (s->shaders[0].type == C2RT_SHADER_PHONG ? MODE_PHONG : 0);
    }
    if (s->big) s->mode = (s->mode & MODE_NESTED) | MODE_BOUNDED | MODE_GENERIC | MODE_BIG;   // the general kernels only
    return C2RT_OK;
}

int upload_to_devices(c2rt_scene* s) {
    s->n_dev = g_ctx.n;
    for (int i = 0; i < C2RT_MAX_GPUS; i++) {
        s->d_texels[i] = nullptr; s->d_bounds[i] = nullptr; s->d_quads[i] = nullptr; s->d_palettes[i] = nullptr;
        for (int k = 0; k < 4; k++) s->d_records[i][k] = nullptr;
    }
    std::vector<float4> bounds((size_t)std::max(1, s->host.n_nodes));
    for (int k = 0; k < s->host.n_nodes; k++) {
        const DevNode& nd = s->nodes[k];
        bounds[k] = (nd.flags & NODE_UNBOUNDED) ? make_float4(0.f, 0.f, 0.f, -1.f) : make_float4(nd.bcf[0], nd.bcf[1], nd.bcf[2], nd.brf);
    }
    for (int i = 0; i < g_ctx.n; i++) {
        CU(cudaSetDevice(g_ctx.d[i].dev));
        CU(cudaMalloc(&s->d_bounds[i], bounds.size() * sizeof(float4)));
        CU(cudaMemcpy(s->d_bounds[i], bounds.data(), bounds.size() * sizeof(float4), cudaMemcpyHostToDevice));
        if (s->big) {   // filled by make_resident (the texture records carry per-device pointers)
            const size_t bytes[4] = {s->nodes.size() * sizeof(DevNode), s->geoms.size() * sizeof(DevGeom),
                                     s->shaders.size() * sizeof(DevShader), s->textures.size() * sizeof(DevTex)};
            for (int k = 0; k < 4; k++) CU(cudaMalloc(&s->d_records[i][k], std::max<size_t>(bytes[k], 16)));
        }
    }
    for (int i = 0; i < g_ctx.n; i++) {
        CU(cudaSetDevice(g_ctx.d[i].dev));
        if (!s->texels.empty()) {
            CU(cudaMalloc(&s->d_texels[i], s->texels.size() * sizeof(float4)));
            CU(cudaMemcpy(s->d_texels[i], s->texels.data(), s->texels.size() * sizeof(float4), cudaMemcpyHostToDevice));
        }
        if (!s->quads.empty()) {
            CU(cudaMalloc(&s->d_quads[i], s->quads.size() * sizeof(uint32_t)));
            CU(cudaMemcpy(s->d_quads[i], s->quads.data(), s->quads.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
            CU(cudaMalloc(&s->d_palettes[i], s->palettes.size() * sizeof(float4)));
            CU(cudaMemcpy(s->d_palettes[i], s->palettes.data(), s->palettes.size() * sizeof(float4), cudaMemcpyHostToDevice));
        }
    }
    return C2RT_OK;
}

// make `scene` the one resident in device slot `di`'s constant memory
int make_resident(c2rt_scene* s, int di, cudaStream_t st) {
    DeviceCtx& c = g_ctx.d[di];
    if (c.uploaded_scene == s->id) return C2RT_OK;
    // A device holds ONE scene block (constant memory).  Frames of the scene it replaces may still be running on other
    // streams of this device and read that block: wait for them before overwriting it.  (A scene switch therefore cannot
    // happen inside a stream capture; first use of a scene on a device must come before the capture: c2rt.h.)
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    CU(cudaStreamIsCapturing(st, &cap));
    if (cap != cudaStreamCaptureStatusNone)
        return fail(C2RT_ERR_INVALID_ARG, "the scene is not resident on this device yet: render it once outside the stream capture first");
    CU(cudaDeviceSynchronize());
    const int n_bmp_slots = s->host.n_textures + (s->host.env_type == C2RT_ENV_CUBEMAP ? 6 : 0);
    for (int t = 0; t < n_bmp_slots; t++) {
        DevTex& tx = t < s->host.n_textures ? s->textures[t] : s->host.env_faces[t - s->host.n_textures];
        const bool bmp = tx.type == C2RT_TEX_BITMAP, pal = bmp && s->quad_offset[t] >= 0;
        tx.texels = (bmp && !pal) ? s->d_texels[di] + s->tex_offset[t] : nullptr;
        tx.quads = pal ? s->d_quads[di] + s->quad_offset[t] : nullptr;
        tx.palette = pal ? s->d_palettes[di] + s->pal_offset[t] : nullptr;
    }
    if (s->big) {
        const void* src[4] = {s->nodes.data(), s->geoms.data(), s->shaders.data(), s->textures.data()};
        const size_t bytes[4] = {s->nodes.size() * sizeof(DevNode), s->geoms.size() * sizeof(DevGeom),
                                 s->shaders.size() * sizeof(DevShader), s->textures.size() * sizeof(DevTex)};
        for (int k = 0; k < 4; k++)
            if (bytes[k]) CU(cudaMemcpyAsync(s->d_records[di][k], src[k], bytes[k], cudaMemcpyHostToDevice, st));
        s->host.g_nodes = (const DevNode*)s->d_records[di][0];
        s->host.g_geoms = (const DevGeom*)s->d_records[di][1];
        s->host.g_shaders = (const DevShader*)s->d_records[di][2];
        s->host.g_textures = (const DevTex*)s->d_records[di][3];
    } else {
        if (!s->nodes.empty()) memcpy(s->host.nodes, s->nodes.data(), s->nodes.size() * sizeof(DevNode));
        if (!s->geoms.empty()) memcpy(s->host.geoms, s->geoms.data(), s->geoms.size() * sizeof(DevGeom));
        if (!s->shaders.empty()) memcpy(s->host.shaders, s->shaders.data(), s->shaders.size() * sizeof(DevShader));
        if (!s->textures.empty()) memcpy(s->host.textures, s->textures.data(), s->textures.size() * sizeof(DevTex));
    }
    CU(upload_scene(s->host, st));
    CU(cudaStreamSynchronize(st));  // the source is pageable host memory that the next device patches
    c.uploaded_scene = s->id;
    return C2RT_OK;
}

int check_frame_args(const c2rt_scene* s, const c2rt_camera* cam, const c2rt_settings* set) {
    if (!s || !cam || !set) return fail(C2RT_ERR_INVALID_ARG, "scene, camera and settings must be non-null");
    if (set->frame_width == 0 || set->frame_height == 0 || set->frame_width > 65536 || set->frame_height > 65536)
        return fail(C2RT_ERR_INVALID_ARG, "bad frame size %ux%u", set->frame_width, set->frame_height);
    if (cam->frame_width == 0 || cam->frame_height == 0) return fail(C2RT_ERR_INVALID_ARG, "camera frame size is zero (setFrameSize not called)");
    if (set->gi_enabled && !cam->dof)   // renderer.d:256-263: the DOF branch is tested first and ignores GIEnabled
        for (int i = 0; i < s->host.n_nodes; i++)
            if (s->shaders[s->nodes[i].shader].type == C2RT_SHADER_PHONG)
                return fail(C2RT_ERR_UNSUPPORTED, "GIEnabled with a Phong-shaded node: Phong.spawnRay / eval are assert(0) in the reference "
                                                  "(shader.d:252-262), it halts as soon as a path reaches that node");
    if (set->gi_enabled && !cam->dof && s->host.env_type != C2RT_ENV_BLACK)
        return fail(C2RT_ERR_UNSUPPORTED, "GIEnabled with a cubemap environment: GI frames are only built for the reference's black environment "
                                          "(every path is provably black there: DESIGN.md section 0, row f-4)");
    if (!std::isfinite(cam->stereo_separation)) return fail(C2RT_ERR_INVALID_ARG, "stereoSeparation is not finite");
    if (cam->dof && cam->num_samples == 0) return fail(C2RT_ERR_INVALID_ARG, "DOF camera with numSamples == 0");
    return C2RT_OK;
}

void fill_params(FrameParams& fp, const c2rt_camera* cam, const c2rt_settings* set, const c2rt_scene* s, int di) {
    memset(&fp, 0, sizeof fp);
    fp.bounds = s->d_bounds[di];
    for (int k = 0; k < 3; k++) {
        fp.pos[k] = cam->pos[k];
        fp.ul_rel[k] = cam->up_left[k] - cam->pos[k];
        fp.du[k] = cam->up_right[k] - cam->up_left[k];   // camera.d:141
        fp.dv[k] = cam->down_left[k] - cam->up_left[k];  // camera.d:142
        fp.right_dir[k] = cam->right_dir[k];
        fp.up_dir[k] = cam->up_dir[k];
        fp.front_dir[k] = cam->front_dir[k];
        fp.ambient[k] = set->ambient_light[k];
    }
    for (int k = 0; k < 3; k++) fp.posf[k] = (float)cam->pos[k];
    fp.posf_len = sqrtf(fp.posf[0] * fp.posf[0] + fp.posf[1] * fp.posf[1] + fp.posf[2] * fp.posf[2]);
    fp.inv_w = 1.0 / (double)cam->frame_width;
    fp.inv_h = 1.0 / (double)cam->frame_height;
    static const double kx[5] = {0.0, 0.3, 0.6, 0.0, 0.6}, ky[5] = {0.0, 0.3, 0.0, 0.6, 0.6};
    for (int t = 0; t < 5; t++)
        for (int k = 0; k < 3; k++) fp.tap_d[t][k] = fp.du[k] * (kx[t] * fp.inv_w) + fp.dv[k] * (ky[t] * fp.inv_h);
    fp.focal_plane_dist = cam->focal_plane_dist;
    fp.disc_multiplier = cam->disc_multiplier;
    fp.stereo_sep = cam->stereo_separation;
    fp.seed = set->rng_seed;
    fp.W = set->frame_width;
    fp.H = set->frame_height;
    fp.aa = set->aa_enabled != 0;
    fp.dof = cam->dof != 0;
    fp.num_samples = cam->num_samples;
    fp.count_rays = set->count_rays != 0;
    // GI frame (renderer.d:289-301,378-463): every path returns exactly black — PointLight.solidAngle is 0 (light.d:72-75) so
    // resultDirect is 0, lights cannot be hit, misses read the black environment — and the pixel is the mean of pathsPerPixel zeros
    fp.gi = set->gi_enabled && !cam->dof;
    fp.gi_fill = set->paths_per_pixel ? 0.f : nanf("");
    fp.prepass_bucket = set->prepass_only ? (set->bucket_size ? set->bucket_size : 48u) : 0u;
    if (s->mode & MODE_SOLO) {   // render_kernel.cu solo_plane_test
        const double y = s->nodes[0].wp[0], h = cam->pos[1] - y, ly = s->host.lights[0].pos[1];
        fp.solo_side = h > 0 ? 1 : h < 0 ? -1 : 0;
        fp.solo_sign = fp.solo_side > 0 ? 0x80000000u : 0u;
        fp.solo_h = h;
        // |d|^2 of the un-normalised pinhole direction is convex in the screen position: its maximum over the sampled rectangle
        // (pixel corners + the AA offsets + DOF's one-pixel jitter, one more pixel of margin) is at a corner; its minimum is at
        // least the squared distance of the screen's plane from the camera
        double dmax2 = 0.0;
        for (int c = 0; c < 4; c++) {
            const double sx = (c & 1) ? ((double)fp.W + 2.0) * fp.inv_w : -fp.inv_w, sy = (c & 2) ? ((double)fp.H + 2.0) * fp.inv_h : -fp.inv_h;
            double l2 = 0.0;
            for (int k = 0; k < 3; k++) { const double v = fp.ul_rel[k] + fp.du[k] * sx + fp.dv[k] * sy; l2 += v * v; }
            dmax2 = std::max(dmax2, l2);
        }
        const double n[3] = {fp.du[1] * fp.dv[2] - fp.du[2] * fp.dv[1], fp.du[2] * fp.dv[0] - fp.du[0] * fp.dv[2], fp.du[0] * fp.dv[1] - fp.du[1] * fp.dv[0]};
        const double nl = std::sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
        const double dmin = nl > 0 ? std::fabs(fp.ul_rel[0] * n[0] + fp.ul_rel[1] * n[1] + fp.ul_rel[2] * n[2]) / nl : 0.0;
        // DOF / stereo move the ray origin inside the lens: by at most `lens` in any direction, `lens_y` in height; a DOF ray
        // runs from there to the focal point, at most focalPlaneDist |d| / (d . front) from the camera position (camera.d:154-173)
        double lens = std::fabs(cam->stereo_separation), lens_y = std::fabs(cam->stereo_separation * cam->right_dir[1]);
        double front_min = 1e300;   // min over the corners of d . front (linear in the screen position)
        for (int c = 0; c < 4; c++) {
            const double sx = (c & 1) ? ((double)fp.W + 2.0) * fp.inv_w : -fp.inv_w, sy = (c & 2) ? ((double)fp.H + 2.0) * fp.inv_h : -fp.inv_h;
            double f = 0.0;
            for (int k = 0; k < 3; k++) f += (fp.ul_rel[k] + fp.du[k] * sx + fp.dv[k] * sy) * cam->front_dir[k];
            front_min = std::min(front_min, f);
        }
        double dray2 = dmax2;
        bool lens_ok = true;
        if (cam->dof) {
            const double dm = std::fabs(cam->disc_multiplier) * (1.0 + 1e-6);
            lens += 2.0 * dm;
            lens_y += dm * (std::fabs(cam->right_dir[1]) + std::fabs(cam->up_dir[1]));
            lens_ok = front_min > 1e-6 && std::isfinite(cam->focal_plane_dist);
            const double reach = lens_ok ? std::fabs(cam->focal_plane_dist) * std::sqrt(dmax2) / front_min + lens : 0.0;
            dray2 = reach * reach;
        }
        fp.graze_dy2 = 1e-18 * dray2 * (1.0 + 1e-6);
        // regular: the rounding of the hit point's y (|h| 1e-15 + an ulp of y) and of the shadow-ray origin cannot reach the
        // 1e-6 offset, the whole lens is on one side of the plane and the light on the same side by more than 1e-5, distances stay
        // far below 1e99; preview frames (prepassOnly: jitter over whole blocks) are left to the general path
        const double mag = std::fabs(h) + std::fabs(y) + std::fabs(cam->pos[1]) + std::fabs(ly) + lens;
        const char* no_fast = getenv("C2RT_NO_SOLO_FAST");   // test hook: every one-plane frame on the general path
        fp.solo_fast = fp.solo_side != 0 && lens_ok && std::isfinite(dray2) && std::isfinite(mag) && mag < 1e6 && dray2 < 1e12 &&
                       std::fabs(h) > lens_y + 1e-5 && (double)fp.solo_side * (ly - y) > 1e-5 && dmin > 1e-6 &&
                       !set->prepass_only && !(no_fast && no_fast[0] == '1');
        // d.y = fma(dv.y, sy, fma(du.y, sx, ul_rel.y)) + tap_d.y (render_kernel.cu screen_dir): with du.y = +-0 the inner fma is
        // the same value for every sx >= 0, so d.y is constant along a row.  Tested on the value the kernel uses, not on the
        // camera's roll: the corners reach the ABI from any host.
        fp.solo_rows = fp.solo_fast && fp.du[1] == 0.0;
        // the same for d.z = fma(dv.z, sy, fma(du.z, sx, ul_rel.z)) + tap_d.z: a camera without yaw or roll has du.z == 0
        fp.solo_zrows = fp.solo_rows && fp.du[2] == 0.0;
    }
}

// The band layout of a launch (c2rt.h c2rt_band: rows in bands of band_rows, band b on rank b % n_ranks; compact outputs hold
// only this rank's rows) and the device's ray counters and sRGB table
void set_bands(FrameParams& fp, const DeviceCtx& c, uint32_t rank, uint32_t n_ranks, uint32_t band_rows, bool compact) {
    fp.rank = rank;
    fp.n_ranks = n_ranks;
    fp.tiles_per_band = band_rows / TILE_H;
    fp.compact = compact;
    fp.counters = c.d_counters;
    fp.lut = c.d_lut;
}

// Reads a device's ray counters behind the work already on `st` (either output may be null) and zeroes them for the next
// frame.  The caller has made c.dev the current device.
int take_ray_counters(const DeviceCtx& c, cudaStream_t st, uint64_t* primary, uint64_t* shadow) {
    unsigned long long v[2];
    CU(cudaMemcpyAsync(v, c.d_counters, sizeof v, cudaMemcpyDeviceToHost, st));
    CU(cudaMemsetAsync(c.d_counters, 0, sizeof v, st));
    CU(cudaStreamSynchronize(st));
    if (primary) *primary = v[0];
    if (shadow) *shadow = v[1];
    return C2RT_OK;
}

// c2rt_cancel bookkeeping: true iff a cancel was requested since the last call; the device flags are lowered again
bool take_cancel_request() {
    if (!g_cancel_requested.exchange(false)) return false;
    for (int i = 0; i < g_ctx.n; i++) {
        DeviceCtx& c = g_ctx.d[i];
        cudaSetDevice(c.dev);
        cudaStreamSynchronize(c.cancel_stream);
        cudaMemset(c.d_cancel, 0, sizeof(int));
    }
    cudaSetDevice(g_ctx.d[0].dev);
    return true;
}

uint32_t local_tile_rows(uint32_t H, uint32_t rank, uint32_t n, uint32_t band_rows) {
    uint32_t rows = c2rt_band_rows_owned(H, rank, n, band_rows);
    return (rows + TILE_H - 1) / TILE_H;
}

// Rows per band of a c2rt_render frame on n devices, a whole number of tiles: device i renders bands i, i + n, i + 2n, ...
// Each band is one launch and one contiguous D2H copy per output plane, and its copy runs while the next band renders.
uint32_t frame_band_rows(int n, uint32_t H, uint32_t W) {
    const uint32_t tile_rows = (H + TILE_H - 1) / TILE_H;
    if (n == 1) {
        // up to 4 bands: the D2H copy of a float frame costs more than rendering it, so most of it should overlap
        const uint32_t bands = tile_rows >= 32 ? 4 : 1;
        return (tile_rows + bands - 1) / bands * TILE_H;
    }
    // 2..16 interleaved bands per device (one band per ~256k pixels): small frames must not be cut into many bands
    // (every launch / copy costs a few host microseconds)
    const uint32_t per_dev = (uint32_t)std::min<size_t>(16, std::max<size_t>(2, (size_t)W * H / (size_t)n / 262144));
    return std::max<uint32_t>(TILE_H, (H / ((uint32_t)n * per_dev) + TILE_H - 1) / TILE_H * TILE_H);
}

// Grows a device buffer to at least `elems` elements; its contents are not kept.
template <class T>
int grow_buffer(T*& buf, size_t& cap, size_t elems) {
    if (cap >= elems) return C2RT_OK;
    cudaFree(buf);
    buf = nullptr; cap = 0;
    CU(cudaMalloc(&buf, std::max<size_t>(elems, 1) * sizeof(T)));
    cap = elems;
    return C2RT_OK;
}

// c2rt_render_pixel and the hit frames refuse GI frames with one rule and one message
const char* const kGiPickMessage = "pixel pick on a GI frame: the reference's lastTracingResult is the last random path segment";

int check_hit_args(const c2rt_scene* s, const c2rt_camera* cam, const c2rt_settings* set, const c2rt_hit_planes* planes) {
    int rc = check_frame_args(s, cam, set);
    if (rc) return rc;
    if (!planes || (!planes->node && !planes->dist && !planes->normal && !planes->uv))
        return fail(C2RT_ERR_INVALID_ARG, "every hit plane is null");
    if (set->gi_enabled && !cam->dof) return fail(C2RT_ERR_UNSUPPORTED, kGiPickMessage);
    return C2RT_OK;
}

// Device slot i's share of an n-device frame: its bands (frame_band_rows) render into the slot's compact buffers, which hold
// only its own rows in order (the whole frame when n == 1), and each band is copied to its rows of the caller's host planes
// on copy_stream once its launch has finished.  A colour frame (c2rt_render: rgb, argb) or, with `hits`, a hit frame
// (c2rt_render_hits: its host planes).  Returns when the copies are complete.
int render_bands(int i, int n, c2rt_scene* s, const c2rt_camera* cam, const c2rt_settings* set, float* rgb, uint32_t* argb,
                 const c2rt_hit_planes* hits, uint32_t* launches_out, float* kernel_ms_out) {
    const uint32_t W = set->frame_width, H = set->frame_height;
    const uint32_t brows = frame_band_rows(n, H, W);
    DeviceCtx& c = g_ctx.d[i];
    CU(cudaSetDevice(c.dev));
    FrameParams fp;
    fill_params(fp, cam, set, s, i);
    set_bands(fp, c, (uint32_t)i, (uint32_t)n, brows, true);
    const size_t need = (size_t)c2rt_band_rows_owned(H, fp.rank, fp.n_ranks, brows) * W;
    // the output planes: host destination, device buffer, 4-byte words per pixel
    struct Plane {
        void* host;
        uint32_t* dev;
        uint32_t words;
    } planes[4] = {};
    c2rt_hit_planes d_hits = {};
    int rc = C2RT_OK;
    if (hits) {
        rc = grow_buffer(c.d_hits, c.hits_cap, need * 7);
        if (rc) return rc;
        planes[0] = {hits->node, c.d_hits, 1};
        planes[1] = {hits->dist, c.d_hits + need, 1};
        planes[2] = {hits->normal, c.d_hits + need * 2, 3};
        planes[3] = {hits->uv, c.d_hits + need * 5, 2};
        d_hits.node = hits->node ? (int32_t*)planes[0].dev : nullptr;
        d_hits.dist = hits->dist ? (float*)planes[1].dev : nullptr;
        d_hits.normal = hits->normal ? (float*)planes[2].dev : nullptr;
        d_hits.uv = hits->uv ? (float*)planes[3].dev : nullptr;
    } else {
        fp.cancel = c.d_cancel;
        rc = rgb ? grow_buffer(c.d_rgb, c.rgb_cap, need * 3) : C2RT_OK;
        if (rc == C2RT_OK && argb) rc = grow_buffer(c.d_argb, c.argb_cap, need);
        if (rc) return rc;
        fp.rgb = rgb ? c.d_rgb : nullptr;
        fp.argb = argb ? c.d_argb : nullptr;
        planes[0] = {rgb, (uint32_t*)c.d_rgb, 3};
        planes[1] = {argb, c.d_argb, 1};
    }
    CU(cudaEventRecord(c.e0, c.stream));
    uint32_t local_row = 0, b = 0;
    for (uint32_t y0 = (uint32_t)i * brows; y0 < H; y0 += (uint32_t)n * brows, b++) {
        const uint32_t rows = std::min<uint32_t>(brows, H - y0);
        if (b >= c.band_done.size()) {
            cudaEvent_t e;
            CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            c.band_done.push_back(e);
        }
        fp.tile_row0 = b * fp.tiles_per_band;
        const uint32_t tile_rows = (rows + TILE_H - 1) / TILE_H;
        if (hits) CU(launch_hits(fp, s->mode, tile_rows, d_hits, c.stream));
        else CU(launch_frame(fp, s->mode, tile_rows, c.stream));
        CU(cudaEventRecord(c.band_done[b], c.stream));
        CU(cudaStreamWaitEvent(c.copy_stream, c.band_done[b], 0));
        for (const Plane& p : planes)
            if (p.host)
                CU(cudaMemcpyAsync((uint32_t*)p.host + (size_t)y0 * W * p.words, p.dev + (size_t)local_row * W * p.words,
                                   (size_t)rows * W * p.words * sizeof(uint32_t), cudaMemcpyDeviceToHost, c.copy_stream));
        local_row += rows;
    }
    CU(cudaEventRecord(c.e1, c.stream));
    CU(cudaStreamSynchronize(c.copy_stream));
    CU(cudaEventSynchronize(c.e1));
    CU(cudaEventElapsedTime(kernel_ms_out, c.e0, c.e1));
    *launches_out = b;   // one launch per band
    return C2RT_OK;
}

}  // namespace

extern "C" {

int c2rt_abi_version(void) { return C2RT_ABI_VERSION; }

const char* c2rt_last_error(void) { return g_err.c_str(); }

int c2rt_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int c2rt_init(int n_gpus, const int* device_ids) {
    std::lock_guard<std::mutex> g(g_mu);
    return init_locked(n_gpus, device_ids);
}

void c2rt_shutdown(void) {
    std::lock_guard<std::mutex> g(g_mu);
    g_pool.stop();
    for (int i = 0; i < g_ctx.n; i++) destroy_device(g_ctx.d[i]);
    g_ctx.n = 0;
    g_ctx.inited = false;
}

uint32_t c2rt_band_rows_owned(uint32_t height, uint32_t rank, uint32_t n_ranks, uint32_t band_rows) {
    if (n_ranks == 0 || band_rows == 0) return 0;
    uint32_t rows = 0;
    for (uint32_t y0 = rank * band_rows; y0 < height; y0 += n_ranks * band_rows) rows += (height - y0 < band_rows) ? height - y0 : band_rows;
    return rows;
}

uint32_t c2rt_rng_u31(uint64_t seed, uint32_t px, uint32_t py, uint32_t tap, uint32_t sample, uint32_t draw) {
    return rng_u31(seed, px, py, tap, sample, draw);   // the kernel's generator (scene_dev.h)
}

void c2rt_srgb_table(uint8_t out[4097]) {
    for (int i = 0; i < 4097; i++) out[i] = srgb8((float)i / 4096.f);
}

int c2rt_scene_create(const c2rt_scene_desc* desc, c2rt_scene** out) {
    if (!out) return fail(C2RT_ERR_INVALID_ARG, "out is null");
    *out = nullptr;
    std::lock_guard<std::mutex> g(g_mu);
    c2rt_scene* s = new c2rt_scene();
    int rc = validate_and_build(desc, s);
    if (rc == C2RT_OK) rc = ensure_init_locked();
    if (rc == C2RT_OK) {
        s->id = g_ctx.next_scene_id++;
        rc = upload_to_devices(s);
    }
    if (rc != C2RT_OK) {
        delete s;
        return rc;
    }
    *out = s;
    return C2RT_OK;
}

void c2rt_scene_destroy(c2rt_scene* s) {
    if (!s) return;
    std::lock_guard<std::mutex> g(g_mu);
    for (int i = 0; i < s->n_dev && i < g_ctx.n; i++) {
        if (s->d_texels[i] || s->d_bounds[i] || s->d_quads[i]) {
            cudaSetDevice(g_ctx.d[i].dev);
            cudaFree(s->d_texels[i]);
            cudaFree(s->d_bounds[i]);
            cudaFree(s->d_quads[i]);
            cudaFree(s->d_palettes[i]);
            for (int k = 0; k < 4; k++) cudaFree(s->d_records[i][k]);
        }
        if (g_ctx.d[i].uploaded_scene == s->id) g_ctx.d[i].uploaded_scene = 0;
    }
    delete s;
}

int c2rt_render_device(c2rt_scene* s, const c2rt_camera* cam, const c2rt_settings* set, const c2rt_band* band, float* d_rgb,
                       uint32_t* d_argb, void* stream, c2rt_stats* stats) {
    int rc = check_frame_args(s, cam, set);
    if (rc) return rc;
    if (!d_rgb) return fail(C2RT_ERR_INVALID_ARG, "d_rgb is null");
    if (set->prepass_only && !set->prepass_enabled) return C2RT_OK;  // renderer.d:110,129-130: nothing is drawn
    std::lock_guard<std::mutex> g(g_mu);
    if (!g_ctx.inited) return fail(C2RT_ERR_NOT_INITIALISED, "c2rt_init has not been called");
    int dev = -1;
    CU(cudaGetDevice(&dev));
    DeviceCtx* c = find_device(dev);
    if (!c) return fail(C2RT_ERR_INVALID_ARG, "current device %d is not part of the c2rt context", dev);
    int di = (int)(c - g_ctx.d);
    if (di >= s->n_dev) return fail(C2RT_ERR_INVALID_ARG, "scene was created under a different c2rt_init configuration");
    cudaStream_t st = (cudaStream_t)stream;
    rc = make_resident(s, di, st);
    if (rc) return rc;
    const c2rt_band whole = {0, 1, TILE_H, 0, nullptr, 0, 0};   // no band: the whole frame on one rank
    const c2rt_band& b = band ? *band : whole;
    if (b.n_ranks == 0 || b.rank >= b.n_ranks || b.band_rows == 0 || b.band_rows % TILE_H != 0)
        return fail(C2RT_ERR_INVALID_ARG, "bad band (rank %u of %u, band_rows %u; band_rows must be a multiple of %d)", b.rank,
                    b.n_ranks, b.band_rows, TILE_H);
    FrameParams fp;
    fill_params(fp, cam, set, s, di);
    set_bands(fp, *c, b.rank, b.n_ranks, b.band_rows, b.compact != 0);
    if (b.done_flags) {
        if (b.n_ranks > 32) return fail(C2RT_ERR_INVALID_ARG, "done_flags: at most 32 ranks");
        fp.frame_no = b.frame_no;
        if (b.rank == 0) {   // rank 0 waits inside its kernel; peers signal behind theirs (below)
            fp.done_flags = (uint32_t*)b.done_flags;
            fp.done_counter = c->d_done_counter;
        }
    }
    if (((uintptr_t)d_rgb & 15u) && (fp.W & 3u) == 0)
        return fail(C2RT_ERR_INVALID_ARG, "d_rgb must be 16-byte aligned when the frame width is a multiple of 4 (float4 band stores)");
    fp.rgb = d_rgb;
    fp.argb = d_argb;
    CU(launch_frame(fp, s->mode, local_tile_rows(fp.H, b.rank, b.n_ranks, b.band_rows), st));
    const bool signals = b.done_flags && b.rank != 0;
    if (signals) CU(launch_signal((uint32_t*)b.done_flags + b.rank, b.frame_no, st));
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->n_gpus = 1;
        stats->launches = signals ? 2 : 1;
    }
    return C2RT_OK;
}

int c2rt_read_ray_counters(c2rt_scene*, void* stream, uint64_t* primary, uint64_t* shadow) {
    std::lock_guard<std::mutex> g(g_mu);
    if (!g_ctx.inited) return fail(C2RT_ERR_NOT_INITIALISED, "c2rt_init has not been called");
    int dev = -1;
    CU(cudaGetDevice(&dev));
    DeviceCtx* c = find_device(dev);
    if (!c) return fail(C2RT_ERR_INVALID_ARG, "current device %d is not part of the c2rt context", dev);
    return take_ray_counters(*c, (cudaStream_t)stream, primary, shadow);
}

int c2rt_render(c2rt_scene* s, const c2rt_camera* cam, const c2rt_settings* set, float* rgb, uint32_t* argb, c2rt_stats* stats) {
    auto t0 = std::chrono::steady_clock::now();
    int rc = check_frame_args(s, cam, set);
    if (rc) return rc;
    if (!rgb && !argb) return fail(C2RT_ERR_INVALID_ARG, "rgb and argb are both null");
    if (set->prepass_only && !set->prepass_enabled) {  // renderer.d:110,129-130: nothing is drawn, the image keeps its contents
        if (stats) memset(stats, 0, sizeof *stats);
        return C2RT_OK;
    }
    std::lock_guard<std::mutex> g(g_mu);
    rc = ensure_init_locked();
    if (rc) return rc;
    if (s->n_dev != g_ctx.n) return fail(C2RT_ERR_INVALID_ARG, "scene was created under a different c2rt_init configuration");
    take_cancel_request();   // a cancel that arrived while no frame was in progress cancels nothing
    const int n = g_ctx.n;
    // scene residency first, on this thread: make_resident patches the shared host copy of the scene block per device
    for (int i = 0; i < n; i++) {
        if (g_ctx.d[i].uploaded_scene == s->id) continue;
        CU(cudaSetDevice(g_ctx.d[i].dev));
        rc = make_resident(s, i, g_ctx.d[i].stream);
        if (rc) return rc;
    }
    // Every device renders its bands and copies them to the host frame over its own PCIe link: the host copy of a float
    // frame is the slow part, so N links beat one.  Worker w of the pool drives device w + 1, this thread drives device 0.
    int rcs[C2RT_MAX_GPUS] = {};
    uint32_t ls[C2RT_MAX_GPUS] = {};
    float kms[C2RT_MAX_GPUS] = {};
    std::string errs[C2RT_MAX_GPUS];
    if (n > 1)
        g_pool.run([&](int w) {
            rcs[w + 1] = render_bands(w + 1, n, s, cam, set, rgb, argb, nullptr, &ls[w + 1], &kms[w + 1]);
            if (rcs[w + 1]) errs[w + 1] = g_err;
        });
    rcs[0] = render_bands(0, n, s, cam, set, rgb, argb, nullptr, &ls[0], &kms[0]);
    if (rcs[0]) errs[0] = g_err;
    if (n > 1) g_pool.wait();
    uint32_t launches = 0;
    double kernel_ms = 0;
    for (int i = 0; i < n; i++) {
        if (rcs[i]) { g_err = errs[i]; return rcs[i]; }
        launches += ls[i];
        if (kms[i] > kernel_ms) kernel_ms = kms[i];
    }
    CU(cudaSetDevice(g_ctx.d[0].dev));
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->kernel_ms = kernel_ms;
        stats->n_gpus = (uint32_t)n;
        stats->launches = launches;
        if (set->count_rays) {
            for (int i = 0; i < n; i++) {
                DeviceCtx& c = g_ctx.d[i];
                CU(cudaSetDevice(c.dev));
                uint64_t p, sh;
                rc = take_ray_counters(c, c.stream, &p, &sh);
                if (rc) return rc;
                stats->primary_rays += p;
                stats->shadow_rays += sh;
            }
            CU(cudaSetDevice(g_ctx.d[0].dev));
        }
        stats->total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
    if (take_cancel_request()) {
        g_err = "frame cancelled by c2rt_cancel: the output holds the tiles rendered before the request";
        return C2RT_CANCELLED;
    }
    return C2RT_OK;
}

int c2rt_cancel(void) {
    // no lock: c2rt_render holds the library mutex for the whole frame, and this must get through while it runs
    if (!g_ctx.inited) return fail(C2RT_ERR_NOT_INITIALISED, "c2rt_init has not been called");
    g_cancel_requested.store(true);
    static const int one = 1;
    int prev = -1;
    cudaGetDevice(&prev);
    for (int i = 0; i < g_ctx.n; i++) {
        const DeviceCtx& c = g_ctx.d[i];
        cudaSetDevice(c.dev);
        cudaMemcpyAsync(c.d_cancel, &one, sizeof(int), cudaMemcpyHostToDevice, c.cancel_stream);
    }
    if (prev >= 0) cudaSetDevice(prev);
    cudaGetLastError();
    return C2RT_OK;
}

int c2rt_render_pixel(c2rt_scene* s, const c2rt_camera* cam, const c2rt_settings* set, int x, int y, float rgb[3], c2rt_hit* hit) {
    int rc = check_frame_args(s, cam, set);
    if (rc) return rc;
    if (!rgb) return fail(C2RT_ERR_INVALID_ARG, "rgb is null");
    if (set->gi_enabled && !cam->dof) return fail(C2RT_ERR_UNSUPPORTED, kGiPickMessage);
    if (x < 0 || y < 0 || (uint32_t)x >= set->frame_width || (uint32_t)y >= set->frame_height)
        return fail(C2RT_ERR_INVALID_ARG, "pixel (%d,%d) outside the %ux%u frame", x, y, set->frame_width, set->frame_height);
    std::lock_guard<std::mutex> g(g_mu);
    rc = ensure_init_locked();
    if (rc) return rc;
    DeviceCtx& c = g_ctx.d[0];
    CU(cudaSetDevice(c.dev));
    rc = make_resident(s, 0, c.stream);
    if (rc) return rc;
    FrameParams fp;
    fill_params(fp, cam, set, s, 0);
    set_bands(fp, c, 0, 1, TILE_H, false);
    fp.count_rays = 0;
    CU(launch_pixel(fp, s->mode, x, y, c.d_pixel, c.stream));
    PixelOut o;
    CU(cudaMemcpyAsync(&o, c.d_pixel, sizeof o, cudaMemcpyDeviceToHost, c.stream));
    CU(cudaStreamSynchronize(c.stream));
    rgb[0] = o.rgb[0]; rgb[1] = o.rgb[1]; rgb[2] = o.rgb[2];
    if (hit) {
        memset(hit, 0, sizeof *hit);
        hit->node = o.node;
        hit->dist = o.dist;
        for (int k = 0; k < 3; k++) { hit->p[k] = o.p[k]; hit->normal[k] = o.n[k]; }
        hit->u = o.u; hit->v = o.v;
    }
    return C2RT_OK;
}

int c2rt_render_hits(c2rt_scene* s, const c2rt_camera* cam, const c2rt_settings* set, const c2rt_hit_planes* planes, c2rt_stats* stats) {
    auto t0 = std::chrono::steady_clock::now();
    int rc = check_hit_args(s, cam, set, planes);
    if (rc) return rc;
    std::lock_guard<std::mutex> g(g_mu);
    rc = ensure_init_locked();
    if (rc) return rc;
    if (s->n_dev != g_ctx.n) return fail(C2RT_ERR_INVALID_ARG, "scene was created under a different c2rt_init configuration");
    const int n = g_ctx.n;
    for (int i = 0; i < n; i++) {   // (as in c2rt_render: residency first, on this thread)
        if (g_ctx.d[i].uploaded_scene == s->id) continue;
        CU(cudaSetDevice(g_ctx.d[i].dev));
        rc = make_resident(s, i, g_ctx.d[i].stream);
        if (rc) return rc;
    }
    int rcs[C2RT_MAX_GPUS] = {};
    uint32_t ls[C2RT_MAX_GPUS] = {};
    float kms[C2RT_MAX_GPUS] = {};
    std::string errs[C2RT_MAX_GPUS];
    if (n > 1)
        g_pool.run([&](int w) {
            rcs[w + 1] = render_bands(w + 1, n, s, cam, set, nullptr, nullptr, planes, &ls[w + 1], &kms[w + 1]);
            if (rcs[w + 1]) errs[w + 1] = g_err;
        });
    rcs[0] = render_bands(0, n, s, cam, set, nullptr, nullptr, planes, &ls[0], &kms[0]);
    if (rcs[0]) errs[0] = g_err;
    if (n > 1) g_pool.wait();
    uint32_t launches = 0;
    double kernel_ms = 0;
    for (int i = 0; i < n; i++) {
        if (rcs[i]) { g_err = errs[i]; return rcs[i]; }
        launches += ls[i];
        if (kms[i] > kernel_ms) kernel_ms = kms[i];
    }
    CU(cudaSetDevice(g_ctx.d[0].dev));
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->kernel_ms = kernel_ms;
        stats->n_gpus = (uint32_t)n;
        stats->launches = launches;
        stats->total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
    return C2RT_OK;
}

int c2rt_render_hits_device(c2rt_scene* s, const c2rt_camera* cam, const c2rt_settings* set, const c2rt_band* band,
                            const c2rt_hit_planes* planes, void* stream, c2rt_stats* stats) {
    int rc = check_hit_args(s, cam, set, planes);
    if (rc) return rc;
    if (band && band->done_flags) return fail(C2RT_ERR_INVALID_ARG, "hit frames have no frame-complete signalling: done_flags must be null");
    std::lock_guard<std::mutex> g(g_mu);
    if (!g_ctx.inited) return fail(C2RT_ERR_NOT_INITIALISED, "c2rt_init has not been called");
    int dev = -1;
    CU(cudaGetDevice(&dev));
    DeviceCtx* c = find_device(dev);
    if (!c) return fail(C2RT_ERR_INVALID_ARG, "current device %d is not part of the c2rt context", dev);
    int di = (int)(c - g_ctx.d);
    if (di >= s->n_dev) return fail(C2RT_ERR_INVALID_ARG, "scene was created under a different c2rt_init configuration");
    cudaStream_t st = (cudaStream_t)stream;
    rc = make_resident(s, di, st);
    if (rc) return rc;
    const c2rt_band whole = {0, 1, TILE_H, 0, nullptr, 0, 0};   // no band: the whole frame on one rank
    const c2rt_band& b = band ? *band : whole;
    if (b.n_ranks == 0 || b.rank >= b.n_ranks || b.band_rows == 0 || b.band_rows % TILE_H != 0)
        return fail(C2RT_ERR_INVALID_ARG, "bad band (rank %u of %u, band_rows %u; band_rows must be a multiple of %d)", b.rank,
                    b.n_ranks, b.band_rows, TILE_H);
    FrameParams fp;
    fill_params(fp, cam, set, s, di);
    set_bands(fp, *c, b.rank, b.n_ranks, b.band_rows, b.compact != 0);
    CU(launch_hits(fp, s->mode, local_tile_rows(fp.H, b.rank, b.n_ranks, b.band_rows), *planes, st));
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->n_gpus = 1;
        stats->launches = 1;
    }
    return C2RT_OK;
}

int c2rt_deinterleave(const void* gathered, void* frame, uint32_t width, uint32_t height, uint32_t elem_words, uint32_t n_ranks,
                      uint32_t band_rows, uint32_t rows_pad, void* stream) {
    if (!gathered || !frame || !width || !height || !elem_words || !n_ranks || !band_rows)
        return fail(C2RT_ERR_INVALID_ARG, "bad deinterleave arguments");
    CU(launch_deinterleave(gathered, frame, width * elem_words, height, n_ranks, band_rows, rows_pad, (cudaStream_t)stream));
    return C2RT_OK;
}

int c2rt_frame_alloc(size_t bytes, void** d_ptr) {
    if (!d_ptr || !bytes) return fail(C2RT_ERR_INVALID_ARG, "bad frame_alloc arguments");
    CU(cudaMalloc(d_ptr, bytes));
    CU(cudaMemset(*d_ptr, 0, bytes));
    return C2RT_OK;
}
int c2rt_frame_free(void* d_ptr) {
    CU(cudaFree(d_ptr));
    return C2RT_OK;
}
int c2rt_frame_export(void* d_ptr, uint8_t handle[64]) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, d_ptr));
    memcpy(handle, &h, 64);
    return C2RT_OK;
}
int c2rt_frame_import(const uint8_t handle[64], void** d_ptr) {
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    CU(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return C2RT_OK;
}
int c2rt_frame_unimport(void* d_ptr) {
    CU(cudaIpcCloseMemHandle(d_ptr));
    return C2RT_OK;
}

int c2rt_frame_memset(void* d_ptr, int byte_value, size_t bytes, void* stream) {
    if (!d_ptr) return fail(C2RT_ERR_INVALID_ARG, "bad frame_memset arguments");
    CU(cudaMemsetAsync(d_ptr, byte_value, bytes, (cudaStream_t)stream));
    return C2RT_OK;
}

int c2rt_frame_download(void* host_dst, const void* d_src, size_t bytes, void* stream) {
    if (!host_dst || !d_src) return fail(C2RT_ERR_INVALID_ARG, "bad frame_download arguments");
    CU(cudaMemcpyAsync(host_dst, d_src, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return C2RT_OK;
}

int c2rt_gate(void* d_flags, uint32_t n_ranks, uint32_t round, void* stream) {
    if (!d_flags || n_ranks < 1 || n_ranks > 32 || round == 0) return fail(C2RT_ERR_INVALID_ARG, "bad gate arguments");
    uint32_t* flags = (uint32_t*)d_flags;
    CU(launch_gate(flags, round, n_ranks, flags + n_ranks, (cudaStream_t)stream));
    return C2RT_OK;
}

int c2rt_pin_host_buffer(void* ptr, size_t bytes) {
    if (!ptr || !bytes) return fail(C2RT_ERR_INVALID_ARG, "bad pin_host_buffer arguments");
    cudaError_t e = cudaHostRegister(ptr, bytes, cudaHostRegisterPortable);
    if (e == cudaErrorHostMemoryAlreadyRegistered) {
        cudaGetLastError();
        return C2RT_OK;
    }
    if (e != cudaSuccess) return fail(C2RT_ERR_CUDA, "cudaHostRegister failed: %s", cudaGetErrorString(e));
    return C2RT_OK;
}
int c2rt_unpin_host_buffer(void* ptr) {
    if (!ptr) return fail(C2RT_ERR_INVALID_ARG, "bad unpin_host_buffer argument");
    cudaError_t e = cudaHostUnregister(ptr);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(C2RT_ERR_CUDA, "cudaHostUnregister failed: %s", cudaGetErrorString(e));
    }
    return C2RT_OK;
}

long long c2rt_selftest_device_pool(int workers, int rounds) {
    if (workers < 1 || workers > 64 || rounds < 1) return -1;
    DevicePool pool;   // a private pool: the library's own one is left alone
    std::vector<std::atomic<long long>> hits(workers);
    for (auto& h : hits) h.store(0);
    long long total = 0;
    for (int phase = 0; phase < 2; phase++) {   // phase 1 runs on a restarted pool
        pool.start(workers);
        for (int r = 0; r < rounds; r++) {
            pool.run([&](int w) { hits[w].fetch_add(1, std::memory_order_relaxed); });
            pool.wait();
            // every so often let the workers fall asleep, so the condition-variable hand-off is taken too
            if (r % 97 == 96) std::this_thread::sleep_for(std::chrono::milliseconds(3));
        }
        pool.stop();
    }
    for (auto& h : hits) {
        if (h.load() != 2LL * rounds) return -2;   // a lost or duplicated round on some worker
        total += h.load();
    }
    return total / 2;
}

int c2rt_measure_fma_peak(int fp64, double* tflops, double* sm_clock_mhz_est) {
    if (!tflops) return fail(C2RT_ERR_INVALID_ARG, "tflops is null");
    int dev = 0;
    CU(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, dev));
    void* d_out = nullptr;
    CU(cudaMalloc(&d_out, 64));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    const int threads = 512, blocks = prop.multiProcessorCount * 4, iters = fp64 ? 2048 : 8192;
    CU(launch_fma_peak(fp64 != 0, blocks, threads, 64, d_out, 0));  // warm-up
    CU(cudaDeviceSynchronize());
    double best = 0;
    for (int rep = 0; rep < 5; rep++) {
        CU(cudaEventRecord(e0, 0));
        CU(launch_fma_peak(fp64 != 0, blocks, threads, iters, d_out, 0));
        CU(cudaEventRecord(e1, 0));
        CU(cudaEventSynchronize(e1));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, e0, e1));
        double flops = 2.0 * 64.0 * (double)iters * threads * (double)blocks;
        double tf = flops / (ms * 1e-3) / 1e12;
        if (tf > best) best = tf;
    }
    *tflops = best;
    if (sm_clock_mhz_est) {
        // lanes per SM per clock: 128 FP32, 64 FP64 on sm_100
        double lanes = fp64 ? 64.0 : 128.0;
        *sm_clock_mhz_est = best * 1e12 / (2.0 * lanes * prop.multiProcessorCount) / 1e6;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d_out);
    return C2RT_OK;
}

}  // extern "C"
