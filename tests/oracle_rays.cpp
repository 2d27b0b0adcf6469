// TEST INFRASTRUCTURE: the CPU oracle's two scene queries on caller-supplied rays, for tests/test_gpu_rays.py, which compiles
// this file against the oracle's headers (oracle/) into a temporary library.  The oracle itself is left as it is.
//   orr_trace_rays       the closest-hit loop of renderPixel / trace (renderer.d:325-376) on (origin, normalize(dir))
//   orr_test_visibility  Scene::testVisibility(from, to) (scene.d:62-78)
// Each query also reports how close its answer came to a tie (the Diag probe of orc_scene.hpp), so that the tests can set
// aside ill-conditioned queries rather than loosen their comparison.
#include "orc_loader.hpp"
#include "orc_render.hpp"

using namespace orc;

namespace {
Vec3 vec(const double* p) { return Vec3(mk_real(p[0]), mk_real(p[1]), mk_real(p[2])); }
thread_local std::string g_err;
}  // namespace

extern "C" {

const char* orr_last_error(void) { return g_err.c_str(); }

void* orr_scene_load(const char* path) {
    try {
        std::unique_ptr<Scene> s = parseSceneFromFile(path);
        s->beginFrame();
        return s.release();
    } catch (const std::exception& e) {
        g_err = e.what();
        return nullptr;
    }
}

void orr_scene_free(void* s) { delete static_cast<Scene*>(s); }

// out[11 i ..]: node (-1 = miss), dist, p[3], normal[3], u, v, gap.  gap: the smallest relative gap between the winning
// distance and another node's hit distance, or between two CSG crossings met on the way (1e300: none).
void orr_trace_rays(void* sp, size_t n, const double* o, const double* d, double* out) {
    const Scene& sc = *static_cast<const Scene*>(sp);
    for (size_t i = 0; i < n; i++) {
        Ray ray;
        ray.orig = vec(o + 3 * i);
        ray.dir = vec(d + 3 * i);
        normalize(ray.dir);
        Diag& dg = tl_diag();
        dg = Diag();
        dg.on = true;
        IntersectionData data;
        data.dist = mk_real(1e99);
        int closest = -1;
        for (size_t k = 0; k < sc.nodes.size(); k++)
            if (sc.nodes[k]->intersect(ray, data)) closest = (int)k;
        if (closest >= 0) {
            const double d1 = raw(data.dist);
            for (size_t k = 0; k < sc.nodes.size(); k++) {
                if ((int)k == closest) continue;
                IntersectionData probe;
                probe.dist = mk_real(1e99);
                if (sc.nodes[k]->intersect(ray, probe)) dg.gap(std::fabs(raw(probe.dist) - d1) / std::max(1.0, std::fabs(d1)));
            }
        }
        dg.on = false;
        double* r = out + 11 * i;
        r[0] = closest;
        r[1] = raw(data.dist);
        r[2] = raw(data.p.x); r[3] = raw(data.p.y); r[4] = raw(data.p.z);
        r[5] = raw(data.normal.x); r[6] = raw(data.normal.y); r[7] = raw(data.normal.z);
        r[8] = raw(data.u); r[9] = raw(data.v);
        r[10] = dg.min_gap;
    }
}

// out[2 i ..]: visible (1 / 0), gap: the smallest distance of a candidate occluder from either end of the segment, or gap
// between two CSG crossings, relative to max(1, |to - from|) (1e300: none).
void orr_test_visibility(void* sp, size_t n, const double* from, const double* to, double* out) {
    const Scene& sc = *static_cast<const Scene*>(sp);
    for (size_t i = 0; i < n; i++) {
        const Vec3 f = vec(from + 3 * i), t = vec(to + 3 * i);
        Diag& dg = tl_diag();
        dg = Diag();
        dg.on = true;   // testVisibility probes every node against the far end
        const bool visible = sc.testVisibility(f, t);
        Ray ray;   // the near end
        ray.orig = f;
        ray.dir = t - f;
        normalize(ray.dir);
        const double maxd = raw(length(t - f));
        for (auto& node : sc.nodes) {
            IntersectionData probe;
            probe.dist = mk_real(1e99);
            if (node->intersect(ray, probe)) dg.gap(std::fabs(raw(probe.dist)) / std::max(1.0, maxd));
        }
        dg.on = false;
        out[2 * i] = visible ? 1.0 : 0.0;
        out[2 * i + 1] = dg.min_gap;
    }
}

}  // extern "C"
