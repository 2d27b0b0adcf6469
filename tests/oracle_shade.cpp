// TEST INFRASTRUCTURE: the CPU oracle's `trace` on caller-supplied rays, for tests/test_gpu_shade.py, which compiles this file
// together with tests/oracle_rays.cpp (scene loading: orr_scene_load / orr_scene_free) against the oracle's headers (oracle/)
// into a temporary library.  The oracle itself is left as it is.
//   orr_shade_rays  Renderer::trace(ray) (renderer.d:325-376) on (origin, normalize(dir)), depth 0
// Each query also reports how close its camera hit and its shadow segments came to a tie, so that the tests can set aside
// ill-conditioned queries rather than loosen their comparison.
#include "orc_loader.hpp"
#include "orc_render.hpp"

using namespace orc;

namespace {
Vec3 vec(const double* p) { return Vec3(mk_real(p[0]), mk_real(p[1]), mk_real(p[2])); }
}  // namespace

extern "C" {

// out[4 i ..]: r, g, b, gap.  gap: the smallest relative gap between the camera hit's distance and another node's hit on the ray,
// or between a lit light's distance and an occluder candidate on the shadow segment from the hit (p + N 1e-6, as the shaders
// start it) to that light (1e300: none).  Ties inside a CSG or at texture cell edges are not counted: the colour there is the
// reference's own discontinuity, and the comparison keeps those queries.
void orr_shade_rays(void* sp, size_t n, const double* o, const double* d, double* out) {
    const Scene& sc = *static_cast<const Scene*>(sp);
    const Renderer r(sc, nullptr);
    for (size_t i = 0; i < n; i++) {
        Ray ray;
        ray.orig = vec(o + 3 * i);
        ray.dir = vec(d + 3 * i);
        normalize(ray.dir);
        const Color c = r.trace(ray);
        double gap = 1e300;
        IntersectionData data;
        data.dist = mk_real(1e99);
        int closest = -1;
        for (size_t k = 0; k < sc.nodes.size(); k++)
            if (sc.nodes[k]->intersect(ray, data)) closest = (int)k;
        if (closest >= 0) {
            const double d1 = raw(data.dist);
            for (size_t k = 0; k < sc.nodes.size(); k++) {
                IntersectionData probe;
                probe.dist = mk_real(1e99);
                if ((int)k != closest && sc.nodes[k]->intersect(ray, probe))
                    gap = std::min(gap, std::fabs(raw(probe.dist) - d1) / std::max(1.0, std::fabs(d1)));
            }
            const Vec3 from = data.p + faceforward(ray.dir, data.normal) * mk_real(1e-6);
            for (auto& light : sc.lights) {
                Vec3 lp;
                Color lc;
                light->getNthSample(0, data.p, lp, lc);
                if (raw(lc.intensity()) == 0) continue;
                Ray sr;
                sr.orig = from;
                sr.dir = lp - from;
                normalize(sr.dir);
                const double maxd = raw(length(lp - from));
                for (auto& node : sc.nodes) {
                    IntersectionData probe;
                    probe.dist = mk_real(1e99);
                    if (node->intersect(sr, probe)) gap = std::min(gap, std::fabs(raw(probe.dist) - maxd) / std::max(1.0, maxd));
                }
            }
        }
        double* q = out + 4 * i;
        q[0] = raw(c.r); q[1] = raw(c.g); q[2] = raw(c.b);
        q[3] = gap;
    }
}

}  // extern "C"
