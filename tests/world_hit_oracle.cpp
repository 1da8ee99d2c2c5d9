// world_hit_oracle.cpp — the CPU reference of rt_world_hit (test infrastructure, like oracle/oracle.cpp).
//
// It is built from the oracle itself (this file includes oracle/oracle.cpp and adds one entry point), so every hit test,
// Transform, BVH box, interval, ConstantMedium::hit and Philox draw is the oracle's own code and arithmetic.
// tests/world_hit_oracle.py compiles it into a temporary directory with the oracle's flags.
//
// For ray k the record is what the oracle's world.hit(r, Interval(t_min, t_max_k)) returns, media enabled, with the path
// context (seed, pixel = k, sample = 0, segment): every ConstantMedium m takes its free-flight draw from
// philox(seed; k, 0, segment, RT_MEDIUM_SLOT(m)).  An empty interval (t_max_k < t_min, or a NaN bound) is a miss that is
// never traced.
#include "../oracle/oracle.cpp"

#include <unordered_map>

extern "C" {

// out[k] for rays[k], t_max_k = t_max_per_ray ? t_max_per_ray[k] : t_max (see the top of the file)
int orc_world_hit(const void* s, const rt_ray* rays, const double* t_max_per_ray, uint64_t n, double t_min, double t_max, uint64_t seed,
                  uint32_t segment, rt_hit_record* out) {
    using namespace orc;
    const Scene* sc = (const Scene*)s;
    std::unordered_map<const Material*, uint32_t> material_index;  // HitRecord::mat back to its materials[] index
    for (size_t m = 0; m < sc->materials.size(); m++) material_index.emplace(sc->materials[m].get(), (uint32_t)m);
#pragma omp parallel for schedule(dynamic, 256)
    for (int64_t k = 0; k < (int64_t)n; k++) {
        rt_hit_record h;
        std::memset(&h, 0, sizeof(h));
        h.t = INF;
        h.kind = RT_HIT_MISS;
        h.prim_id = h.inst_id = h.material = RT_NONE;
        const double t_max_k = t_max_per_ray ? t_max_per_ray[k] : t_max;
        if (t_min <= t_max_k) {
            PathCtx ctx;
            ctx.seed = seed, ctx.pixel = (uint32_t)k, ctx.sample = 0, ctx.segment = segment;
            ctx.media_enabled = true;
            Ray r(Vec3(rays[k].origin), Vec3(rays[k].direction), rays[k].time);
            HitRecord rec;
            if (sc->world->hit(r, Interval::raw(t_min, t_max_k), ctx, rec)) {
                h.t = rec.t;
                for (int c = 0; c < 3; c++) h.p[c] = rec.p[c], h.normal[c] = rec.normal[c];
                h.u = rec.u, h.v = rec.v;
                h.front_face = rec.front_face ? 1u : 0u;
                h.prim_id = rec.prim_id, h.inst_id = rec.inst_id;
                h.kind = dynamic_cast<const ConstantMedium*>(sc->by_object[rec.prim_id]) ? RT_HIT_MEDIUM : RT_HIT_SURFACE;
                h.material = material_index.at(rec.mat);
            }
        }
        out[k] = h;
    }
    return 0;
}

}  // extern "C"
