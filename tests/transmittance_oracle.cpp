// transmittance_oracle.cpp — the CPU reference of rt_transmittance (test infrastructure, like oracle/oracle.cpp).
//
// It is built from the oracle itself (this file includes oracle/oracle.cpp and adds one entry point), so the boundary
// hits, Transforms, BVH boxes and intervals are the oracle's own code and arithmetic.  tests/transmittance_oracle.py
// compiles it into a temporary directory with the oracle's flags.
//
// For one ray and interval [t_min, t_max_i], the value is the probability that world.hit(r, [t_min, t_max_i]) returns
// None when every ConstantMedium draws its own uniform number u (volume.rs:37-73: None iff neg_inv_density * ln(u) >
// distance_inside_boundary, i.e. with probability exp(distance_inside_boundary / neg_inv_density)):
//   - a surface hit in the interval makes Hittables / BVH return it whatever the media do: 0;
//   - otherwise every medium the traversal reaches is asked on the full interval, and the factors multiply in
//     ascending medium index;
//   - an empty interval (t_max_i < t_min, or a NaN bound) gives 1.
#include "../oracle/oracle.cpp"

namespace orc {
namespace {

// The media world.hit asks when no surface is hit: a Hittables asks every child (hits.rs:39-46), a BVH node both children
// when its box meets the interval and neither otherwise (bvh.rs:57-85; with no hit the right child keeps the full
// interval), a Transform its child with the local ray (shapes.rs:88-111).  Each ConstantMedium multiplies
// factor[medium_index] by its pass-through probability, computed as ConstantMedium::hit computes distance_inside_boundary.
void media_factors(const Hittable* h, const Ray& r, const Interval& interval, std::vector<double>& factor) {
    if (const auto* l = dynamic_cast<const Hittables*>(h)) {
        for (const Hittable* o : l->objects) media_factors(o, r, interval, factor);
    } else if (const auto* b = dynamic_cast<const BVHNode*>(h)) {
        if (!b->bbox.hit(r, interval)) return;
        if (b->left) media_factors(b->left, r, interval, factor);
        if (b->right) media_factors(b->right, r, Interval::make(interval.min, interval.max), factor);
    } else if (const auto* t = dynamic_cast<const Transform*>(h)) {
        Vec3 to = r.at(1.0);
        Vec3 local_origin = t->detransform(r.orig);
        Vec3 local_to = t->detransform(to);
        media_factors(t->object, Ray(local_origin, local_to - local_origin, r.time), interval, factor);
    } else if (const auto* m = dynamic_cast<const ConstantMedium*>(h)) {  // volume.rs:42-58
        PathCtx ctx;
        ctx.media_enabled = false;  // a boundary holds surfaces only
        HitRecord rec1, rec2;
        if (!m->boundary->hit(r, UNIVERSE, ctx, rec1)) return;
        if (!m->boundary->hit(r, Interval::make(rec1.t + 0.0001, INF), ctx, rec2)) return;
        if (rec1.t < interval.min) rec1.t = interval.min;  // clamp_min_assign
        if (rec2.t > interval.max) rec2.t = interval.max;  // clamp_max_assign
        if (rec1.t >= rec2.t) return;
        if (rec1.t < 0.0) rec1.t = 0.0;
        double ray_length = length(r.dir);
        double distance_inside_boundary = (rec2.t - rec1.t) * ray_length;
        if (m->medium_index >= factor.size()) factor.resize(m->medium_index + 1, 1.0);
        factor[m->medium_index] *= std::exp(distance_inside_boundary / m->neg_inv_density);
    }
}

}  // namespace
}  // namespace orc

extern "C" {

// out[k] for rays[k], t_max_k = t_max_per_ray ? t_max_per_ray[k] : t_max (see the top of the file)
int orc_transmittance(const void* s, const rt_ray* rays, const double* t_max_per_ray, uint64_t n, double t_min, double t_max, double* out) {
    using namespace orc;
    const Scene* sc = (const Scene*)s;
#pragma omp parallel for schedule(dynamic, 256)
    for (int64_t k = 0; k < (int64_t)n; k++) {
        const double t_max_k = t_max_per_ray ? t_max_per_ray[k] : t_max;
        if (!(t_min <= t_max_k)) {
            out[k] = 1.0;
            continue;
        }
        const Interval iv = Interval::raw(t_min, t_max_k);
        Ray r(Vec3(rays[k].origin), Vec3(rays[k].direction), rays[k].time);
        PathCtx ctx;
        ctx.media_enabled = false;
        HitRecord rec;
        if (sc->world->hit(r, iv, ctx, rec)) {
            out[k] = 0.0;
            continue;
        }
        std::vector<double> factor;
        media_factors(sc->world, r, iv, factor);
        double T = 1.0;
        for (double f : factor) T *= f;
        out[k] = T;
    }
    return 0;
}

}  // extern "C"
