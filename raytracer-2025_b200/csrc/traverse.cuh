// traverse.cuh — closest-hit traversal of the flat BVH2 with binary64 primitive tests.
//
// Box tests run in binary32 but are CONSERVATIVE: boxes are rounded outwards at build time and
// every slab distance is widened by a bound on its rounding error, so a box that the exact test
// would enter is never culled.  The primitive tests are the reference's own arithmetic in
// binary64 (sphere.rs:77-108, quad.rs:71-102, triangle.rs:56-98), which makes the winning t
// bit-identical to the CPU restatement for unbaked primitives.  Exact ties are resolved by the
// per-primitive rank (hits.rs:42: first child wins; bvh.rs:78-84: right child wins).
#pragma once
#include "device_math.cuh"
#include "scene_types.h"

namespace rt {

struct RayD {
    D3 o, d;
    double time;
};

// ---- Transform (shapes.rs:74-101) with the reference's quaternion arithmetic -------------------
struct Quat {
    double w, x, y, z;
};
__device__ __forceinline__ Quat qmul(Quat a, Quat b) {  // quaternion.rs:94-104
    return Quat{a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z, a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y,
                a.w * b.y - a.x * b.z + a.y * b.w + a.z * b.x, a.w * b.z + a.x * b.y - a.y * b.x + a.z * b.w};
}
__device__ __forceinline__ D3 qrotate(Quat q, D3 v) {  // quaternion.rs:72-82: q * (0,v) * conj(q)
    Quat r = qmul(qmul(q, Quat{0.0, v.x, v.y, v.z}), Quat{q.w, -q.x, -q.y, -q.z});
    return D3{r.x, r.y, r.z};
}
struct XformParams {
    D3 offset, scale;
    Quat q;
};
__device__ __forceinline__ XformParams load_xform(const Xform* __restrict__ x) {
    XformParams p;
    p.offset = D3{__ldg(&x->offset[0]), __ldg(&x->offset[1]), __ldg(&x->offset[2])};
    p.q = Quat{__ldg(&x->quat[0]), __ldg(&x->quat[1]), __ldg(&x->quat[2]), __ldg(&x->quat[3])};
    p.scale = D3{__ldg(&x->scale[0]), __ldg(&x->scale[1]), __ldg(&x->scale[2])};
    return p;
}
__device__ __forceinline__ D3 xf_transform(const XformParams& p, D3 v) { return qrotate(p.q, v * p.scale) + p.offset; }  // shapes.rs:74-78
__device__ __forceinline__ D3 xf_detransform(const XformParams& p, D3 v) {                                           // shapes.rs:80-84
    D3 r = qrotate(Quat{p.q.w, -p.q.x, -p.q.y, -p.q.z}, v - p.offset);
    return D3{r.x / p.scale.x, r.y / p.scale.y, r.z / p.scale.z};
}
// Transform::hit entry (shapes.rs:93-101) through the whole chain, outermost first: t is preserved
__device__ __noinline__ RayD ray_to_local(const SceneView& sv, uint32_t xform, RayD r) {
    const Xform* x = sv.xforms + xform;
    const uint32_t n = __ldg(&x->n_chain);
    for (uint32_t k = 0; k < n; k++) {
        XformParams p = load_xform(sv.xforms + __ldg(&x->chain[k]));
        D3 to = r.o + 1.0 * r.d;  // r.at(1.0)
        D3 lo = xf_detransform(p, r.o);
        D3 lt = xf_detransform(p, to);
        r.o = lo;
        r.d = lt - lo;
    }
    return r;
}
// point / direction versions for Transform::pdf_value and ::random (shapes.rs:117-132)
__device__ __forceinline__ D3 point_to_local(const SceneView& sv, uint32_t xform, D3 v) {
    const Xform* x = sv.xforms + xform;
    const uint32_t n = __ldg(&x->n_chain);
    for (uint32_t k = 0; k < n; k++) v = xf_detransform(load_xform(sv.xforms + __ldg(&x->chain[k])), v);
    return v;
}

// binary32 image of the ray for the slab test: t = fma(plane, idf, noidf)
#if RT_SLAB_SIGNSEL
// The absolute error bound of a slab distance is folded into the addend (one copy rounded towards the near side,
// one towards the far side) and the near/far plane of every axis is picked by the sign of 1/d, so a box costs
// 6 selects + 6 FMA + 4 min/max instead of 6 FMA + 6 min/max pairs + 6 adds + 4 min/max.
struct RayF {
    float idx, idy, idz;          // 1/d, clamped to +-1e30
    float nxl, nyl, nzl;          // -o * idf - error bound   (-inf on an axis that takes no part in culling)
    float nxh, nyh, nzh;          // -o * idf + error bound   (+inf ...)
    bool sx, sy, sz;              // 1/d < 0: the far plane is `lo`
};
#else
struct RayF {
    float idx, idy, idz;     // 1/d, clamped to +-1e30
    float nox, noy, noz;     // -o * idf (rounded once from binary64)
    float ex, ey, ez;        // per-axis absolute error bound of the slab distances
};
#endif

// moving: the scene holds a moving sphere (SceneView::moving) and the ray may carry any time.
__device__ __forceinline__ void make_rayf(const RayD& r, RayF& f, bool moving) {
    // An axis whose 1/d overflows binary32 range (d == 0, denormal, NaN) takes no part in culling:
    // its error bound is infinite, so its slab is (-inf, +inf).  Conservative, and only rays exactly
    // parallel to an axis plane pay for it.
    auto inv = [](double d, bool& clamped) {
        double i = 1.0 / d;
        clamped = !(fabs(i) <= 1e30);
        if (clamped) i = copysign(1e30, d);
        return (float)i;
    };
    bool cx, cy, cz;
    f.idx = inv(r.d.x, cx), f.idy = inv(r.d.y, cy), f.idz = inv(r.d.z, cz);
    // The box of a moving sphere bounds its centre over times [0, 1] only (sphere.rs:35-51), while Sphere::hit places it at any
    // time: a ray whose time lies outside (or is NaN) culls no box at all, and gets the brute-force answer by testing every
    // primitive.  Only the query kernels of scenes with a moving sphere pay for the check: the render's rays carry get_ray's
    // times in [0, 1).
    if (moving && !(r.time >= 0.0 && r.time <= 1.0)) cx = cy = cz = true;
    const float nox = (float)(-r.o.x * (double)f.idx);
    const float noy = (float)(-r.o.y * (double)f.idy);
    const float noz = (float)(-r.o.z * (double)f.idz);
    // |t_computed - t_exact| <= (|t| + |o*idf|) * 2^-24 ; the |t| part is applied as a relative slack
    const float k = 1.0f / 4194304.0f;  // 2^-22
#if RT_SLAB_SIGNSEL
    const float ex = fabsf(nox) * k, ey = fabsf(noy) * k, ez = fabsf(noz) * k;
    f.nxl = cx ? -INFINITY : nox - ex, f.nxh = cx ? INFINITY : nox + ex;
    f.nyl = cy ? -INFINITY : noy - ey, f.nyh = cy ? INFINITY : noy + ey;
    f.nzl = cz ? -INFINITY : noz - ez, f.nzh = cz ? INFINITY : noz + ez;
    f.sx = f.idx < 0.f, f.sy = f.idy < 0.f, f.sz = f.idz < 0.f;
#else
    f.nox = nox, f.noy = noy, f.noz = noz;
    f.ex = cx ? INFINITY : fabsf(f.nox) * k;
    f.ey = cy ? INFINITY : fabsf(f.noy) * k;
    f.ez = cz ? INFINITY : fabsf(f.noz) * k;
#endif
}

// returns true when the box may intersect the ray within [tmin_f, tmax_f]; tnear for ordering
__device__ __forceinline__ bool slab(const RayF& f, const float* lo, const float* hi, float tmin_f, float tmax_f, float& tnear) {
#if RT_SLAB_SIGNSEL
    // a NaN candidate (inf - inf on a degenerate axis) is ignored by fmaxf/fminf, i.e. that axis does not cull
    float tn = fmaxf(fmaxf(__fmaf_rn(f.sx ? hi[0] : lo[0], f.idx, f.nxl), __fmaf_rn(f.sy ? hi[1] : lo[1], f.idy, f.nyl)),
                     __fmaf_rn(f.sz ? hi[2] : lo[2], f.idz, f.nzl));
    float tf = fminf(fminf(__fmaf_rn(f.sx ? lo[0] : hi[0], f.idx, f.nxh), __fmaf_rn(f.sy ? lo[1] : hi[1], f.idy, f.nyh)),
                     __fmaf_rn(f.sz ? lo[2] : hi[2], f.idz, f.nzh));
#else
    float x0 = __fmaf_rn(lo[0], f.idx, f.nox), x1 = __fmaf_rn(hi[0], f.idx, f.nox);
    float y0 = __fmaf_rn(lo[1], f.idy, f.noy), y1 = __fmaf_rn(hi[1], f.idy, f.noy);
    float z0 = __fmaf_rn(lo[2], f.idz, f.noz), z1 = __fmaf_rn(hi[2], f.idz, f.noz);
    float tn = fmaxf(fmaxf(fminf(x0, x1) - f.ex, fminf(y0, y1) - f.ey), fminf(z0, z1) - f.ez);
    float tf = fminf(fminf(fmaxf(x0, x1) + f.ex, fmaxf(y0, y1) + f.ey), fmaxf(z0, z1) + f.ez);
#endif
    const float rel = 1.0f / 2097152.0f;  // 2^-21
    tn = __fmaf_rn(-fabsf(tn), rel, tn);
    tf = __fmaf_rn(fabsf(tf), rel, tf);
    tnear = tn;
    // written with negations so that a NaN anywhere keeps the box (conservative)
    return !(tn > tf) && !(tn > tmax_f) && !(tf < tmin_f);
}

__device__ __forceinline__ bool contains(double mn, double mx, double x) { return x >= mn && x <= mx; }  // interval.rs:65-67

// 256-bit read-only global loads (LDG.E.256 on sm_100): a diverged warp pays one L1 tag lookup per lane and
// request, so fetching a 64-byte node or a 128-byte primitive in 32-byte pieces halves the L1 work of the
// 16-byte version.  The address must be 32-byte aligned (nodes and primitive records are).
__device__ __forceinline__ void ldg256(const void* p, float4& a, float4& b) {
#if RT_LDG256
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
                 : "l"(p));
#else
    a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
#endif
}
__device__ __forceinline__ void ldg256(const void* p, double2& a, double2& b) {
#if RT_LDG256
    asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a.x), "=d"(a.y), "=d"(b.x), "=d"(b.y) : "l"(p));
#else
    a = __ldg(reinterpret_cast<const double2*>(p)), b = __ldg(reinterpret_cast<const double2*>(p) + 1);
#endif
}

// Sphere::hit, sphere.rs:77-108 (geometry only)
__device__ __forceinline__ bool sphere_hit_at(D3 center, D3 cvec, double radius, const RayD& r, double tmin, double tmax, double& t_out) {
    D3 current_center = center + r.time * cvec;
    D3 oc = current_center - r.o;
    double a = length_squared(r.d);
    double h = dot(r.d, oc);
    double c = length_squared(oc) - radius * radius;
    double discriminant = h * h - a * c;
    if (discriminant < 0.0) return false;
    double sqrtd = sqrt(discriminant);
    double root = (h - sqrtd) / a;
    if (!contains(tmin, tmax, root)) {
        root = (h + sqrtd) / a;
        if (!contains(tmin, tmax, root)) return false;
    }
    t_out = root;
    return true;
}
__device__ __forceinline__ bool sphere_hit(const double* __restrict__ g, const RayD& r, double tmin, double tmax, double& t_out) {
    double2 a0, a1, a2, a3;
    ldg256(g, a0, a1);
    ldg256(g + 4, a2, a3);
    return sphere_hit_at(D3{a0.x, a0.y, a1.x}, D3{a1.y, a2.x, a2.y}, a3.x, r, tmin, tmax, t_out);
}

struct Planar {
    D3 q, u, v, n, w;
    double D;
};
__device__ __forceinline__ void load_planar(const double* __restrict__ g, Planar& p) {
    const double2* s = reinterpret_cast<const double2*>(g);
    double2 a0 = __ldg(s), a1 = __ldg(s + 1), a2 = __ldg(s + 2), a3 = __ldg(s + 3);
    double2 a4 = __ldg(s + 4), a5 = __ldg(s + 5), a6 = __ldg(s + 6), a7 = __ldg(s + 7);
    p.q = D3{a0.x, a0.y, a1.x};
    p.u = D3{a1.y, a2.x, a2.y};
    p.v = D3{a3.x, a3.y, a4.x};
    p.n = D3{a4.y, a5.x, a5.y};
    p.D = a6.x;
    p.w = D3{a6.y, a7.x, a7.y};
}
// the same from a record that is not in global memory (k_walk's shared-memory copy)
__device__ __forceinline__ void load_planar_plain(const double* g, Planar& p) {
    p.q = ld3(g), p.u = ld3(g + 3), p.v = ld3(g + 6), p.n = ld3(g + 9);
    p.D = g[12];
    p.w = ld3(g + 13);
}
// Quad::hit / Triangle::hit, quad.rs:71-102, triangle.rs:56-98 (geometry only)
__device__ __forceinline__ bool planar_hit_loaded(const Planar& p, bool triangle, const RayD& r, double tmin, double tmax,
                                                  double& t_out, double& alpha, double& beta) {
    double denom = dot(p.n, r.d);
    if (fabs(denom) < 1e-8) return false;
    double t = (p.D - dot(p.n, r.o)) / denom;
    if (!contains(tmin, tmax, t)) return false;
    D3 intersection = r.o + t * r.d;
    D3 hp = intersection - p.q;
    alpha = dot(p.w, cross(hp, p.v));
    beta = dot(p.w, cross(p.u, hp));
    if (!contains(0.0, 1.0, alpha) || !contains(0.0, 1.0, beta)) return false;
    if (triangle && !contains(0.0, 1.0, alpha + beta)) return false;
    t_out = t;
    return true;
}
__device__ __forceinline__ bool planar_hit(const double* __restrict__ g, bool triangle, const RayD& r, double tmin, double tmax, double& t_out) {
    // plane first: most candidates are rejected before the rest of the record is needed
    double2 a4, a5, a6, a7;
    ldg256(g + 8, a4, a5);
    ldg256(g + 12, a6, a7);
    D3 n = D3{a4.y, a5.x, a5.y};
    double denom = dot(n, r.d);
    if (fabs(denom) < 1e-8) return false;
    double t = (a6.x - dot(n, r.o)) / denom;
    if (!contains(tmin, tmax, t)) return false;
    double2 a0, a1, a2, a3;
    ldg256(g, a0, a1);
    ldg256(g + 4, a2, a3);
    D3 q = D3{a0.x, a0.y, a1.x}, u = D3{a1.y, a2.x, a2.y}, v = D3{a3.x, a3.y, a4.x}, w = D3{a6.y, a7.x, a7.y};
    D3 intersection = r.o + t * r.d;
    D3 hp = intersection - q;
    double alpha = dot(w, cross(hp, v));
    double beta = dot(w, cross(u, hp));
    if (!contains(0.0, 1.0, alpha) || !contains(0.0, 1.0, beta)) return false;
    if (triangle && !contains(0.0, 1.0, alpha + beta)) return false;
    t_out = t;
    return true;
}

struct TraceCounters {
    uint32_t nodes, prims;
};

// Shared-memory copy of the breadth-first top of the traversed tree (all of it for book-sized scenes).
//
// Four-wide nodes are staged with the TMA bulk-copy engine: one elected thread arms an mbarrier with the byte count and issues
// cp.async.bulk (global -> shared, UBLKCP in SASS) in 32 KB pieces; every thread then waits on the barrier's phase.  No register
// or LSU traffic is spent on the copy, and it overlaps with the rest of the CTA's prologue.
//
// Binary nodes are stored COMPACT: the 48 bytes of boxes of node i at float4[3 i .. 3 i + 2], its two child references in a
// uint2 array behind the boxes - 56 bytes per node instead of the 64 of the global layout (8 are padding), so that book2_final's
// 3201 nodes fit next to the stacks (188 KB) and the node loop never takes its global-memory path: with 6 % of the nodes left
// in global memory almost every warp-wide visit executed both paths.  All threads copy (4 x LDG.128 -> 3 x STS.128 + STS.64).
constexpr uint32_t SMEM_NODE_BYTES = 56;
__device__ __forceinline__ uint32_t cached_tree_float4(const SceneView& sv) {  // size of the node region in float4 units
    return sv.nodes4 ? 8u * sv.n_cached_nodes : (sv.n_cached_nodes * SMEM_NODE_BYTES + 15u) / 16u;
}
__device__ __forceinline__ void stage_nodes(const SceneView& sv, float4* smem_nodes) {
    __shared__ alignas(8) unsigned long long s_bar;
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&s_bar);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (sv.n_cached_nodes == 0) return;
    if (!sv.nodes4) {
        uint2* children = reinterpret_cast<uint2*>(smem_nodes + 3 * sv.n_cached_nodes);
        for (uint32_t i = threadIdx.x; i < sv.n_cached_nodes; i += blockDim.x) {
            const float4* np = reinterpret_cast<const float4*>(sv.nodes + i);
            float4 n0, n1, n2, n3;
            ldg256(np, n0, n1);
            ldg256(np + 2, n2, n3);
            smem_nodes[3 * i] = n0, smem_nodes[3 * i + 1] = n1, smem_nodes[3 * i + 2] = n2;
            children[i] = make_uint2(__float_as_uint(n3.x), __float_as_uint(n3.y));
        }
        __syncthreads();
        return;
    }
    const uint32_t bytes = sv.n_cached_nodes * (uint32_t)sizeof(Node4);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
        const char* src = reinterpret_cast<const char*>(sv.nodes4);
        const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem_nodes);
        for (uint32_t off = 0; off < bytes; off += 32768u) {
            const uint32_t n = min(32768u, bytes - off);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst + off),
                         "l"(src + off), "r"(n), "r"(bar)
                         : "memory");
        }
    }
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(bar)
            : "memory");
    }
}

// Closest hit below `root` within [tmin, tmax] (both inclusive).  smem_nodes holds nodes
// [0, n_cached_nodes); stack[] is this thread's column of the shared-memory traversal stack (entry i
// at stack[i * stride]).
//
// Loop structure: "while-while" with postponed leaves.  A lane that reaches a leaf parks it and keeps
// descending; the warp switches to the (binary64, expensive) primitive tests when every lane still
// traversing has a parked leaf, or a lane meets a second one.  This keeps the primitive-test code
// converged: the first version ran it with 3-7 of 32 lanes active (profiles/r01_v1_*).
// ANY_TIME: r may carry a time outside [0, 1] (make_rayf).
template <bool COUNT, bool USE_RANK, bool ANY_TIME>
__device__ __forceinline__ bool closest_hit(const SceneView& sv, uint32_t root, const RayD& r, double tmin, double tmax,
                                            const float4* __restrict__ smem_nodes, uint32_t* __restrict__ stack, int stride,
                                            double& best_t, uint32_t& best_prim, TraceCounters* cnt) {
    if (root == INVALID_REF) return false;
    double tbest = tmax;
    uint32_t prim = 0xFFFFFFFFu, prim_rank = 0xFFFFFFFFu;
    uint32_t cached_xform = 0xFFFFFFFFu;  // RT_NONE: the world ray itself
    RayD lr = r;                          // the ray in the local space of cached_xform
    float tmax_f = __double2float_ru(tmax);

    auto test_leaf = [&](uint32_t leaf) {
        uint32_t first = (leaf & ~LEAF_FLAG) >> 3, count = (leaf & 7u) + 1;
        for (uint32_t i = 0; i < count; i++) {
            uint32_t pi = first + i;
            const uint4 km = __ldg(reinterpret_cast<const uint4*>(&sv.meta[pi]));  // kind_mat, rank, object, xform
            const uint32_t kind = km.x >> 30;
            if (km.w != cached_xform) {
                lr = km.w == 0xFFFFFFFFu ? r : ray_to_local(sv, km.w, r);
                cached_xform = km.w;
            }
            const double* g = sv.geom[pi].d;
            double t;
            bool hit = kind == PRIM_SPHERE ? sphere_hit(g, lr, tmin, tbest, t) : planar_hit(g, kind == PRIM_TRIANGLE, lr, tmin, tbest, t);
            if (COUNT) cnt->prims++;
            if (hit) {
                // t <= tbest here; an exact tie keeps the lower rank
                bool better = prim == 0xFFFFFFFFu || t < tbest || (USE_RANK && km.y < prim_rank);
                if (better) {
                    tbest = t;
                    prim = pi;
                    prim_rank = km.y;
                    tmax_f = __double2float_ru(t);
                }
            }
        }
    };

    if (root & LEAF_FLAG) {  // a group of at most MAX_LEAF_PRIMS primitives (e.g. a medium boundary): no boxes
        test_leaf(root);
    } else {
        RayF f;
        make_rayf(r, f, ANY_TIME && sv.moving);
        const float tmin_f = __double2float_rd(tmin);
        int sp = 0;
        uint32_t cur = root;         // node to visit next; INVALID_REF when the stack ran out
        uint32_t parked = INVALID_REF;  // postponed leaf
        while (cur != INVALID_REF) {
            while (!(cur & LEAF_FLAG) && cur != INVALID_REF) {
                float4 n0, n1, n2, n3;  // (global memory: the callers - k_tail, k_walk, the media pass - stage no nodes)
                {
                    const float4* np = reinterpret_cast<const float4*>(sv.nodes + cur);
                    ldg256(np, n0, n1);
                    ldg256(np + 2, n2, n3);
                }
                if (COUNT) cnt->nodes++;
                float lo0[3] = {n0.x, n0.y, n0.z}, hi0[3] = {n0.w, n1.x, n1.y};
                float lo1[3] = {n1.z, n1.w, n2.x}, hi1[3] = {n2.y, n2.z, n2.w};
                uint32_t c0 = __float_as_uint(n3.x), c1 = __float_as_uint(n3.y);
                float t0, t1;
                bool h0 = slab(f, lo0, hi0, tmin_f, tmax_f, t0);
                bool h1 = slab(f, lo1, hi1, tmin_f, tmax_f, t1);
                if (h0 && h1) {
                    bool swap = t1 < t0;
                    stack[(sp++) * stride] = swap ? c0 : c1;
                    cur = swap ? c1 : c0;
                } else if (h0 || h1) {
                    cur = h0 ? c0 : c1;
                } else {
                    cur = sp > 0 ? stack[(--sp) * stride] : INVALID_REF;
                }
                if ((cur & LEAF_FLAG) && parked == INVALID_REF) {  // first leaf: park it, keep descending
                    parked = cur;
                    cur = sp > 0 ? stack[(--sp) * stride] : INVALID_REF;
                }
                if (!__any_sync(__activemask(), parked == INVALID_REF)) break;  // every lane has one
            }
            while (parked != INVALID_REF) {
                test_leaf(parked);
                parked = INVALID_REF;
                if (cur & LEAF_FLAG) {  // the node reached after parking is a leaf too
                    parked = cur;
                    cur = sp > 0 ? stack[(--sp) * stride] : INVALID_REF;
                }
            }
        }
    }
    if (prim == 0xFFFFFFFFu) return false;
    best_t = tbest;
    best_prim = prim;
    return true;
}

// Does a primitive of `leaf` (a leaf reference) beat a scatter point at distance t_scatter with tie rank `rank` - a hit in
// [tmin, t_scatter] that is nearer, or at the same distance with a lower rank (the rule of closest_hit)?  k_walk's test of the
// entry leaves of a medium: no boxes, no stack.
__device__ __forceinline__ bool leaf_beats_scatter(const SceneView& sv, uint32_t leaf, const RayD& r, double tmin, double t_scatter, uint32_t rank) {
    const uint32_t first = (leaf & ~LEAF_FLAG) >> 3, count = (leaf & 7u) + 1;
    uint32_t cached_xform = 0xFFFFFFFFu;
    RayD lr = r;
    bool beaten = false;
    for (uint32_t i = 0; i < count; i++) {
        const uint32_t pi = first + i;
        const uint4 km = __ldg(reinterpret_cast<const uint4*>(&sv.meta[pi]));  // kind_mat, rank, object, xform
        if (km.w != cached_xform) {
            lr = km.w == 0xFFFFFFFFu ? r : ray_to_local(sv, km.w, r);
            cached_xform = km.w;
        }
        const double* g = sv.geom[pi].d;
        const uint32_t kind = km.x >> 30;
        double t;
        const bool hit = kind == PRIM_SPHERE ? sphere_hit(g, lr, tmin, t_scatter, t) : planar_hit(g, kind == PRIM_TRIANGLE, lr, tmin, t_scatter, t);
        beaten = beaten || (hit && (t < t_scatter || km.y < rank));  // t <= t_scatter here
    }
    return beaten;
}

// ------------------------------------------------------------------------------------------------
// Persistent "while-while" traversal fed from a per-warp FIFO of PREPARED rays.
//
// Work items are dealt to CTAs in interleaved groups of 32.  A warp refills its FIFO with all 32 lanes at
// once: lane i loads item i of the warp's next group (one coalesced 2 KB read, prefetched into L2 when the
// group was claimed, one refill earlier), derives the binary32 slab image of the ray (three binary64
// divisions) and stores the prepared ray in shared memory.  A lane whose traversal has finished POPS a
// prepared ray - seven 128-bit shared-memory loads - at the top of a round once `refill_min` lanes are idle.
// Round 1 refilled lanes in place: ~250 warp-instructions at 1-2 active lanes, which is why it was a net
// loss on cache-resident scenes; the FIFO splits that into a converged part and a cheap pop.
//
// Slot layout, 7 x 16 bytes (a stride of 28 words puts the 128-bit accesses of eight consecutive slots on
// disjoint banks, so refill stores and pop loads are conflict free):
//   q0 o.x o.y | q1 o.z d.x | q2 d.y d.z | q3 time tmax | q4 prim0 rank0 item 1/d.x | q5 1/d.y 1/d.z nxl nyl | q6 nzl nxh nyh nzh
//
// Measured alternatives (profiles/README.md, round 2): a step-scheduled loop (one node step per round for every
// lane at an inner node, primitive tests only when `leaf_min` lanes hold a leaf) raised the active lanes from 15
// to 21 but lost 35 % in time on book2_final - every round pays four warp votes and the reconvergence of three
// divergent regions, and the tight node loop below is what hides the L1/shared-memory latency.
//
// PARK = postponed leaves: a lane that reaches a leaf parks it and keeps descending until every lane of the
// warp holds one, so the binary64 primitive tests run converged.  Worth it when traversals are long (1M-triangle
// soup, 106 nodes per ray); on the book scenes (11 nodes + 3.7 primitive tests per ray) the extra votes cost more
// than they save, so rt_scene_create picks per scene (SceneView::park_leaves).
//
// IO::load(item, ray, tmax, prim0, rank0) -> bool, IO::t_min() and IO::store(item, hit, t, prim) bind the routine
// to the path streams (k_extend) or to a plain ray array (k_closest_hit, k_occluded).  An item whose load returns false is
// dropped without a store.
// ------------------------------------------------------------------------------------------------
constexpr uint32_t FIFO_SLOT_WORDS = 28;
constexpr uint32_t FIFO_INVALID_ITEM = 0xFFFFFFFFu;  // a slot of the ragged last group: popped and dropped

// WIDE = traverse the four-wide collapse (sv.nodes4, out-of-cache scenes): four slab tests per fetch, the hit
// children are ordered by entry distance with a five-exchange network, the nearest is followed and the others
// are pushed farthest first.
// (WIDE == 2: the whole four-wide tree is in shared memory - a variant of its own, because a per-visit choice between the two
// node sources costs the global-memory traversal of the big scenes 7 % in Mrays/s; WIDE == 3: the BINARY tree, all of it in
// shared memory, likewise without the global-memory path)
// XF = false: the scene has no Transform at all (the soups): no local-space copy of the ray, no detransform code.
// KINDS: 0 = any primitives, 1 = the scene holds spheres only, 2 = quads / triangles only (a mesh, the soups): the other test is compiled out.
// ANY = any-hit (occlusion): the first primitive test that hits within [tmin, tmax] ends the lane's traversal - its parked leaf,
// the rest of the current leaf and its stack are dropped - and store() is called with hit = true.  The interval never shrinks, so
// no rank, kind or binary32 bound is kept.
template <bool COUNT, bool USE_RANK, bool PARK, int WIDE, bool XF, int KINDS, bool ANY = false, class IO>
__device__ __forceinline__ void trace_persistent(const SceneView& sv, IO& io, uint32_t n, uint32_t* s_cursor,
                                                 const float4* __restrict__ smem_nodes, uint32_t* __restrict__ stack, int stride,
                                                 uint32_t* __restrict__ fifo, uint32_t fifo_slots_arg, TraceCounters* cnt, double* __restrict__ ray_s = nullptr) {
    // the all-in-shared-memory variants run in direct mode only (the shared memory holds the tree, not FIFOs): no FIFO code in them;
    // the four-wide tree in global memory is always fed from the FIFOs (api.cu gives it at least 32 slots): no direct-mode code
    const uint32_t fifo_slots = WIDE >= 2 ? 0u : fifo_slots_arg;
    constexpr bool FIFO_ONLY = WIDE == 1;
    const unsigned FULL = 0xFFFFFFFFu;
    const uint32_t lane = threadIdx.x & 31u;
#if RT_RAY_SMEM
    // The binary64 ray (and its image in the local space of the last Transform met) lives in shared memory, component k of this
    // thread at ray_s[k * stride]: only the leaf tests read it, and 28 registers fewer per thread are four more warps per SM.
    auto put_ray = [&](int base, const RayD& q) {
        ray_s[(base + 0) * stride] = q.o.x, ray_s[(base + 1) * stride] = q.o.y, ray_s[(base + 2) * stride] = q.o.z;
        ray_s[(base + 3) * stride] = q.d.x, ray_s[(base + 4) * stride] = q.d.y, ray_s[(base + 5) * stride] = q.d.z;
        ray_s[(base + 6) * stride] = q.time;
    };
    auto get_ray = [&](int base) {
        RayD q;
        q.o = D3{ray_s[(base + 0) * stride], ray_s[(base + 1) * stride], ray_s[(base + 2) * stride]};
        q.d = D3{ray_s[(base + 3) * stride], ray_s[(base + 4) * stride], ray_s[(base + 5) * stride]};
        q.time = ray_s[(base + 6) * stride];
        return q;
    };
#endif
    const unsigned lt_mask = (1u << lane) - 1u;
    const uint32_t G = gridDim.x, b = blockIdx.x;
    const uint32_t n_groups = (n + 31u) >> 5;
    const uint32_t local_groups = (n_groups + G - 1u - b) / G;  // groups of 32 items dealt to this CTA
    const uint32_t q_mask = fifo_slots - 1u;                    // fifo_slots is 32 or 64
    const uint32_t refill_min = sv.refill_min;

    bool have = false;
    bool exhausted = false;            // warp-uniform: the CTA's cursor ran past its last group
    uint32_t head = 0, avail = 0;      // warp-uniform FIFO state: first filled slot, number of filled slots
    uint32_t item = 0;
#if !RT_RAY_SMEM
    RayD r, lr;
#endif
    RayF f;
    const double tmin = io.t_min();
    const float tmin_f = __double2float_rd(tmin);
    double tbest = 0.0;
    float tmax_f = 0.f;
    uint32_t prim = 0xFFFFFFFFu, prim_rank = 0xFFFFFFFFu, cached_xform = 0xFFFFFFFFu;
    uint32_t prim_meta = 0;         // PrimMeta::kind_mat of the incumbent (kind, shade class, material)
    uint32_t cur = INVALID_REF;     // inner node to visit next | a second leaf met while `parked` is taken (PARK) | INVALID_REF
    uint32_t parked = INVALID_REF;  // the leaf this lane holds
    int sp = 0;

    // the group this warp will load at its next refill: claimed (and prefetched) one refill ahead
    uint32_t next_group = 0;
    {
        if (lane == 0) next_group = atomicAdd(s_cursor, 1u);
        next_group = __shfl_sync(FULL, next_group, 0);
        if (next_group < local_groups) io.prefetch((next_group * G + b) * 32u + lane);
    }

    while (true) {
        const unsigned idle = __ballot_sync(FULL, !have);
        // sv.refill_min: idle lanes a warp waits for before it pops (32 = drain the warp completely)
        if (idle && ((FIFO_ONLY || fifo_slots) ? ((uint32_t)__popc(idle) >= refill_min || idle == FULL) : idle == FULL)) {
            const uint32_t n_idle = __popc(idle);
            if (!FIFO_ONLY && fifo_slots == 0) {
                // ---- direct mode (no FIFO: the shared memory holds the whole tree instead): the warp has drained,
                // every lane prepares the ray it will trace itself ----
                const uint32_t g = next_group;
                if (g >= local_groups) {
                    exhausted = true;
                } else {
                    if (lane == 0) next_group = atomicAdd(s_cursor, 1u);
                    next_group = __shfl_sync(FULL, next_group, 0);
                    if (next_group < local_groups) io.prefetch((next_group * G + b) * 32u + lane);
                    const uint32_t it = (g * G + b) * 32u + lane;
                    prim = 0xFFFFFFFFu, prim_rank = 0xFFFFFFFFu;
#if RT_RAY_SMEM
                    RayD r;
#endif
                    if (it < n && io.load(it, r, tbest, prim, prim_rank)) {
                        item = it;
                        make_rayf(r, f, IO::any_time && sv.moving);
                        have = true;
                        tmax_f = __double2float_ru(tbest);
                        cached_xform = 0xFFFFFFFFu;
#if RT_RAY_SMEM
                        put_ray(0, r);
#else
                        if (XF) lr = r;
#endif
                        sp = 0;
                        const uint32_t root = (WIDE == 1 || WIDE == 2) ? sv.world_root4 : sv.world_root;
                        if (root & LEAF_FLAG)
                            parked = root, cur = INVALID_REF;
                        else
                            parked = INVALID_REF, cur = root;
                    }
                }
            } else {
                // ---- refill: every lane of the warp prepares one ray of the claimed group (converged) ----
                if (avail < n_idle && !exhausted && avail + 32u <= fifo_slots) {
                    const uint32_t g = next_group;
                    if (g >= local_groups) {
                        exhausted = true;
                    } else {
                        if (lane == 0) next_group = atomicAdd(s_cursor, 1u);
                        next_group = __shfl_sync(FULL, next_group, 0);
                        if (next_group < local_groups) io.prefetch((next_group * G + b) * 32u + lane);
                        const uint32_t it = (g * G + b) * 32u + lane;
                        uint32_t* slot = fifo + ((head + avail + lane) & q_mask) * FIFO_SLOT_WORDS;
                        RayD pr;
                        RayF pf;
                        double ptmax = 0.0;
                        uint32_t p0 = 0xFFFFFFFFu, r0 = 0xFFFFFFFFu;
                        uint32_t pit = FIFO_INVALID_ITEM;
                        if (it < n && io.load(it, pr, ptmax, p0, r0)) {
                            pit = it;
                            make_rayf(pr, pf, IO::any_time && sv.moving);
                        } else {
                            pr.o = pr.d = D3{0.0, 0.0, 0.0}, pr.time = 0.0;
                            pf.idx = pf.idy = pf.idz = pf.nxl = pf.nyl = pf.nzl = pf.nxh = pf.nyh = pf.nzh = 0.f;
                        }
                        double2* sd = reinterpret_cast<double2*>(slot);
                        sd[0] = make_double2(pr.o.x, pr.o.y);
                        sd[1] = make_double2(pr.o.z, pr.d.x);
                        sd[2] = make_double2(pr.d.y, pr.d.z);
                        sd[3] = make_double2(pr.time, ptmax);
                        float4* sf = reinterpret_cast<float4*>(slot);
                        sf[4] = make_float4(__uint_as_float(p0), __uint_as_float(r0), __uint_as_float(pit), pf.idx);
                        sf[5] = make_float4(pf.idy, pf.idz, pf.nxl, pf.nyl);
                        sf[6] = make_float4(pf.nzl, pf.nxh, pf.nyh, pf.nzh);
                        avail += 32u;
                        __syncwarp();  // the slots are read by other lanes below
                    }
                }
                // ---- pop: the k-th idle lane takes the k-th filled slot ----
                const uint32_t take = min(n_idle, avail);
                const uint32_t my = __popc(idle & lt_mask);
                if (!have && my < take) {
                    const uint32_t* slot = fifo + ((head + my) & q_mask) * FIFO_SLOT_WORDS;
                    const float4 q4 = reinterpret_cast<const float4*>(slot)[4];
                    item = __float_as_uint(q4.z);
                    if (item != FIFO_INVALID_ITEM) {
                        const double2* sd = reinterpret_cast<const double2*>(slot);
                        const double2 a0 = sd[0], a1 = sd[1], a2 = sd[2], a3 = sd[3];
                        const float4 q5 = reinterpret_cast<const float4*>(slot)[5], q6 = reinterpret_cast<const float4*>(slot)[6];
#if RT_RAY_SMEM
                        RayD r;
#endif
                        r.o = D3{a0.x, a0.y, a1.x};
                        r.d = D3{a1.y, a2.x, a2.y};
                        r.time = a3.x;
                        tbest = a3.y;
                        // prim / prim_rank may start from an incumbent the caller already knows (a medium scatter point)
                        prim = __float_as_uint(q4.x), prim_rank = __float_as_uint(q4.y);
                        f.idx = q4.w, f.idy = q5.x, f.idz = q5.y;
                        f.nxl = q5.z, f.nyl = q5.w, f.nzl = q6.x;
                        f.nxh = q6.y, f.nyh = q6.z, f.nzh = q6.w;
                        f.sx = f.idx < 0.f, f.sy = f.idy < 0.f, f.sz = f.idz < 0.f;
                        have = true;
                        tmax_f = __double2float_ru(tbest);
                        cached_xform = 0xFFFFFFFFu;
#if RT_RAY_SMEM
                        put_ray(0, r);
#else
                        if (XF) lr = r;
#endif
                        sp = 0;
                        const uint32_t root = (WIDE == 1 || WIDE == 2) ? sv.world_root4 : sv.world_root;
                        if (root & LEAF_FLAG)
                            parked = root, cur = INVALID_REF;
                        else
                            parked = INVALID_REF, cur = root;  // INVALID_REF root (empty world) finishes at once
                    }
                }
                head += take, avail -= take;
                __syncwarp();  // pops are complete before a later refill overwrites the slots
            }
        }
        if (__ballot_sync(FULL, have) == 0) {
            if (exhausted && avail == 0) break;
            continue;  // only dropped slots were popped (ragged tail) or the FIFO still holds rays
        }
        if (have) {
            // node phase: descend until this lane has parked a leaf and met another, or ran out
            while (!(cur & LEAF_FLAG) && cur != INVALID_REF) {
                if (WIDE == 1 || WIDE == 2) {
                    float4 a0, a1, a2, a3, a4, a5;
                    uint4 cr;
                    if (WIDE == 2) {
                        const float4* np = smem_nodes + 8 * cur;
                        a0 = np[0], a1 = np[1], a2 = np[2], a3 = np[3], a4 = np[4], a5 = np[5];
                        cr = *reinterpret_cast<const uint4*>(np + 6);
                    } else {
                        const float4* np = reinterpret_cast<const float4*>(sv.nodes4 + cur);
                        ldg256(np, a0, a1);
                        ldg256(np + 2, a2, a3);
                        ldg256(np + 4, a4, a5);
                        cr = __ldg(reinterpret_cast<const uint4*>(np + 6));
                    }
                    if (COUNT) cnt->nodes++;
                    const float l0[3] = {a0.x, a0.y, a0.z}, u0[3] = {a0.w, a1.x, a1.y};
                    const float l1[3] = {a1.z, a1.w, a2.x}, u1[3] = {a2.y, a2.z, a2.w};
                    const float l2[3] = {a3.x, a3.y, a3.z}, u2[3] = {a3.w, a4.x, a4.y};
                    const float l3[3] = {a4.z, a4.w, a5.x}, u3[3] = {a5.y, a5.z, a5.w};
                    float k0, k1, k2, k3;
                    uint32_t r0 = cr.x, r1 = cr.y, r2 = cr.z, r3 = cr.w;
                    // a child that is missed (or an unused slot: inverted box, and the explicit test covers the degenerate ray
                    // whose three axes take no part in culling) becomes INVALID_REF with an infinite key and sorts last
                    if (!slab(f, l0, u0, tmin_f, tmax_f, k0) || r0 == INVALID_REF) r0 = INVALID_REF, k0 = INFINITY;
                    if (!slab(f, l1, u1, tmin_f, tmax_f, k1) || r1 == INVALID_REF) r1 = INVALID_REF, k1 = INFINITY;
                    if (!slab(f, l2, u2, tmin_f, tmax_f, k2) || r2 == INVALID_REF) r2 = INVALID_REF, k2 = INFINITY;
                    if (!slab(f, l3, u3, tmin_f, tmax_f, k3) || r3 == INVALID_REF) r3 = INVALID_REF, k3 = INFINITY;
                    auto cswap = [](float& ka, uint32_t& ra, float& kb, uint32_t& rb) {
                        const bool s = kb < ka;
                        const float kt = s ? kb : ka;
                        const uint32_t rt_ = s ? rb : ra;
                        kb = s ? ka : kb, rb = s ? ra : rb;
                        ka = kt, ra = rt_;
                    };
                    cswap(k0, r0, k1, r1);
                    cswap(k2, r2, k3, r3);
                    cswap(k0, r0, k2, r2);
                    cswap(k1, r1, k3, r3);
                    cswap(k1, r1, k2, r2);
                    // hits sort before misses, except that a NaN key (a box kept because nothing could be decided) may sit
                    // anywhere: validity is the reference, not the key
                    if (r3 != INVALID_REF) stack[(sp++) * stride] = r3;
                    if (r2 != INVALID_REF) stack[(sp++) * stride] = r2;
                    if (r1 != INVALID_REF) stack[(sp++) * stride] = r1;
                    if (r0 != INVALID_REF)
                        cur = r0;
                    else
                        cur = sp > 0 ? stack[(--sp) * stride] : INVALID_REF;
                } else {
                    float4 n0, n1, n2;
                    uint32_t c0, c1;
                    if (WIDE == 3 || cur < sv.n_cached_nodes) {  // compact shared-memory layout (stage_nodes); WIDE == 3: every node is there
                        const float4* np = smem_nodes + 3 * cur;
                        n0 = np[0], n1 = np[1], n2 = np[2];
                        const uint2 cc = reinterpret_cast<const uint2*>(smem_nodes + 3 * sv.n_cached_nodes)[cur];
                        c0 = cc.x, c1 = cc.y;
                    } else {
                        const float4* np = reinterpret_cast<const float4*>(sv.nodes + cur);
                        float4 n3;
                        ldg256(np, n0, n1);
                        ldg256(np + 2, n2, n3);
                        c0 = __float_as_uint(n3.x), c1 = __float_as_uint(n3.y);
                    }
                    if (COUNT) cnt->nodes++;
                    float lo0[3] = {n0.x, n0.y, n0.z}, hi0[3] = {n0.w, n1.x, n1.y};
                    float lo1[3] = {n1.z, n1.w, n2.x}, hi1[3] = {n2.y, n2.z, n2.w};
                    float t0, t1;
                    bool h0 = slab(f, lo0, hi0, tmin_f, tmax_f, t0);
                    bool h1 = slab(f, lo1, hi1, tmin_f, tmax_f, t1);
                    if (h0 && h1) {
                        bool swap = t1 < t0;
                        stack[(sp++) * stride] = swap ? c0 : c1;
                        cur = swap ? c1 : c0;
                    } else if (h0 || h1) {
                        cur = h0 ? c0 : c1;
                    } else {
                        cur = sp > 0 ? stack[(--sp) * stride] : INVALID_REF;
                    }
                }
                if (PARK) {  // keep descending with one postponed leaf until every lane of the warp has one
                    if ((cur & LEAF_FLAG) && parked == INVALID_REF) {
                        parked = cur;
                        cur = sp > 0 ? stack[(--sp) * stride] : INVALID_REF;
                    }
#if RT_PARK_VOTE
                    if (!__any_sync(__activemask(), parked == INVALID_REF)) break;
#endif
                } else if (cur & LEAF_FLAG) {  // plain while-while: leave the node loop with the leaf
                    parked = cur;
                    cur = sp > 0 ? stack[(--sp) * stride] : INVALID_REF;
                    break;
                }
            }
            // leaf phase
            while (parked != INVALID_REF) {
                const uint32_t first = (parked & ~LEAF_FLAG) >> 3, count = (parked & 7u) + 1;
                for (uint32_t i = 0; i < count; i++) {
                    const uint32_t pi = first + i;
                    const uint4 km = __ldg(reinterpret_cast<const uint4*>(&sv.meta[pi]));
                    const uint32_t kind = km.x >> 30;
#if RT_RAY_SMEM
                    if (km.w != 0xFFFFFFFFu && km.w != cached_xform) {
                        put_ray(7, ray_to_local(sv, km.w, get_ray(0)));
                        cached_xform = km.w;
                    }
                    const RayD lr = get_ray(km.w == 0xFFFFFFFFu ? 0 : 7);
#else
                    if (XF && km.w != cached_xform) {
                        lr = km.w == 0xFFFFFFFFu ? r : ray_to_local(sv, km.w, r);
                        cached_xform = km.w;
                    }
#endif
                    const double* g = sv.geom[pi].d;
                    double t;
                    const RayD& tr = XF ? lr : r;
                    bool hit = KINDS == 1   ? sphere_hit(g, tr, tmin, tbest, t)
                               : KINDS == 2 ? planar_hit(g, kind == PRIM_TRIANGLE, tr, tmin, tbest, t)
                               : kind == PRIM_SPHERE ? sphere_hit(g, tr, tmin, tbest, t) : planar_hit(g, kind == PRIM_TRIANGLE, tr, tmin, tbest, t);
                    if (COUNT) cnt->prims++;
                    if (ANY) {
                        if (hit) {
                            prim = pi;
                            cur = INVALID_REF;  // with parked = INVALID_REF below: the traversal is finished
                            break;
                        }
                    } else if (hit && (prim == 0xFFFFFFFFu || t < tbest || (USE_RANK && km.y < prim_rank))) {
                        tbest = t;
                        prim = pi;
                        prim_rank = km.y;
                        prim_meta = km.x;
                        tmax_f = __double2float_ru(t);
                    }
                }
                parked = INVALID_REF;
                if (cur & LEAF_FLAG) {
                    parked = cur;
                    cur = sp > 0 ? stack[(--sp) * stride] : INVALID_REF;
                }
            }
            if (cur == INVALID_REF) {  // traversal finished
                io.store(item, prim != 0xFFFFFFFFu, tbest, prim, prim_meta);
                have = false;
            }
        }
    }
}

// ConstantMedium boundary that is one untransformed-or-transformed Sphere: both boundary hits of
// volume.rs:42-45 share a, h, c and the square root.  Same operations, same order, same results as
// two Sphere::hit calls on (-inf, inf) and [t1 + 1e-4, inf).  near_root / far_root are the two roots Sphere::hit would compute
// for the same sphere and ray whatever the interval (NaN when the discriminant is negative: no interval contains them).
__device__ __forceinline__ bool sphere_entry_exit_at(D3 center, D3 cvec, double radius, const RayD& r, double& t1, double& t2, double& near_root,
                                                     double& far_root) {
    D3 current_center = center + r.time * cvec;
    D3 oc = current_center - r.o;
    double a = length_squared(r.d);
    double h = dot(r.d, oc);
    double c = length_squared(oc) - radius * radius;
    double discriminant = h * h - a * c;
    near_root = far_root = __longlong_as_double(0x7FF8000000000000ll);
    if (discriminant < 0.0) return false;
    double sqrtd = sqrt(discriminant);
    near_root = (h - sqrtd) / a, far_root = (h + sqrtd) / a;
    // first hit on Interval::UNIVERSE: only a NaN root is rejected
    double first = near_root;
    if (!contains(-INFINITY, INFINITY, first)) {
        first = far_root;
        if (!contains(-INFINITY, INFINITY, first)) return false;
    }
    // second hit on [first + 1e-4, inf)
    const double lo = first + 0.0001;
    double second = near_root;
    if (!contains(lo, INFINITY, second)) {
        second = far_root;
        if (!contains(lo, INFINITY, second)) return false;
    }
    t1 = first;
    t2 = second;
    return true;
}
__device__ __forceinline__ bool sphere_entry_exit(const double* __restrict__ g, const RayD& r, double& t1, double& t2) {
    const double2 a0 = __ldg(reinterpret_cast<const double2*>(g));
    const double2 a1 = __ldg(reinterpret_cast<const double2*>(g) + 1);
    const double2 a2 = __ldg(reinterpret_cast<const double2*>(g) + 2);
    const double2 a3 = __ldg(reinterpret_cast<const double2*>(g) + 3);
    double near_root, far_root;
    return sphere_entry_exit_at(D3{a0.x, a0.y, a1.x}, D3{a1.y, a2.x, a2.y}, a3.x, r, t1, t2, near_root, far_root);
}

// ConstantMedium::hit after the two boundary hits t1 < t2 (volume.rs:46-73) on the caller's interval [1e-8, inf): true and the
// scatter distance when the path scatters inside.  lr: the ray in the medium's space.
__device__ __forceinline__ bool medium_free_flight(double t1, double t2, const RayD& lr, double neg_inv_density, double xi, double& tm) {
    if (t1 < 1e-8) t1 = 1e-8;  // clamp to the caller's interval [1e-8, inf)
    if (t1 >= t2) return false;
    if (t1 < 0.0) t1 = 0.0;
    const double ray_length = length(lr.d);
    const double distance_inside_boundary = (t2 - t1) * ray_length;
    // binary32 screen: when even a pessimistic free-flight estimate clears the segment inside the boundary by a wide
    // margin the path does not scatter here and the binary64 ln is not needed (the exact comparison below is unchanged)
    const float hf = (float)neg_inv_density * logf((float)xi);
    const float hf_err = 4e-7f * fabsf((float)neg_inv_density);
    if (hf > (float)distance_inside_boundary * 1.001f + hf_err) return false;
    const double hit_distance = neg_inv_density * log(xi);
    if (hit_distance > distance_inside_boundary) return false;
    tm = t1 + hit_distance / ray_length;
    return true;
}

// binary32 screen of a medium against a known hit at t: the scatter point lies at t1 + dist/len with t1 >= 0, so a free flight
// that clearly overshoots the known hit cannot win whatever the boundary does.  Below |d| = 1e-18 the binary32 squares of the
// components are subnormal or zero and len_f comes out too short, so such a direction is not screened.
__device__ __forceinline__ bool free_flight_overshoots(double neg_inv_density, double xi, double t, const D3& ld) {
    const float hf = (float)neg_inv_density * logf((float)xi);
    const float hf_err = 4e-7f * fabsf((float)neg_inv_density);
    const float len_f = sqrtf((float)ld.x * (float)ld.x + (float)ld.y * (float)ld.y + (float)ld.z * (float)ld.z);
    return len_f >= 1e-18f && hf > (float)t * len_f * 1.001f + hf_err;
}

}  // namespace rt
