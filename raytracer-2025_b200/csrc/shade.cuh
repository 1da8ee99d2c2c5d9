// shade.cuh — textures, materials, pdfs and light sampling on the device, in the reference's
// operation order (texture.rs, material.rs, pdf.rs, utils/perlin.rs, shapes/*.rs pdf_value/random).
#pragma once
#include "disney.cuh"
#include "traverse.cuh"

namespace rt {

// ---- texture.rs ------------------------------------------------------------------------------
__device__ __forceinline__ int32_t as_i32_sat(double x) {  // Rust `as i32`
    if (isnan(x)) return 0;
    if (x >= 2147483647.0) return 2147483647;
    if (x <= -2147483648.0) return (-2147483647 - 1);
    return (int32_t)x;
}
__device__ __forceinline__ uint32_t as_u32_sat(double x) {  // Rust `as u32`
    if (!(x > 0.0)) return 0u;
    if (x >= 4294967295.0) return 0xFFFFFFFFu;
    return (uint32_t)x;
}

// utils/perlin.rs:40-59, 73-89
__device__ inline double perlin_noise(const Perlin* __restrict__ tab, D3 p) {
    double fx = floor(p.x), fy = floor(p.y), fz = floor(p.z);
    long long i = (long long)fx, j = (long long)fy, k = (long long)fz;  // saturating like `as i64`
    double u = p.x - fx, v = p.y - fy, w = p.z - fz;
    double uu = u * u * (3.0 - 2.0 * u), vv = v * v * (3.0 - 2.0 * v), ww = w * w * (3.0 - 2.0 * w);
    double accum = 0.0;
#pragma unroll
    for (int di = 0; di < 2; di++)
#pragma unroll
        for (int dj = 0; dj < 2; dj++)
#pragma unroll
            for (int dk = 0; dk < 2; dk++) {
                uint32_t idx = __ldg(&tab->perm_x[(unsigned long long)(i + di) & 255]) ^ __ldg(&tab->perm_y[(unsigned long long)(j + dj) & 255]) ^
                               __ldg(&tab->perm_z[(unsigned long long)(k + dk) & 255]);
                D3 c = D3{__ldg(&tab->randvec[idx][0]), __ldg(&tab->randvec[idx][1]), __ldg(&tab->randvec[idx][2])};
                D3 weight_v = D3{u - (double)di, v - (double)dj, w - (double)dk};
                accum += ((double)di * uu + (double)(1 - di) * (1.0 - uu)) * ((double)dj * vv + (double)(1 - dj) * (1.0 - vv)) *
                         ((double)dk * ww + (double)(1 - dk) * (1.0 - ww)) * dot(c, weight_v);
            }
    return accum;
}
__device__ inline double perlin_turb(const Perlin* __restrict__ tab, D3 p, int depth) {  // perlin.rs:61-71
    double accum = 0.0, weight = 1.0;
    D3 temp_p = p;
    for (int i = 0; i < depth; i++) {
        accum = accum + weight * perlin_noise(tab, temp_p);
        temp_p = 2.0 * temp_p;
        weight = 0.5 * weight;
    }
    return fabs(accum);
}

// utils/image.rs:63-82 — texels were sRGB-decoded once at upload
__device__ __forceinline__ float4 image_pixel(const SceneView& sv, const Image& im, uint32_t x, uint32_t y) {
    x = min(x, im.width - 1);
    y = min(y, im.height - 1);
    return __ldg(&sv.texels[im.texel_offset + (uint64_t)y * im.width + x]);
}
__device__ inline float4 image_get_pixel(const SceneView& sv, uint32_t image, double u, double v) {  // texture.rs:111-158
    const Image im = sv.images[image];
    u = u - floor(u);
    v = 1.0 - (v - floor(v));
    if (!(im.flags & RT_IMG_INTERP)) {
        uint32_t i = as_u32_sat(u * (double)im.width), j = as_u32_sat(v * (double)im.height);
        return image_pixel(sv, im, i, j);
    }
    double x = u * (double)im.width - 0.5, y = v * (double)im.height - 0.5;
    uint32_t x0 = as_u32_sat(rmax(floor(x), 0.0)), y0 = as_u32_sat(rmax(floor(y), 0.0));
    uint32_t x1 = min(x0 + 1, im.width - 1), y1 = min(y0 + 1, im.height - 1);
    double dx = x - (double)x0, dy = y - (double)y0;
    float4 p00 = image_pixel(sv, im, x0, y0), p10 = image_pixel(sv, im, x1, y0);
    float4 p01 = image_pixel(sv, im, x0, y1), p11 = image_pixel(sv, im, x1, y1);
    float fx = (float)dx, fy = (float)dy;
    auto mix = [&](float a00, float a10, float a01, float a11) {
        float v0 = __fadd_rn(__fmul_rn(a00, 1.0f - fx), __fmul_rn(a10, fx));
        float v1 = __fadd_rn(__fmul_rn(a01, 1.0f - fx), __fmul_rn(a11, fx));
        return __fadd_rn(__fmul_rn(v0, 1.0f - fy), __fmul_rn(v1, fy));
    };
    return make_float4(mix(p00.x, p10.x, p01.x, p11.x), mix(p00.y, p10.y, p01.y, p11.y), mix(p00.z, p10.z, p01.z, p11.z),
                       mix(p00.w, p10.w, p01.w, p11.w));
}

__device__ inline D3 texture_value(const SceneView& sv, uint32_t tex, double u, double v, D3 p) {
    while (true) {
        const Texture& t = sv.textures[tex];
        switch (t.kind) {
            case RT_TEX_SOLID: return ld3(t.color);  // texture.rs:32-36
            case RT_TEX_CHECKER: {                    // texture.rs:59-73
                int32_t xi = as_i32_sat(floor(t.scale * p.x)), yi = as_i32_sat(floor(t.scale * p.y)), zi = as_i32_sat(floor(t.scale * p.z));
                int32_t sum = (int32_t)((uint32_t)xi + (uint32_t)yi + (uint32_t)zi);
                tex = (sum % 2 == 0) ? t.a : t.b;
                continue;
            }
            case RT_TEX_IMAGE: {  // texture.rs:166-174
                if (t.a == RT_NONE) return D3{0.0, 1.0, 1.0};
                float4 px = image_get_pixel(sv, t.a, u, v);
                return D3{(double)px.x, (double)px.y, (double)px.z};
            }
            case RT_TEX_NOISE: {  // texture.rs:191-196
                double s = 1.0 + sin(t.scale * p.z + 10.0 * perlin_turb(&sv.perlins[t.a], p, 7));
                return D3{0.5, 0.5, 0.5} * s;
            }
            default: {  // RT_TEX_GRADIENT_Y
                double a = 0.5 * (p.y + 1.0);
                return (1.0 - a) * ld3(t.color) + a * ld3(t.color2);
            }
        }
    }
}
__device__ __forceinline__ bool texture_needs_uv(const SceneView& sv, uint32_t tex) {
    uint32_t k = sv.textures[tex].kind;
    return k == RT_TEX_IMAGE || k == RT_TEX_CHECKER;
}

// Sphere::get_sphere_uv, sphere.rs:53-61
__device__ __forceinline__ void sphere_uv(D3 p, double& u, double& v) {
    double theta = acos(-p.y);
    double phi = atan2(-p.z, p.x) + RT_PI;
    u = phi / (2.0 * RT_PI);
    v = theta / RT_PI;
}

// ---- hit record ------------------------------------------------------------------------------
struct HitInfo {
    D3 p, normal;  // normal already faces the incoming ray (hit.rs:33-36)
    double u, v;
    bool front_face;
    uint32_t material;
};

// Transform::hit exit (shapes.rs:103-108) for every Transform of the chain, innermost first
__device__ inline bool hit_to_world(const SceneView& sv, uint32_t xform, HitInfo& h) {
    const Xform* x = sv.xforms + xform;
    const uint32_t n = __ldg(&x->n_chain);
    bool ok = true;
    for (uint32_t k = n; k-- > 0;) {
        XformParams p = load_xform(sv.xforms + __ldg(&x->chain[k]));
        h.p = xf_transform(p, h.p);
        D3 ns = D3{h.normal.x / p.scale.x, h.normal.y / p.scale.y, h.normal.z / p.scale.z};
        ok = unit_vector(qrotate(p.q, ns), h.normal) && ok;  // .expect("The transformed normal can't be normalized!")
    }
    return ok;
}

// Rebuild the HitRecord of a surface hit from (prim, t): the same arithmetic the intersection ran.
__device__ inline bool surface_hit_info(const SceneView& sv, uint32_t prim, double t, const RayD& world_ray, bool want_uv, HitInfo& h) {
    const PrimMeta m = sv.meta[prim];
    const uint32_t kind = m.kind_mat >> 30;
    h.material = m.kind_mat & META_MAT_MASK;
    const double* g = sv.geom[prim].d;
    const RayD r = m.xform == RT_NONE ? world_ray : ray_to_local(sv, m.xform, world_ray);
    D3 outward;
    h.p = r.o + t * r.d;  // Ray::at
    h.u = 0.0, h.v = 0.0;
    if (kind == PRIM_SPHERE) {
        D3 center = ld3(g), cvec = ld3(g + 3);
        double radius = g[6];
        D3 current_center = center + r.time * cvec;
        outward = (h.p - current_center) / radius;
        if (want_uv) sphere_uv(outward, h.u, h.v);
    } else {
        Planar pl;
        load_planar(g, pl);
        outward = pl.n;
        D3 hp = h.p - pl.q;
        h.u = dot(pl.w, cross(hp, pl.v));
        h.v = dot(pl.w, cross(pl.u, hp));
    }
    h.front_face = dot(r.d, outward) < 0.0;  // HitRecord::new, hit.rs:33-36 (in local space)
    h.normal = h.front_face ? outward : -outward;
    if (m.xform != RT_NONE) return hit_to_world(sv, m.xform, h);
    return true;
}

// RemappedMaterial::remap_record, shapes/obj.rs:32-62: texture coordinates from the face's uv frame,
// the interpolated (and optionally normal-mapped) shading normal; front_face is kept as it is
__device__ inline bool remap_record(const SceneView& sv, const Remap& rm, HitInfo& h) {
    bool ok = true;
    D3 tex_coord = ld3(rm.tex_ori) + h.u * ld3(rm.tex_u) + h.v * ld3(rm.tex_v);
    D3 n;
    ok = unit_vector((1.0 - h.u - h.v) * ld3(rm.normal[0]) + h.u * ld3(rm.normal[1]) + h.v * ld3(rm.normal[2]), n);
    if (rm.normal_tex != RT_NONE) {
        D3 c = texture_value(sv, rm.normal_tex, tex_coord.x, tex_coord.y, h.p);
        c = c * 2.0 - D3{1.0, 1.0, 1.0};
        if (!rm.has_uv_vecs) ok = false;  // .unwrap() on None
        D3 raw = ld3(rm.u_vec) * c.x + ld3(rm.v_vec) * c.y + n * c.z;
        ok = unit_vector(raw, n) && ok;
    }
    h.normal = n;
    h.u = tex_coord.x;
    h.v = tex_coord.y;
    return ok;
}

// ---- lights: Hittables::pdf_value / random over the flattened leaves (hits.rs:52-75) -----------
// STAGED: `l` is an untransformed light copied out of global memory (LeanLights)
template <bool STAGED = false>
__device__ inline double light_leaf_pdf(const SceneView& sv, const Light& l, D3 origin, D3 direction) {
    if (!STAGED && l.xform != RT_NONE) {  // Transform::pdf_value, shapes.rs:117-123, outermost Transform first
        const Xform* x = sv.xforms + l.xform;
        for (uint32_t k = 0; k < x->n_chain; k++) {
            XformParams p = load_xform(sv.xforms + x->chain[k]);
            D3 lo = xf_detransform(p, origin);
            D3 lt = xf_detransform(p, origin + direction);
            origin = lo;
            direction = lt - lo;
        }
    }
    RayD r{origin, direction, 0.0};
    const double* g = l.g.d;
    if (l.kind == PRIM_SPHERE) {  // sphere.rs:114-132
        double t;
        // own hit test on [1e-8, inf); the light record lives in global memory like any primitive
        if (!(STAGED ? sphere_hit_at(ld3(g), ld3(g + 3), g[6], r, 1e-8, INFINITY, t) : sphere_hit(g, r, 1e-8, INFINITY, t))) return 0.0;
        D3 center = ld3(g);
        double radius = g[6];
        double dist_squared = length_squared((center + 0.0 * ld3(g + 3)) - origin);
        double cos_theta_max = sqrt(1.0 - radius * radius / dist_squared);
        if (isnan(cos_theta_max)) return 1.0 / (4.0 * RT_PI);
        double solid_angle = 2.0 * RT_PI * (1.0 - cos_theta_max);
        return 1.0 / solid_angle;
    }
    // quad.rs:108-120, triangle.rs:104-113
    Planar pl;
    if (STAGED)
        load_planar_plain(g, pl);
    else
        load_planar(g, pl);
    double t, a, b2;
    if (!planar_hit_loaded(pl, l.kind == PRIM_TRIANGLE, r, 1e-8, INFINITY, t, a, b2)) return 0.0;
    double distance_squared = t * t * length_squared(direction);
    double cosine = fabs(dot(direction, pl.n) / length(direction));  // |.| makes the face-forward flip irrelevant
    return distance_squared / (cosine * l.area);
}

__device__ inline double lights_pdf_value(const SceneView& sv, uint32_t lights_flat, D3 origin, D3 direction) {
    double sum = 0.0;
    if (lights_flat) {  // a single-level list: sum / len, hits.rs:57-63
        for (uint32_t i = 0; i < sv.n_lights; i++) sum += light_leaf_pdf(sv, sv.lights[i], origin, direction);
        return sum / (double)sv.n_lights;
    }
    for (uint32_t i = 0; i < sv.n_lights; i++) sum += sv.lights[i].weight * light_leaf_pdf(sv, sv.lights[i], origin, direction);
    return sum;
}

// leaf.random(origin) in the leaf's own space
__device__ inline bool light_leaf_random(const Light& l, D3 origin, double r1, double r2, D3& dir) {
    const double* g = l.g.d;
    bool ok = true;
    if (l.kind == PRIM_SPHERE) {  // sphere.rs:134-144, 63-73
        D3 center = ld3(g);
        double radius = g[6];
        D3 direction = (center + 0.0 * ld3(g + 3)) - origin;
        double distance_squared = length_squared(direction);
        D3 ud;
        ok = unit_vector(direction, ud);
        ONB uvw;
        ok = make_onb(ud, uvw) && ok;
        double y = 1.0 + r2 * (sqrt(1.0 - radius * radius / distance_squared) - 1.0);
        double phi = 2.0 * RT_PI * r1;
        double s, c;
        sincos(phi, &s, &c);
        double x = c * sqrt(1.0 - y * y);
        double z = s * sqrt(1.0 - y * y);
        ok = unit_vector(onb_to_world(uvw, D3{x, y, z}), dir) && ok;
    } else {  // quad.rs:122-125, triangle.rs:115-128
        double ul = r1, vl = r2;
        if (l.kind == PRIM_TRIANGLE && ul + vl > 1.0) {
            double nu = 1.0 - vl, nv = 1.0 - ul;
            ul = nu, vl = nv;
        }
        D3 p = ld3(g) + (ul * ld3(g + 3)) + (vl * ld3(g + 6));
        ok = unit_vector(p - origin, dir);
    }
    return ok;
}

__device__ inline bool lights_random(const SceneView& sv, D3 origin, double pick, double r1, double r2, D3& out) {
    uint32_t leaf = sv.n_lights - 1;
    for (uint32_t i = 0; i < sv.n_lights; i++)
        if (pick < sv.lights[i].cdf) {
            leaf = i;
            break;
        }
    const Light& l = sv.lights[leaf];
    if (l.xform == RT_NONE) return light_leaf_random(l, origin, r1, r2, out);
    // Transform::random nested through the chain (shapes.rs:125-132): origins go down, directions come up
    const Xform* x = sv.xforms + l.xform;
    const uint32_t n = x->n_chain;
    D3 origins[MAX_XFORM_CHAIN + 1];
    origins[0] = origin;
    for (uint32_t k = 0; k < n; k++) origins[k + 1] = xf_detransform(load_xform(sv.xforms + x->chain[k]), origins[k]);
    D3 dir;
    bool ok = light_leaf_random(l, origins[n], r1, r2, dir);
    for (uint32_t k = n; k-- > 0;) {
        XformParams p = load_xform(sv.xforms + x->chain[k]);
        D3 world_to = xf_transform(p, origins[k + 1] + dir);
        ok = unit_vector(world_to - origins[k], dir) && ok;
    }
    out = dir;
    return ok;
}

// The same two over a staged flat list (scene_types.h, LeanLights): no Transform chain, every leaf weighs 1/n.
__device__ __forceinline__ bool lean_lights_random(const LeanLights& L, D3 origin, double pick, double r1, double r2, D3& out) {
    uint32_t leaf = L.n - 1;
    for (uint32_t i = 0; i < L.n; i++)
        if (pick < L.lights[i].cdf) {
            leaf = i;
            break;
        }
    return light_leaf_random(L.lights[leaf], origin, r1, r2, out);
}
// sum / len as lights_pdf_value (x / 1.0 == x: no division for one light)
__device__ __forceinline__ double lean_lights_pdf(const SceneView& sv, const LeanLights& L, D3 origin, D3 direction) {
    double sum = 0.0;
    for (uint32_t i = 0; i < L.n; i++) sum += light_leaf_pdf<true>(sv, L.lights[i], origin, direction);
    return L.n == 1 ? sum : sum / (double)L.n;
}

// shapes/environment.rs:14-24
__device__ inline bool background_value(const SceneView& sv, uint32_t tex, D3 dir, D3& out) {
    D3 p;
    if (!unit_vector(dir, p)) return false;
    double u = 0.0, v = 0.0;
    if (texture_needs_uv(sv, tex)) {
        double theta = acos(-p.y);
        double phi = RT_PI - atan2(-p.z, p.x);
        u = phi / (2.0 * RT_PI);
        v = theta / RT_PI;
    }
    out = texture_value(sv, tex, u, v, p);
    return true;
}

// Material::emitted through DiffuseLight / Mix nesting (material.rs:170-177, 259-267)
__device__ inline D3 material_emitted(const SceneView& sv, uint32_t mat, const HitInfo& h) {
    D3 total = D3{0.0, 0.0, 0.0};
    uint32_t st_mat[8];
    double st_w[8];
    int sp = 0;
    st_mat[sp] = mat, st_w[sp] = 1.0, sp++;
    while (sp > 0) {
        --sp;
        uint32_t m = st_mat[sp];
        double w = st_w[sp];
        while (m != RT_NONE) {
            const Material& M = sv.materials[m];
            if (M.kind == RT_MAT_DIFFUSE_LIGHT) {
                total = total + w * texture_value(sv, M.tex, h.u, h.v, h.p);
                m = M.inner;
            } else if (M.kind == RT_MAT_MIX) {
                double ratio = M.tex == RT_NONE ? M.param : (sv.textures[M.tex].a == RT_NONE ? 1.0 : (double)image_get_pixel(sv, sv.textures[M.tex].a, h.u, h.v).w);
                if (sp < 8) st_mat[sp] = M.inner2, st_w[sp] = w * ratio, sp++;
                w = w * (1.0 - ratio);
                m = M.inner;
            } else
                break;
        }
    }
    return total;
}

}  // namespace rt
