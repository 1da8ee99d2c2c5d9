// shade_step.cuh — one path segment of the wavefront: the camera ray of k_generate, and the emission, scatter, mixture-pdf
// light sampling and throughput update of one hit (camera.rs:247-325) that the shade and walk kernels run.  Kept in a header
// of its own so that tests/device_kat.cu can run the very same code one segment at a time.
#pragma once
#include "kernels.h"
#include "shade.cuh"

namespace rt {

// Camera::get_ray, camera.rs:247-273: the camera ray of stratum sidx (s_i = sidx / sqrt_spp, s_j = sidx % sqrt_spp) through
// pixel (i, j) = (pixel % image_width, pixel / image_width): jitter, defocus disk, time.  `seed` is taken by reference: k_generate
// then reads RenderParams::seed at each draw as it did with this code inline, and its machine code is unchanged.
__device__ __forceinline__ void camera_ray(const rt_camera& cam, const uint64_t& seed, uint32_t pixel, uint32_t sidx, RayD& r) {
    uint32_t i = pixel % cam.image_width, jj = pixel / cam.image_width;
    uint32_t s_i = sidx / cam.sqrt_spp, s_j = sidx % cam.sqrt_spp;
    Rand2 jit = philox_pair(seed, pixel, sidx, 0, RT_SLOT_CAM_JITTER);
    double px = (((double)s_i + jit.a) * cam.recip_sqrt_spp) - 0.5;
    double py = (((double)s_j + jit.b) * cam.recip_sqrt_spp) - 0.5;
    D3 pixel_sample = ld3(cam.pixel00_loc) + (((double)i + px) * ld3(cam.pixel_delta_u)) + (((double)jj + py) * ld3(cam.pixel_delta_v));
    if (cam.defocus_angle_in_degrees <= 0.0) {
        r.o = ld3(cam.center);
    } else {  // defocus_disk_sample, vec3.rs:63-69
        Rand2 dk = philox_pair(seed, pixel, sidx, 0, RT_SLOT_CAM_DISK);
        double theta = (2.0 * RT_PI) * dk.a;
        double rr = sqrt(dk.b);
        double s, c;
        sincos(theta, &s, &c);
        double p0 = rr * c, p1 = rr * s;
        r.o = ld3(cam.center) + (p0 * ld3(cam.defocus_disk_u)) + (p1 * ld3(cam.defocus_disk_v));
    }
    r.d = pixel_sample - r.o;
    r.time = philox_pair(seed, pixel, sidx, 0, RT_SLOT_CAM_TIME).a;
}

__device__ __forceinline__ void contribute(const RenderParams& P, const WavefrontState& W, uint32_t pixel, D3 c) {
    if (isnan(c.x) || isnan(c.y) || isnan(c.z)) {  // camera.rs:323 would panic
        atomicAdd(&W.counters->errors, 1ull);
        return;
    }
    double* a = W.accum + (size_t)pixel * 3;
    if (c.x != 0.0) atomicAdd(a + 0, c.x);
    if (c.y != 0.0) atomicAdd(a + 1, c.y);
    if (c.z != 0.0) atomicAdd(a + 2, c.z);
}

// emitted + scatter + mixture-pdf light sampling for ONE hit (camera.rs:288-321).  Returns whether the path goes on, with the
// next ray and throughput in nr / nbeta.  One instantiation per shade class: everything another class would need is compiled
// out; CLS == SC_OTHER is the fully general version (Mix, Portal, Transparent, lights that wrap a material, misses, media).
// LEAN (SC_DIFFUSE, SC_TEXTURED; scene_types.h, ShadeLean): the light list is the staged flat list `LL`, and a SC_DIFFUSE albedo
// is read straight from its solid texture.
template <uint32_t CLS, bool LEAN = false>
__device__ __forceinline__ bool shade_one(const SceneView& sv, const RenderParams& P, const WavefrontState& W, const RayD& r, D3 beta, uint32_t pixel,
                                          uint32_t sidx, uint32_t segment, double t, uint32_t prim, uint32_t kind, RayD& nr, D3& nbeta,
                                          const LeanLights* LL = nullptr) {
    static_assert(!LEAN || CLS == SC_DIFFUSE || CLS == SC_TEXTURED, "the other lean classes have their own code");
    constexpr bool GENERIC = CLS == SC_OTHER;
    constexpr bool DO_MISS = CLS == SC_MISS;
    constexpr bool DO_MEDIUM = GENERIC || CLS == SC_ISOTROPIC;
    constexpr bool DO_EMIT = GENERIC || CLS == SC_EMISSIVE || CLS == SC_DISNEY;  // Disney below DiffuseLight wrappers (the OBJ loader's `Ke`)
    constexpr bool DO_PDF = GENERIC || CLS == SC_DIFFUSE || CLS == SC_TEXTURED || CLS == SC_ISOTROPIC || CLS == SC_DISNEY;
    constexpr bool DO_REMAP = GENERIC || CLS == SC_DISNEY;
    constexpr bool DO_METAL = GENERIC || CLS == SC_METAL;
    constexpr bool DO_DIELECTRIC = GENERIC || CLS == SC_DIELECTRIC;
            bool alive = false, error = false;
            nr = r;
            nbeta = beta;

            if (DO_MISS || (GENERIC && kind == HIT_MISS)) {
                D3 bg;
                if (background_value(sv, P.cam.background_tex, r.d, bg))
                    contribute(P, W, pixel, beta * bg);
                else
                    error = true;
            } else {
                HitInfo h;
                bool hit_ok = true;
                if (DO_MEDIUM && kind == HIT_MEDIUM) {  // volume.rs:66-72, in the medium's local space
                    const Medium& med = sv.media[prim];
                    const RayD lr = med.xform == RT_NONE ? r : ray_to_local(sv, med.xform, r);
                    h.p = lr.o + t * lr.d;
                    D3 nrm = D3{1.0, 0.0, 0.0};
                    h.front_face = dot(lr.d, nrm) < 0.0;
                    h.normal = h.front_face ? nrm : -nrm;
                    h.u = 0.0, h.v = 0.0;
                    h.material = med.material;
                    if (med.xform != RT_NONE) hit_ok = hit_to_world(sv, med.xform, h);
                } else {
                    uint32_t mat = sv.meta[prim].kind_mat & META_MAT_MASK;
                    hit_ok = surface_hit_info(sv, prim, t, r, sv.materials[mat].needs_uv != 0, h);
                }
                if (!hit_ok) error = true;
                uint32_t mat = h.material;
                // RemappedMaterial is the per-face wrapper the OBJ loader puts outermost (obj.rs:165-176)
                while (DO_REMAP && sv.materials[mat].kind == RT_MAT_REMAPPED) {
                    if (!remap_record(sv, sv.remaps[sv.materials[mat].inner2], h)) error = true;
                    mat = sv.materials[mat].inner;
                }
                // emitted (camera.rs:290) — only light-carrying materials can return non-black
                uint32_t mk = sv.materials[mat].kind;
                if (DO_EMIT && (mk == RT_MAT_DIFFUSE_LIGHT || mk == RT_MAT_MIX)) {
                    D3 e = material_emitted(sv, mat, h);
                    contribute(P, W, pixel, beta * e);
                }
                // resolve DiffuseLight wrappers and Mix picks down to the scattering material
                uint32_t level = 0;
                while (DO_EMIT && mat != RT_NONE) {
                    const Material& M = sv.materials[mat];
                    if (M.kind == RT_MAT_DIFFUSE_LIGHT)
                        mat = M.inner;
                    else if (M.kind == RT_MAT_MIX) {  // material.rs:249-257
                        double ratio = M.tex == RT_NONE ? M.param
                                                        : (sv.textures[M.tex].a == RT_NONE ? 1.0 : (double)image_get_pixel(sv, sv.textures[M.tex].a, h.u, h.v).w);
                        double xi = philox_pair(P.seed, pixel, sidx, segment, RT_SLOT_MIX + 256u * level).a;
                        mat = xi > ratio ? M.inner : M.inner2;
                        level++;
                    } else
                        break;
                }
                if (mat != RT_NONE) {
                    const Material& M = sv.materials[mat];
                    nr.o = h.p;
                    // the material kinds this instantiation can meet
                    const uint32_t mkind = M.kind;
                    const bool is_metal = DO_METAL && (CLS == SC_METAL || mkind == RT_MAT_METAL);
                    const bool is_dielectric = DO_DIELECTRIC && (CLS == SC_DIELECTRIC || mkind == RT_MAT_DIELECTRIC);
                    const bool is_pdf = DO_PDF && (!GENERIC || mkind == RT_MAT_EMPTY || mkind == RT_MAT_LAMBERTIAN || mkind == RT_MAT_ISOTROPIC ||
                                                   mkind == RT_MAT_DISNEY);
                    switch (is_metal ? RT_MAT_METAL : is_dielectric ? RT_MAT_DIELECTRIC : is_pdf ? RT_MAT_LAMBERTIAN : (GENERIC ? mkind : 0xFFFFu)) {
                        case RT_MAT_METAL: {  // material.rs:82-95
                            D3 ud, ur;
                            if (unit_vector(r.d, ud) && unit_vector(reflect(ud, h.normal), ur)) {
                                Rand2 xi = philox_pair(P.seed, pixel, sidx, segment, RT_SLOT_MATERIAL);
                                nr.d = ur + (M.param * random_unit_vector(xi.a, xi.b));
                                nbeta = beta * ld3(M.color);
                                alive = true;
                            }
                            break;
                        }
                        case RT_MAT_DIELECTRIC: {  // material.rs:117-144
                            double ri = h.front_face ? 1.0 / M.param : M.param;
                            D3 ud;
                            if (!unit_vector(r.d, ud)) {
                                error = true;
                                break;
                            }
                            double cos_theta = rmin(dot(-ud, h.normal), 1.0);
                            double sin_theta = sqrt(1.0 - cos_theta * cos_theta);
                            bool cannot_refract = ri * sin_theta > 1.0;
                            double r0 = (1.0 - ri) / (1.0 + ri);
                            double r0s = r0 * r0;
                            double x = 1.0 - cos_theta;
                            double x2 = x * x;
                            double reflectance = r0s + (1.0 - r0s) * (x * (x2 * x2));
                            D3 dir;
                            if (cannot_refract || reflectance > philox_pair(P.seed, pixel, sidx, segment, RT_SLOT_MATERIAL).a) {
                                dir = reflect(ud, h.normal);
                            } else if (!refract(ud, h.normal, ri, dir)) {
                                error = true;
                                break;
                            }
                            nr.d = dir;
                            nbeta = beta * texture_value(sv, M.tex, h.u, h.v, h.p);
                            alive = true;
                            break;
                        }
                        case RT_MAT_TRANSPARENT:  // material.rs:211-218
                            alive = GENERIC;
                            break;
                        case RT_MAT_PORTAL: {  // material/portal.rs:21-30
                            if (!GENERIC) break;
                            nr.o = h.p + ld3(M.v);
                            // quaternion sandwich product, quaternion.rs:72-104
                            double qw = M.v[3], qx = M.v[4], qy = M.v[5], qz = M.v[6];
                            double aw = qw * 0.0 - qx * r.d.x - qy * r.d.y - qz * r.d.z;
                            double ax = qw * r.d.x + qx * 0.0 + qy * r.d.z - qz * r.d.y;
                            double ay = qw * r.d.y - qx * r.d.z + qy * 0.0 + qz * r.d.x;
                            double az = qw * r.d.z + qx * r.d.y - qy * r.d.x + qz * 0.0;
                            double cx = -qx, cy = -qy, cz = -qz;
                            nr.d.x = aw * cx + ax * qw + ay * cz - az * cy;
                            nr.d.y = aw * cy - ax * cz + ay * qw + az * cx;
                            nr.d.z = aw * cz + ax * cy - ay * cx + az * qw;
                            nbeta = beta * ld3(M.color);
                            alive = true;
                            break;
                        }
                        case RT_MAT_LAMBERTIAN: {  // Empty / Lambertian / Isotropic / Disney
                            // ScatterRecord::PDF branch, camera.rs:297-312
                            const bool iso = CLS == SC_ISOTROPIC || (GENERIC && M.kind == RT_MAT_ISOTROPIC);
                            const bool dis = CLS == SC_DISNEY || (GENERIC && M.kind == RT_MAT_DISNEY);
                            D3 albedo = (M.kind == RT_MAT_EMPTY || dis)  ? D3{0.75, 0.75, 0.75}
                                        : (LEAN && CLS == SC_DIFFUSE) ? ld3(sv.textures[M.tex].color)  // texture_value of a solid texture
                                                                      : texture_value(sv, M.tex, h.u, h.v, h.p);
                            ONB uvw;
                            if (!iso && !make_onb(h.normal, uvw)) {
                                error = true;
                                break;
                            }
                            disney::Params DP;
                            D3 v_out_l = D3{0.0, 1.0, 0.0};
                            if (dis) {  // Disney::scatter + DisneyPDF::new, disney.rs:71-91, 522-538
                                DP.base_color = M.tex == RT_NONE ? ld3(M.color) : texture_value(sv, M.tex, h.u, h.v, h.p);
                                DP.roughness = M.v[RT_DISNEY_ROUGHNESS], DP.anisotropic = M.v[RT_DISNEY_ANISOTROPIC], DP.sheen = M.v[RT_DISNEY_SHEEN];
                                DP.sheen_tint = M.v[RT_DISNEY_SHEEN_TINT], DP.clearcoat = M.v[RT_DISNEY_CLEARCOAT];
                                DP.clearcoat_gloss = M.v[RT_DISNEY_CLEARCOAT_GLOSS], DP.specular_tint = M.v[RT_DISNEY_SPECULAR_TINT];
                                DP.metallic = M.v[RT_DISNEY_METALLIC], DP.ior = M.v[RT_DISNEY_IOR], DP.flatness = M.v[RT_DISNEY_FLATNESS];
                                DP.spec_trans = M.v[RT_DISNEY_SPEC_TRANS], DP.diff_trans = M.v[RT_DISNEY_DIFF_TRANS], DP.thin = M.v[RT_DISNEY_THIN] != 0.0;
                                D3 vo;
                                if (!unit_vector(-r.d, vo)) {
                                    error = true;
                                    break;
                                }
                                v_out_l = D3{dot(vo, uvw.u), dot(vo, uvw.v), dot(vo, uvw.w)};  // world_to_onb, onb.rs:40-45
                            }
                            Rand2 pick = philox_pair(P.seed, pixel, sidx, segment, RT_SLOT_MIXTURE);
                            Rand2 dx = philox_pair(P.seed, pixel, sidx, segment, RT_SLOT_DIRECTION);
                            D3 gen = D3{0.0, 0.0, 0.0};
                            const bool have_lights = LEAN ? LL->n > 0 : sv.n_lights > 0;
                            // No `break` inside the divergent sampling branch below: with an early-exit edge the warp would
                            // only reconverge at the end of the switch and run the whole pdf evaluation once per side
                            // (measured: 16 of 32 lanes active from here on).  stop: 1 = the reference panics, 2 = None (black).
                            int stop = 0;
                            if (have_lights && !(pick.a < 0.5)) {
                                if (!(LEAN ? lean_lights_random(*LL, h.p, pick.b, dx.a, dx.b, gen) : lights_random(sv, h.p, pick.b, dx.a, dx.b, gen))) stop = 1;
                            } else if (dis) {
                                Rand2 dpick = philox_pair(P.seed, pixel, sidx, segment, RT_SLOT_DISNEY);
                                D3 v_in_l;
                                bool derr = false;
                                if (!disney::generate_local(DP, v_out_l, h.front_face, dpick, dx, v_in_l, derr))
                                    stop = derr ? 1 : 2;  // None: black (camera.rs:313-315)
                                else if (!unit_vector(onb_to_world(uvw, v_in_l), gen))
                                    stop = 1;
                            } else {
                                gen = iso ? random_unit_vector(dx.a, dx.b) : onb_to_world(uvw, random_cosine_direction(dx.a, dx.b));
                            }
                            // PDF::value, pdf.rs:22-29, 51-57, disney.rs:656-666
                            D3 axp = D3{0.0, 0.0, 0.0};
                            double value0 = 0.0;
                            if (!stop) {
                                if (iso) {
                                    value0 = 1.0 / (4.0 * RT_PI);
                                    axp = albedo / (4.0 * RT_PI);
                                } else {
                                    D3 ud;
                                    if (!unit_vector(gen, ud)) {
                                        stop = 1;
                                    } else if (dis) {
                                        D3 v_in_l = D3{dot(ud, uvw.u), dot(ud, uvw.v), dot(ud, uvw.w)};
                                        bool derr = false;
                                        disney::evaluate_disney(DP, v_out_l, v_in_l, h.front_face, axp, value0, derr);
                                        if (derr) stop = 1;
                                    } else {
                                        double cosine_theta = dot(ud, uvw.v);
                                        value0 = rmax(0.0, cosine_theta / RT_PI);
                                        axp = albedo * rmax(cosine_theta, 0.0) / RT_PI;
                                    }
                                }
                            }
                            double pdf_val = value0;
                            if (!stop && have_lights) {
                                double value1 = LEAN ? lean_lights_pdf(sv, *LL, h.p, gen) : lights_pdf_value(sv, P.lights_flat, h.p, gen);
                                if (isnan(value1) || (value0 == 0.0 && value1 == 0.0))  // hits.rs:64, pdf.rs:105-109
                                    stop = 1;
                                else
                                    pdf_val = value0 * 0.5 + value1 * 0.5;
                            }
                            if (!stop && pdf_val == 0.0) stop = 1;  // camera.rs:309
                            if (!stop) {
                                nr.d = gen;
                                nbeta = beta * (axp / pdf_val);
                                alive = true;
                            }
                            if (stop == 1) error = true;
                            break;
                        }
                        default: break;
                    }
                }
            }
            if (error) {
                atomicAdd(&W.counters->errors, 1ull);
                alive = false;
            }
            // a zero throughput can never contribute again; depth == 0 returns black (camera.rs:282)
            if (alive && (segment + 1 >= P.cam.max_depth || (nbeta.x == 0.0 && nbeta.y == 0.0 && nbeta.z == 0.0))) alive = false;
            return alive;
}

// shade_one<SC_ISOTROPIC> at the scatter point r.at(t) of a medium below no Transform whose Isotropic has a solid albedo
// (axp = albedo / (4 pi)), over a staged flat light list: the same operations in the same order, without the normal, uv, ONB and
// texture lookup a solid Isotropic does not use.  Returns whether the path goes on (nr, nbeta).  Used by k_shade<SC_ISOTROPIC, true>
// and by every segment of the lean k_walk.
__device__ __forceinline__ bool lean_isotropic_scatter(const SceneView& sv, const LeanLights& L, D3 axp, const RenderParams& P, const WavefrontState& W,
                                                       const RayD& r, D3 beta, uint32_t pixel, uint32_t sidx, uint32_t segment, double t, RayD& nr,
                                                       D3& nbeta) {
    nr.o = r.o + t * r.d;  // volume.rs:66-72 (h.p)
    nr.time = r.time;
    const Rand2 pick = philox_pair(P.seed, pixel, sidx, segment, RT_SLOT_MIXTURE);
    const Rand2 dx = philox_pair(P.seed, pixel, sidx, segment, RT_SLOT_DIRECTION);
    D3 gen = D3{0.0, 0.0, 0.0};
    bool panic = false;  // shade_one's stop == 1 (None cannot occur here)
    if (L.n > 0 && !(pick.a < 0.5))
        panic = !lean_lights_random(L, nr.o, pick.b, dx.a, dx.b, gen);
    else
        gen = random_unit_vector(dx.a, dx.b);
    const double value0 = 1.0 / (4.0 * RT_PI);
    double pdf_val = value0;
    if (!panic && L.n > 0) {
        const double value1 = lean_lights_pdf(sv, L, nr.o, gen);
        if (isnan(value1) || (value0 == 0.0 && value1 == 0.0))
            panic = true;
        else
            pdf_val = value0 * 0.5 + value1 * 0.5;
    }
    if (panic || pdf_val == 0.0) {
        atomicAdd(&W.counters->errors, 1ull);
        return false;
    }
    nr.d = gen;
    nbeta = beta * (axp / pdf_val);
    return !(segment + 1 >= P.cam.max_depth || (nbeta.x == 0.0 && nbeta.y == 0.0 && nbeta.z == 0.0));
}

}  // namespace rt
