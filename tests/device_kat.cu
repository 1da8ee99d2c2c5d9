// device_kat.cu — TEST INFRASTRUCTURE ONLY, not part of the product (tests/device_kat.py builds it on first use).
//
// Known-answer harness for the device shading functions: every function of shade.cuh / disney.cuh that the shade kernels call
// gets one thin __global__ wrapper (one element per thread, arrays in, arrays out, plus its ok / error flag), so that
// tests/test_device_kat.py can feed it the oracle's own inputs and compare the numbers one call at a time.  The wrappers call
// the product's header code; there is no second copy of the arithmetic here.  The scene tables come from the product's scene
// compiler (compile_scene), uploaded with plain cudaMalloc / cudaMemcpy.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "kernels.h"  // before shade.cuh: traverse.cuh needs its macros
#include "shade.cuh"
#include "shade_step.cuh"
#include "compile.h"

using namespace rt;

namespace {

thread_local std::string g_err;

int fail(const std::string& e) {
    g_err = e;
    return -1;
}

struct KatScene {
    SceneView sv{};
    uint32_t lights_flat = 1;
    bool has_lean = false;
    LeanLights lean{};
    const ShadeLean* d_shade_lean = nullptr;  // the scene's ShadeLean / WalkLean records on the device, or nullptr
    const WalkLean* d_walk_lean = nullptr;
    uint32_t shade_lean_mask = 0, walk_thick = RT_NONE;
    std::vector<uint32_t> prim_class;  // device primitive -> its compiled shade class (PrimMeta::kind_mat bits 26..29)
    std::vector<Medium> media;
    std::vector<uint32_t> prim_of_object;  // object id -> device primitive index (meta[].object), RT_NONE elsewhere
    uint32_t n_textures = 0, n_materials = 0, n_remaps = 0;
    std::vector<void*> allocs;
    ~KatScene() {
        for (void* p : allocs) cudaFree(p);
    }
    template <class T, class V>
    const T* put(const V& v) {
        if (v.empty()) return nullptr;
        void* d = nullptr;
        if (cudaMalloc(&d, v.size() * sizeof(T)) != cudaSuccess) throw std::string("cudaMalloc failed");
        allocs.push_back(d);
        if (cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess) throw std::string("cudaMemcpy failed");
        return (const T*)d;
    }
};

// device buffers of one call: inputs copied in, outputs copied back
struct Buffers {
    std::vector<void*> p;
    ~Buffers() {
        for (void* x : p) cudaFree(x);
    }
    template <class T>
    T* in(const T* h, size_t n) {
        void* d = nullptr;
        if (cudaMalloc(&d, n * sizeof(T) + 16) != cudaSuccess) throw std::string("cudaMalloc failed");
        p.push_back(d);
        if (n && cudaMemcpy(d, h, n * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess) throw std::string("cudaMemcpy failed");
        return (T*)d;
    }
    template <class T>
    T* out(size_t n) {
        void* d = nullptr;
        if (cudaMalloc(&d, n * sizeof(T) + 16) != cudaSuccess) throw std::string("cudaMalloc failed");
        p.push_back(d);
        return (T*)d;
    }
};

template <class T>
void fetch(T* h, const T* d, size_t n) {
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) throw std::string("kernel: ") + cudaGetErrorString(e);
    if (n && cudaMemcpy(h, d, n * sizeof(T), cudaMemcpyDeviceToHost) != cudaSuccess) throw std::string("cudaMemcpy failed");
}

// 0, or -1 with kat_last_error() set
template <class F>
int guarded(F f) {
    try {
        f();
        return 0;
    } catch (const std::string& e) {
        return fail(e);
    }
}

// every index a wrapper dereferences is checked on the host first: a bad argument is an error, not a device fault
void check_indices(const uint32_t* idx, int n, uint32_t limit, const char* what) {
    for (int i = 0; i < n; i++)
        if (idx[i] >= limit) throw std::string(what) + " index out of range";
}

constexpr int BLOCK = 128;
inline int grid(int n) { return (n + BLOCK - 1) / BLOCK; }

__device__ __forceinline__ void st3(double* o, D3 v) { o[0] = v.x, o[1] = v.y, o[2] = v.z; }

// params15: base_color(3) roughness anisotropic sheen sheen_tint clearcoat clearcoat_gloss specular_tint metallic ior flatness
// spec_trans diff_trans (the order of orc_kat_disney_evaluate)
__device__ disney::Params disney_params(const double* p, int thin) {
    disney::Params P;
    P.base_color = ld3(p);
    P.roughness = p[3], P.anisotropic = p[4], P.sheen = p[5], P.sheen_tint = p[6], P.clearcoat = p[7], P.clearcoat_gloss = p[8];
    P.specular_tint = p[9], P.metallic = p[10], P.ior = p[11], P.flatness = p[12], P.spec_trans = p[13], P.diff_trans = p[14];
    P.thin = thin != 0;
    return P;
}

// ---- wrappers ---------------------------------------------------------------------------------
// out5: reflectance(3), forward pdf, error
__global__ void k_disney_evaluate(const double* params15, int thin, const double* v_out, const double* v_in, const int* front_face, int n, double* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const disney::Params P = disney_params(params15, thin);
    D3 r;
    double pdf;
    bool err = false;
    disney::evaluate_disney(P, ld3(v_out + 3 * i), ld3(v_in + 3 * i), front_face[i] != 0, r, pdf, err);
    st3(out + 5 * i, r);
    out[5 * i + 3] = pdf, out[5 * i + 4] = err ? 1.0 : 0.0;
}

// generate_local, then shade_one's normalisation with an identity basis.  out4: direction(3), rc (1 Some, 0 None, -1 panic)
__global__ void k_disney_generate(const double* params15, int thin, const double* v_out, const int* front_face, const double* pick2, const double* u2, int n,
                                  double* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const disney::Params P = disney_params(params15, thin);
    const ONB id{D3{1.0, 0.0, 0.0}, D3{0.0, 1.0, 0.0}, D3{0.0, 0.0, 1.0}};
    D3 v_in_l = D3{0.0, 0.0, 0.0}, gen = D3{0.0, 0.0, 0.0};
    bool derr = false;
    double rc;
    if (!disney::generate_local(P, ld3(v_out + 3 * i), front_face[i] != 0, Rand2{pick2[2 * i], pick2[2 * i + 1]}, Rand2{u2[2 * i], u2[2 * i + 1]}, v_in_l, derr))
        rc = derr ? -1.0 : 0.0;
    else
        rc = unit_vector(onb_to_world(id, v_in_l), gen) ? 1.0 : -1.0;
    st3(out + 4 * i, gen);
    out[4 * i + 3] = rc;
}

// in5: u, v, p(3); out3
__global__ void k_texture_value(SceneView sv, const uint32_t* tex, const double* in, int n, double* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    st3(out + 3 * i, texture_value(sv, tex[i], in[5 * i], in[5 * i + 1], ld3(in + 5 * i + 2)));
}

// out4: colour(3), ok
__global__ void k_background_value(SceneView sv, uint32_t tex, const double* dir, int n, double* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    D3 c = D3{0.0, 0.0, 0.0};
    bool ok = background_value(sv, tex, ld3(dir + 3 * i), c);
    st3(out + 4 * i, c);
    out[4 * i + 3] = ok ? 1.0 : 0.0;
}

// hit record: p(3) normal(3) u v front_face ok material = 11 doubles
__device__ void st_hit(double* o, const HitInfo& h, bool ok) {
    st3(o, h.p), st3(o + 3, h.normal);
    o[6] = h.u, o[7] = h.v, o[8] = h.front_face ? 1.0 : 0.0, o[9] = ok ? 1.0 : 0.0, o[10] = (double)h.material;
}

__global__ void k_surface_hit_info(SceneView sv, const uint32_t* prim, const double* t, const rt_ray* rays, int n, double* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    RayD r;
    r.o = ld3(rays[i].origin), r.d = ld3(rays[i].direction), r.time = rays[i].time;
    HitInfo h{};
    bool ok = surface_hit_info(sv, prim[i], t[i], r, true, h);
    st_hit(out + 11 * i, h, ok);
}

// in9: p(3) normal(3) u v front_face -> the remapped record
__global__ void k_remap_record(SceneView sv, const uint32_t* remap, const double* in, int n, double* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    HitInfo h{};
    h.p = ld3(in + 9 * i), h.normal = ld3(in + 9 * i + 3), h.u = in[9 * i + 6], h.v = in[9 * i + 7], h.front_face = in[9 * i + 8] != 0.0;
    h.material = RT_NONE;
    bool ok = remap_record(sv, sv.remaps[remap[i]], h);
    st_hit(out + 11 * i, h, ok);
}

__global__ void k_lights_pdf(SceneView sv, uint32_t lights_flat, const LeanLights* lean, const double* origin, const double* dir, int n, double* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = lean ? lean_lights_pdf(sv, *lean, ld3(origin + 3 * i), ld3(dir + 3 * i)) : lights_pdf_value(sv, lights_flat, ld3(origin + 3 * i), ld3(dir + 3 * i));
}

// in3: pick, r1, r2; out4: direction(3), ok
__global__ void k_lights_random(SceneView sv, const LeanLights* lean, const double* origin, const double* in, int n, double* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    D3 d = D3{0.0, 0.0, 0.0};
    const double* x = in + 3 * i;
    bool ok = lean ? lean_lights_random(*lean, ld3(origin + 3 * i), x[0], x[1], x[2], d) : lights_random(sv, ld3(origin + 3 * i), x[0], x[1], x[2], d);
    st3(out + 4 * i, d);
    out[4 * i + 3] = ok ? 1.0 : 0.0;
}

// in5: u, v, p(3); out3
__global__ void k_material_emitted(SceneView sv, const uint32_t* mat, const double* in, int n, double* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    HitInfo h{};
    h.u = in[5 * i], h.v = in[5 * i + 1], h.p = ld3(in + 5 * i + 2);
    st3(out + 3 * i, material_emitted(sv, mat[i], h));
}

// The box test of every traversal: make_rayf + slab (traverse.cuh).  The binary64 interval bounds are converted the way the
// traversal converts them - t_min rounded down, t_max rounded up to binary32 - so a caller passes the query's own bounds.
// in8: o(3) d(3) t_min t_max; box6: lo(3) hi(3); out: 1 when the box is kept
__global__ void k_slab(const double* in, const float* box, int n, uint8_t* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double* x = in + 8 * i;
    RayD r;
    r.o = ld3(x), r.d = ld3(x + 3), r.time = 0.0;
    RayF f;
    make_rayf(r, f, false);
    float tnear;
    out[i] = slab(f, box + 6 * i, box + 6 * i + 3, __double2float_rd(x[6]), __double2float_ru(x[7]), tnear) ? 1 : 0;
}

// medium_free_flight (traverse.cuh) with the medium's ray direction d.  in7: t1 t2 d(3) neg_inv_density xi; out2: ok, tm
__global__ void k_medium_free_flight(const double* in, int n, double* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double* x = in + 7 * i;
    RayD lr;
    lr.o = D3{0.0, 0.0, 0.0}, lr.d = ld3(x + 2), lr.time = 0.0;
    double tm = 0.0;
    const bool ok = medium_free_flight(x[0], x[1], lr, x[5], x[6], tm);
    out[2 * i] = ok ? 1.0 : 0.0, out[2 * i + 1] = tm;
}

// free_flight_overshoots (traverse.cuh).  in6: neg_inv_density xi t d(3); out: 1 when the screen says the free flight overshoots t
__global__ void k_free_flight_overshoots(const double* in, int n, uint8_t* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double* x = in + 6 * i;
    out[i] = free_flight_overshoots(x[0], x[1], x[2], ld3(x + 3)) ? 1 : 0;
}


// One path segment (shade_step.cuh) per element.  in (rays): the ray; in4: beta(3), t; ids6: pixel, sample, segment, prim, kind,
// max_depth; seeds.  out16: the contribution added to the element's own zeroed accumulator(3), next ray o(3) d(3) time, nbeta(3),
// alive, change of the error counter, unused.  LEAN: 0 = shade_one<CLS>; 1 = the lean kernels' code with the ShadeLean record
// (shade_one<CLS, true>, or lean_isotropic_scatter with axp[prim] for SC_ISOTROPIC); 2 = lean_isotropic_scatter with the WalkLean
// record (the lean walk's segment).  nr and nbeta start as the ray and beta, as shade_one sets them.
template <uint32_t CLS, int LEAN>
__global__ void k_shade_step(SceneView sv, RenderParams P0, const ShadeLean* SL, const WalkLean* WL, const rt_ray* rays, const double* in4,
                             const uint32_t* ids6, const uint64_t* seeds, int n, double* acc3, Counters* counters, double* out16) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t* id = ids6 + 6 * i;
    RenderParams P = P0;
    P.seed = seeds[i], P.cam.max_depth = id[5];
    // contribute() adds at accum + 3 * pixel: point accum so that this lands on the element's own three doubles (address
    // arithmetic on integers, the pixel index may be any 28-bit value)
    WavefrontState W{};
    W.accum = reinterpret_cast<double*>(reinterpret_cast<uintptr_t>(acc3 + 3 * (size_t)i) - (uintptr_t)id[0] * 3u * sizeof(double));
    W.counters = counters + i;
    RayD r;
    r.o = ld3(rays[i].origin), r.d = ld3(rays[i].direction), r.time = rays[i].time;
    const D3 beta = ld3(in4 + 4 * i);
    const double t = in4[4 * i + 3];
    RayD nr = r;
    D3 nbeta = beta;
    bool alive;
    if constexpr (LEAN == 2)
        alive = lean_isotropic_scatter(sv, WL->lights, ld3(WL->axp), P, W, r, beta, id[0], id[1], id[2], t, nr, nbeta);
    else if constexpr (LEAN == 1 && CLS == SC_ISOTROPIC)
        alive = lean_isotropic_scatter(sv, SL->lights, ld3(SL->axp[id[3]]), P, W, r, beta, id[0], id[1], id[2], t, nr, nbeta);
    else
        alive = shade_one<CLS, LEAN == 1>(sv, P, W, r, beta, id[0], id[1], id[2], t, id[3], id[4], nr, nbeta, LEAN ? &SL->lights : nullptr);
    double* o = out16 + 16 * i;
    st3(o, nr.o), st3(o + 3, nr.d);
    o[6] = nr.time;
    st3(o + 7, nbeta);
    o[10] = alive ? 1.0 : 0.0;
    o[11] = (double)counters[i].errors;
    o[12] = o[13] = o[14] = o[15] = 0.0;
}

// k_generate's camera ray: camera_ray(cam, seed, j * image_width + i, sidx).  in3: i, j, sidx
__global__ void k_camera_ray(rt_camera cam, uint64_t seed, const uint32_t* in3, int n, rt_ray* out) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const uint32_t* x = in3 + 3 * k;
    RayD r;
    camera_ray(cam, seed, x[1] * cam.image_width + x[0], x[2], r);
    st3(out[k].origin, r.o), st3(out[k].direction, r.d);
    out[k].time = r.time;
}

template <uint32_t CLS, int LEAN>
void launch_shade_step(const KatScene& s, const RenderParams& P, Buffers& b, const rt_ray* rays, const double* in4, const uint32_t* ids6,
                       const uint64_t* seeds, int n, double* out16) {
    double* d_acc = b.out<double>(3 * (size_t)n);
    Counters* d_cnt = b.out<Counters>(n);
    if (cudaMemset(d_acc, 0, 3 * (size_t)n * sizeof(double)) != cudaSuccess || cudaMemset(d_cnt, 0, (size_t)n * sizeof(Counters)) != cudaSuccess)
        throw std::string("cudaMemset failed");
    double* d_out = b.out<double>(16 * (size_t)n);
    k_shade_step<CLS, LEAN><<<grid(n), BLOCK>>>(s.sv, P, s.d_shade_lean, s.d_walk_lean, b.in(rays, n), b.in(in4, 4 * (size_t)n), b.in(ids6, 6 * (size_t)n),
                                                b.in(seeds, n), n, d_acc, d_cnt, d_out);
    fetch(out16, d_out, 16 * (size_t)n);
    std::vector<double> acc(3 * (size_t)n);
    fetch(acc.data(), d_acc, acc.size());
    for (int i = 0; i < n; i++) out16[16 * i + 12] = acc[3 * i], out16[16 * i + 13] = acc[3 * i + 1], out16[16 * i + 14] = acc[3 * i + 2];
}

}  // namespace

// ---- C entry points (ctypes, tests/device_kat.py) -------------------------------------------------
extern "C" {

const char* kat_last_error() { return g_err.c_str(); }

// compile_scene (flags 0) and upload the tables the shading functions read
void* kat_scene_create(const rt_scene_desc* desc) {
    KatScene* s = new KatScene();
    try {
        CompiledScene cs;
        std::string err;
        int rc = compile_scene(*desc, 0, cs, err);
        if (rc != RT_OK) throw "compile_scene: " + err;
        SceneView& v = s->sv;
        v.geom = s->put<PrimGeom>(cs.geom), v.meta = s->put<PrimMeta>(cs.meta), v.xforms = s->put<Xform>(cs.xforms);
        v.materials = s->put<Material>(cs.materials), v.textures = s->put<Texture>(cs.textures), v.images = s->put<Image>(cs.images);
        v.texels = s->put<float4>(cs.texels), v.perlins = s->put<Perlin>(cs.perlins), v.media = s->put<Medium>(cs.media);
        v.lights = s->put<Light>(cs.lights), v.remaps = s->put<Remap>(cs.remaps);
        v.n_media = (uint32_t)cs.media.size(), v.n_lights = (uint32_t)cs.lights.size(), v.n_prims = (uint32_t)cs.geom.size();
        v.n_xforms = (uint32_t)cs.xforms.size();
        // the rule of rt_scene_create (api.cu, "lights is flat"): every leaf has the same weight 1/n
        s->lights_flat = 1;
        for (auto& l : cs.lights)
            if (l.weight != 1.0 / (double)cs.lights.size()) s->lights_flat = 0;
        // the staged list of the lean kernels, when the scene's light list qualifies for one
        if (!cs.shade_lean.empty() && (cs.shade_lean_mask & (1u << SC_DIFFUSE)))
            s->lean = cs.shade_lean[0].lights, s->has_lean = true;
        else if (!cs.walk_lean.empty())
            s->lean = cs.walk_lean[0].lights, s->has_lean = true;
        s->n_textures = (uint32_t)cs.textures.size(), s->n_materials = (uint32_t)cs.materials.size(), s->n_remaps = (uint32_t)cs.remaps.size();
        s->d_shade_lean = s->put<ShadeLean>(cs.shade_lean), s->d_walk_lean = s->put<WalkLean>(cs.walk_lean);
        s->shade_lean_mask = cs.shade_lean.empty() ? 0u : cs.shade_lean_mask;
        s->walk_thick = cs.walk_lean.empty() ? RT_NONE : cs.walk_lean[0].thick;
        for (auto& m : cs.meta) s->prim_class.push_back((m.kind_mat >> META_CLASS_SHIFT) & 15u);
        s->media = cs.media;
        s->prim_of_object.assign(desc->n_objects, RT_NONE);
        for (size_t p = 0; p < cs.meta.size(); p++) s->prim_of_object[cs.meta[p].object] = (uint32_t)p;
        return s;
    } catch (const std::string& e) {
        g_err = e;
    } catch (const std::exception& e) {
        g_err = e.what();
    }
    delete s;
    return nullptr;
}
void kat_scene_destroy(void* s) { delete (KatScene*)s; }

// info: n_lights, lights_flat, has_lean, lean n, n_prims
void kat_scene_info(const void* h, uint32_t* out5) {
    const KatScene& s = *(const KatScene*)h;
    out5[0] = s.sv.n_lights, out5[1] = s.lights_flat, out5[2] = s.has_lean, out5[3] = s.has_lean ? s.lean.n : 0, out5[4] = s.sv.n_prims;
}
// device primitive index of every object id (RT_NONE for containers)
void kat_prim_of_object(const void* h, uint32_t* out, uint32_t n) {
    const KatScene& s = *(const KatScene*)h;
    for (uint32_t i = 0; i < n && i < s.prim_of_object.size(); i++) out[i] = s.prim_of_object[i];
}

// Host only (no device needed): every light leaf of the compiled scene - kind, Transform chain id, weight, cdf.
// Returns the number of leaves (at most cap are written) or -1.
int kat_light_table(const rt_scene_desc* desc, uint32_t* kind, uint32_t* xform, double* weight, double* cdf, uint32_t cap) {
    CompiledScene cs;
    std::string err;
    if (compile_scene(*desc, 0, cs, err) != RT_OK) return fail("compile_scene: " + err);
    for (size_t i = 0; i < cs.lights.size() && i < cap; i++)
        kind[i] = cs.lights[i].kind, xform[i] = cs.lights[i].xform, weight[i] = cs.lights[i].weight, cdf[i] = cs.lights[i].cdf;
    return (int)cs.lights.size();
}

// lean_info: shade_lean_mask (0 without a ShadeLean record), has WalkLean, the WalkLean thick medium (RT_NONE), n_media
void kat_scene_lean_info(const void* h, uint32_t* out4) {
    const KatScene& s = *(const KatScene*)h;
    out4[0] = s.shade_lean_mask, out4[1] = s.d_walk_lean != nullptr, out4[2] = s.walk_thick, out4[3] = (uint32_t)s.media.size();
}
// the compiled shade class of every device primitive (PrimMeta::kind_mat bits 26..29)
void kat_prim_class(const void* h, uint32_t* out, uint32_t n) {
    const KatScene& s = *(const KatScene*)h;
    for (uint32_t i = 0; i < n && i < s.prim_class.size(); i++) out[i] = s.prim_class[i];
}
// every medium: object id of its ConstantMedium, flags (MEDIUM_THICK), Transform chain (RT_NONE: none)
void kat_media(const void* h, uint32_t* object, uint32_t* flags, uint32_t* xform, uint32_t n) {
    const KatScene& s = *(const KatScene*)h;
    for (uint32_t i = 0; i < n && i < s.media.size(); i++) object[i] = s.media[i].object, flags[i] = s.media[i].flags, xform[i] = s.media[i].xform;
}

// One segment per element through shade_one<cls> (lean 0), the lean shade kernels' code (lean 1: classes SC_DIFFUSE, SC_TEXTURED,
// SC_ISOTROPIC) or the lean walk's lean_isotropic_scatter (lean 2).  out16 per element: next ray o(3) d(3) time, nbeta(3), alive,
// errors, contribution(3), unused.
int kat_shade_step(const void* h, const rt_camera* cam, uint32_t cls, int lean, const rt_ray* rays, const double* in4,
                   const uint32_t* ids6, const uint64_t* seeds, int n, double* out16) {
    const KatScene& s = *(const KatScene*)h;
    if (lean == 1 && !(s.shade_lean_mask & (1u << cls))) return fail("class " + std::to_string(cls) + " is not lean in this scene");
    if (lean == 2 && (!s.d_walk_lean || cls != SC_ISOTROPIC)) return fail("the scene has no lean walk");
    if (lean < 0 || lean > 2) return fail("bad lean");
    return guarded([&] {
        for (int i = 0; i < n; i++) {
            const uint32_t* id = ids6 + 6 * i;
            const bool medium = id[4] == HIT_MEDIUM, surface = id[4] == HIT_SURFACE;
            if (id[4] > HIT_MEDIUM || (surface && id[3] >= s.sv.n_prims) || (medium && id[3] >= s.sv.n_media)) throw std::string("primitive index out of range");
            if (id[0] >= (1u << IDS_PIXEL_BITS) || id[1] >= (1u << IDS_SAMPLE_BITS) || id[2] >= (1u << IDS_SEGMENT_BITS)) throw std::string("path id out of range");
            // the hit kinds each instantiation reads: a miss has no primitive, a medium index is no primitive index
            if (id[4] == HIT_MISS && cls != SC_MISS && cls != SC_OTHER) throw std::string("a miss goes to SC_MISS or SC_OTHER");
            if (id[4] != HIT_MISS && cls == SC_MISS) throw std::string("SC_MISS only shades misses");
            if (medium && cls != SC_ISOTROPIC && cls != SC_OTHER) throw std::string("a medium hit goes to SC_ISOTROPIC or SC_OTHER");
            if (lean == 2 && !(medium && id[3] == s.walk_thick)) throw std::string("the lean walk only scatters in its thick medium");
            if (lean == 1 && cls == SC_ISOTROPIC && !(medium && id[3] < SHADE_LEAN_MEDIA)) throw std::string("lean isotropic: not a medium");
        }
        RenderParams P{};
        P.cam = *cam;
        P.lights_flat = s.lights_flat;
        Buffers b;
        switch (cls * 4 + (uint32_t)lean) {
#define RT_KAT_CLS(C)                                                                     \
    case C * 4: launch_shade_step<C, 0>(s, P, b, rays, in4, ids6, seeds, n, out16); break;
            RT_KAT_CLS(SC_MISS) RT_KAT_CLS(SC_DIFFUSE) RT_KAT_CLS(SC_TEXTURED) RT_KAT_CLS(SC_ISOTROPIC) RT_KAT_CLS(SC_METAL)
            RT_KAT_CLS(SC_DIELECTRIC) RT_KAT_CLS(SC_EMISSIVE) RT_KAT_CLS(SC_DISNEY) RT_KAT_CLS(SC_OTHER)
#undef RT_KAT_CLS
            case SC_DIFFUSE * 4 + 1: launch_shade_step<SC_DIFFUSE, 1>(s, P, b, rays, in4, ids6, seeds, n, out16); break;
            case SC_TEXTURED * 4 + 1: launch_shade_step<SC_TEXTURED, 1>(s, P, b, rays, in4, ids6, seeds, n, out16); break;
            case SC_ISOTROPIC * 4 + 1: launch_shade_step<SC_ISOTROPIC, 1>(s, P, b, rays, in4, ids6, seeds, n, out16); break;
            case SC_ISOTROPIC * 4 + 2: launch_shade_step<SC_ISOTROPIC, 2>(s, P, b, rays, in4, ids6, seeds, n, out16); break;
            default: throw std::string("no such shade class instantiation");
        }
    });
}

// camera_ray of k_generate per row.  in3: i, j, sidx
int kat_camera_ray(const rt_camera* cam, uint64_t seed, const uint32_t* in3, int n, rt_ray* out) {
    return guarded([&] {
        Buffers b;
        rt_ray* d_out = b.out<rt_ray>(n);
        k_camera_ray<<<grid(n), BLOCK>>>(*cam, seed, b.in(in3, 3 * (size_t)n), n, d_out);
        fetch(out, d_out, n);
    });
}

int kat_disney_evaluate(const double* params15, int thin, const double* v_out, const double* v_in, const int* front_face, int n, double* out5) {
    return guarded([&] {
        Buffers b; double* d_out = b.out<double>(5 * (size_t)n);
        k_disney_evaluate<<<grid(n), BLOCK>>>(b.in(params15, 15), thin, b.in(v_out, 3 * (size_t)n), b.in(v_in, 3 * (size_t)n), b.in(front_face, n), n, d_out);
        fetch(out5, d_out, 5 * (size_t)n);
    });
}
int kat_disney_generate(const double* params15, int thin, const double* v_out, const int* front_face, const double* pick2, const double* u2, int n, double* out4) {
    return guarded([&] {
        Buffers b; double* d_out = b.out<double>(4 * (size_t)n);
        k_disney_generate<<<grid(n), BLOCK>>>(b.in(params15, 15), thin, b.in(v_out, 3 * (size_t)n), b.in(front_face, n), b.in(pick2, 2 * (size_t)n),
                                              b.in(u2, 2 * (size_t)n), n, d_out);
        fetch(out4, d_out, 4 * (size_t)n);
    });
}
int kat_texture_value(const void* h, const uint32_t* tex, const double* in5, int n, double* out3) {
    const KatScene& s = *(const KatScene*)h;
    return guarded([&] {
        check_indices(tex, n, s.n_textures, "texture");
        Buffers b; double* d_out = b.out<double>(3 * (size_t)n);
        k_texture_value<<<grid(n), BLOCK>>>(s.sv, b.in(tex, n), b.in(in5, 5 * (size_t)n), n, d_out); fetch(out3, d_out, 3 * (size_t)n);
    });
}
int kat_background_value(const void* h, uint32_t tex, const double* dir, int n, double* out4) {
    const KatScene& s = *(const KatScene*)h;
    return guarded([&] {
        check_indices(&tex, 1, s.n_textures, "texture");
        Buffers b; double* d_out = b.out<double>(4 * (size_t)n);
        k_background_value<<<grid(n), BLOCK>>>(s.sv, tex, b.in(dir, 3 * (size_t)n), n, d_out); fetch(out4, d_out, 4 * (size_t)n);
    });
}
int kat_surface_hit_info(const void* h, const uint32_t* prim, const double* t, const rt_ray* rays, int n, double* out11) {
    const KatScene& s = *(const KatScene*)h;
    return guarded([&] {
        check_indices(prim, n, s.sv.n_prims, "primitive");
        Buffers b; double* d_out = b.out<double>(11 * (size_t)n);
        k_surface_hit_info<<<grid(n), BLOCK>>>(s.sv, b.in(prim, n), b.in(t, n), b.in(rays, n), n, d_out); fetch(out11, d_out, 11 * (size_t)n);
    });
}
int kat_remap_record(const void* h, const uint32_t* remap, const double* in9, int n, double* out11) {
    const KatScene& s = *(const KatScene*)h;
    return guarded([&] {
        check_indices(remap, n, s.n_remaps, "remap");
        Buffers b; double* d_out = b.out<double>(11 * (size_t)n);
        k_remap_record<<<grid(n), BLOCK>>>(s.sv, b.in(remap, n), b.in(in9, 9 * (size_t)n), n, d_out); fetch(out11, d_out, 11 * (size_t)n);
    });
}
// lean != 0: lean_lights_pdf over the staged list (the scene must have one)
int kat_lights_pdf(const void* h, int lean, const double* origin, const double* dir, int n, double* out) {
    const KatScene& s = *(const KatScene*)h;
    if (lean && !s.has_lean) return fail("the scene's light list does not qualify for a LeanLights list");
    return guarded([&] {
        Buffers b; double* d_out = b.out<double>(n);
        k_lights_pdf<<<grid(n), BLOCK>>>(s.sv, s.lights_flat, lean ? b.in(&s.lean, 1) : nullptr, b.in(origin, 3 * (size_t)n), b.in(dir, 3 * (size_t)n), n, d_out);
        fetch(out, d_out, n);
    });
}
int kat_lights_random(const void* h, int lean, const double* origin, const double* in3, int n, double* out4) {
    const KatScene& s = *(const KatScene*)h;
    if (lean && !s.has_lean) return fail("the scene's light list does not qualify for a LeanLights list");
    if (!lean && s.sv.n_lights == 0) return fail("the scene has no lights");
    return guarded([&] {
        Buffers b; double* d_out = b.out<double>(4 * (size_t)n);
        k_lights_random<<<grid(n), BLOCK>>>(s.sv, lean ? b.in(&s.lean, 1) : nullptr, b.in(origin, 3 * (size_t)n), b.in(in3, 3 * (size_t)n), n, d_out);
        fetch(out4, d_out, 4 * (size_t)n);
    });
}
int kat_material_emitted(const void* h, const uint32_t* mat, const double* in5, int n, double* out3) {
    const KatScene& s = *(const KatScene*)h;
    return guarded([&] {
        check_indices(mat, n, s.n_materials, "material");
        Buffers b; double* d_out = b.out<double>(3 * (size_t)n);
        k_material_emitted<<<grid(n), BLOCK>>>(s.sv, b.in(mat, n), b.in(in5, 5 * (size_t)n), n, d_out); fetch(out3, d_out, 3 * (size_t)n);
    });
}
int kat_slab(const double* in8, const float* box6, int n, uint8_t* out) {
    return guarded([&] {
        Buffers b; uint8_t* d_out = b.out<uint8_t>(n);
        k_slab<<<grid(n), BLOCK>>>(b.in(in8, 8 * (size_t)n), b.in(box6, 6 * (size_t)n), n, d_out); fetch(out, d_out, n);
    });
}
int kat_medium_free_flight(const double* in7, int n, double* out2) {
    return guarded([&] {
        Buffers b; double* d_out = b.out<double>(2 * (size_t)n);
        k_medium_free_flight<<<grid(n), BLOCK>>>(b.in(in7, 7 * (size_t)n), n, d_out); fetch(out2, d_out, 2 * (size_t)n);
    });
}
int kat_free_flight_overshoots(const double* in6, int n, uint8_t* out) {
    return guarded([&] {
        Buffers b; uint8_t* d_out = b.out<uint8_t>(n);
        k_free_flight_overshoots<<<grid(n), BLOCK>>>(b.in(in6, 6 * (size_t)n), n, d_out); fetch(out, d_out, n);
    });
}

}  // extern "C"
