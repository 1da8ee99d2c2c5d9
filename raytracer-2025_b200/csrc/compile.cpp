// compile.cpp — rt_scene_desc -> CompiledScene.
//
//   1. validate every index of the description;
//   2. copy materials / textures (image texels are sRGB-decoded once here instead of per fetch,
//      utils/image.rs:75-81);
//   3. walk the object graph depth first.  The walk order IS the reference's tie order
//      (SURVEY.md appendix B): `Hittables` children in insertion order (Iterator::min_by keeps the
//      first minimum, hits.rs:42), `BVH` right subtree before left (bvh.rs:78-84) with the tree
//      shape of BVH::from_vec (bvh.rs:16-46) recomputed from the objects' bounding boxes;
//   4. keep primitives below a Transform in its local space (the device takes rays there with the
//      reference's own arithmetic, shapes.rs:74-101) but bound them in WORLD space for the single
//      level BVH; split media boundaries into their own groups;
//   5. flatten the lights tree into leaves with their selection probability;
//   6. build one SAH BVH per group and store primitives in leaf order.
#include "compile.h"

#include <omp.h>

#include <memory>
#include <parallel/algorithm>

#include <chrono>
#include <cstdio>
#include <cstdlib>

#include <vector_functions.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>

namespace rt {

namespace {

struct V3 {
    double x, y, z;
};
inline V3 v3(const double* p) { return V3{p[0], p[1], p[2]}; }
inline V3 operator+(V3 a, V3 b) { return V3{a.x + b.x, a.y + b.y, a.z + b.z}; }
inline V3 operator-(V3 a, V3 b) { return V3{a.x - b.x, a.y - b.y, a.z - b.z}; }
inline V3 operator*(double s, V3 a) { return V3{s * a.x, s * a.y, s * a.z}; }
inline double dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
inline V3 cross(V3 a, V3 b) { return V3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }

struct Affine {
    double A[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    double b[3] = {0, 0, 0};
    bool identity = true;
    uint32_t inst_object = RT_NONE;
    uint32_t xform = RT_NONE;  // index in CompiledScene::xforms of the innermost Transform
    V3 point(V3 p) const {
        return V3{A[0] * p.x + A[1] * p.y + A[2] * p.z + b[0], A[3] * p.x + A[4] * p.y + A[5] * p.z + b[1],
                  A[6] * p.x + A[7] * p.y + A[8] * p.z + b[2]};
    }
    V3 vec(V3 p) const {
        return V3{A[0] * p.x + A[1] * p.y + A[2] * p.z, A[3] * p.x + A[4] * p.y + A[5] * p.z,
                  A[6] * p.x + A[7] * p.y + A[8] * p.z};
    }
    double det() const {
        return A[0] * (A[4] * A[8] - A[5] * A[7]) - A[1] * (A[3] * A[8] - A[5] * A[6]) + A[2] * (A[3] * A[7] - A[4] * A[6]);
    }
    bool inverse(double inv[9]) const {
        double d = det();
        if (d == 0.0 || !std::isfinite(d)) return false;
        double r = 1.0 / d;
        inv[0] = (A[4] * A[8] - A[5] * A[7]) * r;
        inv[1] = (A[2] * A[7] - A[1] * A[8]) * r;
        inv[2] = (A[1] * A[5] - A[2] * A[4]) * r;
        inv[3] = (A[5] * A[6] - A[3] * A[8]) * r;
        inv[4] = (A[0] * A[8] - A[2] * A[6]) * r;
        inv[5] = (A[2] * A[3] - A[0] * A[5]) * r;
        inv[6] = (A[3] * A[7] - A[4] * A[6]) * r;
        inv[7] = (A[1] * A[6] - A[0] * A[7]) * r;
        inv[8] = (A[0] * A[4] - A[1] * A[3]) * r;
        return true;
    }
};

// Transform::transform (shapes.rs:74-78) as a matrix: x -> q * (x .* scale) * conj(q) + offset
Affine affine_of(const rt_transform& t, uint32_t object) {
    const double w = t.quat[0], x = t.quat[1], y = t.quat[2], z = t.quat[3];
    // columns of the rotation = images of the basis vectors under the Hamilton sandwich product;
    // the quaternion is not renormalised (neither is it in quaternion.rs:72-82)
    double R[9] = {w * w + x * x - y * y - z * z, 2 * (x * y - w * z),           2 * (x * z + w * y),
                   2 * (x * y + w * z),           w * w - x * x + y * y - z * z, 2 * (y * z - w * x),
                   2 * (x * z - w * y),           2 * (y * z + w * x),           w * w - x * x - y * y + z * z};
    Affine a;
    for (int r = 0; r < 3; r++)
        for (int c = 0; c < 3; c++) a.A[r * 3 + c] = R[r * 3 + c] * t.scale[c];
    for (int k = 0; k < 3; k++) a.b[k] = t.offset[k];
    a.identity = false;
    a.inst_object = object;
    return a;
}
// outer(inner(x))
Affine compose(const Affine& outer, const Affine& inner) {
    if (outer.identity) return inner;
    Affine r;
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) {
            double s = 0;
            for (int k = 0; k < 3; k++) s += outer.A[i * 3 + k] * inner.A[k * 3 + j];
            r.A[i * 3 + j] = s;
        }
    V3 b = outer.point(V3{inner.b[0], inner.b[1], inner.b[2]});
    r.b[0] = b.x, r.b[1] = b.y, r.b[2] = b.z;
    r.identity = false;
    r.inst_object = inner.inst_object;  // innermost Transform
    return r;
}

struct FlatPrim {
    PrimGeom g;
    PrimMeta m;
    double lo[3], hi[3];
};

float round_down(double x) {
    float f = (float)x;
    if ((double)f > x) f = std::nextafterf(f, -INFINITY);
    return f;
}
float round_up(double x) {
    float f = (float)x;
    if ((double)f < x) f = std::nextafterf(f, INFINITY);
    return f;
}

uint64_t total_order_key(double x) {  // f64::total_cmp (bvh.rs:52)
    uint64_t b;
    std::memcpy(&b, &x, 8);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

uint32_t shade_class_of(const rt_scene_desc& d, const rt_material& m, const std::vector<Material>& done) {
    switch (m.kind) {
        case RT_MAT_DISNEY: return SC_DISNEY;
        // The OBJ loader's chains: RemappedMaterial outermost (obj.rs:165-176), below it the DiffuseLight a `Ke` line adds - exporters
        // write `Ke 0 0 0` on every material, so 95 % of the shipped assets are Remapped(DiffuseLight(Disney)) - then the Disney.
        // They share the Disney kernel (emission included); only Mix / Transparent / Portal chains need the general one, whose
        // code no longer fits the instruction cache (ncu on the assets/Final scene: icc hit rate 46 %, issue active 13 %).
        case RT_MAT_REMAPPED: return done[m.inner].shade_class == SC_DISNEY ? SC_DISNEY : SC_OTHER;
        case RT_MAT_EMPTY: return SC_DIFFUSE;
        case RT_MAT_LAMBERTIAN: return d.textures[m.tex].kind == RT_TEX_SOLID ? SC_DIFFUSE : SC_TEXTURED;
        case RT_MAT_METAL: return SC_METAL;
        case RT_MAT_DIELECTRIC: return SC_DIELECTRIC;
        case RT_MAT_DIFFUSE_LIGHT: return m.inner == RT_NONE ? SC_EMISSIVE : (done[m.inner].shade_class == SC_DISNEY ? SC_DISNEY : SC_OTHER);
        case RT_MAT_ISOTROPIC: return SC_ISOTROPIC;
        default: return SC_OTHER;
    }
}

float srgb_to_linear(float x) {  // palette Srgb::into_linear<f32>, applied per fetch by image.rs:80
    if (x <= 0.04045f) return (float)(1.0 / 12.92) * x;
    return std::pow(std::fma(x, (float)(1.0 / 1.055), (float)(0.055 / 1.055)), 2.4f);
}

struct Compiler {
    const rt_scene_desc& d;
    uint32_t flags;
    CompiledScene& out;
    std::string& err;
    WorldBuilder world_builder = nullptr;
    std::vector<RawVec<FlatPrim>> groups;  // 0 = world surfaces, 1+m = boundary of media[m]
    std::vector<uint32_t> group_of_medium;
    uint32_t next_rank = 0;
    int status = RT_OK;

    bool fail(int code, const std::string& msg) {
        if (status == RT_OK) status = code, err = msg;
        return false;
    }

    bool validate() {
        if (d.version != RT_ABI_VERSION) return fail(RT_ERR_VERSION, "rt_scene_desc.version mismatch");
        if (d.struct_size != sizeof(rt_scene_desc)) return fail(RT_ERR_VERSION, "rt_scene_desc.struct_size mismatch");
        if (d.world_root >= d.n_objects) return fail(RT_ERR_INVALID, "world_root out of range");
        if (d.n_materials > META_MAT_MASK) return fail(RT_ERR_UNSUPPORTED, "more than 2^26 materials");
        if (d.lights_root != RT_NONE && d.lights_root >= d.n_objects) return fail(RT_ERR_INVALID, "lights_root out of range");
        auto need = [&](const void* p, uint64_t n, const char* what) {
            if (n && !p) return fail(RT_ERR_INVALID, std::string(what) + " is null");
            return true;
        };
        if (!need(d.objects, d.n_objects, "objects") || !need(d.children, d.n_children, "children") ||
            !need(d.spheres, d.n_spheres, "spheres") || !need(d.planars, d.n_planars, "planars") ||
            !need(d.transforms, d.n_transforms, "transforms") || !need(d.media, d.n_media, "media") ||
            !need(d.materials, d.n_materials, "materials") || !need(d.textures, d.n_textures, "textures") ||
            !need(d.images, d.n_images, "images") || !need(d.texels, d.n_texels, "texels") ||
            !need(d.perlins, d.n_perlins, "perlins") || !need(d.remaps, d.n_remaps, "remaps"))
            return false;
        for (uint32_t i = 0; i < d.n_perlins; i++)  // utils/perlin.rs:25-38: permutations of 0..255; they index randvec on the device
            for (int k = 0; k < 256; k++)
                if (d.perlins[i].perm_x[k] > 255u || d.perlins[i].perm_y[k] > 255u || d.perlins[i].perm_z[k] > 255u)
                    return fail(RT_ERR_INVALID, "perlin permutation entry out of range");
        for (uint32_t i = 0; i < d.n_remaps; i++)
            if (d.remaps[i].normal_tex != RT_NONE && (d.remaps[i].normal_tex >= d.n_textures || d.textures[d.remaps[i].normal_tex].kind != RT_TEX_IMAGE))
                return fail(RT_ERR_INVALID, "remap normal texture must be an image texture");
        // every image is copied (and sRGB-decoded) by copy_tables, referenced or not: bound them all, overflow-safe
        for (uint32_t i = 0; i < d.n_images; i++) {
            const rt_image& im = d.images[i];
            if (im.width == 0 || im.height == 0) return fail(RT_ERR_INVALID, "image with zero width or height (a missing file is texture.a == RT_NONE)");
            const uint64_t n_texel = (uint64_t)im.width * im.height;  // < 2^64: both factors are 32-bit
            if (n_texel > (d.n_texels >> 2) || im.texel_offset > d.n_texels - 4 * n_texel || (im.texel_offset & 3u))
                return fail(RT_ERR_INVALID, "image texels out of range");
        }
        for (uint32_t i = 0; i < d.n_textures; i++) {
            const rt_texture& t = d.textures[i];
            switch (t.kind) {
                case RT_TEX_SOLID:
                case RT_TEX_GRADIENT_Y: break;
                case RT_TEX_CHECKER:
                    if (t.a >= i || t.b >= i) return fail(RT_ERR_INVALID, "checker children must precede the checker");
                    break;
                case RT_TEX_IMAGE:
                    if (t.a != RT_NONE && t.a >= d.n_images) return fail(RT_ERR_INVALID, "image index out of range");
                    break;
                case RT_TEX_NOISE:
                    if (t.a >= d.n_perlins) return fail(RT_ERR_INVALID, "perlin index out of range");
                    break;
                default: return fail(RT_ERR_INVALID, "unknown texture kind");
            }
        }
        for (uint32_t i = 0; i < d.n_materials; i++) {
            const rt_material& m = d.materials[i];
            auto tex_ok = [&](bool required) { return m.tex < d.n_textures || (!required && m.tex == RT_NONE); };
            switch (m.kind) {
                case RT_MAT_EMPTY:
                case RT_MAT_METAL:
                case RT_MAT_TRANSPARENT:
                case RT_MAT_PORTAL: break;
                case RT_MAT_LAMBERTIAN:
                case RT_MAT_DIELECTRIC:
                case RT_MAT_ISOTROPIC:
                    if (!tex_ok(true)) return fail(RT_ERR_INVALID, "material texture out of range");
                    break;
                case RT_MAT_DIFFUSE_LIGHT:
                    if (!tex_ok(true)) return fail(RT_ERR_INVALID, "material texture out of range");
                    if (m.inner != RT_NONE && m.inner >= i) return fail(RT_ERR_INVALID, "inner material must precede its wrapper");
                    break;
                case RT_MAT_MIX:
                    if (m.inner >= i || m.inner2 >= i) return fail(RT_ERR_INVALID, "Mix children must precede it");
                    if (!tex_ok(false)) return fail(RT_ERR_INVALID, "material texture out of range");
                    if (m.tex != RT_NONE && d.textures[m.tex].kind != RT_TEX_IMAGE)
                        return fail(RT_ERR_INVALID, "Mix ratio texture must be an image");
                    break;
                case RT_MAT_DISNEY:
                    if (!tex_ok(false)) return fail(RT_ERR_INVALID, "material texture out of range");
                    break;
                case RT_MAT_REMAPPED:
                    if (m.inner >= i) return fail(RT_ERR_INVALID, "inner material must precede its wrapper");
                    if (m.inner2 >= d.n_remaps) return fail(RT_ERR_INVALID, "remap index out of range");
                    break;
                default: return fail(RT_ERR_INVALID, "unknown material kind");
            }
        }
        // The graph is a tree (Box<dyn Hittable> owns its children): one parent per object, nesting bounded so that the
        // recursive walks below cannot overflow the stack
        std::vector<uint8_t> seen(d.n_objects, 0);
        std::vector<uint16_t> height(d.n_objects, 0);
        constexpr uint32_t MAX_NESTING = 256;
        for (uint32_t i = 0; i < d.n_objects; i++) {
            const rt_object& o = d.objects[i];
            if ((uint64_t)o.first_child + o.child_count > d.n_children) return fail(RT_ERR_INVALID, "children range out of bounds");
            switch (o.kind) {
                case RT_OBJ_SPHERE:
                    if (o.data >= d.n_spheres || o.material >= d.n_materials) return fail(RT_ERR_INVALID, "sphere payload/material out of range");
                    break;
                case RT_OBJ_QUAD:
                case RT_OBJ_TRIANGLE:
                    if (o.data >= d.n_planars || o.material >= d.n_materials) return fail(RT_ERR_INVALID, "planar payload/material out of range");
                    break;
                case RT_OBJ_LIST: break;
                case RT_OBJ_BVH:
                    if (o.child_count == 0) return fail(RT_ERR_INVALID, "BVH node must contain at least one object");
                    break;
                case RT_OBJ_TRANSFORM:
                    if (o.data >= d.n_transforms || o.child_count != 1) return fail(RT_ERR_INVALID, "bad Transform");
                    break;
                case RT_OBJ_MEDIUM:
                    if (o.data >= d.n_media || o.child_count != 1 || o.material >= d.n_materials) return fail(RT_ERR_INVALID, "bad ConstantMedium");
                    // volume.rs:23-35: the phase function is always an Isotropic; the shade kernels rely on it
                    if (d.materials[o.material].kind != RT_MAT_ISOTROPIC) return fail(RT_ERR_INVALID, "the phase function of a ConstantMedium must be an Isotropic material");
                    break;
                default: return fail(RT_ERR_INVALID, "unknown object kind");
            }
            for (uint32_t k = 0; k < o.child_count; k++) {
                uint32_t c = d.children[o.first_child + k];
                if (c >= d.n_objects) return fail(RT_ERR_INVALID, "child index out of range");
                if (c >= i) return fail(RT_ERR_INVALID, "children must precede their parent (the graph is a tree emitted bottom-up)");
                if (seen[c]) return fail(RT_ERR_INVALID, "an object has two parents (the graph must be a tree)");
                seen[c] = 1;
                height[i] = std::max<uint16_t>(height[i], (uint16_t)(height[c] + 1));
            }
            if (height[i] > MAX_NESTING) return fail(RT_ERR_UNSUPPORTED, "containers nested more than 256 deep");
        }
        if (seen[d.world_root] || (d.lights_root != RT_NONE && (seen[d.lights_root] || d.lights_root == d.world_root)))
            return fail(RT_ERR_INVALID, "world / lights root is the child of another object");
        return true;
    }

    void copy_tables() {
        out.textures.resize(d.n_textures);
        for (uint32_t i = 0; i < d.n_textures; i++) {
            const rt_texture& s = d.textures[i];
            Texture t{};
            t.kind = s.kind, t.a = s.a, t.b = s.b;
            for (int k = 0; k < 3; k++) t.color[k] = s.color[k], t.color2[k] = s.color2[k];
            t.scale = s.scale;
            out.textures[i] = t;
        }
        out.materials.resize(d.n_materials);
        for (uint32_t i = 0; i < d.n_materials; i++) {
            const rt_material& s = d.materials[i];
            Material m{};
            m.kind = s.kind, m.tex = s.tex, m.inner = s.inner, m.inner2 = s.inner2;
            for (int k = 0; k < 3; k++) m.color[k] = s.color[k];
            m.param = s.param;
            for (int k = 0; k < 16; k++) m.v[k] = s.v[k];
            m.shade_class = shade_class_of(d, s, out.materials);
            // does shading this material read the surface coordinates (image / checker lookups)?
            // (kinds that ignore `tex` may carry anything there: bounds first)
            auto tex_uv = [&](uint32_t t) { return t < d.n_textures && (d.textures[t].kind == RT_TEX_IMAGE || d.textures[t].kind == RT_TEX_CHECKER); };
            m.needs_uv = tex_uv(s.tex) ? 1u : 0u;
            if (s.inner != RT_NONE && s.inner < i) m.needs_uv |= out.materials[s.inner].needs_uv;
            if (s.inner2 != RT_NONE && s.inner2 < i) m.needs_uv |= out.materials[s.inner2].needs_uv;
            out.materials[i] = m;
        }
        out.images.resize(d.n_images);
        out.texels.resize(d.n_texels / 4);
        for (uint32_t i = 0; i < d.n_images; i++) {
            const rt_image& s = d.images[i];
            Image im{};
            im.width = s.width, im.height = s.height, im.flags = s.flags;
            im.texel_offset = s.texel_offset / 4;
            out.images[i] = im;
            const float* p = d.texels + s.texel_offset;
            for (uint64_t k = 0; k < (uint64_t)s.width * s.height; k++) {
                float4 t;
                if (s.flags & RT_IMG_LINEAR)
                    t = make_float4(p[4 * k], p[4 * k + 1], p[4 * k + 2], p[4 * k + 3]);
                else
                    t = make_float4(srgb_to_linear(p[4 * k]), srgb_to_linear(p[4 * k + 1]), srgb_to_linear(p[4 * k + 2]), p[4 * k + 3]);
                out.texels[im.texel_offset + k] = t;
            }
        }
        out.remaps.resize(d.n_remaps);
        static_assert(sizeof(Remap) == sizeof(rt_remap), "remap layout");
        for (uint32_t i = 0; i < d.n_remaps; i++) std::memcpy(&out.remaps[i], &d.remaps[i], sizeof(Remap));
        out.perlins.resize(d.n_perlins);
        for (uint32_t i = 0; i < d.n_perlins; i++) std::memcpy(&out.perlins[i], &d.perlins[i], sizeof(Perlin));
        static_assert(sizeof(Perlin) == sizeof(rt_perlin), "perlin layout");
    }

    // register one Transform below `parent` and return the affine image of the whole chain
    bool push_xform(const rt_transform& t, uint32_t object, const Affine& parent, Affine& out_chain) {
        Xform x{};
        for (int k = 0; k < 3; k++) x.offset[k] = t.offset[k], x.scale[k] = t.scale[k];
        for (int k = 0; k < 4; k++) x.quat[k] = t.quat[k];
        x.inst_object = object;
        uint32_t self = (uint32_t)out.xforms.size();
        x.n_chain = 0;
        if (parent.xform != RT_NONE) {
            const Xform& px = out.xforms[parent.xform];
            for (uint32_t k = 0; k < px.n_chain; k++) x.chain[x.n_chain++] = px.chain[k];
        }
        if (x.n_chain >= MAX_XFORM_CHAIN) return fail(RT_ERR_UNSUPPORTED, "more than 4 nested Transforms");
        x.chain[x.n_chain++] = self;
        out.xforms.push_back(x);
        out_chain = compose(parent, affine_of(t, object));
        out_chain.xform = self;
        double inv[9];
        if (!out_chain.inverse(inv)) return fail(RT_ERR_UNSUPPORTED, "singular Transform (zero scale)");
        return true;
    }

    // Local geometry of a leaf shape (verbatim from the description) and its WORLD-space bounds
    // under the affine image of the Transform chain.
    bool leaf(uint32_t obj, const Affine& a, PrimGeom& g, uint32_t& kind, double lo[3], double hi[3], double* area_out, bool quiet = false) {
        const rt_object& o = d.objects[obj];
        std::memset(&g, 0, sizeof(g));
        V3 pts[8];
        int np = 0;
        double pad_r = 0.0;
        if (o.kind == RT_OBJ_SPHERE) {
            const rt_sphere& s = d.spheres[o.data];
            V3 c = v3(s.center), cv = v3(s.center_vec);
            double r = s.radius;
            g.d[0] = c.x, g.d[1] = c.y, g.d[2] = c.z, g.d[3] = cv.x, g.d[4] = cv.y, g.d[5] = cv.z, g.d[6] = r;
            kind = PRIM_SPHERE;
            if (area_out) *area_out = 0.0;
            V3 c1 = c + cv;  // centre at time 1 (sphere.rs:35-51 bounds time in [0,1])
            bool similarity = true;
            double k = 1.0;
            if (!a.identity) {
                k = a.A[0] * a.A[0] + a.A[3] * a.A[3] + a.A[6] * a.A[6];
                for (int i = 0; i < 3 && similarity; i++)
                    for (int j = 0; j < 3; j++) {
                        double s2 = a.A[i] * a.A[j] + a.A[3 + i] * a.A[3 + j] + a.A[6 + i] * a.A[6 + j];
                        if (std::fabs(s2 - (i == j ? k : 0.0)) > 1e-9 * k) similarity = false;
                    }
            }
            if (similarity) {  // still a sphere in world space: tight box around the moving centre
                pts[np++] = a.identity ? c : a.point(c);
                pts[np++] = a.identity ? c1 : a.point(c1);
                pad_r = r * std::sqrt(k) * (1.0 + 1e-9);
            } else {  // an ellipsoid: box of the transformed corners of the local box (like shapes.rs:49-72)
                double mn[3], mx[3];
                double cc[2][3] = {{c.x, c.y, c.z}, {c1.x, c1.y, c1.z}};
                for (int q = 0; q < 3; q++) mn[q] = std::min(cc[0][q], cc[1][q]) - r, mx[q] = std::max(cc[0][q], cc[1][q]) + r;
                for (int m = 0; m < 8; m++) pts[np++] = a.point(V3{(m & 4) ? mx[0] : mn[0], (m & 2) ? mx[1] : mn[1], (m & 1) ? mx[2] : mn[2]});
            }
        } else {
            const rt_planar& p = d.planars[o.data];
            const bool tri = o.kind == RT_OBJ_TRIANGLE;
            kind = tri ? PRIM_TRIANGLE : PRIM_QUAD;
            V3 q = v3(p.anchor), u = v3(p.u), v = v3(p.v);
            double* e = g.d;
            e[0] = q.x, e[1] = q.y, e[2] = q.z, e[3] = u.x, e[4] = u.y, e[5] = u.z, e[6] = v.x, e[7] = v.y, e[8] = v.z;
            e[9] = p.normal[0], e[10] = p.normal[1], e[11] = p.normal[2], e[12] = p.parm_d;
            e[13] = p.w[0], e[14] = p.w[1], e[15] = p.w[2];
            if (area_out) *area_out = p.area;
            V3 corner[4] = {q, q + u, q + v, q + u + v};
            for (int i = 0; i < (tri ? 3 : 4); i++) pts[np++] = a.identity ? corner[i] : a.point(corner[i]);
        }
        for (int k = 0; k < 3; k++) lo[k] = INFINITY, hi[k] = -INFINITY;
        for (int i = 0; i < np; i++) {
            double c[3] = {pts[i].x, pts[i].y, pts[i].z};
            for (int k = 0; k < 3; k++) lo[k] = std::min(lo[k], c[k] - pad_r), hi[k] = std::max(hi[k], c[k] + pad_r);
        }
        if (!a.identity) {
            // the device transforms with quaternion products, this bound with a matrix: cover the
            // last-bit disagreement between the two before the outward rounding to binary32
            for (int k = 0; k < 3; k++) {
                double m = 1e-12 * (std::fabs(lo[k]) + std::fabs(hi[k]) + (hi[k] - lo[k]));
                lo[k] -= m, hi[k] += m;
            }
        }
        for (int k = 0; k < 3; k++)
            if (!std::isfinite(lo[k]) || !std::isfinite(hi[k])) return quiet ? false : fail(RT_ERR_INVALID, "primitive with non-finite bounds");
        return true;
    }

    // Order in which BVH::from_vec + BVH::hit would prefer the children on a tie: right before left.
    // Each node is the reference's split: bounds of the set, longest axis (ties towards z, aabb.rs:80-92),
    // STABLE sort by box-min (bvh.rs:41, f64::total_cmp), halves at len/2.
    //
    // The reference sorts at every node (N log^2 N).  Box-mins never change, so this walk sorts the children
    // ONCE per axis and carries the three sorted lists down the tree by stable partition, like a kd-tree
    // build: O(N) per level, no comparator indirection, subtrees as OpenMP tasks.  Invariant at the entry of
    // a node: each axis list holds the node's children sorted by (box-min on that axis, position in the order P
    // the parent left them in) - exactly what a stable sort of P would produce, so the list of the chosen
    // axis IS the sorted node.  Partitioning keeps a list sorted by box-min but leaves equal keys in the
    // PARENT's P order; runs of equal keys are therefore re-sorted by the position in the new order.
    struct AxisEnt {
        double mn, mx;  // bounding-box interval of the child on this axis
        uint32_t id;    // index into the BVH's child list
        uint32_t pad;
    };
    struct TieOrder {
        const uint32_t* kids = nullptr;  // child list -> object ids
        AxisEnt* list[2][3] = {};        // ping-pong copies of the three axis lists
        uint8_t* side = nullptr;         // scratch, one byte per child: 1 = goes to the right half of its node
        uint32_t* pos = nullptr;         // scratch, written only by nodes that have equal keys: position in the sorted node
    };
    static bool key_less(const AxisEnt& x, const AxisEnt& y) { return total_order_key(x.mn) < total_order_key(y.mn); }
    // p_axis: the axis whose list holds this node's children in the order P their parent left them (the parent's
    // sorted order survives the stable partition); -1 at the root, where the ids themselves are P.
    void tie_order_node(const TieOrder& T, size_t off, size_t len, int buf, int p_axis, uint32_t* out) {
        AxisEnt* const* cur = T.list[buf];
        if (len == 1) {
            out[0] = T.kids[cur[0][off].id];
            return;
        }
        if (len == 2) {  // no sort: left = P[0], right = P[1] (bvh.rs:24-27), right first
            uint32_t a, b;
            if (p_axis >= 0) {
                a = cur[p_axis][off].id, b = cur[p_axis][off + 1].id;
            } else {
                a = std::min(cur[0][off].id, cur[0][off + 1].id), b = std::max(cur[0][off].id, cur[0][off + 1].id);
            }
            out[0] = T.kids[b];
            out[1] = T.kids[a];
            return;
        }
        double s[3];
        for (int k = 0; k < 3; k++) {
            double mn = INFINITY, mx = -INFINITY;
            const AxisEnt* e = cur[k] + off;
            for (size_t i = 0; i < len; i++) mn = std::fmin(mn, e[i].mn), mx = std::fmax(mx, e[i].mx);
            s[k] = std::fmax(mx - mn, 0.0);
        }
        const int axis = s[0] > s[1] ? (s[0] > s[2] ? 0 : 2) : (s[1] > s[2] ? 1 : 2);  // aabb.rs:80-92
        const size_t mid = len / 2, n_right = len - mid;
        {
            // one byte per child instead of its 4-byte position: the partitions below look it up at random, and a
            // quarter of the footprint is what stays in cache on a 10^8-child tree
            const AxisEnt* e = cur[axis] + off;  // the node in sorted order
            for (size_t i = 0; i < len; i++) T.side[e[i].id] = i >= mid;
        }
        AxisEnt* const* nxt = T.list[buf ^ 1];
        bool ties = false;
        for (int k = 0; k < 3; k++) {
            const AxisEnt* e = cur[k] + off;
            AxisEnt* lo = nxt[k] + off;
            AxisEnt* hi = nxt[k] + off + mid;
            if (k == axis) {
                std::memcpy(lo, e, len * sizeof(AxisEnt));
                continue;
            }
            uint64_t last_lo = 0, last_hi = 0;  // keys are never 0 for a finite value... compare only after the first write
            bool any_lo = false, any_hi = false;
            for (size_t i = 0; i < len; i++) {
                const uint64_t key = total_order_key(e[i].mn);
                if (!T.side[e[i].id]) {
                    ties |= any_lo && key == last_lo;
                    last_lo = key, any_lo = true;
                    *lo++ = e[i];
                } else {
                    ties |= any_hi && key == last_hi;
                    last_hi = key, any_hi = true;
                    *hi++ = e[i];
                }
            }
        }
        if (ties) {
            // equal keys: a partitioned list keeps them in the PARENT's order; put them in this node's sorted order
            const AxisEnt* e = cur[axis] + off;
            for (size_t i = 0; i < len; i++) T.pos[e[i].id] = (uint32_t)i;
            for (int k = 0; k < 3; k++) {
                if (k == axis) continue;
                for (AxisEnt* half : {nxt[k] + off, nxt[k] + off + mid}) {
                    const size_t n = half == nxt[k] + off ? mid : n_right;
                    for (size_t i = 0; i + 1 < n;) {
                        size_t j = i + 1;
                        const uint64_t key = total_order_key(half[i].mn);
                        while (j < n && total_order_key(half[j].mn) == key) j++;
                        if (j - i > 1) std::sort(half + i, half + j, [&](const AxisEnt& x, const AxisEnt& y) { return T.pos[x.id] < T.pos[y.id]; });
                        i = j;
                    }
                }
            }
        }
        if (len >= 16384) {
#pragma omp task default(shared)
            tie_order_node(T, off + mid, n_right, buf ^ 1, axis, out);
            tie_order_node(T, off, mid, buf ^ 1, axis, out + n_right);
#pragma omp taskwait
        } else {
            tie_order_node(T, off + mid, n_right, buf ^ 1, axis, out);
            tie_order_node(T, off, mid, buf ^ 1, axis, out + n_right);
        }
    }
    // One BIG node of the walk above, split by ALL threads (the task recursion gives a node to one thread: on a 10^8-child tree
    // the first four levels then run on 1, 2, 4 and 8 of the cores and take as long as all the levels below them together).
    // Same steps as tie_order_node: bounds -> axis, side bytes, stable partition of the two other lists (two passes over
    // per-thread chunks: count, then write at the chunk's offsets), equal-key runs re-sorted by position.  Returns the axis.
    int split_node_parallel(const TieOrder& T, size_t off, size_t len, int buf) {
        AxisEnt* const* cur = T.list[buf];
        AxisEnt* const* nxt = T.list[buf ^ 1];
        double s[3];
        for (int k = 0; k < 3; k++) {
            double mn = INFINITY, mx = -INFINITY;
            const AxisEnt* e = cur[k] + off;
#pragma omp parallel for schedule(static) reduction(min : mn) reduction(max : mx)
            for (size_t i = 0; i < len; i++) mn = std::fmin(mn, e[i].mn), mx = std::fmax(mx, e[i].mx);
            s[k] = std::fmax(mx - mn, 0.0);
        }
        const int axis = s[0] > s[1] ? (s[0] > s[2] ? 0 : 2) : (s[1] > s[2] ? 1 : 2);  // aabb.rs:80-92
        const size_t mid = len / 2;
        {
            const AxisEnt* e = cur[axis] + off;
#pragma omp parallel for schedule(static)
            for (size_t i = 0; i < len; i++) T.side[e[i].id] = i >= mid;
        }
        const int n_chunks = std::max(1, omp_get_max_threads());
        std::vector<size_t> lo_count((size_t)n_chunks + 1);
        bool ties = false;
        for (int k = 0; k < 3; k++) {
            const AxisEnt* e = cur[k] + off;
            if (k == axis) {
#pragma omp parallel for schedule(static)
                for (size_t i = 0; i < len; i++) nxt[k][off + i] = e[i];
                continue;
            }
            auto chunk_begin = [&](int c) { return len * (size_t)c / (size_t)n_chunks; };
#pragma omp parallel for schedule(static, 1)
            for (int c = 0; c < n_chunks; c++) {
                size_t n_lo = 0;
                for (size_t i = chunk_begin(c); i < chunk_begin(c + 1); i++) n_lo += !T.side[e[i].id];
                lo_count[(size_t)c + 1] = n_lo;
            }
            lo_count[0] = 0;
            for (int c = 0; c < n_chunks; c++) lo_count[(size_t)c + 1] += lo_count[(size_t)c];  // lows before chunk c
#pragma omp parallel for schedule(static, 1)
            for (int c = 0; c < n_chunks; c++) {
                AxisEnt* lo = nxt[k] + off + lo_count[(size_t)c];
                AxisEnt* hi = nxt[k] + off + mid + (chunk_begin(c) - lo_count[(size_t)c]);
                for (size_t i = chunk_begin(c); i < chunk_begin(c + 1); i++) {
                    if (!T.side[e[i].id])
                        *lo++ = e[i];
                    else
                        *hi++ = e[i];
                }
            }
            // equal keys next to each other inside a half: the run has to be put into this node's order (below)
            const AxisEnt* o = nxt[k] + off;
            bool t = false;
#pragma omp parallel for schedule(static) reduction(|| : t)
            for (size_t i = 1; i < len; i++)
                if (i != mid && total_order_key(o[i].mn) == total_order_key(o[i - 1].mn)) t = true;
            ties = ties || t;
        }
        if (ties) {
            const AxisEnt* e = cur[axis] + off;
#pragma omp parallel for schedule(static)
            for (size_t i = 0; i < len; i++) T.pos[e[i].id] = (uint32_t)i;
            const size_t n_right = len - mid;
#pragma omp parallel for schedule(dynamic, 1) collapse(2)
            for (int k = 0; k < 3; k++)
                for (int h = 0; h < 2; h++) {
                    if (k == axis) continue;
                    AxisEnt* half = nxt[k] + off + (h ? mid : 0);
                    const size_t n = h ? n_right : mid;
                    for (size_t i = 0; i + 1 < n;) {
                        size_t j = i + 1;
                        const uint64_t key = total_order_key(half[i].mn);
                        while (j < n && total_order_key(half[j].mn) == key) j++;
                        if (j - i > 1) std::sort(half + i, half + j, [&](const AxisEnt& x, const AxisEnt& y) { return T.pos[x.id] < T.pos[y.id]; });
                        i = j;
                    }
                }
        }
        return axis;
    }

    // Stable LSD radix sort of a[0..n) by total_order_key(mn), four 16-bit digits, all threads: every thread counts the digits of
    // its chunk, the offsets are laid out digit-major / thread-minor (which is what keeps equal keys in input order), every
    // thread scatters its chunk.  A digit on which all keys agree costs no pass.  `tmp` is scratch of the same length.
    // (The three lists of 16 M entries on 8 cores: 1.1-1.5 s against 2.2 s for libstdc++'s parallel multiway merge sort.)
    static void radix_sort_by_min(AxisEnt* a, AxisEnt* tmp, size_t n) {
        const int T = std::max(1, omp_get_max_threads());
        std::vector<size_t> hist((size_t)T * 65536);
        AxisEnt* src = a;
        AxisEnt* dst = tmp;
        for (int pass = 0; pass < 4; pass++) {
            const int shift = 16 * pass;
            std::fill(hist.begin(), hist.end(), 0);
#pragma omp parallel num_threads(T)
            {
                const int t = omp_get_thread_num();
                size_t* h = hist.data() + (size_t)t * 65536;
                const size_t i0 = n * (size_t)t / (size_t)T, i1 = n * (size_t)(t + 1) / (size_t)T;
                for (size_t i = i0; i < i1; i++) h[(total_order_key(src[i].mn) >> shift) & 0xFFFFu]++;
            }
            size_t run = 0;
            bool one_bucket = false;
            for (size_t d = 0; d < 65536; d++) {
                size_t in_digit = 0;
                for (int t = 0; t < T; t++) {
                    const size_t c = hist[(size_t)t * 65536 + d];
                    hist[(size_t)t * 65536 + d] = run;
                    run += c, in_digit += c;
                }
                one_bucket = one_bucket || in_digit == n;
            }
            if (one_bucket) continue;  // all keys share this digit: nothing moves
#pragma omp parallel num_threads(T)
            {
                const int t = omp_get_thread_num();
                size_t* h = hist.data() + (size_t)t * 65536;
                const size_t i0 = n * (size_t)t / (size_t)T, i1 = n * (size_t)(t + 1) / (size_t)T;
                for (size_t i = i0; i < i1; i++) dst[h[(total_order_key(src[i].mn) >> shift) & 0xFFFFu]++] = src[i];
            }
            std::swap(src, dst);
        }
        if (src != a) {
#pragma omp parallel for schedule(static)
            for (size_t i = 0; i < n; i++) a[i] = src[i];
        }
    }

    // kids[0..n) -> the same ids in tie order
    void bvh_visit_order(std::vector<uint32_t>& kids) {
        const size_t n = kids.size();
        if (n < 2) return;
        std::unique_ptr<AxisEnt[]> store[2][3];  // not value-initialised: 144 bytes per child that the loops below fill
        std::vector<uint32_t> pos(n), out(n);
        std::vector<uint8_t> side(n);
        TieOrder T;
        T.kids = kids.data();
        T.pos = pos.data();
        T.side = side.data();
        for (int b = 0; b < 2; b++)
            for (int k = 0; k < 3; k++) store[b][k].reset(new AxisEnt[n]), T.list[b][k] = store[b][k].get();
#pragma omp parallel for schedule(static) if (n > 32768)
        for (size_t i = 0; i < n; i++) {
            const double* bb = d.objects[kids[i]].bbox;
            for (int k = 0; k < 3; k++) T.list[0][k][i] = AxisEnt{bb[2 * k], bb[2 * k + 1], (uint32_t)i, 0};
        }
        if (n > 100000) timer.lap("    tie order: fill");
        // the three stable sorts by box-min: a radix sort by all threads for big inputs (the second copy of the list is its scratch;
        // it brings its own team, so it runs outside the task region of the walk)
        size_t radix_min = 32768;
        if (const char* e = getenv("RT2025_TIE_RADIX_MIN")) radix_min = (size_t)std::max(2l, atol(e));  // (the CPU check forces it on small inputs)
        for (int k = 0; k < 3; k++) {
            if (n > radix_min)
                radix_sort_by_min(T.list[0][k], T.list[1][k], n);
            else if (n > 32768)
                __gnu_parallel::stable_sort(T.list[0][k], T.list[0][k] + n, key_less);
            else
                std::stable_sort(T.list[0][k], T.list[0][k] + n, key_less);
        }
        if (n > 100000) timer.lap("    tie order: three stable sorts");
        // the big nodes at the top are split one after the other by all threads; what is left goes to the task recursion
        struct Job {
            size_t off, len;
            int buf, p_axis;
            uint32_t* out;
        };
        size_t par_min = 1u << 20;
        if (const char* e = getenv("RT2025_TIE_PAR_MIN")) par_min = (size_t)std::max(8l, atol(e));  // (the CPU check forces the parallel split on small inputs)
        std::vector<Job> big{{0, n, 0, -1, out.data()}}, rest;
        while (!big.empty()) {
            const Job j = big.back();
            big.pop_back();
            if (j.len < par_min || j.len < 8) {
                rest.push_back(j);
                continue;
            }
            const int axis = split_node_parallel(T, j.off, j.len, j.buf);
            const size_t mid = j.len / 2, n_right = j.len - mid;
            big.push_back({j.off + mid, n_right, j.buf ^ 1, axis, j.out});          // right first (bvh.rs:78-84)
            big.push_back({j.off, mid, j.buf ^ 1, axis, j.out + n_right});
        }
        if (n > 100000) timer.lap("    tie order: big nodes, all threads");
#pragma omp parallel if (n > 32768)  // waking the team costs more than a book-sized tree (a few thousand children) takes
#pragma omp single
        for (const Job& j : rest) {
#pragma omp task default(shared) firstprivate(j)
            tie_order_node(T, j.off, j.len, j.buf, j.p_axis, j.out);
        }
        if (n > 100000) timer.lap("    tie order: subtrees as tasks");
        kids.swap(out);
    }

    // A BVH whose children are all shapes (a mesh, a soup): the leaves of walk() computed by all cores.
    // Returns false - with nothing changed - when a child is a container or fails, so that the serial
    // walk handles it and reports the error.
    bool leaves_in_parallel(const std::vector<uint32_t>& order, const Affine& chain, uint32_t group, bool in_medium) {
        const size_t n = order.size();
        for (uint32_t c : order) {
            const uint32_t k = d.objects[c].kind;
            if (k != RT_OBJ_SPHERE && k != RT_OBJ_QUAD && k != RT_OBJ_TRIANGLE) return false;
        }
        RawVec<FlatPrim>& G = groups[group];
        const size_t base = G.size();
        G.resize(base + n);
        const uint32_t rank0 = next_rank;
        bool ok = true;
        uint64_t n_sph = 0;
#pragma omp parallel for schedule(static) reduction(&& : ok) reduction(+ : n_sph)
        for (size_t i = 0; i < n; i++) {
            // `order` is the tie order, a permutation: the object and its shape record are read at random - ask for them early
            if (i + 16 < n) __builtin_prefetch(&d.objects[order[i + 16]]);
            if (i + 8 < n) {
                const rt_object& po = d.objects[order[i + 8]];
                if (po.kind == RT_OBJ_SPHERE)
                    __builtin_prefetch(&d.spheres[po.data]);
                else
                    __builtin_prefetch(&d.planars[po.data]), __builtin_prefetch((const char*)&d.planars[po.data] + 64), __builtin_prefetch((const char*)&d.planars[po.data] + 128);
            }
            const uint32_t obj = order[i];
            FlatPrim& fp = G[base + i];
            uint32_t kind = 0;
            if (!leaf(obj, chain, fp.g, kind, fp.lo, fp.hi, nullptr, true)) {
                ok = false;
                continue;
            }
            fp.m.kind_mat = (kind << 30) | (out.materials[d.objects[obj].material].shade_class << META_CLASS_SHIFT) | d.objects[obj].material;
            fp.m.object = obj;
            fp.m.rank = in_medium ? 0 : rank0 + (uint32_t)i;
            fp.m.xform = chain.xform;
            if (!in_medium) out.ranks[obj] = fp.m.rank;
            n_sph += kind == PRIM_SPHERE;
        }
        if (!ok) {
            G.resize(base);
            return false;
        }
        if (!in_medium) next_rank += (uint32_t)n;
        out.n_spheres += (uint32_t)n_sph;
        out.n_planars += (uint32_t)(n - n_sph);
        return true;
    }

    // depth-first walk in tie order; group = which primitive set receives the leaves
    void walk(uint32_t obj, const Affine& chain, uint32_t group, bool in_medium) {
        if (status != RT_OK) return;
        const rt_object& o = d.objects[obj];
        switch (o.kind) {
            case RT_OBJ_SPHERE:
            case RT_OBJ_QUAD:
            case RT_OBJ_TRIANGLE: {
                FlatPrim fp;
                uint32_t kind;
                if (!leaf(obj, chain, fp.g, kind, fp.lo, fp.hi, nullptr)) return;
                fp.m.kind_mat = (kind << 30) | (out.materials[o.material].shade_class << META_CLASS_SHIFT) | o.material;
                fp.m.object = obj;
                fp.m.rank = in_medium ? 0 : next_rank++;
                if (!in_medium) out.ranks[obj] = fp.m.rank;
                fp.m.xform = chain.xform;
                groups[group].push_back(fp);
                if (kind == PRIM_SPHERE) out.n_spheres++; else out.n_planars++;
                break;
            }
            case RT_OBJ_LIST:
                for (uint32_t k = 0; k < o.child_count; k++) walk(d.children[o.first_child + k], chain, group, in_medium);
                break;
            case RT_OBJ_BVH: {
                std::vector<uint32_t> order(d.children + o.first_child, d.children + o.first_child + o.child_count);
                if (!((flags & RT_BUILD_NO_REF_RANKS) || in_medium)) bvh_visit_order(order);
                if (order.size() > 100000) timer.lap("  BVH::from_vec tie order");
                if (order.size() >= 4096 && leaves_in_parallel(order, chain, group, in_medium)) break;
                for (uint32_t c : order) walk(c, chain, group, in_medium);
                break;
            }
            case RT_OBJ_TRANSFORM: {
                Affine a;
                if (!push_xform(d.transforms[o.data], obj, chain, a)) return;
                walk(d.children[o.first_child], a, group, in_medium);
                break;
            }
            case RT_OBJ_MEDIUM: {
                if (in_medium) {
                    fail(RT_ERR_UNSUPPORTED, "a ConstantMedium inside the boundary of another medium is not supported");
                    return;
                }
                Medium m{};
                m.material = o.material;
                m.object = obj;
                m.rank = next_rank++;
                out.ranks[obj] = m.rank;
                m.neg_inv_density = d.media[o.data].neg_inv_density;
                m.medium_index = o.data;
                m.xform = chain.xform;
                groups.emplace_back();
                uint32_t g = (uint32_t)groups.size() - 1;
                group_of_medium.push_back(g);
                out.media.push_back(m);
                walk(d.children[o.first_child], chain, g, true);
                break;
            }
        }
    }

    void walk_lights(uint32_t obj, const Affine& chain, double weight) {
        if (status != RT_OK) return;
        const rt_object& o = d.objects[obj];
        switch (o.kind) {
            case RT_OBJ_SPHERE:
            case RT_OBJ_QUAD:
            case RT_OBJ_TRIANGLE: {
                Light l{};
                double lo[3], hi[3];
                if (!leaf(obj, chain, l.g, l.kind, lo, hi, &l.area)) return;
                l.xform = chain.xform;
                l.weight = weight;
                out.lights.push_back(l);
                break;
            }
            case RT_OBJ_LIST:
                if (o.child_count == 0) {
                    fail(RT_ERR_INVALID, "The collection of objects is empty! (lights, hits.rs:73)");
                    return;
                }
                for (uint32_t k = 0; k < o.child_count; k++)
                    walk_lights(d.children[o.first_child + k], chain, weight / (double)o.child_count);
                break;
            case RT_OBJ_TRANSFORM: {
                Affine a;
                if (!push_xform(d.transforms[o.data], obj, chain, a)) return;
                walk_lights(d.children[o.first_child], a, weight);
                break;
            }
            default:
                fail(RT_ERR_UNSUPPORTED, "lights may not contain a BVH or ConstantMedium: pdf_value/random are unimplemented!() there (hit.rs:51-59)");
        }
    }

    // RT2025_TIMING=1 prints the wall time of every phase to stderr
    struct PhaseTimer {
        bool on = getenv("RT2025_TIMING") != nullptr;
        std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
        void lap(const char* what) {
            if (!on) return;
            auto t1 = std::chrono::steady_clock::now();
            fprintf(stderr, "[rt2025 compile] %-28s %8.3f s\n", what, std::chrono::duration<double>(t1 - t0).count());
            t0 = t1;
        }
    };

    struct GroupBox {
        float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    };
    std::vector<GroupBox> group_boxes;
    bool is_world_group(const RawVec<FlatPrim>* g) const { return g == &groups[0]; }

    // leaves of the world tree whose box overlaps `b` (padded): the only primitives a segment inside `b` can meet
    // (sphere != nullptr: the boundary is that static, untransformed sphere {cx, cy, cz, r} - boxes are tested against the ball)
    bool overlapping_leaves(const GroupBox& b, const double* sphere, uint32_t ref, uint32_t* entry, uint32_t& n) const {
        if (ref == INVALID_REF) return true;
        if (ref & LEAF_FLAG) {
            if (n == MEDIUM_MAX_ENTRIES) return false;
            entry[n++] = ref;
            return true;
        }
        const Node& nd = out.nodes[ref];
        auto overlaps = [&](const float* lo, const float* hi) {
            for (int k = 0; k < 3; k++)
                if (!(lo[k] <= b.hi[k] && hi[k] >= b.lo[k])) return false;
            if (sphere) {
                double d2 = 0.0;
                for (int k = 0; k < 3; k++) {
                    const double c = sphere[k], dk = c < (double)lo[k] ? (double)lo[k] - c : (c > (double)hi[k] ? c - (double)hi[k] : 0.0);
                    d2 += dk * dk;
                }
                if (d2 > sphere[3] * sphere[3]) return false;
            }
            return true;
        };
        if (overlaps(nd.lo0, nd.hi0) && !overlapping_leaves(b, sphere, nd.child0, entry, n)) return false;
        if (overlaps(nd.lo1, nd.hi1) && !overlapping_leaves(b, sphere, nd.child1, entry, n)) return false;
        return true;
    }

    PhaseTimer timer;
    int run() {
        if (!validate()) return status;
        timer.lap("validate");
        copy_tables();
        timer.lap("copy tables");
        out.ranks.assign(d.n_objects, RT_NONE);
        groups.emplace_back();
        walk(d.world_root, Affine(), 0, false);
        if (status != RT_OK) return status;
        timer.lap("walk (ranks + leaves)");
        if (d.lights_root != RT_NONE) {
            walk_lights(d.lights_root, Affine(), 1.0);
            if (status != RT_OK) return status;
            double acc = 0.0;
            for (auto& l : out.lights) {
                acc += l.weight;
                l.cdf = acc;
            }
        }
        uint64_t total = 0;
        for (auto& g : groups) total += g.size();
        if (total >= (1ull << 28)) {
            fail(RT_ERR_UNSUPPORTED, "more than 2^28 primitives");
            return status;
        }
        out.geom.resize(total);
        out.meta.resize(total);
        uint32_t base = 0;
        std::vector<uint32_t> roots;
        for (auto& g : groups) {
            RawVec<BuildBox> boxes(g.size());
#pragma omp parallel for schedule(static) if (g.size() > 65536)
            for (size_t i = 0; i < g.size(); i++)
                for (int k = 0; k < 3; k++) boxes[i].lo[k] = round_down(g[i].lo[k]), boxes[i].hi[k] = round_up(g[i].hi[k]);
            {  // world box of the group (the boundary of a medium: MEDIUM_THICK entry leaves below)
                GroupBox gb;
                for (size_t i = 0; i < g.size(); i++)
                    for (int k = 0; k < 3; k++) gb.lo[k] = std::min(gb.lo[k], boxes[i].lo[k]), gb.hi[k] = std::max(gb.hi[k], boxes[i].hi[k]);
                if (!is_world_group(&g)) group_boxes.resize(groups.size()), group_boxes[&g - &groups[0]] = gb;
            }
            RawVec<uint32_t> order;
            timer.lap("build boxes");
            uint32_t root = INVALID_REF;
            const bool is_world = &g == &groups[0];
            if (is_world && world_builder && g.size() >= 4096 && world_builder(boxes, base, out.nodes, order, out.bvh_depth, root)) {
                timer.lap("device LBVH build");
            } else {
                // the boundary groups of the media are walked by the media kernel with a stack of their own depth
                root = build_bvh(boxes, base, out.nodes, order, is_world ? out.bvh_depth : out.media_bvh_depth);
                timer.lap("SAH build");
            }
#pragma omp parallel for schedule(static) if (g.size() > 65536)
            for (size_t i = 0; i < g.size(); i++) {
                out.geom[base + i] = g[order[i]].g;
                out.meta[base + i] = g[order[i]].m;
            }
            roots.push_back(root);
            base += (uint32_t)g.size();
            RawVec<FlatPrim>().swap(g);
            timer.lap("reorder primitives");
        }
        // Scenes that cannot stay in the caches are traversed through a four-wide collapse of the world tree (half
        // the dependent node fetches); RT2025_WIDE_BVH=0/1 overrides the size rule (tests force it on small scenes).
        // Small trees too, when the whole collapse fits in a traversal CTA's shared memory (api.cu checks, and falls back to the
        // binary nodes, which then fit as well): half the node visits at shared-memory latency - cornell extend 28.7 -> 25.9 ms,
        // book1 2.21 -> 2.03 ms.  In between (book2: 3201 nodes, the binary tree fills the shared memory) both are equal
        // and the tree stays binary.
        bool wide = out.nodes.size() > 8192 || out.nodes.size() * sizeof(Node) <= 170 * 1024;
        if (const char* e = getenv("RT2025_WIDE_BVH")) wide = atoi(e) != 0;
        // Renumber the nodes breadth first from the world root (then the media groups): any prefix of
        // the array is then the top of the tree, which the kernels stage in shared memory.  Skipped when the
        // world is traversed through the collapse (which is emitted breadth first itself): only the small media
        // trees still walk these nodes, and a 100 M-node renumbering is 6 s of serial host time.
        if (!wide) {
            const size_t n = out.nodes.size();
            std::vector<uint32_t> order;
            order.reserve(n);
            std::vector<uint32_t> new_index(n, 0xFFFFFFFFu);
            for (uint32_t root : roots) {
                if (root == INVALID_REF || (root & LEAF_FLAG)) continue;
                size_t head = order.size();
                new_index[root] = (uint32_t)order.size();
                order.push_back(root);
                while (head < order.size()) {
                    const Node& nd = out.nodes[order[head++]];
                    for (uint32_t c : {nd.child0, nd.child1})
                        if (!(c & LEAF_FLAG) && c != INVALID_REF) {
                            new_index[c] = (uint32_t)order.size();
                            order.push_back(c);
                        }
                }
            }
            RawVec<Node> sorted(order.size());
            for (size_t i = 0; i < order.size(); i++) {
                Node nd = out.nodes[order[i]];
                if (!(nd.child0 & LEAF_FLAG) && nd.child0 != INVALID_REF) nd.child0 = new_index[nd.child0];
                if (!(nd.child1 & LEAF_FLAG) && nd.child1 != INVALID_REF) nd.child1 = new_index[nd.child1];
                sorted[i] = nd;
            }
            out.nodes.swap(sorted);
            for (uint32_t& root : roots)
                if (root != INVALID_REF && !(root & LEAF_FLAG)) root = new_index[root];
        }
        timer.lap("breadth-first renumbering");
        out.world_root = roots[0];
        {
            if (wide) {
                out.world_root4 = collapse_bvh4(out.nodes, out.world_root, out.nodes4, out.bvh4_depth);
                if (3 * out.bvh4_depth + 2 > (uint32_t)TRAVERSAL_STACK) {  // would not fit the traversal stack: keep the binary tree
                    out.nodes4.clear();
                    out.world_root4 = INVALID_REF;
                }
                timer.lap("four-wide collapse");
            }
        }
        for (size_t m = 0; m < out.media.size(); m++) {
            Medium& med = out.media[m];
            med.root = roots[group_of_medium[m]];
            med.single_sphere = RT_NONE;
            if ((med.root & LEAF_FLAG) && med.root != INVALID_REF && (med.root & 7u) == 0) {
                uint32_t pi = (med.root & ~LEAF_FLAG) >> 3;
                if ((out.meta[pi].kind_mat >> 30) == PRIM_SPHERE) med.single_sphere = pi;
            }
        }
        if (timer.on) fprintf(stderr, "[rt2025 compile] %zu binary nodes (depth %u), %zu four-wide nodes (depth %u), %zu primitives\n", out.nodes.size(), out.bvh_depth, out.nodes4.size(), out.bvh4_depth, out.geom.size());
        // optically thick media (scene_types.h, MEDIUM_THICK): only when the sampling of EVERY medium is the closed-form
        // sphere test, because the random walk looks one segment ahead over all of them
        bool all_spheres = true;
        for (const Medium& med : out.media) all_spheres = all_spheres && med.single_sphere != RT_NONE;
        double min_depth = 1.0;
        if (const char* e = getenv("RT2025_WALK_MIN_DEPTH")) min_depth = atof(e);  // tuning knob; <= 0 switches the walk off
        for (Medium& med : out.media) {
            med.flags = 0;
            if (!all_spheres || !(min_depth > 0.0)) continue;
            const double radius = std::fabs(out.geom[med.single_sphere].d[6]);
            if (radius * std::fabs(1.0 / med.neg_inv_density) >= min_depth) med.flags |= MEDIUM_THICK;
        }
        for (size_t m = 0; m < out.media.size(); m++) {
            Medium& med = out.media[m];
            med.n_entry = MEDIUM_NO_ENTRIES;
            if (!(med.flags & MEDIUM_THICK) || getenv("RT2025_WALK_NO_ENTRIES")) continue;
            GroupBox b = group_boxes[group_of_medium[m]];
            for (int k = 0; k < 3; k++) {  // the scatter points are inside the boundary up to rounding
                const float pad = 1e-4f * std::max(1.0f, std::max(std::fabs(b.lo[k]), std::fabs(b.hi[k])));
                b.lo[k] -= pad, b.hi[k] += pad;
            }
            uint32_t n = 0;
            const double* g = out.geom[med.single_sphere].d;
            const bool plain = med.xform == RT_NONE && out.meta[med.single_sphere].xform == RT_NONE && g[3] == 0.0 && g[4] == 0.0 && g[5] == 0.0;
            const double ball[4] = {g[0], g[1], g[2], std::fabs(g[6]) * (1.0 + 1e-4) + 1e-4};
            if (overlapping_leaves(b, plain ? ball : nullptr, out.world_root, med.entry, n)) med.n_entry = n;
            if (timer.on) fprintf(stderr, "[rt2025 compile] medium %zu is optically thick: %d entry leaves\n", m, (int)med.n_entry);
        }
        walk_lean();
        if (timer.on) fprintf(stderr, "[rt2025 compile] random walk: %s\n", out.walk_lean.empty() ? "generic" : (out.walk_lean[0].shell != RT_NONE ? "lean, shell" : "lean"));
        shade_lean();
        if (timer.on) {
            std::string classes;
            const std::pair<uint32_t, const char*> names[] = {{SC_DIFFUSE, " diffuse"}, {SC_TEXTURED, " textured"}, {SC_ISOTROPIC, " isotropic"}, {SC_EMISSIVE, " emissive"}};
            for (const auto& c : names)
                if (out.shade_lean_mask & (1u << c.first)) classes += c.second;
            fprintf(stderr, "[rt2025 compile] shade lean:%s\n", classes.empty() ? " generic" : classes.c_str());
        }
        return RT_OK;
    }

    // scene_types.h, LeanLights: the staged light list, or false when the scene's list is not flat, is longer than LEAN_LIGHTS or
    // has a leaf below a Transform
    bool lean_lights(LeanLights& L) const {
        std::memset(&L, 0, sizeof(L));
        const size_t n = out.lights.size();
        if (n > LEAN_LIGHTS) return false;
        for (size_t i = 0; i < n; i++) {  // flat: every leaf weighs 1/n (rt_scene_create's test)
            const Light& l = out.lights[i];
            if (l.xform != RT_NONE || l.weight != 1.0 / (double)n) return false;
            L.lights[i] = l;
        }
        L.n = (uint32_t)n;
        return true;
    }

    // albedo / (4 pi) of an Isotropic over a solid texture, as shade_one computes it (D3 / double), or false for any other material
    bool isotropic_axp(uint32_t material, double* axp) const {
        const Material& iso = out.materials[material];
        if (iso.kind != RT_MAT_ISOTROPIC || iso.tex >= out.textures.size() || out.textures[iso.tex].kind != RT_TEX_SOLID) return false;
        for (int k = 0; k < 3; k++) axp[k] = (1.0 / (4.0 * 3.14159265358979323846264338327950288)) * out.textures[iso.tex].color[k];
        return true;
    }

    // scene_types.h, WalkLean: the record of the lean random walk when the scene qualifies, otherwise nothing
    void walk_lean() {
        out.walk_lean.clear();
        const size_t n_media = out.media.size();
        if (n_media > WALK_LEAN_MEDIA) return;
        WalkLean L;
        std::memset(&L, 0, sizeof(L));
        if (!lean_lights(L.lights)) return;
        L.n_media = (uint32_t)n_media, L.thick = RT_NONE, L.shell = RT_NONE;
        for (size_t m = 0; m < n_media; m++) {
            const Medium& med = out.media[m];
            if (med.single_sphere == RT_NONE || med.xform != RT_NONE || out.meta[med.single_sphere].xform != RT_NONE) return;
            if (med.flags & MEDIUM_THICK) {
                if (L.thick != RT_NONE || med.n_entry == MEDIUM_NO_ENTRIES) return;
                L.thick = (uint32_t)m;
            }
            std::memcpy(L.sphere[m], out.geom[med.single_sphere].d, 7 * sizeof(double));
            L.neg_inv_density[m] = med.neg_inv_density;
            L.rank[m] = med.rank, L.medium_index[m] = med.medium_index;
        }
        if (L.thick == RT_NONE) return;
        const Medium& thick = out.media[L.thick];
        if (!isotropic_axp(thick.material, L.axp)) return;
        for (uint32_t e = 0; e < thick.n_entry; e++) {
            const uint32_t first = (thick.entry[e] & ~LEAF_FLAG) >> 3, count = (thick.entry[e] & 7u) + 1;
            for (uint32_t pi = first; pi < first + count; pi++) {
                const PrimMeta& pm = out.meta[pi];
                if (L.n_prims == WALK_LEAN_PRIMS || pm.xform != RT_NONE) return;
                const uint32_t k = L.n_prims++;
                L.prim[k] = out.geom[pi];
                L.prim_kind[k] = pm.kind_mat >> 30, L.prim_rank[k] = pm.rank;
                // bit-identical (memcmp, not ==: -0.0 and NaN must not pass) centre, centre_vec and radius
                if (L.shell == RT_NONE && L.prim_kind[k] == PRIM_SPHERE && std::memcmp(out.geom[pi].d, L.sphere[L.thick], 7 * sizeof(double)) == 0) L.shell = k;
            }
        }
        out.walk_lean.push_back(L);
    }

    // scene_types.h, ShadeLean: which shade classes may run their lean kernel, and the record they stage
    void shade_lean() {
        out.shade_lean.clear();
        out.shade_lean_mask = 0;
        ShadeLean S;
        std::memset(&S, 0, sizeof(S));
        const bool lights = lean_lights(S.lights);
        // SC_ISOTROPIC: the scatter points of every medium that is not MEDIUM_THICK (those go to k_walk) land there
        bool iso = lights && out.media.size() <= SHADE_LEAN_MEDIA;
        for (size_t m = 0; iso && m < out.media.size(); m++) {
            const Medium& med = out.media[m];
            if (med.flags & MEDIUM_THICK) continue;
            iso = med.xform == RT_NONE && isotropic_axp(med.material, S.axp[m]);
        }
        // the classes of the surfaces: one with an Isotropic material would land in SC_ISOTROPIC as well
        bool emissive = true;
        for (size_t p = 0; p < out.meta.size() && (iso || emissive); p++) {
            const PrimMeta& pm = out.meta[p];
            const uint32_t cls = (pm.kind_mat >> META_CLASS_SHIFT) & 15u;
            if (cls == SC_ISOTROPIC) iso = false;
            if (cls == SC_EMISSIVE) {
                const Material& M = out.materials[pm.kind_mat & META_MAT_MASK];
                if (pm.xform != RT_NONE || M.kind != RT_MAT_DIFFUSE_LIGHT || M.inner != RT_NONE || M.tex >= out.textures.size() ||
                    out.textures[M.tex].kind != RT_TEX_SOLID)
                    emissive = false;
            }
        }
        if (lights) out.shade_lean_mask |= 1u << SC_DIFFUSE | 1u << SC_TEXTURED;
        if (iso) out.shade_lean_mask |= 1u << SC_ISOTROPIC;
        if (emissive) out.shade_lean_mask |= 1u << SC_EMISSIVE;
        if (out.shade_lean_mask) out.shade_lean.push_back(S);
    }
};

}  // namespace

int compile_scene(const rt_scene_desc& d, uint32_t flags, CompiledScene& out, std::string& err, WorldBuilder world_builder) {
    Compiler c{d, flags, out, err};
    c.world_builder = world_builder;
    return c.run();
}

}  // namespace rt
