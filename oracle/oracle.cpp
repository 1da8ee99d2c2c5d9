// oracle.cpp — CPU restatement of the reference path tracer (caidj0/Raytracer-2025).
//
// THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/, __graft_entry__.smoke() and the
// cpu_baseline / --impl reference legs of bench.py may load it.  The product (librt2025.so)
// never links, loads or calls anything in this directory.
//
// The reference is a Rust crate and no Rust toolchain exists in this image or on the GPU box,
// so the reference itself cannot be compiled (oracle/_ref does not exist).  This file restates
// its algorithm in C++ binary64 with the reference's container semantics — recursive
// ray_color, virtual dispatch, linear `Hittables`, median-split `BVH`, per-node divisions in the
// slab test — operation for operation; each function cites the file:line it follows.  Compile
// with -ffp-contract=off: rustc never contracts a*b+c into an fma.
//
// Pinning: the reference's own tests hold known answers only for AABB::hit (aabb.rs:213-227),
// longest_axis/union/from_points (aabb.rs:199-253), get_sphere_uv (sphere.rs:152-169), Ray::at,
// Vec3 algebra and quaternion rotation; tests/test_oracle_kat.py checks those through the orc_kat_*
// entry points below.  Hits, scatter, pdfs, media, textures and the tone map have no vectors
// in the reference and the reference cannot be run here; round 2 pinned them by other means:
//   * hand-derived exact vectors (inputs whose every intermediate is representable) for Sphere / Quad / Triangle / Transform /
//     ConstantMedium hits, Dielectric / Metal / Lambertian / Isotropic scatter, CosinePDF and the light pdfs - tests/test_oracle_kat_hand.py;
//   * independent restatements written from the Rust source in plain Python for Perlin noise and NoiseTexture, Disney::evaluate_disney
//     and DisneyPDF::generate with all their samplers, Checker / Image textures, the ACES fit, Portal / Transparent / Mix,
//     RemappedMaterial::remap_record (with and without a normal map) and the Triangle light - tests/test_perlin_restatement.py,
//     tests/test_disney_restatement.py, tests/test_restatements.py.
// What is left "parity unpinned" (SURVEY.md 8c): palette's sRGB encoder (crate not vendored; 8-bit codes are stated to +-1).
//
// The one deliberate difference: the reference draws from the unseeded thread RNG; here every
// draw is an addressed Philox4x32-10 sample (include/rt2025_rng.h), which the CUDA core uses too.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <limits>
#include <memory>
#include <string>
#include <vector>

#ifdef _OPENMP
#include <omp.h>
#endif

#include "rt2025.h"
#include "rt2025_rng.h"

namespace orc {

static const double PI = 3.14159265358979323846264338327950288;
static const double INF = std::numeric_limits<double>::infinity();

// ---------------------------------------------------------------- utils/vec3.rs
struct Vec3 {
    double e[3];
    Vec3() : e{0, 0, 0} {}
    Vec3(double x, double y, double z) : e{x, y, z} {}
    explicit Vec3(const double* p) : e{p[0], p[1], p[2]} {}
    double x() const { return e[0]; }
    double y() const { return e[1]; }
    double z() const { return e[2]; }
    double operator[](int i) const { return e[i]; }
    double& operator[](int i) { return e[i]; }
};
static inline Vec3 operator+(Vec3 a, Vec3 b) { return Vec3(a[0] + b[0], a[1] + b[1], a[2] + b[2]); }
static inline Vec3 operator-(Vec3 a, Vec3 b) { return Vec3(a[0] - b[0], a[1] - b[1], a[2] - b[2]); }
static inline Vec3 operator*(Vec3 a, Vec3 b) { return Vec3(a[0] * b[0], a[1] * b[1], a[2] * b[2]); }
static inline Vec3 vdiv(Vec3 a, Vec3 b) { return Vec3(a[0] / b[0], a[1] / b[1], a[2] / b[2]); }  // impl_op!(Div) vec3.rs:296
static inline Vec3 operator-(Vec3 a) { return Vec3(-a[0], -a[1], -a[2]); }
static inline Vec3 operator*(double s, Vec3 a) { return Vec3(s * a[0], s * a[1], s * a[2]); }   // vec3.rs:140-146
static inline Vec3 operator*(Vec3 a, double s) { return Vec3(a[0] * s, a[1] * s, a[2] * s); }   // vec3.rs:156-162
static inline Vec3 operator/(Vec3 a, double s) { return (1.0 / s) * a; }                        // vec3.rs:222-228
static inline double dot(Vec3 a, Vec3 b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }     // vec3.rs:107-109
static inline Vec3 cross(Vec3 a, Vec3 b) {                                                       // vec3.rs:111-117
    return Vec3(a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]);
}
static inline double length_squared(Vec3 a) { return a[0] * a[0] + a[1] * a[1] + a[2] * a[2]; }  // vec3.rs:96-98
static inline double length(Vec3 a) { return std::sqrt(length_squared(a)); }
// UnitVec3::from_vec3, vec3.rs:303-310
static inline bool unit_vector(Vec3 v, Vec3& out) {
    Vec3 r = v / length(v);
    out = r;
    return std::isfinite(r[0]) && std::isfinite(r[1]) && std::isfinite(r[2]);
}
// Rust f64::min/max return the other operand when one is NaN
static inline double rmin(double a, double b) { return std::isnan(a) ? b : (std::isnan(b) ? a : (a < b ? a : b)); }
static inline double rmax(double a, double b) { return std::isnan(a) ? b : (std::isnan(b) ? a : (a > b ? a : b)); }

// ---------------------------------------------------------------- utils/ray.rs
struct Ray {
    Vec3 orig, dir;
    double time = 0.0;
    Ray() {}
    Ray(Vec3 o, Vec3 d, double t = 0.0) : orig(o), dir(d), time(t) {}
    Vec3 at(double t) const { return orig + t * dir; }  // ray.rs:39-41
};

// ---------------------------------------------------------------- utils/interval.rs
struct Interval {
    double min, max;
    Interval() : min(0), max(0) {}
    static Interval make(double a, double b) {  // Interval::new, interval.rs:10-15
        Interval i;
        i.min = rmin(a, b);
        i.max = rmax(a, b);
        return i;
    }
    static Interval raw(double mn, double mx) {  // from_range / struct literal
        Interval i;
        i.min = mn;
        i.max = mx;
        return i;
    }
    bool contains(double x) const { return x >= min && x <= max; }  // :65-67
    double size() const { return rmax(max - min, 0.0); }            // :42-44
    static bool intersect(const Interval& a, const Interval& b, Interval& out) {  // :46-56
        double mx = rmin(a.max, b.max);
        double mn = rmax(a.min, b.min);
        if (mn <= mx) {
            out = raw(mn, mx);
            return true;
        }
        return false;
    }
    static Interval union_(Interval a, Interval b) { return raw(rmin(a.min, b.min), rmax(a.max, b.max)); }  // :58-63
};
static const Interval UNIVERSE = Interval::raw(-INF, INF);

// ---------------------------------------------------------------- aabb.rs
struct AABB {
    Interval x, y, z;
    static AABB empty() { return AABB{Interval::raw(INF, -INF), Interval::raw(INF, -INF), Interval::raw(INF, -INF)}; }
    static AABB from6(const double* b) { return AABB{Interval::raw(b[0], b[1]), Interval::raw(b[2], b[3]), Interval::raw(b[4], b[5])}; }
    const Interval& axis_interval(int n) const { return n == 0 ? x : (n == 1 ? y : z); }
    AABB pad_to_minimums() const {  // aabb.rs:43-51
        const double DELTA = 0.0001;
        auto f = [&](Interval t) {
            if (t.size() < DELTA) {
                double padding = DELTA / 2.0;  // Interval::expand, interval.rs:29-35
                return Interval::raw(t.min - padding, t.max + padding);
            }
            return t;
        };
        return AABB{f(x), f(y), f(z)};
    }
    static AABB from_points(Vec3 a, Vec3 b) {  // aabb.rs:21-28
        return AABB{Interval::make(a[0], b[0]), Interval::make(a[1], b[1]), Interval::make(a[2], b[2])}.pad_to_minimums();
    }
    // aabb.rs:62-78: one division per axis per call, NaN-suppressing Interval::new, try_fold intersect
    bool hit(const Ray& r, Interval ray_t) const {
        Interval acc = ray_t;
        for (int axis = 0; axis < 3; axis++) {
            const Interval& ax = axis_interval(axis);
            double adinv = 1.0 / r.dir[axis];
            double t0 = (ax.min - r.orig[axis]) * adinv;
            double t1 = (ax.max - r.orig[axis]) * adinv;
            Interval slab = Interval::make(t0, t1);
            Interval next;
            if (!Interval::intersect(acc, slab, next)) return false;
            acc = next;
        }
        return true;
    }
    int longest_axis() const {  // aabb.rs:80-92
        double lx = x.size(), ly = y.size(), lz = z.size();
        if (lx > ly) return lx > lz ? 0 : 2;
        return ly > lz ? 1 : 2;
    }
    static AABB union_(AABB a, AABB b) {  // aabb.rs:94-100
        return AABB{Interval::union_(a.x, b.x), Interval::union_(a.y, b.y), Interval::union_(a.z, b.z)};
    }
};

// ---------------------------------------------------------------- utils/quaternion.rs
struct Quaternion {
    double w, x, y, z;
    Quaternion conjugate() const { return Quaternion{w, -x, -y, -z}; }  // :84-91
    Quaternion mul(const Quaternion& r) const {                         // :94-104
        return Quaternion{w * r.w - x * r.x - y * r.y - z * r.z, w * r.x + x * r.w + y * r.z - z * r.y,
                          w * r.y - x * r.z + y * r.w + z * r.x, w * r.z + x * r.y - y * r.x + z * r.w};
    }
    Vec3 rotate_vector(Vec3 v) const {  // :72-82
        Quaternion qv{0.0, v[0], v[1], v[2]};
        Quaternion r = mul(qv).mul(conjugate());
        return Vec3(r.x, r.y, r.z);
    }
    static Quaternion from_axis_angle(Vec3 axis, double deg) {  // :39-51
        double half = (deg * (PI / 180.0)) * 0.5;
        double s = std::sin(half), c = std::cos(half);
        Vec3 a;
        unit_vector(axis, a);
        return Quaternion{c, a[0] * s, a[1] * s, a[2] * s};
    }
};

// ---------------------------------------------------------------- utils/onb.rs
struct ONB {
    Vec3 axis[3];
    bool ok = true;
    ONB() {}
    explicit ONB(Vec3 n) {  // onb.rs:8-22
        Vec3 a = std::fabs(n.x()) > 0.9 ? Vec3(0.0, 1.0, 0.0) : Vec3(1.0, 0.0, 0.0);
        Vec3 u;
        ok = unit_vector(cross(n, a), u);
        Vec3 w = cross(u, n);
        axis[0] = u, axis[1] = n, axis[2] = w;
    }
    Vec3 onb_to_world(Vec3 v) const { return v[0] * axis[0] + v[1] * axis[1] + v[2] * axis[2]; }  // :34-38
};

// ---------------------------------------------------------------- Philox4x32-10 (rt2025_rng.h)
struct Rand2 {
    double a, b;
};
static inline void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
    for (int r = 0; r < 10; r++) {
        uint64_t p0 = (uint64_t)RT_PHILOX_M0 * c[0];
        uint64_t p1 = (uint64_t)RT_PHILOX_M1 * c[2];
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c[0] = n0, c[1] = n1, c[2] = n2, c[3] = n3;
        k0 += RT_PHILOX_W0;
        k1 += RT_PHILOX_W1;
    }
}
static inline Rand2 philox_pair(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t segment, uint32_t slot) {
    uint32_t c[4] = {pixel, sample, segment, slot};
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    Rand2 r;
    r.a = (double)(((uint64_t)(c[0] >> 5) << 26) | (uint64_t)(c[1] >> 6)) * 0x1.0p-53;
    r.b = (double)(((uint64_t)(c[2] >> 5) << 26) | (uint64_t)(c[3] >> 6)) * 0x1.0p-53;
    return r;
}

// The per-path sampling context: stands in for the thread-local RNG of utils/random.rs.
struct PathCtx {
    uint64_t seed = 0;
    uint32_t pixel = 0, sample = 0, segment = 0;
    bool media_enabled = true;  // orc_closest_hit leaves media out (they are stochastic)
    const double* forced = nullptr;  // known-answer hooks only: every draw returns (forced[0], forced[1]) ...
    const double* forced_direction = nullptr;  // ... except RT_SLOT_DIRECTION, which returns this pair when it is set
    Rand2 draw(uint32_t slot) const {
        if (forced) {
            const double* f = (slot == RT_SLOT_DIRECTION && forced_direction) ? forced_direction : forced;
            return Rand2{f[0], f[1]};
        }
        return philox_pair(seed, pixel, sample, segment, slot);
    }
};

// ---------------------------------------------------------------- sampling helpers, vec3.rs
static inline Vec3 random_unit_vector(double r1, double r2) {  // vec3.rs:313-322
    double x = std::cos(2.0 * PI * r1) * 2.0 * std::sqrt(r2 * (1.0 - r2));
    double y = std::sin(2.0 * PI * r1) * 2.0 * std::sqrt(r2 * (1.0 - r2));
    double z = 1.0 - 2.0 * r2;
    return Vec3(x, y, z);
}
static inline Vec3 random_cosine_direction(double r1, double r2) {  // vec3.rs:333-343
    double phi = 2.0 * PI * r1;
    double x = std::sin(phi) * std::sqrt(r2);
    double y = std::sqrt(1.0 - r2);
    double z = std::cos(phi) * std::sqrt(r2);
    return Vec3(x, y, z);
}
static inline Vec3 reflect(Vec3 v, Vec3 n) { return v - 2.0 * dot(v, n) * n; }  // vec3.rs:71-73
static inline bool refract(Vec3 uv, Vec3 n, double relative_eta, Vec3& out) {  // vec3.rs:345-354
    double cos_theta = rmin(dot(-uv, n), 1.0);
    Vec3 out_perp = relative_eta * (uv + cos_theta * n);
    double out_parallel_length = std::sqrt(1.0 - length_squared(out_perp));
    if (std::isnan(out_parallel_length)) return false;
    Vec3 out_parallel = -out_parallel_length * n;
    out = out_perp + out_parallel;
    return true;
}

// ---------------------------------------------------------------- texture.rs
struct Scene;
struct Texture {
    virtual ~Texture() {}
    virtual Vec3 value(double u, double v, Vec3 p) const = 0;
};
struct SolidColor : Texture {  // texture.rs:32-36
    Vec3 albedo;
    Vec3 value(double, double, Vec3) const override { return albedo; }
};
struct CheckerTexture : Texture {  // texture.rs:59-73
    double inv_scale;
    const Texture *even, *odd;
    static int32_t as_i32(double x) {  // Rust `as i32` saturates, NaN -> 0
        if (std::isnan(x)) return 0;
        if (x >= 2147483647.0) return INT32_MAX;
        if (x <= -2147483648.0) return INT32_MIN;
        return (int32_t)x;
    }
    Vec3 value(double u, double v, Vec3 p) const override {
        int32_t xi = as_i32(std::floor(inv_scale * p.x()));
        int32_t yi = as_i32(std::floor(inv_scale * p.y()));
        int32_t zi = as_i32(std::floor(inv_scale * p.z()));
        int32_t sum = (int32_t)((uint32_t)xi + (uint32_t)yi + (uint32_t)zi);  // release-mode wrap
        bool is_even = sum % 2 == 0;
        return is_even ? even->value(u, v, p) : odd->value(u, v, p);
    }
};
struct ImageTexture : Texture {  // texture.rs:81-174, utils/image.rs:55-82
    uint32_t width = 0, height = 0;
    const float* texels = nullptr;  // RGBA32F
    bool linear = false, interp = false;
    static float srgb_to_linear(float x) {  // palette Srgb::into_linear<f32> (crate not vendored)
        if (x <= 0.04045f) return (float)(1.0 / 12.92) * x;
        return std::pow(std::fma(x, (float)(1.0 / 1.055), (float)(0.055 / 1.055)), 2.4f);
    }
    void pixel_data(uint32_t x, uint32_t y, float out[4]) const {  // image.rs:63-82
        x = std::min(x, width - 1);
        y = std::min(y, height - 1);
        const float* p = texels + ((size_t)y * width + x) * 4;
        if (linear) {
            for (int i = 0; i < 4; i++) out[i] = p[i];
        } else {
            for (int i = 0; i < 3; i++) out[i] = srgb_to_linear(p[i]);
            out[3] = p[3];
        }
    }
    static double abs_fract(double x) { return x - std::floor(x); }  // texture.rs:161-163
    static uint32_t as_u32(double x) {
        if (!(x > 0.0)) return 0;
        if (x >= 4294967295.0) return 0xFFFFFFFFu;
        return (uint32_t)x;
    }
    void get_pixel(double u, double v, float out[4]) const {
        u = abs_fract(u);
        v = 1.0 - abs_fract(v);
        if (!interp) {  // texture.rs:111-119
            uint32_t i = as_u32(u * (double)width), j = as_u32(v * (double)height);
            pixel_data(i, j, out);
            return;
        }
        // texture.rs:121-151
        double x = u * (double)width - 0.5, y = v * (double)height - 0.5;
        uint32_t x0 = as_u32(rmax(std::floor(x), 0.0)), y0 = as_u32(rmax(std::floor(y), 0.0));
        uint32_t x1 = std::min(x0 + 1, width - 1), y1 = std::min(y0 + 1, height - 1);
        double dx = x - (double)x0, dy = y - (double)y0;
        float p00[4], p10[4], p01[4], p11[4];
        pixel_data(x0, y0, p00), pixel_data(x1, y0, p10), pixel_data(x0, y1, p01), pixel_data(x1, y1, p11);
        for (int i = 0; i < 4; i++) {
            float v0 = p00[i] * (1.0f - (float)dx) + p10[i] * ((float)dx);
            float v1 = p01[i] * (1.0f - (float)dx) + p11[i] * ((float)dx);
            out[i] = v0 * (1.0f - (float)dy) + v1 * ((float)dy);
        }
    }
    Vec3 value(double u, double v, Vec3) const override {  // texture.rs:166-174
        if (height == 0) return Vec3(0.0, 1.0, 1.0);
        float px[4];
        get_pixel(u, v, px);
        return Vec3((double)px[0], (double)px[1], (double)px[2]);
    }
    double alpha(double u, double v) const {  // texture.rs:102-109
        if (height == 0) return 1.0;
        float px[4];
        get_pixel(u, v, px);
        return (double)px[3];
    }
};
struct NoiseTexture : Texture {  // texture.rs:191-196, utils/perlin.rs:40-89
    const rt_perlin* tab;
    double scale;
    double noise(Vec3 p) const {
        int64_t ijk[3];
        double uvw[3];
        for (int a = 0; a < 3; a++) {
            double fl = std::floor(p[a]);
            // Rust `as i64`: NaN -> 0, saturating at -2^63 and 2^63 - 1 (every double below 2^63 in magnitude converts exactly)
            ijk[a] = std::isnan(fl) ? 0 : (fl >= 0x1p63 ? INT64_MAX : (fl < -0x1p63 ? INT64_MIN : (int64_t)fl));
            uvw[a] = p[a] - fl;
        }
        Vec3 c[2][2][2];
        for (int di = 0; di < 2; di++)
            for (int dj = 0; dj < 2; dj++)
                for (int dk = 0; dk < 2; dk++) {  // ijk + 1 wraps at INT64_MAX: add in uint64_t
                    uint32_t idx = tab->perm_x[((uint64_t)ijk[0] + di) & 255] ^ tab->perm_y[((uint64_t)ijk[1] + dj) & 255] ^
                                   tab->perm_z[((uint64_t)ijk[2] + dk) & 255];
                    c[di][dj][dk] = Vec3(tab->randvec[idx]);
                }
        // perlin_interp, perlin.rs:73-89
        double u = uvw[0], v = uvw[1], w = uvw[2];
        double uu = u * u * (3.0 - 2.0 * u), vv = v * v * (3.0 - 2.0 * v), ww = w * w * (3.0 - 2.0 * w);
        double accum = 0.0;
        for (int i = 0; i < 2; i++)
            for (int j = 0; j < 2; j++)
                for (int k = 0; k < 2; k++) {
                    Vec3 weight_v(u - (double)i, v - (double)j, w - (double)k);
                    accum += ((double)i * uu + (double)(1 - i) * (1.0 - uu)) * ((double)j * vv + (double)(1 - j) * (1.0 - vv)) *
                             ((double)k * ww + (double)(1 - k) * (1.0 - ww)) * dot(c[i][j][k], weight_v);
                }
        return accum;
    }
    double turb(Vec3 p, int depth) const {  // perlin.rs:61-71
        double accum = 0.0, weight = 1.0;
        Vec3 temp_p = p;
        for (int i = 0; i < depth; i++) {
            accum = accum + weight * noise(temp_p);
            temp_p = 2.0 * temp_p;
            weight = 0.5 * weight;
        }
        return std::fabs(accum);
    }
    Vec3 value(double, double, Vec3 p) const override {
        return Vec3(0.5, 0.5, 0.5) * (1.0 + std::sin(scale * p.z() + 10.0 * turb(p, 7)));
    }
};
struct GradientTexture : Texture {  // RT_TEX_GRADIENT_Y (rt2025.h): the book-1 sky
    Vec3 c0, c1;
    Vec3 value(double, double, Vec3 p) const override {
        double a = 0.5 * (p.y() + 1.0);
        return (1.0 - a) * c0 + a * c1;
    }
};

// ---------------------------------------------------------------- hit.rs
struct Material;
struct HitRecord {
    Vec3 p, normal;
    const Material* mat = nullptr;
    double t = 0, u = 0, v = 0;
    bool front_face = false;
    // a Transform of the chain could not normalise its normal: the reference panics there (shapes.rs:107, .expect)
    bool normal_panic = false;
    uint32_t prim_id = RT_NONE, inst_id = RT_NONE;
    static HitRecord make(Vec3 p, Vec3 normal, const Material* mat, double t, double u, double v, const Ray& r_in) {  // hit.rs:24-43
        HitRecord h;
        h.front_face = dot(r_in.dir, normal) < 0.0;
        h.p = p;
        h.normal = h.front_face ? normal : -normal;
        h.mat = mat;
        h.t = t, h.u = u, h.v = v;
        return h;
    }
};

// ---------------------------------------------------------------- material.rs / pdf.rs
enum ScatterKind { SCATTER_NONE, SCATTER_COSINE, SCATTER_SPHERE, SCATTER_RAY, SCATTER_DISNEY };
// DisneyParameters, material/disney.rs:18-35
struct DisneyParameters {
    Vec3 base_color = Vec3(0.8, 0.8, 0.8);
    double roughness = 0.5, anisotropic = 0.0, sheen = 0.0, sheen_tint = 0.0, clearcoat = 0.0, clearcoat_gloss = 0.0;
    double specular_tint = 0.0, metallic = 0.0, ior = 1.45, flatness = 0.0, spec_trans = 0.0, diff_trans = 0.0;
    bool thin = false;
};
struct ScatterRecord {
    ScatterKind kind = SCATTER_NONE;
    Vec3 attenuation;
    ONB uvw;
    Ray ray;
    bool error = false;  // an unwrap()/expect() of the reference would have panicked
    bool fuzzed = false;  // SCATTER_RAY: the direction went through random_unit_vector (sin, cos), a Metal's fuzz
    // DisneyPDF { uvw, v_out, front_face, params }, disney.rs:515-520
    Vec3 v_out;
    bool front_face = false;
    DisneyParameters params;
};
struct Material {
    virtual ~Material() {}
    virtual ScatterRecord scatter(const Ray&, const HitRecord&, const PathCtx&, uint32_t /*mix level*/) const { return ScatterRecord(); }
    virtual Vec3 emitted(const Ray&, const HitRecord&) const { return Vec3(0, 0, 0); }
};
static ScatterRecord cosine_record(Vec3 albedo, Vec3 normal) {  // CosinePDF::new, pdf.rs:41-48
    ScatterRecord s;
    s.kind = SCATTER_COSINE;
    s.attenuation = albedo;
    s.uvw = ONB(normal);
    s.error = !s.uvw.ok;
    return s;
}
struct EmptyMaterial : Material {  // material.rs:38-47
    ScatterRecord scatter(const Ray&, const HitRecord& rec, const PathCtx&, uint32_t) const override {
        return cosine_record(Vec3(0.75, 0.75, 0.75), rec.normal);
    }
};
struct Lambertian : Material {  // material.rs:59-66
    const Texture* texture;
    ScatterRecord scatter(const Ray&, const HitRecord& rec, const PathCtx&, uint32_t) const override {
        return cosine_record(texture->value(rec.u, rec.v, rec.p), rec.normal);
    }
};
struct Metal : Material {  // material.rs:82-95
    Vec3 albedo;
    double fuzz;
    ScatterRecord scatter(const Ray& r_in, const HitRecord& rec, const PathCtx& ctx, uint32_t) const override {
        ScatterRecord s;
        Vec3 ud;
        if (!unit_vector(r_in.dir, ud)) return s;  // `?` -> None
        Vec3 raw_reflected = reflect(ud, rec.normal);
        Vec3 ur;
        if (!unit_vector(raw_reflected, ur)) return s;
        Rand2 xi = ctx.draw(RT_SLOT_MATERIAL);
        Vec3 reflected = ur + (fuzz * random_unit_vector(xi.a, xi.b));
        s.kind = SCATTER_RAY;
        s.attenuation = albedo;
        s.ray = Ray(rec.p, reflected, r_in.time);
        s.fuzzed = true;
        return s;
    }
};
struct Dielectric : Material {  // material.rs:110-144
    const Texture* attenuation;
    double refraction_index;
    static double reflectance(double cosine, double ri) {  // :110-114
        double r0 = (1.0 - ri) / (1.0 + ri);
        double r0_squared = r0 * r0;
        double x = 1.0 - cosine;
        double x2 = x * x;
        double x5 = x * (x2 * x2);  // powi(5)
        return r0_squared + (1.0 - r0_squared) * x5;
    }
    ScatterRecord scatter(const Ray& r_in, const HitRecord& rec, const PathCtx& ctx, uint32_t) const override {
        ScatterRecord s;
        double ri = rec.front_face ? 1.0 / refraction_index : refraction_index;
        Vec3 unit_direction;
        if (!unit_vector(r_in.dir, unit_direction)) {
            s.error = true;
            return s;
        }
        double cos_theta = rmin(dot(-unit_direction, rec.normal), 1.0);
        double sin_theta = std::sqrt(1.0 - cos_theta * cos_theta);
        bool cannot_refract = ri * sin_theta > 1.0;
        Vec3 direction;
        if (cannot_refract || reflectance(cos_theta, ri) > ctx.draw(RT_SLOT_MATERIAL).a) {
            direction = reflect(unit_direction, rec.normal);
        } else if (!refract(unit_direction, rec.normal, ri, direction)) {
            s.error = true;  // .unwrap() on None
            return s;
        }
        s.kind = SCATTER_RAY;
        s.attenuation = attenuation->value(rec.u, rec.v, rec.p);
        s.ray = Ray(rec.p, direction, r_in.time);
        return s;
    }
};
struct DiffuseLight : Material {  // material.rs:170-186
    const Texture* texture;
    const Material* material = nullptr;
    Vec3 emitted(const Ray& ray, const HitRecord& rec) const override {
        Vec3 self_emit = texture->value(rec.u, rec.v, rec.p);
        Vec3 mat_emit = material ? material->emitted(ray, rec) : Vec3(0, 0, 0);
        return self_emit + mat_emit;
    }
    ScatterRecord scatter(const Ray& r_in, const HitRecord& rec, const PathCtx& ctx, uint32_t lvl) const override {
        return material ? material->scatter(r_in, rec, ctx, lvl) : ScatterRecord();
    }
};
struct Isotropic : Material {  // material.rs:198-207
    const Texture* texture;
    ScatterRecord scatter(const Ray&, const HitRecord& rec, const PathCtx&, uint32_t) const override {
        ScatterRecord s;
        s.kind = SCATTER_SPHERE;
        s.attenuation = texture->value(rec.u, rec.v, rec.p);
        return s;
    }
};
struct Transparent : Material {  // material.rs:211-218
    ScatterRecord scatter(const Ray& r_in, const HitRecord& rec, const PathCtx&, uint32_t) const override {
        ScatterRecord s;
        s.kind = SCATTER_RAY;
        s.attenuation = Vec3(1, 1, 1);
        s.ray = Ray(rec.p, r_in.dir, r_in.time);
        return s;
    }
};
struct Mix : Material {  // material.rs:249-267
    const Material *mat1, *mat2;
    double ratio;
    const ImageTexture* alpha = nullptr;
    double get_ratio(const HitRecord& rec) const { return alpha ? alpha->alpha(rec.u, rec.v) : ratio; }
    ScatterRecord scatter(const Ray& r_in, const HitRecord& rec, const PathCtx& ctx, uint32_t lvl) const override {
        double r = get_ratio(rec);
        if (ctx.draw(RT_SLOT_MIX + 256u * lvl).a > r) return mat1->scatter(r_in, rec, ctx, lvl + 1);
        return mat2->scatter(r_in, rec, ctx, lvl + 1);
    }
    Vec3 emitted(const Ray& r_in, const HitRecord& rec) const override {
        double r = get_ratio(rec);
        return mat1->emitted(r_in, rec) * (1.0 - r) + mat2->emitted(r_in, rec) * r;
    }
};
struct Portal : Material {  // material/portal.rs:14-31
    Vec3 attenuation, offset;
    Quaternion q;
    ScatterRecord scatter(const Ray& r_in, const HitRecord& rec, const PathCtx&, uint32_t) const override {
        ScatterRecord s;
        s.kind = SCATTER_RAY;
        s.attenuation = attenuation;
        s.ray = Ray(rec.p + offset, q.rotate_vector(r_in.dir), r_in.time);
        return s;
    }
};

// PDF::value for the material pdfs — pdf.rs:22-29, 51-57, disney.rs:656-666
// ---------------------------------------------------------------- utils/fresnel.rs, material/disney.rs
namespace disney {
static inline double lerp(double a, double b, double t) { return a * (1.0 - t) + b * t; }  // utils.rs:14-19
static inline Vec3 lerp(Vec3 a, Vec3 b, double t) { return a * (1.0 - t) + b * t; }
static inline double clampd(double x, double lo, double hi) { return x < lo ? lo : (x > hi ? hi : x); }  // f64::clamp (NaN stays NaN)
static inline double pow5(double x) { double x2 = x * x; return x * (x2 * x2); }
// the UnitVec3 helpers of vec3.rs:372-420, quirks included: cos_theta2 is y (not y*y) and
// cos_phi / sin_phi compare against 1e8, so they are always 1
static inline double cos_theta(Vec3 w) { return w.y(); }
static inline double cos_theta2(Vec3 w) { return w.y(); }
static inline double sin_theta2(Vec3 w) { return clampd(1.0 - cos_theta2(w), 0.0, 1.0); }
static inline double sin_theta(Vec3 w) { return std::sqrt(sin_theta2(w)); }
static inline double tan_theta(Vec3 w) { return sin_theta(w) / cos_theta(w); }
static inline double cos_phi2(Vec3 w) { double st = sin_theta(w); double c = std::fabs(st) < 1e8 ? 1.0 : w.x() / st; return c * c; }
static inline double sin_phi2(Vec3 w) { double st = sin_theta(w); double c = std::fabs(st) < 1e8 ? 1.0 : w.z() / st; return c * c; }
static inline Vec3 reflect2(Vec3 v, Vec3 n) { return -v + 2.0 * dot(v, n) * n; }  // vec3.rs:76-78
static inline bool refract2(Vec3 v, Vec3 n, double eta, Vec3& out) {             // vec3.rs:357-366
    double ct = rmin(dot(v, n), 1.0);
    Vec3 out_perp = eta * (-v + ct * n);
    double len = std::sqrt(1.0 - length_squared(out_perp));
    if (std::isnan(len)) return false;
    out = out_perp + (-len * n);
    return true;
}
// fresnel.rs
static inline Vec3 schlick(Vec3 r0, double radians) { double e = pow5(1.0 - radians); return r0 + (Vec3(1, 1, 1) - r0) * e; }
static inline double schlick_weight(double u) { return pow5(clampd(1.0 - u, 0.0, 1.0)); }
static inline double schlick_f64(double r0, double radians) { return lerp(1.0, schlick_weight(radians), r0); }
static inline double schlick_r0_from_relative_ior(double eta) { return ((eta - 1.0) * (eta - 1.0)) / ((eta + 1.0) * (eta + 1.0)); }
static inline double dielectric(double cos_theta_in, double n_in, double n_out) {  // fresnel.rs:22-46
    cos_theta_in = clampd(cos_theta_in, -1.0, 1.0);
    if (cos_theta_in < 0.0) {
        std::swap(n_in, n_out);
        cos_theta_in = -cos_theta_in;
    }
    double sin_in = std::sqrt(rmax(1.0 - cos_theta_in * cos_theta_in, 0.0));
    double sin_out = n_in / n_out * sin_in;
    if (sin_out >= 1.0) return 1.0;
    double cos_out = std::sqrt(rmax(1.0 - sin_out * sin_out, 0.0));
    double r_par = (n_out * cos_theta_in - n_in * cos_out) / (n_out * cos_theta_in + n_in * cos_out);
    double r_perp = (n_in * cos_theta_in - n_out * cos_out) / (n_in * cos_theta_in + n_out * cos_out);
    return (r_par * r_par + r_perp * r_perp) / 2.0;
}
static inline Vec3 calculate_tint(Vec3 base) {  // disney.rs:425-433
    double lum = dot(Vec3(0.3, 0.6, 1.0), base);
    return lum > 0.0 ? base * (1.0 / lum) : Vec3(1, 1, 1);
}
static inline double gtr1(double dot_hl, double a) {  // :435-443
    if (a >= 1.0) return 1.0 / PI;
    double a2 = a * a;
    return (a2 - 1.0) / (PI * std::log(a2) * (1.0 + (a2 - 1.0) * dot_hl * dot_hl));
}
static inline double separable_smith_ggxg1(Vec3 w, double a) {  // :445-450
    double a2 = a * a, nv = w.y();
    return 2.0 / (1.0 + std::sqrt(a2 + (1.0 - a2) * nv * nv));
}
static inline double ggx_anisotropic_d(Vec3 h, double ax, double ay) {  // :452-460
    double hx2 = h.x() * h.x(), hy2 = h.z() * h.z(), ct2 = h.y() * h.y();
    double ax2 = ax * ax, ay2 = ay * ay;
    double q = hx2 / ax2 + hy2 / ay2 + ct2;
    return 1.0 / (PI * ax * ay * (q * q));
}
static inline double aniso_smith_g1(Vec3 w, Vec3 h, double ax, double ay, bool& error) {  // :462-480
    if (dot(w, h) <= 0.0) return 0.0;
    double att = std::fabs(tan_theta(w));
    if (std::isnan(att)) error = true;  // assert!
    if (std::isinf(att)) return 0.0;
    double a = std::sqrt(cos_phi2(w) * ax * ax + sin_phi2(w) * ay * ay);
    double at = a * att;
    double lambda = 0.5 * (-1.0 + std::sqrt(1.0 + at * at));
    return 1.0 / (1.0 + lambda);
}
static inline void aniso_params(double roughness, double anisotropic, double& ax, double& ay) {  // :482-488
    double aspect = std::sqrt(1.0 - 0.9 * anisotropic);
    double r2 = roughness * roughness;
    ax = rmax(0.001, r2 / aspect);
    ay = rmax(0.001, r2 * aspect);
}
static inline void vndf_pdf(Vec3 v_in, Vec3 h, Vec3 v_out, double ax, double ay, double& fwd, double& rev, bool& error) {  // :490-510
    double d = ggx_anisotropic_d(h, ax, ay);
    double g1v = aniso_smith_g1(v_out, h, ax, ay, error);
    fwd = g1v * std::fabs(dot(h, v_out)) * d / std::fabs(cos_theta(v_out));
    double g1l = aniso_smith_g1(v_in, h, ax, ay, error);
    rev = g1l * std::fabs(dot(h, v_in)) * d / std::fabs(cos_theta(v_in));
}
static inline double thin_transmission_roughness(double ior, double roughness) { return clampd((0.65 * ior - 0.35) * roughness, 0.0, 1.0); }

static Vec3 disney_fresnel(const DisneyParameters& P, Vec3 v_out, Vec3 h, Vec3 v_in, double relative_ior) {  // :177-200
    double dot_hv = dot(h, v_out);
    Vec3 tint = calculate_tint(P.base_color);
    Vec3 r0 = schlick_r0_from_relative_ior(relative_ior) * lerp(Vec3(1, 1, 1), tint, P.specular_tint);
    r0 = lerp(r0, P.base_color, P.metallic);
    double df = dielectric(dot_hv, 1.0, P.ior);
    Vec3 mf = schlick(r0, dot(v_in, h));
    return lerp(Vec3(df, df, df), mf, P.metallic);
}
static void evaluate_brdf(const DisneyParameters& P, Vec3 v_out, Vec3 h, Vec3 v_in, double relative_ior, Vec3& value, double& fwd, double& rev, bool& error) {  // :100-130
    double nl = cos_theta(v_in), nv = cos_theta(v_out);
    value = Vec3(0, 0, 0), fwd = 0.0, rev = 0.0;
    if (nl <= 0.0 || nv <= 0.0) return;
    double ax, ay;
    aniso_params(P.roughness, P.anisotropic, ax, ay);
    double d = ggx_anisotropic_d(h, ax, ay);
    double gl = aniso_smith_g1(v_in, h, ax, ay, error), gv = aniso_smith_g1(v_out, h, ax, ay, error);
    Vec3 f = disney_fresnel(P, v_out, h, v_in, relative_ior);
    vndf_pdf(v_in, h, v_out, ax, ay, fwd, rev, error);
    fwd = fwd / (4.0 * std::fabs(dot(v_in, h)));
    rev = rev / (4.0 * std::fabs(dot(v_out, h)));
    value = (d * gl * gv * f) / (4.0 * nl * nv);
}
static Vec3 evaluate_sheen(const DisneyParameters& P, Vec3 h, Vec3 v_in) {  // :132-146
    if (P.sheen <= 0.0) return Vec3(0, 0, 0);
    double dot_hl = dot(h, v_in);
    Vec3 tint = calculate_tint(P.base_color);
    return (P.sheen * lerp(Vec3(1, 1, 1), tint, P.sheen_tint)) * schlick_weight(dot_hl);
}
static void evaluate_clearcoat(const DisneyParameters& P, Vec3 v_out, Vec3 h, Vec3 v_in, double& value, double& fwd, double& rev) {  // :148-175
    value = fwd = rev = 0.0;
    if (P.clearcoat <= 0.0) return;
    double dot_nh = h.y(), dot_hl = dot(h, v_in);
    double d = gtr1(dot_nh, lerp(0.1, 0.001, P.clearcoat_gloss));
    double f = schlick_f64(0.04, dot_hl);
    double gl = separable_smith_ggxg1(v_in, 0.25), gv = separable_smith_ggxg1(v_out, 0.25);
    value = 0.25 * P.clearcoat * d * f * gl * gv;
    fwd = d / (4.0 * std::fabs(dot(v_in, h)));
    rev = d / (4.0 * std::fabs(dot(v_out, h)));
}
static Vec3 evaluate_spec_transmission(const DisneyParameters& P, Vec3 v_out, Vec3 h, Vec3 v_in, double ax, double ay, double relative_ior, bool& error) {  // :202-236
    double n2 = relative_ior * relative_ior;
    double anl = std::fabs(cos_theta(v_in)), anv = std::fabs(cos_theta(v_out));
    double dot_hl = dot(h, v_in), dot_hv = dot(h, v_out);
    double d = ggx_anisotropic_d(h, ax, ay);
    double gl = aniso_smith_g1(v_in, h, ax, ay, error), gv = aniso_smith_g1(v_out, h, ax, ay, error);
    double f = dielectric(dot_hv, 1.0, 1.0 / relative_ior);
    Vec3 color = P.base_color;
    if (P.thin) {
        color = Vec3(std::sqrt(color[0]), std::sqrt(color[1]), std::sqrt(color[2]));
        if (std::isnan(color[0]) || std::isnan(color[1]) || std::isnan(color[2])) error = true;  // Vec3::sqrt panics
    }
    double c = (std::fabs(dot_hl) * std::fabs(dot_hv)) / (anl * anv);
    double q = dot_hl + relative_ior * dot_hv;
    double t = n2 / (q * q);
    return (c * t * (1.0 - f) * gl * gv * d) * color;
}
static double evaluate_retro_diffuse(const DisneyParameters& P, Vec3 v_out, Vec3 v_in) {  // :272-290
    double anl = std::fabs(cos_theta(v_in)), anv = std::fabs(cos_theta(v_out));
    double roughness = P.roughness * P.roughness;
    double rr = 0.5 + 2.0 * anl * anl * roughness;
    double fl = schlick_weight(anl), fv = schlick_weight(anv);
    return rr * (fl + fv + fl * fv * (rr - 1.0));
}
static double evaluate_diffuse(const DisneyParameters& P, Vec3 v_out, Vec3 h, Vec3 v_in, bool thin) {  // :238-270
    double anl = std::fabs(cos_theta(v_in)), anv = std::fabs(cos_theta(v_out));
    double fl = schlick_weight(anl), fv = schlick_weight(anv);
    double hk = 0.0;
    if (thin && P.flatness > 0.0) {
        double roughness = P.roughness * P.roughness;
        double dot_hl = dot(h, v_in);
        double fss90 = dot_hl * dot_hl * roughness;
        double fss = lerp(1.0, fss90, fl) * lerp(1.0, fss90, fv);
        hk = 1.25 * (fss * (1.0 / (anl + anv) - 0.5) + 0.5);
    }
    double retro = evaluate_retro_diffuse(P, v_out, v_in);
    double subsurface = lerp(1.0, hk, thin ? P.flatness : 0.0);
    return 1.0 / PI * (retro + subsurface * (1.0 - 0.5 * fl) * (1.0 - 0.5 * fv));
}
static void lobe_pdfs(const DisneyParameters& P, double& p_spec, double& p_diff, double& p_clear, double& p_trans) {  // :403-422
    double metallic_brdf = P.metallic;
    double specular_bsdf = (1.0 - P.metallic) * P.spec_trans;
    double dielectric_brdf = (1.0 - P.spec_trans) * (1.0 - P.metallic);
    double sw = metallic_brdf + dielectric_brdf, tw = specular_bsdf, dw = dielectric_brdf, cw = 1.0 * clampd(P.clearcoat, 0.0, 1.0);
    double norm = 1.0 / (sw + tw + dw + cw);
    p_spec = sw * norm, p_trans = tw * norm, p_diff = dw * norm, p_clear = cw * norm;
}
// Disney::evaluate_disney, disney.rs:292-401
static void evaluate_disney(const DisneyParameters& P, Vec3 v_out, Vec3 v_in, bool front_face, Vec3& reflectance, double& forward_pdf, bool& error) {
    double relative_ior = front_face ? P.ior : 1.0 / P.ior;
    double nv = cos_theta(v_out), nl = cos_theta(v_in);
    bool is_transmission = nv * nl < 0.0;
    Vec3 h;
    if (!unit_vector(is_transmission ? v_in - v_out : v_in + v_out, h)) error = true;  // .expect
    reflectance = Vec3(0, 0, 0);
    forward_pdf = 0.0;
    double p_brdf, p_diffuse, p_clearcoat, p_spec_trans;
    lobe_pdfs(P, p_brdf, p_diffuse, p_clearcoat, p_spec_trans);
    double diffuse_weight = (1.0 - P.metallic) * (1.0 - P.spec_trans);
    double trans_weight = (1.0 - P.metallic) * P.spec_trans;
    bool upper = nl > 0.0 && nv > 0.0;
    if (upper && P.clearcoat > 0.0) {
        double cc, f, r;
        evaluate_clearcoat(P, v_out, h, v_in, cc, f, r);
        reflectance = reflectance + Vec3(cc, cc, cc);
        forward_pdf += p_clearcoat * f;
    }
    if (diffuse_weight > 0.0) {
        double fwd = std::fabs(cos_theta(v_in));
        double diffuse = evaluate_diffuse(P, v_out, h, v_in, P.thin);
        Vec3 sheen = evaluate_sheen(P, h, v_in);
        reflectance = reflectance + diffuse_weight * (diffuse * P.base_color + sheen);
        forward_pdf += p_diffuse * fwd;
    }
    if (trans_weight > 0.0) {
        double rscaled = P.thin ? thin_transmission_roughness(P.ior, P.roughness) : P.roughness;
        double tax, tay;
        aniso_params(rscaled, P.anisotropic, tax, tay);
        Vec3 t_v_out = is_transmission ? -v_out : v_out;
        Vec3 transmission = evaluate_spec_transmission(P, t_v_out, h, v_in, tax, tay, relative_ior, error);
        reflectance = reflectance + trans_weight * transmission;
        double fwd, rev;
        vndf_pdf(v_in, h, t_v_out, tax, tay, fwd, rev, error);
        double dot_lh = dot(h, v_in), dot_vh = dot(h, t_v_out);
        double q = dot_lh + relative_ior * dot_vh;
        double jacobian = (relative_ior * relative_ior * dot_lh) / (q * q);
        forward_pdf += p_spec_trans * fwd * std::fabs(jacobian);
    }
    if (upper) {
        Vec3 spec;
        double f, r;
        evaluate_brdf(P, v_out, h, v_in, relative_ior, spec, f, r, error);
        reflectance = reflectance + spec;
        forward_pdf += p_brdf * f;
    }
    reflectance = reflectance * std::fabs(nl);
    if (forward_pdf == 0.0) forward_pdf = INF;
}
// sample_ggx_vndf_anisotropic, disney.rs:690-716
static bool sample_vndf(Vec3 v_out, double ax, double ay, double u1, double u2, Vec3& out) {
    Vec3 v;
    if (!unit_vector(Vec3(v_out.x() * ax, v_out.y(), v_out.z() * ay), v)) return false;
    Vec3 t1 = v.y() < 0.9999999 ? cross(v, Vec3(0, 1, 0)) : Vec3(1, 0, 0);
    Vec3 t2 = cross(t1, v);
    double a = 1.0 / (1.0 + v.y());
    double r = std::sqrt(u1);
    double phi = u2 < a ? (u2 / a) * PI : PI + (u2 - a) / (1.0 - a) * PI;
    double p1 = r * std::cos(phi);
    double p2 = r * std::sin(phi) * (u2 < a ? 1.0 : v.y());
    Vec3 n = p1 * t1 + p2 * t2 + std::sqrt(rmax(1.0 - p1 * p1 - p2 * p2, 0.0)) * v;
    return unit_vector(Vec3(ax * n.x(), n.y(), ay * n.z()), out);
}
// DisneyPDF::generate, disney.rs:668-688; returns false for None
static bool generate(const ScatterRecord& s, const PathCtx& ctx, Vec3& out, bool& error) {
    const DisneyParameters& P = s.params;
    double p_spec, p_diff, p_clear, p_trans;
    lobe_pdfs(P, p_spec, p_diff, p_clear, p_trans);
    Rand2 pick = ctx.draw(RT_SLOT_DISNEY);
    Rand2 u = ctx.draw(RT_SLOT_DIRECTION);
    const Vec3 v_out = s.v_out;
    double p = pick.a;
    Vec3 v_in;
    if (p <= p_spec) {  // sample_disney_brdf :540-556
        double ax, ay;
        aniso_params(P.roughness, P.anisotropic, ax, ay);
        Vec3 h;
        if (!sample_vndf(v_out, ax, ay, u.a, u.b, h)) { error = true; return false; }
        if (!unit_vector(reflect2(v_out, h), v_in)) { error = true; return false; }
        if (cos_theta(v_in) <= 0.0) return false;
    } else if (p <= p_spec + p_clear) {  // sample_disney_clearcoat :558-587
        double a = 0.25, a2 = a * a;
        double ct = std::sqrt(rmax((1.0 - std::pow(a2, 1.0 - u.a)) / (1.0 - a2), 0.0));
        double st = std::sqrt(rmax(1.0 - ct * ct, 0.0));
        double phi = 2.0 * PI * u.b;
        Vec3 h(st * std::cos(phi), ct, st * std::sin(phi));
        if (dot(h, v_out) < 0.0) h = -h;
        v_in = reflect2(v_out, h);
        if (dot(v_in, v_out) < 0.0) return false;
    } else if (p <= p_spec + p_diff + p_clear) {  // sample_disney_diffuse :589-605
        double y = cos_theta(v_out);
        double sign = std::isnan(y) ? y : (std::signbit(y) ? -1.0 : 1.0);  // f64::signum
        v_in = sign * random_cosine_direction(u.a, u.b);
        if (pick.b <= P.diff_trans) v_in = -v_in;
        if (cos_theta(v_in) == 0.0) return false;
    } else if (p_trans >= 0.0) {  // disney_spec_transmission :607-664
        double ior = s.front_face ? P.ior : 1.0 / P.ior;
        if (cos_theta(v_out) == 0.0) return false;
        double rscaled = P.thin ? thin_transmission_roughness(ior, P.roughness) : P.roughness;
        double tax, tay;
        aniso_params(rscaled, P.anisotropic, tax, tay);
        Vec3 h;
        if (!sample_vndf(v_out, tax, tay, u.a, u.b, h)) { error = true; return false; }
        double dot_vh = dot(v_out, h);
        if (h.y() < 0.0) dot_vh = -dot_vh;
        double ni = v_out.y() > 0.0 ? 1.0 : ior, nt = v_out.y() > 0.0 ? ior : 1.0;
        double relative_ior = ni / nt;
        double f = dielectric(dot_vh, 1.0, P.ior);
        if (pick.b <= f) {
            if (!unit_vector(reflect2(v_out, h), v_in)) { error = true; return false; }
        } else if (P.thin) {
            Vec3 wi = reflect2(v_out, h);
            if (!unit_vector(Vec3(wi.x(), -wi.y(), wi.z()), v_in)) { error = true; return false; }
        } else if (!refract2(v_out, h, relative_ior, v_in)) {
            if (!unit_vector(reflect2(v_out, h), v_in)) { error = true; return false; }
        }
        if (cos_theta(v_in) == 0.0) return false;
    } else {
        error = true;  // panic!("The conditions should be exhausted!")
        return false;
    }
    if (!unit_vector(s.uvw.onb_to_world(v_in), out)) { error = true; return false; }
    return true;
}
}  // namespace disney

struct Disney : Material {  // material/disney.rs:57-91
    DisneyParameters params;
    const Texture* base_color_tex = nullptr;  // the OBJ loader's param_fn reads base_color from a texture (obj.rs:273-285)
    ScatterRecord scatter(const Ray& r_in, const HitRecord& rec, const PathCtx&, uint32_t) const override {
        ScatterRecord s;
        Vec3 v_out;
        if (!unit_vector(-r_in.dir, v_out)) {
            s.error = true;
            return s;
        }
        s.kind = SCATTER_DISNEY;
        s.uvw = ONB(rec.normal);
        if (!s.uvw.ok) s.error = true;
        s.v_out = Vec3(dot(v_out, s.uvw.axis[0]), dot(v_out, s.uvw.axis[1]), dot(v_out, s.uvw.axis[2]));  // world_to_onb, onb.rs:40-45
        s.front_face = rec.front_face;
        s.params = params;
        if (base_color_tex) s.params.base_color = base_color_tex->value(rec.u, rec.v, rec.p);
        return s;
    }
};

struct RemappedMaterial : Material {  // shapes/obj.rs:20-81
    const Material* material;
    Vec3 tex_ori, tex_u, tex_v, u_vec, v_vec, normal[3];
    bool has_uv_vecs = false;
    const Texture* normal_tex = nullptr;
    HitRecord remap_record(const HitRecord& rec, bool& error) const {  // :32-62
        Vec3 tex_coord = tex_ori + rec.u * tex_u + rec.v * tex_v;
        Vec3 n;
        if (!unit_vector((1.0 - rec.u - rec.v) * normal[0] + rec.u * normal[1] + rec.v * normal[2], n)) error = true;
        if (normal_tex) {
            Vec3 c = normal_tex->value(tex_coord.x(), tex_coord.y(), rec.p);
            c = c * 2.0 - Vec3(1.0, 1.0, 1.0);
            if (!has_uv_vecs) error = true;  // .unwrap() on None
            Vec3 raw = u_vec * c[0] + v_vec * c[1] + n * c[2];
            if (!unit_vector(raw, n)) error = true;
        }
        HitRecord out = rec;
        out.normal = n;
        out.u = tex_coord.x();
        out.v = tex_coord.y();
        return out;
    }
    ScatterRecord scatter(const Ray& r_in, const HitRecord& rec, const PathCtx& ctx, uint32_t lvl) const override {
        bool error = false;
        HitRecord r2 = remap_record(rec, error);
        ScatterRecord s = material->scatter(r_in, r2, ctx, lvl);
        if (error) s.error = true;
        return s;
    }
    Vec3 emitted(const Ray& r_in, const HitRecord& rec) const override {
        bool error = false;
        return material->emitted(r_in, remap_record(rec, error));
    }
};

static bool pdf_value(const ScatterRecord& s, Vec3 direction, Vec3& brdf, double& pdf) {
    if (s.kind == SCATTER_DISNEY) {
        Vec3 ud;
        if (!unit_vector(direction, ud)) return false;  // .unwrap()
        Vec3 v_in(dot(ud, s.uvw.axis[0]), dot(ud, s.uvw.axis[1]), dot(ud, s.uvw.axis[2]));
        bool error = false;
        disney::evaluate_disney(s.params, s.v_out, v_in, s.front_face, brdf, pdf, error);
        return !error;
    }
    if (s.kind == SCATTER_SPHERE) {
        pdf = 1.0 / (4.0 * PI);
        brdf = s.attenuation / (4.0 * PI);
        return true;
    }
    Vec3 ud;
    if (!unit_vector(direction, ud)) return false;  // .unwrap()
    double cosine_theta = dot(ud, s.uvw.axis[1]);
    pdf = rmax(0.0, cosine_theta / PI);
    brdf = s.attenuation * rmax(cosine_theta, 0.0) / PI;
    return true;
}
// PDF::generate; false = None (only the Disney lobes can decline, disney.rs:551,583,600,660)
static bool pdf_generate(const ScatterRecord& s, const PathCtx& ctx, Vec3& out, bool& error) {  // pdf.rs:31-33, 59-63
    if (s.kind == SCATTER_DISNEY) return disney::generate(s, ctx, out, error);
    Rand2 u = ctx.draw(RT_SLOT_DIRECTION);
    out = s.kind == SCATTER_SPHERE ? random_unit_vector(u.a, u.b) : s.uvw.onb_to_world(random_cosine_direction(u.a, u.b));
    return true;
}

// ---------------------------------------------------------------- Hittable and its implementors
struct LightSample {
    uint32_t leaf;  // chosen light leaf (global depth-first index)
    double r1, r2;
    bool error = false;
};
struct Hittable {
    AABB bbox;
    uint32_t id = RT_NONE;
    uint32_t first_leaf = 0, n_leaves = 0;  // light-leaf range when part of a lights tree
    virtual ~Hittable() {}
    virtual bool hit(const Ray& r, const Interval& interval, const PathCtx& ctx, HitRecord& rec) const = 0;
    virtual double pdf_value(Vec3 /*origin*/, Vec3 /*direction*/) const { return std::nan(""); }  // unimplemented!()
    virtual Vec3 random(Vec3 /*origin*/, LightSample& ls) const {
        ls.error = true;
        return Vec3(1, 0, 0);
    }
    virtual bool can_be_light() const { return false; }
    virtual void count_leaves(uint32_t& next) {
        first_leaf = next;
        n_leaves = 1;
        next += 1;
    }
};

struct Sphere : Hittable {  // shapes/sphere.rs
    Vec3 center, center_vec;
    double radius;
    const Material* mat;
    bool can_be_light() const override { return true; }
    static void get_sphere_uv(Vec3 p, double& u, double& v) {  // :53-61
        double theta = std::acos(-p.y());
        double phi = std::atan2(-p.z(), p.x()) + PI;
        u = phi / (2.0 * PI);
        v = theta / PI;
    }
    bool hit(const Ray& r, const Interval& interval, const PathCtx&, HitRecord& rec) const override {  // :77-108
        Vec3 current_center = center + r.time * center_vec;
        Vec3 oc = current_center - r.orig;
        double a = length_squared(r.dir);
        double h = dot(r.dir, oc);
        double c = length_squared(oc) - radius * radius;
        double discriminant = h * h - a * c;
        if (discriminant < 0.0) return false;
        double sqrtd = std::sqrt(discriminant);
        double root = (h - sqrtd) / a;
        if (!interval.contains(root)) {
            root = (h + sqrtd) / a;
            if (!interval.contains(root)) return false;
        }
        Vec3 p = r.at(root);
        Vec3 outward_normal = (p - current_center) / radius;
        double u, v;
        get_sphere_uv(outward_normal, u, v);
        rec = HitRecord::make(p, outward_normal, mat, root, u, v, r);
        rec.prim_id = id;
        return true;
    }
    double pdf_value(Vec3 origin, Vec3 direction) const override {  // :114-132
        HitRecord rec;
        PathCtx none;
        if (!hit(Ray(origin, direction), Interval::make(1e-8, INF), none, rec)) return 0.0;
        double dist_squared = length_squared((center + 0.0 * center_vec) - origin);
        double cos_theta_max = std::sqrt(1.0 - radius * radius / dist_squared);
        if (std::isnan(cos_theta_max)) return 1.0 / (4.0 * PI);
        double solid_angle = 2.0 * PI * (1.0 - cos_theta_max);
        return 1.0 / solid_angle;
    }
    Vec3 random(Vec3 origin, LightSample& ls) const override {  // :134-144, :63-73
        Vec3 direction = (center + 0.0 * center_vec) - origin;
        double distance_squared = length_squared(direction);
        Vec3 ud;
        if (!unit_vector(direction, ud)) ls.error = true;
        ONB uvw(ud);
        if (!uvw.ok) ls.error = true;
        double r1 = ls.r1, r2 = ls.r2;
        double y = 1.0 + r2 * (std::sqrt(1.0 - radius * radius / distance_squared) - 1.0);
        double phi = 2.0 * PI * r1;
        double x = std::cos(phi) * std::sqrt(1.0 - y * y);
        double z = std::sin(phi) * std::sqrt(1.0 - y * y);
        Vec3 out;
        if (!unit_vector(uvw.onb_to_world(Vec3(x, y, z)), out)) ls.error = true;
        return out;
    }
};

struct PlanarShape : Hittable {  // shapes/quad.rs, shapes/triangle.rs
    bool triangle;
    Vec3 anchor, u, v, w, normal;
    double parm_d, area;
    const Material* mat;
    bool can_be_light() const override { return true; }
    bool is_interior(double a, double b) const {  // quad.rs:60-68, triangle.rs:56-65
        const Interval unit = Interval::raw(0.0, 1.0);
        if (triangle) return unit.contains(a) && unit.contains(b) && unit.contains(a + b);
        return unit.contains(a) && unit.contains(b);
    }
    bool hit(const Ray& r, const Interval& interval, const PathCtx&, HitRecord& rec) const override {  // quad.rs:71-102
        double denom = dot(normal, r.dir);
        if (std::fabs(denom) < 1e-8) return false;
        double t = (parm_d - dot(normal, r.orig)) / denom;
        if (!interval.contains(t)) return false;
        Vec3 intersection = r.at(t);
        Vec3 hp = intersection - anchor;
        double alpha = dot(w, cross(hp, v));
        double beta = dot(w, cross(u, hp));
        if (!is_interior(alpha, beta)) return false;
        rec = HitRecord::make(intersection, normal, mat, t, alpha, beta, r);
        rec.prim_id = id;
        return true;
    }
    double pdf_value(Vec3 origin, Vec3 direction) const override {  // quad.rs:108-120
        HitRecord rec;
        PathCtx none;
        if (!hit(Ray(origin, direction), Interval::make(1e-8, INF), none, rec)) return 0.0;
        double distance_squared = rec.t * rec.t * length_squared(direction);
        double cosine = std::fabs(dot(direction, rec.normal) / length(direction));
        return distance_squared / (cosine * area);
    }
    Vec3 random(Vec3 origin, LightSample& ls) const override {  // quad.rs:122-125, triangle.rs:115-128
        double ul = ls.r1, vl = ls.r2;
        if (triangle && ul + vl > 1.0) {
            double nu = 1.0 - vl, nv = 1.0 - ul;
            ul = nu, vl = nv;
        }
        Vec3 p = anchor + (ul * u) + (vl * v);
        Vec3 out;
        if (!unit_vector(p - origin, out)) ls.error = true;
        return out;
    }
};

struct Hittables : Hittable {  // hits.rs
    std::vector<Hittable*> objects;
    bool can_be_light() const override { return true; }
    bool hit(const Ray& r, const Interval& interval, const PathCtx& ctx, HitRecord& rec) const override {  // :39-46
        bool any = false;
        HitRecord tmp;
        for (auto* o : objects) {
            if (o->hit(r, interval, ctx, tmp)) {
                if (!any || tmp.t < rec.t) rec = tmp;  // min_by keeps the first of equal minima
                any = true;
            }
        }
        return any;
    }
    double pdf_value(Vec3 origin, Vec3 direction) const override {  // :52-67
        double sum = 0.0;
        for (auto* o : objects) sum += o->pdf_value(origin, direction);
        return sum / (double)objects.size();
    }
    Vec3 random(Vec3 origin, LightSample& ls) const override {  // :69-75 — child that owns the chosen leaf
        for (auto* o : objects)
            if (ls.leaf >= o->first_leaf && ls.leaf < o->first_leaf + o->n_leaves) return o->random(origin, ls);
        ls.error = true;  // "The collection of objects is empty!"
        return Vec3(1, 0, 0);
    }
    void count_leaves(uint32_t& next) override {
        first_leaf = next;
        for (auto* o : objects) o->count_leaves(next);
        n_leaves = next - first_leaf;
    }
};

struct BVHNode : Hittable {  // bvh.rs
    Hittable *left = nullptr, *right = nullptr;
    bool hit(const Ray& r, const Interval& interval, const PathCtx& ctx, HitRecord& rec) const override {  // :57-85
        if (!bbox.hit(r, interval)) return false;
        bool hit_left = false, hit_right = false;
        HitRecord rec_left, rec_right;
        double closest_so_far = interval.max;
        if (left && left->hit(r, interval, ctx, rec_left)) {
            closest_so_far = rec_left.t;
            hit_left = true;
        }
        if (right) {
            Interval right_interval = Interval::make(interval.min, closest_so_far);
            if (right->hit(r, right_interval, ctx, rec_right)) hit_right = true;
        }
        if (hit_right) {
            rec = rec_right;
            return true;
        }
        if (hit_left) {
            rec = rec_left;
            return true;
        }
        return false;
    }
};

struct Transform : Hittable {  // shapes.rs:23-133
    Hittable* object;
    Vec3 offset, scale;
    Quaternion q;
    bool can_be_light() const override { return object->can_be_light(); }
    Vec3 transform(Vec3 v) const { return q.rotate_vector(v * scale) + offset; }                 // :74-78
    Vec3 detransform(Vec3 v) const { return vdiv(q.conjugate().rotate_vector(v - offset), scale); }  // :80-84
    bool hit(const Ray& r, const Interval& interval, const PathCtx& ctx, HitRecord& rec) const override {  // :88-111
        Vec3 to = r.at(1.0);
        Vec3 local_origin = detransform(r.orig);
        Vec3 local_to = detransform(to);
        Ray local_ray(local_origin, local_to - local_origin, r.time);
        if (!object->hit(local_ray, interval, ctx, rec)) return false;
        rec.p = transform(rec.p);
        Vec3 n;
        if (!unit_vector(q.rotate_vector(vdiv(rec.normal, scale)), n)) rec.normal_panic = true;
        rec.normal = n;
        if (rec.inst_id == RT_NONE) rec.inst_id = id;
        return true;
    }
    double pdf_value(Vec3 origin, Vec3 direction) const override {  // :117-123
        Vec3 local_origin = detransform(origin);
        Vec3 local_to = detransform(origin + direction);
        return object->pdf_value(local_origin, local_to - local_origin);
    }
    Vec3 random(Vec3 origin, LightSample& ls) const override {  // :125-132
        Vec3 local_origin = detransform(origin);
        Vec3 local_dir = object->random(local_origin, ls);
        Vec3 world_to = transform(local_origin + local_dir);
        Vec3 out;
        if (!unit_vector(world_to - origin, out)) ls.error = true;
        return out;
    }
    void count_leaves(uint32_t& next) override {
        first_leaf = next;
        object->count_leaves(next);
        n_leaves = next - first_leaf;
    }
};

struct ConstantMedium : Hittable {  // volume.rs
    Hittable* boundary;
    double neg_inv_density;
    const Material* phase;
    uint32_t medium_index;
    bool hit(const Ray& r, const Interval& interval, const PathCtx& ctx, HitRecord& rec) const override {  // :37-73
        if (!ctx.media_enabled) return false;
        HitRecord rec1, rec2;
        if (!boundary->hit(r, UNIVERSE, ctx, rec1)) return false;
        if (!boundary->hit(r, Interval::make(rec1.t + 0.0001, INF), ctx, rec2)) return false;
        if (rec1.t < interval.min) rec1.t = interval.min;  // clamp_min_assign
        if (rec2.t > interval.max) rec2.t = interval.max;  // clamp_max_assign
        if (rec1.t >= rec2.t) return false;
        if (rec1.t < 0.0) rec1.t = 0.0;
        double ray_length = length(r.dir);
        double distance_inside_boundary = (rec2.t - rec1.t) * ray_length;
        const Rand2 draw = ctx.draw(RT_MEDIUM_SLOT(medium_index));  // rt2025_rng.h: a for even media, b for odd ones
        double hit_distance = neg_inv_density * std::log((medium_index & 1u) ? draw.b : draw.a);
        if (hit_distance > distance_inside_boundary) return false;
        double t = rec1.t + hit_distance / ray_length;
        Vec3 p = r.at(t);
        rec = HitRecord::make(p, Vec3(1.0, 0.0, 0.0), phase, t, 0.0, 0.0, r);
        rec.prim_id = id;
        return true;
    }
};

// ---------------------------------------------------------------- scene assembly from rt_scene_desc
struct LightLeaf {
    double weight, cdf;
};
struct Scene {
    std::vector<std::unique_ptr<Texture>> textures;
    std::vector<std::unique_ptr<Material>> materials;
    std::vector<std::unique_ptr<Hittable>> owned;  // every node incl. BVH internals
    std::vector<Hittable*> by_object;               // desc object index -> node
    std::vector<rt_perlin> perlins;
    std::vector<float> texels;
    Hittable* world = nullptr;
    Hittable* lights = nullptr;
    std::vector<LightLeaf> light_leaves;
    std::vector<uint32_t> ranks;  // per desc object; RT_NONE for containers
    // flattened leaves for brute force: leaf + chain of transforms (outermost first)
    struct Leaf {
        Hittable* prim;
        std::vector<const Transform*> chain;
    };
    std::vector<Leaf> leaves;
    std::string error;
};

static uint64_t total_order_key(double x) {  // f64::total_cmp, bvh.rs:52
    uint64_t b;
    std::memcpy(&b, &x, 8);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

// BVH::from_vec, bvh.rs:16-46
static Hittable* build_bvh(Scene& sc, std::vector<Hittable*> objects) {
    auto* node = new BVHNode();
    sc.owned.emplace_back(node);
    AABB bbox = AABB::empty();
    for (auto* o : objects) bbox = AABB::union_(bbox, o->bbox);
    node->bbox = bbox;
    int axis = bbox.longest_axis();
    size_t len = objects.size();
    if (len == 1) {
        node->left = objects[0];
    } else if (len == 2) {
        node->left = objects[0];
        node->right = objects[1];
    } else {
        std::stable_sort(objects.begin(), objects.end(), [axis](const Hittable* a, const Hittable* b) {
            return total_order_key(a->bbox.axis_interval(axis).min) < total_order_key(b->bbox.axis_interval(axis).min);
        });
        size_t mid = len / 2;
        std::vector<Hittable*> left_vec(objects.begin(), objects.begin() + mid), right_vec(objects.begin() + mid, objects.end());
        node->left = build_bvh(sc, std::move(left_vec));
        node->right = build_bvh(sc, std::move(right_vec));
    }
    return node;
}

static Hittable* build_object(Scene& sc, const rt_scene_desc& d, uint32_t idx) {
    if (idx >= d.n_objects) {
        sc.error = "object index out of range";
        return nullptr;
    }
    const rt_object& o = d.objects[idx];
    Hittable* h = nullptr;
    auto kids = [&](std::vector<Hittable*>& out) {
        for (uint32_t k = 0; k < o.child_count; k++) {
            Hittable* c = build_object(sc, d, d.children[o.first_child + k]);
            if (!c) return false;
            out.push_back(c);
        }
        return true;
    };
    switch (o.kind) {
        case RT_OBJ_SPHERE: {
            auto* s = new Sphere();
            const rt_sphere& p = d.spheres[o.data];
            s->center = Vec3(p.center), s->center_vec = Vec3(p.center_vec), s->radius = p.radius;
            s->mat = sc.materials[o.material].get();
            h = s;
            break;
        }
        case RT_OBJ_QUAD:
        case RT_OBJ_TRIANGLE: {
            auto* q = new PlanarShape();
            const rt_planar& p = d.planars[o.data];
            q->triangle = o.kind == RT_OBJ_TRIANGLE;
            q->anchor = Vec3(p.anchor), q->u = Vec3(p.u), q->v = Vec3(p.v), q->w = Vec3(p.w), q->normal = Vec3(p.normal);
            q->parm_d = p.parm_d, q->area = p.area;
            q->mat = sc.materials[o.material].get();
            h = q;
            break;
        }
        case RT_OBJ_LIST: {
            auto* l = new Hittables();
            if (!kids(l->objects)) {
                delete l;
                return nullptr;
            }
            h = l;
            break;
        }
        case RT_OBJ_BVH: {
            std::vector<Hittable*> v;
            if (!kids(v)) return nullptr;
            if (v.empty()) {
                sc.error = "BVH node must contain at least one object";
                return nullptr;
            }
            h = build_bvh(sc, v);  // already owned
            h->id = idx;
            sc.by_object[idx] = h;
            return h;
        }
        case RT_OBJ_TRANSFORM: {
            auto* t = new Transform();
            const rt_transform& p = d.transforms[o.data];
            t->offset = Vec3(p.offset), t->scale = Vec3(p.scale);
            t->q = Quaternion{p.quat[0], p.quat[1], p.quat[2], p.quat[3]};
            t->object = build_object(sc, d, d.children[o.first_child]);
            if (!t->object) {
                delete t;
                return nullptr;
            }
            h = t;
            break;
        }
        case RT_OBJ_MEDIUM: {
            auto* m = new ConstantMedium();
            m->neg_inv_density = d.media[o.data].neg_inv_density;
            m->medium_index = o.data;
            m->phase = sc.materials[o.material].get();
            m->boundary = build_object(sc, d, d.children[o.first_child]);
            if (!m->boundary) {
                delete m;
                return nullptr;
            }
            h = m;
            break;
        }
        default:
            sc.error = "unknown object kind";
            return nullptr;
    }
    h->bbox = AABB::from6(o.bbox);
    h->id = idx;
    sc.owned.emplace_back(h);
    sc.by_object[idx] = h;
    return h;
}

// Appendix B of SURVEY.md: depth-first, list children in order, BVH right before left.
static void assign_ranks(Scene& sc, Hittable* h, uint32_t& next, std::vector<const Transform*>& chain) {
    if (auto* l = dynamic_cast<Hittables*>(h)) {
        for (auto* o : l->objects) assign_ranks(sc, o, next, chain);
    } else if (auto* b = dynamic_cast<BVHNode*>(h)) {
        if (b->right) assign_ranks(sc, b->right, next, chain);
        if (b->left) assign_ranks(sc, b->left, next, chain);
    } else if (auto* t = dynamic_cast<Transform*>(h)) {
        chain.push_back(t);
        assign_ranks(sc, t->object, next, chain);
        chain.pop_back();
    } else if (dynamic_cast<ConstantMedium*>(h)) {
        sc.ranks[h->id] = next++;  // the medium competes as one candidate; its boundary is private
    } else {
        sc.ranks[h->id] = next++;
        sc.leaves.push_back(Scene::Leaf{h, chain});
    }
}

static void light_weights(Hittable* h, double w, std::vector<LightLeaf>& out) {
    if (auto* l = dynamic_cast<Hittables*>(h)) {
        for (auto* o : l->objects) light_weights(o, w / (double)l->objects.size(), out);
    } else if (auto* t = dynamic_cast<Transform*>(h)) {
        light_weights(t->object, w, out);
    } else {
        out.push_back(LightLeaf{w, 0.0});
    }
}

static Scene* scene_from_desc(const rt_scene_desc* d, std::string& err) {
    auto sc = std::make_unique<Scene>();
    if (!d || d->version != RT_ABI_VERSION) {
        err = "bad descriptor version";
        return nullptr;
    }
    sc->perlins.assign(d->perlins, d->perlins + d->n_perlins);
    sc->texels.assign(d->texels, d->texels + d->n_texels);
    for (uint32_t i = 0; i < d->n_textures; i++) {
        const rt_texture& t = d->textures[i];
        Texture* out = nullptr;
        switch (t.kind) {
            case RT_TEX_SOLID: {
                auto* s = new SolidColor();
                s->albedo = Vec3(t.color);
                out = s;
                break;
            }
            case RT_TEX_CHECKER: {
                auto* c = new CheckerTexture();
                c->inv_scale = t.scale;
                if (t.a >= i || t.b >= i) {
                    err = "checker child texture must precede it";
                    delete c;
                    return nullptr;
                }
                c->even = sc->textures[t.a].get(), c->odd = sc->textures[t.b].get();
                out = c;
                break;
            }
            case RT_TEX_IMAGE: {
                auto* im = new ImageTexture();
                if (t.a != RT_NONE) {
                    const rt_image& ri = d->images[t.a];
                    im->width = ri.width, im->height = ri.height;
                    im->texels = sc->texels.data() + ri.texel_offset;
                    im->linear = (ri.flags & RT_IMG_LINEAR) != 0;
                    im->interp = (ri.flags & RT_IMG_INTERP) != 0;
                }
                out = im;
                break;
            }
            case RT_TEX_NOISE: {
                auto* n = new NoiseTexture();
                n->tab = &sc->perlins[t.a];
                n->scale = t.scale;
                out = n;
                break;
            }
            case RT_TEX_GRADIENT_Y: {
                auto* g = new GradientTexture();
                g->c0 = Vec3(t.color), g->c1 = Vec3(t.color2);
                out = g;
                break;
            }
            default:
                err = "unknown texture kind";
                return nullptr;
        }
        sc->textures.emplace_back(out);
    }
    for (uint32_t i = 0; i < d->n_materials; i++) {
        const rt_material& m = d->materials[i];
        Material* out = nullptr;
        auto tex = [&](uint32_t t) -> const Texture* { return t == RT_NONE ? nullptr : sc->textures[t].get(); };
        auto inner = [&](uint32_t k) -> const Material* { return (k == RT_NONE || k >= i) ? nullptr : sc->materials[k].get(); };
        switch (m.kind) {
            case RT_MAT_EMPTY: out = new EmptyMaterial(); break;
            case RT_MAT_LAMBERTIAN: { auto* x = new Lambertian(); x->texture = tex(m.tex); out = x; break; }
            case RT_MAT_METAL: { auto* x = new Metal(); x->albedo = Vec3(m.color); x->fuzz = m.param; out = x; break; }
            case RT_MAT_DIELECTRIC: { auto* x = new Dielectric(); x->attenuation = tex(m.tex); x->refraction_index = m.param; out = x; break; }
            case RT_MAT_DIFFUSE_LIGHT: { auto* x = new DiffuseLight(); x->texture = tex(m.tex); x->material = inner(m.inner); out = x; break; }
            case RT_MAT_ISOTROPIC: { auto* x = new Isotropic(); x->texture = tex(m.tex); out = x; break; }
            case RT_MAT_TRANSPARENT: out = new Transparent(); break;
            case RT_MAT_MIX: {
                auto* x = new Mix();
                x->mat1 = inner(m.inner), x->mat2 = inner(m.inner2), x->ratio = m.param;
                x->alpha = m.tex == RT_NONE ? nullptr : dynamic_cast<const ImageTexture*>(tex(m.tex));
                if (!x->mat1 || !x->mat2) { err = "Mix children must precede it"; delete x; return nullptr; }
                out = x;
                break;
            }
            case RT_MAT_PORTAL: {
                auto* x = new Portal();
                x->attenuation = Vec3(m.color), x->offset = Vec3(m.v);
                x->q = Quaternion{m.v[3], m.v[4], m.v[5], m.v[6]};
                out = x;
                break;
            }
            case RT_MAT_DISNEY: {
                auto* x = new Disney();
                DisneyParameters& P = x->params;
                P.base_color = Vec3(m.color);
                P.roughness = m.v[RT_DISNEY_ROUGHNESS], P.anisotropic = m.v[RT_DISNEY_ANISOTROPIC], P.sheen = m.v[RT_DISNEY_SHEEN];
                P.sheen_tint = m.v[RT_DISNEY_SHEEN_TINT], P.clearcoat = m.v[RT_DISNEY_CLEARCOAT], P.clearcoat_gloss = m.v[RT_DISNEY_CLEARCOAT_GLOSS];
                P.specular_tint = m.v[RT_DISNEY_SPECULAR_TINT], P.metallic = m.v[RT_DISNEY_METALLIC], P.ior = m.v[RT_DISNEY_IOR];
                P.flatness = m.v[RT_DISNEY_FLATNESS], P.spec_trans = m.v[RT_DISNEY_SPEC_TRANS], P.diff_trans = m.v[RT_DISNEY_DIFF_TRANS];
                P.thin = m.v[RT_DISNEY_THIN] != 0.0;
                x->base_color_tex = tex(m.tex);
                out = x;
                break;
            }
            case RT_MAT_REMAPPED: {
                auto* x = new RemappedMaterial();
                x->material = inner(m.inner);
                if (!x->material || m.inner2 >= d->n_remaps) { err = "bad RemappedMaterial"; delete x; return nullptr; }
                const rt_remap& r = d->remaps[m.inner2];
                x->tex_ori = Vec3(r.tex_ori), x->tex_u = Vec3(r.tex_u), x->tex_v = Vec3(r.tex_v);
                x->u_vec = Vec3(r.u_vec), x->v_vec = Vec3(r.v_vec);
                for (int k = 0; k < 3; k++) x->normal[k] = Vec3(r.normal[k]);
                x->has_uv_vecs = r.has_uv_vecs != 0;
                x->normal_tex = tex(r.normal_tex);
                out = x;
                break;
            }
            default: err = "unknown material kind"; return nullptr;
        }
        sc->materials.emplace_back(out);
    }
    sc->by_object.assign(d->n_objects, nullptr);
    sc->ranks.assign(d->n_objects, RT_NONE);
    sc->world = build_object(*sc, *d, d->world_root);
    if (!sc->world) {
        err = sc->error;
        return nullptr;
    }
    if (d->lights_root != RT_NONE) {
        sc->lights = build_object(*sc, *d, d->lights_root);
        if (!sc->lights) {
            err = sc->error;
            return nullptr;
        }
        if (!sc->lights->can_be_light()) {
            err = "lights contains a BVH or ConstantMedium: pdf_value/random are unimplemented!() (hit.rs:51-59)";
            return nullptr;
        }
        uint32_t next = 0;
        sc->lights->count_leaves(next);
        light_weights(sc->lights, 1.0, sc->light_leaves);
        double acc = 0.0;
        for (auto& l : sc->light_leaves) {
            acc += l.weight;
            l.cdf = acc;
        }
    }
    uint32_t next = 0;
    std::vector<const Transform*> chain;
    assign_ranks(*sc, sc->world, next, chain);
    return sc.release();
}

// ---------------------------------------------------------------- camera.rs
struct RenderCounters {
    uint64_t paths = 0, segments = 0, errors = 0;
};

// shapes/environment.rs:14-24
static Vec3 background_value(const Scene& sc, const rt_camera& cam, const Ray& ray, bool& error) {
    Vec3 p;
    if (!unit_vector(ray.dir, p)) {
        error = true;
        return Vec3(0, 0, 0);
    }
    double theta = std::acos(-p.y());
    double phi = PI - std::atan2(-p.z(), p.x());
    double u = phi / (2.0 * PI);
    double v = theta / PI;
    return sc.textures[cam.background_tex]->value(u, v, p);
}

// One level of Camera::ray_color (camera.rs:286-321): world.hit of r, then emission and the scatter of the hit.  `error` is set
// where the reference would panic.  Returns whether the path goes on with s.next: a ScatterRecord::Ray (s.attenuation), or a
// direction generated by the mixture pdf (s.albedo_x_pscatter, s.pdf_val).
struct Segment {
    bool hit = false;
    HitRecord rec;
    Vec3 background;               // miss: background_value
    Vec3 emission;                 // hit: rec.mat->emitted
    ScatterKind kind = SCATTER_NONE;
    Vec3 attenuation;              // SCATTER_RAY
    bool fuzzed = false;           // SCATTER_RAY: ScatterRecord::fuzzed
    Vec3 albedo_x_pscatter;        // the pdf kinds
    double pdf_val = 0.0;
    bool generated = false;        // the pdf kinds: generate() returned Some
    Ray next;
    bool error = false;
};
// The step after world.hit (camera.rs:288-321) on the HitRecord `rec` of r, or on a miss (rec == nullptr): the background, or
// emission, scatter, the mixture pdf and the next ray.  A record whose Transform normal could not be normalised is the panic of
// Transform::hit; its emission is still evaluated, as the device adds it before it ends the path.
static bool shade_record(const Scene& sc, const rt_camera& cam, const Ray& r, const HitRecord* hit, PathCtx& ctx, Segment& s) {
    bool& error = s.error;
    if (!hit) {
        s.background = background_value(sc, cam, r, error);
        return false;
    }
    s.hit = true;
    s.rec = *hit;
    const HitRecord& rec = s.rec;
    if (rec.normal_panic) error = true;
    s.emission = rec.mat->emitted(r, rec);
    if (error) return false;
    ScatterRecord srec = rec.mat->scatter(r, rec, ctx, 0);
    s.kind = srec.kind;
    if (srec.error) {
        error = true;
        return false;
    }
    if (srec.kind == SCATTER_NONE) return false;
    if (srec.kind == SCATTER_RAY) {
        s.attenuation = srec.attenuation;
        s.fuzzed = srec.fuzzed;
        s.next = srec.ray;
        return true;
    }
    // MixturePDF over (material pdf, HittablePDF(lights)) — camera.rs:297-304, pdf.rs:66-120
    Rand2 pick = ctx.draw(RT_SLOT_MIXTURE);
    Vec3 generate_vec;
    bool generated = true;
    if (sc.lights && !(pick.a < 0.5)) {
        Rand2 dirxi = ctx.draw(RT_SLOT_DIRECTION);
        LightSample ls;
        ls.leaf = (uint32_t)sc.light_leaves.size() - 1;
        for (uint32_t i = 0; i < sc.light_leaves.size(); i++)
            if (pick.b < sc.light_leaves[i].cdf) {
                ls.leaf = i;
                break;
            }
        ls.r1 = dirxi.a, ls.r2 = dirxi.b;
        generate_vec = sc.lights->random(rec.p, ls);
        if (ls.error) error = true;
    } else {
        generated = pdf_generate(srec, ctx, generate_vec, error);
    }
    if (error) return false;
    s.generated = generated;
    if (!generated) return false;  // `generate()` returned None: Color::BLACK (camera.rs:313-315)
    Ray scattered(rec.p, generate_vec, r.time);
    Vec3 albedo_x_pscatter;
    double value0;
    if (!pdf_value(srec, scattered.dir, albedo_x_pscatter, value0)) {
        error = true;
        return false;
    }
    double pdf_val = value0;
    if (sc.lights) {
        double value1 = sc.lights->pdf_value(rec.p, scattered.dir);
        if (std::isnan(value1)) error = true;                 // hits.rs:64 assert
        if (value0 == 0.0 && value1 == 0.0) error = true;     // pdf.rs:105-109 panic
        pdf_val = value0 * 0.5 + value1 * 0.5;
    }
    if (pdf_val == 0.0) error = true;  // camera.rs:309
    s.next = scattered;
    s.albedo_x_pscatter = albedo_x_pscatter;
    s.pdf_val = pdf_val;
    return !error;
}
static bool ray_step(const Scene& sc, const rt_camera& cam, const Ray& r, PathCtx& ctx, Segment& s) {
    HitRecord rec;
    const bool hit = sc.world->hit(r, Interval::raw(1e-8, INF), ctx, rec);
    return shade_record(sc, cam, r, hit ? &rec : nullptr, ctx, s);
}

// Camera::ray_color, camera.rs:275-325: ray_step, then the recursion.  `error` is set where the reference would panic.
static Vec3 ray_color(const Scene& sc, const rt_camera& cam, const Ray& r, uint32_t depth, PathCtx& ctx, RenderCounters& cnt, bool& error) {
    if (depth == 0) return Vec3(0, 0, 0);
    ctx.segment = cam.max_depth - depth;
    cnt.segments++;
    Segment s;
    const bool goes_on = ray_step(sc, cam, r, ctx, s);
    if (s.error) {
        error = true;
        return Vec3(0, 0, 0);
    }
    if (!s.hit) return s.background;
    if (!goes_on) return s.kind == SCATTER_NONE ? s.emission : s.emission + Vec3(0, 0, 0);
    Vec3 L = ray_color(sc, cam, s.next, depth - 1, ctx, cnt, error);
    Vec3 color_from_scatter = s.kind == SCATTER_RAY ? s.attenuation * L : (s.albedo_x_pscatter * L) / s.pdf_val;
    Vec3 ret = s.emission + color_from_scatter;
    if (std::isnan(ret[0]) || std::isnan(ret[1]) || std::isnan(ret[2])) error = true;  // camera.rs:323
    return ret;
}

// Camera::get_ray, camera.rs:247-273
static Ray get_ray(const rt_camera& cam, uint32_t i, uint32_t j, uint32_t s_i, uint32_t s_j, PathCtx& ctx) {
    ctx.segment = 0;
    Rand2 jit = ctx.draw(RT_SLOT_CAM_JITTER);
    double px = (((double)s_i + jit.a) * cam.recip_sqrt_spp) - 0.5;
    double py = (((double)s_j + jit.b) * cam.recip_sqrt_spp) - 0.5;
    Vec3 pixel_sample = Vec3(cam.pixel00_loc) + (((double)i + px) * Vec3(cam.pixel_delta_u)) + (((double)j + py) * Vec3(cam.pixel_delta_v));
    Vec3 ray_origin;
    if (cam.defocus_angle_in_degrees <= 0.0) {
        ray_origin = Vec3(cam.center);
    } else {  // defocus_disk_sample + random_in_unit_disk (vec3.rs:63-69)
        Rand2 d = ctx.draw(RT_SLOT_CAM_DISK);
        double theta = (2.0 * PI) * d.a;
        double rr = std::sqrt(d.b);
        double p0 = rr * std::cos(theta), p1 = rr * std::sin(theta);
        ray_origin = Vec3(cam.center) + (p0 * Vec3(cam.defocus_disk_u)) + (p1 * Vec3(cam.defocus_disk_v));
    }
    Vec3 ray_direction = pixel_sample - ray_origin;
    double ray_time = ctx.draw(RT_SLOT_CAM_TIME).a;
    return Ray(ray_origin, ray_direction, ray_time);
}

// utils/color.rs:14-36
static void to_rgb(Vec3 c, uint32_t toon_map, uint8_t out[3]) {
    if (toon_map == 1) {
        const double A = 2.51, C = 2.43;
        const Vec3 B(0.03, 0.03, 0.03), D(0.59, 0.59, 0.59), E(0.14, 0.14, 0.14);
        Vec3 m = vdiv(c * (A * c + B), c * (C * c + D) + E);
        for (int k = 0; k < 3; k++) c[k] = m[k] < 0.0 ? 0.0 : (m[k] > 1.0 ? 1.0 : m[k]);
    }
    for (int k = 0; k < 3; k++) {
        // palette Srgb::from_linear (crate not vendored): the standard piecewise sRGB curve, then
        // round to 8 bits.  palette's f32->u8 fast path may differ by 1 LSB at rounding boundaries.
        double x = c[k];
        double enc = x <= 0.0031308 ? 12.92 * x : 1.055 * std::pow(x, 1.0 / 2.4) - 0.055;
        if (!(enc > 0.0)) enc = 0.0;
        if (enc > 1.0) enc = 1.0;
        out[k] = (uint8_t)std::lround(enc * 255.0);
    }
}

}  // namespace orc

// =====================================================================================
// C entry points (ctypes)
// =====================================================================================
using namespace orc;

extern "C" {

static thread_local std::string g_orc_err;
const char* orc_last_error() { return g_orc_err.c_str(); }

void* orc_scene_create(const rt_scene_desc* d) {
    std::string err;
    Scene* s = scene_from_desc(d, err);
    if (!s) g_orc_err = err;
    return s;
}
void orc_scene_destroy(void* s) { delete (Scene*)s; }

int orc_get_ranks(const void* s, uint32_t* ranks, uint32_t n) {
    const Scene* sc = (const Scene*)s;
    if (n != sc->ranks.size()) return -1;
    std::copy(sc->ranks.begin(), sc->ranks.end(), ranks);
    return 0;
}

// mode 0: the reference's container semantics (world.hit, media left out)
// mode 1: brute force over every leaf shape with the full interval; exact ties -> lower rank
int orc_closest_hit(const void* s, const rt_ray* rays, uint64_t n, double t_min, double t_max, int mode, rt_hit* out) {
    const Scene* sc = (const Scene*)s;
    Interval iv = Interval::raw(t_min, t_max);
#pragma omp parallel for schedule(dynamic, 256)
    for (int64_t k = 0; k < (int64_t)n; k++) {
        Ray r(Vec3(rays[k].origin), Vec3(rays[k].direction), rays[k].time);
        PathCtx ctx;
        ctx.media_enabled = false;
        HitRecord best;
        bool any = false;
        if (mode == 0) {
            any = sc->world->hit(r, iv, ctx, best);
        } else {
            uint32_t best_rank = RT_NONE;
            for (const auto& leaf : sc->leaves) {
                Ray lr = r;
                for (const Transform* t : leaf.chain) {  // Transform::hit entry, outermost first
                    Vec3 lo = t->detransform(lr.orig), lt = t->detransform(lr.at(1.0));
                    lr = Ray(lo, lt - lo, lr.time);
                }
                HitRecord rec;
                if (!leaf.prim->hit(lr, iv, ctx, rec)) continue;
                uint32_t rank = sc->ranks[leaf.prim->id];
                if (!any || rec.t < best.t || (rec.t == best.t && rank < best_rank)) {
                    best = rec;
                    best_rank = rank;
                    best.inst_id = leaf.chain.empty() ? RT_NONE : leaf.chain.back()->id;
                    any = true;
                }
            }
        }
        rt_hit h;
        h.t = any ? best.t : INF;
        h.prim_id = any ? best.prim_id : RT_NONE;
        h.inst_id = any ? best.inst_id : RT_NONE;
        h.u = any ? (float)best.u : 0.0f;
        h.v = any ? (float)best.v : 0.0f;
        out[k] = h;
    }
    return 0;
}

// The pixel loop of Camera::render (camera.rs:179-197): accum receives sum*pixel_sample_scale
// per pixel (f64, W*H*3) for the requested partition / stratum range (see rt_render_opts).
int orc_render(const void* s, const rt_camera* cam, const rt_render_opts* opts, double* accum, rt_stats* stats, int threads) {
    const Scene* sc = (const Scene*)s;
    const uint32_t W = cam->image_width, H = cam->image_height, S = cam->sqrt_spp;
    uint32_t part_count = opts->part_count ? opts->part_count : 1, part_index = opts->part_index;
    uint32_t s_begin = opts->sample_begin, s_end = opts->sample_end;
    if (s_begin == 0 && s_end == 0) s_end = S * S;
    const uint32_t tiles_x = (W + 7) / 8;
    uint64_t paths = 0, segments = 0, errors = 0;
#ifdef _OPENMP
    const int team = threads > 0 ? threads : omp_get_max_threads();  // this call only: later calls keep the default
#else
    (void)threads;
#endif
#pragma omp parallel for num_threads(team) schedule(dynamic, 16) reduction(+ : paths, segments, errors)
    for (int64_t pix = 0; pix < (int64_t)W * H; pix++) {
        uint32_t i = (uint32_t)(pix % W), j = (uint32_t)(pix / W);
        uint32_t tile = (j / 8) * tiles_x + (i / 8);
        Vec3 pixel_color(0, 0, 0);
        if (tile % part_count == part_index) {
            RenderCounters cnt;
            for (uint32_t sidx = s_begin; sidx < s_end; sidx++) {
                uint32_t s_i = sidx / S, s_j = sidx % S;
                PathCtx ctx;
                ctx.seed = opts->seed, ctx.pixel = (uint32_t)pix, ctx.sample = sidx;
                Ray r = get_ray(*cam, i, j, s_i, s_j, ctx);
                bool error = false;
                Vec3 c = ray_color(*sc, *cam, r, cam->max_depth, ctx, cnt, error);
                cnt.paths++;
                if (error) {
                    cnt.errors++;  // the reference would have aborted; the sample is dropped
                    continue;
                }
                pixel_color = pixel_color + c;
            }
            paths += cnt.paths, segments += cnt.segments, errors += cnt.errors;
        }
        Vec3 scaled = pixel_color * cam->pixel_sample_scale;
        accum[pix * 3 + 0] = scaled[0], accum[pix * 3 + 1] = scaled[1], accum[pix * 3 + 2] = scaled[2];
    }
    if (stats) {
        std::memset(stats, 0, sizeof(*stats));
        stats->paths = paths, stats->segments = segments, stats->errors = errors;
    }
    return 0;
}

int orc_tonemap(const double* accum, uint64_t n_pixels, uint32_t toon_map, uint8_t* rgb) {
    for (uint64_t i = 0; i < n_pixels; i++) to_rgb(Vec3(accum + 3 * i), toon_map, rgb + 3 * i);
    return 0;
}

int orc_num_threads() {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

// ---- known-answer hooks for the vectors the reference's own unit tests hold ----------------
int orc_kat_aabb_hit(const double* a, const double* b, const double* o, const double* d, double tmin, double tmax) {
    return AABB::from_points(Vec3(a), Vec3(b)).hit(Ray(Vec3(o), Vec3(d)), Interval::make(tmin, tmax)) ? 1 : 0;
}
int orc_kat_aabb_longest_axis(const double* a, const double* b) { return AABB::from_points(Vec3(a), Vec3(b)).longest_axis(); }
void orc_kat_aabb_from_points(const double* a, const double* b, double* out6) {
    AABB x = AABB::from_points(Vec3(a), Vec3(b));
    out6[0] = x.x.min, out6[1] = x.x.max, out6[2] = x.y.min, out6[3] = x.y.max, out6[4] = x.z.min, out6[5] = x.z.max;
}
void orc_kat_aabb_union(const double* a6, const double* b6, double* out6) {
    AABB x = AABB::union_(AABB::from6(a6), AABB::from6(b6));
    out6[0] = x.x.min, out6[1] = x.x.max, out6[2] = x.y.min, out6[3] = x.y.max, out6[4] = x.z.min, out6[5] = x.z.max;
}
void orc_kat_sphere_uv(const double* p, double* uv) { Sphere::get_sphere_uv(Vec3(p), uv[0], uv[1]); }
void orc_kat_ray_at(const double* o, const double* d, double t, double* out) {
    Vec3 p = Ray(Vec3(o), Vec3(d)).at(t);
    out[0] = p[0], out[1] = p[1], out[2] = p[2];
}
void orc_kat_vec3(const double* a, const double* b, double s, double* out) {
    // out: add(3) sub(3) mul_scalar(3) div_scalar(3) dot(1) cross(3) length(1) unit(3)
    Vec3 A(a), B(b);
    Vec3 r;
    r = A + B; out[0] = r[0], out[1] = r[1], out[2] = r[2];
    r = A - B; out[3] = r[0], out[4] = r[1], out[5] = r[2];
    r = A * s; out[6] = r[0], out[7] = r[1], out[8] = r[2];
    r = A / s; out[9] = r[0], out[10] = r[1], out[11] = r[2];
    out[12] = dot(A, B);
    r = cross(A, B); out[13] = r[0], out[14] = r[1], out[15] = r[2];
    out[16] = length(A);
    unit_vector(A, r); out[17] = r[0], out[18] = r[1], out[19] = r[2];
}
void orc_kat_quat_axis_angle_rotate(const double* axis, double deg, const double* v, double* out) {
    Vec3 r = Quaternion::from_axis_angle(Vec3(axis), deg).rotate_vector(Vec3(v));
    out[0] = r[0], out[1] = r[1], out[2] = r[2];
}
void orc_kat_quat_mul(const double* a_wxyz, const double* b_wxyz, double* out) {
    Quaternion r = Quaternion{a_wxyz[0], a_wxyz[1], a_wxyz[2], a_wxyz[3]}.mul(Quaternion{b_wxyz[0], b_wxyz[1], b_wxyz[2], b_wxyz[3]});
    out[0] = r.w, out[1] = r.x, out[2] = r.y, out[3] = r.z;
}
void orc_kat_philox(const uint32_t* ctr, const uint32_t* key, uint32_t* out) {
    uint32_t c[4] = {ctr[0], ctr[1], ctr[2], ctr[3]};
    philox4x32_10(c, key[0], key[1]);
    for (int i = 0; i < 4; i++) out[i] = c[i];
}
void orc_kat_draw(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t segment, uint32_t slot, double* ab) {
    Rand2 r = philox_pair(seed, pixel, sample, segment, slot);
    ab[0] = r.a, ab[1] = r.b;
}
// ---- hooks for the hand-derived vectors of tests/test_oracle_kat.py (hit records, scatter, pdfs) ----------
// world.hit with every random draw forced to (xi[0], xi[1]).  out: t, p(3), normal(3), u, v, front_face, prim_id, inst_id
int orc_kat_world_hit(const void* s, const rt_ray* ray, double tmin, double tmax, const double* xi, double* out12) {
    const Scene& sc = *(const Scene*)s;
    PathCtx ctx;
    ctx.forced = xi;
    ctx.media_enabled = xi != nullptr;
    HitRecord rec;
    Ray r(Vec3(ray->origin), Vec3(ray->direction), ray->time);
    if (!sc.world->hit(r, Interval::make(tmin, tmax), ctx, rec)) return 0;
    out12[0] = rec.t;
    for (int k = 0; k < 3; k++) out12[1 + k] = rec.p[k], out12[4 + k] = rec.normal[k];
    out12[7] = rec.u, out12[8] = rec.v, out12[9] = rec.front_face ? 1.0 : 0.0;
    out12[10] = (double)rec.prim_id, out12[11] = (double)rec.inst_id;
    return 1;
}
// materials[mat].scatter on a hand-made hit record.  hit9: p(3) normal(3) u v front_face.  Returns the ScatterKind;
// out: attenuation(3), ray direction(3) (SCATTER_RAY only), error flag
int orc_kat_scatter(const void* s, uint32_t mat, const rt_ray* ray, const double* hit9, const double* xi, double* out7) {
    const Scene& sc = *(const Scene*)s;
    PathCtx ctx;
    ctx.forced = xi;
    HitRecord rec;
    rec.p = Vec3(hit9), rec.normal = Vec3(hit9 + 3), rec.u = hit9[6], rec.v = hit9[7], rec.front_face = hit9[8] != 0.0;
    Ray r(Vec3(ray->origin), Vec3(ray->direction), ray->time);
    ScatterRecord sr = sc.materials[mat]->scatter(r, rec, ctx, 0);
    for (int k = 0; k < 3; k++) out7[k] = sr.attenuation[k], out7[3 + k] = sr.ray.dir[k];
    out7[6] = sr.error ? 1.0 : 0.0;
    return (int)sr.kind;
}
// CosinePDF::new(albedo, normal).value(direction) and .generate() with forced draws (pdf.rs:36-64).  out: brdf(3), pdf, generated(3)
int orc_kat_cosine_pdf(const double* albedo, const double* normal, const double* direction, const double* xi, double* out7) {
    ScatterRecord sr = cosine_record(Vec3(albedo), Vec3(normal));
    if (sr.error) return 0;
    Vec3 brdf;
    double pdf;
    if (!pdf_value(sr, Vec3(direction), brdf, pdf)) return 0;
    PathCtx ctx;
    ctx.forced = xi;
    Vec3 gen;
    bool err = false;
    pdf_generate(sr, ctx, gen, err);
    for (int k = 0; k < 3; k++) out7[k] = brdf[k], out7[4 + k] = gen[k];
    out7[3] = pdf;
    return err ? 0 : 1;
}
// Disney::evaluate_disney (material/disney.rs:289-401) on local-space unit vectors (y = normal).  params15: base_color(3), roughness,
// anisotropic, sheen, sheen_tint, clearcoat, clearcoat_gloss, specular_tint, metallic, ior, flatness, spec_trans, diff_trans; out4:
// reflectance(3), forward pdf.  Returns 0 where the reference would panic.
int orc_kat_disney_evaluate(const double* params15, int thin, const double* v_out, const double* v_in, int front_face, double* out4) {
    DisneyParameters P;
    P.base_color = Vec3(params15);
    P.roughness = params15[3], P.anisotropic = params15[4], P.sheen = params15[5], P.sheen_tint = params15[6], P.clearcoat = params15[7];
    P.clearcoat_gloss = params15[8], P.specular_tint = params15[9], P.metallic = params15[10], P.ior = params15[11], P.flatness = params15[12];
    P.spec_trans = params15[13], P.diff_trans = params15[14], P.thin = thin != 0;
    Vec3 refl;
    double pdf = 0.0;
    bool error = false;
    disney::evaluate_disney(P, Vec3(v_out), Vec3(v_in), front_face != 0, refl, pdf, error);
    for (int k = 0; k < 3; k++) out4[k] = refl[k];
    out4[3] = pdf;
    return error ? 0 : 1;
}
// DisneyPDF::generate (disney.rs:542-720) in the local frame (identity basis, y = normal) with the draws forced: pick2 = the RT_SLOT_DISNEY
// pair (lobe choice, coin of the diffuse-transmission / Fresnel decision), u2 = the RT_SLOT_DIRECTION pair.  Returns 1 and the direction,
// 0 for None, -1 where the reference would panic.
int orc_kat_disney_generate(const double* params15, int thin, const double* v_out, int front_face, const double* pick2, const double* u2, double* out3) {
    ScatterRecord sr;
    sr.kind = SCATTER_DISNEY;
    DisneyParameters& P = sr.params;
    P.base_color = Vec3(params15);
    P.roughness = params15[3], P.anisotropic = params15[4], P.sheen = params15[5], P.sheen_tint = params15[6], P.clearcoat = params15[7];
    P.clearcoat_gloss = params15[8], P.specular_tint = params15[9], P.metallic = params15[10], P.ior = params15[11], P.flatness = params15[12];
    P.spec_trans = params15[13], P.diff_trans = params15[14], P.thin = thin != 0;
    sr.v_out = Vec3(v_out);
    sr.front_face = front_face != 0;
    sr.uvw.axis[0] = Vec3(1, 0, 0), sr.uvw.axis[1] = Vec3(0, 1, 0), sr.uvw.axis[2] = Vec3(0, 0, 1);
    PathCtx ctx;
    ctx.forced = pick2;
    ctx.forced_direction = u2;
    Vec3 out;
    bool error = false;
    const bool some = disney::generate(sr, ctx, out, error);
    if (error) return -1;
    if (!some) return 0;
    for (int k = 0; k < 3; k++) out3[k] = out[k];
    return 1;
}
// lights.pdf_value(origin, direction) and lights.random(origin) of the scene's lights tree (hits.rs:52-75 and the shapes below it)
double orc_kat_lights_pdf_value(const void* s, const double* origin, const double* direction) {
    const Scene& sc = *(const Scene*)s;
    return sc.lights ? sc.lights->pdf_value(Vec3(origin), Vec3(direction)) : std::nan("");
}
int orc_kat_lights_random(const void* s, const double* origin, uint32_t leaf, double r1, double r2, double* out3) {
    const Scene& sc = *(const Scene*)s;
    if (!sc.lights) return 0;
    LightSample ls;
    ls.leaf = leaf, ls.r1 = r1, ls.r2 = r2;
    Vec3 d = sc.lights->random(Vec3(origin), ls);
    for (int k = 0; k < 3; k++) out3[k] = d[k];
    return ls.error ? 0 : 1;
}
static void write_segment(const Segment& g, bool goes_on, double hit_kind, double object, double t, double* o) {
    o[0] = hit_kind, o[1] = object, o[2] = t;
    for (int c = 0; c < 3; c++) {
        o[3 + c] = g.background[c], o[6 + c] = g.emission[c], o[10 + c] = g.attenuation[c], o[13 + c] = g.albedo_x_pscatter[c];
        o[17 + c] = g.next.orig[c], o[20 + c] = g.next.dir[c];
    }
    o[9] = (double)g.kind;
    o[16] = g.pdf_val;
    o[23] = g.next.time;
    o[24] = goes_on ? 1.0 : 0.0, o[25] = g.generated ? 1.0 : 0.0, o[26] = g.error ? 1.0 : 0.0, o[27] = g.fuzzed ? 1.0 : 0.0;
}
// One level of ray_color per row (ray_step), with the draws addressed by (seeds[i]; ids[3i] pixel, ids[3i+1] sample, ids[3i+2]
// segment) and media enabled.  out28 per row: hit (0 miss, 1 surface, 2 medium), object id (the leaf shape or the ConstantMedium),
// t, background(3), emission(3), scatter kind, attenuation(3), albedo_x_pscatter(3), pdf_val, next ray o(3) d(3) time, goes on,
// generated, error, fuzzed (a SCATTER_RAY direction that went through sin / cos).
int orc_kat_shade_step(const void* s, const rt_camera* cam, const rt_ray* rays, const uint64_t* seeds, const uint32_t* ids, uint64_t n, double* out28) {
    const Scene& sc = *(const Scene*)s;
#pragma omp parallel for schedule(dynamic, 64)
    for (int64_t k = 0; k < (int64_t)n; k++) {
        PathCtx ctx;
        ctx.seed = seeds[k], ctx.pixel = ids[3 * k], ctx.sample = ids[3 * k + 1], ctx.segment = ids[3 * k + 2];
        Ray r(Vec3(rays[k].origin), Vec3(rays[k].direction), rays[k].time);
        Segment g;
        const bool goes_on = ray_step(sc, *cam, r, ctx, g);
        const bool medium = g.hit && sc.by_object[g.rec.prim_id] && dynamic_cast<const ConstantMedium*>(sc.by_object[g.rec.prim_id]);
        write_segment(g, goes_on, g.hit ? (medium ? 2.0 : 1.0) : 0.0, g.hit ? (double)g.rec.prim_id : (double)RT_NONE, g.hit ? g.rec.t : INF,
                      out28 + 28 * k);
    }
    return 0;
}
// shade_record on given rt_hit_records, the step rt_shade runs (include/rt2025.h): p, normal, u, v and the material are used as
// given, front_face is != 0; t, prim_id and reserved are not read, nor anything of a miss but its kind.  A record of kind >
// RT_HIT_MEDIUM, or a non-miss record with material >= n_materials, is an error and shades nothing; inst_id != RT_NONE with a
// non-finite normal is the Transform panic.  out28 as orc_kat_shade_step, with hit = the record's kind, object RT_NONE and t NaN.
int orc_kat_shade_record(const void* s, const rt_camera* cam, const rt_ray* rays, const rt_hit_record* records, const uint64_t* seeds,
                         const uint32_t* ids, uint64_t n, double* out28) {
    const Scene& sc = *(const Scene*)s;
#pragma omp parallel for schedule(dynamic, 64)
    for (int64_t k = 0; k < (int64_t)n; k++) {
        PathCtx ctx;
        ctx.seed = seeds[k], ctx.pixel = ids[3 * k], ctx.sample = ids[3 * k + 1], ctx.segment = ids[3 * k + 2];
        Ray r(Vec3(rays[k].origin), Vec3(rays[k].direction), rays[k].time);
        const rt_hit_record& h = records[k];
        Segment g;
        bool goes_on = false;
        if (h.kind > RT_HIT_MEDIUM || (h.kind != RT_HIT_MISS && h.material >= sc.materials.size())) {
            g.error = true;
        } else if (h.kind == RT_HIT_MISS) {
            goes_on = shade_record(sc, *cam, r, nullptr, ctx, g);
        } else {
            HitRecord rec;
            rec.p = Vec3(h.p), rec.normal = Vec3(h.normal), rec.u = h.u, rec.v = h.v, rec.front_face = h.front_face != 0;
            rec.mat = sc.materials[h.material].get();
            rec.inst_id = h.inst_id;
            rec.normal_panic = h.inst_id != RT_NONE && !(std::isfinite(h.normal[0]) && std::isfinite(h.normal[1]) && std::isfinite(h.normal[2]));
            goes_on = shade_record(sc, *cam, r, &rec, ctx, g);
        }
        write_segment(g, goes_on, (double)h.kind, (double)RT_NONE, std::nan(""), out28 + 28 * k);
    }
    return 0;
}
// texture / environment lookups on a built scene (used to cross-check the device textures)
void orc_texture_value(const void* s, uint32_t tex, double u, double v, const double* p, double* out) {
    Vec3 c = ((const Scene*)s)->textures[tex]->value(u, v, Vec3(p));
    out[0] = c[0], out[1] = c[1], out[2] = c[2];
}
void orc_camera_ray(const rt_camera* cam, uint64_t seed, uint32_t i, uint32_t j, uint32_t sidx, rt_ray* out) {
    PathCtx ctx;
    ctx.seed = seed, ctx.pixel = j * cam->image_width + i, ctx.sample = sidx;
    Ray r = get_ray(*cam, i, j, sidx / cam->sqrt_spp, sidx % cam->sqrt_spp, ctx);
    for (int k = 0; k < 3; k++) out->origin[k] = r.orig[k], out->direction[k] = r.dir[k];
    out->time = r.time;
}

}  // extern "C"
