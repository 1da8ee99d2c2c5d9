/*
 * rt2025.h — C ABI of the B200-native path-tracing core for caidj0/Raytracer-2025.
 *
 * The reference crate has no FFI; its only boundary is the public Rust API.  The cut made
 * here is inside `Camera::render` (reference src/camera.rs:161), between `self.initilize()`
 * (:162) and the pixel loop (:179-197): the Rust side (or the C++ host mirror in
 * raytracer-2025_b200/host/) keeps building the trait-object scene, *flattens* it into the
 * plain-old-data object graph below and hands it to this library, which owns everything
 * from camera-ray generation to the accumulated radiance image.
 *
 * Conventions
 *   - every entry point returns 0 (RT_OK) on success and a negative rt_status otherwise;
 *     rt_last_error() returns a thread-local message for the last failure;
 *   - no C++ exception crosses this boundary;
 *   - all pointers are borrowed for the duration of the call only; rt_scene_create copies;
 *   - handles are opaque; distinct handles may be used from distinct host threads;
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     RT_ERR_NO_DEVICE.
 *
 * All geometry is IEEE-754 binary64, like the reference (src/utils/vec3.rs:12-15).
 */
#ifndef RT2025_H
#define RT2025_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_ABI_VERSION 1u
#define RT_NONE 0xFFFFFFFFu

typedef enum rt_status {
    RT_OK = 0,
    RT_ERR_INVALID = -1,      /* malformed description (bad index, bad kind, null pointer) */
    RT_ERR_UNSUPPORTED = -2,  /* a construct the flattener cannot express on the device     */
    RT_ERR_NO_DEVICE = -3,    /* no CUDA device / wrong architecture: there is no CPU path  */
    RT_ERR_CUDA = -4,         /* a CUDA runtime call failed                                 */
    RT_ERR_OOM = -5,
    RT_ERR_VERSION = -6
} rt_status;

/* ------------------------------------------------------------------------------------ */
/* Object graph: one rt_object per `dyn Hittable` in the reference scene.                */
/* ------------------------------------------------------------------------------------ */

typedef enum rt_obj_kind {
    RT_OBJ_SPHERE = 1,    /* shapes/sphere.rs:17-51   payload: spheres[data]              */
    RT_OBJ_QUAD = 2,      /* shapes/quad.rs:18-49     payload: planars[data]              */
    RT_OBJ_TRIANGLE = 3,  /* shapes/triangle.rs:16-46 payload: planars[data]              */
    RT_OBJ_LIST = 4,      /* hits.rs:10-31  `Hittables`; children in insertion order       */
    RT_OBJ_BVH = 5,       /* bvh.rs:5-46    children in the order given to BVH::from_vec   */
    RT_OBJ_TRANSFORM = 6, /* shapes.rs:23-47        payload: transforms[data], one child   */
    RT_OBJ_MEDIUM = 7     /* volume.rs:16-35        payload: media[data], one child        */
} rt_obj_kind;

typedef struct rt_object {
    uint32_t kind;         /* rt_obj_kind */
    uint32_t material;     /* leaf shapes: index into materials[]; MEDIUM: its Isotropic    */
    uint32_t first_child;  /* offset into children[] (LIST/BVH/TRANSFORM/MEDIUM)            */
    uint32_t child_count;  /* 1 for TRANSFORM and MEDIUM                                   */
    uint32_t data;         /* index into the per-kind payload array, RT_NONE if none        */
    uint32_t reserved;
    double bbox[6];        /* `bounding_box()` exactly as the reference computed it:        */
                           /* xmin,xmax,ymin,ymax,zmin,zmax (aabb.rs:9-51, incl. padding)   */
} rt_object;

/* Sphere { center: Ray, radius } — sphere.rs:17-51.  center(time) = center + time*center_vec */
typedef struct rt_sphere {
    double center[3];
    double center_vec[3];
    double radius;
    double reserved;
} rt_sphere;

/* Quad / Triangle share the plane + w-basis representation — quad.rs:18-49, triangle.rs:16-46.
 * The derived fields are copied from the host object so that every consumer intersects with
 * the very same numbers the reference would use. */
typedef struct rt_planar {
    double anchor[3];
    double u[3];
    double v[3];
    double normal[3]; /* unit(cross(u,v)) */
    double parm_d;    /* normal . anchor  */
    double w[3];      /* n / (n.n)        */
    double area;      /* |n| (quad) or |n|/2 (triangle) */
    double reserved;
} rt_planar;

/* Transform { offset, quaternion, scale } — shapes.rs:23-47, utils/quaternion.rs:6-11 */
typedef struct rt_transform {
    double offset[3];
    double quat[4]; /* w, x, y, z */
    double scale[3];
} rt_transform;

/* ConstantMedium — volume.rs:16-35; its phase function is materials[object.material] */
typedef struct rt_medium {
    double neg_inv_density;
    double reserved;
} rt_medium;

/* ------------------------------------------------------------------------------------ */
/* Materials (material.rs) and textures (texture.rs)                                     */
/* ------------------------------------------------------------------------------------ */

typedef enum rt_mat_kind {
    RT_MAT_EMPTY = 0,         /* material.rs:36-47  0.75 grey Lambertian                    */
    RT_MAT_LAMBERTIAN = 1,    /* :49-66   tex                                              */
    RT_MAT_METAL = 2,         /* :68-95   color, param = fuzz (already clamped to [0,1])    */
    RT_MAT_DIELECTRIC = 3,    /* :97-144  tex = attenuation, param = refraction index       */
    RT_MAT_DIFFUSE_LIGHT = 4, /* :146-186 tex, inner = wrapped material or RT_NONE          */
    RT_MAT_ISOTROPIC = 5,     /* :188-207 tex                                              */
    RT_MAT_TRANSPARENT = 6,   /* :209-218                                                  */
    RT_MAT_MIX = 7,           /* :220-268 inner, inner2, param = ratio or tex = alpha image */
    RT_MAT_PORTAL = 8,        /* material/portal.rs:9-31 color, v[0..3)=offset v[3..7)=quat */
    RT_MAT_DISNEY = 9,        /* material/disney.rs:17-116: color = base_color (or tex = base-colour   */
                              /* texture, as the OBJ loader builds it, shapes/obj.rs:271-293), v[] =  */
                              /* the DisneyParameters scalars in RT_DISNEY_* order                     */
    RT_MAT_REMAPPED = 10      /* shapes/obj.rs:20-81 RemappedMaterial: inner = wrapped material,       */
                              /* inner2 = index into remaps[]                                          */
} rt_mat_kind;

/* order of the DisneyParameters scalars in rt_material.v (disney.rs:18-35) */
enum {
    RT_DISNEY_ROUGHNESS = 0, RT_DISNEY_ANISOTROPIC, RT_DISNEY_SHEEN, RT_DISNEY_SHEEN_TINT, RT_DISNEY_CLEARCOAT,
    RT_DISNEY_CLEARCOAT_GLOSS, RT_DISNEY_SPECULAR_TINT, RT_DISNEY_METALLIC, RT_DISNEY_IOR, RT_DISNEY_FLATNESS,
    RT_DISNEY_SPEC_TRANS, RT_DISNEY_DIFF_TRANS, RT_DISNEY_THIN /* 0.0 or 1.0 */, RT_DISNEY_COUNT
};

typedef struct rt_material {
    uint32_t kind;
    uint32_t tex;
    uint32_t inner;
    uint32_t inner2;
    double color[3];
    double param;
    double v[16];
} rt_material;

/* RemappedMaterial { tex_ori, tex_u, tex_v, u_vec, v_vec, normal[3], normal_tex } — obj.rs:20-29 */
typedef struct rt_remap {
    double tex_ori[3], tex_u[3], tex_v[3];
    double u_vec[3], v_vec[3];   /* valid only when has_uv_vecs (both Options are Some)                */
    double normal[3][3];         /* the three vertex normals                                          */
    uint32_t has_uv_vecs;
    uint32_t normal_tex;         /* texture index of the raw normal map, RT_NONE for None             */
} rt_remap;

typedef enum rt_tex_kind {
    RT_TEX_SOLID = 0,    /* texture.rs:9-36    color                                       */
    RT_TEX_CHECKER = 1,  /* :38-73             scale = inv_scale, a = even, b = odd         */
    RT_TEX_IMAGE = 2,    /* :81-174            a = image index or RT_NONE (missing file)    */
    RT_TEX_NOISE = 3,    /* :176-196           a = perlin table index, scale                */
    RT_TEX_GRADIENT_Y = 4 /* not in the crate: (1-s)*color + s*color2, s = 0.5*(p.y+1).     */
                          /* It is the book-1 sky, evaluated on the unit ray direction that */
                          /* Environment::value passes as `p` (environment.rs:14-24).       */
} rt_tex_kind;

typedef struct rt_texture {
    uint32_t kind;
    uint32_t a;
    uint32_t b;
    uint32_t reserved;
    double color[3];
    double color2[3];
    double scale;
    double reserved2;
} rt_texture;

#define RT_IMG_LINEAR 1u /* texels already linear (raw / HDR / EXR): utils/image.rs:71-82 */
#define RT_IMG_INTERP 2u /* bilinear (new_raw_image) instead of nearest: texture.rs:87-100 */

typedef struct rt_image {
    uint32_t width, height;
    uint32_t flags;
    uint32_t reserved;
    uint64_t texel_offset; /* first float of this image in texels[] (RGBA32F, row-major)    */
} rt_image;

/* Perlin tables — utils/perlin.rs:9-14 */
typedef struct rt_perlin {
    double randvec[256][3];
    uint32_t perm_x[256], perm_y[256], perm_z[256];
} rt_perlin;

typedef struct rt_scene_desc {
    uint32_t version;      /* RT_ABI_VERSION */
    uint32_t struct_size;  /* sizeof(rt_scene_desc) */
    uint32_t world_root;   /* object index of `world` passed to Camera::render              */
    uint32_t lights_root;  /* object index of `lights`, RT_NONE for `None`                  */

    uint32_t n_objects, n_children, n_spheres, n_planars;
    uint32_t n_transforms, n_media, n_materials, n_textures;
    uint32_t n_images, n_perlins;
    uint64_t n_texels;     /* number of floats in texels[] */
    uint32_t n_remaps, reserved0;

    const rt_object* objects;
    const uint32_t* children;
    const rt_sphere* spheres;
    const rt_planar* planars;
    const rt_transform* transforms;
    const rt_medium* media;
    const rt_material* materials;
    const rt_texture* textures;
    const rt_image* images;
    const float* texels;
    const rt_perlin* perlins;
    const rt_remap* remaps;
} rt_scene_desc;

/* ------------------------------------------------------------------------------------ */
/* Camera block: the state of `Camera` *after* initilize() — camera.rs:46-75,204-245      */
/* ------------------------------------------------------------------------------------ */

typedef struct rt_camera {
    uint32_t image_width, image_height;
    uint32_t sqrt_spp;   /* floor(sqrt(samples_per_pixel)) — camera.rs:212 */
    uint32_t max_depth;
    uint32_t background_tex;  /* texture index of `background.texture` */
    uint32_t toon_map;        /* 0 = ToonMap::None, 1 = ToonMap::ACES (utils/color.rs:8-11) */
    double recip_sqrt_spp;
    double pixel_sample_scale;
    double center[3];
    double pixel00_loc[3];
    double pixel_delta_u[3];
    double pixel_delta_v[3];
    double defocus_angle_in_degrees;
    double defocus_disk_u[3];
    double defocus_disk_v[3];
} rt_camera;

/* ------------------------------------------------------------------------------------ */
/* Calls                                                                                  */
/* ------------------------------------------------------------------------------------ */

typedef struct rt_scene rt_scene;

#define RT_BUILD_NO_REF_RANKS 1u /* skip the median-split walk that reproduces the reference's
                                    tie order (bvh.rs:78-84, hits.rs:42); ranks = object id  */
#define RT_BUILD_DEVICE_LBVH 2u  /* build the world BVH on the GPU (Morton-code LBVH, one primitive per leaf) instead
                                    of the host binned-SAH builder: a much faster rt_scene_create for very large
                                    scenes, a tree that traverses slower; ids and t do not depend on the tree */

typedef struct rt_build_opts {
    uint32_t struct_size;
    uint32_t flags;
    int32_t device;       /* CUDA ordinal; -1 = current device */
    uint32_t reserved;
} rt_build_opts;

/* Takes the place of everything Camera::render receives by reference - `world: &dyn Hittable` and
 * `lights: Option<&dyn Hittable>` (camera.rs:161) - and of the work BVH::from_vec does when client code builds the
 * scene (bvh.rs:16-46): validates the description, computes the reference's tie order, keeps primitives below a
 * Transform in their local space (shapes.rs:88-111), builds the traversal tree(s) and uploads everything to the
 * device.  The description is copied; the caller may free it on return. */
int rt_scene_create(const rt_scene_desc* desc, const rt_build_opts* opts, rt_scene** out);
/* Drop of the scene (the reference's Box<dyn Hittable> going out of scope). */
int rt_scene_destroy(rt_scene* scene);

/* Any time is valid.  A moving sphere is placed at center + time*center_vec whatever the time, as Sphere::hit does, but
 * its traversal box bounds it over times [0, 1] only (sphere.rs:35-51): in a scene with a moving sphere a ray whose time
 * lies outside [0, 1] (or is NaN) culls no box and tests every primitive.  Its answer is still exact, at brute-force cost;
 * Camera::get_ray draws times in [0, 1). */
typedef struct rt_ray {
    double origin[3];
    double direction[3];
    double time;
} rt_ray;

typedef struct rt_hit {
    double t;          /* ray parameter of the closest surface hit */
    uint32_t prim_id;  /* object index of the leaf shape, RT_NONE = miss */
    uint32_t inst_id;  /* object index of the innermost enclosing Transform, RT_NONE if none */
    float u, v;        /* surface coordinates as HitRecord carries them (hit.rs:17-18) */
} rt_hit;

typedef struct rt_stats {
    uint64_t paths;        /* camera samples traced                                         */
    uint64_t segments;     /* world.hit calls (camera.rs:286)                               */
    uint64_t node_visits;  /* BVH nodes fetched (only when RT_OPT_COUNT is set)              */
    uint64_t prim_tests;   /* primitive tests   (only when RT_OPT_COUNT is set)              */
    uint64_t errors;       /* samples zeroed where the reference would panic (camera.rs:309,323) */
    uint64_t kernel_launches;
    double ms_total;       /* device time of the call, CUDA events on its stream             */
    double ms_raygen, ms_extend, ms_shade, ms_other; /* filled when RT_OPT_STAGE_TIMES is set */
    uint64_t iterations;   /* wavefront iterations                                          */
    uint64_t reserved[4];  /* reserved[0]: of `segments`, those evaluated inside the random-walk kernel of an optically
                              thick ConstantMedium (they never passed through extend);
                              reserved[1]: of reserved[0], those evaluated by its lean variant (scenes whose walk needs
                              no Transform, texture lookup or light-tree code);
                              reserved[2]: hits shaded by the lean variant of a shade-class kernel (diffuse, textured,
                              isotropic or emissive hits of scenes whose class needs no Transform, texture lookup or
                              light-tree code)                                                      */
} rt_stats;

/* Closest surface hit for a batch of rays over `world` (media excluded: they are stochastic,
 * volume.rs:58).  Interval semantics are Interval::contains (utils/interval.rs:65-67).
 * The answer is that of a test of every primitive (the oracle's brute-force mode): the box
 * test never culls a hit, also where the reference's AABB::hit inside a BVH would (rays that
 * graze a box face, edge or corner).  This holds for every query below.
 * A batch holds at most 2^32 - 16 rays: a larger n is RT_ERR_INVALID for every query below and
 * rt_shade, refused before anything is allocated or copied.
 * Host-pointer version copies in and out; the _device version takes device pointers and
 * enqueues on `stream` (a cudaStream_t passed as void*; NULL = default stream). */
#define RT_OPT_COUNT 1u
#define RT_OPT_STAGE_TIMES 2u
int rt_closest_hit(const rt_scene* scene, const rt_ray* rays, uint64_t n, double t_min,
                   double t_max, uint32_t flags, rt_hit* out, rt_stats* stats);
int rt_closest_hit_device(const rt_scene* scene, const rt_ray* d_rays, uint64_t n, double t_min,
                          double t_max, uint32_t flags, rt_hit* d_out, void* stream,
                          rt_stats* stats);

/* Occlusion (any-hit) query for a batch of rays over `world`.  With
 * t_max_i = t_max_per_ray ? t_max_per_ray[i] : t_max,
 *     out[i] = 1 iff some surface primitive has a hit t with Interval::contains(t_min, t_max_i, t)
 *              (inclusive at both ends, utils/interval.rs:65-67), else 0.
 * This is geometric visibility: every surface occludes whatever its material (Dielectric,
 * Transparent, Portal and emitters alike); media are excluded as in rt_closest_hit and no
 * transmittance is computed (rt_transmittance below does).  An empty interval (t_max_i < t_min, or a NaN bound) gives 0.
 * With the same primitive arithmetic as rt_closest_hit, bit for bit:
 *     out[i] == (closest_hit(ray, t_min, +inf).prim_id != RT_NONE && .t <= t_max_i)
 * A ray's traversal ends at the first hit found, so it visits at most the nodes and primitives
 * closest hit would.  `stats` gets segments = n, ms_total and kernel_launches, and node_visits /
 * prim_tests with RT_OPT_COUNT.  Host-pointer version copies in and out; the _device version
 * takes device pointers (t_max_per_ray may be NULL) and enqueues on `stream`. */
int rt_occluded(const rt_scene* scene, const rt_ray* rays, const double* t_max_per_ray /* n values or NULL */,
                uint64_t n, double t_min, double t_max, uint32_t flags, uint8_t* out, rt_stats* stats);
int rt_occluded_device(const rt_scene* scene, const rt_ray* d_rays, const double* d_t_max_per_ray,
                       uint64_t n, double t_min, double t_max, uint32_t flags, uint8_t* d_out,
                       void* stream, rt_stats* stats);

/* Transmittance (visibility through media) for a batch of rays over `world`: out[i] (binary64) is
 * the probability that world.hit(ray, [t_min, t_max_i]) returns None when every ConstantMedium
 * draws its own uniform number, with t_max_i as in rt_occluded:
 *   - an empty interval (t_max_i < t_min, or a NaN bound) gives 1.0 (the ray is not traced);
 *   - where rt_occluded with the same arguments gives 1 the result is 0.0 exactly (every surface
 *     blocks whatever its material);
 *   - otherwise the product, in ascending medium order, of exp(L_m / neg_inv_density_m) over all
 *     media, where L_m is the distance_inside_boundary of ConstantMedium::hit (volume.rs:42-58) on
 *     [t_min, t_max_i]: t1 = boundary.hit(r, UNIVERSE), t2 = boundary.hit(r, [t1 + 1e-4, inf))
 *     (factor 1 if either misses), t1 clamped up to t_min and t2 down to t_max_i (factor 1 if
 *     t1 >= t2), t1 = max(t1, 0), L = (t2 - t1) * |d| with d the direction in the medium's space.
 * Density 0 gives a factor 1, an infinite density a factor 0 wherever L > 0; neither is special-
 * cased.  T == 0 with rt_occluded == 0 happens only by underflow or through an infinite density.
 * Two launches: the occlusion pass of rt_occluded into a stream-ordered scratch buffer, then one
 * media pass.  `stats` gets segments = n, kernel_launches = 2 and ms_total over both, and with
 * RT_OPT_COUNT node_visits / prim_tests summed over both passes (a sphere boundary counts 2
 * primitive tests).  Host-pointer version copies in and out; the _device version takes device
 * pointers (t_max_per_ray may be NULL) and enqueues on `stream`. */
int rt_transmittance(const rt_scene* scene, const rt_ray* rays, const double* t_max_per_ray /* n values or NULL */,
                     uint64_t n, double t_min, double t_max, uint32_t flags, double* out, rt_stats* stats);
int rt_transmittance_device(const rt_scene* scene, const rt_ray* d_rays, const double* d_t_max_per_ray,
                            uint64_t n, double t_min, double t_max, uint32_t flags, double* d_out,
                            void* stream, rt_stats* stats);

/* World hit: the HitRecord world.hit(ray, Interval(t_min, t_max_i)) returns (camera.rs:286, hit.rs:9-60),
 * media included, for a batch of rays over `world`, with t_max_i as in rt_occluded.
 *   - Draws: the ConstantMedium of media[m] draws philox(seed; pixel = i, sample = 0, segment,
 *     RT_MEDIUM_SLOT(m)), component a for even m and b for odd m, as the renderer does.  The same
 *     (seed, segment) reproduces a batch bit for bit; a client path loop passes its bounce number as
 *     `segment`.
 *   - Interval: surfaces use Interval::contains (inclusive at both ends).  A medium runs
 *     ConstantMedium::hit (volume.rs:37-73) on [t_min, t_max_i]: t1 = boundary.hit(r, UNIVERSE),
 *     t2 = boundary.hit(r, [t1 + 1e-4, inf)), t1 clamped up to t_min and t2 down to t_max_i (no hit
 *     if t1 >= t2), t1 = max(t1, 0), then t = t1 + hit_distance / |d| with d the direction in the
 *     medium's space, when hit_distance = neg_inv_density * ln(xi) <= (t2 - t1) * |d|.
 *   - Winner: the smallest t; an exact tie goes to the lower tie rank (rt_scene_get_ranks).
 *   - Medium record: p = r.at(t) and normal (1, 0, 0) flipped by front_face, in the medium's space,
 *     then taken through its Transform chain like a surface's; u = v = 0.
 *   - An empty interval (t_max_i < t_min, or a NaN bound) gives a miss record; it is not traced and
 *     takes no draws.  Miss record: t = +inf, p and normal zero, ids and material RT_NONE,
 *     kind RT_HIT_MISS.
 * Two launches: a closest-hit surface pass into a stream-ordered scratch buffer (16 bytes per ray),
 * then the record pass.  `stats` gets segments = n, kernel_launches = 2 and ms_total over both,
 * and with RT_OPT_COUNT node_visits / prim_tests summed over both passes.  Host-pointer version
 * copies in and out; the _device version takes device pointers (t_max_per_ray may be NULL) and
 * enqueues on `stream`. */
#define RT_HIT_MISS 0u
#define RT_HIT_SURFACE 1u
#define RT_HIT_MEDIUM 2u

typedef struct rt_hit_record { /* HitRecord, hit.rs:9-20, in world space */
    double t;
    double p[3];
    double normal[3];     /* faces the ray (set_face_normal, hit.rs:33-36), after the Transform chain */
    double u, v;          /* binary64; 0, 0 for a medium */
    uint32_t kind;        /* RT_HIT_* */
    uint32_t front_face;  /* 0 / 1 */
    uint32_t prim_id;     /* object index of the leaf shape, or of the RT_OBJ_MEDIUM object; RT_NONE on a miss */
    uint32_t inst_id;     /* innermost enclosing Transform's object index, RT_NONE if none */
    uint32_t material;    /* materials[] index: the shape's material (a RemappedMaterial stays as it is, the
                             remap belongs to scatter) or the medium's phase function; RT_NONE on a miss */
    uint32_t reserved;
} rt_hit_record;          /* 96 bytes */

int rt_world_hit(const rt_scene* scene, const rt_ray* rays, const double* t_max_per_ray /* n values or NULL */,
                 uint64_t n, double t_min, double t_max, uint64_t seed, uint32_t segment, uint32_t flags,
                 rt_hit_record* out, rt_stats* stats);
int rt_world_hit_device(const rt_scene* scene, const rt_ray* d_rays, const double* d_t_max_per_ray,
                        uint64_t n, double t_min, double t_max, uint64_t seed, uint32_t segment,
                        uint32_t flags, rt_hit_record* d_out, void* stream, rt_stats* stats);

/* Shade: the step of ray_color after world.hit (camera.rs:288-321) for a batch of records as rt_world_hit
 * writes them, so that a client can run the path loop itself (INTEGRATION.md):
 *     rays = rt_camera_rays(sample 0); beta = 1; radiance = 0; state = RT_PATH_ALIVE
 *     for segment in 0 .. max_depth: rt_world_hit(rays, t_max_i = state & RT_PATH_ALIVE ? t_max : NaN,
 *                                                  seed, segment); rt_shade(..., seed, segment)
 * reproduces rt_render at one sample per pixel (sqrt_spp = 1).  The path state of row i is updated in place:
 *   - Active rows: row i is active iff state[i] & RT_PATH_ALIVE.  Of an inactive row only the state byte is
 *     read, and nothing is written.
 *   - An active row leaves with state = RT_PATH_ALIVE iff the path goes on, with rays[i] / beta[i] its next
 *     ray and throughput (otherwise they are left as they were), after the render's cuts: segment + 1 >=
 *     max_depth, and a zero throughput.  RT_PATH_ERROR is set iff the render counts an error in rt_stats
 *     for this segment: a case where the reference panics, or a NaN contribution (camera.rs:323); such a
 *     path may still go on.  The other bits are cleared.
 *   - radiance[i] (3 binary64) gets beta * emitted, or beta * the background of camera->background_tex
 *     looked up on the ray direction for a miss; NaN contributions are dropped.
 *   - Draws: philox(seed; pixel = i, sample = 0, segment, slot) in the renderer's slots (MATERIAL,
 *     MIXTURE, DIRECTION, MIX + 256 * level, DISNEY), the addressing rt_world_hit uses for its media.
 *   - The record is the HitRecord: p, normal, u, v, front_face and material are used as given, a
 *     RemappedMaterial is applied here; t, prim_id and reserved are not read, nor any field of a miss
 *     but its kind.  front_face: any nonzero value means front.  inst_id is only a flag, never an
 *     index: a record with inst_id != RT_NONE and a non-finite normal is a Transform normal that
 *     could not be normalised (the reference panics).  A record with kind > RT_HIT_MEDIUM, or a
 *     non-miss record with material >= n_materials, ends its path with RT_PATH_ERROR.
 *   - camera: only max_depth and background_tex are read.  RT_ERR_INVALID for a null pointer,
 *     background_tex >= n_textures or segment >= max_depth (the reference never runs that segment).
 * `stats` gets segments = n, errors = the rows that leave with RT_PATH_ERROR, kernel_launches and
 * ms_total (the launch alone).  `flags` must be 0 (RT_ERR_INVALID otherwise); every refusal comes
 * before anything is copied.  Host-pointer version copies in and out (rays, beta, radiance and state
 * are updated in place); the _device version takes device pointers and enqueues on `stream`. */
#define RT_PATH_ALIVE 1u /* state bit 0: the path goes on with rays[i] / beta[i] */
#define RT_PATH_ERROR 2u /* state bit 1: this segment hit a case where the reference panics */

int rt_shade(const rt_scene* scene, const rt_camera* camera, const rt_hit_record* records, uint64_t n, uint64_t seed,
             uint32_t segment, uint32_t flags, rt_ray* rays, double* beta, double* radiance, uint8_t* state,
             rt_stats* stats);
int rt_shade_device(const rt_scene* scene, const rt_camera* camera /* host pointer */, const rt_hit_record* d_records,
                    uint64_t n, uint64_t seed, uint32_t segment, uint32_t flags, rt_ray* d_rays, double* d_beta,
                    double* d_radiance, uint8_t* d_state, void* stream, rt_stats* stats);

/* Camera rays: Camera::get_ray (camera.rs:247-273) of stratum `sample` (0 <= sample < sqrt_spp^2:
 * s_i = sample / sqrt_spp, s_j = sample % sqrt_spp) through every pixel, the ray rt_render traces first:
 * out[j * image_width + i] for pixel (i, j), image_width * image_height rays, with the draws
 * philox(seed; pixel, sample, 0, RT_SLOT_CAM_*).  Runs on the current device (no scene), like
 * rt_tonemap_device.  RT_ERR_INVALID for a null pointer, a bad sample or more than 2^32 - 16 pixels.
 * The host-pointer version returns when `out` is filled; the _device version enqueues on `stream`. */
int rt_camera_rays(const rt_camera* camera, uint64_t seed, uint32_t sample, rt_ray* out);
int rt_camera_rays_device(const rt_camera* camera, uint64_t seed, uint32_t sample, rt_ray* d_out, void* stream);

/* Path ids: the three entries above with the address of each row's draws given per row, so that a client
 * loop runs any number of samples per pixel and may compact, permute and refill its batch.  The id is
 * the render's own path id (rt2025_rng.h): a row's draws are philox(seed; pixel, sample, segment, slot).
 * Ids are addresses and are not range-checked: a pixel beyond the image or a stratum >= sqrt_spp^2 gets
 * what the same arithmetic gives.
 *   - rt_camera_rays_ids: out[i] = Camera::get_ray of pixel (ids[i].pixel % image_width,
 *     ids[i].pixel / image_width) and stratum ids[i].sample (s_i = sample / sqrt_spp, s_j = sample %
 *     sqrt_spp), with the draws philox(seed; pixel, sample, 0, RT_SLOT_CAM_*); segment is not read.
 *     Runs on the current device (no scene), like rt_camera_rays.  RT_ERR_INVALID for a null pointer,
 *     n > 2^32 - 16, image_width == 0 or sqrt_spp == 0.
 *   - rt_world_hit_ids: rt_world_hit, with the free-flight draw of media[m] for row i at
 *     philox(seed; ids[i].pixel, ids[i].sample, ids[i].segment, RT_MEDIUM_SLOT(m)).  Only rows that take
 *     draws (a scene with media and a non-empty interval) read their id.  Everything else, refusals and
 *     stats included, is rt_world_hit's.
 *   - rt_shade_ids: rt_shade, with the draws of row i addressed by ids[i] and ids[i].segment in place of
 *     `segment`, in the draws and in the depth cut.  radiance + 3 i is still indexed by row: a client
 *     that holds several samples of one pixel sums them itself.  A row that leaves with RT_PATH_ALIVE
 *     gets ids[i].segment += 1; no other field of ids is ever written, and an inactive row reads and
 *     writes nothing but its state byte.  An active row with ids[i].segment >= max_depth (a segment the
 *     reference never runs) ends with RT_PATH_ERROR, counts in stats.errors, and nothing else of it is
 *     read or written.  The refusals are rt_shade's but the segment test.
 * Each pins its twin bit for bit:
 *   - rt_world_hit(..., segment = s) equals rt_world_hit_ids with ids[i] = (i, 0, s);
 *   - rt_shade(..., segment = s) equals rt_shade_ids with the same ids, apart from the segment update;
 *   - rt_camera_rays(sample = s) equals rt_camera_rays_ids with ids[i] = (i, s, any).
 * So the loop of rt_shade, with ids (pixel, stratum, 0) for every path and the rows summed into a
 * framebuffer by pixel, reproduces rt_render at any sqrt_spp (INTEGRATION.md §5).  Host-pointer versions
 * copy in and out (rt_shade_ids copies ids back); the _device versions take device pointers (the camera
 * stays a host pointer) and enqueue on `stream`. */
typedef struct rt_path_id {
    uint32_t pixel;     /* the render's pixel index j * image_width + i */
    uint32_t sample;    /* the stratum s_i * sqrt_spp + s_j */
    uint32_t segment;   /* the number of world.hit calls made on the path before this one */
    uint32_t reserved;  /* never read or written by the library */
} rt_path_id;           /* 16 bytes */

int rt_camera_rays_ids(const rt_camera* camera, uint64_t seed, const rt_path_id* ids, uint64_t n, rt_ray* out);
int rt_camera_rays_ids_device(const rt_camera* camera, uint64_t seed, const rt_path_id* d_ids, uint64_t n,
                              rt_ray* d_out, void* stream);
int rt_world_hit_ids(const rt_scene* scene, const rt_ray* rays, const rt_path_id* ids,
                     const double* t_max_per_ray /* n values or NULL */, uint64_t n, double t_min, double t_max,
                     uint64_t seed, uint32_t flags, rt_hit_record* out, rt_stats* stats);
int rt_world_hit_ids_device(const rt_scene* scene, const rt_ray* d_rays, const rt_path_id* d_ids,
                            const double* d_t_max_per_ray, uint64_t n, double t_min, double t_max, uint64_t seed,
                            uint32_t flags, rt_hit_record* d_out, void* stream, rt_stats* stats);
int rt_shade_ids(const rt_scene* scene, const rt_camera* camera, const rt_hit_record* records, rt_path_id* ids,
                 uint64_t n, uint64_t seed, uint32_t flags, rt_ray* rays, double* beta, double* radiance,
                 uint8_t* state, rt_stats* stats);
int rt_shade_ids_device(const rt_scene* scene, const rt_camera* camera /* host pointer */,
                        const rt_hit_record* d_records, rt_path_id* d_ids, uint64_t n, uint64_t seed, uint32_t flags,
                        rt_ray* d_rays, double* d_beta, double* d_radiance, uint8_t* d_state, void* stream,
                        rt_stats* stats);

typedef enum rt_accum_type { RT_ACCUM_F32 = 0, RT_ACCUM_F64 = 1 } rt_accum_type;

typedef struct rt_render_opts {
    uint32_t struct_size;
    uint32_t flags;          /* RT_OPT_* */
    uint64_t seed;           /* Philox key; the reference RNG is unseeded (utils/random.rs)  */
    uint32_t accum_type;     /* rt_accum_type of the output image                           */
    uint32_t part_index;     /* this caller renders partition part_index of part_count:      */
    uint32_t part_count;     /*   interleaved 8x8 pixel tiles; 0 or 1 = whole image           */
    uint32_t sample_begin;   /* stratum range [sample_begin, sample_end) of sqrt_spp^2;       */
    uint32_t sample_end;     /*   0,0 = all                                                  */
    uint32_t max_paths_in_flight; /* wavefront capacity; 0 = library default                 */
    uint32_t reserved[4];    /* zero.  reserved[0] carries two measurement switches that never change the image:
                                bit 0 = one general shade kernel instead of one per material class,
                                bit 1 = sample the media after the surface hit is known (the order of
                                        Hittables::hit) instead of before it                          */
} rt_render_opts;

/* Render: the pixel loop of Camera::render (camera.rs:179-197) without the 8-bit encode.
 * `accum` is caller-owned, image_width*image_height*3 values of accum_type, and receives the
 * SUM over the rendered samples multiplied by pixel_sample_scale (i.e. the mean linear
 * radiance when all samples and partitions are rendered; partial partitions sum to it). */
int rt_render(const rt_scene* scene, const rt_camera* camera, const rt_render_opts* opts,
              void* accum, rt_stats* stats);
int rt_render_device(const rt_scene* scene, const rt_camera* camera, const rt_render_opts* opts,
                     void* d_accum, void* stream, rt_stats* stats);

/* Camera::render end to end (camera.rs:161-202): render, then Color::to_rgb on the device; only the
 * 3-byte pixels cross PCIe.  `rgb` is a host pointer to image_width*image_height*3 bytes (RgbImage order).
 * Fails with RT_ERR_INVALID if a pixel is NaN (utils/color.rs:28 asserts). */
int rt_render_rgb8(const rt_scene* scene, const rt_camera* camera, const rt_render_opts* opts, uint8_t* rgb,
                   rt_stats* stats);

/* One process, several GPUs: scenes[i] must be the same description created on distinct devices.
 * GPU i renders partition i of n (interleaved 8x8 tiles) from its own host thread into a framebuffer in its own
 * memory; GPU scenes[0]->device then sums the partial frames with one kernel that loads the other GPUs' buffers
 * through peer mappings (NVLink / NVSwitch; staged peer copies where two devices cannot map each other) and only the
 * finished frame crosses PCIe.  This is the in-library form of the reference's single `par_bridge` over pixels
 * (camera.rs:179-181) spread over GPUs.  `accum` as in rt_render.  opts->part_index / part_count must be 0: the
 * partitioning is done here.  stats are totals (times = slowest GPU). */
int rt_render_multi(rt_scene* const* scenes, uint32_t n_scenes, const rt_camera* camera, const rt_render_opts* opts,
                    void* accum, rt_stats* stats);
/* The same, ending like Camera::render (camera.rs:193-194): Color::to_rgb on GPU 0, `rgb` receives the RgbImage bytes. */
int rt_render_multi_rgb8(rt_scene* const* scenes, uint32_t n_scenes, const rt_camera* camera, const rt_render_opts* opts,
                         uint8_t* rgb, rt_stats* stats);

/* Color::to_rgb — utils/color.rs:27-36: optional ACES, then linear -> sRGB 8 bit.
 * `accum` holds mean linear radiance (host pointer), `rgb` receives n_pixels*3 bytes. */
int rt_tonemap(const void* accum, uint32_t accum_type, uint64_t n_pixels, uint32_t toon_map,
               uint8_t* rgb);
/* The same on buffers that already live on the current device (e.g. the framebuffer a multi-GPU client
 * has just reduced with NCCL): `d_accum` and `d_rgb` are device pointers, the work is ordered on
 * `stream` (a cudaStream_t, NULL = default stream) and the call returns once the image is complete. */
int rt_tonemap_device(const void* d_accum, uint32_t accum_type, uint64_t n_pixels, uint32_t toon_map,
                      uint8_t* d_rgb, void* stream);

/* Introspection used by tests and the roofline arithmetic (not needed by a renderer client). */
typedef struct rt_scene_info {
    uint32_t n_prims, n_spheres, n_planars, n_nodes;
    uint32_t n_media, n_lights, n_materials, n_textures;
    uint32_t bvh_depth;
    uint32_t node_bytes; /* bytes read per node visit of a world traversal: 64 (binary tree) or 128 (four-wide collapse
                            used for scenes beyond the caches; node_visits then counts wide nodes) */
    uint64_t device_bytes;
} rt_scene_info;
int rt_scene_get_info(const rt_scene* scene, rt_scene_info* info);
/* tie rank of every flattened primitive, indexed like the desc's objects (RT_NONE for
 * containers): lower rank wins an exact t tie, reproducing hits.rs:42 and bvh.rs:78-84 */
int rt_scene_get_ranks(const rt_scene* scene, uint32_t* ranks, uint32_t n_objects);

const char* rt_last_error(void);
uint32_t rt_abi_version(void);
int rt_device_count(void);

#ifdef __cplusplus
}
#endif
#endif /* RT2025_H */
