// scene_types.h — device-resident scene layout shared by the host compile step and the kernels.
//
// HBM layout (everything 16-byte aligned, read-only during a render):
//   nodes[]   64 B  BVH2 node holding BOTH children's boxes as conservative binary32 bounds and
//                   two child references; one node visit = 4 x LDG.128 and two slab tests.
//   geom[]   128 B  one primitive in BVH leaf order, binary64, the very numbers of the reference's
//                   structs (sphere.rs:17-22, quad.rs:18-29): sphere = centre(3) centre_vec(3)
//                   radius; quad/triangle = anchor(3) u(3) v(3) normal(3) D w(3).  Primitives
//                   below a Transform are stored in that Transform's local space.
//   meta[]    16 B  kind|material, tie rank, object id (rt_hit.prim_id), Transform chain id.
// The BVH is single level over WORLD-space boxes; a leaf primitive that sits below a Transform
// is intersected with the ray taken to its local space (t is preserved, shapes.rs:93-101).
#pragma once
#include <stdint.h>

namespace rt {

constexpr uint32_t LEAF_FLAG = 0x80000000u;
constexpr uint32_t INVALID_REF = 0x7FFFFFFFu;  // empty child / empty group
constexpr int MAX_LEAF_PRIMS = 8;
constexpr int TRAVERSAL_STACK = 64;
constexpr uint32_t META_MAT_MASK = 0x03FFFFFFu;  // PrimMeta::kind_mat
constexpr uint32_t META_CLASS_SHIFT = 26;

// child reference: interior -> node index; leaf -> LEAF_FLAG | first_prim << 3 | (count - 1)
struct alignas(32) Node {
    float lo0[3], hi0[3];
    float lo1[3], hi1[3];
    uint32_t child0, child1;
    uint32_t pad0, pad1;
};
static_assert(sizeof(Node) == 64, "node must be 64 bytes");

// Four-wide node of the collapsed BVH used for scenes that do not fit the caches (world group only): the boxes of
// up to four children as conservative binary32 bounds, child references as in Node.  An unused slot has an
// inverted box and INVALID_REF.  128 bytes = four 256-bit loads; half the dependent fetches of the binary tree.
struct alignas(32) Node4 {
    float box[4][6];  // lo.xyz, hi.xyz per child
    uint32_t child[4];
    uint32_t pad[4];
};
static_assert(sizeof(Node4) == 128, "wide node must be 128 bytes");

enum PrimKind : uint32_t { PRIM_SPHERE = 0, PRIM_QUAD = 1, PRIM_TRIANGLE = 2 };

struct alignas(32) PrimGeom {
    double d[16];
};
static_assert(sizeof(PrimGeom) == 128, "primitive record must be 128 bytes");

struct alignas(16) PrimMeta {
    uint32_t kind_mat;  // kind in bits 30..31, shade class of the material in bits 26..29, material index in bits 0..25
    uint32_t rank;      // lower rank wins an exact t tie (hits.rs:42, bvh.rs:78-84)
    uint32_t object;    // index of the leaf shape in rt_scene_desc.objects
    uint32_t xform;     // index into xforms[] (innermost enclosing Transform) or RT_NONE
};

// One `Transform` (shapes.rs:23-29) plus the chain of Transforms above it.  Primitives below a
// Transform keep their LOCAL geometry; rays are taken to local space with the reference's own
// quaternion arithmetic (shapes.rs:74-101), so t, u, v and the tie behaviour are the reference's.
constexpr int MAX_XFORM_CHAIN = 4;
struct Xform {
    double offset[3];
    double quat[4];  // w x y z
    double scale[3];
    uint32_t chain[MAX_XFORM_CHAIN];  // xform indices from the outermost Transform down to this one
    uint32_t n_chain;
    uint32_t inst_object;  // object id of this Transform (rt_hit.inst_id of the primitives directly below)
};

struct Material {
    uint32_t kind, tex, inner, inner2;
    double color[3];
    double param;
    double v[16];
    uint32_t shade_class, needs_uv;
};

// RemappedMaterial payload (shapes/obj.rs:20-29)
struct Remap {
    double tex_ori[3], tex_u[3], tex_v[3];
    double u_vec[3], v_vec[3];
    double normal[3][3];
    uint32_t has_uv_vecs, normal_tex;
};

struct Texture {
    uint32_t kind, a, b, pad;
    double color[3];
    double color2[3];
    double scale;
};

struct Image {
    uint32_t width, height, flags, pad;
    uint64_t texel_offset;  // in float4 texels
};

struct Perlin {
    double randvec[256][3];
    uint32_t perm_x[256], perm_y[256], perm_z[256];
};

constexpr uint32_t MEDIUM_MAX_ENTRIES = 6, MEDIUM_NO_ENTRIES = 0xFFFFFFFFu;
struct Medium {
    uint32_t root;      // boundary group root reference
    uint32_t material;  // its Isotropic
    uint32_t object;    // object id of the ConstantMedium
    uint32_t rank;
    double neg_inv_density;
    uint32_t xform;     // Transform chain above the medium (ray_length is local, volume.rs:55) or RT_NONE
    uint32_t medium_index;
    uint32_t single_sphere;  // primitive index when the boundary is exactly one Sphere, else RT_NONE
    uint32_t flags;          // MEDIUM_THICK
    // MEDIUM_THICK: every world primitive that can be met by a segment lying inside the boundary sits in one of these
    // leaves of the world tree (leaf references; found by the scene compiler with a box-overlap walk).  n_entry ==
    // MEDIUM_NO_ENTRIES: too many, traverse from the world root.
    uint32_t n_entry;
    uint32_t entry[MEDIUM_MAX_ENTRIES];
    uint32_t pad;
};
// An optically thick medium (boundary radius x density >= 1, every boundary of the scene a single Sphere): a path that
// scatters inside most likely scatters there again, so its scatter points go to the random-walk kernel (k_walk), which
// keeps the path in registers from one scatter point to the next instead of sending it through the streams.
constexpr uint32_t MEDIUM_THICK = 1u;

// One leaf of the lights tree (hits.rs:52-75), geometry in the local space of its Transform chain
struct Light {
    PrimGeom g;
    uint32_t kind;
    uint32_t xform;  // RT_NONE or index into xforms[]
    double weight, cdf, area;
};

// The light list as the lean kernels stage it (WalkLean, ShadeLean): flat - every leaf weighs 1/n - with at most LEAN_LIGHTS
// leaves, none of them below a Transform, so the mixture pdf needs no light-tree or Transform code (kernels.cu, lean_lights_*).
// The scene compiler fills it (compile.cpp, lean_lights) or finds that the scene's list does not qualify.
constexpr uint32_t LEAN_LIGHTS = 4;
struct LeanLights {
    Light lights[LEAN_LIGHTS];  // as in lights[]
    uint32_t n;
    uint32_t pad[7];
};

// The constants of the lean random walk (k_walk<.., LEAN>), gathered by the scene compiler for a scene whose walk needs none of
// the generic machinery: one MEDIUM_THICK medium with its entry leaves, every medium bounded by one untransformed Sphere, an
// Isotropic over a solid texture in the thick one, a LeanLights list and at most WALK_LEAN_PRIMS untransformed primitives in the
// entry leaves.  The kernel copies the record to shared memory once per CTA, so a segment makes no dependent loads through
// media[], materials[], textures[], meta[] or lights[].
constexpr uint32_t WALK_LEAN_MEDIA = 4, WALK_LEAN_PRIMS = 8;
struct WalkLean {
    LeanLights lights;
    PrimGeom prim[WALK_LEAN_PRIMS];      // the primitives of the thick medium's entry leaves, in leaf order
    double sphere[WALK_LEAN_MEDIA][8];   // boundary Sphere of every medium: centre(3) centre_vec(3) radius
    double neg_inv_density[WALK_LEAN_MEDIA];
    double axp[3];                       // albedo / (4 pi) of the thick medium's Isotropic (shade_one's expression)
    double pad0;
    uint32_t rank[WALK_LEAN_MEDIA], medium_index[WALK_LEAN_MEDIA];
    uint32_t prim_kind[WALK_LEAN_PRIMS], prim_rank[WALK_LEAN_PRIMS];
    uint32_t n_media, thick, n_prims;
    // entry primitive whose geometry is bit-identical to the thick boundary sphere (the glass shell around book2's subsurface
    // ball), or RT_NONE: its hit on a segment is decided from the roots the boundary test has already computed
    uint32_t shell;
};

// The constants of the lean shade-class kernels (k_shade<CLS, true>), gathered by the scene compiler; SceneView::shade_lean_mask
// says which classes may use them (bit c: class c):
//   SC_DIFFUSE, SC_TEXTURED - the light list is a LeanLights list;
//   SC_ISOTROPIC            - the same, no surface has an Isotropic material, and every medium that is not MEDIUM_THICK sits below
//                             no Transform and scatters with an Isotropic over a solid texture (its albedo / (4 pi) is in axp);
//   SC_EMISSIVE             - every primitive of the class sits below no Transform and its DiffuseLight (no inner material) has a
//                             solid texture.
// Each CTA copies the record to shared memory, as k_walk does with WalkLean.
constexpr uint32_t SHADE_LEAN_MEDIA = 4;
struct ShadeLean {
    LeanLights lights;
    double axp[SHADE_LEAN_MEDIA][4];  // per medium index: albedo / (4 pi) of its Isotropic (shade_one's expression), w unused
};

// shade work classes used to bin hits (extend -> shade queues)
enum ShadeClass : uint32_t {
    SC_MISS = 0,      // background lookup, path ends
    SC_DIFFUSE = 1,   // cosine pdf with a solid albedo (Lambertian / EmptyMaterial)
    SC_TEXTURED = 2,  // cosine pdf with checker / image / noise albedo
    SC_ISOTROPIC = 3,
    SC_METAL = 4,
    SC_DIELECTRIC = 5,
    SC_EMISSIVE = 6,  // DiffuseLight without inner material: path ends
    SC_DISNEY = 7,    // Disney BSDF, bare or below the OBJ loader's RemappedMaterial / DiffuseLight wrappers
    SC_OTHER = 8,     // Mix, Portal, Transparent, DiffuseLight with inner, anything nested
    SC_WALK = 9,      // scatter point inside an optically thick ConstantMedium (MEDIUM_THICK): k_walk
    SC_COUNT = 10
};

struct SceneView {
    const Node* nodes;
    const PrimGeom* geom;
    const PrimMeta* meta;
    const Xform* xforms;
    const Material* materials;
    const Texture* textures;
    const Image* images;
    const float4* texels;
    const Perlin* perlins;
    const Medium* media;
    const Light* lights;
    const Remap* remaps;
    const Node4* nodes4;  // collapsed four-wide tree of the world group, or nullptr
    uint32_t world_root4; // root reference into nodes4 (only when nodes4 != nullptr)
    uint32_t media_xform;  // some ConstantMedium (or its single-sphere boundary) sits under a Transform
    uint32_t world_root;
    uint32_t n_media, n_lights, n_prims;
    uint32_t n_nodes;
    uint32_t n_cached_nodes;  // nodes [0, n_cached_nodes) (breadth-first top of the tree) are staged in shared memory
    uint32_t stack_entries;   // traversal stack entries per thread
    uint32_t l2_window_bytes; // prefix of nodes[] (breadth first = top of the tree) pinned in L2 by the traversal launches; 0 = none
    uint32_t park_leaves;     // persistent traversal postpones leaves (long traversals) or not (book-sized scenes)
    uint32_t refill_min;      // idle lanes a warp of the persistent traversal waits for before it takes new rays (1..32)
    uint32_t media_stack_entries;  // traversal stack entries per thread of the media kernel (depth of the deepest boundary group)
    uint32_t tail_stack_entries;  // stack entries per thread of k_tail: depth of the deepest binary tree (world or boundary group) + 2
    uint32_t kinds;              // world primitives: 1 = spheres only, 2 = quads / triangles only, 0 = both (or none)
    uint32_t n_xforms;           // Transforms in the scene (0: the traversal needs no local-space rays)
    uint32_t walk_entries_only;  // exactly one MEDIUM_THICK medium and it has its entry leaves: k_walk never traverses from the world root
    uint32_t fifo_slots;      // prepared-ray FIFO slots per warp of the persistent traversal: 32 or 64; 0 = no FIFO (traverse.cuh)
    const WalkLean* walk_lean;  // the scene qualifies for the lean random walk (one record), or nullptr: the generic k_walk
    const ShadeLean* shade_lean;  // the constants of the lean shade-class kernels (one record), or nullptr: every class generic
    uint32_t shade_lean_mask;     // bit c: shade class c runs its lean kernel (ShadeLean)
    uint32_t moving;              // some sphere moves (center_vec != 0): rays with a time outside [0, 1] cull no box (make_rayf)
};

}  // namespace rt
