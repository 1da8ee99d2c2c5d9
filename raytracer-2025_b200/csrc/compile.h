// compile.h — host-side "scene compiler": rt_scene_desc (reference-shaped object graph)
// -> flat device arrays (scene_types.h).
#pragma once
#include <memory>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include <vector_types.h>

#include "rt2025.h"
#include "scene_types.h"

namespace rt {

// std::vector whose resize() leaves trivially constructible elements uninitialised.  The big tables of a scene are
// filled by parallel loops right after they are sized; zero-filling them first is serial page-touching work
// (about 45 GB, 15 s, on a 10^8-primitive scene).
template <class T, class A = std::allocator<T>>
struct default_init_allocator : A {
    using A::A;
    template <class U>
    struct rebind {
        using other = default_init_allocator<U, typename std::allocator_traits<A>::template rebind_alloc<U>>;
    };
    template <class U>
    void construct(U* p) noexcept(std::is_nothrow_default_constructible<U>::value) {
        ::new (static_cast<void*>(p)) U;
    }
    template <class U, class... Args>
    void construct(U* p, Args&&... args) {
        std::allocator_traits<A>::construct(static_cast<A&>(*this), p, std::forward<Args>(args)...);
    }
};
template <class T>
using RawVec = std::vector<T, default_init_allocator<T>>;

struct CompiledScene {
    RawVec<Node> nodes;
    RawVec<Node4> nodes4;  // four-wide collapse of the world tree (empty: not built)
    uint32_t world_root4 = INVALID_REF;
    uint32_t bvh4_depth = 0;
    RawVec<PrimGeom> geom;
    RawVec<PrimMeta> meta;
    std::vector<Xform> xforms;
    std::vector<Material> materials;
    std::vector<Texture> textures;
    std::vector<Image> images;
    std::vector<float4> texels;
    std::vector<Perlin> perlins;
    std::vector<Medium> media;
    std::vector<Light> lights;
    std::vector<Remap> remaps;
    std::vector<uint32_t> ranks;  // per desc object, RT_NONE for containers
    std::vector<WalkLean> walk_lean;  // one record when the scene qualifies for the lean random walk, else empty
    std::vector<ShadeLean> shade_lean;  // one record when some shade class qualifies for its lean kernel, else empty
    uint32_t shade_lean_mask = 0;       // bit c: shade class c runs its lean kernel (scene_types.h, ShadeLean)
    uint32_t world_root = INVALID_REF;
    uint32_t bvh_depth = 0;        // world group (binary tree)
    uint32_t media_bvh_depth = 0;  // deepest ConstantMedium boundary group
    uint32_t n_spheres = 0, n_planars = 0;
};

struct BuildBox;
// Optional replacement for the host SAH builder on the world group (lbvh.cu); same contract as build_bvh below,
// returns false to decline (the host builder then runs).
using WorldBuilder = bool (*)(const RawVec<BuildBox>& boxes, uint32_t first_prim_base, RawVec<Node>& nodes,
                              RawVec<uint32_t>& order, uint32_t& depth_out, uint32_t& root_out);

// returns RT_OK or a negative rt_status and fills err
int compile_scene(const rt_scene_desc& d, uint32_t flags, CompiledScene& out, std::string& err, WorldBuilder world_builder = nullptr);

// Collapse the binary tree below `root` (a reference into `nodes`) into four-wide nodes, breadth first.
// Returns the root reference into `out` (a leaf / INVALID root is returned unchanged) and the depth of the result.
uint32_t collapse_bvh4(const RawVec<Node>& nodes, uint32_t root, RawVec<Node4>& out, uint32_t& depth_out);

// Binned-SAH BVH2 over conservative binary32 boxes.  `order` receives the leaf order (a
// permutation of 0..n-1); nodes are appended to `nodes`; leaf references point at
// first_prim_base + position in `order`.  Returns the root child reference.
struct BuildBox {
    float lo[3], hi[3];
};
uint32_t build_bvh(const RawVec<BuildBox>& boxes, uint32_t first_prim_base, RawVec<Node>& nodes,
                   RawVec<uint32_t>& order, uint32_t& depth_out);
// lbvh.cu: Morton-code LBVH built on the current CUDA device (RT_BUILD_DEVICE_LBVH)
bool build_bvh_device(const RawVec<BuildBox>& boxes, uint32_t first_prim_base, RawVec<Node>& nodes, RawVec<uint32_t>& order,
                      uint32_t& depth_out, uint32_t& root_out);

}  // namespace rt
