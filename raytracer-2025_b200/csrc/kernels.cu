// kernels.cu — the wavefront path tracer and the closest-hit, occlusion, transmittance and world-hit batch kernels (sm_100a).
//
// Pipeline per iteration (all queues and counters live in HBM; no host round trip is needed to
// size a launch — kernels are persistent grid-stride loops that read the counts themselves):
//
//   generate : tops the current ray stream up to capacity with camera rays (Camera::get_ray, camera.rs:247-273)
//   media    : constant-medium sampling (volume.rs:37-73).  When every boundary is a sphere it runs BEFORE extend and
//              leaves the nearest scatter point in the hit stream as the incumbent; otherwise after it, against the
//              surface hit
//   extend   : closest surface hit, persistent traversal (world.hit, camera.rs:286)
//   bin      : the append of every queue position to the shade queue of the winner's material class
//   shade    : one kernel per class - emitted + scatter + mixture-pdf light sampling (camera.rs:290-321);
//              survivors are appended to the other copy of the ray/state streams
//   walk     : the class of scatter points inside optically thick media: the path stays in registers from one scatter point to
//              the next (Isotropic::scatter, then world.hit of the next segment in place) until it leaves the medium or ends
//
// Paths flow through dense, position-indexed streams (kernels.h); terminated paths simply are not
// re-appended.  Radiance is accumulated with binary64 atomics into a per-pixel framebuffer.
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>

#include "kernels.h"
#include "shade.cuh"
#include "shade_step.cuh"

namespace rt {

// ------------------------------------------------------------------------------------------
// closest-hit, occlusion and world-hit surface batch kernels (rt_closest_hit, rt_occluded, rt_world_hit)
// ------------------------------------------------------------------------------------------
struct RayArrayIO {  // rt_closest_hit batches: rays in, rt_hit out
    static constexpr bool any_time = true;  // the caller's rays may carry any time (make_rayf)
    const SceneView& sv;
    const rt_ray* __restrict__ rays;
    rt_hit* __restrict__ out;
    double tmin, tmax;
    __device__ __forceinline__ double t_min() const { return tmin; }
    __device__ __forceinline__ bool load(uint32_t i, RayD& r, double& t1, uint32_t& prim0, uint32_t& rank0) const {
        const double* rp = reinterpret_cast<const double*>(rays + i);
        r.o = D3{rp[0], rp[1], rp[2]};
        r.d = D3{rp[3], rp[4], rp[5]};
        r.time = rp[6];
        t1 = tmax;
        prim0 = 0xFFFFFFFFu, rank0 = 0xFFFFFFFFu;
        return true;
    }
    __device__ __forceinline__ void prefetch(uint32_t i) const { asm volatile("prefetch.global.L2 [%0];" ::"l"(rays + i)); }
    __device__ __forceinline__ void store(uint32_t i, bool hit, double t, uint32_t prim, uint32_t) const {
        rt_hit h;
        if (hit) {
            RayD r;
            double b;
            uint32_t p0, r0;
            load(i, r, b, p0, r0);
            HitInfo hi;
            surface_hit_info(sv, prim, t, r, true, hi);
            const PrimMeta m = sv.meta[prim];
            h.t = t;
            h.prim_id = m.object;
            h.inst_id = m.xform == RT_NONE ? RT_NONE : sv.xforms[m.xform].inst_object;
            h.u = (float)hi.u, h.v = (float)hi.v;
        } else {
            h.t = INFINITY;
            h.prim_id = RT_NONE, h.inst_id = RT_NONE;
            h.u = 0.f, h.v = 0.f;
        }
        out[i] = h;
    }
};

struct OcclusionIO {  // rt_occluded batches: rays and per-ray t_max in, one byte out
    static constexpr bool any_time = true;
    const rt_ray* __restrict__ rays;
    const double* __restrict__ tmax_per_ray;  // nullptr: `tmax` for every ray
    uint8_t* __restrict__ out;
    double tmin, tmax;
    __device__ __forceinline__ double t_min() const { return tmin; }
    __device__ __forceinline__ bool load(uint32_t i, RayD& r, double& t1, uint32_t& prim0, uint32_t& rank0) const {
        const double* rp = reinterpret_cast<const double*>(rays + i);
        r.o = D3{rp[0], rp[1], rp[2]};
        r.d = D3{rp[3], rp[4], rp[5]};
        r.time = rp[6];
        t1 = tmax_per_ray ? tmax_per_ray[i] : tmax;
        prim0 = 0xFFFFFFFFu, rank0 = 0xFFFFFFFFu;
        if (!(tmin <= t1)) {  // an empty interval (t_max_i < t_min, or a NaN bound) contains no t: answered here, never traced
            out[i] = 0;
            return false;
        }
        return true;
    }
    __device__ __forceinline__ void prefetch(uint32_t i) const { asm volatile("prefetch.global.L2 [%0];" ::"l"(rays + i)); }
    __device__ __forceinline__ void store(uint32_t i, bool hit, double, uint32_t, uint32_t) const { out[i] = hit ? 1 : 0; }
};

struct WorldHitIO {  // rt_world_hit's surface pass: rays and per-ray t_max in, the winner (t, kind, internal primitive) out
    static constexpr bool any_time = true;
    const rt_ray* __restrict__ rays;
    const double* __restrict__ tmax_per_ray;  // nullptr: `tmax` for every ray
    HitRec* __restrict__ out;
    double tmin, tmax;
    __device__ __forceinline__ double t_min() const { return tmin; }
    __device__ __forceinline__ bool load(uint32_t i, RayD& r, double& t1, uint32_t& prim0, uint32_t& rank0) const {
        const double* rp = reinterpret_cast<const double*>(rays + i);
        r.o = D3{rp[0], rp[1], rp[2]};
        r.d = D3{rp[3], rp[4], rp[5]};
        r.time = rp[6];
        t1 = tmax_per_ray ? tmax_per_ray[i] : tmax;
        prim0 = 0xFFFFFFFFu, rank0 = 0xFFFFFFFFu;
        if (!(tmin <= t1)) {  // an empty interval (t_max_i < t_min, or a NaN bound) contains no t: answered here, never traced
            store(i, false, 0.0, 0xFFFFFFFFu, 0u);
            return false;
        }
        return true;
    }
    __device__ __forceinline__ void prefetch(uint32_t i) const { asm volatile("prefetch.global.L2 [%0];" ::"l"(rays + i)); }
    __device__ __forceinline__ void store(uint32_t i, bool hit, double t, uint32_t prim, uint32_t) const {
        *reinterpret_cast<double2*>(out + i) = make_double2(hit ? t : INFINITY, __hiloint2double((int)prim, (int)(hit ? HIT_SURFACE : HIT_MISS)));
    }
};

// The persistent traversal of a ray batch, shared by k_closest_hit and k_world_hit_surface (ANY = false) and k_occluded (ANY = true).
template <bool COUNT, bool USE_RANK, bool PARK, int WIDE, bool XF, int KINDS, bool ANY, class IO>
__device__ __forceinline__ void trace_batch(const SceneView& sv, IO& io, uint32_t n, unsigned long long* counters) {
    extern __shared__ float4 s_mem[];  // [cached nodes | traversal stacks | per-warp ray FIFOs]
    __shared__ uint32_t s_cursor;
    uint32_t* stack_base = reinterpret_cast<uint32_t*>(s_mem + cached_tree_float4(sv));
    uint32_t* stack = stack_base + threadIdx.x;
    uint32_t* fifo = stack_base + sv.stack_entries * EXTEND_BLOCK + (threadIdx.x >> 5) * sv.fifo_slots * FIFO_SLOT_WORDS;
    if (threadIdx.x == 0) s_cursor = 0;
    stage_nodes(sv, s_mem);
    TraceCounters cnt{0, 0};
    double* ray_s = reinterpret_cast<double*>(stack_base + sv.stack_entries * EXTEND_BLOCK + (EXTEND_BLOCK / 32) * sv.fifo_slots * FIFO_SLOT_WORDS) + threadIdx.x;
    trace_persistent<COUNT, USE_RANK, PARK, WIDE, XF, KINDS, ANY>(sv, io, n, &s_cursor, s_mem, stack, EXTEND_BLOCK, fifo, sv.fifo_slots, &cnt, ray_s);
    if (COUNT) {
        atomicAdd(&counters[0], (unsigned long long)cnt.nodes);
        atomicAdd(&counters[1], (unsigned long long)cnt.prims);
    }
}

template <bool COUNT, bool PARK, int WIDE, bool XF = true, int KINDS = 0>
__global__ void __launch_bounds__(EXTEND_BLOCK, EXTEND_MIN_BLOCKS) k_closest_hit(SceneView sv, const rt_ray* __restrict__ rays, uint32_t n, double tmin,
                                                                 double tmax, rt_hit* __restrict__ out, unsigned long long* counters) {
    RayArrayIO io{sv, rays, out, tmin, tmax};
    trace_batch<COUNT, true, PARK, WIDE, XF, KINDS, false>(sv, io, n, counters);
}

// any hit: the ray's traversal ends at the first primitive hit, whatever it is (no rank: any hit is the answer)
template <bool COUNT, bool PARK, int WIDE, bool XF = true, int KINDS = 0>
__global__ void __launch_bounds__(EXTEND_BLOCK, EXTEND_MIN_BLOCKS) k_occluded(SceneView sv, const rt_ray* __restrict__ rays, const double* __restrict__ tmax_per_ray,
                                                              uint32_t n, double tmin, double tmax, uint8_t* __restrict__ out, unsigned long long* counters) {
    OcclusionIO io{rays, tmax_per_ray, out, tmin, tmax};
    trace_batch<COUNT, false, PARK, WIDE, XF, KINDS, true>(sv, io, n, counters);
}

// Every instantiation of a batch kernel family that batch_variant() can pick (kernel_setup opts them into the big shared memory).
#define RT_BATCH_VARIANTS(K)                                                                                                            \
    (const void*)K<false, false, 0>, (const void*)K<false, true, 0>, (const void*)K<false, true, 1>, (const void*)K<false, true, 2>,     \
        (const void*)K<true, false, 0>, (const void*)K<true, true, 0>, (const void*)K<true, true, 1>, (const void*)K<true, true, 2>,     \
        (const void*)K<false, false, 3>, (const void*)K<true, false, 3>, (const void*)K<false, true, 1, false, 0>,                      \
        (const void*)K<true, true, 1, false, 0>, (const void*)K<false, true, 1, false, 1>, (const void*)K<true, true, 1, false, 1>,     \
        (const void*)K<false, true, 1, false, 2>, (const void*)K<true, true, 1, false, 2>

// Launch with the top of the BVH pinned in L2.  A scene whose nodes + primitives exceed the L2 makes almost every
// warp-wide node visit wait for at least one lane's DRAM miss; nodes are stored breadth first, so a persisting
// access-policy window over a prefix of the array is "the top of the tree" and keeps it resident while the
// primitive records stream through the rest of the cache.  sv.l2_window_bytes == 0 (cache-resident scenes) is
// a plain launch.  The window is a per-launch attribute: the caller's stream is left untouched.
template <class K, class... Args>
static void launch_with_l2_window(K kernel, const SceneView& sv, int grid, int block, size_t smem, cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid), cfg.blockDim = dim3((unsigned)block);
    cfg.dynamicSmemBytes = smem, cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    if (sv.l2_window_bytes) {
        attr[0].id = cudaLaunchAttributeAccessPolicyWindow;
        attr[0].val.accessPolicyWindow.base_ptr = sv.nodes4 ? (void*)const_cast<Node4*>(sv.nodes4) : (void*)const_cast<Node*>(sv.nodes);
        attr[0].val.accessPolicyWindow.num_bytes = sv.l2_window_bytes;
        attr[0].val.accessPolicyWindow.hitRatio = 1.0f;
        attr[0].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        attr[0].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        cfg.attrs = attr, cfg.numAttrs = 1;
    }
    cudaLaunchKernelEx(&cfg, kernel, args...);
}

// The variant of a batch kernel family a scene runs: one choice for k_closest_hit, k_occluded and k_world_hit_surface.  F::get<COUNT, PARK, WIDE, XF,
// KINDS>() names an instantiation of the family.
template <class F>
static auto batch_variant(const SceneView& sv, bool count) {
    // scenes without any Transform that hold one kind of primitive (a mesh, the soups) have variants without the detransform and
    // without the other primitive test
    auto soup = [&]() {
        if (sv.kinds == 1) return count ? F::template get<true, true, 1, false, 1>() : F::template get<false, true, 1, false, 1>();
        if (sv.kinds == 2) return count ? F::template get<true, true, 1, false, 2>() : F::template get<false, true, 1, false, 2>();
        return count ? F::template get<true, true, 1, false, 0>() : F::template get<false, true, 1, false, 0>();
    };
    return (sv.nodes4 && !sv.n_cached_nodes && !sv.n_xforms) ? soup()
           : sv.nodes4 ? (sv.n_cached_nodes && !sv.fifo_slots ? (count ? F::template get<true, true, 2>() : F::template get<false, true, 2>())
                                                              : (count ? F::template get<true, true, 1>() : F::template get<false, true, 1>()))
           : (!sv.park_leaves && !sv.fifo_slots && sv.n_cached_nodes == sv.n_nodes) ? (count ? F::template get<true, false, 3>() : F::template get<false, false, 3>())
           : count ? (sv.park_leaves ? F::template get<true, true, 0>() : F::template get<true, false, 0>())
                   : (sv.park_leaves ? F::template get<false, true, 0>() : F::template get<false, false, 0>());
}
struct ClosestHitKernels {
    template <bool COUNT, bool PARK, int WIDE, bool XF = true, int KINDS = 0>
    static auto get() { return k_closest_hit<COUNT, PARK, WIDE, XF, KINDS>; }
};
struct OccludedKernels {
    template <bool COUNT, bool PARK, int WIDE, bool XF = true, int KINDS = 0>
    static auto get() { return k_occluded<COUNT, PARK, WIDE, XF, KINDS>; }
};

void launch_closest_hit(const SceneView& sv, const rt_ray* d_rays, uint32_t n, double tmin, double tmax, bool count, rt_hit* d_out,
                        unsigned long long* d_counters, int grid, size_t stack_bytes, cudaStream_t stream) {  // stack_bytes = whole dynamic smem
    launch_with_l2_window(batch_variant<ClosestHitKernels>(sv, count), sv, grid, EXTEND_BLOCK, stack_bytes, stream, sv, d_rays, n, tmin, tmax, d_out,
                          d_counters);
}

void launch_occluded(const SceneView& sv, const rt_ray* d_rays, const double* d_tmax_per_ray, uint32_t n, double tmin, double tmax, bool count,
                     uint8_t* d_out, unsigned long long* d_counters, int grid, size_t stack_bytes, cudaStream_t stream) {
    launch_with_l2_window(batch_variant<OccludedKernels>(sv, count), sv, grid, EXTEND_BLOCK, stack_bytes, stream, sv, d_rays, d_tmax_per_ray, n, tmin,
                          tmax, d_out, d_counters);
}

// ------------------------------------------------------------------------------------------
// wavefront state
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t pack_ids(uint32_t pixel, uint32_t sample, uint32_t segment) {
    return (uint64_t)pixel | ((uint64_t)sample << IDS_PIXEL_BITS) | ((uint64_t)segment << (IDS_PIXEL_BITS + IDS_SAMPLE_BITS));
}
__device__ __forceinline__ void unpack_ids(uint64_t ids, uint32_t& pixel, uint32_t& sample, uint32_t& segment) {
    pixel = (uint32_t)(ids & ((1ull << IDS_PIXEL_BITS) - 1ull));
    sample = (uint32_t)((ids >> IDS_PIXEL_BITS) & ((1ull << IDS_SAMPLE_BITS) - 1ull));
    segment = (uint32_t)(ids >> (IDS_PIXEL_BITS + IDS_SAMPLE_BITS));
}
__device__ __forceinline__ void load_ray(const RayRec* __restrict__ rec, RayD& r, uint64_t& ids) {
    const double2* p = reinterpret_cast<const double2*>(rec);
    double2 a0 = p[0], a1 = p[1], a2 = p[2], a3 = p[3];
    r.o = D3{a0.x, a0.y, a1.x};
    r.d = D3{a1.y, a2.x, a2.y};
    r.time = a3.x;
    ids = (uint64_t)__double_as_longlong(a3.y);
}
__device__ __forceinline__ void store_ray(RayRec* __restrict__ rec, const RayD& r, uint64_t ids) {
    double2* p = reinterpret_cast<double2*>(rec);
    p[0] = make_double2(r.o.x, r.o.y);
    p[1] = make_double2(r.o.z, r.d.x);
    p[2] = make_double2(r.d.y, r.d.z);
    p[3] = make_double2(r.time, __longlong_as_double((long long)ids));
}
__device__ __forceinline__ void store_beta(BetaRec* __restrict__ rec, D3 beta) {
    double2* p = reinterpret_cast<double2*>(rec);
    p[0] = make_double2(beta.x, beta.y);
    p[1] = make_double2(beta.z, 0.0);
}

// warp-aggregated reservation of one entry in queue `q` (lanes with q < 0 reserve nothing);
// returns the reserved position
__device__ __forceinline__ uint32_t queue_reserve(uint32_t* counts, int q) {
    unsigned active = __activemask();
    unsigned peers = __match_any_sync(active, q);
    uint32_t pos = 0;
    if (q >= 0) {
        int leader = __ffs(peers) - 1;
        int lane = threadIdx.x & 31;
        uint32_t base = 0;
        if (lane == leader) base = atomicAdd(&counts[q], (uint32_t)__popc(peers));
        base = __shfl_sync(peers, base, leader);
        pos = base + __popc(peers & ((1u << lane) - 1));
    }
    return pos;
}

// pixel list of this partition: 8x8 tiles dealt round-robin (rt_render_opts.part_index/part_count)
__global__ void k_pixel_list(uint32_t W, uint32_t H, uint32_t part_index, uint32_t part_count, uint32_t* list, uint32_t* count) {
    uint32_t tiles_x = (W + 7) / 8, tiles_y = (H + 7) / 8;
    uint32_t n_tiles = tiles_x * tiles_y;
    // one warp handles one tile = 64 pixels, two per lane; order inside the list is tile-major
    uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) / 32, lane = threadIdx.x & 31;
    uint32_t n_warps = gridDim.x * blockDim.x / 32;
    for (uint32_t tile = warp; tile < n_tiles; tile += n_warps) {
        if (tile % part_count != part_index) continue;
        uint32_t tx = tile % tiles_x, ty = tile / tiles_x;
        // positions in the list are claimed with one atomic per tile (order only affects scheduling)
        uint32_t valid = 0;
        uint32_t px[2], ok[2];
        for (int k = 0; k < 2; k++) {
            uint32_t p = lane + 32 * k;
            uint32_t x = tx * 8 + (p & 7), y = ty * 8 + (p >> 3);
            ok[k] = x < W && y < H;
            px[k] = y * W + x;
            valid += ok[k];
        }
        uint32_t total = valid;
        for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xFFFFFFFFu, total, o);
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(count, total);
        base = __shfl_sync(0xFFFFFFFFu, base, 0);
        // exclusive prefix of `valid` over lanes
        uint32_t incl = valid;
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= (uint32_t)o) incl += v;
        }
        uint32_t pos = base + incl - valid;
        for (int k = 0; k < 2; k++)
            if (ok[k]) list[pos++] = px[k];
    }
}

// after shade the current stream is consumed: its length and the class queues are reset (one thread)
__device__ __forceinline__ void reset_consumed_queues(const WavefrontState& W) {
    Counters* c = W.counters;
    c->n_extend[W.parity] = 0;
    c->walk_cursor = 0;
    for (int k = 0; k < SC_COUNT; k++) c->n_shade[k] = 0;
}
__global__ void k_step(WavefrontState W) { reset_consumed_queues(W); }

// ------------------------------------------------------------------------------------------
// extend
// ------------------------------------------------------------------------------------------
// the free-flight draw of one medium (rt2025_rng.h: one Philox call serves two media; `cache` keeps the pair between the
// iterations of a loop over the media)
struct MediumDraws {
    Rand2 pair;
    uint32_t slot = 0xFFFFFFFFu;
    __device__ __forceinline__ double get(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t segment, uint32_t medium_index) {
        const uint32_t s = RT_MEDIUM_SLOT(medium_index);
        if (s != slot) {
            pair = philox_pair(seed, pixel, sample, segment, s);
            slot = s;
        }
        return (medium_index & 1u) ? pair.b : pair.a;
    }
};

constexpr uint32_t MEDIUM_INCUMBENT = 0x80000000u;  // `prim` of a traversal whose incumbent is a medium scatter point: flag | medium index

// The ray in a medium's space (Medium::xform): ConstantMedium::hit measures ray_length on it (volume.rs:55).  XF: the
// medium may sit under a Transform.
template <bool XF>
__device__ __forceinline__ void medium_ray(const SceneView& sv, const Medium& med, const RayD& r, RayD& lr) {
    lr = r;
    if (XF && med.xform != RT_NONE) lr = ray_to_local(sv, med.xform, r);
}

// The two boundary hits of ConstantMedium::hit (volume.rs:42-45): t1 = boundary.hit(r, UNIVERSE), then
// t2 = boundary.hit(r, [t1 + 1e-4, inf)); false when either misses.  lr = medium_ray(r).
//   SPHERE: the boundary is the single Sphere med.single_sphere; one fused entry/exit test (2 primitive tests) on the
//   sphere's local ray, which is lr unless the sphere sits under a Transform of its own (XF).
//   Otherwise two closest-hit traversals of the boundary group, global nodes only, stacks at `stack` (stride apart).
template <bool COUNT, bool SPHERE, bool XF>
__device__ __forceinline__ bool medium_boundary_hits(const SceneView& sv, const Medium& med, const RayD& r, const RayD& lr, const float4* s_mem,
                                                     uint32_t* stack, int stride, double& t1, double& t2, TraceCounters* cnt) {
    if (SPHERE) {
        RayD br = lr;
        if (XF) {
            const uint32_t bx = sv.meta[med.single_sphere].xform;
            if (bx != med.xform) br = bx == RT_NONE ? r : ray_to_local(sv, bx, r);
        }
        if (COUNT) cnt->prims += 2;
        return sphere_entry_exit(sv.geom[med.single_sphere].d, br, t1, t2);
    }
    uint32_t bp;
    if (!closest_hit<COUNT, false, true>(sv, med.root, r, -INFINITY, INFINITY, s_mem, stack, stride, t1, bp, cnt)) return false;
    return closest_hit<COUNT, false, true>(sv, med.root, r, t1 + 0.0001, INFINITY, s_mem, stack, stride, t2, bp, cnt);
}

// ConstantMedium::hit (volume.rs:37-73) for a medium whose boundary is a single Sphere, on the caller's interval
// [1e-8, inf): true and the scatter distance when the path scatters inside.  XF: the medium or its sphere may sit
// under a Transform.
template <bool COUNT, bool XF>
__device__ __forceinline__ bool sample_sphere_medium(const SceneView& sv, const Medium& med, const RayD& r, double xi, double& tm, TraceCounters* cnt) {
    RayD lr;
    medium_ray<XF>(sv, med, r, lr);
    double t1, t2;
    if (!medium_boundary_hits<COUNT, true, XF>(sv, med, r, lr, nullptr, nullptr, 0, t1, t2, cnt)) return false;
    return medium_free_flight(t1, t2, lr, med.neg_inv_density, xi, tm);
}

// MEDIA: 0 = the ray load does not look at media (none, or they are sampled by k_media after extend);
// 3 = a k_media<PRE> pass ahead of extend left the nearest scatter point of every ray in the hit stream;
// 1 / 2 = every ConstantMedium boundary is a single Sphere and the media are sampled HERE, while the ray is being
// prepared (2: some of them under a Transform).  The nearest scatter point becomes the incumbent of the traversal -
// its distance bounds the search, its tie rank decides an exact tie - so a path scattering inside a dense medium
// (book2's trapped paths bounce there up to max_depth times) costs a traversal of a few units instead of the whole
// scene, and no separate pass re-reads the ray stream.  The winner is the same as with Hittables::hit's order
// (hits.rs:39-46 takes the minimum t over all children, media included).
template <bool COUNT, int MEDIA>
struct PathIO {  // k_extend: rays come from the current ray stream, hits go to the hit stream
    static constexpr bool any_time = false;  // camera rays and their scattered successors carry get_ray's time in [0, 1)
    const SceneView& sv;
    const RayRec* __restrict__ rays;
    HitRec* __restrict__ hits;
    uint8_t* __restrict__ cls;  // nullptr: a media pass follows and writes the class bytes
    uint64_t seed;
    bool bin_by_class, drop_misses;
    TraceCounters* cnt;
    __device__ __forceinline__ double t_min() const { return 1e-8; }  // camera.rs:286
    __device__ __forceinline__ bool load(uint32_t j, RayD& r, double& t1, uint32_t& prim0, uint32_t& rank0) const {
        uint64_t ids;
        load_ray(rays + j, r, ids);
        t1 = INFINITY;
        prim0 = 0xFFFFFFFFu, rank0 = 0xFFFFFFFFu;
        if (MEDIA == 3) {
            const double2 hw = *reinterpret_cast<const double2*>(hits + j);
            if ((uint32_t)__double2loint(hw.y) == HIT_MEDIUM) {  // a surface must beat this point (or tie it with a lower rank)
                const uint32_t m = (uint32_t)__double2hiint(hw.y);
                t1 = hw.x;
                prim0 = MEDIUM_INCUMBENT | m;
                rank0 = sv.media[m].rank;
            }
        } else if (MEDIA) {
            uint32_t pixel, sample, segment;
            unpack_ids(ids, pixel, sample, segment);
            MediumDraws draws;
            for (uint32_t m = 0; m < sv.n_media; m++) {
                const Medium& med = sv.media[m];
                const double xi = draws.get(seed, pixel, sample, segment, med.medium_index);
                double tm;
                if (!sample_sphere_medium<COUNT, MEDIA == 2>(sv, med, r, xi, tm, cnt)) continue;
                // the media compete with each other like any children of a container: nearest, then lower rank
                if (prim0 == 0xFFFFFFFFu || tm < t1 || (tm == t1 && med.rank < rank0)) {
                    t1 = tm;
                    prim0 = MEDIUM_INCUMBENT | m;
                    rank0 = med.rank;
                }
            }
        }
        return true;
    }
    __device__ __forceinline__ void prefetch(uint32_t j) const {
        asm volatile("prefetch.global.L2 [%0];" ::"l"(rays + j));
        if (MEDIA == 3) asm volatile("prefetch.global.L2 [%0];" ::"l"(hits + j));
    }
    __device__ __forceinline__ void store(uint32_t j, bool hit, double t, uint32_t prim, uint32_t prim_meta) const {
        uint32_t kind = HIT_MISS, c = SC_MISS;
        if (hit) {
            if (MEDIA && (prim & MEDIUM_INCUMBENT)) {  // the scatter point kept its place
                kind = HIT_MEDIUM, prim &= ~MEDIUM_INCUMBENT;
                // the phase function of a ConstantMedium is an Isotropic (validated by the scene compiler)
                c = (sv.media[prim].flags & MEDIUM_THICK) ? SC_WALK : SC_ISOTROPIC;
            } else {
                kind = HIT_SURFACE;
                c = (prim_meta >> META_CLASS_SHIFT) & 15u;  // PrimMeta::kind_mat of the winner, kept by the traversal
            }
        }
        *reinterpret_cast<double2*>(hits + j) = make_double2(hit ? t : INFINITY, __hiloint2double((int)prim, (int)kind));
        if (cls) cls[j] = (c == SC_MISS && drop_misses) ? CLASS_DROPPED : (uint8_t)(bin_by_class || c == SC_MISS ? c : SC_DIFFUSE);
    }
};

// closest hit of every path in the extend queue: world.hit (camera.rs:286) over the surfaces and, with MEDIA, the media
template <bool COUNT, bool PARK, int WIDE, int MEDIA>
__global__ void __launch_bounds__(EXTEND_BLOCK, EXTEND_MIN_BLOCKS) k_extend(SceneView sv, RenderParams P, WavefrontState W) {
    extern __shared__ float4 s_mem[];  // [cached nodes | traversal stacks | per-warp ray FIFOs]
    __shared__ uint32_t s_cursor;
    uint32_t* stack_base = reinterpret_cast<uint32_t*>(s_mem + cached_tree_float4(sv));
    uint32_t* stack = stack_base + threadIdx.x;
    uint32_t* fifo = stack_base + sv.stack_entries * EXTEND_BLOCK + (threadIdx.x >> 5) * sv.fifo_slots * FIFO_SLOT_WORDS;
    const uint32_t n = W.counters->n_extend[W.parity];
    if (n == 0) return;
    if (threadIdx.x == 0) s_cursor = 0;
    stage_nodes(sv, s_mem);
    TraceCounters cnt{0, 0};
    // a media pass after extend (classic order, or boundaries that are not spheres) owns the class bytes
    const bool media_pass_follows = sv.n_media != 0 && MEDIA == 0;  // (P.media_first == 0)
    PathIO<COUNT, MEDIA> io{sv, W.ray_q[W.parity], W.hit_q, media_pass_follows ? nullptr : W.cls_q, P.seed, P.bin_by_class != 0, P.drop_misses != 0, &cnt};
    double* ray_s = reinterpret_cast<double*>(stack_base + sv.stack_entries * EXTEND_BLOCK + (EXTEND_BLOCK / 32) * sv.fifo_slots * FIFO_SLOT_WORDS) + threadIdx.x;
    trace_persistent<COUNT, true, PARK, WIDE, true, 0>(sv, io, n, &s_cursor, s_mem, stack, EXTEND_BLOCK, fifo, sv.fifo_slots, &cnt, ray_s);
    if (COUNT) {
        atomicAdd(&W.counters->node_visits, (unsigned long long)cnt.nodes);
        atomicAdd(&W.counters->prim_tests, (unsigned long long)cnt.prims);
    }
}

// ConstantMedium::hit of every medium against the hit known so far (t, prim, kind; kind == HIT_MISS: none): the nearest scatter
// point replaces it when it wins (nearer, or an exact tie with the lower rank).  Returns whether it did.
// `first`: the medium tried first (the winner is the minimum of (t, rank) and does not depend on the order; the one the path
// is most likely to scatter in goes first so that its scatter point screens the others).  FILTER: 0 = every medium,
// 1 = only MEDIUM_THICK ones, 2 = only the others (k_walk asks in two steps and shares the draws between them).
template <bool COUNT, bool GENERIC, bool XF, int FILTER = 0>
__device__ __forceinline__ bool sample_media(const SceneView& sv, uint64_t seed, const RayD& r, uint32_t pixel, uint32_t sample, uint32_t segment, double& t,
                                             uint32_t& prim, uint32_t& kind, const float4* s_mem, uint32_t* stack, int stride, TraceCounters* cntp,
                                             uint32_t first, MediumDraws& draws) {
    uint32_t rank = kind == HIT_SURFACE ? sv.meta[prim].rank : (kind == HIT_MEDIUM ? sv.media[prim].rank : 0xFFFFFFFFu);
    bool changed = false;
        for (uint32_t k = 0; k < sv.n_media; k++) {
            uint32_t m = first + k;
            if (m >= sv.n_media) m -= sv.n_media;
            if (FILTER && ((sv.media[m].flags & MEDIUM_THICK) != 0u) != (FILTER == 1)) continue;
            const Medium& med = sv.media[m];
            const double xi = draws.get(seed, pixel, sample, segment, med.medium_index);
            double tm;
            RayD lr;
            medium_ray<XF>(sv, med, r, lr);
            // skip the boundary test of a medium that cannot beat the known hit
            if (RT_MEDIA_EARLY_SCREEN && kind != HIT_MISS && free_flight_overshoots(med.neg_inv_density, xi, t, lr.d)) continue;
            if (med.single_sphere != RT_NONE) {
                if (!sample_sphere_medium<COUNT, XF>(sv, med, r, xi, tm, cntp)) continue;
            } else if (GENERIC) {
                double t1, t2;
                if (!medium_boundary_hits<COUNT, false, XF>(sv, med, r, lr, s_mem, stack, stride, t1, t2, cntp)) continue;
                if (t1 < 1e-8) t1 = 1e-8;  // clamp to the caller's interval [1e-8, inf)
                if (t1 >= t2) continue;
                if (t1 < 0.0) t1 = 0.0;
                const double ray_length = length(lr.d);
                const double distance_inside_boundary = (t2 - t1) * ray_length;
                const double hit_distance = med.neg_inv_density * log(xi);
                if (hit_distance > distance_inside_boundary) continue;
                tm = t1 + hit_distance / ray_length;
            } else {
                continue;  // unreachable: the host launches the GENERIC instantiation for such scenes
            }
            // the medium competes with the other children of its container like any hit
            if (kind == HIT_MISS || tm < t || (tm == t && med.rank < rank)) {
                t = tm;
                prim = m;
                kind = HIT_MEDIUM;
                rank = med.rank;
                changed = true;
            }
        }
    return changed;
}

template <bool COUNT, bool GENERIC, bool XF>
__device__ __forceinline__ bool sample_media(const SceneView& sv, uint64_t seed, const RayD& r, uint32_t pixel, uint32_t sample, uint32_t segment, double& t,
                                             uint32_t& prim, uint32_t& kind, const float4* s_mem, uint32_t* stack, int stride, TraceCounters* cntp) {
    MediumDraws draws;
    return sample_media<COUNT, GENERIC, XF, 0>(sv, seed, r, pixel, sample, segment, t, prim, kind, s_mem, stack, stride, cntp, 0u, draws);
}

// Camera::get_ray, camera.rs:247-273: tops the current ray stream up to capacity with camera rays
// MEDIA: the scene's media all have sphere boundaries and are sampled ahead of extend (RenderParams::media_first == 1): the
// free-flight draws of segment 0 are taken here, while the ray is in registers, and the nearest scatter point goes to the hit
// stream as extend's incumbent - the sampling pass then only reads the survivors of the last shade stage (a camera ray is a
// quarter to a third of all segments, and this kernel is bound by its stores).  XF as in k_media.
#ifndef RT_GEN_MEDIA_MIN_BLOCKS
#define RT_GEN_MEDIA_MIN_BLOCKS 4
#endif
template <bool MEDIA, bool XF>
__global__ void __launch_bounds__(256, MEDIA ? RT_GEN_MEDIA_MIN_BLOCKS : 4) k_generate(SceneView sv, RenderParams P, WavefrontState W) {
    const uint64_t remaining = W.total_paths - W.counters->next_path;
    const uint32_t extend_base = W.counters->n_extend[W.parity];
    const uint32_t room = W.capacity - extend_base;
    const uint32_t n_new = (uint32_t)(remaining < (uint64_t)room ? remaining : (uint64_t)room);
    const uint64_t first = W.counters->next_path;
    const rt_camera& cam = P.cam;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n_new; j += gridDim.x * blockDim.x) {
        uint64_t g = first + j;
        uint32_t sidx = P.sample_begin + (uint32_t)(g / W.n_pixels);
        uint32_t pixel = W.pixel_list[g % W.n_pixels];
        RayD r;
        camera_ray(cam, P.seed, pixel, sidx, r);
        store_ray(W.ray_q[W.parity] + extend_base + j, r, pack_ids(pixel, sidx, 0u));
        store_beta(W.beta_q[W.parity] + extend_base + j, D3{1.0, 1.0, 1.0});
        if (MEDIA) {
            double t = INFINITY;
            uint32_t prim = 0xFFFFFFFFu, kind = HIT_MISS;
            TraceCounters cnt{0, 0};
            sample_media<false, false, XF>(sv, P.seed, r, pixel, sidx, 0u, t, prim, kind, nullptr, nullptr, 0, &cnt);
            *reinterpret_cast<double2*>(W.hit_q + extend_base + j) = make_double2(t, __hiloint2double((int)prim, (int)kind));
        }
    }
    // Bookkeeping of the stage (it used to be a launch of its own): every block read the counters above before it got here,
    // so the LAST block to arrive may advance them - the next kernel of the stream sees the topped-up queue length.
    __syncthreads();
    if (threadIdx.x == 0) {
        Counters* c = W.counters;
        __threadfence();
        if (atomicAdd(&c->gen_done, 1u) == gridDim.x - 1u) {
            c->gen_done = 0;
            c->next_path += n_new;
            c->n_extend[W.parity] = extend_base + n_new;
            c->n_unsampled = MEDIA ? extend_base : extend_base + n_new;
            c->segments += extend_base + n_new;
            c->iterations += (extend_base + n_new > 0);
            __threadfence();
        }
    }
}

// Media pass AFTER extend (the order of Hittables::hit): ConstantMedium::hit for every medium (volume.rs:37-73)
// against the surface hit k_extend found, one thread per extend-queue entry.  Used when some boundary is not a
// single Sphere (GENERIC: the boundary needs a BVH traversal per lane, kept out of the common instantiation because
// it doubles the register footprint) and for the classic-order A/B switch; sphere-bounded media are otherwise sampled
// by k_extend itself (PathIO<MEDIA>).  Writes the winner back to the hit stream and the class byte of every entry.
//   MODE 1: every boundary is a single Sphere; MODE 2: general boundaries.
//   XF = some medium (or its sphere boundary) sits under a Transform (without the detransform code the single-sphere
//   pass needs 81 registers instead of 126 and runs three CTAs per SM).
//   PRE = the pass runs BEFORE extend (sphere boundaries only): it knows no surface hit and leaves the nearest scatter
//   point (or a miss) in the hit stream; extend takes it as the incumbent (PathIO<3>) and writes the class bytes.
template <bool COUNT, int MODE, bool XF, bool PRE>
__global__ void __launch_bounds__(MEDIA_BLOCK, MODE == 2 ? RT_MEDIA_GENERIC_MIN_BLOCKS : (XF ? RT_MEDIA_MIN_BLOCKS : RT_MEDIA_MIN_BLOCKS_NOXF))
    k_media(SceneView sv, RenderParams P, WavefrontState W) {
    constexpr bool GENERIC = MODE == 2;
    extern __shared__ float4 s_mem[];  // traversal stacks for boundaries that are not a single sphere
    uint32_t* stack = reinterpret_cast<uint32_t*>(s_mem) + threadIdx.x;
    TraceCounters cnt{0, 0};
    const uint32_t n = PRE ? W.counters->n_unsampled : W.counters->n_extend[W.parity];
    const uint32_t n_round = (n + 31u) & ~31u;  // whole warps iterate together
    const RayRec* __restrict__ rays = W.ray_q[W.parity];
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n_round; j += gridDim.x * blockDim.x) {
        {  // pull the next iteration's records towards L1 while this one computes
            const uint32_t jn = j + gridDim.x * blockDim.x;
            if (jn < n) {
                asm volatile("prefetch.global.L1 [%0];" ::"l"(rays + jn));
                if (!PRE) asm volatile("prefetch.global.L1 [%0];" ::"l"(W.hit_q + jn));
            }
        }
        if (j >= n) continue;
        double t = INFINITY;
        uint32_t prim = 0xFFFFFFFFu, kind = HIT_MISS;
        if (!PRE) {
            const double2 hw = *reinterpret_cast<const double2*>(W.hit_q + j);
            t = hw.x;
            prim = (uint32_t)__double2hiint(hw.y), kind = (uint32_t)__double2loint(hw.y);
        }
        RayD r;
        uint64_t ids64;
        load_ray(rays + j, r, ids64);
        uint32_t pixel, sample, segment;
        unpack_ids(ids64, pixel, sample, segment);
        const uint32_t surface_meta = kind == HIT_SURFACE ? __ldg(&sv.meta[prim].kind_mat) : 0u;
        const bool changed = sample_media<COUNT, GENERIC, XF>(sv, P.seed, r, pixel, sample, segment, t, prim, kind, s_mem, stack, MEDIA_BLOCK, &cnt);
        if (PRE || changed) *reinterpret_cast<double2*>(W.hit_q + j) = make_double2(t, __hiloint2double((int)prim, (int)kind));
        if (PRE) continue;  // extend writes the class bytes
        uint32_t c = kind == HIT_MISS     ? (uint32_t)SC_MISS
                     : kind == HIT_MEDIUM ? ((sv.media[prim].flags & MEDIUM_THICK) ? (uint32_t)SC_WALK : (uint32_t)SC_ISOTROPIC)
                                          : ((surface_meta >> META_CLASS_SHIFT) & 15u);
        if (!P.bin_by_class && c != SC_MISS) c = SC_DIFFUSE;
        W.cls_q[j] = (c == SC_MISS && P.drop_misses) ? CLASS_DROPPED : (uint8_t)c;
    }
    if (COUNT) {
        atomicAdd(&W.counters->node_visits, (unsigned long long)cnt.nodes);
        atomicAdd(&W.counters->prim_tests, (unsigned long long)cnt.prims);
    }
}

// rt_transmittance's media pass, after k_occluded left the surface answer of every ray in `occluded`: one ray per thread.
// An occluded ray gets 0 (its ray record is not read), an empty interval 1, every other ray the product over the media, in
// medium order, of the probability that ConstantMedium::hit (volume.rs:37-73) returns None on the caller's interval
// [tmin, t_max_i]: exp(distance_inside_boundary / neg_inv_density).  GENERIC / XF as MODE 2 / XF of k_media.
template <bool COUNT, bool GENERIC, bool XF>
__global__ void __launch_bounds__(MEDIA_BLOCK) k_transmittance(SceneView sv, const rt_ray* __restrict__ rays, const double* __restrict__ tmax_per_ray,
                                                             uint32_t n, double tmin, double tmax, const uint8_t* __restrict__ occluded,
                                                             double* __restrict__ out, unsigned long long* counters) {
    extern __shared__ float4 s_mem[];  // traversal stacks for boundaries that are not a single sphere
    uint32_t* stack = reinterpret_cast<uint32_t*>(s_mem) + threadIdx.x;
    TraceCounters cnt{0, 0};
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        if (occluded[i]) {
            out[i] = 0.0;
            continue;
        }
        const double t_max_i = tmax_per_ray ? tmax_per_ray[i] : tmax;
        if (!(tmin <= t_max_i)) {  // an empty interval (t_max_i < t_min, or a NaN bound): nothing in it can stop the ray
            out[i] = 1.0;
            continue;
        }
        const double* rp = reinterpret_cast<const double*>(rays + i);
        RayD r;
        r.o = D3{rp[0], rp[1], rp[2]};
        r.d = D3{rp[3], rp[4], rp[5]};
        r.time = rp[6];
        double T = 1.0;
        for (uint32_t m = 0; m < sv.n_media; m++) {
            const Medium& med = sv.media[m];
            RayD lr;
            medium_ray<XF>(sv, med, r, lr);
            double t1, t2;
            if (med.single_sphere != RT_NONE) {
                if (!medium_boundary_hits<COUNT, true, XF>(sv, med, r, lr, s_mem, stack, MEDIA_BLOCK, t1, t2, &cnt)) continue;
            } else if (GENERIC) {
                if (!medium_boundary_hits<COUNT, false, XF>(sv, med, r, lr, s_mem, stack, MEDIA_BLOCK, t1, t2, &cnt)) continue;
            } else {
                continue;  // unreachable: the host launches the GENERIC instantiation for such scenes
            }
            if (t1 < tmin) t1 = tmin;  // clamp_min_assign / clamp_max_assign to the caller's interval
            if (t2 > t_max_i) t2 = t_max_i;
            if (t1 >= t2) continue;
            if (t1 < 0.0) t1 = 0.0;
            const double distance_inside_boundary = (t2 - t1) * length(lr.d);
            T *= exp(distance_inside_boundary / med.neg_inv_density);
        }
        out[i] = T;
    }
    if (COUNT) {
        atomicAdd(&counters[0], (unsigned long long)cnt.nodes);
        atomicAdd(&counters[1], (unsigned long long)cnt.prims);
    }
}

// rt_world_hit's record pass, after k_world_hit_surface left the surface winner of every ray in `surface`: one ray per thread.
// Every medium competes on the caller's interval [tmin, t_max_i] as ConstantMedium::hit (volume.rs:37-73) does there, with the
// free-flight draw philox(seed; pixel = i, sample = 0, segment, RT_MEDIUM_SLOT(medium_index)); the nearest t wins, an exact tie
// goes to the lower rank.  The winner's HitRecord is rebuilt in world space.  GENERIC / XF as in k_transmittance.
template <bool COUNT, bool GENERIC, bool XF>
__global__ void __launch_bounds__(MEDIA_BLOCK) k_world_hit_record(SceneView sv, const rt_ray* __restrict__ rays, const double* __restrict__ tmax_per_ray,
                                                                uint32_t n, double tmin, double tmax, uint64_t seed, uint32_t segment,
                                                                const HitRec* __restrict__ surface, rt_hit_record* __restrict__ out,
                                                                unsigned long long* counters) {
    extern __shared__ float4 s_mem[];  // traversal stacks for boundaries that are not a single sphere
    uint32_t* stack = reinterpret_cast<uint32_t*>(s_mem) + threadIdx.x;
    TraceCounters cnt{0, 0};
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const double2 hw = *reinterpret_cast<const double2*>(surface + i);
        double t = hw.x;
        uint32_t kind = (uint32_t)__double2loint(hw.y), prim = (uint32_t)__double2hiint(hw.y);
        const double t_max_i = tmax_per_ray ? tmax_per_ray[i] : tmax;
        // an empty interval (t_max_i < t_min, or a NaN bound) is a miss of the surface pass and takes no draws; a surface miss
        // in a scene without media needs no ray
        const bool media = tmin <= t_max_i && sv.n_media != 0;
        RayD r;
        if (media || kind != HIT_MISS) {
            const double* rp = reinterpret_cast<const double*>(rays + i);
            r.o = D3{rp[0], rp[1], rp[2]};
            r.d = D3{rp[3], rp[4], rp[5]};
            r.time = rp[6];
        }
        uint32_t rank = kind == HIT_SURFACE ? sv.meta[prim].rank : 0xFFFFFFFFu;
        MediumDraws draws;
        for (uint32_t m = 0; media && m < sv.n_media; m++) {
            const Medium& med = sv.media[m];
            RayD lr;
            medium_ray<XF>(sv, med, r, lr);
            double t1, t2;
            if (med.single_sphere != RT_NONE) {
                if (!medium_boundary_hits<COUNT, true, XF>(sv, med, r, lr, s_mem, stack, MEDIA_BLOCK, t1, t2, &cnt)) continue;
            } else if (GENERIC) {
                if (!medium_boundary_hits<COUNT, false, XF>(sv, med, r, lr, s_mem, stack, MEDIA_BLOCK, t1, t2, &cnt)) continue;
            } else {
                continue;  // unreachable: the host launches the GENERIC instantiation for such scenes
            }
            if (t1 < tmin) t1 = tmin;  // clamp_min_assign / clamp_max_assign to the caller's interval
            if (t2 > t_max_i) t2 = t_max_i;
            if (t1 >= t2) continue;
            if (t1 < 0.0) t1 = 0.0;
            const double ray_length = length(lr.d);
            const double distance_inside_boundary = (t2 - t1) * ray_length;
            const double hit_distance = med.neg_inv_density * log(draws.get(seed, i, 0u, segment, med.medium_index));
            if (hit_distance > distance_inside_boundary) continue;
            const double tm = t1 + hit_distance / ray_length;
            // the medium competes with the other children of its container like any hit
            if (kind == HIT_MISS || tm < t || (tm == t && med.rank < rank)) {
                t = tm;
                prim = m;
                kind = HIT_MEDIUM;
                rank = med.rank;
            }
        }
        HitInfo h;
        uint32_t object = RT_NONE, xform = RT_NONE;
        if (kind == HIT_MEDIUM) {  // volume.rs:66-72 in the medium's space, as shade_one builds it
            const Medium& med = sv.media[prim];
            RayD lr;
            medium_ray<XF>(sv, med, r, lr);
            h.p = lr.o + t * lr.d;
            const D3 nrm = D3{1.0, 0.0, 0.0};
            h.front_face = dot(lr.d, nrm) < 0.0;
            h.normal = h.front_face ? nrm : -nrm;
            h.u = 0.0, h.v = 0.0;
            h.material = med.material;
            object = med.object;
            if (XF && med.xform != RT_NONE) {
                xform = med.xform;
                hit_to_world(sv, xform, h);
            }
        } else if (kind == HIT_SURFACE) {
            surface_hit_info(sv, prim, t, r, true, h);
            const PrimMeta pm = sv.meta[prim];
            object = pm.object, xform = pm.xform;
        } else {
            t = INFINITY;
            h.p = h.normal = D3{0.0, 0.0, 0.0};
            h.u = h.v = 0.0;
            h.front_face = false;
            h.material = RT_NONE;
        }
        rt_hit_record rec;
        rec.t = t;
        rec.p[0] = h.p.x, rec.p[1] = h.p.y, rec.p[2] = h.p.z;
        rec.normal[0] = h.normal.x, rec.normal[1] = h.normal.y, rec.normal[2] = h.normal.z;
        rec.u = h.u, rec.v = h.v;
        rec.kind = kind == HIT_MEDIUM ? RT_HIT_MEDIUM : kind == HIT_SURFACE ? RT_HIT_SURFACE : RT_HIT_MISS;
        rec.front_face = h.front_face ? 1u : 0u;
        rec.prim_id = object;
        rec.inst_id = xform == RT_NONE ? RT_NONE : sv.xforms[xform].inst_object;
        rec.material = h.material;
        rec.reserved = 0;
        out[i] = rec;
    }
    if (COUNT) {
        atomicAdd(&counters[0], (unsigned long long)cnt.nodes);
        atomicAdd(&counters[1], (unsigned long long)cnt.prims);
    }
}

// Binning: the append of every queue position to the shade queue of its class byte.  A memory-bound pass (1 byte in,
// 4 bytes out per entry) with one global atomic per class per 256 entries: same-address atomics are what bounds it.
__global__ void __launch_bounds__(MEDIA_BLOCK, 4) k_bin(WavefrontState W) {
    __shared__ uint32_t s_cnt[2][SC_COUNT], s_base[SC_COUNT];
    if (threadIdx.x < 2 * SC_COUNT) (&s_cnt[0][0])[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t n = W.counters->n_extend[W.parity];
    const uint32_t n_round = (n + MEDIA_BLOCK - 1u) / MEDIA_BLOCK * MEDIA_BLOCK;  // whole CTAs iterate together
    uint32_t it = 0;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n_round; j += gridDim.x * blockDim.x, it++) {
        int q = j < n ? (int)W.cls_q[j] : -1;
        if (q == (int)CLASS_DROPPED) q = -1;
        uint32_t* cntb = s_cnt[it & 1];
        const uint32_t local = queue_reserve(cntb, q);
        __syncthreads();
        if (threadIdx.x < SC_COUNT) {
            const uint32_t c = cntb[threadIdx.x];
            if (c) s_base[threadIdx.x] = atomicAdd(&W.counters->n_shade[threadIdx.x], c);
            s_cnt[(it & 1) ^ 1][threadIdx.x] = 0;
        }
        __syncthreads();
        if (q >= 0) W.q_shade[q][s_base[q] + local] = j;
    }
}

// ------------------------------------------------------------------------------------------
// shade
// ------------------------------------------------------------------------------------------
// contribute, shade_one and lean_isotropic_scatter: shade_step.cuh

// CTAs per SM of the lean class kernels, one hex digit per shade class (digit c: class c).  Measured on book2 (torch.profiler, ms
// per frame at 2 / 3 / 4 CTAs): diffuse 39.1 / 34.0 / 35.9, textured 18.3 / 20.0 / 22.5, isotropic 22.5 / 20.9 / 20.6, emissive
// 14.5 / 12.7 / 13.0.  Isotropic keeps three: four is within 0.3 ms and spills more.
#ifndef RT_SHADE_LEAN_BLOCKS
#define RT_SHADE_LEAN_BLOCKS 0x3003230u
#endif
constexpr int shade_lean_blocks(uint32_t cls) { return (int)((RT_SHADE_LEAN_BLOCKS >> (4u * cls)) & 15u); }
constexpr int shade_blocks(uint32_t cls, bool lean) {
    return lean ? shade_lean_blocks(cls) : (((RT_SHADE_3BLOCK_MASK >> cls) & 1u) ? 3 : RT_SHADE_MIN_BLOCKS);
}

// One instantiation per shade class (scene_types.h ShadeClass): the queue it reads only holds hits
// of that class, so everything another class would need is compiled out and the kernel keeps few
// registers.  CLS == SC_OTHER is the fully general version (Mix, Portal, Transparent, lights that
// wrap a material) and is also what runs when binning is switched off.
// LEAN: the scene lets class CLS skip the code it cannot reach (scene_types.h, ShadeLean; SceneView::shade_lean_mask); each CTA
// copies the ShadeLean record to shared memory first.  SC_EMISSIVE then only adds beta * the light's colour: it reads the path
// ids, the throughput and the hit record, and no geometry.
template <uint32_t CLS, bool LEAN = false>
__global__ void __launch_bounds__(SHADE_BLOCK, shade_blocks(CLS, LEAN)) k_shade(SceneView sv, RenderParams P, WavefrontState W, uint32_t queue) {
    constexpr bool EMIT_ONLY = LEAN && CLS == SC_EMISSIVE;
    __shared__ uint32_t s_warp_count[SHADE_BLOCK / 32];
    __shared__ uint32_t s_base;
    extern __shared__ float4 s_lean[];  // LEAN: the ShadeLean record
    const ShadeLean& SL = *reinterpret_cast<const ShadeLean*>(s_lean);
    if (LEAN && !EMIT_ONLY) {
        unsigned long long* dst = reinterpret_cast<unsigned long long*>(s_lean);
        const unsigned long long* src = reinterpret_cast<const unsigned long long*>(sv.shade_lean);
        for (uint32_t k = threadIdx.x; k < sizeof(ShadeLean) / 8; k += SHADE_BLOCK) dst[k] = src[k];
        __syncthreads();
    }
    unsigned long long lean_hits = 0;  // thread 0: the entries this CTA shaded
    const uint32_t n = W.counters->n_shade[queue];
    const RayRec* __restrict__ rays = W.ray_q[W.parity];
    const BetaRec* __restrict__ betas = W.beta_q[W.parity];
    // the loop bound is uniform over the block: the survivor append is aggregated per block
    for (uint32_t j0 = blockIdx.x * blockDim.x; j0 < n; j0 += gridDim.x * blockDim.x) {
        const uint32_t j = j0 + threadIdx.x;
        int q = -1;
        RayD nr;
        D3 nbeta;
        uint32_t pixel = 0, sidx = 0, segment = 0;
#if RT_SHADE_PREFETCH
        {  // the records are gathered through the class queue: start pulling the next round's towards L2/L1 now
            const uint32_t jn = j + gridDim.x * blockDim.x;
            if (jn < n) {
                const uint32_t pn = W.q_shade[queue][jn];
                asm volatile("prefetch.global.L2 [%0];" ::"l"(rays + pn));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(betas + pn));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(W.hit_q + pn));
            }
        }
#endif
        if (LEAN && threadIdx.x == 0) lean_hits += min(n - j0, (uint32_t)SHADE_BLOCK);
        if (j < n) {
            const uint32_t pos = W.q_shade[queue][j];
            if constexpr (EMIT_ONLY) {  // material_emitted of a DiffuseLight over a solid texture; the path ends
                unpack_ids((uint64_t)__double_as_longlong(reinterpret_cast<const double2*>(rays + pos)[3].y), pixel, sidx, segment);
                const double2* sp2 = reinterpret_cast<const double2*>(betas + pos);
                const double2 b0 = sp2[0], b1 = sp2[1];
                const D3 beta = D3{b0.x, b0.y, b1.x};
                const uint32_t prim = (uint32_t)__double2hiint(reinterpret_cast<const double2*>(W.hit_q + pos)->y);
                const uint32_t mat = sv.meta[prim].kind_mat & META_MAT_MASK;
                const D3 e = D3{0.0, 0.0, 0.0} + 1.0 * ld3(sv.textures[sv.materials[mat].tex].color);
                contribute(P, W, pixel, beta * e);
            } else {
                RayD r;
                uint64_t ids64;
                load_ray(rays + pos, r, ids64);
                unpack_ids(ids64, pixel, sidx, segment);
                const double2* sp2 = reinterpret_cast<const double2*>(betas + pos);
                const double2 b0 = sp2[0], b1 = sp2[1];
                D3 beta = D3{b0.x, b0.y, b1.x};
                const double2 hw = *reinterpret_cast<const double2*>(W.hit_q + pos);
                const double t = hw.x;
                const uint32_t prim = (uint32_t)__double2hiint(hw.y), kind = (uint32_t)__double2loint(hw.y);
                bool alive;
                if constexpr (LEAN && CLS == SC_ISOTROPIC)  // only media scatter here (ShadeLean): prim is the medium index
                    alive = lean_isotropic_scatter(sv, SL.lights, ld3(SL.axp[prim]), P, W, r, beta, pixel, sidx, segment, t, nr, nbeta);
                else
                    alive = shade_one<CLS, LEAN>(sv, P, W, r, beta, pixel, sidx, segment, t, prim, kind, nr, nbeta, &SL.lights);
                q = alive ? 0 : -1;
            }
        }
        if constexpr (EMIT_ONLY) continue;  // no survivors
        // survivors are appended to the other copy of the streams: one atomic per block
        const unsigned alive_mask = __ballot_sync(0xFFFFFFFFu, q == 0);
        const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
        if (lane == 0) s_warp_count[warp] = __popc(alive_mask);
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t total = 0;
#pragma unroll
            for (int w = 0; w < SHADE_BLOCK / 32; w++) total += s_warp_count[w];
            s_base = total ? atomicAdd(&W.counters->n_extend[W.parity ^ 1u], total) : 0u;
        }
        __syncthreads();
        uint32_t npos = s_base + __popc(alive_mask & ((1u << lane) - 1u));
        for (uint32_t w = 0; w < warp; w++) npos += s_warp_count[w];
        __syncthreads();  // s_warp_count / s_base are reused by the next iteration
        if constexpr (!EMIT_ONLY) {
            if (q == 0) {
                store_ray(W.ray_q[W.parity ^ 1u] + npos, nr, pack_ids(pixel, sidx, segment + 1));
                store_beta(W.beta_q[W.parity ^ 1u] + npos, nbeta);
            }
        }
    }
    if (LEAN && lean_hits) atomicAdd(&W.counters->shade_lean_hits, lean_hits);
}

// ------------------------------------------------------------------------------------------
// random walk inside an optically thick medium
// ------------------------------------------------------------------------------------------
// A path that scatters inside a dense ConstantMedium (book2's blue subsurface sphere: mean free path 5 in a sphere of radius 70)
// scatters there again and again until max_depth ends it: on book2_final a third of ALL segments are such scatter points, and
// each went through the sampling pass, extend, the binning and the isotropic shade kernel - four trips through HBM and a
// traversal at extend's 15 active lanes for a segment that is a few units long.  k_walk takes the queue of scatter points inside
// MEDIUM_THICK media and keeps every path in registers from one scatter point to the next: Isotropic::scatter + the mixture pdf
// (the SC_ISOTROPIC code of shade_one), then world.hit of the NEXT segment in place - the free-flight draw of every medium
// (volume.rs:37-73, the medium the path is in first, so that its scatter point screens the others) and a traversal bounded by
// the nearest scatter point, with the tie rule of the wavefront (a surface wins with a smaller t, or the same t and a lower
// rank).  While a thick medium wins again the loop goes on; otherwise the new ray is appended to the ray stream like any
// survivor of a shade kernel and the wavefront evaluates that segment itself (one look-ahead per walk is computed twice).
// Every draw is addressed by (pixel, sample, segment, slot), so the radiance is the very sum the wavefront alone produces.
// A lane whose walk ends takes the next queue entry at once (static striding, no atomics): the loop body is the same for every
// lane, so the warp stays converged however long the individual walks are.
#ifndef RT_WALK_BLOCK
#define RT_WALK_BLOCK 128
#endif
constexpr int WALK_BLOCK = RT_WALK_BLOCK;
#ifndef RT_WALK_MIN_BLOCKS
#define RT_WALK_MIN_BLOCKS 4
#endif
#ifndef RT_WALK_LEAN_MIN_BLOCKS
#define RT_WALK_LEAN_MIN_BLOCKS 4
#endif

// One segment of the lean walk (scene_types.h, WalkLean) from a scatter point at t inside the thick medium: lean_isotropic_scatter,
// then the look-ahead of k_walk - the thick medium, the thin ones when it
// scattered, the entry primitives - against the staged constants.  Returns whether the path goes on (nr, nbeta); `stay`: the
// next scatter point (at tn) is again inside the thick medium and nothing beats it.
__device__ __forceinline__ bool walk_lean_segment(const SceneView& sv, const WalkLean& L, const RenderParams& P, const WavefrontState& W, const RayD& r,
                                                  D3 beta, uint32_t pixel, uint32_t sidx, uint32_t segment, double t, uint32_t max_steps,
                                                  uint32_t& steps, RayD& nr, D3& nbeta, double& tn, bool& stay) {
    stay = false;
    if (!lean_isotropic_scatter(sv, L.lights, ld3(L.axp), P, W, r, beta, pixel, sidx, segment, t, nr, nbeta)) return false;

    // world.hit of the next segment, as sample_media<.., 1> then <.., 2> and leaf_beats_scatter
    const uint32_t seg1 = segment + 1u, thick = L.thick;
    MediumDraws draws;
    double near_root, far_root;  // the thick boundary's roots: the shell's Sphere::hit on this ray has the same
    {
        const double* s = L.sphere[thick];
        double t1, t2;
        const double xi = draws.get(P.seed, pixel, sidx, seg1, L.medium_index[thick]);
        const bool inside = sphere_entry_exit_at(ld3(s), ld3(s + 3), s[6], nr, t1, t2, near_root, far_root);
        if (!inside || !medium_free_flight(t1, t2, nr, L.neg_inv_density[thick], xi, tn)) return true;
    }
    if (!(++steps < max_steps)) return true;
    const uint32_t med_rank = L.rank[thick];
    for (uint32_t m = 0; m < L.n_media; m++) {
        if (m == thick) continue;
        const double xi = draws.get(P.seed, pixel, sidx, seg1, L.medium_index[m]);
        if (RT_MEDIA_EARLY_SCREEN && free_flight_overshoots(L.neg_inv_density[m], xi, tn, nr.d)) continue;
        const double* s = L.sphere[m];
        double t1, t2, nroot, froot, tm;
        if (!sphere_entry_exit_at(ld3(s), ld3(s + 3), s[6], nr, t1, t2, nroot, froot) || !medium_free_flight(t1, t2, nr, L.neg_inv_density[m], xi, tm)) continue;
        if (tm < tn || (tm == tn && L.rank[m] < med_rank)) return true;  // a thin medium wins: the walk ends whatever else does
    }
    bool beaten = false;
    for (uint32_t i = 0; i < L.n_prims && !beaten; i++) {
        const double* g = L.prim[i].d;
        double th;
        bool hit;
        if (i == L.shell) {  // sphere_hit's choice: the near root if it lies in [1e-8, tn], else the far one
            th = near_root;
            hit = contains(1e-8, tn, th);
            if (!hit) {
                th = far_root;
                hit = contains(1e-8, tn, th);
            }
        } else if (L.prim_kind[i] == PRIM_SPHERE) {
            hit = sphere_hit_at(ld3(g), ld3(g + 3), g[6], nr, 1e-8, tn, th);
        } else {
            Planar pl;
            load_planar_plain(g, pl);
            double a, b;
            hit = planar_hit_loaded(pl, L.prim_kind[i] == PRIM_TRIANGLE, nr, 1e-8, tn, th, a, b);
        }
        beaten = hit && (th < tn || L.prim_rank[i] < med_rank);
    }
    stay = !beaten;
    return true;
}

// ENTRIES: every thick medium of the scene has its entry leaves and there is only one of them, so the traversal from the world
// root (another medium's scatter point, more leaves than slots) is never needed and is compiled out.
// LEAN: the scene's walk constants are staged (SceneView::walk_lean, implies ENTRIES and !XF): walk_lean_segment.
template <bool XF, bool ENTRIES, bool LEAN = false>
__global__ void __launch_bounds__(WALK_BLOCK, LEAN ? RT_WALK_LEAN_MIN_BLOCKS : RT_WALK_MIN_BLOCKS) k_walk(SceneView sv, RenderParams P, WavefrontState W) {
    extern __shared__ float4 s_mem[];  // traversal stacks (global-memory nodes only) | LEAN: the WalkLean record
    uint32_t* stack = reinterpret_cast<uint32_t*>(s_mem) + threadIdx.x;
    const WalkLean& L = *reinterpret_cast<const WalkLean*>(s_mem);
    if (LEAN) {
        unsigned long long* dst = reinterpret_cast<unsigned long long*>(s_mem);
        const unsigned long long* src = reinterpret_cast<const unsigned long long*>(sv.walk_lean);
        for (uint32_t k = threadIdx.x; k < sizeof(WalkLean) / 8; k += WALK_BLOCK) dst[k] = src[k];
        __syncthreads();
    }
    const uint32_t n = W.counters->n_shade[SC_WALK];
    const RayRec* __restrict__ rays = W.ray_q[W.parity];
    const BetaRec* __restrict__ betas = W.beta_q[W.parity];
    const uint32_t* __restrict__ queue = W.q_shade[SC_WALK];
    const uint32_t lane = threadIdx.x & 31u;
    const unsigned FULL = 0xFFFFFFFFu, lt_mask = (1u << lane) - 1u;
    TraceCounters cnt{0, 0};
    unsigned long long walked = 0;
    bool have = false;
    RayD r;
    D3 beta;
    uint32_t pixel = 0, sidx = 0, segment = 0, medium = 0;
    double t = 0.0;
    // A walk is a serial chain (about 8 us per segment for a warp that has the SM to itself): once the queue is too short to fill the
    // GPU - the drain of a frame, where every iteration would wait some 300 us for the handful of paths that have just entered the
    // medium - a walk is cut after `drain_steps` segments and its path goes back to the ray stream; the wavefront evaluates the
    // next segment, finds the same scatter point and queues the path for the walk of the next iteration.
    const uint32_t max_steps = n <= P.walk_drain_queue ? P.walk_drain_steps : 0xFFFFFFFFu;
    uint32_t steps = 0;
    // queue entries are claimed 32 at a time per warp (one atomic, records prefetched) and handed to the lanes as their walks end
    uint32_t pool_next = 0, pool_end = 0;  // warp-uniform
    bool exhausted = false;                // warp-uniform: the cursor ran past the queue
    while (true) {
        unsigned need = __ballot_sync(FULL, !have);
        while (need && !(exhausted && pool_next == pool_end)) {
            if (pool_next == pool_end) {
                uint32_t base = 0;
                if (lane == 0) base = atomicAdd(&W.counters->walk_cursor, 32u);
                base = __shfl_sync(FULL, base, 0);
                if (base >= n) {
                    exhausted = true;
                    break;
                }
                pool_next = base, pool_end = min(base + 32u, n);
                if (base + lane < pool_end) {
                    const uint32_t pos = queue[base + lane];
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(rays + pos));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(betas + pos));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(W.hit_q + pos));
                }
            }
            const uint32_t take = min((uint32_t)__popc(need), pool_end - pool_next);
            const uint32_t my = __popc(need & lt_mask);
            if (!have && my < take) {
                const uint32_t pos = queue[pool_next + my];
                uint64_t ids64;
                load_ray(rays + pos, r, ids64);
                unpack_ids(ids64, pixel, sidx, segment);
                const double2* sp2 = reinterpret_cast<const double2*>(betas + pos);
                const double2 b0 = sp2[0], b1 = sp2[1];
                beta = D3{b0.x, b0.y, b1.x};
                const double2 hw = *reinterpret_cast<const double2*>(W.hit_q + pos);
                t = hw.x;
                medium = (uint32_t)__double2hiint(hw.y);
                have = true;
                steps = 0;
            }
            pool_next += take;
            need = __ballot_sync(FULL, !have);
        }
        if (need == FULL) break;  // nothing left to claim and every walk of the warp has ended
        if (have) {
            RayD nr;
            D3 nbeta;
            double tn = INFINITY;
            uint32_t pn = medium;
            bool alive, stay = false;
            if constexpr (LEAN) {
                alive = walk_lean_segment(sv, L, P, W, r, beta, pixel, sidx, segment, t, max_steps, steps, nr, nbeta, tn, stay);
            } else if ((alive = shade_one<SC_ISOTROPIC>(sv, P, W, r, beta, pixel, sidx, segment, t, medium, HIT_MEDIUM, nr, nbeta))) {
                // world.hit of the next segment: the thick media first (the one the path is in leads); when none of them scatters
                // the walk is over whatever the thin ones do, otherwise they are screened by the scatter point found
                uint32_t kn = HIT_MISS;
                pn = 0xFFFFFFFFu;
                MediumDraws draws;
                sample_media<false, false, XF, 1>(sv, P.seed, nr, pixel, sidx, segment + 1u, tn, pn, kn, s_mem, stack, WALK_BLOCK, &cnt, medium, draws);
                stay = kn == HIT_MEDIUM && ++steps < max_steps;
                if (stay) {
                    sample_media<false, false, XF, 2>(sv, P.seed, nr, pixel, sidx, segment + 1u, tn, pn, kn, s_mem, stack, WALK_BLOCK, &cnt, 0u, draws);
                    stay = (sv.media[pn].flags & MEDIUM_THICK) != 0u;
                }
                if (stay) {
                    const Medium& mn = sv.media[pn];
                    const uint32_t med_rank = mn.rank;
                    double ts;
                    uint32_t ps;
                    if (ENTRIES || (pn == medium && mn.n_entry != MEDIUM_NO_ENTRIES)) {
                        // both ends of the segment lie inside the same boundary: only the world leaves that overlap it can be met
                        for (uint32_t e = 0; e < mn.n_entry && stay; e++) stay = !leaf_beats_scatter(sv, mn.entry[e], nr, 1e-8, tn, med_rank);
                    } else if (closest_hit<false, true, false>(sv, sv.world_root, nr, 1e-8, tn, s_mem, stack, WALK_BLOCK, ts, ps, &cnt)) {
                        stay = !(ts < tn || sv.meta[ps].rank < med_rank);
                    }
                }
            }
            if (!alive) {
                have = false;
            } else if (stay) {
                r = nr, beta = nbeta, segment++, t = tn, medium = pn;
                walked++;
            } else {
                const uint32_t npos = queue_reserve(&W.counters->n_extend[W.parity ^ 1u], 0);
                store_ray(W.ray_q[W.parity ^ 1u] + npos, nr, pack_ids(pixel, sidx, segment + 1u));
                store_beta(W.beta_q[W.parity ^ 1u] + npos, nbeta);
                have = false;
            }
        }
    }
    if (walked) {
        atomicAdd(&W.counters->segments, walked);
        atomicAdd(&W.counters->walk_segments, walked);
        if (LEAN) atomicAdd(&W.counters->walk_lean_segments, walked);
    }
}
static void launch_walk(const SceneView& sv, const RenderParams& P, const WavefrontState& W, int grid, cudaStream_t s) {
    SceneView wv = sv;
    wv.n_cached_nodes = 0;  // the non-persistent closest_hit() reads the binary tree from global memory
    if (sv.walk_lean) {  // no traversal: the dynamic shared memory holds the staged constants
        k_walk<false, true, true><<<grid / RT_WALK_MIN_BLOCKS * RT_WALK_LEAN_MIN_BLOCKS, WALK_BLOCK, sizeof(WalkLean), s>>>(wv, P, W);
        return;
    }
    const size_t smem = (size_t)std::max(sv.tail_stack_entries, 4u) * WALK_BLOCK * sizeof(uint32_t);
    auto k = sv.media_xform ? (sv.walk_entries_only ? k_walk<true, true> : k_walk<true, false>) : (sv.walk_entries_only ? k_walk<false, true> : k_walk<false, false>);
    k<<<grid, WALK_BLOCK, smem, s>>>(wv, P, W);
}

// ------------------------------------------------------------------------------------------
// tail: the last few thousand paths of a frame, traced to completion by one launch
// ------------------------------------------------------------------------------------------
// Once every camera path has been generated the wavefront only drains: depth-40 stragglers keep it alive for dozens of
// iterations of ~14 launches each that move a few hundred paths - a fixed cost per frame that does not shrink when the frame
// is split over GPUs (round 1: 5.6 % of the 8-GPU step).  k_tail is launched after every iteration and returns at once unless
// generation is over and at most `threshold` paths are left; then one thread takes one path and runs generate-less
// extend -> media -> shade in a loop until the path ends.  The draws are addressed by (pixel, sample, segment, slot), so the
// radiance is the very sum the wavefront would have produced.  The last CTA to finish marks the queue empty.
constexpr int TAIL_BLOCK = MEDIA_BLOCK;
__global__ void __launch_bounds__(TAIL_BLOCK, 1) k_tail(SceneView sv, RenderParams P, WavefrontState W, uint32_t threshold) {
    extern __shared__ float4 s_mem[];  // traversal stacks (global-memory nodes only)
    uint32_t* stack = reinterpret_cast<uint32_t*>(s_mem) + threadIdx.x;
    Counters* c = W.counters;
    // the bookkeeping after shade (nobody in this kernel reads what it resets: the consumed stream's length and the class queues)
    if (blockIdx.x == 0 && threadIdx.x == 0) reset_consumed_queues(W);
    const uint32_t np = W.parity ^ 1u;  // shade has just appended the survivors to the other copy of the streams
    const uint32_t n = c->n_extend[np];
    if (n == 0 || n > threshold || c->next_path < W.total_paths) return;
    const RayRec* __restrict__ rays = W.ray_q[np];
    const BetaRec* __restrict__ betas = W.beta_q[np];
    TraceCounters cnt{0, 0};
    unsigned long long my_segments = 0;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
        RayD r;
        uint64_t ids64;
        load_ray(rays + j, r, ids64);
        uint32_t pixel, sidx, segment;
        unpack_ids(ids64, pixel, sidx, segment);
        const double2* sp2 = reinterpret_cast<const double2*>(betas + j);
        const double2 b0 = sp2[0], b1 = sp2[1];
        D3 beta = D3{b0.x, b0.y, b1.x};
        while (true) {
            my_segments++;
            double t = INFINITY;
            uint32_t prim = 0xFFFFFFFFu, kind = HIT_MISS;
            if (closest_hit<false, true, false>(sv, sv.world_root, r, 1e-8, INFINITY, s_mem, stack, TAIL_BLOCK, t, prim, &cnt)) kind = HIT_SURFACE;
            if (sv.n_media) sample_media<false, true, true>(sv, P.seed, r, pixel, sidx, segment, t, prim, kind, s_mem, stack, TAIL_BLOCK, &cnt);
            RayD nr;
            D3 nbeta;
            if (!shade_one<SC_OTHER>(sv, P, W, r, beta, pixel, sidx, segment, t, prim, kind, nr, nbeta)) break;
            r = nr, beta = nbeta, segment++;
        }
    }
    if (my_segments) atomicAdd(&c->segments, my_segments);
    // every CTA read `n` before it got here, and the last one to arrive does so after all the others have finished
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&c->pad, 1u) == gridDim.x - 1u) {
            c->n_extend[np] = 0;
            c->pad = 0;
            c->iterations += 1;
        }
    }
}
void launch_tail(const SceneView& sv, const RenderParams& P, const WavefrontState& W, uint32_t threshold, int grid, cudaStream_t s) {
    SceneView tv = sv;
    tv.n_cached_nodes = 0;  // the non-persistent closest_hit() reads the binary tree from global memory
    const size_t smem = (size_t)std::max(sv.tail_stack_entries, 4u) * TAIL_BLOCK * sizeof(uint32_t);
    k_tail<<<grid, TAIL_BLOCK, smem, s>>>(tv, P, W, threshold);
}

__global__ void k_finalize(const double* __restrict__ accum, uint64_t n, double scale, void* out, int out_f64) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        double v = accum[i] * scale;
        if (out_f64)
            reinterpret_cast<double*>(out)[i] = v;
        else
            reinterpret_cast<float*>(out)[i] = (float)v;
    }
}


// The multi-GPU reduce: GPU 0 sums the partial framebuffers where they lie.  parts.p[k] for k > 0 are PEER pointers (memory of
// the other GPUs mapped through cudaDeviceEnablePeerAccess), so the loads below cross NVLink / NVSwitch; every value is read once
// and only GPU 0 writes.  The partitions are disjoint pixel tiles, so most addends are zero and the sum is also the gather.
template <class T>
__global__ void __launch_bounds__(256) k_sum_parts(PartList parts, T* __restrict__ out, uint64_t n) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        T acc = reinterpret_cast<const T*>(parts.p[0])[i];
        for (uint32_t k = 1; k < parts.n; k++) acc += reinterpret_cast<const T*>(parts.p[k])[i];
        out[i] = acc;
    }
}
void launch_sum_parts(const PartList& parts, void* out, uint64_t n_values, bool f64, int grid, cudaStream_t s) {
    if (f64)
        k_sum_parts<double><<<grid, 256, 0, s>>>(parts, reinterpret_cast<double*>(out), n_values);
    else
        k_sum_parts<float><<<grid, 256, 0, s>>>(parts, reinterpret_cast<float*>(out), n_values);
}

// Color::to_rgb, utils/color.rs:14-36: optional ACES fit, then linear -> sRGB 8 bit.  palette's
// encoder is not vendored with the reference; this is the standard piecewise curve rounded to
// nearest (palette's f32 fast path may differ by one code at rounding boundaries).
__global__ void k_tonemap(const void* __restrict__ accum, int f64, uint64_t n_pixels, uint32_t toon_map, uint8_t* __restrict__ rgb, int* error_flag) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pixels; i += (uint64_t)gridDim.x * blockDim.x) {
        D3 c;
        if (f64) {
            const double* a = reinterpret_cast<const double*>(accum) + 3 * i;
            c = D3{a[0], a[1], a[2]};
        } else {
            const float* a = reinterpret_cast<const float*>(accum) + 3 * i;
            c = D3{(double)a[0], (double)a[1], (double)a[2]};
        }
        if (isnan(c.x) || isnan(c.y) || isnan(c.z)) *error_flag = 1;  // color.rs:28 assert
        if (toon_map == 1) {  // aces_tonemap, color.rs:14-25
            const double A = 2.51, C = 2.43;
            const D3 B = D3{0.03, 0.03, 0.03}, Dd = D3{0.59, 0.59, 0.59}, E = D3{0.14, 0.14, 0.14};
            D3 num = c * (A * c + B), den = c * (C * c + Dd) + E;
            D3 m = D3{num.x / den.x, num.y / den.y, num.z / den.z};
            c = D3{fmin(fmax(m.x, 0.0), 1.0), fmin(fmax(m.y, 0.0), 1.0), fmin(fmax(m.z, 0.0), 1.0)};
        }
        double v[3] = {c.x, c.y, c.z};
        for (int k = 0; k < 3; k++) {
            double x = v[k];
            double enc = x <= 0.0031308 ? 12.92 * x : 1.055 * pow(x, 1.0 / 2.4) - 0.055;
            if (!(enc > 0.0)) enc = 0.0;
            if (enc > 1.0) enc = 1.0;
            rgb[3 * i + k] = (uint8_t)llrint(floor(enc * 255.0 + 0.5));
        }
    }
}
void launch_tonemap(const void* accum, bool f64, uint64_t n_pixels, uint32_t toon_map, uint8_t* rgb, int* error_flag, cudaStream_t s) {
    int grid = (int)((n_pixels + 255) / 256);
    if (grid > 148 * 8) grid = 148 * 8;
    if (grid < 1) grid = 1;
    k_tonemap<<<grid, 256, 0, s>>>(accum, f64 ? 1 : 0, n_pixels, toon_map, rgb, error_flag);
}

// ------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------
void launch_init(const WavefrontState& W, const RenderParams& P, int grid, cudaStream_t s) {
    k_pixel_list<<<grid, 256, 0, s>>>(P.cam.image_width, P.cam.image_height, P.part_index, P.part_count, W.pixel_list, &W.counters->n_pixels);
}
void launch_generate(const SceneView& sv, const RenderParams& P, const WavefrontState& W, int grid, cudaStream_t s) {
    if (P.media_first == 1 && sv.n_media && P.sample_in_generate) {
        grid = grid / 4 * RT_GEN_MEDIA_MIN_BLOCKS;  // api.cu sizes the grid for four resident CTAs per SM
        sv.media_xform ? k_generate<true, true><<<grid, 256, 0, s>>>(sv, P, W) : k_generate<true, false><<<grid, 256, 0, s>>>(sv, P, W);
    } else
        k_generate<false, false><<<grid, 256, 0, s>>>(sv, P, W);
}
template <int MEDIA>
static void launch_extend_media(const SceneView& sv, const RenderParams& P, const WavefrontState& W, bool count, int grid, size_t stack_bytes, cudaStream_t s) {
    auto k = sv.nodes4 ? (sv.n_cached_nodes && !sv.fifo_slots ? (count ? k_extend<true, true, 2, MEDIA> : k_extend<false, true, 2, MEDIA>)
                                            : (count ? k_extend<true, true, 1, MEDIA> : k_extend<false, true, 1, MEDIA>))
             : (!sv.park_leaves && !sv.fifo_slots && sv.n_cached_nodes == sv.n_nodes) ? (count ? k_extend<true, false, 3, MEDIA> : k_extend<false, false, 3, MEDIA>)
             : count   ? (sv.park_leaves ? k_extend<true, true, 0, MEDIA> : k_extend<true, false, 0, MEDIA>)
                       : (sv.park_leaves ? k_extend<false, true, 0, MEDIA> : k_extend<false, false, 0, MEDIA>);
    launch_with_l2_window(k, sv, grid, EXTEND_BLOCK, stack_bytes, s, sv, P, W);
}
void launch_extend(const SceneView& sv, const RenderParams& P, const WavefrontState& W, bool count, int grid, size_t stack_bytes, cudaStream_t s) {
    if (P.media_first == 2 && sv.n_media)
        sv.media_xform ? launch_extend_media<2>(sv, P, W, count, grid, stack_bytes, s) : launch_extend_media<1>(sv, P, W, count, grid, stack_bytes, s);
    else if (P.media_first == 1 && sv.n_media)
        launch_extend_media<3>(sv, P, W, count, grid, stack_bytes, s);
    else
        launch_extend_media<0>(sv, P, W, count, grid, stack_bytes, s);
}
int launch_media_bin(const SceneView& sv, const RenderParams& P, const WavefrontState& W, bool count, bool generic, int grid, cudaStream_t s, int phase) {
    if (phase == 1) {  // media-first order: the sampling pass ahead of extend (sphere boundaries)
        const bool xf = sv.media_xform != 0;
        auto k = count ? (xf ? k_media<true, 1, true, true> : k_media<true, 1, false, true>) : (xf ? k_media<false, 1, true, true> : k_media<false, 1, false, true>);
        k<<<grid, MEDIA_BLOCK, 0, s>>>(sv, P, W);
        return 1;
    }
    int launches = 1;
    if (phase == 0 && sv.n_media) {  // the media pass after extend: global-memory nodes only (its shared memory holds just the stacks)
        SceneView mv = sv;
        mv.n_cached_nodes = 0;
        const size_t media_smem = generic ? (size_t)sv.media_stack_entries * MEDIA_BLOCK * sizeof(uint32_t) : 0;  // <= 64 KB, opted in by kernel_setup
        const bool xf = sv.media_xform != 0;
        if (generic) {
            auto k = count ? (xf ? k_media<true, 2, true, false> : k_media<true, 2, false, false>) : (xf ? k_media<false, 2, true, false> : k_media<false, 2, false, false>);
            k<<<grid, MEDIA_BLOCK, media_smem, s>>>(mv, P, W);
        } else {
            auto k = count ? (xf ? k_media<true, 1, true, false> : k_media<true, 1, false, false>) : (xf ? k_media<false, 1, true, false> : k_media<false, 1, false, false>);
            k<<<grid, MEDIA_BLOCK, 0, s>>>(mv, P, W);
        }
        launches++;
    }
    k_bin<<<grid, MEDIA_BLOCK, 0, s>>>(W);
    return launches;
}
void launch_transmittance(const SceneView& sv, bool generic, const rt_ray* d_rays, const double* d_tmax_per_ray, uint32_t n, double tmin, double tmax,
                          bool count, const uint8_t* d_occluded, double* d_out, unsigned long long* d_counters, int grid, cudaStream_t s) {
    SceneView mv = sv;  // global-memory nodes only, as the media pass of the render (its shared memory holds just the stacks)
    mv.n_cached_nodes = 0;
    const size_t media_smem = generic ? (size_t)sv.media_stack_entries * MEDIA_BLOCK * sizeof(uint32_t) : 0;  // <= 64 KB, opted in by kernel_setup
    const bool xf = sv.media_xform != 0;
    auto k = generic ? (count ? (xf ? k_transmittance<true, true, true> : k_transmittance<true, true, false>)
                              : (xf ? k_transmittance<false, true, true> : k_transmittance<false, true, false>))
                     : (count ? (xf ? k_transmittance<true, false, true> : k_transmittance<true, false, false>)
                              : (xf ? k_transmittance<false, false, true> : k_transmittance<false, false, false>));
    k<<<grid, MEDIA_BLOCK, media_smem, s>>>(mv, d_rays, d_tmax_per_ray, n, tmin, tmax, d_occluded, d_out, d_counters);
}
void launch_world_hit_record(const SceneView& sv, bool generic, const rt_ray* d_rays, const double* d_tmax_per_ray, uint32_t n, double tmin,
                             double tmax, uint64_t seed, uint32_t segment, bool count, const HitRec* d_surface, rt_hit_record* d_out,
                             unsigned long long* d_counters, int grid, cudaStream_t s) {
    SceneView mv = sv;  // global-memory nodes only, as launch_transmittance
    mv.n_cached_nodes = 0;
    const size_t media_smem = generic ? (size_t)sv.media_stack_entries * MEDIA_BLOCK * sizeof(uint32_t) : 0;  // <= 64 KB, opted in by kernel_setup
    const bool xf = sv.media_xform != 0;
    auto k = generic ? (count ? (xf ? k_world_hit_record<true, true, true> : k_world_hit_record<true, true, false>)
                              : (xf ? k_world_hit_record<false, true, true> : k_world_hit_record<false, true, false>))
                     : (count ? (xf ? k_world_hit_record<true, false, true> : k_world_hit_record<true, false, false>)
                              : (xf ? k_world_hit_record<false, false, true> : k_world_hit_record<false, false, false>));
    k<<<grid, MEDIA_BLOCK, media_smem, s>>>(mv, d_rays, d_tmax_per_ray, n, tmin, tmax, seed, segment, d_surface, d_out, d_counters);
}
template <uint32_t CLS>
static void launch_shade_cls(const SceneView& sv, const RenderParams& P, const WavefrontState& W, uint32_t queue, int grid, cudaStream_t s) {
    // `grid` is sized for RT_SHADE_MIN_BLOCKS resident CTAs per SM; classes compiled for another count get the matching grid
    if constexpr (CLS == SC_DIFFUSE || CLS == SC_TEXTURED || CLS == SC_ISOTROPIC || CLS == SC_EMISSIVE) {
        if (queue == CLS && (sv.shade_lean_mask >> CLS) & 1u) {  // the scene compiler's choice (scene_types.h, ShadeLean)
            static_assert(shade_lean_blocks(CLS) >= 1, "RT_SHADE_LEAN_BLOCKS: no CTA count for a lean class");
            k_shade<CLS, true><<<grid / RT_SHADE_MIN_BLOCKS * shade_lean_blocks(CLS), SHADE_BLOCK, CLS == SC_EMISSIVE ? 0 : sizeof(ShadeLean), s>>>(sv, P, W, queue);
            return;
        }
    }
    if ((RT_SHADE_3BLOCK_MASK >> CLS) & 1u) grid = grid / RT_SHADE_MIN_BLOCKS * 3;
    k_shade<CLS><<<grid, SHADE_BLOCK, 0, s>>>(sv, P, W, queue);
}
// class_mask: bit c set when the scene can produce hits of shade class c (the miss queue always runs).
// The class kernels are independent (own queue each, atomics on the shared outputs): with `fan` they are dealt
// over side streams between a fork and a join event so that the tail of one overlaps the start of the next.
int launch_shade(const SceneView& sv, const RenderParams& P, const WavefrontState& W, uint32_t class_mask, int grid, cudaStream_t s,
                 const ShadeFan* fan, bool tail_follows, int walk_grid) {
    int launches = tail_follows ? 1 : 2;  // the miss kernel (and k_step)
    if (!P.bin_by_class) {  // everything but misses sits in the SC_DIFFUSE queue: general kernel
        launch_shade_cls<SC_MISS>(sv, P, W, SC_MISS, grid, s);
        launch_shade_cls<SC_OTHER>(sv, P, W, SC_DIFFUSE, grid, s);
        launches++;
    } else {
        const int n_side = fan ? fan->n_side : 0;
        if (n_side) {
            cudaEventRecord(fan->fork, s);
            for (int i = 0; i < n_side; i++) cudaStreamWaitEvent(fan->side[i], fan->fork, 0);
        }
        int next = 0;
        auto lane = [&]() {  // main stream first, then the side streams, round robin
            const int k = next++ % (n_side + 1);
            return k == 0 ? s : fan->side[k - 1];
        };
        // the random walk runs longest (one launch takes its paths through dozens of segments): start it first
        if (class_mask & (1u << SC_WALK)) launch_walk(sv, P, W, walk_grid, lane()), launches++;
        // the classes that usually hold most hits first, so they start on different streams
        if (class_mask & (1u << SC_DIFFUSE)) launch_shade_cls<SC_DIFFUSE>(sv, P, W, SC_DIFFUSE, grid, lane()), launches++;
        if (class_mask & (1u << SC_ISOTROPIC)) launch_shade_cls<SC_ISOTROPIC>(sv, P, W, SC_ISOTROPIC, grid, lane()), launches++;
        if (class_mask & (1u << SC_DISNEY)) launch_shade_cls<SC_DISNEY>(sv, P, W, SC_DISNEY, grid, lane()), launches++;
        if (class_mask & (1u << SC_TEXTURED)) launch_shade_cls<SC_TEXTURED>(sv, P, W, SC_TEXTURED, grid, lane()), launches++;
        launch_shade_cls<SC_MISS>(sv, P, W, SC_MISS, grid, lane());
        if (class_mask & (1u << SC_DIELECTRIC)) launch_shade_cls<SC_DIELECTRIC>(sv, P, W, SC_DIELECTRIC, grid, lane()), launches++;
        if (class_mask & (1u << SC_EMISSIVE)) launch_shade_cls<SC_EMISSIVE>(sv, P, W, SC_EMISSIVE, grid, lane()), launches++;
        if (class_mask & (1u << SC_METAL)) launch_shade_cls<SC_METAL>(sv, P, W, SC_METAL, grid, lane()), launches++;
        if (class_mask & (1u << SC_OTHER)) launch_shade_cls<SC_OTHER>(sv, P, W, SC_OTHER, grid, lane()), launches++;
        for (int i = 0; i < n_side; i++) {
            cudaEventRecord(fan->join[i], fan->side[i]);
            cudaStreamWaitEvent(s, fan->join[i], 0);
        }
    }
    if (!tail_follows) k_step<<<1, 1, 0, s>>>(W);  // otherwise k_tail, launched next, resets the consumed queues
    return launches;
}
void launch_finalize(const double* accum, uint64_t n, double scale, void* out, bool out_f64, int grid, cudaStream_t s) {
    k_finalize<<<grid, 256, 0, s>>>(accum, n, scale, out, out_f64 ? 1 : 0);
}

// The surface pass of rt_world_hit: closest hit on [tmin, t_max_i], the internal primitive kept for the record pass.  Defined
// after the render kernels: instantiated ahead of them, the family changes the register assignment of four k_shade
// instantiations (same instructions, permuted registers), and the render's SASS is kept as it was.
template <bool COUNT, bool PARK, int WIDE, bool XF = true, int KINDS = 0>
__global__ void __launch_bounds__(EXTEND_BLOCK, EXTEND_MIN_BLOCKS) k_world_hit_surface(SceneView sv, const rt_ray* __restrict__ rays,
                                                                       const double* __restrict__ tmax_per_ray, uint32_t n, double tmin,
                                                                       double tmax, HitRec* __restrict__ out, unsigned long long* counters) {
    WorldHitIO io{rays, tmax_per_ray, out, tmin, tmax};
    trace_batch<COUNT, true, PARK, WIDE, XF, KINDS, false>(sv, io, n, counters);
}
struct WorldHitSurfaceKernels {
    template <bool COUNT, bool PARK, int WIDE, bool XF = true, int KINDS = 0>
    static auto get() { return k_world_hit_surface<COUNT, PARK, WIDE, XF, KINDS>; }
};
void launch_world_hit_surface(const SceneView& sv, const rt_ray* d_rays, const double* d_tmax_per_ray, uint32_t n, double tmin, double tmax, bool count,
                              HitRec* d_out, unsigned long long* d_counters, int grid, size_t stack_bytes, cudaStream_t stream) {
    launch_with_l2_window(batch_variant<WorldHitSurfaceKernels>(sv, count), sv, grid, EXTEND_BLOCK, stack_bytes, stream, sv, d_rays, d_tmax_per_ray,
                          n, tmin, tmax, d_out, d_counters);
}

// rt_shade: the step of ray_color after world.hit (camera.rs:288-321) for a batch of rt_hit_records, one row per thread, the
// general instantiation of the render's step (shade_hit<SC_OTHER> + end_segment) with the draws philox(seed; pixel = i,
// sample = 0, segment, slot).  contribute() adds to radiance + 3 i.  Defined after the render kernels, as the world-hit family.
__global__ void __launch_bounds__(SHADE_BLOCK, shade_blocks(SC_OTHER, false))
    k_shade_records(SceneView sv, RenderParams P, const rt_hit_record* __restrict__ records, uint64_t n, uint32_t n_materials, uint32_t segment,
                    rt_ray* __restrict__ rays, double* __restrict__ beta, double* __restrict__ radiance, uint8_t* __restrict__ state,
                    unsigned long long* n_errors) {
    // contribute() and end_segment() count errors at &W.counters->errors: that is this thread's own word of s_errors (address
    // arithmetic on integers, as tests/device_kat.cu does), so that a row knows whether its segment added one
    __shared__ unsigned long long s_errors[SHADE_BLOCK];
    WavefrontState W{};
    W.accum = radiance;
    W.counters = reinterpret_cast<Counters*>(reinterpret_cast<uintptr_t>(s_errors + threadIdx.x) - offsetof(Counters, errors));
    unsigned long long errors = 0;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        if (!(state[i] & RT_PATH_ALIVE)) continue;  // an inactive row: nothing else of it is read or written
        s_errors[threadIdx.x] = 0;
        const uint32_t pixel = (uint32_t)i;
        const double* rp = reinterpret_cast<const double*>(rays + i);
        RayD r;
        r.o = D3{rp[0], rp[1], rp[2]};
        r.d = D3{rp[3], rp[4], rp[5]};
        r.time = rp[6];
        const D3 b = ld3(beta + 3 * i);
        const rt_hit_record& rec = records[i];
        const uint32_t kind = rec.kind;
        RayD nr = r;
        D3 nbeta = b;
        bool alive = false, error = false;
        if (kind > RT_HIT_MEDIUM || (kind != RT_HIT_MISS && rec.material >= n_materials)) {
            error = true;  // a malformed record (it comes from outside the library): nothing of it is used
        } else if (kind == RT_HIT_MISS) {
            D3 bg;
            if (background_value(sv, P.cam.background_tex, r.d, bg))
                contribute(P, W, pixel, b * bg);
            else
                error = true;
        } else {
            HitInfo h;
            h.p = ld3(rec.p);
            h.normal = ld3(rec.normal);
            h.u = rec.u, h.v = rec.v;
            h.front_face = rec.front_face != 0;
            h.material = rec.material;
            // shade_one's hit_ok is what surface_hit_info / hit_to_world return: true without a Transform; under one, false iff
            // some Transform of the chain left a normal unit_vector could not make finite.  A non-finite normal stays non-finite
            // through the rest of the chain (scaling and rotating keep an inf or NaN component), and a chain of finite steps ends
            // finite, so the record's normal tells it exactly.
            const bool hit_ok = rec.inst_id == RT_NONE || finite3(h.normal);
            shade_hit<SC_OTHER>(sv, P, W, r, b, pixel, 0u, segment, h, hit_ok, nr, nbeta, alive, error, nullptr);
        }
        alive = end_segment(P, W, segment, alive, error, nbeta);
        const bool err = s_errors[threadIdx.x] != 0;  // a panic, or a NaN contribution contribute() dropped
        errors += err ? 1u : 0u;
        if (alive) {
            double* wp = reinterpret_cast<double*>(rays + i);
            wp[0] = nr.o.x, wp[1] = nr.o.y, wp[2] = nr.o.z;
            wp[3] = nr.d.x, wp[4] = nr.d.y, wp[5] = nr.d.z;
            wp[6] = nr.time;
            beta[3 * i + 0] = nbeta.x, beta[3 * i + 1] = nbeta.y, beta[3 * i + 2] = nbeta.z;
        }
        state[i] = (uint8_t)((alive ? RT_PATH_ALIVE : 0u) | (err ? RT_PATH_ERROR : 0u));
    }
    if (errors && n_errors) atomicAdd(n_errors, errors);
}
void launch_shade_records(const SceneView& sv, const RenderParams& P, const rt_hit_record* d_records, uint64_t n, uint32_t n_materials,
                          uint32_t segment, rt_ray* d_rays, double* d_beta, double* d_radiance, uint8_t* d_state, unsigned long long* d_errors,
                          int grid, cudaStream_t s) {
    k_shade_records<<<grid, SHADE_BLOCK, 0, s>>>(sv, P, d_records, n, n_materials, segment, d_rays, d_beta, d_radiance, d_state, d_errors);
}

// rt_camera_rays: Camera::get_ray of stratum `sample` through every pixel, k_generate's camera_ray, in the render's pixel order
__global__ void __launch_bounds__(256) k_camera_rays(rt_camera cam, uint64_t seed, uint32_t sample, uint64_t n, rt_ray* __restrict__ out) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        RayD r;
        camera_ray(cam, seed, (uint32_t)i, sample, r);
        double* wp = reinterpret_cast<double*>(out + i);
        wp[0] = r.o.x, wp[1] = r.o.y, wp[2] = r.o.z;
        wp[3] = r.d.x, wp[4] = r.d.y, wp[5] = r.d.z;
        wp[6] = r.time;
    }
}
void launch_camera_rays(const rt_camera& cam, uint64_t seed, uint32_t sample, uint64_t n, rt_ray* d_out, int grid, cudaStream_t s) {
    k_camera_rays<<<grid, 256, 0, s>>>(cam, seed, sample, n, d_out);
}

int kernel_setup(size_t smem_bytes, int* extend_blocks_per_sm, int* shade_blocks_per_sm, int* walk_blocks_per_sm) {
    // dynamic shared memory above 48 KB is opt-in
    cudaError_t e = cudaSuccess;
    const void* big_smem[] = {
#define RT_EXTEND_VARIANTS(M)                                                                                                     \
    (const void*)k_extend<false, false, 0, M>, (const void*)k_extend<false, true, 0, M>, (const void*)k_extend<false, true, 1, M>, \
        (const void*)k_extend<false, true, 2, M>, (const void*)k_extend<true, false, 0, M>, (const void*)k_extend<true, true, 0, M>, \
        (const void*)k_extend<true, true, 1, M>, (const void*)k_extend<true, true, 2, M>, (const void*)k_extend<false, false, 3, M>, \
        (const void*)k_extend<true, false, 3, M>
        RT_EXTEND_VARIANTS(0), RT_EXTEND_VARIANTS(1), RT_EXTEND_VARIANTS(2), RT_EXTEND_VARIANTS(3),
#undef RT_EXTEND_VARIANTS
        RT_BATCH_VARIANTS(k_closest_hit), RT_BATCH_VARIANTS(k_occluded), RT_BATCH_VARIANTS(k_world_hit_surface)};
    for (const void* f : big_smem)
        if ((e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(EXTEND_SMEM_MAX - 1024))) != cudaSuccess) return (int)e;
    // the general-boundary media pass: TRAVERSAL_STACK entries per thread is 64 KB
    if ((e = cudaFuncSetAttribute((const void*)k_tail, cudaFuncAttributeMaxDynamicSharedMemorySize, TRAVERSAL_STACK * TAIL_BLOCK * (int)sizeof(uint32_t))) != cudaSuccess) return (int)e;
    for (const void* f : {(const void*)k_walk<false, false>, (const void*)k_walk<true, false>, (const void*)k_walk<false, true>, (const void*)k_walk<true, true>})
        if ((e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, TRAVERSAL_STACK * WALK_BLOCK * (int)sizeof(uint32_t))) != cudaSuccess) return (int)e;
    const void* media_smem[] = {(const void*)k_media<false, 2, false, false>, (const void*)k_media<false, 2, true, false>,
                                (const void*)k_media<true, 2, false, false>, (const void*)k_media<true, 2, true, false>,
                                (const void*)k_transmittance<false, true, false>, (const void*)k_transmittance<false, true, true>,
                                (const void*)k_transmittance<true, true, false>, (const void*)k_transmittance<true, true, true>,
                                (const void*)k_world_hit_record<false, true, false>, (const void*)k_world_hit_record<false, true, true>,
                                (const void*)k_world_hit_record<true, true, false>, (const void*)k_world_hit_record<true, true, true>};
    for (const void* f : media_smem)
        if ((e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, TRAVERSAL_STACK * MEDIA_BLOCK * (int)sizeof(uint32_t))) != cudaSuccess) return (int)e;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(extend_blocks_per_sm, k_extend<false, false, 0, 0>, EXTEND_BLOCK, smem_bytes);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(shade_blocks_per_sm, k_shade<SC_OTHER>, SHADE_BLOCK, 0);  // a class never compiled for three
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(walk_blocks_per_sm, k_walk<true, false>, WALK_BLOCK, 24 * WALK_BLOCK * sizeof(uint32_t));
    return 0;
}

}  // namespace rt
