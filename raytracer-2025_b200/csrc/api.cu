// api.cu — the extern "C" boundary (include/rt2025.h): scene upload, the wavefront driver loop,
// closest-hit batches, tone mapping.  No C++ exception leaves this file.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "compile.h"
#include "kernels.h"
#include "rt2025.h"

using namespace rt;

namespace {

thread_local std::string g_err;

int set_err(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define CU(call)                                                                                              \
    do {                                                                                                      \
        cudaError_t e_ = (call);                                                                              \
        if (e_ != cudaSuccess) {                                                                              \
            throw CudaFail{std::string(#call) + ": " + cudaGetErrorString(e_)};                               \
        }                                                                                                     \
    } while (0)

struct CudaFail {
    std::string what;
};

// All tables of a scene live in ONE stream-ordered allocation (cudaMallocAsync: freed blocks stay in the
// device's pool, so a client that builds a scene per frame - Camera::render does - pays no driver call
// after the first frame; a dozen cudaMalloc/cudaFree pairs per scene cost 10-50 ms with visible jitter).
struct Arena {
    char* base = nullptr;
    size_t size = 0, used = 0;
    template <class V>
    size_t reserve(const V& v) {
        size = (size + 255) & ~size_t(255);
        const size_t at = size;
        size += v.size() * sizeof(typename V::value_type);
        return at;
    }
    void allocate(cudaStream_t st) {
        size = (size + 255) & ~size_t(255);
        if (size) CU(cudaMallocAsync((void**)&base, size, st));
    }
    template <class V, class T = typename V::value_type>
    T* put(const V& v, cudaStream_t st) {
        used = (used + 255) & ~size_t(255);
        if (v.empty()) return nullptr;
        T* d = reinterpret_cast<T*>(base + used);
        CU(cudaMemcpyAsync(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, st));
        used += v.size() * sizeof(T);
        return d;
    }
};

void keep_pool_memory(int device) {  // once per device: the default pool keeps up to 1 GiB of freed blocks
    static std::mutex mu;
    static std::vector<int> done;
    std::lock_guard<std::mutex> lock(mu);
    if (std::find(done.begin(), done.end(), device) != done.end()) return;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        uint64_t threshold = 1ull << 30;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold);
    }
    cudaGetLastError();
    done.push_back(device);
}

// short-lived device buffers of the host-pointer entry points: stream-ordered (default stream), pooled
template <class T>
void scratch_alloc(T** p, size_t bytes) { CU(cudaMallocAsync((void**)p, bytes, nullptr)); }
inline void scratch_free(void* p) {
    if (p) cudaFreeAsync(p, nullptr);
}

// Entry points select the scene's device; the caller's current device is put back on return (the library is
// meant to sit next to torch or another CUDA client in one process).
struct DeviceGuard {
    int prev = -1;
    DeviceGuard() {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        cudaGetLastError();
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// scenes that hold a persisting-L2 window, per device: the carve-out is handed back when the last one dies
std::mutex g_l2_mu;
int g_l2_users[64] = {};

struct Workspace {  // wavefront buffers, cached on the scene between renders
    WavefrontState W{};
    uint32_t capacity = 0;
    uint64_t n_pixels_alloc = 0;
    Counters* h_counters = nullptr;  // pinned, two copies (pipelined read-back)
    cudaEvent_t check_ev[2] = {nullptr, nullptr};
    std::vector<cudaEvent_t> events;  // stage-timing pool: 4 per iteration, read back after the render
    ShadeFan fan;                     // side streams of the shade stage
    bool fan_ready = false;
    const ShadeFan* shade_fan() {
        if (!fan_ready) {
            fan_ready = true;
            int n = RT_SHADE_SIDE_STREAMS;
            if (const char* e = getenv("RT2025_SHADE_STREAMS")) n = std::max(0, std::min(3, atoi(e)));  // tuning knob
            bool ok = cudaEventCreateWithFlags(&fan.fork, cudaEventDisableTiming) == cudaSuccess;
            for (int i = 0; i < n && ok; i++)
                ok = cudaStreamCreateWithFlags(&fan.side[i], cudaStreamNonBlocking) == cudaSuccess &&
                     cudaEventCreateWithFlags(&fan.join[i], cudaEventDisableTiming) == cudaSuccess;
            fan.n_side = ok ? n : 0;
            cudaGetLastError();
        }
        return &fan;
    }
    cudaEvent_t check_event(int slot) {
        if (!check_ev[slot]) cudaEventCreateWithFlags(&check_ev[slot], cudaEventDisableTiming);
        return check_ev[slot];
    }
    cudaEvent_t event(size_t i) {
        while (events.size() <= i) {
            cudaEvent_t e;
            if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
            events.push_back(e);
        }
        return events[i];
    }
    void release() {
        for (auto e : events) cudaEventDestroy(e);
        events.clear();
        for (auto& e : check_ev)
            if (e) cudaEventDestroy(e);
        if (fan.fork) cudaEventDestroy(fan.fork);
        for (int i = 0; i < 3; i++) {
            if (fan.side[i]) cudaStreamDestroy(fan.side[i]);
            if (fan.join[i]) cudaEventDestroy(fan.join[i]);
        }
        for (int k = 0; k < 2; k++) cudaFree(W.ray_q[k]), cudaFree(W.beta_q[k]);
        cudaFree(W.hit_q);
        cudaFree(W.cls_q);
        for (auto& q : W.q_shade) cudaFree(q);
        cudaFree(W.pixel_list);
        cudaFree(W.accum);
        cudaFree(W.counters);
        if (h_counters) cudaFreeHost(h_counters);
        *this = Workspace();
    }
};

}  // namespace

// Wavefront workspaces are pooled per device and shared by all scenes of the process: re-creating a scene (what
// Camera::render does on every call) must not re-allocate half a gigabyte.  A render borrows a free workspace for its
// duration; a second render on the same GPU at the same time (another scene, another host thread) gets one of its own
// instead of queueing behind the first.
namespace {
struct DeviceWorkspace {
    std::mutex mu;
    std::vector<std::unique_ptr<Workspace>> all;
    std::vector<Workspace*> free_list;
};
DeviceWorkspace& device_workspace(int device) {
    static DeviceWorkspace pool[64];
    return pool[device & 63];
}
struct WorkspaceLease {
    DeviceWorkspace& d;
    Workspace* ws = nullptr;
    explicit WorkspaceLease(DeviceWorkspace& dws) : d(dws) {
        std::lock_guard<std::mutex> lock(d.mu);
        if (d.free_list.empty()) {
            d.all.emplace_back(new Workspace());
            ws = d.all.back().get();
        } else {  // the largest one first: it is the least likely to need growing
            auto it = std::max_element(d.free_list.begin(), d.free_list.end(), [](Workspace* a, Workspace* b) { return a->capacity < b->capacity; });
            ws = *it;
            d.free_list.erase(it);
        }
    }
    ~WorkspaceLease() {
        std::lock_guard<std::mutex> lock(d.mu);
        d.free_list.push_back(ws);
    }
};
}  // namespace

struct rt_scene {
    int device = 0;
    int sm_count = 148;
    SceneView view{};
    void* arena = nullptr;  // one stream-ordered allocation holding every table of the view
    std::vector<uint32_t> ranks;
    rt_scene_info info{};
    uint32_t lights_flat = 1;
    uint32_t class_mask = 0;     // shade classes the scene's materials can produce
    bool generic_media = false;  // some ConstantMedium boundary is not a single Sphere
    std::vector<uint8_t> black_texture;  // per texture: a solid colour (0, 0, 0) - a miss against such a background contributes nothing
    int extend_blocks_per_sm = 4, shade_blocks_per_sm = 4, walk_blocks_per_sm = 1;
    size_t stack_bytes = 0;  // dynamic shared memory of the traversal kernels: cached nodes + stacks
};

namespace {

int check_device(int requested, int& device, int& sm_count) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return set_err(RT_ERR_NO_DEVICE, "no CUDA device available: librt2025 has no CPU path");
    }
    if (requested >= 0) {
        if (requested >= n) return set_err(RT_ERR_INVALID, "device ordinal out of range");
        if (cudaSetDevice(requested) != cudaSuccess) return set_err(RT_ERR_CUDA, "cudaSetDevice failed");
    }
    cudaGetDevice(&device);
    // cudaGetDeviceProperties costs 5-45 ms per call on this platform (it was most of rt_tonemap and a third of
    // rt_scene_create): three attributes, asked once per device
    struct Cached {
        int major = -1, minor = 0, sms = 0;
    };
    static std::mutex mu;
    static std::vector<Cached> cache;
    std::lock_guard<std::mutex> lock(mu);
    if ((int)cache.size() <= device) cache.resize(device + 1);
    Cached& c = cache[device];
    if (c.major < 0) {
        int major = 0, minor = 0, sms = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device) != cudaSuccess ||
            cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device) != cudaSuccess ||
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess)
            return set_err(RT_ERR_CUDA, "cudaDeviceGetAttribute failed");
        c.major = major, c.minor = minor, c.sms = sms;
    }
    if (c.major != 10)
        return set_err(RT_ERR_NO_DEVICE, std::string("built for sm_100a only; device is sm_") + std::to_string(c.major) + std::to_string(c.minor));
    sm_count = c.sms;
    return RT_OK;
}

// The batch limit of the ray queries and rt_shade, checked before anything is allocated or copied
static int batch_refusal(uint64_t n) {
    return n > 0xFFFFFFF0ull ? set_err(RT_ERR_INVALID, "more than 2^32 - 16 rays in one batch") : RT_OK;
}

// The body of the _device batch queries: the batch size check, RT_OPT_COUNT counters, event timing and `stats`.
// launch(count, d_counters, grid, stream) enqueues the kernels and returns how many it launched.
template <class Launch>
int run_batch(const rt_scene* s, uint64_t n, uint32_t flags, void* stream, rt_stats* stats, Launch launch) {
    if (stats) std::memset(stats, 0, sizeof(*stats));
    if (n == 0) return RT_OK;
    if (const int refused = batch_refusal(n)) return refused;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long* d_cnt = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    int rc = RT_OK;
    DeviceGuard guard;
    try {
        CU(cudaSetDevice(s->device));
        // counters are only read back through `stats`: without it the kernel runs the uncounted instantiation.
        // The buffer is allocated and freed in stream order on the caller's stream, like the kernel that writes it.
        const bool count = (flags & RT_OPT_COUNT) != 0 && stats != nullptr;
        if (count) {
            CU(cudaMallocAsync((void**)&d_cnt, 2 * sizeof(unsigned long long), st));
            CU(cudaMemsetAsync(d_cnt, 0, 2 * sizeof(unsigned long long), st));
        }
        int grid = s->sm_count * s->extend_blocks_per_sm;
        uint64_t need = (n + EXTEND_BLOCK - 1) / EXTEND_BLOCK;
        if ((uint64_t)grid > need) grid = (int)need;
        if (stats) {
            CU(cudaEventCreate(&e0));
            CU(cudaEventCreate(&e1));
            CU(cudaEventRecord(e0, st));
        }
        const int launches = launch(count, d_cnt, grid, st);
        CU(cudaGetLastError());
        if (stats) {
            CU(cudaEventRecord(e1, st));
            CU(cudaEventSynchronize(e1));
            float ms = 0;
            CU(cudaEventElapsedTime(&ms, e0, e1));
            stats->ms_total = ms;
            stats->ms_extend = ms;
            stats->segments = n;
            stats->kernel_launches = launches;
            if (count) {
                unsigned long long h[2];
                CU(cudaMemcpyAsync(h, d_cnt, sizeof(h), cudaMemcpyDeviceToHost, st));
                CU(cudaStreamSynchronize(st));
                stats->node_visits = h[0], stats->prim_tests = h[1];
            }
        }
    } catch (const CudaFail& f) {
        rc = set_err(RT_ERR_CUDA, f.what);
    }
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    if (d_cnt) cudaFreeAsync(d_cnt, st);
    return rc;
}

}  // namespace

extern "C" {

const char* rt_last_error(void) { return g_err.c_str(); }
uint32_t rt_abi_version(void) { return RT_ABI_VERSION; }
int rt_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int rt_scene_create(const rt_scene_desc* desc, const rt_build_opts* opts, rt_scene** out) {
    if (!desc || !out) return set_err(RT_ERR_INVALID, "null argument");
    *out = nullptr;
    rt_scene* s = nullptr;
    DeviceGuard guard;
    try {
        CompiledScene cs;
        std::string err;
        uint32_t flags = opts ? opts->flags : 0;
        int device = 0, sms = 0;
        int rc = RT_OK;
        const bool device_build = (flags & RT_BUILD_DEVICE_LBVH) != 0;
        if (device_build) {  // the builder runs on the scene's device: select it before compiling
            rc = check_device(opts ? opts->device : -1, device, sms);
            if (rc != RT_OK) return rc;
        }
        rc = compile_scene(*desc, flags, cs, err, device_build ? build_bvh_device : nullptr);
        if (rc != RT_OK) return set_err(rc, err);
        if (!device_build) {
            rc = check_device(opts ? opts->device : -1, device, sms);
            if (rc != RT_OK) return rc;
        }
        {
            // a small scene's four-wide collapse is only used when all of it fits in a traversal CTA's shared memory next to the
            // stacks (compile.cpp); otherwise its binary tree is traversed, which then fits
            const size_t budget = EXTEND_SMEM_MAX / EXTEND_MIN_BLOCKS - 1024;
            const size_t stacks = (size_t)std::min<uint32_t>(std::max(cs.bvh_depth + 2, 3 * cs.bvh4_depth + 2), TRAVERSAL_STACK) * EXTEND_BLOCK * sizeof(uint32_t) + EXTEND_RAY_SMEM_BYTES;
            if (!cs.nodes4.empty() && cs.nodes.size() * sizeof(Node) <= 2 * budget && stacks + cs.nodes4.size() * sizeof(Node4) > budget &&
                !getenv("RT2025_WIDE_BVH")) {
                RawVec<Node4>().swap(cs.nodes4);
                cs.world_root4 = INVALID_REF;
            }
        }
        s = new rt_scene();
        s->device = device;
        s->sm_count = sms;
        SceneView& v = s->view;
        keep_pool_memory(device);
        {
            cudaStream_t st = cudaStreamPerThread;
            Arena a;
            a.reserve(cs.nodes4), a.reserve(cs.nodes), a.reserve(cs.geom), a.reserve(cs.meta), a.reserve(cs.xforms), a.reserve(cs.materials), a.reserve(cs.textures);
            a.reserve(cs.images), a.reserve(cs.texels), a.reserve(cs.perlins), a.reserve(cs.media), a.reserve(cs.lights), a.reserve(cs.remaps), a.reserve(cs.walk_lean), a.reserve(cs.shade_lean);
            a.allocate(st);
            s->arena = a.base;
            v.nodes4 = a.put(cs.nodes4, st), v.world_root4 = cs.world_root4;
            v.nodes = a.put(cs.nodes, st), v.geom = a.put(cs.geom, st), v.meta = a.put(cs.meta, st), v.xforms = a.put(cs.xforms, st);
            v.materials = a.put(cs.materials, st), v.textures = a.put(cs.textures, st), v.images = a.put(cs.images, st);
            v.texels = a.put(cs.texels, st), v.perlins = a.put(cs.perlins, st), v.media = a.put(cs.media, st);
            v.lights = a.put(cs.lights, st), v.remaps = a.put(cs.remaps, st), v.walk_lean = a.put(cs.walk_lean, st);
            v.shade_lean = a.put(cs.shade_lean, st), v.shade_lean_mask = cs.shade_lean_mask;
            CU(cudaStreamSynchronize(st));  // the host vectors die with this call
        }
        v.world_root = cs.world_root;
        v.n_media = (uint32_t)cs.media.size();
        v.n_xforms = (uint32_t)cs.xforms.size();
        v.kinds = (cs.n_spheres && !cs.n_planars) ? 1u : ((cs.n_planars && !cs.n_spheres) ? 2u : 0u);
        v.n_lights = (uint32_t)cs.lights.size();
        v.n_prims = (uint32_t)cs.geom.size();
        v.moving = 0;
        for (size_t p = 0; p < cs.geom.size(); p++)
            if ((cs.meta[p].kind_mat >> 30) == PRIM_SPHERE && (cs.geom[p].d[3] != 0.0 || cs.geom[p].d[4] != 0.0 || cs.geom[p].d[5] != 0.0)) v.moving = 1;
        s->ranks = cs.ranks;
        for (auto& m : cs.media) s->generic_media |= m.single_sphere == RT_NONE;
        v.media_xform = 0;
        for (auto& m : cs.media)
            if (m.xform != RT_NONE || (m.single_sphere != RT_NONE && cs.meta[m.single_sphere].xform != RT_NONE)) v.media_xform = 1;
        for (auto& m : cs.materials) s->class_mask |= 1u << m.shade_class;
        for (auto& t : cs.textures) s->black_texture.push_back(t.kind == RT_TEX_SOLID && t.color[0] == 0.0 && t.color[1] == 0.0 && t.color[2] == 0.0);
        uint32_t n_thick = 0, n_thick_entries = 0;
        for (auto& m : cs.media)
            if (m.flags & MEDIUM_THICK) s->class_mask |= 1u << SC_WALK, n_thick++, n_thick_entries += m.n_entry != MEDIUM_NO_ENTRIES;
        v.walk_entries_only = n_thick == 1 && n_thick_entries == 1;  // scatter points of thick media go to the random-walk kernel
        // lights is "flat" when every leaf has the same weight 1/n (a single-level list)
        s->lights_flat = 1;
        for (auto& l : cs.lights)
            if (l.weight != 1.0 / (double)cs.lights.size()) s->lights_flat = 0;
        rt_scene_info& i = s->info;
        i.n_prims = v.n_prims, i.n_spheres = cs.n_spheres, i.n_planars = cs.n_planars, i.n_nodes = (uint32_t)cs.nodes.size();
        i.n_media = v.n_media, i.n_lights = v.n_lights, i.n_materials = (uint32_t)cs.materials.size(), i.n_textures = (uint32_t)cs.textures.size();
        i.bvh_depth = cs.bvh_depth;
        i.node_bytes = cs.nodes4.empty() ? (uint32_t)sizeof(Node) : (uint32_t)sizeof(Node4);
        i.device_bytes = cs.nodes.size() * sizeof(Node) + cs.nodes4.size() * sizeof(Node4) + cs.geom.size() * sizeof(PrimGeom) +
                         cs.meta.size() * sizeof(PrimMeta) + cs.texels.size() * sizeof(float4) + cs.perlins.size() * sizeof(Perlin);
        // shared memory of the traversal kernels: per-thread stacks sized by this scene's tree depth,
        // the rest (up to 227 KB) holds the breadth-first top of the BVH
        v.n_nodes = (uint32_t)cs.nodes.size();
        // the binary tree pushes one reference per level, the four-wide one up to three (compile.cpp keeps it within the limit)
        v.stack_entries = std::min<uint32_t>(std::max(cs.bvh_depth + 2, cs.nodes4.empty() ? 0u : 3 * cs.bvh4_depth + 2), TRAVERSAL_STACK);
        v.media_stack_entries = std::min<uint32_t>(cs.media_bvh_depth + 2, TRAVERSAL_STACK);
        v.tail_stack_entries = std::min<uint32_t>(std::max(cs.bvh_depth, cs.media_bvh_depth) + 2, TRAVERSAL_STACK);  // the media kernel walks boundary groups only
        const size_t stack_bytes = (size_t)v.stack_entries * EXTEND_BLOCK * sizeof(uint32_t) + EXTEND_RAY_SMEM_BYTES;  // (+ the rays, behind the FIFOs)
        // persistent traversal: a warp whose BVH lives in L1/shared memory is issue-bound and runs best when it
        // drains completely before taking 32 new rays; once node fetches go to L2/HBM the idle lanes are worth
        // more as loads in flight and every finished lane is refilled at once (profiles/README.md: 1M-triangle
        // soup, incoherent rays, 392 vs 274 Mrays/s; book2_final 49.4 vs 48.7 ms the other way round)
        v.refill_min = cs.nodes.size() > 100000 ? 1 : 16;  // FIFO mode: idle lanes a warp collects before it pops (sweeps in profiles/README.md)
        // scenes that do not fit the L2: pin the top of the tree (kernels.cu, launch_with_l2_window)
        v.l2_window_bytes = 0;
        {
            // bytes of the tree the traversal kernels actually read (the four-wide collapse when there is one)
            const size_t tree_bytes = cs.nodes4.empty() ? cs.nodes.size() * sizeof(Node) : cs.nodes4.size() * sizeof(Node4);
            const size_t scene_bytes = tree_bytes + cs.geom.size() * (sizeof(PrimGeom) + sizeof(PrimMeta));
            int l2 = 0, max_persist = 0, max_window = 0;
            cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, device);
            cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, device);
            cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, device);
            size_t want = 0;
            if (const char* e = getenv("RT2025_L2_WINDOW_MB")) want = (size_t)atol(e) << 20;  // tuning knob (0 disables)
            // measured (profiles/README.md): a window that holds the WHOLE node array helps incoherent rays (1M-triangle
            // soup 392 -> 416 Mrays/s, primary unchanged); a partial window over a bigger tree gains 2-5 % on incoherent
            // rays and costs coherent ones up to 15 % (10M soup, 79 MB window), so it is only set when everything fits
            else if (scene_bytes > (size_t)l2 && tree_bytes <= (size_t)max_persist) want = tree_bytes;
            want = std::min({want, (size_t)max_persist, (size_t)max_window, tree_bytes});
            if (want >= (1u << 20)) {
                std::lock_guard<std::mutex> lock(g_l2_mu);
                size_t have = 0;
                cudaDeviceGetLimit(&have, cudaLimitPersistingL2CacheSize);
                // never shrink a carve-out another live scene (or the host framework) asked for
                if (have >= want || cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) == cudaSuccess) {
                    v.l2_window_bytes = (uint32_t)want;
                    g_l2_users[device & 63]++;
                }
                cudaGetLastError();
            }
            if (getenv("RT2025_TIMING")) fprintf(stderr, "[rt2025] L2 %d MB, max persisting %d MB, max window %d MB, scene %zu MB -> window %u MB\n",
                                                 l2 >> 20, max_persist >> 20, max_window >> 20, scene_bytes >> 20, v.l2_window_bytes >> 20);
        }
        // postponed leaves pay off when traversals are long (traverse.cuh); measured crossover between the 3.2 k-node
        // book-2 scene (off: extend 281 vs 299 ms) and the 11.5 k-face mesh scene (on: 487 vs 502 ms)
        v.park_leaves = cs.nodes.size() > 4096 ? 1 : 0;
        if (const char* e = getenv("RT2025_PARK_LEAVES")) v.park_leaves = atoi(e) != 0;  // tuning knob
        if (const char* e = getenv("RT2025_REFILL_MIN")) v.refill_min = (uint32_t)std::min(32l, std::max(1l, atol(e)));  // tuning knob
        // shared memory of a traversal CTA: [cached nodes | stacks | per-warp FIFOs of prepared rays].  The FIFOs come first
        // (64 slots per warp when they fit next to the stacks, else 32), the node cache gets what is left.
        const size_t budget = EXTEND_SMEM_MAX / EXTEND_MIN_BLOCKS - 1024;
        auto fifo_bytes = [](uint32_t slots) { return (size_t)(EXTEND_BLOCK / 32) * slots * 28 * sizeof(uint32_t); };
        v.fifo_slots = stack_bytes + fifo_bytes(64) <= budget ? 64u : 32u;
        // Cache-resident trees keep the round-1 scheme (fifo_slots = 0: a warp takes 32 rays, drains, takes 32 more; the
        // shared memory holds the tree instead).  Measured, extend ms per frame, direct vs FIFO: book2_final (3201 nodes)
        // 40.8 vs 45.9, book1_final 33.5 vs 34.8, cornell 29.0 vs 28.5; trees far beyond shared memory gain from the
        // per-lane refill: the 76 k-node mesh scene 69.6 (drained) vs 61.8, the 1 M soups +12..24 % in Mrays/s.
        if (cs.nodes.size() * sizeof(Node) <= 2 * budget) v.fifo_slots = 0;
        if (const char* e = getenv("RT2025_FIFO_SLOTS")) v.fifo_slots = atoi(e) >= 64 ? 64u : (atoi(e) >= 32 ? 32u : 0u);  // tuning knob
        // a four-wide tree is either all in shared memory (direct mode) or all in global memory and fed from the FIFOs: the kernels
        // have no other four-wide variant
        const bool wide_in_smem = !cs.nodes4.empty() && v.fifo_slots == 0 && stack_bytes + cs.nodes4.size() * sizeof(Node4) + 16 <= budget &&
                                  !(getenv("RT2025_SMEM_NODES_KB") && (size_t)atol(getenv("RT2025_SMEM_NODES_KB")) * 1024 < cs.nodes4.size() * sizeof(Node4));
        if (!cs.nodes4.empty() && !wide_in_smem && v.fifo_slots == 0) v.fifo_slots = 32;
        if (stack_bytes + fifo_bytes(v.fifo_slots) > budget) throw CudaFail{"traversal stacks and ray FIFOs do not fit in shared memory"};
        const size_t room = budget - stack_bytes - fifo_bytes(v.fifo_slots);
        size_t cache_bytes = room;
        if (const char* e = getenv("RT2025_SMEM_NODES_KB")) cache_bytes = std::min<size_t>(room, (size_t)atol(e) * 1024);  // tuning knob
        // the persistent traversal reads ONE tree: the four-wide collapse when there is one (n_cached_nodes then counts Node4)
        const size_t node_size = cs.nodes4.empty() ? 56 : sizeof(Node4);  // traverse.cuh: binary nodes are stored compact (SMEM_NODE_BYTES)
        const size_t tree_nodes = cs.nodes4.empty() ? cs.nodes.size() : cs.nodes4.size();
        v.n_cached_nodes = (uint32_t)std::min<size_t>(tree_nodes, (cache_bytes >= 16 ? cache_bytes - 16 : 0) / node_size);  // (the region is rounded up to 16 bytes)
        // A four-wide tree is only staged when ALL of it fits (RT2025_WIDE_BVH=1 on a book-sized scene): staging the top of a tree
        // that lives in L2 takes the shared memory away from the L1 and buys nothing (measured with the binary top in round 2:
        // synthetic mesh scene extend 30.1 -> 26.8 ms, 1 M-triangle soup +3 % Mrays/s without it)
        if (!cs.nodes4.empty()) v.n_cached_nodes = wide_in_smem ? (uint32_t)tree_nodes : 0u;
        s->stack_bytes = stack_bytes + fifo_bytes(v.fifo_slots) + (((size_t)v.n_cached_nodes * node_size + 15) & ~(size_t)15);
        if (kernel_setup(s->stack_bytes, &s->extend_blocks_per_sm, &s->shade_blocks_per_sm, &s->walk_blocks_per_sm) != 0)
            throw CudaFail{"cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed"};
        if (s->extend_blocks_per_sm < 1) s->extend_blocks_per_sm = 1;
        if (s->shade_blocks_per_sm < 1) s->shade_blocks_per_sm = 1;
        if (s->walk_blocks_per_sm < 1) s->walk_blocks_per_sm = 1;
        if (const char* e = getenv("RT2025_WALK_BLOCKS")) s->walk_blocks_per_sm = std::max(1, std::min(s->walk_blocks_per_sm, atoi(e)));  // tuning knob
        CU(cudaDeviceSynchronize());
        *out = s;
        return RT_OK;
    } catch (const CudaFail& f) {
        if (s) rt_scene_destroy(s);
        return set_err(RT_ERR_CUDA, f.what);
    } catch (const std::bad_alloc&) {
        if (s) rt_scene_destroy(s);
        return set_err(RT_ERR_OOM, "out of host memory");
    } catch (...) {
        if (s) rt_scene_destroy(s);
        return set_err(RT_ERR_INVALID, "unexpected failure in rt_scene_create");
    }
}

int rt_scene_destroy(rt_scene* s) {
    if (!s) return RT_OK;
    DeviceGuard guard;
    cudaSetDevice(s->device);
    if (s->arena) {
        cudaDeviceSynchronize();  // renders of this scene may still be in flight on caller streams
        if (s->view.l2_window_bytes) {
            std::lock_guard<std::mutex> lock(g_l2_mu);
            // hand the pinned lines back to ordinary traffic once no scene of this process uses a window on the device
            if (--g_l2_users[s->device & 63] == 0) cudaCtxResetPersistingL2Cache();
        }
        cudaFreeAsync(s->arena, cudaStreamPerThread);
    }
    delete s;
    return RT_OK;
}

int rt_scene_get_info(const rt_scene* s, rt_scene_info* info) {
    if (!s || !info) return set_err(RT_ERR_INVALID, "null argument");
    *info = s->info;
    return RT_OK;
}

int rt_scene_get_ranks(const rt_scene* s, uint32_t* ranks, uint32_t n) {
    if (!s || !ranks) return set_err(RT_ERR_INVALID, "null argument");
    if (n != s->ranks.size()) return set_err(RT_ERR_INVALID, "n_objects mismatch");
    std::copy(s->ranks.begin(), s->ranks.end(), ranks);
    return RT_OK;
}

int rt_closest_hit_device(const rt_scene* s, const rt_ray* d_rays, uint64_t n, double t_min, double t_max, uint32_t flags,
                          rt_hit* d_out, void* stream, rt_stats* stats) {
    if (!s || (n && (!d_rays || !d_out))) return set_err(RT_ERR_INVALID, "null argument");
    return run_batch(s, n, flags, stream, stats, [&](bool count, unsigned long long* d_cnt, int grid, cudaStream_t st) {
        launch_closest_hit(s->view, d_rays, (uint32_t)n, t_min, t_max, count, d_out, d_cnt, grid, s->stack_bytes, st);
        return 1;
    });
}

int rt_closest_hit(const rt_scene* s, const rt_ray* rays, uint64_t n, double t_min, double t_max, uint32_t flags, rt_hit* out,
                   rt_stats* stats) {
    if (!s || (n && (!rays || !out))) return set_err(RT_ERR_INVALID, "null argument");
    if (n == 0) {
        if (stats) std::memset(stats, 0, sizeof(*stats));
        return RT_OK;
    }
    if (const int refused = batch_refusal(n)) return refused;
    rt_ray* d_rays = nullptr;
    rt_hit* d_out = nullptr;
    int rc = RT_OK;
    DeviceGuard guard;
    try {
        CU(cudaSetDevice(s->device));
        scratch_alloc(&d_rays, n * sizeof(rt_ray));
        scratch_alloc(&d_out, n * sizeof(rt_hit));
        CU(cudaMemcpy(d_rays, rays, n * sizeof(rt_ray), cudaMemcpyHostToDevice));
        rc = rt_closest_hit_device(s, d_rays, n, t_min, t_max, flags, d_out, nullptr, stats);
        if (rc == RT_OK) {
            CU(cudaDeviceSynchronize());
            CU(cudaMemcpy(out, d_out, n * sizeof(rt_hit), cudaMemcpyDeviceToHost));
        }
    } catch (const CudaFail& f) {
        rc = set_err(RT_ERR_CUDA, f.what);
    }
    scratch_free(d_rays);
    scratch_free(d_out);
    return rc;
}

int rt_occluded_device(const rt_scene* s, const rt_ray* d_rays, const double* d_t_max_per_ray, uint64_t n, double t_min, double t_max,
                       uint32_t flags, uint8_t* d_out, void* stream, rt_stats* stats) {
    if (!s || (n && (!d_rays || !d_out))) return set_err(RT_ERR_INVALID, "null argument");
    return run_batch(s, n, flags, stream, stats, [&](bool count, unsigned long long* d_cnt, int grid, cudaStream_t st) {
        launch_occluded(s->view, d_rays, d_t_max_per_ray, (uint32_t)n, t_min, t_max, count, d_out, d_cnt, grid, s->stack_bytes, st);
        return 1;
    });
}

int rt_occluded(const rt_scene* s, const rt_ray* rays, const double* t_max_per_ray, uint64_t n, double t_min, double t_max, uint32_t flags,
                uint8_t* out, rt_stats* stats) {
    if (!s || (n && (!rays || !out))) return set_err(RT_ERR_INVALID, "null argument");
    if (n == 0) {
        if (stats) std::memset(stats, 0, sizeof(*stats));
        return RT_OK;
    }
    if (const int refused = batch_refusal(n)) return refused;
    rt_ray* d_rays = nullptr;
    double* d_tmax = nullptr;
    uint8_t* d_out = nullptr;
    int rc = RT_OK;
    DeviceGuard guard;
    try {
        CU(cudaSetDevice(s->device));
        scratch_alloc(&d_rays, n * sizeof(rt_ray));
        scratch_alloc(&d_out, n);
        CU(cudaMemcpy(d_rays, rays, n * sizeof(rt_ray), cudaMemcpyHostToDevice));
        if (t_max_per_ray) {
            scratch_alloc(&d_tmax, n * sizeof(double));
            CU(cudaMemcpy(d_tmax, t_max_per_ray, n * sizeof(double), cudaMemcpyHostToDevice));
        }
        rc = rt_occluded_device(s, d_rays, d_tmax, n, t_min, t_max, flags, d_out, nullptr, stats);
        if (rc == RT_OK) {
            CU(cudaDeviceSynchronize());
            CU(cudaMemcpy(out, d_out, n, cudaMemcpyDeviceToHost));
        }
    } catch (const CudaFail& f) {
        rc = set_err(RT_ERR_CUDA, f.what);
    }
    scratch_free(d_rays);
    scratch_free(d_tmax);
    scratch_free(d_out);
    return rc;
}

int rt_transmittance_device(const rt_scene* s, const rt_ray* d_rays, const double* d_t_max_per_ray, uint64_t n, double t_min, double t_max,
                            uint32_t flags, double* d_out, void* stream, rt_stats* stats) {
    if (!s || (n && (!d_rays || !d_out))) return set_err(RT_ERR_INVALID, "null argument");
    return run_batch(s, n, flags, stream, stats, [&](bool count, unsigned long long* d_cnt, int grid, cudaStream_t st) {
        // the surface pass writes one occlusion byte per ray to a stream-ordered scratch buffer; the media pass reads it
        uint8_t* d_occ = nullptr;
        CU(cudaMallocAsync((void**)&d_occ, n, st));
        launch_occluded(s->view, d_rays, d_t_max_per_ray, (uint32_t)n, t_min, t_max, count, d_occ, d_cnt, grid, s->stack_bytes, st);
        int grid_m = s->sm_count * 8;
        const uint64_t need = (n + MEDIA_BLOCK - 1) / MEDIA_BLOCK;
        if ((uint64_t)grid_m > need) grid_m = (int)need;
        launch_transmittance(s->view, s->generic_media, d_rays, d_t_max_per_ray, (uint32_t)n, t_min, t_max, count, d_occ, d_out, d_cnt, grid_m, st);
        CU(cudaFreeAsync(d_occ, st));
        return 2;
    });
}

int rt_transmittance(const rt_scene* s, const rt_ray* rays, const double* t_max_per_ray, uint64_t n, double t_min, double t_max,
                     uint32_t flags, double* out, rt_stats* stats) {
    if (!s || (n && (!rays || !out))) return set_err(RT_ERR_INVALID, "null argument");
    if (n == 0) {
        if (stats) std::memset(stats, 0, sizeof(*stats));
        return RT_OK;
    }
    if (const int refused = batch_refusal(n)) return refused;
    rt_ray* d_rays = nullptr;
    double* d_tmax = nullptr;
    double* d_out = nullptr;
    int rc = RT_OK;
    DeviceGuard guard;
    try {
        CU(cudaSetDevice(s->device));
        scratch_alloc(&d_rays, n * sizeof(rt_ray));
        scratch_alloc(&d_out, n * sizeof(double));
        CU(cudaMemcpy(d_rays, rays, n * sizeof(rt_ray), cudaMemcpyHostToDevice));
        if (t_max_per_ray) {
            scratch_alloc(&d_tmax, n * sizeof(double));
            CU(cudaMemcpy(d_tmax, t_max_per_ray, n * sizeof(double), cudaMemcpyHostToDevice));
        }
        rc = rt_transmittance_device(s, d_rays, d_tmax, n, t_min, t_max, flags, d_out, nullptr, stats);
        if (rc == RT_OK) {
            CU(cudaDeviceSynchronize());
            CU(cudaMemcpy(out, d_out, n * sizeof(double), cudaMemcpyDeviceToHost));
        }
    } catch (const CudaFail& f) {
        rc = set_err(RT_ERR_CUDA, f.what);
    }
    scratch_free(d_rays);
    scratch_free(d_tmax);
    scratch_free(d_out);
    return rc;
}

int rt_world_hit_device(const rt_scene* s, const rt_ray* d_rays, const double* d_t_max_per_ray, uint64_t n, double t_min, double t_max,
                        uint64_t seed, uint32_t segment, uint32_t flags, rt_hit_record* d_out, void* stream, rt_stats* stats) {
    if (!s || (n && (!d_rays || !d_out))) return set_err(RT_ERR_INVALID, "null argument");
    return run_batch(s, n, flags, stream, stats, [&](bool count, unsigned long long* d_cnt, int grid, cudaStream_t st) {
        // the surface pass writes the surface winner of every ray (16 bytes) to a stream-ordered scratch buffer; the record pass reads it
        HitRec* d_surface = nullptr;
        CU(cudaMallocAsync((void**)&d_surface, n * sizeof(HitRec), st));
        launch_world_hit_surface(s->view, d_rays, d_t_max_per_ray, (uint32_t)n, t_min, t_max, count, d_surface, d_cnt, grid, s->stack_bytes, st);
        int grid_m = s->sm_count * 8;
        const uint64_t need = (n + MEDIA_BLOCK - 1) / MEDIA_BLOCK;
        if ((uint64_t)grid_m > need) grid_m = (int)need;
        launch_world_hit_record(s->view, s->generic_media, d_rays, d_t_max_per_ray, (uint32_t)n, t_min, t_max, seed, segment, count, d_surface, d_out,
                                d_cnt, grid_m, st);
        CU(cudaFreeAsync(d_surface, st));
        return 2;
    });
}

int rt_world_hit(const rt_scene* s, const rt_ray* rays, const double* t_max_per_ray, uint64_t n, double t_min, double t_max, uint64_t seed,
                 uint32_t segment, uint32_t flags, rt_hit_record* out, rt_stats* stats) {
    if (!s || (n && (!rays || !out))) return set_err(RT_ERR_INVALID, "null argument");
    if (n == 0) {
        if (stats) std::memset(stats, 0, sizeof(*stats));
        return RT_OK;
    }
    if (const int refused = batch_refusal(n)) return refused;
    rt_ray* d_rays = nullptr;
    double* d_tmax = nullptr;
    rt_hit_record* d_out = nullptr;
    int rc = RT_OK;
    DeviceGuard guard;
    try {
        CU(cudaSetDevice(s->device));
        scratch_alloc(&d_rays, n * sizeof(rt_ray));
        scratch_alloc(&d_out, n * sizeof(rt_hit_record));
        CU(cudaMemcpy(d_rays, rays, n * sizeof(rt_ray), cudaMemcpyHostToDevice));
        if (t_max_per_ray) {
            scratch_alloc(&d_tmax, n * sizeof(double));
            CU(cudaMemcpy(d_tmax, t_max_per_ray, n * sizeof(double), cudaMemcpyHostToDevice));
        }
        rc = rt_world_hit_device(s, d_rays, d_tmax, n, t_min, t_max, seed, segment, flags, d_out, nullptr, stats);
        if (rc == RT_OK) {
            CU(cudaDeviceSynchronize());
            CU(cudaMemcpy(out, d_out, n * sizeof(rt_hit_record), cudaMemcpyDeviceToHost));
        }
    } catch (const CudaFail& f) {
        rc = set_err(RT_ERR_CUDA, f.what);
    }
    scratch_free(d_rays);
    scratch_free(d_tmax);
    scratch_free(d_out);
    return rc;
}

// The host-side refusals of rt_shade / rt_shade_device, made before anything is allocated or copied
static int shade_refusal(const rt_scene* s, const rt_camera* cam, uint64_t n, uint32_t segment, uint32_t flags) {
    if (const int refused = batch_refusal(n)) return refused;
    if (flags != 0) return set_err(RT_ERR_INVALID, "rt_shade takes no flags (flags must be 0)");
    if (cam->background_tex >= s->info.n_textures) return set_err(RT_ERR_INVALID, "camera.background_tex out of range");
    if (segment >= cam->max_depth) return set_err(RT_ERR_INVALID, "segment >= camera.max_depth: the reference never runs that segment");
    return RT_OK;
}

int rt_shade_device(const rt_scene* s, const rt_camera* cam, const rt_hit_record* d_records, uint64_t n, uint64_t seed, uint32_t segment,
                    uint32_t flags, rt_ray* d_rays, double* d_beta, double* d_radiance, uint8_t* d_state, void* stream, rt_stats* stats) {
    if (!s || !cam || (n && (!d_records || !d_rays || !d_beta || !d_radiance || !d_state))) return set_err(RT_ERR_INVALID, "null argument");
    if (const int refused = shade_refusal(s, cam, n, segment, flags)) return refused;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long* d_errors = nullptr;
    int rc = RT_OK;
    DeviceGuard guard;
    try {
        // the error count is only kept for `stats`: its word is allocated, cleared and read back outside the timed launch
        if (stats && n) {
            CU(cudaSetDevice(s->device));
            CU(cudaMallocAsync((void**)&d_errors, sizeof(unsigned long long), st));
            CU(cudaMemsetAsync(d_errors, 0, sizeof(unsigned long long), st));
        }
        rc = run_batch(s, n, 0, stream, stats, [&](bool, unsigned long long*, int, cudaStream_t bs) {
            RenderParams P{};
            P.cam = *cam;
            P.seed = seed;
            P.lights_flat = s->lights_flat;
            int grid = s->sm_count * 8;
            const uint64_t need = (n + SHADE_BLOCK - 1) / SHADE_BLOCK;
            if ((uint64_t)grid > need) grid = (int)need;
            launch_shade_records(s->view, P, d_records, n, s->info.n_materials, segment, d_rays, d_beta, d_radiance, d_state, d_errors, grid, bs);
            return 1;
        });
        if (rc == RT_OK && d_errors) {
            unsigned long long h_errors = 0;
            CU(cudaMemcpyAsync(&h_errors, d_errors, sizeof(h_errors), cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            stats->errors = h_errors;
        }
    } catch (const CudaFail& f) {
        rc = set_err(RT_ERR_CUDA, f.what);
    }
    if (d_errors) cudaFreeAsync(d_errors, st);
    return rc;
}

int rt_shade(const rt_scene* s, const rt_camera* cam, const rt_hit_record* records, uint64_t n, uint64_t seed, uint32_t segment, uint32_t flags,
             rt_ray* rays, double* beta, double* radiance, uint8_t* state, rt_stats* stats) {
    if (!s || !cam || (n && (!records || !rays || !beta || !radiance || !state))) return set_err(RT_ERR_INVALID, "null argument");
    if (const int refused = shade_refusal(s, cam, n, segment, flags)) return refused;
    if (n == 0) {
        if (stats) std::memset(stats, 0, sizeof(*stats));
        return RT_OK;
    }
    rt_hit_record* d_rec = nullptr;
    rt_ray* d_rays = nullptr;
    double *d_beta = nullptr, *d_rad = nullptr;
    uint8_t* d_state = nullptr;
    int rc = RT_OK;
    DeviceGuard guard;
    try {
        CU(cudaSetDevice(s->device));
        scratch_alloc(&d_rec, n * sizeof(rt_hit_record));
        scratch_alloc(&d_rays, n * sizeof(rt_ray));
        scratch_alloc(&d_beta, n * 3 * sizeof(double));
        scratch_alloc(&d_rad, n * 3 * sizeof(double));
        scratch_alloc(&d_state, n);
        CU(cudaMemcpy(d_rec, records, n * sizeof(rt_hit_record), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(d_rays, rays, n * sizeof(rt_ray), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(d_beta, beta, n * 3 * sizeof(double), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(d_rad, radiance, n * 3 * sizeof(double), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(d_state, state, n, cudaMemcpyHostToDevice));
        rc = rt_shade_device(s, cam, d_rec, n, seed, segment, flags, d_rays, d_beta, d_rad, d_state, nullptr, stats);
        if (rc == RT_OK) {
            CU(cudaDeviceSynchronize());
            CU(cudaMemcpy(rays, d_rays, n * sizeof(rt_ray), cudaMemcpyDeviceToHost));
            CU(cudaMemcpy(beta, d_beta, n * 3 * sizeof(double), cudaMemcpyDeviceToHost));
            CU(cudaMemcpy(radiance, d_rad, n * 3 * sizeof(double), cudaMemcpyDeviceToHost));
            CU(cudaMemcpy(state, d_state, n, cudaMemcpyDeviceToHost));
        }
    } catch (const CudaFail& f) {
        rc = set_err(RT_ERR_CUDA, f.what);
    }
    scratch_free(d_rec);
    scratch_free(d_rays);
    scratch_free(d_beta);
    scratch_free(d_rad);
    scratch_free(d_state);
    return rc;
}

int rt_camera_rays_device(const rt_camera* cam, uint64_t seed, uint32_t sample, rt_ray* d_out, void* stream) {
    if (!cam || !d_out) return set_err(RT_ERR_INVALID, "null argument");
    if ((uint64_t)sample >= (uint64_t)cam->sqrt_spp * cam->sqrt_spp) return set_err(RT_ERR_INVALID, "sample >= sqrt_spp^2");
    const uint64_t n = (uint64_t)cam->image_width * cam->image_height;
    if (n > 0xFFFFFFF0ull) return set_err(RT_ERR_INVALID, "more than 2^32 - 16 pixels");
    int device, sms;
    int rc = check_device(-1, device, sms);
    if (rc != RT_OK || n == 0) return rc;
    int grid = sms * 8;
    if ((uint64_t)grid > (n + 255) / 256) grid = (int)((n + 255) / 256);
    launch_camera_rays(*cam, seed, sample, n, d_out, grid, (cudaStream_t)stream);
    if (cudaGetLastError() != cudaSuccess) return set_err(RT_ERR_CUDA, "k_camera_rays launch failed");
    return RT_OK;
}

int rt_camera_rays(const rt_camera* cam, uint64_t seed, uint32_t sample, rt_ray* out) {
    if (!cam || !out) return set_err(RT_ERR_INVALID, "null argument");
    if ((uint64_t)sample >= (uint64_t)cam->sqrt_spp * cam->sqrt_spp) return set_err(RT_ERR_INVALID, "sample >= sqrt_spp^2");
    const uint64_t n = (uint64_t)cam->image_width * cam->image_height;
    if (n > 0xFFFFFFF0ull) return set_err(RT_ERR_INVALID, "more than 2^32 - 16 pixels");
    int device, sms;
    int rc = check_device(-1, device, sms);
    if (rc != RT_OK || n == 0) return rc;
    keep_pool_memory(device);
    rt_ray* d = nullptr;
    cudaStream_t st = cudaStreamPerThread;
    try {
        CU(cudaMallocAsync((void**)&d, n * sizeof(rt_ray), st));
        rc = rt_camera_rays_device(cam, seed, sample, d, st);
        if (rc == RT_OK) {
            CU(cudaMemcpyAsync(out, d, n * sizeof(rt_ray), cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
        }
    } catch (const CudaFail& f) {
        rc = set_err(RT_ERR_CUDA, f.what);
    }
    if (d) cudaFreeAsync(d, st);
    return rc;
}

static uint64_t count_partition_pixels(uint32_t W, uint32_t H, uint32_t part_index, uint32_t part_count) {
    uint32_t tiles_x = (W + 7) / 8, tiles_y = (H + 7) / 8;
    uint64_t n = 0;
    for (uint32_t ty = 0; ty < tiles_y; ty++)
        for (uint32_t tx = 0; tx < tiles_x; tx++) {
            uint32_t tile = ty * tiles_x + tx;
            if (tile % part_count != part_index) continue;
            uint32_t w = std::min(8u, W - tx * 8), h = std::min(8u, H - ty * 8);
            n += (uint64_t)w * h;
        }
    return n;
}

int rt_render_device(const rt_scene* cs, const rt_camera* cam, const rt_render_opts* opts, void* d_accum, void* stream, rt_stats* stats) {
    if (!cs || !cam || !d_accum) return set_err(RT_ERR_INVALID, "null argument");
    rt_scene* s = const_cast<rt_scene*>(cs);
    rt_render_opts o{};
    if (opts) {
        if (opts->struct_size != sizeof(rt_render_opts)) return set_err(RT_ERR_VERSION, "rt_render_opts.struct_size mismatch");
        o = *opts;
    }
    if (cam->image_width == 0 || cam->image_height == 0 || cam->sqrt_spp == 0)
        return set_err(RT_ERR_INVALID, "camera has an empty image or zero samples");
    // the path ids travel packed in the ray record (kernels.h): 28 + 24 + 12 bits
    if ((uint64_t)cam->image_width * cam->image_height >= (1ull << IDS_PIXEL_BITS))
        return set_err(RT_ERR_UNSUPPORTED, "more than 2^28 pixels");
    if ((uint64_t)cam->sqrt_spp * cam->sqrt_spp >= (1ull << IDS_SAMPLE_BITS)) return set_err(RT_ERR_UNSUPPORTED, "more than 2^24 samples per pixel");
    if (cam->max_depth >= (1u << IDS_SEGMENT_BITS)) return set_err(RT_ERR_UNSUPPORTED, "max_depth above 4095");
    if (cam->background_tex >= s->info.n_textures) return set_err(RT_ERR_INVALID, "camera.background_tex out of range");
    const uint32_t part_count = o.part_count ? o.part_count : 1;
    if (o.part_index >= part_count) return set_err(RT_ERR_INVALID, "part_index >= part_count");
    uint32_t s_begin = o.sample_begin, s_end = o.sample_end;
    const uint32_t spp = cam->sqrt_spp * cam->sqrt_spp;
    if (s_begin == 0 && s_end == 0) s_end = spp;
    if (s_begin > s_end || s_end > spp) return set_err(RT_ERR_INVALID, "bad sample range");
    if (stats) std::memset(stats, 0, sizeof(*stats));

    WorkspaceLease lease(device_workspace(s->device));
    cudaStream_t st = (cudaStream_t)stream;
    const uint64_t n_px_img = (uint64_t)cam->image_width * cam->image_height;
    const uint64_t n_pixels = count_partition_pixels(cam->image_width, cam->image_height, o.part_index, part_count);
    const uint64_t nominal_paths = n_pixels * (uint64_t)(s_end - s_begin);
    // max_depth == 0: ray_color returns black before it looks at the world (camera.rs:282) - no path is traced
    const uint64_t total_paths = cam->max_depth == 0 ? 0 : nominal_paths;
    // paths in flight: large enough that the ~14 launches of an iteration and the under-filled start and end of every
    // persistent kernel are amortised over many segments, never more than the job needs.  Measured, 800x800x144 book2 frame:
    // 2^23 / 2^24 / 2^25 / 2^26 paths: 90.9 / 87.9 / 86.6 / 85.5 ms (the 1920x1080 mesh scene: 105.0 -> 97.9 ms from 2^24 to 2^25);
    // 2^27 paths are 33 GB of streams (249 B per path), 18 % of a B200's memory; a device that cannot give that much gets half (below).
    // (2^27 since the random walk took a third of the segments out of the streams: 455.9 -> 449.8 ms on the bench frame, 45 -> 39 iterations)
    uint32_t capacity = o.max_paths_in_flight ? o.max_paths_in_flight : (1u << 27);
    if (const char* e = getenv("RT2025_PATHS_IN_FLIGHT")) capacity = (uint32_t)std::max(1024l, atol(e));  // tuning knob
    capacity = (uint32_t)std::min<uint64_t>(capacity, ((total_paths + 1023) / 1024) * 1024);
    capacity = std::max(capacity, 1024u);
    cudaEvent_t ev[8] = {nullptr};
    int rc = RT_OK;
    try {
        CU(cudaSetDevice(s->device));
        Workspace& ws = *lease.ws;
        if (ws.capacity < capacity || ws.n_pixels_alloc < n_px_img) {  // grow-only
            uint32_t capacity_alloc = std::max(ws.capacity, capacity);
            const uint64_t n_px_alloc = std::max<uint64_t>(ws.n_pixels_alloc, n_px_img);
            // the streams are 249 bytes per path in flight (33 GB at the default 2^27): when the device cannot give that much
            // - other tenants, a smaller part - halve the capacity instead of failing; the image does not depend on it
            while (true) {
                ws.release();
                WavefrontState& W = ws.W;
                bool ok = true;
                auto alloc = [&](auto** p, size_t bytes) { ok = ok && cudaMalloc((void**)p, bytes) == cudaSuccess; };
                for (int k = 0; k < 2; k++) {
                    alloc(&W.ray_q[k], (size_t)capacity_alloc * sizeof(RayRec));
                    alloc(&W.beta_q[k], (size_t)capacity_alloc * sizeof(BetaRec));
                }
                alloc(&W.hit_q, (size_t)capacity_alloc * sizeof(HitRec));
                alloc(&W.cls_q, (size_t)capacity_alloc);
                for (auto& q : W.q_shade) alloc(&q, (size_t)capacity_alloc * 4);
                alloc(&W.pixel_list, n_px_alloc * 4);
                alloc(&W.accum, n_px_alloc * 3 * sizeof(double));
                alloc(&W.counters, sizeof(Counters));
                if (ok) break;
                cudaGetLastError();
                if (capacity_alloc <= (1u << 20)) {
                    ws.release();
                    throw CudaFail{"out of device memory for the wavefront streams (even at 2^20 paths in flight)"};
                }
                capacity_alloc >>= 1;
            }
            CU(cudaMallocHost(&ws.h_counters, 2 * sizeof(Counters)));
            ws.capacity = capacity_alloc;
            ws.n_pixels_alloc = n_px_alloc;
        }
        capacity = std::min(capacity, ws.capacity);
        WavefrontState W = ws.W;
        W.capacity = capacity;
        W.n_pixels = (uint32_t)n_pixels;
        W.total_paths = total_paths;
        RenderParams P{};
        P.cam = *cam;
        P.seed = o.seed;
        P.sample_begin = s_begin;
        P.part_index = o.part_index, P.part_count = part_count;
        P.lights_flat = s->lights_flat;
        P.bin_by_class = (o.reserved[0] & 1u) ? 0u : 1u;  // reserved[0] bit 0: disable material binning (A/B evidence)
        // media-first order (kernels.cu, PathIO<MEDIA>: sampled by extend while it prepares the ray) when every boundary is a single sphere.
        // With general boundaries the sampling pass loses its cheapest screen (free flight vs surface distance) and the
        // extra boundary traversals cost more than extend saves (mesh-fog scene 1092 -> 1104 ms), so those keep the
        // classic order.  reserved[0] bit 1 or RT2025_MEDIA_FIRST=0/1 override.
        P.media_first = (s->view.n_media > 0 && !s->generic_media && !(o.reserved[0] & 2u)) ? 1u : 0u;
        // 1 = a sampling pass ahead of extend, 2 = sampled by extend while it prepares the ray.  Measured on book2_final (ms per
        // 800x800x144 frame, extend + media + binning): pass 47.7+2, fused 52.2+2 - the pass runs at 24 warps per SM and streams,
        // inside extend the same binary64 code runs at 16 warps per SM - so the pass is the default; RT2025_MEDIA_FIRST=0/1/2.
        if (const char* e = getenv("RT2025_MEDIA_FIRST")) P.media_first = (s->view.n_media > 0 && !s->generic_media) ? (uint32_t)std::max(0, std::min(2, atoi(e))) : 0u;

        // measured on one eighth of the bench frame (what a rank of an 8-GPU run renders): 66.9 -> 66.0 ms; the whole frame on one GPU is unchanged
        P.walk_drain_queue = 262144, P.walk_drain_steps = 4;
        if (const char* e = getenv("RT2025_WALK_DRAIN_QUEUE")) P.walk_drain_queue = (uint32_t)std::max(0l, atol(e));  // tuning knobs
        if (const char* e = getenv("RT2025_WALK_DRAIN_STEPS")) P.walk_drain_steps = (uint32_t)std::max(1l, atol(e));
        // a miss against a black background adds nothing to the frame: extend drops the path instead of queueing it for the miss kernel
        P.drop_misses = s->black_texture[cam->background_tex] && !getenv("RT2025_KEEP_MISSES");
        P.sample_in_generate = 1;
        if (const char* e = getenv("RT2025_GEN_MEDIA")) P.sample_in_generate = atoi(e) != 0;  // tuning knob
        const bool count = (o.flags & RT_OPT_COUNT) != 0, stage = (o.flags & RT_OPT_STAGE_TIMES) != 0;
        if (count) P.sample_in_generate = 0;  // the counting instantiation of the sampling pass sees every segment
        const int grid_e = s->sm_count * s->extend_blocks_per_sm, grid_s = s->sm_count * s->shade_blocks_per_sm;
        const int grid_g = s->sm_count * 4;
        const int grid_m = s->sm_count * 8;
        for (auto& e : ev) CU(cudaEventCreate(&e));
        CU(cudaEventRecord(ev[0], st));
        Counters init{};
        CU(cudaMemcpyAsync(W.counters, &init, sizeof(init), cudaMemcpyHostToDevice, st));
        CU(cudaMemsetAsync(W.accum, 0, n_px_img * 3 * sizeof(double), st));
        uint64_t launches = 2;
        const Counters* final_counters = nullptr;
        double ms_gen = 0, ms_ext = 0, ms_med = 0, ms_shd = 0;
        if (total_paths > 0) {
            launch_init(W, P, grid_g, st);
            launches += 1;
            // k_tail: below this many live paths (and no camera path left to generate) one launch finishes the frame
            uint32_t tail_threshold = 1u << 16;
            if (const char* e = getenv("RT2025_TAIL_PATHS")) tail_threshold = (uint32_t)std::max(0l, atol(e));  // tuning knob (0 disables)
            size_t iters = 0;
            auto enqueue_iterations = [&](size_t n_iter) {
                for (size_t b = 0; b < n_iter; b++, iters++) {
                    W.parity = (uint32_t)(iters & 1);
                    // stage times: events are only recorded here and read after the render, so the
                    // measurement does not add a host synchronisation to the timed region
                    if (stage) CU(cudaEventRecord(ws.event(6 * iters + 0), st));
                    launch_generate(s->view, P, W, grid_g, st);
                    if (stage) CU(cudaEventRecord(ws.event(6 * iters + 1), st));
                    // media_first 1: a sampling pass ahead of extend leaves the nearest scatter point as the incumbent; 2: extend
                    // samples the sphere-bounded media itself; 0: the media pass runs between extend and the binning
                    if (P.media_first == 1) launches += launch_media_bin(s->view, P, W, count, s->generic_media, grid_m, st, 1);
                    if (stage) CU(cudaEventRecord(ws.event(6 * iters + 5), st));
                    launch_extend(s->view, P, W, count, grid_e, s->stack_bytes, st);
                    if (stage) CU(cudaEventRecord(ws.event(6 * iters + 2), st));
                    launches += launch_media_bin(s->view, P, W, count, s->generic_media, grid_m, st, P.media_first ? 2 : 0);
                    if (stage) CU(cudaEventRecord(ws.event(6 * iters + 3), st));
                    launches += 2 + launch_shade(s->view, P, W, s->class_mask, grid_s, st, ws.shade_fan(), tail_threshold != 0, s->sm_count * s->walk_blocks_per_sm);  // generate, extend + shade
                    if (tail_threshold) {
                        launch_tail(s->view, P, W, tail_threshold, s->sm_count, st);
                        launches += 1;
                    }
                    if (stage) CU(cudaEventRecord(ws.event(6 * iters + 4), st));
                }
            };
            auto read_back = [&](int slot) {
                CU(cudaMemcpyAsync(&ws.h_counters[slot], W.counters, sizeof(Counters), cudaMemcpyDeviceToHost, st));
                CU(cudaEventRecord(ws.check_event(slot), st));
            };
            // The host never idles the GPU to learn whether the frame is finished.  Generation alone takes at least
            // total_paths / capacity iterations: those are enqueued without a look at the counters.  After that the counters of
            // burst k are read while burst k+1 is already queued (two pinned copies, two events); the burst that runs past the
            // last live path is a list of kernels that find empty queues and return (~3 us each).
            enqueue_iterations(std::max<size_t>(1, (size_t)((total_paths + capacity - 1) / capacity)));
            int slot = 0;
            read_back(slot);
            const size_t burst = 2;
            while (true) {
                enqueue_iterations(burst);
                read_back(slot ^ 1);
                CU(cudaEventSynchronize(ws.check_event(slot)));
                const Counters& hc = ws.h_counters[slot];
                if (hc.next_path >= total_paths && hc.n_extend[0] == 0 && hc.n_extend[1] == 0) break;  // (the speculative burst adds nothing to it)
                slot ^= 1;
            }
            final_counters = &ws.h_counters[slot];
            CU(cudaGetLastError());
            if (stage) {
                for (size_t i = 0; i < iters; i++) {
                    float a, b, c, d;
                    CU(cudaEventElapsedTime(&a, ws.events[6 * i], ws.events[6 * i + 1]));
                    float m1;  // generate | media sampling pass (if any) | extend | media pass (if any) + binning | shade
                    CU(cudaEventElapsedTime(&m1, ws.events[6 * i + 1], ws.events[6 * i + 5]));
                    CU(cudaEventElapsedTime(&b, ws.events[6 * i + 5], ws.events[6 * i + 2]));
                    CU(cudaEventElapsedTime(&c, ws.events[6 * i + 2], ws.events[6 * i + 3]));
                    c += m1;
                    CU(cudaEventElapsedTime(&d, ws.events[6 * i + 3], ws.events[6 * i + 4]));
                    ms_gen += a, ms_ext += b, ms_med += c, ms_shd += d;
                    if (getenv("RT2025_ITER_TIMES")) fprintf(stderr, "[rt2025] iteration %3zu: generate %7.3f  media+bin %7.3f  extend %7.3f  shade %7.3f ms\n", i, a, c, b, d);
                }
                // the timing pool grows with the longest render: keep a few hundred iterations' worth
                while (ws.events.size() > 6 * 512) {
                    cudaEventDestroy(ws.events.back());
                    ws.events.pop_back();
                }
            }
        }
        launch_finalize(W.accum, n_px_img * 3, cam->pixel_sample_scale, d_accum, o.accum_type == RT_ACCUM_F64, grid_g, st);
        launches += 1;
        CU(cudaEventRecord(ev[1], st));
        CU(cudaEventSynchronize(ev[1]));
        CU(cudaGetLastError());
        if (stats) {
            float ms = 0;
            CU(cudaEventElapsedTime(&ms, ev[0], ev[1]));
            const Counters zero{};
            const Counters& c = final_counters ? *final_counters : zero;
            stats->paths = nominal_paths;
            stats->segments = total_paths ? c.segments : 0;
            stats->node_visits = total_paths ? c.node_visits : 0;
            stats->prim_tests = total_paths ? c.prim_tests : 0;
            stats->errors = total_paths ? c.errors : 0;
            stats->iterations = total_paths ? c.iterations : 0;
            stats->reserved[0] = total_paths ? c.walk_segments : 0;  // rt_stats.walk_segments
            stats->reserved[1] = total_paths ? c.walk_lean_segments : 0;  // rt_stats.walk_lean_segments
            stats->reserved[2] = total_paths ? c.shade_lean_hits : 0;  // rt_stats.shade_lean_hits
            stats->kernel_launches = launches;
            stats->ms_total = ms;
            stats->ms_raygen = ms_gen, stats->ms_extend = ms_ext, stats->ms_shade = ms_shd;
            stats->ms_other = ms_med;  // the media + binning kernel
        }
    } catch (const CudaFail& f) {
        rc = set_err(RT_ERR_CUDA, f.what);
    }
    for (auto& e : ev)
        if (e) cudaEventDestroy(e);
    return rc;
}

int rt_render(const rt_scene* s, const rt_camera* cam, const rt_render_opts* opts, void* accum, rt_stats* stats) {
    if (!s || !cam || !accum) return set_err(RT_ERR_INVALID, "null argument");
    const size_t elem = (opts && opts->accum_type == RT_ACCUM_F64) ? 8 : 4;
    const size_t bytes = (size_t)cam->image_width * cam->image_height * 3 * elem;
    void* d = nullptr;
    int rc = RT_OK;
    DeviceGuard guard;
    try {
        CU(cudaSetDevice(s->device));
        scratch_alloc(&d, bytes);
        rc = rt_render_device(s, cam, opts, d, nullptr, stats);
        if (rc == RT_OK) CU(cudaMemcpy(accum, d, bytes, cudaMemcpyDeviceToHost));
    } catch (const CudaFail& f) {
        rc = set_err(RT_ERR_CUDA, f.what);
    }
    scratch_free(d);
    return rc;
}

int rt_render_rgb8(const rt_scene* s, const rt_camera* cam, const rt_render_opts* opts, uint8_t* rgb, rt_stats* stats) {
    if (!s || !cam || !rgb) return set_err(RT_ERR_INVALID, "null argument");
    rt_render_opts o{};
    if (opts) o = *opts;
    o.struct_size = sizeof(o);
    o.accum_type = RT_ACCUM_F64;
    const uint64_t n_px = (uint64_t)cam->image_width * cam->image_height;
    double* d_accum = nullptr;
    uint8_t* d_rgb = nullptr;
    int* d_flag = nullptr;
    int rc = RT_OK;
    DeviceGuard guard;
    try {
        CU(cudaSetDevice(s->device));
        scratch_alloc(&d_accum, n_px * 3 * sizeof(double));
        scratch_alloc(&d_rgb, n_px * 3);
        scratch_alloc(&d_flag, sizeof(int));
        CU(cudaMemset(d_flag, 0, sizeof(int)));
        rc = rt_render_device(s, cam, &o, d_accum, nullptr, stats);
        if (rc == RT_OK) {
            launch_tonemap(d_accum, true, n_px, cam->toon_map, d_rgb, d_flag, nullptr);
            CU(cudaGetLastError());
            CU(cudaMemcpy(rgb, d_rgb, n_px * 3, cudaMemcpyDeviceToHost));
            int flag = 0;
            CU(cudaMemcpy(&flag, d_flag, sizeof(int), cudaMemcpyDeviceToHost));
            if (flag) rc = set_err(RT_ERR_INVALID, "NaN radiance in the image (utils/color.rs:28 asserts)");
            if (stats) stats->kernel_launches += 1;
        }
    } catch (const CudaFail& f) {
        rc = set_err(RT_ERR_CUDA, f.what);
    }
    scratch_free(d_accum);
    scratch_free(d_rgb);
    scratch_free(d_flag);
    return rc;
}

namespace {

// The multi-GPU render behind rt_render_multi / rt_render_multi_rgb8: GPU i renders partition i of n from a host thread of
// its own into a framebuffer in ITS memory; GPU 0 then sums the partial frames with one kernel that reads the other GPUs'
// buffers through peer mappings (NVLink loads; a staged cudaMemcpyPeer where two devices cannot map each other).  The
// partitions are disjoint pixel sets, so the sum is also the gather.  On return `parts[0]` (device scenes[0]->device)
// holds the complete frame; the caller reads it back - or encodes it first - and frees every buffer with free_parts().
struct MultiFrame {
    std::vector<void*> parts;   // parts[i] lives on scenes[i]->device
    std::vector<int> devices;
    void* staged = nullptr;     // scratch on device 0 for peers that cannot be mapped
    ~MultiFrame() {
        for (size_t i = 0; i < parts.size(); i++)
            if (parts[i]) {
                cudaSetDevice(devices[i]);
                cudaFreeAsync(parts[i], cudaStreamPerThread);
            }
        if (staged) {
            cudaSetDevice(devices[0]);
            cudaFreeAsync(staged, cudaStreamPerThread);
        }
    }
};

int render_multi_to_device0(rt_scene* const* scenes, uint32_t n, const rt_camera* cam, const rt_render_opts* opts, bool force_f64, MultiFrame& mf,
                            rt_stats* stats) {
    if (!scenes || !n || !cam) return set_err(RT_ERR_INVALID, "null argument");
    if (n > MAX_PARTS) return set_err(RT_ERR_UNSUPPORTED, "more than 16 GPUs");
    rt_render_opts base{};
    if (opts) {
        if (opts->struct_size != sizeof(rt_render_opts)) return set_err(RT_ERR_VERSION, "rt_render_opts.struct_size mismatch");
        base = *opts;
    }
    base.struct_size = sizeof(base);
    if (force_f64) base.accum_type = RT_ACCUM_F64;
    if (base.part_count > 1 || base.part_index != 0) return set_err(RT_ERR_INVALID, "rt_render_multi partitions the image itself");
    for (uint32_t i = 0; i < n; i++) {
        if (!scenes[i]) return set_err(RT_ERR_INVALID, "null scene");
        for (uint32_t j = 0; j < i; j++)
            if (scenes[j]->device == scenes[i]->device) return set_err(RT_ERR_INVALID, "two scenes on the same device");
    }
    const size_t n_val = (size_t)cam->image_width * cam->image_height * 3;
    const bool f64 = base.accum_type == RT_ACCUM_F64;
    const size_t bytes = n_val * (f64 ? 8 : 4);
    mf.parts.assign(n, nullptr);
    mf.devices.resize(n);
    for (uint32_t i = 0; i < n; i++) mf.devices[i] = scenes[i]->device;
    std::vector<rt_stats> st(n);
    std::vector<int> rcs(n, RT_OK);
    std::vector<std::string> errs(n);
    std::vector<std::thread> threads;
    for (uint32_t i = 0; i < n; i++) {
        threads.emplace_back([&, i]() {
            rt_render_opts o = base;
            o.part_index = i;
            o.part_count = n;
            if (cudaSetDevice(scenes[i]->device) != cudaSuccess || cudaMallocAsync(&mf.parts[i], bytes, cudaStreamPerThread) != cudaSuccess) {
                rcs[i] = RT_ERR_CUDA, errs[i] = "cudaMallocAsync of a partial framebuffer failed";
                cudaGetLastError();
                return;
            }
            rcs[i] = rt_render_device(scenes[i], cam, &o, mf.parts[i], cudaStreamPerThread, &st[i]);  // returns when the frame is complete
            if (rcs[i] != RT_OK) errs[i] = rt_last_error();  // thread-local: carry it to the caller's thread
        });
    }
    for (auto& t : threads) t.join();
    for (uint32_t i = 0; i < n; i++)
        if (rcs[i] != RT_OK) return set_err(rcs[i], errs[i]);
    try {
        const int dev0 = scenes[0]->device;
        CU(cudaSetDevice(dev0));
        cudaStream_t st0 = cudaStreamPerThread;
        int launches = 0;
        if (n > 1) {
            PartList mapped{};  // partial frames GPU 0 can load from directly
            mapped.p[mapped.n++] = mf.parts[0];
            for (uint32_t i = 1; i < n; i++) {
                int can = 0;
                cudaDeviceCanAccessPeer(&can, dev0, scenes[i]->device);
                if (can) {
                    // the partial frames are stream-ordered allocations: their visibility to a peer is a property of the owning
                    // device's memory pool (cudaDeviceEnablePeerAccess only covers cudaMalloc memory)
                    cudaMemPool_t pool = nullptr;
                    cudaMemAccessDesc desc{};
                    desc.location.type = cudaMemLocationTypeDevice;
                    desc.location.id = dev0;
                    desc.flags = cudaMemAccessFlagsProtReadWrite;
                    if (cudaDeviceGetDefaultMemPool(&pool, scenes[i]->device) != cudaSuccess || cudaMemPoolSetAccess(pool, &desc, 1) != cudaSuccess) can = 0;
                    cudaGetLastError();
                }
                if (can) {
                    mapped.p[mapped.n++] = mf.parts[i];
                } else {  // no mapping between the two: stage the partial frame on GPU 0 and add it at once
                    if (!mf.staged) CU(cudaMallocAsync(&mf.staged, bytes, st0));
                    CU(cudaMemcpyPeerAsync(mf.staged, dev0, mf.parts[i], scenes[i]->device, bytes, st0));
                    PartList two{};
                    two.p[0] = mf.parts[0], two.p[1] = mf.staged, two.n = 2;
                    launch_sum_parts(two, mf.parts[0], n_val, f64, scenes[0]->sm_count * 4, st0);
                    launches++;
                }
            }
            if (mapped.n > 1) {
                launch_sum_parts(mapped, mf.parts[0], n_val, f64, scenes[0]->sm_count * 4, st0);
                launches++;
            }
            CU(cudaGetLastError());
        }
        CU(cudaStreamSynchronize(st0));
        if (stats) {
            std::memset(stats, 0, sizeof(*stats));
            for (uint32_t i = 0; i < n; i++) {
                stats->paths += st[i].paths, stats->segments += st[i].segments, stats->errors += st[i].errors;
                stats->node_visits += st[i].node_visits, stats->prim_tests += st[i].prim_tests;
                stats->kernel_launches += st[i].kernel_launches, stats->iterations += st[i].iterations;
                stats->ms_total = std::max(stats->ms_total, st[i].ms_total);
                stats->ms_raygen = std::max(stats->ms_raygen, st[i].ms_raygen), stats->ms_extend = std::max(stats->ms_extend, st[i].ms_extend);
                stats->ms_shade = std::max(stats->ms_shade, st[i].ms_shade), stats->ms_other = std::max(stats->ms_other, st[i].ms_other);
            }
            stats->kernel_launches += launches;
        }
    } catch (const CudaFail& f) {
        return set_err(RT_ERR_CUDA, f.what);
    }
    return RT_OK;
}

}  // namespace

int rt_render_multi(rt_scene* const* scenes, uint32_t n, const rt_camera* cam, const rt_render_opts* opts, void* accum, rt_stats* stats) {
    if (!accum) return set_err(RT_ERR_INVALID, "null argument");
    DeviceGuard guard;
    MultiFrame mf;
    int rc = render_multi_to_device0(scenes, n, cam, opts, false, mf, stats);
    if (rc != RT_OK) return rc;
    const size_t bytes = (size_t)cam->image_width * cam->image_height * 3 * ((opts && opts->accum_type == RT_ACCUM_F64) ? 8 : 4);
    if (cudaSetDevice(scenes[0]->device) != cudaSuccess || cudaMemcpy(accum, mf.parts[0], bytes, cudaMemcpyDeviceToHost) != cudaSuccess)
        return set_err(RT_ERR_CUDA, std::string("read-back of the reduced frame: ") + cudaGetErrorString(cudaGetLastError()));
    return RT_OK;
}

int rt_render_multi_rgb8(rt_scene* const* scenes, uint32_t n, const rt_camera* cam, const rt_render_opts* opts, uint8_t* rgb, rt_stats* stats) {
    if (!rgb) return set_err(RT_ERR_INVALID, "null argument");
    DeviceGuard guard;
    MultiFrame mf;
    int rc = render_multi_to_device0(scenes, n, cam, opts, true, mf, stats);
    if (rc != RT_OK) return rc;
    const uint64_t n_px = (uint64_t)cam->image_width * cam->image_height;
    char* d = nullptr;
    cudaStream_t st0 = cudaStreamPerThread;
    try {
        CU(cudaSetDevice(scenes[0]->device));
        const size_t out_bytes = ((size_t)n_px * 3 + 255) & ~size_t(255);
        CU(cudaMallocAsync((void**)&d, out_bytes + 256, st0));
        int* d_flag = reinterpret_cast<int*>(d + out_bytes);
        CU(cudaMemsetAsync(d_flag, 0, sizeof(int), st0));
        launch_tonemap(mf.parts[0], true, n_px, cam->toon_map, reinterpret_cast<uint8_t*>(d), d_flag, st0);
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(rgb, d, (size_t)n_px * 3, cudaMemcpyDeviceToHost, st0));
        int flag = 0;
        CU(cudaMemcpyAsync(&flag, d_flag, sizeof(int), cudaMemcpyDeviceToHost, st0));
        CU(cudaStreamSynchronize(st0));
        if (flag) rc = set_err(RT_ERR_INVALID, "NaN radiance in the image (utils/color.rs:28 asserts)");
        if (stats) stats->kernel_launches += 1;
    } catch (const CudaFail& f) {
        rc = set_err(RT_ERR_CUDA, f.what);
    }
    if (d) cudaFreeAsync(d, st0);
    return rc;
}

int rt_tonemap(const void* accum, uint32_t accum_type, uint64_t n_pixels, uint32_t toon_map, uint8_t* rgb) {
    if (!accum || !rgb) return set_err(RT_ERR_INVALID, "null argument");
    int device, sms;
    int rc = check_device(-1, device, sms);
    if (rc != RT_OK) return rc;
    keep_pool_memory(device);
    const size_t in_bytes = ((size_t)n_pixels * 3 * (accum_type == RT_ACCUM_F64 ? 8 : 4) + 255) & ~size_t(255);
    const size_t out_bytes = ((size_t)n_pixels * 3 + 255) & ~size_t(255);
    char* d = nullptr;
    cudaStream_t st = cudaStreamPerThread;
    try {
        CU(cudaMallocAsync((void**)&d, in_bytes + out_bytes + 256, st));
        int* d_flag = reinterpret_cast<int*>(d + in_bytes + out_bytes);
        CU(cudaMemsetAsync(d_flag, 0, sizeof(int), st));
        CU(cudaMemcpyAsync(d, accum, (size_t)n_pixels * 3 * (accum_type == RT_ACCUM_F64 ? 8 : 4), cudaMemcpyHostToDevice, st));
        launch_tonemap(d, accum_type == RT_ACCUM_F64, n_pixels, toon_map, reinterpret_cast<uint8_t*>(d + in_bytes), d_flag, st);
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(rgb, d + in_bytes, (size_t)n_pixels * 3, cudaMemcpyDeviceToHost, st));
        int flag = 0;
        CU(cudaMemcpyAsync(&flag, d_flag, sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        if (flag) rc = set_err(RT_ERR_INVALID, "NaN radiance in the image (utils/color.rs:28 asserts)");
    } catch (const CudaFail& f) {
        rc = set_err(RT_ERR_CUDA, f.what);
    }
    if (d) cudaFreeAsync(d, st);
    return rc;
}

int rt_tonemap_device(const void* d_accum, uint32_t accum_type, uint64_t n_pixels, uint32_t toon_map, uint8_t* d_rgb, void* stream) {
    if (!d_accum || !d_rgb) return set_err(RT_ERR_INVALID, "null argument");
    int device, sms;
    int rc = check_device(-1, device, sms);
    if (rc != RT_OK) return rc;
    keep_pool_memory(device);
    cudaStream_t st = (cudaStream_t)stream;
    int* d_flag = nullptr;
    try {
        CU(cudaMallocAsync((void**)&d_flag, 256, st));
        CU(cudaMemsetAsync(d_flag, 0, sizeof(int), st));
        launch_tonemap(d_accum, accum_type == RT_ACCUM_F64, n_pixels, toon_map, d_rgb, d_flag, st);
        CU(cudaGetLastError());
        int flag = 0;
        CU(cudaMemcpyAsync(&flag, d_flag, sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        if (flag) rc = set_err(RT_ERR_INVALID, "NaN radiance in the image (utils/color.rs:28 asserts)");
    } catch (const CudaFail& f) {
        rc = set_err(RT_ERR_CUDA, f.what);
    }
    if (d_flag) cudaFreeAsync(d_flag, st);
    return rc;
}

}  // extern "C"
