// kernels.h — state shared between the kernels (kernels.cu) and the C ABI driver (api.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "rt2025.h"
#include "scene_types.h"

namespace rt {

// one CTA per SM: its shared memory holds the top of the BVH (all of it for small scenes) + the stacks
#ifndef RT_EXTEND_BLOCK
#define RT_EXTEND_BLOCK 512
#endif
#ifndef RT_EXTEND_MIN_BLOCKS
#define RT_EXTEND_MIN_BLOCKS 1
#endif
constexpr int EXTEND_BLOCK = RT_EXTEND_BLOCK;
constexpr int EXTEND_MIN_BLOCKS = RT_EXTEND_MIN_BLOCKS;
constexpr size_t EXTEND_SMEM_MAX = 227 * 1024;
constexpr int SHADE_BLOCK = 256;
constexpr int MEDIA_BLOCK = 256;
#ifndef RT_REFILL_MIN
#define RT_REFILL_MIN 32  // SceneView::refill_min default (traverse.cuh, trace_persistent)
#endif
constexpr int REFILL_MIN = RT_REFILL_MIN;
#ifndef RT_SLAB_SIGNSEL
#define RT_SLAB_SIGNSEL 1  // slab test: near/far planes picked by the sign of 1/d, error bound folded into the addend
#endif
#ifndef RT_RAY_SMEM
#define RT_RAY_SMEM 0  // persistent traversal: the binary64 ray lives in shared memory instead of 28 registers (traverse.cuh)
#endif
constexpr size_t EXTEND_RAY_SMEM_BYTES = RT_RAY_SMEM ? (size_t)14 * sizeof(double) * RT_EXTEND_BLOCK : 0;
#ifndef RT_PARK_VOTE
#define RT_PARK_VOTE 1  // postponed leaves: leave the node loop as soon as every lane of the warp holds a leaf (0: only at a second leaf)
#endif
#ifndef RT_LDG256
#define RT_LDG256 1  // 256-bit global loads for nodes and primitive records
#endif
#ifndef RT_SHADE_SIDE_STREAMS
#define RT_SHADE_SIDE_STREAMS 2  // side streams the per-class shade kernels are dealt over (0: all on the render stream)
#endif
#ifndef RT_MEDIA_MIN_BLOCKS
#define RT_MEDIA_MIN_BLOCKS 2
#endif
#ifndef RT_MEDIA_MIN_BLOCKS_NOXF
#define RT_MEDIA_MIN_BLOCKS_NOXF 3
#endif
#ifndef RT_MEDIA_GENERIC_MIN_BLOCKS
#define RT_MEDIA_GENERIC_MIN_BLOCKS 2
#endif
#ifndef RT_MEDIA_BLOCK_AGG
#define RT_MEDIA_BLOCK_AGG 0
#endif
#ifndef RT_MEDIA_TWO_PHASE
#define RT_MEDIA_TWO_PHASE 1
#endif
#ifndef RT_MEDIA_EARLY_SCREEN
#define RT_MEDIA_EARLY_SCREEN 1
#endif
#ifndef RT_SHADE_3BLOCK_MASK
#define RT_SHADE_3BLOCK_MASK 0x73u  // shade classes compiled for three CTAs per SM (85 registers) instead of RT_SHADE_MIN_BLOCKS
#endif
#ifndef RT_SHADE_PREFETCH
#define RT_SHADE_PREFETCH 0  // 1: k_shade prefetches the next round's gathered records into L2 (measured: book2 shade 30.1 -> 30.7 ms, cornell 25.9 -> 26.4: off)
#endif
#ifndef RT_SHADE_MIN_BLOCKS
#define RT_SHADE_MIN_BLOCKS 2
#endif

constexpr uint8_t CLASS_DROPPED = 0xFF;  // cls_q: the path ended in extend, no shade kernel reads the entry
enum HitKind : uint32_t { HIT_MISS = 0, HIT_SURFACE = 1, HIT_MEDIUM = 2 };

// The wavefront state is a set of dense streams indexed by QUEUE POSITION (no per-path slots):
//   ray_q[2]   64 B  o(3) d(3) time + the packed path ids    read by extend/media/shade, written by shade/generate
//   beta_q[2]  32 B  throughput(3) + 8 spare bytes           read by shade, written by shade/generate
//   hit_q      16 B  t, kind, primitive                      written by extend, updated by the media pass, read by shade
//   cls_q       1 B  shade class of the winner               written by extend (or the media pass), read by the binning pass
// The two copies of ray_q/beta_q alternate every iteration (`parity`): shade reads position p of the
// current copy and appends survivors to the other one, generate tops that one up with camera rays.
// Round 1 kept the ids in a 48-byte state record next to the throughput: the media pass and extend then read
// 48 (64 with sector granularity) bytes for 12 bytes of ids, and every stage re-read the ray record.  With the ids
// in the ray record's spare 8 bytes, extend - which now also samples the media while it prepares the ray - reads
// 64 bytes per segment and writes 17; the throughput is touched by shade alone.
struct alignas(16) RayRec {
    double w[7];
    uint64_t ids;  // pack_ids(pixel, sample, segment)
};
struct alignas(16) BetaRec {
    double beta[3];
    double spare;
};
struct alignas(16) HitRec {
    double t;
    uint32_t kind, prim;
};
static_assert(sizeof(RayRec) == 64 && sizeof(BetaRec) == 32 && sizeof(HitRec) == 16, "stream record sizes");
// path ids: pixel (28 bits) | sample (24 bits) | segment (12 bits); rt_render_device rejects frames beyond these
constexpr uint32_t IDS_PIXEL_BITS = 28, IDS_SAMPLE_BITS = 24, IDS_SEGMENT_BITS = 12;

struct Counters {
    uint32_t n_extend[2];  // entries in ray_q/state_q of each parity
    uint32_t n_shade[SC_COUNT];
    uint32_t n_pixels, pad;  // pad: arrival counter of k_tail's CTAs
    uint32_t n_unsampled, pad3;  // entries [0, n_unsampled) of the current ray stream still need the media sampling pass (the camera
                                 // rays behind them were sampled by k_generate while it had them in registers)
    uint32_t gen_done, walk_cursor;  // arrival counter of k_generate's CTAs; next entry of the SC_WALK queue to be claimed (k_walk)
    unsigned long long next_path, segments, iterations, errors, node_visits, prim_tests;
    unsigned long long walk_segments;  // of `segments`: evaluated inside k_walk (they never went through the streams)
    unsigned long long walk_lean_segments;  // of `walk_segments`: evaluated by the lean variant of k_walk (SceneView::walk_lean)
    unsigned long long shade_lean_hits;     // hits shaded by a lean class kernel (k_shade<CLS, true>, SceneView::shade_lean_mask)
};

struct WavefrontState {
    RayRec* ray_q[2];
    BetaRec* beta_q[2];
    HitRec* hit_q;
    uint8_t* cls_q;  // shade class of every hit
    uint32_t* q_shade[SC_COUNT];
    uint32_t* pixel_list;
    double* accum;  // W*H*3 binary64 sums
    Counters* counters;
    uint32_t capacity, n_pixels;
    uint64_t total_paths;
    uint32_t parity, pad;
};

struct RenderParams {
    rt_camera cam;
    uint64_t seed;
    uint32_t sample_begin, part_index, part_count;
    uint32_t lights_flat, bin_by_class;
    uint32_t walk_drain_queue, walk_drain_steps;  // k_walk: queues of at most walk_drain_queue entries cut every walk after walk_drain_steps segments
    uint32_t drop_misses;  // the background is a solid (0, 0, 0): a path that misses everything ends in extend (class byte CLASS_DROPPED)
    uint32_t sample_in_generate;  // media_first == 1: k_generate samples the media for the camera rays it writes (A/B knob RT2025_GEN_MEDIA=0)
    uint32_t media_first;  // 0: media sampled after extend (order of Hittables::hit); 1: by a pass ahead of extend, 2: by extend itself while it
                           // prepares the ray - extend then only looks for surfaces up to the scatter point
};

void launch_closest_hit(const SceneView& sv, const rt_ray* d_rays, uint32_t n, double tmin, double tmax, bool count, rt_hit* d_out,
                        unsigned long long* d_counters, int grid, size_t smem_bytes, cudaStream_t stream);
// d_out[i] = 1 when a surface hit lies in [tmin, d_tmax_per_ray ? d_tmax_per_ray[i] : tmax]; the same variant as launch_closest_hit
void launch_occluded(const SceneView& sv, const rt_ray* d_rays, const double* d_tmax_per_ray, uint32_t n, double tmin, double tmax, bool count,
                     uint8_t* d_out, unsigned long long* d_counters, int grid, size_t smem_bytes, cudaStream_t stream);
// The media pass of rt_transmittance, after launch_occluded wrote d_occluded: d_out[i] = 0 for an occluded ray, else the product
// of exp(L / neg_inv_density) over the media on [tmin, t_max_i] (1 for an empty interval).  generic: some boundary is not a single
// Sphere.  `grid` CTAs of MEDIA_BLOCK threads.
void launch_transmittance(const SceneView& sv, bool generic, const rt_ray* d_rays, const double* d_tmax_per_ray, uint32_t n, double tmin, double tmax,
                          bool count, const uint8_t* d_occluded, double* d_out, unsigned long long* d_counters, int grid, cudaStream_t s);
// The two passes of rt_world_hit.  Surface: d_out[i] = the closest surface hit on [tmin, t_max_i] as a HitRec (internal primitive,
// kind HIT_SURFACE or HIT_MISS; an empty interval is a miss); the same variant as launch_closest_hit.  Record: every medium competes
// with that hit on the caller's interval, drawing philox(seed; i, 0, segment, RT_MEDIUM_SLOT(m)), and the winner's record goes to
// d_out; generic as in launch_transmittance, `grid` CTAs of MEDIA_BLOCK threads.
void launch_world_hit_surface(const SceneView& sv, const rt_ray* d_rays, const double* d_tmax_per_ray, uint32_t n, double tmin, double tmax, bool count,
                              HitRec* d_out, unsigned long long* d_counters, int grid, size_t smem_bytes, cudaStream_t stream);
void launch_world_hit_record(const SceneView& sv, bool generic, const rt_ray* d_rays, const double* d_tmax_per_ray, uint32_t n, double tmin,
                             double tmax, uint64_t seed, uint32_t segment, bool count, const HitRec* d_surface, rt_hit_record* d_out,
                             unsigned long long* d_counters, int grid, cudaStream_t s);
// rt_shade: the render's step after world.hit (shade_hit<SC_OTHER>, end_segment) for every row of d_state with RT_PATH_ALIVE,
// from its rt_hit_record; *d_errors (may be nullptr) gets the rows that end with RT_PATH_ERROR.  `grid` CTAs of SHADE_BLOCK threads.
void launch_shade_records(const SceneView& sv, const RenderParams& P, const rt_hit_record* d_records, uint64_t n, uint32_t n_materials,
                          uint32_t segment, rt_ray* d_rays, double* d_beta, double* d_radiance, uint8_t* d_state, unsigned long long* d_errors,
                          int grid, cudaStream_t s);
// rt_camera_rays: d_out[pixel] = Camera::get_ray of stratum `sample` (k_generate's camera_ray), `grid` CTAs of 256 threads
void launch_camera_rays(const rt_camera& cam, uint64_t seed, uint32_t sample, uint64_t n, rt_ray* d_out, int grid, cudaStream_t s);
// The path-id forms (rt_world_hit_ids, rt_shade_ids, rt_camera_rays_ids): as the three above, with the draws of row i addressed by
// d_ids[i] = (pixel, sample, segment).  launch_shade_records_ids takes each row's segment from d_ids (a row at segment >= max_depth
// ends with RT_PATH_ERROR) and adds one to it on the rows that go on.  launch_camera_rays_ids writes d_out[i] for i < n.
void launch_world_hit_record_ids(const SceneView& sv, bool generic, const rt_ray* d_rays, const double* d_tmax_per_ray, uint32_t n, double tmin,
                                 double tmax, uint64_t seed, const rt_path_id* d_ids, bool count, const HitRec* d_surface, rt_hit_record* d_out,
                                 unsigned long long* d_counters, int grid, cudaStream_t s);
void launch_shade_records_ids(const SceneView& sv, const RenderParams& P, const rt_hit_record* d_records, uint64_t n, uint32_t n_materials,
                              rt_path_id* d_ids, rt_ray* d_rays, double* d_beta, double* d_radiance, uint8_t* d_state, unsigned long long* d_errors,
                              int grid, cudaStream_t s);
void launch_camera_rays_ids(const rt_camera& cam, uint64_t seed, const rt_path_id* d_ids, uint64_t n, rt_ray* d_out, int grid, cudaStream_t s);
void launch_init(const WavefrontState& W, const RenderParams& P, int grid, cudaStream_t s);
void launch_generate(const SceneView& sv, const RenderParams& P, const WavefrontState& W, int grid, cudaStream_t s);
void launch_extend(const SceneView& sv, const RenderParams& P, const WavefrontState& W, bool count, int grid, size_t smem_bytes, cudaStream_t s);
// phase 0: media sampling after extend (classic order / general boundaries) + binning; phase 1: the sampling pass ahead of extend;
// phase 2: binning only (extend wrote the class bytes)
int launch_media_bin(const SceneView& sv, const RenderParams& P, const WavefrontState& W, bool count, bool generic, int grid, cudaStream_t s, int phase);
struct ShadeFan {  // side streams for the per-class shade kernels (owned by the workspace)
    int n_side = 0;
    cudaStream_t side[3] = {};
    cudaEvent_t fork = nullptr, join[3] = {};
};
int launch_shade(const SceneView& sv, const RenderParams& P, const WavefrontState& W, uint32_t class_mask, int grid, cudaStream_t s,
                 const ShadeFan* fan, bool tail_follows, int walk_grid);
// partial framebuffers of a multi-GPU render, as GPU 0 sees them (peer-mapped pointers for the other GPUs)
constexpr uint32_t MAX_PARTS = 16;
struct PartList {
    const void* p[MAX_PARTS];
    uint32_t n;
};
// out[i] = sum over parts of p[k][i] (out may be parts.p[0])
void launch_sum_parts(const PartList& parts, void* out, uint64_t n_values, bool f64, int grid, cudaStream_t s);
// finishes the frame in one launch once generation is over and at most `threshold` paths are left (kernels.cu, k_tail); a no-op otherwise
void launch_tail(const SceneView& sv, const RenderParams& P, const WavefrontState& W, uint32_t threshold, int grid, cudaStream_t s);
void launch_finalize(const double* accum, uint64_t n, double scale, void* out, bool out_f64, int grid, cudaStream_t s);
void launch_tonemap(const void* accum, bool f64, uint64_t n_pixels, uint32_t toon_map, uint8_t* rgb, int* error_flag, cudaStream_t s);
int kernel_setup(size_t smem_bytes, int* extend_blocks_per_sm, int* shade_blocks_per_sm, int* walk_blocks_per_sm);

}  // namespace rt
