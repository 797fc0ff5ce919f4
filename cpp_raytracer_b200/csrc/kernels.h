// kernels.h -- launch interface between the C ABI (api.cu) and the kernels (kernels.cu).
#pragma once
#include <cstdint>
#include <type_traits>
#include <cuda_runtime.h>

#include "shade.cuh"

namespace b200rt {

// Threads per block of the path kernels = pixels per tile of the work pool.  Measured with the pool (B200, 128 spp,
// gpurun_out/r2_variants*.txt -> profiles/r2_tile_shape.md): 8 x 8 / 8 x 16 / 8 x 32 / 8 x 64 / 8 x 128 tiles give
// C2 4020 / 4104 / 4135 / 4134 / 4171 and C4b 3243 / 3384 / 3580 / 3576 / 3629 Mpaths/s; 16- and 32-wide tiles are
// slower than 8-wide ones of the same size (the 32 consecutive items a warp holds form an 8 x 4 pixel patch).
#ifndef B200RT_PATH_BLOCK
#define B200RT_PATH_BLOCK 256
#endif
#ifndef B200RT_TILE_W
#define B200RT_TILE_W 8
#endif
constexpr int kPathBlock = B200RT_PATH_BLOCK;       // threads per block of the path kernels = pixels per tile
constexpr int kPathTileW = B200RT_TILE_W;           // tile = kPathTileW x (kPathBlock / kPathTileW) pixels
constexpr int kPathTileH = kPathBlock / kPathTileW;
static_assert(kPathBlock % kPathTileW == 0 && kPathBlock % 32 == 0, "tile shape");
// Tile columns and tiles of a w x h image (tile t is column t % path_tiles_x(w), row t / path_tiles_x(w)).
__host__ __device__ __forceinline__ uint32_t path_tiles_x(uint32_t w) { return (w + (uint32_t)kPathTileW - 1u) / (uint32_t)kPathTileW; }
__host__ __device__ __forceinline__ uint32_t path_tiles(uint32_t w, uint32_t h) {
    return path_tiles_x(w) * ((h + (uint32_t)kPathTileH - 1u) / (uint32_t)kPathTileH);
}
#ifdef B200RT_PATH_MINB
constexpr int kPathMinBlocks = B200RT_PATH_MINB;    // occupancy experiments
#else
constexpr int kPathMinBlocks = 1024 / kPathBlock;   // 1024 threads = 32 warps per SM at 64 registers
#endif
constexpr uint32_t kRenderAccumulate = 2u;    // == B200RT_FLAG_ACCUMULATE
constexpr uint32_t kRenderThreadPixels = 16u; // == B200RT_FLAG_THREAD_PIXELS
constexpr uint32_t kMaxSamplesPerLaunch = 1u << 22;   // tile items (up to 1024 pixels x samples, + one group) are counted in 32 bits
// Second-moment plane (path_megakernel_pool in PathMode::Moments): the sum of x^2 per pixel and channel is kept in 64-bit
// fixed point of 2^-24 units -- per-sample resolution 6.0e-8, range +-5.5e11 per pixel per launch.  At most 2^16 samples
// per launch, so a mean x^2 of up to 8.4e6 per sample (x up to about 2900) fits; the brightest emitter of the scene
// set (500 x 0.8) gives x^2 <= 1.6e5.
constexpr uint32_t kMaxSamplesPerLaunchMoments = 1u << 16;
// What a launch of the tile-pool path kernel writes (launch_path_megakernel).
enum class PathMode { Plain, Counters, Moments, Adaptive };

struct RenderParams {
    DeviceScene scene;
    CameraParams cam;
    unsigned long long seed;
    uint32_t sample_begin, sample_count;
    float *out;                        // image_h x image_w x 3
    float scale;                       // 1 (sum) or 1/sample_count (mean)
    uint32_t flags;
    unsigned long long *counters;      // [0] rays, [1] node visits, [2] primitive tests, [3] of which quad tests
    uint32_t group_shift;              // work-pool item order: 2^group_shift consecutive items are samples of one pixel
    float *out_m2;                     // moments launches only: image_h x image_w x 3, mean (or sum) of x^2; last, so that
                                       // the fields above keep their parameter offsets
    // Tail of the tile-pool grid (path_megakernel_pool): blocks [0, tail_first) render whole tiles; with tail_chunks > 0,
    // each of the remaining tiles is split into tail_chunks blocks of tail_chunk_samples samples (the last one ragged),
    // which sum into tail_acc and let the last of them to arrive write the pixels.  tail_chunks = 0: whole tiles only.
    uint32_t tail_first, tail_chunks, tail_chunk_samples;
    long long *tail_acc;               // per tail tile: kPathBlock x 3 sums (x 2 with moments), zero between launches
    uint32_t *tail_arrivals;           // per tail tile: chunk blocks done, zero between launches
    // Adaptive launches only (b200rt_render_adaptive): block b renders tile ad_list[b] (its tail chunks: the entries from
    // tail_first on), only the pixels whose bit is set in that tile's ad_mask words, and adds its sums into ad_planes.
    const uint32_t *ad_list;
    uint32_t ad_n_list;
    const uint32_t *ad_mask;
    long long *ad_planes;
};
// Adaptive sampling (b200rt_render_adaptive).  Per tile: kAdaptiveMaskWords 32-bit words, bit lp = tile pixel lp (pool
// numbering, kernels.cu map_tile).  Per pixel: 6 int64 sums -- radiance in 2^-30 units, then x^2 in 2^-24 units, as the
// moments kernel keeps them in shared memory -- and a uint32 sample count.
constexpr int kAdaptiveMaskWords = kPathBlock / 32;
constexpr int kAdaptivePlanes = 6;
struct AdaptiveState {
    uint32_t w, h;
    uint32_t *list;                    // this pass's active tiles
    uint32_t n_list;
    uint32_t *mask;                    // active pixels
    uint32_t *unconv;                  // pixels not converged at their current count (zero outside the pass's tiles)
    const long long *planes;
    uint32_t *counts;
    uint32_t *next_list;               // the next pass's active tiles ...
    uint32_t *totals;                  // ... [0] how many, [1] their active pixels; zero before adaptive_decide
    double rel_noise, abs_noise;
};
// Every pixel active, list = all tiles (tiles x kPathBlock threads).
cudaError_t launch_adaptive_init(const AdaptiveState &A, uint32_t tiles, cudaStream_t st);
// After a pass that took the active pixels to n samples: their counts become n and, with judge, their unconverged bits
// are set from the convergence rule (b200rt.h).
cudaError_t launch_adaptive_judge(const AdaptiveState &A, uint32_t n, bool judge, const DeviceScene &S, cudaStream_t st);
// A pixel stays active if any pixel of its 3 x 3 neighbourhood is unconverged; writes the next list and totals.
cudaError_t launch_adaptive_decide(const AdaptiveState &A, const DeviceScene &S, cudaStream_t st);
// planes + counts -> the output planes (mean, or with sum the sums) and nothing else.
cudaError_t launch_adaptive_finish(const AdaptiveState &A, bool sum, float *out_rgb, float *out_m2, cudaStream_t st);
// Scratch of a launch with `tail_tiles` chunked tail tiles: tail_acc, then tail_arrivals.
size_t tail_scratch_bytes(uint32_t tail_tiles, bool moments);
// Path blocks of the tile-pool kernel resident on the current device at once (occupancy x SM count).
cudaError_t path_resident_blocks(int stack, PathMode mode, bool leaf_first, int sm_count, int *blocks);
#ifdef B200RT_BLOCK_TIMES
cudaError_t set_block_times(unsigned long long *buf, uint32_t n_blocks);   // diagnostic build: see kernels.cu
#endif

// Path-slot pool of the wavefront variant (wavefront.cu); all pointers are device memory.
// One slot = one 128-byte line, read and written with 16-byte vector accesses.
struct alignas(128) PathSlot {
    double ox, oy, oz, dx, dy, dz;   //  0: the ray (direction not normalised)
    double hit_t;                    // 48: closest hit of the last trace ...
    uint32_t hit_ref;                // 56: ... and its primitive reference (kNoHit on a miss)
    uint32_t pixel;                  // 60: pixel index; 0xFFFFFFFF = dead slot
    float tr, tg, tb;                // 64: path throughput
    uint32_t sample;                 // 76
    uint32_t bounce;                 // 80
    uint32_t cls;                    // 84: material class of the last hit (queue it was sorted into)
    uint32_t pad[10];
};
static_assert(sizeof(PathSlot) == 128, "PathSlot must be one 128-byte line");

struct WavefrontPool {
    uint32_t n_slots;
    unsigned long long total_items;     // image_w * image_h * samples of this call
    PathSlot *slots;
    uint32_t *queue;                    // 5 class queues of n_slots entries each
    uint32_t *queue_count;              // [5]
    uint32_t *alive;
    unsigned long long *next_item;
};
size_t wavefront_pool_alloc_bytes(uint32_t n_slots);
void wavefront_pool_layout(void *base, uint32_t n_slots, WavefrontPool &W);
cudaError_t run_wavefront(int stack, const RenderParams &P, const WavefrontPool &W, bool count, cudaStream_t st, int sm_count,
                          unsigned long long *launches);

// `stack` = traversal stack entries the scene needs (3 x depth of the 4-wide tree); the
// launchers pick the smallest instantiation that fits (32 / 64 / 128): with_stack calls f with it as a compile-time constant.
template <typename F>
auto with_stack(int stack, F &&f) {
    if (stack <= 32) return f(std::integral_constant<int, 32>{});
    if (stack <= 64) return f(std::integral_constant<int, 64>{});
    return f(std::integral_constant<int, 128>{});
}
cudaError_t launch_raycast(int stack, const DeviceScene &S, const double *rays, long long n, double tmin, double tmax,
                           int32_t *prim, double *t, cudaStream_t st);
// The path kernel of a render.  mode: what the tile-pool kernel writes besides the image --
//   Counters  also the traversal counters P.counters[1..3]
//   Moments   also the second-moment plane P.out_m2 (at most kMaxSamplesPerLaunchMoments samples per launch)
//   Adaptive  both sums of the active pixels of the tiles in P.ad_list into P.ad_planes, instead of the image
// Plain and Counters run the thread-owns-pixel kernel under kRenderThreadPixels.  leaf_first: order of the two steps
// inside one iteration of the traversal loop (see closest_hit).
cudaError_t launch_path_megakernel(int stack, const RenderParams &P, PathMode mode, bool leaf_first, cudaStream_t st);
// measurement only: 16 lane-accounting counters (see path_lanes_kernel)
cudaError_t launch_path_lanes(int stack, const RenderParams &P, unsigned long long *acc, bool leaf_first, cudaStream_t st);
cudaError_t launch_finalize(float *frame, long long n_pixels, float scale, int32_t *ldr, int clamp, cudaStream_t st);
cudaError_t launch_tonemap(const float *hdr, long long n_pixels, int32_t *out, int clamp, cudaStream_t st);
cudaError_t launch_debug_camera(const CameraParams &C, const uint32_t *pixels, const uint32_t *rnd, long long n, double *rays_out,
                                cudaStream_t st);
cudaError_t launch_debug_philox(const uint32_t *in, long long n, uint32_t *out, cudaStream_t st);
cudaError_t launch_debug_samplers(const uint32_t *rnd, long long n, double *sphere_out, double *disk_out, cudaStream_t st);
// records: n x 88-byte ShadeRecord (kernels.cu)
cudaError_t launch_debug_shade(int stack, const DeviceScene &S, const double *rays, const uint32_t *rnd, long long n, double tmin,
                               double tmax, void *records, cudaStream_t st);

// Peer-memory frame exchange (multi-GPU): per-rank sum buffers addressed from this GPU.
constexpr int kMaxPeers = 16;
struct PeerFrames { const float *p[kMaxPeers]; };
void peer_slice(long long n_pixels, int n_peers, int rank, long long *lo, long long *hi);
// frame += other (multi-GPU exchange without peer mapping: the root adds the copied per-device frames in order)
cudaError_t launch_add_frame(float *frame, const float *other, long long n_floats, cudaStream_t st);
cudaError_t launch_reduce_finalize_peers(const PeerFrames &in, int n_peers, int rank, long long n_pixels, float scale,
                                         float *root_hdr, int32_t *root_ldr, int clamp, cudaStream_t st);

}  // namespace b200rt
