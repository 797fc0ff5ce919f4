// kernels.cu -- the CUDA kernels behind the C ABI (sm_100a only; compiled with -fmad=false so
// FP64 primitive tests reproduce the reference's unfused arithmetic bit for bit).
//
//   raycast_kernel        one thread per ray, closest hit -> (canonical prim index, t)
//                         [BVH::hit_by / Scene::hit_by, reference bvh.h:585-715, scene.h:59-75]
//   path_megakernel_pool  the default path kernel: a block's lanes take its tile's (pixel, sample) items from a pool
//                         [Camera::render<T> + ray_color, reference camera.h:205-297; the rules of a path: path.cuh]
//   path_megakernel       the thread-owns-pixel form (B200RT_FLAG_THREAD_PIXELS): one thread per pixel, all its samples
//   tonemap_kernel        Reinhard + gamma 2 + int(255.999999 v)   [RGB::as_string, rgb.h:90-113]
#include <type_traits>

#include "kernels.h"
#include "path.cuh"

namespace b200rt {

// ------------------------------------------------------------------------------------------
template <int STACK>
__global__ void __launch_bounds__(128) raycast_kernel(DeviceScene S, const double *__restrict__ rays, long long n,
                                                      double tmin, double tmax, int32_t *__restrict__ prim_out,
                                                      double *__restrict__ t_out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double *r = rays + i * 6;
    const Hit h = closest_hit<STACK, false>(S, r[0], r[1], r[2], r[3], r[4], r[5], tmin, tmax, nullptr);
    if (h.ref == kNoHit) {
        prim_out[i] = -1;
        t_out[i] = 0.0;
    } else {
        prim_out[i] = (int32_t)canonical_prim(S, h.ref);
        t_out[i] = h.t;
    }
}

// One surface interaction per ray with the CALLER's random words: closest hit, then shade_hit -- the very
// device function the path kernels call -- on a unit throughput.  Test hook (b200rt_debug_shade): makes the
// hit_info face rule and the four materials checkable ray by ray against the oracle's reflected / refracted /
// reflectance, which the path kernels' own Philox streams do not allow.
struct ShadeRecord {
    double scattered[6];   // origin, direction of the scattered ray (zeros if the path ended)
    double t;
    float atten[3];        // throughput after the interaction (the material's attenuation)
    float emit[3];         // emitted radiance picked up at the hit
    int32_t prim;          // canonical primitive index or -1
    int32_t flags;         // bit 0: a scattered ray continues
};
static_assert(sizeof(ShadeRecord) == 88, "ShadeRecord is mirrored by numpy in capi.py");

// Primary rays for given pixels with the CALLER's random words (test hook b200rt_debug_camera_rays): the
// kernels' camera_ray, checkable against Camera::random_ray_through_pixel draw for draw.
__global__ void debug_camera_kernel(const __grid_constant__ CameraParams C, const uint32_t *__restrict__ pixels,
                                    const uint32_t *__restrict__ rnd, long long n, double *__restrict__ rays_out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Philox4 w{rnd[i * 4 + 0], rnd[i * 4 + 1], rnd[i * 4 + 2], rnd[i * 4 + 3]};
    Ray r;
    PathState p;
    camera_ray(C, pixels[i * 2 + 0], pixels[i * 2 + 1], w, r, p);
    double *o = rays_out + i * 6;
    o[0] = r.ox; o[1] = r.oy; o[2] = r.oz; o[3] = r.dx; o[4] = r.dy; o[5] = r.dz;
}

// Test hooks (b200rt_debug_philox / b200rt_debug_samplers): the generator and the direction samplers exactly as the
// path kernels call them, on caller-supplied inputs.
__global__ void debug_philox_kernel(const uint32_t *__restrict__ in, long long n, uint32_t *__restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Philox4 r = philox4x32_10(in[i * 6 + 0], in[i * 6 + 1], in[i * 6 + 2], in[i * 6 + 3], in[i * 6 + 4], in[i * 6 + 5]);
    out[i * 4 + 0] = r.x; out[i * 4 + 1] = r.y; out[i * 4 + 2] = r.z; out[i * 4 + 3] = r.w;
}
__global__ void debug_samplers_kernel(const uint32_t *__restrict__ rnd, long long n, double *__restrict__ sphere_out,
                                      double *__restrict__ disk_out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double x, y, z;
    sample_unit_sphere(u01(rnd[i * 2 + 0]), u01(rnd[i * 2 + 1]), x, y, z);
    sphere_out[i * 3 + 0] = x; sphere_out[i * 3 + 1] = y; sphere_out[i * 3 + 2] = z;
    double ax, ay;
    sample_unit_disk(u01(rnd[i * 2 + 0]), u01(rnd[i * 2 + 1]), ax, ay);
    disk_out[i * 2 + 0] = ax; disk_out[i * 2 + 1] = ay;
}

template <int STACK>
__global__ void __launch_bounds__(128) debug_shade_kernel(DeviceScene S, const double *__restrict__ rays,
                                                          const uint32_t *__restrict__ rnd, long long n, double tmin, double tmax,
                                                          ShadeRecord *__restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Ray r{rays[i * 6 + 0], rays[i * 6 + 1], rays[i * 6 + 2], rays[i * 6 + 3], rays[i * 6 + 4], rays[i * 6 + 5]};
    const Hit h = closest_hit<STACK, false>(S, r.ox, r.oy, r.oz, r.dx, r.dy, r.dz, tmin, tmax, nullptr);
    ShadeRecord rec{};
    rec.prim = -1;
    if (h.ref != kNoHit) {
        const Philox4 w{rnd[i * 4 + 0], rnd[i * 4 + 1], rnd[i * 4 + 2], rnd[i * 4 + 3]};
        PathState p{1.0f, 1.0f, 1.0f};
        float er = 0.0f, eg = 0.0f, eb = 0.0f;
        const bool cont = shade_hit(S, h, w, r, p, er, eg, eb);
        rec.prim = (int32_t)canonical_prim(S, h.ref);
        rec.t = h.t;
        rec.flags = cont ? 1 : 0;
        if (cont) {
            rec.scattered[0] = r.ox; rec.scattered[1] = r.oy; rec.scattered[2] = r.oz;
            rec.scattered[3] = r.dx; rec.scattered[4] = r.dy; rec.scattered[5] = r.dz;
            rec.atten[0] = p.tr; rec.atten[1] = p.tg; rec.atten[2] = p.tb;
        }
        rec.emit[0] = er; rec.emit[1] = eg; rec.emit[2] = eb;
    }
    out[i] = rec;
}

// ------------------------------------------------------------------------------------------
// Thread -> pixel: a block is an 8 x (kPathBlock / 8) pixel tile, each warp an 8x4 sub-tile, so the 32 primary
// rays of a warp are neighbours on the image plane.
struct PixelMap {
    uint32_t px, py, pixel;
    bool valid;
};
__device__ __forceinline__ PixelMap map_pixel(const CameraParams &C) {
    const uint32_t tiles_x = path_tiles_x(C.w);
    const uint32_t tile_x = blockIdx.x % tiles_x, tile_y = blockIdx.x / tiles_x;
    PixelMap m;
    m.px = tile_x * (uint32_t)kPathTileW + (threadIdx.x % (uint32_t)kPathTileW);
    m.py = tile_y * (uint32_t)kPathTileH + (threadIdx.x / (uint32_t)kPathTileW);
    m.valid = m.px < C.w && m.py < C.h;
    m.pixel = m.py * C.w + m.px;
    return m;
}

// A pixel's three channels, times k: stored, or with accumulate added to what is there.
__device__ __forceinline__ void store_rgb(float *o, float r, float g, float b, float k, bool accumulate) {
    if (accumulate) { o[0] += r * k; o[1] += g * k; o[2] += b * k; }
    else { o[0] = r * k; o[1] = g * k; o[2] = b * k; }
}

__device__ __forceinline__ void write_pixel_and_counters(const RenderParams &P, const PixelMap &m, float sum_r, float sum_g,
                                                         float sum_b, uint32_t lane_rays, bool count,
                                                         const TraversalCounters &ctr) {
    if (m.valid && B200RT_CHECK(P.scene, m.pixel < P.cam.w * P.cam.h, 3))
        store_rgb(P.out + (size_t)m.pixel * 3, sum_r, sum_g, sum_b, P.scale, (P.flags & kRenderAccumulate) != 0);
    write_counters(P, lane_rays, count, ctr);
}

// One path segment's worth of "shade + continue or regenerate": consumes the finished traversal
// in T (if any), and leaves either a new ray in `ray` (returns true) or the lane finished.
struct LaneState {
    PathState p;
    Ray ray;
    uint32_t s = 0, bounce = 0;
    bool has_path = false;
    float sum_r = 0.f, sum_g = 0.f, sum_b = 0.f;   // every contribution (throughput x emission / background) is added here directly
    uint32_t rays = 0;
};
__device__ __forceinline__ bool shade_and_advance(const RenderParams &P, const PixelMap &m, const Hit &best, LaneState &L) {
    if (L.has_path) {
        ++L.rays;
        float er, eg, eb;
        // the sums start at +0 and so are never -0: adding the zero contribution of a hit that is not a light changes no bit
        const bool cont = path_bounce(P, best, m.pixel, L.s, L.bounce, L.ray, L.p, er, eg, eb);
        L.sum_r += er; L.sum_g += eg; L.sum_b += eb;
        if (!cont) {
            L.has_path = false;
            ++L.s;
        }
    }
    if (!L.has_path) {
        if (L.s == P.sample_count) return false;
        path_start(P, m.pixel, m.px, m.py, L.s, L.ray, L.p);
        L.bounce = 0;
        L.has_path = true;
    }
    return true;
}

// ------------------------------------------------------------------------------------------
// Tile work pool.  A block owns an 8 x 32 pixel tile (kPathTileW x kPathTileH) but its THREADS do not own pixels: the tile's (pixel, sample) items
// -- sample-major, so that the lanes of a warp work on neighbouring pixels of the same sample at any time -- are handed
// out through a shared-memory counter, and a lane whose path ends takes the next item whatever pixel it belongs to.
// With thread-owns-pixel a lane on a cheap pixel (sky: one ray per path) ran out of samples long before its neighbours
// on glass (five rays per path) and idled for the rest of the warp's life: 12-22 % of all lane-slots of the node and
// leaf steps (profiles/r2_lane_accounting.md).
//   Radiance is summed per pixel in shared memory as 64-bit FIXED POINT (2^-30 units) with integer atomics: integer
// addition is associative, so the sum -- and with it the image -- is bit-deterministic and does not depend on which
// lane rendered which sample, in which order.  One contribution per path (emission at a light, or the background on a
// miss), so three atomics per path at most.  Resolution 9.3e-10, range +-8.6e9 per pixel per launch.
struct TilePool {
    unsigned int next;                 // next (pixel, sample) item of this tile
    unsigned int slot;                 // BlockWork::slot (kept here rather than in a register through the path loop)
    unsigned int last;                 // chunk blocks: this block arrived last and writes the tile
    long long acc[kPathBlock * 3];     // per tile pixel: sum of radiance x 2^30
};
// The moments instantiation's pool: the same, plus the sum of x^2 per pixel and channel in 2^-24 units (range: kernels.h).
struct TilePoolMoments : TilePool {
    long long acc2[kPathBlock * 3];    // per tile pixel: sum of radiance^2 x 2^24
};
// The adaptive instantiation's pool: the moments pool, plus the tile pixels the block renders.  Its items and its
// accumulators are numbered over that list instead of over the tile's valid pixels.
struct TilePoolAdaptive : TilePoolMoments {
    unsigned char act[kPathBlock];     // active tile pixels, ascending
    unsigned int warp_act[kAdaptiveMaskWords];
};
static_assert(kPathBlock <= 256, "TilePoolAdaptive::act holds tile pixels in bytes");
template <bool MOMENTS, bool ADAPTIVE = false>
using TilePoolOf = std::conditional_t<ADAPTIVE, TilePoolAdaptive, std::conditional_t<MOMENTS, TilePoolMoments, TilePool>>;
constexpr float kFixScale = 1073741824.0f;            // 2^30
constexpr double kFixInv = 1.0 / 1073741824.0;
constexpr float kFix2Scale = 16777216.0f;             // 2^24
constexpr double kFix2Inv = 1.0 / 16777216.0;
// A fixed-point sum of radiance (fix_rgb) or of x^2 (fix_x2) as the float every reader of the sums starts from: the image
// and the second-moment plane (store_tile_pixel), the adaptive rule (pixel_converged) and the adaptive output planes
// (adaptive_finish_kernel).  So a pixel an adaptive render stops at n samples has the bits of an n-sample render_moments.
__device__ __forceinline__ float fix_rgb(long long a) { return (float)((double)a * kFixInv); }
__device__ __forceinline__ float fix_x2(long long q) { return (float)((double)q * kFix2Inv); }

struct TileMap {
    uint32_t x0, y0, vw, n_valid;      // tile origin, valid width, valid pixel count (edge tiles are ragged)
};
// Image column and row of tile pixel lt.
__device__ __forceinline__ uint2 tile_xy(const TileMap &tm, uint32_t lt) { return make_uint2(tm.x0 + lt % tm.vw, tm.y0 + lt / tm.vw); }
__device__ __forceinline__ TileMap map_tile(const CameraParams &C, uint32_t tile) {
    const uint32_t tiles_x = path_tiles_x(C.w);
    const uint32_t tile_x = tile % tiles_x, tile_y = tile / tiles_x;
    TileMap t;
    t.x0 = tile_x * (uint32_t)kPathTileW;
    t.y0 = tile_y * (uint32_t)kPathTileH;
    t.vw = min((uint32_t)kPathTileW, C.w - t.x0);
    t.n_valid = t.vw * min((uint32_t)kPathTileH, C.h - t.y0);
    return t;
}

// What one block of path_megakernel_pool renders: all samples of a tile, or -- in the tail of the grid -- one chunk
// [s_begin, s_end) of a tail tile's samples.  The last whole tiles drain while the short chunk blocks that follow them
// in the grid keep the SMs full, so a frame no longer ends on a partly idle GPU.  Nothing depends on the order in which
// the hardware starts blocks.
struct BlockWork {
    uint32_t tile, s_begin, s_end;
    uint32_t slot;                     // tail-tile ordinal, or kWholeTile
};
constexpr uint32_t kWholeTile = 0xFFFFFFFFu;
__device__ __forceinline__ BlockWork block_work(const RenderParams &P) {
    BlockWork w{blockIdx.x, 0u, P.sample_count, kWholeTile};
    if (P.tail_chunks && blockIdx.x >= P.tail_first) {
        const uint32_t j = blockIdx.x - P.tail_first;
        w.slot = j / P.tail_chunks;
        w.tile = P.tail_first + w.slot;
        w.s_begin = (j - w.slot * P.tail_chunks) * P.tail_chunk_samples;
        w.s_end = min(w.s_begin + P.tail_chunk_samples, P.sample_count);
    }
    return w;
}

// The block's (pixel, sample) items in pool_fetch's numbering: [*first, return value).  A chunk starts, and unless it is
// the last one also ends, on a multiple of 2^group_shift samples (the host rounds the chunk size), so the item ranges of a
// tile's chunks partition the items of the whole tile and every chunk sees the same (pixel, sample) pairs it would there.
__device__ __forceinline__ uint32_t block_items(const RenderParams &P, const TileMap &tm, const BlockWork &w, uint32_t &first) {
    const uint32_t gs = P.group_shift;
    if (P.cam.max_depth == 0) { first = 0u; return 0u; }
    if (gs == 0u) { first = tm.n_valid * w.s_begin; return tm.n_valid * w.s_end; }
    const uint32_t per_block = tm.n_valid << gs;
    first = per_block * (w.s_begin >> gs);
    return per_block * ((w.s_end + (1u << gs) - 1u) >> gs);
}

struct PoolLane {
    PathState p;
    uint32_t pixel = 0, lp = 0, s = 0, bounce = 0;    // image pixel index, pixel within the tile, sample, bounce
    bool has_path = false;
    uint32_t rays = 0;
};

// (The 64-bit shared-memory atomicAdd compiles to a compare-and-swap loop, ATOMS.CAST.SPIN.64.  Splitting it into two native
//  32-bit atomics with an exact carry -- the thread whose addition wrapped the low word carries into the high one -- was
//  measured 2-5 % SLOWER on all six scenes in a same-box A/B, so the plain form stays.)
//   MOMENTS also sums x^2 per channel.  x^2 of a path is the square of its single non-zero contribution: a path adds
// radiance at exactly one interaction -- the light it hits (DiffuseLight emits and never scatters, so the path ends there,
// material.h:248-263) or the background on a miss -- and zero at every other one.  So squaring each contribution here is
// the square of the path's sample radiance, with no per-lane state.
template <bool MOMENTS = false>
__device__ __forceinline__ void pool_contribute(TilePoolOf<MOMENTS> &tp, uint32_t lp, float r, float g, float b) {
    if (r != 0.0f) atomicAdd(reinterpret_cast<unsigned long long *>(&tp.acc[lp * 3 + 0]), (unsigned long long)__float2ll_rn(r * kFixScale));
    if (g != 0.0f) atomicAdd(reinterpret_cast<unsigned long long *>(&tp.acc[lp * 3 + 1]), (unsigned long long)__float2ll_rn(g * kFixScale));
    if (b != 0.0f) atomicAdd(reinterpret_cast<unsigned long long *>(&tp.acc[lp * 3 + 2]), (unsigned long long)__float2ll_rn(b * kFixScale));
    if constexpr (MOMENTS) {
        if (r != 0.0f) atomicAdd(reinterpret_cast<unsigned long long *>(&tp.acc2[lp * 3 + 0]), (unsigned long long)__float2ll_rn(r * r * kFix2Scale));
        if (g != 0.0f) atomicAdd(reinterpret_cast<unsigned long long *>(&tp.acc2[lp * 3 + 1]), (unsigned long long)__float2ll_rn(g * g * kFix2Scale));
        if (b != 0.0f) atomicAdd(reinterpret_cast<unsigned long long *>(&tp.acc2[lp * 3 + 2]), (unsigned long long)__float2ll_rn(b * b * kFix2Scale));
    }
}

// Takes the tile's next (pixel, sample) item into L (false: none left).  Item order: group_shift = 0: sample-major
// (consecutive items = neighbouring pixels of one sample).  group_shift = g: consecutive items = 2^g samples of the SAME
// pixel, so the primary rays a warp starts together are near-identical and traverse in lockstep: C2 +3 %, C4 +5 %,
// C4b +15 %, C5 +5 % -- when the background is black.  With a bright background every escaping path adds to its pixel's
// accumulator and lanes on the same pixel serialise on it (C1 -3 %; warp-aggregating the sums first costs more than it
// saves), so the host picks g = 3 for a black background and 0 otherwise (profiles/r2_tile_shape.md).  The image is the same
// bit for bit under every order.  The items run from pool_init's start to total_items (block_items).  ADAPTIVE: L.lp
// numbers the block's active pixels (tm.n_valid of them); tp.act maps it to the tile pixel.
template <bool ADAPTIVE = false>
__device__ __forceinline__ bool pool_fetch(const RenderParams &P, const TileMap &tm, TilePool &tp, uint32_t total_items, PoolLane &L,
                                           uint32_t &px, uint32_t &py) {
    if (total_items == 0u) return false;
    const uint32_t gs = P.group_shift;
    if (gs == 0u) {
        const uint32_t item = atomicAdd(&tp.next, 1u);
        if (item >= total_items) return false;
        if (tm.n_valid == (uint32_t)kPathBlock) { L.s = item / (uint32_t)kPathBlock; L.lp = item % (uint32_t)kPathBlock; }
        else { L.s = item / tm.n_valid; L.lp = item - L.s * tm.n_valid; }
    } else {
        const uint32_t per_block = tm.n_valid << gs;                             // items per block of 2^g samples
        while (true) {
            const uint32_t item = atomicAdd(&tp.next, 1u);
            if (item >= total_items) return false;
            const uint32_t s_hi = item / per_block, rem = item - s_hi * per_block;
            L.lp = rem >> gs;
            L.s = (s_hi << gs) + (rem & ((1u << gs) - 1u));
            if (L.s < P.sample_count) break;                                      // ragged last block of samples
        }
    }
    uint32_t lt = L.lp;
    if constexpr (ADAPTIVE) lt = static_cast<TilePoolAdaptive &>(tp).act[L.lp];
    const uint32_t lx = tm.vw == (uint32_t)kPathTileW ? lt % (uint32_t)kPathTileW : lt % tm.vw;
    const uint32_t ly = tm.vw == (uint32_t)kPathTileW ? lt / (uint32_t)kPathTileW : lt / tm.vw;
    px = tm.x0 + lx;
    py = tm.y0 + ly;
    L.pixel = py * P.cam.w + px;
    L.bounce = 0;
    return true;
}

// shade_and_advance with the tile pool: the lane's path takes one step or, once ended, the lane takes the next item.
template <bool MOMENTS = false, bool ADAPTIVE = false>
__device__ __forceinline__ bool pool_shade_and_advance(const RenderParams &P, const TileMap &tm, TilePoolOf<MOMENTS, ADAPTIVE> &tp,
                                                       uint32_t total_items, const Hit &best, PoolLane &L, Ray &ray) {
    if (L.has_path) {
        ++L.rays;
        float er, eg, eb;
        const bool cont = path_bounce(P, best, L.pixel, L.s, L.bounce, ray, L.p, er, eg, eb);
        pool_contribute<MOMENTS>(tp, L.lp, er, eg, eb);   // the path's only non-zero contribution, if any (see pool_contribute)
        if (!cont) L.has_path = false;
    }
    if (!L.has_path) {
        uint32_t px, py;
        if (!pool_fetch<ADAPTIVE>(P, tm, tp, total_items, L, px, py)) return false;
        path_start(P, L.pixel, px, py, L.s, ray, L.p);
        L.has_path = true;
    }
    return true;
}

template <bool MOMENTS = false>
__device__ __forceinline__ void pool_init(TilePoolOf<MOMENTS> &tp, uint32_t first_item, uint32_t slot = kWholeTile) {
    if (threadIdx.x == 0) { tp.next = first_item; tp.slot = slot; }
    for (int i = threadIdx.x; i < kPathBlock * 3; i += kPathBlock) tp.acc[i] = 0;
    if constexpr (MOMENTS)
        for (int i = threadIdx.x; i < kPathBlock * 3; i += kPathBlock) tp.acc2[i] = 0;
    __syncthreads();
}

// Tile pixel lp's fixed-point sums a (and, with MOMENTS, its x^2 sums q, scaled the same way) -> the image.
template <bool MOMENTS = false>
__device__ __forceinline__ void store_tile_pixel(const RenderParams &P, const TileMap &tm, uint32_t lp, const long long (&a)[3],
                                                 const long long (&q)[3]) {
    const uint2 xy = tile_xy(tm, lp);
    const uint32_t pixel = xy.y * P.cam.w + xy.x;
    if (B200RT_CHECK(P.scene, pixel < P.cam.w * P.cam.h, 3)) {
        const float k = P.scale;
        store_rgb(P.out + (size_t)pixel * 3, fix_rgb(a[0]), fix_rgb(a[1]), fix_rgb(a[2]), k, (P.flags & kRenderAccumulate) != 0);
        if constexpr (MOMENTS)
            store_rgb(P.out_m2 + (size_t)pixel * 3, fix_x2(q[0]), fix_x2(q[1]), fix_x2(q[2]), k, (P.flags & kRenderAccumulate) != 0);
    }
}

// ADAPTIVE: active pixel lp's sums of this pass are added to its int64 planes.  A pixel has one writer per pass (the
// block of a whole tile, or the last chunk of a tail tile to arrive), so a plain add is exact; the conversion to floats
// happens once, after the last pass (adaptive_finish_kernel, through fix_rgb / fix_x2).
__device__ __forceinline__ void add_tile_pixel(const RenderParams &P, const TileMap &tm, const TilePoolAdaptive &tp, uint32_t lp,
                                               const long long (&a)[3], const long long (&q)[3]) {
    const uint32_t lt = tp.act[lp];
    const uint2 xy = tile_xy(tm, lt);
    const uint32_t pixel = xy.y * P.cam.w + xy.x;
    if (B200RT_CHECK(P.scene, lt < kPathBlock && pixel < P.cam.w * P.cam.h, 3)) {
        long long *o = P.ad_planes + (size_t)pixel * kAdaptivePlanes;
        o[0] += a[0]; o[1] += a[1]; o[2] += a[2];
        o[3] += q[0]; o[4] += q[1]; o[5] += q[2];
    }
}

template <bool MOMENTS, bool ADAPTIVE>
__device__ __forceinline__ void finish_tile_pixel(const RenderParams &P, const TileMap &tm, const TilePoolOf<MOMENTS, ADAPTIVE> &tp,
                                                  uint32_t lp, const long long (&a)[3], const long long (&q)[3]) {
    if constexpr (ADAPTIVE) add_tile_pixel(P, tm, tp, lp, a, q);
    else store_tile_pixel<MOMENTS>(P, tm, lp, a, q);
}

// After the block's last path: thread t writes tile pixel t.
template <bool MOMENTS = false, bool ADAPTIVE = false>
__device__ __forceinline__ void pool_write_tile(const RenderParams &P, const TileMap &tm, TilePoolOf<MOMENTS, ADAPTIVE> &tp) {
    __syncthreads();
    const uint32_t lp = threadIdx.x;
    if (lp < tm.n_valid) {
        const long long a[3] = {tp.acc[lp * 3 + 0], tp.acc[lp * 3 + 1], tp.acc[lp * 3 + 2]};
        long long q[3] = {0, 0, 0};
        if constexpr (MOMENTS) { q[0] = tp.acc2[lp * 3 + 0]; q[1] = tp.acc2[lp * 3 + 1]; q[2] = tp.acc2[lp * 3 + 2]; }
        finish_tile_pixel<MOMENTS, ADAPTIVE>(P, tm, tp, lp, a, q);
    }
}

// After a chunk block's last path: add its sums into the tail tile's slot of P.tail_acc with 64-bit integer atomics (so the
// total does not depend on how the samples were split or in which order the chunks finish), then count the block in.
// The chunk that arrives last takes the totals -- leaving the slot and its counter zero for the next launch -- and writes
// the pixels exactly as pool_write_tile does.  No block waits for another.
template <bool MOMENTS = false, bool ADAPTIVE = false>
__device__ __forceinline__ void pool_merge_chunk(const RenderParams &P, const TileMap &tm, TilePoolOf<MOMENTS, ADAPTIVE> &tp, uint32_t slot) {
    constexpr uint32_t kPlane = (uint32_t)kPathBlock * 3u;
    unsigned long long *part = reinterpret_cast<unsigned long long *>(P.tail_acc) + (size_t)slot * kPlane * (MOMENTS ? 2u : 1u);
    for (uint32_t i = threadIdx.x; i < kPlane; i += kPathBlock) {
        if (tp.acc[i]) atomicAdd(&part[i], (unsigned long long)tp.acc[i]);
        if constexpr (MOMENTS)
            if (tp.acc2[i]) atomicAdd(&part[kPlane + i], (unsigned long long)tp.acc2[i]);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) tp.last = atomicAdd(&P.tail_arrivals[slot], 1u) == P.tail_chunks - 1u;
    __syncthreads();
    if (!tp.last) return;
    __threadfence();
    const uint32_t lp = threadIdx.x;
    long long a[3], q[3] = {0, 0, 0};
    for (int c = 0; c < 3; ++c) {
        a[c] = (long long)atomicExch(&part[lp * 3 + c], 0ull);
        if constexpr (MOMENTS) q[c] = (long long)atomicExch(&part[kPlane + lp * 3 + c], 0ull);
    }
    if (lp == 0) P.tail_arrivals[slot] = 0u;
    if (lp < tm.n_valid) finish_tile_pixel<MOMENTS, ADAPTIVE>(P, tm, tp, lp, a, q);
}

#ifdef B200RT_BLOCK_TIMES
// Diagnostic build (-DB200RT_BLOCK_TIMES, scripts/tail_profile.py): thread 0 of every path_megakernel_pool block records
// {start ns, end ns, SM} of %globaltimer into g_block_times[blockIdx.x] (armed by b200rt_debug_block_times).
__device__ unsigned long long *g_block_times;
__device__ uint32_t g_block_times_n;
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void record_block_time(unsigned long long t_start) {
    if (threadIdx.x != 0 || !g_block_times || blockIdx.x >= g_block_times_n) return;
    uint32_t sm;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(sm));
    unsigned long long *r = g_block_times + (size_t)blockIdx.x * 3;
    r[0] = t_start; r[1] = globaltimer_ns(); r[2] = sm;
}
cudaError_t set_block_times(unsigned long long *buf, uint32_t n_blocks) {
    cudaError_t e = cudaMemcpyToSymbol(g_block_times, &buf, sizeof buf);
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(g_block_times_n, &n_blocks, sizeof n_blocks);
    return e;
}
#endif

// Start of an ADAPTIVE block: the tile of list entry `entry`, and its active pixels (its mask bits) in ascending tile-pixel
// order in tp.act.  Returns the tile's map with n_valid = the number of active pixels, so that block_items and pool_fetch
// number the items over them exactly as they number a whole tile's pixels.
__device__ __forceinline__ TileMap adaptive_tile(const RenderParams &P, uint32_t entry, TilePoolAdaptive &tp) {
    uint32_t tile = 0;
    bool ok = B200RT_CHECK(P.scene, entry < P.ad_n_list, 3);
    if (ok) {
        tile = P.ad_list[entry];
        ok = B200RT_CHECK(P.scene, tile < path_tiles(P.cam.w, P.cam.h), 3);
    }
    TileMap tm = map_tile(P.cam, ok ? tile : 0u);
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u, base = warp * 32u;
    const uint32_t valid = tm.n_valid >= base + 32u ? 0xFFFFFFFFu : (tm.n_valid > base ? (1u << (tm.n_valid - base)) - 1u : 0u);
    uint32_t word = ok ? P.ad_mask[(size_t)tile * kAdaptiveMaskWords + warp] : 0u;
    if (!B200RT_CHECK(P.scene, (word & ~valid) == 0u, 3)) word &= valid;
    if (lane == 0) tp.warp_act[warp] = __popc(word);
    __syncthreads();
    uint32_t before = 0, total = 0;
#pragma unroll
    for (uint32_t k = 0; k < (uint32_t)kAdaptiveMaskWords; ++k) {
        const uint32_t c = tp.warp_act[k];
        before += k < warp ? c : 0u;
        total += c;
    }
    if ((word >> lane) & 1u) tp.act[before + __popc(word & ((1u << lane) - 1u))] = (unsigned char)threadIdx.x;
    tm.n_valid = total;
    return tm;
}

// path_megakernel_pool (variant 0, default): every lane runs traverse-then-shade in a loop and takes the tile's next
// (pixel, sample) item as soon as its path ends.  Moments: also the per-pixel sum of x^2 into P.out_m2
// (b200rt_render_moments).  Adaptive (b200rt_render_adaptive): a block renders the active pixels of an entry of P.ad_list
// and adds both sums into P.ad_planes; the host sets sample_begin to the pass's first sample, so the Philox keys are unchanged.
template <int STACK, PathMode MODE, bool LEAF_FIRST>
__global__ void __launch_bounds__(kPathBlock, kPathMinBlocks) path_megakernel_pool(const __grid_constant__ RenderParams P) {
    constexpr bool COUNT = MODE == PathMode::Counters;
    constexpr bool MOMENTS = MODE == PathMode::Moments || MODE == PathMode::Adaptive;
    constexpr bool ADAPTIVE = MODE == PathMode::Adaptive;
    __shared__ TilePoolOf<MOMENTS, ADAPTIVE> tp;
#ifdef B200RT_BLOCK_TIMES
    const unsigned long long t_start = globaltimer_ns();
#endif
    const CameraParams &C = P.cam;
    const BlockWork w = block_work(P);
    TileMap tm;
    if constexpr (ADAPTIVE) tm = adaptive_tile(P, w.tile, tp);
    else tm = map_tile(C, w.tile);
    uint32_t first_item;
    const uint32_t total_items = block_items(P, tm, w, first_item);
    pool_init<MOMENTS>(tp, first_item, w.slot);
    PoolLane L;
    Ray ray;
    TraversalCounters ctr;
    Hit best{0.0, kNoHit};
    while (pool_shade_and_advance<MOMENTS, ADAPTIVE>(P, tm, tp, total_items, best, L, ray)) {
        best = closest_hit<STACK, COUNT, LEAF_FIRST>(P.scene, ray.ox, ray.oy, ray.oz, ray.dx, ray.dy, ray.dz, kRayTmin, kRayTmax, &ctr);
    }
    __syncthreads();
    const uint32_t slot = tp.slot;
    if (slot == kWholeTile) pool_write_tile<MOMENTS, ADAPTIVE>(P, tm, tp);
    else pool_merge_chunk<MOMENTS, ADAPTIVE>(P, tm, tp, slot);
    write_counters(P, L.rays, COUNT, ctr);
#ifdef B200RT_BLOCK_TIMES
    record_block_time(t_start);
#endif
}

// ------------------------------------------------------------------------------------------
// path_megakernel (thread-owns-pixel form, kept for A/B: B200RT_FLAG_THREAD_PIXELS): every lane runs traverse-then-shade
// in a loop over ITS pixel's samples and starts the next sample as soon as a path ends.  64 registers (16 blocks = 32 warps per SM) measured
// fastest on B200: 8/12/16/20/24 blocks per SM gave 2707/3171/3263/2630/2307 Mpaths/s on C2.
template <int STACK, bool COUNT>
__global__ void __launch_bounds__(kPathBlock, kPathMinBlocks) path_megakernel(const __grid_constant__ RenderParams P) {
    const CameraParams &C = P.cam;
    const PixelMap m = map_pixel(C);
    LaneState L;
    TraversalCounters ctr;
    Hit best{0.0, kNoHit};
    if (m.valid && C.max_depth > 0 && P.sample_count > 0) {
        while (shade_and_advance(P, m, best, L)) {
            best = closest_hit<STACK, COUNT>(P.scene, L.ray.ox, L.ray.oy, L.ray.oz, L.ray.dx, L.ray.dy, L.ray.dz, kRayTmin, kRayTmax, &ctr);
        }
    }
    write_pixel_and_counters(P, m, L.sum_r, L.sum_g, L.sum_b, L.rays, COUNT, ctr);
}

// ------------------------------------------------------------------------------------------
// path_lanes_kernel: MEASUREMENT ONLY (b200rt_debug_lane_accounting).  The default kernel's schedule -- per
// round every lane shades / regenerates, then the warp iterates "node step for the lanes at a node, leaf step for the
// lanes at a leaf" (or the reverse order, as the launcher picks) until its slowest lane is done -- replayed warp-synchronously so that each warp can count, per executed step,
// how many of its 32 lanes took part and what the others were doing:
//   acc[0] shade executions           acc[1] lanes taking part
//   acc[2] node-step executions       acc[3] lanes at a node     acc[4] idle: at a leaf   acc[5] idle: traversal done,
//                                                                waiting for the round    acc[6] idle: pixel out of samples
//   acc[7] leaf-step executions       acc[8] lanes at a leaf     acc[9] idle: at a node   acc[10] idle: done   acc[11] idle: finished
//   acc[12] primitive-test executions (a leaf step loops over its primitives; each       acc[13] lanes taking part
//           scene-spanning primitive, traverse.cuh trav_hoisted, is one more per round)
//   acc[14] warps   acc[15] lane-rounds (shade calls that started a ray)
// Same Philox keys and the same arithmetic as path_megakernel, so it also writes the same image.
template <int STACK, bool POOL>
__global__ void __launch_bounds__(kPathBlock) path_lanes_kernel(const __grid_constant__ RenderParams P, unsigned long long *__restrict__ acc, bool leaf_first) {
    __shared__ TilePool tp;
    const CameraParams &C = P.cam;
    const PixelMap m = map_pixel(C);
    const BlockWork w = block_work(P);   // whole tiles: the measurement launch has no chunked tail
    const TileMap tm = map_tile(C, w.tile);
    uint32_t first_item;
    const uint32_t total_items = block_items(P, tm, w, first_item);
    if (POOL) pool_init(tp, first_item);
    LaneState L;
    PoolLane Lp;
    Trav T;
    uint2 stack[STACK];
    T.cur = kTravDone;
    T.best.t = 0.0; T.best.ref = kNoHit;
    bool finished = POOL ? false : !(m.valid && C.max_depth > 0 && P.sample_count > 0);
    unsigned long long a[16] = {};
    const unsigned full = 0xffffffffu;
    while (true) {
        const unsigned ms = __ballot_sync(full, !finished);
        if (!ms) break;
        a[0]++; a[1] += __popc(ms);
        bool go = false;
        if (!finished) {
            if (POOL) {
                go = pool_shade_and_advance(P, tm, tp, total_items, T.best, Lp, T.ray);
                if (go) trav_setup(T, kRayTmin, kRayTmax);
            } else {
                go = shade_and_advance(P, m, T.best, L);
                if (go) trav_init(T, L.ray.ox, L.ray.oy, L.ray.oz, L.ray.dx, L.ray.dy, L.ray.dz, kRayTmin, kRayTmax);
            }
            if (go) a[15]++;
            else { finished = true; T.cur = kTravDone; }
        }
        {   // the scene-spanning primitives: one primitive-test execution each, by the lanes that started a ray
            const unsigned mg = __ballot_sync(full, go);
            if (mg) { a[12] += P.scene.n_hoisted; a[13] += (unsigned long long)__popc(mg) * P.scene.n_hoisted; }
            if (go) trav_hoisted<false>(P.scene, T, nullptr);
        }
        while (true) {   // one iteration of closest_hit's loop: both kinds of step, in the product's order
            if (!__ballot_sync(full, !finished && !trav_done(T))) break;
#pragma unroll
            for (int phase = 0; phase < 2; ++phase) {
                const bool node_phase = (phase == 0) != leaf_first;
                const bool node = !finished && trav_at_node(T), leaf = !finished && trav_at_leaf(T);
                const unsigned mn = __ballot_sync(full, node), ml = __ballot_sync(full, leaf), mf = __ballot_sync(full, finished);
                const unsigned md = ~(mn | ml | mf);
                if (node_phase) {
                    if (mn) { a[2]++; a[3] += __popc(mn); a[4] += __popc(ml); a[5] += __popc(md); a[6] += __popc(mf); }
                    if (node) trav_node_step(P.scene, T, stack);
                } else {
                    if (ml) {
                        a[7]++; a[8] += __popc(ml); a[9] += __popc(mn); a[10] += __popc(md); a[11] += __popc(mf);
                        const uint32_t cnt = leaf ? ((T.cur >> 26) & 0xFu) : 0u;
                        for (uint32_t i = 0; i < 8; ++i) {
                            const unsigned mi = __ballot_sync(full, cnt > i);
                            if (!mi) break;
                            a[12]++; a[13] += __popc(mi);
                        }
                    }
                    if (leaf) trav_leaf_step(P.scene, T, stack);
                }
            }
        }
    }
    TraversalCounters ctr;
    if (POOL) { pool_write_tile(P, tm, tp); write_counters(P, Lp.rays, false, ctr); }
    else write_pixel_and_counters(P, m, L.sum_r, L.sum_g, L.sum_b, L.rays, false, ctr);
    a[14] = 1;
    unsigned long long rounds = a[15];
    for (int off = 16; off; off >>= 1) rounds += __shfl_down_sync(full, rounds, off);
    a[15] = rounds;
    if ((threadIdx.x & 31) == 0)
        for (int i = 0; i < 16; ++i) atomicAdd(&acc[i], a[i]);
}

// ------------------------------------------------------------------------------------------
// One pixel's tone map into q[0..2]: Reinhard + gamma 2 + int(255.999999 v)   [RGB::as_string, rgb.h:90-113]
__device__ __forceinline__ void tonemap_pixel(double r, double g, double b, int clamp, int32_t *__restrict__ q) {
    const double L = 0.2126 * r + 0.7152 * g + 0.0722 * b;          // rgb.h:28-30
    const double scale = 255 + 0.999999;                             // rgb.h:106
    const double v[3] = {r / (1 + L), g / (1 + L), b / (1 + L)};     // rgb.h:99-104
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        int t = (int)(scale * sqrt(v[c]));                           // pow(v, 1/2), truncation (rgb.h:107-111)
        if (clamp) t = t < 0 ? 0 : (t > 255 ? 255 : t);
        q[c] = t;
    }
}

__global__ void tonemap_kernel(const float *__restrict__ hdr, long long n_pixels, int32_t *__restrict__ out, int clamp) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pixels) return;
    tonemap_pixel(hdr[i * 3 + 0], hdr[i * 3 + 1], hdr[i * 3 + 2], clamp, out + i * 3);
}

// Frame epilogue on the reducing rank: sum -> mean in place (pixel_color /= spp, camera.h:290) and,
// optionally, the tone-mapped integers of the same pixels in the same pass.
__global__ void finalize_kernel(float *__restrict__ frame, long long n_pixels, float scale, int32_t *__restrict__ ldr, int clamp) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pixels) return;
    const float rf = frame[i * 3 + 0] * scale, gf = frame[i * 3 + 1] * scale, bf = frame[i * 3 + 2] * scale;
    frame[i * 3 + 0] = rf; frame[i * 3 + 1] = gf; frame[i * 3 + 2] = bf;
    if (ldr) tonemap_pixel(rf, gf, bf, clamp, ldr + i * 3);
}

// Multi-GPU frame exchange as ONE kernel over peer memory (NVLink / NVSwitch): this rank's slice of
// "sum the per-rank sample sums, /= spp (camera.h:290), tone-map (rgb.h:90-113)" with the result
// written straight into the root rank's buffers.  Every rank runs it on a different slice, so the
// N frames cross the links once, spread over all of them (reduce-scatter + epilogue + gather in one
// pass), instead of funnelling into rank 0.  Peers are added in rank order 0..N-1 whichever rank owns
// the slice, so the result does not depend on the slicing.
//   Block = kPeerTilePx pixels: coalesced float4 loads from each peer -> sum -> scale -> coalesced
//   float4 store to the root HDR frame (may alias peer 0's buffer: each element is read and written by
//   the same thread) -> shared memory -> per-pixel tone map -> coalesced store of the integers.
constexpr int kPeerTilePx = 1024, kPeerThreads = 256;
__global__ void __launch_bounds__(kPeerThreads) reduce_finalize_peers_kernel(const __grid_constant__ PeerFrames in, int n_peers, long long px_lo,
                                                                             long long px_hi, float scale, float *root_hdr,
                                                                             int32_t *root_ldr, int clamp) {
    __shared__ __align__(16) float tile[kPeerTilePx * 3];
    const long long tile_px = px_lo + (long long)blockIdx.x * kPeerTilePx;
    const long long base = tile_px * 3;                                                     // first float of the tile
    const long long n_fl = ((px_hi - tile_px < kPeerTilePx) ? (px_hi - tile_px) : kPeerTilePx) * 3;  // floats in this tile
#pragma unroll
    for (int k = 0; k < kPeerTilePx * 3 / 4 / kPeerThreads; ++k) {
        const int j = (threadIdx.x + k * kPeerThreads) * 4;
        if (j + 3 < n_fl) {
            float4 a = *reinterpret_cast<const float4 *>(in.p[0] + base + j);
            for (int r = 1; r < n_peers; ++r) {
                const float4 b = *reinterpret_cast<const float4 *>(in.p[r] + base + j);
                a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
            }
            a.x *= scale; a.y *= scale; a.z *= scale; a.w *= scale;
            *reinterpret_cast<float4 *>(root_hdr + base + j) = a;
            *reinterpret_cast<float4 *>(tile + j) = a;
        } else {
            for (int e = j; e < n_fl && e < j + 4; ++e) {                                    // ragged end of the frame
                float a = in.p[0][base + e];
                for (int r = 1; r < n_peers; ++r) a += in.p[r][base + e];
                a *= scale;
                root_hdr[base + e] = a;
                tile[e] = a;
            }
        }
    }
    if (!root_ldr) return;
    __syncthreads();
    int32_t q[kPeerTilePx / kPeerThreads][3];
#pragma unroll
    for (int k = 0; k < kPeerTilePx / kPeerThreads; ++k) {
        const int px = threadIdx.x + k * kPeerThreads;
        if (px * 3 < n_fl) tonemap_pixel(tile[px * 3 + 0], tile[px * 3 + 1], tile[px * 3 + 2], clamp, q[k]);
        else q[k][0] = q[k][1] = q[k][2] = 0;                                                // past the ragged end of the frame
    }
    __syncthreads();
    int32_t *itile = reinterpret_cast<int32_t *>(tile);
#pragma unroll
    for (int k = 0; k < kPeerTilePx / kPeerThreads; ++k) {
        const int px = threadIdx.x + k * kPeerThreads;
        itile[px * 3 + 0] = q[k][0]; itile[px * 3 + 1] = q[k][1]; itile[px * 3 + 2] = q[k][2];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kPeerTilePx * 3 / 4 / kPeerThreads; ++k) {
        const int j = (threadIdx.x + k * kPeerThreads) * 4;
        if (j + 3 < n_fl) *reinterpret_cast<int4 *>(root_ldr + base + j) = *reinterpret_cast<const int4 *>(itile + j);
        else for (int e = j; e < n_fl && e < j + 4; ++e) root_ldr[base + e] = itile[e];
    }
}

// ------------------------------------------------------------------------------------------
cudaError_t launch_raycast(int stack, const DeviceScene &S, const double *rays, long long n, double tmin, double tmax,
                           int32_t *prim, double *t, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    const int block = 128;
    with_stack(stack, [&](auto K) {
        raycast_kernel<K.value><<<(unsigned)((n + block - 1) / block), block, 0, st>>>(S, rays, n, tmin, tmax, prim, t);
    });
    return cudaGetLastError();
}

cudaError_t launch_debug_camera(const CameraParams &C, const uint32_t *pixels, const uint32_t *rnd, long long n, double *rays_out,
                                cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    debug_camera_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(C, pixels, rnd, n, rays_out);
    return cudaGetLastError();
}

cudaError_t launch_debug_philox(const uint32_t *in, long long n, uint32_t *out, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    debug_philox_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(in, n, out);
    return cudaGetLastError();
}
cudaError_t launch_debug_samplers(const uint32_t *rnd, long long n, double *sphere_out, double *disk_out, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    debug_samplers_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(rnd, n, sphere_out, disk_out);
    return cudaGetLastError();
}

cudaError_t launch_debug_shade(int stack, const DeviceScene &S, const double *rays, const uint32_t *rnd, long long n, double tmin,
                               double tmax, void *records, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    const unsigned blocks = (unsigned)((n + 127) / 128);
    ShadeRecord *out = static_cast<ShadeRecord *>(records);
    with_stack(stack, [&](auto K) { debug_shade_kernel<K.value><<<blocks, 128, 0, st>>>(S, rays, rnd, n, tmin, tmax, out); });
    return cudaGetLastError();
}

// The tile-pool kernel instance of (stack, mode, leaf_first).  The launch and the occupancy query that sizes its chunked
// tail both take it from here, so they always name the same instance.
template <int STACK, PathMode MODE>
static const void *pool_instance(bool leaf_first) {
    return leaf_first ? (const void *)path_megakernel_pool<STACK, MODE, true> : (const void *)path_megakernel_pool<STACK, MODE, false>;
}
static const void *path_pool_kernel(int stack, PathMode mode, bool leaf_first) {
    return with_stack(stack, [&](auto K) {
        return mode == PathMode::Plain      ? pool_instance<K.value, PathMode::Plain>(leaf_first)
               : mode == PathMode::Counters ? pool_instance<K.value, PathMode::Counters>(leaf_first)
               : mode == PathMode::Moments  ? pool_instance<K.value, PathMode::Moments>(leaf_first)
                                            : pool_instance<K.value, PathMode::Adaptive>(leaf_first);
    });
}

cudaError_t launch_path_megakernel(int stack, const RenderParams &P, PathMode mode, bool leaf_first, cudaStream_t st) {
    // one block per tile, or per entry of the pass's tile list
    const uint32_t units = mode == PathMode::Adaptive ? P.ad_n_list : path_tiles(P.cam.w, P.cam.h);
    if (units == 0) return cudaSuccess;
    if ((P.flags & kRenderThreadPixels) && (mode == PathMode::Plain || mode == PathMode::Counters)) {
        with_stack(stack, [&](auto K) {   // round-1 work distribution: node-then-leaf only
            if (mode == PathMode::Counters) path_megakernel<K.value, true><<<units, kPathBlock, 0, st>>>(P);
            else path_megakernel<K.value, false><<<units, kPathBlock, 0, st>>>(P);
        });
        return cudaGetLastError();
    }
    // tile pool: whole-tile blocks, then tail_chunks chunk blocks for each unit from tail_first on
    const uint32_t blocks = P.tail_chunks ? P.tail_first + (units - P.tail_first) * P.tail_chunks : units;
    void *args[] = {const_cast<RenderParams *>(&P)};
    return cudaLaunchKernel(path_pool_kernel(stack, mode, leaf_first), blocks, kPathBlock, args, 0, st);
}

// ------------------------------------------------------------------------------------------
// Adaptive sampling between passes.  Every kernel below runs one block of kPathBlock threads per tile, thread t on tile
// pixel t, so that warp k owns mask word k of the tile.
__device__ __forceinline__ TileMap adaptive_map(const AdaptiveState &A, uint32_t tile) {
    CameraParams C;
    C.w = A.w;
    C.h = A.h;
    return map_tile(C, tile);
}
__device__ __forceinline__ uint32_t adaptive_tiles(const AdaptiveState &A) { return path_tiles(A.w, A.h); }

__global__ void __launch_bounds__(kPathBlock) adaptive_init_kernel(const __grid_constant__ AdaptiveState A) {
    const uint32_t tile = blockIdx.x, warp = threadIdx.x >> 5;
    const TileMap tm = adaptive_map(A, tile);
    const unsigned bits = __ballot_sync(0xFFFFFFFFu, threadIdx.x < tm.n_valid);
    if ((threadIdx.x & 31u) == 0) {
        A.mask[(size_t)tile * kAdaptiveMaskWords + warp] = bits;
        A.unconv[(size_t)tile * kAdaptiveMaskWords + warp] = 0u;
    }
    if (threadIdx.x == 0) A.list[tile] = tile;
}

// Camera::sample_variance of one channel, from the mean-plane floats of x and x^2 over n >= 2 samples.
__device__ __forceinline__ double channel_variance(float mean, float m2, uint32_t n) {
    const double d = (double)m2 - (double)mean * (double)mean;
    if (d <= ldexp((double)m2, -20) + 0x1p-24) return 0.0;
    return (double)n / (double)(n - 1u) * d;
}

// The convergence rule (b200rt.h, b200rt_render_adaptive): the mean-plane floats exactly as store_tile_pixel writes them
// (fix_rgb / fix_x2 times the float 1/n), then err = sqrt(sum of the channel variances / 3n) against rel_noise x the mean
// of the three channel means + abs_noise.  In double; the library is built with -fmad=false, so nothing is contracted and
// the host can replay it bit for bit.
__device__ __forceinline__ bool pixel_converged(const AdaptiveState &A, const long long *p, uint32_t n) {
    const float inv = (float)(1.0 / (double)n);
    double var = 0.0, level = 0.0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float mean = fix_rgb(p[c]) * inv;
        const float m2 = fix_x2(p[3 + c]) * inv;
        var += channel_variance(mean, m2, n);
        level += (double)mean;
    }
    const double err = sqrt(var / (3.0 * (double)n));
    return err <= A.rel_noise * (level / 3.0) + A.abs_noise;
}

// The pixels a pass rendered now have n samples; with judge, each one's unconverged bit is set from the rule.
__global__ void __launch_bounds__(kPathBlock) adaptive_judge_kernel(const __grid_constant__ AdaptiveState A, uint32_t n, int judge,
                                                                    const __grid_constant__ DeviceScene S) {
    const uint32_t tile = A.list[blockIdx.x];
    if (!B200RT_CHECK(S, tile < adaptive_tiles(A), 3)) return;
    const TileMap tm = adaptive_map(A, tile);
    const uint32_t lp = threadIdx.x, lane = lp & 31u;
    const size_t mw = (size_t)tile * kAdaptiveMaskWords + (lp >> 5);
    bool unconv = false;
    if (((A.mask[mw] >> lane) & 1u) && B200RT_CHECK(S, lp < tm.n_valid, 3)) {
        const uint2 xy = tile_xy(tm, lp);
        const uint32_t pixel = xy.y * A.w + xy.x;
        A.counts[pixel] = n;
        if (judge) unconv = !pixel_converged(A, A.planes + (size_t)pixel * kAdaptivePlanes, n);
    }
    const unsigned bits = __ballot_sync(0xFFFFFFFFu, unconv);
    if (lane == 0) A.unconv[mw] = bits;
}

// A pixel of the pass stays active if any pixel of its 3 x 3 neighbourhood (clipped at the image edge) is unconverged.
// A pixel that stopped earlier was converged when it stopped and its sums have not changed since, so only the pass's own
// tiles can hold unconverged bits; every other tile's are zero.  Stopping is final: a pixel outside the mask stays out.
__global__ void __launch_bounds__(kPathBlock) adaptive_decide_kernel(const __grid_constant__ AdaptiveState A,
                                                                     const __grid_constant__ DeviceScene S) {
    const uint32_t tile = A.list[blockIdx.x];
    if (!B200RT_CHECK(S, tile < adaptive_tiles(A), 3)) return;
    const TileMap tm = adaptive_map(A, tile);
    const uint32_t lp = threadIdx.x, lane = lp & 31u;
    const uint32_t tiles_x = path_tiles_x(A.w);
    const size_t mw = (size_t)tile * kAdaptiveMaskWords + (lp >> 5);
    bool keep = false;
    if (((A.mask[mw] >> lane) & 1u) && lp < tm.n_valid) {
        const uint2 xy = tile_xy(tm, lp);
        const int px = (int)xy.x, py = (int)xy.y;
        for (int qy = max(py - 1, 0); qy <= min(py + 1, (int)A.h - 1); ++qy)
            for (int qx = max(px - 1, 0); qx <= min(px + 1, (int)A.w - 1); ++qx) {
                const uint32_t tq = (uint32_t)qy / (uint32_t)kPathTileH * tiles_x + (uint32_t)qx / (uint32_t)kPathTileW;
                const TileMap tn = adaptive_map(A, tq);
                const uint32_t lq = ((uint32_t)qy - tn.y0) * tn.vw + ((uint32_t)qx - tn.x0);
                keep |= (A.unconv[(size_t)tq * kAdaptiveMaskWords + lq / 32u] >> (lq & 31u)) & 1u;
            }
    }
    const unsigned bits = __ballot_sync(0xFFFFFFFFu, keep);
    if (lane == 0) A.mask[mw] = bits;
    const int n_keep = __syncthreads_count(keep);
    if (threadIdx.x == 0 && n_keep) {
        const uint32_t slot = atomicAdd(&A.totals[0], 1u);
        if (B200RT_CHECK(S, slot < adaptive_tiles(A), 3)) A.next_list[slot] = tile;
        atomicAdd(&A.totals[1], (uint32_t)n_keep);
    }
}

// planes / counts -> the output floats: store_tile_pixel's conversion with the pixel's own count (k = 1 for sums).
__global__ void adaptive_finish_kernel(const __grid_constant__ AdaptiveState A, int sum, float *__restrict__ out_rgb,
                                       float *__restrict__ out_m2) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)A.w * A.h) return;
    const uint32_t n = A.counts[i];
    const float k = sum || n == 0 ? 1.0f : (float)(1.0 / (double)n);
    const long long *p = A.planes + i * kAdaptivePlanes;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        out_rgb[i * 3 + c] = fix_rgb(p[c]) * k;
        out_m2[i * 3 + c] = fix_x2(p[3 + c]) * k;
    }
}

cudaError_t launch_adaptive_init(const AdaptiveState &A, uint32_t tiles, cudaStream_t st) {
    if (tiles == 0) return cudaSuccess;
    adaptive_init_kernel<<<tiles, kPathBlock, 0, st>>>(A);
    return cudaGetLastError();
}
cudaError_t launch_adaptive_judge(const AdaptiveState &A, uint32_t n, bool judge, const DeviceScene &S, cudaStream_t st) {
    if (A.n_list == 0) return cudaSuccess;
    adaptive_judge_kernel<<<A.n_list, kPathBlock, 0, st>>>(A, n, judge ? 1 : 0, S);
    return cudaGetLastError();
}
cudaError_t launch_adaptive_decide(const AdaptiveState &A, const DeviceScene &S, cudaStream_t st) {
    if (A.n_list == 0) return cudaSuccess;
    adaptive_decide_kernel<<<A.n_list, kPathBlock, 0, st>>>(A, S);
    return cudaGetLastError();
}
cudaError_t launch_adaptive_finish(const AdaptiveState &A, bool sum, float *out_rgb, float *out_m2, cudaStream_t st) {
    const long long n = (long long)A.w * A.h;
    if (n == 0) return cudaSuccess;
    adaptive_finish_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(A, sum ? 1 : 0, out_rgb, out_m2);
    return cudaGetLastError();
}

size_t tail_scratch_bytes(uint32_t tail_tiles, bool moments) {
    return (size_t)tail_tiles * ((size_t)kPathBlock * 3 * sizeof(long long) * (moments ? 2 : 1) + sizeof(uint32_t));
}

cudaError_t path_resident_blocks(int stack, PathMode mode, bool leaf_first, int sm_count, int *blocks) {
    int n = 0;
    const cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, path_pool_kernel(stack, mode, leaf_first), kPathBlock, 0);
    *blocks = n * sm_count;
    return e;
}

cudaError_t launch_path_lanes(int stack, const RenderParams &P, unsigned long long *acc, bool leaf_first, cudaStream_t st) {
    const uint32_t tiles = path_tiles(P.cam.w, P.cam.h);
    if (tiles == 0) return cudaSuccess;
    const bool pool = !(P.flags & kRenderThreadPixels);
    with_stack(stack, [&](auto K) {
        if (pool) path_lanes_kernel<K.value, true><<<tiles, kPathBlock, 0, st>>>(P, acc, leaf_first);
        else path_lanes_kernel<K.value, false><<<tiles, kPathBlock, 0, st>>>(P, acc, leaf_first);
    });
    return cudaGetLastError();
}

cudaError_t launch_tonemap(const float *hdr, long long n_pixels, int32_t *out, int clamp, cudaStream_t st) {
    if (n_pixels == 0) return cudaSuccess;
    tonemap_kernel<<<(unsigned)((n_pixels + 255) / 256), 256, 0, st>>>(hdr, n_pixels, out, clamp);
    return cudaGetLastError();
}

cudaError_t launch_finalize(float *frame, long long n_pixels, float scale, int32_t *ldr, int clamp, cudaStream_t st) {
    if (n_pixels == 0) return cudaSuccess;
    finalize_kernel<<<(unsigned)((n_pixels + 255) / 256), 256, 0, st>>>(frame, n_pixels, scale, ldr, clamp);
    return cudaGetLastError();
}

__global__ void add_frame_kernel(float *__restrict__ frame, const float *__restrict__ other, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) frame[i] += other[i];
}
cudaError_t launch_add_frame(float *frame, const float *other, long long n_floats, cudaStream_t st) {
    if (n_floats == 0) return cudaSuccess;
    add_frame_kernel<<<(unsigned)((n_floats + 255) / 256), 256, 0, st>>>(frame, other, n_floats);
    return cudaGetLastError();
}

void peer_slice(long long n_pixels, int n_peers, int rank, long long *lo, long long *hi) {
    long long chunk = (n_pixels + n_peers - 1) / n_peers;
    chunk = (chunk + kPeerTilePx - 1) / kPeerTilePx * kPeerTilePx;        // whole tiles: slices start 16-byte aligned
    const long long a = chunk * rank, b = a + chunk;
    *lo = a < n_pixels ? a : n_pixels;
    *hi = b < n_pixels ? b : n_pixels;
}

cudaError_t launch_reduce_finalize_peers(const PeerFrames &in, int n_peers, int rank, long long n_pixels, float scale,
                                         float *root_hdr, int32_t *root_ldr, int clamp, cudaStream_t st) {
    long long lo, hi;
    peer_slice(n_pixels, n_peers, rank, &lo, &hi);
    if (hi <= lo) return cudaSuccess;
    const unsigned blocks = (unsigned)((hi - lo + kPeerTilePx - 1) / kPeerTilePx);
    reduce_finalize_peers_kernel<<<blocks, kPeerThreads, 0, st>>>(in, n_peers, lo, hi, scale, root_hdr, root_ldr, clamp);
    return cudaGetLastError();
}

}  // namespace b200rt
