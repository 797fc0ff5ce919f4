// path.cuh -- the rules of one path, shared by the tile-pool and thread-owns-pixel kernels (kernels.cu) and the wavefront
// variant (wavefront.cu), so that all of them render the same paths.  They differ only in how lanes get work and where
// contributions are summed.
#pragma once
#include <limits>

#include "kernels.h"

namespace b200rt {

// world.hit_by(ray, Interval::with_min(0.00001))  (camera.h:217).  Compile-time constants, so that trav_setup's
// float_toward folds their FP32 bounds (traverse.cuh).
constexpr double kRayTmin = 0.00001;
constexpr double kRayTmax = std::numeric_limits<double>::infinity();

// Sample s of `pixel` (at image column px, row py): its primary ray and unit throughput (camera.h:184-200).
__device__ __forceinline__ void path_start(const RenderParams &P, uint32_t pixel, uint32_t px, uint32_t py, uint32_t s, Ray &ray,
                                           PathState &p) {
    const Philox4 rnd = philox4x32_10(pixel, P.sample_begin + s, 0u, 0u, (uint32_t)P.seed, (uint32_t)(P.seed >> 32));
    camera_ray(P.cam, px, py, rnd, ray, p);
}

// One step of ray_color (camera.h:205-258) for a ray whose closest hit is `hit`: writes the contribution (throughput x
// background on a miss, x emission at a light, else zero) into er / eg / eb, and returns true if the path continues with
// the scattered ray in `ray`.  Once `bounce` reaches max_depth the path ends: ray_color(scattered, depth_left - 1) would
// contribute nothing (camera.h:211-213).
__device__ __forceinline__ bool path_bounce(const RenderParams &P, const Hit &hit, uint32_t pixel, uint32_t s, uint32_t &bounce,
                                            Ray &ray, PathState &p, float &er, float &eg, float &eb) {
    if (hit.ref == kNoHit) {   // camera.h:248
        er = p.tr * P.cam.background[0]; eg = p.tg * P.cam.background[1]; eb = p.tb * P.cam.background[2];
        return false;
    }
    er = eg = eb = 0.0f;
    const Philox4 rnd = philox4x32_10(pixel, P.sample_begin + s, bounce + 1u, 0u, (uint32_t)P.seed, (uint32_t)(P.seed >> 32));
    return shade_hit(P.scene, hit, rnd, ray, p, er, eg, eb) && ++bounce != P.cam.max_depth;
}

// The rays (and with count the traversal counters) of the warp's lanes into P.counters: one atomic per warp and counter.
__device__ __forceinline__ void write_counters(const RenderParams &P, uint32_t lane_rays, bool count, const TraversalCounters &ctr) {
    unsigned long long rays = lane_rays;
    for (int off = 16; off; off >>= 1) rays += __shfl_down_sync(0xffffffffu, rays, off);
    if ((threadIdx.x & 31) == 0 && rays) atomicAdd(&P.counters[0], rays);
    if (count) {
        unsigned long long a = ctr.nodes, b = ctr.prims, c = ctr.quads;
        for (int off = 16; off; off >>= 1) {
            a += __shfl_down_sync(0xffffffffu, a, off);
            b += __shfl_down_sync(0xffffffffu, b, off);
            c += __shfl_down_sync(0xffffffffu, c, off);
        }
        if ((threadIdx.x & 31) == 0) { atomicAdd(&P.counters[1], a); atomicAdd(&P.counters[2], b); atomicAdd(&P.counters[3], c); }
    }
}

}  // namespace b200rt
