// wavefront.cu -- the wavefront variant of the path kernel (B200RT_VARIANT_WAVEFRONT).
//
// A path is started and advanced by the same functions as in the other path kernels (path.cuh), so
// all of them compute identical per-path radiance; images differ only by FP32 summation order
// (frame accumulation here is atomic).  What changes is the execution
// shape, aimed at the two divergence sources ncu shows in the megakernel (12 of 32 threads active
// per instruction; material code at 6-7):
//
//   * a POOL of path slots lives in HBM (SoA: ray 6 x f64, throughput + pixel, sample/bounce,
//     hit t + ref).  Every slot always holds a live path: when a path ends, the shade stage
//     regenerates the slot with the next (pixel, sample) work item, so every wave traces a full
//     pool until the frame's samples run out.
//   * wf_trace   persistent warps over contiguous chunks of the pool; a lane that finishes its ray
//                parks the result and, once a quarter of the warp is parked, the parked lanes write
//                hit + material class back and take the next slots -- lanes never wait for the
//                longest ray of the warp.
//   * wf_shade   one thread per queue entry, queues concatenated in class order
//                (miss | light | lambertian | metal | dielectric), so a warp shades ONE material.
//
//   * wf_sort    builds the five class queues: compaction by warp ballot + prefix sums.
//
// A slot is one 128-byte line (AoS) accessed with 16-byte vectors, so the class-sorted (random)
// slot order of the shade stage still moves whole sectors.  Traffic per ray segment: trace reads
// 64 B and writes 32 B, sort reads 32 B, shade reads 96 B and writes 96 B: ~0.3 KB.
#include <cstdio>
#include <cstdlib>

#include "kernels.h"
#include "path.cuh"

namespace b200rt {

enum { WF_MISS = 0, WF_LIGHT = 1, WF_LAMBERT = 2, WF_METAL = 3, WF_DIELECTRIC = 4, WF_CLASSES = 5 };
constexpr uint32_t kDeadPixel = 0xFFFFFFFFu;
constexpr int kSortBlock = 256;

__device__ __forceinline__ uint32_t lanemask_lt() {
    uint32_t m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

// (pixel, sample) of work item k: consecutive items are neighbouring pixels of the same sample.
__device__ __forceinline__ void item_to_pixel_sample(unsigned long long k, uint32_t npix, uint32_t &pixel, uint32_t &sample) {
    sample = (uint32_t)(k / npix);
    pixel = (uint32_t)(k - (unsigned long long)sample * npix);
}

// 16-byte views of a slot
__device__ __forceinline__ void slot_store_ray(PathSlot *s, const Ray &r) {
    double2 *v = reinterpret_cast<double2 *>(s);
    v[0] = make_double2(r.ox, r.oy); v[1] = make_double2(r.oz, r.dx); v[2] = make_double2(r.dy, r.dz);
}
__device__ __forceinline__ void slot_load_ray(const PathSlot *s, Ray &r) {
    const double2 *v = reinterpret_cast<const double2 *>(s);
    const double2 a = v[0], b = v[1], c = v[2];
    r.ox = a.x; r.oy = a.y; r.oz = b.x; r.dx = b.y; r.dy = c.x; r.dz = c.y;
}

// Starts the path of work item `item` in slot `s` (camera.h:184-200).
__device__ __forceinline__ void wf_spawn(const RenderParams &P, PathSlot *s, unsigned long long item) {
    const CameraParams &C = P.cam;
    uint32_t pixel, smp;
    item_to_pixel_sample(item, C.w * C.h, pixel, smp);
    Ray r;
    PathState p;
    path_start(P, pixel, pixel % C.w, pixel / C.w, smp, r, p);
    slot_store_ray(s, r);
    reinterpret_cast<uint4 *>(s)[3] = make_uint4(0u, 0u, kNoHit, pixel);                              // hit_t, hit_ref, pixel
    reinterpret_cast<float4 *>(s)[4] = make_float4(p.tr, p.tg, p.tb, __uint_as_float(smp));          // throughput, sample
    reinterpret_cast<uint2 *>(s)[10] = make_uint2(0u, WF_MISS);                                       // bounce, cls
}

__global__ void __launch_bounds__(256) wf_generate(const __grid_constant__ RenderParams P, const WavefrontPool W) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W.n_slots) return;
    if ((unsigned long long)i < W.total_items) wf_spawn(P, W.slots + i, i);
    else W.slots[i].pixel = kDeadPixel;
}

// ------------------------------------------------------------------------------------------
// wf_trace: persistent warps.  Each warp owns a contiguous chunk of the pool; a lane that
// finishes its ray parks the result and, once a quarter of the warp is parked (or nothing is
// left), the parked lanes write their hit + material class back and take the next slots of the
// warp's chunk -- no lane waits for the longest ray of its warp, and there is no global atomic
// on the ray-fetch path.
template <int STACK, bool COUNT>
__global__ void __launch_bounds__(kPathBlock, kPathMinBlocks) wf_trace(const __grid_constant__ RenderParams P, const WavefrontPool W) {
    Trav T;
    uint2 stack[STACK];
    T.cur = kTravDone;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t per_warp = (W.n_slots + n_warps - 1) / n_warps;
    uint32_t cursor = warp * per_warp;                                   // warp-uniform
    const uint32_t chunk_end = min(cursor + per_warp, W.n_slots);
    uint32_t slot = 0;
    bool have = false, parked = false;
    uint32_t rays = 0;
    TraversalCounters ctr;

    while (true) {
        const unsigned idle = __ballot_sync(0xffffffffu, !have);
        if (__popc(idle) >= 8 || idle == 0xffffffffu) {
            // ---- retire: hit + material class back into the slot ----
            if (parked) {
                uint32_t cls = WF_MISS;
                if (T.best.ref != kNoHit) {
                    const uint32_t mat = (T.best.ref & kQuadFlagD) ? __ldg(&P.scene.quad_meta[T.best.ref & ~kQuadFlagD]).y
                                                                   : __ldg(&P.scene.sphere_meta[T.best.ref]).y;
                    const uint32_t kind = __ldg(&P.scene.materials[mat].kind);
                    cls = kind == B200RT_MAT_LIGHT ? WF_LIGHT
                          : (kind == B200RT_MAT_LAMBERTIAN ? WF_LAMBERT : (kind == B200RT_MAT_METAL ? WF_METAL : WF_DIELECTRIC));
                }
                PathSlot *s = W.slots + slot;
                s->hit_t = T.best.t;
                s->hit_ref = T.best.ref;
                s->cls = cls;
                parked = false;
            }
            // ---- refill from the warp's own chunk ----
            if (cursor < chunk_end) {
                const uint32_t idx = cursor + __popc(idle & lanemask_lt());
                cursor += __popc(idle);
                if (!have && idx < chunk_end) {
                    slot = idx;
                    const PathSlot *s = W.slots + slot;
                    if (s->pixel != kDeadPixel) {
                        Ray r;
                        slot_load_ray(s, r);
                        trav_init(T, r.ox, r.oy, r.oz, r.dx, r.dy, r.dz, kRayTmin, kRayTmax);
                        trav_hoisted<COUNT>(P.scene, T, &ctr);
                        have = true;
                    }
                }
            } else if (idle == 0xffffffffu) {
                break;
            }
        }
        if (have) {
            trav_iteration<COUNT>(P.scene, T, stack, &ctr);
            if (trav_done(T)) { have = false; parked = true; ++rays; }
        }
    }
    write_counters(P, rays, COUNT, ctr);
}

// ------------------------------------------------------------------------------------------
// wf_sort: builds the five per-material-class queues of live slots.  Compaction by warp ballot +
// prefix sums: per class, each warp ballots its members (rank = popc of lower lanes), the warp
// totals are prefix-summed through shared memory, and ONE global atomicAdd per class per block
// reserves the block's range of the queue.
__global__ void __launch_bounds__(kSortBlock) wf_sort(const WavefrontPool W) {
    __shared__ uint32_t warp_count[WF_CLASSES][kSortBlock / 32];
    __shared__ uint32_t block_base[WF_CLASSES];
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31u, wid = threadIdx.x >> 5;
    uint32_t cls = 0xFFu;
    if (i < W.n_slots) {
        const uint4 q = reinterpret_cast<const uint4 *>(W.slots + i)[5];   // bounce, cls, pad, pad
        const uint32_t pixel = W.slots[i].pixel;
        if (pixel != kDeadPixel) cls = q.y;
    }
    uint32_t my_rank = 0;
#pragma unroll
    for (int c = 0; c < WF_CLASSES; ++c) {
        const unsigned m = __ballot_sync(0xffffffffu, cls == (uint32_t)c);
        if (cls == (uint32_t)c) my_rank = __popc(m & lanemask_lt());
        if (lane == 0) warp_count[c][wid] = __popc(m);
    }
    __syncthreads();
    if (threadIdx.x < WF_CLASSES) {
        uint32_t total = 0;
        for (int w = 0; w < kSortBlock / 32; ++w) { const uint32_t n = warp_count[threadIdx.x][w]; warp_count[threadIdx.x][w] = total; total += n; }
        block_base[threadIdx.x] = total ? atomicAdd(&W.queue_count[threadIdx.x], total) : 0u;
    }
    __syncthreads();
    if (cls != 0xFFu) W.queue[(size_t)cls * W.n_slots + block_base[cls] + warp_count[cls][wid] + my_rank] = i;
}

// ------------------------------------------------------------------------------------------
// wf_shade: one thread per queue entry; the five queues are walked back to back, so all lanes of
// a warp (except at the four boundaries) shade the same material class.
__global__ void __launch_bounds__(128) wf_shade(const __grid_constant__ RenderParams P, const WavefrontPool W) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t cls = 0;
    bool valid = false;
#pragma unroll
    for (int c = 0; c < WF_CLASSES; ++c) {
        const uint32_t n = W.queue_count[c];
        if (!valid) {
            if (i < n) { cls = c; valid = true; }
            else i -= n;
        }
    }
    if (!valid) return;
    PathSlot *s = W.slots + W.queue[(size_t)cls * W.n_slots + i];
    const uint4 hq = reinterpret_cast<const uint4 *>(s)[3];      // hit_t (2 words), hit_ref, pixel
    const float4 th = reinterpret_cast<const float4 *>(s)[4];    // throughput, sample
    uint32_t bounce = s->bounce;
    const uint32_t pixel = hq.w, smp = __float_as_uint(th.w);
    PathState p{th.x, th.y, th.z};
    const Hit h{__hiloint2double((int)hq.y, (int)hq.x), hq.z};
    Ray r;
    if (h.ref != kNoHit) slot_load_ray(s, r);
    float add_r, add_g, add_b;
    const bool cont = path_bounce(P, h, pixel, smp, bounce, r, p, add_r, add_g, add_b);
    if (add_r != 0.f || add_g != 0.f || add_b != 0.f) {
        float *o = P.out + (size_t)pixel * 3;
        atomicAdd(o + 0, add_r * P.scale); atomicAdd(o + 1, add_g * P.scale); atomicAdd(o + 2, add_b * P.scale);
    }
    if (cont) {
        slot_store_ray(s, r);
        reinterpret_cast<float4 *>(s)[4] = make_float4(p.tr, p.tg, p.tb, th.w);
        s->bounce = bounce;
    } else {
        // path ended: regenerate the slot with the next work item (warp-aggregated fetch)
        const unsigned mask = __activemask();
        const uint32_t lane = threadIdx.x & 31u, leader = __ffs(mask) - 1u;
        unsigned long long base = 0;
        if (lane == leader) base = atomicAdd(W.next_item, (unsigned long long)__popc(mask));
        base = __shfl_sync(mask, base, leader);
        const unsigned long long item = base + __popc(mask & lanemask_lt());
        if (item < W.total_items) {
            wf_spawn(P, s, item);
        } else {
            s->pixel = kDeadPixel;
            atomicAdd(W.alive, 0xFFFFFFFFu);   // -1
        }
    }
}

__global__ void wf_reset(const WavefrontPool W) {
    if (threadIdx.x < WF_CLASSES) W.queue_count[threadIdx.x] = 0;
}

size_t wavefront_pool_alloc_bytes(uint32_t n_slots) {
    return (size_t)n_slots * (sizeof(PathSlot) + WF_CLASSES * sizeof(uint32_t)) + 4096;
}

// Carves the pool out of one device allocation.
void wavefront_pool_layout(void *base, uint32_t n_slots, WavefrontPool &W) {
    char *p = static_cast<char *>(base);
    auto take = [&](size_t bytes) { char *q = p; p += (bytes + 255) / 256 * 256; return q; };
    W.n_slots = n_slots;
    W.slots = (PathSlot *)take((size_t)n_slots * sizeof(PathSlot));
    W.queue = (uint32_t *)take((size_t)WF_CLASSES * n_slots * sizeof(uint32_t));
    W.queue_count = (uint32_t *)take(8 * sizeof(uint32_t));
    W.alive = W.queue_count + 6;
    W.next_item = (unsigned long long *)take(sizeof(unsigned long long));
}

template <int STACK>
static cudaError_t run_wavefront_t(const RenderParams &P, WavefrontPool W, bool count, cudaStream_t st, int sm_count,
                                   unsigned long long *launches) {
    const CameraParams &C = P.cam;
    W.total_items = (unsigned long long)C.w * C.h * P.sample_count;
    cudaError_t e;
    if (!(P.flags & kRenderAccumulate))
        if ((e = cudaMemsetAsync(P.out, 0, (size_t)C.w * C.h * 3 * sizeof(float), st)) != cudaSuccess) return e;
    if (W.total_items == 0 || C.max_depth == 0) return cudaSuccess;
    const uint32_t live = (uint32_t)(W.total_items < W.n_slots ? W.total_items : W.n_slots);
    const unsigned long long first_next = live;
    if ((e = cudaMemcpyAsync(W.next_item, &first_next, sizeof first_next, cudaMemcpyHostToDevice, st)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(W.alive, &live, sizeof live, cudaMemcpyHostToDevice, st)) != cudaSuccess) return e;
    wf_generate<<<(W.n_slots + 255) / 256, 256, 0, st>>>(P, W);
    ++*launches;
    const int trace_blocks = sm_count * kPathMinBlocks;
    uint32_t alive = live;
    unsigned long long waves = 0;
    for (; alive != 0; ++waves) {
        wf_reset<<<1, 32, 0, st>>>(W);
        if (count) wf_trace<STACK, true><<<trace_blocks, kPathBlock, 0, st>>>(P, W);
        else wf_trace<STACK, false><<<trace_blocks, kPathBlock, 0, st>>>(P, W);
        wf_sort<<<(W.n_slots + kSortBlock - 1) / kSortBlock, kSortBlock, 0, st>>>(W);
        wf_shade<<<(W.n_slots + 127) / 128, 128, 0, st>>>(P, W);
        *launches += 4;
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        if ((waves & 7) == 7 || W.total_items <= W.n_slots) {
            // the only host round trip: poll the live-slot counter (every 8 waves in steady state)
            if ((e = cudaMemcpyAsync(&alive, W.alive, sizeof alive, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
            if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
        }
    }
    if (std::getenv("B200RT_WF_DEBUG"))
        std::fprintf(stderr, "[b200rt] wavefront: %llu waves over a pool of %u slots, %llu work items\n", waves, W.n_slots, W.total_items);
    return cudaSuccess;
}

cudaError_t run_wavefront(int stack, const RenderParams &P, const WavefrontPool &W, bool count, cudaStream_t st, int sm_count,
                          unsigned long long *launches) {
    return with_stack(stack, [&](auto K) { return run_wavefront_t<K.value>(P, W, count, st, sm_count, launches); });
}

}  // namespace b200rt
