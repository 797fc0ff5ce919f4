// api.cu -- implementation of the C ABI declared in include/b200rt.h.
//
// Host side of the drop-in boundary: validates the scene description's structure, uploads the
// caller's arrays as they are, has one of the two builders decide the 4-wide BVH and its leaf order
// (bvh_builder.cpp on the host, with primitive bounds exactly as the reference's constructors
// compute them, sphere.h:112-123, parallelogram.h:281-295; or lbvh.cu on the device), has
// scene_layout.cu lay the primitives out in that order and launches the kernels.  There is no CPU
// compute path: every entry point that produces hits or pixels fails with B200RT_ENODEVICE without a GPU.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/b200rt.h"
#include "bvh_builder.h"
#include "devmem.h"
#include "kernels.h"
#include "thread_pool.h"

using namespace b200rt;

namespace b200rt {
cudaError_t build_lbvh_device(const B200rtSphere *d_sph, uint32_t n_sph, const B200rtQuad *d_quads, uint32_t n_quad,
                              uint32_t max_hoisted, uint32_t *sphere_order, uint32_t *quad_order, float4 **nodes_out,
                              uint32_t *n_nodes_out, uint32_t *depth_out, uint32_t *n_hoisted_out, uint32_t hoisted_ref_out[kMaxHoisted]);
cudaError_t assemble_scene_device(const B200rtSphere *sph, const uint32_t *sphere_order, uint32_t n_sph, const B200rtQuad *quads,
                                  const uint32_t *quad_order, uint32_t n_quad, const B200rtMaterial *mats, uint32_t n_mat,
                                  double2 *out_sph, uint2 *out_sph_meta, double2 *out_quads, uint2 *out_quad_meta,
                                  DeviceMaterial *out_mats, int bad_out[2]);
}

namespace {

thread_local std::string g_last_error;

int fail(int code, const std::string &msg) {
    g_last_error = msg;
    return code;
}
#define CUDA_TRY(expr)                                                                         \
    do {                                                                                       \
        cudaError_t e_ = (expr);                                                               \
        if (e_ != cudaSuccess) {                                                               \
            cudaGetLastError();                                                                \
            return fail(e_ == cudaErrorMemoryAllocation ? B200RT_ENOMEM : B200RT_ECUDA,         \
                        std::string(#expr) + ": " + cudaGetErrorString(e_));                   \
        }                                                                                      \
    } while (0)

double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; cudaGetLastError(); }
        ok = cudaSetDevice(dev) == cudaSuccess;
        if (!ok) cudaGetLastError();
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

constexpr uint32_t kSceneMagic = 0xB200577Eu, kMultiMagic = 0xB2003171u;

struct SceneImpl {
    uint32_t magic = kSceneMagic;
    int device = 0;
    std::mutex mu;                   // a handle is not re-entrant: calls on it are serialised
    DeviceScene d{};                 // device pointers
    // [0] nodes, [1] spheres, [2] sphere_meta, [3] quads, [4] quad_meta, [5] materials
    void *allocs[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    size_t alloc_bytes[6] = {0, 0, 0, 0, 0, 0};
    bool peer_visible = false;       // the arrays are peer-visible buffers (devmem.h): a multi-device scene copies them device to device
    B200rtSceneInfo info{};
    int stack = 32;
    unsigned long long *d_counters = nullptr;   // [0] rays, [1] node visits, [2] primitive tests, [3] of which quad tests
    unsigned long long *d_viol = nullptr;       // bounds-checked build only: [4] violation counters
    float *d_frame = nullptr;        // scratch frame for the host-buffer render entry
    size_t frame_floats = 0;
    double *d_rays = nullptr; int32_t *d_prim = nullptr; double *d_t = nullptr;   // raycast scratch
    size_t ray_capacity = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t ev_pool = nullptr;   // wavefront: the path-slot pool is free again (renders of one scene share it)
    void *d_pool = nullptr;          // wavefront path-slot pool
    uint32_t pool_slots = 0;
    cudaEvent_t ev_tail = nullptr;   // the tail scratch is free again (renders of one scene share it)
    void *d_tail = nullptr;          // chunked tail tiles of the path kernel: partial sums and arrival counters, zero between launches
    size_t tail_bytes = 0;
    void *d_adapt = nullptr;         // adaptive sampling: int64 planes, counts, masks and tile lists (AdaptiveBuffers)
    size_t adapt_bytes = 0;
    int sm_count = 148;
};

// The scene resident on several devices of this process (b200rt_scene_create_multi).
struct MultiImpl {
    uint32_t magic = kMultiMagic;
    std::mutex mu;
    std::vector<SceneImpl *> dev;            // dev[0] was built; the others are device-to-device copies of it
    std::vector<cudaStream_t> stream;        // one non-blocking stream per device
    std::vector<cudaEvent_t> ev_render, ev_xchg;
    std::vector<float *> frame;              // per-device FP32 SUM frame
    float *scratch = nullptr;                // devices[0]: landing buffer of the exchange without peer mapping
    size_t frame_floats = 0;
    bool peers = false;                      // every device can dereference every other device's pool memory
    double replicate_ms = 0;
};

// Scene arrays: stream-ordered pool memory, or (multi-device scenes) peer-visible buffers.
cudaError_t scene_alloc(SceneImpl *s, int slot, size_t bytes) {
    void *p = nullptr;
    const cudaError_t e = s->peer_visible ? peer_buffer_acquire(s->device, bytes, &p) : dev_alloc_async(&p, bytes, 0);
    if (e != cudaSuccess) return e;
    s->allocs[slot] = p;
    s->alloc_bytes[slot] = bytes;
    return cudaSuccess;
}
void scene_free_arrays(SceneImpl *s) {
    for (int i = 0; i < 6; ++i) {
        if (s->peer_visible) peer_buffer_release(s->device, s->allocs[i]);
        else dev_free(s->allocs[i]);
        s->allocs[i] = nullptr;
        s->alloc_bytes[i] = 0;
    }
}

SceneImpl *as_scene(void *h) {
    SceneImpl *s = static_cast<SceneImpl *>(h);
    return (s && s->magic == kSceneMagic) ? s : nullptr;
}
MultiImpl *as_multi(void *h) {
    MultiImpl *m = static_cast<MultiImpl *>(h);
    return (m && m->magic == kMultiMagic) ? m : nullptr;
}
// the single-device scene behind either kind of handle (devices[0] of a multi-device one)
SceneImpl *root_scene(void *h) {
    if (MultiImpl *m = as_multi(h)) return m->dev.empty() ? nullptr : m->dev[0];
    return as_scene(h);
}

int device_count_quiet() {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// ---- reference-exact host geometry helpers ------------------------------------------------
struct V3 { double x, y, z; };
inline V3 sub(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
inline V3 add(V3 a, V3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
inline V3 mul(V3 a, double d) { return {a.x * d, a.y * d, a.z * d}; }
inline V3 divv(V3 a, double d) { return mul(a, 1 / d); }   // operator/= multiplies by 1/d (vec3d.h:31)
inline V3 crossv(V3 a, V3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
inline double mag2(V3 a) { return a.x * a.x + a.y * a.y + a.z * a.z; }
inline double mag(V3 a) { return std::sqrt(mag2(a)); }
inline V3 unitv(V3 a) { return divv(a, mag(a)); }
inline V3 v3(const double *p) { return {p[0], p[1], p[2]}; }
inline void put(double *p, V3 v) { p[0] = v.x; p[1] = v.y; p[2] = v.z; }

Box3 sphere_box(const B200rtSphere &s) {   // sphere.h:112-123
    Box3 b;
    for (int a = 0; a < 3; ++a) {
        const double p = s.c[a] - s.r, q = s.c[a] + s.r;
        b.lo[a] = std::fmin(p, q);
        b.hi[a] = std::fmax(p, q);
    }
    return b;
}
Box3 quad_box(const B200rtQuad &q) {       // parallelogram.h:281-295 + aabb.h ensure_min_axis_length
    Box3 b;
    const V3 v = v3(q.v), s1 = v3(q.s1), s2 = v3(q.s2);
    const V3 pts[4] = {v, add(v, s1), add(v, s2), add(add(v, s1), s2)};
    for (int a = 0; a < 3; ++a) { b.lo[a] = std::numeric_limits<double>::infinity(); b.hi[a] = -b.lo[a]; }
    for (const V3 &p : pts) {
        const double c[3] = {p.x, p.y, p.z};
        for (int a = 0; a < 3; ++a) { b.lo[a] = std::fmin(b.lo[a], c[a]); b.hi[a] = std::fmax(b.hi[a], c[a]); }
    }
    for (int a = 0; a < 3; ++a) {
        const double size = b.hi[a] - b.lo[a];
        if (size < 1e-4) { const double pad = (1e-4 - size) / 2; b.lo[a] -= pad; b.hi[a] += pad; }
    }
    return b;
}

int validate_desc(const B200rtSceneDesc *d, bool check_prims = true) {
    if (!d) return fail(B200RT_EINVAL, "scene description is NULL");
    if ((d->n_materials && !d->materials) || (d->n_spheres && !d->spheres) || (d->n_quads && !d->quads))
        return fail(B200RT_EINVAL, "scene description has a count without an array");
    const uint64_t n_prims = d->n_spheres + d->n_quads;
    if (n_prims > 0x7FFFFFFFull) return fail(B200RT_EINVAL, "too many primitives");
    // scene creation checks material kinds and per-primitive indices on the device (scene_layout.cu); the host loops
    // below serve b200rt_selftest_bvh, which runs without one
    if (!check_prims) return B200RT_OK;
    for (uint64_t i = 0; i < d->n_materials; ++i)
        if (d->materials[i].kind > B200RT_MAT_LIGHT)
            return fail(B200RT_EINVAL, "unknown material kind " + std::to_string(d->materials[i].kind) +
                                           " (closed set: Lambertian, Metal, Dielectric, DiffuseLight)");
    for (uint64_t i = 0; i < d->n_spheres; ++i)
        if (d->spheres[i].mat >= d->n_materials || d->spheres[i].prim >= n_prims)
            return fail(B200RT_EINVAL, "sphere " + std::to_string(i) + ": material or primitive index out of range");
    for (uint64_t i = 0; i < d->n_quads; ++i)
        if (d->quads[i].mat >= d->n_materials || d->quads[i].prim >= n_prims)
            return fail(B200RT_EINVAL, "quad " + std::to_string(i) + ": material or primitive index out of range");
    return B200RT_OK;
}

// Runs body(lo, hi) over [0, n) split into chunks on a temporary pool (serial when small).
template <typename F>
void parallel_ranges(uint64_t n, int threads, F body) {
    if (n < (1u << 16) || threads <= 1) { body((uint64_t)0, n); return; }
    ThreadPool pool(threads);
    const int chunks = threads * 4;
    pool.parallel_for(chunks, [&](int c) { body(n * c / chunks, n * (c + 1) / chunks); });
}
int host_threads(const B200rtBuildOpts *o) {
    return (o && o->build_threads > 0) ? o->build_threads : ThreadPool::hardware_threads();
}

void compute_boxes(const B200rtSceneDesc *d, std::vector<Box3> &boxes, int threads) {
    boxes.resize(d->n_spheres + d->n_quads);
    parallel_ranges(d->n_spheres, threads, [&](uint64_t lo, uint64_t hi) {
        for (uint64_t i = lo; i < hi; ++i) boxes[i] = sphere_box(d->spheres[i]);
    });
    parallel_ranges(d->n_quads, threads, [&](uint64_t lo, uint64_t hi) {
        for (uint64_t i = lo; i < hi; ++i) boxes[d->n_spheres + i] = quad_box(d->quads[i]);
    });
}

BuildParams build_params(const B200rtBuildOpts *o) {
    BuildParams p;
    if (o) {
        if (o->max_leaf_prims > 0) p.max_leaf_prims = o->max_leaf_prims;
        if (o->sah_bins > 0) p.sah_bins = o->sah_bins;
        if (o->build_threads > 0) p.threads = o->build_threads;
    }
    return p;
}

void free_scene(SceneImpl *s) {
    if (!s) return;
    DeviceGuard g(s->device);
    cudaDeviceSynchronize();   // kernels of any stream may still read the scene
    scene_free_arrays(s);
    dev_free(s->d_counters);
    dev_free(s->d_viol);
    dev_free(s->d_frame);
    dev_free(s->d_rays);
    dev_free(s->d_prim);
    dev_free(s->d_t);
    dev_free(s->d_pool);
    dev_free(s->d_tail);
    dev_free(s->d_adapt);
    if (s->ev0) cudaEventDestroy(s->ev0);
    if (s->ev1) cudaEventDestroy(s->ev1);
    if (s->ev_pool) cudaEventDestroy(s->ev_pool);
    if (s->ev_tail) cudaEventDestroy(s->ev_tail);
    s->magic = 0;
    delete s;
}

void free_multi(MultiImpl *m) {
    if (!m) return;
    for (size_t i = 0; i < m->dev.size(); ++i) {
        if (!m->dev[i]) continue;
        DeviceGuard g(m->dev[i]->device);
        if (i < m->stream.size() && m->stream[i]) cudaStreamSynchronize(m->stream[i]);
        if (i < m->frame.size()) peer_buffer_release(m->dev[i]->device, m->frame[i]);
        if (i == 0) dev_free(m->scratch);
        if (i < m->ev_render.size() && m->ev_render[i]) cudaEventDestroy(m->ev_render[i]);
        if (i < m->ev_xchg.size() && m->ev_xchg[i]) cudaEventDestroy(m->ev_xchg[i]);
        if (i < m->stream.size() && m->stream[i]) cudaStreamDestroy(m->stream[i]);
    }
    for (SceneImpl *s : m->dev) free_scene(s);
    m->magic = 0;
    delete m;
}

int fill_camera(const B200rtCamera *cam, CameraParams &C) {
    if (!cam) return fail(B200RT_EINVAL, "camera is NULL");
    if (cam->image_w == 0 || cam->image_h == 0 || cam->image_w > 65536 || cam->image_h > 65536 ||
        cam->image_w * cam->image_h > 0x7FFFFFFFull)   // pixel indices are 32-bit
        return fail(B200RT_EINVAL, "image dimensions out of range");
    if (cam->max_depth > 0xFFFFFFFFull) return fail(B200RT_EINVAL, "max_depth out of range");
    for (int a = 0; a < 3; ++a) {
        C.center[a] = cam->center[a]; C.pixel00[a] = cam->pixel00[a];
        C.delta_x[a] = cam->delta_x[a]; C.delta_y[a] = cam->delta_y[a];
        C.disk_x[a] = cam->disk_x[a]; C.disk_y[a] = cam->disk_y[a];
        C.background[a] = (float)cam->background[a];
    }
    C.defocus = cam->defocus_angle > 0 ? 1u : 0u;   // camera.h:186 (defocus_angle <= 0 -> pinhole)
    C.w = (uint32_t)cam->image_w; C.h = (uint32_t)cam->image_h; C.max_depth = (uint32_t)cam->max_depth;
    return B200RT_OK;
}

// Resolves the sample range of a render call: count 0 means camera.spp unless B200RT_FLAG_EXACT_COUNT is set.
int sample_range_of(const B200rtCamera *cam, const B200rtRenderOpts &o, uint64_t *count_out) {
    const uint64_t count = (o.sample_count || (o.flags & B200RT_FLAG_EXACT_COUNT)) ? o.sample_count : cam->spp;
    if (count > 0xFFFFFFFFull || o.sample_offset + count > 0xFFFFFFFFull) return fail(B200RT_EINVAL, "sample range out of range");
    if (o.variant != B200RT_VARIANT_MEGAKERNEL && o.variant != B200RT_VARIANT_WAVEFRONT)
        return fail(B200RT_EINVAL, "unknown kernel variant");
    *count_out = count;
    return B200RT_OK;
}

// What a render of `cam` with `opts` (NULL: the defaults) on scene s takes from its arguments: the options in o; the camera,
// the sample range, the seed, flags and counters in P; and the two schedule rules of the path kernels -- the work-pool
// item order (P.group_shift) and the order of the traversal steps (leaf_first).  The caller sets the outputs and the scale.
int render_setup(SceneImpl *s, const B200rtCamera *cam, const B200rtRenderOpts *opts, B200rtRenderOpts &o, RenderParams &P,
                 bool &leaf_first) {
    if (int rc = fill_camera(cam, P.cam)) return rc;
    o = opts ? *opts : B200rtRenderOpts{};
    uint64_t count = 0;
    if (int rc = sample_range_of(cam, o, &count)) return rc;
    P.scene = s->d;
    P.seed = o.seed;
    P.sample_begin = (uint32_t)o.sample_offset;
    P.sample_count = (uint32_t)count;
    P.flags = o.flags;
    P.counters = s->d_counters;
    // work-pool item order (kernels.cu): same-pixel groups of 8 when only light hits contribute (black background)
    P.group_shift = (cam->background[0] == 0.0 && cam->background[1] == 0.0 && cam->background[2] == 0.0) ? 3u : 0u;
    if (const char *g = std::getenv("B200RT_GROUP_SHIFT")) P.group_shift = (uint32_t)std::min(5, std::max(0, std::atoi(g)));   // experiments
    // order of the node and the leaf step inside a traversal iteration (traverse.cuh): leaf first when quads dominate
    leaf_first = s->info.n_quads > s->info.n_spheres;
    if (const char *lf = std::getenv("B200RT_LEAF_FIRST")) leaf_first = lf[0] == '1';   // experiments
    return B200RT_OK;
}

// Moments and adaptive renders run on the tile-pool kernel without traversal counters; `what` starts the message.
int require_default_kernel(const B200rtRenderOpts &o, const char *what) {
    if (o.variant == B200RT_VARIANT_WAVEFRONT || (o.flags & (B200RT_FLAG_THREAD_PIXELS | B200RT_FLAG_COUNTERS)))
        return fail(B200RT_EINVAL, std::string(what) + " the default kernel only: no wavefront variant, B200RT_FLAG_THREAD_PIXELS or B200RT_FLAG_COUNTERS");
    return B200RT_OK;
}

// The chunked tail of the tile-pool grid (RenderParams::tail_first): the last `tiles` tiles of the image are rendered by
// blocks of about 1/`chunks` of their samples each, so that short blocks fill the SMs while the last whole tiles drain.
// Default: twice the blocks the GPU holds at once, 8 chunks of at least 8 samples.  B200RT_TAIL_TILES=R[,K] forces R tail
// tiles and K chunks per tile (R = 0: whole tiles only), for A/B measurements and tests.
struct TailPlan {
    uint32_t tiles = 0, chunks = 8, min_chunk = 8;
    bool forced = false;
};
int plan_tail(SceneImpl *s, const CameraParams &C, PathMode mode, bool leaf_first, TailPlan *t) {
    const uint32_t tiles = path_tiles(C.w, C.h);
    if (const char *e = std::getenv("B200RT_TAIL_TILES")) {
        long long r = 0, k = 0;
        const int n = std::sscanf(e, "%lld,%lld", &r, &k);
        t->tiles = (uint32_t)std::min<long long>(tiles, std::max(0ll, r));
        if (n == 2) { t->chunks = (uint32_t)std::max(1ll, std::min(k, 1ll << 22)); t->min_chunk = 1; }
        t->forced = true;
        return B200RT_OK;
    }
    int resident = 0;
    if (cudaError_t e = path_resident_blocks(s->stack, mode, leaf_first, s->sm_count, &resident); e != cudaSuccess) {
        cudaGetLastError();
        return fail(B200RT_ECUDA, std::string("path kernel occupancy: ") + cudaGetErrorString(e));
    }
    t->tiles = (uint32_t)std::min<uint64_t>(tiles, 2ull * (uint64_t)std::max(0, resident));
    return B200RT_OK;
}

// Scene-spanning primitives the builders take out of the tree (bvh_builder.h spanning_key): up to kMaxHoisted by
// default.  B200RT_HOISTED=0 keeps every primitive in the tree, for A/B measurements and tests.
uint32_t max_hoisted() {
    const char *e = std::getenv("B200RT_HOISTED");
    return e ? (uint32_t)std::max(0ll, std::min<long long>(std::atoll(e), kMaxHoisted)) : kMaxHoisted;
}

// Points P at the scene's tail scratch for `tail_tiles` tiles, growing it if needed.  Renders of one scene share the
// scratch: the caller's stream waits (on the device) until the previous render is done with it.  Every launch leaves it zero.
cudaError_t tail_scratch(SceneImpl *s, uint32_t tail_tiles, bool moments, cudaStream_t st, RenderParams *P) {
    const size_t bytes = tail_scratch_bytes(tail_tiles, moments);
    if (bytes > s->tail_bytes) {
        if (s->d_tail) { cudaEventSynchronize(s->ev_tail); dev_free(s->d_tail); s->d_tail = nullptr; s->tail_bytes = 0; }
        if (cudaError_t e = dev_alloc(&s->d_tail, bytes); e != cudaSuccess) return e;
        s->tail_bytes = bytes;
        if (cudaError_t e = cudaMemsetAsync(s->d_tail, 0, bytes, st); e != cudaSuccess) return e;
    }
    if (cudaError_t e = cudaStreamWaitEvent(st, s->ev_tail, 0); e != cudaSuccess) return e;
    P->tail_acc = static_cast<long long *>(s->d_tail);
    P->tail_arrivals = reinterpret_cast<uint32_t *>(static_cast<char *>(s->d_tail) + bytes - (size_t)tail_tiles * sizeof(uint32_t));
    return cudaSuccess;
}

// One launch's chunking of its tail tiles: the chunk is a multiple of 2^group_shift samples (so same-pixel item groups
// stay whole and chunks partition the tile's items, kernels.cu block_items).  A launch whose samples make one chunk keeps
// whole tiles, unless the chunk count was forced.  `tiles`: the tiles the launch renders (the last of them are chunked).
void chunk_tail(const TailPlan &t, uint32_t tiles, RenderParams &Q) {
    const uint32_t n = Q.sample_count, group = 1u << Q.group_shift;
    uint32_t chunk = std::max(t.min_chunk, (uint32_t)(((uint64_t)n + t.chunks - 1) / t.chunks));
    chunk = (uint32_t)(((uint64_t)chunk + group - 1) / group * group);
    const uint32_t k = (uint32_t)(((uint64_t)n + chunk - 1) / chunk);
    if (k <= 1 && !t.forced) return;
    Q.tail_first = tiles - std::min(t.tiles, tiles);
    Q.tail_chunks = k;
    Q.tail_chunk_samples = chunk;
}

// After a render enqueued on `st` between s->ev0 and s->ev1: its four counters and its kernel time into *stats.  The copy
// is ordered on st, which may be a caller's non-blocking stream, and st is synchronised.
cudaError_t read_stats(SceneImpl *s, cudaStream_t st, B200rtStats *stats) {
    unsigned long long c[4];
    float ms = 0;
    cudaError_t e = cudaMemcpyAsync(c, s->d_counters, sizeof c, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, s->ev0, s->ev1);
    if (e != cudaSuccess) return e;
    stats->kernel_ms = ms;
    stats->rays = c[0]; stats->node_visits = c[1]; stats->prim_tests = c[2]; stats->quad_tests = c[3];
    return cudaSuccess;
}

// Grows the scene's scratch frame (the host-buffer renders' device output) to at least `floats` floats.
cudaError_t grow_frame(SceneImpl *s, size_t floats) {
    if (floats <= s->frame_floats) return cudaSuccess;
    if (s->d_frame) { dev_free(s->d_frame); s->d_frame = nullptr; s->frame_floats = 0; }
    if (cudaError_t e = dev_alloc(&s->d_frame, floats * sizeof(float)); e != cudaSuccess) return e;
    s->frame_floats = floats;
    return cudaSuccess;
}

// Enqueues the path kernel(s) of one render call on `st` (the caller holds s->mu and has made s->device current).
// d_m2 (optional): the second-moment plane, written by the moments instantiation of the default kernel.
int render_on_device(SceneImpl *s, const B200rtCamera *cam, const B200rtRenderOpts *opts, float *d_out,
                     cudaStream_t st, B200rtStats *stats, bool sync_for_stats, float *d_m2 = nullptr) {
    RenderParams P{};
    B200rtRenderOpts o;
    bool leaf_first;
    if (int rc = render_setup(s, cam, opts, o, P, leaf_first)) return rc;
    if (d_m2)
        if (int rc = require_default_kernel(o, "moments are rendered by")) return rc;
    const uint64_t count = P.sample_count;
    const PathMode mode = d_m2 ? PathMode::Moments : (o.flags & B200RT_FLAG_COUNTERS) ? PathMode::Counters : PathMode::Plain;
    P.out = d_out;
    P.out_m2 = d_m2;
    P.scale = (o.flags & B200RT_FLAG_SUM) || count == 0 ? 1.0f : (float)(1.0 / (double)count);
    CUDA_TRY(cudaMemsetAsync(s->d_counters, 0, 4 * sizeof(unsigned long long), st));
    unsigned long long launches = 1;
    CUDA_TRY(cudaEventRecord(s->ev0, st));
    if (count == 0) {
        // an empty share of a sample split: no samples, so the sum is zero (nothing to add under ACCUMULATE)
        launches = 0;
        if (!(o.flags & B200RT_FLAG_ACCUMULATE)) {
            CUDA_TRY(cudaMemsetAsync(d_out, 0, (size_t)cam->image_w * cam->image_h * 3 * sizeof(float), st));
            if (d_m2) CUDA_TRY(cudaMemsetAsync(d_m2, 0, (size_t)cam->image_w * cam->image_h * 3 * sizeof(float), st));
        }
    } else if (o.variant == B200RT_VARIANT_WAVEFRONT) {
        // pool of path slots: 2^21 by default (B200RT_WF_SLOTS overrides, for experiments).  Renders of one scene
        // share the pool: each waits (on the device) for the previous one to be done with it.
        uint32_t want = 1u << 21;
        if (const char *e = std::getenv("B200RT_WF_SLOTS")) want = (uint32_t)std::max(1024ll, std::atoll(e));
        const unsigned long long items = (unsigned long long)cam->image_w * cam->image_h * count;
        if (items < want) want = (uint32_t)std::max(1024ull, items);
        if (want != s->pool_slots) {
            if (s->d_pool) { cudaEventSynchronize(s->ev_pool); dev_free(s->d_pool); s->d_pool = nullptr; s->pool_slots = 0; }
            CUDA_TRY(dev_alloc(&s->d_pool, wavefront_pool_alloc_bytes(want)));
            s->pool_slots = want;
        }
        CUDA_TRY(cudaStreamWaitEvent(st, s->ev_pool, 0));
        WavefrontPool W{};
        wavefront_pool_layout(s->d_pool, s->pool_slots, W);
        launches = 0;
        CUDA_TRY(run_wavefront(s->stack, P, W, mode == PathMode::Counters, st, s->sm_count, &launches));
        CUDA_TRY(cudaEventRecord(s->ev_pool, st));
    } else {
        TailPlan tail;
        if (!(o.flags & B200RT_FLAG_THREAD_PIXELS)) {
            if (int rc = plan_tail(s, P.cam, mode, leaf_first, &tail)) return rc;
            if (tail.tiles) CUDA_TRY(tail_scratch(s, tail.tiles, d_m2 != nullptr, st, &P));
        }
        // the tile work pool counts (pixel, sample) items in 32 bits: more than 2^22 samples per pixel go in several launches
        // (2^16 with moments: the range of the x^2 accumulator, kernels.h)
        const uint64_t per_launch = d_m2 ? kMaxSamplesPerLaunchMoments : kMaxSamplesPerLaunch;
        launches = 0;
        for (uint64_t done = 0; done < count; done += per_launch) {
            RenderParams Q = P;
            Q.sample_begin = (uint32_t)(o.sample_offset + done);
            Q.sample_count = (uint32_t)std::min<uint64_t>(per_launch, count - done);
            if (done) Q.flags |= kRenderAccumulate;
            if (tail.tiles) chunk_tail(tail, path_tiles(P.cam.w, P.cam.h), Q);
            CUDA_TRY(launch_path_megakernel(s->stack, Q, mode, leaf_first, st));
            ++launches;
        }
        if (tail.tiles) CUDA_TRY(cudaEventRecord(s->ev_tail, st));
    }
    CUDA_TRY(cudaEventRecord(s->ev1, st));
    if (stats) {
        std::memset(stats, 0, sizeof *stats);
        stats->paths = (uint64_t)cam->image_w * cam->image_h * count;
        stats->kernel_launches = launches;
        stats->n_devices = 1;
        if (sync_for_stats) CUDA_TRY(read_stats(s, st, stats));
    }
    return B200RT_OK;
}

// Points s->d at the arrays in s->allocs, takes `info` and the info.n_hoisted references of the scene-spanning primitives,
// sizes the traversal stack from the tree depth and creates the per-scene launch state (counters, events, the
// bounds-check table of the debug build); `s->device` is current.
int finish_scene(SceneImpl *s, const B200rtSceneInfo &info, const uint32_t *hoisted_ref) {
    static_assert(sizeof(s->d.hoisted_ref) / sizeof(s->d.hoisted_ref[0]) == kMaxHoisted, "DeviceScene::hoisted_ref");
    s->d.n_hoisted = info.n_hoisted;
    for (uint32_t k = 0; k < kMaxHoisted; ++k) s->d.hoisted_ref[k] = k < info.n_hoisted ? hoisted_ref[k] : 0u;
    s->d.nodes = static_cast<const float4 *>(s->allocs[0]);
    s->d.spheres = static_cast<const double2 *>(s->allocs[1]);
    s->d.sphere_meta = static_cast<const uint2 *>(s->allocs[2]);
    s->d.quads = static_cast<const double2 *>(s->allocs[3]);
    s->d.quad_meta = static_cast<const uint2 *>(s->allocs[4]);
    s->d.materials = static_cast<const DeviceMaterial *>(s->allocs[5]);
    if (reinterpret_cast<uintptr_t>(s->d.nodes) & 127)   // trav_node_step forms plane addresses with OR / XOR on the low bits
        return fail(B200RT_ECUDA, "node array is not 128-byte aligned");
    s->info = info;
    s->stack = with_stack((int)(3 * info.tree_depth), [](auto K) { return K.value; });
    s->info.stack_entries = (uint32_t)s->stack;
    s->info.device_bytes = 0;
    for (size_t b : s->alloc_bytes) s->info.device_bytes += b;
    cudaError_t e = dev_alloc(&s->d_counters, 4 * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&s->sm_count, cudaDevAttrMultiProcessorCount, s->device);
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev1);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_pool, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_tail, cudaEventDisableTiming);
#ifdef B200RT_DEBUG_BOUNDS
    if (e == cudaSuccess) e = dev_alloc(&s->d_viol, 4 * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemsetAsync(s->d_viol, 0, 4 * sizeof(unsigned long long), 0);
    s->d.dbg.viol = s->d_viol;
    s->d.dbg.n_nodes = (uint32_t)s->info.n_nodes;
    s->d.dbg.n_spheres = (uint32_t)s->info.n_spheres;
    s->d.dbg.n_quads = (uint32_t)s->info.n_quads;
    s->d.dbg.n_materials = (uint32_t)s->info.n_materials;
    s->d.dbg.stack_cap = (uint32_t)s->stack;
    if (const char *cap = std::getenv("B200RT_DEBUG_STACK_CAP")) s->d.dbg.stack_cap = (uint32_t)std::max(0, std::min(s->stack, std::atoi(cap)));
#endif
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { cudaGetLastError(); return fail(B200RT_ECUDA, std::string("scene setup: ") + cudaGetErrorString(e)); }
    return B200RT_OK;
}

// Makes the scene resident on s->device.  The caller's arrays go up as they are; a builder decides the tree and the
// leaf order -- the GPU LBVH (lbvh.cu) when `gpu_build`, the host SAH builder (bvh_builder.cpp) otherwise or when
// the LBVH is too deep for the largest traversal stack -- and scene_layout.cu lays the primitives out in that order
// and checks them, whichever builder ran.  build_ms is the host builder's time when it built the tree, else all of
// it; upload_ms is the rest.
int scene_build(const B200rtSceneDesc *desc, const B200rtBuildOpts *opts, bool gpu_build, SceneImpl *s) {
    const double t0 = now_ms();
    if (desc->n_spheres > kLeafIndexMask || desc->n_quads > kLeafIndexMask)
        return fail(B200RT_EINVAL, "too many primitives for the leaf encoding (2^26 per type)");
    if (desc->n_materials > 0xFFFFFFFFull) return fail(B200RT_EINVAL, "too many materials");
    const uint32_t n_sph = (uint32_t)desc->n_spheres, n_quad = (uint32_t)desc->n_quads, n_mat = (uint32_t)desc->n_materials;
    // the caller's records (pinned staging, pipelined) and the leaf order are scratch; the scene's own arrays are
    // allocated straight into s->allocs so that free_scene releases them on every failure path below
    struct Raw {
        B200rtSphere *sph = nullptr;
        B200rtQuad *quad = nullptr;
        B200rtMaterial *mat = nullptr;
        uint32_t *order = nullptr;   // sphere_order[n_sph], then quad_order[n_quad]
        ~Raw() { dev_free(sph); dev_free(quad); dev_free(mat); dev_free(order); }
    } raw;
    CUDA_TRY(dev_alloc_async(&raw.sph, (size_t)n_sph * sizeof(B200rtSphere), 0));
    CUDA_TRY(dev_alloc_async(&raw.quad, (size_t)n_quad * sizeof(B200rtQuad), 0));
    // the scene's arrays are sized by the description alone: taken before the tree build's temporaries come and go,
    // they find the pool as the previous scene left it instead of fragmented by the build
    const size_t bytes[6] = {0, (size_t)n_sph * 2 * sizeof(double2), (size_t)n_sph * sizeof(uint2), (size_t)n_quad * 8 * sizeof(double2),
                             (size_t)n_quad * sizeof(uint2), (size_t)n_mat * sizeof(DeviceMaterial)};
    for (int i = 1; i < 6; ++i)
        if (bytes[i]) CUDA_TRY(scene_alloc(s, i, bytes[i]));
    CUDA_TRY(dev_alloc_async(&raw.mat, (size_t)n_mat * sizeof(B200rtMaterial), 0));
    CUDA_TRY(dev_alloc_async(&raw.order, ((size_t)n_sph + n_quad) * sizeof(uint32_t), 0));
    CUDA_TRY(staged_upload(raw.sph, desc->spheres, (size_t)n_sph * sizeof(B200rtSphere), 0));
    CUDA_TRY(staged_upload(raw.quad, desc->quads, (size_t)n_quad * sizeof(B200rtQuad), 0));
    CUDA_TRY(staged_upload(raw.mat, desc->materials, (size_t)n_mat * sizeof(B200rtMaterial), 0));
    uint32_t *sphere_order = raw.order, *quad_order = raw.order + n_sph;
    uint32_t n_nodes = 0, depth = 0, n_hoisted = 0, hoisted_ref[kMaxHoisted] = {};
    bool have_tree = false;
    if (gpu_build) {
        const bool trace = std::getenv("B200RT_TRACE") != nullptr;
        if (trace) cudaStreamSynchronize(0);
        const double t_up = now_ms();
        float4 *d_nodes = nullptr;
        const cudaError_t e = build_lbvh_device(raw.sph, n_sph, raw.quad, n_quad, max_hoisted(), sphere_order, quad_order, &d_nodes,
                                                &n_nodes, &depth, &n_hoisted, hoisted_ref);
        if (e != cudaSuccess) { cudaGetLastError(); return fail(B200RT_ECUDA, std::string("GPU BVH build: ") + cudaGetErrorString(e)); }
        if (trace) std::fprintf(stderr, "scene_build: upload %.2f ms, lbvh %.2f ms, depth %u\n", t_up - t0, now_ms() - t_up, depth);
        have_tree = n_nodes && 3 * depth <= 128;
        if (!have_tree) {
            dev_free(d_nodes);   // pathological depth, or too few primitives left for a radix tree: the host builder below takes over
        } else if (s->peer_visible) {
            // the builder sized the node array for the worst case (n - 1 nodes) in pool memory; a multi-device scene
            // keeps an exact-size copy in a peer-visible buffer instead (a device-to-device copy at HBM speed)
            const cudaError_t e2 = scene_alloc(s, 0, (size_t)n_nodes * sizeof(Node4));
            if (e2 == cudaSuccess) cudaMemcpyAsync(s->allocs[0], d_nodes, (size_t)n_nodes * sizeof(Node4), cudaMemcpyDeviceToDevice, 0);
            dev_free(d_nodes);
            if (e2 != cudaSuccess) { cudaGetLastError(); return fail(B200RT_ENOMEM, "node array copy"); }
        } else {
            s->allocs[0] = d_nodes;
            s->alloc_bytes[0] = (size_t)n_nodes * sizeof(Node4);
        }
    }
    double host_ms = -1;
    if (!have_tree) {   // parallel binned SAH + 4-wide collapse on the host; the nodes and the leaf order go up
        const double t1 = now_ms();
        std::vector<Box3> boxes;
        compute_boxes(desc, boxes, host_threads(opts));
        BuiltBVH bvh;
        const char *err = nullptr;
        if (!build_bvh4(boxes, desc->n_spheres, desc->n_quads, select_spanning(boxes, max_hoisted()), build_params(opts), bvh, &err))
            return fail(B200RT_EINVAL, std::string("BVH build failed: ") + (err ? err : "?"));
        host_ms = now_ms() - t1;
        n_hoisted = (uint32_t)bvh.hoisted_ref.size();
        std::copy(bvh.hoisted_ref.begin(), bvh.hoisted_ref.end(), hoisted_ref);
        n_nodes = (uint32_t)bvh.nodes.size();
        depth = bvh.depth;
        if (3 * depth > 128) return fail(B200RT_EINTERNAL, "BVH deeper than the largest traversal stack");
        CUDA_TRY(scene_alloc(s, 0, (size_t)n_nodes * sizeof(Node4)));
        CUDA_TRY(staged_upload(s->allocs[0], bvh.nodes.data(), (size_t)n_nodes * sizeof(Node4), 0));
        CUDA_TRY(staged_upload(sphere_order, bvh.sphere_order.data(), (size_t)n_sph * sizeof(uint32_t), 0));
        CUDA_TRY(staged_upload(quad_order, bvh.quad_order.data(), (size_t)n_quad * sizeof(uint32_t), 0));
    }
    int bad[2] = {0, 0};
    CUDA_TRY(assemble_scene_device(raw.sph, sphere_order, n_sph, raw.quad, quad_order, n_quad, raw.mat, n_mat,
                                   static_cast<double2 *>(s->allocs[1]), static_cast<uint2 *>(s->allocs[2]),
                                   static_cast<double2 *>(s->allocs[3]), static_cast<uint2 *>(s->allocs[4]),
                                   static_cast<DeviceMaterial *>(s->allocs[5]), bad));
    if (bad[1]) return fail(B200RT_EINVAL, "unknown material kind (closed set: Lambertian, Metal, Dielectric, DiffuseLight)");
    if (bad[0]) return fail(B200RT_EINVAL, "a sphere or quad has a material or primitive index out of range");
    B200rtSceneInfo info{};
    info.n_prims = (uint64_t)n_sph + n_quad;
    info.n_spheres = n_sph; info.n_quads = n_quad; info.n_materials = n_mat;
    info.n_nodes = n_nodes;
    info.tree_depth = depth;
    info.n_hoisted = n_hoisted;
    const double total = now_ms() - t0;
    info.build_ms = host_ms >= 0 ? host_ms : total;
    info.upload_ms = total - info.build_ms;
    return finish_scene(s, info, hoisted_ref);
}

// Builds the acceleration structure for `desc` (structure already validated) and makes the scene resident on device `dev`.
int create_scene_on(const B200rtSceneDesc *desc, const B200rtBuildOpts *opts, int dev, bool peer_visible, SceneImpl **out) {
    *out = nullptr;
    SceneImpl *s = new SceneImpl();
    s->device = dev;
    s->peer_visible = peer_visible;
    DeviceGuard g(dev);
    if (!g.ok) { delete s; return fail(B200RT_ECUDA, "cudaSetDevice failed"); }
    const uint64_t n_prims = desc->n_spheres + desc->n_quads;
    int builder = opts ? opts->builder : B200RT_BUILDER_AUTO;
    // AUTO: SAH on the host for small scenes (sub-millisecond, slightly better trees: +5 % on the
    // 4 k-sphere scene), Morton LBVH on the GPU from 64 k primitives up (2.2 M / 3.1 M primitives:
    // tens of ms incl. the upload vs 0.8 / 1.0 s, with equal or better render rates)
    if (builder == B200RT_BUILDER_AUTO) builder = n_prims >= 65536 ? B200RT_BUILDER_GPU_LBVH : B200RT_BUILDER_HOST_SAH;
    if (int rc = scene_build(desc, opts, builder == B200RT_BUILDER_GPU_LBVH && n_prims >= 2, s)) { free_scene(s); return rc; }
    *out = s;
    return B200RT_OK;
}

// A copy of the resident scene `src` on device `dev`: six device-to-device copies (NVLink between peers), no rebuild.
// The copies are enqueued on dev's default stream; the caller synchronises `dev` before the first render.
int replicate_scene_on(const SceneImpl *src, int dev, SceneImpl **out) {
    *out = nullptr;
    SceneImpl *s = new SceneImpl();
    s->device = dev;
    s->peer_visible = true;
    DeviceGuard g(dev);
    if (!g.ok) { delete s; return fail(B200RT_ECUDA, "cudaSetDevice failed"); }
    for (int i = 0; i < 6; ++i) {
        if (!src->allocs[i]) continue;
        cudaError_t e = scene_alloc(s, i, src->alloc_bytes[i]);
        if (e == cudaSuccess) e = cudaMemcpyPeerAsync(s->allocs[i], dev, src->allocs[i], src->device, src->alloc_bytes[i], 0);
        if (e != cudaSuccess) {
            cudaGetLastError();
            free_scene(s);
            return fail(e == cudaErrorMemoryAllocation ? B200RT_ENOMEM : B200RT_ECUDA, std::string("scene copy to a peer device: ") + cudaGetErrorString(e));
        }
    }
    if (int rc = finish_scene(s, src->info, src->d.hoisted_ref)) { free_scene(s); return rc; }
    *out = s;
    return B200RT_OK;
}

// One frame on all devices of `m` into the caller's host buffer(s): sample split, exchange, scale, read back.  With
// out_m2 every device's frame holds [image | second moment] and both planes go through the same per-float exchange.
int render_multi(MultiImpl *m, const B200rtCamera *cam, const B200rtRenderOpts *opts, float *out_rgb, float *out_m2,
                 B200rtStats *stats) {
    std::lock_guard<std::mutex> lk(m->mu);
    const double t0 = now_ms();
    CameraParams C{};
    if (int rc = fill_camera(cam, C)) return rc;
    B200rtRenderOpts o{};
    if (opts) o = *opts;
    uint64_t count = 0;
    if (int rc = sample_range_of(cam, o, &count)) return rc;
    const int n = (int)m->dev.size();
    const long long n_pixels = (long long)cam->image_w * cam->image_h;
    const size_t floats = (size_t)n_pixels * 3;               // one plane
    const int planes = out_m2 ? 2 : 1;
    const size_t all_floats = floats * planes;
    if (all_floats > m->frame_floats) {
        for (int d = 0; d < n; ++d) {
            DeviceGuard g(m->dev[d]->device);
            peer_buffer_release(m->dev[d]->device, m->frame[d]); m->frame[d] = nullptr;
            if (d == 0) { dev_free(m->scratch); m->scratch = nullptr; }
            m->frame_floats = 0;
            CUDA_TRY(peer_buffer_acquire(m->dev[d]->device, all_floats * sizeof(float), reinterpret_cast<void **>(&m->frame[d])));
            if (d == 0 && !m->peers) CUDA_TRY(dev_alloc(&m->scratch, all_floats * sizeof(float)));
        }
        m->frame_floats = all_floats;
    }
    std::vector<B200rtStats> st(n);
    for (int d = 0; d < n; ++d) {   // rank d of n: samples [count*d/n, count*(d+1)/n) of the requested range, as a SUM
        DeviceGuard g(m->dev[d]->device);
        B200rtRenderOpts od = o;
        const uint64_t lo = count * (uint64_t)d / (uint64_t)n, hi = count * (uint64_t)(d + 1) / (uint64_t)n;
        od.sample_offset = o.sample_offset + lo;
        od.sample_count = hi - lo;
        od.flags = (o.flags & (B200RT_FLAG_COUNTERS | B200RT_FLAG_THREAD_PIXELS)) | B200RT_FLAG_SUM | B200RT_FLAG_EXACT_COUNT;
        if (int rc = render_on_device(m->dev[d], cam, &od, m->frame[d], m->stream[d], &st[d], false, out_m2 ? m->frame[d] + floats : nullptr))
            return rc;
        CUDA_TRY(cudaEventRecord(m->ev_render[d], m->stream[d]));
    }
    const float scale = (o.flags & B200RT_FLAG_SUM) || count == 0 ? 1.0f : (float)(1.0 / (double)count);
    cudaEvent_t x0 = nullptr, x1 = nullptr;
    {
        DeviceGuard g(m->dev[0]->device);
        CUDA_TRY(cudaEventCreate(&x0));
        CUDA_TRY(cudaEventCreate(&x1));
    }
    struct EvGuard { cudaEvent_t &a, &b; ~EvGuard() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); } } evg{x0, x1};
    unsigned long long xchg_launches = 0;
    if (m->peers) {
        // one launch per device over peer-mapped frames: device d sums ITS slice of every frame in device order,
        // scales and writes the result into devices[0]'s frame (reduce-scatter + scale + gather in one pass)
        PeerFrames in{};
        for (int r = 0; r < n; ++r) in.p[r] = m->frame[r];
        for (int d = 0; d < n; ++d) {
            DeviceGuard g(m->dev[d]->device);
            for (int r = 0; r < n; ++r)
                if (r != d) CUDA_TRY(cudaStreamWaitEvent(m->stream[d], m->ev_render[r], 0));
            if (d == 0) CUDA_TRY(cudaEventRecord(x0, m->stream[0]));
            CUDA_TRY(launch_reduce_finalize_peers(in, n, d, n_pixels * planes, scale, m->frame[0], nullptr, 0, m->stream[d]));
            CUDA_TRY(cudaEventRecord(m->ev_xchg[d], m->stream[d]));
            ++xchg_launches;
        }
        DeviceGuard g(m->dev[0]->device);
        for (int d = 1; d < n; ++d) CUDA_TRY(cudaStreamWaitEvent(m->stream[0], m->ev_xchg[d], 0));
        CUDA_TRY(cudaEventRecord(x1, m->stream[0]));
    } else {
        // no peer mapping: copy each frame to devices[0] and add there, in device order (the same sums, bit for bit)
        DeviceGuard g(m->dev[0]->device);
        CUDA_TRY(cudaEventRecord(x0, m->stream[0]));
        for (int r = 1; r < n; ++r) {
            CUDA_TRY(cudaStreamWaitEvent(m->stream[0], m->ev_render[r], 0));
            CUDA_TRY(cudaMemcpyPeerAsync(m->scratch, m->dev[0]->device, m->frame[r], m->dev[r]->device, all_floats * sizeof(float), m->stream[0]));
            CUDA_TRY(launch_add_frame(m->frame[0], m->scratch, (long long)all_floats, m->stream[0]));
            ++xchg_launches;
        }
        CUDA_TRY(launch_finalize(m->frame[0], n_pixels * planes, scale, nullptr, 0, m->stream[0]));
        ++xchg_launches;
        CUDA_TRY(cudaEventRecord(x1, m->stream[0]));
    }
    double d2h_ms = 0;
    {
        DeviceGuard g(m->dev[0]->device);
        CUDA_TRY(cudaStreamSynchronize(m->stream[0]));
        const double t1 = now_ms();
        CUDA_TRY(staged_download(out_rgb, m->frame[0], floats * sizeof(float), m->stream[0]));
        if (out_m2) CUDA_TRY(staged_download(out_m2, m->frame[0] + floats, floats * sizeof(float), m->stream[0]));
        d2h_ms = now_ms() - t1;
    }
    B200rtStats total{};
    total.n_devices = (uint32_t)n;
    total.peer_exchange = m->peers ? 1u : 0u;
    for (int d = 0; d < n; ++d) {
        DeviceGuard g(m->dev[d]->device);
        CUDA_TRY(read_stats(m->dev[d], m->stream[d], &st[d]));   // synchronises: nobody reads this device's frame any more
        total.kernel_ms = std::max(total.kernel_ms, st[d].kernel_ms);
        total.paths += st[d].paths; total.rays += st[d].rays;
        total.node_visits += st[d].node_visits; total.prim_tests += st[d].prim_tests; total.quad_tests += st[d].quad_tests;
        total.kernel_launches += st[d].kernel_launches;
    }
    {
        DeviceGuard g(m->dev[0]->device);
        float ms = 0;
        if (cudaEventElapsedTime(&ms, x0, x1) == cudaSuccess) total.exchange_ms = ms; else cudaGetLastError();
    }
    total.kernel_launches += xchg_launches;
    total.d2h_ms = d2h_ms;
    total.d2h_bytes = all_floats * sizeof(float);
    total.replicate_ms = m->replicate_ms;
    total.total_ms = now_ms() - t0;
    if (stats) *stats = total;
    return B200RT_OK;
}

// b200rt_render and b200rt_render_moments: one frame into the caller's host buffer(s).  out_m2 may be NULL (image only);
// otherwise the scene's frame holds [image | second moment] and both planes are read back.
int render_host(void *scene, const B200rtCamera *cam, const B200rtRenderOpts *opts, float *out_rgb, float *out_m2, B200rtStats *stats) {
    if (MultiImpl *m = as_multi(scene)) return render_multi(m, cam, opts, out_rgb, out_m2, stats);
    SceneImpl *s = as_scene(scene);
    if (!s) return fail(B200RT_EINVAL, "bad scene handle");
    {
        CameraParams C{};
        if (int rc = fill_camera(cam, C)) return rc;   // range-checks the dimensions BEFORE anything is sized by them
    }
    std::lock_guard<std::mutex> lk(s->mu);
    DeviceGuard g(s->device);
    const double t0 = now_ms();
    const size_t floats = (size_t)cam->image_w * cam->image_h * 3;   // one plane
    const size_t all_floats = floats * (out_m2 ? 2 : 1);
    CUDA_TRY(grow_frame(s, all_floats));
    B200rtRenderOpts o{};
    if (opts) o = *opts;
    o.flags &= ~(uint32_t)B200RT_FLAG_ACCUMULATE;   // host entry always overwrites
    B200rtStats local{};
    if (int rc = render_on_device(s, cam, &o, s->d_frame, 0, &local, true, out_m2 ? s->d_frame + floats : nullptr)) return rc;
    const double t1 = now_ms();
    CUDA_TRY(staged_download(out_rgb, s->d_frame, floats * sizeof(float), 0));
    if (out_m2) CUDA_TRY(staged_download(out_m2, s->d_frame + floats, floats * sizeof(float), 0));
    const double t2 = now_ms();
    local.d2h_ms = t2 - t1;
    local.d2h_bytes = all_floats * sizeof(float);
    local.total_ms = t2 - t0;
    if (stats) *stats = local;
    return B200RT_OK;
}

// The scene's adaptive-sampling state for one image, carved out of s->d_adapt (grown on first use, like d_frame):
// per pixel 6 int64 sums and a count, per tile two 256-bit masks (active, unconverged) and two tile lists, and the
// two totals the host reads after each pass.
struct AdaptiveBuffers {
    long long *planes;
    uint32_t *counts, *mask, *unconv, *list_a, *list_b, *totals;
};
size_t adaptive_layout(char *base, size_t pixels, size_t tiles, AdaptiveBuffers *b) {
    size_t off = 0;
    auto take = [&](size_t bytes) { char *p = base ? base + off : nullptr; off += (bytes + 255) / 256 * 256; return p; };
    b->planes = reinterpret_cast<long long *>(take(pixels * kAdaptivePlanes * sizeof(long long)));
    b->counts = reinterpret_cast<uint32_t *>(take(pixels * sizeof(uint32_t)));
    b->mask = reinterpret_cast<uint32_t *>(take(tiles * kAdaptiveMaskWords * sizeof(uint32_t)));
    b->unconv = reinterpret_cast<uint32_t *>(take(tiles * kAdaptiveMaskWords * sizeof(uint32_t)));
    b->list_a = reinterpret_cast<uint32_t *>(take(tiles * sizeof(uint32_t)));
    b->list_b = reinterpret_cast<uint32_t *>(take(tiles * sizeof(uint32_t)));
    b->totals = reinterpret_cast<uint32_t *>(take(2 * sizeof(uint32_t)));
    return off;
}

// b200rt_render_adaptive on a single-device scene.  Pass 1 renders min(min_spp, max) samples of every pixel; each later
// pass renders the next min(step_spp, max - n) samples of the pixels still active, all of which have n samples.  Between
// passes two kernels judge the pass's pixels and dilate the result into the next active set and tile list; the host reads
// the next pass's tile and pixel counts, which size its grid or end the loop.
int render_adaptive_host(void *scene, const B200rtCamera *cam, const B200rtRenderOpts *opts, const B200rtAdaptiveOpts *aopts,
                         float *out_rgb, float *out_m2, uint32_t *out_spp, B200rtStats *stats) {
    if (as_multi(scene)) return fail(B200RT_EINVAL, "b200rt_render_adaptive takes a single-device scene");
    SceneImpl *s = as_scene(scene);
    if (!s) return fail(B200RT_EINVAL, "bad scene handle");
    if (!cam || !aopts || !out_rgb) return fail(B200RT_EINVAL, "camera, adaptive options or output pointer is NULL");
    RenderParams P{};
    B200rtRenderOpts o;
    bool leaf_first;
    if (int rc = render_setup(s, cam, opts, o, P, leaf_first)) return rc;
    if (int rc = require_default_kernel(o, "adaptive renders use")) return rc;
    P.flags &= ~(uint32_t)B200RT_FLAG_ACCUMULATE;   // host entry always overwrites
    const uint64_t max_spp = P.sample_count;
    const B200rtAdaptiveOpts a = *aopts;
    if (a.min_spp < 2 || a.step_spp == 0) return fail(B200RT_EINVAL, "adaptive options need min_spp >= 2 and step_spp >= 1");
    if (max_spp > kMaxSamplesPerLaunchMoments) return fail(B200RT_EINVAL, "an adaptive render takes at most 2^16 samples per pixel");
    if (!std::isfinite(a.rel_noise) || !std::isfinite(a.abs_noise) || a.rel_noise < 0 || a.abs_noise < 0)
        return fail(B200RT_EINVAL, "rel_noise and abs_noise must be finite and >= 0");
    std::lock_guard<std::mutex> lk(s->mu);
    DeviceGuard g(s->device);
    const double t0 = now_ms();
    const cudaStream_t st = 0;
    const size_t pixels = (size_t)cam->image_w * cam->image_h, floats = pixels * 3;
    const uint32_t tiles = path_tiles(P.cam.w, P.cam.h);
    CUDA_TRY(grow_frame(s, 2 * floats));
    AdaptiveBuffers b{};
    const size_t bytes = adaptive_layout(nullptr, pixels, tiles, &b);
    if (bytes > s->adapt_bytes) {
        if (s->d_adapt) { dev_free(s->d_adapt); s->d_adapt = nullptr; s->adapt_bytes = 0; }
        CUDA_TRY(dev_alloc(&s->d_adapt, bytes));
        s->adapt_bytes = bytes;
    }
    adaptive_layout(static_cast<char *>(s->d_adapt), pixels, tiles, &b);

    P.ad_mask = b.mask;
    P.ad_planes = b.planes;
    TailPlan tail;
    if (int rc = plan_tail(s, P.cam, PathMode::Adaptive, leaf_first, &tail)) return rc;
    tail.tiles = std::min(tail.tiles, tiles);

    AdaptiveState A{};
    A.w = P.cam.w; A.h = P.cam.h;
    A.list = b.list_a; A.next_list = b.list_b;
    A.mask = b.mask; A.unconv = b.unconv; A.planes = b.planes; A.counts = b.counts; A.totals = b.totals;
    A.rel_noise = a.rel_noise; A.abs_noise = a.abs_noise;

    CUDA_TRY(cudaMemsetAsync(s->d_counters, 0, 4 * sizeof(unsigned long long), st));
    CUDA_TRY(cudaEventRecord(s->ev0, st));
    if (tail.tiles) CUDA_TRY(tail_scratch(s, tail.tiles, true, st, &P));
    CUDA_TRY(cudaMemsetAsync(b.planes, 0, pixels * kAdaptivePlanes * sizeof(long long), st));
    CUDA_TRY(cudaMemsetAsync(b.counts, 0, pixels * sizeof(uint32_t), st));
    CUDA_TRY(launch_adaptive_init(A, tiles, st));
    unsigned long long launches = 1, paths = 0;
    uint64_t n = 0, active_pixels = pixels;
    uint32_t n_list = tiles;
    while (n < max_spp) {
        const uint64_t k = n == 0 ? std::min<uint64_t>(a.min_spp, max_spp) : std::min<uint64_t>(a.step_spp, max_spp - n);
        RenderParams Q = P;
        Q.sample_begin = (uint32_t)(o.sample_offset + n);
        Q.sample_count = (uint32_t)k;
        Q.ad_list = A.list;
        Q.ad_n_list = n_list;
        if (tail.tiles) chunk_tail(tail, n_list, Q);
        CUDA_TRY(launch_path_megakernel(s->stack, Q, PathMode::Adaptive, leaf_first, st));
        paths += active_pixels * k;
        n += k;
        A.n_list = n_list;
        CUDA_TRY(launch_adaptive_judge(A, (uint32_t)n, n < max_spp, s->d, st));
        launches += 2;
        if (n == max_spp) break;
        CUDA_TRY(cudaMemsetAsync(b.totals, 0, 2 * sizeof(uint32_t), st));
        CUDA_TRY(launch_adaptive_decide(A, s->d, st));
        ++launches;
        uint32_t next[2];
        CUDA_TRY(cudaMemcpyAsync(next, b.totals, sizeof next, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        if (next[0] == 0) break;
        std::swap(A.list, A.next_list);
        n_list = next[0];
        active_pixels = next[1];
    }
    CUDA_TRY(launch_adaptive_finish(A, (o.flags & B200RT_FLAG_SUM) != 0, s->d_frame, s->d_frame + floats, st));
    ++launches;
    if (tail.tiles) CUDA_TRY(cudaEventRecord(s->ev_tail, st));
    CUDA_TRY(cudaEventRecord(s->ev1, st));
    B200rtStats local{};
    CUDA_TRY(read_stats(s, st, &local));
    const double t1 = now_ms();
    CUDA_TRY(staged_download(out_rgb, s->d_frame, floats * sizeof(float), st));
    if (out_m2) CUDA_TRY(staged_download(out_m2, s->d_frame + floats, floats * sizeof(float), st));
    if (out_spp) CUDA_TRY(staged_download(out_spp, b.counts, pixels * sizeof(uint32_t), st));
    const double t2 = now_ms();
    if (stats) {
        local.paths = paths;
        local.kernel_launches = launches;
        local.n_devices = 1;
        local.d2h_ms = t2 - t1;
        local.d2h_bytes = (floats * ((out_m2 ? 2 : 1)) + (out_spp ? pixels : 0)) * sizeof(float);
        local.total_ms = t2 - t0;
        *stats = local;
    }
    return B200RT_OK;
}

}  // namespace

// ==========================================================================================
extern "C" {

int b200rt_version(void) { return B200RT_VERSION; }
const char *b200rt_last_error(void) { return g_last_error.c_str(); }
int b200rt_device_count(void) { return device_count_quiet(); }

int b200rt_camera_init(B200rtCamera *c) {
    if (!c) return fail(B200RT_EINVAL, "camera is NULL");
    if (c->image_w == 0 || c->image_h == 0) return fail(B200RT_EINVAL, "image dimensions must be positive");
    if ((c->vfov >= 0) == (c->hfov >= 0)) return fail(B200RT_EINVAL, "exactly one of vfov / hfov must be given");
    // camera.h:87-157, same operations in the same order, in double
    const double aspect = (double)c->image_w / (double)c->image_h;
    const V3 dir = v3(c->dir), center = v3(c->center);
    if (c->focus_dist < 0) c->focus_dist = mag(dir);
    const double focal = c->focus_dist;
    double vw, vh;
    if (c->vfov >= 0) { vh = 2 * focal * std::tan(c->vfov / 2); vw = vh * aspect; }
    else { vw = 2 * focal * std::tan(c->hfov / 2); vh = vw / aspect; }
    const V3 u = unitv(dir);
    const V3 bz = {-u.x, -u.y, -u.z};
    const V3 bx = unitv(crossv(v3(c->up), bz));
    const V3 by = crossv(bz, bx);
    const V3 x_vec = mul(bx, vw), y_vec = mul(by, -vh);
    const V3 dx = divv(x_vec, (double)c->image_w), dy = divv(y_vec, (double)c->image_h);
    const V3 ulc = sub(sub(sub(center, mul(bz, focal)), divv(x_vec, 2)), divv(y_vec, 2));
    const V3 p00 = add(add(ulc, divv(dx, 2)), divv(dy, 2));
    const double rad = focal * std::tan(c->defocus_angle / 2);
    put(c->delta_x, dx); put(c->delta_y, dy); put(c->pixel00, p00);
    put(c->disk_x, mul(bx, rad)); put(c->disk_y, mul(by, rad));
    return B200RT_OK;
}

int b200rt_trim(void) {
    if (device_count_quiet() == 0) return B200RT_OK;
    peer_buffer_trim();
    if (dev_pool_trim_all() != cudaSuccess) { cudaGetLastError(); return fail(B200RT_ECUDA, "cudaMemPoolTrimTo failed"); }
    return B200RT_OK;
}

int b200rt_scene_create(const B200rtSceneDesc *desc, const B200rtBuildOpts *opts, void **scene_out) {
    if (!scene_out) return fail(B200RT_EINVAL, "scene_out is NULL");
    *scene_out = nullptr;
    if (int rc = validate_desc(desc, false)) return rc;   // per-primitive checks: in create_scene_on, by whoever builds
    if (device_count_quiet() == 0) return fail(B200RT_ENODEVICE, "no CUDA device: libb200rt has no CPU path");
    int dev = opts ? opts->device : -1;
    if (dev < 0) { if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); dev = 0; } }
    if (dev >= device_count_quiet() || dev >= kMaxDevices) return fail(B200RT_EINVAL, "device ordinal out of range");
    SceneImpl *s = nullptr;
    if (int rc = create_scene_on(desc, opts, dev, false, &s)) return rc;
    *scene_out = s;
    return B200RT_OK;
}

int b200rt_scene_create_multi(const B200rtSceneDesc *desc, const B200rtBuildOpts *opts, const int32_t *devices, int32_t n_devices,
                              void **scene_out) {
    if (!scene_out) return fail(B200RT_EINVAL, "scene_out is NULL");
    *scene_out = nullptr;
    if (int rc = validate_desc(desc, false)) return rc;
    const int have = device_count_quiet();
    if (have == 0) return fail(B200RT_ENODEVICE, "no CUDA device: libb200rt has no CPU path");
    if (n_devices < 1 || n_devices > kMaxPeers) return fail(B200RT_EINVAL, "device count must be 1 .. 16");
    std::vector<int> devs(n_devices);
    for (int i = 0; i < n_devices; ++i) {
        devs[i] = devices ? devices[i] : i;
        if (devs[i] < 0 || devs[i] >= have || devs[i] >= kMaxDevices) return fail(B200RT_EINVAL, "device ordinal out of range");
    }
    if (n_devices == 1) {
        SceneImpl *s = nullptr;
        if (int rc = create_scene_on(desc, opts, devs[0], false, &s)) return rc;
        *scene_out = s;
        return B200RT_OK;
    }
    MultiImpl *m = new MultiImpl();
    m->dev.assign(n_devices, nullptr);
    m->stream.assign(n_devices, nullptr);
    m->ev_render.assign(n_devices, nullptr);
    m->ev_xchg.assign(n_devices, nullptr);
    m->frame.assign(n_devices, nullptr);
    const double t0 = now_ms();
    // Peer mapping: every device must be able to dereference every other device's pool memory for the fused
    // exchange; cudaMemcpyPeerAsync (the scene copies) works either way but goes over NVLink only between peers.
    bool all_peers = true;
    for (int i = 0; i < n_devices; ++i) {
        DeviceGuard g(devs[i]);
        for (int j = 0; j < n_devices; ++j) {
            if (devs[i] == devs[j]) continue;   // the same GPU listed again: nothing to map
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, devs[i], devs[j]) != cudaSuccess) { cudaGetLastError(); can = 0; }
            if (!can) { all_peers = false; continue; }
            const cudaError_t e = cudaDeviceEnablePeerAccess(devs[j], 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) all_peers = false;
            cudaGetLastError();
        }
    }
    // B200RT_MULTI_NO_PEER=1 forces the exchange without peer mapping (copies + accumulate on devices[0]); tests use it
    // to cover that path on NVLink boxes.  The frames peers dereference are cudaMalloc memory (devmem.h), which
    // cudaDeviceEnablePeerAccess maps; the pools' memory is only ever the source / target of peer COPIES.
    if (const char *np = std::getenv("B200RT_MULTI_NO_PEER")) if (np[0] == '1') all_peers = false;
    m->peers = all_peers;
    if (int rc = create_scene_on(desc, opts, devs[0], true, &m->dev[0])) { free_multi(m); return rc; }
    const double t_built = now_ms();
    for (int i = 1; i < n_devices; ++i)   // all copies are in flight together, one per destination device
        if (int rc = replicate_scene_on(m->dev[0], devs[i], &m->dev[i])) { free_multi(m); return rc; }
    for (int i = 0; i < n_devices; ++i) {
        DeviceGuard g(devs[i]);
        cudaError_t e = cudaStreamCreateWithFlags(&m->stream[i], cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&m->ev_render[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&m->ev_xchg[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaDeviceSynchronize();   // this device's copy of the scene has landed
        if (e != cudaSuccess) { cudaGetLastError(); free_multi(m); return fail(B200RT_ECUDA, std::string("multi-device setup: ") + cudaGetErrorString(e)); }
    }
    m->replicate_ms = now_ms() - t_built;
    if (std::getenv("B200RT_TRACE")) std::fprintf(stderr, "scene_create_multi: peer setup + build %.2f ms, replicate %.2f ms\n", t_built - t0, m->replicate_ms);
    *scene_out = m;
    return B200RT_OK;
}

int b200rt_scene_info(void *scene, B200rtSceneInfo *info) {
    SceneImpl *s = root_scene(scene);
    if (!s || !info) return fail(B200RT_EINVAL, "bad scene handle");
    *info = s->info;
    return B200RT_OK;
}

void b200rt_scene_destroy(void *scene) {
    if (MultiImpl *m = as_multi(scene)) free_multi(m);
    else free_scene(as_scene(scene));
}

int b200rt_debug_bounds(void *scene, uint64_t *out) {
#ifdef B200RT_DEBUG_BOUNDS
    if (!out) return fail(B200RT_EINVAL, "output pointer is NULL");
    for (int k = 0; k < 4; ++k) out[k] = 0;
    std::vector<SceneImpl *> all;
    if (MultiImpl *m = as_multi(scene)) all = m->dev;
    else if (SceneImpl *s = as_scene(scene)) all.push_back(s);
    else return fail(B200RT_EINVAL, "bad scene handle");
    for (SceneImpl *s : all) {
        DeviceGuard g(s->device);
        unsigned long long v[4];
        CUDA_TRY(cudaDeviceSynchronize());
        CUDA_TRY(cudaMemcpy(v, s->d_viol, sizeof v, cudaMemcpyDeviceToHost));
        for (int k = 0; k < 4; ++k) out[k] += v[k];
    }
    return B200RT_OK;
#else
    (void)scene; (void)out;
    return fail(B200RT_EINVAL, "this libb200rt was built without -DB200RT_DEBUG_BOUNDS");
#endif
}

int b200rt_debug_philox(const uint32_t *counters_keys, int64_t n, uint32_t *out, int device) {
    if (n < 0 || (n && (!counters_keys || !out))) return fail(B200RT_EINVAL, "bad debug_philox buffers");
    if (device_count_quiet() == 0) return fail(B200RT_ENODEVICE, "no CUDA device: libb200rt has no CPU path");
    if (n == 0) return B200RT_OK;
    if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) { cudaGetLastError(); device = 0; } }
    DeviceGuard g(device);
    uint32_t *d_in = nullptr, *d_out = nullptr;
    cudaError_t e = dev_alloc(&d_in, (size_t)n * 6 * sizeof(uint32_t));
    if (e == cudaSuccess) e = dev_alloc(&d_out, (size_t)n * 4 * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMemcpy(d_in, counters_keys, (size_t)n * 6 * sizeof(uint32_t), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = launch_debug_philox(d_in, n, d_out, 0);
    if (e == cudaSuccess) e = cudaMemcpy(out, d_out, (size_t)n * 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost);
    cudaStreamSynchronize(0);
    dev_free(d_in); dev_free(d_out);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(B200RT_ECUDA, std::string("debug_philox: ") + cudaGetErrorString(e)); }
    return B200RT_OK;
}

int b200rt_debug_samplers(const uint32_t *rnd_pairs, int64_t n, double *sphere_out, double *disk_out, int device) {
    if (n < 0 || (n && (!rnd_pairs || !sphere_out || !disk_out))) return fail(B200RT_EINVAL, "bad debug_samplers buffers");
    if (device_count_quiet() == 0) return fail(B200RT_ENODEVICE, "no CUDA device: libb200rt has no CPU path");
    if (n == 0) return B200RT_OK;
    if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) { cudaGetLastError(); device = 0; } }
    DeviceGuard g(device);
    uint32_t *d_in = nullptr;
    double *d_s = nullptr, *d_d = nullptr;
    cudaError_t e = dev_alloc(&d_in, (size_t)n * 2 * sizeof(uint32_t));
    if (e == cudaSuccess) e = dev_alloc(&d_s, (size_t)n * 3 * sizeof(double));
    if (e == cudaSuccess) e = dev_alloc(&d_d, (size_t)n * 2 * sizeof(double));
    if (e == cudaSuccess) e = cudaMemcpy(d_in, rnd_pairs, (size_t)n * 2 * sizeof(uint32_t), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = launch_debug_samplers(d_in, n, d_s, d_d, 0);
    if (e == cudaSuccess) e = cudaMemcpy(sphere_out, d_s, (size_t)n * 3 * sizeof(double), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(disk_out, d_d, (size_t)n * 2 * sizeof(double), cudaMemcpyDeviceToHost);
    cudaStreamSynchronize(0);
    dev_free(d_in); dev_free(d_s); dev_free(d_d);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(B200RT_ECUDA, std::string("debug_samplers: ") + cudaGetErrorString(e)); }
    return B200RT_OK;
}

int b200rt_raycast(void *scene, const double *rays, int64_t n, double tmin, double tmax, int32_t *prim_out, double *t_out) {
    SceneImpl *s = root_scene(scene);
    if (!s) return fail(B200RT_EINVAL, "bad scene handle");
    if (n < 0 || (n && (!rays || !prim_out || !t_out))) return fail(B200RT_EINVAL, "bad ray buffers");
    if (n == 0) return B200RT_OK;
    std::lock_guard<std::mutex> lk(s->mu);
    DeviceGuard g(s->device);
    if ((size_t)n > s->ray_capacity) {
        if (s->d_rays) { dev_free(s->d_rays); dev_free(s->d_prim); dev_free(s->d_t); s->d_rays = nullptr; s->d_prim = nullptr; s->d_t = nullptr; }
        s->ray_capacity = 0;
        CUDA_TRY(dev_alloc(&s->d_rays, (size_t)n * 6 * sizeof(double)));
        CUDA_TRY(dev_alloc(&s->d_prim, (size_t)n * sizeof(int32_t)));
        CUDA_TRY(dev_alloc(&s->d_t, (size_t)n * sizeof(double)));
        s->ray_capacity = (size_t)n;
    }
    CUDA_TRY(cudaMemcpy(s->d_rays, rays, (size_t)n * 6 * sizeof(double), cudaMemcpyHostToDevice));
    CUDA_TRY(launch_raycast(s->stack, s->d, s->d_rays, n, tmin, tmax, s->d_prim, s->d_t, 0));
    CUDA_TRY(cudaMemcpy(prim_out, s->d_prim, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(t_out, s->d_t, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost));
    return B200RT_OK;
}

int b200rt_debug_camera_rays(const B200rtCamera *cam, const uint32_t *pixels_xy, const uint32_t *rnd, int64_t n, double *rays_out,
                             int device) {
    CameraParams C{};
    if (int rc = fill_camera(cam, C)) return rc;
    if (n < 0 || (n && (!pixels_xy || !rnd || !rays_out))) return fail(B200RT_EINVAL, "bad debug_camera_rays buffers");
    if (device_count_quiet() == 0) return fail(B200RT_ENODEVICE, "no CUDA device: libb200rt has no CPU path");
    if (n == 0) return B200RT_OK;
    if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) { cudaGetLastError(); device = 0; } }
    DeviceGuard g(device);
    uint32_t *d_pix = nullptr, *d_rnd = nullptr;
    double *d_rays = nullptr;
    cudaError_t e = dev_alloc(&d_pix, (size_t)n * 2 * sizeof(uint32_t));
    if (e == cudaSuccess) e = dev_alloc(&d_rnd, (size_t)n * 4 * sizeof(uint32_t));
    if (e == cudaSuccess) e = dev_alloc(&d_rays, (size_t)n * 6 * sizeof(double));
    if (e == cudaSuccess) e = cudaMemcpy(d_pix, pixels_xy, (size_t)n * 2 * sizeof(uint32_t), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d_rnd, rnd, (size_t)n * 4 * sizeof(uint32_t), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = launch_debug_camera(C, d_pix, d_rnd, n, d_rays, 0);
    if (e == cudaSuccess) e = cudaMemcpy(rays_out, d_rays, (size_t)n * 6 * sizeof(double), cudaMemcpyDeviceToHost);
    cudaStreamSynchronize(0);
    dev_free(d_pix); dev_free(d_rnd); dev_free(d_rays);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(B200RT_ECUDA, std::string("debug_camera_rays: ") + cudaGetErrorString(e)); }
    return B200RT_OK;
}

int b200rt_debug_shade(void *scene, const double *rays, const uint32_t *rnd, int64_t n, double tmin, double tmax,
                       B200rtShadeRecord *records_out) {
    static_assert(sizeof(B200rtShadeRecord) == 88, "record layout is shared with kernels.cu");
    SceneImpl *s = root_scene(scene);
    if (!s) return fail(B200RT_EINVAL, "bad scene handle");
    if (n < 0 || (n && (!rays || !rnd || !records_out))) return fail(B200RT_EINVAL, "bad debug_shade buffers");
    if (n == 0) return B200RT_OK;
    std::lock_guard<std::mutex> lk(s->mu);
    DeviceGuard g(s->device);
    double *d_rays = nullptr;
    uint32_t *d_rnd = nullptr;
    void *d_rec = nullptr;
    cudaError_t e = dev_alloc(&d_rays, (size_t)n * 6 * sizeof(double));
    if (e == cudaSuccess) e = dev_alloc(&d_rnd, (size_t)n * 4 * sizeof(uint32_t));
    if (e == cudaSuccess) e = dev_alloc(&d_rec, (size_t)n * sizeof(B200rtShadeRecord));
    if (e == cudaSuccess) e = cudaMemcpy(d_rays, rays, (size_t)n * 6 * sizeof(double), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d_rnd, rnd, (size_t)n * 4 * sizeof(uint32_t), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = launch_debug_shade(s->stack, s->d, d_rays, d_rnd, n, tmin, tmax, d_rec, 0);
    if (e == cudaSuccess) e = cudaMemcpy(records_out, d_rec, (size_t)n * sizeof(B200rtShadeRecord), cudaMemcpyDeviceToHost);
    cudaStreamSynchronize(0);
    dev_free(d_rays); dev_free(d_rnd); dev_free(d_rec);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(B200RT_ECUDA, std::string("debug_shade: ") + cudaGetErrorString(e)); }
    return B200RT_OK;
}

int b200rt_debug_lane_accounting(void *scene, const B200rtCamera *cam, const B200rtRenderOpts *opts, uint64_t *counters_out) {
    SceneImpl *s = root_scene(scene);
    if (!s) return fail(B200RT_EINVAL, "bad scene handle");
    if (!cam || !counters_out) return fail(B200RT_EINVAL, "camera or output pointer is NULL");
    std::lock_guard<std::mutex> lk(s->mu);
    DeviceGuard g(s->device);
    RenderParams P{};
    B200rtRenderOpts o;
    bool leaf_first;
    if (int rc = render_setup(s, cam, opts, o, P, leaf_first)) return rc;
    float *d_frame = nullptr;
    unsigned long long *d_acc = nullptr;
    CUDA_TRY(dev_alloc(&d_frame, (size_t)cam->image_w * cam->image_h * 3 * sizeof(float)));
    cudaError_t e = dev_alloc(&d_acc, 16 * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemsetAsync(d_acc, 0, 16 * sizeof(unsigned long long), 0);
    if (e == cudaSuccess) e = cudaMemsetAsync(s->d_counters, 0, 4 * sizeof(unsigned long long), 0);
    P.out = d_frame; P.flags &= B200RT_FLAG_THREAD_PIXELS; P.scale = 1.0f;
    if (e == cudaSuccess) e = launch_path_lanes(s->stack, P, d_acc, leaf_first, 0);
    if (e == cudaSuccess) e = cudaMemcpy(counters_out, d_acc, 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
    cudaStreamSynchronize(0);
    dev_free(d_frame); dev_free(d_acc);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(B200RT_ECUDA, std::string("lane accounting: ") + cudaGetErrorString(e)); }
    return B200RT_OK;
}

#ifdef B200RT_BLOCK_TIMES
// Diagnostic build only (-DB200RT_BLOCK_TIMES, scripts/tail_profile.py): from now on every path_megakernel_pool launch on the
// current device writes {start ns, end ns, SM} of block b to device_buf[3 b .. 3 b + 2], for b < n_blocks.  NULL disarms.
int b200rt_debug_block_times(uint64_t *device_buf, uint64_t n_blocks) {
    if (cudaError_t e = set_block_times(reinterpret_cast<unsigned long long *>(device_buf), (uint32_t)std::min<uint64_t>(n_blocks, 0xFFFFFFFFu));
        e != cudaSuccess) {
        cudaGetLastError();
        return fail(B200RT_ECUDA, std::string("block times: ") + cudaGetErrorString(e));
    }
    return B200RT_OK;
}
#endif

int b200rt_render_device(void *scene, const B200rtCamera *cam, const B200rtRenderOpts *opts, float *out_rgb_device,
                         void *stream, B200rtStats *stats) {
    if (as_multi(scene)) return fail(B200RT_EINVAL, "b200rt_render_device takes a single-device scene (a multi-device scene renders through b200rt_render)");
    SceneImpl *s = as_scene(scene);
    if (!s) return fail(B200RT_EINVAL, "bad scene handle");
    if (!out_rgb_device) return fail(B200RT_EINVAL, "output pointer is NULL");
    std::lock_guard<std::mutex> lk(s->mu);
    DeviceGuard g(s->device);
    return render_on_device(s, cam, opts, out_rgb_device, static_cast<cudaStream_t>(stream), stats, stats != nullptr);
}

int b200rt_render(void *scene, const B200rtCamera *cam, const B200rtRenderOpts *opts, float *out_rgb, B200rtStats *stats) {
    if (!cam || !out_rgb) return fail(B200RT_EINVAL, "camera or output pointer is NULL");
    return render_host(scene, cam, opts, out_rgb, nullptr, stats);
}

int b200rt_render_moments(void *scene, const B200rtCamera *cam, const B200rtRenderOpts *opts, float *out_rgb, float *out_m2,
                          B200rtStats *stats) {
    if (!cam || !out_rgb || !out_m2) return fail(B200RT_EINVAL, "camera or output pointer is NULL");
    return render_host(scene, cam, opts, out_rgb, out_m2, stats);
}

int b200rt_render_adaptive(void *scene, const B200rtCamera *cam, const B200rtRenderOpts *opts, const B200rtAdaptiveOpts *aopts,
                           float *out_rgb, float *out_m2_or_null, uint32_t *out_spp_or_null, B200rtStats *stats) {
    return render_adaptive_host(scene, cam, opts, aopts, out_rgb, out_m2_or_null, out_spp_or_null, stats);
}

int b200rt_render_scene_multi(const B200rtSceneDesc *desc, const B200rtCamera *cam, const B200rtRenderOpts *opts,
                              const B200rtBuildOpts *bopts, const int32_t *devices, int32_t n_devices, float *out_rgb,
                              B200rtStats *stats, B200rtSceneInfo *info) {
    const double t0 = now_ms();
    if (!cam || !out_rgb) return fail(B200RT_EINVAL, "camera or output pointer is NULL");
    {
        CameraParams C{};
        if (int rc = fill_camera(cam, C)) return rc;   // reject a bad camera before paying for the build
    }
    void *scene = nullptr;
    if (int rc = b200rt_scene_create_multi(desc, bopts, devices, n_devices, &scene)) return rc;
    const double t1 = now_ms();
    B200rtStats local{};
    int rc = b200rt_render(scene, cam, opts, out_rgb, &local);
    const double t2 = now_ms();
    if (!rc) {
        const SceneImpl *s = root_scene(scene);
        local.h2d_ms = s->info.upload_ms;
        local.h2d_bytes = s->info.device_bytes;
        local.build_ms = s->info.build_ms + s->info.upload_ms;
        if (info) *info = s->info;
    }
    b200rt_scene_destroy(scene);
    local.total_ms = now_ms() - t0;
    if (std::getenv("B200RT_TRACE"))
        std::fprintf(stderr, "b200rt_render_scene_multi: create %.2f ms (build %.2f, replicate %.2f), render %.2f ms (kernel %.2f, exchange %.3f, d2h %.2f), destroy %.2f ms\n",
                     t1 - t0, local.build_ms, local.replicate_ms, t2 - t1, local.kernel_ms, local.exchange_ms, local.d2h_ms, now_ms() - t2);
    if (!rc && stats) *stats = local;
    return rc;
}

int b200rt_render_scene(const B200rtSceneDesc *desc, const B200rtCamera *cam, const B200rtRenderOpts *opts,
                        const B200rtBuildOpts *bopts, float *out_rgb, B200rtStats *stats, B200rtSceneInfo *info) {
    int32_t dev = bopts ? bopts->device : -1;
    if (dev < 0) { int cur = 0; if (cudaGetDevice(&cur) != cudaSuccess) { cudaGetLastError(); cur = 0; } dev = cur; }
    return b200rt_render_scene_multi(desc, cam, opts, bopts, &dev, 1, out_rgb, stats, info);
}

int b200rt_tonemap_device(const float *hdr_device, int64_t n_pixels, int32_t *out_device, int clamp, int device, void *stream) {
    if (n_pixels < 0 || (n_pixels && (!hdr_device || !out_device))) return fail(B200RT_EINVAL, "bad tonemap buffers");
    if (device_count_quiet() == 0) return fail(B200RT_ENODEVICE, "no CUDA device: libb200rt has no CPU path");
    if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) { cudaGetLastError(); device = 0; } }
    DeviceGuard g(device);
    CUDA_TRY(launch_tonemap(hdr_device, n_pixels, out_device, clamp, static_cast<cudaStream_t>(stream)));
    return B200RT_OK;
}

int b200rt_finalize_device(float *frame_device, int64_t n_pixels, double scale, int32_t *ldr_device_or_null, int clamp,
                           int device, void *stream) {
    if (n_pixels < 0 || (n_pixels && !frame_device)) return fail(B200RT_EINVAL, "bad frame buffer");
    if (device_count_quiet() == 0) return fail(B200RT_ENODEVICE, "no CUDA device: libb200rt has no CPU path");
    if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) { cudaGetLastError(); device = 0; } }
    DeviceGuard g(device);
    CUDA_TRY(launch_finalize(frame_device, n_pixels, (float)scale, ldr_device_or_null, clamp, static_cast<cudaStream_t>(stream)));
    return B200RT_OK;
}

int b200rt_finalize_peers_device(const float *const *peer_frames, int n_peers, int rank, int64_t n_pixels, double scale,
                                 float *root_hdr, int32_t *root_ldr_or_null, int clamp, int device, void *stream) {
    if (n_peers < 1 || n_peers > kMaxPeers || rank < 0 || rank >= n_peers) return fail(B200RT_EINVAL, "bad peer count / rank");
    if (n_pixels < 0 || !peer_frames || (n_pixels && !root_hdr)) return fail(B200RT_EINVAL, "bad frame buffers");
    PeerFrames in{};
    for (int r = 0; r < n_peers; ++r) {
        if (n_pixels && (!peer_frames[r] || (reinterpret_cast<uintptr_t>(peer_frames[r]) & 15)))
            return fail(B200RT_EINVAL, "peer frame pointers must be non-null and 16-byte aligned");
        in.p[r] = peer_frames[r];
    }
    if ((reinterpret_cast<uintptr_t>(root_hdr) & 15) || (reinterpret_cast<uintptr_t>(root_ldr_or_null) & 15))
        return fail(B200RT_EINVAL, "root buffers must be 16-byte aligned");
    if (device_count_quiet() == 0) return fail(B200RT_ENODEVICE, "no CUDA device: libb200rt has no CPU path");
    if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) { cudaGetLastError(); device = 0; } }
    DeviceGuard g(device);
    CUDA_TRY(launch_reduce_finalize_peers(in, n_peers, rank, n_pixels, (float)scale, root_hdr, root_ldr_or_null, clamp,
                                          static_cast<cudaStream_t>(stream)));
    return B200RT_OK;
}

int b200rt_tonemap(const float *hdr, int64_t n_pixels, int32_t *out, int clamp) {
    if (n_pixels < 0 || (n_pixels && (!hdr || !out))) return fail(B200RT_EINVAL, "bad tonemap buffers");
    if (device_count_quiet() == 0) return fail(B200RT_ENODEVICE, "no CUDA device: libb200rt has no CPU path");
    if (n_pixels == 0) return B200RT_OK;
    float *d_in = nullptr;
    int32_t *d_out = nullptr;
    CUDA_TRY(dev_alloc(&d_in, (size_t)n_pixels * 3 * sizeof(float)));
    cudaError_t e = dev_alloc(&d_out, (size_t)n_pixels * 3 * sizeof(int32_t));
    if (e == cudaSuccess) e = cudaMemcpy(d_in, hdr, (size_t)n_pixels * 3 * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = launch_tonemap(d_in, n_pixels, d_out, clamp, 0);
    if (e == cudaSuccess) e = cudaMemcpy(out, d_out, (size_t)n_pixels * 3 * sizeof(int32_t), cudaMemcpyDeviceToHost);
    cudaStreamSynchronize(0);
    dev_free(d_in);
    dev_free(d_out);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(B200RT_ECUDA, std::string("tonemap: ") + cudaGetErrorString(e)); }
    return B200RT_OK;
}

// ---- CPU-side self test of the host builder (no GPU needed; used by tests -m "not gpu") -------
// Builds the BVH for `desc`, with the scene-spanning primitives taken out as scene creation takes them out, and checks its
// structural invariants.  Fills depth / node count / hoisted count.
int b200rt_selftest_bvh(const B200rtSceneDesc *desc, const B200rtBuildOpts *opts, B200rtSceneInfo *info) {
    if (int rc = validate_desc(desc)) return rc;
    std::vector<Box3> boxes;
    compute_boxes(desc, boxes, host_threads(opts));
    BuiltBVH bvh;
    const char *err = nullptr;
    const double t0 = now_ms();
    if (!build_bvh4(boxes, desc->n_spheres, desc->n_quads, select_spanning(boxes, max_hoisted()), build_params(opts), bvh, &err))
        return fail(B200RT_EINVAL, std::string("BVH build failed: ") + (err ? err : "?"));
    const double t1 = now_ms();
    if (!validate_bvh4(bvh, boxes, desc->n_spheres, desc->n_quads, &err))
        return fail(B200RT_EINTERNAL, std::string("BVH invariant violated: ") + (err ? err : "?"));
    if (info) {
        std::memset(info, 0, sizeof *info);
        info->n_prims = desc->n_spheres + desc->n_quads;
        info->n_spheres = desc->n_spheres; info->n_quads = desc->n_quads; info->n_materials = desc->n_materials;
        info->n_nodes = bvh.nodes.size();
        info->tree_depth = bvh.depth;
        info->stack_entries = 3 * bvh.depth;
        info->build_ms = t1 - t0;
        info->n_hoisted = (uint32_t)bvh.hoisted_ref.size();
    }
    return B200RT_OK;
}

}  // extern "C"
