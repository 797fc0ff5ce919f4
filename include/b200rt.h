/* b200rt.h -- C ABI of the B200-native path tracer (libb200rt.so).
 *
 * This is the drop-in boundary for ONE path of DeltaPavonis/cpp_raytracer: the render call
 *     Image Camera::render(const Scene &world)                 (reference include/base/camera.h:301-303)
 *     template<T> auto Camera::render(const T &world)          (reference include/base/camera.h:264-297)
 * and the closest-hit query underneath it
 *     BVH::hit_by / Scene::hit_by                              (reference include/acceleration/bvh.h:585-715,
 *                                                               include/base/scene.h:59-75).
 * The reference has no FFI; a maintainer would bind these entry points from Camera::render
 * (see INTEGRATION.md for the stub).  Plain pointers and sizes only; no C++/torch types.
 *
 * Conventions: every function returns 0 on success and a negative B200RT_E* code on failure
 * (never exit()s, unlike the reference's std::exit(-1) in image.h:39-42); the message is
 * available from b200rt_last_error() on the calling thread.  The caller owns every host
 * buffer; the library owns device memory behind the opaque scene handle.  Calls block until
 * their result is in the caller's buffer unless stated otherwise.  A scene handle is NOT re-entrant:
 * calls on one handle are serialised inside the library (a mutex per handle); different handles
 * may be used from different host threads concurrently.  Device memory comes from a private
 * stream-ordered pool per device (the process-wide default pool is never touched); it keeps up to
 * B200RT_POOL_KEEP_MB (environment, default 4096) MiB of freed memory for the next frame and
 * b200rt_trim() returns it.  There is NO CPU fallback: without a CUDA device every compute entry
 * point fails with B200RT_ENODEVICE.
 */
#ifndef B200RT_H
#define B200RT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200RT_VERSION 2

enum {
    B200RT_OK = 0,
    B200RT_EINVAL = -1,      /* bad argument / malformed scene (unknown material kind, index out of range ...) */
    B200RT_ENODEVICE = -2,   /* no usable CUDA device: there is no CPU path */
    B200RT_ECUDA = -3,       /* CUDA runtime error; text in b200rt_last_error() */
    B200RT_ENOMEM = -4,
    B200RT_EINTERNAL = -5
};

/* Material kinds: the closed set of reference materials (include/base/material.h). */
enum {
    B200RT_MAT_LAMBERTIAN = 0,   /* rgb = intrinsic colour                (material.h:58-95)   */
    B200RT_MAT_METAL = 1,        /* rgb = colour, param = fuzz (<= 1)     (material.h:105-152) */
    B200RT_MAT_DIELECTRIC = 2,   /* param = refractive index              (material.h:164-227) */
    B200RT_MAT_LIGHT = 3         /* rgb = colour, param = intensity       (material.h:231-275) */
};

/* Flat scene description.  `prim` is the canonical primitive index: the position of the
 * primitive in Scene::get_primitive_components() order (scene.h:85-105; a Box contributes its
 * six faces in constructor order, box.h:53-84).  b200rt_raycast reports hits by this index. */
#pragma pack(push, 1)
typedef struct B200rtMaterial { uint32_t kind, pad; double rgb[3]; double param; } B200rtMaterial;      /* 40 B */
typedef struct B200rtSphere { double c[3]; double r; uint32_t mat, prim; } B200rtSphere;                /* 40 B, sphere.h:16-22 */
typedef struct B200rtQuad { double v[3], s1[3], s2[3]; uint32_t mat, prim; } B200rtQuad;                /* 80 B, parallelogram.h:14-48 */

/* Camera.  The first block is what the reference's fluent setters store (camera.h:308-406);
 * the second block is what Camera::init() derives from it (camera.h:87-157).
 * b200rt_camera_init() fills the second block from the first, in double precision on the
 * host, operation for operation as the reference does.  Angles are radians; vfov/hfov < 0
 * means "not given" (exactly one of them must be given). */
typedef struct B200rtCamera {
    uint64_t image_w, image_h, spp, max_depth;
    double center[3], dir[3], up[3];
    double focus_dist;            /* < 0: default to |dir| (camera.h:101-103) */
    double defocus_angle;         /* radians; <= 0 turns blur off (camera.h:186) */
    double vfov, hfov;
    double background[3];
    /* derived */
    double pixel00[3], delta_x[3], delta_y[3], disk_x[3], disk_y[3];
} B200rtCamera;
#pragma pack(pop)

typedef struct B200rtSceneDesc {
    uint64_t n_materials, n_spheres, n_quads;
    const B200rtMaterial *materials;
    const B200rtSphere *spheres;
    const B200rtQuad *quads;
} B200rtSceneDesc;

/* Acceleration-structure build knobs (all optional; pass NULL for defaults).  The reference's
 * knobs are BVH(world, num_buckets = 32, max_primitives_in_node = 12) (bvh.h:754-756); the
 * tree here is a different design (4-wide, FP32 conservative boxes), results are tree
 * independent. */
typedef struct B200rtBuildOpts {
    int32_t device;          /* CUDA device ordinal; -1 = current device */
    int32_t max_leaf_prims;  /* 1..8, 0 = default */
    int32_t sah_bins;        /* 4..64, 0 = default */
    int32_t build_threads;   /* host threads for the builder, 0 = all */
    int32_t builder;         /* B200RT_BUILDER_* */
} B200rtBuildOpts;

enum {
    B200RT_BUILDER_AUTO = 0,       /* HOST_SAH below 65536 primitives, GPU_LBVH from there up */
    B200RT_BUILDER_HOST_SAH = 1,   /* parallel binned SAH on the host: best trees, ~0.3 us per primitive */
    B200RT_BUILDER_GPU_LBVH = 2    /* Morton-order LBVH built on the GPU: tens of ms for millions of primitives,
                                      somewhat more node visits per ray; falls back to HOST_SAH if too deep */
};

typedef struct B200rtSceneInfo {
    uint64_t n_prims, n_spheres, n_quads, n_materials;
    uint64_t n_nodes;             /* 4-wide nodes, 128 B each */
    uint64_t device_bytes;        /* total device footprint of the scene */
    uint32_t tree_depth;          /* depth of the 4-wide tree */
    uint32_t stack_entries;       /* traversal stack entries the kernels are instantiated with */
    double build_ms, upload_ms;
    uint32_t n_hoisted;           /* scene-spanning primitives tested by every ray before the tree instead of in it */
} B200rtSceneInfo;

enum {
    B200RT_VARIANT_MEGAKERNEL = 0,          /* one launch for the whole frame, path regeneration (default) */
    B200RT_VARIANT_WAVEFRONT = 1            /* per-material ray queues */
    /* 2 was an experiment (warp-voted step scheduling, measured slower: DESIGN.md section 7); it is no longer
     * part of the library and is rejected with B200RT_EINVAL */
};
enum {
    B200RT_FLAG_SUM = 1,          /* write the per-pixel SUM over the samples of this call instead of the mean */
    B200RT_FLAG_ACCUMULATE = 2,   /* device entry only: add into the output buffer instead of overwriting */
    B200RT_FLAG_COUNTERS = 4,     /* also count node visits and primitive tests (slower; for roofline accounting) */
    B200RT_FLAG_THREAD_PIXELS = 16, /* A/B switch: the round-1 work distribution (a thread owns a pixel and renders all its
                                     samples) instead of the tile work pool (threads take (pixel, sample) items of their
                                     8 x 32 tile as their paths end).  Same paths, same image up to summation order. */
    B200RT_FLAG_EXACT_COUNT = 8   /* sample_count is taken literally: 0 renders NO samples (the output is zeroed /
                                     left alone under ACCUMULATE) instead of meaning "camera.spp" -- what a rank of a
                                     sample split whose share is empty (spp < ranks) must pass */
};

typedef struct B200rtRenderOpts {
    uint64_t seed;             /* RNG key; streams are a pure function of (seed, pixel, sample, bounce) */
    uint64_t sample_offset;    /* first sample index of this call (sample split across GPUs) */
    uint64_t sample_count;     /* samples per pixel rendered by this call; 0 = camera.spp */
    int32_t variant;           /* B200RT_VARIANT_* */
    uint32_t flags;            /* B200RT_FLAG_* */
} B200rtRenderOpts;

typedef struct B200rtStats {
    double kernel_ms;          /* CUDA-event time of the path kernel(s) on their stream */
    double h2d_ms, d2h_ms, total_ms;
    uint64_t paths, rays;      /* pixel-samples and hit_by-equivalent ray casts */
    uint64_t node_visits, prim_tests;   /* only with B200RT_FLAG_COUNTERS */
    uint64_t kernel_launches;
    uint64_t h2d_bytes, d2h_bytes;
    /* v2 */
    double build_ms;           /* acceleration-structure build incl. the upload of the caller's arrays (one-call entries) */
    double replicate_ms;       /* multi-GPU: copying the built scene to the other devices (peer copies, NVLink) */
    double exchange_ms;        /* multi-GPU: summing the per-device frames onto the first device + scaling */
    uint32_t n_devices;        /* devices that rendered */
    uint32_t peer_exchange;    /* 1: fused peer-memory kernel (one launch per device); 0: copies + accumulate on the root */
    uint64_t quad_tests;       /* with B200RT_FLAG_COUNTERS: how many of prim_tests were parallelogram tests (the rest: spheres) */
} B200rtStats;

/* ---- lifetime ------------------------------------------------------------------------- */
int b200rt_device_count(void);
const char *b200rt_last_error(void);
int b200rt_version(void);
/* Returns the freed device memory the library's private pools are holding to the driver (all devices). */
int b200rt_trim(void);

/* Replaces: BVH::BVH(world) + the pointer graph it keeps (bvh.h:754-776).  Flattens the
 * primitives into SoA device arrays, builds the wide BVH and uploads everything. */
int b200rt_scene_create(const B200rtSceneDesc *desc, const B200rtBuildOpts *opts, void **scene_out);
int b200rt_scene_info(void *scene, B200rtSceneInfo *info);
void b200rt_scene_destroy(void *scene);

/* The same scene made resident on SEVERAL GPUs of this process (SURVEY 8(b) "device list / nGPU", 8(e)): the
 * acceleration structure is built ONCE on devices[0] and copied to the others device-to-device
 * (cudaMemcpyPeerAsync: NVLink where the GPUs are peers).  The handle is accepted by b200rt_render
 * (every device renders its share of the samples of every pixel, rank k of n takes samples
 * [k*spp/n, (k+1)*spp/n) of the requested range; the per-device FP32 sum frames are added in device-list order
 * onto devices[0] -- one fused kernel per device over peer-mapped memory when all pairs are peers, else
 * copies + accumulate on devices[0] -- and scaled there; the image equals the single-GPU image up to FP32
 * summation order), b200rt_scene_info, b200rt_raycast / b200rt_debug_shade (answered by devices[0]) and
 * b200rt_scene_destroy.  n_devices == 1 is the same as b200rt_scene_create on that device;
 * devices == NULL means devices 0 .. n_devices-1.  A device may be listed more than once: every entry gets its own
 * copy of the scene, its own stream and its own share of the samples (this is how the test-suite drives the whole
 * multi-device path -- copies, sample split, fused exchange -- on a one-GPU machine).  No torch, no NCCL, one host thread.  Side effect on the
 * process: cudaDeviceEnablePeerAccess is turned on between the listed devices (and left on); the scene arrays and
 * frames of a multi-device scene are plain cudaMalloc buffers cached per device until b200rt_trim().
 * Replaces: nothing in the reference (it has one CPU); this is how `Camera::render` reaches config 5,
 * "sample-split across 8 x B200". */
int b200rt_scene_create_multi(const B200rtSceneDesc *desc, const B200rtBuildOpts *opts, const int32_t *devices,
                              int32_t n_devices, void **scene_out);

/* Replaces: Camera::init() (camera.h:87-157).  Host, double precision. */
int b200rt_camera_init(B200rtCamera *cam);

/* ---- closest hit (deterministic ray-cast harness) -------------------------------------- */
/* Replaces: world.hit_by(ray, Interval(tmin, tmax)) for n rays (bvh.h:585-715 /
 * scene.h:59-75).  rays = n x {ox,oy,oz,dx,dy,dz} doubles (directions NOT normalised, as in
 * the reference).  prim_out[i] = canonical primitive index of the closest hit with
 * tmin < t < tmax, or -1; t_out[i] = its hit time (0 on miss).  Exact ties in t resolve to the
 * lowest canonical index, which is what Scene::hit_by returns. */
int b200rt_raycast(void *scene, const double *rays, int64_t n, double tmin, double tmax,
                   int32_t *prim_out, double *t_out);

/* Test hook: ONE surface interaction per ray, performed by the same device function the path kernels
 * call -- closest hit (as b200rt_raycast), hit point, the hit_info face rule (hittable.h:46-71), then
 * Lambertian / Metal / Dielectric / DiffuseLight scatter + emit (material.h:64-263, vec3d.h:144-200) on a
 * unit throughput -- but with the caller's four 32-bit random words per ray in place of the kernel's
 * Philox stream, so each branch can be checked deterministically.  Word use: Lambertian and Metal
 * sample the unit sphere from words 0,1 (u = (w >> 8) / 2^24; z = 1 - 2 u0, azimuth 2 pi u1); Dielectric
 * compares u(word 2) with the Schlick reflectance (no word is used under total internal reflection). */
typedef struct B200rtShadeRecord {
    double scattered[6];   /* origin (= hit point) and unnormalised direction of the scattered ray; zeros if none */
    double t;              /* hit time */
    float atten[3];        /* attenuation applied (1,1,1 for Dielectric); zeros if the path ended */
    float emit[3];         /* emitted radiance (DiffuseLight: intensity * colour, both faces) */
    int32_t prim;          /* canonical primitive index, -1 = miss */
    int32_t flags;         /* bit 0: scattered ray present */
} B200rtShadeRecord;
int b200rt_debug_shade(void *scene, const double *rays, const uint32_t *rnd, int64_t n, double tmin, double tmax,
                       B200rtShadeRecord *records_out);

/* Test hook: the kernels' primary-ray construction (Camera::random_ray_through_pixel, camera.h:184-200, defocus
 * disk camera.h:160-168) for n pixels (pixels_xy = n x {col, row}) with the caller's four random words per ray
 * (u = (w >> 8) / 2^24): words 0,1 -> the U(-0.5,0.5) factors of delta_x, delta_y; words 2,3 -> the point in the
 * unit disk (radius sqrt(u2), azimuth 2 pi u3), used only when defocus_angle > 0.  rays_out = n x 6 doubles. */
int b200rt_debug_camera_rays(const B200rtCamera *cam, const uint32_t *pixels_xy, const uint32_t *rnd, int64_t n,
                             double *rays_out, int device);

/* Test hooks for the two pieces no oracle can pin through images.  b200rt_debug_philox: the kernels' generator
 * (Philox4x32-10, csrc/rng.cuh) evaluated ON THE DEVICE for n (counter[4], key[2]) inputs -> out = n x 4 words;
 * checked against the Random123 known-answer vectors.  b200rt_debug_samplers: the kernels' direction samplers for n
 * pairs of random words (u = (w >> 8) / 2^24): sphere_out = n x 3 doubles, the unit vector Lambertian / Metal add
 * (stands in for random_unit_vector(), vec3d.h:64-75); disk_out = n x 2 doubles, the defocus-disk point (stands in
 * for random_vector_in_unit_disk(), vec3d.h:79-85). */
int b200rt_debug_philox(const uint32_t *counters_keys, int64_t n, uint32_t *out, int device);
int b200rt_debug_samplers(const uint32_t *rnd_pairs, int64_t n, double *sphere_out, double *disk_out, int device);

/* Bounds-checked build (-DB200RT_DEBUG_BOUNDS; the stand-in for compute-sanitizer, which the GPU pool does not
 * allow): every traversal-stack push, node / primitive / material index and frame store is range-checked on the
 * device; a violation is counted and the access skipped.  out[4] = {stack pushes beyond capacity, node index,
 * primitive or material index, pixel index} violations since the scene was created.  Returns B200RT_EINVAL in a
 * library built without the flag.  B200RT_DEBUG_STACK_CAP (environment, debug build only) lowers the stack
 * capacity the check enforces, to prove the check is live. */
int b200rt_debug_bounds(void *scene, uint64_t *out);

/* Measurement hook: renders `cam` like b200rt_render's default kernel (same schedule: every round each lane of a warp
 * shades / regenerates, then the warp runs one traversal step per lane per iteration until its slowest lane is done)
 * with per-warp accounting of where the 32 lanes are at every executed step.  counters_out[16]:
 *   [0] shade executions, [1] lanes taking part;
 *   [2] node-step executions, [3] lanes at a node, idle lanes: [4] at a leaf, [5] traversal done (waiting for the
 *       slowest lane of the round), [6] pixel out of samples;
 *   [7] leaf-step executions, [8] lanes at a leaf, idle lanes: [9] at a node, [10] done, [11] out of samples;
 *   [12] primitive-test executions, [13] lanes taking part; [14] warps; [15] rays.  No image is returned. */
int b200rt_debug_lane_accounting(void *scene, const B200rtCamera *cam, const B200rtRenderOpts *opts, uint64_t *counters_out);

/* ---- render ---------------------------------------------------------------------------- */
/* Replaces: Camera::render<BVH>(bvh) (camera.h:264-297): for every pixel, the mean (or sum)
 * over the requested samples of ray_color (camera.h:205-258).  out_rgb = image_h x image_w x 3
 * floats, row-major, row 0 at the top, linear HDR (what the reference stores in Image before
 * RGB::as_string tone-maps it).  The image is a pure function of (scene, camera, seed, sample range): per-pixel sums are
 * accumulated in 64-bit fixed point (2^-30 units), so they do not depend on how the GPU distributes the samples over its
 * threads; the sum of one pixel's radiance over one launch (at most 2^22 samples) must stay below 8.6e9. */
int b200rt_render(void *scene, const B200rtCamera *cam, const B200rtRenderOpts *opts,
                  float *out_rgb, B200rtStats *stats);

/* Same, but out_rgb_device is a DEVICE pointer on the scene's device and `stream` a
 * cudaStream_t (NULL = the legacy default stream).  Returns after enqueueing when stats is
 * NULL; with stats it synchronises the stream to read the counters back. */
int b200rt_render_device(void *scene, const B200rtCamera *cam, const B200rtRenderOpts *opts,
                         float *out_rgb_device, void *stream, B200rtStats *stats);

/* b200rt_render plus, for every pixel and channel, the second moment of the sample radiance:
 * out_m2 (image_h x image_w x 3 floats, same layout as out_rgb) = mean over the requested samples of x^2
 * (the SUM of x^2 with B200RT_FLAG_SUM).  out_rgb is the same bits b200rt_render returns for the same
 * arguments (up to FP32 summation order above 2^16 samples per pixel, where both planes are summed
 * over several launches).  SUM frames of both planes add across sample ranges and devices, so the
 * sample variance of a pixel is n/(n-1) * (m2 - mean^2).  Single- and multi-device scenes.
 * The per-pixel sums of x^2 are accumulated in 64-bit fixed point (2^-24 units) over at most 2^16 samples per
 * launch, so they are as independent of the GPU's work distribution as the image; one launch's sum of x^2 of one
 * pixel must stay below 5.5e11 (a mean x^2 of 8.4e6 per sample, x up to about 2900).
 * B200RT_EINVAL with the wavefront variant, B200RT_FLAG_THREAD_PIXELS or B200RT_FLAG_COUNTERS. */
int b200rt_render_moments(void *scene, const B200rtCamera *cam, const B200rtRenderOpts *opts,
                          float *out_rgb, float *out_m2, B200rtStats *stats);

/* Adaptive sampling: every pixel gets samples until IT reaches a noise target.  Pixel p renders samples
 * [offset, offset + n_p) of its own stream, and its out_rgb / out_m2 values are the same bits b200rt_render_moments
 * returns for a uniform render of n_p samples with the same seed and offset; out_spp_or_null[p] = n_p.  The maximum
 * n_p is the sample count of `opts` (resolved as for b200rt_render), at most 2^16.
 *   Passes: the first renders min(min_spp, max) samples of every pixel; each later one renders the next
 * min(step_spp, max - n) samples of every pixel still active, all of which have the same count n.  After a pass,
 * pixel p at count n is CONVERGED when err <= rel_noise * level + abs_noise, evaluated in double without FMA:
 *   mean_c = (float)(S_c * 2^-30) * (float)(1.0 / n),  m2_c = (float)(Q_c * 2^-24) * (float)(1.0 / n)
 *     (the mean-plane floats, from the pixel's fixed-point sums S of x and Q of x^2);
 *   var_c = 0 if d = m2_c - mean_c^2 <= ldexp(m2_c, -20) + 2^-24, else n / (n - 1) * d;
 *   err = sqrt((var_r + var_g + var_b) / (3 n)),  level = (mean_r + mean_g + mean_b) / 3.
 * A pixel stays active while any pixel of its 3 x 3 neighbourhood (clipped at the image edge) is not converged, so a
 * pixel that has not yet seen a light its neighbours see keeps sampling; a pixel that stops never resumes.  With
 * rel_noise = abs_noise = 0 only pixels whose whole neighbourhood has exactly zero variance stop early.
 *   B200RT_FLAG_SUM: both planes are sums.  B200RT_FLAG_ACCUMULATE is ignored.  B200RT_EINVAL with the wavefront
 * variant, B200RT_FLAG_THREAD_PIXELS, B200RT_FLAG_COUNTERS, a multi-device handle, min_spp < 2, step_spp == 0, more
 * than 2^16 samples, or a negative or non-finite rel_noise / abs_noise.  stats->paths is the sum of n_p.  The scene keeps
 * about 52 bytes per pixel of device state for it (int64 sums, counts, masks), grown on first use. */
typedef struct B200rtAdaptiveOpts {
    uint32_t min_spp;     /* samples every pixel gets in the first pass; >= 2 */
    uint32_t step_spp;    /* samples added to each still-active pixel per later pass; >= 1 */
    double rel_noise;     /* converged: err <= rel_noise * level + abs_noise */
    double abs_noise;
} B200rtAdaptiveOpts;
int b200rt_render_adaptive(void *scene, const B200rtCamera *cam, const B200rtRenderOpts *opts,
                           const B200rtAdaptiveOpts *aopts, float *out_rgb, float *out_m2_or_null,
                           uint32_t *out_spp_or_null, B200rtStats *stats);

/* Replaces: Camera::render(const Scene &) end to end (camera.h:301-303): build + upload +
 * render + read back + free, all inside one call on host buffers. */
int b200rt_render_scene(const B200rtSceneDesc *desc, const B200rtCamera *cam,
                        const B200rtRenderOpts *opts, const B200rtBuildOpts *bopts,
                        float *out_rgb, B200rtStats *stats, B200rtSceneInfo *info);

/* Camera::render(const Scene &) end to end on several GPUs: b200rt_scene_create_multi + b200rt_render +
 * destroy in one call on host buffers. */
int b200rt_render_scene_multi(const B200rtSceneDesc *desc, const B200rtCamera *cam, const B200rtRenderOpts *opts,
                              const B200rtBuildOpts *bopts, const int32_t *devices, int32_t n_devices,
                              float *out_rgb, B200rtStats *stats, B200rtSceneInfo *info);

/* ---- tone map --------------------------------------------------------------------------- */
/* Replaces: RGB::as_string() defaults (rgb.h:90-113): Reinhard by luminance, gamma 2,
 * int(255.999999 * v), NO clamp unless clamp != 0 (the reference does not clamp, so a
 * saturated channel can exceed 255).  hdr = n_pixels x 3 floats; out = n_pixels x 3 int32. */
int b200rt_tonemap(const float *hdr, int64_t n_pixels, int32_t *out, int clamp);
int b200rt_tonemap_device(const float *hdr_device, int64_t n_pixels, int32_t *out_device,
                          int clamp, int device, void *stream);

/* Frame epilogue for the multi-GPU sample split, on the rank that holds the reduced SUM frame:
 * frame *= scale in place (pixel_color /= samples_per_pixel, camera.h:290) and, when
 * ldr_device_or_null is given, the tone-mapped integers of the same pixels in the same pass. */
int b200rt_finalize_device(float *frame_device, int64_t n_pixels, double scale, int32_t *ldr_device_or_null,
                           int clamp, int device, void *stream);

/* The same epilogue with the exchange fused in, over peer-mapped memory (NVLink / NVSwitch), in place
 * of "reduce to rank 0, then b200rt_finalize_device": one launch per rank, each rank owning one slice
 * of the frame.  peer_frames[r] is rank r's n_pixels x 3 FP32 SUM buffer as addressable FROM THIS
 * device (CUDA peer / symmetric-memory mapping; peer_frames[rank] is the local one); the kernel adds
 * the n_peers buffers in rank order over its slice, scales, and writes the mean frame into root_hdr
 * and (when given) the tone-mapped integers into root_ldr_or_null -- both pointers into the ROOT
 * rank's memory as addressable from this device.  root_hdr may be peer_frames[0] itself (in place).
 * All pointers must be 16-byte aligned.  The caller orders it: every rank's render must be complete
 * and visible before any rank launches this (a device barrier across ranks), and a second barrier
 * must pass before the root reads the result or any rank reuses its sum buffer.  Slices:
 * chunk = ceil(n_pixels / n_peers) rounded up to 1024 pixels; rank k owns
 * [min(n, k*chunk), min(n, (k+1)*chunk)).  1 <= n_peers <= 16.
 * Replaces: the serial accumulation of camera.h:286-290 across GPUs (no reference counterpart for
 * the exchange itself). */
int b200rt_finalize_peers_device(const float *const *peer_frames, int n_peers, int rank, int64_t n_pixels,
                                 double scale, float *root_hdr, int32_t *root_ldr_or_null, int clamp,
                                 int device, void *stream);

/* ---- host-only self test ---------------------------------------------------------------------- */
/* Builds the acceleration structure for `desc` on the host and checks its invariants (every
 * primitive in exactly one leaf, boxes nested, reported depth exact).  Needs no GPU; fills
 * n_nodes / tree_depth / stack_entries / build_ms of `info`. */
int b200rt_selftest_bvh(const B200rtSceneDesc *desc, const B200rtBuildOpts *opts, B200rtSceneInfo *info);

#ifdef __cplusplus
}
#endif
#endif /* B200RT_H */
