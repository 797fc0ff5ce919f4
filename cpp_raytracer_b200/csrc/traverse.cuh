// traverse.cuh -- device scene layout + closest-hit traversal shared by every kernel.
//
// Stands in for BVH::hit_by (reference include/acceleration/bvh.h:585-715),
// AABB::is_hit_by_optimized (aabb.h:132-174), Sphere::hit_by (sphere.h:45-96) and
// Parallelogram::hit_by (parallelogram.h:177-240).
//
// Precision design (DESIGN.md "Precision"):
//  * Box tests run in FP32 on bounds rounded outward: one FMA per plane against o/d products
//    formed in double and rounded outward, plus a multiplicative slack on the final comparison,
//    so a box test can only err towards "hit".  They never decide the answer, only prune.
//  * Primitive tests run in FP64, operation for operation as the reference writes them, and this
//    translation unit is compiled with -fmad=false (the reference is built for baseline x86-64,
//    no FMA contraction), so for the same ray the hit time is bit-identical to the reference's.
//  * Exact ties in t resolve to the lowest canonical primitive index (what Scene::hit_by,
//    scene.h:59-75, returns), independent of the tree.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace b200rt {

struct DeviceMaterial {   // 32 B, two 16-byte loads
    float r, g, b;        // colour; for lights: intensity * colour (material.h:261-263)
    uint32_t kind;
    double param;         // fuzz | refractive index | intensity
    double pad;
};

// -DB200RT_DEBUG_BOUNDS: the bounds-checked build the GPU test-suite runs in place of compute-sanitizer (which the
// GPU pool does not allow).  Every traversal-stack push, node / primitive / material index and frame store is
// range-checked; a violation is COUNTED (b200rt_debug_bounds) and the access skipped, so a broken tree shows up as
// a failed test instead of silent corruption.  Slots: 0 stack, 1 node index, 2 primitive / material index, 3 pixel.
#ifdef B200RT_DEBUG_BOUNDS
struct DebugBounds {
    unsigned long long *viol;   // [4]
    uint32_t n_nodes, n_spheres, n_quads, n_materials, stack_cap;
};
#define B200RT_CHECK(S, cond, slot) ((cond) ? true : (atomicAdd((S).dbg.viol + (slot), 1ull), false))
#else
#define B200RT_CHECK(S, cond, slot) true
#endif

struct DeviceScene {
    const float4 *nodes;        // 8 x float4 per 4-wide node (bvh_builder.h Node4)
    const double2 *spheres;     // 2 x double2 per sphere, leaf order: {cx, cy}, {cz, r}
    const uint2 *sphere_meta;   // {canonical prim index, material index}
    const double2 *quads;       // 8 x double2 per quad, leaf order: n^[3] V[3] w[3] s1[3] s2[3] pad
    const uint2 *quad_meta;
    const DeviceMaterial *materials;
    // The scene-spanning primitives the tree leaves out (bvh_builder.h spanning_key), tested by every ray before the tree:
    // references as in a leaf (kQuadFlagD | quad position, or sphere position), after the tree's in the leaf order.
    uint32_t n_hoisted;
    uint32_t hoisted_ref[4];
#ifdef B200RT_DEBUG_BOUNDS
    DebugBounds dbg;
#endif
};

constexpr uint32_t kLeafFlagD = 0x80000000u;
constexpr uint32_t kQuadFlagD = 0x40000000u;
constexpr uint32_t kNoHit = 0xFFFFFFFFu;
constexpr float kBoxSlack = 1.0f + 1e-6f;      // covers inv rounding (2^-23) + FMA rounding (2^-24) on both sides: 3.6e-7

struct Ray {
    double ox, oy, oz, dx, dy, dz;   // direction NOT normalised, as in the reference (ray3d.h)
};

struct Hit {
    double t;
    uint32_t ref;   // kNoHit, or (kQuadFlagD?) | index into the leaf-ordered per-type array
};

struct TraversalCounters {
    unsigned long long nodes = 0, prims = 0, quads = 0;   // node visits, primitive tests (all), of which quads
};

__device__ __forceinline__ uint32_t canonical_prim(const DeviceScene &S, uint32_t ref) {
#ifdef B200RT_DEBUG_BOUNDS
    if (!B200RT_CHECK(S, (ref & kQuadFlagD) ? (ref & ~kQuadFlagD) < S.dbg.n_quads : ref < S.dbg.n_spheres, 2)) return 0xFFFFFFFFu;
#endif
    return (ref & kQuadFlagD) ? __ldg(&S.quad_meta[ref & ~kQuadFlagD]).x : __ldg(&S.sphere_meta[ref]).x;
}

// Sphere::hit_by (sphere.h:45-96).  `a` = dot(dir, dir) is hoisted out (same operations, same
// order, so the same bits).  Returns true and the accepted root, or false.
__device__ __forceinline__ bool sphere_root(double ox, double oy, double oz, double dx, double dy, double dz,
                                            double a, double cx, double cy, double cz, double r,
                                            double tmin, double tmax, bool tie_ok, double &root_out) {
#ifdef B200RT_EXP_FP32_LEAF
    // EXPERIMENT ONLY (breaks parity): the sphere test in plain FP32, origin difference formed in double.  Measures
    // the CEILING of any scheme that takes FP64 out of the traversal (deferred exact tests, FP32 intervals): such a
    // scheme still does at least this much work per leaf step.
    {
        const float ocx = (float)(ox - cx), ocy = (float)(oy - cy), ocz = (float)(oz - cz);
        const float fdx = (float)dx, fdy = (float)dy, fdz = (float)dz, fa = (float)a, fr = (float)r;
        const float b_half = fdx * ocx + fdy * ocy + fdz * ocz;
        const float c = (ocx * ocx + ocy * ocy + ocz * ocz) - fr * fr;
        const float disc = b_half * b_half - fa * c;
        if (disc < 0) return false;
        const float sq = sqrtf(disc);
        const float inv_a = __frcp_rn(fa);
        float root = (-b_half - sq) * inv_a;
        if (!((float)tmin < root && root < (float)tmax)) {
            root = (-b_half + sq) * inv_a;
            if (!((float)tmin < root && root < (float)tmax)) return false;
        }
        root_out = (double)root;
        return true;
    }
#endif
    const double ocx = ox - cx, ocy = oy - cy, ocz = oz - cz;
    const double b_half = dx * ocx + dy * ocy + dz * ocz;
    const double c = (ocx * ocx + ocy * ocy + ocz * ocz) - r * r;
    const double disc = b_half * b_half - a * c;
    if (disc < 0) return false;
    const double sq = sqrt(disc);
    const double q1 = -b_half - sq, q2 = -b_half + sq;   // the roots are q1 / a and q2 / a (sphere.h:61,67)
    // A double division costs ~30 instructions, and most sphere tests do not end in a hit: the ray
    // starts ON this sphere (every scattered ray re-tests the sphere it left: q1 ~ 0 < tmin * a) or
    // the sphere lies beyond the current closest hit.  Where the outcome of the reference's
    // `ray_times.contains_exclusive(root)` is certain WITHOUT dividing -- q is away from tmin * a or
    // tmax * a by more than 1e-12 relative, a margin 4 orders above the division's rounding -- skip
    // the division; otherwise do exactly what the reference does.  Outcomes are identical.
    bool try_first = true;
    if (a > 0) {
        const double lo = tmin * a, hi = tmax * a;
        const double lo_m = fabs(lo) * 1e-12, hi_m = fabs(hi) * 1e-12;
        if (q1 > hi + hi_m) return false;                    // smaller root > tmax, so is the larger one
        if (q1 < lo - lo_m) {                                // smaller root < tmin: sphere.h:67 goes to the larger
            if (q2 < lo - lo_m || q2 > hi + hi_m) return false;
            try_first = false;
        }
    }
    double root;
    // Interval::contains_exclusive (interval.h:38); `tie_ok` additionally admits root == tmax so
    // that the caller can break the tie by primitive index.
    if (try_first) {
        root = q1 / a;
        if (tmin < root && (root < tmax || (tie_ok && root == tmax))) { root_out = root; return true; }
        // With a > 0 the larger root is >= the smaller one (q1 <= q2 and division by a positive
        // number are monotone under rounding): a smaller root already past tmin failed on the tmax
        // side, and so does the larger one.
        if (a > 0 && root > tmin) return false;
    }
    root = q2 / a;
    if (!(tmin < root && (root < tmax || (tie_ok && root == tmax)))) return false;
    root_out = root;
    return true;
}

// Parallelogram::hit_by (parallelogram.h:177-240) with the constructor's precomputed
// unit_plane_normal / scaled_plane_normal (parallelogram.h:269-279) supplied by the host.
__device__ __forceinline__ bool quad_root(double ox, double oy, double oz, double dx, double dy, double dz,
                                          const double2 *__restrict__ q, double tmin, double tmax,
                                          bool tie_ok, double &t_out) {
    const double2 q0 = __ldg(q + 0), q1 = __ldg(q + 1), q2 = __ldg(q + 2);
    const double nx = q0.x, ny = q0.y, nz = q1.x, vx = q1.y, vy = q2.x, vz = q2.y;
    const double den = nx * dx + ny * dy + nz * dz;
    if (fabs(den) < 1e-9) return false;
    const double ex = vx - ox, ey = vy - oy, ez = vz - oz;
    const double num = nx * ex + ny * ey + nz * ez;
    {   // The plane is often hit behind the origin or beyond the current closest hit: where num / den is
        // outside (tmin, tmax) by more than 1e-12 relative (far above the division's rounding), the
        // reference's contains_exclusive(hit_time) is certainly false -- skip the double division.
        const double lo = tmin * den, hi = tmax * den;
        const double lo_m = fabs(lo) * 1e-12, hi_m = fabs(hi) * 1e-12;
        if (den > 0 ? (num < lo - lo_m || num > hi + hi_m) : (num > lo + lo_m || num < hi - hi_m)) return false;
    }
    const double t = num / den;
    if (!(tmin < t && (t < tmax || (tie_ok && t == tmax)))) return false;
    const double2 q3 = __ldg(q + 3), q4 = __ldg(q + 4), q5 = __ldg(q + 5), q6 = __ldg(q + 6), q7 = __ldg(q + 7);
    const double wx = q3.x, wy = q3.y, wz = q4.x;
    const double s1x = q4.y, s1y = q5.x, s1z = q5.y;
    const double s2x = q6.x, s2y = q6.y, s2z = q7.x;
    const double px = (ox + t * dx) - vx, py = (oy + t * dy) - vy, pz = (oz + t * dz) - vz;
    // alpha = dot(w, cross(p, s2)); beta = dot(w, cross(s1, p))
    const double c1x = py * s2z - pz * s2y, c1y = pz * s2x - px * s2z, c1z = px * s2y - py * s2x;
    const double alpha = wx * c1x + wy * c1y + wz * c1z;
    const double c2x = s1y * pz - s1z * py, c2y = s1z * px - s1x * pz, c2z = s1x * py - s1y * px;
    const double beta = wx * c2x + wy * c2y + wz * c2z;
    if (!(0 <= alpha && alpha <= 1 && 0 <= beta && beta <= 1)) return false;
    t_out = t;
    return true;
}

#define B200RT_CSWAP(a, b) { const uint32_t lo_ = min(a, b); b = max(a, b); a = lo_; }

constexpr uint32_t kTravDone = 0xFFFFFFFFu;   // `cur` value once the stack has run dry

// Per-ray traversal state.  The traversal is written as STEPS (one interior node, or one leaf)
// so that kernels can either run them in a plain loop (closest_hit below) or let a warp vote
// on which kind of step to execute next (path_megakernel).
struct Trav {
    Ray ray;                         // the ray, exactly as given (FP64; direction not normalised)
    double a;                        // dot(dir, dir), hoisted out of Sphere::hit_by (sphere.h:49)
    double tmin;
    Hit best;                        // best.t doubles as the shrinking ray_times.max (bvh.h:651)
    float fix, fiy, fiz;             // FP32 1/d for the box tests (0 on an axis the ray is parallel to)
    float cnx, cny, cnz;             // o * (1/d), rounded UP   (+ pad): t_near = near_plane * inv - cn
    float cfx, cfy, cfz;             // o * (1/d), rounded DOWN (- pad): t_far  = far_plane  * inv - cf
    float tmin32, tmax32;
    volatile uint32_t near_off[3];   // byte offset of the near-plane float4 of a node per axis; LOCAL MEMORY on purpose
    int sp;
    uint32_t cur;                    // interior node index | leaf reference | kTravDone
};

__device__ __forceinline__ bool trav_at_node(const Trav &T) { return !(T.cur & kLeafFlagD); }
__device__ __forceinline__ bool trav_at_leaf(const Trav &T) { return (T.cur & kLeafFlagD) && T.cur != kTravDone; }
__device__ __forceinline__ bool trav_done(const Trav &T) { return T.cur == kTravDone; }

// double -> float rounded towards -inf / +inf, written with plain casts and integer steps so that it
// constant-folds when the argument is a compile-time constant (the path kernels' kRayTmin / kRayTmax, path.cuh): the
// cvt.rd / cvt.ru intrinsics do not fold, and under the 64-register cap the compiler then re-executes the
// conversion (an XU-pipe instruction) in every node step instead of keeping the value in a register.
__device__ __forceinline__ float float_toward(double x, bool up) {
    float f = (float)x;
    if (up ? ((double)f < x) : ((double)f > x)) {
        int b = __float_as_int(f);
        if (f == 0.0f) b = up ? 0x00000001 : (int)0x80000001;
        else b += ((f > 0.0f) == up) ? 1 : -1;
        f = __int_as_float(b);
    }
    return f;
}

__device__ __forceinline__ void trav_axis(double o, double d, float &inv, float &cn, float &cf) {
    const float fd = (float)d;
    float r = __frcp_rn(fd);
    if (!(fabsf(r) <= 3.4028234e38f) || fd == 0.0f) r = 0.0f;   // parallel / out of FP32 range / NaN
    const double p = o * (double)r;
    const double pad = fabs(p) * 2.4e-7;                         // >= 2 ulp(FP32) of p
    inv = r;
    cn = r == 0.0f ? __int_as_float(0x7f800000) : __double2float_ru(p + pad);
    cf = r == 0.0f ? __int_as_float(0xff800000) : __double2float_rd(p - pad);
}

// Starts the traversal of the ray already stored in T.ray.
__device__ __forceinline__ void trav_setup(Trav &T, double tmin, double tmax) {
    const double ox = T.ray.ox, oy = T.ray.oy, oz = T.ray.oz, dx = T.ray.dx, dy = T.ray.dy, dz = T.ray.dz;
    // Slab tests are  t = plane * inv - o * inv  as ONE FMA per plane.  The product o * inv is formed in
    // double from the exact origin and rounded outward (plus a relative pad that also makes the
    // bound strict), so the origin is never rounded to FP32 and the only relative errors left are
    // the rounding of inv (2^-23) and of the FMA result (2^-24): covered by kBoxSlack.
    // An axis with d == 0 (or |d| below FP32 range) gets inv = 0 and infinite constants, i.e. no
    // constraint from that axis: conservative, and independent of the sign of zero (the
    // reference's own slab test, aabb.h:132-174, mishandles -0.0).
    trav_axis(ox, dx, T.fix, T.cnx, T.cfx);
    trav_axis(oy, dy, T.fiy, T.cny, T.cfy);
    trav_axis(oz, dz, T.fiz, T.cnz, T.cfz);
    T.near_off[0] = T.fix < 0.0f ? 16u : 0u; T.near_off[1] = T.fiy < 0.0f ? 48u : 32u; T.near_off[2] = T.fiz < 0.0f ? 80u : 64u;
    T.tmin = tmin;
    T.tmin32 = float_toward(tmin, false);
    T.tmax32 = float_toward(tmax, true);
    T.a = dx * dx + dy * dy + dz * dz;
    T.best.t = tmax;
    T.best.ref = kNoHit;
    T.sp = 0;
    T.cur = 0;   // root
}
__device__ __forceinline__ void trav_init(Trav &T, double ox, double oy, double oz, double dx, double dy, double dz,
                                          double tmin, double tmax) {
    T.ray.ox = ox; T.ray.oy = oy; T.ray.oz = oz; T.ray.dx = dx; T.ray.dy = dy; T.ray.dz = dz;
    trav_setup(T, tmin, tmax);
}

// Pops the next stack entry that can still contain a closer hit into T.cur (kTravDone if none).
__device__ __forceinline__ void trav_pop(Trav &T, const uint2 *stack) {
    T.cur = kTravDone;
    while (T.sp > 0) {
        const uint2 e = stack[--T.sp];
        if (__uint_as_float(e.y & ~3u) <= T.tmax32 * kBoxSlack) { T.cur = e.x; break; }
    }
}

// One interior node: conservative FP32 slab tests of its four child boxes, nearest-first order.
__device__ __forceinline__ void trav_node_step(const DeviceScene &S, Trav &T, uint2 *stack) {
    // Nodes are 128-byte aligned (checked at scene creation), so the six plane addresses are formed without
    // carries: near = base | (0/16, 32/48, 64/80), far = near ^ 16 -- one logic op each on the low word.
#ifdef B200RT_DEBUG_BOUNDS
    if (!B200RT_CHECK(S, T.cur < S.dbg.n_nodes, 1)) { trav_pop(T, stack); return; }
#endif
    const uintptr_t base = reinterpret_cast<uintptr_t>(S.nodes) + ((uintptr_t)T.cur << 7);
    const uintptr_t pnx = base | T.near_off[0], pny = base | T.near_off[1], pnz = base | T.near_off[2];
#define B200RT_NODE_F4(a) __ldg(reinterpret_cast<const float4 *>(a))
    const float4 bnx = B200RT_NODE_F4(pnx), bfx = B200RT_NODE_F4(pnx ^ 16);
    const float4 bny = B200RT_NODE_F4(pny), bfy = B200RT_NODE_F4(pny ^ 16);
    const float4 bnz = B200RT_NODE_F4(pnz), bfz = B200RT_NODE_F4(pnz ^ 16);
#undef B200RT_NODE_F4
    // The slab tests run one child PAIR per instruction: a plane's float4 holds children 0 and 1 in its .x / .y
    // registers and children 2 and 3 in .z / .w, and sm_100's paired FP32 instructions (FFMA2, FMUL2) take such a pair
    // with the ray's per-axis constants as broadcast scalar operands, so a step issues 12 FFMA2 + 2 FMUL2 instead of
    // 24 FFMA + 4 FMUL and needs no extra registers.  Each half of fma.rn.f32x2 / mul.rn.f32x2 rounds exactly as the
    // scalar fma.rn.f32 / mul.rn.f32 does, so every key -- and with it the sort order, the nodes visited and the
    // frame -- is the same bits as with one instruction per child.
#define B200RT_F2(a, b) make_float2(a, b)
#define B200RT_PLANE(p, lo, hi, inv, c) __ffma2_rn(B200RT_F2(p.lo, p.hi), B200RT_F2(inv, inv), B200RT_F2(-c, -c))
#define B200RT_PAIR(lo, hi, k0, k1)                                                                               \
    uint32_t key##k0, key##k1;                                                                                    \
    {                                                                                                             \
        const float2 nx = B200RT_PLANE(bnx, lo, hi, T.fix, T.cnx), ny = B200RT_PLANE(bny, lo, hi, T.fiy, T.cny);  \
        const float2 nz = B200RT_PLANE(bnz, lo, hi, T.fiz, T.cnz);                                                \
        const float2 fx = B200RT_PLANE(bfx, lo, hi, T.fix, T.cfx), fy = B200RT_PLANE(bfy, lo, hi, T.fiy, T.cfy);  \
        const float2 fz = B200RT_PLANE(bfz, lo, hi, T.fiz, T.cfz);                                                \
        const float tn0 = fmaxf(fmaxf(nx.x, ny.x), fmaxf(nz.x, T.tmin32));                                        \
        const float tn1 = fmaxf(fmaxf(nx.y, ny.y), fmaxf(nz.y, T.tmin32));                                        \
        const float2 tf = __fmul2_rn(B200RT_F2(fminf(fminf(fx.x, fy.x), fminf(fz.x, T.tmax32)),                    \
                                               fminf(fminf(fx.y, fy.y), fminf(fz.y, T.tmax32))),                   \
                                     B200RT_F2(kBoxSlack, kBoxSlack));                                            \
        /* slot, or all ones = miss */                                                                            \
        key##k0 = (__float_as_uint(tn0) & ~3u) | ((tn0 <= tf.x) ? (uint32_t)k0 : 0xFFFFFFFFu);                    \
        key##k1 = (__float_as_uint(tn1) & ~3u) | ((tn1 <= tf.y) ? (uint32_t)k1 : 0xFFFFFFFFu);                    \
    }
    B200RT_PAIR(x, y, 0, 1) B200RT_PAIR(z, w, 2, 3)
#undef B200RT_PAIR
#undef B200RT_PLANE
#undef B200RT_F2
    // Sort the four keys ascending (nearest first); misses sink to the end.  (Pushing the three
    // farther children UNSORTED, each with its entry distance, was measured: node visits per ray
    // unchanged within 0.2 %, but 2-3 % slower -- four predicated pushes cost more than the network.)
    B200RT_CSWAP(key0, key1) B200RT_CSWAP(key2, key3) B200RT_CSWAP(key0, key2)
    B200RT_CSWAP(key1, key3) B200RT_CSWAP(key1, key2)
    // The child reference of a slot is FETCHED from the node just read (an L1 hit) rather than selected from
    // four registers: selection is 5 ALU-pipe operations per pushed entry (or a branchy ?: chain on which the
    // lanes of a warp serialise), and the node step is bound by the ALU pipe (88 of its ~150 instructions;
    // the pipe issues one warp instruction every 2 cycles), not by the load/store unit.
#define B200RT_CHILD(key) __ldg(reinterpret_cast<const uint32_t *>((base | (uint32_t)(((key) << 2) & 0xCu)) + 96))
#define B200RT_PUSH(key) if (key != 0xFFFFFFFFu && B200RT_CHECK(S, (uint32_t)T.sp < S.dbg.stack_cap, 0)) stack[T.sp++] = make_uint2(B200RT_CHILD(key), key);
    if (key0 != 0xFFFFFFFFu) {
        B200RT_PUSH(key3) B200RT_PUSH(key2) B200RT_PUSH(key1)
        T.cur = B200RT_CHILD(key0);
    } else {
        trav_pop(T, stack);
    }
#undef B200RT_PUSH
#undef B200RT_CHILD
}

// One primitive test in the reference's arithmetic (`ref` as in a leaf): a strictly closer hit becomes T.best, and an
// exact tie goes to the lower canonical index (scene.h:59-75).
__device__ __forceinline__ void trav_prim(const DeviceScene &S, Trav &T, uint32_t ref) {
    double t;
    bool hit;
    const uint32_t i = ref & ~kQuadFlagD;
    if (ref & kQuadFlagD) {
        hit = quad_root(T.ray.ox, T.ray.oy, T.ray.oz, T.ray.dx, T.ray.dy, T.ray.dz, S.quads + (size_t)i * 8, T.tmin, T.best.t,
                        T.best.ref != kNoHit, t);
    } else {
        const double2 s0 = __ldg(S.spheres + (size_t)i * 2);
        const double2 s1 = __ldg(S.spheres + (size_t)i * 2 + 1);
        hit = sphere_root(T.ray.ox, T.ray.oy, T.ray.oz, T.ray.dx, T.ray.dy, T.ray.dz, T.a, s0.x, s0.y, s1.x, s1.y, T.tmin, T.best.t,
                          T.best.ref != kNoHit, t);
    }
    if (hit && (t < T.best.t || canonical_prim(S, ref) < canonical_prim(S, T.best.ref))) {
        T.best.t = t;
        T.best.ref = ref;
        T.tmax32 = __double2float_ru(t);
    }
}

// One leaf: FP64 primitive tests in the reference's arithmetic, then pop.
__device__ __forceinline__ uint32_t trav_leaf_step(const DeviceScene &S, Trav &T, const uint2 *stack) {
    const uint32_t cnt = (T.cur >> 26) & 0xFu, first = T.cur & 0x03FFFFFFu;
    const uint32_t type = T.cur & kQuadFlagD;
#ifdef B200RT_DEBUG_BOUNDS
    if (!B200RT_CHECK(S, first + cnt <= (type ? S.dbg.n_quads : S.dbg.n_spheres), 2)) { trav_pop(T, stack); return 0; }
#endif
    for (uint32_t i = 0; i < cnt; ++i) trav_prim(S, T, type | (first + i));
    trav_pop(T, stack);
    return cnt;
}

// The scene-spanning primitives (DeviceScene::hoisted_ref), tested right after trav_setup / trav_init and before the
// tree.  The count is the same for every lane, so the warp runs these tests converged -- a ground the rays would
// otherwise reach in a leaf at a different iteration each tests with all of them -- and the tree traversal then starts
// with tmax already at the ground hit, which culls the subtrees behind it from the first node on.  The closest hit does
// not depend on the order of the tests: each test's answer is the primitive's first root above tmin whatever tmax was,
// and exact ties go to the lower canonical index, so the result is the bits a leaf test gives.  With COUNT these
// tests are counted as primitive tests.
template <bool COUNT>
__device__ __forceinline__ void trav_hoisted(const DeviceScene &S, Trav &T, TraversalCounters *ctr) {
    for (uint32_t k = 0; k < S.n_hoisted; ++k) {
        const uint32_t ref = S.hoisted_ref[k];
#ifdef B200RT_DEBUG_BOUNDS
        if (!B200RT_CHECK(S, (ref & kQuadFlagD) ? (ref & ~kQuadFlagD) < S.dbg.n_quads : ref < S.dbg.n_spheres, 2)) continue;
#endif
        trav_prim(S, T, ref);
        if (COUNT) { ctr->prims++; if (ref & kQuadFlagD) ctr->quads++; }
    }
}

// The traversal loop.  Every iteration offers a lane BOTH kinds of step, one after the other: with NODE-then-LEAF order
// a lane whose node step lands on a leaf tests that leaf in the same iteration, together with the lanes that were
// already at a leaf -- so the expensive FP64 leaf code, the most lane-starved code of the kernel, runs with more
// lanes per execution and the ray needs fewer iterations (a ray's N N L N L takes three iterations instead of
// five).  LEAF_FIRST is the mirror image (a lane that pops a node after its leaf visits it at once): it packs the NODE
// step instead.  Measured against round 1's "one step per iteration" loop (B200, 256-512 spp, same-box A/B):
// node-then-leaf C1 +6.5 %, C2 +5.7 %, C3 +4.6 %, C4 -1.3 %, C4b -1 %, C5 +4.4 %; leaf-then-node C1 +6.5 %, C2 +3.7 %,
// C3 +4.7 %, C4 0 %, C4b +2.5 %, C5 +3.2 %.  The launcher uses leaf-first when quads outnumber spheres.  Two steps of a
// kind per iteration (L N L, N L N) lose again (-1 ... +1 %), and so did round 1's while-while form, which these loops
// replace even on the depth-3 Cornell tree (+4.6 % over it).  With COUNT the steps are counted into *ctr.
template <bool COUNT>
__device__ __forceinline__ void trav_node_counted(const DeviceScene &S, Trav &T, uint2 *stack, TraversalCounters *ctr) {
    if (trav_at_node(T)) { if (COUNT) ctr->nodes++; trav_node_step(S, T, stack); }
}
template <bool COUNT>
__device__ __forceinline__ void trav_leaf_counted(const DeviceScene &S, Trav &T, uint2 *stack, TraversalCounters *ctr) {
    if (trav_at_leaf(T)) {
        const bool is_quad = T.cur & kQuadFlagD;
        const uint32_t c = trav_leaf_step(S, T, stack);
        if (COUNT) { ctr->prims += c; if (is_quad) ctr->quads += c; }
    }
}
template <bool COUNT, bool LEAF_FIRST = false>
__device__ __forceinline__ void trav_iteration(const DeviceScene &S, Trav &T, uint2 *stack, TraversalCounters *ctr) {
    if (LEAF_FIRST) { trav_leaf_counted<COUNT>(S, T, stack, ctr); trav_node_counted<COUNT>(S, T, stack, ctr); }
    else { trav_node_counted<COUNT>(S, T, stack, ctr); trav_leaf_counted<COUNT>(S, T, stack, ctr); }
}

template <int STACK, bool COUNT, bool LEAF_FIRST = false>
__device__ __forceinline__ Hit closest_hit(const DeviceScene &S, double ox, double oy, double oz,
                                           double dx, double dy, double dz, double tmin, double tmax,
                                           TraversalCounters *ctr) {
    Trav T;
    uint2 stack[STACK];
    trav_init(T, ox, oy, oz, dx, dy, dz, tmin, tmax);
    trav_hoisted<COUNT>(S, T, ctr);
    while (!trav_done(T)) trav_iteration<COUNT, LEAF_FIRST>(S, T, stack, ctr);
    return T.best;
}

}  // namespace b200rt
