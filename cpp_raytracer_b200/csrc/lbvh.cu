// lbvh.cu -- acceleration-structure construction ON THE GPU (B200RT_BUILDER_GPU_LBVH).
//
// Stands in for BVH::build_bvh_tree / flatten_bvh_tree (reference include/acceleration/bvh.h:183-550,
// single-threaded: 5.5-7.2 s for the 2.2 M / 3.1 M primitive scenes on the B200 box's host) when
// time-to-first-pixel matters more than tree quality -- the multi-million-primitive scenes, where
// even the parallel host SAH builder (bvh_builder.cpp, ~0.8 s) costs more than the render at 8 GPUs.
//
// Builds the tree and the leaf order only, all device-side from the caller's flat arrays as they are; the
// primitive records are laid out in that order by scene_layout.cu, as for the host builder:
//   1. prim_setup      primitive bounds exactly as the reference's constructors compute them
//                      (sphere.h:112-123, parallelogram.h:281-295) in double, rounded outward to FP32;
//                      the scene's box by warp shuffle + ordered-int atomics
//   2. spanning_keys,  the scene-spanning primitives the tree leaves out (bvh_builder.h spanning_key):
//      pick_spanning   one key per primitive, then one atomicMax pass per pick
//   3. centroid_bounds centroid bounds of the primitives the tree holds
//   4. morton_codes    63-bit Morton code of the centroid (21 bits per axis); the hoisted primitives sort last
//   5. cub radix sort  (key, primitive) pairs                    [library call: a plain sort]
//   6. radix_tree      Karras 2012, "Maximizing parallelism in the construction of BVHs, octrees and
//                      k-d trees": one thread per internal node, duplicates broken by index
//   7. fit_boxes       bottom-up union of child boxes, second arrival continues (atomic counters)
//   8. leaf_order      leaf (= Morton) position -> per-type position: sphere_order / quad_order
//   9. collapse_level  binary -> 4-wide, breadth first, one launch per level: each task pulls up the
//                      larger-area grandchildren until four slots are used, reserves its Node4 with an
//                      atomic counter, patches its parent's child slot and queues its interior children
// Closest-hit results do not depend on the tree, so the parity tests run against this builder too.
#include <algorithm>
#include <cstdio>
#include <cub/cub.cuh>

#include "../../include/b200rt.h"
#include "bvh_builder.h"
#include "devmem.h"

namespace b200rt {

namespace {

#define LB_TRY(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) return e_; } while (0)

__device__ __forceinline__ int float_to_ordered(float f) {
    const int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float ordered_to_float(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }

struct PrimBoxes {
    float *lox, *loy, *loz, *hix, *hiy, *hiz;   // outward-rounded FP32 bounds per primitive
    float *cx, *cy, *cz;                         // centroid
};

// Primitive i's box in double, exactly as the reference's constructors compute it (and api.cu's sphere_box / quad_box).
__device__ __forceinline__ void prim_box(const B200rtSphere *sph, uint32_t n_sph, const B200rtQuad *quads, uint32_t i,
                                         double lo[3], double hi[3]) {
    if (i < n_sph) {                                   // sphere.h:112-123
        const B200rtSphere s = sph[i];
        for (int a = 0; a < 3; ++a) {
            const double p = s.c[a] - s.r, q = s.c[a] + s.r;
            lo[a] = fmin(p, q); hi[a] = fmax(p, q);
        }
    } else {                                           // parallelogram.h:281-295 + ensure_min_axis_length(1e-4)
        const B200rtQuad q = quads[i - n_sph];
        for (int a = 0; a < 3; ++a) {
            const double p0 = q.v[a], p1 = q.v[a] + q.s1[a], p2 = q.v[a] + q.s2[a], p3 = (q.v[a] + q.s1[a]) + q.s2[a];
            lo[a] = fmin(fmin(p0, p1), fmin(p2, p3));
            hi[a] = fmax(fmax(p0, p1), fmax(p2, p3));
            const double size = hi[a] - lo[a];
            if (size < 1e-4) { const double pad = (1e-4 - size) / 2; lo[a] -= pad; hi[a] += pad; }
        }
    }
}

__device__ __forceinline__ long long double_to_ordered(double d) {
    const long long i = __double_as_longlong(d);
    return i >= 0 ? i : i ^ 0x7fffffffffffffffll;
}
__device__ __forceinline__ double ordered_to_double(long long i) { return __longlong_as_double(i >= 0 ? i : i ^ 0x7fffffffffffffffll); }

__global__ void prim_setup(const B200rtSphere *sph, uint32_t n_sph, const B200rtQuad *quads, uint32_t n_quad, PrimBoxes B,
                           long long *sbounds /* [6]: ordered-int64 min xyz, max xyz of the primitive boxes */) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t n = n_sph + n_quad;
    const bool valid = i < n;
    const double inf = __longlong_as_double(0x7ff0000000000000ll);
    double lo[3] = {inf, inf, inf}, hi[3] = {-inf, -inf, -inf};
    if (valid) {
        prim_box(sph, n_sph, quads, i, lo, hi);
        B.lox[i] = __double2float_rd(lo[0]); B.loy[i] = __double2float_rd(lo[1]); B.loz[i] = __double2float_rd(lo[2]);
        B.hix[i] = __double2float_ru(hi[0]); B.hiy[i] = __double2float_ru(hi[1]); B.hiz[i] = __double2float_ru(hi[2]);
        B.cx[i] = (float)(0.5 * lo[0] + 0.5 * hi[0]); B.cy[i] = (float)(0.5 * lo[1] + 0.5 * hi[1]); B.cz[i] = (float)(0.5 * lo[2] + 0.5 * hi[2]);
    }
    // the scene's box (spanning_key): warp reduce, then one atomic per warp and bound
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        double mn = lo[a], mx = hi[a];
        for (int off = 16; off; off >>= 1) {
            mn = fmin(mn, __shfl_down_sync(0xffffffffu, mn, off));
            mx = fmax(mx, __shfl_down_sync(0xffffffffu, mx, off));
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMin(&sbounds[a], double_to_ordered(mn));
            atomicMax(&sbounds[3 + a], double_to_ordered(mx));
        }
    }
}

// spanning_key of every primitive (0: does not span the scene)
__global__ void spanning_keys(const B200rtSphere *sph, uint32_t n_sph, const B200rtQuad *quads, uint32_t n, const long long *sbounds,
                              unsigned long long *keys) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double lo[3], hi[3], slo[3], shi[3];
    prim_box(sph, n_sph, quads, i, lo, hi);
    for (int a = 0; a < 3; ++a) { slo[a] = ordered_to_double(sbounds[a]); shi[a] = ordered_to_double(sbounds[3 + a]); }
    keys[i] = spanning_key(lo, hi, slo, shi, i);
}

// Round r of the selection: the largest key below the one round r - 1 picked (0: none left).
__global__ void pick_spanning(const unsigned long long *keys, uint32_t n, unsigned long long *picked, int r) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long k = keys[i], bound = r ? picked[r - 1] : ~0ull;
    if (k && k < bound) atomicMax(&picked[r], k);
}

struct Hoisted {
    uint32_t n, prim[kMaxHoisted];
    __device__ __forceinline__ bool has(uint32_t i) const {
        bool h = false;
        for (uint32_t k = 0; k < n; ++k) h |= prim[k] == i;
        return h;
    }
};

// Centroid bounds of the primitives the tree holds: warp shuffle + ordered-int atomics.
__global__ void centroid_bounds(PrimBoxes B, uint32_t n, Hoisted H, int *cbounds /* [6]: ordered-int min xyz, max xyz */) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = i < n && !H.has(i);
    const float *c[3] = {B.cx, B.cy, B.cz};
    const float inf = __int_as_float(0x7f800000);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        float mn = valid ? c[a][i] : inf, mx = valid ? c[a][i] : -inf;
        for (int off = 16; off; off >>= 1) {
            mn = fminf(mn, __shfl_down_sync(0xffffffffu, mn, off));
            mx = fmaxf(mx, __shfl_down_sync(0xffffffffu, mx, off));
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMin(&cbounds[a], float_to_ordered(mn));
            atomicMax(&cbounds[3 + a], float_to_ordered(mx));
        }
    }
}

__device__ __forceinline__ unsigned long long spread21(unsigned long long x) {   // 21 bits -> every third bit
    x &= 0x1fffffull;
    x = (x | x << 32) & 0x1f00000000ffffull;
    x = (x | x << 16) & 0x1f0000ff0000ffull;
    x = (x | x << 8) & 0x100f00f00f00f00full;
    x = (x | x << 4) & 0x10c30c30c30c30c3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}

// The hoisted primitives get bit 63, above every 63-bit code: the sort puts them after the tree's primitives.
__global__ void morton_codes(PrimBoxes B, uint32_t n, const int *cbounds, Hoisted H, unsigned long long *keys, uint32_t *vals) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    vals[i] = i;
    if (H.has(i)) { keys[i] = ~0ull; return; }
    unsigned long long code = 0;
    const float *c[3] = {B.cx, B.cy, B.cz};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float lo = ordered_to_float(cbounds[a]), hi = ordered_to_float(cbounds[3 + a]);
        const float ext = hi - lo;
        float u = ext > 0.f ? (c[a][i] - lo) / ext : 0.f;
        u = fminf(fmaxf(u, 0.f), 1.f);
        const unsigned long long q = (unsigned long long)fminf(u * 2097152.0f, 2097151.0f);
        code |= spread21(q) << a;
    }
    keys[i] = code;
}

// Common-prefix length of sorted keys i and j (-1 out of range); equal keys are told apart by index.
__device__ __forceinline__ int delta(const unsigned long long *keys, int n, int i, int j) {
    if (j < 0 || j >= n) return -1;
    const unsigned long long a = keys[i], b = keys[j];
    if (a == b) return 64 + __clz(i ^ j);
    return __clzll((long long)(a ^ b));
}

struct BinTree {
    int *left, *right;        // child: >= 0 internal node index; < 0 leaf ~position (position = ~child)
    int *parent;              // parent of internal node i at [i], of leaf p at [n_internal + p]
    float *lox, *loy, *loz, *hix, *hiy, *hiz;   // internal node boxes
    int *visits;
};

__global__ void radix_tree(const unsigned long long *keys, int n, BinTree T) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    const int d = (delta(keys, n, i, i + 1) - delta(keys, n, i, i - 1)) >= 0 ? 1 : -1;
    const int dmin = delta(keys, n, i, i - d);
    int lmax = 2;
    while (delta(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int t = lmax >> 1; t >= 1; t >>= 1)
        if (delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
    const int j = i + l * d;
    const int dnode = delta(keys, n, i, j);
    int s = 0;
    for (int t = (l + 1) >> 1;; t = (t + 1) >> 1) {
        if (delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
        if (t == 1) break;
    }
    const int gamma = i + s * d + min(d, 0);
    const int lo = min(i, j), hi = max(i, j);
    const int lc = (lo == gamma) ? ~gamma : gamma;
    const int rc = (hi == gamma + 1) ? ~(gamma + 1) : gamma + 1;
    T.left[i] = lc;
    T.right[i] = rc;
    T.parent[lc >= 0 ? lc : (n - 1) + ~lc] = i;
    T.parent[rc >= 0 ? rc : (n - 1) + ~rc] = i;
    if (i == 0) T.parent[0] = -1;
}

__global__ void fit_boxes(PrimBoxes B, const uint32_t *vals, int n, BinTree T) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    int cur = T.parent[(n - 1) + p];
    while (cur >= 0) {
        __threadfence();
        if (atomicAdd(&T.visits[cur], 1) == 0) return;   // the second arrival finds both children done
        float lo[3], hi[3];
        const int ch[2] = {T.left[cur], T.right[cur]};
        for (int a = 0; a < 3; ++a) { lo[a] = __int_as_float(0x7f800000); hi[a] = __int_as_float(0xff800000); }
        for (int k = 0; k < 2; ++k) {
            if (ch[k] >= 0) {
                const int c = ch[k];
                lo[0] = fminf(lo[0], __ldcg(&T.lox[c])); lo[1] = fminf(lo[1], __ldcg(&T.loy[c])); lo[2] = fminf(lo[2], __ldcg(&T.loz[c]));
                hi[0] = fmaxf(hi[0], __ldcg(&T.hix[c])); hi[1] = fmaxf(hi[1], __ldcg(&T.hiy[c])); hi[2] = fmaxf(hi[2], __ldcg(&T.hiz[c]));
            } else {
                const uint32_t prim = vals[~ch[k]];
                lo[0] = fminf(lo[0], B.lox[prim]); lo[1] = fminf(lo[1], B.loy[prim]); lo[2] = fminf(lo[2], B.loz[prim]);
                hi[0] = fmaxf(hi[0], B.hix[prim]); hi[1] = fmaxf(hi[1], B.hiy[prim]); hi[2] = fmaxf(hi[2], B.hiz[prim]);
            }
        }
        T.lox[cur] = lo[0]; T.loy[cur] = lo[1]; T.loz[cur] = lo[2];
        T.hix[cur] = hi[0]; T.hiy[cur] = hi[1]; T.hiz[cur] = hi[2];
        cur = T.parent[cur];
    }
}

__global__ void quad_flags(const uint32_t *vals, uint32_t n, uint32_t n_sph, uint32_t *flags) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) flags[p] = vals[p] >= n_sph ? 1u : 0u;
}

struct CollapseTask { int bnode, parent4, slot; };

__device__ __forceinline__ void child_box(const BinTree &T, const PrimBoxes &B, const uint32_t *vals, int c, float lo[3], float hi[3]) {
    if (c >= 0) {
        lo[0] = T.lox[c]; lo[1] = T.loy[c]; lo[2] = T.loz[c]; hi[0] = T.hix[c]; hi[1] = T.hiy[c]; hi[2] = T.hiz[c];
    } else {
        const uint32_t prim = vals[~c];
        lo[0] = B.lox[prim]; lo[1] = B.loy[prim]; lo[2] = B.loz[prim]; hi[0] = B.hix[prim]; hi[1] = B.hiy[prim]; hi[2] = B.hiz[prim];
    }
}

__global__ void collapse_level(BinTree T, PrimBoxes B, const uint32_t *vals, const uint32_t *quad_rank, uint32_t n_sph,
                               const CollapseTask *tasks, uint32_t n_tasks, CollapseTask *next, uint32_t *next_count,
                               Node4 *nodes4, uint32_t *node_count) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tasks) return;
    const CollapseTask task = tasks[t];
    int kids[4];
    int nk = 0;
    kids[nk++] = T.left[task.bnode];
    kids[nk++] = T.right[task.bnode];
    while (nk < 4) {                       // pull up the interior child with the largest box
        int pick = -1;
        float best = -1.f;
        for (int k = 0; k < nk; ++k) {
            if (kids[k] < 0) continue;
            const int c = kids[k];
            const float ex = T.hix[c] - T.lox[c], ey = T.hiy[c] - T.loy[c], ez = T.hiz[c] - T.loz[c];
            float area = ex * ey + ey * ez + ez * ex;
            if (!(area >= 0.f)) area = 3.4e38f;            // inf/NaN extents: treat as the largest
            if (area > best) { best = area; pick = k; }
        }
        if (pick < 0) break;
        const int c = kids[pick];
        kids[pick] = T.left[c];
        kids[nk++] = T.right[c];
    }
    const uint32_t me = atomicAdd(node_count, 1u);
    if (task.parent4 >= 0) nodes4[task.parent4].child[task.slot] = (int)me;
    Node4 nd;
    const float inf = __int_as_float(0x7f800000);
    for (int k = 0; k < 4; ++k) {
        nd.lox[k] = nd.loy[k] = nd.loz[k] = inf;
        nd.hix[k] = nd.hiy[k] = nd.hiz[k] = -inf;
        nd.child[k] = kEmptyChild;
        nd.pad[k] = 0;
    }
    for (int k = 0; k < nk; ++k) {
        float lo[3], hi[3];
        child_box(T, B, vals, kids[k], lo, hi);
        nd.lox[k] = lo[0]; nd.loy[k] = lo[1]; nd.loz[k] = lo[2];
        nd.hix[k] = hi[0]; nd.hiy[k] = hi[1]; nd.hiz[k] = hi[2];
        if (kids[k] < 0) {
            const uint32_t p = (uint32_t)~kids[k];
            const bool quad = vals[p] >= n_sph;
            const uint32_t typed = quad ? quad_rank[p] : p - quad_rank[p];
            nd.child[k] = (int)(kLeafFlag | (quad ? kQuadFlag : 0u) | (1u << kLeafCountShift) | typed);
        } else {
            nd.child[k] = 0;   // patched by the child's own task
            const uint32_t q = atomicAdd(next_count, 1u);
            next[q] = CollapseTask{kids[k], (int)me, k};
        }
    }
    // the child slots of interior kids are written later by other threads: store everything but those
    Node4 *dst = nodes4 + me;
    for (int k = 0; k < 4; ++k) {
        dst->lox[k] = nd.lox[k]; dst->loy[k] = nd.loy[k]; dst->loz[k] = nd.loz[k];
        dst->hix[k] = nd.hix[k]; dst->hiy[k] = nd.hiy[k]; dst->hiz[k] = nd.hiz[k];
        dst->pad[k] = 0;
        if (k >= nk || kids[k] < 0) dst->child[k] = nd.child[k];
    }
}

// the caller's index of the primitive at each leaf (Morton) position, per type; positions from n_tree on hold the hoisted
// primitives, whose references go to hoisted_ref[p - n_tree]
__global__ void leaf_order(const uint32_t *vals, const uint32_t *quad_rank, uint32_t n, uint32_t n_tree, uint32_t n_sph,
                           uint32_t *sphere_order, uint32_t *quad_order, uint32_t *hoisted_ref) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const uint32_t prim = vals[p];
    const uint32_t ref = prim < n_sph ? p - quad_rank[p] : kQuadFlag | quad_rank[p];
    if (prim < n_sph) sphere_order[ref] = prim;
    else quad_order[quad_rank[p]] = prim - n_sph;
    if (p >= n_tree) hoisted_ref[p - n_tree] = ref;
}

template <typename T>
cudaError_t tmp_alloc(std::vector<void *> &owned, T **p, size_t count) {
    void *q = nullptr;
    cudaError_t e = dev_alloc_async(&q, (count ? count : 1) * sizeof(T), 0);
    if (e != cudaSuccess) return e;
    owned.push_back(q);
    *p = static_cast<T *>(q);
    return cudaSuccess;
}

}  // namespace

// Builds the 4-wide tree on the GPU.  d_sph / d_quads are the caller's flat structs already on the device.
// Outputs: the leaf order, sphere_order[n_sph] / quad_order[n_quad] (allocated by the caller), which ends with the up to
// max_hoisted scene-spanning primitives (spanning_key) the tree leaves out, and their references in
// hoisted_ref_out[*n_hoisted_out]; the Node4 array is allocated here (its size is only known at the end) with
// cudaMallocAsync and handed back through nodes_out.  *n_nodes_out = 0 with nothing allocated: the tree would hold fewer
// than the two primitives a radix tree needs, so the caller builds on the host.
cudaError_t build_lbvh_device(const B200rtSphere *d_sph, uint32_t n_sph, const B200rtQuad *d_quads, uint32_t n_quad,
                              uint32_t max_hoisted, uint32_t *sphere_order, uint32_t *quad_order, float4 **nodes_out,
                              uint32_t *n_nodes_out, uint32_t *depth_out, uint32_t *n_hoisted_out, uint32_t hoisted_ref_out[kMaxHoisted]) {
    const uint32_t n = n_sph + n_quad;
    *n_nodes_out = 0;
    *n_hoisted_out = 0;
    // Encoding limits: a leaf reference holds a 26-bit index into its per-type array (bvh_builder.h), and the radix
    // tree's index arithmetic ((n - 1) + ~child, lmax * d) must stay inside int.  The host builder rejects the same
    // scenes (bvh_builder.cpp); api.cu checks before calling, this is the backstop.
    if (n < 2 || n_sph > kLeafIndexMask || n_quad > kLeafIndexMask || n > (1u << 29)) return cudaErrorInvalidValue;
    std::vector<void *> owned;
    Node4 *nodes4 = nullptr;
    auto cleanup = [&]() { for (void *p : owned) dev_free(p); };
    auto fail = [&](cudaError_t e) { cleanup(); dev_free(nodes4); return e; };
    const int B = 256;
    const unsigned gn = (n + B - 1) / B;
#define LB(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) return fail(e_); } while (0)
    PrimBoxes pb;
    LB(tmp_alloc(owned, &pb.lox, n)); LB(tmp_alloc(owned, &pb.loy, n)); LB(tmp_alloc(owned, &pb.loz, n));
    LB(tmp_alloc(owned, &pb.hix, n)); LB(tmp_alloc(owned, &pb.hiy, n)); LB(tmp_alloc(owned, &pb.hiz, n));
    LB(tmp_alloc(owned, &pb.cx, n)); LB(tmp_alloc(owned, &pb.cy, n)); LB(tmp_alloc(owned, &pb.cz, n));
    long long *sbounds;
    LB(tmp_alloc(owned, &sbounds, 6));
    const long long sinit[6] = {0x7fffffffffffffffll, 0x7fffffffffffffffll, 0x7fffffffffffffffll,
                                (long long)0x8000000000000000ull, (long long)0x8000000000000000ull, (long long)0x8000000000000000ull};
    LB(cudaMemcpyAsync(sbounds, sinit, sizeof sinit, cudaMemcpyHostToDevice, 0));
    prim_setup<<<gn, B>>>(d_sph, n_sph, d_quads, n_quad, pb, sbounds);
    unsigned long long *keys, *keys_alt;
    uint32_t *vals, *vals_alt;
    LB(tmp_alloc(owned, &keys, n)); LB(tmp_alloc(owned, &keys_alt, n));
    LB(tmp_alloc(owned, &vals, n)); LB(tmp_alloc(owned, &vals_alt, n));
    // the scene-spanning primitives: one pass for the keys, then one pass per pick (largest key first)
    Hoisted H{};
    const uint32_t keep = std::min(std::min(max_hoisted, kMaxHoisted), n - 1);
    if (keep) {
        unsigned long long *picked, host_picked[kMaxHoisted];
        LB(tmp_alloc(owned, &picked, kMaxHoisted));
        LB(cudaMemsetAsync(picked, 0, kMaxHoisted * sizeof(unsigned long long), 0));
        spanning_keys<<<gn, B>>>(d_sph, n_sph, d_quads, n, sbounds, keys);
        for (uint32_t r = 0; r < keep; ++r) pick_spanning<<<gn, B>>>(keys, n, picked, (int)r);
        LB(cudaMemcpyAsync(host_picked, picked, sizeof host_picked, cudaMemcpyDeviceToHost, 0));
        LB(cudaStreamSynchronize(0));
        for (uint32_t r = 0; r < keep && host_picked[r]; ++r) H.prim[H.n++] = 0xFFFFFFFFu - (uint32_t)host_picked[r];
    }
    const uint32_t n_tree = n - H.n;
    if (n_tree < 2) { cleanup(); return cudaSuccess; }
    int *cbounds;
    LB(tmp_alloc(owned, &cbounds, 6));
    const int init[6] = {0x7fffffff, 0x7fffffff, 0x7fffffff, (int)0x80000000, (int)0x80000000, (int)0x80000000};
    LB(cudaMemcpyAsync(cbounds, init, sizeof init, cudaMemcpyHostToDevice, 0));
    centroid_bounds<<<gn, B>>>(pb, n, H, cbounds);
    morton_codes<<<gn, B>>>(pb, n, cbounds, H, keys, vals);
    {
        cub::DoubleBuffer<unsigned long long> dk(keys, keys_alt);
        cub::DoubleBuffer<uint32_t> dv(vals, vals_alt);
        const int end_bit = H.n ? 64 : 63;
        size_t tmp_bytes = 0;
        LB(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, dk, dv, (int)n, 0, end_bit));
        char *tmp;
        LB(tmp_alloc(owned, &tmp, tmp_bytes));
        LB(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, dk, dv, (int)n, 0, end_bit));
        keys = dk.Current();
        vals = dv.Current();
    }
    BinTree T;
    LB(tmp_alloc(owned, &T.left, n)); LB(tmp_alloc(owned, &T.right, n)); LB(tmp_alloc(owned, &T.parent, 2 * (size_t)n));
    LB(tmp_alloc(owned, &T.lox, n)); LB(tmp_alloc(owned, &T.loy, n)); LB(tmp_alloc(owned, &T.loz, n));
    LB(tmp_alloc(owned, &T.hix, n)); LB(tmp_alloc(owned, &T.hiy, n)); LB(tmp_alloc(owned, &T.hiz, n));
    LB(tmp_alloc(owned, &T.visits, n));
    LB(cudaMemsetAsync(T.visits, 0, n * sizeof(int), 0));
    radix_tree<<<gn, B>>>(keys, (int)n_tree, T);
    fit_boxes<<<gn, B>>>(pb, vals, (int)n_tree, T);
    // typed (per primitive kind) positions in leaf order
    uint32_t *flags, *quad_rank;
    LB(tmp_alloc(owned, &flags, n)); LB(tmp_alloc(owned, &quad_rank, n));
    quad_flags<<<gn, B>>>(vals, n, n_sph, flags);
    {
        size_t tmp_bytes = 0;
        LB(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, flags, quad_rank, (int)n));
        char *tmp;
        LB(tmp_alloc(owned, &tmp, tmp_bytes));
        LB(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, flags, quad_rank, (int)n));
    }
    uint32_t *hoisted_ref;
    LB(tmp_alloc(owned, &hoisted_ref, kMaxHoisted));
    leaf_order<<<gn, B>>>(vals, quad_rank, n, n_tree, n_sph, sphere_order, quad_order, hoisted_ref);
    // breadth-first collapse to 4-wide nodes (at most n - 1 of them)
    LB(dev_alloc_async(&nodes4, (size_t)(n - 1) * sizeof(Node4), 0));
    CollapseTask *qa, *qb;
    uint32_t *counters;   // [0] next queue size, [1] nodes emitted
    LB(tmp_alloc(owned, &qa, n)); LB(tmp_alloc(owned, &qb, n)); LB(tmp_alloc(owned, &counters, 2));
    LB(cudaMemsetAsync(counters, 0, 2 * sizeof(uint32_t), 0));
    const CollapseTask root{0, -1, 0};
    LB(cudaMemcpyAsync(qa, &root, sizeof root, cudaMemcpyHostToDevice, 0));
    uint32_t n_tasks = 1, depth = 0;
    while (n_tasks) {
        ++depth;
        collapse_level<<<(n_tasks + B - 1) / B, B>>>(T, pb, vals, quad_rank, n_sph, qa, n_tasks, qb, counters, nodes4, counters + 1);
        LB(cudaMemcpyAsync(&n_tasks, counters, sizeof(uint32_t), cudaMemcpyDeviceToHost, 0));
        LB(cudaMemsetAsync(counters, 0, sizeof(uint32_t), 0));
        LB(cudaStreamSynchronize(0));
        std::swap(qa, qb);
        if (depth > 512) return fail(cudaErrorUnknown);
    }
    uint32_t n_nodes = 0;
    LB(cudaMemcpyAsync(&n_nodes, counters + 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, 0));
    LB(cudaMemcpyAsync(hoisted_ref_out, hoisted_ref, H.n * sizeof(uint32_t), cudaMemcpyDeviceToHost, 0));
    LB(cudaStreamSynchronize(0));
    LB(cudaGetLastError());
    cleanup();
    *nodes_out = reinterpret_cast<float4 *>(nodes4);
    *n_nodes_out = n_nodes;
    *depth_out = depth;
    *n_hoisted_out = H.n;
    return cudaSuccess;
#undef LB
}

}  // namespace b200rt
