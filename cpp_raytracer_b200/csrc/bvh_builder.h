// bvh_builder.h -- host-side builder of the 4-wide BVH the device kernels traverse.
//
// Takes the place of the reference's BVH::build_bvh_tree / flatten_bvh_tree
// (reference include/acceleration/bvh.h:183-550) but is a different design: a binned-SAH
// binary tree built in parallel on the host, collapsed to 4-wide nodes whose four child boxes
// are stored SoA in one 128-byte line with FP32 bounds rounded OUTWARD (conservative), and
// leaves that reference contiguous runs of a per-type primitive array in leaf order.
// Closest-hit results do not depend on the tree (only on the primitives), so the tree is free
// to differ from the reference's; see DESIGN.md "Acceleration structure".
#pragma once
#include <cstdint>
#include <cstring>
#include <vector>

#ifdef __CUDACC__
#define B200RT_HD __host__ __device__
#else
#define B200RT_HD
#endif

namespace b200rt {

struct Box3 {
    double lo[3], hi[3];
};

// Scene-spanning primitives (DESIGN.md §5): a primitive whose box has at least half the surface area of the whole
// scene's box -- a ground plane or ground sphere -- is tested by almost every ray.  Up to kMaxHoisted of them, largest
// first, are left out of the tree and tested once per ray before it (traverse.cuh trav_hoisted), with the warp still
// converged, instead of in a divergent leaf step; their boxes no longer widen the tree's nodes either.  At least one
// primitive always stays in the tree.  Both builders select with this one function (select_spanning on the host,
// lbvh.cu on the device) from the primitive boxes in double precision, as the reference's constructors compute them.
constexpr uint32_t kMaxHoisted = 4;
// 0 if primitive `index` with box [lo, hi] does not span the scene box [slo, shi]; else a key that orders the spanning
// ones largest first and equal areas by the lower index: the area's FP32 bits above the complement of the index.  A scene
// whose box has no finite, non-zero area in double (the pathological scene's nested spheres reach 1e166) hoists nothing.
B200RT_HD inline uint64_t spanning_key(const double lo[3], const double hi[3], const double slo[3], const double shi[3],
                                       uint32_t index) {
    const double ex = hi[0] - lo[0], ey = hi[1] - lo[1], ez = hi[2] - lo[2];
    const double sx = shi[0] - slo[0], sy = shi[1] - slo[1], sz = shi[2] - slo[2];
    const double area = ex * ey + ey * ez + ez * ex, scene = sx * sy + sy * sz + sz * sx;   // half surface areas
    if (!(scene > 0 && scene <= 1.7976931348623157e308) || !(area >= 0.5 * scene)) return 0;
    const float f = (float)area;   // positive: its bits order as its value
    uint32_t bits;
    memcpy(&bits, &f, sizeof bits);
    return ((uint64_t)bits << 32) | (0xFFFFFFFFu - index);
}
// The primitives to hoist (indices into prim_boxes, largest first): at most min(max_hoisted, kMaxHoisted), and at most
// prim_boxes.size() - 1.
std::vector<uint32_t> select_spanning(const std::vector<Box3> &prim_boxes, uint32_t max_hoisted);

// One 4-wide node = one 128-byte cache line = eight 16-byte vector loads.
// Child i's box is component i of each float4.  child[i] encodes:
//   >= 0            : index of an interior Node4
//   bit 31 set      : leaf; bit 30 = primitive type (0 sphere, 1 quad); bits 26..29 = count
//                     (0 = empty slot); bits 0..25 = first index in the per-type leaf-ordered array
struct alignas(128) Node4 {
    float lox[4], hix[4], loy[4], hiy[4], loz[4], hiz[4];
    int32_t child[4];
    int32_t pad[4];
};
static_assert(sizeof(Node4) == 128, "Node4 must be exactly one 128-byte line");

constexpr uint32_t kLeafFlag = 0x80000000u;
constexpr uint32_t kQuadFlag = 0x40000000u;
constexpr int kLeafCountShift = 26;
constexpr uint32_t kLeafIndexMask = (1u << kLeafCountShift) - 1;
constexpr int kMaxLeafPrims = 8;
constexpr int32_t kEmptyChild = (int32_t)kLeafFlag;   // leaf with count 0

struct BuildParams {
    int max_leaf_prims = 2;
    int sah_bins = 32;
    int threads = 0;          // 0 = all
    int max_binary_depth = 40;
    double cost_traversal = 1.0;   // relative cost of one child-box test
    double cost_sphere = 2.0;      // relative cost of one FP64 sphere test
    double cost_quad = 3.0;        // relative cost of one FP64 quad test
};

struct BuiltBVH {
    std::vector<Node4> nodes;              // nodes[0] is the root
    std::vector<uint32_t> sphere_order;    // leaf-ordered position -> input sphere index
    std::vector<uint32_t> quad_order;      // leaf-ordered position -> input quad index
    std::vector<uint32_t> hoisted_ref;     // the hoisted primitives, after the tree's in leaf order: sphere position,
                                           // or kQuadFlag | quad position
    uint32_t depth = 0;                    // depth of the 4-wide tree (root = 1)
    uint32_t binary_depth = 0;
    uint64_t n_leaves = 0;
};

// prim_boxes: n_spheres sphere boxes followed by n_quads quad boxes (double precision, as the
// reference computes them: sphere.h:112-123, parallelogram.h:281-295).  hoisted (select_spanning): primitives
// the tree leaves out; they follow the tree's primitives in the leaf order.
// Returns false (with a message in err) if the scene exceeds the node encoding limits.
bool build_bvh4(const std::vector<Box3> &prim_boxes, uint64_t n_spheres, uint64_t n_quads,
                const std::vector<uint32_t> &hoisted, const BuildParams &params, BuiltBVH &out, const char **err);

// Checks the structural invariants of a built tree (every primitive not hoisted in exactly one leaf,
// the hoisted ones at the end of the leaf order and in no leaf, every primitive's box inside every
// ancestor slot box, leaf runs contiguous, depth as reported).
// Used by the CPU test-suite through b200rt_selftest_bvh().
bool validate_bvh4(const BuiltBVH &bvh, const std::vector<Box3> &prim_boxes, uint64_t n_spheres,
                   uint64_t n_quads, const char **err);

}  // namespace b200rt
