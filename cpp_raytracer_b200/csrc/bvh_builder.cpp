// bvh_builder.cpp -- parallel binned-SAH build + collapse to the 4-wide device layout.
// See bvh_builder.h for the role of this file relative to the reference
// (reference include/acceleration/bvh.h:183-550 is the single-threaded builder it stands in for).
#include "bvh_builder.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <functional>
#include <limits>

#include "thread_pool.h"

namespace b200rt {
namespace {

constexpr double kInf = std::numeric_limits<double>::infinity();

inline Box3 empty_box() { return Box3{{kInf, kInf, kInf}, {-kInf, -kInf, -kInf}}; }
// (primitive boxes never hold NaN: plain compares are enough and much cheaper than fmin/fmax)
inline void grow(Box3 &b, const Box3 &o) {
    for (int a = 0; a < 3; ++a) {
        b.lo[a] = o.lo[a] < b.lo[a] ? o.lo[a] : b.lo[a];
        b.hi[a] = o.hi[a] > b.hi[a] ? o.hi[a] : b.hi[a];
    }
}
inline void grow_point(Box3 &b, const double p[3]) {
    for (int a = 0; a < 3; ++a) {
        b.lo[a] = p[a] < b.lo[a] ? p[a] : b.lo[a];
        b.hi[a] = p[a] > b.hi[a] ? p[a] : b.hi[a];
    }
}
inline void centroid(const Box3 &b, double c[3]) {
    // midpoint written so that huge finite coordinates do not overflow
    for (int a = 0; a < 3; ++a) c[a] = 0.5 * b.lo[a] + 0.5 * b.hi[a];
}
// Half surface area of `b` with every extent divided by `scale` (keeps the pathological scene,
// whose coordinates reach 1e166, inside double range).
inline double half_area_scaled(const Box3 &b, double scale) {
    double e[3];
    for (int a = 0; a < 3; ++a) {
        e[a] = (b.hi[a] - b.lo[a]) / scale;
        if (!(e[a] >= 0)) return 0.0;   // empty box
    }
    return e[0] * e[1] + e[1] * e[2] + e[2] * e[0];
}
inline float round_down(double v) {
    float f = (float)v;
    if ((double)f > v) f = std::nextafterf(f, -std::numeric_limits<float>::infinity());
    return f;
}
inline float round_up(double v) {
    float f = (float)v;
    if ((double)f < v) f = std::nextafterf(f, std::numeric_limits<float>::infinity());
    return f;
}
inline int ceil_log2(uint32_t n) {
    int l = 0;
    while ((1u << l) < n) ++l;
    return l;
}

struct BinNode {
    Box3 box;
    uint32_t left = 0, right = 0;    // interior
    uint32_t first = 0, count = 0;   // leaf when count > 0 (range of idx[])
    uint32_t n_prims = 0;            // primitives below this node
    uint8_t type = 0;                // leaf primitive type
};

struct Builder {
    const std::vector<Box3> &boxes;
    const uint64_t n_spheres;
    const BuildParams P;
    std::vector<uint32_t> idx;
    std::vector<BinNode> nodes;
    std::atomic<uint32_t> n_nodes{0};
    std::atomic<uint32_t> max_depth{0};

    static constexpr uint32_t kTopRange = 1u << 16;   // ranges at least this big are split with the whole pool
    static constexpr int kMaxBins = 64;

    Builder(const std::vector<Box3> &b, uint64_t ns, const BuildParams &p) : boxes(b), n_spheres(ns), P(p) {}

    inline int type_of(uint32_t prim) const { return prim >= n_spheres ? 1 : 0; }
    inline double cost_of(int type) const { return type ? P.cost_quad : P.cost_sphere; }

    struct RangeInfo {
        Box3 box = empty_box(), cbox = empty_box();
        uint32_t n_quads = 0;
    };
    void scan_chunk(uint32_t lo, uint32_t hi, RangeInfo &r) const {
        for (uint32_t i = lo; i < hi; ++i) {
            const Box3 &b = boxes[idx[i]];
            grow(r.box, b);
            double c[3];
            centroid(b, c);
            grow_point(r.cbox, c);
            r.n_quads += type_of(idx[i]);
        }
    }
    RangeInfo scan(uint32_t lo, uint32_t hi, ThreadPool *pool) const {
        const uint32_t n = hi - lo;
        RangeInfo r;
        if (!pool) { scan_chunk(lo, hi, r); return r; }
        const int chunks = pool->size() * 4;
        std::vector<RangeInfo> part(chunks);
        pool->parallel_for(chunks, [&](int c) {
            scan_chunk(lo + (uint32_t)((uint64_t)n * c / chunks), lo + (uint32_t)((uint64_t)n * (c + 1) / chunks), part[c]);
        });
        for (auto &p : part) { grow(r.box, p.box); grow(r.cbox, p.cbox); r.n_quads += p.n_quads; }
        return r;
    }

    struct Bin {   // trivially constructible on purpose: only the 3*B bins in use are reset
        Box3 box;
        double weight;
        uint32_t count;
        void reset() { box = empty_box(); weight = 0; count = 0; }
    };
    static inline int bin_of(double c, double cmin, double inv_extent, int B) {
        int b = (int)((c - cmin) * inv_extent);
        return b < 0 ? 0 : (b >= B ? B - 1 : b);
    }
    void bin_chunk(uint32_t lo, uint32_t hi, const RangeInfo &info, const double inv_ext[3], Bin *bins /*3*B*/, int B) const {
        for (uint32_t i = lo; i < hi; ++i) {
            const uint32_t prim = idx[i];
            const Box3 &b = boxes[prim];
            double c[3];
            centroid(b, c);
            const double w = cost_of(type_of(prim));
            for (int a = 0; a < 3; ++a) {
                if (inv_ext[a] == 0) continue;
                Bin &bn = bins[a * B + bin_of(c[a], info.cbox.lo[a], inv_ext[a], B)];
                grow(bn.box, b);
                bn.weight += w;
                bn.count++;
            }
        }
    }

    void make_leaf(uint32_t node, uint32_t lo, uint32_t hi, int type) {
        nodes[node].first = lo;
        nodes[node].count = hi - lo;
        nodes[node].type = (uint8_t)type;
    }

    // Decides what happens to idx[lo,hi) at `node`: returns true if it became a leaf; otherwise
    // partitions the range at `mid` and allocates the two children (l, l+1).
    bool split(uint32_t node, uint32_t lo, uint32_t hi, int depth, ThreadPool *pool, uint32_t &mid, uint32_t &l) {
        {   // track depth
            uint32_t d = (uint32_t)depth, cur = max_depth.load(std::memory_order_relaxed);
            while (d > cur && !max_depth.compare_exchange_weak(cur, d, std::memory_order_relaxed)) {}
        }
        const uint32_t n = hi - lo;
        const RangeInfo info = scan(lo, hi, pool);
        nodes[node].box = info.box;
        nodes[node].n_prims = n;
        const bool pure = info.n_quads == 0 || info.n_quads == n;
        if (n == 1) { make_leaf(node, lo, hi, info.n_quads ? 1 : 0); return true; }

        mid = lo;   // idx[lo,mid) goes left
        bool have_split = false;

        double ext[3], max_ext = 0;
        int max_axis = 0;
        for (int a = 0; a < 3; ++a) {
            ext[a] = info.cbox.hi[a] - info.cbox.lo[a];
            if (ext[a] > max_ext) { max_ext = ext[a]; max_axis = a; }
        }
        const bool depth_exhausted = depth + ceil_log2(n) >= P.max_binary_depth;

        if (!depth_exhausted && max_ext > 0 && std::isfinite(max_ext)) {
            // fewer bins for small ranges: clearing 3 x 32 bins per node would dominate the build
            const int B = n >= 64u ? P.sah_bins : (n >= 16u ? std::min(P.sah_bins, 16) : std::min(P.sah_bins, 8));
            double inv_ext[3];
            for (int a = 0; a < 3; ++a) inv_ext[a] = (ext[a] > 0 && std::isfinite(ext[a])) ? B / ext[a] : 0.0;
            Bin bins[3 * kMaxBins];
            for (int k = 0; k < 3 * B; ++k) bins[k].reset();
            if (!pool) {
                bin_chunk(lo, hi, info, inv_ext, bins, B);
            } else {
                const int chunks = pool->size() * 2;
                std::vector<std::vector<Bin>> part(chunks, std::vector<Bin>(3 * B));
                pool->parallel_for(chunks, [&](int c) {
                    for (auto &b : part[c]) b.reset();
                    bin_chunk(lo + (uint32_t)((uint64_t)n * c / chunks), lo + (uint32_t)((uint64_t)n * (c + 1) / chunks),
                              info, inv_ext, part[c].data(), B);
                });
                for (auto &p : part)
                    for (int k = 0; k < 3 * B; ++k) {
                        grow(bins[k].box, p[k].box);
                        bins[k].weight += p[k].weight;
                        bins[k].count += p[k].count;
                    }
            }
            // node extent used to normalise areas
            double scale = 0;
            for (int a = 0; a < 3; ++a) scale = std::fmax(scale, info.box.hi[a] - info.box.lo[a]);
            if (!(scale > 0) || !std::isfinite(scale)) scale = 1;
            const double node_area = half_area_scaled(info.box, scale);
            double total_w = 0;
            for (int k = 0; k < B; ++k) total_w += bins[max_axis * B + k].weight;

            double best_cost = kInf;
            int best_axis = -1, best_bin = -1;
            double right_area[kMaxBins], right_w[kMaxBins];
            for (int a = 0; a < 3; ++a) {
                if (inv_ext[a] == 0) continue;
                const Bin *bb = &bins[a * B];
                Box3 acc = empty_box();
                double w = 0;
                for (int k = B - 1; k > 0; --k) {
                    grow(acc, bb[k].box);
                    w += bb[k].weight;
                    right_area[k] = half_area_scaled(acc, scale);
                    right_w[k] = w;
                }
                acc = empty_box();
                w = 0;
                uint32_t cnt = 0;
                for (int k = 0; k < B - 1; ++k) {   // split after bin k
                    grow(acc, bb[k].box);
                    w += bb[k].weight;
                    cnt += bb[k].count;
                    if (cnt == 0 || cnt == n) continue;
                    double cost = half_area_scaled(acc, scale) * w + right_area[k + 1] * right_w[k + 1];
                    if (cost < best_cost) { best_cost = cost; best_axis = a; best_bin = k; }
                }
            }
            if (best_axis >= 0 && std::isfinite(best_cost) && node_area > 0) {
                const double split_cost = P.cost_traversal * 2 + best_cost / node_area;
                const double leaf_cost = total_w;
                if ((int)n <= P.max_leaf_prims && pure && leaf_cost <= split_cost) {
                    make_leaf(node, lo, hi, info.n_quads ? 1 : 0);
                    return true;
                }
                const double cmin = info.cbox.lo[best_axis], ie = inv_ext[best_axis];
                auto it = std::partition(idx.begin() + lo, idx.begin() + hi, [&](uint32_t prim) {
                    const Box3 &b = boxes[prim];
                    return bin_of(0.5 * b.lo[best_axis] + 0.5 * b.hi[best_axis], cmin, ie, B) <= best_bin;
                });
                mid = (uint32_t)(it - idx.begin());
                have_split = mid > lo && mid < hi;
            }
        }
        if (!have_split) {
            if ((int)n <= P.max_leaf_prims && pure && !(max_ext > 0)) {   // coincident centroids, small: leaf
                make_leaf(node, lo, hi, info.n_quads ? 1 : 0);
                return true;
            }
            if (!pure && (int)n <= P.max_leaf_prims) {
                // small mixed range: separate the two primitive types so that leaves stay pure
                auto it = std::partition(idx.begin() + lo, idx.begin() + hi, [&](uint32_t prim) { return type_of(prim) == 0; });
                mid = (uint32_t)(it - idx.begin());
            } else {
                // median split along the widest centroid axis (also the depth-cap fallback)
                mid = lo + n / 2;
                if (max_ext > 0) {
                    std::nth_element(idx.begin() + lo, idx.begin() + mid, idx.begin() + hi, [&](uint32_t a, uint32_t b) {
                        return 0.5 * boxes[a].lo[max_axis] + 0.5 * boxes[a].hi[max_axis] <
                               0.5 * boxes[b].lo[max_axis] + 0.5 * boxes[b].hi[max_axis];
                    });
                }
            }
        }
        l = n_nodes.fetch_add(2);
        nodes[node].left = l;
        nodes[node].right = l + 1;
        return false;
    }

    void build_serial(uint32_t node, uint32_t lo, uint32_t hi, int depth) {
        uint32_t mid, l;
        if (split(node, lo, hi, depth, nullptr, mid, l)) return;
        build_serial(l, lo, mid, depth + 1);
        build_serial(l + 1, mid, hi, depth + 1);
    }

    struct Item { uint32_t node, lo, hi; int depth; };
    void build(ThreadPool &pool, uint32_t n) {
        if (pool.size() == 1 || n < kTopRange) { build_serial(0, 0, n, 1); return; }
        // top of the tree: one node at a time, each scanned/binned by the whole pool
        std::vector<Item> top{{0, 0, n, 1}}, subtrees;
        while (!top.empty()) {
            const Item it = top.back();
            top.pop_back();
            if (it.hi - it.lo < kTopRange) { subtrees.push_back(it); continue; }
            uint32_t mid, l;
            if (split(it.node, it.lo, it.hi, it.depth, &pool, mid, l)) continue;
            top.push_back({l, it.lo, mid, it.depth + 1});
            top.push_back({l + 1, mid, it.hi, it.depth + 1});
        }
        // below: independent subtrees, largest first
        std::sort(subtrees.begin(), subtrees.end(), [](const Item &a, const Item &b) { return a.hi - a.lo > b.hi - b.lo; });
        pool.parallel_for((int)subtrees.size(), [&](int i) {
            const Item &it = subtrees[i];
            build_serial(it.node, it.lo, it.hi, it.depth);
        });
    }
};

// Collapses (part of) the binary tree into 4-wide nodes.  Used twice: once serially for the top
// of the tree, where subtrees below `task_threshold` primitives are recorded as tasks instead of
// being descended into, and once per task, in parallel, into task-local arrays that are stitched
// into the final arrays with index offsets afterwards.
struct Emitter {
    struct Task { uint32_t bin_node; int32_t parent; int slot; uint32_t depth4; };
    const Builder &B;
    std::vector<Node4> nodes;
    std::vector<uint32_t> sphere_order, quad_order;
    uint32_t max_depth4 = 0;
    uint64_t n_leaves = 0;
    std::vector<Task> *tasks = nullptr;
    uint32_t task_threshold = 0;

    explicit Emitter(const Builder &b) : B(b) {}

    int32_t encode_leaf(const BinNode &bn) {
        std::vector<uint32_t> &order = bn.type ? quad_order : sphere_order;
        const uint32_t first = (uint32_t)order.size();
        for (uint32_t i = 0; i < bn.count; ++i) {
            uint32_t prim = B.idx[bn.first + i];
            order.push_back(bn.type ? (uint32_t)(prim - B.n_spheres) : prim);
        }
        n_leaves++;
        return (int32_t)(kLeafFlag | (bn.type ? kQuadFlag : 0u) | (bn.count << kLeafCountShift) | first);
    }

    // Emits the 4-wide node for binary interior node `b`; returns its (local) index.
    int32_t emit(uint32_t b, uint32_t depth4) {
        max_depth4 = std::max(max_depth4, depth4);
        const int32_t me = (int32_t)nodes.size();
        nodes.emplace_back();
        uint32_t kids[4];
        int nk = 0;
        kids[nk++] = B.nodes[b].left;
        kids[nk++] = B.nodes[b].right;
        double scale = 0;
        for (int a = 0; a < 3; ++a) scale = std::fmax(scale, B.nodes[b].box.hi[a] - B.nodes[b].box.lo[a]);
        if (!(scale > 0) || !std::isfinite(scale)) scale = 1;
        // Pull up the interior child with the largest box until four slots are used.
        while (nk < 4) {
            int pick = -1;
            double best = -1;
            for (int k = 0; k < nk; ++k) {
                const BinNode &c = B.nodes[kids[k]];
                if (c.count) continue;
                const double area = half_area_scaled(c.box, scale);
                if (area > best) { best = area; pick = k; }
            }
            if (pick < 0) break;
            const BinNode &c = B.nodes[kids[pick]];
            kids[pick] = c.left;
            kids[nk++] = c.right;
        }
        Node4 n4;
        for (int k = 0; k < 4; ++k) {
            n4.lox[k] = n4.loy[k] = n4.loz[k] = std::numeric_limits<float>::infinity();
            n4.hix[k] = n4.hiy[k] = n4.hiz[k] = -std::numeric_limits<float>::infinity();
            n4.child[k] = kEmptyChild;
            n4.pad[k] = 0;
        }
        for (int k = 0; k < nk; ++k) {
            const BinNode &c = B.nodes[kids[k]];
            n4.lox[k] = round_down(c.box.lo[0]); n4.hix[k] = round_up(c.box.hi[0]);
            n4.loy[k] = round_down(c.box.lo[1]); n4.hiy[k] = round_up(c.box.hi[1]);
            n4.loz[k] = round_down(c.box.lo[2]); n4.hiz[k] = round_up(c.box.hi[2]);
            if (c.count) n4.child[k] = encode_leaf(c);
            else if (tasks && c.n_prims <= task_threshold) { tasks->push_back({kids[k], me, k, depth4 + 1}); n4.child[k] = 0; }
            else n4.child[k] = emit(kids[k], depth4 + 1);
        }
        nodes[me] = n4;
        return me;
    }
};

// Collapse + emit of the whole tree rooted at binary node 0 (an interior node) into `out`.
void collapse_tree(const Builder &B, int threads, uint64_t n, BuiltBVH &out) {
    Emitter top(B);
    std::vector<Emitter::Task> tasks;
    if (threads > 1 && n >= (1u << 16)) {
        top.tasks = &tasks;
        top.task_threshold = (uint32_t)std::max<uint64_t>(2048, n / ((uint64_t)threads * 16));
    }
    top.emit(0, 1);
    std::vector<Emitter> parts;
    parts.reserve(tasks.size());
    for (size_t t = 0; t < tasks.size(); ++t) parts.emplace_back(B);
    if (!tasks.empty()) {
        ThreadPool pool(threads);
        pool.parallel_for((int)tasks.size(), [&](int t) {
            parts[t].nodes.reserve(B.nodes[tasks[t].bin_node].n_prims / 2 + 4);
            parts[t].emit(tasks[t].bin_node, tasks[t].depth4);
        });
    }
    // offsets of every part inside the final arrays
    std::vector<uint32_t> node_off(tasks.size() + 1), sph_off(tasks.size() + 1), quad_off(tasks.size() + 1);
    node_off[0] = (uint32_t)top.nodes.size(); sph_off[0] = (uint32_t)top.sphere_order.size(); quad_off[0] = (uint32_t)top.quad_order.size();
    for (size_t t = 0; t < tasks.size(); ++t) {
        node_off[t + 1] = node_off[t] + (uint32_t)parts[t].nodes.size();
        sph_off[t + 1] = sph_off[t] + (uint32_t)parts[t].sphere_order.size();
        quad_off[t + 1] = quad_off[t] + (uint32_t)parts[t].quad_order.size();
    }
    out.nodes.resize(node_off.back());
    out.sphere_order.resize(sph_off.back());
    out.quad_order.resize(quad_off.back());
    std::copy(top.nodes.begin(), top.nodes.end(), out.nodes.begin());
    std::copy(top.sphere_order.begin(), top.sphere_order.end(), out.sphere_order.begin());
    std::copy(top.quad_order.begin(), top.quad_order.end(), out.quad_order.begin());
    out.depth = top.max_depth4;
    out.n_leaves = top.n_leaves;
    for (size_t t = 0; t < tasks.size(); ++t) {
        out.nodes[tasks[t].parent].child[tasks[t].slot] = (int32_t)node_off[t];   // part-local root is index 0
        out.depth = std::max(out.depth, parts[t].max_depth4);
        out.n_leaves += parts[t].n_leaves;
    }
    auto stitch = [&](int t) {
        const Emitter &e = parts[t];
        for (size_t i = 0; i < e.nodes.size(); ++i) {
            Node4 nd = e.nodes[i];
            for (int k = 0; k < 4; ++k) {
                const uint32_t c = (uint32_t)nd.child[k];
                if (!(c & kLeafFlag)) nd.child[k] = (int32_t)(c + node_off[t]);
                else if ((c >> kLeafCountShift) & 0xF) nd.child[k] = (int32_t)(c + ((c & kQuadFlag) ? quad_off[t] : sph_off[t]));
            }
            out.nodes[node_off[t] + i] = nd;
        }
        std::copy(e.sphere_order.begin(), e.sphere_order.end(), out.sphere_order.begin() + sph_off[t]);
        std::copy(e.quad_order.begin(), e.quad_order.end(), out.quad_order.begin() + quad_off[t]);
    };
    if (!tasks.empty()) {
        ThreadPool pool(threads);
        pool.parallel_for((int)tasks.size(), stitch);
    }
}

}  // namespace

std::vector<uint32_t> select_spanning(const std::vector<Box3> &prim_boxes, uint32_t max_hoisted) {
    const size_t n = prim_boxes.size();
    const size_t keep = std::min<size_t>(std::min(max_hoisted, kMaxHoisted), n ? n - 1 : 0);
    if (!keep) return {};
    Box3 scene = empty_box();
    for (const Box3 &b : prim_boxes) grow(scene, b);
    std::vector<uint64_t> keys;
    for (size_t i = 0; i < n; ++i)
        if (const uint64_t k = spanning_key(prim_boxes[i].lo, prim_boxes[i].hi, scene.lo, scene.hi, (uint32_t)i)) keys.push_back(k);
    std::sort(keys.begin(), keys.end(), std::greater<uint64_t>());
    std::vector<uint32_t> out;
    for (size_t k = 0; k < keys.size() && k < keep; ++k) out.push_back(0xFFFFFFFFu - (uint32_t)keys[k]);
    return out;
}

bool build_bvh4(const std::vector<Box3> &prim_boxes, uint64_t n_spheres, uint64_t n_quads,
                const std::vector<uint32_t> &hoisted, const BuildParams &params_in, BuiltBVH &out, const char **err) {
    const uint64_t n_all = n_spheres + n_quads, n = n_all - hoisted.size();   // n: primitives in the tree
    out = BuiltBVH{};
    if (prim_boxes.size() != n_all) { *err = "prim_boxes size mismatch"; return false; }
    if (n_spheres > kLeafIndexMask || n_quads > kLeafIndexMask) { *err = "too many primitives for the leaf encoding (max 2^26 per type)"; return false; }
    std::vector<uint8_t> is_hoisted(n_all, 0);
    for (uint32_t p : hoisted) {
        if (p >= n_all || is_hoisted[p]) { *err = "hoisted primitive out of range or listed twice"; return false; }
        is_hoisted[p] = 1;
    }
    if (n_all && !n) { *err = "every primitive hoisted"; return false; }
    BuildParams P = params_in;
    P.max_leaf_prims = std::clamp(P.max_leaf_prims, 1, kMaxLeafPrims);
    P.sah_bins = std::clamp(P.sah_bins, 4, 64);
    P.max_binary_depth = std::clamp(P.max_binary_depth, 28, 60);
    const int threads = P.threads > 0 ? P.threads : ThreadPool::hardware_threads();

    Node4 root;
    for (int k = 0; k < 4; ++k) {
        root.lox[k] = root.loy[k] = root.loz[k] = std::numeric_limits<float>::infinity();
        root.hix[k] = root.hiy[k] = root.hiz[k] = -std::numeric_limits<float>::infinity();
        root.child[k] = kEmptyChild;
        root.pad[k] = 0;
    }
    if (n == 0) {   // empty scene: a root whose four slots are empty; every ray misses
        out.nodes.push_back(root);
        out.depth = 1;
        return true;
    }

    Builder B(prim_boxes, n_spheres, P);
    B.idx.reserve(n);
    for (uint64_t i = 0; i < n_all; ++i)
        if (!is_hoisted[i]) B.idx.push_back((uint32_t)i);
    B.nodes.resize(2 * n);
    B.n_nodes = 1;
    const auto t_start = std::chrono::steady_clock::now();
    {
        ThreadPool pool(n < Builder::kTopRange ? 1 : threads);
        B.build(pool, (uint32_t)n);
    }
    const auto t_built = std::chrono::steady_clock::now();
    out.binary_depth = B.max_depth.load();

    if (B.nodes[0].count) {
        // single leaf at the root: wrap it in a 4-wide root with one used slot
        Emitter e(B);
        out.nodes.push_back(root);
        const BinNode &c = B.nodes[0];
        Node4 &r = out.nodes[0];
        r.lox[0] = round_down(c.box.lo[0]); r.hix[0] = round_up(c.box.hi[0]);
        r.loy[0] = round_down(c.box.lo[1]); r.hiy[0] = round_up(c.box.hi[1]);
        r.loz[0] = round_down(c.box.lo[2]); r.hiz[0] = round_up(c.box.hi[2]);
        r.child[0] = e.encode_leaf(c);
        out.sphere_order = e.sphere_order;
        out.quad_order = e.quad_order;
        out.n_leaves = 1;
        out.depth = 1;
    } else {
        collapse_tree(B, threads, n, out);
    }
    for (uint32_t p : hoisted) {
        const bool quad = p >= n_spheres;
        std::vector<uint32_t> &order = quad ? out.quad_order : out.sphere_order;
        out.hoisted_ref.push_back((quad ? kQuadFlag : 0u) | (uint32_t)order.size());
        order.push_back(quad ? (uint32_t)(p - n_spheres) : p);
    }
    if (out.sphere_order.size() != n_spheres || out.quad_order.size() != n_quads) { *err = "internal: leaf order size mismatch"; return false; }
    if (std::getenv("B200RT_BUILD_TIMING")) {
        const auto t_end = std::chrono::steady_clock::now();
        std::fprintf(stderr, "[b200rt] bvh build: binary tree %.1f ms (%d threads), collapse+emit %.1f ms, %zu nodes\n",
                     std::chrono::duration<double, std::milli>(t_built - t_start).count(), threads,
                     std::chrono::duration<double, std::milli>(t_end - t_built).count(), out.nodes.size());
    }
    return true;
}

bool validate_bvh4(const BuiltBVH &bvh, const std::vector<Box3> &prim_boxes, uint64_t n_spheres,
                   uint64_t n_quads, const char **err) {
    std::vector<uint8_t> seen_s(n_spheres, 0), seen_q(n_quads, 0);
    struct Item { int32_t node; uint32_t depth; Box3 bound; };
    std::vector<Item> stack;
    Box3 all{{-kInf, -kInf, -kInf}, {kInf, kInf, kInf}};
    stack.push_back({0, 1, all});
    uint32_t depth = 0;
    uint64_t visited = 0;
    auto inside = [](const Box3 &in, const Box3 &outb) {
        for (int a = 0; a < 3; ++a)
            if (in.lo[a] < outb.lo[a] || in.hi[a] > outb.hi[a]) return false;
        return true;
    };
    while (!stack.empty()) {
        Item it = stack.back();
        stack.pop_back();
        if (it.node < 0 || (size_t)it.node >= bvh.nodes.size()) { *err = "child index out of range"; return false; }
        if (++visited > bvh.nodes.size()) { *err = "node graph is not a tree"; return false; }
        depth = std::max(depth, it.depth);
        const Node4 &n = bvh.nodes[it.node];
        for (int k = 0; k < 4; ++k) {
            Box3 slot{{n.lox[k], n.loy[k], n.loz[k]}, {n.hix[k], n.hiy[k], n.hiz[k]}};
            const uint32_t c = (uint32_t)n.child[k];
            if (c & kLeafFlag) {
                const uint32_t cnt = (c >> kLeafCountShift) & 0xF, first = c & kLeafIndexMask;
                const bool quad = c & kQuadFlag;
                if (cnt == 0) continue;
                if (!inside(slot, it.bound)) { *err = "leaf slot box escapes its ancestors"; return false; }
                for (uint32_t i = 0; i < cnt; ++i) {
                    const auto &order = quad ? bvh.quad_order : bvh.sphere_order;
                    if (first + i >= order.size()) { *err = "leaf run out of range"; return false; }
                    const uint32_t p = order[first + i];
                    auto &seen = quad ? seen_q : seen_s;
                    if (p >= seen.size() || seen[p]) { *err = "primitive referenced twice or out of range"; return false; }
                    seen[p] = 1;
                    if (!inside(prim_boxes[quad ? n_spheres + p : p], slot)) { *err = "primitive box not inside its leaf slot box"; return false; }
                }
            } else {
                if (!inside(slot, it.bound)) { *err = "child slot box escapes its ancestors"; return false; }
                stack.push_back({(int32_t)c, it.depth + 1, slot});
            }
        }
    }
    // the hoisted primitives: the last of their type in the leaf order, each in no leaf
    size_t hoisted_of[2] = {0, 0};
    for (uint32_t r : bvh.hoisted_ref) hoisted_of[(r & kQuadFlag) ? 1 : 0]++;
    for (uint32_t r : bvh.hoisted_ref) {
        const bool quad = r & kQuadFlag;
        const auto &order = quad ? bvh.quad_order : bvh.sphere_order;
        const uint32_t pos = r & kLeafIndexMask;
        if ((r & ~(kQuadFlag | kLeafIndexMask)) || pos >= order.size() || pos < order.size() - hoisted_of[quad ? 1 : 0]) {
            *err = "hoisted reference is not among the last of its type in the leaf order"; return false;
        }
        auto &seen = quad ? seen_q : seen_s;
        const uint32_t p = order[pos];
        if (p >= seen.size() || seen[p]) { *err = "hoisted primitive also in the tree, or out of range"; return false; }
        seen[p] = 1;
    }
    for (auto s : seen_s) if (!s) { *err = "sphere missing from the tree"; return false; }
    for (auto s : seen_q) if (!s) { *err = "quad missing from the tree"; return false; }
    if (depth != bvh.depth) { *err = "reported depth differs from actual depth"; return false; }
    return true;
}

}  // namespace b200rt
