// rt_bvh_host.cpp — host-side BVH build with the reference's topology.
//
// The GPU path may traverse in any order (the BVH is a conservative cull), but two things must follow
// the reference's tree (ray-tracer-slave/local-dependencies/bvh/src/bvh/bvh_impl.rs:229-364):
//   * the DFS (left-first) leaf order, which decides exact-distance ties in the nearest-hit min_by
//     (ray-tracer-slave/src/shapes/mod.rs:177-182, bvh_impl.rs:373-398), and
//   * the N = 1 case (root is a leaf, always a candidate).
// So the builder makes the same decisions — centroid-bounds largest axis, 6 SAH buckets with
// bucket = ((c - cmin)/extent * 5.99) as usize, first strictly lower cost wins, halve the list when the
// centroid extent is < 1e-5, one primitive per leaf — evaluated with the same f32 operations, but works
// in place on one index array (stable counting sort by bucket = the reference's bucket concatenation)
// and emits only inner nodes, children encoded as codes, in DFS pre-order.
//
// Build with -ffp-contract=off (no FMA contraction on the host either).
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <mutex>
#include <thread>

#include <emmintrin.h>  // SSE2: the traversal-tree builder bins with it (x86-64 hosts; this image has no other)

#include "rt_host.h"

namespace rtb {
namespace {

constexpr int kBuckets = 6;
// A subtree over n primitives has exactly n - 1 inner nodes and its leaves are idx[lo,hi) in their final order, so
// every node's slot in the DFS pre-order arrays is known before its subtree is built: node `base`, left subtree from
// base + 1, right subtree from base + n_left.  Subtrees above this size are built by their own thread: 2048 on hosts
// with >= 8 hardware threads (on a 16-core host the reference build of 65,536 spheres drops from 30 to 6.5 ms), never
// on smaller hosts.
static const size_t kParallelMin = std::thread::hardware_concurrency() >= 8 ? 2048 : (size_t)-1 / 4;
constexpr float kEpsilon = 0.00001f;  // bvh::EPSILON (lib.rs:80)

// f32::min / f32::max inline (libm's fminf/fmaxf are out-of-line calls under -fno-fast-math and were most of the build
// time).  Their NaN-ignoring branch is not needed: the callers validate every primitive's bounds as finite, and min / max
// / sub / add / div-by-2 of finite or infinite values never produce a NaN here; for equal operands (and for +0 / -0)
// these return the second one, as the previous NaN-aware form did.
inline float nmin(float a, float b) { return a < b ? a : b; }
inline float nmax(float a, float b) { return a > b ? a : b; }

struct Bounds {
    float lo[3], hi[3];
    void clear() {
        for (int a = 0; a < 3; a++) {
            lo[a] = std::numeric_limits<float>::infinity();
            hi[a] = -std::numeric_limits<float>::infinity();
        }
    }
    void join(const Box& b) {  // AABB::join — f32::min/max (NaN-ignoring)
        for (int a = 0; a < 3; a++) {
            lo[a] = nmin(lo[a], b.min[a]);
            hi[a] = nmax(hi[a], b.max[a]);
        }
    }
    void join(const Bounds& b) {
        for (int a = 0; a < 3; a++) {
            lo[a] = nmin(lo[a], b.lo[a]);
            hi[a] = nmax(hi[a], b.hi[a]);
        }
    }
    void grow(const float p[3]) {  // AABB::grow
        for (int a = 0; a < 3; a++) {
            lo[a] = nmin(lo[a], p[a]);
            hi[a] = nmax(hi[a], p[a]);
        }
    }
    bool empty() const { return lo[0] > hi[0] || lo[1] > hi[1] || lo[2] > hi[2]; }
    float area() const {  // AABB::surface_area: 2*(sx*sy + sx*sz + sy*sz)
        float sx = hi[0] - lo[0], sy = hi[1] - lo[1], sz = hi[2] - lo[2];
        return 2.0f * (sx * sy + sx * sz + sy * sz);
    }
    Box box() const {
        Box b;
        for (int a = 0; a < 3; a++) {
            b.min[a] = lo[a];
            b.max[a] = hi[a];
        }
        return b;
    }
};

inline void centre_of(const Box& b, float c[3]) {  // AABB::center: min + (max - min)/2
    for (int a = 0; a < 3; a++) c[a] = b.min[a] + ((b.max[a] - b.min[a]) / 2.0f);
}

struct Builder {
    const std::vector<Box>& boxes;
    std::vector<uint32_t> idx, tmp;
    std::vector<uint8_t> bucket_of;
    std::vector<float> centre;  // AABB::center of every shape, computed once (same f32 operations every time)
    HostBVH* out;
    std::string* err;
    std::atomic<bool> failed{false};
    std::atomic<uint32_t> max_depth{0};
    std::mutex err_mu;

    Builder(const std::vector<Box>& b, HostBVH* o, std::string* e) : boxes(b), out(o), err(e) {
        idx.resize(b.size());
        tmp.resize(b.size());
        bucket_of.resize(b.size());
        centre.resize(3 * b.size());
        for (size_t i = 0; i < b.size(); i++) {
            idx[i] = (uint32_t)i;
            centre_of(b[i], &centre[3 * i]);
        }
    }

    void fail(const char* msg) {
        std::lock_guard<std::mutex> g(err_mu);
        if (!failed.load() && err) *err = msg;
        failed.store(true);
    }
    void note_depth(uint32_t d) {
        uint32_t cur = max_depth.load(std::memory_order_relaxed);
        while (d > cur && !max_depth.compare_exchange_weak(cur, d, std::memory_order_relaxed)) {}
    }

    // Builds the subtree over idx[lo,hi) into inner[base, base + n - 1) and returns its code.  all_in / cent_in: the
    // node's shape bounds and centroid bounds when the parent already has them (the joins of its buckets — min/max are
    // exact and associative, so they equal a pass over the shapes up to the sign of a zero, which no decision sees).
    int32_t build(size_t lo, size_t hi, uint32_t depth, size_t base, const Bounds* all_in = nullptr,
                  const Bounds* cent_in = nullptr) {
        if (failed.load(std::memory_order_relaxed)) return 0;
        if (depth > 4096) {
            fail("BVH deeper than 4096 levels");
            return 0;
        }
        const size_t n = hi - lo;
        if (n == 1) {
            note_depth(depth);
            return ~(int32_t)idx[lo];
        }
        Bounds all, cent;
        if (all_in && cent_in) {
            all = *all_in;
            cent = *cent_in;
        } else {
            all.clear();
            cent.clear();
            for (size_t i = lo; i < hi; i++) {
                all.join(boxes[idx[i]]);
                cent.grow(&centre[3 * (size_t)idx[i]]);
            }
        }
        const int32_t me = (int32_t)base;

        // AABB::largest_axis (aabb.rs:570-580)
        const float sx = cent.hi[0] - cent.lo[0], sy = cent.hi[1] - cent.lo[1], sz = cent.hi[2] - cent.lo[2];
        const int axis = (sx > sy && sx > sz) ? 0 : (sy > sz ? 1 : 2);
        const float extent = cent.hi[axis] - cent.lo[axis];

        size_t mid;
        Bounds bl, br, cl, cr;
        bool child_bounds = false;  // bl/br + cl/cr describe the children completely
        if (n == 2 && extent >= kEpsilon && extent < std::numeric_limits<float>::infinity()) {
            // Two shapes, finite extent (half of all nodes): the centroid at the low end has rel = 0 → bucket 0, the other
            // rel = extent/extent = 1 → bucket 5; every split gives the same cost and the first wins, so the children
            // are (low-end shape, other shape) with their own boxes — the bucket machinery's result, without running it.
            if (!(centre[3 * (size_t)idx[lo] + axis] == cent.lo[axis])) std::swap(idx[lo], idx[lo + 1]);
            mid = lo + 1;
            bl.clear();
            br.clear();
            bl.join(boxes[idx[lo]]);
            br.join(boxes[idx[lo + 1]]);
        } else if (extent < kEpsilon) {
            mid = lo + n / 2;
            bl.clear();
            br.clear();
            for (size_t i = lo; i < mid; i++) bl.join(boxes[idx[i]]);
            for (size_t i = mid; i < hi; i++) br.join(boxes[idx[i]]);
        } else {
            Bounds bb[kBuckets], bc[kBuckets];
            size_t cnt[kBuckets] = {0, 0, 0, 0, 0, 0};
            for (auto& b : bb) b.clear();
            for (auto& b : bc) b.clear();
            for (size_t i = lo; i < hi; i++) {
                const float* c = &centre[3 * (size_t)idx[i]];
                const float rel = (c[axis] - cent.lo[axis]) / extent;
                const float scaled = rel * ((float)kBuckets - 0.01f);
                // `as usize`: truncate, saturate, NaN → 0
                size_t k = (scaled == scaled && scaled > 0.0f) ? (scaled >= 1.8e19f ? (size_t)-1 : (size_t)scaled) : 0;
                if (k >= (size_t)kBuckets) {
                    fail("bucket index out of range (non-finite bounds)");
                    return 0;
                }
                bucket_of[i] = (uint8_t)k;
                cnt[k]++;
                bb[k].join(boxes[idx[i]]);
                bc[k].grow(c);
            }
            int best = 0;
            float best_cost = std::numeric_limits<float>::infinity();
            bl.clear();
            br.clear();
            const float parent_area = all.area();
            for (int s = 0; s < kBuckets - 1; s++) {
                Bounds l, r;
                l.clear();
                r.clear();
                size_t nl = 0, nr = 0;
                for (int k = 0; k <= s; k++) {
                    l.join(bb[k]);
                    nl += cnt[k];
                }
                for (int k = s + 1; k < kBuckets; k++) {
                    r.join(bb[k]);
                    nr += cnt[k];
                }
                const float cost = ((float)nl * l.area() + (float)nr * r.area()) / parent_area;
                if (cost < best_cost) {
                    best = s;
                    best_cost = cost;
                    bl = l;
                    br = r;
                }
            }
            // stable counting sort of idx[lo,hi) by bucket == concatenating the bucket vectors
            size_t start[kBuckets], pos = 0;
            for (int k = 0; k < kBuckets; k++) {
                start[k] = pos;
                pos += cnt[k];
            }
            for (size_t i = lo; i < hi; i++) tmp[lo + start[bucket_of[i]]++] = idx[i];
            std::memcpy(&idx[lo], &tmp[lo], n * sizeof(uint32_t));
            size_t nl = 0;
            for (int k = 0; k <= best; k++) nl += cnt[k];
            mid = lo + nl;
            cl.clear();
            cr.clear();
            for (int k = 0; k <= best; k++) cl.join(bc[k]);
            for (int k = best + 1; k < kBuckets; k++) cr.join(bc[k]);
            child_bounds = true;
        }
        if (bl.empty() || br.empty() || mid == lo || mid == hi) {  // reference: assert!(!child_aabb.is_empty())
            fail("degenerate split (empty child bounds)");
            return 0;
        }
        int32_t l = 0, r = 0;
        std::thread t;
        bool spawned = false;
        if (mid - lo >= kParallelMin && hi - mid >= kParallelMin && depth < 6) {  // at most 63 threads
            try {
                t = std::thread([&] { l = build(lo, mid, depth + 1, base + 1, child_bounds ? &bl : nullptr, child_bounds ? &cl : nullptr); });
                spawned = true;
            } catch (...) {  // no thread to be had: build the left child here
            }
        }
        if (spawned) {
            r = build(mid, hi, depth + 1, base + (mid - lo), child_bounds ? &br : nullptr, child_bounds ? &cr : nullptr);
            t.join();
        } else {
            l = build(lo, mid, depth + 1, base + 1, child_bounds ? &bl : nullptr, child_bounds ? &cl : nullptr);
            r = build(mid, hi, depth + 1, base + (mid - lo), child_bounds ? &br : nullptr, child_bounds ? &cr : nullptr);
        }
        HostNode& nd = out->inner[me];
        nd.box_l = bl.box();
        nd.box_r = br.box();
        nd.left = l;
        nd.right = r;
        return me;
    }
};

}  // namespace

// ---------------------------------------------------------------------------------------------------------
// Traversal-quality tree: binned SAH over all three axes (16 bins), one primitive per leaf.  Used only to
// CULL on the GPU (any conservative tree gives the reference's nearest hit; exact-distance ties are broken by
// the DFS rank of the reference-topology tree, which is still built).  Leaves are codes ~index like above.
// ---------------------------------------------------------------------------------------------------------
namespace {
struct alignas(16) SahRec {  // one primitive, permuted in place: centroid + world position | box min | box max (3 x 16 bytes)
    float c[3];
    uint32_t id;
    float bmin[4], bmax[4];
};
struct alignas(16) Bounds4 {  // lo | hi as two SSE lanes-of-four (w unused)
    __m128 lo, hi;
    void clear() {
        lo = _mm_set1_ps(std::numeric_limits<float>::infinity());
        hi = _mm_set1_ps(-std::numeric_limits<float>::infinity());
    }
    void join(const SahRec& r) {
        lo = _mm_min_ps(lo, _mm_load_ps(r.bmin));
        hi = _mm_max_ps(hi, _mm_load_ps(r.bmax));
    }
    void join(const Bounds4& b) {
        lo = _mm_min_ps(lo, b.lo);
        hi = _mm_max_ps(hi, b.hi);
    }
    float area() const {  // 0 for an empty box
        alignas(16) float d[4];
        _mm_store_ps(d, _mm_sub_ps(hi, lo));
        if (d[0] < 0.0f || d[1] < 0.0f || d[2] < 0.0f) return 0.0f;
        return 2.0f * (d[0] * d[1] + d[0] * d[2] + d[1] * d[2]);
    }
    Box box() const {
        alignas(16) float a[4], b[4];
        _mm_store_ps(a, lo);
        _mm_store_ps(b, hi);
        Box r;
        for (int k = 0; k < 3; k++) {
            r.min[k] = a[k];
            r.max[k] = b[k];
        }
        return r;
    }
};
struct SahBuilder {
    std::vector<SahRec> rec;
    HostBVH* out;
    std::atomic<uint32_t> max_depth{0};
    static constexpr int kBins = 16;

    SahBuilder(const std::vector<Box>& b, HostBVH* o) : out(o) {
        rec.resize(b.size());
        for (size_t i = 0; i < b.size(); i++) {
            rec[i].id = (uint32_t)i;
            for (int a = 0; a < 3; a++) {
                rec[i].bmin[a] = b[i].min[a];
                rec[i].bmax[a] = b[i].max[a];
                rec[i].c[a] = 0.5f * (b[i].min[a] + b[i].max[a]);
            }
            rec[i].bmin[3] = rec[i].bmax[3] = 0.0f;
        }
    }
    void note_depth(uint32_t d) {
        uint32_t cur = max_depth.load(std::memory_order_relaxed);
        while (d > cur && !max_depth.compare_exchange_weak(cur, d, std::memory_order_relaxed)) {}
    }

    int32_t build(size_t lo, size_t hi, uint32_t depth, size_t base) {
        const size_t n = hi - lo;
        if (n == 1) {
            note_depth(depth);
            return ~(int32_t)rec[lo].id;
        }
        // centroid bounds (the id lane rides along and is ignored)
        __m128 cmin4 = _mm_set1_ps(std::numeric_limits<float>::infinity()), cmax4 = _mm_set1_ps(-std::numeric_limits<float>::infinity());
        for (size_t i = lo; i < hi; i++) {
            const __m128 c = _mm_load_ps(rec[i].c);
            cmin4 = _mm_min_ps(cmin4, c);
            cmax4 = _mm_max_ps(cmax4, c);
        }
        alignas(16) float cmin[4], cmax[4];
        _mm_store_ps(cmin, cmin4);
        _mm_store_ps(cmax, cmax4);
        // one pass bins all three axes; small nodes (most of them) use fewer bins, their cost is the per-node set-up
        const int nb = n <= 4 ? 2 : (n <= 16 ? 4 : (n <= 64 ? 8 : kBins));
        Bounds4 bb[3][kBins];
        uint32_t cnt[3][kBins];
        alignas(16) float scale[4] = {0.0f, 0.0f, 0.0f, 0.0f};
        bool use[3];
        for (int a = 0; a < 3; a++) {
            const float ext = cmax[a] - cmin[a];
            use[a] = ext > 0.0f;
            scale[a] = use[a] ? (float)nb * (1.0f - 1e-6f) / ext : 0.0f;
            for (int k = 0; k < nb; k++) { bb[a][k].clear(); cnt[a][k] = 0; }
        }
        cmin[3] = 0.0f;
        const __m128 cm = _mm_load_ps(cmin), sc4 = _mm_load_ps(scale);
        const __m128i top = _mm_set1_epi32(nb - 1), zero = _mm_setzero_si128();
        auto bins_of = [&](const SahRec& r, int k[4]) {  // bin of the centroid on every axis at once
            __m128i b = _mm_cvttps_epi32(_mm_mul_ps(_mm_sub_ps(_mm_load_ps(r.c), cm), sc4));
            b = _mm_max_epi16(_mm_min_epi16(b, top), zero);  // bins are small non-negative ints: 16-bit lanes do
            _mm_storeu_si128(reinterpret_cast<__m128i*>(k), b);
        };
        auto bin_of = [&](const SahRec& r, int a) {
            int k = (int)((r.c[a] - cmin[a]) * scale[a]);
            return k < 0 ? 0 : (k >= nb ? nb - 1 : k);
        };
        for (size_t i = lo; i < hi; i++) {
            int k[4];
            bins_of(rec[i], k);
            for (int a = 0; a < 3; a++) {
                if (!use[a]) continue;
                cnt[a][k[a]]++;
                bb[a][k[a]].join(rec[i]);
            }
        }
        int best_axis = -1, best_split = 0;
        float best_cost = std::numeric_limits<float>::infinity();
        Bounds4 best_l, best_r;
        best_l.clear();
        best_r.clear();
        for (int a = 0; a < 3; a++) {
            if (!use[a]) continue;
            Bounds4 racc[kBins];
            size_t rcnt[kBins];
            Bounds4 acc;
            acc.clear();
            size_t c = 0;
            for (int k = nb - 1; k > 0; k--) {
                acc.join(bb[a][k]);
                c += cnt[a][k];
                racc[k] = acc;
                rcnt[k] = c;
            }
            Bounds4 lacc;
            lacc.clear();
            size_t lc = 0;
            for (int k = 0; k < nb - 1; k++) {
                lacc.join(bb[a][k]);
                lc += cnt[a][k];
                if (lc == 0 || rcnt[k + 1] == 0) continue;
                const float cost = (float)lc * lacc.area() + (float)rcnt[k + 1] * racc[k + 1].area();
                if (cost < best_cost) { best_cost = cost; best_axis = a; best_split = k; best_l = lacc; best_r = racc[k + 1]; }
            }
        }
        size_t mid = lo;
        if (best_axis >= 0) {
            auto it = std::partition(rec.begin() + lo, rec.begin() + hi,
                                     [&](const SahRec& r) { return bin_of(r, best_axis) <= best_split; });
            mid = (size_t)(it - rec.begin());
        }
        if (mid == lo || mid == hi) {  // coincident centroids: halve, bounds by a pass
            mid = lo + n / 2;
            best_l.clear();
            best_r.clear();
            for (size_t i = lo; i < mid; i++) best_l.join(rec[i]);
            for (size_t i = mid; i < hi; i++) best_r.join(rec[i]);
        }
        const int32_t me = (int32_t)base;
        int32_t l = 0, r = 0;
        std::thread t;
        bool spawned = false;
        if (mid - lo >= kParallelMin && hi - mid >= kParallelMin && depth < 6) {  // at most 63 threads
            try {
                t = std::thread([&] { l = build(lo, mid, depth + 1, base + 1); });
                spawned = true;
            } catch (...) {  // no thread to be had: build the left child here
            }
        }
        if (spawned) {
            r = build(mid, hi, depth + 1, base + (mid - lo));
            t.join();
        } else {
            l = build(lo, mid, depth + 1, base + 1);
            r = build(mid, hi, depth + 1, base + (mid - lo));
        }
        HostNode& nd = out->inner[me];
        nd.box_l = best_l.box();
        nd.box_r = best_r.box();
        nd.left = l;
        nd.right = r;
        return me;
    }
};
}  // namespace

bool build_bvh_sah(const std::vector<Box>& boxes, HostBVH* out) {
    out->inner.clear();
    out->leaf_order.clear();
    out->depth = 0;
    if (boxes.empty()) return false;
    out->inner.assign(boxes.size() - 1, HostNode{});
    SahBuilder b(boxes, out);
    out->root = b.build(0, boxes.size(), 0, 0);
    out->leaf_order.resize(boxes.size());
    for (size_t i = 0; i < boxes.size(); i++) out->leaf_order[i] = b.rec[i].id;
    out->depth = b.max_depth.load();
    out->node_count = (uint32_t)(out->inner.size() + out->leaf_order.size());
    return true;
}

bool build_bvh(const std::vector<Box>& boxes, HostBVH* out, std::string* err) {
    out->inner.clear();
    out->leaf_order.clear();
    out->depth = 0;
    if (boxes.empty()) {
        if (err) *err = "empty scene";
        return false;
    }
    out->inner.assign(boxes.size() - 1, HostNode{});
    Builder b(boxes, out, err);
    out->root = b.build(0, boxes.size(), 0, 0);
    out->leaf_order = b.idx;  // the leaves in DFS order are the final order of the index array
    out->depth = b.max_depth.load();
    out->node_count = (uint32_t)(out->inner.size() + out->leaf_order.size());
    return !b.failed.load();
}

}  // namespace rtb
