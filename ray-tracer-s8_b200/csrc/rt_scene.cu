// rt_scene.cu — world ingest: replaces `req.world` ownership + `BVH::build(&mut req.world)` of the reference's
// worker() (ray-tracer-slave/src/main.rs:37,60-61) with a device-resident scene.
//
// Two trees, two critical paths (DESIGN.md section 3):
//   * the tree the kernels TRAVERSE may be any conservative cull: big primitives out of the tree ("split" layout), then
//     a 3-axis binned-SAH tree built here on the host, or from 8192 primitives a Morton LBVH built on the device
//     (rt_bvh_device.cu).  rt_scene_create returns when this tree and the geometry are on the device.
//   * the REFERENCE-topology tree (bvh_impl.rs:229-364, same f32 decisions, rt_bvh_host.cpp) is needed only for what it
//     alone defines: the DFS leaf rank that breaks exact-distance ties (shapes/mod.rs:177-182) and the ancestor boxes a
//     ray with a zero direction component must pass (ray.rs:174-194).  A builder thread makes it beside the upload and
//     sends its tables (rank | ref_up | ref_box) to the device when they are done; a render that starts earlier marks
//     the (measure-zero) pixels that needed them and renders those again (rt_api.cu finish_launch).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>

#include "rt_ctx.h"

using namespace rtb;

namespace {

// leaf codes are ~(pid << 5) in 32 bits: 26-bit primitive ids
constexpr uint64_t MAX_PRIMS = 0x3ffffffu;
constexpr uint32_t kDeviceBuildMin = 8192;  // RT_B200_BUILD=auto: the traversal tree is built on the device from here
constexpr uint32_t kRefSyncBelow = 256;     // the reference tree is built inline below this many primitives
constexpr size_t kRetiredBlobs = 4;         // retired device blobs a context keeps

struct PrimRef {
    uint8_t kind;  // 0 sphere, 1 triangle
    uint32_t idx;  // index in the caller's array
};

// min_by / max_by with partial_cmp().unwrap_or(Equal) (mesh.rs:46-95): min_by returns the first
// argument unless first > second; max_by returns the second unless first > second.
inline float ref_min(float x, float y) { return (x > y) ? y : x; }
inline float ref_max(float x, float y) { return (x > y) ? x : y; }
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
inline bool finite3(const float* v) { return std::isfinite(v[0]) && std::isfinite(v[1]) && std::isfinite(v[2]); }

// World order + bounds (Sphere::aabb sphere.rs:65-72, Triangle::aabb mesh.rs:46-95).
int world_and_boxes(const rt_sphere* spheres, uint32_t n_spheres, const rt_triangle* triangles, uint32_t n_triangles,
                    const uint32_t* world_index, std::vector<PrimRef>* world_out, std::vector<Box>* boxes_out,
                    std::string* err) {
    auto fail = [err](int rc, const char* fmt, uint32_t v) {
        char buf[256];
        snprintf(buf, sizeof buf, fmt, v);
        *err = buf;
        return rc;
    };
    const uint32_t n = n_spheres + n_triangles;
    std::vector<PrimRef>& world = *world_out;
    world.assign(n, PrimRef{0, 0});
    {
        std::vector<uint8_t> seen(n, 0);
        for (uint32_t i = 0; i < n; i++) {
            const uint32_t pos = world_index ? world_index[i] : i;
            if (pos >= n || seen[pos]) return fail(RT_ERR_INVALID_ARG, "world_index is not a permutation of 0..%u", n - 1);
            seen[pos] = 1;
            world[pos] = i < n_spheres ? PrimRef{0, i} : PrimRef{1, i - n_spheres};
        }
    }
    std::vector<Box>& boxes = *boxes_out;
    boxes.resize(n);
    for (uint32_t w = 0; w < n; w++) {
        Box& b = boxes[w];
        if (world[w].kind == 0) {
            const rt_sphere& s = spheres[world[w].idx];
            if (!finite3(s.center) || !std::isfinite(s.radius))
                return fail(RT_ERR_BVH, "sphere %u has non-finite geometry", world[w].idx);
            for (int a = 0; a < 3; a++) {
                b.min[a] = s.center[a] - s.radius;
                b.max[a] = s.center[a] + s.radius;
            }
        } else {
            const rt_triangle& t = triangles[world[w].idx];
            if (!finite3(t.a) || !finite3(t.b) || !finite3(t.c))
                return fail(RT_ERR_BVH, "triangle %u has non-finite geometry", world[w].idx);
            for (int a = 0; a < 3; a++) {
                b.min[a] = ref_min(ref_min(t.a[a], t.c[a]), t.b[a]);
                b.max[a] = ref_max(ref_max(t.a[a], t.c[a]), t.b[a]);
            }
        }
        if (!finite3(b.min) || !finite3(b.max))  // centre +- radius overflowed: the reference's bucket index would panic
            return fail(RT_ERR_BVH, "primitive at world position %u has non-finite bounds", w);
    }
    return RT_OK;
}

// The scene blob, the one statement of its layout: the shared-memory image first (sph | tri | lnode, contiguous, each a
// multiple of 16 bytes, scene_image_bytes long), then 256-byte aligned sections.  rt_scene_create uploads everything
// before sync_bytes; the reference tables and the flag that announces them follow.
struct BlobLayout {
    size_t sph, tri, lnode, sph2, mat, emis, box, big, rank, up, refbox, flag;
    size_t sync_bytes, blob_bytes;
};
BlobLayout blob_layout(uint32_t n_spheres, uint32_t n_triangles, uint32_t lni) {
    const size_t n = (size_t)n_spheres + n_triangles, ni_ref = std::max<size_t>(n - 1, 1);
    BlobLayout L;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        const size_t o = off;
        off = align_up(off + bytes, 256);
        return o;
    };
    L.sph = 0;
    L.tri = L.sph + (size_t)n_spheres * 16;
    L.lnode = L.tri + (size_t)n_triangles * 64;
    off = align_up(scene_image_bytes(n_spheres, n_triangles, lni, true), 256);
    L.sph2 = take((size_t)((n_spheres + 7u) & ~7u) * 16);
    L.mat = take(n * 16);
    L.emis = take(n * 4);
    L.box = take(n * 32);
    L.big = take((size_t)MAX_BIG * 4);
    L.sync_bytes = off;
    L.rank = take(n * 4);
    L.up = take((n + ni_ref) * 4);
    L.refbox = take(ni_ref * 64);
    L.flag = take(4);
    L.blob_bytes = off;
    return L;
}

// The split layout: the primitives whose box is a large share of the scene's (at most MAX_BIG, the largest) are kept
// out of the traversal tree and tested first; the tree covers the rest.
struct Split {
    std::vector<uint32_t> big_world;   // world positions of the primitives kept out of the tree, ascending
    std::vector<uint32_t> rest_world;  // world positions of the primitives the tree covers
    std::vector<Box> rest_store;       // their boxes, when some primitives are big
    // boxes of the primitives the tree covers (without big primitives, `boxes` itself: no copy)
    const std::vector<Box>& rest(const std::vector<Box>& boxes) const { return big_world.empty() ? boxes : rest_store; }
};
void split_big(const std::vector<Box>& boxes, Split* s) {
    const uint32_t n = (uint32_t)boxes.size();
    if (n > 1) {
        auto area_of = [](const Box& b) {
            const double sx = (double)b.max[0] - b.min[0], sy = (double)b.max[1] - b.min[1], sz = (double)b.max[2] - b.min[2];
            return 2.0 * (sx * sy + sx * sz + sy * sz);
        };
        Box all = boxes[0];
        for (uint32_t w = 1; w < n; w++)
            for (int a = 0; a < 3; a++) {
                all.min[a] = fminf(all.min[a], boxes[w].min[a]);
                all.max[a] = fmaxf(all.max[a], boxes[w].max[a]);
            }
        const double thresh = area_of(all) * (1.0 / 16.0);
        std::vector<std::pair<double, uint32_t>> cand;
        for (uint32_t w = 0; w < n; w++) {
            const double a = area_of(boxes[w]);
            if (a > thresh && a > 0.0) cand.push_back({-a, w});
        }
        std::sort(cand.begin(), cand.end());
        if (cand.size() > (size_t)MAX_BIG) cand.resize(MAX_BIG);
        for (auto& c : cand) s->big_world.push_back(c.second);
        std::sort(s->big_world.begin(), s->big_world.end());
    }
    size_t bi = 0;
    s->rest_world.reserve(n - s->big_world.size());
    for (uint32_t w = 0; w < n; w++) {
        if (bi < s->big_world.size() && s->big_world[bi] == w) bi++;
        else s->rest_world.push_back(w);
    }
    if (!s->big_world.empty()) {
        s->rest_store.reserve(s->rest_world.size());
        for (uint32_t w : s->rest_world) s->rest_store.push_back(boxes[w]);
    }
}

// The SAH tree over `rest` (at least two primitives), its leaf codes remapped to world positions.
int host_traversal_tree(rt_ctx* ctx, const std::vector<Box>& rest, const std::vector<uint32_t>& rest_world, HostBVH* t) {
    if (!build_bvh_sah(rest, t)) return set_err(ctx, RT_ERR_BVH, "traversal tree build failed");
    auto remap = [&](int32_t c) { return c >= 0 ? c : ~(int32_t)rest_world[(uint32_t)~c]; };
    for (auto& nd : t->inner) {
        nd.left = remap(nd.left);
        nd.right = remap(nd.right);
    }
    t->root = remap(t->root);
    if (t->depth > (uint32_t)MAX_STACK)
        return set_err(ctx, RT_ERR_UNSUPPORTED, "traversal tree depth %u exceeds the traversal stack (%d)", t->depth, MAX_STACK);
    return RT_OK;
}

// Primitive ids: spheres [0, ns), triangles [ns, n).  In the DFS leaf order of the host-built traversal tree T when
// there is one (neighbours in space are neighbours in memory: the per-hit material / box / rank reads of the lanes of a
// warp share cache lines), else in world order.
void assign_pids(const std::vector<PrimRef>& world, uint32_t n_spheres, const HostBVH* T, std::vector<uint32_t>* pid_of_world) {
    const uint32_t n = (uint32_t)world.size();
    std::vector<uint32_t>& pid = *pid_of_world;
    pid.assign(n, 0xffffffffu);
    uint32_t next_s = 0, next_t = n_spheres;
    auto give = [&](uint32_t w) {
        if (pid[w] == 0xffffffffu) pid[w] = world[w].kind == 0 ? next_s++ : next_t++;
    };
    if (T) {
        std::vector<int32_t> todo;
        todo.push_back(T->root);
        while (!todo.empty()) {
            const int32_t c = todo.back();
            todo.pop_back();
            if (c < 0) {
                give((uint32_t)~c);
            } else {
                todo.push_back(T->inner[(size_t)c].right);
                todo.push_back(T->inner[(size_t)c].left);
            }
        }
    }
    for (uint32_t w = 0; w < n; w++) give(w);
}

// The late tables, in pid indexing, from the reference tree.
struct AuxTables {
    std::vector<uint32_t> rank, up;
    std::vector<float> refbox;  // [ni][side][min xyz . | max xyz .]
};
// Builds the reference tree and its tables, and sets aux's n_nodes, depth and rank_by_world.  false (message in *err):
// the reference's build would panic or never terminate.
bool build_ref_tables(const std::vector<Box>& boxes, const std::vector<uint32_t>& pid_of_world, rt_aux* aux, AuxTables* t,
                      std::string* err) {
    HostBVH bvh;
    if (!build_bvh(boxes, &bvh, err)) return false;
    const uint32_t n = (uint32_t)pid_of_world.size(), ni = (uint32_t)bvh.inner.size();
    t->rank.assign(n, 0);
    t->up.assign((size_t)n + std::max(ni, 1u), UP_ROOT);
    t->refbox.assign((size_t)std::max(ni, 1u) * 16, 0.0f);
    aux->rank_by_world.assign(n, 0);
    for (uint32_t r = 0; r < n; r++) {
        const uint32_t w = bvh.leaf_order[r];
        aux->rank_by_world[w] = r;
        t->rank[pid_of_world[w]] = r;
    }
    for (uint32_t i = 0; i < ni; i++) {
        const HostNode& hn = bvh.inner[i];
        for (uint32_t side = 0; side < 2; side++) {
            const int32_t code = side ? hn.right : hn.left;
            const Box& b = side ? hn.box_r : hn.box_l;
            float* o = t->refbox.data() + ((size_t)2 * i + side) * 8;
            for (int a = 0; a < 3; a++) {
                o[a] = b.min[a];
                o[4 + a] = b.max[a];
            }
            const uint32_t slot = (i << 1) | side;
            if (code >= 0) t->up[(size_t)n + (uint32_t)code] = slot;
            else t->up[pid_of_world[(uint32_t)~code]] = slot;
        }
    }
    aux->n_nodes = bvh.node_count;
    aux->depth = bvh.depth;
    return true;
}

// The retired-blob pool: the smallest retired device blob that fits, else a new allocation in power-of-two size classes
// (>= 256 KB).  Retired blobs fit the next scene of a similar size, and the driver sees few distinct allocation sizes.
cudaError_t take_blob(rt_ctx* ctx, size_t bytes, uint8_t** p, size_t* cap) {
    size_t pick = ctx->retired.size();
    for (size_t i = 0; i < ctx->retired.size(); i++)
        if (ctx->retired[i].cap >= bytes && (pick == ctx->retired.size() || ctx->retired[i].cap < ctx->retired[pick].cap)) pick = i;
    if (pick < ctx->retired.size()) {
        *p = ctx->retired[pick].p;
        *cap = ctx->retired[pick].cap;
        ctx->retired.erase(ctx->retired.begin() + (long)pick);
        return cudaSuccess;
    }
    *cap = (size_t)1 << 18;
    while (*cap < bytes) *cap <<= 1;
    return cudaMalloc(p, *cap);
}
// ctx may be null (its blobs are then freed)
void retire_blob(rt_ctx* ctx, uint8_t* p, size_t cap) {
    if (ctx && ctx->retired.size() < kRetiredBlobs) ctx->retired.push_back({p, cap});
    else cudaFree(p);
}

// The pinned staging buffer holds at least `bytes` (power-of-two size classes, >= 1 MB).
cudaError_t reserve_stage(rt_ctx* ctx, size_t bytes) {
    if (ctx->h_stage_bytes >= bytes) return cudaSuccess;
    if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
    ctx->h_stage = nullptr;
    ctx->h_stage_bytes = 0;
    size_t cap = (size_t)1 << 20;
    while (cap < bytes) cap <<= 1;
    const cudaError_t e = cudaMallocHost(&ctx->h_stage, cap);
    if (e == cudaSuccess) ctx->h_stage_bytes = cap;
    return e;
}

// The reference tree on a thread of its own: its tables go to the blob on aux_stream, then the flag the kernels poll
// (stream order: the tables are there before it).  The flag is lowered first, before anybody can look (device blobs are
// reused).
int start_ref_builder(rt_ctx* ctx, rt_scene* sc, const BlobLayout& L, int delay_ms) {
    CK(ctx, cudaMemsetAsync(sc->d_blob + L.flag, 0, 4, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    sc->aux->worker = std::thread([a = sc->aux.get(), c = ctx, dst = sc->d_blob, L, delay_ms] {
        try {
            if (delay_ms > 0) std::this_thread::sleep_for(std::chrono::milliseconds(delay_ms));
            AuxTables t;
            if (!build_ref_tables(a->boxes, a->pid_of_world, a, &t, &a->err)) {
                a->state.store(-1, std::memory_order_release);
                return;
            }
            static const int one = 1;
            cudaError_t e = cudaSetDevice(c->device);
            if (e == cudaSuccess) e = cudaMemcpyAsync(dst + L.rank, t.rank.data(), t.rank.size() * 4, cudaMemcpyHostToDevice, c->aux_stream);
            if (e == cudaSuccess) e = cudaMemcpyAsync(dst + L.up, t.up.data(), t.up.size() * 4, cudaMemcpyHostToDevice, c->aux_stream);
            if (e == cudaSuccess) e = cudaMemcpyAsync(dst + L.refbox, t.refbox.data(), t.refbox.size() * 4, cudaMemcpyHostToDevice, c->aux_stream);
            if (e == cudaSuccess) e = cudaMemcpyAsync(dst + L.flag, &one, 4, cudaMemcpyHostToDevice, c->aux_stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(c->aux_stream);
            if (e != cudaSuccess) {
                a->err = std::string("upload of the tie-break tables failed: ") + cudaGetErrorString(e);
                a->state.store(-1, std::memory_order_release);
                return;
            }
            a->state.store(1, std::memory_order_release);
        } catch (const std::exception& ex) {
            a->err = ex.what();
            a->state.store(-1, std::memory_order_release);
        } catch (...) {
            a->err = "unknown exception in the builder thread";
            a->state.store(-1, std::memory_order_release);
        }
    });
    return RT_OK;
}

// Geometry, materials, boxes, sphere pairs and big-primitive codes into the staging image h, in pid order.
void fill_image(uint8_t* h, const BlobLayout& L, const std::vector<PrimRef>& world, const rt_sphere* spheres,
                const rt_triangle* triangles, uint32_t n_spheres, const std::vector<Box>& boxes,
                const std::vector<uint32_t>& pid_of_world, const std::vector<uint32_t>& big_world) {
    const uint32_t n = (uint32_t)world.size();
    float* h_sph = (float*)(h + L.sph);
    float* h_tri = (float*)(h + L.tri);
    float* h_mat = (float*)(h + L.mat);
    float* h_em = (float*)(h + L.emis);
    float* h_box = (float*)(h + L.box);
    for (uint32_t w = 0; w < n; w++) {
        const uint32_t pid = pid_of_world[w];
        float* bx = h_box + 8 * (size_t)pid;
        for (int a = 0; a < 3; a++) {
            bx[a] = boxes[w].min[a];
            bx[4 + a] = boxes[w].max[a];
        }
        bx[3] = bx[7] = 0.0f;
        float* m = h_mat + 4 * (size_t)pid;
        if (world[w].kind == 0) {
            const rt_sphere& s = spheres[world[w].idx];
            float* g = h_sph + 4 * (size_t)pid;
            g[0] = s.center[0]; g[1] = s.center[1]; g[2] = s.center[2];
            g[3] = s.radius * s.radius;  // radius.powi(2)
            m[0] = s.albedo[0]; m[1] = s.albedo[1]; m[2] = s.albedo[2]; m[3] = s.roughness;
            h_em[pid] = s.emission;
        } else {
            const rt_triangle& t = triangles[world[w].idx];
            float* g = h_tri + 16 * (size_t)(pid - n_spheres);
            float ab[3], ac[3], amb[3], amc[3];
            for (int a = 0; a < 3; a++) {
                ab[a] = t.b[a] - t.a[a];   // a_to_b (mesh.rs:111)
                ac[a] = t.c[a] - t.a[a];   // a_to_c
                amb[a] = t.a[a] - t.b[a];  // normal_at: (a-b).cross(a-c) (mesh.rs:164)
                amc[a] = t.a[a] - t.c[a];
            }
            // glam cross + normalize_or_zero, single f32 ops (host built with -ffp-contract=off)
            const float cr[3] = {amb[1] * amc[2] - amc[1] * amb[2], amb[2] * amc[0] - amc[2] * amb[0],
                                 amb[0] * amc[1] - amc[0] * amb[1]};
            const float dd = (cr[0] * cr[0] + cr[1] * cr[1]) + cr[2] * cr[2];
            const float rcp = 1.0f / sqrtf(dd);
            float nrm[3] = {0.0f, 0.0f, 0.0f};
            if (std::isfinite(rcp) && rcp > 0.0f) {
                nrm[0] = cr[0] * rcp; nrm[1] = cr[1] * rcp; nrm[2] = cr[2] * rcp;
            }
            for (int a = 0; a < 3; a++) {
                g[0 + a] = t.a[a];
                g[4 + a] = ab[a];
                g[8 + a] = ac[a];
                g[12 + a] = nrm[a];
            }
            g[3] = g[7] = g[11] = g[15] = 0.0f;
            m[0] = t.albedo[0]; m[1] = t.albedo[1]; m[2] = t.albedo[2]; m[3] = t.roughness;
            h_em[pid] = t.emission;
        }
    }
    {   // pair j = spheres 2j, 2j+1: (-c0.x, -c1.x, -c0.y, -c1.y) | (-c0.z, -c1.z, r0^2, r1^2); pads can never pass
        const uint32_t ns8 = (n_spheres + 7u) & ~7u;
        float* h2 = (float*)(h + L.sph2);
        for (uint32_t j = 0; j < ns8 / 2; j++)
            for (uint32_t k = 0; k < 2; k++) {
                const uint32_t pid = 2 * j + k;
                const bool real = pid < n_spheres;
                const float* g = h_sph + 4 * (size_t)pid;
                h2[8 * (size_t)j + 0 + k] = real ? -g[0] : 0.0f;
                h2[8 * (size_t)j + 2 + k] = real ? -g[1] : 0.0f;
                h2[8 * (size_t)j + 4 + k] = real ? -g[2] : 0.0f;
                h2[8 * (size_t)j + 6 + k] = real ? g[3] : -std::numeric_limits<float>::infinity();
            }
    }
    for (size_t i = 0; i < (size_t)MAX_BIG; i++)
        ((int32_t*)(h + L.big))[i] = i < big_world.size() ? ~(int32_t)(pid_of_world[big_world[i]] << 5) : 0;
}

// Traversal-tree records of the host tree T into ln (DFS pre-order numbering, left subtree first); returns the root
// code.  Without T: a single primitive in the tree (rest_world) is the root leaf itself; otherwise the tree is empty or
// built on the device (its root is node 0) and the root code is 0.
int32_t emit_nodes(uint8_t* ln, const HostBVH* T, const std::vector<uint32_t>& rest_world,
                   const std::vector<uint32_t>& pid_of_world) {
    auto leaf_code = [&](int32_t world_code) { return ~(int32_t)(pid_of_world[(uint32_t)~world_code] << 5); };
    if (!T) return rest_world.size() == 1 ? leaf_code(~(int32_t)rest_world[0]) : 0;
    int32_t* lc = (int32_t*)ln;  // the same records: words 12, 13 are the child codes
    struct Item { int32_t code; uint32_t parent; int side; };
    std::vector<Item> todo;
    uint32_t next = 0;
    int32_t lroot = 0;
    todo.push_back(Item{T->root, 0, -1});
    while (!todo.empty()) {
        const Item it = todo.back();
        todo.pop_back();
        const uint32_t me = next++;
        if (it.side < 0) lroot = (int32_t)me * NODE_BYTES;
        else lc[NODE_WORDS * (size_t)it.parent + 12 + it.side] = (int32_t)me * NODE_BYTES;
        const HostNode& hn = T->inner[(size_t)it.code];
        float lcn[3], lhh[3], rcn[3], rhh[3];
        centre_half(hn.box_l.min, hn.box_l.max, lcn, lhh);
        centre_half(hn.box_r.min, hn.box_r.max, rcn, rhh);
        node_box_words(lcn, lhh, rcn, rhh, (float*)ln + NODE_WORDS * (size_t)me);
        for (int k = 14; k < NODE_WORDS; k++) lc[NODE_WORDS * (size_t)me + k] = 0;
        const int32_t kids[2] = {hn.left, hn.right};
        for (int side = 1; side >= 0; side--) {  // push right first so the left subtree is numbered first
            if (kids[side] < 0) {
                lc[NODE_WORDS * (size_t)me + 12 + side] = leaf_code(kids[side]);
            } else {
                todo.push_back(Item{kids[side], me, side});
            }
        }
    }
    return lroot;
}

// The staging image's first stage_bytes to the device blob, then, with device_tree, the LBVH over `rest` into the
// node-record region (which the staging image leaves out).  The staging buffer is free again on return; on an error the
// caller still owns the blob.
int upload(rt_ctx* ctx, rt_scene* sc, const uint8_t* h, const BlobLayout& L, size_t stage_bytes, bool device_tree,
           const std::vector<Box>& rest, const std::vector<uint32_t>& rest_world, const std::vector<uint32_t>& pid_of_world) {
    cudaError_t e;
    if (device_tree) {  // 4 MB of node records at 65,536 primitives are not copied
        e = cudaMemcpyAsync(sc->d_blob, h, L.lnode, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(sc->d_blob + L.sph2, h + L.sph2, stage_bytes - L.sph2, cudaMemcpyHostToDevice, ctx->stream);
    } else {
        e = cudaMemcpyAsync(sc->d_blob, h, stage_bytes, cudaMemcpyHostToDevice, ctx->stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);  // the staging buffer is reused by the next scene
    if (e != cudaSuccess) return set_err(ctx, RT_ERR_CUDA, "scene upload failed: %s", cudaGetErrorString(e));
    if (!device_tree) return RT_OK;
    std::vector<uint32_t> dev_pid(rest.size());
    for (size_t i = 0; i < rest.size(); i++) dev_pid[i] = pid_of_world[rest_world[i]];
    uint32_t depth = 0;
    e = build_lbvh_device(&ctx->dbuild, rest.data(), dev_pid.data(), (uint32_t)dev_pid.size(),
                          (float4*)(sc->d_blob + L.lnode), &depth, ctx->stream);
    if (e != cudaSuccess) return set_err(ctx, RT_ERR_CUDA, "device BVH build failed: %s", cudaGetErrorString(e));
    if (depth > (uint32_t)MAX_STACK)
        return set_err(ctx, RT_ERR_UNSUPPORTED, "device-built tree depth %u exceeds the traversal stack (%d)", depth, MAX_STACK);
    return RT_OK;
}

DevScene make_dev_scene(const uint8_t* blob, const BlobLayout& L, uint32_t n_spheres, uint32_t n_triangles, uint32_t lni,
                        int32_t lroot, bool ltree, uint32_t nbig) {
    DevScene d{};
    d.sph = (const float4*)(blob + L.sph);
    d.tri = (const float4*)(blob + L.tri);
    d.lnode = (const float4*)(blob + L.lnode);
    d.sph2 = (const float4*)(blob + L.sph2);
    d.lni = lni;
    d.lroot = lroot;
    d.ltree = ltree ? 1 : 0;
    d.nbig = nbig;
    d.big_code = (const int*)(blob + L.big);
    d.mat = (const float4*)(blob + L.mat);
    d.emis = (const float*)(blob + L.emis);
    d.rank = (const uint32_t*)(blob + L.rank);
    d.leaf_box = (const float4*)(blob + L.box);
    d.ref_up = (const uint32_t*)(blob + L.up);
    d.ref_box = (const float4*)(blob + L.refbox);
    d.aux_ready = 0;
    d.aux_flag = (const int*)(blob + L.flag);
    d.ns = n_spheres;
    d.nt = n_triangles;
    d.ni = n_spheres + n_triangles - 1;
    return d;
}

}  // namespace

namespace rtb {

int scene_settle(rt_ctx* ctx, const rt_scene* scene) {
    rt_aux* aux = scene->aux.get();
    if (!aux) return RT_OK;
    if (aux->worker.joinable()) aux->worker.join();
    if (aux->state.load(std::memory_order_acquire) < 0) return set_err(ctx, RT_ERR_BVH, "BVH build failed: %s", aux->err.c_str());
    return RT_OK;
}

DevScene scene_view(const rt_scene* scene) {
    DevScene d = scene->dev;
    d.aux_ready = (!scene->aux || scene->aux->state.load(std::memory_order_acquire) == 1) ? 1 : 0;
    return d;
}

}  // namespace rtb

extern "C" {

int rt_bvh_build_host(const rt_sphere* spheres, uint32_t n_spheres, const rt_triangle* triangles, uint32_t n_triangles,
                      const uint32_t* world_index, uint32_t* rank_out, uint32_t* n_nodes, uint32_t* depth) {
    RT_GUARD_BEGIN
    const uint64_t n64 = (uint64_t)n_spheres + n_triangles;
    if (n64 == 0) return RT_ERR_EMPTY_SCENE;
    if (n64 > MAX_PRIMS) return RT_ERR_UNSUPPORTED;
    if ((n_spheres && !spheres) || (n_triangles && !triangles)) return RT_ERR_INVALID_ARG;
    std::vector<PrimRef> world;
    std::vector<Box> boxes;
    std::string err;
    int rc = world_and_boxes(spheres, n_spheres, triangles, n_triangles, world_index, &world, &boxes, &err);
    HostBVH bvh;
    if (rc == RT_OK && !build_bvh(boxes, &bvh, &err)) {
        err = "BVH build failed: " + err;
        rc = RT_ERR_BVH;
    }
    if (rc) return set_err(nullptr, rc, "%s", err.c_str());
    if (rank_out)
        for (uint32_t r = 0; r < (uint32_t)n64; r++) rank_out[bvh.leaf_order[r]] = r;
    if (n_nodes) *n_nodes = bvh.node_count;
    if (depth) *depth = bvh.depth;
    return RT_OK;
    RT_GUARD_END(nullptr)
}

int rt_scene_create(rt_ctx* ctx, const rt_sphere* spheres, uint32_t n_spheres, const rt_triangle* triangles,
                    uint32_t n_triangles, const uint32_t* world_index, rt_scene** out) {
    if (!ctx) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    if (!out) return set_err(ctx, RT_ERR_INVALID_ARG, "rt_scene_create: out is NULL");
    *out = nullptr;
    const uint64_t n64 = (uint64_t)n_spheres + n_triangles;
    if (n64 == 0)
        return set_err(ctx, RT_ERR_EMPTY_SCENE,
                       "empty world: the reference's BVHNode::build never terminates on zero shapes");
    // inner codes are the byte offset of a 64-byte node record and must stay positive (n - 1 records: 25 bits of nodes)
    if (n64 > MAX_PRIMS || (n64 - 1) * (uint64_t)NODE_BYTES > 0x7fffffffull)
        return set_err(ctx, RT_ERR_UNSUPPORTED, "too many primitives (%llu; this build addresses %llu)", (unsigned long long)n64,
                       (unsigned long long)(0x7fffffffull / NODE_BYTES + 1));
    if ((n_spheres && !spheres) || (n_triangles && !triangles))
        return set_err(ctx, RT_ERR_INVALID_ARG, "rt_scene_create: NULL primitive array");
    const uint32_t n = (uint32_t)n64;
    const TestHooks& hooks = test_hooks();

    static std::atomic<uint64_t> next_serial{1};
    std::unique_ptr<rt_scene> sc(new rt_scene());
    sc->ctx = ctx;
    sc->serial = next_serial++;
    sc->n = n;
    sc->aux.reset(new rt_aux());
    rt_aux* aux = sc->aux.get();
    std::vector<PrimRef> world;
    std::string werr;
    const int wrc = world_and_boxes(spheres, n_spheres, triangles, n_triangles, world_index, &world, &aux->boxes, &werr);
    if (wrc) return set_err(ctx, wrc, "%s", werr.c_str());
    const std::vector<Box>& boxes = aux->boxes;  // shared, read-only from here on

    // which tree will be traversed, and who builds it
    Split split;
    split_big(boxes, &split);
    const std::vector<Box>& rest = split.rest(boxes);
    const bool device_tree = rest.size() >= 2 &&
                             (hooks.build_mode == 2 || (hooks.build_mode == 1 && rest.size() >= kDeviceBuildMin));
    HostBVH sah;
    const HostBVH* T = nullptr;  // the host-built traversal tree (leaf codes: world positions)
    if (!device_tree && rest.size() >= 2) {
        const int rc = host_traversal_tree(ctx, rest, split.rest_world, &sah);
        if (rc) return rc;
        T = &sah;
    }
    assign_pids(world, n_spheres, T, &aux->pid_of_world);
    const std::vector<uint32_t>& pid_of_world = aux->pid_of_world;

    // the reference tree: inline for small scenes, else on the builder thread below
    const bool ref_sync = n < kRefSyncBelow;
    AuxTables ref_tables;
    if (ref_sync) {
        std::string berr;
        if (!build_ref_tables(boxes, pid_of_world, aux, &ref_tables, &berr))
            return set_err(ctx, RT_ERR_BVH, "BVH build failed: %s", berr.c_str());
    }

    const uint32_t lni = device_tree ? (uint32_t)rest.size() - 1 : T ? (uint32_t)T->inner.size() : 0;
    const BlobLayout L = blob_layout(n_spheres, n_triangles, lni);
    sc->blob_bytes = L.blob_bytes;
    const size_t stage_bytes = ref_sync ? L.blob_bytes : L.sync_bytes;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, reserve_stage(ctx, stage_bytes));
    CK(ctx, take_blob(ctx, L.blob_bytes, &sc->d_blob, &sc->blob_cap));
    // the builder thread starts now, with pid_of_world final: it overlaps the fill and the upload
    if (!ref_sync) {
        const int rc = start_ref_builder(ctx, sc.get(), L, hooks.aux_delay_ms);
        if (rc) return rc;
    }

    uint8_t* const h = ctx->h_stage;
    fill_image(h, L, world, spheres, triangles, n_spheres, boxes, pid_of_world, split.big_world);
    const int32_t lroot = emit_nodes(h + L.lnode, T, split.rest_world, pid_of_world);
    if (ref_sync) {  // the whole blob is uploaded by this call: the tables and the raised flag go with it
        memcpy(h + L.rank, ref_tables.rank.data(), ref_tables.rank.size() * 4);
        memcpy(h + L.up, ref_tables.up.data(), ref_tables.up.size() * 4);
        memcpy(h + L.refbox, ref_tables.refbox.data(), ref_tables.refbox.size() * 4);
        *(int32_t*)(h + L.flag) = 1;
    }
    const int rc = upload(ctx, sc.get(), h, L, stage_bytes, device_tree, rest, split.rest_world, pid_of_world);
    if (rc) {  // the builder thread may still write to the blob
        if (aux->worker.joinable()) aux->worker.join();
        retire_blob(ctx, sc->d_blob, sc->blob_cap);
        return rc;
    }
    if (ref_sync) aux->state.store(1, std::memory_order_release);

    sc->dev = make_dev_scene(sc->d_blob, L, n_spheres, n_triangles, lni, lroot, !rest.empty(),
                             (uint32_t)split.big_world.size());
    *out = sc.release();
    return RT_OK;
    RT_GUARD_END(ctx)
}

void rt_scene_destroy(rt_ctx* ctx, rt_scene* scene) {
    if (!scene) return;
    if (scene->aux && scene->aux->worker.joinable()) scene->aux->worker.join();
    if (ctx) {
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        cudaStreamSynchronize(ctx->copy_stream);
    }
    if (scene->d_blob) retire_blob(ctx, scene->d_blob, scene->blob_cap);
    delete scene;
}

int rt_scene_wait_ready(rt_ctx* ctx, const rt_scene* scene) {
    if (!ctx || !scene) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    return scene_settle(ctx, scene);
    RT_GUARD_END(ctx)
}

int rt_scene_info(const rt_scene* scene, uint32_t* n_prims, uint32_t* n_nodes, uint32_t* depth, uint32_t* rank_out) {
    if (!scene) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    const int rc = scene_settle(scene->ctx, scene);
    if (rc) return rc;
    if (n_prims) *n_prims = scene->n;
    if (n_nodes) *n_nodes = scene->aux->n_nodes;
    if (depth) *depth = scene->aux->depth;
    if (rank_out) memcpy(rank_out, scene->aux->rank_by_world.data(), scene->n * sizeof(uint32_t));
    return RT_OK;
    RT_GUARD_END(scene->ctx)
}

size_t rt_scene_device_bytes(const rt_scene* scene) { return scene ? scene->blob_bytes : 0; }

}  // extern "C"
