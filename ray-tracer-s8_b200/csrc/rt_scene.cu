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
#include <functional>
#include <limits>

#include "rt_ctx.h"

using namespace rtb;

namespace {

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

// centre / half-extent form of a box (FILTER domain): t = (c - o)*inv -/+ h*|inv|.  h is padded for the rounding of
// the c- and h-terms (<= 2^-24 * (2|c| + h) per axis); the o-term is covered per ray by the kernels.
void centre_half_of(const Box& b, float c[3], float h[3]) {
    double m = 0.0;
    for (int a = 0; a < 3; a++) m = std::fmax(m, std::fmax(std::fabs((double)b.min[a]), std::fabs((double)b.max[a])));
    for (int a = 0; a < 3; a++) {
        const double cc = 0.5 * ((double)b.min[a] + (double)b.max[a]);
        const double hh = 0.5 * ((double)b.max[a] - (double)b.min[a]);
        c[a] = (float)cc;
        h[a] = (float)(hh * (1.0 + 4e-6) + 2e-6 * m + 1e-30);
    }
}

// World order + bounds (Sphere::aabb sphere.rs:65-72, Triangle::aabb mesh.rs:46-95).
int world_and_boxes(const rt_sphere* spheres, uint32_t n_spheres, const rt_triangle* triangles, uint32_t n_triangles,
                    const uint32_t* world_index, std::vector<PrimRef>* world_out, std::vector<Box>* boxes_out,
                    std::string* err) {
    char buf[256];
    const uint32_t n = n_spheres + n_triangles;
    std::vector<PrimRef>& world = *world_out;
    world.assign(n, PrimRef{0, 0});
    {
        std::vector<uint8_t> seen(n, 0);
        for (uint32_t i = 0; i < n; i++) {
            const uint32_t pos = world_index ? world_index[i] : i;
            if (pos >= n || seen[pos]) {
                snprintf(buf, sizeof buf, "world_index is not a permutation of 0..%u", n - 1);
                *err = buf;
                return RT_ERR_INVALID_ARG;
            }
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
            if (!finite3(s.center) || !std::isfinite(s.radius)) {
                snprintf(buf, sizeof buf, "sphere %u has non-finite geometry", world[w].idx);
                *err = buf;
                return RT_ERR_BVH;
            }
            for (int a = 0; a < 3; a++) {
                b.min[a] = s.center[a] - s.radius;
                b.max[a] = s.center[a] + s.radius;
            }
        } else {
            const rt_triangle& t = triangles[world[w].idx];
            if (!finite3(t.a) || !finite3(t.b) || !finite3(t.c)) {
                snprintf(buf, sizeof buf, "triangle %u has non-finite geometry", world[w].idx);
                *err = buf;
                return RT_ERR_BVH;
            }
            for (int a = 0; a < 3; a++) {
                b.min[a] = ref_min(ref_min(t.a[a], t.c[a]), t.b[a]);
                b.max[a] = ref_max(ref_max(t.a[a], t.c[a]), t.b[a]);
            }
        }
        if (!finite3(b.min) || !finite3(b.max)) {  // centre +- radius overflowed: the reference's bucket index would panic
            snprintf(buf, sizeof buf, "primitive at world position %u has non-finite bounds", w);
            *err = buf;
            return RT_ERR_BVH;
        }
    }
    return RT_OK;
}

// The late tables, in pid indexing, from the reference tree.
struct AuxTables {
    std::vector<uint32_t> rank, up;
    std::vector<float> refbox;  // [ni][side][min xyz . | max xyz .]
};
void tables_from_tree(const HostBVH& bvh, const std::vector<uint32_t>& pid_of_world, AuxTables* t,
                      std::vector<uint32_t>* rank_by_world) {
    const uint32_t n = (uint32_t)pid_of_world.size(), ni = (uint32_t)bvh.inner.size();
    t->rank.assign(n, 0);
    t->up.assign((size_t)n + std::max(ni, 1u), UP_ROOT);
    t->refbox.assign((size_t)std::max(ni, 1u) * 16, 0.0f);
    rank_by_world->assign(n, 0);
    for (uint32_t r = 0; r < n; r++) {
        const uint32_t w = bvh.leaf_order[r];
        (*rank_by_world)[w] = r;
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
    if (n64 > 0x3ffffffu) return RT_ERR_UNSUPPORTED;  // leaf codes hold a 26-bit primitive id
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
    // leaf codes are ~(pid << 5) in 32 bits (26-bit ids); inner codes are the byte offset of a 64-byte node record and
    // must stay positive (n - 1 records: 25 bits of nodes)
    if (n64 > 0x3ffffffu || (n64 - 1) * (uint64_t)NODE_BYTES > 0x7fffffffull)
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
    {
        std::string werr;
        const int wrc = world_and_boxes(spheres, n_spheres, triangles, n_triangles, world_index, &world, &aux->boxes, &werr);
        if (wrc) return set_err(ctx, wrc, "%s", werr.c_str());
    }
    const std::vector<Box>& boxes = aux->boxes;  // shared, read-only from here on

    // ---- which tree will be traversed ---------------------------------------------------------------------
    std::vector<uint32_t> big_world;  // split layout: world positions of the primitives kept out of the tree
    std::vector<Box> rest_store;      // boxes and world positions of the primitives the tree covers (without big
    std::vector<uint32_t> rest_world; //   primitives the tree covers `boxes` itself, no copy)
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
        for (auto& c : cand) big_world.push_back(c.second);
        std::sort(big_world.begin(), big_world.end());
    }
    if (big_world.empty()) {
        rest_world.resize(n);
        for (uint32_t w = 0; w < n; w++) rest_world[w] = w;
    } else {
        size_t bi = 0;
        rest_store.reserve(n - big_world.size());
        rest_world.reserve(n - big_world.size());
        for (uint32_t w = 0; w < n; w++) {
            if (bi < big_world.size() && big_world[bi] == w) {
                bi++;
                continue;
            }
            rest_store.push_back(boxes[w]);
            rest_world.push_back(w);
        }
    }
    const std::vector<Box>& rest = big_world.empty() ? boxes : rest_store;
    const bool ltree = !rest.empty();
    constexpr uint32_t kDeviceBuildMin = 8192;
    const bool device_tree = rest.size() >= 2 &&
                             (hooks.build_mode == 2 || (hooks.build_mode == 1 && rest.size() >= kDeviceBuildMin));

    // ---- the reference-topology tree: beside everything else when it is worth a thread -------------------
    const bool ref_sync = n < 256;
    HostBVH ref_bvh;  // synchronous case only
    AuxTables ref_tables;
    if (ref_sync) {
        std::string berr;
        if (!build_bvh(boxes, &ref_bvh, &berr)) return set_err(ctx, RT_ERR_BVH, "BVH build failed: %s", berr.c_str());
        aux->n_nodes = ref_bvh.node_count;
        aux->depth = ref_bvh.depth;
    }

    // ---- host traversal tree ---------------------------------------------------------------------------------
    HostBVH sah;
    const HostBVH* T = nullptr;  // tree to emit as lnode records (leaf codes: world positions)
    if (ltree && !device_tree && rest.size() >= 2) {
        if (!build_bvh_sah(rest, &sah)) return set_err(ctx, RT_ERR_BVH, "traversal tree build failed");
        auto remap = [&](int32_t c) { return c >= 0 ? c : ~(int32_t)rest_world[(uint32_t)~c]; };
        for (auto& nd : sah.inner) {
            nd.left = remap(nd.left);
            nd.right = remap(nd.right);
        }
        sah.root = remap(sah.root);
        T = &sah;
        if (T->depth > (uint32_t)MAX_STACK)
            return set_err(ctx, RT_ERR_UNSUPPORTED, "traversal tree depth %u exceeds the traversal stack (%d)", T->depth, MAX_STACK);
        sc->tree_depth = T->depth;
    }

    // ---- primitive ids: spheres [0, ns), triangles [ns, n).  In the DFS leaf order of the host-built traversal tree
    // when there is one (neighbours in space are neighbours in memory: the per-hit material / box / rank reads of the
    // lanes of a warp share cache lines), else in world order.
    aux->pid_of_world.assign(n, 0xffffffffu);
    {
        uint32_t next_s = 0, next_t = n_spheres;
        auto give = [&](uint32_t w) {
            if (aux->pid_of_world[w] == 0xffffffffu) aux->pid_of_world[w] = world[w].kind == 0 ? next_s++ : next_t++;
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
    const std::vector<uint32_t>& pid_of_world = aux->pid_of_world;
    if (ref_sync) tables_from_tree(ref_bvh, pid_of_world, &ref_tables, &aux->rank_by_world);
    uint32_t lni = 0;
    if (device_tree) lni = (uint32_t)rest.size() - 1;
    else if (T) lni = (uint32_t)T->inner.size();

    // ---- blob layout: the shared-memory image first (contiguous, 16-byte granules), then 256-byte aligned sections
    const uint32_t ni_ref = n - 1;
    const uint32_t ns8 = (n_spheres + 7u) & ~7u;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        const size_t o = off;
        off = align_up(off + bytes, 256);
        return o;
    };
    const size_t o_sph = 0, o_tri = o_sph + (size_t)n_spheres * 16, o_ln = o_tri + (size_t)n_triangles * 64;
    off = align_up(o_ln + (size_t)lni * NODE_BYTES, 256);
    const size_t o_sph2 = take((size_t)ns8 * 16), o_mat = take((size_t)n * 16), o_em = take((size_t)n * 4),
                 o_box = take((size_t)n * 32), o_big = take((size_t)MAX_BIG * 4);
    const size_t sync_bytes = off;  // everything up to here is uploaded by this call
    const size_t o_rank = take((size_t)n * 4), o_up = take(((size_t)n + std::max(ni_ref, 1u)) * 4),
                 o_refbox = take((size_t)std::max(ni_ref, 1u) * 64), o_flag = take(4);
    const size_t blob_bytes = off;
    sc->o_rank = o_rank;
    sc->o_up = o_up;
    sc->o_refbox = o_refbox;
    sc->blob_bytes = blob_bytes;
    const size_t stage_bytes = ref_sync ? blob_bytes : sync_bytes;

    CK(ctx, cudaSetDevice(ctx->device));
    if (ctx->h_stage_bytes < stage_bytes) {
        if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
        ctx->h_stage = nullptr;
        ctx->h_stage_bytes = 0;
        size_t cap = (size_t)1 << 20;
        while (cap < stage_bytes) cap <<= 1;
        CK(ctx, cudaMallocHost(&ctx->h_stage, cap));
        ctx->h_stage_bytes = cap;
    }
    uint8_t* const h = ctx->h_stage;
    {   // smallest retired device blob that fits, else a new allocation in power-of-two size classes (>= 256 KB): retired
        // blobs fit the next scene of a similar size, and the driver sees few distinct allocation sizes
        size_t pick = ctx->retired.size();
        for (size_t i = 0; i < ctx->retired.size(); i++)
            if (ctx->retired[i].cap >= blob_bytes && (pick == ctx->retired.size() || ctx->retired[i].cap < ctx->retired[pick].cap)) pick = i;
        if (pick < ctx->retired.size()) {
            sc->d_blob = ctx->retired[pick].p;
            sc->blob_cap = ctx->retired[pick].cap;
            ctx->retired.erase(ctx->retired.begin() + (long)pick);
        } else {
            size_t cap = (size_t)1 << 18;
            while (cap < blob_bytes) cap <<= 1;
            CK(ctx, cudaMalloc(&sc->d_blob, cap));
            sc->blob_cap = cap;
        }
    }
    auto give_back = [&] {
        if (sc->aux && sc->aux->worker.joinable()) sc->aux->worker.join();
        if (sc->d_blob) ctx->retired.push_back({sc->d_blob, sc->blob_cap});
        sc->d_blob = nullptr;
    };

    // ---- the builder thread starts now: it knows where its tables go ------------------------------------------
    if (!ref_sync) {
        // the flag kernels poll for the tables: down before anybody can look (device blobs are reused)
        CK(ctx, cudaMemsetAsync(sc->d_blob + o_flag, 0, 4, ctx->stream));
        CK(ctx, cudaStreamSynchronize(ctx->stream));
        rt_aux* const a = aux;
        rt_ctx* const c = ctx;
        const size_t dr = o_rank, du = o_up, db = o_refbox, df = o_flag;
        uint8_t* const dst = sc->d_blob;
        const int delay_ms = hooks.aux_delay_ms;
        a->worker = std::thread([a, c, dst, dr, du, db, df, delay_ms] {
            try {
                if (delay_ms > 0) std::this_thread::sleep_for(std::chrono::milliseconds(delay_ms));
                HostBVH bvh;
                AuxTables t;
                std::string berr;
                if (!build_bvh(a->boxes, &bvh, &berr)) {
                    a->err = berr;
                    a->state.store(-1, std::memory_order_release);
                    return;
                }
                tables_from_tree(bvh, a->pid_of_world, &t, &a->rank_by_world);
                a->n_nodes = bvh.node_count;
                a->depth = bvh.depth;
                cudaError_t e = cudaSetDevice(c->device);
                if (e == cudaSuccess) e = cudaMemcpyAsync(dst + dr, t.rank.data(), t.rank.size() * 4, cudaMemcpyHostToDevice, c->aux_stream);
                if (e == cudaSuccess) e = cudaMemcpyAsync(dst + du, t.up.data(), t.up.size() * 4, cudaMemcpyHostToDevice, c->aux_stream);
                if (e == cudaSuccess) e = cudaMemcpyAsync(dst + db, t.refbox.data(), t.refbox.size() * 4, cudaMemcpyHostToDevice, c->aux_stream);
                // ... and then the flag kernels already running poll (stream order: the tables are there before it)
                static const int one = 1;
                if (e == cudaSuccess) e = cudaMemcpyAsync(dst + df, &one, 4, cudaMemcpyHostToDevice, c->aux_stream);
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
    }

    // ---- fill the staging copy ------------------------------------------------------------------------------------
    float* h_sph = (float*)(h + o_sph);
    float* h_tri = (float*)(h + o_tri);
    float* h_mat = (float*)(h + o_mat);
    float* h_em = (float*)(h + o_em);
    float* h_box = (float*)(h + o_box);
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
        float* h2 = (float*)(h + o_sph2);
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
        ((int32_t*)(h + o_big))[i] = i < big_world.size() ? ~(int32_t)(pid_of_world[big_world[i]] << 5) : 0;
    // the flag lives in the late region: inside the staging copy only when the whole blob is uploaded by this call (the
    // asynchronous path zeroes it on the device above and the builder thread raises it)
    if (ref_sync) *(int32_t*)(h + o_flag) = 1;

    // traversal-tree records from the host tree: DFS pre-order numbering, left subtree first
    int32_t lroot = 0;
    auto leaf_code = [&](int32_t world_code) { return ~(int32_t)(pid_of_world[(uint32_t)~world_code] << 5); };
    if (device_tree) {
        lroot = 0;  // nodes 0 .. n-2 are written on the device after the upload; the root is node 0
    } else if (T) {
        float* ln = (float*)(h + o_ln);
        int32_t* lc = (int32_t*)(h + o_ln);  // the same records: words 12, 13 are the child codes
        struct Item { int32_t code; uint32_t parent; int side; };
        std::vector<Item> todo;
        uint32_t next = 0;
        todo.push_back(Item{T->root, 0, -1});
        while (!todo.empty()) {
            const Item it = todo.back();
            todo.pop_back();
            const uint32_t me = next++;
            if (it.side < 0) lroot = (int32_t)me * NODE_BYTES;
            else lc[NODE_WORDS * (size_t)it.parent + 12 + it.side] = (int32_t)me * NODE_BYTES;
            const HostNode& hn = T->inner[(size_t)it.code];
            float lcn[3], lhh[3], rcn[3], rhh[3];
            centre_half_of(hn.box_l, lcn, lhh);
            centre_half_of(hn.box_r, rcn, rhh);
            float* pa = ln + NODE_WORDS * (size_t)me;
            node_box_words(lcn, lhh, rcn, rhh, pa);
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
    } else if (ltree) {  // a single primitive in the tree: the root is its leaf
        lroot = leaf_code(~(int32_t)rest_world[0]);
    }
    if (ref_sync) {
        memcpy(h + o_rank, ref_tables.rank.data(), ref_tables.rank.size() * 4);
        memcpy(h + o_up, ref_tables.up.data(), ref_tables.up.size() * 4);
        memcpy(h + o_refbox, ref_tables.refbox.data(), ref_tables.refbox.size() * 4);
    }

    cudaError_t e;
    const size_t ln_end = align_up(o_ln + (size_t)lni * NODE_BYTES, 256);
    if (device_tree && ln_end < stage_bytes) {
        // the node records are written on the device: nothing of that region is in the staging copy (4 MB at 65,536)
        e = o_ln ? cudaMemcpyAsync(sc->d_blob, h, o_ln, cudaMemcpyHostToDevice, ctx->stream) : cudaSuccess;
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(sc->d_blob + ln_end, h + ln_end, stage_bytes - ln_end, cudaMemcpyHostToDevice, ctx->stream);
    } else {
        e = cudaMemcpyAsync(sc->d_blob, h, stage_bytes, cudaMemcpyHostToDevice, ctx->stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);  // the staging buffer is reused by the next scene
    if (e != cudaSuccess) {
        give_back();
        return set_err(ctx, RT_ERR_CUDA, "scene upload failed: %s", cudaGetErrorString(e));
    }
    if (device_tree) {
        std::vector<float> dev_boxes(6 * rest.size());
        std::vector<uint32_t> dev_pid(rest.size());
        for (size_t i = 0; i < rest.size(); i++) {
            for (int a = 0; a < 3; a++) {
                dev_boxes[6 * i + a] = rest[i].min[a];
                dev_boxes[6 * i + 3 + a] = rest[i].max[a];
            }
            dev_pid[i] = pid_of_world[rest_world[i]];
        }
        uint32_t depth = 0;
        e = build_lbvh_device(&ctx->dbuild, dev_boxes.data(), dev_pid.data(), (uint32_t)dev_pid.size(),
                              (float4*)(sc->d_blob + o_ln), &depth, ctx->stream);
        if (e != cudaSuccess || depth > (uint32_t)MAX_STACK) {
            give_back();
            if (e != cudaSuccess) return set_err(ctx, RT_ERR_CUDA, "device BVH build failed: %s", cudaGetErrorString(e));
            return set_err(ctx, RT_ERR_UNSUPPORTED, "device-built tree depth %u exceeds the traversal stack (%d)", depth, MAX_STACK);
        }
        sc->tree_depth = depth;
        sc->device_tree = true;
    }
    if (ref_sync) aux->state.store(1, std::memory_order_release);

    DevScene& d = sc->dev;
    d.sph = (const float4*)(sc->d_blob + o_sph);
    d.tri = (const float4*)(sc->d_blob + o_tri);
    d.lnode = (const float4*)(sc->d_blob + o_ln);
    d.sph2 = (const float4*)(sc->d_blob + o_sph2);
    d.lni = lni;
    d.lroot = lroot;
    d.ltree = ltree ? 1 : 0;
    d.nbig = (uint32_t)big_world.size();
    d.big_code = (const int*)(sc->d_blob + o_big);
    d.mat = (const float4*)(sc->d_blob + o_mat);
    d.emis = (const float*)(sc->d_blob + o_em);
    d.rank = (const uint32_t*)(sc->d_blob + o_rank);
    d.leaf_box = (const float4*)(sc->d_blob + o_box);
    d.ref_up = (const uint32_t*)(sc->d_blob + o_up);
    d.ref_box = (const float4*)(sc->d_blob + o_refbox);
    d.aux_ready = 0;
    d.aux_flag = (const int*)(sc->d_blob + o_flag);
    d.ns = n_spheres;
    d.nt = n_triangles;
    d.ni = ni_ref;
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
    if (scene->d_blob) {
        if (ctx && ctx->retired.size() < 4) ctx->retired.push_back({scene->d_blob, scene->blob_cap});
        else cudaFree(scene->d_blob);
    }
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
