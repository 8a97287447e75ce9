// rt_api.cu — the C ABI of include/rt_b200.h: context, render calls, frame buffers.
//
// Replaces the body of worker() in ray-tracer-slave/src/main.rs:32-106 (see the header for the mapping); the scene side
// (main.rs:37,60-61) is rt_scene.cu, the one-process multi-GPU frame rt_multi.cu.
// There is no CPU fallback anywhere in this library: every render goes through launch_render().
#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>

#include "rt_ctx.h"

using namespace rtb;

static thread_local std::string g_init_err = "";

namespace rtb {

int set_err(rt_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    try {
        if (ctx) ctx->err = buf;
        else g_init_err = buf;
    } catch (...) {
    }
    return code;
}

// Brute force (K1) is picked only for tiny scenes: on the C5 sweep the BVH kernel already wins at 64 spheres
// (0.152 ms vs 0.247 ms at 1080p), see profiles/r1_c5_sweep.log
constexpr uint32_t kBruteMaxPrims = 16;

int resolve(rt_ctx* ctx, const rt_scene* scene, const rt_params* in, bool whole_frame, Resolved* r) {
    if (!scene || !in) return set_err(ctx, RT_ERR_INVALID_ARG, "NULL scene or params");
    const int rc = resolve_params(ctx, in, whole_frame, r);
    if (rc) return rc;
    r->isect = r->p.intersector == RT_INTERSECT_AUTO ? (scene->n <= kBruteMaxPrims ? RT_INTERSECT_BRUTE : RT_INTERSECT_BVH)
                                                     : (int)r->p.intersector;
    return RT_OK;
}

int resolve_params(rt_ctx* ctx, const rt_params* in, bool whole_frame, Resolved* r) {
    if (!in) return set_err(ctx, RT_ERR_INVALID_ARG, "NULL params");
    rt_params p = *in;
    if (whole_frame) {  // division fields do not apply to a whole-frame call
        p.divisions = 1;
        p.division_no = 0;
    }
    if (p.divisions == 0) p.divisions = 1;
    if (p.spp == 0) p.spp = 100;                                                              // main.rs:51
    if (p.max_bounces == 0 && !(p.flags & RT_PARAM_MAX_BOUNCES_EXPLICIT)) p.max_bounces = 10;  // main.rs:39
    if (p.aperture == 0.0f && !(p.flags & RT_PARAM_APERTURE_EXPLICIT)) p.aperture = 0.1f;      // main.rs:45
    if (p.focus_distance == 0.0f) p.focus_distance = 1.0f;
    if (p.field_of_view == 0.0f) p.field_of_view = 3.14159265358979323846f / 2.0f;  // PI / 2f32
    if (p.focal_length == 0.0f) p.focal_length = 1.0f;
    if (p.width == 0 || p.height == 0) return set_err(ctx, RT_ERR_INVALID_ARG, "zero width or height");
    if (p.height % p.divisions != 0)
        return set_err(ctx, RT_ERR_INVALID_ARG,
                       "height %u is not a multiple of divisions %u (the reference silently drops rows)", p.height,
                       p.divisions);
    if (p.division_no >= p.divisions) return set_err(ctx, RT_ERR_INVALID_ARG, "division_no out of range");
    if (p.max_bounces + 1 > (uint32_t)MAX_PATH)
        return set_err(ctx, RT_ERR_UNSUPPORTED, "max_bounces %u exceeds this build's limit %d", p.max_bounces, MAX_PATH - 1);
    if ((uint64_t)p.width * p.height > 0x7fffffffu) return set_err(ctx, RT_ERR_UNSUPPORTED, "frame too large");
    if (p.intersector > RT_INTERSECT_BVH) return set_err(ctx, RT_ERR_INVALID_ARG, "unknown intersector");
    r->p = p;
    // Camera::new (camera.rs:19-47) with the arguments of main.rs:42-50, single f32 ops in order
    DevCamera& c = r->cam;
    const float aspect = (float)p.width / (float)p.height;
    const float image_height = (float)p.height;
    const float vh = 2.0f * tanf(p.field_of_view / 2.0f);
    const float vw = aspect * vh;
    const float hor[3] = {vw, 0.0f, 0.0f}, ver[3] = {0.0f, vh, 0.0f}, fl[3] = {0.0f, 0.0f, p.focal_length};
    for (int a = 0; a < 3; a++) {
        c.org[a] = p.cam_origin[a];
        c.hor[a] = hor[a];
        c.ver[a] = ver[a];
        c.llc[a] = ((p.cam_origin[a] - hor[a] / 2.0f) - ver[a] / 2.0f) - fl[a];
    }
    c.lens_radius = p.aperture / 2.0f;
    c.u_den = aspect * image_height - 1.0f;
    c.v_den = image_height - 1.0f;
    c.focus = p.focus_distance;
    return RT_OK;
}

// A frame download is streamed in slabs of whole tile rows, about kSlabBytes each and at most kSlabs.
constexpr size_t kSlabs = 16;
constexpr size_t kSlabBytes = (size_t)1 << 20;
static_assert(kSlabs <= (size_t)MAX_SLABS, "a frame's control block has MAX_SLABS counters");
SlabPlan plan_slabs(uint32_t width, uint32_t rows) {
    SlabPlan p;
    p.width = width;
    p.rows = rows;
    const uint32_t tiles_y = (rows + TILE_H - 1) / TILE_H;
    const size_t bytes = (size_t)width * rows * 3;
    uint32_t s = (uint32_t)std::min<size_t>(kSlabs, std::max<size_t>(1, bytes / kSlabBytes));
    s = std::max(1u, std::min(s, tiles_y));
    p.tile_rows = (tiles_y + s - 1) / s;
    p.slabs = (tiles_y + p.tile_rows - 1) / p.tile_rows;
    return p;
}

static int ensure_out(rt_ctx* ctx, size_t bytes) {
    if (ctx->d_out_bytes >= bytes) return RT_OK;
    if (ctx->d_out) {
        CK(ctx, cudaStreamSynchronize(ctx->stream));
        CK(ctx, cudaStreamSynchronize(ctx->copy_stream));
        CK(ctx, cudaFree(ctx->d_out));
        ctx->d_out = nullptr;
        ctx->d_out_bytes = 0;
    }
    const size_t cap = rt_frame_ctl_offset(bytes);
    CK(ctx, cudaMalloc(&ctx->d_out, cap + RT_FRAME_CTL_BYTES));
    ctx->d_out_bytes = cap;
    return RT_OK;
}

// The context's own staging frame.  Its counters start from zero for every launch (frame number OWN_FRAME_SEQ = 1 each
// time): whether a launch counts at all is the launcher's choice (single-rank frames do not, rt_kernels.cu), so nothing
// cumulative can be assumed here — unlike the shared frames of rt_frame_alloc, whose ranks always count.
int own_frame(rt_ctx* ctx, uint32_t width, uint32_t rows, Frame* f) {
    const size_t bytes = (size_t)width * rows * 3;
    const int rc = ensure_out(ctx, bytes);
    if (rc) return rc;
    f->dev = ctx->d_out;
    f->ctl = reinterpret_cast<rt_frame_ctl*>(ctx->d_out + ctx->d_out_bytes);
    f->plan = plan_slabs(width, rows);
    CK(ctx, cudaMemsetAsync(f->ctl, 0, sizeof(rt_frame_ctl), ctx->stream));
    CK(ctx, cudaEventRecord(ctx->ev_sync, ctx->stream));
    CK(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_sync, 0));  // slab waits start after the reset
    return RT_OK;
}

Frame caller_frame(void* frame_dev, uint32_t width, uint32_t height) {
    Frame f;
    f.dev = static_cast<uint8_t*>(frame_dev);
    f.ctl = reinterpret_cast<rt_frame_ctl*>(f.dev + rt_frame_ctl_offset((size_t)width * height * 3));
    f.plan = plan_slabs(width, height);
    return f;
}

int check_frame_out(rt_ctx* ctx, const uint8_t* out_rgb, size_t out_len, uint32_t width, uint32_t height) {
    const size_t bytes = (size_t)width * height * 3;
    if (out_rgb && out_len != bytes) return set_err(ctx, RT_ERR_INVALID_ARG, "out_len %zu != height*width*3 = %zu", out_len, bytes);
    return RT_OK;
}

int launch(rt_ctx* ctx, const rt_scene* scene, const Resolved& r, const LaunchArgs& a, LaunchInfo* info) {
    DevParams pr{};
    pr.width = r.p.width;
    pr.height = r.p.height;
    pr.row0 = a.row0;
    pr.row1 = a.row1;
    pr.spp = r.p.spp;
    pr.depth = r.p.max_bounces + 1;
    pr.seed = r.p.seed;
    pr.tile_rank = a.tile_rank;
    pr.tile_ranks = a.tile_ranks;
    pr.out = a.frame.dev;
    pr.out_row0 = a.out_row0;
    pr.tiles_x = (r.p.width + TILE_W - 1) / TILE_W;
    pr.tiles_y = (a.row1 - a.row0 + TILE_H - 1) / TILE_H;
    pr.counters = ctx->d_ctr;
    pr.tile_counter = reinterpret_cast<unsigned int*>(ctx->d_ctr + RT_CTR_TICKETS);
    pr.redo_count = ctx->d_ctr + RT_CTR_REDO;
    pr.redo_list = ctx->d_redo;
    pr.redo_cap = RT_REDO_CAP;
    pr.pixel_list = a.pixel_list;
    pr.list_count = a.list_count;
    pr.state_in = static_cast<const uint4*>(a.state_in);
    pr.state_out = static_cast<uint4*>(a.state_out);
    pr.s0 = a.s0;
    pr.done = a.frame.ctl ? a.frame.ctl->done : nullptr;
    pr.stage_hint = a.stream ? 1 : 0;
    pr.redo_slab = ctx->d_ctr + RT_CTR_REDO_SLAB;
    pr.slab_tile_rows = a.frame.plan.tile_rows ? a.frame.plan.tile_rows : 1;
    const DevScene dev = scene_view(scene);
    CK(ctx, cudaMemsetAsync(ctx->d_ctr, 0, RT_CTR_SLOTS * sizeof(unsigned long long), ctx->stream));
    if (!a.pixel_list) CK(ctx, cudaMemsetAsync(ctx->d_redo, 0, RT_REDO_CAP * sizeof(unsigned int), ctx->stream));
    CK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    CK(ctx, launch_render(dev, r.cam, pr, r.isect, r.p.collect_counters != 0, ctx->sm_count, ctx->smem_optin, ctx->stream, info));
    CK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    return RT_OK;
}

// Reads the counter block after the kernel has completed (the stream must be synchronised by the caller or here).
static int read_counters(rt_ctx* ctx) {
    CK(ctx, cudaMemcpyAsync(ctx->h_ctr, ctx->d_ctr, RT_CTR_SLOTS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->h_flag[0]) {
        ctx->h_flag[0] = 0;
        return set_err(ctx, RT_ERR_TIMEOUT, "waited %d ms for a frame counter (the owner's \"consumed\" word, or a slab of the frame)", test_hooks().wait_timeout_ms);
    }
    return RT_OK;
}

static float ms_since(std::chrono::steady_clock::time_point t0) {
    return std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
}

// Camera rays of `shares` of the tile_ranks equal shares of the launch's rows: one share is what a rank reports alone;
// all of a frame's ranks together report the whole frame, also when the shares do not divide it evenly.
static uint64_t primary_rays(const Launch& l, uint32_t shares) {
    return (uint64_t)(l.a.row1 - l.a.row0) * l.r.p.width * shares / l.a.tile_ranks * (l.r.p.spp - l.a.s0);
}

// After the kernel of launch() has completed: re-renders the pixels that needed the tie-break tables before they had
// landed (waits for the tables), then fills l.st (total_ms is the caller's).  kernel_launches counts a second launch
// whenever the first pass listed pixels, even when the kernel's own redo rounds took all of them.
static int finish_launch(Launch& l) {
    rt_ctx* const ctx = l.ctx;
    int rc = read_counters(ctx);
    if (rc) return rc;
    const unsigned long long count = ctx->h_ctr[RT_CTR_REDO];
    const unsigned long long taken = ctx->h_ctr[RT_CTR_TICKET2] & 0xffffffffull;  // second passes done inside the kernel
    const uint32_t redone = count == 0 ? 0u : count > RT_REDO_CAP ? 0xffffffffu : (uint32_t)count;
    float first_ms = 0.0f;  // kernel time of the first pass when a second one follows (it re-records ev0 / ev1)
    if (count > RT_REDO_CAP || taken < count) {
        cudaEventElapsedTime(&first_ms, ctx->ev0, ctx->ev1);
        unsigned long long first[NUM_COUNTERS], slab_counts[MAX_SLABS];
        memcpy(first, ctx->h_ctr, sizeof first);
        memcpy(slab_counts, ctx->h_ctr + RT_CTR_REDO_SLAB, sizeof slab_counts);
        rc = scene_settle(ctx, l.scene);  // the tables must be there now
        if (rc) return rc;
        LaunchInfo li;
        LaunchArgs b = l.a;
        if (count > RT_REDO_CAP) {
            // more than the list holds: the whole launch again, without counting (every pixel it had not held back is
            // counted already); the pixels still held back are then counted slab by slab from the first pass's numbers
            b.frame.ctl = nullptr;
            rc = launch(ctx, l.scene, l.r, b, &li);
            if (rc) return rc;
            if (l.a.frame.ctl) {
                memcpy(ctx->h_ctr + RT_CTR_REDO_SLAB, slab_counts, sizeof slab_counts);
                CK(ctx, cudaMemcpyAsync(ctx->d_ctr + RT_CTR_REDO_SLAB, ctx->h_ctr + RT_CTR_REDO_SLAB, sizeof slab_counts,
                                        cudaMemcpyHostToDevice, ctx->stream));
                CK(ctx, launch_add_counts(l.a.frame.ctl->done, ctx->d_ctr + RT_CTR_REDO_SLAB, MAX_SLABS, ctx->stream));
            }
            rc = read_counters(ctx);  // the counters of the repeated launch are the frame's
            if (rc) return rc;
        } else {
            // the listed pixels nobody got to inside the kernel, with the tables: counted now (their first pass held
            // them back)
            b.pixel_list = ctx->d_redo + taken;
            b.list_count = (uint32_t)(count - taken);
            rc = launch(ctx, l.scene, l.r, b, &li);
            if (rc) return rc;
            rc = read_counters(ctx);
            if (rc) return rc;
            for (int i = 0; i < NUM_COUNTERS; i++) ctx->h_ctr[i] += first[i];  // queries of both passes (redo_pixels says so)
        }
    }
    rt_stats& st = l.st;
    memset(&st, 0, sizeof st);
    const unsigned long long* c = ctx->h_ctr;
    st.rays = c[CTR_RAYS];
    st.primary = primary_rays(l, 1);
    st.slab_tests = c[CTR_SLAB];
    st.sphere_tests = c[CTR_SPH_TEST];
    st.sphere_exact = c[CTR_SPH_EXACT];
    st.sphere_hits = c[CTR_SPH_HIT];
    st.tri_tests = c[CTR_TRI_TEST];
    st.tri_stage[0] = c[CTR_TRI_S1];
    st.tri_stage[1] = c[CTR_TRI_S2];
    st.tri_stage[2] = c[CTR_TRI_S3];
    st.tri_hits = c[CTR_TRI_HIT];
    st.shades_sphere = c[CTR_SHADE_SPH];
    st.shades_tri = c[CTR_SHADE_TRI];
    st.emissive = c[CTR_EMISSIVE];
    st.sky = c[CTR_SKY];
    st.active_lane_iters = c[CTR_ACTIVE_LANES];
    st.total_lane_iters = c[CTR_TOTAL_LANES];
    float ms = 0.0f;
    CK(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    st.kernel_ms = ms + first_ms;
    st.intersector_used = (uint32_t)l.r.isect;
    st.kernel_launches = 1u + (redone ? 1u : 0u);
    st.grid_ctas = l.info.grid;
    st.cta_threads = l.info.threads;
    st.ctas_per_sm = (uint32_t)l.info.ctas_per_sm;
    st.scene_in_smem = l.info.scene_in_smem ? 1u : 0u;
    st.dyn_smem_bytes = (uint32_t)l.info.dyn_smem;
    st.redo_pixels = redone;
    return RT_OK;
}

// The statistics of the n launches of one call together (n = 1: the launch's own).  The counters, kernel_launches and
// redo_pixels add up (redo_pixels stays at 0xffffffff, "more than the list held", once a launch reports it); kernel_ms is
// the longest launch's, as the launches run side by side; intersector_used and the launch shape are the first launch's
// (context 0's); primary counts the launches' shares together.  total_ms is the caller's.
static rt_stats combine_stats(const Launch* l, uint32_t n) {
    rt_stats t;
    memset(&t, 0, sizeof t);
    for (uint32_t i = 0; i < n; i++) {
        const rt_stats& s = l[i].st;
        t.rays += s.rays;
        t.slab_tests += s.slab_tests;
        t.sphere_tests += s.sphere_tests;
        t.sphere_exact += s.sphere_exact;
        t.sphere_hits += s.sphere_hits;
        t.tri_tests += s.tri_tests;
        for (int k = 0; k < 3; k++) t.tri_stage[k] += s.tri_stage[k];
        t.tri_hits += s.tri_hits;
        t.shades_sphere += s.shades_sphere;
        t.shades_tri += s.shades_tri;
        t.emissive += s.emissive;
        t.sky += s.sky;
        t.active_lane_iters += s.active_lane_iters;
        t.total_lane_iters += s.total_lane_iters;
        t.kernel_launches += s.kernel_launches;
        t.redo_pixels = (t.redo_pixels == 0xffffffffu || s.redo_pixels == 0xffffffffu) ? 0xffffffffu : t.redo_pixels + s.redo_pixels;
        t.kernel_ms = std::max(t.kernel_ms, s.kernel_ms);
    }
    t.primary = primary_rays(l[0], n);
    t.intersector_used = l[0].st.intersector_used;
    t.grid_ctas = l[0].st.grid_ctas;
    t.cta_threads = l[0].st.cta_threads;
    t.ctas_per_sm = l[0].st.ctas_per_sm;
    t.scene_in_smem = l[0].st.scene_in_smem;
    t.dyn_smem_bytes = l[0].st.dyn_smem_bytes;
    return t;
}

// On the frame owner.  enqueue: for every slab, on the copy stream, wait (on the device) until frame number `seq` of it
// is complete, then copy it towards out_rgb (nullptr: only wait) — asynchronous; a pageable out_rgb is reached through a
// pinned staging frame.  finish: host side of the same — returns when every slab is in out_rgb.  Between the two the
// caller is free to finish its own kernel (second pass included): nothing here blocks the render stream.
struct SlabJob {
    SlabPlan plan;
    uint8_t* out = nullptr;       // caller's destination
    uint8_t* pinned = nullptr;    // where the device copies go (== out when out is pinned)
    uint32_t host_done = 0;       // pageable path: slabs already copied on to `out`
    const rt_frame_ctl* ctl = nullptr;
};

static int enqueue_slab_copies(rt_ctx* ctx, const uint8_t* frame_dev, const rt_frame_ctl* ctl, const SlabPlan& plan, uint64_t seq,
                               uint8_t* out_rgb, SlabJob* job) {
    job->plan = plan;
    job->out = out_rgb;
    job->pinned = out_rgb;
    const size_t bytes = (size_t)plan.rows * plan.width * 3;
    if (out_rgb) {
        cudaPointerAttributes attr;
        const cudaError_t pe = cudaPointerGetAttributes(&attr, out_rgb);
        (void)cudaGetLastError();
        if (pe != cudaSuccess || attr.type == cudaMemoryTypeUnregistered) {
            // pageable destination: an asynchronous copy would block this thread until the slab is complete; go through
            // pinned staging and copy slab by slab on the host as they land
            if (ctx->h_frame_bytes < bytes) {
                if (ctx->h_frame) cudaFreeHost(ctx->h_frame);
                ctx->h_frame = nullptr;
                ctx->h_frame_bytes = 0;
                CK(ctx, cudaMallocHost(&ctx->h_frame, bytes));
                ctx->h_frame_bytes = bytes;
            }
            job->pinned = ctx->h_frame;
            while (ctx->slab_events.size() < plan.slabs) {
                cudaEvent_t e;
                CK(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                ctx->slab_events.push_back(e);
            }
        }
    }
    ctx->h_flag[0] = 0;
    job->ctl = ctl;
    const bool by_value = ctx->stream_wait_value64 != nullptr;
    if (!out_rgb && !by_value)  // the frame stays on the device: one kernel waits for all its slabs
        CK(ctx, launch_wait_all_slabs(ctl->done, (unsigned long long)seq, plan.slabs, plan.tile_rows, plan.rows, plan.width,
                                      ctx->h_flag, ctx->copy_stream));
    for (uint32_t i = 0; (out_rgb || by_value) && i < plan.slabs; i++) {
        // tickets walk the frame bottom-up: the last slab completes first
        const uint32_t s = plan.slabs - 1 - i;
        const unsigned long long target = (unsigned long long)seq * plan.pixels(s);
        if (by_value) {  // CU_STREAM_WAIT_VALUE_GEQ = 0: the stream itself waits, no SM involved
            const int wr = ctx->stream_wait_value64((void*)ctx->copy_stream, (unsigned long long)(uintptr_t)&ctl->done[s], target, 0u);
            if (wr != 0) return set_err(ctx, RT_ERR_CUDA, "cuStreamWaitValue64 failed (%d)", wr);
        } else {
            CK(ctx, launch_wait_slab(&ctl->done[s], target, ctx->h_flag, ctx->copy_stream));
        }
        if (out_rgb) {
            const size_t off = (size_t)plan.first_row(s) * plan.width * 3;
            const size_t nb = (size_t)plan.row_count(s) * plan.width * 3;
            CK(ctx, cudaMemcpyAsync(job->pinned + off, frame_dev + off, nb, cudaMemcpyDeviceToHost, ctx->copy_stream));
            if (job->pinned != out_rgb) CK(ctx, cudaEventRecord(ctx->slab_events[s], ctx->copy_stream));
        }
    }
    // the frame is out of the buffer: ranks waiting to overwrite it may go on (rt_frame_wait_consumed)
    CK(ctx, launch_set_u64(const_cast<unsigned long long*>(&ctl->consumed), (unsigned long long)seq, ctx->copy_stream));
    return RT_OK;
}

// Pageable destination: slab by slab from the pinned staging frame, as each lands.  until_kernel_done: stop (returning the
// number of slabs done) as soon as the render kernel of this context has finished, so that the caller can look after
// pixels the kernel left for a second pass before blocking on slabs that wait for exactly those pixels.
static int host_copy_slabs(rt_ctx* ctx, const SlabJob& job, uint32_t first, bool until_kernel_done, uint32_t* done_out) {
    uint32_t i = first;
    for (; i < job.plan.slabs; i++) {
        const uint32_t s = job.plan.slabs - 1 - i;  // in the order enqueue_slab_copies queued them
        if (until_kernel_done) {
            bool landed = false;
            for (;;) {
                if (cudaEventQuery(ctx->slab_events[s]) == cudaSuccess) { landed = true; break; }
                if (cudaEventQuery(ctx->ev1) == cudaSuccess) break;
                std::this_thread::yield();
            }
            (void)cudaGetLastError();
            if (!landed) break;
        } else {
            const auto t0 = std::chrono::steady_clock::now();
            while (cudaEventQuery(ctx->slab_events[s]) != cudaSuccess) {
                if (std::chrono::steady_clock::now() - t0 > std::chrono::milliseconds(test_hooks().wait_timeout_ms)) {
                    (void)cudaGetLastError();
                    *done_out = i;
                    return RT_OK;  // finish_slab_copies' drain reports the timeout
                }
                std::this_thread::yield();
            }
            (void)cudaGetLastError();
        }
        if (ctx->h_flag[0]) break;
        const size_t off = (size_t)job.plan.first_row(s) * job.plan.width * 3;
        memcpy(job.out + off, job.pinned + off, (size_t)job.plan.row_count(s) * job.plan.width * 3);
    }
    *done_out = i;
    return RT_OK;
}

// A stream that waits by value has no time limit of its own: when the wait limit (RT_B200_WAIT_TIMEOUT_MS, 20 s) is
// over, every wait is satisfied from the side and the caller reports the timeout.
static int drain_copy_stream(rt_ctx* ctx, const SlabJob& job) {
    const auto t0 = std::chrono::steady_clock::now();
    for (;;) {
        const cudaError_t q = cudaStreamQuery(ctx->copy_stream);
        if (q == cudaSuccess) break;
        if (q != cudaErrorNotReady) return set_err(ctx, RT_ERR_CUDA, "copy stream: %s", cudaGetErrorString(q));
        if (std::chrono::steady_clock::now() - t0 > std::chrono::milliseconds(test_hooks().wait_timeout_ms)) {
            ctx->h_flag[0] = 1;
            if (job.ctl) {
                unsigned long long* fill = ctx->h_ctr;  // pinned scratch: RT_CTR_SLOTS >= MAX_SLABS entries
                for (int i = 0; i < MAX_SLABS; i++) fill[i] = 0x7fffffffffffffffull;
                cudaMemcpyAsync(const_cast<unsigned long long*>(job.ctl->done), fill, MAX_SLABS * sizeof(unsigned long long),
                                cudaMemcpyHostToDevice, ctx->aux_stream);
                cudaStreamSynchronize(ctx->aux_stream);
            }
            cudaStreamSynchronize(ctx->copy_stream);
            break;
        }
        std::this_thread::yield();
    }
    (void)cudaGetLastError();
    return RT_OK;
}

static int finish_slab_copies(rt_ctx* ctx, const SlabJob& job) {
    if (job.out && job.pinned != job.out) {
        uint32_t done = 0;
        const int rc = host_copy_slabs(ctx, job, job.host_done, false, &done);
        if (rc) return rc;
    }
    const int rc = drain_copy_stream(ctx, job);
    if (rc) return rc;
    if (ctx->h_flag[0]) {
        ctx->h_flag[0] = 0;  // reported here: the next call starts clean
        return set_err(ctx, RT_ERR_TIMEOUT, "a slab of the frame did not complete within %d ms", test_hooks().wait_timeout_ms);
    }
    return RT_OK;
}

int collect_frame(rt_ctx* owner, const Frame& f, uint64_t seq, uint8_t* out_rgb, Launch* l, uint32_t n, rt_stats* stats,
                  std::chrono::steady_clock::time_point t0) {
    const auto relay = [&](uint32_t i, int rc) {
        if (rc && l[i].ctx != owner) set_err(owner, rc, "context %u: %s", i, l[i].ctx->err.c_str());
        return rc;
    };
    int rc;
    for (uint32_t i = 0; i < n; i++) {
        CK(owner, cudaSetDevice(l[i].ctx->device));
        if ((rc = relay(i, launch(l[i].ctx, l[i].scene, l[i].r, l[i].a, &l[i].info)))) return rc;
    }
    CK(owner, cudaSetDevice(owner->device));
    // The frame streams when every launch counts its finished pixels into the frame's control block and there is more
    // than one slab or rank to wait for.  Streaming waits on the device for the kernels; contexts that share a device
    // also share its hardware queues, where a wait could sit in front of the very kernel it waits for, so such frames
    // are copied after the kernels instead.  With no launch the ranks elsewhere count: the frame always streams.
    bool streamed = true;
    for (uint32_t i = 0; i < n; i++) {
        streamed = streamed && l[i].info.counts_done && f.ctl && (f.plan.slabs > 1 || l[i].a.tile_ranks > 1);
        for (uint32_t j = 0; j < i; j++) streamed = streamed && l[i].ctx->device != l[j].ctx->device;
    }
    SlabJob job;
    const bool late = owner->serial_launches;  // launches block: queue the waits once nothing of ours is outstanding
    if (streamed && !late) {
        rc = enqueue_slab_copies(owner, f.dev, f.ctl, f.plan, seq, out_rgb, &job);
        if (rc) return rc;
        // pageable destination: host copies while the owner's kernel runs (it stops there, never waiting on a second
        // pass that only the loop below runs)
        if (n && job.out && job.pinned != job.out) {
            rc = host_copy_slabs(owner, job, 0, true, &job.host_done);
            if (rc) return rc;
        }
    }
    for (uint32_t i = 0; i < n; i++) {  // kernels done: the pixels they still held back are final (and counted) now
        CK(owner, cudaSetDevice(l[i].ctx->device));
        if ((rc = relay(i, finish_launch(l[i])))) return rc;
    }
    CK(owner, cudaSetDevice(owner->device));
    if (streamed && late) {
        rc = enqueue_slab_copies(owner, f.dev, f.ctl, f.plan, seq, out_rgb, &job);
        if (rc) return rc;
    }
    if (streamed) {
        rc = finish_slab_copies(owner, job);
        if (rc) return rc;
    } else if (out_rgb) {
        CK(owner, cudaMemcpyAsync(out_rgb, f.dev, (size_t)f.plan.rows * f.plan.width * 3, cudaMemcpyDeviceToHost, owner->stream));
        CK(owner, cudaStreamSynchronize(owner->stream));
    }
    if (stats && n) {
        *stats = combine_stats(l, n);
        stats->total_ms = ms_since(t0);
    }
    return RT_OK;
}

}  // namespace rtb

namespace {

int render_rows_to_host(rt_ctx* ctx, const rt_scene* scene, const Resolved& r, uint32_t row0, uint32_t row1,
                        uint8_t* out_rgb, size_t out_len, rt_stats* stats) {
    const auto t0 = std::chrono::steady_clock::now();
    const size_t bytes = (size_t)(row1 - row0) * r.p.width * 3;
    if (!out_rgb) return set_err(ctx, RT_ERR_INVALID_ARG, "out_rgb is NULL");
    if (out_len != bytes)
        return set_err(ctx, RT_ERR_INVALID_ARG, "out_len %zu != (rows %u * width %u * 3) = %zu", out_len, row1 - row0,
                       r.p.width, bytes);
    CK(ctx, cudaSetDevice(ctx->device));
    Launch l{ctx, scene, r};
    l.a.row0 = row0;
    l.a.row1 = row1;
    l.a.out_row0 = row0;
    const int rc = own_frame(ctx, r.p.width, row1 - row0, &l.a.frame);
    if (rc) return rc;
    // Streaming the frame out slab by slab while it renders beats one copy after the kernel on a single GPU when a pixel
    // is many samples of work (C3, 16 spp: stage + counters +0.2 ms, the 25 MB copy 0.5 ms); at few samples per pixel
    // the stage costs more than the copy (C2, 1 spp: +0.09 vs 0.12 ms incl. the slab waits; C4, 4 spp: +2.2 vs 2.0 ms)
    l.a.stream = bytes >= ((size_t)4 << 20) && l.a.frame.plan.slabs > 1 && r.p.spp >= 8;
    return collect_frame(ctx, l.a.frame, OWN_FRAME_SEQ, out_rgb, &l, 1, stats, t0);
}

// Rank tile_rank of tile_ranks of a caller's whole frame.  seq (nullable: not the frame owner's call) must not be 0.
int tiles_args(rt_ctx* ctx, const Resolved& r, void* frame_dev, uint32_t tile_rank, uint32_t tile_ranks, const uint64_t* seq,
               LaunchArgs* a) {
    if (!frame_dev) return set_err(ctx, RT_ERR_INVALID_ARG, "frame_dev is NULL");
    if (tile_ranks == 0 || tile_rank >= tile_ranks || (seq && *seq == 0))
        return set_err(ctx, RT_ERR_INVALID_ARG, seq ? "bad tile_rank/tile_ranks/seq" : "bad tile_rank/tile_ranks");
    a->row1 = r.p.height;
    a->tile_rank = tile_rank;
    a->tile_ranks = tile_ranks;
    a->frame = caller_frame(frame_dev, r.p.width, r.p.height);
    return RT_OK;
}

}  // namespace

extern "C" {

// Nsight Compute (and CUDA_LAUNCH_BLOCKING=1) make every kernel launch synchronous.  The frame owner normally queues
// its slab waits, then runs the second pass that releases the pixels its first pass held back (finish_launch); with
// blocking launches the host would sit in the launch of a wait (or of the kernel behind the value waits) that only its
// own next step can satisfy — measured: bench.py under ncu stopped at the first streamed frame.  So when launches
// block, the waits are queued after the second pass.
static bool launches_block() {
    extern char** environ;
    for (char** e = environ; e && *e; e++)
        if (!strncmp(*e, "NV_NSIGHT_INJECTION", 19) || !strncmp(*e, "NV_COMPUTE_PROFILER", 19) ||
            !strncmp(*e, "CUDA_INJECTION64_PATH=", 22))
            return true;
    const char* b = std::getenv("CUDA_LAUNCH_BLOCKING");
    return b && atoi(b) != 0;
}

int rt_abi_version(void) { return RT_B200_ABI_VERSION; }

void rt_struct_sizes(size_t out[4]) {
    out[0] = sizeof(rt_sphere);
    out[1] = sizeof(rt_triangle);
    out[2] = sizeof(rt_params);
    out[3] = sizeof(rt_stats);
}

const char* rt_last_error(const rt_ctx* ctx) { return ctx ? ctx->err.c_str() : g_init_err.c_str(); }

int rt_init(int device, rt_ctx** out) {
    if (!out) return set_err(nullptr, RT_ERR_INVALID_ARG, "rt_init: out is NULL");
    *out = nullptr;
    RT_GUARD_BEGIN
    (void)test_hooks();  // the environment is read here, once
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return set_err(nullptr, RT_ERR_NO_DEVICE, "no CUDA device (%s); this library has no CPU fallback",
                       e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    if (device < 0 || device >= count)
        return set_err(nullptr, RT_ERR_INVALID_ARG, "device %d out of range [0,%d)", device, count);
    rt_ctx* ctx = new rt_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
#define CKI(call)                                                                                      \
    do {                                                                                               \
        cudaError_t e__ = (call);                                                                      \
        if (e__ != cudaSuccess) {                                                                      \
            set_err(nullptr, RT_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e__));            \
            rt_shutdown(ctx);                                                                          \
            return RT_ERR_CUDA;                                                                        \
        }                                                                                              \
    } while (0)
    CKI(cudaSetDevice(device));
    CKI(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        set_err(nullptr, RT_ERR_NO_DEVICE, "device %d is sm_%d%d; this build carries sm_100a code only", device,
                prop.major, prop.minor);
        rt_shutdown(ctx);
        return RT_ERR_NO_DEVICE;
    }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = (int)prop.sharedMemPerBlockOptin;
    CKI(cudaDeviceGetAttribute(&ctx->clock_khz, cudaDevAttrClockRate, device));
    memcpy(ctx->name, prop.name, 63); ctx->name[63] = 0;
    CKI(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    CKI(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    CKI(cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking));
    CKI(cudaEventCreate(&ctx->ev0));
    CKI(cudaEventCreate(&ctx->ev1));
    CKI(cudaEventCreateWithFlags(&ctx->ev_sync, cudaEventDisableTiming));
    CKI(cudaMalloc(&ctx->d_ctr, RT_CTR_SLOTS * sizeof(unsigned long long)));
    CKI(cudaMallocHost(&ctx->h_ctr, RT_CTR_SLOTS * sizeof(unsigned long long)));
    CKI(cudaMalloc(&ctx->d_redo, RT_REDO_CAP * sizeof(unsigned int)));
    CKI(cudaHostAlloc(&ctx->h_flag, 64, cudaHostAllocMapped));
    ctx->h_flag[0] = 0;
    // load the module and resolve every kernel now: the first division of a job must not pay the lazy load
    CKI(preload_kernels());
    ctx->serial_launches = launches_block();
    {   // stream memory operations, if this driver and device have them (64-bit waits)
        int can64 = 0;
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaDeviceGetAttribute(&can64, static_cast<cudaDeviceAttr>(122) /* CU_DEVICE_ATTRIBUTE_CAN_USE_64_BIT_STREAM_MEM_OPS */, device) == cudaSuccess && can64 &&
            cudaGetDriverEntryPoint("cuStreamWaitValue64", &fn, cudaEnableDefault, &qr) == cudaSuccess &&
            qr == cudaDriverEntryPointSuccess && fn && !test_hooks().no_stream_wait)
            ctx->stream_wait_value64 = reinterpret_cast<int (*)(void*, unsigned long long, unsigned long long, unsigned int)>(fn);
        (void)cudaGetLastError();
    }
#undef CKI
    *out = ctx;
    return RT_OK;
    RT_GUARD_END(nullptr)
}

void rt_shutdown(rt_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    if (ctx->aux_stream) cudaStreamSynchronize(ctx->aux_stream);
    if (ctx->d_out) cudaFree(ctx->d_out);
    if (ctx->d_ctr) cudaFree(ctx->d_ctr);
    if (ctx->h_ctr) cudaFreeHost(ctx->h_ctr);
    if (ctx->d_redo) cudaFree(ctx->d_redo);
    if (ctx->h_flag) cudaFreeHost(ctx->h_flag);
    if (ctx->h_frame) cudaFreeHost(ctx->h_frame);
    for (cudaEvent_t e : ctx->slab_events) cudaEventDestroy(e);
    if (ctx->d_scratch) cudaFree(ctx->d_scratch);
    if (ctx->d_flush) cudaFree(ctx->d_flush);
    free_device_build(&ctx->dbuild);
    for (auto& r : ctx->retired) cudaFree(r.p);
    ctx->retired.clear();
    for (void* p : ctx->host_allocs) cudaFreeHost(p);
    ctx->host_allocs.clear();
    if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->ev_sync) cudaEventDestroy(ctx->ev_sync);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
    delete ctx;
}

int rt_device_info(rt_ctx* ctx, int* sm_count, int* clock_khz, int* smem_optin, char name_out[64]) {
    if (!ctx) return RT_ERR_INVALID_ARG;
    if (sm_count) *sm_count = ctx->sm_count;
    if (clock_khz) *clock_khz = ctx->clock_khz;
    if (smem_optin) *smem_optin = ctx->smem_optin;
    if (name_out) memcpy(name_out, ctx->name, 64);
    return RT_OK;
}

void* rt_stream(rt_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int rt_sync(rt_ctx* ctx) {
    if (!ctx) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->copy_stream));
    return RT_OK;
    RT_GUARD_END(ctx)
}

// -------------------------------------------------------------------------------------------------
// Render
// -------------------------------------------------------------------------------------------------
int rt_render_division(rt_ctx* ctx, const rt_scene* scene, const rt_params* params, uint8_t* out_rgb, size_t out_len,
                       rt_stats* stats) {
    if (!ctx) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    Resolved r;
    int rc = resolve(ctx, scene, params, false, &r);
    if (rc) return rc;
    const uint32_t band = r.p.height / r.p.divisions;  // main.rs:55-56
    const uint32_t row0 = band * r.p.division_no;      // main.rs:66-68
    return render_rows_to_host(ctx, scene, r, row0, row0 + band, out_rgb, out_len, stats);
    RT_GUARD_END(ctx)
}

int rt_render_frame(rt_ctx* ctx, const rt_scene* scene, const rt_params* params, uint8_t* out_rgb, size_t out_len,
                    rt_stats* stats) {
    if (!ctx) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    Resolved r;
    int rc = resolve(ctx, scene, params, true, &r);
    if (rc) return rc;
    return render_rows_to_host(ctx, scene, r, 0, r.p.height, out_rgb, out_len, stats);
    RT_GUARD_END(ctx)
}

int rt_render_tiles_device(rt_ctx* ctx, const rt_scene* scene, const rt_params* params, uint32_t tile_rank,
                           uint32_t tile_ranks, void* frame_dev, int sync, rt_stats* stats) {
    if (!ctx) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    const auto t0 = std::chrono::steady_clock::now();
    Launch l{ctx, scene};
    int rc = resolve(ctx, scene, params, true, &l.r);
    if (rc) return rc;
    rc = tiles_args(ctx, l.r, frame_dev, tile_rank, tile_ranks, nullptr, &l.a);
    if (rc) return rc;
    CK(ctx, cudaSetDevice(ctx->device));
    if (!sync) {  // nobody will be there for a second pass: have the tie-break tables first
        rc = scene_settle(ctx, scene);
        if (rc) return rc;
    }
    rc = launch(ctx, scene, l.r, l.a, &l.info);
    if (rc || !sync) return rc;
    rc = finish_launch(l);
    if (rc) return rc;
    if (stats) {
        *stats = l.st;  // primary: the frame's pixels / ranks (the exact count of this rank's tiles is not needed)
        stats->total_ms = ms_since(t0);
    }
    return RT_OK;
    RT_GUARD_END(ctx)
}

int rt_render_tiles_collect(rt_ctx* ctx, const rt_scene* scene, const rt_params* params, uint32_t tile_rank,
                            uint32_t tile_ranks, void* frame_dev, uint64_t seq, uint8_t* out_rgb, size_t out_len,
                            rt_stats* stats) {
    if (!ctx) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    const auto t0 = std::chrono::steady_clock::now();
    Launch l{ctx, scene};
    int rc = resolve(ctx, scene, params, true, &l.r);
    if (rc) return rc;
    rc = tiles_args(ctx, l.r, frame_dev, tile_rank, tile_ranks, &seq, &l.a);
    if (rc) return rc;
    rc = check_frame_out(ctx, out_rgb, out_len, l.r.p.width, l.r.p.height);
    if (rc) return rc;
    CK(ctx, cudaSetDevice(ctx->device));
    return collect_frame(ctx, l.a.frame, seq, out_rgb, &l, 1, stats, t0);
    RT_GUARD_END(ctx)
}

// -------------------------------------------------------------------------------------------------
// Progressive rendering: resumable per-pixel sample chains
// -------------------------------------------------------------------------------------------------
// The samples of a render at spp = k are the first k samples of a render at any larger spp (no draw depends on spp, the
// sum is folded in order, quantise() divides at the end), so chunks of samples reproduce rt_render_division at the
// cumulative count byte for byte.
int rt_accum_create(rt_ctx* ctx, const rt_params* params, rt_accum** out) {
    if (!ctx) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    if (!out) return set_err(ctx, RT_ERR_INVALID_ARG, "rt_accum_create: out is NULL");
    *out = nullptr;
    Resolved r;
    const int rc = resolve_params(ctx, params, false, &r);
    if (rc) return rc;
    std::unique_ptr<rt_accum> acc(new rt_accum());
    acc->ctx = ctx;
    acc->params = *params;
    acc->params.collect_counters = 0;
    const uint32_t band = r.p.height / r.p.divisions;
    acc->row0 = band * r.p.division_no;
    acc->row1 = acc->row0 + band;
    const size_t bytes = (size_t)band * r.p.width * STATE_RECORD_BYTES;
    CK(ctx, cudaSetDevice(ctx->device));
    for (int i = 0; i < 2; i++) {
        const cudaError_t e = cudaMalloc(&acc->state[i], bytes);
        if (e != cudaSuccess) {
            if (i) cudaFree(acc->state[0]);
            (void)cudaGetLastError();
            return set_err(ctx, RT_ERR_CUDA, "rt_accum_create: cudaMalloc of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
        }
    }
    *out = acc.release();
    return RT_OK;
    RT_GUARD_END(ctx)
}

void rt_accum_destroy(rt_ctx* ctx, rt_accum* acc) {
    if (!acc) return;
    rt_ctx* c = ctx ? ctx : acc->ctx;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    cudaFree(acc->state[0]);
    cudaFree(acc->state[1]);
    delete acc;
}

int rt_accum_reset(rt_ctx* ctx, rt_accum* acc, const rt_params* params) {
    if (!ctx) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    if (!acc || acc->ctx != ctx) return set_err(ctx, RT_ERR_INVALID_ARG, "rt_accum_reset: accum is NULL or of another context");
    if (params) {
        Resolved r;
        const int rc = resolve_params(ctx, params, false, &r);
        if (rc) return rc;
        const uint32_t band = r.p.height / r.p.divisions, row0 = band * r.p.division_no;
        if (r.p.width != acc->params.width || r.p.height != acc->params.height || row0 != acc->row0 || row0 + band != acc->row1)
            return set_err(ctx, RT_ERR_INVALID_ARG, "rt_accum_reset: width, height and band must stay %ux%u, rows [%u, %u)",
                           acc->params.width, acc->params.height, acc->row0, acc->row1);
        acc->params = *params;
        acc->params.collect_counters = 0;
    }
    acc->samples = 0;
    acc->scene_serial = 0;
    return RT_OK;
    RT_GUARD_END(ctx)
}

int rt_accum_samples(const rt_accum* acc, uint32_t* samples_out) {
    if (!acc || !samples_out) return RT_ERR_INVALID_ARG;
    *samples_out = acc->samples;
    return RT_OK;
}

int rt_render_samples(rt_ctx* ctx, const rt_scene* scene, rt_accum* acc, uint32_t n_samples, uint8_t* out_rgb,
                      size_t out_len, rt_stats* stats) {
    if (!ctx) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    const auto t0 = std::chrono::steady_clock::now();
    if (!acc || acc->ctx != ctx) return set_err(ctx, RT_ERR_INVALID_ARG, "rt_render_samples: accum is NULL or of another context");
    if (!scene) return set_err(ctx, RT_ERR_INVALID_ARG, "rt_render_samples: scene is NULL");
    if (n_samples == 0) return set_err(ctx, RT_ERR_INVALID_ARG, "rt_render_samples: n_samples is 0");
    if ((uint64_t)acc->samples + n_samples > 0xffffffffull)
        return set_err(ctx, RT_ERR_INVALID_ARG, "rt_render_samples: %u + %u samples overflow 32 bits", acc->samples, n_samples);
    if (acc->samples && scene->serial != acc->scene_serial)
        return set_err(ctx, RT_ERR_INVALID_ARG, "rt_render_samples: not the scene of the chunks since the last create / reset");
    rt_params p = acc->params;
    p.spp = acc->samples + n_samples;
    Launch l{ctx, scene};
    int rc = resolve(ctx, scene, &p, false, &l.r);
    if (rc) return rc;
    const uint32_t rows = acc->row1 - acc->row0, width = l.r.p.width;
    const size_t bytes = (size_t)rows * width * 3;
    if (out_rgb && out_len != bytes)
        return set_err(ctx, RT_ERR_INVALID_ARG, "out_len %zu != (rows %u * width %u * 3) = %zu", out_len, rows, width, bytes);
    CK(ctx, cudaSetDevice(ctx->device));
    l.a.row0 = acc->row0;
    l.a.row1 = acc->row1;
    l.a.out_row0 = acc->row0;
    rc = own_frame(ctx, width, rows, &l.a.frame);
    if (rc) return rc;
    l.a.stream = false;  // the band is copied after the kernel
    l.a.state_in = acc->state[acc->cur];
    l.a.state_out = acc->state[acc->cur ^ 1];
    l.a.s0 = acc->samples;
    rc = collect_frame(ctx, l.a.frame, OWN_FRAME_SEQ, out_rgb, &l, 1, stats, t0);
    if (rc) return rc;
    acc->cur ^= 1;
    acc->samples += n_samples;
    acc->scene_serial = scene->serial;
    return RT_OK;
    RT_GUARD_END(ctx)
}

int rt_accum_read_linear(rt_ctx* ctx, const rt_accum* acc, float* out, size_t out_len) {
    if (!ctx) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    if (!acc || acc->ctx != ctx) return set_err(ctx, RT_ERR_INVALID_ARG, "rt_accum_read_linear: accum is NULL or of another context");
    if (!out) return set_err(ctx, RT_ERR_INVALID_ARG, "rt_accum_read_linear: out is NULL");
    if (acc->samples == 0) return set_err(ctx, RT_ERR_INVALID_ARG, "rt_accum_read_linear: no samples rendered yet");
    const uint64_t pixels = (uint64_t)(acc->row1 - acc->row0) * acc->params.width;
    const size_t bytes = (size_t)pixels * 3 * sizeof(float);
    if (out_len != bytes) return set_err(ctx, RT_ERR_INVALID_ARG, "out_len %zu != rows * width * 3 * 4 = %zu", out_len, bytes);
    CK(ctx, cudaSetDevice(ctx->device));
    // the buffer the next chunk writes in full serves as the scratch (12 of its 48 bytes per pixel)
    float* scratch = static_cast<float*>(acc->state[acc->cur ^ 1]);
    CK(ctx, launch_accum_linear(acc->state[acc->cur], scratch, pixels, acc->samples, ctx->sm_count, ctx->stream));
    CK(ctx, cudaMemcpyAsync(out, scratch, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return RT_OK;
    RT_GUARD_END(ctx)
}

// -------------------------------------------------------------------------------------------------
// Memory helpers
// -------------------------------------------------------------------------------------------------
int rt_host_alloc(rt_ctx* ctx, size_t bytes, void** out) {
    if (!ctx || !out) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMallocHost(out, bytes ? bytes : 1));
    ctx->host_allocs.push_back(*out);
    return RT_OK;
    RT_GUARD_END(ctx)
}
void rt_host_free(rt_ctx* ctx, void* p) {
    if (!p) return;
    if (ctx) {
        cudaSetDevice(ctx->device);
        auto it = std::find(ctx->host_allocs.begin(), ctx->host_allocs.end(), p);
        if (it == ctx->host_allocs.end()) return;  // not ours (or already freed)
        ctx->host_allocs.erase(it);
    }
    cudaFreeHost(p);
}

int rt_frame_alloc(rt_ctx* ctx, size_t bytes, void** dev_out, uint8_t handle_out[64]) {
    if (!ctx || !dev_out) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CK(ctx, cudaSetDevice(ctx->device));
    const size_t ctl_off = rt_frame_ctl_offset(bytes ? bytes : 1);
    CK(ctx, cudaMalloc(dev_out, ctl_off + RT_FRAME_CTL_BYTES));
    CK(ctx, cudaMemset((uint8_t*)*dev_out + ctl_off, 0, RT_FRAME_CTL_BYTES));
    if (handle_out) {
        cudaIpcMemHandle_t h;
        CK(ctx, cudaIpcGetMemHandle(&h, *dev_out));
        memcpy(handle_out, &h, 64);
    }
    return RT_OK;
    RT_GUARD_END(ctx)
}
int rt_frame_open(rt_ctx* ctx, const uint8_t handle[64], void** dev_out) {
    if (!ctx || !handle || !dev_out) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    CK(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    CK(ctx, cudaIpcOpenMemHandle(dev_out, h, cudaIpcMemLazyEnablePeerAccess));
    return RT_OK;
    RT_GUARD_END(ctx)
}
int rt_frame_close(rt_ctx* ctx, void* dev) {
    if (!ctx) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    CK(ctx, cudaIpcCloseMemHandle(dev));
    return RT_OK;
    RT_GUARD_END(ctx)
}
int rt_frame_free(rt_ctx* ctx, void* dev) {
    if (!ctx) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->copy_stream));
    CK(ctx, cudaFree(dev));
    return RT_OK;
    RT_GUARD_END(ctx)
}
int rt_frame_download(rt_ctx* ctx, const void* frame_dev, uint8_t* out_rgb, size_t bytes) {
    if (!ctx || !frame_dev || !out_rgb) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpyAsync(out_rgb, frame_dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return RT_OK;
    RT_GUARD_END(ctx)
}
int rt_frame_collect(rt_ctx* ctx, const void* frame_dev, const rt_params* params, uint64_t seq, uint8_t* out_rgb,
                     size_t out_len) {
    if (!ctx || !frame_dev || !params) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    const auto t0 = std::chrono::steady_clock::now();
    if (params->width == 0 || params->height == 0 || seq == 0) return set_err(ctx, RT_ERR_INVALID_ARG, "rt_frame_collect: zero size or seq");
    const int rc = check_frame_out(ctx, out_rgb, out_len, params->width, params->height);
    if (rc) return rc;
    CK(ctx, cudaSetDevice(ctx->device));
    // read only here: the ranks elsewhere render into the frame
    const Frame f = caller_frame(const_cast<void*>(frame_dev), params->width, params->height);
    return collect_frame(ctx, f, seq, out_rgb, nullptr, 0, nullptr, t0);
    RT_GUARD_END(ctx)
}

int rt_frame_wait_consumed(rt_ctx* ctx, const void* frame_dev, size_t frame_bytes, uint64_t seq) {
    if (!ctx || !frame_dev) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    if (seq == 0) return RT_OK;
    CK(ctx, cudaSetDevice(ctx->device));
    const rt_frame_ctl* ctl = reinterpret_cast<const rt_frame_ctl*>((const uint8_t*)frame_dev + rt_frame_ctl_offset(frame_bytes));
    CK(ctx, launch_wait_slab(&ctl->consumed, (unsigned long long)seq, ctx->h_flag, ctx->stream));
    return RT_OK;
    RT_GUARD_END(ctx)
}

int rt_l2_flush(rt_ctx* ctx, size_t bytes, float* ms_out) {
    if (!ctx) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    CK(ctx, cudaSetDevice(ctx->device));
    if (ctx->flush_bytes < bytes) {
        if (ctx->d_flush) CK(ctx, cudaFree(ctx->d_flush));
        ctx->d_flush = nullptr;
        ctx->flush_bytes = 0;
        CK(ctx, cudaMalloc(&ctx->d_flush, bytes));
        ctx->flush_bytes = bytes;
    }
    if (ms_out) CK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    CK(ctx, cudaMemsetAsync(ctx->d_flush, 0, bytes, ctx->stream));  // stream-ordered in front of the next render
    if (ms_out) {
        CK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
        CK(ctx, cudaStreamSynchronize(ctx->stream));
        CK(ctx, cudaEventElapsedTime(ms_out, ctx->ev0, ctx->ev1));
    }
    return RT_OK;
    RT_GUARD_END(ctx)
}

// -------------------------------------------------------------------------------------------------
// FP32 roofline denominator
// -------------------------------------------------------------------------------------------------
int rt_measure_fp32_peak(rt_ctx* ctx, double* tflops_out, float* ms_out) {
    if (!ctx || !tflops_out) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    CK(ctx, cudaSetDevice(ctx->device));
    if (!ctx->d_scratch) CK(ctx, cudaMalloc(&ctx->d_scratch, (size_t)ctx->sm_count * 8 * 256 * sizeof(float)));
    const int iters = 4096;
    float best = std::numeric_limits<float>::max();
    for (int rep = 0; rep < 4; rep++) {
        CK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
        CK(ctx, launch_fp32_peak(ctx->d_scratch, ctx->sm_count, iters, ctx->stream));
        CK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
        CK(ctx, cudaStreamSynchronize(ctx->stream));
        float ms = 0.0f;
        CK(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        if (rep > 0 && ms < best) best = ms;
    }
    const double flops = (double)ctx->sm_count * 8 * 256 * (double)iters * 16 * 8 * 2;
    *tflops_out = flops / (best * 1e-3) / 1e12;
    if (ms_out) *ms_out = best;
    return RT_OK;
    RT_GUARD_END(ctx)
}

}  // extern "C"
