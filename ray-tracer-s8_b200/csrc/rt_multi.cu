// rt_multi.cu — one frame on several GPUs from ONE process: the C-ABI form of the controller's fan-out
// (ray-tracer-controller/src/main.rs:47-75: one RenderInfo per slave; :109-119: stitch the slices).
//
// Context i renders the tiles of rank i of n (the rotating interleave of rt_render_tiles_device) of its own copy of the
// scene — the reference replicates the world in every request body too — and stores finished tiles straight into the
// frame that lives in context 0's memory: peer access over NVLink, no staging copy and no collective.  The frame's
// control block counts finished pixels per slab (system-scope releases from every GPU), so the copy of a slab to the
// caller's host buffer starts as soon as all ranks have finished that slab, while the rest of the frame still renders.
// rt_render_samples_multi is the same frame rendered in chunks of samples: each context resumes its tiles' chains.
// rt_render_frame_jpeg renders the frame (on one context or on n) and encodes it where it lies, in context 0's memory.
#include <cstring>
#include <vector>

#include "rt_ctx.h"

using namespace rtb;

namespace {

// The n launches of l towards one frame of width x height in context 0's memory (its staging frame): peer access from
// every other context's device to context 0's, the frame's counters reset on context 0's stream in front of every
// context's launch, and each launch's rows, tile share and frame set.
int shared_frame(rt_ctx* const* ctxs, uint32_t n, uint32_t width, uint32_t height, Launch* l) {
    rt_ctx* const c0 = ctxs[0];
    for (uint32_t i = 1; i < n; i++) {
        if (ctxs[i]->device == c0->device) continue;
        CK(c0, cudaSetDevice(ctxs[i]->device));
        int can = 0;
        CK(c0, cudaDeviceCanAccessPeer(&can, ctxs[i]->device, c0->device));
        if (!can) return set_err(c0, RT_ERR_UNSUPPORTED, "device %d cannot access device %d's memory", ctxs[i]->device, c0->device);
        const cudaError_t e = cudaDeviceEnablePeerAccess(c0->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
            return set_err(c0, RT_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d → %d): %s", ctxs[i]->device, c0->device, cudaGetErrorString(e));
        (void)cudaGetLastError();
    }
    CK(c0, cudaSetDevice(c0->device));
    Frame f;
    const int rc = own_frame(c0, width, height, &f);
    if (rc) return rc;
    // the counters may have been reset on context 0's stream: every other context's kernel comes after that
    CK(c0, cudaEventRecord(c0->ev_sync, c0->stream));
    for (uint32_t i = 1; i < n; i++) {
        CK(c0, cudaSetDevice(ctxs[i]->device));
        CK(c0, cudaStreamWaitEvent(ctxs[i]->stream, c0->ev_sync, 0));
    }
    CK(c0, cudaSetDevice(c0->device));
    for (uint32_t i = 0; i < n; i++) {
        l[i].a.row1 = height;
        l[i].a.tile_rank = i;
        l[i].a.tile_ranks = n;
        l[i].a.frame = f;
    }
    return RT_OK;
}

// What an accum binds that decides the frame (spp, collect_counters and the band are checked elsewhere).
bool same_binding(const rt_params& a, const rt_params& b) {
    return a.width == b.width && a.height == b.height && a.max_bounces == b.max_bounces && a.seed == b.seed &&
           !memcmp(a.cam_origin, b.cam_origin, sizeof a.cam_origin) && !memcmp(&a.aperture, &b.aperture, sizeof(float)) &&
           !memcmp(&a.focus_distance, &b.focus_distance, sizeof(float)) &&
           !memcmp(&a.field_of_view, &b.field_of_view, sizeof(float)) &&
           !memcmp(&a.focal_length, &b.focal_length, sizeof(float)) && a.intersector == b.intersector && a.flags == b.flags;
}

}  // namespace

extern "C" int rt_render_frame_multi(rt_ctx* const* ctxs, const rt_scene* const* scenes, uint32_t n, const rt_params* params,
                                     uint8_t* out_rgb, size_t out_len, rt_stats* stats) {
    if (!ctxs || !scenes || n == 0 || !ctxs[0]) return RT_ERR_INVALID_ARG;
    rt_ctx* const c0 = ctxs[0];
    RT_GUARD_BEGIN
    const auto t0 = std::chrono::steady_clock::now();
    for (uint32_t i = 0; i < n; i++)
        if (!ctxs[i] || !scenes[i]) return set_err(c0, RT_ERR_INVALID_ARG, "rt_render_frame_multi: NULL context or scene %u", i);
    if (!out_rgb) return set_err(c0, RT_ERR_INVALID_ARG, "out_rgb is NULL");
    std::vector<Launch> l;
    for (uint32_t i = 0; i < n; i++) {
        l.push_back({ctxs[i], scenes[i]});
        const int rc = resolve(ctxs[i], scenes[i], params, true, &l[i].r);
        if (rc) {
            if (i) set_err(c0, rc, "context %u: %s", i, ctxs[i]->err.c_str());
            return rc;
        }
    }
    const uint32_t W = l[0].r.p.width, H = l[0].r.p.height;
    int rc = check_frame_out(c0, out_rgb, out_len, W, H);
    if (rc) return rc;
    rc = shared_frame(ctxs, n, W, H, l.data());
    if (rc) return rc;
    return collect_frame(c0, l[0].a.frame, OWN_FRAME_SEQ, out_rgb, l.data(), n, stats, t0);
    RT_GUARD_END(c0)
}

extern "C" int rt_render_samples_multi(rt_ctx* const* ctxs, const rt_scene* const* scenes, rt_accum* const* accs, uint32_t n,
                                       uint32_t n_samples, uint8_t* out_rgb, size_t out_len, rt_stats* stats) {
    if (!ctxs || !scenes || !accs || n == 0 || !ctxs[0]) return RT_ERR_INVALID_ARG;
    rt_ctx* const c0 = ctxs[0];
    RT_GUARD_BEGIN
    const auto t0 = std::chrono::steady_clock::now();
    for (uint32_t i = 0; i < n; i++)
        if (!ctxs[i] || !scenes[i] || !accs[i])
            return set_err(c0, RT_ERR_INVALID_ARG, "rt_render_samples_multi: NULL context, scene or accum %u", i);
    const rt_accum* const a0 = accs[0];
    if (n_samples == 0) return set_err(c0, RT_ERR_INVALID_ARG, "rt_render_samples_multi: n_samples is 0");
    if ((uint64_t)a0->samples + n_samples > 0xffffffffull)
        return set_err(c0, RT_ERR_INVALID_ARG, "rt_render_samples_multi: %u + %u samples overflow 32 bits", a0->samples, n_samples);
    for (uint32_t i = 0; i < n; i++) {
        const rt_accum* const a = accs[i];
        if (a->ctx != ctxs[i]) return set_err(c0, RT_ERR_INVALID_ARG, "rt_render_samples_multi: accum %u is of another context", i);
        if (a->row0 != 0 || a->row1 != a->params.height)
            return set_err(c0, RT_ERR_INVALID_ARG, "rt_render_samples_multi: accum %u holds rows [%u, %u), not the whole frame", i,
                           a->row0, a->row1);
        if (a->tile_ranks && (a->tile_rank != i || a->tile_ranks != n))
            return set_err(c0, RT_ERR_INVALID_ARG, "rt_render_samples_multi: accum %u holds rank %u of %u, not %u of %u until reset",
                           i, a->tile_rank, a->tile_ranks, i, n);
        if (!same_binding(a->params, a0->params))
            return set_err(c0, RT_ERR_INVALID_ARG, "rt_render_samples_multi: accum %u is bound to other params than accum 0", i);
        if (a->samples != a0->samples)
            return set_err(c0, RT_ERR_INVALID_ARG, "rt_render_samples_multi: accum %u has %u samples, accum 0 %u", i, a->samples,
                           a0->samples);
        if (a->samples && scenes[i]->serial != a->scene_serial)
            return set_err(c0, RT_ERR_INVALID_ARG,
                           "rt_render_samples_multi: scene %u is not the scene of the chunks since the last create / reset", i);
    }
    std::vector<Launch> l;
    for (uint32_t i = 0; i < n; i++) {
        rt_params p = accs[i]->params;
        p.spp = a0->samples + n_samples;
        l.push_back({ctxs[i], scenes[i]});
        const int rc = resolve(ctxs[i], scenes[i], &p, true, &l[i].r);
        if (rc) {
            if (i) set_err(c0, rc, "context %u: %s", i, ctxs[i]->err.c_str());
            return rc;
        }
    }
    const uint32_t W = l[0].r.p.width, H = l[0].r.p.height;
    int rc = check_frame_out(c0, out_rgb, out_len, W, H);
    if (rc) return rc;
    rc = shared_frame(ctxs, n, W, H, l.data());
    if (rc) return rc;
    for (uint32_t i = 0; i < n; i++) {
        l[i].a.state_in = accs[i]->state[accs[i]->cur];
        l[i].a.state_out = accs[i]->state[accs[i]->cur ^ 1];
        l[i].a.s0 = a0->samples;
    }
    rc = collect_frame(c0, l[0].a.frame, OWN_FRAME_SEQ, out_rgb, l.data(), n, stats, t0);
    if (rc) return rc;
    // every chain has advanced: only now does any accum move (on an error above none did)
    for (uint32_t i = 0; i < n; i++) {
        rt_accum* const a = accs[i];
        a->cur ^= 1;
        a->samples += n_samples;
        a->scene_serial = scenes[i]->serial;
        a->tile_rank = i;
        a->tile_ranks = n;
    }
    return RT_OK;
    RT_GUARD_END(c0)
}

extern "C" int rt_render_frame_jpeg(rt_ctx* const* ctxs, const rt_scene* const* scenes, uint32_t n, const rt_params* params,
                                    uint32_t quality, uint8_t* out, size_t out_cap, size_t* out_len, rt_stats* stats) {
    if (!ctxs || !scenes || n == 0 || !ctxs[0]) return RT_ERR_INVALID_ARG;
    rt_ctx* const c0 = ctxs[0];
    RT_GUARD_BEGIN
    const auto t0 = std::chrono::steady_clock::now();
    for (uint32_t i = 0; i < n; i++)
        if (!ctxs[i] || !scenes[i]) return set_err(c0, RT_ERR_INVALID_ARG, "rt_render_frame_jpeg: NULL context or scene %u", i);
    std::vector<Launch> l;
    for (uint32_t i = 0; i < n; i++) {
        l.push_back({ctxs[i], scenes[i]});
        const int rc = resolve(ctxs[i], scenes[i], params, true, &l[i].r);
        if (rc) {
            if (i) set_err(c0, rc, "context %u: %s", i, ctxs[i]->err.c_str());
            return rc;
        }
    }
    const uint32_t W = l[0].r.p.width, H = l[0].r.p.height;
    int rc = jpeg_check(c0, W, H, quality, out, out_cap, out_len);
    if (rc) return rc;
    // the frame stays in context 0's staging frame: with no host destination a single launch does not stream
    if (n == 1) {
        CK(c0, cudaSetDevice(c0->device));
        l[0].a.row1 = H;
        rc = own_frame(c0, W, H, &l[0].a.frame);
    } else {
        rc = shared_frame(ctxs, n, W, H, l.data());
    }
    if (rc) return rc;
    rc = collect_frame(c0, l[0].a.frame, OWN_FRAME_SEQ, nullptr, l.data(), n, stats, t0);
    if (rc) return rc;
    for (uint32_t i = 1; i < n; i++) {  // the encode on context 0's stream comes after every rank's last store
        CK(c0, cudaSetDevice(ctxs[i]->device));
        CK(c0, cudaEventRecord(ctxs[i]->ev_sync, ctxs[i]->stream));
        CK(c0, cudaSetDevice(c0->device));
        CK(c0, cudaStreamWaitEvent(c0->stream, ctxs[i]->ev_sync, 0));
    }
    rc = jpeg_encode_device(c0, l[0].a.frame.dev, W, H, quality, out, out_len, nullptr);
    if (rc) return rc;
    if (stats) stats->total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return RT_OK;
    RT_GUARD_END(c0)
}
