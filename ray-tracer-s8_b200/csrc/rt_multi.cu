// rt_multi.cu — one frame on several GPUs from ONE process: the C-ABI form of the controller's fan-out
// (ray-tracer-controller/src/main.rs:47-75: one RenderInfo per slave; :109-119: stitch the slices).
//
// Context i renders the tiles of rank i of n (the rotating interleave of rt_render_tiles_device) of its own copy of the
// scene — the reference replicates the world in every request body too — and stores finished tiles straight into the
// frame that lives in context 0's memory: peer access over NVLink, no staging copy and no collective.  The frame's
// control block counts finished pixels per slab (system-scope releases from every GPU), so the copy of a slab to the
// caller's host buffer starts as soon as all ranks have finished that slab, while the rest of the frame still renders.
#include <vector>

#include "rt_ctx.h"

using namespace rtb;

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

    // peer access to the frame owner
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

    // the frame: context 0's staging frame and its control block
    CK(c0, cudaSetDevice(c0->device));
    Frame f;
    rc = own_frame(c0, W, H, &f);
    if (rc) return rc;
    // the counters may have been reset on context 0's stream: every other context's kernel comes after that
    CK(c0, cudaEventRecord(c0->ev_sync, c0->stream));
    for (uint32_t i = 1; i < n; i++) {
        CK(c0, cudaSetDevice(ctxs[i]->device));
        CK(c0, cudaStreamWaitEvent(ctxs[i]->stream, c0->ev_sync, 0));
    }
    for (uint32_t i = 0; i < n; i++) {
        l[i].a.row1 = H;
        l[i].a.tile_rank = i;
        l[i].a.tile_ranks = n;
        l[i].a.frame = f;
    }
    return collect_frame(c0, f, OWN_FRAME_SEQ, out_rgb, l.data(), n, stats, t0);
    RT_GUARD_END(c0)
}
