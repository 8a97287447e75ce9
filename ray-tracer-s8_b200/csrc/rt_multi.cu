// rt_multi.cu — one frame on several GPUs from ONE process: the C-ABI form of the controller's fan-out
// (ray-tracer-controller/src/main.rs:47-75: one RenderInfo per slave; :109-119: stitch the slices).
//
// Context i renders the tiles of rank i of n (the rotating interleave of rt_render_tiles_device) of its own copy of the
// scene — the reference replicates the world in every request body too — and stores finished tiles straight into the
// frame that lives in context 0's memory: peer access over NVLink, no staging copy and no collective.  The frame's
// control block counts finished pixels per slab (system-scope releases from every GPU), so the copy of a slab to the
// caller's host buffer starts as soon as all ranks have finished that slab, while the rest of the frame still renders.
#include <algorithm>
#include <cstring>

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
    std::vector<Resolved> r(n);
    for (uint32_t i = 0; i < n; i++) {
        const int rc = resolve(ctxs[i], scenes[i], params, true, &r[i]);
        if (rc) {
            if (i) set_err(c0, rc, "context %u: %s", i, ctxs[i]->err.c_str());
            return rc;
        }
    }
    const uint32_t W = r[0].p.width, H = r[0].p.height;
    const size_t bytes = (size_t)W * H * 3;
    if (out_len != bytes) return set_err(c0, RT_ERR_INVALID_ARG, "out_len %zu != height*width*3 = %zu", out_len, bytes);

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
    LaunchArgs a0;
    a0.row0 = 0;
    a0.row1 = H;
    a0.out_row0 = 0;
    int rc = own_frame(c0, W, H, &a0);
    if (rc) return rc;
    // the counters may have been reset on context 0's stream: every other context's kernel comes after that
    CK(c0, cudaEventRecord(c0->ev_sync, c0->stream));

    std::vector<LaunchInfo> li(n);
    std::vector<LaunchArgs> la(n, a0);
    for (uint32_t i = 0; i < n; i++) {
        rt_ctx* c = ctxs[i];
        CK(c0, cudaSetDevice(c->device));
        if (i) CK(c0, cudaStreamWaitEvent(c->stream, c0->ev_sync, 0));
        la[i].tile_rank = i;
        la[i].tile_ranks = n;
        rc = launch(c, scenes[i], r[i], la[i], &li[i]);
        if (rc) {
            if (i) set_err(c0, rc, "context %u: %s", i, c->err.c_str());
            return rc;
        }
    }
    CK(c0, cudaSetDevice(c0->device));
    // Streaming waits on the device for the other contexts' kernels.  Contexts that share a device also share its
    // hardware queues: a wait kernel could then sit in front of the very kernel it waits for, so such frames are
    // copied after the kernels instead.
    bool streamed = true;
    for (uint32_t i = 0; i < n; i++) {
        streamed = streamed && li[i].counts_done;
        for (uint32_t j = 0; j < i; j++) streamed = streamed && ctxs[i]->device != ctxs[j]->device;
    }
    SlabJob job;
    const bool late = c0->serial_launches;  // blocking launches: the waits go behind the second passes (rt_init)
    if (streamed && !late) {
        rc = enqueue_slab_copies(c0, c0->d_out, a0.ctl, a0.plan, c0->out_seq, out_rgb, &job);
        if (rc) return rc;
    }
    // second passes (tie-break tables that had not landed) and counters, context by context
    uint32_t redone = 0;
    rt_stats sum;
    memset(&sum, 0, sizeof sum);
    for (uint32_t i = 0; i < n; i++) {
        rt_ctx* c = ctxs[i];
        CK(c0, cudaSetDevice(c->device));
        uint32_t rd = 0;
        rc = finish_redo(c, scenes[i], r[i], la[i], &rd);
        if (rc) {
            if (i) set_err(c0, rc, "context %u: %s", i, c->err.c_str());
            return rc;
        }
        redone = (rd == 0xffffffffu || redone == 0xffffffffu) ? 0xffffffffu : redone + rd;
        rt_stats st;
        memset(&st, 0, sizeof st);
        st.redo_pixels = rd;
        rc = finish_stats(c, r[i], (uint64_t)W * H / n, &st, t0, li[i]);
        if (rc) return rc;
        uint64_t* dst = &sum.rays;
        const uint64_t* src = &st.rays;
        for (size_t k = 0; k < offsetof(rt_stats, kernel_ms) / sizeof(uint64_t); k++) dst[k] += src[k];
        sum.kernel_ms = std::max(sum.kernel_ms, st.kernel_ms);
        sum.kernel_launches += st.kernel_launches;
        if (i == 0) {
            sum.intersector_used = st.intersector_used;
            sum.grid_ctas = st.grid_ctas;
            sum.cta_threads = st.cta_threads;
            sum.ctas_per_sm = st.ctas_per_sm;
            sum.scene_in_smem = st.scene_in_smem;
            sum.dyn_smem_bytes = st.dyn_smem_bytes;
        }
    }
    CK(c0, cudaSetDevice(c0->device));
    if (streamed && late) {
        CK(c0, cudaSetDevice(c0->device));
        rc = enqueue_slab_copies(c0, c0->d_out, a0.ctl, a0.plan, c0->out_seq, out_rgb, &job);
        if (rc) return rc;
    }
    if (streamed) {  // every context's held-back pixels are final and counted by now: the last slabs complete
        rc = finish_slab_copies(c0, job);
        if (rc) return rc;
    } else {
        CK(c0, cudaMemcpyAsync(out_rgb, c0->d_out, bytes, cudaMemcpyDeviceToHost, c0->stream));
        CK(c0, cudaStreamSynchronize(c0->stream));
    }
    if (stats) {
        sum.primary = (uint64_t)W * H * r[0].p.spp;
        sum.redo_pixels = redone;
        sum.total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
        *stats = sum;
    }
    return RT_OK;
    RT_GUARD_END(c0)
}
