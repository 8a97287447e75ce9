// rt_ctx.h — the objects behind the opaque handles of include/rt_b200.h (shared by rt_api.cu, rt_scene.cu, rt_multi.cu).
#pragma once
#include <atomic>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "rt_device.cuh"
#include "rt_host.h"

// Control block behind every frame buffer (rt_frame_alloc and the context's own staging frame): per-slab counts of the
// pixels written so far, cumulative over the frames rendered into the buffer (frame number `seq` of a slab is complete
// when its counter reaches seq * pixels_in_slab), so no rank ever has to reset a counter another rank may be adding to.
struct rt_frame_ctl {
    unsigned long long done[rtb::MAX_SLABS];
    unsigned long long consumed;  // frames the owner has finished collecting (written by the owner, polled by the ranks
                                  // before they overwrite the buffer: rt_frame_wait_consumed)
};
constexpr size_t RT_FRAME_CTL_BYTES = 1024;
static_assert(sizeof(rt_frame_ctl) <= RT_FRAME_CTL_BYTES, "control block size");
inline size_t rt_frame_ctl_offset(size_t frame_bytes) { return (frame_bytes + 255) / 256 * 256; }

struct rt_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;       // render stream
    cudaStream_t copy_stream = nullptr;  // slab waits + device→host copies, concurrent with the render kernel
    cudaStream_t aux_stream = nullptr;   // late upload of the tie-break tables by the scene's builder thread
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_sync = nullptr;
    int sm_count = 0, clock_khz = 0, smem_optin = 0;
    char name[64] = {0};
    uint8_t* d_out = nullptr;  // band / frame staging in HBM + control block
    size_t d_out_bytes = 0;    // capacity for pixels (the control block follows at rt_frame_ctl_offset(capacity))
    uint64_t out_seq = 1;      // frame number the counters of d_out count towards (reset per launch: always 1)
    unsigned long long* d_ctr = nullptr;  // NUM_COUNTERS counters | 2 tickets (one u64) | redo count (one u64)
    unsigned long long* h_ctr = nullptr;  // pinned mirror
    unsigned int* d_redo = nullptr;       // pixels to render again once the tie-break tables are up (REDO_CAP entries)
    unsigned int* h_flag = nullptr;       // pinned + mapped: [0] a slab wait timed out
    // cuStreamWaitValue64 (driver entry point, resolved in rt_init; null: not available → wait kernels): a stream waits
    // for a counter in device memory without occupying an SM — the render kernel leaves no room for a waiting kernel
    // (1024 threads x 64 registers = the whole register file of every SM)
    int (*stream_wait_value64)(void* stream, unsigned long long addr, unsigned long long value, unsigned int flags) = nullptr;
    bool serial_launches = false;         // kernel launches block the host (profiler, CUDA_LAUNCH_BLOCKING): see rt_init
    uint8_t* h_frame = nullptr;           // pinned staging for frames streamed to a pageable destination
    size_t h_frame_bytes = 0;
    std::vector<cudaEvent_t> slab_events; // one per slab, for the pageable path's per-slab host copies
    float* d_scratch = nullptr;
    void* d_flush = nullptr;              // rt_l2_flush: a buffer larger than L2
    size_t flush_bytes = 0;
    float first_pass_ms = 0.0f;           // kernel time of the first pass when a second one followed (finish_redo)
    rtb::DeviceBuild dbuild;
    // scene upload: one pinned staging buffer the blob is assembled in, and a few retired device blobs kept for the
    // next rt_scene_create (a slave makes one scene per job: cudaMalloc/cudaFree per job were a third of a small job)
    uint8_t* h_stage = nullptr;
    size_t h_stage_bytes = 0;
    struct Retired { uint8_t* p; size_t cap; };
    std::vector<Retired> retired;
    std::vector<void*> host_allocs;  // rt_host_alloc'ed buffers still alive (freed at shutdown)
    std::string err;
};
constexpr uint32_t RT_REDO_CAP = 1u << 16;
constexpr int RT_CTR_TICKETS = rtb::NUM_COUNTERS;      // two 32-bit tickets: whole tiles | the tail's pixels
constexpr int RT_CTR_TICKET2 = rtb::NUM_COUNTERS + 1;  // 32-bit ticket: redo-list entries taken inside the kernel (| pad)
constexpr int RT_CTR_REDO = rtb::NUM_COUNTERS + 2;     // pixels appended to the redo list
constexpr int RT_CTR_REDO_SLAB = rtb::NUM_COUNTERS + 3;  // MAX_SLABS per-slab counts of pixels still held back
constexpr int RT_CTR_SLOTS = rtb::NUM_COUNTERS + 3 + rtb::MAX_SLABS;

// The reference-topology tree (bvh_impl.rs:229-364) is needed only to break exact-distance ties (its DFS leaf order,
// shapes/mod.rs:177-182) and for rays with a zero direction component (ancestor boxes, ray.rs:174-194).  It is built
// beside the upload by a thread of its own; its tables reach the device when they are ready.
struct rt_aux {
    std::thread worker;
    std::atomic<int> state{0};  // 0 running, 1 tables on the device, -1 failed
    std::string err;
    // inputs (owned)
    std::vector<rtb::Box> boxes;            // by world position
    std::vector<uint32_t> pid_of_world;
    // outputs
    std::vector<uint32_t> rank_by_world;    // world position → DFS leaf rank
    uint32_t n_nodes = 0, depth = 0;
};

struct rt_scene {
    rt_ctx* ctx = nullptr;
    uint8_t* d_blob = nullptr;
    size_t blob_bytes = 0, blob_cap = 0;
    rtb::DevScene dev{};
    uint32_t n = 0;
    uint32_t tree_depth = 0;   // depth of the tree the kernels traverse
    bool device_tree = false;  // it was built on the device (LBVH)
    size_t o_rank = 0, o_up = 0, o_refbox = 0;  // blob offsets of the late tables
    std::unique_ptr<rt_aux> aux;
    uint64_t serial = 0;  // unique per process (rt_scene_create): a re-created scene may reuse a destroyed one's address
};

namespace rtb {

int set_err(rt_ctx* ctx, int code, const char* fmt, ...);
// Blocks until the scene's tie-break tables are on the device (or their build failed: returns the status).
int scene_settle(rt_ctx* ctx, const rt_scene* scene);
// DevScene to launch with right now: aux_ready reflects whether the tables have landed.
DevScene scene_view(const rt_scene* scene);

struct Resolved {
    rt_params p;
    DevCamera cam;
    int isect;
};
int resolve(rt_ctx* ctx, const rt_scene* scene, const rt_params* in, bool whole_frame, Resolved* r);
// resolve() without a scene: every check and default except the intersector's pick (r->isect is left unset)
int resolve_params(rt_ctx* ctx, const rt_params* in, bool whole_frame, Resolved* r);

// slab geometry of a launch that renders `rows` image rows: slabs of `tile_rows` tile rows each
struct SlabPlan {
    uint32_t slabs = 1, tile_rows = 1;
    uint32_t width = 0, rows = 0;
    uint32_t first_row(uint32_t s) const { return std::min(rows, s * tile_rows * (uint32_t)TILE_H); }
    uint32_t row_count(uint32_t s) const { return first_row(s + 1) - first_row(s); }
    unsigned long long pixels(uint32_t s) const { return (unsigned long long)row_count(s) * width; }
};
SlabPlan plan_slabs(uint32_t width, uint32_t rows);

struct LaunchArgs {
    uint32_t row0 = 0, row1 = 0, tile_rank = 0, tile_ranks = 1;
    uint8_t* dst = nullptr;       // frame / band buffer (device, possibly a peer's)
    uint32_t out_row0 = 0;
    rt_frame_ctl* ctl = nullptr;  // its control block (nullable: no completion counting)
    SlabPlan plan;
    bool stream = false;          // the frame goes to the host slab by slab while it renders (stage + counters wanted)
    const unsigned int* pixel_list = nullptr;  // redo launch: render exactly these pixels (y * width + x)
    uint32_t list_count = 0;
    const void* state_in = nullptr;  // resumable chains (rt_render_samples): samples [s0, spp) from state_in to state_out
    void* state_out = nullptr;
    uint32_t s0 = 0;
};
// The context's own staging frame (+ control block) for a launch of `rows` rows: fills dst / ctl / plan, bumps out_seq.
int own_frame(rt_ctx* ctx, uint32_t width, uint32_t rows, LaunchArgs* a);
// Launches the render on ctx->stream; timing events ev0 / ev1 are recorded around the kernel.
int launch(rt_ctx* ctx, const rt_scene* scene, const Resolved& r, const LaunchArgs& a, LaunchInfo* info);
// After the kernel of `launch` has completed: re-renders the pixels that needed the tie-break tables before they had
// landed (waits for the tables).  *redone = number of pixels rendered again.
int finish_redo(rt_ctx* ctx, const rt_scene* scene, const Resolved& r, const LaunchArgs& a, uint32_t* redone);
int finish_stats(rt_ctx* ctx, const Resolved& r, uint64_t pixels, rt_stats* st,
                 std::chrono::steady_clock::time_point t0, const LaunchInfo& li);
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
int enqueue_slab_copies(rt_ctx* ctx, const uint8_t* frame_dev, const rt_frame_ctl* ctl, const SlabPlan& plan, uint64_t seq,
                        uint8_t* out_rgb, SlabJob* job);
int finish_slab_copies(rt_ctx* ctx, const SlabJob& job);

}  // namespace rtb

// Sample state of the rows of one frame or division (rt_accum_create).  Two buffers of STATE_RECORD_BYTES per pixel: a
// chunk reads state[cur] and writes state[cur ^ 1], and cur flips only when the chunk has succeeded, so a second pass
// (which starts over from state[cur]) and a failed call both leave the chain where it was.
struct rt_accum {
    rt_ctx* ctx = nullptr;
    rt_params params{};         // as bound (spp and collect_counters ignored); resolved against the scene per chunk
    uint32_t row0 = 0, row1 = 0;
    void* state[2] = {nullptr, nullptr};
    int cur = 0;
    uint32_t samples = 0;       // samples of every pixel's chain done so far
    uint64_t scene_serial = 0;  // the scene of the chunks since the last create / reset (0: none yet)
};

#define CK(ctx, call)                                                                                        \
    do {                                                                                                     \
        cudaError_t e__ = (call);                                                                            \
        if (e__ != cudaSuccess)                                                                              \
            return rtb::set_err(ctx, RT_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__),   \
                                __FILE__, __LINE__);                                                         \
    } while (0)

// Every extern "C" entry runs its body inside this guard: nothing unwinds across the C boundary.
#define RT_GUARD_BEGIN try {
#define RT_GUARD_END(ctx)                                                                          \
    }                                                                                              \
    catch (const std::bad_alloc&) { return rtb::set_err(ctx, RT_ERR_NOMEM, "out of host memory"); } \
    catch (const std::exception& ex__) { return rtb::set_err(ctx, RT_ERR_INTERNAL, "internal error: %s", ex__.what()); } \
    catch (...) { return rtb::set_err(ctx, RT_ERR_INTERNAL, "internal error"); }
