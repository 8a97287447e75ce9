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
    uint32_t* d_bands = nullptr;  // band table of rt_render_divisions' banded launches
    size_t d_bands_cap = 0;       // entries
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
    rtb::DeviceBuild dbuild;
    // scene upload: one pinned staging buffer the blob is assembled in, and a few retired device blobs kept for the
    // next rt_scene_create (a slave makes one scene per job: cudaMalloc/cudaFree per job were a third of a small job)
    uint8_t* h_stage = nullptr;
    size_t h_stage_bytes = 0;
    struct Retired { uint8_t* p; size_t cap; };
    std::vector<Retired> retired;
    std::vector<void*> host_allocs;  // rt_host_alloc'ed buffers still alive (freed at shutdown)
    uint8_t* d_jpeg = nullptr;       // JPEG encoder scratch (rt_jpeg.cu): coefficients, bit offsets, coded and stuffed bytes
    size_t d_jpeg_bytes = 0;
    unsigned long long* h_jpeg_len = nullptr;  // pinned: length of the last encoded segment
    uint8_t* d_wire = nullptr;       // wire format scratch (rt_wire.cu): the world's text and records, ImageSlice bodies
    size_t d_wire_bytes = 0;
    unsigned long long* h_wire = nullptr;  // pinned: a parse's outcome (array end, decline, sphere count)
    uint8_t* d_obj = nullptr;        // OBJ ingest scratch (rt_obj.cu): the body's text, its lines, vertices, corners, triangles
    size_t d_obj_bytes = 0;
    unsigned long long* h_obj = nullptr;   // pinned: counts and the decline flag between the stages of a parse
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
    // inputs (owned; rt_scene_update replaces boxes once the thread has been joined)
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
    std::unique_ptr<rt_aux> aux;
    uint64_t serial = 0;  // unique per process (rt_scene_create, rt_scene_update): a re-created scene may reuse a destroyed
                          // one's address, an updated one keeps its own
    // the topology rt_scene_update keeps (the traversal tree's lni / lroot / ltree are in dev)
    std::vector<uint32_t> world_index;  // as given to rt_scene_create (empty: none)
    std::vector<uint32_t> big_world;    // world positions of the primitives kept out of the traversal tree
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

// A frame buffer on the device (possibly a peer's) with its control block and slab plan.
struct Frame {
    uint8_t* dev = nullptr;
    rt_frame_ctl* ctl = nullptr;  // nullable: no completion counting
    SlabPlan plan;
};
// The context's own staging frame for `rows` rows, its counters reset on ctx->stream: its frame number is always
// OWN_FRAME_SEQ (see own_frame in rt_api.cu).
constexpr uint64_t OWN_FRAME_SEQ = 1;
int own_frame(rt_ctx* ctx, uint32_t width, uint32_t rows, Frame* f);
// A caller's whole frame of width x height (rt_frame_alloc / rt_frame_open): the control block follows the pixels.
Frame caller_frame(void* frame_dev, uint32_t width, uint32_t height);
// out_rgb (nullable: no download) must hold a whole frame of width x height.
int check_frame_out(rt_ctx* ctx, const uint8_t* out_rgb, size_t out_len, uint32_t width, uint32_t height);

struct LaunchArgs {
    uint32_t row0 = 0, row1 = 0, tile_rank = 0, tile_ranks = 1;
    Frame frame;                  // where the launch's rows go
    uint32_t out_row0 = 0;
    bool stream = false;          // the frame goes to the host slab by slab while it renders (stage + counters wanted)
    const unsigned int* pixel_list = nullptr;  // redo launch: render exactly these pixels (y * width + x)
    uint32_t list_count = 0;
    const void* state_in = nullptr;  // resumable chains (rt_render_samples): samples [s0, spp) from state_in to state_out
    void* state_out = nullptr;
    uint32_t s0 = 0;
    const uint32_t* band_table = nullptr;  // banded launch (rt_render_divisions): row0 = 0, rows = bands of band_rows
    uint32_t band_rows = 0;                // stacked in table order (device memory of the context, see DevParams)
};
// Launches the render on ctx->stream; timing events ev0 / ev1 are recorded around the kernel.
int launch(rt_ctx* ctx, const rt_scene* scene, const Resolved& r, const LaunchArgs& a, LaunchInfo* info);

// One context's launch towards a frame, and what it reports: `info` from launch(), `st` from its finish (rt_api.cu).
struct Launch {
    rt_ctx* ctx = nullptr;
    const rt_scene* scene = nullptr;
    Resolved r;
    LaunchArgs a;
    LaunchInfo info;
    rt_stats st{};
};
// The frame owner's sequence, on `owner` (the context whose memory holds frame f): launches the n entries of l (none:
// the frame is rendered by ranks elsewhere), streams frame number `seq` of f to out_rgb (nullptr: none) slab by slab
// while it renders, finishes every launch (second pass, statistics) and returns when the whole frame is in out_rgb.
// Errors of a launch on another context are reported on `owner` as "context i: ...".  stats (nullable; filled when
// n >= 1): the launches' statistics combined, total_ms counted from t0.
int collect_frame(rt_ctx* owner, const Frame& f, uint64_t seq, uint8_t* out_rgb, Launch* l, uint32_t n, rt_stats* stats,
                  std::chrono::steady_clock::time_point t0);

// JPEG (rt_jpeg.cu).  jpeg_check: the refusals shared by every JPEG entry (NULL out, size, quality, out_cap below
// rt_jpeg_bound).  jpeg_encode_device: encodes the width x height RGB8 frame at rgb_dev (device memory of ctx, ordered
// on ctx->stream) into out (checked by jpeg_check) and returns when out holds all *out_len bytes; ms_out (nullable): the
// device time of the encode.
int jpeg_check(rt_ctx* ctx, uint32_t width, uint32_t height, uint32_t quality, const uint8_t* out, size_t out_cap,
               const size_t* out_len);
int jpeg_encode_device(rt_ctx* ctx, const uint8_t* rgb_dev, uint32_t width, uint32_t height, uint32_t quality,
                       uint8_t* out, size_t* out_len, float* ms_out);
cudaError_t jpeg_preload();
// In place: sums[0..n) → their exclusive sum, sums[n] = the total (the carry pass behind the CTA scans of rt_jpeg.cu and
// rt_wire.cu), on stream s.
cudaError_t scan_carry(unsigned long long* sums, uint32_t n, cudaStream_t s);

// Wire format (rt_wire.cu).  slice_json_check: the refusals of rt_render_divisions_json beyond those of
// rt_render_divisions.  slice_json_device: the ImageSlice bodies of the n bands of rows x width stacked at rgb_dev (device
// memory of ctx, ordered on ctx->stream), band k with division_no division_nos[k], packed into out with their lengths in
// out_lens; returns when both are complete.
cudaError_t wire_preload();
int slice_json_check(rt_ctx* ctx, uint32_t n, uint32_t rows, uint32_t width, const char* id, const uint8_t* out,
                     size_t out_cap, const size_t* out_lens);
int slice_json_device(rt_ctx* ctx, const uint8_t* rgb_dev, uint32_t n, uint32_t rows, uint32_t width,
                      const uint32_t* division_nos, const char* id, uint8_t* out, size_t* out_lens);

// OBJ ingest (rt_obj.cu).
cudaError_t obj_preload();

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
    // the tile share of the chunks since the last create / reset (tile_ranks 0: none yet): rt_render_samples is rank 0
    // of 1; rank i of n (rt_render_samples_multi) holds the chains of that rank's tiles only
    uint32_t tile_rank = 0, tile_ranks = 0;
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
