// rt_host.h — host-side declarations shared by rt_api.cu, rt_scene.cu, rt_multi.cu, rt_kernels.cu and rt_bvh_host.cpp.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/rt_b200.h"

namespace rtb {

struct DevScene;
struct DevCamera;
struct DevParams;

constexpr int MAX_SLABS = 64;  // completion counters per frame (frame control block)

// Measurement switches, read from the environment once per process (rt_init forces the read).  Not API.
struct Tunables {
    int smem_override = -1;      // RT_B200_SMEM=0|1: force the scene out of / into shared memory
    int tile_order_reverse = 1;  // RT_B200_TILE_ORDER=topdown: tickets walk the tile grid top-down
    int stage_out = -1;          // RT_B200_STAGE_OUT=0|1: force the output stage + completion counters off / on (-1: shared frames only)
    int tail_permille = 30;      // RT_B200_TAIL_PERMILLE: share of the tickets handed out pixel by pixel
    int build_mode = 1;          // RT_B200_BUILD=host|device|auto: who builds the traversal tree
    int tree_mode = 2;           // RT_B200_TREE=ref|sah|split: which tree is traversed
    bool timing = false;         // RT_B200_TIMING: stage times of rt_scene_create on stderr
    int slabs = 16;              // RT_B200_SLABS: slabs a frame download is streamed in
    bool async_ref = true;       // RT_B200_ASYNC_REF=0: build the reference-topology tree inside rt_scene_create
    int pid_order = 1;           // RT_B200_PID_ORDER=world: primitive ids in world order instead of the traversal tree's DFS order
    int aux_delay_ms = 0;        // RT_B200_AUX_DELAY_MS: the builder thread sleeps first (tests: frames rendered before the tables land)
    int wait_timeout_ms = 20000; // RT_B200_WAIT_TIMEOUT_MS: how long a frame owner waits for a slab / a rank for the owner
    bool count_done = true;      // RT_B200_COUNT_DONE=0: no completion counters (frames are copied after the kernel)
#ifdef RT_B200_EXPERIMENTS
    int bvh_variant = 3;         // RT_B200_BVH_KERNEL=lanes|simple|pools|deferred|wave|wq
    int sched_minb = 2;
    int w[4] = {1, 1, 1, 1}, node_num = 1, node_den = 2;
    int wave_refill = 8;
    int wq_warps = 24, wq_chains = 128, wq_min_active = 20, wq_min_node = 24, wq_burst = 2, wq_t_leaf = 4, wq_t_pend = 6,
        wq_t_fin = 6, wq_sync = 0, wq_budget = 0, tb_alt = 0, tb_burst = 4;
#endif
};
const Tunables& tunables();

struct LaunchInfo {
    unsigned grid = 0, threads = 0;
    size_t dyn_smem = 0;
    int ctas_per_sm = 0;
    bool scene_in_smem = false;
    unsigned launches = 1;
    bool counts_done = true;  // the kernel keeps the frame's completion counters (the A/B kernels do not)
};

// rt_bvh_device.cu: LBVH + refit of the traversal tree on the device (scratch owned by the context)
struct DeviceBuild {
    void* mem = nullptr;
    size_t bytes = 0;
};
void free_device_build(DeviceBuild* b);
cudaError_t build_lbvh_device(DeviceBuild* buf, const float* h_boxes, const uint32_t* h_pid_of, uint32_t n,
                              float4* lnode, float4* legacy_abc, int2* legacy_d, uint32_t* depth_out, cudaStream_t stream);

// rt_kernels.cu
cudaError_t preload_kernels();
cudaError_t launch_render(const DevScene& sc, const DevCamera& cam, const DevParams& pr, int isect, bool count,
                          int sm_count, int smem_optin, cudaStream_t stream, LaunchInfo* info);
cudaError_t launch_wait_slab(const unsigned long long* done, unsigned long long target, unsigned int* timeout_flag,
                             cudaStream_t stream);
cudaError_t launch_wait_all_slabs(const unsigned long long* done, unsigned long long seq, uint32_t slabs, uint32_t tile_rows,
                                  uint32_t rows, uint32_t width, unsigned int* timeout_flag, cudaStream_t stream);
cudaError_t launch_set_u64(unsigned long long* p, unsigned long long v, cudaStream_t stream);
cudaError_t launch_add_counts(unsigned long long* done, const unsigned long long* add, int n, cudaStream_t stream);
cudaError_t launch_fp32_peak(float* scratch, int sm_count, int iters, cudaStream_t stream);
// rows * width * 3 floats: sum / samples of each pixel's state record (rt_accum_read_linear)
cudaError_t launch_accum_linear(const void* state, float* out, unsigned long long pixels, uint32_t samples, int sm_count,
                                cudaStream_t stream);
size_t scene_smem_bytes(const DevScene& sc, int isect);

#ifdef RT_B200_EXPERIMENTS
// device buffers of the wavefront pipeline (owned by the context, grown on demand)
struct WaveBuffers {
    void* slots = nullptr;          // WSlot[capacity]
    uint32_t* q_ray = nullptr;      // [capacity] each
    uint32_t* q_hit = nullptr;
    uint32_t* q_miss = nullptr;
    uint32_t* path_ext = nullptr;   // [(ext_depth) * capacity] path entries beyond the 8 kept in the slot
    void* counters = nullptr;       // WaveCounters[2]
    size_t capacity = 0, ext_entries = 0;
};
void free_wave_buffers(WaveBuffers* wb);
// device buffer of the warp-private wavefront kernel: per-chain state (rt_kernel_wq.cuh), grown on demand
struct WqBuffers {
    void* state = nullptr;
    size_t bytes = 0;
};
void free_wq_buffers(WqBuffers* b);
struct ExperimentBuffers {
    WaveBuffers wave;
    WqBuffers wq;
};
void set_experiment_buffers(ExperimentBuffers* b);  // the context whose launch follows (single-threaded tooling)
void free_experiment_buffers(ExperimentBuffers* b);
bool legacy_node_arrays_needed();  // true when RT_B200_BVH_KERNEL selects a kernel that reads node_* / cnode_*
cudaError_t launch_trace_bench(const DevScene& sc, int variant, bool with_big, const float4* rays, unsigned long long n,
                               unsigned long long* ticket, int2* out, int sm_count, int smem_optin, cudaStream_t stream);
cudaError_t sort_rays_device(const float4* rays, unsigned long long n, const float lo[3], const float hi[3], float4* out,
                             cudaStream_t stream);
#endif

// ---- rt_bvh_host.cpp: SAH BVH with the reference's topology ------------------------------------------
struct Box {
    float min[3], max[3];
};
struct HostNode {       // inner node; children are codes: >= 0 inner index, < 0 leaf of world position ~code
    Box box_l, box_r;
    int32_t left, right;
};
struct HostBVH {
    std::vector<HostNode> inner;        // DFS pre-order
    std::vector<uint32_t> leaf_order;   // rank → world position
    int32_t root = 0;                   // code
    uint32_t depth = 0;                 // deepest leaf (root = 0)
    uint32_t node_count = 0;            // inner + leaves, = 2n-1
};
// boxes[i] = AABB of the primitive at world position i.  Returns false (with a message) when the
// reference's build would panic or never terminate.
bool build_bvh(const std::vector<Box>& boxes, HostBVH* out, std::string* err);
// 3-axis, 16-bin SAH tree over the same primitives, for culling only (leaf order is NOT the reference's).
bool build_bvh_sah(const std::vector<Box>& boxes, HostBVH* out);

}  // namespace rtb
