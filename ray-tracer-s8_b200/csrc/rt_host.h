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
struct Box;

constexpr int MAX_SLABS = 64;  // completion counters per frame (frame control block)

// Test hooks, read from the environment once per process (rt_init forces the read).  They let tests reach paths a
// normal run does not take on a given machine or at a given moment; they are not API.
struct TestHooks {
    int build_mode = 1;          // RT_B200_BUILD=host|device|auto: who builds the traversal tree
    int aux_delay_ms = 0;        // RT_B200_AUX_DELAY_MS: the builder thread sleeps first (frames rendered before the tables land)
    int wait_timeout_ms = 20000; // RT_B200_WAIT_TIMEOUT_MS: how long a frame owner waits for a slab / a rank for the owner
    bool no_stream_wait = false; // RT_B200_NO_STREAM_WAIT: slab waits as one-thread kernels instead of cuStreamWaitValue64
};
const TestHooks& test_hooks();

struct LaunchInfo {
    unsigned grid = 0, threads = 0;
    size_t dyn_smem = 0;
    int ctas_per_sm = 0;
    bool scene_in_smem = false;
    bool counts_done = true;  // the kernel keeps the frame's completion counters
};

// rt_bvh_device.cu: LBVH + refit of the traversal tree on the device (scratch owned by the context)
struct DeviceBuild {
    void* mem = nullptr;
    size_t bytes = 0;
};
void free_device_build(DeviceBuild* b);
cudaError_t build_lbvh_device(DeviceBuild* buf, const Box* h_boxes, const uint32_t* h_pid_of, uint32_t n,
                              float4* lnode, uint32_t* depth_out, cudaStream_t stream);

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
