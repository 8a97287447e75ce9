// rt_bvh_device.cu — device-side build and refit of the TRAVERSAL tree (SURVEY.md §8f row f3): Morton-code LBVH
// (Karras 2012: one thread per inner node finds its key range and split from common prefixes) + bottom-up refit.  The
// refit reads nothing but the scene blob (child codes of the node records, exact leaf boxes), so it serves any tree in
// it: the LBVH below, and rt_scene_update's refit of a host-built or device-built tree to moved primitives.
//
// What it replaces: the host's 3-axis binned-SAH build of the product kernels' culling tree (rt_bvh_host.cpp,
// build_bvh_sah), serial O(N log N) — 42 ms at 65,536 spheres against a 3 ms frame.  What it does NOT replace: the
// reference-topology build (bvh_impl.rs:229-364), whose DFS leaf order decides exact-distance ties and therefore
// stays bit-faithful on the host.  Any conservative tree gives the reference's nearest hit (DESIGN.md §2), so frames
// are bit-identical whichever tree culls; only the number of slab tests differs.
//
// Pipeline (one stream, no host round trip except the depth check):
//   morton_keys   key = 30-bit Morton code of the box centre (10 bits per axis inside the centroid bounds) << 32 | i
//   radix sort    cub::DeviceRadixSort::SortKeys on the 62 significant bits (library sort: not a path kernel)
//   karras_nodes  inner node i ↔ keys [first,last], split by the highest differing bit; the child codes of record i
//   link_nodes    parents of every record's children, from the child codes           (refit from here on)
//   refit_nodes   one thread per leaf walks up; the second arrival at a node joins its two child boxes, writes the
//                 node record's boxes (centre / half-extent form: centre_half, as on the host) and goes on
//   leaf_depths   deepest leaf, for the traversal stack bound (MAX_STACK)               (build only)
#include <cub/device/device_radix_sort.cuh>

#include <cstdlib>

#include "rt_device.cuh"
#include "rt_host.h"

namespace rtb {
namespace {

__device__ __forceinline__ uint32_t expand10(uint32_t v) {  // 10 bits → every third bit
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}

__global__ void morton_keys(const float* __restrict__ boxes, uint32_t n, float3 cmin, float3 cscale,
                            unsigned long long* __restrict__ keys) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* b = boxes + 6 * (size_t)i;
    const float cx = 0.5f * (b[0] + b[3]), cy = 0.5f * (b[1] + b[4]), cz = 0.5f * (b[2] + b[5]);
    const uint32_t qx = (uint32_t)fminf(fmaxf((cx - cmin.x) * cscale.x, 0.0f), 1023.0f);
    const uint32_t qy = (uint32_t)fminf(fmaxf((cy - cmin.y) * cscale.y, 0.0f), 1023.0f);
    const uint32_t qz = (uint32_t)fminf(fmaxf((cz - cmin.z) * cscale.z, 0.0f), 1023.0f);
    const uint32_t code = (expand10(qx) << 2) | (expand10(qy) << 1) | expand10(qz);
    keys[i] = ((unsigned long long)code << 32) | i;  // unique keys: ties between equal codes are broken by the index
}

// length of the common prefix of keys i and j (−1 outside the array); keys are unique
__device__ __forceinline__ int delta(const unsigned long long* keys, int n, int i, int j) {
    if (j < 0 || j >= n) return -1;
    return __clzll((long long)(keys[i] ^ keys[j]));
}

// Karras 2012, Algorithm "construct binary radix tree": inner node i (0 = root) covers sorted keys [first, last].
// Children: index < n-1 → inner node, else leaf (sorted position = index - (n-1)).  Writes the child codes of record i
// (inner: the byte offset of its record; leaf: ~(pid << 5), one primitive per leaf); refit_nodes fills in the boxes.
__global__ void karras_nodes(const unsigned long long* __restrict__ keys, const uint32_t* __restrict__ pid_of, int n,
                             int4* __restrict__ lnode4) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    const int d = (delta(keys, n, i, i + 1) - delta(keys, n, i, i - 1)) >= 0 ? 1 : -1;
    const int dmin = delta(keys, n, i, i - d);
    int lmax = 2;
    while (delta(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int t = lmax >> 1; t >= 1; t >>= 1)
        if (delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
    const int j = i + l * d;
    const int dnode = delta(keys, n, i, j);
    int s = 0;
    for (int t = (l + 1) >> 1;; t = (t + 1) >> 1) {
        if (delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
        if (t == 1) break;
    }
    const int gamma = i + s * d + min(d, 0);
    const int lo = min(i, j), hi = max(i, j);
    const int left = (lo == gamma) ? (n - 1 + gamma) : gamma;
    const int right = (hi == gamma + 1) ? (n - 1 + gamma + 1) : gamma + 1;
    auto code = [&](int c) {
        return c < n - 1 ? c * NODE_BYTES : ~(int)(pid_of[(uint32_t)(keys[c - (n - 1)] & 0xffffffffull)] << 5);
    };
    lnode4[NODE_F4 * (size_t)i + 3] = make_int4(code(left), code(right), 0, 0);
}

struct B6 {
    float lo[3], hi[3];
};

// The parents of every record's children, from the child codes (words 12, 13 of the record): parent[node] for inner
// children, leaf_parent[pid] for leaves.  What no record names keeps the -1 it was set to: the root, big primitives.
__global__ void link_nodes(const int4* __restrict__ lnode4, uint32_t lni, int* __restrict__ parent,
                           int* __restrict__ leaf_parent) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= lni) return;
    const int4 ch = lnode4[NODE_F4 * (size_t)i + 3];
    for (const int c : {ch.x, ch.y}) {
        if (c >= 0) parent[c / NODE_BYTES] = (int)i;
        else leaf_parent[(uint32_t)~c >> 5] = (int)i;
    }
}

// One thread per primitive walks up from its leaf; the second arrival at a node joins its two child boxes (leaves: the
// exact AABB leaf_box[pid]), writes the node record's boxes (centre / half-extent form: centre_half, as on the host)
// and goes on.  The child codes of the records stay as they are.
__global__ void refit_nodes(const float4* __restrict__ leaf_box, uint32_t n_prims, const int* __restrict__ parent,
                            const int* __restrict__ leaf_parent, unsigned int* __restrict__ arrived, B6* nbox,
                            float4* __restrict__ lnode) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_prims) return;
    int node = leaf_parent[p];
    while (node >= 0) {
        __threadfence();
        if (atomicAdd(&arrived[node], 1u) == 0u) return;  // the sibling subtree is not finished: its thread goes on
        __threadfence();
        const int4 ch = reinterpret_cast<const int4*>(lnode)[NODE_F4 * (size_t)node + 3];
        B6 bl, br;
        auto fetch = [&](int c, B6* out) {
            if (c < 0) {
                const uint32_t pid = (uint32_t)~c >> 5;
                const float4 lo = __ldg(leaf_box + 2 * (size_t)pid), hi = __ldg(leaf_box + 2 * (size_t)pid + 1);
                out->lo[0] = lo.x; out->lo[1] = lo.y; out->lo[2] = lo.z;
                out->hi[0] = hi.x; out->hi[1] = hi.y; out->hi[2] = hi.z;
            } else {
                // written by another SM's thread before its atomicAdd: read past L1 (a neighbour in the same line may
                // have been cached earlier in this launch)
                const float* q = reinterpret_cast<const float*>(nbox + c / NODE_BYTES);
                for (int a = 0; a < 3; a++) {
                    out->lo[a] = __ldcg(q + a);
                    out->hi[a] = __ldcg(q + 3 + a);
                }
            }
        };
        fetch(ch.x, &bl);
        fetch(ch.y, &br);
        float lc[3], lh[3], rc[3], rh[3];
        centre_half(bl.lo, bl.hi, lc, lh);
        centre_half(br.lo, br.hi, rc, rh);
        float w[12];
        node_box_words(lc, lh, rc, rh, w);
        lnode[NODE_F4 * (size_t)node + 0] = make_float4(w[0], w[1], w[2], w[3]);
        lnode[NODE_F4 * (size_t)node + 1] = make_float4(w[4], w[5], w[6], w[7]);
        lnode[NODE_F4 * (size_t)node + 2] = make_float4(w[8], w[9], w[10], w[11]);
        B6 u;
        for (int a = 0; a < 3; a++) {
            u.lo[a] = fminf(bl.lo[a], br.lo[a]);
            u.hi[a] = fmaxf(bl.hi[a], br.hi[a]);
        }
        nbox[node] = u;
        node = parent[node];
    }
}

__global__ void leaf_depths(const int* __restrict__ parent, const int* __restrict__ leaf_parent, uint32_t n_prims,
                            unsigned int* __restrict__ max_depth) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned int d = 0;
    if (p < n_prims)
        for (int node = leaf_parent[p]; node >= 0; node = parent[node]) d++;
    for (int ofs = 16; ofs > 0; ofs >>= 1) d = max(d, __shfl_xor_sync(0xffffffffu, d, ofs));
    if ((threadIdx.x & 31) == 0 && d) atomicMax(max_depth, d);
}

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// Sections of the one scratch allocation, 256-byte aligned.
struct Carve {
    size_t off = 0;
    size_t take(size_t bytes) {
        const size_t o = off;
        off = align256(off + bytes);
        return o;
    }
};

// The refit's scratch: parent | leaf_parent (adjacent: one reset to -1) | arrival counters + the deepest leaf | unions.
struct RefitScratch {
    size_t parent, leaf_parent, arrived, nbox;
    RefitScratch(Carve* c, uint32_t n_prims, uint32_t lni)
        : parent(c->take((size_t)lni * 4)), leaf_parent(c->take((size_t)n_prims * 4)), arrived(c->take((size_t)lni * 4 + 4)),
          nbox(c->take((size_t)lni * sizeof(B6))) {}
};

// The scratch buffer holds at least `bytes` (power-of-two size classes, >= 1 MB).
cudaError_t reserve(DeviceBuild* buf, size_t bytes, cudaStream_t stream) {
    if (buf->bytes >= bytes) return cudaSuccess;
    cudaStreamSynchronize(stream);
    free_device_build(buf);
    size_t cap = (size_t)1 << 20;
    while (cap < bytes) cap <<= 1;
    const cudaError_t e = cudaMalloc(&buf->mem, cap);
    if (e == cudaSuccess) buf->bytes = cap;
    return e;
}

// Refit of the lni records at lnode to the leaf boxes; with want_depth, the deepest leaf goes to the word after the
// arrival counters too.  Queued on `stream`.
cudaError_t run_refit(uint8_t* m, const RefitScratch& r, const float4* leaf_box, uint32_t n_prims, float4* lnode,
                      uint32_t lni, bool want_depth, cudaStream_t stream) {
    int* parent = (int*)(m + r.parent);
    int* leaf_parent = (int*)(m + r.leaf_parent);
    unsigned int* arrived = (unsigned int*)(m + r.arrived);
    cudaError_t e = cudaMemsetAsync(parent, 0xff, r.leaf_parent - r.parent + (size_t)n_prims * 4, stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(arrived, 0, (size_t)lni * 4 + 4, stream);
    if (e != cudaSuccess) return e;
    const unsigned T = 256;
    link_nodes<<<(lni + T - 1) / T, T, 0, stream>>>((const int4*)lnode, lni, parent, leaf_parent);
    refit_nodes<<<(n_prims + T - 1) / T, T, 0, stream>>>(leaf_box, n_prims, parent, leaf_parent, arrived,
                                                         (B6*)(m + r.nbox), lnode);
    if (want_depth) leaf_depths<<<(n_prims + T - 1) / T, T, 0, stream>>>(parent, leaf_parent, n_prims, arrived + lni);
    return cudaGetLastError();
}

}  // namespace

void free_device_build(DeviceBuild* b) {
    if (b->mem) cudaFree(b->mem);
    *b = DeviceBuild();
}

// h_boxes: the boxes of the n primitives the tree covers (host); pid_of: their primitive ids (host).  leaf_box (device,
// n_prims pairs min | max by pid) must hold their boxes already.  Writes n - 1 node records to lnode (device); the root is
// node 0.  *depth_out = deepest leaf.
static_assert(sizeof(Box) == 6 * sizeof(float), "the kernels read a Box as min xyz | max xyz");
cudaError_t build_lbvh_device(DeviceBuild* buf, const Box* h_boxes, const uint32_t* h_pid_of, uint32_t n,
                              const float4* leaf_box, uint32_t n_prims, float4* lnode, uint32_t* depth_out,
                              cudaStream_t stream) {
    if (n < 2) return cudaErrorInvalidValue;
    // centroid bounds on the host: one pass over data the host already holds
    float cmin[3] = {3.0e38f, 3.0e38f, 3.0e38f}, cmax[3] = {-3.0e38f, -3.0e38f, -3.0e38f};
    for (uint32_t i = 0; i < n; i++)
        for (int a = 0; a < 3; a++) {
            const float c = 0.5f * (h_boxes[i].min[a] + h_boxes[i].max[a]);
            cmin[a] = c < cmin[a] ? c : cmin[a];
            cmax[a] = c > cmax[a] ? c : cmax[a];
        }
    float3 lo = make_float3(cmin[0], cmin[1], cmin[2]), sc;
    sc.x = cmax[0] > cmin[0] ? 1023.999f / (cmax[0] - cmin[0]) : 0.0f;
    sc.y = cmax[1] > cmin[1] ? 1023.999f / (cmax[1] - cmin[1]) : 0.0f;
    sc.z = cmax[2] > cmin[2] ? 1023.999f / (cmax[2] - cmin[2]) : 0.0f;

    size_t sort_bytes = 0;
    cudaError_t e = cub::DeviceRadixSort::SortKeys(nullptr, sort_bytes, (const unsigned long long*)nullptr,
                                                   (unsigned long long*)nullptr, (int)n, 0, 62, stream);
    if (e != cudaSuccess) return e;
    // one allocation: boxes | pid_of | keys in | keys out | sort scratch | the refit's scratch
    Carve c;
    const size_t o_box = c.take((size_t)n * 24), o_pid = c.take((size_t)n * 4), o_k0 = c.take((size_t)n * 8),
                 o_k1 = c.take((size_t)n * 8), o_sort = c.take(sort_bytes);
    const RefitScratch r(&c, n_prims, n - 1);
    if ((e = reserve(buf, c.off, stream)) != cudaSuccess) return e;
    uint8_t* m = (uint8_t*)buf->mem;
    float* d_boxes = (float*)(m + o_box);
    uint32_t* d_pid = (uint32_t*)(m + o_pid);
    unsigned long long* k0 = (unsigned long long*)(m + o_k0);
    unsigned long long* k1 = (unsigned long long*)(m + o_k1);
    if ((e = cudaMemcpyAsync(d_boxes, h_boxes, (size_t)n * sizeof(Box), cudaMemcpyHostToDevice, stream)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(d_pid, h_pid_of, (size_t)n * 4, cudaMemcpyHostToDevice, stream)) != cudaSuccess) return e;
    const unsigned T = 256, G = (n + T - 1) / T;
    morton_keys<<<G, T, 0, stream>>>(d_boxes, n, lo, sc, k0);
    if ((e = cub::DeviceRadixSort::SortKeys(m + o_sort, sort_bytes, k0, k1, (int)n, 0, 62, stream)) != cudaSuccess) return e;
    karras_nodes<<<G, T, 0, stream>>>(k1, d_pid, (int)n, (int4*)lnode);
    if ((e = run_refit(m, r, leaf_box, n_prims, lnode, n - 1, true, stream)) != cudaSuccess) return e;
    unsigned int depth = 0;
    if ((e = cudaMemcpyAsync(&depth, (unsigned int*)(m + r.arrived) + (n - 1), 4, cudaMemcpyDeviceToHost, stream)) != cudaSuccess)
        return e;
    if ((e = cudaStreamSynchronize(stream)) != cudaSuccess) return e;
    *depth_out = depth;
    return cudaGetLastError();
}

cudaError_t refit_device(DeviceBuild* buf, const float4* leaf_box, uint32_t n_prims, float4* lnode, uint32_t lni,
                         cudaStream_t stream) {
    if (lni == 0) return cudaSuccess;
    Carve c;
    const RefitScratch r(&c, n_prims, lni);
    cudaError_t e = reserve(buf, c.off, stream);
    if (e == cudaSuccess) e = run_refit((uint8_t*)buf->mem, r, leaf_box, n_prims, lnode, lni, false, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    return e;
}

}  // namespace rtb
