// rt_bvh_device.cu — device-side build of the TRAVERSAL tree (SURVEY.md §8f row f3): Morton-code LBVH
// (Karras 2012: one thread per inner node finds its key range and split from common prefixes) + bottom-up refit.
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
//   karras_nodes  inner node i ↔ keys [first,last], split by the highest differing bit; children + parents
//   refit         one thread per leaf walks up; the second arrival at a node joins its two child boxes, writes the
//                 node record (centre / half-extent form, padded exactly like the host's centre_half_of) and goes on
//   leaf_depths   deepest leaf, for the traversal stack bound (MAX_STACK)
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
// Children: index < n-1 → inner node, else leaf (sorted position = index - (n-1)).
__global__ void karras_nodes(const unsigned long long* __restrict__ keys, int n, int2* __restrict__ child,
                             int* __restrict__ parent /* [2n-1]: inner nodes then leaves */) {
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
    child[i] = make_int2(left, right);
    parent[left] = i;
    parent[right] = i;
    if (i == 0) parent[0] = -1;
}

struct B6 {
    float lo[3], hi[3];
};

// centre / half-extent form, padded for the FILTER-domain slab arithmetic — the host's centre_half_of, verbatim
__device__ __forceinline__ void centre_half_dev(const B6& b, float c[3], float h[3]) {
    double m = 0.0;
    for (int a = 0; a < 3; a++) m = fmax(m, fmax(fabs((double)b.lo[a]), fabs((double)b.hi[a])));
    for (int a = 0; a < 3; a++) {
        const double cc = 0.5 * ((double)b.lo[a] + (double)b.hi[a]);
        const double hh = 0.5 * ((double)b.hi[a] - (double)b.lo[a]);
        c[a] = (float)cc;
        h[a] = (float)(hh * (1.0 + 4e-6) + 2e-6 * m + 1e-30);
    }
}

__global__ void refit(const unsigned long long* __restrict__ keys, const float* __restrict__ boxes,
                      const uint32_t* __restrict__ pid_of, int n, const int2* __restrict__ child,
                      const int* __restrict__ parent, unsigned int* __restrict__ arrived, B6* nbox,
                      float4* __restrict__ lnode) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    int node = parent[n - 1 + p];
    while (node >= 0) {
        __threadfence();
        if (atomicAdd(&arrived[node], 1u) == 0u) return;  // the sibling subtree is not finished: its thread goes on
        __threadfence();
        const int2 ch = child[node];
        B6 bl, br;
        int cl, cr;
        auto fetch = [&](int c, B6* out, int* code) {
            if (c >= n - 1) {
                const uint32_t id = (uint32_t)(keys[c - (n - 1)] & 0xffffffffull);
                const float* b = boxes + 6 * (size_t)id;
                for (int a = 0; a < 3; a++) {
                    out->lo[a] = b[a];
                    out->hi[a] = b[3 + a];
                }
                *code = ~(int)((pid_of[id] << 5) | 0u);  // one primitive per leaf
            } else {
                // written by another SM's thread before its atomicAdd: read past L1 (a neighbour in the same line may
                // have been cached earlier in this launch)
                const float* q = reinterpret_cast<const float*>(nbox + c);
                for (int a = 0; a < 3; a++) {
                    out->lo[a] = __ldcg(q + a);
                    out->hi[a] = __ldcg(q + 3 + a);
                }
                *code = c;
            }
        };
        fetch(ch.x, &bl, &cl);
        fetch(ch.y, &br, &cr);
        float lc[3], lh[3], rc[3], rh[3];
        centre_half_dev(bl, lc, lh);
        centre_half_dev(br, rc, rh);
        float w[12];
        node_box_words(lc, lh, rc, rh, w);
        lnode[NODE_F4 * (size_t)node + 0] = make_float4(w[0], w[1], w[2], w[3]);
        lnode[NODE_F4 * (size_t)node + 1] = make_float4(w[4], w[5], w[6], w[7]);
        lnode[NODE_F4 * (size_t)node + 2] = make_float4(w[8], w[9], w[10], w[11]);
        // inner children by the byte offset of their record (rt_device.cuh)
        reinterpret_cast<int4*>(lnode)[NODE_F4 * (size_t)node + 3] =
            make_int4(cl >= 0 ? cl * NODE_BYTES : cl, cr >= 0 ? cr * NODE_BYTES : cr, 0, 0);
        for (int k = 4; k < NODE_F4; k++) lnode[NODE_F4 * (size_t)node + k] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        B6 u;
        for (int a = 0; a < 3; a++) {
            u.lo[a] = fminf(bl.lo[a], br.lo[a]);
            u.hi[a] = fmaxf(bl.hi[a], br.hi[a]);
        }
        nbox[node] = u;
        node = parent[node];
    }
}

__global__ void leaf_depths(const int* __restrict__ parent, int n, unsigned int* __restrict__ max_depth) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned int d = 0;
    if (p < n)
        for (int node = parent[n - 1 + p]; node >= 0; node = parent[node]) d++;
    for (int ofs = 16; ofs > 0; ofs >>= 1) d = max(d, __shfl_xor_sync(0xffffffffu, d, ofs));
    if ((threadIdx.x & 31) == 0 && d) atomicMax(max_depth, d);
}

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

}  // namespace

void free_device_build(DeviceBuild* b) {
    if (b->mem) cudaFree(b->mem);
    *b = DeviceBuild();
}

// boxes: n x (min xyz, max xyz) of the primitives the tree covers (host); pid_of: their primitive ids (host).
// Writes n - 1 node records to lnode (device); the root is node 0.
// *depth_out = deepest leaf.
cudaError_t build_lbvh_device(DeviceBuild* buf, const float* h_boxes, const uint32_t* h_pid_of, uint32_t n,
                              float4* lnode, uint32_t* depth_out, cudaStream_t stream) {
    if (n < 2) return cudaErrorInvalidValue;
    // centroid bounds on the host: one pass over data the host already holds
    float cmin[3] = {3.0e38f, 3.0e38f, 3.0e38f}, cmax[3] = {-3.0e38f, -3.0e38f, -3.0e38f};
    for (uint32_t i = 0; i < n; i++)
        for (int a = 0; a < 3; a++) {
            const float c = 0.5f * (h_boxes[6 * (size_t)i + a] + h_boxes[6 * (size_t)i + 3 + a]);
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
    // one allocation: boxes | pid_of | keys in | keys out | child | parent | arrived + depth | node boxes | sort scratch
    size_t off = 0;
    auto take = [&](size_t bytes) {
        const size_t o = off;
        off = align256(off + bytes);
        return o;
    };
    const size_t o_box = take((size_t)n * 24), o_pid = take((size_t)n * 4), o_k0 = take((size_t)n * 8),
                 o_k1 = take((size_t)n * 8), o_child = take((size_t)(n - 1) * 8), o_parent = take((size_t)(2 * n - 1) * 4),
                 o_arr = take((size_t)n * 4 + 4), o_nbox = take((size_t)(n - 1) * sizeof(B6)), o_sort = take(sort_bytes);
    if (buf->bytes < off) {
        cudaStreamSynchronize(stream);
        free_device_build(buf);
        size_t cap = (size_t)1 << 20;
        while (cap < off) cap <<= 1;
        if ((e = cudaMalloc(&buf->mem, cap)) != cudaSuccess) return e;
        buf->bytes = cap;
    }
    uint8_t* m = (uint8_t*)buf->mem;
    float* d_boxes = (float*)(m + o_box);
    uint32_t* d_pid = (uint32_t*)(m + o_pid);
    unsigned long long* k0 = (unsigned long long*)(m + o_k0);
    unsigned long long* k1 = (unsigned long long*)(m + o_k1);
    int2* d_child = (int2*)(m + o_child);
    int* d_parent = (int*)(m + o_parent);
    unsigned int* d_arr = (unsigned int*)(m + o_arr);
    B6* d_nbox = (B6*)(m + o_nbox);
    if ((e = cudaMemcpyAsync(d_boxes, h_boxes, (size_t)n * 24, cudaMemcpyHostToDevice, stream)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(d_pid, h_pid_of, (size_t)n * 4, cudaMemcpyHostToDevice, stream)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(d_arr, 0, (size_t)n * 4 + 4, stream)) != cudaSuccess) return e;
    const unsigned T = 256, G = (n + T - 1) / T;
    morton_keys<<<G, T, 0, stream>>>(d_boxes, n, lo, sc, k0);
    if ((e = cub::DeviceRadixSort::SortKeys(m + o_sort, sort_bytes, k0, k1, (int)n, 0, 62, stream)) != cudaSuccess) return e;
    karras_nodes<<<G, T, 0, stream>>>(k1, (int)n, d_child, d_parent);
    refit<<<G, T, 0, stream>>>(k1, d_boxes, d_pid, (int)n, d_child, d_parent, d_arr, d_nbox, lnode);
    leaf_depths<<<G, T, 0, stream>>>(d_parent, (int)n, d_arr + n);
    unsigned int depth = 0;
    if ((e = cudaMemcpyAsync(&depth, d_arr + n, 4, cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(stream)) != cudaSuccess) return e;
    *depth_out = depth;
    return cudaGetLastError();
}

}  // namespace rtb
