// rt_obj.cu — the controller's OBJ ++ MTL upload body turned into its triangle world on the device, bit for bit what
// rt_b200/obj.py's build_world (the host path, ray-tracer-controller/src/obj.rs:10-53) returns, or a decline.
//
// The body goes to the device as OBJ '\n' MTL '\n' (the host decodes the two sections separately, so no line crosses
// obj_size; the added line ends keep it so and end the last line of each).  Then, on ctx->stream:
//   obj_ends_kernel (COUNT)   one thread per 64 bytes: the line ends in them (\n \r \v \f \x1c-\x1e: every byte at which
//                             str.splitlines() breaks an ASCII text) and any byte >= 0x80 (a decline); CTA scan,
//                             scan_carry over the CTA totals
//   obj_ends_kernel (WRITE)   the same pass stores each line end at its index
//   obj_line_kernel (COUNT)   one thread per line: the comment cut at '#', the key, and the line's counts (a vertex, its
//                             corners, whether it closes a model (o, g, usemtl), a usemtl, a line the host reads (usemtl;
//                             newmtl, Kd, Ns in the MTL)); a v of fewer than 3 coordinates or an f of fewer than 3 corners
//                             is a decline.  One CTA scan of the five counts, scan_carry over each
//   obj_line_kernel (WRITE)   the same pass, each line at its prefix: vertices parsed into a compact array; corners
//                             resolved (i > 0: i - 1, else the vertex count at the line + i; out of range is a decline)
//                             into a flat array; the start and the usemtl ordinal of each model; the lines the host reads,
//                             with the Kd / Ns numbers of MTL lines already converted
//   host                      materials from the MTL lines in order (a repeated newmtl resets, the last one wins) and
//                             the material of each usemtl ordinal: work in the MTL and usemtl lines only
//   obj_model_kernel          one thread per model: corners / 3 triangles (a model with corners and no material is a
//                             decline); CTA scan, scan_carry → each model's first triangle
//   obj_tri_kernel            one thread per triangle: its model by binary search over the first triangles, its three
//                             corners, and the model's material (roughness = Ns / 1000 in one f32 division)
// The model of a line is the count of o / g / usemtl lines up to it, and its material the latest usemtl before the model
// opened: no usemtl can lie inside a model, since each closes one.  So a triple may span f lines, and the 1 or 2 corners
// left at a model's end are dropped, exactly as the host's flat list cut into triples.
#include <cub/block/block_scan.cuh>

#include <string>
#include <unordered_map>
#include <vector>

#include "rt_ctx.h"
#include "rt_wire_num.cuh"

using namespace rtb;

namespace {

constexpr int kScanThreads = 256;
constexpr uint32_t kTextChunk = 64;  // text bytes per thread of obj_ends_kernel
constexpr int kCounts = 5;

using ScanU32 = cub::BlockScan<uint32_t, kScanThreads>;

// What a line adds to the five prefixes
struct Counts {
    uint32_t v, corners, close, use, named;
};
struct AddCounts {
    __device__ __forceinline__ Counts operator()(const Counts& a, const Counts& b) const {
        return {a.v + b.v, a.corners + b.corners, a.close + b.close, a.use + b.use, a.named + b.named};
    }
};
using ScanCounts = cub::BlockScan<Counts, kScanThreads>;

// A line the host reads: [s, e) with the comment cut (positions in the device text); for an MTL Kd or Ns line, its
// numbers (ok: all of them are in the device grammar; Kd needs 3 tokens, Ns 1)
struct Named {
    uint32_t s, e;
    float v[3];
    uint32_t ok;
};

// The material of a usemtl ordinal, resolved by the host (ok = 0: no material of that name)
struct UseMat {
    float kd[3];
    float ns;
    uint32_t ok;
};

__device__ __forceinline__ bool line_end(uint8_t c) {
    return c == '\n' || c == '\r' || c == 0x0b || c == 0x0c || (c >= 0x1c && c <= 0x1e);
}
// str.split()'s whitespace inside a line (the other ASCII whitespace ends the line)
__host__ __device__ __forceinline__ bool obj_sep(uint8_t c) { return c == ' ' || c == '\t' || c == 0x1f; }

__host__ __device__ __forceinline__ bool next_token(const uint8_t*& p, const uint8_t* end, const uint8_t*& tb,
                                                    const uint8_t*& te) {
    while (p < end && obj_sep(*p)) p++;
    if (p == end) return false;
    tb = p;
    while (p < end && !obj_sep(*p)) p++;
    te = p;
    return true;
}

__device__ __forceinline__ bool is_key(const uint8_t* b, const uint8_t* e, const char* k) {
    for (; b < e && *k; b++, k++)
        if (*b != (uint8_t)*k) return false;
    return b == e && !*k;
}

// int(corner.split("/")[0]) of the corner token [p, end): [+-]? at most 10 digits, then the end or a '/'
__device__ __forceinline__ bool face_index(const uint8_t* p, const uint8_t* end, long long* out) {
    const bool neg = *p == '-';
    p += *p == '-' || *p == '+';
    long long v = 0;
    int n = 0;
    for (; p < end && json_digit(*p); p++, n++) v = v * 10 + (*p - '0');
    if (n == 0 || n > 10 || (p < end && *p != '/')) return false;
    *out = neg ? -v : v;
    return true;
}

// WRITE = false: count the line ends in each thread's bytes (and flag bytes >= 0x80), scan the counts within the CTA.
// WRITE = true: store them at their index (cta_off from scan_carry).
template <bool WRITE>
__global__ void __launch_bounds__(kScanThreads) obj_ends_kernel(const uint8_t* __restrict__ text, uint32_t chunks,
                                                                uint32_t* __restrict__ local,
                                                                unsigned long long* __restrict__ cta_sums,
                                                                uint32_t* __restrict__ ends,
                                                                unsigned int* __restrict__ decline) {
    __shared__ typename ScanU32::TempStorage s_scan;
    const uint32_t c = blockIdx.x * kScanThreads + threadIdx.x;
    uint32_t count = 0, at = 0, high = 0;
    if (c < chunks) {
        if (WRITE) at = (uint32_t)cta_sums[blockIdx.x] + local[c];
        const uint4* q = reinterpret_cast<const uint4*>(text) + (size_t)c * (kTextChunk / 16);
        const uint32_t base = c * kTextChunk;
#pragma unroll
        for (uint32_t v = 0; v < kTextChunk / 16; v++) {
            const uint4 u = q[v];
            const uint32_t w[4] = {u.x, u.y, u.z, u.w};
            if (!WRITE) high |= (w[0] | w[1] | w[2] | w[3]) & 0x80808080u;
#pragma unroll
            for (int j = 0; j < 16; j++) {
                if (line_end((uint8_t)(w[j >> 2] >> (8 * (j & 3))))) {
                    if (WRITE) ends[at++] = base + v * 16 + j;
                    count++;
                }
            }
        }
    }
    if (!WRITE) {
        if (high) atomicOr(decline, 1u);
        uint32_t off, total;
        ScanU32(s_scan).ExclusiveSum(count, off, total);
        if (c < chunks) local[c] = off;
        if (threadIdx.x == 0) cta_sums[blockIdx.x] = total;
    }
}

struct LineOut {
    float* verts;           // 3 per vertex
    uint32_t* corners;      // vertex index per corner
    uint32_t* model_start;  // model k >= 1: its first corner (model 0 starts at 0)
    int32_t* model_use;     // model k >= 1: its usemtl ordinal, -1 none
    Named* named;
};

// Line [s, e) of the device text.  at: the prefixes at the line (WRITE only).
template <bool WRITE>
__device__ __forceinline__ Counts obj_line(const uint8_t* text, uint32_t s, uint32_t e, bool mtl, const Counts& at,
                                           const LineOut& o, unsigned int* decline) {
    Counts c{0, 0, 0, 0, 0};
    const uint8_t* p = text + s;
    const uint8_t* end = p;
    while (end < text + e && *end != '#') end++;
    const uint8_t *kb, *ke, *tb, *te;
    if (!next_token(p, end, kb, ke)) return c;
    const uint32_t kl = (uint32_t)(ke - kb);
    if (!mtl) {
        if (kl == 1 && *kb == 'v') {
            c.v = 1;
            float x[3];
            int n = 0;
            for (; n < 3 && next_token(p, end, tb, te); n++)
                if (WRITE && !obj_number(tb, te, &x[n])) atomicOr(decline, 1u);
            if (n < 3) {
                if (!WRITE) atomicOr(decline, 1u);
            } else if (WRITE) {
                float* v = o.verts + (size_t)at.v * 3;
                v[0] = x[0];
                v[1] = x[1];
                v[2] = x[2];
            }
        } else if (kl == 1 && *kb == 'f') {
            uint32_t n = 0;
            for (; next_token(p, end, tb, te); n++) {
                if (!WRITE) continue;
                long long i;
                if (!face_index(tb, te, &i)) {
                    atomicOr(decline, 1u);
                    continue;
                }
                i = i > 0 ? i - 1 : (long long)at.v + i;  // negative indices are relative to the vertices so far
                if (i < 0 || i >= (long long)at.v) {
                    atomicOr(decline, 1u);
                    continue;
                }
                o.corners[at.corners + n] = (uint32_t)i;
            }
            if (!WRITE && n < 3) atomicOr(decline, 1u);
            c.corners = n;
        } else {
            const bool use = is_key(kb, ke, "usemtl");
            if (use || (kl == 1 && (*kb == 'o' || *kb == 'g'))) {
                c.close = 1;
                c.use = c.named = use;
                if (WRITE) {
                    o.model_start[at.close + 1] = at.corners;
                    o.model_use[at.close + 1] = (int32_t)(at.use + c.use) - 1;
                    if (use) o.named[at.named] = Named{s, (uint32_t)(end - text), {0.f, 0.f, 0.f}, 0};
                }
            }
        }
    } else {
        const bool kd = is_key(kb, ke, "Kd"), ns = is_key(kb, ke, "Ns");
        if (kd || ns || is_key(kb, ke, "newmtl")) {
            c.named = 1;
            if (WRITE) {
                Named nm{s, (uint32_t)(end - text), {0.f, 0.f, 0.f}, 0};
                if (kd || ns) {
                    const int want = kd ? 3 : 1;
                    int n = 0;
                    bool ok = true;
                    for (; n < want && next_token(p, end, tb, te); n++) ok = obj_number(tb, te, &nm.v[n]) && ok;
                    nm.ok = ok && n == want;
                }
                o.named[at.named] = nm;
            }
        }
    }
    return c;
}

template <bool WRITE>
__global__ void __launch_bounds__(kScanThreads) obj_line_kernel(const uint8_t* __restrict__ text,
                                                                const uint32_t* __restrict__ ends, uint32_t n_lines,
                                                                uint32_t mtl_start, Counts* __restrict__ local,
                                                                unsigned long long* __restrict__ cta_sums, uint32_t ctas,
                                                                LineOut o, unsigned int* __restrict__ decline) {
    __shared__ typename ScanCounts::TempStorage s_scan;
    const uint32_t k = blockIdx.x * kScanThreads + threadIdx.x;
    Counts at{0, 0, 0, 0, 0}, c{0, 0, 0, 0, 0};
    if (k < n_lines) {
        const uint32_t s = k ? ends[k - 1] + 1 : 0, e = ends[k];
        if (WRITE) {
            const Counts l = local[k];
            const unsigned long long* cs = cta_sums + blockIdx.x;
            at = {(uint32_t)cs[0] + l.v, (uint32_t)cs[ctas + 1] + l.corners, (uint32_t)cs[2 * (ctas + 1)] + l.close,
                  (uint32_t)cs[3 * (ctas + 1)] + l.use, (uint32_t)cs[4 * (ctas + 1)] + l.named};
        }
        c = obj_line<WRITE>(text, s, e, s >= mtl_start, at, o, decline);
    }
    if (!WRITE) {
        Counts off, total;
        ScanCounts(s_scan).ExclusiveScan(c, off, Counts{0, 0, 0, 0, 0}, AddCounts(), total);
        if (k < n_lines) local[k] = off;
        if (threadIdx.x == 0) {
            const uint32_t t[kCounts] = {total.v, total.corners, total.close, total.use, total.named};
            for (int f = 0; f < kCounts; f++) cta_sums[f * (ctas + 1) + blockIdx.x] = t[f];
        }
    }
}

__device__ __forceinline__ uint32_t model_first(const uint32_t* model_start, uint32_t m) { return m ? model_start[m] : 0; }

// One thread per model: its triangles (corners / 3), their exclusive sum within the CTA
__global__ void __launch_bounds__(kScanThreads) obj_model_kernel(const uint32_t* __restrict__ model_start,
                                                                 const int32_t* __restrict__ model_use, uint32_t n_models,
                                                                 uint32_t n_corners, const UseMat* __restrict__ mats,
                                                                 uint32_t* __restrict__ local,
                                                                 unsigned long long* __restrict__ cta_sums,
                                                                 unsigned int* __restrict__ decline) {
    __shared__ typename ScanU32::TempStorage s_scan;
    const uint32_t m = blockIdx.x * kScanThreads + threadIdx.x;
    uint32_t tris = 0;
    if (m < n_models) {
        const uint32_t n = (m + 1 < n_models ? model_start[m + 1] : n_corners) - model_first(model_start, m);
        if (n) {
            const int32_t u = m ? model_use[m] : -1;
            if (u < 0 || !mats[u].ok) atomicOr(decline, 1u);  // the host's "model without a material"
        }
        tris = n / 3;
    }
    uint32_t off, total;
    ScanU32(s_scan).ExclusiveSum(tris, off, total);
    if (m < n_models) local[m] = off;
    if (threadIdx.x == 0) cta_sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(kScanThreads) obj_tri_kernel(const float* __restrict__ verts,
                                                               const uint32_t* __restrict__ corners,
                                                               const uint32_t* __restrict__ model_start,
                                                               const int32_t* __restrict__ model_use, uint32_t n_models,
                                                               const UseMat* __restrict__ mats,
                                                               const uint32_t* __restrict__ local,
                                                               const unsigned long long* __restrict__ cta_off,
                                                               uint32_t model_ctas, rt_triangle* __restrict__ out) {
    const uint32_t t = blockIdx.x * kScanThreads + threadIdx.x;
    if (t >= cta_off[model_ctas]) return;
    // the last model whose first triangle is <= t (models without triangles before it share its first triangle)
    uint32_t lo = 0, hi = n_models - 1;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) / 2;
        if ((uint32_t)cta_off[mid / kScanThreads] + local[mid] <= t) lo = mid;
        else hi = mid - 1;
    }
    const uint32_t m = lo;
    const int32_t u = m ? model_use[m] : -1;
    if (u < 0) return;  // declined by obj_model_kernel
    const UseMat mat = mats[u];
    const uint32_t g = model_first(model_start, m) + 3 * (t - ((uint32_t)cta_off[m / kScanThreads] + local[m]));
    float* o = reinterpret_cast<float*>(out + t);
    for (int k = 0; k < 3; k++) {
        const float* v = verts + (size_t)corners[g + k] * 3;
        o[3 * k] = v[0];
        o[3 * k + 1] = v[1];
        o[3 * k + 2] = v[2];
    }
    o[9] = mat.kd[0];
    o[10] = mat.kd[1];
    o[11] = mat.kd[2];
    o[12] = __fdiv_rn(mat.ns, 1000.0f);  // np.float32(Ns) / np.float32(1000)
    o[13] = 0.0f;
}

// ------------------------------------------------------------------------------------------------
// Scratch (ctx->d_obj, grows with the input; offsets 256-byte aligned).  The parse carves it in three stages, each
// sized by what the previous one counted; growing keeps the bytes the earlier stages wrote.
// ------------------------------------------------------------------------------------------------
struct Carver {
    size_t o = 0;
    size_t take(size_t bytes) {
        const size_t at = o;
        o += (bytes + 255) / 256 * 256;
        return at;
    }
};

int ensure_obj_scratch(rt_ctx* ctx, size_t bytes, size_t keep) {
    if (!ctx->h_obj) CK(ctx, cudaMallocHost(&ctx->h_obj, 8 * sizeof(unsigned long long)));
    if (ctx->d_obj_bytes >= bytes) return RT_OK;
    uint8_t* p = nullptr;
    CK(ctx, cudaMalloc(&p, bytes));
    if (ctx->d_obj) {
        if (keep) CK(ctx, cudaMemcpyAsync(p, ctx->d_obj, keep, cudaMemcpyDeviceToDevice, ctx->stream));
        CK(ctx, cudaStreamSynchronize(ctx->stream));
        CK(ctx, cudaFree(ctx->d_obj));
    }
    ctx->d_obj = p;
    ctx->d_obj_bytes = bytes;
    return RT_OK;
}

struct Token {
    const uint8_t *b, *e;
};

std::vector<Token> tokens(const uint8_t* p, const uint8_t* end) {
    std::vector<Token> t;
    const uint8_t *b, *e;
    while (next_token(p, end, b, e)) t.push_back({b, e});
    return t;
}

// " ".join(rest): the tokens after the key joined by single spaces
std::string name_of(const std::vector<Token>& t) {
    std::string s;
    for (size_t i = 1; i < t.size(); i++) {
        if (i > 1) s += ' ';
        s.append(reinterpret_cast<const char*>(t[i].b), t[i].e - t[i].b);
    }
    return s;
}

constexpr const char* kOrderKey = "__order__";  // parse_mtl's bookkeeping key: a material of that name is the host's

}  // namespace

namespace rtb {

cudaError_t obj_preload() {
    cudaFuncAttributes a;
    cudaError_t e;
    if ((e = cudaFuncGetAttributes(&a, obj_ends_kernel<false>)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, obj_ends_kernel<true>)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, obj_line_kernel<false>)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, obj_line_kernel<true>)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, obj_model_kernel)) != cudaSuccess) return e;
    return cudaFuncGetAttributes(&a, obj_tri_kernel);
}

}  // namespace rtb

extern "C" {

// An f line with n corners is "f" and n tokens, each after at least one separator: at least 2n + 1 bytes.  So an OBJ
// section of obj_size bytes has at most obj_size / 2 corners, and since each model keeps floor(its corners / 3)
// triangles, at most floor(obj_size / 2) / 3 = floor(obj_size / 6) triangles.
size_t rt_obj_max_triangles(size_t obj_size) { return obj_size / 6; }

int rt_obj_build_world(rt_ctx* ctx, const uint8_t* body, size_t len, size_t obj_size, rt_triangle* triangles, size_t cap,
                       uint32_t* n_triangles) {
    if (!ctx) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    if (!body || !triangles || !n_triangles) return set_err(ctx, RT_ERR_INVALID_ARG, "rt_obj_build_world: NULL pointer");
    if (obj_size > len) return set_err(ctx, RT_ERR_INVALID_ARG, "rt_obj_build_world: obj_size %zu > len %zu", obj_size, len);
    const size_t bound = rt_obj_max_triangles(obj_size);
    if (cap < bound)
        return set_err(ctx, RT_ERR_INVALID_ARG, "rt_obj_build_world: cap %zu < rt_obj_max_triangles(%zu) = %zu", cap,
                       obj_size, bound);
    if (len > 0xFFFFFFFFull - 2 - kTextChunk)
        return set_err(ctx, RT_ERR_UNSUPPORTED, "rt_obj_build_world: %zu bytes (positions are 32-bit)", len);
    CK(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    unsigned long long* h = nullptr;
    const auto declined = [&](const char* why) {
        return set_err(ctx, RT_ERR_UNSUPPORTED, "rt_obj_build_world: %s (outside the device grammar)", why);
    };

    // stage 1: the text and its line ends
    const size_t text_len = len + 2, mtl_start = obj_size + 1;
    const uint32_t chunks = (uint32_t)((text_len + kTextChunk - 1) / kTextChunk);
    const uint32_t text_ctas = (chunks + kScanThreads - 1) / kScanThreads;
    Carver cv;
    const size_t o_text = cv.take((size_t)chunks * kTextChunk), o_clocal = cv.take((size_t)chunks * sizeof(uint32_t)),
                 o_csums = cv.take((text_ctas + 1) * sizeof(unsigned long long)), o_decline = cv.take(sizeof(unsigned int));
    int rc = ensure_obj_scratch(ctx, cv.o, 0);
    if (rc) return rc;
    h = ctx->h_obj;
    uint8_t* m = ctx->d_obj;
    CK(ctx, cudaMemsetAsync(m + o_text + text_len, 0, (size_t)chunks * kTextChunk - text_len, s));
    if (obj_size) CK(ctx, cudaMemcpyAsync(m + o_text, body, obj_size, cudaMemcpyHostToDevice, s));
    if (len > obj_size)
        CK(ctx, cudaMemcpyAsync(m + o_text + mtl_start, body + obj_size, len - obj_size, cudaMemcpyHostToDevice, s));
    CK(ctx, cudaMemsetAsync(m + o_text + obj_size, '\n', 1, s));
    CK(ctx, cudaMemsetAsync(m + o_text + len + 1, '\n', 1, s));
    CK(ctx, cudaMemsetAsync(m + o_decline, 0, sizeof(unsigned int), s));
    obj_ends_kernel<false><<<text_ctas, kScanThreads, 0, s>>>(m + o_text, chunks, reinterpret_cast<uint32_t*>(m + o_clocal),
                                                              reinterpret_cast<unsigned long long*>(m + o_csums), nullptr,
                                                              reinterpret_cast<unsigned int*>(m + o_decline));
    CK(ctx, scan_carry(reinterpret_cast<unsigned long long*>(m + o_csums), text_ctas, s));
    CK(ctx, cudaGetLastError());
    CK(ctx, cudaMemcpyAsync(h, m + o_csums + text_ctas * sizeof(unsigned long long), sizeof(unsigned long long),
                            cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaMemcpyAsync(h + 1, m + o_decline, sizeof(unsigned int), cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    if ((uint32_t)h[1]) return declined("a byte above 0x7F");
    const uint32_t n_lines = (uint32_t)h[0];  // >= 2: the two added line ends

    // stage 2: per line, its end and its counts
    const uint32_t line_ctas = (n_lines + kScanThreads - 1) / kScanThreads;
    const size_t o_ends = cv.take((size_t)n_lines * sizeof(uint32_t)), o_llocal = cv.take((size_t)n_lines * sizeof(Counts)),
                 o_lsums = cv.take((size_t)kCounts * (line_ctas + 1) * sizeof(unsigned long long));
    if ((rc = ensure_obj_scratch(ctx, cv.o, o_ends))) return rc;
    m = ctx->d_obj;
    const uint8_t* d_text = m + o_text;
    uint32_t* ends = reinterpret_cast<uint32_t*>(m + o_ends);
    Counts* llocal = reinterpret_cast<Counts*>(m + o_llocal);
    unsigned long long* lsums = reinterpret_cast<unsigned long long*>(m + o_lsums);
    unsigned int* decline = reinterpret_cast<unsigned int*>(m + o_decline);
    obj_ends_kernel<true><<<text_ctas, kScanThreads, 0, s>>>(d_text, chunks, reinterpret_cast<uint32_t*>(m + o_clocal),
                                                             reinterpret_cast<unsigned long long*>(m + o_csums), ends, decline);
    obj_line_kernel<false><<<line_ctas, kScanThreads, 0, s>>>(d_text, ends, n_lines, (uint32_t)mtl_start, llocal, lsums,
                                                              line_ctas, LineOut{}, decline);
    for (int f = 0; f < kCounts; f++) CK(ctx, scan_carry(lsums + (size_t)f * (line_ctas + 1), line_ctas, s));
    CK(ctx, cudaGetLastError());
    for (int f = 0; f < kCounts; f++)
        CK(ctx, cudaMemcpyAsync(h + f, lsums + (size_t)f * (line_ctas + 1) + line_ctas, sizeof(unsigned long long),
                                cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaMemcpyAsync(h + kCounts, decline, sizeof(unsigned int), cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    if ((uint32_t)h[kCounts]) return declined("a v line of fewer than 3 coordinates or an f line of fewer than 3 corners");
    const uint32_t n_v = (uint32_t)h[0], n_corners = (uint32_t)h[1], n_close = (uint32_t)h[2], n_use = (uint32_t)h[3],
                   n_named = (uint32_t)h[4];
    const uint32_t n_models = n_close + 1, model_ctas = (n_models + kScanThreads - 1) / kScanThreads;
    const uint32_t tri_cap = n_corners / 3;

    // stage 3: vertices, corners, models, the lines the host reads, triangles
    const size_t o_verts = cv.take((size_t)n_v * 3 * sizeof(float)), o_corners = cv.take((size_t)n_corners * sizeof(uint32_t)),
                 o_mstart = cv.take((size_t)n_models * sizeof(uint32_t)),
                 o_muse = cv.take((size_t)n_models * sizeof(int32_t)), o_named = cv.take((size_t)n_named * sizeof(Named)),
                 o_mats = cv.take((size_t)n_use * sizeof(UseMat)), o_mlocal = cv.take((size_t)n_models * sizeof(uint32_t)),
                 o_msums = cv.take((model_ctas + 1) * sizeof(unsigned long long)),
                 o_tris = cv.take((size_t)tri_cap * sizeof(rt_triangle));
    if ((rc = ensure_obj_scratch(ctx, cv.o, o_verts))) return rc;
    m = ctx->d_obj;
    d_text = m + o_text;
    ends = reinterpret_cast<uint32_t*>(m + o_ends);
    llocal = reinterpret_cast<Counts*>(m + o_llocal);
    lsums = reinterpret_cast<unsigned long long*>(m + o_lsums);
    decline = reinterpret_cast<unsigned int*>(m + o_decline);
    const LineOut lo{reinterpret_cast<float*>(m + o_verts), reinterpret_cast<uint32_t*>(m + o_corners),
                     reinterpret_cast<uint32_t*>(m + o_mstart), reinterpret_cast<int32_t*>(m + o_muse),
                     reinterpret_cast<Named*>(m + o_named)};
    obj_line_kernel<true><<<line_ctas, kScanThreads, 0, s>>>(d_text, ends, n_lines, (uint32_t)mtl_start, llocal, lsums,
                                                             line_ctas, lo, decline);
    CK(ctx, cudaGetLastError());
    std::vector<Named> named(n_named);
    if (n_named) CK(ctx, cudaMemcpyAsync(named.data(), lo.named, n_named * sizeof(Named), cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaMemcpyAsync(h, decline, sizeof(unsigned int), cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    if ((uint32_t)h[0]) return declined("a number or a face index");

    // materials (parse_mtl): the MTL lines in order, then the material of each usemtl ordinal
    struct Mat {
        float kd[3] = {0.f, 0.f, 0.f};
        float ns = 0.f;
    };
    std::vector<Mat> mats;
    std::unordered_map<std::string, uint32_t> by_name;
    std::vector<UseMat> use(n_use);
    uint32_t n_obj_named = 0;
    int cur = -1;
    for (const Named& nm : named) {
        if (nm.s < mtl_start) {
            n_obj_named++;
            continue;
        }
        const std::vector<Token> t = tokens(body + nm.s - 1, body + nm.e - 1);  // device text → body: the added '\n'
        const size_t kl = t[0].e - t[0].b;
        if (kl == 6) {  // newmtl
            const std::string name = name_of(t);
            if (name == kOrderKey) return declined("a material named __order__");
            const auto it = by_name.emplace(name, (uint32_t)mats.size()).first;
            if (it->second == mats.size()) mats.emplace_back();
            mats[it->second] = Mat{};
            cur = (int)it->second;
        } else if (cur >= 0 && t.size() >= (kl == 2 && t[0].b[0] == 'K' ? 4u : 2u)) {  // Kd with 3 numbers, Ns with 1
            if (!nm.ok) return declined("a Kd or Ns number");
            if (t[0].b[0] == 'K') {
                for (int j = 0; j < 3; j++) mats[cur].kd[j] = nm.v[j];
            } else {
                mats[cur].ns = nm.v[0];
            }
        }
    }
    if (n_obj_named != n_use) return set_err(ctx, RT_ERR_INTERNAL, "rt_obj_build_world: usemtl lines %u != %u", n_obj_named, n_use);
    for (uint32_t i = 0; i < n_use; i++) {
        const Named& nm = named[i];
        const std::string name = name_of(tokens(body + nm.s, body + nm.e));
        if (name == kOrderKey) return declined("a material named __order__");
        const auto it = by_name.find(name);
        use[i] = UseMat{{0.f, 0.f, 0.f}, 0.f, 0};
        if (it != by_name.end()) {
            const Mat& mt = mats[it->second];
            use[i] = UseMat{{mt.kd[0], mt.kd[1], mt.kd[2]}, mt.ns, 1};
        }
    }
    if (!n_corners) {  // no faces: no triangles, and no model that needs a material
        *n_triangles = 0;
        return RT_OK;
    }

    // triangles
    const UseMat* d_mats = reinterpret_cast<const UseMat*>(m + o_mats);
    uint32_t* mlocal = reinterpret_cast<uint32_t*>(m + o_mlocal);
    unsigned long long* msums = reinterpret_cast<unsigned long long*>(m + o_msums);
    rt_triangle* d_tris = reinterpret_cast<rt_triangle*>(m + o_tris);
    if (n_use) CK(ctx, cudaMemcpyAsync(m + o_mats, use.data(), n_use * sizeof(UseMat), cudaMemcpyHostToDevice, s));
    obj_model_kernel<<<model_ctas, kScanThreads, 0, s>>>(lo.model_start, lo.model_use, n_models, n_corners, d_mats, mlocal,
                                                         msums, decline);
    CK(ctx, scan_carry(msums, model_ctas, s));
    if (tri_cap)
        obj_tri_kernel<<<(tri_cap + kScanThreads - 1) / kScanThreads, kScanThreads, 0, s>>>(
            lo.verts, lo.corners, lo.model_start, lo.model_use, n_models, d_mats, mlocal, msums, model_ctas, d_tris);
    CK(ctx, cudaGetLastError());
    CK(ctx, cudaMemcpyAsync(h, msums + model_ctas, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaMemcpyAsync(h + 1, decline, sizeof(unsigned int), cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    if ((uint32_t)h[1]) return declined("a model with faces and no material");
    const uint32_t n = (uint32_t)h[0];
    if (n) CK(ctx, cudaMemcpyAsync(triangles, d_tris, (size_t)n * sizeof(rt_triangle), cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    *n_triangles = n;
    return RT_OK;
    RT_GUARD_END(ctx)
}

}  // extern "C"
