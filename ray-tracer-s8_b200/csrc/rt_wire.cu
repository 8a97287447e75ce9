// rt_wire.cu — the slave's wire format on the device: the "world" array of a RenderInfo body in, the ImageSlice bodies
// out, each equal to what rt_b200/wire.py (the host path) reads and writes.
//
// Parse (rt_world_parse_json), over the text copied to the device with 256 zero bytes after it (every scan below stops at
// the first byte outside its grammar, so it never reads past them):
//   wire_starts_kernel     one thread per 64 bytes: the Object starts in them, '{' ws* '"Sphere"' or '"Triangle"' (the
//            (COUNT / WRITE)   tag of an Object can be nothing else in the device grammar, which has no string values);
//                          CTA scan of the counts, scan_carry over the CTA totals, then the same pass writes positions
//   wire_object_kernel     one thread per start: fixed-schema descent of the Object (keys in declaration order, numbers
//                          by rt_wire_num.cuh), then what follows it: ',' and exactly the next start, or the array's ']'
//   wire_kind_kernel       one thread per start up to the first that ends the array: any decline, and the exclusive sum
//                          of the sphere flags (CTA scan + scan_carry)
//   wire_scatter_kernel    spheres and triangles compacted in world order, world_index = the Object's position
// Why starts are found by their tag and not by quote parity and bracket depth: in the device grammar the only strings
// are keys, so the tag pattern marks exactly the Objects of a valid world, and the chain check of wire_object_kernel
// (every Object followed by ',' and the next start, the first one by the array's '[') proves that the starts and the
// text between them are exactly one array.  A start found anywhere else breaks the chain or lies past the array's end,
// where it is ignored.  One scan of the text instead of three.
//
// ImageSlice bodies (rt_render_divisions_json), over the n bands where the render left them (stacked in list order):
//   wire_len_kernel        one thread per 16 values: 1-3 digits each plus the comma after every value but a band's last;
//                          CTA scan, scan_carry (the JPEG encoder's carry kernel)
//   wire_band_kernel       one CTA: each band's start in the packed output, its header {"division_no":D,"image":[ and
//                          trailer ],"id":"<id>"}, and its length
//   wire_digits_kernel     one thread per 16 values writes them at their offsets
#include <cub/block/block_scan.cuh>

#include "rt_ctx.h"
#include "rt_wire_num.cuh"

using namespace rtb;

namespace {

constexpr int kScanThreads = 256;
constexpr uint32_t kTextChunk = 64;  // text bytes per thread of wire_starts_kernel
constexpr uint32_t kTextPad = 256;   // zero bytes after the text on the device
constexpr uint32_t kValsPerThread = 16;
constexpr uint32_t kHeaderMax = 35;  // {"division_no":4294967295,"image":[
constexpr uint32_t kTrailer = 46;    // ],"id":"<36>"}
constexpr uint32_t kIdLen = 36;
constexpr uint64_t kNoEnd = ~0ull;

using ScanU32 = cub::BlockScan<uint32_t, kScanThreads>;

// ------------------------------------------------------------------------------------------------
// Parse
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ const uint8_t* skip_ws(const uint8_t* p) {
    while (json_ws(*p)) p++;
    return p;
}

// exactly the bytes of s, no whitespace
__device__ __forceinline__ bool exact(const uint8_t*& p, const char* s) {
    for (; *s; s++, p++)
        if (*p != (uint8_t)*s) return false;
    return true;
}

// Is p (just past a '{') the tag of an Object?  1 Sphere, 2 Triangle, 0 no.
__device__ __forceinline__ int tag_at(const uint8_t* p) {
    p = skip_ws(p);
    const uint8_t* q = p;
    if (exact(q, "\"Sphere\"")) return 1;
    q = p;
    return exact(q, "\"Triangle\"") ? 2 : 0;
}

// An Object of the device grammar, written as the JSON it matches: whitespace may precede every token; a quoted key
// matches exactly; #x is a number stored in record slot x (hex); I is node_index, a non-negative integer whose value is
// ignored (wire.py ignores it; the slave rebuilds it).  Record slots are the float fields of rt_sphere (center, radius,
// albedo, roughness, emission) and of rt_triangle (a, b, c, albedo, roughness, emission).  Field order: shapes/sphere.rs
// and shapes/mesh.rs.
constexpr int kRecFloats = 14;
__constant__ const char c_sphere[] =
    "{\"Sphere\":{\"radius\":#3,\"center\":[#0,#1,#2],\"node_index\":I,\"p_albedo_at\":{\"r\":#4,\"g\":#5,\"b\":#6},"
    "\"p_roughness_at\":#7,\"p_emission_at\":#8}}";
__constant__ const char c_triangle[] =
    "{\"Triangle\":{\"a\":[#0,#1,#2],\"b\":[#3,#4,#5],\"c\":[#6,#7,#8],\"node_index\":I,"
    "\"p_albedo_at\":{\"r\":#9,\"g\":#a,\"b\":#b},\"p_roughness_at\":#c,\"p_emission_at\":#d}}";

// The Object at p against its pattern (by tag), numbers into rec; p ends just past it.  *tri: the tag is Triangle.
__device__ __forceinline__ bool parse_object(const uint8_t*& p, float* rec, bool* tri) {
    if (*p != '{') return false;
    const int tag = tag_at(p + 1);
    if (!tag) return false;
    *tri = tag == 2;
    for (const char* s = tag == 1 ? c_sphere : c_triangle; *s; s++) {
        p = skip_ws(p);
        if (*s == '#') {
            const char h = *++s;
            float v;
            if (!json_number(p, &v)) return false;
            rec[h <= '9' ? h - '0' : h - 'a' + 10] = v;
        } else if (*s == 'I') {
            if (!json_digit(*p)) return false;
            if (*p++ == '0') {
                if (json_digit(*p)) return false;
            } else {
                while (json_digit(*p)) p++;
            }
        } else if (*s == '"') {  // the whole key, quotes included, byte for byte
            do {
                if (*p++ != (uint8_t)*s) return false;
            } while (*++s != '"');
            if (*p++ != '"') return false;
        } else if (*p++ != (uint8_t)*s) {
            return false;
        }
    }
    return true;
}

// WRITE = false: count the starts in each thread's bytes and scan the counts within the CTA.  WRITE = true: store them
// at their index (cta_off from scan_carry).
template <bool WRITE>
__global__ void __launch_bounds__(kScanThreads) wire_starts_kernel(const uint8_t* __restrict__ text, uint32_t len,
                                                                   uint32_t chunks, uint32_t* __restrict__ local,
                                                                   unsigned long long* __restrict__ cta_sums,
                                                                   uint32_t* __restrict__ starts, uint32_t cap) {
    __shared__ typename ScanU32::TempStorage s_scan;
    const uint32_t c = blockIdx.x * kScanThreads + threadIdx.x;
    uint32_t count = 0, at = 0;
    if (c < chunks) {
        if (WRITE) at = (uint32_t)cta_sums[blockIdx.x] + local[c];
        const uint4* q = reinterpret_cast<const uint4*>(text) + (size_t)c * (kTextChunk / 16);
        const uint32_t base = c * kTextChunk;
#pragma unroll
        for (uint32_t v = 0; v < kTextChunk / 16; v++) {
            const uint4 u = q[v];
            const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
            for (int j = 0; j < 16; j++) {
                const uint32_t i = base + v * 16 + j;
                if ((uint8_t)(w[j >> 2] >> (8 * (j & 3))) == '{' && i < len && tag_at(text + i + 1)) {
                    if (WRITE && at < cap) starts[at++] = i;
                    count++;
                }
            }
        }
    }
    if (!WRITE) {
        uint32_t off, total;
        ScanU32(s_scan).ExclusiveSum(count, off, total);
        if (c < chunks) local[c] = off;
        if (threadIdx.x == 0) cta_sums[blockIdx.x] = total;
    }
}

// Status of an Object: the low two bits, bit 2 set for a triangle
constexpr uint8_t kNext = 0, kLast = 1, kBad = 2;

__global__ void __launch_bounds__(kScanThreads) wire_object_kernel(const uint8_t* __restrict__ text,
                                                                   const uint32_t* __restrict__ starts,
                                                                   const unsigned long long* __restrict__ n_starts,
                                                                   uint32_t cap, uint32_t first_open, float* __restrict__ recs,
                                                                   uint8_t* __restrict__ status,
                                                                   unsigned long long* __restrict__ first_end) {
    // starts past cap (possible only after the array's end, or in a text that is not a world) are not stored: a chain
    // that needs one breaks at the last stored start, and the parse is declined
    const uint32_t k = blockIdx.x * kScanThreads + threadIdx.x, n = (uint32_t)min(*n_starts, (unsigned long long)cap);
    if (k >= n) return;
    const uint8_t* p = text + starts[k];
    bool tri = false;
    uint8_t st = kBad;
    if ((k || starts[0] == first_open) && parse_object(p, recs + (size_t)k * kRecFloats, &tri)) {
        p = skip_ws(p);
        if (*p == ',') {
            p = skip_ws(p + 1);
            if (k + 1 < n && (uint32_t)(p - text) == starts[k + 1]) st = kNext;
        } else if (*p == ']') {
            st = kLast;  // the Object with the lowest index that is followed by ']' ends the array
            atomicMin(first_end, (unsigned long long)k << 32 | (uint32_t)(p - text));
        }
    }
    status[k] = st | (tri ? 4 : 0);
}

// Objects 0..last (last = the one that ends the array): a decline if any is bad, and the exclusive sum of the spheres
__global__ void __launch_bounds__(kScanThreads) wire_kind_kernel(const uint8_t* __restrict__ status,
                                                                 const unsigned long long* __restrict__ n_starts,
                                                                 uint32_t cap, const unsigned long long* __restrict__ first_end,
                                                                 uint32_t* __restrict__ local,
                                                                 unsigned long long* __restrict__ cta_sums,
                                                                 unsigned int* __restrict__ decline) {
    __shared__ typename ScanU32::TempStorage s_scan;
    const uint32_t k = blockIdx.x * kScanThreads + threadIdx.x;
    const unsigned long long fe = *first_end;
    const bool in = fe != kNoEnd && k <= (uint32_t)(fe >> 32) && k < min(*n_starts, (unsigned long long)cap);
    uint32_t sphere = 0;
    if (in) {
        const uint8_t s = status[k];
        if ((s & 3) == kBad) atomicOr(decline, 1u);
        sphere = !(s & 4);
    }
    uint32_t off, total;
    ScanU32(s_scan).ExclusiveSum(sphere, off, total);
    if (in) local[k] = off;
    if (threadIdx.x == 0) cta_sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(kScanThreads) wire_scatter_kernel(const uint8_t* __restrict__ status,
                                                                    const float* __restrict__ recs,
                                                                    const unsigned long long* __restrict__ first_end,
                                                                    const uint32_t* __restrict__ local,
                                                                    const unsigned long long* __restrict__ cta_off,
                                                                    uint32_t kind_ctas, rt_sphere* __restrict__ spheres,
                                                                    rt_triangle* __restrict__ triangles,
                                                                    uint32_t* __restrict__ world_index) {
    const uint32_t k = blockIdx.x * kScanThreads + threadIdx.x;
    const unsigned long long fe = *first_end;
    if (fe == kNoEnd || k > (uint32_t)(fe >> 32)) return;
    const uint32_t s = (uint32_t)(cta_off[blockIdx.x] + local[k]), ns = (uint32_t)cta_off[kind_ctas];
    const float* r = recs + (size_t)k * kRecFloats;
    if (!(status[k] & 4)) {
        float* o = reinterpret_cast<float*>(spheres + s);
        for (int i = 0; i < 9; i++) o[i] = r[i];
        world_index[s] = k;
    } else {
        const uint32_t t = k - s;
        float* o = reinterpret_cast<float*>(triangles + t);
        for (int i = 0; i < kRecFloats; i++) o[i] = r[i];
        world_index[ns + t] = k;
    }
}

// ------------------------------------------------------------------------------------------------
// ImageSlice bodies
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t digits(uint32_t v) { return 1 + (v >= 10) + (v >= 100); }

// Characters of value i of the stacked bands (band_vals values per band): its digits and the comma after it
__device__ __forceinline__ uint32_t value_chars(uint8_t v, uint64_t i, uint64_t band_vals) {
    return digits(v) + (i % band_vals != band_vals - 1);
}

__global__ void __launch_bounds__(kScanThreads) wire_len_kernel(const uint8_t* __restrict__ rgb, uint64_t vals,
                                                                uint64_t band_vals, uint32_t* __restrict__ local,
                                                                unsigned long long* __restrict__ cta_sums) {
    __shared__ typename ScanU32::TempStorage s_scan;
    const uint64_t c = (uint64_t)blockIdx.x * kScanThreads + threadIdx.x;
    uint32_t chars = 0;
    for (uint32_t j = 0; j < kValsPerThread; j++) {
        const uint64_t i = c * kValsPerThread + j;
        if (i < vals) chars += value_chars(rgb[i], i, band_vals);
    }
    uint32_t off, total;
    ScanU32(s_scan).ExclusiveSum(chars, off, total);
    if (c * kValsPerThread < vals) local[c] = off;
    if (threadIdx.x == 0) cta_sums[blockIdx.x] = total;
}

struct SliceId {
    char c[kIdLen];
};

// Offset of value i's first character among all the bands' digits and commas
__device__ __forceinline__ unsigned long long value_offset(const uint8_t* rgb, uint64_t i, uint64_t vals, uint64_t band_vals,
                                                           const uint32_t* local, const unsigned long long* cta_off) {
    if (i == vals) return cta_off[(vals + kValsPerThread * kScanThreads - 1) / (kValsPerThread * kScanThreads)];
    const uint64_t c = i / kValsPerThread;
    unsigned long long o = cta_off[c / kScanThreads] + local[c];
    for (uint64_t j = c * kValsPerThread; j < i; j++) o += value_chars(rgb[j], j, band_vals);
    return o;
}

__device__ __forceinline__ uint32_t decimal_len(uint32_t v) {
    uint32_t n = 1;
    for (; v >= 10; v /= 10) n++;
    return n;
}

__device__ __forceinline__ uint32_t write_uint(uint8_t* out, uint32_t v) {
    const uint32_t n = decimal_len(v);
    for (uint32_t j = n; j-- > 0; v /= 10) out[j] = (uint8_t)('0' + v % 10);
    return n;
}

__device__ __forceinline__ uint32_t header_len(uint32_t d) { return 15 + decimal_len(d) + 10; }  // {"division_no":D,"image":[

// One CTA.  band_at[k]: characters before band k's first value (k = 0..n); body_off[k]: where body k starts in out;
// img_off[k]: where its first value goes; lens[k]: its length.
__global__ void __launch_bounds__(kScanThreads) wire_band_kernel(const uint8_t* __restrict__ rgb, uint64_t vals,
                                                                 uint64_t band_vals, const uint32_t* __restrict__ local,
                                                                 const unsigned long long* __restrict__ cta_off,
                                                                 const uint32_t* __restrict__ division_nos, uint32_t n,
                                                                 SliceId id, unsigned long long* __restrict__ band_at,
                                                                 unsigned long long* __restrict__ img_off,
                                                                 unsigned long long* __restrict__ lens,
                                                                 uint8_t* __restrict__ out) {
    for (uint32_t k = threadIdx.x; k <= n; k += kScanThreads)
        band_at[k] = value_offset(rgb, (uint64_t)k * band_vals, vals, band_vals, local, cta_off);
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long o = 0;
        for (uint32_t k = 0; k < n; k++) {
            const uint32_t h = header_len(division_nos[k]);
            img_off[k] = o + h;
            lens[k] = h + (band_at[k + 1] - band_at[k]) + kTrailer;
            o += lens[k];
        }
    }
    __syncthreads();
    for (uint32_t k = threadIdx.x; k < n; k += kScanThreads) {
        const uint32_t h = header_len(division_nos[k]);
        uint8_t* b = out + img_off[k] - h;
        const char* head = "{\"division_no\":";
        for (int j = 0; j < 15; j++) b[j] = (uint8_t)head[j];
        b += 15;
        b += write_uint(b, division_nos[k]);
        const char* img = ",\"image\":[";
        for (int j = 0; j < 10; j++) b[j] = (uint8_t)img[j];
        uint8_t* t = out + img_off[k] + (band_at[k + 1] - band_at[k]);
        const char* tid = "],\"id\":\"";
        for (int j = 0; j < 8; j++) t[j] = (uint8_t)tid[j];
        for (uint32_t j = 0; j < kIdLen; j++) t[8 + j] = (uint8_t)id.c[j];
        t[8 + kIdLen] = '"';
        t[9 + kIdLen] = '}';
    }
}

__global__ void __launch_bounds__(kScanThreads) wire_digits_kernel(const uint8_t* __restrict__ rgb, uint64_t vals,
                                                                   uint64_t band_vals, const uint32_t* __restrict__ local,
                                                                   const unsigned long long* __restrict__ cta_off,
                                                                   const unsigned long long* __restrict__ band_at,
                                                                   const unsigned long long* __restrict__ img_off,
                                                                   uint8_t* __restrict__ out) {
    const uint64_t c = (uint64_t)blockIdx.x * kScanThreads + threadIdx.x;
    if (c * kValsPerThread >= vals) return;
    unsigned long long o = cta_off[blockIdx.x] + local[c];  // among all the bands' characters
    for (uint32_t j = 0; j < kValsPerThread; j++) {
        const uint64_t i = c * kValsPerThread + j;
        if (i >= vals) break;
        const uint64_t k = i / band_vals;
        uint8_t* b = out + img_off[k] + (o - band_at[k]);
        const uint32_t v = rgb[i];
        const uint32_t d = digits(v);
        if (d == 3) *b++ = (uint8_t)('0' + v / 100);
        if (d >= 2) *b++ = (uint8_t)('0' + v / 10 % 10);
        *b++ = (uint8_t)('0' + v % 10);
        const bool comma = i % band_vals != band_vals - 1;
        if (comma) *b = ',';
        o += d + comma;
    }
}

// ------------------------------------------------------------------------------------------------
// Scratch (ctx->d_wire, grows with the input; offsets 256-byte aligned)
// ------------------------------------------------------------------------------------------------
struct Carver {
    size_t o = 0;
    size_t take(size_t bytes) {
        const size_t at = o;
        o += (bytes + 255) / 256 * 256;
        return at;
    }
};

int ensure_wire_scratch(rt_ctx* ctx, size_t bytes) {
    if (!ctx->h_wire) CK(ctx, cudaMallocHost(&ctx->h_wire, 4 * sizeof(unsigned long long)));
    if (ctx->d_wire_bytes >= bytes) return RT_OK;
    if (ctx->d_wire) {
        CK(ctx, cudaStreamSynchronize(ctx->stream));
        CK(ctx, cudaFree(ctx->d_wire));
        ctx->d_wire = nullptr;
        ctx->d_wire_bytes = 0;
    }
    CK(ctx, cudaMalloc(&ctx->d_wire, bytes));
    ctx->d_wire_bytes = bytes;
    return RT_OK;
}

// {"Sphere":{"radius":0,"center":[0,0,0],"node_index":0,"p_albedo_at":{"r":0,"g":0,"b":0},"p_roughness_at":0,"p_emission_at":0}}
// is the shortest Object of the grammar (a Triangle has three vectors), and each but the last is followed by a comma.
constexpr size_t kMinObject = 118;

bool uuid_form(const char* id) {
    for (uint32_t i = 0; i < kIdLen; i++) {
        const char c = id[i];
        const bool ok = (i == 8 || i == 13 || i == 18 || i == 23) ? c == '-' : ((c >= '0' && c <= '9') || (c >= 'a' && c <= 'f'));
        if (!ok) return false;  // a NUL stops here too
    }
    return id[kIdLen] == 0;
}

}  // namespace

namespace rtb {

cudaError_t wire_preload() {
    cudaFuncAttributes a;
    cudaError_t e;
    if ((e = cudaFuncGetAttributes(&a, wire_starts_kernel<false>)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, wire_starts_kernel<true>)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, wire_object_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, wire_kind_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, wire_scatter_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, wire_len_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, wire_band_kernel)) != cudaSuccess) return e;
    return cudaFuncGetAttributes(&a, wire_digits_kernel);
}

int slice_json_check(rt_ctx* ctx, uint32_t n, uint32_t rows, uint32_t width, const char* id, const uint8_t* out,
                     size_t out_cap, const size_t* out_lens) {
    if (!id || !out || !out_lens) return set_err(ctx, RT_ERR_INVALID_ARG, "ImageSlice JSON: id, out or out_lens is NULL");
    if (!uuid_form(id))
        return set_err(ctx, RT_ERR_INVALID_ARG, "ImageSlice JSON: id is not a 36-character hyphenated lowercase uuid");
    const size_t need = (size_t)n * rt_slice_json_bound(rows, width);
    if (out_cap < need)
        return set_err(ctx, RT_ERR_INVALID_ARG, "ImageSlice JSON: out_cap %zu < n %u * rt_slice_json_bound(%u, %u) = %zu",
                       out_cap, n, rows, width, need);
    return RT_OK;
}

int slice_json_device(rt_ctx* ctx, const uint8_t* rgb_dev, uint32_t n, uint32_t rows, uint32_t width,
                      const uint32_t* division_nos, const char* id, uint8_t* out, size_t* out_lens) {
    const uint64_t band_vals = (uint64_t)rows * width * 3, vals = band_vals * n;
    const uint64_t threads = (vals + kValsPerThread - 1) / kValsPerThread;
    const uint32_t ctas = (uint32_t)((threads + kScanThreads - 1) / kScanThreads);
    const size_t body_cap = (size_t)n * rt_slice_json_bound(rows, width);
    Carver cv;
    const size_t o_local = cv.take(threads * sizeof(uint32_t)), o_sums = cv.take((ctas + 1) * sizeof(unsigned long long)),
                 o_nos = cv.take(n * sizeof(uint32_t)), o_at = cv.take((n + 1) * sizeof(unsigned long long)),
                 o_img = cv.take(n * sizeof(unsigned long long)), o_lens = cv.take(n * sizeof(unsigned long long)),
                 o_out = cv.take(body_cap);
    int rc = ensure_wire_scratch(ctx, cv.o);
    if (rc) return rc;
    uint8_t* m = ctx->d_wire;
    uint32_t* local = reinterpret_cast<uint32_t*>(m + o_local);
    unsigned long long* sums = reinterpret_cast<unsigned long long*>(m + o_sums);
    uint32_t* nos = reinterpret_cast<uint32_t*>(m + o_nos);
    unsigned long long* band_at = reinterpret_cast<unsigned long long*>(m + o_at);
    unsigned long long* img = reinterpret_cast<unsigned long long*>(m + o_img);
    unsigned long long* lens = reinterpret_cast<unsigned long long*>(m + o_lens);
    SliceId sid;
    memcpy(sid.c, id, kIdLen);
    cudaStream_t s = ctx->stream;
    CK(ctx, cudaMemcpyAsync(nos, division_nos, n * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
    CK(ctx, cudaEventRecord(ctx->ev0, s));
    wire_len_kernel<<<ctas, kScanThreads, 0, s>>>(rgb_dev, vals, band_vals, local, sums);
    CK(ctx, scan_carry(sums, ctas, s));
    wire_band_kernel<<<1, kScanThreads, 0, s>>>(rgb_dev, vals, band_vals, local, sums, nos, n, sid, band_at, img, lens,
                                                m + o_out);
    wire_digits_kernel<<<ctas, kScanThreads, 0, s>>>(rgb_dev, vals, band_vals, local, sums, band_at, img, m + o_out);
    CK(ctx, cudaGetLastError());
    CK(ctx, cudaEventRecord(ctx->ev1, s));
    static_assert(sizeof(size_t) == sizeof(unsigned long long), "out_lens is copied as u64");
    CK(ctx, cudaMemcpyAsync(out_lens, lens, n * sizeof(size_t), cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    size_t total = 0;
    for (uint32_t k = 0; k < n; k++) total += out_lens[k];
    CK(ctx, cudaMemcpyAsync(out, m + o_out, total, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    return RT_OK;
}

}  // namespace rtb

extern "C" {

size_t rt_world_json_max_objects(size_t len) { return len / (kMinObject + 1) + 1; }

size_t rt_slice_json_bound(uint32_t rows, uint32_t width) {
    return kHeaderMax + (size_t)rows * width * 3 * 4 + kTrailer;  // a value is at most 3 digits and a comma
}

int rt_world_parse_json(rt_ctx* ctx, const char* text, size_t len, rt_sphere* spheres, rt_triangle* triangles,
                        uint32_t* world_index, size_t cap, uint32_t* n_spheres, uint32_t* n_triangles, size_t* consumed) {
    if (!ctx) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    if (!text || !spheres || !triangles || !world_index || !n_spheres || !n_triangles || !consumed)
        return set_err(ctx, RT_ERR_INVALID_ARG, "rt_world_parse_json: NULL pointer");
    const size_t bound = rt_world_json_max_objects(len);
    if (cap < bound)
        return set_err(ctx, RT_ERR_INVALID_ARG, "rt_world_parse_json: cap %zu < rt_world_json_max_objects(%zu) = %zu", cap,
                       len, bound);
    if (len > 0xFFFFFFFFull - kTextPad - kTextChunk)
        return set_err(ctx, RT_ERR_UNSUPPORTED, "rt_world_parse_json: %zu bytes (positions are 32-bit)", len);
    const uint8_t* t = reinterpret_cast<const uint8_t*>(text);
    size_t i = 0;
    while (i < len && json_ws(t[i])) i++;
    if (i == len || t[i] != '[') return set_err(ctx, RT_ERR_UNSUPPORTED, "rt_world_parse_json: no array at the start");
    size_t j = i + 1;
    while (j < len && json_ws(t[j])) j++;
    if (j < len && t[j] == ']') {  // the empty world
        *n_spheres = *n_triangles = 0;
        *consumed = j + 1;
        return RT_OK;
    }
    if (j == len || t[j] != '{') return set_err(ctx, RT_ERR_UNSUPPORTED, "rt_world_parse_json: not an array of Object");
    CK(ctx, cudaSetDevice(ctx->device));
    const uint32_t chunks = (uint32_t)((len + kTextChunk - 1) / kTextChunk), text_ctas = (chunks + kScanThreads - 1) / kScanThreads;
    const uint32_t obj_ctas = (uint32_t)((cap + kScanThreads - 1) / kScanThreads);
    Carver cv;
    const size_t o_text = cv.take((size_t)chunks * kTextChunk + kTextPad), o_local = cv.take((size_t)chunks * sizeof(uint32_t)),
                 o_sums = cv.take((text_ctas + 1) * sizeof(unsigned long long)), o_starts = cv.take(cap * sizeof(uint32_t)),
                 o_recs = cv.take(cap * kRecFloats * sizeof(float)), o_status = cv.take(cap),
                 o_klocal = cv.take((size_t)obj_ctas * kScanThreads * sizeof(uint32_t)),
                 o_ksums = cv.take((obj_ctas + 1) * sizeof(unsigned long long)), o_ctl = cv.take(2 * sizeof(unsigned long long)),
                 o_sph = cv.take(cap * sizeof(rt_sphere)), o_tri = cv.take(cap * sizeof(rt_triangle)),
                 o_wi = cv.take(cap * sizeof(uint32_t));
    int rc = ensure_wire_scratch(ctx, cv.o);
    if (rc) return rc;
    uint8_t* m = ctx->d_wire;
    const uint8_t* d_text = m + o_text;
    uint32_t* local = reinterpret_cast<uint32_t*>(m + o_local);
    unsigned long long* sums = reinterpret_cast<unsigned long long*>(m + o_sums);
    uint32_t* starts = reinterpret_cast<uint32_t*>(m + o_starts);
    float* recs = reinterpret_cast<float*>(m + o_recs);
    uint8_t* status = m + o_status;
    uint32_t* klocal = reinterpret_cast<uint32_t*>(m + o_klocal);
    unsigned long long* ksums = reinterpret_cast<unsigned long long*>(m + o_ksums);
    unsigned long long* first_end = reinterpret_cast<unsigned long long*>(m + o_ctl);
    unsigned int* decline = reinterpret_cast<unsigned int*>(first_end + 1);
    rt_sphere* d_sph = reinterpret_cast<rt_sphere*>(m + o_sph);
    rt_triangle* d_tri = reinterpret_cast<rt_triangle*>(m + o_tri);
    uint32_t* d_wi = reinterpret_cast<uint32_t*>(m + o_wi);
    cudaStream_t s = ctx->stream;
    CK(ctx, cudaMemcpyAsync(m + o_text, text, len, cudaMemcpyHostToDevice, s));
    CK(ctx, cudaMemsetAsync(m + o_text + len, 0, (size_t)chunks * kTextChunk + kTextPad - len, s));
    CK(ctx, cudaMemsetAsync(first_end, 0xFF, sizeof(unsigned long long), s));
    CK(ctx, cudaMemsetAsync(decline, 0, sizeof(unsigned int), s));
    CK(ctx, cudaEventRecord(ctx->ev0, s));
    wire_starts_kernel<false><<<text_ctas, kScanThreads, 0, s>>>(d_text, (uint32_t)len, chunks, local, sums, nullptr, 0);
    CK(ctx, scan_carry(sums, text_ctas, s));
    wire_starts_kernel<true><<<text_ctas, kScanThreads, 0, s>>>(d_text, (uint32_t)len, chunks, local, sums, starts, (uint32_t)cap);
    const unsigned long long* n_starts = sums + text_ctas;
    wire_object_kernel<<<obj_ctas, kScanThreads, 0, s>>>(d_text, starts, n_starts, (uint32_t)cap, (uint32_t)j, recs, status,
                                                          first_end);
    wire_kind_kernel<<<obj_ctas, kScanThreads, 0, s>>>(status, n_starts, (uint32_t)cap, first_end, klocal, ksums, decline);
    CK(ctx, scan_carry(ksums, obj_ctas, s));
    wire_scatter_kernel<<<obj_ctas, kScanThreads, 0, s>>>(status, recs, first_end, klocal, ksums, obj_ctas, d_sph, d_tri, d_wi);
    CK(ctx, cudaGetLastError());
    CK(ctx, cudaEventRecord(ctx->ev1, s));
    unsigned long long* h = ctx->h_wire;
    CK(ctx, cudaMemcpyAsync(h, first_end, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaMemcpyAsync(h + 1, decline, sizeof(unsigned int), cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaMemcpyAsync(h + 2, ksums + obj_ctas, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    if (h[0] == kNoEnd || (uint32_t)h[1])
        return set_err(ctx, RT_ERR_UNSUPPORTED, "rt_world_parse_json: the world is outside the device grammar");
    const uint32_t n = (uint32_t)(h[0] >> 32) + 1, ns = (uint32_t)h[2];
    if (ns) CK(ctx, cudaMemcpyAsync(spheres, d_sph, ns * sizeof(rt_sphere), cudaMemcpyDeviceToHost, s));
    if (n > ns) CK(ctx, cudaMemcpyAsync(triangles, d_tri, (n - ns) * sizeof(rt_triangle), cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaMemcpyAsync(world_index, d_wi, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    *n_spheres = ns;
    *n_triangles = n - ns;
    *consumed = (uint32_t)h[0] + 1;
    return RT_OK;
    RT_GUARD_END(ctx)
}

}  // extern "C"
