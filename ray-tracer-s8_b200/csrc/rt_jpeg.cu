// rt_jpeg.cu — baseline JPEG of an RGB8 frame in device memory, byte-identical to libjpeg's defaults at quality q (the
// controller's JPEG(90), ray-tracer-controller/src/main.rs:95-142): JFIF 1.01, 4:2:0, the standard Huffman tables of
// T.81 Annex K, one scan with no restart markers.  Every step is integer, so "identical" is a byte comparison.
//
//   jpeg_coef_kernel     one CTA per MCU: colour conversion (jccolor.c), 2x2 downsampling with the 1,2 bias (jcsample.c),
//                        edge replication (jcprepct.c), six jpeg_fdct_islow (jfdctint.c), quantisation, dummy blocks
//                        (jccoefct.c compress_data) → int16 coefficients in zigzag order, 384 per MCU
//   jpeg_bits_kernel     one thread per block: Huffman bits of the block (DC against the preceding block of its
//                        component) and their exclusive sum within the CTA
//   jpeg_carry_kernel    one CTA: exclusive sum of the CTA totals → every block's bit offset, and the total
//   jpeg_emit_kernel     one thread per block writes its bits at its offset, MSB first, into zeroed 32-bit words; only
//                        the first and the last word of its span can be shared with a neighbour (atomicOr)
//   jpeg_ff_kernel       one thread per 32-byte chunk of the coded bytes (last byte padded with 1-bits): 0xFF count
//                        and its exclusive sum within the CTA; jpeg_carry_kernel again over the CTA totals
//   jpeg_stuff_kernel    one thread per chunk copies its bytes to their final place with 0x00 after every 0xFF; the
//                        chunk holding the last byte appends EOI and stores the segment's length
// The header (623 bytes) depends only on width, height and quality and is written by the host.
#include <cub/block/block_scan.cuh>

#include <climits>
#include <cstring>

#include "rt_ctx.h"

using namespace rtb;

namespace {

constexpr int kHeaderBytes = 623;
constexpr int kScanThreads = 256;    // blocks / chunks per CTA of the bit-count and 0xFF-count kernels
constexpr int kCarryThreads = 512;
constexpr int kChunkBytes = 32;
constexpr int kMaxBlockBits = 22 + 63 * 26;  // see rt_jpeg_bound

// zigzag index → natural (row-major) index
constexpr uint8_t kZigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                 41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
// Annex K.1 base tables, natural order
constexpr uint8_t kBaseQuant[2][64] = {
    {16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,  14, 13, 16, 24, 40,  57,
     69, 56, 14, 17, 22,  29,  51,  87,  80, 62, 18, 22, 37,  56,  68,  109, 103, 77, 24, 35, 55,  64,
     81, 104, 113, 92, 49, 64, 78,  87,  103, 121, 120, 101, 72, 92, 95, 98,  112, 100, 103, 99},
    {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99,
     99, 99, 47, 66, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
     99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99}};

// Annex K.3 Huffman tables: code counts per length 1..16, then the symbols in code order
struct HuffSpec {
    uint8_t bits[16];
    uint8_t vals[162];
};
constexpr HuffSpec kDcLuma = {{0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0}, {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11}};
constexpr HuffSpec kDcChroma = {{0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0}, {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11}};
constexpr HuffSpec kAcLuma = {
    {0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d},
    {0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71, 0x14,
     0x32, 0x81, 0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72, 0x82, 0x09,
     0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a,
     0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65,
     0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88,
     0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9,
     0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca,
     0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea,
     0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa}};
constexpr HuffSpec kAcChroma = {
    {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77},
    {0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22, 0x32,
     0x81, 0x08, 0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1, 0x0a, 0x16,
     0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36, 0x37, 0x38, 0x39,
     0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64,
     0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x82, 0x83, 0x84, 0x85, 0x86,
     0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7,
     0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8,
     0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9,
     0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa}};

constexpr int spec_count(const HuffSpec& s) {
    int n = 0;
    for (int i = 0; i < 16; i++) n += s.bits[i];
    return n;
}

// Canonical codes (Annex C), one word per symbol: code << 8 | length (0: no code)
struct HuffTables {
    uint32_t dc[2][16];
    uint32_t ac[2][256];
};
constexpr void fill_codes(const HuffSpec& s, uint32_t* out) {
    uint32_t code = 0;
    int k = 0;
    for (int len = 1; len <= 16; len++) {
        for (int i = 0; i < s.bits[len - 1]; i++) out[s.vals[k++]] = code++ << 8 | (uint32_t)len;
        code <<= 1;
    }
}
constexpr HuffTables make_tables() {
    HuffTables t{};
    fill_codes(kDcLuma, t.dc[0]);
    fill_codes(kDcChroma, t.dc[1]);
    fill_codes(kAcLuma, t.ac[0]);
    fill_codes(kAcChroma, t.ac[1]);
    return t;
}
__constant__ HuffTables c_huff = make_tables();
__constant__ uint8_t c_zigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,
                                     12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,  7,  14, 21, 28,
                                     35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51,
                                     58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

struct Quant {
    uint16_t q[2][64];  // luma, chroma: natural order
};

// jpeg_quality_scaling + jpeg_add_quant_table with force_baseline
Quant quant_tables(uint32_t quality) {
    const int scale = quality < 50 ? 5000 / (int)quality : 200 - 2 * (int)quality;
    Quant t;
    for (int c = 0; c < 2; c++)
        for (int i = 0; i < 64; i++) t.q[c][i] = (uint16_t)std::min(255, std::max(1, (kBaseQuant[c][i] * scale + 50) / 100));
    return t;
}

struct Geometry {
    uint32_t width, height, mx, my;  // MCUs per row, MCU rows
    uint32_t bw, bh;                 // luma blocks that hold image data (ceil(w / 8), ceil(h / 8)): the rest are dummies
    uint32_t hc;                     // chroma rows that hold image data: ceil(h / 2)
};
Geometry geometry(uint32_t w, uint32_t h) {
    return {w, h, (w + 15) / 16, (h + 15) / 16, (w + 7) / 8, (h + 7) / 8, (h + 1) / 2};
}

// ------------------------------------------------------------------------------------------------
// Coefficients
// ------------------------------------------------------------------------------------------------
constexpr int FIX_0_298631336 = 2446, FIX_0_390180644 = 3196, FIX_0_541196100 = 4433, FIX_0_765366865 = 6270,
              FIX_0_899976223 = 7373, FIX_1_175875602 = 9633, FIX_1_501321110 = 12299, FIX_1_847759065 = 15137,
              FIX_1_961570560 = 16069, FIX_2_053119869 = 16819, FIX_2_562915447 = 20995, FIX_3_072711026 = 25172;

// One 8-point pass of jpeg_fdct_islow over d[0], d[stride], ... d[7 * stride], in place.  For 8-bit samples every
// intermediate fits 32 bits (as in libjpeg's own SIMD forms).
template <bool FIRST>
__device__ __forceinline__ void fdct_pass(int* d, int stride) {
    constexpr int CONST_BITS = 13, PASS1_BITS = 2;
    constexpr int n = FIRST ? CONST_BITS - PASS1_BITS : CONST_BITS + PASS1_BITS;
    const auto descale = [](int x, int s) { return (x + (1 << (s - 1))) >> s; };
    const int tmp0 = d[0] + d[7 * stride], tmp7 = d[0] - d[7 * stride];
    const int tmp1 = d[stride] + d[6 * stride], tmp6 = d[stride] - d[6 * stride];
    const int tmp2 = d[2 * stride] + d[5 * stride], tmp5 = d[2 * stride] - d[5 * stride];
    const int tmp3 = d[3 * stride] + d[4 * stride], tmp4 = d[3 * stride] - d[4 * stride];
    const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    if (FIRST) {
        d[0] = (tmp10 + tmp11) << PASS1_BITS;
        d[4 * stride] = (tmp10 - tmp11) << PASS1_BITS;
    } else {
        d[0] = descale(tmp10 + tmp11, PASS1_BITS);
        d[4 * stride] = descale(tmp10 - tmp11, PASS1_BITS);
    }
    int z1 = (tmp12 + tmp13) * FIX_0_541196100;
    d[2 * stride] = descale(z1 + tmp13 * FIX_0_765366865, n);
    d[6 * stride] = descale(z1 - tmp12 * FIX_1_847759065, n);
    z1 = tmp4 + tmp7;
    int z2 = tmp5 + tmp6, z3 = tmp4 + tmp6, z4 = tmp5 + tmp7;
    const int z5 = (z3 + z4) * FIX_1_175875602;
    z1 *= -FIX_0_899976223;
    z2 *= -FIX_2_562915447;
    z3 = z3 * -FIX_1_961570560 + z5;
    z4 = z4 * -FIX_0_390180644 + z5;
    d[7 * stride] = descale(tmp4 * FIX_0_298631336 + z1 + z3, n);
    d[5 * stride] = descale(tmp5 * FIX_2_053119869 + z2 + z4, n);
    d[3 * stride] = descale(tmp6 * FIX_3_072711026 + z2 + z3, n);
    d[stride] = descale(tmp7 * FIX_1_501321110 + z1 + z4, n);
}

__global__ void __launch_bounds__(256) jpeg_coef_kernel(const uint8_t* __restrict__ rgb, Geometry g, Quant qt,
                                                        int16_t* __restrict__ coef) {
    __shared__ int s_cb[16][16], s_cr[16][16];  // full-resolution chroma of the MCU's 16 x 16 input pixels
    __shared__ int s_blk[6][64];                // Y00 Y01 Y10 Y11 Cb Cr, natural order, centred on 0, DCT in place
    __shared__ uint16_t s_div[2][64];
    __shared__ uint8_t s_zigzag[64];
    __shared__ int s_dummy_dc[4];               // dummy luma block k: its DC, else INT_MIN
    const uint32_t mcu = blockIdx.x, mcu_x = mcu % g.mx, mcu_y = mcu / g.mx;
    const int t = threadIdx.x;
    if (t < 128) s_div[t >> 6][t & 63] = (uint16_t)(qt.q[t >> 6][t & 63] * 8);
    else if (t < 192) s_zigzag[t - 128] = c_zigzag[t - 128];
    {   // colour conversion (rgb_ycc_convert): columns past the image repeat its last column, rows its last row
        const int px = t & 15, py = t >> 4;
        const uint32_t x = min(mcu_x * 16 + px, g.width - 1), y = min(mcu_y * 16 + py, g.height - 1);
        const uint8_t* p = rgb + ((size_t)y * g.width + x) * 3;
        const int r = p[0], gg = p[1], b = p[2];
        constexpr int ONE_HALF = 1 << 15, CBCR_OFFSET = 128 << 16;
        const int Y = (19595 * r + 38470 * gg + 7471 * b + ONE_HALF) >> 16;  // FIX(0.29900) FIX(0.58700) FIX(0.11400)
        s_cb[py][px] = (-11059 * r - 21709 * gg + 32768 * b + CBCR_OFFSET + ONE_HALF - 1) >> 16;  // FIX(0.16874) FIX(0.33126)
        s_cr[py][px] = (32768 * r - 27439 * gg - 5329 * b + CBCR_OFFSET + ONE_HALF - 1) >> 16;    // FIX(0.41869) FIX(0.08131)
        s_blk[(py >> 3) * 2 + (px >> 3)][(py & 7) * 8 + (px & 7)] = Y - 128;
    }
    __syncthreads();
    if (t < 128) {  // h2v2 downsampling; chroma rows past ceil(h/2) repeat the last downsampled row (jcprepct.c)
        const int c = t >> 6, cx = t & 7, cy = (t >> 3) & 7;
        const int ry = (int)min(mcu_y * 8 + cy, g.hc - 1) - (int)(mcu_y * 8);
        const int(*s)[16] = c ? s_cr : s_cb;
        const int sum = s[2 * ry][2 * cx] + s[2 * ry][2 * cx + 1] + s[2 * ry + 1][2 * cx] + s[2 * ry + 1][2 * cx + 1];
        s_blk[4 + c][cy * 8 + cx] = ((sum + 1 + (cx & 1)) >> 2) - 128;
    }
    __syncthreads();
    if (t < 48) fdct_pass<true>(&s_blk[t >> 3][(t & 7) * 8], 1);  // rows
    __syncthreads();
    if (t < 48) fdct_pass<false>(&s_blk[t >> 3][t & 7], 8);       // columns
    __syncthreads();
    for (int i = t; i < 6 * 64; i += 256) {  // quantise: magnitude rounded half up
        const int b = i >> 6, k = i & 63;
        const int d = s_div[b >= 4][k], x = s_blk[b][k], a = abs(x);
        const int q = a < (d >> 1) ? 0 : (a + (d >> 1)) / d;
        s_blk[b][k] = x < 0 ? -q : q;
    }
    __syncthreads();
    if (t == 0) {  // dummy luma blocks (jccoefct.c): zero, with the DC of the block before in MCU order
        int dc[4];
        for (int k = 0; k < 4; k++) {
            dc[k] = s_blk[k][0];
            s_dummy_dc[k] = INT_MIN;
            if (mcu_y * 2 + (k >> 1) >= g.bh) s_dummy_dc[k] = dc[k] = dc[1];  // bottom row: the last block of the row above
            else if (mcu_x * 2 + (k & 1) >= g.bw) s_dummy_dc[k] = dc[k] = dc[k - 1];  // right edge: the left neighbour
        }
    }
    __syncthreads();
    int16_t* out = coef + (size_t)mcu * 384;
    for (int i = t; i < 6 * 64; i += 256) {
        const int b = i >> 6, k = i & 63;
        int v = s_blk[b][s_zigzag[k]];
        if (b < 4 && s_dummy_dc[b] != INT_MIN) v = k ? 0 : s_dummy_dc[b];
        out[i] = (int16_t)v;
    }
}

// ------------------------------------------------------------------------------------------------
// Entropy coding
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int magnitude_bits(int v) { return v ? 32 - __clz(abs(v)) : 0; }

// Codes block z (zigzag) against the DC predictor `pred` into sink.put(bits, length), length <= 26 per call.
template <class Sink>
__device__ __forceinline__ void code_block(const int16_t* __restrict__ z, int pred, const uint32_t* dc,
                                           const uint32_t* ac, Sink& sink) {
    const uint4* zv = reinterpret_cast<const uint4*>(z);
    const int diff = z[0] - pred;
    int n = magnitude_bits(diff);
    sink.put((dc[n] >> 8) << n | ((diff < 0 ? diff - 1 : diff) & ((1 << n) - 1)), (dc[n] & 0xff) + n);
    int run = 0;
#pragma unroll 1
    for (int w = 0; w < 8; w++) {
        const uint4 u = zv[w];
        const uint32_t pairs[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int j = 0; j < 8; j++) {
            if (w == 0 && j == 0) continue;  // the DC
            const int v = (int16_t)(pairs[j >> 1] >> ((j & 1) * 16));
            if (v == 0) {
                run++;
                continue;
            }
            for (; run >= 16; run -= 16) sink.put(ac[0xF0] >> 8, ac[0xF0] & 0xff);  // ZRL
            n = magnitude_bits(v);
            const uint32_t c = ac[run << 4 | n];
            sink.put((c >> 8) << n | ((v < 0 ? v - 1 : v) & ((1 << n) - 1)), (c & 0xff) + n);
            run = 0;
        }
    }
    if (run) sink.put(ac[0] >> 8, ac[0] & 0xff);  // EOB
}

// DC of the block of the same component that precedes block i (MCU order: Y00 Y01 Y10 Y11 Cb Cr); 0 for the first
__device__ __forceinline__ int dc_pred(const int16_t* __restrict__ coef, uint32_t i) {
    const uint32_t b = i % 6;
    if (b == 1 || b == 2 || b == 3) return coef[(size_t)(i - 1) * 64];
    if (i < 6) return 0;
    return coef[(size_t)(b == 0 ? i - 3 : i - 6) * 64];
}

struct SharedTables {
    uint32_t dc[16], ac[256];
};
__device__ __forceinline__ void load_tables(SharedTables* s) {  // [0] luma, [1] chroma
    for (int i = threadIdx.x; i < 2 * 272; i += blockDim.x) {
        const int c = i / 272, k = i % 272;
        if (k < 16) s[c].dc[k] = c_huff.dc[c][k];
        else s[c].ac[k - 16] = c_huff.ac[c][k - 16];
    }
    __syncthreads();
}

struct BitCount {
    uint32_t bits = 0;
    __device__ __forceinline__ void put(uint32_t, uint32_t len) { bits += len; }
};

using ScanU32 = cub::BlockScan<uint32_t, kScanThreads>;

__global__ void __launch_bounds__(kScanThreads) jpeg_bits_kernel(const int16_t* __restrict__ coef, uint32_t blocks,
                                                                 uint32_t* __restrict__ local,
                                                                 unsigned long long* __restrict__ cta_sum) {
    __shared__ SharedTables s_tab[2];
    __shared__ typename ScanU32::TempStorage s_scan;
    load_tables(s_tab);
    const uint32_t i = blockIdx.x * kScanThreads + threadIdx.x;
    BitCount c;
    if (i < blocks) {
        const SharedTables& tab = s_tab[i % 6 >= 4];
        code_block(coef + (size_t)i * 64, dc_pred(coef, i), tab.dc, tab.ac, c);
    }
    uint32_t off, total;
    ScanU32(s_scan).ExclusiveSum(c.bits, off, total);
    if (i < blocks) local[i] = off;
    if (threadIdx.x == 0) cta_sum[blockIdx.x] = total;
}

// In place: sums[0..n) → their exclusive sum; sums[n] = the total.
__global__ void __launch_bounds__(kCarryThreads) jpeg_carry_kernel(unsigned long long* sums, uint32_t n) {
    using Scan = cub::BlockScan<unsigned long long, kCarryThreads>;
    __shared__ typename Scan::TempStorage s_scan;
    unsigned long long carry = 0;
    for (uint32_t base = 0; base < n; base += kCarryThreads) {
        const uint32_t i = base + threadIdx.x;
        const unsigned long long v = i < n ? sums[i] : 0;
        unsigned long long off, total;
        Scan(s_scan).ExclusiveSum(v, off, total);
        if (i < n) sums[i] = carry + off;
        carry += total;
        __syncthreads();  // s_scan is reused
    }
    if (threadIdx.x == 0) sums[n] = carry;
}

// Bits of one block from absolute bit position `pos` on, MSB first, into 32-bit words (bit 31 first).  Words wholly
// inside the span are stored; the first and the last may hold a neighbour's bits and are ORed in.
struct BitWriter {
    uint32_t* words;
    size_t w;              // word the next full 32 bits go to
    unsigned long long acc = 0;
    uint32_t n;            // bits pending in acc (< 32 between calls)
    bool first = true;
    __device__ BitWriter(uint32_t* words_, unsigned long long pos) : words(words_), w(pos >> 5), n(pos & 31) {}
    __device__ __forceinline__ void put(uint32_t bits, uint32_t len) {
        acc = acc << len | bits;
        n += len;
        if (n >= 32) {
            n -= 32;
            const uint32_t word = (uint32_t)(acc >> n);
            if (first) atomicOr(&words[w], word);
            else words[w] = word;
            first = false;
            w++;
        }
    }
    __device__ __forceinline__ void flush() {
        if (n) atomicOr(&words[w], (uint32_t)(acc << (32 - n)));
    }
};

__global__ void __launch_bounds__(kScanThreads) jpeg_emit_kernel(const int16_t* __restrict__ coef, uint32_t blocks,
                                                                 const uint32_t* __restrict__ local,
                                                                 const unsigned long long* __restrict__ cta_off,
                                                                 uint32_t* __restrict__ words) {
    __shared__ SharedTables s_tab[2];
    load_tables(s_tab);
    const uint32_t i = blockIdx.x * kScanThreads + threadIdx.x;
    if (i >= blocks) return;
    const SharedTables& tab = s_tab[i % 6 >= 4];
    BitWriter wr(words, cta_off[blockIdx.x] + local[i]);
    code_block(coef + (size_t)i * 64, dc_pred(coef, i), tab.dc, tab.ac, wr);
    wr.flush();
}

// Bytes [c * 32, c * 32 + 32) of the coded bits: byte j of the stream is the (j % 4)-th most significant byte of word
// j / 4; the byte holding the last bit is padded with 1-bits.  Returns the number of those bytes that exist.
__device__ __forceinline__ uint32_t load_chunk(const uint32_t* __restrict__ words, uint32_t c,
                                               unsigned long long total_bits, uint8_t (&b)[kChunkBytes]) {
    const unsigned long long nbytes = (total_bits + 7) / 8, first = (unsigned long long)c * kChunkBytes;
    if (first >= nbytes) return 0;
    const uint4* p = reinterpret_cast<const uint4*>(words) + (size_t)c * 2;
    const uint4 u0 = p[0], u1 = p[1];
    const uint32_t w[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
    const uint8_t pad = (uint8_t)((1u << ((8 - (total_bits & 7)) & 7)) - 1);
#pragma unroll
    for (int j = 0; j < kChunkBytes; j++) {
        b[j] = (uint8_t)(w[j >> 2] >> (24 - 8 * (j & 3)));
        if (first + j == nbytes - 1) b[j] |= pad;
    }
    return (uint32_t)min((unsigned long long)kChunkBytes, nbytes - first);
}

__global__ void __launch_bounds__(kScanThreads) jpeg_ff_kernel(const uint32_t* __restrict__ words,
                                                               const unsigned long long* __restrict__ total_bits,
                                                               uint32_t chunks, uint32_t* __restrict__ local,
                                                               unsigned long long* __restrict__ cta_sum) {
    __shared__ typename ScanU32::TempStorage s_scan;
    const uint32_t c = blockIdx.x * kScanThreads + threadIdx.x;
    uint8_t b[kChunkBytes];
    const uint32_t valid = c < chunks ? load_chunk(words, c, *total_bits, b) : 0;
    uint32_t ff = 0;
#pragma unroll
    for (int j = 0; j < kChunkBytes; j++) ff += (uint32_t)j < valid && b[j] == 0xFF;
    uint32_t off, total;
    ScanU32(s_scan).ExclusiveSum(ff, off, total);
    if (c < chunks) local[c] = off;
    if (threadIdx.x == 0) cta_sum[blockIdx.x] = total;
}

__global__ void __launch_bounds__(kScanThreads) jpeg_stuff_kernel(const uint32_t* __restrict__ words,
                                                                  const unsigned long long* __restrict__ total_bits,
                                                                  uint32_t chunks, const uint32_t* __restrict__ local,
                                                                  const unsigned long long* __restrict__ cta_off,
                                                                  uint8_t* __restrict__ seg,
                                                                  unsigned long long* __restrict__ seg_len) {
    const uint32_t c = blockIdx.x * kScanThreads + threadIdx.x;
    if (c >= chunks) return;
    const unsigned long long bits = *total_bits, nbytes = (bits + 7) / 8;
    uint8_t b[kChunkBytes];
    const uint32_t valid = load_chunk(words, c, bits, b);
    if (!valid) return;
    unsigned long long o = (unsigned long long)c * kChunkBytes + cta_off[blockIdx.x] + local[c];
#pragma unroll
    for (uint32_t j = 0; j < kChunkBytes; j++) {
        if (j < valid) {
            seg[o++] = b[j];
            if (b[j] == 0xFF) seg[o++] = 0;
        }
    }
    if ((unsigned long long)c * kChunkBytes + valid == nbytes) {  // the last byte: EOI follows
        seg[o] = 0xFF;
        seg[o + 1] = 0xD9;
        *seg_len = o + 2;
    }
}

// Scratch of one encode, carved from ctx->d_jpeg (all offsets 256-byte aligned)
struct Layout {
    size_t coef, local_bits, sums_bits, words, local_ff, sums_ff, seg, seg_len, bytes;
    uint32_t blocks, bits_ctas, chunks, ff_ctas;
    size_t word_bytes;
};
Layout layout(const Geometry& g) {
    Layout l{};
    const size_t mcus = (size_t)g.mx * g.my;
    l.blocks = (uint32_t)(mcus * 6);
    l.bits_ctas = (l.blocks + kScanThreads - 1) / kScanThreads;
    const size_t raw = (mcus * 6 * kMaxBlockBits + 7) / 8;  // coded bytes before stuffing, at most
    l.chunks = (uint32_t)((raw + kChunkBytes - 1) / kChunkBytes);
    l.ff_ctas = (l.chunks + kScanThreads - 1) / kScanThreads;
    l.word_bytes = (size_t)l.chunks * kChunkBytes;
    size_t o = 0;
    const auto take = [&](size_t bytes) {
        const size_t at = o;
        o += (bytes + 255) / 256 * 256;
        return at;
    };
    l.coef = take(mcus * 384 * sizeof(int16_t));
    l.local_bits = take((size_t)l.blocks * sizeof(uint32_t));
    l.sums_bits = take(((size_t)l.bits_ctas + 1) * sizeof(unsigned long long));
    l.words = take(l.word_bytes);
    l.local_ff = take((size_t)l.chunks * sizeof(uint32_t));
    l.sums_ff = take(((size_t)l.ff_ctas + 1) * sizeof(unsigned long long));
    l.seg = take(2 * raw + 2 + 2);  // every byte stuffed, the padding byte, EOI
    l.seg_len = take(sizeof(unsigned long long));
    l.bytes = o;
    return l;
}

int ensure_jpeg_scratch(rt_ctx* ctx, size_t bytes) {
    if (!ctx->h_jpeg_len) CK(ctx, cudaMallocHost(&ctx->h_jpeg_len, sizeof(unsigned long long)));
    if (ctx->d_jpeg_bytes >= bytes) return RT_OK;
    if (ctx->d_jpeg) {
        CK(ctx, cudaStreamSynchronize(ctx->stream));
        CK(ctx, cudaFree(ctx->d_jpeg));
        ctx->d_jpeg = nullptr;
        ctx->d_jpeg_bytes = 0;
    }
    CK(ctx, cudaMalloc(&ctx->d_jpeg, bytes));
    ctx->d_jpeg_bytes = bytes;
    return RT_OK;
}

// SOI, APP0, DQT x2, SOF0, DHT x4, SOS: what libjpeg writes in front of the scan
void write_header(uint8_t* out, uint32_t w, uint32_t h, const Quant& qt) {
    uint8_t* p = out;
    const auto u8 = [&](int v) { *p++ = (uint8_t)v; };
    const auto u16 = [&](int v) { u8(v >> 8); u8(v & 0xff); };
    u16(0xFFD8);
    u16(0xFFE0); u16(16);
    for (const char c : {'J', 'F', 'I', 'F', '\0'}) u8(c);
    u8(1); u8(1); u8(0); u16(1); u16(1); u8(0); u8(0);  // version 1.01, no units, density 1 x 1, no thumbnail
    for (int t = 0; t < 2; t++) {
        u16(0xFFDB); u16(67); u8(t);
        for (int k = 0; k < 64; k++) u8(qt.q[t][kZigzag[k]]);
    }
    u16(0xFFC0); u16(17); u8(8); u16((int)h); u16((int)w); u8(3);
    u8(1); u8(0x22); u8(0);
    u8(2); u8(0x11); u8(1);
    u8(3); u8(0x11); u8(1);
    const HuffSpec* specs[4] = {&kDcLuma, &kAcLuma, &kDcChroma, &kAcChroma};
    const int classes[4] = {0x00, 0x10, 0x01, 0x11};
    for (int i = 0; i < 4; i++) {
        const int n = spec_count(*specs[i]);
        u16(0xFFC4); u16(19 + n); u8(classes[i]);
        for (int k = 0; k < 16; k++) u8(specs[i]->bits[k]);
        for (int k = 0; k < n; k++) u8(specs[i]->vals[k]);
    }
    u16(0xFFDA); u16(12); u8(3);
    u8(1); u8(0x00);
    u8(2); u8(0x11);
    u8(3); u8(0x11);
    u8(0); u8(63); u8(0);
}

}  // namespace

namespace rtb {

int jpeg_check(rt_ctx* ctx, uint32_t width, uint32_t height, uint32_t quality, const uint8_t* out, size_t out_cap,
               const size_t* out_len) {
    if (!out || !out_len) return set_err(ctx, RT_ERR_INVALID_ARG, "JPEG: out or out_len is NULL");
    if (width == 0 || height == 0 || width > 65535 || height > 65535)
        return set_err(ctx, RT_ERR_INVALID_ARG, "JPEG: %u x %u is outside 1..65535 (the SOF fields)", width, height);
    if (quality < 1 || quality > 100) return set_err(ctx, RT_ERR_INVALID_ARG, "JPEG: quality %u outside 1..100", quality);
    const size_t bound = rt_jpeg_bound(width, height);
    if (out_cap < bound)
        return set_err(ctx, RT_ERR_INVALID_ARG, "JPEG: out_cap %zu < rt_jpeg_bound(%u, %u) = %zu", out_cap, width, height, bound);
    return RT_OK;
}

int jpeg_encode_device(rt_ctx* ctx, const uint8_t* rgb_dev, uint32_t width, uint32_t height, uint32_t quality,
                       uint8_t* out, size_t* out_len, float* ms_out) {
    const Geometry g = geometry(width, height);
    const Layout l = layout(g);
    int rc = ensure_jpeg_scratch(ctx, l.bytes);
    if (rc) return rc;
    const Quant qt = quant_tables(quality);
    write_header(out, width, height, qt);
    uint8_t* m = ctx->d_jpeg;
    int16_t* coef = reinterpret_cast<int16_t*>(m + l.coef);
    uint32_t* local_bits = reinterpret_cast<uint32_t*>(m + l.local_bits);
    unsigned long long* sums_bits = reinterpret_cast<unsigned long long*>(m + l.sums_bits);
    uint32_t* words = reinterpret_cast<uint32_t*>(m + l.words);
    uint32_t* local_ff = reinterpret_cast<uint32_t*>(m + l.local_ff);
    unsigned long long* sums_ff = reinterpret_cast<unsigned long long*>(m + l.sums_ff);
    uint8_t* seg = m + l.seg;
    unsigned long long* seg_len = reinterpret_cast<unsigned long long*>(m + l.seg_len);
    cudaStream_t s = ctx->stream;
    CK(ctx, cudaEventRecord(ctx->ev0, s));
    CK(ctx, cudaMemsetAsync(words, 0, l.word_bytes, s));
    jpeg_coef_kernel<<<g.mx * g.my, 256, 0, s>>>(rgb_dev, g, qt, coef);
    jpeg_bits_kernel<<<l.bits_ctas, kScanThreads, 0, s>>>(coef, l.blocks, local_bits, sums_bits);
    jpeg_carry_kernel<<<1, kCarryThreads, 0, s>>>(sums_bits, l.bits_ctas);
    jpeg_emit_kernel<<<l.bits_ctas, kScanThreads, 0, s>>>(coef, l.blocks, local_bits, sums_bits, words);
    const unsigned long long* total_bits = sums_bits + l.bits_ctas;
    jpeg_ff_kernel<<<l.ff_ctas, kScanThreads, 0, s>>>(words, total_bits, l.chunks, local_ff, sums_ff);
    jpeg_carry_kernel<<<1, kCarryThreads, 0, s>>>(sums_ff, l.ff_ctas);
    jpeg_stuff_kernel<<<l.ff_ctas, kScanThreads, 0, s>>>(words, total_bits, l.chunks, local_ff, sums_ff, seg, seg_len);
    CK(ctx, cudaGetLastError());
    CK(ctx, cudaEventRecord(ctx->ev1, s));
    CK(ctx, cudaMemcpyAsync(ctx->h_jpeg_len, seg_len, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    const size_t n = (size_t)*ctx->h_jpeg_len;
    CK(ctx, cudaMemcpyAsync(out + kHeaderBytes, seg, n, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    *out_len = kHeaderBytes + n;
    if (ms_out) CK(ctx, cudaEventElapsedTime(ms_out, ctx->ev0, ctx->ev1));
    return RT_OK;
}

cudaError_t scan_carry(unsigned long long* sums, uint32_t n, cudaStream_t s) {
    jpeg_carry_kernel<<<1, kCarryThreads, 0, s>>>(sums, n);
    return cudaGetLastError();
}

cudaError_t jpeg_preload() {
    cudaFuncAttributes a;
    cudaError_t e;
    if ((e = cudaFuncGetAttributes(&a, jpeg_coef_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, jpeg_bits_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, jpeg_carry_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, jpeg_emit_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, jpeg_ff_kernel)) != cudaSuccess) return e;
    return cudaFuncGetAttributes(&a, jpeg_stuff_kernel);
}

}  // namespace rtb

extern "C" {

// Header + EOI + the padding byte + every MCU at its largest, each byte stuffed.  A block codes at most 22 bits of DC
// (a code of <= 11 bits and a magnitude of <= 11) and, for each of its 63 AC positions, at most 26 bits (a code of <= 16
// bits and a magnitude of <= 10): a nonzero coefficient codes its own symbol, a ZRL (<= 11 bits) stands for 16 zero
// positions and the EOB (<= 4 bits) for at least one.  So a 4:2:0 MCU (6 blocks) codes at most 6 * 1660 bits = 1245
// bytes, and 2490 once every byte is followed by a stuffed 0x00.
size_t rt_jpeg_bound(uint32_t width, uint32_t height) {
    const Geometry g = geometry(width, height);
    return kHeaderBytes + 2 + 2 + (size_t)g.mx * g.my * 2 * (6 * kMaxBlockBits / 8);
}

int rt_jpeg_encode(rt_ctx* ctx, const uint8_t* rgb, uint32_t width, uint32_t height, uint32_t quality, uint8_t* out,
                   size_t out_cap, size_t* out_len, float* ms_out) {
    if (!ctx) return RT_ERR_INVALID_ARG;
    RT_GUARD_BEGIN
    if (!rgb) return set_err(ctx, RT_ERR_INVALID_ARG, "rt_jpeg_encode: rgb is NULL");
    int rc = jpeg_check(ctx, width, height, quality, out, out_cap, out_len);
    if (rc) return rc;
    CK(ctx, cudaSetDevice(ctx->device));
    Frame f;  // the frame goes up into the context's staging frame
    if ((rc = own_frame(ctx, width, height, &f))) return rc;
    CK(ctx, cudaMemcpyAsync(f.dev, rgb, (size_t)width * height * 3, cudaMemcpyHostToDevice, ctx->stream));
    return jpeg_encode_device(ctx, f.dev, width, height, quality, out, out_len, ms_out);
    RT_GUARD_END(ctx)
}

}  // extern "C"
