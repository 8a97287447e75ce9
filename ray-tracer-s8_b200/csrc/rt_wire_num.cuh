// rt_wire_num.cuh — JSON number tokens to f32 exactly as the host path converts them (rt_b200/wire.py: Python's json
// module, then a float32 structured array): an integer token becomes a Python int, a token with a fraction or an exponent
// Python's correctly rounded float(token); either is then rounded to f32 to nearest.
//   integer, <= 19 digits   u64 exactly → f64 (RN) → f32 (RN); "-0" is the int 0, so +0.0
//   fraction / exponent     Eisel–Lemire (Lemire 2021, the fast_float formulation) → f64, then f32 (RN); "-0.0" is -0.0
// Declined (the host decides): more than 19 significant digits, a nonzero significand with a decimal exponent outside
// the table (rt_wire_pow5.h), and the one case the 128-bit product cannot decide.  Host and device code, so the
// conversion can be checked on a CPU.
// obj_number reads the number tokens of OBJ / MTL lines (rt_obj.cu) with the same conversion: see there.
#pragma once
#include <cstdint>
#include <cstring>

#include "rt_wire_pow5.h"

namespace rtb {

__host__ __device__ __forceinline__ bool json_ws(uint8_t c) { return c == ' ' || c == '\t' || c == '\n' || c == '\r'; }
__host__ __device__ __forceinline__ bool json_digit(uint8_t c) { return c >= '0' && c <= '9'; }

__host__ __device__ __forceinline__ uint64_t mul_hi64(uint64_t a, uint64_t b) {
#ifdef __CUDA_ARCH__
    return __umul64hi(a, b);
#else
    return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}

// w * 10^q as the bits of the nearest f64 (w != 0, q in the table): false when undecided.
__host__ __device__ inline bool eisel_lemire(uint64_t w, int q, uint64_t* bits) {
#ifdef __CUDA_ARCH__
    const int lz = __clzll((long long)w);
#else
    const int lz = __builtin_clzll(w);
#endif
    w <<= lz;
    const uint64_t* t = rt_pow5 + 2 * (q - RT_POW5_QMIN);
    uint64_t hi = mul_hi64(w, t[0]), lo = w * t[0];
    constexpr uint64_t kMask = ~0ull >> 55;  // 52 mantissa bits + 3
    if ((hi & kMask) == kMask) {  // the low word of the power can carry into the bits that decide the rounding
        const uint64_t s = mul_hi64(w, t[1]);
        lo += s;
        hi += lo < s;
    }
    if (lo == ~0ull && (q < -27 || q > 55)) return false;  // outside the range where the product is exact
    const int upper = (int)(hi >> 63), shift = upper + 9;
    uint64_t m = hi >> shift;
    int p2 = ((217706 * q) >> 16) + 63 + upper - lz + 1023;
    if (p2 <= 0) {  // subnormal (or zero)
        if (-p2 + 1 >= 64) {
            *bits = 0;
            return true;
        }
        m >>= -p2 + 1;
        m += m & 1;
        m >>= 1;
        *bits = (m < (1ull << 52) ? 0ull : 1ull << 52) | (m & ((1ull << 52) - 1));
        return true;
    }
    if (lo <= 1 && q >= -4 && q <= 23 && (m & 3) == 1 && (m << shift) == hi) m &= ~1ull;  // exact tie: to even
    m += m & 1;
    m >>= 1;
    if (m >= (2ull << 52)) {
        m = 1ull << 52;
        p2++;
    }
    m &= ~(1ull << 52);
    *bits = p2 >= 0x7FF ? 0x7FFull << 52 : (uint64_t)p2 << 52 | m;
    return true;
}

__host__ __device__ __forceinline__ float f64_bits_to_f32(uint64_t bits) {
#ifdef __CUDA_ARCH__
    return __double2float_rn(__longlong_as_double((long long)bits));
#else
    double d;
    memcpy(&d, &bits, 8);
    return (float)d;
#endif
}

// The JSON number at p (no leading whitespace); on success p is just past it.  false: not a JSON number, or declined.
__host__ __device__ inline bool json_number(const uint8_t*& p, float* out) {
    const uint8_t* s = p;
    const bool neg = *s == '-';
    s += neg;
    if (!json_digit(*s)) return false;
    uint64_t w = 0;
    int sig = 0, nfrac = 0;
    const auto digit = [&](uint8_t c) {
        if (w || c != '0') {  // leading zeros are not significant
            sig += sig <= 19;
            w = w * 10 + (c - '0');
        }
    };
    if (*s == '0') s++;
    else
        while (json_digit(*s)) digit(*s++);
    bool is_int = true;
    if (*s == '.') {
        s++;
        if (!json_digit(*s)) return false;
        while (json_digit(*s)) {
            digit(*s++);
            nfrac += nfrac <= 100000;
        }
        is_int = false;
    }
    int e = 0;
    if (*s == 'e' || *s == 'E') {
        s++;
        const bool eneg = *s == '-';
        s += *s == '-' || *s == '+';
        if (!json_digit(*s)) return false;
        while (json_digit(*s)) {
            if (e < 100000) e = e * 10 + (*s - '0');
            s++;
        }
        e = eneg ? -e : e;
        is_int = false;
    }
    if (sig > 19 || nfrac > 100000) return false;
    if (is_int) {
        const float f = (float)(double)w;
        *out = neg && w ? -f : f;
    } else if (w == 0) {
        *out = neg ? -0.0f : 0.0f;
    } else {
        const int q = e - nfrac;
        uint64_t bits;
        if (q < RT_POW5_QMIN || q > RT_POW5_QMAX || !eisel_lemire(w, q, &bits)) return false;
        *out = f64_bits_to_f32(bits | (neg ? 1ull << 63 : 0));
    }
    p = s;
    return true;
}

// The OBJ / MTL number token [p, end), converted as rt_b200/obj.py does: float(np.float32(token)), i.e. Python's
// correctly rounded float(token), then f32 to nearest ("-0" is -0.0).  The device form is
// [+-]? (digits [. digits*] | . digits) ([eE] [+-]? digits)?; false: any other token (Python also takes "inf", "nan",
// "1_0" ...: the host decides), more than 19 significant digits, a nonzero significand with a decimal exponent outside
// the table, an undecided product, or a result that is not finite.
__host__ __device__ inline bool obj_number(const uint8_t* p, const uint8_t* end, float* out) {
    const bool neg = p < end && *p == '-';
    p += p < end && (*p == '-' || *p == '+');
    uint64_t w = 0;
    int sig = 0, nfrac = 0, ndig = 0;
    const auto digit = [&](uint8_t c) {
        if (w || c != '0') {  // leading zeros are not significant
            sig += sig <= 19;
            w = w * 10 + (c - '0');
        }
        ndig += ndig <= 1;
    };
    while (p < end && json_digit(*p)) digit(*p++);
    if (p < end && *p == '.') {
        p++;
        while (p < end && json_digit(*p)) {
            digit(*p++);
            nfrac += nfrac <= 100000;
        }
    }
    if (!ndig) return false;  // "." or no digits at all
    int e = 0;
    if (p < end && (*p == 'e' || *p == 'E')) {
        p++;
        const bool eneg = p < end && *p == '-';
        p += p < end && (*p == '-' || *p == '+');
        if (p == end || !json_digit(*p)) return false;
        while (p < end && json_digit(*p)) {
            if (e < 100000) e = e * 10 + (*p - '0');
            p++;
        }
        e = eneg ? -e : e;
    }
    if (p != end || sig > 19 || nfrac > 100000) return false;
    if (w == 0) {
        *out = neg ? -0.0f : 0.0f;
        return true;
    }
    const int q = e - nfrac;
    uint64_t bits;
    if (q < RT_POW5_QMIN || q > RT_POW5_QMAX || !eisel_lemire(w, q, &bits)) return false;
    const float f = f64_bits_to_f32(bits | (neg ? 1ull << 63 : 0));
    if (!(f >= -3.40282347e38f && f <= 3.40282347e38f)) return false;  // the host gives inf (with a warning)
    *out = f;
    return true;
}

}  // namespace rtb
