// rt_exact_check.cu — lib/librt_b200_check.so (`make check`), a test library built apart from the product: the guarded
// fast paths of rt_device.cuh against the plain __fdiv_rn / __fsqrt_rn forms they replace, on the device, bit for bit
// (tests/test_exact_fastpath.py).
#include "rt_device.cuh"
#include "../../include/rt_b200.h"

namespace rtb {

__device__ __forceinline__ void fp_count(unsigned long long* n, bool bad) {
    const unsigned m = __ballot_sync(__activemask(), bad);
    if (m && (threadIdx.x & 31) == (uint32_t)(__ffs(__activemask()) - 1)) atomicAdd(n, (unsigned long long)__popc(m));
}
__device__ __forceinline__ bool fp_ne(float a, float b) { return __float_as_uint(a) != __float_as_uint(b); }

// every float32 bit pattern as numerator (and as square-root argument) against every divisor
__global__ void fp_div_kernel(const float* div, uint32_t n_div, unsigned long long* bad, unsigned long long* checked) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    unsigned long long ck = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (1ull << 32); i += stride) {
        const float a = __uint_as_float((uint32_t)i);
        bool wrong = x_sqrt_domain(a) && fp_ne(x_sqrt_fast(a), x_sqrt_ool(a));
        const bool num = x_div_num(a);
        for (uint32_t k = 0; k < n_div; k++) {
            const float b = div[k];
            if (!(num && x_div_mag(b))) continue;
            ck++;
            const float r = x_rcp_refined(b), q = __fdiv_rn(a, b);
            wrong |= fp_ne(x_quot(a, b, r), q);
            if (a != 0.0f) wrong |= fp_ne(x_quot_nz(a, b, r), q);
        }
        fp_count(bad, wrong);
    }
    atomicAdd(checked, ck);
}

// a vector's normalisations and inverse direction, and sphere roots on (d, oc, r2)
__global__ void fp_vec_kernel(const float* v, uint32_t n_vec, const float* s, uint32_t n_sph, unsigned long long* bad) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    bool wrong = false;
    if (i < n_vec) {
        const V3 a = mk(v[3 * i], v[3 * i + 1], v[3 * i + 2]);
        const V3 orv = mk(7.0f, 8.0f, 9.0f);
        auto ne3 = [](V3 p, V3 q) { return fp_ne(p.x, q.x) || fp_ne(p.y, q.y) || fp_ne(p.z, q.z); };
        wrong |= ne3(x_normalize_div(a), x_normalize_div_slow(a));
        const float rcp = x_rcp_length_slow(a);
        const bool some = isfinite(rcp) && rcp > 0.0f;
        wrong |= ne3(x_normalize_or(a, orv), some ? x_scale(a, rcp) : orv);
        V3 t = orv;
        wrong |= x_try_normalize(a, &t) != some || ne3(t, some ? x_scale(a, rcp) : orv);
        wrong |= ne3(x_normalize_div_or_zero(a), x_normalize_div_or_zero_slow(a));
        wrong |= ne3(x_rcp3(a), x_rcp3_slow(a));
        const float l2 = x_dot(a, a);
        wrong |= fp_ne(x_sqrt_domain(l2) ? x_sqrt_fast(l2) : x_sqrt_ool(l2), x_sqrt_ool(l2));
    }
    if (i < n_sph) {
        const float* r = s + 7 * i;
        const V3 d = mk(r[0], r[1], r[2]), oc = mk(r[3], r[4], r[5]);
        float t = -1.0f;
        const bool hit = sphere_root_exact(d, oc, r[6], &t);
        const float ts = sphere_root_slow(d, oc, r[6]);
        wrong |= hit != (ts == ts) || (hit && fp_ne(t, ts));
    }
    fp_count(bad, wrong);
}

}  // namespace rtb

// Every float32 bit pattern is a numerator against each of the n_div divisors, and a square-root argument; vecs holds n_vec
// 3-vectors, sph n_sph records d.xyz, oc.xyz, r*r.  out[0] / out[1] = bitwise mismatches (scalars / vectors and sphere
// roots), out[2] = the number of (numerator, divisor) pairs inside the guarded domain that were compared.
extern "C" int rt_debug_exact_fastpath(const float* divisors, uint32_t n_div, const float* vecs, uint32_t n_vec,
                                       const float* sph, uint32_t n_sph, uint64_t* out) {
    using namespace rtb;
    if (!out || (n_div && !divisors) || (n_vec && !vecs) || (n_sph && !sph)) return RT_ERR_INVALID_ARG;
    float *d_div = nullptr, *d_vec = nullptr, *d_sph = nullptr;
    unsigned long long* d_n = nullptr;
    cudaError_t e = cudaMalloc(&d_div, sizeof(float) * (n_div + 1));
    if (e == cudaSuccess) e = cudaMalloc(&d_vec, sizeof(float) * (3 * (size_t)n_vec + 1));
    if (e == cudaSuccess) e = cudaMalloc(&d_sph, sizeof(float) * (7 * (size_t)n_sph + 1));
    if (e == cudaSuccess) e = cudaMalloc(&d_n, sizeof(unsigned long long) * 3);
    if (e == cudaSuccess) e = cudaMemcpy(d_div, divisors, sizeof(float) * n_div, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d_vec, vecs, sizeof(float) * 3 * (size_t)n_vec, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d_sph, sph, sizeof(float) * 7 * (size_t)n_sph, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemset(d_n, 0, sizeof(unsigned long long) * 3);
    if (e == cudaSuccess) {
        fp_div_kernel<<<148 * 16, 256>>>(d_div, n_div, d_n, d_n + 2);
        const uint32_t n = n_vec > n_sph ? n_vec : n_sph;
        if (n) fp_vec_kernel<<<(n + 255) / 256, 256>>>(d_vec, n_vec, d_sph, n_sph, d_n + 1);
        e = cudaGetLastError();
    }
    unsigned long long h[3] = {0, 0, 0};
    if (e == cudaSuccess) e = cudaMemcpy(h, d_n, sizeof(h), cudaMemcpyDeviceToHost);
    cudaFree(d_div);
    cudaFree(d_vec);
    cudaFree(d_sph);
    cudaFree(d_n);
    if (e != cudaSuccess) return RT_ERR_CUDA;
    out[0] = h[0];  // mismatches: divisions and square roots
    out[1] = h[1];  // mismatches: vectors and sphere roots
    out[2] = h[2];  // (numerator, divisor) pairs inside the division domain that were compared
    return RT_OK;
}
