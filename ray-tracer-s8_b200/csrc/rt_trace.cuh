// rt_trace.cuh — device code of the nearest-hit query and of the per-sample arithmetic (sm_100a).
//
// Included by the render kernel (rt_kernels.cu).  Everything that decides a path is in the EXACT domain of
// rt_device.cuh; the FILTER-domain tests here only cull.
//
//   K1 (trace_brute):  every primitive per query; the sphere FILTER runs on pairs of spheres in packed f32x2
//                      arithmetic (FADD2 / FMUL2 / FFMA2), exact reference arithmetic only where it passes.
//   K2 (trace_bvh_ch): ordered, distance-culled traversal of the traversal tree (DESIGN.md section 3: big primitives
//                      first, then a SAH or LBVH tree over the rest) with conservative FMA slab tests in
//                      centre/half-extent form and a branch-free visit; exact arithmetic at the leaves.
#pragma once
#include "rt_device.cuh"

namespace rtb {

constexpr int THREADS = 256;  // CTA size of the instrumented (COUNT) instantiations and of the global-memory kernels

struct Hit {
    float dist;  // length(point - origin), exact domain
    int pid;     // -1 = miss.  While a query runs, HIT_UNSURE may be set in a non-negative pid (see consider)
    V3 p;        // ray.at(t)
    bool unsure; // set by the trace functions when they return: the decision needed the tie-break tables before they
                 // had landed, the pixel is rendered again
};
// Carried in bit 30 of Hit::pid during a query instead of in a register of its own (pids are 26 bits; the kernel
// runs at its register cap and one more live value in the traversal loop costs more than these few masks).
constexpr int HIT_UNSURE = 0x40000000;
__device__ __forceinline__ void hit_finish(Hit& h) {
    h.unsure = h.pid >= 0 && (h.pid & HIT_UNSURE);
    if (h.pid >= 0) h.pid &= ~HIT_UNSURE;
}

struct Ctr {
    unsigned long long v[NUM_COUNTERS];
};

// Shared-memory view of the geometry arrays (or the global pointers when SMEM == false)
struct SceneView {
    const float4* sph2;  // brute-force kernel only
    const float4* sph;
    const float4* tri;
    uint32_t nodes_s;       // shared-memory kernel: shared-window address of node record 0 (already inside the child codes)
    const char* nodes_g;    // global-memory kernel: DevScene::lnode
};

// ld.shared by 32-bit shared-window address (a node code of the shared-memory kernel IS such an address)
#define RT_LDS_F4(v, addr, off) \
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4+" #off "];" : "=f"((v).x), "=f"((v).y), "=f"((v).z), "=f"((v).w) : "r"(addr))
#define RT_LDS_I2(v, addr, off) asm volatile("ld.shared.v2.s32 {%0,%1}, [%2+" #off "];" : "=r"((v).x), "=r"((v).y) : "r"(addr))

// ---------------------------------------------------------------------------------------------
// Leaf tests.  `best` is updated iff the candidate wins the reference's min_by: smaller
// length(p - o), ties to the smaller DFS leaf rank (shapes/mod.rs:174-182, bvh_impl.rs:373-398).
// ---------------------------------------------------------------------------------------------
// FILTER-domain shortcut for the reference's slab test on the shape's own box: when the hit point is inside
// the box by a margin that dominates every rounding error of ray.rs:174-194 (2^-23 relative on each slab
// product, plus the ~1e-6*t disagreement between a triangle's Moeller-Trumbore t and its flat box's slab t),
// the reference test passes for certain.  Axes on which the box is flat (lo == hi: an axis-aligned triangle)
// give the reference tmin == tmax bit for bit, so only the other axes need the margin.
__device__ __forceinline__ bool robustly_inside(V3 p, float t, V3 lo, V3 hi, float extra = 0.0f) {
    const float m0 = fmaf(4e-5f, fabsf(t), extra);
    bool ok = true;
    {
        const float m = fmaf(1e-6f, fabsf(p.x) + fabsf(lo.x) + fabsf(hi.x), m0);
        ok = ok && ((lo.x == hi.x) || ((p.x - lo.x >= m) && (hi.x - p.x >= m)));
    }
    {
        const float m = fmaf(1e-6f, fabsf(p.y) + fabsf(lo.y) + fabsf(hi.y), m0);
        ok = ok && ((lo.y == hi.y) || ((p.y - lo.y >= m) && (hi.y - p.y >= m)));
    }
    {
        const float m = fmaf(1e-6f, fabsf(p.z) + fabsf(lo.z) + fabsf(hi.z), m0);
        ok = ok && ((lo.z == hi.z) || ((p.z - lo.z >= m) && (hi.z - p.z >= m)));
    }
    return ok;
}

// What consider() reads of the scene, by value: a reference to the kernel's DevScene parameter must never reach an
// out-of-line function — taking its address makes the compiler copy the whole parameter block to local memory and
// read `sc.*` from there in the hot loops as well (measured: C3 38 → 50 ms).
struct HitCtx {
    const float4* leaf_box;
    const uint32_t* rank;
    const uint32_t* ref_up;
    const float4* ref_box;
    const int* aux_flag;
    uint32_t n;
    int aux_ready;
};
// Have the tie-break tables landed?  Known at launch, or polled (acquire: the tables were written before the flag).
__device__ __forceinline__ bool aux_now(const HitCtx& hc) {
    if (hc.aux_ready) return true;
    int v;
    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(hc.aux_flag) : "memory");
    return v != 0;
}
__device__ __forceinline__ HitCtx hit_ctx(const DevScene& sc) {
    return HitCtx{sc.leaf_box, sc.rank, sc.ref_up, sc.ref_box, sc.aux_flag, sc.ns + sc.nt, sc.aux_ready};
}

// Rays with a direction component of exactly +-0 make the reference's slab test produce inf / NaN planes
// (ray.rs:133-143,174-194 with the crate's own min/max, ray.rs:82-112), and then "the shape's own box passes"
// no longer implies that every ancestor's child box passes (e.g. d.z == 0 with o.z exactly on an ancestor's max
// plane gives tmax = NaN and the subtree is dropped; d.x == -0.0 makes every box fail).  Such rays re-run the
// reference's own test on every box of the leaf's ancestor chain in the REFERENCE tree, root side last.
__device__ __noinline__ bool ref_ancestors_pass(const uint32_t* ref_up, const float4* ref_box, uint32_t n, V3 o, V3 d, int pid) {
    // plain loads (not the read-only path): the tables may have landed while this kernel was running
    uint32_t u = ref_up[pid];  // (parent << 1) | side of the leaf; its own box is tested by the caller
    while (u != UP_ROOT) {
        u = ref_up[n + (u >> 1)];  // the parent's own slot in ITS parent
        if (u == UP_ROOT) break;   // the root node's box is never tested (bvh_impl.rs:373-398)
        const V3 lo = ld3(ref_box[2 * u]), hi = ld3(ref_box[2 * u + 1]);
        if (!ref_intersects_aabb(o, d, lo, hi)) return false;
    }
    return true;
}

__device__ __forceinline__ void consider(const HitCtx& hc, V3 o, V3 d, float t, int pid, Hit& best) {
    V3 p = x_add(o, x_scale(d, t));   // Ray::at: origin + t*direction
    int flag = 0;
    // bvh.traverse() (main.rs:113): the shape is a candidate only if the reference's slab test lets it through
    if (hc.n > 1) {
        const V3 blo = ld3(__ldg(&hc.leaf_box[2 * pid])), bhi = ld3(__ldg(&hc.leaf_box[2 * pid + 1]));
        const bool degenerate = (d.x == 0.0f) || (d.y == 0.0f) || (d.z == 0.0f);  // +-0: inf / NaN slabs
        if (degenerate) {
            if (!ref_intersects_aabb(o, d, blo, bhi)) return;
            if (!aux_now(hc)) flag = HIT_UNSURE;  // whether the ancestors pass is decided in the second pass
            else if (!ref_ancestors_pass(hc.ref_up, hc.ref_box, hc.n, o, d, pid)) return;
        } else if (!robustly_inside(p, t, blo, bhi) && !ref_intersects_aabb(o, d, blo, bhi)) {
            return;
        }
    }
    const V3 po = x_sub(p, o);
    const float dist2 = x_dot(po, po);
    const float dist = x_sqrt_domain(dist2) ? x_sqrt_fast(dist2) : x_sqrt_ool(dist2);  // = x_length(po)
    bool take;
    if (best.pid < 0) {
        take = true;
    } else if (best.dist > dist) {
        take = true;
        flag |= best.pid & HIT_UNSURE;  // sticky for the rest of the query
    } else if (best.dist == dist) {
        if (aux_now(hc)) {
            take = hc.rank[pid] < hc.rank[best.pid & ~HIT_UNSURE];  // plain loads: the tables may have landed mid-kernel
        } else {
            take = false;
            flag = HIT_UNSURE;
        }
    } else {
        take = false;  // includes NaN: partial_cmp → None → Less → incumbent kept
    }
    if (take) {
        best.dist = dist;
        best.pid = pid | flag;
        best.p = p;
    } else if (flag) {
        best.pid |= flag;  // best.pid >= 0 here: a candidate is only ever refused in favour of an incumbent
    }
}

// FMA Moeller-Trumbore with error-scaled margins: false only when the exact test (mesh.rs:109-161) must
// reject, or when the hit would be farther than the current best by more than the tie margin.
__device__ __forceinline__ bool triangle_filter(const float4* tri, int tidx, V3 o, V3 d, float cull) {
    const V3 a = ld3(tri[4 * tidx + 0]), ab = ld3(tri[4 * tidx + 1]), ac = ld3(tri[4 * tidx + 2]);
    const float ux = fmaf(d.y, ac.z, -ac.y * d.z), uy = fmaf(d.z, ac.x, -ac.z * d.x), uz = fmaf(d.x, ac.y, -ac.x * d.y);
    const float det = fmaf(ab.z, uz, fmaf(ab.y, uy, ab.x * ux));
    const float sdet = fabsf(ab.x * ux) + fabsf(ab.y * uy) + fabsf(ab.z * uz);
    if (fabsf(det) < 1e-5f + 1e-4f * sdet) return true;  // near-parallel: let the exact test decide
    const float inv = __frcp_rn(det), ainv = fabsf(inv);
    const float aox = o.x - a.x, aoy = o.y - a.y, aoz = o.z - a.z;
    const float mag = fabsf(aox) + fabsf(aoy) + fabsf(aoz);
    const float mab = fabsf(ab.x) + fabsf(ab.y) + fabsf(ab.z), mac = fabsf(ac.x) + fabsf(ac.y) + fabsf(ac.z);
    const float u = fmaf(aoz, uz, fmaf(aoy, uy, aox * ux)) * inv;
    // 1e-4 = ~800 ulp on the products actually summed; the second term covers cancellation inside d x ac
    const float eu = (1e-4f * (fabsf(aox * ux) + fabsf(aoy * uy) + fabsf(aoz * uz)) + 2e-6f * mag * mac) * ainv + 1e-5f;
    if (u < -eu || u > 1.0f + eu) return false;
    const float vx = fmaf(aoy, ab.z, -ab.y * aoz), vy = fmaf(aoz, ab.x, -ab.z * aox), vz = fmaf(aox, ab.y, -ab.x * aoy);
    const float v = fmaf(d.z, vz, fmaf(d.y, vy, d.x * vx)) * inv;
    const float ev = 1e-4f * mag * mab * ainv + 1e-5f;  // |d| = 1
    if (v < -ev || u + v > 1.0f + eu + ev) return false;
    const float t = fmaf(ac.z, vz, fmaf(ac.y, vy, ac.x * vx)) * inv;
    const float et = 1e-4f * mag * mab * mac * ainv + 1e-6f;
    if (t < 0.0009f - et || t > cull + et) return false;  // exact needs t in [T_MIN, T_MAX) and a chance to win
    return true;
}

// ---------------------------------------------------------------------------------------------
// K1: brute force
// ---------------------------------------------------------------------------------------------
// The hot loop is the FILTER alone, 11 FMA-pipe instructions + compare + branch per sphere:
//   oc = o - c (3 FADD, the reference's own first operation, so the exact path reuses it)
//   bh = d.oc, oc2 = oc.oc (2 FMUL + 4 FFMA);  m = bh*bh + (r^2 - 0.99998*oc2) (2 FFMA)
// m >= 0  <=>  the reference's discriminant 4*(bh^2 - (|oc|^2 - r^2)) is above -8e-5*|oc|^2 (~300 ulp of slack).
// Everything else (roots behind the origin, exact roots, slab check, min_by) runs only for the few spheres that pass.
template <bool COUNT>
__device__ __noinline__ void brute_sphere_slow(const HitCtx sc, const float4 s, int pid, V3 o, V3 d, Hit& best,
                                               Ctr& ctr) {
    const V3 oc = mk(x_sub(o.x, s.x), x_sub(o.y, s.y), x_sub(o.z, s.z));
    const float bh = fmaf(oc.z, d.z, fmaf(oc.y, d.y, oc.x * d.x));
    const float oc2 = fmaf(oc.z, oc.z, fmaf(oc.y, oc.y, oc.x * oc.x));
    if (bh > 0.0f && (oc2 - s.w) > 1e-4f * oc2) return;  // both roots behind the origin: not in [T_MIN, T_MAX)
    if (COUNT) ctr.v[CTR_SPH_EXACT]++;
    float t;
    if (!sphere_root_exact(d, oc, s.w, &t)) return;
    if (COUNT) ctr.v[CTR_SPH_HIT]++;
    consider(sc, o, d, t, pid, best);
}

__device__ __forceinline__ float brute_margin(const float4 s, V3 o, V3 d) {
    const float ocx = x_sub(o.x, s.x), ocy = x_sub(o.y, s.y), ocz = x_sub(o.z, s.z);
    const float bh = fmaf(ocz, d.z, fmaf(ocy, d.y, ocx * d.x));
    const float oc2 = fmaf(ocz, ocz, fmaf(ocy, ocy, ocx * ocx));
    return fmaf(bh, bh, fmaf(oc2, -0.99998f, s.w));
}

// a group of 8 spheres (first is a multiple of 8) in which at least one passed the filter: the four pairs once more
// in packed arithmetic, this time keeping WHICH spheres passed, then the slow path for exactly those
template <bool COUNT>
__device__ __noinline__ void brute_group_slow(const HitCtx sc, const float4* sph, const float4* sph2, int first, int count,
                                              V3 o, V3 d, bool all, Hit& best, Ctr& ctr) {
    const f32x2 ox2 = pk2(o.x, o.x), oy2 = pk2(o.y, o.y), oz2 = pk2(o.z, o.z);
    const f32x2 dx2 = pk2(d.x, d.x), dy2 = pk2(d.y, d.y), dz2 = pk2(d.z, d.z);
    const f32x2 kk2 = pk2(-0.99998f, -0.99998f);
    unsigned mask = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const float4 A = sph2[2 * ((first >> 1) + k)], B = sph2[2 * ((first >> 1) + k) + 1];
        const f32x2 ocx = add2(ox2, pk2(A.x, A.y)), ocy = add2(oy2, pk2(A.z, A.w)), ocz = add2(oz2, pk2(B.x, B.y));
        const f32x2 bh = fma2(ocz, dz2, fma2(ocy, dy2, mul2(ocx, dx2)));
        const f32x2 oc2 = fma2(ocz, ocz, fma2(ocy, ocy, mul2(ocx, ocx)));
        float m_lo, m_hi;
        upk2(fma2(bh, bh, fma2(oc2, kk2, pk2(B.z, B.w))), m_lo, m_hi);
        mask |= (!(m_lo < 0.0f) ? 1u : 0u) << (2 * k);
        mask |= (!(m_hi < 0.0f) ? 1u : 0u) << (2 * k + 1);
    }
    if (all) mask = 0xffu;  // a non-finite ray: every sphere goes through the exact arithmetic
    mask &= (1u << count) - 1u;
    while (mask) {
        const int k = __ffs(mask) - 1;
        mask &= mask - 1u;
        brute_sphere_slow<COUNT>(sc, sph[first + k], first + k, o, d, best, ctr);
    }
}

// a triangle in the brute-force kernel: out of line like the spheres' slow path (K1's hot loop is the packed sphere
// filter; everything else is kept out of its instruction stream)
template <bool COUNT>
__device__ __noinline__ void brute_triangle_slow(const HitCtx hc, const float4* tri, int tidx, int pid, V3 o, V3 d, Hit& best, Ctr& ctr) {
    const V3 a = ld3(tri[4 * tidx + 0]), ab = ld3(tri[4 * tidx + 1]), ac = ld3(tri[4 * tidx + 2]);
    if (COUNT) ctr.v[CTR_TRI_TEST]++;
    float t;
    int stage;
    const bool hit = triangle_root_exact(o, d, a, ab, ac, &t, &stage);
    if (COUNT) {
        if (stage >= 1) ctr.v[CTR_TRI_S1]++;
        if (stage >= 2) ctr.v[CTR_TRI_S2]++;
        if (stage >= 3) ctr.v[CTR_TRI_S3]++;
        if (hit) ctr.v[CTR_TRI_HIT]++;
    }
    if (hit) consider(hc, o, d, t, pid, best);
}

template <bool COUNT>
__device__ __forceinline__ void trace_brute_impl(const DevScene& sc, const SceneView& sv, V3 o, V3 d, Hit& best, Ctr& ctr) {
    best.pid = -1;
    best.dist = 0.0f;
    const int ns = (int)sc.ns;
    // a non-finite ray makes the margins NaN, which fmaxf would drop: send such a ray through the slow path whole
    const bool weird = !(isfinite(o.x) && isfinite(o.y) && isfinite(o.z) && isfinite(d.x) && isfinite(d.y) && isfinite(d.z));
    // Packed pairs: two spheres per instruction — 3 FADD2 + 2 FMUL2 + 6 FFMA2 per PAIR (5.5 FMA-pipe issue slots per
    // sphere instead of 11), two LDS.128 per pair, one FMNMX3 per pair, one branch per 16 spheres.  The FMA pipe still
    // does 11 lane-operations per sphere, so the loop is bound by the pipe, not by issue (profiles/r1_notes.md).
    const f32x2 ox2 = pk2(o.x, o.x), oy2 = pk2(o.y, o.y), oz2 = pk2(o.z, o.z);
    const f32x2 dx2 = pk2(d.x, d.x), dy2 = pk2(d.y, d.y), dz2 = pk2(d.z, d.z);
    const f32x2 kk2 = pk2(-0.99998f, -0.99998f);
    auto pair_margin = [&](int j, float m) {
        const float4 A = sv.sph2[2 * j], B = sv.sph2[2 * j + 1];
        const f32x2 ocx = add2(ox2, pk2(A.x, A.y)), ocy = add2(oy2, pk2(A.z, A.w)), ocz = add2(oz2, pk2(B.x, B.y));
        const f32x2 bh = fma2(ocz, dz2, fma2(ocy, dy2, mul2(ocx, dx2)));
        const f32x2 oc2 = fma2(ocz, ocz, fma2(ocy, ocy, mul2(ocx, ocx)));
        const f32x2 mm = fma2(bh, bh, fma2(oc2, kk2, pk2(B.z, B.w)));
        float m_lo, m_hi;
        upk2(mm, m_lo, m_hi);
        return fmaxf(fmaxf(m, m_lo), m_hi);
    };
    const int ns8 = (ns + 7) & ~7;
    const float NEG = -3.0e38f;
    const HitCtx hc = hit_ctx(sc);
    int i = 0;
    for (; i + 16 <= ns8; i += 16) {
        float m0 = NEG, m1 = NEG;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            m0 = pair_margin((i >> 1) + k, m0);
            m1 = pair_margin((i >> 1) + 4 + k, m1);
        }
        if (COUNT) ctr.v[CTR_SPH_TEST] += min(16, ns - i);
        if (!(fmaxf(m0, m1) < 0.0f) || weird) {
            if (!(m0 < 0.0f) || weird) brute_group_slow<COUNT>(hc, sv.sph, sv.sph2, i, min(8, ns - i), o, d, weird, best, ctr);
            if ((!(m1 < 0.0f) || weird) && i + 8 < ns) brute_group_slow<COUNT>(hc, sv.sph, sv.sph2, i + 8, min(8, ns - i - 8), o, d, weird, best, ctr);
        }
    }
    if (i < ns8) {
        float m0 = NEG;
#pragma unroll
        for (int k = 0; k < 4; k++) m0 = pair_margin((i >> 1) + k, m0);
        if (COUNT) ctr.v[CTR_SPH_TEST] += ns - i;
        if (!(m0 < 0.0f) || weird) brute_group_slow<COUNT>(hc, sv.sph, sv.sph2, i, ns - i, o, d, weird, best, ctr);
    }
    const int nt = (int)sc.nt;
#pragma unroll 1
    for (int j = 0; j < nt; j++) brute_triangle_slow<COUNT>(hc, sv.tri, j, ns + j, o, d, best, ctr);
}

// ---------------------------------------------------------------------------------------------
// Camera::get_ray (camera.rs:109-129) — EXACT
// ---------------------------------------------------------------------------------------------
static __device__ __noinline__ float2 camera_uv_slow(float nu, float nv, float u_den, float v_den) {
    return make_float2(x_div_ool(nu, u_den), x_div_ool(nv, v_den));
}
__device__ __forceinline__ void primary_ray(const DevCamera& cam, uint32_t x, uint32_t y_cam, Rng& rng, V3* o_out,
                                            V3* d_out) {
    float a, b;
    unit_disc(rng, a, b);
    V3 offset = mk(x_mul(a, cam.lens_radius), x_mul(b, cam.lens_radius), 0.0f);
    const float nu = x_add((float)x, rng.gen_range_0_1());
    const float nv = x_add((float)y_cam, rng.gen_range_0_1());
    // u = nu / u_den, v = nv / v_den behind one guard
    float u = x_quot(nu, cam.u_den, x_rcp_refined(cam.u_den));
    float v = x_quot(nv, cam.v_den, x_rcp_refined(cam.v_den));
    if (!(x_div_num(nu) && x_div_num(nv) && x_div_mag(cam.u_den) && x_div_mag(cam.v_den))) {
        const float2 uv = camera_uv_slow(nu, nv, cam.u_den, cam.v_den);
        u = uv.x;
        v = uv.y;
    }
    V3 org = mk(cam.org[0], cam.org[1], cam.org[2]);
    V3 llc = mk(cam.llc[0], cam.llc[1], cam.llc[2]);
    V3 hor = mk(cam.hor[0], cam.hor[1], cam.hor[2]);
    V3 ver = mk(cam.ver[0], cam.ver[1], cam.ver[2]);
    // lower_left_corner + u*horizontal + v*vertical - origin
    V3 target = x_sub(x_add(x_add(llc, x_scale(hor, u)), x_scale(ver, v)), org);
    // Ray::new(origin, normalize_or_zero(target)).at(focus_distance); Ray::new renormalises by division
    V3 d1 = x_normalize_div_or_zero(target);
    V3 focal_point = x_add(org, x_scale(d1, cam.focus));
    V3 fo = x_add(org, offset);
    *o_out = fo;
    *d_out = x_normalize_div_or_zero(x_sub(focal_point, fo));
}

// `(c * 255.999) as u8`: truncation, saturation, NaN → 0 (color.rs:13-19)
static __device__ __noinline__ float x_sqrt_div_slow(float a, float b) { return x_sqrt_ool(x_div_ool(a, b)); }
__device__ __forceinline__ uint32_t quantise(float sum, float spp_f) {
    // sqrt(sum / spp): a zero mean (a black pixel) is its own square root, and the fast square root is NaN there
    const float m = x_quot(sum, spp_f, x_rcp_refined(spp_f));
    float c = (m == 0.0f) ? m : x_sqrt_fast(m);
    if (!(x_div_num(sum) && x_div_mag(spp_f) && (m == 0.0f || x_sqrt_domain(m)))) c = x_sqrt_div_slow(sum, spp_f);
    float s = x_mul(c, 255.999f);
    uint32_t q = __float2uint_rz(s);  // saturating, NaN → 0
    return q > 255u ? 255u : q;
}

// ---------------------------------------------------------------------------------------------
// K2 traversal, second form: centre/half-extent slab test (9 FFMA + 4 FMNMX per box instead of 6 FFMA +
// 10 FMNMX: the first form saturated the ALU pipe at 75 % with the FMA pipe at 23 %), FMA pre-filter in
// front of the exact triangle test.  Same while-while structure, same results.
// ---------------------------------------------------------------------------------------------
// One node visit's loads.  Shared-memory kernel: the code of an inner node is the shared-window address of its record
// (no address arithmetic in the loop); global-memory kernel: its byte offset from DevScene::lnode.
template <bool SMEM>
__device__ __forceinline__ void load_node(const SceneView& sv, int cur, float4& a, float4& b, float4& c, int2& ch) {
    if (SMEM) {
        RT_LDS_F4(a, cur, 0);
        RT_LDS_F4(b, cur, 16);
        RT_LDS_F4(c, cur, 32);
        RT_LDS_I2(ch, cur, 48);
    } else {
        const float4* nrec = reinterpret_cast<const float4*>(sv.nodes_g + cur);
        a = __ldg(nrec); b = __ldg(nrec + 1); c = __ldg(nrec + 2);
        ch = __ldg(reinterpret_cast<const int2*>(nrec + 3));
    }
}
constexpr int TR_DONE = (int)0x80000000;  // traversal finished (never a leaf code: first_pid < 2^26)
template <bool COUNT, bool SMEM>
__device__ __forceinline__ void trace_bvh_ch_impl(const DevScene& sc, const SceneView& sv, V3 o, V3 d, Hit& best, Ctr& ctr) {
    best.pid = -1;
    best.dist = 0.0f;
    // FILTER-domain ray constants; |1/d| is clamped so 0*inf never produces NaN slabs
    const float BIG = 1e30f;
    float ix = fminf(fmaxf(__frcp_rn(d.x), -BIG), BIG);
    float iy = fminf(fmaxf(__frcp_rn(d.y), -BIG), BIG);
    float iz = fminf(fmaxf(__frcp_rn(d.z), -BIG), BIG);
    if (!(fabsf(d.x) > 0.0f)) ix = BIG;
    if (!(fabsf(d.y) > 0.0f)) iy = BIG;
    if (!(fabsf(d.z) > 0.0f)) iz = BIG;
    const float ax = fabsf(ix), ay = fabsf(iy), az = fabsf(iz);
    const float qx = -o.x * ix, qy = -o.y * iy, qz = -o.z * iz;
    // rounding of the o-term: <= 3 * 2^-24 * |o*inv| per axis, in t (the c- and h-terms are padded on the host)
    const float slack = 4.8e-7f * fmaxf(fmaxf(fabsf(qx), fabsf(qy)), fabsf(qz)) + 1e-30f;
    const f32x2 i_xy = pk2(ix, iy), q_xy = pk2(qx, qy), a_xy = pk2(ax, ay), na_xy = pk2(-ax, -ay);
    const f32x2 i_zz = pk2(iz, iz), q_zz = pk2(qz, qz), a_zz = pk2(az, az), na_zz = pk2(-az, -az);
    const f32x2 slack2 = pk2(slack, slack);
    float cull = 1001.0f;  // a hit has t < T_MAX and length(p-o) ~ t
    const int ns = (int)sc.ns;
    const HitCtx hc = hit_ctx(sc);
    // The stack starts as: sentinel | tree root | leaf codes of the big primitives (split layout), first one on top.
    // The big primitives are therefore popped and tested before the tree is entered (their hits shorten everything that
    // follows) by the SAME leaf code as every other primitive: the exact arithmetic exists once in the kernel, which
    // matters because this kernel's working set of instructions sits at the edge of the instruction cache.
    int stack[MAX_STACK + 1 + MAX_BIG];
    stack[0] = TR_DONE;  // popping the sentinel ends the traversal, so a pop needs no emptiness test
    int* top = stack + 1;  // next free entry
    if (sc.ltree) *top++ = (SMEM && sc.lroot >= 0) ? sc.lroot + (int)sv.nodes_s : sc.lroot;
#pragma unroll 1
    for (int i = (int)sc.nbig - 1; i >= 0; i--) *top++ = __ldg(&sc.big_code[i]);
    int cur = *--top;
    for (;;) {
        while (cur >= 0) {
            float4 a, b, c;
            int2 ch;
            load_node<SMEM>(sv, cur, a, b, c, ch);
            // a = l.c.xy | l.h.xy, b = r.c.xy | r.h.xy, c = l.c.z r.c.z | l.h.z r.h.z: the eighteen FMAs of the two slab
            // tests are nine packed ones (x|y of each box, z of both boxes); results are the scalar FMAs' bit for bit
            const f32x2 lc2 = fma2(pk2(a.x, a.y), i_xy, q_xy), rc2 = fma2(pk2(b.x, b.y), i_xy, q_xy);
            const f32x2 ln2 = fma2(na_xy, pk2(a.z, a.w), lc2), lf2 = fma2(a_xy, pk2(a.z, a.w), lc2);
            const f32x2 rn2 = fma2(na_xy, pk2(b.z, b.w), rc2), rf2 = fma2(a_xy, pk2(b.z, b.w), rc2);
            const f32x2 cz2 = fma2(pk2(c.x, c.y), i_zz, q_zz);
            const f32x2 nz2 = fma2(na_zz, pk2(c.z, c.w), cz2), fz2 = fma2(a_zz, pk2(c.z, c.w), cz2);
            float lnx, lny, lfx, lfy, rnx, rny, rfx, rfy, lnz, rnz, lfz, rfz;
            upk2(ln2, lnx, lny); upk2(lf2, lfx, lfy); upk2(rn2, rnx, rny); upk2(rf2, rfx, rfy);
            upk2(nz2, lnz, rnz); upk2(fz2, lfz, rfz);
            const float tl = fmaxf(fmaxf(lnx, lny), fmaxf(lnz, 0.0f));
            const float fl = fminf(fminf(lfx, lfy), fminf(lfz, cull));
            const float tr = fmaxf(fmaxf(rnx, rny), fmaxf(rnz, 0.0f));
            const float fr = fminf(fminf(rfx, rfy), fminf(rfz, cull));
            float fls, frs;
            upk2(add2(pk2(fl, fr), slack2), fls, frs);
            const bool hl = tl <= fls;
            const bool hr = tr <= frs;
            if (COUNT) ctr.v[CTR_SLAB] += 2;
            // branch-light step: push and pop are short predicated blocks, the loop has one exit
            const bool swap = tr < tl;
            if (hl && hr) *top++ = swap ? ch.x : ch.y;
            int nxt = (hr && (!hl || swap)) ? ch.y : ch.x;  // the nearer (or the only) child
            if (!(hl || hr)) nxt = *--top;
            cur = nxt;
        }
        if (cur == TR_DONE) return;
        // leaf = one primitive: code = ~(pid << 5).  FILTER first, then the reference's arithmetic for the root, then ONE
        // consider() for both kinds.
        const int pid = (~cur) >> 5;
        float t = 0.0f;
        bool cand = false;
        if (pid < ns) {
            const float4 s = sv.sph[pid];
            // oc = origin - center is a single exact subtraction: shared by filter and exact path
            const V3 oc = mk(x_sub(o.x, s.x), x_sub(o.y, s.y), x_sub(o.z, s.z));
            // FILTER: the reference's discriminant is 4*(bh*bh - (|oc|^2 - r^2)), bh = d.oc.  Evaluated with FMAs, rejected
            // only when negative by more than a generous rounding bound (~300 ulp of |oc|^2), or when both roots lie
            // behind the origin (ray points away, origin outside): cannot be in [T_MIN, T_MAX)
            const float bh = fmaf(oc.z, d.z, fmaf(oc.y, d.y, oc.x * d.x));
            const float oc2 = fmaf(oc.z, oc.z, fmaf(oc.y, oc.y, oc.x * oc.x));
            const float cf = oc2 - s.w;
            const float disc = fmaf(bh, bh, -cf);
            if (COUNT) ctr.v[CTR_SPH_TEST]++;
            if (!(fmaf(oc2, 2e-5f, disc) < 0.0f) && !(bh > 0.0f && cf > 1e-4f * oc2)) {
                if (COUNT) ctr.v[CTR_SPH_EXACT]++;
                cand = sphere_root_exact(d, oc, s.w, &t);
                if (COUNT && cand) ctr.v[CTR_SPH_HIT]++;
            }
        } else {
            if (COUNT) ctr.v[CTR_TRI_TEST]++;
            if (triangle_filter(sv.tri, pid - ns, o, d, cull)) {
                const V3 a = ld3(sv.tri[4 * (pid - ns) + 0]), ab = ld3(sv.tri[4 * (pid - ns) + 1]), ac = ld3(sv.tri[4 * (pid - ns) + 2]);
                int stage;
                cand = triangle_root_exact(o, d, a, ab, ac, &t, &stage);
                if (COUNT) {
                    if (stage >= 1) ctr.v[CTR_TRI_S1]++;
                    if (stage >= 2) ctr.v[CTR_TRI_S2]++;
                    if (stage >= 3) ctr.v[CTR_TRI_S3]++;
                    if (cand) ctr.v[CTR_TRI_HIT]++;
                }
            }
        }
        if (cand) {
            consider(hc, o, d, t, pid, best);
            cull = fmaf(best.dist, 1.00001f, 1e-6f);
        }
        cur = *--top;
    }
}

// The queries as the kernels call them: the nearest hit, with Hit::unsure resolved out of the pid bit it travelled in.
template <bool COUNT>
__device__ __forceinline__ void trace_brute(const DevScene& sc, const SceneView& sv, V3 o, V3 d, Hit& best, Ctr& ctr) {
    trace_brute_impl<COUNT>(sc, sv, o, d, best, ctr);
    hit_finish(best);
}
template <bool COUNT, bool SMEM>
__device__ __forceinline__ void trace_bvh_ch(const DevScene& sc, const SceneView& sv, V3 o, V3 d, Hit& best, Ctr& ctr) {
    trace_bvh_ch_impl<COUNT, SMEM>(sc, sv, o, d, best, ctr);
    hit_finish(best);
}

}  // namespace rtb
