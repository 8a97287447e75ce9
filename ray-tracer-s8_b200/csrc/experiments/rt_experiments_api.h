/* rt_experiments_api.h — entry points that exist only in lib/librt_b200_exp.so (built with -DRT_B200_EXPERIMENTS). */
#ifndef RT_B200_EXPERIMENTS_API_H
#define RT_B200_EXPERIMENTS_API_H
#include "../../../include/rt_b200.h"
#ifdef __cplusplus
extern "C" {
#endif
/* Trace-only benchmark (development aid, csrc/experiments/rt_trace_bench.cuh; with_big 2 / 3 = 0 / 1 on rays sorted by
 * octant + cell): renders one frame while recording up to max_rays of its nearest-hit queries, then times the query alone
 * over the recorded rays as (a) the product kernel's while-while traversal and (b) a ballot-scheduled state machine with
 * dynamic fetch, and counts rays whose answers differ.  with_big = 0 leaves the split layout's big primitives out of
 * both.  The scene must fit shared memory. */
int rt_debug_trace_bench(rt_ctx* ctx, const rt_scene* scene, const rt_params* params, uint64_t max_rays, int with_big,
                         uint64_t* n_rays_out, float* ms_while_while, float* ms_state_machine, uint64_t* mismatches_out);
/* Test aid (csrc/experiments/rt_exact_fastpath.cuh): the guarded fast divisions, square roots, normalisations and sphere
 * roots of rt_device.cuh against the plain __fdiv_rn / __fsqrt_rn forms, on the device.  Every float32 bit pattern is a
 * numerator against each of the n_div divisors, and a square-root argument; vecs holds n_vec 3-vectors, sph n_sph
 * records d.xyz, oc.xyz, r*r.  out[0] / out[1] = bitwise mismatches (scalars / vectors and sphere roots), out[2] = the
 * number of (numerator, divisor) pairs inside the guarded domain that were compared. */
int rt_debug_exact_fastpath(const float* divisors, uint32_t n_div, const float* vecs, uint32_t n_vec, const float* sph,
                            uint32_t n_sph, uint64_t* out);
#ifdef __cplusplus
}
#endif
#endif
