/* rt_b200.h — C ABI of the B200-native render path for ray-tracer-s8's slave.
 *
 * The reference (actuday6418/ray-tracer-s8) has no plugin / FFI interface: its hot path is the body
 * of `worker()` in ray-tracer-slave/src/main.rs:32-106.  This header puts a C ABI exactly there:
 *
 *   reference (Rust, CPU)                                   replacement (this ABI, sm_100a CUDA)
 *   -----------------------------------------------------   -----------------------------------------
 *   req.world: Vec<Object>  (main.rs:37, lib.rs:11-15)  →   rt_scene_create()   once per job
 *   BVH::build(&mut req.world)          (main.rs:60)     →   rt_scene_create()   (host SAH build + upload)
 *   img_buff.par_chunks_exact_mut(...)  (main.rs:53-83)  →   rt_render_division()
 *   ImageSlice.image: Vec<u8>           (main.rs:85-90)  →   out_rgb (caller-owned, (h/div)*w*3 bytes)
 *
 * Plain pointers and sizes only; no C++/torch types.  Every call returns RT_OK (0) or a negative
 * rt_status and never throws or unwinds across the boundary: every entry point catches host exceptions
 * (RT_ERR_NOMEM / RT_ERR_INTERNAL) (the reference `.unwrap()`s and kills its worker thread instead,
 * main.rs:98,152).  There is no CPU fallback: without a CUDA device
 * rt_init fails with RT_ERR_NO_DEVICE.
 *
 * Threading: one rt_ctx = one GPU + one stream, single owner, calls serialised by the caller — the
 * same contract as the reference's single worker thread (main.rs:34-35,160).  Distinct contexts
 * are independent.
 */
#ifndef RT_B200_H
#define RT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_B200_ABI_VERSION 2

typedef enum rt_status {
    RT_OK = 0,
    RT_ERR_INVALID_ARG = -1,   /* null pointer, zero size, out_len mismatch, height % divisions != 0 ... */
    RT_ERR_EMPTY_SCENE = -2,   /* n_spheres + n_triangles == 0 (reference: BVHNode::build never returns) */
    RT_ERR_NO_DEVICE = -3,     /* no usable CUDA device; there is no CPU fallback */
    RT_ERR_CUDA = -4,          /* CUDA runtime error, text in rt_last_error */
    RT_ERR_BVH = -5,           /* scene the reference's BVH build would panic on (NaN bounds, depth) */
    RT_ERR_UNSUPPORTED = -6,   /* parameter outside this build's limits (e.g. max_bounces > 62) */
    RT_ERR_NOMEM = -7,         /* host allocation failed */
    RT_ERR_INTERNAL = -8,      /* an unexpected host exception was caught at the boundary */
    RT_ERR_TIMEOUT = -9        /* a frame slab never completed (a rank of a multi-GPU frame died) */
} rt_status;

typedef struct rt_ctx rt_ctx;     /* device, stream, staging buffers */
typedef struct rt_scene rt_scene; /* device-resident scene: primitive SoA + BVH */

/* Sphere {radius, center, p_albedo_at, p_roughness_at, p_emission_at}
 * (ray-tracer-slave/src/shapes/sphere.rs:13-20; node_index is rebuilt by the library). */
typedef struct rt_sphere {
    float center[3];
    float radius;
    float albedo[3];
    float roughness; /* reference convention: 1 = mirror, 0 = Lambertian (main.rs:119-122) */
    float emission;  /* > 0 terminates the path with emission*albedo (main.rs:116-117) */
} rt_sphere;

/* Triangle {a, b, c, p_albedo_at, p_roughness_at, p_emission_at}
 * (ray-tracer-slave/src/shapes/mesh.rs:15-23). Two-sided, geometric normal (a-b)x(a-c). */
typedef struct rt_triangle {
    float a[3], b[3], c[3];
    float albedo[3];
    float roughness;
    float emission;
} rt_triangle;

typedef enum rt_intersector {
    RT_INTERSECT_AUTO = 0,  /* library picks by primitive count */
    RT_INTERSECT_BRUTE = 1, /* K1: every primitive, scene staged in shared memory */
    RT_INTERSECT_BVH = 2    /* K2: BVH traversal (reference SAH topology, ordered, culled) */
} rt_intersector;

/* RenderMeta + division_no (ray-tracer-slave/src/lib.rs:11-15,25-30) plus the values the reference
 * hard-codes in worker() (main.rs:39-51).  A zero field means "the reference's literal". */
typedef struct rt_params {
    uint32_t width;        /* render_meta.width  */
    uint32_t height;       /* render_meta.height */
    uint32_t divisions;    /* render_meta.divisions; 0 → 1.  height % divisions must be 0 */
    uint32_t division_no;  /* band index, 0 = top of the image */
    uint32_t spp;          /* 0 → 100  (main.rs:51) */
    uint32_t max_bounces;  /* 0 → 10   (main.rs:39); a sample makes at most max_bounces+1 queries */
    uint64_t seed;         /* pixel (x, y_global) draws from SmallRng::seed_from_u64(seed + y_global*width + x) */
    float cam_origin[3];   /* (0,0,0)  (main.rs:43) */
    float aperture;        /* 0 → 0.1  (main.rs:45) */
    float focus_distance;  /* 0 → 1    (main.rs:46) */
    float field_of_view;   /* 0 → PI/2 (main.rs:47) */
    float focal_length;    /* 0 → 1    (main.rs:48) */
    uint32_t intersector;  /* rt_intersector */
    uint32_t collect_counters; /* != 0: run the instrumented kernel variant and fill every rt_stats field */
    uint32_t flags;        /* rt_param_flags: fields whose zero is a value, not "the reference's literal" */
} rt_params;

typedef enum rt_param_flags {
    RT_PARAM_MAX_BOUNCES_EXPLICIT = 1, /* max_bounces is taken as given: 0 = camera rays only */
    RT_PARAM_APERTURE_EXPLICIT = 2     /* aperture is taken as given: 0 = pinhole camera */
} rt_param_flags;

/* Work counters (for the roofline: SURVEY.md §8d / Appendix C) and timings of the last call. */
typedef struct rt_stats {
    uint64_t rays;          /* nearest-hit queries = ray_color calls with depth > 0 (always filled) */
    uint64_t primary;       /* camera rays = pixels * spp (always filled) */
    /* the rest (to total_lane_iters) is filled only when params.collect_counters != 0 (instrumented kernel variant) */
    uint64_t slab_tests;    /* child-box tests during BVH traversal */
    uint64_t sphere_tests;  /* sphere candidate tests (discriminant filter) */
    uint64_t sphere_exact;  /* ... that went through the exact reference arithmetic */
    uint64_t sphere_hits;   /* ... that produced an in-range root */
    uint64_t tri_tests;     /* triangle tests */
    uint64_t tri_stage[3];  /* tests that passed the determinant / u / v checks (mesh.rs:127,140,150) */
    uint64_t tri_hits;      /* in-range triangle hits */
    uint64_t shades_sphere; /* non-terminal hits (scatter) on spheres */
    uint64_t shades_tri;    /* ... on triangles */
    uint64_t emissive;      /* paths ended on an emitter */
    uint64_t sky;           /* paths ended on the sky */
    uint64_t active_lane_iters; /* sum over nearest-hit queries of participating lanes */
    uint64_t total_lane_iters;  /* 32 * warp-level query trips: ratio = SIMT efficiency at query level */
    float kernel_ms;        /* device time of the render kernel, CUDA events on the ctx stream */
    float total_ms;         /* host wall time of the call, copies included */
    uint32_t intersector_used; /* rt_intersector actually run */
    uint32_t kernel_launches;  /* kernels launched by the call */
    uint32_t grid_ctas, cta_threads, ctas_per_sm, scene_in_smem; /* launch shape of the render kernel */
    uint32_t dyn_smem_bytes;
    uint32_t redo_pixels;   /* pixels rendered a second time because a query needed the tie-break tables of the scene
                               (rt_scene_create builds them beside the upload) before they had landed */
} rt_stats;

/* ---- lifecycle -------------------------------------------------------------------------------- */
int rt_abi_version(void);
/* sizeof(rt_sphere), sizeof(rt_triangle), sizeof(rt_params), sizeof(rt_stats) as compiled: lets a
 * binding check its struct layouts at load time. */
void rt_struct_sizes(size_t out[4]);
/* Create a context on CUDA device `device` (one stream, one event pair). */
int rt_init(int device, rt_ctx** out);
void rt_shutdown(rt_ctx* ctx);
/* Last error text of this context (or of the failed rt_init when ctx is NULL). Never NULL. */
const char* rt_last_error(const rt_ctx* ctx);

/* ---- scene: replaces `req.world` ownership + BVH::build (main.rs:60-61) ------------------------- */
/* world_index (nullable): position of each primitive in the reference's Vec<Object>, spheres first
 * then triangles, a permutation of 0..n-1.  NULL = spheres in order, then triangles.  The world order
 * decides exact-distance ties the way the reference's BVH leaf order does (shapes/mod.rs:177-182).
 * RT_ERR_EMPTY_SCENE for an empty world (the reference's build never terminates on it), RT_ERR_UNSUPPORTED above
 * 2^25 primitives (tree node offsets are 31 bits of 64-byte records) or when the traversal tree is deeper than the
 * traversal stack (64). */
int rt_scene_create(rt_ctx* ctx, const rt_sphere* spheres, uint32_t n_spheres, const rt_triangle* triangles,
                    uint32_t n_triangles, const uint32_t* world_index, rt_scene** out);
void rt_scene_destroy(rt_ctx* ctx, rt_scene* scene);
/* rt_scene_create returns as soon as the geometry and the tree the kernels traverse are on the device.  The reference-
 * topology tree (bvh_impl.rs:229-364), which only decides exact-distance ties and the fate of rays with a zero direction
 * component, is finished by a builder thread; renders started before it lands are correct all the same (the few pixels
 * that needed it are rendered again).  This call blocks until it has landed; RT_ERR_BVH if the reference's build would
 * have panicked on this world. */
int rt_scene_wait_ready(rt_ctx* ctx, const rt_scene* scene);
/* BVH facts for tests / tooling: node count (2n-1 like bvh_impl.rs), depth, and the DFS leaf rank of every
 * primitive in world order (rank_out nullable, n entries).  Waits for the builder thread. */
int rt_scene_info(const rt_scene* scene, uint32_t* n_prims, uint32_t* n_nodes, uint32_t* depth, uint32_t* rank_out);
/* Bytes rt_scene_create copied host→device for this scene (primitive SoA + BVH nodes + materials). */
size_t rt_scene_device_bytes(const rt_scene* scene);

/* Host-only BVH build (no GPU needed): the DFS leaf rank of every primitive in world order, as
 * rt_scene_create computes it. For tests and tooling. Outputs nullable. */
int rt_bvh_build_host(const rt_sphere* spheres, uint32_t n_spheres, const rt_triangle* triangles, uint32_t n_triangles,
                      const uint32_t* world_index, uint32_t* rank_out, uint32_t* n_nodes, uint32_t* depth);

/* ---- render: replaces main.rs:53-83 -------------------------------------------------------------- */
/* Renders band `division_no` into host memory: (height/divisions) rows * width * 3 bytes, RGB, row 0 =
 * top of the band.  Returns after out_rgb is complete.  stats is nullable. */
int rt_render_division(rt_ctx* ctx, const rt_scene* scene, const rt_params* params, uint8_t* out_rgb,
                       size_t out_len, rt_stats* stats);
/* All divisions in one launch: height*width*3 bytes into host memory (what the controller stitches at
 * ray-tracer-controller/src/main.rs:109-119). params->division_no is ignored. */
int rt_render_frame(rt_ctx* ctx, const rt_scene* scene, const rt_params* params, uint8_t* out_rgb,
                    size_t out_len, rt_stats* stats);

/* One frame on n GPUs from ONE process (the controller's fan-out, ray-tracer-controller/src/main.rs:47-75,109-119,
 * without HTTP): ctxs[i] renders the tiles t with t % n == (i + t / n) % n — the interleave of rt_render_tiles_device —
 * of the scene scenes[i] (the same world, created on ctxs[i]) straight into a frame in ctxs[0]'s memory over peer
 * access (NVLink stores), and finished slabs of the frame stream to out_rgb (host, height*width*3 bytes) while the rest
 * still renders.  Contexts may share a device.  stats (nullable): counters summed over the contexts, kernel_ms the
 * slowest context's.  params->division_no is ignored. */
int rt_render_frame_multi(rt_ctx* const* ctxs, const rt_scene* const* scenes, uint32_t n, const rt_params* params,
                          uint8_t* out_rgb, size_t out_len, rt_stats* stats);

/* Device-side entry for the multi-GPU tile scheduler: renders the 8x4-pixel tiles of the whole frame that belong to
 * rank tile_rank of tile_ranks (tile t, row-major over the tile grid, belongs to rank (t % ranks - t / ranks) mod ranks:
 * a rotating interleave) into a full-frame DEVICE buffer `frame_dev` (height*width*3 bytes;
 * may be a peer-mapped pointer into another GPU's memory, in which case the stores travel over NVLink).
 * Asynchronous on the ctx stream unless `sync` != 0. stats (nullable) is filled only when sync != 0. */
int rt_render_tiles_device(rt_ctx* ctx, const rt_scene* scene, const rt_params* params, uint32_t tile_rank,
                           uint32_t tile_ranks, void* frame_dev, int sync, rt_stats* stats);
/* The frame owner's form of the call above: renders this context's tiles into frame_dev (allocated by this context with
 * rt_frame_alloc) and, while they render, copies every slab of frame number `seq` to out_rgb as soon as ALL ranks have
 * finished it (see rt_frame_collect).  Returns with the complete frame in out_rgb (height*width*3 bytes); out_rgb may be
 * NULL: the call then only waits until the frame is complete on the device. */
int rt_render_tiles_collect(rt_ctx* ctx, const rt_scene* scene, const rt_params* params, uint32_t tile_rank,
                            uint32_t tile_ranks, void* frame_dev, uint64_t seq, uint8_t* out_rgb, size_t out_len,
                            rt_stats* stats);

/* ---- progressive rendering: resumable per-pixel sample chains, rendered in chunks ------------------ */
/* A pixel's chain is sequential but resumable: between two samples its whole state is the xoshiro256++ state and three
 * running sums, and the samples of a render at spp = k are the first k samples of a render at any larger spp.  So a band
 * rendered in chunks of samples is byte-identical at every step to rt_render_division at the cumulative count: a cheap
 * preview that improves (1 sample, then 2, 4, 8 ...), or more samples added to a finished frame without paying again for
 * the samples it has. */
typedef struct rt_accum rt_accum;
/* Sample state of the rows rt_render_division would render for *params (divisions / division_no honoured; 1 = whole
 * frame), every pixel at sample 0.  Binds width, height, band, seed, camera, max_bounces, flags, intersector;
 * params->spp and collect_counters are ignored.  Device memory: 2 x 48 bytes per pixel. */
int rt_accum_create(rt_ctx* ctx, const rt_params* params, rt_accum** out);
void rt_accum_destroy(rt_ctx* ctx, rt_accum* acc);
/* Back to sample 0, optionally re-bound to new params (same width, height and band; NULL = keep): a camera move.
 * RT_ERR_INVALID_ARG for another size or band. */
int rt_accum_reset(rt_ctx* ctx, rt_accum* acc, const rt_params* params);
int rt_accum_samples(const rt_accum* acc, uint32_t* samples_out);
/* Advances every pixel by n_samples (samples [done, done + n) of its chain) and, if out_rgb != NULL, writes the band as
 * it now stands: byte-identical to rt_render_division with spp = done + n.  Every chunk since the last create / reset
 * must render the same scene (another one, a re-created one included, is RT_ERR_INVALID_ARG; RT_INTERSECT_AUTO is
 * resolved against the scene of each call).  RT_ERR_INVALID_ARG also for n_samples == 0, done + n_samples above
 * 2^32 - 1, out_len != rows*width*3 with out_rgb != NULL, and an accum of another context.  On any error the state is
 * unchanged.  stats (nullable): rays, primary (pixels * n_samples), kernel_ms, total_ms, intersector_used,
 * kernel_launches, the launch shape and redo_pixels; the counters of collect_counters are not filled (0). */
int rt_render_samples(rt_ctx* ctx, const rt_scene* scene, rt_accum* acc, uint32_t n_samples, uint8_t* out_rgb,
                      size_t out_len, rt_stats* stats);
/* Linear radiance of the band: rows*width*3 float32 (out_len in bytes), sum / samples per channel (the exact-domain
 * division quantise() does: sqrt, * 255.999, truncate, saturate, NaN -> 0 give the RGB8 band).  RT_ERR_INVALID_ARG before
 * the first chunk. */
int rt_accum_read_linear(rt_ctx* ctx, const rt_accum* acc, float* out, size_t out_len);

int rt_sync(rt_ctx* ctx);
/* The ctx stream as a cudaStream_t, for callers that order their own work (NCCL, copies) after a render. */
void* rt_stream(rt_ctx* ctx);

/* ---- pinned host memory for callers that want full-rate D2H ------------------------------------- */
int rt_host_alloc(rt_ctx* ctx, size_t bytes, void** out);
void rt_host_free(rt_ctx* ctx, void* p);

/* ---- cross-process frame sharing on one NVLink box (fused render + gather) ----------------------- */
/* Rank 0 allocates the frame and exports a 64-byte handle; other ranks open it and pass the mapped
 * pointer as frame_dev to rt_render_tiles_device. */
int rt_frame_alloc(rt_ctx* ctx, size_t bytes, void** dev_out, uint8_t handle_out[64]);
int rt_frame_open(rt_ctx* ctx, const uint8_t handle[64], void** dev_out);
int rt_frame_close(rt_ctx* ctx, void* dev);
int rt_frame_free(rt_ctx* ctx, void* dev);
int rt_frame_download(rt_ctx* ctx, const void* frame_dev, uint8_t* out_rgb, size_t bytes);
/* Every frame from rt_frame_alloc carries a control block: the render kernels of all ranks add the pixels they finish
 * to per-slab counters in it (system-scope releases, also over NVLink).  On the frame's owner: wait until frame number
 * `seq` (1 = the first frame rendered into this buffer; counters are cumulative, the frame size must not change) is
 * complete — no barrier between the ranks is needed — and, if out_rgb is not NULL, copy each slab to the host as soon
 * as it is complete, while other slabs still render.  RT_ERR_TIMEOUT if a slab does not complete within 20 s. */
int rt_frame_collect(rt_ctx* ctx, const void* frame_dev, const rt_params* params, uint64_t seq, uint8_t* out_rgb,
                     size_t out_len);
/* Flow control for ranks that do not own the frame: everything queued on this context's stream after this call (the
 * next rt_render_tiles_device into frame_dev) waits, on the device, until the owner has finished collecting frame
 * number `seq` of the buffer (rt_frame_collect / rt_render_tiles_collect mark it).  seq == 0 is a no-op.  A rank that
 * renders frame k of a buffer calls this with k - 1; with two buffers used alternately ranks run a frame ahead. */
int rt_frame_wait_consumed(rt_ctx* ctx, const void* frame_dev, size_t frame_bytes, uint64_t seq);

/* ---- measurement helpers --------------------------------------------------------------------------- */
/* FFMA-chain micro-benchmark: achieved FP32 TFLOP/s (2 flops per FFMA) on this device, for the
 * roofline denominator (MEASURED_PEAKS.json has no CUDA-core figure). */
int rt_measure_fp32_peak(rt_ctx* ctx, double* tflops_out, float* ms_out);
/* Writes `bytes` (choose more than the 126 MB L2) of a scratch buffer on the context's stream, asynchronously in front
 * of whatever is queued next: benchmarks flush L2 between timed frames with it without a host synchronisation.
 * ms_out (nullable): when given, the call synchronises and reports the flush's device time. */
int rt_l2_flush(rt_ctx* ctx, size_t bytes, float* ms_out);
/* Device properties: sm_count, clock_khz (max SM clock), smem_optin bytes. Nullable outputs. */
int rt_device_info(rt_ctx* ctx, int* sm_count, int* clock_khz, int* smem_optin, char name_out[64]);

#ifdef __cplusplus
}
#endif
#endif /* RT_B200_H */
