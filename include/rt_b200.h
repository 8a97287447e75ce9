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
/* Replaces the primitives of `scene` with a world of the same shape: n_spheres and n_triangles as created, the
 * world_index given at creation still applies.  Geometry, materials and emission may all change.  Renders queued on
 * ctx before the call see the old world, renders after it the new one, byte-identical to a scene created from it.
 * The traversal tree keeps its topology and is refitted to the new boxes on the device (a tree that motion has made
 * loose costs time, never correctness; re-create the scene to rebuild it); when no primitive's box changes (materials
 * only) only the primitive data is uploaded.  The reference-topology tree is rebuilt as by rt_scene_create, beside the
 * upload from 256 primitives on; a failure of that build is reported by rt_scene_wait_ready, rt_scene_info or a render
 * that needs it.  rt_scene_info then reports the new world; rt_scene_device_bytes does not change.
 * Every successful update gives the scene a new serial: an rt_accum with samples of the old world refuses it
 * (RT_ERR_INVALID_ARG from rt_render_samples) until rt_accum_reset.
 * RT_ERR_INVALID_ARG: NULL ctx or scene, a scene of another context, counts other than the creation counts, a NULL array
 * with a nonzero count.  RT_ERR_BVH: non-finite geometry or bounds.  On either the scene is untouched and still renders
 * the old world.  RT_ERR_CUDA leaves the scene undefined: destroy it. */
int rt_scene_update(rt_ctx* ctx, rt_scene* scene, const rt_sphere* spheres, uint32_t n_spheres,
                    const rt_triangle* triangles, uint32_t n_triangles);
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
/* Several divisions of one job in one launch: band division_nos[k] of *params (params->division_no is ignored) is
 * written to out_rgb + k * rows * width * 3, rows = height / divisions, byte-identical to rt_render_division with
 * division_no = division_nos[k].  out_len = n * rows * width * 3.  A list that is one ascending run of bands renders as
 * that row range (the path of rt_render_division and rt_render_frame); any other list renders its bands stacked in list
 * order in one banded launch.  RT_ERR_INVALID_ARG, before anything is launched: a NULL pointer, n == 0, a division
 * number >= divisions or listed twice, a wrong out_len, and every check of rt_render_division.  Returns after all n
 * bands are in out_rgb.  stats (nullable): as rt_render_division for all n bands (primary = n * rows * width * spp); the
 * counters of collect_counters are not filled (0), as for rt_render_samples. */
int rt_render_divisions(rt_ctx* ctx, const rt_scene* scene, const rt_params* params, const uint32_t* division_nos,
                        uint32_t n, uint8_t* out_rgb, size_t out_len, rt_stats* stats);
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

/* ---- JPEG ------------------------------------------------------------------------------------------ */
/* The controller's output format (ray-tracer-controller/src/main.rs:95-142 encodes the stitched frame as JPEG(90)),
 * encoded on the device.  The bytes are identical to libjpeg's defaults at the same quality (what PIL's
 * save(format="JPEG", quality=q) writes): JFIF 1.01, 4:2:0, the standard Huffman tables, no restart markers.
 * RT_ERR_INVALID_ARG, before anything is launched: a NULL pointer, a width or height of 0 or above 65535, a quality
 * outside 1..100, out_cap < rt_jpeg_bound(width, height).  *out_len: the bytes written to out. */

/* Bytes enough for any JPEG the two calls below write for width x height, at any quality. */
size_t rt_jpeg_bound(uint32_t width, uint32_t height);
/* Baseline JPEG of an RGB8 frame in host memory (height*width*3 bytes, row-major, row 0 on top), byte-identical to
 * libjpeg's defaults at this quality (JFIF, 4:2:0, standard Huffman tables, no restart markers).  ms_out (nullable):
 * device time of the encode. */
int rt_jpeg_encode(rt_ctx* ctx, const uint8_t* rgb, uint32_t width, uint32_t height, uint32_t quality,
                   uint8_t* out, size_t out_cap, size_t* out_len, float* ms_out);
/* Renders the whole frame as rt_render_frame (n == 1) or rt_render_frame_multi (n > 1), then encodes it on ctxs[0]
 * from device memory: the RGB frame never reaches the host.  The bytes equal rt_jpeg_encode of that call's frame.
 * Refused as rt_jpeg_encode and as the render entry it wraps.  stats (nullable): the render's, with total_ms including
 * the encode and the download. */
int rt_render_frame_jpeg(rt_ctx* const* ctxs, const rt_scene* const* scenes, uint32_t n, const rt_params* params,
                         uint32_t quality, uint8_t* out, size_t out_cap, size_t* out_len, rt_stats* stats);

/* ---- wire format: the slave's request and result bodies (ray-tracer-slave/src/lib.rs:10-30) --------- */
/* Upper bound on the Objects in `len` bytes of world JSON (len / the shortest accepted Object, derived in rt_wire.cu). */
size_t rt_world_json_max_objects(size_t len);
/* Parses the JSON array of Object that starts at text[0] (leading JSON whitespace allowed): the "world" value of a
 * RenderInfo.  Writes the spheres and the triangles in world order and the world position of each (spheres first, then
 * triangles), exactly the arrays rt_b200/wire.py's parse_render_info puts in its World, and *consumed = the offset just
 * past the array's ']'.  spheres, triangles and world_index must each hold cap >= rt_world_json_max_objects(len) entries.
 * The device grammar is a strict subset of JSON, serde's canonical layout: every Object {"Sphere":{...}} or
 * {"Triangle":{...}} with its fields in declaration order, JSON whitespace anywhere, JSON numbers of at most 19 significant
 * digits, node_index a non-negative integer (its value is ignored).  Numbers convert as Python's json + float32 do: an
 * integer exactly to f64, then to f32; any other token correctly rounded to f64, then to f32 (both to nearest).
 * RT_ERR_UNSUPPORTED: the text is outside the device grammar (a backslash, an unknown, missing, repeated or reordered key,
 * NaN / Infinity, a number of more than 19 digits or with an exponent outside the conversion table, malformed JSON ...);
 * nothing is promised about the outputs, and the caller parses the text on the host, which decides whether it is valid.
 * RT_ERR_INVALID_ARG: a NULL pointer, cap below the bound. */
int rt_world_parse_json(rt_ctx* ctx, const char* text, size_t len, rt_sphere* spheres, rt_triangle* triangles,
                        uint32_t* world_index, size_t cap, uint32_t* n_spheres, uint32_t* n_triangles, size_t* consumed);
/* Bytes enough for the ImageSlice JSON of one band of rows x width. */
size_t rt_slice_json_bound(uint32_t rows, uint32_t width);
/* rt_render_divisions, then band k written on the device as the body the slave POSTs to /result,
 * {"division_no":D,"image":[v,v,...],"id":"ID"} with no spaces: the bytes of serde_json's json!(ImageSlice) and of
 * wire.ImageSlice(D, band, ID).to_json().  The bodies are packed back to back in out, body k (band division_nos[k]) first
 * after body k - 1; out_lens[k] is its length.  id: the 36-character hyphenated lowercase uuid.  The RGB bands never reach
 * the host.  Refused as rt_render_divisions (out_rgb / out_len aside), and with RT_ERR_INVALID_ARG, before anything is
 * launched: a NULL id, out or out_lens, an id not of that form, out_cap < n * rt_slice_json_bound(rows, width).  stats
 * (nullable): as rt_render_divisions, with total_ms including the bodies and their download. */
int rt_render_divisions_json(rt_ctx* ctx, const rt_scene* scene, const rt_params* params, const uint32_t* division_nos,
                             uint32_t n, const char* id, uint8_t* out, size_t out_cap, size_t* out_lens, rt_stats* stats);

/* ---- OBJ ingest: the controller's /upload body (ray-tracer-controller/src/obj.rs:10-53) ------------------------- */
/* Bytes-derived upper bound on the triangles of an OBJ section of obj_size bytes (obj_size / 6, derived in rt_obj.cu). */
size_t rt_obj_max_triangles(size_t obj_size);
/* obj::build_world (ray-tracer-controller/src/obj.rs:10-53) on the device: body[0, obj_size) is the OBJ, body[obj_size,
 * len) the MTL.  Writes the triangles in world order, exactly the TRIANGLE_DTYPE array rt_b200/obj.py's build_world
 * returns (a, b, c from the corner triples of each model, albedo = Kd, roughness = f32(Ns) / 1000 in f32, emission 0),
 * and *n_triangles.  triangles must hold cap >= rt_obj_max_triangles(obj_size) entries.  A body without faces gives
 * RT_OK and 0 triangles.
 * The device grammar is ASCII, lines broken at \n \r \v \f \x1c \x1d \x1e, '#' cutting the rest of a line, tokens
 * separated by space, \t and \x1f; keys v, f, o, g, usemtl in the OBJ and newmtl, Kd, Ns in the MTL (any other line is
 * ignored); numbers [+-]? (digits [. digits] | . digits) ([eE] [+-]? digits)? of at most 19 significant digits, converted
 * as float(np.float32(token)) (correctly rounded to f64, then to f32, both to nearest); face indices [+-]? digits of at
 * most 10 digits, then the corner's end or a '/'.
 * RT_ERR_UNSUPPORTED: the body is outside the device grammar (a byte above 0x7F, inf / nan, a number with '_' or of
 * more than 19 digits, a non-finite result, an exponent outside the conversion table, a longer face index, a material
 * named __order__) or is one the host rejects (a v of fewer than 3 coordinates, an f of fewer than 3 corners, a bad
 * number or an index out of range, a model with faces and no material, a bad Kd or Ns after a newmtl), or positions
 * would not fit 32 bits.  Nothing is promised about the outputs, and the caller builds the world on the host, which
 * decides whether the body is valid and what its error is.
 * RT_ERR_INVALID_ARG, before anything is launched: a NULL pointer, obj_size > len, cap below the bound. */
int rt_obj_build_world(rt_ctx* ctx, const uint8_t* body, size_t len, size_t obj_size, rt_triangle* triangles, size_t cap,
                       uint32_t* n_triangles);

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
 * unchanged.  RT_ERR_INVALID_ARG for an accum bound to several ranks by rt_render_samples_multi until it is reset.
 * stats (nullable): rays, primary (pixels * n_samples), kernel_ms, total_ms, intersector_used,
 * kernel_launches, the launch shape and redo_pixels; the counters of collect_counters are not filled (0). */
int rt_render_samples(rt_ctx* ctx, const rt_scene* scene, rt_accum* acc, uint32_t n_samples, uint8_t* out_rgb,
                      size_t out_len, rt_stats* stats);
/* Linear radiance of the band: rows*width*3 float32 (out_len in bytes), sum / samples per channel (the exact-domain
 * division quantise() does: sqrt, * 255.999, truncate, saturate, NaN -> 0 give the RGB8 band).  RT_ERR_INVALID_ARG before
 * the first chunk, and for an accum bound to several ranks by rt_render_samples_multi (each holds only its rank's tiles;
 * there is no multi-GPU linear readback). */
int rt_accum_read_linear(rt_ctx* ctx, const rt_accum* acc, float* out, size_t out_len);
/* One progressive frame on n contexts: accs[i] (rt_accum_create on ctxs[i], whole frame: divisions 1) holds the chains of
 * rank i's tiles (the interleave of rt_render_frame_multi).  Advances every pixel by n_samples and, if out_rgb != NULL,
 * streams the frame (height*width*3 bytes) to the host: byte-identical to rt_render_frame at spp = done + n_samples.
 * Context i renders its tiles of scenes[i] (the same world, created on ctxs[i]) into a frame in ctxs[0]'s memory, as
 * rt_render_frame_multi does; each accum keeps a whole-frame state buffer, of which only its rank's records are used.
 * An accum is bound to the tile share of its first chunk after create / reset: rank 0 of 1 for rt_render_samples, rank
 * i of n here; until rt_accum_reset any other share is refused (n = 1 is the share of rt_render_samples).
 * RT_ERR_INVALID_ARG, before anything is launched: a NULL handle, accs[i] not of ctxs[i], an accum that is not whole-frame,
 * bound to another rank or n, bound params (size, seed, camera, max_bounces, flags, intersector) or sample counts that
 * differ between the accums, a scene other than the one of the chunks since the last reset, n_samples == 0, done +
 * n_samples above 2^32 - 1, out_len != height*width*3 with out_rgb != NULL.  On any error no accum moves.  stats
 * (nullable): as rt_render_samples, counters summed over the contexts, kernel_ms the slowest context's. */
int rt_render_samples_multi(rt_ctx* const* ctxs, const rt_scene* const* scenes, rt_accum* const* accs, uint32_t n,
                            uint32_t n_samples, uint8_t* out_rgb, size_t out_len, rt_stats* stats);

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
