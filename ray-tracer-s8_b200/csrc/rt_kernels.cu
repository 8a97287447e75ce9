// rt_kernels.cu — the render megakernel (sm_100a) and its launcher.
//
// One persistent launch renders a set of 8x4-pixel tiles.  Warps pull tiles from a global ticket counter; a lane
// owns one pixel at a time and runs that pixel's whole sample/bounce chain from its own xoshiro256++ stream,
// because the reference draws all of a pixel's samples and bounces sequentially from one generator
// (ray-tracer-slave/src/main.rs:69-77).  The reference's recursion (ray_color, main.rs:108-146) is flattened into
// ONE loop whose trip is a single nearest-hit query.  Lanes are independent workers: a lane that finishes its pixel
// takes the next pixel of the warp's tile instead of idling until the slowest pixel of the tile is done.
//
//   * scene staging: geometry + traversal tree are one contiguous image in the scene blob and reach shared memory
//     by ONE cp.async.bulk per CTA, completion on an mbarrier (UBLKCP in SASS); one 1024-thread CTA per SM, so one
//     copy of the scene per SM and the rest of the 228 KB left to L1 for the traversal stacks
//   * output: finished pixels are staged in a per-warp shared-memory tile; a complete tile leaves as twelve
//     8-byte row vectors (the frame may be peer memory: these are the NVLink stores of the fused render + gather)
//   * completion: the lane that completes a tile adds its pixel count to the warp's batching word; one system-scope
//     release (red.release.sys) per warp and slab adds it to the slab's counter in the frame's control block, which the
//     frame owner's copy stream waits on by value: finished slabs reach the host while the rest still renders
//   * tail: the last tickets are handed out pixel by pixel, so no lane idles while a neighbour finishes a tile
//
// The nearest-hit query itself (K1 brute force / K2 BVH) lives in rt_trace.cuh.
#include "rt_trace.cuh"
#include "rt_host.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>

namespace rtb {

constexpr int SMEM_TPB = 1024;
constexpr int OUT_SLOTS = 4;                        // tiles a warp can have in flight in its output stage
constexpr int TILE_PIX = TILE_W * TILE_H;
constexpr int TILE_BYTES = TILE_PIX * 3;
constexpr uint32_t KEY_FREE = 0xffffffffu;

// ---- bulk-copy staging (TMA engine, non-tensor form) ----------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
    uint32_t done = 0;
    for (uint32_t spin = 0; !done; spin++) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (spin > (1u << 22)) __trap();  // a copy that never lands must not hang the device
    }
}

// ---------------------------------------------------------------------------------------------
// Output stage helpers (cold code, out of line: the hot loop's instruction footprint matters more than a call here)
// ---------------------------------------------------------------------------------------------
struct OutDesc {  // where finished pixels go (by value: never a reference to the kernel's parameter block)
    uint8_t* out;
    unsigned long long* done;
    uint32_t width, out_row0, row0, slab_tile_rows;
};
__device__ __forceinline__ uint32_t slab_of_row(const OutDesc& od, uint32_t y) { return ((y - od.row0) / TILE_H) / od.slab_tile_rows; }

// Completion counts leave a warp in batches: a system-scope release costs microseconds (it waits for every store of
// the warp to be acknowledged, over NVLink for a peer frame).  A warp keeps the pixels it has written to the frame since
// its last release in one shared-memory word, slab << 24 | count (`cntw`): the slab is the one of the warp's current
// tile; counts of that slab are added to the word, counts of any other slab (stragglers) are released at once; the word
// is released when the warp fetches a tile of another slab and when it runs out of work (both converged: the barrier
// there orders the other lanes' stores before the releasing lane's fence).
// A RELEASE only (red.release.sys): it orders this lane's earlier stores — and, cumulatively, the other lanes' stores that
// a __syncwarp ordered before this lane — in front of the count.  __threadfence_system() would be an acquire as well and
// costs a CCTL.IVALL: the SM's whole L1, where the traversal stacks live, thrown away at every release.
__device__ __forceinline__ void release_count(unsigned long long* done, uint32_t slab, uint32_t cnt) {
    asm volatile("red.release.sys.global.add.u64 [%0], %1;" ::"l"(done + slab), "l"((unsigned long long)cnt) : "memory");
}
__device__ __forceinline__ void count_pixels(const OutDesc& od, uint32_t slab, uint32_t cnt, uint32_t* cntw) {
    if (!od.done || cnt == 0) return;
    if (cntw && (*reinterpret_cast<volatile uint32_t*>(cntw) >> 24) == slab) atomicAdd(cntw, cnt);
    else release_count(od.done, slab, cnt);
}

// ONE lane — the one that staged the last missing pixel of a tile: the tile (st = its 96 staged bytes, origin x0 / y0,
// `valid` = the pixels that exist) goes to the frame as twelve 8-byte row vectors and is counted, minus the `hold`
// pixels a second pass will count.  Every store of the tile is this lane's own, so is the release if one is due.
__device__ __noinline__ void complete_tile(const OutDesc od, const uint8_t* st, uint32_t x0, uint32_t y0, uint32_t valid,
                                           uint32_t hold, uint32_t* cntw) {
    const bool vec = valid == 0xffffffffu && ((od.width & 7u) == 0) && ((reinterpret_cast<uintptr_t>(od.out) & 7u) == 0);
    if (vec) {
#pragma unroll 1
        for (uint32_t r = 0; r < (uint32_t)TILE_H; r++) {
            uint2* dst = reinterpret_cast<uint2*>(od.out + ((size_t)(y0 + r - od.out_row0) * od.width + x0) * 3);
            const uint2* src = reinterpret_cast<const uint2*>(st + r * 24);
            const uint2 v0 = src[0], v1 = src[1], v2 = src[2];
            dst[0] = v0; dst[1] = v1; dst[2] = v2;
        }
    } else {
        for (uint32_t m = valid; m; m &= m - 1u) {
            const uint32_t j = (uint32_t)__ffs(m) - 1u;
            uint8_t* dst = od.out + ((size_t)(y0 + (j >> 3) - od.out_row0) * od.width + x0 + (j & 7u)) * 3;
            dst[0] = st[j * 3 + 0]; dst[1] = st[j * 3 + 1]; dst[2] = st[j * 3 + 2];
        }
    }
    count_pixels(od, slab_of_row(od, y0), (uint32_t)__popc(valid) - hold, cntw);
}

// All 32 lanes (tile fetch found no free slot): the pixels `mask` staged so far of an unfinished tile leave as bytes;
// the lanes still working on that tile will find its slot re-keyed and store directly.
__device__ __noinline__ void evict_tile(const OutDesc od, const uint8_t* st, uint32_t x0, uint32_t y0, uint32_t mask, uint32_t hold,
                                        uint32_t* cntw) {
    const int lane = threadIdx.x & 31;
    if ((mask >> lane) & 1u) {
        const size_t off = ((size_t)(y0 + (lane >> 3) - od.out_row0) * od.width + x0 + (lane & 7)) * 3;
        od.out[off + 0] = st[lane * 3 + 0];
        od.out[off + 1] = st[lane * 3 + 1];
        od.out[off + 2] = st[lane * 3 + 2];
    }
    __syncwarp();
    if (lane == 0) count_pixels(od, slab_of_row(od, y0), (uint32_t)__popc(mask) - hold, cntw);
}

// One lane: a finished pixel straight to the frame (no stage slot — the tail's pixel tickets — or the slot was evicted).
__device__ __noinline__ void store_pixel(const OutDesc od, uint32_t x, uint32_t y, uint32_t rgb, bool count, uint32_t* cntw) {
    const size_t off = ((size_t)(y - od.out_row0) * od.width + x) * 3;
    od.out[off + 0] = (uint8_t)rgb;
    od.out[off + 1] = (uint8_t)(rgb >> 8);
    od.out[off + 2] = (uint8_t)(rgb >> 16);
    if (count) count_pixels(od, slab_of_row(od, y), 1u, cntw);
}

// ---------------------------------------------------------------------------------------------
// The megakernel
// ---------------------------------------------------------------------------------------------
// per-lane state word                       warp-uniform state word
constexpr uint32_t L_HAVE = 1u;           constexpr uint32_t W_TILES_LEFT = 1u;
constexpr uint32_t L_FINISHED = 2u;       constexpr uint32_t W_IN_TAIL = 2u;
                                          constexpr int W_SLOT_SHIFT = 4;    // 3 bits: slot + 1 of the warp's current tile
constexpr uint32_t L_REDO = 8u;           constexpr int W_NEXT_SHIFT = 8;    // 6 bits: next pixel of the current tile
constexpr int L_SLOT_SHIFT = 4;           // 3 bits: output-stage slot + 1 of this lane's pixel (0: straight to the frame)
constexpr uint32_t L_SECOND = 128u;       // this pixel comes from the redo list: its first pass was held back, not counted

// RESUME: the launch renders samples [pr.s0, pr.spp) of each pixel's chain from the state in pr.state_in and leaves the
// state in pr.state_out (rt_render_samples, rt_render_samples_multi); the other instantiations render samples [0, pr.spp).
// With the output stage (a frame shared between ranks) a held-back pixel stores no state but is counted in s_hold like
// any other: its second pass, in the kernel or by the host, starts over from the same state_in and counts it then.
// BANDS: the launch's rows are the bands of pr.band_table stacked (rt_render_divisions).  px / py stay in launch rows for
// the stage, the counters, the redo list and the output; the image row, which only the seed and the camera ray need, is
// looked up where it is used rather than held through the traversal.
template <int ISECT, bool SMEM, bool COUNT, bool STAGE, int MINB, int TPB, bool RESUME = false, bool BANDS = false>
__global__ void __launch_bounds__(TPB, MINB) render_kernel_lanes(const DevScene sc, const DevCamera cam,
                                                                const DevParams pr) {
    extern __shared__ float4 smem_dyn[];
    constexpr int NW = TPB / 32;
    // output stage, per warp: OUT_SLOTS tiles of RGB8 + which tile each slot holds (key = tile index in this launch's
    // grid), which of its pixels are staged, which exist (edge tiles are partial), how many staged pixels are held back
    __shared__ __align__(16) uint8_t s_stage[STAGE ? NW : 1][OUT_SLOTS][TILE_BYTES];
    __shared__ uint32_t s_key[STAGE ? NW : 1][OUT_SLOTS], s_fill[STAGE ? NW : 1][OUT_SLOTS],
        s_valid[STAGE ? NW : 1][OUT_SLOTS], s_hold[STAGE ? NW : 1][OUT_SLOTS],
        s_cnt[STAGE ? NW : 1];  // completion count not released yet: slab << 24 | pixels (see count_pixels)
    __shared__ __align__(8) unsigned long long s_bar;

    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;

    SceneView sv;
    if (SMEM) {
        // image = blob layout, scene_image_bytes long: sph | tri | lnode (BVH) or sph | tri + sph2 (brute force)
        const uint32_t geom = sc.ns * 16u + sc.nt * 64u;
        const uint32_t rest = (ISECT == RT_INTERSECT_BVH) ? sc.lni * (uint32_t)NODE_BYTES
                                                          : ((sc.ns + 7u) & ~7u) * 16u;
        uint8_t* base = reinterpret_cast<uint8_t*>(smem_dyn);
        if (threadIdx.x == 0) mbar_init(&s_bar, 1);
        __syncthreads();
        if (threadIdx.x == 0) {
            mbar_expect_tx(&s_bar, geom + rest);
            if (ISECT == RT_INTERSECT_BVH) {
                bulk_g2s(base, sc.sph, geom + rest, &s_bar);  // the whole image in one copy
            } else {
                if (geom) bulk_g2s(base, sc.sph, geom, &s_bar);
                if (rest) bulk_g2s(base + geom, sc.sph2, rest, &s_bar);
            }
        }
        sv.sph = reinterpret_cast<const float4*>(base);
        sv.tri = reinterpret_cast<const float4*>(base + sc.ns * 16u);
        sv.sph2 = reinterpret_cast<const float4*>(base + geom);
        sv.nodes_s = (uint32_t)__cvta_generic_to_shared(base + geom);
        sv.nodes_g = nullptr;
    } else {
        sv.sph2 = sc.sph2;
        sv.sph = sc.sph; sv.tri = sc.tri;
        sv.nodes_s = 0;
        sv.nodes_g = reinterpret_cast<const char*>(sc.lnode);
    }
    if (STAGE && lane < OUT_SLOTS) {
        s_key[warp][lane] = KEY_FREE;
        s_fill[warp][lane] = 0u;
        s_hold[warp][lane] = 0u;
        if (lane == 0) s_cnt[warp] = 0xffu << 24;  // no slab yet
    }
    if (SMEM) mbar_wait(&s_bar, 0);  // every thread observes the completed transaction itself
    if (SMEM && ISECT == RT_INTERSECT_BVH) {
        // inner-node child codes arrive as byte offsets from record 0: make them shared-window addresses, once
        for (uint32_t i = threadIdx.x; i < sc.lni; i += TPB) {
            int2* ch = reinterpret_cast<int2*>(reinterpret_cast<uint8_t*>(smem_dyn) + sc.ns * 16u + sc.nt * 64u +
                                               i * (uint32_t)NODE_BYTES + 48u);
            int2 v = *ch;
            if (v.x >= 0) v.x += (int)sv.nodes_s;
            if (v.y >= 0) v.y += (int)sv.nodes_s;
            *ch = v;
        }
        __syncthreads();
    }
    __syncwarp();

    const unsigned lt_mask = (1u << lane) - 1u;
    const uint32_t total_tiles = pr.tiles_x * pr.tiles_y;
    const uint32_t tail_pixels = pr.pixel_list ? pr.list_count : (pr.my_tickets - pr.tail_first) * (uint32_t)TILE_PIX;
    const float spp_f = (float)pr.spp;

    Ctr ctr;
#pragma unroll
    for (int i = 0; i < NUM_COUNTERS; i++) ctr.v[i] = 0;
    unsigned long long rays = 0;

    uint32_t st = 0;                 // per-lane state word (L_*)
    uint32_t ws = W_TILES_LEFT | ((uint32_t)TILE_PIX << W_NEXT_SHIFT);  // warp-uniform state word (W_*): no tile yet
    uint32_t tile_g = 0;             // warp-uniform: tile index (row-major in this launch's grid) of the current tile
    uint32_t px = 0, py = 0, s = 0, left = 0, np = 0;
    float sr = 0.0f, sg = 0.0f, sb = 0.0f;
    Rng rng;
    rng.s0 = rng.s1 = rng.s2 = rng.s3 = 0;
    V3 o = mk(0, 0, 0), d = mk(0, 0, 1);
    uint32_t path[MAX_PATH];  // pids of the non-terminal hits of the current sample

    // ticket → tile of this rank: group k of `tile_ranks` tiles, rotated; bottom-up so the sky rows end the launch
    auto tile_of_ticket = [&](uint32_t k) -> uint32_t {
        uint32_t g = k * pr.tile_ranks + (pr.tile_rank + k) % pr.tile_ranks;
        if (g < total_tiles) g = total_tiles - 1 - g;
        return g;
    };
    auto out_desc = [&]() { return OutDesc{pr.out, pr.done, pr.width, pr.out_row0, pr.row0, pr.slab_tile_rows}; };
    // launch row → image row (the identity outside BANDS)
    auto image_row = [&](uint32_t y) -> uint32_t {
        if constexpr (BANDS) return __ldg(&pr.band_table[y / pr.band_rows]) * pr.band_rows + y % pr.band_rows;
        else return y;
    };

    for (;;) {
        // ---- hand out pixels: warp-cooperative, tile by tile ----
        unsigned want = __ballot_sync(FULL, (st & (L_HAVE | L_FINISHED)) == 0);
        if (want) {
            while (want) {
                // (1) warp-uniform: a unit to hand out from — the current tile, a new tile, or the tail's pixel tickets
                if (((ws >> W_NEXT_SHIFT) & 63u) >= (uint32_t)TILE_PIX && !(ws & W_IN_TAIL)) {
                    if (!(ws & W_TILES_LEFT)) {
                        if (!(st & L_HAVE)) st |= L_FINISHED;
                        break;
                    }
                    uint32_t k = 0;
                    if (lane == 0) k = atomicAdd(&pr.tile_counter[0], 1u);
                    k = __shfl_sync(FULL, k, 0);
                    const uint32_t g = k < pr.tail_first ? tile_of_ticket(k) : total_tiles;
                    if (g >= total_tiles) {  // the whole-tile tickets are gone (only the last ticket group can be short)
                        ws |= W_IN_TAIL;
                    } else {
                        tile_g = g;
                        ws &= ~((63u << W_NEXT_SHIFT) | (7u << W_SLOT_SHIFT));  // next = 0, no slot
                        if (STAGE) {
                            // a free slot, else evict one: its staged pixels leave as bytes and the lanes still
                            // working on that tile will find the key changed and store directly
                            int sl = -1;
#pragma unroll
                            for (int i = OUT_SLOTS - 1; i >= 0; i--)
                                if (s_key[warp][i] == KEY_FREE) sl = i;
                            if (sl < 0) {
                                sl = (int)(k % OUT_SLOTS);
                                const uint32_t f = s_fill[warp][sl], og = s_key[warp][sl];
                                __syncwarp();
                                if (f) evict_tile(out_desc(), s_stage[warp][sl], (og % pr.tiles_x) * TILE_W,
                                                  pr.row0 + (og / pr.tiles_x) * TILE_H, f, s_hold[warp][sl], &s_cnt[warp]);
                            }
                            const uint32_t x0 = (g % pr.tiles_x) * TILE_W, y0 = pr.row0 + (g / pr.tiles_x) * TILE_H;
                            const uint32_t vm = __ballot_sync(FULL, (x0 + (lane & 7) < pr.width) && (y0 + (lane >> 3) < pr.row1));
                            __syncwarp();
                            if (lane == 0) {
                                s_key[warp][sl] = g;
                                s_fill[warp][sl] = 0u;
                                s_hold[warp][sl] = 0u;
                                s_valid[warp][sl] = vm;
                                // the batching word follows the warp's current tile: a new slab releases the old count
                                // (the barrier above ordered every lane's stores before this lane)
                                const uint32_t slab = ((g / pr.tiles_x) / pr.slab_tile_rows) & 0xffu, w = s_cnt[warp];
                                if ((w >> 24) != slab) {
                                    if (pr.done && (w & 0xffffffu)) release_count(pr.done, w >> 24, w & 0xffffffu);
                                    s_cnt[warp] = slab << 24;
                                }
                            }
                            __syncwarp();
                            ws |= (uint32_t)(sl + 1) << W_SLOT_SHIFT;
                        }
                    }
                }
                // (2) per wanting lane: a candidate pixel (x == width: none)
                uint32_t x = pr.width, y = 0, slot1 = 0, second = 0;
                const uint32_t my = __popc(want & lt_mask);
                const bool wants = (st & (L_HAVE | L_FINISHED)) == 0;
                // (a probe for waiting list entries beside every tile ticket, so that they are rendered again as soon as the
                // tables land instead of at the end, cost more than it saved: C3 37.7 -> 38.0 ms, 2 GPUs 19.7 -> 20.3)
                bool redo_round = false, exhausted = false;
                uint32_t base = 0;
                if (ws & W_IN_TAIL) {
                    // the tail of the launch (or a second pass over a pixel list): pixel tickets, one per wanting lane
                    if (lane == 0) base = atomicAdd(&pr.tile_counter[1], (unsigned int)__popc(want));
                    base = __shfl_sync(FULL, base, 0);
                    redo_round = exhausted = base >= tail_pixels;
                }
                if (redo_round) {
                    // Pixels that waited for the tie-break tables are rendered again by lanes that want work, once the
                    // tables have landed: lane 0 takes up to one list entry per wanting lane.
                    uint32_t t0 = 0, n_take = 0;
                    if (!pr.pixel_list && lane == 0) {
                        int landed = sc.aux_ready;
                        if (!landed) asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(landed) : "l"(sc.aux_flag) : "memory");
                        const unsigned long long cnt = *reinterpret_cast<volatile unsigned long long*>(pr.redo_count);
                        if (landed && cnt <= pr.redo_cap) {  // more than the list holds: the host repeats the launch
                            for (;;) {
                                t0 = *reinterpret_cast<volatile unsigned int*>(&pr.tile_counter[2]);
                                n_take = min((uint32_t)__popc(want), (uint32_t)cnt - min((uint32_t)cnt, t0));
                                if (n_take == 0 || atomicCAS(&pr.tile_counter[2], t0, t0 + n_take) == t0) break;
                            }
                        }
                    }
                    t0 = __shfl_sync(FULL, t0, 0);
                    n_take = __shfl_sync(FULL, n_take, 0);
                    if (n_take == 0 && exhausted) {  // the tickets are gone and nothing waits: this warp is done
                        ws &= ~(W_TILES_LEFT | W_IN_TAIL);
                        if (!(st & L_HAVE)) st |= L_FINISHED;
                        break;
                    }
                    if (n_take) {
                        if (wants && my < n_take) {
                            uint32_t e;  // the entry is written right after its index was reserved: wait for it
                            for (uint32_t spin = 0;; spin++) {
                                e = *reinterpret_cast<volatile unsigned int*>(&pr.redo_list[t0 + my]);
                                if (e & REDO_VALID) break;
                                if (spin > (1u << 24)) __trap();
                            }
                            e &= ~REDO_VALID;
                            x = e % pr.width;
                            y = e / pr.width;
                            second = L_SECOND;
                        }
                        base = tail_pixels;  // this round hands out list entries only
                    }
                }
                if (redo_round && base >= tail_pixels) {
                    // (nothing else this round)
                } else if (ws & W_IN_TAIL) {
                    const uint32_t idx = base + my;
                    if (wants && idx < tail_pixels) {
                        if (pr.pixel_list) {  // the host's second pass: exactly the listed pixels
                            const uint32_t p = pr.pixel_list[idx] & ~REDO_VALID;
                            x = p % pr.width;
                            y = p / pr.width;
                        } else {
                            const uint32_t g = tile_of_ticket(pr.tail_first + idx / TILE_PIX);
                            const uint32_t j = idx % TILE_PIX;
                            if (g < total_tiles) {
                                x = (g % pr.tiles_x) * TILE_W + (j & (TILE_W - 1));
                                y = pr.row0 + (g / pr.tiles_x) * TILE_H + (j / TILE_W);
                            }
                        }
                    }
                } else {
                    const uint32_t next = (ws >> W_NEXT_SHIFT) & 63u, avail = (uint32_t)TILE_PIX - next;
                    if (wants && my < avail) {
                        const uint32_t j = next + my;
                        x = (tile_g % pr.tiles_x) * TILE_W + (j & (TILE_W - 1));
                        y = pr.row0 + (tile_g / pr.tiles_x) * TILE_H + (j / TILE_W);
                        slot1 = (ws >> W_SLOT_SHIFT) & 7u;
                    }
                    ws += min((uint32_t)__popc(want), avail) << W_NEXT_SHIFT;
                }
                // (3) the lane takes its pixel (tiles on the right / bottom edge are partial)
                if (x < pr.width && y < pr.row1) {
                    px = x; py = y;
                    st = L_HAVE | (slot1 << L_SLOT_SHIFT) | second;
                    if constexpr (RESUME) {
                        if (pr.s0 == 0) {  // the chain's start: nothing to read
                            rng.seed_from_u64(pr.seed + ((uint64_t)y * pr.width + x));
                            sr = sg = sb = 0.0f;
                        } else {
                            const uint4* rec = pr.state_in + ((size_t)(y - pr.row0) * pr.width + x) * 3;
                            const uint4 a = __ldcs(rec), b = __ldcs(rec + 1), c = __ldcs(rec + 2);
                            rng.s0 = ((uint64_t)a.y << 32) | a.x;
                            rng.s1 = ((uint64_t)a.w << 32) | a.z;
                            rng.s2 = ((uint64_t)b.y << 32) | b.x;
                            rng.s3 = ((uint64_t)b.w << 32) | b.z;
                            sr = __uint_as_float(c.x); sg = __uint_as_float(c.y); sb = __uint_as_float(c.z);
                        }
                        s = pr.s0;
                    } else {
                        rng.seed_from_u64(pr.seed + ((uint64_t)image_row(y) * pr.width + x));
                        sr = sg = sb = 0.0f;
                        s = 0;
                    }
                    left = 0;
                }
                want = __ballot_sync(FULL, (st & (L_HAVE | L_FINISHED)) == 0);
            }
        }
        if (__ballot_sync(FULL, st & L_HAVE) == 0) break;

        if (st & L_HAVE) {
            if (left == 0) {  // start sample s
                primary_ray(cam, px, pr.height - image_row(py) - 1, rng, &o, &d);  // y_cam = h - y - 1 (main.rs:71)
                left = pr.depth;
                np = 0;
            }
            // ---- one nearest-hit query (ray_color with depth > 0) ----
            rays++;
            if (COUNT) {
                ctr.v[CTR_ACTIVE_LANES]++;
                unsigned am = __activemask();
                if (lane == (__ffs(am) - 1)) ctr.v[CTR_TOTAL_LANES] += 32;
            }
            Hit h;
            if (ISECT == RT_INTERSECT_BRUTE) trace_brute<COUNT>(sc, sv, o, d, h, ctr);
            else trace_bvh_ch<COUNT, SMEM>(sc, sv, o, d, h, ctr);
            if (h.unsure) st |= L_REDO;

            bool done;
            float Lr, Lg, Lb;
            if (h.pid >= 0) {
                const float e = __ldg(&sc.emis[h.pid]);
                const float4 m = __ldg(&sc.mat[h.pid]);
                if (e > 0.0f) {  // emission * albedo (main.rs:116-117)
                    Lr = x_mul(m.x, e); Lg = x_mul(m.y, e); Lb = x_mul(m.z, e);
                    done = true;
                    if (COUNT) ctr.v[CTR_EMISSIVE]++;
                } else {
                    V3 n;
                    if (COUNT) ctr.v[h.pid < (int)sc.ns ? CTR_SHADE_SPH : CTR_SHADE_TRI]++;
                    if (h.pid < (int)sc.ns) {
                        n = x_normalize_or_zero(x_sub(h.p, ld3(sv.sph[h.pid])));  // sphere.rs:49-51
                    } else {
                        n = ld3(sv.tri[4 * (h.pid - (int)sc.ns) + 3]);  // mesh.rs:163-165 (host, same ops)
                    }
                    V3 diffuse = x_add(unit_sphere(rng), n);
                    float kk = x_mul(2.0f, x_dot(d, n));
                    V3 glossy = x_sub(d, x_scale(n, kk));
                    V3 scat = x_add(diffuse, x_scale(x_sub(glossy, diffuse), m.w));
                    const V3 nd = x_normalize_or(scat, n);  // try_normalize(..).unwrap_or(normal) (main.rs:126)
                    o = h.p;
                    d = x_normalize_div(nd);  // Ray::new
                    path[np++] = (uint32_t)h.pid;
                    left--;
                    done = (left == 0);       // next call has depth == 0 → BLACK, no query
                    Lr = Lg = Lb = 0.0f;
                }
            } else {  // sky (main.rs:135-144)
                if (COUNT) ctr.v[CTR_SKY]++;
                const float ny = x_normalize_or_zero(d).y;
                float t = x_add(x_mul(ny, 0.5f), 1.0f);
                float k1 = x_sub(1.0f, t);
                float w = x_mul(1.0f, t);
                Lr = x_add(w, x_mul(0.3f, k1));
                Lg = Lr;
                Lb = x_add(w, x_mul(0.8f, k1));
                done = true;
            }
            if (done) {
                // fold albedo ⊙ (albedo ⊙ (... ⊙ L)) innermost first, like the recursion unwinding
#pragma unroll 1
                while (np > 0) {
                    const float4 m = __ldg(&sc.mat[path[--np]]);
                    Lr = x_mul(m.x, Lr); Lg = x_mul(m.y, Lg); Lb = x_mul(m.z, Lb);
                }
                sr = x_add(sr, Lr); sg = x_add(sg, Lg); sb = x_add(sb, Lb);
                s++;
                left = 0;
                if (s == pr.spp) {  // pixel finished (main.rs:78-81)
                    if constexpr (RESUME) {
                        // a pixel held back for the second pass leaves its state there (from the same state_in)
                        if (!(st & L_REDO)) {
                            uint4* rec = pr.state_out + ((size_t)(py - pr.row0) * pr.width + px) * 3;
                            __stcs(rec, make_uint4((uint32_t)rng.s0, (uint32_t)(rng.s0 >> 32), (uint32_t)rng.s1, (uint32_t)(rng.s1 >> 32)));
                            __stcs(rec + 1, make_uint4((uint32_t)rng.s2, (uint32_t)(rng.s2 >> 32), (uint32_t)rng.s3, (uint32_t)(rng.s3 >> 32)));
                            __stcs(rec + 2, make_uint4(__float_as_uint(sr), __float_as_uint(sg), __float_as_uint(sb), 0u));
                        }
                    }
                    const uint32_t rgb = quantise(sr, spp_f) | (quantise(sg, spp_f) << 8) | (quantise(sb, spp_f) << 16);
                    // a pixel that goes to the second pass is counted there: a slab whose count is complete is final
                    const bool hold = (st & L_REDO) != 0;
                    const int my_sl = (int)((st >> L_SLOT_SHIFT) & 7u) - 1;
                    bool staged = false;
                    if (STAGE && my_sl >= 0) {
                        const uint32_t key = ((py - pr.row0) / TILE_H) * pr.tiles_x + px / TILE_W;
                        if (s_key[warp][my_sl] == key) {  // the slot still holds this pixel's tile (not evicted)
                            const uint32_t j = (px & (TILE_W - 1)) + TILE_W * ((py - pr.row0) & (TILE_H - 1));
                            uint8_t* dst = s_stage[warp][my_sl] + 3 * j;
                            dst[0] = (uint8_t)rgb; dst[1] = (uint8_t)(rgb >> 8); dst[2] = (uint8_t)(rgb >> 16);
                            if (hold) atomicAdd(&s_hold[warp][my_sl], 1u);
                            // the bytes before the bit: shared-memory operations of ONE warp are performed in issue order,
                            // and only this warp touches its stage, so a compiler barrier is all the ordering needed
                            // (a __threadfence_block() here is a MEMBAR.SC.CTA per finished pixel: +30 % at 1 spp)
                            asm volatile("" ::: "memory");
                            const uint32_t now = atomicOr(&s_fill[warp][my_sl], 1u << j) | (1u << j);
                            if (now == s_valid[warp][my_sl]) {  // the last missing pixel: this lane sends the tile off
                                complete_tile(out_desc(), s_stage[warp][my_sl], px & ~(uint32_t)(TILE_W - 1),
                                              py - ((py - pr.row0) & (TILE_H - 1)), now, s_hold[warp][my_sl], &s_cnt[warp]);
                                s_fill[warp][my_sl] = 0u;
                                s_hold[warp][my_sl] = 0u;
                                asm volatile("" ::: "memory");
                                s_key[warp][my_sl] = KEY_FREE;
                            }
                            staged = true;
                        }
                    }
                    if (!staged) store_pixel(out_desc(), px, py, rgb, !hold, STAGE ? &s_cnt[warp] : nullptr);
                    if (st & L_REDO) {  // (a second pass never gets here: the tables are there for it)
                        atomicAdd(&pr.redo_slab[((py - pr.row0) / TILE_H) / pr.slab_tile_rows], 1ull);
                        const unsigned long long at = atomicAdd(pr.redo_count, 1ull);
                        if (at < pr.redo_cap) pr.redo_list[at] = REDO_VALID | (py * pr.width + px);
                    } else if (st & L_SECOND) {
                        atomicAdd(&pr.redo_slab[((py - pr.row0) / TILE_H) / pr.slab_tile_rows], ~0ull);  // no longer held back
                    }
                    st &= ~(L_HAVE | L_REDO | L_SECOND);
                }
            }
        }
    }

    if (STAGE && pr.done) {  // the warp is out of work: what it still holds is released now
        __syncwarp();
        const uint32_t w = s_cnt[warp];
        if (lane == 0 && (w & 0xffffffu)) release_count(pr.done, w >> 24, w & 0xffffffu);
    }
    ctr.v[CTR_RAYS] = rays;
#pragma unroll
    for (int i = 0; i < NUM_COUNTERS; i++) {
        if (!COUNT && i != CTR_RAYS) continue;
        unsigned long long v = ctr.v[i];
#pragma unroll
        for (int ofs = 16; ofs > 0; ofs >>= 1) v += __shfl_down_sync(FULL, v, ofs);
        if (lane == 0 && v) atomicAdd(&pr.counters[i], v);
    }
}

// Spins (one thread) until a counter of a frame's control block reaches `target`.  Used by the ranks that wait for the
// owner's "consumed" word in front of their next kernel, and — only when the driver has no 64-bit stream waits
// (rt_init: cuStreamWaitValue64) — by the owner in front of each slab's device→host copy: beside 1024-thread CTAs that
// own every register of their SM such a kernel becomes resident only when the render kernel ends.  Bounded: a rank
// that died must not hang anybody.
__global__ void wait_slab_kernel(const unsigned long long* done, unsigned long long target, unsigned int* timeout_flag,
                                 unsigned long long max_ns) {
    if (*reinterpret_cast<volatile unsigned int*>(timeout_flag)) return;  // an earlier wait of this frame gave up already
    unsigned long long t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
        unsigned long long v;
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(done) : "memory");
        if (v >= target) return;
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        if (t - t0 > max_ns) {
            *reinterpret_cast<volatile unsigned int*>(timeout_flag) = 1u;  // mapped host memory
            __threadfence_system();
            return;
        }
        __nanosleep(200);
    }
}

// All slabs of a frame at once (nobody copies them out: the frame stays on the device): thread s waits for slab s.
__global__ void wait_all_slabs_kernel(const unsigned long long* done, unsigned long long seq, uint32_t slabs, uint32_t tile_rows,
                                      uint32_t rows, uint32_t width, unsigned int* timeout_flag, unsigned long long max_ns) {
    const uint32_t s = threadIdx.x;
    if (s >= slabs) return;
    const uint32_t r0 = min(rows, s * tile_rows * (uint32_t)TILE_H), r1 = min(rows, (s + 1) * tile_rows * (uint32_t)TILE_H);
    const unsigned long long target = seq * (unsigned long long)(r1 - r0) * width;
    unsigned long long t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
        unsigned long long v;
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(done + s) : "memory");
        if (v >= target) return;
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        if (t - t0 > max_ns) {
            *reinterpret_cast<volatile unsigned int*>(timeout_flag) = 1u;
            __threadfence_system();
            return;
        }
        __nanosleep(200);
    }
}

__global__ void set_u64_kernel(unsigned long long* p, unsigned long long v) {
    __threadfence_system();
    *reinterpret_cast<volatile unsigned long long*>(p) = v;
    __threadfence_system();
}

// done[s] += add[s] with a system-scope release: the counts a second pass over a whole launch could not attribute
__global__ void add_counts_kernel(unsigned long long* done, const unsigned long long* add, int n) {
    const int i = threadIdx.x;
    if (i < n && add[i]) {
        __threadfence_system();
        atomicAdd(&done[i], add[i]);
    }
}

// rt_accum_read_linear: sum / samples per channel of every pixel's state record (the exact-domain division quantise()
// starts with), rows * width * 3 floats.
__global__ void accum_linear_kernel(const uint4* state, float* out, unsigned long long pixels, float samples) {
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < pixels;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint4 c = state[3 * i + 2];
        out[3 * i + 0] = x_div(__uint_as_float(c.x), samples);
        out[3 * i + 1] = x_div(__uint_as_float(c.y), samples);
        out[3 * i + 2] = x_div(__uint_as_float(c.z), samples);
    }
}

// ---------------------------------------------------------------------------------------------
// FFMA-chain micro-benchmark for the FP32 roofline denominator
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) fp32_peak_kernel(float* out, int iters, float seed) {
    float a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6,
          a7 = a0 + 7;
    const float m = 0.999f + seed * 1e-6f, c = 1e-3f + seed;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 16; k++) {
            a0 = fmaf(a0, m, c); a1 = fmaf(a1, m, c); a2 = fmaf(a2, m, c); a3 = fmaf(a3, m, c);
            a4 = fmaf(a4, m, c); a5 = fmaf(a5, m, c); a6 = fmaf(a6, m, c); a7 = fmaf(a7, m, c);
        }
    }
    float r = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
    if (r == 123.456f) out[blockIdx.x * blockDim.x + threadIdx.x] = r;
}

// ---------------------------------------------------------------------------------------------
// Test hooks: read from the environment ONCE (rt_init forces the read); not API
// ---------------------------------------------------------------------------------------------
static int env_int(const char* name, int dflt) {
    const char* e = std::getenv(name);
    return e ? std::atoi(e) : dflt;
}
static bool env_is(const char* name, const char* value) {
    const char* e = std::getenv(name);
    return e && std::strcmp(e, value) == 0;
}
const TestHooks& test_hooks() {
    static const TestHooks t = [] {
        TestHooks v;
        v.build_mode = env_is("RT_B200_BUILD", "host") ? 0 : (env_is("RT_B200_BUILD", "device") ? 2 : 1);
        v.aux_delay_ms = std::max(0, env_int("RT_B200_AUX_DELAY_MS", 0));
        v.wait_timeout_ms = std::max(1, env_int("RT_B200_WAIT_TIMEOUT_MS", 20000));
        v.no_stream_wait = std::getenv("RT_B200_NO_STREAM_WAIT") != nullptr;
        return v;
    }();
    return t;
}

// ---------------------------------------------------------------------------------------------
// Launcher
// ---------------------------------------------------------------------------------------------
typedef void (*KernelFn)(const DevScene, const DevCamera, const DevParams);

// instantiations: the product shapes (one 1024-thread CTA per SM with the scene in shared memory; 4 x 256 threads at
// 64 registers when the scene is read through L1/L2 and the BVH kernel is latency bound — 65,536 spheres 3.13 → 2.84 ms)
// with and without the output stage, and the instrumented (COUNT) form at 3 x 256 threads
template <int ISECT, bool SMEM>
static KernelFn pick_lanes(bool count, bool stage, int* threads) {
    if (count) {
        *threads = THREADS;
        return (KernelFn)render_kernel_lanes<ISECT, SMEM, true, false, 3, THREADS>;
    }
    if (SMEM) {
        // one CTA per SM, as many warps as a CTA can have: C3 40.6 ms at 640 threads, 38.0 at 768 (74 registers), 37.65 at
        // 896 (72), 36.7 at 1024 (64 registers, 48 bytes of spills) — profiles/r2_ab_cta_size.log
        *threads = SMEM_TPB;
        return stage ? (KernelFn)render_kernel_lanes<ISECT, SMEM, false, true, 1, SMEM_TPB>
                     : (KernelFn)render_kernel_lanes<ISECT, SMEM, false, false, 1, SMEM_TPB>;
    }
    *threads = THREADS;
    if (ISECT == RT_INTERSECT_BVH)
        return stage ? (KernelFn)render_kernel_lanes<ISECT, SMEM, false, true, 4, THREADS>
                     : (KernelFn)render_kernel_lanes<ISECT, SMEM, false, false, 4, THREADS>;
    return stage ? (KernelFn)render_kernel_lanes<ISECT, SMEM, false, true, 3, THREADS>
                 : (KernelFn)render_kernel_lanes<ISECT, SMEM, false, false, 3, THREADS>;
}

// the resumable form (rt_render_samples, rt_render_samples_multi): the same CTA shapes with and without the output
// stage, no instrumented variant
template <int ISECT, bool SMEM>
static KernelFn pick_resume(bool stage, int* threads) {
    if constexpr (SMEM) {
        *threads = SMEM_TPB;
        return stage ? (KernelFn)render_kernel_lanes<ISECT, SMEM, false, true, 1, SMEM_TPB, true>
                     : (KernelFn)render_kernel_lanes<ISECT, SMEM, false, false, 1, SMEM_TPB, true>;
    } else {
        *threads = THREADS;
        if constexpr (ISECT == RT_INTERSECT_BVH)
            return stage ? (KernelFn)render_kernel_lanes<ISECT, SMEM, false, true, 4, THREADS, true>
                         : (KernelFn)render_kernel_lanes<ISECT, SMEM, false, false, 4, THREADS, true>;
        else
            return stage ? (KernelFn)render_kernel_lanes<ISECT, SMEM, false, true, 3, THREADS, true>
                         : (KernelFn)render_kernel_lanes<ISECT, SMEM, false, false, 3, THREADS, true>;
    }
}

// the banded form (rt_render_divisions with a list that is not one contiguous run): the product CTA shapes with and
// without the output stage, no instrumented or resumable variant
template <int ISECT, bool SMEM>
static KernelFn pick_bands(bool stage, int* threads) {
    if constexpr (SMEM) {
        *threads = SMEM_TPB;
        return stage ? (KernelFn)render_kernel_lanes<ISECT, SMEM, false, true, 1, SMEM_TPB, false, true>
                     : (KernelFn)render_kernel_lanes<ISECT, SMEM, false, false, 1, SMEM_TPB, false, true>;
    } else {
        *threads = THREADS;
        if constexpr (ISECT == RT_INTERSECT_BVH)
            return stage ? (KernelFn)render_kernel_lanes<ISECT, SMEM, false, true, 4, THREADS, false, true>
                         : (KernelFn)render_kernel_lanes<ISECT, SMEM, false, false, 4, THREADS, false, true>;
        else
            return stage ? (KernelFn)render_kernel_lanes<ISECT, SMEM, false, true, 3, THREADS, false, true>
                         : (KernelFn)render_kernel_lanes<ISECT, SMEM, false, false, 3, THREADS, false, true>;
    }
}

// Resolves every kernel variant once per context so that the first render does not pay the lazy module load.
cudaError_t preload_kernels() {
    cudaFuncAttributes a;
    cudaError_t e;
    int th;
#define RT_TOUCH(fn)                                                    \
    if ((e = cudaFuncGetAttributes(&a, fn)) != cudaSuccess) return e;
    for (int count = 0; count < 2; count++)
        for (int stage = 0; stage < 2; stage++) {
            RT_TOUCH((pick_lanes<RT_INTERSECT_BVH, true>(count, stage, &th)));
            RT_TOUCH((pick_lanes<RT_INTERSECT_BVH, false>(count, stage, &th)));
            RT_TOUCH((pick_lanes<RT_INTERSECT_BRUTE, true>(count, stage, &th)));
            RT_TOUCH((pick_lanes<RT_INTERSECT_BRUTE, false>(count, stage, &th)));
        }
    for (int stage = 0; stage < 2; stage++) {
        RT_TOUCH((pick_resume<RT_INTERSECT_BVH, true>(stage, &th)));
        RT_TOUCH((pick_resume<RT_INTERSECT_BVH, false>(stage, &th)));
        RT_TOUCH((pick_resume<RT_INTERSECT_BRUTE, true>(stage, &th)));
        RT_TOUCH((pick_resume<RT_INTERSECT_BRUTE, false>(stage, &th)));
        RT_TOUCH((pick_bands<RT_INTERSECT_BVH, true>(stage, &th)));
        RT_TOUCH((pick_bands<RT_INTERSECT_BVH, false>(stage, &th)));
        RT_TOUCH((pick_bands<RT_INTERSECT_BRUTE, true>(stage, &th)));
        RT_TOUCH((pick_bands<RT_INTERSECT_BRUTE, false>(stage, &th)));
    }
    RT_TOUCH(accum_linear_kernel);
    RT_TOUCH(wait_slab_kernel);
    RT_TOUCH(wait_all_slabs_kernel);
    RT_TOUCH(add_counts_kernel);
    RT_TOUCH(set_u64_kernel);
    RT_TOUCH(fp32_peak_kernel);
#undef RT_TOUCH
    return cudaSuccess;
}

// Share of a launch's tickets handed out pixel by pixel at its end.  0 to 300 permille measured the same on C3 at 8
// ranks (4.67 / 4.68 / 4.67 / 4.67 / 4.64 ms), 600 and more slower (profiles/r2_final_tail_sweep.log).
constexpr uint64_t kTailPermille = 30;

cudaError_t launch_render(const DevScene& sc, const DevCamera& cam, const DevParams& pr, int isect, bool count,
                          int sm_count, int smem_optin, cudaStream_t stream, LaunchInfo* info) {
    const bool resume = pr.state_out != nullptr;  // rt_render_samples
    const bool bands = pr.band_table != nullptr;  // rt_render_divisions
    if (resume || bands) count = false;
    const size_t static_smem = (SMEM_TPB / 32) * (OUT_SLOTS * (TILE_BYTES + 16) + 4) + 64;
    const size_t need = scene_image_bytes(sc.ns, sc.nt, sc.lni, isect == RT_INTERSECT_BVH);
    // Stage the scene in shared memory when one 1024-thread CTA per SM fits with it (scenes up to ~200 KB); larger
    // scenes are read through L1/L2 (measured on the C5 sweep, profiles/r1_c5_sweep.log)
    if (info) info->counts_done = true;
    const bool smem = !count ? (need + static_smem + 1024 <= (size_t)smem_optin)
                             : ((need + static_smem + 1024) * 3 <= (size_t)smem_optin);
    // The output stage and the completion counters cost ~0.03 ns per pixel (C3: +0.2 ms of 38.0; C2, 1 spp: +0.07 of 0.24);
    // the copy they let the owner overlap costs 0.06 ns per pixel.  On for frames shared between ranks and for frames the
    // caller streams to the host; a frame that stays on one device keeps round 1's byte stores (profiles/r2_notes.md).
    // The same for the resumable form: rt_render_samples_multi's shared frames stage, rt_render_samples' bands do not.
    const bool stage = !count && (pr.tile_ranks > 1 || pr.stage_hint) && pr.done != nullptr;
    int threads = THREADS;
    KernelFn fn;
    if (resume) fn = isect == RT_INTERSECT_BRUTE ? (smem ? pick_resume<RT_INTERSECT_BRUTE, true>(stage, &threads) : pick_resume<RT_INTERSECT_BRUTE, false>(stage, &threads))
                                                 : (smem ? pick_resume<RT_INTERSECT_BVH, true>(stage, &threads) : pick_resume<RT_INTERSECT_BVH, false>(stage, &threads));
    else if (bands) fn = isect == RT_INTERSECT_BRUTE ? (smem ? pick_bands<RT_INTERSECT_BRUTE, true>(stage, &threads) : pick_bands<RT_INTERSECT_BRUTE, false>(stage, &threads))
                                                     : (smem ? pick_bands<RT_INTERSECT_BVH, true>(stage, &threads) : pick_bands<RT_INTERSECT_BVH, false>(stage, &threads));
    else if (isect == RT_INTERSECT_BRUTE) fn = smem ? pick_lanes<RT_INTERSECT_BRUTE, true>(count, stage, &threads) : pick_lanes<RT_INTERSECT_BRUTE, false>(count, stage, &threads);
    else fn = smem ? pick_lanes<RT_INTERSECT_BVH, true>(count, stage, &threads) : pick_lanes<RT_INTERSECT_BVH, false>(count, stage, &threads);
    const size_t dyn = smem ? need : 0;
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
    if (e != cudaSuccess) return e;
    int per_sm = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, threads, dyn);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    const uint64_t total_tiles = (uint64_t)pr.tiles_x * pr.tiles_y;
    const uint64_t my_tiles = (total_tiles + pr.tile_ranks - 1) / pr.tile_ranks;
    const uint64_t want_ctas = (my_tiles + (threads / 32) - 1) / (threads / 32);
    uint64_t grid = (uint64_t)sm_count * per_sm;
    if (grid > want_ctas) grid = want_ctas;
    if (grid < 1) grid = 1;
    DevParams prm = pr;
    if (!stage && !count) {  // without the stage every pixel would pay a system-scope release of its own (the
                             // instrumented kernel does: it is not a timed path)
        prm.done = nullptr;
        if (info) info->counts_done = false;
    }
    prm.my_tickets = (uint32_t)my_tiles;
    if (pr.pixel_list) {  // second pass over a pixel list: pixel tickets only
        const uint64_t warps = ((uint64_t)pr.list_count + 31) / 32;
        grid = std::max<uint64_t>(1, std::min<uint64_t>(grid, (warps + (threads / 32) - 1) / (threads / 32)));
    }
    // the tail: the last kTailPermille / 1000 of the tickets (at least two tiles per warp-slot of the grid would be
    // pointless to split further: small launches are all tail)
    uint64_t tail = my_tiles * kTailPermille / 1000;
    if (my_tiles <= grid * (uint64_t)(threads / 32)) tail = my_tiles;  // fewer tiles than warps: pixel tickets only
    prm.tail_first = (uint32_t)(my_tiles - std::min<uint64_t>(tail, my_tiles));
    if (pr.pixel_list) prm.tail_first = 0;
    fn<<<(unsigned)grid, threads, dyn, stream>>>(sc, cam, prm);
    if (info) {
        info->grid = (unsigned)grid;
        info->threads = threads;
        info->dyn_smem = dyn;
        info->ctas_per_sm = per_sm;
        info->scene_in_smem = smem;
    }
    return cudaGetLastError();
}

cudaError_t launch_wait_slab(const unsigned long long* done, unsigned long long target, unsigned int* timeout_flag,
                             cudaStream_t stream) {
    wait_slab_kernel<<<1, 1, 0, stream>>>(done, target, timeout_flag, (unsigned long long)test_hooks().wait_timeout_ms * 1000000ull);
    return cudaGetLastError();
}

cudaError_t launch_wait_all_slabs(const unsigned long long* done, unsigned long long seq, uint32_t slabs, uint32_t tile_rows,
                                  uint32_t rows, uint32_t width, unsigned int* timeout_flag, cudaStream_t stream) {
    wait_all_slabs_kernel<<<1, MAX_SLABS, 0, stream>>>(done, seq, slabs, tile_rows, rows, width, timeout_flag,
                                                       (unsigned long long)test_hooks().wait_timeout_ms * 1000000ull);
    return cudaGetLastError();
}

cudaError_t launch_set_u64(unsigned long long* p, unsigned long long v, cudaStream_t stream) {
    set_u64_kernel<<<1, 1, 0, stream>>>(p, v);
    return cudaGetLastError();
}

cudaError_t launch_add_counts(unsigned long long* done, const unsigned long long* add, int n, cudaStream_t stream) {
    add_counts_kernel<<<1, MAX_SLABS, 0, stream>>>(done, add, n);
    return cudaGetLastError();
}

cudaError_t launch_accum_linear(const void* state, float* out, unsigned long long pixels, uint32_t samples, int sm_count,
                                cudaStream_t stream) {
    const unsigned long long blocks = std::min<unsigned long long>((pixels + 255) / 256, (unsigned long long)sm_count * 8);
    accum_linear_kernel<<<(unsigned)std::max<unsigned long long>(1, blocks), 256, 0, stream>>>(
        static_cast<const uint4*>(state), out, pixels, (float)samples);
    return cudaGetLastError();
}

cudaError_t launch_fp32_peak(float* scratch, int sm_count, int iters, cudaStream_t stream) {
    fp32_peak_kernel<<<sm_count * 8, 256, 0, stream>>>(scratch, iters, 0.0f);
    return cudaGetLastError();
}

}  // namespace rtb
