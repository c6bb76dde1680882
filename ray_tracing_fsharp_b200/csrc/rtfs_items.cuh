// rtfs_items.cuh — the item loop of the lockstep render kernels, shared by render_kernel (rtfs_device.cu: one frame) and
// render_views_kernel (rtfs_views.cu: several views of one scene stacked as one tall frame).  The two differ only in how a
// lane finds the pixel, camera and RNG key of a path; that is the `Pixels` parameter of render_items (below).
#pragma once
#include "rtfs_device.h"

#include <type_traits>

namespace rtfs {

template <int SMEM>
__device__ __forceinline__ SceneAccess<SMEM> stage_scene(const FrameParams &fp) {
    SceneAccess<SMEM> sc;
    sc.g = fp.g;
    const uint32_t window = uint32_t(__cvta_generic_to_shared(rtfs_smem));
    sc.s_nodes = window + 16u * fp.s_nodes;
    sc.s_spheres = window + 16u * fp.s_spheres;
    sc.s_mats = window + 16u * fp.s_mats;
    if (SMEM) {
        sc.stage_tree(fp.s_nodes, fp.s_spheres, fp.s_mats);
    }
    return sc;
}

// per-warp scratch in shared memory: item slots (one being issued, the others with their last paths still in flight).
// 400 bytes each: for a scene read from global memory what shared memory the slots take is L1 the walk does not get.
// A pixel's red and green sums share a word (16 bits each): a chunk is at most kMaxChunkSamples = 256 samples, 256 x 255 < 2^16.
struct ItemSlot {
    int cursor;    // next path of the item's pool
    int j_begin;   // first local sample index of the item's chunk
    int j_len;     // samples in the chunk (also what the flush adds to the pixels' count field)
    int to_b;      // probe: the chunk belongs to the second accumulator set
    int pix[32];   // each of the 32 pixels as the kernel's Pixels::pack encodes it, -1: none
    unsigned acc_rg[32]; // sum of red | sum of green << 16
    unsigned acc_b[32];  // sum of blue
};
// The slot of the kernels that also sum r^2 + g^2 + b^2 per pixel (RT_FLAG_NOISE): one more word per lane, 528 bytes.  A chunk's
// word stays below 3 x 255^2 x 256 < 2^26.
struct NoiseItemSlot : ItemSlot {
    unsigned acc_q[32]; // sum of r^2 + g^2 + b^2
};
static_assert(sizeof(ItemSlot) == 400 && sizeof(NoiseItemSlot) == 528, "item slot sizes");
static_assert(sizeof(ItemSlot) % 16 == 0 && sizeof(NoiseItemSlot) % 16 == 0, "ItemSlot must be a multiple of 16 bytes");
constexpr size_t warp_scratch_bytes(bool staged, bool noise = false) { // per warp
    return size_t(item_slots(staged)) * (noise ? sizeof(NoiseItemSlot) : sizeof(ItemSlot));
}

__device__ __forceinline__ void flush_counters(unsigned long long *counters, uint32_t paths, uint32_t rays, TraversalCounters cn, bool count) {
    for (int off = 16; off > 0; off >>= 1) {
        paths += __shfl_down_sync(0xffffffffu, paths, off);
        rays += __shfl_down_sync(0xffffffffu, rays, off);
        if (count) {
            cn.box_tests += __shfl_down_sync(0xffffffffu, cn.box_tests, off);
            cn.prim_tests += __shfl_down_sync(0xffffffffu, cn.prim_tests, off);
        }
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(counters + CN_PATHS, (unsigned long long)paths);
        atomicAdd(counters + CN_RAYS, (unsigned long long)rays);
        if (count) {
            atomicAdd(counters + CN_BOX, (unsigned long long)cn.box_tests);
            atomicAdd(counters + CN_PRIM, (unsigned long long)cn.prim_tests);
        }
    }
}

// The body of the lockstep render kernels.  Persistent warps pull work items from a global cursor; an item is a unit of 32
// pixels times a chunk of sample indices.  Inside an item the 32 lanes pull (pixel, sample) paths from a warp-local pool,
// so every lane traces until the pool is dry (path regeneration); per-sample results are added to the pixels'
// integer accumulators in shared memory (PixelStats.add, Pixel.fs:87-95) and flushed with one RED per channel.
//   PROBE = true : unit = one 8x4 tile owned by this rank; samples = the 2*firstTrial+1 probe samples of
//                  renderPixel (Scene.fs:172-182): those up to firstTrial go to `stats`, the rest to `stats_b`
//                  (no chunk straddles the two), so that probe_flags_kernel can compare the two means.
//   PROBE = false: unit = 32 consecutive entries of the flagged-pixel list; samples = this rank's share of the
//                  remaining sample indices (Scene.fs:191-192).
// A warp issues one instruction every ~7.6 cycles whatever the load, so the kernel ends one whole item after the
// work runs out: hence chunks of decreasing length, the last ones a single sample (see build_chunks).
//   NOISE = true : also sum r^2 + g^2 + b^2 of every finished path per pixel (one more shared word per slot lane, flushed
//                  with one 64-bit RED per pixel into fp.sq), for the noise estimate of progressive frames (rt_frame_noise).
//                  The probe adds to the same sum whichever accumulator set its chunk belongs to.
// Pixels maps the frame's flat pixel ids (fp.cam.rows x fp.cam.cols) to what a slot holds and back, and starts a path:
//   Path                                the path state (PathStateT of the kernel's generator);
//   int pack(int pixel)                 the slot's encoding of a pixel (>= 0);
//   size_t index(int packed)            the flat pixel id again (the sums' index);
//   bool begin(Path &, int packed, uint32_t sample)   path_begin with the pixel's camera, key and coordinates.
template <bool PROBE, int SMEM, bool COUNT, bool SSTACK, bool WIDE, bool NOISE, class Pixels>
__device__ __forceinline__ void render_items(const FrameParams &fp, const Pixels &px) {
    using Slot = typename std::conditional<NOISE, NoiseItemSlot, ItemSlot>::type;
    const SceneAccess<SMEM> sc = stage_scene<SMEM>(fp);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    typename std::conditional<SSTACK, SharedStack, LocalStack>::type stack;
    if constexpr (SSTACK) {
        stack.base = uint32_t(__cvta_generic_to_shared(rtfs_smem)) + 16u * fp.s_stack + 4u * threadIdx.x;
        stack.stride = 4u * blockDim.x; // words of one stack level (wide walk: two levels per entry)
        stack.levels = fp.stack_levels;
    }
    constexpr int kSlots = SMEM ? kItemSlots : kGlobalItemSlots;
    Slot *const slots = reinterpret_cast<Slot *>(rtfs_smem + fp.s_warp) + warp * kSlots; // this warp's item slots
    unsigned long long *work = fp.counters + (PROBE ? CN_WORK_PROBE : CN_WORK_MAIN);
    uint32_t n_paths = 0, n_rays = 0;
    TraversalCounters cn{0, 0};

    const unsigned n_list = PROBE ? 0u : (unsigned)fp.counters[CN_LIST];
    const unsigned n_units = PROBE ? unsigned((fp.tiles_x * fp.tiles_y - fp.rank + fp.world - 1) / fp.world) : (n_list + 31u) / 32u;
    const unsigned long long n_items = (unsigned long long)n_units * (unsigned long long)fp.n_chunks;

    // Loads work item `item` into a slot: chunk-major numbering; this lane's pixel; the pool.  Returns the pool size.
    auto load_item = [&](Slot *sl, unsigned long long item, int &n_entries) -> int {
        const int k = int(item / n_units);
        const unsigned unit = unsigned(item - (unsigned long long)k * n_units);
        const int j_begin = int(fp.chunk_begin[k]), j_len = int(fp.chunk_len[k]);
        int my_pixel = -1;
        n_entries = 32;
        if constexpr (PROBE) {
            int tile = int(unit) * fp.world + fp.rank;
            int ty = tile / fp.tiles_x, tx = tile - ty * fp.tiles_x;
            int r = ty * kTileH + (lane >> 3), c = tx * kTileW + (lane & 7);
            if (r < fp.cam.rows && c < fp.cam.cols) my_pixel = r * fp.cam.cols + c;
        } else {
            unsigned e = unit * 32u + lane;
            if (e < n_list) my_pixel = int(fp.list[e]);
            n_entries = int(min(32u, n_list - unit * 32u));
        }
        sl->acc_rg[lane] = 0u; sl->acc_b[lane] = 0u;
        if constexpr (NOISE) sl->acc_q[lane] = 0u;
        sl->pix[lane] = my_pixel < 0 ? -1 : px.pack(my_pixel);
        if (lane == 0) {
            sl->cursor = 0;
            sl->j_begin = j_begin;
            sl->j_len = j_len;
            sl->to_b = (PROBE && j_begin > fp.first_trial) ? 1 : 0;
        }
        __syncwarp();
        return n_entries * j_len;
    };
    // Retires a slot whose paths have all finished: one RED per channel and pixel (PixelStats.add, Pixel.fs:87-95)
    auto flush_item = [&](Slot *sl) {
        __syncwarp();
        const int rc = sl->pix[lane];
        if (rc >= 0) {
            const size_t p = px.index(rc);
            int *st = (sl->to_b ? fp.stats_b : fp.stats) + 4 * p;
            const unsigned rg = sl->acc_rg[lane];
            atomicAdd(st + 0, int(rg & 0xffffu));
            atomicAdd(st + 1, int(rg >> 16));
            atomicAdd(st + 2, int(sl->acc_b[lane]));
            atomicAdd(st + 3, sl->j_len);
            if constexpr (NOISE) atomicAdd(fp.sq + p, (unsigned long long)sl->acc_q[lane]);
        }
        __syncwarp();
    };
    auto fetch_item = [&]() -> unsigned long long { // lane 0 pulls the next item number; consumed (shuffled) later
        return lane == 0 ? atomicAdd(work, 1ull) : 0ull;
    };

    unsigned long long item = __shfl_sync(0xffffffffu, fetch_item(), 0);
    if (threadIdx.x == 0 && item < n_items) atomicAdd(fp.counters + CN_BUSY_BLOCKS, 1ull); // blocks that found work: the resident ones
    if (item < n_items) {
        // kItemSlots slots per warp: lanes pull paths from slot `cur`; when its pool is dry the next item is loaded into a
        // free slot straight away, so lanes do not idle while the last paths of an item complete.  A slot is free once
        // its in-flight paths have finished and it has been flushed; with long, uneven paths (big scenes) several older
        // items can have stragglers at once, hence more than two slots.  Only the warp's final items drain.
        int cur = 0;
        unsigned holds = 1u; // slots that hold an item not yet flushed
        bool finishing = false;
        int n_entries;
        int pool = load_item(&slots[0], item, n_entries);
        int j_begin = slots[0].j_begin;
        unsigned long long prefetched = fetch_item();
        typename Pixels::Path ps;
        bool active = false, dry = false;
        int lane_slot = 0, my = 0; // my: slot index of this lane's path; lane_slot: its pixel within the item
        for (;;) {
            if (!active && !dry) {
                Slot *sl = &slots[cur];
                int q = atomicAdd(&sl->cursor, 1);
                if (q >= pool) {
                    dry = true;
                } else {
                    int j = (n_entries == 32) ? (q >> 5) : (q / n_entries);
                    lane_slot = q - j * n_entries;
                    my = cur;
                    int rc = sl->pix[lane_slot]; // packed pixel, or -1 where the tile overhangs the image edge
                    if (rc >= 0) {
                        uint32_t sample = uint32_t(PROBE ? j_begin + j : fp.sample_begin + fp.rank + (j_begin + j) * fp.world);
                        ++n_paths;
                        active = px.begin(ps, rc, sample); // false: Ray.make' failed (the reference throws)
                        if (!active) atomicAdd(fp.counters + CN_DEGENERATE, 1ull);
                    }
                }
            }
            // Every lane votes, every iteration: this is where the warp reconverges (lanes that regenerate a path and lanes
            // that do not would otherwise drift apart for good and the traversal would run at a fraction of the warp width).
            if (__any_sync(0xffffffffu, dry)) {
                // the current pool is exhausted: retire the older slots whose paths have all finished, then move on
                if (!finishing) {
                    int free_slot = -1;
#pragma unroll
                    for (int sidx = 0; sidx < kSlots; ++sidx) {
                        if (sidx == cur) continue;
                        if ((holds >> sidx) & 1u) {
                            if (__any_sync(0xffffffffu, active && my == sidx)) continue; // stragglers
                            flush_item(&slots[sidx]);
                            holds &= ~(1u << sidx);
                        }
                        if (free_slot < 0) free_slot = sidx;
                    }
                    if (free_slot >= 0) {
                        item = __shfl_sync(0xffffffffu, prefetched, 0);
                        if (item < n_items) {
                            Slot *next = &slots[free_slot];
                            pool = load_item(next, item, n_entries);
                            j_begin = next->j_begin;
                            prefetched = fetch_item();
                            cur = free_slot;
                            holds |= 1u << free_slot;
                            dry = false;
                        } else {
                            finishing = true;
                        }
                    }
                }
                if (finishing && !__any_sync(0xffffffffu, active)) break;
            }
            const unsigned tracing = __ballot_sync(0xffffffffu, active);
            if (active) {
                uint32_t result;
                ++n_rays;
                if (path_step<SMEM, COUNT, decltype(stack), WIDE>(ps, sc, fp.cam.depth, result, cn, tracing, stack)) {
                    RTFS_BOUNDS(my >= 0 && my < kSlots && lane_slot >= 0 && lane_slot < 32);
                    Slot *mine = &slots[my]; // PixelStats.add into the item's accumulators
                    atomicAdd(&mine->acc_rg[lane_slot], ((result >> 16) & 255u) | ((result << 8) & 0x00ff0000u));
                    atomicAdd(&mine->acc_b[lane_slot], result & 255u);
                    if constexpr (NOISE) {
                        const unsigned r = (result >> 16) & 255u, g = (result >> 8) & 255u, b = result & 255u;
                        atomicAdd(&mine->acc_q[lane_slot], r * r + g * g + b * b);
                    }
                    if (result & kDegenerate) atomicAdd(fp.counters + CN_DEGENERATE, 1ull);
                    active = false;
                }
            }
        }
        for (int sidx = 0; sidx < kSlots; ++sidx) // no path is in flight any more
            if ((holds >> sidx) & 1u) flush_item(&slots[sidx]);
    }
    flush_counters(fp.counters, n_paths, n_rays, cn, COUNT);
}

} // namespace rtfs
