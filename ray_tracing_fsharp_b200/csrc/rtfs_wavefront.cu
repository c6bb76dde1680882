// rtfs_wavefront.cu — the wavefront (ray-queue) variant of the render path, RT_MODE_WAVEFRONT.
//
// Same device functions as the megakernel (rtfs_core.cuh), different schedule: path state lives in HBM, and
// every bounce is a pair of launches over the queue of live paths,
//     extend  : Scene.hitObject for every live path              -> hit record (t, primitive)
//     shade   : Hittable.Reflection; finished paths add their Pixel to the integer accumulators
//               (PixelStats.add) with global atomics, survivors are appended to the next queue
//               (warp-aggregated compaction),
// after a `generate` launch that writes the camera rays of a batch (Scene.traceOnce's ray generation).
// It exists because the north star asks for the megakernel-versus-wavefront choice to be made on ncu
// counters (warp execution efficiency, FP32 pipe utilisation, L2 / HBM bytes per ray): DESIGN.md has the
// numbers.  Results are bit-identical to the megakernel's (same RNG keys, same integer sums).
// Single device only.
#include "rtfs_device.h"

#include <cstring>
#include <memory>

namespace rtfs {
namespace {

constexpr int kWfThreads = 256;

struct WfState {
    float4 *s0;        // o.xyz, d.x
    float4 *s1;        // d.y, d.z, colour (bits), last primitive (bits)
    uint4 *s2;         // row << 16 | col, sample, bounces, accumulator set (probe: 0 = first firstTrial+1 samples, 1 = the rest)
    uint2 *hit;        // t (bits), primitive
    uint32_t *queue_a; // live slots (ping)
    uint32_t *queue_b; // live slots (pong)
    uint32_t *counts;  // [0]: live in queue_a, [1]: live in queue_b
    size_t capacity = 0;
    void *block = nullptr;
};

struct WfParams {
    SceneGlobal g;
    DevCamera cam;
    uint32_t k0, k1;
    int32_t first_trial, n_probe, sample_begin;
    int32_t probe;           // 1: paths of the probe phase (all pixels x n_probe samples), 0: main phase over the list
    uint32_t n_list;         // main phase: number of flagged pixels
    const uint32_t *list;    // main phase: flagged pixel ids
    unsigned long long first_path; // index of the batch's first path in the phase's path numbering
    uint32_t n_batch;
    int32_t *stats_a, *stats_b; // accumulators (stats_b only in the probe phase)
    WfState st;
    const uint32_t *queue_in;
    uint32_t *queue_out;
    const uint32_t *count_in; // nullptr: the queue is the identity over [0, n_batch)
    uint32_t *count_out;
    unsigned long long *counters;
    uint32_t s_nodes, s_spheres, s_mats;
};

template <bool SMEM>
__device__ __forceinline__ SceneAccess<SMEM> wf_stage(const WfParams &p) {
    SceneAccess<SMEM> sc;
    sc.g = p.g;
    const uint32_t window = uint32_t(__cvta_generic_to_shared(rtfs_smem));
    sc.s_nodes = window + 16u * p.s_nodes;
    sc.s_spheres = window + 16u * p.s_spheres;
    sc.s_mats = window + 16u * p.s_mats;
    if (SMEM) sc.stage_tree(p.s_nodes, p.s_spheres, p.s_mats);
    return sc;
}

// Scene.traceOnce's ray generation (Scene.fs:129-144) for one batch of paths
__global__ void __launch_bounds__(kWfThreads) wf_generate(const WfParams p) {
    uint32_t made = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < p.n_batch; i += gridDim.x * blockDim.x) {
        unsigned long long path = p.first_path + i;
        uint32_t rc, sample, set = 0;
        bool valid = true;
        if (p.probe) { // path -> (sample, pixel): consecutive threads are consecutive pixels of one sample
            unsigned long long n_pix = (unsigned long long)p.cam.rows * p.cam.cols;
            uint32_t smp = uint32_t(path / n_pix), pix = uint32_t(path - (unsigned long long)smp * n_pix);
            rc = ((pix / p.cam.cols) << 16) | (pix % p.cam.cols);
            sample = smp;
            set = int(smp) > p.first_trial ? 1u : 0u;
        } else {
            uint32_t smp = uint32_t(path / p.n_list), e = uint32_t(path - (unsigned long long)smp * p.n_list);
            uint32_t pix = p.list[e];
            rc = ((pix / p.cam.cols) << 16) | (pix % p.cam.cols);
            sample = uint32_t(p.sample_begin) + smp;
        }
        PathState ps;
        valid = path_begin(ps, p.cam, p.k0, p.k1, int(rc >> 16), int(rc & 0xffff), sample);
        ++made;
        p.st.s0[i] = make_float4(ps.o.x, ps.o.y, ps.o.z, ps.d.x);
        p.st.s1[i] = make_float4(ps.d.y, ps.d.z, __uint_as_float(ps.colour), __int_as_float(valid ? kNoPrim : -2));
        p.st.s2[i] = make_uint4(rc, sample, 0u, set);
    }
    for (int off = 16; off > 0; off >>= 1) made += __shfl_down_sync(0xffffffffu, made, off);
    if ((threadIdx.x & 31) == 0 && made) atomicAdd(p.counters + CN_PATHS, (unsigned long long)made);
}

// Scene.hitObject (Scene.fs:62-91) for every live path
template <bool SMEM>
__global__ void __launch_bounds__(kWfThreads) wf_extend(const WfParams p) {
    const SceneAccess<SMEM> sc = wf_stage<SMEM>(p);
    const uint32_t n = p.count_in ? *p.count_in : p.n_batch;
    uint32_t rays = 0;
    TraversalCounters cn{0, 0};
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        uint32_t slot = p.count_in ? p.queue_in[i] : i;
        float4 a = p.st.s0[slot], b = p.st.s1[slot];
        int last = __float_as_int(b.w);
        if (last == -2) { // Ray.make' failed at generation: the reference throws; treated as a miss
            p.st.hit[slot] = make_uint2(0u, uint32_t(kNoPrim));
            continue;
        }
        Hit h = closest_hit<SMEM, false>(sc, f3(a.x, a.y, a.z), f3(a.w, b.x, b.y), last, cn, 1u << (threadIdx.x & 31));
        ++rays;
        p.st.hit[slot] = make_uint2(__float_as_uint(h.t), uint32_t(h.prim));
    }
    for (int off = 16; off > 0; off >>= 1) rays += __shfl_down_sync(0xffffffffu, rays, off);
    if ((threadIdx.x & 31) == 0 && rays) atomicAdd(p.counters + CN_RAYS, (unsigned long long)rays);
}

// Hittable.Reflection + the bookkeeping of Scene.traceRay (Scene.fs:93-114) for every live path
template <bool SMEM>
__global__ void __launch_bounds__(kWfThreads) wf_shade(const WfParams p) {
    const SceneAccess<SMEM> sc = wf_stage<SMEM>(p);
    const uint32_t n = p.count_in ? *p.count_in : p.n_batch;
    const uint32_t n_round = (n + 31u) & ~31u; // whole warps iterate together (ballot below)
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_round; i += gridDim.x * blockDim.x) {
        bool survives = false;
        uint32_t slot = 0;
        if (i < n) {
            slot = p.count_in ? p.queue_in[i] : i;
            float4 a = p.st.s0[slot], b = p.st.s1[slot];
            uint4 m = p.st.s2[slot];
            uint2 hr = p.st.hit[slot];
            int prim = int(hr.y);
            float3 o = f3(a.x, a.y, a.z), d = f3(a.w, b.x, b.y);
            uint32_t colour = __float_as_uint(b.z);
            int last = __float_as_int(b.w);
            uint32_t result = kBlack;
            if (prim != kNoPrim) {
                const int row = int(m.x >> 16), col = int(m.x & 0xffff);
                CounterRng rng{p.k0, p.k1, uint32_t(row * p.cam.cols + col), m.y, m.z + 1u, 0u};
                float3 strike = fma3(__uint_as_float(hr.x), d, o);
                ScatterResult r = scatter(sc, prim, last, o, d, strike, colour, rng, (bool *)nullptr);
                if (r == SCATTER_ABSORBED) {
                    result = colour;
                } else if (r == SCATTER_ERROR) {
                    result = kBlack;
                } else if (int(m.z) + 1 > p.cam.depth) { // while bounces <= maxCount, Scene.fs:98; not done => HotPink :114
                    result = kHotPink;
                } else {
                    survives = true;
                    p.st.s0[slot] = make_float4(o.x, o.y, o.z, d.x);
                    p.st.s1[slot] = make_float4(d.y, d.z, __uint_as_float(colour), __int_as_float(prim));
                    p.st.s2[slot] = make_uint4(m.x, m.y, m.z + 1u, m.w);
                }
            }
            if (!survives) { // PixelStats.add, Pixel.fs:87-95
                int32_t *st = (m.w ? p.stats_b : p.stats_a) + 4 * size_t((m.x >> 16) * uint32_t(p.cam.cols) + (m.x & 0xffff));
                atomicAdd(st + 0, int((result >> 16) & 255u));
                atomicAdd(st + 1, int((result >> 8) & 255u));
                atomicAdd(st + 2, int(result & 255u));
                atomicAdd(st + 3, 1);
            }
        }
        unsigned live = __ballot_sync(0xffffffffu, survives);
        if (live) {
            uint32_t base = 0;
            if ((threadIdx.x & 31) == 0) base = atomicAdd(p.count_out, uint32_t(__popc(live)));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (survives) p.queue_out[base + __popc(live & ((1u << (threadIdx.x & 31)) - 1u))] = slot;
        }
    }
}

int wf_reserve(DeviceWorkspace *ws, WfState &st, size_t capacity) {
    // the state block is not pooled: the wavefront mode is a measurement variant, not the default path
    (void)ws;
    const size_t per_path = sizeof(float4) * 2 + sizeof(uint4) + sizeof(uint2) + sizeof(uint32_t) * 2;
    RT_CUDA(cudaMalloc(&st.block, capacity * per_path + 256));
    uint8_t *p = static_cast<uint8_t *>(st.block);
    st.s0 = reinterpret_cast<float4 *>(p); p += capacity * sizeof(float4);
    st.s1 = reinterpret_cast<float4 *>(p); p += capacity * sizeof(float4);
    st.s2 = reinterpret_cast<uint4 *>(p); p += capacity * sizeof(uint4);
    st.hit = reinterpret_cast<uint2 *>(p); p += capacity * sizeof(uint2);
    st.queue_a = reinterpret_cast<uint32_t *>(p); p += capacity * sizeof(uint32_t);
    st.queue_b = reinterpret_cast<uint32_t *>(p); p += capacity * sizeof(uint32_t);
    st.counts = reinterpret_cast<uint32_t *>(p);
    st.capacity = capacity;
    return RT_OK;
}

} // namespace

int render_wavefront(RtScene *scene, const RtCamera *camera, int32_t max_w, int32_t max_h, const RtRenderOpts *opts, uint8_t *rgb_out,
                     int32_t *sums_out, RtStats *stats) {
    auto *ds = static_cast<DeviceScene *>(scene->dev);
    DeviceWorkspace *ws = ds->ws;
    RT_CUDA(cudaSetDevice(ds->device));
    cudaStream_t st = ws->stream;
    const size_t n_pixels = size_t(2 * max_w + 1) * size_t(2 * max_h + 1);
    int rc = ensure_frame_buffers(ws, n_pixels);
    if (rc == RT_OK) rc = ensure_list(ws, n_pixels);
    if (rc == RT_OK) rc = ensure_probe_sums(ws, n_pixels);
    if (rc != RT_OK) return rc;
    FrameParams fp;
    fill_frame(fp, ds, *camera, max_w, max_h, *opts, 0, 1);
    fp.stats = ws->d_stats;
    fp.flags = ws->d_flags;

    const size_t batch = size_t(8) << 20; // paths in flight
    WfState wf;
    if ((rc = wf_reserve(ws, wf, batch)) != RT_OK) return rc;
    const std::unique_ptr<void, cudaError_t (*)(void *)> free_state(wf.block, cudaFree);

    // shared-memory staging plan (persistent grid-stride blocks)
    const bool no_smem = (opts->flags & RT_FLAG_NO_SMEM) != 0;
    const size_t nodes_q = size_t(ds->g.n_nodes) * kStagedNodeQuads, sph_q = size_t(ds->g.n_bounded), mat_q = size_t(ds->g.n_bounded + ds->g.n_unbounded) * 2;
    const size_t scene_bytes = (nodes_q + sph_q + mat_q) * 16;
    const bool smem = !no_smem && ds->g.n_bounded > 0 && scene_bytes * 2 + 2048 <= ws->smem_optin; // two blocks per SM
    const size_t smem_bytes = smem ? scene_bytes : 0;
    auto k_extend = smem ? wf_extend<true> : wf_extend<false>;
    auto k_shade = smem ? wf_shade<true> : wf_shade<false>;
    cudaFuncSetAttribute((const void *)k_extend, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem_bytes));
    cudaFuncSetAttribute((const void *)k_shade, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem_bytes));
    int per_sm_e = 1, per_sm_s = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_e, (const void *)k_extend, kWfThreads, smem_bytes);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_s, (const void *)k_shade, kWfThreads, smem_bytes);
    const int grid_e = std::max(1, per_sm_e) * ws->sm_count, grid_s = std::max(1, per_sm_s) * ws->sm_count;

    int launches = 0;
    uint32_t *h_count = reinterpret_cast<uint32_t *>(ws->h_counters + CN_SLOTS - 1); // pinned scratch word
    WfParams p{};
    p.g = ds->g;
    p.cam = fp.cam;
    p.k0 = fp.k0;
    p.k1 = fp.k1;
    p.first_trial = fp.first_trial;
    p.n_probe = fp.n_probe;
    p.sample_begin = fp.sample_begin;
    p.st = wf;
    p.counters = ws->d_counters;
    p.s_nodes = 0;
    p.s_spheres = uint32_t(nodes_q);
    p.s_mats = uint32_t(nodes_q + sph_q);
    p.stats_a = ws->d_stats;
    p.stats_b = ws->d_stats_b;

    cudaError_t err = cudaSuccess;
    auto run_phase = [&](bool probe, unsigned long long n_paths, uint32_t n_list) -> int {
        for (unsigned long long first = 0; first < n_paths; first += batch) {
            p.probe = probe ? 1 : 0;
            p.n_list = n_list;
            p.list = ws->d_list;
            p.first_path = first;
            p.n_batch = uint32_t(std::min<unsigned long long>(batch, n_paths - first));
            int gen_grid = int(std::min<size_t>((p.n_batch + kWfThreads - 1) / kWfThreads, size_t(ws->sm_count) * 16));
            wf_generate<<<gen_grid, kWfThreads, 0, st>>>(p);
            ++launches;
            bool a_is_in = true;
            uint32_t live = p.n_batch;
            for (int bounce = 0; bounce <= fp.cam.depth && live > 0; ++bounce) {
                p.count_in = bounce == 0 ? nullptr : (a_is_in ? wf.counts : wf.counts + 1);
                p.queue_in = a_is_in ? wf.queue_a : wf.queue_b;
                p.queue_out = a_is_in ? wf.queue_b : wf.queue_a;
                p.count_out = a_is_in ? wf.counts + 1 : wf.counts;
                if ((err = cudaMemsetAsync(p.count_out, 0, sizeof(uint32_t), st)) != cudaSuccess) return RT_ERR_CUDA;
                int ge = int(std::min<size_t>((live + kWfThreads - 1) / kWfThreads, size_t(grid_e)));
                int gs = int(std::min<size_t>((live + kWfThreads - 1) / kWfThreads, size_t(grid_s)));
                k_extend<<<ge, kWfThreads, smem_bytes, st>>>(p);
                k_shade<<<gs, kWfThreads, smem_bytes, st>>>(p);
                launches += 2;
                if ((err = cudaMemcpyAsync(h_count, p.count_out, sizeof(uint32_t), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return RT_ERR_CUDA;
                if ((err = cudaStreamSynchronize(st)) != cudaSuccess) return RT_ERR_CUDA;
                live = *h_count;
                a_is_in = !a_is_in;
            }
        }
        return RT_OK;
    };
    auto fail_cuda = [&](const char *what) {
        return fail(RT_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(err != cudaSuccess ? err : cudaGetLastError()));
    };

    FrameEvents &ev = ws->ev;
    ev.record(FrameEvents::BEGIN, st);
    cudaMemsetAsync(ws->d_counters, 0, CN_SLOTS * sizeof(unsigned long long), st);
    cudaMemsetAsync(ws->d_stats, 0, n_pixels * 4 * sizeof(int32_t), st);
    cudaMemsetAsync(ws->d_stats_b, 0, n_pixels * 4 * sizeof(int32_t), st);
    ev.record(FrameEvents::ZEROED, st);
    if (fp.adaptive) {
        if (run_phase(true, (unsigned long long)n_pixels * fp.n_probe, 0) != RT_OK) return fail_cuda("wavefront probe phase");
        launch_probe_flags(fp, ws->d_stats_b, fp.sample_end > fp.sample_begin, st, &launches);
    } else {
        cudaMemsetAsync(ws->d_flags, 1, n_pixels, st);
    }
    // the flagged-pixel list (same kernel as the megakernel path uses)
    launch_compact(ds, fp, single_flags(ws->d_flags), ws->d_list, st, &launches);
    cudaMemcpyAsync(ws->h_counters, ws->d_counters, CN_SLOTS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st);
    if ((err = cudaStreamSynchronize(st)) != cudaSuccess) return fail_cuda("wavefront compaction");
    const unsigned long long n_list = ws->h_counters[CN_LIST];
    const int n_main = fp.sample_end - fp.sample_begin;
    if (n_main > 0 && n_list > 0)
        if (run_phase(false, n_list * (unsigned long long)n_main, uint32_t(n_list)) != RT_OK) return fail_cuda("wavefront main phase");
    ev.record(FrameEvents::TRACED, st);
    if ((rc = launch_finalize(ws->d_stats, n_pixels, opts->gamma, ws->d_rgb, st, &launches)) != RT_OK) return rc;
    if ((rc = frame_finish(ds, fp, ws->d_rgb, rgb_out, sums_out, st, ev)) != RT_OK) return rc;
    RT_CUDA(cudaStreamSynchronize(st));
    if (stats) { // no main_ms: the main phase is many launches with host synchronisations between them
        read_stats(ds, n_pixels, fp.adaptive != 0, launches, nullptr, stats);
        stats->kernel_ms = ev.ms(FrameEvents::ZEROED, FrameEvents::TRACED);
        stats->total_ms = ev.ms(FrameEvents::BEGIN, FrameEvents::END);
    }
    return RT_OK;
}

} // namespace rtfs
