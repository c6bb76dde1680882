// rtfs_frame.cu — progressive frames (rt_frame_*): rt_render's frame, cut into passes over windows of sample indices.
// The probe and the compaction run once, in the opener; every rt_frame_advance is one launch_samples per part over
// [samples_done, samples_done + k), i.e. the same render_kernel<PROBE = false> that rt_render's main
// phase launches, with the same chunking.  Sums are integers keyed by (seed, pixel, sample index), so a frame that has
// reached samples_done is bit for bit rt_render's frame at samples_per_pixel = samples_done (include/rtfs_b200.h).
// A frame opened with RT_FLAG_NOISE also holds per pixel the sum of squares Q (render_kernel<NOISE = true>), from which
// rt_frame_noise derives a per-pixel standard error and a summary over the flagged pixels, and with which a convergence rule
// (rt_frame_set_convergence) stops sampling each pixel once its estimate is within a tolerance.
// rt_frame_begin_views opens the same frame over rt_render_views' tall frame of a batch of views (its kernels are in
// rtfs_views.cu); the probe flags, the compaction, the checks and the output tail work per pixel and need no change for it,
// and rt_frame_view_noise reduces each view as rt_frame_noise reduces a frame of its own.  rt_multi_frame_begin_views splits
// that frame over an RtMulti: every part holds a copy of the table of view cameras and keys on its own device.
// rt_frame_begin_window opens it over a window of rt_render's frame (its kernels are in rtfs_window.cu): the frame's buffers,
// maps and counts are the window's, and every per-pixel kernel runs over the window unchanged.
// rt_frame_features and rt_frame_denoise (kernels in rtfs_denoise.cu) read the frame and keep buffers of their own.
// A frame records its scene's edit count: once rt_scene_update has changed the scene, the calls that would trace or read the
// scene refuse the frame, and the others keep working on what it holds.
// Every frame is split into parts (FramePart, below), one per device: rt_frame_begin* open one, and rt_multi_frame_begin
// one per device of an RtMulti.  Part r probes its tiles and traces its sample indices, and every part runs the same
// opener, pass and end of step.  The totals, the shared flags and everything that reads them live on the first device: the
// only part of a frame of one device traces into them directly, and over several devices the parts trace into buffers of
// their own that the exchange kernel (rtfs_multi.cu) sums into the totals.
// rt_frame_save writes a frame's totals, flags and counters into a snapshot, and rt_frame_resume / rt_multi_frame_resume
// open a frame from one on any device count: frame_alloc, then a restore in place of the probe (kernels in rtfs_snapshot.cu).
#include "rtfs_device.h"

#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstring>

using namespace rtfs;

namespace rtfs {

// rt_frame_noise's reduction: a fixed grid, every block a fixed contiguous range of pixels, every thread a fixed stride of
// it, then a fixed tree in shared memory, then one block over the partials in block order: no result depends on scheduling
// (no floating-point atomics), so the summary is bit-identical from call to call.
struct NoisePartial {
    unsigned long long pixels, above;
    double max_se, sum_se;
};
constexpr int kNoiseBlocks = 512, kNoiseThreads = 256;

__device__ __forceinline__ void noise_combine(NoisePartial &a, const NoisePartial &b) {
    a.pixels += b.pixels;
    a.above += b.above;
    a.max_se = fmax(a.max_se, b.max_se);
    a.sum_se += b.sum_se;
}

__device__ __forceinline__ void noise_block_reduce(NoisePartial acc, NoisePartial *out) {
    __shared__ NoisePartial part[kNoiseThreads];
    part[threadIdx.x] = acc;
    __syncthreads();
    for (int half = kNoiseThreads / 2; half > 0; half >>= 1) {
        if (int(threadIdx.x) < half) noise_combine(part[threadIdx.x], part[threadIdx.x + half]);
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = part[0];
}

// blockIdx.y is the view of a batch (rt_frame_view_noise: n_pixels is then one view's pixels, view v starts at v n_pixels, and
// its partials and summary at v (kNoiseBlocks + 1)): each view is reduced exactly as a frame of its own pixels would be.
__global__ void __launch_bounds__(kNoiseThreads) noise_kernel(const int4 *stats, const unsigned long long *sq, const uint8_t *flags, size_t n_pixels,
                                                              double tolerance, float *se, NoisePartial *partial) {
    const size_t per_block = (n_pixels + kNoiseBlocks - 1) / kNoiseBlocks, base = size_t(blockIdx.y) * n_pixels;
    const size_t begin = base + size_t(blockIdx.x) * per_block;
    const size_t end = size_t(blockIdx.x) * per_block + per_block < n_pixels ? begin + per_block : base + n_pixels;
    NoisePartial acc{0ull, 0ull, 0.0, 0.0};
    for (size_t p = begin + threadIdx.x; p < end; p += kNoiseThreads) {
        const int4 s = stats[p];
        const double e = pixel_standard_error(s.w, s.x, s.y, s.z, sq[p]);
        if (se) se[p] = float(e);
        if (flags[p]) {
            acc.pixels += 1;
            acc.above += e > tolerance ? 1 : 0;
            acc.max_se = fmax(acc.max_se, e);
            acc.sum_se += e;
        }
    }
    noise_block_reduce(acc, partial + size_t(blockIdx.y) * (kNoiseBlocks + 1) + blockIdx.x);
}

// one block per view (blockIdx.x) over that view's partials, in block order
__global__ void __launch_bounds__(kNoiseThreads) noise_summary_kernel(NoisePartial *partial) {
    partial += size_t(blockIdx.x) * (kNoiseBlocks + 1);
    NoisePartial acc{0ull, 0ull, 0.0, 0.0};
    for (int b = threadIdx.x; b < kNoiseBlocks; b += kNoiseThreads) noise_combine(acc, partial[b]);
    noise_block_reduce(acc, partial + kNoiseBlocks);
}

// The check of a convergence rule at a checkpoint: a pixel still being sampled whose E over the samples it holds is <= the
// tolerance stops there (its flag is cleared; the compaction that follows drops it from the list).  E is rt_frame_noise's,
// so `<=` is exactly the complement of its summary's `e > tolerance`.
__global__ void __launch_bounds__(256) converge_kernel(const int4 *stats, const unsigned long long *sq, uint8_t *flags, size_t n_pixels,
                                                       double tolerance) {
    const size_t p = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (p >= n_pixels || !flags[p]) return;
    const int4 s = stats[p];
    if (pixel_standard_error(s.w, s.x, s.y, s.z, sq[p]) <= tolerance) flags[p] = 0;
}

// One device's part of a frame: rank r of world traces the tiles t with t mod world == r in the probe and, in a pass over
// [s, s + k), the sample indices s + r + j world, into sums, Q and flags on its device, and compacts the frame's flags into
// a list and a counter block of its own.  The only part of a frame of one device traces into the frame's own sums, Q and
// flags; over several devices every part has its own.
struct FramePart {
    RtScene *scene = nullptr; // the rank's replica; its workspace's stream carries the rank's work
    FrameParams fp;
    int32_t *d_stats = nullptr;
    unsigned long long *d_sq = nullptr;
    uint8_t *d_flags = nullptr;
    uint32_t *d_list = nullptr;
    unsigned long long *d_counters = nullptr;
    unsigned long long h_counters[CN_SLOTS] = {};
    // a batch of views: the table of view cameras and keys the rank's render kernels read, on the rank's device (every
    // path start and every draw reads it); the first part's is the frame's own
    ViewCamera *d_views = nullptr;
    FrameEvents ev;                 // the probe: ZEROED -> END; a pass: BEGIN -> END
    cudaEvent_t traced = nullptr;   // the rank's samples so far are in its sums and Q
    cudaEvent_t gathered = nullptr; // the rank's slice of the totals is written
    cudaEvent_t listed = nullptr;   // (rank 0) the shared flags are final: the ranks may compact from them
};

// What a frame was opened with, as its opener's caller gave it: rt_frame_save writes it into the snapshot, and resuming
// opens the frame again from it (so the snapshot does not depend on the layout of the device's tables)
struct FrameSpec {
    RtCamera camera{};             // the frame's camera; a batch's first
    std::vector<RtCamera> cameras; // a batch of views: every view's camera and seed (empty otherwise)
    std::vector<uint64_t> seeds;
    bool has_window = false;
    FrameWindow window{};
    int32_t max_w = 0, max_h = 0;
    RtRenderOpts opts{};
};

} // namespace rtfs

// A frame owns everything a pass writes: sums, flags, the image and, in its parts, the flagged-pixel lists and counter
// blocks (paths, rays, the list length and the work cursors), so rt_render and other frames can use the scene between
// passes.  It has one part per device, in rank order: one for rt_frame_begin*, one per device of the RtMulti for
// rt_multi_frame_begin.  Its own sums and Q are the totals of the parts on the first device, and its flags the flags every
// part compacts from; over several devices every call that reads the frame gathers the totals first.  The noise estimate,
// the check's converge_kernel, the features, the filter and the read all run on the first device, over those buffers.
struct RtFrame {
    RtScene *scene = nullptr; // the first device's
    FrameParams fp;
    size_t n_pixels = 0;
    int32_t *d_stats = nullptr;
    uint8_t *d_flags = nullptr;
    uint8_t *d_rgb = nullptr;
    unsigned long long *d_sq = nullptr; // RT_FLAG_NOISE: per pixel the sum of r^2 + g^2 + b^2 (null otherwise)
    float *d_se = nullptr;              // rt_frame_noise's map, allocated on first use
    NoisePartial *d_partial = nullptr;  // and its per-block partial summaries, then the summary (kNoiseBlocks + 1 per view)
    // a batch of views (rt_frame_begin_views): the frame's own table of view cameras and keys, since rt_render_views
    // rewrites the workspace's between two passes; null for a frame of one camera
    ViewCamera *d_views = nullptr;
    int32_t n_views = 1;
    // rt_frame_features' buffers, allocated on first use and computed once per feature_samples (0: not computed yet)
    FrameFeatures feat{};
    int32_t feat_samples = 0;
    float4 *d_denoise = nullptr; // rt_frame_denoise's two levels (2 n_pixels), allocated on first use
    uint64_t paths_done = 0;     // the parts' paths, summed at the end of every step
    uint64_t pixels_listed = 0;  // the length of the list every part compacted last
    int32_t samples_done = 0, samples_target = 0;
    uint64_t pixels_flagged = 0;
    double ms_per_sample = -1.0; // measured device time of one sample index of every flagged pixel (< 0: not known yet)
    double last_pass_ms = 0.0, device_ms = 0.0;
    int32_t passes = 0;
    // convergence rule (rt_frame_set_convergence; conv_interval == 0: none): checkpoints conv_min + j conv_interval
    double conv_tolerance = 0.0;
    int32_t conv_min = 0, conv_interval = 0, conv_checks = 0;
    uint64_t pixels_active = 0; // pixels still being sampled: the list's length (pixels_flagged until a check)
    uint64_t generation = 0;    // the scene's edit count when the frame opened (rt_scene_update)
    std::vector<FramePart> parts;
    bool gathered = true; // the totals hold every part's samples (always, with one part)
    FrameSpec spec;
    uint64_t paths_base = 0; // a resumed frame: the paths of the snapshot (its parts' counter blocks start at zero)
};

namespace {

DeviceScene *part_scene(const FramePart &p) { return static_cast<DeviceScene *>(p.scene->dev); }

void frame_free(RtFrame *f) {
    if (!f) return;
    for (FramePart &p : f->parts) {
        if (!p.scene) continue; // (an opener that failed before reaching this part)
        cudaSetDevice(part_scene(p)->device);
        cudaStreamSynchronize(part_scene(p)->ws->stream);
        if (f->parts.size() > 1) { // (the only part of a frame traces into the frame's own buffers, freed below)
            cudaFree(p.d_stats);
            cudaFree(p.d_sq);
            cudaFree(p.d_flags);
            if (p.d_views != f->d_views) cudaFree(p.d_views);
        }
        cudaFree(p.d_list);
        cudaFree(p.d_counters);
        p.ev.destroy();
        for (cudaEvent_t e : {p.traced, p.gathered, p.listed})
            if (e) cudaEventDestroy(e);
    }
    cudaSetDevice(static_cast<DeviceScene *>(f->scene->dev)->device); // (its stream, the first part's, is synchronised above)
    cudaFree(f->d_stats);
    cudaFree(f->d_flags);
    cudaFree(f->d_rgb);
    cudaFree(f->d_sq);
    cudaFree(f->d_se);
    cudaFree(f->d_partial);
    cudaFree(f->d_views);
    cudaFree(f->feat.prim);
    cudaFree(f->feat.albedo);
    cudaFree(f->feat.normal);
    cudaFree(f->feat.depth);
    cudaFree(f->d_denoise);
    delete f;
}

// the first checkpoint of the frame's rule above samples_done (int64: m + j k may pass INT32_MAX)
int64_t next_checkpoint(const RtFrame *f) {
    const int64_t m = f->conv_min, k = f->conv_interval, s = f->samples_done;
    return s < m ? m : m + ((s - m) / k + 1) * k;
}

void frame_progress(const RtFrame *f, RtFrameProgress *p) {
    if (!p) return;
    std::memset(p, 0, sizeof *p);
    const uint64_t n_probe = uint64_t(f->fp.n_probe);
    p->samples_done = f->samples_done;
    p->samples_target = f->samples_target;
    p->paths_done = f->paths_done;
    p->paths_target = uint64_t(f->n_pixels) * n_probe + f->pixels_flagged * (uint64_t(f->samples_target) - n_probe);
    // with a rule: exact if nothing more converges, so it only shrinks at a check
    if (f->conv_interval) p->paths_target = p->paths_done + f->pixels_active * uint64_t(f->samples_target - f->samples_done);
    p->pixels_flagged = f->pixels_flagged;
    p->last_pass_ms = f->last_pass_ms;
    p->device_ms = f->device_ms;
    p->passes = f->passes;
    p->done = f->samples_done == f->samples_target ? 1 : 0;
}

// ---- the parts of a frame ------------------------------------------------------------------------------------------------
// Devices are ordered by CUDA events only: a rank waits for the others' events on its own stream, and no kernel spins.

// The totals on the first device, over several parts: once every rank's work so far is done, rank r sums its slice of the
// pixels of every rank (launch_gather, peer loads), and at the probe also ORs the ranks' flags into the frame's flags; the
// first device's stream then waits for every slice.
int frame_gather(RtFrame *f, bool probe_flags) {
    const int world = int(f->parts.size());
    GatherTargets t{};
    t.world = world;
    for (int r = 0; r < world; ++r) {
        t.stats[r] = f->parts[r].d_stats;
        t.sq[r] = f->parts[r].d_sq;
        t.flags[r] = f->parts[r].d_flags;
    }
    t.total_stats = f->d_stats;
    t.total_sq = f->d_sq;
    t.total_flags = probe_flags ? f->d_flags : nullptr;
    for (FramePart &p : f->parts) {
        RT_CUDA(cudaSetDevice(part_scene(p)->device));
        RT_CUDA(cudaEventRecord(p.traced, part_scene(p)->ws->stream));
    }
    for (int r = 0; r < world; ++r) {
        DeviceScene *ds = part_scene(f->parts[r]);
        RT_CUDA(cudaSetDevice(ds->device));
        for (int j = 0; j < world; ++j)
            if (j != r) RT_CUDA(cudaStreamWaitEvent(ds->ws->stream, f->parts[j].traced, 0));
        int rc = launch_gather(t, r, f->n_pixels, ds->ws->stream);
        if (rc != RT_OK) return rc;
        RT_CUDA(cudaEventRecord(f->parts[r].gathered, ds->ws->stream));
    }
    DeviceScene *ds0 = part_scene(f->parts[0]);
    RT_CUDA(cudaSetDevice(ds0->device));
    for (int j = 1; j < world; ++j) RT_CUDA(cudaStreamWaitEvent(ds0->ws->stream, f->parts[j].gathered, 0));
    f->gathered = true;
    return RT_OK;
}

// the totals, gathered if a pass has run since they last were (then on the first device's stream)
int ensure_totals(RtFrame *f) { return f->gathered ? RT_OK : frame_gather(f, false); }

// After the probe (probe: over several parts, the frame's flags become the OR of the ranks' probe flags) or a pass that
// ends on a checkpoint (converge: converge_kernel clears the converged pixels' flags on the first device): every rank
// compacts the frame's flags into its own list, so every rank samples the same pixels.  With one part nothing is gathered
// and no stream waits for another.
int frame_relist(RtFrame *f, bool probe, bool converge) {
    const size_t world = f->parts.size();
    int rc;
    if (world > 1 && (rc = frame_gather(f, probe)) != RT_OK) return rc;
    cudaStream_t st0 = part_scene(f->parts[0])->ws->stream;
    if (converge) {
        converge_kernel<<<unsigned((f->n_pixels + 255) / 256), 256, 0, st0>>>(reinterpret_cast<const int4 *>(f->d_stats), f->d_sq, f->d_flags,
                                                                              f->n_pixels, f->conv_tolerance);
        RT_CUDA(cudaGetLastError());
    }
    if (world > 1) RT_CUDA(cudaEventRecord(f->parts[0].listed, st0));
    int launches = 0;
    for (size_t r = 0; r < world; ++r) {
        FramePart &p = f->parts[r];
        DeviceScene *ds = part_scene(p);
        RT_CUDA(cudaSetDevice(ds->device));
        if (r) RT_CUDA(cudaStreamWaitEvent(ds->ws->stream, f->parts[0].listed, 0));
        if ((rc = launch_compact(ds, p.fp, single_flags(f->d_flags), p.d_list, ds->ws->stream, &launches)) != RT_OK) return rc;
    }
    return RT_OK;
}

// The end of a step (the opener's or a pass), on every rank: END, its counters to the host, then a synchronisation of every
// rank's stream.  The frame's paths are then the ranks' paths summed, and its list length the shared list's; returns the
// slowest rank's `from` -> END span.
int frame_sync(RtFrame *f, FrameEvents::Which from, double *span_ms) {
    for (FramePart &p : f->parts) {
        DeviceScene *ds = part_scene(p);
        RT_CUDA(cudaSetDevice(ds->device));
        RT_CUDA(p.ev.record(FrameEvents::END, ds->ws->stream));
        RT_CUDA(cudaMemcpyAsync(p.h_counters, p.d_counters, CN_SLOTS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ds->ws->stream));
    }
    *span_ms = 0.0;
    f->paths_done = f->paths_base;
    for (FramePart &p : f->parts) {
        RT_CUDA(cudaSetDevice(part_scene(p)->device));
        RT_CUDA(cudaStreamSynchronize(part_scene(p)->ws->stream));
        *span_ms = std::max(*span_ms, double(p.ev.ms(from, FrameEvents::END)));
        f->paths_done += p.h_counters[CN_PATHS];
    }
    f->pixels_listed = f->parts[0].h_counters[CN_LIST];
    return RT_OK;
}

// The half of every opener that allocates, once its arguments are checked: the frame's sums, Q, flags and image on the
// first device, one part per scene (the scene of rt_frame_begin*, or the replicas of an RtMulti in rank order), and every
// part's parameters and table of views.  A batch's frame is the tall frame of rt_render_views (rtfs_views.cu) with its own
// table; a window's frame holds the window's pixels only (rtfs_window.cu).  frame_open then probes; frame_resume restores a
// snapshot instead.  On failure nothing is left allocated.
int frame_alloc(const std::vector<RtScene *> &scenes, const FrameSpec &spec, RtFrame **out, const char *who) {
    const int world = int(scenes.size());
    const RtRenderOpts *opts = &spec.opts;
    const int32_t max_w = spec.max_w, max_h = spec.max_h;
    const FrameWindow *window = spec.has_window ? &spec.window : nullptr;
    const std::vector<ViewCamera> views = spec.cameras.empty() ? std::vector<ViewCamera>()
                                                               : view_table(spec.cameras.data(), spec.seeds.data(), int32_t(spec.cameras.size()),
                                                                            max_w, max_h, opts->seed);
    const bool noise = (opts->flags & RT_FLAG_NOISE) != 0;
    int rc;
    for (RtScene *s : scenes)
        if ((rc = prepare_frame(s, opts)) != RT_OK) return rc;
    auto *ds0 = static_cast<DeviceScene *>(scenes[0]->dev);
    RT_CUDA(cudaSetDevice(ds0->device));
    auto *f = new RtFrame();
    f->scene = scenes[0];
    f->generation = scenes[0]->generation;
    f->spec = spec;
    auto bail = [&](int code) {
        frame_free(f);
        return code;
    };
    const size_t view_pixels = size_t(2 * max_w + 1) * size_t(2 * max_h + 1);
    const size_t n = window ? size_t(window->rows) * size_t(window->cols) : view_pixels * std::max<size_t>(1, views.size());
    f->n_pixels = n;
    f->n_views = std::max(1, int32_t(views.size()));
    bool ok = cudaMalloc((void **)&f->d_stats, n * 4 * sizeof(int32_t)) == cudaSuccess && cudaMalloc((void **)&f->d_flags, n) == cudaSuccess &&
              cudaMalloc((void **)&f->d_rgb, n * 3) == cudaSuccess;
    if (noise) ok = ok && cudaMalloc((void **)&f->d_sq, n * sizeof(unsigned long long)) == cudaSuccess;
    if (!views.empty()) ok = ok && cudaMalloc((void **)&f->d_views, views.size() * sizeof(ViewCamera)) == cudaSuccess;
    f->parts.resize(size_t(world));
    for (int r = 0; r < world && ok; ++r) {
        FramePart &p = f->parts[size_t(r)];
        p.scene = scenes[size_t(r)];
        ok = cudaSetDevice(part_scene(p)->device) == cudaSuccess && cudaMalloc((void **)&p.d_list, n * sizeof(uint32_t)) == cudaSuccess &&
             cudaMalloc((void **)&p.d_counters, CN_SLOTS * sizeof(unsigned long long)) == cudaSuccess && p.ev.create() &&
             cudaEventCreateWithFlags(&p.traced, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&p.gathered, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&p.listed, cudaEventDisableTiming) == cudaSuccess;
        p.d_views = f->d_views;
        if (world == 1) { // the only part traces into the frame's own buffers: its totals need no gather
            p.d_stats = f->d_stats;
            p.d_flags = f->d_flags;
            p.d_sq = f->d_sq;
            continue;
        }
        ok = ok && cudaMalloc((void **)&p.d_stats, n * 4 * sizeof(int32_t)) == cudaSuccess && cudaMalloc((void **)&p.d_flags, n) == cudaSuccess;
        if (noise) ok = ok && cudaMalloc((void **)&p.d_sq, n * sizeof(unsigned long long)) == cudaSuccess;
        if (r > 0 && !views.empty()) {
            p.d_views = nullptr;
            ok = ok && cudaMalloc((void **)&p.d_views, views.size() * sizeof(ViewCamera)) == cudaSuccess;
        }
    }
    if (!ok) return bail(fail(RT_ERR_CUDA, std::string(who) + ": allocation failed: " + cudaGetErrorString(cudaGetLastError())));

    // the frame's parameters are one device's (the features, the filter, the pacing and rt_frame_extend read them); each
    // part has its own, of rank r of world
    auto fill = [&](FrameParams &fp, DeviceScene *ds, const ViewCamera *d_views, int r, int w) {
        fill_frame(fp, ds, spec.camera, max_w, max_h, *opts, r, w);
        if (!views.empty()) set_views(fp, d_views, f->n_views, int32_t(view_pixels));
        if (window) set_window(fp, *window);
    };
    fill(f->fp, ds0, f->d_views, 0, 1);
    f->samples_done = f->fp.n_probe; // 0 without the early-out
    f->samples_target = f->fp.sample_end;
    for (int r = 0; r < world; ++r) {
        FramePart &p = f->parts[size_t(r)];
        DeviceScene *ds = part_scene(p);
        if (cudaSetDevice(ds->device) != cudaSuccess) return bail(fail(RT_ERR_CUDA, std::string(who) + ": cudaSetDevice failed"));
        // a batch: the rank's table on its device (from pageable memory: staged before the call returns, and the probe
        // or the restore follows it on the stream)
        if (!views.empty() &&
            cudaMemcpyAsync(p.d_views, views.data(), views.size() * sizeof(ViewCamera), cudaMemcpyHostToDevice, ds->ws->stream) != cudaSuccess)
            return bail(fail(RT_ERR_CUDA, std::string(who) + ": view table upload failed: " + cudaGetErrorString(cudaGetLastError())));
        fill(p.fp, ds, p.d_views, r, world);
        p.fp.stats = p.d_stats;
        p.fp.flags = p.d_flags;
        p.fp.list = p.d_list;
        p.fp.counters = p.d_counters;
        p.fp.sq = p.d_sq; // non-null: plan_launch picks the kernels that also sum the squares
    }
    *out = f;
    return RT_OK;
}

// Every opener: frame_alloc, then the split probe and the compaction.
int frame_open(const std::vector<RtScene *> &scenes, const FrameSpec &spec, RtFrame **out, RtFrameProgress *progress, const char *who) {
    RtFrame *f = nullptr;
    int rc = frame_alloc(scenes, spec, &f, who);
    if (rc != RT_OK) return rc;
    auto bail = [&](int code) {
        frame_free(f);
        return code;
    };
    int launches = 0;
    for (FramePart &p : f->parts) {
        DeviceScene *ds = part_scene(p);
        if (cudaSetDevice(ds->device) != cudaSuccess) return bail(fail(RT_ERR_CUDA, std::string(who) + ": cudaSetDevice failed"));
        // the probe of the rank's tiles; with its own counter block the rank keeps the raw "means differ" flags, also where
        // this target has no main phase: the frame can be extended
        if ((rc = frame_probe(ds, p.fp, ds->ws->stream, &p.ev, &launches)) != RT_OK) return bail(rc);
    }
    if ((rc = frame_relist(f, true, false)) != RT_OK) return bail(rc);
    if ((rc = frame_sync(f, FrameEvents::ZEROED, &f->device_ms)) != RT_OK) return bail(rc);
    f->pixels_flagged = f->pixels_active = f->pixels_listed;
    // the probe traced n_probe samples of every pixel, a pass traces samples of the flagged pixels only; over several
    // devices the slowest rank probed 1 / world of the pixels and a pass gives it 1 / world of the indices
    if (f->fp.adaptive) f->ms_per_sample = f->device_ms * double(f->pixels_flagged) / (double(f->n_pixels) * double(f->fp.n_probe));
    *out = f;
    frame_progress(f, progress);
    return RT_OK;
}

// The spec of an opener's arguments (seeds null: every view has opts->seed)
FrameSpec frame_spec(const RtCamera *cameras, const uint64_t *seeds, int32_t n_views, const FrameWindow *window, int32_t max_w, int32_t max_h,
                     const RtRenderOpts *opts) {
    FrameSpec s;
    s.camera = cameras[0];
    if (n_views > 0) {
        s.cameras.assign(cameras, cameras + n_views);
        s.seeds.assign(size_t(n_views), opts->seed);
        if (seeds) s.seeds.assign(seeds, seeds + n_views);
    }
    if (window) {
        s.has_window = true;
        s.window = *window;
    }
    s.max_w = max_w;
    s.max_h = max_h;
    s.opts = *opts;
    return s;
}

// one pass of every rank over [s, s + k) with s = samples_done (rank r: the indices s + r + j world) and, when it
// ends on a checkpoint, the check; *span_ms is the slowest rank's BEGIN -> END
int frame_pass(RtFrame *f, int k, bool check, double *span_ms) {
    int launches = 0;
    for (FramePart &p : f->parts) {
        DeviceScene *ds = part_scene(p);
        RT_CUDA(cudaSetDevice(ds->device));
        cudaStream_t st = ds->ws->stream;
        FrameParams fp = p.fp;
        fp.cam.spp = f->fp.cam.spp; // (rt_frame_extend changes the frame's parameters only)
        fp.sample_begin = f->samples_done;
        fp.sample_end = f->samples_done + k;
        RT_CUDA(cudaMemsetAsync(p.d_counters + CN_WORK_MAIN, 0, sizeof(unsigned long long), st));
        RT_CUDA(p.ev.record(FrameEvents::BEGIN, st));
        int rc = launch_samples(ds, fp, st, &launches);
        if (rc != RT_OK) return rc;
    }
    f->gathered = f->parts.size() == 1;
    if (check) {
        int rc = frame_relist(f, false, true);
        if (rc != RT_OK) return rc;
    }
    return frame_sync(f, FrameEvents::BEGIN, span_ms);
}

// rt_frame_view_noise reduces at most this many views per launch: the grid's y extent stays far below its limit (65535),
// and the partials stay at most 16.8 MB however many views a batch of small extents has
constexpr int32_t kNoiseViewChunk = 1024;

// What rt_frame_noise and rt_frame_view_noise share before they reduce: their checks, the totals, and the partial summaries
// (kNoiseBlocks + 1 per view of one chunk of views, allocated on first use); *st is the first device's stream.
int noise_begin(RtFrame *f, double tolerance, const char *who, cudaStream_t *st) {
    if (!f->d_sq) return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": the frame was opened without RT_FLAG_NOISE");
    if (!(tolerance >= 0.0)) return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": tolerance must be >= 0");
    int rc = ensure_totals(f);
    if (rc != RT_OK) return rc;
    auto *ds = static_cast<DeviceScene *>(f->scene->dev);
    RT_CUDA(cudaSetDevice(ds->device));
    *st = ds->ws->stream;
    const size_t views = size_t(std::min(f->n_views, kNoiseViewChunk));
    if (!f->d_partial) RT_CUDA(cudaMalloc((void **)&f->d_partial, views * (kNoiseBlocks + 1) * sizeof(NoisePartial)));
    return RT_OK;
}

// The reduction of views [v0, v0 + nv) of view_pixels pixels each, every view as rt_frame_noise reduces a frame of its
// pixels (the same 512 ranges, tree and block order): view v0 + i's summary is then at d_partial + i (kNoiseBlocks + 1) +
// kNoiseBlocks.  se (or null) receives E of every pixel of those views.
int launch_noise(RtFrame *f, int32_t v0, int32_t nv, size_t view_pixels, double tolerance, float *se, cudaStream_t st) {
    const size_t at = size_t(v0) * view_pixels;
    noise_kernel<<<dim3(kNoiseBlocks, unsigned(nv)), kNoiseThreads, 0, st>>>(reinterpret_cast<const int4 *>(f->d_stats) + at, f->d_sq + at,
                                                                              f->d_flags + at, view_pixels, tolerance, se, f->d_partial);
    RT_CUDA(cudaGetLastError());
    noise_summary_kernel<<<unsigned(nv), kNoiseThreads, 0, st>>>(f->d_partial);
    RT_CUDA(cudaGetLastError());
    return RT_OK;
}

void fill_noise(const NoisePartial &total, double tolerance, RtFrameNoise *out) {
    out->pixels = total.pixels;
    out->pixels_above = total.above;
    out->max_se = total.max_se;
    out->mean_se = total.pixels ? total.sum_se / double(total.pixels) : 0.0;
    out->tolerance = tolerance;
}

// the frame's features of sample indices [0, samples), computed on first use of that count (they never change with passes)
int ensure_features(RtFrame *f, int32_t samples, cudaStream_t st) {
    const size_t n = f->n_pixels;
    if (!f->feat.prim) RT_CUDA(cudaMalloc((void **)&f->feat.prim, n * sizeof(int32_t)));
    if (!f->feat.albedo) RT_CUDA(cudaMalloc((void **)&f->feat.albedo, n * 3));
    if (!f->feat.normal) RT_CUDA(cudaMalloc((void **)&f->feat.normal, n * 3 * sizeof(float)));
    if (!f->feat.depth) RT_CUDA(cudaMalloc((void **)&f->feat.depth, n * sizeof(float)));
    if (f->feat_samples != samples) {
        f->feat_samples = 0;
        int rc = launch_features(f->fp, n, samples, f->feat, st);
        if (rc != RT_OK) return rc;
        f->feat_samples = samples;
    }
    return RT_OK;
}

// RT_ERR_INVALID_ARGUMENT if the scene was edited since the frame opened: its probe, flags and samples are of the old scene
int check_current(const RtFrame *f, const char *who) {
    if (f->generation != f->scene->generation)
        return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": the scene changed (rt_scene_update) since the frame was opened; open a new frame");
    return RT_OK;
}

// ---- snapshots (rt_frame_save, rt_frame_resume; the format is in include/rtfs_b200.h, the kernels in rtfs_snapshot.cu) ----

constexpr char kSnapshotMagic[8] = {'R', 'T', 'F', 'S', 'S', 'N', 'A', 'P'};
constexpr size_t kViewEntryBytes = sizeof(RtCamera) + sizeof(uint64_t); // a batch's view: the caller's camera and seed

// the byte offsets of a snapshot's view table, its pixel sections and its end
struct SnapshotLayout {
    size_t table, sections, total;
};
SnapshotLayout snapshot_layout(int32_t kind, size_t n_views, size_t n_pixels, bool noise) {
    SnapshotLayout l;
    l.table = sizeof(RtSnapshotHeader);
    l.sections = l.table + (kind == RT_FRAME_VIEWS ? n_views * kViewEntryBytes : 0);
    l.total = l.sections + 8 * snapshot_section_words(n_pixels, noise);
    return l;
}

int32_t frame_kind(const RtFrame *f) { return f->spec.has_window ? RT_FRAME_WINDOW : f->spec.cameras.empty() ? RT_FRAME_CAMERA : RT_FRAME_VIEWS; }

// the sum of the checksum terms of the header (its checksum field read as 0) and the view table, bytes [0, sections)
uint64_t snapshot_head_checksum(const uint8_t *bytes, size_t sections) {
    RtSnapshotHeader h;
    std::memcpy(&h, bytes, sizeof h);
    h.checksum = 0;
    return snapshot_checksum(&h, sizeof h, 0) + snapshot_checksum(bytes + sizeof h, sections - sizeof h, sizeof h / 8);
}

// a device allocation freed when the call returns, on whichever path
struct StagingBuffer {
    void *p = nullptr;
    ~StagingBuffer() { cudaFree(p); }
};

// rt_frame_resume's and rt_multi_frame_resume's body, once the handle is checked: the header's checks, the scene's
// fingerprint and the opener's checks, all before any device allocation; then frame_alloc, the restore of the sections
// into the first part's sums and Q and the frame's flags (the other parts start from zero), and the relist and end of step
// that follow a probe.
int frame_resume(const std::vector<RtScene *> &scenes, bool multi, const void *snapshot, size_t len, RtFrame **out, RtFrameProgress *progress,
                 const char *who) {
    const std::string w(who);
    RtScene *scene = scenes[0];
    if (!scene->dev) return fail(RT_ERR_UNSUPPORTED, w + ": the scene was created without a device (device = -1)");
    if (!snapshot || len < sizeof(RtSnapshotHeader)) return fail(RT_ERR_INVALID_ARGUMENT, w + ": the snapshot is null or shorter than its header");
    const auto *bytes = static_cast<const uint8_t *>(snapshot);
    RtSnapshotHeader h;
    std::memcpy(&h, bytes, sizeof h);
    if (std::memcmp(h.magic, kSnapshotMagic, sizeof kSnapshotMagic) != 0) return fail(RT_ERR_INVALID_ARGUMENT, w + ": not a frame snapshot (bad magic)");
    if (h.version != RT_SNAPSHOT_VERSION)
        return fail(RT_ERR_INVALID_ARGUMENT, w + ": snapshot format version " + std::to_string(h.version) + "; this library reads version 1");
    const bool noise = (h.opts.flags & RT_FLAG_NOISE) != 0;
    if (h.header_bytes != sizeof h || h.total_bytes != len || h.kind < RT_FRAME_CAMERA || h.kind > RT_FRAME_WINDOW || h.n_views < 1 ||
        (h.kind != RT_FRAME_VIEWS && h.n_views != 1) || h.n_pixels == 0 || h.n_pixels >= (uint64_t(1) << 31) ||
        snapshot_layout(h.kind, size_t(h.n_views), size_t(h.n_pixels), noise).total != len)
        return fail(RT_ERR_INVALID_ARGUMENT, w + ": the snapshot's lengths do not match its header");
    const SnapshotLayout L = snapshot_layout(h.kind, size_t(h.n_views), size_t(h.n_pixels), noise);
    const uint64_t head_sum = snapshot_head_checksum(bytes, L.sections);
    if (head_sum + snapshot_checksum(bytes + L.sections, len - L.sections, L.sections / 8) != h.checksum)
        return fail(RT_ERR_INVALID_ARGUMENT, w + ": the snapshot's checksum does not match its bytes");
    if (h.kind == RT_FRAME_WINDOW && multi)
        return fail(RT_ERR_UNSUPPORTED, w + ": a window runs on one GPU; resume it with rt_frame_resume");
    if (h.n_objects != int32_t(scene->objects.size()) || h.n_textures != int32_t(scene->textures.size()) ||
        h.scene_fingerprint != scene_fingerprint(scene))
        return fail(RT_ERR_INVALID_ARGUMENT, w + ": the scene's objects or textures differ from those of the saved frame's scene");

    // the opener's arguments, and its checks
    FrameSpec spec;
    spec.camera = h.camera;
    spec.max_w = h.max_width_coord;
    spec.max_h = h.max_height_coord;
    spec.opts = h.opts;
    int rc;
    if (h.kind == RT_FRAME_VIEWS) {
        spec.cameras.resize(size_t(h.n_views));
        spec.seeds.resize(size_t(h.n_views));
        for (size_t v = 0; v < size_t(h.n_views); ++v) {
            std::memcpy(&spec.cameras[v], bytes + L.table + v * kViewEntryBytes, sizeof(RtCamera));
            std::memcpy(&spec.seeds[v], bytes + L.table + v * kViewEntryBytes + sizeof(RtCamera), sizeof(uint64_t));
        }
        rc = check_views(scene, spec.cameras.data(), h.n_views, spec.max_w, spec.max_h, &spec.opts, who);
    } else if (h.kind == RT_FRAME_WINDOW) {
        spec.has_window = true;
        spec.window = FrameWindow{h.window[0], h.window[1], h.window[2], h.window[3]};
        rc = check_window(spec.window, spec.max_w, spec.max_h, who);
        if (rc == RT_OK) rc = check_frame_args(scene, &spec.camera, spec.max_w, spec.max_h, &spec.opts);
    } else {
        rc = check_frame_args(scene, &spec.camera, spec.max_w, spec.max_h, &spec.opts);
    }
    if (rc != RT_OK) return rc;
    if ((rc = check_frame_mode(&spec.opts, who, h.kind != RT_FRAME_CAMERA)) != RT_OK) return rc;

    // the frame's state against what its arguments allow (rt_frame_extend, rt_frame_set_convergence)
    const bool adaptive = h.opts.adaptive != 0;
    const int32_t first_trial = adaptive ? std::min(5, h.camera.samples_per_pixel / 2) : 0, n_probe = adaptive ? 2 * first_trial + 1 : 0;
    const int32_t spp = h.samples_per_pixel, target = adaptive ? std::max(n_probe, spp) : spp;
    const size_t view_pixels = size_t(2 * spec.max_w + 1) * size_t(2 * spec.max_h + 1);
    const size_t n_pixels = spec.has_window ? size_t(spec.window.rows) * size_t(spec.window.cols) : view_pixels * size_t(h.n_views);
    const bool rule_ok = h.conv_interval == 0 ? h.conv_min == 0 && h.conv_checks == 0
                                               : noise && h.conv_interval >= 1 && h.conv_min >= 2 && h.conv_tolerance >= 0.0 && h.conv_checks >= 0;
    if (h.n_pixels != n_pixels || h.n_probe != n_probe || spp < 1 || spp > (1 << 22) || (adaptive && std::min(5, spp / 2) != first_trial) ||
        h.samples_target != target || h.samples_done < n_probe || h.samples_done > target || h.passes < 0 || h.pace_devices < 1 ||
        h.pixels_active > h.pixels_flagged || h.pixels_flagged > h.n_pixels || !rule_ok)
        return fail(RT_ERR_INVALID_ARGUMENT, w + ": the snapshot's frame state is not one its arguments allow");

    RtFrame *f = nullptr;
    if ((rc = frame_alloc(scenes, spec, &f, who)) != RT_OK) return rc;
    auto bail = [&](int code) {
        frame_free(f);
        return code;
    };
    f->fp.cam.spp = spp; // (as rt_frame_extend leaves it)
    f->fp.sample_end = target;
    f->samples_done = h.samples_done;
    f->samples_target = target;
    f->passes = h.passes;
    f->pixels_flagged = h.pixels_flagged;
    f->pixels_active = h.pixels_active;
    f->paths_base = h.paths_done;
    f->conv_tolerance = h.conv_tolerance;
    f->conv_min = h.conv_min;
    f->conv_interval = h.conv_interval;
    f->conv_checks = h.conv_checks;
    // a pass over world devices gives each 1 / world of the indices
    f->ms_per_sample = h.ms_per_sample > 0.0 ? h.ms_per_sample * double(h.pace_devices) / double(f->parts.size()) : h.ms_per_sample;

    const size_t words = snapshot_section_words(n_pixels, noise);
    StagingBuffer staging;
    SnapshotTally tally{};
    {
        for (size_t r = 0; r < f->parts.size(); ++r) { // ZEROED: the counters (and the other parts' sums and Q) are clear
            FramePart &p = f->parts[r];
            DeviceScene *ds = part_scene(p);
            cudaStream_t st = ds->ws->stream;
            if (cudaSetDevice(ds->device) != cudaSuccess || cudaMemsetAsync(p.d_counters, 0, CN_SLOTS * sizeof(unsigned long long), st) != cudaSuccess ||
                (r > 0 && cudaMemsetAsync(p.d_stats, 0, n_pixels * 4 * sizeof(int32_t), st) != cudaSuccess) ||
                (r > 0 && p.d_sq && cudaMemsetAsync(p.d_sq, 0, n_pixels * sizeof(unsigned long long), st) != cudaSuccess) ||
                p.ev.record(FrameEvents::ZEROED, st) != cudaSuccess)
                return bail(fail(RT_ERR_CUDA, w + ": clearing the parts failed: " + cudaGetErrorString(cudaGetLastError())));
        }
        FramePart &p0 = f->parts[0];
        DeviceScene *ds0 = part_scene(p0);
        cudaStream_t st0 = ds0->ws->stream;
        if (cudaSetDevice(ds0->device) != cudaSuccess || cudaMalloc(&staging.p, words * 8 + sizeof(SnapshotTally)) != cudaSuccess)
            return bail(fail(RT_ERR_CUDA, w + ": allocation failed: " + cudaGetErrorString(cudaGetLastError())));
        auto *d_words = static_cast<unsigned long long *>(staging.p);
        auto *d_tally = reinterpret_cast<SnapshotTally *>(d_words + words);
        if (cudaMemcpyAsync(d_words, bytes + L.sections, words * 8, cudaMemcpyHostToDevice, st0) != cudaSuccess ||
            cudaMemsetAsync(d_tally, 0, sizeof(SnapshotTally), st0) != cudaSuccess ||
            cudaMemsetAsync(&d_tally->first_bad, 0xff, sizeof d_tally->first_bad, st0) != cudaSuccess)
            return bail(fail(RT_ERR_CUDA, w + ": snapshot upload failed: " + cudaGetErrorString(cudaGetLastError())));
        const SnapshotSections sec{d_words, L.sections / 8, n_pixels, noise};
        const SnapshotRules rules{h.samples_done, n_probe, h.conv_min, h.conv_interval};
        if ((rc = launch_snapshot_unpack(sec, rules, p0.d_stats, p0.d_sq, f->d_flags, d_tally, st0)) != RT_OK) return bail(rc);
        if (cudaMemcpyAsync(&tally, d_tally, sizeof tally, cudaMemcpyDeviceToHost, st0) != cudaSuccess)
            return bail(fail(RT_ERR_CUDA, w + ": reading the restore's tally failed"));
    }
    if ((rc = frame_relist(f, false, false)) != RT_OK) return bail(rc);
    if ((rc = frame_sync(f, FrameEvents::ZEROED, &f->device_ms)) != RT_OK) return bail(rc);
    if (tally.first_bad != ~0ull)
        return bail(fail(RT_ERR_INVALID_ARGUMENT, w + ": pixel " + std::to_string(tally.first_bad) + " of the snapshot breaks the frame's rules"));
    if (head_sum + tally.checksum != h.checksum) return bail(fail(RT_ERR_INVALID_ARGUMENT, w + ": the sections changed on their way to the device"));
    if (tally.counts != h.paths_done || tally.active != h.pixels_active || tally.flagged != h.pixels_flagged || f->pixels_listed != h.pixels_active)
        return bail(fail(RT_ERR_INVALID_ARGUMENT, w + ": the snapshot's pixels do not add up to its paths_done, pixels_active and pixels_flagged"));
    *out = f;
    frame_progress(f, progress);
    return RT_OK;
}

} // namespace

extern "C" {

int rt_frame_begin(RtScene *scene, const RtCamera *camera, int32_t max_w, int32_t max_h, const RtRenderOpts *opts, RtFrame **out,
                   RtFrameProgress *progress) {
    int rc = check_frame_args(scene, camera, max_w, max_h, opts);
    if (rc != RT_OK) return rc;
    if (!out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_begin: out is null");
    *out = nullptr;
    if ((rc = check_frame_mode(opts, "rt_frame_begin", false)) != RT_OK) return rc;
    return frame_open({scene}, frame_spec(camera, nullptr, 0, nullptr, max_w, max_h, opts), out, progress, "rt_frame_begin");
}

int rt_frame_begin_views(RtScene *scene, const RtCamera *cameras, const uint64_t *seeds, int32_t n_views, int32_t max_w, int32_t max_h,
                         const RtRenderOpts *opts, RtFrame **out, RtFrameProgress *progress) {
    // rt_render_views' checks, then rt_frame_begin's
    int rc = check_views(scene, cameras, n_views, max_w, max_h, opts, "rt_frame_begin_views");
    if (rc != RT_OK) return rc;
    if (!out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_begin_views: out is null");
    *out = nullptr;
    if ((rc = check_frame_mode(opts, "rt_frame_begin_views", true)) != RT_OK) return rc;
    return frame_open({scene}, frame_spec(cameras, seeds, n_views, nullptr, max_w, max_h, opts), out, progress, "rt_frame_begin_views");
}

int rt_frame_begin_window(RtScene *scene, const RtCamera *camera, int32_t max_w, int32_t max_h, int32_t row0, int32_t col0, int32_t rows,
                          int32_t cols, const RtRenderOpts *opts, RtFrame **out, RtFrameProgress *progress) {
    // rt_render_window's checks, then rt_frame_begin's
    const FrameWindow w{row0, col0, rows, cols};
    int rc = check_window(w, max_w, max_h, "rt_frame_begin_window");
    if (rc != RT_OK) return rc;
    if (!out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_begin_window: out is null");
    *out = nullptr;
    if ((rc = check_frame_args(scene, camera, max_w, max_h, opts)) != RT_OK) return rc;
    if ((rc = check_frame_mode(opts, "rt_frame_begin_window", true)) != RT_OK) return rc;
    return frame_open({scene}, frame_spec(camera, nullptr, 0, &w, max_w, max_h, opts), out, progress, "rt_frame_begin_window");
}

int rt_multi_frame_begin(RtMulti *multi, const RtCamera *camera, int32_t max_w, int32_t max_h, const RtRenderOpts *opts, RtFrame **out,
                         RtFrameProgress *progress) {
    if (!out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_multi_frame_begin: out is null");
    *out = nullptr;
    if (!multi || multi_scenes(multi).empty()) return fail(RT_ERR_INVALID_ARGUMENT, "rt_multi_frame_begin: null handle");
    // rt_frame_begin's checks and refusals, on the first device's replica
    int rc = check_frame_args(multi_scenes(multi)[0], camera, max_w, max_h, opts);
    if (rc != RT_OK) return rc;
    if ((rc = check_frame_mode(opts, "rt_multi_frame_begin", false)) != RT_OK) return rc;
    return frame_open(multi_scenes(multi), frame_spec(camera, nullptr, 0, nullptr, max_w, max_h, opts), out, progress, "rt_multi_frame_begin");
}

int rt_multi_frame_begin_views(RtMulti *multi, const RtCamera *cameras, const uint64_t *seeds, int32_t n_views, int32_t max_w, int32_t max_h,
                               const RtRenderOpts *opts, RtFrame **out, RtFrameProgress *progress) {
    if (!out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_multi_frame_begin_views: out is null");
    *out = nullptr;
    if (!multi || multi_scenes(multi).empty()) return fail(RT_ERR_INVALID_ARGUMENT, "rt_multi_frame_begin_views: null handle");
    // rt_frame_begin_views' checks and refusals, on the first device's replica
    int rc = check_views(multi_scenes(multi)[0], cameras, n_views, max_w, max_h, opts, "rt_multi_frame_begin_views");
    if (rc != RT_OK) return rc;
    if ((rc = check_frame_mode(opts, "rt_multi_frame_begin_views", true)) != RT_OK) return rc;
    return frame_open(multi_scenes(multi), frame_spec(cameras, seeds, n_views, nullptr, max_w, max_h, opts), out, progress,
                      "rt_multi_frame_begin_views");
}

int rt_frame_advance(RtFrame *f, int32_t max_samples, double target_ms, RtFrameProgress *progress) {
    if (!f) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_advance: null frame");
    if (int rc = check_current(f, "rt_frame_advance"); rc != RT_OK) return rc;
    if (max_samples < 0 || !(target_ms >= 0.0)) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_advance: max_samples and target_ms must be >= 0");
    const bool rule = f->conv_interval > 0;
    if (rule && f->pixels_active == 0) f->samples_done = f->samples_target; // every pixel has stopped: nothing to trace
    const int left = f->samples_target - f->samples_done;
    if (left > 0) {
        int k = left;
        if (max_samples > 0) k = std::min(k, max_samples);
        if (target_ms > 0.0) {
            int paced = 1; // no rate known yet (no probe without the early-out): one sample index
            if (f->ms_per_sample == 0.0) paced = left; // nothing to trace (no pixel is flagged)
            else if (f->ms_per_sample > 0.0) paced = int(std::min(double(left), std::floor(target_ms / f->ms_per_sample)));
            // over several devices a paced window that the end does not cut is a multiple of the device count: no rank idles
            const int world = int(f->parts.size());
            if (world > 1 && paced < left && paced >= world) paced -= paced % world;
            k = std::min(k, std::max(1, paced));
        }
        if (rule) k = int(std::min<int64_t>(k, next_checkpoint(f) - f->samples_done)); // a pass never crosses a checkpoint
        const bool check = rule && f->samples_done + k == next_checkpoint(f);
        double span_ms = 0.0;
        if (int rc = frame_pass(f, k, check, &span_ms); rc != RT_OK) return rc;
        f->samples_done += k;
        f->passes += 1;
        f->last_pass_ms = span_ms;
        f->device_ms += f->last_pass_ms;
        const uint64_t before = f->pixels_active;
        if (check) {
            f->pixels_active = f->pixels_listed;
            f->conv_checks += 1;
            if (f->pixels_active == 0) f->samples_done = f->samples_target; // done, without a launch
        }
        // the next pass traces the pixels still listed
        f->ms_per_sample = before ? f->last_pass_ms / k * (double(f->pixels_active) / double(before)) : 0.0;
    }
    frame_progress(f, progress);
    return RT_OK;
}

int rt_frame_read(RtFrame *f, int32_t gamma, uint8_t *rgb_out, int32_t *sums_out) {
    if (!f) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_read: null frame");
    if (int rc = ensure_totals(f); rc != RT_OK) return rc;
    auto *ds = static_cast<DeviceScene *>(f->scene->dev);
    RT_CUDA(cudaSetDevice(ds->device));
    cudaStream_t st = ds->ws->stream;
    if (rgb_out) {
        int launches = 0;
        int rc = launch_finalize(f->d_stats, f->n_pixels, gamma, f->d_rgb, st, &launches);
        if (rc != RT_OK) return rc;
        RT_CUDA(cudaMemcpyAsync(rgb_out, f->d_rgb, f->n_pixels * 3, cudaMemcpyDeviceToHost, st));
    }
    if (sums_out) RT_CUDA(cudaMemcpyAsync(sums_out, f->d_stats, f->n_pixels * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    RT_CUDA(cudaStreamSynchronize(st));
    return RT_OK;
}

int rt_frame_extend(RtFrame *f, int32_t spp) {
    if (!f) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_extend: null frame");
    if (int rc = check_current(f, "rt_frame_extend"); rc != RT_OK) return rc;
    if (spp < 1 || spp > (1 << 22)) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_extend: samples_per_pixel must be in [1, 2^22]");
    FrameParams &fp = f->fp;
    if (fp.adaptive && std::min(5, spp / 2) != fp.first_trial) // Scene.fs:172
        return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_extend: this samples_per_pixel changes firstTrial, i.e. the probe the frame already ran");
    const int target = fp.adaptive ? std::max(fp.n_probe, spp) : spp;
    if (target < f->samples_done) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_extend: the frame already holds more samples than that");
    f->samples_target = target;
    fp.sample_end = target;
    fp.cam.spp = spp;
    return RT_OK;
}

void rt_frame_destroy(RtFrame *f) { frame_free(f); }

int rt_frame_noise(RtFrame *f, double tolerance, float *se_out, uint64_t *sq_out, RtFrameNoise *summary) {
    if (!f) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_noise: null frame");
    cudaStream_t st;
    int rc = noise_begin(f, tolerance, "rt_frame_noise", &st);
    if (rc != RT_OK) return rc;
    if (se_out && !f->d_se) RT_CUDA(cudaMalloc((void **)&f->d_se, f->n_pixels * sizeof(float)));
    if ((rc = launch_noise(f, 0, 1, f->n_pixels, tolerance, se_out ? f->d_se : nullptr, st)) != RT_OK) return rc;
    NoisePartial total;
    RT_CUDA(cudaMemcpyAsync(&total, f->d_partial + kNoiseBlocks, sizeof total, cudaMemcpyDeviceToHost, st));
    if (se_out) RT_CUDA(cudaMemcpyAsync(se_out, f->d_se, f->n_pixels * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (sq_out) RT_CUDA(cudaMemcpyAsync(sq_out, f->d_sq, f->n_pixels * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    RT_CUDA(cudaStreamSynchronize(st));
    if (summary) fill_noise(total, tolerance, summary);
    return RT_OK;
}

int rt_frame_view_noise(RtFrame *f, double tolerance, RtFrameNoise *per_view) {
    if (!f || !per_view) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_view_noise: null frame or output");
    cudaStream_t st;
    int rc = noise_begin(f, tolerance, "rt_frame_view_noise", &st);
    if (rc != RT_OK) return rc;
    const size_t view_pixels = f->n_pixels / size_t(f->n_views);
    std::vector<NoisePartial> totals(size_t(f->n_views));
    for (int32_t v0 = 0; v0 < f->n_views; v0 += kNoiseViewChunk) {
        const int32_t nv = std::min(kNoiseViewChunk, f->n_views - v0);
        if ((rc = launch_noise(f, v0, nv, view_pixels, tolerance, nullptr, st)) != RT_OK) return rc;
    // (the next chunk's kernels follow this copy on the stream before they overwrite the partials)
        RT_CUDA(cudaMemcpy2DAsync(totals.data() + v0, sizeof(NoisePartial), f->d_partial + kNoiseBlocks, (kNoiseBlocks + 1) * sizeof(NoisePartial),
                                  sizeof(NoisePartial), size_t(nv), cudaMemcpyDeviceToHost, st));
    }
    RT_CUDA(cudaStreamSynchronize(st));
    for (int32_t v = 0; v < f->n_views; ++v) fill_noise(totals[size_t(v)], tolerance, per_view + v);
    return RT_OK;
}

int rt_frame_set_convergence(RtFrame *f, double tolerance, int32_t min_samples, int32_t interval) {
    if (!f) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_set_convergence: null frame");
    if (int rc = check_current(f, "rt_frame_set_convergence"); rc != RT_OK) return rc;
    if (!f->d_sq) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_set_convergence: the frame was opened without RT_FLAG_NOISE");
    if (f->passes > 0) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_set_convergence: a pass has already run");
    if (!(tolerance >= 0.0)) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_set_convergence: tolerance must be >= 0");
    if (interval < 1) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_set_convergence: interval must be >= 1");
    if (min_samples < 2 || min_samples <= f->samples_done)
        return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_set_convergence: min_samples must be >= 2 and above the probe's samples");
    f->conv_tolerance = tolerance;
    f->conv_min = min_samples;
    f->conv_interval = interval;
    return RT_OK;
}

int rt_frame_convergence(RtFrame *f, RtFrameConvergence *out) {
    if (!f || !out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_convergence: null frame or output");
    if (!f->conv_interval) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_convergence: the frame has no convergence rule");
    out->tolerance = f->conv_tolerance;
    out->min_samples = f->conv_min;
    out->interval = f->conv_interval;
    out->next_check = int32_t(std::min<int64_t>(next_checkpoint(f), INT32_MAX));
    out->checks = f->conv_checks;
    out->pixels_active = f->pixels_active;
    out->pixels_converged = f->pixels_flagged - f->pixels_active;
    return RT_OK;
}

int rt_frame_features(RtFrame *f, int32_t samples, int32_t *prim_out, uint8_t *albedo_out, float *normal_out, float *depth_out) {
    if (!f) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_features: null frame");
    if (int rc = check_current(f, "rt_frame_features"); rc != RT_OK) return rc;
    if (samples < 1 || samples > kMaxFeatureSamples) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_features: samples must be in [1, 64]");
    auto *ds = static_cast<DeviceScene *>(f->scene->dev);
    RT_CUDA(cudaSetDevice(ds->device));
    cudaStream_t st = ds->ws->stream;
    int rc = ensure_features(f, samples, st);
    if (rc != RT_OK) return rc;
    const size_t n = f->n_pixels;
    if (prim_out) RT_CUDA(cudaMemcpyAsync(prim_out, f->feat.prim, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (albedo_out) RT_CUDA(cudaMemcpyAsync(albedo_out, f->feat.albedo, n * 3, cudaMemcpyDeviceToHost, st));
    if (normal_out) RT_CUDA(cudaMemcpyAsync(normal_out, f->feat.normal, n * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (depth_out) RT_CUDA(cudaMemcpyAsync(depth_out, f->feat.depth, n * sizeof(float), cudaMemcpyDeviceToHost, st));
    RT_CUDA(cudaStreamSynchronize(st));
    return RT_OK;
}

int rt_frame_denoise(RtFrame *f, const RtDenoiseOpts *opts, uint8_t *rgb_out, float *linear_out) {
    int rc = check_denoise_opts(opts, "rt_frame_denoise");
    if (rc != RT_OK) return rc;
    if (!f) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_denoise: null frame");
    if ((rc = check_current(f, "rt_frame_denoise")) != RT_OK) return rc;
    if (!f->d_sq) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_denoise: the frame was opened without RT_FLAG_NOISE");
    if ((rc = ensure_totals(f)) != RT_OK) return rc;
    auto *ds = static_cast<DeviceScene *>(f->scene->dev);
    RT_CUDA(cudaSetDevice(ds->device));
    cudaStream_t st = ds->ws->stream;
    if ((rc = ensure_features(f, opts->feature_samples, st)) != RT_OK) return rc;
    const size_t n = f->n_pixels;
    if (!f->d_denoise) RT_CUDA(cudaMalloc((void **)&f->d_denoise, 2 * n * sizeof(float4)));
    const int view_rows = f->fp.cam.rows / f->n_views; // the tall frame of a batch: taps stay inside their view
    uint8_t *d_rgb = nullptr;
    float *d_linear = nullptr;
    if ((rc = launch_denoise(f->d_stats, f->d_sq, f->feat, n, view_rows, f->fp.cam.cols, *opts, f->d_denoise, rgb_out != nullptr,
                             linear_out != nullptr, &d_rgb, &d_linear, st)) != RT_OK)
        return rc;
    if (rgb_out) RT_CUDA(cudaMemcpyAsync(rgb_out, d_rgb, n * 3, cudaMemcpyDeviceToHost, st));
    if (linear_out) RT_CUDA(cudaMemcpyAsync(linear_out, d_linear, n * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
    RT_CUDA(cudaStreamSynchronize(st));
    return RT_OK;
}

int rt_pixel_noise(const int32_t *sums, const uint64_t *sq, size_t n, float *se_out) {
    if (n && (!sums || !sq || !se_out)) return fail(RT_ERR_INVALID_ARGUMENT, "rt_pixel_noise: null buffer");
    for (size_t p = 0; p < n; ++p)
        se_out[p] = float(pixel_standard_error(sums[4 * p + 3], sums[4 * p], sums[4 * p + 1], sums[4 * p + 2], sq[p]));
    return RT_OK;
}

int rt_frame_save(RtFrame *f, void *out, size_t cap, size_t *len) {
    if (!f || !len) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_save: null frame or len");
    const bool noise = f->d_sq != nullptr;
    const int32_t kind = frame_kind(f);
    const SnapshotLayout L = snapshot_layout(kind, size_t(f->n_views), f->n_pixels, noise);
    *len = L.total;
    if (int rc = check_current(f, "rt_frame_save"); rc != RT_OK) return rc;
    if (!out && cap == 0) return RT_OK; // sizing only
    if (!out || cap < L.total)
        return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_save: the buffer holds " + std::to_string(cap) + " bytes; the snapshot takes " + std::to_string(L.total));
    int rc = ensure_totals(f);
    if (rc != RT_OK) return rc;
    auto *ds = static_cast<DeviceScene *>(f->scene->dev);
    RT_CUDA(cudaSetDevice(ds->device));
    cudaStream_t st = ds->ws->stream;
    const size_t words = snapshot_section_words(f->n_pixels, noise);
    StagingBuffer staging;
    RT_CUDA(cudaMalloc(&staging.p, (words + 1) * 8));
    auto *d_words = static_cast<unsigned long long *>(staging.p);
    RT_CUDA(cudaMemsetAsync(d_words + words, 0, 8, st));
    const SnapshotSections sec{d_words, L.sections / 8, f->n_pixels, noise};
    if ((rc = launch_snapshot_pack(f->d_stats, f->d_sq, f->d_flags, sec, d_words + words, st)) != RT_OK) return rc;
    auto *b = static_cast<uint8_t *>(out);
    uint64_t sections_sum = 0;
    RT_CUDA(cudaMemcpyAsync(b + L.sections, d_words, words * 8, cudaMemcpyDeviceToHost, st));
    RT_CUDA(cudaMemcpyAsync(&sections_sum, d_words + words, 8, cudaMemcpyDeviceToHost, st));

    // the header and the view table, written while the copy runs
    RtSnapshotHeader h;
    std::memset(&h, 0, sizeof h);
    std::memcpy(h.magic, kSnapshotMagic, sizeof h.magic);
    h.version = RT_SNAPSHOT_VERSION;
    h.header_bytes = sizeof h;
    h.total_bytes = L.total;
    h.scene_fingerprint = scene_fingerprint(f->scene);
    h.n_objects = int32_t(f->scene->objects.size());
    h.n_textures = int32_t(f->scene->textures.size());
    h.kind = kind;
    h.n_views = f->n_views;
    h.camera = f->spec.camera;
    h.max_width_coord = f->spec.max_w;
    h.max_height_coord = f->spec.max_h;
    if (f->spec.has_window) {
        h.window[0] = f->spec.window.row0;
        h.window[1] = f->spec.window.col0;
        h.window[2] = f->spec.window.rows;
        h.window[3] = f->spec.window.cols;
    }
    h.opts = f->spec.opts;
    h.samples_per_pixel = f->fp.cam.spp;
    h.samples_done = f->samples_done;
    h.samples_target = f->samples_target;
    h.n_probe = f->fp.n_probe;
    h.passes = f->passes;
    h.n_pixels = f->n_pixels;
    h.pixels_flagged = f->pixels_flagged;
    h.pixels_active = f->pixels_active;
    h.paths_done = f->paths_done;
    h.conv_tolerance = f->conv_tolerance;
    h.conv_min = f->conv_min;
    h.conv_interval = f->conv_interval;
    h.conv_checks = f->conv_checks;
    h.pace_devices = int32_t(f->parts.size());
    h.ms_per_sample = f->ms_per_sample;
    std::memcpy(b, &h, sizeof h);
    for (size_t v = 0; v < f->spec.cameras.size(); ++v) {
        std::memcpy(b + L.table + v * kViewEntryBytes, &f->spec.cameras[v], sizeof(RtCamera));
        std::memcpy(b + L.table + v * kViewEntryBytes + sizeof(RtCamera), &f->spec.seeds[v], sizeof(uint64_t));
    }
    const uint64_t head_sum = snapshot_head_checksum(b, L.sections);
    RT_CUDA(cudaStreamSynchronize(st));
    h.checksum = head_sum + sections_sum;
    std::memcpy(b + offsetof(RtSnapshotHeader, checksum), &h.checksum, sizeof h.checksum);
    return RT_OK;
}

int rt_frame_resume(RtScene *scene, const void *snapshot, size_t len, RtFrame **out, RtFrameProgress *progress) {
    if (!out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_resume: out is null");
    *out = nullptr;
    if (!scene) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_resume: null scene");
    return frame_resume({scene}, false, snapshot, len, out, progress, "rt_frame_resume");
}

int rt_multi_frame_resume(RtMulti *multi, const void *snapshot, size_t len, RtFrame **out, RtFrameProgress *progress) {
    if (!out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_multi_frame_resume: out is null");
    *out = nullptr;
    if (!multi || multi_scenes(multi).empty()) return fail(RT_ERR_INVALID_ARGUMENT, "rt_multi_frame_resume: null handle");
    return frame_resume(multi_scenes(multi), true, snapshot, len, out, progress, "rt_multi_frame_resume");
}

} // extern "C"
