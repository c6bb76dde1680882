// rtfs_frame.cu — progressive frames (rt_frame_*): rt_render's frame on one device, cut into passes over windows of
// sample indices.  The probe and the compaction run once, in rt_frame_begin; every rt_frame_advance is one
// launch_samples over [samples_done, samples_done + k), i.e. the same render_kernel<PROBE = false> that rt_render's main
// phase launches, with the same chunking.  Sums are integers keyed by (seed, pixel, sample index), so a frame that has
// reached samples_done is bit for bit rt_render's frame at samples_per_pixel = samples_done (include/rtfs_b200.h).
// A frame opened with RT_FLAG_NOISE also holds per pixel the sum of squares Q (render_kernel<NOISE = true>), from which
// rt_frame_noise derives a per-pixel standard error and a summary over the flagged pixels, and with which a convergence rule
// (rt_frame_set_convergence) stops sampling each pixel once its estimate is within a tolerance.
// rt_frame_begin_views opens the same frame over rt_render_views' tall frame of a batch of views (its kernels are in
// rtfs_views.cu); the probe flags, the compaction, the checks and the output tail work per pixel and need no change for it,
// and rt_frame_view_noise reduces each view as rt_frame_noise reduces a frame of its own.
// rt_frame_begin_window opens it over a window of rt_render's frame (its kernels are in rtfs_window.cu): the frame's buffers,
// maps and counts are the window's, and every per-pixel kernel runs over the window unchanged.
// rt_frame_features and rt_frame_denoise (kernels in rtfs_denoise.cu) read the frame and keep buffers of their own.
#include "rtfs_device.h"

#include <algorithm>
#include <cmath>
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

} // namespace rtfs

// A frame owns everything a pass writes: sums, flags, the flagged-pixel list, the image and its own counter block
// (paths, rays, the list length and the work cursors), so rt_render and other frames can use the scene between passes.
struct RtFrame {
    RtScene *scene = nullptr;
    FrameParams fp;
    size_t n_pixels = 0;
    int32_t *d_stats = nullptr;
    uint8_t *d_flags = nullptr;
    uint32_t *d_list = nullptr;
    uint8_t *d_rgb = nullptr;
    unsigned long long *d_counters = nullptr;
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
    unsigned long long h_counters[CN_SLOTS] = {};
    FrameEvents ev; // rt_frame_begin: ZEROED -> TRACED; a pass: BEGIN -> END
    int32_t samples_done = 0, samples_target = 0;
    uint64_t pixels_flagged = 0;
    double ms_per_sample = -1.0; // measured device time of one sample index of every flagged pixel (< 0: not known yet)
    double last_pass_ms = 0.0, device_ms = 0.0;
    int32_t passes = 0;
    // convergence rule (rt_frame_set_convergence; conv_interval == 0: none): checkpoints conv_min + j conv_interval
    double conv_tolerance = 0.0;
    int32_t conv_min = 0, conv_interval = 0, conv_checks = 0;
    uint64_t pixels_active = 0; // pixels still being sampled: the list's length (pixels_flagged until a check)
};

namespace {

void frame_free(RtFrame *f) {
    if (!f) return;
    auto *ds = static_cast<DeviceScene *>(f->scene->dev);
    cudaSetDevice(ds->device);
    cudaStreamSynchronize(ds->ws->stream);
    cudaFree(f->d_stats);
    cudaFree(f->d_flags);
    cudaFree(f->d_list);
    cudaFree(f->d_rgb);
    cudaFree(f->d_counters);
    cudaFree(f->d_sq);
    cudaFree(f->d_se);
    cudaFree(f->d_partial);
    cudaFree(f->d_views);
    cudaFree(f->feat.prim);
    cudaFree(f->feat.albedo);
    cudaFree(f->feat.normal);
    cudaFree(f->feat.depth);
    cudaFree(f->d_denoise);
    f->ev.destroy();
    delete f;
}

// one small device->host copy of the frame's counters and a synchronisation of the scene's stream
int frame_sync(RtFrame *f, cudaStream_t st) {
    RT_CUDA(cudaMemcpyAsync(f->h_counters, f->d_counters, CN_SLOTS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    RT_CUDA(cudaStreamSynchronize(st));
    return RT_OK;
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
    p->paths_done = f->h_counters[CN_PATHS];
    p->paths_target = uint64_t(f->n_pixels) * n_probe + f->pixels_flagged * (uint64_t(f->samples_target) - n_probe);
    // with a rule: exact if nothing more converges, so it only shrinks at a check
    if (f->conv_interval) p->paths_target = p->paths_done + f->pixels_active * uint64_t(f->samples_target - f->samples_done);
    p->pixels_flagged = f->pixels_flagged;
    p->last_pass_ms = f->last_pass_ms;
    p->device_ms = f->device_ms;
    p->passes = f->passes;
    p->done = f->samples_done == f->samples_target ? 1 : 0;
}

// rt_frame_begin (views empty, no window), rt_frame_begin_views and rt_frame_begin_window, once their arguments are checked:
// allocates the frame, and runs the probe and the compaction.  A batch's frame is the tall frame of rt_render_views
// (rtfs_views.cu) with its own table; a window's frame holds the window's pixels only (rtfs_window.cu).
int frame_open(RtScene *scene, const RtCamera &camera, const std::vector<ViewCamera> &views, const FrameWindow *window, int32_t max_w,
               int32_t max_h, const RtRenderOpts *opts, RtFrame **out, RtFrameProgress *progress, const char *who) {
    const bool noise = (opts->flags & RT_FLAG_NOISE) != 0;
    int rc = prepare_frame(scene, opts);
    if (rc != RT_OK) return rc;
    auto *ds = static_cast<DeviceScene *>(scene->dev);
    RT_CUDA(cudaSetDevice(ds->device));
    auto *f = new RtFrame();
    f->scene = scene;
    auto bail = [&](int code) {
        frame_free(f);
        return code;
    };
    const size_t view_pixels = size_t(2 * max_w + 1) * size_t(2 * max_h + 1);
    const size_t n = window ? size_t(window->rows) * size_t(window->cols) : view_pixels * std::max<size_t>(1, views.size());
    f->n_pixels = n;
    bool ok = cudaMalloc((void **)&f->d_stats, n * 4 * sizeof(int32_t)) == cudaSuccess && cudaMalloc((void **)&f->d_flags, n) == cudaSuccess &&
              cudaMalloc((void **)&f->d_list, n * sizeof(uint32_t)) == cudaSuccess && cudaMalloc((void **)&f->d_rgb, n * 3) == cudaSuccess &&
              cudaMalloc((void **)&f->d_counters, CN_SLOTS * sizeof(unsigned long long)) == cudaSuccess;
    if (noise) ok = ok && cudaMalloc((void **)&f->d_sq, n * sizeof(unsigned long long)) == cudaSuccess;
    if (!views.empty()) ok = ok && cudaMalloc((void **)&f->d_views, views.size() * sizeof(ViewCamera)) == cudaSuccess;
    ok = ok && f->ev.create();
    if (!ok) return bail(fail(RT_ERR_CUDA, std::string(who) + ": allocation failed: " + cudaGetErrorString(cudaGetLastError())));

    cudaStream_t st = ds->ws->stream;
    FrameParams &fp = f->fp;
    fill_frame(fp, ds, camera, max_w, max_h, *opts, 0, 1);
    if (!views.empty()) {
        // (from pageable memory: staged before the call returns; the probe below follows it on the stream)
        if (cudaMemcpyAsync(f->d_views, views.data(), views.size() * sizeof(ViewCamera), cudaMemcpyHostToDevice, st) != cudaSuccess)
            return bail(fail(RT_ERR_CUDA, std::string(who) + ": view table upload failed: " + cudaGetErrorString(cudaGetLastError())));
        f->n_views = int32_t(views.size());
        fp.cam.rows *= f->n_views; // the tall frame: probe tiles, flags, list, sums and Q run over it as over one frame
        fp.tiles_y = (fp.cam.rows + kTileH - 1) / kTileH;
        fp.views = f->d_views;
        fp.n_views = f->n_views;
        fp.view_pixels = int32_t(view_pixels);
    }
    if (window) set_window(fp, *window);
    fp.stats = f->d_stats;
    fp.flags = f->d_flags;
    fp.list = f->d_list;
    fp.counters = f->d_counters;
    fp.sq = f->d_sq; // non-null: plan_launch picks the kernels that also sum the squares
    f->samples_done = fp.n_probe; // 0 without the early-out
    f->samples_target = fp.sample_end;
    int launches = 0;
    // with its own counter block, the frame's probe keeps the raw "means differ" flags, also where this target has no main
    // phase: the frame can be extended
    auto enqueue = [&]() -> int {
        int rc2 = frame_probe(ds, fp, st, &f->ev, &launches);
        if (rc2 != RT_OK) return rc2;
        if ((rc2 = launch_compact(ds, fp, single_flags(f->d_flags), f->d_list, st, &launches)) != RT_OK) return rc2;
        RT_CUDA(f->ev.record(FrameEvents::TRACED, st));
        return frame_sync(f, st);
    };
    if ((rc = enqueue()) != RT_OK) return bail(rc);
    f->pixels_flagged = f->pixels_active = f->h_counters[CN_LIST];
    f->device_ms = f->ev.ms(FrameEvents::ZEROED, FrameEvents::TRACED);
    // the probe traced n_probe samples of every pixel; a pass traces samples of the flagged pixels only
    if (fp.adaptive) f->ms_per_sample = f->device_ms * double(f->pixels_flagged) / (double(n) * double(fp.n_probe));
    *out = f;
    frame_progress(f, progress);
    return RT_OK;
}

// rt_frame_view_noise reduces at most this many views per launch: the grid's y extent stays far below its limit (65535),
// and the partials stay at most 16.8 MB however many views a batch of small extents has
constexpr int32_t kNoiseViewChunk = 1024;

// the noise reductions' partial summaries, kNoiseBlocks + 1 per view of one chunk of views, allocated on first use
int ensure_partials(RtFrame *f) {
    const size_t views = size_t(std::min(f->n_views, kNoiseViewChunk));
    if (!f->d_partial) RT_CUDA(cudaMalloc((void **)&f->d_partial, views * (kNoiseBlocks + 1) * sizeof(NoisePartial)));
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

// the refusals of both openers, after their own argument checks
int check_frame_mode(const RtRenderOpts *opts, const char *who) {
    if (opts->mode == RT_MODE_WAVEFRONT) return fail(RT_ERR_UNSUPPORTED, std::string(who) + ": progressive frames run the megakernel only");
    if (opts->mode != RT_MODE_MEGAKERNEL) return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": unknown mode");
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
    if ((rc = check_frame_mode(opts, "rt_frame_begin")) != RT_OK) return rc;
    if ((opts->flags & RT_FLAG_NOISE) && (opts->flags & (RT_FLAG_FLOW | RT_FLAG_COUNTERS)))
        return fail(RT_ERR_UNSUPPORTED, "rt_frame_begin: RT_FLAG_NOISE has no flow-schedule or counting kernel");
    return frame_open(scene, *camera, {}, nullptr, max_w, max_h, opts, out, progress, "rt_frame_begin");
}

int rt_frame_begin_views(RtScene *scene, const RtCamera *cameras, const uint64_t *seeds, int32_t n_views, int32_t max_w, int32_t max_h,
                         const RtRenderOpts *opts, RtFrame **out, RtFrameProgress *progress) {
    // rt_render_views' checks, then rt_frame_begin's
    if (n_views < 1) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_begin_views: n_views must be >= 1");
    if (!cameras) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_begin_views: cameras is null");
    int rc = check_frame_args(scene, &cameras[0], max_w, max_h, opts);
    if (rc != RT_OK) return rc;
    for (int32_t v = 1; v < n_views; ++v)
        if (cameras[v].samples_per_pixel != cameras[0].samples_per_pixel || cameras[v].bounce_depth != cameras[0].bounce_depth)
            return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_begin_views: every camera must have the same samples_per_pixel and bounce_depth");
    if (size_t(2 * max_w + 1) * size_t(2 * max_h + 1) * size_t(n_views) >= (size_t(1) << 31))
        return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_begin_views: n_views x rows x cols must be below 2^31");
    if (!out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_begin_views: out is null");
    *out = nullptr;
    if ((rc = check_frame_mode(opts, "rt_frame_begin_views")) != RT_OK) return rc;
    if (opts->flags & (RT_FLAG_FLOW | RT_FLAG_COUNTERS))
        return fail(RT_ERR_UNSUPPORTED, "rt_frame_begin_views: a batch of views has no flow-schedule or counting kernel");
    std::vector<ViewCamera> table(n_views);
    for (int32_t v = 0; v < n_views; ++v) {
        const uint64_t seed = seeds ? seeds[v] : opts->seed;
        table[v].cam = make_dev_camera(cameras[v], max_w, max_h);
        table[v].k0 = uint32_t(seed);
        table[v].k1 = uint32_t(seed >> 32);
    }
    return frame_open(scene, cameras[0], table, nullptr, max_w, max_h, opts, out, progress, "rt_frame_begin_views");
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
    if ((rc = check_frame_mode(opts, "rt_frame_begin_window")) != RT_OK) return rc;
    if (opts->flags & (RT_FLAG_FLOW | RT_FLAG_COUNTERS))
        return fail(RT_ERR_UNSUPPORTED, "rt_frame_begin_window: a window has no flow-schedule or counting kernel");
    return frame_open(scene, *camera, {}, &w, max_w, max_h, opts, out, progress, "rt_frame_begin_window");
}

int rt_frame_advance(RtFrame *f, int32_t max_samples, double target_ms, RtFrameProgress *progress) {
    if (!f) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_advance: null frame");
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
            k = std::min(k, std::max(1, paced));
        }
        if (rule) k = int(std::min<int64_t>(k, next_checkpoint(f) - f->samples_done)); // a pass never crosses a checkpoint
        const bool check = rule && f->samples_done + k == next_checkpoint(f);
        auto *ds = static_cast<DeviceScene *>(f->scene->dev);
        RT_CUDA(cudaSetDevice(ds->device));
        cudaStream_t st = ds->ws->stream;
        FrameParams fp = f->fp;
        fp.sample_begin = f->samples_done;
        fp.sample_end = f->samples_done + k;
        int launches = 0;
        RT_CUDA(cudaMemsetAsync(f->d_counters + CN_WORK_MAIN, 0, sizeof(unsigned long long), st));
        RT_CUDA(f->ev.record(FrameEvents::BEGIN, st));
        int rc = launch_samples(ds, fp, st, &launches);
        if (rc != RT_OK) return rc;
        if (check) { // the pass ends on a checkpoint: stop the converged pixels and list the others
            converge_kernel<<<unsigned((f->n_pixels + 255) / 256), 256, 0, st>>>(reinterpret_cast<const int4 *>(f->d_stats), f->d_sq, f->d_flags,
                                                                                 f->n_pixels, f->conv_tolerance);
            RT_CUDA(cudaGetLastError());
            if ((rc = launch_compact(ds, fp, single_flags(f->d_flags), f->d_list, st, &launches)) != RT_OK) return rc;
        }
        RT_CUDA(f->ev.record(FrameEvents::END, st));
        if ((rc = frame_sync(f, st)) != RT_OK) return rc;
        f->samples_done += k;
        f->passes += 1;
        f->last_pass_ms = f->ev.ms(FrameEvents::BEGIN, FrameEvents::END);
        f->device_ms += f->last_pass_ms;
        const uint64_t before = f->pixels_active;
        if (check) {
            f->pixels_active = f->h_counters[CN_LIST];
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
    if (!f->d_sq) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_noise: the frame was opened without RT_FLAG_NOISE");
    if (!(tolerance >= 0.0)) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_noise: tolerance must be >= 0");
    auto *ds = static_cast<DeviceScene *>(f->scene->dev);
    RT_CUDA(cudaSetDevice(ds->device));
    cudaStream_t st = ds->ws->stream;
    int rc = ensure_partials(f);
    if (rc != RT_OK) return rc;
    if (se_out && !f->d_se) RT_CUDA(cudaMalloc((void **)&f->d_se, f->n_pixels * sizeof(float)));
    noise_kernel<<<kNoiseBlocks, kNoiseThreads, 0, st>>>(reinterpret_cast<const int4 *>(f->d_stats), f->d_sq, f->d_flags, f->n_pixels, tolerance,
                                                         se_out ? f->d_se : nullptr, f->d_partial);
    RT_CUDA(cudaGetLastError());
    noise_summary_kernel<<<1, kNoiseThreads, 0, st>>>(f->d_partial);
    RT_CUDA(cudaGetLastError());
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
    if (!f->d_sq) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_view_noise: the frame was opened without RT_FLAG_NOISE");
    if (!(tolerance >= 0.0)) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_view_noise: tolerance must be >= 0");
    auto *ds = static_cast<DeviceScene *>(f->scene->dev);
    RT_CUDA(cudaSetDevice(ds->device));
    cudaStream_t st = ds->ws->stream;
    int rc = ensure_partials(f);
    if (rc != RT_OK) return rc;
    // every view reduced as rt_frame_noise reduces a frame of its pixels: the same 512 ranges, tree and block order
    const size_t view_pixels = f->n_pixels / size_t(f->n_views);
    std::vector<NoisePartial> totals(size_t(f->n_views));
    for (int32_t v0 = 0; v0 < f->n_views; v0 += kNoiseViewChunk) {
        const int32_t nv = std::min(kNoiseViewChunk, f->n_views - v0);
        const size_t at = size_t(v0) * view_pixels;
        noise_kernel<<<dim3(kNoiseBlocks, unsigned(nv)), kNoiseThreads, 0, st>>>(reinterpret_cast<const int4 *>(f->d_stats) + at, f->d_sq + at,
                                                                                  f->d_flags + at, view_pixels, tolerance, nullptr, f->d_partial);
        RT_CUDA(cudaGetLastError());
        noise_summary_kernel<<<unsigned(nv), kNoiseThreads, 0, st>>>(f->d_partial);
        RT_CUDA(cudaGetLastError());
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
    if (!f->d_sq) return fail(RT_ERR_INVALID_ARGUMENT, "rt_frame_denoise: the frame was opened without RT_FLAG_NOISE");
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

} // extern "C"
