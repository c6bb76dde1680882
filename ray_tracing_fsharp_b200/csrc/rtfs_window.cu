// rtfs_window.cu — rt_render_window: a window [row0, row0 + rows) x [col0, col0 + cols) of rt_render's frame, bit for bit,
// in one call (and the progressive frame of that window, rt_frame_begin_window in rtfs_frame.cu).  The window runs
// rt_render's sequence over its own pixels: fp.cam.rows x fp.cam.cols are the window's, so the probe tiles, the flags, the
// list, the sums and the output tail cover the window only.  The only new device work is here: the render kernel's item
// loop (rtfs_items.cuh) with a lane's window pixel mapped back to its place in the frame, where its path starts and from
// which its RNG pixel word comes.  A path is a pure function of (seed, frame pixel word, sample index) and the camera's full
// extents, and the probe flag of a pixel depends on its own samples only, so no bit of a window pixel depends on the window.
#include "rtfs_items.cuh"

#include <cstdint>

namespace rtfs {

// A slot holds the window's pixel id p itself.  A path starts at the frame's (R, C) = (win_row0 + r, win_col0 + c) with the
// frame's key and rt_render's pixel word R (2 max_w + 1) + C; path_begin cannot be used, since it forms that word from
// cam.cols, which here is the window's width.  One camera and one key: the generator is CounterRng, as in render_kernel,
// and nothing is added per draw.
struct WindowPixels {
    using Path = PathState;
    const FrameParams &fp;
    __device__ __forceinline__ int pack(int pixel) const { return pixel; }
    __device__ __forceinline__ size_t index(int p) const { return size_t(p); }
    __device__ __forceinline__ bool begin(PathState &ps, int p, uint32_t sample) const {
        const int r = p / fp.cam.cols, c = p - r * fp.cam.cols;
        const int R = fp.win_row0 + r, C = fp.win_col0 + c;
        ps.rng.k0 = fp.k0;
        ps.rng.k1 = fp.k1;
        ps.rng.pixel = uint32_t(R * (2 * fp.cam.max_w + 1) + C);
        ps.rng.sample = sample;
        return path_start(ps, fp.cam, R, C);
    }
};

// The lockstep kernels without counters, as render_kernel<PROBE, SMEM, false, SSTACK, WIDE>, over a window of a frame.
template <bool PROBE, int SMEM, bool SSTACK, bool WIDE>
__global__ void __launch_bounds__(block_threads(SMEM), blocks_per_sm(SMEM)) render_window_kernel(const FrameParams fp) {
    render_items<PROBE, SMEM, false, SSTACK, WIDE, false>(fp, WindowPixels{fp});
}

// The same twelve shapes that also sum r^2 + g^2 + b^2 per pixel into fp.sq, as render_kernel<..., NOISE = true>: the
// progressive frames of a window opened with RT_FLAG_NOISE.
template <bool PROBE, int SMEM, bool SSTACK, bool WIDE>
__global__ void __launch_bounds__(block_threads(SMEM), blocks_per_sm(SMEM)) render_window_noise_kernel(const FrameParams fp) {
    render_items<PROBE, SMEM, false, SSTACK, WIDE, true>(fp, WindowPixels{fp});
}

template <bool PROBE, int SMEM, bool SSTACK, bool WIDE>
static RenderKernelFn pick_noise(bool noise) {
    return noise ? render_window_noise_kernel<PROBE, SMEM, SSTACK, WIDE> : render_window_kernel<PROBE, SMEM, SSTACK, WIDE>;
}
template <bool PROBE>
static RenderKernelFn pick_window(bool smem, bool lean, bool sstack, bool wide, bool noise) {
    if (smem) return lean ? pick_noise<PROBE, 2, false, false>(noise) : pick_noise<PROBE, 1, false, false>(noise);
    if (wide) return sstack ? pick_noise<PROBE, 0, true, true>(noise) : pick_noise<PROBE, 0, false, true>(noise);
    return sstack ? pick_noise<PROBE, 0, true, false>(noise) : pick_noise<PROBE, 0, false, false>(noise);
}
RenderKernelFn pick_window_kernel(bool probe, bool smem, bool lean, bool sstack, bool wide, bool noise) {
    return probe ? pick_window<true>(smem, lean, sstack, wide, noise) : pick_window<false>(smem, lean, sstack, wide, noise);
}

int check_window(const FrameWindow &w, int max_w, int max_h, const char *who) {
    if (w.rows < 1 || w.cols < 1) return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": rows and cols must be >= 1");
    if (w.row0 < 0 || w.col0 < 0) return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": row0 and col0 must be >= 0");
    if (int64_t(w.row0) + w.rows > 2 * int64_t(max_h) + 1 || int64_t(w.col0) + w.cols > 2 * int64_t(max_w) + 1)
        return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": the window must lie inside the (2 max_h + 1) x (2 max_w + 1) frame");
    return RT_OK;
}

void set_window(FrameParams &fp, const FrameWindow &w) {
    fp.cam.rows = w.rows;
    fp.cam.cols = w.cols;
    fp.tiles_x = (w.cols + kTileW - 1) / kTileW;
    fp.tiles_y = (w.rows + kTileH - 1) / kTileH;
    fp.window = 1;
    fp.win_row0 = w.row0;
    fp.win_col0 = w.col0;
}

} // namespace rtfs

using namespace rtfs;

extern "C" {

int rt_render_window(RtScene *scene, const RtCamera *camera, int32_t max_w, int32_t max_h, int32_t row0, int32_t col0, int32_t rows,
                     int32_t cols, const RtRenderOpts *opts, uint8_t *rgb_out, int32_t *sums_out, RtStats *stats) {
    const FrameWindow w{row0, col0, rows, cols};
    int rc = check_window(w, max_w, max_h, "rt_render_window");
    if (rc != RT_OK) return rc;
    if (!rgb_out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_render_window: rgb_out is null");
    if ((rc = check_frame_args(scene, camera, max_w, max_h, opts)) != RT_OK) return rc;
    if (opts->mode == RT_MODE_WAVEFRONT) return fail(RT_ERR_UNSUPPORTED, "rt_render_window: a window runs the megakernel only");
    if (opts->mode != RT_MODE_MEGAKERNEL) return fail(RT_ERR_INVALID_ARGUMENT, "rt_render_window: unknown mode");
    if (opts->flags & (RT_FLAG_FLOW | RT_FLAG_COUNTERS))
        return fail(RT_ERR_UNSUPPORTED, "rt_render_window: a window has no flow-schedule or counting kernel");
    if ((rc = prepare_frame(scene, opts)) != RT_OK) return rc;
    auto *ds = static_cast<DeviceScene *>(scene->dev);
    RT_CUDA(cudaSetDevice(ds->device));
    DeviceWorkspace *ws = ds->ws;
    const size_t n_pixels = size_t(rows) * size_t(cols);
    if ((rc = ensure_frame_buffers(ws, n_pixels)) != RT_OK) return rc;
    cudaStream_t st = ws->stream;
    FrameParams fp;
    fill_frame(fp, ds, *camera, max_w, max_h, *opts, 0, 1);
    set_window(fp, w);
    fp.stats = ws->d_stats;
    fp.flags = ws->d_flags;
    int launches = 0;
    if ((rc = frame_probe(ds, fp, st, &ws->ev, &launches)) != RT_OK) return rc;
    if ((rc = frame_main(ds, fp, st, ws->ev, &launches)) != RT_OK) return rc;
    if ((rc = launch_finalize(ws->d_stats, n_pixels, opts->gamma, ws->d_rgb, st, &launches)) != RT_OK) return rc;
    if ((rc = frame_finish(ds, fp, ws->d_rgb, rgb_out, sums_out, st, ws->ev)) != RT_OK) return rc;
    RT_CUDA(cudaStreamSynchronize(st));
    if (stats) read_stats(ds, n_pixels, fp.adaptive != 0, launches, &ws->ev, stats);
    return RT_OK;
}

} // extern "C"
