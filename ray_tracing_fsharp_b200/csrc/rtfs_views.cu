// rtfs_views.cu — rt_render_views: n views of one scene (same extents and samples per pixel; camera and seed per view) in
// one submission.  The views are stacked as one tall frame of n_views x rows rows, global pixel P = v rows cols + r cols + c,
// and that frame runs rt_render's sequence once: one probe, one compaction, one main phase, one finalize, one device->host
// copy and one synchronisation.  The only new device work is here: the render kernel's item loop (rtfs_items.cuh) with a
// lane's pixel mapped to its view's camera and key, so that view v is bit for bit rt_render of camera v and seed v.
#include "rtfs_items.cuh"

#include <cstring>
#include <vector>

namespace rtfs {

// The generator of a path of a batch: CounterRng's draws, with the key of the path's view and the pixel word of its pixel
// within the view, both found from the tall-frame pixel P it holds.  (Holding the key itself would keep two more words live
// through the whole item loop, where render_kernel reads its one key from the kernel parameters: those words spill.)
struct ViewRng {
    uint32_t P, sample, bounce, retry;
    const ViewCamera *views;
    uint32_t view_pixels;
    __device__ __forceinline__ float4 next() {
        const uint32_t v = P / view_pixels;
        const ViewCamera *vc = views + v;
        uint4 w = philox4x32_10(make_uint4(P - v * view_pixels, sample, bounce, retry), vc->k0, vc->k1);
        ++retry;
        return make_float4(u01(w.x), u01(w.y), u01(w.z), u01(w.w));
    }
};

// A slot holds the tall frame's pixel id P itself: render_kernel's row << 16 | col stops at row 65535, and a tall frame
// passes it.  A path starts at P's local (r, c) from its view's camera, so its RNG pixel word is rt_render's r cols + c.
// A probe tile straddles two views where rows % 4 != 0: every lane finds its own view.
struct ViewPixels {
    using Path = PathStateT<ViewRng>;
    const FrameParams &fp;
    __device__ __forceinline__ int pack(int pixel) const { return pixel; }
    __device__ __forceinline__ size_t index(int P) const { return size_t(P); }
    __device__ __forceinline__ bool begin(Path &ps, int P, uint32_t sample) const {
        const int v = P / fp.view_pixels, p = P - v * fp.view_pixels;
        const int r = p / fp.cam.cols, c = p - r * fp.cam.cols;
        ps.rng.P = uint32_t(P);
        ps.rng.sample = sample;
        ps.rng.views = fp.views;
        ps.rng.view_pixels = uint32_t(fp.view_pixels);
        return path_start(ps, fp.views[v].cam, r, c);
    }
};

// The lockstep kernels without counters, as render_kernel<PROBE, SMEM, false, SSTACK, WIDE>, over a batch of views.
template <bool PROBE, int SMEM, bool SSTACK, bool WIDE>
__global__ void __launch_bounds__(block_threads(SMEM), blocks_per_sm(SMEM)) render_views_kernel(const FrameParams fp) {
    render_items<PROBE, SMEM, false, SSTACK, WIDE, false>(fp, ViewPixels{fp});
}

// The same twelve shapes that also sum r^2 + g^2 + b^2 per pixel into fp.sq, as render_kernel<..., NOISE = true>: the
// progressive frames of a batch opened with RT_FLAG_NOISE (rt_frame_begin_views).  A kernel of its own rather than a
// parameter of render_views_kernel, whose twelve instantiations stay what they are.
template <bool PROBE, int SMEM, bool SSTACK, bool WIDE>
__global__ void __launch_bounds__(block_threads(SMEM), blocks_per_sm(SMEM)) render_views_noise_kernel(const FrameParams fp) {
    render_items<PROBE, SMEM, false, SSTACK, WIDE, true>(fp, ViewPixels{fp});
}

template <bool PROBE, int SMEM, bool SSTACK, bool WIDE>
static RenderKernelFn pick_noise(bool noise) {
    return noise ? render_views_noise_kernel<PROBE, SMEM, SSTACK, WIDE> : render_views_kernel<PROBE, SMEM, SSTACK, WIDE>;
}
template <bool PROBE>
static RenderKernelFn pick_views(bool smem, bool lean, bool sstack, bool wide, bool noise) {
    if (smem) return lean ? pick_noise<PROBE, 2, false, false>(noise) : pick_noise<PROBE, 1, false, false>(noise);
    if (wide) return sstack ? pick_noise<PROBE, 0, true, true>(noise) : pick_noise<PROBE, 0, false, true>(noise);
    return sstack ? pick_noise<PROBE, 0, true, false>(noise) : pick_noise<PROBE, 0, false, false>(noise);
}
RenderKernelFn pick_views_kernel(bool probe, bool smem, bool lean, bool sstack, bool wide, bool noise) {
    return probe ? pick_views<true>(smem, lean, sstack, wide, noise) : pick_views<false>(smem, lean, sstack, wide, noise);
}

// grow-only, like the frame buffers
static int ensure_views(DeviceWorkspace *ws, size_t n_views) {
    if (ws->views_cap >= n_views) return RT_OK;
    cudaFree(ws->d_views);
    ws->d_views = nullptr;
    ws->views_cap = 0;
    RT_CUDA(cudaMalloc((void **)&ws->d_views, n_views * sizeof(ViewCamera)));
    ws->views_cap = n_views;
    return RT_OK;
}

} // namespace rtfs

using namespace rtfs;

extern "C" {

int rt_render_views(RtScene *scene, const RtCamera *cameras, const uint64_t *seeds, int32_t n_views, int32_t max_w, int32_t max_h,
                    const RtRenderOpts *opts, uint8_t *rgb_out, int32_t *sums_out, RtStats *stats) {
    if (n_views < 1) return fail(RT_ERR_INVALID_ARGUMENT, "rt_render_views: n_views must be >= 1");
    if (!cameras || !rgb_out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_render_views: cameras or rgb_out is null");
    int rc = check_frame_args(scene, &cameras[0], max_w, max_h, opts);
    if (rc != RT_OK) return rc;
    // the probe's firstTrial, the chunk table and the bounce budget are the batch's
    for (int32_t v = 1; v < n_views; ++v)
        if (cameras[v].samples_per_pixel != cameras[0].samples_per_pixel || cameras[v].bounce_depth != cameras[0].bounce_depth)
            return fail(RT_ERR_INVALID_ARGUMENT, "rt_render_views: every camera must have the same samples_per_pixel and bounce_depth");
    const size_t view_pixels = size_t(2 * max_w + 1) * size_t(2 * max_h + 1);
    const size_t n_pixels = view_pixels * size_t(n_views);
    if (n_pixels >= (size_t(1) << 31)) return fail(RT_ERR_INVALID_ARGUMENT, "rt_render_views: n_views x rows x cols must be below 2^31");
    if (opts->mode == RT_MODE_WAVEFRONT) return fail(RT_ERR_UNSUPPORTED, "rt_render_views: a batch of views runs the megakernel only");
    if (opts->mode != RT_MODE_MEGAKERNEL) return fail(RT_ERR_INVALID_ARGUMENT, "rt_render_views: unknown mode");
    if (opts->flags & (RT_FLAG_FLOW | RT_FLAG_COUNTERS))
        return fail(RT_ERR_UNSUPPORTED, "rt_render_views: a batch of views has no flow-schedule or counting kernel");
    if ((rc = prepare_frame(scene, opts)) != RT_OK) return rc;
    auto *ds = static_cast<DeviceScene *>(scene->dev);
    RT_CUDA(cudaSetDevice(ds->device));
    DeviceWorkspace *ws = ds->ws;
    if ((rc = ensure_frame_buffers(ws, n_pixels)) != RT_OK) return rc;
    if ((rc = ensure_views(ws, size_t(n_views))) != RT_OK) return rc;
    cudaStream_t st = ws->stream;
    std::vector<ViewCamera> table(n_views);
    for (int32_t v = 0; v < n_views; ++v) {
        const uint64_t seed = seeds ? seeds[v] : opts->seed;
        table[v].cam = make_dev_camera(cameras[v], max_w, max_h);
        table[v].k0 = uint32_t(seed);
        table[v].k1 = uint32_t(seed >> 32);
    }
    // (from pageable memory: the call returns once the table is staged, so it may go out of scope)
    RT_CUDA(cudaMemcpyAsync(ws->d_views, table.data(), table.size() * sizeof(ViewCamera), cudaMemcpyHostToDevice, st));
    FrameParams fp;
    fill_frame(fp, ds, cameras[0], max_w, max_h, *opts, 0, 1);
    fp.cam.rows *= n_views; // the tall frame: probe tiles, flags, list and sums run over it as over one frame
    fp.tiles_y = (fp.cam.rows + kTileH - 1) / kTileH;
    fp.views = ws->d_views;
    fp.n_views = n_views;
    fp.view_pixels = int32_t(view_pixels);
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
