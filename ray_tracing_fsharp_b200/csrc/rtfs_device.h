// rtfs_device.h — declarations shared by the device translation units of librtfs_b200.so.
#pragma once
#include "rtfs_core.cuh"

#include <string>
#include <vector>

namespace rtfs {

// ---------------------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------------------
#define RT_CUDA(expr)                                                                                         \
    do {                                                                                                      \
        cudaError_t e__ = (expr);                                                                             \
        if (e__ != cudaSuccess)                                                                               \
            return fail(RT_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));                    \
    } while (0)

inline int require_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        cudaGetLastError();
        return fail(RT_ERR_NO_DEVICE, "no CUDA device is visible: librtfs_b200 has no CPU fallback");
    }
    if (device < 0 || device >= n) return fail(RT_ERR_INVALID_ARGUMENT, "CUDA device ordinal out of range");
    RT_CUDA(cudaSetDevice(device));
    return RT_OK;
}

// ---------------------------------------------------------------------------------------------------
// device scene
// ---------------------------------------------------------------------------------------------------
enum CounterSlot { CN_PATHS = 0, CN_RAYS = 1, CN_BOX = 2, CN_PRIM = 3, CN_LIST = 4, CN_WORK_PROBE = 5, CN_WORK_MAIN = 6, CN_DEGENERATE = 7, CN_BUSY_BLOCKS = 8, CN_SLOTS = 16 };
// (the last slot of the pinned copy is a scratch word of the wavefront driver; the pinned buffer holds a second set of
// CN_SLOTS words: the snapshot taken between the probe and the main phase)

// The events a frame records on its stream, in stream order: BEGIN; ZEROED once the counters and sums are cleared;
// MAIN_BEGIN and MAIN_END around the main phase; TRACED once the last render kernel is done; END once the results and
// the counters are copied.  RtStats: kernel_ms = ZEROED -> TRACED, main_ms = MAIN_BEGIN -> MAIN_END, total_ms = BEGIN -> END.
struct FrameEvents {
    enum Which { BEGIN, ZEROED, MAIN_BEGIN, MAIN_END, TRACED, END, COUNT };
    cudaEvent_t ev[COUNT] = {};
    bool create() {
        bool ok = true;
        for (auto &e : ev) ok = ok && cudaEventCreate(&e) == cudaSuccess;
        return ok;
    }
    void destroy() {
        for (auto &e : ev)
            if (e) cudaEventDestroy(e);
    }
    cudaError_t record(Which w, cudaStream_t st) { return cudaEventRecord(ev[w], st); }
    float ms(Which from, Which to) const {
        float t = 0.f;
        cudaEventElapsedTime(&t, ev[from], ev[to]);
        return t;
    }
};

// one view of a batch (rt_render_views): its camera and its Philox key
struct ViewCamera {
    DevCamera cam;
    uint32_t k0, k1;
};

// Frame buffers, scratch, stream and events of one device.  Allocating these costs milliseconds, so they are
// pooled: a scene handle borrows one for its lifetime and returns it on destroy (handles stay independent of
// one another; nothing is shared between two live handles).
struct DeviceWorkspace {
    int device = 0;
    int sm_count = 0;
    size_t smem_optin = 0;
    size_t probe_pixels = 0; // second accumulator set of the probe phase
    int32_t *d_stats_b = nullptr;
    size_t ws_pixels = 0; // frame buffers of rt_render
    int32_t *d_stats = nullptr;
    uint8_t *d_flags = nullptr;
    uint8_t *d_rgb = nullptr;
    size_t list_pixels = 0; // flagged-pixel list of the main phase
    uint32_t *d_list = nullptr;
    // the scene blob of the handle that holds this workspace, and its pinned staging copy: pooled with the workspace so
    // that creating a scene costs one copy, not a cudaMalloc / cudaFree pair (grow-only)
    void *d_blob = nullptr;
    void *h_blob = nullptr;
    size_t blob_cap = 0;
    size_t views_cap = 0; // the per-view cameras and keys of rt_render_views
    ViewCamera *d_views = nullptr;
    unsigned long long *d_counters = nullptr;
    unsigned long long *h_counters = nullptr; // pinned
    cudaStream_t stream = nullptr;
    FrameEvents ev;
};
int workspace_acquire(int device, DeviceWorkspace **out);
void workspace_release(DeviceWorkspace *ws);
// grow-only: the sums, flags and RGB8 of rt_render's frame; the flagged-pixel list; the probe's second accumulator set
int ensure_frame_buffers(DeviceWorkspace *ws, size_t n_pixels);
int ensure_list(DeviceWorkspace *ws, size_t n_pixels);
int ensure_probe_sums(DeviceWorkspace *ws, size_t n_pixels);

struct PooledTexture { // an image texture's array + texture object, pooled by (device, width, height)
    int device, w, h;
    cudaArray_t array;
    cudaTextureObject_t object;
};
struct DeviceScene {
    int device = 0;
    SceneGlobal g{};
    DRefNode *ref_nodes = nullptr;
    int32_t n_ref_nodes = 0;
    void *blob = nullptr; // nodes | spheres | materials | unbounded | textures, in the workspace's pooled allocation (not owned)
    void *wide_blob = nullptr; // the 8-wide compressed tree: nodes | spheres in its order | the two index maps
    int32_t wide_depth = 0;
    std::vector<PooledTexture> images; // image textures borrowed from the pool
    size_t bytes = 0;
    int32_t max_depth = 0; // depth of the tree: the walk's stack never holds more entries
    bool lean = false;     // no FP64 unbounded object, no texture index: the staged kernels have a variant without that code
    DeviceWorkspace *ws = nullptr;
};

constexpr int kTileW = 8, kTileH = 4; // a warp's 32 pixels
constexpr int kMaxChunks = 192;
constexpr int kMaxChunkSamples = 256;                    // samples of one pixel in a work item (16-bit colour sums: 256 x 255 < 2^16)
constexpr int kMaxLaunchSamples = 160 * kMaxChunkSamples; // sample indices of one rank a single main-phase launch covers (build_chunks)
// Launch shape of the render kernels (measured on B200, DESIGN.md 5).
//   scene staged in shared memory: ONE persistent block of 1024 threads per SM at 64 registers per thread.  That kernel is bound
//     by instruction issue and its walk loop wants the registers (896 threads at 72 registers and 2 x 640 at 48 both lost);
//   scene read from global memory / L2 (big scenes): TWO blocks of 768 threads per SM at 40 registers per thread.  That kernel
//     waits on L2 (long-scoreboard stalls), so 48 warps per SM hide more latency than 32: 100 k spheres at 32 spp 219 -> 203 ms;
//     the spills land outside the walk loop.  (2 x 640 at 48 registers: 211 ms; 2 x 1024 at 32: 253 ms, spills inside the loop.)
// The macros exist for A/B builds.
#ifndef RTFS_BLOCK_THREADS
#define RTFS_BLOCK_THREADS 1024
#endif
#ifndef RTFS_BLOCKS_PER_SM
#define RTFS_BLOCKS_PER_SM 1
#endif
#ifndef RTFS_GLOBAL_BLOCK_THREADS
#define RTFS_GLOBAL_BLOCK_THREADS 768
#endif
#ifndef RTFS_GLOBAL_BLOCKS_PER_SM
#define RTFS_GLOBAL_BLOCKS_PER_SM 2
#endif
#ifndef RTFS_ITEM_SLOTS
#define RTFS_ITEM_SLOTS 4
#endif
#ifndef RTFS_GLOBAL_ITEM_SLOTS
#define RTFS_GLOBAL_ITEM_SLOTS 4
#endif
constexpr int kBlockThreads = RTFS_BLOCK_THREADS;
constexpr int kBlocksPerSm = RTFS_BLOCKS_PER_SM;
constexpr int kGlobalBlockThreads = RTFS_GLOBAL_BLOCK_THREADS;
constexpr int kGlobalBlocksPerSm = RTFS_GLOBAL_BLOCKS_PER_SM;
// Work-item slots per warp (rtfs_device.cu, 400 bytes each, 528 with the sum of squares of RT_FLAG_NOISE).  Four keep a warp fed best: on the 100 k-sphere scene (two blocks of
// 768 threads per SM) four slots 199.5 ms, three 202, two 222 (warps run dry).
constexpr int kItemSlots = RTFS_ITEM_SLOTS, kGlobalItemSlots = RTFS_GLOBAL_ITEM_SLOTS;
constexpr int item_slots(bool staged) { return staged ? kItemSlots : kGlobalItemSlots; }
constexpr int block_threads(bool staged) { return staged ? kBlockThreads : kGlobalBlockThreads; }
constexpr int blocks_per_sm(bool staged) { return staged ? kBlocksPerSm : kGlobalBlocksPerSm; }

struct FrameParams {
    SceneGlobal g;
    DevCamera cam;
    uint32_t k0, k1;
    int32_t rank, world;
    int32_t tiles_x, tiles_y;
    int32_t first_trial;  // min 5 (spp / 2), Scene.fs:172
    int32_t n_probe;      // 2 * first_trial + 1
    int32_t sample_begin; // first sample index of the main phase
    int32_t sample_end;   // one past the last
    int32_t adaptive;
    // work items: (unit, chunk k) where a unit is 32 pixels and chunk k covers this rank's local sample indices
    // [chunk_begin[k], chunk_begin[k] + chunk_len[k]); chunks are sorted by decreasing length and items are
    // numbered chunk-major, so the persistent warps meet the long items first and the short ones last
    int32_t n_chunks;
    uint32_t chunk_begin[kMaxChunks];
    uint32_t chunk_len[kMaxChunks];
    int32_t *stats;       // rows*cols*4 {sumR, sumG, sumB, count}
    int32_t *stats_b;     // probe phase: sums of the samples after the first firstTrial + 1 (same layout)
    uint8_t *flags;       // rows*cols
    const uint32_t *list; // flagged pixel ids (main phase)
    unsigned long long *counters;
    // shared-memory staging
    uint32_t s_nodes, s_spheres, s_mats, s_warp; // offsets in uint4 units
    uint32_t s_stack; // SSTACK kernels: the walk stacks, one column of `stack_levels` words per thread (uint4 units)
    int32_t opt_flags; // RtRenderOpts.flags
    int32_t stack_levels; // words per thread of the shared-memory walk stacks
    int32_t quantum;      // flow kernel: node visits between two schedule points
    // last, so that no other parameter moves: rows*cols per-pixel sums of r^2 + g^2 + b^2 over the pixel's samples
    // (progressive frames opened with RT_FLAG_NOISE; null otherwise, and then the kernels without that sum run)
    unsigned long long *sq;
    // a batch of views (rt_render_views, rtfs_views.cu): n_views views of view_pixels pixels each, stacked as one tall frame
    // (cam.rows = n_views x the rows of a view), and the camera and key of every view; null otherwise, and then the kernels
    // of one frame run
    const ViewCamera *views;
    int32_t n_views;
    int32_t view_pixels;
    // a window of rt_render's frame (rt_render_window, rt_frame_begin_window: rtfs_window.cu): cam.rows x cam.cols are the
    // window's, at row win_row0 and column win_col0 of the (2 max_h + 1) x (2 max_w + 1) frame; window = 0 otherwise, and
    // then the kernels of one frame run
    int32_t window;
    int32_t win_row0, win_col0;
};

// a window of rt_render's frame: rows x cols pixels from (row0, col0), counted as rt_render's output (row 0 = top row)
struct FrameWindow {
    int32_t row0, col0, rows, cols;
};
// RT_ERR_INVALID_ARGUMENT unless the window is non-empty and lies inside the (2 max_h + 1) x (2 max_w + 1) frame
int check_window(const FrameWindow &w, int max_w, int max_h, const char *who);
// narrows a frame filled by fill_frame to the window: probe tiles, flags, list, sums and the output tail run over its pixels
void set_window(FrameParams &fp, const FrameWindow &w);


constexpr int kMaxDevices = 16;
// where the main phase finds the probe flags: one buffer (single device, or already combined by the
// caller's all-reduce), or one buffer per rank, each holding the flags of the tiles that rank probed
struct FlagsView {
    const uint8_t *by_rank[kMaxDevices];
    int32_t world;
};
inline FlagsView single_flags(const uint8_t *p) {
    FlagsView v{};
    v.by_rank[0] = p;
    v.world = 1;
    return v;
}

int check_frame_args(const RtScene *scene, const RtCamera *camera, int max_w, int max_h, const RtRenderOpts *opts);
void fill_frame(FrameParams &fp, DeviceScene *ds, const RtCamera &cam, int max_w, int max_h, const RtRenderOpts &opts, int rank, int world);
// The launch helpers pick their kernels from fp.opt_flags (RT_FLAG_COUNTERS, RT_FLAG_NO_SMEM, ...) and count what they
// launch in *launches.
// raw_flags: flag every pixel whose two probe means differ even where the frame has no main phase (progressive frames
// keep them so that the frame can be extended to more samples); otherwise only where a main phase follows
int launch_probe(DeviceScene *ds, FrameParams fp, cudaStream_t st, int *launches, bool raw_flags);
// merges the probe's two accumulator sets (fp.stats += stats_b) and raises fp.flags on the pixels of this rank's tiles
// whose two means differ (more: only if samples follow)
int launch_probe_flags(const FrameParams &fp, const int32_t *stats_b, bool more, cudaStream_t st, int *launches);
// compaction + the main phase over [fp.sample_begin, fp.sample_end); the two halves are also launched on their own
// (progressive frames, rtfs_frame.cu: compaction once, then one launch_samples per pass)
int launch_main(DeviceScene *ds, FrameParams fp, const FlagsView &flags, cudaStream_t st, int *launches);
int launch_compact(DeviceScene *ds, const FrameParams &fp, const FlagsView &flags, uint32_t *list, cudaStream_t st, int *launches);
int launch_samples(DeviceScene *ds, FrameParams fp, cudaStream_t st, int *launches);
// the kernel of a batch of views (rtfs_views.cu) for the launch plan_launch has decided: scene staged in shared memory
// (and lean), or read from global memory with shared or local walk stacks over the binary or the 8-wide tree; with noise,
// the kernel that also sums the squares (progressive frames of a batch opened with RT_FLAG_NOISE)
typedef void (*RenderKernelFn)(const FrameParams);
RenderKernelFn pick_views_kernel(bool probe, bool smem, bool lean, bool sstack, bool wide, bool noise);
// the same choice among the kernels of a window of one frame (rtfs_window.cu)
RenderKernelFn pick_window_kernel(bool probe, bool smem, bool lean, bool sstack, bool wide, bool noise);
// PixelStats.mean + the optional gamma of a whole frame: sums -> RGB8
int launch_finalize(const int32_t *stats, size_t n_pixels, int gamma, uint8_t *rgb, cudaStream_t st, int *launches);

// One rank's frame, in three steps on its stream; fp.stats, fp.flags and fp.counters (and fp.sq) are the frame's.
// frame_probe: BEGIN, zero the counters, the sums (and fp.sq), ZEROED, then the probe, or every flag raised without the
//   early-out.  A split probe (fp.world > 1) writes the flags of its own tiles only, so the others are cleared first;
//   a frame with its own counter block (progressive frames) keeps the raw flags.  ev may be null: no events.
// frame_main: the counter snapshot into ws->h_counters + CN_SLOTS, MAIN_BEGIN, compaction + samples over the flags in
//   fp.flags, MAIN_END, TRACED.
// frame_finish: RGB8 (from d_rgb) and sums to the host if asked, the counters into ws->h_counters, END.
int frame_probe(DeviceScene *ds, const FrameParams &fp, cudaStream_t st, FrameEvents *ev, int *launches);
int frame_main(DeviceScene *ds, const FrameParams &fp, cudaStream_t st, FrameEvents &ev, int *launches);
int frame_finish(DeviceScene *ds, const FrameParams &fp, const uint8_t *d_rgb, uint8_t *rgb_out, int32_t *sums_out, cudaStream_t st,
                 FrameEvents &ev);
// RtStats from the counters last copied into ds->ws->h_counters; with ev, also the frame's times and main_rays
void read_stats(const DeviceScene *ds, size_t n_pixels, bool adaptive, int launches, const FrameEvents *ev, RtStats *stats);

// The tail of a frame split over ranks, for one rank's slice of the pixels: sum the ranks' sums (peer loads over NVLink),
// truncating mean, gamma, RGB8 into each of rgb[0, n_rgb) and, if given, the summed int4 into sums.  Four pixels per
// thread, so that the RGB8 stores are whole 32-bit words.  (rtfs_multi.cu)
struct ReduceTargets {
    const int32_t *stats[kMaxDevices];
    int32_t world;
    uint8_t *rgb[kMaxDevices];
    int32_t n_rgb;
    int32_t *sums;
};
int launch_reduce_finalize(const ReduceTargets &t, int rank, size_t n_pixels, int gamma, cudaStream_t st, int *launches);

// PixelOutput.correct (ImageOutput.fs:11-18): the block fills `lut` with the 8-bit output of every mean, gamma or not
__device__ __forceinline__ void fill_gamma_lut(uint8_t *lut, int gamma) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        int v = i;
        if (gamma) {
            v = __double2int_rn(sqrt(double(i) / 255.0) * 255.0); // Math.Round: half to even
            if (v == 256) v = 255;
        }
        lut[i] = uint8_t(v);
    }
    __syncthreads();
}
// PixelStats.mean (Pixel.fs:103-108): the truncating mean of each channel, through the table
__device__ __forceinline__ void pixel_rgb8(int4 s, const uint8_t *lut, uint8_t *out) {
    int n = s.w > 0 ? s.w : 1;
    out[0] = lut[(s.x / n) & 255];
    out[1] = lut[(s.y / n) & 255];
    out[2] = lut[(s.z / n) & 255];
}

// E of a pixel from its moments: n samples, channel sums t0..t2, sum of squares q (include/rtfs_b200.h, rt_frame_noise).
// D = n q - sum t_c^2 is exact in int64 for n <= 2^22 (each term < 3.5e18); the double arithmetic is the same, in the same
// order, on the device and on the host (rt_pixel_noise), and IEEE division and square root round correctly on both.
__host__ __device__ __forceinline__ double pixel_standard_error(int32_t n, int32_t t0, int32_t t1, int32_t t2, uint64_t q) {
    if (n < 2) return HUGE_VAL;
    // unsigned wrap-around arithmetic, then the int64 value: the same bits as the signed formula wherever that is defined
    const uint64_t tt = uint64_t(int64_t(t0) * t0) + uint64_t(int64_t(t1) * t1) + uint64_t(int64_t(t2) * t2);
    const int64_t d = int64_t(uint64_t(n) * q - tt);
    const double nd = double(n);
    return sqrt(double(d) / (3.0 * nd * nd * double(n - 1)));
}

// ---------------------------------------------------------------------------------------------------
// denoised previews of progressive frames (rtfs_denoise.cu; rt_frame_features, rt_frame_denoise)
// ---------------------------------------------------------------------------------------------------
constexpr int kMaxDenoiseIterations = 10, kMaxFeatureSamples = 64;
// per pixel, in rt_frame_features' layouts: prim n, albedo n*3, normal n*3, depth n
struct FrameFeatures {
    int32_t *prim;
    uint8_t *albedo;
    float *normal;
    float *depth;
};
// the first-hit features of sample indices [0, samples) of the n_pixels pixels of the frame fp describes (one camera, a
// batch of views or a window)
int launch_features(const FrameParams &fp, size_t n_pixels, int samples, const FrameFeatures &out, cudaStream_t st);
// RT_ERR_INVALID_ARGUMENT unless every option of rt_frame_denoise is in range
int check_denoise_opts(const RtDenoiseOpts *o, const char *who);
// the filter over a frame's sums and Q, views of view_rows rows each: buf holds 2 n_pixels float4 (the two levels); the RGB8
// and the linear output it was asked for are left in device memory at *d_rgb and *d_linear (inside buf)
int launch_denoise(const int32_t *stats, const unsigned long long *sq, const FrameFeatures &feat, size_t n_pixels, int view_rows, int cols,
                   const RtDenoiseOpts &o, float4 *buf, bool want_rgb, bool want_linear, uint8_t **d_rgb, float **d_linear, cudaStream_t st);

// makes sure the tree the frame will walk is on the device (the wide tree is built on first use for small scenes)
int prepare_frame(RtScene *scene, const RtRenderOpts *opts);
bool frame_walks_wide_tree(const DeviceScene *ds, int opt_flags, bool smem_fits);

inline DevCamera make_dev_camera(const RtCamera &c, int max_w, int max_h) {
    DevCamera d{};
    d.ox = float(c.view_origin[0]); d.oy = float(c.view_origin[1]); d.oz = float(c.view_origin[2]);
    d.cx = float(c.xaxis_origin[0] - c.view_origin[0]);
    d.cy = float(c.xaxis_origin[1] - c.view_origin[1]);
    d.cz = float(c.xaxis_origin[2] - c.view_origin[2]);
    d.xx = float(c.xaxis_dir[0]); d.xy = float(c.xaxis_dir[1]); d.xz = float(c.xaxis_dir[2]);
    d.yx = float(c.yaxis_dir[0]); d.yy = float(c.yaxis_dir[1]); d.yz = float(c.yaxis_dir[2]);
    d.sx = float(c.viewport_width / double(max_w));
    d.sy = float(c.viewport_height / double(max_h));
    d.max_w = max_w;
    d.max_h = max_h;
    d.rows = 2 * max_h + 1; // Scene.fs:208-209
    d.cols = 2 * max_w + 1;
    d.spp = c.samples_per_pixel;
    d.depth = c.bounce_depth;
    return d;
}


} // namespace rtfs
