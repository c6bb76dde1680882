// rtfs_multi.cu — one frame or one batch of views split over several GPUs of this process (rt_multi_*, rt_render_multi).
//
// Replicated scene, sample-index split (SURVEY.md §8e).  The devices exchange data only through NVLink
// peer memory, inside the kernels that need it:
//   probe    : device r probes the tiles t with t mod world == r (Scene.fs:172-188), writing sums and
//              flags into its own buffers;
//   compact  : every device builds the flagged-pixel list reading each tile's flags from the owner's
//              buffer with peer loads;
//   main     : device r adds its share (sample index mod world == r) of the remaining samples of every
//              flagged pixel into its own sum buffer (Scene.fs:191-192);
//   reduce + finalize (one kernel): device r sums the world's buffers for its slice of the pixels with
//              128-bit peer loads, divides (PixelStats.mean, Pixel.fs:103-108), applies the optional
//              gamma (ImageOutput.fs:11-18) and stores RGB8 straight into pinned host memory.
// Integer sums keyed by sample index make the image bit-identical for every device count.
// rt_multi_render_views runs the same sequence over rt_render_views' tall frame of a batch of views: the split, the
// exchange and the reduce work per pixel, and every rank reads the table of view cameras and keys from its own device.
// (The one-process-per-GPU form of the same split, with NCCL all-reduces between rt_device_probe /
// rt_device_main / rt_device_finalize, is driven from bench.py through torch.distributed.)
#include "rtfs_device.h"

#include <chrono>
#include <cstdlib>
#include <cstring>
#include <memory>

struct RtMulti {
    std::vector<int> devices;
    std::vector<RtScene *> scenes;
    std::vector<int32_t *> d_stats;
    std::vector<uint8_t *> d_flags;
    std::vector<cudaStream_t> streams;
    std::vector<cudaEvent_t> ev_begin, ev_probe, ev_main, ev_end;
    size_t ws_pixels = 0;
    uint8_t *h_rgb = nullptr;  // pinned, portable
    int32_t *h_sums = nullptr; // pinned, portable (only when sums are requested)
    size_t h_sums_pixels = 0;
};

namespace rtfs {
namespace {

__global__ void reduce_finalize_kernel(const ReduceTargets t, int n_pixels, int quad_begin, int quad_end, int gamma) {
    __shared__ uint8_t lut[256];
    fill_gamma_lut(lut, gamma);
    const int quad = quad_begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (quad >= quad_end) return;
    uint8_t out[12];
    const int n_valid = min(4, n_pixels - 4 * quad);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int px = 4 * quad + k;
        int4 s = make_int4(0, 0, 0, 0);
        if (k < n_valid) {
            for (int r = 0; r < t.world; ++r) {
                const int4 v = reinterpret_cast<const int4 *>(t.stats[r])[px];
                s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
            }
            if (t.sums) reinterpret_cast<int4 *>(t.sums)[px] = s;
        }
        pixel_rgb8(s, lut, out + 3 * k);
    }
    const uint32_t w0 = uint32_t(out[0]) | (uint32_t(out[1]) << 8) | (uint32_t(out[2]) << 16) | (uint32_t(out[3]) << 24);
    const uint32_t w1 = uint32_t(out[4]) | (uint32_t(out[5]) << 8) | (uint32_t(out[6]) << 16) | (uint32_t(out[7]) << 24);
    const uint32_t w2 = uint32_t(out[8]) | (uint32_t(out[9]) << 8) | (uint32_t(out[10]) << 16) | (uint32_t(out[11]) << 24);
    for (int r = 0; r < t.n_rgb; ++r) {
        if (n_valid == 4) {
            uint32_t *dst = reinterpret_cast<uint32_t *>(t.rgb[r] + 12 * size_t(quad));
            dst[0] = w0; dst[1] = w1; dst[2] = w2;
        } else {
            for (int k = 0; k < 3 * n_valid; ++k) t.rgb[r][12 * size_t(quad) + k] = out[k];
        }
    }
}

// A progressive frame's exchange (launch_gather): four pixels per thread, so that every rank's sums are four 128-bit peer
// loads, its Q two, and its four probe flags one 32-bit load (flags are 0 or 1 bytes, so OR-ing the words ORs the pixels).
__global__ void gather_kernel(const GatherTargets t, size_t n_pixels, size_t quad_begin, size_t quad_end) {
    const size_t quad = quad_begin + size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (quad >= quad_end) return;
    const size_t p0 = 4 * quad;
    if (p0 + 4 <= n_pixels) {
        int4 s[4];
        ulonglong2 q[2];
#pragma unroll
        for (int k = 0; k < 4; ++k) s[k] = make_int4(0, 0, 0, 0);
        q[0] = q[1] = make_ulonglong2(0ull, 0ull);
        uint32_t f = 0;
        for (int r = 0; r < t.world; ++r) {
            const int4 *src = reinterpret_cast<const int4 *>(t.stats[r]) + p0;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int4 v = src[k];
                s[k].x += v.x; s[k].y += v.y; s[k].z += v.z; s[k].w += v.w;
            }
            if (t.total_sq) {
                const ulonglong2 *qs = reinterpret_cast<const ulonglong2 *>(t.sq[r] + p0);
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    const ulonglong2 v = qs[k];
                    q[k].x += v.x; q[k].y += v.y;
                }
            }
            if (t.total_flags) f |= *reinterpret_cast<const uint32_t *>(t.flags[r] + p0);
        }
        int4 *dst = reinterpret_cast<int4 *>(t.total_stats) + p0;
#pragma unroll
        for (int k = 0; k < 4; ++k) dst[k] = s[k];
        if (t.total_sq) {
            reinterpret_cast<ulonglong2 *>(t.total_sq + p0)[0] = q[0];
            reinterpret_cast<ulonglong2 *>(t.total_sq + p0)[1] = q[1];
        }
        if (t.total_flags) *reinterpret_cast<uint32_t *>(t.total_flags + p0) = f;
        return;
    }
    for (size_t p = p0; p < n_pixels; ++p) { // the last quad of a frame whose size is not a multiple of four
        int4 s = make_int4(0, 0, 0, 0);
        unsigned long long q = 0;
        uint8_t f = 0;
        for (int r = 0; r < t.world; ++r) {
            const int4 v = reinterpret_cast<const int4 *>(t.stats[r])[p];
            s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
            if (t.total_sq) q += t.sq[r][p];
            if (t.total_flags) f |= t.flags[r][p];
        }
        reinterpret_cast<int4 *>(t.total_stats)[p] = s;
        if (t.total_sq) t.total_sq[p] = q;
        if (t.total_flags) t.total_flags[p] = f;
    }
}

void multi_free(RtMulti *m) {
    if (!m) return;
    for (size_t i = 0; i < m->devices.size(); ++i) {
        cudaSetDevice(m->devices[i]);
        if (i < m->d_stats.size()) cudaFree(m->d_stats[i]);
        if (i < m->d_flags.size()) cudaFree(m->d_flags[i]);
        if (i < m->ev_begin.size() && m->ev_begin[i]) cudaEventDestroy(m->ev_begin[i]);
        if (i < m->ev_probe.size() && m->ev_probe[i]) cudaEventDestroy(m->ev_probe[i]);
        if (i < m->ev_main.size() && m->ev_main[i]) cudaEventDestroy(m->ev_main[i]);
        if (i < m->ev_end.size() && m->ev_end[i]) cudaEventDestroy(m->ev_end[i]);
        if (i < m->streams.size() && m->streams[i]) cudaStreamDestroy(m->streams[i]);
    }
    if (m->h_rgb) cudaFreeHost(m->h_rgb);
    if (m->h_sums) cudaFreeHost(m->h_sums);
    for (RtScene *s : m->scenes) rt_scene_destroy(s);
    delete m;
}

int multi_workspace(RtMulti *m, size_t n_pixels, bool want_sums) {
    const size_t n = m->devices.size();
    if (m->ws_pixels < n_pixels) {
        for (size_t i = 0; i < n; ++i) {
            RT_CUDA(cudaSetDevice(m->devices[i]));
            cudaFree(m->d_stats[i]);
            cudaFree(m->d_flags[i]);
            m->d_stats[i] = nullptr;
            m->d_flags[i] = nullptr;
        }
        if (m->h_rgb) cudaFreeHost(m->h_rgb);
        m->h_rgb = nullptr;
        m->ws_pixels = 0;
        for (size_t i = 0; i < n; ++i) {
            RT_CUDA(cudaSetDevice(m->devices[i]));
            RT_CUDA(cudaMalloc((void **)&m->d_stats[i], n_pixels * 4 * sizeof(int32_t)));
            RT_CUDA(cudaMalloc((void **)&m->d_flags[i], n_pixels));
        }
        RT_CUDA(cudaHostAlloc((void **)&m->h_rgb, n_pixels * 3 + 16, cudaHostAllocPortable | cudaHostAllocMapped));
        m->ws_pixels = n_pixels;
    }
    if (want_sums && m->h_sums_pixels < n_pixels) {
        if (m->h_sums) cudaFreeHost(m->h_sums);
        m->h_sums = nullptr;
        m->h_sums_pixels = 0;
        RT_CUDA(cudaHostAlloc((void **)&m->h_sums, n_pixels * 4 * sizeof(int32_t), cudaHostAllocPortable | cudaHostAllocMapped));
        m->h_sums_pixels = n_pixels;
    }
    return RT_OK;
}

// rt_multi_render's body, once its arguments are checked: one frame (views empty), or rt_render_views' tall frame of a
// batch (views: the table of every view's camera and key).  Every rank uploads the table into its replica's workspace
// (ws->d_views, on its own device), so the render kernels read every view's camera and key from local memory; the probe,
// the compaction, the main phase and the reduce then run over the tall frame as over one frame.
int multi_render(RtMulti *m, const RtCamera &camera, const std::vector<ViewCamera> &views, int32_t max_w, int32_t max_h,
                 const RtRenderOpts *opts, uint8_t *rgb_out, int32_t *sums_out, RtStats *stats) {
    const auto t0 = std::chrono::steady_clock::now();
    const int world = int(m->devices.size());
    const size_t view_pixels = size_t(2 * max_w + 1) * size_t(2 * max_h + 1);
    const size_t n_pixels = view_pixels * std::max<size_t>(1, views.size());
    int rc = multi_workspace(m, n_pixels, sums_out != nullptr);
    if (rc != RT_OK) return rc;
    for (RtScene *s : m->scenes)
        if ((rc = prepare_frame(s, opts)) != RT_OK) return rc;
    std::vector<int> launches(world, 0);
    std::vector<FrameParams> fps(world);
    FlagsView flags{};
    flags.world = world;
    for (int i = 0; i < world; ++i) flags.by_rank[i] = m->d_flags[i];

    // phase 1 on every device
    for (int i = 0; i < world; ++i) {
        auto *ds = static_cast<DeviceScene *>(m->scenes[i]->dev);
        RT_CUDA(cudaSetDevice(m->devices[i]));
        cudaStream_t st = m->streams[i];
        fill_frame(fps[i], ds, camera, max_w, max_h, *opts, i, world);
        if (!views.empty()) { // (from pageable memory: staged before the call returns, and the probe follows it on the stream)
            if ((rc = ensure_views(ds->ws, views.size())) != RT_OK) return rc;
            RT_CUDA(cudaMemcpyAsync(ds->ws->d_views, views.data(), views.size() * sizeof(ViewCamera), cudaMemcpyHostToDevice, st));
            set_views(fps[i], ds->ws->d_views, int32_t(views.size()), int32_t(view_pixels));
        }
        fps[i].stats = m->d_stats[i];
        fps[i].flags = m->d_flags[i];
        RT_CUDA(cudaEventRecord(m->ev_begin[i], st));
        if ((rc = frame_probe(ds, fps[i], st, nullptr, &launches[i])) != RT_OK) return rc;
        RT_CUDA(cudaEventRecord(m->ev_probe[i], st));
    }
    // phase 2: needs everyone's flags
    for (int i = 0; i < world; ++i) {
        auto *ds = static_cast<DeviceScene *>(m->scenes[i]->dev);
        RT_CUDA(cudaSetDevice(m->devices[i]));
        cudaStream_t st = m->streams[i];
        for (int j = 0; j < world; ++j)
            if (j != i) RT_CUDA(cudaStreamWaitEvent(st, m->ev_probe[j], 0));
        if ((rc = launch_main(ds, fps[i], flags, st, &launches[i])) != RT_OK) return rc;
        RT_CUDA(cudaMemcpyAsync(ds->ws->h_counters, ds->ws->d_counters, CN_SLOTS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        RT_CUDA(cudaEventRecord(m->ev_main[i], st));
    }
    // reduce + finalize: needs everyone's sums; each device owns a slice of the pixels
    ReduceTargets t{};
    for (int j = 0; j < world; ++j) t.stats[j] = m->d_stats[j];
    t.world = world;
    t.n_rgb = 1;
    for (int i = 0; i < world; ++i) {
        RT_CUDA(cudaSetDevice(m->devices[i]));
        cudaStream_t st = m->streams[i];
        for (int j = 0; j < world; ++j)
            if (j != i) RT_CUDA(cudaStreamWaitEvent(st, m->ev_main[j], 0));
        RT_CUDA(cudaHostGetDevicePointer((void **)&t.rgb[0], m->h_rgb, 0));
        if (sums_out) RT_CUDA(cudaHostGetDevicePointer((void **)&t.sums, m->h_sums, 0));
        if ((rc = launch_reduce_finalize(t, i, n_pixels, opts->gamma, st, &launches[i])) != RT_OK) return rc;
        RT_CUDA(cudaEventRecord(m->ev_end[i], st));
    }
    for (int i = 0; i < world; ++i) {
        RT_CUDA(cudaSetDevice(m->devices[i]));
        RT_CUDA(cudaStreamSynchronize(m->streams[i]));
    }
    std::memcpy(rgb_out, m->h_rgb, n_pixels * 3);
    if (sums_out) std::memcpy(sums_out, m->h_sums, n_pixels * 4 * sizeof(int32_t));
    if (stats) {
        std::memset(stats, 0, sizeof *stats);
        for (int i = 0; i < world; ++i) {
            RtStats d;
            read_stats(static_cast<DeviceScene *>(m->scenes[i]->dev), n_pixels, opts->adaptive != 0, launches[i], nullptr, &d);
            stats->paths += d.paths;
            stats->rays += d.rays;
            stats->box_tests += d.box_tests;
            stats->prim_tests += d.prim_tests;
            stats->degenerate_paths += d.degenerate_paths;
            stats->launches += d.launches;
            stats->pixels_early_out = d.pixels_early_out; // every device compacted the same flags
            float ms = 0.f;
            cudaEventElapsedTime(&ms, m->ev_begin[i], m->ev_end[i]);
            stats->kernel_ms = std::max(stats->kernel_ms, double(ms)); // device time of the slowest GPU, probe -> reduce
        }
        stats->total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
    return RT_OK;
}

} // namespace

int launch_reduce_finalize(const ReduceTargets &t, int rank, size_t n_pixels, int gamma, cudaStream_t st, int *launches) {
    const long long n_quads = (long long)(n_pixels + 3) / 4;
    const int quad_begin = int(n_quads * rank / t.world), quad_end = int(n_quads * (rank + 1) / t.world);
    if (quad_end <= quad_begin) return RT_OK;
    reduce_finalize_kernel<<<(quad_end - quad_begin + 255) / 256, 256, 0, st>>>(t, int(n_pixels), quad_begin, quad_end, gamma);
    RT_CUDA(cudaGetLastError());
    ++*launches;
    return RT_OK;
}

int launch_gather(const GatherTargets &t, int rank, size_t n_pixels, cudaStream_t st) {
    const size_t n_quads = (n_pixels + 3) / 4;
    const size_t quad_begin = n_quads * size_t(rank) / size_t(t.world), quad_end = n_quads * size_t(rank + 1) / size_t(t.world);
    if (quad_end <= quad_begin) return RT_OK;
    gather_kernel<<<unsigned((quad_end - quad_begin + 255) / 256), 256, 0, st>>>(t, n_pixels, quad_begin, quad_end);
    RT_CUDA(cudaGetLastError());
    return RT_OK;
}

const std::vector<RtScene *> &multi_scenes(const RtMulti *m) { return m->scenes; }

} // namespace rtfs

using namespace rtfs;

extern "C" {

int rt_multi_create(const RtHittable *objects, int32_t n_objects, const RtTexture *textures, int32_t n_textures, const int32_t *devices,
                    int32_t n_devices, RtMulti **out) {
    if (!out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_multi_create: out is null");
    *out = nullptr;
    if (!devices || n_devices < 1 || n_devices > kMaxDevices) return fail(RT_ERR_INVALID_ARGUMENT, "rt_multi_create: 1..16 devices");
    int visible = rt_device_count();
    if (visible <= 0) return fail(RT_ERR_NO_DEVICE, "no CUDA device is visible: librtfs_b200 has no CPU fallback");
    // RTFS_MULTI_SHARE_DEVICES (tests): ranks may share a device, so that the split, its exchange and its cross-stream
    // ordering run on a machine with fewer GPUs than ranks; each rank still has its own replica, workspace and stream
    const bool share = std::getenv("RTFS_MULTI_SHARE_DEVICES") != nullptr;
    for (int i = 0; i < n_devices; ++i) {
        if (devices[i] < 0 || devices[i] >= visible) return fail(RT_ERR_INVALID_ARGUMENT, "rt_multi_create: device ordinal out of range");
        for (int j = 0; j < i; ++j)
            if (devices[j] == devices[i] && !share) return fail(RT_ERR_INVALID_ARGUMENT, "rt_multi_create: duplicate device");
    }
    // every device must be able to read every other device's buffers (NVLink / NVSwitch peer access)
    for (int i = 0; i < n_devices; ++i) {
        RT_CUDA(cudaSetDevice(devices[i]));
        for (int j = 0; j < n_devices; ++j) {
            if (devices[i] == devices[j]) continue;
            int can = 0;
            RT_CUDA(cudaDeviceCanAccessPeer(&can, devices[i], devices[j]));
            if (!can) return fail(RT_ERR_UNSUPPORTED, "rt_multi_create: devices without peer access cannot share a frame");
            cudaError_t e = cudaDeviceEnablePeerAccess(devices[j], 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
            else if (e != cudaSuccess) return fail(RT_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
        }
    }
    auto *m = new RtMulti();
    m->devices.assign(devices, devices + n_devices);
    m->d_stats.assign(n_devices, nullptr);
    m->d_flags.assign(n_devices, nullptr);
    m->streams.assign(n_devices, nullptr);
    m->ev_begin.assign(n_devices, nullptr);
    m->ev_probe.assign(n_devices, nullptr);
    m->ev_main.assign(n_devices, nullptr);
    m->ev_end.assign(n_devices, nullptr);
    for (int i = 0; i < n_devices; ++i) {
        RtScene *s = nullptr;
        int rc = rt_scene_create(objects, n_objects, textures, n_textures, devices[i], &s);
        if (rc != RT_OK) {
            multi_free(m);
            return rc;
        }
        m->scenes.push_back(s);
        if (cudaSetDevice(devices[i]) != cudaSuccess || cudaStreamCreateWithFlags(&m->streams[i], cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreate(&m->ev_begin[i]) != cudaSuccess || cudaEventCreate(&m->ev_probe[i]) != cudaSuccess ||
            cudaEventCreate(&m->ev_main[i]) != cudaSuccess || cudaEventCreate(&m->ev_end[i]) != cudaSuccess) {
            multi_free(m);
            return fail(RT_ERR_CUDA, "rt_multi_create: stream / event creation failed");
        }
    }
    *out = m;
    return RT_OK;
}

void rt_multi_destroy(RtMulti *multi) { multi_free(multi); }

int rt_multi_render(RtMulti *m, const RtCamera *camera, int32_t max_w, int32_t max_h, const RtRenderOpts *opts, uint8_t *rgb_out,
                    int32_t *sums_out, RtStats *stats) {
    if (!m || m->scenes.empty()) return fail(RT_ERR_INVALID_ARGUMENT, "rt_multi_render: null handle");
    int rc = check_frame_args(m->scenes[0], camera, max_w, max_h, opts);
    if (rc != RT_OK) return rc;
    if (!rgb_out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_multi_render: rgb_out is null");
    if (opts->mode != RT_MODE_MEGAKERNEL) return fail(RT_ERR_UNSUPPORTED, "rt_multi_render: only RT_MODE_MEGAKERNEL is split over devices");
    return multi_render(m, *camera, {}, max_w, max_h, opts, rgb_out, sums_out, stats);
}

int rt_multi_render_views(RtMulti *m, const RtCamera *cameras, const uint64_t *seeds, int32_t n_views, int32_t max_w, int32_t max_h,
                          const RtRenderOpts *opts, uint8_t *rgb_out, int32_t *sums_out, RtStats *stats) {
    // the union of rt_multi_render's and rt_render_views' checks, before any device work
    if (!m || m->scenes.empty()) return fail(RT_ERR_INVALID_ARGUMENT, "rt_multi_render_views: null handle");
    if (!rgb_out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_multi_render_views: rgb_out is null");
    int rc = check_views(m->scenes[0], cameras, n_views, max_w, max_h, opts, "rt_multi_render_views");
    if (rc != RT_OK) return rc;
    if ((rc = check_frame_mode(opts, "rt_multi_render_views", true)) != RT_OK) return rc;
    return multi_render(m, cameras[0], view_table(cameras, seeds, n_views, max_w, max_h, opts->seed), max_w, max_h, opts, rgb_out, sums_out,
                        stats);
}

int rt_render_multi(const RtHittable *objects, int32_t n_objects, const RtTexture *textures, int32_t n_textures, const int32_t *devices,
                    int32_t n_devices, const RtCamera *camera, int32_t max_w, int32_t max_h, const RtRenderOpts *opts, uint8_t *rgb_out,
                    int32_t *sums_out, RtStats *stats) {
    RtMulti *m = nullptr;
    int rc = rt_multi_create(objects, n_objects, textures, n_textures, devices, n_devices, &m);
    if (rc != RT_OK) return rc;
    rc = rt_multi_render(m, camera, max_w, max_h, opts, rgb_out, sums_out, stats);
    std::string keep = rt_last_error();
    rt_multi_destroy(m);
    if (rc != RT_OK) set_error(keep);
    return rc;
}

} // extern "C"
