// rtfs_device.cu — device half of librtfs_b200.so: scene upload, the render kernels (probe / compact /
// main / finalize), the per-primitive conformance kernels and the C-ABI entry points that launch them.
// Compiled for sm_100a only.  There is no CPU fallback: every entry point here needs a CUDA device.
#include "rtfs_core.cuh"
#include "rtfs_device.h"
#include "rtfs_items.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

namespace rtfs {

// ---------------------------------------------------------------------------------------------------
// workspace pool
// ---------------------------------------------------------------------------------------------------
static std::mutex g_pool_mutex;
static std::vector<DeviceWorkspace *> g_pool;

static void workspace_destroy(DeviceWorkspace *ws) {
    if (!ws) return;
    cudaSetDevice(ws->device);
    cudaFree(ws->d_stats);
    cudaFree(ws->d_flags);
    cudaFree(ws->d_rgb);
    cudaFree(ws->d_list);
    cudaFree(ws->d_views);
    cudaFree(ws->d_stats_b);
    cudaFree(ws->d_counters);
    cudaFree(ws->d_blob);
    if (ws->h_blob) cudaFreeHost(ws->h_blob);
    if (ws->h_counters) cudaFreeHost(ws->h_counters);
    ws->ev.destroy();
    if (ws->stream) cudaStreamDestroy(ws->stream);
    delete ws;
}

int workspace_acquire(int device, DeviceWorkspace **out) {
    *out = nullptr;
    {
        std::lock_guard<std::mutex> lock(g_pool_mutex);
        for (size_t i = 0; i < g_pool.size(); ++i)
            if (g_pool[i]->device == device) {
                *out = g_pool[i];
                g_pool.erase(g_pool.begin() + i);
                return RT_OK;
            }
    }
    auto *ws = new DeviceWorkspace();
    ws->device = device;
    cudaDeviceProp prop;
    bool ok = cudaGetDeviceProperties(&prop, device) == cudaSuccess;
    if (ok) {
        ws->sm_count = prop.multiProcessorCount;
        ws->smem_optin = prop.sharedMemPerBlockOptin;
        ok = cudaMalloc((void **)&ws->d_counters, CN_SLOTS * sizeof(unsigned long long)) == cudaSuccess &&
             cudaMallocHost((void **)&ws->h_counters, 2 * CN_SLOTS * sizeof(unsigned long long)) == cudaSuccess &&
             cudaStreamCreateWithFlags(&ws->stream, cudaStreamNonBlocking) == cudaSuccess && ws->ev.create();
    }
    if (!ok) {
        std::string why = cudaGetErrorString(cudaGetLastError());
        workspace_destroy(ws);
        return fail(RT_ERR_CUDA, "device workspace allocation failed: " + why);
    }
    *out = ws;
    return RT_OK;
}

void workspace_release(DeviceWorkspace *ws) {
    if (!ws) return;
    cudaSetDevice(ws->device);
    cudaStreamSynchronize(ws->stream);
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    if (g_pool.size() < 32) {
        g_pool.push_back(ws);
        return;
    }
    workspace_destroy(ws);
}

// Image textures: cudaMallocArray / cudaCreateTextureObject / their destructors cost milliseconds to tens of
// milliseconds, so arrays are pooled by (device, width, height) like the workspaces; a reused array is overwritten.
static std::vector<PooledTexture> g_texture_pool;

static bool texture_acquire(int device, int w, int h, PooledTexture &out) {
    {
        std::lock_guard<std::mutex> lock(g_pool_mutex);
        for (size_t i = 0; i < g_texture_pool.size(); ++i)
            if (g_texture_pool[i].device == device && g_texture_pool[i].w == w && g_texture_pool[i].h == h) {
                out = g_texture_pool[i];
                g_texture_pool.erase(g_texture_pool.begin() + i);
                return true;
            }
    }
    out = PooledTexture{device, w, h, nullptr, 0};
    cudaChannelFormatDesc desc = cudaCreateChannelDesc<uchar4>();
    if (cudaMallocArray(&out.array, &desc, w, h) != cudaSuccess) return false;
    cudaResourceDesc res;
    std::memset(&res, 0, sizeof res);
    res.resType = cudaResourceTypeArray;
    res.res.array.array = out.array;
    cudaTextureDesc td;
    std::memset(&td, 0, sizeof td);
    td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp;
    td.filterMode = cudaFilterModePoint;
    td.readMode = cudaReadModeElementType;
    td.normalizedCoords = 0;
    if (cudaCreateTextureObject(&out.object, &res, &td, nullptr) != cudaSuccess) {
        cudaFreeArray(out.array);
        return false;
    }
    return true;
}
static void texture_release(const PooledTexture &t) {
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    if (g_texture_pool.size() < 16) {
        g_texture_pool.push_back(t);
        return;
    }
    cudaSetDevice(t.device);
    cudaDestroyTextureObject(t.object);
    cudaFreeArray(t.array);
}

// ---------------------------------------------------------------------------------------------------
// device scene
// ---------------------------------------------------------------------------------------------------
void device_scene_free(RtScene *scene) {
    auto *ds = static_cast<DeviceScene *>(scene->dev);
    if (!ds) return;
    cudaSetDevice(ds->device);
    // rt_device_probe / rt_device_main / rt_comm_render launch on the caller's stream, not the workspace's: quiesce the whole
    // device before the workspace and the texture arrays go back to pools another handle may draw from at once
    cudaDeviceSynchronize();
    cudaFree(ds->ref_nodes);
    cudaFree(ds->wide_blob); // (the main blob lives in the workspace)
    if (ds->ws) workspace_release(ds->ws);
    for (const PooledTexture &t : ds->images) texture_release(t);
    delete ds;
    scene->dev = nullptr;
}

size_t device_scene_bytes(const RtScene *scene) {
    auto *ds = static_cast<const DeviceScene *>(scene->dev);
    return ds ? ds->bytes : 0;
}

int device_scene_upload(RtScene *scene) {
    int rc = require_device(scene->device);
    if (rc != RT_OK) return rc;
    auto *ds = new DeviceScene();
    scene->dev = ds;
    ds->device = scene->device;
    const HostSceneLayout &L = scene->layout;
    auto bail = [&](int code) {
        device_scene_free(scene);
        return code;
    };
    if ((rc = workspace_acquire(ds->device, &ds->ws)) != RT_OK) return bail(rc);

    // textures: image texels go into a cudaArray read through a texture object (point sampling)
    std::vector<DTexture> dt(scene->textures.size());
    for (size_t i = 0; i < scene->textures.size(); ++i) {
        const RtTexture &t = scene->textures[i];
        DTexture &o = dt[i];
        std::memset(&o, 0, sizeof o);
        o.kind = t.kind;
        o.rgb = (uint32_t(t.colour[0]) << 16) | (uint32_t(t.colour[1]) << 8) | uint32_t(t.colour[2]);
        o.w = t.width;
        o.h = t.height;
        o.even = t.even;
        o.odd = t.odd;
        o.grid = float(t.grid_size);
        o.cx = float(t.map_centre[0]);
        o.cy = float(t.map_centre[1]);
        o.cz = float(t.map_centre[2]);
        o.inv_radius = float(1.0 / (t.map_radius != 0.0 ? t.map_radius : 1.0));
        if (t.kind == RT_TEX_IMAGE) {
            std::vector<uchar4> texels(size_t(t.width) * t.height);
            for (size_t k = 0; k < texels.size(); ++k) texels[k] = make_uchar4(t.rgb8[3 * k], t.rgb8[3 * k + 1], t.rgb8[3 * k + 2], 255);
            PooledTexture pt;
            if (!texture_acquire(ds->device, t.width, t.height, pt)) return bail(fail(RT_ERR_CUDA, "texture allocation failed for an image texture"));
            ds->images.push_back(pt);
            if (cudaMemcpy2DToArray(pt.array, 0, 0, texels.data(), size_t(t.width) * sizeof(uchar4), size_t(t.width) * sizeof(uchar4), t.height,
                                    cudaMemcpyHostToDevice) != cudaSuccess)
                return bail(fail(RT_ERR_CUDA, "cudaMemcpy2DToArray failed for an image texture"));
            o.tex = pt.object;
            ds->bytes += texels.size() * sizeof(uchar4);
        }
    }

    // everything else travels as one blob: one allocation, one host->device copy
    auto align = [](size_t x) { return (x + 255) & ~size_t(255); };
    const size_t off_nodes = 0;
    const size_t off_spheres = align(off_nodes + L.nodes.size() * sizeof(DNode));
    const size_t off_mats = align(off_spheres + L.spheres.size() * sizeof(DSphere));
    const size_t off_unb = align(off_mats + L.materials.size() * sizeof(DMaterial));
    const size_t off_ref = align(off_unb + L.unbounded.size() * sizeof(DUnbounded));
    const size_t off_tex = off_ref;
    const size_t total = align(off_tex + dt.size() * sizeof(DTexture)) + 256;
    DeviceWorkspace *ws = ds->ws;
    if (ws->blob_cap < total) { // grow the pooled blob and its pinned staging copy
        cudaFree(ws->d_blob);
        if (ws->h_blob) cudaFreeHost(ws->h_blob);
        ws->d_blob = ws->h_blob = nullptr;
        ws->blob_cap = 0;
        const size_t cap = std::max<size_t>(total + total / 2, 256 << 10);
        if (cudaMalloc(&ws->d_blob, cap) != cudaSuccess || cudaMallocHost(&ws->h_blob, cap) != cudaSuccess) {
            cudaFree(ws->d_blob);
            ws->d_blob = nullptr;
            return bail(fail(RT_ERR_CUDA, "cudaMalloc failed for the scene"));
        }
        ws->blob_cap = cap;
    }
    uint8_t *host = static_cast<uint8_t *>(ws->h_blob);
    auto put = [&](size_t off, const void *src, size_t n) {
        if (n) std::memcpy(host + off, src, n);
    };
    { // the device walks centre / half-extent boxes (rtfs_internal.h)
        DNode *dn = reinterpret_cast<DNode *>(host + off_nodes);
        for (size_t i = 0; i < L.nodes.size(); ++i) dn[i] = device_node_of(L.nodes[i]);
    }
    put(off_spheres, L.spheres.data(), L.spheres.size() * sizeof(DSphere));
    put(off_mats, L.materials.data(), L.materials.size() * sizeof(DMaterial));
    put(off_unb, L.unbounded.data(), L.unbounded.size() * sizeof(DUnbounded));
    put(off_tex, dt.data(), dt.size() * sizeof(DTexture));
    ds->blob = ws->d_blob;
    if (cudaMemcpyAsync(ds->blob, host, total, cudaMemcpyHostToDevice, ws->stream) != cudaSuccess || cudaStreamSynchronize(ws->stream) != cudaSuccess)
        return bail(fail(RT_ERR_CUDA, "host->device copy of the scene failed"));
    ds->bytes += total;
    uint8_t *base = static_cast<uint8_t *>(ds->blob);
    ds->g.nodes = reinterpret_cast<const uint4 *>(base + off_nodes);
    ds->g.spheres = reinterpret_cast<const float4 *>(base + off_spheres);
    ds->g.mats = reinterpret_cast<const uint4 *>(base + off_mats);
    ds->g.unb = reinterpret_cast<const DUnbounded *>(base + off_unb);
    ds->g.tex = reinterpret_cast<const DTexture *>(base + off_tex);
    ds->g.n_nodes = int32_t(L.nodes.size());
    ds->g.n_bounded = L.n_bounded;
    ds->g.n_unbounded = int32_t(L.unbounded.size());
    ds->g.n_tex = int32_t(scene->textures.size());
    ds->max_depth = L.max_depth;
    // lean: nothing in this scene needs the FP64 evaluation of an unbounded object or a texture lookup (SceneAccess, rtfs_core.cuh)
    ds->lean = true;
    for (const DUnbounded &u : L.unbounded) ds->lean = ds->lean && u.fp32 == 1;
    for (const DMaterial &m : L.materials) ds->lean = ds->lean && m.texture < 0;
    if (!L.wide_nodes.empty()) return device_scene_ensure_wide(scene); // built at creation for big scenes
    return RT_OK;
}

// uploads the 8-wide compressed tree (building it first if the scene was too small to get one at creation)
int device_scene_ensure_wide(RtScene *scene) {
    auto *ds = static_cast<DeviceScene *>(scene->dev);
    if (!ds || ds->wide_blob || ds->g.n_bounded <= 0) return RT_OK;
    HostSceneLayout &L = scene->layout;
    build_wide_layout(L);
    if (L.wide_depth > 30) return fail(RT_ERR_UNSUPPORTED, "the wide BVH is deeper than the traversal stack");
    auto align = [](size_t x) { return (x + 255) & ~size_t(255); };
    const size_t off_nodes = 0;
    const size_t off_sph = align(L.wide_nodes.size() * sizeof(DWideNode));
    const size_t off_w2d = align(off_sph + L.wide_spheres.size() * sizeof(DSphere));
    const size_t off_d2w = align(off_w2d + L.wide_to_dev.size() * sizeof(int32_t));
    const size_t total = align(off_d2w + L.dev_to_wide.size() * sizeof(int32_t)) + 256;
    std::vector<uint8_t> host(total, 0);
    std::memcpy(host.data() + off_nodes, L.wide_nodes.data(), L.wide_nodes.size() * sizeof(DWideNode));
    std::memcpy(host.data() + off_sph, L.wide_spheres.data(), L.wide_spheres.size() * sizeof(DSphere));
    std::memcpy(host.data() + off_w2d, L.wide_to_dev.data(), L.wide_to_dev.size() * sizeof(int32_t));
    std::memcpy(host.data() + off_d2w, L.dev_to_wide.data(), L.dev_to_wide.size() * sizeof(int32_t));
    RT_CUDA(cudaSetDevice(ds->device));
    RT_CUDA(cudaMalloc(&ds->wide_blob, total));
    RT_CUDA(cudaMemcpy(ds->wide_blob, host.data(), total, cudaMemcpyHostToDevice));
    ds->bytes += total;
    uint8_t *base = static_cast<uint8_t *>(ds->wide_blob);
    ds->g.wide_nodes = reinterpret_cast<const uint4 *>(base + off_nodes);
    ds->g.wide_spheres = reinterpret_cast<const float4 *>(base + off_sph);
    ds->g.wide_to_dev = reinterpret_cast<const int32_t *>(base + off_w2d);
    ds->g.dev_to_wide = reinterpret_cast<const int32_t *>(base + off_d2w);
    ds->wide_depth = L.wide_depth;
    return RT_OK;
}

// which tree a frame walks: the binary SAH tree (staged in shared memory when the scene fits there, read from global
// memory otherwise) unless the caller asks for the 8-wide compressed one.  Measured on B200 (DESIGN.md 5): the wide
// walk executes more instructions per ray than the binary one (eight quantised boxes decoded and tested per visit for a
// third as many visits) and these kernels are issue-bound, not bandwidth-bound, so it is not the default for any size.
bool frame_walks_wide_tree(const DeviceScene *ds, int opt_flags, bool smem_fits) {
    (void)smem_fits;
    if (ds->g.n_bounded <= 0 || (opt_flags & RT_FLAG_BVH2)) return false;
    return (opt_flags & RT_FLAG_WIDE_BVH) != 0;
}
int prepare_frame(RtScene *scene, const RtRenderOpts *opts) {
    if (opts->flags & RT_FLAG_WIDE_BVH) return device_scene_ensure_wide(scene);
    return RT_OK;
}

// uploads the reference-topology tree the first time the conformance traversal asks for it
int device_scene_ensure_reference(RtScene *scene) {
    auto *ds = static_cast<DeviceScene *>(scene->dev);
    if (!ds || ds->ref_nodes) return RT_OK;
    scene_ensure_reference(scene);
    const auto &nodes = scene->layout.ref_nodes;
    RT_CUDA(cudaSetDevice(ds->device));
    RT_CUDA(cudaMalloc((void **)&ds->ref_nodes, std::max<size_t>(nodes.size(), 1) * sizeof(DRefNode)));
    if (!nodes.empty()) RT_CUDA(cudaMemcpy(ds->ref_nodes, nodes.data(), nodes.size() * sizeof(DRefNode), cudaMemcpyHostToDevice));
    ds->n_ref_nodes = int32_t(nodes.size());
    return RT_OK;
}

// ---------------------------------------------------------------------------------------------------
// render kernels
// ---------------------------------------------------------------------------------------------------
// rt_render's frame: a slot holds row << 16 | col of a pixel; every path starts from fp.cam with the frame's key
struct FramePixels {
    using Path = PathState;
    const FrameParams &fp;
    __device__ __forceinline__ int pack(int pixel) const { return ((pixel / fp.cam.cols) << 16) | (pixel % fp.cam.cols); }
    __device__ __forceinline__ size_t index(int rc) const { return size_t(rc >> 16) * size_t(fp.cam.cols) + size_t(rc & 0xffff); }
    __device__ __forceinline__ bool begin(PathState &ps, int rc, uint32_t sample) const {
        return path_begin(ps, fp.cam, fp.k0, fp.k1, rc >> 16, rc & 0xffff, sample);
    }
};

// The render kernel: the item loop of rtfs_items.cuh over one frame.
template <bool PROBE, int SMEM, bool COUNT, bool SSTACK, bool WIDE, bool NOISE = false>
__global__ void __launch_bounds__(block_threads(SMEM), blocks_per_sm(SMEM)) render_kernel(const FrameParams fp) {
    render_items<PROBE, SMEM, COUNT, SSTACK, WIDE, NOISE>(fp, FramePixels{fp});
}


#include "rtfs_flow.cuh" // render_flow_kernel: the flow schedule (RT_FLAG_FLOW)

// End of the probe phase (Scene.fs:177-188) for the tiles this rank owns: merge the two accumulator sets into
// `stats`, flag the pixels whose two truncated means differ (PixelStats.mean Pixel.fs:103-108, Pixel.difference :113-116)
__global__ void probe_flags_kernel(int32_t *stats, const int32_t *stats_b, uint8_t *flags, int rows, int cols, int tiles_x, int rank, int world,
                                   int first_trial, int n_probe, int more) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= rows * cols) return;
    int r = p / cols, c = p - r * cols;
    int tile = (r / kTileH) * tiles_x + c / kTileW;
    if (tile % world != rank) return;
    int4 a = reinterpret_cast<int4 *>(stats)[p], b = reinterpret_cast<const int4 *>(stats_b)[p];
    int n_old = first_trial + 1;
    int4 s = make_int4(a.x + b.x, a.y + b.y, a.z + b.z, n_probe);
    int diff = abs(s.x / n_probe - a.x / n_old) + abs(s.y / n_probe - a.y / n_old) + abs(s.z / n_probe - a.z / n_old);
    reinterpret_cast<int4 *>(stats)[p] = s;
    flags[p] = (diff != 0 && more) ? 1 : 0;
}

// flags -> list of flagged pixel ids, one warp per 8x4 tile so that list neighbours are image neighbours
// (with several devices in one process the flag of a tile is read from its owner's buffer over NVLink)
__global__ void compact_kernel(const FlagsView flags, uint32_t *list, unsigned long long *counters, int rows, int cols, int tiles_x,
                               int tiles_y) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int tile = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; tile < tiles_x * tiles_y; tile += warps) {
        int ty = tile / tiles_x, tx = tile - ty * tiles_x;
        int r = ty * kTileH + (lane >> 3), c = tx * kTileW + (lane & 7);
        const uint8_t *owner = flags.by_rank[flags.world > 1 ? tile % flags.world : 0];
        bool f = (r < rows && c < cols) && owner[r * cols + c] != 0;
        unsigned m = __ballot_sync(0xffffffffu, f);
        if (m == 0) continue;
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(counters + CN_LIST, (unsigned long long)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (f) list[base + __popc(m & ((1u << lane) - 1u))] = uint32_t(r * cols + c);
    }
}

// PixelStats.mean (Pixel.fs:103-108) and, optionally, PixelOutput.correct (ImageOutput.fs:11-18)
__global__ void finalize_kernel(const int32_t *stats, int n_pixels, int gamma, uint8_t *rgb) {
    __shared__ uint8_t lut[256];
    fill_gamma_lut(lut, gamma);
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pixels) return;
    pixel_rgb8(reinterpret_cast<const int4 *>(stats)[p], lut, rgb + 3 * size_t(p));
}

// ---------------------------------------------------------------------------------------------------
// frame driver
// ---------------------------------------------------------------------------------------------------
int check_frame_args(const RtScene *scene, const RtCamera *camera, int max_w, int max_h, const RtRenderOpts *opts) {
    if (!scene || !camera || !opts) return fail(RT_ERR_INVALID_ARGUMENT, "render: null argument");
    if (!scene->dev) return fail(RT_ERR_NO_DEVICE, "render: the scene was created without a device (device = -1); there is no CPU fallback");
    if (max_w <= 0 || max_h <= 0) return fail(RT_ERR_INVALID_ARGUMENT, "render: maxWidthCoord and maxHeightCoord must be positive");
    if (max_w > 32767 || max_h > 16383) return fail(RT_ERR_INVALID_ARGUMENT, "render: image too large (at most 65535 x 32767)");
    if (camera->samples_per_pixel < 1 || camera->samples_per_pixel > (1 << 22))
        return fail(RT_ERR_INVALID_ARGUMENT, "render: samples_per_pixel must be in [1, 2^22] (integer sums are 32-bit)");
    if (camera->bounce_depth < 0) return fail(RT_ERR_INVALID_ARGUMENT, "render: bounce_depth must be non-negative");
    return RT_OK;
}

struct LaunchPlan {
    bool smem;
    size_t smem_bytes;
    int blocks, threads;
};

// count and noise never come together (rt_frame_begin refuses RT_FLAG_NOISE with RT_FLAG_COUNTERS; plan_launch checks)
template <bool PROBE, int SMEM, bool SSTACK, bool WIDE>
static RenderKernelFn pick_count(bool count, bool noise) {
    if (noise) return render_kernel<PROBE, SMEM, false, SSTACK, WIDE, true>;
    return count ? render_kernel<PROBE, SMEM, true, SSTACK, WIDE> : render_kernel<PROBE, SMEM, false, SSTACK, WIDE>;
}
template <bool PROBE>
static RenderKernelFn pick_global(bool sstack, bool wide, bool count, bool noise) { // the scene is read from global memory
    if (wide) return sstack ? pick_count<PROBE, 0, true, true>(count, noise) : pick_count<PROBE, 0, false, true>(count, noise);
    return sstack ? pick_count<PROBE, 0, true, false>(count, noise) : pick_count<PROBE, 0, false, false>(count, noise);
}
template <bool PROBE>
static RenderKernelFn pick_flow(bool smem, bool count) {
    if (smem) return count ? render_flow_kernel<PROBE, true, true> : render_flow_kernel<PROBE, true, false>;
    return count ? render_flow_kernel<PROBE, false, true> : render_flow_kernel<PROBE, false, false>;
}
static RenderKernelFn pick_kernel(bool probe, bool smem, bool lean, bool count, bool sstack, bool wide, bool noise) {
    if (smem && lean) return probe ? pick_count<true, 2, false, false>(count, noise) : pick_count<false, 2, false, false>(count, noise);
    if (probe) return smem ? pick_count<true, 1, false, false>(count, noise) : pick_global<true>(sstack, wide, count, noise);
    return smem ? pick_count<false, 1, false, false>(count, noise) : pick_global<false>(sstack, wide, count, noise);
}

// does a block with `bytes` of dynamic shared memory leave room for `per_sm` of its kind on an SM (1 KB reserved per block)
static bool smem_fits(const DeviceScene *ds, size_t bytes, int per_sm) {
    return (bytes + 1024) * size_t(per_sm) <= ds->ws->smem_optin + (per_sm > 1 ? 1024 : 0);
}

// 16-byte quads of the scene a staged block holds: nodes | spheres | materials
static size_t staged_scene_quads(const DeviceScene *ds) {
    return size_t(ds->g.n_nodes) * kStagedNodeQuads + size_t(ds->g.n_bounded) + size_t(ds->g.n_bounded + ds->g.n_unbounded) * 2;
}

// the scene is staged in shared memory when it fits beside `warp_bytes` of scratch per warp (one block of kBlockThreads per SM)
static bool scene_staged(const DeviceScene *ds, size_t warp_bytes) {
    const size_t warp_q = (kBlockThreads / 32) * warp_bytes / 16;
    return smem_fits(ds, (staged_scene_quads(ds) + warp_q) * 16, kBlocksPerSm) && ds->g.n_bounded > 0;
}

// lays out shared memory and sizes the persistent grid
static int plan_launch(DeviceScene *ds, FrameParams &fp, bool probe, LaunchPlan &plan, RenderKernelFn &fn) {
    const bool count = (fp.opt_flags & RT_FLAG_COUNTERS) != 0, no_smem = (fp.opt_flags & RT_FLAG_NO_SMEM) != 0;
    const bool wide_asked = frame_walks_wide_tree(ds, fp.opt_flags, true);
    // the flow schedule (ring of rays per warp) on request only — measured slower than lockstep on B200 (DESIGN.md 5) —
    // and not with the wide tree (no flow variant) nor when the bounce budget does not fit the byte it shares with the colour
    const bool flow = (fp.opt_flags & RT_FLAG_FLOW) && !(fp.opt_flags & RT_FLAG_LOCKSTEP) && !wide_asked && fp.cam.depth <= kMaxFlowDepth;
    // the sum of squares of progressive frames opened with RT_FLAG_NOISE: lockstep kernels without counters only
    const bool noise = fp.sq != nullptr;
    if (noise && (flow || count)) return fail(RT_ERR_UNSUPPORTED, "render: the noise estimate has no flow-schedule or counting kernel");
    // a batch of views (rt_render_views, rt_frame_begin_views): lockstep kernels without counters, with or without the sum
    // of squares
    const bool views = fp.views != nullptr;
    if (views && (flow || count)) return fail(RT_ERR_UNSUPPORTED, "render: a batch of views has no flow-schedule or counting kernel");
    // a window of one frame (rt_render_window, rt_frame_begin_window): the same kernels as a batch, over the window's pixels
    const bool window = fp.window != 0;
    if (window && (flow || count)) return fail(RT_ERR_UNSUPPORTED, "render: a window has no flow-schedule or counting kernel");
    const size_t nodes_q = size_t(ds->g.n_nodes) * kStagedNodeQuads, sph_q = size_t(ds->g.n_bounded);
    const size_t scene_q = staged_scene_quads(ds);
    bool smem = scene_staged(ds, flow ? sizeof(FlowWarp) : warp_scratch_bytes(true, noise));
    const bool wide = frame_walks_wide_tree(ds, fp.opt_flags, smem);
    if (no_smem || wide) smem = false;
    // the launch shape follows from where the scene is read (rtfs_device.h); the flow kernels keep one block of 1024
    plan.threads = flow ? kBlockThreads : block_threads(smem);
    const int want_per_sm = flow ? 1 : blocks_per_sm(smem);
    const size_t warp_q = size_t(plan.threads / 32) * (flow ? sizeof(FlowWarp) : warp_scratch_bytes(smem, noise)) / 16;
    fp.s_nodes = 0;
    fp.s_spheres = uint32_t(nodes_q);
    fp.s_mats = uint32_t(nodes_q + sph_q);
    fp.s_warp = smem ? uint32_t(scene_q) : 0u;
    plan.smem = smem;
    // A scene read from L2 leaves shared memory free: the walk stacks go there when tree depth x block size words fit
    // (measured on the 100 k-sphere scene at 16 spp: 124.3 against 128.2 ms; with the scene itself in shared memory the
    // same change is within noise, 67.1 against 67.4 ms on C2, 137.7 against 136.7 on C4, so those kernels keep a local stack)
    const size_t used_q = (smem ? scene_q : 0) + warp_q;
    const size_t stack_q = size_t(wide ? 2 * (ds->wide_depth + 1) : ds->max_depth + 1) * size_t(plan.threads) * 4 / 16;
    // RTFS_LOCAL_STACK (A/B runs, tests): keep the walk stacks in local memory even where shared memory has room for them
    static const bool local_stack = std::getenv("RTFS_LOCAL_STACK") != nullptr;
    const bool sstack = !flow && !smem && !local_stack && ds->g.n_bounded > 0 && smem_fits(ds, (used_q + stack_q) * 16, want_per_sm);
    fp.s_stack = uint32_t(used_q);
    {
        static const int forced = [] {
            const char *e = std::getenv("RTFS_FLOW_QUANTUM");
            return e ? std::max(1, std::min(64, std::atoi(e))) : 0;
        }();
        fp.quantum = forced ? forced : (smem ? kFlowQuantumSmall : kFlowQuantumBig);
    }
    fp.stack_levels = int32_t(stack_q * 16 / (size_t(plan.threads) * 4));
    plan.smem_bytes = (used_q + (sstack ? stack_q : 0)) * 16;
    const bool lean = ds->lean && !(fp.opt_flags & RT_FLAG_NO_LEAN);
    if (views) fn = pick_views_kernel(probe, smem, lean, sstack, wide, noise);
    else if (window) fn = pick_window_kernel(probe, smem, lean, sstack, wide, noise);
    else fn = flow ? (probe ? pick_flow<true>(smem, count) : pick_flow<false>(smem, count)) : pick_kernel(probe, smem, lean, count, sstack, wide, noise);
    {
        static const bool show = std::getenv("RTFS_DEBUG_PLAN") != nullptr;
        if (show) {
            char views_field[24] = ""; // a batch of views adds its size to the line
            if (views) std::snprintf(views_field, sizeof views_field, " views=%d", fp.n_views);
            char window_field[64] = ""; // a window adds its size and offset
            if (window) std::snprintf(window_field, sizeof window_field, " window=%dx%d@%d,%d", fp.cam.rows, fp.cam.cols, fp.win_row0, fp.win_col0);
            std::fprintf(stderr, "rtfs: plan probe=%d staged=%d lean=%d count=%d sstack=%d wide=%d flow=%d noise=%d smem_bytes=%zu threads=%d%s%s\n",
                         int(probe), int(smem), int(smem && lean), int(count), int(sstack), int(wide), int(flow), int(noise), plan.smem_bytes,
                         plan.threads, views_field, window_field);
        }
    }
    { // The dynamic shared-memory limit of a kernel is a per-function, per-device setting: it is only ever RAISED here
      // (to the largest size any scene has asked for), and the occupancy of a (kernel, size, device) triple is asked once.
        struct Known {
            const void *fn;
            size_t smem;
            int device, per_sm;
        };
        static std::mutex mutex;
        static std::vector<Known> known; // smem = the size the entry's occupancy was computed for
        static std::vector<Known> limits; // smem = the limit currently set for (fn, device)
        std::lock_guard<std::mutex> lock(mutex);
        Known *limit = nullptr;
        for (Known &k : limits)
            if (k.fn == (const void *)fn && k.device == ds->device) limit = &k;
        if (!limit || limit->smem < plan.smem_bytes) {
            RT_CUDA(cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, int(plan.smem_bytes)));
            // Two blocks per SM must both be resident (a persistent kernel's second wave finds no work left).  The occupancy
            // query below answers 2 whenever the SM COULD hold them, but the carve-out the driver picks by default at launch
            // is not always large enough for both (measured: with 61 KB of dynamic shared memory per block only 148 of the 296
            // blocks ever ran, 100 k spheres 279 ms instead of 202), so the largest carve-out is asked for explicitly.
            if (!smem && !flow) RT_CUDA(cudaFuncSetAttribute((const void *)fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
            if (limit) limit->smem = plan.smem_bytes;
            else limits.push_back(Known{(const void *)fn, plan.smem_bytes, ds->device, 0});
        }
        int per_sm = -1;
        for (const Known &k : known)
            if (k.fn == (const void *)fn && k.smem == plan.smem_bytes && k.device == ds->device) per_sm = k.per_sm;
        if (per_sm < 0) {
            RT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void *)fn, plan.threads, plan.smem_bytes));
            known.push_back(Known{(const void *)fn, plan.smem_bytes, ds->device, per_sm});
        }
        if (per_sm < 1) return fail(RT_ERR_CUDA, "render kernel does not fit on an SM");
        plan.blocks = per_sm * ds->ws->sm_count;
    }
    return RT_OK;
}

int ensure_frame_buffers(DeviceWorkspace *ws, size_t n_pixels) {
    if (ws->ws_pixels >= n_pixels) return RT_OK;
    cudaFree(ws->d_stats);
    cudaFree(ws->d_flags);
    cudaFree(ws->d_rgb);
    ws->d_stats = nullptr;
    ws->d_flags = nullptr;
    ws->d_rgb = nullptr;
    ws->ws_pixels = 0;
    RT_CUDA(cudaMalloc((void **)&ws->d_stats, n_pixels * 4 * sizeof(int32_t)));
    RT_CUDA(cudaMalloc((void **)&ws->d_flags, n_pixels));
    RT_CUDA(cudaMalloc((void **)&ws->d_rgb, n_pixels * 3));
    ws->ws_pixels = n_pixels;
    return RT_OK;
}

int ensure_list(DeviceWorkspace *ws, size_t n_pixels) {
    if (ws->list_pixels >= n_pixels) return RT_OK;
    cudaFree(ws->d_list);
    ws->d_list = nullptr;
    ws->list_pixels = 0;
    RT_CUDA(cudaMalloc((void **)&ws->d_list, n_pixels * sizeof(uint32_t)));
    ws->list_pixels = n_pixels;
    return RT_OK;
}

int ensure_probe_sums(DeviceWorkspace *ws, size_t n_pixels) {
    if (ws->probe_pixels >= n_pixels) return RT_OK;
    cudaFree(ws->d_stats_b);
    ws->d_stats_b = nullptr;
    ws->probe_pixels = 0;
    RT_CUDA(cudaMalloc((void **)&ws->d_stats_b, n_pixels * 4 * sizeof(int32_t)));
    ws->probe_pixels = n_pixels;
    return RT_OK;
}

void fill_frame(FrameParams &fp, DeviceScene *ds, const RtCamera &cam, int max_w, int max_h, const RtRenderOpts &opts, int rank, int world) {
    std::memset(&fp, 0, sizeof fp);
    fp.g = ds->g;
    fp.cam = make_dev_camera(cam, max_w, max_h);
    fp.k0 = uint32_t(opts.seed);
    fp.k1 = uint32_t(opts.seed >> 32);
    fp.rank = rank;
    fp.world = world;
    fp.tiles_x = (fp.cam.cols + kTileW - 1) / kTileW;
    fp.tiles_y = (fp.cam.rows + kTileH - 1) / kTileH;
    fp.adaptive = opts.adaptive ? 1 : 0;
    if (fp.adaptive) {
        fp.first_trial = std::min(5, cam.samples_per_pixel / 2); // Scene.fs:172
        fp.n_probe = 2 * fp.first_trial + 1;
        fp.sample_begin = fp.n_probe;
        fp.sample_end = std::max(fp.n_probe, cam.samples_per_pixel); // the third loop runs spp - 2 firstTrial - 1 times, Scene.fs:191
    } else {
        fp.first_trial = 0;
        fp.n_probe = 0;
        fp.sample_begin = 0;
        fp.sample_end = cam.samples_per_pixel;
    }
    fp.counters = ds->ws->d_counters;
    fp.opt_flags = opts.flags;
}

// Cuts this rank's local sample range [0, n_local) into chunks: `bulk` samples per chunk, then a taper
// bulk/2, bulk/4, ..., 2, 1, 1 so that the last layers of items are short (a warp cannot be sped up, so the
// kernel ends one item after the work runs out).  No chunk straddles `boundary` (probe: firstTrial + 1, the first
// sample of the second accumulator set).  Chunks are stored by decreasing length: items are numbered chunk-major.
static int build_chunks(FrameParams &fp, int n_local, int boundary, size_t n_units, int resident_warps) {
    fp.n_chunks = 0;
    if (n_local <= 0) return RT_OK;
    // bulk chunk: every warp should see ~16 bulk items; at most 32 samples (1024 paths) per item
    long long bulk = (long long)(n_units * size_t(n_local)) / (16LL * std::max(1, resident_warps));
    bulk = std::max(1LL, std::min(32LL, bulk));
    bulk = std::max(bulk, (long long)((n_local + 159) / 160)); // the table has kMaxChunks entries; n_local <= kMaxLaunchSamples keeps bulk <= kMaxChunkSamples
    std::vector<int> sizes;
    for (int t = int(bulk) / 2; t >= 1; t /= 2) sizes.push_back(t);
    if (bulk > 1) sizes.push_back(1);
    int taper = 0;
    for (int t : sizes) taper += t;
    while (!sizes.empty() && taper > n_local) { // short range: drop the longest taper chunks
        taper -= sizes.front();
        sizes.erase(sizes.begin());
    }
    int rest = n_local - taper;
    std::vector<int> all;
    while (rest > 0) {
        int c = int(std::min<long long>(bulk, rest));
        all.push_back(c);
        rest -= c;
    }
    all.insert(all.end(), sizes.begin(), sizes.end());
    std::vector<std::pair<int, int>> chunks;
    int at = 0;
    for (int c : all) {
        if (boundary > at && boundary < at + c) { // split at the boundary
            chunks.push_back({at, boundary - at});
            chunks.push_back({boundary, at + c - boundary});
        } else {
            chunks.push_back({at, c});
        }
        at += c;
    }
    std::stable_sort(chunks.begin(), chunks.end(), [](const std::pair<int, int> &a, const std::pair<int, int> &b) { return a.second > b.second; });
    if (chunks.size() > size_t(kMaxChunks)) return fail(RT_ERR_UNSUPPORTED, "render: the sample range needs more chunks than the work table holds");
    fp.n_chunks = int(chunks.size());
    for (int k = 0; k < fp.n_chunks; ++k) {
        fp.chunk_begin[k] = uint32_t(chunks[k].first);
        fp.chunk_len[k] = uint32_t(chunks[k].second);
    }
    return RT_OK;
}

int launch_probe(DeviceScene *ds, FrameParams fp, cudaStream_t st, int *launches, bool raw_flags) {
    DeviceWorkspace *ws = ds->ws;
    const size_t n_pixels = size_t(fp.cam.rows) * fp.cam.cols;
    int rc = ensure_probe_sums(ws, n_pixels);
    if (rc != RT_OK) return rc;
    RT_CUDA(cudaMemsetAsync(ws->d_stats_b, 0, n_pixels * 4 * sizeof(int32_t), st));
    RT_CUDA(cudaMemsetAsync(fp.counters + CN_WORK_PROBE, 0, sizeof(unsigned long long), st));
    fp.stats_b = ws->d_stats_b;
    LaunchPlan plan;
    RenderKernelFn fn;
    if ((rc = plan_launch(ds, fp, true, plan, fn)) != RT_OK) return rc;
    const size_t n_units = size_t((fp.tiles_x * fp.tiles_y - fp.rank + fp.world - 1) / fp.world);
    rc = build_chunks(fp, fp.n_probe, fp.first_trial + 1, n_units, plan.blocks * (plan.threads / 32));
    if (rc != RT_OK) return rc;
    fn<<<plan.blocks, plan.threads, plan.smem_bytes, st>>>(fp);
    RT_CUDA(cudaGetLastError());
    ++*launches;
    return launch_probe_flags(fp, ws->d_stats_b, raw_flags || fp.sample_end > fp.sample_begin, st, launches);
}

int launch_probe_flags(const FrameParams &fp, const int32_t *stats_b, bool more, cudaStream_t st, int *launches) {
    const size_t n_pixels = size_t(fp.cam.rows) * fp.cam.cols;
    probe_flags_kernel<<<unsigned((n_pixels + 255) / 256), 256, 0, st>>>(fp.stats, stats_b, fp.flags, fp.cam.rows, fp.cam.cols, fp.tiles_x,
                                                                          fp.rank, fp.world, fp.first_trial, fp.n_probe, more ? 1 : 0);
    RT_CUDA(cudaGetLastError());
    ++*launches;
    return RT_OK;
}

// flags -> the flagged-pixel list `list`, its length in fp.counters[CN_LIST]; zeroes the main phase's work cursor
int launch_compact(DeviceScene *ds, const FrameParams &fp, const FlagsView &flags, uint32_t *list, cudaStream_t st, int *launches) {
    RT_CUDA(cudaMemsetAsync(fp.counters + CN_LIST, 0, sizeof(unsigned long long), st));
    RT_CUDA(cudaMemsetAsync(fp.counters + CN_WORK_MAIN, 0, sizeof(unsigned long long), st));
    compact_kernel<<<ds->ws->sm_count * 4, 256, 0, st>>>(flags, list, fp.counters, fp.cam.rows, fp.cam.cols, fp.tiles_x, fp.tiles_y);
    RT_CUDA(cudaGetLastError());
    ++*launches;
    return RT_OK;
}

// The main phase over the sample window [fp.sample_begin, fp.sample_end) (this rank's share of it) for the pixels of
// fp.list; the work cursor fp.counters[CN_WORK_MAIN] must be zero on entry
int launch_samples(DeviceScene *ds, FrameParams fp, cudaStream_t st, int *launches) {
    const size_t n_pixels = size_t(fp.cam.rows) * fp.cam.cols;
    LaunchPlan plan;
    RenderKernelFn fn;
    int rc = plan_launch(ds, fp, false, plan, fn);
    if (rc != RT_OK) return rc;
    int n_span = fp.sample_end - fp.sample_begin - fp.rank;
    int n_local = n_span > 0 ? (n_span + fp.world - 1) / fp.world : 0;
    // the list length is only known on the device; size the chunks for the whole frame (an upper bound on the units)
    // one launch covers at most kMaxLaunchSamples of this rank's sample indices (a chunk stays within kMaxChunkSamples: the
    // 16-bit halves of an item's red | green word); a frame with more is several launches
    for (int base = 0; base < n_local; base += kMaxLaunchSamples) {
        rc = build_chunks(fp, std::min(kMaxLaunchSamples, n_local - base), -1, (n_pixels + 31) / 32, plan.blocks * (plan.threads / 32));
        if (rc != RT_OK) return rc;
        for (int k = 0; k < fp.n_chunks; ++k) fp.chunk_begin[k] += uint32_t(base);
        if (base > 0) RT_CUDA(cudaMemsetAsync(fp.counters + CN_WORK_MAIN, 0, sizeof(unsigned long long), st));
        fn<<<plan.blocks, plan.threads, plan.smem_bytes, st>>>(fp);
        RT_CUDA(cudaGetLastError());
        ++*launches;
    }
    return RT_OK;
}

int launch_main(DeviceScene *ds, FrameParams fp, const FlagsView &flags, cudaStream_t st, int *launches) {
    int rc = ensure_list(ds->ws, size_t(fp.cam.rows) * fp.cam.cols);
    if (rc != RT_OK) return rc;
    if ((rc = launch_compact(ds, fp, flags, ds->ws->d_list, st, launches)) != RT_OK) return rc;
    fp.list = ds->ws->d_list;
    return launch_samples(ds, fp, st, launches);
}

int launch_finalize(const int32_t *stats, size_t n_pixels, int gamma, uint8_t *rgb, cudaStream_t st, int *launches) {
    finalize_kernel<<<unsigned((n_pixels + 255) / 256), 256, 0, st>>>(stats, int(n_pixels), gamma, rgb);
    RT_CUDA(cudaGetLastError());
    ++*launches;
    return RT_OK;
}

int frame_probe(DeviceScene *ds, const FrameParams &fp, cudaStream_t st, FrameEvents *ev, int *launches) {
    const size_t n_pixels = size_t(fp.cam.rows) * fp.cam.cols;
    if (ev) RT_CUDA(ev->record(FrameEvents::BEGIN, st));
    RT_CUDA(cudaMemsetAsync(fp.counters, 0, CN_SLOTS * sizeof(unsigned long long), st));
    RT_CUDA(cudaMemsetAsync(fp.stats, 0, n_pixels * 4 * sizeof(int32_t), st));
    if (fp.sq) RT_CUDA(cudaMemsetAsync(fp.sq, 0, n_pixels * sizeof(unsigned long long), st));
    if (ev) RT_CUDA(ev->record(FrameEvents::ZEROED, st));
    if (!fp.adaptive) {
        RT_CUDA(cudaMemsetAsync(fp.flags, 1, n_pixels, st));
        return RT_OK;
    }
    if (fp.world > 1) RT_CUDA(cudaMemsetAsync(fp.flags, 0, n_pixels, st));
    return launch_probe(ds, fp, st, launches, fp.counters != ds->ws->d_counters);
}

int frame_main(DeviceScene *ds, const FrameParams &fp, cudaStream_t st, FrameEvents &ev, int *launches) {
    RT_CUDA(cudaMemcpyAsync(ds->ws->h_counters + CN_SLOTS, fp.counters, CN_SLOTS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    RT_CUDA(ev.record(FrameEvents::MAIN_BEGIN, st));
    int rc = launch_main(ds, fp, single_flags(fp.flags), st, launches);
    if (rc != RT_OK) return rc;
    RT_CUDA(ev.record(FrameEvents::MAIN_END, st));
    RT_CUDA(ev.record(FrameEvents::TRACED, st));
    return RT_OK;
}

int frame_finish(DeviceScene *ds, const FrameParams &fp, const uint8_t *d_rgb, uint8_t *rgb_out, int32_t *sums_out, cudaStream_t st,
                 FrameEvents &ev) {
    const size_t n_pixels = size_t(fp.cam.rows) * fp.cam.cols;
    if (rgb_out) RT_CUDA(cudaMemcpyAsync(rgb_out, d_rgb, n_pixels * 3, cudaMemcpyDeviceToHost, st));
    if (sums_out) RT_CUDA(cudaMemcpyAsync(sums_out, fp.stats, n_pixels * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    RT_CUDA(cudaMemcpyAsync(ds->ws->h_counters, fp.counters, CN_SLOTS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    RT_CUDA(ev.record(FrameEvents::END, st));
    return RT_OK;
}

void read_stats(const DeviceScene *ds, size_t n_pixels, bool adaptive, int launches, const FrameEvents *ev, RtStats *stats) {
    const unsigned long long *h = ds->ws->h_counters;
    std::memset(stats, 0, sizeof *stats);
    stats->paths = h[CN_PATHS];
    stats->rays = h[CN_RAYS];
    stats->box_tests = h[CN_BOX];
    stats->prim_tests = h[CN_PRIM];
    stats->pixels_early_out = adaptive ? (unsigned long long)n_pixels - h[CN_LIST] : 0;
    stats->degenerate_paths = h[CN_DEGENERATE];
    stats->launches = launches;
    if (ev) {
        stats->kernel_ms = ev->ms(FrameEvents::ZEROED, FrameEvents::TRACED);
        stats->total_ms = ev->ms(FrameEvents::BEGIN, FrameEvents::END);
        stats->main_ms = ev->ms(FrameEvents::MAIN_BEGIN, FrameEvents::MAIN_END);
        stats->main_rays = h[CN_RAYS] - h[CN_SLOTS + CN_RAYS];
    }
    if (std::getenv("RTFS_DEBUG_BLOCKS")) std::fprintf(stderr, "rtfs: blocks that found work (probe + main): %llu\n", h[CN_BUSY_BLOCKS]);
}

// one device->host copy of the counters into ds->ws->h_counters and a synchronisation of the stream
static int sync_counters(DeviceScene *ds, cudaStream_t st) {
    RT_CUDA(cudaMemcpyAsync(ds->ws->h_counters, ds->ws->d_counters, CN_SLOTS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    RT_CUDA(cudaStreamSynchronize(st));
    return RT_OK;
}

// implemented in rtfs_wavefront.cu
int render_wavefront(RtScene *scene, const RtCamera *camera, int32_t max_w, int32_t max_h, const RtRenderOpts *opts, uint8_t *rgb_out,
                     int32_t *sums_out, RtStats *stats);

} // namespace rtfs

using namespace rtfs;

// =================================================================================================
// C ABI — device entry points
// =================================================================================================
extern "C" {

int rt_host_pin(void *ptr, size_t bytes) {
    if (!ptr || !bytes) return fail(RT_ERR_INVALID_ARGUMENT, "rt_host_pin: null or empty buffer");
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        return fail(RT_ERR_NO_DEVICE, "rt_host_pin: no CUDA device is visible");
    }
    RT_CUDA(cudaHostRegister(ptr, bytes, cudaHostRegisterPortable));
    return RT_OK;
}
int rt_host_unpin(void *ptr) {
    if (!ptr) return fail(RT_ERR_INVALID_ARGUMENT, "rt_host_unpin: null buffer");
    RT_CUDA(cudaHostUnregister(ptr));
    return RT_OK;
}

int rt_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// bytes of the scene each persistent block stages in shared memory (0: the BVH is read from global memory / L2)
size_t rt_scene_shared_memory_bytes(const RtScene *scene) {
    if (!scene || !scene->dev) return 0;
    auto *ds = static_cast<const DeviceScene *>(scene->dev);
    // with the default (lockstep) schedule's per-warp scratch
    return scene_staged(ds, warp_scratch_bytes(true)) ? staged_scene_quads(ds) * 16 : 0;
}

int rt_device_probe(RtScene *scene, const RtCamera *camera, int32_t max_w, int32_t max_h, const RtRenderOpts *opts, int32_t rank,
                    int32_t world, int32_t *d_stats, uint8_t *d_flags, void *stream, RtStats *stats) {
    int rc = check_frame_args(scene, camera, max_w, max_h, opts);
    if (rc != RT_OK) return rc;
    if (world < 1 || rank < 0 || rank >= world || !d_stats || !d_flags) return fail(RT_ERR_INVALID_ARGUMENT, "rt_device_probe: bad rank/world/buffers");
    if ((rc = prepare_frame(scene, opts)) != RT_OK) return rc;
    auto *ds = static_cast<DeviceScene *>(scene->dev);
    RT_CUDA(cudaSetDevice(ds->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    FrameParams fp;
    fill_frame(fp, ds, *camera, max_w, max_h, *opts, rank, world);
    fp.stats = d_stats;
    fp.flags = d_flags;
    const size_t n_pixels = size_t(fp.cam.rows) * fp.cam.cols;
    int launches = 0;
    RT_CUDA(cudaMemsetAsync(ds->ws->d_counters, 0, CN_SLOTS * sizeof(unsigned long long), st));
    if (!fp.adaptive) {
        // no probe phase: every pixel takes all its samples in the main phase (rank 0 raises the flags once)
        if (rank == 0) RT_CUDA(cudaMemsetAsync(d_flags, 1, n_pixels, st));
    } else if ((rc = launch_probe(ds, fp, st, &launches, false)) != RT_OK) {
        return rc;
    }
    if (stats) {
        if ((rc = sync_counters(ds, st)) != RT_OK) return rc;
        read_stats(ds, n_pixels, false, launches, nullptr, stats);
    }
    return RT_OK;
}

int rt_device_main(RtScene *scene, const RtCamera *camera, int32_t max_w, int32_t max_h, const RtRenderOpts *opts, int32_t rank,
                   int32_t world, int32_t *d_stats, const uint8_t *d_flags, void *stream, RtStats *stats) {
    int rc = check_frame_args(scene, camera, max_w, max_h, opts);
    if (rc != RT_OK) return rc;
    if (world < 1 || rank < 0 || rank >= world || !d_stats || !d_flags) return fail(RT_ERR_INVALID_ARGUMENT, "rt_device_main: bad rank/world/buffers");
    if ((rc = prepare_frame(scene, opts)) != RT_OK) return rc;
    auto *ds = static_cast<DeviceScene *>(scene->dev);
    RT_CUDA(cudaSetDevice(ds->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    FrameParams fp;
    fill_frame(fp, ds, *camera, max_w, max_h, *opts, rank, world);
    fp.stats = d_stats;
    fp.flags = const_cast<uint8_t *>(d_flags);
    int launches = 0;
    if ((rc = launch_main(ds, fp, single_flags(d_flags), st, &launches)) != RT_OK) return rc;
    if (stats) {
        if ((rc = sync_counters(ds, st)) != RT_OK) return rc;
        read_stats(ds, size_t(fp.cam.rows) * fp.cam.cols, fp.adaptive != 0, launches, nullptr, stats);
    }
    return RT_OK;
}

// paths / rays / tests accumulated on this scene since the last rt_device_probe (one D2H copy + a stream sync)
int rt_device_counters(RtScene *scene, void *stream, RtStats *stats) {
    if (!scene || !stats) return fail(RT_ERR_INVALID_ARGUMENT, "rt_device_counters: null argument");
    if (!scene->dev) return fail(RT_ERR_NO_DEVICE, "rt_device_counters: the scene has no device");
    auto *ds = static_cast<DeviceScene *>(scene->dev);
    RT_CUDA(cudaSetDevice(ds->device));
    int rc = sync_counters(ds, static_cast<cudaStream_t>(stream));
    if (rc != RT_OK) return rc;
    std::memset(stats, 0, sizeof *stats);
    stats->paths = ds->ws->h_counters[CN_PATHS];
    stats->rays = ds->ws->h_counters[CN_RAYS];
    stats->box_tests = ds->ws->h_counters[CN_BOX];
    stats->prim_tests = ds->ws->h_counters[CN_PRIM];
    stats->pixels_early_out = ds->ws->h_counters[CN_LIST]; // NOTE: here the number of pixels that went on to phase 2
    return RT_OK;
}

int rt_device_finalize(int32_t device, const int32_t *d_stats, int32_t n_pixels, int32_t gamma, uint8_t *d_rgb, void *stream) {
    int rc = require_device(device);
    if (rc != RT_OK) return rc;
    if (!d_stats || !d_rgb || n_pixels <= 0) return fail(RT_ERR_INVALID_ARGUMENT, "rt_device_finalize: bad argument");
    int launches = 0;
    return launch_finalize(d_stats, size_t(n_pixels), gamma, d_rgb, static_cast<cudaStream_t>(stream), &launches);
}

int rt_render(RtScene *scene, const RtCamera *camera, int32_t max_w, int32_t max_h, const RtRenderOpts *opts, uint8_t *rgb_out,
              int32_t *sums_out, RtStats *stats) {
    int rc = check_frame_args(scene, camera, max_w, max_h, opts);
    if (rc != RT_OK) return rc;
    if (!rgb_out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_render: rgb_out is null");
    if (opts->mode == RT_MODE_WAVEFRONT) return render_wavefront(scene, camera, max_w, max_h, opts, rgb_out, sums_out, stats);
    if (opts->mode != RT_MODE_MEGAKERNEL) return fail(RT_ERR_INVALID_ARGUMENT, "rt_render: unknown mode");
    if ((rc = prepare_frame(scene, opts)) != RT_OK) return rc;
    auto *ds = static_cast<DeviceScene *>(scene->dev);
    RT_CUDA(cudaSetDevice(ds->device));
    DeviceWorkspace *ws = ds->ws;
    const size_t n_pixels = size_t(2 * max_w + 1) * size_t(2 * max_h + 1);
    if ((rc = ensure_frame_buffers(ws, n_pixels)) != RT_OK) return rc;
    cudaStream_t st = ws->stream;
    FrameParams fp;
    fill_frame(fp, ds, *camera, max_w, max_h, *opts, 0, 1);
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
