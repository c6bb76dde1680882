// rtfs_comm.cu — one rank of a multi-process job (one process per GPU), with the collectives INSIDE the library
// (rt_comm_*).  Replicated scene, sample-index split (SURVEY.md §8e); the exchange steps are NCCL calls issued by
// this file on the same stream as the kernels, so a caller (bench.py under torchrun, or one F# process per GPU) makes
// one call per frame:
//
//   probe          rank r probes the tiles t with t mod world == r                      (Scene.fs:172-188)
//   ncclAllReduce  flags, uint8 MAX                                   n_pixels bytes   [adaptive only]
//   compact + main rank r adds samples n_probe + r + j*world of every flagged pixel    (Scene.fs:191-192)
//   reduce + finalize + gather, ONE kernel over NVLink peer memory (the ranks' buffers mapped into one another with CUDA
//                  IPC when the communicator's buffers are allocated): rank r sums every rank's {sumR, sumG, sumB, count}
//                  for ITS slice of the pixels with 128-bit peer loads, divides (PixelStats.mean, Pixel.fs:103-108),
//                  applies the optional gamma (ImageOutput.fs:11-18) and stores the RGB8 of the slice into EVERY rank's
//                  frame with peer stores; a 4-byte ncclAllReduce before and after it are the stream-ordered barriers
//                  ("all sums are final", "all slices have landed and nobody reads my sums any more")
//     — or, where the buffers cannot be mapped (no peer access, IPC refused; RTFS_COMM_NO_PEER=1 forces it):
//   ncclReduceScatter (int32 SUM: rank r receives the totals of its slice) -> finalize_kernel on the slice ->
//   ncclAllGather of the RGB8 slices (3 n_pixels bytes instead of another 16 n_pixels)
//   copy           device -> host on the ranks that asked for the image
//
// (With sums_out the sums are all-reduced instead, so that every rank can return them.)  Integer sums keyed by sample
// index make the image bit-identical for every world size and identical to rt_render's.
//
// NCCL is bound at run time (dlopen of libnccl.so.2, preferring a copy the process has already mapped): the library
// must keep loading on a single-GPU host without NCCL, and a process that also holds PyTorch must not end up with two
// different NCCL builds behind one soname.  Only the symbols below are used; nccl.h supplies the types.
#include "rtfs_device.h"

#include <dlfcn.h>
#include <nccl.h>

#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

namespace rtfs {
namespace {

struct NcclApi {
    void *handle = nullptr;
    ncclResult_t (*GetVersion)(int *) = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*ReduceScatter)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    std::string path;
};
std::mutex g_nccl_mutex;
NcclApi g_nccl;

int nccl_api(NcclApi **out) {
    std::lock_guard<std::mutex> lock(g_nccl_mutex);
    if (!g_nccl.handle) {
        void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD); // a copy the process already holds (PyTorch's), if any
        if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
        if (!h) return fail(RT_ERR_UNSUPPORTED, std::string("rt_comm: libnccl.so.2 cannot be loaded: ") + dlerror());
        NcclApi a;
        a.handle = h;
        bool ok = true;
        auto sym = [&](const char *name) {
            void *p = dlsym(h, name);
            ok = ok && p != nullptr;
            return p;
        };
        a.GetVersion = reinterpret_cast<decltype(a.GetVersion)>(sym("ncclGetVersion"));
        a.GetUniqueId = reinterpret_cast<decltype(a.GetUniqueId)>(sym("ncclGetUniqueId"));
        a.CommInitRank = reinterpret_cast<decltype(a.CommInitRank)>(sym("ncclCommInitRank"));
        a.CommDestroy = reinterpret_cast<decltype(a.CommDestroy)>(sym("ncclCommDestroy"));
        a.GetErrorString = reinterpret_cast<decltype(a.GetErrorString)>(sym("ncclGetErrorString"));
        a.AllReduce = reinterpret_cast<decltype(a.AllReduce)>(sym("ncclAllReduce"));
        a.ReduceScatter = reinterpret_cast<decltype(a.ReduceScatter)>(sym("ncclReduceScatter"));
        a.AllGather = reinterpret_cast<decltype(a.AllGather)>(sym("ncclAllGather"));
        if (!ok) {
            dlclose(h);
            return fail(RT_ERR_UNSUPPORTED, "rt_comm: libnccl.so.2 lacks a symbol this library needs");
        }
        Dl_info info;
        if (dladdr(reinterpret_cast<void *>(a.AllReduce), &info) && info.dli_fname) a.path = info.dli_fname;
        g_nccl = a;
    }
    *out = &g_nccl;
    return RT_OK;
}

#define RT_NCCL(api, expr)                                                                                    \
    do {                                                                                                      \
        ncclResult_t r__ = (expr);                                                                            \
        if (r__ != ncclSuccess) return fail(RT_ERR_CUDA, std::string(#expr) + ": " + (api)->GetErrorString(r__)); \
    } while (0)

} // namespace
} // namespace rtfs

struct RtComm {
    rtfs::NcclApi *api = nullptr;
    ncclComm_t comm = nullptr;
    int rank = 0, world = 1, device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    rtfs::FrameEvents ev;
    size_t last_pixels = 0;
    bool last_adaptive = false;
    int last_launches = 0;
    // frame buffers, padded so that the pixels split into `world` equal slices
    size_t slice_px = 0;      // pixels per slice
    int32_t *d_stats = nullptr; // world * slice_px * 4
    uint8_t *d_flags = nullptr; // world * slice_px
    uint8_t *d_rgb = nullptr;   // world * slice_px * 3
    // peer memory: every rank's d_stats and d_rgb as this process sees them (own pointers at [rank]); empty: NCCL path
    bool peer = false;
    int32_t *peer_stats[rtfs::kMaxDevices] = {};
    uint8_t *peer_rgb[rtfs::kMaxDevices] = {};
    int32_t *d_sync = nullptr;  // the word the barrier all-reduces sum
    uint8_t *d_handles = nullptr; // staging for the exchange of the IPC handles
};

using namespace rtfs;

namespace {
void peer_close(RtComm *c) {
    for (int r = 0; r < c->world; ++r) {
        if (r != c->rank) {
            if (c->peer_stats[r]) cudaIpcCloseMemHandle(c->peer_stats[r]);
            if (c->peer_rgb[r]) cudaIpcCloseMemHandle(c->peer_rgb[r]);
        }
        c->peer_stats[r] = nullptr;
        c->peer_rgb[r] = nullptr;
    }
    c->peer = false;
}

// Maps every rank's sum and frame buffers into this process (collective: called by all ranks when their buffers have
// just been allocated).  Any failure on any rank leaves every rank on the NCCL path.
int peer_open(RtComm *c) {
    peer_close(c);
    if (c->world < 2) return RT_OK;
    if (const char *e = std::getenv("RTFS_COMM_NO_PEER"))
        if (e[0] == '1') return RT_OK; // every rank reads the same environment under torchrun / mpirun
    NcclApi *api = c->api;
    cudaStream_t st = c->stream;
    constexpr size_t kPer = 2 * sizeof(cudaIpcMemHandle_t);
    if (!c->d_handles) RT_CUDA(cudaMalloc((void **)&c->d_handles, kPer * kMaxDevices));
    if (!c->d_sync) {
        RT_CUDA(cudaMalloc((void **)&c->d_sync, sizeof(int32_t)));
        RT_CUDA(cudaMemset(c->d_sync, 0, sizeof(int32_t)));
    }
    cudaIpcMemHandle_t mine[2];
    int ok = cudaIpcGetMemHandle(&mine[0], c->d_stats) == cudaSuccess && cudaIpcGetMemHandle(&mine[1], c->d_rgb) == cudaSuccess ? 1 : 0;
    if (!ok) {
        cudaGetLastError();
        std::memset(mine, 0, sizeof mine);
    }
    std::vector<cudaIpcMemHandle_t> all(2 * size_t(c->world));
    RT_CUDA(cudaMemcpyAsync(c->d_handles + kPer * c->rank, mine, kPer, cudaMemcpyHostToDevice, st));
    RT_NCCL(api, api->AllGather(c->d_handles + kPer * c->rank, c->d_handles, kPer, ncclUint8, c->comm, st));
    RT_CUDA(cudaMemcpyAsync(all.data(), c->d_handles, kPer * c->world, cudaMemcpyDeviceToHost, st));
    RT_CUDA(cudaStreamSynchronize(st));
    for (int r = 0; r < c->world && ok; ++r) {
        if (r == c->rank) {
            c->peer_stats[r] = c->d_stats;
            c->peer_rgb[r] = c->d_rgb;
            continue;
        }
        void *ps = nullptr, *pr = nullptr;
        if (cudaIpcOpenMemHandle(&ps, all[2 * r], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess ||
            cudaIpcOpenMemHandle(&pr, all[2 * r + 1], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
            cudaGetLastError();
            if (ps) cudaIpcCloseMemHandle(ps);
            ok = 0;
            break;
        }
        c->peer_stats[r] = static_cast<int32_t *>(ps);
        c->peer_rgb[r] = static_cast<uint8_t *>(pr);
    }
    // all or nothing, agreed by everybody: MIN over the ranks' flags
    int32_t flag = ok, agreed = 0;
    RT_CUDA(cudaMemcpyAsync(c->d_sync, &flag, sizeof flag, cudaMemcpyHostToDevice, st));
    RT_NCCL(api, api->AllReduce(c->d_sync, c->d_sync, 1, ncclInt32, ncclMin, c->comm, st));
    RT_CUDA(cudaMemcpyAsync(&agreed, c->d_sync, sizeof agreed, cudaMemcpyDeviceToHost, st));
    RT_CUDA(cudaMemsetAsync(c->d_sync, 0, sizeof(int32_t), st));
    RT_CUDA(cudaStreamSynchronize(st));
    if (agreed == 1) c->peer = true;
    else peer_close(c);
    return RT_OK;
}

void comm_free(RtComm *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    const bool had_peers = c->peer;
    peer_close(c);
    if (had_peers && c->comm && c->api && c->d_sync) {
        // rt_comm_destroy is collective when buffers are shared: nobody frees a buffer a peer still has mapped
        if (c->api->AllReduce(c->d_sync, c->d_sync, 1, ncclInt32, ncclSum, c->comm, c->stream) == ncclSuccess) cudaStreamSynchronize(c->stream);
    }
    if (c->comm && c->api) c->api->CommDestroy(c->comm);
    cudaFree(c->d_sync);
    cudaFree(c->d_handles);
    cudaFree(c->d_stats);
    cudaFree(c->d_flags);
    cudaFree(c->d_rgb);
    c->ev.destroy();
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

int comm_workspace(RtComm *c, size_t n_pixels) {
    size_t slice = (n_pixels + size_t(c->world) - 1) / size_t(c->world);
    slice = (slice + 3) & ~size_t(3); // whole 16-byte groups of RGB8 per slice
    if (c->slice_px >= slice) return RT_OK;
    if (c->stream) RT_CUDA(cudaStreamSynchronize(c->stream));
    peer_close(c); // the peers close their mappings of these buffers in the same call (frames are collective)
    if (c->world > 1) { // nobody frees a buffer a peer may still have mapped: a host-side rendezvous through NCCL
        if (!c->d_sync) {
            RT_CUDA(cudaMalloc((void **)&c->d_sync, sizeof(int32_t)));
            RT_CUDA(cudaMemset(c->d_sync, 0, sizeof(int32_t)));
        }
        RT_NCCL(c->api, c->api->AllReduce(c->d_sync, c->d_sync, 1, ncclInt32, ncclSum, c->comm, c->stream));
        RT_CUDA(cudaStreamSynchronize(c->stream));
    }
    cudaFree(c->d_stats);
    cudaFree(c->d_flags);
    cudaFree(c->d_rgb);
    c->d_stats = nullptr;
    c->d_flags = nullptr;
    c->d_rgb = nullptr;
    c->slice_px = 0;
    const size_t padded = slice * size_t(c->world);
    RT_CUDA(cudaMalloc((void **)&c->d_stats, padded * 4 * sizeof(int32_t)));
    RT_CUDA(cudaMalloc((void **)&c->d_flags, padded));
    RT_CUDA(cudaMalloc((void **)&c->d_rgb, padded * 3));
    RT_CUDA(cudaMemset(c->d_stats, 0, padded * 4 * sizeof(int32_t))); // a frame clears its pixels only: the padding stays zero
    c->slice_px = slice;
    return peer_open(c);
}
} // namespace

extern "C" {

int rt_comm_unique_id(uint8_t *id_out) {
    if (!id_out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_comm_unique_id: null argument");
    static_assert(sizeof(ncclUniqueId) == RT_COMM_ID_BYTES, "RT_COMM_ID_BYTES must equal sizeof(ncclUniqueId)");
    NcclApi *api;
    int rc = nccl_api(&api);
    if (rc != RT_OK) return rc;
    ncclUniqueId id;
    RT_NCCL(api, api->GetUniqueId(&id));
    std::memcpy(id_out, &id, sizeof id);
    return RT_OK;
}

int rt_comm_nccl_version(int32_t *version_out, char *path_out, size_t path_cap) {
    NcclApi *api;
    int rc = nccl_api(&api);
    if (rc != RT_OK) return rc;
    int v = 0;
    RT_NCCL(api, api->GetVersion(&v));
    if (version_out) *version_out = v;
    if (path_out && path_cap) {
        std::strncpy(path_out, api->path.c_str(), path_cap - 1);
        path_out[path_cap - 1] = 0;
    }
    return RT_OK;
}

int rt_comm_create(const uint8_t *id, int32_t rank, int32_t world, int32_t device, void *stream, RtComm **out) {
    if (!out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_comm_create: out is null");
    *out = nullptr;
    if ((!id && world > 1) || world < 1 || world > kMaxDevices || rank < 0 || rank >= world) return fail(RT_ERR_INVALID_ARGUMENT, "rt_comm_create: bad id / rank / world");
    int rc = require_device(device);
    if (rc != RT_OK) return rc;
    NcclApi *api = nullptr;
    if (world > 1 && (rc = nccl_api(&api)) != RT_OK) return rc; // a single rank needs no collective and no NCCL
    auto *c = new RtComm();
    c->api = api;
    c->rank = rank;
    c->world = world;
    c->device = device;
    bool ok = true;
    if (stream) {
        c->stream = static_cast<cudaStream_t>(stream);
    } else {
        ok = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) == cudaSuccess;
        c->own_stream = ok;
    }
    ok = ok && c->ev.create();
    if (!ok) {
        comm_free(c);
        return fail(RT_ERR_CUDA, "rt_comm_create: stream / event creation failed");
    }
    if (world > 1) {
        ncclUniqueId uid;
        std::memcpy(&uid, id, sizeof uid);
        ncclResult_t r = api->CommInitRank(&c->comm, world, uid, rank);
        if (r != ncclSuccess) {
            c->comm = nullptr;
            comm_free(c);
            return fail(RT_ERR_CUDA, std::string("ncclCommInitRank: ") + api->GetErrorString(r));
        }
    }
    *out = c;
    return RT_OK;
}

void rt_comm_destroy(RtComm *comm) { comm_free(comm); }

int rt_comm_render(RtComm *c, RtScene *scene, const RtCamera *camera, int32_t max_w, int32_t max_h, const RtRenderOpts *opts, uint8_t *rgb_out,
                   int32_t *sums_out, RtStats *stats) {
    if (!c) return fail(RT_ERR_INVALID_ARGUMENT, "rt_comm_render: null communicator");
    int rc = check_frame_args(scene, camera, max_w, max_h, opts);
    if (rc != RT_OK) return rc;
    if (opts->mode != RT_MODE_MEGAKERNEL) return fail(RT_ERR_UNSUPPORTED, "rt_comm_render: only RT_MODE_MEGAKERNEL is split over ranks");
    if ((rc = prepare_frame(scene, opts)) != RT_OK) return rc;
    auto *ds = static_cast<DeviceScene *>(scene->dev);
    if (ds->device != c->device) return fail(RT_ERR_INVALID_ARGUMENT, "rt_comm_render: the scene lives on another device than the communicator");
    RT_CUDA(cudaSetDevice(c->device));
    const size_t n_pixels = size_t(2 * max_w + 1) * size_t(2 * max_h + 1);
    if ((rc = comm_workspace(c, n_pixels)) != RT_OK) return rc;
    cudaStream_t st = c->stream;
    NcclApi *api = c->api;
    FrameParams fp;
    fill_frame(fp, ds, *camera, max_w, max_h, *opts, c->rank, c->world);
    fp.stats = c->d_stats;
    fp.flags = c->d_flags;
    int launches = 0;
    if ((rc = frame_probe(ds, fp, st, &c->ev, &launches)) != RT_OK) return rc;
    if (fp.adaptive && c->world > 1) RT_NCCL(api, api->AllReduce(c->d_flags, c->d_flags, n_pixels, ncclUint8, ncclMax, c->comm, st));
    if ((rc = frame_main(ds, fp, st, c->ev, &launches)) != RT_OK) return rc;
    if (c->world == 1 || sums_out) {
        // every rank returns the sums: all-reduce them, then divide the whole frame locally
        if (c->world > 1) RT_NCCL(api, api->AllReduce(c->d_stats, c->d_stats, n_pixels * 4, ncclInt32, ncclSum, c->comm, st));
        if ((rc = launch_finalize(c->d_stats, n_pixels, opts->gamma, c->d_rgb, st, &launches)) != RT_OK) return rc;
    } else if (c->peer) {
        // one kernel over peer memory between two 4-byte barriers: this rank's slice into every rank's frame
        RT_NCCL(api, api->AllReduce(c->d_sync, c->d_sync, 1, ncclInt32, ncclSum, c->comm, st)); // every rank's sums are final
        ReduceTargets t{};
        for (int r = 0; r < c->world; ++r) {
            t.stats[r] = c->peer_stats[r];
            t.rgb[r] = c->peer_rgb[r];
        }
        t.world = t.n_rgb = c->world;
        if ((rc = launch_reduce_finalize(t, c->rank, n_pixels, opts->gamma, st, &launches)) != RT_OK) return rc;
        RT_NCCL(api, api->AllReduce(c->d_sync, c->d_sync, 1, ncclInt32, ncclSum, c->comm, st)); // every slice has landed everywhere
    } else {
        // reduce-scatter (in place: rank r's totals land in its own slice), divide the slice, all-gather RGB8 (in place)
        int32_t *slice_stats = c->d_stats + size_t(c->rank) * c->slice_px * 4;
        uint8_t *slice_rgb = c->d_rgb + size_t(c->rank) * c->slice_px * 3;
        RT_NCCL(api, api->ReduceScatter(c->d_stats, slice_stats, c->slice_px * 4, ncclInt32, ncclSum, c->comm, st));
        if ((rc = launch_finalize(slice_stats, c->slice_px, opts->gamma, slice_rgb, st, &launches)) != RT_OK) return rc;
        RT_NCCL(api, api->AllGather(slice_rgb, c->d_rgb, c->slice_px * 3, ncclUint8, c->comm, st));
    }
    if ((rc = frame_finish(ds, fp, c->d_rgb, rgb_out, sums_out, st, c->ev)) != RT_OK) return rc;
    c->last_pixels = n_pixels;
    c->last_adaptive = fp.adaptive != 0;
    c->last_launches = launches;
    if (!rgb_out && !sums_out && !stats) return RT_OK; // device-resident frame: the caller synchronises the stream it gave us
    RT_CUDA(cudaStreamSynchronize(st));
    if (stats) return rt_comm_last_stats(c, scene, stats);
    return RT_OK;
}

int rt_comm_last_stats(RtComm *c, RtScene *scene, RtStats *stats) {
    if (!c || !scene || !scene->dev || !stats) return fail(RT_ERR_INVALID_ARGUMENT, "rt_comm_last_stats: null argument");
    auto *ds = static_cast<DeviceScene *>(scene->dev);
    if (!c->last_pixels) return fail(RT_ERR_INVALID_ARGUMENT, "rt_comm_last_stats: no frame has been rendered on this communicator");
    RT_CUDA(cudaSetDevice(c->device));
    RT_CUDA(cudaEventSynchronize(c->ev.ev[FrameEvents::END])); // the counter copy precedes it
    read_stats(ds, c->last_pixels, c->last_adaptive, c->last_launches, &c->ev, stats); // this rank's paths and rays
    return RT_OK;
}

// 1: the ranks' buffers are mapped into one another (CUDA IPC) and the tail of a frame is the fused peer-memory kernel;
// 0: the NCCL reduce-scatter / all-gather path
int rt_comm_uses_peer_memory(const RtComm *c) { return c && c->peer ? 1 : 0; }

// the frame of the last rt_comm_render as it lies in device memory (RGB8, rows*cols*3; valid until the next call)
int rt_comm_frame(RtComm *c, const uint8_t **d_rgb_out, const int32_t **d_stats_out) {
    if (!c) return fail(RT_ERR_INVALID_ARGUMENT, "rt_comm_frame: null communicator");
    if (d_rgb_out) *d_rgb_out = c->d_rgb;
    if (d_stats_out) *d_stats_out = c->d_stats;
    return RT_OK;
}

} // extern "C"
