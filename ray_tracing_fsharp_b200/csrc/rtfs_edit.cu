// rtfs_edit.cu — rt_scene_update: edits objects and textures of a scene on its device and refits its tree there.
//
// The changed device records (spheres, materials, unbounded objects, textures) are packed on the host into the workspace's
// pinned staging blob as 16-byte words with their destination word in the scene blob, travel in ONE host->device copy, and
// edit_scatter_kernel writes each word to its place.  Image texels go into the texture's pooled array as at creation.
//
// The refit keeps the tree's topology, its leaf order and the device primitive ids, and recomputes the boxes above the moved
// spheres only: work proportional to (spheres moved x depth), not to the scene.  The node records hold each child's box in
// centre / half-extent form, rounded outwards, which is not closed under union, so the refit keeps the min / max form of the
// tree beside it (as the host build left it, uploaded by the first edit that moves a sphere) with a parent link per node and
// per leaf.  refit_mark_kernel counts each node's dirty children; refit_climb_kernel runs one thread per moved leaf, forms
// the leaf box exactly as build_device_layout does (FP64 subtraction and addition of the FP32 values, rounded down and up),
// and climbs: the last child to arrive at a node forms the union of its two child boxes, converts the node with
// device_node_of (the host's function) and goes on to the parent.  min and max are exact and rounding is monotone, so the
// union of rounded leaf boxes is the rounded union, every box equals what a host build of this topology would hold, and no
// result depends on the order of arrival.
#include "rtfs_device.h"

#include <algorithm>
#include <cstring>

using namespace rtfs;

namespace rtfs {

constexpr int kEditThreads = 256;

__global__ void __launch_bounds__(kEditThreads) edit_scatter_kernel(const uint4 *words, const uint32_t *dst, int32_t n, uint4 *blob) {
    const int32_t i = int32_t(blockIdx.x) * kEditThreads + int32_t(threadIdx.x);
    if (i < n) blob[dst[i]] = words[i];
}

// One thread per moved leaf: the first child to mark a node marks the node's own parent in turn, so each dirty child adds
// exactly one to its parent's count (a leaf belongs to one object and indices are unique).
__global__ void __launch_bounds__(kEditThreads) refit_mark_kernel(const int32_t *moved, int32_t n, RefitView r) {
    const int32_t i = int32_t(blockIdx.x) * kEditThreads + int32_t(threadIdx.x);
    if (i >= n) return;
    int32_t link = r.leaf_parent[moved[i]];
    while (link >= 0) {
        const int32_t node = link >> 1;
        if (atomicAdd(&r.dirty[node], 1u) != 0u) return; // another child has marked this node and its ancestors
        link = r.node_parent[node];
    }
}

__device__ __forceinline__ DNode load_minmax(const DNode *p) { // past L1: the other children's boxes were written by other SMs
    DNode d;
    const uint4 *src = reinterpret_cast<const uint4 *>(p);
    uint4 *out = reinterpret_cast<uint4 *>(&d);
#pragma unroll
    for (int q = 0; q < 4; ++q) out[q] = __ldcg(src + q);
    return d;
}

__global__ void __launch_bounds__(kEditThreads) refit_climb_kernel(const int32_t *moved, int32_t n, const float4 *spheres, RefitView r,
                                                                   uint4 *nodes) {
    const int32_t i = int32_t(blockIdx.x) * kEditThreads + int32_t(threadIdx.x);
    if (i >= n) return;
    const int32_t k = moved[i];
    const float4 s = spheres[k];
    const float c[3] = {s.x, s.y, s.z};
    float mn[3], mx[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) { // build_device_layout's leaf box
        mn[a] = round_down(double(c[a]) - double(s.w));
        mx[a] = round_up(double(c[a]) + double(s.w));
    }
    int32_t link = r.leaf_parent[k];
    for (;;) {
        const int32_t node = link >> 1;
        DNode *m = r.minmax + node;
        float *bmn = (link & 1) ? m->r_mn : m->l_mn, *bmx = (link & 1) ? m->r_mx : m->l_mx;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            bmn[a] = mn[a];
            bmx[a] = mx[a];
        }
        const uint32_t need = r.dirty[node]; // read before arriving: the last arrival clears it
        __threadfence();
        if (atomicAdd(&r.arrive[node], 1u) + 1u < need) return; // a sibling still climbs towards this node: it goes on
        __threadfence();
        const DNode box = load_minmax(m);
        const DNode dev = device_node_of(box);
        const uint4 *q = reinterpret_cast<const uint4 *>(&dev);
        nodes[4 * size_t(node) + 0] = q[0]; // the twelve box floats; the child refs (q3) stay
        nodes[4 * size_t(node) + 1] = q[1];
        nodes[4 * size_t(node) + 2] = q[2];
        r.arrive[node] = 0u;
        r.dirty[node] = 0u;
        atomicAdd(r.refit_nodes, 1u);
        link = r.node_parent[node];
        if (link < 0) return; // the root: its own box is stored nowhere
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            mn[a] = fminf(box.l_mn[a], box.r_mn[a]);
            mx[a] = fmaxf(box.l_mx[a], box.r_mx[a]);
        }
    }
}

namespace {

size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

// The refit's state, allocated and uploaded from the host layout by the first edit that moves a sphere (scenes that are
// never edited pay nothing; rt_scene_rebuild leaves it written for the tree it built).  The one-sphere tree's root holds
// the leaf on the left and the never-entered {+inf} box on the right, which no edit touches.
int ensure_refit(RtScene *scene, DeviceScene *ds, RefitView &r) {
    const HostSceneLayout &L = scene->layout;
    const size_t nn = L.nodes.size(), nb = size_t(L.n_bounded);
    size_t total = 0, off_dirty = 0;
    const RefitView offsets = refit_view(nullptr, nn, nb, &total, &off_dirty);
    if (!ds->refit) {
        std::vector<uint8_t> host(off_dirty, 0);
        std::memcpy(host.data(), L.nodes.data(), nn * sizeof(DNode));
        int32_t *np = reinterpret_cast<int32_t *>(host.data() + size_t(offsets.node_parent)),
                *lp = reinterpret_cast<int32_t *>(host.data() + size_t(offsets.leaf_parent));
        np[0] = -1;
        for (size_t i = 0; i < nn; ++i) {
            const DNode &nd = L.nodes[i];
            for (int side = 0; side < 2; ++side) {
                if (side == 1 && L.root_is_leaf && i == 0) continue;
                const int32_t child = side ? nd.right : nd.left, link = int32_t(i << 1) | side;
                if (child >= 0) np[child] = link;
                else lp[~child] = link;
            }
        }
        RT_CUDA(cudaMalloc(&ds->refit, total));
        RT_CUDA(cudaMemcpy(ds->refit, host.data(), off_dirty, cudaMemcpyHostToDevice));
        RT_CUDA(cudaMemset(static_cast<uint8_t *>(ds->refit) + off_dirty, 0, total - off_dirty));
        ds->bytes += total;
    }
    r = refit_view(ds->refit, nn, nb, &total, &off_dirty);
    return RT_OK;
}

} // namespace

RefitView refit_view(void *base, size_t nn, size_t nb, size_t *total, size_t *zeroed_from) {
    const size_t off_np = align256(nn * sizeof(DNode));
    const size_t off_lp = align256(off_np + nn * sizeof(int32_t));
    const size_t off_dirty = align256(off_lp + nb * sizeof(int32_t));
    const size_t off_arrive = align256(off_dirty + nn * sizeof(uint32_t));
    const size_t off_count = align256(off_arrive + nn * sizeof(uint32_t));
    *total = off_count + 256;
    *zeroed_from = off_dirty;
    uint8_t *b = static_cast<uint8_t *>(base);
    return RefitView{reinterpret_cast<DNode *>(b), reinterpret_cast<int32_t *>(b + off_np), reinterpret_cast<int32_t *>(b + off_lp),
                     reinterpret_cast<uint32_t *>(b + off_dirty), reinterpret_cast<uint32_t *>(b + off_arrive),
                     reinterpret_cast<uint32_t *>(b + off_count)};
}

int check_indices(const int32_t *index, int32_t n, int32_t count, const char *what, const char *who) {
    std::vector<int32_t> sorted(index, index + n);
    std::sort(sorted.begin(), sorted.end());
    for (int32_t i = 0; i < n; ++i) {
        if (sorted[i] < 0 || sorted[i] >= count)
            return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": " + what + " index " + std::to_string(sorted[i]) + " is out of range");
        if (i > 0 && sorted[i] == sorted[i - 1])
            return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": " + what + " index " + std::to_string(sorted[i]) + " appears twice");
    }
    return RT_OK;
}

namespace {

bool same_texture(const RtTexture &a, const RtTexture &b) { // every field but the texel pointer, and the texels
    if (a.kind != b.kind || std::memcmp(a.colour, b.colour, 3) != 0 || a.width != b.width || a.height != b.height || a.even != b.even ||
        a.odd != b.odd || a.grid_size != b.grid_size || a.map_radius != b.map_radius)
        return false;
    for (int k = 0; k < 3; ++k)
        if (a.map_centre[k] != b.map_centre[k]) return false;
    return a.kind != RT_TEX_IMAGE || std::memcmp(a.rgb8, b.rgb8, size_t(a.width) * a.height * 3) == 0;
}

} // namespace

void invalidate_wide(RtScene *scene, DeviceScene *ds) {
    HostSceneLayout &L = scene->layout;
    L.wide_nodes.clear();
    L.wide_spheres.clear();
    L.wide_to_dev.clear();
    L.dev_to_wide.clear();
    L.wide_depth = 0;
    if (!ds->wide_blob) return;
    cudaFree(ds->wide_blob);
    ds->wide_blob = nullptr;
    ds->bytes -= ds->wide_bytes;
    ds->wide_bytes = 0;
    ds->wide_depth = 0;
    ds->g.wide_nodes = nullptr;
    ds->g.wide_spheres = nullptr;
    ds->g.wide_to_dev = nullptr;
    ds->g.dev_to_wide = nullptr;
}
void invalidate_reference(RtScene *scene, DeviceScene *ds) {
    scene->ref_built = false;
    scene->ref_tree.clear();
    scene->layout.ref_nodes.clear();
    cudaFree(ds->ref_nodes);
    ds->ref_nodes = nullptr;
    ds->n_ref_nodes = 0;
}

int device_scene_sync_layout(RtScene *scene) {
    if (!scene->layout_stale && !scene->records_stale) return RT_OK;
    auto *ds = static_cast<DeviceScene *>(scene->dev);
    HostSceneLayout &L = scene->layout;
    RT_CUDA(cudaSetDevice(ds->device));
    if (scene->records_stale) { // after rt_scene_rebuild: the records in leaf order, and the caller's index -> device id map
        const size_t nb = size_t(L.n_bounded), nu = size_t(ds->g.n_unbounded);
        L.spheres.resize(nb);
        L.materials.resize(nb + nu);
        L.unbounded.resize(nu);
        L.device_id_of.resize(scene->objects.size());
        RT_CUDA(cudaMemcpy(L.spheres.data(), ds->g.spheres, nb * sizeof(DSphere), cudaMemcpyDeviceToHost));
        RT_CUDA(cudaMemcpy(L.materials.data(), ds->g.mats, (nb + nu) * sizeof(DMaterial), cudaMemcpyDeviceToHost));
        RT_CUDA(cudaMemcpy(L.unbounded.data(), ds->g.unb, nu * sizeof(DUnbounded), cudaMemcpyDeviceToHost));
        RT_CUDA(cudaMemcpy(L.device_id_of.data(), ds->dev_of, L.device_id_of.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
        scene->records_stale = false;
    }
    if (scene->layout_stale) {
        scene->device_nodes.resize(L.nodes.size());
        RT_CUDA(cudaMemcpy(L.nodes.data(), ds->refit, L.nodes.size() * sizeof(DNode), cudaMemcpyDeviceToHost));
        RT_CUDA(cudaMemcpy(scene->device_nodes.data(), ds->g.nodes, L.nodes.size() * sizeof(DNode), cudaMemcpyDeviceToHost));
        scene->layout_stale = false;
    }
    return RT_OK;
}

} // namespace rtfs

extern "C" {

int rt_scene_update(RtScene *scene, const int32_t *object_index, const RtHittable *objects, int32_t n_objects, const int32_t *texture_index,
                    const RtTexture *textures, int32_t n_textures, RtSceneUpdate *info) {
    constexpr const char *who = "rt_scene_update";
    if (!scene) return fail(RT_ERR_INVALID_ARGUMENT, "rt_scene_update: null scene");
    if (n_objects < 0 || n_textures < 0 || (n_objects > 0 && (!object_index || !objects)) || (n_textures > 0 && (!texture_index || !textures)))
        return fail(RT_ERR_INVALID_ARGUMENT, "rt_scene_update: bad array arguments");
    if (scene->device < 0 || !scene->dev)
        return fail(RT_ERR_UNSUPPORTED, "rt_scene_update: the scene was created without a device (device = -1)");
    const int32_t n_obj_all = int32_t(scene->objects.size()), n_tex_all = int32_t(scene->textures.size());
    int rc = check_indices(object_index, n_objects, n_obj_all, "object", who);
    if (rc == RT_OK) rc = check_indices(texture_index, n_textures, n_tex_all, "texture", who);
    if (rc != RT_OK) return rc;

    // ---- every check before any change: structure, then what rt_scene_create checks in the edited arrays
    auto structural = [&](const std::string &what) {
        return fail(RT_ERR_INVALID_ARGUMENT, "rt_scene_update: " + what + " (a structural change: create a new scene)");
    };
    for (int32_t i = 0; i < n_objects; ++i) {
        const int32_t at = object_index[i];
        const RtHittable &h = objects[i], &old = scene->objects[size_t(at)];
        if (h.shape != old.shape) return structural("object " + std::to_string(at) + " changes its shape");
        if (h.shape == RT_SHAPE_SPHERE && (h.radius >= 0.0) != (old.radius >= 0.0))
            return structural("sphere " + std::to_string(at) + " changes the sign of its radius, i.e. whether the tree holds it");
        if ((rc = check_object(h, at, n_tex_all, who)) != RT_OK) return fail(RT_ERR_INVALID_ARGUMENT, rt_last_error());
    }
    for (int32_t j = 0; j < n_textures; ++j) {
        const int32_t at = texture_index[j];
        const RtTexture &t = textures[j], &old = scene->textures[size_t(at)];
        if (t.kind != old.kind) return structural("texture " + std::to_string(at) + " changes its kind");
        if (t.kind == RT_TEX_IMAGE && (t.width != old.width || t.height != old.height))
            return structural("image texture " + std::to_string(at) + " changes its size");
    }
    if (n_textures > 0) {
        std::vector<RtTexture> table(scene->textures);
        for (int32_t j = 0; j < n_textures; ++j) table[size_t(texture_index[j])] = textures[j];
        if ((rc = check_textures(table.data(), n_tex_all, who)) != RT_OK) return fail(RT_ERR_INVALID_ARGUMENT, rt_last_error());
    }
    if ((rc = require_device(scene->device)) != RT_OK) return rc;
    if (scene->records_stale && (rc = device_scene_sync_layout(scene)) != RT_OK) return rc; // after a rebuild: the records it placed

    // ---- the changed device records, as 16-byte words with their destination word in the scene blob
    auto *ds = static_cast<DeviceScene *>(scene->dev);
    HostSceneLayout &L = scene->layout;
    const uint8_t *blob = static_cast<const uint8_t *>(ds->blob);
    auto word_of = [&](const void *p) { return uint32_t((static_cast<const uint8_t *>(p) - blob) / 16); };
    const uint32_t w_sph = word_of(ds->g.spheres), w_mat = word_of(ds->g.mats), w_unb = word_of(ds->g.unb), w_tex = word_of(ds->g.tex);
    std::vector<uint4> words;
    std::vector<uint32_t> dst;
    std::vector<int32_t> moved; // device ids of the bounded spheres that moved
    auto push = [&](uint32_t at, const void *rec, size_t bytes) {
        for (size_t q = 0; q < bytes / 16; ++q) {
            uint4 w;
            std::memcpy(&w, static_cast<const uint8_t *>(rec) + 16 * q, 16);
            words.push_back(w);
            dst.push_back(at + uint32_t(q));
        }
    };
    RtSceneUpdate out{};
    bool spheres_reshaped = false; // a sphere's centre or radius changed: the reference-topology tree is stale
    for (int32_t i = 0; i < n_objects; ++i) {
        const int32_t at = object_index[i];
        const RtHittable &h = objects[i];
        RtHittable &old = scene->objects[size_t(at)];
        if (std::memcmp(&h, &old, sizeof h) != 0) out.objects += 1;
        if (h.shape == RT_SHAPE_SPHERE && (std::memcmp(h.p, old.p, sizeof h.p) != 0 || h.radius != old.radius)) spheres_reshaped = true;
        const int32_t dev = L.device_id_of[size_t(at)]; // -1: a bounded sphere of negative radius, never hit (F16)
        if (dev >= 0) {
            const DMaterial m = make_material(h, at);
            DMaterial &om = L.materials[size_t(dev)];
            if (std::memcmp(&m, &om, sizeof m) != 0) {
                ds->n_textured += (m.texture >= 0 ? 1 : 0) - (om.texture >= 0 ? 1 : 0);
                push(w_mat + 2u * uint32_t(dev), &m, sizeof m);
                om = m;
            }
            if (dev < L.n_bounded) {
                const DSphere sp{float(h.p[0]), float(h.p[1]), float(h.p[2]), float(h.radius)};
                if (std::memcmp(&sp, &L.spheres[size_t(dev)], sizeof sp) != 0) {
                    push(w_sph + uint32_t(dev), &sp, sizeof sp);
                    moved.push_back(dev);
                    L.spheres[size_t(dev)] = sp;
                }
            } else {
                const DUnbounded u = make_unbounded(h);
                DUnbounded &ou = L.unbounded[size_t(dev - L.n_bounded)];
                if (std::memcmp(&u, &ou, sizeof u) != 0) {
                    ds->n_fp64 += (u.fp32 ? 0 : 1) - (ou.fp32 ? 0 : 1);
                    push(w_unb + 4u * uint32_t(dev - L.n_bounded), &u, sizeof u);
                    ou = u;
                }
            }
        }
        old = h;
    }
    struct TexelCopy {
        cudaArray_t array;
        std::vector<uchar4> texels;
        int32_t w, h;
    };
    std::vector<TexelCopy> texel_copies;
    if (n_textures > 0) {
        std::vector<int32_t> image_slot(size_t(n_tex_all), -1); // ds->images holds the image textures in index order
        for (int32_t t = 0, k = 0; t < n_tex_all; ++t)
            if (scene->textures[size_t(t)].kind == RT_TEX_IMAGE) image_slot[size_t(t)] = k++;
        for (int32_t j = 0; j < n_textures; ++j) {
            const int32_t at = texture_index[j];
            const RtTexture &t = textures[j];
            RtTexture &old = scene->textures[size_t(at)];
            if (same_texture(t, old)) continue;
            out.textures += 1;
            DTexture d = device_texture_of(t);
            if (t.kind == RT_TEX_IMAGE) {
                const PooledTexture &pt = ds->images[size_t(image_slot[size_t(at)])];
                d.tex = pt.object;
                const size_t bytes = size_t(t.width) * t.height * 3;
                if (std::memcmp(t.rgb8, old.rgb8, bytes) != 0) {
                    texel_copies.push_back(TexelCopy{pt.array, texels_of(t), t.width, t.height});
                    scene->texture_pixels[size_t(at)].assign(t.rgb8, t.rgb8 + bytes);
                }
            }
            push(w_tex + 4u * uint32_t(at), &d, sizeof d);
            old = t;
            old.rgb8 = t.kind == RT_TEX_IMAGE ? scene->texture_pixels[size_t(at)].data() : nullptr;
        }
    }

    // ---- one copy, the scatter, the refit
    DeviceWorkspace *ws = ds->ws;
    cudaStream_t st = ws->stream;
    RT_CUDA(cudaSetDevice(ds->device));
    RefitView r{};
    if (!moved.empty() && (rc = ensure_refit(scene, ds, r)) != RT_OK) return rc;
    const int32_t n_words = int32_t(words.size()), n_moved = int32_t(moved.size());
    const size_t off_dst = align256(words.size() * sizeof(uint4)), off_moved = align256(off_dst + dst.size() * sizeof(uint32_t));
    const size_t bytes = off_moved + moved.size() * sizeof(int32_t);
    if (ws->h_blob_cap < bytes) {
        if (ws->h_blob) cudaFreeHost(ws->h_blob);
        ws->h_blob = nullptr;
        ws->h_blob_cap = 0;
        RT_CUDA(cudaMallocHost(&ws->h_blob, bytes));
        ws->h_blob_cap = bytes;
    }
    if (ds->edit_stage_cap < bytes) {
        cudaFree(ds->edit_stage);
        ds->edit_stage = nullptr;
        ds->edit_stage_cap = 0;
        RT_CUDA(cudaMalloc(&ds->edit_stage, bytes));
        ds->edit_stage_cap = bytes;
    }
    uint8_t *host = static_cast<uint8_t *>(ws->h_blob);
    if (n_words) {
        std::memcpy(host, words.data(), words.size() * sizeof(uint4));
        std::memcpy(host + off_dst, dst.data(), dst.size() * sizeof(uint32_t));
    }
    if (n_moved) std::memcpy(host + off_moved, moved.data(), moved.size() * sizeof(int32_t));
    const uint8_t *stage = static_cast<const uint8_t *>(ds->edit_stage);
    const int32_t *d_moved = reinterpret_cast<const int32_t *>(stage + off_moved);
    uint32_t refit_nodes = 0;
    RT_CUDA(ws->ev.record(FrameEvents::BEGIN, st));
    for (const TexelCopy &c : texel_copies)
        RT_CUDA(cudaMemcpy2DToArrayAsync(c.array, 0, 0, c.texels.data(), size_t(c.w) * sizeof(uchar4), size_t(c.w) * sizeof(uchar4), size_t(c.h),
                                         cudaMemcpyHostToDevice, st));
    if (bytes) RT_CUDA(cudaMemcpyAsync(ds->edit_stage, host, bytes, cudaMemcpyHostToDevice, st));
    if (n_words) {
        edit_scatter_kernel<<<unsigned((n_words + kEditThreads - 1) / kEditThreads), kEditThreads, 0, st>>>(
            reinterpret_cast<const uint4 *>(stage), reinterpret_cast<const uint32_t *>(stage + off_dst), n_words, static_cast<uint4 *>(ds->blob));
        RT_CUDA(cudaGetLastError());
        out.launches += 1;
    }
    if (n_moved) {
        const unsigned blocks = unsigned((n_moved + kEditThreads - 1) / kEditThreads);
        RT_CUDA(cudaMemsetAsync(r.refit_nodes, 0, sizeof(uint32_t), st));
        refit_mark_kernel<<<blocks, kEditThreads, 0, st>>>(d_moved, n_moved, r);
        RT_CUDA(cudaGetLastError());
        refit_climb_kernel<<<blocks, kEditThreads, 0, st>>>(d_moved, n_moved, ds->g.spheres, r,
                                                            reinterpret_cast<uint4 *>(const_cast<uint4 *>(ds->g.nodes)));
        RT_CUDA(cudaGetLastError());
        out.launches += 2;
        RT_CUDA(cudaMemcpyAsync(&refit_nodes, r.refit_nodes, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    }
    RT_CUDA(ws->ev.record(FrameEvents::END, st));
    RT_CUDA(cudaStreamSynchronize(st));

    // ---- the scene's state: lean, the derived trees, the edit count
    ds->lean = ds->n_fp64 == 0 && ds->n_textured == 0;
    if (n_moved) {
        scene->layout_stale = true; // layout.nodes: downloaded when a host consumer asks (device_scene_sync_layout)
        scene->sah_built = false;
        invalidate_wide(scene, ds);
    }
    if (spheres_reshaped) invalidate_reference(scene, ds);
    if (n_objects + n_textures > 0) scene->generation += 1;
    if (info) {
        out.spheres_moved = n_moved;
        out.nodes_refit = int32_t(refit_nodes);
        out.generation = scene->generation;
        out.device_ms = ws->ev.ms(FrameEvents::BEGIN, FrameEvents::END);
        *info = out;
    }
    return RT_OK;
}

} // extern "C"
