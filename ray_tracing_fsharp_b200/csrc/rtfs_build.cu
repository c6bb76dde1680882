// rtfs_build.cu — rt_scene_rebuild: removes and appends objects of a scene and builds its tree on the device.
//
// The tree is built by PLOC, parallel locally-ordered clustering (Meister & Bittner, "Parallel Locally-Ordered Clustering for
// Bounding Volume Hierarchy Construction", TVCG 2018), over the FP32 sphere boxes.  Every step is a pure function of the
// object array after the call, so the tree does not depend on the scene's history or on scheduling:
//   1. collect: the survivors' device records are gathered from the scene blob into arrays in the new caller order (their
//      material's host_index rewritten), the appended records follow from one host->device copy; the centroid bounds are an
//      exact min / max reduction and the lean counts integer sums;
//   2. sort: 30-bit Morton codes of the FP32 centres over the centroid bounds, keys (morton << 32 | caller index), sorted
//      by cub::DeviceRadixSort (the keys are unique, so the order is);
//   3. cluster: each cluster's nearest neighbour among the kPlocRadius clusters either side (distance: the FP32 surface
//      area of the union box, rounded in a written order; ties to the lower index); mutual nearest neighbours merge into
//      the lower slot, and an order-keeping prefix sum compacts the clusters.  The pair of least distance, lowest index
//      first, is always mutual, so every iteration merges;
//   4. flatten: top-down, one launch per clustering iteration (every node's parent was made by a later one), each node
//      learns its DFS pre-order index, its first leaf and its depth, writes its min / max record and its parent links
//      (the refit's state: rt_scene_update refits this tree) and its device record (device_node_of), and places the
//      spheres and materials of its leaf children in leaf order.  Unbounded objects follow in array order.
// tests/ploc_rule.py restates all of it in numpy; the device tree equals it node for node.
//
// A tree deeper than the walk stacks allow (60, rt_scene_create's limit) is replaced by the host SAH build of the same
// array, uploaded as rt_scene_create would (on_device = 0).
#include "rtfs_device.h"

#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>

using namespace rtfs;

namespace rtfs {

constexpr int kBuildThreads = 256;
constexpr int kScanThreads = 1024; // one element per thread: a block scans 1024
constexpr int kPlocRadius = 16;    // the search radius of the clustering (tests/ploc_rule.py: RADIUS)
constexpr int kMaxTreeDepth = 60;  // rt_scene_create's limit: the walk stacks are sized from the depth

// the class of an object of the new array: no device record (a bounded sphere of negative radius, F16), a sphere of the
// tree, an unbounded object
enum : int32_t { OBJ_NONE = 0, OBJ_BOUNDED = 1, OBJ_UNBOUNDED = 2 };

// what the builder counts, on the device; the host sets the initial values in the staged copy
struct BuildCounters {
    uint32_t n_fp64, n_textured, depth, pad0;
    int32_t cmin[3], pad1; // the centroid bounds as order-preserving integers (float_key)
    int32_t cmax[3], pad2;
    unsigned long long total; // the grand total of the last scan
    unsigned long long pad3;
};
static_assert(sizeof(BuildCounters) == 64, "BuildCounters is one 64-byte block");

// a cluster: its box, its tree ref (>= 0 a node being built, < 0 the leaf of sorted position ~ref) and its leaf count
struct Cluster {
    float mn[3], mx[3];
    int32_t ref, leaves;
};
// a node being built, numbered in order of creation: its two children's boxes and refs, its leaf count
struct BuildNode {
    float l_mn[3], l_mx[3], r_mn[3], r_mx[3];
    int32_t left, right, leaves, pad;
};

__device__ __forceinline__ int32_t float_key(float f) { // the order of floats as signed integers (-0 below +0)
    const int32_t k = __float_as_int(f);
    return k >= 0 ? k : k ^ 0x7fffffff;
}
__device__ __forceinline__ float key_float(int32_t k) { return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff); }

// the clustering distance: the FP32 surface area (halved) of the union of two boxes, in this order and without contraction;
// NaN (an infinite extent times a zero one) counts as +inf, so that distances are totally ordered
__device__ __forceinline__ float union_area(const Cluster &a, const Cluster &b) {
    float d[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) d[k] = __fsub_rn(fmaxf(a.mx[k], b.mx[k]), fminf(a.mn[k], b.mn[k]));
    const float s = __fadd_rn(__fadd_rn(__fmul_rn(d[0], d[1]), __fmul_rn(d[1], d[2])), __fmul_rn(d[2], d[0]));
    return s != s ? __int_as_float(0x7f800000) : s;
}

// exclusive prefix sum of v over the block (blockDim.x a multiple of 32, at most 1024); *total: the block's sum
__device__ unsigned long long block_exclusive_scan(unsigned long long v, unsigned long long *total) {
    __shared__ unsigned long long warp_sums[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
    unsigned long long x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_sums[warp] = x;
    __syncthreads();
    if (warp == 0) {
        unsigned long long w = lane < warps ? warp_sums[lane] : 0ull;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long y = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += y;
        }
        warp_sums[lane] = w;
    }
    __syncthreads();
    const unsigned long long before = warp == 0 ? 0ull : warp_sums[warp - 1];
    *total = warp_sums[warps - 1];
    __syncthreads(); // warp_sums may be reused by the caller's next scan
    return before + x - v;
}

// The scans count two things at once, packed as lo | hi << 32 (neither reaches 2^32).  The exclusive prefix of element i is
// out[i] + top[i / kScanThreads] once scan_top_kernel has run.
struct KeepFlag { // the old objects that survive
    const uint8_t *removed;
    __device__ unsigned long long operator()(int32_t i) const { return removed[i] ? 0ull : 1ull; }
};
struct ClassFlag { // spheres of the tree (lo) and unbounded objects (hi) of the new array
    const int32_t *cls;
    __device__ unsigned long long operator()(int32_t i) const {
        return cls[i] == OBJ_BOUNDED ? 1ull : (cls[i] == OBJ_UNBOUNDED ? 1ull << 32 : 0ull);
    }
};
__device__ __forceinline__ bool ploc_mutual(const int32_t *nn, int32_t i) { return nn[nn[i]] == i; }
struct ClusterFlag { // clusters that stay a slot (lo: every one but the higher of a merging pair) and merges (hi)
    const int32_t *nn;
    __device__ unsigned long long operator()(int32_t i) const {
        const int32_t j = nn[i];
        const bool mutual = ploc_mutual(nn, i);
        return (mutual && j < i) ? 0ull : (1ull | (mutual ? 1ull << 32 : 0ull));
    }
};

template <class Flag>
__global__ void __launch_bounds__(kScanThreads) scan_local_kernel(Flag flag, int32_t n, unsigned long long *out, unsigned long long *top) {
    const int32_t i = int32_t(blockIdx.x) * kScanThreads + int32_t(threadIdx.x);
    unsigned long long total;
    const unsigned long long ex = block_exclusive_scan(i < n ? flag(i) : 0ull, &total);
    if (i < n) out[i] = ex;
    if (threadIdx.x == 0) top[blockIdx.x] = total;
}

// one block: the blocks' totals -> their exclusive prefix, and the grand total
__global__ void __launch_bounds__(kScanThreads) scan_top_kernel(unsigned long long *top, int32_t n_blocks, unsigned long long *grand) {
    unsigned long long carry = 0;
    for (int32_t base = 0; base < n_blocks; base += kScanThreads) {
        const int32_t i = base + int32_t(threadIdx.x);
        unsigned long long total;
        const unsigned long long ex = block_exclusive_scan(i < n_blocks ? top[i] : 0ull, &total);
        if (i < n_blocks) top[i] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) *grand = carry;
}
__device__ __forceinline__ unsigned long long scanned(const unsigned long long *out, const unsigned long long *top, int32_t i) {
    return out[i] + top[i / kScanThreads];
}

__global__ void __launch_bounds__(kBuildThreads) rebuild_mark_kernel(const int32_t *remove, int32_t n, uint8_t *removed) {
    const int32_t i = int32_t(blockIdx.x) * kBuildThreads + int32_t(threadIdx.x);
    if (i < n) removed[remove[i]] = 1;
}

// the records of the new array in caller order: thread t < n_old gathers old object t if it survives, the others take the
// appended records (the host made their materials with their new index, which is their slot); the centroid bounds and the
// lean counts accumulate (min, max and integer sums: free of order)
struct CollectArgs {
    int32_t n_old, n_append, nb_old;
    const uint8_t *removed;
    const unsigned long long *kscan, *ktop;
    const int32_t *dev_of; // old caller index -> old device id
    const float4 *old_spheres;
    const DMaterial *old_mats;
    const DUnbounded *old_unb;
    const int32_t *app_cls; // the appended records, staged by the host
    const float4 *app_sph;
    const DMaterial *app_mat;
    const DUnbounded *app_unb;
    int32_t *cls; // out, per new caller index
    float4 *sph;
    DMaterial *mat;
    DUnbounded *unb;
    BuildCounters *counters;
};
__global__ void __launch_bounds__(kBuildThreads) rebuild_collect_kernel(const CollectArgs a) {
    const int32_t t = int32_t(blockIdx.x) * kBuildThreads + int32_t(threadIdx.x);
    int32_t c = -1, at = 0;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    DMaterial m{};
    DUnbounded u{};
    if (t < a.n_old && !a.removed[t]) {
        at = int32_t(scanned(a.kscan, a.ktop, t) & 0xffffffffu);
        const int32_t dev = a.dev_of[t];
        c = dev < 0 ? OBJ_NONE : (dev < a.nb_old ? OBJ_BOUNDED : OBJ_UNBOUNDED);
        if (c != OBJ_NONE) {
            m = a.old_mats[dev];
            m.host_index = at;
        }
        if (c == OBJ_BOUNDED) s = a.old_spheres[dev];
        if (c == OBJ_UNBOUNDED) u = a.old_unb[dev - a.nb_old];
    } else if (t >= a.n_old && t < a.n_old + a.n_append) {
        const int32_t j = t - a.n_old;
        c = a.app_cls[j];
        m = a.app_mat[j];
        at = m.host_index;
        if (c == OBJ_BOUNDED) s = a.app_sph[j];
        if (c == OBJ_UNBOUNDED) u = a.app_unb[j];
    }
    if (c >= 0) a.cls[at] = c;
    if (c >= OBJ_BOUNDED) a.mat[at] = m;
    if (c == OBJ_BOUNDED) a.sph[at] = s;
    if (c == OBJ_UNBOUNDED) a.unb[at] = u;
    // one atomic per warp and quantity
    const bool bounded = c == OBJ_BOUNDED;
    const int32_t big = 0x7fffffff, small = int32_t(0x80000000u);
    const int32_t kx = bounded ? float_key(s.x) : big, ky = bounded ? float_key(s.y) : big, kz = bounded ? float_key(s.z) : big;
    const int32_t mnx = __reduce_min_sync(0xffffffffu, kx), mny = __reduce_min_sync(0xffffffffu, ky), mnz = __reduce_min_sync(0xffffffffu, kz);
    const int32_t mxx = __reduce_max_sync(0xffffffffu, bounded ? kx : small), mxy = __reduce_max_sync(0xffffffffu, bounded ? ky : small),
                  mxz = __reduce_max_sync(0xffffffffu, bounded ? kz : small);
    const unsigned n_tex = __popc(__ballot_sync(0xffffffffu, c >= OBJ_BOUNDED && m.texture >= 0));
    const unsigned n_fp64 = __popc(__ballot_sync(0xffffffffu, c == OBJ_UNBOUNDED && u.fp32 == 0));
    if ((threadIdx.x & 31) == 0) {
        if (mnx != big) {
            atomicMin(&a.counters->cmin[0], mnx);
            atomicMin(&a.counters->cmin[1], mny);
            atomicMin(&a.counters->cmin[2], mnz);
            atomicMax(&a.counters->cmax[0], mxx);
            atomicMax(&a.counters->cmax[1], mxy);
            atomicMax(&a.counters->cmax[2], mxz);
        }
        if (n_tex) atomicAdd(&a.counters->n_textured, n_tex);
        if (n_fp64) atomicAdd(&a.counters->n_fp64, n_fp64);
    }
}

// the 10 bits of v spread to every third bit
__device__ __forceinline__ uint32_t spread_bits(uint32_t v) {
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}
// an axis of a centre quantised to 10 bits over the centroid bounds: floor((c - lo) * (1024 / (hi - lo))), at most 1023
__device__ __forceinline__ uint32_t morton_axis(float c, float lo, float hi) {
    const float ext = __fsub_rn(hi, lo);
    if (!(ext > 0.f)) return 0u;
    const float q = __fmul_rn(__fsub_rn(c, lo), __fdiv_rn(1024.f, ext));
    return q >= 1023.f ? 1023u : uint32_t(q);
}
// keys (morton << 32 | caller index) of the spheres of the tree; every other object sorts last
__global__ void __launch_bounds__(kBuildThreads) rebuild_keys_kernel(const int32_t *cls, const float4 *sph, int32_t n, const BuildCounters *counters,
                                                                      unsigned long long *keys) {
    const int32_t i = int32_t(blockIdx.x) * kBuildThreads + int32_t(threadIdx.x);
    if (i >= n) return;
    if (cls[i] != OBJ_BOUNDED) {
        keys[i] = ~0ull;
        return;
    }
    const float4 s = sph[i];
    const float c[3] = {s.x, s.y, s.z};
    uint32_t m = 0;
#pragma unroll
    for (int a = 0; a < 3; ++a) m |= spread_bits(morton_axis(c[a], key_float(counters->cmin[a]), key_float(counters->cmax[a]))) << (2 - a);
    keys[i] = (static_cast<unsigned long long>(m) << 32) | uint32_t(i);
}

// build_device_layout's leaf box of a sphere: the FP64 difference and sum of the FP32 centre and radius, rounded outwards
__device__ __forceinline__ void leaf_box(const float4 s, float *mn, float *mx) {
    const float c[3] = {s.x, s.y, s.z};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        mn[a] = round_down(double(c[a]) - double(s.w));
        mx[a] = round_up(double(c[a]) + double(s.w));
    }
}

__global__ void __launch_bounds__(kBuildThreads) ploc_init_kernel(const unsigned long long *sorted, const float4 *sph, int32_t nb, Cluster *out) {
    const int32_t p = int32_t(blockIdx.x) * kBuildThreads + int32_t(threadIdx.x);
    if (p >= nb) return;
    Cluster c;
    leaf_box(sph[uint32_t(sorted[p])], c.mn, c.mx);
    c.ref = ~p;
    c.leaves = 1;
    out[p] = c;
}

// each cluster's nearest neighbour within kPlocRadius slots either side: least union_area, ties to the lower index
__global__ void __launch_bounds__(kBuildThreads) ploc_nearest_kernel(const Cluster *cl, int32_t m, int32_t *nn) {
    const int32_t i = int32_t(blockIdx.x) * kBuildThreads + int32_t(threadIdx.x);
    if (i >= m) return;
    const Cluster me = cl[i];
    const int32_t lo = max(0, i - kPlocRadius), hi = min(m - 1, i + kPlocRadius);
    int32_t best = -1;
    float best_d = 0.f;
    for (int32_t j = lo; j <= hi; ++j) {
        if (j == i) continue;
        const float d = union_area(me, cl[j]);
        if (best < 0 || d < best_d) {
            best = j;
            best_d = d;
        }
    }
    nn[i] = best;
}

// mutual pairs merge into the lower slot as node `node_base + (merges before it)`, the others move to their compacted slot
__global__ void __launch_bounds__(kBuildThreads) ploc_merge_kernel(const Cluster *cl, int32_t m, const int32_t *nn, const unsigned long long *fscan,
                                                                   const unsigned long long *ftop, int32_t node_base, Cluster *out, BuildNode *nodes) {
    const int32_t i = int32_t(blockIdx.x) * kBuildThreads + int32_t(threadIdx.x);
    if (i >= m) return;
    const int32_t j = nn[i];
    const bool mutual = ploc_mutual(nn, i);
    if (mutual && j < i) return; // merged into slot j
    const unsigned long long at = scanned(fscan, ftop, i);
    const int32_t slot = int32_t(at & 0xffffffffu);
    const Cluster a = cl[i];
    if (!mutual) {
        out[slot] = a;
        return;
    }
    const Cluster b = cl[j];
    const int32_t id = node_base + int32_t(at >> 32);
    BuildNode n;
    Cluster u;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        n.l_mn[k] = a.mn[k];
        n.l_mx[k] = a.mx[k];
        n.r_mn[k] = b.mn[k];
        n.r_mx[k] = b.mx[k];
        u.mn[k] = fminf(a.mn[k], b.mn[k]);
        u.mx[k] = fmaxf(a.mx[k], b.mx[k]);
    }
    n.left = a.ref;
    n.right = b.ref;
    n.leaves = a.leaves + b.leaves;
    n.pad = 0;
    nodes[id] = n;
    u.ref = id;
    u.leaves = n.leaves;
    out[slot] = u;
}

// where the flattened tree and the records go
struct PlaceArgs {
    const unsigned long long *sorted; // sorted keys: leaf p is the caller's object uint32(sorted[p])
    const float4 *sph;
    const DMaterial *mat;
    RefitView r;
    uint4 *nodes; // the device records in the scene blob
    float4 *spheres;
    DMaterial *mats;
    int32_t *dev_of;
    BuildCounters *counters;
};
// a leaf child of the node at DFS index d: the sphere of sorted position p becomes device primitive q
__device__ __forceinline__ void place_leaf(const PlaceArgs &a, int32_t p, int32_t q, int32_t link) {
    const uint32_t idx = uint32_t(a.sorted[p]);
    a.spheres[q] = a.sph[idx];
    a.mats[q] = a.mat[idx];
    a.dev_of[idx] = q;
    a.r.leaf_parent[q] = link;
}
__device__ __forceinline__ void write_node(const PlaceArgs &a, int32_t d, const DNode &mm) {
    a.r.minmax[d] = mm;
    const DNode dev = device_node_of(mm);
    const uint4 *q = reinterpret_cast<const uint4 *>(&dev);
#pragma unroll
    for (int k = 0; k < 4; ++k) a.nodes[4 * size_t(d) + k] = q[k];
}

// the nodes [first, first + count) made by one clustering iteration; state[t] = {DFS index, first leaf, depth} was set by the
// node's parent (the root's by the host)
__global__ void __launch_bounds__(kBuildThreads) ploc_flatten_kernel(const BuildNode *bn, int4 *state, int32_t first, int32_t count, PlaceArgs a) {
    const int32_t k = int32_t(blockIdx.x) * kBuildThreads + int32_t(threadIdx.x);
    if (k >= count) return;
    const int32_t t = first + k;
    const BuildNode n = bn[t];
    const int4 st = state[t];
    const int32_t d = st.x, lo = st.y, depth = st.z;
    const int32_t leaves_l = n.left < 0 ? 1 : bn[n.left].leaves;
    DNode mm;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        mm.l_mn[c] = n.l_mn[c];
        mm.l_mx[c] = n.l_mx[c];
        mm.r_mn[c] = n.r_mn[c];
        mm.r_mx[c] = n.r_mx[c];
    }
    mm.pad0 = mm.pad1 = 0;
    if (n.left >= 0) {
        const int32_t dl = d + 1;
        state[n.left] = make_int4(dl, lo, depth + 1, 0);
        a.r.node_parent[dl] = d << 1;
        mm.left = dl;
    } else {
        place_leaf(a, ~n.left, lo, d << 1);
        mm.left = ~lo;
    }
    if (n.right >= 0) {
        const int32_t dr = d + leaves_l; // past this node and the leaves_l - 1 nodes of the left subtree
        state[n.right] = make_int4(dr, lo + leaves_l, depth + 1, 0);
        a.r.node_parent[dr] = (d << 1) | 1;
        mm.right = dr;
    } else {
        place_leaf(a, ~n.right, lo + leaves_l, (d << 1) | 1);
        mm.right = ~(lo + leaves_l);
    }
    write_node(a, d, mm);
    atomicMax(&a.counters->depth, uint32_t(depth));
}

// one sphere: a node with the leaf on the left and the never-entered box {+inf} on the right, as the host builds it
__global__ void ploc_single_kernel(PlaceArgs a) {
    DNode mm;
    float4 s = a.sph[uint32_t(a.sorted[0])];
    leaf_box(s, mm.l_mn, mm.l_mx);
    for (int c = 0; c < 3; ++c) mm.r_mn[c] = mm.r_mx[c] = __int_as_float(0x7f800000);
    mm.left = mm.right = ~0;
    mm.pad0 = mm.pad1 = 0;
    place_leaf(a, 0, 0, 0);
    a.r.node_parent[0] = -1;
    write_node(a, 0, mm);
    a.counters->depth = 1u;
}

// unbounded objects after the spheres, in array order; objects without a record map to -1
__global__ void __launch_bounds__(kBuildThreads) rebuild_place_unbounded_kernel(const int32_t *cls, const unsigned long long *cscan, const unsigned long long *ctop,
                                                                                 int32_t n, int32_t nb, const DMaterial *mat, const DUnbounded *unb,
                                                                                 DMaterial *mats_out, DUnbounded *unb_out, int32_t *dev_of) {
    const int32_t i = int32_t(blockIdx.x) * kBuildThreads + int32_t(threadIdx.x);
    if (i >= n) return;
    const int32_t c = cls[i];
    if (c == OBJ_NONE) dev_of[i] = -1;
    if (c != OBJ_UNBOUNDED) return;
    const int32_t r = int32_t(scanned(cscan, ctop, i) >> 32);
    mats_out[nb + r] = mat[i];
    unb_out[r] = unb[i];
    dev_of[i] = nb + r;
}

namespace {

size_t align256(size_t x) { return (x + 255) & ~size_t(255); }
unsigned blocks_for(size_t n, int threads) { return unsigned((n + size_t(threads) - 1) / size_t(threads)); }

// a bump allocator over offsets: first with base = null to size, then over the allocation
struct Carve {
    uint8_t *base;
    size_t at = 0;
    template <class T>
    T *take(size_t n) {
        T *p = reinterpret_cast<T *>(base + at);
        at = align256(at + n * sizeof(T));
        return p;
    }
};

// the class of an object (what its device record is)
int32_t class_of(const RtHittable &h) {
    if (h.shape != RT_SHAPE_SPHERE) return OBJ_UNBOUNDED;
    return h.radius < 0.0 ? OBJ_NONE : OBJ_BOUNDED;
}

// a scan of n elements: the local kernel, then the top kernel; returns the number of launches
template <class Flag>
int launch_scan(Flag flag, int32_t n, unsigned long long *out, unsigned long long *top, unsigned long long *grand, cudaStream_t st) {
    const unsigned blocks = std::max(1u, blocks_for(size_t(n), kScanThreads));
    scan_local_kernel<<<blocks, kScanThreads, 0, st>>>(flag, n, out, top);
    scan_top_kernel<<<1, kScanThreads, 0, st>>>(top, int32_t(blocks), grand);
    return 2;
}

} // namespace
} // namespace rtfs

extern "C" {

int rt_scene_rebuild(RtScene *scene, const int32_t *remove, int32_t n_remove, const RtHittable *append, int32_t n_append, RtSceneRebuild *info) {
    constexpr const char *who = "rt_scene_rebuild";
    if (!scene) return fail(RT_ERR_INVALID_ARGUMENT, "rt_scene_rebuild: null scene");
    if (n_remove < 0 || n_append < 0 || (n_remove > 0 && !remove) || (n_append > 0 && !append))
        return fail(RT_ERR_INVALID_ARGUMENT, "rt_scene_rebuild: bad array arguments");
    if (scene->device < 0 || !scene->dev)
        return fail(RT_ERR_UNSUPPORTED, "rt_scene_rebuild: the scene was created without a device (device = -1)");
    const int32_t n_old = int32_t(scene->objects.size()), n_tex = int32_t(scene->textures.size());
    int rc = check_indices(remove, n_remove, n_old, "remove", who);
    if (rc != RT_OK) return rc;
    const int64_t n_new64 = int64_t(n_old) - n_remove + n_append;
    if (n_new64 > int64_t(0x7fffffff)) return fail(RT_ERR_INVALID_ARGUMENT, "rt_scene_rebuild: more than 2^31 - 1 objects");
    const int32_t n_surv = n_old - n_remove, n = int32_t(n_new64);
    for (int32_t j = 0; j < n_append; ++j)
        if ((rc = check_object(append[j], n_surv + j, n_tex, who)) != RT_OK) return rc;
    if ((rc = require_device(scene->device)) != RT_OK) return rc;

    // ---- the new counts, from the removed and appended objects alone
    auto *ds = static_cast<DeviceScene *>(scene->dev);
    HostSceneLayout &L = scene->layout;
    DeviceWorkspace *ws = ds->ws;
    cudaStream_t st = ws->stream;
    const int32_t nb_old = ds->g.n_bounded, nu_old = ds->g.n_unbounded;
    int32_t nb = nb_old, nu = nu_old;
    for (int32_t i = 0; i < n_remove; ++i) {
        const int32_t c = class_of(scene->objects[size_t(remove[i])]);
        nb -= c == OBJ_BOUNDED;
        nu -= c == OBJ_UNBOUNDED;
    }
    for (int32_t j = 0; j < n_append; ++j) {
        const int32_t c = class_of(append[j]);
        nb += c == OBJ_BOUNDED;
        nu += c == OBJ_UNBOUNDED;
    }
    const int32_t nn = nb >= 2 ? nb - 1 : nb; // one node holds a single sphere
    const BlobLayout old_blob = blob_layout(size_t(ds->g.n_nodes), size_t(nb_old), size_t(nu_old), size_t(n_tex));
    const BlobLayout B = blob_layout(size_t(nn), size_t(nb), size_t(nu), size_t(n_tex));

    // ---- the staged records: initial counters | remove list | the appended objects' class, sphere, material, unbounded record
    Carve hs{nullptr};
    hs.take<BuildCounters>(1);
    hs.take<int32_t>(size_t(n_remove));
    hs.take<int32_t>(size_t(n_append));
    hs.take<float4>(size_t(n_append));
    hs.take<DMaterial>(size_t(n_append));
    hs.take<DUnbounded>(size_t(n_append));
    const size_t stage_bytes = hs.at;

    // ---- scratch: the stage, then the builder's arrays
    const size_t n_old_blocks = std::max<size_t>(1, blocks_for(size_t(n_old), kScanThreads)), n_blocks = std::max<size_t>(1, blocks_for(size_t(n), kScanThreads)),
                 nb_blocks = std::max<size_t>(1, blocks_for(size_t(nb), kScanThreads));
    size_t sort_bytes = 0;
    RT_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, sort_bytes, static_cast<unsigned long long *>(nullptr), static_cast<unsigned long long *>(nullptr),
                                           std::max(n, 1), 0, 62, st));
    struct Scratch {
        uint8_t *stage;
        uint8_t *removed;
        unsigned long long *kscan, *ktop, *cscan, *ctop, *fscan, *ftop, *keys, *sorted;
        void *sort_tmp;
        int32_t *cls, *nn;
        float4 *sph;
        DMaterial *mat;
        DUnbounded *unb;
        Cluster *ca, *cb;
        BuildNode *bn;
        int4 *state;
        DTexture *tex;
    };
    auto lay = [&](uint8_t *base, Scratch &s) {
        Carve c{base};
        s.stage = c.take<uint8_t>(stage_bytes);
        s.removed = c.take<uint8_t>(size_t(n_old));
        s.kscan = c.take<unsigned long long>(size_t(n_old));
        s.ktop = c.take<unsigned long long>(n_old_blocks);
        s.cls = c.take<int32_t>(size_t(n));
        s.sph = c.take<float4>(size_t(n));
        s.mat = c.take<DMaterial>(size_t(n));
        s.unb = c.take<DUnbounded>(size_t(n));
        s.cscan = c.take<unsigned long long>(size_t(n));
        s.ctop = c.take<unsigned long long>(n_blocks);
        s.keys = c.take<unsigned long long>(size_t(n));
        s.sorted = c.take<unsigned long long>(size_t(n));
        s.sort_tmp = c.take<uint8_t>(sort_bytes);
        s.ca = c.take<Cluster>(size_t(nb));
        s.cb = c.take<Cluster>(size_t(nb));
        s.nn = c.take<int32_t>(size_t(nb));
        s.fscan = c.take<unsigned long long>(size_t(nb));
        s.ftop = c.take<unsigned long long>(nb_blocks);
        s.bn = c.take<BuildNode>(size_t(nb));
        s.state = c.take<int4>(size_t(nb));
        s.tex = c.take<DTexture>(size_t(n_tex));
        return c.at;
    };
    Scratch sc{};
    const size_t scratch_bytes = lay(nullptr, sc) + 256;
    size_t refit_bytes = 0, refit_zeroed = 0, old_refit_bytes = 0, unused = 0;
    refit_view(nullptr, size_t(nn), size_t(nb), &refit_bytes, &refit_zeroed);
    refit_view(nullptr, size_t(ds->g.n_nodes), size_t(nb_old), &old_refit_bytes, &unused);

    // ---- every allocation before any change: scratch, the id map, pinned staging, the new refit state, a bigger blob
    RT_CUDA(cudaSetDevice(ds->device));
    if (ds->build_scratch_cap < scratch_bytes) {
        cudaFree(ds->build_scratch);
        ds->build_scratch = nullptr;
        ds->build_scratch_cap = 0;
        RT_CUDA(cudaMalloc(&ds->build_scratch, scratch_bytes + scratch_bytes / 4));
        ds->build_scratch_cap = scratch_bytes + scratch_bytes / 4;
    }
    const size_t id_cap = size_t(std::max(n, n_old)) + 1;
    if (ds->dev_of_cap < id_cap) {
        int32_t *grown = nullptr;
        RT_CUDA(cudaMalloc(&grown, (id_cap + id_cap / 4) * sizeof(int32_t)));
        if (ds->dev_of_valid && cudaMemcpyAsync(grown, ds->dev_of, size_t(n_old) * sizeof(int32_t), cudaMemcpyDeviceToDevice, st) != cudaSuccess) {
            cudaFree(grown);
            return fail(RT_ERR_CUDA, "rt_scene_rebuild: copy of the id map failed");
        }
        RT_CUDA(cudaStreamSynchronize(st));
        cudaFree(ds->dev_of);
        ds->dev_of = grown;
        ds->dev_of_cap = id_cap + id_cap / 4;
    }
    if (ws->h_blob_cap < stage_bytes) {
        if (ws->h_blob) cudaFreeHost(ws->h_blob);
        ws->h_blob = nullptr;
        ws->h_blob_cap = 0;
        RT_CUDA(cudaMallocHost(&ws->h_blob, stage_bytes));
        ws->h_blob_cap = stage_bytes;
    }
    void *refit = nullptr;
    RT_CUDA(cudaMalloc(&refit, refit_bytes));
    void *blob = ws->d_blob; // rebuilt in place: the builder reads the old records into scratch before it writes the blob
    size_t blob_cap = ws->blob_cap;
    if (blob_cap < B.total) {
        blob_cap = std::max<size_t>(B.total + B.total / 2, 256 << 10);
        if (cudaMalloc(&blob, blob_cap) != cudaSuccess) {
            cudaFree(refit);
            return fail(RT_ERR_CUDA, "rt_scene_rebuild: cudaMalloc failed for the grown scene");
        }
    }

    // ---- stage: counters, remove list, the appended records (made with their new indices)
    uint8_t *host = static_cast<uint8_t *>(ws->h_blob);
    {
        Carve h{host};
        BuildCounters *cnt = h.take<BuildCounters>(1);
        std::memset(cnt, 0, sizeof *cnt);
        for (int a = 0; a < 3; ++a) {
            cnt->cmin[a] = 0x7fffffff;
            cnt->cmax[a] = int32_t(0x80000000u);
        }
        int32_t *rm = h.take<int32_t>(size_t(n_remove));
        if (n_remove) std::memcpy(rm, remove, size_t(n_remove) * sizeof(int32_t));
        int32_t *acls = h.take<int32_t>(size_t(n_append));
        float4 *asph = h.take<float4>(size_t(n_append));
        DMaterial *amat = h.take<DMaterial>(size_t(n_append));
        DUnbounded *aunb = h.take<DUnbounded>(size_t(n_append));
        for (int32_t j = 0; j < n_append; ++j) {
            const RtHittable &o = append[j];
            acls[j] = class_of(o);
            asph[j] = make_float4(float(o.p[0]), float(o.p[1]), float(o.p[2]), float(o.radius));
            amat[j] = make_material(o, n_surv + j);
            aunb[j] = acls[j] == OBJ_UNBOUNDED ? make_unbounded(o) : DUnbounded{};
        }
    }
    lay(static_cast<uint8_t *>(ds->build_scratch), sc);
    const uint8_t *sbase = sc.stage;
    Carve sv{const_cast<uint8_t *>(sbase)};
    BuildCounters *d_cnt = sv.take<BuildCounters>(1);
    int32_t *d_remove = sv.take<int32_t>(size_t(n_remove));
    int32_t *d_acls = sv.take<int32_t>(size_t(n_append));
    float4 *d_asph = sv.take<float4>(size_t(n_append));
    DMaterial *d_amat = sv.take<DMaterial>(size_t(n_append));
    DUnbounded *d_aunb = sv.take<DUnbounded>(size_t(n_append));
    if (!ds->dev_of_valid) // the scene's records came from the host (creation, or the host fallback): its id map
        RT_CUDA(cudaMemcpyAsync(ds->dev_of, L.device_id_of.data(), size_t(n_old) * sizeof(int32_t), cudaMemcpyHostToDevice, st));

    static const bool trace = std::getenv("RTFS_DEBUG_REBUILD") != nullptr;
    enum { S_BEGIN, S_COLLECT, S_SORT, S_CLUSTER, S_FLATTEN, S_END, S_COUNT };
    cudaEvent_t stage_ev[S_COUNT] = {};
    if (trace)
        for (auto &e : stage_ev) cudaEventCreate(&e);
    auto mark = [&](int which) {
        if (trace) cudaEventRecord(stage_ev[which], st);
    };
    int launches = 0;
    RT_CUDA(ws->ev.record(FrameEvents::BEGIN, st));
    mark(S_BEGIN);
    RT_CUDA(cudaMemcpyAsync(sc.stage, host, stage_bytes, cudaMemcpyHostToDevice, st));

    // ---- 1. collect the new array's records (reads the old blob), and the textures' records
    const uint8_t *old_base = static_cast<const uint8_t *>(ds->blob);
    if (n_old) RT_CUDA(cudaMemsetAsync(sc.removed, 0, size_t(n_old), st));
    if (n_remove) {
        rebuild_mark_kernel<<<blocks_for(size_t(n_remove), kBuildThreads), kBuildThreads, 0, st>>>(d_remove, n_remove, sc.removed);
        launches += 1;
    }
    launches += launch_scan(KeepFlag{sc.removed}, n_old, sc.kscan, sc.ktop, &d_cnt->total, st);
    if (n_old + n_append) {
        CollectArgs ca{n_old,     n_append, nb_old,  sc.removed, sc.kscan, sc.ktop, ds->dev_of, ds->g.spheres,
                       reinterpret_cast<const DMaterial *>(ds->g.mats), ds->g.unb, d_acls, d_asph, d_amat, d_aunb,
                       sc.cls,    sc.sph,   sc.mat,  sc.unb,     d_cnt};
        rebuild_collect_kernel<<<blocks_for(size_t(n_old + n_append), kBuildThreads), kBuildThreads, 0, st>>>(ca);
        launches += 1;
    }
    if (n_tex) RT_CUDA(cudaMemcpyAsync(sc.tex, old_base + old_blob.tex, size_t(n_tex) * sizeof(DTexture), cudaMemcpyDeviceToDevice, st));
    launches += launch_scan(ClassFlag{sc.cls}, n, sc.cscan, sc.ctop, &d_cnt->total, st);
    mark(S_COLLECT);

    // ---- 2. Morton keys and the sort
    if (n) {
        rebuild_keys_kernel<<<blocks_for(size_t(n), kBuildThreads), kBuildThreads, 0, st>>>(sc.cls, sc.sph, n, d_cnt, sc.keys);
        RT_CUDA(cub::DeviceRadixSort::SortKeys(sc.sort_tmp, sort_bytes, sc.keys, sc.sorted, n, 0, 62, st));
        launches += 2;
    }
    mark(S_SORT);

    // ---- 3. clustering: one iteration per round trip of the cluster count
    uint8_t *nb_base = static_cast<uint8_t *>(blob);
    const RefitView rv = refit_view(refit, size_t(nn), size_t(nb), &refit_bytes, &refit_zeroed);
    PlaceArgs pa{sc.sorted, sc.sph, sc.mat, rv, reinterpret_cast<uint4 *>(nb_base + B.nodes), reinterpret_cast<float4 *>(nb_base + B.spheres),
                 reinterpret_cast<DMaterial *>(nb_base + B.mats), ds->dev_of, d_cnt};
    std::vector<std::pair<int32_t, int32_t>> rounds; // the nodes each iteration made: (first, count)
    if (nb >= 2) {
        ploc_init_kernel<<<blocks_for(size_t(nb), kBuildThreads), kBuildThreads, 0, st>>>(sc.sorted, sc.sph, nb, sc.ca);
        launches += 1;
        int32_t m = nb, made = 0;
        Cluster *in = sc.ca, *out = sc.cb;
        while (m > 1) {
            const unsigned blocks = blocks_for(size_t(m), kBuildThreads);
            ploc_nearest_kernel<<<blocks, kBuildThreads, 0, st>>>(in, m, sc.nn);
            launches += 1 + launch_scan(ClusterFlag{sc.nn}, m, sc.fscan, sc.ftop, &d_cnt->total, st);
            ploc_merge_kernel<<<blocks, kBuildThreads, 0, st>>>(in, m, sc.nn, sc.fscan, sc.ftop, made, out, sc.bn);
            launches += 1;
            unsigned long long total = 0;
            RT_CUDA(cudaMemcpyAsync(&total, &d_cnt->total, sizeof total, cudaMemcpyDeviceToHost, st));
            RT_CUDA(cudaStreamSynchronize(st));
            const int32_t kept = int32_t(total & 0xffffffffu), merged = int32_t(total >> 32);
            if (merged <= 0 || kept != m - merged) { // cannot happen (a mutual pair always exists); never loop on it
                cudaFree(refit);
                if (blob != ws->d_blob) cudaFree(blob);
                return fail(RT_ERR_DEGENERATE, "rt_scene_rebuild: a clustering iteration made no progress");
            }
            rounds.emplace_back(made, merged);
            made += merged;
            m = kept;
            std::swap(in, out);
        }
    }
    mark(S_CLUSTER);

    // ---- 4. flatten top-down into the blob and the refit state; then the unbounded objects and the textures
    if (nn) RT_CUDA(cudaMemsetAsync(static_cast<uint8_t *>(refit) + refit_zeroed, 0, refit_bytes - refit_zeroed, st));
    if (nb >= 2) {
        const int4 root = make_int4(0, 0, 1, 0);
        const int32_t root_id = nb - 2;
        const int32_t minus_one = -1;
        RT_CUDA(cudaMemcpyAsync(sc.state + root_id, &root, sizeof root, cudaMemcpyHostToDevice, st));
        RT_CUDA(cudaMemcpyAsync(rv.node_parent, &minus_one, sizeof minus_one, cudaMemcpyHostToDevice, st));
        for (size_t k = rounds.size(); k-- > 0;) {
            ploc_flatten_kernel<<<blocks_for(size_t(rounds[k].second), kBuildThreads), kBuildThreads, 0, st>>>(sc.bn, sc.state, rounds[k].first,
                                                                                                             rounds[k].second, pa);
            launches += 1;
        }
    } else if (nb == 1) {
        ploc_single_kernel<<<1, 1, 0, st>>>(pa);
        launches += 1;
    }
    if (n) {
        rebuild_place_unbounded_kernel<<<blocks_for(size_t(n), kBuildThreads), kBuildThreads, 0, st>>>(
            sc.cls, sc.cscan, sc.ctop, n, nb, sc.mat, sc.unb, reinterpret_cast<DMaterial *>(nb_base + B.mats),
            reinterpret_cast<DUnbounded *>(nb_base + B.unb), ds->dev_of);
        launches += 1;
    }
    if (n_tex) RT_CUDA(cudaMemcpyAsync(nb_base + B.tex, sc.tex, size_t(n_tex) * sizeof(DTexture), cudaMemcpyDeviceToDevice, st));
    RT_CUDA(cudaGetLastError());
    BuildCounters got{};
    RT_CUDA(cudaMemcpyAsync(&got, d_cnt, sizeof got, cudaMemcpyDeviceToHost, st));
    mark(S_FLATTEN);
    RT_CUDA(ws->ev.record(FrameEvents::END, st));
    mark(S_END);
    RT_CUDA(cudaStreamSynchronize(st));
    const double device_ms = ws->ev.ms(FrameEvents::BEGIN, FrameEvents::END);
    if (trace) {
        float t[S_COUNT] = {};
        for (int k = 1; k < S_COUNT; ++k) cudaEventElapsedTime(&t[k], stage_ev[k - 1], stage_ev[k]);
        std::fprintf(stderr, "rtfs: rebuild n=%d bounded=%d rounds=%zu collect_ms=%.4f sort_ms=%.4f cluster_ms=%.4f flatten_ms=%.4f device_ms=%.4f\n", n, nb,
                     rounds.size(), t[S_COLLECT], t[S_SORT], t[S_CLUSTER], t[S_FLATTEN], device_ms);
        for (auto &e : stage_ev) cudaEventDestroy(e);
    }

    // ---- the scene's state: host copy of the array, the blob's sections, the counts, the refit state, the derived trees
    if (blob != ws->d_blob) {
        cudaFree(ws->d_blob);
        ws->d_blob = blob;
        ws->blob_cap = blob_cap;
    }
    ds->blob = blob;
    ds->bytes += B.total - old_blob.total;
    if (ds->refit) {
        cudaFree(ds->refit);
        ds->bytes -= old_refit_bytes;
    }
    ds->refit = refit;
    ds->bytes += refit_bytes;
    {
        std::vector<uint8_t> gone(size_t(n_old), 0);
        for (int32_t i = 0; i < n_remove; ++i) gone[size_t(remove[i])] = 1;
        size_t w = 0;
        for (size_t i = 0; i < size_t(n_old); ++i)
            if (!gone[i]) scene->objects[w++] = scene->objects[i];
        scene->objects.resize(w);
        scene->objects.insert(scene->objects.end(), append, append + n_append);
    }
    ds->g.nodes = reinterpret_cast<const uint4 *>(nb_base + B.nodes);
    ds->g.spheres = reinterpret_cast<const float4 *>(nb_base + B.spheres);
    ds->g.mats = reinterpret_cast<const uint4 *>(nb_base + B.mats);
    ds->g.unb = reinterpret_cast<const DUnbounded *>(nb_base + B.unb);
    ds->g.tex = reinterpret_cast<const DTexture *>(nb_base + B.tex);
    ds->g.n_nodes = nn;
    ds->g.n_bounded = nb;
    ds->g.n_unbounded = nu;
    ds->n_fp64 = int32_t(got.n_fp64);
    ds->n_textured = int32_t(got.n_textured);
    ds->lean = ds->n_fp64 == 0 && ds->n_textured == 0;
    ds->dev_of_valid = true;
    invalidate_wide(scene, ds);
    invalidate_reference(scene, ds);
    scene->sah_built = false;
    L.n_bounded = nb;
    L.root_is_leaf = nb == 1 ? 1 : 0;
    L.max_depth = int32_t(got.depth);
    L.nodes.resize(size_t(nn));
    scene->layout_stale = nn > 0; // layout.nodes from the refit state, the records from the blob: on a host consumer's demand
    scene->records_stale = true;
    if (nn == 0) scene->device_nodes.clear();
    int32_t on_device = 1;
    if (L.max_depth > kMaxTreeDepth) { // deeper than the walk stacks: the host SAH tree of the same array, as rt_scene_create builds it
        on_device = 0;
        std::vector<HostNode> unused_tree;
        build_device_layout(scene->objects.data(), n, L, unused_tree);
        scene->layout_stale = scene->records_stale = false;
        scene->device_nodes.clear();
        cudaFree(ds->refit); // rt_scene_update uploads the refit state of this tree when it first needs it
        ds->refit = nullptr;
        ds->bytes -= refit_bytes;
        ds->dev_of_valid = false;
        const size_t head = B.unb; // nodes | spheres | materials (the unbounded part is the same in both trees)
        if (ws->h_blob_cap < head) {
            if (ws->h_blob) cudaFreeHost(ws->h_blob);
            ws->h_blob = nullptr;
            ws->h_blob_cap = 0;
            RT_CUDA(cudaMallocHost(&ws->h_blob, head));
            ws->h_blob_cap = head;
        }
        uint8_t *hb = static_cast<uint8_t *>(ws->h_blob);
        std::memset(hb, 0, head);
        DNode *dn = reinterpret_cast<DNode *>(hb + B.nodes);
        for (size_t i = 0; i < L.nodes.size(); ++i) dn[i] = device_node_of(L.nodes[i]);
        std::memcpy(hb + B.spheres, L.spheres.data(), L.spheres.size() * sizeof(DSphere));
        std::memcpy(hb + B.mats, L.materials.data(), L.materials.size() * sizeof(DMaterial));
        RT_CUDA(cudaMemcpyAsync(nb_base, hb, head, cudaMemcpyHostToDevice, st));
        RT_CUDA(cudaStreamSynchronize(st));
    }
    ds->max_depth = L.max_depth;
    scene->generation += 1;
    if (info) {
        RtSceneRebuild out{};
        out.objects_removed = n_remove;
        out.objects_appended = n_append;
        out.n_objects = n;
        out.n_bounded = nb;
        out.nodes = nn;
        out.depth = L.max_depth;
        out.on_device = on_device;
        out.launches = launches;
        out.generation = scene->generation;
        out.device_ms = device_ms;
        *info = out;
    }
    return RT_OK;
}

} // extern "C"
