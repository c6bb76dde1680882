// rtfs_internal.h — types shared by the host (rtfs_host.cpp) and device (rtfs_device.cu) halves of
// librtfs_b200.so.  Not part of the public ABI.
#pragma once
#include "../../include/rtfs_b200.h"

#include <cmath>
#include <cstddef>
#include <cstdint>
#include <limits>
#include <string>
#include <vector>

// functions compiled for the host and, in the CUDA translation units, for the device too (one piece of code for both)
#ifdef __CUDACC__
#define RTFS_HOST_DEVICE __host__ __device__ inline
#else
#define RTFS_HOST_DEVICE inline
#endif

namespace rtfs {

// ---- error plumbing ---------------------------------------------------------------------------
void set_error(const std::string &msg);
int fail(int code, const std::string &msg);

// ---- host BVH ---------------------------------------------------------------------------------
// Flattened tree in DFS pre-order (left child = i + 1), the format rt_scene_bvh_nodes exposes.
struct HostNode {
    double mn[3], mx[3];
    int32_t right; // -1: leaf
    int32_t prim;  // leaf: index into the caller's Hittable array
};

// BoundingBoxTree.make (RayTracing/BoundingBoxTree.fs:9-43): median split on box.Min[axis], axis by
// minimum volume(L)+volume(R); leaves hold one object.  `prims` are indices of bounded objects in
// array order (Scene.fs:16-22).
void build_reference_tree(const RtHittable *objs, const std::vector<int32_t> &prims, std::vector<HostNode> &out);

// ---- device-side scene layout (what rtfs_device.cu uploads) --------------------------------------
// Bounded spheres, in SAH leaf order.  16 B each, one 128-bit load.
struct DSphere {
    float cx, cy, cz, r;
};
// BVH2 node with both children's boxes inline: 64 B = four 128-bit loads.
//   q0 = {l.min.x, l.min.y, l.min.z, l.max.x}
//   q1 = {l.max.y, l.max.z, r.min.x, r.min.y}
//   q2 = {r.min.z, r.max.x, r.max.y, r.max.z}
//   q3 = {left, right, -, -} as int bits: >= 0 internal node index, < 0 leaf holding sphere ~idx
struct DNode {
    float l_mn[3], l_mx[3];
    float r_mn[3], r_mx[3];
    int32_t left, right;
    int32_t pad0, pad1;
};
static_assert(sizeof(DNode) == 64, "DNode must be 64 bytes");
// What the DEVICE holds per node: the same two boxes as centre c and half-extent h >= 0, left and right child side by side
// (same 64 bytes):
//   q0 = {c.x l, c.x r, c.y l, c.y r}   q1 = {c.z l, c.z r, h.x l, h.x r}   q2 = {h.y l, h.y r, h.z l, h.z r}   q3 as above
// For a ray with reciprocal direction inv and noi = -o * inv the slab distances of an axis are  t_c -+ h |inv|  with
// t_c = c * inv + noi: near and far come out ordered, so no min / max pair per axis (ALU pipe) is needed, and because the two
// children's values sit in adjacent, even-aligned registers after a 128-bit load, each step is ONE packed FFMA2
// (fma.rn.f32x2, sm_100) for both boxes with the ray's constant as a broadcast operand: ten FMA-pipe instructions per visit
// (slab_pair, rtfs_core.cuh).  device_node_of() converts, rounding the half-extent upwards so that the box never shrinks.

// the FP32 value nearest v towards -inf / +inf (the directed roundings of the leaf boxes and half-extents)
RTFS_HOST_DEVICE float round_down(double v) {
#ifdef __CUDA_ARCH__
    return __double2float_rd(v);
#else
    float f = float(v);
    if (double(f) > v) f = std::nextafterf(f, -std::numeric_limits<float>::infinity());
    return f;
#endif
}
RTFS_HOST_DEVICE float round_up(double v) {
#ifdef __CUDA_ARCH__
    return __double2float_ru(v);
#else
    float f = float(v);
    if (double(f) < v) f = std::nextafterf(f, std::numeric_limits<float>::infinity());
    return f;
#endif
}

// min / max boxes -> centre / half-extent boxes in the paired layout above, never smaller than the original.  The host
// upload and the device refit (rtfs_edit.cu) both convert with this function, so the two give the same bytes.
RTFS_HOST_DEVICE DNode device_node_of(const DNode &n) {
    DNode d = n;
    float c[2][3], h[2][3];
    for (int side = 0; side < 2; ++side) {
        const float *mn = side ? n.r_mn : n.l_mn, *mx = side ? n.r_mx : n.l_mx;
        for (int a = 0; a < 3; ++a) {
#ifdef __CUDA_ARCH__
            const bool finite = isfinite(mn[a]) && isfinite(mx[a]);
#else
            const bool finite = std::isfinite(mn[a]) && std::isfinite(mx[a]);
#endif
            if (!finite) { // the never-entered dummy box of a one-sphere tree
                c[side][a] = 1e30f;
                h[side][a] = 0.f;
                continue;
            }
            const float cf = float(0.5 * (double(mn[a]) + double(mx[a])));
            const double lo = double(cf) - double(mn[a]), hi = double(mx[a]) - double(cf);
            const float hf = round_up(hi < lo ? lo : hi);
            c[side][a] = cf;
#ifdef __CUDA_ARCH__
            h[side][a] = nextafterf(hf, __int_as_float(0x7f800000));
#else
            h[side][a] = std::nextafterf(hf, std::numeric_limits<float>::infinity());
#endif
        }
    }
    // {c.x l, c.x r, c.y l, c.y r | c.z l, c.z r, h.x l, h.x r | h.y l, h.y r, h.z l, h.z r}: the twelve floats of the struct in order
    float *q = d.l_mn;
    static_assert(offsetof(DNode, left) == 12 * sizeof(float), "the twelve box floats are contiguous");
    for (int a = 0; a < 3; ++a)
        for (int side = 0; side < 2; ++side) {
            q[2 * a + side] = c[side][a];
            q[6 + 2 * a + side] = h[side][a];
        }
    return d;
}

// Per-primitive material record, 32 B = two 128-bit loads.  Index = device primitive id.
struct DMaterial {
    double albedo;      // FP64 so that Pixel.darken's round-half-even is bit-exact (Pixel.fs:144-151)
    float p0;           // fuzz (FUZZED) | ior (DIELECTRIC, GLASS) | cap threshold cx + 0.75 r (LIGHT_SOURCE_CAP)
    float p1;           // prob (DIELECTRIC)
    uint32_t style_rgb; // style << 24 | r << 16 | g << 8 | b
    int32_t texture;    // index into textures, -1: constant colour
    uint32_t flags;     // bit0: flipped (radius < 0, Sphere.fs:321); bit1: plane
    int32_t host_index; // index into the caller's Hittable array
};
static_assert(sizeof(DMaterial) == 32, "DMaterial must be 32 bytes");
// the material record of object host_index
DMaterial make_material(const RtHittable &h, int32_t host_index);

// Unbounded objects (UnboundedSphere, InfinitePlane), tested linearly after the tree (Scene.fs:77-86).
// These spheres are typically huge (r = 1000, 2000), and |o - c|^2 - r^2 evaluated from o - c cancels catastrophically
// in FP32.  Two evaluations (classify_unbounded picks per object, on the host):
//   fp32 = 1  the EXPANDED forms  |o|^2 - 2 o.c + k  (k = |c|^2 - r^2)  and  k - n.o  (k = n.p0), k computed in FP64
//             and rounded once: every term is then of the size of the scene, not of the sphere, and FP32 keeps
//             ~1e-7 relative accuracy on the result.  Used when the centre is exactly representable in FP32 and k is
//             small enough next to the scene (see classify_unbounded) — the floor, the sky dome, planes near the origin;
//   fp32 = 0  the FP64 evaluation of exactly the cancelling terms (any other object).
struct DUnbounded {
    double p[3];   // centre / point on plane
    double r2;     // radius^2 (sphere)
    float n[3];    // plane: normal; sphere with fp32 = 1: the centre as floats (exactly p)
    float r;       // signed radius (sphere)
    int32_t shape; // RT_SHAPE_UNBOUNDED_SPHERE | RT_SHAPE_INFINITE_PLANE
    int32_t fp32;
    float k;       // sphere: |c|^2 - r^2; plane: n . p0
    int32_t pad;
};
// fills fp32 / k (and n for spheres) of an object whose p, r, r2, n, shape are set
void classify_unbounded(DUnbounded &u);
// the device record of an unbounded object (UnboundedSphere, InfinitePlane), classified
DUnbounded make_unbounded(const RtHittable &h);
static_assert(sizeof(DUnbounded) == 64, "DUnbounded must be 64 bytes");

struct DTexture {
    int32_t kind;
    uint32_t rgb; // r << 16 | g << 8 | b
    int32_t w, h;
    unsigned long long tex; // cudaTextureObject_t (uchar4, point sampling, unnormalised coords)
    int32_t even, odd;
    float grid;
    float cx, cy, cz, inv_radius;
    int32_t pad[3];
};
static_assert(sizeof(DTexture) == 64, "DTexture must be 64 bytes");

// Reference-topology tree for the exhaustive-DFS conformance traversal (F12).
struct DRefNode {
    float mn[3], mx[3];
    int32_t right; // -1 leaf
    int32_t prim;  // leaf: device primitive id, -1 if the object is not representable (never)
};
static_assert(sizeof(DRefNode) == 32, "DRefNode must be 32 bytes");

// 8-wide compressed BVH node (after Ylitie, Karras, Laine, "Efficient Incoherent Ray Traversal on GPUs Through
// Compressed Wide BVHs", HPG 2017): 80 B = five 128-bit loads.  The eight child boxes are quantised to 8 bits per
// plane on a per-node grid: coordinate q stands for p + q * 2^e (rounded outwards at build time).
//   q0 = {p.x, p.y, p.z, ex' | ey' << 8 | ez' << 16 | imask << 24}   e' = e + 127 + 15: the bits of the float 2^(e+15) >> 23
//   q1 = {child_base, prim_base, meta[0..3], meta[4..7]}
//   q2 = {qlo.x[0..3], qlo.x[4..7], qlo.y[0..3], qlo.y[4..7]}
//   q3 = {qlo.z[0..3], qlo.z[4..7], qhi.x[0..3], qhi.x[4..7]}
//   q4 = {qhi.y[0..3], qhi.y[4..7], qhi.z[0..3], qhi.z[4..7]}
// Children sit in slots 0..7; slot s is the child lying towards the octant with signs (x: bit 2, y: bit 1, z: bit 0), so
// that `slot XOR octant-of-the-ray` orders the children roughly front to back without computing distances.
// imask: which slots hold internal nodes; those are stored consecutively from child_base in slot order.
// meta[s]: 0 = empty; internal node: 0b001 << 5 | (24 + s); leaf: (unary count of spheres) << 5 | offset from prim_base.
struct DWideNode {
    float p[3];
    uint8_t e[3];
    uint8_t imask;
    uint32_t child_base, prim_base;
    uint8_t meta[8];
    uint8_t qlo_x[8], qlo_y[8], qlo_z[8], qhi_x[8], qhi_y[8], qhi_z[8];
};
static_assert(sizeof(DWideNode) == 80, "DWideNode must be 80 bytes");

struct HostSceneLayout {
    // device primitive ids: [0, n_bounded) bounded spheres in SAH leaf order, then unbounded in array order
    std::vector<DSphere> spheres;
    std::vector<DNode> nodes;
    std::vector<DMaterial> materials; // n_bounded + n_unbounded
    std::vector<DUnbounded> unbounded;
    std::vector<DRefNode> ref_nodes;
    std::vector<int32_t> device_id_of; // caller's Hittable index -> device primitive id (-1: never hit, F16)
    int32_t n_bounded = 0;
    int32_t root_is_leaf = 0;
    int32_t max_depth = 0;
    // the 8-wide compressed tree over the same spheres (build_wide_layout): its own sphere order (the spheres of a node
    // are consecutive), mapped to and from device primitive ids
    std::vector<DWideNode> wide_nodes;
    std::vector<DSphere> wide_spheres;
    std::vector<int32_t> wide_to_dev, dev_to_wide;
    int32_t wide_depth = 0;
};

// SAH BVH2 over the bounded spheres with radius >= 0 (a bounded sphere with negative radius has an
// inverted box and is never hit in the reference, F16).  Fills layout.spheres/nodes and the bounded
// part of layout.materials; also exports the tree in HostNode form for inspection.
void build_device_layout(const RtHittable *objs, int32_t n_objs, HostSceneLayout &layout, std::vector<HostNode> &sah_tree_out);
// The checks rt_scene_create makes of one object and of the texture table; `who` names the caller in the message.
int check_object(const RtHittable &h, int32_t i, int32_t n_textures, const char *who);
int check_textures(const RtTexture *textures, int32_t n_textures, const char *who);
// Collapses the SAH BVH2 of `layout` into the 8-wide compressed tree (fills layout.wide_*).  Idempotent.
void build_wide_layout(HostSceneLayout &layout);
// (built on first use: a render with RT_FLAG_WIDE_BVH, rt_test_hit_object(traversal = 2), rt_scene_wide_bvh_check)

} // namespace rtfs

// The opaque scene handle.
struct RtScene {
    std::vector<RtHittable> objects;
    std::vector<RtTexture> textures;
    std::vector<std::vector<uint8_t>> texture_pixels;
    std::vector<rtfs::HostNode> ref_tree, sah_tree;
    bool ref_built = false; // the reference-topology tree is built on first use (scene_ensure_reference)
    bool sah_built = false; // likewise the inspection form of the SAH tree (scene_ensure_sah_tree)
    rtfs::HostSceneLayout layout;
    int32_t device = -1;
    void *dev = nullptr; // rtfs_device.cu: DeviceScene*
    // rt_scene_update (rtfs_edit.cu): the edit count, which progressive frames record when they open; after a refit the
    // tree's boxes live on the device and layout.nodes is stale until device_scene_sync_layout downloads them, together with
    // the node records the device walks (device_nodes, which rt_scene_device_bvh_check holds to device_node_of)
    uint64_t generation = 0;
    bool layout_stale = false;
    std::vector<rtfs::DNode> device_nodes;
    // rt_scene_rebuild (rtfs_build.cu) builds the tree on the device and places the records there: layout.spheres,
    // materials, unbounded and device_id_of are stale until device_scene_sync_layout downloads them
    bool records_stale = false;
};

// implemented in rtfs_device.cu
namespace rtfs {
void scene_ensure_reference(RtScene *scene);
void scene_ensure_sah_tree(RtScene *scene);
int device_scene_upload(RtScene *scene);
int device_scene_ensure_reference(RtScene *scene);
int device_scene_ensure_wide(RtScene *scene);
// brings layout.nodes (and scene->device_nodes) up to date after rt_scene_update refit the tree, and the records of the
// layout after rt_scene_rebuild placed them on the device (rtfs_edit.cu)
int device_scene_sync_layout(RtScene *scene);
void device_scene_free(RtScene *scene);
size_t device_scene_bytes(const RtScene *scene);
} // namespace rtfs
