// rtfs_host.cpp — host half of librtfs_b200.so: error plumbing, Camera.makeBasic, the P3 writer,
// the two BVH builders and the scene handle.  Nothing in this file needs a GPU.
#include "rtfs_internal.h"

#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <limits>
#include <numeric>

namespace rtfs {

static thread_local std::string g_last_error;
void set_error(const std::string &msg) { g_last_error = msg; }
int fail(int code, const std::string &msg) {
    g_last_error = msg;
    return code;
}

namespace {

struct D3 {
    double x, y, z;
};
inline D3 operator+(D3 a, D3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
inline D3 operator-(D3 a, D3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
inline D3 operator*(double s, D3 a) { return {s * a.x, s * a.y, s * a.z}; }
inline double dot(D3 a, D3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
inline D3 cross(D3 a, D3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - b.x * a.y}; }
inline D3 load(const double *p) { return {p[0], p[1], p[2]}; }
inline void store(double *p, D3 v) {
    p[0] = v.x;
    p[1] = v.y;
    p[2] = v.z;
}
constexpr double kTol = 1e-8; // Float.tolerance, RayTracing/Float.fs:80
// Vector.unitise (Point.fs:28-35): fails when |v.v| < 1e-8, multiplies by the reciprocal root.
inline bool unitise(D3 v, D3 &out) {
    double d = dot(v, v);
    if (std::fabs(d) < kTol) return false;
    out = (1.0 / std::sqrt(d)) * v;
    return true;
}

} // namespace

// ---------------------------------------------------------------------------------------------
// BoundingBoxTree.make, RayTracing/BoundingBoxTree.fs:9-43
// ---------------------------------------------------------------------------------------------
namespace {
struct RefBox {
    double mn[3], mx[3];
};
inline RefBox sphere_box(const RtHittable &h) { // Sphere.make, Sphere.fs:333-336 (inverted when radius < 0)
    RefBox b;
    for (int a = 0; a < 3; ++a) {
        b.mn[a] = h.p[a] + (-h.radius);
        b.mx[a] = h.p[a] + h.radius;
    }
    return b;
}
inline RefBox merge(const RefBox &i, const RefBox &j) { // BoundingBox.mergeTwo, BoundingBox.fs:96-108
    RefBox o;
    for (int a = 0; a < 3; ++a) {
        o.mn[a] = std::min(i.mn[a], j.mn[a]);
        o.mx[a] = std::max(i.mx[a], j.mx[a]);
    }
    return o;
}
inline double volume(const RefBox &b) { return (b.mx[0] - b.mn[0]) * (b.mx[1] - b.mn[1]) * (b.mx[2] - b.mn[2]); }
inline RefBox merge_all(const RtHittable *objs, const std::vector<int32_t> &v) {
    RefBox b = sphere_box(objs[v[0]]);
    for (size_t i = 1; i < v.size(); ++i) b = merge(b, sphere_box(objs[v[i]]));
    return b;
}

int32_t ref_go(const RtHittable *objs, const std::vector<int32_t> &boxes, std::vector<HostNode> &out) {
    int32_t me = int32_t(out.size());
    out.push_back(HostNode{});
    RefBox all = merge_all(objs, boxes);
    auto put_box = [&](const RefBox &b) {
        for (int a = 0; a < 3; ++a) {
            out[me].mn[a] = b.mn[a];
            out[me].mx[a] = b.mx[a];
        }
    };
    put_box(all);
    out[me].right = -1;
    out[me].prim = -1;
    if (boxes.size() == 1) {
        out[me].prim = boxes[0];
        return me;
    }
    if (boxes.size() == 2) {
        ref_go(objs, {boxes[0]}, out);
        int32_t r = ref_go(objs, {boxes[1]}, out);
        out[me].right = r;
        return me;
    }
    std::vector<int32_t> best_left, best_right;
    double best_cost = 0.0;
    for (int axis = 0; axis < 3; ++axis) {
        std::vector<int32_t> sorted = boxes;
        // Array.sortBy is unstable in .NET; a stable sort is one of its admissible outcomes.
        std::stable_sort(sorted.begin(), sorted.end(), [&](int32_t a, int32_t b) {
            return (objs[a].p[axis] + (-objs[a].radius)) < (objs[b].p[axis] + (-objs[b].radius));
        });
        size_t half = sorted.size() / 2;
        std::vector<int32_t> left(sorted.begin(), sorted.begin() + half + 1); // boxes.[0 .. n/2] is inclusive
        std::vector<int32_t> right(sorted.begin() + half + 1, sorted.end());
        double cost = volume(merge_all(objs, left)) + volume(merge_all(objs, right));
        if (axis == 0 || cost < best_cost) { // Array.minBy keeps the first minimum
            best_cost = cost;
            best_left.swap(left);
            best_right.swap(right);
        }
    }
    ref_go(objs, best_left, out);
    int32_t r = ref_go(objs, best_right, out);
    out[me].right = r;
    return me;
}
} // namespace

void build_reference_tree(const RtHittable *objs, const std::vector<int32_t> &prims, std::vector<HostNode> &out) {
    out.clear();
    if (prims.empty()) return;
    ref_go(objs, prims, out);
}

// ---------------------------------------------------------------------------------------------
// SAH BVH2 for the render kernels
// ---------------------------------------------------------------------------------------------
namespace {
struct BuildPrim {
    float mn[3], mx[3];
    float c[3];
    int32_t obj;
};
struct FBox {
    float mn[3], mx[3];
    void reset() {
        for (int a = 0; a < 3; ++a) {
            mn[a] = std::numeric_limits<float>::infinity();
            mx[a] = -std::numeric_limits<float>::infinity();
        }
    }
    void grow(const float *pmn, const float *pmx) {
        for (int a = 0; a < 3; ++a) {
            mn[a] = std::min(mn[a], pmn[a]);
            mx[a] = std::max(mx[a], pmx[a]);
        }
    }
    double area() const {
        double dx = double(mx[0]) - mn[0], dy = double(mx[1]) - mn[1], dz = double(mx[2]) - mn[2];
        if (dx < 0 || dy < 0 || dz < 0) return 0.0;
        return 2.0 * (dx * dy + dy * dz + dz * dx);
    }
};

struct SahBuilder {
    std::vector<BuildPrim> prims;
    const RtHittable *objs;
    HostSceneLayout *layout;
    int max_depth = 0;

    FBox bounds(int lo, int hi) const {
        FBox b;
        b.reset();
        for (int i = lo; i < hi; ++i) b.grow(prims[i].mn, prims[i].mx);
        return b;
    }
    int32_t emit_leaf(int i) {
        const RtHittable &h = objs[prims[i].obj];
        int32_t idx = int32_t(layout->spheres.size());
        layout->spheres.push_back(DSphere{float(h.p[0]), float(h.p[1]), float(h.p[2]), float(h.radius)});
        leaf_obj.push_back(prims[i].obj);
        return ~idx;
    }
    std::vector<int32_t> leaf_obj;

    int split(int lo, int hi, int depth) {
        int n = hi - lo;
        int mid = -1;
        FBox cb;
        cb.reset();
        for (int i = lo; i < hi; ++i) cb.grow(prims[i].c, prims[i].c);
        constexpr int kSmall = 12;
        if (n > 2 && n <= kSmall && depth < 40) {
            // Small ranges (most nodes of the tree): the same binned SAH evaluated over the primitives themselves.  A split
            // "after bin k" only matters at the bins that hold something, and the boxes of "bins <= k" are unions of
            // primitive boxes whichever way they are accumulated, so sorting the few primitives by bin index and sweeping
            // them gives the costs, the minimum and the first-minimum tie-break of the 16-bin sweep below exactly —
            // without resetting and walking 3 x 16 mostly empty bins per node.
            constexpr int BINS = 16;
            double best = std::numeric_limits<double>::infinity();
            int best_axis = -1, best_bin = -1;
            for (int axis = 0; axis < 3; ++axis) {
                float ext = cb.mx[axis] - cb.mn[axis];
                if (!(ext > 0.f)) continue;
                const float scale = float(BINS) / ext;
                int key[kSmall], idx[kSmall];
                for (int i = 0; i < n; ++i) { // insertion sort by bin index (stable: equal bins keep their order, which does not matter)
                    int k = std::min(BINS - 1, std::max(0, int((prims[lo + i].c[axis] - cb.mn[axis]) * scale)));
                    int j = i;
                    while (j > 0 && key[j - 1] > k) {
                        key[j] = key[j - 1];
                        idx[j] = idx[j - 1];
                        --j;
                    }
                    key[j] = k;
                    idx[j] = lo + i;
                }
                double right_area[kSmall + 1];
                FBox acc;
                acc.reset();
                right_area[n] = 0.0;
                for (int j = n - 1; j > 0; --j) {
                    acc.grow(prims[idx[j]].mn, prims[idx[j]].mx);
                    right_area[j] = acc.area();
                }
                acc.reset();
                for (int j = 0; j < n - 1; ++j) { // split after sorted position j, allowed where the bin index changes
                    acc.grow(prims[idx[j]].mn, prims[idx[j]].mx);
                    if (key[j] == key[j + 1] || key[j] >= BINS - 1) continue;
                    double cost = acc.area() * (j + 1) + right_area[j + 1] * (n - 1 - j);
                    if (cost < best) {
                        best = cost;
                        best_axis = axis;
                        best_bin = key[j];
                    }
                }
            }
            if (best_axis >= 0) {
                const float ext = cb.mx[best_axis] - cb.mn[best_axis];
                const float sc = float(BINS) / ext, c0 = cb.mn[best_axis];
                auto it = std::partition(prims.begin() + lo, prims.begin() + hi, [&](const BuildPrim &p) {
                    int k = std::min(BINS - 1, std::max(0, int((p.c[best_axis] - c0) * sc)));
                    return k <= best_bin;
                });
                mid = int(it - prims.begin());
            }
        } else if (n > 2 && depth < 40) {
            constexpr int BINS = 16;
            // one pass over the primitives fills the bins of all three axes
            FBox bb[3][BINS];
            int cnt[3][BINS];
            float scale[3];
            bool live[3];
            for (int axis = 0; axis < 3; ++axis) {
                float ext = cb.mx[axis] - cb.mn[axis];
                live[axis] = ext > 0.f;
                scale[axis] = live[axis] ? float(BINS) / ext : 0.f;
                for (int k = 0; k < BINS; ++k) {
                    bb[axis][k].reset();
                    cnt[axis][k] = 0;
                }
            }
            for (int i = lo; i < hi; ++i) {
                const BuildPrim &p = prims[i];
                for (int axis = 0; axis < 3; ++axis) {
                    if (!live[axis]) continue;
                    int k = std::min(BINS - 1, std::max(0, int((p.c[axis] - cb.mn[axis]) * scale[axis])));
                    bb[axis][k].grow(p.mn, p.mx);
                    cnt[axis][k]++;
                }
            }
            double best = std::numeric_limits<double>::infinity();
            int best_axis = -1, best_bin = -1;
            for (int axis = 0; axis < 3; ++axis) {
                if (!live[axis]) continue;
                double right_area[BINS];
                int right_cnt[BINS];
                FBox acc;
                acc.reset();
                int c = 0;
                double area = 0.0; // of `acc`: recomputed only when a bin adds something (most bins of a small node are empty)
                for (int k = BINS - 1; k > 0; --k) {
                    if (cnt[axis][k]) {
                        acc.grow(bb[axis][k].mn, bb[axis][k].mx);
                        area = acc.area();
                    }
                    c += cnt[axis][k];
                    right_area[k] = area;
                    right_cnt[k] = c;
                }
                acc.reset();
                c = 0;
                area = 0.0;
                for (int k = 0; k < BINS - 1; ++k) {
                    if (cnt[axis][k]) {
                        acc.grow(bb[axis][k].mn, bb[axis][k].mx);
                        area = acc.area();
                    }
                    c += cnt[axis][k];
                    if (c == 0 || right_cnt[k + 1] == 0) continue;
                    double cost = area * c + right_area[k + 1] * right_cnt[k + 1];
                    if (cost < best) {
                        best = cost;
                        best_axis = axis;
                        best_bin = k;
                    }
                }
            }
            if (best_axis >= 0) {
                const float sc = scale[best_axis], c0 = cb.mn[best_axis];
                auto it = std::partition(prims.begin() + lo, prims.begin() + hi, [&](const BuildPrim &p) {
                    int k = std::min(BINS - 1, std::max(0, int((p.c[best_axis] - c0) * sc)));
                    return k <= best_bin;
                });
                mid = int(it - prims.begin());
            }
        }
        if (mid <= lo || mid >= hi) { // median split on the widest centroid axis
            int axis = 0;
            for (int a = 1; a < 3; ++a)
                if (cb.mx[a] - cb.mn[a] > cb.mx[axis] - cb.mn[axis]) axis = a;
            mid = lo + n / 2;
            std::nth_element(prims.begin() + lo, prims.begin() + mid, prims.begin() + hi,
                             [&](const BuildPrim &a, const BuildPrim &b) { return a.c[axis] < b.c[axis]; });
        }
        return mid;
    }

    // builds an internal node over [lo, hi), hi - lo >= 2; returns its index
    int32_t build(int lo, int hi, int depth) {
        max_depth = std::max(max_depth, depth);
        int32_t me = int32_t(layout->nodes.size());
        layout->nodes.push_back(DNode{});
        int mid = split(lo, hi, depth);
        FBox lb = bounds(lo, mid), rb = bounds(mid, hi);
        int32_t left = (mid - lo == 1) ? emit_leaf(lo) : build(lo, mid, depth + 1);
        int32_t right = (hi - mid == 1) ? emit_leaf(mid) : build(mid, hi, depth + 1);
        DNode &nd = layout->nodes[me];
        for (int a = 0; a < 3; ++a) {
            nd.l_mn[a] = lb.mn[a];
            nd.l_mx[a] = lb.mx[a];
            nd.r_mn[a] = rb.mn[a];
            nd.r_mx[a] = rb.mx[a];
        }
        nd.left = left;
        nd.right = right;
        nd.pad0 = nd.pad1 = 0;
        return me;
    }
};

void export_sah(const HostSceneLayout &L, const std::vector<int32_t> &leaf_obj, int32_t ref, const float *mn, const float *mx,
                std::vector<HostNode> &out) {
    int32_t me = int32_t(out.size());
    out.push_back(HostNode{});
    for (int a = 0; a < 3; ++a) {
        out[me].mn[a] = mn[a];
        out[me].mx[a] = mx[a];
    }
    out[me].right = -1;
    out[me].prim = -1;
    if (ref < 0) {
        out[me].prim = leaf_obj[~ref];
        return;
    }
    const DNode nd = L.nodes[ref];
    export_sah(L, leaf_obj, nd.left, nd.l_mn, nd.l_mx, out);
    int32_t r = int32_t(out.size());
    export_sah(L, leaf_obj, nd.right, nd.r_mn, nd.r_mx, out);
    out[me].right = r;
}
} // namespace

DMaterial make_material(const RtHittable &h, int32_t host_index) {
    DMaterial m{};
    m.albedo = h.albedo;
    m.p0 = 0.f;
    m.p1 = 0.f;
    switch (h.style) {
    case RT_STYLE_FUZZED_REFLECTION: m.p0 = float(h.fuzz); break;
    case RT_STYLE_DIELECTRIC:
        m.p0 = float(h.ior);
        m.p1 = float(h.prob);
        break;
    case RT_STYLE_GLASS: m.p0 = float(h.ior); break;
    case RT_STYLE_LIGHT_SOURCE_CAP: m.p0 = float(h.p[0] + (h.radius - (h.radius / 4.0))); break; // Sphere.fs:191-192
    default: break;
    }
    m.style_rgb = (uint32_t(h.style) << 24) | (uint32_t(h.colour[0]) << 16) | (uint32_t(h.colour[1]) << 8) | uint32_t(h.colour[2]);
    m.texture = h.texture;
    m.flags = 0;
    if (h.shape != RT_SHAPE_INFINITE_PLANE && std::fabs(h.radius - 0.0) >= kTol && h.radius < 0.0) m.flags |= 1u; // Float.compare r 0 = Less
    if (h.shape == RT_SHAPE_INFINITE_PLANE) m.flags |= 2u;
    m.host_index = host_index;
    return m;
}

// FP32 (expanded form) or FP64 for an unbounded object — see DUnbounded.  The expanded forms lose accuracy only through
// the size of k next to the quantity wanted (2 r h for a ray origin at height h above a sphere, h for a plane): absolute
// error ~ 6e-8 (|o|^2 + 2 |o.c| + |k|).  With origins inside a scene of extent ~100 that is below 1e-6 in h when the
// sphere is at least as big as its distance from the world origin (|c| <= |r|, r >= 8: floors, domes) and for planes
// with |n.p0| <= 16; everything else keeps the FP64 path.
void classify_unbounded(DUnbounded &u) {
    u.fp32 = 0;
    u.k = 0.f;
    bool exact = true;
    for (int a = 0; a < 3; ++a) exact = exact && double(float(u.p[a])) == u.p[a];
    if (u.shape == RT_SHAPE_INFINITE_PLANE) {
        double k = double(u.n[0]) * u.p[0] + double(u.n[1]) * u.p[1] + double(u.n[2]) * u.p[2];
        if (std::fabs(k) <= 16.0) {
            u.fp32 = 1;
            u.k = float(k);
        }
        return;
    }
    double c2 = u.p[0] * u.p[0] + u.p[1] * u.p[1] + u.p[2] * u.p[2];
    double r = std::fabs(double(u.r));
    if (exact && r >= 8.0 && c2 <= r * r * 1.0000001 && double(u.r) * double(u.r) == u.r2) {
        u.fp32 = 1;
        u.k = float(c2 - u.r2);
        for (int a = 0; a < 3; ++a) u.n[a] = float(u.p[a]);
    }
}

DUnbounded make_unbounded(const RtHittable &h) {
    DUnbounded u{};
    for (int a = 0; a < 3; ++a) {
        u.p[a] = h.p[a];
        u.n[a] = float(h.n[a]);
    }
    u.r2 = h.radius * h.radius; // Sphere.make, Sphere.fs:326
    u.r = float(h.radius);
    u.shape = h.shape;
    classify_unbounded(u);
    return u;
}

void build_device_layout(const RtHittable *objs, int32_t n_objs, HostSceneLayout &L, std::vector<HostNode> &sah_tree_out) {
    L = HostSceneLayout{};
    sah_tree_out.clear();
    SahBuilder b;
    b.objs = objs;
    b.layout = &L;
    std::vector<int32_t> unbounded;
    for (int32_t i = 0; i < n_objs; ++i) {
        const RtHittable &h = objs[i];
        if (h.shape != RT_SHAPE_SPHERE) {
            unbounded.push_back(i);
            continue;
        }
        if (h.radius < 0.0) continue; // inverted box: never hit in the reference (F16); kept only in the reference tree
        BuildPrim p;
        float cf[3] = {float(h.p[0]), float(h.p[1]), float(h.p[2])};
        float rf = float(h.radius);
        for (int a = 0; a < 3; ++a) {
            p.mn[a] = round_down(double(cf[a]) - double(rf));
            p.mx[a] = round_up(double(cf[a]) + double(rf));
            p.c[a] = cf[a];
        }
        p.obj = i;
        b.prims.push_back(p);
    }
    int n = int(b.prims.size());
    if (n == 1) {
        // a single leaf: wrap it in a node whose right child is the box {+inf, +inf}, which no ray enters
        L.nodes.push_back(DNode{});
        int32_t leaf = b.emit_leaf(0);
        DNode &nd = L.nodes[0];
        for (int a = 0; a < 3; ++a) {
            nd.l_mn[a] = b.prims[0].mn[a];
            nd.l_mx[a] = b.prims[0].mx[a];
            nd.r_mn[a] = std::numeric_limits<float>::infinity();
            nd.r_mx[a] = std::numeric_limits<float>::infinity();
        }
        nd.left = leaf;
        nd.right = leaf;
        L.root_is_leaf = 1;
        b.max_depth = 1;
    } else if (n >= 2) {
        b.build(0, n, 1);
    }
    L.n_bounded = int32_t(L.spheres.size());
    L.max_depth = b.max_depth;
    std::vector<int32_t> device_id_of(n_objs, -1);
    for (int32_t k = 0; k < L.n_bounded; ++k) {
        L.materials.push_back(make_material(objs[b.leaf_obj[k]], b.leaf_obj[k]));
        device_id_of[b.leaf_obj[k]] = k;
    }
    for (int32_t i : unbounded) {
        device_id_of[i] = L.n_bounded + int32_t(L.unbounded.size());
        L.unbounded.push_back(make_unbounded(objs[i]));
        L.materials.push_back(make_material(objs[i], i));
    }
    L.device_id_of = device_id_of; // bounded spheres with negative radius keep id -1: they can never be returned
    (void)sah_tree_out; // the inspection form of the tree is made on first request (scene_ensure_sah_tree)
}

// The SAH tree in the HostNode form rt_scene_bvh_nodes hands out: only inspection asks for it, so it is built on first use.
void scene_ensure_sah_tree(RtScene *s) {
    if (s->sah_built) return;
    s->sah_built = true;
    const HostSceneLayout &L = s->layout;
    s->sah_tree.clear();
    if (L.n_bounded < 1) return;
    std::vector<int32_t> leaf_obj(size_t(L.n_bounded));
    for (int32_t k = 0; k < L.n_bounded; ++k) leaf_obj[k] = L.materials[k].host_index;
    FBox rootb;
    rootb.reset();
    if (L.root_is_leaf) {
        rootb.grow(L.nodes[0].l_mn, L.nodes[0].l_mx);
        export_sah(L, leaf_obj, L.nodes[0].left, rootb.mn, rootb.mx, s->sah_tree);
    } else {
        rootb.grow(L.nodes[0].l_mn, L.nodes[0].l_mx);
        rootb.grow(L.nodes[0].r_mn, L.nodes[0].r_mx);
        export_sah(L, leaf_obj, 0, rootb.mn, rootb.mx, s->sah_tree);
    }
}

// ---------------------------------------------------------------------------------------------
// 8-wide compressed BVH: greedy collapse of the SAH BVH2 (open the child of largest area until there are eight),
// children placed in octant-ordered slots, boxes quantised outwards to 8 bits on a per-node power-of-two grid
// ---------------------------------------------------------------------------------------------
void build_wide_layout(HostSceneLayout &L) {
    if (!L.wide_nodes.empty() || L.n_bounded < 1) return;
    struct Child {
        int32_t ref; // BVH2 ref: >= 0 internal node, < 0 leaf ~sphere
        float mn[3], mx[3];
    };
    auto area = [](const Child &c) {
        double dx = double(c.mx[0]) - c.mn[0], dy = double(c.mx[1]) - c.mn[1], dz = double(c.mx[2]) - c.mn[2];
        return (dx < 0 || dy < 0 || dz < 0) ? 0.0 : dx * dy + dy * dz + dz * dx;
    };
    auto children_of = [&](int32_t node, std::vector<Child> &out) {
        const DNode &nd = L.nodes[node];
        Child l{nd.left, {nd.l_mn[0], nd.l_mn[1], nd.l_mn[2]}, {nd.l_mx[0], nd.l_mx[1], nd.l_mx[2]}};
        Child r{nd.right, {nd.r_mn[0], nd.r_mn[1], nd.r_mn[2]}, {nd.r_mx[0], nd.r_mx[1], nd.r_mx[2]}};
        out.push_back(l);
        if (!(L.root_is_leaf && node == 0)) out.push_back(r); // a one-sphere scene: the right child is a never-entered dummy
    };
    // spheres below each BVH2 node: a subtree of at most kLeafMax spheres can sit in ONE leaf slot of a wide node
    constexpr int kLeafMax = 3;
    std::vector<int32_t> below(L.nodes.size(), 0);
    for (int32_t i = int32_t(L.nodes.size()) - 1; i >= 0; --i) { // children have larger indices (DFS pre-order)
        const DNode &nd = L.nodes[i];
        below[i] = (nd.left < 0 ? 1 : below[nd.left]) + ((L.root_is_leaf && i == 0) ? 0 : (nd.right < 0 ? 1 : below[nd.right]));
    }
    auto count_of = [&](int32_t ref) { return ref < 0 ? 1 : below[ref]; };
    std::vector<int32_t> gathered;
    auto gather = [&](int32_t ref, auto &&self) -> void { // device ids of the spheres below `ref`, in tree order
        if (ref < 0) {
            gathered.push_back(~ref);
            return;
        }
        self(L.nodes[ref].left, self);
        if (!(L.root_is_leaf && ref == 0)) self(L.nodes[ref].right, self);
    };
    struct Work {
        int32_t bvh2;
        uint32_t index;
        int32_t depth;
    };
    L.wide_nodes.assign(1, DWideNode{});
    L.wide_spheres.clear();
    L.wide_to_dev.clear();
    std::vector<Work> work{{0, 0u, 1}};
    for (size_t w = 0; w < work.size(); ++w) {
        const Work job = work[w];
        L.wide_depth = std::max(L.wide_depth, job.depth);
        std::vector<Child> ch;
        children_of(job.bvh2, ch);
        // open the child of largest area until there are eight: first the subtrees too big for a leaf slot, then (slots
        // permitting) the small ones, whose spheres then get boxes of their own
        for (int pass = 0; pass < 2; ++pass)
            while (ch.size() < 8) {
                int pick = -1;
                double best = -1.0;
                for (size_t i = 0; i < ch.size(); ++i)
                    if (ch[i].ref >= 0 && (pass == 1 || count_of(ch[i].ref) > kLeafMax) && area(ch[i]) > best) {
                        best = area(ch[i]);
                        pick = int(i);
                    }
                if (pick < 0) break;
                const int32_t open = ch[pick].ref;
                ch.erase(ch.begin() + pick);
                children_of(open, ch);
            }
        const int n = int(ch.size());
        float lo[3], hi[3];
        for (int a = 0; a < 3; ++a) {
            lo[a] = ch[0].mn[a];
            hi[a] = ch[0].mx[a];
            for (int i = 1; i < n; ++i) {
                lo[a] = std::min(lo[a], ch[i].mn[a]);
                hi[a] = std::max(hi[a], ch[i].mx[a]);
            }
        }
        // octant-ordered slots: greedily give each (child, slot) pair of largest projection of the child's centre
        // (relative to the node's) on the slot's diagonal
        int slot_of[8], child_in[8];
        std::fill(slot_of, slot_of + 8, -1);
        std::fill(child_in, child_in + 8, -1);
        double cost[8][8];
        for (int i = 0; i < n; ++i)
            for (int s = 0; s < 8; ++s) {
                double c = 0.0;
                for (int a = 0; a < 3; ++a) {
                    double rel = 0.5 * (double(ch[i].mn[a]) + ch[i].mx[a]) - 0.5 * (double(lo[a]) + hi[a]);
                    c += ((s >> (2 - a)) & 1) ? rel : -rel;
                }
                cost[i][s] = c;
            }
        for (int k = 0; k < n; ++k) {
            int bi = -1, bs = -1;
            for (int i = 0; i < n; ++i) {
                if (slot_of[i] >= 0) continue;
                for (int s = 0; s < 8; ++s)
                    if (child_in[s] < 0 && (bi < 0 || cost[i][s] > cost[bi][bs])) {
                        bi = i;
                        bs = s;
                    }
            }
            slot_of[bi] = bs;
            child_in[bs] = bi;
        }
        DWideNode nd{};
        int ebits[3];
        double step[3];
        for (int a = 0; a < 3; ++a) {
            nd.p[a] = lo[a];
            double ext = double(hi[a]) - double(lo[a]);
            int e = ext > 0.0 ? int(std::ceil(std::log2(ext / 255.0))) : -100;
            e = std::max(-100, std::min(100, e));
            while (std::ldexp(255.0, e) < ext) ++e; // log2 rounding: the grid must span the node
            ebits[a] = e;
            step[a] = std::ldexp(1.0, e);
            nd.e[a] = uint8_t(e + 127 + 15);
        }
        nd.child_base = uint32_t(L.wide_nodes.size());
        nd.prim_base = uint32_t(L.wide_spheres.size());
        int n_internal = 0, n_prims = 0;
        for (int s = 0; s < 8; ++s) {
            nd.qlo_x[s] = nd.qlo_y[s] = nd.qlo_z[s] = 255; // empty slot: an inverted box
            nd.qhi_x[s] = nd.qhi_y[s] = nd.qhi_z[s] = 0;
            const int i = child_in[s];
            if (i < 0) continue;
            uint8_t *qlo[3] = {nd.qlo_x, nd.qlo_y, nd.qlo_z}, *qhi[3] = {nd.qhi_x, nd.qhi_y, nd.qhi_z};
            for (int a = 0; a < 3; ++a) {
                double l = std::floor((double(ch[i].mn[a]) - double(lo[a])) / step[a]);
                double h = std::ceil((double(ch[i].mx[a]) - double(lo[a])) / step[a]);
                qlo[a][s] = uint8_t(std::max(0.0, std::min(255.0, l)));
                qhi[a][s] = uint8_t(std::max(0.0, std::min(255.0, h)));
            }
            if (ch[i].ref >= 0 && count_of(ch[i].ref) > kLeafMax) {
                nd.imask |= uint8_t(1u << s);
                nd.meta[s] = uint8_t((1u << 5) | (24u + unsigned(s)));
                work.push_back(Work{ch[i].ref, nd.child_base + uint32_t(n_internal), job.depth + 1});
                ++n_internal;
            } else { // a leaf slot: one to three spheres, the count in unary
                gathered.clear();
                gather(ch[i].ref, gather);
                nd.meta[s] = uint8_t((((1u << gathered.size()) - 1u) << 5) | unsigned(n_prims));
                for (int32_t dev : gathered) {
                    L.wide_spheres.push_back(L.spheres[dev]);
                    L.wide_to_dev.push_back(dev);
                    ++n_prims;
                }
            }
        }
        (void)ebits;
        L.wide_nodes.resize(L.wide_nodes.size() + n_internal);
        L.wide_nodes[job.index] = nd;
    }
    L.dev_to_wide.assign(L.n_bounded, -1);
    for (size_t k = 0; k < L.wide_to_dev.size(); ++k) L.dev_to_wide[L.wide_to_dev[k]] = int32_t(k);
}

// The reference-topology tree is only needed by the conformance traversal and by inspection; it is built on
// first use (its median-split build sorts every range three times: half a second for 100 000 spheres).
void scene_ensure_reference(RtScene *s) {
    if (s->ref_built) return;
    s->ref_built = true;
    std::vector<int32_t> bounded;
    for (int32_t i = 0; i < int32_t(s->objects.size()); ++i)
        if (s->objects[i].shape == RT_SHAPE_SPHERE) bounded.push_back(i); // Hittable.BoundingBox, Hittable.fs:14-18
    build_reference_tree(s->objects.data(), bounded, s->ref_tree);
    HostSceneLayout &L = s->layout;
    L.ref_nodes.clear();
    for (const HostNode &hn : s->ref_tree) {
        DRefNode r{};
        for (int a = 0; a < 3; ++a) {
            bool inverted = hn.mn[a] > hn.mx[a];
            r.mn[a] = inverted ? float(hn.mn[a]) : round_down(hn.mn[a]);
            r.mx[a] = inverted ? float(hn.mx[a]) : round_up(hn.mx[a]);
        }
        r.right = hn.right;
        r.prim = hn.prim >= 0 ? L.device_id_of[hn.prim] : -1;
        L.ref_nodes.push_back(r);
    }
}

// Scene.make's preconditions on one object (shape, style, plane cases, texture index, finite coordinates)
int check_object(const RtHittable &h, int32_t i, int32_t n_textures, const char *who) {
    if (h.shape < RT_SHAPE_SPHERE || h.shape > RT_SHAPE_INFINITE_PLANE)
        return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": object " + std::to_string(i) + " has an unknown shape");
    if (h.style < RT_STYLE_LIGHT_SOURCE || h.style > RT_STYLE_GLASS)
        return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": object " + std::to_string(i) + " has an unknown style");
    if (h.shape == RT_SHAPE_INFINITE_PLANE) {
        // InfinitePlaneStyle has four cases only (InfinitePlane.fs:3-13, F13)
        if (h.style == RT_STYLE_LIGHT_SOURCE_CAP || h.style == RT_STYLE_DIELECTRIC || h.style == RT_STYLE_GLASS)
            return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": object " + std::to_string(i) + ": InfinitePlaneStyle has no such case");
        double nn = h.n[0] * h.n[0] + h.n[1] * h.n[1] + h.n[2] * h.n[2];
        if (std::fabs(nn - 1.0) > 1e-6)
            return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": object " + std::to_string(i) + ": plane normal must be a unit vector");
        if (h.style != RT_STYLE_LIGHT_SOURCE && h.texture >= 0)
            return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": object " + std::to_string(i) + ": reflecting planes carry a colour, not a texture");
    }
    if (h.texture >= n_textures) return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": object " + std::to_string(i) + " references a missing texture");
    for (int a = 0; a < 3; ++a)
        if (!std::isfinite(h.p[a])) return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": object " + std::to_string(i) + " has a non-finite coordinate");
    if (h.shape != RT_SHAPE_INFINITE_PLANE && !std::isfinite(h.radius))
        return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": object " + std::to_string(i) + " has a non-finite radius");
    return RT_OK;
}

// the texture table: image sizes, checker sub-texture indices, map radii, and no checker cycle or nest deeper than the device follows
int check_textures(const RtTexture *textures, int32_t n_textures, const char *who) {
    for (int32_t t = 0; t < n_textures; ++t) {
        const RtTexture &x = textures[t];
        if (x.kind == RT_TEX_IMAGE) {
            if (x.width <= 0 || x.height <= 0 || !x.rgb8) return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": image texture " + std::to_string(t) + " is empty");
        } else if (x.kind == RT_TEX_CHECKERED) {
            if (x.even < 0 || x.even >= n_textures || x.odd < 0 || x.odd >= n_textures || x.even == t || x.odd == t)
                return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": checkered texture " + std::to_string(t) + " has bad sub-textures");
        } else if (x.kind != RT_TEX_COLOUR) {
            return fail(RT_ERR_UNSUPPORTED, std::string(who) + ": texture " + std::to_string(t) + " is of a kind the device cannot evaluate (closures must be baked to an image)");
        }
        if (x.kind != RT_TEX_COLOUR && !(std::fabs(x.map_radius) > 0.0))
            return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": texture " + std::to_string(t) + " has map_radius 0");
    }
    // Checkered textures nest (Texture.fs:56-62); the device follows at most kMaxCheckerDepth levels, so deeper nests and
    // cycles (which the reference's immutable values cannot even express) are refused here rather than rendered black
    {
        constexpr int kMaxCheckerDepth = 8;
        std::vector<int> depth(size_t(n_textures), -1); // -1 unknown, -2 on the current path
        std::vector<std::pair<int32_t, int>> stack;
        for (int32_t root = 0; root < n_textures; ++root) {
            if (depth[root] >= 0) continue;
            stack.push_back({root, 0});
            while (!stack.empty()) {
                auto [t, phase] = stack.back();
                const RtTexture &x = textures[t];
                if (x.kind != RT_TEX_CHECKERED) {
                    depth[t] = 0;
                    stack.pop_back();
                    continue;
                }
                if (phase == 0) {
                    depth[t] = -2;
                    stack.back().second = 1;
                    for (int32_t c : {x.even, x.odd}) {
                        if (depth[c] == -2) return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": checkered texture " + std::to_string(t) + " is part of a cycle");
                        if (depth[c] == -1) stack.push_back({c, 0});
                    }
                } else {
                    depth[t] = 1 + std::max(depth[x.even], depth[x.odd]);
                    if (depth[t] > kMaxCheckerDepth)
                        return fail(RT_ERR_UNSUPPORTED, std::string(who) + ": checkered textures nested deeper than " + std::to_string(kMaxCheckerDepth) + " levels");
                    stack.pop_back();
                }
            }
        }
    }
    return RT_OK;
}

} // namespace rtfs

using namespace rtfs;

// =================================================================================================
// C ABI — host-side entry points
// =================================================================================================
extern "C" {

int rt_abi_version(void) { return RT_ABI_VERSION; }
const char *rt_last_error(void) { return g_last_error.c_str(); }

// Camera.makeBasic, RayTracing/Camera.fs:34-59
int rt_camera_make_basic(int32_t samples_per_pixel, double focal_length, double aspect_ratio, const double origin[3],
                         const double view_direction[3], const double view_up[3], RtCamera *out) {
    if (!origin || !view_direction || !view_up || !out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_camera_make_basic: null argument");
    D3 o = load(origin), view = load(view_direction), up = load(view_up);
    if (std::fabs(dot(view, view) - 1.0) > 1e-6)
        return fail(RT_ERR_INVALID_ARGUMENT, "rt_camera_make_basic: view_direction must be a unit vector (UnitVector in the reference)");
    const double height = 2.0;
    D3 corner = o + focal_length * view; // Ray.walkAlong view focalLength
    // Plane.makeNormalTo' corner viewDirection, Plane.fs:22-38
    D3 v1 = (std::fabs(view.z - 0.0) < kTol) ? D3{0.0, 0.0, 1.0} : D3{1.0, 1.0, (-view.x - view.y) / view.z};
    D3 p_v2, p_v1;
    if (!unitise(cross(view, v1), p_v2) || !unitise(v1, p_v1))
        return fail(RT_ERR_DEGENERATE, "rt_camera_make_basic: Plane.makeNormalTo failed to normalise (the reference throws)");
    // Plane.basis viewUp viewPlane, Plane.fs:82-97
    D3 upn;
    if (!unitise(up, upn)) return fail(RT_ERR_DEGENERATE, "rt_camera_make_basic: viewUp has zero length (the reference throws)");
    double c1 = dot(p_v1, upn), c2 = dot(p_v2, upn);
    D3 yv, xv;
    if (!unitise(c1 * p_v1 + c2 * p_v2, yv) || !unitise(c2 * p_v1 + (-c1) * p_v2, xv))
        return fail(RT_ERR_DEGENERATE, "rt_camera_make_basic: viewUp is parallel to the view direction (the reference throws)");
    std::memset(out, 0, sizeof *out);
    store(out->view_origin, o);
    store(out->view_dir, view);
    store(out->xaxis_origin, corner);
    store(out->xaxis_dir, xv);
    store(out->yaxis_dir, yv);
    out->viewport_height = height;
    out->viewport_width = aspect_ratio * height;
    out->focal_length = focal_length;
    out->samples_per_pixel = samples_per_pixel;
    out->bounce_depth = 150; // Camera.fs:58
    return RT_OK;
}

// PixelOutput.correct, RayTracing/ImageOutput.fs:11-18
uint8_t rt_gamma_correct(uint8_t b) {
    int i = int(std::nearbyint(std::sqrt(double(b) / 255.0) * 255.0)); // Math.Round: half to even
    if (i == 256) i = 255;
    return uint8_t(i);
}

// ImageOutput.writePpm, RayTracing/ImageOutput.fs:163-197
static void ppm_build(const uint8_t *rgb, int32_t rows, int32_t cols, bool gamma, std::string &s) {
    uint8_t lut[256];
    for (int i = 0; i < 256; ++i) lut[i] = gamma ? rt_gamma_correct(uint8_t(i)) : uint8_t(i);
    char num[256][4];
    int len[256];
    for (int i = 0; i < 256; ++i) len[i] = std::snprintf(num[i], 4, "%d", i);
    s.clear();
    s.reserve(size_t(rows) * cols * 12 + 32);
    s += "P3\n";
    s += std::to_string(cols) + " " + std::to_string(rows) + "\n";
    s += "255\n";
    for (int32_t r = 0; r < rows; ++r) {
        for (int32_t c = 0; c < cols; ++c) {
            const uint8_t *p = rgb + (size_t(r) * cols + c) * 3;
            for (int k = 0; k < 3; ++k) {
                uint8_t v = lut[p[k]];
                s.append(num[v], size_t(len[v]));
                if (k != 2) s.push_back(' ');
            }
            if (c != cols - 1) s.push_back(' ');
        }
        if (r != rows - 1) s.push_back('\n');
    }
}
int rt_ppm_format(const uint8_t *rgb, int32_t rows, int32_t cols, int32_t gamma_correct, char *out, size_t cap, size_t *len) {
    if (!rgb || rows <= 0 || cols <= 0 || !len) return fail(RT_ERR_INVALID_ARGUMENT, "rt_ppm_format: bad argument");
    std::string s;
    ppm_build(rgb, rows, cols, gamma_correct != 0, s);
    *len = s.size();
    if (out && cap) std::memcpy(out, s.data(), std::min(cap, s.size()));
    return RT_OK;
}
int rt_ppm_write_file(const uint8_t *rgb, int32_t rows, int32_t cols, int32_t gamma_correct, const char *path) {
    if (!rgb || rows <= 0 || cols <= 0 || !path) return fail(RT_ERR_INVALID_ARGUMENT, "rt_ppm_write_file: bad argument");
    std::string s;
    ppm_build(rgb, rows, cols, gamma_correct != 0, s);
    FILE *f = std::fopen(path, "wb");
    if (!f) return fail(RT_ERR_IO, std::string("rt_ppm_write_file: cannot open ") + path);
    size_t w = std::fwrite(s.data(), 1, s.size(), f);
    std::fclose(f);
    if (w != s.size()) return fail(RT_ERR_IO, "rt_ppm_write_file: short write");
    return RT_OK;
}

// Scene.make, RayTracing/Scene.fs:15-28
int rt_scene_create(const RtHittable *objects, int32_t n_objects, const RtTexture *textures, int32_t n_textures,
                    int32_t device, RtScene **out) {
    if (!out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_scene_create: out is null");
    *out = nullptr;
    if (n_objects < 0 || n_textures < 0 || (n_objects > 0 && !objects) || (n_textures > 0 && !textures))
        return fail(RT_ERR_INVALID_ARGUMENT, "rt_scene_create: bad array arguments");
    for (int32_t i = 0; i < n_objects; ++i) {
        int rc = check_object(objects[i], i, n_textures, "rt_scene_create");
        if (rc != RT_OK) return rc;
    }
    int rc = check_textures(textures, n_textures, "rt_scene_create");
    if (rc != RT_OK) return rc;
    auto *s = new RtScene();
    s->objects.assign(objects, objects + n_objects);
    s->textures.assign(textures, textures + n_textures);
    s->texture_pixels.resize(n_textures);
    for (int32_t t = 0; t < n_textures; ++t) {
        if (textures[t].kind == RT_TEX_IMAGE) {
            size_t bytes = size_t(textures[t].width) * textures[t].height * 3;
            s->texture_pixels[t].assign(textures[t].rgb8, textures[t].rgb8 + bytes);
            s->textures[t].rgb8 = s->texture_pixels[t].data();
        } else {
            s->textures[t].rgb8 = nullptr;
        }
    }
    build_device_layout(s->objects.data(), n_objects, s->layout, s->sah_tree);
    if (s->layout.max_depth > 60) {
        delete s;
        return fail(RT_ERR_UNSUPPORTED, "rt_scene_create: BVH deeper than the traversal stack");
    }
    s->device = device;
    if (device >= 0) {
        int rc = device_scene_upload(s);
        if (rc != RT_OK) {
            delete s;
            return rc;
        }
    }
    *out = s;
    return RT_OK;
}

void rt_scene_destroy(RtScene *scene) {
    if (!scene) return;
    if (scene->dev) device_scene_free(scene);
    delete scene;
}

int rt_scene_bvh_node_count(const RtScene *scene, int32_t which) {
    if (!scene) return fail(RT_ERR_INVALID_ARGUMENT, "rt_scene_bvh_node_count: null scene");
    if (int rc = device_scene_sync_layout(const_cast<RtScene *>(scene)); rc != RT_OK) return rc;
    if (which == RT_BVH_REFERENCE) scene_ensure_reference(const_cast<RtScene *>(scene));
    else scene_ensure_sah_tree(const_cast<RtScene *>(scene));
    return int(which == RT_BVH_REFERENCE ? scene->ref_tree.size() : scene->sah_tree.size());
}
int rt_scene_bvh_nodes(const RtScene *scene, int32_t which, double *bounds, int32_t *right, int32_t *prim) {
    if (!scene || !bounds || !right || !prim) return fail(RT_ERR_INVALID_ARGUMENT, "rt_scene_bvh_nodes: null argument");
    if (int rc = device_scene_sync_layout(const_cast<RtScene *>(scene)); rc != RT_OK) return rc;
    if (which == RT_BVH_REFERENCE) scene_ensure_reference(const_cast<RtScene *>(scene));
    else scene_ensure_sah_tree(const_cast<RtScene *>(scene));
    const auto &t = which == RT_BVH_REFERENCE ? scene->ref_tree : scene->sah_tree;
    for (size_t i = 0; i < t.size(); ++i) {
        for (int a = 0; a < 3; ++a) {
            bounds[6 * i + a] = t[i].mn[a];
            bounds[6 * i + 3 + a] = t[i].mx[a];
        }
        right[i] = t[i].right;
        prim[i] = t[i].prim;
    }
    return RT_OK;
}
size_t rt_scene_device_bytes(const RtScene *scene) { return scene ? device_scene_bytes(scene) : 0; }

// Builds (if need be) and checks the 8-wide compressed tree on the host: every bounded sphere sits in exactly one leaf
// slot, and the decoded box of every slot contains all the spheres below it (each plane decoded as p + q 2^e).
int rt_scene_wide_bvh_check(RtScene *scene, int32_t *n_nodes, int32_t *depth, int32_t *n_spheres, double *mean_children) {
    if (!scene) return fail(RT_ERR_INVALID_ARGUMENT, "rt_scene_wide_bvh_check: null scene");
    if (int rc = device_scene_sync_layout(scene); rc != RT_OK) return rc;
    HostSceneLayout &L = scene->layout;
    build_wide_layout(L);
    std::vector<int> seen(size_t(L.n_bounded), 0);
    size_t children = 0;
    struct Item {
        uint32_t node;
        double mn[3], mx[3]; // what the ancestors' slots promise to contain
        bool bounded;
    };
    std::vector<Item> todo;
    if (!L.wide_nodes.empty()) todo.push_back(Item{0u, {0, 0, 0}, {0, 0, 0}, false});
    while (!todo.empty()) {
        Item it = todo.back();
        todo.pop_back();
        if (it.node >= L.wide_nodes.size()) return fail(RT_ERR_DEGENERATE, "wide BVH: child index out of range");
        const DWideNode &nd = L.wide_nodes[it.node];
        int internal = 0;
        for (int s = 0; s < 8; ++s) {
            if (nd.meta[s] == 0) continue;
            ++children;
            const uint8_t *qlo[3] = {nd.qlo_x, nd.qlo_y, nd.qlo_z}, *qhi[3] = {nd.qhi_x, nd.qhi_y, nd.qhi_z};
            Item c{0u, {0, 0, 0}, {0, 0, 0}, true};
            for (int a = 0; a < 3; ++a) {
                double step = std::ldexp(1.0, int(nd.e[a]) - 127 - 15);
                c.mn[a] = double(nd.p[a]) + qlo[a][s] * step;
                c.mx[a] = double(nd.p[a]) + qhi[a][s] * step;
                if (it.bounded) { // a child's box may stick out of its parent's by quantisation only if the content does not
                    c.mn[a] = std::max(c.mn[a], it.mn[a]);
                    c.mx[a] = std::min(c.mx[a], it.mx[a]);
                }
            }
            const bool inner = (nd.imask >> s) & 1u;
            if (inner) {
                if (nd.meta[s] != uint8_t((1u << 5) | (24u + unsigned(s)))) return fail(RT_ERR_DEGENERATE, "wide BVH: bad meta of an internal slot");
                c.node = nd.child_base + uint32_t(internal++);
                todo.push_back(c);
            } else {
                int count = nd.meta[s] >> 5, off = nd.meta[s] & 31;
                count = count == 1 ? 1 : (count == 3 ? 2 : (count == 7 ? 3 : -1));
                if (count < 0 || off + count > 24) return fail(RT_ERR_DEGENERATE, "wide BVH: bad meta of a leaf slot");
                for (int k = 0; k < count; ++k) {
                    size_t w = size_t(nd.prim_base) + off + k;
                    if (w >= L.wide_to_dev.size()) return fail(RT_ERR_DEGENERATE, "wide BVH: sphere index out of range");
                    int32_t dev = L.wide_to_dev[w];
                    if (dev < 0 || dev >= L.n_bounded || L.dev_to_wide[dev] != int32_t(w)) return fail(RT_ERR_DEGENERATE, "wide BVH: index maps disagree");
                    ++seen[dev];
                    const DSphere &sp = L.spheres[dev];
                    const float c3[3] = {sp.cx, sp.cy, sp.cz};
                    for (int a = 0; a < 3; ++a)
                        if (double(c3[a]) - double(sp.r) < c.mn[a] || double(c3[a]) + double(sp.r) > c.mx[a])
                            return fail(RT_ERR_DEGENERATE, "wide BVH: a sphere sticks out of a box above it");
                }
            }
        }
    }
    for (int v : seen)
        if (v != 1) return fail(RT_ERR_DEGENERATE, "wide BVH: a sphere is missing or duplicated");
    if (n_nodes) *n_nodes = int32_t(L.wide_nodes.size());
    if (depth) *depth = L.wide_depth;
    if (n_spheres) *n_spheres = int32_t(L.wide_to_dev.size());
    if (mean_children) *mean_children = L.wide_nodes.empty() ? 0.0 : double(children) / double(L.wide_nodes.size());
    return RT_OK;
}

// Checks the nodes as the DEVICE will read them (device_node_of: centre / half-extent boxes, left and right child side by
// side): every decoded box c -+ h contains the min / max box it was made from (so also every sphere below it), h >= 0, the
// child refs are untouched, every bounded sphere is the leaf of exactly one node, and the tree is as deep as max_depth says
// (the render kernels size their walk stacks from it).  After rt_scene_update refit the tree on the device, the nodes are
// the device's min / max boxes, and every node record the device walks must also be device_node_of of them (the device's
// conversion is the host's).
int rt_scene_device_bvh_check(RtScene *scene, int32_t *n_nodes, int32_t *depth, int32_t *n_spheres) {
    if (!scene) return fail(RT_ERR_INVALID_ARGUMENT, "rt_scene_device_bvh_check: null scene");
    if (int rc = device_scene_sync_layout(scene); rc != RT_OK) return rc;
    const HostSceneLayout &L = scene->layout;
    if (!scene->device_nodes.empty()) {
        if (scene->device_nodes.size() != L.nodes.size()) return fail(RT_ERR_DEGENERATE, "device BVH: node count differs on the device");
        for (size_t i = 0; i < L.nodes.size(); ++i) {
            const DNode host = device_node_of(L.nodes[i]);
            if (std::memcmp(&host, &scene->device_nodes[i], sizeof(DNode)) != 0)
                return fail(RT_ERR_DEGENERATE, "device BVH: node " + std::to_string(i) + " on the device is not device_node_of its min / max boxes");
        }
    }
    std::vector<int> seen(size_t(L.n_bounded), 0);
    int deepest = 0;
    struct Item {
        int32_t ref;
        int depth;
    };
    std::vector<Item> todo;
    if (L.n_bounded > 0) todo.push_back(Item{0, 1});
    size_t visited = 0;
    while (!todo.empty()) {
        const Item it = todo.back();
        todo.pop_back();
        if (it.ref < 0 || size_t(it.ref) >= L.nodes.size()) return fail(RT_ERR_DEGENERATE, "device BVH: child index out of range");
        if (++visited > L.nodes.size()) return fail(RT_ERR_DEGENERATE, "device BVH: a node is reachable twice");
        deepest = std::max(deepest, it.depth);
        const DNode &src = L.nodes[size_t(it.ref)];
        const DNode dev = device_node_of(src);
        const float *q = dev.l_mn; // the twelve box floats in device order
        if (dev.left != src.left || dev.right != src.right) return fail(RT_ERR_DEGENERATE, "device BVH: child refs changed by the conversion");
        for (int side = 0; side < 2; ++side) {
            if (L.root_is_leaf && it.ref == 0 && side == 1) continue; // the never-entered dummy of a one-sphere tree
            const float *mn = side ? src.r_mn : src.l_mn, *mx = side ? src.r_mx : src.l_mx;
            for (int a = 0; a < 3; ++a) {
                const double c = q[2 * a + side], h = q[6 + 2 * a + side];
                if (!(h >= 0.0) || !(c - h <= double(mn[a])) || !(c + h >= double(mx[a])))
                    return fail(RT_ERR_DEGENERATE, "device BVH: a centre / half-extent box is smaller than the box it was made from");
            }
            const int32_t child = side ? src.right : src.left;
            if (child >= 0) {
                todo.push_back(Item{child, it.depth + 1});
                continue;
            }
            const int32_t k = ~child;
            if (k < 0 || k >= L.n_bounded) return fail(RT_ERR_DEGENERATE, "device BVH: leaf sphere index out of range");
            ++seen[size_t(k)];
            const DSphere &sp = L.spheres[size_t(k)];
            const float cs[3] = {sp.cx, sp.cy, sp.cz};
            for (int a = 0; a < 3; ++a) {
                const double c = q[2 * a + side], h = q[6 + 2 * a + side], r = std::fabs(double(sp.r));
                if (!(c - h <= double(cs[a]) - r) || !(c + h >= double(cs[a]) + r)) return fail(RT_ERR_DEGENERATE, "device BVH: a leaf box does not contain its sphere");
            }
        }
    }
    for (int v : seen)
        if (v != 1) return fail(RT_ERR_DEGENERATE, "device BVH: a sphere is missing or duplicated");
    if (L.n_bounded > 0 && deepest > L.max_depth) return fail(RT_ERR_DEGENERATE, "device BVH: deeper than max_depth (the walk stacks are sized from it)");
    if (n_nodes) *n_nodes = int32_t(L.nodes.size());
    if (depth) *depth = deepest;
    if (n_spheres) *n_spheres = L.n_bounded;
    return RT_OK;
}

} // extern "C"
