// rtfs_host_debug.cpp — the device functions of rtfs_core.cuh compiled for the HOST, under AddressSanitizer and
// UndefinedBehaviorSanitizer, with a scalar driver of the frame (probe -> flags -> main -> mean).  Test infrastructure
// (tests/test_host_debug_asan.py): compute-sanitizer is closed on this pool, so memory safety of the traversal, the
// scatter and the item bookkeeping is checked here instead — every array access of path_begin / path_step goes through
// the same code the kernels compile, with the stacks and the scene arrays as ordinary host allocations that ASan guards.
// The arithmetic differs from the device's only where a MUFU approximation or an FMA contraction does, so frames are
// compared with the oracle the way the GPU's are (almost all pixels byte-identical under the shared counter RNG).
//
// Never linked into librtfs_b200.so.
#define RTFS_HOST_DEBUG 1
#define RTFS_HD inline
#include <cstdint>

#include <cuda_runtime.h> // vector types only

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

// ---- host stand-ins for the device intrinsics rtfs_core.cuh uses ----
static inline float __uint_as_float(uint32_t u) { float f; std::memcpy(&f, &u, 4); return f; }
static inline float __int_as_float(int i) { float f; std::memcpy(&f, &i, 4); return f; }
static inline double __longlong_as_double(long long i) { double f; std::memcpy(&f, &i, 8); return f; }
static inline uint32_t __float_as_uint(float f) { uint32_t u; std::memcpy(&u, &f, 4); return u; }
static inline uint32_t __umulhi(uint32_t a, uint32_t b) { return uint32_t((uint64_t(a) * uint64_t(b)) >> 32); }
static inline float __uint2float_rn(uint32_t w) { return float(w); }
static inline int __double2int_rn(double x) { return int(std::nearbyint(x)); }
static inline double __hiloint2double(int hi, int lo) {
    uint64_t u = (uint64_t(uint32_t(hi)) << 32) | uint32_t(lo);
    double d; std::memcpy(&d, &u, 8); return d;
}
template <class T> static inline T __ldg(const T *p) { return *p; }
static inline int min(int a, int b) { return a < b ? a : b; }
static inline int max(int a, int b) { return a > b ? a : b; }

struct HostTexels { const uint8_t *rgb; int w, h; };
static inline uint32_t fetch_texel(unsigned long long tex, int x, int y) {
    const HostTexels *t = reinterpret_cast<const HostTexels *>(tex);
    if (x < 0 || y < 0 || x >= t->w || y >= t->h) { std::fprintf(stderr, "fetch_texel: (%d, %d) outside %d x %d\n", x, y, t->w, t->h); std::abort(); }
    const uint8_t *p = t->rgb + 3 * (size_t(y) * t->w + x);
    return (uint32_t(p[0]) << 16) | (uint32_t(p[1]) << 8) | uint32_t(p[2]);
}
namespace rtfs { using ::fetch_texel; }

#include "../rtfs_core.cuh"

#include <memory>
#include <vector>

using namespace rtfs;

// the device half of the library is absent here: rt_scene_create is only ever called with device = -1
namespace rtfs {
int device_scene_upload(RtScene *) { return fail(RT_ERR_NO_DEVICE, "host debug build"); }
int device_scene_ensure_reference(RtScene *) { return RT_OK; }
int device_scene_ensure_wide(RtScene *) { return RT_OK; }
int device_scene_sync_layout(RtScene *) { return RT_OK; }
void device_scene_free(RtScene *) {}
size_t device_scene_bytes(const RtScene *) { return 0; }
} // namespace rtfs

namespace {
struct HostScene {
    RtScene *scene = nullptr;
    std::vector<DTexture> tex;
    std::vector<HostTexels> texels;
    // exact-size copies, so that ASan sees an overrun by one element
    std::unique_ptr<uint4[]> nodes, mats, wide_nodes;
    std::unique_ptr<float4[]> spheres, wide_spheres;
    std::unique_ptr<DUnbounded[]> unb;
    std::unique_ptr<int32_t[]> w2d, d2w;
    SceneGlobal g{};
};
template <class T, class S>
std::unique_ptr<T[]> exact_copy(const std::vector<S> &v) {
    const size_t bytes = v.size() * sizeof(S);
    std::unique_ptr<T[]> p(new T[bytes / sizeof(T) ? bytes / sizeof(T) : 0]);
    if (bytes) std::memcpy(p.get(), v.data(), bytes);
    return p;
}
int build(HostScene &hs, const RtHittable *objects, int n_objects, const RtTexture *textures, int n_textures, int wide) {
    int rc = rt_scene_create(objects, n_objects, textures, n_textures, -1, &hs.scene);
    if (rc != RT_OK) return rc;
    HostSceneLayout &L = hs.scene->layout;
    if (wide) build_wide_layout(L);
    hs.texels.resize(n_textures);
    hs.tex.resize(n_textures);
    for (int i = 0; i < n_textures; ++i) {
        const RtTexture &t = hs.scene->textures[i];
        DTexture &o = hs.tex[i];
        std::memset(&o, 0, sizeof o);
        o.kind = t.kind;
        o.rgb = (uint32_t(t.colour[0]) << 16) | (uint32_t(t.colour[1]) << 8) | uint32_t(t.colour[2]);
        o.w = t.width; o.h = t.height; o.even = t.even; o.odd = t.odd;
        o.grid = float(t.grid_size);
        o.cx = float(t.map_centre[0]); o.cy = float(t.map_centre[1]); o.cz = float(t.map_centre[2]);
        o.inv_radius = float(1.0 / (t.map_radius != 0.0 ? t.map_radius : 1.0));
        hs.texels[i] = HostTexels{t.rgb8, t.width, t.height};
        o.tex = reinterpret_cast<unsigned long long>(&hs.texels[i]);
    }
    std::vector<DNode> dev_nodes(L.nodes.size());
    for (size_t i = 0; i < L.nodes.size(); ++i) dev_nodes[i] = device_node_of(L.nodes[i]); // what device_scene_upload does
    hs.nodes = exact_copy<uint4>(dev_nodes);
    hs.spheres = exact_copy<float4>(L.spheres);
    hs.mats = exact_copy<uint4>(L.materials);
    hs.unb.reset(new DUnbounded[L.unbounded.size()]);
    std::copy(L.unbounded.begin(), L.unbounded.end(), hs.unb.get());
    hs.wide_nodes = exact_copy<uint4>(L.wide_nodes);
    hs.wide_spheres = exact_copy<float4>(L.wide_spheres);
    hs.w2d = exact_copy<int32_t>(L.wide_to_dev);
    hs.d2w = exact_copy<int32_t>(L.dev_to_wide);
    hs.g.nodes = hs.nodes.get();
    hs.g.spheres = hs.spheres.get();
    hs.g.mats = hs.mats.get();
    hs.g.unb = hs.unb.get();
    hs.g.tex = hs.tex.data();
    hs.g.n_nodes = int32_t(L.nodes.size());
    hs.g.n_bounded = L.n_bounded;
    hs.g.n_unbounded = int32_t(L.unbounded.size());
    hs.g.n_tex = n_textures;
    hs.g.wide_nodes = hs.wide_nodes.get();
    hs.g.wide_spheres = hs.wide_spheres.get();
    hs.g.wide_to_dev = hs.w2d.get();
    hs.g.dev_to_wide = hs.d2w.get();
    return RT_OK;
}

DevCamera dev_camera(const RtCamera &c, int max_w, int max_h) { // = make_dev_camera (rtfs_device.h)
    DevCamera d{};
    d.ox = float(c.view_origin[0]); d.oy = float(c.view_origin[1]); d.oz = float(c.view_origin[2]);
    d.cx = float(c.xaxis_origin[0] - c.view_origin[0]);
    d.cy = float(c.xaxis_origin[1] - c.view_origin[1]);
    d.cz = float(c.xaxis_origin[2] - c.view_origin[2]);
    d.xx = float(c.xaxis_dir[0]); d.xy = float(c.xaxis_dir[1]); d.xz = float(c.xaxis_dir[2]);
    d.yx = float(c.yaxis_dir[0]); d.yy = float(c.yaxis_dir[1]); d.yz = float(c.yaxis_dir[2]);
    d.sx = float(c.viewport_width / double(max_w));
    d.sy = float(c.viewport_height / double(max_h));
    d.max_w = max_w; d.max_h = max_h;
    d.rows = 2 * max_h + 1; d.cols = 2 * max_w + 1;
    d.spp = c.samples_per_pixel; d.depth = c.bounce_depth;
    return d;
}

// optional trace of the work per ray (slab tests, primitive tests), path by path: feeds the warp-scheduling
// simulations under profiles/ (how much of a warp's time is lost to the longest walk of its 32 lanes)
std::vector<uint32_t> *g_ray_log = nullptr;
std::vector<float> *g_ray_geometry = nullptr; // with it: origin, direction and bounce index of every logged ray (7 floats)

template <bool WIDE>
uint32_t trace_one(const SceneAccess<false> &sc, const DevCamera &cam, uint64_t seed, int r, int c, uint32_t sample, uint64_t &rays) {
    PathState ps;
    uint32_t result = kBlack;
    TraversalCounters cn{0, 0};
    LocalStack stack;
    if (!path_begin(ps, cam, uint32_t(seed), uint32_t(seed >> 32), r, c, sample)) return kBlack;
    for (;;) {
        ++rays;
        const TraversalCounters before = cn;
        if (g_ray_geometry) g_ray_geometry->insert(g_ray_geometry->end(), {ps.o.x, ps.o.y, ps.o.z, ps.d.x, ps.d.y, ps.d.z, float(ps.bounces)});
        const bool done = path_step<false, true, LocalStack, WIDE>(ps, sc, cam.depth, result, cn, 1u, stack);
        if (g_ray_log) g_ray_log->push_back(((cn.box_tests - before.box_tests) << 8) | ((cn.prim_tests - before.prim_tests) & 255u) | (done ? 0x80000000u : 0u));
        if (done) break;
    }
    return result;
}
} // namespace

extern "C" {

// One frame, scalar: renderPixel's three loops (Scene.fs:157-194) with the device's sample numbering, so that the sums
// are the ones the kernels produce (up to MUFU / FMA rounding).  sums_out: rows*cols*4 int32; rgb_out: rows*cols*3.
int dbg_render(const RtHittable *objects, int n_objects, const RtTexture *textures, int n_textures, const RtCamera *camera, int max_w, int max_h,
               uint64_t seed, int adaptive, int wide, uint8_t *rgb_out, int32_t *sums_out, uint64_t *rays_out) {
    HostScene hs;
    int rc = build(hs, objects, n_objects, textures, n_textures, wide);
    if (rc != RT_OK) return rc;
    SceneAccess<false> sc;
    sc.g = hs.g;
    sc.s_nodes = sc.s_spheres = sc.s_mats = 0;
    const DevCamera cam = dev_camera(*camera, max_w, max_h);
    const int spp = camera->samples_per_pixel;
    const int first_trial = std::min(5, spp / 2), n_probe = 2 * first_trial + 1;
    uint64_t rays = 0;
    for (int r = 0; r < cam.rows; ++r)
        for (int c = 0; c < cam.cols; ++c) {
            int32_t s[4] = {0, 0, 0, 0};
            auto add = [&](uint32_t sample) {
                uint32_t px = wide ? trace_one<true>(sc, cam, seed, r, c, sample, rays) : trace_one<false>(sc, cam, seed, r, c, sample, rays);
                s[0] += int((px >> 16) & 255u); s[1] += int((px >> 8) & 255u); s[2] += int(px & 255u); s[3] += 1;
            };
            if (adaptive) {
                for (int j = 0; j <= first_trial; ++j) add(uint32_t(j));
                int32_t old[3] = {s[0] / s[3], s[1] / s[3], s[2] / s[3]};
                for (int j = first_trial + 1; j < n_probe; ++j) add(uint32_t(j));
                int diff = std::abs(s[0] / s[3] - old[0]) + std::abs(s[1] / s[3] - old[1]) + std::abs(s[2] / s[3] - old[2]);
                if (diff != 0)
                    for (int j = n_probe; j < std::max(n_probe, spp); ++j) add(uint32_t(j));
            } else {
                for (int j = 0; j < spp; ++j) add(uint32_t(j));
            }
            const size_t p = size_t(r) * cam.cols + c;
            for (int k = 0; k < 4; ++k) sums_out[4 * p + k] = s[k];
            for (int k = 0; k < 3; ++k) rgb_out[3 * p + k] = uint8_t(s[k] / (s[3] > 0 ? s[3] : 1));
        }
    if (rays_out) *rays_out = rays;
    rt_scene_destroy(hs.scene);
    return RT_OK;
}

// dbg_render with a log of the work of every ray: log_out[i] = box tests << 8 | primitive tests, bit 31 = last ray of its path
int dbg_render_logged(const RtHittable *objects, int n_objects, const RtTexture *textures, int n_textures, const RtCamera *camera, int max_w,
                      int max_h, uint64_t seed, int adaptive, int wide, uint8_t *rgb_out, int32_t *sums_out, uint32_t *log_out, uint64_t log_cap,
                      uint64_t *log_len) {
    std::vector<uint32_t> log;
    g_ray_log = &log;
    uint64_t rays = 0;
    int rc = dbg_render(objects, n_objects, textures, n_textures, camera, max_w, max_h, seed, adaptive, wide, rgb_out, sums_out, &rays);
    g_ray_log = nullptr;
    *log_len = log.size();
    std::memcpy(log_out, log.data(), sizeof(uint32_t) * std::min<uint64_t>(log_cap, log.size()));
    return rc;
}

// dbg_render_logged plus the geometry of every ray (7 floats per ray: origin, direction, bounce index), for the experiments
// under profiles/ that ask how well a ray's walk length can be predicted before the walk
int dbg_render_logged_geometry(const RtHittable *objects, int n_objects, const RtTexture *textures, int n_textures, const RtCamera *camera,
                               int max_w, int max_h, uint64_t seed, int adaptive, uint8_t *rgb_out, int32_t *sums_out, uint32_t *log_out,
                               float *geometry_out, uint64_t log_cap, uint64_t *log_len) {
    std::vector<float> geometry;
    g_ray_geometry = &geometry;
    int rc = dbg_render_logged(objects, n_objects, textures, n_textures, camera, max_w, max_h, seed, adaptive, 0, rgb_out, sums_out, log_out, log_cap,
                               log_len);
    g_ray_geometry = nullptr;
    std::memcpy(geometry_out, geometry.data(), sizeof(float) * 7 * std::min<uint64_t>(log_cap, geometry.size() / 7));
    return rc;
}

// The order of node visits ('I') and leaf visits ('L') of every ray of a frame, rays separated by '.', for the warp
// simulations under profiles/ (what batching the leaf visits of a warp would buy).  Walks the binary tree exactly as
// bvh_closest does, visit by visit.
int dbg_visit_trace(const RtHittable *objects, int n_objects, const RtTexture *textures, int n_textures, const RtCamera *camera, int max_w,
                    int max_h, uint64_t seed, int spp, char *out, uint64_t cap, uint64_t *len) {
    HostScene hs;
    int rc = build(hs, objects, n_objects, textures, n_textures, 0);
    if (rc != RT_OK) return rc;
    SceneAccess<false> sc;
    sc.g = hs.g;
    sc.s_nodes = sc.s_spheres = sc.s_mats = 0;
    const DevCamera cam = dev_camera(*camera, max_w, max_h);
    uint64_t n = 0;
    auto emit = [&](char c) {
        if (n < cap) out[n] = c;
        ++n;
    };
    for (int r = 0; r < cam.rows; ++r)
        for (int c = 0; c < cam.cols; ++c)
            for (int j = 0; j < spp; ++j) {
                PathState ps;
                if (!path_begin(ps, cam, uint32_t(seed), uint32_t(seed >> 32), r, c, uint32_t(j))) continue;
                for (;;) {
                    TraversalCounters cn{0, 0};
                    LocalStack stack;
                    float best_t = kNoHitT;
                    int best_ref = kNoRef;
                    if (sc.g.n_bounded > 0) {
                        const RaySlabs rs = make_slabs(ps.o, ps.d);
                        int sp = 0, node = sc.root();
                        for (;;) {
                            emit(node >= 0 ? 'I' : 'L');
                            if (bvh_visit<false, true>(sc, rs, ps.o, ps.d, ps.last, node, sp, stack, best_t, best_ref, cn)) break;
                        }
                    }
                    emit('.');
                    Hit h = finish_hit<false, true>(sc, ps.o, ps.d, ps.last, best_t, best_ref, cn);
                    uint32_t result;
                    if (path_after_hit<false>(ps, sc, h, cam.depth, result)) break;
                }
                emit('/'); // end of path
            }
    *len = n;
    rt_scene_destroy(hs.scene);
    return RT_OK;
}

// hitObject through both trees for explicit rays: prim_out = index into the caller's Hittable array, or -1
int dbg_hit_object(const RtHittable *objects, int n_objects, int wide, int n, const float *o, const float *d, int32_t *prim_out, float *t_out) {
    HostScene hs;
    int rc = build(hs, objects, n_objects, nullptr, 0, wide);
    if (rc != RT_OK) return rc;
    SceneAccess<false> sc;
    sc.g = hs.g;
    sc.s_nodes = sc.s_spheres = sc.s_mats = 0;
    const DMaterial *mats = reinterpret_cast<const DMaterial *>(hs.mats.get());
    for (int i = 0; i < n; ++i) {
        TraversalCounters cn{0, 0};
        float3 ro = f3(o[3 * i], o[3 * i + 1], o[3 * i + 2]), rd = f3(d[3 * i], d[3 * i + 1], d[3 * i + 2]);
        Hit h = wide ? closest_hit<false, true, true>(sc, ro, rd, kNoPrim, cn, 1u) : closest_hit<false, true, false>(sc, ro, rd, kNoPrim, cn, 1u);
        prim_out[i] = h.prim == kNoPrim ? -1 : mats[h.prim].host_index;
        t_out[i] = h.t;
    }
    rt_scene_destroy(hs.scene);
    return RT_OK;
}

// deliberately walks off the end of the traversal stack: the bounds assert (or ASan) must stop the process
int dbg_stack_overflow(int entries) {
    LocalStack stack;
    for (int i = 0; i < entries; ++i) stack.put(i, i);
    int sum = 0;
    for (int i = 0; i < entries; ++i) sum += stack.get(i);
    return sum;
}

} // extern "C"
