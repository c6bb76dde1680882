// rtfs_conformance.cu — per-primitive conformance entry points (rt_test_*) and the FP32 FMA
// microbenchmark.  Each kernel runs one thread per test vector through exactly the __device__
// function of rtfs_core.cuh that the render kernels execute.  Inputs and outputs are host arrays of
// doubles (the reference's types); they are rounded to FP32 on upload where the device works in FP32.
#include "rtfs_device.h"

#include <cstring>
#include <vector>

namespace rtfs {
namespace {

template <class T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    ~DevBuf() { cudaFree(p); }
    int alloc(size_t count) {
        n = count;
        RT_CUDA(cudaMalloc((void **)&p, std::max<size_t>(count, 1) * sizeof(T)));
        return RT_OK;
    }
    int put(const std::vector<T> &h) {
        int rc = alloc(h.size());
        if (rc != RT_OK) return rc;
        if (!h.empty()) RT_CUDA(cudaMemcpy(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
        return RT_OK;
    }
    int get(std::vector<T> &h) const {
        h.resize(n);
        if (n) RT_CUDA(cudaMemcpy(h.data(), p, n * sizeof(T), cudaMemcpyDeviceToHost));
        return RT_OK;
    }
};

std::vector<float> to_f32(const double *src, size_t n) {
    std::vector<float> v(n);
    for (size_t i = 0; i < n; ++i) v[i] = float(src[i]);
    return v;
}
#define RT_TRY(expr)              \
    do {                          \
        int rc__ = (expr);        \
        if (rc__ != RT_OK) return rc__; \
    } while (0)

inline int finish_launch() {
    RT_CUDA(cudaGetLastError());
    RT_CUDA(cudaDeviceSynchronize());
    return RT_OK;
}
inline unsigned grid_for(int n) { return unsigned((n + 127) / 128); }

__device__ __forceinline__ float3 ld3(const float *p, int i) { return f3(p[3 * i], p[3 * i + 1], p[3 * i + 2]); }
__device__ __forceinline__ void st3(float *p, int i, float3 v) {
    p[3 * i] = v.x;
    p[3 * i + 1] = v.y;
    p[3 * i + 2] = v.z;
}

__global__ void k_sphere_hit(int n, const float *o, const float *d, const float *c, const float *r, float *t_out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float t;
    float3 cc = ld3(c, i);
    bool hit = sphere_hit(ld3(o, i), ld3(d, i), make_float4(cc.x, cc.y, cc.z, r[i]), false, t);
    t_out[i] = hit ? t : CUDART_NAN_F;
}
__global__ void k_plane_hit(int n, const float *o, const float *d, const double *p, const float *nrm, float *t_out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    DUnbounded u;
    u.p[0] = p[3 * i]; u.p[1] = p[3 * i + 1]; u.p[2] = p[3 * i + 2];
    u.n[0] = nrm[3 * i]; u.n[1] = nrm[3 * i + 1]; u.n[2] = nrm[3 * i + 2];
    u.shape = RT_SHAPE_INFINITE_PLANE;
    // classify_unbounded's rule for planes (rtfs_host.cpp), so that each vector takes the path a scene object would
    const double k = double(u.n[0]) * u.p[0] + double(u.n[1]) * u.p[1] + double(u.n[2]) * u.p[2];
    u.fp32 = fabs(k) <= 16.0 ? 1 : 0;
    u.k = float(k);
    float t;
    bool hit = u.fp32 ? plane_hit_big_f32(ld3(o, i), ld3(d, i), u, false, t) : plane_hit_big(d3(ld3(o, i)), d3(ld3(d, i)), u, false, t);
    t_out[i] = hit ? t : CUDART_NAN_F;
}
__global__ void k_aabb_hit(int n, const float *o, const float *d, const float *mn, const float *mx, uint8_t *out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float a[3] = {mn[3 * i], mn[3 * i + 1], mn[3 * i + 2]}, b[3] = {mx[3 * i], mx[3 * i + 1], mx[3 * i + 2]};
    float3 dir = ld3(d, i);
    out[i] = aabb_hits_ref(inverse_directions(dir), ld3(o, i), a, b) ? 1 : 0;
}
__global__ void k_hit_object(SceneGlobal g, const DRefNode *ref_nodes, int n_ref, int traversal, int n, const float *o, const float *d,
                             int32_t *prim_out, float *t_out, float *strike_out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Hit h;
    if (traversal == 1) {
        h = closest_hit_reference(ref_nodes, n_ref, g, ld3(o, i), ld3(d, i), kNoPrim);
    } else {
        SceneAccess<false> sc;
        sc.g = g;
        sc.s_nodes = sc.s_spheres = sc.s_mats = 0;
        TraversalCounters cn{0, 0};
        if (traversal == 2)
            h = closest_hit<false, false, true>(sc, ld3(o, i), ld3(d, i), kNoPrim, cn, 1u << (threadIdx.x & 31));
        else
            h = closest_hit<false, false>(sc, ld3(o, i), ld3(d, i), kNoPrim, cn, 1u << (threadIdx.x & 31));
    }
    if (h.prim == kNoPrim) {
        prim_out[i] = -1;
        t_out[i] = CUDART_NAN_F;
        st3(strike_out, i, f3(0.f, 0.f, 0.f));
    } else {
        prim_out[i] = int32_t(__ldg(g.mats + 2 * h.prim + 1).w); // DMaterial.host_index
        t_out[i] = h.t;
        st3(strike_out, i, h.strike);
    }
}
__global__ void k_reflection(SceneGlobal g, int n, const int32_t *prim, const float *o, const float *d, const float *strike,
                             const uint8_t *colour_in, const float *uniforms, uint8_t *absorbed, uint8_t *colour_out, float *o_out,
                             float *d_out, uint8_t *inside_out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    SceneAccess<false> sc;
    sc.g = g;
    sc.s_nodes = sc.s_spheres = sc.s_mats = 0;
    ExplicitRng rng;
    for (int k = 0; k < 4; ++k) rng.u[k] = uniforms[4 * i + k];
    rng.rot = 0;
    float3 ro = ld3(o, i), rd = ld3(d, i);
    uint32_t colour = (uint32_t(colour_in[3 * i]) << 16) | (uint32_t(colour_in[3 * i + 1]) << 8) | uint32_t(colour_in[3 * i + 2]);
    bool inside = false;
    ScatterResult r = scatter(sc, prim[i], kNoPrim, ro, rd, ld3(strike, i), colour, rng, &inside);
    absorbed[i] = uint8_t(r);
    colour_out[3 * i] = uint8_t(colour >> 16);
    colour_out[3 * i + 1] = uint8_t(colour >> 8);
    colour_out[3 * i + 2] = uint8_t(colour);
    st3(o_out, i, ro);
    st3(d_out, i, rd);
    inside_out[i] = inside ? 1 : 0;
}
__global__ void k_camera_rays(DevCamera cam, int n, const int32_t *row, const int32_t *col, const float *r1, const float *r2, float *o_out,
                              float *d_out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float3 o, d = f3(CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F);
    camera_ray(cam, row[i], col[i], r1[i], r2[i], o, d);
    st3(o_out, i, o);
    st3(d_out, i, d);
}
__global__ void k_texture(SceneGlobal g, int n, const int32_t *prim, const float *point, uint8_t *colour_out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint4 b = __ldg(g.mats + 2 * prim[i] + 1);
    int tex = int(b.y);
    uint32_t c = tex < 0 ? (b.x & 0x00FFFFFFu) : texture_colour(g, tex, ld3(point, i));
    colour_out[3 * i] = uint8_t(c >> 16);
    colour_out[3 * i + 1] = uint8_t(c >> 8);
    colour_out[3 * i + 2] = uint8_t(c);
}
__global__ void k_combine_darken(int n, const uint8_t *a, const uint8_t *b, const double *albedo, uint8_t *out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t pa = (uint32_t(a[3 * i]) << 16) | (uint32_t(a[3 * i + 1]) << 8) | uint32_t(a[3 * i + 2]);
    uint32_t pb = (uint32_t(b[3 * i]) << 16) | (uint32_t(b[3 * i + 1]) << 8) | uint32_t(b[3 * i + 2]);
    uint32_t c = darken(albedo[i], combine(pa, pb));
    out[3 * i] = uint8_t(c >> 16);
    out[3 * i + 1] = uint8_t(c >> 8);
    out[3 * i + 2] = uint8_t(c);
}
__global__ void k_rng(uint32_t k0, uint32_t k1, int n, const uint32_t *pixel, const uint32_t *sample, const uint32_t *bounce,
                      const uint32_t *retry, uint32_t *words, float *uniforms) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint4 w = philox4x32_10(make_uint4(pixel[i], sample[i], bounce[i], retry[i]), k0, k1);
    words[4 * i] = w.x; words[4 * i + 1] = w.y; words[4 * i + 2] = w.z; words[4 * i + 3] = w.w;
    CounterRng rng{k0, k1, pixel[i], sample[i], bounce[i], retry[i]};
    float4 u = rng.next();
    uniforms[4 * i] = u.x; uniforms[4 * i + 1] = u.y; uniforms[4 * i + 2] = u.z; uniforms[4 * i + 3] = u.w;
}
__global__ void k_trace_samples(SceneGlobal g, DevCamera cam, uint32_t k0, uint32_t k1, int n, const int32_t *row_idx, const int32_t *col_idx,
                                const int32_t *sample, uint8_t *colour_out, int32_t *rays_out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    SceneAccess<false> sc;
    sc.g = g;
    sc.s_nodes = sc.s_spheres = sc.s_mats = 0;
    PathState ps;
    uint32_t result = kBlack;
    int rays = 0;
    TraversalCounters cn{0, 0};
    LocalStack stack;
    if (path_begin(ps, cam, k0, k1, row_idx[i], col_idx[i], uint32_t(sample[i]))) {
        for (;;) {
            ++rays;
            if (path_step<false, false>(ps, sc, cam.depth, result, cn, 1u << (threadIdx.x & 31), stack)) break; // lanes run independently here
        }
    }
    colour_out[3 * i] = uint8_t(result >> 16);
    colour_out[3 * i + 1] = uint8_t(result >> 8);
    colour_out[3 * i + 2] = uint8_t(result);
    rays_out[i] = rays;
}

// Dependent FFMA chains, 8 per thread: the measured FP32 FMA peak used as the roofline denominator.
__global__ void __launch_bounds__(256) k_fma_peak(float *sink, int iters, float a, float b) {
    float x0 = threadIdx.x * 1e-3f, x1 = x0 + 1.f, x2 = x0 + 2.f, x3 = x0 + 3.f, x4 = x0 + 4.f, x5 = x0 + 5.f, x6 = x0 + 6.f, x7 = x0 + 7.f;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
            x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
        }
    }
    float s = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
    if (s == 123.456f) sink[0] = s;
}

int scene_device(RtScene *scene, DeviceScene **out) {
    if (!scene) return fail(RT_ERR_INVALID_ARGUMENT, "null scene");
    if (!scene->dev) return fail(RT_ERR_NO_DEVICE, "the scene was created without a device (device = -1); there is no CPU fallback");
    *out = static_cast<DeviceScene *>(scene->dev);
    RT_CUDA(cudaSetDevice((*out)->device));
    return device_scene_sync_layout(scene); // after a rebuild: the device ids the primitive indices map to
}

int map_prims(const RtScene *scene, int n, const int32_t *prim, std::vector<int32_t> &out) {
    out.resize(n);
    for (int i = 0; i < n; ++i) {
        if (prim[i] < 0 || prim[i] >= int32_t(scene->objects.size())) return fail(RT_ERR_INVALID_ARGUMENT, "primitive index out of range");
        int32_t id = scene->layout.device_id_of[prim[i]];
        if (id < 0)
            return fail(RT_ERR_INVALID_ARGUMENT,
                        "primitive is a bounded sphere with negative radius: its box is inverted and the reference can never hit it (F16)");
        out[i] = id;
    }
    return RT_OK;
}

} // namespace
} // namespace rtfs

using namespace rtfs;

extern "C" {

int rt_test_sphere_hit(int32_t device, int32_t n, const double *origin, const double *dir, const double *centre, const double *radius,
                       double *t_out) {
    RT_TRY(require_device(device));
    if (n < 0 || !origin || !dir || !centre || !radius || !t_out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_test_sphere_hit: bad argument");
    DevBuf<float> o, d, c, r, t;
    RT_TRY(o.put(to_f32(origin, 3 * size_t(n))));
    RT_TRY(d.put(to_f32(dir, 3 * size_t(n))));
    RT_TRY(c.put(to_f32(centre, 3 * size_t(n))));
    RT_TRY(r.put(to_f32(radius, size_t(n))));
    RT_TRY(t.alloc(n));
    if (n) k_sphere_hit<<<grid_for(n), 128>>>(n, o.p, d.p, c.p, r.p, t.p);
    RT_TRY(finish_launch());
    std::vector<float> h;
    RT_TRY(t.get(h));
    for (int i = 0; i < n; ++i) t_out[i] = double(h[i]);
    return RT_OK;
}

int rt_test_plane_hit(int32_t device, int32_t n, const double *origin, const double *dir, const double *point, const double *normal,
                      double *t_out) {
    RT_TRY(require_device(device));
    if (n < 0 || !origin || !dir || !point || !normal || !t_out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_test_plane_hit: bad argument");
    DevBuf<float> o, d, nr, t;
    DevBuf<double> p;
    RT_TRY(o.put(to_f32(origin, 3 * size_t(n))));
    RT_TRY(d.put(to_f32(dir, 3 * size_t(n))));
    RT_TRY(nr.put(to_f32(normal, 3 * size_t(n))));
    RT_TRY(p.put(std::vector<double>(point, point + 3 * size_t(n))));
    RT_TRY(t.alloc(n));
    if (n) k_plane_hit<<<grid_for(n), 128>>>(n, o.p, d.p, p.p, nr.p, t.p);
    RT_TRY(finish_launch());
    std::vector<float> h;
    RT_TRY(t.get(h));
    for (int i = 0; i < n; ++i) t_out[i] = double(h[i]);
    return RT_OK;
}

int rt_test_aabb_hit(int32_t device, int32_t n, const double *origin, const double *dir, const double *box_min, const double *box_max,
                     uint8_t *hit_out) {
    RT_TRY(require_device(device));
    if (n < 0 || !origin || !dir || !box_min || !box_max || !hit_out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_test_aabb_hit: bad argument");
    DevBuf<float> o, d, a, b;
    DevBuf<uint8_t> h;
    RT_TRY(o.put(to_f32(origin, 3 * size_t(n))));
    RT_TRY(d.put(to_f32(dir, 3 * size_t(n))));
    RT_TRY(a.put(to_f32(box_min, 3 * size_t(n))));
    RT_TRY(b.put(to_f32(box_max, 3 * size_t(n))));
    RT_TRY(h.alloc(n));
    if (n) k_aabb_hit<<<grid_for(n), 128>>>(n, o.p, d.p, a.p, b.p, h.p);
    RT_TRY(finish_launch());
    std::vector<uint8_t> out;
    RT_TRY(h.get(out));
    if (n) std::memcpy(hit_out, out.data(), n);
    return RT_OK;
}

int rt_test_hit_object(RtScene *scene, int32_t traversal, int32_t n, const double *origin, const double *dir, int32_t *prim_out,
                       double *t_out, double *strike_out) {
    DeviceScene *ds;
    RT_TRY(scene_device(scene, &ds));
    if (n < 0 || !origin || !dir || !prim_out || !t_out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_test_hit_object: bad argument");
    if (traversal < 0 || traversal > 2) return fail(RT_ERR_INVALID_ARGUMENT, "rt_test_hit_object: traversal must be 0, 1 or 2");
    if (traversal == 1) RT_TRY(device_scene_ensure_reference(scene));
    if (traversal == 2) RT_TRY(device_scene_ensure_wide(scene));
    DevBuf<float> o, d, t, s;
    DevBuf<int32_t> p;
    RT_TRY(o.put(to_f32(origin, 3 * size_t(n))));
    RT_TRY(d.put(to_f32(dir, 3 * size_t(n))));
    RT_TRY(t.alloc(n));
    RT_TRY(s.alloc(3 * size_t(n)));
    RT_TRY(p.alloc(n));
    if (n) k_hit_object<<<grid_for(n), 128>>>(ds->g, ds->ref_nodes, ds->n_ref_nodes, traversal, n, o.p, d.p, p.p, t.p, s.p);
    RT_TRY(finish_launch());
    std::vector<float> ht, hs;
    std::vector<int32_t> hp;
    RT_TRY(t.get(ht));
    RT_TRY(s.get(hs));
    RT_TRY(p.get(hp));
    for (int i = 0; i < n; ++i) {
        prim_out[i] = hp[i];
        t_out[i] = double(ht[i]);
        if (strike_out)
            for (int k = 0; k < 3; ++k) strike_out[3 * i + k] = double(hs[3 * i + k]);
    }
    return RT_OK;
}

int rt_test_reflection(RtScene *scene, int32_t n, const int32_t *prim, const double *origin, const double *dir, const double *strike,
                       const uint8_t *colour_in, const double *uniforms, uint8_t *absorbed_out, uint8_t *colour_out, double *origin_out,
                       double *dir_out, uint8_t *inside_out) {
    DeviceScene *ds;
    RT_TRY(scene_device(scene, &ds));
    if (n < 0 || !prim || !origin || !dir || !strike || !colour_in || !uniforms || !absorbed_out || !colour_out || !origin_out || !dir_out)
        return fail(RT_ERR_INVALID_ARGUMENT, "rt_test_reflection: bad argument");
    std::vector<int32_t> ids;
    RT_TRY(map_prims(scene, n, prim, ids));
    DevBuf<int32_t> p;
    DevBuf<float> o, d, s, u, oo, dd;
    DevBuf<uint8_t> ci, ab, co, in;
    RT_TRY(p.put(ids));
    RT_TRY(o.put(to_f32(origin, 3 * size_t(n))));
    RT_TRY(d.put(to_f32(dir, 3 * size_t(n))));
    RT_TRY(s.put(to_f32(strike, 3 * size_t(n))));
    RT_TRY(u.put(to_f32(uniforms, 4 * size_t(n))));
    RT_TRY(ci.put(std::vector<uint8_t>(colour_in, colour_in + 3 * size_t(n))));
    RT_TRY(ab.alloc(n));
    RT_TRY(co.alloc(3 * size_t(n)));
    RT_TRY(in.alloc(n));
    RT_TRY(oo.alloc(3 * size_t(n)));
    RT_TRY(dd.alloc(3 * size_t(n)));
    if (n) k_reflection<<<grid_for(n), 128>>>(ds->g, n, p.p, o.p, d.p, s.p, ci.p, u.p, ab.p, co.p, oo.p, dd.p, in.p);
    RT_TRY(finish_launch());
    std::vector<uint8_t> hab, hco, hin;
    std::vector<float> hoo, hdd;
    RT_TRY(ab.get(hab));
    RT_TRY(co.get(hco));
    RT_TRY(in.get(hin));
    RT_TRY(oo.get(hoo));
    RT_TRY(dd.get(hdd));
    for (int i = 0; i < n; ++i) {
        absorbed_out[i] = hab[i];
        if (inside_out) inside_out[i] = hin[i];
        for (int k = 0; k < 3; ++k) {
            colour_out[3 * i + k] = hco[3 * i + k];
            origin_out[3 * i + k] = double(hoo[3 * i + k]);
            dir_out[3 * i + k] = double(hdd[3 * i + k]);
        }
    }
    return RT_OK;
}

int rt_test_camera_rays(int32_t device, const RtCamera *camera, int32_t max_w, int32_t max_h, int32_t n, const int32_t *row,
                        const int32_t *col, const double *rand1, const double *rand2, double *origin_out, double *dir_out) {
    RT_TRY(require_device(device));
    if (!camera || max_w <= 0 || max_h <= 0 || n < 0 || !row || !col || !rand1 || !rand2 || !origin_out || !dir_out)
        return fail(RT_ERR_INVALID_ARGUMENT, "rt_test_camera_rays: bad argument");
    DevBuf<int32_t> r, c;
    DevBuf<float> r1, r2, o, d;
    RT_TRY(r.put(std::vector<int32_t>(row, row + n)));
    RT_TRY(c.put(std::vector<int32_t>(col, col + n)));
    RT_TRY(r1.put(to_f32(rand1, n)));
    RT_TRY(r2.put(to_f32(rand2, n)));
    RT_TRY(o.alloc(3 * size_t(n)));
    RT_TRY(d.alloc(3 * size_t(n)));
    if (n) k_camera_rays<<<grid_for(n), 128>>>(make_dev_camera(*camera, max_w, max_h), n, r.p, c.p, r1.p, r2.p, o.p, d.p);
    RT_TRY(finish_launch());
    std::vector<float> ho, hd;
    RT_TRY(o.get(ho));
    RT_TRY(d.get(hd));
    for (size_t i = 0; i < 3 * size_t(n); ++i) {
        origin_out[i] = double(ho[i]);
        dir_out[i] = double(hd[i]);
    }
    return RT_OK;
}

int rt_test_texture(RtScene *scene, int32_t n, const int32_t *prim, const double *point, uint8_t *colour_out) {
    DeviceScene *ds;
    RT_TRY(scene_device(scene, &ds));
    if (n < 0 || !prim || !point || !colour_out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_test_texture: bad argument");
    std::vector<int32_t> ids;
    RT_TRY(map_prims(scene, n, prim, ids));
    DevBuf<int32_t> p;
    DevBuf<float> pt;
    DevBuf<uint8_t> co;
    RT_TRY(p.put(ids));
    RT_TRY(pt.put(to_f32(point, 3 * size_t(n))));
    RT_TRY(co.alloc(3 * size_t(n)));
    if (n) k_texture<<<grid_for(n), 128>>>(ds->g, n, p.p, pt.p, co.p);
    RT_TRY(finish_launch());
    std::vector<uint8_t> h;
    RT_TRY(co.get(h));
    if (n) std::memcpy(colour_out, h.data(), 3 * size_t(n));
    return RT_OK;
}

int rt_test_combine_darken(int32_t device, int32_t n, const uint8_t *a, const uint8_t *b, const double *albedo, uint8_t *out) {
    RT_TRY(require_device(device));
    if (n < 0 || !a || !b || !albedo || !out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_test_combine_darken: bad argument");
    DevBuf<uint8_t> da, db, dout;
    DevBuf<double> dal;
    RT_TRY(da.put(std::vector<uint8_t>(a, a + 3 * size_t(n))));
    RT_TRY(db.put(std::vector<uint8_t>(b, b + 3 * size_t(n))));
    RT_TRY(dal.put(std::vector<double>(albedo, albedo + n)));
    RT_TRY(dout.alloc(3 * size_t(n)));
    if (n) k_combine_darken<<<grid_for(n), 128>>>(n, da.p, db.p, dal.p, dout.p);
    RT_TRY(finish_launch());
    std::vector<uint8_t> h;
    RT_TRY(dout.get(h));
    if (n) std::memcpy(out, h.data(), 3 * size_t(n));
    return RT_OK;
}

int rt_test_rng(int32_t device, uint64_t seed, int32_t n, const uint32_t *pixel, const uint32_t *sample, const uint32_t *bounce,
                const uint32_t *retry, uint32_t *words_out, double *uniforms_out) {
    RT_TRY(require_device(device));
    if (n < 0 || !pixel || !sample || !bounce || !retry || !words_out || !uniforms_out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_test_rng: bad argument");
    DevBuf<uint32_t> p, s, b, r, w;
    DevBuf<float> u;
    RT_TRY(p.put(std::vector<uint32_t>(pixel, pixel + n)));
    RT_TRY(s.put(std::vector<uint32_t>(sample, sample + n)));
    RT_TRY(b.put(std::vector<uint32_t>(bounce, bounce + n)));
    RT_TRY(r.put(std::vector<uint32_t>(retry, retry + n)));
    RT_TRY(w.alloc(4 * size_t(n)));
    RT_TRY(u.alloc(4 * size_t(n)));
    if (n) k_rng<<<grid_for(n), 128>>>(uint32_t(seed), uint32_t(seed >> 32), n, p.p, s.p, b.p, r.p, w.p, u.p);
    RT_TRY(finish_launch());
    std::vector<uint32_t> hw;
    std::vector<float> hu;
    RT_TRY(w.get(hw));
    RT_TRY(u.get(hu));
    for (size_t i = 0; i < 4 * size_t(n); ++i) {
        words_out[i] = hw[i];
        uniforms_out[i] = double(hu[i]);
    }
    return RT_OK;
}

int rt_test_trace_samples(RtScene *scene, const RtCamera *camera, int32_t max_w, int32_t max_h, uint64_t seed, int32_t n,
                          const int32_t *row_idx, const int32_t *col_idx, const int32_t *sample, uint8_t *colour_out, int32_t *rays_out) {
    DeviceScene *ds;
    RT_TRY(scene_device(scene, &ds));
    if (!camera || max_w <= 0 || max_h <= 0 || n < 0 || !row_idx || !col_idx || !sample || !colour_out)
        return fail(RT_ERR_INVALID_ARGUMENT, "rt_test_trace_samples: bad argument");
    DevBuf<int32_t> r, c, s, rays;
    DevBuf<uint8_t> co;
    RT_TRY(r.put(std::vector<int32_t>(row_idx, row_idx + n)));
    RT_TRY(c.put(std::vector<int32_t>(col_idx, col_idx + n)));
    RT_TRY(s.put(std::vector<int32_t>(sample, sample + n)));
    RT_TRY(rays.alloc(n));
    RT_TRY(co.alloc(3 * size_t(n)));
    if (n)
        k_trace_samples<<<grid_for(n), 128>>>(ds->g, make_dev_camera(*camera, max_w, max_h), uint32_t(seed), uint32_t(seed >> 32), n, r.p, c.p, s.p,
                                              co.p, rays.p);
    RT_TRY(finish_launch());
    std::vector<uint8_t> h;
    std::vector<int32_t> hr;
    RT_TRY(co.get(h));
    RT_TRY(rays.get(hr));
    if (n) std::memcpy(colour_out, h.data(), 3 * size_t(n));
    if (rays_out)
        for (int i = 0; i < n; ++i) rays_out[i] = hr[i];
    return RT_OK;
}

int rt_measure_fp32_peak(int32_t device, double *tflops_out) {
    RT_TRY(require_device(device));
    if (!tflops_out) return fail(RT_ERR_INVALID_ARGUMENT, "rt_measure_fp32_peak: null output");
    cudaDeviceProp prop;
    RT_CUDA(cudaGetDeviceProperties(&prop, device));
    DevBuf<float> sink;
    RT_TRY(sink.alloc(1));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    cudaEvent_t e0, e1;
    RT_CUDA(cudaEventCreate(&e0));
    RT_CUDA(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0);
        k_fma_peak<<<blocks, threads>>>(sink.p, iters, 1.0000001f, 1e-7f);
        cudaEventRecord(e1);
        if (cudaEventSynchronize(e1) != cudaSuccess) break;
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        double flops = double(blocks) * threads * double(iters) * 16.0 * 8.0 * 2.0;
        if (rep > 0 && ms > 0.f) best = std::max(best, flops / (double(ms) * 1e-3) / 1e12);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    RT_CUDA(cudaGetLastError());
    *tflops_out = best;
    return RT_OK;
}

} // extern "C"
