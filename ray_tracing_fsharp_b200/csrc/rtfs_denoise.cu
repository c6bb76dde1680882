// rtfs_denoise.cu — denoised previews of progressive frames (rt_frame_features, rt_frame_denoise in rtfs_frame.cu).
// features_kernel traces, for every pixel of a frame, the camera rays of its first F sample indices, exactly as the render
// kernels of the frame's kind start those paths, and keeps first-hit data: the caller's primitive hit by sample 0, the colour
// the first scatter leaves in a white path (the albedo), the shading normal and the hit distance.  The filter is an
// edge-avoiding a-trous wavelet (Dammertz et al., HPG 2010) whose colour weight is scaled by each pixel's own standard error
// (as SVGF scales it by its variance, Schied et al., HPG 2017), stopped at edges by those features.  It reads the frame's sums
// and Q and writes buffers of its own; nothing a pass reads or writes is touched.
// Every filter operation is an IEEE float32 + - x / with round-to-nearest written as an intrinsic (no contraction), over a
// fixed tap order, so tests/denoise_rule.py restates the filter bit for bit.  The formulas are in include/rtfs_b200.h.
#include "rtfs_device.h"

#include <cmath>

namespace rtfs {

constexpr int kFeatureThreads = 128; // each thread holds a walk stack of kLocalStackWords words in local memory
constexpr int kFilterThreads = 256;

// One thread per frame pixel.  The pixel's camera, key, frame coordinates and RNG pixel word are the ones its paths take
// (path_begin for one frame; ViewPixels of rtfs_views.cu for a batch; WindowPixels of rtfs_window.cu for a window), so sample s
// here is the first segment of the path the frame traces for sample index s.  The tree is read from global memory through the
// binary SAH tree walk (closest_hit, as rt_test_hit_object with traversal 0); the first scatter is scatter itself with a white
// colour, and the generator of bounce 1, although the colour and the normal do not depend on its draws.
__global__ void __launch_bounds__(kFeatureThreads) features_kernel(const FrameParams fp, size_t n_pixels, int samples, FrameFeatures out) {
    const size_t p = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (p >= n_pixels) return;
    int r = int(p / size_t(fp.cam.cols)), c = int(p - size_t(r) * size_t(fp.cam.cols));
    DevCamera cam = fp.cam;
    uint32_t k0 = fp.k0, k1 = fp.k1, word = uint32_t(p);
    if (fp.views) { // view v of the tall frame: its camera and key, its pixel within the view
        const int v = int(p / size_t(fp.view_pixels)), q = int(p) - v * fp.view_pixels;
        cam = fp.views[v].cam;
        k0 = fp.views[v].k0;
        k1 = fp.views[v].k1;
        r = q / fp.cam.cols;
        c = q - r * fp.cam.cols;
        word = uint32_t(q);
    } else if (fp.window) { // the window's pixel at its place in the frame, and the frame's pixel word
        r += fp.win_row0;
        c += fp.win_col0;
        word = uint32_t(r * (2 * fp.cam.max_w + 1) + c);
    }
    SceneAccess<0> sc;
    sc.g = fp.g;
    sc.s_nodes = sc.s_spheres = sc.s_mats = 0;
    TraversalCounters cn{0, 0};
    const unsigned self = 1u << (threadIdx.x & 31);
    int32_t prim0 = -1;
    uint32_t ar = 0, ag = 0, ab = 0;
    int hits = 0;
    float nx = 0.f, ny = 0.f, nz = 0.f, t = 0.f;
    for (int s = 0; s < samples; ++s) {
        PathState ps;
        ps.rng = CounterRng{k0, k1, word, uint32_t(s), 0u, 0u};
        if (!path_start(ps, cam, r, c)) continue; // a camera ray the reference cannot make: no hit, black
        const Hit h = closest_hit<0, false>(sc, ps.o, ps.d, kNoPrim, cn, self);
        if (h.prim == kNoPrim) continue;
        if (s == 0) prim0 = int32_t(__ldg(fp.g.mats + 2 * h.prim + 1).w); // DMaterial.host_index
        ps.rng.bounce = 1u;
        ps.rng.retry = 0u;
        uint32_t colour = kWhite;
        float3 n = f3(0.f, 0.f, 0.f); // a scatter that fails before it has a normal adds nothing
        if (scatter(sc, h.prim, kNoPrim, ps.o, ps.d, h.strike, colour, ps.rng, nullptr, &n) == SCATTER_ERROR) colour = kBlack;
        ar += (colour >> 16) & 255u;
        ag += (colour >> 8) & 255u;
        ab += colour & 255u;
        nx = __fadd_rn(nx, n.x);
        ny = __fadd_rn(ny, n.y);
        nz = __fadd_rn(nz, n.z);
        t = __fadd_rn(t, h.t);
        ++hits;
    }
    out.prim[p] = prim0;
    out.albedo[3 * p] = uint8_t(ar / uint32_t(samples));
    out.albedo[3 * p + 1] = uint8_t(ag / uint32_t(samples));
    out.albedo[3 * p + 2] = uint8_t(ab / uint32_t(samples));
    const float fh = float(hits);
    out.normal[3 * p] = hits ? __fdiv_rn(nx, fh) : 0.f;
    out.normal[3 * p + 1] = hits ? __fdiv_rn(ny, fh) : 0.f;
    out.normal[3 * p + 2] = hits ? __fdiv_rn(nz, fh) : 0.f;
    out.depth[p] = hits ? __fdiv_rn(t, fh) : CUDART_INF_F;
}

// Level 0's input: per pixel (c_r, c_g, c_b, v) with c = float(T) / float(n) and v = float(E)^2, E as rt_frame_noise computes
// it; v = -1 marks a pixel without samples, which is output black and is no pixel's neighbour.
__global__ void __launch_bounds__(kFilterThreads) denoise_input_kernel(const int4 *stats, const unsigned long long *sq, size_t n_pixels,
                                                                       float4 *out) {
    const size_t p = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (p >= n_pixels) return;
    const int4 s = stats[p];
    if (s.w == 0) {
        out[p] = make_float4(0.f, 0.f, 0.f, -1.f);
        return;
    }
    const float n = __int2float_rn(s.w);
    const float e = __double2float_rn(pixel_standard_error(s.w, s.x, s.y, s.z, sq[p]));
    out[p] = make_float4(__fdiv_rn(__int2float_rn(s.x), n), __fdiv_rn(__int2float_rn(s.y), n), __fdiv_rn(__int2float_rn(s.z), n), __fmul_rn(e, e));
}

__device__ __forceinline__ float norm2(float a, float b, float c) {
    return __fadd_rn(__fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b)), __fmul_rn(c, c));
}
// the edge-stopping function w(x) = 1 / (1 + x (1 + x / 2)): exp(-x) to second order, 1 at x = 0, 0 at x = +inf
__device__ __forceinline__ float edge_weight(float x) {
    return __fdiv_rn(1.f, __fadd_rn(1.f, __fmul_rn(x, __fadd_rn(1.f, __fmul_rn(0.5f, x)))));
}

// One a-trous level: 5 x 5 taps at spacing `step`, B3-spline weights h = (1, 4, 6, 4, 1) (the 1/16 cancels in the
// normalisation), rows outer and columns inner.  A tap is skipped outside the frame, outside the pixel's view (view_rows rows
// each) and on a pixel without samples.  sc, sn, sa are this level's sigma_colour (halved per level), sigma_normal and
// sigma_albedo, squared here; sz is sigma_depth.
__global__ void __launch_bounds__(kFilterThreads) atrous_kernel(const float4 *__restrict__ in, float4 *__restrict__ out, FrameFeatures f,
                                                                size_t n_pixels, int view_rows, int cols, int step, float sc, float sn, float sa,
                                                                float sz) {
    const size_t p = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (p >= n_pixels) return;
    const float4 cp = __ldg(in + p);
    if (cp.w < 0.f) {
        out[p] = cp;
        return;
    }
    const float sc2 = __fmul_rn(sc, sc), sn2 = __fmul_rn(sn, sn), sa2 = __fmul_rn(sa, sa);
    const int r = int(p / size_t(cols)), c = int(p - size_t(r) * size_t(cols));
    const int v0 = r - r % view_rows;
    const float anr = float(__ldg(f.albedo + 3 * p)), ang = float(__ldg(f.albedo + 3 * p + 1)), anb = float(__ldg(f.albedo + 3 * p + 2));
    const float npx = __ldg(f.normal + 3 * p), npy = __ldg(f.normal + 3 * p + 1), npz = __ldg(f.normal + 3 * p + 2);
    const float zp = __ldg(f.depth + p);
    const float zscale = __fmul_rn(sz, zp);
    constexpr int kB3[5] = {1, 4, 6, 4, 1};
    float ws = 0.f, sr = 0.f, sg = 0.f, sb = 0.f;
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        const int rr = r + (j - 2) * step;
        if (rr < v0 || rr >= v0 + view_rows) continue;
#pragma unroll
        for (int i = 0; i < 5; ++i) {
            const int cc = c + (i - 2) * step;
            if (cc < 0 || cc >= cols) continue;
            const size_t q = size_t(rr) * size_t(cols) + size_t(cc);
            const float4 cq = __ldg(in + q);
            if (cq.w < 0.f) continue;
            const float dc = norm2(__fsub_rn(cp.x, cq.x), __fsub_rn(cp.y, cq.y), __fsub_rn(cp.z, cq.z));
            const float xc = dc == 0.f ? 0.f : __fdiv_rn(dc, __fmul_rn(sc2, __fadd_rn(cp.w, cq.w)));
            const float dn = norm2(__fsub_rn(npx, __ldg(f.normal + 3 * q)), __fsub_rn(npy, __ldg(f.normal + 3 * q + 1)),
                                   __fsub_rn(npz, __ldg(f.normal + 3 * q + 2)));
            const float da = norm2(__fsub_rn(anr, float(__ldg(f.albedo + 3 * q))), __fsub_rn(ang, float(__ldg(f.albedo + 3 * q + 1))),
                                   __fsub_rn(anb, float(__ldg(f.albedo + 3 * q + 2))));
            const float zq = __ldg(f.depth + q);
            float xz = 0.f;
            if (zp != zq) {
                if (isinf(zp) || isinf(zq)) {
                    xz = CUDART_INF_F;
                } else {
                    const float tz = __fdiv_rn(__fsub_rn(zp, zq), zscale);
                    xz = __fmul_rn(tz, tz);
                }
            }
            float w = float(kB3[j] * kB3[i]);
            w = __fmul_rn(w, edge_weight(xc));
            w = __fmul_rn(w, edge_weight(__fdiv_rn(dn, sn2)));
            w = __fmul_rn(w, edge_weight(__fdiv_rn(da, sa2)));
            w = __fmul_rn(w, edge_weight(xz));
            ws = __fadd_rn(ws, w);
            sr = __fadd_rn(sr, __fmul_rn(w, cq.x));
            sg = __fadd_rn(sg, __fmul_rn(w, cq.y));
            sb = __fadd_rn(sb, __fmul_rn(w, cq.z));
        }
    }
    // the centre tap always counts, with weight 36: ws > 0
    out[p] = make_float4(__fdiv_rn(sr, ws), __fdiv_rn(sg, ws), __fdiv_rn(sb, ws), cp.w);
}

// the last level to the caller's layouts: linear n*3 floats, RGB8 clamped to [0, 255], truncated, through PixelOutput.correct
__global__ void __launch_bounds__(kFilterThreads) denoise_output_kernel(const float4 *in, size_t n_pixels, int gamma, uint8_t *rgb, float *linear) {
    __shared__ uint8_t lut[256];
    fill_gamma_lut(lut, gamma);
    const size_t p = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (p >= n_pixels) return;
    const float4 v = in[p];
    if (linear) {
        linear[3 * p] = v.x;
        linear[3 * p + 1] = v.y;
        linear[3 * p + 2] = v.z;
    }
    if (rgb) {
        rgb[3 * p] = lut[int(fminf(fmaxf(v.x, 0.f), 255.f))];
        rgb[3 * p + 1] = lut[int(fminf(fmaxf(v.y, 0.f), 255.f))];
        rgb[3 * p + 2] = lut[int(fminf(fmaxf(v.z, 0.f), 255.f))];
    }
}

static unsigned grid_of(size_t n, int threads) { return unsigned((n + size_t(threads) - 1) / size_t(threads)); }

int launch_features(const FrameParams &fp, size_t n_pixels, int samples, const FrameFeatures &out, cudaStream_t st) {
    features_kernel<<<grid_of(n_pixels, kFeatureThreads), kFeatureThreads, 0, st>>>(fp, n_pixels, samples, out);
    RT_CUDA(cudaGetLastError());
    return RT_OK;
}

// a sigma as the filter uses it: the float32 nearest the double, finite and > 0
static bool sigma_ok(double s) {
    const float f = float(s);
    return f > 0.f && std::isfinite(f);
}

int check_denoise_opts(const RtDenoiseOpts *o, const char *who) {
    if (!o) return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": opts is null");
    if (o->iterations < 1 || o->iterations > kMaxDenoiseIterations)
        return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": iterations must be in [1, 10]");
    if (o->feature_samples < 1 || o->feature_samples > kMaxFeatureSamples)
        return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": feature_samples must be in [1, 64]");
    if (!sigma_ok(o->sigma_colour) || !sigma_ok(o->sigma_normal) || !sigma_ok(o->sigma_albedo) || !sigma_ok(o->sigma_depth))
        return fail(RT_ERR_INVALID_ARGUMENT, std::string(who) + ": every sigma must be > 0 and finite in float32");
    return RT_OK;
}

int launch_denoise(const int32_t *stats, const unsigned long long *sq, const FrameFeatures &feat, size_t n_pixels, int view_rows, int cols,
                   const RtDenoiseOpts &o, float4 *buf, bool want_rgb, bool want_linear, uint8_t **d_rgb, float **d_linear, cudaStream_t st) {
    float4 *level[2] = {buf, buf + n_pixels};
    const unsigned grid = grid_of(n_pixels, kFilterThreads);
    denoise_input_kernel<<<grid, kFilterThreads, 0, st>>>(reinterpret_cast<const int4 *>(stats), sq, n_pixels, level[0]);
    RT_CUDA(cudaGetLastError());
    const float sc = float(o.sigma_colour), sn = float(o.sigma_normal), sa = float(o.sigma_albedo), sz = float(o.sigma_depth);
    for (int k = 0; k < o.iterations; ++k) {
        // sigma_colour / 2^k: exact in float32 (a power-of-two scaling)
        atrous_kernel<<<grid, kFilterThreads, 0, st>>>(level[k & 1], level[(k + 1) & 1], feat, n_pixels, view_rows, cols, 1 << k,
                                                       std::ldexp(sc, -k), sn, sa, sz);
        RT_CUDA(cudaGetLastError());
    }
    // the outputs go to the other buffer: n*3 floats, then n*3 bytes (15 of its 16 bytes per pixel)
    const float4 *last = level[o.iterations & 1];
    float *linear = reinterpret_cast<float *>(level[(o.iterations + 1) & 1]);
    uint8_t *rgb = reinterpret_cast<uint8_t *>(linear + 3 * n_pixels);
    *d_linear = want_linear ? linear : nullptr;
    *d_rgb = want_rgb ? rgb : nullptr;
    if (want_rgb || want_linear) {
        denoise_output_kernel<<<grid, kFilterThreads, 0, st>>>(last, n_pixels, o.gamma, *d_rgb, *d_linear);
        RT_CUDA(cudaGetLastError());
    }
    return RT_OK;
}

} // namespace rtfs
