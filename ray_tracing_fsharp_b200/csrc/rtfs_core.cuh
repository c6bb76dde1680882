// rtfs_core.cuh — the device functions of the render path: counter RNG, vector algebra, integer
// colour, camera ray generation, sphere / plane / box intersection, BVH traversal, scatter and
// texture lookup.  Everything the render kernels and the conformance kernels execute lives here, so
// that a conformance entry point runs exactly the function the render kernel runs.
//
// Arithmetic: FP32, except (a) Pixel.darken's product (FP64, so that .NET's round-half-to-even is
// reproduced bit-for-bit), (b) the unbounded objects (huge spheres, planes), whose quadratic is
// evaluated in FP64 because |o-c|^2 - r^2 cancels catastrophically in FP32 for r ~ 1000.
//
// Self-intersection.  The reference rejects the t ~ 0 root of a ray that starts on a surface with the
// absolute test t > 1e-8, which works in FP64 (strike points lie within ~1e-13 of the surface) and
// cannot work in FP32 (~1e-6).  A ray therefore carries the id of the primitive it left (`last`), and
// the test against that primitive uses the exact on-surface form (c = 0 => roots 0 and -2b): the same
// decisions as the reference makes, without the cancellation.  See DESIGN.md §"FP32 and 1e-8".
#pragma once
#include "rtfs_internal.h"

#include <cuda_runtime.h>
#include <math_constants.h>

#ifndef RTFS_HD
#define RTFS_HD __device__ __forceinline__
#endif

// Bounds checks on the traversal stacks and the item bookkeeping: always on in the host build that runs under ASan /
// UBSan (host_debug/), and in a device build made with -DRTFS_DEBUG_BOUNDS (make bounds); compiled out otherwise.
#if defined(RTFS_HOST_DEBUG)
#define RTFS_BOUNDS(cond)                                                                                  \
    do {                                                                                                   \
        if (!(cond)) {                                                                                     \
            std::fprintf(stderr, "rtfs bounds check failed: %s (%s:%d)\n", #cond, __FILE__, __LINE__);      \
            std::abort();                                                                                  \
        }                                                                                                  \
    } while (0)
#elif defined(RTFS_DEBUG_BOUNDS)
#define RTFS_BOUNDS(cond)                                                                                  \
    do {                                                                                                   \
        if (!(cond)) {                                                                                     \
            printf("rtfs bounds check failed: %s (%s:%d)\n", #cond, __FILE__, __LINE__);                   \
            __trap();                                                                                      \
        }                                                                                                  \
    } while (0)
#else
#define RTFS_BOUNDS(cond) ((void)0)
#endif

namespace rtfs {

constexpr float kTolF = 1e-8f;   // Float.tolerance, RayTracing/Float.fs:80
constexpr double kTolD = 1e-8;
constexpr uint32_t kWhite = 0x00FFFFFFu, kBlack = 0u, kHotPink = (205u << 16) | (105u << 8) | 180u; // Pixel.fs:18-66
constexpr uint32_t kDegenerate = 0x80000000u; // flag on a path's result: it ended where the reference would throw (rendered Black)
constexpr int kNoPrim = -1;
constexpr int kNoRef = 0x7fffffff; // "no primitive" where primitives are named by ref (see SceneAccess)
constexpr float kNoHitT = 3.402823466e38f; // "bestFloat = infinity" (Scene.fs:65) as the largest finite float

// reconvergence point for the given lanes of the warp (no-op in the host-compiled debug build)
RTFS_HD void converge(unsigned lanes) {
#ifdef __CUDA_ARCH__
    __syncwarp(lanes);
#else
    (void)lanes;
#endif
}

// ---- Float.compare, Float.fs:88-96 ------------------------------------------------------------
enum Cmp { CMP_GREATER = 0, CMP_EQUAL = 1, CMP_LESS = 2 };
RTFS_HD Cmp fcmp(float a, float b) { return (fabsf(a - b) < kTolF) ? CMP_EQUAL : (a < b ? CMP_LESS : CMP_GREATER); }
RTFS_HD Cmp fcmp(double a, double b) { return (fabs(a - b) < kTolD) ? CMP_EQUAL : (a < b ? CMP_LESS : CMP_GREATER); }

// ---- one-instruction reciprocal / square root -----------------------------------------------------
// For arguments known to be normal numbers (or zero, for sqrt): a single MUFU (<= 2 ulp) instead of the IEEE
// sequences with their denormal rescaling and slow paths (4 to 12 instructions each, several per bounce).  The
// contract on this path is 1e-5 relative; decisions against the reference's 1e-8 tolerances move by an ulp or two.
RTFS_HD float rcp_fast(float x) { // 1 / x for |x| in the normal range: one MUFU.RCP (1 ulp), no denormal rescaling
#ifdef __CUDA_ARCH__
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#else
    return 1.0f / x;
#endif
}
RTFS_HD float rsqrt_fast(float x) { // 1 / sqrt(x), x a normal number: one MUFU.RSQ
#ifdef __CUDA_ARCH__
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#else
    return 1.0f / sqrtf(x);
#endif
}
RTFS_HD float sqrt_fast(float x) {
#ifdef __CUDA_ARCH__
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#else
    return sqrtf(x);
#endif
}

// ---- vectors (Point.fs:17-100) ------------------------------------------------------------------
RTFS_HD float3 f3(float x, float y, float z) { return make_float3(x, y, z); }
RTFS_HD float3 operator+(float3 a, float3 b) { return f3(a.x + b.x, a.y + b.y, a.z + b.z); }
RTFS_HD float3 operator-(float3 a, float3 b) { return f3(a.x - b.x, a.y - b.y, a.z - b.z); }
RTFS_HD float3 operator*(float s, float3 a) { return f3(s * a.x, s * a.y, s * a.z); }
RTFS_HD float3 operator-(float3 a) { return f3(-a.x, -a.y, -a.z); }
RTFS_HD float dot(float3 a, float3 b) { return fmaf(a.x, b.x, fmaf(a.y, b.y, a.z * b.z)); }
RTFS_HD float3 fma3(float s, float3 a, float3 b) { return f3(fmaf(s, a.x, b.x), fmaf(s, a.y, b.y), fmaf(s, a.z, b.z)); }
// Vector.unitise (Point.fs:28-35) / Ray.overwriteWithMake (Ray.fs:11-24): fails iff |v.v| < 1e-8
RTFS_HD bool unitise(float3 v, float3 &out) {
    float d = dot(v, v);
    if (fabsf(d) < kTolF) return false;
    out = rsqrt_fast(d) * v; // d >= 1e-8: a normal number; 2 ulp, renormalisation error stays ~1e-7
    return true;
}

struct D3 {
    double x, y, z;
};
RTFS_HD D3 d3(float3 a) { return D3{double(a.x), double(a.y), double(a.z)}; }
RTFS_HD D3 operator-(D3 a, D3 b) { return D3{a.x - b.x, a.y - b.y, a.z - b.z}; }
RTFS_HD double dot(D3 a, D3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }

// ---- counter RNG ---------------------------------------------------------------------------------
// Philox4x32-10 keyed by the frame seed, counter = (pixel, sample, bounce, retry).  Replaces the
// reference's shared, time-seeded xorshift producers (Float.fs:13-76, Scene.fs:205).  One block gives
// the 1-3 uniforms a bounce consumes (SURVEY.md Appendix A); `retry` advances on every further block.
RTFS_HD uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return c;
}
// FloatProducer's toDouble (Float.fs:29): w / (2^32 - 1) in [0, 1] inclusive.  In FP32 1/(2^32-1)
// rounds to 2^-32 and float(0xFFFFFFFF) = 2^32, so the range is preserved.
RTFS_HD float u01(uint32_t w) { return __uint2float_rn(w) * 2.3283064365386963e-10f; }

struct CounterRng {
    uint32_t k0, k1, pixel, sample, bounce, retry;
    RTFS_HD float4 next() {
        uint4 w = philox4x32_10(make_uint4(pixel, sample, bounce, retry), k0, k1);
        ++retry;
        return make_float4(u01(w.x), u01(w.y), u01(w.z), u01(w.w));
    }
};
// explicit uniforms for the conformance entry points: four values, rotated by one per block
struct ExplicitRng {
    float u[4];
    int rot;
    RTFS_HD float4 next() {
        float4 r = make_float4(u[rot & 3], u[(rot + 1) & 3], u[(rot + 2) & 3], u[(rot + 3) & 3]);
        ++rot;
        return r;
    }
};

// UnitVector.random, Point.fs:49-59: cube-normalised (F4), retry only when |v|^2 < 1e-8
template <class Rng>
RTFS_HD float3 unit_random(Rng &rng) {
    for (;;) {
        float4 u = rng.next();
        float3 v = f3(2.0f * u.x - 1.0f, 2.0f * u.y - 1.0f, 2.0f * u.z - 1.0f);
        float3 out;
        if (unitise(v, out)) return out;
    }
}

// ---- colour (Pixel.fs:136-151) --------------------------------------------------------------------
// colours are packed r << 16 | g << 8 | b
RTFS_HD uint32_t div255(uint32_t x) { return (x * 0x8081u) >> 23; } // exact for x < 65536
RTFS_HD uint32_t combine(uint32_t a, uint32_t b) {                  // Pixel.combine: (a * b) / 255, truncating
    uint32_t r = div255(((a >> 16) & 255u) * ((b >> 16) & 255u));
    uint32_t g = div255(((a >> 8) & 255u) * ((b >> 8) & 255u));
    uint32_t bl = div255((a & 255u) * (b & 255u));
    return (r << 16) | (g << 8) | bl;
}
RTFS_HD uint32_t darken(double albedo, uint32_t p) { // Pixel.darken: Math.Round (half to even) of a double product
    uint32_t r = uint32_t(__double2int_rn(double((p >> 16) & 255u) * albedo)) & 255u;
    uint32_t g = uint32_t(__double2int_rn(double((p >> 8) & 255u) * albedo)) & 255u;
    uint32_t b = uint32_t(__double2int_rn(double(p & 255u) * albedo)) & 255u;
    return (r << 16) | (g << 8) | b;
}

// ---- camera (Scene.fs:129-144) ----------------------------------------------------------------------
struct DevCamera {
    float ox, oy, oz;    // View.Origin
    float cx, cy, cz;    // ViewportXAxis.Origin - View.Origin (subtracted on the host in FP64)
    float xx, xy, xz;    // ViewportXAxis.Vector
    float yx, yy, yz;    // ViewportYAxis.Vector
    float sx, sy;        // ViewportWidth / maxWidthCoord, ViewportHeight / maxHeightCoord
    int32_t max_w, max_h, rows, cols;
    int32_t spp, depth;
};
// row / col are the signed coordinates renderPixel receives.  Returns false where Ray.make' would fail.
RTFS_HD bool camera_ray(const DevCamera &c, int row, int col, float r1, float r2, float3 &o, float3 &d) {
    float landing = (float(col) + r1) * c.sx;
    float walk = (float(row) + r2) * c.sy;
    float3 v = f3(fmaf(walk, c.yx, fmaf(landing, c.xx, c.cx)), fmaf(walk, c.yy, fmaf(landing, c.xy, c.cy)),
                  fmaf(walk, c.yz, fmaf(landing, c.xz, c.cz)));
    o = f3(c.ox, c.oy, c.oz);
    return unitise(v, d);
}

// ---- BoundingBox.hits with inverseDirections (BoundingBox.fs:25-94) -----------------------------------
// Decision-exact restatement: same comparison order, same +-inf / NaN behaviour (a NaN from 0 * inf
// fails every comparison and so leaves tMin / tMax unchanged).  No early return is needed: the bail-outs
// have no side effects, so evaluating all three axes and combining the predicates is equivalent.
RTFS_HD bool aabb_hits_ref(float3 inv, float3 o, const float mn[3], const float mx[3]) {
    float t_min = -CUDART_INF_F, t_max = CUDART_INF_F;
    float t0 = (mn[0] - o.x) * inv.x, t1 = (mx[0] - o.x) * inv.x;
    if (inv.x < 0.0f) { float s = t0; t0 = t1; t1 = s; }
    t_min = (t0 > t_min) ? t0 : t_min;
    t_max = (t1 < t_max) ? t1 : t_max;
    bool ok = !(t_max < t_min || 0.0f >= t_max);
    t0 = (mn[1] - o.y) * inv.y; t1 = (mx[1] - o.y) * inv.y;
    if (inv.y < 0.0f) { float s = t0; t0 = t1; t1 = s; }
    t_min = (t0 > t_min) ? t0 : t_min;
    t_max = (t1 < t_max) ? t1 : t_max;
    ok = ok && !(t_max < t_min || 0.0f >= t_max);
    t0 = (mn[2] - o.z) * inv.z; t1 = (mx[2] - o.z) * inv.z;
    if (inv.z < 0.0f) { float s = t0; t0 = t1; t1 = s; }
    t_min = (t0 > t_min) ? t0 : t_min;
    t_max = (t1 < t_max) ? t1 : t_max;
    return ok && (t_max >= t_min && t_max >= 0.0f);
}
RTFS_HD float3 inverse_directions(float3 d) { return f3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z); }

// Slab test of the render traversal.  Per ray: inv = 1 / d (components clamped away from zero, so no
// 0 * inf = NaN arises), noi = -o * inv, and pad = an absolute bound on the rounding of c * inv + noi; per box:
// ten packed FMA-pipe operations and a handful of min / max / compare for both children (see slab_pair).  Conservative: boxes are rounded outwards on
// the host, t_far is padded by 5 ulp (Ize, "Robust BVH Ray Traversal") plus `pad`.  Returns the entry distance for ordering and culls against the best hit so far
// (a finite number: kNoHitT while nothing is hit, so that the box {+inf, +inf} of a one-leaf tree is never
// entered).  It may accept a box the reference rejects only for rays within rounding of a box face; closest-hit
// results do not depend on it (rt_test_hit_object(traversal = 0) checks them against the oracle).
struct RaySlabs {
    float3 inv, noi, ainv; // 1 / d, -o / d, |1 / d|
    float pad;
};
RTFS_HD RaySlabs make_slabs(float3 o, float3 d) {
    const float tiny = 1e-30f;
    float x = fabsf(d.x) < tiny ? copysignf(tiny, d.x) : d.x;
    float y = fabsf(d.y) < tiny ? copysignf(tiny, d.y) : d.y;
    float z = fabsf(d.z) < tiny ? copysignf(tiny, d.z) : d.z;
    RaySlabs r;
    // approximate reciprocals (1 ulp): the slab test is padded, and noi is built from the same inv
    r.inv = f3(rcp_fast(x), rcp_fast(y), rcp_fast(z)); // |x|, |y|, |z| >= 1e-30: normal numbers
    r.noi = f3(-o.x * r.inv.x, -o.y * r.inv.y, -o.z * r.inv.z);
    r.ainv = f3(fabsf(r.inv.x), fabsf(r.inv.y), fabsf(r.inv.z));
    r.pad = 7.2e-7f * fmaxf(fmaxf(fabsf(r.noi.x), fabsf(r.noi.y)), fabsf(r.noi.z));
    return r;
}
// Two FP32 fused multiply-adds in one instruction: fma.rn.f32x2 (sm_100, SASS FFMA2) on register pairs, each half rounded
// exactly as fmaf rounds.  The render kernel is bound by instruction issue, not by the FMA pipe, so halving the issue slots
// of the slab arithmetic pays.  An operand whose halves are the same value (or the same value under |x| / -x) costs no extra
// register: ptxas folds the pack into a broadcast operand of FFMA2 (`|R27|.F32`).
RTFS_HD void fma2(float ax, float ay, float bx, float by, float cx, float cy, float &rx, float &ry) {
#ifdef __CUDA_ARCH__
    asm("{\n\t.reg .b64 a, b, c, r;\n\tmov.b64 a, {%2, %3};\n\tmov.b64 b, {%4, %5};\n\tmov.b64 c, {%6, %7};\n\t"
        "fma.rn.f32x2 r, a, b, c;\n\tmov.b64 {%0, %1}, r;\n\t}"
        : "=f"(rx), "=f"(ry)
        : "f"(ax), "f"(ay), "f"(bx), "f"(by), "f"(cx), "f"(cy));
#else
    rx = fmaf(ax, bx, cx);
    ry = fmaf(ay, by, cy);
#endif
}
// The two child boxes of a node at once.  Boxes come as centre c and half-extent h >= 0 with the left and the right child's
// values side by side (rtfs_internal.h, device_node_of): per axis the plane distances are t_c -+ h |inv| with t_c = c inv + noi,
// so near and far need no min / max pair (FMNMX, ALU pipe), and each of the three steps is one FFMA2 per axis for both
// boxes: ten FMA-pipe instructions per visit with the padding.  Three roundings per distance instead of one: t_far is padded
// by 5 ulp + pad.  hit = t_near <= min(t_far, best_t); the entry distances order the descent.
RTFS_HD void slab_pair(const RaySlabs &r, const uint4 &q0, const uint4 &q1, const uint4 &q2, float best_t, bool &hit_l, bool &hit_r, float &entry_l,
                       float &entry_r) {
    const float cxl = __uint_as_float(q0.x), cxr = __uint_as_float(q0.y), cyl = __uint_as_float(q0.z), cyr = __uint_as_float(q0.w);
    const float czl = __uint_as_float(q1.x), czr = __uint_as_float(q1.y), hxl = __uint_as_float(q1.z), hxr = __uint_as_float(q1.w);
    const float hyl = __uint_as_float(q2.x), hyr = __uint_as_float(q2.y), hzl = __uint_as_float(q2.z), hzr = __uint_as_float(q2.w);
    float txl, txr, tyl, tyr, tzl, tzr;
    fma2(cxl, cxr, r.inv.x, r.inv.x, r.noi.x, r.noi.x, txl, txr);
    fma2(cyl, cyr, r.inv.y, r.inv.y, r.noi.y, r.noi.y, tyl, tyr);
    fma2(czl, czr, r.inv.z, r.inv.z, r.noi.z, r.noi.z, tzl, tzr);
    float nxl, nxr, nyl, nyr, nzl, nzr, fxl, fxr, fyl, fyr, fzl, fzr;
    fma2(hxl, hxr, -r.ainv.x, -r.ainv.x, txl, txr, nxl, nxr);
    fma2(hyl, hyr, -r.ainv.y, -r.ainv.y, tyl, tyr, nyl, nyr);
    fma2(hzl, hzr, -r.ainv.z, -r.ainv.z, tzl, tzr, nzl, nzr);
    fma2(hxl, hxr, r.ainv.x, r.ainv.x, txl, txr, fxl, fxr);
    fma2(hyl, hyr, r.ainv.y, r.ainv.y, tyl, tyr, fyl, fyr);
    fma2(hzl, hzr, r.ainv.z, r.ainv.z, tzl, tzr, fzl, fzr);
    float fl, fr;
    fma2(fminf(fminf(fxl, fyl), fzl), fminf(fminf(fxr, fyr), fzr), 1.0000005960464478f, 1.0000005960464478f, r.pad, r.pad, fl, fr);
    entry_l = fmaxf(fmaxf(nxl, nyl), fmaxf(nzl, 0.0f));
    entry_r = fmaxf(fmaxf(nxr, nyr), fmaxf(nzr, 0.0f));
    hit_l = entry_l <= fminf(fl, best_t);
    hit_r = entry_r <= fminf(fr, best_t);
}

// ---- Sphere.firstIntersection (Sphere.fs:349-386) -------------------------------------------------------
// FP32 form for the bounded spheres.  The discriminant is evaluated as r^2 - |oc - b d|^2 (Haines et al.,
// "Precision Improvements for Ray/Sphere Intersection"), algebraically the reference's b^2 - (|oc|^2 - r^2)
// for unit d.  Root selection follows the reference line by line.  `self`: the ray starts on this sphere.
RTFS_HD bool sphere_hit(float3 o, float3 d, float4 s, bool self, float &t_out) {
    float3 oc = f3(o.x - s.x, o.y - s.y, o.z - s.z);
    float b = dot(d, oc);
    if (self) { // c = 0: roots 0 and -2b; the reference keeps the one that is `positive`
        float t = -2.0f * b;
        t_out = t;
        return t > kTolF;
    }
    float3 l = fma3(-b, d, oc);
    float disc = fmaf(s.w, s.w, -dot(l, l));
    // Sphere.fs:349-386 decides in three steps: Float.compare disc 0 (Equal: the one root -b; Less: miss), then which of
    // i1 = -b + sqrt(disc), i2 = -b - sqrt(disc) is `positive`, then the smaller of two positive roots.  Since i2 <= i1,
    // and they are 2 sqrt(disc) >= 2e-4 apart whenever disc >= 1e-8, that is: the root is i2 if i2 is positive, else i1,
    // and the ray hits iff that root is positive — the same decisions in two compares and a select (the ALU pipe is
    // the busiest unit of the render kernel).  disc within the tolerance of 0 is the case sqrt(disc) = 0 of the same formula.
    if (disc <= -kTolF) return false;
    const float im = disc < kTolF ? 0.0f : sqrt_fast(disc); // disc >= 1e-8 where the root is taken
    const float i2 = -(b + im), i1 = im - b;
    const float ip = i2 > kTolF ? i2 : i1;
    t_out = ip;
    return ip > kTolF;
}
// Unbounded spheres (typically huge: the r = 1000 floor, the r = 2000 light dome).  |o - c|^2 - r^2 and
// b^2 - c cancel catastrophically in FP32, so exactly those terms are evaluated in FP64 (on the FP32 ray promoted
// exactly); the square root and the roots are FP32, each root in its cancellation-free form (the product of the
// roots is c / a).  d is unit only to ~1e-7, so the quadratic keeps its leading coefficient a = d.d.
// Root selection follows Sphere.firstIntersection (Sphere.fs:349-386) line by line.
RTFS_HD bool sphere_hit_big(D3 o, D3 d, double a, const DUnbounded &s, bool self, float &t_out) {
    D3 oc = o - D3{s.p[0], s.p[1], s.p[2]};
    double b = dot(d, oc);
    float inv_a = rcp_fast(float(a)); // a = d.d ~ 1
    if (self) { // c = 0: roots 0 and -2b / a; the reference keeps the one that is `positive`
        float t = -2.0f * float(b) * inv_a;
        t_out = t;
        return t > kTolF;
    }
    double c = dot(oc, oc) - s.r2;
    float disc = float(b * b - a * c), bf = float(b), cf = float(c);
    float ip;
    if (fabsf(disc) < kTolF) { // Float.compare disc 0 = Equal
        ip = -bf * inv_a;
    } else if (disc < 0.0f) {
        return false;
    } else {
        float im = sqrt_fast(disc); // disc >= 1e-8 here
        float q1 = im - bf, q2 = -(bf + im); // i1 = q1 / a (the larger root), i2 = q2 / a; q1 * q2 = a * c
        float i1, i2;
        if (bf < 0.0f) { // |q1| >= im >= 1e-4
            i1 = q1 * inv_a;
            i2 = cf * rcp_fast(q1);
        } else { // |q2| >= im >= 1e-4
            i2 = q2 * inv_a;
            i1 = cf * rcp_fast(q2);
        }
        bool p1 = i1 > kTolF, p2 = i2 > kTolF;
        if (p1 && p2)
            ip = (fabsf(i1 - i2) < kTolF || i1 < i2) ? i1 : i2;
        else if (p1)
            ip = i1;
        else if (p2)
            ip = i2;
        else
            return false;
    }
    t_out = ip;
    return ip > kTolF;
}
// The same sphere from the expanded quadratic, all FP32 (DUnbounded.fp32 = 1): c = |o|^2 - 2 o.C + k with k = |C|^2 - r^2
// from the host, b = d.o - d.C.  No term is larger than scene-size x sphere-size, and nothing of the size of the
// sphere squared is ever subtracted from its like.  Root selection as above.
RTFS_HD float big_sphere_c(float3 o, const DUnbounded &s) {
    const float3 C = f3(s.n[0], s.n[1], s.n[2]);
    return fmaf(-2.0f, dot(o, C), dot(o, o)) + s.k;
}
RTFS_HD bool sphere_hit_big_f32(float3 o, float3 d, float a, const DUnbounded &s, bool self, float &t_out) {
    const float3 C = f3(s.n[0], s.n[1], s.n[2]);
    const float bf = dot(d, o) - dot(d, C);
    const float inv_a = rcp_fast(a); // a = d.d ~ 1
    if (self) { // c = 0: roots 0 and -2b / a; the reference keeps the one that is `positive`
        float t = -2.0f * bf * inv_a;
        t_out = t;
        return t > kTolF;
    }
    const float cf = big_sphere_c(o, s);
    const float disc = fmaf(bf, bf, -a * cf);
    if (disc <= -kTolF) return false; // Float.compare disc 0 = Less
    float ip;
    if (disc < kTolF) { // Equal: the one root
        ip = -bf * inv_a;
    } else {
        const float im = sqrt_fast(disc); // disc >= 1e-8 here
        // i1 = q1 / a is the larger root, i2 = q2 / a the smaller; q1 * q2 = a * c gives whichever of them cancels in its
        // own formula from the other.  As in sphere_hit: the root is i2 if it is positive, else i1 (they are >= 2e-4 apart).
        const float q = bf < 0.0f ? im - bf : -(bf + im); // |q| >= im >= 1e-4
        const float via_q = q * inv_a, via_c = cf * rcp_fast(q);
        const float i1 = bf < 0.0f ? via_q : via_c, i2 = bf < 0.0f ? via_c : via_q;
        ip = i2 > kTolF ? i2 : i1;
    }
    t_out = ip;
    return ip > kTolF;
}
// and the plane: n.(p0 - o) = k - n.o
RTFS_HD bool plane_hit_big_f32(float3 o, float3 d, const DUnbounded &p, bool self, float &t_out) {
    if (self) return false;
    const float3 n = f3(p.n[0], p.n[1], p.n[2]);
    const float den = dot(n, d);
    if (fabsf(den) < kTolF) return false;
    float t = (p.k - dot(n, o)) * rcp_fast(den); // |den| >= 1e-8
    t_out = t;
    return t > kTolF;
}
// InfinitePlane.intersection (InfinitePlane.fs:125-136): numerator and denominator in FP64, quotient in FP32
RTFS_HD bool plane_hit_big(D3 o, D3 d, const DUnbounded &p, bool self, float &t_out) {
    if (self) return false; // the numerator is 0 on the plane: t = 0 is never `positive`
    D3 n{double(p.n[0]), double(p.n[1]), double(p.n[2])};
    float den = float(dot(n, d));
    if (fabsf(den) < kTolF) return false;
    float t = float(dot(n, D3{p.p[0], p.p[1], p.p[2]} - o)) * rcp_fast(den); // |den| >= 1e-8
    t_out = t;
    return t > kTolF;
}
// ---- scene access ------------------------------------------------------------------------------------
// The render kernels read the flattened BVH either from global memory through the read-only path
// (128-bit __ldg) or from a copy staged in shared memory (128-bit LDS); the template parameter picks.
struct SceneGlobal {
    const uint4 *nodes;
    const float4 *spheres;
    const uint4 *mats;
    const DUnbounded *unb;
    const DTexture *tex;
    int32_t n_nodes, n_bounded, n_unbounded, n_tex;
    // the 8-wide compressed tree (null until built: big scenes at creation, others on first use)
    const uint4 *wide_nodes;      // 5 per node
    const float4 *wide_spheres;   // the spheres in the wide tree's order
    const int32_t *wide_to_dev;   // wide sphere index -> device primitive id
    const int32_t *dev_to_wide;   // and back
};

#ifdef __CUDACC__
extern __shared__ uint4 rtfs_smem[];
// 128-bit load from a 32-bit shared-window address (one LDS.128, no generic-address arithmetic)
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
#endif

RTFS_HD float4 ldg_sphere(const float4 *p) {
#ifdef __CUDA_ARCH__
    return __ldg(p);
#else
    return *p;
#endif
}

// A staged node takes FIVE quads of shared memory, not four: with a stride of 64 bytes quad q of every node lies in one
// of only two 16-byte bank groups, so the LDS.128 of a walk's divergent lanes (each at a node of its own) collide several
// ways within every quarter-warp (ncu: 39 % of all shared-memory wavefronts were bank conflicts).  At 80 bytes quad q of node
// i starts at bank group (5 i + q) mod 8: every group equally likely.  Child refs are byte addresses, so a visit pays nothing.
constexpr uint32_t kStagedNodeQuads = 5;
// SMEM: 0 = the scene is read from global memory, 1 = from the copy staged in shared memory, 2 = staged and LEAN: the host has
// seen that every unbounded object is cleared for FP32 and no material has a texture index (DeviceScene::lean), so the FP64
// evaluations of unbounded objects and the texture lookup are compiled out of that kernel (fewer instructions per ray — the
// compiler hoists the FP64 conversions of the ray out of the loop over the objects, for every ray — and a smaller kernel).
template <int SMEM>
struct SceneAccess {
    static constexpr bool kLean = SMEM == 2;
    SceneGlobal g;
    uint32_t s_nodes, s_spheres, s_mats; // SMEM only: byte addresses of the staged copies in the shared window
    // one 64-byte node: four LDS.128 from the staged copy, or two 256-bit read-only loads from global memory
    // (sm_100 has LDG.256: half as many L1 requests per divergent node fetch as four 128-bit loads)
    // Child references.  A walk holds a `ref`: >= 0 an internal node, < 0 a leaf.  Read from global memory a ref is
    // the node index / ~sphere index the host wrote.  In the staged copy (SMEM) stage_tree() has rewritten every
    // ref into the shared-window byte address of what it points at (node: address; leaf: ~address of the sphere), so
    // a visit needs no address arithmetic at all (the compiler would otherwise rebuild base + 64 i from special
    // registers on every visit rather than keep the base in a register).
    RTFS_HD int root() const { return SMEM ? int(s_nodes) : 0; }
    RTFS_HD int ref_of_sphere(int k) const { return SMEM ? ~int(s_spheres + 16u * uint32_t(k)) : ~k; }
    RTFS_HD int sphere_of_ref(int ref) const { return SMEM ? int((uint32_t(~ref) - s_spheres) >> 4) : ~ref; }
    RTFS_HD void node(int i, uint4 &q0, uint4 &q1, uint4 &q2, uint4 &q3) const {
#ifdef __CUDACC__
        if (SMEM) {
            const uint32_t a = uint32_t(i);
            q0 = lds128(a);
            q1 = lds128(a + 16u);
            q2 = lds128(a + 32u);
            q3 = lds128(a + 48u);
            return;
        }
        const uint4 *p = g.nodes + 4 * i;
        asm volatile("ld.global.nc.v8.u32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=r"(q0.x), "=r"(q0.y), "=r"(q0.z), "=r"(q0.w), "=r"(q1.x), "=r"(q1.y), "=r"(q1.z), "=r"(q1.w)
                     : "l"(p));
        asm volatile("ld.global.nc.v8.u32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=r"(q2.x), "=r"(q2.y), "=r"(q2.z), "=r"(q2.w), "=r"(q3.x), "=r"(q3.y), "=r"(q3.z), "=r"(q3.w)
                     : "l"(p + 2));
#else
        q0 = g.nodes[4 * i];
        q1 = g.nodes[4 * i + 1];
        q2 = g.nodes[4 * i + 2];
        q3 = g.nodes[4 * i + 3];
#endif
    }
    RTFS_HD float4 sphere_at(int ref) const { // the sphere a leaf ref points at
#ifdef __CUDACC__
        if (SMEM) {
            uint4 v = lds128(uint32_t(~ref));
            return make_float4(__uint_as_float(v.x), __uint_as_float(v.y), __uint_as_float(v.z), __uint_as_float(v.w));
        }
#endif
        return __ldg(g.spheres + ~ref);
    }
#ifdef __CUDACC__
    // Copies the whole scene (SMEM) into shared memory at s_nodes / s_spheres / s_mats, rewriting the child refs
    // of the nodes (see above).  Every thread of the block must call it; ends in __syncthreads().
    __device__ __forceinline__ void stage_tree(uint32_t q_nodes, uint32_t q_spheres, uint32_t q_mats) const {
        const int n_nodes_q = g.n_nodes * 4, n_sph_q = g.n_bounded, n_mat_q = (g.n_bounded + g.n_unbounded) * 2;
        for (int i = threadIdx.x; i < n_nodes_q; i += blockDim.x) {
            uint4 v = __ldg(g.nodes + i);
            if ((i & 3) == 3) { // {left, right, -, -}
                v.x = int(v.x) >= 0 ? s_nodes + 16u * kStagedNodeQuads * v.x : uint32_t(ref_of_sphere(~int(v.x)));
                v.y = int(v.y) >= 0 ? s_nodes + 16u * kStagedNodeQuads * v.y : uint32_t(ref_of_sphere(~int(v.y)));
            }
            rtfs_smem[q_nodes + (i >> 2) * kStagedNodeQuads + (i & 3)] = v;
        }
        for (int i = threadIdx.x; i < n_sph_q; i += blockDim.x) rtfs_smem[q_spheres + i] = __ldg(reinterpret_cast<const uint4 *>(g.spheres) + i);
        for (int i = threadIdx.x; i < n_mat_q; i += blockDim.x) rtfs_smem[q_mats + i] = __ldg(g.mats + i);
        __syncthreads();
    }
#endif
    RTFS_HD float4 sphere(int i) const {
#ifdef __CUDACC__
        if (SMEM) {
            uint4 v = lds128(s_spheres + 16u * uint32_t(i));
            return make_float4(__uint_as_float(v.x), __uint_as_float(v.y), __uint_as_float(v.z), __uint_as_float(v.w));
        }
#endif
        return __ldg(g.spheres + i);
    }
    RTFS_HD uint4 mat_q(int i, int q) const {
#ifdef __CUDACC__
        if (SMEM) return lds128(s_mats + 32u * uint32_t(i) + 16u * uint32_t(q));
#endif
        return __ldg(g.mats + 2 * i + q);
    }
};

struct Hit {
    float t;
    int32_t prim; // device primitive id, kNoPrim: nothing hit
    int32_t ref;  // the same primitive as a walk names it: leaf ref (bounded sphere) | device id (unbounded) | kNoRef
    float3 strike;
};

struct TraversalCounters {
    uint32_t box_tests, prim_tests;
};

// The walk's stack of postponed children: a per-thread array in local memory, or (render kernels, when shared memory
// has room for tree depth x block size words) a column of shared memory per thread.  Thread t's entry i sits at word
// i * blockDim + t: lanes are always in distinct banks, whatever their depths, so a push or pop is one conflict-free
// wavefront, where lanes at different depths of a local-memory stack touch a cache line each.
constexpr int kLocalStackWords = 64;
struct LocalStack {
    int a[kLocalStackWords];
    RTFS_HD void put(int i, int v) {
        RTFS_BOUNDS(i >= 0 && i < kLocalStackWords);
        a[i] = v;
    }
    RTFS_HD int get(int i) const {
        RTFS_BOUNDS(i >= 0 && i < kLocalStackWords);
        return a[i];
    }
    // two-word entries (the wide walk's node groups)
    RTFS_HD void put2(int i, uint2 v) {
        RTFS_BOUNDS(i >= 0 && 2 * i + 1 < kLocalStackWords);
        a[2 * i] = int(v.x);
        a[2 * i + 1] = int(v.y);
    }
    RTFS_HD uint2 get2(int i) const {
        RTFS_BOUNDS(i >= 0 && 2 * i + 1 < kLocalStackWords);
        return make_uint2(uint32_t(a[2 * i]), uint32_t(a[2 * i + 1]));
    }
};
#ifdef __CUDACC__
struct SharedStack {
    uint32_t base, stride; // byte address of this thread's entry 0 in the shared window; bytes between entries
    int levels;            // words per thread (checked with -DRTFS_DEBUG_BOUNDS only)
    __device__ __forceinline__ void put(int i, int v) {
        RTFS_BOUNDS(i >= 0 && i < levels);
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(base + uint32_t(i) * stride), "r"(v));
    }
    __device__ __forceinline__ int get(int i) const {
        RTFS_BOUNDS(i >= 0 && i < levels);
        int v;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(base + uint32_t(i) * stride));
        return v;
    }
    __device__ __forceinline__ void put2(int i, uint2 v) {
        RTFS_BOUNDS(i >= 0 && 2 * i + 1 < levels);
        const uint32_t a = base + uint32_t(2 * i) * stride;
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v.x));
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(a + stride), "r"(v.y));
    }
    __device__ __forceinline__ uint2 get2(int i) const {
        RTFS_BOUNDS(i >= 0 && 2 * i + 1 < levels);
        const uint32_t a = base + uint32_t(2 * i) * stride;
        uint2 v;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v.x) : "r"(a));
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v.y) : "r"(a + stride));
        return v;
    }
};
#endif

// Scene.hitObject (Scene.fs:62-91) over the SAH tree: ordered, culled by the best hit so far.  The
// closest hit does not depend on tree topology or visiting order (only exact ties in t do, F12), so the
// result equals the reference's exhaustive left-then-right DFS.  Then the unbounded objects in array
// order, which must win by Float.compare t^2 best^2 = Less (Scene.fs:77-86).
// One visit of the walk over the tree: `node` is an internal node (>= 0: test both children's boxes, descend into
// the nearer one, push the other) or a leaf (~k: test sphere k, pop).  Returns true when the walk is over.
// `node`, `last_ref`, `best` and the stack entries are refs (SceneAccess); best >= 0 (kNoRef): nothing hit yet.
template <int SMEM, bool COUNT, class Stack>
RTFS_HD bool bvh_visit(const SceneAccess<SMEM> &sc, const RaySlabs &rs, float3 o, float3 d, int last_ref, int &node, int &sp, Stack &stack,
                       float &best_t, int &best, TraversalCounters &cn) {
    if (node >= 0) {
        uint4 q0, q1, q2, q3;
        sc.node(node, q0, q1, q2, q3);
        float tl, tr;
        bool hl, hr;
        slab_pair(rs, q0, q1, q2, best_t, hl, hr, tl, tr);
        if (COUNT) cn.box_tests += 2;
        int left = int(q3.x), right = int(q3.y);
        if (hl && hr) {
            bool left_first = tl <= tr;
            stack.put(sp++, left_first ? right : left);
            node = left_first ? left : right;
            return false;
        }
        if (hl) { node = left; return false; }
        if (hr) { node = right; return false; }
    } else {
        float4 s = sc.sphere_at(node);
        float t;
        if (COUNT) cn.prim_tests += 1;
        if (sphere_hit(o, d, s, node == last_ref, t) && t < best_t) {
            best_t = t;
            best = node;
        }
    }
    if (sp == 0) return true;
    node = stack.get(--sp);
    return false;
}
// ---- the 8-wide compressed tree (scenes read from global memory) -------------------------------------------------
// After Ylitie, Karras, Laine (HPG 2017).  A visit loads one 80-byte node (five 128-bit read-only loads: three 32-byte
// sectors instead of the two per BVH2 visit, for a third as many visits), tests its eight quantised child boxes against
// the ray and the best hit so far, and turns the outcome into one 32-bit mask: bits 24..31 = internal children that
// were hit, at position 24 + (slot XOR octant of the ray), so that the highest set bit is always the child to enter
// next (front to back without computing or sorting distances); bits 0..23 = spheres of the node's leaf children.  The
// walk holds a "node group" {child_base, hit bits | imask}: popping a child is a find-highest-bit and a popcount; a
// group with children left over goes on the stack as ONE two-word entry.
//
// A quantised plane byte b becomes the float 1 + b 2^-15 with one PRMT (b dropped into the mantissa of 1.0f), so a
// plane distance is one FFMA, t = f S + C, with per node and axis S = 2^(e+15) / d and C = (p - o) / d - S: no integer to
// float conversions (a quarter-rate pipe).  The test is conservative: boxes are quantised outwards, t_far is padded.
// Refs here: a sphere is named ~k with k its index in the WIDE sphere order (wide_to_dev maps it to the device id).
#ifdef __CUDACC__
RTFS_HD float wide_plane(uint32_t q4, int j) { // byte j of q4 -> 1 + b 2^-15
    return __uint_as_float(__byte_perm(q4, 0x3F800000u, 0x7604u | (uint32_t(j) << 4)));
}
RTFS_HD uint4 ldg128(const uint4 *p) { return __ldg(p); }
#else
RTFS_HD float wide_plane(uint32_t q4, int j) { return 1.0f + float((q4 >> (8 * j)) & 255u) * 3.0517578125e-05f; }
RTFS_HD uint4 ldg128(const uint4 *p) { return *p; }
RTFS_HD int __clz(uint32_t x) { return x ? __builtin_clz(x) : 32; }
RTFS_HD int __popc(uint32_t x) { return __builtin_popcount(x); }
#endif
template <bool COUNT, class Stack>
RTFS_HD void wide_closest(const SceneGlobal &g, float3 o, float3 d, int last_ref, float &best_t, int &best_ref, TraversalCounters &cn, Stack &stack) {
    best_t = kNoHitT;
    best_ref = kNoRef;
    if (g.n_bounded <= 0) return;
    const RaySlabs rs = make_slabs(o, d);
    const bool nx = rs.inv.x < 0.0f, ny = rs.inv.y < 0.0f, nz = rs.inv.z < 0.0f;
    const uint32_t octinv = (nx ? 0u : 4u) | (ny ? 0u : 2u) | (nz ? 0u : 1u);
    const uint32_t octinv4 = octinv * 0x01010101u;
    uint2 ngroup = make_uint2(0u, 0x80000000u); // the root: "child 0 of a group at base 0"
    int sp = 0;
    for (;;) {
        // ---- enter the nearest child of the current group ----
        const uint32_t bit = 31u - uint32_t(__clz(ngroup.y));
        const uint32_t imask_bits = ngroup.y;
        ngroup.y &= ~(1u << bit);
        if (ngroup.y > 0x00FFFFFFu) stack.put2(sp++, ngroup);
        const uint32_t slot = (bit - 24u) ^ octinv;
        const uint32_t node = ngroup.x + uint32_t(__popc(imask_bits & ~(0xFFFFFFFFu << slot)));
        const uint4 *np = g.wide_nodes + 5 * size_t(node);
        const uint4 n0 = ldg128(np), n1 = ldg128(np + 1), n2 = ldg128(np + 2), n3 = ldg128(np + 3), n4 = ldg128(np + 4);
        if (COUNT) cn.box_tests += 8;
        // per node and axis: t(b) = f(b) S + C
        const float sx = __uint_as_float((n0.w & 0xffu) << 23) * rs.inv.x;
        const float sy = __uint_as_float((n0.w & 0xff00u) << 15) * rs.inv.y;
        const float sz = __uint_as_float((n0.w & 0xff0000u) << 7) * rs.inv.z;
        const float bx = fmaf(__uint_as_float(n0.x), rs.inv.x, rs.noi.x), by = fmaf(__uint_as_float(n0.y), rs.inv.y, rs.noi.y),
                    bz = fmaf(__uint_as_float(n0.z), rs.inv.z, rs.noi.z);
        const float cx = bx - sx, cy = by - sy, cz = bz - sz;
        // rounding of b (relative to |b|), of C (relative to |b| + |S|) and of noi (rs.pad), as an absolute pad on t_far
        const float pad = fmaf(2.4e-7f, fmaxf(fmaxf(fabsf(bx) + fabsf(sx), fabsf(by) + fabsf(sy)), fabsf(bz) + fabsf(sz)), rs.pad);
        uint32_t hits = 0;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const uint32_t meta4 = half ? n1.w : n1.z;
            const uint32_t is_inner4 = (meta4 & (meta4 << 1)) & 0x10101010u;
            const uint32_t inner_mask4 = (is_inner4 >> 4) * 0xffu; // 0xff in the bytes of internal children (no carries: 1 * 0xff)
            const uint32_t bit_index4 = (meta4 ^ (octinv4 & inner_mask4)) & 0x1F1F1F1Fu;
            const uint32_t child_bits4 = (meta4 >> 5) & 0x07070707u;
            const uint32_t qlx = half ? n2.y : n2.x, qly = half ? n2.w : n2.z, qlz = half ? n3.y : n3.x;
            const uint32_t qhx = half ? n3.w : n3.z, qhy = half ? n4.y : n4.x, qhz = half ? n4.w : n4.z;
            const uint32_t near_x = nx ? qhx : qlx, far_x = nx ? qlx : qhx;
            const uint32_t near_y = ny ? qhy : qly, far_y = ny ? qly : qhy;
            const uint32_t near_z = nz ? qhz : qlz, far_z = nz ? qlz : qhz;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float t0x = fmaf(wide_plane(near_x, j), sx, cx), t1x = fmaf(wide_plane(far_x, j), sx, cx);
                const float t0y = fmaf(wide_plane(near_y, j), sy, cy), t1y = fmaf(wide_plane(far_y, j), sy, cy);
                const float t0z = fmaf(wide_plane(near_z, j), sz, cz), t1z = fmaf(wide_plane(far_z, j), sz, cz);
                const float t_near = fmaxf(fmaxf(t0x, t0y), fmaxf(t0z, 0.0f));
                const float t_far = fminf(fminf(t1x, t1y), fminf(t1z, best_t));
                if (t_near <= fmaf(t_far, 1.0000003576278687f, pad)) hits |= ((child_bits4 >> (8 * j)) & 0xffu) << ((bit_index4 >> (8 * j)) & 0xffu);
            }
        }
        ngroup = make_uint2(n1.x, (hits & 0xFF000000u) | (n0.w >> 24));
        // ---- the spheres of this node's leaf children that the ray may hit ----
        uint32_t prims = hits & 0x00FFFFFFu;
        while (prims) {
            const uint32_t pb = 31u - uint32_t(__clz(prims));
            prims &= ~(1u << pb);
            const int k = int(n1.y + pb);
            float t;
            if (COUNT) cn.prim_tests += 1;
            if (sphere_hit(o, d, ldg_sphere(g.wide_spheres + k), ~k == last_ref, t) && t < best_t) {
                best_t = t;
                best_ref = ~k;
            }
        }
        if (ngroup.y <= 0x00FFFFFFu) {
            if (sp == 0) return;
            ngroup = stack.get2(--sp);
        }
    }
}

// A path remembers the primitive its ray leaves as the walk names it: the leaf ref of a bounded sphere (< 0), the
// device id of an unbounded object (>= n_bounded), kNoRef for a camera ray.  From a device primitive id:
template <int SMEM, bool WIDE = false>
RTFS_HD int ref_of_prim(const SceneAccess<SMEM> &sc, int prim) {
    if (WIDE) return prim < 0 ? kNoRef : (prim < sc.g.n_bounded ? ~sc.g.dev_to_wide[prim] : prim);
    return prim < 0 ? kNoRef : (prim < sc.g.n_bounded ? sc.ref_of_sphere(prim) : prim);
}
// the bounded part of hitObject: the closest sphere of the tree, if any
template <int SMEM, bool COUNT, class Stack>
RTFS_HD void bvh_closest(const SceneAccess<SMEM> &sc, float3 o, float3 d, int last_ref, float &best_t, int &best_ref, TraversalCounters &cn,
                         Stack &stack) {
    best_t = kNoHitT;
    best_ref = kNoRef;
    if (sc.g.n_bounded <= 0) return;
    const RaySlabs rs = make_slabs(o, d);
    int sp = 0;
    int node = sc.root();
    while (!bvh_visit<SMEM, COUNT>(sc, rs, o, d, last_ref, node, sp, stack, best_t, best_ref, cn)) {
    }
}
// the unbounded objects, after the tree (Scene.fs:77-86), and the strike point (:91)
// (`last_ref` and `best_ref` are refs; an unbounded object's ref is its device id)
template <int SMEM, bool COUNT, bool WIDE = false>
RTFS_HD Hit finish_hit(const SceneAccess<SMEM> &sc, float3 o, float3 d, int last_ref, float best_t, int best_ref, TraversalCounters &cn) {
    const int last = last_ref;
    int best = best_ref;
    if (sc.g.n_unbounded > 0) {
        const float af = dot(d, d);
        for (int i = 0; i < sc.g.n_unbounded; ++i) {
            const DUnbounded &u = sc.g.unb[i];
            float t;
            bool self = (sc.g.n_bounded + i) == last;
            bool hit;
            if (SceneAccess<SMEM>::kLean || u.fp32) { // warp-uniform: every lane is at object i
                hit = (u.shape == RT_SHAPE_INFINITE_PLANE) ? plane_hit_big_f32(o, d, u, self, t) : sphere_hit_big_f32(o, d, af, u, self, t);
            } else {
                const D3 od = d3(o), dd = d3(d);
                hit = (u.shape == RT_SHAPE_INFINITE_PLANE) ? plane_hit_big(od, dd, u, self, t) : sphere_hit_big(od, dd, dot(dd, dd), u, self, t);
            }
            if (COUNT) cn.prim_tests += 1;
            // Float.compare (t * t) bestFloat = Less, Scene.fs:82
            if (hit && fcmp(t * t, best_t * best_t) == CMP_LESS) {
                best_t = t;
                best = sc.g.n_bounded + i;
            }
        }
    }
    Hit h;
    h.t = best_t;
    h.ref = best;
    h.prim = best < 0 ? (WIDE ? sc.g.wide_to_dev[~best] : sc.sphere_of_ref(best)) : (best == kNoRef ? kNoPrim : best);
    h.strike = fma3(best_t, d, o); // Ray.walkAlong ray bestLength, Scene.fs:91
    return h;
}
// `lanes`: the lanes of this warp that are tracing a ray in this call.  They leave the walk at different times and
// wait for one another before the unbounded tests, so that those and the scatter that follows run once per warp at
// full width instead of once per straggler group.
// (Tried and dropped: parking a leaf and testing it after the walk, converged, instead of during it at ~4 active
// lanes — the lost culling costs 5 % more slab tests and the C2 frame got 3 % slower.)
template <int SMEM, bool COUNT, class Stack, bool WIDE = false>
RTFS_HD Hit closest_hit_from(const SceneAccess<SMEM> &sc, float3 o, float3 d, int last_ref, TraversalCounters &cn, unsigned lanes, Stack &stack) {
    float best_t;
    int best_ref;
    if (WIDE)
        wide_closest<COUNT>(sc.g, o, d, last_ref, best_t, best_ref, cn, stack);
    else
        bvh_closest<SMEM, COUNT>(sc, o, d, last_ref, best_t, best_ref, cn, stack);
    converge(lanes);
    return finish_hit<SMEM, COUNT, WIDE>(sc, o, d, last_ref, best_t, best_ref, cn);
}
// the same with the ray's previous primitive given as a device primitive id (conformance entry points, wavefront)
template <int SMEM, bool COUNT, bool WIDE = false>
RTFS_HD Hit closest_hit(const SceneAccess<SMEM> &sc, float3 o, float3 d, int last, TraversalCounters &cn, unsigned lanes) {
    LocalStack stack;
    return closest_hit_from<SMEM, COUNT, LocalStack, WIDE>(sc, o, d, ref_of_prim<SMEM, WIDE>(sc, last), cn, lanes, stack);
}

// The reference's own traversal (Scene.fs:30-60, F12): exhaustive left-then-right DFS of the
// reference-topology tree with the decision-exact slab test and no culling.  Conformance only.
RTFS_HD Hit closest_hit_reference(const DRefNode *ref_nodes, int n_ref_nodes, const SceneGlobal &g, float3 o, float3 d, int last) {
    float best_t = CUDART_INF_F;
    int best = kNoPrim;
    if (n_ref_nodes > 0) {
        float3 inv = inverse_directions(d);
        int stack[64];
        int sp = 0;
        int node = 0;
        for (;;) {
            const DRefNode nd = ref_nodes[node];
            bool descend = false;
            if (aabb_hits_ref(inv, o, nd.mn, nd.mx)) {
                if (nd.right < 0) {
                    if (nd.prim >= 0) {
                        float t;
                        if (sphere_hit(o, d, __ldg(g.spheres + nd.prim), nd.prim == last, t) && t * t < best_t * best_t) {
                            best_t = t;
                            best = nd.prim;
                        }
                    }
                } else {
                    stack[sp++] = nd.right;
                    node = node + 1;
                    descend = true;
                }
            }
            if (descend) continue;
            if (sp == 0) break;
            node = stack[--sp];
        }
    }
    const D3 od = d3(o), dd = d3(d);
    const double a = dot(dd, dd);
    const float af = dot(d, d);
    if (best == kNoPrim) best_t = kNoHitT;
    for (int i = 0; i < g.n_unbounded; ++i) {
        const DUnbounded &u = g.unb[i];
        float t;
        bool self = (g.n_bounded + i) == last;
        bool hit;
        if (u.fp32)
            hit = (u.shape == RT_SHAPE_INFINITE_PLANE) ? plane_hit_big_f32(o, d, u, self, t) : sphere_hit_big_f32(o, d, af, u, self, t);
        else
            hit = (u.shape == RT_SHAPE_INFINITE_PLANE) ? plane_hit_big(od, dd, u, self, t) : sphere_hit_big(od, dd, a, u, self, t);
        if (hit && fcmp(t * t, best_t * best_t) == CMP_LESS) {
            best_t = t;
            best = g.n_bounded + i;
        }
    }
    Hit h;
    h.t = best_t;
    h.prim = best;
    h.ref = kNoRef; // not used by the callers of the conformance traversal
    h.strike = fma3(best_t, d, o);
    return h;
}

// ---- textures (Texture.fs:12-15, :50-67; Sphere.planeMapInverse Sphere.fs:55-61) ------------------------
#ifndef RTFS_HOST_DEBUG
RTFS_HD uint32_t fetch_texel(unsigned long long tex, int x, int y) {
    uchar4 v = tex2D<uchar4>(cudaTextureObject_t(tex), float(x) + 0.5f, float(y) + 0.5f);
    return (uint32_t(v.x) << 16) | (uint32_t(v.y) << 8) | uint32_t(v.z);
}
#endif
RTFS_HD uint32_t texture_colour(const SceneGlobal &g, int tex, float3 p) {
    DTexture t = g.tex[tex];
    if (t.kind == RT_TEX_COLOUR) return t.rgb;
    float3 q = t.inv_radius * f3(p.x - t.cx, p.y - t.cy, p.z - t.cz);
    float theta = acosf(fminf(1.0f, fmaxf(-1.0f, -q.y)));
    float phi = atan2f(-q.z, q.x) + CUDART_PI_F;
    float u = phi * (0.5f / CUDART_PI_F), v = theta * (1.0f / CUDART_PI_F); // constants fold; a multiply instead of an IEEE division
    for (int guard = 0; guard < 8 && t.kind == RT_TEX_CHECKERED; ++guard) { // Texture.fs:56-62
        float sine = sinf(t.grid * u) * sinf(t.grid * v);
        t = g.tex[(fcmp(sine, 0.0f) == CMP_LESS) ? t.even : t.odd];
    }
    if (t.kind == RT_TEX_COLOUR) return t.rgb;
    if (t.kind == RT_TEX_IMAGE) { // Texture.fs:63-67: truncating nearest lookup with the u flip
        int x = int((1.0f - u) * float(t.w - 1));
        int y = int(v * float(t.h - 1));
        x = min(max(x, 0), t.w - 1);
        y = min(max(y, 0), t.h - 1);
        return fetch_texel(t.tex, x, y);
    }
    return kBlack;
}

// ---- scatter ----------------------------------------------------------------------------------------------
struct Material {
    double albedo;
    float p0, p1;
    uint32_t style, rgb;
    int32_t texture;
    uint32_t flags;
    int32_t host_index;
};
template <int SMEM>
RTFS_HD Material load_material(const SceneAccess<SMEM> &sc, int prim) {
    uint4 a = sc.mat_q(prim, 0), b = sc.mat_q(prim, 1);
    Material m;
    m.albedo = __hiloint2double(int(a.y), int(a.x));
    m.p0 = __uint_as_float(a.z);
    m.p1 = __uint_as_float(a.w);
    m.style = b.x >> 24;
    m.rgb = b.x & 0x00FFFFFFu;
    m.texture = int(b.y);
    m.flags = b.z;
    m.host_index = int(b.w);
    return m;
}

// Sphere.reflectWithoutFuzz (Sphere.fs:68-87) / InfinitePlane.pureOutgoing (InfinitePlane.fs:18-38).
// With T = unit(d - (n.d) n) the reference's -(n.d) n + (T.d) T equals d - 2 (n.d) n; when the tangent
// cannot be normalised (|d - (n.d) n|^2 < 1e-8: the ray runs along the normal) it flips the ray.
// `tangent` = d - (n.d) n is shared with refract_dir.
RTFS_HD float3 reflect_dir(float3 n, float3 d, float nd, float3 tangent) {
    if (fabsf(dot(tangent, tangent)) < kTolF) return -d;
    float3 r = fma3(-nd, n, tangent);
    float3 out;
    if (!unitise(r, out)) return -d; // unreachable: |r| = 1
    return out;
}
// Sphere.refract (Sphere.fs:108-146); `refl` is what reflectWithoutFuzz gives (total internal reflection)
RTFS_HD float3 refract_dir(bool inside, float3 n, float3 d, float3 tangent, float3 refl, float incoming_cos, float ior) {
    float inv_index = inside ? ior : rcp_fast(ior); // 1 / index, index = inside ? 1 / ior : ior (Sphere.fs:118-119)
    float3 tu;
    if (!unitise(tangent, tu)) return d; // parallel to the normal: straight through
    float incoming_sin = sqrt_fast(fmaxf(0.0f, 1.0f - incoming_cos * incoming_cos));
    float outgoing_sin = incoming_sin * inv_index;
    if (fcmp(outgoing_sin, 1.0f) == CMP_GREATER) return refl;
    float outgoing_cos = sqrt_fast(fmaxf(0.0f, 1.0f - outgoing_sin * outgoing_sin));
    float3 v = fma3(outgoing_sin, tu, (-outgoing_cos) * n);
    float3 out;
    if (!unitise(v, out)) return d;
    return out;
}

enum ScatterResult { SCATTER_CONTINUE = 0, SCATTER_ABSORBED = 1, SCATTER_ERROR = 2 };

// Hittable.Reflection (Hittable.fs:8-12) -> Sphere.reflection (Sphere.fs:150-300) /
// InfinitePlane.reflection (InfinitePlane.fs:43-99).  On SCATTER_CONTINUE the ray (o, d) and the colour
// are updated in place; on SCATTER_ABSORBED `colour` is the emitted result.  `inside_out` and `normal_out` (optional) receive
// the inside flag and the shading normal, oriented against the ray (F10, F11), once they are known.
//
// Written so that a warp whose lanes hit different materials shares as much as possible: one normal /
// inside computation, one colour update, ONE block of the counter RNG for whichever style draws
// (Lambert and Fuzzed: GetThree; Dielectric and Glass: Get — always the first block of the bounce), one
// reflection, and a common "unit(base + scale * offset)" tail; only the few style-specific lines diverge.
template <int SMEM, class Rng>
RTFS_HD ScatterResult scatter(const SceneAccess<SMEM> &sc, int prim, int last, float3 &o, float3 &d, float3 strike, uint32_t &colour,
                              Rng &rng, bool *inside_out, float3 *normal_out = nullptr) {
    const Material m = load_material(sc, prim);
    const bool is_plane = (m.flags & 2u) != 0;
    const bool flipped = (m.flags & 1u) != 0;
    const uint32_t style = m.style;

    // ---- normal and inside flag: Sphere.fs:162-182 (F10); planes use their normal unflipped (F11) ----
    float3 n;
    bool inside = false;
    if (is_plane) {
        const DUnbounded &pl = sc.g.unb[prim - sc.g.n_bounded];
        n = f3(pl.n[0], pl.n[1], pl.n[2]);
    } else {
        Cmp where;
        if (prim < sc.g.n_bounded) {
            float4 s = sc.sphere(prim);
            float3 v = f3(strike.x - s.x, strike.y - s.y, strike.z - s.z);
            if (!unitise(v, n)) return SCATTER_ERROR; // Sphere.normal's ValueOption.get
            float3 co = f3(s.x - o.x, s.y - o.y, s.z - o.z);
            where = (prim == last) ? CMP_EQUAL : fcmp(dot(co, co), s.w * s.w);
        } else {
            const DUnbounded &u = sc.g.unb[prim - sc.g.n_bounded];
            if (SceneAccess<SMEM>::kLean || u.fp32) {
                // strike - C rounds at the size of the sphere (~6e-5 for r = 1000): 6e-8 of the normal's direction;
                // inside / outside is the sign of the expanded |o - C|^2 - r^2 (Float.compare's 1e-8 band kept)
                float3 vf = f3(strike.x - u.n[0], strike.y - u.n[1], strike.z - u.n[2]);
                if (!unitise(vf, n)) return SCATTER_ERROR;
                const float c = big_sphere_c(o, u);
                where = (prim == last || fabsf(c) < kTolF) ? CMP_EQUAL : (c < 0.0f ? CMP_LESS : CMP_GREATER);
            } else {
                D3 c{u.p[0], u.p[1], u.p[2]};
                D3 v = d3(strike) - c;
                float3 vf = f3(float(v.x), float(v.y), float(v.z)); // the subtraction is what needs FP64 (|c| ~ 1000)
                if (!unitise(vf, n)) return SCATTER_ERROR;
                D3 co = c - d3(o);
                where = (prim == last) ? CMP_EQUAL : fcmp(dot(co, co), u.r2);
            }
        }
        if (where != CMP_GREATER) {
            if (!flipped) { inside = true; n = -n; }
        } else if (flipped) {
            inside = true;
            n = -n;
        }
    }
    if (inside_out) *inside_out = inside;
    if (normal_out) *normal_out = n;

    // ---- emitters ----
    if (style == RT_STYLE_LIGHT_SOURCE) { // Sphere.fs:185-189, InfinitePlane.fs:52-56
        colour = combine(colour, (SceneAccess<SMEM>::kLean || m.texture < 0) ? m.rgb : texture_colour(sc.g, m.texture, strike));
        return SCATTER_ABSORBED;
    }
    if (style == RT_STYLE_LIGHT_SOURCE_CAP) { // Sphere.fs:190-200; p0 = centre.x + (r - r / 4)
        colour = (fcmp(strike.x, m.p0) == CMP_GREATER) ? combine(m.rgb, colour) : kBlack;
        return SCATTER_ABSORBED;
    }
    if (style > RT_STYLE_GLASS || (is_plane && style > RT_STYLE_LAMBERT_REFLECTION)) return SCATTER_ERROR;

    // ---- colour: darken albedo (combine incoming texture), Sphere.fs:203-207 etc., InfinitePlane.fs:40-41 ----
    const uint32_t surface = (SceneAccess<SMEM>::kLean || is_plane || m.texture < 0) ? m.rgb : texture_colour(sc.g, m.texture, strike);
    const uint32_t nc = darken(m.albedo, combine(colour, surface));

    // ---- the bounce's first RNG block, for every style that draws ----
    float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
    if (style != RT_STYLE_PURE_REFLECTION) u = rng.next();

    // ---- mirror direction, for every style but Lambert ----
    const float nd = dot(n, d);
    const float3 tangent = fma3(-nd, n, d);
    float3 refl = d;
    if (style != RT_STYLE_LAMBERT_REFLECTION) refl = reflect_dir(n, d, nd, tangent);

    float3 out = refl;      // PureReflection: Sphere.fs:224-233, InfinitePlane.fs:95-99
    float3 base = n;        // Lambert: unit(n + offset), Sphere.fs:211-220, InfinitePlane.fs:78-86
    float scale = 1.0f;
    bool random_offset = (style == RT_STYLE_LAMBERT_REFLECTION);
    if (style == RT_STYLE_FUZZED_REFLECTION) { // unit(reflected + fuzz * offset), Sphere.fs:89-104 (kept even if it points inwards, F11)
        base = refl;
        scale = m.p0;
        random_offset = true;
    } else if (style == RT_STYLE_DIELECTRIC) { // Sphere.fs:248-267
        if (!(u.x > m.p1)) out = refract_dir(inside, n, d, tangent, refl, nd, m.p0);
    } else if (style == RT_STYLE_GLASS) { // Sphere.fs:269-300
        float incoming_cos = -nd;
        float refr = inside ? rcp_fast(m.p0) : m.p0;
        float param = (1.0f - refr) * rcp_fast(1.0f + refr);
        param = param * param;
        float x = 1.0f - incoming_cos;
        float x2 = x * x;
        float reflection_prob = param + (1.0f - param) * (x2 * x2 * x);
        if (!(u.x < reflection_prob)) out = refract_dir(inside, n, d, tangent, refl, incoming_cos, m.p0);
    }
    if (random_offset) {
        // UnitVector.random (Point.fs:49-59) redraws while |v|^2 < 1e-8; the callers redraw while the sum cannot be
        // normalised — except InfinitePlane's Lambert, which takes one offset and throws (InfinitePlane.fs:86)
        for (;;) {
            float3 offset;
            if (unitise(f3(2.0f * u.x - 1.0f, 2.0f * u.y - 1.0f, 2.0f * u.z - 1.0f), offset)) {
                if (unitise(fma3(scale, offset, base), out)) break;
                if (is_plane && style == RT_STYLE_LAMBERT_REFLECTION) return SCATTER_ERROR;
            }
            u = rng.next();
        }
    }
    colour = nc;
    o = strike;
    d = out;
    return SCATTER_CONTINUE;
}

// ---- one path (Scene.traceOnce :118-155 + Scene.traceRay :93-114) as a state machine -------------------
// `begin` starts a camera sample; `step` performs one hitObject + Reflection and reports whether the
// path ended.  The render kernels call `step` from a single flat loop so that the lanes of a warp stay
// converged on the traversal while their paths are at different bounces (path regeneration).
// Rng: CounterRng, or a generator with the same draws that finds its key and pixel word another way (rtfs_views.cu); it
// has the counter words `bounce` and `retry` and a `next()`.
template <class Rng = CounterRng>
struct PathStateT {
    float3 o, d;
    uint32_t colour;
    int32_t last; // the primitive the ray leaves, as a ref (see ref_of_prim)
    int32_t bounces;
    Rng rng;
};
using PathState = PathStateT<>;
// the camera sample of a path whose generator already holds its key, pixel and sample index
template <class Rng>
RTFS_HD bool path_start(PathStateT<Rng> &p, const DevCamera &cam, int row_idx, int col_idx) {
    p.rng.bounce = 0;
    p.rng.retry = 0;
    float4 u = p.rng.next(); // rand.GetTwo (), Scene.fs:129
    p.colour = kWhite;
    p.last = kNoRef;
    p.bounces = 0;
    int row = cam.max_h - row_idx - 1; // Scene.fs:219
    int col = col_idx - cam.max_w;     // Scene.fs:226
    return camera_ray(cam, row, col, u.x, u.y, p.o, p.d);
}
RTFS_HD bool path_begin(PathState &p, const DevCamera &cam, uint32_t k0, uint32_t k1, int row_idx, int col_idx, uint32_t sample) {
    p.rng.k0 = k0;
    p.rng.k1 = k1;
    p.rng.pixel = uint32_t(row_idx * cam.cols + col_idx);
    p.rng.sample = sample;
    return path_start(p, cam, row_idx, col_idx);
}
// the part of a step that follows hitObject: Reflection, bounce count (Scene.fs:102-114).
// Returns true when the path is finished; `result` is then its Pixel.
template <int SMEM, class Rng>
RTFS_HD bool path_after_hit(PathStateT<Rng> &p, const SceneAccess<SMEM> &sc, const Hit &h, int max_count, uint32_t &result) {
    if (h.prim == kNoPrim) { // the ray goes off into the distance
        result = kBlack;
        return true;
    }
    p.rng.bounce = uint32_t(p.bounces + 1);
    p.rng.retry = 0;
    ScatterResult r = scatter(sc, h.prim, h.ref == p.last ? h.prim : kNoPrim, p.o, p.d, h.strike, p.colour, p.rng, (bool *)nullptr);
    if (r == SCATTER_ABSORBED) {
        result = p.colour;
        return true;
    }
    if (r == SCATTER_ERROR) { // the reference throws here; unreachable on non-degenerate input: Black, and counted
        result = kBlack | kDegenerate;
        return true;
    }
    p.last = h.ref;
    p.bounces += 1;
    if (p.bounces > max_count) { // while bounces <= maxCount, Scene.fs:98; not done => HotPink :114
        result = kHotPink;
        return true;
    }
    return false;
}
// one whole step: hitObject + Reflection; returns true when the path is finished
template <int SMEM, bool COUNT, class Stack, bool WIDE = false, class Rng>
RTFS_HD bool path_step(PathStateT<Rng> &p, const SceneAccess<SMEM> &sc, int max_count, uint32_t &result, TraversalCounters &cn, unsigned lanes,
                       Stack &stack) {
    Hit h = closest_hit_from<SMEM, COUNT, Stack, WIDE>(sc, p.o, p.d, p.last, cn, lanes, stack);
    return path_after_hit<SMEM>(p, sc, h, max_count, result);
}

} // namespace rtfs
