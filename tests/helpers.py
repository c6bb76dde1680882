"""Shared fixtures for the parity tests: seeded scenes, cameras and ray generators."""
import numpy as np

import oracle
from ray_tracing_fsharp_b200 import abi, sample_images
from ray_tracing_fsharp_b200.domain import marshal


def unit(v):
    v = np.asarray(v, float)
    return v / np.sqrt((v * v).sum(-1, keepdims=True))


def random_unit_vectors(rng, n):
    return unit(rng.normal(size=(n, 3)))


def f32(a):
    """Round to FP32-representable doubles, so that the oracle and the device see the same inputs."""
    return np.asarray(a, np.float32).astype(np.float64)


def oracle_camera(spec):
    cam = oracle.camera_make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    cam.bounce_depth = spec.bounce_depth
    return cam


def scene_pair(spec, device=0):
    """(oracle scene, device scene handle, camera) for a SceneSpec."""
    from ray_tracing_fsharp_b200 import native
    hs, ts, keep = marshal(spec.objects)
    osc = oracle.Scene(hs, ts)
    dsc = native.SceneHandle(hs, ts, device, keepalive=keep)
    return osc, dsc, oracle_camera(spec)


def small_random_spheres(n_side=4, seed=3):
    """A reduced RTOW-style scene (same material mix, fewer spheres) for cases the oracle must finish quickly."""
    rng = np.random.default_rng(seed)
    from ray_tracing_fsharp_b200.domain import Colour, Hittable, Pixel, Sphere, SphereStyle, Texture
    objs = []
    for a in range(-n_side, n_side):
        for b in range(-n_side, n_side):
            choice = rng.random()
            centre = (a + 0.9 * rng.random(), 0.2, b + 0.9 * rng.random())
            if choice < 0.6:
                style = SphereStyle.LambertReflection(rng.random() * rng.random(), Texture.Colour(Colour.random(rng)))
            elif choice < 0.8:
                style = SphereStyle.FuzzedReflection(rng.random() / 2 + 0.5, Texture.Colour(Colour.random(rng)), rng.random() / 2)
            elif choice < 0.9:
                style = SphereStyle.Glass(1.0, Texture.Colour(Colour.White), 1.5)
            else:
                style = SphereStyle.Dielectric(0.95, Texture.Colour(Colour.random(rng)), 1.4, 0.8)
            objs.append(Hittable.Sphere(Sphere.make(style, centre, 0.2)))
    objs.append(Hittable.Sphere(Sphere.make(SphereStyle.Glass(1.0, Texture.Colour(Colour.White), 1.5), (0.0, 1.0, 0.0), 1.0)))
    objs.append(Hittable.Sphere(Sphere.make(SphereStyle.PureReflection(1.0, Texture.Colour(Pixel(180, 150, 128))), (2.5, 1.0, 0.0), 1.0)))
    objs.append(Hittable.UnboundedSphere(Sphere.make(SphereStyle.LightSource(Texture.Colour(Pixel(200, 200, 255))), (0.0, 0.0, 0.0), 2000.0)))
    objs.append(Hittable.UnboundedSphere(Sphere.make(SphereStyle.LambertReflection(0.5, Texture.Colour(Colour.White)), (0.0, -1000.0, 0.0),
                                                     1000.0)))
    return sample_images.SceneSpec("reduced RTOW scene", objs, 32, 6.0, 1.5, (8.0, 2.0, -3.0), (0.0, 0.5, 0.0), (0.0, 1.0, 0.0), 60, 40, 50)


# ---- frames rebuilt sample by sample --------------------------------------------------------------------------------------
# Every sample is a pure function of (seed, pixel, sample index), so a frame's accumulators are the sums of the colours a
# tracer (rt_test_trace_samples, or the oracle) gives for the pixel's sample indices.
BATCH = 1 << 24  # paths per tracer call


def sample_moments(tracer, cam, mw, mh, seed, pixels, s_begin, s_end):
    """Per pixel, the colour sums ([n, 3] int64), the sum of r^2 + g^2 + b^2 ([n] int64) and the rays taken, of samples
    s_begin .. s_end - 1."""
    cols = 2 * mw + 1
    m = s_end - s_begin
    sums = np.zeros((len(pixels), 3), np.int64)
    sq = np.zeros(len(pixels), np.int64)
    rays = 0
    if m <= 0 or len(pixels) == 0:
        return sums, sq, rays
    per_call = max(1, BATCH // m)
    smp = np.arange(s_begin, s_end, dtype=np.int32)
    for lo in range(0, len(pixels), per_call):
        pix = pixels[lo:lo + per_call]
        row = np.repeat((pix // cols).astype(np.int32), m)
        col = np.repeat((pix % cols).astype(np.int32), m)
        colour, r = tracer.trace_samples(cam, mw, mh, seed, row, col, np.tile(smp, len(pix)))
        c = colour.astype(np.int64).reshape(len(pix), m, 3)
        sums[lo:lo + len(pix)] = c.sum(1)
        sq[lo:lo + len(pix)] = (c * c).sum((1, 2))
        rays += int(r.sum(dtype=np.int64))
    return sums, sq, rays


def expected_sums(tracer, cam, max_w, max_h, seed, adaptive, pixels):
    """What the frame's accumulators of the flat pixel ids `pixels` must hold: ([n, 4] int64 sums with the count in the last
    column, the per-pixel count, the rays of all those samples).  renderPixel's rule (Scene.fs:157-194) exactly as fill_frame /
    probe_flags_kernel and the oracle's render_pixel apply it: samples 0 .. firstTrial give the old mean, samples
    0 .. 2 firstTrial the new one; a pixel whose truncated means differ takes samples up to spp - 1, if there are more."""
    pixels = np.asarray(pixels, np.int64)
    spp = int(cam.samples_per_pixel)
    if adaptive:
        ft = min(5, spp // 2)
        n_probe = 2 * ft + 1
        a, _, rays_a = sample_moments(tracer, cam, max_w, max_h, seed, pixels, 0, ft + 1)
        b, _, rays_b = sample_moments(tracer, cam, max_w, max_h, seed, pixels, ft + 1, n_probe)
        s = a + b
        flagged = (np.abs(s // n_probe - a // (ft + 1)).sum(1) != 0) & (spp > n_probe)
        more, _, rays_c = sample_moments(tracer, cam, max_w, max_h, seed, pixels[flagged], n_probe, spp)
        s[flagged] += more
        count = np.where(flagged, spp, n_probe)
        rays = rays_a + rays_b + rays_c
    else:
        s, _, rays = sample_moments(tracer, cam, max_w, max_h, seed, pixels, 0, spp)
        count = np.full(len(pixels), spp, np.int64)
    return np.concatenate([s, count[:, None]], 1), count, rays


def expected_moments(tracer, cam, mw, mh, seed, adaptive, pixels, samples_done):
    """([n, 4] sums with the count, [n] Q) of the flat pixel ids `pixels` in a frame of cam.samples_per_pixel that has reached
    samples_done.  renderPixel's rule: samples 0 .. firstTrial give the old mean, 0 .. 2 firstTrial the new one; a frame keeps
    the raw "means differ" flags, and a flagged pixel holds sample indices 0 .. samples_done - 1."""
    pixels = np.asarray(pixels, np.int64)
    spp = int(cam.samples_per_pixel)
    if adaptive:
        ft = min(5, spp // 2)
        n_probe = 2 * ft + 1
        a, qa, _ = sample_moments(tracer, cam, mw, mh, seed, pixels, 0, ft + 1)
        b, qb, _ = sample_moments(tracer, cam, mw, mh, seed, pixels, ft + 1, n_probe)
        s, q = a + b, qa + qb
        flagged = np.abs(s // n_probe - a // (ft + 1)).sum(1) != 0
        more, qm, _ = sample_moments(tracer, cam, mw, mh, seed, pixels[flagged], n_probe, samples_done)
        s[flagged] += more
        q[flagged] += qm
        count = np.where(flagged, samples_done, n_probe)
    else:
        s, q, _ = sample_moments(tracer, cam, mw, mh, seed, pixels, 0, samples_done)
        count = np.full(len(pixels), samples_done, np.int64)
    return np.concatenate([s, count[:, None]], 1), q


def camera_sample_rays(spec, cam, rng, n):
    """Primary rays of random pixels as the oracle generates them: FP32-representable origins, unit directions in
    double (the oracle's formulas assume |d| = 1 to double precision, as the reference's UnitVector guarantees; the
    device receives the same direction rounded to FP32)."""
    row = rng.integers(-spec.max_height_coord - 1, spec.max_height_coord, n).astype(np.int32)
    col = rng.integers(-spec.max_width_coord, spec.max_width_coord + 1, n).astype(np.int32)
    o, d = oracle.camera_rays(cam, spec.max_width_coord, spec.max_height_coord, row, col, rng.random(n), rng.random(n))
    return f32(o), d


def fp32_safe_closest_hit(hittables, o, d, win_prim, win_t, chunk=2000):
    """Which rays have a closest-primitive decision that FP32 cannot legitimately flip?  Brute force over every object
    of the scene in double precision (no tree), same pattern as the per-primitive sphere test:

      * no object is grazed by the ray: a sphere whose discriminant is within 1e-3 r^2 of zero, or a plane met at
        |n.d| < 1e-4, may flip between hit and miss in FP32 — unless the root it would produce lies beyond the winner
        by more than 1 %, in which case the flip cannot change the answer;
      * the ray does not start within 1 % of the surface of a bounded sphere (the t ~ 0 cancellation regime), nor within
        1e-4 of an unbounded one (whose quadratic the device evaluates in FP64);
      * the winning t leads every other candidate root by more than 1e-4 relative.

    `win_prim`, `win_t`: the oracle's answer (prim < 0: nothing hit).  Bounded spheres of negative radius are never hit
    (F16) and are ignored.  Returns a boolean mask over the rays."""
    shape = np.array([h.shape for h in hittables])
    p = np.array([[h.p[0], h.p[1], h.p[2]] for h in hittables])
    nrm = np.array([[h.n[0], h.n[1], h.n[2]] for h in hittables])
    r = np.array([h.radius for h in hittables])
    is_plane = shape == abi.RT_SHAPE_INFINITE_PLANE
    bounded = shape == abi.RT_SHAPE_SPHERE
    ignore = bounded & (r < 0)
    o, d = np.asarray(o, float), np.asarray(d, float)
    safe = np.ones(len(o), bool)
    for lo in range(0, len(o), chunk):
        oo, dd = o[lo:lo + chunk, None, :], d[lo:lo + chunk, None, :]
        tw = np.where(win_prim[lo:lo + chunk] >= 0, win_t[lo:lo + chunk], np.inf)[:, None]
        oc = oo - p[None]
        b = (dd * oc).sum(2)
        dist2 = (oc * oc).sum(2)
        disc = b * b - (dist2 - r * r)
        root = np.sqrt(np.maximum(disc, 0.0))
        t1, t2 = -b - root, -b + root
        # candidate roots of every sphere: the positive ones (1e-8 as Float.positive)
        cand = np.where(t1 > 1e-8, t1, np.where(t2 > 1e-8, t2, np.inf))
        cand = np.where(disc < 0, np.inf, cand)
        grazing = np.abs(disc) <= 1e-3 * r * r
        would_be = np.abs(b)  # where a grazed sphere's root would lie
        near = np.where(bounded, np.abs(np.sqrt(dist2) - np.abs(r)) <= 1e-2 * np.abs(r), np.abs(np.sqrt(dist2) - np.abs(r)) <= 1e-4)
        den = (dd * nrm[None]).sum(2)
        with np.errstate(divide="ignore", invalid="ignore"):
            tp = ((p[None] - oo) * nrm[None]).sum(2) / den
        plane_graze = np.abs(den) < 1e-4
        plane_cand = np.where((np.abs(den) >= 1e-8) & (tp > 1e-8), tp, np.inf)
        cand = np.where(is_plane, plane_cand, cand)
        grazing = np.where(is_plane, plane_graze, grazing)
        would_be = np.where(is_plane, np.where(np.isfinite(tp), np.abs(tp), 0.0), would_be)
        near = np.where(is_plane, np.abs(((oo - p[None]) * nrm[None]).sum(2)) <= 1e-4, near)
        cand = np.where(ignore, np.inf, cand)
        dangerous_graze = grazing & ~ignore & (would_be < 1.01 * tw)
        near = near & ~ignore
        srt = np.sort(cand, axis=1)
        first, second = srt[:, 0], srt[:, 1] if cand.shape[1] > 1 else np.full(len(srt), np.inf)
        lead = np.where(np.isfinite(first), (second - first) > 1e-4 * first, True)
        safe[lo:lo + chunk] = ~dangerous_graze.any(1) & ~near.any(1) & lead
    return safe
