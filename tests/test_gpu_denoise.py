"""Denoised previews of progressive frames (rt_frame_features, rt_frame_denoise, Frame.features, Frame.denoise).
Features are rebuilt sample by sample from the conformance entry points (rt_test_rng for the camera draws, rt_test_camera_rays,
rt_test_hit_object with traversal 0, rt_test_reflection with a white colour): prim, albedo and depth EXACTLY, normals within
1e-5 (the entry points give the inside flag, and the normal is restated from the scene's geometry).  The filter must EQUAL
tests/denoise_rule.py run on the frame's own sums, Q and features, and must leave the frame as it was.  Cases: C1-C5 and a
scene one sphere past the staging limit; F = 1 and 4; passes, pacing, a convergence rule and extension; windows (the crop of
the frame's features) and batches of views (each view as the frame of its camera and seed); the early-out on and off; gamma;
interleaving with rt_render and another frame.  A sanity check: on C2 at 16 spp the denoised image is closer to a 1024-spp
frame of another seed than the raw one is."""
import numpy as np
import pytest

from ray_tracing_fsharp_b200 import abi, native
from ray_tracing_fsharp_b200.domain import marshal

import denoise_rule
from test_gpu_views import device_scene, orbit

pytestmark = pytest.mark.gpu

NOISE = abi.RT_FLAG_NOISE
OPTS = dict(iterations=3, feature_samples=4, sigma_colour=4.0, sigma_normal=0.1, sigma_albedo=16.0, sigma_depth=0.02)


def camera(spec, spp=None):
    cam = orbit(spec, 1)[0]
    if spp is not None:
        cam.samples_per_pixel = spp
    return cam


def expected_features(spec, dsc, cam, seed, R, C, samples):
    """(prim, albedo, normal, depth) of frame pixels (R, C), rebuilt from the conformance entry points."""
    mw, mh = spec.max_width_coord, spec.max_height_coord
    hs, _, _ = marshal(spec.objects)
    n = len(R)
    word = (R * (2 * mw + 1) + C).astype(np.uint32)
    zeros = np.zeros(n, np.uint32)
    albedo = np.zeros((n, 3), np.int64)
    nsum = np.zeros((n, 3), np.float32)
    tsum = np.zeros(n, np.float32)
    hits = np.zeros(n, np.int64)
    prim0 = None
    for s in range(samples):
        smp = np.full(n, s, np.uint32)
        _, u = native.rng(seed, word, smp, zeros, zeros)
        o, d = native.camera_rays(cam, mw, mh, (mh - R - 1).astype(np.int32), (C - mw).astype(np.int32), u[:, 0], u[:, 1])
        prim, t, strike = dsc.hit_object(o, d, traversal=0)
        if s == 0:
            prim0 = prim.copy()
        hit = prim >= 0
        if not hit.any():
            continue
        _, u1 = native.rng(seed, word[hit], smp[hit], zeros[hit] + 1, zeros[hit])
        white = np.full((int(hit.sum()), 3), 255, np.uint8)
        code, colour, _, _, inside = dsc.reflection(prim[hit], o[hit], d[hit], strike[hit], white, u1)
        colour = np.where((code == 2)[:, None], 0, colour)  # a scatter that fails: black
        albedo[hit] += colour
        # the outward normal as scatter forms it, in float32: the plane's normal, or unit(strike - centre)
        outward = np.zeros((int(hit.sum()), 3), np.float32)
        for k, (p, st) in enumerate(zip(prim[hit], strike[hit])):
            h = hs[int(p)]
            if h.shape == abi.RT_SHAPE_INFINITE_PLANE:
                outward[k] = np.asarray(h.n[:], np.float32)
            else:
                v = st.astype(np.float32) - np.asarray(h.p[:], np.float32)
                outward[k] = v / np.sqrt(np.float32(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]))
        nrm = np.where(inside[:, None] == 1, -outward, outward).astype(np.float32)
        nsum[hit] = nsum[hit] + nrm
        tsum[hit] = tsum[hit] + t[hit].astype(np.float32)
        hits += hit
    fh = hits.astype(np.float32)
    with np.errstate(all="ignore"):
        normal = np.where(hits[:, None] > 0, nsum / fh[:, None], np.float32(0))
        depth = np.where(hits > 0, tsum / fh, np.float32(np.inf))
    return prim0, (albedo // samples).astype(np.uint8), normal, depth.astype(np.float32)


# ---- 1. features against the conformance entry points ---------------------------------------------------------------------
@pytest.mark.parametrize("samples", [1, 4])
@pytest.mark.parametrize("name", ["C1", "C2", "C3", "C4", "C5", "stage-n*+1"])
def test_features_match_the_entry_points(name, samples):
    spec, dsc = device_scene(name)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    rows, cols = 2 * mh + 1, 2 * mw + 1
    cam = camera(spec)
    seed = 2 ** 64 - 5
    frame = dsc.open_frame(cam, mw, mh, seed=seed)
    prim, albedo, normal, depth = frame.features(samples)
    assert prim.shape == (rows, cols) and albedo.shape == (rows, cols, 3) and normal.shape == (rows, cols, 3) and depth.shape == (rows, cols)
    pix = np.arange(0, rows * cols, max(1, rows * cols // 1500) | 1)
    R, C = pix // cols, pix % cols
    e_prim, e_albedo, e_normal, e_depth = expected_features(spec, dsc, cam, seed, R, C, samples)
    assert np.array_equal(prim[R, C], e_prim)
    assert np.array_equal(albedo[R, C], e_albedo)
    assert np.array_equal(depth[R, C], e_depth)
    assert np.abs(normal[R, C] - e_normal).max() <= 1e-5
    assert (prim >= 0).any() and (albedo > 0).any()
    frame.close()


# ---- 2. features do not depend on passes ----------------------------------------------------------------------------------
def test_features_are_the_same_before_and_after_passes():
    spec, dsc = device_scene("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    frame = dsc.open_frame(camera(spec, 64), mw, mh, seed=3, flags=NOISE)
    frame.set_convergence(2.0, 16, 16)
    before = {f: frame.features(f) for f in (1, 4)}
    frame.advance(max_samples=5)
    assert all(np.array_equal(a, b) for a, b in zip(frame.features(4), before[4]))
    while not frame.advance(max_samples=7).done:
        pass
    assert frame.convergence().checks > 0
    frame.extend(128)
    frame.advance()
    for f in (1, 4, 1):  # recomputed whenever F changes
        assert all(np.array_equal(a, b) for a, b in zip(frame.features(f), before[f])), f
    frame.close()


def test_window_features_are_the_crop():
    spec, dsc = device_scene("C3")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cam = camera(spec)
    full = dsc.open_frame(cam, mw, mh, seed=9).features(4)
    for w in [(5, 7, 20, 30), (0, 0, 1, 1), (2 * mh, 2 * mw, 1, 1), (0, 3, 2 * mh + 1, 5)]:
        win = dsc.open_frame_window(cam, mw, mh, w, seed=9)
        for a, b in zip(win.features(4), full):
            assert np.array_equal(a, b[w[0]:w[0] + w[2], w[1]:w[1] + w[3]]), w
        win.close()


def test_view_features_are_those_of_each_camera():
    spec, dsc = device_scene("C4")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cams, seeds = orbit(spec, 3), [5, 2 ** 63 + 1, 7]
    batch = dsc.open_frame_views(cams, mw, mh, seeds=seeds)
    feats = batch.features(4)
    assert feats[0].shape == (3, 2 * mh + 1, 2 * mw + 1)
    for v, cam in enumerate(cams):
        one = dsc.open_frame(cam, mw, mh, seed=seeds[v]).features(4)
        for a, b in zip(feats, one):
            assert np.array_equal(a[v], b), v
    batch.close()


# ---- 3. the filter against the rule ---------------------------------------------------------------------------------------
def check_rule(frame, gamma=False, **opts):
    o = dict(OPTS, **opts)
    rgb, lin = frame.denoise(gamma=gamma, want_linear=True, **o)
    _, sums = frame.read(want_sums=True)
    _, _, sq = frame.noise(0.0, want_map=False, want_sq=True)
    _, albedo, normal, depth = frame.features(o["feature_samples"])
    e_rgb, e_lin = denoise_rule.denoise(sums, sq, albedo, normal, depth, o["iterations"], o["sigma_colour"], o["sigma_normal"],
                                        o["sigma_albedo"], o["sigma_depth"], gamma=gamma)
    assert np.array_equal(lin.view(np.uint32), e_lin.view(np.uint32)), np.argwhere(lin != e_lin)[:5]
    assert np.array_equal(rgb, e_rgb)
    return rgb, lin


def test_denoise_equals_the_rule_on_c2_at_full_size():
    spec, dsc = device_scene("C2")
    frame = dsc.open_frame(camera(spec, 16), spec.max_width_coord, spec.max_height_coord, seed=21, flags=NOISE)
    while not frame.advance(max_samples=6).done:
        pass
    check_rule(frame)
    frame.close()


@pytest.mark.parametrize("adaptive", [True, False])
@pytest.mark.parametrize("name", ["C3", "C4"])
def test_denoise_equals_the_rule_after_passes(name, adaptive):
    spec, dsc = device_scene(name)
    frame = dsc.open_frame(camera(spec, 24), spec.max_width_coord, spec.max_height_coord, seed=4, adaptive=adaptive, flags=NOISE)
    if not adaptive:  # no sample yet: every pixel black
        rgb, lin = check_rule(frame)
        assert not rgb.any() and not lin.any()
    k = 0
    while not frame.progress.done:
        frame.advance(max_samples=5)
        k += 1
        check_rule(frame, gamma=k % 2 == 1, iterations=1 + k % 5, feature_samples=1 + k % 3, sigma_colour=1.0 + k)
    frame.close()


def test_view_denoise_is_the_denoise_of_each_camera():
    spec, dsc = device_scene("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cams, seeds = orbit(spec, 3), [1, 2, 3]
    for c in cams:
        c.samples_per_pixel = 24
    batch = dsc.open_frame_views(cams, mw, mh, seeds=seeds, flags=NOISE)
    batch.advance(max_samples=9)
    rgb, lin = check_rule(batch, gamma=True)
    for v, cam in enumerate(cams):
        one = dsc.open_frame(cam, mw, mh, seed=seeds[v], flags=NOISE)
        one.advance(max_samples=9)
        r1, l1 = one.denoise(gamma=True, want_linear=True, **OPTS)
        assert np.array_equal(rgb[v], r1) and np.array_equal(lin[v].view(np.uint32), l1.view(np.uint32)), v
        one.close()
    batch.close()


def test_window_denoise_equals_the_rule():
    spec, dsc = device_scene("stage-n*+1")
    frame = dsc.open_frame_window(camera(spec), spec.max_width_coord, spec.max_height_coord, (3, 4, 20, 33), seed=8, flags=NOISE)
    frame.advance(max_samples=4)
    check_rule(frame)
    frame.close()


# ---- 4. a denoise leaves the frame as it was ------------------------------------------------------------------------------
def snapshot(frame):
    rgb, sums = frame.read(want_sums=True)
    _, se, sq = frame.noise(0.5, want_map=True, want_sq=True)
    return rgb, sums, sq, se.view(np.uint32)


def test_denoise_leaves_the_frame_as_it_was():
    spec, dsc = device_scene("C3")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cam = camera(spec, 96)
    a = dsc.open_frame(cam, mw, mh, seed=12, flags=NOISE)
    b = dsc.open_frame(cam, mw, mh, seed=12, flags=NOISE)
    for f in (a, b):
        f.set_convergence(1.5, 16, 8)
    while not a.progress.done:
        a.advance(max_samples=6)
        before = snapshot(a)
        a.denoise(**OPTS)
        a.features(2)
        after = snapshot(a)
        assert all(np.array_equal(x, y) for x, y in zip(before, after))
    while not b.advance(max_samples=11).done:
        pass
    assert all(np.array_equal(x, y) for x, y in zip(snapshot(a), snapshot(b)))
    ca, cb = a.convergence(), b.convergence()
    assert (ca.pixels_active, ca.pixels_converged) == (cb.pixels_active, cb.pixels_converged)
    assert np.array_equal(a.denoise(**OPTS)[0], b.denoise(**OPTS)[0])


def test_interleaving_with_render_and_another_frame():
    spec, dsc = device_scene("C4")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cam, cam2 = camera(spec, 32), orbit(spec, 4)[1]
    cam2.samples_per_pixel = 32
    a = dsc.open_frame(cam, mw, mh, seed=1, flags=NOISE)
    b = dsc.open_frame(cam2, mw, mh, seed=2, flags=NOISE)
    while not (a.progress.done and b.progress.done):
        a.advance(max_samples=7)
        dsc.render(cam2, mw, mh, seed=5)
        b.denoise(**OPTS)
        b.advance(max_samples=5)
        a.features(3)
    for f, c, s in ((a, cam, 1), (b, cam2, 2)):
        ref = dsc.open_frame(c, mw, mh, seed=s, flags=NOISE)
        ref.advance()
        assert np.array_equal(f.denoise(want_linear=True, **OPTS)[1], ref.denoise(want_linear=True, **OPTS)[1])
        ref.close()


# ---- 5. the Python surface and its errors ---------------------------------------------------------------------------------
def test_argument_errors():
    spec, dsc = device_scene("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    plain = dsc.open_frame(camera(spec), mw, mh)
    with pytest.raises(native.RtError) as e:
        plain.denoise(**OPTS)
    assert e.value.code == abi.RT_ERR_INVALID_ARGUMENT
    plain.features(64)
    for bad in (0, 65):
        with pytest.raises(native.RtError) as e:
            plain.features(bad)
        assert e.value.code == abi.RT_ERR_INVALID_ARGUMENT
    noisy = dsc.open_frame(camera(spec), mw, mh, flags=NOISE)
    for kw in (dict(iterations=0), dict(iterations=11), dict(feature_samples=65), dict(sigma_depth=float("nan")), dict(sigma_colour=0.0)):
        with pytest.raises(native.RtError) as e:
            noisy.denoise(**dict(OPTS, **kw))
        assert e.value.code == abi.RT_ERR_INVALID_ARGUMENT, kw
    rgb, lin = noisy.denoise()
    assert rgb.shape == (2 * mh + 1, 2 * mw + 1, 3) and lin is None


# ---- 6. sanity: the denoised image is closer to the converged one ----------------------------------------------------------
def rms(a, b):
    d = a.astype(np.float64) - b.astype(np.float64)
    return float(np.sqrt((d * d).mean()))


def test_denoised_c2_is_closer_to_a_converged_frame():
    spec, dsc = device_scene("C2")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    _, ref_sums, _ = dsc.render(camera(spec, 1024), mw, mh, seed=1001, adaptive=False, want_sums=True)
    ref = ref_sums[..., :3] / ref_sums[..., 3:]
    frame = dsc.open_frame(camera(spec, 16), mw, mh, seed=77, adaptive=False, flags=NOISE)
    frame.advance()
    _, sums = frame.read(want_sums=True)
    _, lin = frame.denoise(want_linear=True)
    raw_err, den_err = rms(sums[..., :3] / sums[..., 3:], ref), rms(lin, ref)
    print(f"C2 16 spp: RMS error raw {raw_err:.3f}, denoised {den_err:.3f} (8-bit levels)")
    assert den_err < raw_err
