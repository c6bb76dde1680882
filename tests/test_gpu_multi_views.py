"""Batches of views split over several GPUs (rt_multi_render_views, rt_multi_frame_begin_views, MultiHandle.render_views and
open_frame_views, Scene.render_views and render_views_progressive on a scene made with devices=[...]) against the batch of
one GPU (SceneHandle.render_views, open_frame_views) of the same scene, cameras, seeds, flags and rule.  Every comparison is
np.array_equal or equality of struct fields.
Worlds of 1, 2, 3 and max(4, visible devices) ranks run on any machine: ranks share devices where fewer GPUs are visible
(RTFS_MULTI_SHARE_DEVICES), each with its own replica, workspace, stream, buffers and table of views.
Cases: C1, C1 at 19 x 11 (rows % 4 != 0, so probe tiles straddle two views), C2 at full size with the early-out on and off,
C4, C5 at reduced size and a scene one sphere past the staging limit; seeds per view and none; NO_SMEM, WIDE_BVH and NO_LEAN;
batches of one view; pass shapes, extension, convergence rules, view_noise over more than 1 024 views, features and
denoising; interleaving with other work on the same RtMulti; refusals; the Python wrappers."""
import ctypes as C

import numpy as np
import pytest

from ray_tracing_fsharp_b200 import abi, native
from ray_tracing_fsharp_b200.scene import Image, Scene

from test_gpu_multi_progressive import PROGRESS, assert_same, camera, devices, extents, fields, lockstep, multi, run_to_end, shared, single, spec_of
from test_gpu_views import orbit

pytestmark = pytest.mark.gpu

NOISE = abi.RT_FLAG_NOISE
WORLDS = [1, 2, 3, "all"]
STATS = ("paths", "rays", "degenerate_paths", "pixels_early_out")


def cameras(name, n, spp=None):
    """A turntable of n cameras of the scene, at its samples per pixel or `spp`."""
    spec = spec_of(name)
    cams = orbit(spec, n)
    for c in cams:
        c.samples_per_pixel = spp or spec.spp
        c.bounce_depth = spec.bounce_depth
    return cams


def seeds_of(n):
    return [1000 + 7 * v for v in range(n)]


def check_render_views(name, world, n, seeds, adaptive=True, flags=0, spp=None):
    """rt_multi_render_views over the world against rt_render_views on one device: sums, RGB8, gamma RGB8 and the counts."""
    cams, (mw, mh) = cameras(name, n, spp), extents(name)
    mh_ = multi(name, devices(world))
    kw = dict(seeds=seeds, seed=5, adaptive=adaptive, flags=flags)
    rgb, sums, st = mh_.render_views(cams, mw, mh, want_sums=True, **kw)
    ref_rgb, ref_sums, ref_st = single(name).render_views(cams, mw, mh, want_sums=True, **kw)
    assert rgb.shape == ref_rgb.shape == (n, 2 * mh + 1, 2 * mw + 1, 3)
    assert np.array_equal(sums, ref_sums)
    assert np.array_equal(rgb, ref_rgb)
    assert np.array_equal(mh_.render_views(cams, mw, mh, gamma=True, **kw)[0], single(name).render_views(cams, mw, mh, gamma=True, **kw)[0])
    assert fields(st, STATS) == fields(ref_st, STATS)
    assert st.box_tests == 0 and st.prim_tests == 0 and st.kernel_ms > 0.0
    return cams


# ---- one call ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("name,n,adaptive", [("C1", 5, True), ("C1-odd", 6, True), ("C1-odd", 6, False), ("C2", 2, True), ("C2", 2, False),
                                             ("C4", 3, True), ("C5", 2, True), ("stage-n*+1", 3, True)])
def test_render_views_scene_families(name, n, adaptive, world):
    check_render_views(name, world, n, seeds_of(n), adaptive=adaptive)


@pytest.mark.parametrize("world", WORLDS)
def test_render_views_one_seed_for_every_view(world):
    check_render_views("C1", world, 4, None)


@pytest.mark.parametrize("world", [1, 2, "all"])
@pytest.mark.parametrize("flag", ["no-smem", "wide-bvh", "no-lean"])
@pytest.mark.parametrize("name", ["C1", "stage-n*+1"])
def test_flags(name, flag, world):
    f = {"no-smem": abi.RT_FLAG_NO_SMEM, "wide-bvh": abi.RT_FLAG_WIDE_BVH, "no-lean": abi.RT_FLAG_NO_LEAN}[flag]
    cams = check_render_views(name, world, 3, seeds_of(3), flags=f)
    (mw, mh), devs = extents(name), devices(world)
    for flags in (f, f | NOISE):
        a = single(name).open_frame_views(cams, mw, mh, seeds=seeds_of(3), flags=flags)
        b = multi(name, devs).open_frame_views(cams, mw, mh, seeds=seeds_of(3), flags=flags)
        with a, b:
            lockstep(a, b, [4, 0])


@pytest.mark.parametrize("world", WORLDS)
def test_single_view(world):
    """A batch of one view is rt_multi_render (and rt_multi_frame_begin) of its camera and seed; one view of a batch is
    rt_render of its camera and seed."""
    name = "C1"
    cams, (mw, mh), mh_ = cameras(name, 3), extents(name), multi(name, devices(world))
    rgb, sums, st = mh_.render_views(cams[1:2], mw, mh, seeds=[77], want_sums=True)
    one_rgb, one_sums, one_st = mh_.render(cams[1], mw, mh, seed=77, want_sums=True)
    assert np.array_equal(sums[0], one_sums) and np.array_equal(rgb[0], one_rgb)
    assert fields(st, STATS) == fields(one_st, STATS)
    _, batch_sums, _ = mh_.render_views(cams, mw, mh, seeds=seeds_of(3), want_sums=True)
    for v in range(3):
        _, ref, _ = single(name).render(cams[v], mw, mh, seed=seeds_of(3)[v], want_sums=True)
        assert np.array_equal(batch_sums[v], ref), v
    with mh_.open_frame_views(cams[1:2], mw, mh, seeds=[77], flags=NOISE) as a, mh_.open_frame(cams[1], mw, mh, seed=77, flags=NOISE) as b:
        for k in (5, 0):
            a.advance(k)
            b.advance(k)
            assert fields(a.progress, PROGRESS) == fields(b.progress, PROGRESS)
            (ra, sa), (rb, sb) = a.read(want_sums=True), b.read(want_sums=True)
            assert np.array_equal(sa[0], sb) and np.array_equal(ra[0], rb)
            (na, ea, qa), (nb, eb, qb) = a.noise(1.0, want_sq=True), b.noise(1.0, want_sq=True)
            assert fields(na) == fields(nb) and np.array_equal(ea[0], eb) and np.array_equal(qa[0], qb)


# ---- progressive frames -----------------------------------------------------------------------------------------------------
def open_pair(name, world, n=3, spp=None, seeds=None, adaptive=True, flags=NOISE):
    """(batch frame of one device, batch frame over the world's devices) of the same cameras, seeds and flags."""
    cams, (mw, mh) = cameras(name, n, spp), extents(name)
    seeds = seeds_of(n) if seeds is None else seeds
    a = single(name).open_frame_views(cams, mw, mh, seeds=seeds, adaptive=adaptive, flags=flags)
    b = multi(name, devices(world)).open_frame_views(cams, mw, mh, seeds=seeds, adaptive=adaptive, flags=flags)
    return a, b


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("name,n,adaptive,flags", [("C1", 3, True, NOISE), ("C1-odd", 5, True, NOISE), ("C1-odd", 5, False, 0), ("C2", 2, True, NOISE),
                                                   ("C2", 2, False, 0), ("C4", 3, True, NOISE), ("C5", 2, True, NOISE),
                                                   ("stage-n*+1", 3, True, NOISE)])
def test_progressive_scene_families(name, n, adaptive, flags, world):
    a, b = open_pair(name, world, n=n, adaptive=adaptive, flags=flags)
    with a, b:
        assert_same(a, b)
        lockstep(a, b, [5, 3, 0])


@pytest.mark.parametrize("world", WORLDS)
def test_progressive_one_seed_for_every_view(world):
    name = "C1"
    cams, (mw, mh) = cameras(name, 3), extents(name)
    a = single(name).open_frame_views(cams, mw, mh, seed=9, flags=NOISE)
    b = multi(name, devices(world)).open_frame_views(cams, mw, mh, seed=9, flags=NOISE)
    with a, b:
        lockstep(a, b, [6, 0])


@pytest.mark.parametrize("world", WORLDS)
def test_pass_shapes_end_in_the_same_batch(world):
    name, spp = "C1", 160
    cams, (mw, mh) = cameras(name, 3, spp), extents(name)
    with single(name).open_frame_views(cams, mw, mh, seeds=seeds_of(3), flags=NOISE) as ref:
        sums, (noise, se, sq), progress = run_to_end(ref, "unpaced")
        per_view = [fields(x) for x in ref.view_noise(1.0)]
    for shape in (1, 7, 64, "paced", "unpaced"):
        with multi(name, devices(world)).open_frame_views(cams, mw, mh, seeds=seeds_of(3), flags=NOISE) as f:
            if shape == 1:
                for _ in range(3):  # windows of one sample index: every rank but the first idles
                    f.advance(1)
            s, (nz, e, q), p = run_to_end(f, shape)
            assert np.array_equal(s, sums) and np.array_equal(q, sq) and np.array_equal(e, se), shape
            assert fields(nz) == fields(noise) and fields(p, PROGRESS) == fields(progress, PROGRESS), shape
            assert [fields(x) for x in f.view_noise(1.0)] == per_view, shape


@pytest.mark.parametrize("world", [1, 2, "all"])
def test_extension_equals_a_batch_opened_at_the_target(world):
    name = "C1"
    (mw, mh), devs = extents(name), devices(world)
    with multi(name, devs).open_frame_views(cameras(name, 3, 256), mw, mh, seeds=seeds_of(3), flags=NOISE) as f, \
            single(name).open_frame_views(cameras(name, 3, 512), mw, mh, seeds=seeds_of(3), flags=NOISE) as ref:
        f.advance(100)
        f.extend(512)
        f.advance()
        ref.advance()
        assert_same(ref, f)


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("tau,m,k", [(0.0, 64, 64), (0.5, 64, 64), (1.0, 64, 64), (1.0, 37, 23)])
def test_convergence(tau, m, k, world):
    name = "C1"
    a, b = open_pair(name, world, n=3, spp=256)
    with a, b:
        a.set_convergence(tau, m, k)
        b.set_convergence(tau, m, k)
        while not b.progress.done:
            a.advance(40)
            b.advance(40)
            assert_same(a, b, tol=tau)
        assert a.progress.done


@pytest.mark.parametrize("world", [2, "all"])
def test_view_noise_of_more_views_than_one_chunk(world):
    """1 500 views of 3 x 3 pixels: rt_frame_view_noise reduces them in two chunks of views."""
    name, n = "C1", 1500
    cams, seeds = cameras(name, n), [3 * v + 1 for v in range(n)]
    a = single(name).open_frame_views(cams, 1, 1, seeds=seeds, adaptive=False, flags=NOISE)
    b = multi(name, devices(world)).open_frame_views(cams, 1, 1, seeds=seeds, adaptive=False, flags=NOISE)
    with a, b:
        for k in (3, 0):
            a.advance(k)
            b.advance(k)
            va, vb = a.view_noise(2.0), b.view_noise(2.0)
            assert len(vb) == n and [fields(x) for x in va] == [fields(x) for x in vb]
            assert np.array_equal(a.read(want_sums=True)[1], b.read(want_sums=True)[1])


@pytest.mark.parametrize("world", [1, 2, "all"])
def test_features_and_denoise(world):
    other = dict(iterations=5, feature_samples=1, sigma_colour=2.0, sigma_normal=0.3, sigma_albedo=8.0, sigma_depth=0.1, gamma=True)
    a, b = open_pair("C1-odd", world, n=4, spp=64)
    with a, b:
        for calls in ([], [20], [0]):
            lockstep(a, b, calls)
            for samples in (1, 4):
                for x, y in zip(a.features(samples), b.features(samples)):
                    assert np.array_equal(x, y), samples
            for opts in ({}, other):
                for x, y in zip(a.denoise(want_linear=True, **opts), b.denoise(want_linear=True, **opts)):
                    assert np.array_equal(x, y), opts


@pytest.mark.parametrize("world", [1, 2, "all"])
def test_interleaving_with_other_work_on_the_multi(world):
    """rt_multi_render, rt_multi_render_views and a second frame run on the RtMulti between the batch frame's passes."""
    name = "C1"
    cams, (mw, mh) = cameras(name, 3, 48), extents(name)
    mh_ = multi(name, devices(world))
    a, b = open_pair(name, world, n=3, spp=48)
    with a, b:
        lockstep(a, b, [6])
        _, sums, _ = mh_.render(cams[0], mw, mh, seed=4, want_sums=True)
        assert np.array_equal(sums, single(name).render(cams[0], mw, mh, seed=4, want_sums=True)[1])
        lockstep(a, b, [6])
        # a batch of other views: the one-call path rewrites its own tables, not the frame's
        other_cams = cameras(name, 5, 48)
        _, sums, _ = mh_.render_views(other_cams, mw, mh, seeds=seeds_of(5), want_sums=True)
        assert np.array_equal(sums, single(name).render_views(other_cams, mw, mh, seeds=seeds_of(5), want_sums=True)[1])
        second = mh_.open_frame_views(other_cams, mw, mh, seeds=seeds_of(5))
        second.advance(10)
        lockstep(a, b, [6])
        second.close()  # destroyed mid-way
        lockstep(a, b, [0])


def test_refusals():
    name = "C1"
    cams, (mw, mh) = cameras(name, 2), extents(name)
    mh_ = multi(name, devices(1))
    lib = native.lib()
    arr = (abi.RtCamera * 2)(*cams)
    rgb = np.empty((2, 2 * mh + 1, 2 * mw + 1, 3), np.uint8)
    rgb_p = C.c_void_p(rgb.ctypes.data)

    def both(cams_arr, n, mw_, mh_coord, opts, code, what):
        assert lib.rt_multi_render_views(mh_.ptr, cams_arr, None, n, mw_, mh_coord, C.byref(opts), rgb_p, None, None) == code, what
        out = C.c_void_p(12345)
        assert lib.rt_multi_frame_begin_views(mh_.ptr, cams_arr, None, n, mw_, mh_coord, C.byref(opts), C.byref(out), None) == code, what
        assert out.value is None, what

    for mode, flags, code in [(abi.RT_MODE_WAVEFRONT, 0, abi.RT_ERR_UNSUPPORTED), (abi.RT_MODE_MEGAKERNEL, abi.RT_FLAG_FLOW, abi.RT_ERR_UNSUPPORTED),
                              (abi.RT_MODE_MEGAKERNEL, abi.RT_FLAG_COUNTERS, abi.RT_ERR_UNSUPPORTED),
                              (abi.RT_MODE_MEGAKERNEL, NOISE | abi.RT_FLAG_FLOW, abi.RT_ERR_UNSUPPORTED), (7, 0, abi.RT_ERR_INVALID_ARGUMENT)]:
        both(arr, 2, mw, mh, abi.RtRenderOpts(1, 1, mode, 0, flags), code, (mode, flags))
    opts = abi.RtRenderOpts(1, 1, abi.RT_MODE_MEGAKERNEL, 0, 0)
    both(arr, 0, mw, mh, opts, abi.RT_ERR_INVALID_ARGUMENT, "no views")
    both(None, 2, mw, mh, opts, abi.RT_ERR_INVALID_ARGUMENT, "null cameras")
    both(arr, 2, 0, mh, opts, abi.RT_ERR_INVALID_ARGUMENT, "bad extents")
    for field, value in (("samples_per_pixel", cams[0].samples_per_pixel + 1), ("bounce_depth", cams[0].bounce_depth + 1)):
        odd = (abi.RtCamera * 2)(*cams)
        setattr(odd[1], field, value)
        both(odd, 2, mw, mh, opts, abi.RT_ERR_INVALID_ARGUMENT, field)
    many = (abi.RtCamera * 600)(*([cams[0]] * 600))  # 600 x 2001 x 2001 pixels >= 2^31
    both(many, 600, 1000, 1000, opts, abi.RT_ERR_INVALID_ARGUMENT, "2^31")
    assert lib.rt_multi_render_views(mh_.ptr, arr, None, 2, mw, mh, C.byref(opts), None, None, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_multi_frame_begin_views(mh_.ptr, arr, None, 2, mw, mh, C.byref(opts), None, None) == abi.RT_ERR_INVALID_ARGUMENT
    with mh_.open_frame_views(cams, mw, mh) as f:  # no RT_FLAG_NOISE: the noise calls refuse the frame
        for call in (lambda: f.noise(1.0), lambda: f.view_noise(1.0), lambda: f.set_convergence(1.0), lambda: f.denoise()):
            with pytest.raises(native.RtError) as e:
                call()
            assert e.value.code == abi.RT_ERR_INVALID_ARGUMENT


# ---- the Python wrappers ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, "all"])
def test_scene_render_views_on_several_devices(world):
    spec = spec_of("C1")
    (mw, mh), n = extents("C1"), 3
    cams = cameras("C1", n, 48)
    one = Scene.make(spec.objects, device=0)
    with shared(devices(world)):
        several = Scene.make(spec.objects, devices=list(devices(world)))
    assert isinstance(several.handle, native.MultiHandle)
    ticks = {"one": 0, "several": 0}

    def tick(which):
        def f(_):
            ticks[which] += 1
        return f

    total_a, ref = Scene.render_views(tick("one"), print, mw, mh, cams, one, seeds=seeds_of(n))
    total_b, got = Scene.render_views(tick("several"), print, mw, mh, cams, several, seeds=seeds_of(n))
    assert total_a == total_b == float((2 * mh + 1) * n)
    for x, y in zip(ref, got):
        assert np.array_equal(Image.render(x), Image.render(y))
    assert ticks == {"one": (2 * mh + 1) * n, "several": (2 * mh + 1) * n}
    for kw in (dict(), dict(converge_tolerance=1.0, converge_min_samples=32, converge_interval=16)):
        ticks = {"one": 0, "several": 0}
        passes = []
        ref = Scene.render_views_progressive(tick("one"), print, mw, mh, cams, one, seeds=seeds_of(n), target_ms=1.0, **kw)
        got = Scene.render_views_progressive(tick("several"), print, mw, mh, cams, several, seeds=seeds_of(n), target_ms=1.0,
                                             on_pass=lambda p, fr: passes.append(p.samples_done), **kw)
        assert all(np.array_equal(x, y) for x, y in zip(ref, got)), kw
        assert ticks == {"one": (2 * mh + 1) * n, "several": (2 * mh + 1) * n}
        assert passes
