"""Progressive frames split over several GPUs (rt_multi_frame_begin, MultiHandle.open_frame, Scene.render_progressive on a
scene made with devices=[...]) against the progressive frame of one GPU (SceneHandle.open_frame) of the same scene, camera,
seed, flags and rule, driven with the same max_samples per call.  Every comparison is np.array_equal or equality of struct
fields: sums, RGB8 with and without gamma, Q, the E map, the noise summary, view_noise, every field of RtFrameProgress and
RtFrameConvergence but the _ms fields and passes, the features and the denoised image.
World 1 (an RtMulti of one device) and worlds of 2, 3 and max(4, visible devices) ranks run on any machine: where fewer
GPUs are visible than ranks, ranks share devices (RTFS_MULTI_SHARE_DEVICES), each with its own replica, workspace, stream and
buffers, so the tile-split probe, the exchange kernel over several ranks, the cross-stream event ordering and the pacing run
as they do over several GPUs; only the peer loads then stay on one device.
Cases: C1 and a frame of 19 x 11 (neither side a multiple of the 8 x 4 tile), C2 at full size with the early-out on and off,
C4 (the staged general kernel), C5 at reduced size (the global-memory kernels), a scene one sphere past the staging limit;
NO_SMEM, WIDE_BVH and NO_LEAN; FLOW and COUNTERS without noise; pass shapes (one sample index, so that ranks idle, 7, 64,
paced and unpaced passes) and extension; convergence rules; features and denoising; interleaving with rt_multi_render and a
second frame on the same RtMulti; refusals."""
import contextlib
import ctypes as C
import functools
import os

import numpy as np
import pytest

from ray_tracing_fsharp_b200 import abi, native, sample_images
from ray_tracing_fsharp_b200.domain import marshal
from ray_tracing_fsharp_b200.scene import Scene

from test_gpu_views import _past_staging_limit

pytestmark = pytest.mark.gpu

NOISE = abi.RT_FLAG_NOISE
PROGRESS = ("samples_done", "samples_target", "paths_done", "paths_target", "pixels_flagged", "done")
SPECS = {
    "C1": lambda: sample_images.few_spheres(max_w=40, max_h=21, spp=24),       # 81 x 43
    "C1-odd": lambda: sample_images.few_spheres(max_w=9, max_h=5, spp=24),     # 19 x 11
    "C2": lambda: sample_images.random_spheres(spp=24),                        # full size, 1201 x 801
    "C4": lambda: sample_images.mixed_planes(max_w=48, max_h=27, spp=24),
    "C5": lambda: sample_images.many_spheres(max_w=240, max_h=135, spp=16),    # 100 k spheres, 481 x 271
    "stage-n*+1": _past_staging_limit,
}


def devices(world):
    """The device of each rank of a world of 1, 2 or 3 ranks, or "all": every visible device and at least four ranks.  Ranks
    are spread over the visible devices and share them where there are fewer devices than ranks."""
    n = native.device_count()
    ranks = max(n, 4) if world == "all" else world
    return tuple(r % n for r in range(ranks))


@contextlib.contextmanager
def shared(devs):
    """rt_multi_create accepts repeated device ordinals while this is open (only when the ranks share devices)."""
    share = len(set(devs)) < len(devs)
    if share:
        os.environ["RTFS_MULTI_SHARE_DEVICES"] = "1"
    try:
        yield
    finally:
        if share:
            os.environ.pop("RTFS_MULTI_SHARE_DEVICES", None)


@functools.lru_cache(maxsize=None)
def spec_of(name):
    return SPECS[name]()


@functools.lru_cache(maxsize=None)
def single(name):
    hs, ts, keep = marshal(spec_of(name).objects)
    return native.SceneHandle(hs, ts, 0, keepalive=keep)


@functools.lru_cache(maxsize=None)
def multi(name, devs):
    hs, ts, keep = marshal(spec_of(name).objects)
    with shared(devs):
        return native.MultiHandle(hs, ts, list(devs), keepalive=keep)


def camera(name, spp=None):
    spec = spec_of(name)
    cam = native.camera_make_basic(spp or spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    cam.bounce_depth = spec.bounce_depth
    return cam


def extents(name):
    spec = spec_of(name)
    return spec.max_width_coord, spec.max_height_coord


def fields(s, names=None):
    return {n: getattr(s, n) for n in (names or [f for f, _ in s._fields_])}


def open_pair(name, world, spp=None, seed=7, adaptive=True, flags=0):
    """(frame of one device, frame over the world's devices) of the same camera, seed and flags."""
    cam, (mw, mh) = camera(name, spp), extents(name)
    a = single(name).open_frame(cam, mw, mh, seed=seed, adaptive=adaptive, flags=flags)
    b = multi(name, devices(world)).open_frame(cam, mw, mh, seed=seed, adaptive=adaptive, flags=flags)
    return a, b


def assert_same(a, b, tol=1.0):
    """Frame b (over several devices) is frame a (one device) in every output."""
    assert fields(a.progress, PROGRESS) == fields(b.progress, PROGRESS)
    ra, sa = a.read(want_sums=True)
    rb, sb = b.read(want_sums=True)
    assert np.array_equal(sa, sb), f"sums differ at {a.progress.samples_done} samples"
    assert np.array_equal(ra, rb)
    assert np.array_equal(a.read(gamma=True)[0], b.read(gamma=True)[0])
    try:
        na, ea, qa = a.noise(tol, want_sq=True)
    except native.RtError:
        with pytest.raises(native.RtError):
            b.noise(tol)
        return
    nb, eb, qb = b.noise(tol, want_sq=True)
    assert fields(na) == fields(nb)
    assert np.array_equal(qa, qb) and np.array_equal(ea, eb)
    assert [fields(x) for x in a.view_noise(tol)] == [fields(x) for x in b.view_noise(tol)]
    try:
        ca = a.convergence()
    except native.RtError:
        return
    assert fields(ca) == fields(b.convergence())


def lockstep(a, b, calls, tol=1.0, every=True):
    """Drives both frames with the same max_samples per call (0: everything left), comparing after every pass."""
    for k in calls:
        a.advance(k)
        b.advance(k)
        if every:
            assert_same(a, b, tol)
    assert_same(a, b, tol)


@pytest.mark.parametrize("flags", [0, NOISE])
def test_world_of_one_device_after_every_pass(flags):
    a, b = open_pair("C1", 1, spp=64, flags=flags)
    with a, b:
        assert_same(a, b)
        lockstep(a, b, [7] * 8 + [0])
        assert b.progress.done


@pytest.mark.parametrize("world", [2, 3, "all"])
@pytest.mark.parametrize("name,adaptive,flags", [("C1", True, NOISE), ("C1-odd", True, NOISE), ("C1-odd", False, 0), ("C2", True, NOISE),
                                                 ("C2", False, 0), ("C4", True, NOISE), ("C5", True, NOISE), ("stage-n*+1", True, NOISE),
                                                 ("stage-n*+1", False, NOISE)])
def test_scene_families(name, adaptive, flags, world):
    a, b = open_pair(name, world, adaptive=adaptive, flags=flags)
    with a, b:
        assert_same(a, b)
        lockstep(a, b, [5, 3, 0])


@pytest.mark.parametrize("world", [1, 2, "all"])
@pytest.mark.parametrize("flag", ["no-smem", "wide-bvh", "no-lean"])
@pytest.mark.parametrize("name", ["C1", "stage-n*+1"])
def test_flags(name, flag, world):
    f = {"no-smem": abi.RT_FLAG_NO_SMEM, "wide-bvh": abi.RT_FLAG_WIDE_BVH, "no-lean": abi.RT_FLAG_NO_LEAN}[flag]
    for flags in (f, f | NOISE):
        a, b = open_pair(name, world, flags=flags)
        with a, b:
            lockstep(a, b, [4, 0])


@pytest.mark.parametrize("world", [1, 2, "all"])
@pytest.mark.parametrize("flag", [abi.RT_FLAG_FLOW, abi.RT_FLAG_COUNTERS])
def test_flow_and_counters_without_noise(flag, world):
    a, b = open_pair("C1", world, flags=flag)
    with a, b:
        lockstep(a, b, [6, 0])


def run_to_end(frame, shape):
    if shape == "paced":
        while not frame.progress.done:
            frame.advance(target_ms=0.5)
    elif shape == "unpaced":
        frame.advance()
    else:
        while not frame.progress.done:
            frame.advance(shape)
    return frame.read(want_sums=True)[1], frame.noise(1.0, want_sq=True), frame.progress


@pytest.mark.parametrize("world", [1, 2, 3, "all"])
def test_pass_shapes_end_in_the_same_frame(world):
    name, spp = "C1", 160
    cam, (mw, mh) = camera(name, spp), extents(name)
    with single(name).open_frame(cam, mw, mh, seed=3, flags=NOISE) as ref:
        sums, (noise, se, sq), progress = run_to_end(ref, "unpaced")
    for shape in (1, 7, 64, "paced", "unpaced"):
        with multi(name, devices(world)).open_frame(cam, mw, mh, seed=3, flags=NOISE) as f:
            if shape == 1:
                for _ in range(3):  # windows of one sample index: every rank but the first idles
                    f.advance(1)
            s, (n, e, q), p = run_to_end(f, shape)
            assert np.array_equal(s, sums) and np.array_equal(q, sq) and np.array_equal(e, se), shape
            assert fields(n) == fields(noise) and fields(p, PROGRESS) == fields(progress, PROGRESS), shape


@pytest.mark.parametrize("world", [1, 2, "all"])
def test_paced_windows_are_multiples_of_the_device_count(world):
    devs = devices(world)
    name = "C2"
    cam, (mw, mh) = camera(name, 400), extents(name)
    with multi(name, devs).open_frame(cam, mw, mh, seed=3) as f:
        done, cut = f.progress.samples_done, 0
        for _ in range(3):
            p = f.advance(target_ms=20.0)
            k = p.samples_done - done
            done = p.samples_done
            if not p.done and k >= len(devs):
                assert k % len(devs) == 0, (k, len(devs))
                cut += 1
        assert cut > 0  # at least one paced window held a whole number of rounds


@pytest.mark.parametrize("world", [1, 2, "all"])
def test_extension_equals_a_frame_opened_at_the_target(world):
    name = "C1"
    (mw, mh), devs = extents(name), devices(world)
    with multi(name, devs).open_frame(camera(name, 256), mw, mh, seed=11, flags=NOISE) as f, \
            single(name).open_frame(camera(name, 512), mw, mh, seed=11, flags=NOISE) as ref:
        f.advance(100)
        f.extend(512)
        f.advance()
        ref.advance()
        assert_same(ref, f)


@pytest.mark.parametrize("world", [1, 2, 3, "all"])
@pytest.mark.parametrize("tau,m,k", [(0.0, 64, 64), (0.5, 64, 64), (1.0, 64, 64), (1.0, 37, 23)])
def test_convergence(tau, m, k, world):
    name, spp = "C1", 256
    cam, (mw, mh) = camera(name, spp), extents(name)
    a, b = open_pair(name, world, spp=spp, seed=5, flags=NOISE)
    with a, b:
        a.set_convergence(tau, m, k)
        b.set_convergence(tau, m, k)
        checks = 0
        while not b.progress.done:
            a.advance(40)
            b.advance(40)
            assert_same(a, b, tol=tau)
            c = b.convergence()
            if c.checks > checks and not b.progress.done:  # right after a check every pixel still sampled is above tau
                summary = b.noise(tau, want_map=False)[0]
                assert summary.pixels_above == summary.pixels == c.pixels_active
            checks = c.checks
        assert a.progress.done
        # every pixel is rt_render's pixel at its own sample count
        _, sums = b.read(want_sums=True)
        counts = sums[..., 3]
        for n in np.unique(counts):
            _, ref, _ = single(name).render(camera(name, int(n)), mw, mh, seed=5, want_sums=True)
            at = counts == n
            assert np.array_equal(sums[at], ref[at]), int(n)


@pytest.mark.parametrize("world", [1, 2, "all"])
def test_features_and_denoise(world):
    other = dict(iterations=5, feature_samples=1, sigma_colour=2.0, sigma_normal=0.3, sigma_albedo=8.0, sigma_depth=0.1, gamma=True)
    a, b = open_pair("C1", world, spp=64, seed=9, flags=NOISE)
    with a, b:
        for calls in ([], [20], [0]):
            lockstep(a, b, calls)
            for samples in (1, 4, 64):
                for x, y in zip(a.features(samples), b.features(samples)):
                    assert np.array_equal(x, y), samples
            for opts in ({}, other):
                for x, y in zip(a.denoise(want_linear=True, **opts), b.denoise(want_linear=True, **opts)):
                    assert np.array_equal(x, y), opts


@pytest.mark.parametrize("world", [1, 2, "all"])
def test_interleaving_with_render_and_other_frames(world):
    name = "C1"
    cam, (mw, mh) = camera(name, 48), extents(name)
    mh_ = multi(name, devices(world))
    a = single(name).open_frame(cam, mw, mh, seed=21, flags=NOISE)
    b = mh_.open_frame(cam, mw, mh, seed=21, flags=NOISE)
    with a, b:
        lockstep(a, b, [6])
        rgb, sums, _ = mh_.render(cam, mw, mh, seed=4, want_sums=True)
        _, ref_sums, _ = single(name).render(cam, mw, mh, seed=4, want_sums=True)
        assert np.array_equal(sums, ref_sums)
        other = mh_.open_frame(camera(name, 96), mw, mh, seed=22)
        other.advance(10)
        lockstep(a, b, [6])
        other.advance(10)
        other.close()  # destroyed mid-way
        third = mh_.open_frame(cam, mw, mh, seed=23, flags=NOISE)
        lockstep(a, b, [6])
        third.advance(3)
        lockstep(a, b, [0])
        third.close()


def test_refusals():
    name = "C1"
    cam, (mw, mh) = camera(name), extents(name)
    mh_ = multi(name, devices(1))
    lib = native.lib()
    for mode, flags, code in [(abi.RT_MODE_WAVEFRONT, 0, abi.RT_ERR_UNSUPPORTED), (abi.RT_MODE_MEGAKERNEL, NOISE | abi.RT_FLAG_FLOW, abi.RT_ERR_UNSUPPORTED),
                              (abi.RT_MODE_MEGAKERNEL, NOISE | abi.RT_FLAG_COUNTERS, abi.RT_ERR_UNSUPPORTED), (7, 0, abi.RT_ERR_INVALID_ARGUMENT)]:
        opts = abi.RtRenderOpts(1, 1, mode, 0, flags)
        out = C.c_void_p()
        assert lib.rt_multi_frame_begin(mh_.ptr, C.byref(cam), mw, mh, C.byref(opts), C.byref(out), None) == code, (mode, flags)
        assert out.value is None
    opts = abi.RtRenderOpts(1, 1, abi.RT_MODE_MEGAKERNEL, 0, 0)
    out = C.c_void_p()
    assert lib.rt_multi_frame_begin(mh_.ptr, None, mw, mh, C.byref(opts), C.byref(out), None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_multi_frame_begin(mh_.ptr, C.byref(cam), 0, mh, C.byref(opts), C.byref(out), None) == abi.RT_ERR_INVALID_ARGUMENT
    assert out.value is None
    if "RTFS_MULTI_SHARE_DEVICES" not in os.environ:  # ranks share a device only on request
        hs, ts, keep = marshal(spec_of(name).objects)
        with pytest.raises(native.RtError) as e:
            native.MultiHandle(hs, ts, [0, 0], keepalive=keep)
        assert e.value.code == abi.RT_ERR_INVALID_ARGUMENT
    with mh_.open_frame(cam, mw, mh) as f:  # no RT_FLAG_NOISE: the noise calls refuse the frame
        for call in (lambda: f.noise(1.0), lambda: f.view_noise(1.0), lambda: f.set_convergence(1.0), lambda: f.denoise()):
            with pytest.raises(native.RtError) as e:
                call()
            assert e.value.code == abi.RT_ERR_INVALID_ARGUMENT


@pytest.mark.parametrize("world", [2, "all"])
def test_scene_render_progressive(world):
    spec = spec_of("C1")
    mw, mh = extents("C1")
    cam = camera("C1", 96)
    one = Scene.make(spec.objects, device=0)
    with shared(devices(world)):
        several = Scene.make(spec.objects, devices=list(devices(world)))
    assert isinstance(several.handle, native.MultiHandle)
    for kw in (dict(), dict(noise_tolerance=2.0), dict(converge_tolerance=1.0, converge_min_samples=32, converge_interval=16)):
        ticks = {"one": 0, "several": 0}
        passes = []

        def tick(which):
            def f(_):
                ticks[which] += 1
            return f

        ref = Scene.render_progressive(tick("one"), print, mw, mh, cam, one, seed=17, target_ms=1.0, **kw)
        got = Scene.render_progressive(tick("several"), print, mw, mh, cam, several, seed=17, target_ms=1.0,
                                       on_pass=lambda p, fr: passes.append(p.samples_done), **kw)
        assert np.array_equal(got, ref), kw
        assert ticks == {"one": 2 * mh + 1, "several": 2 * mh + 1}
        assert passes
    with pytest.raises(NotImplementedError):
        Scene.render_progressive(lambda _: None, print, mw, mh, cam, several, seed=17, window=(0, 0, 4, 4))
