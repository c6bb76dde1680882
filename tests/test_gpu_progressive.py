"""Progressive frames (rt_frame_*, native.Frame, Scene.render_progressive) against rt_render, bit for bit.

A frame that has reached samples_done must hold exactly rt_render's frame at samples_per_pixel = samples_done (same
seed, extents, early-out and flags): sums keyed by (seed, pixel, sample index) and added as integers do not depend on
how the sample indices are cut into passes.  Every comparison here is np.array_equal, with no tolerance.  The frames are
the production ones (C2 is the frame bench.py times; C3, C4 and C5 at full size) so that the passes run with the
production chunking and, for C5, the global-memory kernel with its walk stacks in shared memory."""
import ctypes as C
import hashlib

import numpy as np
import pytest

from helpers import oracle_camera
from ray_tracing_fsharp_b200 import abi, native, sample_images
from ray_tracing_fsharp_b200.domain import marshal
from ray_tracing_fsharp_b200.scene import Image, Scene

pytestmark = pytest.mark.gpu

# bench.py's frame_hashes: the C2 frame at seed 424242 through rt_render (profiles/r02h_bench_n1.json, "frame_sha256")
C2_BENCH_SEED = 424242
C2_BENCH_RGB8 = "df1007c6bb1b210f65b3d16f72e9fc87ba62e85f5015b5bc35494f749e24f8e4"
C2_BENCH_SUMS = "88ff5c728e3f659a7cf1df46a2d06095e925a7b3316dbd8414d383331a8596e2"


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def scenes():
    cache = {}

    def get(name):
        if name not in cache:
            spec = sample_images.CONFIGS[name]()
            hs, ts, keep = marshal(spec.objects)
            cache[name] = (spec, native.SceneHandle(hs, ts, 0, keepalive=keep), oracle_camera(spec))
        return cache[name]

    yield get
    for _, h, _ in cache.values():
        h.close()


def with_spp(cam, spp):
    c = abi.RtCamera.from_buffer_copy(cam)
    c.samples_per_pixel = spp
    return c


def n_probe_of(spp, adaptive):
    return 2 * min(5, spp // 2) + 1 if adaptive else 0


def assert_is_render_at(h, frame, cam, mw, mh, seed, adaptive, flags, progress):
    """The frame equals rt_render at samples_done: sums, RGB8 with and without gamma, and the path count."""
    s = progress.samples_done
    ref_cam = with_spp(cam, s)
    rgb, sums, stats = h.render(ref_cam, mw, mh, seed=seed, adaptive=adaptive, flags=flags, want_sums=True)
    got_rgb, got_sums = frame.read(want_sums=True)
    assert np.array_equal(got_sums, sums), f"sums differ from rt_render at {s} spp"
    assert np.array_equal(got_rgb, rgb), f"RGB8 differs from rt_render at {s} spp"
    rgb_g, _, _ = h.render(ref_cam, mw, mh, seed=seed, adaptive=adaptive, flags=flags, gamma=True)
    got_g, _ = frame.read(gamma=True)
    assert np.array_equal(got_g, rgb_g), f"gamma-corrected RGB8 differs from rt_render at {s} spp"
    n_pixels = (2 * mw + 1) * (2 * mh + 1)
    n_probe = n_probe_of(cam.samples_per_pixel, adaptive)
    assert progress.paths_done == n_pixels * n_probe + progress.pixels_flagged * (s - n_probe)
    assert progress.paths_done == stats.paths
    return stats


def run_windows(h, cam, mw, mh, seed, adaptive, windows, flags=0):
    """Opens a frame, checks it after the probe and after every forced window; returns the last progress."""
    spp = cam.samples_per_pixel
    n_pixels = (2 * mw + 1) * (2 * mh + 1)
    with h.open_frame(cam, mw, mh, seed=seed, adaptive=adaptive, flags=flags) as frame:
        p = frame.progress
        n_probe = n_probe_of(spp, adaptive)
        assert p.samples_done == n_probe and p.passes == 0
        assert p.samples_target == max(n_probe, spp)
        target_paths = p.paths_target
        assert target_paths == n_pixels * n_probe + p.pixels_flagged * (p.samples_target - n_probe)
        if adaptive:
            assert_is_render_at(h, frame, cam, mw, mh, seed, adaptive, flags, p)
        else:
            assert p.pixels_flagged == n_pixels and p.paths_done == 0
        for w in windows:
            before = p.samples_done
            p = frame.advance(max_samples=w)
            assert p.samples_done == (min(p.samples_target, before + w) if w else p.samples_target)
            assert p.paths_target == target_paths
            stats = assert_is_render_at(h, frame, cam, mw, mh, seed, adaptive, flags, p)
        assert p.done == 1 and p.samples_done == spp
        assert p.paths_done == target_paths  # exact from rt_frame_begin on
        if adaptive and spp > n_probe:
            assert p.pixels_flagged == n_pixels - stats.pixels_early_out
        # advance after done: nothing traced, done reported
        q = frame.advance()
        assert q.done == 1 and q.passes == p.passes and q.samples_done == p.samples_done and q.paths_done == p.paths_done
        return p


@pytest.mark.parametrize("config,spp,adaptive,windows", [
    ("C2", 500, True, (1, 7, 32, 100, 0)),
    ("C2", 500, False, (1, 7, 32, 100, 0)),
    ("C3", 256, True, (1, 7, 32, 100, 0)),
    ("C4", 1024, True, (1, 7, 32, 100, 0)),
    ("C5", 64, True, (1, 7, 32, 0)),
])
def test_every_pass_is_a_lower_spp_frame(scenes, config, spp, adaptive, windows):
    spec, h, cam = scenes(config)
    p = run_windows(h, with_spp(cam, spp), spec.max_width_coord, spec.max_height_coord, 77, adaptive, windows)
    assert p.passes == len(windows)


@pytest.mark.parametrize("flags", [abi.RT_FLAG_NO_SMEM, abi.RT_FLAG_NO_LEAN, abi.RT_FLAG_WIDE_BVH, abi.RT_FLAG_FLOW, abi.RT_FLAG_COUNTERS])
def test_render_flags_act_as_in_rt_render(scenes, flags):
    spec, h, cam = scenes("C2")
    run_windows(h, with_spp(cam, 64), spec.max_width_coord, spec.max_height_coord, 78, True, (7, 0), flags=flags)


def test_final_frame_is_the_bench_frame(scenes):
    spec, h, cam = scenes("C2")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    with h.open_frame(cam, mw, mh, seed=C2_BENCH_SEED) as frame:
        p = frame.progress
        while not p.done:
            p = frame.advance(target_ms=250.0)
        rgb, sums = frame.read(want_sums=True)
    ref_rgb, ref_sums, stats = h.render(cam, mw, mh, seed=C2_BENCH_SEED, want_sums=True)
    assert np.array_equal(rgb, ref_rgb) and np.array_equal(sums, ref_sums)
    assert p.paths_done == stats.paths
    assert sha(rgb) == C2_BENCH_RGB8
    assert sha(sums) == C2_BENCH_SUMS


def test_extension(scenes):
    spec, h, cam = scenes("C2")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    seed = 91
    # rendered to 100 spp, then continued to 500
    with h.open_frame(with_spp(cam, 100), mw, mh, seed=seed) as frame:
        p = frame.advance()
        assert p.done and p.samples_done == 100
        assert_is_render_at(h, frame, with_spp(cam, 100), mw, mh, seed, True, 0, p)
        frame.extend(500)
        p = frame.advance(0, 0.0)
        assert p.done and p.samples_done == 500 and p.samples_target == 500
        assert_is_render_at(h, frame, with_spp(cam, 500), mw, mh, seed, True, 0, p)
        with pytest.raises(native.RtError) as e:  # below what the frame holds
            frame.extend(499)
        assert e.value.code == abi.RT_ERR_INVALID_ARGUMENT
        with pytest.raises(native.RtError) as e:  # above 2^22
            frame.extend((1 << 22) + 1)
        assert e.value.code == abi.RT_ERR_INVALID_ARGUMENT
    # opened at 11 spp: the probe is the whole frame, yet it continues to 64
    with h.open_frame(with_spp(cam, 11), mw, mh, seed=seed) as frame:
        p = frame.progress
        assert p.done and p.samples_done == 11
        assert_is_render_at(h, frame, with_spp(cam, 11), mw, mh, seed, True, 0, p)
        frame.extend(64)
        assert not frame.advance(max_samples=20).done
        p = frame.advance()
        assert p.done and p.samples_done == 64
        assert_is_render_at(h, frame, with_spp(cam, 64), mw, mh, seed, True, 0, p)
    # the target may also come down, to no less than what is done
    with h.open_frame(cam, mw, mh, seed=seed) as frame:
        frame.advance(max_samples=100)
        frame.extend(150)
        p = frame.advance()
        assert p.done and p.samples_done == 150
        assert_is_render_at(h, frame, with_spp(cam, 150), mw, mh, seed, True, 0, p)
    # 6 -> 64 changes firstTrial (3 -> 5), i.e. the probe already run
    with h.open_frame(with_spp(cam, 6), mw, mh, seed=seed) as frame:
        with pytest.raises(native.RtError) as e:
            frame.extend(64)
        assert e.value.code == abi.RT_ERR_INVALID_ARGUMENT
        frame.extend(7)  # firstTrial 3 as well: accepted


def test_isolation_between_passes(scenes):
    spec, h, cam = scenes("C2")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cam_a = with_spp(cam, 200)
    c1 = sample_images.CONFIGS["C1"]()
    cam_b = oracle_camera(c1)
    cam_b.samples_per_pixel = 64
    with h.open_frame(cam_a, mw, mh, seed=5) as a:
        a.advance(max_samples=20)
        other, _, _ = h.render(with_spp(cam_b, 33), 300, 170, seed=6)  # another camera and size on the same scene
        with h.open_frame(cam_b, c1.max_width_coord, c1.max_height_coord, seed=7) as b:
            b.advance(max_samples=10)
            pa = a.advance()
            assert pa.done
            assert_is_render_at(h, a, cam_a, mw, mh, 5, True, 0, pa)
            pb = b.advance()
            assert pb.done
            assert_is_render_at(h, b, cam_b, c1.max_width_coord, c1.max_height_coord, 7, True, 0, pb)
    again, _, _ = h.render(with_spp(cam_b, 33), 300, 170, seed=6)
    assert np.array_equal(other, again)


def test_pacing_does_not_change_results(scenes):
    spec, h, cam = scenes("C2")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    with h.open_frame(cam, mw, mh, seed=3) as frame:
        one = frame.advance()
        assert one.passes == 1
        ref_rgb, ref_sums = frame.read(want_sums=True)
    with h.open_frame(cam, mw, mh, seed=3) as frame:
        p = frame.progress
        sizes = []
        while not p.done:
            before = p.samples_done
            p = frame.advance(target_ms=5.0)
            sizes.append(p.samples_done - before)
            assert p.last_pass_ms > 0
        rgb, sums = frame.read(want_sums=True)
    assert p.passes == len(sizes) > 1 and min(sizes) >= 1
    assert np.array_equal(sums, ref_sums) and np.array_equal(rgb, ref_rgb)
    assert p.paths_done == one.paths_done


def test_render_progressive_python_mirror(scenes):
    spec = sample_images.CONFIGS["C2"]()
    cam = oracle_camera(spec)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    rows = 2 * mh + 1
    s = Scene.make(spec.objects, device=0)
    ticks, seen = [], []

    def on_pass(progress, frame):
        seen.append((progress.samples_done, progress.done, len(ticks)))

    img = Scene.render_progressive(lambda x: ticks.append(x), lambda _: None, mw, mh, cam, s, seed=11, target_ms=10.0, on_pass=on_pass)
    assert len(ticks) == rows and all(t == 1.0 for t in ticks)
    assert len(seen) > 1 and seen[-1][1] == 1 and seen[-1][0] == spec.spp
    assert 0 < seen[-1][2] < rows  # ticks came in before the last pass completed
    assert [n for _, _, n in seen] == sorted(n for _, _, n in seen)
    _, image = Scene.render(lambda _: None, lambda _: None, mw, mh, cam, s, seed=11)
    assert np.array_equal(img, Image.render(image))

    # stopped after the first pass: the image is rt_render's at that pass's samples_done
    ticks.clear()
    stopped = {}

    def stop(progress, frame):
        stopped["spp"] = progress.samples_done
        stopped["rgb"], stopped["sums"] = frame.read(want_sums=True)
        return True

    img = Scene.render_progressive(lambda x: ticks.append(x), lambda _: None, mw, mh, cam, s, seed=12, target_ms=10.0, on_pass=stop)
    assert len(ticks) == rows
    assert 11 < stopped["spp"] < spec.spp
    ref_rgb, ref_sums, _ = s.handle.render(with_spp(cam, stopped["spp"]), mw, mh, seed=12, want_sums=True)
    assert np.array_equal(stopped["sums"], ref_sums) and np.array_equal(stopped["rgb"], ref_rgb)
    assert np.array_equal(img, ref_rgb)


def test_errors(scenes):
    spec, h, cam = scenes("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    with pytest.raises(native.RtError) as e:
        h.open_frame(cam, mw, mh, mode=abi.RT_MODE_WAVEFRONT)
    assert e.value.code == abi.RT_ERR_UNSUPPORTED
    lib = native.lib()
    opts = abi.RtRenderOpts(1, 1, abi.RT_MODE_MEGAKERNEL, 0, 0)
    out = C.c_void_p()
    progress = abi.RtFrameProgress()
    buf = np.empty(16, np.int32)
    bad = abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_frame_begin(None, C.byref(cam), mw, mh, C.byref(opts), C.byref(out), None) == bad
    assert lib.rt_frame_begin(h.ptr, None, mw, mh, C.byref(opts), C.byref(out), None) == bad
    assert lib.rt_frame_begin(h.ptr, C.byref(cam), mw, mh, None, C.byref(out), None) == bad
    assert lib.rt_frame_begin(h.ptr, C.byref(cam), mw, mh, C.byref(opts), None, None) == bad
    assert lib.rt_frame_advance(None, 0, 0.0, C.byref(progress)) == bad
    assert lib.rt_frame_read(None, 0, native.ptr(buf), None) == bad
    assert lib.rt_frame_extend(None, 10) == bad
    lib.rt_frame_destroy(None)
    with h.open_frame(cam, mw, mh) as frame:
        assert lib.rt_frame_advance(frame.ptr, -1, 0.0, None) == bad
        assert lib.rt_frame_advance(frame.ptr, 0, -1.0, None) == bad
        assert lib.rt_frame_advance(frame.ptr, 0, float("nan"), None) == bad
        assert lib.rt_frame_extend(frame.ptr, 0) == bad
        assert frame.advance().done  # still usable
