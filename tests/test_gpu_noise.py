"""The noise estimate of progressive frames (RT_FLAG_NOISE, rt_frame_noise, Frame.noise, render_progressive's stop rule).

Every sample is a pure function of (seed, pixel, sample index) and rt_test_trace_samples reproduces it, so the per-pixel sum
of squares Q a frame keeps is checked EXACTLY against the sum of r^2 + g^2 + b^2 over the pixel's sample indices, with
renderPixel's early-out rule applied to the same colours (helpers.expected_moments).  A frame
opened with the flag must still be rt_render's frame at samples_done, bit for bit; the estimate derived from Q must equal a
numpy restatement; and render_progressive must stop at the first check that meets its rule."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

if __name__ == "__main__":  # the child process of test_noise_kernels_with_local_walk_stacks
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from helpers import expected_moments, oracle_camera  # noqa: E402
from ray_tracing_fsharp_b200 import abi, native, sample_images  # noqa: E402
from ray_tracing_fsharp_b200.domain import marshal  # noqa: E402
from ray_tracing_fsharp_b200.scene import Image, Scene  # noqa: E402

pytestmark = pytest.mark.gpu

NOISE = abi.RT_FLAG_NOISE


@pytest.fixture(scope="module")
def scenes():
    cache = {}

    def get(name):
        if name not in cache:
            spec = sample_images.CONFIGS[name]() if name != "small" else sample_images.few_spheres(max_w=40, max_h=22, spp=40)
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


def numpy_se(sums, sq):
    """D = n Q - sum_c T_c^2 in int64, E = sqrt(D / (3 n^2 (n - 1))) in float64, +inf where n < 2."""
    sums = np.asarray(sums).astype(np.int64)
    n = sums[..., 3]
    t = sums[..., :3]
    d = n * np.asarray(sq).astype(np.int64) - (t[..., 0] * t[..., 0] + t[..., 1] * t[..., 1] + t[..., 2] * t[..., 2])
    nd = n.astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        e = np.sqrt(d.astype(np.float64) / (3.0 * nd * nd * (n - 1).astype(np.float64)))
    return np.where(n < 2, np.inf, e)


# ---- reconstruction from single samples (helpers.expected_moments) ----------------------------------------------------
def row_subset(rows, cols, stride, n_random, seed):
    """Rows 0-3, the last four rows, every `stride`-th row between them, and `n_random` pixels anywhere (flat ids)."""
    picked = np.unique(np.concatenate([np.arange(4), np.arange(4, rows - 4, stride), np.arange(rows - 4, rows)]))
    pixels = (picked[:, None] * cols + np.arange(cols)[None, :]).ravel()
    extra = np.random.default_rng(seed).integers(0, rows * cols, n_random)
    return np.unique(np.concatenate([pixels, extra]))


def assert_moments_exact(h, frame, cam, mw, mh, seed, adaptive, pixels, what):
    """Sums and Q of the frame at `pixels` equal the reconstruction at the frame's samples_done."""
    _, sums = frame.read(want_sums=True)
    _, _, sq = frame.noise(0.0, want_map=False, want_sq=True)
    want_sums, want_q = expected_moments(h, cam, mw, mh, seed, adaptive, pixels, frame.progress.samples_done)
    got_sums = sums.reshape(-1, 4)[pixels].astype(np.int64)
    got_q = sq.reshape(-1)[pixels].astype(np.int64)
    bad = np.flatnonzero((got_sums != want_sums).any(1) | (got_q != want_q))
    cols = 2 * mw + 1
    detail = "; ".join(f"(row {pixels[i] // cols}, col {pixels[i] % cols}) frame {got_sums[i].tolist()} Q {got_q[i]}, samples "
                       f"{want_sums[i].tolist()} Q {want_q[i]}" for i in bad[:6])
    assert bad.size == 0, f"{what} at {frame.progress.samples_done} spp: {bad.size} of {len(pixels)} pixels differ: {detail}"
    assert (got_q > 0).any()


def test_q_of_the_bench_frame_after_the_probe_and_a_pass(scenes):
    """The C2 frame bench.py times (seed 424242), rows 0-3, every 9th row, the last four and 300 random pixels."""
    spec, h, cam = scenes("C2")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    pixels = row_subset(spec.rows, spec.cols, 9, 300, 1)
    with h.open_frame(cam, mw, mh, seed=424242, flags=NOISE) as frame:
        assert_moments_exact(h, frame, cam, mw, mh, 424242, True, pixels, "C2 after the probe")
        frame.advance(max_samples=89)
        assert frame.progress.samples_done == 100
        assert_moments_exact(h, frame, cam, mw, mh, 424242, True, pixels, "C2 mid-frame")


@pytest.mark.parametrize("config,stride", [("C3", 15), ("C4", 27), ("C5", 15)])
def test_q_of_full_size_frames_at_64_spp(scenes, config, stride):
    """C3 (texture lookups), C4 (planes, FP64 objects, depth 100), C5 (the scene read from global memory) at 64 spp."""
    spec, h, cam = scenes(config)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cam64 = with_spp(cam, 64)
    pixels = row_subset(spec.rows, spec.cols, stride, 300, 2)
    with h.open_frame(cam64, mw, mh, seed=21, flags=NOISE) as frame:
        frame.advance(max_samples=20)
        frame.advance()
        assert frame.progress.done
        assert_moments_exact(h, frame, cam64, mw, mh, 21, True, pixels, config)


@pytest.mark.parametrize("adaptive", [True, False])
def test_q_of_a_small_frame_every_pixel(scenes, adaptive):
    spec, h, cam = scenes("small")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    pixels = np.arange(spec.rows * spec.cols)
    with h.open_frame(cam, mw, mh, seed=5, adaptive=adaptive, flags=NOISE) as frame:
        if adaptive:
            assert_moments_exact(h, frame, cam, mw, mh, 5, adaptive, pixels, "small frame")
        for w in (1, 7, 0):
            frame.advance(max_samples=w)
            assert_moments_exact(h, frame, cam, mw, mh, 5, adaptive, pixels, "small frame")


# ---- the frame itself is unchanged -----------------------------------------------------------------------------------------
def assert_is_render_at(h, frame, cam, mw, mh, seed, adaptive, flags, progress):
    s = progress.samples_done
    rgb, sums, stats = h.render(with_spp(cam, s), mw, mh, seed=seed, adaptive=adaptive, flags=flags, want_sums=True)
    got_rgb, got_sums = frame.read(want_sums=True)
    assert np.array_equal(got_sums, sums), f"sums differ from rt_render at {s} spp"
    assert np.array_equal(got_rgb, rgb), f"RGB8 differs from rt_render at {s} spp"
    assert progress.paths_done == stats.paths


def run_windows(h, cam, mw, mh, seed, windows, flags):
    """A NOISE frame checked against rt_render after the probe and after every window; returns its final Q."""
    with h.open_frame(cam, mw, mh, seed=seed, flags=flags | NOISE) as frame:
        assert_is_render_at(h, frame, cam, mw, mh, seed, True, flags, frame.progress)
        for w in windows:
            p = frame.advance(max_samples=w)
            assert_is_render_at(h, frame, cam, mw, mh, seed, True, flags, p)
        assert p.done
        return frame.noise(0.0, want_map=False, want_sq=True)[2]


@pytest.mark.parametrize("config,spp,windows", [("C2", 500, (1, 7, 32, 100, 0)), ("C5", 64, (1, 7, 32, 0))])
def test_noise_frames_are_rt_render_frames(scenes, config, spp, windows):
    spec, h, cam = scenes(config)
    run_windows(h, with_spp(cam, spp), spec.max_width_coord, spec.max_height_coord, 31, windows, 0)


def test_noise_frames_with_each_render_flag(scenes):
    """Every flag that works with RT_FLAG_NOISE: the same frame, and the same Q, as the default kernels give."""
    spec, h, cam = scenes("C2")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cam64 = with_spp(cam, 64)
    q0 = run_windows(h, cam64, mw, mh, 32, (7, 0), 0)
    for flags in (abi.RT_FLAG_NO_SMEM, abi.RT_FLAG_NO_LEAN, abi.RT_FLAG_WIDE_BVH, abi.RT_FLAG_BVH2, abi.RT_FLAG_LOCKSTEP,
                  abi.RT_FLAG_NO_SMEM | abi.RT_FLAG_WIDE_BVH):
        q = run_windows(h, cam64, mw, mh, 32, (7, 0), flags)
        assert np.array_equal(q, q0), f"flags {flags}: Q differs from the default kernels'"


# ---- the global kernels with their walk stacks in local memory -------------------------------------------------------------
# On the scenes above, a scene read from global memory always has room for its walk stacks in shared memory, so the four
# NOISE kernels that keep them in local memory (probe and main phase, binary and 8-wide tree) never run there.  A child
# process with RTFS_LOCAL_STACK set (read once, by the first launch plan) runs them on a reduced C2 frame read from global
# memory, and reports its launch plans (RTFS_DEBUG_PLAN) on stderr.
def local_stack_child():
    spec = sample_images.CONFIGS["C2"]()
    spec.max_width_coord, spec.max_height_coord, spec.spp = 100, 60, 40
    hs, ts, keep = marshal(spec.objects)
    h = native.SceneHandle(hs, ts, 0, keepalive=keep)
    cam = oracle_camera(spec)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    pixels = np.arange(spec.rows * spec.cols)
    for flags in (abi.RT_FLAG_NO_SMEM, abi.RT_FLAG_NO_SMEM | abi.RT_FLAG_WIDE_BVH):
        with h.open_frame(cam, mw, mh, seed=51, flags=flags | NOISE) as frame:
            assert_is_render_at(h, frame, cam, mw, mh, 51, True, flags, frame.progress)
            assert_moments_exact(h, frame, cam, mw, mh, 51, True, pixels, f"flags {flags}, local stacks")
            for w in (7, 0):
                p = frame.advance(max_samples=w)
                assert_is_render_at(h, frame, cam, mw, mh, 51, True, flags, p)
                assert_moments_exact(h, frame, cam, mw, mh, 51, True, pixels, f"flags {flags}, local stacks")
            assert p.done
    h.close()
    print("local-stack child: ok")


def test_noise_kernels_with_local_walk_stacks():
    env = dict(os.environ, RTFS_LOCAL_STACK="1", RTFS_DEBUG_PLAN="1")
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "local-stack"], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "local-stack child: ok" in r.stdout, r.stdout[-4000:] + r.stderr[-4000:]
    ran = set()
    for line in r.stderr.splitlines():
        if line.startswith("rtfs: plan "):
            kv = dict(x.split("=") for x in line[len("rtfs: plan "):].split())
            if kv["noise"] == "1":
                assert (kv["staged"], kv["sstack"]) == ("0", "0"), line
                ran.add((kv["probe"], kv["wide"]))
    assert ran == {("1", "0"), ("0", "0"), ("1", "1"), ("0", "1")}, ran


# ---- pacing --------------------------------------------------------------------------------------------------------------
def test_q_does_not_depend_on_pacing(scenes):
    spec, h, cam = scenes("C2")
    mw, mh = spec.max_width_coord, spec.max_height_coord

    def q_of(frame):
        return frame.noise(0.0, want_map=False, want_sq=True)[2]

    with h.open_frame(cam, mw, mh, seed=3, flags=NOISE) as a, h.open_frame(cam, mw, mh, seed=3, flags=NOISE) as b:
        for w in (1, 7, 32):
            a.advance(max_samples=w)
        b.advance(max_samples=40)
        assert a.progress.samples_done == b.progress.samples_done == 51
        assert np.array_equal(q_of(a), q_of(b))
        while not a.progress.done:
            a.advance(target_ms=5.0)
        b.advance()
        assert a.progress.passes > 3 and b.progress.passes == 2
        assert np.array_equal(q_of(a), q_of(b))
        q500 = q_of(a)
    # extended: 100 -> 500, and 11 (the probe only) -> 64, against frames opened at the higher target
    with h.open_frame(with_spp(cam, 100), mw, mh, seed=3, flags=NOISE) as f:
        f.advance()
        f.extend(500)
        f.advance()
        assert f.progress.samples_done == 500
        assert np.array_equal(q_of(f), q500)
    with h.open_frame(with_spp(cam, 11), mw, mh, seed=3, flags=NOISE) as f, \
            h.open_frame(with_spp(cam, 64), mw, mh, seed=3, flags=NOISE) as g:
        f.extend(64)
        f.advance()
        g.advance()
        assert np.array_equal(q_of(f), q_of(g))


# ---- the estimate ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("adaptive", [True, False])
def test_estimate_matches_numpy(scenes, adaptive):
    spec, h, cam = scenes("C2")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    with h.open_frame(cam, mw, mh, seed=41, adaptive=adaptive, flags=NOISE) as frame:
        frame.advance(max_samples=50)
        s = frame.progress.samples_done
        _, sums = frame.read(want_sums=True)
        e = numpy_se(sums, frame.noise(0.0, want_map=False, want_sq=True)[2])
        flagged = sums[..., 3] == s  # past the probe, exactly the pixels that go on hold samples_done samples
        assert int(flagged.sum()) == frame.progress.pixels_flagged
        ef = e[flagged]
        assert np.isfinite(ef).all()
        for tol in (0.0, float(np.median(ef)), float(np.quantile(ef, 0.99)), float(ef.max()), float("inf")):
            summary, se, sq = frame.noise(tol, want_sq=True)
            assert np.array_equal(numpy_se(sums, sq), e)
            assert se.dtype == np.float32 and np.array_equal(se, e.astype(np.float32))
            assert summary.pixels == int(flagged.sum())
            assert summary.pixels_above == int((ef > tol).sum())
            assert summary.max_se == ef.max()
            assert summary.mean_se == pytest.approx(ef.mean(), rel=1e-12)
            assert summary.tolerance == tol
            again, _, _ = frame.noise(tol, want_map=False)
            assert bytes(again) == bytes(summary)  # bit-identical from call to call
        # the host helper gives the same map from the saved moments
        assert np.array_equal(native.pixel_noise(sums, sq), se)


def test_estimate_after_the_probe(scenes):
    """After the probe every pixel holds n_probe samples; the summary covers the pixels flagged to go on."""
    spec, h, cam = scenes("C2")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    with h.open_frame(cam, mw, mh, seed=42, flags=NOISE) as frame:
        summary, se, sq = frame.noise(4.0, want_sq=True)
        _, sums = frame.read(want_sums=True)
        assert (sums[..., 3] == 11).all()
        assert summary.pixels == frame.progress.pixels_flagged > 0
        assert np.array_equal(se, numpy_se(sums, sq).astype(np.float32))
        assert summary.max_se <= float(se.max())


# ---- render_progressive's stop rule ------------------------------------------------------------------------------------------
def test_render_progressive_stops_on_the_noise_rule(scenes):
    spec = sample_images.CONFIGS["C2"]()
    cam = oracle_camera(spec)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    rows = 2 * mh + 1
    s = Scene.make(spec.objects, device=0)
    fraction = 0.01
    # the tolerance: the 99th percentile of E over the flagged pixels at 200 spp, so that the rule is met near there
    with s.handle.open_frame(cam, mw, mh, seed=13, flags=NOISE) as frame:
        frame.advance(max_samples=200 - 11)
        summary, se, _ = frame.noise(0.0)
        _, sums = frame.read(want_sums=True)
        tol = float(np.quantile(se[sums[..., 3] == 200], 1.0 - fraction))
    ticks, seen = [], []

    def on_pass(progress, frame):
        summary, _, _ = frame.noise(tol, want_map=False)
        seen.append((progress.samples_done, progress.done, summary.pixels_above, summary.pixels))

    img = Scene.render_progressive(lambda x: ticks.append(x), lambda _: None, mw, mh, cam, s, seed=13, target_ms=10.0, on_pass=on_pass,
                                   noise_tolerance=tol, noise_fraction=fraction)
    assert len(ticks) == rows and all(t == 1.0 for t in ticks)
    meets = [above <= fraction * pixels for _, _, above, pixels in seen]
    assert len(seen) > 2 and meets[-1] and not any(meets[:-1]), seen  # stopped at the first check that met the rule
    done = seen[-1][0]
    assert 11 < done < spec.spp and not seen[-1][1]
    ref_rgb, _, _ = s.handle.render(with_spp(cam, done), mw, mh, seed=13)
    assert np.array_equal(img, ref_rgb)
    # without a tolerance the same call renders the whole frame
    ticks.clear()
    img = Scene.render_progressive(lambda x: ticks.append(x), lambda _: None, mw, mh, cam, s, seed=13, target_ms=50.0)
    _, image = Scene.render(lambda _: None, lambda _: None, mw, mh, cam, s, seed=13)
    assert np.array_equal(img, Image.render(image)) and len(ticks) == rows


def test_render_progressive_stops_after_the_probe(scenes):
    """A tolerance every flagged pixel meets after the probe: no pass runs, the image is the probe's frame."""
    spec = sample_images.CONFIGS["C2"]()
    cam = oracle_camera(spec)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    s = Scene.make(spec.objects, device=0)
    ticks, seen = [], []
    img = Scene.render_progressive(lambda x: ticks.append(x), lambda _: None, mw, mh, cam, s, seed=14,
                                   on_pass=lambda p, f: seen.append(p.samples_done), noise_tolerance=float("inf"))
    assert seen == [] and len(ticks) == 2 * mh + 1
    ref_rgb, _, _ = s.handle.render(with_spp(cam, 11), mw, mh, seed=14)
    assert np.array_equal(img, ref_rgb)


# ---- errors ---------------------------------------------------------------------------------------------------------------
def test_errors(scenes):
    spec, h, cam = scenes("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    for other in (abi.RT_FLAG_FLOW, abi.RT_FLAG_COUNTERS):
        with pytest.raises(native.RtError) as e:
            h.open_frame(cam, mw, mh, flags=NOISE | other)
        assert e.value.code == abi.RT_ERR_UNSUPPORTED
    with h.open_frame(cam, mw, mh) as frame:
        with pytest.raises(native.RtError) as e:
            frame.noise(1.0)
        assert e.value.code == abi.RT_ERR_INVALID_ARGUMENT
    with h.open_frame(cam, mw, mh, flags=NOISE) as frame:
        lib = native.lib()
        summary = abi.RtFrameNoise()
        assert lib.rt_frame_noise(frame.ptr, -1.0, None, None, C.byref(summary)) == abi.RT_ERR_INVALID_ARGUMENT
        assert lib.rt_frame_noise(frame.ptr, float("nan"), None, None, C.byref(summary)) == abi.RT_ERR_INVALID_ARGUMENT
        assert lib.rt_frame_noise(frame.ptr, 1.0, None, None, None) == abi.RT_OK  # every output optional
        assert frame.advance().done  # still usable
    # rt_render ignores the bit: the same frame as without it
    a, sa, _ = h.render(cam, mw, mh, seed=4, flags=NOISE, want_sums=True)
    b, sb, _ = h.render(cam, mw, mh, seed=4, want_sums=True)
    assert np.array_equal(a, b) and np.array_equal(sa, sb)


if __name__ == "__main__" and sys.argv[1:] == ["local-stack"]:
    local_stack_child()
