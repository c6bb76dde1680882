"""The convergence rule of progressive frames (rt_frame_set_convergence, Frame.set_convergence, render_progressive's
converge_tolerance).

Under the rule every pixel p holds the sums and Q of sample indices [0, n_p), n_p being the probe's count, the first
checkpoint at which its standard error was within the tolerance, or samples_done.  Every sample is a pure function of
(seed, pixel, sample index), so the frame is checked EXACTLY: against the rule restated in numpy (convergence_rule.py) over
colours from rt_test_trace_samples, and at production size against a plain RT_FLAG_NOISE frame snapshotted at every
checkpoint."""
import ctypes as C

import numpy as np
import pytest

from convergence_rule import checkpoints, converge, numpy_se, probe
from helpers import BATCH, oracle_camera
from ray_tracing_fsharp_b200 import abi, native, sample_images
from ray_tracing_fsharp_b200.domain import marshal
from ray_tracing_fsharp_b200.scene import Scene

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


def state(frame, pixels=None):
    """(int64 sums [n, 4], int64 Q [n]) of the frame, at `pixels` (flat ids) or everywhere."""
    _, sums = frame.read(want_sums=True)
    _, _, sq = frame.noise(0.0, want_map=False, want_sq=True)
    sums, sq = sums.reshape(-1, 4).astype(np.int64), sq.reshape(-1).astype(np.int64)
    return (sums, sq) if pixels is None else (sums[pixels], sq[pixels])


class Samples:
    """The colours of samples [0, spp) of the flat pixel ids `pixels`, traced one by one (rt_test_trace_samples); moments()
    is the source of samples convergence_rule reads."""

    def __init__(self, h, cam, mw, mh, seed, pixels, spp):
        cols = 2 * mw + 1
        self.colours = np.empty((len(pixels), spp, 3), np.uint8)
        per_call = max(1, BATCH // spp)
        smp = np.arange(spp, dtype=np.int32)
        for lo in range(0, len(pixels), per_call):
            pix = pixels[lo:lo + per_call]
            colour, _ = h.trace_samples(cam, mw, mh, seed, np.repeat(pix // cols, spp), np.repeat(pix % cols, spp), np.tile(smp, len(pix)))
            self.colours[lo:lo + len(pix)] = colour.reshape(len(pix), spp, 3)

    def moments(self, idx, s0, s1):
        c = self.colours[idx, s0:s1].astype(np.int64)
        return c.sum(1), (c * c).sum((1, 2))


def median_e_at(samples, start, m, k):
    """A tolerance that about half the pixels still sampled at the first checkpoint meet there."""
    s0, q0, _, flagged = start
    sums, q, _, _ = converge(samples.moments, s0, q0, flagged, m, -1.0, m, k)
    return float(np.median(numpy_se(sums, q)[flagged]))


def assert_rule_holds(frame, samples, pixels, start, tol, m, k, what):
    """The frame at `pixels` equals the numpy rule at its samples_done; returns the rule's (active mask, checks)."""
    s0, q0, _, flagged = start
    done = frame.progress.samples_done
    want_sums, want_q, active, checks = converge(samples.moments, s0, q0, flagged, done, tol, m, k)
    got_sums, got_q = state(frame, pixels)
    bad = np.flatnonzero((got_sums != want_sums).any(1) | (got_q != want_q))
    assert bad.size == 0, (f"{what} at {done} spp: {bad.size} of {len(pixels)} pixels differ, e.g. frame {got_sums[bad[0]].tolist()} "
                           f"Q {got_q[bad[0]]}, rule {want_sums[bad[0]].tolist()} Q {want_q[bad[0]]}")
    return active, checks


def row_subset(rows, cols, stride, n_random, seed):
    picked = np.unique(np.concatenate([np.arange(4), np.arange(4, rows - 4, stride), np.arange(rows - 4, rows)]))
    pixels = (picked[:, None] * cols + np.arange(cols)[None, :]).ravel()
    return np.unique(np.concatenate([pixels, np.random.default_rng(seed).integers(0, rows * cols, n_random)]))


# ---- 1. exact against single samples ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("config,spp,m,k", [("small", 40, 16, 8), ("C2", 200, 64, 32)])
@pytest.mark.parametrize("adaptive", [True, False])
def test_frame_is_the_rule_on_single_samples(scenes, config, spp, m, k, adaptive):
    spec, h, cam = scenes(config)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cam = with_spp(cam, spp)
    n = spec.rows * spec.cols
    pixels = np.arange(n) if config == "small" else row_subset(spec.rows, spec.cols, 40, 300, 3)
    samples = Samples(h, cam, mw, mh, 17, pixels, spp)
    start = probe(samples.moments, len(pixels), spp, adaptive)
    tol = median_e_at(samples, start, m, k)
    with h.open_frame(cam, mw, mh, seed=17, adaptive=adaptive, flags=NOISE) as frame:
        frame.set_convergence(tol, m, k)
        assert_rule_holds(frame, samples, pixels, start, tol, m, k, f"{config} after the probe")
        seen_stopped = 0
        while not frame.progress.done:
            frame.advance(max_samples=11)
            active, checks = assert_rule_holds(frame, samples, pixels, start, tol, m, k, config)
            conv = frame.convergence()
            assert conv.checks == checks
            seen_stopped = int((start[3] & ~active).sum())
            if config == "small":  # every pixel: the frame's counts are the rule's
                assert conv.pixels_active == int(active.sum()) and conv.pixels_converged == seen_stopped
                assert frame.progress.paths_done == int(state(frame)[0][:, 3].sum())
        assert 0 < seen_stopped < int(start[3].sum())


# ---- 2. exact against the plain frame at production size ----------------------------------------------------------------
def plain_snapshots(h, cam, mw, mh, seed, m, k, quantile):
    """A plain RT_FLAG_NOISE frame advanced checkpoint by checkpoint: (tolerance, the frame the rule must give, active mask,
    checks).  The tolerance is the `quantile` of E over the pixels still sampled at the first checkpoint."""
    with h.open_frame(cam, mw, mh, seed=seed, flags=NOISE) as plain:
        target = plain.progress.samples_target
        want_sums = want_q = active = tol = None
        checks = 0
        for c in checkpoints(m, k, target):
            plain.advance(max_samples=c - plain.progress.samples_done)
            assert plain.progress.samples_done == c
            sums, q = state(plain)
            if want_sums is None:
                want_sums, want_q, active = sums, q, sums[:, 3] == c
                tol = float(np.quantile(numpy_se(sums, q)[active], quantile))
            if not active.any():
                break
            want_sums[active], want_q[active] = sums[active], q[active]
            active &= ~(numpy_se(sums, q) <= tol)
            checks += 1
        plain.advance()
        sums, q = state(plain)
        want_sums[active], want_q[active] = sums[active], q[active]
        return tol, want_sums, want_q, active, checks


@pytest.mark.parametrize("config,spp", [("C2", 500), ("C4", 1024), ("C5", 256)])
def test_frame_is_the_plain_frame_at_its_checkpoints(scenes, config, spp):
    """C2 and C4 run the staged lean and staged general kernels, C5 the one reading the scene from global memory."""
    spec, h, cam = scenes(config)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cam = with_spp(cam, spp)
    tol, want_sums, want_q, active, checks = plain_snapshots(h, cam, mw, mh, 23, 64, 64, 0.5)
    with h.open_frame(cam, mw, mh, seed=23, flags=NOISE) as frame:
        frame.set_convergence(tol, 64, 64)
        while not frame.progress.done:
            frame.advance(target_ms=100.0)
        sums, q = state(frame)
        conv = frame.convergence()
        flagged = frame.progress.pixels_flagged
    bad = np.flatnonzero((sums != want_sums).any(1) | (q != want_q))
    assert bad.size == 0, f"{config}: {bad.size} pixels differ from the plain frame's snapshots"
    assert conv.pixels_active == int(active.sum()) and conv.pixels_converged == flagged - int(active.sum())
    assert conv.checks == checks and 0 < conv.pixels_converged < flagged


# ---- 3. and 4. pacing and extension --------------------------------------------------------------------------------------
def run(h, cam, mw, mh, seed, tol, step, extend_from=None):
    """(sums, Q, RtFrameConvergence bytes) of a converging C2 frame advanced by `step()` until done."""
    c0 = with_spp(cam, extend_from) if extend_from else cam
    with h.open_frame(c0, mw, mh, seed=seed, flags=NOISE) as f:
        f.set_convergence(tol, 64, 64)
        if extend_from:
            while not f.progress.done:
                step(f)
            f.extend(cam.samples_per_pixel)
            step(f)  # progress is read back by rt_frame_advance: the extended frame's first pass
        while not f.progress.done:
            step(f)
        sums, q = state(f)
        return sums, q, bytes(f.convergence())


def c2_tolerance(h, cam, mw, mh, seed):
    with h.open_frame(cam, mw, mh, seed=seed, flags=NOISE) as f:
        f.advance(max_samples=64 - f.progress.samples_done)
        summary, se, _ = f.noise(0.0)
        _, sums = f.read(want_sums=True)
        return float(np.median(se[sums[..., 3] == 64]))


def test_pacing_does_not_change_the_frame(scenes):
    spec, h, cam = scenes("C2")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    tol = c2_tolerance(h, cam, mw, mh, 7)
    ref = run(h, cam, mw, mh, 7, tol, lambda f: f.advance())
    for step in (lambda f: f.advance(max_samples=1), lambda f: f.advance(max_samples=7), lambda f: f.advance(max_samples=64),
                 lambda f: f.advance(target_ms=2.0)):
        got = run(h, cam, mw, mh, 7, tol, step)
        assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]) and got[2] == ref[2]


def test_extended_frame_is_the_frame_opened_at_the_target(scenes):
    spec, h, cam = scenes("C2")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    tol = c2_tolerance(h, cam, mw, mh, 8)
    cam512 = with_spp(cam, 512)
    ref = run(h, cam512, mw, mh, 8, tol, lambda f: f.advance(max_samples=100))
    for start in (256, 300):
        got = run(h, cam512, mw, mh, 8, tol, lambda f: f.advance(max_samples=100), extend_from=start)
        assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]) and got[2] == ref[2]


# ---- 5. tau = 0 -------------------------------------------------------------------------------------------------------------
def test_zero_tolerance_with_the_early_out_is_the_plain_frame(scenes):
    spec, h, cam = scenes("C2")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cam = with_spp(cam, 200)
    with h.open_frame(cam, mw, mh, seed=9, flags=NOISE) as frame:
        frame.set_convergence(0.0, 16, 16)
        while not frame.progress.done:
            p = frame.advance(max_samples=40)
            rgb, sums, stats = h.render(with_spp(cam, p.samples_done), mw, mh, seed=9, want_sums=True)
            got_rgb, got_sums = frame.read(want_sums=True)
            assert np.array_equal(got_sums, sums) and np.array_equal(got_rgb, rgb), p.samples_done
            assert p.paths_done == stats.paths
        conv = frame.convergence()
        assert conv.pixels_converged == 0 and conv.checks == len(checkpoints(16, 16, 200))


def test_zero_tolerance_without_the_early_out_stops_the_constant_pixels(scenes):
    spec, h, cam = scenes("small")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    pixels = np.arange(spec.rows * spec.cols)
    samples = Samples(h, cam, mw, mh, 10, pixels, spec.spp)
    constant = (samples.colours[:, :16] == samples.colours[:, :1]).all((1, 2))
    assert 0 < constant.sum() < len(pixels)
    with h.open_frame(cam, mw, mh, seed=10, adaptive=False, flags=NOISE) as frame:
        frame.set_convergence(0.0, 16, 8)
        while not frame.progress.done:
            frame.advance()
        sums, q = state(frame)
        assert np.array_equal(sums[:, 3] == 16, constant) and (sums[~constant, 3] == spec.spp).all()
        assert frame.convergence().pixels_converged == int(constant.sum())
        e = numpy_se(sums, q)
        assert (e[constant] == 0).all() and (e[~constant] > 0).all()


# ---- 6. progress -------------------------------------------------------------------------------------------------------------
def test_progress_with_a_rule(scenes):
    spec, h, cam = scenes("C2")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    tol = c2_tolerance(h, cam, mw, mh, 11)
    with h.open_frame(cam, mw, mh, seed=11, flags=NOISE) as frame:
        frame.set_convergence(tol, 64, 64)
        targets = [frame.progress.paths_target]
        while not frame.progress.done:
            p = frame.advance(max_samples=50)
            targets.append(p.paths_target)
            sums, _ = state(frame)
            assert p.paths_done == int(sums[:, 3].sum())  # every traced path is in a pixel's count
            conv = frame.convergence()
            assert p.paths_target == p.paths_done + conv.pixels_active * (p.samples_target - p.samples_done)
            assert p.pixels_flagged == conv.pixels_active + conv.pixels_converged
            if not p.done and (p.samples_done - 64) % 64 == 0:  # right after a check
                summary, _, _ = frame.noise(tol, want_map=False)
                assert summary.pixels == conv.pixels_active and summary.pixels_above == summary.pixels
        assert all(a >= b for a, b in zip(targets, targets[1:])) and targets[-1] < targets[0]
    # a tolerance every pixel meets: everything stops at the first check, done without tracing further
    with h.open_frame(cam, mw, mh, seed=11, flags=NOISE) as frame:
        frame.set_convergence(float("inf"), 64, 64)
        p = frame.advance()
        assert p.samples_done == 64 or p.done
        p = frame.advance() if not p.done else p
        assert p.done and p.samples_done == p.samples_target and p.paths_done == p.paths_target
        assert frame.convergence().pixels_active == 0 and frame.convergence().checks == 1
        sums, _ = state(frame)
        assert set(np.unique(sums[:, 3]).tolist()) <= {11, 64}


# ---- 7. argument errors --------------------------------------------------------------------------------------------------
def test_argument_errors(scenes):
    spec, h, cam = scenes("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    lib = native.lib()
    cam64 = with_spp(cam, 64)
    with h.open_frame(cam64, mw, mh) as frame:  # no RT_FLAG_NOISE
        assert lib.rt_frame_set_convergence(frame.ptr, 1.0, 32, 8) == abi.RT_ERR_INVALID_ARGUMENT
    with h.open_frame(cam64, mw, mh, flags=NOISE) as frame:
        out = abi.RtFrameConvergence()
        assert lib.rt_frame_convergence(frame.ptr, C.byref(out)) == abi.RT_ERR_INVALID_ARGUMENT  # no rule yet
        for tol, m, k in ((-1.0, 32, 8), (float("nan"), 32, 8), (1.0, 32, 0), (1.0, 1, 8), (1.0, 11, 8), (1.0, 5, 8)):
            assert lib.rt_frame_set_convergence(frame.ptr, tol, m, k) == abi.RT_ERR_INVALID_ARGUMENT, (tol, m, k)
        assert lib.rt_frame_set_convergence(frame.ptr, 1.0, 12, 1) == abi.RT_OK  # the lowest min_samples after an 11-sample probe
        frame.set_convergence(2.0, 32, 8)  # replaces the rule
        conv = frame.convergence()
        assert (conv.tolerance, conv.min_samples, conv.interval, conv.next_check, conv.checks) == (2.0, 32, 8, 32, 0)
        assert lib.rt_frame_convergence(frame.ptr, None) == abi.RT_ERR_INVALID_ARGUMENT
        frame.advance(max_samples=1)
        assert lib.rt_frame_set_convergence(frame.ptr, 1.0, 32, 8) == abi.RT_ERR_INVALID_ARGUMENT  # after the first pass
        assert frame.convergence().min_samples == 32
    with h.open_frame(cam64, mw, mh, adaptive=False, flags=NOISE) as frame:
        assert lib.rt_frame_set_convergence(frame.ptr, 1.0, 1, 8) == abi.RT_ERR_INVALID_ARGUMENT
        assert lib.rt_frame_set_convergence(frame.ptr, 1.0, 2, 8) == abi.RT_OK  # no probe: 2 samples are enough


# ---- 8. other work on the scene ----------------------------------------------------------------------------------------------
def test_render_and_a_second_frame_between_passes(scenes):
    spec, h, cam = scenes("C2")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    tol = c2_tolerance(h, cam, mw, mh, 12)
    ref = run(h, cam, mw, mh, 12, tol, lambda f: f.advance())
    ref_rgb, ref_sums, _ = h.render(cam, mw, mh, seed=12, want_sums=True)
    with h.open_frame(cam, mw, mh, seed=12, flags=NOISE) as a, h.open_frame(cam, mw, mh, seed=12, flags=NOISE) as b:
        a.set_convergence(tol, 64, 64)
        while not a.progress.done:
            a.advance(max_samples=50)
            b.advance(max_samples=30)
            rgb, sums, _ = h.render(cam, mw, mh, seed=12, want_sums=True)
            assert np.array_equal(sums, ref_sums) and np.array_equal(rgb, ref_rgb)
        b.advance()
        sums, q = state(a)
        assert np.array_equal(sums, ref[0]) and np.array_equal(q, ref[1]) and bytes(a.convergence()) == ref[2]
        _, b_sums = b.read(want_sums=True)
        assert np.array_equal(b_sums, ref_sums)  # the plain frame is rt_render's


# ---- 9. render_progressive -----------------------------------------------------------------------------------------------
def test_render_progressive_with_a_rule(scenes):
    spec = sample_images.CONFIGS["C2"]()
    cam = oracle_camera(spec)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    s = Scene.make(spec.objects, device=0)
    tol = c2_tolerance(s.handle, cam, mw, mh, 13)
    ticks, seen = [], []
    img = Scene.render_progressive(lambda x: ticks.append(x), lambda _: None, mw, mh, cam, s, seed=13, target_ms=10.0,
                                   on_pass=lambda p, f: seen.append(f.convergence().checks), converge_tolerance=tol)
    assert len(ticks) == 2 * mh + 1 and all(t == 1.0 for t in ticks)
    assert len(seen) > 2 and seen[-1] == len(checkpoints(64, 64, spec.spp))
    with s.handle.open_frame(cam, mw, mh, seed=13, flags=NOISE) as f:
        f.set_convergence(tol, 64, 64)
        while not f.progress.done:
            f.advance()
        want, _ = f.read()
    assert np.array_equal(img, want)
