"""Progressive frames of a batch of views (rt_frame_begin_views, rt_frame_view_noise, SceneHandle.open_frame_views,
Scene.render_views_progressive).  Every sample is keyed by (view seed, pixel within the view, sample index) and the sums, Q
and counts are integers, so every check is EXACT: after every pass view v of the batch must equal rt_render of camera v and
seed v at samples_done (sums, RGB8, gamma RGB8) and a single RT_FLAG_NOISE frame of that view (Q, the E map); under a
convergence rule it must equal a single converging frame of that view at every checkpoint, the batch's counts must be the
sums of the single frames', and rt_frame_view_noise must give each single frame's rt_frame_noise summary bit for bit.
Cases: early-out on and off; 1, 2, 3 and 37 views; rows % 4 != 0 (probe tiles straddle views); pacing and extension; the
scene families and flags of test_gpu_views; interleaving with other work on the scene; argument errors.  Two child
processes report the launch plans (RTFS_DEBUG_PLAN, one with RTFS_LOCAL_STACK): all twelve render_views_noise_kernel
shapes must be launched."""
import ctypes as C
import math
import os
import subprocess
import sys

import numpy as np
import pytest

if __name__ == "__main__":  # the child processes of test_every_batched_noise_kernel_is_launched
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from ray_tracing_fsharp_b200 import abi, native, sample_images  # noqa: E402
from ray_tracing_fsharp_b200.scene import Scene  # noqa: E402
from test_gpu_views import FLAGS, device_scene, orbit  # noqa: E402

pytestmark = pytest.mark.gpu

NOISE = abi.RT_FLAG_NOISE


def with_spp(cams, spp):
    out = []
    for c in cams:
        c = abi.RtCamera.from_buffer_copy(c)
        c.samples_per_pixel = spp
        out.append(c)
    return out


def bits(summary):
    return bytes(summary)


def state(frame):
    """(sums int32 [..., rows, cols, 4], Q uint64 [..., rows, cols], E float32 bits [..., rows, cols]) of a frame or a batch."""
    _, sums = frame.read(want_sums=True)
    _, se, sq = frame.noise(0.0, want_map=True, want_sq=True)
    return sums, sq, se.view(np.uint32)


def open_pair(dsc, cams, mw, mh, seeds, adaptive=True, flags=NOISE, rule=None):
    """The batch and one frame per view, both with the same flags and rule."""
    batch = dsc.open_frame_views(cams, mw, mh, seeds=seeds, adaptive=adaptive, flags=flags)
    singles = [dsc.open_frame(c, mw, mh, seed=s, adaptive=adaptive, flags=flags) for c, s in zip(cams, seeds)]
    if rule is not None:
        for f in [batch] + singles:
            f.set_convergence(*rule)
    return batch, singles


def assert_matches_singles(batch, singles, what, noise=True, tol=None):
    """The batch's views equal the single frames: sums, RGB8, gamma RGB8 (and Q, E map, per-view summary with noise)."""
    rgb, sums = batch.read(want_sums=True)
    rgb_g, _ = batch.read(gamma=True)
    if noise:
        _, se, sq = batch.noise(0.0, want_map=True, want_sq=True)
        per_view = batch.view_noise(tol if tol is not None else 1.0)
    for v, f in enumerate(singles):
        assert f.progress.samples_done == batch.progress.samples_done, what
        r1, s1 = f.read(want_sums=True)
        g1, _ = f.read(gamma=True)
        assert np.array_equal(sums[v], s1), f"{what}: view {v} sums differ"
        assert np.array_equal(rgb[v], r1) and np.array_equal(rgb_g[v], g1), f"{what}: view {v} RGB8 differs"
        if noise:
            summary, se1, sq1 = f.noise(tol if tol is not None else 1.0, want_map=True, want_sq=True)
            assert np.array_equal(sq[v], sq1), f"{what}: view {v} Q differs"
            assert np.array_equal(se[v].view(np.uint32), se1.view(np.uint32)), f"{what}: view {v} E differs"
            assert bits(per_view[v]) == bits(summary), (what, v, per_view[v].pixels, summary.pixels, per_view[v].max_se, summary.max_se)


def assert_equals_render(dsc, batch, cams, mw, mh, seeds, adaptive, flags, views=None):
    """View v at samples_done is rt_render of camera v and seed v at samples_per_pixel = samples_done."""
    done = batch.progress.samples_done
    rgb, sums = batch.read(want_sums=True)
    rgb_g, _ = batch.read(gamma=True)
    for v in (range(len(cams)) if views is None else views):
        cam = with_spp([cams[v]], done)[0]
        r1, s1, _ = dsc.render(cam, mw, mh, seed=seeds[v], adaptive=adaptive, flags=flags & ~NOISE, want_sums=True)
        g1, _, _ = dsc.render(cam, mw, mh, seed=seeds[v], adaptive=adaptive, flags=flags & ~NOISE, gamma=True)
        assert np.array_equal(sums[v], s1), f"view {v} at {done} spp: sums differ from rt_render"
        assert np.array_equal(rgb[v], r1) and np.array_equal(rgb_g[v], g1), f"view {v} at {done} spp: RGB8 differs from rt_render"


def close(*frames):
    for f in frames:
        f.close()


# ---- 1. every pass: rt_render and the single noise frame -------------------------------------------------------------------
@pytest.mark.parametrize("adaptive", [True, False])
@pytest.mark.parametrize("n", [1, 2, 3, 37])
def test_every_pass_equals_render_and_single_frames(n, adaptive):
    spec, dsc = device_scene("C1")  # 81 x 43: 43 % 4 == 3, probe tiles straddle views
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cams = orbit(spec, n)
    seeds = [100 + 7 * v + (v << 40) for v in range(n)]
    batch, singles = open_pair(dsc, cams, mw, mh, seeds, adaptive)
    rows, cols = 2 * mh + 1, 2 * mw + 1
    assert batch.n_views == n and batch.progress.samples_target == singles[0].progress.samples_target
    assert batch.progress.pixels_flagged == sum(f.progress.pixels_flagged for f in singles)
    step = 0
    while True:
        assert batch.progress.paths_done == sum(f.progress.paths_done for f in singles)
        assert batch.progress.paths_target == sum(f.progress.paths_target for f in singles)
        assert_matches_singles(batch, singles, f"n={n} pass {step}")
        if batch.progress.samples_done > 0:
            assert_equals_render(dsc, batch, cams, mw, mh, seeds, adaptive, NOISE, views=None if n <= 3 else [0, 17, 36])
        if batch.progress.done:
            break
        batch.advance(max_samples=3)
        for f in singles:
            f.advance(max_samples=3)
        step += 1
    rgb, sums = batch.read(want_sums=True)
    assert rgb.shape == (n, rows, cols, 3) and sums.shape == (n, rows, cols, 4)
    if n == 1:  # a one-view batch's view summary is its frame summary
        assert bits(batch.view_noise(0.5)[0]) == bits(batch.noise(0.5, want_map=False)[0])
    close(batch, *singles)


# ---- 2. a convergence rule: every checkpoint --------------------------------------------------------------------------------
@pytest.mark.parametrize("adaptive", [True, False])
@pytest.mark.parametrize("tol", [0.0, 0.5, 1.0])
def test_converging_batch_equals_converging_frames(tol, adaptive):
    spec, dsc = device_scene("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cams = with_spp(orbit(spec, 3), 48)
    seeds = [5, 1 << 33, 2 ** 64 - 1]
    rule = (tol, 16, 8)
    batch, singles = open_pair(dsc, cams, mw, mh, seeds, adaptive, rule=rule)
    converged = 0
    while not batch.progress.done:
        batch.advance(max_samples=5)
        for f in singles:
            f.advance(max_samples=5)
        assert_matches_singles(batch, singles, f"tau={tol} at {batch.progress.samples_done}", tol=tol)
        conv, ones = batch.convergence(), [f.convergence() for f in singles]
        assert conv.checks == ones[0].checks and all(o.checks == conv.checks for o in ones)
        assert conv.next_check == ones[0].next_check
        assert conv.pixels_active == sum(o.pixels_active for o in ones)
        assert conv.pixels_converged == sum(o.pixels_converged for o in ones)
        assert batch.progress.paths_done == sum(f.progress.paths_done for f in singles)
        assert batch.progress.paths_target == sum(f.progress.paths_target for f in singles)
        converged = conv.pixels_converged
        done = batch.progress.samples_done
        if conv.pixels_active and done >= 16 and done % 8 == 0:  # right after a check every pixel still sampled is above tau
            assert all(s.pixels_above == s.pixels for s in batch.view_noise(tol))
    assert all(f.progress.done for f in singles)
    if not adaptive and tol > 0.0:
        assert converged > 0
    close(batch, *singles)


# ---- 3. pacing and extension ------------------------------------------------------------------------------------------------
def _run(dsc, cams, mw, mh, seeds, rule, pace, spp=None):
    f = dsc.open_frame_views(with_spp(cams, spp) if spp else cams, mw, mh, seeds=seeds, flags=NOISE)
    f.set_convergence(*rule)
    while not f.progress.done:
        f.advance(**pace)
    out = state(f), f.convergence().pixels_converged, f.progress.paths_done
    f.close()
    return out


def test_pacing_does_not_change_the_batch():
    spec, dsc = device_scene("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cams = with_spp(orbit(spec, 4), 64)
    seeds = [1, 2, 3, 4]
    rule = (1.0, 16, 8)
    want = _run(dsc, cams, mw, mh, seeds, rule, {})
    for pace in ({"max_samples": 1}, {"max_samples": 7}, {"target_ms": 0.5}):
        got = _run(dsc, cams, mw, mh, seeds, rule, pace)
        for a, b in zip(want[0], got[0]):
            assert np.array_equal(a, b), pace
        assert want[1:] == got[1:], pace


def test_extended_batch_equals_batch_opened_there():
    spec, dsc = device_scene("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cams = with_spp(orbit(spec, 3), 256)
    seeds = [9, 10, 11]
    rule = (1.0, 64, 64)
    f = dsc.open_frame_views(cams, mw, mh, seeds=seeds, flags=NOISE)
    f.set_convergence(*rule)
    while not f.progress.done:
        f.advance(max_samples=100)
    f.extend(512)
    while not f.advance(max_samples=100).done:
        pass
    got = state(f)
    f.close()
    want = _run(dsc, cams, mw, mh, seeds, rule, {}, spp=512)[0]
    for a, b in zip(want, got):
        assert np.array_equal(a, b)


# ---- 4. scene families and flags --------------------------------------------------------------------------------------------
def _family(name, n, flags, spp=24, rule=(1.0, 12, 4), adaptive=True):
    spec, dsc = device_scene(name)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cams = with_spp(orbit(spec, n), spp)
    seeds = [41 + v for v in range(n)]
    noise = bool(flags & NOISE)
    batch, singles = open_pair(dsc, cams, mw, mh, seeds, adaptive, flags, rule if noise else None)
    while not batch.progress.done:
        batch.advance(max_samples=5)
        for f in singles:
            f.advance(max_samples=5)
        assert_matches_singles(batch, singles, f"{name} flags={flags} at {batch.progress.samples_done}", noise=noise,
                               tol=rule[0] if noise else None)
    if not noise:
        assert_equals_render(dsc, batch, cams, mw, mh, seeds, adaptive, flags)
    close(batch, *singles)


@pytest.mark.parametrize("name,n", [("C1", 3), ("C3", 3), ("C4", 3), ("C5", 3), ("stage-n*+1", 3), ("C2", 2)])
def test_scene_families(name, n):
    _family(name, n, NOISE)


@pytest.mark.parametrize("flag", sorted(FLAGS))
@pytest.mark.parametrize("name", ["C1", "C3", "stage-n*+1"])
def test_flags(name, flag):
    for adaptive in (True, False):
        _family(name, 3, NOISE | FLAGS[flag], adaptive=adaptive)


@pytest.mark.parametrize("flag", sorted(FLAGS))
def test_batch_without_noise_is_exact(flag):
    """Without RT_FLAG_NOISE the batch runs render_views_kernel, pass by pass."""
    _family("C1", 3, FLAGS[flag])


def test_view_noise_of_many_views_of_a_small_extent():
    """70 000 views of 3 x 3 pixels: more views than one launch's grid has rows, reduced in chunks of views.  Sampled views
    equal single frames' summaries bit for bit, and the views' pixel counts add up to the batch's."""
    spec, dsc = device_scene("C1")
    n = 70000
    cams = orbit(spec, n)
    seeds = [3 * v + 1 for v in range(n)]
    with dsc.open_frame_views(cams, 1, 1, seeds=seeds, adaptive=False, flags=NOISE) as batch:
        batch.advance(max_samples=4)
        per_view = batch.view_noise(2.0)
        whole, _, _ = batch.noise(2.0, want_map=False)
        assert len(per_view) == n
        assert sum(s.pixels for s in per_view) == whole.pixels == 9 * n
        assert sum(s.pixels_above for s in per_view) == whole.pixels_above
        for v in (0, 1023, 1024, 65535, 65536, n - 1):
            with dsc.open_frame(cams[v], 1, 1, seed=seeds[v], adaptive=False, flags=NOISE) as one:
                one.advance(max_samples=4)
                assert bits(per_view[v]) == bits(one.noise(2.0, want_map=False)[0]), v


# ---- 5. launch plans ----------------------------------------------------------------------------------------------------------
PLAN_SCENES = {"C1": ["default", "no-lean", "no-smem", "wide-bvh"], "C3": ["default"], "stage-n*+1": ["default", "wide-bvh"]}


def plans_child():
    for name, flags in PLAN_SCENES.items():
        spec, dsc = device_scene(name)
        for flag in flags:
            with dsc.open_frame_views(orbit(spec, 2), spec.max_width_coord, spec.max_height_coord, seeds=[1, 2],
                                      flags=NOISE | FLAGS[flag]) as f:
                f.advance()
    print("plans child: ok")


def _plans(extra_env):
    env = dict(os.environ, RTFS_DEBUG_PLAN="1", **extra_env)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "plans"], env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0 and "plans child: ok" in r.stdout, r.stdout[-4000:] + r.stderr[-4000:]
    reached = set()
    for line in r.stderr.splitlines():
        if not line.startswith("rtfs: plan "):
            continue
        kv = dict(x.split("=") for x in line[len("rtfs: plan "):].split())
        assert kv["views"] == "2" and kv["noise"] == "1" and kv["count"] == "0" and kv["flow"] == "0", line
        reached.add((kv["probe"], kv["staged"], kv["lean"], kv["sstack"], kv["wide"]))
    return reached


def test_every_batched_noise_kernel_is_launched():
    reached = _plans({}) | _plans({"RTFS_LOCAL_STACK": "1"})
    want = set()
    for probe in "10":
        want |= {(probe, "1", "1", "0", "0"), (probe, "1", "0", "0", "0")}
        want |= {(probe, "0", "0", s, w) for s in "01" for w in "01"}
    assert len(want) == 12
    assert want <= reached, sorted(want - reached)


# ---- 6. interleaving ----------------------------------------------------------------------------------------------------------
def test_interleaved_with_other_work_on_the_scene():
    """Between two passes: rt_render_views with other (and more) cameras, which rewrites and grows the workspace's view
    table, rt_render, and another progressive frame.  The batch owns its table, so it stays exact."""
    spec, dsc = device_scene("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cams = with_spp(orbit(spec, 3), 40)
    seeds = [21, 22, 23]
    rule = (0.5, 16, 8)
    want = _run(dsc, cams, mw, mh, seeds, rule, {"max_samples": 6})
    batch = dsc.open_frame_views(cams, mw, mh, seeds=seeds, flags=NOISE)
    batch.set_convergence(*rule)
    other = dsc.open_frame(orbit(spec, 5)[4], mw, mh, seed=77)
    k = 0
    while not batch.progress.done:
        batch.advance(max_samples=6)
        others = orbit(spec, 7 + k)
        dsc.render_views(others, mw + k, mh, seeds=list(range(len(others))))
        dsc.render(others[1], mw, mh, seed=3)
        other.advance(max_samples=2)
        k += 1
    got = state(batch), batch.convergence().pixels_converged, batch.progress.paths_done
    for a, b in zip(want[0], got[0]):
        assert np.array_equal(a, b)
    assert want[1:] == got[1:]
    close(batch, other)


# ---- 7. errors and Scene.render_views_progressive --------------------------------------------------------------------------
def _raw(dsc, cams, n, mw, mh, opts, out=True):
    arr = (abi.RtCamera * max(1, len(cams)))(*cams) if cams is not None else None
    ptr = C.c_void_p()
    rc = native.lib().rt_frame_begin_views(dsc.ptr, arr, None, n, mw, mh, C.byref(opts), C.byref(ptr) if out else None, None)
    if ptr.value:
        native.lib().rt_frame_destroy(ptr)
    return rc


def test_argument_errors():
    spec, dsc = device_scene("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cams = orbit(spec, 2)
    opts = abi.RtRenderOpts(1, 1, abi.RT_MODE_MEGAKERNEL, 0, NOISE)
    assert _raw(dsc, cams, 2, mw, mh, opts) == abi.RT_OK
    assert _raw(dsc, cams, 0, mw, mh, opts) == abi.RT_ERR_INVALID_ARGUMENT
    assert _raw(dsc, cams, -3, mw, mh, opts) == abi.RT_ERR_INVALID_ARGUMENT
    assert _raw(dsc, None, 2, mw, mh, opts) == abi.RT_ERR_INVALID_ARGUMENT
    assert _raw(dsc, cams, 2, mw, mh, opts, out=False) == abi.RT_ERR_INVALID_ARGUMENT
    for field, value in (("samples_per_pixel", spec.spp + 1), ("bounce_depth", spec.bounce_depth + 1)):
        odd = orbit(spec, 2)
        setattr(odd[1], field, value)
        assert _raw(dsc, odd, 2, mw, mh, opts) == abi.RT_ERR_INVALID_ARGUMENT, field
    assert _raw(dsc, cams, 2, 32767, 16383, opts) == abi.RT_ERR_INVALID_ARGUMENT  # 2 x 65535 x 32767 >= 2^31
    for extra in (0, NOISE):
        for mode, flags in ((abi.RT_MODE_WAVEFRONT, 0), (abi.RT_MODE_MEGAKERNEL, abi.RT_FLAG_FLOW),
                            (abi.RT_MODE_MEGAKERNEL, abi.RT_FLAG_COUNTERS), (abi.RT_MODE_MEGAKERNEL, abi.RT_FLAG_FLOW | abi.RT_FLAG_LOCKSTEP)):
            o = abi.RtRenderOpts(1, 1, mode, 0, flags | extra)
            assert _raw(dsc, cams, 2, mw, mh, o) == abi.RT_ERR_UNSUPPORTED, (mode, flags, extra)
    with pytest.raises(ValueError):
        dsc.open_frame_views(cams, mw, mh, seeds=[1])
    lib = native.lib()
    with dsc.open_frame_views(cams, mw, mh, seeds=[1, 2]) as plain:
        out = (abi.RtFrameNoise * 2)()
        assert lib.rt_frame_view_noise(plain.ptr, 1.0, out) == abi.RT_ERR_INVALID_ARGUMENT  # without RT_FLAG_NOISE
    with dsc.open_frame_views(cams, mw, mh, seeds=[1, 2], flags=NOISE) as f:
        out = (abi.RtFrameNoise * 2)()
        assert lib.rt_frame_view_noise(f.ptr, 1.0, None) == abi.RT_ERR_INVALID_ARGUMENT
        assert lib.rt_frame_view_noise(f.ptr, -1.0, out) == abi.RT_ERR_INVALID_ARGUMENT
        assert lib.rt_frame_view_noise(f.ptr, math.nan, out) == abi.RT_ERR_INVALID_ARGUMENT
        assert lib.rt_frame_view_noise(None, 1.0, out) == abi.RT_ERR_INVALID_ARGUMENT
        assert lib.rt_frame_view_noise(f.ptr, 1.0, out) == abi.RT_OK
    # a frame of one camera has one view
    with dsc.open_frame(cams[0], mw, mh, seed=1, flags=NOISE) as f:
        assert bits(f.view_noise(2.0)[0]) == bits(f.noise(2.0, want_map=False)[0])


def test_scene_render_views_progressive():
    spec = sample_images.few_spheres(max_w=20, max_h=10, spp=48)
    scene = Scene.make(spec.objects, device=0)
    cams = orbit(spec, 3)
    rows = spec.rows
    for rule in (None, 1.0):
        ticks = []
        images = Scene.render_views_progressive(ticks.append, lambda _: None, spec.max_width_coord, spec.max_height_coord, cams, scene,
                                                seeds=[4, 5, 6], target_ms=0.05, converge_tolerance=rule, converge_min_samples=16,
                                                converge_interval=8)
        assert len(images) == 3 and len(ticks) == rows * 3
        for v, img in enumerate(images):
            want = Scene.render_progressive(lambda _: None, lambda _: None, spec.max_width_coord, spec.max_height_coord, cams[v], scene,
                                            seed=4 + v, converge_tolerance=rule, converge_min_samples=16, converge_interval=8)
            assert img.shape == (rows, spec.cols, 3) and np.array_equal(img, want), (rule, v)
    # stopping through on_pass: the views of the samples done at the stop
    seen = []

    def stop(progress, frame):
        seen.append(progress.samples_done)
        return len(seen) == 2

    ticks = []
    images = Scene.render_views_progressive(ticks.append, lambda _: None, spec.max_width_coord, spec.max_height_coord, cams, scene,
                                            seeds=[4, 5, 6], target_ms=0.0, on_pass=stop)
    assert len(seen) == 1 and len(ticks) == rows * 3  # target_ms = 0: one pass takes everything left
    ticks = []
    seen.clear()

    def stop_early(progress, frame):
        seen.append(progress.samples_done)
        return True

    dsc = scene.handle
    images = Scene.render_views_progressive(ticks.append, lambda _: None, spec.max_width_coord, spec.max_height_coord, cams, scene,
                                            seeds=[4, 5, 6], target_ms=1e-6, on_pass=stop_early)
    assert len(seen) == 1 and seen[0] < 48 and len(ticks) == rows * 3
    for v, img in enumerate(images):
        want, _, _ = dsc.render(with_spp([cams[v]], seen[0])[0], spec.max_width_coord, spec.max_height_coord, seed=4 + v)
        assert np.array_equal(img, want)


if __name__ == "__main__" and sys.argv[1:] == ["plans"]:
    plans_child()
