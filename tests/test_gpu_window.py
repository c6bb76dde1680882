"""Windows of a frame (rt_render_window, rt_frame_begin_window, SceneHandle.render_window / open_frame_window,
Scene.render_window, Scene.render_progressive(window=...)).  Every sample is keyed by (seed, frame pixel, sample index) and the
sums, Q and counts are integers, so every check is EXACT: a window must equal the crop of rt_render's frame (sums, RGB8, gamma
RGB8), its paths must be what its own pixels take, tiles of uneven grids must reassemble into the frame, and after every pass
a progressive window must equal the crop of the full progressive frame (sums, Q, E map; under a convergence rule too).
Cases: C1-C5 and a scene one sphere past the staging limit; early-out on and off; the flags of test_gpu_views; two seeds;
the whole frame, one pixel, one row, one column, the corners and odd windows off the 8 x 4 tile grid; pacing and extension;
the noise summary; interleaving with other work on the scene; the mode refusals.  Two child processes report the launch plans
(RTFS_DEBUG_PLAN, one with RTFS_LOCAL_STACK): all 24 window kernels must be launched and named."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

if __name__ == "__main__":  # the child processes of test_every_window_kernel_is_launched
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from ray_tracing_fsharp_b200 import abi, native, sample_images  # noqa: E402
from ray_tracing_fsharp_b200.scene import Image, Scene  # noqa: E402
from test_gpu_views import FLAGS, device_scene, orbit  # noqa: E402

pytestmark = pytest.mark.gpu

NOISE = abi.RT_FLAG_NOISE


def camera(spec, spp=None):
    cam = orbit(spec, 1)[0]  # the spec's own camera (angle 0)
    if spp is not None:
        cam.samples_per_pixel = spp
    return cam


def windows(rows, cols):
    """(row0, col0, rows, cols): the whole frame, one pixel, one row, one column, the four corners, odd windows off the tiles."""
    h, w = min(5, rows), min(7, cols)
    return [(0, 0, rows, cols), (rows // 2, cols // 2, 1, 1), (rows // 3, 0, 1, cols), (0, cols // 3, rows, 1),
            (0, 0, h, w), (0, cols - w, h, w), (rows - h, 0, h, w), (rows - h, cols - w, h, w),
            (1, 3, min(9, rows - 1), min(13, cols - 3)), (rows // 2 + 1, cols // 2 + 5, min(11, rows - rows // 2 - 1), min(17, cols - cols // 2 - 5)),
            (2, 5, rows - 3, cols - 6)]


def crop(a, w):
    r0, c0, r, c = w
    return a[r0:r0 + r, c0:c0 + c]


def n_probe_of(spp, adaptive):
    return 2 * min(5, spp // 2) + 1 if adaptive else 0


def check_windows(dsc, cam, mw, mh, wins, seed, adaptive=True, flags=0):
    """Each window against the crop of one rt_render: sums, RGB8 and gamma RGB8 equal; paths from the frame's counts."""
    full, full_sums, full_st = dsc.render(cam, mw, mh, seed=seed, adaptive=adaptive, flags=flags, want_sums=True)
    full_g, _, _ = dsc.render(cam, mw, mh, seed=seed, adaptive=adaptive, flags=flags, gamma=True)
    n_probe = n_probe_of(cam.samples_per_pixel, adaptive)
    spp = max(n_probe, cam.samples_per_pixel)
    for w in wins:
        rgb, sums, st = dsc.render_window(cam, mw, mh, w, seed=seed, adaptive=adaptive, flags=flags, want_sums=True)
        rgb_g, _, _ = dsc.render_window(cam, mw, mh, w, seed=seed, adaptive=adaptive, flags=flags, gamma=True)
        assert rgb.shape == (w[2], w[3], 3) and sums.shape == (w[2], w[3], 4)
        assert np.array_equal(sums, crop(full_sums, w)), f"window {w}: sums differ"
        assert np.array_equal(rgb, crop(full, w)), f"window {w}: RGB8 differs"
        assert np.array_equal(rgb_g, crop(full_g, w)), f"window {w}: gamma RGB8 differs"
        flagged = int((crop(full_sums, w)[..., 3] > n_probe).sum())
        assert st.paths == w[2] * w[3] * n_probe + flagged * (spp - n_probe), (w, st.paths)
        assert st.pixels_early_out == (w[2] * w[3] - flagged if adaptive else 0), w
        if w[2:] == (2 * mh + 1, 2 * mw + 1):  # the whole frame: rt_render in every output
            for k in ("paths", "rays", "pixels_early_out", "degenerate_paths", "launches", "box_tests", "prim_tests"):
                assert getattr(st, k) == getattr(full_st, k), (k, getattr(st, k), getattr(full_st, k))
            assert st.kernel_ms > 0.0
    return full_sums, full_st


# ---- 1. windows of one frame ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("adaptive", [True, False])
@pytest.mark.parametrize("name", ["C1", "C2", "C3", "C4", "C5", "stage-n*+1"])
def test_windows_equal_the_crop_of_render(name, adaptive):
    spec, dsc = device_scene(name)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cam = camera(spec)
    for seed in (7, 2 ** 64 - 3):
        check_windows(dsc, cam, mw, mh, windows(2 * mh + 1, 2 * mw + 1), seed, adaptive)


@pytest.mark.parametrize("flag", sorted(FLAGS))
@pytest.mark.parametrize("name", ["C1", "C3", "stage-n*+1"])
def test_flags(name, flag):
    spec, dsc = device_scene(name)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    rows, cols = 2 * mh + 1, 2 * mw + 1
    for adaptive in (True, False):
        check_windows(dsc, camera(spec), mw, mh, [(0, 0, rows, cols), (1, 3, 9, 13), (rows - 6, cols - 11, 6, 11)], 5, adaptive,
                      FLAGS[flag])


def test_noise_flag_is_ignored():
    spec, dsc = device_scene("C1")
    cam, w = camera(spec), (2, 3, 17, 29)
    a = dsc.render_window(cam, spec.max_width_coord, spec.max_height_coord, w, seed=9, want_sums=True)
    b = dsc.render_window(cam, spec.max_width_coord, spec.max_height_coord, w, seed=9, want_sums=True, flags=NOISE)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


# ---- 2. tiles -----------------------------------------------------------------------------------------------------------------
def uneven_cuts(n, parts, rng):
    cuts = np.sort(rng.choice(np.arange(1, n), parts - 1, replace=False))
    return [0] + [int(c) for c in cuts] + [n]


@pytest.mark.parametrize("name,grid", [("C2", (4, 4)), ("C4", (3, 5))])
def test_tiles_reassemble_into_the_frame(name, grid):
    spec, dsc = device_scene(name)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    rows, cols = 2 * mh + 1, 2 * mw + 1
    cam = camera(spec)
    rng = np.random.default_rng(len(name) + grid[0])
    for adaptive in (True, False):
        full, full_sums, full_st = dsc.render(cam, mw, mh, seed=31, adaptive=adaptive, want_sums=True)
        rgb = np.zeros_like(full)
        sums = np.full_like(full_sums, -1)
        paths = rays = early = 0
        rc, cc = uneven_cuts(rows, grid[0], rng), uneven_cuts(cols, grid[1], rng)
        for i in range(grid[0]):
            for j in range(grid[1]):
                w = (rc[i], cc[j], rc[i + 1] - rc[i], cc[j + 1] - cc[j])
                t_rgb, t_sums, st = dsc.render_window(cam, mw, mh, w, seed=31, adaptive=adaptive, want_sums=True)
                rgb[w[0]:w[0] + w[2], w[1]:w[1] + w[3]] = t_rgb
                sums[w[0]:w[0] + w[2], w[1]:w[1] + w[3]] = t_sums
                paths, rays, early = paths + st.paths, rays + st.rays, early + st.pixels_early_out
        assert np.array_equal(sums, full_sums) and np.array_equal(rgb, full), (name, adaptive)
        assert (paths, rays, early) == (full_st.paths, full_st.rays, full_st.pixels_early_out)


# ---- 3. progressive windows -------------------------------------------------------------------------------------------------
def state(frame):
    """(sums int32 [rows, cols, 4], Q uint64 [rows, cols], E float32 bits [rows, cols])."""
    _, sums = frame.read(want_sums=True)
    _, se, sq = frame.noise(0.0, want_map=True, want_sq=True)
    return sums, sq, se.view(np.uint32)


def assert_crop_of(win, full, w, what):
    for a, b, k in zip(state(win), state(full), ("sums", "Q", "E")):
        assert np.array_equal(a, crop(b, w)), f"{what}: {k} differ"


@pytest.mark.parametrize("adaptive", [True, False])
@pytest.mark.parametrize("w", [(0, 0, 43, 81), (5, 9, 13, 30), (40, 0, 3, 81), (0, 77, 43, 4), (21, 40, 1, 1)])
def test_every_pass_equals_the_crop(w, adaptive):
    spec, dsc = device_scene("C1")  # 81 x 43
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cam = camera(spec, 16)
    seed = 123 + (1 << 40)
    win = dsc.open_frame_window(cam, mw, mh, w, seed=seed, adaptive=adaptive, flags=NOISE)
    full = dsc.open_frame(cam, mw, mh, seed=seed, adaptive=adaptive, flags=NOISE)
    n_probe = n_probe_of(16, adaptive)
    assert win.progress.samples_target == full.progress.samples_target
    step = 0
    while True:
        p = win.progress
        assert p.samples_done == full.progress.samples_done
        assert_crop_of(win, full, w, f"{w} pass {step}")
        _, full_sums = full.read(want_sums=True)
        flagged = int((crop(full_sums, w)[..., 3] > n_probe).sum()) if p.samples_done > n_probe else p.pixels_flagged
        assert p.pixels_flagged == flagged
        assert p.paths_target == w[2] * w[3] * n_probe + flagged * (p.samples_target - n_probe)
        if p.samples_done > 0:
            at = camera(spec, p.samples_done)
            r1, s1, _ = dsc.render(at, mw, mh, seed=seed, adaptive=adaptive, want_sums=True)
            g1, _, _ = dsc.render(at, mw, mh, seed=seed, adaptive=adaptive, gamma=True)
            rgb, sums = win.read(want_sums=True)
            rgb_g, _ = win.read(gamma=True)
            assert np.array_equal(sums, crop(s1, w)) and np.array_equal(rgb, crop(r1, w)) and np.array_equal(rgb_g, crop(g1, w)), step
        if p.done:
            break
        win.advance(max_samples=3)
        full.advance(max_samples=3)
        step += 1
    assert p.paths_done == p.paths_target
    win.close()
    full.close()


@pytest.mark.parametrize("adaptive", [True, False])
@pytest.mark.parametrize("tol", [0.0, 0.5, 1.0])
def test_converging_window_equals_the_crop_of_the_converging_frame(tol, adaptive):
    spec, dsc = device_scene("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cam = camera(spec, 48)
    w = (3, 11, 29, 45)
    rule = (tol, 16, 8)
    win = dsc.open_frame_window(cam, mw, mh, w, seed=5, adaptive=adaptive, flags=NOISE)
    full = dsc.open_frame(cam, mw, mh, seed=5, adaptive=adaptive, flags=NOISE)
    for f in (win, full):
        f.set_convergence(*rule)
    while not (win.progress.done and full.progress.done):
        win.advance(max_samples=5)
        full.advance(max_samples=5)
        assert win.progress.samples_done == full.progress.samples_done or win.progress.done
        if win.progress.samples_done == full.progress.samples_done:
            assert_crop_of(win, full, w, f"tau={tol} at {win.progress.samples_done}")
    assert_crop_of(win, full, w, f"tau={tol} at the end")
    conv = win.convergence()
    _, full_sums = full.read(want_sums=True)
    counts = crop(full_sums, w)[..., 3]
    n_probe = n_probe_of(48, adaptive)
    assert conv.pixels_active + conv.pixels_converged == win.progress.pixels_flagged
    assert conv.pixels_converged >= int(((counts > n_probe) & (counts < 48)).sum())  # (those stopped at 48 look like the rest)
    if not adaptive and tol > 0.0:
        assert conv.pixels_converged > 0
    win.close()
    full.close()


def _run(dsc, cam, mw, mh, w, rule, pace):
    f = dsc.open_frame_window(cam, mw, mh, w, seed=77, flags=NOISE)
    f.set_convergence(*rule)
    while not f.progress.done:
        f.advance(**pace)
    out = state(f), f.convergence().pixels_converged, f.progress.paths_done
    f.close()
    return out


def test_pacing_does_not_change_the_window():
    spec, dsc = device_scene("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cam, w, rule = camera(spec, 64), (4, 6, 31, 57), (1.0, 16, 8)
    want = _run(dsc, cam, mw, mh, w, rule, {})
    for pace in ({"max_samples": 1}, {"max_samples": 7}, {"target_ms": 0.5}):
        got = _run(dsc, cam, mw, mh, w, rule, pace)
        for a, b in zip(want[0], got[0]):
            assert np.array_equal(a, b), pace
        assert want[1:] == got[1:], pace


def test_extended_window_equals_window_opened_there():
    spec, dsc = device_scene("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    w, rule = (9, 2, 21, 63), (1.0, 64, 64)
    f = dsc.open_frame_window(camera(spec, 256), mw, mh, w, seed=77, flags=NOISE)
    f.set_convergence(*rule)
    while not f.progress.done:
        f.advance(max_samples=100)
    f.extend(512)
    while not f.advance(max_samples=100).done:
        pass
    got = state(f)
    f.close()
    want = _run(dsc, camera(spec, 512), mw, mh, w, rule, {})[0]
    for a, b in zip(want, got):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("name", ["C2", "C4", "C5", "stage-n*+1"])
def test_progressive_scene_families(name):
    spec, dsc = device_scene(name)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    rows, cols = 2 * mh + 1, 2 * mw + 1
    cam = camera(spec, 24)
    w = (rows // 4 + 1, cols // 4 + 3, rows // 2, cols // 2)
    win = dsc.open_frame_window(cam, mw, mh, w, seed=41, flags=NOISE)
    full = dsc.open_frame(cam, mw, mh, seed=41, flags=NOISE)
    for f in (win, full):
        f.set_convergence(1.0, 12, 4)
    while not full.progress.done:
        win.advance(max_samples=5)
        full.advance(max_samples=5)
        assert_crop_of(win, full, w, f"{name} at {full.progress.samples_done}")
    win.close()
    full.close()


# ---- 4. the noise summary ------------------------------------------------------------------------------------------------------
def standard_error(sums, sq):
    """E of every pixel in double, exactly as the library computes it (include/rtfs_b200.h, rt_frame_noise)."""
    n = sums[..., 3].astype(np.int64)
    t = sums[..., :3].astype(np.int64)
    d = (n.astype(np.uint64) * sq - (t * t).sum(-1).astype(np.uint64)).astype(np.int64)
    nd = n.astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        e = np.sqrt(d.astype(np.float64) / (3.0 * nd * nd * (n - 1).astype(np.float64)))
    return np.where(n < 2, np.inf, e)


@pytest.mark.parametrize("adaptive", [True, False])
def test_noise_summary_is_the_crop_of_the_frame(adaptive):
    spec, dsc = device_scene("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cam = camera(spec, 40)
    w = (6, 13, 27, 51)
    with dsc.open_frame_window(cam, mw, mh, w, seed=3, adaptive=adaptive, flags=NOISE) as win, \
            dsc.open_frame(cam, mw, mh, seed=3, adaptive=adaptive, flags=NOISE) as full:
        for k in (13, 9):
            win.advance(max_samples=k)
            full.advance(max_samples=k)
            _, full_sums = full.read(want_sums=True)
            _, full_se, full_sq = full.noise(0.0, want_map=True, want_sq=True)
            e = standard_error(full_sums, full_sq)
            assert np.array_equal(e.astype(np.float32).view(np.uint32), full_se.view(np.uint32))
            done = full.progress.samples_done
            flagged = crop(full_sums, w)[..., 3] == done  # the pixels later passes still sample (done > n_probe here)
            ec = crop(e, w)[flagged]
            for tol in (0.0, 0.7, 2.5):
                summary, _, _ = win.noise(tol, want_map=False)
                assert summary.pixels == flagged.sum() and summary.pixels_above == int((ec > tol).sum())
                assert summary.max_se == (ec.max() if ec.size else 0.0)
                assert abs(summary.mean_se - ec.mean()) <= 1e-12 * abs(ec.mean())
                per_view = win.view_noise(tol)
                assert len(per_view) == 1 and bytes(per_view[0]) == bytes(summary)


# ---- 5. interleaving --------------------------------------------------------------------------------------------------------
def test_interleaved_with_other_work_on_the_scene():
    """Between two passes: rt_render, rt_render_views, rt_render_window and another progressive frame on the same scene."""
    spec, dsc = device_scene("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cam, w, rule = camera(spec, 40), (7, 20, 19, 33), (0.5, 16, 8)
    want = _run(dsc, cam, mw, mh, w, rule, {"max_samples": 6})
    f = dsc.open_frame_window(cam, mw, mh, w, seed=77, flags=NOISE)
    f.set_convergence(*rule)
    other = dsc.open_frame(orbit(spec, 5)[4], mw, mh, seed=78)
    k = 0
    while not f.progress.done:
        f.advance(max_samples=6)
        others = orbit(spec, 3 + k)
        dsc.render_views(others, mw + k, mh, seeds=list(range(len(others))))
        dsc.render(others[1], mw, mh + k, seed=3)
        dsc.render_window(others[2], mw + 2, mh + 1, (k, k, 9 + k, 40), seed=4)
        other.advance(max_samples=2)
        k += 1
    got = state(f), f.convergence().pixels_converged, f.progress.paths_done
    for a, b in zip(want[0], got[0]):
        assert np.array_equal(a, b)
    assert want[1:] == got[1:]
    f.close()
    other.close()


# ---- 6. refusals on the device path -----------------------------------------------------------------------------------------
def test_modes_refused():
    spec, dsc = device_scene("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cam, w = camera(spec), (1, 2, 10, 20)
    lib = native.lib()
    rgb = np.zeros((10, 20, 3), np.uint8)
    for extra in (0, NOISE):
        for mode, flags in ((abi.RT_MODE_WAVEFRONT, 0), (abi.RT_MODE_MEGAKERNEL, abi.RT_FLAG_FLOW),
                            (abi.RT_MODE_MEGAKERNEL, abi.RT_FLAG_COUNTERS), (abi.RT_MODE_MEGAKERNEL, abi.RT_FLAG_FLOW | abi.RT_FLAG_LOCKSTEP)):
            o = abi.RtRenderOpts(1, 1, mode, 0, flags | extra)
            assert lib.rt_render_window(dsc.ptr, C.byref(cam), mw, mh, *w, C.byref(o), native.ptr(rgb), None, None) == abi.RT_ERR_UNSUPPORTED
            out = C.c_void_p()
            assert lib.rt_frame_begin_window(dsc.ptr, C.byref(cam), mw, mh, *w, C.byref(o), C.byref(out), None) == abi.RT_ERR_UNSUPPORTED
            assert out.value is None
    for bad in ((0, 0, 44, 81), (0, 1, 43, 81), (-1, 0, 2, 2), (0, 0, 0, 1)):
        with pytest.raises(native.RtError) as e:
            dsc.render_window(cam, mw, mh, bad)
        assert e.value.code == abi.RT_ERR_INVALID_ARGUMENT
    check_windows(dsc, cam, mw, mh, [w], 2)  # the scene still renders after the refusals


# ---- 7. launch plans ----------------------------------------------------------------------------------------------------------
PLAN_SCENES = {"C1": ["default", "no-lean", "no-smem", "wide-bvh"], "C3": ["default"], "stage-n*+1": ["default", "wide-bvh"]}
PLAN_WINDOW = (3, 5, 20, 30)


def plans_child():
    for name, flags in PLAN_SCENES.items():
        spec, dsc = device_scene(name)
        cam = camera(spec, 24)
        for flag in flags:
            dsc.render_window(cam, spec.max_width_coord, spec.max_height_coord, PLAN_WINDOW, seed=1, flags=FLAGS[flag])
            with dsc.open_frame_window(cam, spec.max_width_coord, spec.max_height_coord, PLAN_WINDOW, seed=1, flags=NOISE | FLAGS[flag]) as f:
                f.advance()
    spec, dsc = device_scene("C1")
    sys.stderr.write("single frame\n")
    dsc.render(camera(spec), spec.max_width_coord, spec.max_height_coord, seed=1)
    print("plans child: ok")


def _plans(extra_env):
    env = dict(os.environ, RTFS_DEBUG_PLAN="1", **extra_env)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "plans"], env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0 and "plans child: ok" in r.stdout, r.stdout[-4000:] + r.stderr[-4000:]
    reached, single, after = set(), [], False
    r0, c0, rows, cols = PLAN_WINDOW
    for line in r.stderr.splitlines():
        if line == "single frame":
            after = True
        if not line.startswith("rtfs: plan "):
            continue
        kv = dict(x.split("=") for x in line[len("rtfs: plan "):].split())
        if after:
            single.append(kv)
            continue
        assert kv["window"] == f"{rows}x{cols}@{r0},{c0}" and "views" not in kv, line
        assert kv["count"] == "0" and kv["flow"] == "0", line
        reached.add((kv["noise"], kv["probe"], kv["staged"], kv["lean"], kv["sstack"], kv["wide"]))
    assert single and all("window" not in kv and "views" not in kv for kv in single)  # rt_render's line is unchanged
    return reached


def test_every_window_kernel_is_launched():
    reached = _plans({}) | _plans({"RTFS_LOCAL_STACK": "1"})
    want = set()
    for noise in "01":
        for probe in "10":
            want |= {(noise, probe, "1", "1", "0", "0"), (noise, probe, "1", "0", "0", "0")}
            want |= {(noise, probe, "0", "0", s, w) for s in "01" for w in "01"}
    assert len(want) == 24
    assert want <= reached, sorted(want - reached)


# ---- 8. Scene.render_window and Scene.render_progressive(window=...) ----------------------------------------------------------
def test_scene_wrappers():
    spec = sample_images.few_spheres(max_w=20, max_h=10, spp=48)
    scene = Scene.make(spec.objects, device=0)
    cam = camera(spec)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    w = (2, 3, 11, 29)
    ticks = []
    total, img = Scene.render_window(ticks.append, lambda _: None, mw, mh, cam, scene, w, seed=4)
    assert total == float(w[2]) and img.RowCount == w[2] and img.ColCount == w[3] and not ticks  # lazy
    _, ref = Scene.render(lambda _: None, lambda _: None, mw, mh, cam, scene, seed=4)
    got = Image.render(img)
    assert got.shape == (w[2], w[3], 3) and np.array_equal(got, crop(Image.render(ref), w)) and len(ticks) == w[2]
    assert scene.last_stats.paths > 0
    for rule in (None, 1.0):
        ticks = []
        got = Scene.render_progressive(ticks.append, lambda _: None, mw, mh, cam, scene, seed=4, target_ms=0.05, converge_tolerance=rule,
                                       converge_min_samples=16, converge_interval=8, window=w)
        want = Scene.render_progressive(lambda _: None, lambda _: None, mw, mh, cam, scene, seed=4, converge_tolerance=rule,
                                        converge_min_samples=16, converge_interval=8)
        assert got.shape == (w[2], w[3], 3) and np.array_equal(got, crop(want, w)), rule
        assert len(ticks) == w[2]


if __name__ == "__main__" and sys.argv[1:] == ["plans"]:
    plans_child()
