"""Many views of one scene in one call (rt_render_views): every view must EQUAL rt_render of its camera and seed — the int32
sums, the RGB8 image and the gamma RGB8 image — and the batch's path, ray, early-out and degenerate counts must equal the sums
of the per-view counts.  Cases: early-out on and off; 1, 2, 3 and 37 views; rows % 4 != 0 (probe tiles straddle two views);
one seed for every view and one seed per view; cameras that differ in viewport and focal length; identical cameras.  Scenes:
a C1 turntable, C2 at full size, C3 (image texture), C4 (planes, depth 100), the 100 k-sphere scene (global-memory kernels)
and a scene one sphere past the staging limit.  Flags: default, NO_SMEM, WIDE_BVH, NO_LEAN.  Two child processes report the
launch plans (RTFS_DEBUG_PLAN, one with RTFS_LOCAL_STACK): all twelve batched kernels must be launched."""
import ctypes as C
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

if __name__ == "__main__":  # the child processes of test_every_batched_kernel_is_launched
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from ray_tracing_fsharp_b200 import abi, native, sample_images  # noqa: E402
from ray_tracing_fsharp_b200.domain import marshal  # noqa: E402
from ray_tracing_fsharp_b200.scene import Image, Scene  # noqa: E402

pytestmark = pytest.mark.gpu

FLAGS = {"default": 0, "no-smem": abi.RT_FLAG_NO_SMEM, "wide-bvh": abi.RT_FLAG_WIDE_BVH, "no-lean": abi.RT_FLAG_NO_LEAN}


@functools.lru_cache(maxsize=None)
def device_scene(name):
    spec = {
        "C1": lambda: sample_images.few_spheres(max_w=40, max_h=21, spp=16),  # 81 x 43: 43 % 4 == 3
        "C2": lambda: sample_images.random_spheres(spp=8),                    # full size, 1201 x 801
        "C3": lambda: sample_images.earth(max_w=48, max_h=25, spp=24),
        "C4": lambda: sample_images.mixed_planes(max_w=48, max_h=27, spp=24),
        "C5": lambda: sample_images.many_spheres(max_w=40, max_h=22, spp=4),
        "stage-n*+1": lambda: _past_staging_limit(),
    }[name]()
    hs, ts, keep = marshal(spec.objects)
    return spec, native.SceneHandle(hs, ts, 0, keepalive=keep)


def _past_staging_limit():
    from test_gpu_kernel_matrix import random_spheres, staging_counts
    spec = random_spheres(staging_counts()[0] + 1)
    spec.max_width_coord, spec.max_height_coord, spec.spp = 30, 17, 20  # 61 x 35
    return spec


def orbit(spec, n, focal=None, aspect=None):
    """n cameras on a circle around the spec's look-at point, through its origin (a turntable)."""
    origin, look = np.asarray(spec.origin, float), np.asarray(spec.look_at, float)
    rel = origin - look
    cams = []
    for v in range(n):
        a = 2.0 * np.pi * v / max(n, 1)
        ca, sa = np.cos(a), np.sin(a)
        o = look + np.array([ca * rel[0] + sa * rel[2], rel[1], -sa * rel[0] + ca * rel[2]])
        d = look - o
        cam = native.camera_make_basic(spec.spp, focal if focal is not None else spec.focal_length,
                                       aspect if aspect is not None else spec.aspect_ratio, o, d / np.linalg.norm(d), spec.view_up)
        cam.bounce_depth = spec.bounce_depth
        cams.append(cam)
    return cams


def check_views(dsc, cams, mw, mh, seeds=None, seed=7, adaptive=True, flags=0):
    """The batch against one rt_render per view: sums, RGB8 and gamma RGB8 equal; counts equal the sums of the views'."""
    rgb, sums, st = dsc.render_views(cams, mw, mh, seeds=seeds, seed=seed, adaptive=adaptive, flags=flags, want_sums=True)
    rgb_g, _, _ = dsc.render_views(cams, mw, mh, seeds=seeds, seed=seed, adaptive=adaptive, flags=flags, gamma=True)
    rows, cols = 2 * mh + 1, 2 * mw + 1
    assert rgb.shape == (len(cams), rows, cols, 3) and sums.shape == (len(cams), rows, cols, 4)
    total = dict(paths=0, rays=0, pixels_early_out=0, degenerate_paths=0)
    launches = None
    for v, cam in enumerate(cams):
        s_v = seeds[v] if seeds is not None else seed
        r1, s1, st1 = dsc.render(cam, mw, mh, seed=s_v, adaptive=adaptive, flags=flags, want_sums=True)
        g1, _, _ = dsc.render(cam, mw, mh, seed=s_v, adaptive=adaptive, flags=flags, gamma=True)
        assert np.array_equal(sums[v], s1), f"view {v}: sums differ"
        assert np.array_equal(rgb[v], r1), f"view {v}: RGB8 differs"
        assert np.array_equal(rgb_g[v], g1), f"view {v}: gamma RGB8 differs"
        for k in total:
            total[k] += getattr(st1, k)
        launches = st1.launches
    for k, want in total.items():
        assert getattr(st, k) == want, (k, getattr(st, k), want)
    assert st.launches == launches and st.kernel_ms > 0.0  # one frame sequence for the whole batch
    return rgb, sums, st


@pytest.mark.parametrize("adaptive", [True, False])
@pytest.mark.parametrize("n", [1, 2, 3, 37])
def test_c1_turntable(n, adaptive):
    spec, dsc = device_scene("C1")
    cams = orbit(spec, n)
    check_views(dsc, cams, spec.max_width_coord, spec.max_height_coord, seed=11, adaptive=adaptive)
    check_views(dsc, cams, spec.max_width_coord, spec.max_height_coord, seeds=[100 + 7 * v + (v << 40) for v in range(n)], adaptive=adaptive)


@pytest.mark.parametrize("mw,mh", [(14, 4), (11, 5), (7, 5), (9, 6)])
def test_row_counts_across_tile_boundaries(mw, mh):
    """9, 11, 11 and 13 rows (rows are odd, so never a multiple of the 4-high tile): probe tiles straddle views lane by lane."""
    spec, dsc = device_scene("C1")
    check_views(dsc, orbit(spec, 5), mw, mh, seeds=[3, 1 << 33, 5, 0, 2 ** 64 - 1])


def test_cameras_differ_in_viewport_and_focal_length():
    spec, dsc = device_scene("C1")
    cams = orbit(spec, 2) + orbit(spec, 1, focal=0.6, aspect=1.0) + orbit(spec, 2, focal=2.5, aspect=3.0)
    assert len({(c.viewport_width, c.viewport_height, c.focal_length) for c in cams}) == 3
    check_views(dsc, cams, spec.max_width_coord, spec.max_height_coord, seeds=[1, 2, 3, 4, 5])


def test_identical_cameras_give_identical_views():
    spec, dsc = device_scene("C1")
    cams = orbit(spec, 1) * 4
    rgb, sums, _ = check_views(dsc, cams, spec.max_width_coord, spec.max_height_coord, seed=23)
    for v in range(1, 4):
        assert np.array_equal(rgb[v], rgb[0]) and np.array_equal(sums[v], sums[0])


@pytest.mark.parametrize("name,n", [("C2", 2), ("C3", 3), ("C4", 3), ("C5", 3), ("stage-n*+1", 3)])
def test_scene_families(name, n):
    spec, dsc = device_scene(name)
    cams = orbit(spec, n)
    check_views(dsc, cams, spec.max_width_coord, spec.max_height_coord, seeds=[41 + v for v in range(n)])


@pytest.mark.parametrize("flag", sorted(FLAGS))
@pytest.mark.parametrize("name", ["C1", "C3", "stage-n*+1"])
def test_flags(name, flag):
    spec, dsc = device_scene(name)
    cams = orbit(spec, 3)
    for adaptive in (True, False):
        check_views(dsc, cams, spec.max_width_coord, spec.max_height_coord, seeds=[5, 6, 7], adaptive=adaptive, flags=FLAGS[flag])


def test_noise_flag_is_ignored():
    spec, dsc = device_scene("C1")
    cams = orbit(spec, 3)
    a = dsc.render_views(cams, spec.max_width_coord, spec.max_height_coord, seed=9, want_sums=True)
    b = dsc.render_views(cams, spec.max_width_coord, spec.max_height_coord, seed=9, want_sums=True, flags=abi.RT_FLAG_NOISE)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def _raw(dsc, cams, n, mw, mh, opts, rgb):
    arr = (abi.RtCamera * max(1, len(cams)))(*cams) if cams is not None else None
    return native.lib().rt_render_views(dsc.ptr, arr, None, n, mw, mh, C.byref(opts), native.ptr(rgb), None, None)


def test_argument_errors():
    spec, dsc = device_scene("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cams = orbit(spec, 2)
    rgb = np.zeros((2, 2 * mh + 1, 2 * mw + 1, 3), np.uint8)
    opts = abi.RtRenderOpts(1, 1, abi.RT_MODE_MEGAKERNEL, 0, 0)
    assert _raw(dsc, cams, 0, mw, mh, opts, rgb) == abi.RT_ERR_INVALID_ARGUMENT
    assert _raw(dsc, cams, -3, mw, mh, opts, rgb) == abi.RT_ERR_INVALID_ARGUMENT
    assert _raw(dsc, None, 2, mw, mh, opts, rgb) == abi.RT_ERR_INVALID_ARGUMENT
    assert _raw(dsc, cams, 2, mw, mh, opts, None) == abi.RT_ERR_INVALID_ARGUMENT
    for field, value in (("samples_per_pixel", spec.spp + 1), ("bounce_depth", spec.bounce_depth + 1)):
        odd = orbit(spec, 2)
        setattr(odd[1], field, value)
        assert _raw(dsc, odd, 2, mw, mh, opts, rgb) == abi.RT_ERR_INVALID_ARGUMENT, field
    # 2 x 65535 x 32767 pixels >= 2^31 (refused before anything is allocated or written)
    assert _raw(dsc, cams, 2, 32767, 16383, opts, rgb) == abi.RT_ERR_INVALID_ARGUMENT
    for mode, flags in ((abi.RT_MODE_WAVEFRONT, 0), (abi.RT_MODE_MEGAKERNEL, abi.RT_FLAG_FLOW), (abi.RT_MODE_MEGAKERNEL, abi.RT_FLAG_COUNTERS),
                        (abi.RT_MODE_MEGAKERNEL, abi.RT_FLAG_FLOW | abi.RT_FLAG_LOCKSTEP)):
        o = abi.RtRenderOpts(1, 1, mode, 0, flags)
        assert _raw(dsc, cams, 2, mw, mh, o, rgb) == abi.RT_ERR_UNSUPPORTED, (mode, flags)
    with pytest.raises(ValueError):
        dsc.render_views(cams, mw, mh, seeds=[1])
    # the scene still renders after the refusals
    check_views(dsc, cams, mw, mh, seed=2)


def test_interleaved_with_render_and_progressive_frames():
    """rt_render and a progressive frame between two batches; then a larger batch, so the buffers grow."""
    spec, dsc = device_scene("C1")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    cams = orbit(spec, 3)
    first, first_sums, _ = dsc.render_views(cams, mw, mh, seeds=[1, 2, 3], want_sums=True)
    one, one_sums, _ = dsc.render(cams[1], mw, mh, seed=2, want_sums=True)
    assert np.array_equal(one_sums, first_sums[1]) and np.array_equal(one, first[1])
    with dsc.open_frame(cams[2], mw, mh, seed=3) as frame:
        frame.advance(max_samples=2)
        mid = dsc.render_views(cams, mw, mh, seeds=[1, 2, 3], want_sums=True)
        assert np.array_equal(mid[1], first_sums)
        frame.advance()
        rgb, sums = frame.read(want_sums=True)
    assert np.array_equal(sums, first_sums[2]) and np.array_equal(rgb, first[2])
    check_views(dsc, orbit(spec, 9), mw + 13, mh + 6, seeds=list(range(9)))  # larger: the tall buffers grow
    again, again_sums, _ = dsc.render_views(cams, mw, mh, seeds=[1, 2, 3], want_sums=True)
    assert np.array_equal(again_sums, first_sums) and np.array_equal(again, first)


def test_scene_render_views():
    """Scene.render_views: one Image per camera, Scene.render's image with the same seed; rows x views progress ticks."""
    spec = sample_images.few_spheres(max_w=20, max_h=10, spp=8)
    scene = Scene.make(spec.objects, device=0)
    cams = orbit(spec, 3)
    ticks = []
    total, images = Scene.render_views(ticks.append, lambda _: None, spec.max_width_coord, spec.max_height_coord, cams, scene,
                                       seeds=[4, 5, 6])
    assert total == float(spec.rows * 3) and len(images) == 3
    for v, img in enumerate(images):
        _, ref = Scene.render(lambda _: None, lambda _: None, spec.max_width_coord, spec.max_height_coord, cams[v], scene, seed=4 + v)
        assert np.array_equal(Image.render(img), Image.render(ref))
    assert len(ticks) == spec.rows * 3


# ---- launch plans -------------------------------------------------------------------------------------------------------
PLAN_SCENES = {"C1": ["default", "no-lean", "no-smem", "wide-bvh"], "C3": ["default"], "stage-n*+1": ["default", "wide-bvh"]}


def plans_child():
    for name, flags in PLAN_SCENES.items():
        spec, dsc = device_scene(name)
        for flag in flags:
            dsc.render_views(orbit(spec, 2), spec.max_width_coord, spec.max_height_coord, seed=1, flags=FLAGS[flag])
    spec, dsc = device_scene("C1")
    sys.stderr.write("single frame\n")
    dsc.render(orbit(spec, 1)[0], spec.max_width_coord, spec.max_height_coord, seed=1)
    print("plans child: ok")


def _plans(extra_env):
    env = dict(os.environ, RTFS_DEBUG_PLAN="1", **extra_env)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "plans"], env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0 and "plans child: ok" in r.stdout, r.stdout[-4000:] + r.stderr[-4000:]
    batched, single, after = set(), [], False
    for line in r.stderr.splitlines():
        if line == "single frame":
            after = True
        if not line.startswith("rtfs: plan "):
            continue
        kv = dict(x.split("=") for x in line[len("rtfs: plan "):].split())
        if after:
            single.append(kv)
            continue
        assert kv["views"] == "2" and kv["count"] == "0" and kv["flow"] == "0" and kv["noise"] == "0", line
        batched.add((kv["probe"], kv["staged"], kv["lean"], kv["sstack"], kv["wide"]))
    assert single and all("views" not in kv for kv in single)  # rt_render's line is unchanged
    return batched


def test_every_batched_kernel_is_launched():
    reached = _plans({}) | _plans({"RTFS_LOCAL_STACK": "1"})
    want = set()
    for probe in "10":
        want |= {(probe, "1", "1", "0", "0"), (probe, "1", "0", "0", "0")}
        want |= {(probe, "0", "0", s, w) for s in "01" for w in "01"}
    assert len(want) == 12
    assert want <= reached, sorted(want - reached)


if __name__ == "__main__" and sys.argv[1:] == ["plans"]:
    plans_child()
