"""Saving a progressive frame and resuming it (rt_frame_save, rt_frame_resume, rt_multi_frame_resume, Frame.save,
SceneHandle / MultiHandle.resume_frame, Scene.resume_progressive).  Every case opens two identical frames, advances both
with the same max_samples sequence, saves one, destroys it and resumes the snapshot, then advances the resumed frame and the
uninterrupted twin with the same max_samples sequence, comparing after every pass with np.array_equal or field for field:
sums, RGB8 with and without gamma, Q, the E map, the noise summary, view_noise, every field of RtFrameProgress and
RtFrameConvergence but the _ms fields (and passes, which continue from the snapshot), features and the denoised image.
Device counts at save and at resume: 1 -> 1, 1 -> 2, 2 -> 1, 3 -> 2 and 1 -> max(4, visible devices), ranks sharing devices
where fewer GPUs are visible (RTFS_MULTI_SHARE_DEVICES), as in test_gpu_multi_progressive.py."""
import ctypes as C

import numpy as np
import pytest

import snapshot_rule as rule
from ray_tracing_fsharp_b200 import abi, native, sample_images
from ray_tracing_fsharp_b200.domain import marshal
from ray_tracing_fsharp_b200.scene import Camera, Scene

from test_gpu_multi_progressive import NOISE, assert_same, camera, devices, extents, multi, shared, single, spec_of

pytestmark = pytest.mark.gpu

ONE = "one"  # a SceneHandle: the frame of rt_frame_begin*; any other world is an RtMulti of that many ranks


def owner(name, world):
    return single(name) if world == ONE else multi(name, devices(world))


def opener(name, spp=None, seed=7, adaptive=True, flags=0):
    cam, (mw, mh) = camera(name, spp), extents(name)
    return lambda o: o.open_frame(cam, mw, mh, seed=seed, adaptive=adaptive, flags=flags)


def views_opener(name, n=3, seeds=(11, 12, 13), flags=NOISE, spp=None):
    spec = spec_of(name)
    mw, mh = extents(name)
    cams = []
    for v in range(n):
        origin = tuple(spec.origin[a] + 0.3 * v * (a == 0) for a in range(3))
        cam = native.camera_make_basic(spp or spec.spp, spec.focal_length, spec.aspect_ratio, origin, spec.view_direction, spec.view_up)
        cam.bounce_depth = spec.bounce_depth
        cams.append(cam)
    return lambda o: o.open_frame_views(cams, mw, mh, seeds=None if seeds is None else list(seeds)[:n], seed=5, flags=flags)


def resume_case(name, open_fn, save_world, resume_world, before, after, rule_=None, tol=1.0):
    """The twin and the resumed frame, compared after every pass of `after` (max_samples per call) and at the end."""
    src, twin = open_fn(owner(name, save_world)), open_fn(owner(name, save_world))
    with twin:
        with src:
            if rule_ is not None:
                src.set_convergence(*rule_)
                twin.set_convergence(*rule_)
            for k in before:
                src.advance(k)
                twin.advance(k)
            data = src.save()
            assert src.save() == data  # two saves without a pass between them
            assert_same(twin, src, tol)  # saving changed nothing
        with owner(name, resume_world).resume_frame(data) as r:
            assert r.progress.passes == twin.progress.passes
            assert_same(twin, r, tol)
            if resume_world == save_world:
                assert r.save() == data  # save -> resume -> save: the same bytes
            for k in after:
                r.advance(k)
                twin.advance(k)
                assert_same(twin, r, tol)
            return data, r.progress


WORLDS = [(ONE, ONE), (ONE, 2), (2, ONE), (3, 2), (ONE, "all")]


@pytest.mark.parametrize("save_world,resume_world", WORLDS)
@pytest.mark.parametrize("flags", [0, NOISE])
def test_device_counts(save_world, resume_world, flags):
    resume_case("C1", opener("C1", spp=64, flags=flags), save_world, resume_world, [7, 5], [7] * 4 + [0])


@pytest.mark.parametrize("name", ["C1", "C1-odd", "C2", "C4", "C5", "stage-n*+1"])
def test_scene_families(name):
    resume_case(name, opener(name, flags=NOISE), ONE, 2, [3], [5, 0])


@pytest.mark.parametrize("before", [[], [9], [0]], ids=["after-opener", "mid-frame", "done"])
def test_save_points(before):
    data, progress = resume_case("C1", opener("C1", spp=64, flags=NOISE), ONE, ONE, before, [9, 0])
    assert progress.done


def test_after_extend_and_extend_after_resume():
    o = owner("C1", ONE)
    twin = opener("C1", spp=256, flags=NOISE)(o)
    with opener("C1", spp=256, flags=NOISE)(o) as src:
        for f in (src, twin):
            f.advance(0)
            f.extend(512)
            f.advance(40)
        data = src.save()
    with twin, owner("C1", 2).resume_frame(data) as r:
        assert_same(twin, r)
        for k in (100, 0):
            r.advance(k)
            twin.advance(k)
            assert_same(twin, r)
        # done, then extended again
        for f in (r, twin):
            f.extend(600)
            f.advance(0)
        assert_same(twin, r)


def test_done_frame_extended_after_resume():
    o = owner("C1", ONE)
    twin = opener("C1", spp=32, flags=NOISE)(o)
    with opener("C1", spp=32, flags=NOISE)(o) as src:
        src.advance(0)
        twin.advance(0)
        data = src.save()
    with twin, owner("C1", "all").resume_frame(data) as r:
        assert r.progress.done
        for f in (r, twin):
            f.extend(96)
        for k in (17, 0):
            r.advance(k)
            twin.advance(k)
            assert_same(twin, r)


@pytest.mark.parametrize("tau,m,k", [(0.5, 64, 64), (1.0, 64, 64), (1.0, 37, 23)])
@pytest.mark.parametrize("save_world,resume_world", [(ONE, ONE), (ONE, 2), (3, 2)])
def test_convergence_checkpoints(tau, m, k, save_world, resume_world):
    # max_samples 0 runs to the next checkpoint: the save lands on a checkpoint, right after its check
    resume_case("C1", opener("C1", spp=256, flags=NOISE), save_world, resume_world, [0], [0] * 8, rule_=(tau, m, k), tol=tau)


def test_set_convergence_accepted_exactly_when_the_saved_frame_would_accept_it():
    o = owner("C1", ONE)
    with opener("C1", spp=128, flags=NOISE)(o) as f:
        fresh = f.save()
        f.advance(5)
        later = f.save()
    with o.resume_frame(fresh) as r:
        r.set_convergence(1.0, 64, 64)
    with o.resume_frame(later) as r:
        with pytest.raises(native.RtError) as e:
            r.set_convergence(1.0, 64, 64)
        assert e.value.code == abi.RT_ERR_INVALID_ARGUMENT


@pytest.mark.parametrize("mode", ["no-early-out", "no-smem", "wide-bvh", "no-lean", "flow", "counters"])
def test_modes(mode):
    adaptive = mode != "no-early-out"
    flags = {"no-early-out": NOISE, "no-smem": NOISE | abi.RT_FLAG_NO_SMEM, "wide-bvh": NOISE | abi.RT_FLAG_WIDE_BVH,
             "no-lean": NOISE | abi.RT_FLAG_NO_LEAN, "flow": abi.RT_FLAG_FLOW, "counters": abi.RT_FLAG_COUNTERS}[mode]
    resume_case("C1", opener("C1", spp=48, adaptive=adaptive, flags=flags), ONE, 2, [6], [6, 0])


@pytest.mark.parametrize("seeds", [(11, 12, 13), None], ids=["seeds", "no-seeds"])
@pytest.mark.parametrize("save_world,resume_world", [(ONE, ONE), (ONE, 2), (2, ONE)])
def test_views(seeds, save_world, resume_world):
    resume_case("C1-odd", views_opener("C1-odd", seeds=seeds), save_world, resume_world, [5], [5, 0])


def test_window():
    name = "C1"
    cam, (mw, mh) = camera(name, 64), extents(name)
    open_fn = lambda o: o.open_frame_window(cam, mw, mh, (3, 5, 17, 29), seed=7, flags=NOISE)  # noqa: E731
    data, _ = resume_case(name, open_fn, ONE, ONE, [6], [6, 0])
    assert rule.parse(data)["header"].kind == abi.RT_FRAME_WINDOW
    with pytest.raises(native.RtError) as e:
        owner(name, 2).resume_frame(data)
    assert e.value.code == abi.RT_ERR_UNSUPPORTED


@pytest.mark.parametrize("save_world,resume_world", [(ONE, 2), (2, ONE)])
def test_features_and_denoise_after_resume(save_world, resume_world):
    o = owner("C1", save_world)
    with opener("C1", spp=64, flags=NOISE)(o) as src, opener("C1", spp=64, flags=NOISE)(o) as twin:
        for f in (src, twin):
            f.advance(12)
        data = src.save()
        with owner("C1", resume_world).resume_frame(data) as r:
            for x, y in zip(twin.features(4), r.features(4)):
                assert np.array_equal(x, y)
            for x, y in zip(twin.denoise(want_linear=True), r.denoise(want_linear=True)):
                assert np.array_equal(x, y)


def test_snapshot_matches_the_rule_and_the_frame():
    o = owner("C1", ONE)
    with opener("C1", spp=64, flags=NOISE)(o) as f:
        f.advance(9)
        data = f.save()
        parts = rule.parse(data)
        _, sums = f.read(want_sums=True)
        _, _, sq = f.noise(1.0, want_map=False, want_sq=True)
        p = f.progress
    h = parts["header"]
    assert h.checksum == rule.checksum(data) and rule.write(parts) == data
    assert np.array_equal(parts["sums"], sums.reshape(-1, 4)) and np.array_equal(parts["sq"], sq.reshape(-1))
    assert (h.samples_done, h.paths_done, h.pixels_flagged) == (p.samples_done, p.paths_done, p.pixels_flagged)
    assert int(parts["active"].sum()) == h.pixels_active and int(sums[..., 3].sum()) == h.paths_done


def _resume_refused(o, data, code=abi.RT_ERR_INVALID_ARGUMENT, fn=None):
    out = C.c_void_p(12345)
    lib = native.lib()
    fn = fn or (lib.rt_frame_resume if isinstance(o, native.SceneHandle) else lib.rt_multi_frame_resume)
    assert fn(o.ptr, data, len(data), C.byref(out), None) == code, lib.rt_last_error()
    assert out.value is None
    return lib.rt_last_error().decode()


def test_refusals_leave_out_null_and_the_scene_usable():
    o = owner("C1", ONE)
    with opener("C1", spp=64, flags=NOISE)(o) as f:
        f.advance(9)
        data = f.save()
        n = C.c_size_t()
        assert native.lib().rt_frame_save(f.ptr, None, 0, C.byref(n)) == abi.RT_OK and n.value == len(data)
        small = np.empty(len(data) - 1, np.uint8)
        assert native.lib().rt_frame_save(f.ptr, native.ptr(small), small.size, C.byref(n)) == abi.RT_ERR_INVALID_ARGUMENT
        assert n.value == len(data)
    _, at, _ = rule.sections(rule.parse(data)["header"])
    npx = rule.parse(data)["header"].n_pixels
    assert _resume_refused(o, data[:-8])
    assert _resume_refused(o, data[:100])
    for byte in (0, 8, 60, 300, at + 5, at + 16 * npx + 3, len(data) - 2):  # magic, version, camera, header tail, sums, Q, flags
        bad = bytearray(data)
        bad[byte] ^= 0x10
        assert _resume_refused(o, bytes(bad))
    parts = rule.parse(data)
    parts["header"].magic = b"RTFSSNAQ"
    assert "magic" in _resume_refused(o, rule.write(parts))
    parts = rule.parse(data)
    parts["header"].version = 2
    assert "version" in _resume_refused(o, rule.write(parts))
    # one inconsistent pixel under a correct checksum: refused and named
    parts = rule.parse(data)
    p = int(np.flatnonzero(parts["active"])[3])
    parts["sums"][p, 3] -= 1
    assert f"pixel {p}" in _resume_refused(o, rule.write(parts))
    parts = rule.parse(data)
    parts["sums"][p, 0] = 255 * parts["sums"][p, 3] + 1
    assert f"pixel {p}" in _resume_refused(o, rule.write(parts))
    parts = rule.parse(data)
    parts["header"].paths_done += 1
    assert "paths_done" in _resume_refused(o, rule.write(parts))
    # the scene is still usable, and the good snapshot still resumes
    with o.resume_frame(data) as r:
        r.advance(0)


def test_scene_content_must_match_and_an_edit_back_is_accepted():
    spec = sample_images.earth(max_w=30, max_h=17, spp=24, bitmap=sample_images.synthetic_earthmap(64, 32))
    hs, ts, keep = marshal(spec.objects)
    h = native.SceneHandle(hs, ts, 0, keepalive=keep)
    cam = native.camera_make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    cam.bounce_depth = spec.bounce_depth
    with h.open_frame(cam, spec.max_width_coord, spec.max_height_coord, seed=3, flags=NOISE) as f:
        f.advance(5)
        data = f.save()
        # a stale frame's save is refused
        sphere = [i for i in range(len(hs)) if hs[i].shape == abi.RT_SHAPE_SPHERE][0]
        moved = abi.RtHittable.from_buffer_copy(bytes(hs[sphere]))
        moved.p[0] += 0.25
        h.update([sphere], [moved])
        n = C.c_size_t()
        assert native.lib().rt_frame_save(f.ptr, None, 0, C.byref(n)) == abi.RT_ERR_INVALID_ARGUMENT
    assert "differ" in _resume_refused(h, data)
    h.update([sphere], [hs[sphere]])  # back to the saved arrays
    with h.resume_frame(data) as r:
        r.advance(0)
    img = [t for t in range(len(ts)) if ts[t].kind == abi.RT_TEX_IMAGE][0]
    old = np.ctypeslib.as_array(ts[img].rgb8, shape=(ts[img].height, ts[img].width, 3))
    texels = np.ascontiguousarray(old.copy())
    texels[0, 0, 0] ^= 1
    tex = abi.RtTexture.from_buffer_copy(bytes(ts[img]))
    tex.rgb8 = texels.ctypes.data_as(C.POINTER(C.c_uint8))
    h.update([], [], [img], [tex])
    assert "differ" in _resume_refused(h, data)
    h.update([], [], [img], [ts[img]])
    with h.resume_frame(data) as r:
        r.advance(0)
    # a scene created anew from the same arrays takes the snapshot too
    with native.SceneHandle(hs, ts, 0, keepalive=keep).resume_frame(data) as r:
        r.advance(0)


def test_interleaving_and_frames_side_by_side():
    o = owner("C1", ONE)
    cam, (mw, mh) = camera("C1", 64), extents("C1")
    with opener("C1", spp=64, flags=NOISE)(o) as src, opener("C1", spp=64, flags=NOISE)(o) as twin:
        for f in (src, twin):
            f.advance(8)
        data = src.save()
        o.render(cam, mw, mh, seed=99)  # other work on the scene between save and resume
        with opener("C1", spp=64)(o) as other:
            other.advance(0)
            with o.resume_frame(data) as r:  # the original frame is still alive beside it
                for k in (8, 0):
                    for f in (src, twin, r):
                        f.advance(k)
                    assert_same(twin, r)
                    assert_same(twin, src)


@pytest.mark.parametrize("devs", [None, "all"])
def test_scene_resume_progressive(devs):
    spec = spec_of("C1")
    cam = Camera.make_basic(64, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    cam.bounce_depth = spec.bounce_depth
    devs = None if devs is None else devices(devs)
    with shared(devs or ()):
        s = Scene.make(spec.objects, devices=None if devs is None else list(devs))
    ticks = []
    want = Scene.render_progressive(lambda x: ticks.append(x), lambda _: None, spec.max_width_coord, spec.max_height_coord, cam, s, seed=4,
                                    target_ms=1.0)
    saved = []

    def stop_after_two(progress, frame):
        saved.append(frame.save())
        return len(saved) == 2

    first = []
    Scene.render_progressive(lambda x: first.append(x), lambda _: None, spec.max_width_coord, spec.max_height_coord, cam, s, seed=4,
                             target_ms=1.0, on_pass=stop_after_two)
    rest = []
    got = Scene.resume_progressive(lambda x: rest.append(x), lambda _: None, saved[-1], s, target_ms=1.0)
    assert np.array_equal(want, got)
    assert len(ticks) == len(rest) == 2 * spec.max_height_coord + 1
