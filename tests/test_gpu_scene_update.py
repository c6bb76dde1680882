"""In-place scene edits (rt_scene_update, SceneHandle.update, Scene.update).  After an edit a scene must render EXACTLY as a scene
created from the edited arrays: every comparison is np.array_equal against rt_scene_create of those arrays, over rt_render
(flags 0, NO_SMEM, NO_LEAN, WIDE_BVH; sums, RGB8, paths and rays), rt_render_views, rt_render_window, a progressive frame with
noise and a convergence rule opened after the edit, and rt_frame_features.
Scenes: C1-C5 and one sphere past the staging limit with moved spheres and recoloured objects; C3 with its image-textured sphere
moved together with its map centre and its texels replaced; C4 with planes and unbounded spheres edited, one of them flipped
between the FP32 and FP64 classes.  Also: the lean plan follows a texture index on and off; the tree after edits passes
rt_scene_device_bvh_check, equals tests/refit_rule.py, and comes back byte for byte when the edit is undone; the refit touches
at most depth nodes for one sphere and none for a material edit; a 50-step C2 animation; stale frames; every refusal, each
leaving the scene as it was; rendering and frames between edits; and the Python wrappers."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from ray_tracing_fsharp_b200 import abi, native, sample_images
from ray_tracing_fsharp_b200.domain import Hittable, Sphere, marshal
from ray_tracing_fsharp_b200.scene import Scene

import refit_rule
from test_gpu_views import _past_staging_limit, orbit

pytestmark = pytest.mark.gpu

NOISE = abi.RT_FLAG_NOISE
SPECS = {
    "C1": lambda: sample_images.few_spheres(max_w=40, max_h=21, spp=16),
    "C2": lambda: sample_images.random_spheres(spp=8),
    "C3": lambda: sample_images.earth(max_w=48, max_h=25, spp=24),
    "C4": lambda: sample_images.mixed_planes(max_w=48, max_h=27, spp=24),
    "C5": lambda: sample_images.many_spheres(max_w=40, max_h=22, spp=4),
    "stage-n*+1": lambda: _past_staging_limit(),
}


def copy(arr, ctype):
    """A ctypes array holding copies of the records of `arr` (a ctypes array or a list of records)."""
    out = (ctype * max(1, len(arr)))()
    if isinstance(arr, C.Array):
        C.memmove(out, arr, C.sizeof(ctype) * len(arr))
    else:
        for i, rec in enumerate(arr):
            out[i] = rec
    return out


def create(hs, ts):
    return native.SceneHandle(hs, ts, 0)


def camera(spec):
    return orbit(spec, 1)[0]


def assert_same_frames(edited, fresh, spec, seed=11, full=True):
    """Every entry point of `edited` against `fresh`, bit for bit."""
    cam, mw, mh = camera(spec), spec.max_width_coord, spec.max_height_coord
    for flags in (0, abi.RT_FLAG_NO_SMEM, abi.RT_FLAG_NO_LEAN, abi.RT_FLAG_WIDE_BVH):
        a, sa, st_a = edited.render(cam, mw, mh, seed=seed, flags=flags, want_sums=True)
        b, sb, st_b = fresh.render(cam, mw, mh, seed=seed, flags=flags, want_sums=True)
        assert np.array_equal(sa, sb), f"flags {flags}: sums differ"
        assert np.array_equal(a, b), f"flags {flags}: RGB8 differs"
        assert (st_a.paths, st_a.rays) == (st_b.paths, st_b.rays), flags
    if not full:
        return
    cams = orbit(spec, 2)
    va, vsa, _ = edited.render_views(cams, mw, mh, seeds=[3, 4], want_sums=True)
    vb, vsb, _ = fresh.render_views(cams, mw, mh, seeds=[3, 4], want_sums=True)
    assert np.array_equal(vsa, vsb) and np.array_equal(va, vb), "views differ"
    rows, cols = 2 * mh + 1, 2 * mw + 1
    win = (rows // 4, cols // 3, rows // 2, cols // 2)
    wa, wsa, _ = edited.render_window(cam, mw, mh, win, seed=seed, want_sums=True)
    wb, wsb, _ = fresh.render_window(cam, mw, mh, win, seed=seed, want_sums=True)
    assert np.array_equal(wsa, wsb) and np.array_equal(wa, wb), "windows differ"
    fa, fb = edited.open_frame(cam, mw, mh, seed=seed, flags=NOISE), fresh.open_frame(cam, mw, mh, seed=seed, flags=NOISE)
    with fa, fb:
        if cam.samples_per_pixel > 12:
            fa.set_convergence(2.0, 12, 4)
            fb.set_convergence(2.0, 12, 4)
        while not fa.progress.done:
            pa, pb = fa.advance(max_samples=5), fb.advance(max_samples=5)
            assert (pa.samples_done, pa.paths_done) == (pb.samples_done, pb.paths_done)
            ra, sa = fa.read(want_sums=True)
            rb, sb = fb.read(want_sums=True)
            assert np.array_equal(sa, sb) and np.array_equal(ra, rb), "progressive frames differ"
            assert np.array_equal(fa.noise(1.0, want_sq=True)[2], fb.noise(1.0, want_sq=True)[2])
        for x, y in zip(fa.features(4), fb.features(4)):
            assert np.array_equal(x, y), "features differ"


def bounded(hs):
    return [i for i in range(len(hs)) if hs[i].shape == abi.RT_SHAPE_SPHERE and hs[i].radius >= 0]


def move_and_recolour(hs, rng, n_move, n_colour):
    """A copy of hs with n_move bounded spheres moved and resized and n_colour objects recoloured; and the indices edited."""
    out = copy(hs, abi.RtHittable)
    b = bounded(hs)
    moved = rng.choice(b, size=min(n_move, len(b)), replace=False).tolist()
    for i in moved:
        o = out[i]
        for a in range(3):
            o.p[a] += rng.normal(0, 0.3 * o.radius + 0.01)
        o.radius *= rng.uniform(0.8, 1.2)
    coloured = rng.choice(len(hs), size=min(n_colour, len(hs)), replace=False).tolist()
    for i in coloured:
        o = out[i]
        o.colour[0], o.colour[1] = int(rng.integers(0, 256)), int(rng.integers(0, 256))
        o.albedo = float(rng.uniform(0.2, 1.0))
    return out, sorted(set(moved) | set(coloured))


# ---- 1. the scene families ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(SPECS))
def test_moved_and_recoloured_scenes_render_as_created(name):
    spec = SPECS[name]()
    hs, ts, keep = marshal(spec.objects)
    h = create(hs, ts)
    rng = np.random.default_rng(1)
    n_move = 1000 if name == "C5" else 7
    edited, idx = move_and_recolour(hs, rng, n_move, 5)
    info = h.update(idx, [edited[i] for i in idx])
    assert info.generation == 1 and info.spheres_moved > 0 and info.nodes_refit > 0 and info.device_ms > 0
    fresh = create(edited, ts)
    assert_same_frames(h, fresh, spec, full=name != "C5")
    h.device_bvh_check()
    bounds, right, prim = h.bvh_nodes()
    assert np.array_equal(refit_rule.refit(right, prim, edited).astype(np.float64), bounds)
    h.wide_bvh_check()
    # a second edit on top of the first
    edited2, idx2 = move_and_recolour(edited, rng, n_move, 3)
    info2 = h.update(idx2, [edited2[i] for i in idx2])
    assert info2.generation == 2
    assert_same_frames(h, create(edited2, ts), spec, full=False)
    h.device_bvh_check()


def test_textured_sphere_moved_with_its_map_and_texels_replaced():
    spec = SPECS["C3"]()
    hs, ts, keep = marshal(spec.objects)
    h = create(hs, ts)
    img = [t for t in range(len(ts)) if ts[t].kind == abi.RT_TEX_IMAGE][0]
    users = [i for i in range(len(hs)) if hs[i].texture == img]
    assert users
    edited = copy(hs, abi.RtHittable)
    tex = copy(ts, abi.RtTexture)
    delta = (0.15, -0.05, 0.1)
    for i in users:
        for a in range(3):
            edited[i].p[a] += delta[a]
    for a in range(3):
        tex[img].map_centre[a] += delta[a]
    old = np.ctypeslib.as_array(ts[img].rgb8, shape=(ts[img].height, ts[img].width, 3))
    texels = np.ascontiguousarray(255 - old[:, ::-1])
    tex[img].rgb8 = texels.ctypes.data_as(C.POINTER(C.c_uint8))
    info = h.update(users, [edited[i] for i in users], [img], [tex[img]])
    assert info.textures == 1 and info.spheres_moved == len([i for i in users if i in bounded(hs)])
    assert_same_frames(h, create(edited, list(tex)[:len(ts)]), spec)


def test_planes_and_unbounded_spheres_edited_across_the_fp32_fp64_classes():
    spec = SPECS["C4"]()
    hs, ts, keep = marshal(spec.objects)
    h = create(hs, ts)
    edited = copy(hs, abi.RtHittable)
    planes = [i for i in range(len(hs)) if hs[i].shape == abi.RT_SHAPE_INFINITE_PLANE]
    unb = [i for i in range(len(hs)) if hs[i].shape == abi.RT_SHAPE_UNBOUNDED_SPHERE]
    assert planes and unb
    p = edited[planes[0]]
    n = np.array(list(p.n)) + np.array([0.03, 0.0, -0.02])
    n /= np.linalg.norm(n)
    p.n[:] = n.tolist()
    p.p[1] += 0.25
    u = edited[unb[0]]
    u.p[0] += 1e-9  # no longer exact in FP32: the FP64 class (or still it, moved)
    u.colour[2] = 17
    idx = [planes[0], unb[0]]
    info = h.update(idx, [edited[i] for i in idx])
    assert info.spheres_moved == 0 and info.nodes_refit == 0
    assert_same_frames(h, create(edited, ts), spec)
    # and back: an unbounded object returns to the FP32 class
    info = h.update(idx, [hs[i] for i in idx])
    assert_same_frames(h, create(hs, ts), spec, full=False)


# ---- 2. lean ----------------------------------------------------------------------------------------------------------------------
LEAN_CHILD = r'''
import sys
sys.path.insert(0, sys.argv[1])
from ray_tracing_fsharp_b200 import abi, native, sample_images
from ray_tracing_fsharp_b200.domain import marshal
spec = sample_images.few_spheres(max_w=20, max_h=10, spp=4)
hs, _, _ = marshal(spec.objects)
tex = (abi.RtTexture * 1)()
tex[0].kind = abi.RT_TEX_COLOUR
tex[0].colour[:] = [10, 200, 30]
h = native.SceneHandle(hs, tex, 0)
cam = native.camera_make_basic(4, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
def mark(s):
    sys.stderr.write(s + "\n"); sys.stderr.flush()
mark("BEFORE"); h.render(cam, 20, 10)
i = [k for k in range(len(hs)) if hs[k].shape == abi.RT_SHAPE_SPHERE][0]
e = (abi.RtHittable * 1)(hs[i]); e[0].texture = 0
h.update([i], [e[0]]); mark("TEXTURED"); h.render(cam, 20, 10)
h.update([i], [hs[i]]); mark("REVERTED"); h.render(cam, 20, 10)
'''


def test_lean_follows_a_texture_index():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RTFS_DEBUG_PLAN="1")
    res = subprocess.run([sys.executable, "-c", LEAN_CHILD, root], env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    section, lean = None, {}
    for line in res.stderr.splitlines():
        if line in ("BEFORE", "TEXTURED", "REVERTED"):
            section = line
        elif "rtfs: plan" in line and section:
            lean.setdefault(section, set()).add(" lean=1" in line)
    assert lean == {"BEFORE": {True}, "TEXTURED": {False}, "REVERTED": {True}}, (lean, res.stderr[-2000:])


# ---- 3. the tree ------------------------------------------------------------------------------------------------------------------
def test_tree_comes_back_byte_for_byte_and_refits_no_more_than_needed():
    spec = SPECS["C2"]()
    hs, ts, keep = marshal(spec.objects)
    h = create(hs, ts)
    before = h.bvh_nodes()
    depth = h.device_bvh_check()["depth"]
    rng = np.random.default_rng(3)
    edited, idx = move_and_recolour(hs, rng, 40, 10)
    h.update(idx, [edited[i] for i in idx])
    h.device_bvh_check()
    assert not np.array_equal(h.bvh_nodes()[0], before[0])
    h.update(idx, [hs[i] for i in idx])
    after = h.bvh_nodes()
    assert all(np.array_equal(a, b) for a, b in zip(before, after))
    h.device_bvh_check()
    assert_same_frames(h, create(hs, ts), spec, full=False)
    # one sphere: only its ancestors
    i = bounded(hs)[5]
    one = copy(hs, abi.RtHittable)
    one[i].p[1] += 0.01
    info = h.update([i], [one[i]])
    assert info.spheres_moved == 1 and 1 <= info.nodes_refit <= depth, (info.nodes_refit, depth)
    # a material only: no refit
    mat = copy(one, abi.RtHittable)
    mat[i].albedo = 0.123
    info = h.update([i], [mat[i]])
    assert info.objects == 1 and info.spheres_moved == 0 and info.nodes_refit == 0 and info.launches == 1
    assert_same_frames(h, create(mat, ts), spec, full=False)


def test_one_sphere_tree():
    spec = sample_images.few_spheres(max_w=20, max_h=10, spp=8)
    hs, ts, keep = marshal(spec.objects)
    keep_idx = [i for i in range(len(hs)) if hs[i].shape != abi.RT_SHAPE_SPHERE][:2] + bounded(hs)[:1]
    one = (abi.RtHittable * len(keep_idx))(*[hs[i] for i in keep_idx])
    h = create(one, ts)
    edited = copy(one, abi.RtHittable)
    k = len(keep_idx) - 1
    edited[k].p[0] += 0.2
    edited[k].radius *= 1.3
    info = h.update([k], [edited[k]])
    assert info.spheres_moved == 1 and info.nodes_refit == 1
    assert_same_frames(h, create(edited, ts), spec)
    h.device_bvh_check()


# ---- 4. animation -----------------------------------------------------------------------------------------------------------------
def bob(objects, step, steps=120):
    """C2's small spheres bob on a sine: step `step` of `steps`."""
    out = []
    for k, o in enumerate(objects):
        if isinstance(o, Hittable.Sphere) and o.sphere.Radius == 0.2:
            c = o.sphere.Centre
            y = c[1] + 0.15 * np.sin(2.0 * np.pi * step / steps + 0.7 * k)
            o = Hittable.Sphere(Sphere.make(o.sphere.Style, (c[0], y, c[2]), o.sphere.Radius))
        out.append(o)
    return out


def test_animation_matches_recreated_scenes():
    spec = sample_images.random_spheres(max_w=150, max_h=100, spp=8)
    s = Scene.make(spec.objects, device=0)
    cam = camera(spec)
    for step in range(1, 51):
        objs = bob(spec.objects, step)
        info = Scene.update(s, objs)
        assert info.spheres_moved > 0
        if step % 10 == 0:
            a, sa, _ = s.handle.render(cam, spec.max_width_coord, spec.max_height_coord, seed=step, want_sums=True)
            fresh = Scene.make(objs, device=0)
            b, sb, _ = fresh.handle.render(cam, spec.max_width_coord, spec.max_height_coord, seed=step, want_sums=True)
            assert np.array_equal(sa, sb) and np.array_equal(a, b), step


# ---- 5. stale frames, refusals, interleaving --------------------------------------------------------------------------------------
def test_stale_frames():
    spec = SPECS["C1"]()
    hs, ts, keep = marshal(spec.objects)
    h = create(hs, ts)
    cam = camera(spec)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    f = h.open_frame(cam, mw, mh, seed=2, flags=NOISE)
    f.advance(max_samples=3)
    conv = h.open_frame(cam, mw, mh, seed=2, flags=NOISE)
    conv.set_convergence(1.0, 12, 4)
    before = (f.read(want_sums=True), f.noise(1.0, want_sq=True), f.view_noise(1.0), conv.convergence())
    edited, idx = move_and_recolour(hs, np.random.default_rng(4), 3, 3)
    h.update(idx, [edited[i] for i in idx])
    lib = native.lib()
    opts = abi.RtDenoiseOpts(3, 4, 4.0, 0.1, 16.0, 0.02, 0, 0)
    for rc in (lib.rt_frame_advance(f.ptr, 1, 0.0, None), lib.rt_frame_extend(f.ptr, 32),
               lib.rt_frame_set_convergence(f.ptr, 1.0, 30, 4), lib.rt_frame_features(f.ptr, 4, None, None, None, None),
               lib.rt_frame_denoise(f.ptr, C.byref(opts), None, None), lib.rt_frame_advance(conv.ptr, 0, 0.0, None)):
        assert rc == abi.RT_ERR_INVALID_ARGUMENT
        assert b"scene changed" in lib.rt_last_error()
    after = (f.read(want_sums=True), f.noise(1.0, want_sq=True), f.view_noise(1.0), conv.convergence())
    for x, y in zip(before[0], after[0]):
        assert np.array_equal(x, y)
    s0, s1 = before[1], after[1]
    assert bytes(s0[0]) == bytes(s1[0]) and np.array_equal(s0[1], s1[1]) and np.array_equal(s0[2], s1[2])
    assert bytes(before[2][0]) == bytes(after[2][0]) and bytes(before[3]) == bytes(after[3])
    f.close()
    conv.close()
    # a frame opened after the edit runs
    with h.open_frame(cam, mw, mh, seed=2, flags=NOISE) as g:
        g.advance()
        g.features(4)


def test_refusals_leave_the_scene_as_it_was():
    spec = SPECS["C3"]()
    hs, ts, keep = marshal(spec.objects)
    h = create(hs, ts)
    cam = camera(spec)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    ref = h.render(cam, mw, mh, seed=5, want_sums=True)[1]
    nodes = h.bvh_nodes()
    sph = bounded(hs)[0]
    img = [t for t in range(len(ts)) if ts[t].kind == abi.RT_TEX_IMAGE][0]
    chk = [t for t in range(len(ts)) if ts[t].kind == abi.RT_TEX_CHECKERED]
    lib = native.lib()

    def rec(i, **kw):
        e = copy(hs, abi.RtHittable)[i]
        for k, v in kw.items():
            setattr(e, k, v)
        return e

    def tex(t, **kw):
        e = copy(ts, abi.RtTexture)[t]
        for k, v in kw.items():
            setattr(e, k, v)
        return e

    moved = rec(sph)
    moved.p[0] += 1.0
    cases = [
        ([sph], [rec(sph, shape=abi.RT_SHAPE_UNBOUNDED_SPHERE)], [], []),  # structural: shape
        ([sph], [rec(sph, radius=-hs[sph].radius - 0.1)], [], []),          # structural: tree membership
        ([len(hs)], [hs[0]], [], []),                                       # out of range
        ([-1], [hs[0]], [], []),
        ([sph, 0, sph], [moved, hs[0], moved], [], []),                     # duplicate
        ([sph], [rec(sph, style=99)], [], []),                              # what rt_scene_create refuses
        ([sph], [rec(sph, texture=len(ts))], [], []),
        ([sph], [rec(sph, radius=float("nan"))], [], []),
        ([], [], [img], [tex(img, kind=abi.RT_TEX_COLOUR)]),                # structural: texture kind
        ([], [], [img], [tex(img, width=ts[img].width + 1)]),               # structural: image size
        ([], [], [img], [tex(img, map_radius=0.0)]),
        ([], [], [len(ts)], [ts[0]]),
        ([], [], [img, img], [ts[img], ts[img]]),
    ]
    if chk:
        cases.append(([], [], [chk[0]], [tex(chk[0], even=chk[0])]))
    for oi, objs, ti, texs in cases:
        with pytest.raises(native.RtError) as e:
            h.update(oi, objs, ti, texs)
        assert e.value.code == abi.RT_ERR_INVALID_ARGUMENT, (oi, ti, e.value)
    # raw argument errors
    one = np.zeros(1, np.int32)
    assert lib.rt_scene_update(h.ptr, native.ptr(one), None, 1, None, None, 0, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_scene_update(h.ptr, None, None, -1, None, None, 0, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_scene_update(h.ptr, None, None, 0, None, None, -2, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_scene_update(h.ptr, None, None, 0, native.ptr(one), None, 1, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert np.array_equal(h.render(cam, mw, mh, seed=5, want_sums=True)[1], ref)
    assert all(np.array_equal(a, b) for a, b in zip(nodes, h.bvh_nodes()))
    assert h.update([], []).generation == 0  # an empty call edits nothing


def test_interleaving_renders_frames_and_edits():
    spec = SPECS["C2"]()
    spec.max_width_coord, spec.max_height_coord = 150, 100
    hs, ts, keep = marshal(spec.objects)
    h = create(hs, ts)
    cam = camera(spec)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    rng = np.random.default_rng(8)
    cur = hs
    for k in range(4):
        with h.open_frame(cam, mw, mh, seed=k, flags=NOISE) as f:
            f.advance(max_samples=2)
            h.render(cam, mw, mh, seed=k + 100)
            f.advance()
            got = f.read(want_sums=True)[1]
        fresh = create(cur, ts)
        with fresh.open_frame(cam, mw, mh, seed=k, flags=NOISE) as g:
            g.advance()
            assert np.array_equal(got, g.read(want_sums=True)[1]), k
        cur, idx = move_and_recolour(cur, rng, 20, 5)
        h.update(idx, [cur[i] for i in idx])
        assert np.array_equal(h.render(cam, mw, mh, seed=k, want_sums=True)[1], create(cur, ts).render(cam, mw, mh, seed=k, want_sums=True)[1])


# ---- 6. the Python wrappers --------------------------------------------------------------------------------------------------------
def test_scene_update_sends_only_changed_records():
    spec = sample_images.random_spheres(max_w=60, max_h=40, spp=8)
    s = Scene.make(spec.objects, device=0)
    objs = list(spec.objects)
    o = objs[7]
    objs[7] = Hittable.Sphere(Sphere.make(o.sphere.Style, (o.sphere.Centre[0] + 0.1,) + tuple(o.sphere.Centre[1:]), o.sphere.Radius))
    info = Scene.update(s, objs)
    assert info.objects == 1 and info.spheres_moved == 1 and info.textures == 0
    assert Scene.update(s, objs).objects == 0  # nothing changed: nothing sent
    cam = camera(spec)
    a = s.handle.render(cam, spec.max_width_coord, spec.max_height_coord, seed=1, want_sums=True)[1]
    b = Scene.make(objs, device=0).handle.render(cam, spec.max_width_coord, spec.max_height_coord, seed=1, want_sums=True)[1]
    assert np.array_equal(a, b)
    with pytest.raises(ValueError):
        Scene.update(s, objs[:-1])
    # textures: C3's texture table is diffed too
    spec3 = SPECS["C3"]()
    s3 = Scene.make(spec3.objects, device=0)
    assert Scene.update(s3, list(spec3.objects)).objects == 0


def test_scene_update_refuses_a_scene_over_several_devices():
    if native.device_count() < 2:
        # a scene record around an RtMulti handle, as Scene.make(devices=[0, 1]) makes it (the wrapper decides by the type)
        s = Scene(native.MultiHandle.__new__(native.MultiHandle), [], [], [], [0, 1])
        with pytest.raises(NotImplementedError):
            Scene.update(s, [])
        return
    spec = sample_images.few_spheres(max_w=10, max_h=5, spp=2)
    s = Scene.make(spec.objects, devices=[0, 1])
    with pytest.raises(NotImplementedError):
        Scene.update(s, spec.objects)
