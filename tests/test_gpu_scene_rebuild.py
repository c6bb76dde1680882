"""Structural edits of a live scene (rt_scene_rebuild, SceneHandle.rebuild, Scene.add / remove / rebuild).  After a rebuild a
scene must render EXACTLY as a scene created from the new array: every comparison is np.array_equal against rt_scene_create of
that array, over rt_render (flags 0, NO_SMEM, NO_LEAN, WIDE_BVH), views, a window, a progressive frame with noise and a
convergence rule, and features (the helpers of test_gpu_scene_update).
The device tree equals tests/ploc_rule.py node for node and passes both tree checks; it depends on the array only, not on the
edits that led to it; rays hit the same objects through every traversal; the scene grows past the shared-memory staging limit
and back; C4's planes and unbounded spheres keep their array order; the tree can lose every sphere or keep one; a chain of
nested spheres too deep for the walk stacks falls back to the host tree; rt_scene_update refits the new tree; stale frames,
refusals and interleaving; and the Python wrappers."""
import numpy as np
import pytest

from ray_tracing_fsharp_b200 import abi, native, sample_images
from ray_tracing_fsharp_b200.domain import Hittable, marshal
from ray_tracing_fsharp_b200.scene import Scene

import ploc_rule
from test_gpu_scene_update import SPECS, assert_same_frames, bounded, camera, copy, create, move_and_recolour
from test_gpu_views import _past_staging_limit

pytestmark = pytest.mark.gpu

NOISE = abi.RT_FLAG_NOISE


def edited_array(hs, remove, append):
    """The array rt_scene_rebuild(remove, append) leaves: hs without `remove`, then `append`."""
    gone = set(int(i) for i in remove)
    recs = [hs[i] for i in range(len(hs)) if i not in gone] + list(append)
    return copy(recs, abi.RtHittable) if recs else (abi.RtHittable * 0)(), len(recs)


def fresh_spheres(hs, rng, n):
    """n new bounded spheres with the materials of random existing ones, in a row just above every bounded sphere of `hs` and
    apart from one another: no new sphere meets another sphere, so no closest hit can be an exact tie in t between two bounded
    spheres (the one case in which trees of different topology may pick different hits)."""
    b = bounded(hs)
    c = np.array([list(hs[i].p) for i in b])
    r = np.array([hs[i].radius for i in b])
    small = r <= np.median(r)
    rad = 0.3 * float(np.median(r))
    top = float((c[:, 1] + r)[small].max()) if small.any() else float((c[:, 1] + r).max())
    top = max(top, float((c[:, 1] + r)[r < 50 * np.median(r)].max()))
    centre = c[small].mean(axis=0)
    out = []
    for k, src in enumerate(rng.choice(b, size=n, replace=len(b) < n)):
        o = copy(hs, abi.RtHittable)[int(src)]
        o.p[0] = float(centre[0] + (k - n / 2.0) * 3.0 * rad + rng.uniform(-0.2, 0.2) * rad)
        o.p[1] = top + 1.5 * rad + float(rng.uniform(0, 0.3)) * rad
        o.p[2] = float(centre[2] + rng.uniform(-0.5, 0.5) * rad)
        o.radius = rad
        out.append(o)
    return out


def assert_tree_is_the_rule(h, arr, n):
    """The device tree (rt_scene_bvh_nodes) is tests/ploc_rule.py's, node for node, and passes both checks."""
    bounds, right, prim = h.bvh_nodes()
    rb, rr, rp, depth = ploc_rule.build([arr[i] for i in range(n)])
    assert np.array_equal(bounds, rb) and np.array_equal(right, rr) and np.array_equal(prim, rp)
    if len(rb):
        info = h.device_bvh_check()
        assert info["depth"] == depth and info["spheres"] == int((rp >= 0).sum())
        h.wide_bvh_check()
    return depth


def check_edit(spec, h, hs, ts, remove, append, full=True):
    arr, n = edited_array(hs, remove, append)
    info = h.rebuild(remove, append)
    assert (info.objects_removed, info.objects_appended, info.n_objects, info.on_device) == (len(remove), len(append), n, 1)
    depth = assert_tree_is_the_rule(h, arr, n)
    assert info.depth == depth and info.device_ms > 0
    assert_same_frames(h, create(arr, ts), spec, full=full)
    return arr, n


# ---- 1. the scene families: remove, append, both, a pure rebuild ----------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(SPECS))
def test_structural_edits_render_as_created(name):
    spec = SPECS[name]()
    hs, ts, keep = marshal(spec.objects)
    h = create(hs, ts)
    rng = np.random.default_rng(len(hs))
    b = bounded(hs)
    cur, n = copy(hs, abi.RtHittable), len(hs)
    # a few removed (bounded spheres, and the first object whatever it is), a few appended, both together (the last object
    # and object 1 out, two in), and a pure rebuild
    steps = [
        lambda n: (sorted(set(rng.choice(b, size=min(3, len(b) - 1), replace=False).tolist()) | {0}), []),
        lambda n: ([], fresh_spheres(hs, rng, 4)),
        lambda n: ([1, n - 1], fresh_spheres(hs, rng, 2)),
        lambda n: ([], []),
    ]
    for step in steps:
        remove, append = step(n)
        cur, n = check_edit(spec, h, cur, ts, remove, append, full=name in ("C1", "C4", "stage-n*+1"))
        assert h.n_objects == n


def test_same_array_same_tree_whatever_the_history():
    spec = SPECS["C2"]()
    hs, ts, keep = marshal(spec.objects)
    rng = np.random.default_rng(6)
    extra = fresh_spheres(hs, rng, 6)
    # history A: remove 10 and 20, then append all six
    a = create(hs, ts)
    a.rebuild([10, 20], [])
    a.rebuild([], extra)
    # history B: append three, remove, append the rest, rebuild twice more
    b = create(hs, ts)
    b.rebuild([], extra[:3])
    b.rebuild([20, 10], [])
    b.rebuild([], extra[3:])
    b.rebuild()
    b.rebuild()
    # history C: one call
    c = create(hs, ts)
    c.rebuild([10, 20], extra)
    trees = [x.bvh_nodes() for x in (a, b, c)]
    for t in trees[1:]:
        assert all(np.array_equal(p, q) for p, q in zip(trees[0], t))
    for x in (b, c):
        assert a.device_bvh_check() == x.device_bvh_check()
    arr, n = edited_array(hs, [10, 20], extra)
    assert_same_frames(a, create(arr, ts), spec, full=False)


def test_hit_object_through_every_traversal():
    spec = SPECS["C4"]()
    hs, ts, keep = marshal(spec.objects)
    h = create(hs, ts)
    rng = np.random.default_rng(2)
    remove, append = [1, 3], fresh_spheres(hs, rng, 3)
    h.rebuild(remove, append)
    arr, n = edited_array(hs, remove, append)
    fresh = create(arr, ts)
    o = np.asarray(spec.origin, float) + rng.normal(0, 0.5, (4000, 3))
    d = rng.normal(0, 1, (4000, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    for traversal in (0, 1, 2):
        pa, ta, _ = h.hit_object(o, d, traversal)
        pb, tb, _ = fresh.hit_object(o, d, traversal)
        assert np.array_equal(pa, pb) and np.array_equal(ta, tb), traversal


def test_growth_across_the_staging_limit_and_back():
    spec = _past_staging_limit()
    hs, ts, keep = marshal(spec.objects)
    b = bounded(hs)
    # start below the limit: the scene without 40 spheres
    below = sorted(b[-40:])
    small, n_small = edited_array(hs, below, [])
    h = create(small, ts)
    assert h.shared_memory_bytes() > 0
    back = [copy(hs, abi.RtHittable)[i] for i in below]
    big, n_big = check_edit(spec, h, small, ts, [], back, full=False)
    assert h.shared_memory_bytes() == 0
    check_edit(spec, h, big, ts, list(range(n_big - 40, n_big)), [], full=False)
    assert h.shared_memory_bytes() > 0


def test_planes_and_unbounded_spheres_keep_their_array_order():
    spec = SPECS["C4"]()
    hs, ts, keep = marshal(spec.objects)
    h = create(hs, ts)
    unb = [i for i in range(len(hs)) if hs[i].shape != abi.RT_SHAPE_SPHERE]
    assert len(unb) >= 2
    # remove the first unbounded object, append copies of two others (their array order is their tie-break order)
    append = [copy(hs, abi.RtHittable)[unb[-1]], copy(hs, abi.RtHittable)[unb[1]]]
    arr, n = check_edit(spec, h, hs, ts, [unb[0]], append)
    # a plane moved to the end of the array
    cur_unb = [i for i in range(n) if arr[i].shape == abi.RT_SHAPE_INFINITE_PLANE]
    if cur_unb:
        check_edit(spec, h, arr, ts, [cur_unb[0]], [copy(arr, abi.RtHittable)[cur_unb[0]]])


def test_every_bounded_sphere_removed_then_one_left():
    spec = SPECS["C4"]()
    hs, ts, keep = marshal(spec.objects)
    h = create(hs, ts)
    b = bounded(hs)
    arr, n = edited_array(hs, b, [])
    info = h.rebuild(b, [])
    assert info.n_bounded == 0 and info.nodes == 0 and info.depth == 0
    assert_same_frames(h, create(arr, ts), spec)
    one = [copy(hs, abi.RtHittable)[b[0]]]
    arr2, n2 = check_edit(spec, h, arr, ts, [], one)
    assert h.device_bvh_check()["nodes"] == 1
    # rt_scene_update moves the one sphere of the rebuilt tree
    moved = copy(arr2, abi.RtHittable)
    moved[n2 - 1].p[0] += 0.2
    assert h.update([n2 - 1], [moved[n2 - 1]]).nodes_refit == 1
    assert_same_frames(h, create(moved, ts), spec, full=False)


def test_deep_chain_falls_back_to_the_host_tree():
    spec = sample_images.few_spheres(max_w=30, max_h=17, spp=8)
    hs, ts, keep = marshal(spec.objects)
    h = create(hs, ts)
    chain = []
    base = copy(hs, abi.RtHittable)[bounded(hs)[0]]
    for i in range(70):
        o = copy([base], abi.RtHittable)[0]
        o.p[0], o.p[1], o.p[2] = 0.25, 0.5, -2.0
        o.radius = 1e-4 * 1.3 ** i
        chain.append(o)
    arr, n = edited_array(hs, [], chain)
    assert ploc_rule.build([arr[i] for i in range(n)])[3] > 60
    info = h.rebuild([], chain)
    assert info.on_device == 0 and info.depth <= 60
    fresh = create(arr, ts)
    assert all(np.array_equal(p, q) for p, q in zip(h.bvh_nodes(), fresh.bvh_nodes()))  # rt_scene_create's tree
    h.device_bvh_check()
    assert_same_frames(h, fresh, spec)
    # and the next rebuild starts from the host records
    info = h.rebuild(list(range(n - 70, n)), [])
    assert info.on_device == 1
    assert_same_frames(h, create(hs, ts), spec, full=False)


def test_update_refits_the_rebuilt_tree():
    spec = SPECS["C2"]()
    hs, ts, keep = marshal(spec.objects)
    h = create(hs, ts)
    rng = np.random.default_rng(12)
    arr, n = check_edit(spec, h, hs, ts, [5, 6, 7], fresh_spheres(hs, rng, 5), full=False)
    for k in range(3):
        arr, idx = move_and_recolour(arr, rng, 30, 5)
        info = h.update(idx, [arr[i] for i in idx])
        assert info.spheres_moved > 0
        h.device_bvh_check()
        assert_same_frames(h, create(arr, ts), spec, full=k == 2)


# ---- 2. stale frames, refusals, interleaving -----------------------------------------------------------------------------------
def test_stale_frames():
    spec = SPECS["C1"]()
    hs, ts, keep = marshal(spec.objects)
    h = create(hs, ts)
    cam = camera(spec)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    f = h.open_frame(cam, mw, mh, seed=2, flags=NOISE)
    f.advance(max_samples=3)
    before = f.read(want_sums=True)
    g0 = h.rebuild([], []).generation
    assert g0 == 1
    lib = native.lib()
    assert lib.rt_frame_advance(f.ptr, 1, 0.0, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert b"scene changed" in lib.rt_last_error()
    after = f.read(want_sums=True)
    assert all(np.array_equal(x, y) for x, y in zip(before, after))
    f.close()
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
    good = copy(hs, abi.RtHittable)[bounded(hs)[0]]

    def rec(**kw):
        e = copy([good], abi.RtHittable)[0]
        for k, v in kw.items():
            setattr(e, k, v)
        return e

    cases = [
        ([len(hs)], []), ([-1], []), ([2, 2], []), ([0, 1, 0], []),
        ([], [rec(style=99)]), ([], [rec(texture=len(ts))]), ([], [rec(radius=float("nan"))]), ([], [rec(shape=7)]),
        ([0], [good, rec(texture=len(ts) + 3)]),
    ]
    for remove, append in cases:
        with pytest.raises(native.RtError) as e:
            h.rebuild(remove, append)
        assert e.value.code == abi.RT_ERR_INVALID_ARGUMENT, (remove, e.value)
    lib = native.lib()
    one = np.zeros(1, np.int32)
    assert lib.rt_scene_rebuild(None, None, 0, None, 0, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_scene_rebuild(h.ptr, None, 1, None, 0, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_scene_rebuild(h.ptr, None, -1, None, 0, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_scene_rebuild(h.ptr, native.ptr(one), 1, None, 1, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_scene_rebuild(h.ptr, None, 0, None, -3, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert np.array_equal(h.render(cam, mw, mh, seed=5, want_sums=True)[1], ref)
    assert all(np.array_equal(a, b) for a, b in zip(nodes, h.bvh_nodes()))
    assert h.update([], []).generation == 0  # nothing changed, not even the edit count
    assert h.device_bvh_check()["spheres"] == len(bounded(hs))


def test_interleaving_renders_frames_and_rebuilds():
    spec = SPECS["C2"]()
    spec.max_width_coord, spec.max_height_coord = 150, 100
    hs, ts, keep = marshal(spec.objects)
    h = create(hs, ts)
    cam = camera(spec)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    rng = np.random.default_rng(8)
    cur, n = copy(hs, abi.RtHittable), len(hs)
    for k in range(4):
        with h.open_frame(cam, mw, mh, seed=k, flags=NOISE) as f:
            f.advance(max_samples=2)
            h.render(cam, mw, mh, seed=k + 100)
            f.advance()
            got = f.read(want_sums=True)[1]
        with create(cur, ts).open_frame(cam, mw, mh, seed=k, flags=NOISE) as g:
            g.advance()
            assert np.array_equal(got, g.read(want_sums=True)[1]), k
        remove = sorted(rng.choice(n, size=3, replace=False).tolist())
        append = fresh_spheres(cur, rng, 2 + k)
        h.rebuild(remove, append)
        cur, n = edited_array(cur, remove, append)
        a = h.render(cam, mw, mh, seed=k, want_sums=True)[1]
        assert np.array_equal(a, create(cur, ts).render(cam, mw, mh, seed=k, want_sums=True)[1])


# ---- 3. the Python wrappers ---------------------------------------------------------------------------------------------------
def test_scene_add_remove_rebuild():
    spec = sample_images.earth(max_w=48, max_h=25, spp=16)
    s = Scene.make(spec.objects, device=0)
    objs = list(spec.objects)
    cam = camera(spec)
    mw, mh = spec.max_width_coord, spec.max_height_coord

    def same(expected):
        a = s.handle.render(cam, mw, mh, seed=1, want_sums=True)[1]
        b = Scene.make(expected, device=0).handle.render(cam, mw, mh, seed=1, want_sums=True)[1]
        assert np.array_equal(a, b)

    textured = [o for o in objs if isinstance(o, Hittable.Sphere)][-1]  # the textured earth, if any, is a sphere
    info = Scene.add(s, [objs[1], textured])
    assert info.objects_appended == 2 and info.n_objects == len(objs) + 2
    objs = objs + [objs[1], textured]
    same(objs)
    Scene.remove(s, [0, 2])
    objs = [o for i, o in enumerate(objs) if i not in (0, 2)]
    same(objs)
    assert Scene.rebuild(s).objects_removed == 0
    same(objs)
    # Scene.update diffs against the restructured records
    assert Scene.update(s, objs).objects == 0
    with pytest.raises(native.RtError):
        Scene.remove(s, [len(objs)])
    multi = Scene(native.MultiHandle.__new__(native.MultiHandle), [], [], [], [0, 1])
    for call in (lambda: Scene.add(multi, []), lambda: Scene.remove(multi, []), lambda: Scene.rebuild(multi)):
        with pytest.raises(NotImplementedError):
            call()
