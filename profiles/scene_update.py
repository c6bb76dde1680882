"""What an in-place edit (rt_scene_update) costs against creating the scene anew, and how a refit tree ages under animation.

1. Update cost on C5 (100 k spheres): 1, 1 000 and 100 000 moved spheres (random steps of 0.05 radii), each edit applied with
   SceneHandle.update and timed by a host clock (the call ends in a stream synchronisation) and by its device_ms; against
   rt_scene_create of the edited array (SAH build and upload: SceneHandle of the marshalled records) and against Python's
   marshal() of the domain objects.  Rounds alternate the two, medians and min / max are reported.
2. Tree-quality drift.  C2 (1201 x 801) at 64 spp per step: its small spheres bob on a sine over 120 steps (Scene.update with the
   whole new object list), every step's frame timed on the refit tree against a scene recreated from the same objects.  C5 at
   961 x 541 and 16 spp: every sphere takes a random-walk step of 0.05 radii per step for 30 steps.  Frame time is RtStats
   kernel_ms.
3. In every step of every run the sums of the edited scene and of the recreated one are compared (np.array_equal).  A step
   whose sums differ is examined: how many pixels differ; whether the refit tree passes rt_scene_device_bvh_check and equals
   tests/refit_rule.py over the edited spheres (then it holds exactly the boxes a host build of its topology would); and
   whether the recreated scene's own binary and 8-wide trees disagree on that frame, i.e. whether the frame has a closest hit
   that is an exact tie in t between two spheres, which different topologies may resolve differently.
The card's name, power limit and clock limit are read in the same run.  Writes one JSON document to stdout and, with --out, to
that file.

  python profiles/scene_update.py --out profiles/scene_update_b200.json
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ray_tracing_fsharp_b200 import abi, native, sample_images  # noqa: E402
from ray_tracing_fsharp_b200.domain import Hittable, Sphere, marshal  # noqa: E402
from ray_tracing_fsharp_b200.scene import Scene  # noqa: E402
from profiles.progressive_passes import card  # noqa: E402

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import refit_rule  # noqa: E402


def camera(spec, spp=None):
    cam = native.camera_make_basic(spp or spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    cam.bounce_depth = spec.bounce_depth
    return cam


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


def bob(objects, step, steps=120):
    """C2's small spheres bob on a sine: step `step` of `steps`."""
    out = []
    for k, o in enumerate(objects):
        if isinstance(o, Hittable.Sphere) and o.sphere.Radius == 0.2:
            c = o.sphere.Centre
            o = Hittable.Sphere(Sphere.make(o.sphere.Style, (c[0], c[1] + 0.15 * np.sin(2.0 * np.pi * step / steps + 0.7 * k), c[2]),
                                            o.sphere.Radius))
        out.append(o)
    return out


def update_cost(rounds):
    spec = sample_images.many_spheres()
    t0 = time.perf_counter()
    hs, ts, keep = marshal(spec.objects)
    marshal_ms = (time.perf_counter() - t0) * 1e3
    h = native.SceneHandle(hs, ts, 0, keepalive=keep)
    bounded = np.array([i for i in range(len(hs)) if hs[i].shape == abi.RT_SHAPE_SPHERE and hs[i].radius >= 0])
    rng = np.random.default_rng(3)
    cur = (abi.RtHittable * len(hs))()
    C.memmove(cur, hs, C.sizeof(cur))
    out = {"scene": "C5, 100 000 spheres", "objects": len(hs), "marshal_ms": marshal_ms, "cases": []}
    h.update([int(bounded[0])], [cur[int(bounded[0])]])  # the first edit that moves a sphere uploads the min / max tree
    for n in (1, 1000, len(bounded)):
        wall, dev, create_ms, refit = [], [], [], []
        equal = True
        for _ in range(rounds):
            idx = np.sort(rng.choice(bounded, size=n, replace=False))
            for i in idx:
                o = cur[int(i)]
                for a in range(3):
                    o.p[a] += rng.normal(0, 0.05 * o.radius)
            recs = (abi.RtHittable * n)(*[cur[int(i)] for i in idx])
            oi = idx.astype(np.int32)
            t0 = time.perf_counter()
            info = h.update(oi, recs)
            wall.append((time.perf_counter() - t0) * 1e3)
            dev.append(info.device_ms)
            refit.append(info.nodes_refit)
            t0 = time.perf_counter()
            fresh = native.SceneHandle(cur, ts, 0)
            create_ms.append((time.perf_counter() - t0) * 1e3)
            cam = camera(spec, 1)
            a = h.render(cam, 120, 68, seed=1, want_sums=True)[1]
            b = fresh.render(cam, 120, 68, seed=1, want_sums=True)[1]
            equal = equal and bool(np.array_equal(a, b))
            fresh.close()
        out["cases"].append({"spheres_moved": n, "update_wall_ms": spread(wall), "update_device_ms": spread(dev),
                             "nodes_refit": spread(refit), "create_wall_ms": spread(create_ms), "sums_equal_every_round": equal})
    h.close()
    return out


def drift_c2(steps, spp):
    spec = sample_images.random_spheres(spp=spp)
    cam = camera(spec)
    s = Scene.make(spec.objects, device=0)
    rows = []
    for step in range(1, steps + 1):
        objs = bob(spec.objects, step)
        t0 = time.perf_counter()
        info = Scene.update(s, objs)
        upd = (time.perf_counter() - t0) * 1e3
        _, a, st_a = s.handle.render(cam, spec.max_width_coord, spec.max_height_coord, seed=step, want_sums=True)
        fresh = Scene.make(objs, device=0)
        _, b, st_b = fresh.handle.render(cam, spec.max_width_coord, spec.max_height_coord, seed=step, want_sums=True)
        row = {"step": step, "refit_kernel_ms": st_a.kernel_ms, "recreated_kernel_ms": st_b.kernel_ms, "scene_update_wall_ms": upd,
               "update_device_ms": info.device_ms, "sums_equal": bool(np.array_equal(a, b))}
        if not row["sums_equal"]:
            row["examined"] = examine(s.handle, fresh.handle, marshal(objs)[0], cam, spec, step, a, b)
        fresh.handle.close()
        rows.append(row)
    return summarise("C2 1201 x 801, small spheres bobbing on a sine", steps, spp, rows)


def drift_c5(steps, spp):
    spec = sample_images.many_spheres(max_w=480, max_h=270, spp=spp)
    cam = camera(spec)
    hs, ts, keep = marshal(spec.objects)
    h = native.SceneHandle(hs, ts, 0, keepalive=keep)
    bounded = np.array([i for i in range(len(hs)) if hs[i].shape == abi.RT_SHAPE_SPHERE and hs[i].radius >= 0])
    cur = (abi.RtHittable * len(hs))()
    C.memmove(cur, hs, C.sizeof(cur))
    rng = np.random.default_rng(4)
    rows = []
    for step in range(1, steps + 1):
        for i in bounded:
            o = cur[int(i)]
            for a in range(3):
                o.p[a] += rng.normal(0, 0.05 * o.radius)
        recs = (abi.RtHittable * len(bounded))(*[cur[int(i)] for i in bounded])
        info = h.update(bounded.astype(np.int32), recs)
        _, a, st_a = h.render(cam, spec.max_width_coord, spec.max_height_coord, seed=step, want_sums=True)
        fresh = native.SceneHandle(cur, ts, 0)
        _, b, st_b = fresh.render(cam, spec.max_width_coord, spec.max_height_coord, seed=step, want_sums=True)
        row = {"step": step, "refit_kernel_ms": st_a.kernel_ms, "recreated_kernel_ms": st_b.kernel_ms, "update_device_ms": info.device_ms,
               "sums_equal": bool(np.array_equal(a, b))}
        if not row["sums_equal"]:
            row["examined"] = examine(h, fresh, cur, cam, spec, step, a, b)
        fresh.close()
        rows.append(row)
    h.close()
    return summarise("C5 961 x 541, 100 k spheres in a random walk of 0.05 radii per step", steps, spp, rows)


def examine(h, fresh, records, cam, spec, seed, a, b):
    """Why the sums `a` (edited scene h) and `b` (recreated scene) of one frame differ (see the module's note 3)."""
    mw, mh = spec.max_width_coord, spec.max_height_coord
    out = {"pixels_differing": int((a != b).any(axis=-1).sum())}
    try:
        h.device_bvh_check()
        out["device_bvh_check"] = "passed"
    except native.RtError as e:
        out["device_bvh_check"] = str(e)
    bounds, right, prim = h.bvh_nodes()
    out["tree_equals_refit_rule"] = bool(np.array_equal(refit_rule.refit(right, prim, records).astype(np.float64), bounds))
    wide = fresh.render(cam, mw, mh, seed=seed, want_sums=True, flags=abi.RT_FLAG_WIDE_BVH)[1]
    out["recreated_binary_vs_wide_pixels_differing"] = int((wide != b).any(axis=-1).sum())
    return out


def summarise(name, steps, spp, rows):
    ratio = [r["refit_kernel_ms"] / r["recreated_kernel_ms"] for r in rows]
    return {"scene": name, "steps": steps, "spp": spp, "sums_equal_every_step": all(r["sums_equal"] for r in rows),
            "steps_differing": [r["step"] for r in rows if not r["sums_equal"]],
            "refit_over_recreated": {"first_10": statistics.median(ratio[:10]), "last_10": statistics.median(ratio[-10:]),
                                     "max": max(ratio)},
            "steps_detail": rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--c2-steps", type=int, default=120)
    ap.add_argument("--c5-steps", type=int, default=30)
    ap.add_argument("--out")
    args = ap.parse_args()
    if native.device_count() < 1:
        raise SystemExit("scene_update.py measures on a GPU: no CUDA device is visible")
    doc = {"card": card(), "update_cost": update_cost(args.rounds), "drift": [drift_c2(args.c2_steps, 64), drift_c5(args.c5_steps, 16)]}
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
