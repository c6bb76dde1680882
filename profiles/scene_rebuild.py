"""What a structural edit (rt_scene_rebuild) costs against creating the scene anew, and how fast its tree is to walk.

1. Device time of a rebuild of the current objects (RtSceneRebuild.device_ms) on C2 and C5, split by stage (collect, sort,
   cluster, flatten) from the library's RTFS_DEBUG_REBUILD trace, which records CUDA events between the stages.
2. Host wall time on C5 (100 k spheres) of adding one sphere, removing one and adding 1 000 (SceneHandle.rebuild, which ends in
   a stream synchronisation), against rt_scene_create of the same array (SceneHandle of the records: host SAH build and upload).
   Rounds alternate the two.
3. Frame time (RtStats.kernel_ms) on the device tree against the host SAH tree of the same array: C2 at 1201 x 801 and 500 spp,
   C5 at 961 x 541 and 16 spp (DESIGN.md section 20's drift sizes).  Rounds alternate, and every round compares the two
   frames' sums (np.array_equal).
Medians with min / max.  The card's name, power limit and clock limit are read in the same run.  Writes one JSON document to
stdout and, with --out, to that file.

  python profiles/scene_rebuild.py --out profiles/scene_rebuild_b200.json
"""
import argparse
import ctypes as C
import json
import os
import re
import statistics
import sys
import tempfile
import time

import numpy as np

os.environ["RTFS_DEBUG_REBUILD"] = "1"  # read once, at the first rebuild
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ray_tracing_fsharp_b200 import abi, native, sample_images  # noqa: E402
from ray_tracing_fsharp_b200.domain import marshal  # noqa: E402
from profiles.progressive_passes import card  # noqa: E402


def camera(spec, spp=None):
    cam = native.camera_make_basic(spp or spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    cam.bounce_depth = spec.bounce_depth
    return cam


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


class Trace:
    """Captures what the library writes to stderr (file descriptor 2) during a block."""

    def __enter__(self):
        self.f = tempfile.TemporaryFile(mode="w+b")
        sys.stderr.flush()
        self.saved = os.dup(2)
        os.dup2(self.f.fileno(), 2)
        return self

    def __exit__(self, *exc):
        os.dup2(self.saved, 2)
        os.close(self.saved)
        self.f.seek(0)
        self.text = self.f.read().decode("utf-8", "replace")
        self.f.close()


STAGES = ("collect_ms", "sort_ms", "cluster_ms", "flatten_ms", "device_ms")


def stage_times(name, spec, rounds):
    hs, ts, keep = marshal(spec.objects)
    h = native.SceneHandle(hs, ts, 0, keepalive=keep)
    h.rebuild()  # warm-up: scratch allocation, module load
    per = {k: [] for k in STAGES}
    info = None
    for _ in range(rounds):
        with Trace() as t:
            info = h.rebuild()
        line = [x for x in t.text.splitlines() if x.startswith("rtfs: rebuild")][-1]
        for k in STAGES:
            per[k].append(float(re.search(k + r"=([0-9.]+)", line).group(1)))
        per.setdefault("rounds", []).append(int(re.search(r"rounds=([0-9]+)", line).group(1)))
    h.close()
    return {"scene": name, "objects": len(hs), "spheres": info.n_bounded, "depth": info.depth, "nodes": info.nodes,
            "clustering_iterations": per.pop("rounds")[-1], "launches": info.launches, **{k: spread(v) for k, v in per.items()}}


def host_cost(rounds):
    spec = sample_images.many_spheres()
    hs, ts, keep = marshal(spec.objects)
    h = native.SceneHandle(hs, ts, 0, keepalive=keep)
    h.rebuild()
    rng = np.random.default_rng(3)
    bounded = [i for i in range(len(hs)) if hs[i].shape == abi.RT_SHAPE_SPHERE and hs[i].radius >= 0]
    size = C.sizeof(abi.RtHittable)
    cur = bytearray(bytes(hs))
    out = []

    def new_spheres(k):
        recs = []
        for i in rng.choice(bounded, size=k, replace=False):
            o = abi.RtHittable.from_buffer_copy(cur, int(i) * size)
            for a in range(3):
                o.p[a] += float(rng.normal(0, 2.0))
            recs.append(o)
        return recs

    for case, n_remove, n_add in (("add 1", 0, 1), ("remove 1", 1, 0), ("add 1000", 0, 1000)):
        wall, dev, create = [], [], []
        for _ in range(rounds):
            n = len(cur) // size
            remove = sorted(rng.choice(n, size=n_remove, replace=False).tolist())
            add = new_spheres(n_add)
            t0 = time.perf_counter()
            info = h.rebuild(remove, add)
            wall.append((time.perf_counter() - t0) * 1e3)
            dev.append(info.device_ms)
            arr = np.frombuffer(bytes(cur), np.uint8).reshape(-1, size)
            keep_rows = np.ones(n, bool)
            keep_rows[remove] = False
            cur = bytearray(arr[keep_rows].tobytes() + b"".join(bytes(o) for o in add))
            recs = (abi.RtHittable * (len(cur) // size)).from_buffer_copy(cur)
            t0 = time.perf_counter()
            fresh = native.SceneHandle(recs, ts, 0, keepalive=keep)
            create.append((time.perf_counter() - t0) * 1e3)
            fresh.close()
        out.append({"case": case, "rebuild_wall_ms": spread(wall), "rebuild_device_ms": spread(dev), "create_wall_ms": spread(create)})
    h.close()
    return {"scene": "C5, 100 000 spheres", "cases": out}


def frame_time(name, spec, rounds):
    hs, ts, keep = marshal(spec.objects)
    dev_tree = native.SceneHandle(hs, ts, 0, keepalive=keep)
    dev_tree.rebuild()
    host_tree = native.SceneHandle(hs, ts, 0, keepalive=keep)
    cam = camera(spec)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    for h in (dev_tree, host_tree):  # warm-up
        h.render(cam, mw, mh, seed=99)
    t_dev, t_host, equal = [], [], True
    for r in range(rounds):
        _, sa, st_a = dev_tree.render(cam, mw, mh, seed=r, want_sums=True)
        _, sb, st_b = host_tree.render(cam, mw, mh, seed=r, want_sums=True)
        t_dev.append(st_a.kernel_ms)
        t_host.append(st_b.kernel_ms)
        equal = equal and bool(np.array_equal(sa, sb))
    md, mh_ = statistics.median(t_dev), statistics.median(t_host)
    return {"scene": name, "pixels": f"{2 * mw + 1} x {2 * mh + 1}", "spp": spec.spp, "device_tree": dev_tree.device_bvh_check(),
            "host_tree": host_tree.device_bvh_check(), "device_tree_kernel_ms": spread(t_dev), "host_tree_kernel_ms": spread(t_host),
            "ratio_of_medians": md / mh_, "sums_equal_every_round": equal}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--frame-rounds", type=int, default=5)
    ap.add_argument("--out")
    a = ap.parse_args()
    doc = {"card": card(),
           "stages": [stage_times("C2", sample_images.random_spheres(spp=4), a.rounds),
                      stage_times("C5", sample_images.many_spheres(), a.rounds)],
           "host_cost": host_cost(a.rounds),
           "frames": [frame_time("C2", sample_images.random_spheres(max_w=600, max_h=400, spp=500), a.frame_rounds),
                      frame_time("C5", sample_images.many_spheres(max_w=480, max_h=270, spp=16), a.frame_rounds)]}
    text = json.dumps(doc, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
