"""What rendering many views in one rt_render_views call gains over one rt_render call per view, alternated in one process on
one GPU.

Workloads: a 64-view C1 turntable (401 x 225, 16 spp); 24 previews of the RTOW scene (C2's objects) at max coordinates
(200, 133), 32 spp; 8 full C2 views (1201 x 801, 500 spp), where one frame already fills the GPU.  Per workload and round it
times the batch and the loop of the same views: device time (CUDA events: RtStats.total_ms of the batch, the sum of the
views' total_ms for the loop; the loop's device time leaves out the host gaps between its calls) and wall time (host clock
around the call or the loop; every call ends in a stream synchronisation).  The timed calls copy the images back, not the
sums.  It reports medians, the spread (min and max over the rounds) and the gain of the batch in %, and checks that the
batch's int32 sums equal the loop's in every round.
The card's name, power limit and clock limit are read in the same run.  Writes one JSON document to stdout and, with
--out, to that file.

  python profiles/views_throughput.py --out /tmp/views_throughput.json
"""
import argparse
import hashlib
import json
import os
import statistics
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ray_tracing_fsharp_b200 import native, sample_images  # noqa: E402
from ray_tracing_fsharp_b200.domain import marshal  # noqa: E402
from profiles.progressive_passes import card  # noqa: E402


def orbit(spec, n):
    """n cameras on a circle around the spec's look-at point, through its origin."""
    origin, look = np.asarray(spec.origin, float), np.asarray(spec.look_at, float)
    rel = origin - look
    cams = []
    for v in range(n):
        a = 2.0 * np.pi * v / n
        ca, sa = np.cos(a), np.sin(a)
        o = look + np.array([ca * rel[0] + sa * rel[2], rel[1], -sa * rel[0] + ca * rel[2]])
        d = look - o
        cam = native.camera_make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, o, d / np.linalg.norm(d), spec.view_up)
        cam.bounce_depth = spec.bounce_depth
        cams.append(cam)
    return cams


WORKLOADS = {
    "C1 turntable, 64 views": (lambda: sample_images.few_spheres(), 64, 15),
    "RTOW previews, 24 views at (200, 133), 32 spp": (lambda: sample_images.random_spheres(max_w=200, max_h=133, spp=32), 24, 10),
    "C2, 8 full views at 500 spp": (lambda: sample_images.random_spheres(), 8, 4),
}


# The timed calls return the images only, as a viewer would; the sums that are compared come from an untimed call of the
# same form right after (the sums of 64 C1 views are 92 MB, whose copy would otherwise dominate the device time).
def batch_once(h, cams, spec, seeds):
    t0 = time.perf_counter()
    _, _, st = h.render_views(cams, spec.max_width_coord, spec.max_height_coord, seeds=seeds)
    wall = (time.perf_counter() - t0) * 1e3
    _, sums, _ = h.render_views(cams, spec.max_width_coord, spec.max_height_coord, seeds=seeds, want_sums=True)
    return {"device_ms": st.total_ms, "kernel_ms": st.kernel_ms, "wall_ms": wall, "launches": st.launches, "paths": st.paths,
            "sums": hashlib.sha256(sums.tobytes()).hexdigest()}


def loop_once(h, cams, spec, seeds):
    device = kernel = 0.0
    launches = paths = 0
    t0 = time.perf_counter()
    for cam, seed in zip(cams, seeds):
        _, _, st = h.render(cam, spec.max_width_coord, spec.max_height_coord, seed=seed)
        device += st.total_ms
        kernel += st.kernel_ms
        launches += st.launches
        paths += st.paths
    wall = (time.perf_counter() - t0) * 1e3
    parts = [h.render(cam, spec.max_width_coord, spec.max_height_coord, seed=seed, want_sums=True)[1] for cam, seed in zip(cams, seeds)]
    return {"device_ms": device, "kernel_ms": kernel, "wall_ms": wall, "launches": launches, "paths": paths,
            "sums": hashlib.sha256(np.stack(parts).tobytes()).hexdigest()}


def summary(runs, key):
    xs = [r[key] for r in runs]
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--rounds-scale", type=float, default=1.0, help="multiplies every workload's number of rounds")
    args = ap.parse_args()
    if native.device_count() < 1:
        raise SystemExit("views_throughput.py needs a CUDA device")
    doc = {"card": card(), "workloads": {}}
    for name, (make, n, rounds) in WORKLOADS.items():
        spec = make()
        hs, ts, keep = marshal(spec.objects)
        h = native.SceneHandle(hs, ts, 0, keepalive=keep)
        cams = orbit(spec, n)
        seeds = [1000 + v for v in range(n)]
        batch_once(h, cams, spec, seeds)  # warm-up: modules, buffers, launch plans
        loop_once(h, cams, spec, seeds)
        batch, loop = [], []
        for _ in range(max(1, int(round(rounds * args.rounds_scale)))):
            batch.append(batch_once(h, cams, spec, seeds))
            loop.append(loop_once(h, cams, spec, seeds))
        equal = all(b["sums"] == lp["sums"] for b, lp in zip(batch, loop))
        w = {"views": n, "rows": spec.rows, "cols": spec.cols, "spp": spec.spp, "rounds": len(batch), "sums_equal": equal,
             "paths_per_call": batch[0]["paths"], "launches": {"batch": batch[0]["launches"], "loop": loop[0]["launches"]}}
        for key in ("device_ms", "kernel_ms", "wall_ms"):
            b, lp = summary(batch, key), summary(loop, key)
            w[key] = {"batch": b, "loop": lp, "gain_pct": 100.0 * (lp["median"] - b["median"]) / lp["median"]}
        w["mpaths_per_s_device"] = {"batch": batch[0]["paths"] / w["device_ms"]["batch"]["median"] / 1e3,
                                    "loop": loop[0]["paths"] / w["device_ms"]["loop"]["median"] / 1e3}
        doc["workloads"][name] = w
        h.close()
        print(f"{name}: device {w['device_ms']['batch']['median']:.2f} vs {w['device_ms']['loop']['median']:.2f} ms "
              f"({w['device_ms']['gain_pct']:+.1f} %), wall {w['wall_ms']['batch']['median']:.2f} vs {w['wall_ms']['loop']['median']:.2f} ms "
              f"({w['wall_ms']['gain_pct']:+.1f} %), sums equal: {equal}", file=sys.stderr)
        if not equal:
            raise SystemExit(f"{name}: the batch's sums differ from the loop's")
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
