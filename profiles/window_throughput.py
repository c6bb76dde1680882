"""What a window of a frame (rt_render_window) costs against the whole frame (rt_render), alternated in one process on one GPU.

Workloads:
  C2 (1201 x 801, 500 spp): the full frame; centred windows holding 1/4 and 1/16 of the pixels (half and a quarter of the rows
    and of the columns); and the frame as a 4 x 4 grid of uneven tiles, timed as the sum of the 16 calls, against one
    rt_render.  The tiles' fixed costs are what the 16 calls take beyond the one frame.
  C5 (3841 x 2161, 100 k spheres, 256 spp): a centred window of 1/64 of the pixels (480 x 270) against the full frame.
Per round every variant runs once, in turn.  Device time is RtStats.total_ms (CUDA events from the first memset to the end of
the copies back; the sum over the calls for the tiles), kernel time RtStats.kernel_ms, wall time a host clock around the call
(every call ends in a stream synchronisation).  Every timed call copies back the image and the int32 sums, and every round
checks that each window's sums equal the crop of that round's full frame and that the tiles assemble into it.  It reports
medians and the spread (min and max over the rounds), the window's share of the frame's paths, and its device time as a share
of the frame's.  The card's name, power limit and clock limit are read in the same run.  Writes one JSON document to stdout
and, with --out, to that file.

  python profiles/window_throughput.py --out profiles/window_throughput_b200.json
"""
import argparse
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

SEED = 2024


def camera(spec):
    cam = native.camera_make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    cam.bounce_depth = spec.bounce_depth
    return cam


def centred(rows, cols, k):
    """The centred window of rows // k x cols // k pixels: 1/k^2 of the frame."""
    r, c = rows // k, cols // k
    return ((rows - r) // 2, (cols - c) // 2, r, c)


def uneven_tiles(rows, cols, n):
    """An n x n grid whose row and column bands grow by a third from first to last (so no band is a multiple of the tiles)."""
    def cuts(total):
        weights = np.linspace(1.0, 1.33, n)
        edges = np.concatenate([[0.0], np.cumsum(weights)]) / weights.sum() * total
        return [int(round(e)) for e in edges]
    rc, cc = cuts(rows), cuts(cols)
    return [(rc[i], cc[j], rc[i + 1] - rc[i], cc[j + 1] - cc[j]) for i in range(n) for j in range(n)]


def full_once(h, cam, spec):
    t0 = time.perf_counter()
    _, sums, st = h.render(cam, spec.max_width_coord, spec.max_height_coord, seed=SEED, want_sums=True)
    wall = (time.perf_counter() - t0) * 1e3
    return {"device_ms": st.total_ms, "kernel_ms": st.kernel_ms, "wall_ms": wall, "paths": st.paths, "launches": st.launches}, sums


def window_once(h, cam, spec, w):
    t0 = time.perf_counter()
    _, sums, st = h.render_window(cam, spec.max_width_coord, spec.max_height_coord, w, seed=SEED, want_sums=True)
    wall = (time.perf_counter() - t0) * 1e3
    return {"device_ms": st.total_ms, "kernel_ms": st.kernel_ms, "wall_ms": wall, "paths": st.paths, "launches": st.launches}, sums


def tiles_once(h, cam, spec, tiles, rows, cols):
    out = {"device_ms": 0.0, "kernel_ms": 0.0, "wall_ms": 0.0, "paths": 0, "launches": 0}
    sums = np.full((rows, cols, 4), -1, np.int32)
    for w in tiles:
        r, s = window_once(h, cam, spec, w)
        for k in out:
            out[k] += r[k]
        sums[w[0]:w[0] + w[2], w[1]:w[1] + w[3]] = s
    return out, sums


def summary(runs, key):
    xs = [r[key] for r in runs]
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


def crop(a, w):
    return a[w[0]:w[0] + w[2], w[1]:w[1] + w[3]]


WORKLOADS = {
    "C2 at 500 spp": (lambda: sample_images.random_spheres(), {"window 1/4": 2, "window 1/16": 4}, True, 5),
    "C5 at 256 spp": (lambda: sample_images.many_spheres(spp=256), {"window 1/64": 8}, False, 5),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--rounds-scale", type=float, default=1.0, help="multiplies every workload's number of rounds")
    args = ap.parse_args()
    if native.device_count() < 1:
        raise SystemExit("window_throughput.py needs a CUDA device")
    doc = {"card": card(), "seed": SEED, "workloads": {}}
    for name, (make, wins, with_tiles, rounds) in WORKLOADS.items():
        spec = make()
        rows, cols = spec.rows, spec.cols
        hs, ts, keep = marshal(spec.objects)
        h = native.SceneHandle(hs, ts, 0, keepalive=keep)
        cam = camera(spec)
        windows = {k: centred(rows, cols, d) for k, d in wins.items()}
        tiles = uneven_tiles(rows, cols, 4) if with_tiles else None
        # warm-up: modules, buffers, launch plans
        full_once(h, cam, spec)
        for w in windows.values():
            window_once(h, cam, spec, w)
        runs = {"full frame": [], **{k: [] for k in windows}}
        if tiles:
            runs["4 x 4 uneven tiles"] = []
            tiles_once(h, cam, spec, tiles, rows, cols)
        equal = True
        for _ in range(max(1, int(round(rounds * args.rounds_scale)))):
            r, full_sums = full_once(h, cam, spec)
            runs["full frame"].append(r)
            for k, w in windows.items():
                r, s = window_once(h, cam, spec, w)
                runs[k].append(r)
                equal = equal and np.array_equal(s, crop(full_sums, w))
            if tiles:
                r, s = tiles_once(h, cam, spec, tiles, rows, cols)
                runs["4 x 4 uneven tiles"].append(r)
                equal = equal and np.array_equal(s, full_sums)
        full_dev = summary(runs["full frame"], "device_ms")["median"]
        full_paths = runs["full frame"][0]["paths"]
        wl = {"rows": rows, "cols": cols, "spp": spec.spp, "rounds": len(runs["full frame"]), "sums_equal": equal, "variants": {}}
        for k, rs in runs.items():
            v = {key: summary(rs, key) for key in ("device_ms", "kernel_ms", "wall_ms")}
            v["paths"] = rs[0]["paths"]
            v["launches"] = rs[0]["launches"]
            v["path_share"] = rs[0]["paths"] / full_paths
            v["device_share"] = v["device_ms"]["median"] / full_dev
            if k in windows:
                v["window"] = list(windows[k])
                v["pixel_share"] = windows[k][2] * windows[k][3] / (rows * cols)
            if k.endswith("tiles"):
                v["tiles"] = [list(t) for t in tiles]
                v["fixed_cost_ms"] = v["device_ms"]["median"] - full_dev
                v["fixed_cost_ms_per_tile"] = v["fixed_cost_ms"] / len(tiles)
            wl["variants"][k] = v
            print(f"{name}, {k}: device {v['device_ms']['median']:.2f} ms [{v['device_ms']['min']:.2f}, {v['device_ms']['max']:.2f}], "
                  f"{100 * v['device_share']:.2f} % of the frame's for {100 * v['path_share']:.2f} % of its paths", file=sys.stderr)
        doc["workloads"][name] = wl
        h.close()
        if not equal:
            raise SystemExit(f"{name}: a window's sums differ from the crop of the frame")
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
