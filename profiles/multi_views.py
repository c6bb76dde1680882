"""What a batch of views split over several GPUs gains (rt_multi_render_views, rt_multi_frame_begin_views), alternated in one
process with the forms it replaces, for every world from 1 to the number of visible devices.

Workloads: section 16's three batches, in one call: a 64-view C1 turntable (401 x 225, 16 spp); 24 previews of the RTOW scene
(C2's objects) at max coordinates (200, 133), 32 spp; 8 full C2 views (1201 x 801, 500 spp).  And section 17's progressive C1
turntable (64 views at 1024 spp, RT_FLAG_NOISE, rule tau = 1, m = k = 64, passes of 250 ms).
Forms, alternated within every round at world w (devices 0 .. w - 1, one rank each; ranks never share a device here):
  batch_w   the batch over the w devices (MultiHandle.render_views / open_frame_views);
  loop_w    one rt_multi_render (rt_multi_frame_begin) per view on the same w devices;
  one_gpu   rt_render_views (rt_frame_begin_views) on device 0.
Times: wall time (host clock around the call or the loop; every call returns with its device work done) and device time
(one call: RtStats.kernel_ms of the multi forms, the slowest device's probe -> reduce span, which includes the RGB8 stores
into pinned host memory, against RtStats.total_ms of rt_render_views, which includes its device -> host copy; progressive:
RtFrameProgress.device_ms).  The loops' device times are sums over their calls and leave out the host gaps between them.
The timed calls return images only; the sums compared are from untimed calls of the same forms right after.  In every round
the int32 sums (and Q, progressive) of the three forms must be equal ("sums_equal").
With one device visible only world 1 is measured, and the multi-GPU columns are recorded as not measured.  The card's name,
power limit and SM clock limit are read in the same run.  Writes one JSON document to stdout and, with --out, to that file.

  python profiles/multi_views.py --out profiles/multi_views_b200.json
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
from ray_tracing_fsharp_b200 import abi, native, sample_images  # noqa: E402
from ray_tracing_fsharp_b200.domain import marshal  # noqa: E402
from profiles.multi_progressive import card  # noqa: E402
from profiles.views_throughput import orbit  # noqa: E402

NOISE = abi.RT_FLAG_NOISE
TARGET_MS = 250.0
RULE = (1.0, 64, 64)

ONE_CALL = {
    "C1 turntable, 64 views": (lambda: sample_images.few_spheres(), 64, 5),
    "RTOW previews, 24 views at (200, 133), 32 spp": (lambda: sample_images.random_spheres(max_w=200, max_h=133, spp=32), 24, 5),
    "C2, 8 full views at 500 spp": (lambda: sample_images.random_spheres(), 8, 3),
}
PROGRESSIVE = {"C1 turntable, 64 views at 1024 spp": (lambda: sample_images.few_spheres(spp=1024), 64, 2)}


def sha(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


# ---- one call -------------------------------------------------------------------------------------------------------------
def batch_once(h, cams, spec, seeds, device_field):
    t0 = time.perf_counter()
    _, _, st = h.render_views(cams, spec.max_width_coord, spec.max_height_coord, seeds=seeds)
    wall = (time.perf_counter() - t0) * 1e3
    _, sums, _ = h.render_views(cams, spec.max_width_coord, spec.max_height_coord, seeds=seeds, want_sums=True)
    return {"device_ms": getattr(st, device_field), "wall_ms": wall, "paths": st.paths, "sums": sha(sums)}


def loop_once(m, cams, spec, seeds):
    device, wall, paths = 0.0, 0.0, 0
    for cam, seed in zip(cams, seeds):
        t0 = time.perf_counter()
        _, _, st = m.render(cam, spec.max_width_coord, spec.max_height_coord, seed=seed)
        wall += (time.perf_counter() - t0) * 1e3
        device += st.kernel_ms
        paths += st.paths
    parts = [m.render(cam, spec.max_width_coord, spec.max_height_coord, seed=seed, want_sums=True)[1] for cam, seed in zip(cams, seeds)]
    return {"device_ms": device, "wall_ms": wall, "paths": paths, "sums": sha(np.stack(parts))}


# ---- progressive ----------------------------------------------------------------------------------------------------------
def drive(f):
    f.set_convergence(*RULE)
    while not f.progress.done:
        f.advance(target_ms=TARGET_MS)
    f.read()
    return f.progress


def frame_batch_once(h, cams, spec, seeds):
    t0 = time.perf_counter()
    with h.open_frame_views(cams, spec.max_width_coord, spec.max_height_coord, seeds=seeds, flags=NOISE) as f:
        p = drive(f)
        wall = (time.perf_counter() - t0) * 1e3
        _, sums = f.read(want_sums=True)
        sq = f.noise(0.0, want_map=False, want_sq=True)[2]
    return {"device_ms": p.device_ms, "wall_ms": wall, "passes": p.passes, "paths": p.paths_done, "sums": sha(sums, sq)}


def frame_loop_once(m, cams, spec, seeds):
    device, wall, passes, paths, sums, sqs = 0.0, 0.0, 0, 0, [], []
    for cam, seed in zip(cams, seeds):
        t0 = time.perf_counter()
        with m.open_frame(cam, spec.max_width_coord, spec.max_height_coord, seed=seed, flags=NOISE) as f:
            p = drive(f)
            wall += (time.perf_counter() - t0) * 1e3
            sums.append(f.read(want_sums=True)[1])
            sqs.append(f.noise(0.0, want_map=False, want_sq=True)[2])
        device, passes, paths = device + p.device_ms, passes + p.passes, paths + p.paths_done
    return {"device_ms": device, "wall_ms": wall, "passes": passes, "paths": paths, "sums": sha(np.stack(sums), np.stack(sqs))}


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


def compare(runs, keys):
    """Medians and spreads per form, and the gain of the batch over the loop and over one GPU (% of their median)."""
    out = {form: {k: spread([r[k] for r in rs]) for k in keys} for form, rs in runs.items()}
    for k in ("device_ms", "wall_ms"):
        b = out["batch"][k]["median"]
        out[f"{k}_gain_over_loop_pct"] = 100.0 * (out["loop"][k]["median"] - b) / out["loop"][k]["median"]
        out[f"{k}_gain_over_one_gpu_pct"] = 100.0 * (out["one_gpu"][k]["median"] - b) / out["one_gpu"][k]["median"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds-scale", type=float, default=1.0, help="multiplies every workload's number of rounds")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    n_dev = native.device_count()
    if n_dev < 1:
        raise SystemExit("multi_views.py needs a CUDA device")
    worlds = list(range(1, n_dev + 1))
    doc = {"card": card(), "devices_visible": n_dev, "worlds_measured": worlds,
           "multi_gpu": "measured" if n_dev > 1 else "not measured: one device visible",
           "progressive_rule": {"tolerance": RULE[0], "min_samples": RULE[1], "interval": RULE[2], "target_ms": TARGET_MS},
           "one_call": {}, "progressive": {}}
    for table, key, keys in ((ONE_CALL, "one_call", ("device_ms", "wall_ms")), (PROGRESSIVE, "progressive", ("device_ms", "wall_ms", "passes"))):
        for name, (make, n, rounds) in table.items():
            spec = make()
            hs, ts, keep = marshal(spec.objects)
            one = native.SceneHandle(hs, ts, 0, keepalive=keep)
            cams = orbit(spec, n)
            seeds = [1000 + v for v in range(n)]
            w_doc = {"views": n, "rows": spec.rows, "cols": spec.cols, "spp": spec.spp, "worlds": {}}
            for w in worlds:
                m = native.MultiHandle(hs, ts, list(range(w)), keepalive=keep)
                if key == "one_call":
                    forms = {"batch": lambda: batch_once(m, cams, spec, seeds, "kernel_ms"), "loop": lambda: loop_once(m, cams, spec, seeds),
                             "one_gpu": lambda: batch_once(one, cams, spec, seeds, "total_ms")}
                else:
                    forms = {"batch": lambda: frame_batch_once(m, cams, spec, seeds), "loop": lambda: frame_loop_once(m, cams, spec, seeds),
                             "one_gpu": lambda: frame_batch_once(one, cams, spec, seeds)}
                for f in forms.values():  # warm-up: modules, buffers, launch plans
                    f()
                runs = {k: [] for k in forms}
                equal = []
                for _ in range(max(1, int(round(rounds * args.rounds_scale)))):
                    for k, f in forms.items():
                        runs[k].append(f())
                    equal.append(len({runs[k][-1]["sums"] for k in forms}) == 1)
                r = compare(runs, keys)
                r["rounds"] = len(equal)
                r["sums_equal"] = equal
                r["paths"] = {k: runs[k][0]["paths"] for k in forms}
                if w == 1:
                    r["note"] = ("world 1: batch is rt_multi_render_views on one device and one_gpu is rt_render_views "
                                 "(rt_frame_begin_views), timed alternately; compare them within the spread")
                w_doc["worlds"][str(w)] = r
                m.close()
                print(f"{name}, world {w}: batch {r['batch']['wall_ms']['median']:.2f} ms, loop {r['loop']['wall_ms']['median']:.2f} ms, "
                      f"one GPU {r['one_gpu']['wall_ms']['median']:.2f} ms (wall), sums equal: {equal}", file=sys.stderr, flush=True)
                if not all(equal):
                    raise SystemExit(f"{name}, world {w}: the forms' sums differ")
            if n_dev == 1:
                w_doc["worlds"]["2..8"] = "not measured: one device visible"
            one.close()
            doc[key][name] = w_doc
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
