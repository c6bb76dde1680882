"""What rendering a batch of views as one converging progressive frame (rt_frame_begin_views) gains over a loop of single
converging frames (rt_frame_begin per view) with the same seeds and rule, alternated in one process on one GPU.

Workloads: a 64-view C1 turntable (401 x 225, 1024 spp); 24 previews of the RTOW scene (C2's objects) at max coordinates
(200, 133), 256 spp; 8 full C2 views (1201 x 801, 500 spp).  Every frame carries RT_FLAG_NOISE and the rule tau = 1,
m = k = 64, and is advanced in passes of about 250 ms of device time until done, then its images are read, as a viewer
would.  Device time is RtFrameProgress.device_ms (CUDA events: the probe and every pass) of the batch, and the sum over the
views for the loop (which leaves out the host gaps between its calls).  Wall time is the host clock from the open to the
read; every call ends in a stream synchronisation.  Medians, min and max over the rounds, and the gain of the batch in %.
The batch's int32 sums and Q must equal the loop's in every round.
Also, on the turntable: the price of the flag on the batch, i.e. the batch with RT_FLAG_NOISE and no rule against the batch
without RT_FLAG_NOISE (same passes).
The card's name, power limit and clock limit are read in the same run.  Writes one JSON document to stdout and, with --out,
to that file.

  python profiles/views_progressive.py --out /tmp/views_progressive.json
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
from profiles.progressive_passes import card  # noqa: E402
from profiles.views_throughput import orbit  # noqa: E402

TARGET_MS = 250.0
RULE = (1.0, 64, 64)
NOISE = abi.RT_FLAG_NOISE

WORKLOADS = {
    "C1 turntable, 64 views at 1024 spp": (lambda: sample_images.few_spheres(spp=1024), 64, 3),
    "RTOW previews, 24 views at (200, 133), 256 spp": (lambda: sample_images.random_spheres(max_w=200, max_h=133, spp=256), 24, 5),
    "C2, 8 full views at 500 spp": (lambda: sample_images.random_spheres(), 8, 3),
}


def drive(frame, rule):
    if rule is not None:
        frame.set_convergence(*rule)
    while not frame.progress.done:
        frame.advance(target_ms=TARGET_MS)
    frame.read()
    p = frame.progress
    conv = frame.convergence() if rule is not None else None
    return p.device_ms, p.passes, p.paths_done, p.pixels_flagged, (conv.pixels_converged if conv else 0)


def digest(frame, flags):
    _, sums = frame.read(want_sums=True)
    h = hashlib.sha256(sums.tobytes())
    if flags & NOISE:
        h.update(frame.noise(0.0, want_map=False, want_sq=True)[2].tobytes())
    return h.hexdigest()


def batch_once(h, cams, spec, seeds, flags=NOISE, rule=RULE):
    t0 = time.perf_counter()
    f = h.open_frame_views(cams, spec.max_width_coord, spec.max_height_coord, seeds=seeds, flags=flags)
    device, passes, paths, flagged, converged = drive(f, rule)
    wall = (time.perf_counter() - t0) * 1e3
    out = {"device_ms": device, "wall_ms": wall, "passes": passes, "paths": paths, "pixels_flagged": flagged,
           "pixels_converged": converged, "sums": digest(f, flags)}
    f.close()
    return out


def loop_once(h, cams, spec, seeds, flags=NOISE, rule=RULE):
    device, passes, paths, flagged, converged = 0.0, 0, 0, 0, 0
    frames, wall = [], 0.0
    for cam, seed in zip(cams, seeds):
        t0 = time.perf_counter()
        f = h.open_frame(cam, spec.max_width_coord, spec.max_height_coord, seed=seed, flags=flags)
        d, p, n, fl, c = drive(f, rule)
        wall += (time.perf_counter() - t0) * 1e3
        device, passes, paths, flagged, converged = device + d, passes + p, paths + n, flagged + fl, converged + c
        frames.append(f)
    hsh = hashlib.sha256()
    for f in frames:
        _, sums = f.read(want_sums=True)
        hsh.update(sums.tobytes())
    if flags & NOISE:
        for f in frames:
            hsh.update(f.noise(0.0, want_map=False, want_sq=True)[2].tobytes())
    for f in frames:
        f.close()
    # the batch's digest hashes the sums of every view, then Q of every view: the same bytes in the same order
    return {"device_ms": device, "wall_ms": wall, "passes": passes, "paths": paths, "pixels_flagged": flagged,
            "pixels_converged": converged, "sums": hsh.hexdigest()}


def summary(runs, key):
    xs = [r[key] for r in runs]
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


def compare(a_runs, b_runs, a, b):
    out = {}
    for key in ("device_ms", "wall_ms"):
        sa, sb = summary(a_runs, key), summary(b_runs, key)
        out[key] = {a: sa, b: sb, "gain_pct": 100.0 * (sb["median"] - sa["median"]) / sb["median"]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--rounds-scale", type=float, default=1.0, help="multiplies every workload's number of rounds")
    args = ap.parse_args()
    if native.device_count() < 1:
        raise SystemExit("views_progressive.py needs a CUDA device")
    doc = {"card": card(), "target_ms": TARGET_MS, "rule": {"tolerance": RULE[0], "min_samples": RULE[1], "interval": RULE[2]},
           "workloads": {}}
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
        w = {"views": n, "rows": spec.rows, "cols": spec.cols, "spp": spec.spp, "rounds": len(batch), "sums_and_q_equal": equal,
             "paths": batch[0]["paths"], "pixels_flagged": batch[0]["pixels_flagged"],
             "converged_fraction": batch[0]["pixels_converged"] / max(1, batch[0]["pixels_flagged"]),
             "passes": {"batch": batch[0]["passes"], "loop": loop[0]["passes"]}}
        w.update(compare(batch, loop, "batch", "loop"))
        if n == 64:  # the price of RT_FLAG_NOISE on the batch: no rule, with and without the flag
            batch_once(h, cams, spec, seeds, flags=0, rule=None)
            plain, flagged = [], []
            for _ in range(max(1, int(round(rounds * args.rounds_scale)))):
                plain.append(batch_once(h, cams, spec, seeds, flags=0, rule=None))
                flagged.append(batch_once(h, cams, spec, seeds, flags=NOISE, rule=None))
            price = compare(plain, flagged, "without_noise", "with_noise")
            for key in price:  # what the flag adds, in % of the time without it
                price[key].pop("gain_pct")
                p, f = price[key]["without_noise"]["median"], price[key]["with_noise"]["median"]
                price[key]["cost_pct"] = 100.0 * (f - p) / p
            price["passes"] = {"without_noise": plain[0]["passes"], "with_noise": flagged[0]["passes"]}
            w["noise_flag_price"] = price
        doc["workloads"][name] = w
        h.close()
        print(f"{name}: device {w['device_ms']['batch']['median']:.2f} vs {w['device_ms']['loop']['median']:.2f} ms "
              f"({w['device_ms']['gain_pct']:+.1f} %), wall {w['wall_ms']['batch']['median']:.2f} vs {w['wall_ms']['loop']['median']:.2f} ms "
              f"({w['wall_ms']['gain_pct']:+.1f} %), sums and Q equal: {equal}", file=sys.stderr)
        if not equal:
            raise SystemExit(f"{name}: the batch's sums or Q differ from the loop's")
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
