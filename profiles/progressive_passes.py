"""What rendering a frame in passes costs: the same frame through rt_render and through rt_frame_* (native.Frame) with
passes of about --target-ms of device time each, alternated in one process on one GPU.

Per config and form it reports the device time (rt_render: RtStats.kernel_ms, probe + main phase; a frame: the probe and
compaction plus every pass, RtFrameProgress.device_ms, both from CUDA events on the scene's stream), the host wall time of
the whole call (with the frame: rt_frame_begin, every rt_frame_advance, rt_frame_read), the number of passes, the overhead
against rt_render in % (medians over the rounds), and whether the final int32 sums are equal.  The card's name, power limit
and clock limit are read in the same run.  Writes one JSON document to stdout and, with --out, to that file.

  python profiles/progressive_passes.py --out /tmp/progressive_passes.json
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ray_tracing_fsharp_b200 import native, sample_images  # noqa: E402
from ray_tracing_fsharp_b200.domain import marshal  # noqa: E402
from ray_tracing_fsharp_b200.scene import Camera  # noqa: E402


def card():
    try:
        q = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                                    text=True, timeout=30).strip()
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "clocks_max_sm": clock}
    except Exception as e:  # the figures are then reported without a card, and say so
        return {"name": f"not read ({e})"}


def render_once(h, cam, spec, seed):
    t0 = time.perf_counter()
    rgb, sums, st = h.render(cam, spec.max_width_coord, spec.max_height_coord, seed=seed, want_sums=True)
    wall = (time.perf_counter() - t0) * 1e3
    return {"device_ms": st.kernel_ms, "wall_ms": wall, "passes": 1, "launches": st.launches, "paths": st.paths,
            "sums": hashlib.sha256(sums.tobytes()).hexdigest()}


def frame_once(h, cam, spec, seed, target_ms):
    t0 = time.perf_counter()
    with h.open_frame(cam, spec.max_width_coord, spec.max_height_coord, seed=seed) as f:
        p = f.progress
        passes_ms = []
        while not p.done:
            p = f.advance(target_ms=target_ms)
            passes_ms.append(p.last_pass_ms)
        rgb, sums = f.read(want_sums=True)
    wall = (time.perf_counter() - t0) * 1e3
    return {"device_ms": p.device_ms, "wall_ms": wall, "passes": p.passes, "paths": p.paths_done,
            "pass_ms": [round(x, 3) for x in passes_ms], "sums": hashlib.sha256(sums.tobytes()).hexdigest()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="C2,C4,C5")
    ap.add_argument("--target-ms", default="250,50")
    ap.add_argument("--rounds", default="C2:5,C4:5,C5:2", help="alternations per config")
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    targets = [float(x) for x in args.target_ms.split(",")]
    rounds = {k: int(v) for k, v in (x.split(":") for x in args.rounds.split(","))}
    doc = {"card": card(), "seed": args.seed, "configs": {}}
    for name in args.configs.split(","):
        spec = sample_images.CONFIGS[name]()
        cam = Camera.make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
        cam.bounce_depth = spec.bounce_depth
        hs, ts, keep = marshal(spec.objects)
        h = native.SceneHandle(hs, ts, 0, keepalive=keep)
        # warm-up of both forms (module load, launch attributes, allocations) on a cheap frame of the same extents
        wcam = type(cam).from_buffer_copy(cam)
        wcam.samples_per_pixel = 16
        render_once(h, wcam, spec, args.seed - 1)
        frame_once(h, wcam, spec, args.seed - 1, targets[0])
        forms = ["rt_render"] + [f"frame_{t:g}ms" for t in targets]
        runs = {f: [] for f in forms}
        for r in range(rounds.get(name, 3)):
            for f in (forms if r % 2 == 0 else forms[::-1]):  # alternate the order between rounds
                runs[f].append(render_once(h, cam, spec, args.seed) if f == "rt_render" else frame_once(h, cam, spec, args.seed, float(f[6:-2])))
                print(name, f, {k: v for k, v in runs[f][-1].items() if k not in ("sums", "pass_ms")}, file=sys.stderr, flush=True)
        base_dev = statistics.median(x["device_ms"] for x in runs["rt_render"])
        base_wall = statistics.median(x["wall_ms"] for x in runs["rt_render"])
        ref_sums = runs["rt_render"][0]["sums"]
        out = {"frame": f"{spec.cols}x{spec.rows}", "spp": spec.spp, "depth": spec.bounce_depth, "forms": {}}
        for f in forms:
            dev = statistics.median(x["device_ms"] for x in runs[f])
            wall = statistics.median(x["wall_ms"] for x in runs[f])
            out["forms"][f] = {
                "device_ms_median": round(dev, 3), "device_ms": [round(x["device_ms"], 3) for x in runs[f]],
                "wall_ms_median": round(wall, 3), "wall_ms": [round(x["wall_ms"], 3) for x in runs[f]],
                "passes": sorted({x["passes"] for x in runs[f]}),
                "overhead_device_pct": round(100.0 * (dev - base_dev) / base_dev, 3),
                "overhead_wall_pct": round(100.0 * (wall - base_wall) / base_wall, 3),
                "sums_equal_rt_render": all(x["sums"] == ref_sums for x in runs[f]),
                "paths": sorted({x["paths"] for x in runs[f]}),
            }
            if f != "rt_render":
                out["forms"][f]["pass_ms_last_run"] = runs[f][-1]["pass_ms"]
        doc["configs"][name] = out
        h.close()
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
