"""What a progressive frame over several GPUs costs (rt_multi_frame_begin, MultiHandle.open_frame), alternated in one process
with the forms it is compared with, on 1, 2, 4 and 8 GPUs (as many of those as are visible).

  c5_paced    C5 (100 k spheres, 3841 x 2161) at 4096 spp in passes of --target-ms against rt_multi_render at the same device
              count: device time (the frame's RtFrameProgress.device_ms against RtStats.kernel_ms, both the slowest device's
              CUDA-event spans), host wall time, passes, overhead %, and strong-scaling efficiency against the frame on one GPU.
  c5_noise    C5 at 1024 spp opened with RT_FLAG_NOISE under the rule tau = 1, m = k = 64 (passes of 64 sample indices, so
              every pass ends on a check) against the plain frame and the noise frame without a rule, driven in the same
              64-index passes: device-time ratios, and the time of the first check (the exchange, converge_kernel and the
              compaction: the first pass of the rule's frame minus the first pass of the noise frame, which trace the same
              samples).
  c2_paced    C2 (1201 x 801) at 500 spp in passes of --target-ms against rt_multi_render: one pass, so the overhead is the
              opener's and the synchronisations'.
  c5_denoise  Frame.denoise of the C5 frame after 64 spp, wall time of the call, which gathers the totals first.

Medians and the spread (min, max) over the rounds; in every round the final int32 sums of the compared forms must be equal
(recorded as "sums_equal").  The card's name, power limit and clock limit are read in the same run.  Writes one JSON
document to stdout and, with --out, to that file.

  python profiles/multi_progressive.py --out profiles/multi_progressive_b200.json
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
from ray_tracing_fsharp_b200 import abi, native, sample_images  # noqa: E402
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


def sha(a):
    return hashlib.sha256(a.tobytes()).hexdigest()


def camera(spec, spp):
    cam = Camera.make_basic(spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    cam.bounce_depth = spec.bounce_depth
    return cam


def render_once(m, spec, cam, seed):
    t0 = time.perf_counter()
    _, sums, st = m.render(cam, spec.max_width_coord, spec.max_height_coord, seed=seed, want_sums=True)
    return {"device_ms": st.kernel_ms, "wall_ms": (time.perf_counter() - t0) * 1e3, "passes": 1, "sums": sha(sums)}


def frame_once(m, spec, cam, seed, target_ms=0.0, max_samples=0, flags=0, rule=None, first_samples=0):
    t0 = time.perf_counter()
    with m.open_frame(cam, spec.max_width_coord, spec.max_height_coord, seed=seed, flags=flags) as f:
        if rule:
            f.set_convergence(*rule)
        p = f.progress
        probe_ms = p.device_ms
        pass_ms = []
        while not p.done:
            p = f.advance(max_samples=first_samples if first_samples and not pass_ms else max_samples, target_ms=target_ms)
            pass_ms.append(p.last_pass_ms)
        _, sums = f.read(want_sums=True)
        checks = f.convergence().checks if rule else 0
    return {"device_ms": p.device_ms, "wall_ms": (time.perf_counter() - t0) * 1e3, "passes": p.passes, "probe_ms": probe_ms,
            "pass_ms": [round(x, 3) for x in pass_ms], "checks": checks, "sums": sha(sums)}


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


def summarise(runs, keys=("device_ms", "wall_ms", "passes")):
    return {k: spread([r[k] for r in runs]) for k in keys}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worlds", default="1,2,4,8")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--target-ms", type=float, default=250.0)
    ap.add_argument("--c5-spp", type=int, default=4096)
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    n_dev = native.device_count()
    worlds = [w for w in (int(x) for x in args.worlds.split(",")) if w <= n_dev]
    doc = {"card": card(), "devices_visible": n_dev, "target_ms": args.target_ms, "rounds": args.rounds, "seed": args.seed, "results": {}}
    c5, c2 = sample_images.many_spheres(), sample_images.random_spheres()
    specs = {"C5": c5, "C2": c2}
    marshalled = {k: marshal(s.objects) for k, s in specs.items()}
    res = doc["results"]
    for w in worlds:
        handles = {k: native.MultiHandle(hs, ts, list(range(w)), keepalive=keep) for k, (hs, ts, keep) in marshalled.items()}
        m5, m2 = handles["C5"], handles["C2"]
        # warm-up of every form at a small sample count (modules, launch plans, buffers)
        for m, spec in ((m5, c5), (m2, c2)):
            render_once(m, spec, camera(spec, 16), args.seed)
            frame_once(m, spec, camera(spec, 16), args.seed, target_ms=args.target_ms, flags=abi.RT_FLAG_NOISE, rule=(1.0, 12, 2))
        r = res.setdefault(str(w), {})

        runs = {"render": [], "frame": []}
        equal = []
        cam = camera(c5, args.c5_spp)
        for _ in range(args.rounds):
            runs["render"].append(render_once(m5, c5, cam, args.seed))
            runs["frame"].append(frame_once(m5, c5, cam, args.seed, target_ms=args.target_ms))
            equal.append(runs["render"][-1]["sums"] == runs["frame"][-1]["sums"])
        dr, df = summarise(runs["render"]), summarise(runs["frame"])
        r["c5_paced"] = {"spp": args.c5_spp, "render": dr, "frame": df, "sums_equal": equal,
                         "overhead_device_pct": 100.0 * (df["device_ms"]["median"] / dr["device_ms"]["median"] - 1.0),
                         "overhead_wall_pct": 100.0 * (df["wall_ms"]["median"] / dr["wall_ms"]["median"] - 1.0),
                         "frame_pass_ms": runs["frame"][-1]["pass_ms"], "frame_probe_ms": runs["frame"][-1]["probe_ms"]}

        # the noise frame with the rule against the plain frame and against the noise frame without a rule, all in the same
        # windows: [n_probe, 64), then 64 indices a pass; the rule's first pass traces exactly what the noise frame's first pass
        # traces (no pixel stops before the first check), so their difference is the first check: the gather, converge_kernel
        # and the compaction
        runs = {"plain": [], "noise": [], "rule": []}
        equal = []
        cam = camera(c5, 1024)
        first = 64 - 11  # C5 at 1024 spp probes 11 sample indices
        for _ in range(args.rounds):
            runs["plain"].append(frame_once(m5, c5, cam, args.seed, max_samples=64, first_samples=first))
            runs["noise"].append(frame_once(m5, c5, cam, args.seed, max_samples=64, flags=abi.RT_FLAG_NOISE, first_samples=first))
            runs["rule"].append(frame_once(m5, c5, cam, args.seed, max_samples=64, flags=abi.RT_FLAG_NOISE, rule=(1.0, 64, 64)))
            # the rule stops pixels, so its sums differ from the other frames'; the noise frame's must equal the plain one's
            equal.append(runs["noise"][-1]["sums"] == runs["plain"][-1]["sums"] and runs["rule"][-1]["sums"] == runs["rule"][0]["sums"])
        dp, dn, dr = summarise(runs["plain"]), summarise(runs["noise"]), summarise(runs["rule"])
        first_check = [b["pass_ms"][0] - a["pass_ms"][0] for a, b in zip(runs["noise"], runs["rule"])]
        r["c5_noise"] = {"spp": 1024, "plain": dp, "noise": dn, "noise_rule": dr, "sums_equal": equal,
                         "checks": runs["rule"][-1]["checks"],
                         "rule_over_plain_device_ratio": dr["device_ms"]["median"] / dp["device_ms"]["median"],
                         "noise_over_plain_device_ratio": dn["device_ms"]["median"] / dp["device_ms"]["median"],
                         "first_check_ms": spread(first_check),
                         "rule_pass_ms": runs["rule"][-1]["pass_ms"], "noise_pass_ms": runs["noise"][-1]["pass_ms"]}

        runs = {"render": [], "frame": []}
        equal = []
        cam = camera(c2, 500)
        for _ in range(args.rounds + 1):
            runs["render"].append(render_once(m2, c2, cam, args.seed))
            runs["frame"].append(frame_once(m2, c2, cam, args.seed, target_ms=args.target_ms))
            equal.append(runs["render"][-1]["sums"] == runs["frame"][-1]["sums"])
        dr, df = summarise(runs["render"]), summarise(runs["frame"])
        r["c2_paced"] = {"spp": 500, "render": dr, "frame": df, "sums_equal": equal,
                         "overhead_device_pct": 100.0 * (df["device_ms"]["median"] / dr["device_ms"]["median"] - 1.0),
                         "overhead_wall_pct": 100.0 * (df["wall_ms"]["median"] / dr["wall_ms"]["median"] - 1.0)}

        with m5.open_frame(camera(c5, 64), c5.max_width_coord, c5.max_height_coord, seed=args.seed, flags=abi.RT_FLAG_NOISE) as f:
            f.advance()
            f.denoise()  # the features and the filter's buffers, computed once
            times = []
            for _ in range(3):  # the totals are gathered already: the filter alone
                t0 = time.perf_counter()
                f.denoise()
                times.append((time.perf_counter() - t0) * 1e3)
        with m5.open_frame(camera(c5, 64), c5.max_width_coord, c5.max_height_coord, seed=args.seed, flags=abi.RT_FLAG_NOISE) as f:
            f.features(4)
            f.advance()  # the totals are stale now: the next denoise gathers them first
            t0 = time.perf_counter()
            f.denoise()
            with_gather = (time.perf_counter() - t0) * 1e3
        r["c5_denoise"] = {"wall_ms_features_kept": spread(times), "wall_ms_with_gather": with_gather}
        for h in handles.values():
            h.close()
        print(json.dumps({w: r}), file=sys.stderr, flush=True)

    one = res.get("1", {}).get("c5_paced")
    if one:
        for w, r in res.items():
            r["c5_paced"]["strong_scaling_efficiency"] = one["frame"]["device_ms"]["median"] / (int(w) * r["c5_paced"]["frame"]["device_ms"]["median"])
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
