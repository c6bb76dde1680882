"""What the noise estimate costs: the same progressive frame with and without RT_FLAG_NOISE (the render kernels that also
sum r^2 + g^2 + b^2 per pixel), alternated in one process on one GPU.

Per config and form it reports the device time of the whole frame (probe and compaction plus every pass,
RtFrameProgress.device_ms, CUDA events on the scene's stream), the passes, the overhead against the frame without the flag
in % (medians over the rounds), whether the final int32 sums are equal, and which kernel plan_launch picked for the probe and
for the passes (staged in shared memory or read from global memory, lean, walk stacks in shared memory, bytes of dynamic
shared memory: the RTFS_DEBUG_PLAN lines the library prints).  With the flag it also times rt_frame_noise (the estimate
and its summary over the frame, host wall time around the synchronous call).  The card's name, power limit and clock limit
are read in the same run.  Writes one JSON document to stdout and, with --out, to that file.

  python profiles/noise_overhead.py --out /tmp/noise_overhead.json
"""
import argparse
import contextlib
import hashlib
import json
import os
import statistics
import sys
import tempfile
import time

os.environ["RTFS_DEBUG_PLAN"] = "1"  # read once, by the first launch plan
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ray_tracing_fsharp_b200 import abi, native, sample_images  # noqa: E402
from ray_tracing_fsharp_b200.domain import marshal  # noqa: E402
from ray_tracing_fsharp_b200.scene import Camera  # noqa: E402
from profiles.progressive_passes import card  # noqa: E402


@contextlib.contextmanager
def captured_stderr(lines):
    """Collects what the library writes to file descriptor 2 meanwhile (one line per launch plan)."""
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+b") as tmp:
        os.dup2(tmp.fileno(), 2)
        try:
            yield
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            tmp.seek(0)
            lines.extend(tmp.read().decode("utf-8", "replace").splitlines())


def plans(lines):
    """{'probe': ..., 'main': ...}: the distinct kernel choices of the launch plans among `lines`."""
    out = {"probe": set(), "main": set()}
    for ln in lines:
        if not ln.startswith("rtfs: plan "):
            continue
        kv = dict(x.split("=") for x in ln[len("rtfs: plan "):].split())
        kind = "global" if kv["staged"] == "0" else ("staged lean" if kv["lean"] == "1" else "staged")
        if kind == "global":
            kind += (" wide" if kv["wide"] == "1" else "") + (" sstack" if kv["sstack"] == "1" else " local stack")
        out["probe" if kv["probe"] == "1" else "main"].add(f"{kind}, {kv['smem_bytes']} B shared, {kv['threads']} threads")
    return {k: sorted(v) for k, v in out.items()}


def frame_once(h, cam, spec, seed, target_ms, flags):
    lines = []
    with captured_stderr(lines):
        with h.open_frame(cam, spec.max_width_coord, spec.max_height_coord, seed=seed, flags=flags) as f:
            p = f.progress
            while not p.done:
                p = f.advance(target_ms=target_ms)
            _, sums = f.read(want_sums=True)
            noise_ms = []
            if flags & abi.RT_FLAG_NOISE:
                for _ in range(5):
                    t0 = time.perf_counter()
                    summary, _, _ = f.noise(1.0, want_map=False)
                    noise_ms.append((time.perf_counter() - t0) * 1e3)
    return {"device_ms": p.device_ms, "passes": p.passes, "paths": p.paths_done, "sums": hashlib.sha256(sums.tobytes()).hexdigest(),
            "plans": plans(lines), "noise_call_ms": statistics.median(noise_ms) if noise_ms else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="C2,C4,C5")
    ap.add_argument("--spp", default="C5:4096", help="samples per pixel overriding a config's own")
    ap.add_argument("--target-ms", type=float, default=250.0)
    ap.add_argument("--rounds", default="C2:6,C4:4,C5:2", help="alternations per config")
    ap.add_argument("--seed", type=int, default=2025)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    rounds = {k: int(v) for k, v in (x.split(":") for x in args.rounds.split(","))}
    spp_of = {k: int(v) for k, v in (x.split(":") for x in args.spp.split(",") if x)}
    doc = {"card": card(), "seed": args.seed, "target_ms": args.target_ms, "configs": {}}
    forms = {"plain": 0, "noise": abi.RT_FLAG_NOISE}
    for name in args.configs.split(","):
        spec = sample_images.CONFIGS[name]()
        if name in spp_of:
            spec.spp = spp_of[name]
        cam = Camera.make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
        cam.bounce_depth = spec.bounce_depth
        hs, ts, keep = marshal(spec.objects)
        h = native.SceneHandle(hs, ts, 0, keepalive=keep)
        # warm-up of both forms (module load, launch attributes, allocations) on a cheap frame of the same extents
        wcam = type(cam).from_buffer_copy(cam)
        wcam.samples_per_pixel = 16
        for flags in forms.values():
            frame_once(h, wcam, spec, args.seed - 1, args.target_ms, flags)
        runs = {f: [] for f in forms}
        for r in range(rounds.get(name, 3)):
            for f in (list(forms) if r % 2 == 0 else list(forms)[::-1]):  # alternate the order between rounds
                runs[f].append(frame_once(h, cam, spec, args.seed, args.target_ms, forms[f]))
                print(name, f, {k: v for k, v in runs[f][-1].items() if k != "sums"}, file=sys.stderr, flush=True)
        base = statistics.median(x["device_ms"] for x in runs["plain"])
        out = {"frame": f"{spec.cols}x{spec.rows}", "spp": spec.spp, "depth": spec.bounce_depth, "forms": {}}
        for f in forms:
            dev = statistics.median(x["device_ms"] for x in runs[f])
            out["forms"][f] = {
                "device_ms_median": round(dev, 3), "device_ms": [round(x["device_ms"], 3) for x in runs[f]],
                "passes": sorted({x["passes"] for x in runs[f]}),
                "overhead_device_pct": round(100.0 * (dev - base) / base, 3),
                "sums_equal_plain": all(x["sums"] == runs["plain"][0]["sums"] for x in runs[f]),
                "paths": sorted({x["paths"] for x in runs[f]}),
                "kernels": runs[f][-1]["plans"],
            }
            if f == "noise":
                out["forms"][f]["rt_frame_noise_ms_median"] = round(statistics.median(x["noise_call_ms"] for x in runs[f]), 3)
        doc["configs"][name] = out
        h.close()
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
