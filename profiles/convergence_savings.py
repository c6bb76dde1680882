"""What the convergence rule of progressive frames saves, what it costs, and what it does to the image.

Per config, in one process on one GPU, all frames progressive with RT_FLAG_NOISE and passes of about --target-ms:
  * the plain frame (no rule) and converging frames at each tolerance of --tolerances (min_samples = interval = 64):
    device time (RtFrameProgress.device_ms, CUDA events: probe and compaction plus every pass, checks included), paths,
    passes, the share of the flagged pixels that converged, the largest E over the flagged pixels at the end, and against a
    reference frame of another seed at 4x the samples (C5: --ref-spp) the RMS and the mean signed error of the per-pixel
    means (sum / count of each channel, 8-bit levels, before gamma) over the flagged pixels;
  * the price of the machinery: tau = 0 with the early-out (the flagged pixels' samples are never all equal, so nothing
    converges and the frame is the plain one) against the plain frame, alternated, medians over --rounds.
The card's name, power limit and clock limit are read in the same run.  Writes one JSON document to stdout and, with --out,
to that file.

  python profiles/convergence_savings.py --out /tmp/convergence_savings.json
"""
import argparse
import hashlib
import json
import os
import statistics
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ray_tracing_fsharp_b200 import abi, native, sample_images  # noqa: E402
from ray_tracing_fsharp_b200.domain import marshal  # noqa: E402
from ray_tracing_fsharp_b200.scene import Camera  # noqa: E402
from profiles.progressive_passes import card  # noqa: E402

NOISE = abi.RT_FLAG_NOISE


def frame_once(h, cam, spec, seed, target_ms, tol=None, keep=False):
    with h.open_frame(cam, spec.max_width_coord, spec.max_height_coord, seed=seed, flags=NOISE) as f:
        if tol is not None:
            f.set_convergence(tol, 64, 64)
        p = f.progress
        while not p.done:
            p = f.advance(target_ms=target_ms)
        _, sums = f.read(want_sums=True)
        out = {"device_ms": p.device_ms, "passes": p.passes, "paths": p.paths_done, "flagged": p.pixels_flagged,
               "sums": hashlib.sha256(sums.tobytes()).hexdigest()}
        if tol is not None:
            c = f.convergence()
            out.update(checks=c.checks, converged=c.pixels_converged)
        if keep:
            _, se, _ = f.noise(0.0)
            out.update(sums_array=sums.reshape(-1, 4), se=se.reshape(-1))
    return out


def means(sums):
    return sums[:, :3].astype(np.float64) / np.maximum(sums[:, 3:4], 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="C2,C4,C5")
    ap.add_argument("--spp", default="C5:1024", help="samples per pixel overriding a config's own")
    ap.add_argument("--ref-spp", default="C5:4096", help="the reference frame's samples per pixel (default 4x the frame's)")
    ap.add_argument("--tolerances", default="0.5,1,2")
    ap.add_argument("--target-ms", type=float, default=250.0)
    ap.add_argument("--rounds", default="C2:6,C4:4,C5:3", help="alternations of the tau = 0 / plain comparison per config")
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    rounds = {k: int(v) for k, v in (x.split(":") for x in args.rounds.split(","))}
    spp_of = {k: int(v) for k, v in (x.split(":") for x in args.spp.split(",") if x)}
    ref_spp_of = {k: int(v) for k, v in (x.split(":") for x in args.ref_spp.split(",") if x)}
    tols = [float(x) for x in args.tolerances.split(",")]
    doc = {"card": card(), "seed": args.seed, "target_ms": args.target_ms, "min_samples": 64, "interval": 64, "configs": {}}
    for name in args.configs.split(","):
        spec = sample_images.CONFIGS[name]()
        if name in spp_of:
            spec.spp = spp_of[name]
        cam = Camera.make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
        cam.bounce_depth = spec.bounce_depth
        hs, ts, keep = marshal(spec.objects)
        h = native.SceneHandle(hs, ts, 0, keepalive=keep)
        wcam = type(cam).from_buffer_copy(cam)
        wcam.samples_per_pixel = 128
        frame_once(h, wcam, spec, args.seed - 1, args.target_ms)  # warm-up: module load, allocations
        frame_once(h, wcam, spec, args.seed - 1, args.target_ms, tol=1.0)

        rcam = type(cam).from_buffer_copy(cam)
        rcam.samples_per_pixel = ref_spp_of.get(name, 4 * spec.spp)
        ref = frame_once(h, rcam, spec, args.seed + 1, args.target_ms, keep=True)
        ref_means = means(ref["sums_array"])
        del ref["sums_array"], ref["se"]

        out = {"frame": f"{spec.cols}x{spec.rows}", "spp": spec.spp, "reference_spp": rcam.samples_per_pixel,
               "reference_device_ms": round(ref["device_ms"], 3), "forms": {}}
        plain = frame_once(h, cam, spec, args.seed, args.target_ms, keep=True)
        flagged = plain["sums_array"][:, 3] == spec.spp
        forms = {"plain": plain}
        for tol in tols:
            forms[f"tau={tol:g}"] = frame_once(h, cam, spec, args.seed, args.target_ms, tol=tol, keep=True)
            print(name, tol, {k: v for k, v in forms[f"tau={tol:g}"].items() if k not in ("sums_array", "se")}, file=sys.stderr, flush=True)
        for key, r in forms.items():
            err = (means(r["sums_array"]) - ref_means)[flagged]
            out["forms"][key] = {
                "device_ms": round(r["device_ms"], 3), "device_vs_plain": round(r["device_ms"] / plain["device_ms"], 4),
                "paths": r["paths"], "paths_vs_plain": round(r["paths"] / plain["paths"], 4), "passes": r["passes"],
                "converged_fraction": round(r.get("converged", 0) / max(1, r["flagged"]), 4), "checks": r.get("checks", 0),
                "max_se_flagged": round(float(r["se"][flagged].max()), 4),
                "rms_error_flagged": round(float(np.sqrt((err * err).mean())), 4), "mean_signed_error_flagged": round(float(err.mean()), 5),
            }
        out["flagged_pixels"] = int(flagged.sum())

        # the price of the machinery: tau = 0 (nothing converges) against the plain frame, alternated
        runs = {"plain": [], "tau=0": []}
        for r in range(rounds.get(name, 3)):
            for f in (["plain", "tau=0"] if r % 2 == 0 else ["tau=0", "plain"]):
                runs[f].append(frame_once(h, cam, spec, args.seed, args.target_ms, tol=0.0 if f == "tau=0" else None))
        base = statistics.median(x["device_ms"] for x in runs["plain"])
        zero = statistics.median(x["device_ms"] for x in runs["tau=0"])
        out["machinery"] = {
            "plain_device_ms": [round(x["device_ms"], 3) for x in runs["plain"]],
            "tau0_device_ms": [round(x["device_ms"], 3) for x in runs["tau=0"]],
            "plain_passes": sorted({x["passes"] for x in runs["plain"]}), "tau0_passes": sorted({x["passes"] for x in runs["tau=0"]}),
            "tau0_checks": sorted({x["checks"] for x in runs["tau=0"]}), "tau0_converged": sorted({x["converged"] for x in runs["tau=0"]}),
            "overhead_device_pct": round(100.0 * (zero - base) / base, 3),
            "sums_equal": all(x["sums"] == runs["plain"][0]["sums"] for x in runs["plain"] + runs["tau=0"]),
        }
        print(name, out["machinery"], file=sys.stderr, flush=True)
        doc["configs"][name] = out
        h.close()
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
