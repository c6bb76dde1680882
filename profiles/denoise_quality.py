"""What rt_frame_denoise buys and costs: error of raw and denoised progressive frames against a converged frame, and the device
time of the features and of the filter.

Workloads (full size): C2 (1201 x 801, RTOW spheres), C3 (1921 x 1081, the textured earth and planes), C4 (1921 x 1081, planes
and glass).  Every frame is progressive with RT_FLAG_NOISE and without the early-out, so every pixel holds the same samples.
  sweep     on each scene at 16 spp (seed 2025), the RMS error of the denoised image over a grid of options; the defaults of
            Frame.denoise (DESIGN.md section 19) are the options with the lowest error summed over the three scenes.
  quality   at 4, 16 and 64 spp (seed 2024), the RMS and mean signed error of the raw image (per-pixel means) and of the
            denoised one (linear_out, the defaults), both in 8-bit levels before gamma, over every pixel, against rt_render
            of another seed (7777) at 4096 spp (C4: 1024), without the early-out.
  equivalent the raw sample count whose error matches the denoised 16-spp image: raw errors of one frame advanced to 1, 2, 4,
            ... 1024 samples, interpolated in log(spp) between the two counts around the denoised error.
  timing    the device time of rt_frame_features (F = 4) and of rt_frame_denoise
            (no outputs copied), from torch.profiler's CUDA kernel records (features_kernel; denoise_input_kernel + atrous_kernel
            + denoise_output_kernel), on C2 at 16 spp and on C5 (3841 x 2161, 100 k spheres) at 4 spp; also the host clock
            around each call, which returns with its work complete.  The features are recomputed each time by asking for
            F = 3 and then F = 4; only the F = 4 launches are reported.
The card's name, power limit and clock limit are read in the same run.  Writes one JSON document to stdout and, with --out,
to that file.

  python profiles/denoise_quality.py --out profiles/denoise_quality_b200.json
"""
import argparse
import ctypes as C
import itertools
import json
import math
import os
import statistics
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ray_tracing_fsharp_b200 import abi, native, sample_images  # noqa: E402
from ray_tracing_fsharp_b200.domain import marshal  # noqa: E402
from profiles.progressive_passes import card  # noqa: E402

SEED, SWEEP_SEED, REF_SEED = 2024, 2025, 7777
GRID = dict(iterations=(3, 4, 5, 6), sigma_colour=(1.0, 2.0, 4.0, 8.0), sigma_normal=(0.1, 0.3, 1.0), sigma_albedo=(4.0, 16.0, 64.0),
            sigma_depth=(0.02, 0.1, 0.5))


def camera(spec, spp):
    cam = native.camera_make_basic(spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    cam.bounce_depth = spec.bounce_depth
    return cam


def means(sums):
    return sums[..., :3].astype(np.float64) / sums[..., 3:].astype(np.float64)


def errors(img, ref):
    d = img.astype(np.float64) - ref
    return {"rms": float(np.sqrt((d * d).mean())), "mean_signed": float(d.mean())}


def frame_at(h, spec, spp, seed):
    f = h.open_frame(camera(spec, spp), spec.max_width_coord, spec.max_height_coord, seed=seed, adaptive=False, flags=abi.RT_FLAG_NOISE)
    f.advance()
    return f


def kernel_records(fn, names, reps):
    """Per kernel named, the device times (ms) of its launches in `reps` calls of fn, in launch order (torch.profiler's CUDA
    records)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    recs = {n: [] for n in names}
    for ev in prof.events():
        for n in names:
            if n in ev.name and ev.device_type.name == "CUDA":
                recs[n].append((ev.time_range.start, ev.device_time / 1e3))
    return {n: [t for _, t in sorted(r)] for n, r in recs.items()}


def wall_ms(fn, reps):
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        out.append((time.perf_counter() - t0) * 1e3)
    return {"median": statistics.median(out), "min": min(out), "max": max(out)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    doc = {"card": card(), "grid": GRID, "scenes": {}}
    scenes = {"C2": (sample_images.random_spheres(), 4096), "C3": (sample_images.earth(), 4096), "C4": (sample_images.mixed_planes(), 1024)}
    handles, refs = {}, {}
    for name, (spec, ref_spp) in scenes.items():
        hs, ts, keep = marshal(spec.objects)
        h = handles[name] = native.SceneHandle(hs, ts, 0, keepalive=keep)
        _, s, _ = h.render(camera(spec, ref_spp), spec.max_width_coord, spec.max_height_coord, seed=REF_SEED, adaptive=False, want_sums=True)
        refs[name] = means(s)
        doc["scenes"][name] = {"rows": 2 * spec.max_height_coord + 1, "cols": 2 * spec.max_width_coord + 1, "reference_spp": ref_spp}

    # sweep: the options with the lowest summed RMS error at 16 spp
    keys = list(GRID)
    score = {}
    for name, (spec, _) in scenes.items():
        f = frame_at(handles[name], spec, 16, SWEEP_SEED)
        for combo in itertools.product(*[GRID[k] for k in keys]):
            o = dict(zip(keys, combo))
            _, lin = f.denoise(feature_samples=4, want_linear=True, **o)
            score[combo] = score.get(combo, 0.0) + errors(lin, refs[name])["rms"]
        f.close()
    best = dict(zip(keys, min(score, key=score.get)))
    best["feature_samples"] = 4
    doc["defaults"] = best
    doc["sweep_best_summed_rms"] = min(score.values())

    for name, (spec, _) in scenes.items():
        h, ref, out = handles[name], refs[name], doc["scenes"][name]
        out["quality"] = {}
        for spp in (4, 16, 64):
            f = frame_at(h, spec, spp, SEED)
            _, sums = f.read(want_sums=True)
            _, lin = f.denoise(want_linear=True, **best)
            out["quality"][str(spp)] = {"raw": errors(means(sums), ref), "denoised": errors(lin, ref)}
            f.close()
        # equivalent spp of the denoised 16-spp image
        target = out["quality"]["16"]["denoised"]["rms"]
        f = h.open_frame(camera(spec, 1024), spec.max_width_coord, spec.max_height_coord, seed=SEED, adaptive=False, flags=abi.RT_FLAG_NOISE)
        curve = []
        for spp in (1, 2, 4, 8, 16, 32, 64, 128, 256, 512, 1024):
            f.advance(max_samples=spp - f.progress.samples_done)
            curve.append((spp, errors(means(f.read(want_sums=True)[1]), ref)["rms"]))
        f.close()
        out["raw_rms_by_spp"] = {str(s): e for s, e in curve}
        eq = None
        for (s0, e0), (s1, e1) in zip(curve, curve[1:]):
            if e0 >= target >= e1:
                a = (e0 - target) / (e0 - e1) if e0 != e1 else 0.0
                eq = math.exp(math.log(s0) + a * (math.log(s1) - math.log(s0)))
                break
        out["equivalent_spp_of_denoised_16"] = eq if eq is not None else f"beyond {curve[-1][0]}" if target < curve[-1][1] else "below 1"

    # timing: C2 at 16 spp and C5 at 4 spp
    doc["timing"] = {}
    c5 = sample_images.many_spheres()
    hs, ts, keep = marshal(c5.objects)
    handles["C5"] = native.SceneHandle(hs, ts, 0, keepalive=keep)
    for name, spec, spp in (("C2", scenes["C2"][0], 16), ("C5", c5, 4)):
        f = frame_at(handles[name], spec, spp, SEED)
        opts = abi.RtDenoiseOpts(best["iterations"], 4, best["sigma_colour"], best["sigma_normal"], best["sigma_albedo"],
                                 best["sigma_depth"], 0, 0)

        def features():  # F = 3, then F = 4: both are computed afresh
            f.features(3)
            f.features(4)

        def denoise():  # the filter alone: no output copied
            native.check(native.lib().rt_frame_denoise(f.ptr, C.byref(opts), None, None))

        feat = kernel_records(features, ["features_kernel"], args.reps)["features_kernel"]
        f.features(4)
        den = kernel_records(denoise, ["denoise_input_kernel", "atrous_kernel", "denoise_output_kernel"], args.reps)
        f4 = feat[1::2]  # every second launch is F = 4
        filt = {k: sum(v) / args.reps for k, v in den.items()}
        doc["timing"][name] = {
            "pixels": int(f.rows * f.cols), "spp": spp, "frame_device_ms": f.progress.device_ms,
            "features_f4_ms": {"median": statistics.median(f4), "min": min(f4), "max": max(f4)},
            "filter_ms_per_call": sum(filt.values()), "filter_kernels_ms_per_call": filt,
            "atrous_levels_per_call": len(den["atrous_kernel"]) / args.reps,
            "features_f3_then_f4_call_wall_ms": wall_ms(features, args.reps),
            "denoise_call_wall_ms": wall_ms(denoise, args.reps),
        }
        f.close()
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
