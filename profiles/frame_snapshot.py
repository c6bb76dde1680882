"""What saving and resuming a progressive frame costs (rt_frame_save, rt_frame_resume), and what checkpointing a long frame
costs against the same frame left alone.

Save and resume, for C2 (1201 x 801, 500 spp, RT_FLAG_NOISE, run to its end) and C5 (3841 x 2161, RT_FLAG_NOISE, after four
passes of 250 ms), with the caller's buffer pageable (np.empty) and pinned (rt_host_pin), alternated within every round:
  save_wall_ms     host clock around rt_frame_save (it returns with the snapshot in the buffer);
  resume_wall_ms   host clock around rt_frame_resume (header checks, the checksum over the whole buffer on the host, the
                   fingerprint, the allocation, the copy, the restore kernel, the compaction);
  resume_device_ms RtFrameProgress.device_ms of the resumed frame: the restore and the compaction on the device;
  pack_ms / unpack_ms  the device time of snapshot_pack_kernel and snapshot_unpack_kernel, from torch.profiler in a
                   separate, profiled round.
Checkpointing: C5 at 4096 spp (RT_FLAG_NOISE) in passes of 250 ms, saved into a pinned buffer every N passes, against the
same frame not saved, in the same process; wall times.  In every round the resumed frame's sums and Q, and the checkpointed
frame's final sums, must equal the uninterrupted frame's ("sums_equal").
The card's name, power limit and SM clock limit are read in the same run.  Writes one JSON document to stdout and, with
--out, to that file.

  python profiles/frame_snapshot.py --out profiles/frame_snapshot_b200.json
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ray_tracing_fsharp_b200 import abi, native, sample_images  # noqa: E402
from ray_tracing_fsharp_b200.domain import marshal  # noqa: E402
from profiles.multi_progressive import camera, card  # noqa: E402

NOISE = abi.RT_FLAG_NOISE
TARGET_MS = 250.0
CASES = {
    "C2 1201x801, 500 spp, noise, done": (lambda: sample_images.random_spheres(), 500, None),
    "C5 3841x2161, noise, after 4 passes of 250 ms": (lambda: sample_images.many_spheres(), 4096, 4),
}


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "n": len(xs)}


def open_frame(h, spec, spp, passes):
    f = h.open_frame(camera(spec, spp), spec.max_width_coord, spec.max_height_coord, seed=11, flags=NOISE)
    k = 0
    while not f.progress.done and (passes is None or k < passes):
        f.advance(target_ms=TARGET_MS)
        k += 1
    return f


def buffer(n, pinned):
    b = np.zeros(n, np.uint8)
    if pinned:
        native.check(native.lib().rt_host_pin(native.ptr(b), b.nbytes))
    return b


def save_resume(h, f, buf):
    lib = native.lib()
    n = C.c_size_t()
    t0 = time.perf_counter()
    native.check(lib.rt_frame_save(f.ptr, native.ptr(buf), buf.size, C.byref(n)))
    t1 = time.perf_counter()
    out, progress = C.c_void_p(), abi.RtFrameProgress()
    native.check(lib.rt_frame_resume(h.ptr, native.ptr(buf), n.value, C.byref(out), C.byref(progress)))
    t2 = time.perf_counter()
    r = native.Frame.__new__(native.Frame)
    r.scene, r.ptr, r.progress, r.rows, r.cols = h, out, progress, f.rows, f.cols
    with r:
        _, a = f.read(want_sums=True)
        _, b = r.read(want_sums=True)
        _, _, qa = f.noise(1.0, want_map=False, want_sq=True)
        _, _, qb = r.noise(1.0, want_map=False, want_sq=True)
    return {"save_wall_ms": 1e3 * (t1 - t0), "resume_wall_ms": 1e3 * (t2 - t1), "resume_device_ms": progress.device_ms, "bytes": n.value,
            "sums_equal": bool(np.array_equal(a, b) and np.array_equal(qa, qb))}


def kernel_times(h, f, buf):
    """Device time of the two snapshot kernels in one profiled save and resume (torch.profiler, CUDA activities)."""
    try:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            save_resume(h, f, buf)
        out = {}
        for e in prof.events():
            for key, name in (("pack_ms", "snapshot_pack_kernel"), ("unpack_ms", "snapshot_unpack_kernel")):
                if name in e.name:
                    us = getattr(e, "device_time", None)
                    out[key] = (us if us is not None else e.cuda_time) / 1e3
        return out or {"pack_ms": "not measured (no kernel events)", "unpack_ms": "not measured (no kernel events)"}
    except Exception as e:  # reported as not measured, with the reason
        return {"pack_ms": f"not measured ({e})", "unpack_ms": f"not measured ({e})"}


def checkpointing(h, spec, every, rounds):
    lib = native.lib()
    runs = {"unsaved": [], f"saved every {every} passes": []}
    equal = []
    for _ in range(rounds):
        finals = []
        for key in runs:
            f = h.open_frame(camera(spec, 4096), spec.max_width_coord, spec.max_height_coord, seed=11, flags=NOISE)
            with f:
                n = C.c_size_t()
                native.check(lib.rt_frame_save(f.ptr, None, 0, C.byref(n)))
                buf = buffer(n.value, True) if key != "unsaved" else None
                saves = 0
                t0 = time.perf_counter()
                while not f.progress.done:
                    f.advance(target_ms=TARGET_MS)
                    if buf is not None and f.progress.passes % every == 0:
                        native.check(lib.rt_frame_save(f.ptr, native.ptr(buf), buf.size, C.byref(n)))
                        saves += 1
                wall = 1e3 * (time.perf_counter() - t0)
                runs[key].append({"wall_ms": wall, "device_ms": f.progress.device_ms, "passes": f.progress.passes, "saves": saves})
                finals.append(f.read(want_sums=True)[1])
                if buf is not None:
                    lib.rt_host_unpin(native.ptr(buf))
        equal.append(bool(np.array_equal(finals[0], finals[1])))
    out = {k: {"wall_ms": spread([r["wall_ms"] for r in v]), "device_ms": spread([r["device_ms"] for r in v]), "passes": v[0]["passes"],
               "saves": v[0]["saves"]} for k, v in runs.items()}
    out["sums_equal"] = equal
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--every", type=int, default=10)
    ap.add_argument("--out")
    args = ap.parse_args()
    if native.device_count() < 1:
        raise SystemExit("frame_snapshot.py measures on a GPU; none is visible")
    doc = {"card": card(), "target_ms": TARGET_MS, "cases": {}}
    c5 = None
    for name, (make, spp, passes) in CASES.items():
        spec = make()
        hs, ts, keep = marshal(spec.objects)
        h = native.SceneHandle(hs, ts, 0, keepalive=keep)
        if name.startswith("C5"):
            c5 = (h, spec)
        with open_frame(h, spec, spp, passes) as f:
            n = C.c_size_t()
            native.check(native.lib().rt_frame_save(f.ptr, None, 0, C.byref(n)))
            bufs = {"pageable": buffer(n.value, False), "pinned": buffer(n.value, True)}
            save_resume(h, f, bufs["pinned"])  # warm-up
            rounds = {k: [] for k in bufs}
            for _ in range(args.rounds):
                for k, b in bufs.items():
                    rounds[k].append(save_resume(h, f, b))
            entry = {"bytes": n.value, "pixels": f.rows * f.cols, "samples_done": f.progress.samples_done}
            for k, rs in rounds.items():
                entry[k] = {m: spread([r[m] for r in rs]) for m in ("save_wall_ms", "resume_wall_ms", "resume_device_ms")}
                entry[k]["sums_equal"] = [r["sums_equal"] for r in rs]
            entry["kernels"] = kernel_times(h, f, bufs["pinned"])
            native.lib().rt_host_unpin(native.ptr(bufs["pinned"]))
        doc["cases"][name] = entry
    h, spec = c5
    doc["checkpointing"] = {"case": "C5 3841x2161, 4096 spp, noise, passes of 250 ms", **checkpointing(h, spec, args.every, max(1, args.rounds - 1))}
    doc["multi_gpu"] = "not measured: this script times one device"
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
