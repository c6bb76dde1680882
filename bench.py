#!/usr/bin/env python
"""bench.py — Mrays/s and Mpaths/s of the render path on the RTOW final scene (BASELINE.json configs[1]).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, sm_100a)
    python bench.py --impl reference --gpus N ...            # the CPU arm: C++ restatement of the F# algorithm

A step is one frame: Scene.render of the C2 scene (1201x801, 500 spp, depth 50, adaptive early-out as the
reference does it).  Every frame is one library call, rt_comm_render: probe + [all-reduce of flags] + compact +
main + [reduce-scatter of sums] + finalize + [all-gather of RGB8], kernels and NCCL collectives enqueued by
librtfs_b200.so on the stream bench.py hands it.  `value` times the device-resident frame with CUDA events on that
stream, L2 flushed between steps, max over ranks.  `e2e` times the public API with host buffers: Scene.make
(marshal + BVH build + host->device upload) + Scene.render + Image.render (device->host image).  The line also
carries: `roofline` (SURVEY 8d's algorithmic FLOPs of the reference traversal) and `roofline_useful` (the tests our
traversal executed), `traversal`, `frame_sha256` (one fixed-seed frame hashed through every product path: equal
for every N), `other_configs` (C1, C3, C4, the author's native 2401x1601 depth-150 frame, C5 at its full 4096 spp),
`cpu_baseline`.  Prints ONE JSON line on rank 0.

`--dump-outputs DIR` writes the frame the last timed step left in device memory as DIR/rgb.npy (RGB8, float32) and, with one
rank, DIR/sums.npy (the int32 PixelStats sums, float64), so that two builds can be compared output for output: the scene and
the seeds depend only on the arguments.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the checkout may be read-only: nothing is written into it

import numpy as np  # noqa: E402

# FLOPs of the reference algorithm per ray (SURVEY.md §8d): 3 (inverse directions) + 12 per slab test +
# 20 per sphere test + 14 per plane test + 1 per candidate + 6 (strike point)
def flops_per_ray(c):
    rays = max(1, c["rays"])
    return 3.0 + 12.0 * c["box_tests"] / rays + 20.0 * c["sphere_tests"] / rays + 14.0 * c["plane_tests"] / rays + c["candidates"] / rays + 6.0


# the same figure per config, measured by the oracle (DESIGN.md §3); used when the CPU sample does not run (N > 1)
FLOPS_PER_RAY = {"C1": 96.0, "C2": 414.0, "C3": 75.0, "C4": 131.0, "C5": 1927.0}


def metric_name(spec, config):
    if config == "C2":
        return "Mrays/s, RTOW final scene 1201x801 500spp depth 50 (Mpaths/s alongside)"
    return f"Mrays/s, {spec.name}, {spec.cols}x{spec.rows} {spec.spp}spp depth {spec.bounce_depth} (Mpaths/s alongside)"


def build_spec(args):
    from ray_tracing_fsharp_b200 import sample_images
    fn = sample_images.CONFIGS[args.config]
    spec = fn()
    if args.spp:
        spec.spp = args.spp
    if args.half_extents:
        spec.max_width_coord, spec.max_height_coord = args.half_extents
    return spec


def workload_name(spec, adaptive):
    return (f"{spec.name}, {spec.cols}x{spec.rows}, {spec.spp} spp, depth {spec.bounce_depth}, "
            f"adaptive early-out {'on (Scene.fs:157-194)' if adaptive else 'off'}")


# ---------------------------------------------------------------------------------------------------
# CPU arm: the oracle (C++ restatement of the F# algorithm), all host threads, bounded sample
# ---------------------------------------------------------------------------------------------------
def cpu_sample(spec, target_seconds, threads, seed=7):
    """Renders every `row_step`-th row of the frame at full spp with the oracle, sized for ~target_seconds."""
    import oracle
    from ray_tracing_fsharp_b200.domain import marshal
    hs, ts, _keep = marshal(spec.objects)
    scene = oracle.Scene(hs, ts)
    cam = oracle.camera_make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    cam.bounce_depth = spec.bounce_depth
    # calibrate on a few rows spread over the frame, at no more than 64 spp (a row of the 100 k-sphere frame at 4096 spp
    # takes the host cores 20 s); the time of a row is at most linear in spp beyond that
    step0 = max(1, spec.rows // 8)
    spp_cal = min(spec.spp, 64)
    cam_cal = oracle.camera_make_basic(spp_cal, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    cam_cal.bounce_depth = spec.bounce_depth
    t0 = time.perf_counter()
    _, _, c0, rows0 = scene.render(cam_cal, spec.max_width_coord, spec.max_height_coord, seed=seed, rng_mode=0, adaptive=True, threads=threads,
                                   row_begin=step0 // 2, row_step=step0)
    dt0 = time.perf_counter() - t0
    per_row = dt0 / max(1, rows0) * (spec.spp / spp_cal)
    n_rows = int(min(spec.rows, max(1, target_seconds / max(per_row, 1e-9))))
    row_step = max(1, spec.rows // max(1, n_rows))
    t0 = time.perf_counter()
    _, _, c, rows = scene.render(cam, spec.max_width_coord, spec.max_height_coord, seed=seed + 1, rng_mode=0, adaptive=True, threads=threads,
                                 row_begin=row_step // 2, row_step=row_step)
    dt = time.perf_counter() - t0
    return {"seconds": dt, "rows": rows, "row_step": row_step, "counters": c}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    spec = build_spec(args)
    threads = os.cpu_count() or 1
    per_step = []
    counters = None
    rows = row_step = 0
    # every step is a bounded sample of the frame; size it so that the whole run stays within a couple of minutes
    per_step_seconds = min(args.cpu_seconds, 120.0 / max(1, args.warmup + args.steps))
    for i in range(args.warmup + args.steps):
        s = cpu_sample(spec, per_step_seconds, threads, seed=100 + i)
        if i >= args.warmup:
            per_step.append(s)
        counters, rows, row_step = s["counters"], s["rows"], s["row_step"]
    secs = sum(s["seconds"] for s in per_step)
    rays = sum(s["counters"]["rays"] for s in per_step)
    paths = sum(s["counters"]["paths"] for s in per_step)
    mrays = rays / secs / 1e6
    sample = f"every {row_step}th row of the frame ({rows} of {spec.rows} rows) at full spp per step"
    line = {
        "impl": "reference",
        "metric": metric_name(spec, args.config),
        "note": "CPU arm = the oracle, a C++ restatement of the F# CPU renderer, row-parallel on all host threads (.NET is absent from this image)",
        "value": mrays, "unit": "Mrays/s", "mpaths_per_s": paths / secs / 1e6,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / max(1, len(per_step)),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(spec, True), "sample": sample},
        "cpu_baseline": {"value": mrays, "unit": "Mrays/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": mrays, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "flops_per_ray_reference_algorithm": flops_per_ray(counters),
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.perf_counter(), line.strip()))

    def stop(self, t_begin, t_end):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, line in self.samples:
            if t < t_begin or t > t_end + 0.1:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def executed_flops_per_ray(c, n_planes):
    """SURVEY 8d's formula on the tests OUR traversal executed (RT_FLAG_COUNTERS): every ray tests every unbounded
    object, so `n_planes` of the primitive tests per ray are plane tests (14 FLOP) and the rest sphere tests (20)."""
    rays = max(1, c["rays"])
    prim = c["prim_tests"] / rays
    return 3.0 + 12.0 * c["box_tests"] / rays + 20.0 * max(0.0, prim - n_planes) + 14.0 * n_planes + 1.0 + 6.0


class Runner:
    """One rank of the job: torch for the stream, the events, the barrier and the max-over-ranks; every frame is ONE
    library call, rt_comm_render (kernels + NCCL collectives enqueued by librtfs_b200.so on the stream it is given)."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from ray_tracing_fsharp_b200 import native
        from ray_tracing_fsharp_b200.distributed import comm_from_torch_distributed
        self.torch, self.dist, self.native, self.args = torch, dist, native, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if native.device_count() < 1:
            raise RuntimeError("bench.py needs a CUDA device: the product path has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.ctl = None
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
            self.ctl = dist.new_group(backend="gloo")  # host-side barrier for the phases where rank 0 drives every GPU itself
        # a stream of our own, made current: the legacy default stream's handle is NULL, which the library reads as "use your own"
        self.stream = torch.cuda.Stream(self.dev)
        torch.cuda.set_stream(self.stream)
        self.comm = comm_from_torch_distributed(self.local_rank, self.stream.cuda_stream)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)  # > 126 MB L2
        self.adaptive = not args.no_adaptive
        self.flags = 0  # RtRenderOpts.flags of every frame

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def host_barrier(self):
        self.torch.cuda.synchronize(self.dev)
        if self.world > 1:
            self.dist.barrier(group=self.ctl)

    def reduce(self, values, op):
        t = self.torch.tensor(values, dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=getattr(self.dist.ReduceOp, op))
        return [float(x) for x in t.tolist()]

    def scene(self, spec):
        from ray_tracing_fsharp_b200.domain import marshal
        from ray_tracing_fsharp_b200.scene import Camera
        hs, ts, keep = marshal(spec.objects)
        handle = self.native.SceneHandle(hs, ts, self.local_rank, keepalive=keep)
        cam = Camera.make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
        cam.bounce_depth = spec.bounce_depth
        return handle, cam

    def enqueue(self, handle, cam, spec, seed, flags=None):
        """One device-resident frame: nothing crosses PCIe, nothing synchronises."""
        self.comm.render(handle, cam, spec.max_width_coord, spec.max_height_coord, seed=seed, adaptive=self.adaptive,
                         flags=self.flags if flags is None else flags, want_rgb=False, want_sums=False, want_stats=False)

    def measure(self, handle, cam, spec, steps, warmup, seed0=2000):
        """W untimed frames, then K timed ones: L2 flushed, barrier + synchronize on both sides, CUDA events on the stream the
        library enqueues on, max over ranks.  Returns whole-job totals plus rank 0's main-phase kernel figures."""
        torch = self.torch
        for i in range(warmup):
            self.enqueue(handle, cam, spec, seed0 - 1000 + i)
        self.barrier()
        out = {"ms": 0.0, "rays": 0, "paths": 0, "launches": 0, "main_ms": [], "main_rays": [], "degenerate": 0, "last_seed": seed0 + steps - 1}
        for i in range(steps):
            self.flush.fill_(i & 0xFF)
            self.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(self.stream)
            self.enqueue(handle, cam, spec, seed0 + i)
            e1.record(self.stream)
            self.barrier()
            st = self.comm.last_stats(handle)  # this rank's counters and the events the library recorded around its kernels
            ms, = self.reduce([e0.elapsed_time(e1)], "MAX")
            rays, paths, launches, degenerate = self.reduce([st.rays, st.paths, st.launches, st.degenerate_paths], "SUM")
            out["ms"] += ms
            out["rays"] += int(rays)
            out["paths"] += int(paths)
            out["launches"] += int(launches)
            out["degenerate"] += int(degenerate)
            out["main_ms"].append(st.main_ms)
            out["main_rays"].append(int(st.main_rays))
        return out

    def device_frame(self, spec):
        """The frame the last rt_comm_render left in device memory, copied to the host: RGB8 [rows, cols, 3] and, where this
        rank holds all of them (one rank), the int32 PixelStats sums [rows, cols, 4].  Call after synchronising."""
        d_rgb, d_sums = self.comm.frame_pointers()
        host = lambda a: self.torch.as_tensor(a, device=self.dev).cpu().numpy()  # noqa: E731
        rgb = host(DeviceArray(d_rgb, (spec.rows, spec.cols, 3), "|u1"))
        sums = host(DeviceArray(d_sums, (spec.rows, spec.cols, 4), "<i4")) if self.world == 1 else None
        return rgb, sums

    def counters(self, handle, cam, spec, seed=4000):
        """One untimed frame with RT_FLAG_COUNTERS (a slower kernel variant): the tests OUR traversal executes."""
        from ray_tracing_fsharp_b200 import abi
        _, _, st = self.comm.render(handle, cam, spec.max_width_coord, spec.max_height_coord, seed=seed, adaptive=self.adaptive,
                                    flags=self.flags | abi.RT_FLAG_COUNTERS, want_rgb=False, want_sums=False, want_stats=True)
        rays, paths, box, prim = self.reduce([st.rays, st.paths, st.box_tests, st.prim_tests], "SUM")
        return {"rays": rays, "paths": paths, "box_tests": box, "prim_tests": prim}


class DeviceArray:
    """A buffer in device memory that the library owns, described by __cuda_array_interface__ so that torch can read it."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"data": (ptr, False), "shape": shape, "typestr": typestr, "version": 2}


DUMP_BYTES = 64_000_000  # all files together, .npy headers included


def dump_outputs(out_dir, rgb, sums, seed=0):
    """Writes the frame as out_dir/rgb.npy (float32) and out_dir/sums.npy (float64; omitted when None), both exact.  A frame
    larger than DUMP_BYTES in all is cut to a fixed, seeded sample of its pixels ([n, 3] / [n, 4]), whose flat indices go to
    out_dir/pixel_index.npy.  Returns {file name: shape}."""
    arrays = {"rgb": rgb.astype(np.float32)}
    if sums is not None:
        arrays["sums"] = sums.astype(np.float64)
    n_pixels = rgb.shape[0] * rgb.shape[1]
    per_pixel = sum(a.nbytes for a in arrays.values()) // n_pixels
    budget = DUMP_BYTES - 1024  # a .npy header is 128 bytes
    if n_pixels * per_pixel > budget:
        keep = budget // (per_pixel + 8)
        idx = np.sort(np.random.default_rng(seed).choice(n_pixels, keep, replace=False))
        arrays = {k: a.reshape(n_pixels, -1)[idx] for k, a in arrays.items()}
        arrays["pixel_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
    return {f"{name}.npy": list(a.shape) for name, a in arrays.items()}


def n_planes_of(spec):
    from ray_tracing_fsharp_b200.domain import Hittable
    return sum(1 for o in spec.objects if isinstance(o, Hittable.InfinitePlane))


def frame_hashes(r, handle, cam, spec, seed=424242):
    """One extra untimed frame with a fixed seed through every product path; SHA-256 of the RGB8 frame and of the int32
    PixelStats sums.  Equal hashes across N = 1, 2, 4, 8 and across the paths are the multi-GPU correctness evidence."""
    import hashlib
    from ray_tracing_fsharp_b200 import native
    mw, mh = spec.max_width_coord, spec.max_height_coord
    sha = lambda a: hashlib.sha256(a.tobytes()).hexdigest()  # noqa: E731
    paths = {}
    rgb, sums, _ = r.comm.render(handle, cam, mw, mh, seed=seed, adaptive=r.adaptive, flags=r.flags, want_rgb=True, want_sums=True)
    ref_rgb, ref_sums = sha(rgb), sha(sums)
    paths["rt_comm_render, sums all-reduced"] = ref_rgb
    rgb2, _, _ = r.comm.render(handle, cam, mw, mh, seed=seed, adaptive=r.adaptive, flags=r.flags, want_rgb=True, want_sums=False)
    paths["rt_comm_render, sums reduce-scattered + RGB8 all-gathered"] = sha(rgb2)
    out = {"seed": seed, "rgb8": ref_rgb, "sums_int32": ref_sums}
    r.host_barrier()
    if r.rank == 0:
        if r.world == 1:
            rgb3, sums3, _ = handle.render(cam, mw, mh, seed=seed, adaptive=r.adaptive, flags=r.flags, want_sums=True)
            paths["rt_render"] = sha(rgb3)
            out["sums_int32_rt_render"] = sha(sums3)
        elif native.device_count() >= r.world:
            # one process (this one) driving all N devices through peer memory: what a single F# host process would call
            from ray_tracing_fsharp_b200.domain import marshal
            hs, ts, keep = marshal(spec.objects)
            multi = native.MultiHandle(hs, ts, list(range(r.world)), keepalive=keep)
            multi.render(cam, mw, mh, seed=seed - 1, adaptive=r.adaptive, flags=r.flags)  # first use: allocations
            t0 = time.perf_counter()
            rgb3, sums3, st3 = multi.render(cam, mw, mh, seed=seed, adaptive=r.adaptive, flags=r.flags, want_sums=True)
            wall = time.perf_counter() - t0
            paths["rt_multi_render (one process, peer memory)"] = sha(rgb3)
            out["sums_int32_rt_multi_render"] = sha(sums3)
            out["rt_multi_render"] = {"device_ms": st3.kernel_ms, "wall_ms_with_sums_copy": 1e3 * wall, "rays": int(st3.rays), "devices": r.world}
            t0 = time.perf_counter()
            rgb4, _, st4 = multi.render(cam, mw, mh, seed=seed, adaptive=r.adaptive, flags=r.flags)  # the call a host makes: frame into a host buffer
            wall = time.perf_counter() - t0
            out["rt_multi_render"].update({"wall_ms": 1e3 * wall, "mrays_per_s_wall": st4.rays / wall / 1e6})
            paths["rt_multi_render, second call"] = sha(rgb4)
            multi.close()
    r.host_barrier()
    out["paths"] = paths
    out["all_paths_equal"] = len(set(paths.values())) == 1 and all(out.get(k, ref_sums) == ref_sums for k in ("sums_int32_rt_render", "sums_int32_rt_multi_render"))
    return out


def e2e_frames(r, spec, cam, n_e2e):
    """The public API with HOST buffers, every step: Scene.make (marshal + BVH build + host->device upload of the scene) +
    Scene.render + Image.render (kernels, collectives, device->host copy of the frame).  Wall clock, max over ranks."""
    from ray_tracing_fsharp_b200 import native
    from ray_tracing_fsharp_b200.domain import marshal
    from ray_tracing_fsharp_b200.scene import Image, Scene
    mw, mh = spec.max_width_coord, spec.max_height_coord
    secs, rays_total, h2d, d2h = 0.0, 0, 0, 0
    ring = native.FrameRing((spec.rows, spec.cols, 3), count=2)  # the host's own two frame arrays, reused explicitly
    for i in range(-2, n_e2e):  # two untimed iterations: first-use allocations (the library's handle pool)
        r.barrier()
        t0 = time.perf_counter()
        if r.world == 1:
            sc = Scene.make(spec.objects, device=r.local_rank)
            _, image = Scene.render(lambda _p: None, lambda _s: None, mw, mh, cam, sc, seed=3000 + i, adaptive=r.adaptive, flags=r.flags, frames=ring)
            pixels = Image.render(image)
            rays = sc.last_stats.rays
            h2d = sc.handle.device_bytes()
            d2h = pixels.nbytes + 128
            sc.handle.close()
        else:
            hs, ts, keep = marshal(spec.objects)
            sc = native.SceneHandle(hs, ts, r.local_rank, keepalive=keep)
            rgb, _, st = r.comm.render(sc, cam, mw, mh, seed=3000 + i, adaptive=r.adaptive, flags=r.flags, want_rgb=(r.rank == 0), want_stats=True,
                                       rgb_out=ring.next() if r.rank == 0 else None)
            rays = st.rays
            h2d = sc.device_bytes()
            d2h = (rgb.nbytes if rgb is not None else 0) + 128
            sc.close()
        own = time.perf_counter() - t0  # this rank's wall time from the common start; the collectives inside the frame tie the ranks together
        r.barrier()
        dt, = r.reduce([own], "MAX")
        rr, h2d_all, d2h_all = r.reduce([rays, h2d, d2h], "SUM")
        if i >= 0:
            secs += dt
            rays_total += int(rr)
    return {"secs": secs, "rays": rays_total, "h2d": int(h2d_all), "d2h": int(d2h_all)}


def other_config_specs(args):
    from ray_tracing_fsharp_b200 import sample_images
    out = []
    for name in args.other_configs.split(","):
        name = name.strip()
        if not name or name == args.config:
            continue
        if name == "native":
            # the author's own workload: randomSpheres at (1200, 800) half-extents, BounceDepth 150 as Camera.makeBasic sets it
            # (RayTracing.App/SampleImages.fs:818-827, :960; Camera.fs:58)
            spec = sample_images.random_spheres(max_w=1200, max_h=800, spp=500, depth=150)
            spec.name = "RTOW final scene at the author's native size (random-spheres)"
            out.append((name, spec, "C2", 2))
        else:
            out.append((name, sample_images.CONFIGS[name](), name, 1 if name == "C5" else 3))
    return out


def run_ours(args):
    from ray_tracing_fsharp_b200 import abi, native
    r = Runner(args)
    torch, rank, world = r.torch, r.rank, r.world
    r.flags = ((abi.RT_FLAG_NO_SMEM if args.no_smem else 0) | {"auto": 0, "binary": abi.RT_FLAG_BVH2, "wide": abi.RT_FLAG_WIDE_BVH}[args.bvh]
               | (abi.RT_FLAG_FLOW if args.schedule == "flow" else 0) | (abi.RT_FLAG_NO_LEAN if args.no_lean else 0))
    spec = build_spec(args)
    handle, cam = r.scene(spec)
    fp32_peak = native.measure_fp32_peak(r.local_rank) if rank == 0 else 0.0

    sampler = ClockSampler(r.local_rank)
    for i in range(args.warmup):  # warm-up outside the clock window
        r.enqueue(handle, cam, spec, 1000 + i)
    r.barrier()
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    t_begin = time.perf_counter()
    m = r.measure(handle, cam, spec, args.steps, 0)
    t_end = time.perf_counter()
    clocks = sampler.stop(t_begin, t_end) if rank == 0 else None
    secs = m["ms"] / 1e3
    value = m["rays"] / secs / 1e6
    main_ms = sum(m["main_ms"]) / max(1, len(m["main_ms"]))
    main_rays = sum(m["main_rays"]) / max(1, len(m["main_rays"]))
    dumped = None
    if args.dump_outputs and rank == 0:  # before the next rt_comm_render replaces the frame
        dumped = {"dir": os.path.abspath(args.dump_outputs), "frame_seed": m["last_seed"],
                  "files": dump_outputs(args.dump_outputs, *r.device_frame(spec))}

    n_e2e = max(1, min(args.steps, 3))
    e2e = e2e_frames(r, spec, cam, n_e2e)
    trav = r.counters(handle, cam, spec)
    hashes = frame_hashes(r, handle, cam, spec) if not args.no_hash else None

    # ---- the other BASELINE configs (and the author's native frame), each a short measurement of its own ----
    others = {}
    for name, ospec, fkey, osteps in ([] if args.no_other_configs else other_config_specs(args)):
        oh, ocam = r.scene(ospec)
        if name == "C5":  # a full-spp warm-up frame would cost as much as the measurement: warm up on a 16-spp frame
            wcam = type(ocam).from_buffer_copy(ocam)
            wcam.samples_per_pixel = 16
            r.enqueue(oh, wcam, ospec, 900)
            r.barrier()
            om = r.measure(oh, ocam, ospec, osteps, 0, seed0=5000)
        else:
            om = r.measure(oh, ocam, ospec, osteps, 1, seed0=5000)
        oc = r.counters(oh, ocam, ospec) if name != "C5" else None
        o_main_ms = sum(om["main_ms"]) / len(om["main_ms"])
        o_main_rays = sum(om["main_rays"]) / len(om["main_rays"])
        f_ref = FLOPS_PER_RAY[fkey]
        entry = {"workload": workload_name(ospec, r.adaptive), "steps": osteps, "ms_per_step": om["ms"] / osteps,
                 "mrays_per_s": om["rays"] / (om["ms"] / 1e3) / 1e6, "mpaths_per_s": om["paths"] / (om["ms"] / 1e3) / 1e6,
                 "rays_per_step": om["rays"] / osteps, "main_kernel_ms": o_main_ms,
                 "flops_per_ray_reference_algorithm": f_ref,
                 "frac": (o_main_rays / (o_main_ms / 1e3) * f_ref / 1e12 / fp32_peak) if (rank == 0 and fp32_peak and o_main_ms > 0) else None,
                 "scene_bytes_staged_in_shared_memory": oh.shared_memory_bytes()}
        if oc:
            f_exec = executed_flops_per_ray(oc, n_planes_of(ospec))
            entry["traversal"] = {"box_tests_per_ray": oc["box_tests"] / max(1, oc["rays"]), "prim_tests_per_ray": oc["prim_tests"] / max(1, oc["rays"])}
            entry["frac_executed_tests"] = (o_main_rays / (o_main_ms / 1e3) * f_exec / 1e12 / fp32_peak) if (rank == 0 and fp32_peak and o_main_ms > 0) else None
        others[name] = entry
        oh.close()

    peer_memory = r.comm.uses_peer_memory()
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            s = cpu_sample(spec, args.cpu_seconds, threads)
            cpu = {"value": s["counters"]["rays"] / s["seconds"] / 1e6, "unit": "Mrays/s", "cores": threads, "kind": "port",
                   "sample": f"every {s['row_step']}th row of the frame ({s['rows']} of {spec.rows} rows) at full spp, {s['seconds']:.1f} s",
                   "mpaths_per_s": s["counters"]["paths"] / s["seconds"] / 1e6, "counters": s["counters"]}
        # algorithmic FLOPs per ray of the REFERENCE traversal on this scene (SURVEY 8d): measured by the oracle on the CPU
        # sample when it ran, else the figure recorded in DESIGN.md for the config
        f_ray = flops_per_ray(cpu["counters"]) if cpu else (args.flops_per_ray or FLOPS_PER_RAY[args.config])
        f_exec = executed_flops_per_ray(trav, n_planes_of(spec))
        rate = main_rays / (main_ms / 1e3) if main_ms > 0 else 0.0
        achieved, achieved_exec = rate * f_ray / 1e12, rate * f_exec / 1e12
        traffic = l2_per_ray = hbm_per_ray = None
        tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tp) and args.config == "C2" and not args.spp and not args.half_extents:  # the ncu capture is of the C2 main kernel
            try:
                tj = json.load(open(tp))
                traffic = tj.get("dram_bytes_per_launch")
                if tj.get("rays_per_launch"):
                    hbm_per_ray = tj["dram_bytes_per_launch"] / tj["rays_per_launch"]
                    l2_per_ray = tj.get("l2_bytes_per_launch", 0) / tj["rays_per_launch"] or None
            except Exception:
                traffic = None
        line = {
            "metric": metric_name(spec, args.config),
            "value": value, "unit": "Mrays/s", "mpaths_per_s": m["paths"] / secs / 1e6,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": m["ms"] / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(spec, r.adaptive), "l2": "flushed between steps (256 MiB fill)",
                       "parallelism": f"sample-split x{world}" + (", exchange steps issued by librtfs_b200.so (rt_comm_render): NCCL all-reduce of the flags (uint8 max); "
                                                                    "the sums reduced, divided and gathered as config.frame_tail says" if world > 1 else ""),
                       "scene_bytes_staged_in_shared_memory": 0 if args.no_smem else handle.shared_memory_bytes()},
            "rays_per_step": m["rays"] / args.steps, "paths_per_step": m["paths"] / args.steps, "degenerate_paths": m["degenerate"],
            "e2e": {"value": e2e["rays"] / e2e["secs"] / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": e2e["h2d"], "d2h_bytes_per_step": e2e["d2h"],
                    "ms_per_step": 1e3 * e2e["secs"] / n_e2e, "steps": n_e2e,
                    "what": ("Scene.make (marshal + BVH build + upload) + Scene.render + Image.render with host buffers" if world == 1 else
                             "per rank: marshal + rt_scene_create (BVH build + upload) + rt_comm_render (kernels and NCCL collectives inside the library); "
                             "rank 0 receives the frame in a host buffer; bytes are summed over ranks")},
            "gpu_launches": m["launches"],
            "clocks": clocks,
            "roofline": {"bound": "fp32", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s", "frac": achieved / fp32_peak if fp32_peak else None,
                         "traffic": traffic, "flops_per_ray": f_ray,
                         "kernel": "render_kernel<PROBE=0> (main phase), rank 0", "kernel_ms_per_launch": main_ms, "rays_per_launch": main_rays,
                         "hbm_bytes_per_ray": hbm_per_ray, "l2_bytes_per_ray": l2_per_ray,
                         "note": "achieved = rays per launch x FLOPs the REFERENCE traversal spends per ray (exhaustive DFS, SURVEY 8d: the contract's "
                                 "algorithmic figure) / duration of the launch from CUDA events the library records around it on its stream; the tests "
                                 "the device actually executes are under roofline_useful; peak = FP32 FMA microbenchmark measured in this run "
                                 "(MEASURED_PEAKS.json has no FP32 figure); traffic, hbm/l2 bytes per ray = ncu, profiles/roofline_traffic.json"},
            "roofline_useful": {"bound": "fp32", "achieved": achieved_exec, "peak": fp32_peak, "unit": "TFLOP/s",
                                "frac": achieved_exec / fp32_peak if fp32_peak else None, "flops_per_ray": f_exec,
                                "note": "the same launch counted with the slab / primitive tests OUR ordered, culled traversal executed "
                                        "(RT_FLAG_COUNTERS frame), SURVEY 8d's per-test weights; shading, RNG and control flow are not counted"},
            "traversal": {"box_tests_per_ray": trav["box_tests"] / max(1, trav["rays"]), "prim_tests_per_ray": trav["prim_tests"] / max(1, trav["rays"]),
                          "rays_per_path": trav["rays"] / max(1, trav["paths"])},
        }
        if dumped:
            line["dumped_outputs"] = dumped
        if hashes:
            line["frame_sha256"] = hashes
        if others:
            line["other_configs"] = others
        if world > 1:
            v, path = native.CommHandle.nccl_version()
            line["config"]["nccl"] = f"{v} bound by librtfs_b200.so from {path}"
            line["config"]["frame_tail"] = ("one kernel over NVLink peer memory (CUDA IPC): sum over ranks, divide, gamma, gather; two 4-byte all-reduces as barriers"
                                            if peer_memory else "ncclReduceScatter + finalize_kernel + ncclAllGather (peer mapping unavailable)")
        if cpu:
            line["cpu_baseline"] = {k: v for k, v in cpu.items() if k != "counters"}
        print(json.dumps(line), flush=True)
    handle.close()
    r.comm.close()
    if world > 1:
        r.dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2", choices=["C1", "C2", "C3", "C4", "C5"])
    ap.add_argument("--spp", type=int, default=0, help="override samples per pixel (a reduced-size run; not the headline)")
    ap.add_argument("--half-extents", type=int, nargs=2, default=None, help="override maxWidthCoord maxHeightCoord")
    ap.add_argument("--no-adaptive", action="store_true")
    ap.add_argument("--no-smem", action="store_true")
    ap.add_argument("--no-lean", action="store_true", help="A/B: do not use the kernel specialised for scenes without FP64 objects and texture lookups")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--bvh", default="auto", choices=["auto", "binary", "wide"],
                    help="which tree the kernels walk: auto = binary in shared memory when the scene fits, else 8-wide compressed (A/B runs)")
    ap.add_argument("--schedule", default="lockstep", choices=["flow", "lockstep"],
                    help="lockstep = one ray per lane per pass (default); flow = a ring of 64 rays per warp, walks pulled by the "
                         "lanes, scatters in full-width passes (measured slower; for A/B runs)")
    ap.add_argument("--no-hash", action="store_true", help="skip the fixed-seed frame hashed through every product path")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the short measurements of the other BASELINE configs")
    ap.add_argument("--other-configs", default="C1,C3,C4,native,C5", help="which of C1..C5 / native to measure after the headline config")
    ap.add_argument("--cpu-seconds", type=float, default=25.0)
    ap.add_argument("--flops-per-ray", type=float, default=0.0, help="FLOPs of the reference traversal per ray, used when the CPU sample does not run (default: the config's figure from DESIGN.md)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame of the last timed step as DIR/rgb.npy and DIR/sums.npy (at most 64 MB in all; a larger frame is a "
                         "fixed, seeded sample of its pixels, indices in DIR/pixel_index.npy)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the frames of --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
