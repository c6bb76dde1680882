"""Frames rebuilt sample by sample.  The counter RNG makes every sample a pure function of (seed, pixel, sample index),
and rt_test_trace_samples traces one sample per thread with the same path_begin / path_step the render kernels run.
So the int32 accumulators of every pixel of a rendered frame must EQUAL the sum of the tracer's colours over sample
indices 0 .. count - 1, count being renderPixel's early-out rule applied to those same colours.  No tolerance: a sample
lost, traced twice, traced under another index or credited to another pixel shows, as does any difference between the
tracer's arithmetic and the render kernels'.  The tracer itself is tied to the oracle sample by sample (the level-1
test_trace_samples_match_oracle_sample_for_sample, and the oracle checks below on the reconstructed samples).

The frames are the production ones (the C2 frame bench.py times, the native 2401x1601 frame, C3, C4, C5 at full size),
where the schedule takes its production shape: bulk chunks of 32 samples, persistent warps recycling their item slots,
the 100 k-sphere kernel with its walk stacks in shared memory, tile overhang at the frame's edges, a flagged list ending
in a partial unit; and the limits of the frame arguments."""
import os
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import oracle
from helpers import expected_sums, oracle_camera, small_random_spheres, unit
from ray_tracing_fsharp_b200 import abi, sample_images
from ray_tracing_fsharp_b200.domain import marshal


class ParallelTracer:
    """`trace_samples` of a tracer that runs on one thread (orc_trace_samples), split over a thread pool (ctypes releases
    the GIL for the call)."""

    def __init__(self, tracer, threads=None):
        self.tracer = tracer
        self.threads = threads or os.cpu_count() or 1

    def trace_samples(self, cam, max_w, max_h, seed, row, col, sample):
        n = len(row)
        parts = max(1, min(self.threads, n // 256))
        cut = np.linspace(0, n, parts + 1).astype(np.int64)
        with ThreadPoolExecutor(parts) as pool:
            out = list(pool.map(lambda i: self.tracer.trace_samples(cam, max_w, max_h, seed, row[cut[i]:cut[i + 1]], col[cut[i]:cut[i + 1]],
                                                                    sample[cut[i]:cut[i + 1]]), range(parts)))
        return np.concatenate([c for c, _ in out]), np.concatenate([r for _, r in out])


def assert_exact(sums, pixels, want, what):
    """The frame's accumulators at `pixels` equal `want`, every channel and the count."""
    cols = sums.shape[1]
    got = sums.reshape(-1, 4)[pixels].astype(np.int64)
    bad = np.flatnonzero((got != want).any(1))
    detail = "; ".join(f"(row {pixels[i] // cols}, col {pixels[i] % cols}) frame {got[i].tolist()} samples {want[i].tolist()}" for i in bad[:6])
    assert bad.size == 0, f"{what}: {bad.size} of {len(pixels)} pixels are not the sum of their samples: {detail}"


def row_subset(rows, cols, stride, n_random, seed):
    """Flat ids of every pixel of the first tile band (rows 0-3), the last four rows and every `stride`-th row between them
    (an odd stride meets every row of an 8x4 tile), plus `n_random` pixels anywhere."""
    picked = np.unique(np.concatenate([np.arange(4), np.arange(4, rows - 4, stride), np.arange(rows - 4, rows)]))
    pixels = (picked[:, None] * cols + np.arange(cols)[None, :]).ravel()
    extra = np.random.default_rng(seed).integers(0, rows * cols, n_random)
    return np.unique(np.concatenate([pixels, extra]))


def _small(config, max_w, max_h, spp):
    spec = sample_images.CONFIGS[config]()
    spec.max_width_coord, spec.max_height_coord, spec.spp = max_w, max_h, spp
    return spec


# ---- the helper against the oracle's render_pixel (no GPU) ------------------------------------------------------------
@pytest.mark.parametrize("adaptive", [True, False])
@pytest.mark.parametrize("which", ["reduced", "C4"])
def test_expected_sums_is_the_oracle_render(which, adaptive):
    """With the oracle as tracer, expected_sums reproduces orc_render's accumulators (shared counter RNG) bit for bit: the
    early-out rule restated here is renderPixel's, including spp below the probe (spp 4 takes 5 samples)."""
    spec = small_random_spheres() if which == "reduced" else _small("C4", 40, 22, 33)
    hs, ts, _keep = marshal(spec.objects)
    osc = oracle.Scene(hs, ts)
    cam = oracle_camera(spec)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    tracer = ParallelTracer(osc)
    pixels = np.arange(spec.rows * spec.cols)
    for spp in (1, 2, 4, 10, 11, 12, 33):
        cam.samples_per_pixel = spp
        _, ref_stats, counters, _ = osc.render(cam, mw, mh, seed=17, rng_mode=1, adaptive=adaptive)
        want, count, rays = expected_sums(tracer, cam, mw, mh, 17, adaptive, pixels)
        assert np.array_equal(want, ref_stats.reshape(-1, 4)), (which, adaptive, spp)
        assert int(count.sum()) == counters["paths"] and rays == counters["rays"], (which, adaptive, spp)
        if adaptive and spp > 2 * min(5, spp // 2) + 1:
            assert 0 < (count == spp).sum() < len(count), (which, spp)  # both branches of the rule are taken


# ---- full-size frames --------------------------------------------------------------------------------------------------
# Row strides of the reconstructed subsets (odd: every row of a tile is met), chosen for the time the tracer takes on a B200.
STRIDE = {"C2-fixed": 9, "native": 15, "C3": 15, "C4": 27, "C5": 15}
SEED = {"C2": 424242, "C2-fixed": 7, "native": 8, "C3": 9, "C4": 10, "C5": 11}


def _frame_spec(name):
    if name == "native":  # bench.py's: randomSpheres at its author's half-extents, depth 150 as Camera.makeBasic sets it
        return sample_images.random_spheres(max_w=1200, max_h=800, spp=500, depth=150)
    spec = sample_images.CONFIGS[name]()
    if name == "C5":
        spec.spp = 64  # two bulk chunks of 32 samples
    return spec


class Frames:
    """Scenes and default frames, made once per module (the 100 k-sphere scene takes a while to marshal).  "C2-fixed" is the
    bench frame without the early-out."""

    def __init__(self):
        self._scenes = {}
        self._frames = {}

    def scene(self, name):
        from ray_tracing_fsharp_b200 import native
        key = "C2" if name == "C2-fixed" else name
        if key not in self._scenes:
            spec = _frame_spec(key)
            hs, ts, keep = marshal(spec.objects)
            self._scenes[key] = (spec, oracle.Scene(hs, ts), native.SceneHandle(hs, ts, 0, keepalive=keep), oracle_camera(spec), (hs, ts, keep))
        return self._scenes[key]

    def frame(self, name):
        """(spec, osc, dsc, cam, adaptive, sums, stats) of the default render of frame `name`."""
        spec, osc, dsc, cam, _ = self.scene(name)
        adaptive = name != "C2-fixed"
        if name not in self._frames:
            _, sums, stats = dsc.render(cam, spec.max_width_coord, spec.max_height_coord, seed=SEED[name], adaptive=adaptive, want_sums=True)
            self._frames[name] = (sums, stats)
        return (spec, osc, dsc, cam, adaptive) + self._frames[name]


@pytest.fixture(scope="module")
def frames():
    return Frames()


@pytest.mark.gpu
def test_bench_frame_is_the_sum_of_its_samples(frames):
    """The C2 frame bench.py times (1201x801, 500 spp, adaptive), every pixel, and the frame's path, ray and early-out counts."""
    spec, osc, dsc, cam, adaptive, sums, stats = frames.frame("C2")
    pixels = np.arange(spec.rows * spec.cols)
    t0 = time.perf_counter()
    want, count, rays = expected_sums(dsc, cam, spec.max_width_coord, spec.max_height_coord, SEED["C2"], adaptive, pixels)
    print(f"C2 1201x801: {int(count.sum())} paths, {rays} rays reconstructed in {time.perf_counter() - t0:.1f} s")
    assert_exact(sums, pixels, want, "C2 bench frame")
    assert int(stats.paths) == int(count.sum())
    assert int(stats.rays) == rays
    assert int(stats.pixels_early_out) == int((count == 11).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["C2-fixed", "native", "C3", "C4", "C5"])
def test_full_size_frame_rows_are_the_sum_of_their_samples(frames, name):
    """C2 with the early-out off; the native 2401x1601 frame at depth 150; C3 (texture lookups, the full kernel); C4 (planes,
    FP64 objects, depth 100); C5 at 64 spp (the scene read from global memory, walk stacks in shared memory)."""
    spec, osc, dsc, cam, adaptive, sums, stats = frames.frame(name)
    pixels = row_subset(spec.rows, spec.cols, STRIDE[name], 300, SEED[name])
    t0 = time.perf_counter()
    want, count, rays = expected_sums(dsc, cam, spec.max_width_coord, spec.max_height_coord, SEED[name], adaptive, pixels)
    print(f"{name} {spec.cols}x{spec.rows}, stride {STRIDE[name]}: {len(pixels)} pixels, {int(count.sum())} paths reconstructed in "
          f"{time.perf_counter() - t0:.1f} s")
    if name == "C5":
        assert dsc.shared_memory_bytes() == 0  # the global-memory kernel
    assert_exact(sums, pixels, want, name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["C2", "C2-fixed", "native", "C3", "C4", "C5"])
def test_oracle_traces_the_reconstructed_samples(frames, name):
    """The oracle on a random subset of the (pixel, sample) pairs the frames above are rebuilt from, with the bars of
    test_trace_samples_match_oracle_sample_for_sample (the C5 oracle walks the 100 k spheres exhaustively: fewer paths)."""
    spec, osc, dsc, cam, adaptive, sums, stats = frames.frame(name)
    rng = np.random.default_rng(SEED[name] + 1)
    n = 8_000 if name == "C5" else 200_000
    pixels = np.arange(spec.rows * spec.cols) if name == "C2" else row_subset(spec.rows, spec.cols, STRIDE[name], 300, SEED[name])
    pix = rng.choice(pixels, n)
    smp = (rng.random(n) * sums.reshape(-1, 4)[pix, 3]).astype(np.int32)
    row, col = (pix // spec.cols).astype(np.int32), (pix % spec.cols).astype(np.int32)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    wc, wr = ParallelTracer(osc).trace_samples(cam, mw, mh, SEED[name], row, col, smp)
    gc, gr = dsc.trace_samples(cam, mw, mh, SEED[name], row, col, smp)
    same = (wc == gc).all(1)
    if name != "C5":
        assert same.mean() > 0.998, same.mean()
        assert (wr == gr).mean() > 0.998
    else:
        assert same.mean() > 0.985, same.mean()
        assert (wr == gr).mean() > 0.85
    assert np.abs(gc.astype(float).mean(0) - wc.astype(float).mean(0)).max() < 0.5


@pytest.mark.gpu
def test_bench_frame_rows_match_the_oracle_render(frames):
    """The oracle renders the bench frame's strided rows with the shared counter RNG: the early-out decisions (count field)
    agree on the share of pixels test_frame_matches_oracle_with_shared_rng asks for, and the early-out share within 0.01."""
    spec, osc, dsc, cam, adaptive, sums, stats = frames.frame("C2")
    stride = STRIDE["C2-fixed"]
    _, ref_stats, _, n_rows = osc.render(cam, spec.max_width_coord, spec.max_height_coord, seed=SEED["C2"], rng_mode=1, adaptive=True,
                                         row_begin=4, row_step=stride)
    rows = np.arange(4, spec.rows, stride)
    assert n_rows == len(rows)
    got, ref = sums[rows, :, 3], ref_stats[rows, :, 3]
    assert (got == ref).mean() > 0.99, (got == ref).mean()
    assert abs((got == 11).mean() - (ref == 11).mean()) < 0.01


# ---- product paths at full size: the same frame bit for bit ---------------------------------------------------------------
C2_VARIANTS = ["no-lean", "no-smem", "wide-bvh", "bvh2", "flow", "counters", "wavefront", "split-3", "split-8", "comm-1"]
_FLAG = {"no-lean": abi.RT_FLAG_NO_LEAN, "no-smem": abi.RT_FLAG_NO_SMEM, "wide-bvh": abi.RT_FLAG_WIDE_BVH, "bvh2": abi.RT_FLAG_BVH2,
         "flow": abi.RT_FLAG_FLOW, "counters": abi.RT_FLAG_COUNTERS}


def _split_frame(dsc, cam, mw, mh, seed, adaptive, world):
    """The sample split run rank by rank on one device, as test_sample_split_is_invariant_emulated_on_one_gpu runs it."""
    import torch
    from ray_tracing_fsharp_b200.distributed import DeviceBackend
    backends = [DeviceBackend(dsc, cam, mw, mh, seed=seed, adaptive=adaptive) for _ in range(world)]
    bufs = [b.alloc() for b in backends]
    # the ranks share the scene's work counters, which a probe resets and a main phase adds to
    probe = []
    for r in range(world):
        backends[r].probe(r, world, *bufs[r])
        probe.append(backends[r].counters())
    flags = torch.stack([f for _, f in bufs]).max(0).values.contiguous()  # all_reduce(MAX)
    for r in range(world):
        bufs[r][1].copy_(flags)
        backends[r].main(r, world, *bufs[r])
    last = backends[-1].counters()  # the last rank's probe and every rank's main phase
    paths = int(last.paths) + sum(int(c.paths) for c in probe[:-1])
    rays = int(last.rays) + sum(int(c.rays) for c in probe[:-1])
    total = torch.stack([s for s, _ in bufs]).sum(0).to(torch.int32)  # all_reduce(SUM)
    early_out = int((flags == 0).sum().item()) if adaptive else 0
    return total.cpu().numpy(), paths, rays, early_out


@pytest.mark.gpu
@pytest.mark.parametrize("variant", C2_VARIANTS)
def test_product_paths_give_the_bench_frame(frames, variant):
    from ray_tracing_fsharp_b200 import native
    spec, osc, dsc, cam, adaptive, sums, stats = frames.frame("C2")
    mw, mh, seed = spec.max_width_coord, spec.max_height_coord, SEED["C2"]
    if variant in _FLAG:
        _, got, st = dsc.render(cam, mw, mh, seed=seed, adaptive=adaptive, want_sums=True, flags=_FLAG[variant])
        paths, rays, early_out = int(st.paths), int(st.rays), int(st.pixels_early_out)
    elif variant == "wavefront":
        _, got, st = dsc.render(cam, mw, mh, seed=seed, adaptive=adaptive, want_sums=True, mode=abi.RT_MODE_WAVEFRONT)
        paths, rays, early_out = int(st.paths), int(st.rays), int(st.pixels_early_out)
    elif variant.startswith("split-"):
        got, paths, rays, early_out = _split_frame(dsc, cam, mw, mh, seed, adaptive, int(variant[len("split-"):]))
    else:
        comm = native.CommHandle(None, 0, 1, 0)
        _, got, st = comm.render(dsc, cam, mw, mh, seed=seed, adaptive=adaptive, want_rgb=True, want_sums=True)
        comm.close()
        paths, rays, early_out = int(st.paths), int(st.rays), int(st.pixels_early_out)
    got = got.reshape(sums.shape)
    assert np.array_equal(got, sums), f"{variant}: {int((got != sums).any(2).sum())} pixels differ from the default frame"
    assert (paths, rays, early_out) == (int(stats.paths), int(stats.rays), int(stats.pixels_early_out))


# The 8-wide tree (opt-in) and the binary tree visit spheres in different orders, and where two spheres are met at exactly
# the same FP32 t the order decides the winner (F12).  Among the 100 k overlapping spheres of C5 that happens on about one
# ray in 40 M, and 17 of the 8.3 M pixels of this frame differed on a B200.  That the walks differ only on such ties is
# test_wide_and_binary_walks_differ_only_on_exact_ties.  Strict: this starts failing once the two walks break ties alike.
WIDE_C5 = pytest.param("wide-bvh", marks=pytest.mark.xfail(strict=True, reason="exact ties in t: the visiting order picks the sphere (F12)"))


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [WIDE_C5, "flow"])
def test_large_scene_paths_give_the_c5_frame(frames, variant):
    spec, osc, dsc, cam, adaptive, sums, stats = frames.frame("C5")
    _, got, st = dsc.render(cam, spec.max_width_coord, spec.max_height_coord, seed=SEED["C5"], adaptive=adaptive, want_sums=True,
                            flags=_FLAG[variant])
    assert np.array_equal(got, sums), f"{variant}: {int((got != sums).any(2).sum())} pixels differ from the default frame"
    assert (int(st.paths), int(st.rays), int(st.pixels_early_out)) == (int(stats.paths), int(stats.rays), int(stats.pixels_early_out))


@pytest.mark.gpu
def test_wide_and_binary_walks_differ_only_on_exact_ties(frames):
    """Where the two C5 frames differ: the closest hit of the 8-wide walk against the binary walk on 8 M camera rays of the 100 k
    spheres and on as many rays leaving the camera rays' first strike points.  Same sphere and same t, or two spheres at exactly the same
    t, where the visiting order decides (F12); a sphere the quantised boxes lost would show as a miss or a larger t."""
    from ray_tracing_fsharp_b200 import native
    spec, osc, dsc, cam, _ = frames.scene("C5")
    mw, mh = spec.max_width_coord, spec.max_height_coord
    rng = np.random.default_rng(43)
    ties = 0
    for _ in range(4):
        n = 2_000_000
        row = rng.integers(-mh - 1, mh, n).astype(np.int32)
        col = rng.integers(-mw, mw + 1, n).astype(np.int32)
        o, d = native.camera_rays(cam, mw, mh, row, col, rng.random(n), rng.random(n))
        prim, _, strike = dsc.hit_object(o, d, 0)
        hit = prim >= 0
        for oo, dd in ((o, d), (strike[hit], unit(rng.normal(size=(int(hit.sum()), 3))))):
            p0, t0, _ = dsc.hit_object(oo, dd, 0)
            p2, t2, _ = dsc.hit_object(oo, dd, 2)
            assert np.array_equal(p0 >= 0, p2 >= 0), int((p0 >= 0).sum() - (p2 >= 0).sum())
            h = p0 >= 0
            assert np.array_equal(t0[h], t2[h]), [(int(p0[i]), int(p2[i]), float(t0[i]), float(t2[i])) for i in np.flatnonzero(h & (t0 != t2))[:6]]
            ties += int((p0 != p2).sum())
    print(f"C5: {ties} rays whose closest spheres tie exactly")


@pytest.mark.gpu
def test_devices_of_one_process_give_the_bench_frame(frames):
    from ray_tracing_fsharp_b200 import native
    n = native.device_count()
    if n < 2:
        pytest.skip("needs two GPUs")
    spec, osc, dsc, cam, adaptive, sums, stats = frames.frame("C2")
    hs, ts, keep = frames.scene("C2")[4]
    for world in sorted({2, n}):
        m = native.MultiHandle(hs, ts, list(range(world)), keepalive=keep)
        _, got, st = m.render(cam, spec.max_width_coord, spec.max_height_coord, seed=SEED["C2"], adaptive=adaptive, want_sums=True)
        m.close()
        assert np.array_equal(got, sums), world
        assert (int(st.paths), int(st.rays)) == (int(stats.paths), int(stats.rays)), world


# ---- limits and boundaries ---------------------------------------------------------------------------------------------------
def _device_pair(spec):
    from ray_tracing_fsharp_b200 import native
    hs, ts, keep = marshal(spec.objects)
    return oracle.Scene(hs, ts), native.SceneHandle(hs, ts, 0, keepalive=keep), oracle_camera(spec)


def _check_against_oracle(osc, cam, max_w, max_h, seed, adaptive, rgb, sums, stats):
    """The crop bars of test_frame_matches_oracle_with_shared_rng."""
    ref, ref_stats, counters, _ = osc.render(cam, max_w, max_h, seed=seed, rng_mode=1, adaptive=adaptive)
    assert (rgb == ref).all(2).mean() > 0.985, (rgb == ref).all(2).mean()
    assert (sums == ref_stats).all(2).mean() > 0.97, (sums == ref_stats).all(2).mean()
    assert (sums[..., 3] != ref_stats[..., 3]).mean() < 0.01
    assert abs(int(stats.paths) - counters["paths"]) <= 0.01 * counters["paths"]
    assert abs(int(stats.rays) - counters["rays"]) <= 0.01 * counters["rays"]
    assert np.abs(rgb.astype(int) - ref.astype(int)).mean() < 0.3


def _reconstruct_whole_frame(osc, dsc, cam, max_w, max_h, seed, adaptive, oracle_too=True):
    rgb, sums, stats = dsc.render(cam, max_w, max_h, seed=seed, adaptive=adaptive, want_sums=True)
    pixels = np.arange(sums.shape[0] * sums.shape[1])
    want, count, rays = expected_sums(dsc, cam, max_w, max_h, seed, adaptive, pixels)
    what = f"{sums.shape[1]}x{sums.shape[0]} {int(cam.samples_per_pixel)} spp adaptive {adaptive}"
    assert_exact(sums, pixels, want, what)
    assert (int(stats.paths), int(stats.rays)) == (int(count.sum()), rays), what
    if oracle_too:
        _check_against_oracle(osc, cam, max_w, max_h, seed, adaptive, rgb, sums, stats)
    return sums, count


@pytest.mark.gpu
@pytest.mark.parametrize("max_w,max_h", [(32767, 1), (1, 16383)], ids=["widest", "tallest"])
def test_largest_frame_extents(max_w, max_h):
    """65535 x 3 (columns need all 16 bits of an item's packed pixel) and 3 x 32767, probe-only (8 spp: the probe takes 9)
    and with every pixel in the main phase."""
    osc, dsc, cam = _device_pair(_small("C1", max_w, max_h, 8))
    for adaptive in (True, False):
        _reconstruct_whole_frame(osc, dsc, cam, max_w, max_h, 23, adaptive)


@pytest.mark.gpu
def test_camera_rays_at_the_widest_columns():
    """Camera rays at columns up to +-32767, with test_camera_rays' bars."""
    from ray_tracing_fsharp_b200 import native
    spec = sample_images.few_spheres()
    cam = native.camera_make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    rng = np.random.default_rng(29)
    n = 50_000
    max_w, max_h = 32767, 1
    col = rng.integers(-max_w, max_w + 1, n).astype(np.int32)
    col[:8] = [-32767, -32767, 32767, 32767, -32766, 32766, 0, 1]
    row = rng.integers(-max_h - 1, max_h, n).astype(np.int32)
    r1, r2 = [np.asarray(rng.random(n), np.float32).astype(np.float64) for _ in range(2)]
    wo, wd = oracle.camera_rays(cam, max_w, max_h, row, col, r1, r2)
    go, gd = native.camera_rays(cam, max_w, max_h, row, col, r1, r2)
    assert np.abs(go - wo).max() <= 1e-6 * (1 + np.abs(wo).max())
    assert np.abs(gd - wd).max() <= 1e-5
    assert np.abs((gd * gd).sum(1) - 1).max() < 1e-6


@pytest.mark.gpu
def test_one_past_each_limit_is_an_invalid_argument():
    from ray_tracing_fsharp_b200 import native
    osc, dsc, cam = _device_pair(_small("C1", 1, 1, 4))
    for max_w, max_h, spp in [(32768, 1, 4), (1, 16384, 4), (1, 1, (1 << 22) + 1)]:
        cam.samples_per_pixel = spp
        with pytest.raises(native.RtError) as err:
            dsc.render(cam, max_w, max_h, seed=1)
        assert err.value.code == abi.RT_ERR_INVALID_ARGUMENT, (max_w, max_h, spp)


@pytest.mark.gpu
@pytest.mark.parametrize("main_samples", [40959, 40960, 40961, 81921])
def test_main_phase_launch_boundaries(main_samples):
    """One main-phase launch covers 40960 sample indices of a rank (kMaxLaunchSamples): adaptive frames of 5 x 3 pixels whose
    flagged pixels take just under, exactly, just over one launch, and just over two."""
    spp = 11 + main_samples
    osc, dsc, cam = _device_pair(_small("C1", 2, 1, spp))
    sums, count = _reconstruct_whole_frame(osc, dsc, cam, 2, 1, 31, True, oracle_too=False)
    assert (count == spp).any() and (count == 11).any()


@pytest.mark.gpu
def test_most_samples_per_pixel():
    """spp = 2^22, the largest the library takes, 3 x 3 pixels without the early-out: 37.7 M paths into int32 sums, a light of
    (255, 255, 255) seen straight on by most of them."""
    from ray_tracing_fsharp_b200.domain import Colour, Hittable, Pixel, Sphere, SphereStyle, Texture
    spec = sample_images.few_spheres(max_w=1, max_h=1, spp=1 << 22)
    spec.objects = [o for o in spec.objects if type(o).__name__ != "UnboundedSphere"]
    spec.objects.append(Hittable.UnboundedSphere(Sphere.make(SphereStyle.LightSource(Texture.Colour(Pixel(255, 255, 255))), (0.0, 0.0, 0.0),
                                                             200.0)))
    osc, dsc, cam = _device_pair(spec)
    sums, count = _reconstruct_whole_frame(osc, dsc, cam, 1, 1, 37, False, oracle_too=False)
    assert sums[..., :3].max() == 255 << 22  # a pixel of nothing but light: the largest sum there can be


@pytest.mark.gpu
@pytest.mark.parametrize("max_h", [24, 25])
@pytest.mark.parametrize("max_w", [48, 49, 50, 51])
def test_frames_that_end_in_partial_tiles(max_w, max_h):
    """cols = 97, 99, 101, 103 (every odd residue mod the 8-wide tile) by rows = 49, 51 (both odd residues mod 4), adaptive
    and not; without the early-out the flagged list holds every pixel, an odd number, so it ends in a partial unit of 32."""
    osc, dsc, cam = _device_pair(_small("C1", max_w, max_h, 16))
    for adaptive in (True, False):
        _reconstruct_whole_frame(osc, dsc, cam, max_w, max_h, 41 + max_w + max_h, adaptive)
