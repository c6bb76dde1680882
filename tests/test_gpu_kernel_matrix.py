"""Every render kernel the library can launch, on every kind of scene, against the sample-by-sample reconstruction.

A frame's int32 sums must EQUAL the sums of the colours rt_test_trace_samples gives for each pixel's sample indices, with
renderPixel's early-out rule applied to those colours (helpers.expected_sums).  This file keeps two tables, one of scenes
and one of variants (flag sets that select kernel instantiations through the public API), and checks every cell of their
product against one reconstruction per (scene, seed, spp, adaptive): the four int32 fields of every pixel, the path, ray
and early-out counts, the sum of squares Q of progressive NOISE frames after every pass, and, among the counting kernels
that walk the binary tree, the box and primitive test counts.  Retiring a mode is deleting a row.

The new scene families are tied to the double-precision oracle sample by sample, so that the exact check does not only
show that the kernels agree with each other.  Two child processes report the launch plans (RTFS_DEBUG_PLAN) of every
cell, one of them with the walk stacks forced into local memory (RTFS_LOCAL_STACK); together they must reach every
render_kernel and render_flow_kernel instantiation the library holds (tests/golden/render_kernels_sass.json) and the twelve
NOISE instantiations."""
import functools
import json
import os
import subprocess
import sys
import time

import numpy as np
import pytest

if __name__ == "__main__":  # the child processes of test_every_instantiation_is_reached
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import oracle  # noqa: E402
from helpers import expected_moments, expected_sums, f32, oracle_camera, random_unit_vectors  # noqa: E402
from ray_tracing_fsharp_b200 import abi, native, sample_images  # noqa: E402
from ray_tracing_fsharp_b200.domain import (Colour, Hittable, InfinitePlane, InfinitePlaneStyle, ParameterisedTexture, Pixel,  # noqa: E402
                                            Sphere, SphereStyle, Texture, marshal)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MW, MH = 24, 13  # 49 x 27 pixels: neither a multiple of the 8-wide nor of the 4-high tile
SPP = 24         # adaptive: the 11-sample probe, then 13 samples in the main phase


# ---- scenes ------------------------------------------------------------------------------------------------------------
def _sized(spec, mw=MW, mh=MH, spp=SPP):
    spec.max_width_coord, spec.max_height_coord, spec.spp = mw, mh, spp
    return spec


def _reference_sample(name):
    # the scales give half-extents near (23, 13)
    pixels = {"shiny-floor": 400, "fuzzy-floor": 400, "spheres": 200, "inside-sphere": 1200, "total-refraction": 300, "glass": 200,
              "textured-sphere": 200, "moved-camera": 300}[name]
    spec = sample_images.REFERENCE_SAMPLES[name](13.0 / pixels)
    spec.spp = SPP
    return spec


def _col(r, g, b):
    return Texture.Colour(Pixel(r, g, b))


def _spec(name, objs, origin=(0.0, 1.0, -4.0), look_at=(0.0, 0.5, 0.0), depth=50):
    return sample_images.SceneSpec(name, objs, SPP, 1.0, 16.0 / 9.0, origin, look_at, (0.0, 1.0, 0.0), MW, MH, depth)


def planes_only():
    """No bounded sphere (n_bounded == 0): no tree, nothing staged, no walk stack."""
    objs = [Hittable.InfinitePlane(InfinitePlane.make(InfinitePlaneStyle.LambertReflection(0.7, Pixel(200, 180, 40)), (0.0, -0.5, 0.0), (0.0, 1.0, 0.0))),
            Hittable.InfinitePlane(InfinitePlane.make(InfinitePlaneStyle.FuzzedReflection(0.9, Pixel(180, 200, 255), 0.2), (0.0, 0.0, 6.0),
                                                      (0.0, 0.0, -1.0))),
            Hittable.InfinitePlane(InfinitePlane.make(InfinitePlaneStyle.LightSource(_col(255, 255, 230)), (0.0, 5.0, 0.0), (0.0, -1.0, 0.0))),
            Hittable.UnboundedSphere(Sphere.make(SphereStyle.LightSource(_col(90, 90, 160)), (0.0, 0.0, 0.0), 300.0))]
    return _spec("planes only", objs)


def _image(w, h, seed):
    return ParameterisedTexture.Image(np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8))


def one_sphere():
    """A single bounded sphere (the root is its leaf, the right box is {+inf, +inf}) with an image texture, over a plane."""
    interpret = Sphere.plane_map_inverse(1.0, (0.0, 0.5, 1.0))
    objs = [Hittable.Sphere(Sphere.make(SphereStyle.LambertReflection(0.9, ParameterisedTexture.to_texture(interpret, _image(16, 9, 1))),
                                        (0.0, 0.5, 1.0), 1.0)),
            Hittable.InfinitePlane(InfinitePlane.make(InfinitePlaneStyle.PureReflection(0.8, Pixel(230, 230, 240)), (0.0, -0.5, 0.0), (0.0, 1.0, 0.0))),
            Hittable.UnboundedSphere(Sphere.make(SphereStyle.LightSource(_col(200, 200, 230)), (0.0, 0.0, 0.0), 200.0))]
    return _spec("one bounded sphere", objs)


ODD_SIZES = [(1, 1), (1, 7), (7, 1), (3, 5), (1025, 3)]  # (width, height) of the image textures


def checker_nest(depth, leaf_even, leaf_odd, grid=7.0):
    """`depth` checkers nested inside each other, both children of every level the next level: every lookup walks all of them."""
    t = ParameterisedTexture.Checkered(leaf_even, leaf_odd, grid)
    for _ in range(depth - 1):
        t = ParameterisedTexture.Checkered(t, t, grid)
    return t


def odd_textures():
    """Spheres with image textures of 1x1, 1x7, 7x1, 3x5 and 1025x3 texels, and one whose texture is a checker nest exactly as
    deep as the library accepts (8), with an image and a colour as leaves.  Object i is the sphere of ODD_SIZES[i]; object 5 the
    checker."""
    objs = []
    for i, size in enumerate(ODD_SIZES + [None]):
        centre = (-2.5 + 1.0 * i, 0.3 + 0.2 * (i % 2), 1.0 + 0.3 * (i % 3))
        interpret = Sphere.plane_map_inverse(0.45, centre)
        tex = _image(*size, 10 + i) if size else checker_nest(8, _image(3, 5, 30), ParameterisedTexture.Colour(Pixel(20, 200, 60)))
        objs.append(Hittable.Sphere(Sphere.make(SphereStyle.LambertReflection(0.95, ParameterisedTexture.to_texture(interpret, tex)), centre, 0.45)))
    objs += [Hittable.InfinitePlane(InfinitePlane.make(InfinitePlaneStyle.LambertReflection(0.5, Pixel(200, 200, 200)), (0.0, -0.5, 0.0), (0.0, 1.0, 0.0))),
             Hittable.UnboundedSphere(Sphere.make(SphereStyle.LightSource(_col(230, 230, 255)), (0.0, 0.0, 0.0), 200.0))]
    return _spec("odd textures", objs, origin=(0.0, 1.0, -3.0), look_at=(0.0, 0.4, 1.0))


@functools.lru_cache(maxsize=None)
def _random_sphere_objects(n_max=3000, seed=17):
    rng = np.random.default_rng(seed)
    objs = []
    for i in range(n_max):
        c = (float(rng.uniform(-12, 12)), float(rng.uniform(0.1, 4.0)), float(rng.uniform(-2, 22)))
        k = rng.random()
        col = Texture.Colour(Colour.random(rng))
        style = (SphereStyle.LambertReflection(float(rng.random()), col) if k < 0.8 else
                 SphereStyle.FuzzedReflection(0.8, col, float(rng.random() / 2)) if k < 0.95 else SphereStyle.Glass(1.0, Texture.Colour(Colour.White), 1.5))
        objs.append(Hittable.Sphere(Sphere.make(style, c, float(rng.uniform(0.1, 0.35)))))
    return objs


def random_spheres(n):
    """n random spheres (C2's material mix) under a sky, over a floor: the size decides where the scene is read from."""
    objs = list(_random_sphere_objects()[:n])
    objs += [Hittable.UnboundedSphere(Sphere.make(SphereStyle.LightSource(_col(200, 200, 255)), (0.0, 0.0, 0.0), 2000.0)),
             Hittable.UnboundedSphere(Sphere.make(SphereStyle.LambertReflection(0.5, Texture.Colour(Colour.White)), (0.0, -1000.0, 0.0), 1000.0))]
    return _spec(f"{n} random spheres", objs, origin=(0.0, 3.0, -8.0), look_at=(0.0, 1.0, 6.0))


def deep_tree():
    """4000 spheres at distances growing geometrically over ten decades along the view direction, scattered sideways in
    proportion: the SAH peels a few at each level, and the device tree is 45-60 levels deep.  Too big to stage and too deep for
    walk stacks in shared memory, so production runs the global kernel with local stacks."""
    rng = np.random.default_rng(0)
    n = 4000
    dist = 10.0 ** (10.0 * np.arange(n) / n)
    origin = np.array([0.0, 1.0, -5.0])
    c = origin[None] + np.outer(2 + dist, [0.0, 0.0, 1.0]) + rng.normal(size=(n, 3)) * 2.0 * dist[:, None]
    kind = rng.random(n)
    objs = []
    for i in range(n):
        col = _col(*[int(x) for x in rng.integers(0, 256, 3)])
        style = (SphereStyle.LightSource(col) if kind[i] < 0.15 else SphereStyle.FuzzedReflection(0.9, col, 0.3) if kind[i] < 0.3 else
                 SphereStyle.LambertReflection(0.8, col))
        objs.append(Hittable.Sphere(Sphere.make(style, tuple(float(x) for x in c[i]), float(0.2 * dist[i]))))
    return _spec("deep tree", objs, origin=tuple(origin), look_at=(0.0, 1.0, 0.0))


def _config(name):
    return lambda: _sized(sample_images.CONFIGS[name]())


NEW_FAMILIES = {"planes-only": planes_only, "one-sphere": one_sphere, "odd-textures": odd_textures, "deep-tree": deep_tree}


@functools.lru_cache(maxsize=None)
def staging_counts():
    """(n*, the noise-window count): n* is the largest number of random spheres the library stages in shared memory
    (SceneHandle.shared_memory_bytes() > 0), found by bisection.  The kernels with RT_FLAG_NOISE keep 128 more bytes per item
    slot, so a scene staged without the flag but within that much of the limit is read from global memory with it: the
    largest count whose staged bytes are at least 4 KB below n*'s (one more sphere adds far less than 4 KB, the NOISE slots of
    a block far more)."""
    def staged_bytes(n):
        hs, ts, keep = marshal(random_spheres(n).objects)
        h = native.SceneHandle(hs, ts, 0, keepalive=keep)
        b = h.shared_memory_bytes()
        h.close()
        return b

    lo, hi = 1, len(_random_sphere_objects())
    assert staged_bytes(lo) > 0 and staged_bytes(hi) == 0
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if staged_bytes(mid) > 0 else (lo, mid)
    top = staged_bytes(lo)
    a, b = 1, lo
    while b - a > 1:
        mid = (a + b) // 2
        a, b = (mid, b) if staged_bytes(mid) <= top - 4096 else (a, mid)
    return lo, a


def scene_builders():
    """name -> SceneSpec builder, every family of the matrix.  The staging scenes need a device to be sized."""
    table = {f"ref-{k}": functools.partial(_reference_sample, k) for k in sorted(sample_images.REFERENCE_SAMPLES)}
    table.update({"C1": _config("C1"), "C3": _config("C3"), "C4": _config("C4")})
    table.update(NEW_FAMILIES)
    n_star, n_noise = staging_counts()
    table.update({"stage-n*": functools.partial(random_spheres, n_star), "stage-n*+1": functools.partial(random_spheres, n_star + 1),
                  "noise-window": functools.partial(random_spheres, n_noise)})
    return table


SCENE_NAMES = ([f"ref-{k}" for k in sorted(sample_images.REFERENCE_SAMPLES)] + ["C1", "C3", "C4"] + list(NEW_FAMILIES)
               + ["stage-n*", "stage-n*+1", "noise-window"])
SEED = {name: 1000 + i for i, name in enumerate(SCENE_NAMES)}


@functools.lru_cache(maxsize=None)
def device_scene(name):
    spec = scene_builders()[name]()
    hs, ts, keep = marshal(spec.objects)
    return spec, native.SceneHandle(hs, ts, 0, keepalive=keep), oracle_camera(spec), (hs, ts, keep)


# ---- variants ----------------------------------------------------------------------------------------------------------
F = abi
VARIANTS = {
    "default": dict(flags=0),
    "no-lean": dict(flags=F.RT_FLAG_NO_LEAN),
    "no-smem": dict(flags=F.RT_FLAG_NO_SMEM),
    "wide-bvh": dict(flags=F.RT_FLAG_WIDE_BVH),
    "counters": dict(flags=F.RT_FLAG_COUNTERS),
    "no-lean+counters": dict(flags=F.RT_FLAG_NO_LEAN | F.RT_FLAG_COUNTERS),
    "no-smem+counters": dict(flags=F.RT_FLAG_NO_SMEM | F.RT_FLAG_COUNTERS),
    "wide-bvh+counters": dict(flags=F.RT_FLAG_WIDE_BVH | F.RT_FLAG_COUNTERS),
    "flow": dict(flags=F.RT_FLAG_FLOW),
    "flow+no-smem": dict(flags=F.RT_FLAG_FLOW | F.RT_FLAG_NO_SMEM),
    "flow+counters": dict(flags=F.RT_FLAG_FLOW | F.RT_FLAG_COUNTERS),
    "wavefront": dict(flags=0, mode=F.RT_MODE_WAVEFRONT),
    "noise": dict(flags=0, noise=True),
    "noise+no-smem": dict(flags=F.RT_FLAG_NO_SMEM, noise=True),
    "noise+wide-bvh": dict(flags=F.RT_FLAG_WIDE_BVH, noise=True),
    "split-3": dict(flags=0, split=3),
}
BINARY_COUNTING = ["counters", "no-lean+counters", "no-smem+counters", "flow+counters"]  # must agree on box and primitive tests
LOCAL_STACK_VARIANTS = ["no-smem", "wide-bvh", "no-smem+counters", "wide-bvh+counters", "noise+no-smem", "noise+wide-bvh"]
WINDOWS = (1, 7, 0)  # progressive passes: one sample, seven, the rest


WIDE_STACK_LEVELS = 30  # the deepest 8-wide tree the wide walk's stack holds (device_scene_ensure_wide)


@functools.lru_cache(maxsize=None)
def wide_depth(name):
    """Depth of the scene's 8-wide tree, built and verified on the host."""
    return device_scene(name)[1].wide_bvh_check()["depth"]


def wide_unsupported(name, variant):
    """A frame on the 8-wide tree of a scene whose wide tree is deeper than the wide walk's stack: the library refuses it."""
    return bool(VARIANTS[variant]["flags"] & F.RT_FLAG_WIDE_BVH) and wide_depth(name) > WIDE_STACK_LEVELS


class Reconstruction:
    """The expected frame of one (scene, seed, spp, adaptive), rebuilt once from single samples."""

    def __init__(self, dsc, cam, mw, mh, seed, adaptive):
        self.dsc, self.cam, self.mw, self.mh, self.seed, self.adaptive = dsc, cam, mw, mh, seed, adaptive
        self.pixels = np.arange((2 * mw + 1) * (2 * mh + 1))
        self.want, self.count, self.rays = expected_sums(dsc, cam, mw, mh, seed, adaptive, self.pixels)
        spp = int(cam.samples_per_pixel)
        self.n_probe = 2 * min(5, spp // 2) + 1 if adaptive else 0
        self.early_out = len(self.pixels) - int((self.count > self.n_probe).sum()) if adaptive else 0

    def check_sums(self, sums, what):
        got = np.asarray(sums).reshape(-1, 4).astype(np.int64)
        bad = np.flatnonzero((got != self.want).any(1))
        cols = 2 * self.mw + 1
        detail = "; ".join(f"(row {p // cols}, col {p % cols}) frame {got[p].tolist()} samples {self.want[p].tolist()}" for p in bad[:4])
        assert bad.size == 0, f"{what}: {bad.size} of {len(got)} pixels are not the sum of their samples: {detail}"

    def check_q(self, frame, what):
        _, sums = frame.read(want_sums=True)
        _, _, sq = frame.noise(0.0, want_map=False, want_sq=True)
        s = frame.progress.samples_done
        want_sums, want_q = expected_moments(self.dsc, self.cam, self.mw, self.mh, self.seed, self.adaptive, self.pixels, s)
        assert np.array_equal(sums.reshape(-1, 4).astype(np.int64), want_sums), f"{what} at {s} samples: sums"
        bad = np.flatnonzero(sq.reshape(-1).astype(np.int64) != want_q)
        assert bad.size == 0, f"{what} at {s} samples: Q of {bad.size} pixels, e.g. pixel {bad[:4].tolist()}"


def run_variant(dsc, cam, mw, mh, seed, adaptive, variant, rec=None):
    """Runs one variant; returns (sums, paths, rays or None, early_out or None, box_tests, prim_tests).  With `rec`, a NOISE
    frame is checked against it after the probe and after every pass."""
    v = VARIANTS[variant]
    flags = v["flags"]
    if v.get("noise"):
        with dsc.open_frame(cam, mw, mh, seed=seed, adaptive=adaptive, flags=flags | F.RT_FLAG_NOISE) as frame:
            if rec is not None and adaptive:
                rec.check_q(frame, variant)
            for w in WINDOWS:
                frame.advance(max_samples=w)
                if rec is not None:
                    rec.check_q(frame, variant)
            assert frame.progress.done
            _, sums = frame.read(want_sums=True)
            return sums, int(frame.progress.paths_done), None, None, 0, 0
    if v.get("split"):
        from test_gpu_frame_reconstruction import _split_frame
        total, paths, rays, early_out = _split_frame(dsc, cam, mw, mh, seed, adaptive, v["split"])
        return total, paths, rays, early_out, 0, 0
    _, sums, st = dsc.render(cam, mw, mh, seed=seed, adaptive=adaptive, want_sums=True, flags=flags, mode=v.get("mode", F.RT_MODE_MEGAKERNEL))
    return sums, int(st.paths), int(st.rays), int(st.pixels_early_out), int(st.box_tests), int(st.prim_tests)


def check_cell(name, dsc, cam, mw, mh, seed, adaptive, variant, rec):
    what = f"{name} / {variant} / {int(cam.samples_per_pixel)} spp / adaptive {adaptive}"
    if wide_unsupported(name, variant):
        with pytest.raises(native.RtError) as err:
            run_variant(dsc, cam, mw, mh, seed, adaptive, variant, rec)
        assert err.value.code == F.RT_ERR_UNSUPPORTED, what
        return None
    sums, paths, rays, early_out, box, prim = run_variant(dsc, cam, mw, mh, seed, adaptive, variant, rec)
    rec.check_sums(sums, what)
    assert paths == int(rec.count.sum()), what
    if rays is not None:
        assert rays == rec.rays, what
    if early_out is not None:
        assert early_out == rec.early_out, what
    return box, prim


def check_scene(name, spp, variants, adaptives=(True, False)):
    spec, dsc, cam0, _ = device_scene(name)
    cam = abi.RtCamera.from_buffer_copy(cam0)
    cam.samples_per_pixel = spp
    mw, mh, seed = spec.max_width_coord, spec.max_height_coord, SEED[name]
    for adaptive in adaptives:
        rec = Reconstruction(dsc, cam, mw, mh, seed, adaptive)
        counts = {}
        for variant in variants:
            counts[variant] = check_cell(name, dsc, cam, mw, mh, seed, adaptive, variant, rec)
        binary = {v: counts[v] for v in BINARY_COUNTING if v in counts}
        if binary:
            assert len(set(binary.values())) == 1, f"{name} {spp} spp adaptive {adaptive}: box / prim tests differ: {binary}"
            if dsc.device_bvh_check()["spheres"] > 0:
                assert next(iter(binary.values()))[0] > 0


# ---- the matrix ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", SCENE_NAMES)
def test_every_variant_gives_the_reconstructed_frame(name):
    t0 = time.perf_counter()
    check_scene(name, SPP, list(VARIANTS))
    print(f"{name}: {len(VARIANTS)} variants x adaptive on / off in {time.perf_counter() - t0:.1f} s")


@pytest.mark.parametrize("name", ["odd-textures", "stage-n*"])
@pytest.mark.parametrize("spp", [1, 2, 3, 12, 33, 300])
def test_spp_sweep(name, spp):
    """Probe-only frames (spp <= 11 adaptive), a one-sample main phase (12), several chunks (33), a long main phase (300)."""
    check_scene(name, spp, list(VARIANTS))


def test_staging_boundaries_are_where_the_planner_puts_them():
    n_star, n_noise = staging_counts()
    print(f"staged up to {n_star} random spheres; {n_noise} are staged without RT_FLAG_NOISE only")
    assert device_scene("stage-n*")[1].shared_memory_bytes() > 0
    assert device_scene("stage-n*+1")[1].shared_memory_bytes() == 0
    assert device_scene("noise-window")[1].shared_memory_bytes() > 0
    info = device_scene("deep-tree")[1].device_bvh_check()
    print(f"deep tree: binary tree {info['depth']} levels, 8-wide tree {wide_depth('deep-tree')} levels")
    assert 45 <= info["depth"] <= 60, info


# ---- the new scenes against the double-precision oracle --------------------------------------------------------------------
@pytest.mark.parametrize("name", list(NEW_FAMILIES) + ["stage-n*"])
def test_new_scenes_trace_like_the_oracle(name):
    """Random (pixel, sample) pairs traced by the device tracer and by the oracle, with the bars of
    test_trace_samples_match_oracle_sample_for_sample."""
    spec, dsc, cam, (hs, ts, _) = device_scene(name)
    osc = oracle.Scene(hs, ts)
    rng = np.random.default_rng(SEED[name])
    n = 8_000 if name in ("deep-tree", "stage-n*") else 30_000  # the oracle walks big scenes exhaustively
    row = rng.integers(0, spec.rows, n).astype(np.int32)
    col = rng.integers(0, spec.cols, n).astype(np.int32)
    smp = rng.integers(0, 300, n).astype(np.int32)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    wc, wr = osc.trace_samples(cam, mw, mh, 99, row, col, smp)
    gc, gr = dsc.trace_samples(cam, mw, mh, 99, row, col, smp)
    same = (wc == gc).all(1)
    print(f"{name}: {same.mean():.5f} of samples identical, {(wr == gr).mean():.5f} equal ray counts")
    assert same.mean() > 0.998, same.mean()
    assert (wr == gr).mean() > 0.998
    assert np.abs(gc.astype(float).mean(0) - wc.astype(float).mean(0)).max() < 0.5
    assert gc.max() > 0


@pytest.mark.parametrize("index", range(len(ODD_SIZES) + 1), ids=[f"{w}x{h}" for w, h in ODD_SIZES] + ["checker-nest-8"])
def test_odd_texture_lookups_match_the_oracle(index):
    """The texel-edge bar of test_image_texture_lookup everywhere, and exact where a texture has a single texel along an axis at
    every point whose texel coordinate along the other axis lies more than 1e-4 from an edge (FP32 cannot move it across one):
    for 1x1 that is every point, and a lookup that scaled the wrong extent or flipped the wrong axis shows on most of them."""
    spec, dsc, cam, (hs, ts, _) = device_scene("odd-textures")
    osc = oracle.Scene(hs, ts)
    obj = spec.objects[index].sphere
    rng = np.random.default_rng(60 + index)
    p = f32(np.asarray(obj.Centre, float) + obj.Radius * random_unit_vectors(rng, 50_000))
    prim = np.full(len(p), index, np.int32)
    want, got = osc.texture(prim, p), dsc.texture(prim, p)
    same = (want == got).all(1)
    assert same.mean() > 0.998, same.mean()
    if index < len(ODD_SIZES) and 1 in ODD_SIZES[index]:
        w, h = ODD_SIZES[index]
        uv = np.array([oracle.plane_map_inverse(obj.Radius, obj.Centre, q) for q in p])
        x, y = (1.0 - uv[:, 0]) * (w - 1), uv[:, 1] * (h - 1)  # Texture.fs:63-67, before truncation
        clear = ((w == 1) | (np.abs(x - np.round(x)) > 1e-4)) & ((h == 1) | (np.abs(y - np.round(y)) > 1e-4))  # an axis of one texel has no edge
        assert clear.mean() > 0.99, clear.mean()
        assert same[clear].all(), (ODD_SIZES[index], int((~same[clear]).sum()))
    assert len(np.unique(got, axis=0)) > 1 or ODD_SIZES[index] == (1, 1)


# ---- coverage of the instantiations ------------------------------------------------------------------------------------------
PLAN_KEYS = ("probe", "staged", "lean", "count", "sstack", "wide", "flow", "noise")


def kernel_of(plan):
    """The instantiation a plan line names."""
    p = {k: plan[k] == "1" for k in PLAN_KEYS}
    b = lambda x: "true" if x else "false"  # noqa: E731
    if p["flow"]:
        return f"render_flow_kernel<{b(p['probe'])}, {b(p['staged'])}, {b(p['count'])}>"
    smem = 2 if p["lean"] else 1 if p["staged"] else 0
    noise = ", true" if p["noise"] else ""
    return f"render_kernel<{b(p['probe'])}, {smem}, {b(p['count'])}, {b(p['sstack'])}, {b(p['wide'])}{noise}>"


def library_instantiations():
    with open(os.path.join(ROOT, "tests", "golden", "render_kernels_sass.json")) as f:
        names = json.load(f)["kernels"]
    out = set()
    for full in names:
        for k in ("render_kernel<", "render_flow_kernel<"):
            if k in full:
                out.add(full[full.index(k):full.index(">") + 1])
    # the NOISE kernels pick_count returns: the lockstep kernels without counters, with NOISE = true
    out |= {k[:-1] + ", true>" for k in out if k.startswith("render_kernel<") and k.split(", ")[2] == "false"}
    return out


def _marker(text):
    os.write(2, f"cell {text}\n".encode())


def plans_child():
    """One short pass of every cell (adaptive: the probe and a main phase), each preceded by a marker line on stderr."""
    for name in SCENE_NAMES:
        spec, dsc, cam0, _ = device_scene(name)
        cam = abi.RtCamera.from_buffer_copy(cam0)
        cam.samples_per_pixel = 16
        for variant in VARIANTS:
            _marker(f"{name} {variant}")
            try:
                run_variant(dsc, cam, spec.max_width_coord, spec.max_height_coord, 1, True, variant)
            except native.RtError as e:
                assert wide_unsupported(name, variant) and e.code == F.RT_ERR_UNSUPPORTED, (name, variant, e)
    print("plans child: ok")


def local_stack_child():
    """The global kernels with their walk stacks in local memory, on every scene, with the exact check."""
    for name in SCENE_NAMES:
        _marker(f"{name} -")  # not a cell: the exact check's launches
        check_scene(name, SPP, LOCAL_STACK_VARIANTS)
        for variant in LOCAL_STACK_VARIANTS:
            _marker(f"{name} {variant}")
            spec, dsc, cam, _ = device_scene(name)
            try:
                run_variant(dsc, cam, spec.max_width_coord, spec.max_height_coord, 1, True, variant)
            except native.RtError as e:
                assert wide_unsupported(name, variant) and e.code == F.RT_ERR_UNSUPPORTED, (name, variant, e)
    print("local-stack child: ok")


def _run_child(mode, extra_env):
    env = dict(os.environ, RTFS_DEBUG_PLAN="1", **extra_env)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), mode], env=env, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0 and f"{mode} child: ok" in r.stdout, r.stdout[-4000:] + r.stderr[-4000:]
    cells, cell = {}, None
    for line in r.stderr.splitlines():
        if line.startswith("cell "):
            cell = tuple(line.split()[1:3])
            if cell[1] == "-":
                cell = None
            else:
                cells.setdefault(cell, set())
        elif line.startswith("rtfs: plan ") and cell is not None:
            kv = dict(x.split("=") for x in line[len("rtfs: plan "):].split())
            cells[cell].add(tuple(kv[k] for k in PLAN_KEYS))
    return cells


def test_every_instantiation_is_reached():
    production = _run_child("plans", {})
    local = _run_child("local-stack", {"RTFS_LOCAL_STACK": "1"})
    reached = {}
    for where, cells in (("production", production), ("RTFS_LOCAL_STACK", local)):
        for (name, variant), plans in sorted(cells.items()):
            kernels = sorted({kernel_of(dict(zip(PLAN_KEYS, p))) for p in plans})
            print(f"{where:16s} {name:22s} {variant:18s} {' '.join(kernels) if kernels else '(no plan: wavefront mode or refused)'}")
            for k in kernels:
                reached.setdefault(k, set()).add(where)
    want = library_instantiations()
    assert len(want) == 44, len(want)  # 24 render_kernel, 8 render_flow_kernel, 12 NOISE
    print("instantiation table:")
    for k in sorted(want):
        print(f"  {'reached' if k in reached else 'MISSED ':8s} {k:52s} {', '.join(sorted(reached.get(k, ())))}")
    assert want <= set(reached), sorted(want - set(reached))

    def plans_of(cells, name, variant):
        return {dict(zip(PLAN_KEYS, p))["staged"] for p in cells[(name, variant)]}

    # where the planner switches: staged at n*, not at n* + 1; the noise window staged without the flag only
    assert plans_of(production, "stage-n*", "default") == {"1"}
    assert plans_of(production, "stage-n*+1", "default") == {"0"}
    assert plans_of(production, "noise-window", "default") == {"1"}
    assert plans_of(production, "noise-window", "noise") == {"0"}
    # the deep tree runs the global kernel with local walk stacks in production
    assert {(dict(zip(PLAN_KEYS, p))["staged"], dict(zip(PLAN_KEYS, p))["sstack"]) for p in production[("deep-tree", "default")]} == {("0", "0")}
    # no bounded sphere: nothing staged, no walk stack
    assert plans_of(production, "planes-only", "default") == {"0"}


if __name__ == "__main__" and sys.argv[1:] == ["plans"]:
    plans_child()
if __name__ == "__main__" and sys.argv[1:] == ["local-stack"]:
    local_stack_child()
