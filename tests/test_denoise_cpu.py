"""CPU-side checks of denoised previews (no GPU): the two prototypes against the header and the ctypes declarations, the
RtDenoiseOpts mirror against the header's layout, the refusals that come before any device work, the no-device error, the
registers and spills of the new kernels (the filter kernels spill nothing), and properties of tests/denoise_rule.py, the
numpy restatement the device filter is held to bit for bit."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from ray_tracing_fsharp_b200 import abi, native, sample_images
from ray_tracing_fsharp_b200.domain import marshal

import denoise_rule
from test_noise_cpu import _build_product
from test_window_cpu import _header_args, _kernel_report

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("iterations", "feature_samples", "sigma_colour", "sigma_normal", "sigma_albedo", "sigma_depth", "gamma", "_pad0")


def test_prototypes_match_header():
    src = r'''
#include <stdio.h>
#include "rtfs_b200.h"
int main(void) {
    int (*f)(RtFrame *, int32_t, int32_t *, uint8_t *, float *, float *) = rt_frame_features;
    int (*d)(RtFrame *, const RtDenoiseOpts *, uint8_t *, float *) = rt_frame_denoise;
    printf("%d %d %d\n", RT_ABI_VERSION, f != 0, d != 0);
    return 0;
}
'''
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "p.c")
        open(c, "w").write(src)
        subprocess.check_call(["gcc", "-Werror", "-Wincompatible-pointer-types", "-I", os.path.join(ROOT, "include"), "-c", c, "-o",
                               os.path.join(td, "p.o")])
    assert _header_args("rt_frame_features") == 6 and len(native.lib().rt_frame_features.argtypes) == 6
    assert _header_args("rt_frame_denoise") == 4 and len(native.lib().rt_frame_denoise.argtypes) == 4
    assert {"rt_frame_features", "rt_frame_denoise"} <= set(native.EXPORTS)
    assert abi.RT_ABI_VERSION == 6 and native.lib().rt_abi_version() == 6


def test_denoise_opts_mirror_matches_header_layout():
    src = "#include <stdio.h>\n#include <stddef.h>\n#include \"rtfs_b200.h\"\nint main(void) {\n"
    src += '  printf("%zu\\n", sizeof(RtDenoiseOpts));\n'
    for f in FIELDS:
        src += f'  printf("%zu\\n", offsetof(RtDenoiseOpts, {f}));\n'
    src += "  return 0; }\n"
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(td, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        got = [int(x) for x in subprocess.check_output([exe], text=True).split()]
    assert [f[0] for f in abi.RtDenoiseOpts._fields_] == list(FIELDS)
    assert got == [C.sizeof(abi.RtDenoiseOpts)] + [getattr(abi.RtDenoiseOpts, f).offset for f in FIELDS]


def _opts(**kw):
    o = dict(iterations=5, feature_samples=4, sigma_colour=4.0, sigma_normal=0.3, sigma_albedo=16.0, sigma_depth=0.1, gamma=0, _pad0=0)
    o.update(kw)
    return abi.RtDenoiseOpts(*[o[f] for f in FIELDS])


BAD_OPTS = [dict(iterations=0), dict(iterations=11), dict(iterations=-1), dict(feature_samples=0), dict(feature_samples=65)] + [
    {s: v} for s in ("sigma_colour", "sigma_normal", "sigma_albedo", "sigma_depth") for v in (0.0, -1.0, float("nan"), float("inf"), 1e-50, 1e39)]


def test_refusals_before_any_device_work():
    lib = native.lib()
    rgb = np.zeros(3, np.uint8)
    for kw in BAD_OPTS:
        # the options are checked first: the message names the option, not the (missing) frame
        assert lib.rt_frame_denoise(None, C.byref(_opts(**kw)), native.ptr(rgb), None) == abi.RT_ERR_INVALID_ARGUMENT, kw
        assert b"null frame" not in lib.rt_last_error(), (kw, lib.rt_last_error())
    assert lib.rt_frame_denoise(None, None, None, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_frame_denoise(None, C.byref(_opts()), native.ptr(rgb), None) == abi.RT_ERR_INVALID_ARGUMENT
    assert b"null frame" in lib.rt_last_error()
    for samples in (0, 65, -1, 1, 64):
        assert lib.rt_frame_features(None, samples, None, None, None, None) == abi.RT_ERR_INVALID_ARGUMENT


def test_without_a_device():
    spec = sample_images.few_spheres(max_w=20, max_h=10, spp=4)
    hs, ts, keep = marshal(spec.objects)
    h = native.SceneHandle(hs, ts, device=-1, keepalive=keep)
    cam = native.camera_make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    # no frame to denoise: opening one is the no-device error
    with pytest.raises(native.RtError) as e:
        h.open_frame(cam, spec.max_width_coord, spec.max_height_coord, flags=abi.RT_FLAG_NOISE)
    assert e.value.code == abi.RT_ERR_NO_DEVICE
    h.close()


def test_denoise_kernels_registers_and_spills():
    kernels = _kernel_report(_build_product("rtfs_denoise.ptxas.log"))
    names = {n.split("(")[0].replace("void ", ""): v for n, v in kernels.items()}
    assert set(names) == {"rtfs::features_kernel", "rtfs::denoise_input_kernel", "rtfs::atrous_kernel", "rtfs::denoise_output_kernel"}
    for k in ("rtfs::denoise_input_kernel", "rtfs::atrous_kernel", "rtfs::denoise_output_kernel"):
        regs, st, ld = names[k]
        assert st == 0 and ld == 0, (k, st, ld)
        assert regs <= 64, (k, regs)  # 256 threads a block: at most 4 blocks of 64 registers per SM stay resident
    regs, st, ld = names["rtfs::features_kernel"]
    assert regs <= 255 and st <= 64 and ld <= 64, (regs, st, ld)


# ---- the rule's own properties ------------------------------------------------------------------------------------------------
SIGMAS = dict(sigma_colour=4.0, sigma_normal=0.3, sigma_albedo=16.0, sigma_depth=0.1)


def frame(rng, rows, cols, n=16, lo=0, hi=256):
    """Random moments of pixels of n samples each, and random features."""
    vals = rng.integers(lo, hi, (rows, cols, n, 3)).astype(np.int64)
    sums = np.concatenate([vals.sum(2), np.full((rows, cols, 1), n)], 2).astype(np.int32)
    sq = (vals * vals).sum((2, 3)).astype(np.uint64)
    albedo = rng.integers(0, 256, (rows, cols, 3)).astype(np.uint8)
    normal = rng.normal(size=(rows, cols, 3)).astype(np.float32)
    depth = rng.uniform(1, 10, (rows, cols)).astype(np.float32)
    depth[rng.random((rows, cols)) < 0.1] = np.inf
    return sums, sq, albedo, normal, depth


def test_constant_image_is_a_fixed_point():
    rng = np.random.default_rng(1)
    rows, cols = 23, 31
    sums, sq, albedo, normal, depth = frame(rng, rows, cols)
    # every pixel's mean 100.25 (exact in float32, and so are its products with the integer tap weights)
    sums[..., :3] = 1604
    for guides in ((np.zeros_like(albedo), np.zeros_like(normal), np.ones_like(depth)), (albedo, normal, depth)):
        _, lin = denoise_rule.denoise(sums, sq, *guides, iterations=1, **SIGMAS)
        if guides[0] is albedo:  # weights that are not integers: within rounding
            assert np.allclose(lin, np.float32(100.25), rtol=1e-6, atol=0)
        else:
            assert np.array_equal(lin, np.full((rows, cols, 3), np.float32(100.25)))


def test_lone_bright_pixel_with_zero_noise_stays_put():
    rows, cols = 17, 19
    n = 8
    sums = np.zeros((rows, cols, 4), np.int32)
    sums[..., 3] = n
    sums[8, 9, :3] = 255 * n  # every sample 255: E = 0, as for its neighbours (every sample 0)
    sq = np.zeros((rows, cols), np.uint64)
    sq[8, 9] = 3 * 255 * 255 * n
    albedo = np.zeros((rows, cols, 3), np.uint8)
    normal = np.zeros((rows, cols, 3), np.float32)
    depth = np.ones((rows, cols), np.float32)
    rgb, lin = denoise_rule.denoise(sums, sq, albedo, normal, depth, iterations=4, **SIGMAS)
    expect = np.zeros((rows, cols, 3), np.float32)
    expect[8, 9] = 255
    assert np.array_equal(lin, expect) and np.array_equal(rgb, expect.astype(np.uint8))


def test_taps_never_cross_a_view_boundary():
    rng = np.random.default_rng(2)
    rows, cols = 13, 21
    views = [frame(rng, rows, cols, lo=a, hi=b) for a, b in ((0, 40), (200, 256), (0, 256))]
    stacked = [np.stack([v[k] for v in views]) for k in range(5)]
    rgb, lin = denoise_rule.denoise(*stacked, iterations=4, gamma=True, **SIGMAS)
    tall_rgb, tall_lin = denoise_rule.denoise(*[a.reshape((-1,) + a.shape[2:]) for a in stacked], iterations=4, gamma=True,
                                              view_rows=rows, **SIGMAS)
    assert np.array_equal(rgb.reshape(tall_rgb.shape), tall_rgb) and np.array_equal(lin.reshape(tall_lin.shape), tall_lin)
    for v, f in enumerate(views):
        one_rgb, one_lin = denoise_rule.denoise(*f, iterations=4, gamma=True, **SIGMAS)
        assert np.array_equal(rgb[v], one_rgb) and np.array_equal(lin[v], one_lin), v
    # and without the cut the views do bleed into one another (the check above is not vacuous)
    _, bled = denoise_rule.denoise(*[a.reshape((-1,) + a.shape[2:]) for a in stacked], iterations=4, gamma=True, **SIGMAS)
    assert not np.array_equal(bled.reshape(lin.shape), lin)


def test_pixels_without_samples_are_black_and_no_neighbour():
    rng = np.random.default_rng(3)
    rows, cols = 11, 12
    sums, sq, albedo, normal, depth = frame(rng, rows, cols)
    hole = rng.random((rows, cols)) < 0.3
    with_hole = sums.copy()
    with_hole[hole] = 0
    sq_hole = np.where(hole, np.uint64(0), sq)
    rgb, lin = denoise_rule.denoise(with_hole, sq_hole, albedo, normal, depth, iterations=3, **SIGMAS)
    assert (lin[hole] == 0).all() and (rgb[hole] == 0).all()
    # what a hole held does not matter
    other = with_hole.copy()
    other[hole, :3] = 12345
    _, lin2 = denoise_rule.denoise(other, sq_hole, albedo, normal, depth, iterations=3, **SIGMAS)
    assert np.array_equal(lin[~hole], lin2[~hole])
