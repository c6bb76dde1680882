"""CPU-side checks of batches of views over several GPUs (no GPU): both prototypes against the header and the ctypes
declarations, the ABI version they leave as it was, and the refusals of a null handle, output or frame pointer that come
before any device work."""
import ctypes as C
import os
import subprocess
import tempfile

from ray_tracing_fsharp_b200 import abi, native, sample_images

from test_window_cpu import _header_args

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_prototypes_match_header():
    src = r'''
#include <stdio.h>
#include "rtfs_b200.h"
int main(void) {
    int (*r)(RtMulti *, const RtCamera *, const uint64_t *, int32_t, int32_t, int32_t, const RtRenderOpts *, uint8_t *, int32_t *,
             RtStats *) = rt_multi_render_views;
    int (*b)(RtMulti *, const RtCamera *, const uint64_t *, int32_t, int32_t, int32_t, const RtRenderOpts *, RtFrame **,
             RtFrameProgress *) = rt_multi_frame_begin_views;
    printf("%d %d %d\n", RT_ABI_VERSION, r != 0, b != 0);
    return 0;
}
'''
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "p.c")
        open(c, "w").write(src)
        subprocess.check_call(["gcc", "-Werror", "-Wincompatible-pointer-types", "-I", os.path.join(ROOT, "include"), "-c", c, "-o",
                               os.path.join(td, "p.o")])
    assert _header_args("rt_multi_render_views") == 10 and len(native.lib().rt_multi_render_views.argtypes) == 10
    assert _header_args("rt_multi_frame_begin_views") == 9 and len(native.lib().rt_multi_frame_begin_views.argtypes) == 9
    assert {"rt_multi_render_views", "rt_multi_frame_begin_views"} <= set(native.EXPORTS)
    # the feature only adds functions: the version callers compare is unchanged
    assert abi.RT_ABI_VERSION == 6 and native.lib().rt_abi_version() == 6


def test_null_handle_output_or_frame_is_refused_before_any_device_work():
    spec = sample_images.few_spheres(max_w=20, max_h=10, spp=4)
    cam = native.camera_make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    cams = (abi.RtCamera * 2)(cam, cam)
    lib = native.lib()
    rgb = (C.c_uint8 * (2 * 41 * 21 * 3))()
    for flags in (0, abi.RT_FLAG_NOISE):
        opts = abi.RtRenderOpts(1, 1, abi.RT_MODE_MEGAKERNEL, 0, flags)
        # no RtMulti: refused as a null handle, with or without an output
        for out_rgb in (rgb, None):
            assert lib.rt_multi_render_views(None, cams, None, 2, 20, 10, C.byref(opts), out_rgb, None, None) == abi.RT_ERR_INVALID_ARGUMENT
            assert "null" in lib.rt_last_error().decode()
        out = C.c_void_p(12345)  # a stale value the call must clear
        assert lib.rt_multi_frame_begin_views(None, cams, None, 2, 20, 10, C.byref(opts), C.byref(out), None) == abi.RT_ERR_INVALID_ARGUMENT
        assert out.value is None
        assert lib.rt_multi_frame_begin_views(None, cams, None, 2, 20, 10, C.byref(opts), None, None) == abi.RT_ERR_INVALID_ARGUMENT
        assert "null" in lib.rt_last_error().decode()
