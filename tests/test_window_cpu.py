"""CPU-side checks of windows of a frame (no GPU): the two prototypes against the header and the ctypes declarations, the ABI
version they leave as it was, the refusals of a bad window or a null output that come before any device work, the no-device
error, and the machine code of the 24 window kernels: each stays within its launch bound (64 staged, 40 global) and spills
at most 16 bytes more than its render_kernel<PROBE, SMEM, false, SSTACK, WIDE, NOISE> counterpart."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from ray_tracing_fsharp_b200 import abi, native, sample_images
from ray_tracing_fsharp_b200.domain import marshal

from test_noise_cpu import _build_product, _demangle, _ptxas_report

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_args(name):
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "rtfs_b200.h")).read(), flags=re.S)
    m = re.search(r"int " + name + r"\(([^)]*)\);", text)
    assert m, name
    return len(m.group(1).split(","))


def test_prototypes_match_header():
    src = r'''
#include <stdio.h>
#include "rtfs_b200.h"
int main(void) {
    int (*r)(RtScene *, const RtCamera *, int32_t, int32_t, int32_t, int32_t, int32_t, int32_t, const RtRenderOpts *, uint8_t *,
             int32_t *, RtStats *) = rt_render_window;
    int (*b)(RtScene *, const RtCamera *, int32_t, int32_t, int32_t, int32_t, int32_t, int32_t, const RtRenderOpts *, RtFrame **,
             RtFrameProgress *) = rt_frame_begin_window;
    printf("%d %d %d\n", RT_ABI_VERSION, r != 0, b != 0);
    return 0;
}
'''
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "p.c")
        open(c, "w").write(src)
        subprocess.check_call(["gcc", "-Werror", "-Wincompatible-pointer-types", "-I", os.path.join(ROOT, "include"), "-c", c, "-o",
                               os.path.join(td, "p.o")])
    assert _header_args("rt_render_window") == 12 and len(native.lib().rt_render_window.argtypes) == 12
    assert _header_args("rt_frame_begin_window") == 11 and len(native.lib().rt_frame_begin_window.argtypes) == 11
    assert {"rt_render_window", "rt_frame_begin_window"} <= set(native.EXPORTS)
    # the feature only adds functions: the version callers compare is unchanged
    assert abi.RT_ABI_VERSION == 6 and native.lib().rt_abi_version() == 6


def _host_scene():
    spec = sample_images.few_spheres(max_w=20, max_h=10, spp=4)  # 41 x 21
    hs, ts, keep = marshal(spec.objects)
    h = native.SceneHandle(hs, ts, device=-1, keepalive=keep)
    cam = native.camera_make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    return spec, h, cam


def test_without_a_device():
    spec, h, cam = _host_scene()
    mw, mh = spec.max_width_coord, spec.max_height_coord
    with pytest.raises(native.RtError) as e:
        h.render_window(cam, mw, mh, (3, 4, 5, 6))
    assert e.value.code == abi.RT_ERR_NO_DEVICE
    for flags in (0, abi.RT_FLAG_NOISE):
        with pytest.raises(native.RtError) as e:
            h.open_frame_window(cam, mw, mh, (0, 0, 2 * mh + 1, 2 * mw + 1), flags=flags)
        assert e.value.code == abi.RT_ERR_NO_DEVICE
    h.close()


# (row0, col0, rows, cols) refused on the 41 x 21 frame of _host_scene
BAD_WINDOWS = [(0, 0, 0, 5), (0, 0, 5, 0), (0, 0, -1, 5), (-1, 0, 5, 5), (0, -1, 5, 5), (17, 0, 5, 5), (0, 37, 5, 5), (0, 0, 22, 41),
               (0, 0, 21, 42), (20, 40, 2, 1), (2 ** 31 - 1, 0, 1, 1), (0, 2 ** 31 - 1, 1, 1), (1, 1, 2 ** 31 - 1, 1)]


def test_refusals_before_any_device_work():
    spec, h, cam = _host_scene()
    lib = native.lib()
    mw, mh = spec.max_width_coord, spec.max_height_coord
    opts = abi.RtRenderOpts(1, 1, abi.RT_MODE_MEGAKERNEL, 0, abi.RT_FLAG_NOISE)
    rgb = np.zeros(21 * 41 * 3, np.uint8)
    for w in BAD_WINDOWS:
        assert lib.rt_render_window(h.ptr, C.byref(cam), mw, mh, *w, C.byref(opts), native.ptr(rgb), None, None) == abi.RT_ERR_INVALID_ARGUMENT, w
        out = C.c_void_p()
        assert lib.rt_frame_begin_window(h.ptr, C.byref(cam), mw, mh, *w, C.byref(opts), C.byref(out), None) == abi.RT_ERR_INVALID_ARGUMENT, w
        assert out.value is None
    ok = (0, 0, 2 * mh + 1, 2 * mw + 1)
    assert lib.rt_render_window(h.ptr, C.byref(cam), mw, mh, *ok, C.byref(opts), None, None, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_frame_begin_window(h.ptr, C.byref(cam), mw, mh, *ok, C.byref(opts), None, None) == abi.RT_ERR_INVALID_ARGUMENT
    # rt_render's own argument errors
    out = C.c_void_p()
    assert lib.rt_render_window(None, C.byref(cam), mw, mh, *ok, C.byref(opts), native.ptr(rgb), None, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_render_window(h.ptr, None, mw, mh, *ok, C.byref(opts), native.ptr(rgb), None, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_render_window(h.ptr, C.byref(cam), mw, mh, *ok, None, native.ptr(rgb), None, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_frame_begin_window(None, C.byref(cam), mw, mh, *ok, C.byref(opts), C.byref(out), None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_frame_begin_window(h.ptr, C.byref(cam), mw, mh, *ok, None, C.byref(out), None) == abi.RT_ERR_INVALID_ARGUMENT
    assert out.value is None
    with pytest.raises(native.RtError) as e:
        h.render_window(cam, mw, mh, (0, 0, 0, 3))
    assert e.value.code == abi.RT_ERR_INVALID_ARGUMENT
    with pytest.raises(native.RtError) as e:
        h.open_frame_window(cam, mw, mh, (5, 5, 100, 3))
    assert e.value.code == abi.RT_ERR_INVALID_ARGUMENT
    h.close()


def _kernel_report(log):
    info, cur = {}, None
    for line in open(log):
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur = m.group(1)
            info[cur] = [None, None, None]
            continue
        if cur is None:
            continue
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m:
            info[cur][1:] = [int(m.group(1)), int(m.group(2))]
        m = re.search(r"Used (\d+) registers", line)
        if m:
            info[cur][0] = int(m.group(1))
    return {n: tuple(info[k]) for k, n in _demangle(list(info)).items()}


def test_window_kernels_registers_and_spills():
    """render_window(_noise)_kernel<PROBE, SMEM, SSTACK, WIDE> against render_kernel<PROBE, SMEM, false, SSTACK, WIDE, NOISE>."""
    base = _ptxas_report()
    pat = re.compile(r"void rtfs::render_window(_noise)?_kernel<(true|false), (\d), (true|false), (true|false)>\(rtfs::FrameParams\)$")
    kernels = {}
    for name, v in _kernel_report(_build_product("rtfs_window.ptxas.log")).items():
        m = pat.match(name)
        if m:
            kernels[(m.group(1) is not None,) + m.groups()[1:]] = v
    assert len(kernels) == 24
    shapes = {("2", "false", "false"), ("1", "false", "false")} | {("0", s, w) for s in ("false", "true") for w in ("false", "true")}
    for noise in (False, True):
        for probe in ("true", "false"):
            assert {k[2:] for k in kernels if k[0] == noise and k[1] == probe} == shapes
    for (noise, probe, smem, sstack, wide), (regs, st, ld) in kernels.items():
        key = f"void rtfs::render_kernel<{probe}, {smem}, false, {sstack}, {wide}, {'true' if noise else 'false'}>(rtfs::FrameParams)"
        _, base_st, base_ld = base[key]
        bound = 40 if smem == "0" else 64
        assert regs <= bound, (noise, probe, smem, sstack, wide, regs)
        assert st <= base_st + 16 and ld <= base_ld + 16, ((noise, probe, smem, sstack, wide), (st, ld), (base_st, base_ld))
