"""CPU-side checks of progressive frames of a batch of views (no GPU): the two prototypes against the header and the ctypes
declarations, the ABI version they leave as it was, the refusals that come before any device work, the no-device error, and
the machine code of the twelve render_views_noise_kernel shapes: each stays within its launch bound (64 staged, 40 global)
and spills at most 16 bytes more than its render_kernel<PROBE, SMEM, false, SSTACK, WIDE, true> counterpart."""
import ctypes as C
import os
import re
import subprocess
import tempfile

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
    int (*b)(RtScene *, const RtCamera *, const uint64_t *, int32_t, int32_t, int32_t, const RtRenderOpts *, RtFrame **,
             RtFrameProgress *) = rt_frame_begin_views;
    int (*n)(RtFrame *, double, RtFrameNoise *) = rt_frame_view_noise;
    printf("%d %d %d\n", RT_ABI_VERSION, b != 0, n != 0);
    return 0;
}
'''
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "p.c")
        open(c, "w").write(src)
        subprocess.check_call(["gcc", "-Werror", "-Wincompatible-pointer-types", "-I", os.path.join(ROOT, "include"), "-c", c, "-o",
                               os.path.join(td, "p.o")])
    assert _header_args("rt_frame_begin_views") == 9 and len(native.lib().rt_frame_begin_views.argtypes) == 9
    assert _header_args("rt_frame_view_noise") == 3 and len(native.lib().rt_frame_view_noise.argtypes) == 3
    assert {"rt_frame_begin_views", "rt_frame_view_noise"} <= set(native.EXPORTS)
    # the feature only adds functions: the version callers compare is unchanged
    assert abi.RT_ABI_VERSION == 6 and native.lib().rt_abi_version() == 6


def _host_scene():
    spec = sample_images.few_spheres(max_w=20, max_h=10, spp=4)
    hs, ts, keep = marshal(spec.objects)
    h = native.SceneHandle(hs, ts, device=-1, keepalive=keep)
    cam = native.camera_make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    return spec, h, cam


def test_without_a_device():
    spec, h, cam = _host_scene()
    for flags in (0, abi.RT_FLAG_NOISE):
        with pytest.raises(native.RtError) as e:
            h.open_frame_views([cam, cam], spec.max_width_coord, spec.max_height_coord, seeds=[1, 2], flags=flags)
        assert e.value.code == abi.RT_ERR_NO_DEVICE
    h.close()


def test_refusals_before_any_device_work():
    spec, h, cam = _host_scene()
    lib = native.lib()
    cams = (abi.RtCamera * 2)(cam, cam)
    opts = abi.RtRenderOpts(1, 1, abi.RT_MODE_MEGAKERNEL, 0, abi.RT_FLAG_NOISE)
    out = C.c_void_p()
    mw, mh = spec.max_width_coord, spec.max_height_coord
    assert lib.rt_frame_begin_views(h.ptr, cams, None, 0, mw, mh, C.byref(opts), C.byref(out), None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_frame_begin_views(h.ptr, None, None, 2, mw, mh, C.byref(opts), C.byref(out), None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_frame_begin_views(None, cams, None, 2, mw, mh, C.byref(opts), C.byref(out), None) == abi.RT_ERR_INVALID_ARGUMENT
    assert out.value is None
    noise = (abi.RtFrameNoise * 1)()
    assert lib.rt_frame_view_noise(None, 1.0, noise) == abi.RT_ERR_INVALID_ARGUMENT
    with pytest.raises(native.RtError) as e:
        h.open_frame_views([], mw, mh)
    assert e.value.code == abi.RT_ERR_INVALID_ARGUMENT
    with pytest.raises(ValueError):
        h.open_frame_views([cam, cam], mw, mh, seeds=[1])
    h.close()


def test_batched_noise_kernels_registers_and_spills():
    """render_views_noise_kernel<PROBE, SMEM, SSTACK, WIDE> against render_kernel<PROBE, SMEM, false, SSTACK, WIDE, true>."""
    base = _ptxas_report()
    log = _build_product("rtfs_views.ptxas.log")
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
    pat = re.compile(r"void rtfs::render_views_noise_kernel<(true|false), (\d), (true|false), (true|false)>\(rtfs::FrameParams\)$")
    batched = {}
    for name, v in ((n, tuple(info[k])) for k, n in _demangle(list(info)).items()):
        m = pat.match(name)
        if m:
            batched[m.groups()] = v
    assert len(batched) == 12
    assert {(k[1], k[2], k[3]) for k in batched} == {("2", "false", "false"), ("1", "false", "false")} | {
        ("0", s, w) for s in ("false", "true") for w in ("false", "true")}
    for (probe, smem, sstack, wide), (regs, st, ld) in batched.items():
        _, base_st, base_ld = base[f"void rtfs::render_kernel<{probe}, {smem}, false, {sstack}, {wide}, true>(rtfs::FrameParams)"]
        bound = 40 if smem == "0" else 64
        assert regs <= bound, (probe, smem, sstack, wide, regs)
        assert st <= base_st + 16 and ld <= base_ld + 16, ((probe, smem, sstack, wide), (st, ld), (base_st, base_ld))
