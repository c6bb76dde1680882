"""CPU-side checks of rt_render_views (no GPU): the prototype and the ctypes declaration against the header, the refusals
that come before any device work, the no-device error, and the machine code of the twelve batched render kernels: they keep
their render_kernel counterparts' register budget (64 staged, 40 global: the launch bounds) and spill at most 16 bytes more."""
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


def test_prototype_matches_header():
    """The header's prototype compiles against the declaration below, and ctypes passes as many arguments."""
    src = r'''
#include <stdio.h>
#include "rtfs_b200.h"
int main(void) {
    int (*f)(RtScene *, const RtCamera *, const uint64_t *, int32_t, int32_t, int32_t, const RtRenderOpts *, uint8_t *, int32_t *,
             RtStats *) = rt_render_views;
    printf("%d %d\n", RT_ABI_VERSION, f != 0);
    return 0;
}
'''
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "p.c")
        open(c, "w").write(src)
        obj = os.path.join(td, "p.o")
        subprocess.check_call(["gcc", "-Werror", "-Wincompatible-pointer-types", "-I", os.path.join(ROOT, "include"), "-c", c, "-o", obj])
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "rtfs_b200.h")).read(), flags=re.S)
    m = re.search(r"int rt_render_views\(([^)]*)\);", text)
    assert m and len(m.group(1).split(",")) == 10
    assert len(native.lib().rt_render_views.argtypes) == 10
    assert abi.RT_ABI_VERSION == 6 and native.lib().rt_abi_version() == 6


def _host_scene():
    spec = sample_images.few_spheres(max_w=20, max_h=10, spp=4)
    hs, ts, keep = marshal(spec.objects)
    h = native.SceneHandle(hs, ts, device=-1, keepalive=keep)
    cam = native.camera_make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    return spec, h, cam


def test_without_a_device():
    spec, h, cam = _host_scene()
    with pytest.raises(native.RtError) as e:
        h.render_views([cam, cam], spec.max_width_coord, spec.max_height_coord, seeds=[1, 2])
    assert e.value.code == abi.RT_ERR_NO_DEVICE
    h.close()


def test_refusals_before_any_device_work():
    spec, h, cam = _host_scene()
    lib = native.lib()
    cams = (abi.RtCamera * 2)(cam, cam)
    opts = abi.RtRenderOpts(1, 1, abi.RT_MODE_MEGAKERNEL, 0, 0)
    rgb = np.zeros(16, np.uint8)
    mw, mh = spec.max_width_coord, spec.max_height_coord
    assert lib.rt_render_views(h.ptr, cams, None, 0, mw, mh, C.byref(opts), native.ptr(rgb), None, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_render_views(h.ptr, None, None, 2, mw, mh, C.byref(opts), native.ptr(rgb), None, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_render_views(h.ptr, cams, None, 2, mw, mh, C.byref(opts), None, None, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_render_views(None, cams, None, 2, mw, mh, C.byref(opts), native.ptr(rgb), None, None) == abi.RT_ERR_INVALID_ARGUMENT
    with pytest.raises(native.RtError) as e:
        h.render_views([], mw, mh)
    assert e.value.code == abi.RT_ERR_INVALID_ARGUMENT
    h.close()


def test_batched_kernels_registers_and_spills():
    """render_views_kernel<PROBE, SMEM, SSTACK, WIDE> against render_kernel<PROBE, SMEM, false, SSTACK, WIDE, false>."""
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
    pat = re.compile(r"void rtfs::render_views_kernel<(true|false), (\d), (true|false), (true|false)>\(rtfs::FrameParams\)$")
    batched = {}
    for name, v in ((n, tuple(info[k])) for k, n in _demangle(list(info)).items()):
        m = pat.match(name)
        if m:
            batched[m.groups()] = v
    assert len(batched) == 12
    assert {(k[1], k[2], k[3]) for k in batched} == {("2", "false", "false"), ("1", "false", "false")} | {
        ("0", s, w) for s in ("false", "true") for w in ("false", "true")}
    for (probe, smem, sstack, wide), (regs, st, ld) in batched.items():
        base_regs, base_st, base_ld = base[f"void rtfs::render_kernel<{probe}, {smem}, false, {sstack}, {wide}, false>(rtfs::FrameParams)"]
        bound = 40 if smem == "0" else 64
        assert regs <= bound and base_regs == bound, (probe, smem, sstack, wide, regs)
        assert st <= base_st + 16 and ld <= base_ld + 16, ((probe, smem, sstack, wide), (st, ld), (base_st, base_ld))
