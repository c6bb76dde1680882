"""CPU-side checks of in-place scene edits (no GPU): the prototype and the RtSceneUpdate mirror against the header, the
errors a call gets without a device, the registers and spills of the edit kernels, and tests/refit_rule.py, the numpy
restatement of the refit the device is held to exactly: on an unedited scene it reproduces the host build's tree, and over
moved spheres every box it forms contains what lies below it."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from ray_tracing_fsharp_b200 import abi, native, sample_images
from ray_tracing_fsharp_b200.domain import marshal

import refit_rule
from test_noise_cpu import _build_product
from test_window_cpu import _header_args, _kernel_report

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("objects", "textures", "spheres_moved", "nodes_refit", "generation", "device_ms", "launches", "_pad0")


def test_prototype_matches_header():
    src = r'''
#include <stdio.h>
#include "rtfs_b200.h"
int main(void) {
    int (*u)(RtScene *, const int32_t *, const RtHittable *, int32_t, const int32_t *, const RtTexture *, int32_t, RtSceneUpdate *) =
        rt_scene_update;
    printf("%d %d\n", RT_ABI_VERSION, u != 0);
    return 0;
}
'''
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "p.c")
        open(c, "w").write(src)
        subprocess.check_call(["gcc", "-Werror", "-Wincompatible-pointer-types", "-I", os.path.join(ROOT, "include"), "-c", c, "-o",
                               os.path.join(td, "p.o")])
    assert _header_args("rt_scene_update") == 8 and len(native.lib().rt_scene_update.argtypes) == 8
    assert "rt_scene_update" in native.EXPORTS
    assert abi.RT_ABI_VERSION == 6 and native.lib().rt_abi_version() == 6


def test_scene_update_mirror_matches_header_layout():
    src = "#include <stdio.h>\n#include <stddef.h>\n#include \"rtfs_b200.h\"\nint main(void) {\n"
    src += '  printf("%zu\\n", sizeof(RtSceneUpdate));\n'
    for f in FIELDS:
        src += f'  printf("%zu\\n", offsetof(RtSceneUpdate, {f}));\n'
    src += "  return 0; }\n"
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(td, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        got = [int(x) for x in subprocess.check_output([exe], text=True).split()]
    assert [f[0] for f in abi.RtSceneUpdate._fields_] == list(FIELDS)
    assert got == [C.sizeof(abi.RtSceneUpdate)] + [getattr(abi.RtSceneUpdate, f).offset for f in FIELDS]


def test_without_a_device():
    lib = native.lib()
    spec = sample_images.few_spheres(max_w=20, max_h=10, spp=4)
    hs, ts, keep = marshal(spec.objects)
    # a host-only scene cannot be edited: it has no device records
    h = native.SceneHandle(hs, ts, device=-1, keepalive=keep)
    with pytest.raises(native.RtError) as e:
        h.update([0], [hs[0]])
    assert e.value.code == abi.RT_ERR_UNSUPPORTED
    # argument errors come first
    assert lib.rt_scene_update(None, None, None, 0, None, None, 0, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_scene_update(h.ptr, None, None, -1, None, None, 0, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_scene_update(h.ptr, None, None, 1, None, None, 0, None) == abi.RT_ERR_INVALID_ARGUMENT
    h.close()
    # and without a device there is no device scene to edit: creating one is the no-device error
    if native.device_count() == 0:
        with pytest.raises(native.RtError) as e:
            native.SceneHandle(hs, ts, device=0, keepalive=keep)
        assert e.value.code == abi.RT_ERR_NO_DEVICE


def test_edit_kernels_registers_and_spills():
    kernels = _kernel_report(_build_product("rtfs_edit.ptxas.log"))
    names = {n.split("(")[0].replace("void ", ""): v for n, v in kernels.items()}
    assert set(names) == {"rtfs::edit_scatter_kernel", "rtfs::refit_mark_kernel", "rtfs::refit_climb_kernel"}
    for k, (regs, st, ld) in names.items():
        assert st == 0 and ld == 0, (k, st, ld)
        assert regs <= 64, (k, regs)  # 256 threads a block


# ---- the rule -------------------------------------------------------------------------------------------------------------------
def host_scene(spec):
    hs, ts, keep = marshal(spec.objects)
    return hs, native.SceneHandle(hs, ts, device=-1, keepalive=keep)


SPECS = {
    "C1": lambda: sample_images.few_spheres(max_w=20, max_h=10, spp=4),
    "C2": lambda: sample_images.random_spheres(spp=4),
    "C4": lambda: sample_images.mixed_planes(max_w=20, max_h=10, spp=4),
}


@pytest.mark.parametrize("name", sorted(SPECS))
def test_rule_reproduces_the_host_build(name):
    hs, h = host_scene(SPECS[name]())
    bounds, right, prim = h.bvh_nodes(abi.RT_BVH_SAH)
    boxes = refit_rule.refit(right, prim, hs)
    assert np.array_equal(boxes.astype(np.float64), bounds)
    # the device form of every child box contains the box it is made from
    for i in np.nonzero(right >= 0)[0]:
        for child in (i + 1, right[i]):
            c, hh = refit_rule.device_node_of(boxes[child, :3], boxes[child, 3:])
            assert (hh >= 0).all()
            assert (c.astype(np.float64) - hh <= boxes[child, :3]).all() and (c.astype(np.float64) + hh >= boxes[child, 3:]).all()
    h.close()


def test_rule_contains_moved_spheres():
    spec = sample_images.random_spheres(spp=4)
    hs, h = host_scene(spec)
    bounds, right, prim = h.bvh_nodes(abi.RT_BVH_SAH)
    rng = np.random.default_rng(5)
    moved = (abi.RtHittable * len(hs))()
    C.memmove(moved, hs, C.sizeof(moved))
    leaves = prim[right < 0]
    for i in rng.choice(leaves, size=len(leaves) // 3, replace=False):
        o = moved[int(i)]
        for a in range(3):
            o.p[a] += rng.normal(0, 2.0)
        o.radius = abs(o.radius * rng.uniform(0.5, 2.0))
    boxes = refit_rule.refit(right, prim, moved)
    # every box contains every FP32 sphere below it, and its own children's boxes
    below = [[] for _ in range(len(right))]
    for i in range(len(right) - 1, -1, -1):
        below[i] = [int(prim[i])] if right[i] < 0 else below[i + 1] + below[right[i]]
    for i in range(len(right)):
        for k in below[i]:
            c = np.array(list(moved[k].p), np.float32).astype(np.float64)
            r = np.float64(np.float32(moved[k].radius))
            assert (boxes[i, :3] <= c - r).all() and (boxes[i, 3:] >= c + r).all(), (i, k)
    assert not np.array_equal(boxes.astype(np.float64), bounds)
    h.close()


def test_rule_leaf_box_is_the_directed_rounding():
    rng = np.random.default_rng(9)
    for _ in range(2000):
        c = rng.normal(0, 10 ** rng.uniform(-3, 4), 3)
        r = abs(rng.normal(0, 10 ** rng.uniform(-4, 3)))
        mn, mx = refit_rule.leaf_box(c, r)
        c32, r32 = c.astype(np.float32).astype(np.float64), np.float64(np.float32(r))
        lo, hi = c32 - r32, c32 + r32
        assert (mn.astype(np.float64) <= lo).all() and (mx.astype(np.float64) >= hi).all()
        # tight: the next float inwards would cut the sphere
        assert (np.nextafter(mn, np.float32(np.inf)).astype(np.float64) > lo).all()
        assert (np.nextafter(mx, np.float32(-np.inf)).astype(np.float64) < hi).all()
