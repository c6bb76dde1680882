"""CPU-side checks of structural scene edits (no GPU): the prototype and the RtSceneRebuild mirror against the header, the
errors a call gets without a device or on a host-only scene, the registers and spills of the builder's kernels, and
tests/ploc_rule.py, the numpy restatement of the device builder: on C1-C5 every sphere is in exactly one leaf, every box
contains what lies below it, the tree does not depend on the order in which the array was reached, and the depth is reported.
Its SAH cost is printed next to the host SAH tree's (not asserted)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from ray_tracing_fsharp_b200 import abi, native, sample_images
from ray_tracing_fsharp_b200.domain import marshal

import ploc_rule
from test_noise_cpu import _build_product
from test_window_cpu import _header_args, _kernel_report

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("objects_removed", "objects_appended", "n_objects", "n_bounded", "nodes", "depth", "on_device", "launches", "generation",
          "device_ms")


def test_prototype_matches_header():
    src = r'''
#include <stdio.h>
#include "rtfs_b200.h"
int main(void) {
    int (*r)(RtScene *, const int32_t *, int32_t, const RtHittable *, int32_t, RtSceneRebuild *) = rt_scene_rebuild;
    printf("%d %d\n", RT_ABI_VERSION, r != 0);
    return 0;
}
'''
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "p.c")
        open(c, "w").write(src)
        subprocess.check_call(["gcc", "-Werror", "-Wincompatible-pointer-types", "-I", os.path.join(ROOT, "include"), "-c", c, "-o",
                               os.path.join(td, "p.o")])
    assert _header_args("rt_scene_rebuild") == 6 and len(native.lib().rt_scene_rebuild.argtypes) == 6
    assert "rt_scene_rebuild" in native.EXPORTS
    assert abi.RT_ABI_VERSION == 6 and native.lib().rt_abi_version() == 6


def test_scene_rebuild_mirror_matches_header_layout():
    src = "#include <stdio.h>\n#include <stddef.h>\n#include \"rtfs_b200.h\"\nint main(void) {\n"
    src += '  printf("%zu\\n", sizeof(RtSceneRebuild));\n'
    for f in FIELDS:
        src += f'  printf("%zu\\n", offsetof(RtSceneRebuild, {f}));\n'
    src += "  return 0; }\n"
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(td, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        got = [int(x) for x in subprocess.check_output([exe], text=True).split()]
    assert [f[0] for f in abi.RtSceneRebuild._fields_] == list(FIELDS)
    assert got == [C.sizeof(abi.RtSceneRebuild)] + [getattr(abi.RtSceneRebuild, f).offset for f in FIELDS]


def test_without_a_device():
    lib = native.lib()
    spec = sample_images.few_spheres(max_w=20, max_h=10, spp=4)
    hs, ts, keep = marshal(spec.objects)
    h = native.SceneHandle(hs, ts, device=-1, keepalive=keep)
    with pytest.raises(native.RtError) as e:
        h.rebuild([0], [])
    assert e.value.code == abi.RT_ERR_UNSUPPORTED
    with pytest.raises(native.RtError) as e:
        h.rebuild()
    assert e.value.code == abi.RT_ERR_UNSUPPORTED
    # argument errors come first
    one = np.zeros(1, np.int32)
    assert lib.rt_scene_rebuild(None, None, 0, None, 0, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_scene_rebuild(h.ptr, None, -1, None, 0, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_scene_rebuild(h.ptr, None, 0, None, -1, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_scene_rebuild(h.ptr, None, 1, None, 0, None) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_scene_rebuild(h.ptr, native.ptr(one), 0, None, 1, None) == abi.RT_ERR_INVALID_ARGUMENT
    h.close()
    if native.device_count() == 0:
        with pytest.raises(native.RtError) as e:
            native.SceneHandle(hs, ts, device=0, keepalive=keep)
        assert e.value.code == abi.RT_ERR_NO_DEVICE


def test_builder_kernels_registers_and_spills():
    kernels = _kernel_report(_build_product("rtfs_build.ptxas.log"))
    names = {n.split("(")[0].replace("void ", ""): v for n, v in kernels.items() if "rtfs::" in n.split("(")[0] and "cub" not in n.split("(")[0]}
    ours = {"rtfs::rebuild_mark_kernel", "rtfs::rebuild_collect_kernel", "rtfs::rebuild_keys_kernel", "rtfs::ploc_init_kernel",
            "rtfs::ploc_nearest_kernel", "rtfs::ploc_merge_kernel", "rtfs::ploc_flatten_kernel", "rtfs::ploc_single_kernel",
            "rtfs::rebuild_place_unbounded_kernel", "rtfs::scan_top_kernel"}
    assert ours <= set(k.split("<")[0] for k in names), sorted(names)
    for k, (regs, st, ld) in names.items():
        assert st == 0 and ld == 0, (k, st, ld)
        limit = 64 if "scan" in k else 128  # the scans run 1024 threads a block, the others 256
        assert regs <= limit, (k, regs)


# ---- the rule -------------------------------------------------------------------------------------------------------------------
SPECS = {
    "C1": lambda: sample_images.few_spheres(max_w=20, max_h=10, spp=4),
    "C2": lambda: sample_images.random_spheres(spp=4),
    "C3": lambda: sample_images.earth(max_w=20, max_h=10, spp=4),
    "C4": lambda: sample_images.mixed_planes(max_w=20, max_h=10, spp=4),
    "C5": lambda: sample_images.many_spheres(n=100_000, max_w=20, max_h=10, spp=4),
}


def check_tree(objects, bounds, right, prim, depth):
    n = len(right)
    spheres = [i for i in range(len(objects)) if objects[i].shape == abi.RT_SHAPE_SPHERE and objects[i].radius >= 0]
    assert sorted(prim[prim >= 0].tolist()) == spheres  # every sphere in exactly one leaf
    assert (prim[right >= 0] == -1).all() and (right[right >= 0] > np.nonzero(right >= 0)[0]).all()
    # every box contains its children's (and so everything below it); a leaf's box contains its FP32 sphere
    inner = np.nonzero(right >= 0)[0]
    for kids in (inner + 1, right[inner]):
        assert (bounds[inner, :3] <= bounds[kids, :3]).all() and (bounds[inner, 3:] >= bounds[kids, 3:]).all()
    for i in np.nonzero(right < 0)[0]:
        h = objects[int(prim[i])]
        c = np.array(list(h.p), np.float32).astype(np.float64)
        r = np.float64(np.float32(h.radius))
        assert (bounds[i, :3] <= c - r).all() and (bounds[i, 3:] >= c + r).all()
    # the depth in internal nodes, root 1
    d = np.zeros(n, np.int64)
    if n:
        d[0] = 1
    for i in range(n):
        if right[i] >= 0:
            d[i + 1] = d[right[i]] = d[i] + 1
    assert depth == (int(d[right >= 0].max()) if len(inner) else (1 if n else 0))


@pytest.mark.parametrize("name", sorted(SPECS))
def test_rule_tree_properties_and_sah_cost(name):
    hs, ts, keep = marshal(SPECS[name]().objects)
    objects = [hs[i] for i in range(len(hs))]
    bounds, right, prim, depth = ploc_rule.build(objects)
    check_tree(objects, bounds, right, prim, depth)
    host = native.SceneHandle(hs, ts, device=-1, keepalive=keep)
    hb, hr, hp = host.bvh_nodes(abi.RT_BVH_SAH)
    host.close()
    ploc, sah = ploc_rule.sah_cost(bounds, right), ploc_rule.sah_cost(hb, hr)
    print(f"{name}: {len(prim[prim >= 0])} spheres, PLOC depth {depth}, SAH cost {ploc:.3f} against the host tree's {sah:.3f} "
          f"(ratio {ploc / sah if sah else float('nan'):.3f})")


def test_rule_is_a_function_of_the_array_alone():
    hs, ts, keep = marshal(SPECS["C2"]().objects)
    objects = [hs[i] for i in range(len(hs))]
    a = ploc_rule.build(objects)
    # the same array reached from a shuffled copy by putting the records back: equal records give an equal tree
    rng = np.random.default_rng(4)
    perm = rng.permutation(len(objects))
    shuffled = [objects[i] for i in perm]
    back = [None] * len(objects)
    for k, i in enumerate(perm):
        back[i] = shuffled[k]
    b = ploc_rule.build(back)
    assert all(np.array_equal(x, y) for x, y in zip(a[:3], b[:3])) and a[3] == b[3]
    # a different order of the same spheres is a different array: the leaves' caller indices follow it
    c = ploc_rule.build(shuffled)
    assert sorted(perm[c[2][c[2] >= 0]].tolist()) == sorted(a[2][a[2] >= 0].tolist())


def test_rule_edge_cases():
    hs, ts, keep = marshal(SPECS["C4"]().objects)
    objects = [hs[i] for i in range(len(hs))]
    unb = [o for o in objects if o.shape != abi.RT_SHAPE_SPHERE]
    sph = [o for o in objects if o.shape == abi.RT_SHAPE_SPHERE and o.radius >= 0]
    b, r, p, d = ploc_rule.build(unb)
    assert len(b) == 0 and d == 0
    b, r, p, d = ploc_rule.build(unb + sph[:1])
    assert len(b) == 1 and r[0] == -1 and p[0] == len(unb) and d == 1
    b, r, p, d = ploc_rule.build(sph[:2])
    assert list(r) == [2, -1, -1] and d == 1


def test_rule_nested_chain_is_deeper_than_the_walk_stacks():
    hs, ts, keep = marshal(SPECS["C1"]().objects)
    base = [hs[i] for i in range(len(hs)) if hs[i].shape == abi.RT_SHAPE_SPHERE][0]
    chain = []
    for i in range(70):
        o = abi.RtHittable()
        C.memmove(C.byref(o), C.byref(base), C.sizeof(o))
        o.p[0], o.p[1], o.p[2] = 0.25, 0.5, -2.0
        o.radius = 1e-4 * 1.3 ** i
        chain.append(o)
    b, r, p, d = ploc_rule.build(chain)
    assert d == 69  # one merge per iteration: a chain
