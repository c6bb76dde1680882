"""CPU-side checks of saving and resuming progressive frames (no GPU): the three prototypes and the snapshot header against
the header file and the ctypes declarations, the exports, the ABI version they leave as it was, the refusals that come before
any device work (null arguments, a host-only scene, a damaged snapshot), the machine code of the two new kernels, and the
format restated in tests/snapshot_rule.py: a parse / write round trip and the checksum's properties."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import snapshot_rule as rule
from ray_tracing_fsharp_b200 import abi, native, sample_images
from ray_tracing_fsharp_b200.domain import marshal

from test_noise_cpu import _build_product
from test_window_cpu import _header_args, _kernel_report

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_prototypes_and_header_layout_match():
    src = r'''
#include <stddef.h>
#include <stdio.h>
#include "rtfs_b200.h"
int main(void) {
    int (*s)(RtFrame *, void *, size_t, size_t *) = rt_frame_save;
    int (*r)(RtScene *, const void *, size_t, RtFrame **, RtFrameProgress *) = rt_frame_resume;
    int (*m)(RtMulti *, const void *, size_t, RtFrame **, RtFrameProgress *) = rt_multi_frame_resume;
    printf("%d %d %zu %zu %zu %zu %zu\n", RT_ABI_VERSION, RT_SNAPSHOT_VERSION, sizeof(RtSnapshotHeader), offsetof(RtSnapshotHeader, checksum),
           offsetof(RtSnapshotHeader, opts), offsetof(RtSnapshotHeader, n_pixels), offsetof(RtSnapshotHeader, ms_per_sample));
    return !(s && r && m);
}
'''
    with tempfile.TemporaryDirectory() as td:
        c, exe = os.path.join(td, "p.c"), os.path.join(td, "p")
        open(c, "w").write(src)
        subprocess.check_call(["gcc", "-Werror", "-Wincompatible-pointer-types", "-I", os.path.join(ROOT, "include"), c, "-o", exe,
                               "-Wl,--unresolved-symbols=ignore-all"])
        got = subprocess.run([exe], capture_output=True, text=True).stdout.split()
    h = abi.RtSnapshotHeader
    assert got == [str(x) for x in (6, abi.RT_SNAPSHOT_VERSION, C.sizeof(h), h.checksum.offset, h.opts.offset, h.n_pixels.offset,
                                    h.ms_per_sample.offset)]
    assert C.sizeof(h) == rule.HEADER_BYTES == 344
    for name, n in (("rt_frame_save", 4), ("rt_frame_resume", 5), ("rt_multi_frame_resume", 5)):
        assert _header_args(name) == n and len(getattr(native.lib(), name).argtypes) == n
    assert {"rt_frame_save", "rt_frame_resume", "rt_multi_frame_resume"} <= set(native.EXPORTS)
    # the feature only adds functions and a struct: the version callers compare is unchanged
    assert abi.RT_ABI_VERSION == 6 and native.lib().rt_abi_version() == 6


def test_null_arguments_are_refused_before_any_device_work():
    lib = native.lib()
    n = C.c_size_t(7)
    assert lib.rt_frame_save(None, None, 0, C.byref(n)) == abi.RT_ERR_INVALID_ARGUMENT
    assert "null" in lib.rt_last_error().decode()
    data = rule.synthetic()
    for fn in (lib.rt_frame_resume, lib.rt_multi_frame_resume):
        out = C.c_void_p(12345)  # a stale value the call must clear
        assert fn(None, data, len(data), C.byref(out), None) == abi.RT_ERR_INVALID_ARGUMENT
        assert out.value is None
        assert fn(None, data, len(data), None, None) == abi.RT_ERR_INVALID_ARGUMENT
        assert "null" in lib.rt_last_error().decode()


def test_a_host_only_scene_is_refused():
    spec = sample_images.few_spheres(max_w=20, max_h=10, spp=4)
    hs, ts, keep = marshal(spec.objects)
    scene = native.SceneHandle(hs, ts, -1, keepalive=keep)  # device = -1: no device work ever
    out = C.c_void_p(12345)
    data = rule.synthetic()
    assert native.lib().rt_frame_resume(scene.ptr, data, len(data), C.byref(out), None) == abi.RT_ERR_UNSUPPORTED
    assert out.value is None
    with pytest.raises(native.RtError) as e:
        scene.resume_frame(data)
    assert e.value.code == abi.RT_ERR_UNSUPPORTED


def test_snapshot_kernels_registers_and_spills():
    kernels = _kernel_report(_build_product("rtfs_snapshot.ptxas.log"))
    for name in ("snapshot_pack_kernel", "snapshot_unpack_kernel"):
        found = [v for k, v in kernels.items() if name in k]
        assert len(found) == 1, sorted(kernels)
        regs, st, ld = found[0]
        assert st == 0 and ld == 0, (name, st, ld)
        assert regs <= 64, (name, regs)  # 256 threads a block: several blocks a SM stay resident


@pytest.mark.parametrize("noise", [False, True])
@pytest.mark.parametrize("kind,n_views,n_pixels", [(abi.RT_FRAME_CAMERA, 1, 1), (abi.RT_FRAME_CAMERA, 1, 150), (abi.RT_FRAME_VIEWS, 3, 192),
                                                   (abi.RT_FRAME_WINDOW, 1, 64)])
def test_parse_and_write_round_trip(kind, n_views, n_pixels, noise):
    data = rule.synthetic(n_pixels, noise, kind, n_views)
    parts = rule.parse(data)
    h = parts["header"]
    assert (h.kind, h.n_views, h.n_pixels, h.total_bytes) == (kind, n_views, n_pixels, len(data))
    assert len(data) % 8 == 0 and h.checksum == rule.checksum(data)
    assert (parts["sq"] is not None) == noise and parts["sums"].shape == (n_pixels, 4)
    assert len(parts["cameras"]) == (n_views if kind == abi.RT_FRAME_VIEWS else 0)
    assert rule.write(parts) == data


def test_checksum_changes_with_any_flipped_bit():
    data = rule.synthetic(150, True)
    base = rule.checksum(data)
    rng = np.random.default_rng(1)
    skip = range(8 * rule.CHECKSUM_WORD, 8 * rule.CHECKSUM_WORD + 8)
    positions = [b for b in list(range(len(data))) if b not in skip]
    for byte in list(positions[:64]) + list(rng.choice(positions, 400, replace=False)) + [len(data) - 1]:
        for bit in (0, 3, 7):
            flipped = bytearray(data)
            flipped[byte] ^= 1 << bit
            assert rule.checksum(bytes(flipped)) != base, (byte, bit)
    # the checksum field itself is read as zero
    flipped = bytearray(data)
    flipped[8 * rule.CHECKSUM_WORD] ^= 1
    assert rule.checksum(bytes(flipped)) == base
    # the sum does not depend on the order its terms are added in, but a term does depend on its word's position
    w = np.frombuffer(data, "<u8").copy()
    w[rule.CHECKSUM_WORD] = 0
    i = np.arange(w.size, dtype=np.uint64)
    perm = rng.permutation(w.size)
    with np.errstate(over="ignore"):
        assert int(rule.mix(i[perm], w[perm]).sum(dtype=np.uint64)) == base
    swapped = w.copy()
    swapped[[50, 51]] = swapped[[51, 50]]
    if swapped[50] != swapped[51]:
        with np.errstate(over="ignore"):
            assert int(rule.mix(i, swapped).sum(dtype=np.uint64)) != base
