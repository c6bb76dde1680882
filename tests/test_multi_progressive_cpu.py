"""CPU-side checks of progressive frames over several GPUs (no GPU): the prototype against the header and the ctypes
declaration, the ABI version it leaves as it was, the refusals of a null handle or output that come before any device work,
and the machine code of the exchange kernel: no spills, and at most 64 registers a thread."""
import ctypes as C
import os
import subprocess
import tempfile

from ray_tracing_fsharp_b200 import abi, native, sample_images

from test_noise_cpu import _build_product
from test_window_cpu import _header_args, _kernel_report

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_prototype_matches_header():
    src = r'''
#include <stdio.h>
#include "rtfs_b200.h"
int main(void) {
    int (*b)(RtMulti *, const RtCamera *, int32_t, int32_t, const RtRenderOpts *, RtFrame **, RtFrameProgress *) = rt_multi_frame_begin;
    printf("%d %d\n", RT_ABI_VERSION, b != 0);
    return 0;
}
'''
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "p.c")
        open(c, "w").write(src)
        subprocess.check_call(["gcc", "-Werror", "-Wincompatible-pointer-types", "-I", os.path.join(ROOT, "include"), "-c", c, "-o",
                               os.path.join(td, "p.o")])
    assert _header_args("rt_multi_frame_begin") == 7 and len(native.lib().rt_multi_frame_begin.argtypes) == 7
    assert "rt_multi_frame_begin" in native.EXPORTS
    # the feature only adds a function: the version callers compare is unchanged
    assert abi.RT_ABI_VERSION == 6 and native.lib().rt_abi_version() == 6


def test_null_handle_or_output_is_refused_before_any_device_work():
    spec = sample_images.few_spheres(max_w=20, max_h=10, spp=4)
    cam = native.camera_make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    lib = native.lib()
    for flags in (0, abi.RT_FLAG_NOISE):
        opts = abi.RtRenderOpts(1, 1, abi.RT_MODE_MEGAKERNEL, 0, flags)
        out = C.c_void_p(12345)  # a stale value the call must clear
        assert lib.rt_multi_frame_begin(None, C.byref(cam), 20, 10, C.byref(opts), C.byref(out), None) == abi.RT_ERR_INVALID_ARGUMENT
        assert out.value is None
        assert lib.rt_multi_frame_begin(None, C.byref(cam), 20, 10, C.byref(opts), None, None) == abi.RT_ERR_INVALID_ARGUMENT
        assert "null" in lib.rt_last_error().decode()


def test_gather_kernel_registers_and_spills():
    kernels = _kernel_report(_build_product("rtfs_multi.ptxas.log"))
    names = {n.replace("(anonymous namespace)::", "").split("(")[0].replace("void ", ""): v for n, v in kernels.items()}
    assert "rtfs::gather_kernel" in names, sorted(names)
    regs, st, ld = names["rtfs::gather_kernel"]
    assert st == 0 and ld == 0, (st, ld)
    assert regs <= 64, regs  # 256 threads a block: four such blocks a SM stay resident
