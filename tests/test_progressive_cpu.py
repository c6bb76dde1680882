"""CPU-side checks of the progressive-frame surface (no GPU): RtFrameProgress's ctypes mirror against the header, the
no-device error of rt_frame_begin, and the tick distribution of Scene.render_progressive."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from ray_tracing_fsharp_b200 import abi, native, sample_images
from ray_tracing_fsharp_b200.domain import marshal
from ray_tracing_fsharp_b200.scene import ProgressTicks

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

FIELDS = ("samples_done", "samples_target", "paths_done", "paths_target", "pixels_flagged", "last_pass_ms", "device_ms", "passes", "done")


def test_frame_progress_mirror_matches_header_layout():
    src = "#include <stdio.h>\n#include <stddef.h>\n#include \"rtfs_b200.h\"\nint main(void) {\n"
    src += '  printf("%zu\\n", sizeof(RtFrameProgress));\n'
    for f in FIELDS:
        src += f'  printf("%zu\\n", offsetof(RtFrameProgress, {f}));\n'
    src += "  return 0; }\n"
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(td, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        got = [int(x) for x in subprocess.check_output([exe], text=True).split()]
    assert [f[0] for f in abi.RtFrameProgress._fields_] == list(FIELDS)
    assert got == [C.sizeof(abi.RtFrameProgress)] + [getattr(abi.RtFrameProgress, f).offset for f in FIELDS]


def test_frame_begin_without_a_device():
    spec = sample_images.few_spheres(max_w=20, max_h=10, spp=4)
    hs, ts, keep = marshal(spec.objects)
    h = native.SceneHandle(hs, ts, device=-1, keepalive=keep)
    cam = native.camera_make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    with pytest.raises(native.RtError) as e:
        h.open_frame(cam, spec.max_width_coord, spec.max_height_coord)
    assert e.value.code == abi.RT_ERR_NO_DEVICE
    h.close()


def test_progress_ticks_total_exactly_rows():
    rng = np.random.default_rng(0)
    for rows in (1, 3, 801, 2161):
        for _ in range(50):
            target = int(rng.integers(1, 10**12))
            done = np.sort(rng.integers(0, target, int(rng.integers(0, 40))))
            t = ProgressTicks(rows)
            emitted = [t.update(int(d), target) for d in done]
            assert all(n >= 0 for n in emitted)
            # the fractional part carries: after each update the total is floor(rows * done / target)
            assert list(np.cumsum(emitted)) == [rows * int(d) // target for d in done]
            assert sum(emitted) + t.finish() == rows
            assert t.finish() == 0


def test_progress_ticks_small_steps_carry():
    t = ProgressTicks(10)
    got = [t.update(d, 1000) for d in range(0, 1000, 7)]  # each step is 0.07 of a tick
    assert sum(got) == 10 * 994 // 1000 and max(got) == 1
    assert t.update(1000, 1000) == 10 - sum(got)  # reaching the target hands out the rest
    assert t.finish() == 0


def test_progress_ticks_whole_frame_at_once():
    t = ProgressTicks(801)
    assert t.update(0, 5) == 0
    assert t.update(5, 5) == 801
    assert t.update(7, 5) == 0
    assert t.finish() == 0
