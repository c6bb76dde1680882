"""CPU-side checks of the convergence rule of progressive frames (no GPU): RtFrameConvergence's ctypes mirror against the
header, the no-device error, the null-frame errors, ProgressTicks under a target that shrinks, and the numpy restatement of
the rule (convergence_rule.py) that the GPU tests compare frames with."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from convergence_rule import checkpoints, converge, next_checkpoint, numpy_se, probe
from ray_tracing_fsharp_b200 import abi, native, sample_images
from ray_tracing_fsharp_b200.domain import marshal
from ray_tracing_fsharp_b200.scene import ProgressTicks, Scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

FIELDS = ("tolerance", "min_samples", "interval", "next_check", "checks", "pixels_active", "pixels_converged")


def test_frame_convergence_mirror_matches_header_layout():
    src = "#include <stdio.h>\n#include <stddef.h>\n#include \"rtfs_b200.h\"\nint main(void) {\n"
    src += '  printf("%zu\\n", sizeof(RtFrameConvergence));\n'
    for f in FIELDS:
        src += f'  printf("%zu\\n", offsetof(RtFrameConvergence, {f}));\n'
    src += '  printf("%d\\n", RT_ABI_VERSION);\n  return 0; }\n'
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(td, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        got = [int(x) for x in subprocess.check_output([exe], text=True).split()]
    assert [f[0] for f in abi.RtFrameConvergence._fields_] == list(FIELDS)
    assert got == [C.sizeof(abi.RtFrameConvergence)] + [getattr(abi.RtFrameConvergence, f).offset for f in FIELDS] + [abi.RT_ABI_VERSION]


def test_converging_frame_without_a_device():
    spec = sample_images.few_spheres(max_w=20, max_h=10, spp=4)
    hs, ts, keep = marshal(spec.objects)
    h = native.SceneHandle(hs, ts, device=-1, keepalive=keep)
    cam = native.camera_make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    s = Scene(h, hs, ts, keep, [-1])
    with pytest.raises(native.RtError) as e:
        Scene.render_progressive(lambda _: None, lambda _: None, spec.max_width_coord, spec.max_height_coord, cam, s, seed=1,
                                 converge_tolerance=1.0)
    assert e.value.code == abi.RT_ERR_NO_DEVICE
    h.close()


def test_convergence_null_frame():
    lib = native.lib()
    out = abi.RtFrameConvergence()
    assert lib.rt_frame_set_convergence(None, 1.0, 64, 64) == abi.RT_ERR_INVALID_ARGUMENT
    assert lib.rt_frame_convergence(None, C.byref(out)) == abi.RT_ERR_INVALID_ARGUMENT


def test_progress_ticks_with_a_shrinking_target():
    """paths_target of a converging frame drops at every check (paths_done + active (target - samples_done)) and never
    grows; the ticks still never go negative and total `rows`."""
    rng = np.random.default_rng(1)
    for rows in (1, 45, 801, 2161):
        for _ in range(50):
            n, spp, step = int(rng.integers(1, 10**6)), int(rng.integers(64, 4096)), int(rng.integers(1, 64))
            active, done, paths = n, 0, 0
            t = ProgressTicks(rows)
            emitted, targets = [], []
            while done < spp and active:
                k = min(step, spp - done)
                paths += active * k
                done += k
                active = int(active * rng.random()) if rng.random() < 0.5 else active
                targets.append(paths + active * (spp - done))
                emitted.append(t.update(paths, targets[-1]))
            assert all(a >= b for a, b in zip(targets, targets[1:]))
            assert all(e >= 0 for e in emitted)
            assert sum(emitted) + t.finish() == rows


# ---- the numpy restatement ---------------------------------------------------------------------------------------------
def test_checkpoint_lattice():
    assert checkpoints(64, 64, 500) == [64, 128, 192, 256, 320, 384, 448]
    assert checkpoints(64, 64, 63) == [] and checkpoints(64, 64, 64) == [64]
    assert checkpoints(16, 8, 40) == [16, 24, 32, 40]
    for m, k in ((2, 1), (16, 8), (64, 64), (100, 7)):
        for s in range(0, 400):
            c = next_checkpoint(m, k, s)
            assert c > s and (c - m) % k == 0 and c >= m
            assert c - k <= s or c == m  # the first one above s


def random_colours(n, spp, seed):
    """[n, spp, 3] uint8 samples: a third of the pixels constant (sky), a third low noise, a third high noise."""
    rng = np.random.default_rng(seed)
    base = rng.integers(20, 230, (n, 1, 3))
    spread = np.where(np.arange(n)[:, None, None] % 3 == 0, 0, np.where(np.arange(n)[:, None, None] % 3 == 1, 4, 120))
    return np.clip(base + rng.integers(-1, 2, (n, spp, 3)) * spread + rng.integers(0, 2, (n, spp, 3)) * (spread > 0), 0, 255).astype(np.uint8)


def moments_of(colours):
    def moments(idx, s0, s1):
        c = colours[idx, s0:s1].astype(np.int64)
        return c.sum(1), (c * c).sum((1, 2))
    return moments


def e_at(moments, p, d):
    """E of pixel p over samples [0, d)."""
    t, q = moments(np.array([p]), 0, d)
    return numpy_se(np.append(t[0], d)[None], q)[0]


@pytest.mark.parametrize("adaptive", [True, False])
def test_rule_restated(adaptive):
    """Every pixel holds [0, n_p) with n_p the probe, the first checkpoint where E <= tolerance, or samples_done."""
    n, spp, m, k = 600, 200, 16, 24
    colours = random_colours(n, spp, 2)
    moments = moments_of(colours)
    s0, q0, n_probe, flagged = probe(moments, n, spp, adaptive)
    for tol in (0.0, 0.5, 2.0, 10.0, np.inf):
        for done in (n_probe, m - 1, m, m + 5, m + k, 150, spp):
            sums, q, active, checks = converge(moments, s0, q0, flagged, done, tol, m, k)
            n_p = sums[:, 3]
            want_s, want_q = moments(np.arange(n), 0, 0)
            for p in range(n):
                t, qq = moments(np.array([p]), 0, int(n_p[p]))
                want_s[p], want_q[p] = t[0], qq[0]
            assert np.array_equal(sums[:, :3], want_s) and np.array_equal(q, want_q)
            assert (n_p[~flagged] == n_probe).all()
            stopped = flagged & ~active
            if active.any():
                assert (n_p[active] == done).all()
                assert checks == len(checkpoints(m, k, done))
            for p in np.flatnonzero(stopped):
                c = int(n_p[p])
                assert c in checkpoints(m, k, done)
                e = [e_at(moments, p, d) for d in checkpoints(m, k, c)]
                assert e[-1] <= tol and all(x > tol for x in e[:-1])  # converged at c, at no earlier checkpoint
            if tol == 0.0 and adaptive:
                # a flagged pixel's two probe means differ, so its samples are not all equal: E > 0 forever
                assert (active == flagged).all()
            if tol == 0.0 and not adaptive and done >= m:
                assert (~active == (colours[:, :m] == colours[:, :1]).all((1, 2))).all()
