"""CPU-side checks of the noise estimate (no GPU): the RtFrameNoise ctypes mirror against the header, the no-device error of
a frame opened with RT_FLAG_NOISE, rt_pixel_noise (the estimate's formula, shared with the device kernel) against a numpy
restatement, and the machine code of the render kernels: the kernels without the sum of squares are the instructions they
were before it existed, and the ones with it do not spill more than their counterparts."""
import ctypes as C
import hashlib
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile

import numpy as np
import pytest

if __name__ == "__main__":  # write-sass-digests, below
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ray_tracing_fsharp_b200 import abi, native, sample_images  # noqa: E402
from ray_tracing_fsharp_b200.domain import marshal  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "ray_tracing_fsharp_b200", "csrc", "build")
NVCC = "/usr/local/cuda/bin/nvcc"
CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"

FIELDS = ("pixels", "pixels_above", "max_se", "mean_se", "tolerance")


def numpy_se(sums, sq):
    """The estimate restated: D = n Q - sum_c T_c^2 in int64, E = sqrt(D / (3 n^2 (n - 1))) in float64, +inf where n < 2."""
    sums = np.asarray(sums).astype(np.int64)
    n = sums[..., 3]
    t = sums[..., :3]
    d = n * np.asarray(sq).astype(np.int64) - (t[..., 0] * t[..., 0] + t[..., 1] * t[..., 1] + t[..., 2] * t[..., 2])
    nd = n.astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        e = np.sqrt(d.astype(np.float64) / (3.0 * nd * nd * (n - 1).astype(np.float64)))
    return np.where(n < 2, np.inf, e)


def moments(values, counts):
    """Sums {T_r, T_g, T_b, n} and Q of pixels whose samples take value values[p, k, c] counts[p, k] times."""
    v = values.astype(np.int64)
    c = counts.astype(np.int64)
    n = c.sum(1)
    t = (v * c[:, :, None]).sum(1)
    q = (v * v * c[:, :, None]).sum((1, 2))
    return np.concatenate([t, n[:, None]], 1).astype(np.int32), q.astype(np.uint64)


def test_frame_noise_mirror_matches_header_layout():
    src = "#include <stdio.h>\n#include <stddef.h>\n#include \"rtfs_b200.h\"\nint main(void) {\n"
    src += '  printf("%zu\\n", sizeof(RtFrameNoise));\n'
    for f in FIELDS:
        src += f'  printf("%zu\\n", offsetof(RtFrameNoise, {f}));\n'
    src += '  printf("%d\\n", RT_FLAG_NOISE);\n  return 0; }\n'
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(td, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        got = [int(x) for x in subprocess.check_output([exe], text=True).split()]
    assert [f[0] for f in abi.RtFrameNoise._fields_] == list(FIELDS)
    assert got == [C.sizeof(abi.RtFrameNoise)] + [getattr(abi.RtFrameNoise, f).offset for f in FIELDS] + [abi.RT_FLAG_NOISE]


def test_noise_frame_without_a_device():
    spec = sample_images.few_spheres(max_w=20, max_h=10, spp=4)
    hs, ts, keep = marshal(spec.objects)
    h = native.SceneHandle(hs, ts, device=-1, keepalive=keep)
    cam = native.camera_make_basic(spec.spp, spec.focal_length, spec.aspect_ratio, spec.origin, spec.view_direction, spec.view_up)
    for flags in (abi.RT_FLAG_NOISE, abi.RT_FLAG_NOISE | abi.RT_FLAG_NO_SMEM):
        with pytest.raises(native.RtError) as e:
            h.open_frame(cam, spec.max_width_coord, spec.max_height_coord, flags=flags)
        assert e.value.code == abi.RT_ERR_NO_DEVICE
    h.close()


def test_frame_noise_null_frame():
    assert native.lib().rt_frame_noise(None, 1.0, None, None, None) == abi.RT_ERR_INVALID_ARGUMENT


def test_pixel_noise_random_moments():
    """Pixels of 1 to 300 samples drawn from [0, 255], and pixels of up to 2^22 samples spread over a few values."""
    rng = np.random.default_rng(5)
    small = rng.integers(0, 256, (4000, 300, 3))
    counts = (np.arange(300)[None, :] < rng.integers(1, 301, 4000)[:, None]).astype(np.int64)
    big_values = rng.integers(0, 256, (4000, 4, 3))
    big_counts = rng.multinomial(1 << 22, [0.25] * 4, 4000) // rng.integers(1, 5000, 4000)[:, None]
    for values, cnt in ((small, counts), (big_values, big_counts)):
        sums, sq = moments(values, cnt)
        want = numpy_se(sums, sq)
        got = native.pixel_noise(sums, sq)
        assert got.dtype == np.float32 and got.shape == sq.shape
        assert np.array_equal(got, want.astype(np.float32))
        assert np.isfinite(got[sums[:, 3] >= 2]).all()


def test_pixel_noise_extremes():
    n22 = 1 << 22
    values = np.array([
        [[0, 0, 0], [255, 255, 255]],      # 2^22 samples alternating 0 and 255: every term of D near its largest
        [[17, 200, 3], [17, 200, 3]],      # all samples equal: D = 0
        [[255, 255, 255], [0, 0, 0]],      # one sample: +inf
        [[0, 0, 0], [0, 0, 0]],            # no sample: +inf
        [[255, 0, 255], [255, 255, 0]],    # two samples
    ])
    counts = np.array([[n22 // 2, n22 // 2], [n22 - 5, 5], [1, 0], [0, 0], [1, 1]])
    sums, sq = moments(values, counts)
    got = native.pixel_noise(sums, sq)
    assert np.array_equal(got, numpy_se(sums, sq).astype(np.float32))
    # the alternating pixel: D = 3 255^2 2^42, E = 255 / (2 sqrt(2^22 - 1))
    assert int(sq[0]) * n22 - 3 * (255 * n22 // 2) ** 2 == 3 * 255 ** 2 * 2 ** 42
    assert got[0] == np.float32(255.0 / (2.0 * np.sqrt(n22 - 1.0)))
    assert got[1] == 0.0 and np.isinf(got[2]) and np.isinf(got[3])
    assert got[4] == np.float32(np.sqrt(2 * 255.0 ** 2 / 12.0))  # T = (510, 255, 255), Q = 4 255^2: D = 2 255^2
    # shapes of a frame: [rows, cols, 4] and [rows, cols]
    frame_sums = np.broadcast_to(sums[0], (3, 5, 4))
    assert np.array_equal(native.pixel_noise(frame_sums, np.full((3, 5), sq[0])), np.full((3, 5), got[0]))
    with pytest.raises(ValueError):
        native.pixel_noise(sums[:2], sq)


# ---- machine code -------------------------------------------------------------------------------------------------------
# tests/golden/render_kernels_sass.json: SHA-256 of the SASS (cuobjdump -sass, instruction lines) of every kernel of
# rtfs_device.cu as compiled before the noise estimate existed, with the nvcc that compiled them.  render_kernel's trailing
# NOISE parameter changes the kernels' names: a name with NOISE = false maps back to the five-parameter name.
# The digests belong to one compiler: with another nvcc the comparison is skipped, and says so.  To take them again (after a
# toolkit change, or a deliberate change to the render kernels), build rtfs_device.cu of the reference commit with that
# nvcc (make -C ray_tracing_fsharp_b200/csrc) and run
#     python tests/test_noise_cpu.py write-sass-digests <that build>/rtfs_device.cu.o
# The build products are what build() leaves in csrc/build: where the library is built they must be there, and a test
# that misses them fails rather than skips.
SASS_GOLDEN = os.path.join(ROOT, "tests", "golden", "render_kernels_sass.json")


def _demangle(names):
    out = subprocess.check_output(["c++filt"], input="\n".join(names), text=True).split("\n")
    return dict(zip(names, out))


def sass_functions(obj):
    """{kernel name without NOISE = false: instruction text} of a device object; the NOISE = true kernels are left out."""
    text = subprocess.check_output([CUOBJDUMP, "-sass", obj], text=True)
    body, cur = {}, None
    for line in text.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            body[cur] = []
        elif cur and line.strip():
            body[cur].append(line)
    out = {}
    for mangled, name in _demangle(list(body)).items():
        m = re.match(r"void rtfs::render_kernel<(.*)>\(rtfs::FrameParams\)$", name)
        if m:
            args = m.group(1).split(", ")
            if len(args) == 6:
                if args[5] == "true":
                    continue
                name = "void rtfs::render_kernel<" + ", ".join(args[:5]) + ">(rtfs::FrameParams)"
        out[name] = "\n".join(body[mangled])
    return out


def _nvcc_version():
    return subprocess.check_output([NVCC, "--version"], text=True).strip().splitlines()[-1]


def _build_product(name):
    """A file build() leaves in csrc/build (make keeps the objects and ptxas -v logs there), and the tools to read it."""
    path = os.path.join(BUILD, name)
    if not os.path.exists(path):
        pytest.fail(f"{path} is missing: build the library with __graft_entry__.build() (make -C ray_tracing_fsharp_b200/csrc), "
                    "which keeps its objects and ptxas logs in csrc/build")
    if not os.path.exists(CUOBJDUMP) or not shutil.which("c++filt"):
        pytest.fail(f"{CUOBJDUMP} (CUDA toolkit) and c++filt (binutils) are needed to read the machine code")
    return path


def write_sass_digests(obj, path=SASS_GOLDEN):
    """Writes the digests of the kernels of the device object `obj`, with the version of the nvcc at NVCC."""
    doc = {"nvcc": _nvcc_version(), "object": "rtfs_device.cu.o",
           "kernels": {k: hashlib.sha256(v.encode()).hexdigest() for k, v in sorted(sass_functions(obj).items())}}
    with open(path, "w") as fh:
        json.dump(doc, fh, indent=1)


def test_kernels_without_noise_are_unchanged():
    obj = _build_product("rtfs_device.cu.o")
    golden = json.load(open(SASS_GOLDEN))
    if _nvcc_version() != golden["nvcc"]:
        pytest.skip(f"the digests were taken with {golden['nvcc']}, this nvcc is {_nvcc_version()}: take them again "
                    "(see the comment above SASS_GOLDEN)")
    got = {k: hashlib.sha256(v.encode()).hexdigest() for k, v in sass_functions(obj).items()}
    assert sum("render_kernel" in k for k in golden["kernels"]) == 24
    assert set(got) == set(golden["kernels"])
    changed = sorted(k for k in got if got[k] != golden["kernels"][k])
    assert not changed, f"machine code changed: {changed}"


def _ptxas_report():
    """{demangled kernel: (registers, spill store bytes, spill load bytes)} from the build's ptxas -v log."""
    log = _build_product("rtfs_device.ptxas.log")
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
    names = _demangle(list(info))
    return {names[k]: tuple(v) for k, v in info.items()}


def test_noise_kernels_registers_and_spills():
    """The 12 kernels with the sum of squares (the lockstep kernels without counters, probe and main phase) keep their
    counterparts' register budget (64 staged, 40 global: the launch bounds) and spill at most 16 bytes more.  (The global
    kernels spill a few hundred bytes under their 40-register bound, with or without the sum; those spills lie outside the
    walk loop, DESIGN.md 5.)"""
    rep = _ptxas_report()
    pat = re.compile(r"void rtfs::render_kernel<(true|false), (\d), (true|false), (true|false), (true|false), (true|false)>\(rtfs::FrameParams\)$")
    kernels = {}
    for name, v in rep.items():
        m = pat.match(name)
        if m:
            kernels[m.groups()] = v
    noisy = sorted(k for k in kernels if k[5] == "true")
    assert len(noisy) == 12 and len(kernels) == 36
    assert all(k[2] == "false" for k in noisy)  # no counting variant
    for k in noisy:
        regs, st, ld = kernels[k]
        base_regs, base_st, base_ld = kernels[k[:5] + ("false",)]
        assert regs == base_regs == (40 if k[1] == "0" else 64), k
        assert st <= base_st + 16 and ld <= base_ld + 16, (k, (st, ld), (base_st, base_ld))


if __name__ == "__main__" and len(sys.argv) == 3 and sys.argv[1] == "write-sass-digests":
    write_sass_digests(sys.argv[2])
