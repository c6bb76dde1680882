"""bench.py on the device: --dump-outputs writes the frame of the last timed step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import scene_pair
from ray_tracing_fsharp_b200 import sample_images

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_hold_the_frame_of_the_last_timed_step(tmp_path):
    out_dir = tmp_path / "outputs"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "4", "--warmup", "1", "--config", "C1", "--spp", "16",
           "--half-extents", "40", "22", "--no-cpu-baseline", "--no-other-configs", "--no-hash", "--dump-outputs", str(out_dir)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=tmp_path)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["steps"] == 4 and d["warmup"] == 1 and d["value"] > 0
    dumped = d["dumped_outputs"]
    assert dumped["files"] == {"rgb.npy": [45, 81, 3], "sums.npy": [45, 81, 4]}
    assert sorted(os.listdir(out_dir)) == ["rgb.npy", "sums.npy"]
    rgb, sums = np.load(out_dir / "rgb.npy"), np.load(out_dir / "sums.npy")
    assert rgb.dtype == np.float32 and sums.dtype == np.float64
    # the same frame through rt_render, with the seed the last timed step used
    spec = sample_images.CONFIGS["C1"]()
    spec.max_width_coord, spec.max_height_coord, spec.spp = 40, 22, 16
    _osc, dsc, cam = scene_pair(spec)
    want_rgb, want_sums, _ = dsc.render(cam, 40, 22, seed=dumped["frame_seed"], adaptive=True, want_sums=True)
    assert np.array_equal(rgb, want_rgb) and np.array_equal(sums, want_sums)
    # another seed gives another frame: the dump is not some earlier frame that happens to match
    other, _, _ = dsc.render(cam, 40, 22, seed=dumped["frame_seed"] - 1, adaptive=True)
    assert not np.array_equal(rgb, other)
