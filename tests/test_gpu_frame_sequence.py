"""Every render entry point drives a frame through the same sequence (csrc/rtfs_device.h: frame_probe, frame_main,
frame_finish): the same frame through rt_render, a one-rank communicator, a one-device MultiHandle and the wavefront mode
gives the same image, the same counts and the same launches."""
import numpy as np
import pytest

from helpers import scene_pair, small_random_spheres
from ray_tracing_fsharp_b200 import abi, native
from ray_tracing_fsharp_b200.domain import marshal

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def frame():
    spec = small_random_spheres()
    _osc, dsc, cam = scene_pair(spec)
    hs, ts, keep = marshal(spec.objects)
    multi = native.MultiHandle(hs, ts, devices=(0,), keepalive=keep)
    yield spec, dsc, cam, multi
    multi.close()
    dsc.close()


@pytest.mark.parametrize("adaptive", [True, False])
def test_one_device_multi_render_equals_rt_render(frame, adaptive):
    spec, dsc, cam, multi = frame
    mw, mh = spec.max_width_coord, spec.max_height_coord
    for gamma in (False, True):
        want_rgb, want_sums, want = dsc.render(cam, mw, mh, seed=17, adaptive=adaptive, gamma=gamma, want_sums=True)
        want_rgb, want_sums = want_rgb.copy(), want_sums.copy()
        rgb, sums, got = multi.render(cam, mw, mh, seed=17, adaptive=adaptive, gamma=gamma, want_sums=True)
        assert np.array_equal(rgb, want_rgb) and np.array_equal(sums, want_sums)
        assert (got.paths, got.rays, got.pixels_early_out) == (want.paths, want.rays, want.pixels_early_out)
    if adaptive:
        assert 0 < want.pixels_early_out < (2 * mw + 1) * (2 * mh + 1)


@pytest.mark.parametrize("adaptive", [True, False])
def test_entry_points_issue_the_same_launches(frame, adaptive):
    spec, dsc, cam, multi = frame
    mw, mh = spec.max_width_coord, spec.max_height_coord
    n_pixels = (2 * mw + 1) * (2 * mh + 1)
    # probe + flags + compact + main + tail; without the early-out compact + main + tail (the main phase fits one launch)
    want = 5 if adaptive else 3
    _, want_sums, st = dsc.render(cam, mw, mh, seed=5, adaptive=adaptive, want_sums=True)
    want_sums = want_sums.copy()
    comm = native.CommHandle(None, 0, 1, 0)
    try:
        _, sums_c, st_c = comm.render(dsc, cam, mw, mh, seed=5, adaptive=adaptive, want_sums=True)
    finally:
        comm.close()
    _, sums_m, st_m = multi.render(cam, mw, mh, seed=5, adaptive=adaptive, want_sums=True)
    assert np.array_equal(sums_c, want_sums) and np.array_equal(sums_m, want_sums)
    assert (st.launches, st_c.launches, st_m.launches) == (want, want, want)
    for s in (st, st_c):
        assert 0 < s.main_ms <= s.kernel_ms <= s.total_ms
    assert 0 < st_m.kernel_ms <= st_m.total_ms

    # the wavefront mode at bounce depth 0: one generate + extend + shade per phase (one batch each), then the probe
    # flags, the compaction and the tail; the main phase only if a pixel is flagged
    cam0 = type(cam).from_buffer_copy(cam)
    cam0.bounce_depth = 0
    _, _, want_wf = dsc.render(cam0, mw, mh, seed=5, adaptive=adaptive, want_sums=True)
    _, _, st_w = dsc.render(cam0, mw, mh, seed=5, adaptive=adaptive, want_sums=True, mode=abi.RT_MODE_WAVEFRONT)
    assert (st_w.paths, st_w.rays, st_w.pixels_early_out) == (want_wf.paths, want_wf.rays, want_wf.pixels_early_out)
    main = 3 if st_w.pixels_early_out < n_pixels else 0
    assert st_w.launches == (3 + 1 + 1 + main + 1 if adaptive else 1 + 3 + 1)
    assert 0 < st_w.kernel_ms <= st_w.total_ms
