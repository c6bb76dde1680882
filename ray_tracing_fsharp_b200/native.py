"""ctypes binding of librtfs_b200.so (include/rtfs_b200.h).

This is the only way the package reaches the compute path, and it fails loudly: a missing library
raises ImportError-like RuntimeError with the build command, a missing GPU surfaces as
RtError(RT_ERR_NO_DEVICE) from the library itself.  There is no CPU fallback anywhere.
"""
import ctypes as C
import os

import numpy as np

from . import abi
from .abi import (RtCamera, RtDenoiseOpts, RtFrameConvergence, RtFrameNoise, RtFrameProgress, RtHittable, RtRenderOpts, RtSceneRebuild, RtSceneUpdate,
                  RtSnapshotHeader, RtStats, RtTexture)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librtfs_b200.so")


class RtError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"librtfs_b200 error {code}: {message}")
        self.code = code


_lib = None

_vp = C.c_void_p
_i32 = C.c_int32


def _declare(lib):
    sig = {
        "rt_abi_version": (C.c_int, []),
        "rt_last_error": (C.c_char_p, []),
        "rt_device_count": (C.c_int, []),
        "rt_host_pin": (C.c_int, [_vp, C.c_size_t]),
        "rt_host_unpin": (C.c_int, [_vp]),
        "rt_camera_make_basic": (C.c_int, [_i32, C.c_double, C.c_double, _vp, _vp, _vp, C.POINTER(RtCamera)]),
        "rt_ppm_format": (C.c_int, [_vp, _i32, _i32, _i32, _vp, C.c_size_t, C.POINTER(C.c_size_t)]),
        "rt_ppm_write_file": (C.c_int, [_vp, _i32, _i32, _i32, C.c_char_p]),
        "rt_gamma_correct": (C.c_uint8, [C.c_uint8]),
        "rt_scene_create": (C.c_int, [_vp, _i32, _vp, _i32, _i32, C.POINTER(_vp)]),
        "rt_scene_destroy": (None, [_vp]),
        "rt_scene_bvh_node_count": (C.c_int, [_vp, _i32]),
        "rt_scene_bvh_nodes": (C.c_int, [_vp, _i32, _vp, _vp, _vp]),
        "rt_scene_wide_bvh_check": (C.c_int, [_vp, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i32), C.POINTER(C.c_double)]),
        "rt_scene_device_bvh_check": (C.c_int, [_vp, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i32)]),
        "rt_scene_device_bytes": (C.c_size_t, [_vp]),
        "rt_scene_shared_memory_bytes": (C.c_size_t, [_vp]),
        "rt_scene_update": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _vp, _i32, C.POINTER(RtSceneUpdate)]),
        "rt_scene_rebuild": (C.c_int, [_vp, _vp, _i32, _vp, _i32, C.POINTER(RtSceneRebuild)]),
        "rt_render": (C.c_int, [_vp, C.POINTER(RtCamera), _i32, _i32, C.POINTER(RtRenderOpts), _vp, _vp, C.POINTER(RtStats)]),
        "rt_render_views": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, C.POINTER(RtRenderOpts), _vp, _vp, C.POINTER(RtStats)]),
        "rt_frame_begin": (C.c_int, [_vp, C.POINTER(RtCamera), _i32, _i32, C.POINTER(RtRenderOpts), C.POINTER(_vp),
                                     C.POINTER(RtFrameProgress)]),
        "rt_frame_advance": (C.c_int, [_vp, _i32, C.c_double, C.POINTER(RtFrameProgress)]),
        "rt_frame_read": (C.c_int, [_vp, _i32, _vp, _vp]),
        "rt_frame_extend": (C.c_int, [_vp, _i32]),
        "rt_frame_destroy": (None, [_vp]),
        "rt_frame_noise": (C.c_int, [_vp, C.c_double, _vp, _vp, C.POINTER(RtFrameNoise)]),
        "rt_frame_set_convergence": (C.c_int, [_vp, C.c_double, _i32, _i32]),
        "rt_frame_convergence": (C.c_int, [_vp, C.POINTER(RtFrameConvergence)]),
        "rt_frame_begin_views": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, C.POINTER(RtRenderOpts), C.POINTER(_vp),
                                           C.POINTER(RtFrameProgress)]),
        "rt_frame_view_noise": (C.c_int, [_vp, C.c_double, _vp]),
        "rt_render_window": (C.c_int, [_vp, C.POINTER(RtCamera), _i32, _i32, _i32, _i32, _i32, _i32, C.POINTER(RtRenderOpts), _vp, _vp,
                                       C.POINTER(RtStats)]),
        "rt_frame_begin_window": (C.c_int, [_vp, C.POINTER(RtCamera), _i32, _i32, _i32, _i32, _i32, _i32, C.POINTER(RtRenderOpts),
                                            C.POINTER(_vp), C.POINTER(RtFrameProgress)]),
        "rt_frame_features": (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp]),
        "rt_frame_denoise": (C.c_int, [_vp, C.POINTER(RtDenoiseOpts), _vp, _vp]),
        "rt_pixel_noise": (C.c_int, [_vp, _vp, C.c_size_t, _vp]),
        "rt_render_multi": (C.c_int, [_vp, _i32, _vp, _i32, _vp, _i32, C.POINTER(RtCamera), _i32, _i32, C.POINTER(RtRenderOpts), _vp,
                                      _vp, C.POINTER(RtStats)]),
        "rt_multi_create": (C.c_int, [_vp, _i32, _vp, _i32, _vp, _i32, C.POINTER(_vp)]),
        "rt_multi_render": (C.c_int, [_vp, C.POINTER(RtCamera), _i32, _i32, C.POINTER(RtRenderOpts), _vp, _vp, C.POINTER(RtStats)]),
        "rt_multi_destroy": (None, [_vp]),
        "rt_multi_frame_begin": (C.c_int, [_vp, C.POINTER(RtCamera), _i32, _i32, C.POINTER(RtRenderOpts), C.POINTER(_vp),
                                           C.POINTER(RtFrameProgress)]),
        "rt_multi_render_views": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, C.POINTER(RtRenderOpts), _vp, _vp, C.POINTER(RtStats)]),
        "rt_multi_frame_begin_views": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, C.POINTER(RtRenderOpts), C.POINTER(_vp),
                                                 C.POINTER(RtFrameProgress)]),
        "rt_frame_save": (C.c_int, [_vp, _vp, C.c_size_t, C.POINTER(C.c_size_t)]),
        "rt_frame_resume": (C.c_int, [_vp, _vp, C.c_size_t, C.POINTER(_vp), C.POINTER(RtFrameProgress)]),
        "rt_multi_frame_resume": (C.c_int, [_vp, _vp, C.c_size_t, C.POINTER(_vp), C.POINTER(RtFrameProgress)]),
        "rt_device_probe": (C.c_int, [_vp, C.POINTER(RtCamera), _i32, _i32, C.POINTER(RtRenderOpts), _i32, _i32, _vp, _vp, _vp,
                                      C.POINTER(RtStats)]),
        "rt_device_main": (C.c_int, [_vp, C.POINTER(RtCamera), _i32, _i32, C.POINTER(RtRenderOpts), _i32, _i32, _vp, _vp, _vp,
                                     C.POINTER(RtStats)]),
        "rt_device_counters": (C.c_int, [_vp, _vp, C.POINTER(RtStats)]),
        "rt_device_finalize": (C.c_int, [_i32, _vp, _i32, _i32, _vp, _vp]),
        "rt_comm_unique_id": (C.c_int, [_vp]),
        "rt_comm_create": (C.c_int, [_vp, _i32, _i32, _i32, _vp, C.POINTER(_vp)]),
        "rt_comm_destroy": (None, [_vp]),
        "rt_comm_uses_peer_memory": (C.c_int, [_vp]),
        "rt_comm_nccl_version": (C.c_int, [C.POINTER(_i32), C.c_char_p, C.c_size_t]),
        "rt_comm_render": (C.c_int, [_vp, _vp, C.POINTER(RtCamera), _i32, _i32, C.POINTER(RtRenderOpts), _vp, _vp, C.POINTER(RtStats)]),
        "rt_comm_last_stats": (C.c_int, [_vp, _vp, C.POINTER(RtStats)]),
        "rt_comm_frame": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp)]),
        "rt_test_sphere_hit": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, _vp]),
        "rt_test_plane_hit": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, _vp]),
        "rt_test_aabb_hit": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, _vp]),
        "rt_test_hit_object": (C.c_int, [_vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
        "rt_test_reflection": (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
        "rt_test_camera_rays": (C.c_int, [_i32, C.POINTER(RtCamera), _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
        "rt_test_texture": (C.c_int, [_vp, _i32, _vp, _vp, _vp]),
        "rt_test_combine_darken": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp]),
        "rt_test_rng": (C.c_int, [_i32, C.c_uint64, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
        "rt_test_trace_samples": (C.c_int, [_vp, C.POINTER(RtCamera), _i32, _i32, C.c_uint64, _i32, _vp, _vp, _vp, _vp, _vp]),
        "rt_measure_fp32_peak": (C.c_int, [_i32, C.POINTER(C.c_double)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export what the header declares
        fn.restype = res
        fn.argtypes = args
    return sorted(sig)


EXPORTS = None


def lib():
    """The loaded library.  Raises if it has not been built (python -c 'import __graft_entry__ as g; g.build()')."""
    global _lib, EXPORTS
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `make -C ray_tracing_fsharp_b200/csrc` "
                "(or __graft_entry__.build()).  There is no CPU fallback.")
        handle = C.CDLL(LIB_PATH)
        EXPORTS = _declare(handle)
        if handle.rt_abi_version() != abi.RT_ABI_VERSION:
            raise RuntimeError("librtfs_b200.so was built from a different include/rtfs_b200.h (ABI version mismatch)")
        _lib = handle
    return _lib


def check(rc):
    if rc != abi.RT_OK:
        raise RtError(rc, lib().rt_last_error().decode("utf-8", "replace"))
    return rc


def ptr(a):
    """void* of a C-contiguous numpy array (or None)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return C.c_void_p(a.ctypes.data)


def f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a.reshape(shape) if shape is not None else a


class FrameRing:
    """Explicit recycling of output frames, for a host that renders frame after frame: hands out `count` uint8 arrays of
    one shape in turn (`next()`), each already touched.  Opt-in — pass `rgb_out=ring.next()` (or `frames=ring` to
    Scene.render): the caller states that it is done with the frame it got `count` calls ago.  Without it every render
    returns a fresh array that is never handed out again.  (A fresh np.empty is untouched memory, and the device->host copy
    into it pays a page fault per 4 KiB — 1.3 ms for the 2.9 MB C2 frame; a .NET caller's zero-initialised, reused array
    does not.)"""

    def __init__(self, shape, count=2):
        if count < 1:
            raise ValueError("FrameRing needs at least one frame")
        self.shape = tuple(shape)
        self._frames = [np.zeros(self.shape, np.uint8) for _ in range(count)]
        self._pinned = []
        for f in self._frames:
            f.fill(0)  # touch the pages now
            # page-lock it where a device is present (rt_host_pin): the device->host copy then runs at PCIe speed
            if lib().rt_host_pin(C.c_void_p(f.ctypes.data), f.nbytes) == abi.RT_OK:
                self._pinned.append(f)
        self._at = 0

    def __del__(self):
        try:
            for f in self._pinned:
                lib().rt_host_unpin(C.c_void_p(f.ctypes.data))
            self._pinned = []
        except Exception:
            pass

    def next(self):
        f = self._frames[self._at % len(self._frames)]
        self._at += 1
        return f


def _frame_buffer(shape):
    """A fresh output frame (never recycled behind the caller's back; see FrameRing for the opt-in)."""
    return np.empty(shape, np.uint8)


def _as_array(ctype, items):
    """A ctypes array of `items` for the ABI: marshal()'s array is passed through as it is (no per-element copy)."""
    if isinstance(items, C.Array) and items._type_ is ctype and len(items) > 0:
        return items
    return (ctype * max(1, len(items)))(*items)


def device_count():
    return int(lib().rt_device_count())


def _views_args(cameras, seeds):
    """(n, the RtCamera array, the uint64 seeds or None) of a batch of views, as rt_render_views and its kin take them."""
    n = len(cameras)
    cams = (RtCamera * max(1, n))(*cameras)
    sd = None
    if seeds is not None:
        if len(seeds) != n:
            raise ValueError(f"{len(seeds)} seeds for {n} cameras")
        sd = np.ascontiguousarray([int(x) for x in seeds], np.uint64)
    return n, cams, sd


def _views_frame(owner, out, progress, max_w, max_h, n):
    """The Frame of a batch of n views opened into `out`; it holds `owner` (a SceneHandle or MultiHandle)."""
    frame = Frame.__new__(Frame)
    frame.scene, frame.ptr, frame.progress = owner, out, progress
    frame.rows, frame.cols = 2 * max_h + 1, 2 * max_w + 1
    frame.n_views = n
    return frame


def _resume(owner, resume_fn, data):
    """The Frame resume_fn (rt_frame_resume or rt_multi_frame_resume) opens from the snapshot `data` (bytes-like) on `owner`
    (a SceneHandle or MultiHandle), with the shape of the frame that was saved: a tall frame for a batch of views, the
    window's rows and cols for a window."""
    buf = np.frombuffer(data, np.uint8)
    out = C.c_void_p()
    progress = RtFrameProgress()
    check(resume_fn(owner.ptr, C.c_void_p(buf.ctypes.data if buf.size else None), buf.size, C.byref(out), C.byref(progress)))
    h = RtSnapshotHeader.from_buffer_copy(buf[:C.sizeof(RtSnapshotHeader)].tobytes())
    if h.kind == abi.RT_FRAME_VIEWS:
        return _views_frame(owner, out, progress, h.max_width_coord, h.max_height_coord, h.n_views)
    frame = Frame.__new__(Frame)
    frame.scene, frame.ptr, frame.progress = owner, out, progress
    if h.kind == abi.RT_FRAME_WINDOW:
        frame.rows, frame.cols = h.window[2], h.window[3]
    else:
        frame.rows, frame.cols = 2 * h.max_height_coord + 1, 2 * h.max_width_coord + 1
    return frame


class SceneHandle:
    """Owner of an RtScene* (rt_scene_create / rt_scene_destroy)."""

    def __init__(self, hittables, textures=(), device=0, keepalive=None):
        self.n_objects = len(hittables)
        self._h = _as_array(RtHittable, hittables)
        self._t = _as_array(RtTexture, textures)
        self._keep = keepalive
        self.device = device
        out = C.c_void_p()
        check(lib().rt_scene_create(self._h, len(hittables), self._t, len(textures), device, C.byref(out)))
        self.ptr = out

    def close(self):
        if getattr(self, "ptr", None):
            lib().rt_scene_destroy(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def update(self, object_index, hittables, texture_index=None, textures=None) -> RtSceneUpdate:
        """Edits the scene on its device (rt_scene_update): object object_index[i] becomes hittables[i], texture
        texture_index[j] becomes textures[j], and the tree is refit there.  The scene then renders bit for bit as one
        created from the edited arrays.  Structural changes (shape, the sign of a bounded sphere's radius, a texture's kind or
        image size), bad or repeated indices and anything creation refuses: RtError RT_ERR_INVALID_ARGUMENT, the scene left
        as it was.  Frames opened before the call are stale (see Frame).  Returns the RtSceneUpdate."""
        oi = np.ascontiguousarray(list(object_index), np.int32)
        ti = np.ascontiguousarray(list(texture_index) if texture_index is not None else [], np.int32)
        textures = list(textures) if textures is not None else []
        if len(hittables) != len(oi) or len(textures) != len(ti):
            raise ValueError("one record per index")
        h = _as_array(RtHittable, hittables)
        t = _as_array(RtTexture, textures)
        info = RtSceneUpdate()
        check(lib().rt_scene_update(self.ptr, ptr(oi), h, len(oi), ptr(ti), t, len(ti), C.byref(info)))
        return info

    def rebuild(self, remove=(), append=()) -> RtSceneRebuild:
        """Removes and appends objects and builds the tree anew on the device (rt_scene_rebuild): the objects `remove`
        (indices) are taken out, the others keep their order, and `append` (RtHittable records) are added at the end.  The
        scene then renders bit for bit as one created from the new array.  With neither, the tree of the current objects is
        rebuilt.  Bad or repeated indices and anything creation refuses in an appended object: RtError
        RT_ERR_INVALID_ARGUMENT, the scene left as it was.  Frames opened before the call are stale (see Frame).  Returns the
        RtSceneRebuild."""
        rm = np.ascontiguousarray(list(remove), np.int32)
        append = list(append)
        a = _as_array(RtHittable, append)
        info = RtSceneRebuild()
        check(lib().rt_scene_rebuild(self.ptr, ptr(rm), len(rm), a, len(append), C.byref(info)))
        self.n_objects = info.n_objects
        return info

    def bvh_nodes(self, which=abi.RT_BVH_SAH):
        n = lib().rt_scene_bvh_node_count(self.ptr, which)
        bounds = np.empty((n, 6))
        right = np.empty(n, np.int32)
        prim = np.empty(n, np.int32)
        if n:
            check(lib().rt_scene_bvh_nodes(self.ptr, which, ptr(bounds), ptr(right), ptr(prim)))
        return bounds, right, prim

    def wide_bvh_check(self):
        """Builds (if need be) and verifies the 8-wide compressed tree on the host; returns its figures."""
        n, depth, ns, mc = _i32(), _i32(), _i32(), C.c_double()
        check(lib().rt_scene_wide_bvh_check(self.ptr, C.byref(n), C.byref(depth), C.byref(ns), C.byref(mc)))
        return {"nodes": n.value, "depth": depth.value, "spheres": ns.value, "mean_children": mc.value}

    def device_bvh_check(self):
        """Verifies on the host the binary tree in the form the render kernels read it; returns its figures."""
        n, depth, ns = _i32(), _i32(), _i32()
        check(lib().rt_scene_device_bvh_check(self.ptr, C.byref(n), C.byref(depth), C.byref(ns)))
        return {"nodes": n.value, "depth": depth.value, "spheres": ns.value}

    def device_bytes(self):
        return int(lib().rt_scene_device_bytes(self.ptr))

    def shared_memory_bytes(self):
        return int(lib().rt_scene_shared_memory_bytes(self.ptr))

    # ---- render ----
    def render(self, camera, max_w, max_h, seed=0, adaptive=True, mode=abi.RT_MODE_MEGAKERNEL, gamma=False, flags=0,
               want_sums=False, rgb_out=None):
        rows, cols = 2 * max_h + 1, 2 * max_w + 1
        rgb = rgb_out if rgb_out is not None else _frame_buffer((rows, cols, 3))
        sums = np.empty((rows, cols, 4), np.int32) if want_sums else None
        opts = RtRenderOpts(seed, int(adaptive), mode, int(gamma), flags)
        stats = RtStats()
        check(lib().rt_render(self.ptr, C.byref(camera), max_w, max_h, C.byref(opts), ptr(rgb), ptr(sums), C.byref(stats)))
        return rgb, sums, stats

    def render_views(self, cameras, max_w, max_h, seeds=None, adaptive=True, gamma=False, flags=0, want_sums=False, seed=0):
        """n views of this scene in one submission (rt_render_views): `cameras` a sequence of RtCamera (same
        samples_per_pixel and bounce_depth), `seeds` one per view or None (then `seed` for every view).  Returns
        (uint8 [n, rows, cols, 3], int32 [n, rows, cols, 4] or None, RtStats of the batch); view v is exactly
        render(cameras[v], max_w, max_h, seed=seeds[v]).  RtError RT_ERR_INVALID_ARGUMENT for an empty batch."""
        n, cams, sd = _views_args(cameras, seeds)
        rows, cols = 2 * max_h + 1, 2 * max_w + 1
        rgb = _frame_buffer((n, rows, cols, 3))
        sums = np.empty((n, rows, cols, 4), np.int32) if want_sums else None
        opts = RtRenderOpts(seed, int(adaptive), abi.RT_MODE_MEGAKERNEL, int(gamma), flags)
        stats = RtStats()
        check(lib().rt_render_views(self.ptr, cams, ptr(sd), n, max_w, max_h, C.byref(opts), ptr(rgb), ptr(sums), C.byref(stats)))
        return rgb, sums, stats

    def open_frame(self, camera, max_w, max_h, seed=0, adaptive=True, flags=0, mode=abi.RT_MODE_MEGAKERNEL):
        """A progressive frame of this scene (rt_frame_begin: runs the probe).  See Frame."""
        return Frame(self, camera, max_w, max_h, seed, adaptive, flags, mode)

    def open_frame_views(self, cameras, max_w, max_h, seeds=None, seed=0, adaptive=True, flags=0):
        """A progressive frame of a batch of views of this scene (rt_frame_begin_views: runs the probe), cameras and seeds as
        render_views.  A Frame whose read, noise and sums have shape [n_views, rows, cols, ...]; view v is exactly
        open_frame(cameras[v], max_w, max_h, seed=seeds[v]) at the same samples_done, and Frame.view_noise summarises
        each view.  RtError RT_ERR_INVALID_ARGUMENT for an empty batch."""
        n, cams, sd = _views_args(cameras, seeds)
        opts = RtRenderOpts(seed, int(adaptive), abi.RT_MODE_MEGAKERNEL, 0, flags)
        out = C.c_void_p()
        progress = RtFrameProgress()
        check(lib().rt_frame_begin_views(self.ptr, cams, ptr(sd), n, max_w, max_h, C.byref(opts), C.byref(out), C.byref(progress)))
        return _views_frame(self, out, progress, max_w, max_h, n)

    def render_window(self, camera, max_w, max_h, window, seed=0, adaptive=True, gamma=False, flags=0, want_sums=False, rgb_out=None):
        """The window (row0, col0, rows, cols) of render(camera, max_w, max_h, ...) without tracing the rest of the frame
        (rt_render_window).  Returns (uint8 [rows, cols, 3], int32 [rows, cols, 4] or None, RtStats of the window);
        window pixel (r, c) is exactly pixel (row0 + r, col0 + c) of render's frame.  RtError RT_ERR_INVALID_ARGUMENT for a
        window that is empty or does not lie inside the (2 max_h + 1) x (2 max_w + 1) frame."""
        row0, col0, rows, cols = (int(x) for x in window)
        rgb = rgb_out if rgb_out is not None else _frame_buffer((max(rows, 0), max(cols, 0), 3))
        sums = np.empty((max(rows, 0), max(cols, 0), 4), np.int32) if want_sums else None
        opts = RtRenderOpts(seed, int(adaptive), abi.RT_MODE_MEGAKERNEL, int(gamma), flags)
        stats = RtStats()
        check(lib().rt_render_window(self.ptr, C.byref(camera), max_w, max_h, row0, col0, rows, cols, C.byref(opts), ptr(rgb), ptr(sums),
                                     C.byref(stats)))
        return rgb, sums, stats

    def open_frame_window(self, camera, max_w, max_h, window, seed=0, adaptive=True, flags=0):
        """A progressive frame of the window (row0, col0, rows, cols) of this scene's frame (rt_frame_begin_window: runs the
        probe over the window).  A Frame whose read, noise and sums have shape [rows, cols, ...]; after any pass (and under a
        convergence rule) it is exactly the crop of open_frame(camera, max_w, max_h, seed=seed) at the same samples_done."""
        row0, col0, rows, cols = (int(x) for x in window)
        opts = RtRenderOpts(seed, int(adaptive), abi.RT_MODE_MEGAKERNEL, 0, flags)
        out = C.c_void_p()
        progress = RtFrameProgress()
        check(lib().rt_frame_begin_window(self.ptr, C.byref(camera), max_w, max_h, row0, col0, rows, cols, C.byref(opts), C.byref(out),
                                          C.byref(progress)))
        frame = Frame.__new__(Frame)
        frame.scene, frame.ptr, frame.progress = self, out, progress
        frame.rows, frame.cols = rows, cols
        return frame

    def resume_frame(self, data):
        """A progressive frame opened from a snapshot written by Frame.save (rt_frame_resume), on this scene: after every
        further pass it is exactly the saved frame continued without interruption, whatever device count saved it.  The
        scene must hold the objects and textures of the saved frame's scene.  RtError RT_ERR_INVALID_ARGUMENT for a damaged
        snapshot or a scene with other content."""
        return _resume(self, lib().rt_frame_resume, data)

    # ---- conformance ----
    def hit_object(self, o, d, traversal=0):
        o, d = f64(o, (-1, 3)), f64(d, (-1, 3))
        n = len(o)
        prim = np.empty(n, np.int32)
        t = np.empty(n)
        strike = np.empty((n, 3))
        check(lib().rt_test_hit_object(self.ptr, traversal, n, ptr(o), ptr(d), ptr(prim), ptr(t), ptr(strike)))
        return prim, t, strike

    def reflection(self, prim, o, d, strike, colour_in, uniforms):
        prim = np.ascontiguousarray(prim, np.int32)
        o, d, strike = f64(o, (-1, 3)), f64(d, (-1, 3)), f64(strike, (-1, 3))
        colour_in = np.ascontiguousarray(colour_in, np.uint8).reshape(-1, 3)
        uniforms = f64(uniforms, (-1, 4))
        n = len(prim)
        absorbed = np.empty(n, np.uint8)
        colour = np.empty((n, 3), np.uint8)
        oo = np.empty((n, 3))
        do = np.empty((n, 3))
        inside = np.empty(n, np.uint8)
        check(lib().rt_test_reflection(self.ptr, n, ptr(prim), ptr(o), ptr(d), ptr(strike), ptr(colour_in), ptr(uniforms), ptr(absorbed),
                                       ptr(colour), ptr(oo), ptr(do), ptr(inside)))
        return absorbed, colour, oo, do, inside

    def texture(self, prim, point):
        prim = np.ascontiguousarray(prim, np.int32)
        point = f64(point, (-1, 3))
        out = np.empty((len(prim), 3), np.uint8)
        check(lib().rt_test_texture(self.ptr, len(prim), ptr(prim), ptr(point), ptr(out)))
        return out

    def trace_samples(self, camera, max_w, max_h, seed, row_idx, col_idx, sample):
        row_idx, col_idx, sample = [np.ascontiguousarray(a, np.int32) for a in (row_idx, col_idx, sample)]
        n = len(row_idx)
        colour = np.empty((n, 3), np.uint8)
        rays = np.empty(n, np.int32)
        check(lib().rt_test_trace_samples(self.ptr, C.byref(camera), max_w, max_h, seed, n, ptr(row_idx), ptr(col_idx), ptr(sample),
                                          ptr(colour), ptr(rays)))
        return colour, rays


class Frame:
    """Owner of an RtFrame* (rt_frame_begin / rt_frame_destroy): rt_render's frame advanced in passes over windows of
    sample indices.  After every pass the frame is exactly rt_render's at samples_per_pixel = progress.samples_done.
    Holds its scene handle, so the scene outlives it.  A frame of a batch of views (SceneHandle.open_frame_views) has
    n_views set, and its images, sums and maps carry a leading view axis; a frame of a window (SceneHandle.open_frame_window)
    has the window's rows and cols.  Once its scene is edited (SceneHandle.update) the frame is stale: advance, extend,
    set_convergence, features and denoise raise RtError RT_ERR_INVALID_ARGUMENT; read, noise, view_noise and convergence
    still return what it holds."""

    n_views = None  # a frame of one camera

    def _shape(self, *tail):
        return ((self.n_views,) if self.n_views is not None else ()) + (self.rows, self.cols) + tail

    def __init__(self, scene: SceneHandle, camera, max_w, max_h, seed=0, adaptive=True, flags=0, mode=abi.RT_MODE_MEGAKERNEL):
        self.scene = scene
        self.rows, self.cols = 2 * max_h + 1, 2 * max_w + 1
        opts = RtRenderOpts(seed, int(adaptive), mode, 0, flags)
        out = C.c_void_p()
        self.progress = RtFrameProgress()
        check(lib().rt_frame_begin(scene.ptr, C.byref(camera), max_w, max_h, C.byref(opts), C.byref(out), C.byref(self.progress)))
        self.ptr = out

    def advance(self, max_samples=0, target_ms=0.0) -> RtFrameProgress:
        """One pass of at most `max_samples` sample indices (0: no limit) predicted to take about `target_ms` of device time
        (0: no limit).  A no-op once the frame is done."""
        progress = RtFrameProgress()
        check(lib().rt_frame_advance(self.ptr, int(max_samples), float(target_ms), C.byref(progress)))
        self.progress = progress
        return progress

    def read(self, gamma=False, want_sums=False, rgb_out=None):
        """The current image (uint8 [rows, cols, 3]) and, with want_sums, the int32 sums [rows, cols, 4]."""
        rgb = rgb_out if rgb_out is not None else _frame_buffer(self._shape(3))
        sums = np.empty(self._shape(4), np.int32) if want_sums else None
        check(lib().rt_frame_read(self.ptr, int(gamma), ptr(rgb), ptr(sums)))
        return rgb, sums

    def extend(self, spp):
        """Raises the frame's target to `spp` samples per pixel (RtError RT_ERR_INVALID_ARGUMENT if that would change the
        probe, or is below what the frame already holds)."""
        check(lib().rt_frame_extend(self.ptr, int(spp)))

    def noise(self, tolerance, want_map=True, want_sq=False):
        """The noise estimate of a frame opened with abi.RT_FLAG_NOISE (rt_frame_noise): (RtFrameNoise summary over the
        flagged pixels against `tolerance`, the per-pixel standard error float32 [rows, cols] or None, the per-pixel sum of
        r^2 + g^2 + b^2 uint64 [rows, cols] or None)."""
        summary = RtFrameNoise()
        se = np.empty(self._shape(), np.float32) if want_map else None
        sq = np.empty(self._shape(), np.uint64) if want_sq else None
        check(lib().rt_frame_noise(self.ptr, float(tolerance), ptr(se), ptr(sq), C.byref(summary)))
        return summary, se, sq

    def view_noise(self, tolerance):
        """One RtFrameNoise per view (rt_frame_view_noise; one for a frame of one camera): view v's summary over its pixels
        still being sampled, bit for bit noise(tolerance)[0] of the frame of camera v alone.  pixels == 0: the view is
        finished."""
        out = (RtFrameNoise * (self.n_views or 1))()
        check(lib().rt_frame_view_noise(self.ptr, float(tolerance), out))
        return list(out)

    def set_convergence(self, tolerance, min_samples=64, interval=64):
        """Stops sampling each pixel once its noise estimate is within `tolerance` (8-bit levels), checked at the sample
        counts min_samples + j * interval (rt_frame_set_convergence).  Only on a frame opened with abi.RT_FLAG_NOISE, before
        its first pass.  Every pixel is then exactly rt_render's pixel at the sample count it stopped at."""
        check(lib().rt_frame_set_convergence(self.ptr, float(tolerance), int(min_samples), int(interval)))

    def convergence(self) -> RtFrameConvergence:
        """The rule and its state (rt_frame_convergence): next checkpoint, checks run, pixels still sampled and stopped."""
        out = RtFrameConvergence()
        check(lib().rt_frame_convergence(self.ptr, C.byref(out)))
        return out

    def features(self, samples=4):
        """First-hit features of sample indices 0 .. samples - 1 of every pixel (rt_frame_features): (prim int32 [rows, cols],
        the caller's Hittable index hit by sample 0 or -1; albedo uint8 [rows, cols, 3], the truncating mean of the colour the
        first scatter leaves in a white path; normal float32 [rows, cols, 3] and depth float32 [rows, cols], the means over the
        samples that hit, depth +inf where none did).  Exact functions of (seed, pixel, samples): passes do not change them."""
        prim = np.empty(self._shape(), np.int32)
        albedo = np.empty(self._shape(3), np.uint8)
        normal = np.empty(self._shape(3), np.float32)
        depth = np.empty(self._shape(), np.float32)
        check(lib().rt_frame_features(self.ptr, int(samples), ptr(prim), ptr(albedo), ptr(normal), ptr(depth)))
        return prim, albedo, normal, depth

    def denoise(self, iterations=3, feature_samples=4, sigma_colour=4.0, sigma_normal=0.1, sigma_albedo=16.0, sigma_depth=0.02, gamma=False,
                want_linear=False):
        """A denoised preview of the frame's current image (rt_frame_denoise: an edge-avoiding a-trous filter guided by each
        pixel's noise estimate and by features(feature_samples)).  Only on a frame opened with abi.RT_FLAG_NOISE; the frame
        itself is left as it was.  Returns (uint8 [rows, cols, 3], float32 [rows, cols, 3] filtered means in 8-bit levels or
        None).  The defaults are DESIGN.md section 19's."""
        opts = RtDenoiseOpts(int(iterations), int(feature_samples), float(sigma_colour), float(sigma_normal), float(sigma_albedo),
                             float(sigma_depth), int(gamma), 0)
        rgb = np.empty(self._shape(3), np.uint8)
        linear = np.empty(self._shape(3), np.float32) if want_linear else None
        check(lib().rt_frame_denoise(self.ptr, C.byref(opts), ptr(rgb), ptr(linear)))
        return rgb, linear

    def save(self) -> bytes:
        """The frame as a snapshot (rt_frame_save): bytes that SceneHandle.resume_frame or MultiHandle.resume_frame open again
        as this frame, in this process or another, on any device count.  The frame is left as it was.  RtError
        RT_ERR_INVALID_ARGUMENT for a stale frame."""
        n = C.c_size_t()
        check(lib().rt_frame_save(self.ptr, None, 0, C.byref(n)))
        buf = np.empty(n.value, np.uint8)
        check(lib().rt_frame_save(self.ptr, ptr(buf), buf.size, C.byref(n)))
        return buf.tobytes()

    def close(self):
        if getattr(self, "ptr", None):
            lib().rt_frame_destroy(self.ptr)
            self.ptr = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiHandle:
    """Owner of an RtMulti* (rt_multi_create / rt_multi_destroy): one frame split over several GPUs of this process."""

    def __init__(self, hittables, textures=(), devices=(0,), keepalive=None):
        self._h = _as_array(RtHittable, hittables)
        self._t = _as_array(RtTexture, textures)
        self._keep = keepalive
        self.devices = list(devices)
        dv = (C.c_int32 * len(self.devices))(*self.devices)
        out = C.c_void_p()
        check(lib().rt_multi_create(self._h, len(hittables), self._t, len(textures), dv, len(self.devices), C.byref(out)))
        self.ptr = out

    def close(self):
        if getattr(self, "ptr", None):
            lib().rt_multi_destroy(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def render(self, camera, max_w, max_h, seed=0, adaptive=True, gamma=False, flags=0, want_sums=False, rgb_out=None):
        rows, cols = 2 * max_h + 1, 2 * max_w + 1
        rgb = rgb_out if rgb_out is not None else _frame_buffer((rows, cols, 3))
        sums = np.empty((rows, cols, 4), np.int32) if want_sums else None
        opts = RtRenderOpts(seed, int(adaptive), abi.RT_MODE_MEGAKERNEL, int(gamma), flags)
        stats = RtStats()
        check(lib().rt_multi_render(self.ptr, C.byref(camera), max_w, max_h, C.byref(opts), ptr(rgb), ptr(sums), C.byref(stats)))
        return rgb, sums, stats

    def open_frame(self, camera, max_w, max_h, seed=0, adaptive=True, flags=0, mode=abi.RT_MODE_MEGAKERNEL):
        """A progressive frame split over this handle's devices (rt_multi_frame_begin: runs the probe).  A Frame that is bit
        for bit SceneHandle.open_frame's frame of one device after every pass; it holds this handle, so the handle outlives
        it."""
        opts = RtRenderOpts(seed, int(adaptive), mode, 0, flags)
        out = C.c_void_p()
        progress = RtFrameProgress()
        check(lib().rt_multi_frame_begin(self.ptr, C.byref(camera), max_w, max_h, C.byref(opts), C.byref(out), C.byref(progress)))
        frame = Frame.__new__(Frame)
        frame.scene, frame.ptr, frame.progress = self, out, progress
        frame.rows, frame.cols = 2 * max_h + 1, 2 * max_w + 1
        return frame

    def render_views(self, cameras, max_w, max_h, seeds=None, adaptive=True, gamma=False, flags=0, want_sums=False, seed=0):
        """A batch of views split over this handle's devices (rt_multi_render_views): arguments and return shapes of
        SceneHandle.render_views, and bit for bit its images, sums and the stats' paths, rays, degenerate_paths and
        pixels_early_out."""
        n, cams, sd = _views_args(cameras, seeds)
        rows, cols = 2 * max_h + 1, 2 * max_w + 1
        rgb = _frame_buffer((n, rows, cols, 3))
        sums = np.empty((n, rows, cols, 4), np.int32) if want_sums else None
        opts = RtRenderOpts(seed, int(adaptive), abi.RT_MODE_MEGAKERNEL, int(gamma), flags)
        stats = RtStats()
        check(lib().rt_multi_render_views(self.ptr, cams, ptr(sd), n, max_w, max_h, C.byref(opts), ptr(rgb), ptr(sums), C.byref(stats)))
        return rgb, sums, stats

    def open_frame_views(self, cameras, max_w, max_h, seeds=None, seed=0, adaptive=True, flags=0):
        """A progressive frame of a batch of views split over this handle's devices (rt_multi_frame_begin_views: runs the
        probe), arguments as SceneHandle.open_frame_views.  A Frame that is bit for bit SceneHandle.open_frame_views' frame of
        one device after every pass; it holds this handle, so the handle outlives it."""
        n, cams, sd = _views_args(cameras, seeds)
        opts = RtRenderOpts(seed, int(adaptive), abi.RT_MODE_MEGAKERNEL, 0, flags)
        out = C.c_void_p()
        progress = RtFrameProgress()
        check(lib().rt_multi_frame_begin_views(self.ptr, cams, ptr(sd), n, max_w, max_h, C.byref(opts), C.byref(out), C.byref(progress)))
        return _views_frame(self, out, progress, max_w, max_h, n)

    def resume_frame(self, data):
        """SceneHandle.resume_frame split over this handle's devices (rt_multi_frame_resume).  A snapshot of a window raises
        RtError RT_ERR_UNSUPPORTED: windows run on one GPU."""
        return _resume(self, lib().rt_multi_frame_resume, data)


class CommHandle:
    """Owner of an RtComm* (rt_comm_create / rt_comm_destroy): this process's rank of a one-process-per-GPU job whose
    collectives the library issues itself (NCCL, bound at run time).  Creation is collective over the ranks."""

    @staticmethod
    def _torch_first():
        """The library binds whatever libnccl.so.2 the process already holds, else the system's.  A process that will
        ALSO import PyTorch must import it first: PyTorch needs the (newer) NCCL build it bundles, and the dynamic loader
        keeps a single library per soname — binding the system's copy first makes `import torch` fail afterwards."""
        import importlib.util
        import sys
        if "torch" not in sys.modules and importlib.util.find_spec("torch") is not None:
            import torch  # noqa: F401

    @staticmethod
    def unique_id() -> bytes:
        CommHandle._torch_first()
        buf = (C.c_uint8 * abi.RT_COMM_ID_BYTES)()
        check(lib().rt_comm_unique_id(buf))
        return bytes(buf)

    @staticmethod
    def nccl_version():
        CommHandle._torch_first()
        v = _i32()
        path = C.create_string_buffer(512)
        check(lib().rt_comm_nccl_version(C.byref(v), path, 512))
        return int(v.value), path.value.decode("utf-8", "replace")

    def __init__(self, unique_id: bytes, rank: int, world: int, device: int, stream=None):
        if unique_id is None and world == 1:
            unique_id = bytes(abi.RT_COMM_ID_BYTES)
        if len(unique_id) != abi.RT_COMM_ID_BYTES:
            raise ValueError("unique_id must be RT_COMM_ID_BYTES long")
        if world > 1:
            CommHandle._torch_first()
        self.rank, self.world, self.device = rank, world, device
        idb = (C.c_uint8 * abi.RT_COMM_ID_BYTES).from_buffer_copy(unique_id)  # ignored by the library when world == 1
        out = C.c_void_p()
        check(lib().rt_comm_create(idb, rank, world, device, C.c_void_p(stream) if stream else None, C.byref(out)))
        self.ptr = out

    def close(self):
        if getattr(self, "ptr", None):
            lib().rt_comm_destroy(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def render(self, scene: "SceneHandle", camera, max_w, max_h, seed=0, adaptive=True, gamma=False, flags=0, want_rgb=True,
               want_sums=False, want_stats=True, rgb_out=None):
        """One frame, collectively.  want_rgb / want_sums / want_stats all False: enqueue only (device-resident)."""
        rows, cols = 2 * max_h + 1, 2 * max_w + 1
        rgb = (rgb_out if rgb_out is not None else _frame_buffer((rows, cols, 3))) if want_rgb else None
        sums = np.empty((rows, cols, 4), np.int32) if want_sums else None
        opts = RtRenderOpts(seed, int(adaptive), abi.RT_MODE_MEGAKERNEL, int(gamma), flags)
        stats = RtStats() if (want_stats or want_rgb or want_sums) else None
        check(lib().rt_comm_render(self.ptr, scene.ptr, C.byref(camera), max_w, max_h, C.byref(opts), ptr(rgb), ptr(sums),
                                   C.byref(stats) if stats is not None else None))
        return rgb, sums, stats

    def uses_peer_memory(self) -> bool:
        return bool(lib().rt_comm_uses_peer_memory(self.ptr))

    def last_stats(self, scene: "SceneHandle"):
        """Timing / counters of the last enqueue-only render (call after synchronising the stream)."""
        stats = RtStats()
        check(lib().rt_comm_last_stats(self.ptr, scene.ptr, C.byref(stats)))
        return stats

    def frame_pointers(self):
        rgb, stats = C.c_void_p(), C.c_void_p()
        check(lib().rt_comm_frame(self.ptr, C.byref(rgb), C.byref(stats)))
        return rgb.value, stats.value


# ---- free-standing conformance wrappers ---------------------------------------------------------
def sphere_hit(o, d, c, r, device=0):
    o, d, c, r = f64(o, (-1, 3)), f64(d, (-1, 3)), f64(c, (-1, 3)), f64(r, (-1,))
    t = np.empty(len(o))
    check(lib().rt_test_sphere_hit(device, len(o), ptr(o), ptr(d), ptr(c), ptr(r), ptr(t)))
    return t


def plane_hit(o, d, p, n, device=0):
    o, d, p, n = [f64(a, (-1, 3)) for a in (o, d, p, n)]
    t = np.empty(len(o))
    check(lib().rt_test_plane_hit(device, len(o), ptr(o), ptr(d), ptr(p), ptr(n), ptr(t)))
    return t


def aabb_hit(o, d, bmin, bmax, device=0):
    o, d, bmin, bmax = [f64(a, (-1, 3)) for a in (o, d, bmin, bmax)]
    hit = np.empty(len(o), np.uint8)
    check(lib().rt_test_aabb_hit(device, len(o), ptr(o), ptr(d), ptr(bmin), ptr(bmax), ptr(hit)))
    return hit.astype(bool)


def camera_rays(camera, max_w, max_h, row, col, r1, r2, device=0):
    row, col = np.ascontiguousarray(row, np.int32), np.ascontiguousarray(col, np.int32)
    r1, r2 = f64(r1), f64(r2)
    n = len(row)
    o = np.empty((n, 3))
    d = np.empty((n, 3))
    check(lib().rt_test_camera_rays(device, C.byref(camera), max_w, max_h, n, ptr(row), ptr(col), ptr(r1), ptr(r2), ptr(o), ptr(d)))
    return o, d


def combine_darken(a, b, albedo, device=0):
    a = np.ascontiguousarray(a, np.uint8).reshape(-1, 3)
    b = np.ascontiguousarray(b, np.uint8).reshape(-1, 3)
    albedo = np.ascontiguousarray(np.broadcast_to(f64(albedo), (len(a),)))
    out = np.empty_like(a)
    check(lib().rt_test_combine_darken(device, len(a), ptr(a), ptr(b), ptr(albedo), ptr(out)))
    return out


def rng(seed, pixel, sample, bounce, retry, device=0):
    pixel, sample, bounce, retry = [np.ascontiguousarray(a, np.uint32) for a in (pixel, sample, bounce, retry)]
    n = len(pixel)
    words = np.empty((n, 4), np.uint32)
    u = np.empty((n, 4))
    check(lib().rt_test_rng(device, seed, n, ptr(pixel), ptr(sample), ptr(bounce), ptr(retry), ptr(words), ptr(u)))
    return words, u


def measure_fp32_peak(device=0):
    out = C.c_double()
    check(lib().rt_measure_fp32_peak(device, C.byref(out)))
    return out.value


def camera_make_basic(spp, focal, aspect, origin, view_dir, view_up):
    cam = RtCamera()
    origin, view_dir, view_up = f64(origin), f64(view_dir), f64(view_up)
    check(lib().rt_camera_make_basic(spp, focal, aspect, ptr(origin), ptr(view_dir), ptr(view_up), C.byref(cam)))
    return cam


def pixel_noise(sums, sq):
    """rt_pixel_noise on the host: the per-pixel standard error (float32, the shape of `sq`) from saved moments, `sums`
    int32 [..., 4] {sumR, sumG, sumB, count} and `sq` uint64 [...] (the sum of r^2 + g^2 + b^2).  Needs no device."""
    sums = np.ascontiguousarray(sums, np.int32)
    sq = np.ascontiguousarray(sq, np.uint64)
    if sums.shape != sq.shape + (4,):
        raise ValueError(f"sums {sums.shape} must be sq's shape {sq.shape} + (4,)")
    se = np.empty(sq.shape, np.float32)
    check(lib().rt_pixel_noise(ptr(sums), ptr(sq), sq.size, ptr(se)))
    return se


def ppm_format(rgb, gamma=False):
    rgb = np.ascontiguousarray(rgb, np.uint8)
    rows, cols = rgb.shape[0], rgb.shape[1]
    n = C.c_size_t()
    check(lib().rt_ppm_format(ptr(rgb), rows, cols, int(gamma), None, 0, C.byref(n)))
    buf = C.create_string_buffer(n.value)
    check(lib().rt_ppm_format(ptr(rgb), rows, cols, int(gamma), C.cast(buf, C.c_void_p), n.value, C.byref(n)))
    return buf.raw[:n.value]


def ppm_write_file(rgb, path, gamma=False):
    rgb = np.ascontiguousarray(rgb, np.uint8)
    check(lib().rt_ppm_write_file(ptr(rgb), rgb.shape[0], rgb.shape[1], int(gamma), os.fsencode(path)))


def gamma_correct(b):
    return int(lib().rt_gamma_correct(int(b)))
