"""Host-side mirror of the reference's render surface: Camera, Scene, Image, ImageOutput.

Same names, argument order and meaning as the F# modules, so that callers (and tests) read like the
reference's.  Everything that computes goes through the C ABI (native.py); nothing here traces rays.

  Camera.make_basic     RayTracing/Camera.fs:34-59
  Scene.make            RayTracing/Scene.fs:15-28
  Scene.update          Scene.make of an edited object list, done in place on the device (rt_scene_update)
  Scene.render          RayTracing/Scene.fs:196-236
  Scene.render_views    Scene.render of many cameras of one scene in one submission (rt_render_views; one GPU or several)
  Scene.render_progressive  the same frame in sample passes, progress ticks as passes finish (native.Frame, one GPU or several)
  Scene.render_views_progressive  Scene.render_views in sample passes, as one progressive frame of the batch (one GPU or several)
  Scene.resume_progressive  a progressive frame saved by Frame.save, continued to its target (one GPU or several)
  Scene.render_window   a window (row0, col0, rows, cols) of Scene.render's image, without tracing the rest (rt_render_window)
  Image / Image.render  RayTracing/Domain.fs:9-31
  ImageOutput.write_ppm RayTracing/ImageOutput.fs:163-197, PixelOutput.correct :11-18
"""
import ctypes as C
import os
import secrets
from dataclasses import dataclass
from typing import Callable, List, Optional, Sequence

import numpy as np

from . import abi, native
from .domain import marshal


class Camera:
    @staticmethod
    def make_basic(samples_per_pixel: int, focal_length: float, aspect_ratio: float, origin, view_direction, view_up) -> abi.RtCamera:
        """Camera.makeBasic.  BounceDepth is 150 as in the reference (Camera.fs:58); override the field
        like `{ camera with BounceDepth = 50 }`: `cam.bounce_depth = 50`."""
        return native.camera_make_basic(samples_per_pixel, focal_length, aspect_ratio, origin, view_direction, view_up)


@dataclass
class Image:
    """Domain.fs:9-15: `Rows` is a sequence of deferred rows; here each is a thunk returning uint8 [cols, 3]."""
    Rows: Sequence[Callable[[], np.ndarray]]
    RowCount: int
    ColCount: int
    # set by Scene.render: forces every row at once (one frame, one progress call per row) without 2·maxH+1 array copies
    _all_rows: Optional[Callable[[], np.ndarray]] = None

    @staticmethod
    def row_count(i: "Image") -> int:
        return i.RowCount

    @staticmethod
    def col_count(i: "Image") -> int:
        return i.ColCount

    @staticmethod
    def render(i: "Image") -> np.ndarray:
        """Image.render (Domain.fs:23-24): force every row; returns uint8 [rows, cols, 3]."""
        if i._all_rows is not None:
            return i._all_rows()
        return np.stack([row() for row in i.Rows]) if i.RowCount else np.zeros((0, i.ColCount, 3), np.uint8)


class Scene:
    """Scene.make / Scene.render.  The record is opaque, as in the reference (Scene.fs:5-9)."""

    def __init__(self, handle, hittables, textures, keep, devices):
        self._handle = handle
        self._hittables, self._textures, self._keep = hittables, textures, keep
        self._devices = devices
        self.last_stats: Optional[abi.RtStats] = None

    @staticmethod
    def make(objects, device: int = 0, devices: Optional[List[int]] = None) -> "Scene":
        """Scene.make: partitions bounded / unbounded objects and builds the BVH (host), uploads it.
        `devices=[...]` (more than one) splits every frame over those GPUs of this process."""
        hittables, textures, keep = marshal(objects)
        if devices is not None and len(devices) > 1:
            handle = native.MultiHandle(hittables, textures, devices, keepalive=keep)
            return Scene(handle, hittables, textures, keep, list(devices))
        dev = devices[0] if devices else device
        handle = native.SceneHandle(hittables, textures, dev, keepalive=keep)
        return Scene(handle, hittables, textures, keep, [dev])

    @property
    def handle(self):
        return self._handle

    @staticmethod
    def update(s: "Scene", objects) -> abi.RtSceneUpdate:
        """The scene Scene.make(objects) would give, made in place: `objects` is the whole new object list (as F# holds it, an
        immutable array).  It is marshalled and diffed against the scene's current records, and only the changed objects and
        textures go to the device (rt_scene_update), which refits the tree there; the scene then renders bit for bit as
        Scene.make(objects).  The structure must stay: the object count, each object's shape, the sign of each bounded
        sphere's radius, and the texture table (its size, each texture's kind, an image's size); otherwise ValueError (make a
        new scene).  Progressive frames opened before the call are stale.  A scene made with devices=[...] (several GPUs):
        NotImplementedError.  Returns the RtSceneUpdate."""
        if not isinstance(s._handle, native.SceneHandle):
            raise NotImplementedError("Scene.update edits a scene of one device; make a scene split over devices=[...] anew")
        hittables, textures, keep = marshal(objects)
        if len(hittables) != len(s._hittables):
            raise ValueError(f"Scene.update: {len(hittables)} objects for a scene of {len(s._hittables)}: make a new scene")
        if len(textures) != len(s._textures) or any(_texture_shape(a) != _texture_shape(b) for a, b in zip(textures, s._textures)):
            raise ValueError("Scene.update: the texture table changes its structure (count, kinds or image sizes): make a new scene")
        size = C.sizeof(abi.RtHittable)
        new = np.frombuffer(hittables, np.uint8).reshape(-1, size) if len(hittables) else np.zeros((0, size), np.uint8)
        old = np.frombuffer(s._hittables, np.uint8).reshape(-1, size) if len(s._hittables) else np.zeros((0, size), np.uint8)
        changed = np.nonzero((new != old).any(axis=1))[0].tolist()
        tex_changed = [j for j, (a, b) in enumerate(zip(textures, s._textures)) if not _same_texture(a, b)]
        info = s._handle.update(changed, [hittables[i] for i in changed], tex_changed, [textures[j] for j in tex_changed])
        s._hittables, s._textures, s._keep = hittables, textures, keep
        s._handle._h, s._handle._t, s._handle._keep = hittables, native._as_array(abi.RtTexture, textures), keep
        return info

    @staticmethod
    def add(s: "Scene", objects) -> abi.RtSceneRebuild:
        """Appends `objects` to the scene, in place (rt_scene_rebuild): the scene then renders bit for bit as Scene.make of its
        objects followed by these, and the new objects take the next indices.  Their textures must be textures the scene
        already holds (a texture table cannot grow here; otherwise ValueError: make a new scene).  Progressive frames opened
        before the call are stale.  A scene made with devices=[...] (several GPUs): NotImplementedError."""
        hittables, textures, keep = marshal(objects)
        remap = []
        for t in textures:
            same = [j for j, u in enumerate(s._textures) if _same_texture(t, u)]
            if not same:
                raise ValueError("Scene.add: an object brings a texture the scene does not hold: make a new scene")
            remap.append(same[0])
        for h in hittables:
            if h.texture >= 0:
                h.texture = remap[h.texture]
        return Scene._restructure(s, [], list(hittables), keep)

    @staticmethod
    def remove(s: "Scene", indices) -> abi.RtSceneRebuild:
        """Removes the objects at `indices`, in place (rt_scene_rebuild): the others keep their order and are renumbered
        densely, and the scene renders bit for bit as Scene.make of them.  Bad or repeated indices: RtError
        RT_ERR_INVALID_ARGUMENT.  Progressive frames opened before the call are stale.  A scene made with devices=[...]:
        NotImplementedError."""
        return Scene._restructure(s, list(indices), [], None)

    @staticmethod
    def rebuild(s: "Scene") -> abi.RtSceneRebuild:
        """Builds the scene's tree anew on the device from its current objects: the remedy for a tree that Scene.update's
        refits have left slow to walk (DESIGN.md section 20).  Frames are unchanged bit for bit; progressive frames opened
        before the call are stale.  A scene made with devices=[...]: NotImplementedError."""
        return Scene._restructure(s, [], [], None)

    @staticmethod
    def _restructure(s: "Scene", remove, append, keep) -> abi.RtSceneRebuild:
        if not isinstance(s._handle, native.SceneHandle):
            raise NotImplementedError("structural edits change a scene of one device; make a scene split over devices=[...] anew")
        info = s._handle.rebuild(remove, append)
        size = C.sizeof(abi.RtHittable)
        old = np.frombuffer(s._hittables, np.uint8).reshape(-1, size) if len(s._hittables) else np.zeros((0, size), np.uint8)
        kept = np.ones(len(old), bool)
        kept[np.asarray(remove, np.int64)] = False
        buf = bytearray(old[kept].tobytes() + b"".join(bytes(h) for h in append))
        n = len(buf) // size
        hittables = (abi.RtHittable * n).from_buffer(buf) if n else (abi.RtHittable * 0)()
        s._hittables = hittables
        s._keep = (s._keep, keep) if keep is not None else s._keep
        s._handle._h, s._handle._keep = hittables, s._keep
        return info

    @staticmethod
    def render(progress_increment: Callable[[float], None], print_fn: Callable[[str], None], max_width_coord: int, max_height_coord: int,
               camera: abi.RtCamera, s: "Scene", seed: Optional[int] = None, adaptive: bool = True, mode: int = abi.RT_MODE_MEGAKERNEL,
               flags: int = 0, frames: Optional["native.FrameRing"] = None):
        """Scene.render: returns (total progress, Image).  Like the reference it is lazy: nothing is
        traced until a row is forced; the first forced row renders the whole frame on the GPU.
        `seed`: key of the counter RNG; None draws one from the OS as `FloatProducer (Random ())` does
        (Scene.fs:205).  `frames`: a native.FrameRing to take the output array from (explicit reuse by a host that renders
        frame after frame); by default every frame is a fresh array.  `print_fn` is accepted and ignored exactly as the reference ignores it (Scene.fs:158)."""
        rows, cols = 2 * max_height_coord + 1, 2 * max_width_coord + 1  # Scene.fs:208-209
        if seed is None:
            seed = secrets.randbits(64)
        state = {}

        def frame():
            if "rgb" not in state:
                out = frames.next() if frames is not None else None
                if isinstance(s._handle, native.MultiHandle):
                    rgb, _, stats = s._handle.render(camera, max_width_coord, max_height_coord, seed=seed, adaptive=adaptive, flags=flags,
                                                     rgb_out=out)
                else:
                    rgb, _, stats = s._handle.render(camera, max_width_coord, max_height_coord, seed=seed, adaptive=adaptive, mode=mode,
                                                     flags=flags, rgb_out=out)
                s.last_stats = stats
                state["rgb"] = rgb
            return state["rgb"]

        def row_thunk(r):
            def force():
                out = frame()[r]
                progress_increment(1.0)  # Scene.fs:232
                return out
            return force

        def all_rows():
            out = frame()
            for _ in range(rows):
                progress_increment(1.0)
            return out

        return float(rows), Image([row_thunk(r) for r in range(rows)], rows, cols, all_rows)

    @staticmethod
    def render_views(progress_increment: Callable[[float], None], print_fn: Callable[[str], None], max_width_coord: int,
                     max_height_coord: int, cameras: Sequence[abi.RtCamera], s: "Scene", seed: Optional[int] = None,
                     seeds: Optional[Sequence[int]] = None, adaptive: bool = True, flags: int = 0):
        """Scene.render for every camera of `cameras` (same samples_per_pixel and bounce_depth; a turntable, a fly-through,
        stereo pairs, previews), rendered together by one GPU (native.SceneHandle.render_views).  Returns (total progress,
        [Image per camera]); lazy like Scene.render: the first forced row renders every view.  The progress ticks total
        rows * len(cameras), one per row forced.  `seeds`: one RNG key per view; otherwise `seed` (None: one drawn from the
        OS) for every view.  With the same camera and seed, view v is Scene.render's image.  On a scene made with
        devices=[...] the batch is split over those GPUs (native.MultiHandle.render_views), bit for bit the batch of one GPU.
        `print_fn` is ignored."""
        rows, cols = 2 * max_height_coord + 1, 2 * max_width_coord + 1
        n = len(cameras)
        if seed is None and seeds is None:
            seed = secrets.randbits(64)
        state = {}

        def frames():
            if "rgb" not in state:
                rgb, _, stats = s._handle.render_views(list(cameras), max_width_coord, max_height_coord, seeds=seeds, seed=seed or 0,
                                                       adaptive=adaptive, flags=flags)
                s.last_stats = stats
                state["rgb"] = rgb
            return state["rgb"]

        def image(v):
            def row_thunk(r):
                def force():
                    out = frames()[v, r]
                    progress_increment(1.0)
                    return out
                return force

            def all_rows():
                out = frames()[v]
                for _ in range(rows):
                    progress_increment(1.0)
                return out
            return Image([row_thunk(r) for r in range(rows)], rows, cols, all_rows)

        return float(rows * n), [image(v) for v in range(n)]

    @staticmethod
    def render_window(progress_increment: Callable[[float], None], print_fn: Callable[[str], None], max_width_coord: int,
                      max_height_coord: int, camera: abi.RtCamera, s: "Scene", window, seed: Optional[int] = None, adaptive: bool = True,
                      flags: int = 0):
        """The window (row0, col0, rows, cols) of Scene.render's image, rendered by one GPU without the rest of the frame
        (native.SceneHandle.render_window): a closer look at one part of a frame, or one tile of a frame split into tiles.
        Returns (total progress, Image of rows x cols); lazy like Scene.render: the first forced row renders the window, and
        the progress ticks total the window's rows.  With the same camera and seed, window pixel (r, c) is Scene.render's
        pixel (row0 + r, col0 + c).  `print_fn` is ignored."""
        if not isinstance(s._handle, native.SceneHandle):
            raise NotImplementedError("a window runs on one GPU: make the scene with a single device")
        row0, col0, rows, cols = (int(x) for x in window)
        if seed is None:
            seed = secrets.randbits(64)
        state = {}

        def frame():
            if "rgb" not in state:
                rgb, _, stats = s._handle.render_window(camera, max_width_coord, max_height_coord, (row0, col0, rows, cols), seed=seed,
                                                        adaptive=adaptive, flags=flags)
                s.last_stats = stats
                state["rgb"] = rgb
            return state["rgb"]

        def row_thunk(r):
            def force():
                out = frame()[r]
                progress_increment(1.0)
                return out
            return force

        def all_rows():
            out = frame()
            for _ in range(rows):
                progress_increment(1.0)
            return out

        return float(rows), Image([row_thunk(r) for r in range(rows)], rows, cols, all_rows)

    @staticmethod
    def render_progressive(progress_increment: Callable[[float], None], print_fn: Callable[[str], None], max_width_coord: int,
                           max_height_coord: int, camera: abi.RtCamera, s: "Scene", seed: Optional[int] = None, adaptive: bool = True,
                           target_ms: float = 250.0, on_pass: Optional[Callable[[abi.RtFrameProgress, "native.Frame"], object]] = None,
                           flags: int = 0, noise_tolerance: Optional[float] = None, noise_fraction: float = 0.0,
                           converge_tolerance: Optional[float] = None, converge_min_samples: int = 64,
                           converge_interval: int = 64, window=None) -> np.ndarray:
        """Scene.render's frame rendered in passes of about `target_ms` of device time each (native.Frame; on a scene made
        with devices=[...], one frame split over those GPUs, bit for bit the frame of one GPU).
        `progress_increment(1.0)` is called as passes complete, in proportion to the paths traced so far out of the frame's
        total, and exactly `rows` times in all, like the reference's one call per row (Scene.fs:232).  After every pass
        `on_pass(progress, frame)` is called, if given: it may read the current image (`frame.read()`, exactly the frame of
        `progress.samples_done` samples per pixel) and stops the frame by returning True.  Returns the pixels (uint8
        [rows, cols, 3], before gamma): with the same seed, Scene.render's image, or that of the samples done when stopped.
        `print_fn` is accepted and ignored as in Scene.render.  To checkpoint the frame, `on_pass` may call `frame.save()`:
        Scene.resume_progressive continues the snapshot later, in this process or another, bit for bit.
        With `noise_tolerance` (8-bit levels) the frame also keeps its noise estimate (abi.RT_FLAG_NOISE, Frame.noise) and
        stops at the first check where at most `noise_fraction` of the pixels still being sampled have a standard error
        of the mean above the tolerance.  The check runs after the probe and after every pass (after `on_pass`); the image
        returned is then rt_render's at the samples done.
        With `converge_tolerance` (8-bit levels) each pixel stops being sampled once its standard error is within it, checked
        at converge_min_samples + j * converge_interval samples (Frame.set_convergence): every pixel is then rt_render's pixel
        at the sample count it stopped at.  It composes with the `noise_tolerance` stop, whose summary then covers the pixels
        still being sampled.
        With `window` = (row0, col0, rows, cols) only that window of the frame is traced (native.SceneHandle.open_frame_window):
        the progress ticks total the window's rows, and the pixels returned ([rows, cols, 3]) are exactly that crop of the
        frame rendered without it; a window runs on one GPU (NotImplementedError on a scene made with devices=[...])."""
        if window is not None and not isinstance(s._handle, native.SceneHandle):
            raise NotImplementedError("a window runs on one GPU: make the scene with a single device")
        rows = 2 * max_height_coord + 1 if window is None else int(window[2])
        if seed is None:
            seed = secrets.randbits(64)
        if noise_tolerance is not None or converge_tolerance is not None:
            flags |= abi.RT_FLAG_NOISE
        if window is None:
            opened = s._handle.open_frame(camera, max_width_coord, max_height_coord, seed=seed, adaptive=adaptive, flags=flags)
        else:
            opened = s._handle.open_frame_window(camera, max_width_coord, max_height_coord, window, seed=seed, adaptive=adaptive, flags=flags)
        with opened as frame:
            if converge_tolerance is not None:
                frame.set_convergence(converge_tolerance, converge_min_samples, converge_interval)
            return _run_passes(frame, rows, progress_increment, target_ms, on_pass, noise_tolerance, noise_fraction)

    @staticmethod
    def render_views_progressive(progress_increment: Callable[[float], None], print_fn: Callable[[str], None], max_width_coord: int,
                                 max_height_coord: int, cameras: Sequence[abi.RtCamera], s: "Scene", seeds: Optional[Sequence[int]] = None,
                                 seed: Optional[int] = None, adaptive: bool = True, target_ms: float = 250.0,
                                 on_pass: Optional[Callable[[abi.RtFrameProgress, "native.Frame"], object]] = None, flags: int = 0,
                                 converge_tolerance: Optional[float] = None, converge_min_samples: int = 64,
                                 converge_interval: int = 64) -> List[np.ndarray]:
        """render_progressive for every camera of `cameras` (same samples_per_pixel and bounce_depth), as one progressive frame
        of the batch (native.SceneHandle.open_frame_views): each pass of about `target_ms` of device time advances every view.
        The progress ticks total rows * len(cameras), spread over the paths traced as in render_progressive.  `on_pass(progress,
        frame)` after every pass may read the views (`frame.read()`, [n, rows, cols, 3]) and stops the batch by returning True.
        `seeds`: one RNG key per view; otherwise `seed` (None: one drawn from the OS) for every view.  With
        `converge_tolerance` every pixel of every view stops once its standard error is within it, checked at
        converge_min_samples + j * converge_interval samples (Frame.set_convergence).  Returns one uint8 [rows, cols, 3] image
        per view (before gamma): with the same camera and seed, view v is render_progressive's image of camera v with the same
        rule, or, stopped early, that of the samples done.  On a scene made with devices=[...] the frame is split over those
        GPUs (native.MultiHandle.open_frame_views), bit for bit the frame of one GPU after every pass.  `print_fn` is
        ignored."""
        rows, n = 2 * max_height_coord + 1, len(cameras)
        if seed is None and seeds is None:
            seed = secrets.randbits(64)
        if converge_tolerance is not None:
            flags |= abi.RT_FLAG_NOISE
        with s._handle.open_frame_views(list(cameras), max_width_coord, max_height_coord, seeds=seeds, seed=seed or 0, adaptive=adaptive,
                                        flags=flags) as frame:
            if converge_tolerance is not None:
                frame.set_convergence(converge_tolerance, converge_min_samples, converge_interval)
            rgb = _run_passes(frame, rows * n, progress_increment, target_ms, on_pass, None, 0.0)
        return [rgb[v] for v in range(n)]

    @staticmethod
    def resume_progressive(progress_increment: Callable[[float], None], print_fn: Callable[[str], None], snapshot, s: "Scene",
                           target_ms: float = 250.0, on_pass: Optional[Callable[[abi.RtFrameProgress, "native.Frame"], object]] = None,
                           noise_tolerance: Optional[float] = None, noise_fraction: float = 0.0):
        """Continues a frame saved by Frame.save (for instance from render_progressive's `on_pass`) to its target, on `s`,
        which must hold the objects and textures of the scene the frame was saved from (one GPU or devices=[...], whatever
        the device count that saved it).  Returns what render_progressive (or render_views_progressive, for a batch of
        views) would have returned had the frame never stopped: bit for bit the same pixels.  The progress ticks total the
        same rows (times views) as the original call; the share already done is emitted at once.  `target_ms`, `on_pass`,
        `noise_tolerance` and `noise_fraction` act as in render_progressive (the noise stop needs a frame saved with its
        noise estimate); the convergence rule the frame was saved with still applies.  `print_fn` is ignored."""
        with s._handle.resume_frame(snapshot) as frame:
            rows = frame.rows * (frame.n_views or 1)
            rgb = _run_passes(frame, rows, progress_increment, target_ms, on_pass, noise_tolerance, noise_fraction)
        return rgb if frame.n_views is None else [rgb[v] for v in range(frame.n_views)]


def _run_passes(frame: "native.Frame", total_ticks: int, progress_increment: Callable[[float], None], target_ms: float, on_pass,
                noise_tolerance: Optional[float], noise_fraction: float) -> np.ndarray:
    """The passes of render_progressive and its kin, from the frame's current state to its target, an `on_pass` that
    returns True, or the noise stop: `total_ticks` progress ticks spread over the paths traced (what the frame already
    holds is emitted at once), then the frame's pixels."""
    ticks = ProgressTicks(total_ticks)

    def emit(n):
        for _ in range(n):
            progress_increment(1.0)

    def converged(progress):
        if noise_tolerance is None or progress.done:
            return False
        summary, _, _ = frame.noise(noise_tolerance, want_map=False)
        return summary.pixels_above <= noise_fraction * summary.pixels

    progress = frame.progress
    emit(ticks.update(progress.paths_done, progress.paths_target))  # the probe (or what a resumed frame holds)
    stop = converged(progress)
    while not progress.done and not stop:
        progress = frame.advance(target_ms=target_ms)
        if not progress.done:
            emit(ticks.update(progress.paths_done, progress.paths_target))
        if on_pass is not None and on_pass(progress, frame):
            break
        stop = converged(progress)
    rgb, _ = frame.read()
    emit(ticks.finish())  # the last pass's share, or the rest of the frame when on_pass stopped it
    return rgb


def _texture_shape(t: abi.RtTexture):
    """What rt_scene_update must keep of a texture: its kind and, for an image, its size."""
    return (t.kind, t.width, t.height) if t.kind == abi.RT_TEX_IMAGE else (t.kind,)


def _texels(t: abi.RtTexture) -> bytes:
    return C.string_at(t.rgb8, t.width * t.height * 3) if t.kind == abi.RT_TEX_IMAGE else b""


def _same_texture(a: abi.RtTexture, b: abi.RtTexture) -> bool:
    """Every field but the texel pointer, and the texels."""
    fields = [f for f, _ in abi.RtTexture._fields_ if f != "rgb8"]
    return all(_plain(getattr(a, f)) == _plain(getattr(b, f)) for f in fields) and _texels(a) == _texels(b)


def _plain(v):
    return list(v) if isinstance(v, C.Array) else v


class ProgressTicks:
    """Spreads `total` progress ticks over a quantity that grows towards a target: after update(done, target) the ticks
    handed out so far are floor(total * done / target), so the fractional part carries into the next update, and
    finish() hands out the rest.  However the updates fall, the ticks add up to exactly `total`."""

    def __init__(self, total: int):
        self.total = int(total)
        self.emitted = 0

    def update(self, done: int, target: int) -> int:
        """Number of ticks to emit now."""
        want = self.total if target <= 0 or done >= target else (self.total * int(done)) // int(target)
        n = max(0, want - self.emitted)
        self.emitted += n
        return n

    def finish(self) -> int:
        n = self.total - self.emitted
        self.emitted = self.total
        return n


class PixelOutput:
    @staticmethod
    def correct(b: int) -> int:
        """PixelOutput.correct (ImageOutput.fs:11-18)."""
        return native.gamma_correct(b)


class ImageOutput:
    @staticmethod
    def write_ppm(gamma_correct: bool, pixels: np.ndarray, path: Optional[os.PathLike] = None) -> bytes:
        """ImageOutput.writePpm (ImageOutput.fs:163-197): P3 text, byte-identical format."""
        data = native.ppm_format(pixels, gamma_correct)
        if path is not None:
            native.ppm_write_file(pixels, path, gamma_correct)
        return data
