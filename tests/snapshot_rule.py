"""The snapshot format of rt_frame_save / rt_frame_resume (include/rtfs_b200.h) restated in numpy: parse a snapshot into its
header, view table and pixel sections, write one back, and compute its checksum.  The tests compare the library's bytes with
what this module reads and writes, and build snapshots the library must refuse."""
import ctypes as C

import numpy as np

from ray_tracing_fsharp_b200 import abi

MAGIC = b"RTFSSNAP"
HEADER_BYTES = C.sizeof(abi.RtSnapshotHeader)
VIEW_ENTRY_BYTES = C.sizeof(abi.RtCamera) + 8
CHECKSUM_WORD = abi.RtSnapshotHeader.checksum.offset // 8
GOLDEN = np.uint64(0x9E3779B97F4A7C15)


def mix(i, w):
    """splitmix64's finalizer of w + (i + 1) golden, elementwise over uint64 arrays (mod 2^64)."""
    with np.errstate(over="ignore"):
        z = w.astype(np.uint64) + (i.astype(np.uint64) + np.uint64(1)) * GOLDEN
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def checksum(data: bytes) -> int:
    """sum over the file's uint64 words of mix(i, w_i) mod 2^64, the checksum field read as 0."""
    w = np.frombuffer(data, "<u8").copy()
    w[CHECKSUM_WORD] = 0
    with np.errstate(over="ignore"):
        return int(mix(np.arange(w.size, dtype=np.uint64), w).sum(dtype=np.uint64))


def sections(header):
    """(byte offset of the view table, of the pixel sections, total bytes) for a header."""
    n, noise = int(header.n_pixels), bool(header.opts.flags & abi.RT_FLAG_NOISE)
    table = HEADER_BYTES
    at = table + (header.n_views * VIEW_ENTRY_BYTES if header.kind == abi.RT_FRAME_VIEWS else 0)
    return table, at, at + 8 * (n * (3 if noise else 2) + (n + 63) // 64)


def parse(data: bytes):
    """{header, cameras, seeds, sums int32 [n, 4], sq uint64 [n] or None, active bool [n]} of a snapshot."""
    h = abi.RtSnapshotHeader.from_buffer_copy(data[:HEADER_BYTES])
    assert h.magic == MAGIC and h.version == abi.RT_SNAPSHOT_VERSION and h.header_bytes == HEADER_BYTES
    table, at, total = sections(h)
    assert h.total_bytes == total == len(data)
    cameras, seeds = [], []
    if h.kind == abi.RT_FRAME_VIEWS:
        for v in range(h.n_views):
            e = table + v * VIEW_ENTRY_BYTES
            cameras.append(abi.RtCamera.from_buffer_copy(data[e:e + C.sizeof(abi.RtCamera)]))
            seeds.append(int(np.frombuffer(data[e + C.sizeof(abi.RtCamera):e + VIEW_ENTRY_BYTES], "<u8")[0]))
    n = int(h.n_pixels)
    sums = np.frombuffer(data, "<i4", 4 * n, at).reshape(n, 4).copy()
    at += 16 * n
    sq = None
    if h.opts.flags & abi.RT_FLAG_NOISE:
        sq = np.frombuffer(data, "<u8", n, at).copy()
        at += 8 * n
    words = np.frombuffer(data, "<u4", 2 * ((n + 63) // 64), at)
    active = np.unpackbits(words.view(np.uint8), bitorder="little")[:n].astype(bool)
    return {"header": h, "cameras": cameras, "seeds": seeds, "sums": sums, "sq": sq, "active": active}


def write(parts) -> bytes:
    """The snapshot of parse()'s dict, with total_bytes and the checksum recomputed (the other header fields as given)."""
    h = abi.RtSnapshotHeader.from_buffer_copy(bytes(parts["header"]))
    n = int(h.n_pixels)
    _, _, total = sections(h)
    h.total_bytes = total
    h.checksum = 0
    out = bytearray(bytes(h))
    if h.kind == abi.RT_FRAME_VIEWS:
        for cam, seed in zip(parts["cameras"], parts["seeds"]):
            out += bytes(cam) + np.uint64(seed).tobytes()
    out += np.ascontiguousarray(parts["sums"], "<i4").tobytes()
    if h.opts.flags & abi.RT_FLAG_NOISE:
        out += np.ascontiguousarray(parts["sq"], "<u8").tobytes()
    bits = np.zeros(64 * ((n + 63) // 64), np.uint8)
    bits[:n] = np.asarray(parts["active"], bool)
    out += np.packbits(bits, bitorder="little").tobytes()
    assert len(out) == total
    c = checksum(bytes(out))
    out[8 * CHECKSUM_WORD:8 * CHECKSUM_WORD + 8] = np.uint64(c).tobytes()
    return bytes(out)


def synthetic(n_pixels=150, noise=True, kind=abi.RT_FRAME_CAMERA, n_views=1, seed=0):
    """A snapshot of made-up, self-consistent content (for format tests without a device)."""
    rng = np.random.default_rng(seed)
    h = abi.RtSnapshotHeader()
    h.magic, h.version, h.header_bytes = MAGIC, abi.RT_SNAPSHOT_VERSION, HEADER_BYTES
    h.kind, h.n_views, h.n_pixels = kind, n_views, n_pixels
    h.opts.flags = abi.RT_FLAG_NOISE if noise else 0
    h.samples_done, h.n_probe = 40, 11
    counts = np.where(rng.random(n_pixels) < 0.5, 40, 11).astype(np.int32)
    sums = np.zeros((n_pixels, 4), np.int32)
    sums[:, 3] = counts
    sums[:, :3] = (rng.integers(0, 256, (n_pixels, 3)) * counts[:, None]).astype(np.int32)
    active = counts == 40
    h.paths_done, h.pixels_active, h.pixels_flagged = int(counts.sum()), int(active.sum()), int(active.sum())
    cams = [abi.RtCamera(samples_per_pixel=64, bounce_depth=v) for v in range(n_views)] if kind == abi.RT_FRAME_VIEWS else []
    sq = rng.integers(0, 3 * 255 * 255, n_pixels).astype(np.uint64) * counts.astype(np.uint64) if noise else None
    return write({"header": h, "cameras": cams, "seeds": [1000 + v for v in range(len(cams))], "sums": sums, "sq": sq, "active": active})
