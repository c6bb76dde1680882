"""numpy restatement of the tree refit of rt_scene_update (csrc/rtfs_edit.cu), which the device is held to exactly.

A leaf's box is the directed rounding of its FP32 sphere, computed in FP64: [round_down(c - r), round_up(c + r)] per axis, c and r
the FP32 centre and radius (build_device_layout).  A node's box is the union of its two children's boxes.  device_node_of turns a
node's two child boxes into the centre / half-extent form the render kernels walk.

The tree is given as rt_scene_bvh_nodes hands it out (DFS pre-order, left child = i + 1, `right`, `prim` the caller's object
index of a leaf); refit() recomputes every box of that topology from the objects' current centres and radii."""
import numpy as np

F32, F64 = np.float32, np.float64


def round_down(v):
    """The FP32 value nearest each FP64 v towards -inf."""
    v = np.asarray(v, F64)
    f = v.astype(F32)
    return np.where(f.astype(F64) > v, np.nextafter(f, F32(-np.inf)), f).astype(F32)


def round_up(v):
    """The FP32 value nearest each FP64 v towards +inf."""
    v = np.asarray(v, F64)
    f = v.astype(F32)
    return np.where(f.astype(F64) < v, np.nextafter(f, F32(np.inf)), f).astype(F32)


def leaf_box(centre, radius):
    """(min, max) float32 [3] of the sphere with FP64 centre [3] and radius, as the host build and the device refit form it."""
    c = np.asarray(centre, F64).astype(F32).astype(F64)
    r = F64(F32(radius))
    return round_down(c - r), round_up(c + r)


def refit(right, prim, objects):
    """Boxes float32 [n, 6] (min xyz, max xyz) of every node of the tree (right, prim) over `objects` (a sequence of
    RtHittable): leaves from their spheres, every other node the union of its children."""
    n = len(right)
    boxes = np.zeros((n, 6), F32)
    for i in range(n - 1, -1, -1):  # children come after their parent in pre-order
        if right[i] < 0:
            h = objects[int(prim[i])]
            mn, mx = leaf_box(list(h.p), h.radius)
        else:
            l, r = boxes[i + 1], boxes[right[i]]
            mn, mx = np.minimum(l[:3], r[:3]), np.maximum(l[3:], r[3:])
        boxes[i, :3], boxes[i, 3:] = mn, mx
    return boxes


def device_node_of(mn, mx):
    """(centre, half-extent) float32 [3] of one child box in the form the render kernels walk: the centre rounded to nearest
    from the FP64 midpoint, the half-extent the larger FP64 distance to either face rounded up, then one ulp more; a
    non-finite box (the never-entered right child of a one-sphere tree) becomes centre 1e30, half-extent 0."""
    mn, mx = np.asarray(mn, F32), np.asarray(mx, F32)
    finite = np.isfinite(mn) & np.isfinite(mx)
    m64, x64 = np.where(finite, mn, 0).astype(F64), np.where(finite, mx, 0).astype(F64)
    c = (F64(0.5) * (m64 + x64)).astype(F32)
    h = round_up(np.maximum(x64 - c.astype(F64), c.astype(F64) - m64))
    h = np.nextafter(h, F32(np.inf))
    return np.where(finite, c, F32(1e30)), np.where(finite, h, F32(0))
