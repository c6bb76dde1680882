"""numpy restatement of the device tree builder of rt_scene_rebuild (csrc/rtfs_build.cu), which the device is held to node for
node.

PLOC, parallel locally-ordered clustering (Meister & Bittner, TVCG 2018), over the spheres of the tree (shape sphere, radius
>= 0) of an object array:
  - leaf boxes are refit_rule.leaf_box, the host build's directed roundings of the FP32 sphere;
  - 30-bit Morton codes of the FP32 centres over their exact min / max bounds: per axis floor((c - lo) * (1024 / (hi - lo))),
    each operation rounded to FP32, at most 1023 (0 on an axis without extent); keys (morton << 32 | caller index), sorted;
  - clustering: each cluster's nearest neighbour among RADIUS clusters either side by the FP32 area
    (dx dy + dy dz) + dz dx of the union box (NaN counts as +inf), ties to the lower index; mutual pairs merge into the
    lower slot as a node numbered in slot order after the nodes of earlier iterations (left child the lower slot's
    cluster), and the clusters keep their order;
  - the tree is written in DFS pre-order from the last node made, which is the root.

build() returns the tree as rt_scene_bvh_nodes hands it out: per record (leaves included) its box as float64 [6] (min xyz,
max xyz), `right` (-1 for a leaf) and `prim` (the caller's object index of a leaf, -1 otherwise); and the depth in internal
nodes (root 1) that RtSceneRebuild reports."""
import numpy as np

import refit_rule

F32 = np.float32
RADIUS = 16
SHAPE_SPHERE = 0


def bounded_spheres(objects):
    """Caller indices, FP32 centres [n, 3] and FP32 radii [n] of the spheres of the tree."""
    idx = [i for i, h in enumerate(objects) if h.shape == SHAPE_SPHERE and h.radius >= 0.0]
    c = np.array([list(objects[i].p) for i in idx], np.float64).reshape(-1, 3).astype(F32)
    r = np.array([objects[i].radius for i in idx], np.float64).astype(F32)
    return np.array(idx, np.int64), c, r


def morton_keys(idx, c):
    lo, hi = c.min(axis=0), c.max(axis=0)
    code = np.zeros(len(idx), np.uint64)
    for a in range(3):
        ext = F32(hi[a] - lo[a])
        if ext > 0:
            q = ((c[:, a] - lo[a]).astype(F32) * F32(F32(1024) / ext)).astype(F32)
            v = np.where(q >= F32(1023), 1023, q.astype(np.int64)).astype(np.uint64)
        else:
            v = np.zeros(len(idx), np.uint64)
        spread = np.zeros(len(idx), np.uint64)
        for b in range(10):
            spread |= ((v >> np.uint64(b)) & np.uint64(1)) << np.uint64(3 * b)
        code |= spread << np.uint64(2 - a)
    return (code << np.uint64(32)) | idx.astype(np.uint64)


def union_area(mn_a, mx_a, mn_b, mx_b):
    d = (np.maximum(mx_a, mx_b) - np.minimum(mn_a, mn_b)).astype(F32)
    with np.errstate(invalid="ignore", over="ignore"):
        s = ((d[..., 0] * d[..., 1]).astype(F32) + (d[..., 1] * d[..., 2]).astype(F32)).astype(F32) + (d[..., 2] * d[..., 0]).astype(F32)
    s = s.astype(F32)
    return np.where(np.isnan(s), F32(np.inf), s)


def nearest(mn, mx):
    m = len(mn)
    best = np.full(m, -1, np.int64)
    best_d = np.zeros(m, F32)
    i = np.arange(m)
    for off in range(-RADIUS, RADIUS + 1):  # ascending j: a strict < keeps the lower index on ties
        if off == 0:
            continue
        j = i + off
        ok = (j >= 0) & (j < m)
        jj = np.clip(j, 0, m - 1)
        d = union_area(mn, mx, mn[jj], mx[jj])
        take = ok & ((best < 0) | (d < best_d))
        best = np.where(take, j, best)
        best_d = np.where(take, d, best_d)
    return best


def cluster(mn, mx):
    """Clusters the leaves (boxes in sorted order); returns the nodes made, in order: (left ref, right ref, l box, r box),
    a ref >= 0 a node, < 0 the leaf of sorted position ~ref; and the number of iterations."""
    ref = -1 - np.arange(len(mn))
    nodes = []
    rounds = 0
    while len(mn) > 1:
        nn = nearest(mn, mx)
        i = np.arange(len(mn))
        mutual = nn[nn] == i
        keep = ~(mutual & (nn < i))
        merge = mutual & (i < nn)
        new_ref = ref.copy()
        new_mn, new_mx = mn.copy(), mx.copy()
        for k in np.nonzero(merge)[0]:
            j = nn[k]
            nodes.append((int(ref[k]), int(ref[j]), np.concatenate([mn[k], mx[k]]), np.concatenate([mn[j], mx[j]])))
            new_ref[k] = len(nodes) - 1
            new_mn[k], new_mx[k] = np.minimum(mn[k], mn[j]), np.maximum(mx[k], mx[j])
        ref, mn, mx = new_ref[keep], new_mn[keep], new_mx[keep]
        rounds += 1
    return nodes, rounds


def build(objects):
    """(bounds [k, 6] float64, right [k], prim [k], depth) of the device tree over `objects` (a sequence of RtHittable)."""
    idx, c, r = bounded_spheres(objects)
    n = len(idx)
    if n == 0:
        return np.zeros((0, 6)), np.zeros(0, np.int32), np.zeros(0, np.int32), 0
    order = np.argsort(morton_keys(idx, c), kind="stable")
    leaf_obj = idx[order]
    boxes = [refit_rule.leaf_box(c[k].astype(np.float64), r[k]) for k in order]
    mn = np.array([b[0] for b in boxes], F32).reshape(-1, 3)
    mx = np.array([b[1] for b in boxes], F32).reshape(-1, 3)
    if n == 1:
        return np.concatenate([mn[0], mx[0]]).astype(np.float64)[None, :], np.array([-1], np.int32), np.array([leaf_obj[0]], np.int32), 1
    nodes, _ = cluster(mn, mx)
    out_box, out_right, out_prim = [], [], []
    depth = 0
    root = nodes[-1]
    stack = [(len(nodes) - 1, np.concatenate([np.minimum(root[2][:3], root[3][:3]), np.maximum(root[2][3:], root[3][3:])]), 1, None)]
    while stack:  # pre-order: a node, its left subtree, its right subtree
        ref, box, d, parent_slot = stack.pop()
        me = len(out_box)
        if parent_slot is not None:
            out_right[parent_slot] = me
        out_box.append(box.astype(np.float64))
        out_right.append(-1)
        if ref < 0:
            out_prim.append(int(leaf_obj[-1 - ref]))
            continue
        out_prim.append(-1)
        depth = max(depth, d)
        left, right, lb, rb = nodes[ref]
        stack.append((right, rb, d + 1, me))
        stack.append((left, lb, d + 1, None))
    return np.array(out_box), np.array(out_right, np.int32), np.array(out_prim, np.int32), depth


def sah_cost(bounds, right):
    """The SAH cost of a tree in rt_scene_bvh_nodes form, relative to its root's area: the area of every record, internal
    nodes and leaves alike (cost 1 each), over the root's."""
    if len(bounds) == 0:
        return 0.0
    d = bounds[:, 3:] - bounds[:, :3]
    area = d[:, 0] * d[:, 1] + d[:, 1] * d[:, 2] + d[:, 2] * d[:, 0]
    return float(area.sum() / area[0])
