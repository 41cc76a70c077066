"""K8 (rendered-depth cost, include/pgp.h) restated in numpy: the checker, never the product.

Points 1-7 of the contract, in the order they are written there, in int64 / float32 / float64 exactly as specified.  Each
triangle is evaluated over the samples of its covered pixel box; the boxes of many triangles are expanded into one candidate list
at a time (vectorised), which changes nothing: coverage and depth of a sample depend on that triangle alone, and the z-test keeps
the minimum key.  RESTATED, PARITY UNPINNED: the reference's OpenGL renderer and computeCost are not available."""
from __future__ import annotations

import numpy as np

from oracle.segment_port import decode_depth

F32 = np.float32
NEAR = F32(0.1)
GUARD = F32(1 << 20)
EMPTY = np.uint64(0xFFFFFFFFFFFFFFFF)


def pose_f32(pose44) -> np.ndarray:
    """1. the pose rounded to an fp32 3x4 (utilities::convertToMatrix)."""
    return np.asarray(pose44, np.float64).reshape(4, 4)[:3, :4].astype(np.float32)


def transform(T: np.ndarray, v: np.ndarray):
    """1. camera-frame X, Y, Z per row ((m0 x + m1 y) + m2 z) + m3, each operation rounded to fp32."""
    x, y, z = v[:, 0], v[:, 1], v[:, 2]
    with np.errstate(all="ignore"):
        return [((T[r, 0] * x + T[r, 1] * y) + T[r, 2] * z) + T[r, 3] for r in range(3)]


def project(K, X, Y, Z):
    """2. + 3. projection, snapping to 1/256 px and the per-vertex validity (finite, Z > 0.1f, inside the 2^20 px guard band)."""
    K = np.asarray(K, np.float32).reshape(9)
    fx, fy, cx, cy = K[0], K[4], K[2], K[5]
    with np.errstate(all="ignore"):
        sx = ((fx * X) / Z) + cx
        sy = ((fy * Y) / Z) + cy
        ok = np.isfinite(X) & np.isfinite(Y) & np.isfinite(Z) & (Z > NEAR) & (np.abs(sx) <= GUARD) & (np.abs(sy) <= GUARD)
        ix = np.where(ok, np.rint(sx * F32(256)), 0).astype(np.int64)
        iy = np.where(ok, np.rint(sy * F32(256)), 0).astype(np.int64)
    return ix, iy, ok


def edge(ax, ay, bx, by, px, py):
    """4. E(a, b, p) in int64 (exact: every operand is below 2^30)."""
    return (bx - ax) * (py - ay) - (by - ay) * (px - ax)


def owns(e, ax, ay, bx, by):
    """4. inside an edge, or on it when the edge a -> b is a top-left edge."""
    dx, dy = bx - ax, by - ay
    return (e > 0) | ((e == 0) & ((dy < 0) | ((dy == 0) & (dx > 0))))


def setup(ix, iy, ok, Z, tri, rows, cols):
    """3. + 4. culling and orientation; returns the kept triangles' oriented vertex ids and their covered pixel boxes."""
    tri = np.asarray(tri, np.int64).reshape(-1, 3)
    a, b, c = tri[:, 0].copy(), tri[:, 1].copy(), tri[:, 2].copy()
    keep = ok[a] & ok[b] & ok[c]
    area = edge(ix[a], iy[a], ix[b], iy[b], ix[c], iy[c])
    swap = area < 0
    b, c = np.where(swap, c, b), np.where(swap, b, c)
    keep &= area != 0
    xs, ys = np.stack([ix[a], ix[b], ix[c]]), np.stack([iy[a], iy[b], iy[c]])
    c0 = np.maximum((xs.min(0) + 255) >> 8, 0)
    c1 = np.minimum(xs.max(0) >> 8, cols - 1)
    r0 = np.maximum((ys.min(0) + 255) >> 8, 0)
    r1 = np.minimum(ys.max(0) >> 8, rows - 1)
    keep &= (c0 <= c1) & (r0 <= r1)
    k = np.nonzero(keep)[0]
    return a[k], b[k], c[k], c0[k], c1[k], r0[k], r1[k]


def fragments(projected, Z, tri, rows, cols, batch=1 << 22):
    """4. + 5. every covered (pixel, depth) of a mesh already transformed and projected (`projected` = project(...)): yields
    (flat pixel, fp32 depth, triangle) arrays batch by batch; `triangle` indexes the kept, oriented triangles in mesh order."""
    ix, iy, ok = projected
    a, b, c, c0, c1, r0, r1 = setup(ix, iy, ok, Z, tri, rows, cols)
    iz = 1.0 / Z.astype(np.float64)
    w, h = c1 - c0 + 1, r1 - r0 + 1
    n = w * h
    start = 0
    while start < len(a):
        csum = np.cumsum(n[start:])
        stop = start + max(1, int(np.searchsorted(csum, batch, side="right")))
        t = np.repeat(np.arange(start, stop), n[start:stop])
        first = np.repeat(np.cumsum(n[start:stop]) - n[start:stop], n[start:stop])
        local = np.arange(len(t)) - first
        cc = c0[t] + local % w[t]
        rr = r0[t] + local // w[t]
        px, py = cc * 256, rr * 256
        xa, ya, xb, yb, xc, yc = ix[a[t]], iy[a[t]], ix[b[t]], iy[b[t]], ix[c[t]], iy[c[t]]
        e0 = edge(xb, yb, xc, yc, px, py)
        e1 = edge(xc, yc, xa, ya, px, py)
        e2 = edge(xa, ya, xb, yb, px, py)
        inside = owns(e0, xb, yb, xc, yc) & owns(e1, xc, yc, xa, ya) & owns(e2, xa, ya, xb, yb)
        e0, e1, e2, t = e0[inside], e1[inside], e2[inside], t[inside]
        den = (e0.astype(np.float64) * iz[a[t]] + e1.astype(np.float64) * iz[b[t]]) + e2.astype(np.float64) * iz[c[t]]
        with np.errstate(over="ignore"):
            depth = ((e0 + e1 + e2).astype(np.float64) / den).astype(np.float32)
        yield rr[inside] * cols + cc[inside], depth, t
        start = stop


def _mesh_fragments(mesh, pose44, K, rows, cols):
    verts, tri = mesh[0], mesh[1]
    X, Y, Z = transform(pose_f32(pose44), np.asarray(verts, np.float32).reshape(-1, 3))
    return fragments(project(K, X, Y, Z), Z, tri, rows, cols)


def zbuffer(meshes, obj_ids, poses44, K, rows, cols) -> np.ndarray:
    """6. the per-pixel minimum of (float_bits(depth) << 32) | slot over one state; EMPTY where nothing is drawn."""
    z = np.full(rows * cols, EMPTY, np.uint64)
    for slot, (obj, pose) in enumerate(zip(obj_ids, poses44)):
        for p, d, _ in _mesh_fragments(meshes[obj], pose, K, rows, cols):
            np.minimum.at(z, p, (d.view(np.uint32).astype(np.uint64) << np.uint64(32)) | np.uint64(slot))
    return z


def render(meshes, obj_ids, poses44, K, rows, cols):
    """pgp_render_depth: (depth rows x cols fp32, 0 = nothing; slot rows x cols int32, -1 = nothing)."""
    z = zbuffer(meshes, obj_ids, poses44, K, rows, cols)
    hit = z != EMPTY
    depth = np.where(hit, (z >> np.uint64(32)).astype(np.uint32), 0).astype(np.uint32).view(np.float32)
    slot = np.where(hit, (z & np.uint64(0xFFFFFFFF)).astype(np.int64), -1).astype(np.int32)
    return depth.reshape(rows, cols), slot.reshape(rows, cols)


def counts_from_images(depth, slot, n_slots, depth_raw, class_mask, class_ids, tau) -> np.ndarray:
    """7. (n_slots, 5) int32 {rendered, agree, in_front, behind, on_segment} from one state's depth and slot images."""
    out = np.zeros((n_slots, 5), np.int64)
    s = slot.reshape(-1)
    hit = s >= 0
    r = depth.reshape(-1)[hit]
    sl = s[hit]
    o = decode_depth(np.asarray(depth_raw).reshape(-1))[hit]
    valid = (o.astype(np.float64) > 0.1) & (o.astype(np.float64) < 2.0)
    tau = F32(tau)
    with np.errstate(over="ignore", invalid="ignore"):
        agree = valid & (np.abs(r - o) <= tau)
        in_front = valid & ~agree & ((o - r) > tau)
        behind = valid & ~agree & ~in_front & ((r - o) > tau)
    np.add.at(out[:, 0], sl, 1)
    np.add.at(out[:, 1], sl, agree.astype(np.int64))
    np.add.at(out[:, 2], sl, in_front.astype(np.int64))
    np.add.at(out[:, 3], sl, behind.astype(np.int64))
    if class_mask is not None:
        lab = np.asarray(class_mask).reshape(-1)[hit].astype(np.int64)
        np.add.at(out[:, 4], sl, (lab == np.asarray(class_ids, np.int64)[sl]).astype(np.int64))
    return out.astype(np.int32)


def depth_cost(meshes, states, K, rows, cols, depth_raw, class_mask, tau) -> np.ndarray:
    """pgp_depth_cost: states = [(obj_ids, poses44), ...]; meshes[obj] = (verts, tri, class_id).  One record per placed object."""
    recs = [np.zeros((0, 5), np.int32)]
    for obj_ids, poses in states:
        if len(obj_ids) == 0:
            continue
        depth, slot = render(meshes, obj_ids, poses, K, rows, cols)
        recs.append(counts_from_images(depth, slot, len(obj_ids), depth_raw, class_mask, [meshes[o][2] for o in obj_ids], tau))
    return np.concatenate(recs)


def class_pixels(depth_raw, class_mask) -> np.ndarray:
    """pgp_set_depth_observation's class_pixels_out: pixels of each label with valid depth."""
    o = decode_depth(np.asarray(depth_raw).reshape(-1)).astype(np.float64)
    valid = (o > 0.1) & (o < 2.0)
    return np.bincount(np.asarray(class_mask).reshape(-1)[valid].astype(np.int64), minlength=256).astype(np.int64)


def coverage(mesh, pose44, K, rows, cols) -> np.ndarray:
    """How many triangles of one mesh cover each sample (no z-test): the watertightness check."""
    cov = np.zeros(rows * cols, np.int64)
    for p, _, _ in _mesh_fragments(mesh, pose44, K, rows, cols):
        np.add.at(cov, p, 1)
    return cov.reshape(rows, cols)
