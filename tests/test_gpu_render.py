"""K8, the rendered-depth cost (include/pgp.h): pgp_set_mesh, pgp_set_depth_observation, pgp_render_depth, pgp_depth_cost.

RESTATED, PARITY UNPINNED: the reference's OpenGL renderer and UCTState::computeCost are not available.  On the CPU the numpy
restatement oracle/render_port.py is checked against independent facts (watertight coverage, exact depth of a fronto-parallel
quad, float64 ray casting of a box).  On the GPU every image and count is compared bit for bit with that restatement."""
import os

import numpy as np
import pytest

from oracle import render_port as rp
from physimglobalpose_b200 import synth

G = os.path.join(os.path.dirname(__file__), "golden")
C1_CLASSES = {"kleenex_tissue_box": 8, "expo_dry_erase_board_eraser": 2, "folgers_classic_roast_coffee": 3}


def kmat(fx, fy, cx, cy):
    return np.array([[fx, 0, cx], [0, fy, cy], [0, 0, 1]], np.float32)


def pose(R=None, t=(0.0, 0.0, 0.0)):
    P = np.eye(4)
    if R is not None:
        P[:3, :3] = R
    P[:3, 3] = t
    return P


def encode_depth(dec_u16):
    """Inverse of K7's decode: the raw value whose ((d << 13) | (d >> 3)) is dec_u16."""
    d = np.asarray(dec_u16, np.uint32) & 0xFFFF
    return (((d << 3) | (d >> 13)) & 0xFFFF).astype(np.uint16)


def c1_frame():
    g = np.load(os.path.join(G, "c1_test_scene.npz"))
    raw = np.repeat(g["depth_raw_rle"][0], g["depth_raw_rle"][1]).astype(np.uint16).reshape(480, 640)
    mask = np.repeat(g["mask_all_rle"][0], g["mask_all_rle"][1]).astype(np.uint8).reshape(480, 640)
    return g, raw, mask


# ------------------------------------------------------------------------------------------------ CPU: the restatement
PIX = kmat(100.0, 100.0, 0.0, 0.0)          # pixel (c, r) <-> model point (c / 100, r / 100, 0) at Z = 1


def _pixel_mesh(pts, tris):
    """Vertices given in pixel units on the plane Z = 1 (pose: translation (0, 0, 1)); they snap exactly onto samples."""
    v = np.zeros((len(pts), 3), np.float32)
    v[:, :2] = (np.asarray(pts, np.float64) / 100.0).astype(np.float32)
    return v, np.asarray(tris, np.int32)


def _strict_inside(poly, rows, cols):
    """Samples strictly inside a convex polygon given in pixel units (either orientation), exact in integers."""
    c, r = np.meshgrid(np.arange(cols), np.arange(rows))
    poly = np.asarray(poly, np.int64)
    s = []
    for i in range(len(poly)):
        a, b = poly[i], poly[(i + 1) % len(poly)]
        s.append((b[0] - a[0]) * (r - a[1]) - (b[1] - a[1]) * (c - a[0]))
    s = np.stack(s)
    return np.all(s > 0, 0) | np.all(s < 0, 0), np.all(s >= 0, 0) | np.all(s <= 0, 0)


def _check_watertight(pts, tris, poly, rows=48, cols=64):
    v, t = _pixel_mesh(pts, tris)
    cov = rp.coverage((v, t), pose(t=(0, 0, 1)), PIX, rows, cols)
    inside, closed = _strict_inside(poly, rows, cols)
    assert np.all(cov[inside] == 1), np.argwhere(inside & (cov != 1))[:5]
    assert cov.max() <= 1
    assert np.all(cov[~closed] == 0)


def _wind(tris, rng):
    """Random windings: the rasterizer has no back-face culling."""
    tris = np.array(tris)
    flip = rng.random(len(tris)) < 0.5
    tris[flip] = tris[flip][:, [0, 2, 1]]
    return tris


def test_watertight_grid():
    rng = np.random.default_rng(1)
    xs, ys = np.arange(2, 43, 4), np.arange(3, 34, 4)
    pts = [(x, y) for y in ys for x in xs]
    nx = len(xs)
    tris = []
    for j in range(len(ys) - 1):
        for i in range(nx - 1):
            a, b, c, d = j * nx + i, j * nx + i + 1, (j + 1) * nx + i + 1, (j + 1) * nx + i
            tris += [(a, b, c), (a, c, d)] if (i + j) % 2 == 0 else [(a, b, d), (b, c, d)]
    _check_watertight(pts, _wind(tris, rng), [(2, 3), (42, 3), (42, 31), (2, 31)])


def test_watertight_fan():
    rng = np.random.default_rng(2)
    ring = [(x, 12) for x in range(22, 38, 4)] + [(38, y) for y in range(12, 28, 4)] + \
           [(x, 28) for x in range(38, 22, -4)] + [(22, y) for y in range(28, 12, -4)]
    pts = [(30, 20)] + ring
    tris = [(0, 1 + i, 1 + (i + 1) % len(ring)) for i in range(len(ring))]
    _check_watertight(pts, _wind(tris, rng), [(22, 12), (38, 12), (38, 28), (22, 28)])


@pytest.mark.parametrize("d", [(8, 0), (8, 8), (0, 8), (-8, 8), (-8, 0), (-8, -8), (0, -8), (8, -8)])
def test_watertight_shared_edge(d):
    rng = np.random.default_rng(3)
    P = np.array([30, 20])
    Q = P + d
    M = P + np.array(d) // 2
    perp = np.array([-d[1], d[0]]) // 2
    pts = [tuple(P), tuple(Q), tuple(M + perp), tuple(M - perp)]
    _check_watertight(pts, _wind([(0, 1, 2), (1, 0, 3)], rng), [pts[0], pts[2], pts[1], pts[3]])


def test_fronto_parallel_quad_depth_is_exact():
    g = np.load(os.path.join(G, "c1_test_scene.npz"))
    for z0 in (0.4, 0.7317, 1.93):
        v = np.array([[-0.1, -0.08, 0], [0.12, -0.08, 0], [0.12, 0.09, 0], [-0.1, 0.09, 0]], np.float32)
        t = np.array([[0, 1, 2], [0, 3, 2]], np.int32)
        depth, slot = rp.render({0: (v, t, -1)}, [0], [pose(t=(0.01, -0.02, z0))], g["K"], 480, 640)
        hit = slot >= 0
        assert hit.sum() > 2000
        assert np.all(depth[hit] == np.float32(z0)) and np.all(depth[~hit] == 0)


def test_box_depth_matches_ray_casting():
    """A box mesh at the synthetic generator's GT pose, away from silhouette pixels, against float64 ray casting: (1) to 1e-6 m
    against the plane of the covering triangle through its SNAPPED vertices (back-projected at their depths), i.e. perspective-
    correct interpolation checked by an independent formula; (2) against the exact box (slab intersection) within what the 1/256 px
    snap can move a surface: |depth gradient| x 2^-9 px per axis."""
    g = np.load(os.path.join(G, "c1_test_scene.npz"))
    K = g["K"].astype(np.float64)
    fx, fy, cx, cy = K[0, 0], K[1, 1], K[0, 2], K[1, 2]
    v, t = synth.box_mesh(synth.BOX, 4)
    P = pose(synth.rot_axis_angle(synth.GT_AXIS, synth.GT_ANGLE), synth.GT_T)
    depth, slot = rp.render({0: (v, t, -1)}, [0], [P], g["K"], 480, 640)
    hit = slot >= 0
    inner = hit.copy()                                  # away from the silhouette: all 8 neighbours covered too
    for dr in (-1, 0, 1):
        for dc in (-1, 0, 1):
            inner &= np.roll(np.roll(hit, dr, 0), dc, 1)
    # (1) the front triangle of each pixel, its snapped vertices back-projected, the ray / plane intersection
    X, Y, Z = rp.transform(rp.pose_f32(P), v)
    ix, iy, ok = rp.project(g["K"], X, Y, Z)
    a, b, c, *_ = rp.setup(ix, iy, ok, Z, t, 480, 640)
    front = np.full(480 * 640, -1)
    best = np.full(480 * 640, np.inf, np.float32)
    for pix, d, tri in rp.fragments((ix, iy, ok), Z, t, 480, 640):
        order = np.lexsort((tri, d))                    # nearest first; the z-test keeps the smaller depth
        pix, d, tri = pix[order], d[order], tri[order]
        u, first = np.unique(pix, return_index=True)
        closer = d[first] < best[u]
        best[u[closer]], front[u[closer]] = d[first][closer], tri[first][closer]
    r, col = np.nonzero(inner)
    assert len(r) > 2000
    k = front[r * 640 + col]
    Zd = Z.astype(np.float64)
    def back(i):                                        # snapped screen position at the vertex depth -> camera frame
        return np.stack([(ix[i] / 256.0 - cx) * Zd[i] / fx, (iy[i] / 256.0 - cy) * Zd[i] / fy, Zd[i]], 1)
    A, B, Cc = back(a[k]), back(b[k]), back(c[k])
    n = np.cross(B - A, Cc - A)
    ray = np.stack([(col - cx) / fx, (r - cy) / fy, np.ones(len(r))], 1)
    t_plane = np.einsum("ij,ij->i", n, A) / np.einsum("ij,ij->i", n, ray)
    err1 = np.abs(depth[r, col].astype(np.float64) - t_plane)
    assert err1.max() <= 1e-6, err1.max()
    # (2) the exact box
    R, tt = P[:3, :3], P[:3, 3]
    half = np.asarray(synth.BOX) / 2

    def cast(cc, rr):
        d = np.stack([(cc - cx) / fx, (rr - cy) / fy, np.ones(len(cc))], 1)
        o_m, d_m = R.T @ (-tt), d @ R
        with np.errstate(divide="ignore"):
            t1, t2 = (-half - o_m) / d_m, (half - o_m) / d_m
        return np.minimum(t1, t2).max(1)
    exact = cast(col, r)
    gx = np.abs(cast(col + 0.5, r) - cast(col - 0.5, r))
    gy = np.abs(cast(col, r + 0.5) - cast(col, r - 0.5))
    err2 = np.abs(depth[r, col].astype(np.float64) - exact)
    assert np.all(err2 <= 1.5 * (gx + gy) / 512 + 1e-6), (err2 - 1.5 * (gx + gy) / 512).max()
    assert np.median(err2) < 1e-6


def test_class_pixels_restatement():
    _, raw, mask = c1_frame()
    h = rp.class_pixels(raw, mask)
    o = rp.decode_depth(raw).astype(np.float64)
    for cls in C1_CLASSES.values():
        assert h[cls] == int(((mask == cls) & (o > 0.1) & (o < 2.0)).sum()) > 0


# ------------------------------------------------------------------------------------------------ GPU: bit for bit
def _set_meshes(engine, meshes):
    for obj, (v, t, cls) in meshes.items():
        engine.set_mesh(obj, v, t, cls)


def _check_state(engine, meshes, obj_ids, poses, K, raw, mask, tau):
    rows, cols = raw.shape
    depth, slot = engine.render_depth(obj_ids, poses)
    want_d, want_s = rp.render(meshes, obj_ids, poses, K, rows, cols)
    assert np.array_equal(depth.view(np.uint32), want_d.view(np.uint32)), np.argwhere(depth.view(np.uint32) != want_d.view(np.uint32))[:5]
    assert np.array_equal(slot, want_s)
    got = engine.depth_cost([(obj_ids, poses)], tau)
    want = rp.counts_from_images(want_d, want_s, len(obj_ids), raw, mask, [meshes[o][2] for o in obj_ids], tau)
    assert np.array_equal(got, want), (got, want)
    # the counts taken on the host from the device's own images
    assert np.array_equal(got, rp.counts_from_images(depth, slot, len(obj_ids), raw, mask, [meshes[o][2] for o in obj_ids], tau))
    return depth, slot, got


def _random_obs(rng, rows, cols, lo=0.3, hi=1.2):
    dec = rng.integers(int(lo * 10000), int(hi * 10000), (rows, cols))
    dec[rng.random((rows, cols)) < 0.1] = 0
    return encode_depth(dec), rng.integers(0, 4, (rows, cols)).astype(np.uint8)


def _random_triangles(rng, n, K, rows, cols, spread):
    """n independent triangles with vertices around random screen points (sizes from sub-pixel to `spread` px), depth 0.3-1.5 m."""
    fx, fy, cx, cy = K[0, 0], K[1, 1], K[0, 2], K[1, 2]
    centre = np.stack([rng.uniform(-0.2 * cols, 1.2 * cols, n), rng.uniform(-0.2 * rows, 1.2 * rows, n)], 1)
    size = np.exp(rng.uniform(np.log(0.05), np.log(spread), n))
    px = centre[:, None, :] + rng.normal(size=(n, 3, 2)) * size[:, None, None]
    Z = rng.uniform(0.3, 1.5, (n, 3))
    X = (px[..., 0] - cx) * Z / fx
    Y = (px[..., 1] - cy) * Z / fy
    v = np.stack([X, Y, Z], -1).reshape(-1, 3).astype(np.float32)
    return v, np.arange(3 * n, dtype=np.int32).reshape(-1, 3)


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols", [(1, 1), (1, 33), (17, 13), (480, 640), (479, 641)])
def test_random_triangles_every_size(engine, rows, cols):
    rng = np.random.default_rng(rows * 1000 + cols)
    K = kmat(500.0, 510.0, cols / 2 - 0.3, rows / 2 + 0.2)
    raw, mask = _random_obs(rng, rows, cols)
    engine.set_depth_observation(raw, mask, K)
    meshes = {0: _random_triangles(rng, 3000, K, rows, cols, 40.0) + (1,), 1: _random_triangles(rng, 200, K, rows, cols, 2000.0) + (2,)}
    _set_meshes(engine, meshes)
    _check_state(engine, meshes, [0, 1], [pose(), pose(t=(0.001, 0, 0.05))], K, raw, mask, 0.01)


@pytest.mark.gpu
def test_watertight_meshes_on_device(engine):
    rows, cols = 48, 64
    raw = encode_depth(np.full((rows, cols), 10000))
    engine.set_depth_observation(raw, None, PIX)
    rng = np.random.default_rng(4)
    xs, ys = np.arange(2, 43, 4), np.arange(3, 34, 4)
    pts = [(x, y) for y in ys for x in xs]
    nx = len(xs)
    tris = []
    for j in range(len(ys) - 1):
        for i in range(nx - 1):
            a, b, c, d = j * nx + i, j * nx + i + 1, (j + 1) * nx + i + 1, (j + 1) * nx + i
            tris += [(a, b, c), (a, c, d)] if (i + j) % 2 == 0 else [(a, b, d), (b, c, d)]
    v, t = _pixel_mesh(pts, _wind(tris, rng))
    meshes = {0: (v, t, -1)}
    _set_meshes(engine, meshes)
    depth, slot, counts = _check_state(engine, meshes, [0], [pose(t=(0, 0, 1))], PIX, raw, None, 0.0)
    assert counts[0, 0] == (slot >= 0).sum() > 1000 and counts[0, 1] == counts[0, 0]
    for d in [(8, 0), (8, 8), (0, 8), (-8, 8), (-8, 0), (-8, -8), (0, -8), (8, -8)]:
        P = np.array([30, 20])
        M, perp = P + np.array(d) // 2, np.array([-d[1], d[0]]) // 2
        v, t = _pixel_mesh([tuple(P), tuple(P + d), tuple(M + perp), tuple(M - perp)], _wind([(0, 1, 2), (1, 0, 3)], rng))
        meshes = {0: (v, t, -1)}
        _set_meshes(engine, meshes)
        _check_state(engine, meshes, [0], [pose(t=(0, 0, 1))], PIX, raw, None, 0.0)


@pytest.mark.gpu
def test_offscreen_near_plane_and_guard_band(engine):
    rows, cols = 64, 80
    K = kmat(100.0, 100.0, 40.0, 32.0)
    rng = np.random.default_rng(5)
    raw, mask = _random_obs(rng, rows, cols)
    engine.set_depth_observation(raw, mask, K)
    big = 5000.0                                                          # 5e5 px from the centre: inside the 2^20 px guard band
    v = np.array([
        [-0.5, -0.4, 0], [0.5, -0.4, 0], [0.0, 0.5, 0],                   # partly off-screen at Z = 1
        [5, 5, 0], [6, 5, 0], [5, 6, 0],                                  # fully off-screen
        [-big, -big, 0], [big, -big, 0], [0, big, 0],                     # larger than the image, inside the guard band
        [-0.1, -0.1, -0.9], [0.1, -0.1, -0.9], [0, 0.1, -0.9],             # Z = fl(1 - 0.9f), just above 0.1: kept
        [-0.1, -0.1, 0], [0.1, -0.1, 0], [0, 0.1, 0],                     # at the pose's Z (the near-plane slide below)
        [-2e4, -0.1, 0], [0.1, -0.1, 0], [0, 0.1, 0],                     # |sx| > 2^20 px: dropped
        [0, 0, 0], [0.1, 0, 0], [0.2, 0, 0],                              # zero area
        [0, 0, 0], [0, 0, 0], [0.1, 0.1, 0],                              # repeated vertex
    ], np.float32)
    t = np.arange(len(v), dtype=np.int32).reshape(-1, 3)
    t = np.concatenate([t, [[21, 21, 23], [18, 18, 18]]]).astype(np.int32)   # repeated indices
    meshes = {0: (v, t, 1)}
    _set_meshes(engine, meshes)
    above = float(np.nextafter(np.float32(0.1), np.float32(1)))
    _check_state(engine, meshes, [0], [pose(t=(0, 0, 1))], K, raw, mask, 0.02)
    # the same mesh slid towards the camera: the near plane at 0.1 exactly (dropped) and one float above it (kept)
    for z in (0.1, above, 0.0999):
        d, s, _ = _check_state(engine, meshes, [0], [pose(t=(0, 0, z))], K, raw, mask, 0.02)
    big_only = {0: (v[6:9], np.array([[0, 1, 2]], np.int32), 1)}
    _set_meshes(engine, big_only)
    d, s, _ = _check_state(engine, big_only, [0], [pose(t=(0, 0, 1))], K, raw, mask, 0.02)
    assert np.all(s == 0)                                                 # a triangle larger than the image covers it all


@pytest.mark.gpu
def test_same_pose_ties_go_to_the_smaller_slot(engine):
    g, raw, mask = c1_frame()
    engine.set_depth_observation(raw, mask, g["K"])
    v, t = synth.box_mesh((0.1, 0.1, 0.1), 2)
    meshes = {3: (v, t, 8), 5: (v.copy(), t[:, [0, 2, 1]].copy(), 2)}
    _set_meshes(engine, meshes)
    P = pose(synth.rot_axis_angle((1, 2, 3), 0.4), (0.0, 0.02, 0.5))
    for ids in ([3, 5], [5, 3]):
        d, s, counts = _check_state(engine, meshes, ids, [P, P], g["K"], raw, mask, 0.005)
        assert counts[0, 0] > 0 and counts[1, 0] == 0 and np.all(s[s >= 0] == 0)


@pytest.mark.gpu
def test_mesh_sizes_and_refill(engine):
    g, raw, mask = c1_frame()
    engine.set_depth_observation(raw, mask, g["K"])
    one = (np.array([[-0.05, -0.05, 0], [0.05, -0.05, 0], [0, 0.05, 0]], np.float32), np.array([[0, 1, 2]], np.int32), 8)
    box = synth.box_mesh((0.08, 0.1, 0.12), 1) + (2,)
    ell = synth.ellipsoid_mesh((0.06, 0.05, 0.08), 160, 320) + (3,)
    assert len(one[1]) == 1 and len(box[1]) == 12 and 95_000 < len(ell[1]) < 105_000
    meshes = {0: one, 1: box, 2: ell}
    _set_meshes(engine, meshes)
    R = synth.rot_axis_angle((0.2, 1, 0.4), 0.9)
    poses = [pose(R, (-0.1, 0.0, 0.45)), pose(R.T, (0.0, 0.03, 0.5)), pose(R, (0.05, -0.02, 0.55))]
    _check_state(engine, meshes, [0, 1, 2], poses, g["K"], raw, mask, 0.01)
    meshes[1] = synth.ellipsoid_mesh((0.03, 0.04, 0.05), 8, 16) + (2,)      # slot 1 refilled with a different mesh
    engine.set_mesh(1, *meshes[1])
    _check_state(engine, meshes, [0, 1, 2], poses, g["K"], raw, mask, 0.01)


def _table_states(g, rng, n_states, max_objs):
    """Box meshes placed around the test scene's three segments (on the table), jittered."""
    cents = [g[f"{n}_seg_xyz"].astype(np.float64).mean(0) for n in g["names"]]
    states = []
    for _ in range(n_states):
        k = int(rng.integers(0, max_objs + 1))
        ids = rng.integers(0, 3, k)
        poses = [pose(synth.rot_axis_angle(rng.normal(size=3), rng.uniform(0, 0.5)), cents[i] + rng.normal(scale=0.02, size=3)) for i in ids]
        states.append((ids.astype(np.int32), np.array(poses).reshape(-1, 4, 4)))
    return states


def _table_meshes(g):
    return {i: synth.box_mesh(d, 2) + (C1_CLASSES[str(n)],) for i, (n, d) in enumerate(zip(g["names"], [(0.12, 0.1, 0.24), (0.15, 0.05, 0.035), (0.1, 0.1, 0.15)]))}


@pytest.mark.gpu
def test_test_scene_observation(engine):
    g, raw, mask = c1_frame()
    hist = engine.set_depth_observation(raw, mask, g["K"])
    assert np.array_equal(hist, rp.class_pixels(raw, mask))
    meshes = _table_meshes(g)
    _set_meshes(engine, meshes)
    rng = np.random.default_rng(6)
    for ids, poses in _table_states(g, rng, 4, 3):
        _check_state(engine, meshes, list(ids), poses, g["K"], raw, mask, 0.01)
    # the three objects near their segments agree with the observation on most of their pixels and lie on their labels
    ids, poses = [0, 1, 2], [pose(t=g[f"{n}_seg_xyz"].astype(np.float64).mean(0) + [0, 0, 0.03]) for n in g["names"]]
    _, _, counts = _check_state(engine, meshes, ids, poses, g["K"], raw, mask, 0.02)
    assert np.all(counts[:, 4] > 0.3 * counts[:, 0])
    # no mask: on_segment stays 0
    assert np.all(engine.set_depth_observation(raw, None, g["K"]) == 0)
    _, _, counts = _check_state(engine, meshes, ids, poses, g["K"], raw, None, 0.02)
    assert np.all(counts[:, 4] == 0)


@pytest.mark.gpu
def test_tau_and_validity_edges(engine):
    rows, cols = 24, 32
    K = kmat(60.0, 60.0, 16.0, 12.0)
    v = np.array([[-1, -1, 0], [1, -1, 0], [1, 1, 0], [-1, 1, 0]], np.float32)
    t = np.array([[0, 1, 2], [0, 2, 3]], np.int32)
    meshes = {0: (v, t, 7), 1: (v, t, -1)}
    rng = np.random.default_rng(7)
    dec = rng.integers(4000, 6000, (rows, cols))
    dec[0, :8] = [0, 1000, 20000, 19999, 1001, 999, 65535, 5000]         # 0, 0.1, 2.0 and their neighbours
    raw = encode_depth(dec)
    mask = np.where(rng.random((rows, cols)) < 0.5, 7, 3).astype(np.uint8)
    engine.set_depth_observation(raw, mask, K)
    _set_meshes(engine, meshes)
    z = 0.5
    o = rp.decode_depth(raw)
    r = np.float32(z)
    diff = np.abs(r - o[o > 0])
    for tau in (0.0, float(np.sort(diff)[len(diff) // 2]), float(np.nextafter(np.sort(diff)[len(diff) // 2], np.float32(0))), 0.05):
        for ids in ([0], [1]):
            _, _, counts = _check_state(engine, meshes, ids, [pose(t=(0, 0, z))], K, raw, mask, tau)
            assert counts[0, 0] == rows * cols
    # one pixel with |r - o| exactly tau counts as agree; o - r one float above tau as in_front
    dec2 = np.full((rows, cols), 5000)
    dec2[3, 4] = 5100
    raw2 = encode_depth(dec2)
    engine.set_depth_observation(raw2, mask, K)
    tau = float(np.float32(np.float32(0.51) - np.float32(0.5)))
    _, _, c_eq = _check_state(engine, meshes, [0], [pose(t=(0, 0, 0.5))], K, raw2, mask, tau)
    _, _, c_lt = _check_state(engine, meshes, [0], [pose(t=(0, 0, 0.5))], K, raw2, mask, float(np.nextafter(np.float32(tau), np.float32(0))))
    assert c_eq[0, 1] == rows * cols and c_lt[0, 1] == rows * cols - 1 and c_lt[0, 2] == 1


@pytest.mark.gpu
@pytest.mark.parametrize("n_states,max_objs", [(0, 0), (1, 3), (25, 64), (4000, 3)])
def test_batches_equal_states_alone(engine, n_states, max_objs):
    g, raw, mask = c1_frame()
    engine.set_depth_observation(raw, mask, g["K"])
    meshes = _table_meshes(g)
    _set_meshes(engine, meshes)
    rng = np.random.default_rng(n_states)
    states = _table_states(g, rng, n_states, max_objs)
    if n_states == 4000:                                  # more states than one chunk holds (4M (state, tile) bins at 640 x 480)
        states[0] = (np.zeros(0, np.int32), np.zeros((0, 4, 4)))
    got = engine.depth_cost(states, 0.01)
    assert got.shape == (sum(len(i) for i, _ in states), 5)
    off = 0
    for k, (ids, poses) in enumerate(states):
        alone = engine.depth_cost([(ids, poses)], 0.01)
        assert np.array_equal(got[off:off + len(ids)], alone), k
        if n_states <= 25 and len(ids):
            want = rp.depth_cost(meshes, [(ids, poses)], g["K"], 480, 640, raw, mask, 0.01)
            assert np.array_equal(alone, want), k
        off += len(ids)


@pytest.mark.gpu
def test_refusals_leave_outputs_untouched(engine):
    from physimglobalpose_b200 import _lib
    lib, ctx = _lib.load(), engine._ctx
    g, raw, mask = c1_frame()
    K = g["K"].astype(np.float32).reshape(9)
    v, t = synth.box_mesh((0.1, 0.1, 0.1), 1)
    p = lambda a: a.ctypes.data                            # noqa: E731
    # a depth call before any observation: a fresh context
    from physimglobalpose_b200.engine import PoseEngine
    fresh = PoseEngine(0)
    assert lib.pgp_set_mesh(fresh._ctx, 0, p(v), len(v), p(t), len(t), -1) == 0
    offs = np.array([0, 1], np.int64)
    ids = np.zeros(1, np.int32)
    P = np.eye(4).reshape(1, 16) + np.array([0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0.5, 0, 0, 0, 0])
    out = np.full((1, 5), -7, np.int32)
    depth = np.full((480, 640), -3.0, np.float32)
    assert lib.pgp_depth_cost(fresh._ctx, p(offs), 1, p(ids), p(P), 0.01, p(out)) == -1 and np.all(out == -7)
    assert lib.pgp_render_depth(fresh._ctx, p(ids), p(P), 1, p(depth), None) == -1 and np.all(depth == -3)
    fresh.close()
    # pgp_set_mesh
    bad_v = v.copy()
    bad_v[2, 1] = np.nan
    bad_t = t.copy()
    bad_t[5, 2] = len(v)
    neg_t = t.copy()
    neg_t[0, 0] = -1
    assert lib.pgp_set_mesh(ctx, 9, p(bad_v), len(v), p(t), len(t), -1) == -1
    assert lib.pgp_set_mesh(ctx, 9, p(v), len(v), p(bad_t), len(t), -1) == -1
    assert lib.pgp_set_mesh(ctx, 9, p(v), len(v), p(neg_t), len(t), -1) == -1
    assert lib.pgp_set_mesh(ctx, 9, p(v), 2, p(t), len(t), -1) == -1
    assert lib.pgp_set_mesh(ctx, 9, p(v), len(v), p(t), 0, -1) == -1
    assert lib.pgp_set_mesh(ctx, 64, p(v), len(v), p(t), len(t), -1) == -1
    # pgp_set_depth_observation
    hist = np.full(256, -5, np.int64)
    for KK in (np.where(np.arange(9) == 2, np.inf, K), np.where(np.arange(9) == 7, np.nan, K), np.where(np.arange(9) == 0, 0, K),
               np.where(np.arange(9) == 4, -1, K)):
        KK = KK.astype(np.float32)
        assert lib.pgp_set_depth_observation(ctx, p(raw), p(mask), 480, 640, p(KK), p(hist)) == -1 and np.all(hist == -5)
    assert lib.pgp_set_depth_observation(ctx, p(raw), p(mask), 0, 640, p(K), p(hist)) == -1
    assert lib.pgp_set_depth_observation(ctx, p(raw), p(mask), 480, 0, p(K), p(hist)) == -1
    assert lib.pgp_set_depth_observation(ctx, p(raw), p(mask), 480, 640, p(K), p(hist)) == 0
    assert lib.pgp_set_mesh(ctx, 0, p(v), len(v), p(t), len(t), 8) == 0
    # pgp_depth_cost / pgp_render_depth
    out = np.full((70, 5), -7, np.int32)
    depth = np.full((480, 640), -3.0, np.float32)
    P70 = np.tile(P, (70, 1))
    ids70 = np.zeros(70, np.int32)

    def refused(offs, ids=ids70, P=P70, tau=0.01, code=-1):
        offs = np.asarray(offs, np.int64)
        assert lib.pgp_depth_cost(ctx, p(offs), len(offs) - 1, p(ids), p(P), tau, p(out)) == code
        assert np.all(out == -7)
    refused([0, 1], tau=-0.001)
    refused([0, 1], tau=float("nan"))
    refused([0, 1], tau=float("inf"))
    refused([1, 2])                                        # not from 0
    refused([0, 3, 2])                                     # decreasing
    refused([0, 65])                                       # more than PGP_MAX_OBJECTS objects in one state
    nanP = P70.copy()
    nanP[1, 3] = np.nan
    refused([0, 2], P=nanP)
    refused([0, 1], ids=np.full(70, 64, np.int32))         # object id out of range
    refused([0, 1], ids=np.full(70, 40, np.int32), code=-4)   # no mesh in slot 40: PGP_E_NO_MODEL
    assert lib.pgp_render_depth(ctx, p(ids70), p(nanP[1:]), 1, p(depth), None) == -1 and np.all(depth == -3)
    assert lib.pgp_render_depth(ctx, p(ids70), p(P70), 65, p(depth), None) == -1 and np.all(depth == -3)
    assert lib.pgp_render_depth(ctx, p(np.full(1, 40, np.int32)), p(P70), 1, p(depth), None) == -4 and np.all(depth == -3)
    # valid edge cases: no states, empty states
    assert lib.pgp_depth_cost(ctx, None, 0, None, None, 0.01, None) == 0
    assert lib.pgp_depth_cost(ctx, p(np.zeros(4, np.int64)), 3, None, None, 0.01, None) == 0
    assert lib.pgp_render_depth(ctx, None, None, 0, p(depth), None) == 0 and np.all(depth == 0)
