"""K7, the segment preparation (pgp_prepare_segment, k7_segment.cu), against its float64 restatement oracle/segment_port.py at the
edges: every raw depth value, frame shapes and intrinsics, voxel-boundary coordinates, leaf / radius / min_neighbors sweeps on
synthetic surfaces in both modes, neighbours at exactly the radius, line-like segments, degenerate inputs, scratch history and the
refusals.  Frames are ray-cast per pixel, quantised to the 0.1 mm of the depth format and encoded back to raw.

What "agree" means, per output point (the reference's neighbourhood decides how well the point is determined):
  - the kept set, the pixel count and, with k7_mls = 0, every position: identical (positions bit for bit);
  - a normal whose PCA plane is determined (eigen-gap (l1 - l0) / l2 >= 1e-9 of the neighbourhood covariance): equal to fp32
    rounding, |dn|_inf <= 1.2e-7, plus the eigenvector's own float64 sensitivity 1e-13 / gap and, when the polynomial was solved,
    1e-14 x the condition number of its (diagonally scaled) 6x6 system;
  - a neighbourhood on one line (l1 <= 1e-10 l2): its normal is any direction across the line, so only |n . line| <= 1e-6;
  - a normal perpendicular to its viewing ray (|n . p| <= 1e-6 |p|, e.g. a strip in a plane through the camera, or the crease of
    a symmetric ridge) has no side towards the camera, and either sign is the flip's rounding: compared up to sign;
  - k7_mls = 1: positions to 1e-6 m wherever the 6x6 system is decided the same on both sides -- not solved (fewer than 6
    neighbours, or a Cholesky pivot at or below 1e-12 of its diagonal, far under the 1e-10 that refuses it) or well conditioned
    (smallest relative pivot >= 1e-8, scaled condition number <= 1e8).  Between those (thin strips, where the depth's 0.1 mm
    steps are all that keeps the neighbours off one or two lines), float64 does not determine the polynomial step, nor whether it
    is taken: positions to 1e-6 m plus twice the reference's own step off the PCA plane, normals unit length only.
GPU tests are marked; the reference-only tests run anywhere."""
import contextlib
import ctypes as C

import numpy as np
import pytest

from oracle import segment_port as sp

gpu = pytest.mark.gpu
PGP_E_INVALID, PGP_E_CAPACITY = -1, -8
COND_MAX, PIVOT_SOLVED, PIVOT_REFUSED = 1e8, 1e-8, 1e-12


def encode_depth(dec_u16):
    """Inverse of K7's decode: the raw value whose ((d << 13) | (d >> 3)) is dec_u16."""
    d = np.asarray(dec_u16, np.uint32) & 0xFFFF
    return (((d << 3) | (d >> 13)) & 0xFFFF).astype(np.uint16)


def kmat(fx, fy, cx, cy):
    return np.array([[fx, 0, cx], [0, fy, cy], [0, 0, 1]], np.float32)


def raycast(kind, rows, cols, K, noise=0.0, seed=0):
    """Decoded depth (units of 0.1 mm) of a surface seen through pixel rays (a, b, 1); 0 where the ray misses or leaves (0, 6.5 m)."""
    fx, fy, cx, cy = (float(K[0, 0]), float(K[1, 1]), float(K[0, 2]), float(K[1, 2]))
    u, v = np.mgrid[0:rows, 0:cols].astype(np.float64)
    a, b = (v - cx) / fx, (u - cy) / fy
    with np.errstate(divide="ignore", invalid="ignore"):
        if kind == "plane":                      # through (0, 0, 0.7), normal (0.3, -0.2, -1)
            n = np.array([0.3, -0.2, -1.0])
            z = (n[2] * 0.7) / (n[0] * a + n[1] * b + n[2])
        elif kind == "sphere":                   # cap of a 0.35 m sphere centred at (0.02, -0.01, 1.0), the near side
            c = np.array([0.02, -0.01, 1.0])
            dd = a * a + b * b + 1.0
            dc = a * c[0] + b * c[1] + c[2]
            disc = dc * dc - dd * (c @ c - 0.35 ** 2)
            z = np.where(disc >= 0, (dc - np.sqrt(np.maximum(disc, 0))) / dd, np.nan)
        elif kind == "corner":                   # convex box corner at (0.01, -0.02, 0.6) pointing at the camera: max of 3 planes
            p0 = np.array([0.01, -0.02, 0.6])
            zs = []
            for n in ([0.8, 0.5, -1.0], [-0.8, 0.5, -1.0], [0.0, -0.9, -1.0]):
                n = np.asarray(n)
                zs.append((n @ p0) / (n[0] * a + n[1] * b + n[2]))
            z = np.max(zs, axis=0)
        elif kind == "ridge":                    # the V ridge z = z0 + 3 |x|: z = z0 / (1 - 3 |a|)
            den = 1.0 - 3.0 * np.abs(a)
            z = np.where(den > 0, 0.5 / den, np.nan)
        else:
            raise ValueError(kind)
    if noise:
        z = z + np.random.default_rng(seed).normal(0.0, noise, z.shape)
    ok = np.isfinite(z) & (z > 0) & (z < 6.5)
    return np.where(ok, np.round(np.where(ok, z, 0) * 10000.0), 0).astype(np.uint16)


@contextlib.contextmanager
def mls_mode(engine, mls):
    engine.set_option("k7_mls", int(mls))
    try:
        yield
    finally:
        engine.set_option("k7_mls", 1)


# ------------------------------------------------------------------------------------------------ the reference, with its diagnostics
def reference(raw, mask, cls, K, leaf, nr, orr, mn, mls):
    """oracle/segment_port.py's prepare_segment, step by step so that every output row keeps its centroid index."""
    dec = sp.decode_depth(raw)
    pts = sp.backproject(dec, mask, cls, K)
    if len(pts) == 0:
        z = np.zeros((0, 3), np.float32)
        return dict(xyz=z, nrm=z, n_raw=0, cen=z, idx=np.zeros(0, np.int64))
    cen = sp.voxel_centroids(pts, leaf)
    if mls:
        proj, nrm, valid = sp.mls_project(cen, nr)
        idx = np.flatnonzero(valid)
        idx = idx[sp.radius_outlier_keep(proj[idx], orr, mn)]
        return dict(xyz=proj[idx], nrm=nrm[idx], n_raw=len(pts), cen=cen, idx=idx)
    nrm = sp.pca_normals(cen, nr)
    idx = np.flatnonzero(sp.radius_outlier_keep(cen, orr, mn))
    return dict(xyz=cen[idx], nrm=nrm[idx], n_raw=len(pts), cen=cen, idx=idx)


def diagnostics(cen, i, nb, nr):
    """float64 facts of centroid i's neighbourhood: covariance eigenvalues / the line direction, and for >= 6 neighbours the MLS
    6x6 system as mls_project builds it -- its smallest relative Cholesky pivot and its diagonally scaled condition number."""
    q = cen[nb].astype(np.float64)
    c = cen[i].astype(np.float64)
    mean = q.mean(axis=0)
    w, vec = np.linalg.eigh((q - mean).T @ (q - mean))
    n = vec[:, 0]
    point = c - np.dot(c - mean, n) * n
    out = dict(cnt=len(nb), gap=(w[1] - w[0]) / w[2] if w[2] > 0 else 0.0, line=w[2] > 0 and w[1] <= 1e-10 * w[2], e2=vec[:, 2],
               plane_point=point, pivot=None, cond=None)
    if len(nb) >= 6:
        de = q - point
        r = float(np.float32(nr))
        wgt = np.exp(-np.einsum("ij,ij->i", de, de) / (r * r))
        va = sp._unit_orthogonal(n)
        ua = np.cross(n, va)
        uu, vv = de @ ua, de @ va
        P = np.stack([np.ones_like(uu), vv, vv * vv, uu, uu * vv, uu * uu])
        A = (P * wgt) @ P.T
        if not np.all(np.diag(A) > 0):                                   # a basis function zero at every neighbour: refused
            out["pivot"], out["cond"] = 0.0, np.inf
            return out
        s = 1.0 / np.sqrt(np.diag(A))
        out["cond"] = float(np.linalg.cond(A * s[:, None] * s[None, :]))
        piv, L = [], np.zeros((6, 6))
        for j in range(6):
            d = A[j, j] - L[j, :j] @ L[j, :j]
            piv.append(d / A[j, j])
            if not d > 0:
                break
            L[j, j] = np.sqrt(d)
            L[j + 1:, j] = (A[j + 1:, j] - L[j + 1:, :j] @ L[j, :j]) / L[j, j]
        out["pivot"] = min(piv)
    return out


def compare(got, want, nr, mls, min_tight=0.0):
    """Assert the per-point rules of the module docstring; min_tight: the share of points that must be held to the tight bounds."""
    xyz, nrm, n_raw = got
    assert n_raw == want["n_raw"]
    assert xyz.shape == want["xyz"].shape, (xyz.shape, want["xyz"].shape)
    if len(xyz) == 0:
        return 0
    assert np.all(np.isfinite(xyz)) and np.all(np.isfinite(nrm))
    assert np.all(np.abs(np.linalg.norm(nrm.astype(np.float64), axis=1) - 1) < 1e-6)
    if not mls:
        assert np.array_equal(xyz, want["xyz"])
    cen, idx = want["cen"], want["idx"]
    nbs = sp.neighbours(cen, nr)
    tight, bad = 0, []
    for row, i in enumerate(idx):
        dg = diagnostics(cen, i, nbs[i], nr)
        dp = np.abs(xyz[row].astype(np.float64) - want["xyz"][row]).max()
        wn = want["nrm"][row].astype(np.float64)
        p = want["xyz"][row].astype(np.float64)
        if abs(wn @ p) <= 1e-6 * np.linalg.norm(p):                       # across the viewing ray: no side faces the camera
            wn = wn if nrm[row] @ wn >= 0 else -wn
        dn = np.abs(nrm[row].astype(np.float64) - wn).max()
        solved = mls and dg["pivot"] is not None and dg["pivot"] > PIVOT_REFUSED
        if dg["cnt"] < 3:                                                  # PCA mode only: the normal is -c on both sides
            ok_p, ok_n = True, dn <= 1.2e-7
        elif dg["line"]:
            ok_p = dp <= 1e-6 if mls else True
            ok_n = abs(float(nrm[row] @ dg["e2"])) <= 1e-6
        elif dg["gap"] >= 1e-9 and (not solved or (dg["pivot"] >= PIVOT_SOLVED and dg["cond"] <= COND_MAX)):
            ok_p = dp <= 1e-6
            ok_n = dn <= 1.2e-7 + 1e-13 / dg["gap"] + (1e-14 * dg["cond"] if solved else 0.0)
        elif mls:
            step = np.abs(want["xyz"][row].astype(np.float64) - dg["plane_point"]).max()
            ok_p, ok_n = dp <= 1e-6 + 2 * step, True
            if not ok_p:
                bad.append((row, int(i), dp, dn, dg["cnt"], dg["gap"], dg["pivot"], dg["cond"]))
            continue
        else:
            continue
        tight += 1
        if not (ok_p and ok_n):
            bad.append((row, int(i), dp, dn, dg["cnt"], dg["gap"], dg["pivot"], dg["cond"]))
    assert not bad, f"{len(bad)} points differ (row, centroid, |dp|, |dn|, nb, gap, pivot, cond): {bad[:8]}"
    assert tight >= min_tight * len(idx), (tight, len(idx))
    return tight


def run_both(engine, raw, mask, cls, K, leaf=0.01, nr=0.02, orr=0.03, mn=10, modes=(0, 1), min_tight=0.0):
    for mls in modes:
        with mls_mode(engine, mls):
            got = engine.prepare_segment(raw, mask, cls, K, leaf, nr, orr, mn)
        compare(got, reference(raw, mask, cls, K, leaf, nr, orr, mn, mls), nr, mls, min_tight)


# ------------------------------------------------------------------------------------------------ frames
def tie_frame(n=24):
    """Fronto-parallel plane at 0.5 m, pixel pitch 0.5 / 75 = r / 3 for r = 0.02 (one pixel per 5 mm voxel, so every centroid is
    its pixel): pairs three pixels apart sit exactly at 0.02f, a rounding either side of it, and between 0.02f and 0.02."""
    K = kmat(75.0, 75.0, (n - 1) / 2 + 0.25, (n - 1) / 2 - 0.25)
    raw = encode_depth(np.full((n, n), 5000, np.uint16))
    return raw, np.ones((n, n), np.uint8), K


def pair_d2(cen):
    c = cen.astype(np.float64)
    d = c[:, None, :] - c[None, :, :]
    return (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]


# ------------------------------------------------------------------------------------------------ CPU: the restatement itself
def test_tie_frame_has_pairs_on_every_side_of_the_radius():
    raw, mask, K = tie_frame()
    cen = sp.voxel_centroids(sp.backproject(sp.decode_depth(raw), mask, 1, K), 0.005)
    assert len(cen) == mask.size                                          # one pixel per voxel
    d2 = pair_d2(cen)
    r32 = float(np.float32(0.02))
    below = float(np.nextafter(np.float32(0.02), np.float32(0))) ** 2
    assert (d2 == r32 * r32).sum() > 0                                    # exactly at the fp32 radius
    assert ((d2 > r32 * r32) & (d2 <= 0.02 * 0.02)).sum() > 0             # between 0.02f and 0.02
    assert ((d2 >= below) & (d2 < r32 * r32)).sum() > 0                   # within an fp32 ulp below


def test_neighbour_predicate_is_the_kernels():
    """segment_port.neighbours against a brute-force float64 form of the kernel's predicate ((dx*dx + dy*dy) + dz*dz <= r*r,
    r the fp32 radius), over every pair of the tie frame and of a noisy surface; the kd-tree's own radius test (0.02, its own
    summation) is shown to differ on the tie frame -- it counts the pairs between 0.02f and 0.02."""
    from scipy.spatial import cKDTree
    raw, mask, K = tie_frame()
    tie = sp.voxel_centroids(sp.backproject(sp.decode_depth(raw), mask, 1, K), 0.005)
    Ks = kmat(300.0, 300.0, 29.5, 19.5)
    noisy = sp.voxel_centroids(sp.backproject(sp.decode_depth(encode_depth(raycast("sphere", 40, 60, Ks, 5e-4))),
                                              np.ones((40, 60), np.uint8), 1, Ks), 0.005)
    for cen in (tie, noisy):
        d2 = pair_d2(cen)
        for r in (0.02, 0.015, 0.03):
            r32 = float(np.float32(r))
            brute = [np.flatnonzero(row <= r32 * r32).tolist() for row in d2]
            assert sp.neighbours(cen, r) == brute
    old = cKDTree(tie).query_ball_point(tie, 0.02)
    assert sum(len(o) for o in old) > sum(len(n) for n in sp.neighbours(tie, 0.02))


def test_chol6_port_solves_and_refuses_like_the_kernel():
    """segment_port.chol6_solve: a well-conditioned system is solved to float64 rounding; the systems of points on one line and
    on two lines (singular up to rounding, pivots near 1e-16 of the diagonal) are refused whatever the rounding."""
    rng = np.random.default_rng(3)
    M = rng.normal(size=(6, 6))
    A = M @ M.T + 6 * np.eye(6)
    b = rng.normal(size=6)
    x = sp.chol6_solve(A, b)
    assert np.abs(A @ x - b).max() < 1e-12
    t = np.linspace(-0.02, 0.02, 9)
    for uu, vv in ((t, 0.3 * t), (np.r_[t, t], np.r_[np.full(9, -0.005), np.full(9, 0.005)])):
        P = np.stack([np.ones_like(uu), vv, vv * vv, uu, uu * vv, uu * uu])
        A = (P * np.exp(-(uu * uu + vv * vv) / 4e-4)) @ P.T
        assert sp.chol6_solve(A, np.ones(6)) is None


# ------------------------------------------------------------------------------------------------ GPU: decode and validity
@gpu
def test_every_raw_depth_value(engine):
    """All 65536 raw values in one 256 x 256 frame, the whole mask the class, PCA mode and min_neighbors 0 (every centroid kept):
    the pixel count is the restatement's -- decoded 1000 .. 19999, since (double)0.1f > 0.1 and 2.0 is not < 2.0 -- and every
    point is bit for bit the restatement's."""
    raw = np.arange(65536, dtype=np.uint32).astype(np.uint16).reshape(256, 256)
    mask = np.full((256, 256), 9, np.uint8)
    K = kmat(211.0, 197.0, 127.3, 128.6)
    want = reference(raw, mask, 9, K, 0.01, 0.02, 0.03, 0, False)
    assert want["n_raw"] == 19000
    with mls_mode(engine, 0):
        got = engine.prepare_segment(raw, mask, 9, K, 0.01, 0.02, 0.03, 0)
    compare(got, want, 0.02, False)
    assert len(got[0]) == len(want["cen"])


# ------------------------------------------------------------------------------------------------ GPU: frame shapes and intrinsics
SHAPES = [  # rows, cols, K, class, other labels
    (1, 1, kmat(500.0, 500.0, 0.3, 0.7), 0, ()),
    (1, 33, kmat(-480.0, 510.0, 16.25, 0.4), 255, (0, 3)),
    (17, 13, kmat(90.0, -75.5, 6.6, 8.3), 0, (255, 1)),
    (479, 641, kmat(-533.5, 529.25, 320.7, 239.2), 255, (0, 254, 7)),
    (480, 640, kmat(525.0, 531.0, 319.5, 239.5), 0, (255, 12)),
]


@gpu
@pytest.mark.parametrize("rows,cols,K,cls,others", SHAPES, ids=[f"{s[0]}x{s[1]}" for s in SHAPES])
def test_frame_shapes_and_intrinsics(engine, rows, cols, K, cls, others):
    """Frame sizes from 1 x 1 up, non-integer principal points, fx != fy, negative focal lengths, class ids 0 and 255 with other
    labels interleaved in the mask; the principal point inside the frame puts points and voxel indices on both sides of 0."""
    dec = raycast("sphere" if rows * cols > 1000 else "plane", rows, cols, np.abs(K), 3e-4, seed=rows)
    u, v = np.mgrid[0:rows, 0:cols]
    mask = np.full((rows, cols), cls, np.uint8)
    for k, o in enumerate(others):
        mask[(u * 7 + v * 3 + k) % (len(others) + 3) == 0] = o
    run_both(engine, encode_depth(dec), mask, cls, K)


def boundary_frame():
    """Depths 0.4 .. 1.1875 m in steps of 12.5 mm, mixed over the frame, x = (v - cx) d / fx: many x / leaf and y / leaf land exactly
    on an integer in fp32 or one ulp either side."""
    rows, cols = 40, 81
    K = kmat(100.0, 100.0, 40.0, 20.0)
    u, v = np.mgrid[0:rows, 0:cols]
    dec = (4000 + 125 * ((u * 7 + v * 5) % 64)).astype(np.uint16)
    return encode_depth(dec), np.ones((rows, cols), np.uint8), K


def test_boundary_frame_reaches_the_voxel_edges():
    raw, mask, K = boundary_frame()
    pts = sp.backproject(sp.decode_depth(raw), mask, 1, K)
    leaf = np.float32(0.01)
    for axis in (0, 1):
        q = (pts[:, axis] / leaf).astype(np.float32)
        f = np.floor(q)
        up, down = np.nextafter(f, np.float32(np.inf)), np.nextafter(f + 1, np.float32(-np.inf))
        assert (q == f).sum() > 10 and (q == up).sum() > 0 and (q == down).sum() > 0
        assert (q < 0).sum() > 10 and (q > 0).sum() > 10


@gpu
def test_voxel_boundaries(engine):
    raw, mask, K = boundary_frame()
    run_both(engine, raw, mask, 1, K, mn=1)


# ------------------------------------------------------------------------------------------------ GPU: parameters and surfaces
LEAVES = [0.0025, 0.005, 0.01, 0.02]
SURFACES = ["plane", "sphere", "corner", "ridge"]
RADII = [(2.0, 3.0, 10), (16.0, 2.0, 1), (8.0, 16.0, 400), (4.0, 1.5, 0), (16.0, 16.0, 10), (1.5, 4.0, 1), (3.0, 8.0, 25), (6.0, 12.0, 0)]
CASES = [(s, noisy, leaf) for s in SURFACES for noisy in (False, True) for leaf in LEAVES]


@gpu
@pytest.mark.parametrize("surface,noisy,leaf", CASES, ids=[f"{s}-{'noisy' if n else 'exact'}-{leaf * 1000:g}mm" for s, n, leaf in CASES])
def test_parameters_on_surfaces(engine, surface, noisy, leaf):
    """Leaf 2.5 .. 20 mm, radii from 1.5 to 16 leaves, min_neighbors 0, 1, 10 and above any count, both modes, on a tilted plane,
    a sphere cap, a box corner and the V ridge, exact and with 0.5 mm depth noise.  The pixel pitch is about half a leaf."""
    k = CASES.index((surface, noisy, leaf))
    fn, fo, mn = RADII[k % len(RADII)]
    fx = 0.7 / (0.5 * leaf)
    K = kmat(fx, fx * 1.01, 39.7, 31.4)
    dec = raycast(surface, 64, 80, K, 5e-4 if noisy else 0.0, seed=k)
    nr, orr = float(np.float32(fn * leaf)), float(np.float32(fo * leaf))
    run_both(engine, encode_depth(dec), np.ones((64, 80), np.uint8), 1, K, leaf, nr, orr, mn, min_tight=0.5)


def ridge_frame():
    K = kmat(300.0, 300.0, 44.5, 29.5)
    return encode_depth(raycast("ridge", 60, 90, K)), np.ones((60, 90), np.uint8), K


@gpu
@pytest.mark.parametrize("leaf,nr,orr,mn", [(0.005, 0.08, 0.01, 10), (0.0025, 0.04, 0.01, 10), (0.0025, 0.04, 0.01, 30)])
def test_mls_outlier_window_covers_the_displacement(engine, leaf, nr, orr, mn):
    """The V ridge with a wide MLS radius: the projection moves points near the crease by up to 3.3 cm, more than the 2 x 2 voxels
    the outlier search once allowed, so neighbours of the projected cloud lie outside a window sized for normal_r <= 2 leaves."""
    raw, mask, K = ridge_frame()
    want = reference(raw, mask, 1, K, leaf, nr, orr, mn, True)
    disp = np.linalg.norm(want["xyz"].astype(np.float64) - want["cen"][want["idx"]], axis=1)
    assert disp.max() > 2 * leaf + orr
    with mls_mode(engine, 1):
        got = engine.prepare_segment(raw, mask, 1, K, leaf, nr, orr, mn)
    compare(got, want, nr, True)


# ------------------------------------------------------------------------------------------------ GPU: ties at the radius
@gpu
@pytest.mark.parametrize("mls", [0, 1])
def test_neighbours_at_the_radius(engine, mls):
    """The tie frame with normal_r = outlier_r = 0.02: min_neighbors set to the count of a point with a pair exactly at 0.02f
    (kept only if that pair counts) and to one more than the count of a point with a pair between 0.02f and 0.02 (kept only if
    that pair wrongly counts).  On the exact plane MLS leaves every point where it is, so the ties survive the projection."""
    raw, mask, K = tie_frame()
    cen = sp.voxel_centroids(sp.backproject(sp.decode_depth(raw), mask, 1, K), 0.005)
    d2 = pair_d2(cen)
    r32 = float(np.float32(0.02))
    cnt = (d2 <= r32 * r32).sum(axis=1)
    at = np.flatnonzero((d2 == r32 * r32).any(axis=1))
    between = np.flatnonzero(((d2 > r32 * r32) & (d2 <= 0.02 * 0.02)).any(axis=1))
    for mn in sorted({int(cnt[at].min()), int(cnt[at].max()), int(cnt[between].min()) + 1, int(cnt[between].max()) + 1}):
        run_both(engine, raw, mask, 1, K, 0.005, 0.02, 0.02, mn, modes=(mls,))


# ------------------------------------------------------------------------------------------------ GPU: line-like segments
def strip_masks(rows, cols):
    u, v = np.mgrid[0:rows, 0:cols]
    return {"row": u == rows // 2, "column": v == cols // 2, "diagonal": u == v, "two_rows": (u == rows // 2) | (u == rows // 2 + 1),
            "anti_diagonal_pair": (u + v == cols // 2) | (u + v == cols // 2 + 1)}


@gpu
@pytest.mark.parametrize("strip", ["row", "column", "diagonal", "two_rows", "anti_diagonal_pair"])
@pytest.mark.parametrize("surface", ["plane", "sphere"])
def test_line_like_segments(engine, strip, surface):
    """Thin masks on a plane and on a sphere, one pixel per 5 mm voxel so that the strips stay strips: centroids on one or two
    lines up to the depth's 0.1 mm steps, whose 6x6 systems are singular or nearly so.  Same points kept, positions as the
    module docstring says, in both modes."""
    rows = cols = 48
    K = kmat(110.0, 110.0, 23.5, 23.5)
    dec = raycast(surface, rows, cols, K)
    mask = strip_masks(rows, cols)[strip].astype(np.uint8) * 4
    for nr, orr, mn in ((0.02, 0.03, 3), (0.04, 0.02, 1), (0.08, 0.08, 10)):
        run_both(engine, encode_depth(dec), mask, 4, K, 0.005, nr, orr, mn)


# ------------------------------------------------------------------------------------------------ GPU: degenerate inputs
def raw_call(engine, raw, mask, cls, K, leaf=0.01, nr=0.02, orr=0.03, mn=10, cap=64, rows=None, cols=None):
    """pgp_prepare_segment on sentinel-filled outputs: (rc, xyz, nrm, n_valid_pixels) with whatever the call left in them."""
    d = np.ascontiguousarray(raw, np.uint16)
    m = np.ascontiguousarray(mask, np.uint8)
    k9 = np.ascontiguousarray(np.asarray(K, np.float32).reshape(9))
    xyz = np.full((max(cap, 1), 3), -7.0, np.float32)
    nrm = np.full((max(cap, 1), 3), -7.0, np.float32)
    nval = C.c_int(-12345)
    p = lambda a: C.c_void_p(a.ctypes.data)
    rc = engine._lib.pgp_prepare_segment(engine._ctx, p(d), p(m), d.shape[0] if rows is None else rows, d.shape[1] if cols is None else cols,
                                         int(cls), p(k9), float(leaf), float(nr), float(orr), int(mn), p(xyz), p(nrm), int(cap), C.byref(nval))
    return rc, xyz, nrm, nval.value


@gpu
@pytest.mark.parametrize("mls", [0, 1])
def test_one_valid_pixel(engine, mls):
    """A single valid pixel: PCA mode returns it with the normal -c / |c|; MLS drops it (fewer than 3 neighbours)."""
    raw = np.zeros((9, 11), np.uint16)
    raw[4, 7] = encode_depth(np.uint16(6543))
    mask = np.ones((9, 11), np.uint8)
    K = kmat(300.0, 310.0, 5.2, 3.9)
    with mls_mode(engine, mls):
        xyz, nrm, n_raw = engine.prepare_segment(raw, mask, 1, K, min_neighbors=1)
    assert n_raw == 1
    if mls:
        assert len(xyz) == 0
    else:
        want = reference(raw, mask, 1, K, 0.01, 0.02, 0.03, 1, False)
        assert np.array_equal(xyz, want["xyz"]) and len(xyz) == 1
        c = xyz[0].astype(np.float64)
        assert np.array_equal(nrm[0], (-c / np.linalg.norm(c)).astype(np.float32))


@gpu
@pytest.mark.parametrize("mls", [0, 1])
def test_empty_results_write_nothing(engine, mls):
    """No valid depth (zeros, too near, 2 m and beyond, another class): n = 0 and no count; every point an outlier: n = 0 with the
    pixel count.  Neither writes a point."""
    K = kmat(200.0, 200.0, 15.5, 11.5)
    dec = raycast("plane", 24, 32, K)
    mask = np.ones((24, 32), np.uint8)
    bad = dec.copy()
    bad[:8] = 0
    bad[8:16] = 1000 - 1
    bad[16:] = 20000
    with mls_mode(engine, mls):
        for raw, cls, mn, n_raw in ((encode_depth(bad), 1, 0, 0), (encode_depth(dec), 2, 0, 0), (encode_depth(dec), 1, 10 ** 6, 24 * 32)):
            rc, xyz, nrm, nval = raw_call(engine, raw, mask, cls, K, mn=mn)
            assert rc == 0 and nval == n_raw
            assert np.all(xyz == -7.0) and np.all(nrm == -7.0)


@gpu
def test_capacity_edge(engine):
    """cap equal to the number of points succeeds and fills exactly cap rows; cap one less is PGP_E_CAPACITY with no point written."""
    K = kmat(200.0, 200.0, 15.5, 11.5)
    raw = encode_depth(raycast("sphere", 24, 32, K))
    mask = np.ones((24, 32), np.uint8)
    xyz, nrm, _ = engine.prepare_segment(raw, mask, 1, K, 0.005, 0.02, 0.02, 3)
    n = len(xyz)
    assert n > 10
    rc, x, nr_, _ = raw_call(engine, raw, mask, 1, K, 0.005, 0.02, 0.02, 3, cap=n)
    assert rc == n and np.array_equal(x, xyz) and np.array_equal(nr_, nrm)
    rc, x, nr_, _ = raw_call(engine, raw, mask, 1, K, 0.005, 0.02, 0.02, 3, cap=n - 1)
    assert rc == PGP_E_CAPACITY and np.all(x == -7.0) and np.all(nr_ == -7.0)


# ------------------------------------------------------------------------------------------------ GPU: scratch history
@gpu
@pytest.mark.parametrize("mls", [0, 1])
def test_scratch_history(engine, mls):
    """A large frame, a small one, the large one again on one engine: each result bit for bit what a fresh engine returns."""
    from physimglobalpose_b200.engine import PoseEngine
    Kb, Ks = kmat(525.0, 525.0, 319.5, 239.5), kmat(150.0, 150.0, 20.5, 14.5)
    big = (encode_depth(raycast("corner", 480, 640, Kb, 5e-4)), np.ones((480, 640), np.uint8), 1, Kb, 0.005, 0.02, 0.03, 10)
    small = (encode_depth(raycast("sphere", 30, 40, Ks, 5e-4, seed=2)), np.ones((30, 40), np.uint8), 1, Ks, 0.01, 0.08, 0.05, 5)
    fresh = {}
    for name, args in (("big", big), ("small", small)):
        e = PoseEngine(0)
        try:
            e.set_option("k7_mls", mls)
            fresh[name] = e.prepare_segment(*args)
        finally:
            e.close()
    with mls_mode(engine, mls):
        for name, args in (("big", big), ("small", small), ("big", big)):
            got = engine.prepare_segment(*args)
            want = fresh[name]
            assert got[2] == want[2] and np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), name


# ------------------------------------------------------------------------------------------------ GPU: refusals
@gpu
@pytest.mark.parametrize("entry,value", [(0, np.nan), (2, np.inf), (4, -np.inf), (5, np.nan), (8, np.nan), (1, np.inf)])
def test_refuses_non_finite_intrinsics(engine, entry, value):
    K = kmat(200.0, 200.0, 15.5, 11.5)
    raw = encode_depth(raycast("plane", 24, 32, K))
    K = K.copy()
    K.reshape(9)[entry] = value
    rc, xyz, nrm, nval = raw_call(engine, raw, np.ones((24, 32), np.uint8), 1, K)
    assert rc == PGP_E_INVALID and nval == -12345 and np.all(xyz == -7.0) and np.all(nrm == -7.0)


@gpu
def test_refuses_tiny_leaf(engine):
    """A leaf so small that a voxel index could pass 2^30 is refused before anything runs (its index span would wrap an int); the
    smallest leaf the bound allows for the same frame still runs."""
    K = kmat(200.0, 200.0, 15.5, 11.5)
    raw = encode_depth(raycast("plane", 24, 32, K))
    mask = np.ones((24, 32), np.uint8)
    for leaf in (1e-10, 1e-9, 1.8e-9):
        rc, xyz, nrm, nval = raw_call(engine, raw, mask, 1, K, leaf, 16 * leaf, 16 * leaf, 1)
        assert rc == PGP_E_INVALID and nval == -12345 and np.all(xyz == -7.0) and np.all(nrm == -7.0)
    coord = max(2.0, 2.0 * max(16.5, 15.5) / 200.0, 2.0 * max(12.5, 11.5) / 200.0)
    leaf = float(np.float32(coord / 2 ** 30 * 1.001))
    rc, *_ = raw_call(engine, raw, mask, 1, K, leaf, leaf, leaf, 1)
    assert rc in (0, -6)                                                  # runs; the table may be too large (PGP_E_TOO_LARGE)


@gpu
def test_refuses_overflowing_frame_size(engine):
    """rows x cols beyond int (and beyond the 2^30 pixels K7 indexes) is refused before a byte of the frame is read."""
    K = kmat(200.0, 200.0, 15.5, 11.5)
    raw = np.zeros((1, 1), np.uint16)
    mask = np.ones((1, 1), np.uint8)
    for rows, cols in ((65536, 65536), (46341, 46341), (1 << 15, (1 << 15) + 1), (3, 1 << 30)):
        rc, xyz, nrm, nval = raw_call(engine, raw, mask, 1, K, rows=rows, cols=cols)
        assert rc == PGP_E_INVALID and nval == -12345 and np.all(xyz == -7.0)
    # the engine is untouched by the refusals
    xyz, nrm, n_raw = engine.prepare_segment(encode_depth(raycast("plane", 24, 32, K)), np.ones((24, 32), np.uint8), 1, K)
    assert n_raw == 24 * 32 and len(xyz) > 0
