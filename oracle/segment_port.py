"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the segment preparation that precedes the PCS -> LCP path
(PPE = /root/reference/src/physim_pose_estimation):
  depth decode     utilities::readDepthImage           PPE/src/misc/utilities.cpp:47-61   ((d << 13) | (d >> 3)) as u16, / 10000
  mask             GTSegmentation::compute2dSegment    PPE/src/segmentation/Segmentation.cpp:187-207
  back-projection  utilities::convert3dUnOrganizedRGB  PPE/src/misc/utilities.cpp:210-228  fp32 ((v - cx) * depth) / fx, 0.1 < depth < 2.0
  voxel centroids  pcl::VoxelGrid, leaf 1 cm           Segmentation.cpp:226-229  (centroid per voxel, output in voxel-index order)
  normals          pcl::MovingLeastSquares, r = 2 cm   Segmentation.cpp:231-238  -- mls_project (polynomial fit of order 2, projection +
                                                                                   normal); pca_normals = round 1's stand-in
  outlier removal  pcl::RadiusOutlierRemoval 3 cm / 10 PPE/src/hypothesis_generation/ObjectPoseCandidateSet.cpp:28-32
  normal flip      pcl::flipNormalTowardsViewpoint + renormalise  :39-51
PCL is not vendored in the reference tree and not installed: the three PCL filters are RESTATED, PARITY UNPINNED (VoxelGrid's
index convention and MLS's polynomial projection in particular).  The device kernels (k7_segment.cu) are checked against THIS file;
tests/golden/make_c1.py uses it to prepare the configs[0] fixture.  Only tests/ and tests/golden/ import it."""
from __future__ import annotations

import numpy as np


def decode_depth(raw_u16: np.ndarray) -> np.ndarray:
    raw = raw_u16.astype(np.uint16)
    dec = ((raw << np.uint16(13)) | (raw >> np.uint16(3))).astype(np.uint16)
    return (dec.astype(np.float32) / np.float32(10000)).astype(np.float32)


def backproject(depth_m: np.ndarray, mask: np.ndarray, cls: int, K: np.ndarray) -> np.ndarray:
    obj = np.where(mask == cls, depth_m, np.float32(0))
    o64 = obj.astype(np.float64)                                     # `depth > 0.1 && depth < 2.0` promotes the float to double
    u, v = np.nonzero((o64 > 0.1) & (o64 < 2.0))                     # row-major pixel order, like the double loop
    d = obj[u, v].astype(np.float32)
    x = ((v.astype(np.float32) - K[0, 2]) * d / K[0, 0]).astype(np.float32)
    y = ((u.astype(np.float32) - K[1, 2]) * d / K[1, 1]).astype(np.float32)
    return np.stack([x, y, d], axis=1)


def voxel_centroids(pts: np.ndarray, leaf: float = 0.01) -> np.ndarray:
    leaf = np.float32(leaf)
    ijk = np.floor(pts / leaf).astype(np.int64)
    ijk -= ijk.min(axis=0)
    dims = ijk.max(axis=0) + 1
    key = ijk[:, 0] + dims[0] * (ijk[:, 1] + dims[1] * ijk[:, 2])
    order = np.argsort(key, kind="stable")
    key, pts = key[order], pts[order]
    starts = np.flatnonzero(np.r_[True, key[1:] != key[:-1]])
    cnt = np.diff(np.r_[starts, len(key)])
    return (np.add.reduceat(pts.astype(np.float64), starts, axis=0) / cnt[:, None]).astype(np.float32)


def neighbours(cen: np.ndarray, radius: float) -> list:
    """Per point, the ascending indices of the points q with ((dx*dx + dy*dy) + dz*dz) <= r*r: the kernel's predicate, in double
    from the fp32 coordinates, each operation rounded, with r the fp32 radius the C ABI receives promoted to double (0.02f, not 0.02).
    The kd-tree only proposes candidates, within a slightly larger radius; the predicate decides."""
    from scipy.spatial import cKDTree
    r = float(np.float32(radius))
    c64 = cen.astype(np.float64)
    out = []
    for i, cand in enumerate(cKDTree(cen).query_ball_point(cen, r * (1.0 + 1e-6), return_sorted=True)):
        cand = np.asarray(cand, np.int64)
        d = c64[cand] - c64[i]
        d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        out.append(cand[d2 <= r * r].tolist())
    return out


def pca_normals(cen: np.ndarray, radius: float = 0.02) -> np.ndarray:
    nrm = np.zeros_like(cen)
    for i, nb in enumerate(neighbours(cen, radius)):
        q = cen[nb].astype(np.float64)
        if len(nb) >= 3:
            w, vec = np.linalg.eigh(np.cov((q - q.mean(axis=0)).T))
            n = vec[:, 0]
        else:
            n = -cen[i].astype(np.float64)
        if np.dot(n, cen[i]) > 0:
            n = -n
        nrm[i] = (n / np.linalg.norm(n)).astype(np.float32)
    return nrm


def _unit_orthogonal(n: np.ndarray) -> np.ndarray:
    """Eigen's Vector3d::unitOrthogonal() (what pcl::MovingLeastSquares builds its local frame with)."""
    x, y, z = n
    if not (abs(x) <= abs(z) * 1e-12) or not (abs(y) <= abs(z) * 1e-12):
        inv = 1.0 / np.sqrt(x * x + y * y)
        return np.array([-y * inv, x * inv, 0.0])
    inv = 1.0 / np.sqrt(y * y + z * z)
    return np.array([0.0, -z * inv, y * inv])


CHOL6_REL_PIVOT = 1e-10


def chol6_solve(A: np.ndarray, b: np.ndarray):
    """k7_segment.cu::chol6_solve, operation for operation in Python floats (IEEE double, no fused multiply-add): Cholesky of the
    lower triangle, then the two triangular solves.  None when a pivot is not above CHOL6_REL_PIVOT times its column's diagonal --
    a system singular up to rounding (neighbours on one or two lines) is not solved, on both sides, whatever the rounding."""
    n = len(b)
    L = [[float(A[i][j]) for j in range(n)] for i in range(n)]
    x = [float(v) for v in b]
    for j in range(n):
        d = L[j][j]
        for k in range(j):
            d -= L[j][k] * L[j][k]
        if not (d > CHOL6_REL_PIVOT * L[j][j]):
            return None
        d = float(np.sqrt(d))
        L[j][j] = d
        for i in range(j + 1, n):
            v = L[i][j]
            for k in range(j):
                v -= L[i][k] * L[j][k]
            L[i][j] = v / d
    for i in range(n):
        v = x[i]
        for k in range(i):
            v -= L[i][k] * x[k]
        x[i] = v / L[i][i]
    for i in range(n - 1, -1, -1):
        v = x[i]
        for k in range(i + 1, n):
            v -= L[k][i] * x[k]
        x[i] = v / L[i][i]
    return np.array(x)


def mls_project(cen: np.ndarray, radius: float = 0.02, order: int = 2):
    """pcl::MovingLeastSquares with setPolynomialFit(true), setComputeNormals(true), no upsampling, as the reference configures it
    (PPE/src/segmentation/Segmentation.cpp:231-238): per point, the (unweighted) PCA plane of its neighbours within `radius`, the
    query projected onto it, a weighted (exp(-d^2 / radius^2)) least-squares polynomial of total degree `order` in the plane's
    (u, v) frame over the same neighbours, the point moved along the plane normal by the polynomial's value at (0, 0) and the
    normal tilted by its gradient there.  Restated from PCL's published algorithm (mls.hpp, computeMLSPointNormal): PCL is not
    available here, PARITY UNPINNED.  Returns (points, unit normals oriented to the camera at the origin, valid mask): points
    with fewer than 3 neighbours are dropped by PCL (valid = False)."""
    n_coef = (order + 1) * (order + 2) // 2
    r = float(np.float32(radius))                                    # the weights use the fp32 radius, as the kernel does
    out_p = cen.astype(np.float64).copy()
    out_n = np.zeros((len(cen), 3))
    valid = np.zeros(len(cen), dtype=bool)
    for i, nb in enumerate(neighbours(cen, radius)):
        if len(nb) < 3:
            continue
        q = cen[nb].astype(np.float64)
        c = cen[i].astype(np.float64)
        mean = q.mean(axis=0)
        w_, vec = np.linalg.eigh((q - mean).T @ (q - mean))
        n = vec[:, 0]
        point = c - np.dot(c - mean, n) * n
        normal = n.copy()
        if len(nb) >= n_coef:
            de = q - point
            wgt = np.exp(-np.einsum("ij,ij->i", de, de) / (r * r))
            v_axis = _unit_orthogonal(n)
            u_axis = np.cross(n, v_axis)
            u, v, f = de @ u_axis, de @ v_axis, de @ n
            P = np.stack([u ** ui * v ** vi for ui in range(order + 1) for vi in range(order + 1 - ui)])     # [1, v, v^2, u, uv, u^2]
            A = (P * wgt) @ P.T
            b = (P * wgt) @ f
            coef = chol6_solve(A, b)
            if coef is not None:
                point = point + coef[0] * n
                normal = n - coef[order + 1] * u_axis - coef[1] * v_axis
        if np.dot(normal, point) > 0:
            normal = -normal
        out_p[i] = point
        out_n[i] = normal / np.linalg.norm(normal)
        valid[i] = True
    return out_p.astype(np.float32), out_n.astype(np.float32), valid


def radius_outlier_keep(cen: np.ndarray, radius: float = 0.03, min_neighbors: int = 10) -> np.ndarray:
    return np.array([len(nb) >= min_neighbors for nb in neighbours(cen, radius)], dtype=bool)      # the point itself counts, as in PCL


def prepare_segment(depth_m, mask, cls, K, leaf=0.01, normal_radius=0.02, outlier_radius=0.03, min_neighbors=10, mls=False):
    pts = backproject(depth_m, mask, cls, K)
    cen = voxel_centroids(pts, leaf)
    if mls:
        # the reference's order: MLS on the voxel centroids (points with < 3 neighbours vanish), then the radius-outlier filter on
        # the PROJECTED cloud (ObjectPoseCandidateSet.cpp:28-32)
        proj, nrm, valid = mls_project(cen, normal_radius)
        proj, nrm = proj[valid], nrm[valid]
        keep = radius_outlier_keep(proj, outlier_radius, min_neighbors)
        return proj[keep], nrm[keep], len(pts)
    nrm = pca_normals(cen, normal_radius)
    keep = radius_outlier_keep(cen, outlier_radius, min_neighbors)
    return cen[keep], nrm[keep], len(pts)
