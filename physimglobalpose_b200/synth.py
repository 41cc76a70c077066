"""Seeded synthetic clouds and pose hypotheses of the shapes BASELINE.json names.

Generator spec: SURVEY.md 8(d) / BASELINE.md 3 (box model, GT pose, plane + clutter scene,
GT / perturbed / uniform hypotheses handed over as fp32 centred-frame 3x4 matrices).  The
same bytes go to the CUDA path, to the C restatement and to the compiled reference, so the
RNG only has to be deterministic (numpy PCG64), not the survey's std::mt19937 stream;
k-bar and the roofline bytes are always recomputed from the actual inputs (bench.py).
"""
from __future__ import annotations

import dataclasses

import numpy as np

BOX = (0.10, 0.15, 0.20)
GT_T = (0.10, -0.05, 0.60)
GT_AXIS = (0.3, 0.5, 0.8)
GT_ANGLE = 0.7


def rot_axis_angle(axis, angle) -> np.ndarray:
    a = np.asarray(axis, dtype=np.float64)
    a = a / np.linalg.norm(a)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(angle) * K + (1 - np.cos(angle)) * (K @ K)


def sample_box(rng: np.random.Generator, n: int, dims) -> tuple[np.ndarray, np.ndarray]:
    """n points uniform (area-weighted) on the six faces of a box centred at 0; outward normals."""
    dx, dy, dz = dims
    areas = np.array([dy * dz, dy * dz, dx * dz, dx * dz, dx * dy, dx * dy])
    face = rng.choice(6, size=n, p=areas / areas.sum())
    u = rng.uniform(-0.5, 0.5, size=n)
    v = rng.uniform(-0.5, 0.5, size=n)
    pts = np.zeros((n, 3))
    nrm = np.zeros((n, 3))
    half = np.array(dims) / 2
    for f in range(6):
        m = face == f
        ax = f // 2
        sgn = 1.0 if f % 2 == 0 else -1.0
        o1, o2 = [a for a in range(3) if a != ax]
        pts[m, ax] = sgn * half[ax]
        pts[m, o1] = u[m] * dims[o1]
        pts[m, o2] = v[m] * dims[o2]
        nrm[m, ax] = sgn
    return pts, nrm


def box_mesh(dims, n: int = 1) -> tuple[np.ndarray, np.ndarray]:
    """Box centred at 0, every face an n x n grid of quads split into two triangles: 12 n^2 triangles, fp32 vertices, int32
    indices.  Neighbouring faces do not share vertices (a render of the box is closed all the same: the seams coincide)."""
    half = np.asarray(dims, np.float64) / 2
    g = np.linspace(-1.0, 1.0, n + 1)
    verts, tris = [], []
    for ax in range(3):
        o1, o2 = [a for a in range(3) if a != ax]
        for sgn in (1.0, -1.0):
            u, v = np.meshgrid(g, g, indexing="ij")
            p = np.zeros((n + 1, n + 1, 3))
            p[..., ax] = sgn * half[ax]
            p[..., o1] = u * half[o1]
            p[..., o2] = v * half[o2]
            base = sum(len(x) for x in verts)
            i = np.arange(n)[:, None] * (n + 1) + np.arange(n)[None, :]
            q = np.stack([i, i + n + 1, i + n + 2, i + 1], -1).reshape(-1, 4) + base
            tris.append(np.concatenate([q[:, [0, 1, 2]], q[:, [0, 2, 3]]]))
            verts.append(p.reshape(-1, 3))
    return np.concatenate(verts).astype(np.float32), np.concatenate(tris).astype(np.int32)


def ellipsoid_mesh(radii, n_lat: int, n_lon: int) -> tuple[np.ndarray, np.ndarray]:
    """UV-sphere scaled to `radii`: 2 n_lon (n_lat - 1) triangles, shared vertices, poles included."""
    th = np.linspace(0, np.pi, n_lat + 1)[1:-1]
    ph = np.linspace(0, 2 * np.pi, n_lon, endpoint=False)
    T, P = np.meshgrid(th, ph, indexing="ij")
    ring = np.stack([np.sin(T) * np.cos(P), np.sin(T) * np.sin(P), np.cos(T)], -1).reshape(-1, 3)
    verts = np.concatenate([[[0, 0, 1]], ring, [[0, 0, -1]]]) * np.asarray(radii, np.float64)
    j = np.arange(n_lon)
    jn = (j + 1) % n_lon
    tris = [np.stack([np.zeros(n_lon, int), 1 + j, 1 + jn], -1)]
    for r in range(n_lat - 2):
        a, b = 1 + r * n_lon, 1 + (r + 1) * n_lon
        tris += [np.stack([a + j, b + j, b + jn], -1), np.stack([a + j, b + jn, a + jn], -1)]
    last, pole = 1 + (n_lat - 2) * n_lon, len(verts) - 1
    tris.append(np.stack([last + j, np.full(n_lon, pole), last + jn], -1))
    return verts.astype(np.float32), np.concatenate(tris).astype(np.int32)


def seq_centroid_f32(xyz: np.ndarray) -> np.ndarray:
    """Sequential fp32 sum / n, the way Match4PCSBase::init accumulates centroids
    (/root/reference/src/3rdparty/super4pcs/src/super4pcs/algorithms/match4pcsBase.cc:242-250)."""
    x = np.ascontiguousarray(xyz, dtype=np.float32)
    s = np.add.accumulate(x, axis=0, dtype=np.float32)[-1]
    return (s / np.float32(x.shape[0])).astype(np.float32)


@dataclasses.dataclass
class Problem:
    scene_xyz: np.ndarray      # (Ns,3) f32, camera frame
    scene_nrm: np.ndarray      # (Ns,3) f32 unit
    scene_prior: np.ndarray    # (Ns,)  f32
    model_xyz: np.ndarray      # (Nm,3) f32, model frame (validation == search sampling)
    model_nrm: np.ndarray      # (Nm,3) f32 unit
    delta: float
    gt_pose: np.ndarray        # (4,4) f64 model -> camera
    c_scene: np.ndarray        # (3,) f32 sequential centroid of the scene
    c_model: np.ndarray        # (3,) f32 sequential centroid of the (search) model


def make_problem(n_model: int = 2000, n_scene: int = 100_000, delta: float = 0.01, seed: int = 1234) -> Problem:
    rng = np.random.default_rng(seed)
    mp, mn = sample_box(rng, n_model, BOX)
    R = rot_axis_angle(GT_AXIS, GT_ANGLE)
    t = np.array(GT_T)
    gt = np.eye(4)
    gt[:3, :3] = R
    gt[:3, 3] = t

    n_obj = int(round(0.15 * n_scene))
    n_plane = int(round(0.45 * n_scene))
    n_clut = n_scene - n_obj - n_plane
    op, on = sample_box(rng, n_obj, BOX)
    op = op @ R.T + t
    on = on @ R.T
    pp = np.stack([rng.uniform(-0.5, 0.5, n_plane), rng.uniform(-0.5, 0.5, n_plane), np.full(n_plane, 0.75)], axis=1)
    pn = np.tile(np.array([0.0, 0.0, -1.0]), (n_plane, 1))
    cps, cns = [], []
    per = [n_clut // 6 + (1 if i < n_clut % 6 else 0) for i in range(6)]
    for i in range(6):
        cp, cn = sample_box(rng, per[i], (0.15, 0.12, 0.20))
        ang = 2 * np.pi * i / 6
        Rz = rot_axis_angle((0, 0, 1), ang + 0.3)
        cps.append(cp @ Rz.T + np.array([0.3 * np.cos(ang), 0.3 * np.sin(ang), 0.6]))
        cns.append(cn @ Rz.T)
    sp = np.concatenate([op, pp] + cps)
    sn = np.concatenate([on, pn] + cns)
    sp = sp + rng.uniform(-0.001, 0.001, size=sp.shape)
    perm = rng.permutation(sp.shape[0])
    sp, sn = sp[perm], sn[perm]

    scene_xyz = np.ascontiguousarray(sp, dtype=np.float32)
    model_xyz = np.ascontiguousarray(mp, dtype=np.float32)
    return Problem(
        scene_xyz=scene_xyz,
        scene_nrm=np.ascontiguousarray(sn, dtype=np.float32),
        scene_prior=np.ones(scene_xyz.shape[0], dtype=np.float32),
        model_xyz=model_xyz,
        model_nrm=np.ascontiguousarray(mn, dtype=np.float32),
        delta=float(delta),
        gt_pose=gt,
        c_scene=seq_centroid_f32(scene_xyz),
        c_model=seq_centroid_f32(model_xyz),
    )


def make_segment_problem(n_model: int = 1000, n_segment: int = 2000, delta: float = 0.005, seed: int = 77,
                         noise: float = 0.001) -> Problem:
    """Test-scene-sized object request: the scene is ONE object's segment -- the camera-visible part
    of the model surface at the GT pose (camera at the origin), jittered by +-noise -- as
    CongruentSetMatching::generate hands it to the matcher
    (/root/reference/src/physim_pose_estimation/src/hypothesis_generation/ObjectPoseCandidateSet.cpp:23-74)."""
    rng = np.random.default_rng(seed)
    mp, mn = sample_box(rng, n_model, BOX)
    R = rot_axis_angle(GT_AXIS, GT_ANGLE)
    t = np.array(GT_T)
    gt = np.eye(4)
    gt[:3, :3] = R
    gt[:3, 3] = t
    pts, nrm = [], []
    while sum(len(p) for p in pts) < n_segment:
        sp, sn = sample_box(rng, 4 * n_segment, BOX)
        sp = sp @ R.T + t
        sn = sn @ R.T
        vis = np.einsum("ij,ij->i", sn, sp) < 0          # normal faces the camera at the origin
        pts.append(sp[vis]); nrm.append(sn[vis])
    sp = np.concatenate(pts)[:n_segment]
    sn = np.concatenate(nrm)[:n_segment]
    sp = sp + rng.uniform(-noise, noise, size=sp.shape)
    scene_xyz = np.ascontiguousarray(sp, dtype=np.float32)
    model_xyz = np.ascontiguousarray(mp, dtype=np.float32)
    return Problem(scene_xyz=scene_xyz, scene_nrm=np.ascontiguousarray(sn, dtype=np.float32),
                   scene_prior=np.ones(len(scene_xyz), np.float32), model_xyz=model_xyz,
                   model_nrm=np.ascontiguousarray(mn, dtype=np.float32), delta=float(delta), gt_pose=gt,
                   c_scene=seq_centroid_f32(scene_xyz), c_model=seq_centroid_f32(model_xyz))


def pose_error(pose_a: np.ndarray, pose_b: np.ndarray) -> tuple[float, float]:
    """(translation distance in metres, rotation angle in radians) between two 4x4 poses."""
    dt = float(np.linalg.norm(pose_a[:3, 3] - pose_b[:3, 3]))
    Rr = pose_a[:3, :3].T @ pose_b[:3, :3]
    ang = float(np.arccos(np.clip((np.trace(Rr) - 1) / 2, -1, 1)))
    return dt, ang


def centre_pose(pose: np.ndarray, c_scene: np.ndarray, c_model: np.ndarray) -> np.ndarray:
    """World pose(s) (…,4,4) f64 -> centred-frame row-major 3x4 fp32: Tr(-c_P) . T . Tr(c_Q)."""
    pose = np.asarray(pose, dtype=np.float64)
    R = pose[..., :3, :3]
    t = pose[..., :3, 3]
    tc = t + np.einsum("...ij,j->...i", R, c_model.astype(np.float64)) - c_scene.astype(np.float64)
    out = np.concatenate([R, tc[..., None]], axis=-1)
    return np.ascontiguousarray(out, dtype=np.float32)


def uncentre_pose(T: np.ndarray, c_scene: np.ndarray, c_model: np.ndarray) -> np.ndarray:
    """Inverse of centre_pose: centred 3x4 -> world 4x4 f64 (translation as in
    match4pcsBase.cc:1474-1482: c1 + cP - R (c2 + cQ) collapses to t_c + cP - R cQ)."""
    T = np.asarray(T, dtype=np.float64)
    R = T[..., :3, :3]
    t = T[..., :3, 3] + c_scene.astype(np.float64) - np.einsum("...ij,j->...i", R, c_model.astype(np.float64))
    out = np.zeros(T.shape[:-2] + (4, 4))
    out[..., :3, :3] = R
    out[..., :3, 3] = t
    out[..., 3, 3] = 1.0
    return out


def make_hypotheses(prob: Problem, n: int, seed: int = 4321, chunk: int = 1 << 20) -> np.ndarray:
    """(n,3,4) fp32 centred-frame transforms: 0 = GT, odd = GT o small perturbation
    (sigma_t 2 cm, sigma_theta 0.2 rad about a random axis), even = uniform pose in the scene volume."""
    rng = np.random.default_rng(seed)
    out = np.empty((n, 3, 4), dtype=np.float32)
    gt = prob.gt_pose
    for s in range(0, n, chunk):
        m = min(chunk, n - s)
        axis = rng.normal(size=(m, 3))
        axis /= np.linalg.norm(axis, axis=1, keepdims=True)
        idx = np.arange(s, s + m)
        odd = (idx % 2) == 1
        ang = np.where(odd, rng.normal(0, 0.2, size=m), rng.uniform(0, 2 * np.pi, size=m))
        K = np.zeros((m, 3, 3))
        K[:, 0, 1], K[:, 0, 2] = -axis[:, 2], axis[:, 1]
        K[:, 1, 0], K[:, 1, 2] = axis[:, 2], -axis[:, 0]
        K[:, 2, 0], K[:, 2, 1] = -axis[:, 1], axis[:, 0]
        Rr = np.eye(3)[None] + np.sin(ang)[:, None, None] * K + (1 - np.cos(ang))[:, None, None] * (K @ K)
        pose = np.zeros((m, 4, 4))
        pose[:, 3, 3] = 1
        # odd: GT o perturbation (perturbation applied in the model frame, then GT)
        dt = rng.normal(0, 0.02, size=(m, 3))
        R_odd = gt[:3, :3][None] @ Rr
        t_odd = gt[:3, 3][None] + dt
        # even: uniform pose in the scene volume
        t_even = np.stack([rng.uniform(-0.5, 0.5, m), rng.uniform(-0.5, 0.5, m), rng.uniform(0.4, 0.9, m)], axis=1)
        pose[:, :3, :3] = np.where(odd[:, None, None], R_odd, Rr)
        pose[:, :3, 3] = np.where(odd[:, None], t_odd, t_even)
        out[s:s + m] = centre_pose(pose, prob.c_scene, prob.c_model)
    if n > 0:
        out[0] = centre_pose(gt, prob.c_scene, prob.c_model)
    return out


def make_hypotheses_range(prob: Problem, lo: int, hi: int, seed: int = 4321, block: int = 1 << 18) -> np.ndarray:
    """Hypotheses [lo, hi) of an arbitrarily long list whose content depends only on (seed, index): the list is cut into blocks
    of `block` hypotheses, block b drawn with its own generator seeded (seed, b) exactly like make_hypotheses draws one chunk.
    Lets every rank of a sharded run build just its shard of the SAME global list (index 0 = GT)."""
    out = np.empty((max(hi - lo, 0), 3, 4), dtype=np.float32)
    b = lo // block
    while b * block < hi:
        s0, s1 = b * block, (b + 1) * block
        full = make_hypotheses(prob, block, seed=(seed * 1_000_003 + b) & 0x7FFFFFFF, chunk=block)
        if b != 0:                                  # only the list's first hypothesis is the exact GT
            full[0] = make_hypotheses(prob, 2, seed=(seed * 1_000_003 + b + 77) & 0x7FFFFFFF)[1]
        a, e = max(lo, s0), min(hi, s1)
        out[a - lo:e - lo] = full[a - s0:e - s0]
        b += 1
    return out


def kbar_27(prob: Problem, T: np.ndarray, max_hyp: int = 256) -> tuple[float, float]:
    """Mean number of scene points in the 27 delta-cells around a transformed model point
    (k-bar of SURVEY.md 8(d)) and the fraction of point-queries whose 27-neighbourhood is
    non-empty, over the first max_hyp hypotheses.  Grid anchored at the centred scene AABB min."""
    P = prob.scene_xyz - prob.c_scene
    V = prob.model_xyz - prob.c_model
    d = np.float32(prob.delta)
    lo = P.min(axis=0)
    dims = np.floor((P.max(axis=0) - lo) / d).astype(np.int64) + 1
    cell = np.floor((P - lo) / d).astype(np.int64)
    occ = np.zeros(tuple(dims + 2), dtype=np.int32)      # 1-cell apron
    np.add.at(occ, (cell[:, 0] + 1, cell[:, 1] + 1, cell[:, 2] + 1), 1)
    # 27-neighbourhood sum by separable box filter
    s = occ.astype(np.int64)
    for ax in range(3):
        s = s + np.roll(s, 1, axis=ax) + np.roll(s, -1, axis=ax)  # apron is empty so roll wrap is harmless
    T = T[:max_hyp].astype(np.float64)
    tp = np.einsum("hij,nj->hni", T[:, :, :3], V.astype(np.float64)) + T[:, None, :, 3]
    c = np.floor((tp - lo) / d).astype(np.int64) + 1
    inside = np.all((c >= 0) & (c < (dims + 2)), axis=-1)
    c = np.clip(c, 0, dims + 1)
    k = np.where(inside, s[c[..., 0], c[..., 1], c[..., 2]], 0)
    return float(k.mean()), float((k > 0).mean())
