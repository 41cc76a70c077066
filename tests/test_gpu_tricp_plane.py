"""K5's point-to-plane fit (`pgp_tricp_plane`) against a plain numpy restatement.

`plane_ref` follows the contract in include/pgp.h stage by stage, in float64 where the kernel uses double and in fp32 where it
uses fp32.  Start transform, queries, nearest neighbours, trim and stop are those of `tricp_ref` (tests/test_gpu_tricp.py), whose
helpers it reuses; per kept pair it forms r = n . (p' - q) and a = [p' x n, n] in double, sums E = sum r^2, H = sum a a^T and
g = -sum a r, solves x = H^+ g with the scaled, truncated pseudo-inverse (here through numpy's eigh, independently of the
kernel's Jacobi), and composes dR = Rz(gamma) Ry(beta) Rx(alpha), dt = x[3:] onto the fp32 transform.  The fit restates PCL's
TransformationEstimationPointToPlaneLLS (not vendored: parity unpinned), so the reference is pinned on the CPU against
independent facts: a noise-free box is recovered exactly, a plane moves only along its constrained directions, and the Euler
construction equals scipy's."""
import math

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

from physimglobalpose_b200 import _lib, synth
from tests.test_gpu_tricp import (FMAX, F32, PGP_E_INVALID, _far, _lattice_ties, _near, _problem, _trim_for, _ulp_close, inv_pose,
                                  morton_order, n_keep_of, nearest, query, retry_reached, tricp_ref)

PGP_E_NO_MODEL = -4
gpu = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------------------ the reference
def unit_normals(nrm):
    """pgp_set_model's stored normal in fp32: s = (n0^2 + n1^2) + n2^2, zero below 0.01, else n / sqrtf(s)."""
    n = np.asarray(nrm, F32).reshape(-1, 3)
    s = (n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1]) + n[:, 2] * n[:, 2]
    out = np.zeros_like(n)
    ok = s >= F32(0.01)
    out[ok] = n[ok] / np.sqrt(s[ok])[:, None]
    return out


def pinv_solve(H, g):
    """x = S V L^+ V^T S g with s_j = 1/sqrt(H_jj) (0 where H_jj <= 0), eigenvalues <= 1e-9 lambda_max dropped; and the rank kept."""
    H, g = np.asarray(H, np.float64), np.asarray(g, np.float64)
    d = np.diag(H)
    s = np.where(d > 0, 1.0 / np.sqrt(np.where(d > 0, d, 1.0)), 0.0)
    w, V = np.linalg.eigh(s[:, None] * H * s[None, :])
    lmax = w.max()
    keep = (w > 1e-9 * lmax) if lmax > 0 else np.zeros(6, bool)
    Vk = V[:, keep]
    return s * (Vk @ ((Vk.T @ (s * g)) / w[keep])), int(keep.sum())


def euler_zyx(x):
    """Rz(gamma) Ry(beta) Rx(alpha) in the kernel's association."""
    a, b, c = (float(v) for v in x[:3])
    ca, sa, cb, sb, cg, sg = math.cos(a), math.sin(a), math.cos(b), math.sin(b), math.cos(c), math.sin(c)
    return np.array([[cg * cb, -sg * ca + (cg * sb) * sa, sg * sa + (cg * sb) * ca],
                     [sg * cb, cg * ca + (sg * sb) * sa, -cg * sa + (sg * sb) * ca],
                     [-sb, cb * sa, cb * ca]])


def plane_rows(P, Q, N):
    """r and a = [p x n, n] per pair, in double."""
    P, Q, N = (np.asarray(v, np.float64) for v in (P, Q, N))
    r = ((P[:, 0] - Q[:, 0]) * N[:, 0] + (P[:, 1] - Q[:, 1]) * N[:, 1]) + (P[:, 2] - Q[:, 2]) * N[:, 2]
    a = np.stack([P[:, 1] * N[:, 2] - P[:, 2] * N[:, 1], P[:, 2] * N[:, 0] - P[:, 0] * N[:, 2], P[:, 0] * N[:, 1] - P[:, 1] * N[:, 0],
                  N[:, 0], N[:, 1], N[:, 2]], axis=1)
    return r, a


def plane_ref(seg, tgt, nrm, pose, trim=0.5, ratio=0.99, max_iter=100):
    """One pose.  Returns dict(pose, iters, energy, taus, energies, xs (the update of every fit), ranks)."""
    seg, tgt = np.asarray(seg, F32).reshape(-1, 3), np.asarray(tgt, F32).reshape(-1, 3)
    un = unit_normals(nrm)
    pose = np.asarray(pose, np.float64).reshape(4, 4)
    ns = len(seg)
    n_keep = n_keep_of(trim, ns)
    out = dict(pose=pose.copy(), iters=0, energy=F32(0), taus=[], energies=[], xs=[], ranks=[])
    if n_keep < 3:
        return out
    src = seg[morton_order(seg)]
    pos = np.arange(ns)
    T = inv_pose(pose)[:3].astype(F32)
    energy, it = FMAX, 0
    while True:
        q = query(T, src)
        d2, nn = nearest(q, tgt)
        kept = np.lexsort((pos, d2))[:n_keep]
        r, a = plane_rows(q[kept], tgt[nn[kept]], un[nn[kept]])
        with np.errstate(all="ignore"):
            old, energy = energy, F32(np.sum(r * r))
        if not energy <= FMAX:
            energy = F32(np.inf)
        out["taus"].append(d2[kept[-1]])
        out["energies"].append(energy)
        it += 1
        if energy <= FMAX:
            x, rank = pinv_solve(a.T @ a, -(a.T @ r))
            out["xs"].append(x)
            out["ranks"].append(rank)
            R = euler_zyx(x)
            T64 = T.astype(np.float64)
            T = np.concatenate([R @ T64[:, :3], (R @ T64[:, 3] + x[3:])[:, None]], axis=1).astype(F32)
        with np.errstate(all="ignore"):
            go = (energy / old) < F32(ratio) and it < max(1, max_iter)
        if not go:
            break
    out["iters"], out["energy"] = it, energy
    if energy <= FMAX:
        M = np.eye(4)
        M[:3] = T.astype(np.float64)
        out["pose"] = inv_pose(M)
    return out


# ------------------------------------------------------------------------------------------------------------ CPU: the 6x6 solve
@pytest.fixture(scope="module")
def lib():
    return _lib.load()


def _solve(lib, H, g):
    H, g = np.ascontiguousarray(H, np.float64), np.ascontiguousarray(g, np.float64)
    x = np.zeros(6)
    rank = lib.pgp_host_solve_plane6(H.ctypes.data, g.ctypes.data, x.ctypes.data)
    return x, rank


def _rows_of(shape, rng):
    """Point / unit-normal rows of a cylinder, two planes or one plane, in a random rigid placement."""
    n = 400
    if shape == "cylinder":
        th, z = rng.uniform(0, 2 * np.pi, n), rng.uniform(-0.05, 0.05, n)
        P = np.stack([0.04 * np.cos(th), 0.04 * np.sin(th), z], 1)
        N = np.stack([np.cos(th), np.sin(th), np.zeros(n)], 1)
    else:
        P = np.stack([rng.uniform(-0.05, 0.05, n), rng.uniform(-0.05, 0.05, n), np.zeros(n)], 1)
        N = np.tile([0.0, 0.0, 1.0], (n, 1))
        if shape == "two_planes":
            half = n // 2
            P[half:] = P[half:][:, [2, 1, 0]]                 # the plane x = 0
            N[half:] = [1.0, 0.0, 0.0]
    R = synth.rot_axis_angle(rng.normal(size=3), rng.uniform(0.3, 2.5))
    return P @ R.T + rng.normal(0, 0.2, 3), N @ R.T


def _agree(x, ref, w=None):
    w = np.ones(6) if w is None else w
    return np.linalg.norm(w * (x - ref)) <= 1e-12 * np.linalg.norm(w * ref) + 1e-300


def test_solve_plane6_matches_an_eigh_pseudo_inverse(lib):
    rng = np.random.default_rng(17)
    for _ in range(20):                                         # symmetric positive definite
        A = rng.normal(size=(6, 6))
        H = A @ A.T + 0.1 * np.eye(6)
        g = rng.normal(size=6)
        x, rank = _solve(lib, H, g)
        ref, rref = pinv_solve(H, g)
        assert rank == rref == 6 and _agree(x, ref)
        assert np.linalg.norm(H @ x - g) <= 1e-11 * np.linalg.norm(g)
    # rank-deficient matrices of real point / normal rows: a cylinder leaves the rotation about and the translation along its
    # axis free (rank 4), two planes the translation along their common line (rank 5), one plane its in-plane motion (rank 3)
    for shape, want in (("cylinder", 4), ("two_planes", 5), ("plane", 3)):
        for seed in range(4):
            P, N = _rows_of(shape, np.random.default_rng(seed))
            r = rng.normal(0, 1e-3, len(P))
            a = plane_rows(P, np.zeros_like(P), N)[1]
            H, g = a.T @ a, -(a.T @ r)
            x, rank = _solve(lib, H, g)
            ref, rref = pinv_solve(H, g)
            assert rank == rref == want, (shape, rank, rref)
            assert _agree(x, ref), (shape, x, ref)
            assert np.linalg.norm(H @ x - g) <= 1e-9 * np.linalg.norm(g), shape      # g lies in the range of H: solved there
    x, rank = _solve(lib, np.zeros((6, 6)), rng.normal(size=6))
    assert rank == 0 and not x.any()
    # diagonal scalings 1e-6 .. 1e6: D H D x' = D g has x' = D^-1 x, which the scaling recovers
    A = rng.normal(size=(6, 6))
    H, g = A @ A.T + 0.1 * np.eye(6), rng.normal(size=6)
    x0, _ = _solve(lib, H, g)
    for lo, hi in ((1e-6, 1e6), (1e-6, 1e-6), (1e6, 1e6), (1e-3, 1e3)):
        D = np.geomspace(lo, hi, 6)[rng.permutation(6)]
        x, rank = _solve(lib, D[:, None] * H * D[None, :], D * g)
        ref, _ = pinv_solve(D[:, None] * H * D[None, :], D * g)
        assert rank == 6 and _agree(x, ref, D) and _agree(D * x, x0), (lo, hi)


def test_euler_construction_is_extrinsic_xyz():
    rng = np.random.default_rng(5)
    for x in [np.zeros(3), *rng.uniform(-np.pi, np.pi, (20, 3)), *rng.normal(0, 1e-3, (5, 3))]:
        want = Rotation.from_euler("xyz", x).as_matrix()
        assert np.abs(euler_zyx(x) - want).max() <= 1e-15, x


# ------------------------------------------------------------------------------------------------------------ CPU: pin the reference
def _box_segment(seed=3, n_model=3000):
    """A noise-free box model with exact normals, and the model points of its camera-facing faces placed at the GT pose."""
    prob = synth.make_segment_problem(n_model, 10, 0.005, seed=seed, noise=0.0)
    R, t = prob.gt_pose[:3, :3], prob.gt_pose[:3, 3]
    cam = prob.model_xyz @ R.T + t
    vis = np.einsum("ij,ij->i", prob.model_nrm @ R.T, cam) < 0
    return prob, np.ascontiguousarray(cam[vis], F32)


def _offset(pose, ang, trans, seed):
    rng = np.random.default_rng(seed)
    P = pose.copy()
    P[:3, :3] = P[:3, :3] @ synth.rot_axis_angle(rng.normal(size=3), ang)
    d = rng.normal(size=3)
    P[:3, 3] += d / np.linalg.norm(d) * trans
    return P


def test_reference_recovers_a_noise_free_box():
    prob, seg = _box_segment()
    for seed in range(3):
        start = _offset(prob.gt_pose, math.radians(3), 0.01, seed)
        ref = plane_ref(seg, prob.model_xyz, prob.model_nrm, start, trim=0.9, ratio=0.99, max_iter=100)
        dt = np.linalg.norm(ref["pose"][:3, 3] - prob.gt_pose[:3, 3])
        ang = Rotation.from_matrix(ref["pose"][:3, :3] @ prob.gt_pose[:3, :3].T).magnitude()
        assert dt <= 1e-6 and ang <= 1e-6, (seed, dt, ang, ref["iters"])
        assert ref["ranks"][-1] == 6


def test_reference_keeps_the_free_motion_of_a_plane():
    """One plane (z = 0, normal +z): every update has gamma = tx = ty = 0 exactly, the segment ends on the plane, and the
    in-plane translation and the rotation about the normal change only through the composition with the tilts."""
    rng = np.random.default_rng(7)
    tgt = np.stack([rng.uniform(-0.1, 0.1, 3000), rng.uniform(-0.1, 0.1, 3000), np.zeros(3000)], 1).astype(F32)
    nrm = np.tile(np.array([0, 0, 1], F32), (len(tgt), 1))
    seg = np.stack([rng.uniform(-0.05, 0.05, 800), rng.uniform(-0.05, 0.05, 800), np.zeros(800)], 1)
    place = np.eye(4)
    place[:3, :3] = synth.rot_axis_angle([0, 0, 1], 0.3) @ synth.rot_axis_angle([1, 0.5, 0], 0.02)
    place[:3, 3] = [0.01, -0.02, 0.004]
    seg = (seg @ place[:3, :3].T + place[:3, 3]).astype(F32)
    start = np.eye(4)
    start[:3, :3] = synth.rot_axis_angle([0, 0, 1], -0.2)
    start[:3, 3] = [0.003, 0.002, 0.0]
    ref = plane_ref(seg, tgt, nrm, start, trim=1.0, ratio=0.99, max_iter=100)
    assert ref["iters"] >= 2 and all(rk == 3 for rk in ref["ranks"])
    xs = np.array(ref["xs"])
    assert not xs[:, 2:5].any()                                 # gamma, tx, ty
    T = inv_pose(ref["pose"])
    on_plane = seg.astype(np.float64) @ T[:3, :3].T + T[:3, 3]
    assert np.abs(on_plane[:, 2]).max() <= 1e-6
    T0 = inv_pose(start)
    yaw = lambda M: math.atan2(M[1, 0], M[0, 0])                # noqa: E731
    assert abs(yaw(T) - yaw(T0)) <= 1e-3 and np.abs(T[:2, 3] - T0[:2, 3]).max() <= 1e-4


# ------------------------------------------------------------------------------------------------------------ GPU
def _set(engine, prob, tgt=None, nrm=None):
    engine.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    engine.set_model(0, prob.model_xyz, prob.model_nrm, tgt if tgt is not None else prob.model_xyz,
                     nrm if nrm is not None else prob.model_nrm)


def _check(refined, iters, energy, refs, what="", pose_tol=1e-6):
    for k, r in enumerate(refs):
        assert iters[k] == r["iters"], (what, k, iters[k], r["iters"])
        assert _ulp_close(energy[k], r["energy"]), (what, k, float(energy[k]), float(r["energy"]))
        err = np.abs(refined[k] - r["pose"]).max()
        assert err <= pose_tol, (what, k, err, iters[k])


@gpu
@pytest.mark.parametrize("ns", [3, 4, 5, 1023, 1024, 2047, 2048, 2049, 4097, 20000])
def test_one_and_two_iterations(engine, ns):
    prob, seg = _problem(2000, max(ns, 600), seed=21, clutter=0)
    rng = np.random.default_rng(ns)
    seg = seg[rng.permutation(len(seg))[:ns]] if ns < len(seg) else seg
    seg = np.ascontiguousarray(seg[:ns], F32)
    _set(engine, prob)
    poses = np.concatenate([_near(prob, 2, ns), _far(prob, 1, ns + 1)])
    for spec in ("keep2", "keep3", 0.5, 1.0):
        trim = _trim_for(spec, ns)
        nk = n_keep_of(trim, ns)
        for max_iter in (0, 1, 2):
            refined, iters, energy = engine.tricp_plane(0, seg, poses, trim=trim, ratio=2.0, max_iter=max_iter)
            refs = [plane_ref(seg, prob.model_xyz, prob.model_nrm, P, trim=trim, ratio=2.0, max_iter=max_iter) for P in poses]
            _check(refined, iters, energy, refs, what=(ns, spec, max_iter))
            if nk < 3:
                assert np.array_equal(refined, poses) and not iters.any() and not energy.any()
            else:
                assert np.all(iters == max(1, max_iter))


def _cap_problem():
    """A 2.5 cm patch of one face turned by 0.01 rad about its centre, plus one exact point 8 cm away (tests/test_gpu_tricp.py's
    cap case), with the face's normals."""
    big = synth.make_segment_problem(20000, 10, 0.005, seed=12)
    tgt, nrm = big.model_xyz, big.model_nrm
    face = tgt[tgt[:, 2] == tgt[:, 2].max()]
    c = face[np.argmin(np.abs(face[:, 0] + 0.035) + np.abs(face[:, 1]))]
    lone = face[np.argmin(np.abs(face[:, 0] - 0.045) + np.abs(face[:, 1]))]
    patch = face[np.linalg.norm(face[:, :2] - c[:2], axis=1) < 0.025]
    src = np.concatenate([(patch - c) @ synth.rot_axis_angle([0, 1, 0], 0.01).T + c, lone[None]]).astype(F32)
    return tgt, nrm, src


@gpu
def test_full_loop_near_and_far_with_clutter(engine):
    prob, seg = _problem(2000, 2500, seed=9, clutter=600)
    _set(engine, prob)
    poses = np.concatenate([_near(prob, 4, 31), _far(prob, 8, 32)])
    refined, iters, energy = engine.tricp_plane(0, seg, poses, trim=0.5, ratio=0.99, max_iter=100)
    refs = [plane_ref(seg, prob.model_xyz, prob.model_nrm, P, trim=0.5, ratio=0.99, max_iter=100) for P in poses]
    _check(refined, iters, energy, refs)
    assert max(r["iters"] for r in refs) >= 5
    assert any(retry_reached(r["taus"]) for r in refs) or _cap_retry(engine)


def _cap_retry(engine):
    tgt, nrm, src = _cap_problem()
    prob = synth.make_segment_problem(500, 500, 0.005, seed=1)
    engine.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    engine.set_model(0, prob.model_xyz, prob.model_nrm, tgt, nrm)
    start = np.eye(4)[None]
    refined, iters, energy = engine.tricp_plane(0, src, start, trim=1.0, ratio=0.99, max_iter=100)
    ref = plane_ref(src, tgt, nrm, start[0], trim=1.0, ratio=0.99, max_iter=100)
    _check(refined, iters, energy, [ref], what="cap")
    return retry_reached(ref["taus"])


@gpu
@pytest.mark.parametrize("k", [0, 1, 74, 75, 150])
def test_batch_sizes(engine, k):
    prob, seg = _problem(2000, 1500, seed=23, clutter=100)
    _set(engine, prob)
    poses = np.concatenate([_near(prob, k - k // 2, 7), _far(prob, k // 2, 8)]) if k else np.zeros((0, 4, 4))
    refined, iters, energy = engine.tricp_plane(0, seg, poses, trim=0.5, ratio=2.0, max_iter=1)
    assert refined.shape == (k, 4, 4)
    refs = [plane_ref(seg, prob.model_xyz, prob.model_nrm, P, trim=0.5, max_iter=1) for P in poses]
    _check(refined, iters, energy, refs, what=k)
    if k == 150:
        refined, iters, energy = engine.tricp_plane(0, seg, poses, trim=0.5, ratio=0.99, max_iter=30)
        for j in range(k):
            r1, i1, e1 = engine.tricp_plane(0, seg, poses[j:j + 1], trim=0.5, ratio=0.99, max_iter=30)
            assert np.array_equal(r1[0], refined[j]) and i1[0] == iters[j] and e1[0].tobytes() == energy[j].tobytes(), j


@gpu
def test_ties_at_the_trim_threshold(engine):
    """The lattice of tests/test_gpu_tricp.py with random unit normals: which tied correspondences are admitted shows in the
    point-to-plane energy and update."""
    tgt, src = _lattice_ties()
    nrm = np.random.default_rng(11).normal(size=tgt.shape).astype(F32)
    prob = synth.make_segment_problem(500, 500, 0.005, seed=1)
    engine.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    engine.set_model(0, tgt, nrm)
    ns = len(src)
    pose = np.eye(4)[None]
    d2, _ = nearest(src, tgt)
    small = int((d2 == F32(2.0 ** -12 / 64)).sum())
    assert 1000 < small < ns - 1000
    for nk in (small // 3, small - 1, small + 777, ns - 5):
        trim = float(F32((nk + 0.5) / ns))
        assert n_keep_of(trim, ns) == nk
        for max_iter in (1, 2, 100):
            refined, iters, energy = engine.tricp_plane(0, src, pose, trim=trim, ratio=0.99, max_iter=max_iter)
            ref = plane_ref(src, tgt, nrm, pose[0], trim=trim, ratio=0.99, max_iter=max_iter)
            _check(refined, iters, energy, [ref], what=(nk, max_iter))


@gpu
def test_degenerate_targets(engine):
    prob, seg = _problem(2000, 1500, seed=33, clutter=100)
    poses = np.concatenate([_near(prob, 3, 51), _far(prob, 2, 52)])
    # a planar model: rank 3, only the tilts and the normal offset move
    flat = prob.model_xyz.copy()
    flat[:, 2] = F32(0.01)
    up = np.tile(np.array([0, 0, 1], F32), (len(flat), 1))
    _set(engine, prob, flat, up)
    refined, iters, energy = engine.tricp_plane(0, seg, poses, trim=0.5, ratio=0.99, max_iter=100)
    refs = [plane_ref(seg, flat, up, P, trim=0.5, ratio=0.99, max_iter=100) for P in poses]
    _check(refined, iters, energy, refs, what="planar")
    for r in refs:
        assert all(rk == 3 for rk in r["ranks"]) and not np.array(r["xs"])[:, 2:5].any()
    # kept normals all zero: x = 0, the transform stays the fp32 start, and 0 / 0 stops the loop at iteration 2
    _set(engine, prob, prob.model_xyz, np.zeros_like(prob.model_xyz))
    refined, iters, energy = engine.tricp_plane(0, seg, poses, trim=0.5, ratio=0.99, max_iter=100)
    for k, P in enumerate(poses):
        M = np.eye(4)
        M[:3] = inv_pose(P)[:3].astype(F32)
        assert iters[k] == 2 and energy[k] == 0 and np.array_equal(refined[k], inv_pose(M)), k
    # 1e20 along the normal of target point 0 (where every overflowing query lands): the energy overflows fp32
    _set(engine, prob)
    far = poses.copy()
    far[1][:3, 3] += 1e20 * (far[1][:3, :3] @ prob.model_nrm[0].astype(np.float64))
    refined, iters, energy = engine.tricp_plane(0, seg, far, trim=0.5, ratio=0.99, max_iter=100)
    assert iters[1] == 1 and energy[1] == np.inf and np.array_equal(refined[1], far[1])
    ref = plane_ref(seg, prob.model_xyz, prob.model_nrm, far[1])
    assert ref["iters"] == 1 and ref["energy"] == np.inf
    alone, it0, en0 = engine.tricp_plane(0, seg, far[[0, 2, 3, 4]], trim=0.5, ratio=0.99, max_iter=100)
    assert np.array_equal(alone, refined[[0, 2, 3, 4]]) and np.array_equal(it0, iters[[0, 2, 3, 4]])


def _raw(engine, fn, seg, poses, obj=0, trim=0.5, ratio=0.99, max_iter=100):
    seg = np.ascontiguousarray(seg, F32)
    P = np.ascontiguousarray(poses, np.float64).reshape(-1, 16).copy()
    it, en = np.zeros(len(P), np.int32), np.zeros(len(P), F32)
    rc = getattr(engine._lib, fn)(engine._ctx, obj, seg.ctypes.data, len(seg), P.ctypes.data, len(P), float(trim), float(ratio),
                                  int(max_iter), it.ctypes.data, en.ctypes.data)
    return rc, P.reshape(-1, 4, 4), it, en


@gpu
def test_refusals(engine):
    prob, seg = _problem(2000, 1500, seed=37, clutter=50)
    _set(engine, prob)
    poses = _near(prob, 4, 61)
    for bad in (np.nan, np.inf, -np.inf):
        P = poses.copy()
        P[1][1, 3] = bad
        rc, out = _raw(engine, "pgp_tricp_plane", seg, P)[:2]
        assert rc == PGP_E_INVALID and np.array_equal(out, P, equal_nan=True), bad
        S = seg.copy()
        S[777, 1] = bad
        rc, out = _raw(engine, "pgp_tricp_plane", S, poses)[:2]
        assert rc == PGP_E_INVALID and np.array_equal(out, poses), bad
    for trim, ratio in ((np.nan, 0.99), (0.5, np.nan), (0.0, 0.99), (-0.5, 0.99), (0.5, 0.0), (0.5, -1.0)):
        rc, out = _raw(engine, "pgp_tricp_plane", seg, poses, trim=trim, ratio=ratio)[:2]
        assert rc == PGP_E_INVALID and np.array_equal(out, poses), (trim, ratio)
    rc, out = _raw(engine, "pgp_tricp_plane", seg, poses, obj=7)[:2]
    assert rc == PGP_E_NO_MODEL and np.array_equal(out, poses)
    sx = np.ascontiguousarray(prob.model_xyz, F32)
    sn = np.ascontiguousarray(prob.model_nrm, F32)
    assert engine._lib.pgp_set_model(engine._ctx, 1, sx.ctypes.data, sn.ctypes.data, len(sx), sx.ctypes.data, None, len(sx)) == 0
    rc, out = _raw(engine, "pgp_tricp_plane", seg, poses, obj=1)[:2]
    assert rc == PGP_E_INVALID and np.array_equal(out, poses)
    rc, out = _raw(engine, "pgp_tricp", seg, poses, obj=1)[:2]     # the point-to-point fit needs no normals
    assert rc == 0


@gpu
def test_shared_scratch_leaves_tricp_unchanged(engine):
    prob, seg = _problem(2000, 2500, seed=9, clutter=600)
    _set(engine, prob)
    poses = np.concatenate([_near(prob, 6, 81), _far(prob, 6, 82)])
    before = engine.tricp(0, seg, poses, trim=0.5, ratio=0.99, max_iter=100)
    engine.tricp_plane(0, seg[:1700], np.concatenate([poses, poses]), trim=0.7, ratio=0.99, max_iter=100)
    after = engine.tricp(0, seg, poses, trim=0.5, ratio=0.99, max_iter=100)
    assert all(a.tobytes() == b.tobytes() for a, b in zip(before, after))
    refs = [tricp_ref(seg, prob.model_xyz, P, trim=0.5, ratio=0.99, max_iter=100) for P in poses[:2]]
    assert [r["iters"] for r in refs] == list(before[1][:2])
