"""K5 (trimmed ICP, `pgp_tricp` / `pgp_mcts_tricp`) and K6 (explained-point removal) against plain numpy restatements.

`tricp_ref` states the kernel's documented semantics stage by stage, in float64 where the kernel uses double and in fp32 where it
uses fp32, independently of the C restatement `lo_tricp`:
  start transform  T0 = fp32 of the double inverse of the pose ([R t]^-1 = [R^T, -R^T t]);
  query            ((T0 x + T1 y) + T2 z) + T3 per row, fp32, not fused;
  distance         d2 = (dx^2 + dy^2) + dz^2, fp32 left to right;
  nearest          exact, by brute force, ties to the smaller index of the VALIDATION cloud; a query with no d2 below FLT_MAX
                   (NaN or overflow) gets target 0 at FLT_MAX;
  trim             n_keep = min(ns, (int)|fp32(trim) * fp32(ns)|), tau = the n_keep-th smallest d2, the values equal to tau
                   admitted in the Morton order the host uploads the source in (key restated below);
  sums / fit       the 16 sums in double, the rigid fit by SVD (Umeyama without scale, proper rotation) in float64, cast to fp32;
  stop             energy / old_energy < ratio && it < max(1, max_iter) in fp32, old_energy starting at FLT_MAX;
  result           pose = double inverse of the fp32 transform; a pose whose energy is not finite is returned as given;
                   n_keep < 3 leaves the pose as given with iters = 0, energy = 0.
With the SVD and Horn's eigenvector agreeing to ~1e-15, the fp32 transforms of kernel and reference agree bit for bit almost
always, so the device trajectory is compared tightly: iteration counts equal, energies within 1 fp32 ulp (only the order of the
double sums differs), poses within 1e-6."""
import math

import numpy as np
import pytest

from physimglobalpose_b200 import synth

F32 = np.float32
FMAX = F32(np.finfo(np.float32).max)
PGP_E_INVALID = -1
gpu = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------------------ the reference
def inv_pose(P):
    """k5_tricp.cu::invert_pose in double, the same association."""
    P = np.asarray(P, np.float64).reshape(16)
    out = np.zeros((4, 4))
    for r in range(3):
        for c in range(3):
            out[r, c] = P[4 * c + r]
        out[r, 3] = -((P[r] * P[3] + P[4 + r] * P[7]) + P[8 + r] * P[11])
    out[3, 3] = 1.0
    return out


def _spread(v):
    x = v.astype(np.uint64) & np.uint64(0x1FFFFF)
    for sh, m in ((32, 0x1F00000000FFFF), (16, 0x1F0000FF0000FF), (8, 0x100F00F00F00F00F), (4, 0x10C30C30C30C30C3), (2, 0x1249249249249249)):
        x = (x | (x << np.uint64(sh))) & np.uint64(m)
    return x


def morton_order(seg):
    """The host's upload order of the source: 30-bit Morton key of the fp32 position in the segment's bounding cube, ties by index."""
    seg = np.asarray(seg, F32)
    lo, hi = seg.min(0), seg.max(0)
    e = hi - lo
    ext = max(max(e[0], e[1]), max(e[2], F32(1e-12)))
    key = np.zeros(len(seg), np.uint64)
    for c in range(3):
        u = (seg[:, c] - lo[c]) / ext
        q = np.minimum(F32(1023.0), np.maximum(F32(0.0), u * F32(1024.0))).astype(np.uint32)
        key |= _spread(q) << np.uint64(c)
    return np.lexsort((np.arange(len(seg)), key))


def query(T, src):
    return np.stack([((T[r, 0] * src[:, 0] + T[r, 1] * src[:, 1]) + T[r, 2] * src[:, 2]) + T[r, 3] for r in range(3)], axis=1)


def nearest(q, tgt):
    """Exact fp32 nearest neighbour by brute force (ties: smaller target index); no d2 below FLT_MAX -> (FLT_MAX, 0)."""
    q, tgt = np.asarray(q, F32), np.asarray(tgt, F32)
    d2 = np.empty(len(q), F32)
    nn = np.empty(len(q), np.int64)
    step = max(1, (1 << 22) // len(tgt))
    with np.errstate(all="ignore"):
        for a in range(0, len(q), step):
            qq = q[a:a + step]
            dx, dy, dz = (qq[:, None, c] - tgt[None, :, c] for c in range(3))
            d = (dx * dx + dy * dy) + dz * dz
            d[np.isnan(d)] = np.inf
            j = d.argmin(1)
            v = d[np.arange(len(qq)), j]
            miss = ~(v < FMAX)
            j[miss], v[miss] = 0, FMAX
            d2[a:a + step], nn[a:a + step] = v, j
    return d2, nn


def n_keep_of(trim, ns):
    kf = abs(F32(trim) * F32(ns))
    return min(ns, int(kf)) if kf < 2.0 ** 31 else ns


def rigid_fit(n, Ss, Sg, Ssg):
    """R, t minimising sum |R s + t - g|^2 from the sums (SVD, proper rotation), float64."""
    cs, cg = Ss / n, Sg / n
    H = Ssg - n * np.outer(cs, cg)
    U, _, Vt = np.linalg.svd(H)
    D = np.diag([1.0, 1.0, -1.0 if np.linalg.det(Vt.T @ U.T) < 0 else 1.0])
    R = Vt.T @ D @ U.T
    return R, cg - R @ cs


def tricp_ref(seg, tgt, pose, trim=0.5, ratio=0.99, max_iter=100):
    """One pose.  Returns dict(pose, iters, energy, taus, energies, pairs (kept source / target of the last iteration), R, t)."""
    seg, tgt = np.asarray(seg, F32).reshape(-1, 3), np.asarray(tgt, F32).reshape(-1, 3)
    pose = np.asarray(pose, np.float64).reshape(4, 4)
    ns = len(seg)
    n_keep = n_keep_of(trim, ns)
    out = dict(pose=pose.copy(), iters=0, energy=F32(0), taus=[], energies=[], unique=[], pairs=None, R=None, t=None)
    if n_keep < 3:
        return out
    src = seg[morton_order(seg)]
    pos = np.arange(ns)
    T = inv_pose(pose)[:3].astype(F32)
    energy, it = FMAX, 0
    while True:
        d2, nn = nearest(query(T, src), tgt)
        kept = np.lexsort((pos, d2))[:n_keep]
        s, g = src[kept].astype(np.float64), tgt[nn[kept]].astype(np.float64)
        with np.errstate(over="ignore"):
            old, energy = energy, F32(np.sum(d2[kept].astype(np.float64)))
        out["taus"].append(d2[kept[-1]])
        out["energies"].append(energy)
        out["pairs"] = (s, g)
        it += 1
        if energy <= FMAX:
            R, t = rigid_fit(float(n_keep), s.sum(0), g.sum(0), s.T @ g)
            out["R"], out["t"] = R, t
            sv = np.linalg.svd(s.T @ g - n_keep * np.outer(s.mean(0), g.mean(0)), compute_uv=False)
            # rank >= 2 (far above the rounding of the sums): one best proper rotation
            out["unique"].append(bool(sv[1] > 1e-9 * n_keep * np.abs(s).max() * np.abs(g).max()))
            T = np.concatenate([R, t[:, None]], axis=1).astype(F32)
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


def retry_reached(taus):
    """True when the kernel's capped search must be redone uncapped: tau_{i+1} >= fp32(max(4 tau_i, 1e-12))."""
    return any(b >= max(F32(4.0) * a, F32(1e-12)) for a, b in zip(taus, taus[1:]))


# ------------------------------------------------------------------------------------------------------------ problems
def _problem(n_model=2000, n_seg=1500, seed=9, clutter=0):
    prob = synth.make_segment_problem(n_model, n_seg, 0.005, seed=seed)
    seg = prob.scene_xyz
    if clutter:
        rng = np.random.default_rng(seed + 100)
        d = rng.normal(size=(clutter, 3))
        d /= np.linalg.norm(d, axis=1, keepdims=True)
        centre = prob.gt_pose[:3, 3]
        # 0.3-1 m from the model's surface: the box's half-diagonal is ~0.14 m
        seg = np.concatenate([seg, (centre + d * rng.uniform(0.45, 1.15, size=(clutter, 1))).astype(F32)])
    return prob, np.ascontiguousarray(seg, F32)


def _starts(prob, n, seed, ang=(0.0, 0.08), trans=0.006):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        P = prob.gt_pose.copy()
        a = rng.uniform(*ang) if ang[0] > 0 else rng.normal(0, ang[1])
        P[:3, :3] = P[:3, :3] @ synth.rot_axis_angle(rng.normal(size=3), a)
        off = rng.normal(size=3)
        P[:3, 3] += off / np.linalg.norm(off) * (rng.uniform(*trans) if isinstance(trans, tuple) else rng.normal(0, trans))
        out.append(P)
    return np.array(out).reshape(-1, 4, 4)


def _near(prob, n, seed):
    return _starts(prob, n, seed)


def _far(prob, n, seed):
    """20-40 degrees and 3-8 cm from the ground truth."""
    return _starts(prob, n, seed, ang=(math.radians(20), math.radians(40)), trans=(0.03, 0.08))


def _set(engine, prob, val=None):
    engine.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    if val is None:
        engine.set_model(0, prob.model_xyz, prob.model_nrm)
    else:
        engine.set_model(0, prob.model_xyz, prob.model_nrm, val, np.zeros_like(val))


def _ulp_close(a, b, ulps=1):
    a, b = F32(a), F32(b)
    if a == b:
        return True
    return bool(np.isfinite(a) and np.isfinite(b) and abs(float(a) - float(b)) <= ulps * float(np.spacing(max(abs(a), abs(b)))))


def _objective(pairs, R, t):
    s, g = pairs
    return float(np.sum((s @ R.T + t - g) ** 2))


def _check_fit(pose, ref, what=""):
    """For a fit whose rotation is not unique: a finite proper rotation that reaches the least-squares minimum of the kept pairs
    (the objective to 1e-9 relative, evaluated with the rotation nearest to the fp32 matrix, plus the fp32 rounding of the
    transform when the minimum is 0)."""
    T = inv_pose(pose)                                          # the device's fp32 transform, in double
    R, t = T[:3, :3], T[:3, 3]
    assert np.all(np.isfinite(T)), what
    assert np.abs(R.T @ R - np.eye(3)).max() <= 1e-6 and abs(np.linalg.det(R) - 1.0) <= 1e-6, (what, R)
    U, _, Vt = np.linalg.svd(R)                                 # undo the fp32 rounding's scaling: nearest rotation
    want = _objective(ref["pairs"], ref["R"], ref["t"])
    got = _objective(ref["pairs"], U @ Vt, t)
    assert abs(got - want) <= 1e-9 * want + len(ref["pairs"][0]) * 1e-12, (what, got, want)


def _check(refined, iters, energy, refs, pose_tol=1e-6, what=""):
    """Iteration counts, energies to 1 ulp, poses to pose_tol.  A rotation the kept pairs leave free is compared through the
    objective when it is the last fit; when it is not, what follows depends on the free rotation and only the count is compared."""
    for k, r in enumerate(refs):
        assert iters[k] == r["iters"], (what, k, iters[k], r["iters"])
        if not all(r["unique"][:-1]):
            continue
        assert _ulp_close(energy[k], r["energy"]), (what, k, float(energy[k]), float(r["energy"]))
        if not all(r["unique"]):
            _check_fit(refined[k], r, what=(what, k))
            continue
        err = np.abs(refined[k] - r["pose"]).max()
        assert err <= pose_tol, (what, k, err, iters[k])


def _check_loop(refined, iters, energy, refs, what=""):
    for k, r in enumerate(refs):
        assert iters[k] == r["iters"], (what, k, iters[k], r["iters"])
        assert _ulp_close(energy[k], r["energy"]), (what, k, float(energy[k]), float(r["energy"]))
        assert all(r["unique"]), (what, k)
        dt = np.linalg.norm(refined[k][:3, 3] - r["pose"][:3, 3])
        ang = np.linalg.norm(refined[k][:3, :3] - r["pose"][:3, :3]) / math.sqrt(2.0)    # small angle: |R_a - R_b|_F = sqrt(2) angle
        assert dt <= 1e-6 and ang <= 1e-6, (what, k, dt, ang)


# ------------------------------------------------------------------------------------------------------------ CPU: pin the reference
@pytest.mark.parametrize("seed", [3, 4, 5])
@pytest.mark.parametrize("trim", [0.5, 0.9])
def test_reference_equals_lo_tricp(port_lib, seed, trim):
    """The numpy reference walks the same iterations to the same transform as the C restatement lo_tricp (the problems of
    test_tricp_crosscheck.py), so it is pinned without a GPU."""
    prob = synth.make_segment_problem(800, 600, 0.005, seed=seed)
    rng = np.random.default_rng(seed)
    pose = prob.gt_pose.copy()
    pose[:3, :3] = pose[:3, :3] @ synth.rot_axis_angle(rng.normal(size=3), 0.06)
    pose[:3, 3] += rng.normal(0, 0.004, size=3)
    ref = tricp_ref(prob.scene_xyz, prob.model_xyz, pose, trim=trim)
    o = port_lib.PortOracle(prob.scene_xyz, prob.scene_nrm, prob.model_xyz, prob.model_nrm, prob.model_xyz, prob.model_nrm, prob.delta)
    T_c, it_c, e_c = o.tricp(prob.scene_xyz, prob.model_xyz, inv_pose(pose)[:3].astype(F32), trim=trim, ratio=0.99, max_iter=100)
    assert it_c == ref["iters"] >= 2
    assert abs(e_c - ref["energy"]) <= 1e-6 * ref["energy"]
    assert np.abs(T_c - inv_pose(ref["pose"])[:3]).max() <= 1e-6


def test_reference_primitives():
    """Morton key, nearest-neighbour ties and overflow, n_keep and the pose inverse, on hand-made inputs."""
    seg = np.array([[1, 1, 1], [0, 0, 0], [1, 0, 0], [0, 1, 0]], F32)
    assert list(morton_order(seg)) == [1, 2, 3, 0]              # keys 0, 1, 2, 7 (x is the lowest bit)
    tgt = np.array([[1, 0, 0], [-1, 0, 0], [0, 0, 0]], F32)
    d2, nn = nearest(np.array([[0, 0, 0], [0.5, 0, 0], [0, 0, 0]], F32), tgt[:2])
    assert list(nn) == [0, 0, 0] and list(d2) == [1.0, 0.25, 1.0]   # tie -> smaller index
    d2, nn = nearest(np.array([[1e20, 0, 0], [np.nan, 0, 0], [np.inf, 0, 0]], F32), tgt)
    assert list(nn) == [0, 0, 0] and np.all(d2 == FMAX)
    assert n_keep_of(0.5, 1001) == 500 and n_keep_of(1.5, 7) == 7 and n_keep_of(np.inf, 7) == 7
    P = np.eye(4)
    P[:3, :3] = synth.rot_axis_angle([1, 2, 3], 0.4)
    P[:3, 3] = [0.1, -0.2, 0.7]
    assert np.allclose(inv_pose(P), np.linalg.inv(P), atol=1e-15)


def test_lo_tricp_survives_an_overflowing_pose(port_lib):
    """A translation of 1e20 overflows every squared distance: lo_tricp takes target 0 at FLT_MAX (it used to read tgt[-3]),
    stops after one iteration with energy +Inf and leaves the transform as given -- the same as K5 and the reference."""
    prob = synth.make_segment_problem(800, 600, 0.005, seed=3)
    pose = prob.gt_pose.copy()
    pose[:3, 3] += 1e20
    T0 = inv_pose(pose)[:3].astype(F32)
    o = port_lib.PortOracle(prob.scene_xyz, prob.scene_nrm, prob.model_xyz, prob.model_nrm, prob.model_xyz, prob.model_nrm, prob.delta)
    T, it, e = o.tricp(prob.scene_xyz, prob.model_xyz, T0, trim=0.5, ratio=0.99, max_iter=100)
    assert it == 1 and e == np.inf and np.array_equal(T, T0)
    ref = tricp_ref(prob.scene_xyz, prob.model_xyz, pose)
    assert ref["iters"] == 1 and ref["energy"] == np.inf and np.array_equal(ref["pose"], pose)


# ------------------------------------------------------------------------------------------------------------ GPU: K5
def _trim_for(spec, ns):
    if spec == "keep2":
        t = F32(2.5 / ns)
    elif spec == "keep3":
        t = F32(3.5 / ns)
    else:
        return float(spec)
    return float(t)


@gpu
@pytest.mark.parametrize("ns", [3, 4, 5, 1023, 1024, 2047, 2048, 2049, 4097, 20000])
def test_one_and_two_iterations(engine, ns):
    """max_iter 1 and 2 (and 0, which behaves like 1) over segment sizes around the 1024-thread chunk and the two-CTA split,
    and trims keeping 2 (early return), 3, half, all and 'more than all' of the points."""
    prob, seg = _problem(2000, max(ns, 600), seed=21, clutter=0)
    rng = np.random.default_rng(ns)
    seg = seg[rng.permutation(len(seg))[:ns]] if ns < len(seg) else seg
    seg = np.ascontiguousarray(seg[:ns], F32)
    _set(engine, prob)
    poses = np.concatenate([_near(prob, 2, ns), _far(prob, 1, ns + 1)])
    for spec in ("keep2", "keep3", 0.5, 1.0, 1.5):
        trim = _trim_for(spec, ns)
        nk = n_keep_of(trim, ns)
        assert nk == {"keep2": 2, "keep3": 3}.get(spec, nk)
        for max_iter in (0, 1, 2):
            refined, iters, energy = engine.tricp(0, seg, poses, trim=trim, ratio=2.0, max_iter=max_iter)
            refs = [tricp_ref(seg, prob.model_xyz, P, trim=trim, ratio=2.0, max_iter=max_iter) for P in poses]
            _check(refined, iters, energy, refs, what=(ns, spec, max_iter))
            assert all(all(r["unique"]) for r in refs[:2]), (ns, spec)        # the near starts are compared matrix for matrix
            if nk < 3:
                assert np.array_equal(refined, poses) and not iters.any() and not energy.any()
            else:
                assert np.all(iters == max(1, max_iter))


@gpu
@pytest.mark.parametrize("k", [0, 1, 74, 75, 150])
def test_batch_sizes(engine, k):
    """More clusters than fit one wave on 148 SMs; k = 0 is a no-op."""
    prob, seg = _problem(2000, 1500, seed=23, clutter=100)
    _set(engine, prob)
    poses = np.concatenate([_near(prob, k - k // 2, 7), _far(prob, k // 2, 8)]) if k else np.zeros((0, 4, 4))
    refined, iters, energy = engine.tricp(0, seg, poses, trim=0.5, ratio=2.0, max_iter=1)
    assert refined.shape == (k, 4, 4)
    refs = [tricp_ref(seg, prob.model_xyz, P, trim=0.5, max_iter=1) for P in poses]
    _check(refined, iters, energy, refs, what=k)


@gpu
def test_full_loop_near_and_far_with_clutter(engine):
    """Whole refinements from near and from 20-40 degree / several-cm starts with clutter 0.3-1 m from the model: same iteration
    counts, same final poses, same energies.  At least one trajectory more than quadruples the squared trim radius between two
    iterations, which is exactly when the kernel's capped search must be redone without the cap."""
    prob, seg = _problem(2000, 2500, seed=9, clutter=600)
    _set(engine, prob)
    poses = np.concatenate([_near(prob, 4, 31), _far(prob, 8, 32)])
    refined, iters, energy = engine.tricp(0, seg, poses, trim=0.5, ratio=0.99, max_iter=100)
    refs = [tricp_ref(seg, prob.model_xyz, P, trim=0.5, ratio=0.99, max_iter=100) for P in poses]
    _check_loop(refined, iters, energy, refs)
    assert max(r["iters"] for r in refs) >= 20
    # These starts shrink the trim radius steadily.  A start the cap cuts into: a 2.5 cm patch of one face turned by 0.01 rad
    # about its centre, and one exact point 8 cm away.  The fit follows the patch and swings the lone point out by ~0.7 mm, so
    # with trim = 1 the squared trim radius grows ~7x from the first iteration to the second.
    tgt = synth.make_segment_problem(20000, 10, 0.005, seed=12).model_xyz
    face = tgt[tgt[:, 2] == tgt[:, 2].max()]
    c = face[np.argmin(np.abs(face[:, 0] + 0.035) + np.abs(face[:, 1]))]
    lone = face[np.argmin(np.abs(face[:, 0] - 0.045) + np.abs(face[:, 1]))]
    patch = face[np.linalg.norm(face[:, :2] - c[:2], axis=1) < 0.025]
    src = np.concatenate([(patch - c) @ synth.rot_axis_angle([0, 1, 0], 0.01).T + c, lone[None]]).astype(F32)
    engine.set_model(0, prob.model_xyz, prob.model_nrm, tgt, np.zeros_like(tgt))
    start = np.stack([np.eye(4), _near(prob, 1, 5)[0] @ np.linalg.inv(prob.gt_pose)])
    refined, iters, energy = engine.tricp(0, src, start, trim=1.0, ratio=0.99, max_iter=100)
    refs = [tricp_ref(src, tgt, P, trim=1.0, ratio=0.99, max_iter=100) for P in start]
    _check_loop(refined, iters, energy, refs, what="cap")
    assert retry_reached(refs[0]["taus"]), refs[0]["taus"]


@gpu
def test_batch_independence(engine):
    """Every pose of a 150-pose batch is bit-identical to the same pose refined alone."""
    prob, seg = _problem(1500, 1800, seed=29, clutter=200)
    _set(engine, prob)
    poses = np.concatenate([_near(prob, 75, 41), _far(prob, 75, 42)])
    refined, iters, energy = engine.tricp(0, seg, poses, trim=0.5, ratio=0.99, max_iter=30)
    for k in range(len(poses)):
        r1, i1, e1 = engine.tricp(0, seg, poses[k:k + 1], trim=0.5, ratio=0.99, max_iter=30)
        assert np.array_equal(r1[0], refined[k]) and i1[0] == iters[k] and e1[0].tobytes() == energy[k].tobytes(), k


def _lattice_ties(n_side=(24, 24, 12), h=2.0 ** -6, seed=5):
    """Target: a dyadic lattice (exact in fp32, mirror-symmetric).  Source: lattice points moved by +-h/4 or +-h/8 along one
    axis, some of them twice, some mirrored through the lattice centre: every squared distance is h^2/16 or h^2/64 exactly,
    so thousands of DIFFERENT correspondences tie at each value."""
    rng = np.random.default_rng(seed)
    ax = [np.arange(n, dtype=np.float64) * h for n in n_side]
    tgt = np.stack(np.meshgrid(*ax, indexing="ij"), -1).reshape(-1, 3)
    inner = tgt[(tgt[:, 0] > 0) & (tgt[:, 1] > 0) & (tgt[:, 2] > 0) & (tgt[:, 0] < ax[0][-1]) & (tgt[:, 1] < ax[1][-1]) & (tgt[:, 2] < ax[2][-1])]
    pick = inner[rng.permutation(len(inner))[:3000]]
    off = np.zeros_like(pick)
    off[np.arange(len(pick)), rng.integers(0, 3, len(pick))] = rng.choice([-h / 4, h / 4, -h / 8, h / 8], len(pick))
    src = pick + off
    centre = np.array([a[-1] / 2 for a in ax])
    src = np.concatenate([src, src[:1200], 2 * centre - src[1200:2400]])          # duplicated, mirrored
    return tgt.astype(F32), src[rng.permutation(len(src))].astype(F32)


@gpu
def test_ties_at_the_trim_threshold(engine):
    """ns = 5400 > 4096: the tie sets span both CTAs of the cluster and several 1024-point chunks of each.  n_keep falls inside
    the h^2/64 and inside the h^2/16 group; which of the tied correspondences are admitted (the first in Morton order) moves
    the fit's centroids, so a wrong admission order shows in the transform."""
    tgt, src = _lattice_ties()
    prob = synth.make_segment_problem(500, 500, 0.005, seed=1)
    engine.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    engine.set_model(0, tgt, np.zeros_like(tgt))
    ns = len(src)
    assert ns > 4096
    pose = np.eye(4)[None]
    d2, _ = nearest(src, tgt)
    small = int((d2 == F32(2.0 ** -12 / 64)).sum())
    assert 1000 < small < ns - 1000
    for nk in (small // 3, small - 1, small + 777, ns - 5):
        trim = float(F32((nk + 0.5) / ns))
        assert n_keep_of(trim, ns) == nk
        for max_iter in (1, 2, 100):
            refined, iters, energy = engine.tricp(0, src, pose, trim=trim, ratio=0.99, max_iter=max_iter)
            ref = tricp_ref(src, tgt, pose[0], trim=trim, ratio=0.99, max_iter=max_iter)
            _check(refined, iters, energy, [ref], what=(nk, max_iter))


def _host_would_fallback(engine, pairs):
    """Horn's 4x4 matrix of the kept pairs; the host copy of max_eigvec4 returns 0 exactly when the device takes Jacobi."""
    import ctypes as C
    s, g = pairs
    n = float(len(s))
    H = s.T @ g - n * np.outer(s.mean(0), g.mean(0))
    (Sxx, Sxy, Sxz), (Syx, Syy, Syz), (Szx, Szy, Szz) = H
    N = np.array([[Sxx + Syy + Szz, Syz - Szy, Szx - Sxz, Sxy - Syx], [Syz - Szy, Sxx - Syy - Szz, Sxy + Syx, Szx + Sxz],
                  [Szx - Sxz, Sxy + Syx, -Sxx + Syy - Szz, Syz + Szy], [Sxy - Syx, Szx + Sxz, Syz + Szy, -Sxx - Syy + Szz]])
    q = np.zeros(4)
    f = engine._lib.pgp_host_max_eigvec4
    f.restype, f.argtypes = C.c_int, [C.c_void_p, C.c_void_p]
    return f(np.ascontiguousarray(N).ctypes.data, q.ctypes.data) == 0


@gpu
@pytest.mark.parametrize("case", ["collinear", "identical", "exact"])
def test_degenerate_fits(engine, case):
    """Kept correspondences that leave the rotation undetermined force the device's Jacobi fallback.  The rotation must come
    out finite and proper, and reach the least-squares minimum: where the rotation is not unique the objective is compared,
    not the matrix."""
    rng = np.random.default_rng(3)
    prob = synth.make_segment_problem(500, 500, 0.005, seed=1)
    engine.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    if case == "collinear":
        tgt = np.zeros((400, 3), F32)
        tgt[:, 0] = np.sort(rng.uniform(0, 0.3, 400))
        src = np.zeros((300, 3), F32)
        src[:, 0] = rng.uniform(0.01, 0.29, 300)
        src[:, 1] = 0.004                                       # a parallel line: every correspondence lies in one direction
        pose, trim, max_iter = np.eye(4), 1.0, 1
    elif case == "identical":
        # dyadic, so every sum is exact and the cross-covariance is exactly 0: Horn's matrix is 0
        p = np.array([2.0 ** -6, 2.0 ** -5, -(2.0 ** -5)])
        tgt = np.concatenate([prob.model_xyz, (p + [2.0 ** -8, 0, 0])[None]]).astype(F32)
        src = np.tile(p.astype(F32), (700, 1))
        pose, trim, max_iter = np.eye(4), 0.5, 1
    else:
        tgt = prob.model_xyz
        src = tgt[rng.permutation(len(tgt))[:300]]
        pose, trim, max_iter = np.eye(4), 0.6, 100
    engine.set_model(0, prob.model_xyz, prob.model_nrm, tgt, np.zeros_like(tgt))
    refined, iters, energy = engine.tricp(0, src, pose[None], trim=trim, ratio=0.99, max_iter=max_iter)
    ref = tricp_ref(src, tgt, pose, trim=trim, ratio=0.99, max_iter=max_iter)
    assert iters[0] == ref["iters"] and _ulp_close(energy[0], ref["energy"])
    if case == "exact":
        assert all(ref["unique"])
    else:
        assert not ref["unique"][-1]
    _check_fit(refined[0], ref, what=case)
    if case == "exact":
        assert ref["iters"] == 2 and energy[0] == 0.0             # 0 / FLT_MAX continues, 0 / 0 stops
        assert np.abs(refined[0] - np.eye(4)).max() <= 1e-6
    else:
        assert _host_would_fallback(engine, ref["pairs"])


@gpu
@pytest.mark.parametrize("shape", ["planar", "one_point", "far_outlier", "val_differs", "reloaded"])
def test_target_grid_shapes(engine, shape):
    """Target grids of one cell layer, one cell, 96 cells with nearly every point in one of them, a validation cloud that
    differs from the search cloud, and a slot refilled after a refinement (its grid must be rebuilt)."""
    prob, seg = _problem(2000, 1500, seed=33, clutter=100)
    engine.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    rng = np.random.default_rng(4)
    tgt = prob.model_xyz
    max_iter = 100
    if shape == "planar":
        tgt = tgt.copy()
        tgt[:, 2] = F32(0.01)
    elif shape == "one_point":
        tgt = tgt[:1].copy()                                    # every correspondence the same point: the rotation is free
        max_iter = 1
    elif shape == "far_outlier":
        big = synth.make_segment_problem(110_000, 10, 0.005, seed=2).model_xyz      # > 107 171 points: 96 cells
        tgt = np.concatenate([big, np.array([[10.0, 0.0, 0.0]], F32)])
        max_iter = 3
    elif shape == "val_differs":
        tgt = (prob.model_xyz + rng.normal(0, 0.002, prob.model_xyz.shape)).astype(F32)
    if shape == "reloaded":
        engine.set_model(0, prob.model_xyz[::-1].copy() * F32(1.5), prob.model_nrm)
        engine.tricp(0, seg, _near(prob, 2, 1), trim=0.5)
        engine.set_model(0, prob.model_xyz, prob.model_nrm)
    else:
        engine.set_model(0, prob.model_xyz, prob.model_nrm, tgt, np.zeros_like(tgt))
    poses = np.concatenate([_near(prob, 3, 51), _far(prob, 3, 52)])
    refined, iters, energy = engine.tricp(0, seg, poses, trim=0.5, ratio=0.99, max_iter=max_iter)
    refs = [tricp_ref(seg, tgt, P, trim=0.5, ratio=0.99, max_iter=max_iter) for P in poses]
    if shape == "one_point":
        _check(refined, iters, energy, refs, what=shape)
        assert not any(r["unique"][0] for r in refs)
    else:
        _check_loop(refined, iters, energy, refs, what=shape)


def _grid_of(tgt):
    """k5_tricp.cu::build_target_grid in fp32: lo, g, inv_g, dim."""
    tgt = np.asarray(tgt, F32)
    lo, hi = tgt.min(0), tgt.max(0)
    ext = max(F32(hi[k] - lo[k]) for k in range(3))
    cells = max(1, min(96, math.ceil(2.0 * np.cbrt(float(len(tgt))))))
    g = max(F32(ext / F32(cells)), F32(1e-6))
    inv_g = F32(F32(1.0) / g)
    dim = [max(1, int(np.floor(F32(F32(hi[k] - lo[k]) * inv_g))) + 1) for k in range(3)]
    return lo, g, inv_g, dim


def _cell_face_problem():
    """A 97 x 97 x 12 lattice on the cell faces lo + j g of a 96-cell grid (non-dyadic lo and g, so the fp32 cell coordinate
    fl(fl(x - lo) * inv_g) is rounded), and far above it, for every face j, a query q whose x cell is j - 1 and a point P just
    across face j + 1 -- two cells away -- at x distance d_P within 2e-5 of a cell of g, plus a point B in the neighbouring
    y cell slightly FARTHER than P (1e-7 .. 1e-5 of a cell).  P is the nearest neighbour.  Where rounding puts q and P less
    than g apart, B is placed inside the stop bound (r - 1) g * (1 - 5e-7) of ring 2 taken without the rounding of the cell
    coordinate: a search with that bound accepts B after ring 1.  (y is near 0 so that B's offset can be set finely.)"""
    g0 = F32(0.0104173)
    lo0 = np.array([0.3137, -0.4862, 0.1171], F32)
    faces = [(lo0[k] + np.arange(97, dtype=F32) * g0).astype(F32) for k in range(3)]
    X, Y, Z = np.meshgrid(faces[0], faces[1], faces[2][:12], indexing="ij")
    lattice = np.stack([X, Y, Z], -1).reshape(-1, 3)
    lo, g, inv_g, dim = _grid_of(lattice)
    assert dim[0] == 97 and len(lattice) > 107_171

    def cell(x, k):
        return int(np.floor(F32(F32(F32(x) - lo[k]) * inv_g)))

    def step(x, d):
        return np.nextafter(F32(x), F32(d * np.inf)).astype(F32)

    b2_unslacked = F32(F32(g * g) * F32(0.999999))
    rng = np.random.default_rng(8)
    y0 = cell(F32(0.0), 1)
    slots = [(y0 + dy, zc) for dy in (0, 4, -4, 8, -8) for zc in range(20, 93, 4)]
    pairs = []
    for j in range(1, 95):
        xq = F32(lo[0] + F32(j) * g)                      # largest fp32 in x cell j - 1
        while cell(xq, 0) >= j:
            xq = step(xq, -1)
        while cell(step(xq, 1), 0) < j:
            xq = step(xq, 1)
        xp = F32(lo[0] + F32(j + 1) * g)                  # smallest fp32 in x cell j + 1
        while cell(xp, 0) < j + 1:
            xp = step(xp, 1)
        while cell(step(xp, -1), 0) >= j + 1:
            xp = step(xp, -1)
        dxp = F32(xq - xp)
        pairs.append((F32(dxp * dxp) >= b2_unslacked, j, xq, xp, dxp))
    src, extra, old_misses = [], [], 0
    for (yc, zc), (_, j, xq, xp, dxp) in zip(slots, sorted(pairs, key=lambda p: (p[0], p[1]))):
        yq = F32(lo[1] + (F32(yc) + F32(0.5)) * g)
        zq = F32(lo[2] + (F32(zc) + F32(0.5)) * g)
        d2p = F32(dxp * dxp)
        if d2p < b2_unslacked:
            yb = F32(yq + F32(np.sqrt(0.5 * (float(d2p) + float(b2_unslacked)))))
        else:
            yb = F32(yq + F32(float(-dxp) * (1 + 10.0 ** rng.uniform(-7, -5))))
        while F32(F32(yq - yb) ** 2) <= d2p:
            yb = step(yb, 1)
        d2b = F32(F32(yq - yb) ** 2)
        assert cell(yb, 1) == yc + 1 and cell(xp, 0) == j + 1 and cell(xq, 0) == j - 1 and cell(yq, 1) == yc
        old_misses += bool(d2b <= b2_unslacked)
        src.append([xq, yq, zq])
        extra += [[xp, yq, zq], [xq, yb, zq]]
    tgt = np.concatenate([lattice, np.array(extra, F32)])
    return tgt, np.array(src, F32), old_misses


@gpu
def test_cell_faces(engine):
    """Nearest neighbours just across a cell face, observed through the one-iteration energy and transform with trim = 1."""
    tgt, src, old_misses = _cell_face_problem()
    assert old_misses >= 3                                   # the construction does reach the rounding sliver
    prob = synth.make_segment_problem(500, 500, 0.005, seed=1)
    engine.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    engine.set_model(0, prob.model_xyz, prob.model_nrm, tgt, np.zeros_like(tgt))
    pose = np.eye(4)[None]
    _, nn = nearest(src, tgt)
    assert np.all(nn == len(tgt) - 2 * len(src) + 2 * np.arange(len(src)))     # P, not B, is the nearest point of every query
    refined, iters, energy = engine.tricp(0, src, pose, trim=1.0, ratio=0.99, max_iter=1)
    ref = tricp_ref(src, tgt, pose[0], trim=1.0, max_iter=1)
    _check(refined, iters, energy, [ref])


def _raw_tricp(engine, seg, poses, trim=0.5, ratio=0.99, max_iter=100):
    seg = np.ascontiguousarray(seg, F32)
    P = np.ascontiguousarray(poses, np.float64).reshape(-1, 16).copy()
    it, en = np.zeros(len(P), np.int32), np.zeros(len(P), F32)
    rc = engine._lib.pgp_tricp(engine._ctx, 0, seg.ctypes.data, len(seg), P.ctypes.data, len(P), float(trim), float(ratio), int(max_iter),
                               it.ctypes.data, en.ctypes.data)
    return rc, P.reshape(-1, 4, 4), it, en


def _raw_mcts(engine, seg, poses, trim=0.5, ratio=0.99):
    seg = np.ascontiguousarray(seg, F32)
    P = np.ascontiguousarray(poses, np.float64).reshape(-1, 16).copy()
    it, en = np.zeros(len(P), np.int32), np.zeros(len(P), F32)
    import ctypes as C
    nun = C.c_int(0)
    rc = engine._lib.pgp_mcts_tricp(engine._ctx, 0, seg.ctypes.data, len(seg), None, 0, 0.008, P.ctypes.data, len(P), float(trim), float(ratio),
                                    100, it.ctypes.data, en.ctypes.data, C.byref(nun))
    return rc, P.reshape(-1, 4, 4)


@gpu
def test_non_finite_and_overflowing_input(engine):
    """NaN / Inf in a pose or a segment point, and a NaN trim or ratio, are refused before anything runs; a finite pose whose
    queries overflow fp32 (translation 1e20) stops after one iteration with energy +Inf and is returned as given, and the
    other poses of its batch are bit-identical to a batch without it."""
    prob, seg = _problem(2000, 1500, seed=37, clutter=50)
    _set(engine, prob)
    poses = _near(prob, 4, 61)
    for bad in (np.nan, np.inf, -np.inf):
        for where in ((0, 0), (1, 3), (2, 2)):
            P = poses.copy()
            P[1][where] = bad
            for call in (_raw_tricp, _raw_mcts):
                rc, out = call(engine, seg, P)[:2]
                assert rc == PGP_E_INVALID and np.array_equal(out, P, equal_nan=True), (bad, where, call.__name__)
        S = seg.copy()
        S[777, 1] = bad
        for call in (_raw_tricp, _raw_mcts):
            rc, out = call(engine, S, poses)[:2]
            assert rc == PGP_E_INVALID and np.array_equal(out, poses)
    for trim, ratio in ((np.nan, 0.99), (0.5, np.nan), (0.0, 0.99), (0.5, -1.0)):
        for call in (_raw_tricp, _raw_mcts):
            rc, out = call(engine, seg, poses, trim=trim, ratio=ratio)[:2]
            assert rc == PGP_E_INVALID and np.array_equal(out, poses), (trim, ratio)
    far = poses.copy()
    far[2][:3, 3] += 1e20
    rc, out, it, en = _raw_tricp(engine, seg, far)
    rc0, out0, it0, en0 = _raw_tricp(engine, seg, poses[[0, 1, 3]])
    assert rc == 0 and rc0 == 0
    assert it[2] == 1 and en[2] == np.inf and np.array_equal(out[2], far[2])
    assert np.array_equal(out[[0, 1, 3]], out0) and np.array_equal(it[[0, 1, 3]], it0) and en[[0, 1, 3]].tobytes() == en0.tobytes()
    ref = tricp_ref(seg, prob.model_xyz, far[2])
    assert ref["iters"] == 1 and ref["energy"] == np.inf
    # trim = 1 with one source point at 1e20: its squared distance overflows, the energy does not (FLT_MAX + the rest rounds
    # to FLT_MAX), so one fit runs -- with target point 0 for that correspondence, and sums that the 1e20 coordinate has
    # cancelled to rounding noise -- and energy / old_energy = 1 stops.  Defined means: one iteration and a finite pose.
    S = seg.copy()
    S[5] = [1e20, 0.0, 0.0]
    refined, iters, energy = engine.tricp(0, S, poses[:2], trim=1.0, ratio=0.99, max_iter=100)
    refs = [tricp_ref(S, prob.model_xyz, P, trim=1.0) for P in poses[:2]]
    assert [r["iters"] for r in refs] == [1, 1] and all(r["energy"] == FMAX for r in refs)
    assert np.all(iters == 1) and np.all(energy == FMAX) and np.all(np.isfinite(refined))


# ------------------------------------------------------------------------------------------------------------ GPU: K6
def explained_ref(seg, model, placed, threshold):
    """pgp_remove_explained restated in fp32: the model placed at fp32(pose[:3]) row by row ((m0 x + m1 y) + m2 z) + m3, and a
    segment point is explained iff some placed point has (dx^2 + dy^2) + dz^2 < fl(threshold^2)."""
    seg, model = np.asarray(seg, F32), np.asarray(model, F32)
    r2 = F32(F32(threshold) * F32(threshold))
    flags = np.zeros(len(seg), bool)
    for P in np.asarray(placed, np.float64).reshape(-1, 4, 4):
        ex = query(P[:3].astype(F32), model)
        for a in range(0, len(seg), 512):
            s = seg[a:a + 512]
            dx, dy, dz = (s[:, None, c] - ex[None, :, c] for c in range(3))
            flags[a:a + 512] |= ((dx * dx + dy * dy) + dz * dz < r2).any(1)
    return flags


@gpu
@pytest.mark.parametrize("nv", [1, 255, 256, 257, 3000])
def test_explained_point_removal_bitwise(engine, nv):
    """Explained-cloud sizes around the 256-point tile, segments that are not a multiple of 256, up to 8 placed poses, threshold
    0 and the strict d2 < r^2 at exact equality."""
    rng = np.random.default_rng(nv)
    prob = synth.make_segment_problem(3000, 2000, 0.005, seed=43)
    engine.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    model = prob.model_xyz[rng.permutation(len(prob.model_xyz))[:nv]]
    engine.set_model(0, prob.model_xyz, prob.model_nrm, model, np.zeros_like(model))
    seg = prob.scene_xyz[:1999]
    for n_placed in (1, 2, 8):
        placed = np.concatenate([prob.gt_pose[None], _near(prob, n_placed - 1, n_placed)])
        placed[1:, :3, 3] += rng.normal(0, 0.03, (n_placed - 1, 3))
        for thr in (0.0, 0.004, 0.008, 0.02):
            got = engine.remove_explained(0, seg, placed, thr)
            want = explained_ref(seg, model, placed, thr)
            assert np.array_equal(got, want), (n_placed, thr, int((got != want).sum()))
            if thr == 0.0:
                assert not got.any()
    # exact equality with dyadic coordinates: distance 2^-7 along one axis is NOT explained at threshold 2^-7, 2^-7 - 2^-20 is
    h = 2.0 ** -7
    m0 = model[0].astype(np.float64)
    base = np.round(m0 * 2 ** 10) / 2 ** 10                  # dyadic, so every difference below is exact
    pose = np.eye(4)
    model1 = np.array([base], F32)
    engine.set_model(0, prob.model_xyz, prob.model_nrm, model1, np.zeros_like(model1))
    seg_eq = np.array([base + [h, 0, 0], base - [0, h, 0], base + [0, 0, h], base + [h - 2 ** -20, 0, 0], base + [0.0, 0.0, 0.0]], F32)
    got = engine.remove_explained(0, seg_eq, pose[None], h)
    assert list(got) == [False, False, False, True, True]
    assert np.array_equal(got, explained_ref(seg_eq, model1, pose[None], h))


@gpu
def test_mcts_tricp_when_everything_or_almost_everything_is_explained(engine):
    prob, seg = _problem(2000, 1200, seed=47)
    _set(engine, prob)
    cand = _near(prob, 3, 71)
    placed = prob.gt_pose[None]
    # a threshold that explains every segment point: nothing left to refine
    refined, iters, energy, n_un = engine.mcts_tricp(0, seg, placed, cand, 1.0, trim=0.5, ratio=0.99)
    assert n_un == 0 and not iters.any() and not energy.any() and np.array_equal(refined, cand)
    # exactly two points remain: n_keep < 3 leaves the poses as given
    far = np.array([[5.0, 5.0, 5.0], [-5.0, 5.0, 5.0]], F32)
    refined, iters, energy, n_un = engine.mcts_tricp(0, np.concatenate([seg, far]), placed, cand, 1.0, trim=1.0, ratio=0.99)
    assert n_un == 2 and not iters.any() and not energy.any() and np.array_equal(refined, cand)
    # and some explained: removal + refinement == refinement of the survivors, and == the reference
    shifted = placed.copy()
    shifted[0, :3, 3] += 0.05
    refined, iters, energy, n_un = engine.mcts_tricp(0, seg, shifted, cand, 0.008)
    keep = ~explained_ref(seg, prob.model_xyz, shifted, 0.008)
    assert n_un == int(keep.sum()) and 0 < n_un < len(seg)
    refs = [tricp_ref(seg[keep], prob.model_xyz, P) for P in cand]
    _check_loop(refined, iters, energy, refs)
