"""K4d (pgp_distinct_dev, pgp_topk_distinct) against its float64 restatement (oracle/select_port.py), bitwise: kept records,
their order, the counts and the camera-frame poses."""
import math

import numpy as np
import pytest

from oracle.select_port import centred_to_pose, distinct
from physimglobalpose_b200 import synth
from physimglobalpose_b200.engine import HYP_DTYPE, PoseGroup

gpu = pytest.mark.gpu
PGP_OK, PGP_E_INVALID, PGP_E_NO_SCENE, PGP_E_NO_MODEL = 0, -1, -3, -4
SLOTS = (50, 51, 52, 53)                     # model slots of this module (cleared of symmetries at the end)
FLIPS = [np.diag(d) for d in ([-1.0, -1.0, 1.0], [-1.0, 1.0, -1.0], [1.0, -1.0, -1.0])]   # a box's three 180 degree turns
COS10 = math.cos(math.radians(10.0))


def rand_rot(rng, n):
    q = rng.normal(size=(n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    w, x, y, z = q.T
    return np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                     2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                     2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], -1).reshape(n, 3, 3)


def small_rot(rng, n, max_rad):
    axis = rng.normal(size=(n, 3))
    axis /= np.linalg.norm(axis, axis=1, keepdims=True)
    return np.stack([synth.rot_axis_angle(a, th) for a, th in zip(axis, rng.uniform(0, max_rad, n))])


def pool_records(T12, index=None, seed=0):
    T12 = np.asarray(T12, np.float32).reshape(-1, 12)
    rng = np.random.default_rng(seed)
    r = np.zeros(len(T12), HYP_DTYPE)
    r["T"] = T12
    r["index"] = np.arange(len(T12)) * 3 + 5 if index is None else index
    r["count"] = rng.integers(0, 1000, len(T12))
    r["score"] = rng.uniform(0, 1, len(T12)).astype(np.float32)
    return r


def make_pool(kind, m, n_syms, seed):
    """uniform: rotations and translations anywhere in a 10 cm box; clustered: tight jitter (2 mm, 2 degrees) around a few
    centres, each member turned by one of the symmetries at random."""
    rng = np.random.default_rng(seed)
    if kind == "uniform":
        R, t = rand_rot(rng, m), rng.uniform(-0.05, 0.05, (m, 3))
    else:
        nc = 5
        cR, ct = rand_rot(rng, nc), rng.uniform(-0.05, 0.05, (nc, 3))
        c = rng.integers(0, nc, m)
        R = np.einsum("nij,njk->nik", cR[c], small_rot(rng, m, math.radians(2.0)))
        t = ct[c] + rng.uniform(-0.002, 0.002, (m, 3))
        if n_syms:
            S = np.stack([np.eye(3)] + FLIPS[:n_syms])[rng.integers(0, n_syms + 1, m)]
            R = np.einsum("nij,njk->nik", R, S)
    T = np.zeros((m, 3, 4))
    T[:, :, :3], T[:, :, 3] = R, t
    return pool_records(T.reshape(m, 12), seed=seed)


def dev_tensor(records):
    import torch
    return torch.from_numpy(np.ascontiguousarray(records).view(np.uint8).copy()).cuda()


class Call:
    """One pgp_distinct_dev call through the C ABI with an exact cos_angle; sentinel-filled outputs."""

    def __init__(self, objs, pools, k, max_dist, cos_angle, poses=True, n_kept=True):
        import torch
        self.objs = np.asarray(objs, np.int32)
        self.off = np.concatenate([[0], np.cumsum([len(p) for p in pools])]).astype(np.int64)
        self.pools, self.k, self.max_dist, self.cos_angle = pools, k, max_dist, cos_angle
        self.pool = dev_tensor(np.concatenate(pools))
        n = len(pools)
        self.out = torch.full((n * k * 64,), 0x5A, dtype=torch.uint8, device="cuda")
        self.poses = torch.full((n * k, 16), -3.0, dtype=torch.float64, device="cuda") if poses else None
        self.n_kept = torch.full((n,), -9, dtype=torch.int32, device="cuda") if n_kept else None
        torch.cuda.synchronize()

    def run(self, eng, **over):
        a = dict(objs=self.objs.ctypes.data, off=self.off.ctypes.data, n=len(self.objs), pool=self.pool.data_ptr(), k=self.k,
                 max_dist=self.max_dist, cos_angle=self.cos_angle, out=self.out.data_ptr(),
                 poses=None if self.poses is None else self.poses.data_ptr(), n_kept=None if self.n_kept is None else self.n_kept.data_ptr())
        a.update(over)
        return eng._lib.pgp_distinct_dev(eng._ctx, a["objs"], a["off"], a["n"], a["pool"], a["k"], a["max_dist"], a["cos_angle"], a["out"],
                                         a["poses"], a["n_kept"])

    def results(self, eng):
        import torch
        eng.synchronize()
        torch.cuda.synchronize()
        out = self.out.cpu().numpy().view(HYP_DTYPE).reshape(len(self.objs), self.k)
        poses = None if self.poses is None else self.poses.cpu().numpy().reshape(len(self.objs), self.k, 16)
        n_kept = None if self.n_kept is None else self.n_kept.cpu().numpy()
        return out, poses, n_kept


def same_records(a, b):
    return np.ascontiguousarray(a).view(np.uint8).tobytes() == np.ascontiguousarray(b).view(np.uint8).tobytes()


def padding(n):
    r = np.zeros(n, HYP_DTYPE)
    r["index"] = -1
    return r


def check_list(out_row, n_kept, pool, k, max_dist, cos_angle, syms, poses_row=None, eng=None, obj=None):
    want = distinct(pool["T"], pool["index"], k, max_dist, cos_angle, syms)
    assert n_kept == len(want)
    assert same_records(out_row[:n_kept], pool[want])
    assert same_records(out_row[n_kept:], padding(k - n_kept))
    if poses_row is not None:
        cP, cQ = eng.centroids(obj)
        assert np.array_equal(poses_row[:n_kept].view(np.uint64), centred_to_pose(pool[want]["T"], cP, cQ).view(np.uint64))
        assert np.array_equal(poses_row[n_kept:], np.tile(np.eye(4).reshape(16), (k - n_kept, 1)))
    return want


@pytest.fixture(scope="module")
def sc(engine):
    prob = synth.make_problem(400, 8000, 0.01, seed=91)
    engine.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    for i, obj in enumerate(SLOTS):          # different subsamples: different centroids per slot
        engine.set_model(obj, prob.model_xyz[i:], prob.model_nrm[i:])
        engine.set_symmetries(obj, None)
    yield engine, prob
    for obj in SLOTS:
        engine.set_symmetries(obj, None)


@gpu
@pytest.mark.parametrize("kind", ["uniform", "clustered"])
@pytest.mark.parametrize("n_syms", [0, 1, 3])
@pytest.mark.parametrize("m", [1, 2, 63, 64, 65, 1000, 4096])
def test_random_pools_match_the_restatement(sc, kind, n_syms, m):
    eng, _ = sc
    obj = SLOTS[0]
    syms = FLIPS[:n_syms]
    eng.set_symmetries(obj, syms)
    pool = make_pool(kind, m, n_syms, seed=m * 7 + n_syms)
    max_dist, cos_angle = (0.03, 0.5) if kind == "uniform" else (0.01, COS10)
    full = distinct(pool["T"], pool["index"], m, max_dist, cos_angle, syms)     # greedy with a stop at k is a prefix of the full walk
    for k in sorted({1, 64, m}):
        c = Call([obj], [pool], k, max_dist, cos_angle)
        assert c.run(eng) == PGP_OK, eng._lib.pgp_last_error(eng._ctx)
        out, poses, n_kept = c.results(eng)
        want = full[:k]
        assert n_kept[0] == len(want)
        assert same_records(out[0, :len(want)], pool[want]) and same_records(out[0, len(want):], padding(k - len(want)))
        cP, cQ = eng.centroids(obj)
        assert np.array_equal(poses[0, :len(want)].view(np.uint64), centred_to_pose(pool[want]["T"], cP, cQ).view(np.uint64))
        assert np.array_equal(poses[0, len(want):], np.tile(np.eye(4).reshape(16), (k - len(want), 1)))
    if kind == "clustered" and m >= 1000:
        assert len(full) < m / 10, "the clustered pool should collapse to a few placements"
    eng.set_symmetries(obj, None)


@gpu
def test_padding_and_nan_records(sc):
    eng, _ = sc
    obj = SLOTS[1]
    pool = make_pool("clustered", 300, 0, seed=5)
    pool["index"][::7] = -1
    pool["T"][3::11, 3] = np.nan
    pool["T"][5::13, 4] = np.nan
    c = Call([obj], [pool], 300, 0.01, COS10)
    assert c.run(eng) == PGP_OK
    out, poses, n_kept = c.results(eng)
    want = check_list(out[0], n_kept[0], pool, 300, 0.01, COS10, [], poses[0], eng, obj)
    assert np.isnan(pool["T"][want]).any(axis=1).sum() == np.isnan(pool["T"][pool["index"] >= 0]).any(axis=1).sum()


def rotz32(deg):
    R = np.eye(3, dtype=np.float32)
    c, s = np.float32(math.cos(math.radians(deg))), np.float32(math.sin(math.radians(deg)))
    R[0, 0], R[0, 1], R[1, 0], R[1, 1] = c, -s, s, c
    return R


def tr_of(Ra, Rb):
    """The contract's trace for S = I, in double from the fp32 entries."""
    a, b = Ra.astype(np.float64).reshape(9), Rb.astype(np.float64).reshape(9)
    tr = a[0] * b[0]
    for e in range(1, 9):
        tr = tr + a[e] * b[e]
    return tr


@gpu
@pytest.mark.parametrize("trans", ["at", "past"])
@pytest.mark.parametrize("rot", ["at", "past"])
def test_thresholds_exactly_and_one_ulp_past(sc, trans, rot):
    eng, _ = sc
    obj = SLOTS[0]
    Ra, Rb = rotz32(0.0), rotz32(7.3)
    tr = tr_of(Ra, Rb)
    cos_at = (tr - 1.0) / 2.0
    assert 1.0 + 2.0 * cos_at == tr
    cos_past = (np.nextafter(tr, 4.0) - 1.0) / 2.0
    assert 1.0 + 2.0 * cos_past == np.nextafter(tr, 4.0)
    a = np.zeros((3, 4), np.float32)
    b = np.zeros((3, 4), np.float32)
    a[:, :3], b[:, :3] = Ra, Rb
    a[:, 3] = (0.25, -0.5, 1.0)
    b[:, 3] = (0.25 + 3 / 1024, -0.5 + 4 / 1024, 1.0)           # d2 = 25 * 2^-20 exactly
    dist_at = 5 / 1024
    dist = dist_at if trans == "at" else float(np.nextafter(dist_at, 0.0))
    cos = cos_at if rot == "at" else cos_past
    pool = pool_records(np.stack([a.reshape(12), b.reshape(12)]))
    c = Call([obj], [pool], 2, dist, cos)
    assert c.run(eng) == PGP_OK
    out, _, n_kept = c.results(eng)
    assert n_kept[0] == (1 if trans == rot == "at" else 2)
    check_list(out[0], n_kept[0], pool, 2, dist, cos, [])


@gpu
def test_symmetry_threshold_exact(sc):
    eng, _ = sc
    obj = SLOTS[2]
    Rb = rotz32(180.0 + 4.0)
    S = np.diag([-1.0, -1.0, 1.0])
    G = np.zeros((3, 3))
    Rb64 = Rb.astype(np.float64)
    for r in range(3):
        for cc in range(3):
            G[r, cc] = (Rb64[r, 0] * S[0, cc] + Rb64[r, 1] * S[1, cc]) + Rb64[r, 2] * S[2, cc]
    tr = tr_of(np.eye(3, dtype=np.float32), G)
    cos_at = (tr - 1.0) / 2.0
    cos_past = (np.nextafter(tr, 4.0) - 1.0) / 2.0
    a, b = np.zeros((3, 4), np.float32), np.zeros((3, 4), np.float32)
    a[:, :3], b[:, :3] = np.eye(3), Rb
    pool = pool_records(np.stack([a.reshape(12), b.reshape(12)]))
    for syms, cos, want in (([S], cos_at, 1), ([S], cos_past, 2), ([], cos_at, 2)):
        eng.set_symmetries(obj, syms)
        c = Call([obj], [pool], 2, 0.0, cos)
        assert c.run(eng) == PGP_OK
        out, _, n_kept = c.results(eng)
        assert n_kept[0] == want
        check_list(out[0], n_kept[0], pool, 2, 0.0, cos, syms)
    eng.set_symmetries(obj, None)


@gpu
@pytest.mark.parametrize("mode", ["count", "weighted"])
def test_topk_distinct_is_the_restatement_on_topk(sc, mode):
    eng, prob = sc
    obj = SLOTS[0]
    eng.set_symmetries(obj, FLIPS[:1])
    T = synth.make_hypotheses(prob, 20000, seed=17)
    eng.score_lcp(obj, T, mode)
    for m, k, d, ang in ((4096, 64, 0.01, 10.0), (1000, 1000, 0.005, 5.0), (64, 1, 0.01, 10.0)):
        pool = eng.topk(obj, m)
        got = eng.topk_distinct(obj, m, k, d, math.radians(ang))
        want = distinct(pool["T"], pool["index"], k, d, math.cos(math.radians(ang)), FLIPS[:1])
        assert same_records(got, pool[want])
    eng.set_symmetries(obj, None)


@gpu
def test_multi_list_equals_single_lists_in_any_order(sc):
    eng, _ = sc
    syms = {SLOTS[0]: [], SLOTS[1]: FLIPS[:1], SLOTS[2]: FLIPS, SLOTS[3]: FLIPS[1:2]}
    for obj, s in syms.items():
        eng.set_symmetries(obj, s)
    rng = np.random.default_rng(3)
    lists = [(SLOTS[i % 4], make_pool("clustered" if i % 3 else "uniform", int(m), len(syms[SLOTS[i % 4]]) % 4, seed=100 + i))
             for i, m in enumerate([4096, 1, 65, 700, 64, 2000, 3, 4096, 130])]
    k = 64
    singles = []
    for obj, pool in lists:
        c = Call([obj], [pool], k, 0.01, COS10)
        assert c.run(eng) == PGP_OK
        singles.append(c.results(eng))
    for order in (np.arange(len(lists)), rng.permutation(len(lists))):
        c = Call([lists[i][0] for i in order], [lists[i][1] for i in order], k, 0.01, COS10)
        assert c.run(eng) == PGP_OK
        out, poses, n_kept = c.results(eng)
        for row, i in enumerate(order):
            s_out, s_poses, s_n = singles[i]
            assert n_kept[row] == s_n[0] and same_records(out[row], s_out[0]) and np.array_equal(poses[row], s_poses[0])
            obj, pool = lists[i]
            check_list(out[row], n_kept[row], pool, k, 0.01, COS10, syms[obj], poses[row], eng, obj)
    for obj in syms:
        eng.set_symmetries(obj, None)


@gpu
def test_asynchronous_on_the_context_stream(sc):
    import torch
    eng, _ = sc
    s = torch.cuda.Stream()
    one = [(SLOTS[0], make_pool("clustered", 4096, 0, seed=1))]
    many = [(SLOTS[i % 4], make_pool("clustered", 4096, 0, seed=2 + i)) for i in range(8)]
    eng.set_stream(s.cuda_stream)
    try:
        for lists in (one, many):                 # warm: scratch and pinned staging at these sizes
            Call([o for o, _ in lists], [p for _, p in lists], 64, 0.01, COS10).run(eng)
        eng.synchronize()
        calls, grew = [], []
        for lists in (one, many):
            c = Call([o for o, _ in lists], [p for _, p in lists], 64, 0.01, COS10)
            with torch.cuda.stream(s):
                torch.cuda._sleep(500_000_000)
                before = eng.launch_count
                assert c.run(eng) == PGP_OK
                grew.append(eng.launch_count - before)
                assert not s.query(), "the call waited for the stream"
            calls.append((lists, c))
        assert grew[0] == grew[1] == 2
        for lists, c in calls:
            out, poses, n_kept = c.results(eng)
            for row, (obj, pool) in enumerate(lists):
                check_list(out[row], n_kept[row], pool, 64, 0.01, COS10, [], poses[row], eng, obj)
    finally:
        eng.set_stream(None)


def _refusals():
    P = {}
    P["n_lists < 0"] = dict(n=-1)
    P["k = 0"] = dict(k=0)
    P["k = 4097"] = dict(k=4097)
    P["max_dist NaN"] = dict(max_dist=float("nan"))
    P["max_dist inf"] = dict(max_dist=float("inf"))
    P["max_dist < 0"] = dict(max_dist=-1e-3)
    P["cos_angle NaN"] = dict(cos_angle=float("nan"))
    P["null objs"] = dict(objs=None)
    P["null offsets"] = dict(off=None)
    P["null pool"] = dict(pool=None)
    P["null out"] = dict(out=None)
    return P


REFUSALS = _refusals()
HOST_SHAPES = ("offset 0 not 0", "empty list", "list of 4097", "obj out of range", "obj without model", "pool on the host",
               "out on the host", "poses on the host", "n_kept on the host", "no scene for poses")


@gpu
@pytest.mark.parametrize("case", list(REFUSALS) + list(HOST_SHAPES))
def test_refusals_queue_nothing(sc, case):
    import torch
    eng, prob = sc
    pools = [make_pool("clustered", 100, 0, seed=9), make_pool("clustered", 50, 0, seed=10)]
    c = Call([SLOTS[0], SLOTS[1]], pools, 16, 0.01, COS10)
    over, code = dict(REFUSALS.get(case, {})), PGP_E_INVALID
    host = np.zeros(4096 * 64, np.uint8)
    if case == "offset 0 not 0":
        c.off[:] = (1, 101, 151)
    elif case == "empty list":
        c.off[:] = (0, 0, 150)
    elif case == "list of 4097":
        big = make_pool("uniform", 4097, 0, seed=11)
        c = Call([SLOTS[0]], [big], 16, 0.01, COS10)
    elif case == "obj out of range":
        c.objs[1] = 64
    elif case == "obj without model":
        c.objs[1] = 63
        code = PGP_E_NO_MODEL
    elif case in ("pool on the host", "out on the host"):
        over = {case.split()[0]: host.ctypes.data}
    elif case in ("poses on the host", "n_kept on the host"):
        over = {case.split()[0]: host.ctypes.data}
    before = eng.launch_count
    if case == "no scene for poses":
        from physimglobalpose_b200.engine import PoseEngine
        e2 = PoseEngine(0)
        try:
            e2.set_model(SLOTS[0], prob.model_xyz, prob.model_nrm)
            e2.set_model(SLOTS[1], prob.model_xyz, prob.model_nrm)
            assert c.run(e2) == PGP_E_NO_SCENE
            assert e2.launch_count == 0
        finally:
            e2.close()
    else:
        assert c.run(eng, **over) == code, case
    assert eng.launch_count == before
    out, poses, n_kept = c.results(eng)
    assert (out.view(np.uint8) == 0x5A).all() and (poses == -3.0).all() and (n_kept == -9).all()
    torch.cuda.synchronize()


@gpu
def test_set_symmetries_refusals(sc):
    eng, _ = sc
    lib, ctx = eng._lib, eng._ctx
    R = np.tile(np.eye(3).reshape(9), (24, 1))
    assert lib.pgp_set_symmetries(ctx, 64, R.ctypes.data, 1) == PGP_E_INVALID
    assert lib.pgp_set_symmetries(ctx, -1, R.ctypes.data, 1) == PGP_E_INVALID
    assert lib.pgp_set_symmetries(ctx, SLOTS[0], R.ctypes.data, -1) == PGP_E_INVALID
    assert lib.pgp_set_symmetries(ctx, SLOTS[0], R.ctypes.data, 24) == PGP_E_INVALID
    assert lib.pgp_set_symmetries(ctx, SLOTS[0], None, 2) == PGP_E_INVALID
    bad = R.copy()
    bad[1, 4] = np.inf
    assert lib.pgp_set_symmetries(ctx, SLOTS[0], bad.ctypes.data, 2) == PGP_E_INVALID
    assert lib.pgp_set_symmetries(ctx, SLOTS[0], R.ctypes.data, 23) == PGP_OK
    assert lib.pgp_set_symmetries(ctx, SLOTS[0], None, 0) == PGP_OK


@gpu
def test_set_model_keeps_the_symmetries(sc):
    eng, prob = sc
    obj = SLOTS[3]
    a, b = np.zeros((3, 4), np.float32), np.zeros((3, 4), np.float32)
    a[:, :3], b[:, :3] = np.eye(3), FLIPS[0]
    pool = pool_records(np.stack([a.reshape(12), b.reshape(12)]))
    eng.set_symmetries(obj, FLIPS[:1])
    eng.set_model(obj, prob.model_xyz[3:], prob.model_nrm[3:])
    c = Call([obj], [pool], 2, 0.01, COS10)
    assert c.run(eng) == PGP_OK
    assert c.results(eng)[2][0] == 1
    eng.set_symmetries(obj, None)


@gpu
def test_chain_topk_distinct_refine_without_host_sync(sc):
    import torch
    eng, prob = sc
    k, m = 16, 4096
    T = synth.make_hypotheses(prob, 30000, seed=23)
    Td = torch.from_numpy(T.reshape(-1, 12)).cuda()
    counts = [torch.zeros(len(T), dtype=torch.int32, device="cuda") for _ in SLOTS]
    scores = [torch.zeros(len(T), dtype=torch.float32, device="cuda") for _ in SLOTS]
    pool = torch.zeros(len(SLOTS) * m * 64, dtype=torch.uint8, device="cuda")
    out = torch.zeros(len(SLOTS) * k * 64, dtype=torch.uint8, device="cuda")
    poses = torch.zeros((len(SLOTS) * k, 16), dtype=torch.float64, device="cuda")
    n_kept = torch.zeros(len(SLOTS), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    for i, obj in enumerate(SLOTS):
        eng.score_lcp_device(obj, Td, counts[i], scores[i], "weighted")
        eng.topk_device(obj, m, 0, pool[i * m * 64:(i + 1) * m * 64])
    eng.distinct_device(list(SLOTS), np.arange(len(SLOTS) + 1) * m, pool, k, 0.01, math.radians(10.0), out, poses, n_kept)
    seg = torch.from_numpy(prob.scene_xyz).cuda()
    items = np.array([(obj, 0, 0, 0) for obj in SLOTS], np.int32)
    status = torch.full((1,), 55, dtype=torch.int32, device="cuda")
    eng.refine_batch_device(seg, np.array([0, len(prob.scene_xyz)]), torch.zeros((0, 16), dtype=torch.float64, device="cuda"), items,
                            np.arange(len(SLOTS) + 1) * k, poses, status)
    eng.synchronize()
    torch.cuda.synchronize()
    assert int(status.item()) == PGP_OK
    rec = out.cpu().numpy().view(HYP_DTYPE).reshape(len(SLOTS), k)
    nk = n_kept.cpu().numpy()
    refined = poses.cpu().numpy().reshape(len(SLOTS), k, 4, 4)
    pools = pool.cpu().numpy().view(HYP_DTYPE).reshape(len(SLOTS), m)
    host_items = []
    for i, obj in enumerate(SLOTS):
        check_list(rec[i], nk[i], pools[i], k, 0.01, math.cos(math.radians(10.0)), [])
        assert nk[i] >= 1
        host_items.append((obj, 0, np.zeros((0, 4, 4)), eng.centred_to_pose(obj, rec[i]["T"][:nk[i]])))
    want = eng.refine_batch([prob.scene_xyz], host_items)
    for i in range(len(SLOTS)):
        assert np.array_equal(refined[i, :nk[i]], want[i][0])
        assert np.isfinite(refined[i]).all()


@gpu
def test_two_devices_equal_one_context():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from physimglobalpose_b200.engine import PoseEngine
    prob = synth.make_problem(400, 8000, 0.01, seed=92)
    T = synth.make_hypotheses(prob, 50001, seed=29)
    one = PoseEngine(0)
    g2 = PoseGroup([0, 1])
    try:
        for e in (one, g2):
            e.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
            e.set_model(0, prob.model_xyz, prob.model_nrm)
            e.set_symmetries(0, FLIPS[:1])
        for mode in ("count", "weighted"):
            one.score_lcp(0, T, mode)
            g2.score_lcp(0, T, mode)
            for m, k in ((4096, 64), (300, 300)):
                a = one.topk_distinct(0, m, k, 0.01, math.radians(10.0))
                b = g2.topk_distinct(0, m, k, 0.01, math.radians(10.0))
                assert same_records(a, b)
    finally:
        g2.close()
        one.close()
