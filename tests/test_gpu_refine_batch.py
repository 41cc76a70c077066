"""pgp_refine_batch (many items of explained-point removal + trimmed ICP in one call) against the single calls it batches.

Every comparison is bitwise, on the same context: item i's poses, iterations, energies and n_unexplained equal
  point, n_placed > 0: pgp_mcts_tricp;      point, n_placed = 0: pgp_tricp on the whole segment;
  plane, n_placed > 0: pgp_remove_explained, the survivors in order, pgp_tricp_plane;   plane, n_placed = 0: pgp_tricp_plane;
with pgp_mcts_tricp's edges (no survivor or n_keep < 3: poses as given, iters = energy = 0)."""
import numpy as np
import pytest

from physimglobalpose_b200 import synth
from tests.test_gpu_tricp import _far, _near

gpu = pytest.mark.gpu
PGP_E_INVALID, PGP_E_NO_MODEL = -1, -4
SIZES = (300, 1000, 2000, 5000)
SLOT = 20                     # model slots SLOT .. SLOT + 3 (with normals); SLOT + 4: the 2000-point model without normals
THR = 0.008
REC = np.dtype([("obj", "<i4"), ("seg", "<i4"), ("placed_lo", "<i4"), ("n_placed", "<i4")])


class Frame:
    """Four objects of different model sizes, their segments, and two more segments: the 2000-point model placed at its ground
    truth (every point explained by that model at that pose) and the same with two far points (1 m away: only they survive)."""

    def __init__(self, engine):
        self.probs = [synth.make_segment_problem(n, 2000, 0.005, seed=300 + i) for i, n in enumerate(SIZES)]
        for k, p in enumerate(self.probs):
            engine.set_model(SLOT + k, p.model_xyz, p.model_nrm)
        p2 = self.probs[2]
        xl, nl = p2.model_xyz, p2.model_nrm
        assert engine._lib.pgp_set_model(engine._ctx, SLOT + 4, xl.ctypes.data, nl.ctypes.data, len(xl), xl.ctypes.data, None, len(xl)) == 0
        gt = p2.gt_pose
        onto = (p2.model_xyz.astype(np.float64) @ gt[:3, :3].T + gt[:3, 3]).astype(np.float32)
        far = (gt[:3, 3] + np.array([[1.0, 0, 0], [0, 1.0, 0]])).astype(np.float32)
        self.segs = [p.scene_xyz for p in self.probs] + [onto, np.concatenate([onto, far])]
        self.gt = gt

    def shifted_others(self, k, which=None):
        """The other objects' ground-truth poses shifted 5 cm along x (as tools/configs_run.py places them)."""
        js = [j for j in range(4) if j != k] if which is None else list(which)
        P = np.array([self.probs[j].gt_pose for j in js]).reshape(-1, 4, 4)
        P[:, 0, 3] += 0.05
        return P

    def items(self):
        """Every case of the mixed frame: no placed objects, shifted others, all explained, 2 survivors; k in {0, 1, 7, 64}."""
        out = []
        ks = (64, 7, 1, 0)
        for k in range(4):
            pr = self.probs[k]
            out.append((SLOT + k, k, np.zeros((0, 4, 4)), _near(pr, ks[k], 10 + k)))
            out.append((SLOT + k, k, self.shifted_others(k), _far(pr, ks[(k + 1) % 4], 20 + k)))
        out.append((SLOT + 2, 4, self.gt[None], _near(self.probs[2], 7, 30)))        # every point explained
        out.append((SLOT + 2, 5, self.gt[None], _near(self.probs[2], 64, 31)))       # two survivors: n_keep = 1
        out.append((SLOT + 2, 5, self.gt[None], _near(self.probs[2], 0, 32)))
        out.append((SLOT + 3, 0, self.shifted_others(0, (1, 2)), _near(self.probs[0], 1, 33)))
        return out


@pytest.fixture(scope="module")
def frame(engine):
    return Frame(engine)


def single(engine, metric, segs, item):
    """What the single calls give for one item: (poses, iters, energy, n_unexplained)."""
    obj, s, placed, poses = item
    seg = segs[s]
    poses = np.asarray(poses, np.float64).reshape(-1, 4, 4)
    k = len(poses)
    if len(placed):
        mask = engine.remove_explained(obj, seg, placed, THR)
        nun = int((~mask).sum())
        if k == 0:
            return poses, np.zeros(0, np.int32), np.zeros(0, np.float32), nun
        if metric == "point":
            P, it, en, n2 = engine.mcts_tricp(obj, seg, placed, poses, THR)
            assert n2 == nun
            return P, it, en, nun
        surv = seg[~mask]
        if len(surv) == 0:
            return poses.copy(), np.zeros(k, np.int32), np.zeros(k, np.float32), 0
        P, it, en = engine.tricp_plane(obj, surv, poses)
        return P, it, en, nun
    fit = engine.tricp if metric == "point" else engine.tricp_plane
    P, it, en = fit(obj, seg, poses)
    return P, it, en, len(seg)


def same(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def check_against_singles(engine, metric, segs, items, got):
    assert len(got) == len(items)
    for i, (item, g) in enumerate(zip(items, got)):
        want = single(engine, metric, segs, item)
        for name, a, b in zip(("poses", "iters", "energy"), g[:3], want[:3]):
            assert same(a, b), f"item {i} ({metric}): {name} differ from the single calls"
        assert g[3] == want[3], f"item {i} ({metric}): n_unexplained {g[3]} != {want[3]}"


@gpu
@pytest.mark.parametrize("metric", ["point", "plane"])
def test_mixed_frame_equals_single_calls(engine, frame, metric):
    items = frame.items()
    got = engine.refine_batch(frame.segs, items, metric, THR)
    check_against_singles(engine, metric, frame.segs, items, got)
    # the frame covers what it says it covers
    nun = [g[3] for g in got]
    assert nun[8] == 0 and nun[9] == 2 and 0 < nun[1] < len(frame.segs[0])
    assert all((g[1] == 0).all() and (g[2] == 0).all() for g in got[8:11])
    assert {len(g[0]) for g in got} == {0, 1, 7, 64}
    assert any((g[1] > 1).any() for g in got[:8])


@gpu
@pytest.mark.parametrize("metric", ["point", "plane"])
def test_results_do_not_depend_on_item_order_or_company(engine, frame, metric):
    items = frame.items()
    base = engine.refine_batch(frame.segs, items, metric, THR)
    perm = np.random.default_rng(5).permutation(len(items))
    got = engine.refine_batch(frame.segs, [items[i] for i in perm], metric, THR)
    for j, i in enumerate(perm):
        assert all(same(a, b) for a, b in zip(got[j][:3], base[i][:3])) and got[j][3] == base[i][3]
    rep = [items[1], items[0], items[1], items[9], items[1]]
    got = engine.refine_batch(frame.segs, rep, metric, THR)
    for j, i in enumerate((1, 0, 1, 9, 1)):
        assert all(same(a, b) for a, b in zip(got[j][:3], base[i][:3])) and got[j][3] == base[i][3]


@gpu
@pytest.mark.parametrize("metric", ["point", "plane"])
def test_rollout_shaped_batch(engine, frame, metric):
    rng = np.random.default_rng(41)
    items = []
    for r in range(320):
        k = int(rng.integers(4))
        others = [j for j in range(4) if j != k]
        which = rng.permutation(others)[:int(rng.integers(4))]
        placed = frame.shifted_others(k, which) if len(which) else np.zeros((0, 4, 4))
        items.append((SLOT + k, k, placed, _near(frame.probs[k], 1, 1000 + r)))
    got = engine.refine_batch(frame.segs, items, metric, THR)
    check_against_singles(engine, metric, frame.segs, items, got)


@gpu
def test_scratch_history_does_not_matter():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from physimglobalpose_b200.engine import PoseEngine
    e = PoseEngine(0)
    try:
        f = Frame(e)
        pr = f.probs[1]
        starts = _far(pr, 16, 7)
        before = [e.tricp(SLOT + 1, pr.scene_xyz, starts), e.tricp_plane(SLOT + 1, pr.scene_xyz, starts),
                  e.mcts_tricp(SLOT + 1, pr.scene_xyz, f.shifted_others(1), starts, THR)]
        small = f.items()[:3]
        for metric in ("point", "plane"):
            a = e.refine_batch(f.segs, small, metric, THR)
            e.refine_batch(f.segs, f.items() * 3, metric, THR)
            b = e.refine_batch(f.segs, small, metric, THR)
            for x, y in zip(a, b):
                assert all(same(u, v) for u, v in zip(x[:3], y[:3])) and x[3] == y[3]
        after = [e.tricp(SLOT + 1, pr.scene_xyz, starts), e.tricp_plane(SLOT + 1, pr.scene_xyz, starts),
                 e.mcts_tricp(SLOT + 1, pr.scene_xyz, f.shifted_others(1), starts, THR)]
        for x, y in zip(before, after):
            assert all(same(u, v) for u, v in zip(x[:3], y[:3]))
        assert before[2][3] == after[2][3]
    finally:
        e.close()


@gpu
@pytest.mark.parametrize("metric", ["point", "plane"])
def test_poisoned_pose_reports_inf_and_stays(engine, frame, metric):
    items = frame.items()
    obj, s, placed, poses = items[1]
    poses = poses.copy()
    poses[3, 0, 3] = 1e20
    items[1] = (obj, s, placed, poses)
    got = engine.refine_batch(frame.segs, items, metric, THR)
    assert got[1][2][3] == np.inf and same(got[1][0][3], poses[3])
    check_against_singles(engine, metric, frame.segs, items, got)


# ------------------------------------------------------------------------------------------------------------ refusals
class Raw:
    """A valid raw call (two segments, three placed rows shared by two items, 5 poses) with sentinel-filled outputs."""

    def __init__(self, frame):
        self.metric = 0
        self.seg = np.ascontiguousarray(np.concatenate([frame.segs[0][:500], frame.segs[1][:400]]), np.float32)
        self.seg_off = np.array([0, 500, 900], np.int64)
        self.n_segs = 2
        self.placed = np.ascontiguousarray(frame.shifted_others(0).reshape(-1, 16))
        self.n_rows = 3
        self.rec = np.array([(SLOT, 0, 0, 3), (SLOT + 1, 1, 1, 2), (SLOT + 1, 1, 0, 0)], REC)
        self.pose_off = np.array([0, 2, 4, 5], np.int64)
        self.n_items = 3
        self.poses = np.ascontiguousarray(np.concatenate([_near(frame.probs[0], 2, 1), _near(frame.probs[1], 3, 2)]).reshape(-1, 16))
        self.thr, self.trim, self.ratio, self.max_iter = THR, 0.5, 0.99, 100
        self.iters = np.full(5, 12345, np.int32)
        self.energy = np.full(5, -7.0, np.float32)
        self.nun = np.full(3, -99, np.int32)

    def outputs(self):
        return [self.poses.tobytes(), self.iters.tobytes(), self.energy.tobytes(), self.nun.tobytes()]

    def call(self, engine):
        p = lambda a: None if a is None else a.ctypes.data
        return engine._lib.pgp_refine_batch(engine._ctx, self.metric, p(self.seg), p(self.seg_off), self.n_segs, p(self.placed), self.n_rows,
                                            p(self.rec), p(self.pose_off), self.n_items, p(self.poses), self.thr, self.trim, self.ratio,
                                            self.max_iter, p(self.iters), p(self.energy), p(self.nun))


def _set(**kw):
    return lambda r: [setattr(r, k, v) for k, v in kw.items()]


def _poke(name, idx, value):
    def f(r):
        a = getattr(r, name).copy()
        a[idx] = value
        setattr(r, name, a)
    return f


def _rec(i, field, value):
    def f(r):
        r.rec = r.rec.copy()
        r.rec[i][field] = value
    return f


def _empty_segment(r):
    r.seg_off = np.array([0, 500, 500, 900], np.int64)
    r.n_segs = 3
    r.rec = r.rec.copy()
    r.rec[1]["seg"] = 1


def _too_many_poses(r):
    r.pose_off = np.array([0, 2, 4, (1 << 20) + 1], np.int64)


def _too_much_scratch(r):
    r.seg = np.ascontiguousarray(np.tile(r.seg, (2, 1)))
    r.seg_off = np.array([0, 500, 1800], np.int64)   # segment 1: 1300 points
    k = (1 << 30) // 1300 + 1                         # k x 1300 points > 2^30, k < 2^20
    r.pose_off = np.array([0, 2, 4, 4 + k], np.int64)
    r.poses = np.zeros((4 + k, 16))
    r.poses[:, [0, 5, 10, 15]] = 1.0


REFUSALS = {
    "metric 2": (_set(metric=2), PGP_E_INVALID),
    "metric -1": (_set(metric=-1), PGP_E_INVALID),
    "n_items < 0": (_set(n_items=-1), PGP_E_INVALID),
    "seg_offsets not from 0": (_poke("seg_off", 0, 1), PGP_E_INVALID),
    "seg_offsets decreasing": (_poke("seg_off", 1, 950), PGP_E_INVALID),
    "segment index = n_segs": (_rec(0, "seg", 2), PGP_E_INVALID),
    "segment index < 0": (_rec(0, "seg", -1), PGP_E_INVALID),
    "empty segment": (_empty_segment, PGP_E_INVALID),
    "placed rows past the end": (_rec(1, "n_placed", 3), PGP_E_INVALID),
    "placed_lo < 0": (_rec(0, "placed_lo", -1), PGP_E_INVALID),
    "n_placed < 0": (_rec(2, "n_placed", -1), PGP_E_INVALID),
    "pose_offsets not from 0": (_poke("pose_off", 0, 1), PGP_E_INVALID),
    "pose_offsets decreasing": (_poke("pose_off", 2, 1), PGP_E_INVALID),
    "NaN segment coordinate": (_poke("seg", (700, 1), np.nan), PGP_E_INVALID),
    "infinite placed entry": (_poke("placed", (2, 3), np.inf), PGP_E_INVALID),
    "NaN pose entry": (_poke("poses", (4, 7), np.nan), PGP_E_INVALID),
    "trim 0": (_set(trim=0.0), PGP_E_INVALID),
    "trim NaN": (_set(trim=float("nan")), PGP_E_INVALID),
    "ratio 0": (_set(ratio=0.0), PGP_E_INVALID),
    "threshold < 0": (_set(thr=-0.001), PGP_E_INVALID),
    "threshold NaN": (_set(thr=float("nan")), PGP_E_INVALID),
    "plane without normals": (lambda r: (_set(metric=1)(r), _rec(2, "obj", SLOT + 4)(r)), PGP_E_INVALID),
    "too many poses": (_too_many_poses, PGP_E_INVALID),
    "too much scratch": (_too_much_scratch, PGP_E_INVALID),
    "no model": (_rec(1, "obj", 63), PGP_E_NO_MODEL),
}


@gpu
@pytest.mark.parametrize("case", sorted(REFUSALS))
def test_refusals_leave_outputs_untouched(engine, frame, case):
    r = Raw(frame)
    mutate, code = REFUSALS[case]
    mutate(r)
    before = r.outputs()
    assert r.call(engine) == code
    assert r.outputs() == before


@gpu
def test_valid_raw_call_shared_rows_and_empty_batches(engine, frame):
    r = Raw(frame)
    assert r.call(engine) == 0
    segs = [r.seg[:500], r.seg[500:]]
    placed = r.placed.reshape(-1, 4, 4)
    P0 = Raw(frame).poses.reshape(-1, 4, 4)
    want = [single(engine, "point", segs, (SLOT, 0, placed[0:3], P0[0:2])), single(engine, "point", segs, (SLOT + 1, 1, placed[1:3], P0[2:4])),
            single(engine, "point", segs, (SLOT + 1, 1, placed[:0], P0[4:5]))]
    for i, (lo, hi) in enumerate(((0, 2), (2, 4), (4, 5))):
        assert same(r.poses.reshape(-1, 4, 4)[lo:hi], want[i][0]) and same(r.iters[lo:hi], want[i][1]) and same(r.energy[lo:hi], want[i][2])
        assert r.nun[i] == want[i][3]
    # n_items = 0: a no-op
    r = Raw(frame)
    r.n_items, r.pose_off = 0, np.zeros(1, np.int64)
    before = r.outputs()
    assert r.call(engine) == 0 and r.outputs() == before
    # every k = 0: only n_unexplained is written
    r = Raw(frame)
    r.pose_off = np.zeros(4, np.int64)
    before = r.outputs()
    assert r.call(engine) == 0
    assert r.outputs()[:3] == before[:3]
    assert list(r.nun) == [want[0][3], want[1][3], 400]
    # NULL outputs are allowed
    r = Raw(frame)
    r.iters = r.energy = r.nun = None
    assert r.call(engine) == 0 and same(r.poses.reshape(-1, 4, 4)[0:2], want[0][0])
