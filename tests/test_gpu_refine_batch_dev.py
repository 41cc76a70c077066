"""pgp_refine_batch_dev (the batch on device data, asynchronous on the context's stream) against the single calls and against
pgp_refine_batch, bitwise, on the same context.  The single calls order the source on the host (morton_source); the batch orders
it on the device (k5_prep_items), so every comparison here also pins the device Morton order: a different order changes the
double sums, and ties at the trim threshold are admitted in that order."""
import numpy as np
import pytest

from physimglobalpose_b200 import synth
from tests.test_gpu_refine_batch import REFUSALS, SLOT, THR, Frame, Raw, _poke, check_against_singles, same
from tests.test_gpu_tricp import _near

gpu = pytest.mark.gpu
PGP_OK, PGP_E_INVALID = 0, -1
SORT_SHARED = 8192            # k5_tricp.cu K5_SORT_SHARED: larger segments sort their survivors in global memory
BIG = 30                      # model slot of the 20,000-point segment's object
VALUE_REFUSALS = ("NaN segment coordinate", "infinite placed entry", "NaN pose entry")


@pytest.fixture(scope="module")
def frame(engine):
    return Frame(engine)


def pack(segs, items):
    """The arrays of pgp_refine_batch for (obj, seg, placed (m, 4, 4), poses (k, 4, 4)) items, as PoseEngine.refine_batch packs them."""
    seg = np.ascontiguousarray(np.concatenate([np.asarray(s, np.float32).reshape(-1, 3) for s in segs]))
    seg_off = np.concatenate([[0], np.cumsum([len(s) for s in segs])]).astype(np.int64)
    placed = [np.asarray(it[2], np.float64).reshape(-1, 16) for it in items]
    poses = [np.asarray(it[3], np.float64).reshape(-1, 16) for it in items]
    lo = np.concatenate([[0], np.cumsum([len(p) for p in placed])])
    rec = np.array([(it[0], it[1], lo[i], len(placed[i])) for i, it in enumerate(items)], np.int32).reshape(-1, 4)
    pose_off = np.concatenate([[0], np.cumsum([len(p) for p in poses])]).astype(np.int64)
    return seg, seg_off, np.concatenate(placed + [np.zeros((0, 16))]), rec, pose_off, np.concatenate(poses + [np.zeros((0, 16))])


class DevCall:
    """One refine_batch_device call: the device inputs, sentinel-filled device outputs (None: a NULL output) and its status."""

    def __init__(self, segs, items, outputs=True):
        import torch
        seg, self.seg_off, placed, self.rec, self.pose_off, poses = pack(segs, items)
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        self.seg, self.placed, self.poses = dev(seg), dev(placed), dev(poses)
        n, p = len(items), len(poses)
        self.iters = dev(np.full(p, 12345, np.int32)) if outputs else None
        self.energy = dev(np.full(p, -7.0, np.float32)) if outputs else None
        self.nun = dev(np.full(n, -99, np.int32)) if outputs else None
        self.status = dev(np.full(1, 55, np.int32))
        torch.cuda.synchronize()

    def run(self, engine, metric):
        engine.refine_batch_device(self.seg, self.seg_off, self.placed, self.rec, self.pose_off, self.poses, self.status, self.iters, self.energy,
                                   self.nun, metric=metric, threshold=THR)

    def results(self, engine):
        """Status and one (poses, iters, energy, n_unexplained) per item, after a sync."""
        import torch
        engine.synchronize()
        torch.cuda.synchronize()
        P = self.poses.cpu().numpy()
        it = self.iters.cpu().numpy() if self.iters is not None else None
        en = self.energy.cpu().numpy() if self.energy is not None else None
        nun = self.nun.cpu().numpy() if self.nun is not None else None
        out = [(P[a:b].reshape(-1, 4, 4), None if it is None else it[a:b], None if en is None else en[a:b], None if nun is None else int(nun[i]))
               for i, (a, b) in enumerate(zip(self.pose_off[:-1], self.pose_off[1:]))]
        return int(self.status.cpu()[0]), out


def run_dev(engine, segs, items, metric):
    c = DevCall(segs, items)
    c.run(engine, metric)
    return c.results(engine)


def equal_results(a, b):
    return len(a) == len(b) and all(all(same(u, v) for u, v in zip(x[:3], y[:3])) and x[3] == y[3] for x, y in zip(a, b))


def rollout_items(frame, n=320, seed=41):
    rng = np.random.default_rng(seed)
    items = []
    for r in range(n):
        k = int(rng.integers(4))
        which = rng.permutation([j for j in range(4) if j != k])[:int(rng.integers(4))]
        placed = frame.shifted_others(k, which) if len(which) else np.zeros((0, 4, 4))
        items.append((SLOT + k, k, placed, _near(frame.probs[k], 1, 1000 + r)))
    return items


@gpu
@pytest.mark.parametrize("metric", ["point", "plane"])
def test_mixed_frame_equals_single_calls_and_host_batch(engine, frame, metric):
    items = frame.items()
    status, got = run_dev(engine, frame.segs, items, metric)
    assert status == PGP_OK
    check_against_singles(engine, metric, frame.segs, items, got)
    assert equal_results(got, engine.refine_batch(frame.segs, items, metric, THR))
    nun = [g[3] for g in got]
    assert nun[8] == 0 and nun[9] == 2 and {len(g[0]) for g in got} == {0, 1, 7, 64}


@gpu
@pytest.mark.parametrize("metric", ["point", "plane"])
def test_item_order_repeats_and_rollout(engine, frame, metric):
    items = frame.items()
    _, base = run_dev(engine, frame.segs, items, metric)
    perm = np.random.default_rng(5).permutation(len(items))
    status, got = run_dev(engine, frame.segs, [items[i] for i in perm], metric)
    assert status == PGP_OK and equal_results(got, [base[i] for i in perm])
    rep = (1, 0, 1, 9, 1)
    status, got = run_dev(engine, frame.segs, [items[i] for i in rep], metric)
    assert status == PGP_OK and equal_results(got, [base[i] for i in rep])
    roll = rollout_items(frame)
    status, got = run_dev(engine, frame.segs, roll, metric)
    assert status == PGP_OK
    check_against_singles(engine, metric, frame.segs, roll, got)


@pytest.fixture(scope="module")
def sorting_case(engine, frame):
    """Segments on both sides of the shared-memory sort: 20,000 points (global memory, with and without placed objects), exactly
    SORT_SHARED points (shared memory, at its limit), SORT_SHARED + 1 (global), and one of duplicated and coincident points (many
    equal Morton codes, ties at the trim threshold)."""
    big = synth.make_segment_problem(2000, 20000, 0.005, seed=900)
    engine.set_model(BIG, big.model_xyz, big.model_nrm)
    rng = np.random.default_rng(9)
    base = frame.probs[2].scene_xyz[:700]
    dup = np.ascontiguousarray(np.concatenate([base, base, base[:300]])[rng.permutation(1700)])
    segs = [big.scene_xyz, big.scene_xyz[:SORT_SHARED], big.scene_xyz[:SORT_SHARED + 1], dup]
    near = big.gt_pose.copy()
    near[0, 3] += 0.01
    items = [(BIG, 0, np.zeros((0, 4, 4)), _near(big, 4, 1)), (BIG, 0, near[None], _near(big, 2, 2)),
             (BIG, 1, np.zeros((0, 4, 4)), _near(big, 4, 3)), (BIG, 2, np.zeros((0, 4, 4)), _near(big, 4, 4)),
             (SLOT + 2, 3, np.zeros((0, 4, 4)), _near(frame.probs[2], 7, 5)), (SLOT + 2, 3, frame.shifted_others(2), _near(frame.probs[2], 3, 6))]
    assert len(segs[0]) == 20000 and len(segs[1]) == SORT_SHARED and len(segs[2]) == SORT_SHARED + 1
    return segs, items


@gpu
@pytest.mark.parametrize("metric", ["point", "plane"])
def test_sort_paths_and_equal_codes(engine, sorting_case, metric):
    segs, items = sorting_case
    status, got = run_dev(engine, segs, items, metric)
    assert status == PGP_OK
    check_against_singles(engine, metric, segs, items, got)
    assert equal_results(got, engine.refine_batch(segs, items, metric, THR))
    assert 0 < got[1][3] < 20000 and all(g[3] == len(segs[it[1]]) for g, it in zip(got, items) if len(it[2]) == 0)
    assert all((g[1] > 0).all() for g in got)


@gpu
@pytest.mark.parametrize("metric", ["point", "plane"])
def test_poisoned_pose_reports_inf_and_stays(engine, frame, metric):
    items = frame.items()
    obj, s, placed, poses = items[1]
    poses = poses.copy()
    poses[3, 0, 3] = 1e20
    items[1] = (obj, s, placed, poses)
    status, got = run_dev(engine, frame.segs, items, metric)
    assert status == PGP_OK and got[1][2][3] == np.inf and same(got[1][0][3], poses[3])
    check_against_singles(engine, metric, frame.segs, items, got)


# ------------------------------------------------------------------------------------------------------------ refusals
class RawDev:
    """Raw's call (tests/test_gpu_refine_batch.py) through pgp_refine_batch_dev: its bulk arrays on the device, sentinel-filled
    device outputs and a status word of 55.  ptr overrides a pointer argument (a host buffer, or 0 for NULL)."""

    def __init__(self, r):
        import torch
        self.r = r
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        self.t = dict(seg=dev(r.seg), placed=dev(r.placed), poses=dev(r.poses), iters=dev(r.iters), energy=dev(r.energy), nun=dev(r.nun),
                      status=dev(np.full(1, 55, np.int32)))
        torch.cuda.synchronize()
        self.initial = self.outputs()

    def call(self, engine, **ptr):
        p = {k: v.data_ptr() for k, v in self.t.items()}
        p.update({k: (v or None) for k, v in ptr.items()})
        r = self.r
        return engine._lib.pgp_refine_batch_dev(engine._ctx, r.metric, p["seg"], r.seg_off.ctypes.data, r.n_segs, p["placed"], r.n_rows,
                                                r.rec.ctypes.data, r.pose_off.ctypes.data, r.n_items, p["poses"], r.thr, r.trim, r.ratio, r.max_iter,
                                                p["iters"], p["energy"], p["nun"], p["status"])

    def outputs(self):
        import torch
        torch.cuda.synchronize()
        return {k: self.t[k].cpu().numpy().tobytes() for k in ("poses", "iters", "energy", "nun", "status")}


def _check_valid_call(engine, frame):
    """A valid call: status PGP_OK and every result bitwise pgp_refine_batch's."""
    d = RawDev(Raw(frame))
    assert d.call(engine) == 0
    engine.synchronize()
    host = Raw(frame)
    assert host.call(engine) == 0
    got = d.outputs()
    assert got["status"] == np.int32(PGP_OK).tobytes()
    assert [got[k] for k in ("poses", "iters", "energy", "nun")] == host.outputs()


@gpu
@pytest.mark.parametrize("case", VALUE_REFUSALS)
def test_device_value_refusal_writes_nothing_and_does_not_carry_over(engine, frame, case):
    r = Raw(frame)
    REFUSALS[case][0](r)
    d = RawDev(r)
    assert d.call(engine) == 0                      # queued: the value is found on the device
    engine.synchronize()
    got = d.outputs()
    assert got["status"] == np.int32(PGP_E_INVALID).tobytes()
    assert all(got[k] == d.initial[k] for k in ("poses", "iters", "energy", "nun"))
    _check_valid_call(engine, frame)


HOST_REFUSALS = sorted(set(REFUSALS) - set(VALUE_REFUSALS)) + ["null status", "host segments", "host poses", "host placed", "host iters",
                                                                "host status"]


@gpu
@pytest.mark.parametrize("case", HOST_REFUSALS)
def test_host_refusals_queue_nothing(engine, frame, case):
    r = Raw(frame)
    ptr, code = {}, PGP_E_INVALID
    if case in REFUSALS:
        mutate, code = REFUSALS[case]
        mutate(r)
    d = RawDev(r)
    host_buf = {"host segments": ("seg", r.seg), "host poses": ("poses", r.poses), "host placed": ("placed", r.placed),
                "host iters": ("iters", r.iters), "host status": ("status", np.zeros(1, np.int32))}
    if case == "null status":
        ptr["status"] = 0
    elif case in host_buf:
        ptr[host_buf[case][0]] = host_buf[case][1].ctypes.data
    launches = engine.launch_count
    assert d.call(engine, **ptr) == code
    assert engine.launch_count == launches
    engine.synchronize()
    assert d.outputs() == d.initial
    if case in host_buf:
        assert Raw(frame).outputs()[0] == r.poses.tobytes()          # the host buffer was not written either


# ------------------------------------------------------------------------------------------------------------ ordering
@gpu
def test_asynchronous_on_the_context_stream(engine, frame):
    import torch
    s = torch.cuda.Stream()
    small = frame.items()[:4]
    roll = rollout_items(frame, seed=43)
    engine.set_stream(s.cuda_stream)
    try:
        for items in (small, roll):                 # warm: target grids, scratch and pinned staging at these sizes
            DevCall(frame.segs, items).run(engine, "point")
        engine.synchronize()
        calls, grew = [], []
        for items in (small, roll):
            c = DevCall(frame.segs, items)
            with torch.cuda.stream(s):
                torch.cuda._sleep(500_000_000)
                before = engine.launch_count
                c.run(engine, "point")
                grew.append(engine.launch_count - before)
                assert not s.query(), "the call waited for the stream"
            calls.append(c)
        assert grew[0] == grew[1]
        st, got_small = calls[0].results(engine)
        assert st == PGP_OK
        check_against_singles(engine, "point", frame.segs, small, got_small)
        st, got_roll = calls[1].results(engine)
        assert st == PGP_OK and equal_results(got_roll, engine.refine_batch(frame.segs, roll, "point", THR))
    finally:
        engine.set_stream(None)


@gpu
def test_back_to_back_calls_without_sync(engine, frame):
    a_items, b_items = frame.items(), rollout_items(frame, n=64, seed=44)
    a, b = DevCall(frame.segs, a_items), DevCall(frame.segs, b_items)
    a.run(engine, "plane")
    b.run(engine, "point")
    sa, got_a = a.results(engine)
    sb, got_b = b.results(engine)
    assert sa == sb == PGP_OK
    assert equal_results(got_a, engine.refine_batch(frame.segs, a_items, "plane", THR))
    assert equal_results(got_b, engine.refine_batch(frame.segs, b_items, "point", THR))


@gpu
def test_null_outputs_and_empty_batch(engine, frame):
    items = frame.items()
    c = DevCall(frame.segs, items, outputs=False)
    c.run(engine, "point")
    status, got = c.results(engine)
    want = engine.refine_batch(frame.segs, items, "point", THR)
    assert status == PGP_OK and all(same(g[0], w[0]) for g, w in zip(got, want))
    # n_items = 0: nothing to refine, the values are still checked
    for bad, code in ((False, PGP_OK), (True, PGP_E_INVALID)):
        r = Raw(frame)
        if bad:
            _poke("seg", (3, 0), np.nan)(r)
        r.n_items, r.pose_off = 0, np.zeros(1, np.int64)
        d = RawDev(r)
        assert d.call(engine) == 0
        engine.synchronize()
        got = d.outputs()
        assert got["status"] == np.int32(code).tobytes() and all(got[k] == d.initial[k] for k in ("poses", "iters", "energy", "nun"))
