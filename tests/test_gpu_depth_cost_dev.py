"""pgp_depth_cost_dev (the rendered-depth cost on device data, asynchronous on the context's stream) against pgp_depth_cost,
bitwise, on the same context; chained behind pgp_refine_batch_dev; its device status (PGP_E_INVALID, PGP_E_CAPACITY) and its
host refusals.  The capacity cases also pin the host forms' re-run in smaller chunks (pgp_depth_cost, pgp_render_depth)."""
import numpy as np
import pytest

from physimglobalpose_b200 import synth
from tests.test_gpu_refine_batch import SLOT, THR, Frame
from tests.test_gpu_refine_batch_dev import DevCall, rollout_items
from tests.test_gpu_render import (PIX, _pixel_mesh, _random_obs, _random_triangles, _set_meshes, _table_meshes, _table_states, c1_frame, kmat,
                                   pose)

gpu = pytest.mark.gpu
PGP_OK, PGP_E_INVALID, PGP_E_NO_MODEL, PGP_E_CAPACITY = 0, -1, -4, -8


class Call:
    """One depth_cost_device call: the states' poses on the device, out filled with -7 and status with 55."""

    def __init__(self, states):
        import torch
        self.ids = [np.asarray(i, np.int32).reshape(-1) for i, _ in states]
        P = np.concatenate([np.asarray(p, np.float64).reshape(-1, 16) for _, p in states] + [np.zeros((0, 16))])
        self.poses = torch.from_numpy(np.ascontiguousarray(P)).cuda()
        self.out = torch.full((len(P), 5), -7, dtype=torch.int32, device="cuda")
        self.status = torch.full((1,), 55, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()

    def run(self, engine, tau):
        engine.depth_cost_device(self.ids, self.poses, self.out, self.status, tau)

    def results(self, engine):
        import torch
        engine.synchronize()
        torch.cuda.synchronize()
        return int(self.status.cpu()[0]), self.out.cpu().numpy()


def run_dev(engine, states, tau):
    c = Call(states)
    c.run(engine, tau)
    return c.results(engine)


def check_equal(engine, states, tau):
    status, got = run_dev(engine, states, tau)
    want = engine.depth_cost(states, tau)
    assert status == PGP_OK
    assert np.array_equal(got, want), np.argwhere(got != want)[:5]
    return got


# ------------------------------------------------------------------------------------------------------------ equality
@gpu
@pytest.mark.parametrize("n_states,max_objs", [(0, 0), (1, 3), (25, 64), (4000, 3)])
def test_table_batches_equal_host_form(engine, n_states, max_objs):
    g, raw, mask = c1_frame()
    engine.set_depth_observation(raw, mask, g["K"])
    _set_meshes(engine, _table_meshes(g))
    states = _table_states(g, np.random.default_rng(100 + n_states), n_states, max_objs)
    got = check_equal(engine, states, 0.01)
    if n_states >= 25:
        assert got[:, 0].sum() > 0 and got[:, 4].sum() > 0


@gpu
@pytest.mark.parametrize("rows,cols", [(1, 1), (17, 13), (479, 641)])
def test_random_triangles_equal_host_form(engine, rows, cols):
    rng = np.random.default_rng(rows * 7 + cols)
    K = kmat(500.0, 510.0, cols / 2 - 0.3, rows / 2 + 0.2)
    raw, mask = _random_obs(rng, rows, cols)
    engine.set_depth_observation(raw, mask, K)
    _set_meshes(engine, {0: _random_triangles(rng, 3000, K, rows, cols, 40.0) + (1,), 1: _random_triangles(rng, 200, K, rows, cols, 2000.0) + (2,)})
    states = [([0, 1], [pose(), pose(t=(0.001, 0, 0.05))]), ([1], [pose(t=(0, 0.002, 0.01))]), ([], np.zeros((0, 4, 4))), ([1, 0], [pose(), pose()])]
    got = check_equal(engine, states, 0.01)
    assert got[:, 0].sum() > 0


@gpu
def test_refilled_mesh_and_no_mask(engine):
    g, raw, mask = c1_frame()
    engine.set_depth_observation(raw, mask, g["K"])
    meshes = _table_meshes(g)
    _set_meshes(engine, meshes)
    states = _table_states(g, np.random.default_rng(7), 12, 3)
    before = check_equal(engine, states, 0.01)
    engine.set_mesh(1, *synth.ellipsoid_mesh((0.03, 0.04, 0.05), 8, 16), meshes[1][2])     # slot 1 refilled with a different mesh
    after = check_equal(engine, states, 0.01)
    assert not np.array_equal(before, after)
    engine.set_depth_observation(raw, None, g["K"])                                         # no class mask: on_segment stays 0
    got = check_equal(engine, states, 0.01)
    assert np.all(got[:, 4] == 0) and got[:, 0].sum() > 0


# ------------------------------------------------------------------------------------------------------------ chained
@gpu
def test_chained_behind_refinement(engine):
    """refine_batch_device writes the poses, depth_cost_device scores that same tensor on the same stream with no synchronisation
    in between; equal to refine_batch then depth_cost on the host.  State j places the objects of items 2j and 2j + 1."""
    frame = Frame(engine)
    g, raw, mask = c1_frame()
    engine.set_depth_observation(raw, mask, g["K"])
    for k in range(4):
        engine.set_mesh(SLOT + k, *synth.box_mesh(synth.BOX, 2), k + 1)
    items = rollout_items(frame, n=64, seed=45)
    ids = [np.array([items[2 * j][0], items[2 * j + 1][0]], np.int32) for j in range(len(items) // 2)]
    ref = DevCall(frame.segs, items)
    import torch
    out = torch.full((len(items), 5), -7, dtype=torch.int32, device="cuda")
    status = torch.full((1,), 55, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ref.run(engine, "point")
    engine.depth_cost_device(ids, ref.poses, out, status, 0.01)
    st_refine, _ = ref.results(engine)
    assert st_refine == PGP_OK and int(status.cpu()[0]) == PGP_OK
    host = engine.refine_batch(frame.segs, items, "point", THR)
    P = np.concatenate([h[0] for h in host])
    assert P.tobytes() == ref.poses.cpu().numpy().tobytes()
    want = engine.depth_cost([(i, P[2 * j:2 * j + 2]) for j, i in enumerate(ids)], 0.01)
    got = out.cpu().numpy()
    assert np.array_equal(got, want) and got[:, 0].sum() > 0


# ------------------------------------------------------------------------------------------------------------ ordering
@gpu
def test_asynchronous_on_the_context_stream(engine):
    import torch
    g, raw, mask = c1_frame()
    engine.set_depth_observation(raw, mask, g["K"])
    _set_meshes(engine, _table_meshes(g))
    small = _table_states(g, np.random.default_rng(21), 25, 3)
    big = _table_states(g, np.random.default_rng(22), 600, 3)
    s = torch.cuda.Stream()
    engine.set_stream(s.cuda_stream)
    try:
        warm = [Call(small), Call(big)]              # warm: scratch and pinned staging at these sizes
        for c in warm:
            c.run(engine, 0.01)
        engine.synchronize()
        calls = [Call(small), Call(big)]
        for c in calls:                              # back to back, no synchronisation in between
            with torch.cuda.stream(s):
                torch.cuda._sleep(500_000_000)
                c.run(engine, 0.01)
                assert not s.query(), "the call waited for the stream"
        for c, states in zip(calls, (small, big)):
            st, got = c.results(engine)
            assert st == PGP_OK and np.array_equal(got, engine.depth_cost(states, 0.01))
    finally:
        engine.set_stream(None)


# ------------------------------------------------------------------------------------------------------------ device status
@gpu
@pytest.mark.parametrize("value", [np.nan, np.inf])
def test_value_refusal_writes_nothing_and_does_not_carry_over(engine, value):
    g, raw, mask = c1_frame()
    engine.set_depth_observation(raw, mask, g["K"])
    _set_meshes(engine, _table_meshes(g))
    states = _table_states(g, np.random.default_rng(31), 25, 3)
    j = next(j for j, (ids, _) in enumerate(states) if len(ids) > 1)
    ids, P = states[j]
    P = P.copy()
    P[1, 3, 2] = value                               # the bottom row too: all 16 entries are checked
    bad = states[:j] + [(ids, P)] + states[j + 1:]
    st, got = run_dev(engine, bad, 0.01)
    assert st == PGP_E_INVALID and np.all(got == -7)
    check_equal(engine, states, 0.01)                # the next call reports PGP_OK
    c = Call([])                                     # n_states = 0 sets PGP_OK too
    c.run(engine, 0.01)
    assert c.results(engine)[0] == PGP_OK


def _full_frame_mesh(n_copies):
    """n_copies of one triangle (pixel units on the plane Z = 1 under PIX) that covers a 128 x 128 frame at Z in 1 .. 1.5."""
    v, t = _pixel_mesh([(-10, -10), (400, -10), (-10, 400)], [(0, 1, 2)])
    return v, np.tile(t, (n_copies, 1))


@gpu
def test_capacity(engine):
    """More than 2^25 (triangle, tile) entries in one chunk: the dev form reports PGP_E_CAPACITY; the host forms re-run in chunks
    that fit and give exactly what one copy of the triangle gives (coincident triangles tie on the same key)."""
    rng = np.random.default_rng(41)
    one_v, one_t = _full_frame_mesh(1)
    engine.set_mesh(50, one_v, one_t, 2)
    # one state: 2.2M copies over the 16 tiles of a 64 x 64 frame
    raw, mask = _random_obs(rng, 64, 64, 0.8, 1.3)
    engine.set_depth_observation(raw, mask, PIX)
    engine.set_mesh(51, *_full_frame_mesh(2_200_000), 2)
    P = [pose(t=(0, 0, 1.1))]
    st, got = run_dev(engine, [([51], P)], 0.01)
    assert st == PGP_E_CAPACITY and np.all(got == -7)
    want = engine.depth_cost([([50], P)], 0.01)
    assert want[0, 0] == 64 * 64 and np.array_equal(engine.depth_cost([([51], P)], 0.01), want)
    d1, s1 = engine.render_depth([50], P)
    d2, s2 = engine.render_depth([51], P)
    assert np.array_equal(d1.view(np.uint32), d2.view(np.uint32)) and np.array_equal(s1, s2) and np.all(s2 == 0)
    # several states in one chunk, 300k copies each over the 64 tiles of a 128 x 128 frame: 1.9 x 10^7 entries a state
    raw, mask = _random_obs(rng, 128, 128, 0.8, 1.6)
    engine.set_depth_observation(raw, mask, PIX)
    engine.set_mesh(52, *_full_frame_mesh(300_000), 3)
    states = [([52], [pose(t=(0, 0, 1.0))]), ([52, 50], [pose(t=(0, 0, 1.2)), pose(t=(0, 0, 1.1))]), ([50], [pose(t=(0, 0, 1.3))]),
              ([], np.zeros((0, 4, 4))), ([50, 52], [pose(t=(0, 0, 1.4)), pose(t=(0, 0, 1.05))])]
    st, got = run_dev(engine, states, 0.02)
    assert st == PGP_E_CAPACITY and np.all(got == -7)
    batch = engine.depth_cost(states, 0.02)
    alone = np.concatenate([engine.depth_cost([s], 0.02) for s in states])
    assert np.array_equal(batch, alone) and batch[:, 0].sum() == 4 * 128 * 128
    assert batch[1, 0] == 0 and np.array_equal(batch[2], engine.depth_cost([([50], [pose(t=(0, 0, 1.1))])], 0.02)[0])   # the nearer one takes all


# ------------------------------------------------------------------------------------------------------------ host refusals
HOST_REFUSALS = ["no observation", "offsets not from 0", "offsets decrease", "65 objects", "id out of range", "no mesh", "negative tau",
                 "nan tau", "inf tau", "null status", "host poses", "host out", "host status"]


@gpu
@pytest.mark.parametrize("case", HOST_REFUSALS)
def test_host_refusals_queue_nothing(engine, case):
    import torch
    from physimglobalpose_b200.engine import PoseEngine
    g, raw, mask = c1_frame()
    engine.set_depth_observation(raw, mask, g["K"])
    _set_meshes(engine, _table_meshes(g))
    P = np.tile(pose(t=(0.0, 0.0, 0.6)).reshape(1, 16), (70, 1))
    ids = np.zeros(70, np.int32)
    offs, tau, code = np.array([0, 1, 3], np.int64), 0.01, PGP_E_INVALID
    c = Call([(ids[:1], P[:1]), (ids[1:3], P[1:3])])
    dev = {"poses": c.poses.data_ptr(), "out": c.out.data_ptr(), "status": c.status.data_ptr()}
    host_P, host_out, host_status = P[:3].copy(), np.full((3, 5), -7, np.int32), np.full(1, 55, np.int32)
    ctx, fresh = engine._ctx, None
    if case == "no observation":
        fresh = PoseEngine(0)
        v, t = synth.box_mesh((0.1, 0.1, 0.1), 1)
        fresh.set_mesh(0, v, t)
        ctx = fresh._ctx
    elif case == "offsets not from 0":
        offs = np.array([1, 2, 3], np.int64)
    elif case == "offsets decrease":
        offs = np.array([0, 3, 2], np.int64)
    elif case == "65 objects":
        offs = np.array([0, 65], np.int64)
    elif case == "id out of range":
        ids[1] = 64
    elif case == "no mesh":
        ids[2], code = 40, PGP_E_NO_MODEL
    elif case.endswith("tau"):
        tau = {"negative tau": -0.001, "nan tau": float("nan"), "inf tau": float("inf")}[case]
    elif case == "null status":
        dev["status"] = None
    else:
        dev[case[5:]] = {"host poses": host_P, "host out": host_out, "host status": host_status}[case].ctypes.data
    before = c.results(engine)
    launches = engine.launch_count
    try:
        assert engine._lib.pgp_depth_cost_dev(ctx, offs.ctypes.data, len(offs) - 1, ids.ctypes.data, dev["poses"], tau, dev["out"], dev["status"]) == code
    finally:
        if fresh is not None:
            fresh.close()
    assert engine.launch_count == launches
    after = c.results(engine)
    assert after[0] == before[0] == 55 and np.array_equal(after[1], before[1])
    assert np.all(host_out == -7) and host_status[0] == 55
    torch.cuda.synchronize()
