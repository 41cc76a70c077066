"""pgp_render_depth_dev (many states rendered into device frames, asynchronous on the context's stream) against pgp_render_depth,
bitwise, state by state; chained behind pgp_refine_batch_dev; its device status and host refusals.  pgp_set_depth_observation_dev
(the observed frame taken from device memory) against pgp_set_depth_observation, and its stream order."""
import os

import numpy as np
import pytest

from oracle import render_port as rp
from physimglobalpose_b200 import _lib, synth
from tests.test_gpu_depth_cost_dev import Call, _full_frame_mesh
from tests.test_gpu_refine_batch import SLOT, THR, Frame
from tests.test_gpu_refine_batch_dev import DevCall, rollout_items
from tests.test_gpu_render import PIX, _random_obs, _random_triangles, _set_meshes, _table_meshes, _table_states, c1_frame, kmat, pose

gpu = pytest.mark.gpu
PGP_OK, PGP_E_INVALID, PGP_E_NO_MODEL, PGP_E_CAPACITY = 0, -1, -4, -8
EMPTY = (np.zeros((0,), np.int32), np.zeros((0, 4, 4)))


def test_device_forms_are_exported():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    lib = _lib.load()
    for name in ("pgp_render_depth_dev", "pgp_set_depth_observation_dev"):
        assert hasattr(lib, name) and name in _lib.exported_symbols()


class RCall:
    """One render_depth_device call: the states' poses on the device, depth filled with -3.0, slot with -9 (slot=False: None) and
    status with 55."""

    def __init__(self, states, shape, slot=True):
        import torch
        self.ids = [np.asarray(i, np.int32).reshape(-1) for i, _ in states]
        P = np.concatenate([np.asarray(p, np.float64).reshape(-1, 16) for _, p in states] + [np.zeros((0, 16))])
        self.poses = torch.from_numpy(np.ascontiguousarray(P)).cuda()
        self.depth = torch.full((len(states),) + tuple(shape), -3.0, dtype=torch.float32, device="cuda")
        self.slot = torch.full((len(states),) + tuple(shape), -9, dtype=torch.int32, device="cuda") if slot else None
        self.status = torch.full((1,), 55, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()

    def run(self, engine):
        engine.render_depth_device(self.ids, self.poses, self.depth, self.status, self.slot)

    def status_after(self, engine):
        import torch
        engine.synchronize()
        torch.cuda.synchronize()
        return int(self.status.cpu()[0])

    def frames(self, a, b):
        """Host copies of frames [a, b): (depth, slot or None)."""
        return self.depth[a:b].cpu().numpy(), None if self.slot is None else self.slot[a:b].cpu().numpy()

    def untouched(self):
        import torch
        ok = bool(torch.all(self.depth == -3.0))
        return ok and (self.slot is None or bool(torch.all(self.slot == -9)))


def run_render(engine, states, slot=True):
    c = RCall(states, engine._frame, slot)
    c.run(engine)
    assert c.status_after(engine) == PGP_OK
    return c


def check_frames(engine, c, states, block=128):
    """Every frame of a finished call is bitwise render_depth of its state alone."""
    for a in range(0, len(states), block):
        d, s = c.frames(a, a + block)
        for k, (ids, P) in enumerate(states[a:a + block]):
            want_d, want_s = engine.render_depth(ids, P)
            assert np.array_equal(d[k].view(np.uint32), want_d.view(np.uint32)), (a + k, np.argwhere(d[k].view(np.uint32) != want_d.view(np.uint32))[:5])
            if s is not None:
                assert np.array_equal(s[k], want_s), a + k


# ------------------------------------------------------------------------------------------------------------ equality
@gpu
@pytest.mark.parametrize("n_states,max_objs", [(0, 0), (1, 3), (25, 64), (4000, 3)])
def test_table_batches_equal_host_render(engine, n_states, max_objs):
    g, raw, mask = c1_frame()
    engine.set_depth_observation(raw, mask, g["K"])
    meshes = _table_meshes(g)
    _set_meshes(engine, meshes)
    states = _table_states(g, np.random.default_rng(200 + n_states), n_states, max_objs)
    c = run_render(engine, states)
    check_frames(engine, c, states)
    if n_states == 25:                                # the counts taken on the host from the device frames equal depth_cost
        d, s = c.frames(0, n_states)
        for k, (ids, P) in enumerate(states):
            want = rp.counts_from_images(d[k], s[k], len(ids), raw, mask, [meshes[o][2] for o in ids], 0.01)
            assert np.array_equal(engine.depth_cost([(ids, P)], 0.01), want), k
        assert sum(int((s[k] >= 0).sum()) for k in range(n_states)) > 0


@gpu
@pytest.mark.parametrize("rows,cols", [(1, 1), (17, 13), (479, 641)])
def test_random_triangles_equal_host_render_and_restatement(engine, rows, cols):
    rng = np.random.default_rng(rows * 11 + cols)
    K = kmat(500.0, 510.0, cols / 2 - 0.3, rows / 2 + 0.2)
    raw, mask = _random_obs(rng, rows, cols)
    engine.set_depth_observation(raw, mask, K)
    meshes = {0: _random_triangles(rng, 3000, K, rows, cols, 40.0) + (1,), 1: _random_triangles(rng, 200, K, rows, cols, 2000.0) + (2,)}
    _set_meshes(engine, meshes)
    states = [([0, 1], [pose(), pose(t=(0.001, 0, 0.05))]), ([1], [pose(t=(0, 0.002, 0.01))]), EMPTY, ([1, 0], [pose(), pose()])]
    c = run_render(engine, states)
    check_frames(engine, c, states)
    d, s = c.frames(0, len(states))
    for k, (ids, P) in enumerate(states):
        want_d, want_s = rp.render(meshes, list(ids), P, K, rows, cols)
        assert np.array_equal(d[k].view(np.uint32), want_d.view(np.uint32)) and np.array_equal(s[k], want_s), k
        assert np.array_equal(engine.depth_cost([(ids, P)], 0.01), rp.counts_from_images(d[k], s[k], len(ids), raw, mask, [meshes[o][2] for o in ids], 0.01))
    assert np.all(d[2] == 0) and np.all(s[2] == -1) and (s[0] >= 0).sum() > 0


@gpu
def test_empty_states_and_no_slot_frames(engine):
    g, raw, mask = c1_frame()
    engine.set_depth_observation(raw, mask, g["K"])
    _set_meshes(engine, _table_meshes(g))
    c = run_render(engine, [EMPTY, EMPTY, EMPTY])                 # no placed object at all: only the frames are cleared
    d, s = c.frames(0, 3)
    assert np.all(d.view(np.uint32) == 0) and np.all(s == -1)
    states = _table_states(g, np.random.default_rng(8), 12, 3)
    states[5] = EMPTY
    c = run_render(engine, states, slot=False)
    check_frames(engine, c, states)
    assert np.all(c.frames(5, 6)[0].view(np.uint32) == 0)


@gpu
def test_refilled_mesh_and_reversed_order(engine):
    g, raw, mask = c1_frame()
    engine.set_depth_observation(raw, mask, g["K"])
    meshes = _table_meshes(g)
    _set_meshes(engine, meshes)
    states = _table_states(g, np.random.default_rng(9), 20, 3)
    before = run_render(engine, states)
    check_frames(engine, before, states)
    rev = run_render(engine, states[::-1])                        # the same states reversed: the same frames, permuted
    assert np.array_equal(rev.depth.flip(0).cpu().numpy().view(np.uint32), before.depth.cpu().numpy().view(np.uint32))
    assert np.array_equal(rev.slot.flip(0).cpu().numpy(), before.slot.cpu().numpy())
    engine.set_mesh(1, *synth.ellipsoid_mesh((0.03, 0.04, 0.05), 8, 16), meshes[1][2])     # slot 1 refilled with a different mesh
    after = run_render(engine, states)
    check_frames(engine, after, states)
    assert not np.array_equal(before.depth.cpu().numpy(), after.depth.cpu().numpy())


# ------------------------------------------------------------------------------------------------------------ chained
@gpu
def test_chained_behind_refinement(engine):
    """refine_batch_device writes the poses, render_depth_device renders that same tensor on the same stream with no synchronisation
    in between; equal to refine_batch then render_depth on the host.  State j places the objects of items 2j and 2j + 1."""
    import torch
    frame = Frame(engine)
    g, raw, mask = c1_frame()
    engine.set_depth_observation(raw, mask, g["K"])
    for k in range(4):
        engine.set_mesh(SLOT + k, *synth.box_mesh(synth.BOX, 2), k + 1)
    items = rollout_items(frame, n=64, seed=46)
    ids = [np.array([items[2 * j][0], items[2 * j + 1][0]], np.int32) for j in range(len(items) // 2)]
    ref = DevCall(frame.segs, items)
    depth = torch.full((len(ids), 480, 640), -3.0, dtype=torch.float32, device="cuda")
    slot = torch.full((len(ids), 480, 640), -9, dtype=torch.int32, device="cuda")
    status = torch.full((1,), 55, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ref.run(engine, "point")
    engine.render_depth_device(ids, ref.poses, depth, status, slot)
    st_refine, _ = ref.results(engine)
    assert st_refine == PGP_OK and int(status.cpu()[0]) == PGP_OK
    host = engine.refine_batch(frame.segs, items, "point", THR)
    P = np.concatenate([h[0] for h in host])
    assert P.tobytes() == ref.poses.cpu().numpy().tobytes()
    d, s = depth.cpu().numpy(), slot.cpu().numpy()
    for j, i in enumerate(ids):
        want_d, want_s = engine.render_depth(i, P[2 * j:2 * j + 2])
        assert np.array_equal(d[j].view(np.uint32), want_d.view(np.uint32)) and np.array_equal(s[j], want_s), j
    assert (s >= 0).sum() > 0


# ------------------------------------------------------------------------------------------------------------ ordering
@gpu
def test_asynchronous_on_the_context_stream(engine):
    import torch
    g, raw, mask = c1_frame()
    engine.set_depth_observation(raw, mask, g["K"])
    _set_meshes(engine, _table_meshes(g))
    small = _table_states(g, np.random.default_rng(23), 25, 3)
    big = _table_states(g, np.random.default_rng(24), 600, 3)
    s = torch.cuda.Stream()
    engine.set_stream(s.cuda_stream)
    try:
        for states in (small, big):                  # warm: scratch and pinned staging at these sizes
            RCall(states, (480, 640)).run(engine)
        engine.synchronize()
        calls = [RCall(small, (480, 640)), RCall(big, (480, 640))]
        for c in calls:                              # back to back, no synchronisation in between
            with torch.cuda.stream(s):
                torch.cuda._sleep(500_000_000)
                c.run(engine)
                assert not s.query(), "the call waited for the stream"
        for c, states in zip(calls, (small, big)):
            assert c.status_after(engine) == PGP_OK
            check_frames(engine, c, states)
    finally:
        engine.set_stream(None)


# ------------------------------------------------------------------------------------------------------------ device status
@gpu
@pytest.mark.parametrize("value", [np.nan, np.inf])
def test_value_refusal_writes_nothing_and_does_not_carry_over(engine, value):
    g, raw, mask = c1_frame()
    engine.set_depth_observation(raw, mask, g["K"])
    _set_meshes(engine, _table_meshes(g))
    states = _table_states(g, np.random.default_rng(33), 25, 3)
    j = next(j for j, (ids, _) in enumerate(states) if len(ids) > 1)
    for entry in range(16):                          # every one of the 16 entries is checked, the bottom row too
        ids, P = states[j]
        P = P.copy()
        P[1].reshape(16)[entry] = value
        c = RCall(states[:j] + [(ids, P)] + states[j + 1:], (480, 640))
        c.run(engine)
        assert c.status_after(engine) == PGP_E_INVALID and c.untouched(), entry
    c = run_render(engine, states)                   # the next call reports PGP_OK
    check_frames(engine, c, states)
    c = RCall([], (480, 640))                        # n_states = 0 sets PGP_OK too
    c.run(engine)
    assert c.status_after(engine) == PGP_OK


@gpu
def test_capacity(engine):
    """More than 2^25 (triangle, tile) entries in one chunk: PGP_E_CAPACITY; render_depth renders that state."""
    rng = np.random.default_rng(43)
    raw, mask = _random_obs(rng, 64, 64, 0.8, 1.3)
    engine.set_depth_observation(raw, mask, PIX)
    engine.set_mesh(50, *_full_frame_mesh(1), 2)
    engine.set_mesh(51, *_full_frame_mesh(2_200_000), 2)
    P = [pose(t=(0, 0, 1.1))]
    c = RCall([([51], P)], (64, 64))
    c.run(engine)
    assert c.status_after(engine) == PGP_E_CAPACITY
    d1, s1 = engine.render_depth([50], P)
    d2, s2 = engine.render_depth([51], P)
    assert np.array_equal(d1.view(np.uint32), d2.view(np.uint32)) and np.all(s2 == 0)


# ------------------------------------------------------------------------------------------------------------ observation
def _obs_device(raw, mask, int16=False):
    import torch
    r = torch.from_numpy(np.ascontiguousarray(raw).view(np.int16)).cuda()
    if not int16:
        r = r.view(torch.uint16)
    m = None if mask is None else torch.from_numpy(np.ascontiguousarray(mask, np.uint8)).cuda()
    return r, m, torch.full((256,), -5, dtype=torch.int64, device="cuda")


def _observation_case(engine, raw, mask, K, states, int16=False):
    """The host and the device form of one observation give the same histogram, depth_cost and render_depth."""
    import torch
    want_hist = engine.set_depth_observation(raw, mask, K)
    want_cost = engine.depth_cost(states, 0.01)
    want_frames = [engine.render_depth(i, P) for i, P in states]
    engine.set_depth_observation(encode_other(raw), None, K)      # a different observation in between
    r, m, hist = _obs_device(raw, mask, int16)
    torch.cuda.synchronize()
    engine.set_depth_observation_device(r, m, K, hist)
    engine.synchronize()
    assert np.array_equal(hist.cpu().numpy(), want_hist) and np.array_equal(want_hist, rp.class_pixels(raw, mask) if mask is not None else 0 * want_hist)
    assert np.array_equal(engine.depth_cost(states, 0.01), want_cost)
    for (i, P), (wd, ws) in zip(states, want_frames):
        d, s = engine.render_depth(i, P)
        assert np.array_equal(d.view(np.uint32), wd.view(np.uint32)) and np.array_equal(s, ws)
    return want_cost


def encode_other(raw):
    return np.ascontiguousarray(raw[::-1, ::-1])


@gpu
@pytest.mark.parametrize("with_mask", [True, False])
def test_observation_device_form_test_scene(engine, with_mask):
    g, raw, mask = c1_frame()
    _set_meshes(engine, _table_meshes(g))
    states = _table_states(g, np.random.default_rng(51), 6, 3)
    cost = _observation_case(engine, raw, mask if with_mask else None, g["K"], states, int16=not with_mask)
    assert cost[:, 0].sum() > 0 and (cost[:, 4].sum() > 0) == with_mask


@gpu
@pytest.mark.parametrize("rows,cols", [(1, 1), (17, 13), (479, 641)])
@pytest.mark.parametrize("with_mask", [True, False])
def test_observation_device_form_random_frames(engine, rows, cols, with_mask):
    rng = np.random.default_rng(rows * 13 + cols)
    K = kmat(500.0, 510.0, cols / 2 - 0.3, rows / 2 + 0.2)
    raw, mask = _random_obs(rng, rows, cols)
    _set_meshes(engine, {0: _random_triangles(rng, 2000, K, rows, cols, 40.0) + (1,), 1: _random_triangles(rng, 100, K, rows, cols, 2000.0) + (2,)})
    states = [([0, 1], [pose(), pose(t=(0.001, 0, 0.05))]), EMPTY, ([1], [pose(t=(0, 0.002, 0.01))])]
    _observation_case(engine, raw, mask if with_mask else None, K, states)


@gpu
def test_observations_follow_stream_order(engine):
    """Two observations, each followed by depth_cost_device and render_depth_device, queued back to back behind a busy stream: each
    call sees the observation queued before it."""
    import torch
    g, raw, mask = c1_frame()
    _set_meshes(engine, _table_meshes(g))
    states = _table_states(g, np.random.default_rng(52), 25, 3)
    raws = [raw, encode_other(raw)]
    masks = [mask, np.ascontiguousarray(mask[::-1, ::-1])]
    want = []
    for r, m in zip(raws, masks):
        want.append((engine.set_depth_observation(r, m, g["K"]), engine.depth_cost(states, 0.01)))
    assert not np.array_equal(want[0][1], want[1][1])
    s = torch.cuda.Stream()
    engine.set_stream(s.cuda_stream)
    try:
        obs = [_obs_device(r, m) for r, m in zip(raws, masks)]
        costs = [Call(states) for _ in raws]
        renders = [RCall(states[:3], (480, 640)) for _ in raws]
        for (r, m, h), c, rc in zip(obs, costs, renders):            # warm at these sizes
            engine.set_depth_observation_device(r, m, g["K"], h)
            c.run(engine, 0.01)
            rc.run(engine)
        engine.synchronize()
        for t in [h for _, _, h in obs] + [c.out for c in costs] + [rc.depth for rc in renders]:
            t.fill_(-5)
        torch.cuda.synchronize()
        with torch.cuda.stream(s):
            torch.cuda._sleep(500_000_000)
            for (r, m, h), c, rc in zip(obs, costs, renders):
                engine.set_depth_observation_device(r, m, g["K"], h)
                c.run(engine, 0.01)
                rc.run(engine)
            assert not s.query(), "a call waited for the stream"
        for (_, _, h), c, rc, (w_hist, w_cost) in zip(obs, costs, renders, want):
            st, got = c.results(engine)
            assert st == PGP_OK and np.array_equal(got, w_cost) and np.array_equal(h.cpu().numpy(), w_hist)
            assert rc.status_after(engine) == PGP_OK
            check_frames(engine, rc, states[:3])
    finally:
        engine.set_stream(None)


# ------------------------------------------------------------------------------------------------------------ host refusals
RENDER_REFUSALS = ["no observation", "offsets not from 0", "offsets decrease", "65 objects", "id out of range", "no mesh", "null status",
                   "null depth", "host poses", "host depth", "host slot", "host status"]


@gpu
@pytest.mark.parametrize("case", RENDER_REFUSALS)
def test_render_host_refusals_queue_nothing(engine, case):
    import torch
    from physimglobalpose_b200.engine import PoseEngine
    g, raw, mask = c1_frame()
    engine.set_depth_observation(raw, mask, g["K"])
    _set_meshes(engine, _table_meshes(g))
    P = np.tile(pose(t=(0.0, 0.0, 0.6)).reshape(1, 16), (70, 1))
    ids = np.zeros(70, np.int32)
    offs, code = np.array([0, 1, 3], np.int64), PGP_E_INVALID
    c = RCall([(ids[:1], P[:1]), (ids[1:3], P[1:3])], (480, 640))
    dev = {"poses": c.poses.data_ptr(), "depth": c.depth.data_ptr(), "slot": c.slot.data_ptr(), "status": c.status.data_ptr()}
    host = {"poses": P[:3].copy(), "depth": np.full((2, 480, 640), -3.0, np.float32), "slot": np.full((2, 480, 640), -9, np.int32),
            "status": np.full(1, 55, np.int32)}
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
    elif case.startswith("null"):
        dev[case[5:]] = None
    else:
        dev[case[5:]] = host[case[5:]].ctypes.data
    torch.cuda.synchronize()
    launches = engine.launch_count
    try:
        assert engine._lib.pgp_render_depth_dev(ctx, offs.ctypes.data, len(offs) - 1, ids.ctypes.data, dev["poses"], dev["depth"], dev["slot"],
                                                dev["status"]) == code
    finally:
        if fresh is not None:
            fresh.close()
    assert engine.launch_count == launches
    assert c.status_after(engine) == 55 and c.untouched()
    assert np.all(host["depth"] == -3.0) and np.all(host["slot"] == -9) and host["status"][0] == 55


OBSERVATION_REFUSALS = ["rows 0", "cols 0", "rows 16385", "K inf", "K nan", "fx 0", "fy negative", "null raw", "null K", "host raw",
                        "host mask", "host class pixels"]


@gpu
@pytest.mark.parametrize("case", OBSERVATION_REFUSALS)
def test_observation_host_refusals_queue_nothing(engine, case):
    import torch
    g, raw, mask = c1_frame()
    engine.set_depth_observation(raw, mask, g["K"])
    _set_meshes(engine, _table_meshes(g))
    states = _table_states(g, np.random.default_rng(53), 4, 3)
    want = engine.depth_cost(states, 0.01)
    r, m, hist = _obs_device(encode_other(raw), mask)
    K = g["K"].astype(np.float32).reshape(9).copy()
    host_hist = np.full(256, -5, np.int64)
    args = {"raw": r.data_ptr(), "mask": m.data_ptr(), "rows": 480, "cols": 640, "K": K.ctypes.data, "class pixels": hist.data_ptr()}
    if case.startswith("rows") or case.startswith("cols"):
        args[case[:4]] = int(case[5:])
    elif case.startswith("K") or case.startswith("f"):
        K[{"K inf": 2, "K nan": 7, "fx 0": 0, "fy negative": 4}[case]] = {"K inf": np.inf, "K nan": np.nan, "fx 0": 0.0, "fy negative": -1.0}[case]
    elif case.startswith("null"):
        args[case[5:]] = None
    else:
        args[case[5:]] = {"raw": raw, "mask": mask, "class pixels": host_hist}[case[5:]].ctypes.data
    torch.cuda.synchronize()
    launches = engine.launch_count
    assert engine._lib.pgp_set_depth_observation_dev(engine._ctx, args["raw"], args["mask"], args["rows"], args["cols"], args["K"],
                                                     args["class pixels"]) == PGP_E_INVALID
    assert engine.launch_count == launches
    torch.cuda.synchronize()
    assert bool(torch.all(hist == -5)) and np.all(host_hist == -5)
    assert np.array_equal(engine.depth_cost(states, 0.01), want)                # the observation before the refusal still holds
