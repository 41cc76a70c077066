"""GPU parity of K1 + K3 + K4 against the CPU oracle, through the C ABI (libpgp.so)."""
import numpy as np
import pytest

from physimglobalpose_b200 import synth

pytestmark = pytest.mark.gpu


class _Checker:
    """The CPU checker of these tests: the reference engine itself (oracle/_ref/libs4ref.so -- built from /root/reference where
    that exists and shipped to the GPU box as a built file) answers every question it can (Verify, WeightedVerify, centroids,
    priors); the C restatement (pinned to it by tests/test_oracle_golden.py) only fills in what the reference does not expose
    per call (per-point nearest ids, the chain scan, the multi-threaded driver)."""

    def __init__(self, port_lib, args, kw):
        self.port = port_lib.PortOracle(*args, **kw)
        self.ref = port_lib.RefOracle(*args, **kw) if port_lib.have_ref() else None
        self.first = self.ref or self.port

    def verify(self, T):
        return self.first.verify(T)

    def weighted_verify(self, T, reg_of=-1):
        return self.first.weighted_verify(T, reg_of=reg_of)

    def centroids(self):
        return self.first.centroids()

    def priors(self):
        return self.first.priors()

    def __getattr__(self, name):
        return getattr(self.port, name)


def _oracle(port_lib, prob, **kw):
    return _Checker(port_lib, (prob.scene_xyz, prob.scene_nrm, prob.model_xyz, prob.model_nrm, prob.model_xyz, prob.model_nrm, prob.delta), kw)


def test_gpu_tests_check_against_the_reference_engine_when_it_travelled(port_lib, small_problem):
    """On the GPU box oracle/_ref/libs4ref.so is present (gpurun ships built files): the parity tests below then compare the CUDA
    path with Match4PCSBase::Verify / WeightedVerify directly, not only with the C restatement."""
    import os
    prob, _ = small_problem
    o = _oracle(port_lib, prob)
    assert (o.ref is not None) == os.path.exists(port_lib.REF_SO)


def _setup(engine, prob, obj=0):
    engine.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    engine.set_model(obj, prob.model_xyz, prob.model_nrm)


def test_centroids_and_conversion(engine, port_lib, small_problem):
    prob, T = small_problem
    _setup(engine, prob)
    o = _oracle(port_lib, prob)
    cP, cQ = engine.centroids(0)
    oP, oQ = o.centroids()
    assert np.array_equal(cP, oP) and np.array_equal(cQ, oQ)      # bit-exact sequential fp32 sums
    pose = engine.centred_to_pose(0, T[:5])
    back = engine.pose_to_centred(0, pose)
    assert np.allclose(back, T[:5], atol=1e-6)


def test_count_parity_small(engine, port_lib, small_problem):
    prob, T = small_problem
    _setup(engine, prob)
    want = _oracle(port_lib, prob).verify(T)
    counts, scores = engine.score_lcp(0, T, "count")
    assert np.array_equal(counts, want)                            # integer inlier counts: bit-exact
    assert counts[0] == len(prob.model_xyz) and counts.argmax() == want.argmax() == 0
    assert np.array_equal(scores, (want.astype(np.float32) / np.float32(len(prob.model_xyz))))


def test_weighted_parity_small(engine, port_lib, small_problem):
    prob, T = small_problem
    _setup(engine, prob)
    o = _oracle(port_lib, prob)
    ws, wn, reg = o.weighted_verify(T, reg_of=1)
    counts, scores = engine.score_lcp(0, T, "weighted")
    assert np.array_equal(counts, wn.astype(np.uint32))
    assert np.array_equal(scores, ws)
    assert np.array_equal(engine.registered_points(0, T[1]), reg)
    assert np.array_equal(engine.nearest_in_range(0, T[3]), o.nn_ids(T[3]))


def test_weighted_general_priors_bit_exact(engine, port_lib, small_problem):
    prob, T = small_problem
    _setup(engine, prob)
    rng = np.random.default_rng(3)
    img = rng.integers(0, 10001, size=(480, 640)).astype(np.uint16)
    K = np.array([[600.0, 0, 320], [0, 600.0, 240], [0, 0, 1]], np.float32)
    o = _oracle(port_lib, prob, K=K, prior_img=img)
    engine.set_scene_prior_image(img, K)
    assert np.array_equal(engine.scene_priors(), o.priors())
    ws, wn = o.weighted_verify(T[:200])
    counts, scores = engine.score_lcp(0, T[:200], "weighted")
    assert np.array_equal(counts, wn.astype(np.uint32))
    assert np.array_equal(scores, ws)                               # ordered fp32 accumulation: bit-exact


def test_topk_and_chain(engine, port_lib, small_problem):
    prob, T = small_problem
    _setup(engine, prob)
    o = _oracle(port_lib, prob)
    want = o.verify(T)
    counts, scores = engine.score_lcp(0, T, "count")
    top = engine.topk(0, 16)
    order = np.lexsort((np.arange(len(want)), -want.astype(np.int64)))[:16]
    assert np.array_equal(top["index"], order)
    assert np.array_equal(top["count"], want[order])
    assert np.array_equal(top["T"].reshape(-1, 3, 4), T[order])
    # improving chain in a shuffled generation order (so it is longer than one element)
    perm = np.random.default_rng(5).permutation(len(T))
    counts, scores = engine.score_lcp(0, T[perm], "count")
    chain = engine.improving_chain(0)
    assert np.array_equal(chain["index"], o.improving_chain(scores))
    assert chain["score"][-1] == scores.max() and np.all(np.diff(chain["score"]) > 0)


def test_fine_grid_equals_coarse_path_and_oracle(engine, port_lib):
    """The tri-state fast path (K1b labels + FMA voxel transform) must give the same integer counts as
    the plain 27-cell exact path and as the oracle, including for degenerate / huge / NaN matrices."""
    prob = synth.make_problem(800, 30000, 0.01, seed=21)
    T = synth.make_hypotheses(prob, 3000, seed=22).copy()
    rng = np.random.default_rng(0)
    T[5] = 0.0                                   # collapses the model onto one point
    T[6] = T[1] * 1e4                            # huge entries: intermediates beyond pos_bound -> exact path
    T[7, 0, 0] = np.nan
    T[8, :, 3] = np.inf
    T[9] = rng.normal(size=(3, 4)).astype(np.float32)        # not a rotation
    T[10, :, :3] *= 1.5                          # scaled
    _setup(engine, prob)
    want = _oracle(port_lib, prob).verify(T)
    fine, _ = engine.score_lcp(0, T, "count")
    engine.set_option("force_coarse", 1)
    try:
        coarse, _ = engine.score_lcp(0, T, "count")
    finally:
        engine.set_option("force_coarse", 0)
    assert np.array_equal(coarse, want)
    assert np.array_equal(fine, want)


def test_weighted_lists_equal_coarse_path_and_oracle(engine, port_lib):
    """WeightedVerify on the K1c nearest-candidate lists (OUT cull + per-voxel lists) must pick the same nearest
    scene point as the 27-cell search and as the oracle's kd-tree: same gated counts, same scores -- with binary
    priors (integer sums, fast kernel) and with general priors (ordered fp32 sums)."""
    prob = synth.make_problem(800, 30000, 0.01, seed=31)
    T = synth.make_hypotheses(prob, 2000, seed=32).copy()
    rng = np.random.default_rng(1)
    T[5] = 0.0
    T[6] = T[1] * 1e4
    T[7, 0, 0] = np.nan
    T[8, :, 3] = np.inf
    T[9] = rng.normal(size=(3, 4)).astype(np.float32)
    T[10, :, :3] *= 1.5
    _setup(engine, prob)
    o = _oracle(port_lib, prob)
    ws, wn = o.weighted_verify(T)
    counts, scores = engine.score_lcp(0, T, "weighted")
    engine.set_option("force_coarse", 1)
    try:
        c2, s2 = engine.score_lcp(0, T, "weighted")
    finally:
        engine.set_option("force_coarse", 0)
    assert np.array_equal(c2, wn.astype(np.uint32)) and np.array_equal(s2, ws)
    assert np.array_equal(counts, wn.astype(np.uint32)) and np.array_equal(scores, ws)
    # general priors: the ordered kernel on the lists
    img = rng.integers(0, 10001, size=(480, 640)).astype(np.uint16)
    K = np.array([[600.0, 0, 320], [0, 600.0, 240], [0, 0, 1]], np.float32)
    o2 = _oracle(port_lib, prob, K=K, prior_img=img)
    engine.set_scene_prior_image(img, K)
    ws, wn = o2.weighted_verify(T[:300])
    counts, scores = engine.score_lcp(0, T[:300], "weighted")
    assert np.array_equal(counts, wn.astype(np.uint32)) and np.array_equal(scores, ws)


def test_multi_tile_model(engine, port_lib):
    """A validation model larger than one shared-memory tile (8192 points): partial sums are combined with atomics."""
    prob = synth.make_problem(9000, 20000, 0.01, seed=41)
    T = synth.make_hypotheses(prob, 96, seed=42)
    _setup(engine, prob)
    o = _oracle(port_lib, prob)
    want = o.verify(T)
    counts, scores = engine.score_lcp(0, T, "count")
    assert np.array_equal(counts, want)
    assert np.array_equal(scores, want.astype(np.float32) / np.float32(9000))
    ws, wn = o.weighted_verify(T)
    counts, scores = engine.score_lcp(0, T, "weighted")
    assert np.array_equal(counts, wn.astype(np.uint32)) and np.array_equal(scores, ws)


def test_c5_shape_parity(engine, port_lib):
    """configs[4] shape (30k-point model, 300k-point scene): the model spans several shared-memory tiles, and in count mode the
    scene's 96 KB bitmap+rank table is staged in shared memory next to each tile; counts and weighted scores on a sample of
    hypotheses equal the oracle's.  (The table read through L1 in count mode: test_gpu_golden.py::test_lcp_delta_5mm_golden.)"""
    prob = synth.make_problem(30000, 300000, 0.01, seed=51)
    T = synth.make_hypotheses(prob, 48, seed=52)
    _setup(engine, prob)
    # 8 bytes per 32 cells; k3_score stages it while its plan fits in 216 KB, and the rest of the plan is < 68 KB here
    assert engine.grid_info()["n_cells"] // 4 < 148 * 1024
    o = _oracle(port_lib, prob)
    want = o.verify(T)
    counts, _ = engine.score_lcp(0, T, "count")
    assert np.array_equal(counts, want) and counts[0] == 30000
    ws, wn = o.weighted_verify(T[:24])
    c2, s2 = engine.score_lcp(0, T[:24], "weighted")
    assert np.array_equal(c2, wn.astype(np.uint32)) and np.array_equal(s2, ws)


def test_tail_split_units(engine, port_lib):
    """With enough hypotheses the last wave of the persistent grid is handed out in quarter-model work units whose partial sums
    are combined with atomics: results must not depend on the split, and must equal the oracle's."""
    prob = synth.make_problem(600, 20000, 0.01, seed=61)
    T = synth.make_hypotheses(prob, 52000, seed=62)      # > 2 x 24000: the host-buffer call is also cut into two overlapped chunks
    _setup(engine, prob)
    o = _oracle(port_lib, prob)
    res = {}
    for split in (4, 1, 3):
        engine.set_option("tail_split", split)
        res[split] = (engine.score_lcp(0, T, "count"), engine.score_lcp(0, T, "weighted"))
    engine.set_option("tail_split", 4)
    for split in (1, 3):
        for mode in (0, 1):
            assert np.array_equal(res[4][mode][0], res[split][mode][0]) and np.array_equal(res[4][mode][1], res[split][mode][1])
    sel = np.r_[0:300, len(T) - 1500:len(T)]
    assert np.array_equal(res[4][0][0][sel], o.verify(T[sel]))
    ws, wn = o.weighted_verify(T[sel])
    assert np.array_equal(res[4][1][1][sel], ws) and np.array_equal(res[4][1][0][sel], wn.astype(np.uint32))


def test_k3_kernel_shape_is_not_an_option(engine):
    """K3's fine kernel is built once per mode (32 warps; the cell table staged in count mode when it fits, read through L1
    otherwise and in weighted mode): warp-count and table-placement names are refused like any unknown option, and the
    remaining options are still accepted."""
    from physimglobalpose_b200 import _lib
    for name in ("k3_warps_count", "k3_warps_weighted", "k3_smem_table"):
        with pytest.raises(_lib.PgpError) as e:
            engine.set_option(name, 32)
        assert _lib.STATUS[e.value.code] == "PGP_E_INVALID" and "unknown option" in str(e.value)
    engine.set_option("tail_split", 4)


def test_group_cull_is_exact(engine, port_lib):
    """K3 drops whole 32-point groups whose bounding sphere cannot reach the scene (K1d distance field).  The cull must never
    change a count: rigid poses, poses far outside the grid, and non-rigid matrices (scaled / sheared: the sphere radius is
    stretched by the matrix norm) give the oracle's counts with the cull on, and the same counts with it off; both modes."""
    prob = synth.make_problem(1500, 40000, 0.01, seed=31)
    T = synth.make_hypotheses(prob, 4000, seed=32).copy()
    rng = np.random.default_rng(7)
    for i in range(20, 120):                      # anisotropic scale / shear around poses near the ground truth and random ones
        A = np.eye(3) + rng.normal(scale=0.4, size=(3, 3))
        T[i, :, :3] = (A @ T[i, :, :3].astype(np.float64)).astype(np.float32)
    T[120:160, :, 3] += rng.normal(scale=2.0, size=(40, 3)).astype(np.float32)      # far outside the scene grid
    T[160:200, :, :3] *= rng.uniform(0.05, 3.0, size=(40, 1, 1)).astype(np.float32)  # uniform scales
    _setup(engine, prob)
    o = _oracle(port_lib, prob)
    want = o.verify(T)
    ws, wn = o.weighted_verify(T)
    on_c, _ = engine.score_lcp(0, T, "count")
    on_w, on_ws = engine.score_lcp(0, T, "weighted")
    engine.set_option("group_cull", 0)
    try:
        off_c, _ = engine.score_lcp(0, T, "count")
        off_w, off_ws = engine.score_lcp(0, T, "weighted")
    finally:
        engine.set_option("group_cull", 1)
    assert np.array_equal(off_c, want) and np.array_equal(on_c, want)
    assert np.array_equal(off_w, wn.astype(np.uint32)) and np.array_equal(on_w, wn.astype(np.uint32))
    assert np.array_equal(on_ws, ws) and np.array_equal(off_ws, ws)


def test_score_begin_end_equals_blocking_call(engine, port_lib):
    """pgp_score_lcp_begin / _end (the pipelined host-buffer call bench.py's e2e step uses) fills the same counts and scores as
    pgp_score_lcp, with the top-k queued between the two halves; large enough for the streamed-upload path (>= 32768)."""
    import torch
    prob = synth.make_problem(600, 20000, 0.01, seed=41)
    T = synth.make_hypotheses(prob, 40000, seed=42)
    _setup(engine, prob)
    want_c, want_s = engine.score_lcp(0, T, "count")
    want_top = engine.topk(0, 16)
    Th = torch.from_numpy(T.reshape(-1, 12).copy()).pin_memory()
    ch = torch.zeros(len(T), dtype=torch.int32).pin_memory()
    sh = torch.zeros(len(T), dtype=torch.float32).pin_memory()
    engine.score_lcp_begin(0, Th.data_ptr(), len(T), ch.data_ptr(), sh.data_ptr(), "count")
    top = engine.topk(0, 16)                      # queued behind the scoring launch, before the wait
    if engine.score_lcp_end():
        top = engine.topk(0, 16)
    assert np.array_equal(ch.numpy().astype(np.uint32), want_c)
    assert np.array_equal(sh.numpy(), want_s)
    assert np.array_equal(top["index"], want_top["index"]) and np.array_equal(top["count"], want_top["count"])
    assert np.array_equal(want_c[:2000], _oracle(port_lib, prob).verify(T[:2000]))


@pytest.mark.parametrize("n_model", [1, 5, 31, 32, 33, 65])
def test_ragged_model_sizes(engine, port_lib, n_model):
    """Validation models that are not a multiple of the 32-point group / 128-point step (a single point, a partial group, one
    group plus one point): the NaN-padded tail and the dummy group must never count.  Both modes against the oracle."""
    prob = synth.make_problem(200, 8000, 0.01, seed=51)
    rng = np.random.default_rng(n_model)
    sel = rng.choice(len(prob.model_xyz), n_model, replace=False)
    mx, mn = prob.model_xyz[sel].copy(), prob.model_nrm[sel].copy()
    T = synth.make_hypotheses(prob, 600, seed=52)
    engine.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    engine.set_model(0, prob.model_xyz, prob.model_nrm, mx, mn)              # search cloud (centroid) as usual, ragged validation cloud
    o = port_lib.PortOracle(prob.scene_xyz, prob.scene_nrm, prob.model_xyz, prob.model_nrm, mx, mn, prob.delta)
    want = o.verify(T)
    ws, wn = o.weighted_verify(T)
    c, _ = engine.score_lcp(0, T, "count")
    wc, wsc = engine.score_lcp(0, T, "weighted")
    assert np.array_equal(c, want) and c.max() <= n_model
    assert np.array_equal(wc, wn.astype(np.uint32)) and np.array_equal(wsc, ws)


def test_empty_batch_and_tiny_scene(engine, port_lib):
    """Zero hypotheses is a no-op; a scene of one / two points still builds its grid and scores exactly."""
    prob = synth.make_problem(300, 5000, 0.01, seed=61)
    _setup(engine, prob)
    c, s = engine.score_lcp(0, np.zeros((0, 3, 4), np.float32), "count")
    assert len(c) == 0 and len(s) == 0
    T = synth.make_hypotheses(prob, 300, seed=62)
    for n_scene in (1, 2):
        sx, sn = prob.scene_xyz[:n_scene].copy(), prob.scene_nrm[:n_scene].copy()
        engine.set_scene(sx, sn, prob.delta)
        engine.set_model(0, prob.model_xyz, prob.model_nrm)
        o = port_lib.PortOracle(sx, sn, prob.model_xyz, prob.model_nrm, prob.model_xyz, prob.model_nrm, prob.delta)
        # poses that drop the model onto the lone scene point(s), plus the generic ones
        Tn = T.copy()
        Tn[:100, :, 3] = (sx[0] - o.centroids()[0])[None, :] + np.random.default_rng(3).normal(scale=0.02, size=(100, 3)).astype(np.float32)
        c, _ = engine.score_lcp(0, Tn, "count")
        assert np.array_equal(c, o.verify(Tn))


def test_full_size_properties(engine, port_lib):
    """BASELINE.json configs[1] at its full size (2k-pt model, 100k-pt scene, 100k hypotheses), through properties that do not
    need the oracle on every hypothesis: permutation equivariance, shard independence (two halves == whole: what the multi-GPU
    split relies on), weighted <= count, the ground-truth pose at index 0 scores every model point and is the arg-max, the
    top-k is the sorted prefix; plus the oracle itself on a 1 500-hypothesis sample spread over the batch."""
    prob = synth.make_problem(2000, 100000, 0.01, seed=1234)
    T = synth.make_hypotheses(prob, 100000, seed=4321)
    _setup(engine, prob)
    c, s = engine.score_lcp(0, T, "count")
    top = engine.topk(0, 64)
    order = np.lexsort((np.arange(len(c)), -c.astype(np.int64)))[:64]
    assert np.array_equal(top["index"], order) and np.array_equal(top["count"], c[order])
    assert c[0] == 2000 and int(c.argmax()) == 0 and c.max() <= 2000
    rng = np.random.default_rng(9)
    perm = rng.permutation(len(T))
    cp, _ = engine.score_lcp(0, T[perm], "count")
    assert np.array_equal(cp, c[perm])
    ca, _ = engine.score_lcp(0, T[:50000], "count")
    cb, _ = engine.score_lcp(0, T[50000:], "count")
    assert np.array_equal(np.concatenate([ca, cb]), c)
    wc, ws = engine.score_lcp(0, T, "weighted")
    assert np.all(wc <= c) and np.array_equal(ws, wc.astype(np.float32) / np.float32(2000))      # priors are all 1: score = gated count / n
    sample = np.sort(rng.choice(len(T), 1500, replace=False))
    o = _oracle(port_lib, prob)
    assert np.array_equal(c[sample], o.verify(T[sample]))
    wso, wno = o.weighted_verify(T[sample[:500]])
    assert np.array_equal(wc[sample[:500]], wno.astype(np.uint32)) and np.array_equal(ws[sample[:500]], wso)
