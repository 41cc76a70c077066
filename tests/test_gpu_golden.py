"""CUDA path vs the golden vectors minted from the compiled reference engine (tests/golden/*.npz).
These run on the GPU box, where /root/reference does not exist."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def lcp():
    return np.load(os.path.join(G, "lcp_small.npz"))


def test_lcp_count_golden(engine, lcp):
    engine.set_scene(lcp["scene_xyz"], lcp["scene_nrm"], float(lcp["delta"]))
    engine.set_model(0, lcp["model_xyz"], lcp["model_nrm"])
    cP, cQ = engine.centroids(0)
    assert np.array_equal(cP, lcp["cP"]) and np.array_equal(cQ, lcp["cQ"])
    counts, scores = engine.score_lcp(0, lcp["T"], "count")
    assert np.array_equal(counts, lcp["counts"])                       # bit-exact vs Match4PCSBase::Verify
    chain = engine.improving_chain(0)
    # the reference's running-best scan with early termination ends on the same hypothesis with the same score
    assert chain["index"][-1] == int(lcp["running_best"])
    assert chain["score"][-1] == lcp["running_frac"][int(lcp["running_best"])]
    engine.set_option("force_coarse", 1)
    try:
        c2, _ = engine.score_lcp(0, lcp["T"], "count")
    finally:
        engine.set_option("force_coarse", 0)
    assert np.array_equal(c2, lcp["counts"])


def test_lcp_weighted_golden(engine, lcp):
    engine.set_scene(lcp["scene_xyz"], lcp["scene_nrm"], float(lcp["delta"]))
    engine.set_model(0, lcp["model_xyz"], lcp["model_nrm"])
    counts, scores = engine.score_lcp(0, lcp["T"], "weighted")
    assert np.array_equal(scores, lcp["weighted_score"])               # bit-exact vs WeightedVerify
    assert np.array_equal(counts, lcp["weighted_nreg"].astype(np.uint32))
    reg = engine.registered_points(0, lcp["T"][int(lcp["registered_of"])])
    assert np.array_equal(reg, lcp["registered"])
    # probability image -> per-point priors -> ordered fp32 accumulation
    engine.set_scene_prior_image(lcp["prior_img"], lcp["K"])
    assert np.array_equal(engine.scene_priors(), lcp["priors"])
    counts, scores = engine.score_lcp(0, lcp["T"], "weighted")
    assert np.array_equal(scores, lcp["weighted_score_img"])
    assert np.array_equal(counts, lcp["weighted_nreg_img"].astype(np.uint32))


def test_lcp_delta_5mm_golden(engine, lcp):
    d5 = np.load(os.path.join(G, "lcp_small_d5.npz"))
    engine.set_scene(lcp["scene_xyz"], lcp["scene_nrm"], 0.005)
    engine.set_model(0, lcp["model_xyz"], lcp["model_nrm"])
    # the bitmap+rank table (8 bytes per 32 cells) is larger than the 216 KB shared-memory plan: count mode reads it through L1
    assert engine.grid_info()["n_cells"] // 4 > 216 * 1024
    counts, _ = engine.score_lcp(0, lcp["T"], "count")
    assert np.array_equal(counts, d5["counts"])
    _, ws = engine.score_lcp(0, lcp["T"], "weighted")
    assert np.array_equal(ws, d5["weighted_score"])


def _pairset(a):
    a = np.asarray(a).reshape(-1, a.shape[-1])
    return set(map(tuple, a.tolist()))


def test_pcs_golden(engine):
    g = np.load(os.path.join(G, "pcs_small.npz"))
    delta = float(g["delta"])
    engine.set_scene(g["scene_xyz"], g["scene_nrm"], delta)
    engine.set_model(0, g["model_xyz"], g["model_nrm"])
    for k, (b, inv) in enumerate(zip(g["bases"], g["invariants"])):
        p1 = engine.extract_pairs(0, float(g[f"b{k}_d1"]), delta)
        p2 = engine.extract_pairs(0, float(g[f"b{k}_d2"]), delta)
        assert _pairset(p1) == _pairset(g[f"b{k}_p1"])                 # pair SETS equal MatchSuper4PCS::ExtractPairs
        assert _pairset(p2) == _pairset(g[f"b{k}_p2"])
        # the join is fed the reference's own pair lists so that only the join is under test
        q = engine.find_quads(0, b, inv[0], inv[1], delta, g[f"b{k}_p1"], g[f"b{k}_p2"])
        # quad SETS equal MatchSuper4PCS::FindCongruentQuadrilaterals: the reference's quantised join (power-of-two position
        # grid, 7^3 direction grid, rasterised cone) is reproduced cell for cell -- index work, exact
        ours, ref = _pairset(q), _pairset(g[f"b{k}_quads"])
        assert ours == ref, (k, sorted(ours - ref)[:5], sorted(ref - ours)[:5])
        # rigid transforms of the reference's first quads
        nq = len(g[f"b{k}_T"])
        T, ok = engine.rigid_from_quads(0, b, g[f"b{k}_quads"][:nq])
        assert np.array_equal(ok, g[f"b{k}_ok"])
        assert np.allclose(T, g[f"b{k}_T"], atol=5e-6)                 # fp32 frame alignment, not bit-pinned (Eigen association)
        pose = engine.centred_to_pose(0, T)
        assert np.allclose(pose, g[f"b{k}_pose"], atol=1e-5)


def test_mode0_join_equals_reference_live(engine):
    """The same check against the reference engine itself (oracle/_ref/libs4ref.so travels to the GPU box as a built file), on
    bases and pair lists the golden file does not hold: for every base the reference's SelectQuadrilateral draws, its
    ExtractPairs lists go through both joins; the quad sets must be identical, every differing quad is printed."""
    from oracle import pyoracle
    from physimglobalpose_b200 import synth
    if not pyoracle.have_ref():
        pytest.skip("oracle/_ref/libs4ref.so not built")
    prob = synth.make_segment_problem(700, 900, 0.005, seed=31)
    engine.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    engine.set_model(0, prob.model_xyz, prob.model_nrm)
    ref = pyoracle.RefOracle(prob.scene_xyz, prob.scene_nrm, prob.model_xyz, prob.model_nrm, prob.model_xyz, prob.model_nrm, prob.delta)
    P = prob.scene_xyz - engine.centroids(0)[0]
    n_bases = n_quads = 0
    diffs = []
    for seed in range(1, 40):
        ok, b, inv = ref.select_quadrilateral(seed)
        if not ok:
            continue
        d1 = float(np.linalg.norm((P[b[0]] - P[b[1]]).astype(np.float32)))
        d2 = float(np.linalg.norm((P[b[2]] - P[b[3]]).astype(np.float32)))
        p1, p2 = ref.extract_pairs(d1, prob.delta), ref.extract_pairs(d2, prob.delta)
        if len(p1) == 0 or len(p2) == 0:
            continue
        want = _pairset(ref.find_quads(b, float(inv[0]), float(inv[1]), prob.delta, p1, p2))
        got = _pairset(engine.find_quads(0, b, float(inv[0]), float(inv[1]), prob.delta, p1, p2))
        n_bases += 1; n_quads += len(want)
        if got != want:
            diffs.append((seed, sorted(got - want)[:8], sorted(want - got)[:8]))
    assert n_bases >= 10 and n_quads > 1000, (n_bases, n_quads)
    assert not diffs, diffs


def test_stocs_golden(engine):
    """operMode 1, the generator the reference ships: computePPF keys, the PPF-map builder, SelectQuadrilateralStoCS (with the
    reference's own std::default_random_engine + std::discrete_distribution draw reproduced for a pinned engine seed) and the
    mode-1 congruent sets, against vectors minted from the compiled reference (tests/golden/make_golden.py::mint_stocs)."""
    g = np.load(os.path.join(G, "stocs_small.npz"))
    delta = float(g["delta"])
    engine.set_scene(g["scene_xyz"], g["scene_nrm"], delta)
    engine.set_model(0, g["model_xyz"], g["model_nrm"])
    assert np.array_equal(engine.scene_ppf_keys(g["scene_pairs"]), g["scene_keys"])          # computePPF, bit-exact bins
    # the builder the reference lacks == the reference's computePPF over all ordered model pairs
    engine.build_ppf_map(0)
    keys, offs, pairs = engine.get_ppf_map(0)
    assert np.array_equal(keys, g["map_keys"]) and np.array_equal(offs, g["map_offsets"]) and np.array_equal(pairs, g["map_pairs"])
    # the same map handed over the way the ROS node does (PPFMap argument)
    engine.set_ppf_map(0, g["map_keys"], g["map_offsets"], g["map_pairs"])
    n_bases = len(g["base_ok"])
    n = engine.generate_pcs(0, seed=int(g["user_seed"]), max_hyp=1_000_000, n_bases=n_bases, max_quads_per_base=0, mode=1)
    ids, inv, ok = engine.get_bases(0)
    assert np.array_equal(ok, g["base_ok"])
    assert np.array_equal(ids, g["base_ids"])                    # same four points, same pairing
    assert np.array_equal(inv, g["base_inv"])                    # same invariants, bit for bit
    # congruent sets of the bases the golden file holds: pair lists = map rows of the two base edges
    rows = {tuple(k): (int(a), int(b)) for k, a, b in zip(g["map_keys"].tolist(), g["map_offsets"][:-1], g["map_offsets"][1:])}
    total = 0
    for name in g.files:
        if not name.startswith("quads_b"):
            continue
        b = int(name[len("quads_b"):])
        k1 = tuple(engine.scene_ppf_keys([[ids[b, 0], ids[b, 1]]])[0].tolist())
        k2 = tuple(engine.scene_ppf_keys([[ids[b, 2], ids[b, 3]]])[0].tolist())
        p1 = g["map_pairs"][rows[k1][0]:rows[k1][1]]
        p2 = g["map_pairs"][rows[k2][0]:rows[k2][1]]
        q = engine.find_quads(0, ids[b], inv[b, 0], inv[b, 1], delta, p1, p2)
        assert _pairset(q) == _pairset(g[name])
        total += len(q)
    assert total > 0 and n > 0
    # and the generated batch scores like any other
    engine.score_generated(0, "weighted")
    T, counts, scores = engine.get_generated(0)
    assert len(T) == n and scores.max() > 0


def _c1_mask(g, name):
    edges = g[f"{name}_mask_rle"]
    flat = np.zeros(480 * 640 + 1, np.int8)
    np.add.at(flat, edges[0::2], 1)
    np.add.at(flat, edges[1::2], -1)
    return (np.cumsum(flat)[:-1] > 0).reshape(480, 640)


def test_c1_test_scene_golden(engine):
    """configs[0] of BASELINE.json: the reference's own test-scene (frame-000000 + mask.png), three objects.  On the prepared
    segment clouds the CUDA path must give the reference's numbers for the reference's own hypotheses: priors from the mask
    image, inlier counts, weighted scores, and therefore the same arg-max pose."""
    g = np.load(os.path.join(G, "c1_test_scene.npz"))
    for name in g["names"]:
        engine.set_scene(g[f"{name}_seg_xyz"], g[f"{name}_seg_nrm"], float(g["delta"]))
        engine.set_scene_prior_image(np.where(_c1_mask(g, name), 10000, 0).astype(np.uint16), g["K"])
        assert np.array_equal(engine.scene_priors(), g[f"{name}_priors"])
        engine.set_model(0, g[f"{name}_model_xyz"], g[f"{name}_model_nrm"])
        T = g[f"{name}_T"]
        counts, _ = engine.score_lcp(0, T, "count")
        assert np.array_equal(counts, g[f"{name}_counts"])
        wn, ws = engine.score_lcp(0, T, "weighted")
        assert np.array_equal(ws, g[f"{name}_wscore"]) and np.array_equal(wn, g[f"{name}_wnreg"].astype(np.uint32))
        top = engine.topk(0, 1)
        assert top["index"][0] == int(np.lexsort((np.arange(len(ws)), -ws))[0])
        # our own generator on the same clouds reaches a comparable best score (different RNG, same algorithm)
        engine.generate_pcs(0, seed=7, max_hyp=20000)
        engine.score_generated(0, "weighted")
        assert engine.topk(0, 1)["score"][0] >= 0.6 * ws.max()


C1_CLASSES = {"kleenex_tissue_box": 8, "expo_dry_erase_board_eraser": 2, "folgers_classic_roast_coffee": 3}


def test_segment_preparation_on_device(engine):
    """K7 (depth decode, mask, back-projection, 1 cm voxel centroids, PCA normals, radius-outlier removal) on the test-scene frame
    against the numpy restatement the configs[0] fixture was prepared with: same pixel count, same points bit for bit, same
    normals (the eigenvector of a nearly isotropic neighbourhood is ill-conditioned, hence a tolerance on a few of them); and the
    device-prepared segment scores exactly like the fixture's."""
    g = np.load(os.path.join(G, "c1_test_scene.npz"))
    raw = np.repeat(g["depth_raw_rle"][0], g["depth_raw_rle"][1]).astype(np.uint16).reshape(480, 640)
    mask = np.repeat(g["mask_all_rle"][0], g["mask_all_rle"][1]).astype(np.uint8).reshape(480, 640)
    engine.set_option("k7_mls", 0)                      # the fixture was prepared with the PCA-normal variant
    for name in g["names"]:
        xyz, nrm, n_raw = engine.prepare_segment(raw, mask, C1_CLASSES[str(name)], g["K"])
        want_xyz, want_nrm = g[f"{name}_seg_xyz"], g[f"{name}_seg_nrm"]
        assert n_raw == int(g[f"{name}_n_raw"])
        assert xyz.shape == want_xyz.shape
        assert np.array_equal(xyz, want_xyz)
        cosang = np.einsum("ij,ij->i", nrm.astype(np.float64), want_nrm.astype(np.float64))
        assert np.all(np.abs(np.linalg.norm(nrm, axis=1) - 1) < 1e-6)
        assert (cosang > 1 - 1e-6).mean() > 0.98 and cosang.min() > 0.99, (cosang.min(), (cosang > 1 - 1e-6).mean())     # fp32 unit vectors
    # a class that is not in the mask: empty segment, no error
    xyz, nrm, n_raw = engine.prepare_segment(raw, mask, 77, g["K"])
    assert len(xyz) == 0 and n_raw == 0
    engine.set_option("k7_mls", 1)


def test_segment_preparation_mls_on_device(engine):
    """K7 in its default mode -- pcl::MovingLeastSquares as the reference configures it (polynomial fit of order 2 + normals,
    PPE/src/segmentation/Segmentation.cpp:231-238), then the radius-outlier filter on the PROJECTED cloud
    (ObjectPoseCandidateSet.cpp:28-32) -- against the numpy restatement oracle/segment_port.py::mls_project on the test-scene frame:
    same points kept, projected positions equal to 1e-6 m, normals to fp32 rounding (both sides solve the same 6x6 normal equations in
    double; PCL itself is not available: parity with PCL is unpinned)."""
    from oracle import segment_port
    g = np.load(os.path.join(G, "c1_test_scene.npz"))
    raw = np.repeat(g["depth_raw_rle"][0], g["depth_raw_rle"][1]).astype(np.uint16).reshape(480, 640)
    mask = np.repeat(g["mask_all_rle"][0], g["mask_all_rle"][1]).astype(np.uint8).reshape(480, 640)
    dec = segment_port.decode_depth(raw)
    engine.set_option("k7_mls", 1)
    for name in g["names"]:
        cls = C1_CLASSES[str(name)]
        xyz, nrm, n_raw = engine.prepare_segment(raw, mask, cls, g["K"])
        want_xyz, want_nrm, want_raw = segment_port.prepare_segment(dec, mask, cls, g["K"], mls=True)
        assert n_raw == want_raw
        assert xyz.shape == want_xyz.shape, (name, xyz.shape, want_xyz.shape)
        assert np.abs(xyz.astype(np.float64) - want_xyz.astype(np.float64)).max() < 1e-6
        cosang = np.einsum("ij,ij->i", nrm.astype(np.float64), want_nrm.astype(np.float64))
        assert np.all(np.abs(np.linalg.norm(nrm, axis=1) - 1) < 1e-6)
        assert (cosang > 1 - 1e-6).mean() > 0.98 and cosang.min() > 0.99, (name, cosang.min(), (cosang > 1 - 1e-6).mean())     # fp32 unit vectors
        # the projection is a smoothing of the centroids, not a different cloud: every point moved by less than the fit radius
        pca_xyz = g[f"{name}_seg_xyz"]
        from scipy.spatial import cKDTree
        d, _ = cKDTree(pca_xyz).query(xyz)
        assert d.max() < 0.02 and np.median(d) < 0.002


def test_v4pcs_golden(engine):
    """operMode 2: the device's bit-matrix join returns, for the reference's own tetrahedron bases, exactly the quads of the
    reference's ExtractCongruentSet / FindCongruentQuadrilateralsV4PCS (tests/golden/mode2_small.npz), and every quad's rigid
    transform is what pgp_rigid_from_quads gives for the operMode-0 path (same function of the reference)."""
    g = np.load(os.path.join(G, "mode2_small.npz"))
    engine.set_scene(g["scene_xyz"], g["scene_nrm"], float(g["delta"]))
    engine.set_model(0, g["model_xyz"], g["model_nrm"])
    offs = g["quad_offsets"]
    for k, b in enumerate(g["bases"]):
        want = g["quads"][offs[k]:offs[k + 1]]
        got = engine.find_quads_v4pcs(0, b, float(g["delta"]))
        assert np.array_equal(got, want)


def test_generate_v4pcs_finds_the_pose(engine, port_lib):
    """pgp_generate_pcs in operMode 2 end to end on a segment problem: tetrahedron bases -> quads -> rigid transforms.  The
    best-scoring hypothesis reaches (most of) the LCP of the ground-truth pose -- the objective the search maximises; a partial
    view of a box admits other alignments of the same quality, so the pose itself is not asserted -- the generated transforms are
    rigid, the device scores equal the oracle's, and a seed reproduces the batch bit for bit."""
    from physimglobalpose_b200 import synth
    seg = synth.make_segment_problem(600, 800, 0.005, seed=411)
    engine.set_scene(seg.scene_xyz, seg.scene_nrm, seg.delta)
    engine.set_model(0, seg.model_xyz, seg.model_nrm)
    n = engine.generate_pcs(0, seed=3, max_hyp=20000, n_bases=60, max_quads_per_base=100, mode=2)
    assert n > 100
    T1 = engine.get_generated(0)[0].copy()
    R = T1[:, :, :3].astype(np.float64)
    assert np.allclose(R @ R.transpose(0, 2, 1), np.eye(3), atol=1e-4)
    engine.score_generated(0, "count")
    _, counts, _ = engine.get_generated(0)
    o = port_lib.PortOracle(seg.scene_xyz, seg.scene_nrm, seg.model_xyz, seg.model_nrm, seg.model_xyz, seg.model_nrm, seg.delta)
    assert np.array_equal(counts[:300], o.verify(T1[:300]))
    gt_count = int(o.verify(engine.pose_to_centred(0, seg.gt_pose[None]))[0])
    top = engine.topk(0, 1)
    assert top["count"][0] >= 0.7 * gt_count, (int(top["count"][0]), gt_count)
    n2 = engine.generate_pcs(0, seed=3, max_hyp=20000, n_bases=60, max_quads_per_base=100, mode=2)
    assert n2 == n and np.array_equal(engine.get_generated(0)[0], T1)


def test_lcp_full_shapes_golden(engine):
    """BASELINE configs[1] (2k / 100k) and configs[4] (30k / 300k) at full cloud sizes against numbers minted from the reference
    itself (tests/golden/lcp_full_shapes.npz): inlier counts, weighted scores and gated counts bit for bit."""
    from physimglobalpose_b200 import synth

    def _full_shape(g, tag):          # the clouds and hypotheses come from the seeded generator; the file holds the reference's numbers
        nm, ns, n_hyp, seed_p, seed_t = (int(x) for x in g[f"{tag}_shape"])
        prob = synth.make_problem(nm, ns, 0.01, seed=seed_p)
        T = synth.make_hypotheses(prob, n_hyp, seed=seed_t)
        idx = g[f"{tag}_idx"]
        assert np.array_equal(T[idx[:4]], g[f"{tag}_T_check"])
        return prob, T[idx]

    g = np.load(os.path.join(G, "lcp_full_shapes.npz"))
    for tag in ("c2", "c5"):
        prob, T = _full_shape(g, tag)
        engine.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
        engine.set_model(0, prob.model_xyz, prob.model_nrm)
        counts, _ = engine.score_lcp(0, T, "count")
        assert np.array_equal(counts, g[f"{tag}_counts"])
        wn, ws = engine.score_lcp(0, T, "weighted")
        assert np.array_equal(ws, g[f"{tag}_wscore"]) and np.array_equal(wn, g[f"{tag}_wnreg"].astype(np.uint32))
