"""The CPU oracle (oracle/lcp_oracle.c, a plain-C restatement) against the golden vectors minted
from the reference engine itself (tests/golden/make_golden.py), and -- where the reference build
exists (this container) -- against the reference live.  This is what pins the oracle."""
import os

import numpy as np
import pytest

from physimglobalpose_b200 import synth

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def lcp():
    return np.load(os.path.join(G, "lcp_small.npz"))


def _port(port_lib, g, delta=None, **kw):
    return port_lib.PortOracle(g["scene_xyz"], g["scene_nrm"], g["model_xyz"], g["model_nrm"], g["model_xyz"], g["model_nrm"],
                               float(g["delta"]) if delta is None else delta, **kw)


def test_port_lcp_matches_reference_golden(port_lib, lcp):
    o = _port(port_lib, lcp)
    cP, cQ = o.centroids()
    assert np.array_equal(cP, lcp["cP"]) and np.array_equal(cQ, lcp["cQ"])
    assert np.array_equal(o.verify(lcp["T"]), lcp["counts"])
    frac, best = o.verify_running_best(lcp["T"])
    assert best == int(lcp["running_best"]) and np.array_equal(frac, lcp["running_frac"])
    ws, wn, reg = o.weighted_verify(lcp["T"], reg_of=int(lcp["registered_of"]))
    assert np.array_equal(ws, lcp["weighted_score"]) and np.array_equal(wn, lcp["weighted_nreg"])
    assert np.array_equal(reg, lcp["registered"])
    # the improving chain ends at the running best
    chain = o.improving_chain(lcp["counts"].astype(np.float32) / np.float32(len(lcp["model_xyz"])))
    assert chain[-1] == int(lcp["running_best"])


def test_port_priors_and_weighted_with_image(port_lib, lcp):
    o = _port(port_lib, lcp, K=lcp["K"], prior_img=lcp["prior_img"])
    assert np.array_equal(o.priors(), lcp["priors"])
    ws, wn = o.weighted_verify(lcp["T"])
    assert np.array_equal(ws, lcp["weighted_score_img"]) and np.array_equal(wn, lcp["weighted_nreg_img"])


def test_port_delta_5mm(port_lib, lcp):
    d5 = np.load(os.path.join(G, "lcp_small_d5.npz"))
    o = _port(port_lib, lcp, delta=0.005)
    assert np.array_equal(o.verify(lcp["T"]), d5["counts"])
    assert np.array_equal(o.weighted_verify(lcp["T"])[0], d5["weighted_score"])


def test_port_pcs_pieces_match_reference_golden(port_lib):
    g = np.load(os.path.join(G, "pcs_small.npz"))
    o = _port(port_lib, g)
    for k, b in enumerate(g["bases"]):
        for which in ("1", "2"):
            got = o.extract_pairs(float(g[f"b{k}_d{which}"]), float(g["delta"]))
            assert set(map(tuple, got.tolist())) == set(map(tuple, g[f"b{k}_p{which}"].tolist()))
        for quad, T, ok, pose in zip(g[f"b{k}_quads"], g[f"b{k}_T"], g[f"b{k}_ok"], g[f"b{k}_pose"]):
            ok2, T4, P4 = o.rigid_from_quad(b, quad)
            assert ok2 == bool(ok)
            assert np.allclose(T4[:3], T, atol=5e-6) and np.allclose(P4, pose, atol=1e-5)


def test_lcp_invariants(port_lib):
    """Properties the reference's (disabled) tests would assert: identity on a copy -> full count; far
    translation -> 0; monotone in delta."""
    prob = synth.make_segment_problem(300, 600, 0.005, seed=4)
    args = (prob.model_xyz, prob.model_nrm, prob.model_xyz, prob.model_nrm, prob.model_xyz, prob.model_nrm)   # scene := model
    I = np.eye(4)
    T_id = synth.centre_pose(I, synth.seq_centroid_f32(prob.model_xyz), synth.seq_centroid_f32(prob.model_xyz))
    far = I.copy(); far[:3, 3] = 5.0
    T_far = synth.centre_pose(far, synth.seq_centroid_f32(prob.model_xyz), synth.seq_centroid_f32(prob.model_xyz))
    last = None
    for d in (0.001, 0.005, 0.02):
        o = port_lib.PortOracle(*args, d)
        c = o.verify(np.stack([T_id, T_far]))
        assert c[0] == len(prob.model_xyz) and c[1] == 0
        T = synth.make_hypotheses(prob, 32, seed=1)
        cur = port_lib.PortOracle(prob.scene_xyz, prob.scene_nrm, prob.model_xyz, prob.model_nrm, prob.model_xyz, prob.model_nrm, d).verify(T)
        if last is not None:
            assert np.all(cur >= last)
        last = cur


def test_port_equals_reference_live(port_lib, lcp):
    """The C restatement, its multi-threaded CPU-baseline driver included, against the reference's own Verify / WeightedVerify /
    running-best answers stored in lcp_small.npz and lcp_full_shapes.npz; where the reference engine is built (oracle/_ref), also
    against the reference itself on fresh seeded inputs."""
    o = _port(port_lib, lcp)
    assert np.array_equal(o.verify(lcp["T"]), lcp["counts"])
    ws, wn = o.weighted_verify(lcp["T"])
    assert np.array_equal(ws, lcp["weighted_score"]) and np.array_equal(wn, lcp["weighted_nreg"])
    frac, best = o.verify_running_best(lcp["T"])
    assert best == int(lcp["running_best"]) and np.array_equal(frac, lcp["running_frac"])
    assert np.array_equal(o.verify_mt(lcp["T"], 3)[0], lcp["counts"])
    g = np.load(os.path.join(G, "lcp_full_shapes.npz"))
    prob, T = _full_shape(g, "c2")
    full = port_lib.PortOracle(prob.scene_xyz, prob.scene_nrm, prob.model_xyz, prob.model_nrm, prob.model_xyz, prob.model_nrm, prob.delta)
    assert np.array_equal(full.verify_mt(T, 3)[0], g["c2_counts"])
    if not port_lib.have_ref():
        return
    prob = synth.make_problem(400, 9000, 0.01, seed=31)
    T = synth.make_hypotheses(prob, 200, seed=32)
    args = (prob.scene_xyz, prob.scene_nrm, prob.model_xyz, prob.model_nrm, prob.model_xyz, prob.model_nrm, prob.delta)
    ref, port = port_lib.RefOracle(*args), port_lib.PortOracle(*args)
    assert np.array_equal(ref.verify(T), port.verify(T))
    a, b = ref.weighted_verify(T), port.weighted_verify(T)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    fa, ba = ref.verify_running_best(T)
    fb, bb = port.verify_running_best(T)
    assert ba == bb and np.array_equal(fa, fb)
    cm, _ = ref.verify_mt(T, 3)
    assert np.array_equal(cm, ref.verify(T))                       # the multi-thread CPU baseline driver is consistent
    cp, _ = port.verify_mt(T, 3)
    assert np.array_equal(cp, cm)


# ---------------------------------------------------------------- operMode 1 (StoCS + PPF map)
def _stocs_inputs(g):
    from physimglobalpose_b200 import synth
    P = (g["scene_xyz"] - synth.seq_centroid_f32(g["scene_xyz"])).astype(np.float32)
    N = g["scene_nrm"] / np.linalg.norm(g["scene_nrm"], axis=1, keepdims=True)
    return P, N.astype(np.float32)


def test_stocs_port_matches_reference_golden():
    """The numpy restatement of computePPF / SelectQuadrilateralStoCS / TryQuadrilateral (oracle/stocs_port.py) reproduces the
    vectors minted from the compiled reference: same keys, same four points, same pairing, same invariants."""
    from oracle import stocs_port
    from physimglobalpose_b200 import _lib
    g = np.load(os.path.join(G, "stocs_small.npz"))
    P, N = _stocs_inputs(g)
    sp, sk = g["scene_pairs"][:600], g["scene_keys"][:600]
    got = np.array([stocs_port.compute_ppf(P[i], N[i], P[j], N[j]) for i, j in sp])
    assert np.array_equal(got, sk)
    keyset = set(map(tuple, g["map_keys"].tolist()))
    prior = np.ones(len(P), np.float32)
    lib = _lib.load()
    for b in range(8):
        seed = int(lib.pgp_stocs_engine_seed(int(g["user_seed"]), b, int(g["base_attempts"][b])))
        ok, ids, inv = stocs_port.select_stocs(P, N, prior, keyset, seed)
        assert ok == bool(g["base_ok"][b])
        assert np.array_equal(ids, g["base_ids"][b]) and np.array_equal(inv, g["base_inv"][b])
        if g["base_attempts"][b] > 0:       # the attempt before the accepted one fails in the port too
            seed0 = int(lib.pgp_stocs_engine_seed(int(g["user_seed"]), b, int(g["base_attempts"][b]) - 1))
            assert not stocs_port.select_stocs(P, N, prior, keyset, seed0)[0]


def test_stocs_port_equals_reference_live():
    from oracle import pyoracle, stocs_port
    if not pyoracle.have_ref():
        pytest.skip("oracle/_ref not built (needs /root/reference)")
    g = np.load(os.path.join(G, "stocs_small.npz"))
    ref = pyoracle.RefOracle(g["scene_xyz"], g["scene_nrm"], g["model_xyz"], g["model_nrm"], g["model_xyz"], g["model_nrm"], float(g["delta"]))
    ref.set_ppf_map(g["map_keys"], g["map_offsets"], g["map_pairs"])
    P, N = ref.centred(0)
    P0, N0 = _stocs_inputs(g)
    assert np.array_equal(P, P0) and np.allclose(N, N0, atol=1e-6)
    keyset = set(map(tuple, g["map_keys"].tolist()))
    for seed in (11, 12, 13, 14, 15, 16):
        ok, ids, inv = ref.select_stocs(seed)
        ok2, ids2, inv2 = stocs_port.select_stocs(P, N, ref.priors(), keyset, seed)
        assert ok == ok2
        if ok:
            assert np.array_equal(ids, ids2) and np.array_equal(inv, inv2)


# ---------------------------------------------------------------- configs[0]: the reference's test-scene
def test_port_c1_test_scene_matches_reference_golden(port_lib):
    """The C restatement reproduces the reference's Verify / WeightedVerify on the three test-scene objects (segments prepared from
    frame-000000 + mask.png, hypotheses from the reference's own Perform_N_steps; tests/golden/make_c1.py)."""
    g = np.load(os.path.join(G, "c1_test_scene.npz"))
    for name in g["names"]:
        mask = _c1_mask(g, name)
        prior_img = np.where(mask, 10000, 0).astype(np.uint16)
        o = port_lib.PortOracle(g[f"{name}_seg_xyz"], g[f"{name}_seg_nrm"], g[f"{name}_model_xyz"], g[f"{name}_model_nrm"], g[f"{name}_model_xyz"],
                                g[f"{name}_model_nrm"], float(g["delta"]), K=g["K"], prior_img=prior_img)
        assert np.array_equal(o.priors(), g[f"{name}_priors"])
        T = g[f"{name}_T"]
        assert np.array_equal(o.verify(T), g[f"{name}_counts"])
        ws, wn = o.weighted_verify(T)
        assert np.array_equal(ws, g[f"{name}_wscore"]) and np.array_equal(wn, g[f"{name}_wnreg"])


def _c1_mask(g, name):
    edges = g[f"{name}_mask_rle"]
    flat = np.zeros(480 * 640 + 1, np.int8)
    np.add.at(flat, edges[0::2], 1)
    np.add.at(flat, edges[1::2], -1)
    return (np.cumsum(flat)[:-1] > 0).reshape(480, 640)


C1_CLASSES = {"kleenex_tissue_box": 8, "expo_dry_erase_board_eraser": 2, "folgers_classic_roast_coffee": 3}     # gt_info.yml / obj_config.yml


def _c1_images(g):
    raw = np.repeat(g["depth_raw_rle"][0], g["depth_raw_rle"][1]).astype(np.uint16).reshape(480, 640)
    mask = np.repeat(g["mask_all_rle"][0], g["mask_all_rle"][1]).astype(np.uint8).reshape(480, 640)
    return raw, mask


def test_segment_port_reproduces_the_fixture_clouds():
    """The segment-preparation restatement (oracle/segment_port.py), run on the test-scene's depth + mask images stored in the
    fixture, yields exactly the segment clouds the configs[0] vectors were minted on; the bit-twiddled depth decode matches the
    stored crop."""
    from oracle import segment_port
    g = np.load(os.path.join(G, "c1_test_scene.npz"))
    raw, mask = _c1_images(g)
    assert np.array_equal(raw[200:216, 300:316], g["depth_raw_crop"])
    dec = segment_port.decode_depth(raw)
    assert np.array_equal((dec[200:216, 300:316] * np.float32(10000)).round().astype(np.uint16), g["depth_dec_crop"])
    for name in g["names"]:
        xyz, nrm, n_raw = segment_port.prepare_segment(dec, mask, C1_CLASSES[str(name)], g["K"])
        assert n_raw == int(g[f"{name}_n_raw"])
        assert np.array_equal(xyz, g[f"{name}_seg_xyz"]) and np.array_equal(nrm, g[f"{name}_seg_nrm"])


# ---------------------------------------------------------------- operMode 2 (V4PCS)
def test_v4pcs_port_matches_reference_golden():
    """The numpy restatement of ExtractCongruentSet in operMode 2 (six pair extractions + FindCongruentQuadrilateralsV4PCS,
    match4pcsBase.cc:978-1044,1929-2039) gives the reference's quads for the reference's own tetrahedron bases
    (tests/golden/mode2_small.npz, minted from oracle/_ref); live against the reference too where it is built."""
    from oracle import pyoracle
    from physimglobalpose_b200 import synth
    g = np.load(os.path.join(G, "mode2_small.npz"))
    cP = synth.seq_centroid_f32(g["scene_xyz"]); cQ = synth.seq_centroid_f32(g["model_xyz"])
    P = (g["scene_xyz"] - cP).astype(np.float32); Q = (g["model_xyz"] - cQ).astype(np.float32)
    offs = g["quad_offsets"]
    for k, b in enumerate(g["bases"]):
        want = g["quads"][offs[k]:offs[k + 1]]
        got = pyoracle.v4pcs_quads_port(P, Q, b, float(g["delta"]))
        assert np.array_equal(got, want)
    if pyoracle.have_ref():
        ref = pyoracle.RefOracle(g["scene_xyz"], g["scene_nrm"], g["model_xyz"], g["model_nrm"], g["model_xyz"], g["model_nrm"], float(g["delta"]))
        assert np.array_equal(ref.centred(0)[0], P) and np.array_equal(ref.centred(1)[0], Q)
        for seed in (21, 22, 23):
            ok, b = ref.select_tetrahedron(seed)
            assert ok
            q = ref.congruent_set_mode2(b)
            assert len(set(map(tuple, q.tolist()))) == len(q)
            assert np.array_equal(np.array(sorted(map(tuple, q.tolist())), np.int32).reshape(-1, 4), pyoracle.v4pcs_quads_port(P, Q, b, float(g["delta"])))


# ---------------------------------------------------------------- full-size shapes (configs[1], configs[4])
def _full_shape(g, tag):
    from physimglobalpose_b200 import synth
    nm, ns, n_hyp, seed_p, seed_t = (int(x) for x in g[f"{tag}_shape"])
    prob = synth.make_problem(nm, ns, 0.01, seed=seed_p)
    T = synth.make_hypotheses(prob, n_hyp, seed=seed_t)
    idx = g[f"{tag}_idx"]
    assert np.array_equal(T[idx[:4]], g[f"{tag}_T_check"])      # the seeded generator reproduces the hypotheses the vectors were minted on
    return prob, T[idx]


def test_port_matches_reference_golden_at_full_shapes(port_lib):
    """The C restatement against the reference's own Verify / WeightedVerify at the FULL cloud sizes of BASELINE configs[1]
    (2k / 100k) and configs[4] (30k / 300k): tests/golden/lcp_full_shapes.npz holds the reference's numbers for a hypothesis sample
    spread over the benchmark's batch; the clouds are regenerated from the seeded generator."""
    g = np.load(os.path.join(G, "lcp_full_shapes.npz"))
    for tag, n_w in (("c2", 400), ("c5", 24)):
        prob, T = _full_shape(g, tag)
        o = port_lib.PortOracle(prob.scene_xyz, prob.scene_nrm, prob.model_xyz, prob.model_nrm, prob.model_xyz, prob.model_nrm, prob.delta)
        assert np.array_equal(o.verify(T), g[f"{tag}_counts"])
        ws, wn = o.weighted_verify(T[:n_w])
        assert np.array_equal(ws, g[f"{tag}_wscore"][:n_w]) and np.array_equal(wn, g[f"{tag}_wnreg"][:n_w])


def test_mls_restatement_smooths_and_fits_known_surfaces():
    from oracle import segment_port
    """oracle/segment_port.py::mls_project (pcl::MovingLeastSquares with polynomial fit, restated; the checker of K7): on a plane
    the projection removes the noise component along the normal and returns the plane's normal; on a sphere patch -- a surface an
    order-2 polynomial follows -- the projected points lie closer to the sphere than the input and the normals closer to the
    radial direction than plain PCA normals; isolated points vanish."""
    rng = np.random.default_rng(0)
    # plane z = 0.6 + 0.2 x, noise along z
    xy = rng.uniform(-0.1, 0.1, size=(1500, 2))
    z = 0.6 + 0.2 * xy[:, 0] + rng.normal(0, 5e-4, 1500)
    pts = np.column_stack([xy, z]).astype(np.float32)
    pts = np.vstack([pts, np.array([[0.5, 0.5, 0.9]], dtype=np.float32)])          # one isolated point
    P, N, V = segment_port.mls_project(pts, 0.02)
    assert V[:-1].all() and not V[-1]
    n_true = np.array([0.2, 0.0, -1.0]) / np.linalg.norm([0.2, 0.0, -1.0])         # towards the camera at the origin
    inner = (np.abs(pts[:-1, 0]) < 0.07) & (np.abs(pts[:-1, 1]) < 0.07)
    res_in = np.abs(pts[:-1, 2] - (0.6 + 0.2 * pts[:-1, 0]))[inner]
    res_out = np.abs(P[:-1, 2] - (0.6 + 0.2 * P[:-1, 0]))[inner]
    assert np.sqrt((res_out ** 2).mean()) < 0.5 * np.sqrt((res_in ** 2).mean())
    assert (N[:-1][inner] @ n_true).min() > np.cos(np.radians(5.0))
    assert ((P[:-1] * N[:-1]).sum(axis=1) <= 0).all()                              # oriented to the camera
    # sphere patch
    th, ph = rng.uniform(0, 0.6, 3000), rng.uniform(0, 2 * np.pi, 3000)
    d = np.stack([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), -np.cos(th)], axis=1)
    ctr = np.array([0, 0, 0.7])
    cen = segment_port.voxel_centroids((ctr + d * (0.1 + rng.normal(0, 7e-4, 3000))[:, None]).astype(np.float32), 0.005)
    P, N, V = segment_port.mls_project(cen, 0.02)
    assert V.all()
    r_in = np.linalg.norm(cen - ctr, axis=1) - 0.1
    r_out = np.linalg.norm(P - ctr, axis=1) - 0.1
    assert np.sqrt((r_out ** 2).mean()) < 0.5 * np.sqrt((r_in ** 2).mean())
    rad = (P - ctr) / np.linalg.norm(P - ctr, axis=1, keepdims=True)
    ang_mls = np.degrees(np.arccos(np.clip(np.abs((rad * N).sum(axis=1)), 0, 1)))
    radc = (cen - ctr) / np.linalg.norm(cen - ctr, axis=1, keepdims=True)
    ang_pca = np.degrees(np.arccos(np.clip(np.abs((radc * segment_port.pca_normals(cen, 0.02)).sum(axis=1)), 0, 1)))
    assert np.median(ang_mls) < np.median(ang_pca)
