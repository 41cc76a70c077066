"""K3's exact test in AMBIG voxels whose candidate lists run past the two records each voxel keeps inline in its 32-byte slot.

Every scene point is present three times at the same coordinates.  Equal points are never dominated, and a closer point cannot
dominate the closest-so-far, so all three copies of a voxel's closest point are kept: every AMBIG voxel has n >= 3 candidates, its
slot holds two copies of the closest point, and any hit on another scene point has to come from the overflow records."""
import numpy as np
import pytest

from physimglobalpose_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def tripled_problem():
    prob = synth.make_problem(800, 30000, 0.01, seed=71)
    xyz = np.ascontiguousarray(np.repeat(prob.scene_xyz, 3, axis=0))
    nrm = np.ascontiguousarray(np.repeat(prob.scene_nrm, 3, axis=0))
    T = synth.make_hypotheses(prob, 3000, seed=72)
    return prob, xyz, nrm, T


@pytest.fixture(scope="module")
def tripled_oracle(port_lib, tripled_problem):
    prob, xyz, nrm, _ = tripled_problem
    cls = port_lib.RefOracle if port_lib.have_ref() else port_lib.PortOracle
    return cls(xyz, nrm, prob.model_xyz, prob.model_nrm, prob.model_xyz, prob.model_nrm, prob.delta)


def _setup(engine, tripled_problem):
    prob, xyz, nrm, T = tripled_problem
    engine.set_scene(xyz, nrm, prob.delta)
    engine.set_model(0, prob.model_xyz, prob.model_nrm)
    return T


def test_overflow_records_are_built(engine, tripled_problem):
    _setup(engine, tripled_problem)
    st = engine.label_stats()
    assert st["voxels_ambig"] > 0
    # n >= 3 candidates in every AMBIG voxel: at least one overflow record each
    assert st["ambig_overflow_records"] >= st["voxels_ambig"]


def test_count_mode_equals_coarse_path_and_oracle(engine, tripled_problem, tripled_oracle):
    T = _setup(engine, tripled_problem)
    want = tripled_oracle.verify(T)
    fine, _ = engine.score_lcp(0, T, "count")
    engine.set_option("force_coarse", 1)
    try:
        coarse, _ = engine.score_lcp(0, T, "count")
    finally:
        engine.set_option("force_coarse", 0)
    assert np.array_equal(coarse, want)
    assert np.array_equal(fine, want)
    assert want.max() > 0


def test_weighted_mode_equals_oracle(engine, tripled_problem, tripled_oracle):
    T = _setup(engine, tripled_problem)
    ws, wn = tripled_oracle.weighted_verify(T)
    counts, scores = engine.score_lcp(0, T, "weighted")
    assert np.array_equal(counts, wn.astype(np.uint32))
    assert np.array_equal(scores, ws)
