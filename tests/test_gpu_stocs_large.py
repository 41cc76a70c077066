"""StoCS base selection (operMode 1) on either side of the scene size at which the weight vectors leave shared memory.

k2s_select_bases keeps one base's weights (n floats + n doubles) in shared memory while n * 12 + 16 <= 200 KB, i.e. for scenes of
up to 17 065 points, and in global memory beyond.  Both placements must reproduce SelectQuadrilateralStoCS + TryQuadrilateral
(oracle/stocs_port.py) for the engine seed of every (base, attempt): the same acceptance, four points, pairing and invariants,
bit for bit.  The port is plain Python (about a second per attempt at this size), so only a few bases are drawn."""
import numpy as np
import pytest

from physimglobalpose_b200 import synth

pytestmark = pytest.mark.gpu

SHARED_MAX = 17065           # largest scene whose weights fit the 200 KB of dynamic shared memory
N_BASES = 4
SEED = 29


@pytest.fixture(scope="module", params=[SHARED_MAX, SHARED_MAX + 2935], ids=["shared", "global"])
def scene(request):
    prob = synth.make_segment_problem(300, request.param, 0.005, seed=41)
    assert len(prob.scene_xyz) == request.param
    return prob


def _stocs_inputs(prob):
    P = (prob.scene_xyz - synth.seq_centroid_f32(prob.scene_xyz)).astype(np.float32)
    N = prob.scene_nrm / np.linalg.norm(prob.scene_nrm, axis=1, keepdims=True)
    return P, N.astype(np.float32)


def test_stocs_bases_equal_port(engine, scene):
    from oracle import stocs_port
    engine.set_scene(scene.scene_xyz, scene.scene_nrm, scene.delta)
    engine.set_scene_priors(np.ones(len(scene.scene_xyz), np.float32))
    engine.set_model(0, scene.model_xyz, scene.model_nrm)
    engine.build_ppf_map(0)
    keys, _, _ = engine.get_ppf_map(0)
    keyset = set(map(tuple, keys.tolist()))
    engine.generate_pcs(0, seed=SEED, max_hyp=1000, n_bases=N_BASES, max_quads_per_base=0, mode=1)
    ids, inv, ok = engine.get_bases(0)
    assert len(ok) == N_BASES
    P, N = _stocs_inputs(scene)
    prior = np.ones(len(P), np.float32)
    for b in range(N_BASES):
        want_ok, want_ids, want_inv = False, None, None
        for a in range(16):                       # the device re-draws up to 16 times, with the engine seed of each attempt
            want_ok, want_ids, want_inv = stocs_port.select_stocs(P, N, prior, keyset, engine.stocs_engine_seed(SEED, b, a))
            if want_ok:
                break
        assert ok[b] == want_ok, b
        if want_ok:
            assert np.array_equal(ids[b], want_ids), (b, ids[b], want_ids)
            assert np.array_equal(inv[b], want_inv), (b, inv[b], want_inv)
    assert ok.any()
