"""The float64 restatement of K4d (oracle/select_port.py) on pools with hand-computed answers.  No GPU needed."""
import math

import numpy as np

from oracle.select_port import centred_to_pose, distinct

COS10 = math.cos(math.radians(10.0))
FLIP_Z = np.diag([-1.0, -1.0, 1.0])            # the 180 degree turn of a box about its z axis


def pose(t=(0.0, 0.0, 0.0), R=np.eye(3)):
    T = np.zeros((3, 4), np.float32)
    T[:, :3] = R
    T[:, 3] = t
    return T.reshape(12)


def rot_z(deg):
    c, s = math.cos(math.radians(deg)), math.sin(math.radians(deg))
    return np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])


def run(poses, k=64, max_dist=0.01, cos_angle=COS10, syms=(), index=None):
    T = np.stack(poses)
    idx = np.arange(len(T)) if index is None else np.asarray(index)
    return distinct(T, idx, k, max_dist, cos_angle, syms).tolist()


def test_chain_a_b_c_keeps_c():
    # a suppresses b (8 mm), b would suppress c (8 mm) but b is not kept, and a is 16 mm from c: c stays
    assert run([pose((0, 0, 0)), pose((0.008, 0, 0)), pose((0.016, 0, 0))]) == [0, 2]


def test_only_kept_records_suppress():
    # the same chain with b first: b suppresses a and c
    assert run([pose((0.008, 0, 0)), pose((0, 0, 0)), pose((0.016, 0, 0))]) == [0]


def test_translation_alone_or_rotation_alone_does_not_suppress():
    assert run([pose(), pose((0.02, 0, 0))]) == [0, 1]                 # same rotation, 2 cm apart
    assert run([pose(), pose(R=rot_z(20))]) == [0, 1]                  # same place, 20 degrees apart
    assert run([pose(), pose((0.005, 0, 0), rot_z(5))]) == [0]         # 5 mm and 5 degrees: one placement


def test_early_stop_at_k():
    far = [pose((0.1 * i, 0, 0)) for i in range(6)]
    assert run(far, k=3) == [0, 1, 2]
    assert run(far, k=1) == [0]
    assert run(far, k=64) == list(range(6))


def test_padding_is_skipped():
    # a padding record at a's place neither keeps nor suppresses
    assert run([pose(), pose((0.001, 0, 0)), pose((0.5, 0, 0))], index=[-1, 7, 8]) == [1, 2]
    assert run([pose(), pose()], index=[-1, -1]) == []


def test_nan_records_are_kept_and_suppress_nothing():
    nan_t = pose()
    nan_t[3] = np.nan
    nan_r = pose()
    nan_r[5] = np.nan
    # first: kept, and its twin after it is not suppressed by it
    assert run([nan_t, pose()]) == [0, 1]
    assert run([nan_r, pose()]) == [0, 1]
    # after a clean record at the same place: never suppressed
    assert run([pose(), nan_t, nan_r, pose()]) == [0, 1, 2]


def test_flipped_box_needs_its_symmetry():
    twins = [pose((0.1, 0.2, 0.3)), pose((0.1, 0.2, 0.3), FLIP_Z)]
    assert run(twins) == [0, 1]
    assert run(twins, syms=[FLIP_Z]) == [0]
    # a symmetry that does not map one onto the other changes nothing
    assert run(twins, syms=[np.diag([1.0, -1.0, -1.0])]) == [0, 1]


def test_thresholds_are_inclusive_and_exact():
    # d2 = 25 * 2^-20 exactly, max_dist = 5 * 2^-10: suppressed at equality, not one ulp below
    a, b = pose((0.25, -0.5, 1.0)), pose((0.25 + 3 / 1024, -0.5 + 4 / 1024, 1.0))
    assert run([a, b], max_dist=5 / 1024) == [0]
    assert run([a, b], max_dist=np.nextafter(5 / 1024, 0.0)) == [0, 1]
    # identical rotations give tr = 3: cos_angle = 1 is the threshold itself
    assert run([pose(), pose()], max_dist=0.0, cos_angle=1.0) == [0]
    assert run([pose(), pose()], max_dist=0.0, cos_angle=np.nextafter(1.0, 2.0)) == [0, 1]


def test_centred_to_pose_order():
    T = pose((0.1, 0.2, 0.3), rot_z(30))
    cP, cQ = np.float32([0.5, -0.25, 1.0]), np.float32([0.01, 0.02, -0.03])
    P = centred_to_pose(T, cP, cQ).reshape(4, 4)
    R = T.reshape(3, 4)[:, :3].astype(np.float64)
    for r in range(3):
        t = float(T[4 * r + 3]) + float(cP[r])
        for c in range(3):
            t = t - float(R[r, c]) * float(cQ[c])
        assert P[r, 3] == t
    assert np.array_equal(P[:3, :3], R) and np.array_equal(P[3], [0, 0, 0, 1])
