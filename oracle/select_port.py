"""float64 restatement of K4d (pgp_distinct_dev, pgp_topk_distinct): greedy non-maximum suppression in pose space.

The contract of include/pgp.h, operation for operation.  numpy applies every elementwise operation on its own and rounds it once
(no fused multiply-add), and every sum below is written out in the contract's order, so the answers are bitwise the kernel's.

    distinct(pool_T12, pool_index, k, max_dist, cos_angle, syms) -> positions of the kept records in the pool, in pool order
"""
from __future__ import annotations

import numpy as np


def _suppressed_by(a: np.ndarray, B: np.ndarray, max_d2: float, min_tr: float, syms: np.ndarray) -> np.ndarray:
    """Which rows of B (n x 12 fp32) the record a (12 fp32) suppresses."""
    a = a.astype(np.float64)
    B = B.astype(np.float64)
    dx, dy, dz = a[3] - B[:, 3], a[7] - B[:, 7], a[11] - B[:, 11]
    d2 = (dx * dx + dy * dy) + dz * dz
    near = d2 <= max_d2
    Ra = a[[0, 1, 2, 4, 5, 6, 8, 9, 10]]
    Rb = B[:, [0, 1, 2, 4, 5, 6, 8, 9, 10]]

    def trace(G):
        tr = Ra[0] * G[:, 0]
        for e in range(1, 9):
            tr = tr + Ra[e] * G[:, e]
        return tr

    hit = trace(Rb) >= min_tr
    for S in syms:
        G = np.empty_like(Rb)
        for r in range(3):
            for c in range(3):
                G[:, 3 * r + c] = (Rb[:, 3 * r] * S[0, c] + Rb[:, 3 * r + 1] * S[1, c]) + Rb[:, 3 * r + 2] * S[2, c]
        hit |= trace(G) >= min_tr
    return near & hit


def distinct(pool_T12, pool_index, k: int, max_dist: float, cos_angle: float, syms=()) -> np.ndarray:
    """Sequential greedy walk: record i is kept iff no earlier kept record suppresses it; stops after k are kept; records with
    index < 0 are skipped.  pool_T12: m x 12 fp32 centred transforms; syms: n x 3 x 3 (row-major) symmetries, the identity implied.
    Returns the kept positions (int64)."""
    T = np.ascontiguousarray(pool_T12, np.float32).reshape(-1, 12)
    idx = np.asarray(pool_index, np.int64).reshape(-1)
    S = np.asarray(syms, np.float64).reshape(-1, 3, 3)
    max_d2 = float(max_dist) * float(max_dist)
    min_tr = 1.0 + 2.0 * float(cos_angle)
    m = len(T)
    removed = np.zeros(m, bool)
    kept = []
    for i in range(m):
        if len(kept) == k:
            break
        if idx[i] < 0 or removed[i]:
            continue
        kept.append(i)
        if i + 1 < m:
            with np.errstate(all="ignore"):          # NaN / Inf entries: the comparisons decide, as on the device
                removed[i + 1:] |= _suppressed_by(T[i], T[i + 1:], max_d2, min_tr, S)
    return np.asarray(kept, np.int64)


def centred_to_pose(T12, cP, cQ) -> np.ndarray:
    """pgp_centred_to_pose in float64: rotation unchanged, translation ((t_c + c_P) - R_0 c_Q,0) - R_1 c_Q,1 - R_2 c_Q,2."""
    T = np.asarray(T12, np.float32).reshape(-1, 12).astype(np.float64)
    cP = np.asarray(cP, np.float32).astype(np.float64)
    cQ = np.asarray(cQ, np.float32).astype(np.float64)
    P = np.zeros((len(T), 16))
    for r in range(3):
        t = T[:, 4 * r + 3] + cP[r]
        for c in range(3):
            P[:, 4 * r + c] = T[:, 4 * r + c]
            t = t - T[:, 4 * r + c] * cQ[c]
        P[:, 4 * r + 3] = t
    P[:, 15] = 1.0
    return P
