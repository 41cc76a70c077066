"""Host-side checks that need no GPU: the C ABI library loads and exports every symbol
include/pgp.h declares, fails loudly without a device, and the host logic (shard ranges, top-k
merge, pose conversions of the synthetic generator) behaves."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from physimglobalpose_b200 import _lib, sharding, synth
from physimglobalpose_b200.engine import HYP_DTYPE, PoseEngine, exchange_merge, topk_merge, wire_block

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return _lib.load()


def test_every_declared_symbol_is_exported(lib):
    hdr = open(os.path.join(ROOT, "include", "pgp.h")).read()
    declared = set(re.findall(r"PGP_API\s+[\w\s\*]+?\b(pgp_\w+)\s*\(", hdr))
    assert len(declared) >= 30
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in pgp.h but not exported by libpgp.so"
    assert declared == set(_lib.exported_symbols()), declared ^ set(_lib.exported_symbols())
    assert b"sm_100a" in lib.pgp_version()


def test_no_silent_cpu_fallback(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(_lib.PgpError) as e:
        PoseEngine(0)
    assert "no CPU path" in str(e.value) or "CUDA" in str(e.value)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "physimglobalpose_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cc", ".h")):
                src = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "import oracle" not in src and "from oracle" not in src and "lcp_oracle" not in src, os.path.join(dirpath, f)


def test_shard_ranges_cover_exactly():
    for n in (0, 1, 7, 100_000, 1_000_003):
        for world in (1, 2, 3, 8):
            rs = [sharding.shard_range(n, r, world) for r in range(world)]
            assert rs[0][0] == 0 and rs[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(rs, rs[1:]))
            sizes = [hi - lo for lo, hi in rs]
            assert max(sizes) - min(sizes) <= 1


def _records(rng, n, base):
    r = np.zeros(n, HYP_DTYPE)
    r["index"] = base + rng.permutation(n)
    r["count"] = rng.integers(0, 50, size=n)
    r["score"] = r["count"].astype(np.float32) / np.float32(50)
    r["T"] = rng.normal(size=(n, 12)).astype(np.float32)
    return r


def _signed_records(rng, n, base):
    """Scores with negative values, -0.0 and +0.0 (priors may be negative): many ties, zeros of both signs tie."""
    r = _records(rng, n, base)
    r["score"] = rng.choice(np.array([-1.5, -0.25, -1e-30, -0.0, 0.0, 1e-30, 0.25, 1.5], np.float32), size=n)
    return r


def _fp32_order(rec):
    """(score desc, index asc) with scores compared as fp32 values: -0 == +0, the index decides."""
    s = rec["score"].astype(np.float64)
    s[s == 0] = 0.0
    return np.lexsort((rec["index"], -s))


def test_topk_merge_is_independent_of_the_sharding(lib):
    for make in (_records, _signed_records):
        rng = np.random.default_rng(0)
        allrec = make(rng, 4000, 0)
        want = allrec[_fp32_order(allrec)][:64]
        for world in (1, 2, 4, 8):
            lists = []
            for r in range(world):
                lo, hi = sharding.shard_range(len(allrec), r, world)
                part = allrec[lo:hi]
                lists.append(part[_fp32_order(part)][:64])
            got = topk_merge(lists, 64)
            assert got.tobytes() == want.tobytes(), make.__name__
    # short lists are padded with index = -1 and skipped
    got = topk_merge([allrec[:3], allrec[3:5]], 64)
    assert len(got) == 5


def test_exchange_merge_orders_signed_scores_like_the_serial_scan(lib):
    """WEIGHTED records with negative, -0.0 and +0.0 scores: the merged top-k is the fp32 order over the union, and the merged
    chain is the serial scan over the concatenation (best starts at 0, strict '>': a score <= 0 never enters)."""
    rng = np.random.default_rng(4)
    allrec = _signed_records(rng, 3000, 0)
    allrec["index"] = np.arange(len(allrec))                              # generation order: the chain scans it
    allrec["score"][:40] = -np.arange(1, 41, dtype=np.float32)          # a negative prefix: a positive score later still enters
    rise = np.sort(rng.choice(np.arange(40, 3000), 30, replace=False))
    allrec["score"][rise] = np.arange(2, 32, dtype=np.float32)
    want = allrec[_fp32_order(allrec)][:64]
    best, keep = np.float32(0), []
    for i, s in enumerate(allrec["score"]):
        if s > best:
            keep.append(i)
            best = s
    want_chain = allrec[keep]
    assert len(want_chain) >= 30 and np.all(want_chain["score"] > 0)
    for world in (1, 2, 3, 8):
        blocks, chains = [], []
        for r in range(world):
            lo, hi = sharding.shard_range(len(allrec), r, world)
            part = allrec[lo:hi].copy()
            part["index"] -= lo                                              # shard-local indices: auto_base numbers them
            blocks.append(wire_block(part[_fp32_order(part)][:64], hi - lo, 64))
            b, ch = np.float32(0), []
            for i, s in enumerate(part["score"]):
                if s > b:
                    ch.append(i)
                    b = s
            chains.append(wire_block(part[ch], hi - lo, 255))
        assert exchange_merge(np.concatenate(blocks), world, 64, auto_base=True).tobytes() == want.tobytes()
        assert exchange_merge(np.concatenate(chains), world, 255, kind=1, mode="weighted", auto_base=True).tobytes() == want_chain.tobytes()


def test_synth_pose_round_trip():
    prob = synth.make_problem(200, 3000, 0.01, seed=2)
    T = synth.make_hypotheses(prob, 50, seed=3)
    back = synth.centre_pose(synth.uncentre_pose(T, prob.c_scene, prob.c_model), prob.c_scene, prob.c_model)
    assert np.allclose(back, T, atol=1e-6)
    kbar, nonempty = synth.kbar_27(prob, T, max_hyp=50)
    assert kbar > 0 and 0 < nonempty <= 1
