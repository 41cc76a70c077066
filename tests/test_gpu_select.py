"""K4 selection (csrc/k4_select.cu) against plain sequential references: the top-k and the strictly improving chain, through every
entry point that returns them (pgp_topk, pgp_topk_dev, pgp_topk_begin / _end, pgp_improving_chain, pgp_group_topk,
pgp_group_improving_chain), on keys crafted to sit where a radix select, a capped compaction and a segmented max-scan go wrong:
ties at the k-th key, key widths on the 11-bit digit boundaries, k near 4096 and k > n, n where the grid stops growing, chain
steps across CTA segments, chains longer than the capacities, 64-bit index bases, fp32 keys, negative and signed-zero scores.

Crafted keys reach K4 through a scored batch: the caller owns the device buffers pgp_score_lcp_dev scores into, and the selection
reads the last batch from them.  Every hypothesis translates the model 100 m off the scene, so scoring is a cull; the counts,
scores and transforms are then overwritten in place.  T[i] holds a bit pattern that encodes i, so a record is traced back to its
row and compared completely: index (with index_base), count, score bits and all 12 T words.

References: top-k = the first k of (key desc, index asc), keys compared as fp32 values (-0 == +0); chain = keep i iff its key
> max(0, every earlier key), the scan of match4pcsBase.cc:1888-1901 (cross-checked against the C restatement of the oracle)."""
import zlib

import numpy as np
import pytest

from physimglobalpose_b200 import _lib, synth
from physimglobalpose_b200.engine import HYP_DTYPE, PoseEngine, PoseGroup

pytestmark = pytest.mark.gpu

AUTO = _lib.PGP_INDEX_AUTO
BIG_BASE = (1 << 33) + 5
BASES = (0, BIG_BASE, AUTO)
E_INVALID, E_CAPACITY = -1, -8
KMAX = 4096
CHAIN_EXCHANGE_CAP = 255
KS = (1, 2, 63, 64, 65, 2048, 2049, 4095, 4096)
NV_SLOT = {1: 1, 2: 2, 2047: 3, 2048: 4, 30000: 5}        # validation-cloud size -> object slot
NV_COUNT, NV_WEIGHTED = 30000, 2048                        # slots of the generic count / weighted cases
T_PATTERN = 0x40000000                                     # T[i][c] bits = T_PATTERN + 16 i + c: finite, normal, unique
FLT_MAX_BITS, INF_BITS = 0x7F7FFFFF, 0x7F800000


def bits_for(v):
    """k4_select.cu bits_for: the key width of a value."""
    b = 1
    while b < 64 and (v >> b):
        b += 1
    return b


def _f32(bits):
    return np.asarray(bits, np.uint32).view(np.float32)


# ------------------------------------------------------------------------------------------------------------ fixtures
class _Sel:
    def __init__(self, e, g, sm):
        self.e, self.g, self.sm = e, g, sm

    def resolve(self, n):
        """n as a parameter: an int, or ("sm", d) = sm_count * 1024 + d (the size where the grid stops growing)."""
        return self.sm * 1024 + n[1] if isinstance(n, tuple) else n


def _scene_and_models(x, prob, vx, vn):
    x.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    for nv, obj in NV_SLOT.items():
        x.set_model(obj, prob.model_xyz, prob.model_nrm, vx[:nv], vn[:nv])


def _val_cloud(n, seed):
    rng = np.random.default_rng(seed)
    vx = rng.uniform(-0.05, 0.05, size=(n, 3)).astype(np.float32)
    vn = rng.normal(size=(n, 3))
    return vx, (vn / np.linalg.norm(vn, axis=1, keepdims=True)).astype(np.float32)


@pytest.fixture(scope="module")
def sel():
    """A context and a fresh one-device group (no pgp_group_score_lcp: no shard ranges), both with the object slots of NV_SLOT."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    prob = synth.make_problem(300, 4000, 0.01, seed=71)
    vx, vn = _val_cloud(max(NV_SLOT), 72)
    e, g = PoseEngine(0), PoseGroup([0])
    _scene_and_models(e, prob, vx, vn)
    _scene_and_models(g, prob, vx, vn)
    yield _Sel(e, g, torch.cuda.get_device_properties(0).multi_processor_count)
    g.close()
    e.close()


class Batch:
    """A crafted batch on one device, registered as the last scored batch of `obj` on every context of `ctxs` (they share the
    buffers).  with_scores=False: COUNT mode without a score buffer (records then carry fl(count / nv))."""

    def __init__(self, ctxs, obj, n, mode, with_scores=True, device=0, row0=0):
        import torch
        dev = torch.device("cuda", device)
        self.obj, self.n, self.mode, self.row0 = obj, n, mode, row0
        self.T = torch.zeros((n, 12), dtype=torch.float32, device=dev)
        self.T[:, [0, 5, 10]] = 1.0
        self.T[:, [3, 7, 11]] = 100.0                      # 100 m off the scene: the group cull rejects everything at once
        self.counts = torch.zeros(n, dtype=torch.int32, device=dev)
        self.scores = torch.zeros(n, dtype=torch.float32, device=dev) if with_scores else None
        for e in ctxs:
            if with_scores:
                e.score_lcp_device(obj, self.T, self.counts, self.scores, mode)
            else:
                e.score_lcp_ptr(obj, self.T.data_ptr(), n, self.counts.data_ptr(), 0, mode, host=False)
            e.synchronize()
        rows = torch.arange(row0, row0 + n, dtype=torch.int64, device=dev)
        words = T_PATTERN + rows[:, None] * 16 + torch.arange(12, dtype=torch.int64, device=dev)
        self.T.copy_(words.to(torch.int32).view(torch.float32))
        torch.cuda.synchronize(dev)

    def set(self, counts, scores=None):
        import torch
        self.counts.copy_(torch.from_numpy(np.ascontiguousarray(counts, np.uint32).view(np.int32)))
        if self.scores is not None:
            self.scores.copy_(torch.from_numpy(np.ascontiguousarray(scores, np.float32)))
        torch.cuda.synchronize(self.counts.device)


# ------------------------------------------------------------------------------------------------------------ references
def t_words(rows):
    rows = np.asarray(rows, np.int64)
    return _f32((T_PATTERN + rows[:, None] * 16 + np.arange(12)).astype(np.uint32))


def records(rows, counts, scores, nv, base, T=None):
    """The records a selection of `rows` must return: scores=None -> fl(count / nv)."""
    rows = np.asarray(rows, np.int64)
    r = np.zeros(len(rows), HYP_DTYPE)
    r["index"] = rows + (0 if base == AUTO else base)
    r["count"] = counts[rows]
    r["score"] = scores[rows] if scores is not None else counts[rows].astype(np.float32) / np.float32(nv)
    r["T"] = t_words(rows) if T is None else np.asarray(T, np.float32).reshape(-1, 12)[rows]
    return r


def order_key(mode, counts, scores):
    """The value selection orders by, as float64: the count, or the fp32 score with -0 folded into +0."""
    if mode == "count":
        return counts.astype(np.float64)
    s = scores.astype(np.float64)
    s[s == 0] = 0.0
    return s


def ref_topk(key, k):
    n = len(key)
    k = min(k, n)
    cand = np.arange(n)
    if n > 4 * k:
        kth = np.partition(key, n - k)[n - k]
        cand = np.flatnonzero(key >= kth)
    return cand[np.lexsort((cand, -key[cand]))[:k]]


def ref_chain(key):
    """best = 0; keep i iff key[i] > best (strict), then best = key[i]."""
    before = np.maximum.accumulate(np.concatenate(([0.0], key[:-1])))
    return np.flatnonzero(key > before)


def assert_records(got, want, what):
    assert got.dtype == HYP_DTYPE
    g = np.ascontiguousarray(got).view(np.uint8).reshape(-1, 64)
    w = np.ascontiguousarray(want).view(np.uint8).reshape(-1, 64)
    if g.shape == w.shape and np.array_equal(g, w):
        return
    m = min(len(g), len(w))
    bad = np.flatnonzero(np.any(g[:m] != w[:m], axis=1))[:3]
    raise AssertionError(f"{what}: {len(got)} records, want {len(want)}; first differing rows {bad.tolist()}: "
                         f"got {got[bad].tolist()} want {want[bad].tolist()}")


# ------------------------------------------------------------------------------------------------------------ key distributions
def _levels(mode, rng, n, lo, hi):
    """n random keys in [lo, hi] (COUNT: integers; WEIGHTED: fp32 values in [lo / 64, hi / 64])."""
    if mode == "count":
        return rng.integers(lo, hi + 1, size=n).astype(np.uint32)
    return (rng.integers(lo, hi + 1, size=n) / 64.0).astype(np.float32)


def _fp32_keys(rng, n):
    """Random bit patterns in [+0, +Inf], with subnormals, the normal boundary, FLT_MAX, +Inf, 1-ulp neighbours and repeats."""
    b = rng.integers(0, INF_BITS + 1, size=n, dtype=np.int64)
    special = np.array([0, 1, 2, 0x007FFFFF, 0x00800000, 0x00800001, 0x3F7FFFFF, 0x3F800000, 0x3F800001,
                        FLT_MAX_BITS - 1, FLT_MAX_BITS, INF_BITS, INF_BITS])
    pos = rng.choice(n, min(n, len(special)), replace=False)
    b[pos] = special[: len(pos)]
    if n > 32:
        src = rng.choice(n, n // 8, replace=False)                   # 1-ulp neighbours of random keys
        b[rng.choice(n, n // 8, replace=False)] = np.minimum(b[src] + rng.integers(-1, 2, size=len(src)), INF_BITS).clip(0)
        b[rng.choice(n, n // 16, replace=False)] = b[rng.choice(n, n // 16, replace=False)]     # repeats
    return _f32(b.astype(np.uint32))


def _signed_keys(rng, n):
    """Negative, -0.0, +0.0 and positive scores, +-FLT_MAX, +Inf and 1-ulp neighbours on both sides of zero."""
    b = rng.integers(0, 1 << 32, size=n, dtype=np.int64)
    b[(b & 0x7FFFFFFF) > INF_BITS] &= 0x3FFFFFFF                     # no NaN
    b[(b & 0x7FFFFFFF) == INF_BITS] = 0xFF7FFFFF                      # no -Inf, +Inf below
    special = np.array([0, 0x80000000, 0, 0x80000000, 1, 0x80000001, 0xBF800000, 0x3F800000, FLT_MAX_BITS, 0xFF7FFFFF, INF_BITS])
    pos = rng.choice(n, min(n, len(special)), replace=False)
    b[pos] = special[: len(pos)]
    if n > 16:
        z = rng.choice(n, n // 8, replace=False)                     # plenty of signed zeros: ties broken by the index
        b[z] = rng.choice([0, 0x80000000], size=len(z))
    return _f32(b.astype(np.uint32))


def make_keys(mode, dist, rng, n, nv, k=None):
    """(counts, scores) of one distribution.  WEIGHTED counts are arbitrary (records must carry them through)."""
    top = nv if mode == "count" else 60000
    if dist == "equal":
        key = _levels(mode, rng, 1, 1, top).repeat(n)
    elif dist == "zero":
        key = np.zeros(n, np.uint32 if mode == "count" else np.float32)
    elif dist == "two":
        a, b = sorted(_levels(mode, rng, 2, 0, top))
        if a == b:
            a, b = (0, top) if mode == "count" else (np.float32(0.25), np.float32(0.75))
        key = np.where(rng.random(n) < 0.5, a, b).astype(np.uint32 if mode == "count" else np.float32)
    elif dist == "lowbit":
        if mode == "count":
            key = ((top - 1) // 2 * 2 + rng.integers(0, 2, size=n)).astype(np.uint32) if top >= 1 else np.zeros(n, np.uint32)
        else:
            key = _f32(0x3E2AAAAA + rng.integers(0, 2, size=n).astype(np.uint32))
    elif dist == "tie":
        # a large block equal to the k-th key, at random positions (so across every CTA): the last digit and the index decide
        kk = min(k, n)
        above = int(rng.integers(0, kk))
        below = int(rng.integers(0, n - kk + 1)) // 2
        mid = top // 2
        lv = np.concatenate([_levels(mode, rng, above, mid + 1, top), _levels(mode, rng, n - above - below, mid, mid),
                             _levels(mode, rng, below, 0, mid - 1)])
        key = lv[rng.permutation(n)]
    elif dist == "fp32":
        key = _fp32_keys(rng, n)
    elif dist == "signed":
        key = _signed_keys(rng, n)
    elif dist == "zeros_signed":
        key = _f32(rng.choice([0, 0x80000000], size=n).astype(np.uint32))
        few = rng.choice(n, max(1, n // 16), replace=False)
        key[few] = rng.choice([-0.5, 0.5, -1e-30, 1e-30], size=len(few)).astype(np.float32)
    else:
        raise ValueError(dist)
    if mode == "count":
        counts = np.asarray(key, np.uint32)
        assert counts.max(initial=0) <= nv
        return counts, counts.astype(np.float32) / np.float32(nv)
    return rng.integers(0, nv + 1, size=n).astype(np.uint32), np.asarray(key, np.float32)


# ------------------------------------------------------------------------------------------------------------ entry points
def check_topk(S, b, mode, counts, scores, nv, k, bases=BASES, group=True):
    """pgp_topk, pgp_topk_dev (with the padding when k > n), pgp_topk_begin / _end and the one-device group against the reference."""
    import torch
    rows = ref_topk(order_key(mode, counts, scores), k)
    for base in bases:
        want = records(rows, counts, scores, nv, base)
        assert_records(S.e.topk(b.obj, k, base), want, f"pgp_topk k={k} base={base}")
        buf = torch.full((k * 64,), 0xAB, dtype=torch.uint8, device="cuda:0")
        torch.cuda.synchronize(0)                          # K4 writes on the context's stream, not torch's
        S.e.topk_device(b.obj, k, base, buf)
        S.e.synchronize()
        pad = np.zeros(k - len(rows), HYP_DTYPE)
        pad["index"] = -1
        assert_records(buf.cpu().numpy().view(HYP_DTYPE), np.concatenate([want, pad]), f"pgp_topk_dev k={k} base={base}")
        assert_records(S.e.topk_end(S.e.topk_begin(b.obj, k, base)), want, f"pgp_topk_begin/_end k={k} base={base}")
    if group:
        assert_records(S.g.topk(b.obj, k), records(rows, counts, scores, nv, 0), f"pgp_group_topk k={k}")


def check_chain(S, b, mode, counts, scores, nv, bases=BASES, group=True):
    rows = ref_chain(order_key(mode, counts, scores))
    assert len(rows) <= KMAX
    for base in bases:
        got = S.e.improving_chain(b.obj, base, KMAX)
        assert_records(got, records(rows, counts, scores, nv, base), f"pgp_improving_chain base={base}")
    if group:
        if len(rows) <= CHAIN_EXCHANGE_CAP:
            assert_records(S.g.improving_chain(b.obj, KMAX), records(rows, counts, scores, nv, 0), "pgp_group_improving_chain")
        else:
            with pytest.raises(_lib.PgpError) as e:
                S.g.improving_chain(b.obj, KMAX)
            assert e.value.code == E_CAPACITY
    return rows


# ------------------------------------------------------------------------------------------------------------ top-k and chain over n x distribution
SMALL_N = (1, 2, 3, 1023, 1024, 1025, ("sm", -1), ("sm", 0), ("sm", 1))
COUNT_DISTS = ("equal", "zero", "two", "tie", "lowbit")
WEIGHTED_DISTS = ("equal", "zero", "two", "tie", "lowbit", "fp32", "signed", "zeros_signed")
CASES = ([(n, "count", d) for n in SMALL_N for d in COUNT_DISTS] + [(n, "weighted", d) for n in SMALL_N for d in WEIGHTED_DISTS]
         + [((1 << 20) + 7, "count", "tie"), ((1 << 20) + 7, "weighted", "fp32"), ((1 << 20) + 7, "weighted", "signed"),
            (1 << 23, "weighted", "tie"), (1 << 23, "count", "lowbit")])


def _nid(n):
    return f"sm*1024{n[1]:+d}" if isinstance(n, tuple) else str(n)


@pytest.mark.parametrize("n,mode,dist", CASES, ids=[f"{_nid(n)}-{m}-{d}" for n, m, d in CASES])
def test_select_equals_the_sequential_reference(sel, n, mode, dist):
    n = sel.resolve(n)
    nv = NV_COUNT if mode == "count" else NV_WEIGHTED
    rng = np.random.default_rng(zlib.crc32(f"{n}-{mode}-{dist}".encode()))
    b = Batch((sel.e, sel.g.engine(0)), NV_SLOT[nv], n, mode)
    ks = KS + ((n + 1,) if n + 1 <= KMAX and n + 1 not in KS else ()) if n < (1 << 20) else (1, 64, 2049, KMAX)
    counts, scores = make_keys(mode, dist, rng, n, nv, k=1)
    b.set(counts, scores)
    for k in ks:
        if dist == "tie":
            counts, scores = make_keys(mode, dist, rng, n, nv, k=k)
            b.set(counts, scores)
        check_topk(sel, b, mode, counts, scores, nv, k)
    check_chain(sel, b, mode, counts, scores, nv)


def test_k_above_4096_is_invalid(sel):
    b = Batch((sel.e,), NV_SLOT[NV_COUNT], 5000, "count")
    b.set(*make_keys("count", "two", np.random.default_rng(1), 5000, NV_COUNT))
    for call in (lambda: sel.e.topk(b.obj, KMAX + 1), lambda: sel.e.topk_begin(b.obj, KMAX + 1)):
        with pytest.raises(_lib.PgpError) as e:
            call()
        assert e.value.code == E_INVALID
    assert len(sel.e.topk(b.obj, KMAX)) == KMAX


# ------------------------------------------------------------------------------------------------------------ digit boundaries
def _digit_cases():
    """(mode, nv, n) with ibits + kbits on, one below and one above every multiple of 11 reachable with n <= 2^23."""
    out = []
    for mode, kb_of in (("count", {nv: bits_for(nv) for nv in NV_SLOT}), ("weighted", {NV_WEIGHTED: 32})):
        for m11 in range(11, 64, 11):
            for t in (m11 - 1, m11, m11 + 1):
                best = None
                for nv, kb in kb_of.items():
                    ib = t - kb
                    if 1 <= ib <= 23 and (best is None or ib < best[1]):
                        best = (nv, ib)
                if best:
                    nv, ib = best
                    n = 1 << 23 if ib == 23 else (1 << (ib - 1)) + 1        # the smallest n of that index width (n = 2^23 at 23)
                    assert bits_for(n - 1) + bits_for(nv if mode == "count" else (1 << 32) - 1) == t
                    out.append((mode, nv, n))
    return out


DIGIT_CASES = _digit_cases()


@pytest.mark.parametrize("mode,nv,n", DIGIT_CASES,
                         ids=[f"{m}-nv{nv}-n{n}-bits{bits_for(n - 1) + (bits_for(nv) if m == 'count' else 32)}" for m, nv, n in DIGIT_CASES])
def test_key_width_on_the_digit_boundaries(sel, mode, nv, n):
    rng = np.random.default_rng(n * 7 + nv)
    b = Batch((sel.e, sel.g.engine(0)), NV_SLOT[nv], n, mode)
    if mode == "count":
        counts = rng.integers(0, nv + 1, size=n).astype(np.uint32)
        counts[rng.choice(n, min(n, 3), replace=False)] = [nv, 0, nv][: min(n, 3)]
        scores = counts.astype(np.float32) / np.float32(nv)
    else:
        counts, scores = make_keys(mode, "fp32", rng, n, nv)
    b.set(counts, scores)
    for k in (1, 64, 2049, KMAX):
        check_topk(sel, b, mode, counts, scores, nv, k, bases=(BIG_BASE,))
    check_chain(sel, b, mode, counts, scores, nv, bases=(BIG_BASE,))


# ------------------------------------------------------------------------------------------------------------ COUNT without a score buffer
@pytest.mark.parametrize("nv", sorted(NV_SLOT))
@pytest.mark.parametrize("n", (3, ("sm", 1)), ids=_nid)
def test_count_mode_without_score_buffer(sel, nv, n):
    """pgp_score_lcp_dev with scores = NULL: records carry fl(count / nv), computed on the device."""
    n = sel.resolve(n)
    rng = np.random.default_rng(nv + n)
    b = Batch((sel.e, sel.g.engine(0)), NV_SLOT[nv], n, "count", with_scores=False)
    counts = rng.integers(0, nv + 1, size=n).astype(np.uint32)
    b.set(counts)
    for k in (1, 65, KMAX, n + 1):
        if k <= KMAX:
            check_topk(sel, b, "count", counts, None, nv, k)
    check_chain(sel, b, "count", counts, None, nv)


# ------------------------------------------------------------------------------------------------------------ chain shapes
def _grid(sm, n):
    g = min(sm, -(-n // 1024))
    return g, -(-n // g)


def _chain_keys(kind, mode, rng, n, sm):
    """Scores of one chain shape, in [0, 30000] (COUNT) or fp32 (WEIGHTED)."""
    grid, seg = _grid(sm, n)
    if kind == "staircase":
        # a step at every CTA segment boundary: equal keys on both sides of the boundary (strict '>' keeps only the first), the
        # next element one higher; a few rising keys inside each segment
        key = rng.integers(0, 40, size=n).astype(np.float64)
        for g in range(grid):
            lvl = 100 + 200 * g
            s0, s1 = g * seg, min(n, (g + 1) * seg)
            inner = np.sort(rng.choice(np.arange(s0 + 2, max(s0 + 3, s1 - 2)), min(3, max(0, s1 - s0 - 4)), replace=False))
            key[inner] = lvl + 50 + np.arange(len(inner)) * 10
            if g + 1 < grid:
                bnd = (g + 1) * seg
                key[bnd - 1] = key[bnd] = lvl + 190
                if bnd + 1 < n:
                    key[bnd + 1] = lvl + 191
    elif kind == "max_last":
        key = rng.integers(0, 1000, size=n).astype(np.float64)
        key[(grid - 1) * seg + int(rng.integers(0, n - (grid - 1) * seg))] = 5000
    elif kind == "empty":
        key = np.zeros(n) if mode == "count" else -rng.integers(0, 1000, size=n).astype(np.float64)
    else:
        raise ValueError(kind)
    if mode == "count":
        c = key.astype(np.uint32)
        return c, c.astype(np.float32) / np.float32(NV_COUNT)
    s = (key / 1024.0).astype(np.float32)
    if kind == "empty":
        s[rng.choice(n, max(1, n // 4), replace=False)] = rng.choice([0.0, -0.0], size=max(1, n // 4)).astype(np.float32)
    return rng.integers(0, NV_COUNT + 1, size=n).astype(np.uint32), s


CHAIN_N = (1, 1025, 3000, ("sm", -1), ("sm", 1), (1 << 20) + 7)
CHAIN_CASES = [(n, m, kind) for n in CHAIN_N for m in ("count", "weighted") for kind in ("staircase", "max_last", "empty")]


@pytest.mark.parametrize("n,mode,kind", CHAIN_CASES, ids=[f"{_nid(n)}-{m}-{k}" for n, m, k in CHAIN_CASES])
def test_chain_shapes(sel, port_lib, small_problem, n, mode, kind):
    n = sel.resolve(n)
    nv = NV_COUNT
    rng = np.random.default_rng(zlib.crc32(f"{n}-{mode}-{kind}".encode()))
    b = Batch((sel.e, sel.g.engine(0)), NV_SLOT[nv], n, mode)
    counts, scores = _chain_keys(kind, mode, rng, n, sel.sm)
    b.set(counts, scores)
    rows = check_chain(sel, b, mode, counts, scores, nv)
    if kind == "empty":
        assert len(rows) == 0
    if kind == "staircase" and n > 1:
        assert len(rows) >= _grid(sel.sm, n)[0]
    # the vectorised reference is the sequential scan of the C restatement
    prob, _ = small_problem
    o = port_lib.PortOracle(prob.scene_xyz, prob.scene_nrm, prob.model_xyz, prob.model_nrm, prob.model_xyz, prob.model_nrm, prob.delta)
    assert np.array_equal(o.improving_chain(scores, cap=KMAX), rows)


def test_chain_ignores_scores_up_to_zero(sel):
    """WEIGHTED: negative, -0 and +0 scores never enter the chain, and positive improvements after them still do."""
    n = 5000
    b = Batch((sel.e, sel.g.engine(0)), NV_SLOT[NV_WEIGHTED], n, "weighted")
    rng = np.random.default_rng(12)
    s = -rng.random(n).astype(np.float32)
    s[:10] = [-0.0, 0.0, -3e38, -1e-45, 0.0, -0.0, -1.0, 0.0, -0.5, -0.0]
    up = np.sort(rng.choice(np.arange(10, n), 40, replace=False))
    s[up] = np.sort(rng.random(40).astype(np.float32) + 0.001)
    s[up[5]] = s[up[4]]                                    # an equal score does not enter
    counts = rng.integers(0, NV_WEIGHTED + 1, size=n).astype(np.uint32)
    b.set(counts, s)
    rows = check_chain(sel, b, "weighted", counts, s, NV_WEIGHTED)
    assert rows[0] == up[0] and up[5] not in rows and len(rows) == 39
    for k in (1, 64, n + 7 if n + 7 <= KMAX else KMAX):
        check_topk(sel, b, "weighted", counts, s, NV_WEIGHTED, k)


# ------------------------------------------------------------------------------------------------------------ chain capacities
def _chain_of_length(mode, rng, n, length):
    pos = np.sort(rng.choice(n, length, replace=False))
    if mode == "count":
        c = np.zeros(n, np.uint32)
        c[pos] = np.arange(1, length + 1)
        return c, c.astype(np.float32) / np.float32(NV_COUNT)
    s = np.zeros(n, np.float32)
    s[pos] = np.arange(1, length + 1, dtype=np.float32) / np.float32(8.0)
    return rng.integers(0, NV_COUNT + 1, size=n).astype(np.uint32), s


CAP_CASES = [(m, length, cap) for m in ("count", "weighted")
             for length, cap in ((1, 1), (100, 100), (101, 100), (2, 1), (4095, 4095), (4096, 4096), (4096, 4095), (4097, 4096), (4097, 100))]


@pytest.mark.parametrize("mode,length,cap", CAP_CASES, ids=[f"{m}-len{l}-cap{c}" for m, l, c in CAP_CASES])
def test_chain_capacity(sel, mode, length, cap):
    """length <= cap: the chain; cap < length <= 4096: PGP_E_CAPACITY with the last cap elements written; length > 4096:
    PGP_E_CAPACITY and the output is declared unusable."""
    n = max(3 * length, sel.sm * 1024 + 1)
    rng = np.random.default_rng(length * 31 + cap)
    b = Batch((sel.e,), NV_SLOT[NV_COUNT], n, mode)
    counts, scores = _chain_of_length(mode, rng, n, length)
    b.set(counts, scores)
    rows = ref_chain(order_key(mode, counts, scores))
    assert len(rows) == length
    if length <= cap:
        assert_records(sel.e.improving_chain(b.obj, BIG_BASE, cap), records(rows, counts, scores, NV_COUNT, BIG_BASE), "chain")
        return
    out = np.zeros(cap, HYP_DTYPE)
    rc = sel.e._lib.pgp_improving_chain(sel.e._ctx, b.obj, BIG_BASE, out.ctypes.data, cap)
    msg = sel.e._lib.pgp_last_error(sel.e._ctx).decode()
    assert rc == E_CAPACITY, (rc, msg)
    if length <= KMAX:
        assert "the last" in msg
        assert_records(out, records(rows[-cap:], counts, scores, NV_COUNT, BIG_BASE), "chain tail after PGP_E_CAPACITY")
    else:
        assert "unusable" in msg and "the last" not in msg


@pytest.mark.parametrize("mode", ("count", "weighted"))
def test_group_chain_exchange_cap(sel, mode):
    """A device may send at most 255 chain records: 255 is a result, 256 is PGP_E_CAPACITY (the header's overflow flag)."""
    n = sel.sm * 1024 + 1
    for length in (CHAIN_EXCHANGE_CAP, CHAIN_EXCHANGE_CAP + 1):
        rng = np.random.default_rng(length)
        b = Batch((sel.g.engine(0),), NV_SLOT[NV_COUNT], n, mode)
        counts, scores = _chain_of_length(mode, rng, n, length)
        b.set(counts, scores)
        rows = ref_chain(order_key(mode, counts, scores))
        if length <= CHAIN_EXCHANGE_CAP:
            assert_records(sel.g.improving_chain(b.obj, KMAX), records(rows, counts, scores, NV_COUNT, 0), "group chain")
        else:
            with pytest.raises(_lib.PgpError) as e:
                sel.g.improving_chain(b.obj, KMAX)
            assert e.value.code == E_CAPACITY
        del b


# ------------------------------------------------------------------------------------------------------------ two devices
def test_two_device_group_equals_one_context_on_the_concatenation(sel):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    prob = synth.make_problem(300, 4000, 0.01, seed=71)
    vx, vn = _val_cloud(max(NV_SLOT), 72)
    g2 = PoseGroup([0, 1])
    try:
        _scene_and_models(g2, prob, vx, vn)
        for mode, dist in (("count", "tie"), ("weighted", "signed"), ("weighted", "fp32")):
            nv = NV_COUNT if mode == "count" else NV_WEIGHTED
            obj = NV_SLOT[nv]
            n0, n1 = 70001, 90003
            rng = np.random.default_rng(len(dist))
            counts, scores = make_keys(mode, dist, rng, n0 + n1, nv, k=64)
            whole = Batch((sel.e,), obj, n0 + n1, mode)
            whole.set(counts, scores)
            shards = [Batch((g2.engine(0),), obj, n0, mode, device=0, row0=0),
                      Batch((g2.engine(1),), obj, n1, mode, device=1, row0=n0)]
            shards[0].set(counts[:n0], scores[:n0])
            shards[1].set(counts[n0:], scores[n0:])
            key = order_key(mode, counts, scores)
            for k in (1, 64, 4096):
                want = records(ref_topk(key, k), counts, scores, nv, 0)
                assert_records(sel.e.topk(obj, k), want, f"one context k={k}")
                assert_records(g2.topk(obj, k), want, f"two devices k={k}")
            want = records(ref_chain(key), counts, scores, nv, 0)
            assert_records(sel.e.improving_chain(obj), want, "one context chain")
            assert_records(g2.improving_chain(obj), want, "two devices chain")
    finally:
        g2.close()


# ------------------------------------------------------------------------------------------------------------ priors
def test_negative_priors_end_to_end(engine, port_lib, small_problem):
    """Priors with negative values (and signed zeros): the ordered weighted sum is exact, so scores are negative where the gated
    points' priors sum below zero; top-k and chain then follow fp32 order, and a score <= 0 never enters the chain."""
    prob, T = small_problem
    T = T[:200]
    nv = len(prob.model_xyz)
    engine.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    engine.set_model(0, prob.model_xyz, prob.model_nrm)
    rng = np.random.default_rng(91)
    prior = (rng.random(len(prob.scene_xyz)) - 0.5).astype(np.float32)
    prior[rng.choice(len(prior), 500, replace=False)] = rng.choice([0.0, -0.0], size=500).astype(np.float32)
    engine.set_scene_priors(prior)
    assert np.array_equal(engine.scene_priors().view(np.uint32), prior.view(np.uint32))
    counts, scores = engine.score_lcp(0, T, "weighted")

    o = port_lib.PortOracle(prob.scene_xyz, prob.scene_nrm, prob.model_xyz, prob.model_nrm, prob.model_xyz, prob.model_nrm, prob.delta)
    want_s = np.zeros(len(T), np.float32)
    want_c = np.zeros(len(T), np.uint32)
    for i in range(len(T)):
        _, _, reg = o.weighted_verify(T[i:i + 1], reg_of=0)            # gated scene indices, in model-point order
        acc = np.float32(0.0)
        for j in reg:
            acc = np.float32(acc + prior[j])
        want_s[i] = acc / np.float32(nv)
        want_c[i] = len(reg)
    assert np.array_equal(counts, want_c)
    assert np.array_equal(scores.view(np.uint32), want_s.view(np.uint32))
    assert (scores < 0).any() and (scores > 0).any()

    key = order_key("weighted", counts, scores)
    top = records(ref_topk(key, 64), counts, scores, nv, 0, T=T)
    chain = records(ref_chain(key), counts, scores, nv, 0, T=T)
    assert len(chain) >= 1 and np.all(chain["score"] > 0)
    assert_records(engine.topk(0, 64), top, "pgp_topk")
    assert_records(engine.improving_chain(0), chain, "pgp_improving_chain")
    g = PoseGroup([0])
    try:
        g.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
        g.set_model(0, prob.model_xyz, prob.model_nrm)
        g.set_scene_priors(prior)
        gc, gs = g.score_lcp(0, T, "weighted")
        assert np.array_equal(gc, want_c) and np.array_equal(gs.view(np.uint32), want_s.view(np.uint32))
        assert_records(g.topk(0, 64), top, "pgp_group_topk")
        assert_records(g.improving_chain(0), chain, "pgp_group_improving_chain")
    finally:
        g.close()


@pytest.mark.parametrize("bad", (np.nan, np.inf, -np.inf), ids=("nan", "inf", "-inf"))
def test_non_finite_priors_are_refused(engine, small_problem, bad):
    prob, _ = small_problem
    engine.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    good = np.linspace(-1, 1, len(prob.scene_xyz)).astype(np.float32)
    engine.set_scene_priors(good)
    prior = good.copy()
    prior[len(prior) // 3] = bad
    with pytest.raises(_lib.PgpError) as e:
        engine.set_scene_priors(prior)
    assert e.value.code == E_INVALID
    assert np.array_equal(engine.scene_priors(), good)                 # the previous priors stay
    g = PoseGroup([0])
    try:
        g.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
        with pytest.raises(_lib.PgpError) as e:
            g.set_scene_priors(prior)
        assert e.value.code == E_INVALID
        assert np.array_equal(g.engine(0).scene_priors(), np.ones(len(prior), np.float32))
    finally:
        g.close()
