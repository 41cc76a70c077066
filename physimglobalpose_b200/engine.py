"""Host-side mirror of the reference's per-object matcher (match_4pcs::MatchSuper4PCS as
`getProbableTransformsSuper4PCS` drives it, S4/super4pcs_test.cc:39-111) over the C ABI of
include/pgp.h.  numpy arrays are host buffers; torch CUDA tensors are passed by pointer.

S4 = /root/reference/src/3rdparty/super4pcs/src/super4pcs (citations only; nothing is read from
the reference tree at run time)."""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional, Sequence

import numpy as np

from . import _lib
from ._lib import PGP_COMM_ID_BYTES, PGP_INDEX_AUTO, PGP_LCP_COUNT, PGP_LCP_WEIGHTED, PgpError, PgpHyp, PgpPcsOpts

MODES = {"count": PGP_LCP_COUNT, "weighted": PGP_LCP_WEIGHTED, PGP_LCP_COUNT: PGP_LCP_COUNT, PGP_LCP_WEIGHTED: PGP_LCP_WEIGHTED}

HYP_DTYPE = np.dtype([("index", "<i8"), ("count", "<u4"), ("score", "<f4"), ("T", "<f4", (12,))])
assert HYP_DTYPE.itemsize == C.sizeof(PgpHyp) == 64


def _f32(a, cols=None):
    if a is None:
        return None
    a = np.ascontiguousarray(a, dtype=np.float32)
    if cols is not None:
        a = a.reshape(-1, cols)
    return a


def _ptr(a):
    return None if a is None else a.ctypes.data


class PoseEngine:
    """One context on one GPU.  Scene = the segmented cloud of one object request ("P"); model
    slots hold the search / validation clouds ("Q", "Q_validation")."""

    def __init__(self, device: int = 0, _borrowed_ctx=None):
        self._lib = _lib.load()
        self._owned = _borrowed_ctx is None
        self._ctx = self._lib.pgp_create(int(device)) if self._owned else _borrowed_ctx
        if not self._ctx:
            raise PgpError(-2, self._lib.pgp_last_error(None).decode())
        self.device = int(device)
        self._nv = {}
        self._nq = {}
        self._ns = 0
        self._keep = {}

    # ------------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, "_ctx", None):
            if self._owned:
                self._lib.pgp_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int) -> int:
        if rc < 0:
            raise PgpError(rc, self._lib.pgp_last_error(self._ctx).decode())
        return rc

    def set_stream(self, cuda_stream: Optional[int]):
        """cudaStream_t handle (e.g. torch.cuda.current_stream().cuda_stream); None = the context's own
        stream.  torch's default stream has handle 0, which is passed on as cudaStreamLegacy (0x1)."""
        if cuda_stream is not None and int(cuda_stream) == 0:
            cuda_stream = 1
        self._check(self._lib.pgp_set_stream(self._ctx, cuda_stream))

    def set_option(self, name: str, value: int):
        self._check(self._lib.pgp_set_option(self._ctx, name.encode(), int(value)))

    def synchronize(self):
        self._check(self._lib.pgp_synchronize(self._ctx))

    @property
    def launch_count(self) -> int:
        return int(self._lib.pgp_launch_count(self._ctx))

    # ------------------------------------------------------------------ K1
    def set_scene(self, xyz, normals=None, delta: float = 0.005):
        """Match4PCSBase::init for P: centring + spatial index (match4pcsBase.cc:242-270)."""
        xyz = _f32(xyz, 3)
        normals = _f32(normals, 3)
        if normals is not None and len(normals) != len(xyz):
            raise ValueError("normals / points length mismatch")
        self._check(self._lib.pgp_set_scene(self._ctx, _ptr(xyz), _ptr(normals), len(xyz), float(delta)))
        self._ns = len(xyz)

    def set_scene_prior_image(self, img_u16, K):
        img = np.ascontiguousarray(img_u16, dtype=np.uint16)
        K = _f32(K).reshape(9)
        self._check(self._lib.pgp_set_scene_prior_image(self._ctx, _ptr(img), img.shape[0], img.shape[1], _ptr(K)))

    def set_scene_priors(self, prior):
        prior = _f32(prior).reshape(-1)
        if len(prior) != self._ns:
            raise ValueError("one prior per scene point")
        self._check(self._lib.pgp_set_scene_priors(self._ctx, _ptr(prior)))

    def scene_priors(self) -> np.ndarray:
        out = np.zeros(self._ns, np.float32)
        self._check(self._lib.pgp_get_scene_priors(self._ctx, _ptr(out)))
        return out

    def set_model(self, obj: int, search_xyz, search_normals, val_xyz=None, val_normals=None):
        sx, sn = _f32(search_xyz, 3), _f32(search_normals, 3)
        vx = sx if val_xyz is None else _f32(val_xyz, 3)
        vn = sn if val_xyz is None else _f32(val_normals, 3)
        self._check(self._lib.pgp_set_model(self._ctx, obj, _ptr(sx), _ptr(sn), len(sx), _ptr(vx), _ptr(vn), len(vx)))
        self._nq[obj], self._nv[obj] = len(sx), len(vx)

    def centroids(self, obj: int = 0):
        cP, cQ = np.zeros(3, np.float32), np.zeros(3, np.float32)
        self._check(self._lib.pgp_get_centroids(self._ctx, obj, _ptr(cP), _ptr(cQ)))
        return cP, cQ

    def pose_to_centred(self, obj: int, pose44) -> np.ndarray:
        P = np.ascontiguousarray(pose44, dtype=np.float64).reshape(-1, 16)
        out = np.zeros((len(P), 12), np.float32)
        for i in range(len(P)):
            self._check(self._lib.pgp_pose_to_centred(self._ctx, obj, P[i].ctypes.data, out[i].ctypes.data))
        return out.reshape(-1, 3, 4)

    def centred_to_pose(self, obj: int, T) -> np.ndarray:
        T = _f32(T).reshape(-1, 12)
        out = np.zeros((len(T), 16), np.float64)
        for i in range(len(T)):
            self._check(self._lib.pgp_centred_to_pose(self._ctx, obj, T[i].ctypes.data, out[i].ctypes.data))
        return out.reshape(-1, 4, 4)

    def grid_info(self) -> dict:
        dims = (C.c_int * 3)()
        nc, no, b = C.c_int64(), C.c_int64(), C.c_int64()
        cell = C.c_float()
        self._check(self._lib.pgp_grid_info(self._ctx, dims, C.byref(nc), C.byref(no), C.byref(cell), C.byref(b)))
        return dict(dims=tuple(dims), n_cells=nc.value, n_occupied=no.value, cell=cell.value, bytes=b.value)

    def label_stats(self) -> dict:
        """Tri-state label structure of the current scene (pgp_label_stats).  `ambig_overflow_records`: candidates of AMBIG voxels
        beyond the two each voxel keeps inline in its 32-byte slot."""
        out = np.zeros(8, np.int64)
        self._check(self._lib.pgp_label_stats(self._ctx, _ptr(out)))
        keys = ("cells_all_out", "cells_all_in", "cells_mixed", "voxels_out", "voxels_in", "voxels_ambig", "ambig_overflow_records", "nearest_list_entries")
        return dict(zip(keys, (int(v) for v in out)))

    # ------------------------------------------------------------------ K3
    def score_lcp(self, obj: int, T, mode="count"):
        """Host buffers in, host buffers out (counts u32, scores f32); copies are inside the call."""
        T = _f32(T).reshape(-1, 12)
        n = len(T)
        counts = np.zeros(n, np.uint32)
        scores = np.zeros(n, np.float32)
        self._check(self._lib.pgp_score_lcp(self._ctx, obj, _ptr(T), n, MODES[mode], _ptr(counts), _ptr(scores)))
        return counts, scores

    def score_lcp_into(self, obj: int, T: np.ndarray, counts: np.ndarray, scores: Optional[np.ndarray], mode="count"):
        """Same, with caller-owned (ideally pinned) host buffers -- the bench's e2e call."""
        n = T.size // 12
        self._check(self._lib.pgp_score_lcp(self._ctx, obj, T.ctypes.data, n, MODES[mode], counts.ctypes.data,
                                            None if scores is None else scores.ctypes.data))

    def score_lcp_ptr(self, obj: int, T_ptr: int, n: int, counts_ptr: int, scores_ptr: int, mode="count", host: bool = True):
        """Raw-pointer form (pinned torch tensors / device tensors)."""
        fn = self._lib.pgp_score_lcp if host else self._lib.pgp_score_lcp_dev
        self._check(fn(self._ctx, obj, T_ptr, n, MODES[mode], counts_ptr, scores_ptr))

    def score_lcp_begin(self, obj: int, T_ptr: int, n: int, counts_ptr: int, scores_ptr: int, mode="count"):
        """pgp_score_lcp_begin: enqueue upload + scoring + downloads of a pinned host batch and return (see include/pgp.h)."""
        self._check(self._lib.pgp_score_lcp_begin(self._ctx, obj, T_ptr, n, MODES[mode], counts_ptr, scores_ptr))

    def score_lcp_end(self) -> bool:
        """pgp_score_lcp_end: wait for the batch; True when it had to be re-scored (work queued in between must be redone)."""
        return self._check(self._lib.pgp_score_lcp_end(self._ctx)) > 0

    def score_lcp_device(self, obj: int, T_dev, counts_dev, scores_dev, mode="count"):
        """torch CUDA tensors: T (n,12) f32, counts (n,) i32/u32-as-int32, scores (n,) f32.  Asynchronous."""
        n = T_dev.shape[0]
        assert T_dev.is_cuda and T_dev.is_contiguous() and counts_dev.is_cuda and scores_dev.is_cuda
        self._keep[obj] = (T_dev, counts_dev, scores_dev)
        self._check(self._lib.pgp_score_lcp_dev(self._ctx, obj, T_dev.data_ptr(), n, MODES[mode], counts_dev.data_ptr(), scores_dev.data_ptr()))

    def registered_points(self, obj: int, T) -> np.ndarray:
        T = _f32(T).reshape(12)
        out = np.zeros(self._nv[obj], np.int32)
        k = self._check(self._lib.pgp_registered_points(self._ctx, obj, _ptr(T), _ptr(out), len(out)))
        return out[:k].copy()

    def nearest_in_range(self, obj: int, T) -> np.ndarray:
        T = _f32(T).reshape(12)
        out = np.zeros(self._nv[obj], np.int32)
        self._check(self._lib.pgp_nearest_in_range(self._ctx, obj, _ptr(T), _ptr(out)))
        return out

    # ------------------------------------------------------------------ K4
    def topk(self, obj: int, k: int, index_base: int = 0) -> np.ndarray:
        out = np.zeros(max(k, 1), HYP_DTYPE)
        m = self._check(self._lib.pgp_topk(self._ctx, obj, k, index_base, _ptr(out)))
        return out[:m].copy()

    def topk_device(self, obj: int, k: int, index_base: int, out_dev):
        """Asynchronous: k 64-byte records into a torch CUDA uint8 tensor of k*64 bytes (an all-gather send buffer)."""
        assert out_dev.is_cuda and out_dev.numel() * out_dev.element_size() >= 64 * k
        self._check(self._lib.pgp_topk_dev(self._ctx, obj, k, index_base, out_dev.data_ptr()))

    def topk_begin(self, obj: int, k: int, index_base: int = 0) -> int:
        """pgp_topk_begin: K4 on the context's stream, all-gather + download on its exchange stream; returns a ticket."""
        self._tickets = getattr(self, "_tickets", {})
        t = self._check(self._lib.pgp_topk_begin(self._ctx, obj, k, index_base))
        self._tickets[t] = k
        return t

    def topk_stream_wait(self, ticket: int):
        self._check(self._lib.pgp_topk_stream_wait(self._ctx, ticket))

    def topk_end(self, ticket: int) -> np.ndarray:
        """pgp_topk_end: wait for the ticket, merge -> the global top-k (the same on every rank)."""
        out = np.zeros(max(self._tickets.pop(ticket), 1), HYP_DTYPE)
        m = self._check(self._lib.pgp_topk_end(self._ctx, ticket, _ptr(out)))
        return out[:m].copy()

    # ------------------------------------------------------------------ K4d
    def set_symmetries(self, obj: int, R=None):
        """Discrete symmetries of model slot obj: (n, 3, 3) rotations in the centred model frame, the identity implied; None or an
        empty array clears the set (pgp_set_symmetries)."""
        R9 = np.ascontiguousarray(np.zeros((0, 9)) if R is None else R, np.float64).reshape(-1, 9)
        self._check(self._lib.pgp_set_symmetries(self._ctx, int(obj), _ptr(R9) if len(R9) else None, len(R9)))

    def topk_distinct(self, obj: int, m: int, k: int, max_dist: float, max_angle: float) -> np.ndarray:
        """pgp_topk_distinct: the top m by score, then greedy suppression of every record within max_dist (metres, centred
        translation) and max_angle (radians, up to the object's symmetries) of an earlier kept one; at most k records, in score order.
        The kernel sees cos_angle = math.cos(max_angle)."""
        out = np.zeros(max(int(k), 1), HYP_DTYPE)
        n = self._check(self._lib.pgp_topk_distinct(self._ctx, int(obj), int(m), int(k), float(max_dist), math.cos(max_angle), _ptr(out)))
        return out[:n].copy()

    def distinct_device(self, objs, pool_offsets, pool, k: int, max_dist: float, max_angle: float, out, poses=None, n_kept=None):
        """pgp_distinct_dev: pose-distinct selection over many pools on device data, asynchronous on the context's stream (set_stream).
        Structure, numpy: objs (n_lists,) model slots; pool_offsets (n_lists + 1,) int64.  Device data, torch CUDA tensors: pool, the
        concatenated 64-byte records (any dtype, pool_offsets[-1] x 64 bytes, e.g. topk_device's output); out, n_lists x k records
        (kept ones first, then index = -1); poses (n_lists x k, 16) or (n_lists x k, 4, 4) f64 or None, the camera-frame poses (identity
        after the kept ones); n_kept (n_lists,) i32 or None.  The kernel sees cos_angle = math.cos(max_angle).  The tensors are kept
        alive until the next call."""
        import torch
        o = np.ascontiguousarray(objs, np.int32).reshape(-1)
        off = np.ascontiguousarray(pool_offsets, np.int64).reshape(-1)
        if len(off) != len(o) + 1:
            raise ValueError("pool_offsets needs n_lists + 1 entries")
        nbytes = lambda t: t.numel() * t.element_size()   # noqa: E731
        for name, t, need in (("pool", pool, 64 * int(off[-1])), ("out", out, 64 * len(o) * int(k))):
            if not (isinstance(t, torch.Tensor) and t.is_cuda and t.is_contiguous() and nbytes(t) >= need):
                raise ValueError(f"{name} must be a contiguous CUDA tensor of at least {need} bytes")
        want = {"poses": (poses, torch.float64, 16 * len(o) * int(k)), "n_kept": (n_kept, torch.int32, len(o))}
        for name, (t, dt, numel) in want.items():
            if t is not None and not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dt and t.is_contiguous() and t.numel() >= numel):
                raise ValueError(f"{name} must be a contiguous CUDA tensor of {numel} {dt}")
        self._keep["distinct"] = (pool, out, poses, n_kept)
        dp = lambda t: None if t is None else t.data_ptr()   # noqa: E731
        self._check(self._lib.pgp_distinct_dev(self._ctx, _ptr(o) if len(o) else None, _ptr(off), len(o), dp(pool), int(k), float(max_dist),
                                               math.cos(max_angle), dp(out), dp(poses), dp(n_kept)))

    # ------------------------------------------------------------------ multi-GPU (one process per GPU)
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = C.create_string_buffer(PGP_COMM_ID_BYTES)
        rc = _lib.load().pgp_comm_unique_id(buf)
        if rc < 0:
            raise PgpError(rc, _lib.load().pgp_last_error(None).decode())
        return buf.raw

    def comm_init(self, unique_id: Optional[bytes], rank: int, world: int):
        """pgp_comm_init (collective): joins this context to the communicator; pgp_topk / improving_chain become collective."""
        buf = C.create_string_buffer(unique_id, PGP_COMM_ID_BYTES) if unique_id is not None else None
        self._check(self._lib.pgp_comm_init(self._ctx, buf, int(rank), int(world)))

    def comm_destroy(self):
        self._check(self._lib.pgp_comm_destroy(self._ctx))

    @property
    def comm_rank(self) -> int:
        return int(self._lib.pgp_comm_rank(self._ctx))

    @property
    def comm_world(self) -> int:
        return int(self._lib.pgp_comm_world(self._ctx))

    def generate_pcs_range(self, obj: int, base_lo: int, base_hi: int, seed: int = 1, max_hyp: int = 10000, **opts) -> int:
        """pgp_generate_pcs_range: bases [base_lo, base_hi) of the request's n_bases (bases shard across GPUs)."""
        o = PgpPcsOpts()
        self._lib.pgp_pcs_default_opts(C.byref(o))
        for k, v in opts.items():
            setattr(o, k, v)
        n = C.c_int64(0)
        self._check(self._lib.pgp_generate_pcs_range(self._ctx, obj, C.byref(o), int(seed), int(base_lo), int(base_hi), int(max_hyp), C.byref(n)))
        self._ngen = getattr(self, "_ngen", {})
        self._ngen[obj] = n.value
        return n.value

    def sync_generated(self, obj: int, max_hyp: int = 0):
        """pgp_comm_sync_generated (collective): global cap in rank order; returns (index_base of this rank, global total)."""
        base, tot = C.c_int64(0), C.c_int64(0)
        self._check(self._lib.pgp_comm_sync_generated(self._ctx, obj, int(max_hyp), C.byref(base), C.byref(tot)))
        self._ngen = getattr(self, "_ngen", {})
        return base.value, tot.value

    def bench_sector_gather(self, footprint_bytes: int, loads_per_thread: int = 256) -> float:
        """pgp_bench_sector_gather: random 32-byte-sector gather throughput in GB/s."""
        g = C.c_float(0)
        self._check(self._lib.pgp_bench_sector_gather(self._ctx, int(footprint_bytes), int(loads_per_thread), C.byref(g)))
        return float(g.value)

    def improving_chain(self, obj: int, index_base: int = 0, cap: int = 4096) -> np.ndarray:
        out = np.zeros(cap, HYP_DTYPE)
        m = self._check(self._lib.pgp_improving_chain(self._ctx, obj, index_base, _ptr(out), cap))
        return out[:m].copy()

    # ------------------------------------------------------------------ K2
    def extract_pairs(self, obj: int, dist: float, eps: float, cap: int = 1 << 22) -> np.ndarray:
        out = np.zeros((cap, 2), np.int32)
        n = C.c_int64(0)
        self._check(self._lib.pgp_extract_pairs(self._ctx, obj, float(dist), float(eps), _ptr(out), cap, C.byref(n)))
        if n.value > cap:
            return self.extract_pairs(obj, dist, eps, cap=int(n.value))
        return out[: n.value].copy()

    def find_quads(self, obj: int, base4, inv1, inv2, eps, pairs1, pairs2, cap: int = 1 << 20) -> np.ndarray:
        b = np.ascontiguousarray(base4, np.int32)
        p1 = np.ascontiguousarray(pairs1, np.int32).reshape(-1, 2)
        p2 = np.ascontiguousarray(pairs2, np.int32).reshape(-1, 2)
        out = np.zeros((cap, 4), np.int32)
        n = C.c_int64(0)
        self._check(self._lib.pgp_find_quads(self._ctx, obj, _ptr(b), float(inv1), float(inv2), float(eps), _ptr(p1), len(p1),
                                             _ptr(p2), len(p2), _ptr(out), cap, C.byref(n)))
        if n.value > cap:
            return self.find_quads(obj, base4, inv1, inv2, eps, pairs1, pairs2, cap=int(n.value))
        return out[: n.value].copy()

    def find_quads_v4pcs(self, obj: int, base4, eps: float, cap: int = 1 << 22) -> np.ndarray:
        """operMode 2: congruent quads of one base (4 scene ids), sorted by (v1, v2, v3, v4)."""
        b = np.ascontiguousarray(base4, np.int32)
        out = np.zeros((cap, 4), np.int32)
        n = C.c_int64(0)
        self._check(self._lib.pgp_find_quads_v4pcs(self._ctx, obj, _ptr(b), float(eps), _ptr(out), cap, C.byref(n)))
        return out[: min(n.value, cap)].copy()

    def rigid_from_quads(self, obj: int, base4, quads):
        b = np.ascontiguousarray(base4, np.int32)
        q = np.ascontiguousarray(quads, np.int32).reshape(-1, 4)
        T = np.zeros((len(q), 12), np.float32)
        ok = np.zeros(len(q), np.uint8)
        self._check(self._lib.pgp_rigid_from_quads(self._ctx, obj, _ptr(b), _ptr(q), len(q), _ptr(T), _ptr(ok)))
        return T.reshape(-1, 3, 4), ok.astype(bool)

    def generate_pcs(self, obj: int, seed: int = 1, max_hyp: int = 10000, **opts) -> int:
        o = PgpPcsOpts()
        self._lib.pgp_pcs_default_opts(C.byref(o))
        for k, v in opts.items():
            setattr(o, k, v)
        n = C.c_int64(0)
        self._check(self._lib.pgp_generate_pcs(self._ctx, obj, C.byref(o), int(seed), int(max_hyp), C.byref(n)))
        self._ngen = getattr(self, "_ngen", {})
        self._ngen[obj] = n.value
        return n.value

    def score_generated(self, obj: int, mode="count"):
        self._check(self._lib.pgp_score_generated(self._ctx, obj, MODES[mode]))

    def get_generated(self, obj: int):
        n = self._ngen.get(obj, 0)
        T = np.zeros((n, 12), np.float32)
        counts = np.zeros(n, np.uint32)
        scores = np.zeros(n, np.float32)
        self._check(self._lib.pgp_get_generated(self._ctx, obj, _ptr(T), _ptr(counts), _ptr(scores), n))
        return T.reshape(-1, 3, 4), counts, scores

    def set_ppf_map(self, obj: int, keys4, offsets, pairs):
        """Installs the model's PPF map (rows: key (4 ints) -> pairs[offsets[k]:offsets[k+1]]), the PPFMap argument of
        getProbableTransformsSuper4PCS."""
        k = np.ascontiguousarray(keys4, np.int32).reshape(-1, 4)
        o = np.ascontiguousarray(offsets, np.int64)
        p = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        assert len(o) == len(k) + 1
        self._check(self._lib.pgp_set_ppf_map(self._ctx, obj, _ptr(k), _ptr(o), _ptr(p), len(k)))

    def build_ppf_map(self, obj: int):
        self._check(self._lib.pgp_build_ppf_map(self._ctx, obj))

    def get_ppf_map(self, obj: int):
        nk, npr = C.c_int64(0), C.c_int64(0)
        self._check(self._lib.pgp_get_ppf_map(self._ctx, obj, None, 0, None, None, 0, C.byref(nk), C.byref(npr)))
        keys = np.zeros((nk.value, 4), np.int32)
        offs = np.zeros(nk.value + 1, np.int64)
        pairs = np.zeros((npr.value, 2), np.int32)
        self._check(self._lib.pgp_get_ppf_map(self._ctx, obj, _ptr(keys), nk.value, _ptr(offs), _ptr(pairs), npr.value, C.byref(nk), C.byref(npr)))
        return keys, offs, pairs

    def scene_ppf_keys(self, pairs) -> np.ndarray:
        p = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        out = np.zeros((len(p), 4), np.int32)
        self._check(self._lib.pgp_scene_ppf_keys(self._ctx, _ptr(p), len(p), _ptr(out)))
        return out

    def stocs_engine_seed(self, seed: int, base: int, attempt: int = 0) -> int:
        return int(self._lib.pgp_stocs_engine_seed(int(seed), int(base), int(attempt)))

    def get_bases(self, obj: int, cap: int = 4096):
        """Bases of the last generate_pcs call: (ids (n,4) scene indices, invariants (n,2), ok (n,) bool)."""
        ids = np.zeros((cap, 4), np.int32)
        inv = np.zeros((cap, 2), np.float32)
        ok = np.zeros(cap, np.uint8)
        n = self._check(self._lib.pgp_get_bases(self._ctx, obj, _ptr(ids), _ptr(inv), _ptr(ok), cap))
        return ids[:n].copy(), inv[:n].copy(), ok[:n].astype(bool)

    # ------------------------------------------------------------------ K5
    def tricp(self, obj: int, segment_xyz, poses44, trim: float = 0.5, ratio: float = 0.99, max_iter: int = 100):
        seg = _f32(segment_xyz, 3)
        P = np.ascontiguousarray(poses44, dtype=np.float64).reshape(-1, 16).copy()
        iters = np.zeros(len(P), np.int32)
        energy = np.zeros(len(P), np.float32)
        self._check(self._lib.pgp_tricp(self._ctx, obj, _ptr(seg), len(seg), _ptr(P), len(P), float(trim), float(ratio), int(max_iter),
                                        _ptr(iters), _ptr(energy)))
        return P.reshape(-1, 4, 4), iters, energy

    def tricp_plane(self, obj: int, segment_xyz, poses44, trim: float = 0.5, ratio: float = 0.99, max_iter: int = 100):
        """Trimmed point-to-plane ICP (utilities::pointToPlaneICP): tricp's search, trim and stop, fitted to the validation normals
        with 6x6 normal equations.  Returns (refined poses, iterations, point-to-plane trimmed energies)."""
        seg = _f32(segment_xyz, 3)
        P = np.ascontiguousarray(poses44, dtype=np.float64).reshape(-1, 16).copy()
        iters = np.zeros(len(P), np.int32)
        energy = np.zeros(len(P), np.float32)
        self._check(self._lib.pgp_tricp_plane(self._ctx, obj, _ptr(seg), len(seg), _ptr(P), len(P), float(trim), float(ratio), int(max_iter),
                                              _ptr(iters), _ptr(energy)))
        return P.reshape(-1, 4, 4), iters, energy

    # ------------------------------------------------------------------ K6
    def remove_explained(self, obj: int, segment_xyz, placed_poses44, threshold: float = 0.008) -> np.ndarray:
        """Boolean mask of the segment points EXPLAINED by the placed objects (UCTState.cpp:149-174)."""
        seg = _f32(segment_xyz, 3)
        P = np.ascontiguousarray(placed_poses44, dtype=np.float64).reshape(-1, 16)
        flag = np.zeros(len(seg), np.uint8)
        self._check(self._lib.pgp_remove_explained(self._ctx, obj, _ptr(seg), len(seg), _ptr(P) if len(P) else None, len(P), float(threshold), _ptr(flag)))
        return flag.astype(bool)

    def mcts_tricp(self, obj: int, segment_xyz, placed_poses44, poses44, threshold: float = 0.008, trim: float = 0.5, ratio: float = 0.99,
                   max_iter: int = 100):
        """UCTState::performTrICP for a batch of candidate poses: explained-point removal + trimmed ICP."""
        seg = _f32(segment_xyz, 3)
        placed = np.ascontiguousarray(placed_poses44, dtype=np.float64).reshape(-1, 16)
        P = np.ascontiguousarray(poses44, dtype=np.float64).reshape(-1, 16).copy()
        iters = np.zeros(len(P), np.int32)
        energy = np.zeros(len(P), np.float32)
        nun = C.c_int(0)
        self._check(self._lib.pgp_mcts_tricp(self._ctx, obj, _ptr(seg), len(seg), _ptr(placed) if len(placed) else None, len(placed), float(threshold),
                                             _ptr(P), len(P), float(trim), float(ratio), int(max_iter), _ptr(iters), _ptr(energy), C.byref(nun)))
        return P.reshape(-1, 4, 4), iters, energy, nun.value

    def refine_batch(self, segments, items, metric: str = "point", threshold: float = 0.008, trim: float = 0.5, ratio: float = 0.99,
                     max_iter: int = 100):
        """Many refinements in one call (pgp_refine_batch).  segments: list of (n, 3) clouds; items: list of
        (obj, seg index, placed poses (m, 4, 4), candidate poses (k, 4, 4)); metric "point" (pgp_tricp's fit) or "plane"
        (pgp_tricp_plane's).  Returns one (refined poses, iterations, energies, n_unexplained) per item, each equal to that
        item's mcts_tricp (point) or remove_explained + tricp_plane (plane) result."""
        icp = {"point": _lib.PGP_ICP_POINT, "plane": _lib.PGP_ICP_PLANE}[metric]
        segs = [_f32(s, 3) for s in segments]
        seg = np.ascontiguousarray(np.concatenate(segs) if segs else np.zeros((0, 3), np.float32))
        seg_off = np.zeros(len(segs) + 1, np.int64)
        seg_off[1:] = np.cumsum([len(s) for s in segs])
        placed = [np.ascontiguousarray(it[2], dtype=np.float64).reshape(-1, 16) for it in items]
        poses = [np.ascontiguousarray(it[3], dtype=np.float64).reshape(-1, 16) for it in items]
        rec = np.zeros(len(items), np.dtype([("obj", "<i4"), ("seg", "<i4"), ("placed_lo", "<i4"), ("n_placed", "<i4")]))
        lo = 0
        for i, it in enumerate(items):
            rec[i] = (int(it[0]), int(it[1]), lo, len(placed[i]))
            lo += len(placed[i])
        pl = np.ascontiguousarray(np.concatenate(placed) if placed else np.zeros((0, 16)))
        P = np.ascontiguousarray(np.concatenate(poses) if poses else np.zeros((0, 16)))
        pose_off = np.zeros(len(items) + 1, np.int64)
        pose_off[1:] = np.cumsum([len(p) for p in poses])
        iters = np.zeros(len(P), np.int32)
        energy = np.zeros(len(P), np.float32)
        nun = np.zeros(len(items), np.int32)
        self._check(self._lib.pgp_refine_batch(self._ctx, icp, _ptr(seg), _ptr(seg_off), len(segs), _ptr(pl), len(pl), _ptr(rec), _ptr(pose_off),
                                               len(items), _ptr(P), float(threshold), float(trim), float(ratio), int(max_iter), _ptr(iters),
                                               _ptr(energy), _ptr(nun)))
        return [(P[a:b].reshape(-1, 4, 4), iters[a:b], energy[a:b], int(nun[i]))
                for i, (a, b) in enumerate(zip(pose_off[:-1], pose_off[1:]))]

    def refine_batch_device(self, seg_xyz, seg_offsets, placed, items, pose_offsets, poses, status, iters=None, energy=None,
                            n_unexplained=None, metric: str = "point", threshold: float = 0.008, trim: float = 0.5, ratio: float = 0.99,
                            max_iter: int = 100):
        """pgp_refine_batch_dev: refine_batch on device data, asynchronous on the context's stream (set_stream).
        Device data, torch CUDA tensors: seg_xyz (n, 3) f32; placed (m, 4, 4) or (m, 16) f64; poses (p, 4, 4) or (p, 16) f64,
        refined in place; status (1,) i32, PGP_OK or PGP_E_INVALID once the work has run; optional outputs iters (p,) i32,
        energy (p,) f32, n_unexplained (len(items),) i32.  Structure, numpy: seg_offsets (n_segs + 1,) int64; items (n, 4) int32
        rows (obj, seg, placed_lo, n_placed); pose_offsets (len(items) + 1,) int64.  The tensors are kept alive until the next call."""
        import torch
        icp = {"point": _lib.PGP_ICP_POINT, "plane": _lib.PGP_ICP_PLANE}[metric]
        want = {"seg_xyz": (seg_xyz, torch.float32), "placed": (placed, torch.float64), "poses": (poses, torch.float64), "status": (status, torch.int32),
                "iters": (iters, torch.int32), "energy": (energy, torch.float32), "n_unexplained": (n_unexplained, torch.int32)}
        for name, (t, dt) in want.items():
            if t is not None and not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dt and t.is_contiguous()):
                raise ValueError(f"{name} must be a contiguous CUDA tensor of {dt}")
        seg_off = np.ascontiguousarray(seg_offsets, np.int64)
        rec = np.ascontiguousarray(items, np.int32).reshape(-1, 4)
        pose_off = np.ascontiguousarray(pose_offsets, np.int64)
        self._keep["refine_batch"] = (seg_xyz, placed, poses, status, iters, energy, n_unexplained)
        dp = lambda t: None if t is None or t.numel() == 0 else t.data_ptr()
        self._check(self._lib.pgp_refine_batch_dev(self._ctx, icp, dp(seg_xyz), _ptr(seg_off), len(seg_off) - 1, dp(placed), placed.numel() // 16,
                                                   _ptr(rec) if len(rec) else None, _ptr(pose_off), len(rec), dp(poses), float(threshold), float(trim),
                                                   float(ratio), int(max_iter), dp(iters), dp(energy), dp(n_unexplained), status.data_ptr()))

    # ------------------------------------------------------------------ K7
    def prepare_segment(self, depth_raw_u16, class_mask_u8, class_id: int, K, leaf: float = 0.01, normal_radius: float = 0.02,
                        outlier_radius: float = 0.03, min_neighbors: int = 10, cap: int = 1 << 20):
        """Depth frame + class mask -> the object's segment cloud (points, unit normals) and the number of valid-depth pixels."""
        d = np.ascontiguousarray(depth_raw_u16, np.uint16)
        m = np.ascontiguousarray(class_mask_u8, np.uint8)
        assert d.shape == m.shape and d.ndim == 2
        K = _f32(K).reshape(9)
        xyz = np.zeros((cap, 3), np.float32)
        nrm = np.zeros((cap, 3), np.float32)
        nraw = C.c_int(0)
        n = self._check(self._lib.pgp_prepare_segment(self._ctx, _ptr(d), _ptr(m), d.shape[0], d.shape[1], int(class_id), _ptr(K), float(leaf),
                                                      float(normal_radius), float(outlier_radius), int(min_neighbors), _ptr(xyz), _ptr(nrm), cap,
                                                      C.byref(nraw)))
        return xyz[:n].copy(), nrm[:n].copy(), nraw.value

    # ------------------------------------------------------------------ K8
    def set_mesh(self, obj: int, vert_xyz, tri3, class_id: int = -1):
        """Triangle mesh of object slot `obj` in its model frame; class_id = its label in the class mask (-1: none)."""
        v = _f32(vert_xyz, 3)
        t = np.ascontiguousarray(tri3, np.int32).reshape(-1, 3)
        self._check(self._lib.pgp_set_mesh(self._ctx, int(obj), _ptr(v), len(v), _ptr(t), len(t), int(class_id)))

    def set_depth_observation(self, depth_raw_u16, class_mask_u8, K) -> np.ndarray:
        """Observed frame (raw depth as stored, class mask or None, 3x3 intrinsics).  Returns the pixels of each label with valid depth."""
        d = np.ascontiguousarray(depth_raw_u16, np.uint16)
        assert d.ndim == 2
        m = None if class_mask_u8 is None else np.ascontiguousarray(class_mask_u8, np.uint8)
        assert m is None or m.shape == d.shape
        K = _f32(K).reshape(9)
        hist = np.zeros(256, np.int64)
        self._check(self._lib.pgp_set_depth_observation(self._ctx, _ptr(d), _ptr(m), d.shape[0], d.shape[1], _ptr(K), _ptr(hist)))
        self._frame = d.shape
        return hist

    def render_depth(self, obj_ids, poses44):
        """One state rendered in full: (depth rows x cols fp32 metres, 0 = nothing; slot rows x cols int32, -1 = nothing)."""
        ids = np.ascontiguousarray(obj_ids, np.int32).reshape(-1)
        P = np.ascontiguousarray(poses44, np.float64).reshape(-1, 16)
        rows, cols = getattr(self, "_frame", (1, 1))
        depth = np.zeros((rows, cols), np.float32)
        slot = np.zeros((rows, cols), np.int32)
        self._check(self._lib.pgp_render_depth(self._ctx, _ptr(ids), _ptr(P), len(ids), _ptr(depth), _ptr(slot)))
        return depth, slot

    def depth_cost(self, states, tau: float) -> np.ndarray:
        """states: [(obj_ids, poses44), ...].  Returns (n_slots, 5) int32 {rendered, agree, in_front, behind, on_segment}, one row per
        placed object in state order."""
        ids = [np.asarray(o, np.int32).reshape(-1) for o, _ in states]
        poses = [np.asarray(p, np.float64).reshape(-1, 16) for _, p in states]
        offs = np.zeros(len(states) + 1, np.int64)
        offs[1:] = np.cumsum([len(i) for i in ids])
        flat_ids = np.ascontiguousarray(np.concatenate(ids) if ids else np.zeros(0, np.int32), np.int32)
        flat_P = np.ascontiguousarray(np.concatenate(poses) if poses else np.zeros((0, 16)), np.float64)
        out = np.zeros((int(offs[-1]), 5), np.int32)
        self._check(self._lib.pgp_depth_cost(self._ctx, _ptr(offs), len(states), _ptr(flat_ids), _ptr(flat_P), float(tau), _ptr(out)))
        return out

    def depth_cost_device(self, states_ids, poses, out, status, tau: float):
        """pgp_depth_cost_dev: depth_cost on device data, asynchronous on the context's stream (set_stream).
        Structure, numpy: states_ids, one int array of object ids per state.  Device data, torch CUDA tensors, one row per placed
        object in state order: poses (n, 4, 4) or (n, 16) f64; out (n, 5) i32 {rendered, agree, in_front, behind, on_segment},
        written once the work has run with status PGP_OK; status (1,) i32: PGP_OK, PGP_E_INVALID (a pose entry is not finite) or
        PGP_E_CAPACITY (a chunk needed more (triangle, tile) entries than it reserved; depth_cost evaluates such states).  The
        tensors are kept alive until the next call."""
        import torch
        want = {"poses": (poses, torch.float64), "out": (out, torch.int32), "status": (status, torch.int32)}
        for name, (t, dt) in want.items():
            if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dt and t.is_contiguous()):
                raise ValueError(f"{name} must be a contiguous CUDA tensor of {dt}")
        ids = [np.asarray(i, np.int32).reshape(-1) for i in states_ids]
        offs = np.zeros(len(ids) + 1, np.int64)
        offs[1:] = np.cumsum([len(i) for i in ids])
        n = int(offs[-1])
        if poses.numel() != 16 * n or out.numel() != 5 * n or status.numel() != 1:
            raise ValueError(f"{n} placed objects: poses needs {n} x 16 entries, out {n} x 5, status 1")
        flat_ids = np.ascontiguousarray(np.concatenate(ids) if ids else np.zeros(0, np.int32), np.int32)
        self._keep["depth_cost"] = (poses, out, status)
        dp = lambda t: None if t.numel() == 0 else t.data_ptr()   # noqa: E731
        self._check(self._lib.pgp_depth_cost_dev(self._ctx, _ptr(offs), len(ids), _ptr(flat_ids), dp(poses), float(tau), dp(out),
                                                 status.data_ptr()))

    def render_depth_device(self, states_ids, poses, depth, status, slot=None):
        """pgp_render_depth_dev: every state rendered into device frames, asynchronous on the context's stream (set_stream).
        Structure, numpy: states_ids, one int array of object ids per state.  Device data, torch CUDA tensors: poses (n, 4, 4) or
        (n, 16) f64, one row per placed object in state order; depth (n_states, rows, cols) f32 metres (0 = nothing) and slot
        (n_states, rows, cols) i32 (-1 = nothing) or None, frame s equal to render_depth of state s; status (1,) i32: PGP_OK,
        PGP_E_INVALID (a pose entry is not finite; no frame written) or PGP_E_CAPACITY (a chunk needed more (triangle, tile) entries
        than it reserved; the frames are unspecified and render_depth renders such states).  The tensors are kept alive until the
        next call."""
        import torch
        want = {"poses": (poses, torch.float64), "depth": (depth, torch.float32), "status": (status, torch.int32), "slot": (slot, torch.int32)}
        for name, (t, dt) in want.items():
            if (t is not None or name != "slot") and not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dt and t.is_contiguous()):
                raise ValueError(f"{name} must be a contiguous CUDA tensor of {dt}")
        ids = [np.asarray(i, np.int32).reshape(-1) for i in states_ids]
        offs = np.zeros(len(ids) + 1, np.int64)
        offs[1:] = np.cumsum([len(i) for i in ids])
        n, px = int(offs[-1]), len(ids) * int(np.prod(getattr(self, "_frame", (1, 1))))
        if poses.numel() != 16 * n or depth.numel() != px or (slot is not None and slot.numel() != px) or status.numel() != 1:
            raise ValueError(f"{n} placed objects in {len(ids)} states: poses needs {n} x 16 entries, depth and slot {px}, status 1")
        flat_ids = np.ascontiguousarray(np.concatenate(ids) if ids else np.zeros(0, np.int32), np.int32)
        self._keep["render_depth"] = (poses, depth, slot, status)
        dp = lambda t: None if t is None or t.numel() == 0 else t.data_ptr()   # noqa: E731
        self._check(self._lib.pgp_render_depth_dev(self._ctx, _ptr(offs), len(ids), _ptr(flat_ids), dp(poses), dp(depth), dp(slot),
                                                   status.data_ptr()))

    def set_depth_observation_device(self, depth_raw, class_mask, K, class_pixels=None):
        """pgp_set_depth_observation_dev: set_depth_observation on device data, asynchronous on the context's stream (set_stream).
        Torch CUDA tensors: depth_raw (rows, cols) u16 or i16 (the same bits) as stored; class_mask (rows, cols) u8 or None;
        class_pixels (256,) i64 or None, the pixels of each label with valid depth once the work has run.  K: 3x3 intrinsics on the
        host.  Calls queued after this one on the stream see this observation.  The tensors are kept alive until the next call."""
        import torch
        if not (isinstance(depth_raw, torch.Tensor) and depth_raw.is_cuda and depth_raw.dtype in (torch.uint16, torch.int16)
                and depth_raw.is_contiguous() and depth_raw.dim() == 2):
            raise ValueError("depth_raw must be a contiguous 2-D CUDA tensor of torch.uint16 or torch.int16")
        want = {"class_mask": (class_mask, torch.uint8, depth_raw.numel()), "class_pixels": (class_pixels, torch.int64, 256)}
        for name, (t, dt, numel) in want.items():
            if t is not None and not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dt and t.is_contiguous() and t.numel() == numel):
                raise ValueError(f"{name} must be a contiguous CUDA tensor of {numel} {dt}")
        K = _f32(K).reshape(9)
        self._keep["observation"] = (depth_raw, class_mask, class_pixels)
        dp = lambda t: None if t is None else t.data_ptr()   # noqa: E731
        self._check(self._lib.pgp_set_depth_observation_dev(self._ctx, dp(depth_raw), dp(class_mask), depth_raw.shape[0], depth_raw.shape[1],
                                                            _ptr(K), dp(class_pixels)))
        self._frame = tuple(depth_raw.shape)


class PoseGroup:
    """One process, n GPUs (pgp_group_*): replicated scene / models, bases or hypotheses sharded over the devices, NCCL
    all-gather + deterministic merge of the selections.  `engine(i)` gives device i's context for the per-device calls."""

    def __init__(self, devices: Sequence[int]):
        self._lib = _lib.load()
        ids = (C.c_int * len(devices))(*[int(d) for d in devices])
        self._g = self._lib.pgp_group_create(len(devices), ids)
        if not self._g:
            raise PgpError(-9, self._lib.pgp_last_error(None).decode())
        self.devices = list(devices)
        self._engines = [PoseEngine(d, _borrowed_ctx=self._lib.pgp_group_ctx(self._g, i)) for i, d in enumerate(devices)]

    def close(self):
        if getattr(self, "_g", None):
            for e in self._engines:
                e.close()
            self._lib.pgp_group_destroy(self._g)
            self._g = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int) -> int:
        if rc < 0:
            raise PgpError(rc, self._lib.pgp_group_last_error(self._g).decode())
        return rc

    def __len__(self):
        return len(self.devices)

    def engine(self, i: int) -> PoseEngine:
        return self._engines[i]

    def set_scene(self, xyz, normals=None, delta: float = 0.005):
        xyz, normals = _f32(xyz, 3), _f32(normals, 3)
        self._check(self._lib.pgp_group_set_scene(self._g, _ptr(xyz), _ptr(normals), len(xyz), float(delta)))
        for e in self._engines:
            e._ns = len(xyz)

    def set_scene_priors(self, prior):
        prior = _f32(prior).reshape(-1)
        self._check(self._lib.pgp_group_set_scene_priors(self._g, _ptr(prior)))

    def set_scene_prior_image(self, img_u16, K):
        img = np.ascontiguousarray(img_u16, dtype=np.uint16)
        K = _f32(K).reshape(9)
        self._check(self._lib.pgp_group_set_scene_prior_image(self._g, _ptr(img), img.shape[0], img.shape[1], _ptr(K)))

    def set_model(self, obj: int, search_xyz, search_normals, val_xyz=None, val_normals=None):
        sx, sn = _f32(search_xyz, 3), _f32(search_normals, 3)
        vx = sx if val_xyz is None else _f32(val_xyz, 3)
        vn = sn if val_xyz is None else _f32(val_normals, 3)
        self._check(self._lib.pgp_group_set_model(self._g, obj, _ptr(sx), _ptr(sn), len(sx), _ptr(vx), _ptr(vn), len(vx)))
        for e in self._engines:
            e._nq[obj], e._nv[obj] = len(sx), len(vx)

    def build_ppf_map(self, obj: int):
        self._check(self._lib.pgp_group_build_ppf_map(self._g, obj))

    def set_ppf_map(self, obj: int, keys4, offsets, pairs):
        k = np.ascontiguousarray(keys4, np.int32).reshape(-1, 4)
        o = np.ascontiguousarray(offsets, np.int64)
        p = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        self._check(self._lib.pgp_group_set_ppf_map(self._g, obj, _ptr(k), _ptr(o), _ptr(p), len(k)))

    def generate_pcs(self, obj: int, seed: int = 1, max_hyp: int = 10000, **opts) -> int:
        o = PgpPcsOpts()
        self._lib.pgp_pcs_default_opts(C.byref(o))
        for k, v in opts.items():
            setattr(o, k, v)
        n = C.c_int64(0)
        self._check(self._lib.pgp_group_generate_pcs(self._g, obj, C.byref(o), int(seed), int(max_hyp), C.byref(n)))
        return n.value

    def score_generated(self, obj: int, mode="count"):
        self._check(self._lib.pgp_group_score_generated(self._g, obj, MODES[mode]))

    def score_lcp(self, obj: int, T, mode="count"):
        T = _f32(T).reshape(-1, 12)
        counts = np.zeros(len(T), np.uint32)
        scores = np.zeros(len(T), np.float32)
        self._check(self._lib.pgp_group_score_lcp(self._g, obj, _ptr(T), len(T), MODES[mode], _ptr(counts), _ptr(scores)))
        return counts, scores

    def topk(self, obj: int, k: int) -> np.ndarray:
        out = np.zeros(max(k, 1), HYP_DTYPE)
        m = self._check(self._lib.pgp_group_topk(self._g, obj, k, _ptr(out)))
        return out[:m].copy()

    def improving_chain(self, obj: int, cap: int = 4096) -> np.ndarray:
        out = np.zeros(cap, HYP_DTYPE)
        m = self._check(self._lib.pgp_group_improving_chain(self._g, obj, _ptr(out), cap))
        return out[:m].copy()

    def set_symmetries(self, obj: int, R=None):
        R9 = np.ascontiguousarray(np.zeros((0, 9)) if R is None else R, np.float64).reshape(-1, 9)
        self._check(self._lib.pgp_group_set_symmetries(self._g, int(obj), _ptr(R9) if len(R9) else None, len(R9)))

    def topk_distinct(self, obj: int, m: int, k: int, max_dist: float, max_angle: float) -> np.ndarray:
        """PoseEngine.topk_distinct over the group's merged top m: the same answer as one context on the concatenated batch."""
        out = np.zeros(max(int(k), 1), HYP_DTYPE)
        n = self._check(self._lib.pgp_group_topk_distinct(self._g, int(obj), int(m), int(k), float(max_dist), math.cos(max_angle), _ptr(out)))
        return out[:n].copy()


def exchange_merge(wire: np.ndarray, world: int, k: int, kind: int = 0, mode="count", auto_base: bool = False, cap: int = 4096) -> np.ndarray:
    """pgp_exchange_merge: `wire` = world x (k + 1) records (header + k records per rank), as the all-gather delivers them."""
    lib = _lib.load()
    w = np.ascontiguousarray(wire, HYP_DTYPE).reshape(world, k + 1)
    out = np.zeros(max(cap, 1), HYP_DTYPE)
    m = lib.pgp_exchange_merge(w.ctypes.data, world, k, kind, MODES[mode], 1 if auto_base else 0, out.ctypes.data, cap)
    if m < 0:
        raise PgpError(m, "pgp_exchange_merge")
    return out[:m].copy()


def wire_block(records: np.ndarray, batch_size: int, k: int) -> np.ndarray:
    """One rank's block of the exchange: header {batch size, number of records} + k record slots."""
    blk = np.zeros(k + 1, HYP_DTYPE)
    blk["index"][1:] = -1
    n = min(len(records), k)
    blk[0]["index"], blk[0]["count"] = batch_size, n
    blk[1:1 + n] = records[:n]
    return blk


def topk_merge(lists: Sequence[np.ndarray], k: int) -> np.ndarray:
    """Deterministic merge of per-rank top-k record arrays (pgp_topk_merge)."""
    lib = _lib.load()
    k_each = max((len(a) for a in lists), default=0)
    buf = np.zeros((len(lists), max(k_each, 1)), HYP_DTYPE)
    buf["index"] = -1
    for i, a in enumerate(lists):
        buf[i, : len(a)] = a
    out = np.zeros(max(k, 1), HYP_DTYPE)
    m = lib.pgp_topk_merge(buf.ctypes.data, len(lists), max(k_each, 1), k, out.ctypes.data)
    if m < 0:
        raise PgpError(m, "pgp_topk_merge")
    return out[:m].copy()
