"""ctypes binding of libpgp.so (include/pgp.h).  There is no fallback: if the library is not
built, or no B200 is present, every entry point raises."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libpgp.so")

PGP_LCP_COUNT = 0
PGP_LCP_WEIGHTED = 1
PGP_ICP_POINT = 0
PGP_ICP_PLANE = 1

STATUS = {0: "PGP_OK", -1: "PGP_E_INVALID", -2: "PGP_E_CUDA", -3: "PGP_E_NO_SCENE", -4: "PGP_E_NO_MODEL",
          -5: "PGP_E_NO_SCORES", -6: "PGP_E_TOO_LARGE", -7: "PGP_E_NOMEM", -8: "PGP_E_CAPACITY", -9: "PGP_E_COMM"}
PGP_INDEX_AUTO = -1
PGP_COMM_ID_BYTES = 128


class PgpHyp(C.Structure):
    """pgp_hyp of include/pgp.h (64 bytes)."""
    _fields_ = [("index", C.c_int64), ("count", C.c_uint32), ("score", C.c_float), ("T", C.c_float * 12)]


class PgpPcsOpts(C.Structure):
    _fields_ = [("n_bases", C.c_int), ("max_quads_per_base", C.c_int), ("max_base_diameter", C.c_float),
                ("overlap", C.c_float), ("base_trials", C.c_int), ("mode", C.c_int)]


class PgpError(RuntimeError):
    def __init__(self, code: int, text: str):
        super().__init__(f"{STATUS.get(code, code)}: {text}")
        self.code = code


_vp, _i, _i64, _f = C.c_void_p, C.c_int, C.c_int64, C.c_float
_SIGNATURES = {
    "pgp_create": (_vp, [_i]),
    "pgp_destroy": (None, [_vp]),
    "pgp_last_error": (C.c_char_p, [_vp]),
    "pgp_version": (C.c_char_p, []),
    "pgp_set_stream": (_i, [_vp, _vp]),
    "pgp_synchronize": (_i, [_vp]),
    "pgp_set_scene": (_i, [_vp, _vp, _vp, _i, _f]),
    "pgp_set_scene_prior_image": (_i, [_vp, _vp, _i, _i, _vp]),
    "pgp_set_scene_priors": (_i, [_vp, _vp]),
    "pgp_get_scene_priors": (_i, [_vp, _vp]),
    "pgp_set_model": (_i, [_vp, _i, _vp, _vp, _i, _vp, _vp, _i]),
    "pgp_get_centroids": (_i, [_vp, _i, _vp, _vp]),
    "pgp_pose_to_centred": (_i, [_vp, _i, _vp, _vp]),
    "pgp_centred_to_pose": (_i, [_vp, _i, _vp, _vp]),
    "pgp_grid_info": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "pgp_label_stats": (_i, [_vp, _vp]),
    "pgp_score_lcp": (_i, [_vp, _i, _vp, _i64, _i, _vp, _vp]),
    "pgp_score_lcp_dev": (_i, [_vp, _i, _vp, _i64, _i, _vp, _vp]),
    "pgp_score_lcp_begin": (_i, [_vp, _i, _vp, _i64, _i, _vp, _vp]),
    "pgp_score_lcp_end": (_i, [_vp]),
    "pgp_registered_points": (_i, [_vp, _i, _vp, _vp, _i]),
    "pgp_nearest_in_range": (_i, [_vp, _i, _vp, _vp]),
    "pgp_set_option": (_i, [_vp, C.c_char_p, _i]),
    "pgp_launch_count": (_i64, [_vp]),
    "pgp_topk": (_i, [_vp, _i, _i, _i64, _vp]),
    "pgp_topk_dev": (_i, [_vp, _i, _i, _i64, _vp]),
    "pgp_topk_merge": (_i, [_vp, _i, _i, _i, _vp]),
    "pgp_improving_chain": (_i, [_vp, _i, _i64, _vp, _i]),
    "pgp_set_symmetries": (_i, [_vp, _i, _vp, _i]),
    "pgp_distinct_dev": (_i, [_vp, _vp, _vp, _i, _vp, _i, C.c_double, C.c_double, _vp, _vp, _vp]),
    "pgp_topk_distinct": (_i, [_vp, _i, _i, _i, C.c_double, C.c_double, _vp]),
    "pgp_pcs_default_opts": (None, [_vp]),
    "pgp_extract_pairs": (_i, [_vp, _i, _f, _f, _vp, _i64, _vp]),
    "pgp_find_quads": (_i, [_vp, _i, _vp, _f, _f, _f, _vp, _i64, _vp, _i64, _vp, _i64, _vp]),
    "pgp_find_quads_v4pcs": (_i, [_vp, _i, _vp, _f, _vp, _i64, _vp]),
    "pgp_rigid_from_quads": (_i, [_vp, _i, _vp, _vp, _i64, _vp, _vp]),
    "pgp_generate_pcs": (_i, [_vp, _i, _vp, C.c_uint64, _i64, _vp]),
    "pgp_score_generated": (_i, [_vp, _i, _i]),
    "pgp_get_generated": (_i, [_vp, _i, _vp, _vp, _vp, _i64]),
    "pgp_set_ppf_map": (_i, [_vp, _i, _vp, _vp, _vp, _i64]),
    "pgp_build_ppf_map": (_i, [_vp, _i]),
    "pgp_get_ppf_map": (_i, [_vp, _i, _vp, _i64, _vp, _vp, _i64, _vp, _vp]),
    "pgp_scene_ppf_keys": (_i, [_vp, _vp, _i64, _vp]),
    "pgp_stocs_engine_seed": (C.c_uint32, [C.c_uint64, _i, _i]),
    "pgp_get_bases": (_i, [_vp, _i, _vp, _vp, _vp, _i]),
    "pgp_remove_explained": (_i, [_vp, _i, _vp, _i, _vp, _i, _f, _vp]),
    "pgp_mcts_tricp": (_i, [_vp, _i, _vp, _i, _vp, _i, _f, _vp, _i, _f, _f, _i, _vp, _vp, _vp]),
    "pgp_refine_batch": (_i, [_vp, _i, _vp, _vp, _i, _vp, _i64, _vp, _vp, _i, _vp, _f, _f, _f, _i, _vp, _vp, _vp]),
    "pgp_refine_batch_dev": (_i, [_vp, _i, _vp, _vp, _i, _vp, _i64, _vp, _vp, _i, _vp, _f, _f, _f, _i, _vp, _vp, _vp, _vp]),
    "pgp_prepare_segment": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _f, _f, _f, _i, _vp, _vp, _i, _vp]),
    "pgp_tricp": (_i, [_vp, _i, _vp, _i, _vp, _i, _f, _f, _i, _vp, _vp]),
    "pgp_tricp_plane": (_i, [_vp, _i, _vp, _i, _vp, _i, _f, _f, _i, _vp, _vp]),
    "pgp_set_mesh": (_i, [_vp, _i, _vp, _i, _vp, _i, _i]),
    "pgp_set_depth_observation": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp]),
    "pgp_render_depth": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "pgp_depth_cost": (_i, [_vp, _vp, _i, _vp, _vp, _f, _vp]),
    "pgp_depth_cost_dev": (_i, [_vp, _vp, _i, _vp, _vp, _f, _vp, _vp]),
    "pgp_render_depth_dev": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "pgp_set_depth_observation_dev": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp]),
    # multi-GPU
    "pgp_generate_pcs_range": (_i, [_vp, _i, _vp, C.c_uint64, _i, _i, _i64, _vp]),
    "pgp_topk_begin": (_i, [_vp, _i, _i, _i64]),
    "pgp_topk_end": (_i, [_vp, _i, _vp]),
    "pgp_topk_stream_wait": (_i, [_vp, _i]),
    "pgp_exchange_merge": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i]),
    "pgp_comm_unique_id": (_i, [_vp]),
    "pgp_comm_init": (_i, [_vp, _vp, _i, _i]),
    "pgp_comm_init_all": (_i, [_vp, _i]),
    "pgp_comm_rank": (_i, [_vp]),
    "pgp_comm_world": (_i, [_vp]),
    "pgp_comm_destroy": (_i, [_vp]),
    "pgp_comm_sync_generated": (_i, [_vp, _i, _i64, _vp, _vp]),
    "pgp_group_create": (_vp, [_i, _vp]),
    "pgp_group_destroy": (None, [_vp]),
    "pgp_group_size": (_i, [_vp]),
    "pgp_group_ctx": (_vp, [_vp, _i]),
    "pgp_group_last_error": (C.c_char_p, [_vp]),
    "pgp_group_set_scene": (_i, [_vp, _vp, _vp, _i, _f]),
    "pgp_group_set_scene_prior_image": (_i, [_vp, _vp, _i, _i, _vp]),
    "pgp_group_set_scene_priors": (_i, [_vp, _vp]),
    "pgp_group_set_model": (_i, [_vp, _i, _vp, _vp, _i, _vp, _vp, _i]),
    "pgp_group_set_ppf_map": (_i, [_vp, _i, _vp, _vp, _vp, _i64]),
    "pgp_group_build_ppf_map": (_i, [_vp, _i]),
    "pgp_group_generate_pcs": (_i, [_vp, _i, _vp, C.c_uint64, _i64, _vp]),
    "pgp_group_score_generated": (_i, [_vp, _i, _i]),
    "pgp_group_score_lcp": (_i, [_vp, _i, _vp, _i64, _i, _vp, _vp]),
    "pgp_group_topk": (_i, [_vp, _i, _i, _vp]),
    "pgp_group_improving_chain": (_i, [_vp, _i, _vp, _i]),
    "pgp_group_set_symmetries": (_i, [_vp, _i, _vp, _i]),
    "pgp_group_topk_distinct": (_i, [_vp, _i, _i, _i, C.c_double, C.c_double, _vp]),
    "pgp_bench_sector_gather": (_i, [_vp, _i64, _i, _vp]),
    "pgp_generated_cap_split": (_i, [_vp, _i, _i64, _i, _vp, _vp, _vp]),
    "pgp_host_chain_sum_equal": (C.c_float, [C.c_float, C.c_longlong]),
    "pgp_host_max_eigvec4": (_i, [_vp, _vp]),
    "pgp_host_solve_plane6": (_i, [_vp, _vp, _vp]),
}

_lib = None


def load() -> C.CDLL:
    """Loads libpgp.so; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(or `make -C physimglobalpose_b200/csrc`).  There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header / library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def exported_symbols() -> list[str]:
    return sorted(_SIGNATURES)
