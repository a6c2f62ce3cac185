"""ctypes binding of the C ABI in include/psulvsb.h (libpsulvsb_b200.so).

This is the host-side plumbing of the product: it loads the CUDA library and fails loudly when it
is missing -- there is no CPU fallback and nothing here imports the oracle.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpsulvsb_b200.so")

OK, ERR_INVALID, ERR_CUDA, ERR_NO_DEVICE, ERR_CAPACITY, ERR_UNSUPPORTED, ERR_INTERNAL = range(7)
DOMAIN_L_SAMPLED, DOMAIN_BASIC, DOMAIN_UNIFORM, DOMAIN_SCALE, DOMAIN_TUPLE = 1, 2, 3, 4, 5

# every symbol include/psulvsb.h declares (checked by tests/test_capi_symbols.py against the header)
SYMBOLS = [
    "psulvsb_version", "psulvsb_last_error", "psulvsb_default_params", "psulvsb_device_count",
    "psulvsb_create", "psulvsb_destroy", "psulvsb_solve", "psulvsb_solve_batch", "psulvsb_batch_upload",
    "psulvsb_batch_solve_resident", "psulvsb_batch_submit", "psulvsb_batch_wait", "psulvsb_batch_resident_size", "psulvsb_debug_set", "psulvsb_launch_count", "psulvsb_last_device_ms", "psulvsb_last_stage_ms",
    "psulvsb_last_ticks", "psulvsb_last_chunk_ticks", "psulvsb_set_batching", "psulvsb_set_host_threads", "psulvsb_pack_points", "psulvsb_consistency_mask", "psulvsb_consistency_mask_rows",
    "psulvsb_mask_symmetrize", "psulvsb_compact_edges", "psulvsb_ratio_reduced_set", "psulvsb_sample_workspace_bytes",
    "psulvsb_sample_default_max_draws", "psulvsb_sample", "psulvsb_philox_fill", "psulvsb_gnc_tls_rotation",
    "psulvsb_kabsch_batch", "psulvsb_tls_translation", "psulvsb_score_batch", "psulvsb_score_one",
    "psulvsb_max_clique", "psulvsb_max_clique_scratch_words", "psulvsb_gnc_tls_rotation_batch",
    "psulvsb_compute_tims_host", "psulvsb_scale_inliers_host", "psulvsb_tls_scale_host",
    "psulvsb_gnc_tls_rotation_host", "psulvsb_tls_translation_host", "psulvsb_estimate_normals", "psulvsb_estimate_normals_host",
    "psulvsb_comm_unique_id", "psulvsb_comm_create", "psulvsb_comm_destroy", "psulvsb_comm_rank", "psulvsb_comm_world",
    "psulvsb_comm_allreduce_sum_u32", "psulvsb_comm_allreduce_max_u64", "psulvsb_score_batch_sharded",
    "psulvsb_solve_sharded", "psulvsb_shard_row_range",
    "psulvsb_fpfh_workspace_bytes", "psulvsb_fpfh", "psulvsb_fpfh_host", "psulvsb_feature_nn", "psulvsb_match_host",
    "psulvsb_icp_default_params", "psulvsb_icp_workspace_bytes", "psulvsb_icp", "psulvsb_icp_host",
    "psulvsb_icp_batch_workspace_bytes", "psulvsb_icp_batch", "psulvsb_icp_batch_host",
    "psulvsb_fpfh_batch_workspace_bytes", "psulvsb_fpfh_batch", "psulvsb_fpfh_batch_host",
    "psulvsb_match_batch_workspace_bytes", "psulvsb_match_batch", "psulvsb_match_batch_host",
    "psulvsb_gicp", "psulvsb_gicp_host", "psulvsb_gicp_batch_workspace_bytes", "psulvsb_gicp_batch",
    "psulvsb_gicp_batch_host",
    "psulvsb_normals_workspace_bytes", "psulvsb_normals", "psulvsb_normals_host",
    "psulvsb_normals_batch_workspace_bytes", "psulvsb_normals_batch", "psulvsb_normals_batch_host",
    "psulvsb_voxel_down_sample_workspace_bytes", "psulvsb_voxel_down_sample", "psulvsb_voxel_down_sample_host",
    "psulvsb_voxel_down_sample_batch_workspace_bytes", "psulvsb_voxel_down_sample_batch",
    "psulvsb_voxel_down_sample_batch_host",
]
UNIQUE_ID_BYTES = 128


class PsulvsbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"psulvsb error {code}: {msg}")
        self.code = code


class Params(C.Structure):
    """psulvsb_params_t == RobustRegistrationSolver::Params (registration.h:378-473) + lifted constants."""
    _fields_ = [
        ("noise_bound", C.c_double),
        ("cbar2", C.c_double),
        ("estimate_scaling", C.c_int),
        ("rotation_max_iterations", C.c_int),
        ("rotation_gnc_factor", C.c_double),
        ("rotation_cost_threshold", C.c_double),
        ("inlier_selection_mode", C.c_int),
        ("kcore_heuristic_threshold", C.c_double),
        ("score_noise_bound", C.c_double),
        ("inloop_noise_bound", C.c_double),
        ("inloop_cbar2", C.c_double),
        ("inloop_max_iterations", C.c_int),
        ("inloop_gnc_factor", C.c_double),
        ("inloop_cost_threshold", C.c_double),
        ("rotation_similar", C.c_double),
        ("local_max_iter", C.c_int),
        ("tpro_host", C.c_double),
        ("tpro_local", C.c_double),
        ("host_round_limit", C.c_int),
        ("wallclock_cap_s", C.c_double),
        ("self_update", C.c_int),
        ("seed", C.c_uint64),
    ]


class Problem(C.Structure):
    _fields_ = [
        ("src", C.POINTER(C.c_double)),
        ("dst", C.POINTER(C.c_double)),
        ("C", C.c_int),
        ("ori_src", C.POINTER(C.c_double)),
        ("ori_dst", C.POINTER(C.c_double)),
        ("M", C.c_int),
        ("keep_mask", C.POINTER(C.c_int)),
        ("reduce_map", C.POINTER(C.c_int)),
    ]


class Solution(C.Structure):
    _fields_ = [
        ("valid", C.c_int),
        ("scale", C.c_double),
        ("final_inlier_count", C.c_int),
        ("translation", C.c_double * 3),
        ("rotation", C.c_double * 9),
        ("host_rounds", C.c_int),
        ("local_iters", C.c_int),
        ("n_line_vectors", C.c_longlong),
        ("n_reduced", C.c_longlong),
        ("final_C", C.c_int),
        ("refined", C.c_int),
        ("escalations", C.c_int),
        ("borderline_pairs", C.c_longlong),
        ("status", C.c_int),
    ]

    @property
    def R(self) -> np.ndarray:
        return np.array(self.rotation[:]).reshape(3, 3, order="F")

    @property
    def t(self) -> np.ndarray:
        return np.array(self.translation[:])


class LocalTrace(C.Structure):
    _fields_ = [
        ("host_round", C.c_int), ("local_iter", C.c_int), ("n_sampled_lines", C.c_int),
        ("n_sampled_points", C.c_int), ("basic_choose", C.c_int), ("gnc_iterations", C.c_int),
        ("rot_inliers", C.c_int), ("n_rot_points", C.c_int), ("similar", C.c_int), ("curr_count", C.c_int),
        ("best_count", C.c_int), ("local_r", C.c_int),
        ("p_local", C.c_double), ("l_rate", C.c_double), ("b_rate", C.c_double), ("scale", C.c_double),
        ("R", C.c_double * 9), ("t", C.c_double * 3),
    ]


class HostTrace(C.Structure):
    _fields_ = [
        ("host_round", C.c_int), ("curr_count", C.c_int), ("best_host", C.c_int), ("new_corr_count", C.c_int),
        ("inlier_map_size", C.c_int), ("host_r", C.c_int), ("p_host", C.c_double),
    ]


class Trace(C.Structure):
    _fields_ = [
        ("local", C.POINTER(LocalTrace)), ("local_cap", C.c_int), ("local_n", C.c_int),
        ("host", C.POINTER(HostTrace)), ("host_cap", C.c_int), ("host_n", C.c_int),
        ("final_inliers", C.POINTER(C.c_int)), ("inlier_counter", C.POINTER(C.c_int)),
        ("reduce_map_out", C.POINTER(C.c_int)),
    ]


class IcpParams(C.Structure):
    """psulvsb_icp_params_t."""
    _fields_ = [
        ("max_correspondence_distance", C.c_double),
        ("relative_fitness", C.c_double),
        ("relative_rmse", C.c_double),
        ("max_iterations", C.c_int),
        ("point_to_plane", C.c_int),
    ]


class IcpResult(C.Structure):
    """psulvsb_icp_result_t (rotation column-major)."""
    _fields_ = [
        ("rotation", C.c_double * 9),
        ("translation", C.c_double * 3),
        ("fitness", C.c_double),
        ("inlier_rmse", C.c_double),
        ("n_correspondences", C.c_int),
        ("iterations", C.c_int),
        ("status", C.c_int),
    ]


class IcpIteration(C.Structure):
    """psulvsb_icp_iteration_t: the evaluation of T_k."""
    _fields_ = [
        ("rotation", C.c_double * 9),
        ("translation", C.c_double * 3),
        ("fitness", C.c_double),
        ("inlier_rmse", C.c_double),
        ("n_correspondences", C.c_int),
    ]


class IcpPair(C.Structure):
    """psulvsb_icp_pair_t: one problem of a batch (R0 column-major)."""
    _fields_ = [
        ("src", C.c_void_p),
        ("n_s", C.c_int),
        ("tgt", C.c_void_p),
        ("n_t", C.c_int),
        ("tgt_normals", C.c_void_p),
        ("R0", C.c_double * 9),
        ("t0", C.c_double * 3),
    ]


class GicpPair(C.Structure):
    """psulvsb_gicp_pair_t: one generalized-ICP problem of a batch (R0 column-major)."""
    _fields_ = [
        ("src", C.c_void_p),
        ("n_s", C.c_int),
        ("tgt", C.c_void_p),
        ("n_t", C.c_int),
        ("src_normals", C.c_void_p),
        ("tgt_normals", C.c_void_p),
        ("R0", C.c_double * 9),
        ("t0", C.c_double * 3),
    ]


class FpfhCloud(C.Structure):
    """psulvsb_fpfh_cloud_t: one cloud of an FPFH batch."""
    _fields_ = [
        ("pts", C.c_void_p),
        ("n", C.c_int),
        ("viewpoint", C.c_double * 3),
    ]


class MatchPair(C.Structure):
    """psulvsb_match_pair_t: one pair of a matcher batch."""
    _fields_ = [
        ("src", C.c_void_p),
        ("n_src", C.c_int),
        ("tgt", C.c_void_p),
        ("n_tgt", C.c_int),
        ("fs", C.c_void_p),
        ("ft", C.c_void_p),
        ("seed", C.c_uint64),
    ]


_lib = None
_vp = C.c_void_p
_ull = C.c_ulonglong


def lib() -> C.CDLL:
    """Loads libpsulvsb_b200.so; raises if it has not been built (no fallback of any kind)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PsulvsbError(ERR_INTERNAL, f"{LIB_PATH} is missing: run __graft_entry__.build() "
                                             "(nvcc, sm_100a); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        _declare(L)
        _lib = L
    return _lib


def _declare(L: C.CDLL) -> None:
    L.psulvsb_version.restype = C.c_int
    L.psulvsb_last_error.restype = C.c_char_p
    L.psulvsb_default_params.argtypes = [C.POINTER(Params)]
    L.psulvsb_default_params.restype = None
    L.psulvsb_device_count.restype = C.c_int
    L.psulvsb_create.argtypes = [C.POINTER(_vp), C.c_int]
    L.psulvsb_destroy.argtypes = [_vp]
    L.psulvsb_solve.argtypes = [_vp, C.POINTER(Params), C.POINTER(Problem), C.POINTER(Solution), C.POINTER(Trace)]
    L.psulvsb_solve_batch.argtypes = [_vp, C.POINTER(Params), C.POINTER(Problem), C.c_int, C.POINTER(C.c_uint64),
                                      C.POINTER(Solution)]
    L.psulvsb_batch_submit.argtypes = [_vp, C.POINTER(Params), C.POINTER(Problem), C.c_int, C.POINTER(C.c_uint64),
                                       C.POINTER(Solution), C.POINTER(C.c_uint64)]
    L.psulvsb_batch_wait.argtypes = [_vp, C.c_uint64]
    L.psulvsb_batch_upload.argtypes = [_vp, C.POINTER(Problem), C.c_int]
    L.psulvsb_batch_solve_resident.argtypes = [_vp, C.POINTER(Params), C.POINTER(C.c_uint64), C.POINTER(Solution),
                                               C.c_int]
    L.psulvsb_debug_set.argtypes = [C.c_char_p, C.c_double]
    L.psulvsb_batch_resident_size.argtypes = [_vp]
    L.psulvsb_batch_resident_size.restype = C.c_int
    L.psulvsb_launch_count.argtypes = [_vp]
    L.psulvsb_launch_count.restype = C.c_longlong
    L.psulvsb_last_device_ms.argtypes = [_vp]
    L.psulvsb_last_device_ms.restype = C.c_double
    L.psulvsb_last_stage_ms.argtypes = [_vp, C.c_int]
    L.psulvsb_last_stage_ms.restype = C.c_double
    L.psulvsb_last_ticks.argtypes = [_vp]
    L.psulvsb_last_ticks.restype = C.c_int
    L.psulvsb_last_chunk_ticks.argtypes = [_vp, C.POINTER(C.c_int), C.c_int]
    L.psulvsb_last_chunk_ticks.restype = C.c_int
    L.psulvsb_set_batching.argtypes = [_vp, C.c_int, C.c_int]
    L.psulvsb_set_host_threads.argtypes = [_vp, C.c_int]
    L.psulvsb_pack_points.argtypes = [_vp, _vp, C.c_int, C.POINTER(C.c_double), _vp]
    L.psulvsb_consistency_mask.argtypes = [_vp, _vp, _vp, _vp, _vp, C.c_int, C.c_double, C.c_double, _vp, C.c_int,
                                           _vp, _vp]
    L.psulvsb_consistency_mask_rows.argtypes = [_vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_double,
                                                C.c_double, _vp, C.c_int, _vp, _vp]
    L.psulvsb_mask_symmetrize.argtypes = [_vp, _vp, C.c_int, C.c_int]
    L.psulvsb_compact_edges.argtypes = [_vp, _vp, C.c_int, C.c_int, _vp, _vp, _vp, _ull, _vp]
    L.psulvsb_ratio_reduced_set.argtypes = [_vp, _vp, _vp, C.c_int, _vp, _vp, _ull, C.POINTER(_ull),
                                            C.POINTER(C.c_double), C.POINTER(C.c_uint)]
    L.psulvsb_sample_workspace_bytes.argtypes = [_ull, _ull, _ull]
    L.psulvsb_sample_workspace_bytes.restype = _ull
    L.psulvsb_sample_default_max_draws.argtypes = [_ull, _ull]
    L.psulvsb_sample_default_max_draws.restype = _ull
    L.psulvsb_sample.argtypes = [_vp, C.c_uint64, C.c_uint32, C.c_uint32, _ull, _ull, _ull, _vp, _vp, _vp]
    L.psulvsb_philox_fill.argtypes = [_vp, C.c_uint64, C.c_uint32, C.c_uint32, _ull, _ull, _vp]
    L.psulvsb_gnc_tls_rotation.argtypes = [_vp, _vp, _vp, _vp, _ull, C.c_double, C.c_double, C.c_int, C.c_double,
                                           C.c_double, _vp, _vp, _vp, _vp, _vp, _vp]
    L.psulvsb_kabsch_batch.argtypes = [_vp, _vp, _vp, _vp, _vp, C.c_int, _ull, _vp, _vp]
    L.psulvsb_tls_translation.argtypes = [_vp, _vp, _vp, _vp, C.c_int, C.c_double, _vp, C.c_double, _vp, _vp, _vp]
    L.psulvsb_score_batch.argtypes = [_vp, _vp, _vp, _vp, _vp, C.c_int, _vp, _ull, _ull, C.c_double, C.c_double,
                                      C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double), _vp, _vp, _vp]
    L.psulvsb_estimate_normals.argtypes = [_vp, _vp, C.c_int, C.c_int, C.POINTER(C.c_double), _vp]
    L.psulvsb_estimate_normals_host.argtypes = [C.POINTER(C.c_double), C.c_int, C.c_int, C.POINTER(C.c_double),
                                                C.POINTER(C.c_double)]
    L.psulvsb_max_clique.argtypes = [_vp, _vp, _ull, C.c_int, _vp, _vp, _vp, C.c_int]
    L.psulvsb_max_clique_scratch_words.argtypes = [C.c_int]
    L.psulvsb_gnc_tls_rotation_batch.argtypes = [_vp, _vp, _vp, C.c_int, _vp, _ull, C.c_int, C.c_double, C.c_int,
                                                 C.c_double, C.c_double, C.c_int, _vp, _vp, _ull, _vp, _vp, _vp, _vp, _vp]
    L.psulvsb_compute_tims_host.argtypes = [_vp, C.c_int, _vp, _vp]
    L.psulvsb_scale_inliers_host.argtypes = [_vp, _vp, _ull, C.c_double, C.c_double, _vp]
    L.psulvsb_tls_scale_host.argtypes = [_vp, _vp, C.c_int, C.c_double, C.c_double, C.c_uint64, C.c_uint32, _vp, _vp, _vp]
    L.psulvsb_gnc_tls_rotation_host.argtypes = [_vp, _vp, _ull, C.c_double, C.c_int, C.c_double, C.c_double, _vp, _vp,
                                                _vp, _vp, _vp]
    L.psulvsb_tls_translation_host.argtypes = [_vp, _vp, C.c_int, C.c_double, C.c_double, _vp, _vp, _vp]
    L.psulvsb_max_clique_scratch_words.restype = _ull
    L.psulvsb_comm_unique_id.argtypes = [_vp]
    L.psulvsb_comm_create.argtypes = [_vp, C.c_int, C.c_int, _vp]
    L.psulvsb_comm_destroy.argtypes = [_vp]
    L.psulvsb_comm_rank.argtypes = [_vp]
    L.psulvsb_comm_world.argtypes = [_vp]
    L.psulvsb_comm_allreduce_sum_u32.argtypes = [_vp, _vp, _vp, _ull]
    L.psulvsb_comm_allreduce_max_u64.argtypes = [_vp, _vp, _vp, _ull]
    L.psulvsb_score_batch_sharded.argtypes = [_vp] + list(L.psulvsb_score_batch.argtypes)
    L.psulvsb_solve_sharded.argtypes = [_vp, C.POINTER(Params), C.POINTER(Problem), C.POINTER(Solution), C.POINTER(Trace)]
    L.psulvsb_shard_row_range.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.psulvsb_score_one.argtypes = [_vp, _vp, _vp, C.c_int, C.c_double, _vp, _vp, C.c_double, _vp, _vp, _vp]
    L.psulvsb_fpfh_workspace_bytes.argtypes = [C.c_int]
    L.psulvsb_fpfh_workspace_bytes.restype = _ull
    L.psulvsb_fpfh.argtypes = [_vp, _vp, C.c_int, C.c_double, C.c_double, C.POINTER(C.c_double), _vp, _vp, _vp]
    L.psulvsb_fpfh_host.argtypes = [_vp, C.c_int, C.c_double, C.c_double, C.POINTER(C.c_double), _vp, _vp]
    L.psulvsb_feature_nn.argtypes = [_vp, _vp, C.c_int, _vp, C.c_int, _vp, _vp]
    L.psulvsb_match_host.argtypes = [_vp, C.c_int, _vp, C.c_int, _vp, _vp, C.c_int, C.c_int, C.c_double, C.c_uint64,
                                     _vp, C.c_longlong, C.POINTER(C.c_longlong)]
    L.psulvsb_icp_default_params.argtypes = [C.POINTER(IcpParams)]
    L.psulvsb_icp_default_params.restype = None
    L.psulvsb_icp_workspace_bytes.argtypes = [C.c_int, C.c_int]
    L.psulvsb_icp_workspace_bytes.restype = _ull
    L.psulvsb_icp.argtypes = [_vp, _vp, C.c_int, _vp, C.c_int, _vp, C.POINTER(IcpParams), C.POINTER(C.c_double),
                              C.POINTER(C.c_double), _vp, _vp, _vp, _vp]
    L.psulvsb_icp_host.argtypes = [_vp, C.c_int, _vp, C.c_int, _vp, C.POINTER(IcpParams), C.POINTER(C.c_double),
                                   C.POINTER(C.c_double), _vp, _vp, _vp]
    L.psulvsb_icp_batch_workspace_bytes.argtypes = [C.POINTER(IcpPair), C.c_int]
    L.psulvsb_icp_batch_workspace_bytes.restype = _ull
    L.psulvsb_icp_batch.argtypes = [_vp, C.POINTER(IcpPair), C.c_int, C.POINTER(IcpParams), _vp, _vp, _vp, _vp]
    L.psulvsb_icp_batch_host.argtypes = [C.POINTER(IcpPair), C.c_int, C.POINTER(IcpParams), _vp, _vp, _vp]
    L.psulvsb_gicp.argtypes = [_vp, _vp, C.c_int, _vp, _vp, C.c_int, _vp, C.POINTER(IcpParams), C.c_double,
                               C.POINTER(C.c_double), C.POINTER(C.c_double), _vp, _vp, _vp, _vp]
    L.psulvsb_gicp_host.argtypes = [_vp, C.c_int, _vp, _vp, C.c_int, _vp, C.POINTER(IcpParams), C.c_double,
                                    C.POINTER(C.c_double), C.POINTER(C.c_double), _vp, _vp, _vp]
    L.psulvsb_gicp_batch_workspace_bytes.argtypes = [C.POINTER(GicpPair), C.c_int]
    L.psulvsb_gicp_batch_workspace_bytes.restype = _ull
    L.psulvsb_gicp_batch.argtypes = [_vp, C.POINTER(GicpPair), C.c_int, C.POINTER(IcpParams), C.c_double, _vp, _vp,
                                     _vp, _vp]
    L.psulvsb_gicp_batch_host.argtypes = [C.POINTER(GicpPair), C.c_int, C.POINTER(IcpParams), C.c_double, _vp, _vp,
                                          _vp]
    L.psulvsb_fpfh_batch_workspace_bytes.argtypes = [C.POINTER(FpfhCloud), C.c_int]
    L.psulvsb_fpfh_batch_workspace_bytes.restype = _ull
    L.psulvsb_fpfh_batch.argtypes = [_vp, C.POINTER(FpfhCloud), C.c_int, C.c_double, C.c_double, _vp, _vp, _vp]
    L.psulvsb_fpfh_batch_host.argtypes = [C.POINTER(FpfhCloud), C.c_int, C.c_double, C.c_double, _vp, _vp]
    L.psulvsb_normals_workspace_bytes.argtypes = [C.c_int]
    L.psulvsb_normals_workspace_bytes.restype = _ull
    L.psulvsb_normals.argtypes = [_vp, _vp, C.c_int, C.c_double, C.c_int, C.POINTER(C.c_double), _vp, _vp]
    L.psulvsb_normals_host.argtypes = [_vp, C.c_int, C.c_double, C.c_int, C.POINTER(C.c_double), _vp]
    L.psulvsb_normals_batch_workspace_bytes.argtypes = [C.POINTER(FpfhCloud), C.c_int]
    L.psulvsb_normals_batch_workspace_bytes.restype = _ull
    L.psulvsb_normals_batch.argtypes = [_vp, C.POINTER(FpfhCloud), C.c_int, C.c_double, C.c_int, _vp, _vp]
    L.psulvsb_normals_batch_host.argtypes = [C.POINTER(FpfhCloud), C.c_int, C.c_double, C.c_int, _vp]
    L.psulvsb_voxel_down_sample_workspace_bytes.argtypes = [C.c_int]
    L.psulvsb_voxel_down_sample_workspace_bytes.restype = _ull
    L.psulvsb_voxel_down_sample.argtypes = [_vp, _vp, C.c_int, C.c_double, _vp, _vp, _vp]
    L.psulvsb_voxel_down_sample_host.argtypes = [_vp, C.c_int, C.c_double, _vp, _vp]
    L.psulvsb_voxel_down_sample_batch_workspace_bytes.argtypes = [C.POINTER(FpfhCloud), C.c_int]
    L.psulvsb_voxel_down_sample_batch_workspace_bytes.restype = _ull
    L.psulvsb_voxel_down_sample_batch.argtypes = [_vp, C.POINTER(FpfhCloud), C.c_int, C.c_double, _vp, _vp, _vp]
    L.psulvsb_voxel_down_sample_batch_host.argtypes = [C.POINTER(FpfhCloud), C.c_int, C.c_double, _vp, _vp]
    L.psulvsb_match_batch_workspace_bytes.argtypes = [C.POINTER(MatchPair), C.c_int, C.c_int, C.c_int]
    L.psulvsb_match_batch_workspace_bytes.restype = _ull
    L.psulvsb_match_batch.argtypes = [_vp, C.POINTER(MatchPair), C.c_int, C.c_int, C.c_int, C.c_double, _vp, _vp, _vp]
    L.psulvsb_match_batch_host.argtypes = [C.POINTER(MatchPair), C.c_int, C.c_int, C.c_int, C.c_double, _vp, _vp]
    for name in SYMBOLS:
        getattr(L, name)  # AttributeError here = the library does not export what the header declares


def check(rc: int) -> None:
    if rc != OK:
        raise PsulvsbError(rc, lib().psulvsb_last_error().decode("utf-8", "replace"))


def debug_set(name: str, value: float) -> None:
    """psulvsb_debug_set: test switches between equivalent code paths ("reset" restores the defaults)."""
    check(lib().psulvsb_debug_set(name.encode(), float(value)))


def comm_unique_id() -> bytes:
    """psulvsb_comm_unique_id: rank 0 makes it, the caller carries the bytes to the other ranks."""
    buf = C.create_string_buffer(UNIQUE_ID_BYTES)
    check(lib().psulvsb_comm_unique_id(buf))
    return buf.raw


def shard_row_range(n: int, rank: int, world: int):
    """psulvsb_shard_row_range: the consistency rows psulvsb_solve_sharded gives `rank` (host arithmetic)."""
    b, e = C.c_int(0), C.c_int(0)
    check(lib().psulvsb_shard_row_range(n, rank, world, C.byref(b), C.byref(e)))
    return b.value, e.value


def default_params(**kw) -> Params:
    p = Params()
    lib().psulvsb_default_params(C.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise AttributeError(k)
        setattr(p, k, v)
    return p


def _cm(a) -> np.ndarray:
    a = np.asarray(a, dtype=np.float64)
    if a.ndim != 2 or a.shape[0] != 3:
        raise ValueError(f"expected a 3xN matrix, got {a.shape}")
    return np.asfortranarray(a)


_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


class HostProblem:
    """Owns the host arrays of one registration problem in the C ABI's layout (column-major 3xN)."""

    def __init__(self, src, dst, ori_src=None, ori_dst=None, keep_mask=None, reduce_map=None):
        self.src = _cm(src)
        self.dst = _cm(dst)
        if self.src.shape != self.dst.shape:
            raise ValueError("src and dst must have the same shape")
        if ori_src is None:
            ori_src, ori_dst = self.src, self.dst
        self.ori_src = _cm(ori_src)
        self.ori_dst = _cm(ori_dst)
        M = self.ori_src.shape[1]
        if keep_mask is None:
            if self.src.shape[1] != M:
                raise ValueError("keep_mask / reduce_map are required when C != M")
            keep_mask = np.ones(M, dtype=np.int32)
            reduce_map = np.arange(M, dtype=np.int32)
        self.keep_mask = np.ascontiguousarray(keep_mask, dtype=np.int32)
        self.reduce_map = np.ascontiguousarray(reduce_map, dtype=np.int32)
        if self.keep_mask.size != M or self.reduce_map.size != M:
            raise ValueError("keep_mask / reduce_map must have M entries")

    @property
    def nbytes(self) -> int:
        """Bytes the library copies to the device for this problem (ori_* passed as the very same arrays as src / dst
        -- no pre-filter -- are uploaded once)."""
        aliased = (self.ori_src.ctypes.data == self.src.ctypes.data and self.ori_dst.ctypes.data == self.dst.ctypes.data
                   and self.ori_src.shape == self.src.shape)
        ori = 0 if aliased else self.ori_src.nbytes + self.ori_dst.nbytes
        return self.src.nbytes + self.dst.nbytes + ori + self.keep_mask.nbytes + self.reduce_map.nbytes

    def c_struct(self) -> Problem:
        if getattr(self, "_cs", None) is None:  # the arrays are owned by this object: build the view once
            self._cs = self._build_c_struct()
        return self._cs

    def _build_c_struct(self) -> Problem:
        return Problem(self.src.ctypes.data_as(_dp), self.dst.ctypes.data_as(_dp), self.src.shape[1],
                       self.ori_src.ctypes.data_as(_dp), self.ori_dst.ctypes.data_as(_dp), self.ori_src.shape[1],
                       self.keep_mask.ctypes.data_as(_ip), self.reduce_map.ctypes.data_as(_ip))


class Handle:
    """psulvsb_handle_t: one device, one stream, private arenas."""

    def __init__(self, device: int = 0):
        self._h = _vp()
        check(lib().psulvsb_create(C.byref(self._h), device))
        self._problems = None

    def close(self) -> None:
        if self._h:
            lib().psulvsb_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def solve(self, params: Params, problem: HostProblem, trace_cap: int = 0):
        sol = Solution()
        if trace_cap > 0:
            M = problem.ori_src.shape[1]
            loc = (LocalTrace * trace_cap)()
            hst = (HostTrace * trace_cap)()
            fin = np.zeros(M, dtype=np.int32)
            cnt = np.zeros(M, dtype=np.int32)
            rmap = np.zeros(M, dtype=np.int32)
            tr = Trace(C.cast(loc, C.POINTER(LocalTrace)), trace_cap, 0, C.cast(hst, C.POINTER(HostTrace)), trace_cap,
                       0, fin.ctypes.data_as(_ip), cnt.ctypes.data_as(_ip), rmap.ctypes.data_as(_ip))
            ps = problem.c_struct()
            check(lib().psulvsb_solve(self._h, C.byref(params), C.byref(ps), C.byref(sol), C.byref(tr)))
            trace = {"local": [loc[i] for i in range(tr.local_n)], "host": [hst[i] for i in range(tr.host_n)],
                     "final_inliers": fin, "inlier_counter": cnt, "reduce_map": rmap}
            return sol, trace
        ps = problem.c_struct()
        check(lib().psulvsb_solve(self._h, C.byref(params), C.byref(ps), C.byref(sol), None))
        return sol, None

    @staticmethod
    def _problem_array(problems):
        arr = (Problem * len(problems))()
        for i, p in enumerate(problems):
            arr[i] = p.c_struct()
        return arr

    def solve_batch(self, params: Params, problems, seeds=None):
        arr = self._problem_array(problems)
        sols = (Solution * len(problems))()
        sd = None
        if seeds is not None:
            sd = (C.c_uint64 * len(problems))(*[int(s) for s in seeds])
        check(lib().psulvsb_solve_batch(self._h, C.byref(params), arr, len(problems), sd, sols))
        return list(sols)

    def submit(self, params: Params, problems, seeds=None):
        """psulvsb_batch_submit: queue a batch, return a ticket for wait().  The ticket keeps the host arrays alive."""
        arr = self._problem_array(problems)
        sols = (Solution * len(problems))()
        sd = None
        if seeds is not None:
            sd = (C.c_uint64 * len(problems))(*[int(s) for s in seeds])
        tk = C.c_uint64(0)
        check(lib().psulvsb_batch_submit(self._h, C.byref(params), arr, len(problems), sd, sols, C.byref(tk)))
        return (tk.value, sols, arr, sd, list(problems))

    def wait(self, ticket):
        """psulvsb_batch_wait: the solutions of a submitted batch."""
        check(lib().psulvsb_batch_wait(self._h, C.c_uint64(ticket[0])))
        return list(ticket[1])

    def upload(self, problems) -> None:
        self._problems = list(problems)  # keep the host arrays alive
        arr = self._problem_array(self._problems)
        check(lib().psulvsb_batch_upload(self._h, arr, len(self._problems)))

    @property
    def resident_size(self) -> int:
        return lib().psulvsb_batch_resident_size(self._h)

    def solve_resident(self, params: Params, seeds=None):
        n = self.resident_size  # (solve / solve_batch on this handle replace the resident batch)
        if n <= 0:
            raise PsulvsbError(ERR_INVALID, "solve_resident: nothing is resident on this handle (upload first)")
        sols = (Solution * n)()
        sd = None
        if seeds is not None:
            if len(seeds) != n:
                raise PsulvsbError(ERR_INVALID, f"solve_resident: {len(seeds)} seeds for a resident batch of {n}")
            sd = (C.c_uint64 * n)(*[int(s) for s in seeds])
        check(lib().psulvsb_batch_solve_resident(self._h, C.byref(params), sd, sols, n))
        return list(sols)

    def set_host_threads(self, n: int = 0) -> None:
        """psulvsb_set_host_threads: staging threads of uploads (0 = the CPUs available to the process)."""
        check(lib().psulvsb_set_host_threads(self._h, n))

    def comm_create(self, rank: int, world: int, unique_id: bytes) -> None:
        if len(unique_id) != UNIQUE_ID_BYTES:
            raise ValueError("unique_id must have UNIQUE_ID_BYTES bytes")
        check(lib().psulvsb_comm_create(self._h, rank, world, C.c_char_p(unique_id)))

    def comm_destroy(self) -> None:
        check(lib().psulvsb_comm_destroy(self._h))

    @property
    def comm_world(self) -> int:
        return lib().psulvsb_comm_world(self._h)

    def comm_allreduce_sum_u32(self, d_ptr: int, n: int, stream: int = 0) -> None:
        check(lib().psulvsb_comm_allreduce_sum_u32(self._h, stream, d_ptr, n))

    def comm_allreduce_max_u64(self, d_ptr: int, n: int, stream: int = 0) -> None:
        check(lib().psulvsb_comm_allreduce_max_u64(self._h, stream, d_ptr, n))

    def solve_sharded(self, params: Params, problem: HostProblem) -> Solution:
        """psulvsb_solve_sharded: every rank passes the same problem; the consistency rows are split over the ranks."""
        sol = Solution()
        ps = problem.c_struct()
        check(lib().psulvsb_solve_sharded(self._h, C.byref(params), C.byref(ps), C.byref(sol), None))
        return sol

    @property
    def launch_count(self) -> int:
        return lib().psulvsb_launch_count(self._h)

    @property
    def last_device_ms(self) -> float:
        return lib().psulvsb_last_device_ms(self._h)

    def last_stage_ms(self, which: int) -> float:
        return lib().psulvsb_last_stage_ms(self._h, which)

    @property
    def last_ticks(self) -> int:
        return lib().psulvsb_last_ticks(self._h)

    @property
    def last_chunk_ticks(self):
        buf = (C.c_int * 256)()
        n = lib().psulvsb_last_chunk_ticks(self._h, buf, 256)
        return [buf[i] for i in range(min(n, 256))]

    def set_batching(self, chunk: int = 0, lanes: int = 0) -> None:
        """psulvsb_set_batching: registrations per lock-step chunk / chunks in flight (0 = defaults)."""
        check(lib().psulvsb_set_batching(self._h, chunk, lanes))
