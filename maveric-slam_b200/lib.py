"""ctypes binding of libmaveric_b200.so (the drop-in C ABI).

The library is the product; there is no Python or CPU fallback.  Loading fails with an
explicit error if the shared object has not been built (``python maveric-slam_b200/build.py``
or ``__graft_entry__.build()``), and creating a context fails with ``MV_ERR_NO_DEVICE`` when no
sm_100 GPU is visible.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# MV_LIB_PATH: an A/B build of the same library (build.py MV_OUT=...); never anything but this library
SO_PATH = os.environ.get("MV_LIB_PATH") or os.path.join(HERE, "libmaveric_b200.so")

MV_OK, MV_ERR_NO_DEVICE, MV_ERR_CUDA, MV_ERR_BAD_ARG, MV_ERR_TOO_MANY_VALID = range(5)

# Every symbol include/maveric_b200.h and include/maveric_slam_compat.h declare.
NEW_SYMBOLS = [
    "mv_ctx_create", "mv_ctx_destroy", "mv_ctx_set_stream", "mv_ctx_sync", "mv_last_error", "mv_status_str",
    "mv_ctx_launch_count", "mv_ctx_profile", "mv_ctx_profile_read", "mv_ctx_pnp_work", "mv_ctx_match_work", "mv_pnp_has_ab_forms", "mv_softmax_batch", "mv_top_n_batch",
    "compute_softmax_ex", "compute_top_N_ex", "mv_match_params_default", "mv_match_batch",
    "mv_match_pair_host", "mv_ransac_identity_batch", "mv_pnp_params_default", "mv_pnp_gn_batch",
    "mv_build_corr_batch", "mv_track_params_default", "mv_track_sequence", "mv_track_sequence_host",
    "mv_chain_transforms", "mv_results_to_transforms", "mv_nms_batch", "run_nms_ex", "mv_synth_frames",
    "mv_lba_schur_batch",
    "mv_lba_solve_batch",
    "mv_bow_set_vocabulary", "mv_bow_assign_batch", "mv_landmarks_init", "mv_landmarks_observe",
    "mv_landmarks_remove_old", "mv_landmarks_lookup", "mv_build_corr_landmarks_batch", "mv_landmarks_sequence",
    "mv_track_sequence_landmarks", "mv_track_sequence_landmarks_host", "mv_landmarks_speculate",
    "mv_landmarks_resolve", "mv_lm_spec_release", "mv_track_landmarks_prepare", "mv_track_landmarks_step_table",
    "mv_track_landmarks_solve", "mv_track_landmarks_release", "mv_track_landmarks_prepare_host",
    "mv_loop_candidates", "mv_lcd_word_weights", "mv_loop_params_default", "mv_detect_loops",
]
LEGACY_SYMBOLS = [
    "add_Vector2f", "add_Vector3f", "mult_Quaternionf", "create_Quaternionf", "Quaternionf_from_Vector3f",
    "conjugate_Quaternionf", "Vector3f_from_Quaternionf", "apply_rotation", "apply_transform", "frame_create",
    "compute_top_N", "compute_softmax", "normalize_points", "compute_essential_matrix",
    "compute_reprojection_error", "ransac_essential_matrix", "recover_pose_from_essential_matrix",
    "create_ProjectionFactor", "project2d", "cam_project", "compute_error_ProjectionFactor", "matmul", "matmul2",
    "track", "init_local_feature", "init_local_feature_with_id", "update_local_feature", "remove_old_frame",
    "init_hash_entry", "delete_hash_entry", "hash", "init_local_feature_pool", "local_feature_pool_insert",
    "chain_replacement", "local_feature_pool_delete", "local_feature_pool_rehash",
    "local_feature_pool_load_factor", "local_feature_pool_remove_old", "local_feature_pool_valid_keys",
    "local_feature_pool_check_invariant",
]


class MatchParams(C.Structure):
    _fields_ = [("rows", C.c_int), ("cols", C.c_int), ("shift_x", C.c_int), ("shift_y", C.c_int),
                ("radius", C.c_int), ("max_matches", C.c_int), ("match_threshold", C.c_double),
                ("min_prob0", C.c_double), ("use_tensor_cores", C.c_int)]


class PnpParams(C.Structure):
    _fields_ = [("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float),
                ("hypotheses", C.c_int), ("sample_size", C.c_int), ("sample_iters", C.c_int),
                ("refine_iters", C.c_int), ("gate_sq", C.c_float), ("min_depth", C.c_float),
                ("damping", C.c_float), ("seed", C.c_uint64), ("lanes_per_hypothesis", C.c_int), ("first_pair", C.c_int)]


class TrackParams(C.Structure):
    _fields_ = [("match", MatchParams), ("pnp", PnpParams), ("top_n", C.c_int), ("max_valid", C.c_int),
                ("ransac_iterations", C.c_int), ("ransac_threshold", C.c_float)]


class PairResult(C.Structure):
    _fields_ = [("q", C.c_float * 4), ("t", C.c_float * 3), ("pnp_inliers", C.c_float), ("pnp_cost", C.c_float),
                ("num_matches", C.c_int32), ("ransac_inliers", C.c_int32), ("best_hypothesis", C.c_int32),
                ("status", C.c_int32), ("pad", C.c_int32 * 3)]


class LoopParams(C.Structure):
    _fields_ = [("match", MatchParams), ("pnp", PnpParams), ("top_n", C.c_int), ("max_valid", C.c_int),
                ("min_gap", C.c_int), ("k", C.c_int), ("min_score", C.c_int), ("min_inliers", C.c_int)]


class LoopResult(C.Structure):
    _fields_ = [("frame", C.c_int32), ("bow_score", C.c_int32), ("bow_rank", C.c_int32), ("num_matches", C.c_int32),
                ("pnp_inliers", C.c_float), ("pnp_cost", C.c_float), ("q", C.c_float * 4), ("t", C.c_float * 3),
                ("status", C.c_int32), ("pad", C.c_int32 * 2)]


class SynthParams(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("rows", C.c_int), ("cols", C.c_int), ("keypoint_permille", C.c_int),
                ("noise_amp", C.c_int)]


assert C.sizeof(PairResult) == 64
assert C.sizeof(LoopResult) == 64

_lib = None


class LibraryMissing(RuntimeError):
    pass


def load() -> C.CDLL:
    """Loads the shared library; never falls back to anything else."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise LibraryMissing(
            f"{SO_PATH} is not built. Run `python maveric-slam_b200/build.py` (nvcc, sm_100a). "
            "There is no CPU fallback for the tracking hot path.")
    L = C.CDLL(SO_PATH)
    vp, i32, f32 = C.c_void_p, C.c_int, C.c_float
    L.mv_ctx_create.argtypes = [i32, C.POINTER(vp)]
    L.mv_ctx_destroy.argtypes = [vp]
    L.mv_ctx_destroy.restype = None
    L.mv_ctx_set_stream.argtypes = [vp, vp]
    L.mv_ctx_sync.argtypes = [vp]
    L.mv_last_error.argtypes = [vp]
    L.mv_last_error.restype = C.c_char_p
    L.mv_status_str.argtypes = [i32]
    L.mv_status_str.restype = C.c_char_p
    L.mv_ctx_launch_count.argtypes = [vp]
    L.mv_ctx_launch_count.restype = C.c_ulonglong
    L.mv_ctx_profile.argtypes = [vp, i32]
    L.mv_ctx_profile_read.argtypes = [vp, C.c_char_p, C.POINTER(C.c_double), C.POINTER(i32)]
    L.mv_ctx_pnp_work.argtypes = [vp, C.POINTER(C.c_ulonglong)]
    L.mv_ctx_match_work.argtypes = [vp, C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]
    L.mv_pnp_has_ab_forms.argtypes = []
    L.mv_pnp_has_ab_forms.restype = i32
    L.mv_lba_schur_batch.argtypes = [vp, i32, i32, i32, i32, vp, vp]
    L.mv_lba_solve_batch.argtypes = [vp, i32, i32, C.c_float, vp, vp, vp]
    L.mv_softmax_batch.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp]
    L.mv_top_n_batch.argtypes = [vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp]
    L.compute_softmax_ex.argtypes = [vp, f32, vp, i32, C.POINTER(i32), vp, vp]
    L.compute_top_N_ex.argtypes = [vp, f32, vp, i32, i32, i32, C.POINTER(i32), vp, vp, vp]
    L.mv_match_params_default.argtypes = [C.POINTER(MatchParams), i32, i32]
    L.mv_match_params_default.restype = None
    L.mv_match_batch.argtypes = [vp, C.POINTER(MatchParams), i32, i32, i32] + [vp] * 13
    L.mv_match_pair_host.argtypes = [vp, C.POINTER(MatchParams), vp, vp, vp, vp, i32, vp, vp, vp, vp,
                                     C.POINTER(i32), vp, vp]
    L.mv_ransac_identity_batch.argtypes = [vp, i32, i32, vp, vp, i32, f32, vp, vp, vp]
    L.mv_pnp_params_default.argtypes = [C.POINTER(PnpParams)]
    L.mv_pnp_params_default.restype = None
    L.mv_pnp_gn_batch.argtypes = [vp, C.POINTER(PnpParams), i32, i32, vp, vp, vp, vp, vp, vp]
    L.mv_build_corr_batch.argtypes = [vp, i32, i32, i32, i32, vp, vp, f32, f32, f32, f32, vp, vp, vp, vp]
    L.mv_track_params_default.argtypes = [C.POINTER(TrackParams), i32, i32]
    L.mv_track_params_default.restype = None
    L.mv_track_sequence.argtypes = [vp, C.POINTER(TrackParams), i32, vp, vp, vp, vp, vp]
    L.mv_track_sequence_host.argtypes = [vp, C.POINTER(TrackParams), i32, vp, vp, vp, vp, vp,
                                         C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]
    L.mv_bow_set_vocabulary.argtypes = [vp, i32, i32, vp, vp, vp, vp]
    L.mv_bow_assign_batch.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp, vp, vp]
    L.mv_landmarks_init.argtypes = [vp, i32, vp]
    L.mv_landmarks_observe.argtypes = [vp, i32, vp, i32, i32, vp, vp]
    L.mv_landmarks_remove_old.argtypes = [vp, i32, vp, i32]
    L.mv_landmarks_lookup.argtypes = [vp, i32, vp, i32, vp, vp, vp]
    L.mv_build_corr_landmarks_batch.argtypes = [vp, i32, i32, i32, i32] + [vp] * 10
    L.mv_landmarks_sequence.argtypes = [vp, i32, vp, i32, i32, i32, vp, vp, vp, vp]
    L.mv_track_sequence_landmarks.argtypes = [vp, C.POINTER(TrackParams), i32, i32, vp, vp, vp, vp, vp, i32, vp, vp, vp]
    L.mv_track_sequence_landmarks_host.argtypes = [vp, C.POINTER(TrackParams), i32, i32, vp, vp, vp, vp, vp, i32, vp, vp,
                                                   vp, C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]
    L.mv_landmarks_speculate.argtypes = [vp, i32, i32, i32, i32, i32, vp, vp, vp, C.POINTER(vp)]
    L.mv_landmarks_resolve.argtypes = [vp, vp, vp, vp, vp]
    L.mv_lm_spec_release.argtypes = [vp]
    L.mv_lm_spec_release.restype = None
    L.mv_track_landmarks_prepare.argtypes = [vp, C.POINTER(TrackParams), i32, i32, i32, vp, vp, vp, vp, vp, i32,
                                             C.POINTER(vp)]
    L.mv_track_landmarks_prepare_host.argtypes = [vp, C.POINTER(TrackParams), i32, i32, i32, vp, vp, vp, vp, vp, i32,
                                                  C.POINTER(vp), C.POINTER(C.c_ulonglong)]
    L.mv_track_landmarks_step_table.argtypes = [vp, vp, vp, vp]
    L.mv_track_landmarks_solve.argtypes = [vp, vp, vp, vp]
    L.mv_track_landmarks_release.argtypes = [vp]
    L.mv_track_landmarks_release.restype = None
    L.mv_loop_candidates.argtypes = [vp, i32, i32, i32, i32, vp, vp, vp, i32, i32, i32, vp, vp]
    L.mv_lcd_word_weights.argtypes = [vp, i32, i32, i32, vp, vp, vp]
    L.mv_loop_params_default.argtypes = [C.POINTER(LoopParams), i32, i32]
    L.mv_loop_params_default.restype = None
    L.mv_detect_loops.argtypes = [vp, C.POINTER(LoopParams), i32, i32, vp, vp, vp, vp, vp, vp, vp]
    L.mv_synth_frames.argtypes = [vp, C.POINTER(SynthParams), i32, i32, vp, vp, vp, vp]
    L.mv_nms_batch.argtypes = [vp, i32, i32, i32, vp, vp]
    L.run_nms_ex.argtypes = [vp, i32, i32, vp, vp]
    L.mv_chain_transforms.argtypes = [vp, i32, vp, vp]
    L.mv_results_to_transforms.argtypes = [vp, i32, vp, vp]
    # legacy symbols used from Python
    L.compute_softmax.argtypes = [f32, vp, C.POINTER(i32), vp, vp]
    L.compute_softmax.restype = None
    L.compute_top_N.argtypes = [f32, vp, i32, C.POINTER(i32), vp, vp, vp]
    L.compute_top_N.restype = None
    L.ransac_essential_matrix.argtypes = [i32, vp, vp, vp, i32, f32, vp, vp, C.POINTER(i32)]
    L.ransac_essential_matrix.restype = None
    L.recover_pose_from_essential_matrix.argtypes = [vp, vp, vp, vp]
    L.recover_pose_from_essential_matrix.restype = None
    L.compute_reprojection_error.argtypes = [vp, vp, vp]
    L.compute_reprojection_error.restype = f32
    L.normalize_points.argtypes = [i32, vp, vp, vp]
    L.normalize_points.restype = None
    L.compute_essential_matrix.argtypes = [i32, vp, vp, vp]
    L.compute_essential_matrix.restype = None
    L.matmul.argtypes = [C.c_size_t] * 3 + [vp] * 3 + [C.c_size_t] * 3 + [f32] * 2 + [C.c_bool] * 2
    L.matmul.restype = None
    L.matmul2.argtypes = [C.c_size_t] * 3 + [vp] * 4 + [C.c_size_t] * 4 + [f32] * 3 + [C.c_bool] * 2
    L.matmul2.restype = None
    _lib = L
    return L


class MvError(RuntimeError):
    pass


class Context:
    """Owns one mv_ctx (one GPU, one compute stream)."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self.lib = load()
        h = C.c_void_p()
        st = self.lib.mv_ctx_create(device, C.byref(h))
        if st != MV_OK:
            raise MvError(f"mv_ctx_create(device={device}): {self.lib.mv_status_str(st).decode()}")
        self.h = h
        if stream is not None:
            self.check(self.lib.mv_ctx_set_stream(self.h, C.c_void_p(stream)))

    def check(self, st: int) -> None:
        if st != MV_OK:
            raise MvError(f"{self.lib.mv_status_str(st).decode()}: {self.lib.mv_last_error(self.h).decode()}")

    def sync(self) -> None:
        self.check(self.lib.mv_ctx_sync(self.h))

    @property
    def launches(self) -> int:
        return int(self.lib.mv_ctx_launch_count(self.h))

    def profile(self, on: bool) -> None:
        self.check(self.lib.mv_ctx_profile(self.h, 1 if on else 0))

    def profile_read(self, tag: str):
        ms = C.c_double(0)
        n = C.c_int(0)
        self.check(self.lib.mv_ctx_profile_read(self.h, tag.encode(), C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def pnp_work(self) -> int:
        """accepted correspondence-passes of the profiled PnP launches since the last read"""
        v = C.c_ulonglong(0)
        self.check(self.lib.mv_ctx_pnp_work(self.h, C.byref(v)))
        return int(v.value)

    def match_work(self):
        """(tiles, chunks) the tensor-core matcher executed in its last launch on this context"""
        t, c = C.c_ulonglong(0), C.c_ulonglong(0)
        self.check(self.lib.mv_ctx_match_work(self.h, C.byref(t), C.byref(c)))
        return int(t.value), int(c.value)

    def close(self) -> None:
        if getattr(self, "h", None):
            self.lib.mv_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
