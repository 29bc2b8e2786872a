"""ctypes binding of libmmw.so (include/mmw.h).  Fails loudly when the library is missing
or a call fails -- there is no CPU fallback behind this module."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MMW_LIB", os.path.join(_HERE, "libmmw.so"))   # MMW_LIB: alternative build (profiling experiments)

MMW_POSE_2D, MMW_POSE_3D = 0, 1
STEP_POSE, STEP_DEVICE_INPUT, STEP_RECORD_LABELS, STEP_PIPELINE, STEP_INPUT_I16 = 0x1, 0x2, 0x4, 0x8, 0x10
SCENE_POINT_OVERFLOW, SCENE_TRACK_OVERFLOW = 0x1, 0x2
RESULT_FLOATS = 72
ABI_VERSION = 7            # MMW_ABI_VERSION of include/mmw.h this binding was written against
KERNEL_NAMES = ["step", "pose_index", "pose_features", "conv", "fc1", "fc2", "dbscan_big", "packets"]


class MmwError(RuntimeError):
    pass


class Config(C.Structure):
    """mmw_config: mirror of the reference's constants.py (see include/mmw.h)."""
    _fields_ = [
        ("s_height", C.c_double), ("s_tilt_deg", C.c_double), ("z_max", C.c_double),
        ("frames_batch", C.c_int32), ("db_min_samples", C.c_int32),
        ("db_z_weight", C.c_double), ("db_range_weight", C.c_double), ("db_eps", C.c_double),
        ("tr_max_tracks", C.c_int32), ("kf_enable_est", C.c_int32),
        ("tr_lifetime_dynamic", C.c_double), ("tr_lifetime_static", C.c_double),
        ("tr_vel_thres", C.c_double), ("tr_gate", C.c_double),
        ("kf_q_var", C.c_double), ("kf_p_init", C.c_double), ("kf_group_disp_init", C.c_double),
        ("kf_a_n", C.c_double), ("kf_a_spr", C.c_double), ("kf_spread_lim", C.c_double * 6),
        ("kf_est_pointnum", C.c_int32), ("xyz_q_format", C.c_int32),
        ("intensity_mu", C.c_double), ("intensity_std", C.c_double),
        ("x_nudge_thres", C.c_double), ("x_nudge_gain", C.c_double),
        ("default_posture", C.c_float * 57), ("reserved1", C.c_float),
        ("m_x", C.c_double), ("m_y", C.c_double), ("m_z", C.c_double),
        ("fade_size_max", C.c_double), ("fade_size_min", C.c_double), ("fade_weight", C.c_double),
        ("doppler_res", C.c_double),
    ]


class SceneSensor(C.Structure):
    """mmw_scene_sensor: one scene's sensor mounting and radar profile (see include/mmw.h)."""
    _fields_ = [
        ("s_height", C.c_double), ("s_tilt_deg", C.c_double), ("z_max", C.c_double), ("doppler_res", C.c_double),
        ("xyz_q_format", C.c_int32), ("num_doppler_bins", C.c_int32),
    ]


SCENE_SENSOR_DTYPE = np.dtype([
    ("s_height", "<f8"), ("s_tilt_deg", "<f8"), ("z_max", "<f8"), ("doppler_res", "<f8"),
    ("xyz_q_format", "<i4"), ("num_doppler_bins", "<i4"),
], align=False)
assert SCENE_SENSOR_DTYPE.itemsize == C.sizeof(SceneSensor), (SCENE_SENSOR_DTYPE.itemsize, C.sizeof(SceneSensor))


class SceneTracker(C.Structure):
    """mmw_scene_tracker: one scene's tracker and DBSCAN constants (see include/mmw.h)."""
    _fields_ = [
        ("db_eps", C.c_double), ("db_z_weight", C.c_double), ("db_range_weight", C.c_double),
        ("tr_lifetime_dynamic", C.c_double), ("tr_lifetime_static", C.c_double), ("tr_vel_thres", C.c_double),
        ("tr_gate", C.c_double), ("kf_q_var", C.c_double), ("kf_p_init", C.c_double),
        ("kf_group_disp_init", C.c_double), ("kf_a_n", C.c_double), ("kf_a_spr", C.c_double),
        ("kf_spread_lim", C.c_double * 6), ("x_nudge_thres", C.c_double), ("x_nudge_gain", C.c_double),
        ("db_min_samples", C.c_int32), ("tr_max_tracks", C.c_int32), ("kf_enable_est", C.c_int32),
        ("kf_est_pointnum", C.c_int32),
    ]


SCENE_TRACKER_DTYPE = np.dtype([
    ("db_eps", "<f8"), ("db_z_weight", "<f8"), ("db_range_weight", "<f8"),
    ("tr_lifetime_dynamic", "<f8"), ("tr_lifetime_static", "<f8"), ("tr_vel_thres", "<f8"),
    ("tr_gate", "<f8"), ("kf_q_var", "<f8"), ("kf_p_init", "<f8"),
    ("kf_group_disp_init", "<f8"), ("kf_a_n", "<f8"), ("kf_a_spr", "<f8"),
    ("kf_spread_lim", "<f8", (6,)), ("x_nudge_thres", "<f8"), ("x_nudge_gain", "<f8"),
    ("db_min_samples", "<i4"), ("tr_max_tracks", "<i4"), ("kf_enable_est", "<i4"), ("kf_est_pointnum", "<i4"),
], align=False)
assert SCENE_TRACKER_DTYPE.itemsize == C.sizeof(SceneTracker), (SCENE_TRACKER_DTYPE.itemsize, C.sizeof(SceneTracker))


SCENE_BLOB_MAGIC = 0x4D4D574D    # MMW_SCENE_BLOB_MAGIC


class SceneBlobHeader(C.Structure):
    """mmw_scene_blob_header: the 64 bytes that open a scene blob (mmw_export_scenes)."""
    _fields_ = [
        ("magic", C.c_uint32), ("abi_version", C.c_uint32), ("n", C.c_int32), ("max_points_per_frame", C.c_int32),
        ("max_tracks", C.c_int32), ("frames_batch", C.c_int32), ("record_bytes", C.c_uint64),
        ("total_bytes", C.c_uint64), ("reserved", C.c_uint32 * 6),
    ]


assert C.sizeof(SceneBlobHeader) == 64


class TrackOut(C.Structure):
    """mmw_track_out"""
    _fields_ = [
        ("id", C.c_int32), ("point_num", C.c_int32), ("is_static", C.c_int32), ("ring_frames", C.c_int32),
        ("ring_counts", C.c_int32 * 3), ("reserved", C.c_int32),
        ("lifetime", C.c_double), ("n_est", C.c_double),
        ("x", C.c_double * 9), ("P", C.c_double * 81), ("spread_est", C.c_double * 6),
        ("group_disp_est", C.c_double * 36), ("centroid", C.c_double * 6),
        ("min_vals", C.c_double * 6), ("max_vals", C.c_double * 6),
        ("keypoints", C.c_float * 57), ("reserved2", C.c_float),
    ]


TRACK_DTYPE = np.dtype([
    ("id", "<i4"), ("point_num", "<i4"), ("is_static", "<i4"), ("ring_frames", "<i4"),
    ("ring_counts", "<i4", (3,)), ("reserved", "<i4"),
    ("lifetime", "<f8"), ("n_est", "<f8"), ("x", "<f8", (9,)), ("P", "<f8", (9, 9)),
    ("spread_est", "<f8", (6,)), ("group_disp_est", "<f8", (6, 6)), ("centroid", "<f8", (6,)),
    ("min_vals", "<f8", (6,)), ("max_vals", "<f8", (6,)), ("keypoints", "<f4", (57,)), ("reserved2", "<f4"),
], align=False)
assert TRACK_DTYPE.itemsize == C.sizeof(TrackOut), (TRACK_DTYPE.itemsize, C.sizeof(TrackOut))

# name -> (restype, argtypes).  Every symbol include/mmw.h declares is listed here (tests check the list
# against the header and against the built library).
_p = C.c_void_p
SIGNATURES = {
    "mmw_abi_version": (C.c_int, []),
    "mmw_last_error": (C.c_char_p, []),
    "mmw_default_config": (C.c_int, [C.POINTER(Config)]),
    "mmw_create": (C.c_int, [C.POINTER(Config), C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_p)]),
    "mmw_destroy": (C.c_int, [_p]),
    "mmw_reset": (C.c_int, [_p]),
    "mmw_set_doppler_resolution": (C.c_int, [_p, C.c_double]),
    "mmw_set_scene_sensors": (C.c_int, [_p, C.c_int, C.c_int, _p]),
    "mmw_get_scene_sensors": (C.c_int, [_p, C.c_int, C.c_int, _p]),
    "mmw_set_scene_trackers": (C.c_int, [_p, C.c_int, C.c_int, _p]),
    "mmw_get_scene_trackers": (C.c_int, [_p, C.c_int, C.c_int, _p]),
    "mmw_reset_scenes": (C.c_int, [_p, _p, C.c_int]),
    "mmw_state_size": (C.c_size_t, [_p]),
    "mmw_state_dump": (C.c_int, [_p, _p, C.c_size_t]),
    "mmw_state_restore": (C.c_int, [_p, _p, C.c_size_t]),
    "mmw_scene_state_size": (C.c_size_t, [_p, C.c_int]),
    "mmw_export_scenes": (C.c_int, [_p, _p, C.c_int, _p, C.c_size_t]),
    "mmw_import_scenes": (C.c_int, [_p, _p, C.c_int, _p, C.c_size_t]),
    "mmw_load_pose_weights": (C.c_int, [_p, C.c_int, _p, C.c_size_t]),
    "mmw_step": (C.c_int, [_p, _p, _p, _p, C.c_uint32]),
    "mmw_estimate_posture": (C.c_int, [_p]),
    "mmw_pose_features_only": (C.c_int, [_p]),
    "mmw_set_keypoints": (C.c_int, [_p, C.c_int, C.c_int, _p]),
    "mmw_sync": (C.c_int, [_p]),
    "mmw_stream": (_p, [_p]),
    "mmw_get_tracks": (C.c_int, [_p, _p, _p]),
    "mmw_get_scene_summary": (C.c_int, [_p, _p, _p, _p]),
    "mmw_get_point_assoc": (C.c_int, [_p, _p, C.c_size_t]),
    "mmw_get_labels": (C.c_int, [_p, _p, _p]),
    "mmw_get_status": (C.c_int, [_p, _p]),
    "mmw_get_ring_counts": (C.c_int, [_p, _p]),
    "mmw_ring_pop": (C.c_int, [_p, C.c_int]),
    "mmw_ring_clear": (C.c_int, [_p, C.c_int]),
    "mmw_get_pose_rows": (C.c_int, [_p, _p, _p, _p, _p, C.c_size_t]),
    "mmw_preprocess": (C.c_int, [_p, _p, C.c_size_t, _p, _p]),
    "mmw_dbscan": (C.c_int, [_p, _p, _p, C.c_int, C.c_double, C.c_int, _p]),
    "mmw_kalman_predict": (C.c_int, [_p, _p, _p, _p, C.c_int]),
    "mmw_kalman_update": (C.c_int, [_p, _p, _p, _p, _p, _p, C.c_int]),
    "mmw_gate": (C.c_int, [_p, _p, C.c_int, _p, _p, C.c_int, _p, _p]),
    "mmw_pose": (C.c_int, [_p, _p, C.c_int, _p]),
    "mmw_decode_tlv": (C.c_int, [_p, _p, _p, C.c_int, C.c_double, C.c_double, _p, C.c_size_t, _p, _p, _p]),
    "mmw_step_packets": (C.c_int, [_p, _p, _p, _p, C.c_uint32, _p, _p]),
    "mmw_export_track0": (C.c_int, [_p, _p, _p, _p]),
    "mmw_pack_results": (C.c_int, [_p, _p]),
    "mmw_gather_nccl": (C.c_int, [_p, _p, C.c_int, _p]),
    "mmw_nccl_unique_id": (C.c_int, [_p]),
    "mmw_nccl_comm_init": (C.c_int, [_p, _p, C.c_int, C.c_int, C.POINTER(_p)]),
    "mmw_nccl_comm_destroy": (C.c_int, [_p]),
    "mmw_read_results_async": (C.c_int, [_p, _p, C.POINTER(C.c_int)]),
    "mmw_wait_results": (C.c_int, [_p, C.c_int]),
    "mmw_run_frames": (C.c_int, [_p, C.c_int, _p, _p, _p, _p, _p, C.c_uint32]),
    "mmw_run_frames_compact": (C.c_int, [_p, C.c_int, _p, _p, _p, _p, _p, _p, C.c_uint32]),
    "mmw_get_counters": (C.c_int, [_p, _p, C.c_int]),
    "mmw_set_dense_path": (C.c_int, [_p, C.c_int]),
    "mmw_pose_intermediate": (C.c_int, [_p, C.c_int, C.POINTER(C.c_int), _p, C.c_size_t]),
    "mmw_profile": (C.c_int, [_p, C.c_int]),
    "mmw_get_kernel_ms": (C.c_int, [_p, _p, _p]),
    "mmw_phase_clocks": (C.c_int, [_p, C.c_int, _p]),
    "mmw_scene_cycles": (C.c_int, [_p, _p]),
    "mmw_dbscan_big_clocks": (C.c_int, [_p, _p]),
    "mmw_launch_count": (C.c_uint64, [_p]),
}

_lib = None


def load() -> C.CDLL:
    """Loads libmmw.so (built in-tree by __graft_entry__.build() / csrc/Makefile)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise MmwError("libmmw.so not found at %s -- build it with `python -c 'import __graft_entry__ as g; "
                       "g.build()'` (or make -C mmwave_msc_b200/csrc); there is no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.mmw_abi_version() != ABI_VERSION:   # a stale libmmw.so would mis-read the config struct: fail loudly
        raise MmwError("libmmw.so at %s has ABI version %d, this binding needs %d -- rebuild it"
                       % (LIB_PATH, lib.mmw_abi_version(), ABI_VERSION))
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().mmw_last_error()
        raise MmwError("libmmw error %d: %s" % (rc, msg.decode() if msg else "?"))


def ptr(a) -> C.c_void_p:
    """Pointer of a C-contiguous numpy array / int device address / None."""
    if a is None:
        return C.c_void_p(0)
    if isinstance(a, int):
        return C.c_void_p(a)
    if not a.flags["C_CONTIGUOUS"]:
        raise ValueError("array must be C-contiguous")
    return C.c_void_p(a.ctypes.data)
