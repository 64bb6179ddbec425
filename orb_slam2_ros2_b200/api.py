"""Python host-side mirror of the reference interface, bound to liborbx.so through ctypes.

The names follow the reference (include/ORB_SLAM2/ORBExtractor.h:99-161, include/ORB_SLAM2/Frame.h:303-371,
include/ORB_SLAM2/ORBMatcher.h:39): ``ORBExtractor(image, nFeatures, pyramidLevels, scaleFactor, bfTemFp, maxThreshold,
minThreshold).extract()``, ``Frame.createStereo(...)``, ``Frame.createRGBD(...)``.  All compute happens in the CUDA
library; there is no CPU fallback -- loading fails loudly when liborbx.so or a CUDA device is missing.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "liborbx.so")

KP_DTYPE = np.dtype(
    [("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"), ("octave", "<i4"), ("class_id", "<i4")]
)
AREA_QUERY_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("radius", "<f4"), ("octave", "<i4"), ("min_level", "<i4"), ("max_level", "<i4")])

ORBX_OK = 0
ORBX_ERR_INVALID_ARG = -1
ORBX_ERR_IMAGE_SIZE = -2
ORBX_ERR_FILE_NOT_OPEN = -3
ORBX_ERR_CUDA = -4
ORBX_ERR_NO_DEVICE = -5
ORBX_ERR_CAPACITY = -6
ORBX_ERR_STATE = -7
ORBX_ERR_COMM = -8
COMM_ID_BYTES, IPC_HANDLE_BYTES = 128, 64
TRANSPORT_NONE, TRANSPORT_NCCL, TRANSPORT_PEER = 0, 1, 2
DEPTH_U16, DEPTH_F32 = 0, 1
N_STAGES = 7  # ORBX_N_STAGES


# the reference's exception types (include/ORB_SLAM2/Error.h:13-98)
class ORBSlam2Error(RuntimeError):
    pass


class ImageSizeError(ORBSlam2Error):
    pass


class FileNotOpenError(ORBSlam2Error):
    pass


class OrbxCudaError(ORBSlam2Error):
    pass


class OrbxConfig(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("n_features", C.c_int32), ("n_levels", C.c_int32), ("scale_factor", C.c_float),
        ("ini_th_fast", C.c_int32), ("min_th_fast", C.c_int32), ("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float),
        ("bf", C.c_float), ("dist", C.c_float * 5), ("depth_scale", C.c_float), ("max_batch", C.c_int32), ("device", C.c_int32),
        ("pattern", C.POINTER(C.c_float)),
    ]


class OrbxDeviceResults(C.Structure):
    _fields_ = [
        ("kps", C.c_void_p), ("kps_und", C.c_void_p), ("desc", C.c_void_p), ("n_kps", C.c_void_p), ("u_right", C.c_void_p), ("depth", C.c_void_p),
        ("n_matches", C.c_void_p), ("n_images", C.c_int32), ("n_frames", C.c_int32), ("n_features", C.c_int32),
        ("grid_start", C.c_void_p), ("grid_entries", C.c_void_p), ("grid_rows", C.c_int32), ("grid_cols", C.c_int32),
    ]


EXPORTS = [
    "orbx_default_config", "orbx_create", "orbx_destroy", "orbx_status_string", "orbx_last_error", "orbx_load_brief_template", "orbx_set_stream",
    "orbx_num_levels", "orbx_level_info", "orbx_extract", "orbx_get_pyramid", "orbx_stereo_frame", "orbx_rgbd_frame", "orbx_stereo_batch",
    "orbx_stereo_batch_device", "orbx_extract_batch_device", "orbx_rgbd_batch_device", "orbx_synchronize", "orbx_launch_count", "orbx_algorithmic_bytes",
    "orbx_debug_level_corners", "orbx_debug_level_selected", "orbx_read_device", "orbx_profile_stereo_batch_device", "orbx_stage_name", "orbx_debug_run_quadtree", "orbx_grid_info", "orbx_get_grid",
    "orbx_search_in_area", "orbx_search_in_area_batch_device", "orbx_verify_angle",
    "orbx_serialized_capacity", "orbx_serialize_keyframe", "orbx_serialize_keyframe_text", "orbx_serialize_keyframes_device",
    "orbx_vocab_create", "orbx_vocab_load_text", "orbx_vocab_destroy", "orbx_vocab_info", "orbx_bow_transform", "orbx_bow_transform_batch_device",
    "orbx_search_by_bow",
    "orbx_frame_epoch", "orbx_set_graph", "orbx_debug_quadtree_stats", "orbx_frame_range", "orbx_comm_unique_id", "orbx_comm_create", "orbx_comm_ipc_handle", "orbx_comm_open_peers",
    "orbx_comm_create_local", "orbx_comm_destroy", "orbx_comm_info", "orbx_record_layout_get", "orbx_sequence_stereo",
    "orbx_serialized_capacity_bow", "orbx_serialize_keyframe_bow", "orbx_serialize_keyframes_bow_device", "orbx_keyframe_list_head",
    "orbx_keyframe_list_entry_prefix", "orbx_sequence_stereo_keyframes", "orbx_vocab_build", "orbx_vocab_save_text", "orbx_vocab_arrays",
    "orbx_bowdb_build", "orbx_bowdb_destroy", "orbx_bowdb_info", "orbx_bowdb_query_range", "orbx_bowdb_query_frame",
    "orbx_loopver_build", "orbx_loopver_destroy", "orbx_loopver_verify",
]

class OrbxRecordLayout(C.Structure):
    _fields_ = [("record_bytes", C.c_int64), ("off_kps_left", C.c_int64), ("off_desc_left", C.c_int64), ("off_kps_right", C.c_int64),
                ("off_desc_right", C.c_int64), ("off_u_right", C.c_int64), ("off_depth", C.c_int64), ("n_features", C.c_int32), ("reserved", C.c_int32)]


class OrbxSequenceIO(C.Structure):
    _fields_ = [("left", C.c_void_p), ("right", C.c_void_p), ("stride", C.c_size_t), ("frame_stride", C.c_size_t), ("input_on_device", C.c_int32),
                ("records_on_device", C.c_int32), ("records", C.c_void_p), ("record_stride", C.c_size_t), ("gathered_desc_host", C.c_void_p),
                ("gathered_n_host", C.c_void_p)]


class OrbxSequenceResult(C.Structure):
    _fields_ = [("frame_lo", C.c_int64), ("frame_hi", C.c_int64), ("block", C.c_int64), ("gathered_desc", C.c_void_p), ("gathered_n", C.c_void_p),
                ("n_features", C.c_int32), ("world", C.c_int32)]


class OrbxKeyframeIO(C.Structure):
    _fields_ = [("vocab", C.c_void_p), ("levelsup", C.c_int32), ("with_map_points", C.c_int32), ("id0", C.c_uint64), ("pose_rt", C.c_void_p),
                ("on_device", C.c_int32), ("out", C.c_void_p), ("stride", C.c_size_t), ("sizes", C.c_void_p)]


VOCAB_MAX_ITERS, VOCAB_MAX_K = 100, 32  # ORBX_VOCAB_MAX_ITERS / ORBX_VOCAB_MAX_K
BOW_MAX_STRIDE = 16384  # ORBX_BOW_MAX_STRIDE: most descriptors per frame of the bag-of-words entry points


class OrbxVocabTrain(C.Structure):
    _fields_ = [("desc", C.c_void_p), ("n_kps", C.c_void_p), ("n_frames", C.c_int32), ("stride", C.c_int32), ("on_device", C.c_int32), ("k", C.c_int32),
                ("L", C.c_int32), ("seed", C.c_uint64), ("iters", C.c_void_p), ("n_capped", C.c_void_p), ("level_ms", C.c_void_p)]


class OrbxDeviceBow(C.Structure):
    _fields_ = [("bow_ids", C.c_void_p), ("bow_vals", C.c_void_p), ("n_bow", C.c_void_p), ("fv_nodes", C.c_void_p), ("fv_start", C.c_void_p),
                ("fv_feats", C.c_void_p), ("n_fv_nodes", C.c_void_p), ("stride", C.c_int32)]


BOWDB_MAX_FRAMES = 98304  # ORBX_BOWDB_MAX_FRAMES


class OrbxBowdbIO(C.Structure):
    _fields_ = [("exclude_window", C.c_int32), ("min_score", C.c_float), ("top_k", C.c_int32), ("on_device", C.c_int32), ("cand_frame", C.c_void_p),
                ("cand_score", C.c_void_p), ("cand_common", C.c_void_p), ("n_sharing", C.c_void_p), ("max_common", C.c_void_p), ("n_scored", C.c_void_p),
                ("n_kept", C.c_void_p)]


LOOPVER_JACOBI_SWEEPS = 16  # ORBX_LOOPVER_JACOBI_SWEEPS


class OrbxLoopverParams(C.Structure):
    _fields_ = [("ratio", C.c_float), ("min_matches", C.c_int32), ("min_inliers", C.c_int32), ("max_iterations", C.c_int32), ("probability", C.c_double),
                ("seed", C.c_uint64)]


class OrbxLoopverIO(C.Structure):
    _fields_ = [("on_device", C.c_int32), ("cand_frame", C.c_void_p), ("top_k", C.c_int32), ("n_bow", C.c_void_p), ("n_matches", C.c_void_p),
                ("n_corr", C.c_void_p), ("n_iters", C.c_void_p), ("hypothesis", C.c_void_p), ("n_inliers", C.c_void_p), ("accepted", C.c_void_p),
                ("T", C.c_void_p), ("match", C.c_void_p), ("loop_frame", C.c_void_p)]


_lib = None


def load_library(build_if_missing: bool = True):
    """dlopen liborbx.so (building it with nvcc first when absent).  Raises if it cannot be loaded."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        if not build_if_missing:
            raise OSError(f"{LIB_PATH} is missing: run `python -m orb_slam2_ros2_b200.build`")
        from . import build as _b

        _b.build()
    L = C.CDLL(LIB_PATH)
    vp, u8p, i32p, f64p, sz = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t
    L.orbx_default_config.argtypes = [C.POINTER(OrbxConfig)]
    L.orbx_default_config.restype = None
    L.orbx_create.argtypes = [C.POINTER(OrbxConfig), C.POINTER(vp)]
    L.orbx_destroy.argtypes = [vp]
    L.orbx_destroy.restype = None
    L.orbx_status_string.argtypes = [C.c_int]
    L.orbx_status_string.restype = C.c_char_p
    L.orbx_last_error.argtypes = [vp]
    L.orbx_last_error.restype = C.c_char_p
    L.orbx_load_brief_template.argtypes = [C.c_char_p, C.POINTER(C.c_float)]
    L.orbx_set_stream.argtypes = [vp, vp]
    L.orbx_num_levels.argtypes = [vp]
    L.orbx_level_info.argtypes = [vp, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_float), C.POINTER(C.c_int32)]
    L.orbx_extract.argtypes = [vp, u8p, sz, vp, u8p, i32p]
    L.orbx_get_pyramid.argtypes = [vp, C.c_int, C.c_int, C.c_int, u8p, sz]
    L.orbx_stereo_frame.argtypes = [vp, u8p, sz, u8p, sz, vp, u8p, i32p, vp, u8p, i32p, f64p, f64p, i32p]
    L.orbx_rgbd_frame.argtypes = [vp, u8p, sz, vp, sz, C.c_int, vp, vp, u8p, i32p, f64p, f64p]
    L.orbx_stereo_batch.argtypes = [vp, C.c_int, u8p, u8p, sz, sz, vp, u8p, i32p, vp, u8p, i32p, f64p, f64p, i32p]
    L.orbx_stereo_batch_device.argtypes = [vp, C.c_int, vp, vp, sz, sz, C.POINTER(OrbxDeviceResults)]
    L.orbx_extract_batch_device.argtypes = [vp, C.c_int, vp, sz, sz, C.POINTER(OrbxDeviceResults)]
    L.orbx_rgbd_batch_device.argtypes = [vp, C.c_int, vp, sz, sz, vp, sz, sz, C.c_int, C.POINTER(OrbxDeviceResults)]
    L.orbx_synchronize.argtypes = [vp]
    L.orbx_read_device.argtypes = [vp, vp, vp, sz]
    L.orbx_profile_stereo_batch_device.argtypes = [vp, C.c_int, vp, vp, sz, sz, C.POINTER(C.c_float)]
    L.orbx_stage_name.argtypes = [C.c_int]
    L.orbx_stage_name.restype = C.c_char_p
    L.orbx_launch_count.argtypes = [vp]
    L.orbx_launch_count.restype = C.c_int64
    L.orbx_algorithmic_bytes.argtypes = [vp, C.c_int]
    L.orbx_algorithmic_bytes.restype = C.c_int64
    L.orbx_debug_level_corners.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, C.c_int, vp]
    L.orbx_debug_level_selected.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, C.c_int, vp]
    L.orbx_debug_run_quadtree.argtypes = [vp, C.c_int, vp, vp, vp, C.c_int]
    L.orbx_grid_info.argtypes = [vp, C.POINTER(C.c_int32), C.POINTER(C.c_int32)] + [C.POINTER(C.c_float)] * 4
    L.orbx_get_grid.argtypes = [vp, C.c_int, vp, vp]
    L.orbx_search_in_area.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp]
    L.orbx_search_in_area_batch_device.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp]
    L.orbx_verify_angle.argtypes = [vp, C.c_int, vp, vp, vp, vp, C.c_int, vp, C.c_int, C.POINTER(C.c_int32)]
    L.orbx_serialized_capacity.argtypes = [vp]
    L.orbx_serialized_capacity.restype = C.c_int64
    L.orbx_serialize_keyframe.argtypes = [vp, C.c_int, C.c_uint64, vp, C.c_int, vp, sz, C.POINTER(C.c_int64)]
    L.orbx_serialize_keyframes_device.argtypes = [vp, C.c_int, C.c_uint64, vp, C.c_int, vp, sz, vp]
    L.orbx_serialize_keyframe_text.argtypes = [vp, C.c_int, C.c_uint64, vp, C.c_int, C.c_int, C.c_uint64, vp, sz, C.POINTER(C.c_int64)]
    L.orbx_vocab_create.argtypes = [vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, C.POINTER(vp)]
    L.orbx_vocab_load_text.argtypes = [vp, C.c_char_p, C.POINTER(vp)]
    L.orbx_vocab_destroy.argtypes = [vp]
    L.orbx_vocab_destroy.restype = None
    L.orbx_vocab_info.argtypes = [vp] + [C.POINTER(C.c_int32)] * 4
    L.orbx_bow_transform.argtypes = [vp, vp, C.c_int, C.c_int, vp, vp, C.POINTER(C.c_int32), vp, vp, vp, C.POINTER(C.c_int32)]
    L.orbx_bow_transform_batch_device.argtypes = [vp, vp, C.c_int, C.c_int, C.POINTER(OrbxDeviceBow)]
    L.orbx_search_by_bow.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, vp, C.c_int, vp, vp, vp, vp, vp, vp]
    L.orbx_frame_epoch.argtypes = [vp]
    L.orbx_debug_quadtree_stats.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.orbx_set_graph.argtypes = [vp, C.c_int]
    L.orbx_frame_epoch.restype = C.c_uint64
    L.orbx_frame_range.argtypes = [C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.orbx_frame_range.restype = None
    L.orbx_comm_unique_id.argtypes = [vp]
    L.orbx_comm_create.argtypes = [vp, C.c_int, C.c_int, vp, C.c_int64, C.POINTER(vp)]
    L.orbx_comm_ipc_handle.argtypes = [vp, vp]
    L.orbx_comm_open_peers.argtypes = [vp, vp]
    L.orbx_comm_create_local.argtypes = [C.POINTER(vp), C.c_int, C.c_int64, C.POINTER(vp)]
    L.orbx_comm_destroy.argtypes = [vp]
    L.orbx_comm_destroy.restype = None
    L.orbx_comm_info.argtypes = [vp] + [C.POINTER(C.c_int32)] * 3
    L.orbx_record_layout_get.argtypes = [vp, C.POINTER(OrbxRecordLayout)]
    L.orbx_sequence_stereo.argtypes = [vp, vp, C.c_int64, C.POINTER(OrbxSequenceIO), C.POINTER(OrbxSequenceResult)]
    L.orbx_serialized_capacity_bow.argtypes = [vp]
    L.orbx_serialized_capacity_bow.restype = C.c_int64
    L.orbx_serialize_keyframe_bow.argtypes = [vp, C.c_int, C.c_uint64, vp, C.c_int, vp, sz, C.POINTER(C.c_int64)]
    L.orbx_serialize_keyframes_bow_device.argtypes = [vp, C.c_int, C.c_uint64, vp, C.c_int, vp, sz, vp]
    L.orbx_keyframe_list_head.argtypes = [vp, C.c_uint64, vp, sz, C.POINTER(C.c_int64)]
    L.orbx_keyframe_list_entry_prefix.argtypes = [C.c_int64, vp]
    L.orbx_sequence_stereo_keyframes.argtypes = [vp, vp, C.c_int64, C.POINTER(OrbxSequenceIO), C.POINTER(OrbxKeyframeIO), C.POINTER(OrbxSequenceResult)]
    L.orbx_vocab_build.argtypes = [vp, C.POINTER(OrbxVocabTrain), C.POINTER(vp)]
    L.orbx_vocab_save_text.argtypes = [vp, C.c_char_p]
    L.orbx_vocab_arrays.argtypes = [vp, vp, vp, vp, vp]
    L.orbx_bowdb_build.argtypes = [vp, vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, C.POINTER(vp)]
    L.orbx_bowdb_destroy.argtypes = [vp]
    L.orbx_bowdb_destroy.restype = None
    L.orbx_bowdb_info.argtypes = [vp, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int64)]
    L.orbx_bowdb_query_range.argtypes = [vp, vp, C.c_int64, C.c_int64, C.POINTER(OrbxBowdbIO)]
    L.orbx_bowdb_query_frame.argtypes = [vp, vp, C.c_int, C.POINTER(OrbxBowdbIO)]
    L.orbx_loopver_build.argtypes = [vp, vp, C.c_int32, vp, sz, C.c_int32, C.c_int32, C.POINTER(vp)]
    L.orbx_loopver_destroy.argtypes = [vp]
    L.orbx_loopver_destroy.restype = None
    L.orbx_loopver_verify.argtypes = [vp, vp, C.c_int64, C.c_int64, C.POINTER(OrbxLoopverParams), C.POINTER(OrbxLoopverIO)]
    _lib = L
    return L


def _check(ctx, rc: int, what: str):
    if rc == ORBX_OK:
        return
    L = load_library()
    msg = L.orbx_status_string(rc).decode()
    detail = L.orbx_last_error(ctx).decode() if ctx else ""
    text = f"{what}: {msg}" + (f" ({detail})" if detail else "")
    if rc == ORBX_ERR_IMAGE_SIZE:
        raise ImageSizeError(text)
    if rc == ORBX_ERR_FILE_NOT_OPEN:
        raise FileNotOpenError(text)
    if rc in (ORBX_ERR_CUDA, ORBX_ERR_NO_DEVICE, ORBX_ERR_COMM):
        raise OrbxCudaError(text)
    raise ValueError(text)


def load_brief_template(path: str) -> np.ndarray:
    """ORBExtractor::initBriefTemplate (src/ORBExtractor.cc:242-267) -> (256, 4) float32; FileNotOpenError if missing."""
    out = np.zeros(1024, np.float32)
    rc = load_library().orbx_load_brief_template(path.encode(), out.ctypes.data_as(C.POINTER(C.c_float)))
    _check(None, rc, f"BRIEF template {path!r}")
    return out.reshape(256, 4)


@dataclass
class Camera:
    """ORB_SLAM2_ROS2::Camera statics (include/ORB_SLAM2/Camera.h:23-32) as set by System::setSetting (src/System.cc:27-73)."""

    fx: float = 718.856
    fy: float = 718.856
    cx: float = 607.1928
    cy: float = 185.2157
    bl: float = 0.537166
    dist: tuple = (0.0, 0.0, 0.0, 0.0, 0.0)
    depth_scale: float = 1.0

    @property
    def bf(self) -> np.float32:
        return np.float32(self.fx) * np.float32(self.bl)  # Camera::mfBf = mfFx * mfBl in float (src/System.cc:60)


class Context:
    """One configured front-end (owns all device memory).  Thin wrapper over orbx_create / orbx_destroy."""

    def __init__(self, width, height, n_features=2000, n_levels=8, scale_factor=1.2, ini_th=20, min_th=7, camera: Camera | None = None, max_batch=1,
                 device=-1, pattern: np.ndarray | None = None):
        L = load_library()
        cam = camera or Camera()
        cfg = OrbxConfig()
        L.orbx_default_config(C.byref(cfg))
        cfg.width, cfg.height, cfg.n_features, cfg.n_levels = int(width), int(height), int(n_features), int(n_levels)
        cfg.scale_factor, cfg.ini_th_fast, cfg.min_th_fast = float(scale_factor), int(ini_th), int(min_th)
        cfg.fx, cfg.fy, cfg.cx, cfg.cy, cfg.bf = cam.fx, cam.fy, cam.cx, cam.cy, float(cam.bf)
        for i in range(5):
            cfg.dist[i] = float(cam.dist[i]) if i < len(cam.dist) else 0.0
        cfg.depth_scale, cfg.max_batch, cfg.device = float(cam.depth_scale), int(max_batch), int(device)
        self._pattern = None
        if pattern is not None:
            self._pattern = np.ascontiguousarray(pattern, np.float32).reshape(-1)
            cfg.pattern = self._pattern.ctypes.data_as(C.POINTER(C.c_float))
        self._h = C.c_void_p()
        self.width, self.height, self.n_features, self.n_levels, self.max_batch = int(width), int(height), int(n_features), int(n_levels), int(max_batch)
        self.camera = cam
        rc = L.orbx_create(C.byref(cfg), C.byref(self._h))
        if rc != ORBX_OK:
            self._h = C.c_void_p()
        _check(None, rc, "orbx_create")
        self._L = L

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._L.orbx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- tables -------------------------------------------------------------------------------------------
    def level_info(self, level: int):
        w, h, q, s = C.c_int32(), C.c_int32(), C.c_int32(), C.c_float()
        _check(self._h, self._L.orbx_level_info(self._h, level, C.byref(w), C.byref(h), C.byref(s), C.byref(q)), "orbx_level_info")
        return w.value, h.value, np.float32(s.value), q.value

    def scaled_factors(self) -> np.ndarray:
        return np.array([self.level_info(l)[2] for l in range(self.n_levels)], np.float32)

    def set_stream(self, cuda_stream_ptr: int | None):
        """None restores the context's own stream; 0 (torch's legacy default stream) is passed as cudaStreamLegacy"""
        if cuda_stream_ptr is None:
            ptr = 0
        else:
            ptr = int(cuda_stream_ptr) or 1  # cudaStreamLegacy == (cudaStream_t)0x1
        _check(self._h, self._L.orbx_set_stream(self._h, C.c_void_p(ptr)), "orbx_set_stream")

    def set_graph(self, enable: bool):
        """single-pair calls as one CUDA graph launch (default) or as plain stream launches"""
        _check(self._h, self._L.orbx_set_graph(self._h, int(bool(enable))), "orbx_set_graph")

    def synchronize(self):
        _check(self._h, self._L.orbx_synchronize(self._h), "orbx_synchronize")

    def read_device(self, device_ptr: int, shape, dtype) -> np.ndarray:
        """copy a device result array (a pointer from OrbxDeviceResults) to a new numpy array"""
        out = np.zeros(shape, dtype)
        _check(self._h, self._L.orbx_read_device(self._h, C.c_void_p(device_ptr), out.ctypes.data, out.nbytes), "orbx_read_device")
        return out

    @property
    def launch_count(self) -> int:
        return int(self._L.orbx_launch_count(self._h))

    def algorithmic_bytes(self, stereo: bool = True) -> int:
        return int(self._L.orbx_algorithmic_bytes(self._h, 1 if stereo else 0))

    # ---- single frame, host buffers -----------------------------------------------------------------------------
    def extract(self, image: np.ndarray):
        img = _as_u8(image, self.height, self.width)
        N = self.n_features
        kps, desc, n = np.zeros(N, KP_DTYPE), np.zeros((N, 32), np.uint8), C.c_int32(0)
        rc = self._L.orbx_extract(self._h, img.ctypes.data, img.strides[0], kps.ctypes.data, desc.ctypes.data, C.addressof(n))
        _check(self._h, rc, "orbx_extract")
        return kps[: n.value], desc[: n.value]

    def get_pyramid(self, side: int = 0, blurred: bool = False):
        out = []
        for l in range(self.n_levels):
            w, h, _, _ = self.level_info(l)
            a = np.zeros((h, w), np.uint8)
            _check(self._h, self._L.orbx_get_pyramid(self._h, side, l, int(blurred), a.ctypes.data, a.strides[0]), "orbx_get_pyramid")
            out.append(a)
        return out

    def stereo_frame(self, left: np.ndarray, right: np.ndarray):
        l, r = _as_u8(left, self.height, self.width), _as_u8(right, self.height, self.width)
        N = self.n_features
        kl, kr = np.zeros(N, KP_DTYPE), np.zeros(N, KP_DTYPE)
        dl, dr = np.zeros((N, 32), np.uint8), np.zeros((N, 32), np.uint8)
        ur, dp = np.zeros(N, np.float64), np.zeros(N, np.float64)
        nl, nr, nm = C.c_int32(0), C.c_int32(0), C.c_int32(0)
        rc = self._L.orbx_stereo_frame(self._h, l.ctypes.data, l.strides[0], r.ctypes.data, r.strides[0], kl.ctypes.data, dl.ctypes.data, C.addressof(nl),
                                       kr.ctypes.data, dr.ctypes.data, C.addressof(nr), ur.ctypes.data, dp.ctypes.data, C.addressof(nm))
        _check(self._h, rc, "orbx_stereo_frame")
        a, b = nl.value, nr.value
        return StereoResult(kl[:a], dl[:a], kr[:b], dr[:b], ur[:a], dp[:a], nm.value)

    def rgbd_frame(self, gray: np.ndarray, depth_image: np.ndarray):
        g = _as_u8(gray, self.height, self.width)
        if depth_image.dtype == np.float32:
            d, dt = np.ascontiguousarray(depth_image), DEPTH_F32
        else:
            d, dt = np.ascontiguousarray(depth_image, np.uint16), DEPTH_U16
        assert d.shape == (self.height, self.width)
        N = self.n_features
        kraw, kund = np.zeros(N, KP_DTYPE), np.zeros(N, KP_DTYPE)
        desc, ur, dp, n = np.zeros((N, 32), np.uint8), np.zeros(N, np.float64), np.zeros(N, np.float64), C.c_int32(0)
        rc = self._L.orbx_rgbd_frame(self._h, g.ctypes.data, g.strides[0], d.ctypes.data, d.strides[0], dt, kraw.ctypes.data, kund.ctypes.data,
                                     desc.ctypes.data, C.addressof(n), ur.ctypes.data, dp.ctypes.data)
        _check(self._h, rc, "orbx_rgbd_frame")
        k = n.value
        return RGBDResult(kraw[:k], kund[:k], desc[:k], ur[:k], dp[:k])

    # ---- stage-level read-back (parity tests) --------------------------------------------------------------------
    def _debug_list(self, fn, image, level, cap):
        xs, ys, sc, n = np.zeros(cap, np.int32), np.zeros(cap, np.int32), np.zeros(cap, np.int32), C.c_int32(0)
        _check(self._h, fn(self._h, image, level, xs.ctypes.data, ys.ctypes.data, sc.ctypes.data, cap, C.addressof(n)), "orbx_debug")
        k = min(n.value, cap)
        return np.stack([xs[:k], ys[:k], sc[:k]], 1)

    def level_corners(self, image: int, level: int) -> np.ndarray:
        """(n,3) int32 (x_roi, y_roi, score): the level's FAST corners in the reference's detection order"""
        w, h, _, _ = self.level_info(level)
        return self._debug_list(self._L.orbx_debug_level_corners, image, level, w * h // 4 + 16)

    def level_selected(self, image: int, level: int) -> np.ndarray:
        """(n,3) int32 (x, y, score) in level coordinates: the quadtree survivors of the level"""
        return self._debug_list(self._L.orbx_debug_level_selected, image, level, self.n_features + 8)

    def grid_info(self):
        """(rows, cols, mfMinU, mfMinV, mfMaxU, mfMaxV) of VirtualFrame (include/ORB_SLAM2/Frame.h:33-43, src/Frame.cc:55-56)"""
        r, c = C.c_int32(), C.c_int32()
        b = [C.c_float() for _ in range(4)]
        _check(self._h, self._L.orbx_grid_info(self._h, C.byref(r), C.byref(c), *[C.byref(x) for x in b]), "orbx_grid_info")
        return (r.value, c.value, *[np.float32(x.value) for x in b])

    def get_grid(self, frame: int = 0):
        """VirtualFrame::mGrids of a frame of the last stereo / RGB-D call: list[rows][cols] of ascending keypoint indices"""
        rows, cols = self.grid_info()[:2]
        start = np.zeros(rows * cols + 1, np.int32)
        ent = np.zeros(self.n_features, np.int32)
        _check(self._h, self._L.orbx_get_grid(self._h, frame, start.ctypes.data, ent.ctypes.data), "orbx_get_grid")
        return [[ent[start[r * cols + c] : start[r * cols + c + 1]].copy() for c in range(cols)] for r in range(rows)]

    def quadtree_stats(self):
        """(loop-free, sequential) counts of the (image, level) quadtree problems solved so far"""
        a, b = C.c_int64(), C.c_int64()
        _check(self._h, self._L.orbx_debug_quadtree_stats(self._h, C.byref(a), C.byref(b), None), "orbx_debug_quadtree_stats")
        return a.value, b.value

    def quadtree_phase_cycles(self):
        """SM cycles per phase of the loop-free quadtree path, summed over the problems solved so far"""
        a, b = C.c_int64(), C.c_int64()
        ph = (C.c_int64 * 8)()
        _check(self._h, self._L.orbx_debug_quadtree_stats(self._h, C.byref(a), C.byref(b), ph), "orbx_debug_quadtree_stats")
        return a.value, list(ph)

    def run_quadtree(self, level: int, xs, ys, scores) -> np.ndarray:
        """run only the quadtree kernel on a corner list (ROI coords, detection order) -> (m,3) survivors in ROI coords"""
        xs, ys, sc = (np.ascontiguousarray(a, np.int32) for a in (xs, ys, scores))
        _check(self._h, self._L.orbx_debug_run_quadtree(self._h, level, xs.ctypes.data, ys.ctypes.data, sc.ctypes.data, len(xs)), "orbx_debug_run_quadtree")
        sel = self.level_selected(0, level)
        sel[:, :2] -= 16
        return sel

    # ---- tracking-side matchers (SURVEY section 8(f) rank 2) ----------------------------------------------------------
    def search_in_area(self, queries: np.ndarray, query_desc: np.ndarray, exclude: np.ndarray | None = None, frame: int = 0) -> dict:
        """findFeaturesInArea (src/Frame.cc:286-311) + exclusion (src/ORBMatcher.cc:322-331) + getBestMatch (:967-990) for
        every query against frame `frame` of the last stereo / RGB-D call -> dict(best_idx, best_dist, ratio, n_cand)"""
        q = np.ascontiguousarray(queries, AREA_QUERY_DTYPE)
        d = np.ascontiguousarray(query_desc, np.uint8)
        n = len(q)
        assert d.shape == (n, 32)
        ex = None
        if exclude is not None:
            ex = np.zeros(self.n_features, np.uint8)
            ex[: len(exclude)] = np.asarray(exclude).astype(bool)
        bi, bd, nc = np.full(n, -1, np.int32), np.zeros(n, np.int32), np.zeros(n, np.int32)
        ra = np.zeros(n, np.float32)
        rc = self._L.orbx_search_in_area(self._h, frame, n, q.ctypes.data, d.ctypes.data, ex.ctypes.data if ex is not None else None, bi.ctypes.data,
                                         bd.ctypes.data, ra.ctypes.data, nc.ctypes.data)
        _check(self._h, rc, "orbx_search_in_area")
        return dict(best_idx=bi, best_dist=bd, ratio=ra, n_cand=nc)

    def search_in_area_batch_device(self, n_frames, query_stride, d_queries, d_query_desc, d_n_queries, d_exclude, d_best_idx, d_best_dist, d_ratio,
                                    d_n_cand):
        """device-pointer variant over the frames of the last *_device call (asynchronous on the context's stream)"""
        rc = self._L.orbx_search_in_area_batch_device(self._h, n_frames, query_stride, *[C.c_void_p(x or 0) for x in (
            d_queries, d_query_desc, d_n_queries, d_exclude, d_best_idx, d_best_dist, d_ratio, d_n_cand)])
        _check(self._h, rc, "orbx_search_in_area_batch_device")

    def verify_angle(self, query_idx, train_idx, distance, kps1: np.ndarray, kps2: np.ndarray):
        """ORBMatcher::verifyAngle (src/ORBMatcher.cc:1013-1051) -> (query_idx, train_idx, distance) of the survivors"""
        qi = np.ascontiguousarray(query_idx, np.int32).copy()
        ti = np.ascontiguousarray(train_idx, np.int32).copy()
        di = np.ascontiguousarray(distance, np.float32).copy()
        k1, k2 = np.ascontiguousarray(kps1, KP_DTYPE), np.ascontiguousarray(kps2, KP_DTYPE)
        m = C.c_int32(0)
        rc = self._L.orbx_verify_angle(self._h, len(qi), qi.ctypes.data, ti.ctypes.data, di.ctypes.data, k1.ctypes.data, len(k1), k2.ctypes.data, len(k2),
                                       C.byref(m))
        _check(self._h, rc, "orbx_verify_angle")
        return qi[: m.value], ti[: m.value], di[: m.value]

    # ---- result serialisation (SURVEY section 8(f) rank 4) ------------------------------------------------------------
    def serialized_capacity(self) -> int:
        return int(self._L.orbx_serialized_capacity(self._h))

    def serialized_capacity_bow(self) -> int:
        return int(self._L.orbx_serialized_capacity_bow(self._h))

    def serialize_keyframe(self, kf_id: int, pose_rt=None, with_map_points: bool = True, frame: int = 0, bow: bool = False) -> bytes:
        """orbslam2.KeyFrameData bytes (proto/Keyframe.proto:45-64; writer src/KeyFrame.cc:553-647) of a frame of the last call.
        bow=True fills bow_vector / feature_vector from the frame's resident bow_transform() result (KeyFrame.cc:585-599)."""
        cap = self.serialized_capacity_bow() if bow else self.serialized_capacity()
        out = np.zeros(cap, np.uint8)
        pose = None if pose_rt is None else np.ascontiguousarray(pose_rt, np.float32)
        assert pose is None or pose.size == 12
        n = C.c_int64(0)
        fn, name = (self._L.orbx_serialize_keyframe_bow, "orbx_serialize_keyframe_bow") if bow else (self._L.orbx_serialize_keyframe, "orbx_serialize_keyframe")
        rc = fn(self._h, frame, kf_id, pose.ctypes.data if pose is not None else None, int(with_map_points), out.ctypes.data, cap, C.byref(n))
        _check(self._h, rc, name)
        return out[: n.value].tobytes()

    def serialize_keyframe_text(self, kf_id: int, pose_rt=None, with_map_points: bool = True, frame: int = 0, scale_header_next_id=None) -> bytes:
        """the text variant of the keyframe record, operator<<(std::ostream &, KeyFrame &) (src/KeyFrame.cc:423-533); the one-off
        "nextId scales" header line is written when scale_header_next_id is given"""
        cap = 256 + self.n_features * 320
        out = np.zeros(cap, np.uint8)
        pose = None if pose_rt is None else np.ascontiguousarray(pose_rt, np.float32)
        assert pose is None or pose.size == 12
        n = C.c_int64(0)
        rc = self._L.orbx_serialize_keyframe_text(self._h, frame, kf_id, pose.ctypes.data if pose is not None else None, int(with_map_points),
                                                  int(scale_header_next_id is not None), int(scale_header_next_id or 0), out.ctypes.data, cap, C.byref(n))
        _check(self._h, rc, "orbx_serialize_keyframe_text")
        return out[: n.value].tobytes()

    def serialize_keyframes_device(self, n_frames, id0, d_out, frame_stride, d_sizes, d_pose_rt=0, with_map_points=True):
        rc = self._L.orbx_serialize_keyframes_device(self._h, n_frames, id0, C.c_void_p(d_pose_rt or 0), int(with_map_points), C.c_void_p(d_out), frame_stride,
                                                     C.c_void_p(d_sizes))
        _check(self._h, rc, "orbx_serialize_keyframes_device")

    def serialize_keyframes_bow_device(self, n_frames, id0, d_out, frame_stride, d_sizes, d_pose_rt=0, with_map_points=True):
        rc = self._L.orbx_serialize_keyframes_bow_device(self._h, n_frames, id0, C.c_void_p(d_pose_rt or 0), int(with_map_points), C.c_void_p(d_out),
                                                         frame_stride, C.c_void_p(d_sizes))
        _check(self._h, rc, "orbx_serialize_keyframes_bow_device")

    def keyframe_list_head(self, next_id: int) -> bytes:
        """KeyFrameList fields 1 (next_id, left out when 0) and 2 (the level scale factors, packed): the bytes before the records"""
        out = np.zeros(16 + 4 * self.n_levels, np.uint8)
        n = C.c_int64(0)
        _check(self._h, self._L.orbx_keyframe_list_head(self._h, next_id, out.ctypes.data, out.size, C.byref(n)), "orbx_keyframe_list_head")
        return out[: n.value].tobytes()

    # ---- bag-of-words transform (SURVEY section 8(f) rank 3) ---------------------------------------------------------
    def bow_transform(self, vocab: "Vocabulary", frame: int = 0, levelsup: int = 4) -> dict:
        """VirtualFrame::computeBow (include/ORB_SLAM2/Frame.h:224-231) = DBoW3 Vocabulary::transform(descriptors, BowVector,
        FeatureVector, levelsup) -> dict(bow_ids, bow_vals, fv_nodes, fv_start, fv_feats)"""
        N = self.n_features
        ids, vals = np.zeros(N, np.int32), np.zeros(N, np.float64)
        fn, fs, ff = np.zeros(N, np.int32), np.zeros(N + 1, np.int32), np.zeros(N, np.int32)
        nb, nf = C.c_int32(0), C.c_int32(0)
        rc = self._L.orbx_bow_transform(self._h, vocab._h, frame, levelsup, ids.ctypes.data, vals.ctypes.data, C.byref(nb), fn.ctypes.data, fs.ctypes.data,
                                        ff.ctypes.data, C.byref(nf))
        _check(self._h, rc, "orbx_bow_transform")
        m, k = nb.value, nf.value
        return dict(bow_ids=ids[:m], bow_vals=vals[:m], fv_nodes=fn[:k], fv_start=fs[: k + 1], fv_feats=ff[: fs[k]])

    def bow_transform_batch_device(self, vocab: "Vocabulary", n_frames: int, levelsup: int = 4) -> OrbxDeviceBow:
        res = OrbxDeviceBow()
        _check(self._h, self._L.orbx_bow_transform_batch_device(self._h, vocab._h, n_frames, levelsup, C.byref(res)), "orbx_bow_transform_batch_device")
        return res

    def search_by_bow(self, kf_bow: dict, kf_desc: np.ndarray, kf_query_ok=None, frame_cand_ok=None, frame: int = 0) -> dict:
        """matching loop of ORBMatcher::searchByBow (src/ORBMatcher.cc:170-255) against a frame whose bow_transform() was just
        computed; kf_bow = a bow_transform() result of the keyframe.  -> dict(kf_idx, best_idx, best_dist, ratio, n_cand) with
        one row per visited keyframe feature that had candidates (the reference's ++nMatch)"""
        kn, ks, kf = (np.ascontiguousarray(kf_bow[k], np.int32) for k in ("fv_nodes", "fv_start", "fv_feats"))
        kd = np.ascontiguousarray(kf_desc, np.uint8)
        qm = None if kf_query_ok is None else np.ascontiguousarray(kf_query_ok, np.uint8)
        cm = None
        if frame_cand_ok is not None:
            cm = np.zeros(self.n_features, np.uint8)
            cm[: len(frame_cand_ok)] = np.asarray(frame_cand_ok).astype(bool)
        n = len(kf)
        bi, bd, nc = np.full(n, -1, np.int32), np.zeros(n, np.int32), np.zeros(n, np.int32)
        ra = np.zeros(n, np.float32)
        rc = self._L.orbx_search_by_bow(self._h, frame, len(kn), kn.ctypes.data, ks.ctypes.data, kf.ctypes.data, kd.ctypes.data, len(kd),
                                        qm.ctypes.data if qm is not None else None, cm.ctypes.data if cm is not None else None, bi.ctypes.data, bd.ctypes.data,
                                        ra.ctypes.data, nc.ctypes.data)
        _check(self._h, rc, "orbx_search_by_bow")
        ok = nc > 0
        return dict(kf_idx=kf[ok], best_idx=bi[ok], best_dist=bd[ok], ratio=ra[ok], n_cand=nc[ok])

    # ---- batches ----------------------------------------------------------------------------------------------------
    def stereo_batch(self, left: np.ndarray, right: np.ndarray, out: "StereoBatchBuffers | None" = None):
        """left/right: (n, H, W) uint8 host arrays (pinned memory makes the copies asynchronous)."""
        n = left.shape[0]
        assert left.shape == right.shape == (n, self.height, self.width) and left.strides == right.strides and left.dtype == np.uint8
        ob = out or StereoBatchBuffers.numpy(n, self.n_features)
        rc = self._L.orbx_stereo_batch(self._h, n, left.ctypes.data, right.ctypes.data, left.strides[1], left.strides[0], ob.kps_left.ctypes.data,
                                       ob.desc_left.ctypes.data, ob.n_left.ctypes.data, ob.kps_right.ctypes.data, ob.desc_right.ctypes.data,
                                       ob.n_right.ctypes.data, ob.u_right.ctypes.data, ob.depth.ctypes.data, ob.n_matches.ctypes.data)
        _check(self._h, rc, "orbx_stereo_batch")
        return ob

    def stereo_batch_ptr(self, n_frames, left_ptr, right_ptr, stride, frame_stride, ptrs):
        """raw-pointer variant of stereo_batch (host pointers; ptrs = 9 output addresses or 0)."""
        rc = self._L.orbx_stereo_batch(self._h, n_frames, left_ptr, right_ptr, stride, frame_stride, *[C.c_void_p(q or 0) for q in ptrs])
        _check(self._h, rc, "orbx_stereo_batch")

    def stereo_batch_device(self, n_frames, d_left_ptr, d_right_ptr, stride, frame_stride) -> OrbxDeviceResults:
        res = OrbxDeviceResults()
        rc = self._L.orbx_stereo_batch_device(self._h, n_frames, C.c_void_p(d_left_ptr), C.c_void_p(d_right_ptr), stride, frame_stride, C.byref(res))
        _check(self._h, rc, "orbx_stereo_batch_device")
        return res

    def profile_stereo_batch_device(self, n_frames, d_left_ptr, d_right_ptr, stride, frame_stride) -> dict:
        """device milliseconds per stage (events between the kernels; blocks)"""
        ms = (C.c_float * N_STAGES)()
        rc = self._L.orbx_profile_stereo_batch_device(self._h, n_frames, C.c_void_p(d_left_ptr), C.c_void_p(d_right_ptr), stride, frame_stride, ms)
        _check(self._h, rc, "orbx_profile_stereo_batch_device")
        return {self._L.orbx_stage_name(i).decode(): float(ms[i]) for i in range(N_STAGES)}

    # ---- whole sequences sharded by frame (SURVEY section 8e) --------------------------------------------------------
    @property
    def frame_epoch(self) -> int:
        return int(self._L.orbx_frame_epoch(self._h))

    def record_layout(self) -> OrbxRecordLayout:
        lay = OrbxRecordLayout()
        _check(self._h, self._L.orbx_record_layout_get(self._h, C.byref(lay)), "orbx_record_layout_get")
        return lay

    def record_dtype(self) -> np.dtype:
        """numpy view of one frame record (orbx_record_layout): fields n_left, n_right, n_matches, kps_left, desc_left, ..."""
        lay, N = self.record_layout(), self.n_features
        return np.dtype({"names": ["n_left", "n_right", "n_matches", "kps_left", "desc_left", "kps_right", "desc_right", "u_right", "depth"],
                         "formats": ["<i4", "<i4", "<i4", (KP_DTYPE, (N,)), ("u1", (N, 32)), (KP_DTYPE, (N,)), ("u1", (N, 32)), ("<f8", (N,)), ("<f8", (N,))],
                         "offsets": [0, 4, 8, lay.off_kps_left, lay.off_desc_left, lay.off_kps_right, lay.off_desc_right, lay.off_u_right, lay.off_depth],
                         "itemsize": lay.record_bytes})

    def sequence_stereo_ptr(self, n_frames_total: int, left_ptr: int, right_ptr: int, stride: int, frame_stride: int, comm: "Communicator | None" = None,
                            input_on_device: bool = False, records_ptr: int = 0, record_stride: int = 0, records_on_device: bool = False,
                            gathered_desc_host_ptr: int = 0, gathered_n_host_ptr: int = 0) -> OrbxSequenceResult:
        """orbx_sequence_stereo on raw pointers: left/right = THIS RANK'S block of the sequence"""
        io = OrbxSequenceIO(left_ptr, right_ptr, stride, frame_stride, int(input_on_device), int(records_on_device), records_ptr or None,
                            record_stride, gathered_desc_host_ptr or None, gathered_n_host_ptr or None)
        res = OrbxSequenceResult()
        rc = self._L.orbx_sequence_stereo(self._h, comm._h if comm is not None else None, n_frames_total, C.byref(io), C.byref(res))
        _check(self._h, rc, "orbx_sequence_stereo")
        return res

    def sequence_stereo(self, left: np.ndarray, right: np.ndarray, n_frames_total: int | None = None, comm: "Communicator | None" = None,
                        gather_to_host: bool = True):
        """left/right: (n_local, H, W) uint8 host arrays holding this rank's block.  -> (records, gathered_desc, gathered_n):
        records = numpy structured array (record_dtype) of the block's frames; gathered_* cover the WHOLE sequence."""
        n = left.shape[0]
        F = n if n_frames_total is None else int(n_frames_total)
        assert left.shape == right.shape == (n, self.height, self.width) and left.strides == right.strides and left.dtype == np.uint8
        rec = np.zeros(max(n, 1), self.record_dtype())
        gd = np.zeros((F, self.n_features, 32), np.uint8) if gather_to_host else None
        gn = np.zeros(F, np.int32) if gather_to_host else None
        res = self.sequence_stereo_ptr(F, left.ctypes.data, right.ctypes.data, left.strides[1], left.strides[0], comm, False, rec.ctypes.data,
                                       rec.dtype.itemsize, False, gd.ctypes.data if gather_to_host else 0, gn.ctypes.data if gather_to_host else 0)
        assert res.frame_hi - res.frame_lo == n, "left/right must hold exactly this rank's block (orbx_frame_range)"
        return rec[:n], gd, gn

    def sequence_stereo_keyframes_ptr(self, n_frames_total: int, left_ptr: int, right_ptr: int, stride: int, frame_stride: int,
                                      kf_out_ptr: int, kf_stride: int, kf_sizes_ptr: int, vocab: "Vocabulary | None" = None, levelsup: int = 4,
                                      id0: int = 0, with_map_points: bool = True, poses_ptr: int = 0, kf_on_device: bool = False,
                                      comm: "Communicator | None" = None, input_on_device: bool = False, records_ptr: int = 0, record_stride: int = 0,
                                      records_on_device: bool = False, gathered_desc_host_ptr: int = 0, gathered_n_host_ptr: int = 0) -> OrbxSequenceResult:
        """orbx_sequence_stereo_keyframes on raw pointers: the sequence_stereo_ptr outputs plus this rank's keyframe records
        (kf_out_ptr[i * kf_stride], sizes in kf_sizes_ptr, poses_ptr[n_local][12] or 0; all in the memory kf_on_device names)"""
        io = OrbxSequenceIO(left_ptr, right_ptr, stride, frame_stride, int(input_on_device), int(records_on_device), records_ptr or None,
                            record_stride, gathered_desc_host_ptr or None, gathered_n_host_ptr or None)
        kio = OrbxKeyframeIO(vocab._h if vocab is not None else None, int(levelsup), int(with_map_points), int(id0), poses_ptr or None, int(kf_on_device),
                             kf_out_ptr or None, int(kf_stride), kf_sizes_ptr or None)
        res = OrbxSequenceResult()
        rc = self._L.orbx_sequence_stereo_keyframes(self._h, comm._h if comm is not None else None, n_frames_total, C.byref(io), C.byref(kio), C.byref(res))
        _check(self._h, rc, "orbx_sequence_stereo_keyframes")
        return res

    def sequence_stereo_keyframes(self, left: np.ndarray, right: np.ndarray, vocab: "Vocabulary | None" = None, levelsup: int = 4, id0: int = 0,
                                  with_map_points: bool = True, poses=None, comm: "Communicator | None" = None, n_frames_total: int | None = None,
                                  gather_to_host: bool = True):
        """sequence_stereo plus the KeyFrameData record of every frame of this rank's block (bag of words from `vocab`, or
        present-but-empty without one; id = id0 + global frame index; poses: (n_local, 12) Tcw or None = identity).
        -> (records, gathered_desc, gathered_n, keyframes, sizes): keyframes = (n_local, stride) uint8, record i is
        keyframes[i, :sizes[i]]; write_keyframe_list() frames them as a KeyFrameList."""
        n = left.shape[0]
        F = n if n_frames_total is None else int(n_frames_total)
        assert left.shape == right.shape == (n, self.height, self.width) and left.strides == right.strides and left.dtype == np.uint8
        pose = None if poses is None else np.ascontiguousarray(poses, np.float32).reshape(n, 12)
        ks = self.serialized_capacity_bow() if vocab is not None else self.serialized_capacity()
        kf = _aligned_zeros((max(n, 1), ks))
        sizes = np.zeros(max(n, 1), np.int64)
        rec = np.zeros(max(n, 1), self.record_dtype())
        gd = np.zeros((F, self.n_features, 32), np.uint8) if gather_to_host else None
        gn = np.zeros(F, np.int32) if gather_to_host else None
        res = self.sequence_stereo_keyframes_ptr(F, left.ctypes.data, right.ctypes.data, left.strides[1], left.strides[0], kf.ctypes.data, ks, sizes.ctypes.data,
                                                 vocab, levelsup, id0, with_map_points, pose.ctypes.data if pose is not None else 0, False, comm, False,
                                                 rec.ctypes.data, rec.dtype.itemsize, False, gd.ctypes.data if gather_to_host else 0,
                                                 gn.ctypes.data if gather_to_host else 0)
        assert res.frame_hi - res.frame_lo == n, "left/right must hold exactly this rank's block (orbx_frame_range)"
        return rec[:n], gd, gn, kf[:n], sizes[:n]

    def extract_batch_device(self, n_images, d_ptr, stride, frame_stride) -> OrbxDeviceResults:
        res = OrbxDeviceResults()
        rc = self._L.orbx_extract_batch_device(self._h, n_images, C.c_void_p(d_ptr), stride, frame_stride, C.byref(res))
        _check(self._h, rc, "orbx_extract_batch_device")
        return res

    def rgbd_batch_device(self, n_frames, d_gray, gstride, gframe, d_depth, dstride, dframe, depth_type) -> OrbxDeviceResults:
        res = OrbxDeviceResults()
        rc = self._L.orbx_rgbd_batch_device(self._h, n_frames, C.c_void_p(d_gray), gstride, gframe, C.c_void_p(d_depth), dstride, dframe, depth_type,
                                            C.byref(res))
        _check(self._h, rc, "orbx_rgbd_batch_device")
        return res


def _aligned_zeros(shape, align: int = 16) -> np.ndarray:
    n = int(np.prod(shape))
    raw = np.zeros(n + align, np.uint8)
    k = (-raw.ctypes.data) % align
    return raw[k : k + n].reshape(shape)


def write_keyframe_list(fileobj, ctx: Context, records, sizes, next_id: int, head: bool = True) -> int:
    """Writes records[i, :sizes[i]] as the keyframes (field 3) of an orbslam2.KeyFrameList (proto/Keyframe.proto:66-70, writer
    src/Map.cc:205-224), preceded by the head (next_id, the context's scale factors) when `head`; piece by piece, without
    assembling the list in memory.  Rank 0 of a sharded export writes the head, the others entries only: their outputs
    concatenated in rank order are one list.  -> bytes written"""
    L = ctx._L
    pre = (C.c_uint8 * 11)()
    total = 0
    if head:
        h = ctx.keyframe_list_head(next_id)
        fileobj.write(h)
        total += len(h)
    recs = np.asarray(records)
    for i, sz in enumerate(np.asarray(sizes, np.int64)):
        k = L.orbx_keyframe_list_entry_prefix(int(sz), pre)
        _check(ctx._h, k if k < 0 else ORBX_OK, "orbx_keyframe_list_entry_prefix")
        fileobj.write(bytes(pre[:k]))
        fileobj.write(memoryview(recs[i, : int(sz)]))
        total += k + int(sz)
    return total


def frame_range(n_frames_total: int, rank: int, world: int) -> range:
    """orbx_frame_range: the contiguous block of rank `rank` (SURVEY.md section 8e)"""
    lo, hi = C.c_int64(), C.c_int64()
    load_library().orbx_frame_range(n_frames_total, rank, world, C.byref(lo), C.byref(hi))
    return range(lo.value, hi.value)


class Communicator:
    """orbx_comm: the ranks that share one frame-sharded sequence.  Multi-process: rank 0 makes `unique_id()`, ships it to
    the others (e.g. torch.distributed.broadcast_object_list), every rank builds Communicator(ctx, rank, world, id, F)."""

    def __init__(self, ctx: Context, rank: int, world: int, unique_id: bytes, max_frames_total: int, _handle=None):
        self._L, self.ctx = ctx._L, ctx
        self._h = C.c_void_p()
        if _handle is not None:
            self._h = _handle
            return
        buf = (C.c_uint8 * COMM_ID_BYTES).from_buffer_copy(unique_id)
        _check(ctx._h, self._L.orbx_comm_create(ctx._h, rank, world, buf, max_frames_total, C.byref(self._h)), "orbx_comm_create")

    @staticmethod
    def unique_id() -> bytes:
        buf = (C.c_uint8 * COMM_ID_BYTES)()
        _check(None, load_library().orbx_comm_unique_id(buf), "orbx_comm_unique_id")
        return bytes(buf)

    @staticmethod
    def local(ctxs, max_frames_total: int):
        """one process driving len(ctxs) ranks (peer-memory transport, no NCCL) -> list of Communicators"""
        L = load_library()
        n = len(ctxs)
        hs = (C.c_void_p * n)(*[c._h for c in ctxs])
        out = (C.c_void_p * n)()
        _check(ctxs[0]._h, L.orbx_comm_create_local(hs, n, max_frames_total, out), "orbx_comm_create_local")
        return [Communicator(ctxs[r], r, n, b"", max_frames_total, _handle=C.c_void_p(out[r])) for r in range(n)]

    def ipc_handle(self) -> bytes:
        buf = (C.c_uint8 * IPC_HANDLE_BYTES)()
        _check(self.ctx._h, self._L.orbx_comm_ipc_handle(self._h, buf), "orbx_comm_ipc_handle")
        return bytes(buf)

    def open_peers(self, handles):
        """handles[r] = rank r's ipc_handle(); switches the data path to peer-memory stores (ORBX_TRANSPORT_PEER)"""
        blob = b"".join(handles)
        buf = (C.c_uint8 * len(blob)).from_buffer_copy(blob)
        _check(self.ctx._h, self._L.orbx_comm_open_peers(self._h, buf), "orbx_comm_open_peers")

    def info(self):
        v = [C.c_int32() for _ in range(3)]
        self._L.orbx_comm_info(self._h, *[C.byref(x) for x in v])
        return dict(rank=v[0].value, world=v[1].value, transport=v[2].value)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._L.orbx_comm_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _as_u8(a: np.ndarray, h: int, w: int) -> np.ndarray:
    if a.dtype != np.uint8 or a.ndim != 2 or a.shape != (h, w):
        raise ValueError(f"expected a {h}x{w} uint8 image, got {a.shape} {a.dtype}")
    if a.strides[1] != 1:
        a = np.ascontiguousarray(a)
    return a


@dataclass
class StereoResult:
    kps_left: np.ndarray
    desc_left: np.ndarray
    kps_right: np.ndarray
    desc_right: np.ndarray
    u_right: np.ndarray
    depth: np.ndarray
    n_matches: int


@dataclass
class RGBDResult:
    kps_raw: np.ndarray
    kps: np.ndarray
    desc: np.ndarray
    u_right: np.ndarray
    depth: np.ndarray


@dataclass
class StereoBatchBuffers:
    kps_left: np.ndarray
    desc_left: np.ndarray
    n_left: np.ndarray
    kps_right: np.ndarray
    desc_right: np.ndarray
    n_right: np.ndarray
    u_right: np.ndarray
    depth: np.ndarray
    n_matches: np.ndarray

    @staticmethod
    def numpy(n: int, n_features: int) -> "StereoBatchBuffers":
        N = n_features
        return StereoBatchBuffers(np.zeros((n, N), KP_DTYPE), np.zeros((n, N, 32), np.uint8), np.zeros(n, np.int32), np.zeros((n, N), KP_DTYPE),
                                  np.zeros((n, N, 32), np.uint8), np.zeros(n, np.int32), np.zeros((n, N), np.float64), np.zeros((n, N), np.float64),
                                  np.zeros(n, np.int32))


# ----------------------------------------------------------------------------------------------------------------
# reference-shaped classes
# ----------------------------------------------------------------------------------------------------------------
_ctx_cache: dict = {}


def _context_for(h, w, n_features, n_levels, scale, ini_th, min_th, camera: Camera, pattern_key, pattern) -> Context:
    key = (h, w, n_features, n_levels, float(scale), ini_th, min_th, camera.fx, camera.fy, camera.cx, camera.cy, camera.bl, tuple(camera.dist),
           camera.depth_scale, pattern_key)
    ctx = _ctx_cache.get(key)
    if ctx is None:
        ctx = Context(w, h, n_features, n_levels, scale, ini_th, min_th, camera, max_batch=1, pattern=pattern)
        _ctx_cache[key] = ctx
    return ctx


class ORBExtractor:
    """Mirror of ORB_SLAM2_ROS2::ORBExtractor (include/ORB_SLAM2/ORBExtractor.h:99-161).

    The constructor takes the image (the reference builds the pyramid there, src/ORBExtractor.cc:205-214); ``extract()``
    returns (keypoints, descriptors) where descriptors[i] is the reference's i-th 1x32 CV_8U Mat.
    """

    mnBorderSize = 19

    def __init__(self, image: np.ndarray, nFeatures: int, pyramidLevels: int, scaleFactor: float, bfTemFp: str | None, maxThreshold: int,
                 minThreshold: int, camera: Camera | None = None):
        pattern = load_brief_template(bfTemFp) if bfTemFp else None  # FileNotOpenError like :247-250
        self._image = image
        h, w = image.shape
        self._ctx = _context_for(h, w, nFeatures, pyramidLevels, scaleFactor, maxThreshold, minThreshold, camera or Camera(), bfTemFp, pattern)
        self._done = False

    def extract(self):
        kps, desc = self._ctx.extract(self._image)
        self._done = True
        return kps, desc

    def getPyramid(self):
        if not self._done:
            self.extract()
        return self._ctx.get_pyramid(0)

    def getScaledFactors(self) -> np.ndarray:
        return self._ctx.scaled_factors()


@dataclass
class Frame:
    """The per-frame outputs of ORB_SLAM2_ROS2::Frame that belong to the hot path (include/ORB_SLAM2/Frame.h:263-274)."""

    mvFeatsLeft: np.ndarray
    mvLeftDescriptor: np.ndarray
    mvFeatsRight: np.ndarray | None
    mRightDescriptor: np.ndarray | None
    mvFeatsRightU: np.ndarray
    mvDepths: np.ndarray
    mnN: int
    extra: dict = field(default_factory=dict)

    @staticmethod
    def createStereo(leftImg, rightImg, nFeatures, briefFp, maxThresh, minThresh, pVoc=None, nLevels=8, scale=1.2, camera: Camera | None = None) -> "Frame":
        """Frame::createStereo (include/ORB_SLAM2/Frame.h:313-322)."""
        pattern = load_brief_template(briefFp) if briefFp else None
        h, w = leftImg.shape
        ctx = _context_for(h, w, nFeatures, nLevels, scale, maxThresh, minThresh, camera or Camera(), briefFp, pattern)
        r = ctx.stereo_frame(leftImg, rightImg)
        return Frame(r.kps_left, r.desc_left, r.kps_right, r.desc_right, r.u_right, r.depth, r.n_matches, {"ctx": ctx})

    @staticmethod
    def createRGBD(colorImg, depthImg, nFeatures, briefF, maxThresh, minThresh, pVoc=None, dScale=1.0, nLevels=8, scale=1.2,
                   camera: Camera | None = None) -> "Frame":
        """Frame::createRGBD (include/ORB_SLAM2/Frame.h:325-331)."""
        import dataclasses

        cam = dataclasses.replace(camera or Camera(), depth_scale=float(dScale))
        pattern = load_brief_template(briefF) if briefF else None
        h, w = colorImg.shape
        ctx = _context_for(h, w, nFeatures, nLevels, scale, maxThresh, minThresh, cam, briefF, pattern)
        r = ctx.rgbd_frame(colorImg, depthImg)
        return Frame(r.kps, r.desc, None, None, r.u_right, r.depth, int((r.depth > 0).sum()), {"ctx": ctx, "kps_raw": r.kps_raw})


class ORBMatcher:
    """Host mirror of the tracking-side entry points of ORB_SLAM2_ROS2::ORBMatcher (include/ORB_SLAM2/ORBMatcher.h:17-124)
    whose inner loops run on the device (Context.search_in_area / verify_angle).  Map points are not modelled: the callers
    pass the per-keypoint "has a usable map point" masks the reference derives from them."""

    mnMaxThreshold, mnMinThreshold, mnMeanThreshold = 100, 50, 75  # src/ORBMatcher.cc:1086-1088
    mnBinNum, mnBinChoose = 30, 3                                   # :1091-1092

    def __init__(self, ratio: float = 0.6, checkOri: bool = True):
        self.mfRatio = np.float32(ratio)
        self.mbCheckOri = checkOri

    def searchByProjection(self, pFrame1: "Frame", kps2: np.ndarray, desc2: np.ndarray, valid2: np.ndarray, hasMp1: np.ndarray | None, th: float,
                           tlc_z: float = 0.0, baseline: float = 0.0, bFuse: bool = False) -> np.ndarray:
        """searchByProjection(pFrame1, pFrame2, matches, th, bFuse) (src/ORBMatcher.cc:265-347).  kps2/desc2 = pFrame2's
        left keypoints/descriptors, valid2[idx] = "mps2[idx] is a good map point" (and, for bFuse, in view of pFrame1),
        hasMp1[i] = "pFrame1 keypoint i already has a good map point" (dropped from the candidates unless bFuse),
        tlc_z = z of pFrame1's camera centre in pFrame2's camera frame (:275-281).  -> (m, 3) int32 rows (queryIdx =
        pFrame1 keypoint, trainIdx = idx, distance), ascending idx."""
        ctx: Context = pFrame1.extra["ctx"]
        idx = np.nonzero(np.asarray(valid2).astype(bool))[0]
        q = np.zeros(len(idx), AREA_QUERY_DTYPE)
        q["x"], q["y"], q["octave"], q["radius"] = kps2["x"][idx], kps2["y"][idx], kps2["octave"][idx], np.float32(th)
        up = abs(np.float32(tlc_z)) > np.float32(baseline) and tlc_z > 0
        down = abs(np.float32(tlc_z)) > np.float32(baseline) and not tlc_z > 0
        if up:
            q["min_level"], q["max_level"] = q["octave"], 7
        elif down:
            q["min_level"], q["max_level"] = 0, q["octave"]
        else:
            q["min_level"], q["max_level"] = np.maximum(0, q["octave"] - 1), np.minimum(q["octave"] + 1, 7)
        r = ctx.search_in_area(q, desc2[idx], None if bFuse else hasMp1, frame=pFrame1.extra.get("frame", 0))
        ok = (r["n_cand"] > 0) & (r["ratio"] < self.mfRatio) & (r["best_dist"] < self.mnMinThreshold)
        return np.stack([r["best_idx"][ok], idx[ok].astype(np.int32), r["best_dist"][ok]], axis=1).astype(np.int32)

    def searchByProjectionMapPoints(self, pframe: "Frame", uv: np.ndarray, octave: np.ndarray, cosTheta: np.ndarray, mp_desc: np.ndarray, th: float,
                                    hasMp: np.ndarray, bFuse: bool = False, nLevels: int = 8):
        """searchByProjection(pframe, mapPoints, th, matches, bFuse) (src/ORBMatcher.cc:561-621) for the map points that
        passed isInVision: uv = projections, octave = predictLevel(distance), cosTheta = viewing-angle cosine, mp_desc =
        their descriptors, hasMp[i] = "pframe keypoint i has a good map point".
        -> (nMatches, matches): matches = (m, 3) int32 rows (keypoint idx, map point idx, distance); for bFuse = False these
        are the map points newly assigned (first map point to claim a free keypoint wins, :594-601)."""
        ctx: Context = pframe.extra["ctx"]
        n = len(uv)
        q = np.zeros(n, AREA_QUERY_DTYPE)
        q["x"], q["y"], q["octave"] = uv[:, 0], uv[:, 1], octave
        q["radius"] = np.where(np.asarray(cosTheta, np.float32) > np.float32(0.998), np.float32(2.5), np.float32(4.0)) * np.float32(th)
        q["min_level"], q["max_level"] = np.maximum(0, q["octave"] - 1), np.minimum(nLevels - 1, q["octave"] + 1)
        r = ctx.search_in_area(q, mp_desc, None, frame=pframe.extra.get("frame", 0))
        ok = (r["n_cand"] > 0) & (r["best_dist"] < self.mnMinThreshold) & (r["ratio"] < self.mfRatio)
        taken = np.asarray(hasMp).astype(bool).copy()
        n_matches = 0 if bFuse else int(taken.sum())
        out = []
        for i in np.nonzero(ok)[0]:
            k = int(r["best_idx"][i])
            if bFuse:
                out.append((k, i, r["best_dist"][i]))
                n_matches += 1
            elif not taken[k]:
                taken[k] = True
                out.append((k, i, r["best_dist"][i]))
                n_matches += 1
        return n_matches, np.asarray(out, np.int32).reshape(-1, 3)

    def searchByBow(self, pFrame: "Frame", vocab: "Vocabulary", kf_kps: np.ndarray, kf_desc: np.ndarray, kf_bow: dict, kfGood: np.ndarray,
                    frameGood: np.ndarray, bAddMPs: bool = False, bLoop: bool = False, levelsup: int = 4) -> np.ndarray:
        """searchByBow(pFrame, pKframe, matches, bAddMPs, bLoop) (src/ORBMatcher.cc:170-255).  kfGood[i] / frameGood[i] = "the
        feature has a good map point" (for bAddMPs: "... that is in the map").  -> (m, 3) int32 rows (queryIdx = frame
        feature, trainIdx = keyframe feature, distance) after verifyAngle when mbCheckOri."""
        ctx: Context = pFrame.extra["ctx"]
        ctx.bow_transform(vocab, frame=pFrame.extra.get("frame", 0), levelsup=levelsup)  # pFrame->computeBow() (levelsup 4, Frame.h:229)
        kg, fg = np.asarray(kfGood).astype(bool), np.asarray(frameGood).astype(bool)
        if bAddMPs:
            q_ok, c_ok = ~kg, ~fg          # both sides without a map point (:198-201, :221-225)
        elif bLoop:
            q_ok, c_ok = np.ones_like(kg), np.ones_like(fg)
        else:
            q_ok, c_ok = kg, ~fg           # keyframe side has one, frame side does not (:207-211, :230-233)
        r = ctx.search_by_bow(kf_bow, kf_desc, q_ok, c_ok, frame=pFrame.extra.get("frame", 0))
        keep = ~((r["best_dist"] > self.mnMinThreshold) | (r["ratio"] > self.mfRatio))
        m = np.stack([r["best_idx"][keep], r["kf_idx"][keep], r["best_dist"][keep]], axis=1).astype(np.int32).reshape(-1, 3)
        if self.mbCheckOri and len(m):
            m = self.verifyAngle(ctx, m, pFrame.mvFeatsLeft, kf_kps)
        return m

    def verifyAngle(self, ctx: Context, matches: np.ndarray, keyPoints1: np.ndarray, keyPoints2: np.ndarray) -> np.ndarray:
        """ORBMatcher::verifyAngle (src/ORBMatcher.cc:1013-1051) on (m, 3) rows (queryIdx, trainIdx, distance)"""
        qi, ti, di = ctx.verify_angle(matches[:, 0], matches[:, 1], matches[:, 2].astype(np.float32), keyPoints1, keyPoints2)
        return np.stack([qi, ti, di.astype(np.int32)], axis=1).astype(np.int32).reshape(-1, 3)


class Vocabulary:
    """DBoW3::Vocabulary resident on a context's device (the reference loads it in src/System.cc:93)."""

    def __init__(self, ctx: Context, k: int, L: int, parent, is_leaf, desc, weight):
        parent = np.ascontiguousarray(parent, np.int32)
        is_leaf = np.ascontiguousarray(is_leaf, np.uint8)
        desc = np.ascontiguousarray(desc, np.uint8)
        weight = np.ascontiguousarray(weight, np.float64)
        assert desc.shape == (len(parent), 32) and len(is_leaf) == len(parent) == len(weight)
        self._L = ctx._L
        self._h = C.c_void_p()
        rc = self._L.orbx_vocab_create(ctx._h, k, L, len(parent), parent.ctypes.data, is_leaf.ctypes.data, desc.ctypes.data, weight.ctypes.data,
                                       C.byref(self._h))
        _check(ctx._h, rc, "orbx_vocab_create")

    @classmethod
    def load_text(cls, ctx: Context, path: str) -> "Vocabulary":
        """ORB-SLAM2 / DBoW3 text vocabulary (ORBvoc.txt)"""
        self = cls.__new__(cls)
        self._L = ctx._L
        self._h = C.c_void_p()
        _check(ctx._h, self._L.orbx_vocab_load_text(ctx._h, path.encode(), C.byref(self._h)), "orbx_vocab_load_text")
        return self

    @classmethod
    def build(cls, ctx: Context, desc, counts, n_frames: int | None = None, k: int = 10, L: int = 6, seed: int = 0, stride: int | None = None,
              stats: dict | None = None) -> "Vocabulary":
        """DBoW TemplatedVocabulary::create on the device (orbx_vocab_build) from the training set desc[f][i], i < counts[f].
        desc / counts: numpy arrays ((F, stride, 32) uint8 and (F,) int32), or device pointers (ints) of ctx's device, e.g.
        OrbxSequenceResult.gathered_desc / gathered_n, which then need n_frames (the sequence's F: padding rows are not
        frames) and stride (its n_features).  stats, if given, receives iters (per level), n_capped and level_ms (device time
        per level, then of the TF_IDF step)."""
        self = cls.__new__(cls)
        self._L = ctx._L
        self._h = C.c_void_p()
        on_device = isinstance(desc, int)
        if on_device:
            assert isinstance(counts, int) and n_frames is not None and stride is not None, "device pointers need n_frames and stride"
            F, S, dp, cp = int(n_frames), int(stride), desc, counts
        else:
            d = np.ascontiguousarray(desc, np.uint8)
            assert d.ndim == 3 and d.shape[2] == 32
            F = d.shape[0] if n_frames is None else int(n_frames)
            S = d.shape[1]
            d = np.ascontiguousarray(d[:F])
            cnt = np.ascontiguousarray(np.asarray(counts)[:F], np.int32)
            assert len(cnt) == F
            dp, cp = d.ctypes.data, cnt.ctypes.data
        iters, capped, ms = np.zeros(max(int(L), 1), np.int32), C.c_int32(0), np.zeros(max(int(L), 1) + 1, np.float32)
        tr = OrbxVocabTrain(dp, cp, F, S, int(on_device), int(k), int(L), int(seed) & (2**64 - 1), iters.ctypes.data, C.addressof(capped), ms.ctypes.data)
        _check(ctx._h, self._L.orbx_vocab_build(ctx._h, C.byref(tr), C.byref(self._h)), "orbx_vocab_build")
        if stats is not None:
            stats.update(iters=iters[: int(L)].tolist(), n_capped=int(capped.value), level_ms=ms[: int(L) + 1].tolist())
        return self

    def save_text(self, path: str):
        """ORBvoc.txt text format (TemplatedVocabulary::saveToTextFile), readable by load_text"""
        _check(None, self._L.orbx_vocab_save_text(self._h, path.encode()), f"orbx_vocab_save_text {path!r}")

    def arrays(self) -> dict:
        """the nodes as text-format records (record i = node i + 1): parent, is_leaf, desc (n, 32), weight"""
        n = self.info()["n_nodes"] - 1
        par, leaf, desc, w = np.zeros(n, np.int32), np.zeros(n, np.uint8), np.zeros((n, 32), np.uint8), np.zeros(n, np.float64)
        _check(None, self._L.orbx_vocab_arrays(self._h, par.ctypes.data, leaf.ctypes.data, desc.ctypes.data, w.ctypes.data), "orbx_vocab_arrays")
        return dict(parent=par, is_leaf=leaf, desc=desc, weight=w)

    def info(self):
        v = [C.c_int32() for _ in range(4)]
        self._L.orbx_vocab_info(self._h, *[C.byref(x) for x in v])
        return dict(k=v[0].value, L=v[1].value, n_nodes=v[2].value, n_words=v[3].value)

    def close(self):
        if getattr(self, "_h", None):
            self._L.orbx_vocab_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


BOWDB_OUTPUTS = ("cand_frame", "cand_score", "cand_common", "n_sharing", "max_common", "n_scored", "n_kept")


class BowDatabase:
    """Keyframe database over a sequence (orbx_bowdb_*): the BoW inverted file and the first stage of ORB-SLAM2's
    KeyFrameDatabase::DetectLoopCandidates / DetectRelocalizationCandidates, built once on a context's device."""

    @classmethod
    def build(cls, ctx: Context, vocab: Vocabulary, desc, counts, n_frames: int | None = None, stride: int | None = None) -> "BowDatabase":
        """from the descriptors desc[f][i], i < counts[f]: numpy arrays ((F, stride, 32) uint8 and (F,) int32), or device
        pointers (ints) of ctx's device such as OrbxSequenceResult.gathered_desc / gathered_n, which then need n_frames (the
        sequence's F) and stride (its n_features)"""
        self = cls.__new__(cls)
        self._L, self.ctx = ctx._L, ctx
        self._h = C.c_void_p()
        on_device = isinstance(desc, int)
        if on_device:
            assert isinstance(counts, int) and n_frames is not None and stride is not None, "device pointers need n_frames and stride"
            F, S, dp, cp = int(n_frames), int(stride), desc, counts
        else:
            d = np.ascontiguousarray(desc, np.uint8)
            assert d.ndim == 3 and d.shape[2] == 32
            F = d.shape[0] if n_frames is None else int(n_frames)
            S = d.shape[1]
            d = np.ascontiguousarray(d[:F])
            cnt = np.ascontiguousarray(np.asarray(counts)[:F], np.int32)
            assert len(cnt) == F
            dp, cp = d.ctypes.data, cnt.ctypes.data
        _check(ctx._h, self._L.orbx_bowdb_build(ctx._h, vocab._h, dp, cp, F, S, int(on_device), C.byref(self._h)), "orbx_bowdb_build")
        return self

    def info(self) -> dict:
        f, w, p = C.c_int32(), C.c_int32(), C.c_int64()
        _check(None, self._L.orbx_bowdb_info(self._h, C.byref(f), C.byref(w), C.byref(p)), "orbx_bowdb_info")
        return dict(n_frames=f.value, n_words=w.value, n_postings=p.value)

    def _io(self, window, min_score, top_k, on_device, ptrs) -> OrbxBowdbIO:
        return OrbxBowdbIO(int(window), float(min_score), int(top_k), int(on_device), *[p or None for p in ptrs])

    def query_ptr(self, q_lo: int, q_hi: int, top_k: int, exclude_window: int, min_score: float, ptrs, on_device: bool = True):
        """orbx_bowdb_query_range with raw output pointers, in BOWDB_OUTPUTS order (0 = not wanted)"""
        io = self._io(exclude_window, min_score, top_k, on_device, ptrs)
        _check(self.ctx._h, self._L.orbx_bowdb_query_range(self.ctx._h, self._h, int(q_lo), int(q_hi), C.byref(io)), "orbx_bowdb_query_range")

    def query_frame_ptr(self, frame: int, top_k: int, min_score: float, ptrs, on_device: bool = True):
        """orbx_bowdb_query_frame with raw output pointers, in BOWDB_OUTPUTS order (0 = not wanted)"""
        io = self._io(-1, min_score, top_k, on_device, ptrs)
        _check(self.ctx._h, self._L.orbx_bowdb_query_frame(self.ctx._h, self._h, int(frame), C.byref(io)), "orbx_bowdb_query_frame")

    @staticmethod
    def _outputs(nq: int, top_k: int) -> dict:
        k = max(int(top_k), 0)
        return dict(cand_frame=np.zeros((nq, k), np.int32), cand_score=np.zeros((nq, k), np.float32), cand_common=np.zeros((nq, k), np.int32),
                    **{n: np.zeros(nq, np.int32) for n in BOWDB_OUTPUTS[3:]})

    def query(self, q_lo: int, q_hi: int, top_k: int, exclude_window: int = 0, min_score: float = 0.0) -> dict:
        """loop candidates of frames q_lo .. q_hi - 1 (each excludes the frames within exclude_window of itself) -> dict of
        cand_frame / cand_score / cand_common [n][top_k] and n_sharing / max_common / n_scored / n_kept [n]"""
        out = self._outputs(max(int(q_hi) - int(q_lo), 0), top_k)
        self.query_ptr(q_lo, q_hi, top_k, exclude_window, min_score, [out[n].ctypes.data for n in BOWDB_OUTPUTS], on_device=False)
        return out

    def query_frame(self, frame: int = 0, top_k: int = 10, min_score: float = 0.0) -> dict:
        """relocalisation candidates of frame `frame` of the context's most recent call, whose bow_transform() with this
        database's vocabulary is resident; nothing is excluded.  -> the dict of query() with one row"""
        out = self._outputs(1, top_k)
        self.query_frame_ptr(frame, top_k, min_score, [out[n].ctypes.data for n in BOWDB_OUTPUTS], on_device=False)
        return out

    def close(self):
        if getattr(self, "_h", None):
            self._L.orbx_bowdb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


LOOPVER_OUTPUTS = ("n_bow", "n_matches", "n_corr", "n_iters", "hypothesis", "n_inliers", "accepted", "T", "match", "loop_frame")


class LoopVerifier:
    """Loop verification over the frames of a stereo sequence (orbx_loopver_*): ORB-SLAM2's LoopClosing::ComputeSim3 check --
    searchByBow between a query and each of its loop candidates, the rotation check, and a fixed-scale Horn RANSAC --
    for every (query, candidate) pair of a table such as BowDatabase.query's cand_frame, built once on a context's device."""

    @classmethod
    def build(cls, ctx: Context, vocab: Vocabulary, records, n_frames: int, levelsup: int = 4, record_stride: int | None = None) -> "LoopVerifier":
        """from the frames' records (the layout of ctx.record_dtype(), e.g. sequence_stereo's): a host array of n_frames
        records, or a device pointer (int) of ctx's device, which then needs record_stride when it is not record_bytes"""
        self = cls.__new__(cls)
        self._L, self.ctx, self.n_frames = ctx._L, ctx, int(n_frames)
        self._h = C.c_void_p()
        if isinstance(records, int):
            ptr, stride, on_device = records, int(record_stride or ctx.record_layout().record_bytes), 1
        else:
            rec = np.ascontiguousarray(records).view(np.uint8).reshape(len(records), -1)[: int(n_frames)]
            assert len(rec) == int(n_frames)
            ptr, stride, on_device = rec.ctypes.data, rec.shape[1], 0
        _check(ctx._h, self._L.orbx_loopver_build(ctx._h, vocab._h, int(levelsup), ptr, stride, int(n_frames), on_device, C.byref(self._h)),
               "orbx_loopver_build")
        return self

    @staticmethod
    def params(ratio=0.75, min_matches=20, min_inliers=20, max_iterations=300, probability=0.99, seed=0) -> OrbxLoopverParams:
        return OrbxLoopverParams(float(ratio), int(min_matches), int(min_inliers), int(max_iterations), float(probability), int(seed) & (2**64 - 1))

    def verify_ptr(self, q_lo: int, n_queries: int, cand_ptr: int, top_k: int, ptrs, on_device: bool = True, **params):
        """orbx_loopver_verify with a raw table pointer and raw output pointers in LOOPVER_OUTPUTS order (0 = not wanted)"""
        io = OrbxLoopverIO(int(on_device), cand_ptr or None, int(top_k), *[p or None for p in ptrs])
        prm = self.params(**params)
        _check(self.ctx._h, self._L.orbx_loopver_verify(self.ctx._h, self._h, int(q_lo), int(n_queries), C.byref(prm), C.byref(io)), "orbx_loopver_verify")

    def verify(self, q_lo: int, cand_frame, ratio=0.75, min_matches=20, min_inliers=20, max_iterations=300, probability=0.99, seed=0) -> dict:
        """verifies queries q_lo .. q_lo + len(cand_frame) - 1 against their rows of cand_frame ([n][top_k], -1 = empty slot)
        -> dict of n_bow / n_matches / n_corr / n_iters / hypothesis / n_inliers / accepted [n][top_k], T [n][top_k][12],
        match [n][top_k][n_features] and loop_frame [n]"""
        tab = np.ascontiguousarray(cand_frame, np.int32)
        assert tab.ndim == 2
        nq, k, N = tab.shape[0], tab.shape[1], self.ctx.n_features
        out = {n: np.zeros((nq, k), np.int32) for n in LOOPVER_OUTPUTS[:7]}
        out.update(T=np.zeros((nq, k, 12), np.float64), match=np.zeros((nq, k, N), np.int32), loop_frame=np.zeros(nq, np.int32))
        self.verify_ptr(q_lo, nq, tab.ctypes.data, k, [out[n].ctypes.data for n in LOOPVER_OUTPUTS], on_device=False, ratio=ratio,
                        min_matches=min_matches, min_inliers=min_inliers, max_iterations=max_iterations, probability=probability, seed=seed)
        return out

    def close(self):
        if getattr(self, "_h", None):
            self._L.orbx_loopver_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
