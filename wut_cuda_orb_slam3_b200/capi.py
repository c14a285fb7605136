"""ctypes binding of liborbx.so (include/orbx.h).  No torch types cross this boundary: pointers and sizes only.

The library is built in-tree by `make -C wut_cuda_orb_slam3_b200/csrc` (see __graft_entry__.build()).  If it is
missing the import fails loudly — there is no Python/CPU fallback for any compute entry point.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(HERE, "liborbx.so")

KP_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"),
                     ("octave", "<i4"), ("class_id", "<i4")])
assert KP_DTYPE.itemsize == 28

ORBX_OK = 0
ORBX_ERR_EMPTY_IMAGE = -1
ORBX_ERR_INVALID_ARG = -2
ORBX_ERR_NO_DEVICE = -3
ORBX_ERR_CUDA = -4
ORBX_ERR_CAPACITY = -5
ORBX_ERR_UNSUPPORTED = -6
ORBX_ERR_OOM = -7

_vp, _sz, _i, _f = C.c_void_p, C.c_size_t, C.c_int, C.c_float
_i64, _u32 = C.c_int64, C.c_uint32

# name -> (restype, argtypes); every symbol declared in include/orbx.h
SIGNATURES = {
    "orbx_last_error": (C.c_char_p, []),
    "orbx_version": (_i, []),
    "orbx_device_count": (_i, []),
    "orbx_create": (_i, [_i, _f, _i, _i, _i, _i, _i, _i, _i, C.POINTER(_vp)]),
    "orbx_destroy": (None, [_vp]),
    "orbx_get_levels": (_i, [_vp]),
    "orbx_get_scale_factor": (_f, [_vp]),
    "orbx_get_tables": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "orbx_compute_tables": (_i, [_i, _f, _i, _vp, _vp, _vp, _vp, _vp]),
    "orbx_level_size": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "orbx_max_keypoints": (_i, [_vp]),
    "orbx_max_keypoints_for": (_i, [_vp, _i, _i]),
    "orbx_extract": (_i, [_vp, _vp, _i, _i, _sz, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "orbx_extract_color": (_i, [_vp, _vp, _i, _i, _sz, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "orbx_cvt_gray_device": (_i, [_i, _vp, _sz, _sz, _i, _i, _i, _i, _i, _vp, _sz, _sz, _vp]),
    "orbx_extract_batch": (_i, [_vp, _vp, _i, _i, _i, _sz, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "orbx_extract_batch_device": (_i, [_vp, _vp, _sz, _i, _i, _i, _sz, _i, _i, _vp, _vp, _i, _vp, _vp, _vp]),
    "orbx_sync": (_i, [_vp]),
    "orbx_get_pyramid_level": (_i, [_vp, _i, _i, _vp, _sz, _i]),
    "orbx_set_pyramid_mirror": (_i, [_vp, _i]),
    "orbx_get_pyramid_mirror": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "orbx_get_blurred_level": (_i, [_vp, _i, _i, _vp, _sz]),
    "orbx_get_candidates": (_i, [_vp, _i, _i, _vp, _vp, _vp, _i]),
    "orbx_get_level_keypoints": (_i, [_vp, _i, _i, _vp, _vp, _i]),
    "orbx_distribute_octree": (_i, [_i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _i, _vp]),
    "orbx_descriptor_distance": (_i, [_vp, _vp]),
    "orbx_knn2": (_i, [_i, _vp, _i, _vp, _i64, _vp, _vp]),
    "orbx_knn2_device": (_i, [_i, _vp, _i, _vp, _i64, C.c_int32, _vp, _vp, _vp]),
    "orbx_knn2_merge_device": (_i, [_i, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "orbx_ratio_test": (_i, [_vp, _i, _f, _i, _i, _vp]),
    "orbx_rotation_consistency": (_i, [_vp, _vp, _i, _vp]),
    "orbx_distinctive_descriptor": (_i, [_vp, _i, _vp]),
    "orbx_distinctive_descriptors": (_i, [_i, _vp, _vp, _i, _vp]),
    "orbx_serialize_matrix_u8": (_i64, [_i, _vp, _i, _i, _sz, _vp, _sz]),
    "orbx_deserialize_matrix_u8": (_i64, [_i, _vp, _sz, _vp, _vp, _vp, _sz, _sz]),
    "orbx_serialize_keypoints": (_i64, [_i, _vp, _i, _vp, _sz]),
    "orbx_deserialize_keypoints": (_i64, [_i, _vp, _sz, _vp, _vp, _i]),
    "orbx_stereo_match": (_i, [_vp, _i, _vp, _i, _vp, _vp, _i, _vp, _vp, _i, _f, _f, _vp, _vp]),
    "orbx_stereo_match_device": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _i, _f, _f, _vp, _vp, _vp]),
    "orbx_extract_stereo": (_i, [_vp, _vp, _vp, _vp, _i, _i, _sz, _vp, _vp, _vp, _vp, _vp, _vp, _i, _f, _f, _vp, _vp]),
    "orbx_extract_stereo_batch": (_i, [_vp, _vp, _vp, _i, _i, _i, _sz, _f, _f, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp]),
    "orbx_extract_stereo_batch_device": (_i, [_vp, _vp, _vp, _sz, _i, _i, _i, _sz, _f, _f, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "orbx_extract_rgbd": (_i, [_vp, _vp, _i, _i, _sz, _i, _i, _vp, _i, _sz, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "orbx_extract_rgbd_batch": (_i, [_vp, _vp, _vp, _i, _i, _i, _sz, _i, _sz, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "orbx_extract_rgbd_batch_device": (_i, [_vp, _vp, _sz, _sz, _vp, _sz, _sz, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "orbx_comm_unique_id": (_i, [_vp]),
    "orbx_comm_create": (_i, [_i, _i, _i, _vp, C.POINTER(_vp)]),
    "orbx_comm_from_nccl": (_i, [_i, _vp, _i, _i, C.POINTER(_vp)]),
    "orbx_comm_destroy": (None, [_vp]),
    "orbx_comm_info": (_i, [_vp, _vp, _vp, _vp]),
    "orbx_shard_rows": (None, [_i64, _i, _i, _vp, _vp]),
    "orbx_knn2_sharded": (_i, [_vp, _vp, _i, _vp, _i64, _i64, _vp, _vp, _vp]),
    "orbx_vocab_create": (_i, [_i, _i, _vp, _vp, _vp, _i, _i, _i, _i, C.POINTER(_vp)]),
    "orbx_vocab_load_text": (_i, [_i, C.c_char_p, C.POINTER(_vp)]),
    "orbx_vocab_destroy": (None, [_vp]),
    "orbx_vocab_info": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "orbx_bow_transform": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp]),
    "orbx_compute_bow": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "orbx_bow_score": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _i, C.POINTER(C.c_double)]),
    "orbx_search_by_bow": (_i, [_i, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _vp, _i, _f, _i, _vp, _vp, _vp]),
    "orbx_search_by_bow_batch": (_i, [_i, _i, _vp, _vp, _vp, _i, _vp, _i, _i, _vp, _f, _i, _vp, _vp]),
    "orbx_search_for_triangulation": (_i, [_i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _i,
                                           _i, _i, _vp, _vp]),
    "orbx_search_for_triangulation_batch": (_i, [_i, _vp, _vp, _vp, _vp, _i, _vp, _i, _vp, _i, _i, _vp, _vp]),
    "orbx_assign_features_to_grid": (_i, [_i, _vp, _vp, _vp]),
    "orbx_get_features_in_area": (_i, [_i, _vp, _f, _f, _f, _i, _i, _vp, _i, _vp]),
    "orbx_search_by_projection_map": (_i, [_i, _vp, _vp, _f, _i, _f, _f, _vp, _vp]),
    "orbx_search_by_projection_last": (_i, [_i, _vp, _f, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _i, _i, _i, _vp, _vp]),
    "orbx_search_by_projection_kf": (_i, [_i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _i, _i, _vp, _vp]),
    "orbx_search_for_initialization": (_i, [_i, _vp, _vp, _i, _vp, _vp, _i, _f, _i, _vp, _vp]),
    "orbx_fuse": (_i, [_i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _vp, _vp]),
    "orbx_search_by_projection_sim3": (_i, [_i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _f, _f, _vp, _vp]),
    "orbx_fuse_sim3": (_i, [_i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _f, _vp, _vp]),
    "orbx_projection_rounds": (_i, []),
    "orbx_undistort_keypoints": (_i, [_i, _vp, _i, _vp, _vp, _i, _vp, _vp]),
    "orbx_rectifier_create": (_i, [_i, _vp, _vp, _sz, _i, _i, C.POINTER(_vp)]),
    "orbx_resizer_create": (_i, [_i, _i, _i, _i, _i, C.POINTER(_vp)]),
    "orbx_rectifier_destroy": (None, [_vp]),
    "orbx_remap": (_i, [_vp, _vp, _i, _i, _sz, _vp, _sz]),
    "orbx_remap_device": (_i, [_vp, _vp, _i, _i, _sz, _sz, _i, _vp, _sz, _sz, _vp]),
    "orbx_profile_begin": (_i, [_vp]),
    "orbx_profile_end": (_i, [_vp, _vp, _vp]),
    "orbx_measure_popc_peak": (_i, [_i, C.POINTER(C.c_double)]),
    "orbx_launch_count": (_i64, []),
    "orbx_synth_image_host": (None, [_u32, _i, _i, _i, _i, _vp, _sz]),
    "orbx_synth_images_device": (_i, [_i, _u32, _i, _i, _i, _i, _i, _vp, _sz, _sz, _vp]),
    "orbx_synth_descriptors_host": (None, [_u32, _i, _i64, _i64, _i64, _i, _vp]),
    "orbx_synth_descriptors_device": (_i, [_i, _u32, _i, _i64, _i64, _i64, _i, _vp, _vp]),
}


class FeatureVectorC(C.Structure):
    """orbx_feature_vector (include/orbx.h): a DBoW2::FeatureVector in CSR form."""
    _fields_ = [("n_nodes", C.c_int), ("node_ids", _vp), ("offsets", _vp), ("indices", _vp)]


class BowViewC(C.Structure):
    """orbx_bow_view (include/orbx.h): one key frame of orbx_search_by_bow_batch."""
    _fields_ = [("n", C.c_int), ("desc", _vp), ("angle", _vp), ("valid", _vp), ("fv", FeatureVectorC)]


class TriangulationViewC(C.Structure):
    """orbx_triangulation_view (include/orbx.h): one neighbour of orbx_search_for_triangulation_batch."""
    _fields_ = [("n", C.c_int), ("kp", _vp), ("desc", _vp), ("free", _vp), ("stereo", _vp), ("fv", FeatureVectorC),
                ("F12", _f * 9), ("ep", _f * 2), ("scale", _vp), ("sigma2", _vp), ("n_levels", C.c_int), ("coarse", C.c_int)]


class FrameViewC(C.Structure):
    """orbx_frame_view (include/orbx.h): the slice of ORB_SLAM3::Frame the projection searches read."""
    _fields_ = [("n", C.c_int), ("keys_un", _vp), ("descriptors", _vp), ("u_right", _vp), ("occupied", _vp),
                ("min_x", _f), ("min_y", _f), ("max_x", _f), ("max_y", _f), ("grid_w_inv", _f), ("grid_h_inv", _f),
                ("scale_factors", _vp), ("n_levels", C.c_int)]


class KeyFrameViewC(C.Structure):
    """orbx_keyframe_view (include/orbx.h): a frame view plus mvInvLevelSigma2 and mbf, what ORBmatcher::Fuse reads."""
    _fields_ = [("frame", FrameViewC), ("inv_level_sigma2", _vp), ("bf", _f)]


class TrackPointsC(C.Structure):
    """orbx_track_points (include/orbx.h)."""
    _fields_ = [("n", C.c_int), ("in_view", _vp), ("bad", _vp), ("proj_x", _vp), ("proj_y", _vp), ("proj_xr", _vp),
                ("view_cos", _vp), ("track_depth", _vp), ("scale_level", _vp), ("n_obs", _vp), ("descriptors", _vp)]


class RgbdCalibC(C.Structure):
    """orbx_rgbd_calib (include/orbx.h): mK, mDistCoef, mbf and Tracking::mDepthMapFactor."""
    _fields_ = [("K", _f * 4), ("dist", _vp), ("n_dist", C.c_int), ("bf", _f), ("depth_factor", _f)]


class OrbxError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("orbx error %d: %s" % (code, message))
        self.code = code


_lib = None


def lib():
    """Load liborbx.so (once).  Raises if the CUDA extension has not been built: no fallback exists."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ImportError("liborbx.so not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(nvcc, sm_100a).  The ORB front end has no CPU fallback.")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)          # AttributeError here = header and library disagree
            fn.restype = res
            fn.argtypes = args
        L.orbx_debug_sort_replay.restype = None
        L.orbx_debug_sort_replay.argtypes = [_vp, _i]
        L.orbx_debug_sort_replay32.restype = None
        L.orbx_debug_sort_replay32.argtypes = [_vp, _i]
        for nm in ("orbx_debug_sort_replay_ranges", "orbx_debug_sort_replay_ranges32"):
            getattr(L, nm).restype = None
            getattr(L, nm).argtypes = [_vp, _i]
        _lib = L
    return _lib


def check(rc):
    if rc != ORBX_OK:
        raise OrbxError(rc, lib().orbx_last_error().decode("utf-8", "replace"))
    return rc


def ptr(a):
    """Raw address of a numpy array / torch tensor / int."""
    if a is None:
        return None
    if isinstance(a, int):
        return _vp(a)
    if isinstance(a, np.ndarray):
        return _vp(a.ctypes.data)
    if hasattr(a, "data_ptr"):
        return _vp(a.data_ptr())
    raise TypeError(type(a))
