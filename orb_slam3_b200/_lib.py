"""ctypes loader for liborbb200.so.  Fails loudly: there is no Python/CPU
fallback for any compute entry point."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liborbb200.so")

KP_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"),
                     ("response", "<f4"), ("octave", "<i4"), ("class_id", "<i4")])

ORB_E = {-1: "ORB_E_EMPTY", -2: "ORB_E_ARG", -3: "ORB_E_CUDA", -4: "ORB_E_CAPACITY",
         -5: "ORB_E_NODEVICE", -6: "ORB_E_NCCL"}


class OrbError(RuntimeError):
    def __init__(self, rc, msg):
        super().__init__("%s (%d): %s" % (ORB_E.get(rc, "ORB_E_?"), rc, msg))
        self.rc = rc


_lib = None

# name -> (restype, argtypes); every symbol include/orb_b200.h declares
_vp, _i, _f, _sz = C.c_void_p, C.c_int, C.c_float, C.c_size_t
SIGNATURES = {
    "orb_version": (C.c_char_p, []),
    "orb_last_error": (C.c_char_p, []),
    "orb_device_count": (_i, []),
    "orb_create": (_i, [_i, _f, _i, _i, _i, _i, C.POINTER(_vp)]),
    "orb_destroy": (None, [_vp]),
    "orb_get_levels": (_i, [_vp]),
    "orb_get_scale_factor": (_f, [_vp]),
    "orb_get_scale_factors": (_i, [_vp, _vp]),
    "orb_get_inverse_scale_factors": (_i, [_vp, _vp]),
    "orb_get_scale_sigma_squares": (_i, [_vp, _vp]),
    "orb_get_inverse_scale_sigma_squares": (_i, [_vp, _vp]),
    "orb_get_features_per_level": (_i, [_vp, _vp]),
    "orb_extract": (_i, [_vp, _vp, _i, _i, _sz, _i, _i, _vp, _vp, _i, C.POINTER(_i)]),
    "orb_extract_batch": (_i, [_vp, _i, _vp, _i, _i, _sz, _vp, _vp, _vp, _i, _vp, _vp]),
    "orb_extract_batch_device": (_i, [_vp, _i, _vp, _sz, _i, _i, _sz, _vp, _vp]),
    "orb_device_results": (_i, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp),
                                C.POINTER(_i)]),
    "orb_download_results": (_i, [_vp, _i, _vp, _vp, _i, C.POINTER(_i)]),
    "orb_synchronize": (_i, [_vp]),
    "orb_pyramid": (_i, [_vp, _i, _i, C.POINTER(_vp), C.POINTER(_i), C.POINTER(_i), C.POINTER(_sz)]),
    "ham_distance": (_i, [_vp, _vp]),
    "match_create": (_i, [_i, C.POINTER(_vp)]),
    "match_destroy": (None, [_vp]),
    "match_project_local": (_i, [_vp, _vp, _vp, _f, _f, _i, _f, _vp]),
    "match_project_last": (_i, [_vp, _vp, _vp, _vp, _i, _i, _f, _i, _vp]),
    "match_triangulate": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _i]),
    "match_project_last_batch": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _f, _i, _vp, _vp, _i]),
    "match_project_local_batch": (_i, [_vp, _i, _vp, _vp, _f, _f, _i, _f, _vp, _vp, _i]),
    "match_triangulate_batch": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _i, _vp, _i]),
    "match_bow_frame": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _f, _i, _vp]),
    "match_bow_keyframes": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _i, _vp]),
    "match_bow_frame_batch": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _f, _i, _vp, _vp, _i]),
    "match_bow_keyframes_batch": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _f, _i, _vp, _vp, _i]),
    "match_set_stream": (_i, [_vp, _vp]),
    "match_set_async": (_i, [_vp, _i]),
    "match_synchronize": (_i, [_vp]),
    "match_kernel_launches": (C.c_longlong, [_vp]),
    "match_last_ms": (C.c_double, [_vp]),
    "lba_create": (_i, [_i, C.POINTER(_vp)]),
    "lba_destroy": (None, [_vp]),
    "lba_nccl_unique_id": (_i, [_vp]),
    "lba_comm_init": (_i, [_vp, _i, _i, _vp]),
    "lba_solve": (_i, [_vp, _vp, _vp, _i, C.c_double, _vp, _vp, _vp, _vp, _vp]),
    "lba_kernel_launches": (C.c_longlong, [_vp]),
    "lba_measure_fp64_mma_peak": (_i, [_i, _i, _vp]),
    "lba_debug_two_sided_plan": (_i, [_i, _vp, _vp, _vp, _vp]),
    "stereo_create": (_i, [_i, _vp]),
    "stereo_destroy": (None, [_vp]),
    "stereo_match": (_i, [_vp, _vp, _vp, C.c_float, C.c_float, _vp, _vp, _i]),
    "stereo_match_batch": (_i, [_vp, _vp, _vp, _i, C.c_float, C.c_float, _vp, _vp, _i, _vp, _i, _vp]),
    "stereo_device_results": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "stereo_kernel_launches": (C.c_longlong, [_vp]),
    "stereo_last_ms": (C.c_float, [_vp]),
    "poseopt_create": (_i, [_i, _vp]),
    "poseopt_destroy": (None, [_vp]),
    "pose_optimize": (_i, [_vp, _vp, _vp, _vp]),
    "pose_optimize_batch": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "poseopt_kernel_launches": (C.c_longlong, [_vp]),
    "poseopt_last_ms": (C.c_float, [_vp]),
    "frustum_create": (_i, [_i, _vp]),
    "frustum_destroy": (None, [_vp]),
    "frame_is_in_frustum": (_i, [_vp, _vp, C.c_float, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "frame_is_in_frustum_device": (_i, [_vp, _vp, C.c_float, _vp]),
    "frustum_device_results": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "frustum_kernel_launches": (C.c_longlong, [_vp]),
    "frustum_last_ms": (C.c_float, [_vp]),
    "frustum_debug_host": (_i, [_vp, C.c_float, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "vocab_create": (_i, [_i, _vp, _vp]),
    "vocab_destroy": (None, [_vp]),
    "bow_transform": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i]),
    "bow_transform_extracted": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i]),
    "bow_kernel_launches": (C.c_longlong, [_vp]),
    "bow_last_ms": (C.c_float, [_vp]),
    "bow_debug_host": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i]),
    "lia_create": (_i, [_i, _vp]),
    "lia_destroy": (None, [_vp]),
    "lia_solve": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "lia_kernel_launches": (C.c_longlong, [_vp]),
    "lia_last_ms": (C.c_float, [_vp]),
    "lia_debug_host": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "orb_set_profiling": (_i, [_vp, _i]),
    "orb_stage_times": (_i, [_vp, _vp, _vp, _i]),
    "orb_stage_name": (C.c_char_p, [_i]),
    "orb_kernel_launches": (C.c_longlong, [_vp]),
    "orb_debug_candidates": (_i, [_vp, _i, _i, _vp, _i]),
    "orb_debug_octree_host": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _vp, _i]),
    "orb_debug_introsort": (_i, [_vp, _vp, _i, _vp]),
    "orb_debug_introsort_levels": (_i, [_vp, _vp, _i, _vp]),
    "orb_debug_sincos_device": (_i, [_i, _vp, _sz, _vp, _vp]),
    "orb_debug_sincos_host": (_i, [_vp, _sz, _vp, _vp, _i]),
}


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "%s is missing: build it with `python -m orb_slam3_b200.build` "
                "(nvcc, sm_100a). orb_slam3_b200 has no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the ABI lost a symbol
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc < 0:
        raise OrbError(rc, lib().orb_last_error().decode())
    return rc


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)
