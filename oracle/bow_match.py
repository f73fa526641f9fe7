"""ctypes bindings for SearchByBoW (TEST INFRASTRUCTURE ONLY): the oracle's restatement (orc_bow_match.cpp, part of
liborb_oracle.so) and the reference's own object code (oracle/_ref/libref_front_bow.so, built by ref_front_bow.mk where
the reference tree exists).  The views are the ctypes structs of orb_slam3_b200/views.py (interface types)."""
import ctypes as C
import os
import subprocess

import numpy as np

from . import oracle as _o
from . import ref as _ref

_HERE = os.path.dirname(os.path.abspath(__file__))
REF_LIB_PATH = os.path.join(_HERE, "_ref", "libref_front_bow.so")
_vp = C.c_void_p


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _oracle():
    L = _o.lib()
    L.orc_match_bow_frame.argtypes = [_vp] * 5 + [C.c_float, C.c_int, _vp]
    L.orc_match_bow_keyframes.argtypes = [_vp] * 6 + [C.c_float, C.c_int, _vp]
    return L


def match_bow_frame(kf, kf_mp_ok, fv_kf, F, fv_f, nn_ratio, check_ori=True):
    """ORBmatcher(nn_ratio, check_ori).SearchByBoW(KeyFrame*, Frame&, ...): (nmatches, assign[F.n]); assign = KF
    keypoint index, -1 untouched, -2 cleared by the rotation check."""
    ok = np.ascontiguousarray(kf_mp_ok, np.uint8)
    out = np.empty(F.n, np.int32)
    n = _oracle().orc_match_bow_frame(C.byref(kf), _p(ok), C.byref(fv_kf), C.byref(F), C.byref(fv_f), nn_ratio,
                                      int(check_ori), _p(out))
    return n, out


def match_bow_keyframes(kf1, mp_ok1, fv1, kf2, mp_ok2, fv2, nn_ratio, check_ori=True):
    """ORBmatcher(nn_ratio, check_ori).SearchByBoW(KeyFrame*, KeyFrame*, ...): (nmatches, match12[kf1.n])."""
    ok1 = np.ascontiguousarray(mp_ok1, np.uint8)
    ok2 = np.ascontiguousarray(mp_ok2, np.uint8)
    out = np.empty(kf1.n, np.int32)
    n = _oracle().orc_match_bow_keyframes(C.byref(kf1), _p(ok1), C.byref(fv1), C.byref(kf2), _p(ok2), C.byref(fv2),
                                          nn_ratio, int(check_ori), _p(out))
    return n, out


# ---- the reference's own SearchByBoW
_ref_lib = None


def build_ref(force=False):
    """Build oracle/_ref/libref_front_bow.so; None where the reference tree is absent."""
    if not os.path.exists(os.path.join(_ref.REFERENCE, "src", "ORBmatcher.cc")):
        return None
    _o.build()
    cmd = ["make", "-C", _HERE, "-f", "ref_front_bow.mk", "REF=" + _ref.REFERENCE] + (["-B"] if force else []) + \
        ["_ref/libref_front_bow.so"]
    subprocess.check_call(cmd, stdout=subprocess.DEVNULL)
    return REF_LIB_PATH


def ref_available():
    return os.path.exists(REF_LIB_PATH) or build_ref() is not None


def ref_lib():
    global _ref_lib
    if _ref_lib is None:
        if not os.path.exists(REF_LIB_PATH) and build_ref() is None:
            raise FileNotFoundError("oracle/_ref/libref_front_bow.so is not built and %s is absent" % _ref.REFERENCE)
        _o.lib()
        L = C.CDLL(REF_LIB_PATH)
        L.ref_front_bow_frame.argtypes = [_vp] * 5 + [C.c_float, C.c_int, _vp]
        L.ref_front_bow_keyframes.argtypes = [_vp] * 6 + [C.c_float, C.c_int, _vp]
        _ref_lib = L
    return _ref_lib


def ref_bow_frame(kf, kf_mp_ok, fv_kf, F, fv_f, nn_ratio, check_ori=True):
    """The reference's ORBmatcher(nn_ratio, check_ori).SearchByBoW(KeyFrame*, Frame&, ...): (n, assign[F.n]), -1 where
    the vector holds NULL (never matched, or cleared by the rotation check)."""
    ok = np.ascontiguousarray(kf_mp_ok, np.uint8)
    out = np.empty(F.n, np.int32)
    n = ref_lib().ref_front_bow_frame(C.byref(kf), _p(ok), C.byref(fv_kf), C.byref(F), C.byref(fv_f), nn_ratio,
                                      int(check_ori), _p(out))
    return n, out


def ref_bow_keyframes(kf1, mp_ok1, fv1, kf2, mp_ok2, fv2, nn_ratio, check_ori=True):
    """The reference's ORBmatcher(nn_ratio, check_ori).SearchByBoW(KeyFrame*, KeyFrame*, ...): (n, match12[kf1.n])."""
    ok1 = np.ascontiguousarray(mp_ok1, np.uint8)
    ok2 = np.ascontiguousarray(mp_ok2, np.uint8)
    out = np.empty(kf1.n, np.int32)
    n = ref_lib().ref_front_bow_keyframes(C.byref(kf1), _p(ok1), C.byref(fv1), C.byref(kf2), _p(ok2), C.byref(fv2),
                                          nn_ratio, int(check_ori), _p(out))
    return n, out
