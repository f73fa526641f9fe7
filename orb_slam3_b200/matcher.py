"""Host-side mirror of ORB_SLAM3::ORBmatcher (include/ORBmatcher.h:43-76) for the
hot-path methods, over the C ABI.  Frames/KeyFrames/MapPoints are passed
as the flat views of views.py.  No CPU fallback."""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import check, ptr


class ORBmatcher:
    TH_HIGH = 100
    TH_LOW = 50
    HISTO_LENGTH = 30

    def __init__(self, nnratio=0.6, checkOri=True, device=0):
        self._lib = _lib.lib()
        self.mfNNratio = float(nnratio)
        self.mbCheckOrientation = bool(checkOri)
        h = C.c_void_p()
        check(self._lib.match_create(int(device), C.byref(h)))
        self._h = h

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._lib.match_destroy(h)
            self._h = None

    @staticmethod
    def DescriptorDistance(a, b):
        a = np.ascontiguousarray(a, np.uint8)
        b = np.ascontiguousarray(b, np.uint8)
        return _lib.lib().ham_distance(ptr(a), ptr(b))

    def SearchByProjection(self, F, vpMapPoints, th=3.0, bFarPoints=False, thFarPoints=50.0):
        """(nmatches, assign[F.n]) -- assign[i] = index into vpMapPoints or -1."""
        out = np.empty(F.n, np.int32)
        n = check(self._lib.match_project_local(self._h, C.byref(F), C.byref(vpMapPoints), float(th),
                                                self.mfNNratio, int(bFarPoints), float(thFarPoints), ptr(out)))
        return n, out

    def SearchByProjectionLast(self, CurrentFrame, LastFrame, Tcw_qt7, th, bForward=False, bBackward=False):
        """SearchByProjection(Frame& Cur, const Frame& Last, th, bMono): (nmatches, assign[Cur.n]);
        assign = last-frame keypoint index, -1 untouched, -2 cleared by the rotation check."""
        T = np.ascontiguousarray(Tcw_qt7, np.float32)
        out = np.empty(CurrentFrame.n, np.int32)
        n = check(self._lib.match_project_last(self._h, C.byref(CurrentFrame), C.byref(LastFrame), ptr(T),
                                               int(bForward), int(bBackward), float(th),
                                               int(self.mbCheckOrientation), ptr(out)))
        return n, out

    def SearchForTriangulation(self, KF1, KF2, fv1, fv2, F12, ep, bOnlyStereo=False, bCoarse=False, cap=None):
        cap = cap or max(KF1.n, 1)
        F12 = np.ascontiguousarray(F12, np.float32).reshape(9)
        ep = np.ascontiguousarray(ep, np.float32).reshape(2)
        out = np.empty((cap, 2), np.int32)
        n = check(self._lib.match_triangulate(self._h, C.byref(KF1), C.byref(KF2), C.byref(fv1), C.byref(fv2),
                                              ptr(F12), ptr(ep), int(bOnlyStereo), int(bCoarse),
                                              int(self.mbCheckOrientation), ptr(out), cap))
        return n, out[:n]

    def SearchByBoW(self, pKF, kf_mp_ok, fv_kf, F, fv_f):
        """SearchByBoW(KeyFrame* pKF, Frame& F, vpMapPointMatches): (nmatches, assign[F.n]); assign = KF keypoint
        index whose map point lands in vpMapPointMatches[i], -1 untouched, -2 cleared by the rotation check.
        kf_mp_ok[i] = the KF's map point i exists and is not bad."""
        ok = np.ascontiguousarray(kf_mp_ok, np.uint8)
        out = np.empty(F.n, np.int32)
        n = check(self._lib.match_bow_frame(self._h, C.byref(pKF), ptr(ok), C.byref(fv_kf), C.byref(F), C.byref(fv_f),
                                            self.mfNNratio, int(self.mbCheckOrientation), ptr(out)))
        return n, out

    def SearchByBoWKeyFrames(self, pKF1, mp_ok1, fv1, pKF2, mp_ok2, fv2):
        """SearchByBoW(KeyFrame* pKF1, KeyFrame* pKF2, vpMatches12): (nmatches, match12[pKF1.n]); match12 = KF2
        keypoint index, -1 untouched, -2 cleared by the rotation check."""
        ok1 = np.ascontiguousarray(mp_ok1, np.uint8)
        ok2 = np.ascontiguousarray(mp_ok2, np.uint8)
        out = np.empty(pKF1.n, np.int32)
        n = check(self._lib.match_bow_keyframes(self._h, C.byref(pKF1), ptr(ok1), C.byref(fv1), C.byref(pKF2), ptr(ok2),
                                                C.byref(fv2), self.mfNNratio, int(self.mbCheckOrientation), ptr(out)))
        return n, out

    # ---- batched submissions (independent problems)
    def project_last_batch(self, curs, lasts, Tcw, th, forward=None, backward=None, on_device=False,
                           assign_ptrs=None):
        B = len(curs)
        from .views import orb_frame_view, orb_lastframe_view
        ca = (orb_frame_view * B)(*curs)
        la = (orb_lastframe_view * B)(*lasts)
        T = np.ascontiguousarray(Tcw, np.float32).reshape(B, 7)
        fw = np.ascontiguousarray(np.zeros(B) if forward is None else forward, np.int32)
        bw = np.ascontiguousarray(np.zeros(B) if backward is None else backward, np.int32)
        res = np.zeros(B, np.int32)
        self._last_res = res  # must outlive an asynchronous batch
        if int(on_device) == 1:
            outs = None
            arr = (C.c_void_p * B)(*assign_ptrs)
        else:  # 0: host views; 2: only keys / u_right / desc of the frame views are device pointers
            outs = [np.empty(c.n, np.int32) for c in curs]
            arr = (C.c_void_p * B)(*[o.ctypes.data for o in outs])
        check(self._lib.match_project_last_batch(self._h, B, ca, la, ptr(T), ptr(fw), ptr(bw), float(th),
                                                 int(self.mbCheckOrientation), arr, ptr(res), int(on_device)))
        return res, outs

    def project_local_batch(self, frames, mps, th=3.0, bFarPoints=False, thFarPoints=50.0, on_device=False,
                            assign_ptrs=None):
        B = len(frames)
        from .views import orb_frame_view, orb_mappoint_view
        fa = (orb_frame_view * B)(*frames)
        ma = (orb_mappoint_view * B)(*mps)
        res = np.zeros(B, np.int32)
        self._last_res = res
        if int(on_device) == 1:
            outs = None
            arr = (C.c_void_p * B)(*assign_ptrs)
        else:
            outs = [np.empty(f.n, np.int32) for f in frames]
            arr = (C.c_void_p * B)(*[o.ctypes.data for o in outs])
        check(self._lib.match_project_local_batch(self._h, B, fa, ma, float(th), self.mfNNratio, int(bFarPoints),
                                                  float(thFarPoints), arr, ptr(res), int(on_device)))
        return res, outs

    def triangulate_batch(self, kf1s, kf2s, fv1s, fv2s, F12s, eps, bOnlyStereo=False, bCoarse=False, cap=4096):
        B = len(kf1s)
        from .views import orb_frame_view, orb_featvec_view
        a1 = (orb_frame_view * B)(*kf1s)
        a2 = (orb_frame_view * B)(*kf2s)
        f1 = (orb_featvec_view * B)(*fv1s)
        f2 = (orb_featvec_view * B)(*fv2s)
        F = np.ascontiguousarray(F12s, np.float32).reshape(B, 9)
        e = np.ascontiguousarray(eps, np.float32).reshape(B, 2)
        outs = [np.empty((cap, 2), np.int32) for _ in range(B)]
        arr = (C.c_void_p * B)(*[o.ctypes.data for o in outs])
        res = np.zeros(B, np.int32)
        check(self._lib.match_triangulate_batch(self._h, B, a1, a2, f1, f2, ptr(F), ptr(e), int(bOnlyStereo),
                                                int(bCoarse), int(self.mbCheckOrientation), arr, cap, ptr(res), 0))
        return res, [o[:r] for o, r in zip(outs, res)]

    def bow_frame_batch(self, kfs, kf_mp_oks, fv_kfs, frames, fv_fs, on_device=0, out_ptrs=None):
        """SearchByBoW(KeyFrame*, Frame&) for each (kfs[k], frames[k]).  on_device = 2: the frame views' keys / desc
        are an extractor's device results; 1: every array is device memory and out_ptrs are device outputs.
        Returns (nmatches[B], assign lists or None)."""
        from .views import orb_frame_view, orb_featvec_view
        B = len(kfs)
        oks = [np.ascontiguousarray(o, np.uint8) for o in kf_mp_oks] if int(on_device) != 1 else None
        ok_arr = (C.c_void_p * B)(*([o.ctypes.data for o in oks] if oks is not None else kf_mp_oks))
        res = np.zeros(B, np.int32)
        if int(on_device) == 1:
            outs = None
            arr = (C.c_void_p * B)(*out_ptrs)
        else:
            outs = [np.empty(f.n, np.int32) for f in frames]
            arr = (C.c_void_p * B)(*[o.ctypes.data for o in outs])
        check(self._lib.match_bow_frame_batch(self._h, B, (orb_frame_view * B)(*kfs), ok_arr,
                                              (orb_featvec_view * B)(*fv_kfs), (orb_frame_view * B)(*frames),
                                              (orb_featvec_view * B)(*fv_fs), self.mfNNratio,
                                              int(self.mbCheckOrientation), arr, ptr(res), int(on_device)))
        return res, outs

    def bow_keyframes_batch(self, kf1s, mp_ok1s, fv1s, kf2s, mp_ok2s, fv2s, on_device=0, out_ptrs=None):
        """SearchByBoW(KeyFrame*, KeyFrame*) for each pair.  Returns (nmatches[B], match12 lists or None)."""
        from .views import orb_frame_view, orb_featvec_view
        B = len(kf1s)
        dev = int(on_device) == 1
        keep = [] if dev else [np.ascontiguousarray(o, np.uint8) for o in list(mp_ok1s) + list(mp_ok2s)]
        p1 = list(mp_ok1s) if dev else [o.ctypes.data for o in keep[:B]]
        p2 = list(mp_ok2s) if dev else [o.ctypes.data for o in keep[B:]]
        res = np.zeros(B, np.int32)
        if dev:
            outs = None
            arr = (C.c_void_p * B)(*out_ptrs)
        else:
            outs = [np.empty(k.n, np.int32) for k in kf1s]
            arr = (C.c_void_p * B)(*[o.ctypes.data for o in outs])
        check(self._lib.match_bow_keyframes_batch(self._h, B, (orb_frame_view * B)(*kf1s), (C.c_void_p * B)(*p1),
                                                  (orb_featvec_view * B)(*fv1s), (orb_frame_view * B)(*kf2s),
                                                  (C.c_void_p * B)(*p2), (orb_featvec_view * B)(*fv2s), self.mfNNratio,
                                                  int(self.mbCheckOrientation), arr, ptr(res), int(on_device)))
        return res, outs

    def set_stream(self, cuda_stream):
        check(self._lib.match_set_stream(self._h, C.c_void_p(cuda_stream) if cuda_stream else None))

    def set_async(self, on):
        check(self._lib.match_set_async(self._h, int(on)))

    def synchronize(self):
        check(self._lib.match_synchronize(self._h))

    def last_ms(self):
        return float(self._lib.match_last_ms(self._h))

    def kernel_launches(self):
        return int(self._lib.match_kernel_launches(self._h))
