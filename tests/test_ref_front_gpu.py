"""CUDA path against the reference's own front-end object code (oracle/_ref/libref_front.so: ORBmatcher.cc, Frame.cc,
KeyFrame.cc, MapPoint.cc compiled unmodified, see tests/test_ref_front.py) -- no restatement in between: the matchers'
assignment / pair lists, isInFrustum's outputs and ComputeStereoMatches' mvuRight / mvDepth, through the C ABI.
Where oracle/_ref is absent the matchers, isInFrustum and ComputeStereoMatches are held to the committed results of the
same calls (tests/golden/ref_gpu.json); SearchForTriangulation takes F12 and the epipole from the reference and needs it."""
import numpy as np
import pytest

from orb_slam3_b200 import scenes
from orb_slam3_b200.synth import synth_frame, shifted_frame, stereo_right
from oracle import ref
from test_ref_parity import digest, recorded

pytestmark = pytest.mark.gpu
LIVE = ref.front_available()


@pytest.fixture(scope="module")
def feats(oracle):
    a = synth_frame(720, 1280, 41)
    b = shifted_frame(a, 5, -3, 42)
    ex = oracle.OracleExtractor(2000)
    ka, da, _ = ex.extract(a)
    kb, db, _ = ex.extract(b)
    return ka, da, kb, db


@pytest.fixture(scope="module")
def matcher():
    from orb_slam3_b200.matcher import ORBmatcher
    return ORBmatcher


@pytest.mark.parametrize("stereo", [False, True])
def test_search_local_points_cuda_is_the_reference(matcher, feats, stereo):
    ka, da, _, _ = feats
    for th, ratio, far in [(1.0, 0.8, False), (3.0, 0.8, True), (15.0, 0.9, False)]:
        F, mps = scenes.local_map_scene(ka, da, 1280, 720, 1000, seed=int(th) + 7 * stereo, stereo=stereo)
        n, a = matcher(ratio).SearchByProjection(F, mps, th, far, 40.0)
        if not LIVE:
            z = recorded("local_%d_%s_%d_%d" % (stereo, th, ratio * 10, far))
            assert (n, digest(a)) == (z["n"], z["assign"]), (th, ratio, far, n, z["n"])
            assert n > 50
            continue
        n_ref, a_ref = ref.front_project_local(F, mps, th, ratio, far, 40.0)
        assert n == n_ref and np.array_equal(a, a_ref), (th, ratio, far, n, n_ref)
        assert n_ref > 50


@pytest.mark.parametrize("stereo", [False, True])
def test_search_last_frame_cuda_is_the_reference(matcher, feats, stereo):
    ka, da, kb, db = feats
    cur, last, Tcw = scenes.last_frame_scene(ka, da, kb, db, 1280, 720, (5, -3), seed=3, stereo=stereo)
    for th in (7.0, 15.0):
        for (fw, bw) in ((0, 0), (1, 0), (0, 1)) if stereo else ((0, 0),):
            for ori in (True, False):
                n, a = matcher(0.9, ori).SearchByProjectionLast(cur, last, Tcw, th, fw, bw)
                # the reference leaves NULL where the rotation check cleared a match; the C ABI reports those as -2
                a = np.where(a < 0, -1, a)
                if not LIVE:
                    z = recorded("last_%d_%s_%d_%d_%d" % (stereo, th, fw, bw, ori))
                    assert (n, digest(a)) == (z["n"], z["assign"]), (th, fw, bw, ori, n, z["n"])
                    continue
                n_ref, a_ref = ref.front_project_last(cur, last, Tcw, th, fw, bw, ori)
                assert n == n_ref and np.array_equal(a, a_ref), (th, fw, bw, ori, n, n_ref)
    assert n > 50


@pytest.mark.skipif(not LIVE, reason="oracle/_ref/libref_front.so not built and the reference tree is absent")
def test_search_for_triangulation_cuda_is_the_reference(matcher, feats):
    ka, da, kb, db = feats
    T1 = np.array([0, 0, 0, 1, 0.3, -0.1, 0.2], np.float32)
    for stereo, dt in [(True, [-0.1, 0.06, -0.003]), (False, [-0.1, 0.06, -0.003]), (True, [0.05, 0.09, 0.004])]:
        k1, k2, fv1, fv2, _, _ = scenes.triangulation_scene(ka, da, kb, db, 1280, 720, seed=3, stereo=stereo)
        T2 = T1.copy()
        T2[4:] += np.array(dt, np.float32)
        for only_stereo in (False, True):
            for coarse in (False, True):
                for ori in (True, False):
                    n_ref, p_ref, F12, ep = ref.front_triangulate(k1, k2, fv1, fv2, T1, T2, only_stereo, coarse, ori)
                    n, p = matcher(0.6, ori).SearchForTriangulation(k1, k2, fv1, fv2, F12, ep, only_stereo, coarse)
                    assert n == n_ref and np.array_equal(p, p_ref), (stereo, dt, only_stereo, coarse, ori, n, n_ref)


@pytest.mark.parametrize("n,seed,cos_limit", [(3000, 0, 0.5), (50000, 1, 0.5), (20000, 3, 0.9)])
def test_is_in_frustum_cuda_is_the_reference(n, seed, cos_limit):
    from orb_slam3_b200.frustum import FrustumCuller
    v, _ = scenes.frustum_scene(n, seed=seed)
    n_got, got = FrustumCuller().isInFrustum(v, cos_limit)
    inside = got["track_in_view"] != 0
    fields = ("proj_x", "proj_y", "proj_xr", "scale_level", "view_cos", "depth")
    if not LIVE:
        z = recorded("frustum_%d_%d_%s" % (n, seed, cos_limit))
        assert (n_got, digest(got["track_in_view"])) == (z["n"], z["track_in_view"]) and n_got > n // 50
        assert [digest(got[k][inside]) for k in fields] == z["inside"]
        return
    n_ref, r = ref.front_is_in_frustum(v, cos_limit)
    assert n_got == n_ref and n_ref > n // 50
    assert np.array_equal(got["track_in_view"], r["track_in_view"])
    for k in fields:
        assert np.array_equal(got[k][inside], r[k][inside]), k


@pytest.mark.parametrize("h,w,nf,disp", [(480, 752, 1000, (12,)), (720, 1280, 2000, (5, 30, 17))])
def test_compute_stereo_matches_cuda_is_the_reference(oracle, h, w, nf, disp):
    from orb_slam3_b200.extractor import ORBextractor
    from orb_slam3_b200.stereo import StereoMatcher
    left = synth_frame(h, w, 9)
    right = stereo_right(left, 109, disparities=disp)
    el, er = oracle.OracleExtractor(nf), oracle.OracleExtractor(nf)   # inputs of the reference call: its own pyramid levels
    kl, dl, _ = el.extract(left)
    kr, dr, _ = er.extract(right)
    gl, gr, sm = ORBextractor(nf, 1.2, 8, 20, 7), ORBextractor(nf, 1.2, 8, 20, 7), StereoMatcher()
    _, gk, _ = gl(left)
    gr(right)
    assert np.array_equal(gk["x"], kl["x"]) and np.array_equal(gk["y"], kl["y"])
    n, ur, dp = sm.ComputeStereoMatches(gl, gr, len(gk), 386.0, 0.5514)
    if not LIVE:
        z = recorded("stereo_%d_%d_%d" % (h, w, nf))
        assert (n, digest(ur), digest(dp)) == (z["n"], z["u_right"], z["depth"]) and n > 100
        return
    n_ref, ur_ref, dp_ref = ref.front_stereo_match(kl, dl, kr, dr, [el.level_image(l) for l in range(8)],
                                                   [er.level_image(l) for l in range(8)], 386.0, 0.5514)
    assert n == n_ref and n > 100
    assert np.array_equal(ur, ur_ref) and np.array_equal(dp, dp_ref)
