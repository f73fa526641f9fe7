"""ORBmatcher::SearchByBoW, both overloads: the oracle (oracle/orc_bow_match.cpp) against a slow Python restatement of the
reference's loops, and the argument checks of the C ABI, which reject malformed input before any device work."""
import ctypes as C
import math

import numpy as np
import pytest

from oracle import bow_match as orc
from orb_slam3_b200 import scenes
from orb_slam3_b200.views import make_featvec_view, make_frame_view

TH_LOW, HISTO_LENGTH = 50, 30
POPC = np.array([bin(i).count("1") for i in range(256)], np.int32)


def ham(a, b):
    """Hamming distances between the rows of a (m, 32) and b (k, 32)."""
    return POPC[a[:, None, :] ^ b[None, :, :]].sum(-1)


def three_maxima(sizes):
    """ORBmatcher::ComputeThreeMaxima (ORBmatcher.cc:2012-2053)."""
    m1 = m2 = m3 = 0
    i1 = i2 = i3 = -1
    for i, s in enumerate(sizes):
        if s > m1:
            m3, m2, m1, i3, i2, i1 = m2, m1, s, i2, i1, i
        elif s > m2:
            m3, m2, i3, i2 = m2, s, i2, i
        elif s > m3:
            m3, i3 = s, i
    if np.float32(m2) < np.float32(0.1) * np.float32(m1):
        i2 = i3 = -1
    elif np.float32(m3) < np.float32(0.1) * np.float32(m1):
        i3 = -1
    return i1, i2, i3


def rot_bin(a1, a2):
    rot = np.float32(a1) - np.float32(a2)
    if rot < 0:
        rot = np.float32(rot + np.float32(360.0))
    b = int(math.floor(float(np.float32(rot * np.float32(1.0 / HISTO_LENGTH))) + 0.5))  # std::round, rot >= 0
    return 0 if b == HISTO_LENGTH else b


def py_search_by_bow(kind, q, okq, fvq, c, okc, fvc, ratio, check_ori):
    """kind 0: SearchByBoW(KeyFrame* = q, Frame& = c); kind 1: SearchByBoW(KeyFrame* = q, KeyFrame* = c)."""
    kq, dq, kc, dc = q._keep[0], q._keep[1], c._keep[0], c._keep[1]
    fq, fc = fvq._keep, fvc._keep
    out = -np.ones(c.n if kind == 0 else q.n, np.int32)
    taken = np.zeros(c.n, bool)
    hist = [[] for _ in range(HISTO_LENGTH)]
    nm = 0
    where_c = {int(nid): k for k, nid in enumerate(fc["node_ids"])}
    for a, nid in enumerate(fq["node_ids"]):        # ascending node ids: the merge walk visits the shared ones
        b = where_c.get(int(nid))
        if b is None:
            continue
        Q = fq["idx"][fq["ptr"][a]:fq["ptr"][a + 1]]
        Cn = fc["idx"][fc["ptr"][b]:fc["ptr"][b + 1]]
        D = ham(dq[Q], dc[Cn]) if len(Q) and len(Cn) else np.zeros((len(Q), len(Cn)), np.int32)
        for qi, i1 in enumerate(Q):
            if not okq[i1]:
                continue
            alive = ~taken[Cn] if kind == 0 else (~taken[Cn] & (okc[Cn] != 0))
            d = np.where(alive, D[qi], 1 << 20)
            best, second, j = 256, 256, -1
            if alive.any():
                j = int(np.argmin(d))                     # first position with the minimum
                best = int(d[j])
                srt = np.sort(D[qi][alive])
                second = int(srt[1]) if len(srt) > 1 else 256
            passed = best <= TH_LOW if kind == 0 else best < TH_LOW
            if passed and np.float32(best) < np.float32(ratio) * np.float32(second):
                i2 = int(Cn[j])
                taken[i2] = True
                rec = i2 if kind == 0 else int(i1)
                out[rec] = int(i1) if kind == 0 else i2
                if check_ori:
                    hist[rot_bin(kq["angle"][i1], kc["angle"][i2])].append(rec)
                nm += 1
    if check_ori:
        keep = three_maxima([len(h) for h in hist])
        for i, h in enumerate(hist):
            if i not in keep:
                for rec in h:
                    out[rec] = -2
                    nm -= 1
    return nm, out


def run_both(oracle, kind, s, ratio, ori):
    if kind == 0:
        got = orc.match_bow_frame(s["kf1"], s["ok1"], s["fv1"], s["kf2"], s["fv2"], ratio, ori)
        ref = py_search_by_bow(0, s["kf1"], s["ok1"], s["fv1"], s["kf2"], None, s["fv2"], ratio, ori)
    else:
        got = orc.match_bow_keyframes(s["kf1"], s["ok1"], s["fv1"], s["kf2"], s["ok2"], s["fv2"], ratio, ori)
        ref = py_search_by_bow(1, s["kf1"], s["ok1"], s["fv1"], s["kf2"], s["ok2"], s["fv2"], ratio, ori)
    return got, ref


@pytest.fixture(scope="module")
def node_fns(oracle):
    voc = scenes.synth_vocabulary(10, 4, seed=5)

    def by_vocab(levelsup):
        def f(desc):
            r = oracle.bow_transform(voc, desc, levelsup)
            return scenes.nodes_from_featvec(len(desc), r["fv_node_ids"], r["fv_ptr"], r["fv_idx"])
        return f
    # depth-2 nodes (as ORBvoc, k = 10, L = 6, with levelsup = 4), one root node (levelsup = L), 1000 hash buckets
    return {"depth2": by_vocab(2), "root": by_vocab(4), "hash1000": lambda d: scenes.hash_nodes(d, 1000)}


@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("nodes", ["depth2", "root", "hash1000"])
@pytest.mark.parametrize("kind", [0, 1])
def test_oracle_equals_python_restatement(oracle, node_fns, seed, nodes, kind):
    s = scenes.bow_match_scene(400, seed, node_fns[nodes])
    total = 0
    for ratio in (0.7, 0.75, 0.9):
        for ori in (True, False):
            (n, out), (n_ref, out_ref) = run_both(oracle, kind, s, ratio, ori)
            assert n == n_ref and np.array_equal(out, out_ref), (ratio, ori, n, n_ref)
            assert n == int((out >= 0).sum())
            total += n
            if ori:
                assert (out == -2).any() or nodes == "hash1000", "the rotation check cleared nothing"
    assert total > 100


# ---- targeted cases: one node, hand-made distances
def _desc_at(base, dist, rng):
    """A descriptor at Hamming distance `dist` from base."""
    bits = np.unpackbits(base)
    bits[rng.choice(256, dist, replace=False)] ^= 1
    return np.packbits(bits)


def case(q_desc, c_desc, q_angle=None, c_angle=None, okq=None, okc=None, q_nodes=None, c_nodes=None):
    q_desc, c_desc = np.asarray(q_desc, np.uint8), np.asarray(c_desc, np.uint8)
    nq, nc = len(q_desc), len(c_desc)
    sf = scenes.scale_factors()

    def kp(n, ang):
        from orb_slam3_b200._lib import KP_DTYPE
        k = np.zeros(n, KP_DTYPE)
        k["x"], k["y"] = 100.0, 100.0
        k["angle"] = 0.0 if ang is None else ang
        return k
    return dict(kf1=make_frame_view(kp(nq, q_angle), q_desc.reshape(nq, 32), 640, 480, sf),
                kf2=make_frame_view(kp(nc, c_angle), c_desc.reshape(nc, 32), 640, 480, sf),
                ok1=np.ones(nq, np.uint8) if okq is None else np.asarray(okq, np.uint8),
                ok2=np.ones(nc, np.uint8) if okc is None else np.asarray(okc, np.uint8),
                fv1=make_featvec_view(np.zeros(nq) if q_nodes is None else q_nodes),
                fv2=make_featvec_view(np.zeros(nc) if c_nodes is None else c_nodes))


def check_case(oracle, kind, s, ratio, ori, expect_n, expect_out):
    (n, out), (n_ref, out_ref) = run_both(oracle, kind, s, ratio, ori)
    assert (n_ref, out_ref.tolist()) == (expect_n, list(expect_out))
    assert (n, out.tolist()) == (expect_n, list(expect_out))


def test_threshold_is_le_for_frames_and_lt_for_keyframes(oracle):
    rng = np.random.default_rng(0)
    q = rng.integers(0, 256, 32, dtype=np.uint8)
    s = case([q], [_desc_at(q, 50, rng), _desc_at(q, 100, rng)])
    check_case(oracle, 0, s, 0.9, False, 1, [0, -1])      # bestDist1 <= TH_LOW
    check_case(oracle, 1, s, 0.9, False, 0, [-1])         # bestDist1 < TH_LOW
    s = case([q], [_desc_at(q, 49, rng), _desc_at(q, 100, rng)])
    check_case(oracle, 1, s, 0.9, False, 1, [0])


def test_ratio_is_strict(oracle):
    rng = np.random.default_rng(1)
    q = rng.integers(0, 256, 32, dtype=np.uint8)
    s = case([q], [_desc_at(q, 40, rng), _desc_at(q, 30, rng)])   # 30 < 0.75 * 40 = 30.0 is false
    for kind in (0, 1):
        check_case(oracle, kind, s, 0.75, False, 0, [-1] * (2 if kind == 0 else 1))
    s = case([q], [_desc_at(q, 40, rng), _desc_at(q, 29, rng)])
    check_case(oracle, 0, s, 0.75, False, 1, [-1, 0])
    check_case(oracle, 1, s, 0.75, False, 1, [1])


def test_ties_at_the_minimum(oracle):
    rng = np.random.default_rng(2)
    q = rng.integers(0, 256, 32, dtype=np.uint8)
    s = case([q], [_desc_at(q, 20, rng), _desc_at(q, 10, rng), _desc_at(q, 10, rng)])
    check_case(oracle, 0, s, 0.9, False, 0, [-1, -1, -1])   # bestDist2 == bestDist1: no ratio below 1 passes
    check_case(oracle, 0, s, 1.5, False, 1, [-1, 0, -1])    # ... above 1 the FIRST candidate at the minimum wins
    check_case(oracle, 1, s, 1.5, False, 1, [1])


def test_rotation_bins_near_360_and_bin_30(oracle):
    rng = np.random.default_rng(3)
    # ten queries, each with its own node and one candidate at distance 5; rotations (query - candidate angle):
    # 1 x 0 deg and 3 x 900 deg -> bin 0 (900 / 30 = 30 -> 0), 3 x 359.5 deg -> bin 12 (the 1/30 quirk),
    # 2 x 240 deg -> bin 8, 1 x 300 deg -> bin 10: the three maxima are bins 0, 12, 8 and bin 10 is cleared
    rot = np.array([0, 900, 900, 900, 359.5, 359.5, 359.5, 240, 240, 300], np.float32)
    q = rng.integers(0, 256, (10, 32), dtype=np.uint8)
    c = np.stack([_desc_at(x, 5, rng) for x in q])
    s = case(q, c, q_angle=rot, c_angle=np.zeros(10), q_nodes=np.arange(10), c_nodes=np.arange(10))
    for kind in (0, 1):
        check_case(oracle, kind, s, 0.9, True, 9, list(range(9)) + [-2])
        check_case(oracle, kind, s, 0.9, False, 10, list(range(10)))
    assert rot_bin(359.5, 0) == 12 and rot_bin(900, 0) == 0


def test_empty_and_degenerate(oracle):
    rng = np.random.default_rng(4)
    q = rng.integers(0, 256, (3, 32), dtype=np.uint8)
    c = np.stack([_desc_at(x, 3, rng) for x in q])
    for kind in (0, 1):
        n_out = 3
        # empty FeatureVectors, disjoint node ids
        check_case(oracle, kind, case(q, c, q_nodes=-np.ones(3), c_nodes=np.zeros(3)), 0.9, True, 0, [-1] * n_out)
        check_case(oracle, kind, case(q, c, q_nodes=np.arange(3), c_nodes=np.arange(3) + 3), 0.9, True, 0, [-1] * n_out)
        # no valid map point on the query side
        check_case(oracle, kind, case(q, c, okq=np.zeros(3)), 0.9, True, 0, [-1] * n_out)
        # nodes shared, one match each
        check_case(oracle, kind, case(q, c, q_nodes=np.arange(3), c_nodes=np.arange(3)), 0.9, True, 3, [0, 1, 2])
    # keyframe-keyframe: no candidate has a valid map point
    check_case(oracle, 1, case(q, c, okc=np.zeros(3)), 0.9, True, 0, [-1] * 3)
    # every candidate taken: three identical queries, one candidate -- the first query takes it
    s = case(np.stack([q[0]] * 3), c[:1])
    check_case(oracle, 0, s, 0.9, True, 1, [0])
    check_case(oracle, 1, s, 0.9, True, 1, [0, -1, -1])
    # no keypoints at all
    e = case(np.zeros((0, 32)), np.zeros((0, 32)))
    check_case(oracle, 0, e, 0.9, True, 0, [])
    check_case(oracle, 1, e, 0.9, True, 0, [])


# ---- the C ABI rejects bad arguments before it looks for a device
def _fv(ids, ptr, idx):
    from orb_slam3_b200.views import orb_featvec_view
    a = dict(node_ids=np.asarray(ids, np.uint32), ptr=np.asarray(ptr, np.int32), idx=np.asarray(idx, np.int32))
    v = orb_featvec_view()
    v.n_nodes = len(ids)
    v.node_ids, v.ptr, v.idx = a["node_ids"].ctypes.data, a["ptr"].ctypes.data, a["idx"].ctypes.data
    v._keep = a
    return v


MALFORMED = {
    "index >= n": _fv([1, 2], [0, 2, 3], [0, 1, 4]),
    "negative index": _fv([1], [0, 1], [-1]),
    "index twice in one node": _fv([1], [0, 2], [1, 1]),
    "index in two nodes": _fv([1, 2], [0, 1, 2], [1, 1]),
    "node ids not ascending": _fv([2, 1], [0, 1, 2], [0, 1]),
    "repeated node id": _fv([1, 1], [0, 1, 2], [0, 1]),
    "ptr decreasing": _fv([1, 2], [0, 2, 1], [0, 1]),
    "negative n_nodes": _fv([], [0], []),
}
MALFORMED["negative n_nodes"].n_nodes = -1


@pytest.mark.parametrize("what", sorted(MALFORMED))
@pytest.mark.parametrize("side", ["query", "candidate"])
def test_abi_rejects_malformed_featvec(what, side):
    from orb_slam3_b200 import _lib as L
    lib = L.lib()
    rng = np.random.default_rng(5)
    s = case(rng.integers(0, 256, (4, 32), dtype=np.uint8), rng.integers(0, 256, (4, 32), dtype=np.uint8))
    fv1, fv2 = (MALFORMED[what], s["fv2"]) if side == "query" else (s["fv1"], MALFORMED[what])
    h = C.c_void_p()
    assert lib.match_create(0, C.byref(h)) == 0
    out = np.zeros(4, np.int32)
    try:
        assert lib.match_bow_frame(h, C.byref(s["kf1"]), L.ptr(s["ok1"]), C.byref(fv1), C.byref(s["kf2"]), C.byref(fv2),
                                   0.75, 1, L.ptr(out)) == -2
        assert lib.match_bow_keyframes(h, C.byref(s["kf1"]), L.ptr(s["ok1"]), C.byref(fv1), C.byref(s["kf2"]),
                                       L.ptr(s["ok2"]), C.byref(fv2), 0.9, 1, L.ptr(out)) == -2
        assert "FeatureVector" in lib.orb_last_error().decode()
    finally:
        lib.match_destroy(h)


def test_abi_rejects_bad_arguments():
    from orb_slam3_b200 import _lib as L
    lib = L.lib()
    rng = np.random.default_rng(6)
    s = case(rng.integers(0, 256, (4, 32), dtype=np.uint8), rng.integers(0, 256, (4, 32), dtype=np.uint8))
    h = C.c_void_p()
    assert lib.match_create(0, C.byref(h)) == 0
    out = np.zeros(4, np.int32)
    k1, k2, f1, f2 = C.byref(s["kf1"]), C.byref(s["kf2"]), C.byref(s["fv1"]), C.byref(s["fv2"])
    ok = L.ptr(s["ok1"])
    try:
        assert lib.match_bow_frame(None, k1, ok, f1, k2, f2, 0.75, 1, L.ptr(out)) == -2
        assert lib.match_bow_frame(h, k1, None, f1, k2, f2, 0.75, 1, L.ptr(out)) == -2        # no map point flags
        assert lib.match_bow_frame(h, k1, ok, f1, k2, f2, 0.75, 1, None) == -2                # no output
        assert lib.match_bow_keyframes(h, k1, ok, f1, k2, None, f2, 0.9, 1, L.ptr(out)) == -2  # no KF2 flags
        oks = (C.c_void_p * 1)(s["ok1"].ctypes.data)
        outs = (C.c_void_p * 1)(out.ctypes.data)
        res = np.zeros(1, np.int32)
        assert lib.match_bow_frame_batch(h, 0, k1, oks, f1, k2, f2, 0.75, 1, outs, L.ptr(res), 0) == -2  # count 0
        assert lib.match_bow_frame_batch(h, 1, k1, oks, f1, k2, f2, 0.75, 1, outs, L.ptr(res), 3) == -2
        assert lib.match_bow_keyframes_batch(h, 1, k1, oks, f1, k2, oks, f2, 0.9, 1, outs, L.ptr(res), 2) == -2
        if lib.orb_device_count() == 0:   # well-formed input gets as far as the device search
            assert lib.match_bow_frame(h, k1, ok, f1, k2, f2, 0.75, 1, L.ptr(out)) == -5
    finally:
        lib.match_destroy(h)
