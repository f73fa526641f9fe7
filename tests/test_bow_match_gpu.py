"""ORBmatcher::SearchByBoW on the device (through the C ABI) against the CPU oracle: exact output arrays and match
counts, single calls and batches, shared-memory and global-memory nodes, and the extractor -> bow_transform_extracted
-> match_bow_frame_batch(on_device=2) chain."""
import ctypes as C

import numpy as np
import pytest

from oracle import bow_match as orc
from orb_slam3_b200 import scenes
from orb_slam3_b200._lib import KP_DTYPE
from orb_slam3_b200.views import make_featvec_view, make_frame_view, orb_featvec_view, orb_frame_view

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def node_fns(oracle):
    voc = scenes.synth_vocabulary(10, 4, seed=5)

    def by_vocab(levelsup):
        def f(desc):
            r = oracle.bow_transform(voc, desc, levelsup)
            return scenes.nodes_from_featvec(len(desc), r["fv_node_ids"], r["fv_ptr"], r["fv_idx"])
        return f
    return {"depth2": by_vocab(2), "root": by_vocab(4), "hash1000": lambda d: scenes.hash_nodes(d, 1000)}


def oracle_run(oracle, kind, s, ratio, ori):
    if kind == 0:
        return orc.match_bow_frame(s["kf1"], s["ok1"], s["fv1"], s["kf2"], s["fv2"], ratio, ori)
    return orc.match_bow_keyframes(s["kf1"], s["ok1"], s["fv1"], s["kf2"], s["ok2"], s["fv2"], ratio, ori)


def cuda_run(kind, s, ratio, ori):
    from orb_slam3_b200.matcher import ORBmatcher
    m = ORBmatcher(ratio, ori)
    if kind == 0:
        return m.SearchByBoW(s["kf1"], s["ok1"], s["fv1"], s["kf2"], s["fv2"])
    return m.SearchByBoWKeyFrames(s["kf1"], s["ok1"], s["fv1"], s["kf2"], s["ok2"], s["fv2"])


@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("nodes", ["depth2", "root", "hash1000"])
@pytest.mark.parametrize("kind", [0, 1])
def test_cuda_equals_oracle(oracle, node_fns, seed, nodes, kind):
    s = scenes.bow_match_scene(2000, seed, node_fns[nodes])
    for ratio in (0.7, 0.75, 0.9):
        for ori in (True, False):
            n_ref, out_ref = oracle_run(oracle, kind, s, ratio, ori)
            n, out = cuda_run(kind, s, ratio, ori)
            assert n == n_ref and np.array_equal(out, out_ref), (ratio, ori, n, n_ref, int((out != out_ref).sum()))
    assert n_ref > 100


def test_batches_equal_singles_and_repeat(oracle, node_fns):
    from orb_slam3_b200.matcher import ORBmatcher
    scs = [scenes.bow_match_scene(1500, 10 + i, node_fns[("depth2", "root", "hash1000")[i % 3]]) for i in range(6)]
    # Relocalization shape: one frame view (the same object) against several keyframes
    frame = scs[0]
    reloc = [dict(s, kf2=frame["kf2"], fv2=frame["fv2"]) for s in scs]
    for ratio, ori in ((0.75, True), (0.9, False)):
        m = ORBmatcher(ratio, ori)
        for batch in (scs, reloc):
            res, outs = m.bow_frame_batch([s["kf1"] for s in batch], [s["ok1"] for s in batch], [s["fv1"] for s in batch],
                                          [s["kf2"] for s in batch], [s["fv2"] for s in batch])
            launches = m.kernel_launches()
            res2, outs2 = m.bow_frame_batch([s["kf1"] for s in batch], [s["ok1"] for s in batch], [s["fv1"] for s in batch],
                                            [s["kf2"] for s in batch], [s["fv2"] for s in batch])
            assert m.kernel_launches() - launches == 3 and m.last_ms() > 0
            for k, s in enumerate(batch):
                n, out = m.SearchByBoW(s["kf1"], s["ok1"], s["fv1"], s["kf2"], s["fv2"])
                n_ref, out_ref = oracle_run(oracle, 0, s, ratio, ori)
                assert res[k] == n == n_ref and np.array_equal(outs[k], out) and np.array_equal(out, out_ref), k
                assert res2[k] == res[k] and np.array_equal(outs2[k], outs[k])
        res, outs = m.bow_keyframes_batch([s["kf1"] for s in scs], [s["ok1"] for s in scs], [s["fv1"] for s in scs],
                                          [s["kf2"] for s in scs], [s["ok2"] for s in scs], [s["fv2"] for s in scs])
        for k, s in enumerate(scs):
            n, out = m.SearchByBoWKeyFrames(s["kf1"], s["ok1"], s["fv1"], s["kf2"], s["ok2"], s["fv2"])
            n_ref, out_ref = oracle_run(oracle, 1, s, ratio, ori)
            assert res[k] == n == n_ref and np.array_equal(outs[k], out) and np.array_equal(out, out_ref), k


@pytest.mark.parametrize("n", [2000, 10000])
def test_one_large_node(oracle, n):
    """A whole frame in one node (levelsup >= L; monocular initialisation has 5 x nFeatures): the global-memory path."""
    s = scenes.bow_match_scene(n, 7, lambda d: np.zeros(len(d), np.int64))
    assert s["fv1"].n_nodes == s["fv2"].n_nodes == 1
    for kind in (0, 1):
        n_ref, out_ref = oracle_run(oracle, kind, s, 0.9, True)
        got, out = cuda_run(kind, s, 0.9, True)
        assert got == n_ref and np.array_equal(out, out_ref), (kind, got, n_ref)
        assert n_ref > n // 10


def test_device_resident_views(oracle, node_fns):
    """on_device = 1: every array, FeatureVectors and outputs included, is device memory."""
    import torch
    from orb_slam3_b200.matcher import ORBmatcher
    scs = [scenes.bow_match_scene(1000, 20 + i, node_fns["depth2"]) for i in range(3)]
    keep = []

    def dev(a):
        t = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()
        keep.append(t)
        return t.data_ptr()

    def dview(v):
        w = orb_frame_view()
        C.memmove(C.byref(w), C.byref(v), C.sizeof(w))
        w.keys, w.desc = dev(v._keep[0]), dev(v._keep[1])
        return w

    def dfv(f):
        w = orb_featvec_view()
        w.n_nodes = f.n_nodes
        w.node_ids, w.ptr, w.idx = dev(f._keep["node_ids"]), dev(f._keep["ptr"]), dev(f._keep["idx"])
        return w
    m = ORBmatcher(0.75, True)
    out = torch.full((3, 1000), -7, dtype=torch.int32, device="cuda")
    ptrs = [out.data_ptr() + 4 * 1000 * k for k in range(3)]
    res, _ = m.bow_frame_batch([dview(s["kf1"]) for s in scs], [dev(s["ok1"]) for s in scs],
                               [dfv(s["fv1"]) for s in scs], [dview(s["kf2"]) for s in scs],
                               [dfv(s["fv2"]) for s in scs], on_device=1, out_ptrs=ptrs)
    for k, s in enumerate(scs):
        n_ref, out_ref = oracle_run(oracle, 0, s, 0.75, True)
        assert res[k] == n_ref and np.array_equal(out[k, :s["kf2"].n].cpu().numpy(), out_ref), k
    res, _ = m.bow_keyframes_batch([dview(s["kf1"]) for s in scs], [dev(s["ok1"]) for s in scs],
                                   [dfv(s["fv1"]) for s in scs], [dview(s["kf2"]) for s in scs],
                                   [dev(s["ok2"]) for s in scs], [dfv(s["fv2"]) for s in scs], on_device=1, out_ptrs=ptrs)
    for k, s in enumerate(scs):
        n_ref, out_ref = oracle_run(oracle, 1, s, 0.75, True)
        assert res[k] == n_ref and np.array_equal(out[k, :s["kf1"].n].cpu().numpy(), out_ref), k


def test_extractor_bow_transform_matcher_chain(oracle):
    """Relocalization's frame: extracted on the device, ComputeBoW from the device descriptors, matched against
    keyframes with on_device = 2 (the frame's keypoints and descriptors are never uploaded again)."""
    from orb_slam3_b200.bow import ORBVocabulary
    from orb_slam3_b200.extractor import ORBextractor
    from orb_slam3_b200.matcher import ORBmatcher
    from orb_slam3_b200.synth import shifted_frame, synth_frame
    voc = scenes.synth_vocabulary(10, 4, seed=2)
    gv = ORBVocabulary(voc)
    img = synth_frame(720, 1280, 11)
    ext = ORBextractor(2000, 1.2, 8, 20, 7)
    ext.extract_batch([img])
    fv_f = gv.transform_extracted(ext, frame=0, levelsup=2)
    _, kf_keys, kf_desc = ext.download_results(0)
    kp_dev, desc_dev, _, _, cap = ext.device_results()
    F = make_frame_view(kf_keys, kf_desc, 1280, 720, scenes.scale_factors())
    Fd = orb_frame_view()
    C.memmove(C.byref(Fd), C.byref(F), C.sizeof(Fd))
    Fd.keys, Fd.desc = kp_dev, desc_dev
    fvF = make_featvec_view(scenes.nodes_from_featvec(F.n, fv_f["fv_node_ids"], fv_f["fv_ptr"], fv_f["fv_idx"]))
    kfs, oks, fvs = [], [], []
    rng = np.random.default_rng(3)
    for i in range(4):
        k, d, _ = oracle.OracleExtractor(2000).extract(shifted_frame(img, 3 * i, -2 * i, 20 + i))
        r = oracle.bow_transform(voc, d, 2)
        kfs.append(make_frame_view(k, d, 1280, 720, scenes.scale_factors()))
        oks.append((rng.random(len(k)) > 0.3).astype(np.uint8))
        fvs.append(make_featvec_view(scenes.nodes_from_featvec(len(k), r["fv_node_ids"], r["fv_ptr"], r["fv_idx"])))
    m = ORBmatcher(0.75, True)
    res, outs = m.bow_frame_batch(kfs, oks, fvs, [Fd] * 4, [fvF] * 4, on_device=2)
    for i in range(4):
        n_ref, out_ref = orc.match_bow_frame(kfs[i], oks[i], fvs[i], F, fvF, 0.75, True)
        assert res[i] == n_ref and np.array_equal(outs[i], out_ref), i
    assert res[0] > 100


def test_empty_and_degenerate_inputs(oracle):
    from orb_slam3_b200.matcher import ORBmatcher
    rng = np.random.default_rng(4)
    sf = scenes.scale_factors()
    d = rng.integers(0, 256, (5, 32), dtype=np.uint8)
    k = np.zeros(5, KP_DTYPE)
    v = make_frame_view(k, d, 640, 480, sf)
    e = make_frame_view(k[:0], d[:0], 640, 480, sf)
    fv, fv_none, fv_other = make_featvec_view(np.zeros(5)), make_featvec_view(-np.ones(5)), make_featvec_view(np.ones(5))
    fv_e = make_featvec_view(np.zeros(0))
    ones, zeros = np.ones(5, np.uint8), np.zeros(5, np.uint8)
    m = ORBmatcher(0.9, True)
    for (q, okq, fq, c, okc, fc) in [(v, ones, fv, v, ones, fv_none), (v, ones, fv, v, ones, fv_other),
                                     (v, zeros, fv, v, ones, fv), (v, ones, fv, v, zeros, fv),
                                     (e, zeros[:0], fv_e, e, zeros[:0], fv_e), (v, ones, fv, e, zeros[:0], fv_e)]:
        n0, o0 = m.SearchByBoW(q, okq, fq, c, fc)
        r0 = orc.match_bow_frame(q, okq, fq, c, fc, 0.9, True)
        n1, o1 = m.SearchByBoWKeyFrames(q, okq, fq, c, okc, fc)
        r1 = orc.match_bow_keyframes(q, okq, fq, c, okc, fc, 0.9, True)
        assert (n0, o0.tolist()) == (r0[0], r0[1].tolist()) and (n1, o1.tolist()) == (r1[0], r1[1].tolist())
    # identical descriptors on both sides: every query ties with itself only, distance 0
    n, out = m.SearchByBoW(v, ones, fv, v, fv)
    assert n == 5 and out.tolist() == list(range(5))
