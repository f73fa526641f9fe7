"""The SearchByBoW oracle (oracle/orc_bow_match.cpp) against the reference's own ORBmatcher::SearchByBoW, both overloads,
as object code (oracle/_ref/libref_front_bow.so: real KeyFrame / Frame / MapPoint objects).  The reference's vectors hold NULL
both for "never matched" and for "cleared by the rotation check", so the oracle's -2 reads -1 here.  Skips where the
library cannot be built."""
import numpy as np
import pytest

from oracle import bow_match as orc
from orb_slam3_b200 import scenes


@pytest.fixture(scope="module")
def ref():
    if not orc.ref_available():
        pytest.skip("oracle/_ref/libref_front_bow.so needs the reference tree")
    return orc


@pytest.fixture(scope="module")
def node_fns(oracle):
    voc = scenes.synth_vocabulary(10, 4, seed=5)

    def by_vocab(levelsup):
        def f(desc):
            r = oracle.bow_transform(voc, desc, levelsup)
            return scenes.nodes_from_featvec(len(desc), r["fv_node_ids"], r["fv_ptr"], r["fv_idx"])
        return f
    return {"depth2": by_vocab(2), "root": by_vocab(4), "hash1000": lambda d: scenes.hash_nodes(d, 1000)}


@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("nodes", ["depth2", "root", "hash1000"])
def test_oracle_equals_reference(oracle, ref, node_fns, seed, nodes):
    s = scenes.bow_match_scene(800, seed, node_fns[nodes])
    for ratio in (0.7, 0.75, 0.9):
        for ori in (True, False):
            n, out = orc.match_bow_frame(s["kf1"], s["ok1"], s["fv1"], s["kf2"], s["fv2"], ratio, ori)
            n_ref, out_ref = ref.ref_bow_frame(s["kf1"], s["ok1"], s["fv1"], s["kf2"], s["fv2"], ratio, ori)
            assert n == n_ref and np.array_equal(np.where(out == -2, -1, out), out_ref), ("frame", ratio, ori)
            n, out = orc.match_bow_keyframes(s["kf1"], s["ok1"], s["fv1"], s["kf2"], s["ok2"], s["fv2"], ratio, ori)
            n_ref, out_ref = ref.ref_bow_keyframes(s["kf1"], s["ok1"], s["fv1"], s["kf2"], s["ok2"], s["fv2"], ratio,
                                                   ori)
            assert n == n_ref and np.array_equal(np.where(out == -2, -1, out), out_ref), ("keyframes", ratio, ori)
