"""SearchByBoW on the device against the single-threaded CPU oracle, for the three shapes ORB-SLAM3 calls it in:

  reloc  Tracking::Relocalization: one 1280x720 frame with 2000 features, extracted on the device, its FeatureVector
         computed from the device descriptors, matched against 32 candidate keyframes in one batch (on_device = 2);
  loop   LoopClosing: 32 keyframe pairs in one batch, host views;
  trk    Tracking::TrackReferenceKeyFrame: one keyframe-frame call through host views.

Keyframes are frames of the same synthetic scene at other offsets; FeatureVectors come from a 10-ary vocabulary of
depth 4 at levelsup 2 (nodes at depth 2, as ORBvoc with levelsup 4).  Device time is CUDA events on the matcher's
stream (match_last_ms: upload, three kernels, read-back), wall time a host clock around the blocking call; both are
medians over --reps repetitions after --warmup.  `pairs` is the algorithmic count sum |Q| * |C| over shared nodes
(every query with a valid map point against every candidate of its node).  Prints one JSON line; writes nothing."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power = out[0].split(", ")
        return name, power
    except Exception as e:  # the measurement still stands; the card is then unnamed in the output
        return "unknown (%s)" % e, "unknown"


def shared_pairs(fvq, okq, fvc, okc=None):
    fq, fc = fvq._keep, fvc._keep
    where = {int(n): k for k, n in enumerate(fc["node_ids"])}
    total = 0
    for a, nid in enumerate(fq["node_ids"]):
        b = where.get(int(nid))
        if b is None:
            continue
        nq = int(okq[fq["idx"][fq["ptr"][a]:fq["ptr"][a + 1]]].sum())
        cand = fc["idx"][fc["ptr"][b]:fc["ptr"][b + 1]]
        total += nq * (len(cand) if okc is None else int(okc[cand].sum()))
    return total


def timed(fn, m, warmup, reps):
    for _ in range(warmup):
        fn()
    dev, wall = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        wall.append((time.perf_counter() - t0) * 1e3)
        dev.append(m.last_ms())
    return float(np.median(dev)), float(np.median(wall)), out


def oracle_ms(fn, reps=3):
    best = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        best.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(best)), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--keyframes", type=int, default=32)
    args = ap.parse_args()
    if args.reps < 50:
        ap.error("--reps must be at least 50")

    from oracle import bow_match as orc
    from orb_slam3_b200 import scenes
    from orb_slam3_b200.bow import ORBVocabulary
    from orb_slam3_b200.extractor import ORBextractor
    from orb_slam3_b200.matcher import ORBmatcher
    from orb_slam3_b200.synth import shifted_frame, synth_frame
    from orb_slam3_b200.views import make_featvec_view, make_frame_view, orb_frame_view
    import ctypes as C

    K = args.keyframes
    H, W, NF = 720, 1280, 2000
    sf = scenes.scale_factors()
    voc = scenes.synth_vocabulary(10, 4, seed=2)
    gv = ORBVocabulary(voc)
    rng = np.random.default_rng(0)
    img = synth_frame(H, W, 11)
    kf_imgs = [shifted_frame(img, 2 * (i % 8) - 7, (i // 8) - 2, 100 + i) for i in range(K + 1)]

    # keyframes: extracted (device), downloaded, FeatureVectors from their descriptors
    ex_kf = ORBextractor(NF, 1.2, 8, 20, 7, max_batch=K + 1)
    kfs, oks, fvs = [], [], []
    for mono, k, d in ex_kf.extract_batch(kf_imgs):
        r = gv.transform(d, 2)
        kfs.append(make_frame_view(k, d, W, H, sf))
        oks.append((rng.random(len(k)) >= 0.3).astype(np.uint8))
        fvs.append(make_featvec_view(scenes.nodes_from_featvec(len(k), r["fv_node_ids"], r["fv_ptr"], r["fv_idx"])))

    # the relocalising frame: extracted on the device, ComputeBoW from the device descriptors
    ex = ORBextractor(NF, 1.2, 8, 20, 7)
    ex.extract_batch([img])
    r = gv.transform_extracted(ex, 0, 2)
    _, fk, fd = ex.download_results(0)
    F = make_frame_view(fk, fd, W, H, sf)
    fvF = make_featvec_view(scenes.nodes_from_featvec(F.n, r["fv_node_ids"], r["fv_ptr"], r["fv_idx"]))
    kp_dev, desc_dev, _, _, _ = ex.device_results()
    Fd = orb_frame_view()
    C.memmove(C.byref(Fd), C.byref(F), C.sizeof(Fd))
    Fd.keys, Fd.desc = kp_dev, desc_dev

    result = {}
    parity = True

    # ---- Relocalization: 32 keyframes against the frame, ORBmatcher(0.75, true)
    m = ORBmatcher(0.75, True)
    ms_dev, ms_wall, (res, outs) = timed(lambda: m.bow_frame_batch(kfs[:K], oks[:K], fvs[:K], [Fd] * K, [fvF] * K,
                                                                      on_device=2), m, args.warmup, args.reps)
    ms_orc, ref = oracle_ms(lambda: [orc.match_bow_frame(kfs[i], oks[i], fvs[i], F, fvF, 0.75, True) for i in range(K)])
    ok = all(res[i] == ref[i][0] and np.array_equal(outs[i], ref[i][1]) for i in range(K))
    parity &= ok
    result["reloc"] = dict(problems=K, ms_device=ms_dev, ms_wall=ms_wall, ms_oracle_1thread=ms_orc,
                           pairs=sum(shared_pairs(fvs[i], oks[i], fvF) for i in range(K)),
                           nmatches=int(np.sum(res)), parity=bool(ok))

    # ---- LoopClosing: 32 keyframe pairs (i, i + 1), ORBmatcher(0.75, true), host views
    m = ORBmatcher(0.75, True)
    a, b = list(range(K)), list(range(1, K + 1))
    ms_dev, ms_wall, (res, outs) = timed(lambda: m.bow_keyframes_batch([kfs[i] for i in a], [oks[i] for i in a],
                                                                         [fvs[i] for i in a], [kfs[j] for j in b],
                                                                         [oks[j] for j in b], [fvs[j] for j in b]),
                                         m, args.warmup, args.reps)
    ms_orc, ref = oracle_ms(lambda: [orc.match_bow_keyframes(kfs[i], oks[i], fvs[i], kfs[j], oks[j], fvs[j], 0.75, True)
                                     for i, j in zip(a, b)])
    ok = all(res[k] == ref[k][0] and np.array_equal(outs[k], ref[k][1]) for k in range(K))
    parity &= ok
    result["loop"] = dict(problems=K, ms_device=ms_dev, ms_wall=ms_wall, ms_oracle_1thread=ms_orc,
                          pairs=sum(shared_pairs(fvs[i], oks[i], fvs[j], oks[j]) for i, j in zip(a, b)),
                          nmatches=int(np.sum(res)), parity=bool(ok))

    # ---- TrackReferenceKeyFrame: one call, ORBmatcher(0.7, true), host views
    m = ORBmatcher(0.7, True)
    ms_dev, ms_wall, (n, out) = timed(lambda: m.SearchByBoW(kfs[0], oks[0], fvs[0], F, fvF), m, args.warmup, args.reps)
    ms_orc, (n_ref, out_ref) = oracle_ms(lambda: orc.match_bow_frame(kfs[0], oks[0], fvs[0], F, fvF, 0.7, True), 20)
    ok = n == n_ref and np.array_equal(out, out_ref)
    parity &= ok
    result["trk"] = dict(problems=1, ms_device=ms_dev, ms_wall=ms_wall, ms_oracle_1thread=ms_orc,
                         pairs=shared_pairs(fvs[0], oks[0], fvF), nmatches=int(n), parity=bool(ok))

    name, power = gpu_info()
    print(json.dumps(dict(bench="search_by_bow", gpu=name, power_limit=power, reps=args.reps, warmup=args.warmup,
                          features=NF, image="%dx%d" % (W, H), parity=bool(parity), **result)))
    return 0 if parity else 1


if __name__ == "__main__":
    sys.exit(main())
