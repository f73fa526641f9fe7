#!/usr/bin/env python3
"""Generate tests/golden/ref_gpu.json: the results the GPU tests compare the CUDA path with where the reference's object
code (oracle/_ref) is absent -- test_ref_parity.py::test_cuda_equals_reference_object_code and test_ref_front_gpu.py.
Each output is stored as the sha256 of its dtype, shape and bytes (test_ref_parity.digest).

With oracle/_ref present the results are the reference's own.  Without it they are the oracle's: on the extractor cases
test_ref_parity.py::test_reference_object_code_equals_oracle holds the oracle bit for bit to the reference on exactly these
inputs, and test_ref_front.py holds its matchers, isInFrustum and ComputeStereoMatches to the reference's front-end object
code.  `source` in the file says which one wrote it.

    python scripts/make_golden_ref_gpu.py"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from oracle import oracle as O  # noqa: E402
from oracle import ref as R  # noqa: E402
from orb_slam3_b200 import scenes  # noqa: E402
from orb_slam3_b200.synth import synth_frame, shifted_frame, stereo_right  # noqa: E402
from test_ref_parity import CASES, digest, extract_key  # noqa: E402

O.build()
live_ext, live_front = R.available(), R.front_available()
cases = {}

for h, w, nf, seed, low, lap in CASES:
    img = synth_frame(h, w, seed, low_texture=low)
    ex = R.RefExtractor(nf) if live_ext else O.OracleExtractor(nf)
    k, d, mono = ex.extract(img, lap)
    cases[extract_key(h, w, nf, seed, low, lap)] = {
        "n": len(k), "mono": int(mono), "kps": digest(k), "desc": digest(d),
        "levels": [digest(ex.level_image(l)) for l in range(8)]}

# test_ref_front_gpu.py: the feats fixture, then every call the tests make
a = synth_frame(720, 1280, 41)
b = shifted_frame(a, 5, -3, 42)
fx = O.OracleExtractor(2000)
ka, da, _ = fx.extract(a)
kb, db, _ = fx.extract(b)
for stereo in (False, True):
    for th, ratio, far in [(1.0, 0.8, False), (3.0, 0.8, True), (15.0, 0.9, False)]:
        F, mps = scenes.local_map_scene(ka, da, 1280, 720, 1000, seed=int(th) + 7 * stereo, stereo=stereo)
        n, asg = (R.front_project_local(F, mps, th, ratio, far, 40.0) if live_front else
                  O.match_project_local(F, mps, th, ratio, far_points=far, th_far=40.0))
        cases["local_%d_%s_%d_%d" % (stereo, th, ratio * 10, far)] = {"n": int(n), "assign": digest(asg)}
    cur, last, Tcw = scenes.last_frame_scene(ka, da, kb, db, 1280, 720, (5, -3), seed=3, stereo=stereo)
    for th in (7.0, 15.0):
        for (fw, bw) in ((0, 0), (1, 0), (0, 1)) if stereo else ((0, 0),):
            for ori in (True, False):
                n, asg = (R.front_project_last(cur, last, Tcw, th, fw, bw, ori) if live_front else
                          O.match_project_last(cur, last, Tcw, th, forward=fw, backward=bw, check_ori=ori))
                asg = np.where(asg < 0, -1, asg)   # the reference's NULL, whichever way the match was refused
                cases["last_%d_%s_%d_%d_%d" % (stereo, th, fw, bw, ori)] = {"n": int(n), "assign": digest(asg)}
for n_pts, seed, cos_limit in [(3000, 0, 0.5), (50000, 1, 0.5), (20000, 3, 0.9)]:
    v, _ = scenes.frustum_scene(n_pts, seed=seed)
    n, r = R.front_is_in_frustum(v, cos_limit) if live_front else O.is_in_frustum(v, cos_limit)
    inside = r["track_in_view"] != 0
    cases["frustum_%d_%d_%s" % (n_pts, seed, cos_limit)] = {
        "n": int(n), "track_in_view": digest(r["track_in_view"]),
        "inside": [digest(r[k][inside]) for k in ("proj_x", "proj_y", "proj_xr", "scale_level", "view_cos", "depth")]}
for h, w, nf, disp in [(480, 752, 1000, (12,)), (720, 1280, 2000, (5, 30, 17))]:
    left = synth_frame(h, w, 9)
    right = stereo_right(left, 109, disparities=disp)
    el, er = O.OracleExtractor(nf), O.OracleExtractor(nf)
    kl, dl, _ = el.extract(left)
    kr, dr, _ = er.extract(right)
    pl, pr = [el.level_image(l) for l in range(8)], [er.level_image(l) for l in range(8)]
    n, ur, dp = (R.front_stereo_match(kl, dl, kr, dr, pl, pr, 386.0, 0.5514) if live_front else
                 O.stereo_match(kl, dl, kr, dr, pl, pr, 386.0, 0.5514)[:3])
    cases["stereo_%d_%d_%d" % (h, w, nf)] = {"n": int(n), "u_right": digest(ur), "depth": digest(dp)}

out = {"source": {"extract": "reference object code (oracle/_ref)" if live_ext else "oracle",
                  "front": "reference object code (oracle/_ref)" if live_front else "oracle"},
       "cases": cases}
with open(os.path.join(ROOT, "tests", "golden", "ref_gpu.json"), "w") as f:
    json.dump(out, f, indent=1, sort_keys=True)
    f.write("\n")
print(len(cases), "cases,", out["source"])
