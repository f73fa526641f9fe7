#!/usr/bin/env python3
"""LocalBundleAdjustment timings (stats of the third of three solves) for one graph, as one JSON line.
Usage: python scripts/lba_prof.py [K L]"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from orb_slam3_b200 import scenes  # noqa: E402
from orb_slam3_b200.optimizer import LocalBundleAdjustment  # noqa: E402

K, L = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (200, 80000)
g, _ = scenes.lba_graph(K, L, seed=0)
lba = LocalBundleAdjustment()
gv = scenes.lba_view(g)
for rep in range(3):
    st = lba(gv)["stats"]
print(json.dumps({k: st[k] for k in ("iterations", "trials", "ms_total", "ms_linearize", "ms_schur", "ms_solve", "ms_update",
                                     "solver_kind", "envelope_rows_max", "ms_host_prep", "ms_wall")}))
