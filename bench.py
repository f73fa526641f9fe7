#!/usr/bin/env python3
"""bench.py -- BASELINE.json metric on synthetic data.

python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the front-end hot path over one batch (128 per GPU) of synthetic
1280x720 frames (BASELINE.json configs[1]: 8 levels, 2000 features): per frame
ORB extract -> SearchByProjection against the previous frame (th 15, rotation
check) -> SearchByProjection against ~3000 local map points (th 3).  One
process per GPU (torchrun for N>1); frames are independent so ranks share
nothing on this path: weak scaling, no data-path collective.

  value : frames/s with the batch already resident in HBM (CUDA events on the
          launching stream, max over ranks)
  e2e   : frames/s through the host-buffer C ABI: pinned host frames -> H2D ->
          kernels -> D2H keypoints + descriptors, then host views -> match ->
          D2H assignments
  lba   : LocalBA LM iterations/s (optimize(10) incl. rejected trials) on the
          synthetic config-4 graph (N=1) / config-5 graph sharded by landmark
          with one NCCL all-reduce per trial (N>1)
  roofline / cpu_baseline : see DESIGN.md "Measurement"

--dump-outputs DIR writes what the last timed step handed back on rank 0 (keypoints, descriptors, match
assignments; see dump_outputs) as DIR/<name>.npy, so that two builds can be compared on identical inputs.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, NFEAT, NLEVELS = 720, 1280, 2000, 8
N_LOCAL_EXTRA = 1000          # random map points on top of one per keypoint (~3000 total)
TH_LAST, TH_LOCAL = 15.0, 3.0
METRIC = "frames/sec ORB extract+match 1280x720x8lvl"
WORKLOAD = ("configs[1]: 1280x720 8-level 2000-feature ORB extract + SearchByProjection "
            "(last frame th=15 + ~3000 local map points th=3), synthetic stream")


def level_pixels():
    inv = [np.float32(1.0)]
    sc = np.float32(1.0)
    for _ in range(1, NLEVELS):
        sc = np.float32(np.float64(sc) * np.float64(np.float32(1.2)))
        inv.append(np.float32(1.0) / sc)
    return [int(np.rint(np.float32(W) * s)) * int(np.rint(np.float32(H) * s)) for s in inv]


N_STREAMS, STREAM_LEN = 8, 32      # 8 camera streams x 32 frames = 256 distinct frames (+ the 8 stream heads)


def make_streams(rank, n_streams=N_STREAMS, length=STREAM_LEN):
    """SURVEY.md 8(d): stream s of this rank = synth frame seed 1000*(rank*n_streams+s), then `length` frames each the
    previous one shifted by (dx,dy) in [-8,8]^2.  Returns (frames[n_streams*(length+1)], shifts, index of the
    predecessor of every frame or -1 for a stream head)."""
    frames, shifts, prev = [], [], []
    for s in range(n_streams):
        f, sh = make_frames(length + 1, 1000 * (rank * n_streams + s) + 1)
        base = len(frames)
        frames.extend(f)
        shifts.extend(sh)
        prev.extend([-1] + [base + t - 1 for t in range(1, length + 1)])
    return np.stack(frames), shifts, prev


def make_frames(n, seed0):
    """A synthetic stream: frame t+1 = frame t shifted by (dx,dy) in [-8,8]^2."""
    from orb_slam3_b200.synth import synth_frame, shifted_frame
    rng = np.random.default_rng(seed0)
    frames, shifts = [synth_frame(H, W, seed0)], [(0, 0)]
    for t in range(1, n):
        dx, dy = (int(v) for v in rng.integers(-8, 9, size=2))
        frames.append(shifted_frame(frames[-1], dx, dy, seed0 * 1000 + t))
        shifts.append((dx, dy))
    return np.stack(frames), shifts


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons during the timed region.  NVML in-process (pynvml) so that no
    nvidia-smi process has to be spawned next to the measurement; nvidia-smi is the fallback."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.sm, self.mx, self.reasons = [], [], set()
        self.samples = 0
        self.stop_flag = False
        self.nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[gpu_index]) if vis and vis.split(",")[gpu_index].isdigit() else gpu_index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nv = pynvml
        except Exception:
            self.nv = None

    def _sample_nvml(self):
        nv = self.nv
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
        self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)))
        try:
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        table = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
        for name, bit in table.items():
            if r & bit:
                self.reasons.add(name)
        self.samples += 1

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout.strip()
        if not out:
            return
        r = [c.strip() for c in out.split(",")]
        try:
            self.sm.append(float(r[1]))
            self.mx.append(float(r[2]))
        except ValueError:
            pass
        for nm, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[5:9]):
            if v.lower().startswith("active"):
                self.reasons.add(nm)
        self.samples += 1

    def run(self):
        while not self.stop_flag:
            try:
                if self.nv:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            time.sleep(0.01 if self.nv else 0.2)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": self.samples,
                "source": "nvml" if self.nv else "nvidia-smi"}


# --------------------------------------------------------------------------- CPU arm
def cpu_extractor():
    """(extract_throughput(frames, nfeatures, threads, iters) -> (fps, done, seconds), kind).  kind "reference": the
    reference's own ORBextractor.cc as object code (oracle/_ref, built in the container that has /root/reference and
    shipped prebuilt) over cv2-pinned image primitives; "port": the restated oracle when that library is absent."""
    from oracle import oracle as O
    from oracle import ref as R
    if os.path.exists(R.LIB_PATH):
        def thr(frames, nfeatures, threads, iters):
            dt, _ = R.extract_throughput(frames, nfeatures, threads, iters)
            return threads * iters / dt, threads * iters, dt
        return thr, "reference"
    return O.extract_throughput, "port"


def cpu_extract_fps(frames, threads, seconds_budget):
    thr, _ = cpu_extractor()
    fps1, _, _ = thr(frames, NFEAT, 1, 2)
    iters = int(min(64, max(2, seconds_budget * fps1)))
    return thr(frames, NFEAT, threads, iters)


_BEST_THREADS = {}


def best_cpu_threads():
    """Thread count that gives the reference arm its best throughput on this host:
    shared boxes often expose more logical CPUs than the process can really use."""
    if "n" in _BEST_THREADS:
        return _BEST_THREADS["n"]
    thr, _ = cpu_extractor()
    ncpu = os.cpu_count() or 1
    frames, _ = make_frames(4, 1)
    cands = sorted({c for c in (4, 8, 16, 32, 64, ncpu) if c <= ncpu})
    best, best_fps = ncpu, 0.0
    for c in cands:
        fps, _, _ = thr(frames, NFEAT, c, 3)
        if fps > best_fps:
            best, best_fps = c, fps
    _BEST_THREADS["n"] = best
    return best


def cpu_match_seconds_per_frame(frames, shifts, n_pairs=3):
    """Oracle matchers (one thread, like the Tracking thread) on a few frame pairs."""
    from oracle import oracle as O
    from orb_slam3_b200 import scenes
    ex = O.OracleExtractor(NFEAT)
    feats = [ex.extract(f)[:2] for f in frames[:n_pairs + 1]]
    t_m = 0.0
    for t in range(1, n_pairs + 1):
        (ka, da), (kb, db) = feats[t - 1], feats[t]
        cur, last, Tcw = scenes.last_frame_scene(ka, da, kb, db, W, H, shifts[t], seed=2 * t)
        F, mps = scenes.local_map_scene(kb, db, W, H, N_LOCAL_EXTRA, seed=7 * t)
        t1 = time.perf_counter()
        O.match_project_last(cur, last, Tcw, TH_LAST)
        O.match_project_local(F, mps, TH_LOCAL, 0.8)
        t_m += time.perf_counter() - t1
    return t_m / n_pairs


def cpu_lba(K, L, seed=0):
    from oracle import oracle as O
    from orb_slam3_b200 import scenes
    g, _ = scenes.lba_graph(K, L, seed=seed)
    r = O.lba_solve(scenes.lba_view(g))
    st = r["stats"]
    return {"config": "%d KF x %d landmarks, %d edges" % (K, L, len(g["e_kf"])), "iterations": st["iterations"],
            "trials": st["trials"], "seconds": st["ms_total"] / 1e3,
            "value": st["trials"] / (st["ms_total"] / 1e3), "unit": "LM iterations/s", "threads": 1}


def lba_rig_leg(device):
    """SURVEY.md 8a row a17 in the bench line: a fisheye stereo rig window (KannalaBrandt8 cameras on the mono edges,
    EdgeSE3ProjectXYZToBody edges for the second camera) of config-4 size through lba_solve, beside the oracle port on
    one host thread (timed = its CPU baseline; its result = the parity figures)."""
    from oracle import oracle as O
    from orb_slam3_b200 import scenes
    from orb_slam3_b200.optimizer import LocalBundleAdjustment
    K, L = 50, 20000
    g, _ = scenes.lba_rig_graph(K, L, seed=0)
    gv = scenes.lba_view(g)
    lba = LocalBundleAdjustment(device=device)
    best, res = None, None
    for rep in range(3):
        r = lba(gv)
        if rep > 0 and (best is None or r["stats"]["ms_total"] < best["ms_total"]):
            best, res = r["stats"], r
    ref = O.lba_solve(gv)
    dref, dgot = ref["mp_pos"] - g["mp_pos"], res["mp_pos"] - g["mp_pos"]
    tref, tgot = ref["kf_pose"][:, 4:] - g["kf_pose"][:, 4:], res["kf_pose"][:, 4:] - g["kf_pose"][:, 4:]
    return {"config": "fisheye stereo rig: %d KF x %d landmarks, %d mono (KannalaBrandt8) + %d second-camera edges"
                      % (K, L, int((g["e_stereo"] == 0).sum()), int((g["e_stereo"] == 2).sum())),
            "iterations": best["iterations"], "trials": best["trials"], "ms_total": best["ms_total"],
            "value": best["trials"] / (best["ms_total"] * 1e-3), "unit": "LM iterations/s",
            "cpu_port": {"value": ref["stats"]["trials"] / (ref["stats"]["ms_total"] / 1e3), "unit": "LM iterations/s", "threads": 1},
            "parity_vs_oracle": {"same_iterations_and_trials": bool(ref["iterations"] == res["iterations"] and
                                                                     ref["stats"]["trials"] == best["trials"]),
                                 "rel_delta_points": float(np.linalg.norm(dgot - dref) / max(np.linalg.norm(dref), 1e-30)),
                                 "rel_delta_translations": float(np.linalg.norm(tgot - tref) / max(np.linalg.norm(tref), 1e-30)),
                                 "tolerance": 1e-4}}


def run_reference(args):
    """The reference's own CPU implementation of the path: ORBextractor.cc compiled unmodified (oracle/_ref) when
    that library was built (kind "reference"), else the oracle port; matchers and LBA are the oracle port (their
    translation units need Eigen).  All host threads for the per-frame work (one extractor instance per thread),
    single thread for LBA like g2o."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    O.build()
    threads = best_cpu_threads()
    frames, shifts = make_frames(8, 1)
    K, Wm = args.steps, args.warmup
    t_match = cpu_match_seconds_per_frame(frames, shifts)
    vals = []
    for i in range(Wm + K):
        fps, done, dt = cpu_extract_fps(frames, threads, seconds_budget=1.0)
        if i >= Wm:
            vals.append((done, dt))
    done = sum(v[0] for v in vals)
    secs = sum(v[1] for v in vals)
    # matching runs on the same threads: add its per-frame cost to each thread's frame time
    t_ext_frame_thread = secs * threads / max(done, 1)
    fps = threads / (t_ext_frame_thread + t_match)
    lba = cpu_lba(50, 20000)
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": K, "warmup": Wm, "ms_per_step": 1e3 * secs / max(K, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "frames_per_step": int(vals[0][0]) if vals else 0},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": cpu_extractor()[1],
                         "sample": "%d frames/step over %d std::threads (best of 4..nproc); extract = %s, -O3 x86-64-v3, "
                                   "%.2f ms/frame/thread measured with all threads busy; SearchByProjection x2 = oracle port, "
                                   "%.2f ms/frame measured on one thread; value = threads / (extract + match) -- a composition "
                                   "of two measurements, not one loop"
                                   % (vals[0][0] if vals else 0, threads,
                                      "the reference's ORBextractor.cc object code (oracle/_ref) over scalar cv2-pinned "
                                      "resize/FAST/blur (OpenCV's SIMD versions would be faster)"
                                      if cpu_extractor()[1] == "reference" else "oracle C++ port",
                                      1e3 * t_ext_frame_thread, 1e3 * t_match)},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "lba": lba,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------- GPU arm
class Workload:
    """POOL distinct batches of B frames with everything the matchers need."""

    def __init__(self, B, POOL, rank, device, stream, share=None):
        import torch
        from orb_slam3_b200 import scenes
        from orb_slam3_b200.extractor import ORBextractor
        from orb_slam3_b200.matcher import ORBmatcher
        self.torch, self.B, self.POOL = torch, B, POOL
        self.ext = ORBextractor(NFEAT, 1.2, NLEVELS, 20, 7, device=device)
        self.m_last = ORBmatcher(0.9, True, device=device)
        self.m_local = ORBmatcher(0.8, True, device=device)
        self.stream = stream
        for m in (self.m_last, self.m_local):
            m.set_stream(stream)
        cap = self.ext.cap
        self.cap = cap
        if share is not None:
            # extra e2e worker: same inputs, own engine handles and output buffers
            self.uniq, self.host_pool, self.dev_pool, self.meta = share.uniq, share.host_pool, None, share.meta
            self.sf, self.sf2 = share.sf, share.sf2
            self._alloc_outputs(torch, B, cap)
            return
        uniq, shifts, prev = make_streams(rank)
        self.uniq = uniq
        succ = [i for i in range(len(uniq)) if prev[i] >= 0]   # the 256 frames that have a predecessor
        nu = len(succ)
        self.n_distinct = nu
        self.host_pool, self.dev_pool, self.meta = [], [], []
        self.sf = scenes.scale_factors()
        self.sf2 = (self.sf * self.sf).astype(np.float32)
        # one untimed extraction of the distinct frames (GPU) to build the match inputs
        res = self.ext.extract_batch(list(uniq))
        scene_cache = {}
        for p in range(POOL):
            t = torch.empty((B, H, W), dtype=torch.uint8).pin_memory()
            idx = [succ[(b + p * B) % nu] for b in range(B)]  # frame idx[b]; its predecessor is prev[idx[b]]
            for b in range(B):
                t[b] = torch.from_numpy(uniq[idx[b]])
            self.host_pool.append(t)
            self.dev_pool.append(t.cuda())
            entry = {"n": [], "cur": [], "last": [], "T": [], "F": [], "mps": [], "d_last": [], "d_mps": [],
                     "d_taken": []}
            for b in range(B):
                i = idx[b]
                if i not in scene_cache:  # only len(uniq)-1 distinct frames exist
                    _, kb, db = res[i]
                    _, ka, da = res[prev[i]]
                    cur, last, Tcw = scenes.last_frame_scene(ka, da, kb, db, W, H, shifts[i], seed=2 * i)
                    F, mps = scenes.local_map_scene(kb, db, W, H, N_LOCAL_EXTRA, seed=7 * i)
                    scene_cache[i] = (
                        len(kb), cur, last, Tcw, F, mps,
                        {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in last._keep.items()},
                        {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in mps._keep.items()},
                        (torch.from_numpy(cur._keep[5]).cuda(), torch.from_numpy(F._keep[5]).cuda()))
                n_i, cur, last, Tcw, F, mps, dl, dm, dtk = scene_cache[i]
                entry["n"].append(n_i)
                entry["cur"].append(cur); entry["last"].append(last); entry["T"].append(Tcw)
                entry["F"].append(F); entry["mps"].append(mps)
                entry["d_last"].append(dl); entry["d_mps"].append(dm); entry["d_taken"].append(dtk)
            entry["T"] = np.stack(entry["T"])
            self.meta.append(entry)
        self.d_assign_last = torch.empty((B, cap), dtype=torch.int32, device="cuda")
        self.d_assign_local = torch.empty((B, cap), dtype=torch.int32, device="cuda")
        self._alloc_outputs(torch, B, cap)

    def _alloc_outputs(self, torch, B, cap):
        self.out_k = torch.empty((B, cap * 28), dtype=torch.uint8).pin_memory()
        self.out_d = torch.empty((B, cap * 32), dtype=torch.uint8).pin_memory()
        self.out_n = np.zeros(B, np.int32)
        self.out_m = np.zeros(B, np.int32)
        self.nmatch_last = np.zeros(B, np.int32)
        self.nmatch_local = np.zeros(B, np.int32)
        self._dev_views = {}
        self._host_views = {}

    # views whose frame side points at the extractor's device results (built once per pool entry)
    def _device_views(self, p):
        from orb_slam3_b200.views import orb_frame_view, orb_lastframe_view, orb_mappoint_view
        kp, ds, _, _, cap = self.ext.device_results()   # double-buffered: the set of the extraction just submitted
        p = (p, kp)
        if p in self._dev_views:
            return self._dev_views[p]
        e = self.meta[p[0]]
        curs, lasts, Fs, Ms = [], [], [], []
        for b in range(self.B):
            for which, src, lst in ((0, e["cur"][b], curs), (1, e["F"][b], Fs)):
                v = orb_frame_view()
                C.memmove(C.byref(v), C.byref(src), C.sizeof(v))
                v.n = e["n"][b]
                v.keys = kp + b * cap * 28
                v.desc = ds + b * cap * 32
                v.u_right = None
                v.kp_taken = e["d_taken"][b][which].data_ptr()
                v.scale_factors, v.level_sigma2 = self.sf.ctypes.data, self.sf2.ctypes.data
                lst.append(v)
            lv = orb_lastframe_view()
            lv.n = e["last"][b].n
            for k in ("has_mp", "has_obs", "world_pos", "desc", "octave", "angle"):
                setattr(lv, k, e["d_last"][b][k].data_ptr())
            lasts.append(lv)
            mv = orb_mappoint_view()
            mv.n = e["mps"][b].n
            for k in ("track_in_view", "is_bad", "has_obs", "proj_x", "proj_y", "proj_xr", "scale_level",
                      "view_cos", "depth", "desc"):
                setattr(mv, k, e["d_mps"][b][k].data_ptr())
            Ms.append(mv)
        a1 = [self.d_assign_last.data_ptr() + 4 * b * self.cap for b in range(self.B)]
        a2 = [self.d_assign_local.data_ptr() + 4 * b * self.cap for b in range(self.B)]
        self._dev_views[p] = (curs, lasts, Fs, Ms, a1, a2)
        return self._dev_views[p]

    def enable_side_streams(self, main_stream):
        """The two projection matchers only depend on the extraction, not on each other: give each
        its own stream so their latency-bound kernels overlap (joined back before the next step)."""
        torch = self.torch
        self.main_stream = main_stream
        self.side = (torch.cuda.Stream(), torch.cuda.Stream())
        self._match_done = {}
        self.m_last.set_stream(self.side[0].cuda_stream)
        self.m_local.set_stream(self.side[1].cuda_stream)

    def step_device(self, i):
        p = i % self.POOL
        d = self.dev_pool[p]
        side = getattr(self, "side", None)
        if side:
            # the extractor's results are double-buffered: this extraction overwrites the set the matchers of
            # step i-2 read (their end was recorded then), while the matchers of step i-1 may still be running
            done = self._match_done.pop(i - 2, None)
            if done:
                for ev in done:
                    self.main_stream.wait_event(ev)
        self.ext.extract_batch_device(d.data_ptr(), self.B, H, W, W, H * W, stream=self.stream)
        curs, lasts, Fs, Ms, a1, a2 = self._device_views(p)
        if side:
            for st in side:
                st.wait_stream(self.main_stream)
        r1, _ = self.m_last.project_last_batch(curs, lasts, self.meta[p]["T"], TH_LAST, on_device=True,
                                               assign_ptrs=a1)
        r2, _ = self.m_local.project_local_batch(Fs, Ms, TH_LOCAL, on_device=True, assign_ptrs=a2)
        if side:
            evs = []
            for st in side:
                ev = self.torch.cuda.Event()
                ev.record(st)
                evs.append(ev)
            self._match_done[i] = evs
        self.nmatch_last, self.nmatch_local = r1, r2  # filled when the asynchronous batches complete

    def finish_device(self):
        self.m_last.synchronize()
        self.m_local.synchronize()
        side = getattr(self, "side", None)
        if side:  # the timed region ends on the main stream: join the matcher streams into it
            for st in side:
                self.main_stream.wait_stream(st)

    def step_host(self, i):
        from orb_slam3_b200._lib import check, ptr
        from orb_slam3_b200.views import orb_frame_view
        p = i % self.POOL
        t = self.host_pool[p]
        B, cap = self.B, self.cap
        arr = (C.c_void_p * B)(*[t.data_ptr() + b * H * W for b in range(B)])
        check(self.ext._lib.orb_extract_batch(self.ext._h, B, arr, H, W, W, None, C.c_void_p(self.out_k.data_ptr()),
                                              C.c_void_p(self.out_d.data_ptr()), cap, ptr(self.out_n),
                                              ptr(self.out_m)))
        e = self.meta[p]
        kp, ds, _, _, dcap = self.ext.device_results()
        key = (p, kp)
        if key not in self._host_views:
            # the keypoints / descriptors were downloaded for the caller above; the matchers read the
            # extractor's device copy (on_device = 2) instead of uploading them again.  The views only differ
            # from step to step in n, so they are built once per (batch, result buffer)
            curs, Fs = [], []
            for b in range(B):
                for src, lst in ((e["cur"][b], curs), (e["F"][b], Fs)):
                    v = orb_frame_view()
                    C.memmove(C.byref(v), C.byref(src), C.sizeof(v))
                    v.keys = kp + b * dcap * 28
                    v.desc = ds + b * dcap * 32
                    v.u_right = None
                    lst.append(v)
            self._host_views[key] = (curs, Fs)
        curs, Fs = self._host_views[key]
        for b in range(B):
            curs[b].n = Fs[b].n = int(self.out_n[b])
        r1, _ = self.m_last.project_last_batch(curs, e["last"], e["T"], TH_LAST, on_device=2)
        r2, _ = self.m_local.project_local_batch(Fs, e["mps"], TH_LOCAL, on_device=2)
        self.nmatch_last, self.nmatch_local = r1, r2

    def e2e_bytes(self):
        e = self.meta[0]
        h2d = self.B * H * W
        d2h = int(self.B * (NFEAT + 4 * NLEVELS) * 60 + 8 * self.B)
        for b in range(self.B):
            n = e["n"][b]
            h2d += 2 * n * 1 + e["last"][b].n * 50 + e["mps"][b].n * 59   # kp_taken only: keys / desc stay on the device
            d2h += 2 * n * 4
        return h2d, d2h


DUMP_BYTES = 64 * 10**6


def dump_outputs(wl, step, out_dir):
    """Write what step `step` of the device-resident loop handed back, per frame of its batch: the keypoints and
    descriptors of the extraction, the assignments and match counts of both projection matchers.  Per-keypoint
    arrays are the frames' rows one after the other (keypoints_per_frame gives the split).  Integers and bytes are
    stored as float32, which holds them exactly.  A batch whose outputs could exceed DUMP_BYTES is represented by a
    fixed (seed 0) sample of its frames, listed in frames.npy."""
    p = step % wl.POOL
    e = wl.meta[p]
    per_frame = wl.cap * (6 + 32 + 2) * 4 + 5 * 4
    max_frames = (DUMP_BYTES - 4096) // per_frame   # 4096: the .npy headers
    frames = np.arange(wl.B)
    if wl.B > max_frames:
        frames = np.sort(np.random.default_rng(0).choice(wl.B, max_frames, replace=False))
    assign_last = wl.d_assign_last.cpu().numpy()
    assign_local = wl.d_assign_local.cpu().numpy()
    kps, desc, mono, n_kp, a_last, a_local = [], [], [], [], [], []
    for b in frames:
        m, k, d = wl.ext.download_results(int(b))
        mono.append(m)
        n_kp.append(len(k))
        kps.append(np.stack([k[f].astype(np.float32) for f in ("x", "y", "size", "angle", "response", "octave")], 1))
        desc.append(d.astype(np.float32))
        a_last.append(assign_last[b, :e["n"][b]])     # the matchers' frame views hold e["n"][b] keypoints
        a_local.append(assign_local[b, :e["n"][b]])
    out = {"frames": frames, "mono_index": mono, "keypoints_per_frame": n_kp,
           "keypoints": np.concatenate(kps), "descriptors": np.concatenate(desc),
           "assign_last": np.concatenate(a_last), "assign_local": np.concatenate(a_local),
           "matches_last": wl.nmatch_last[frames], "matches_local": wl.nmatch_local[frames]}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float32))


def run_lba_gpu(rank, world, device):
    """LocalBA on the GPU: configs 4 and 5 at N=1, config 5 sharded by landmark for N>1 (one ncclAllReduce of the
    envelope of [S | b_s] per LM trial).  `value` = LM trials / device time of optimize(10); `e2e` = the same count
    over the host wall time of the C-ABI call (edge sort, CSR / pair lists, ordering, H2D, kernels, D2H).  At N>1
    rank 0 also solves the unsharded graph and reports whether the sharded solve reproduces it."""
    import ctypes as C
    import torch
    import torch.distributed as dist
    from orb_slam3_b200 import _lib, scenes
    from orb_slam3_b200.optimizer import LocalBundleAdjustment
    out = {}
    lba = LocalBundleAdjustment(device=device)
    configs = [("config4", 50, 20000), ("config5", 200, 80000)] if world == 1 else [("config5", 200, 80000)]
    if world > 1:
        uid = [LocalBundleAdjustment.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        lba.init_comm(rank, world, uid[0])
    peak = C.c_double(0.0)
    fp64_peak = None
    if rank == 0 and _lib.lib().lba_measure_fp64_mma_peak(device, 10, C.byref(peak)) == 0:
        fp64_peak = peak.value
    tensor_pct = None
    try:
        tensor_pct = json.load(open(os.path.join(ROOT, "profiles", "schur_pairs_r2.json")))["sm__pipe_tensor_cycles_active_pct"]
    except Exception:
        pass
    for name, K, L in configs:
        g, _ = scenes.lba_graph(K, L, seed=0)
        sub, lm_ids, _ = (g, None, None) if world == 1 else scenes.shard_graph(g, rank, world)
        gv = scenes.lba_view(sub)
        best, res = None, None
        for rep in range(4):  # the first run warms up allocations
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            r = lba(gv)
            st = r["stats"]
            if rep > 0 and (best is None or st["ms_total"] < best["ms_total"]):
                best, res = st, r
        ms = torch.tensor([best["ms_total"], best["ms_wall"]], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms_total, ms_wall = (float(v) for v in ms.tolist())
        schur_tf = best["schur_flops"] * best["trials"] / max(best["ms_schur"], 1e-9) / 1e9   # TFLOP/s (useful, block-sparse)
        entry = {
            "config": "%d KF x %d landmarks, %d edges%s" % (K, L, len(g["e_kf"]),
                                                            "" if world == 1 else ", landmark shards + ncclAllReduce"),
            "iterations": best["iterations"], "trials": best["trials"], "ms_total": ms_total,
            "value": best["trials"] / (ms_total * 1e-3), "unit": "LM iterations/s",
            "e2e": {"value": best["trials"] / (ms_wall * 1e-3), "unit": "LM iterations/s", "ms_wall": ms_wall,
                    "ms_host_prep": best["ms_host_prep"],
                    "h2d_bytes": int(len(sub["e_kf"]) * 45 + len(sub["mp_pos"]) * 24 + len(g["kf_fixed"]) * 77),
                    "d2h_bytes": int(len(sub["e_kf"]) * 9 + len(sub["mp_pos"]) * 24 + len(g["kf_fixed"]) * 56)},
            "chi2_initial": best["chi2_initial"], "chi2_final": best["chi2_final"],
            "stage_ms": {k: best[k] for k in ("ms_linearize", "ms_schur", "ms_solve", "ms_update")},
            "reduced_solver": {0: "dense cooperative LDLT", 1: "envelope LDLT (32-column panels, one CTA)",
                               2: "window-resident envelope LDLT (8-column panels, one CTA)",
                               3: "window-resident envelope LDLT from both ends (two CTAs + dense separator block)"}[best["solver_kind"]],
            "envelope_rows_max": best["envelope_rows_max"],
            "schur_gflops_sparse": 1e3 * schur_tf,
            "roofline": {"bound": "tensor", "kernel": "schur_pairs_kernel (fp64 DMMA m8n8k4)", "achieved": schur_tf,
                         "peak": fp64_peak, "unit": "TFLOP/s", "frac": (schur_tf / fp64_peak) if fp64_peak else None,
                         "peak_source": "measured in this run: DMMA m8n8k4 from registers, full grid, best of 10 (lba_measure_fp64_mma_peak)",
                         "tensor_pipe_pct": tensor_pct,
                         "flops": "block-sparse useful flops per trial (SURVEY.md 8d) x trials / time between the Schur events"},
            "n_pose_pairs": best["n_pairs"],
            "allreduce_bytes_per_trial": best["allreduce_bytes_per_trial"],
        }
        if world > 1:
            # NCCL parity carried by the scaling run itself: rank 0 solves the unsharded graph on its own GPU
            flag = torch.zeros(3, dtype=torch.float64, device="cuda")
            if rank == 0:
                single = LocalBundleAdjustment(device=device)(scenes.lba_view(g))
                dpose = float(np.abs(single["kf_pose"] - res["kf_pose"]).max())
                dpts = float(np.abs(single["mp_pos"][lm_ids] - res["mp_pos"]).max())
                same_counts = (single["iterations"] == res["iterations"] and
                               single["stats"]["trials"] == res["stats"]["trials"])
                flag = torch.tensor([1.0 if (same_counts and dpose < 1e-7 and dpts < 1e-6) else 0.0, dpose, dpts],
                                    dtype=torch.float64, device="cuda")
            dist.broadcast(flag, src=0)
            entry["sharded_equals_single"] = bool(flag[0].item() == 1.0)
            entry["max_abs_dpose_vs_single"] = float(flag[1].item())
            entry["max_abs_dpoint_vs_single"] = float(flag[2].item())
        out[name] = entry
    return out


def run_stereo_gpu(rank, world, device, tstream, pairs=64, reps=5, cpu=True):
    """BASELINE.json configs[2] (SURVEY.md 8d config 3, rows 8f-1 + a12): one stereo camera stream per rank / GPU.
    A step = `pairs` rectified 1280x720 stereo pairs of this rank's stream: both eyes extracted by their own
    handle, Frame::ComputeStereoMatches on the device-resident results, then SearchForTriangulation between
    consecutive left keyframes (synthetic FeatureVectors, ~1000 nodes) through the host-buffer batch call.
    Weak scaling: every rank runs its own stream; value = all pairs / max-over-ranks time."""
    import torch
    import torch.distributed as dist
    from orb_slam3_b200 import scenes
    from orb_slam3_b200.extractor import ORBextractor
    from orb_slam3_b200.matcher import ORBmatcher
    from orb_slam3_b200.stereo import StereoMatcher
    from orb_slam3_b200.synth import stereo_right
    bf, b = 386.0, 386.0 / 700.0
    uniq = 16
    lefts, shifts = make_frames(uniq + 1, 9000 + 1000 * rank)
    rights = [stereo_right(l, 9100 + 17 * rank + i, disparities=(6, 24, 12)) for i, l in enumerate(lefts)]
    idx = [1 + i % uniq for i in range(pairs)]
    dl = torch.from_numpy(np.stack([lefts[i] for i in idx])).cuda()
    dr = torch.from_numpy(np.stack([rights[i] for i in idx])).cuda()
    el = ORBextractor(NFEAT, 1.2, NLEVELS, 20, 7, device=device)
    er = ORBextractor(NFEAT, 1.2, NLEVELS, 20, 7, device=device)
    sm = StereoMatcher(device)
    tri = ORBmatcher(0.6, False, device=device)      # LocalMapping.cc:466: ORBmatcher matcher(0.6, false)
    cs = tstream.cuda_stream
    # triangulation inputs: keyframe pairs (frame i, its predecessor) from one untimed extraction of the left stream
    feats = el.extract_batch(list(lefts))
    tri_in = {}
    for i in range(1, uniq + 1):
        _, k2, d2 = feats[i]
        _, k1, d1 = feats[i - 1]
        tri_in[i] = scenes.triangulation_scene(k1, d1, k2, d2, W, H, seed=31 * i, n_nodes=1000, shift=shifts[i])
    targs = [[tri_in[i][j] for i in idx] for j in range(6)]

    def step():
        el.extract_batch_device(dl.data_ptr(), pairs, H, W, W, H * W, stream=cs)
        er.extract_batch_device(dr.data_ptr(), pairs, H, W, W, H * W, stream=cs)
        sm.compute_batch(el, er, pairs, bf, b, on_device=True, cuda_stream=cs)

    for _ in range(3):
        step()
    n_tri, _ = tri.triangulate_batch(*targs)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(reps):
        step()
    e1.record()
    ms_tri_dev = 0.0
    for _ in range(reps):   # SearchForTriangulation of the same keyframes (host views -> H2D -> kernels -> D2H pair lists)
        n_tri, _ = tri.triangulate_batch(*targs)
        ms_tri_dev += tri.last_ms()
    torch.cuda.synchronize()
    ms_wall = (time.perf_counter() - t0) * 1e3 / reps
    ms_all = e0.elapsed_time(e1) / reps
    ms_tri_dev /= reps
    ms_match = 0.0
    for _ in range(reps):  # the stereo matcher alone, device time between its own events
        sm.compute_batch(el, er, pairs, bf, b, on_device=True, cuda_stream=cs)
        ms_match += sm.last_ms()
    ms_match /= reps
    kept, ur, dp = sm.compute_batch(el, er, pairs, bf, b)
    t = torch.tensor([ms_all + ms_tri_dev, ms_wall], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev_max, ms_wall_max = (float(v) for v in t.tolist())
    out = {"config": "configs[2]: %d stereo streams (one per GPU) x %d pairs 1280x720 per step, 2000 features per eye, "
                     "disparity bands 6/24/12 px, %d distinct pairs per stream; + SearchForTriangulation per keyframe pair"
                     % (world, pairs, uniq),
           "value": world * pairs / (ms_dev_max * 1e-3), "unit": "stereo pairs/s (2 x extract + ComputeStereoMatches + SearchForTriangulation), device time, max over ranks",
           "e2e_value": world * pairs / (ms_wall_max * 1e-3),
           "e2e_unit": "stereo pairs/s, host wall clock (frames resident; triangulation through host buffers)",
           "n_gpus": world, "scaling": "weak",
           "pairs_per_s": pairs / (ms_all * 1e-3), "ms_per_step": ms_all,
           "stereo_match_us_per_pair": 1e3 * ms_match / pairs, "matches_per_pair": float(kept.mean()),
           "triangulate_us_per_kf_pair": 1e3 * ms_tri_dev / pairs, "triangulation_pairs_per_kf_pair": float(n_tri.mean()),
           "gpu_launches_per_step": 3 + int(tri.kernel_launches() // (reps + 1))}
    if cpu and rank == 0:
        from oracle import oracle as O
        exl, exr = O.OracleExtractor(NFEAT), O.OracleExtractor(NFEAT)
        t0 = time.perf_counter()
        kl, d1, _ = exl.extract(lefts[1])
        kr, d2, _ = exr.extract(rights[1])
        t_ext = time.perf_counter() - t0
        pl = [exl.level_image(l) for l in range(NLEVELS)]
        pr = [exr.level_image(l) for l in range(NLEVELS)]
        t0 = time.perf_counter()
        for _ in range(5):
            n_ref, ur_ref, dp_ref, _ = O.stereo_match(kl, d1, kr, d2, pl, pr, bf, b)
        t_sm = (time.perf_counter() - t0) / 5
        a1 = tri_in[1]
        t0 = time.perf_counter()
        for _ in range(5):
            n_tref, p_tref = O.match_triangulate(*a1, False, False, False)
        t_tri = (time.perf_counter() - t0) / 5
        n0 = len(kl)
        got_n, got_p = tri.triangulate_batch(*[[a1[j]] for j in range(6)])
        out["cpu_baseline"] = {"stereo_match_ms_per_pair": 1e3 * t_sm, "extract2_ms_per_pair": 1e3 * t_ext,
                               "triangulate_ms_per_kf_pair": 1e3 * t_tri, "threads": 1, "kind": "port",
                               "parity_pair0": bool(np.array_equal(ur[0, :n0], ur_ref) and np.array_equal(dp[0, :n0], dp_ref)),
                               "parity_triangulation0": bool(int(got_n[0]) == n_tref and np.array_equal(got_p[0], p_tref))}
    return out


def run_pose_gpu(device, frames=128, edges=1000, reps=5, cpu=True):
    """SURVEY.md 8(f-2): `frames` independent Optimizer::PoseOptimization problems (one per tracked frame,
    `edges` matched MapPoints each, 80 % stereo, 10 % gross mismatches) per step, one kernel launch."""
    from orb_slam3_b200 import scenes
    from orb_slam3_b200.optimizer import PoseOptimization
    po = PoseOptimization(device)
    uniq = 16
    base = [scenes.pose_scene(edges, seed=100 + i)[0] for i in range(uniq)]
    views = [base[i % uniq] for i in range(frames)]
    po.batch(views)
    ms_dev, t0 = 0.0, time.perf_counter()
    for _ in range(reps):
        inl, pose, outs, stats = po.batch(views)
        ms_dev += po.last_ms()
    ms_wall = (time.perf_counter() - t0) * 1e3 / reps
    ms_dev /= reps
    out = {"config": "%d frames x %d edges (80%% stereo, 10%% mismatches), 4 rounds x optimize(10)" % (frames, edges),
           "value": frames / (ms_dev * 1e-3), "unit": "PoseOptimization calls/s (kernel, CUDA events)",
           "e2e_value": frames / (ms_wall * 1e-3), "e2e_unit": "calls/s through the host-buffer C ABI (H2D + kernel + D2H)",
           "ms_per_step": ms_dev, "gpu_launches_per_step": 1,
           "lm_trials_per_frame": float(stats[:, 2].mean()), "inliers_per_frame": float(inl.mean())}
    if cpu:
        from oracle import oracle as O
        t0 = time.perf_counter()
        refs = [O.pose_optimize(v) for v in base]
        t_cpu = (time.perf_counter() - t0) / uniq
        ok = all(np.array_equal(outs[i], refs[i]["outlier"]) and
                 np.abs(pose[i] - refs[i]["pose"]).max() < 1e-7 for i in range(uniq))
        out["cpu_baseline"] = {"ms_per_call": 1e3 * t_cpu, "threads": 1, "kind": "port", "parity_first_%d" % uniq: bool(ok)}
    return out


def run_frustum_gpu(device, cpu=True):
    """SURVEY.md 8(f-3): Frame::isInFrustum over the local map of one frame (5000 points, the
    Tracking::SearchLocalPoints shape) and over 2^20 points (streaming rate of the kernel)."""
    from orb_slam3_b200 import scenes
    from orb_slam3_b200.frustum import FrustumCuller
    fc = FrustumCuller(device)
    out = {}
    for name, n, reps in (("local_map_5000", 5000, 20), ("stream_1M", 1 << 20, 5)):
        v, _ = scenes.frustum_scene(n, seed=3)
        k, o = fc.isInFrustum(v)
        ms_dev, t0 = 0.0, time.perf_counter()
        for _ in range(reps):
            k, o = fc.isInFrustum(v, out=o)
            ms_dev += fc.last_ms()
        ms_wall = (time.perf_counter() - t0) * 1e3 / reps
        ms_dev /= reps
        e = {"points": n, "in_view": int(k), "kernel_us": 1e3 * ms_dev, "host_call_us": 1e3 * ms_wall,
             "kernel_GBps_algorithmic": n * 57 / (ms_dev * 1e-3) / 1e9, "bytes_per_point": 57}
        if cpu:
            from oracle import oracle as O
            t0 = time.perf_counter()
            for _ in range(3):
                k_ref, ref = O.is_in_frustum(v)
            e["cpu_port_us"] = (time.perf_counter() - t0) / 3 * 1e6
            e["parity"] = bool(k_ref == k and all(np.array_equal(o[f], ref[f]) for f in ref))
        out[name] = e
    return out


def run_bow_gpu(device, cpu=True):
    """SURVEY.md 8(f-4): Frame::ComputeBoW = DBoW2 transform(levelsup 4) of one frame's 2000 descriptors
    against a resident synthetic 10-ary depth-5 vocabulary (the ORB vocabulary is 10-ary, depth 6)."""
    from orb_slam3_b200 import scenes
    from orb_slam3_b200.bow import ORBVocabulary
    from orb_slam3_b200.extractor import ORBextractor
    from orb_slam3_b200.synth import synth_frame
    voc = scenes.synth_vocabulary(10, 5, seed=3)
    gv = ORBVocabulary(voc, device)
    ext = ORBextractor(NFEAT, 1.2, NLEVELS, 20, 7, device=device)
    _, kps, desc = ext(synth_frame(H, W, 4242))
    got = gv.transform_extracted(ext, 0, 4)
    reps, ms_dev, t0 = 20, 0.0, time.perf_counter()
    for _ in range(reps):
        got = gv.transform_extracted(ext, 0, 4)
        ms_dev += gv.last_ms()
    ms_wall = (time.perf_counter() - t0) * 1e3 / reps
    out = {"config": "%d descriptors, vocabulary %d nodes (k=10, L=5), levelsup 4" % (len(desc), voc.n_nodes),
           "kernels_us": 1e3 * ms_dev / reps, "call_us_descriptors_on_device": 1e3 * ms_wall, "gpu_launches_per_call": 2,
           "words": int(len(got["bow_ids"])), "fv_nodes": int(len(got["fv_node_ids"]))}
    if cpu:
        from oracle import oracle as O
        t0 = time.perf_counter()
        for _ in range(3):
            ref = O.bow_transform(voc, desc, 4)
        out["cpu_port_us"] = (time.perf_counter() - t0) / 3 * 1e6
        out["parity"] = bool(all(np.array_equal(got[k], ref[k]) for k in ("bow_ids", "bow_vals", "fv_node_ids", "fv_ptr", "fv_idx")))
    return out


def run_latency_gpu(device, cpu=True, reps=30):
    """Batch-1 latency of the calls the Tracking thread makes once per frame, through the host-buffer C ABI
    (wall clock around the call: H2D + kernels + D2H + sync), median of `reps`, beside the CPU port on one thread."""
    from orb_slam3_b200 import scenes
    from orb_slam3_b200.extractor import ORBextractor
    from orb_slam3_b200.matcher import ORBmatcher
    from orb_slam3_b200.optimizer import PoseOptimization
    from orb_slam3_b200.stereo import StereoMatcher
    from orb_slam3_b200.synth import stereo_right
    frames, shifts = make_frames(3, 777)
    right = stereo_right(frames[1], 778, disparities=(6, 24, 12))
    ext = ORBextractor(NFEAT, 1.2, NLEVELS, 20, 7, device=device)
    ext_r = ORBextractor(NFEAT, 1.2, NLEVELS, 20, 7, device=device)
    m_last, m_local = ORBmatcher(0.9, True, device=device), ORBmatcher(0.8, True, device=device)
    po, sm = PoseOptimization(device), StereoMatcher(device)
    _, ka, da = ext(frames[0])
    _, kb, db = ext(frames[1])
    cur, last, Tcw = scenes.last_frame_scene(ka, da, kb, db, W, H, shifts[1], seed=5)
    F, mps = scenes.local_map_scene(kb, db, W, H, N_LOCAL_EXTRA, seed=6)
    pv, _ = scenes.pose_scene(1000, seed=8)
    ext_r(right)
    bf, b = 386.0, 386.0 / 700.0

    def med(fn):
        fn(); fn()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        return 1e6 * float(np.median(ts))

    out = {"unit": "microseconds per call, batch 1, host buffers in and out (median of %d)" % reps,
           "orb_extract_1280x720": {"gpu_us": med(lambda: ext(frames[1]))},
           "match_project_last": {"gpu_us": med(lambda: m_last.SearchByProjectionLast(cur, last, Tcw, TH_LAST))},
           "match_project_local": {"gpu_us": med(lambda: m_local.SearchByProjection(F, mps, TH_LOCAL))},
           "pose_optimize_1000_edges": {"gpu_us": med(lambda: po(pv))},
           "stereo_match": {"gpu_us": med(lambda: sm.ComputeStereoMatches(ext, ext_r, len(kb), bf, b))}}
    if cpu:
        from oracle import oracle as O
        ex, exr = O.OracleExtractor(NFEAT), O.OracleExtractor(NFEAT)
        out["orb_extract_1280x720"]["cpu_port_us"] = med(lambda: ex.extract(frames[1]))
        out["match_project_last"]["cpu_port_us"] = med(lambda: O.match_project_last(cur, last, Tcw, TH_LAST))
        out["match_project_local"]["cpu_port_us"] = med(lambda: O.match_project_local(F, mps, TH_LOCAL, 0.8))
        out["pose_optimize_1000_edges"]["cpu_port_us"] = med(lambda: O.pose_optimize(pv))
        kl, dl_, _ = ex.extract(frames[1])
        kr, dr_, _ = exr.extract(right)
        pl = [ex.level_image(l) for l in range(NLEVELS)]
        pr = [exr.level_image(l) for l in range(NLEVELS)]
        out["stereo_match"]["cpu_port_us"] = med(lambda: O.stereo_match(kl, dl_, kr, dr_, pl, pr, bf, b))
        for v in out.values():
            if isinstance(v, dict) and "cpu_port_us" in v:
                v["speedup_vs_one_cpu_thread"] = v["cpu_port_us"] / v["gpu_us"]
    return out


def _guarded(fn, *a, **k):
    """The extra legs must never cost the headline line."""
    try:
        return fn(*a, **k)
    except Exception as e:  # noqa: BLE001
        return {"error": "%s: %s" % (type(e).__name__, e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--batch", type=int, default=128, help="frames per step per GPU")
    ap.add_argument("--pool", type=int, default=2, help="distinct batches rotated through (L2 defeat); 2 x 128 = the 256 distinct frames")
    ap.add_argument("--e2e-workers", type=int, default=4, help="host threads feeding the GPU in the e2e leg")
    ap.add_argument("--no-lba", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-stereo", action="store_true", help="skip the 8(f) legs (ComputeStereoMatches, PoseOptimization, isInFrustum, ComputeBoW)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; --impl reference has none")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # stdout carries exactly one JSON line: libraries that write to fd 1 (NCCL prints its version banner
    # there) are pointed at stderr, the line itself goes to a duplicate of the original stdout
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: orb_slam3_b200 has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        # NUMA: keep this rank's host threads (and the first touch of its pinned buffers) on the CPUs next to its GPU
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[local_rank]) if vis and vis.split(",")[local_rank].isdigit() else local_rank
            words = pynvml.nvmlDeviceGetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(phys), (os.cpu_count() + 63) // 64)
            cpus = {64 * w + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1}
            if cpus:
                os.sched_setaffinity(0, cpus & os.sched_getaffinity(0) or cpus)
        except Exception:
            pass
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    B, K, Wm, POOL = args.batch, args.steps, max(args.warmup, 3), args.pool

    tstream = torch.cuda.Stream()  # non-default stream: the engines launch where the events are recorded
    torch.cuda.set_stream(tstream)
    wl = Workload(B, POOL, rank, local_rank, tstream.cuda_stream)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def launches_now():
        return wl.ext.kernel_launches() + wl.m_last.kernel_launches() + wl.m_local.kernel_launches()

    # ---- device-resident metric (matcher batches are asynchronous: the host prepares the next
    # submission while the GPU works; everything is ordered on one stream)
    for m in (wl.m_last, wl.m_local):
        m.set_async(True)
    wl.enable_side_streams(tstream)
    for i in range(Wm):
        wl.step_device(i)
    wl.finish_device()
    launches0 = launches_now()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        wl.step_device(i)
    e1.record()
    wl.finish_device()
    barrier()
    ms_dev = e0.elapsed_time(e1)
    launches = launches_now() - launches0
    nm_last, nm_local = int(wl.nmatch_last.sum()), int(wl.nmatch_local.sum())
    if args.dump_outputs and rank == 0:
        dump_outputs(wl, K - 1, args.dump_outputs)
    # ---- end to end through the host-buffer ABI (wall clock brackets every copy and sync).
    # Batches come from independent camera streams, so `--e2e-workers` host threads (each with its
    # own extractor + matcher handles, i.e. its own CUDA streams) work on different batches at once:
    # one batch's PCIe copies and host staging overlap another batch's kernels.
    from concurrent.futures import ThreadPoolExecutor
    for m in (wl.m_last, wl.m_local):
        m.set_async(False)
    workers = [wl] + [Workload(B, POOL, rank, local_rank, None, share=wl) for _ in range(args.e2e_workers - 1)]
    for w in workers[1:]:
        for m in (w.m_last, w.m_local):
            m.set_stream(None)
    for m in (wl.m_last, wl.m_local):
        m.set_stream(None)
    pool_exec = ThreadPoolExecutor(len(workers))

    def run_host_steps(k):
        def work(widx):
            torch.cuda.set_device(local_rank)
            for i in range(widx, k, len(workers)):
                workers[widx].step_host(i)
        list(pool_exec.map(work, range(len(workers))))

    run_host_steps(max(Wm, len(workers)))
    barrier()
    t0 = time.perf_counter()
    run_host_steps(K)
    barrier()
    ms_e2e = (time.perf_counter() - t0) * 1e3
    for m in (wl.m_last, wl.m_local):
        m.set_stream(tstream.cuda_stream)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    nkp = int(wl.out_n.sum())

    # ---- per-kernel times for the roofline (events around each launch; separate pass)
    wl.ext.set_profiling(True)
    wl.ext.stage_times(reset=True)
    ms_match = [0.0, 0.0]
    for m in (wl.m_last, wl.m_local):
        m.set_async(False)
        m.set_stream(tstream.cuda_stream)
    wl.side = None
    for i in range(K):
        wl.step_device(i)
        ms_match[0] += wl.m_last.last_ms()
        ms_match[1] += wl.m_local.last_ms()
    wl.ext.synchronize()
    st = wl.ext.stage_times(reset=True)
    wl.ext.set_profiling(False)

    tens = torch.tensor([ms_dev, ms_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tens, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e = tens.tolist()

    lba = None
    if not args.no_lba:
        lba = run_lba_gpu(rank, world, local_rank)
    stereo = None
    if not args.no_stereo:   # configs[2]: every rank runs its own stereo stream
        stereo = run_stereo_gpu(rank, world, local_rank, tstream, cpu=(world == 1 and not args.no_cpu))
    pose = None
    if rank == 0 and not args.no_stereo:
        pose = _guarded(run_pose_gpu, local_rank, cpu=(world == 1 and not args.no_cpu))
    frustum = None
    if rank == 0 and not args.no_stereo:
        frustum = _guarded(run_frustum_gpu, local_rank, cpu=(world == 1 and not args.no_cpu))
    bow = None
    if rank == 0 and not args.no_stereo:
        bow = _guarded(run_bow_gpu, local_rank, cpu=(world == 1 and not args.no_cpu))
    latency = None
    if rank == 0 and not args.no_stereo:
        latency = _guarded(run_latency_gpu, local_rank, cpu=(world == 1 and not args.no_cpu))
    if world > 1:
        dist.barrier()

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        P = sum(level_pixels())
        n_mp = NFEAT + N_LOCAL_EXTRA
        # algorithmic bytes per frame and per kernel (DESIGN.md "Kernels")
        alg = {
            "pyramid": W * H + (P - W * H),           # read level 0, write levels 1..7
            "fast": P,                                # one read of the pyramid
            "blur": 2 * P,                            # read + write blurred pyramid
            "octree": 38000 * 8,                      # candidate records in
            "describe": NFEAT * (28 + 32) + NFEAT * (31 * 31 + 512),
        }
        kern = {k: v for k, v in st.items() if k in alg and v[1] > 0}

        def per_launch_ms(k):
            n_l = kern[k][1] if k != "pyramid" else kern[k][1] / (NLEVELS - 1)
            return kern[k][0] / n_l

        dom = max(kern, key=lambda k: kern[k][0])
        achieved = alg[dom] * B / (per_launch_ms(dom) * 1e-3) / 1e9
        total_ms = sum(v[0] for v in kern.values()) + sum(ms_match)
        traffic = None
        try:  # DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture
            tp = os.path.join(ROOT, "profiles", "fast_traffic_r2.json")
            tr = json.load(open(tp if os.path.exists(tp) else os.path.join(ROOT, "profiles", "fast_cells_traffic_r1.json")))
            if dom == "fast":
                traffic = tr["dram_bytes_per_launch"] * B / tr["batch"]
        except Exception:
            pass
        fps_dev = world * B * K / (ms_dev * 1e-3)
        fps_e2e = world * B * K / (ms_e2e * 1e-3)
        stage = {k: v[0] / K for k, v in st.items()}
        stage["match_last(th15)"] = ms_match[0] / K
        stage["match_local(th3)"] = ms_match[1] / K
        per_kernel = {}
        for k in kern:
            gbs = alg[k] * B / (per_launch_ms(k) * 1e-3) / 1e9
            per_kernel[k] = {"GB/s": gbs, "frac_of_hbm": gbs / hbm_peak}
        b_match = (NFEAT + n_mp) * 32 + NFEAT * 16 + n_mp * 24 + 64 * 48 * 4 + NFEAT * 4
        gbs = b_match * B / (max(ms_match[1], 1e-9) / K * 1e-3) / 1e9
        per_kernel["match_local"] = {"GB/s": gbs, "frac_of_hbm": gbs / hbm_peak}
        cpu = None
        if world == 1 and not args.no_cpu:
            from oracle import oracle as O
            O.build()
            threads = best_cpu_threads()
            fps_cpu, done, dt = cpu_extract_fps(wl.uniq[:8], threads, seconds_budget=8.0)
            fps_1, _, _ = cpu_extract_fps(wl.uniq[:8], 1, seconds_budget=3.0)
            t_match = cpu_match_seconds_per_frame(*make_frames(4, 1))
            t_ext = threads / fps_cpu
            kind = cpu_extractor()[1]
            cpu = {"value": threads / (t_ext + t_match), "unit": "frames/s", "cores": threads, "kind": kind,
                   "sample": "extract (%s): %d frames over %d std::threads in %.1fs (%.1f frames/s; 1 thread %.1f frames/s); "
                             "match: %.2f ms/frame/thread (oracle C++ port, one thread); value = threads / (extract + match): "
                             "a composition of the two measurements; the image primitives under the reference code are the "
                             "scalar cv2-pinned ones, OpenCV's SIMD FAST/resize/blur would be several times faster"
                             % ("reference ORBextractor.cc object code, oracle/_ref" if kind == "reference" else "oracle C++ port",
                                done, threads, dt, fps_cpu, fps_1, 1e3 * t_match)}
            if lba is not None:
                lba["cpu_baseline_config4"] = cpu_lba(50, 20000)
                lba["config4_fisheye_rig"] = _guarded(lba_rig_leg, local_rank)
        h2d, d2h = wl.e2e_bytes()
        line = {
            "metric": METRIC, "value": fps_dev, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_step_per_gpu": B,
                       "distinct_frames_per_gpu": wl.n_distinct, "streams_per_gpu": N_STREAMS,
                       "l2": "inputs+pyramids %.0f MB per rotation > 126 MB L2 (%d batches rotated)"
                             % (POOL * B * (W * H + 2 * P) / 1e6, POOL),
                       "keypoints_last_step": nkp, "matches_last_step": {"last": nm_last, "local": nm_local}},
            "e2e": {"value": fps_e2e, "unit": "frames/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "host_threads": args.e2e_workers},
            "gpu_launches": int(launches),
            "clocks": sampler.summary(),
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                         "frac": achieved / hbm_peak, "traffic": traffic, "algorithmic_bytes_per_launch": alg[dom] * B,
                         "peak_source": peak_src,
                         "share_of_step": kern[dom][0] / total_ms, "stage_ms_per_step": stage,
                         "per_kernel": per_kernel},
            "cpu_baseline": cpu,
            "lba": lba,
            "stereo": stereo,
            "pose_optimization": pose,
            "is_in_frustum": frustum,
            "compute_bow": bow,
            "latency_batch1": latency,
        }
        print(json.dumps(line), file=real_stdout, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
