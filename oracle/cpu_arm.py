"""Timed harness of the reference's CPU path on the box's host cores -- used ONLY by bench.py's `cpu_baseline` leg and
`bench.py --impl reference` (this directory is test / measurement infrastructure, never the product).

What runs: per frame of one stream, the reference's front-end calls on cv2 (the OpenCV the reference links: forward + backward
`calcOpticalFlowPyrLK` as IG/tracking/tracking.cc:385-403 calls it) and one `gvinsOptimization` window solve (5 LM iterations, chi-square
culling, 15 iterations; IG/ic_gvins.cc:1130-1239) on the BA PORT (oracle/ba_ref.cpp -- Ceres is neither vendored nor installed, so this
leg is our restatement, compiled `-O3 -march=native` into a temporary directory on the machine that runs it, so that the source
tree is only read; the parity copy keeps `-O2 -ffp-contract=off`).

How it is measured (throughput mode, like the GPU arm: independent streams):
  * one PROCESS per usable core (spawn), each pinned with os.sched_setaffinity to its own core, cv2 / the port single-threaded inside;
  * FIXED work per repetition (n frames = n KLT pairs + n window solves per process), not a time box;
  * all processes start a repetition together (barrier); the repetition's wall time is max(end) - min(start) on CLOCK_MONOTONIC
    (system-wide), frames/s = processes x n / wall;
  * the median over the repetitions is reported, with the per-repetition values, nproc, CPU model and load average."""
from __future__ import annotations

import ctypes as C
import multiprocessing as mp
import os
import pickle
import subprocess
import sys
import tempfile
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def cpu_model() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def build_perf(out_dir: str, verbose: bool = False) -> str:
    """-O3 -march=native copy of the oracle for TIMING (<out_dir>/libicg_oracle_perf.so), built where it runs."""
    out = os.path.join(out_dir, "libicg_oracle_perf.so")
    srcs = [os.path.join(HERE, f) for f in ("klt_ref.c", "detect_ref.c", "clahe_ref.c", "ba_ref.cpp")]
    objs = []
    for s in srcs:
        o = os.path.join(out_dir, os.path.basename(s) + ".o")
        cc = ["g++", "-std=c++17", "-pthread"] if s.endswith(".cpp") else ["gcc", "-std=c11"]
        cmd = cc + ["-O3", "-march=native", "-fPIC", "-fno-fast-math", "-c", s, "-o", o]
        if verbose:
            print(" ".join(cmd))
        subprocess.run(cmd, check=True)
        objs.append(o)
    subprocess.run(["g++", "-shared", "-pthread", "-o", out] + objs + ["-lm"], check=True)
    return out


# ------------------------------------------------------------------------------------------------ worker (one per core)
def _gvins_optimization(oa, olib, prob, threads=1):
    import copy
    p = copy.deepcopy(prob)
    p["gnss_huber"] = 1
    oa.ba_solve(olib, p, 5, threads)
    rc, gc = oa.ba_residual_costs(olib, p)
    std = p["gnss_std"].reshape(-1, 3)
    for g in range(p["n_gnss"]):
        if 2 * gc[g] > 7.815:
            std[g] *= np.sqrt(2 * gc[g] / 7.815)
    p["gnss_std"] = std.reshape(-1)
    p["f_active"][2 * rc > 5.991] = 0
    p["gnss_huber"] = 0
    oa.ba_solve(olib, p, 15, threads)
    return p


def _worker(idx, core, data_path, reps, n_frames, do_ba, barrier, q, perf_so):
    try:
        os.sched_setaffinity(0, {core})
    except OSError:
        pass
    sys.path.insert(0, ROOT)
    data = pickle.load(open(data_path, "rb"))
    frames, pairs, probs = data["frames"], data["pairs"], data["probs"]
    try:
        import cv2
        cv2.setNumThreads(1)
        crit = (cv2.TERM_CRITERIA_COUNT + cv2.TERM_CRITERIA_EPS, 30, 0.01)

        def klt_one(k):
            fa, fb, prev, init = pairs[k % len(pairs)]
            fwd, st, _ = cv2.calcOpticalFlowPyrLK(frames[fa], frames[fb], prev.reshape(-1, 1, 2), init.reshape(-1, 1, 2).copy(), winSize=(21, 21), maxLevel=3,
                                                  criteria=crit, flags=cv2.OPTFLOW_USE_INITIAL_FLOW)
            cv2.calcOpticalFlowPyrLK(frames[fb], frames[fa], fwd, prev.reshape(-1, 1, 2).copy(), winSize=(21, 21), maxLevel=3, criteria=crit,
                                     flags=cv2.OPTFLOW_USE_INITIAL_FLOW)
        klt_kind = "cv2 " + cv2.__version__
    except Exception:  # noqa: BLE001  -- no OpenCV on this box: the C port of the tracker
        klt_kind = "oracle/klt_ref.c"
        klt_one = None
    from tests import oracle_api as oa
    olib = C.CDLL(perf_so)
    oa.declare(olib)
    oa.declare_ba(olib)
    if klt_one is None:
        def klt_one(k):
            fa, fb, prev, init = pairs[k % len(pairs)]
            oa.track_fb(olib, frames[fa], frames[fb], prev, init)
    klt_one(idx)
    if do_ba:
        _gvins_optimization(oa, olib, probs[idx % len(probs)])
    for r in range(reps):
        barrier.wait()
        t0 = time.monotonic()
        for i in range(n_frames):
            klt_one(idx * 131 + r * 17 + i)
        t1 = time.monotonic()
        if do_ba:
            for i in range(n_frames):
                _gvins_optimization(oa, olib, probs[(idx + i) % len(probs)])
        t2 = time.monotonic()
        q.put((idx, r, t0, t1, t2, klt_kind))


def measure(frames, pairs, probs, reps=5, n_frames=8, do_ba=True, max_procs=None):
    """frames: list of u8 images; pairs: list of (fa, fb, prev_pts, init_pts); probs: list of window-problem dicts (oracle layout).
    Returns a dict with the median frames/s over `reps` fixed-work repetitions and the context the judge asked for."""
    cores = sorted(os.sched_getaffinity(0))
    if max_procs:
        cores = cores[:max_procs]
    with tempfile.TemporaryDirectory(prefix="icg_cpu_arm_") as td:
        perf_so = build_perf(td)
        path = os.path.join(td, "inputs.pkl")
        with open(path, "wb") as f:
            pickle.dump(dict(frames=frames, pairs=pairs, probs=probs if do_ba else []), f, protocol=pickle.HIGHEST_PROTOCOL)
        return _measure(cores, perf_so, path, reps, n_frames, do_ba)


def _measure(cores, perf_so, path, reps, n_frames, do_ba):
    """one pinned worker per core; `perf_so` and the pickled inputs at `path` live in measure()'s temporary directory"""
    nproc = len(cores)
    ctx = mp.get_context("spawn")
    barrier, q = ctx.Barrier(nproc), ctx.Queue()
    load0 = os.getloadavg()
    procs = [ctx.Process(target=_worker, args=(i, cores[i], path, reps, n_frames, do_ba, barrier, q, perf_so), daemon=True) for i in range(nproc)]
    for p in procs:
        p.start()
    rows = []
    try:
        import queue
        deadline = time.monotonic() + 900
        while len(rows) < nproc * reps:
            try:
                rows.append(q.get(timeout=2))
            except queue.Empty:
                dead = [p.exitcode for p in procs if p.exitcode not in (None, 0)]
                if dead or time.monotonic() > deadline:
                    raise RuntimeError(f"cpu_arm: worker processes failed (exit codes {dead})") from None
    finally:
        for p in procs:
            p.join(30)
            if p.is_alive():
                p.kill()
    per_rep, klt_rep, ba_rep = [], [], []
    for r in range(reps):
        rr = [x for x in rows if x[1] == r]
        t0, t1, t2 = min(x[2] for x in rr), max(x[3] for x in rr), max(x[4] for x in rr)
        per_rep.append(nproc * n_frames / (t2 - t0))
        klt_rep.append(nproc * n_frames / (t1 - t0))
        if do_ba:  # the solve phase of a process starts when ITS KLT phase ends: rate from the summed busy time
            busy = sum(x[4] - x[3] for x in rr) / nproc
            ba_rep.append(nproc * n_frames / busy)
    value = float(np.median(per_rep))
    return {
        "value": value, "unit": "frames/s", "cores": nproc,
        "kind": ("reference (cv2 KLT: the OpenCV the reference links) + port (BA: oracle/ba_ref.cpp restatement of Ceres LM + DENSE_SCHUR, "
                 "-O3 -march=native; Ceres itself is not installable here)") if do_ba else "reference (cv2 KLT)",
        "sample": f"median of {reps} repetitions; each: {nproc} pinned processes (one per core) x {n_frames} frames "
                  f"(= {n_frames} fwd+bwd LK pairs of 300 pts on 1280x560" + (f" + {n_frames} gvinsOptimization solves K=10 L=300, 5+15 LM its" if do_ba else "")
                  + "), fixed work, wall = max(end) - min(start)",
        "per_repetition": [round(v, 2) for v in per_rep],
        "klt_frames_per_s": float(np.median(klt_rep)), "ba_solves_per_s": float(np.median(ba_rep)) if do_ba else None,
        "klt_impl": rows[0][5], "nproc": nproc, "cpu_model": cpu_model(), "loadavg_before": [round(v, 2) for v in load0],
        "loadavg_after": [round(v, 2) for v in os.getloadavg()],
    }
