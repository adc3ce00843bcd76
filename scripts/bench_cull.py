"""Cost of the post-solve outlier culling in the keyframe sequence (icg_ba_outlier_culling_resident between the two-pass solve and the
resident marginalization), on bench.py's batch shape: 296 cfg-3 windows (synth_cull: pixel key points, injected outliers) on two handles.

  A: gvinsOptimization -> marginalize_resident              (what the keyframe path did before)
  B: gvinsOptimization -> outlier culling -> marginalize_resident
Reported: median wall time per batch of A and B, the device time of the culling call (H2D + kernel + D2H, CUDA events on the handle's
stream) and the culling kernel's own time (torch.profiler over many calls), with the card name and power limit read in the same run.

Usage: python scripts/bench_cull.py [--windows 296] [--handles 2] [--reps 20] [--out profiles/r3_bench_cull.json]
"""
import argparse
import copy
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=296)
    ap.add_argument("--handles", type=int, default=2)
    ap.add_argument("--distinct", type=int, default=16)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_bench_cull.json"))
    a = ap.parse_args()
    import torch
    from datagen import synth_cull
    from ic_gvins_b200.ba import WindowSolver, imu_preintegrate

    def pre(st, iewn, g, nz, imu):
        blob, end = imu_preintegrate(st, iewn, g, nz, imu)
        return blob, np.zeros((imu.shape[0] - 1, 4)), end

    base = [synth_cull.make_cull_window(pre, K=10, L=300, seed=3000 + i) for i in range(a.distinct)]
    wins = [copy.deepcopy(base[i % len(base)]) for i in range(a.windows)]
    bounds = [(a.windows * k) // a.handles for k in range(a.handles + 1)]
    maxF = max(w[0]["F"] for w in wins)
    streams = [torch.cuda.Stream() for _ in range(a.handles)]
    parts = []
    for k in range(a.handles):
        sv = WindowSolver(max_windows=bounds[k + 1] - bounds[k], max_K=10, max_L=300, max_F=maxF, max_gnss=8, max_marg_r=1, stream=streams[k].cuda_stream)
        ws = wins[bounds[k]:bounds[k + 1]]
        probs, cins = [w[0] for w in ws], [w[1] for w in ws]
        init = [{q: np.array(p[q], copy=True) for q in ("pose", "mix", "ext", "invdepth", "f_active", "gnss_std")} for p in probs]
        parts.append((sv, probs, cins, init, sv.marg_prepare(probs, 1, want_schur=False)))
    cull_ms = []

    def step(cull):
        for k, (sv, probs, cins, init, mc) in enumerate(parts):
            for p, ini in zip(probs, init):
                for q, v in ini.items():
                    p[q][...] = v
            sv.gvins_optimization_batch(probs, 20)
            if cull:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(streams[k])
                sv.outlier_culling(probs, cins, want_geometry=False)
                e1.record(streams[k])
                e1.synchronize()
                cull_ms.append(e0.elapsed_time(e1))
            sv.marg_run(mc, resident=True)
        torch.cuda.synchronize()

    res = {}
    for name, cull in (("solve_marg", False), ("solve_cull_marg", True), ("solve_marg_again", False), ("solve_cull_marg_again", True)):
        step(cull)  # warm-up
        ts = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            step(cull)
            ts.append((time.perf_counter() - t0) * 1e3)
        res[name] = dict(median_ms=float(np.median(ts)), min_ms=float(np.min(ts)), per_rep_ms=ts)
    dev_ms = cull_ms[len(parts):]  # drop the warm-up calls
    # the kernel alone: torch.profiler (CUPTI) over many culling calls on the resident windows
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(50):
            for sv, probs, cins, _, _ in parts:
                sv.outlier_culling(probs, cins, want_geometry=False)
        torch.cuda.synchronize()
    kern = [e for e in prof.events() if "ba_outlier_cull" in e.name]
    k_us = [e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total for e in kern]
    name = torch.cuda.get_device_name()
    try:
        plim = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        plim = "unavailable (%s)" % e
    counts = np.array([o["counts"] for sv, probs, cins, _, _ in parts for o in sv.outlier_culling(probs, cins, want_geometry=False)])
    out = dict(
        workload="%d cfg-3 windows (synth_cull, %d distinct) on %d handles: gvinsOptimization(5 + 15) -> [outlier culling] -> marginalize_resident(1 node)"
                 % (a.windows, a.distinct, a.handles, ),
        device=name, power_limit=plim, reps=a.reps, results=res,
        added_ms_per_batch=res["solve_cull_marg"]["median_ms"] - res["solve_marg"]["median_ms"],
        added_ms_per_batch_again=res["solve_cull_marg_again"]["median_ms"] - res["solve_marg_again"]["median_ms"],
        cull_call_device_ms=dict(median=float(np.median(dev_ms)), min=float(np.min(dev_ms)), n=len(dev_ms),
                                 note="CUDA events around one icg_ba_outlier_culling_resident call on the handle's stream (%d windows): H2D + kernel + D2H"
                                      % (bounds[1] - bounds[0])),
        cull_kernel_us=dict(median=float(np.median(k_us)) if k_us else None, min=float(np.min(k_us)) if k_us else None, n=len(k_us)),
        observations_per_window=float(np.mean([w[0]["F"] + w[0]["L"] for w in wins])),
        counts_mean_per_window=dict(zip(["outliers_0", "outliers_1", "num1", "num2", "num3"], counts.mean(0).tolist())),
    )
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k != "results"}))
    for sv, *_ in parts:
        sv.close()


if __name__ == "__main__":
    main()
