#!/usr/bin/env python
"""bench.py -- headline benchmark of the IC-GVINS hot paths on B200 (contract: see the task statement / DESIGN.md).

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torch.distributed.run, one rank / GPU)
    python bench.py --impl reference ...                     (the reference's CPU path: cv2 LK + the BA oracle port)
    python bench.py ... --dump-outputs DIR                   (+ what the headline path returned in its last timed step, DIR/<name>.npy)

A "step" = one frame of every one of B independent 1280x560 synthetic streams resident on this GPU:
pyramid build (levels 1..3) of the B new frames + fused forward/backward KLT of 300 points per stream
(+ one 10-KF / 300-landmark window solve per frame once `--ba` is on).  value = frames/s over all ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, NPTS = 1280, 560, 300
WORKLOAD = ("cfg5-style throughput mode (cfg2 + cfg3 per frame): B independent synthetic 1280x560 streams per GPU; per frame: pyramid levels 1..3 + "
            "fused fwd+bwd 21x21 LK of 300 pts, and one 10-KF / 300-landmark window solve (reprojection + IMU-preintegration + GNSS "
            "factors, gvinsOptimization protocol 5 + chi2 culling + 15 LM iterations; every frame treated as a keyframe)")
WORKLOAD_KLT = "cfg2 x B: B independent synthetic 1280x560 streams per GPU, pyramid + fused fwd+bwd LK of 300 pts (KLT only, --no-ba)"
NFRAMES = 6           # distinct frames per stream (ping-pong sequence 0..5..0)
KLT_BYTES_PER_FRAME_TRACK = 2 * 952_000 + 58 * NPTS                     # tracker kernel only (both pyramids + point I/O)
KLT_BYTES_PER_FRAME_TOTAL = int(W * H * (1 + 5 / 16 + 21 / 64 + 2 * 85 / 64) + 58 * NPTS)  # SURVEY 8d: 3 097 400
# dram__bytes_read.sum + dram__bytes_write.sum of klt_track_kernel from the ncu --set full capture in profiles/r1_klt_v2_ncu.md
# (266.831 MB + 7.692 MB for one launch over B = 148 frames), per frame; the bench scales it to its own B
KLT_DRAM_BYTES_PER_FRAME_NCU = (266_830_592 + 7_691_520) / 148.0


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=296, help="independent streams (frames in flight) per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-frames", type=int, default=8, help="frames (LK pairs + window solves) per host process per CPU-arm repetition")
    ap.add_argument("--no-ba", action="store_true")
    ap.add_argument("--ba-handles", type=int, default=2, help="solver handles (CUDA streams) the B windows are split over")
    ap.add_argument("--no-sharded", action="store_true", help="skip the cfg-4 landmark-sharded BA section")
    ap.add_argument("--sharded-windows", type=int, default=128, help="cfg-4 windows in the landmark-sharded batch")
    ap.add_argument("--no-marg", action="store_true", help="skip the marginalization section")
    ap.add_argument("--no-detect", action="store_true", help="skip the block-detection section")
    ap.add_argument("--no-clahe", action="store_true", help="skip the CLAHE section")
    ap.add_argument("--no-keyframe", action="store_true", help="skip the full-keyframe-path line")
    ap.add_argument("--no-e2e-pipeline", action="store_true", help="e2e: one set of solver handles (the host packs and the GPU solves in turn)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the arrays the headline path returned in its last timed step to DIR/<name>.npy "
                                                          "(rank 0; float32 / float64; a fixed sample of the streams beyond 64 MB)")
    return ap.parse_args()


# ----------------------------------------------------------------------------------------------- synthetic stream
def make_stream(seed: int):
    from datagen import synth_klt as synth
    st = synth.KltStream(W, H, NPTS, seed)
    frames = [st.frame(t) for t in range(NFRAMES)]
    pts = [st.points(t) for t in range(NFRAMES)]
    return frames, pts


def frame_sequence(n_steps: int):
    """ping-pong frame indices so that consecutive entries are always adjacent frames of the stream"""
    period = list(range(NFRAMES)) + list(range(NFRAMES - 2, 0, -1))
    return [period[i % len(period)] for i in range(n_steps + 1)]


def pair_points(pts, fa, fb, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    prev = pts[fa].astype(np.float32)
    init = (pts[fb] + rng.normal(0.0, 1.0, size=pts[fb].shape)).astype(np.float32)
    return prev, init


def write_outputs(out_dir, arrays, limit=64 << 20):
    """Save each array (leading axis = stream) as out_dir/<name>.npy, float64 kept and everything else as float32.  Beyond `limit` bytes in
    all, every array keeps the same seeded sample of streams, so that two builds run with the same arguments stay comparable."""
    arrays = {k: a.astype(np.float64 if a.dtype == np.float64 else np.float32) for k, a in arrays.items()}
    n = len(next(iter(arrays.values())))
    per_stream = sum(a.nbytes for a in arrays.values()) / n
    if per_stream * n > limit:
        keep = np.sort(np.random.default_rng(0).choice(n, int(limit // per_stream), replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


# ----------------------------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self._stop, self._th = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._th = threading.Thread(target=self._run, daemon=True)
        self._th.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._th.join(timeout=6)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- CPU reference arm
def cpu_arm_inputs(frames, pts, n_probs=4):
    """Inputs of oracle/cpu_arm.py: the 10 adjacent frame pairs of the ping-pong sequence with their points, a few cfg-3 windows."""
    import ctypes as C
    import oracle
    from tests import oracle_api as oa
    seq = frame_sequence(10)
    pairs = []
    for k in range(10):
        prev, init = pair_points(pts, seq[k], seq[k + 1], 99 + k)
        pairs.append((seq[k], seq[k + 1], prev, init))
    olib = C.CDLL(oracle.LIB)  # built by __graft_entry__.build(): the bench only reads the source tree
    oa.declare(olib)
    oa.declare_ba(olib)
    probs = make_windows(n_probs, lambda *a: oa.preintegrate(olib, *a))
    return pairs, probs


def cpu_throughput(frames, pts, reps, n_frames, do_ba=True):
    """The reference's CPU path in throughput mode on every usable host core (one pinned process per core, fixed work, median of `reps`):
    oracle/cpu_arm.py.  Returns its result dict."""
    from oracle import cpu_arm
    pairs, probs = cpu_arm_inputs(frames, pts)
    return cpu_arm.measure(frames, pairs, probs, reps=reps, n_frames=n_frames, do_ba=do_ba)


def cpu_single_stream(frames, pts, seconds: float = 1.5):
    """Context for the throughput-mode baseline: ONE stream the way the reference runs it (cv2's own threading over all cores for LK,
    one 4-thread solve at a time as Ceres is configured, IG/ic_gvins.cc:1146).  Returns (klt frames/s, ba solves/s)."""
    import copy
    import ctypes as C
    import oracle
    from tests import oracle_api as oa
    klt = None
    try:
        import cv2
        cv2.setNumThreads(os.cpu_count() or 1)
        crit = (cv2.TERM_CRITERIA_COUNT + cv2.TERM_CRITERIA_EPS, 30, 0.01)
        seq = frame_sequence(1000)
        t0, k = time.perf_counter(), 0
        while time.perf_counter() - t0 < seconds:
            fa, fb = seq[k % 10], seq[k % 10 + 1]
            prev, init = pair_points(pts, fa, fb, 7 + k)
            fwd, _, _ = cv2.calcOpticalFlowPyrLK(frames[fa], frames[fb], prev.reshape(-1, 1, 2), init.reshape(-1, 1, 2).copy(), winSize=(21, 21),
                                                 maxLevel=3, criteria=crit, flags=cv2.OPTFLOW_USE_INITIAL_FLOW)
            cv2.calcOpticalFlowPyrLK(frames[fb], frames[fa], fwd, prev.reshape(-1, 1, 2).copy(), winSize=(21, 21), maxLevel=3, criteria=crit,
                                     flags=cv2.OPTFLOW_USE_INITIAL_FLOW)
            k += 1
        klt = k / (time.perf_counter() - t0)
    except Exception:
        pass
    olib = C.CDLL(oracle.LIB)
    oa.declare(olib)
    oa.declare_ba(olib)
    prob = make_windows(1, lambda *a: oa.preintegrate(olib, *a))[0]
    t0, k = time.perf_counter(), 0
    while time.perf_counter() - t0 < seconds:
        p = copy.deepcopy(prob)
        oa.ba_solve(olib, p, 5, 4)
        oa.ba_solve(olib, p, 15, 4)
        k += 1
    return klt, k / (time.perf_counter() - t0)


def make_windows(n, preintegrate, seed0=2024):
    from datagen import synth_ba
    return [synth_ba.make_window(preintegrate, K=10, L=300, seed=seed0 + b)[0] for b in range(n)]


def run_reference(args):
    """`--impl reference`: the reference's CPU path on the box's host cores (rank 0 only).  Each of the W + K steps is one fixed-work
    repetition of oracle/cpu_arm.py (every usable core: one pinned process, 8 frames each); value = median over the K timed steps."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    frames, pts = make_stream(1234)
    reps = max(1, args.steps + args.warmup)
    res = cpu_throughput(frames, pts, reps=reps, n_frames=args.cpu_frames, do_ba=not args.no_ba)
    timed = res["per_repetition"][args.warmup:] or res["per_repetition"]
    v = float(np.median(timed))
    res = dict(res, value=v, per_repetition_timed=timed)
    line = {"impl": "reference", "metric": "frames/sec (KLT+BA) 1280x560 300-feat 10-KF window", "value": v, "unit": "frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * res["cores"] * args.cpu_frames / v,
            "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8/int32 fixed point + f32 (KLT), f64 (BA)", "data": "synthetic",
            "config": {"workload": WORKLOAD if not args.no_ba else WORKLOAD_KLT, "streams_per_gpu": res["cores"],
                       "note": "CPU arm: one independent stream per host core (streams_per_gpu = host processes here)"},
            "cpu_baseline": res,
            "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------- B200 arm
def run_b200(args):
    # the contract is ONE JSON line on stdout: libraries that chat on fd 1 (e.g. "NCCL version ..." at communicator creation) are sent
    # to stderr for the duration of the run; the saved descriptor is used for the final line
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from ic_gvins_b200 import lib
    from ic_gvins_b200.ba import BaProblem, BaSummary, WindowSolver, imu_preintegrate, to_struct
    from ic_gvins_b200.klt import KltTracker
    import ctypes as C

    B = args.streams
    use_ba = not args.no_ba
    stream = torch.cuda.Stream(device=dev)       # KLT stream (tracking thread of the reference)
    stream_ba = torch.cuda.Stream(device=dev)    # BA stream (optimization thread of the reference)
    frames, pts = make_stream(1234 + rank)
    n_slots = NFRAMES * B
    trk = KltTracker(W, H, n_slots=n_slots, max_points=B * NPTS, device=local_rank, stream=stream.cuda_stream)

    # ---- KLT inputs: pinned host frames; level-0 planes resident in HBM: slot = f * B + b
    h_frames = [torch.from_numpy(f.copy()).pin_memory() for f in frames]
    frame_ptrs = [[h_frames[f].data_ptr()] * B for f in range(NFRAMES)]  # the B streams replicate one 6-frame sequence (distinct device slots)
    for f in range(NFRAMES):
        for b in range(B):
            trk.upload_ptr(f * B + b, h_frames[f].data_ptr(), W, build=False)
    trk.sync()
    total = args.warmup + args.steps
    seq = frame_sequence(total + 1)
    n_total = B * NPTS
    h_prev = torch.empty((total, n_total, 2), dtype=torch.float32).pin_memory()
    h_init = torch.empty((total, n_total, 2), dtype=torch.float32).pin_memory()
    h_slots = torch.empty((total, n_total, 2), dtype=torch.int32).pin_memory()
    for s in range(total):
        fa, fb = seq[s], seq[s + 1]
        for b in range(B):
            p, i = pair_points(pts, fa, fb, 1000 * s + b)
            h_prev[s, b * NPTS:(b + 1) * NPTS] = torch.from_numpy(p)
            h_init[s, b * NPTS:(b + 1) * NPTS] = torch.from_numpy(i)
            h_slots[s, b * NPTS:(b + 1) * NPTS, 0] = fa * B + b
            h_slots[s, b * NPTS:(b + 1) * NPTS, 1] = fb * B + b
    d_prev, d_init, d_slots = h_prev.to(dev), h_init.to(dev), h_slots.to(dev)
    d_fwd = torch.empty((n_total, 2), dtype=torch.float32, device=dev)
    d_bwd = torch.empty((n_total, 2), dtype=torch.float32, device=dev)
    d_st = torch.empty((n_total,), dtype=torch.uint8, device=dev)
    h_fwd = torch.empty((n_total, 2), dtype=torch.float32).pin_memory()
    h_st = torch.empty((n_total,), dtype=torch.uint8).pin_memory()
    e_prev = torch.empty((n_total, 2), dtype=torch.float32, device=dev)
    e_init = torch.empty((n_total, 2), dtype=torch.float32, device=dev)
    e_slots = torch.empty((n_total, 2), dtype=torch.int32, device=dev)

    # ---- BA inputs: one cfg-3 window per stream (the product's own host-side preintegration builds the IMU factors)
    solvers, e2e_parts, e2e_sets = [], [], [([], [])]
    if use_ba:
        def pre(st, iewn, g, nz, imu):
            blob, end = imu_preintegrate(st, iewn, g, nz, imu)
            return blob, np.zeros((imu.shape[0] - 1, 4)), end
        import copy
        base = make_windows(min(B, 64), pre, seed0=2024 + 1000 * rank)  # 64 distinct windows, repeated to fill the batch
        windows = [copy.deepcopy(base[i % len(base)]) for i in range(B)]
        maxF = max(w_["F"] for w_ in windows)
        NH = max(1, min(args.ba_handles, B))
        bounds = [(B * k) // NH for k in range(NH + 1)]
        ba_streams = [stream_ba] + [torch.cuda.Stream(device=dev) for _ in range(NH - 1)]
        e2e_parts = []
        for k in range(NH):
            part = windows[bounds[k]:bounds[k + 1]]
            sv = WindowSolver(max_windows=len(part), max_K=10, max_L=300, max_F=maxF, max_gnss=8, max_marg_r=1, device=local_rank,
                              stream=ba_streams[k].cuda_stream)
            sv.upload(part)
            sv.sync()
            solvers.append(sv)
            # e2e: the struct array over host arrays is what the reference's optimization thread would hand over each keyframe
            pe = [copy.deepcopy(w_) for w_ in part]
            init = [{q: np.array(w_[q], copy=True) for q in ("pose", "mix", "ext", "invdepth", "f_active", "gnss_std")} for w_ in pe]
            e2e_parts.append((pe, init, (BaProblem * len(pe))(*[to_struct(w_) for w_ in pe]), (BaSummary * (2 * len(pe)))()))
        # e2e: a second set of handles, so that the host packs keyframe s + 1 while the GPU solves keyframe s (the reference's optimization thread
        # runs beside its tracking thread the same way); every step still moves its own inputs H2D and its own results D2H inside the timed region
        solvers_b, e2e_parts_b = [], []
        if not args.no_e2e_pipeline:
            for k in range(NH):
                part = windows[bounds[k]:bounds[k + 1]]
                st_b = torch.cuda.Stream(device=dev)
                ba_streams.append(st_b)
                sv = WindowSolver(max_windows=len(part), max_K=10, max_L=300, max_F=maxF, max_gnss=8, max_marg_r=1, device=local_rank, stream=st_b.cuda_stream)
                solvers_b.append(sv)
                pe = [copy.deepcopy(w_) for w_ in part]
                init = [{q: np.array(w_[q], copy=True) for q in ("pose", "mix", "ext", "invdepth", "f_active", "gnss_std")} for w_ in pe]
                e2e_parts_b.append((pe, init, (BaProblem * len(pe))(*[to_struct(w_) for w_ in pe]), (BaSummary * (2 * len(pe)))()))
        e2e_sets = [(solvers, e2e_parts)] + ([(solvers_b, e2e_parts_b)] if solvers_b else [])
        # what icg_ba_upload moves per window (arrays are capacity-strided: max_F factor slots, max_K = 10 IMU slots): slot-ordered factor constants +
        # (landmark, ref, obs, id) + pair index + activity, parameters, IMU blobs + sqrt-information, CSR offsets, GNSS
        ba_h2d = int(len(windows) * (maxF * (14 * 8 + 16 + 4 + 1) + 10 * 16 * 8 + 8 * 8 + 300 * 8 + 10 * (480 + 225) * 8 + 301 * 4 + 91 * 8 + 8 * 56))
        ba_d2h = int(sum(10 * 16 * 8 + 8 * 8 + 300 * 8 + w_["F"] for w_ in windows))
    else:
        ba_h2d = ba_d2h = 0
        ba_streams = []

    def klt_resident(s):
        fb = seq[s + 1]
        trk.build_pyramids(fb * B, B)
        trk.track_batch_dev(n_total, d_slots[s].data_ptr(), d_prev[s].data_ptr(), d_init[s].data_ptr(), d_fwd.data_ptr(),
                            d_bwd.data_ptr(), d_st.data_ptr(), 1)

    def step_resident(s):
        klt_resident(s)
        for sv in solvers:
            sv.run_gvins(20, restart=True)

    e2e_host = {"klt_enqueue_ms": [], "ba_begin_ms": [], "ba_end_ms": []}  # host wall time of the phases of an e2e step (where the step goes)

    def step_e2e(s):
        t_0 = time.perf_counter()
        fb = seq[s + 1]
        trk.upload_batch_ptrs(fb * B, frame_ptrs[fb], W)  # H2D of this step's B new frames from pinned host memory (one call, linear DMA)
        with torch.cuda.stream(stream):
            e_prev.copy_(h_prev[s], non_blocking=True)
            e_init.copy_(h_init[s], non_blocking=True)
            e_slots.copy_(h_slots[s], non_blocking=True)
        trk.build_pyramids(fb * B, B)
        trk.track_batch_dev(n_total, e_slots.data_ptr(), e_prev.data_ptr(), e_init.data_ptr(), d_fwd.data_ptr(), d_bwd.data_ptr(),
                            d_st.data_ptr(), 1)
        with torch.cuda.stream(stream):
            h_fwd.copy_(d_fwd, non_blocking=True)
            h_st.copy_(d_st, non_blocking=True)
        t_1 = time.perf_counter()

        if not use_ba:
            return
        svs, parts = e2e_sets[s % len(e2e_sets)]
        for k in range(len(svs)):
            sv, (pe, init, arr, summ) = svs[k], parts[k]
            for w_, ini in zip(pe, init):  # fresh initial guess every step (the solve updates in place)
                for q, v in ini.items():
                    w_[q][...] = v
            rc = lib().icg_ba_gvins_optimization_begin(sv._h, len(pe), arr, 20)  # pack + upload + enqueue (asynchronous)
            if rc != 0:
                raise RuntimeError(lib().icg_last_error().decode())
        t_2 = time.perf_counter()
        e2e_pending.append(s)
        e2e_finish(keep=len(e2e_sets) - 1)  # two handle sets: collect the PREVIOUS keyframe while this one is on the GPU
        t_3 = time.perf_counter()
        e2e_host["klt_enqueue_ms"].append((t_1 - t_0) * 1e3), e2e_host["ba_begin_ms"].append((t_2 - t_1) * 1e3), e2e_host["ba_end_ms"].append((t_3 - t_2) * 1e3)

    e2e_pending = []

    def e2e_finish(keep=0):
        """synchronise + write back the keyframes in flight (all but the newest `keep`)"""
        while len(e2e_pending) > keep:
            s_ = e2e_pending.pop(0)
            svs, parts = e2e_sets[s_ % len(e2e_sets)]
            for sv, (pe, init, arr, summ) in zip(svs, parts):
                rc = lib().icg_ba_gvins_optimization_end(sv._h, len(pe), arr, summ, None)
                if rc != 0:
                    raise RuntimeError(lib().icg_last_error().decode())

    # ---- the FULL keyframe path of every stream, end to end through the C ABI: what one keyframe costs when nothing is left out.
    #      H2D of the raw frame -> CLAHE + histogram-gate statistic (batched, device-resident) -> pyramid -> fwd+bwd LK + gates -> block detection
    #      (goodFeaturesToTrack + cornerSubPix on the 18 blocks of every frame) -> gvinsOptimization (host arrays in / out) -> gvinsMarginalization
    #      (host arrays in, prior out).  Every frame is treated as a keyframe (conservative).
    kf = None
    if use_ba and not args.no_keyframe:
        from ic_gvins_b200.clahe import Clahe
        from ic_gvins_b200.detect import Detector, block_rois
        import ctypes as C2
        d_raw = torch.from_numpy(np.stack(frames)).to(dev)  # the raw (un-equalised) frames of the sequence, device-resident staging of the H2D copy
        kcl = Clahe(W, H, 3.0, (21, 21), device=local_rank, stream=stream.cuda_stream)
        rois, quota, min_dist, _ = block_rois(W, H, NPTS)
        kdet = Detector(W, H, max_blocks=B * len(rois), max_corners_per_block=32, max_roi_pixels=213 * 186, device=local_rank, stream=stream.cuda_stream)
        p0_, p1_, pit_ = C2.c_void_p(), C2.c_void_p(), C2.c_int()
        lib().icg_klt_slot_level0(trk._h, 0, C2.byref(p0_), C2.byref(pit_))
        lib().icg_klt_slot_level0(trk._h, 1, C2.byref(p1_), C2.byref(pit_))
        slot_stride, slot_pitch, slot0 = p1_.value - p0_.value, pit_.value, p0_.value
        kf_mcalls = [solvers[k].marg_prepare(e2e_parts[k][0], 1, want_schur=False) for k in range(len(solvers))]
        h_raw = torch.empty((B, H, W), dtype=torch.uint8).pin_memory()
        d_rawB = torch.empty((B, H, W), dtype=torch.uint8, device=dev)
        kf_hist = [None]

        kf_host = {"clahe_ms": [], "klt_enqueue_ms": [], "detect_ms": [], "ba_marg_join_ms": []}  # host wall time of the phases (BA threads run beside detection)

        def step_keyframe(s):
            t_0 = time.perf_counter()
            fb = seq[s + 1]
            with torch.cuda.stream(stream):
                d_rawB.copy_(h_raw, non_blocking=True)   # H2D of the B raw frames (pinned)
                e_prev.copy_(h_prev[s], non_blocking=True)
                e_init.copy_(h_init[s], non_blocking=True)
                e_slots.copy_(h_slots[s], non_blocking=True)
            # CLAHE of the B frames into their slots' level-0 planes + the histogram-gate statistic of the raw frames (synchronises: the host decides)
            kf_hist[0] = kcl.apply_batch_dev(B, d_rawB.data_ptr(), W, W * H, slot0 + fb * B * slot_stride, slot_pitch, slot_stride, want_hist=True)
            t_1 = time.perf_counter()
            trk.build_pyramids(fb * B, B)
            trk.track_batch_dev(n_total, e_slots.data_ptr(), e_prev.data_ptr(), e_init.data_ptr(), d_fwd.data_ptr(), d_bwd.data_ptr(), d_st.data_ptr(), 1)
            with torch.cuda.stream(stream):
                h_fwd.copy_(d_fwd, non_blocking=True)
                h_st.copy_(d_st, non_blocking=True)
            t_2 = time.perf_counter()

            def ba_part(k):
                sv, (pe, init, arr, summ) = solvers[k], e2e_parts[k]
                for w_, ini in zip(pe, init):
                    for q, v in ini.items():
                        w_[q][...] = v
                rc = lib().icg_ba_gvins_optimization_begin(sv._h, len(pe), arr, 20)
                if rc == 0:
                    rc = lib().icg_ba_gvins_optimization_end(sv._h, len(pe), arr, summ, None)
                if rc != 0:
                    raise RuntimeError(lib().icg_last_error().decode())
                sv.marg_run(kf_mcalls[k], resident=True)  # gvinsMarginalization of the window just optimised: prior out to host arrays
            ths = [threading.Thread(target=ba_part, args=(k,)) for k in range(len(solvers))]
            for t_ in ths:
                t_.start()
            # block detection of the B equalised frames (device-resident input, corners back on the host), beside the BA threads
            kdet.detect_blocks_dev(B, slot0 + fb * B * slot_stride, slot_pitch, slot_stride, rois, [quota] * len(rois), 0.01, float(min_dist))
            t_3 = time.perf_counter()
            for t_ in ths:
                t_.join()
            t_4 = time.perf_counter()
            kf_host["clahe_ms"].append((t_1 - t_0) * 1e3), kf_host["klt_enqueue_ms"].append((t_2 - t_1) * 1e3)
            kf_host["detect_ms"].append((t_3 - t_2) * 1e3), kf_host["ba_marg_join_ms"].append((t_4 - t_3) * 1e3)
        for b in range(B):
            h_raw[b].copy_(h_frames[0])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def headline_outputs():
        """What the last step_resident handed its caller, one row per stream: the fused LK results and, per window, the solved parameters
        with the pass-2 summary.  The solvers download into copies: the uploaded windows feed the later sections unchanged."""
        out = {"klt_fwd_xy": d_fwd.cpu().numpy().reshape(B, NPTS, 2), "klt_bwd_xy": d_bwd.cpu().numpy().reshape(B, NPTS, 2),
               "klt_status": d_st.cpu().numpy().reshape(B, NPTS)}
        if use_ba:
            par = ("pose", "mix", "ext", "invdepth")
            got = {q: [] for q in par + ("final_cost", "iterations")}
            for k, sv in enumerate(solvers):
                part = [dict(w_, **{q: np.array(w_[q], np.float64) for q in par}) for w_ in windows[bounds[k]:bounds[k + 1]]]
                arr, summ = (BaProblem * len(part))(*[to_struct(w_) for w_ in part]), (BaSummary * len(part))()
                if lib().icg_ba_download(sv._h, len(part), arr, summ) != 0:
                    raise RuntimeError(lib().icg_last_error().decode())
                for w_, s_ in zip(part, summ):
                    for q in par:
                        got[q].append(w_[q])
                    got["final_cost"].append(s_.final_cost)
                    got["iterations"].append(s_.iterations)
            out.update({"ba_" + q: np.array(v, np.float64) for q, v in got.items()})
            out["ba_pose"], out["ba_mix"] = out["ba_pose"].reshape(B, -1, 7), out["ba_mix"].reshape(B, -1, 9)
        return out

    def timed(step_fn, mode="step", finish_fn=None):
        for s in range(args.warmup):
            if step_fn is not None:
                step_fn(s)
            elif mode == "ba_only":
                for sv in solvers:
                    sv.run_gvins(20, restart=True)
        if finish_fn is not None:
            finish_fn()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        kev = []
        torch.cuda.synchronize()
        ev0.record(stream)
        for bs in ba_streams:
            bs.wait_stream(stream)
        for s in range(args.warmup, total):
            if mode == "klt_kernel":
                fb = seq[s + 1]
                trk.build_pyramids(fb * B, B)
                a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                trk.track_batch_dev(n_total, d_slots[s].data_ptr(), d_prev[s].data_ptr(), d_init[s].data_ptr(), d_fwd.data_ptr(),
                                    d_bwd.data_ptr(), d_st.data_ptr(), 1)
                b_.record(stream)
                kev.append((a, b_))
            elif mode == "ba_only":
                a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                for bs in ba_streams:
                    bs.wait_stream(stream)
                for sv in solvers:
                    sv.run_gvins(20, restart=True)
                for bs in ba_streams:
                    stream.wait_stream(bs)
                b_.record(stream)
                kev.append((a, b_))
            else:
                step_fn(s)
        if finish_fn is not None:
            finish_fn()                 # the last keyframe in flight is collected inside the timed region
        for bs in ba_streams:
            stream.wait_stream(bs)      # the step ends when the tracking and all optimization streams are done
        ev1.record(stream)
        barrier()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        kms = [a.elapsed_time(b_) for a, b_ in kev]
        return ms, kms

    lib().icg_launch_count_reset()
    with ClockSampler(local_rank) as clk:
        ms_res, _ = timed(step_resident)
        launches = int(lib().icg_launch_count())
        if args.dump_outputs and rank == 0:
            write_outputs(args.dump_outputs, headline_outputs())
        ms_e2e, _ = timed(step_e2e, finish_fn=e2e_finish)
        _, kms = timed(klt_resident, mode="klt_kernel")
        bms = timed(None, mode="ba_only")[1] if use_ba else []
        ms_klt, _ = timed(klt_resident)
        if use_ba and not args.no_keyframe:
            ms_kf, _ = timed(step_keyframe)
            kf = {"workload": "FULL keyframe path of B streams end to end through the C ABI: H2D raw frame, CLAHE + histogram gate (batched), pyramid, fwd+bwd LK, "
                              "block detection (18 blocks x B frames, one call), gvinsOptimization (host arrays in / out) and gvinsMarginalization of the window "
                              "just optimised (icg_ba_marginalize_resident, prior out to host arrays); 2 handles, one host thread each; every frame a keyframe", "value": B * world * args.steps / (ms_kf / 1e3), "unit": "frames/s",
                  "ms_per_step": ms_kf / args.steps,
                  "host_ms_per_step": {k_: float(np.mean(v_[args.warmup:])) for k_, v_ in kf_host.items() if len(v_) > args.warmup}}
    clocks = clk.summary()
    good = int(d_st.sum().item())
    ba_info = None
    if use_ba:
        sm = [x for sv in solvers for x in sv.download(write_back=False)]
        ba_info = {"ms_per_batch": float(np.mean(bms)), "windows_per_batch": B, "solves_per_s": B / (float(np.mean(bms)) / 1e3) * world,
                   "mean_lm_iterations_pass2": float(np.mean([x["iterations"] for x in sm])),
                   "final_cost_mean": float(np.mean([x["final_cost"] for x in sm]))}

    # ---- CLAHE pre-pass (SURVEY 8f rank 2; tracking.cc:141): device-resident, in place, one frame per call on the KLT stream
    clahe = None
    if not args.no_clahe:
        from ic_gvins_b200.clahe import Clahe
        NC = 148
        cbuf = torch.from_numpy(np.stack([frames[k % NFRAMES] for k in range(NC)])).to(dev)
        cl = Clahe(W, H, 3.0, (21, 21), device=local_rank, stream=stream.cuda_stream)
        for k in range(8):
            cl.apply_dev(cbuf[k].data_ptr(), W, cbuf[k].data_ptr(), W)
        barrier()
        ca, cb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ca.record(stream)
        for k in range(NC):
            cl.apply_dev(cbuf[k].data_ptr(), W, cbuf[k].data_ptr(), W)
        cb.record(stream)
        barrier()
        cms = ca.elapsed_time(cb) / NC
        # the same NC frames in ONE batched launch pair (+ the fused histogram-gate statistic on a second pass)
        cl.apply_batch_dev(NC, cbuf.data_ptr(), W, W * H, cbuf.data_ptr(), W, W * H)
        barrier()
        ca.record(stream)
        for _ in range(5):
            cl.apply_batch_dev(NC, cbuf.data_ptr(), W, W * H, cbuf.data_ptr(), W, W * H)
        cb.record(stream)
        barrier()
        cmsb = ca.elapsed_time(cb) / (5 * NC)
        clahe = {"workload": "icg_clahe_apply_dev (clip 3.0, 21x21 tiles) in place on HBM-resident 1280x560 frames, one frame per call; "
                             "batched: icg_clahe_apply_batch_dev, 148 frames per launch pair",
                 "ms_per_frame": cms, "frames_per_s": 1e3 / cms * world, "algorithmic_bytes_per_frame": 3 * W * H,
                 "achieved_GBps": 3 * W * H / (cms * 1e-3) / 1e9,
                 "batched_ms_per_frame": cmsb, "batched_frames_per_s": 1e3 / cmsb * world, "batched_achieved_GBps": 3 * W * H / (cmsb * 1e-3) / 1e9}
        cl.close()
        del cbuf
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            try:
                import cv2
                cv2.setNumThreads(os.cpu_count() or 1)
                cc = cv2.createCLAHE(3.0, (21, 21))
                t0 = time.perf_counter()
                for k in range(20):
                    cc.apply(frames[k % NFRAMES])
                clahe["cpu_cv2_ms_per_frame"] = (time.perf_counter() - t0) / 20 * 1e3
            except Exception:
                pass

    # ---- featuresDetection (SURVEY 8a row A4): all 18 blocks of a frame in one host-buffer call (image H2D + corners D2H inside)
    detect = None
    if not args.no_detect:
        from ic_gvins_b200.detect import Detector, block_rois
        det = Detector(W, H, max_blocks=32, max_corners_per_block=64, device=local_rank)
        rois, quota, min_dist, _ = block_rois(W, H, NPTS)
        want = [quota] * len(rois)
        got = det.detect_blocks(frames[0], rois, want, 0.01, float(min_dist), None, subpix=True)
        barrier()
        reps = 20
        tcall = []
        for k in range(reps):  # per-call wall time, median: one stalled host round trip (seen once: 4.8 ms mean on a box whose median was 0.7) is not the call's cost
            t0 = time.perf_counter()
            det.detect_blocks(frames[k % NFRAMES], rois, want, 0.01, float(min_dist), None, subpix=True)
            tcall.append(time.perf_counter() - t0)
        dtd = float(np.median(tcall))
        detect = {"workload": "icg_detect_blocks: goodFeaturesToTrack + cornerSubPix on the 18 blocks of a 1280x560 frame, empty mask, "
                              "host buffers (synchronous call, one frame at a time: the reference's per-keyframe use)",
                  "ms_per_frame": dtd * 1e3, "ms_per_frame_mean": float(np.mean(tcall)) * 1e3, "ms_per_frame_max": float(np.max(tcall)) * 1e3,
                  "frames_per_s": 1.0 / dtd * world, "corners": int(sum(len(g) for g in got))}
        det.close()
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            try:
                import cv2
                cv2.setNumThreads(os.cpu_count() or 1)
                t0 = time.perf_counter()
                for k in range(5):
                    img = frames[k % NFRAMES]
                    for (x0, y0, bw, bh), n in zip(rois, want):  # cv2 on numpy slices (the C++ ROI reads beyond the block edge; timing only)
                        blk = np.ascontiguousarray(img[y0:y0 + bh, x0:x0 + bw])
                        c = cv2.goodFeaturesToTrack(blk, n, 0.01, float(min_dist))
                        if c is not None and len(c):
                            cv2.cornerSubPix(blk, c, (5, 5), (-1, -1), (cv2.TERM_CRITERIA_COUNT + cv2.TERM_CRITERIA_EPS, 20, 0.01))
                detect["cpu_cv2_ms_per_frame"] = (time.perf_counter() - t0) / 5 * 1e3
            except Exception:
                pass

    # ---- gvinsMarginalization (SURVEY 8a row B10): the step that follows the solve at every keyframe, through the host-buffer C ABI
    marg = None
    if use_ba and not args.no_marg:
        part = windows[bounds[0]:bounds[1]]
        solvers[0].marginalize(part[:2], 1, want_schur=False)  # workspace allocation + warm-up
        barrier()
        reps = 5
        mcall = solvers[0].marg_prepare(part, 1, want_schur=False)  # argument block (structs over host arrays, output arrays): kept across keyframes
        solvers[0].marg_run(mcall)
        t0 = time.perf_counter()
        for _ in range(reps):
            solvers[0].marg_run(mcall)                 # icg_ba_marginalize: pack + upload + linearise + 2 eigendecompositions + D2H + write-out
        dtm = (time.perf_counter() - t0) / reps
        msum = (BaSummary * (2 * len(part)))()
        if lib().icg_ba_gvins_optimization(solvers[0]._h, len(part), mcall["arr"], 20, msum, None) != 0:  # two-pass solve, written back to `part`
            raise RuntimeError(lib().icg_last_error().decode())
        t0 = time.perf_counter()
        for _ in range(reps):
            solvers[0].marg_run(mcall, resident=True)  # icg_ba_marginalize_resident: the windows the handle has just solved (no pack / upload)
        dtr = (time.perf_counter() - t0) / reps
        pri = solvers[0].marg_collect(mcall)
        marg = {"workload": "icg_ba_marginalize: oldest node + the landmarks anchored in it out of a cfg-3 window (host buffers in, prior out; "
                            "pack + upload + linearisation + two Jacobi eigendecompositions + D2H inside the timed region); resident_*: "
                            "icg_ba_marginalize_resident on the windows the handle has just solved (the reference's order: gvinsOptimization, then "
                            "gvinsMarginalization on the same window), prior out to host arrays",
                "windows_per_call": len(part), "ms_per_call": dtm * 1e3, "windows_per_s": len(part) / dtm * world,
                "resident_ms_per_call": dtr * 1e3, "resident_windows_per_s": len(part) / dtr * world,
                "m": int(pri[0]["m"]), "r": int(pri[0]["r"])}
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            import ctypes as C
            import oracle
            from tests import oracle_api as oa
            olib = C.CDLL(oracle.LIB)
            oa.declare_ba(olib)
            pw = make_windows(1, lambda *a: oa.preintegrate(olib, *a))[0]
            oa.ba_marginalize(olib, pw, 1)
            t0 = time.perf_counter()
            for _ in range(3):
                oa.ba_marginalize(olib, pw, 1)
            marg["cpu_port_ms_per_window"] = (time.perf_counter() - t0) / 3 * 1e3

    # ---- cfg 4: 20-KF / 2000-landmark windows, landmarks sharded over the ranks with an NCCL all-reduce per LM attempt
    sharded = None
    if use_ba and not args.no_sharded:
        from ic_gvins_b200.ba import connect_shards, shard_window
        NW4 = args.sharded_windows
        import copy as _copy
        nd4 = min(NW4, 8)  # distinct cfg-4 windows (host-side generation is ~1 s each), repeated to fill the batch
        big0 = [__import__("datagen.synth_ba", fromlist=["x"]).make_window(pre, K=20, L=2000, seed=4000 + i)[0] for i in range(nd4)]
        big = [_copy.deepcopy(big0[i % nd4]) for i in range(NW4)]
        shards = [shard_window(p_, rank, world) for p_ in big]
        s4 = WindowSolver(max_windows=NW4, max_K=20, max_L=max(x["L"] for x in shards), max_F=max(x["F"] for x in shards), max_gnss=16,
                          max_marg_r=1, device=local_rank, stream=stream_ba.cuda_stream)
        if world > 1:
            connect_shards(s4, rank, world, "p2p", dist)   # peer-memory transport: P2P stores over NVLink, no NCCL on the data path
        s4.upload(shards)
        for _ in range(2):
            s4.run_gvins(20, restart=True)
        barrier()
        a4, b4 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps4 = 5
        a4.record(stream_ba)
        for _ in range(reps4):
            s4.run_gvins(20, restart=True)
        b4.record(stream_ba)
        barrier()
        ms4 = a4.elapsed_time(b4) / reps4
        if world > 1:
            t4 = torch.tensor([ms4], device=dev, dtype=torch.float64)
            dist.all_reduce(t4, op=dist.ReduceOp.MAX)
            ms4 = float(t4.item())
        sm4 = s4.download(write_back=False)
        pk = 127 * 128 // 2 + 3 * 127 + 4
        sharded = {"workload": "cfg4: batch of 20-KF / 2000-landmark windows (gvinsOptimization 5 + 15), landmarks block-partitioned over the ranks; window w "
                               "is reduced and solved by rank w mod ranks: packed reduced-camera operands P2P-stored into the owner's inbox over NVLink, "
                               "cluster Cholesky on the owner, camera step stored back to every rank (strong scaling of one batch)",
                   "windows": NW4, "ranks": world, "transport": "p2p" if world > 1 else "local",
                   "factors_per_window": int(np.mean([p_["F"] for p_ in big])), "ms_per_batch": ms4, "window_solves_per_s": NW4 / (ms4 / 1e3),
                   "reduce_bytes_per_attempt_per_rank": int(NW4 * pk * 8 * (world - 1) / max(1, world)), "final_cost_window0": sm4[0]["final_cost"],
                   "mean_lm_iterations_pass2": float(np.mean([x["iterations"] for x in sm4]))}
        s4.close()

    frames_per_step = B * world
    value = frames_per_step * args.steps / (ms_res / 1e3)
    e2e = frames_per_step * args.steps / (ms_e2e / 1e3)
    k_ms = float(np.mean(kms))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = B * KLT_BYTES_PER_FRAME_TRACK / (k_ms / 1e3) / 1e9
    line = {
        "metric": "frames/sec (KLT+BA) 1280x560 300-feat 10-KF window", "value": value, "unit": "frames/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/int32 fixed point + f32 (KLT), f64 (BA)", "data": "synthetic",
        "config": {"workload": WORKLOAD if use_ba else WORKLOAD_KLT, "streams_per_gpu": B, "points_per_frame": NPTS, "ba_solver_handles": len(solvers),
                   "l2": f"inputs larger than L2: {B * 2 * 1.127:.0f} MB of pyramids touched per step",
                   "replication": "the B streams replay ONE rendered 6-frame sequence (distinct device slots, so HBM traffic and H2D volume are real) and the BA "
                                  "batch repeats 64 distinct cfg-3 windows"},
        "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": B * (W * H + NPTS * 24) + ba_h2d,
                "d2h_bytes_per_step": B * NPTS * 9 + ba_d2h, "ms_per_step": ms_e2e / args.steps,
                "keyframes_in_flight": len(e2e_sets) if use_ba else 1,
                "host_ms_per_step": {k_: float(np.mean(v_[args.warmup:])) if len(v_) > args.warmup else None for k_, v_ in e2e_host.items()}},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {"kernel": "klt_track_kernel", "bound": "hbm", "achieved": achieved, "peak": peak,
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                     "unit": "GB/s", "frac": achieved / peak, "traffic": int(B * KLT_DRAM_BYTES_PER_FRAME_NCU),
                     "traffic_source": "ncu --set full, one launch at B = 148 (profiles/r1_klt_v2_ncu.md), scaled to this B", "kernel_ms": k_ms,
                     "algorithmic_bytes_per_launch": B * KLT_BYTES_PER_FRAME_TRACK},
        # second roofline, informative: the window solve as a whole against the FP64 rate measured on this part (scripts/fp64_probe.cu:
        # 36.3 TFLOP/s DFMA, 37.0 DMMA).  Algorithmic flops = SURVEY 8d's 5 MFLOP per LM iteration of a cfg-3 window x the 22 linearise +
        # solve iterations of gvinsOptimization (5 + 15 + the two bookkeeping passes) x B windows; the path is latency-bound (profiles/r1_ba_stages.md)
        "roofline_ba": ({"kernels": "gvinsOptimization kernel sequence (ba_lin_vis .. ba_accept), whole batch", "bound": "fp64", "unit": "TFLOP/s",
                         "achieved": 5.0e6 * 22 * B / (ba_info["ms_per_batch"] * 1e-3) / 1e12, "peak": 36.3,
                         "peak_source": "scripts/fp64_probe.cu on the gpurun B200 (profiles/r1_ba_stages.md)",
                         "frac": 5.0e6 * 22 * B / (ba_info["ms_per_batch"] * 1e-3) / 1e12 / 36.3,
                         "algorithmic_flops_per_batch": 5.0e6 * 22 * B} if ba_info else None),
        "klt_only": {"value": frames_per_step * args.steps / (ms_klt / 1e3), "unit": "frames/s"},
        "keyframe_path": kf,
        "ba_only": ba_info,
        "sharded_ba": sharded,
        "marginalization": marg,
        "detection": detect,
        "clahe": clahe,
        "tracked_fraction": good / float(n_total),
    }
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        res = cpu_throughput(frames, pts, reps=5, n_frames=args.cpu_frames, do_ba=use_ba)
        if use_ba:
            ss_klt, ss_ba = cpu_single_stream(frames, pts)
            res["single_stream"] = {"klt_frames_per_s": ss_klt, "ba_solves_per_s": ss_ba,
                                    "note": "context: ONE stream as the reference runs it (cv2 LK with all threads, one 4-thread solve at a time)"}
        line["cpu_baseline"] = res
    if rank == 0:
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    trk.close()
    for sv in solvers + (solvers_b if use_ba else []):
        sv.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
