"""Host-side mirror of the reference's window-solve seam (IG/ic_gvins.cc:1130-1239): `WindowSolver` plays the role of
`ceres::Problem` + `ceres::Solver::Solve`, `gvins_optimization()` restates the two-pass protocol of
GVINS::gvinsOptimization (solve N/4 -> chi-square culling -> solve N - N/4).  All arithmetic runs in libicgvins_b200.so.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from ._lib import check, lib, vp

IMU_BLOB = 480
dp = C.POINTER(C.c_double)
ip = C.POINTER(C.c_int32)
bp = C.POINTER(C.c_uint8)


class BaProblem(C.Structure):
    """ctypes image of `icg_ba_problem` (include/icgvins_b200.h)."""
    _fields_ = [
        ("K", C.c_int32), ("L", C.c_int32), ("F", C.c_int32),
        ("pose", dp), ("mix", dp), ("ext", dp), ("invdepth", dp),
        ("ext_const", C.c_int32), ("td_const", C.c_int32),
        ("f_lm", ip), ("f_ref", ip), ("f_obs", ip), ("f_const", dp), ("f_active", bp),
        ("reproj_std", C.c_double), ("reproj_huber", C.c_int32),
        ("n_imu", C.c_int32), ("imu_blob", dp), ("has_imu_error", C.c_int32),
        ("has_pose_prior", C.c_int32), ("pose_prior", dp), ("pose_prior_std", dp),
        ("has_mix_prior", C.c_int32), ("mix_prior", dp), ("mix_prior_std", dp),
        ("n_gnss", C.c_int32), ("gnss_node", ip), ("gnss_blh", dp), ("gnss_std", dp), ("lever", C.c_double * 3),
        ("gnss_huber", C.c_int32),
        ("marg_r", C.c_int32), ("marg_nblocks", C.c_int32), ("marg_block_type", ip), ("marg_block_node", ip),
        ("marg_x0", dp), ("marg_J0", dp), ("marg_e0", dp),
    ]


class BaPrior(C.Structure):
    """ctypes image of `icg_ba_prior`."""
    _fields_ = [("m", C.c_int32), ("r", C.c_int32), ("nblocks", C.c_int32), ("rcap", C.c_int32), ("block_type", ip), ("block_node", ip),
                ("x0", dp), ("J0", dp), ("e0", dp), ("Hp", dp), ("bp", dp)]


class Camera(C.Structure):
    """ctypes image of `icg_camera`."""
    _fields_ = [(k, C.c_double) for k in ("fx", "fy", "cx", "cy", "skew", "k1", "k2", "p1", "p2", "k3")]


class CullInput(C.Structure):
    """ctypes image of `icg_ba_cull_input`."""
    _fields_ = [("cam", Camera), ("reprojection_error_std", C.c_double), ("estimate_extrinsic", C.c_int32), ("reserved", C.c_int32),
                ("R_bc", C.c_double * 9), ("t_bc", C.c_double * 3), ("f_kp", C.POINTER(C.c_float)), ("lm_ref_kp", C.POINTER(C.c_float)),
                ("lm_ref_node", ip), ("lm_ref_pos", ip)]


class CullOutput(C.Structure):
    """ctypes image of `icg_ba_cull_output`."""
    _fields_ = [("ext_updated", C.c_int32), ("counts", C.c_int32 * 5), ("R_bc", C.c_double * 9), ("t_bc", C.c_double * 3),
                ("cam_pose", dp), ("lm_pos", dp), ("lm_depth", dp), ("f_outlier", bp), ("lm_ref_outlier", bp), ("lm_outlier", bp)]


class BaSummary(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("num_successful_steps", C.c_int32), ("termination", C.c_int32), ("reserved", C.c_int32),
                ("initial_cost", C.c_double), ("final_cost", C.c_double), ("final_radius", C.c_double)]


_ARR = dict(pose=np.float64, mix=np.float64, ext=np.float64, invdepth=np.float64, f_lm=np.int32, f_ref=np.int32, f_obs=np.int32,
            f_const=np.float64, f_active=np.uint8, imu_blob=np.float64, pose_prior=np.float64, pose_prior_std=np.float64,
            mix_prior=np.float64, mix_prior_std=np.float64, gnss_node=np.int32, gnss_blh=np.float64, gnss_std=np.float64,
            marg_block_type=np.int32, marg_block_node=np.int32, marg_x0=np.float64, marg_J0=np.float64, marg_e0=np.float64)
_SCAL = ["K", "L", "F", "ext_const", "td_const", "reproj_std", "reproj_huber", "n_imu", "has_imu_error", "has_pose_prior",
         "has_mix_prior", "n_gnss", "gnss_huber", "marg_r", "marg_nblocks"]


def to_struct(prob: dict) -> BaProblem:
    """Build the C struct over the dict's numpy arrays IN PLACE (arrays are made contiguous inside the dict so that the
    solve's in/out parameter updates are visible to the caller)."""
    s = BaProblem()
    for k, dt in _ARR.items():
        a = np.ascontiguousarray(prob[k], dtype=dt)
        prob[k] = a
        ptr_t = dp if dt == np.float64 else ip if dt == np.int32 else bp
        setattr(s, k, a.ctypes.data_as(ptr_t) if a.size else ptr_t())
    for k in _SCAL:
        setattr(s, k, prob[k])
    for i in range(3):
        s.lever[i] = float(prob["lever"][i])
    return s


def shard_window(prob: dict, rank: int, world: int) -> dict:
    """Landmark shard `rank` of `world` of one window problem (SURVEY.md 8e): block partition of the landmarks, each landmark keeps
    all of its reprojection factors (the per-landmark loop at IG/ic_gvins.cc:1777-1834); the camera-side problem is replicated.
    Returns a new dict whose `invdepth`, `f_*` arrays are the local slices (landmark indices remapped) plus `lm_lo`, `lm_hi`
    (global landmark range) and `f_index` (global factor indices) for merging results back."""
    L, F = prob["L"], prob["F"]
    lo, hi = (L * rank) // world, (L * (rank + 1)) // world
    f_lm = np.asarray(prob["f_lm"])
    sel = np.nonzero((f_lm >= lo) & (f_lm < hi))[0]
    out = dict(prob)
    out.update(L=hi - lo, F=len(sel), invdepth=np.array(prob["invdepth"][lo:hi], np.float64),
               f_lm=(f_lm[sel] - lo).astype(np.int32), f_ref=np.asarray(prob["f_ref"])[sel].astype(np.int32),
               f_obs=np.asarray(prob["f_obs"])[sel].astype(np.int32),
               f_const=np.asarray(prob["f_const"], np.float64).reshape(-1, 14)[sel].reshape(-1).copy(),
               f_active=np.asarray(prob["f_active"], np.uint8)[sel].copy(), lm_lo=lo, lm_hi=hi, f_index=sel)
    for k in ("pose", "mix", "ext", "gnss_std"):
        out[k] = np.array(prob[k], copy=True)
    return out


def merge_shard(prob: dict, shard: dict) -> None:
    """Write a solved shard's landmark results back into the full problem dict (camera-side blocks are identical on all shards)."""
    prob["invdepth"][shard["lm_lo"]:shard["lm_hi"]] = shard["invdepth"]
    prob["f_active"][shard["f_index"]] = shard["f_active"]
    for k in ("pose", "mix", "ext", "gnss_std"):
        prob[k][...] = shard[k]


def connect_shards(solver: "WindowSolver", rank: int, world: int, transport: str, dist) -> None:
    """Join `solver` to the landmark-shard group of `world` processes (one per GPU).  The only transport is "p2p": peer-memory stores over
    NVLink.  `dist` is an initialised torch.distributed module (any backend): it only carries the rendezvous blobs, the CUDA IPC handles of
    the exchange buffers."""
    if transport != "p2p":
        raise ValueError(transport)
    mine = solver.shard_export(rank, world)
    blobs = [None] * world
    dist.all_gather_object(blobs, mine)
    solver.shard_connect(blobs)
    dist.barrier()


def imu_preintegrate(state16, iewn, gravity, noise5, imu):
    """B3 host-side propagation in the product library (PreintegrationEarth::integrationProcess, preintegration_earth.cc:205-303)."""
    imu = np.ascontiguousarray(imu, np.float64)
    n = imu.shape[0]
    blob = np.zeros(IMU_BLOB)
    end = np.zeros(10)
    st, g, nz = (np.ascontiguousarray(x, np.float64) for x in (state16, gravity, noise5))
    iw = np.ascontiguousarray(iewn, np.float64) if iewn is not None else None  # None: PreintegrationNormal (iswithearth false)
    check(lib().icg_imu_preintegrate(vp(st.ctypes.data), vp(iw.ctypes.data) if iw is not None else None, vp(g.ctypes.data), vp(nz.ctypes.data),
                                     vp(imu.ctypes.data), n, vp(blob.ctypes.data), vp(end.ctypes.data)), "icg_imu_preintegrate")
    return blob, end


class WindowSolver:
    """Batched sliding-window solver handle (one per optimization thread / GPU)."""

    def __init__(self, max_windows=1, max_K=10, max_L=300, max_F=2700, max_gnss=16, max_marg_r=160, device=0, stream=None):
        self._h = vp()
        check(lib().icg_ba_create(C.byref(self._h), max_windows, max_K, max_L, max_F, max_gnss, max_marg_r, device,
                                  vp(stream) if stream else None), "icg_ba_create")

    def close(self):
        if getattr(self, "_h", None):
            lib().icg_ba_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def shard_export(self, rank: int, world: int) -> bytes:
        """Allocate this rank's peer-memory exchange buffer for a group of `world` ranks; returns the blob the other ranks need."""
        buf = (C.c_uint8 * 128)()
        check(lib().icg_ba_shard_export(self._h, rank, world, buf), "icg_ba_shard_export")
        return bytes(buf)

    def shard_connect(self, blobs) -> None:
        """blobs: the `world` export blobs in rank order."""
        raw = b"".join(blobs)
        buf = (C.c_uint8 * len(raw)).from_buffer_copy(raw)
        check(lib().icg_ba_shard_connect(self._h, buf), "icg_ba_shard_connect")

    def solve(self, problems, max_num_iterations: int):
        """ceres::Solver::Solve on a list of problem dicts (updated in place).  Returns a list of summaries."""
        if isinstance(problems, dict):
            problems = [problems]
        n = len(problems)
        arr = (BaProblem * n)(*[to_struct(p) for p in problems])
        summ = (BaSummary * n)()
        check(lib().icg_ba_solve(self._h, n, arr, max_num_iterations, summ), "icg_ba_solve")
        return [dict(iterations=s.iterations, num_successful_steps=s.num_successful_steps, termination=s.termination,
                     initial_cost=s.initial_cost, final_cost=s.final_cost, final_radius=s.final_radius) for s in summ]

    def solve_structs(self, arr, n, max_num_iterations, summ):
        check(lib().icg_ba_solve(self._h, n, arr, max_num_iterations, summ), "icg_ba_solve")

    # -- device-resident stages
    def upload(self, problems):
        n = len(problems)
        self._keep = (BaProblem * n)(*[to_struct(p) for p in problems])
        self._n = n
        check(lib().icg_ba_upload(self._h, n, self._keep), "icg_ba_upload")

    def run(self, max_num_iterations: int, restart: bool = False):
        check(lib().icg_ba_run(self._h, max_num_iterations, 1 if restart else 0), "icg_ba_run")

    def download(self, write_back: bool = True):
        summ = (BaSummary * self._n)()
        check(lib().icg_ba_download(self._h, self._n, self._keep if write_back else None, summ), "icg_ba_download")
        return [dict(iterations=s.iterations, num_successful_steps=s.num_successful_steps, termination=s.termination,
                     initial_cost=s.initial_cost, final_cost=s.final_cost, final_radius=s.final_radius) for s in summ]

    def sync(self):
        check(lib().icg_ba_sync(self._h), "icg_ba_sync")

    def residual_costs(self, prob):
        s = to_struct(prob)
        rc = np.zeros(prob["F"])
        gc = np.zeros(prob["n_gnss"])
        check(lib().icg_ba_residual_costs(self._h, C.byref(s), vp(rc.ctypes.data), vp(gc.ctypes.data) if gc.size else None),
              "icg_ba_residual_costs")
        return rc, gc

    def gvins_optimization_batch(self, problems, num_iterations=20):
        """GVINS::gvinsOptimization on a list of windows in one device-resident call (icg_ba_gvins_optimization)."""
        n = len(problems)
        arr = (BaProblem * n)(*[to_struct(p) for p in problems])
        summ = (BaSummary * (2 * n))()
        culled = (C.c_int32 * (2 * n))()
        check(lib().icg_ba_gvins_optimization(self._h, n, arr, num_iterations, summ, culled), "icg_ba_gvins_optimization")
        f = lambda s: dict(iterations=s.iterations, num_successful_steps=s.num_successful_steps, termination=s.termination,
                           initial_cost=s.initial_cost, final_cost=s.final_cost, final_radius=s.final_radius)
        return [dict(pass1=f(summ[2 * w]), pass2=f(summ[2 * w + 1]), reproj_removed=culled[2 * w], gnss_reweighted=culled[2 * w + 1])
                for w in range(n)]

    def run_gvins(self, num_iterations: int = 20, restart: bool = False):
        check(lib().icg_ba_run_gvins(self._h, num_iterations, 1 if restart else 0), "icg_ba_run_gvins")

    def gvins_optimization(self, prob, num_iterations=20):
        """GVINS::gvinsOptimization (IG/ic_gvins.cc:1130-1239): pass 1 (N/4 iterations, Huber on GNSS + reprojection),
        GNSS chi2 re-weighting (:1241-1267), reprojection chi2 removal (:1269-1297), pass 2 (N - N/4, GNSS without loss)."""
        first = num_iterations // 4
        second = num_iterations - first
        prob["gnss_huber"] = 1
        s1 = self.solve(prob, first)[0]
        rc, gc = self.residual_costs(prob)
        gnss_std = prob["gnss_std"].reshape(-1, 3)
        n_gnss_out = 0
        for g in range(prob["n_gnss"]):
            chi2 = 2.0 * gc[g]
            if chi2 > 7.815:
                gnss_std[g] *= np.sqrt(chi2 / 7.815)
                n_gnss_out += 1
        prob["gnss_std"] = gnss_std.reshape(-1)
        act = prob["f_active"]
        out = (2.0 * rc > 5.991) & (act != 0)
        act[out] = 0
        prob["gnss_huber"] = 0
        s2 = self.solve(prob, second)[0]
        return dict(pass1=s1, pass2=s2, reproj_removed=int(out.sum()), gnss_reweighted=n_gnss_out)

    def marginalize(self, problems, num_marg=1, want_schur=True, resident=False):
        """MarginalizationInfo::marginalization as GVINS::gvinsMarginalization drives it (IG/ic_gvins.cc:1412-1640) on a list of
        windows: removes the `num_marg` oldest nodes + the landmarks anchored in them.  Returns one dict per window with the new
        prior in the layout the problem dict's marg_* entries use (node indices already shifted).  resident=True: the windows are the
        ones this handle has just solved (icg_ba_marginalize_resident: nothing is uploaded again)."""
        if isinstance(problems, dict):
            problems = [problems]
        call = self.marg_prepare(problems, num_marg, want_schur)
        self.marg_run(call, resident)
        return self.marg_collect(call)

    def outlier_culling(self, problems, cull_inputs, want_geometry=True):
        """GVINS::updateParametersFromOptimizer + gvinsOutlierCulling (IG/ic_gvins.cc:1299-1389, 1035-1128) on the windows this handle has just
        solved (icg_ba_outlier_culling_resident; `problems` = the list of that solve).  cull_inputs: one dict per window with `cam` (fx, fy, cx,
        cy[, skew]), `reprojection_error_std` (px), `estimate_extrinsic`, `R_bc` (3x3), `t_bc`, `f_kp` (F x 2), `lm_ref_kp` (L x 2),
        `lm_ref_node`, `lm_ref_pos` (L).  Each problem's f_active becomes the culling mask (in place).  Returns one dict per window: ext_updated,
        R_bc, t_bc, counts (outliers_[0], outliers_[1], num1, num2, num3), f_outlier, lm_ref_outlier, lm_outlier (bits num1 | num2 << 1 | num3 << 2)
        and, with want_geometry, cam_pose (K x 12: R_wc row-major, t_wc), lm_pos (L x 3), lm_depth."""
        if isinstance(problems, dict):
            problems, cull_inputs = [problems], [cull_inputs]
        n = len(problems)
        arr = (BaProblem * n)(*[to_struct(p) for p in problems])
        cin, cout = (CullInput * n)(), (CullOutput * n)()
        keep, res = [], []
        for w, (p, c) in enumerate(zip(problems, cull_inputs)):
            cam = list(c["cam"]) + [0.0] * (10 - len(c["cam"]))
            cin[w].cam = Camera(*[float(x) for x in cam])
            cin[w].reprojection_error_std = float(c["reprojection_error_std"])
            cin[w].estimate_extrinsic = int(bool(c["estimate_extrinsic"]))
            cin[w].R_bc[:] = [float(x) for x in np.asarray(c["R_bc"], np.float64).ravel()]
            cin[w].t_bc[:] = [float(x) for x in np.asarray(c["t_bc"], np.float64).ravel()]
            dts = dict(f_kp=np.float32, lm_ref_kp=np.float32, lm_ref_node=np.int32, lm_ref_pos=np.int32)
            a = {k: np.ascontiguousarray(c[k], dt) for k, dt in dts.items() if c[k] is not None}  # None passes NULL (argument checks)
            o = dict(f_outlier=np.zeros(p["F"], np.uint8), lm_ref_outlier=np.zeros(p["L"], np.uint8), lm_outlier=np.zeros(p["L"], np.uint8))
            if want_geometry:
                o.update(cam_pose=np.zeros((p["K"], 12)), lm_pos=np.zeros((p["L"], 3)), lm_depth=np.zeros(p["L"]))
            for k, v in a.items():
                setattr(cin[w], k, v.ctypes.data_as(C.POINTER(C.c_float) if v.dtype == np.float32 else ip) if v.size else None)
            for k, v in o.items():
                setattr(cout[w], k, v.ctypes.data_as(dp if v.dtype == np.float64 else bp) if v.size else None)
            keep.append(a)
            res.append(o)
        check(lib().icg_ba_outlier_culling_resident(self._h, n, arr, cin, cout), "icg_ba_outlier_culling_resident")
        for w, o in enumerate(res):
            o.update(ext_updated=int(cout[w].ext_updated), counts=np.array(cout[w].counts[:], np.int32),
                     R_bc=np.array(cout[w].R_bc[:]).reshape(3, 3), t_bc=np.array(cout[w].t_bc[:]))
        return res

    def marg_prepare(self, problems, num_marg=1, want_schur=True):
        """The argument block of one icg_ba_marginalize call (struct array over the problems' host arrays + caller-allocated output arrays):
        what a C++ caller keeps alive across keyframes.  marg_run issues the call, marg_collect turns the outputs into dicts."""
        n = len(problems)
        nm = np.full(n, num_marg, np.int32) if np.isscalar(num_marg) else np.ascontiguousarray(num_marg, np.int32)
        arr = (BaProblem * n)(*[to_struct(p) for p in problems])
        pri = (BaPrior * n)()
        bufs = []
        for w, p in enumerate(problems):
            rcap = 15 * p["K"] + 7
            b = dict(bt=np.zeros(2 * p["K"] + 2, np.int32), bn=np.zeros(2 * p["K"] + 2, np.int32), x0=np.zeros(16 * p["K"] + 8),
                     J0=np.zeros(rcap * rcap), e0=np.zeros(rcap))
            if want_schur:
                b.update(Hp=np.zeros(rcap * rcap), bp=np.zeros(rcap))
            bufs.append(b)
            pri[w].rcap = rcap
            pri[w].block_type, pri[w].block_node = b["bt"].ctypes.data_as(ip), b["bn"].ctypes.data_as(ip)
            pri[w].x0, pri[w].J0, pri[w].e0 = b["x0"].ctypes.data_as(dp), b["J0"].ctypes.data_as(dp), b["e0"].ctypes.data_as(dp)
            if want_schur:
                pri[w].Hp, pri[w].bp = b["Hp"].ctypes.data_as(dp), b["bp"].ctypes.data_as(dp)
        return dict(n=n, nm=nm, arr=arr, pri=pri, bufs=bufs, want_schur=want_schur, problems=problems)

    def marg_run(self, call, resident=False):
        fn = lib().icg_ba_marginalize_resident if resident else lib().icg_ba_marginalize
        check(fn(self._h, call["n"], call["arr"], vp(call["nm"].ctypes.data), call["pri"]), "icg_ba_marginalize")

    def marg_collect(self, call):
        out = []
        gs = {0: 7, 1: 9, 2: 7, 3: 1}
        pri, want_schur = call["pri"], call["want_schur"]
        for w, b in enumerate(call["bufs"]):
            r, nb = pri[w].r, pri[w].nblocks
            nx = sum(gs[int(t)] for t in b["bt"][:nb])
            out.append(dict(m=pri[w].m, r=r, block_type=b["bt"][:nb].copy(), block_node=b["bn"][:nb].copy(), x0=b["x0"][:nx].copy(),
                            J0=b["J0"][:r * r].reshape(r, r).copy(), e0=b["e0"][:r].copy(),
                            Hp=b["Hp"][:r * r].reshape(r, r).copy() if want_schur else None, bp=b["bp"][:r].copy() if want_schur else None))
        return out

    # -- single-factor Evaluate (Ceres CostFunction contract), computed on the device
    def reproj_evaluate(self, pose0, pose1, ext, invdepth, td, const14, std, want_jac=True):
        a = [np.ascontiguousarray(x, np.float64) for x in (pose0, pose1, ext, np.atleast_1d(invdepth), np.atleast_1d(td), const14)]
        r = np.zeros(2)
        Js = [np.zeros((2, 7)), np.zeros((2, 7)), np.zeros((2, 7)), np.zeros((2, 1)), np.zeros((2, 1))]
        jp = (vp * 5)(*[vp(j.ctypes.data) for j in Js])
        check(lib().icg_ba_reproj_evaluate(self._h, *[vp(x.ctypes.data) for x in a], float(std), vp(r.ctypes.data),
                                           jp if want_jac else None), "icg_ba_reproj_evaluate")
        return r, Js

    def gnss_evaluate(self, pose, blh, std3, lever):
        a = [np.ascontiguousarray(x, np.float64) for x in (pose, blh, std3, lever)]
        r, J = np.zeros(3), np.zeros((3, 7))
        jp = (vp * 1)(vp(J.ctypes.data))
        check(lib().icg_ba_gnss_evaluate(self._h, *[vp(x.ctypes.data) for x in a], vp(r.ctypes.data), jp), "icg_ba_gnss_evaluate")
        return r, J

    def pose_prior_evaluate(self, pose, prior7, std6):
        a = [np.ascontiguousarray(x, np.float64) for x in (pose, prior7, std6)]
        r, J = np.zeros(6), np.zeros((6, 7))
        jp = (vp * 1)(vp(J.ctypes.data))
        check(lib().icg_ba_pose_prior_evaluate(self._h, *[vp(x.ctypes.data) for x in a], vp(r.ctypes.data), jp), "icg_ba_pose_prior_evaluate")
        return r, J

    def mix_prior_evaluate(self, mix, prior9, std9):
        a = [np.ascontiguousarray(x, np.float64) for x in (mix, prior9, std9)]
        r, J = np.zeros(9), np.zeros((9, 9))
        jp = (vp * 1)(vp(J.ctypes.data))
        check(lib().icg_ba_mix_prior_evaluate(self._h, *[vp(x.ctypes.data) for x in a], vp(r.ctypes.data), jp), "icg_ba_mix_prior_evaluate")
        return r, J

    def imu_error_evaluate(self, mix):
        m = np.ascontiguousarray(mix, np.float64)
        r, J = np.zeros(6), np.zeros((6, 9))
        jp = (vp * 1)(vp(J.ctypes.data))
        check(lib().icg_ba_imu_error_evaluate(self._h, vp(m.ctypes.data), vp(r.ctypes.data), jp), "icg_ba_imu_error_evaluate")
        return r, J

    def marg_factor_evaluate(self, block_type, params, x0, J0, e0):
        """MarginalizationFactor::Evaluate: params = list of the remained blocks' current values (global sizes)."""
        bt = np.ascontiguousarray(block_type, np.int32)
        ps = [np.ascontiguousarray(x, np.float64) for x in params]
        x0, J0, e0 = (np.ascontiguousarray(x, np.float64) for x in (x0, J0, e0))
        r = len(e0)
        gs = {0: 7, 1: 9, 2: 7, 3: 1}
        res = np.zeros(r)
        Js = [np.zeros((r, gs[int(t)])) for t in bt]
        pp = (vp * len(ps))(*[vp(x.ctypes.data) for x in ps])
        jp = (vp * len(Js))(*[vp(x.ctypes.data) for x in Js])
        check(lib().icg_ba_marg_factor_evaluate(self._h, r, len(bt), vp(bt.ctypes.data), pp, vp(x0.ctypes.data), vp(J0.ctypes.data), vp(e0.ctypes.data),
                                                vp(res.ctypes.data), jp), "icg_ba_marg_factor_evaluate")
        return res, Js

    def imu_evaluate(self, blob, pose0, mix0, pose1, mix1, want_jac=True):
        a = [np.ascontiguousarray(x, np.float64) for x in (blob, pose0, mix0, pose1, mix1)]
        r = np.zeros(15)
        Js = [np.zeros((15, 7)), np.zeros((15, 9)), np.zeros((15, 7)), np.zeros((15, 9))]
        jp = (vp * 4)(*[vp(j.ctypes.data) for j in Js])
        check(lib().icg_ba_imu_evaluate(self._h, *[vp(x.ctypes.data) for x in a], vp(r.ctypes.data), jp if want_jac else None),
              "icg_ba_imu_evaluate")
        return r, Js
