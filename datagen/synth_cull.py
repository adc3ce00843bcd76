"""Synthetic windows for the post-solve outlier culling (GVINS::gvinsOutlierCulling, IG/ic_gvins.cc:1035-1128).  Input generator only.

Built on synth_ba.make_window (unchanged): the key points become pixels of the camera fx = fy = 787, cx = 640, cy = 280 -- float32
cam2pixel of the window's normalised points -- and f_const is re-derived from them with pixel2cam, as the reference builds its factors from
keyPoint() (IG/ic_gvins.cc:1777-1834).  The reference observation sits at position 0, 1 (the triangulation order, IG/tracking/tracking.cc:769-778)
or last of the landmark's observation list.  Injected:
  - gross outliers: a few % of the observations displaced by 6-30 px (feature outliers);
  - num3 landmarks: every non-reference observation displaced by 2-3 px;
  - depth outliers: landmarks moved along their reference ray behind the camera or beyond 200 m, observations re-projected from the truth.
    They trip the depth gate at the reference observation (num1, with the loop's break) -- the only way the reference observation can be
    bad, since the map point is placed on the reference ray and reprojects onto its own key point.
Every decision of the culling, evaluated at the truth parameters, is at least `MARGIN` (px or m) away from its threshold; injections are
re-drawn until it is, so that FP64 rounding cannot flip a decision at those parameters.
"""
from __future__ import annotations

import numpy as np

from . import synth_ba

CAM = (787.0, 787.0, 640.0, 280.0, 0.0)
STD_PX = 1.5
MARGIN = 1e-6


def cam2pixel(cam, pc):
    """float32 pixels of camera points (..., 3) (Camera::cam2pixel, IG/tracking/camera.cc:132-134)."""
    fx, fy, cx, cy, skew = cam[:5]
    pc = np.asarray(pc, np.float64)
    return np.stack([(fx * pc[..., 0] + skew * pc[..., 1]) / pc[..., 2] + cx, fy * pc[..., 1] / pc[..., 2] + cy], -1).astype(np.float32)


def pixel2cam(cam, px):
    """normalised (x, y) of float pixels (..., 2) (Camera::pixel2cam, :126-130)."""
    fx, fy, cx, cy, skew = cam[:5]
    px = np.asarray(px, np.float32).astype(np.float64)
    y = (px[..., 1] - cy) / fy
    x = (px[..., 0] - cx - skew * y) / fx
    return np.stack([x, y], -1)


def camera_poses(pose, ext, K):
    """(R_wc, t_wc) per node from pose (K x 7, p + q_xyzw) and ext (t_bc, q_bc)."""
    Rbc, tbc = synth_ba.q_mat(ext[3:7] / np.linalg.norm(ext[3:7])), np.asarray(ext[:3])
    out = []
    for k in range(K):
        Rk = synth_ba.q_mat(pose[k, 3:] / np.linalg.norm(pose[k, 3:]))
        out.append((Rk @ Rbc, pose[k, :3] + Rk @ tbc))
    return out


def decision_margin(prob, cin, pose=None, ext=None, invdepth=None):
    """Smallest distance of any culling decision from its threshold (px for errors, m for depths) at the given parameters (default: the
    problem's).  Every observation is included, also those the loop would not reach."""
    K, L = prob["K"], prob["L"]
    pose = np.asarray(prob["pose"] if pose is None else pose, np.float64).reshape(-1, 7)
    ext = np.asarray(prob["ext"] if ext is None else ext, np.float64)
    rho = np.asarray(prob["invdepth"] if invdepth is None else invdepth, np.float64)
    poses = camera_poses(pose, ext, K)
    cam, thr = cin["cam"], 3.0 * cin["reprojection_error_std"]
    xy = pixel2cam(cam, cin["lm_ref_kp"])
    m = np.inf
    f_lm, f_obs = np.asarray(prob["f_lm"]), np.asarray(prob["f_obs"])
    for l in range(L):
        R, t = poses[int(cin["lm_ref_node"][l])]
        pw = R @ (np.array([xy[l, 0], xy[l, 1], 1.0]) / rho[l]) + t
        errs = []
        fs = np.nonzero(f_lm == l)[0]
        for node, kp in [(int(cin["lm_ref_node"][l]), cin["lm_ref_kp"][l])] + [(int(f_obs[f]), cin["f_kp"][f]) for f in fs]:
            Rn, tn = poses[node]
            pc = Rn.T @ (pw - tn)
            m = min(m, abs(pc[2] - 1.0), abs(pc[2] - 200.0))
            e = float(np.linalg.norm(cam2pixel(cam, pc).astype(np.float64) - np.asarray(kp, np.float64)))
            if 1.0 < pc[2] < 200.0:
                m = min(m, abs(e - thr))
                if e <= thr:
                    errs.append(e)
        for n_ in range(2, len(errs) + 1):  # the mean over any prefix the loop might keep
            m = min(m, abs(np.mean(errs[:n_]) - cin["reprojection_error_std"]))
    return m


def make_cull_window(preintegrate, K=10, L=300, seed=2024, gross=0.03, num3=0.02, depth=0.02, estimate_extrinsic=True, **kw):
    """Returns (prob, cin, truth): the problem dict (f_const re-derived from the pixel key points), the culling inputs
    (WindowSolver.outlier_culling's cull_inputs entry) and make_window's truth with the depth outliers moved."""
    prob0, truth0 = synth_ba.make_window(preintegrate, K=K, L=L, seed=seed, **kw)
    F = prob0["F"]
    f_lm, f_ref, f_obs = prob0["f_lm"], prob0["f_ref"], prob0["f_obs"]
    fc0 = prob0["f_const"].reshape(-1, 14)
    ref_node = np.array([j % 5 if K > 5 else j % max(1, K - 1) for j in range(L)], np.int32)  # make_window's reference frame of landmark j
    nf = np.bincount(f_lm, minlength=L)
    Rbc = synth_ba.q_mat(truth0["ext"][3:7])
    for attempt in range(100):
        rng = np.random.Generator(np.random.PCG64([seed, attempt, 7]))
        prob = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in prob0.items()}
        truth = {k: v.copy() for k, v in truth0.items()}
        f_kp = cam2pixel(CAM, fc0[:, 3:6])
        lm_kp = np.zeros((L, 2), np.float32)
        first = np.full(L, -1)
        for f in range(F - 1, -1, -1):
            first[f_lm[f]] = f
        for l in range(L):
            lm_kp[l] = cam2pixel(CAM, fc0[first[l], 0:3]) if first[l] >= 0 else np.array([640.0, 280.0], np.float32) + rng.uniform(-200, 200, 2).astype(np.float32)
        choice = rng.integers(0, 3, L)
        lm_pos = np.where(choice == 0, 0, np.where(choice == 1, np.minimum(1, nf), nf)).astype(np.int32)
        kinds = rng.random(L)
        is_depth = (kinds < depth) & (nf >= 1)
        is_num3 = (kinds >= depth) & (kinds < depth + num3) & (nf >= 2)
        rho = prob["invdepth"].copy()
        for l in np.nonzero(is_depth)[0]:  # move the point along its reference ray: behind the camera or beyond 200 m
            d = -rng.uniform(10.0, 40.0) if rng.random() < 0.5 else rng.uniform(400.0, 1000.0)
            x, y = pixel2cam(CAM, lm_kp[l])
            r = ref_node[l]
            Rr = synth_ba.q_mat(truth["pose"][r, 3:])
            pw = Rr @ (Rbc @ (np.array([x, y, 1.0]) * d) + truth["ext"][:3]) + truth["pose"][r, :3]
            for f in np.nonzero(f_lm == l)[0]:
                o = f_obs[f]
                pb = synth_ba.q_mat(truth["pose"][o, 3:]).T @ (pw - truth["pose"][o, :3])
                f_kp[f] = cam2pixel(CAM, Rbc.T @ (pb - truth["ext"][:3]))
            truth["invdepth"][l] = 1.0 / d
            rho[l] = (1.0 / d) * (1.0 + rng.normal(0, 0.05))
        for l in np.nonzero(is_num3)[0]:
            for f in np.nonzero(f_lm == l)[0]:
                a = rng.uniform(0, 2 * np.pi)
                f_kp[f] += (rng.uniform(2.0, 3.0) * np.array([np.cos(a), np.sin(a)])).astype(np.float32)
        gross_f = np.nonzero(rng.random(F) < gross)[0]
        for f in gross_f:
            a = rng.uniform(0, 2 * np.pi)
            f_kp[f] += (rng.uniform(6.0, 30.0) * np.array([np.cos(a), np.sin(a)])).astype(np.float32)
        fc = fc0.copy()
        fc[:, 0:2] = pixel2cam(CAM, lm_kp[f_lm])
        fc[:, 2] = 1.0
        fc[:, 3:5] = pixel2cam(CAM, f_kp)
        fc[:, 5] = 1.0
        # the extrinsic translation is not observable on the planar synthetic trajectory (a free solve drifts it by metres, the gate then
        # rejects it and every observation looks bad): the windows hold it constant, the gate still runs on the (unchanged) solved value
        prob.update(f_const=fc.reshape(-1).copy(), invdepth=rho, reproj_std=STD_PX / CAM[0], ext_const=1, td_const=1)
        Rb = synth_ba.q_mat(prob["ext"][3:7] / np.linalg.norm(prob["ext"][3:7]))
        cin = dict(cam=CAM, reprojection_error_std=STD_PX, estimate_extrinsic=int(estimate_extrinsic), R_bc=Rb, t_bc=prob["ext"][:3].copy(),
                   f_kp=f_kp, lm_ref_kp=lm_kp, lm_ref_node=ref_node, lm_ref_pos=lm_pos)
        assert np.array_equal(f_ref, ref_node[f_lm])
        truth_pose = truth["pose"].reshape(-1)
        if decision_margin(prob, cin, truth_pose, truth["ext"], truth["invdepth"]) >= MARGIN:
            return prob, cin, dict(truth, gross=gross_f, num3=np.nonzero(is_num3)[0], depth=np.nonzero(is_depth)[0])
    raise RuntimeError("make_cull_window: no draw kept every decision %g away from its threshold" % MARGIN)
