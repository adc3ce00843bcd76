"""Hand-built windows for the post-solve outlier culling, one landmark per behaviour of gvinsOutlierCulling (IG/ic_gvins.cc:1035-1128),
and the oracle's two-pass solve (GVINS::gvinsOptimization, :1130-1239) used to produce solved windows.  Shared by the CPU and GPU tests."""
import math

import numpy as np

from tests import oracle_api as oa

CAM = (787.0, 787.0, 640.0, 280.0, 0.0)
STD = 1.5
# nodes: identity attitude, camera = body; node 2 sits 4.1 m ahead of node 0, node 3 245 m behind it
NODE_P = np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.0, 0.0, 4.1], [0.0, 0.0, -245.0]])


def _px(P, k, d=(0.0, 0.0)):
    pc = P - NODE_P[k]
    return np.array([CAM[0] * pc[0] / pc[2] + CAM[2] + d[0], CAM[1] * pc[1] / pc[2] + CAM[3] + d[1]], np.float32)


# landmark: (point, reference position in the observation list, [(observing node, pixel offset, f_active)]); reference node 0
LANDMARKS = [
    ((0.3, 0.1, 5.0), 0, [(1, (0.01, 0.0), 1), (2, (0.01, 0.0), 1), (3, (0.0, 0.01), 1)]),  # depth 0.9 m (node 2) and 250 m (node 3): feature outliers
    ((0.1, 0.05, 0.9), 1, [(1, (0.0, 0.0), 1), (3, (0.0, 0.0), 1)]),                         # reference bad at position 1 after a bad position 0
    ((0.2, 0.1, 250.0), 0, [(1, (0.0, 0.0), 1), (2, (0.0, 0.0), 1)]),                        # reference bad at position 0: immediate break
    ((0.3, -0.1, 8.0), 2, [(1, (3.0, 0.0), 1), (2, (0.0, 3.0), 1)]),                         # errors 0, 3, 3 px: mean 2 px > 1.5 (num3)
    ((0.0, 0.0, 6.0), 0, []),                                                                # no factors: one error (num2)
    ((-0.2, 0.1, 7.0), 1, [(1, (0.0, 4.0), 0), (2, (0.2, 0.0), 1)]),                         # chi2-removed factor with a 4 px error: kept
]
# expected per landmark: f_outlier of its factors, lm_outlier bits, lm_ref_outlier
EXPECT = [([0, 1, 1], 0, 0), ([1, 0], 3, 1), ([0, 0], 3, 1), ([0, 0], 4, 0), ([], 2, 0), ([0, 0], 0, 0)]
EXPECT_COUNTS = [6, 3, 2, 3, 1]


def empty_problem(K, L, F):
    return dict(K=K, L=L, F=F, pose=np.zeros(7 * K), mix=np.zeros(9 * K), ext=np.array([0, 0, 0, 0, 0, 0, 1.0, 0]), invdepth=np.zeros(L),
                ext_const=1, td_const=1, f_lm=np.zeros(F, np.int32), f_ref=np.zeros(F, np.int32), f_obs=np.zeros(F, np.int32),
                f_const=np.zeros(14 * F), f_active=np.ones(F, np.uint8), reproj_std=STD / CAM[0], reproj_huber=1, n_imu=0,
                imu_blob=np.zeros(0), has_imu_error=0, has_pose_prior=0, pose_prior=np.zeros(7), pose_prior_std=np.ones(6), has_mix_prior=0,
                mix_prior=np.zeros(9), mix_prior_std=np.ones(9), n_gnss=0, gnss_node=np.zeros(0, np.int32), gnss_blh=np.zeros(0),
                gnss_std=np.zeros(0), lever=np.zeros(3), gnss_huber=0, marg_r=0, marg_nblocks=0, marg_block_type=np.zeros(0, np.int32),
                marg_block_node=np.zeros(0, np.int32), marg_x0=np.zeros(0), marg_J0=np.zeros(0), marg_e0=np.zeros(0))


def cull_input(prob, f_kp, lm_kp, lm_node, lm_pos, estimate_extrinsic=1, R_bc=None, t_bc=None):
    return dict(cam=CAM, reprojection_error_std=STD, estimate_extrinsic=estimate_extrinsic, R_bc=np.eye(3) if R_bc is None else R_bc,
                t_bc=np.zeros(3) if t_bc is None else t_bc, f_kp=np.asarray(f_kp, np.float32).reshape(-1, 2),
                lm_ref_kp=np.asarray(lm_kp, np.float32).reshape(-1, 2), lm_ref_node=np.asarray(lm_node, np.int32), lm_ref_pos=np.asarray(lm_pos, np.int32))


def hand_window():
    """(prob, cin): the LANDMARKS window (K = 4, identity extrinsic, estimate_extrinsic on: the gate takes the unchanged extrinsic)."""
    F = sum(len(o) for _, _, o in LANDMARKS)
    prob = empty_problem(4, len(LANDMARKS), F)
    pose = prob["pose"].reshape(-1, 7)
    pose[:, :3], pose[:, 6] = NODE_P, 1.0
    f_kp, lm_kp, lm_pos = [], [], []
    f = 0
    for l, (P, rpos, obs) in enumerate(LANDMARKS):
        P = np.array(P)
        prob["invdepth"][l] = 1.0 / P[2]
        lm_kp.append(_px(P, 0))
        lm_pos.append(rpos)
        for node, d, act in obs:
            prob["f_lm"][f], prob["f_ref"][f], prob["f_obs"][f], prob["f_active"][f] = l, 0, node, act
            f_kp.append(_px(P, node, d))
            f += 1
    return prob, cull_input(prob, f_kp, lm_kp, [0] * len(LANDMARKS), lm_pos)


def rot(axis, deg):
    a = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    h = math.radians(deg) / 2
    return np.concatenate([math.sin(h) * a, [math.cos(h)]])  # xyzw


def gate_window(q_xyzw, t, estimate_extrinsic=1):
    """K = 2 window without landmarks whose solved extrinsic is (t, q); baseline identity / 0."""
    prob = empty_problem(2, 0, 0)
    prob["pose"].reshape(-1, 7)[:, 6] = 1.0
    prob["pose"].reshape(-1, 7)[1, 0] = 1.0
    prob["ext"] = np.concatenate([t, q_xyzw, [0.0]])
    return prob, cull_input(prob, np.zeros((0, 2)), np.zeros((0, 2)), [], [], estimate_extrinsic)


def two_pass(lib, po, n=20):
    """GVINS::gvinsOptimization on the oracle: N/4 iterations, GNSS re-weighting + reprojection chi2 removal, N - N/4 iterations.
    Returns the chi2-removed mask."""
    po["gnss_huber"] = 1
    oa.ba_solve(lib, po, n // 4)
    rc, gc = oa.ba_residual_costs(lib, po)
    std = po["gnss_std"].reshape(-1, 3)
    for g in range(po["n_gnss"]):
        if 2 * gc[g] > 7.815:
            std[g] *= np.sqrt(2 * gc[g] / 7.815)
    po["gnss_std"] = std.reshape(-1)
    out = (2 * rc > 5.991) & (po["f_active"] != 0)
    po["f_active"][out] = 0
    po["gnss_huber"] = 0
    oa.ba_solve(lib, po, n - n // 4)
    return out
