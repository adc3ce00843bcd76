"""CPU: the restatement of updateParametersFromOptimizer + gvinsOutlierCulling (IG/ic_gvins.cc:1299-1389, 1035-1128; tests/cull_oracle.py)
against an independent numpy formulation, on hand-built windows (one behaviour each) and on synth_cull windows solved by the oracle's
two-pass protocol; and the effect on the marginalization prior."""
import copy
import math

import numpy as np
import pytest

from datagen import synth_cull
from tests import cull_cases as cc
from tests import cull_oracle as co
from tests import oracle_api as oa


@pytest.fixture(scope="module")
def olib(oracle):
    oa.declare_ba(oracle)
    return oracle


def _qmat(q):  # x y z w -> R, explicit sums
    x, y, z, w = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def _mm(A, B):
    return np.array([[A[i, 0] * B[0, j] + A[i, 1] * B[1, j] + A[i, 2] * B[2, j] for j in range(3)] for i in range(3)])


def _mv(A, v):
    return np.array([A[i, 0] * v[0] + A[i, 1] * v[1] + A[i, 2] * v[2] for i in range(3)])


def restate(prob, cin):
    """The same contract from the formulas (rotation angle from the trace, vectorised projections), a plain loop for the break."""
    ext = np.asarray(prob["ext"], np.float64)
    Rb, tb, upd = np.asarray(cin["R_bc"], np.float64), np.asarray(cin["t_bc"], np.float64), 0
    if cin["estimate_extrinsic"]:
        R = _qmat(ext[3:7] / math.sqrt(sum(ext[3:7] ** 2)))
        D = _mm(R, Rb.T)
        half_sin = math.sqrt(max(0.0, 1.0 - (1.0 + D[0, 0] + D[1, 1] + D[2, 2]) / 4.0))  # |vec(q)| = sin(theta / 2)
        d = ext[:3] - tb
        if not (math.sqrt(d[0] ** 2 + d[1] ** 2 + d[2] ** 2) > 1.0 or half_sin * 180.0 / math.pi > 5.0):
            Rb, tb, upd = R, ext[:3].copy(), 1
    pose = np.asarray(prob["pose"], np.float64).reshape(-1, 7)
    Rw, tw = [], []
    for k in range(prob["K"]):
        Rq = _qmat(pose[k, 3:] / math.sqrt(sum(pose[k, 3:] ** 2)))
        Rw.append(_mm(Rq, Rb)), tw.append(pose[k, :3] + _mv(Rq, tb))
    fx, fy, cx, cy, sk = cin["cam"][:5]
    kp = np.asarray(cin["lm_ref_kp"], np.float32).astype(np.float64)
    yy = (kp[:, 1] - cy) / fy
    xx = (kp[:, 0] - cx - sk * yy) / fx
    depth = 1.0 / np.asarray(prob["invdepth"], np.float64)
    pos = np.array([_mv(Rw[n], np.array([xx[l], yy[l], 1.0]) * depth[l]) + tw[n] for l, n in enumerate(cin["lm_ref_node"])]).reshape(-1, 3)

    def test(node, l, k2):
        pc = _mv(Rw[node].T, pos[l] - tw[node])
        u = np.float32((fx * pc[0] + sk * pc[1]) / pc[2] + cx)
        v = np.float32(fy * pc[1] / pc[2] + cy)
        e = math.hypot(float(u - np.float32(k2[0])), float(v - np.float32(k2[1])))
        return (1.0 < pc[2] < 200.0) and e <= 3.0 * cin["reprojection_error_std"], e

    F, L = prob["F"], prob["L"]
    fo, lro, lo = np.zeros(F, np.uint8), np.zeros(L, np.uint8), np.zeros(L, np.uint8)
    counts = np.zeros(5, np.int32)
    for l in range(L):
        facs = list(np.nonzero(np.asarray(prob["f_lm"]) == l)[0])
        seq = facs[:cin["lm_ref_pos"][l]] + [-1] + facs[cin["lm_ref_pos"][l]:]
        errs = []
        for f in seq:
            good, e = test(int(cin["lm_ref_node"][l]), l, cin["lm_ref_kp"][l]) if f < 0 else test(int(prob["f_obs"][f]), l, cin["f_kp"][f])
            if good:
                errs.append(e)
            elif f < 0:
                lro[l], lo[l] = 1, 1
                counts[0] += 1
                counts[2] += 1
                break
            else:
                fo[f] = 1
                counts[1] += 1
        if len(errs) < 2:
            lo[l] |= 2
            counts[0] += 1
            counts[3] += 1
        elif sum(errs) / len(errs) > cin["reprojection_error_std"]:
            lo[l] |= 4
            counts[0] += 1
            counts[4] += 1
    act = ((fo == 0) & (lo[np.asarray(prob["f_lm"], np.int64)] == 0)).astype(np.uint8) if F else np.zeros(0, np.uint8)
    return dict(ext_updated=upd, R_bc=Rb, t_bc=tb, counts=counts, f_outlier=fo, lm_ref_outlier=lro, lm_outlier=lo,
                cam_pose=np.array([np.concatenate([Rw[k].ravel(), tw[k]]) for k in range(prob["K"])]), lm_pos=pos, lm_depth=depth, f_active=act)


def assert_same(a, b, tol=1e-12):
    for k in ("ext_updated",):
        assert a[k] == b[k], k
    for k in ("counts", "f_outlier", "lm_ref_outlier", "lm_outlier", "f_active"):
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), k
    for k in ("R_bc", "t_bc", "cam_pose", "lm_pos", "lm_depth"):
        x, y = np.asarray(a[k], np.float64), np.asarray(b[k], np.float64)
        assert x.shape == y.shape and (x.size == 0 or np.abs(x - y).max() <= tol * max(1.0, np.abs(y).max())), k


def solved_cull_window(olib, seed, **kw):
    prob, cin, truth = synth_cull.make_cull_window(lambda *a: oa.preintegrate(olib, *a), seed=seed, **kw)
    po = copy.deepcopy(prob)
    removed = cc.two_pass(olib, po)
    return po, cin, truth, removed


@pytest.mark.parametrize("seed", [5, 6, 7])
def test_oracle_matches_restatement_on_solved_windows(olib, seed):
    po, cin, truth, removed = solved_cull_window(olib, seed)
    assert synth_cull.decision_margin(po, cin) > 1e-6  # no decision within rounding of its threshold at the solved parameters
    o = co.outlier_culling(po, cin)
    assert_same(o, restate(po, cin))
    c = o["counts"]
    assert c[1] > 0 and c[2] > 0 and c[3] > 0 and c[4] > 0 and o["ext_updated"] == 1
    assert c[0] == int(((o["lm_outlier"] & 1) > 0).sum() + ((o["lm_outlier"] & 6) > 0).sum())
    assert o["f_outlier"][truth["gross"]].mean() > 0.85  # gross outliers are flagged (unless the solve absorbed one along its epipolar line)
    assert np.all(o["lm_outlier"][truth["depth"]] & 1)  # depth outliers: num1 at the reference observation
    assert np.all(o["lm_outlier"][truth["depth"]] == 3)  # ... and num2 after the break


def test_hand_built_behaviours():
    prob, cin = cc.hand_window()
    o = co.outlier_culling(prob, cin)
    assert_same(o, restate(prob, cin))
    f = 0
    for l, (fo, bits, ro) in enumerate(cc.EXPECT):
        assert o["lm_outlier"][l] == bits and o["lm_ref_outlier"][l] == ro, l
        assert list(o["f_outlier"][f:f + len(fo)]) == fo, l
        f += len(fo)
    assert list(o["counts"]) == cc.EXPECT_COUNTS
    assert o["ext_updated"] == 1 and np.array_equal(o["R_bc"], np.eye(3))
    # the chi2-removed factor (4 px, f_active 0 on entry) is evaluated, kept, and active afterwards
    assert prob["f_active"][-2] == 0 and o["f_active"][-2] == 1 and o["f_active"][-1] == 1


@pytest.mark.parametrize("q,t,est,taken", [
    (cc.rot([0.3, 1.0, 0.2], 9.0), [0.1, 0.0, 0.0], 1, 1),   # sin(4.5 deg) * 57.3 = 4.5 < 5: accepted
    (cc.rot([0.3, 1.0, 0.2], 11.0), [0.0, 0.0, 0.0], 1, 0),  # 5.5 > 5: rejected
    (cc.rot([1.0, 0.0, 0.0], 1.0), [1.2, 0.0, 0.0], 1, 0),   # 1.2 m: rejected
    (cc.rot([0.3, 1.0, 0.2], 2.0), [0.1, 0.0, 0.0], 0, 0),   # estimate_extrinsic off: baseline kept
])
def test_extrinsic_gate(q, t, est, taken):
    prob, cin = cc.gate_window(np.array(q), np.array(t), est)
    prob["ext"][3:7] *= 1.001  # a solved quaternion is not exactly unit: normalised first
    o = co.outlier_culling(prob, cin)
    assert_same(o, restate(prob, cin))
    assert o["ext_updated"] == taken
    R = co.to_rotation_matrix(*co.quat_normalized(q[3], q[0], q[1], q[2]))
    assert np.allclose(o["R_bc"], R if taken else np.eye(3), atol=1e-15) and np.allclose(o["t_bc"], t if taken else 0.0)
    pose1 = o["cam_pose"][1]  # node 1 at (1, 0, 0), identity attitude: R_wc = R_bc, t_wc = p + t_bc
    assert np.allclose(pose1[:9], o["R_bc"].ravel()) and np.allclose(pose1[9:], np.array([1.0, 0, 0]) + o["t_bc"])


def test_culling_changes_the_marginalization_prior(olib):
    """gvinsMarginalization builds its reprojection factors from the map after the culling, not from the chi2-surviving set: on a window with
    outliers the two masks differ, and so do the priors."""
    po, cin, truth, removed = solved_cull_window(olib, 5)
    o = co.outlier_culling(po, cin)
    assert not np.array_equal(o["f_active"], po["f_active"])
    a, b = copy.deepcopy(po), copy.deepcopy(po)
    b["f_active"] = o["f_active"].copy()
    pa, pb = oa.ba_marginalize(olib, a, 1), oa.ba_marginalize(olib, b, 1)
    assert pa["r"] == pb["r"]
    sc = np.sqrt(np.abs(np.diag(pa["Hp"])))
    sc[sc == 0] = 1
    assert np.abs((pa["Hp"] - pb["Hp"]) / np.outer(sc, sc)).max() > 1e-6
