"""CPU restatement of the end of GVINS::gvinsOptimization (TEST INFRASTRUCTURE ONLY): updateParametersFromOptimizer
(ic_gvins/ic_gvins/ic_gvins.cc:1299-1389) and gvinsOutlierCulling (:1035-1128), line by line, in Python scalars.

Python floats are IEEE doubles without contraction, np.float32 rounds to nearest, and the operation order is that of the Eigen / OpenCV
calls the reference makes (written out as in csrc/geom_core.cuh), so the results are those of an uncontracted FP64 build of the reference.
The map is modelled as the window holds it: landmark l has the observations [reference observation at lm_ref_pos[l], its factors in
ascending factor index around it] (mappoint->observations() in insertion order), every one of them in a keyframe of the window.
"""
import math

import numpy as np

R2D = 180.0 / math.pi
F32 = np.float32


def quat_normalized(w, x, y, z):  # Eigen Quaternion::normalized(): coeffs (x, y, z, w) / sqrt(squaredNorm)
    n = math.sqrt(((x * x + y * y) + z * z) + w * w)
    return w / n, x / n, y / n, z / n


def to_rotation_matrix(w, x, y, z):  # Eigen QuaternionBase::toRotationMatrix, row-major 3 x 3 list
    tx, ty, tz = 2 * x, 2 * y, 2 * z
    twx, twy, twz = tx * w, ty * w, tz * w
    txx, txy, txz, tyy, tyz, tzz = tx * x, ty * x, tz * x, ty * y, tz * y, tz * z
    return [[1 - (tyy + tzz), txy - twz, txz + twy], [txy + twz, 1 - (txx + tzz), tyz - twx], [txz - twy, tyz + twx, 1 - (txx + tyy)]]


def from_rotation_matrix(m):  # Eigen Quaternion(const Matrix3d &): returns (w, x, y, z)
    t = (m[0][0] + m[1][1]) + m[2][2]
    if t > 0.0:
        t = math.sqrt(t + 1.0)
        w = 0.5 * t
        t = 0.5 / t
        return w, (m[2][1] - m[1][2]) * t, (m[0][2] - m[2][0]) * t, (m[1][0] - m[0][1]) * t
    i = 0
    if m[1][1] > m[0][0]:
        i = 1
    if m[2][2] > m[i][i]:
        i = 2
    j, k = (i + 1) % 3, (i + 2) % 3
    c = [0.0, 0.0, 0.0]
    t = math.sqrt(((m[i][i] - m[j][j]) - m[k][k]) + 1.0)
    c[i] = 0.5 * t
    t = 0.5 / t
    w = (m[k][j] - m[j][k]) * t
    c[j] = (m[j][i] + m[i][j]) * t
    c[k] = (m[k][i] + m[i][k]) * t
    return w, c[0], c[1], c[2]


def matmul(a, b):
    return [[(a[i][0] * b[0][j] + a[i][1] * b[1][j]) + a[i][2] * b[2][j] for j in range(3)] for i in range(3)]


def matvec(a, v):
    return [(a[i][0] * v[0] + a[i][1] * v[1]) + a[i][2] * v[2] for i in range(3)]


def transpose(a):
    return [[a[j][i] for j in range(3)] for i in range(3)]


def pixel2cam(cam, u, v):  # Camera::pixel2cam (IG/tracking/camera.cc:126-130), u / v float key point
    fx, fy, cx, cy, skew = cam[:5]
    y = (float(v) - cy) / fy
    x = (float(u) - cx - skew * y) / fx
    return x, y


def cam2pixel(cam, pc):  # Camera::cam2pixel (:132-134): cv::Point2f of doubles
    fx, fy, cx, cy, skew = cam[:5]
    return F32((fx * pc[0] + skew * pc[1]) / pc[2] + cx), F32(fy * pc[1] / pc[2] + cy)


def world2cam(pw, R, t):  # Camera::world2cam: R^T (pw - t)
    return matvec(transpose(R), [pw[0] - t[0], pw[1] - t[1], pw[2] - t[2]])


def reprojection_error(cam, R, t, pw, kp):  # Camera::reprojectionError (:153-157) .norm(): float difference, double norm
    u, v = cam2pixel(cam, world2cam(pw, R, t))
    ex, ey = float(u - F32(kp[0])), float(v - F32(kp[1]))
    return math.sqrt(ex * ex + ey * ey)


def is_good_to_track(cam, std, kp, R, t, pw, scale=3.0):  # Tracking::isGoodToTrack (tracking.cc:813-828) + isGoodDepth (:247-249)
    pc = world2cam(pw, R, t)
    if not (pc[2] > 1.0 and pc[2] < 200.0):
        return False
    return not (reprojection_error(cam, R, t, pw, kp) > std * scale)


def update_parameters(prob, cin):
    """updateParametersFromOptimizer: (ext_updated, R_bc, t_bc, camera poses [(R, t)] per node, map points, depths)."""
    ext = [float(x) for x in prob["ext"]]
    R_bc = [[float(cin["R_bc"][i][j]) for j in range(3)] for i in range(3)]
    t_bc = [float(x) for x in cin["t_bc"]]
    updated = 0
    if cin["estimate_extrinsic"]:
        t = ext[0:3]
        R = to_rotation_matrix(*quat_normalized(ext[6], ext[3], ext[4], ext[5]))
        d = [t[0] - t_bc[0], t[1] - t_bc[1], t[2] - t_bc[2]]
        dt = math.sqrt((d[0] * d[0] + d[1] * d[1]) + d[2] * d[2])
        _, qx, qy, qz = from_rotation_matrix(matmul(R, transpose(R_bc)))
        dr = math.sqrt((qx * qx + qy * qy) + qz * qz) * R2D
        if not (dt > 1.0 or dr > 5.0):
            R_bc, t_bc, updated = R, t, 1
    pose = np.asarray(prob["pose"], np.float64).reshape(-1, 7)
    poses = []
    for k in range(prob["K"]):  # MISC::stateToCameraPose (misc.cc:102-108)
        p = [float(x) for x in pose[k]]
        Rq = to_rotation_matrix(*quat_normalized(p[6], p[3], p[4], p[5]))
        rt = matvec(Rq, t_bc)
        poses.append((matmul(Rq, R_bc), [p[0] + rt[0], p[1] + rt[1], p[2] + rt[2]]))
    pos, depths = [], []
    for l in range(prob["L"]):
        depth = 1.0 / float(prob["invdepth"][l])
        x, y = pixel2cam(cin["cam"], F32(cin["lm_ref_kp"][l][0]), F32(cin["lm_ref_kp"][l][1]))
        R, t = poses[int(cin["lm_ref_node"][l])]
        pc = matvec(R, [x * depth, y * depth, 1.0 * depth])
        pos.append([pc[0] + t[0], pc[1] + t[1], pc[2] + t[2]])
        depths.append(depth)
    return updated, R_bc, t_bc, poses, pos, depths


def outlier_culling(prob, cin):
    """updateParametersFromOptimizer + gvinsOutlierCulling on one window.  Returns the dict WindowSolver.outlier_culling returns, plus
    `f_active` = the mask gvinsMarginalization would find in the map."""
    updated, R_bc, t_bc, poses, pos, depths = update_parameters(prob, cin)
    F, L, std, cam = prob["F"], prob["L"], float(cin["reprojection_error_std"]), cin["cam"]
    f_lm = np.asarray(prob["f_lm"])
    facs = [[] for _ in range(L)]
    for f in range(F):
        facs[int(f_lm[f])].append(f)
    f_outlier = np.zeros(F, np.uint8)
    lm_ref_outlier = np.zeros(L, np.uint8)
    lm_outlier = np.zeros(L, np.uint8)
    n_map = n_feat = num1 = num2 = num3 = 0
    for l in range(L):
        obs = [("f", f) for f in facs[l]]
        obs.insert(int(cin["lm_ref_pos"][l]), ("ref", l))
        errors = []
        for kind, i in obs:
            if kind == "ref":
                R, t = poses[int(cin["lm_ref_node"][l])]
                kp = cin["lm_ref_kp"][l]
            else:
                R, t = poses[int(prob["f_obs"][i])]
                kp = cin["f_kp"][i]
            error = reprojection_error(cam, R, t, pos[l], kp)
            if not is_good_to_track(cam, std, kp, R, t, pos[l]):
                if kind == "ref":
                    lm_ref_outlier[l] = 1
                    lm_outlier[l] |= 1
                    n_map += 1
                    num1 += 1
                    break
                f_outlier[i] = 1
                n_feat += 1
            else:
                errors.append(error)
        if len(errors) < 2:
            lm_outlier[l] |= 2
            n_map += 1
            num2 += 1
        else:
            acc = 0.0
            for e in errors:  # std::accumulate(begin, end, 0.0)
                acc = acc + e
            if acc / float(len(errors)) > std:
                lm_outlier[l] |= 4
                n_map += 1
                num3 += 1
    f_active = np.array([0 if (f_outlier[f] or lm_outlier[f_lm[f]]) else 1 for f in range(F)], np.uint8)
    cam_pose = np.array([[*R[0], *R[1], *R[2], *t] for R, t in poses], np.float64).reshape(-1, 12)
    return dict(ext_updated=updated, R_bc=np.array(R_bc), t_bc=np.array(t_bc), counts=np.array([n_map, n_feat, num1, num2, num3], np.int32),
                f_outlier=f_outlier, lm_ref_outlier=lm_ref_outlier, lm_outlier=lm_outlier, cam_pose=cam_pose,
                lm_pos=np.array(pos, np.float64).reshape(-1, 3), lm_depth=np.array(depths), f_active=f_active)
