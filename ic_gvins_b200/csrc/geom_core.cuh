// geom_core.cuh -- __host__ __device__ cores of the point-wise front-end geometry and of the IMU propagation, shared by the host entry
// points (camera.cu, fundamental.cu, ba.cu: icg_camera_*, icg_find_fundamental_mat_ransac, icg_triangulate_points, icg_imu_preintegrate)
// and by their batched device versions (geom.cu).  One definition of the arithmetic -> host and device results agree to the last ulp of
// the libm calls.  References as in the callers (IG/ = ic_gvins/ic_gvins/).
#pragma once
#include <float.h>
#include <math.h>
#include <stdint.h>

#include "../../include/icgvins_b200.h"
#include "ba_math.cuh"

namespace icg {
namespace gc {

#define GC_HD __host__ __device__ inline

// ------------------------------------------------------------------------------------------------ camera model (IG/tracking/camera.cc)
GC_HD void pixel2cam(const icg_camera &c, double u, double v, double &x, double &y) {  // camera.cc:126-130
    y = (v - c.cy) / c.fy;
    x = (u - c.cx - c.skew * y) / c.fx;
}
GC_HD void cam2pixel(const icg_camera &c, double x, double y, double z, float &u, float &v) {  // camera.cc:132-134
    u = (float) ((c.fx * x + c.skew * y) / z + c.cx);
    v = (float) (c.fy * y / z + c.cy);
}
GC_HD void distort_xy(const icg_camera &c, double x, double y, double &xd, double &yd) {  // camera.cc:79-86
    const double r2 = x * x + y * y;
    const double rr = (1 + c.k1 * r2 + c.k2 * r2 * r2 + c.k3 * r2 * r2 * r2);
    xd = x * rr + 2 * c.p1 * x * y + c.p2 * (r2 + 2 * x * x);
    yd = y * rr + c.p1 * (r2 + 2 * y * y) + 2 * c.p2 * x * y;
}
// cv::undistortPoints(pts, pts, K, D, Mat(), K) on one point (calib3d: five fixed-point iterations, skew ignored when normalising, P = K)
GC_HD void undistort_point(const icg_camera &c, float *p) {
    const double ifx = 1.0 / c.fx, ify = 1.0 / c.fy;
    double x = ((double) p[0] - c.cx) * ifx, y = ((double) p[1] - c.cy) * ify;
    const double x0 = x, y0 = y;
    for (int j = 0; j < 5; j++) {
        const double r2 = x * x + y * y;
        const double icdist = 1.0 / (1 + ((c.k3 * r2 + c.k2) * r2 + c.k1) * r2);
        if (icdist < 0) {
            x = x0, y = y0;
            break;
        }
        const double dx = 2 * c.p1 * x * y + c.p2 * (r2 + 2 * x * x), dy = c.p1 * (r2 + 2 * y * y) + 2 * c.p2 * x * y;
        x = (x0 - dx) * icdist;
        y = (y0 - dy) * icdist;
    }
    p[0] = (float) (c.fx * x + c.skew * y + c.cx);
    p[1] = (float) (c.fy * y + c.cy);
}
GC_HD void distort_point(const icg_camera &c, float *p) {  // Camera::distortPoint (camera.cc:88-104)
    double x, y, xd, yd;
    pixel2cam(c, p[0], p[1], x, y);
    distort_xy(c, x, y, xd, yd);
    cam2pixel(c, xd, yd, 1.0, p[0], p[1]);
}

// ------------------------------------------------------------------------------------------------ cv::findFundamentalMat(FM_RANSAC)
struct CvRng {  // cv::RNG: multiply-with-carry, CV_RNG_COEFF = 4164903690
    uint64_t state;
    GC_HD explicit CvRng(uint64_t s = 0xffffffffffffffffull) : state(s ? s : 0xffffffffffffffffull) {}
    GC_HD unsigned next() {
        state = (uint64_t) (unsigned) state * 4164903690u + (unsigned) (state >> 32);
        return (unsigned) state;
    }
    GC_HD int uniform(int a, int b) { return a == b ? a : (int) (next() % (unsigned) (b - a) + a); }
};
// haveCollinearPoints (fundam.cpp): the LAST of `count` points against every pair of earlier ones
GC_HD bool collinear_last(const float *p, int count) {
    const int i = count - 1;
    for (int j = 0; j < i; j++) {
        const double dx1 = p[2 * j] - p[2 * i], dy1 = p[2 * j + 1] - p[2 * i + 1];
        for (int k = 0; k < j; k++) {
            const double dx2 = p[2 * k] - p[2 * i], dy2 = p[2 * k + 1] - p[2 * i + 1];
            if (fabs(dx2 * dy1 - dy2 * dx1) <= FLT_EPSILON * (fabs(dx1) + fabs(dy1) + fabs(dx2) + fabs(dy2))) return true;
        }
    }
    return false;
}
// RANSACPointSetRegistrator::getSubset: 7 distinct indices, redrawn while either image has collinear points (<= 10000 attempts)
GC_HD bool draw_subset(CvRng &rng, const float *p1, const float *p2, int n, int *idx) {
    float ms1[14], ms2[14];
    for (int attempts = 0; attempts < 10000; attempts++) {
        for (int i = 0; i < 7; i++) {
            int v;
            bool dup;
            do {
                v = rng.uniform(0, n);
                dup = false;
                for (int j = 0; j < i; j++) dup = dup || idx[j] == v;
            } while (dup);
            idx[i] = v;
            ms1[2 * i] = p1[2 * v], ms1[2 * i + 1] = p1[2 * v + 1], ms2[2 * i] = p2[2 * v], ms2[2 * i + 1] = p2[2 * v + 1];
        }
        if (collinear_last(ms1, 7) || collinear_last(ms2, 7)) continue;
        return true;
    }
    return false;
}
// cv::solveCubic: c[0] x^3 + c[1] x^2 + c[2] x + c[3] = 0, real roots in OpenCV's order
GC_HD int solve_cubic(const double c[4], double r[3]) {
    const double PI = 3.14159265358979323846;
    double a0 = c[0], a1 = c[1], a2 = c[2], a3 = c[3];
    if (a0 == 0) {
        if (a1 == 0) {
            if (a2 == 0) return a3 == 0 ? -1 : 0;
            r[0] = -a3 / a2;
            return 1;
        }
        double d = a2 * a2 - 4 * a1 * a3;
        if (d >= 0) {
            d = sqrt(d);
            const double q1 = (-a2 + d) * 0.5, q2 = (a2 + d) * -0.5;
            if (fabs(q1) > fabs(q2)) {
                r[0] = q1 / a1;
                r[1] = a3 / q1;
            } else {
                r[0] = q2 / a1;
                r[1] = a3 / q2;
            }
            return d > 0 ? 2 : 1;
        }
        return 0;
    }
    a0 = 1. / a0;
    a1 *= a0, a2 *= a0, a3 *= a0;
    const double Q = (a1 * a1 - 3 * a2) * (1. / 9), R = (2 * a1 * a1 * a1 - 9 * a1 * a2 + 27 * a3) * (1. / 54), Qcubed = Q * Q * Q;
    double d = Qcubed - R * R;
    if (d > 0) {
        const double theta = acos(R / sqrt(Qcubed)), sqrtQ = sqrt(Q), t0 = -2 * sqrtQ, t1 = theta * (1. / 3), t2 = a1 * (1. / 3);
        r[0] = t0 * cos(t1) - t2;
        r[1] = t0 * cos(t1 + (2. * PI / 3)) - t2;
        r[2] = t0 * cos(t1 + (4. * PI / 3)) - t2;
        return 3;
    }
    if (d == 0) {
        if (R >= 0) {
            r[0] = -2 * pow(R, 1. / 3) - a1 / 3;
            r[1] = pow(R, 1. / 3) - a1 / 3;
        } else {
            r[0] = 2 * pow(-R, 1. / 3) - a1 / 3;
            r[1] = -pow(-R, 1. / 3) - a1 / 3;
        }
        return 2;
    }
    d = sqrt(-d);
    double e = pow(d + fabs(R), 1. / 3);
    if (R > 0) e = -e;
    r[0] = (e + Q / e) - a1 * (1. / 3);
    return 1;
}
// right null space of the 7 x 9 system: one-sided (Hestenes) Jacobi on the columns of A; the two columns of V whose A-images have the
// smallest norms span it.  f1 = v7, f2 = v8 in the descending-singular-value order of cv::SVDecomp.
GC_HD void null_space_7x9(const double a[7 * 9], double f1[9], double f2[9]) {
    double G[9][7], V[9][9];
    for (int c = 0; c < 9; c++) {
        for (int r = 0; r < 7; r++) G[c][r] = a[r * 9 + c];
        for (int r = 0; r < 9; r++) V[c][r] = r == c ? 1.0 : 0.0;
    }
    for (int sweep = 0; sweep < 60; sweep++) {
        bool rotated = false;
        for (int p = 0; p < 8; p++)
            for (int q = p + 1; q < 9; q++) {
                double al = 0, be = 0, ga = 0;
                for (int r = 0; r < 7; r++) al += G[p][r] * G[p][r], be += G[q][r] * G[q][r], ga += G[p][r] * G[q][r];
                if (ga == 0.0 || fabs(ga) <= 1e-16 * sqrt(al * be)) continue;
                rotated = true;
                const double zeta = (be - al) / (2.0 * ga);
                const double t = (zeta >= 0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
                const double cs = 1.0 / sqrt(1.0 + t * t), sn = cs * t;
                for (int r = 0; r < 7; r++) {
                    const double x = G[p][r], y = G[q][r];
                    G[p][r] = cs * x - sn * y, G[q][r] = sn * x + cs * y;
                }
                for (int r = 0; r < 9; r++) {
                    const double x = V[p][r], y = V[q][r];
                    V[p][r] = cs * x - sn * y, V[q][r] = sn * x + cs * y;
                }
            }
        if (!rotated) break;
    }
    int order[9];
    double nrm[9];
    for (int c = 0; c < 9; c++) {
        order[c] = c, nrm[c] = 0;
        for (int r = 0; r < 7; r++) nrm[c] += G[c][r] * G[c][r];
    }
    for (int i = 1; i < 9; i++) {  // stable insertion sort, descending norm (== std::stable_sort with nrm[x] > nrm[y])
        const int oi = order[i];
        int j = i - 1;
        while (j >= 0 && nrm[order[j]] < nrm[oi]) order[j + 1] = order[j], j--;
        order[j + 1] = oi;
    }
    for (int r = 0; r < 9; r++) f1[r] = V[order[7]][r], f2[r] = V[order[8]][r];
}
// run7Point (fundam.cpp): up to three fundamental matrices through seven correspondences
GC_HD int run_7point(const float *m1, const float *m2, double F[3][9]) {
    double a[7 * 9], f1[9], f2[9], c[4], r[3] = {0, 0, 0};
    for (int i = 0; i < 7; i++) {
        const double x0 = m1[2 * i], y0 = m1[2 * i + 1], x1 = m2[2 * i], y1 = m2[2 * i + 1];
        double *row = a + i * 9;
        row[0] = x1 * x0, row[1] = x1 * y0, row[2] = x1, row[3] = y1 * x0, row[4] = y1 * y0, row[5] = y1, row[6] = x0, row[7] = y0, row[8] = 1;
    }
    null_space_7x9(a, f1, f2);
    for (int i = 0; i < 9; i++) f1[i] -= f2[i];
    double t0 = f2[4] * f2[8] - f2[5] * f2[7], t1 = f2[3] * f2[8] - f2[5] * f2[6], t2 = f2[3] * f2[7] - f2[4] * f2[6];
    c[3] = f2[0] * t0 - f2[1] * t1 + f2[2] * t2;
    c[2] = f1[0] * t0 - f1[1] * t1 + f1[2] * t2 - f1[3] * (f2[1] * f2[8] - f2[2] * f2[7]) + f1[4] * (f2[0] * f2[8] - f2[2] * f2[6]) -
           f1[5] * (f2[0] * f2[7] - f2[1] * f2[6]) + f1[6] * (f2[1] * f2[5] - f2[2] * f2[4]) - f1[7] * (f2[0] * f2[5] - f2[2] * f2[3]) +
           f1[8] * (f2[0] * f2[4] - f2[1] * f2[3]);
    t0 = f1[4] * f1[8] - f1[5] * f1[7], t1 = f1[3] * f1[8] - f1[5] * f1[6], t2 = f1[3] * f1[7] - f1[4] * f1[6];
    c[0] = f1[0] * t0 - f1[1] * t1 + f1[2] * t2;
    c[1] = f2[0] * t0 - f2[1] * t1 + f2[2] * t2 - f2[3] * (f1[1] * f1[8] - f1[2] * f1[7]) + f2[4] * (f1[0] * f1[8] - f1[2] * f1[6]) -
           f2[5] * (f1[0] * f1[7] - f1[1] * f1[6]) + f2[6] * (f1[1] * f1[5] - f1[2] * f1[4]) - f2[7] * (f1[0] * f1[5] - f1[2] * f1[3]) +
           f2[8] * (f1[0] * f1[4] - f1[1] * f1[3]);
    const int n = solve_cubic(c, r);
    if (n < 1 || n > 3) return n;
    for (int k = 0; k < n; k++) {
        double lambda = r[k], mu = 1.;
        const double s = f1[8] * r[k] + f2[8];
        if (fabs(s) > DBL_EPSILON) {  // normalise so that F(3,3) == 1
            mu = 1. / s;
            lambda *= mu;
            F[k][8] = 1.;
        } else {
            F[k][8] = 0.;
        }
        for (int i = 0; i < 8; i++) F[k][i] = f1[i] * lambda + f2[i] * mu;
    }
    return n;
}
// FMEstimatorCallback::computeError + findInliers (ptsetreg.cpp) for pair i: err = max(d1^2 s1, d2^2 s2) rounded to float <= thresh^2
GC_HD bool is_inlier(const float *m1, const float *m2, int i, const double *F, double thresh) {
    const float t = (float) (thresh * thresh);
    const double x1 = m1[2 * i], y1 = m1[2 * i + 1], x2 = m2[2 * i], y2 = m2[2 * i + 1];
    double a = F[0] * x1 + F[1] * y1 + F[2], b = F[3] * x1 + F[4] * y1 + F[5], c = F[6] * x1 + F[7] * y1 + F[8];
    const double s2 = 1. / (a * a + b * b), d2 = x2 * a + y2 * b + c;
    a = F[0] * x2 + F[3] * y2 + F[6], b = F[1] * x2 + F[4] * y2 + F[7], c = F[2] * x2 + F[5] * y2 + F[8];
    const double s1 = 1. / (a * a + b * b), d1 = x1 * a + y1 * b + c;
    const double e1 = d1 * d1 * s1, e2 = d2 * d2 * s2;
    const float err = (float) (e1 > e2 ? e1 : e2);  // std::max(a, b): b unless a > b... max(a, b) = (a < b) ? b : a
    return err <= t;
}
inline int update_num_iters(double p, double ep, int model_points, int max_iters) {  // RANSACUpdateNumIters (host: replay loop only)
    p = p < 0. ? 0. : p > 1. ? 1. : p, ep = ep < 0. ? 0. : ep > 1. ? 1. : ep;
    double num = 1. - p > DBL_MIN ? 1. - p : DBL_MIN, denom = 1. - pow(1. - ep, model_points);
    if (denom < DBL_MIN) return 0;
    num = log(num), denom = log(denom);
    return denom >= 0 || -num >= max_iters * (-denom) ? max_iters : (int) lrint(num / denom);
}

// ------------------------------------------------------------------------------------------------ Tracking::triangulatePoint (tracking.cc:796-808)
// rows of the 4 x 4 design matrix: pc0.x P0.row(2) - P0.row(0), pc0.y P0.row(2) - P0.row(1), pc1.x P1.row(2) - P1.row(0), pc1.y P1.row(2) - P1.row(1)
// (P = T_c_w, 3 x 4 row-major); pw = right singular vector of the smallest singular value (one-sided Jacobi), dehomogenised
GC_HD void triangulate_point(const double *P0, const double *P1, const double *pc0, const double *pc1, double *pw) {
    double G[4][4], V[4][4];
    for (int c = 0; c < 4; c++) {
        G[c][0] = pc0[0] * P0[8 + c] - P0[c];
        G[c][1] = pc0[1] * P0[8 + c] - P0[4 + c];
        G[c][2] = pc1[0] * P1[8 + c] - P1[c];
        G[c][3] = pc1[1] * P1[8 + c] - P1[4 + c];
        for (int r = 0; r < 4; r++) V[c][r] = r == c ? 1.0 : 0.0;
    }
    for (int sweep = 0; sweep < 60; sweep++) {
        bool rotated = false;
        for (int p = 0; p < 3; p++)
            for (int q = p + 1; q < 4; q++) {
                double al = 0, be = 0, ga = 0;
                for (int r = 0; r < 4; r++) al += G[p][r] * G[p][r], be += G[q][r] * G[q][r], ga += G[p][r] * G[q][r];
                if (ga == 0.0 || fabs(ga) <= 1e-16 * sqrt(al * be)) continue;
                rotated = true;
                const double zeta = (be - al) / (2.0 * ga);
                const double t = (zeta >= 0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
                const double cs = 1.0 / sqrt(1.0 + t * t), sn = cs * t;
                for (int r = 0; r < 4; r++) {
                    const double x = G[p][r], y = G[q][r];
                    G[p][r] = cs * x - sn * y, G[q][r] = sn * x + cs * y;
                    const double vx = V[p][r], vy = V[q][r];
                    V[p][r] = cs * vx - sn * vy, V[q][r] = sn * vx + cs * vy;
                }
            }
        if (!rotated) break;
    }
    int best = 0;
    double bn = 1e300;
    for (int c = 0; c < 4; c++) {
        double nn = 0;
        for (int r = 0; r < 4; r++) nn += G[c][r] * G[c][r];
        if (nn < bn) bn = nn, best = c;
    }
    for (int k = 0; k < 3; k++) pw[k] = V[best][k] / V[best][3];
}

// ------------------------------------------------------------------------------------------------ IMU preintegration propagation
// PreintegrationEarth::resetState / integrationProcess / updateJacobianAndCovariance (IG/preintegration/preintegration_earth.cc:205-338) or, with
// iewn3 == NULL, PreintegrationNormal (PreintegrationBase::integration, preintegration_base.cc:39-70 + preintegration_normal.cc:195-232).
// state16 = p[3] q_xyzw[4] v[3] bg[3] ba[3]; noise5 = gyr_arw, acc_vrw, gyr_bias_std, acc_bias_std, corr_time; imu = n rows (dt, dtheta[3], dvel[3]).
GC_HD void preintegrate_core(const double *state16, const double *iewn3, const double *gravity3, const double *noise5, const double *imu, int n, double *blob,
                             double *end_state10) {
    using namespace bam;
    const bool normal = iewn3 == nullptr;
    V3 cur_p = mk(state16[0], state16[1], state16[2]), cur_v = mk(state16[7], state16[8], state16[9]);
    Q cur_q = mkq(state16[6], state16[3], state16[4], state16[5]);
    const Q q0 = cur_q;
    const V3 bg = mk(state16[10], state16[11], state16[12]), ba = mk(state16[13], state16[14], state16[15]);
    const V3 iewn = normal ? mk(0, 0, 0) : mk(iewn3[0], iewn3[1], iewn3[2]), grav = mk(gravity3[0], gravity3[1], gravity3[2]);
    const double corr = noise5[4];
    double noise[12];
    for (int k = 0; k < 3; k++) {
        noise[k] = noise5[0] * noise5[0], noise[3 + k] = noise5[1] * noise5[1];
        noise[6 + k] = 2 * noise5[2] * noise5[2] / corr, noise[9 + k] = 2 * noise5[3] * noise5[3] / corr;
    }
    double jac[225], cov[225];
    for (int i = 0; i < 225; i++) jac[i] = 0, cov[i] = 0;
    for (int i = 0; i < 15; i++) jac[i * 15 + i] = 1;
    V3 dp = mk(0, 0, 0), dv = mk(0, 0, 0);
    Q dq = mkq(1, 0, 0, 0);
    double delta_time = 0, s0 = 0;
    V3 s1 = mk(0, 0, 0);
    for (int s = 1; s < n; s++) {
        const double *pr = imu + 7 * (size_t) (s - 1), *cu = imu + 7 * (size_t) s;
        const double dt = cu[0];
        V3 pth = mk(pr[1], pr[2], pr[3]) - pr[0] * bg, pvl = mk(pr[4], pr[5], pr[6]) - pr[0] * ba;  // compensationBias (preintegration_base.cc:84-90)
        V3 cth = mk(cu[1], cu[2], cu[3]) - dt * bg, cvl = mk(cu[4], cu[5], cu[6]) - dt * ba;
        delta_time += dt;
        V3 dvfb = cvl + 0.5 * cross(cth, cvl) + (1.0 / 12.0) * (cross(pth, cvl) + cross(pvl, cth));
        V3 dtheta = cth + (1.0 / 12.0) * cross(pth, cth);
        M3 cbb0;
        if (!normal) {
            V3 dv_cor_g = dt * (grav - 2.0 * cross(iewn, cur_v));
            Q qnn = rotvec2q(-(dt * iewn));
            V3 dvel = mul(scale(0.5, add(ident(), qmat(qnn))), mul(qmat(cur_q), dvfb)) + dv_cor_g;
            cur_p = cur_p + dt * cur_v + (0.5 * dt) * dvel;
            cur_v = cur_v + dvel;
            s0 += dt;
            s1 = s1 + dt * cur_p;
            cur_q = qnormalized(qmul(qmul(qnn, cur_q), rotvec2q(dtheta)));
            V3 dnn = -((delta_time - 0.5 * dt) * iewn);
            dvel = mul(qmat(qmul(qmul(qmul(qinv(q0), rotvec2q(dnn)), q0), dq)), dvfb);
            dp = dp + dt * dv + (0.5 * dt) * dvel;
            dv = dv + dvel;
            dq = qnormalized(qmul(dq, rotvec2q(dtheta)));
            cbb0 = neg(qmat(qmul(qmul(qmul(qinv(q0), rotvec2q(-(delta_time * iewn))), q0), dq)));
        } else {
            V3 dvel = mul(qmat(cur_q), dvfb) + dt * grav;
            cur_p = cur_p + dt * cur_v + (0.5 * dt) * dvel;
            cur_v = cur_v + dvel;
            cur_q = qnormalized(qmul(cur_q, rotvec2q(dtheta)));
            dvel = mul(qmat(dq), dvfb);
            dp = dp + dt * dv + (0.5 * dt) * dvel;
            dv = dv + dvel;
            dq = qnormalized(qmul(dq, rotvec2q(dtheta)));
            // phi(3,6) = -R(dq) [dvel]x, phi(3,12) = -R(dq) dt; gt(3,3) = R(dq), gt(6,0) = +I (preintegration_normal.cc:207-225): with a diagonal
            // noise matrix G = gt noise gt^T does not see the sign of a column block of gt, so the Earth form below with cbb0 = -R(dq) is the same
            cbb0 = neg(qmat(dq));
        }
        // updateJacobianAndCovariance: phi = I + F dt; the non-trivial blocks are applied directly (phi is sparse)
        double phi[225], gt[180];
        for (int i = 0; i < 225; i++) phi[i] = 0;
        for (int i = 0; i < 180; i++) gt[i] = 0;
        auto put = [](double *M, int nc, int r0, int c0, const M3 &m) {
            for (int i = 0; i < 3; i++)
                for (int j = 0; j < 3; j++) M[(r0 + i) * nc + c0 + j] = m.m[3 * i + j];
        };
        put(phi, 15, 0, 0, ident());
        put(phi, 15, 0, 3, scale(dt, ident()));
        put(phi, 15, 3, 3, ident());
        put(phi, 15, 3, 6, mul(cbb0, skew(cvl)));
        put(phi, 15, 3, 12, scale(dt, cbb0));
        put(phi, 15, 6, 6, sub(ident(), skew(cth)));
        put(phi, 15, 6, 9, scale(-dt, ident()));
        put(phi, 15, 9, 9, scale(1 - dt / corr, ident()));
        put(phi, 15, 12, 12, scale(1 - dt / corr, ident()));
        double tmp[225];
        for (int i = 0; i < 15; i++)
            for (int j = 0; j < 15; j++) {
                double a = 0;
                for (int k = 0; k < 15; k++) a += phi[i * 15 + k] * jac[k * 15 + j];
                tmp[i * 15 + j] = a;
            }
        for (int i = 0; i < 225; i++) jac[i] = tmp[i];
        put(gt, 12, 3, 3, cbb0);
        put(gt, 12, 6, 0, neg(ident()));
        put(gt, 12, 9, 6, ident());
        put(gt, 12, 12, 9, ident());
        double G[225], pg[225], pc[225];
        for (int i = 0; i < 15; i++)
            for (int j = 0; j < 15; j++) {
                double a = 0;
                for (int k = 0; k < 12; k++) a += gt[i * 12 + k] * noise[k] * gt[j * 12 + k];
                G[i * 15 + j] = a;
            }
        for (int i = 0; i < 15; i++)
            for (int j = 0; j < 15; j++) {
                double a = 0, c = 0;
                for (int k = 0; k < 15; k++) a += phi[i * 15 + k] * G[k * 15 + j], c += phi[i * 15 + k] * cov[k * 15 + j];
                pg[i * 15 + j] = a, pc[i * 15 + j] = c;
            }
        for (int i = 0; i < 15; i++)
            for (int j = 0; j < 15; j++) {
                double a = 0, gpt = 0;
                for (int k = 0; k < 15; k++) a += pc[i * 15 + k] * phi[j * 15 + k], gpt += G[i * 15 + k] * phi[j * 15 + k];
                tmp[i * 15 + j] = a + 0.5 * dt * (pg[i * 15 + j] + gpt);
            }
        for (int i = 0; i < 225; i++) cov[i] = tmp[i];
    }
    for (int i = 0; i < ICG_IMU_BLOB_DOUBLES; i++) blob[i] = 0;
    blob[0] = delta_time;
    blob[1] = dp.x, blob[2] = dp.y, blob[3] = dp.z, blob[4] = dv.x, blob[5] = dv.y, blob[6] = dv.z;
    blob[7] = dq.x, blob[8] = dq.y, blob[9] = dq.z, blob[10] = dq.w;
    for (int k = 0; k < 3; k++) blob[11 + k] = state16[10 + k], blob[14 + k] = state16[13 + k], blob[17 + k] = gravity3[k];
    blob[20] = iewn.x, blob[21] = iewn.y, blob[22] = iewn.z;
    blob[23] = s0, blob[24] = s1.x, blob[25] = s1.y, blob[26] = s1.z;
    for (int i = 0; i < 225; i++) blob[27 + i] = jac[i], blob[252 + i] = cov[i];
    blob[477] = normal ? 1.0 : 0.0;
    if (end_state10) {
        end_state10[0] = cur_p.x, end_state10[1] = cur_p.y, end_state10[2] = cur_p.z;
        end_state10[3] = cur_q.x, end_state10[4] = cur_q.y, end_state10[5] = cur_q.z, end_state10[6] = cur_q.w;
        end_state10[7] = cur_v.x, end_state10[8] = cur_v.y, end_state10[9] = cur_v.z;
    }
}

// ------------------------------------------------------------------------------------------------ post-solve update + outlier culling
// GVINS::updateParametersFromOptimizer (IG/ic_gvins.cc:1299-1389) and the per-observation test of GVINS::gvinsOutlierCulling (:1035-1128).
// Written out operation by operation (no library products) so that host, device and a plain scalar restatement
// round alike; the device copy is compiled without FMA contraction (the float cast in cam2pixel makes the decisions sensitive to it).
// Eigen's Quaternion::normalized(): coeffs (x, y, z, w) / sqrt(squaredNorm), squared norm summed in storage order
GC_HD bam::Q quat_normalized(bam::Q q) {
    const double n = sqrt(((q.x * q.x + q.y * q.y) + q.z * q.z) + q.w * q.w);
    return bam::mkq(q.w / n, q.x / n, q.y / n, q.z / n);
}
// Eigen's Quaternion(const Matrix3 &) (quaternionbase_assign_impl<Other, 3, 3>), row-major R
GC_HD bam::Q rot_to_quat(const double *R) {
    bam::Q q;
    double t = (R[0] + R[4]) + R[8];
    if (t > 0.0) {
        t = sqrt(t + 1.0);
        q.w = 0.5 * t;
        t = 0.5 / t;
        q.x = (R[7] - R[5]) * t;
        q.y = (R[2] - R[6]) * t;
        q.z = (R[3] - R[1]) * t;
    } else {
        int i = 0;
        if (R[4] > R[0]) i = 1;
        if (R[8] > R[3 * i + i]) i = 2;
        const int j = (i + 1) % 3, k = (j + 1) % 3;
        double c[3];
        t = sqrt(((R[3 * i + i] - R[3 * j + j]) - R[3 * k + k]) + 1.0);
        c[i] = 0.5 * t;
        t = 0.5 / t;
        q.w = (R[3 * k + j] - R[3 * j + k]) * t;
        c[j] = (R[3 * j + i] + R[3 * i + j]) * t;
        c[k] = (R[3 * k + i] + R[3 * i + k]) * t;
        q.x = c[0], q.y = c[1], q.z = c[2];
    }
    return q;
}
// the extrinsic gate of updateParametersFromOptimizer (:1311-1331): candidate (t, R) from ext = (t, q_xyzw, td), accepted unless
// |t - t_bc| > 1 m or |vec(quaternion(R R_bc^T))| * R2D > 5 (sin(theta / 2) in "degrees": the gate trips near theta = 10 deg, as written).
// R_bc / t_bc are updated in place; returns 1 when the candidate was taken.
GC_HD int extrinsic_gate(const double *ext, double *R_bc, double *t_bc) {
    const bam::Q q = quat_normalized(bam::mkq(ext[6], ext[3], ext[4], ext[5]));
    const bam::M3 R = bam::qmat(q);
    const double dx = ext[0] - t_bc[0], dy = ext[1] - t_bc[1], dz = ext[2] - t_bc[2];
    const double dt = sqrt((dx * dx + dy * dy) + dz * dz);
    bam::M3 Rb;
    for (int i = 0; i < 9; i++) Rb.m[i] = R_bc[i];
    const bam::M3 D = bam::mul(R, bam::tr(Rb));
    const bam::Q qd = rot_to_quat(D.m);
    const double dr = sqrt((qd.x * qd.x + qd.y * qd.y) + qd.z * qd.z) * (180.0 / 3.14159265358979323846);
    if (dt > 1.0 || dr > 5.0) return 0;
    for (int i = 0; i < 9; i++) R_bc[i] = R.m[i];
    for (int i = 0; i < 3; i++) t_bc[i] = ext[i];
    return 1;
}
// MISC::stateToCameraPose (IG/misc.cc:102-108) of a node pose7 = (p, q_xyzw): R_wc = R(q) R_bc, t_wc = p + R(q) t_bc (q normalised first,
// PreintegrationBase::stateFromData, preintegration_base.cc:115-125)
GC_HD void camera_pose(const double *pose7, const double *R_bc, const double *t_bc, double *R_wc, double *t_wc) {
    const bam::M3 Rq = bam::qmat(quat_normalized(bam::mkq(pose7[6], pose7[3], pose7[4], pose7[5])));
    bam::M3 Rb;
    for (int i = 0; i < 9; i++) Rb.m[i] = R_bc[i];
    const bam::M3 Rw = bam::mul(Rq, Rb);
    const bam::V3 rt = bam::mul(Rq, bam::mk(t_bc[0], t_bc[1], t_bc[2]));
    for (int i = 0; i < 9; i++) R_wc[i] = Rw.m[i];
    t_wc[0] = pose7[0] + rt.x, t_wc[1] = pose7[1] + rt.y, t_wc[2] = pose7[2] + rt.z;
}
// map point from its reference key point and inverse depth (:1379-1386): pos = R_ref (pixel2cam(kp) * depth) + t_ref, depth = 1 / invdepth
GC_HD void mappoint_position(const icg_camera &c, const double *R_ref, const double *t_ref, float ku, float kv, double invdepth, double *pos, double &depth) {
    depth = 1.0 / invdepth;
    double x, y;
    pixel2cam(c, ku, kv, x, y);
    const bam::V3 pw = bam::mul(*(const bam::M3 *) R_ref, bam::mk(x * depth, y * depth, 1.0 * depth));
    pos[0] = pw.x + t_ref[0], pos[1] = pw.y + t_ref[1], pos[2] = pw.z + t_ref[2];
}
// Tracking::isGoodToTrack(kp, pose, pos, scale) (IG/tracking/tracking.cc:813-828): depth gate 1 < z_c < 200 (isGoodDepth, :247-249) and the
// reprojection error |world2pixel(pos) - kp| (Camera::reprojectionError, camera.cc:153-157: float difference, double norm) <= threshold.
// err receives that error; it is what gvinsOutlierCulling averages (:1075).
GC_HD bool good_to_track(const icg_camera &c, const double *R_wc, const double *t_wc, const double *pos, float ku, float kv, double threshold, double &err) {
    const double vx = pos[0] - t_wc[0], vy = pos[1] - t_wc[1], vz = pos[2] - t_wc[2];
    const double pcx = (R_wc[0] * vx + R_wc[3] * vy) + R_wc[6] * vz;  // R^T (pw - t)
    const double pcy = (R_wc[1] * vx + R_wc[4] * vy) + R_wc[7] * vz;
    const double pcz = (R_wc[2] * vx + R_wc[5] * vy) + R_wc[8] * vz;
    float u, v;
    cam2pixel(c, pcx, pcy, pcz, u, v);
    const double ex = (double) (u - ku), ey = (double) (v - kv);
    err = sqrt(ex * ex + ey * ey);
    if (!(pcz > 1.0 && pcz < 200.0)) return false;
    return !(err > threshold);
}

}  // namespace gc
}  // namespace icg
