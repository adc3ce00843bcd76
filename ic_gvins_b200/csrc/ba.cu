// ba.cu -- Path B: batched sliding-window factor-graph solve on sm_100a.
//
// Replaces `ceres::Solver::Solve` (LEVENBERG_MARQUARDT + DENSE_SCHUR, IG/ic_gvins.cc:1143-1146,1183,1217) and the
// per-factor `CostFunction::Evaluate` calls Ceres drives (IG/factors/*.h, IG/preintegration/*.h) for MANY independent
// windows at once (throughput mode: one window per stream).  Ceres is an un-vendored dependency of the reference; the
// trust-region loop restated here follows its published algorithm and the defaults the reference leaves untouched.
//
// Device-resident LM: the host only enqueues a fixed kernel sequence per iteration; every decision (step validity,
// accept/reject, radius update, convergence) is taken on the device in per-window LM state.
//
// Per window: n = 15K+7 camera-side columns laid out [pose_0..pose_{K-1} (6 each) | extrinsic 6 | td 1 | mix_0..mix_{K-1} (9 each)];
// the vision factors only touch the first NCV = 6K+7 ("vision columns").  Landmarks (inverse depths) are eliminated:
//   lin_vis    : thread / reprojection factor -> residual, local Jacobians, Huber correction -> 40-double record
//   lin_lm     : warp / landmark -> h_l, g_l and the dense coupling row w_l (A_W, landmark-major)
//   pair_gram  : factors grouped by (reference node, observing node): 20x20 Gram matrix per group on the FP64 tensor cores
//                (DMMA.8x8x4), then a one-writer-per-entry gather into the vision part of H_cc and g_c
//   schur_dmma : sum_l phi_l w_l w_l^T with phi_l = s_l^2 / (s_l^2 h_l + D_l^2) on the FP64 tensor cores
//   lin_cam    : one CTA / window (second stream, beside the vision chain) -> IMU preintegration, GNSS, bias, prior and
//                marginalization factors -> H_c, g_c
//   solve      : one CTA / window -> Jacobi scaling, LM diagonal, S = s(H - Schur)s + D^2, packed Cholesky in shared memory
//                (panel updates on DMMA), triangular solves, landmark back-substitution, model cost change, candidate x (+) delta
//   cost       : candidate cost (all factors, residuals only);   accept : Ceres step acceptance + radius update
//   ba_marg.cuh: sliding-window marginalization (MarginalizationInfo) on the same device-resident linearisation
#include <unistd.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <thread>
#include <vector>

#include "ba_cull.cuh"
#include "ba_math.cuh"
#include "common.cuh"
#include "geom_core.cuh"

namespace icg {
using namespace bam;

constexpr int BA_SPLIT_J = 1;   // the vision Gram matrix is produced whole by ba_pair_gram
constexpr int BA_SPLIT_W = 4;   // row splits of the Schur SYRK (partials summed in fixed order -> deterministic)
constexpr int BA_CHOL_NB = 8;   // Cholesky block width
constexpr int BA_MARG_MAXB = 72;  // remained blocks of a prior: <= 2 max_K + 2 = 66 at max_K = 32 (table stride)
constexpr int BA_MAX_NODES = 32;  // icg_ba_create: max_K <= 32

struct BaCaps {
    int NW, K, L, F, G, R;     // capacities
    int NCV, N, NS, NCA, RJ, LP, NVB;  // derived strides: NCV = 6K+7, N = 15K+7, NS = N padded, NCA = roundup4(NCV+1), RJ = 2F padded, LP = L padded
};

struct WinDims {  // per-window actual sizes
    int K, L, F, n_imu, n_gnss, marg_r, marg_nb;
    int ext_const, td_const, reproj_huber, gnss_huber, has_imu_error, has_pose_prior, has_mix_prior;
    double reproj_sinv;
};

struct LmState {
    double radius, decrease_factor, x_cost, x_norm, cand_cost, model_cost_change, step_norm, gmax, initial_cost, cost_cam;
    int iter, n_success, n_invalid, done, need_lin, last_success, first, step_valid, fresh_lin, max_iter, chol_ok;
};

// Exchange state of the split pipeline (ba_split.cuh): one buffer per rank holding the inbox of reduction operands, the step broadcast, the
// scalar exchange and the epoch flags; `peer[r]` is rank r's buffer as mapped into this process (peer memory, CUDA IPC or same process)
struct ShardDev {
    int split;                 // 1: the split pipeline drives this handle (large systems and / or landmark shards)
    int PK, BS, RV;            // packed partial length, step-broadcast stride, reduced-vector stride (doubles)
    double *peer[8];
    size_t off_inbox, off_bcast, off_scal, off_flagA, off_flagB, off_flagC;  // offsets in doubles, identical on every rank
    double *redv;              // [NW][RV] owner-side reduced vectors: diag H_vis | g_vis | W phi g_l | cost, sum rho^2, max |g_l|
    int *err;                  // device error word (flag wait timed out)
    double *slm;               // [NW][STEP_SLICES][8] partial sums of ba_step_lm's landmark slices
    int *slm_cnt;              // [NW] slices arrived (resets itself)
};

struct BaDev {  // device pointers (flat, capacity-strided by window)
    ShardDev S;
    WinDims *dims;
    LmState *st;
    double *pose, *mix, *ext, *rho;          // current parameters
    double *pose_c, *mix_c, *ext_c, *rho_c;  // candidate
    double *pose_0, *mix_0, *ext_0, *rho_0;  // initial copy (for re-running the same problem: bench)
    uint8_t *f_active_0;                     // pristine copies of what the two-pass protocol mutates (restart re-solves the UPLOADED problem)
    double *gnss_std_0;
    uint8_t *f_active;                       // by factor id
    int *lm_off;  // CSR offsets of the factor records by landmark
    int *vb_lm0;  // [NW][NVB] first landmark of every lin_vis run (runs hold whole landmarks, <= 128 factors); last entry = run count
    int *f_meta_s;       // per record slot: (landmark, reference node, observing node, factor id)
    double *f_const_s;   // per record slot: the factor's 14 constants (copy of f_const in slot order)
    int *pair_off, *pair_ro, *pair_fidx, *npairs;  // factors grouped by (reference node, observing node)
    double *Mp;                                    // per-pair 20x20 Gram matrices (upper, 210 entries)
    double *AW, *CJ, *CW;  // Schur SYRK input; vision Gram matrix; Schur partials
    double *jcomp, *costf;  // per-factor record (40 doubles, landmark-CSR order), cost
    double *hl, *gl, *scale_l, *scale_c;
    double *Hc, *gc;
    double *Hs;  // H_c + vision Gram - Schur term (lower triangle, ld NS): the operand ba_solve scales and factorises
    double *imu_blob, *imu_U;
    int *gnss_node;
    double *gnss_blh, *gnss_std, *lever;
    double *pose_prior, *pose_prior_sinfo, *mix_prior, *mix_prior_std;
    int *marg_type, *marg_node;
    double *marg_x0, *marg_H0, *marg_b0, *marg_c0;
    double *cost_part;  // [NW][ncost_blocks]
    double *red2;       // [NW][4]: model cost change, step norm^2, non-finite count, candidate cost
    int rank, world;    // landmark shard of this process (split pipeline; 0 / 1 otherwise)
    double *step_c, *step_l;
    double *Sglobal;    // fallback Cholesky workspace when the packed system does not fit shared memory
    unsigned long long *clk;  // ICG_BA_PROFILE: SM-clock totals of ba_solve's phases for window 0 (nullptr otherwise)
};

__device__ __forceinline__ int col_pose(int k) { return 6 * k; }
__device__ __forceinline__ int col_ext(int K) { return 6 * K; }
__device__ __forceinline__ int col_td(int K) { return 6 * K + 6; }
__device__ __forceinline__ int col_mix(int K, int k) { return 6 * K + 7 + 9 * k; }

// ------------------------------------------------------------------------------------------------ lin_vis (+ landmark rows)
__device__ __forceinline__ int jc_off(int a) { return a < 18 ? (a / 6) * 12 + (a % 6) : 36 + 2 * (a - 18); }  // row 0 offset in a record
__device__ __forceinline__ int jc_row1(int a) { return a < 18 ? 6 : 1; }                                           // + this for row 1
// One CTA linearises a run of WHOLE landmarks (<= 128 reprojection factors; the host packs the runs at upload).
//  phase 1: thread / factor, in record (landmark-CSR slot) order -> residual, local Jacobians, Huber correction -> 40-double record
//           [Ji 12 | Jj 12 | Je 12 | Jt 2 | r 2] + [j_rho 2 | observing node | reference node], staged in shared memory;
//  phase 2: the records leave as contiguous, fully used 128-byte lines (a thread-per-record store pattern costs 32 sectors per
//           instruction and made the store pipe the bottleneck) -- ba_pair_gram1 consumes them;
//  phase 3: eight lanes per landmark reduce its records, straight from shared memory, to h_l, g_l and the coupling row
//           w_l[c] = sum_f J_f[:, c]^T j_rho,f of A_W (landmark-major [l][NCA]: zeroed, then the <= 13 + 6 n_obs non-zeros).  All
//           factors of a landmark share the reference node, the extrinsic and td (accumulated); each observing node appears once
//           (written directly; icg_ba_upload checks it).
constexpr int LV_LD = 45;  // shared-memory record row: 44 doubles padded to an odd length (conflict-free)
constexpr size_t LV_SMEM = sizeof(double) * (128 * LV_LD + (BA_MAX_NODES + 1) * NODE_FRAME_LD);  // records + node frames (49.5 KB: dynamic, opted in at create)
__global__ void __launch_bounds__(128, 4) ba_lin_vis(BaCaps C, BaDev D) {
    extern __shared__ double lv_sm[];
    double (*s_rec)[LV_LD] = (double (*)[LV_LD]) lv_sm;
    double (*s_frame)[NODE_FRAME_LD] = (double (*)[NODE_FRAME_LD]) (lv_sm + 128 * LV_LD);
    const int w = blockIdx.y;
    const LmState &st = D.st[w];
    if (st.done || !st.need_lin) return;
    const int *vb = D.vb_lm0 + (size_t) w * C.NVB;
    if ((int) blockIdx.x >= vb[C.NVB - 1]) return;  // last entry = number of runs of this window
    const WinDims dm = D.dims[w];
    const int tid = threadIdx.x;
    const int *off = D.lm_off + (size_t) w * (C.L + 1);
    const int lmA = vb[blockIdx.x], lmB = vb[blockIdx.x + 1];
    const int s0 = off[lmA], nslot = off[lmB] - s0;
    // ---- phase 0: the window's K + 1 node frames (rotation matrix | position of every pose and of the extrinsic), once per CTA
    if (tid <= dm.K) node_frame(tid < dm.K ? D.pose + ((size_t) w * C.K + tid) * 7 : D.ext + (size_t) w * 8, s_frame[tid]);
    __syncthreads();
    // ---- phase 1
    if (tid < nslot) {
        const int q = s0 + tid;
        double r[2], Ji[12], Jj[12], Je[12], Jr[2], Jt[2], cost = 0;
        const int4 meta = ((const int4 *) D.f_meta_s)[(size_t) w * C.F + q];  // (landmark, reference node, observing node, factor id)
        const int i = meta.y, j = meta.z, f = meta.w;
        if (D.f_active[(size_t) w * C.F + f] != 0) {
            const double *ext = D.ext + (size_t) w * 8;
            reproj_eval_frames(s_frame[i], s_frame[j], s_frame[dm.K], D.rho[(size_t) w * C.L + meta.x], ext[7],
                               D.f_const_s + ((size_t) w * C.F + q) * 14, dm.reproj_sinv, true, r, Ji, Jj, Je, Jr, Jt);
            if (dm.ext_const)
                for (int k = 0; k < 12; k++) Je[k] = 0;
            if (dm.td_const) Jt[0] = Jt[1] = 0;
            double sq = r[0] * r[0] + r[1] * r[1], sc = 1.0;
            if (dm.reproj_huber)
                huber(sq, cost, sc);
            else
                cost = 0.5 * sq;
            if (sc != 1.0) {
                for (int k = 0; k < 12; k++) Ji[k] *= sc, Jj[k] *= sc, Je[k] *= sc;
                Jr[0] *= sc, Jr[1] *= sc, Jt[0] *= sc, Jt[1] *= sc, r[0] *= sc, r[1] *= sc;
            }
        } else {
            for (int k = 0; k < 12; k++) Ji[k] = Jj[k] = Je[k] = 0;
            Jr[0] = Jr[1] = Jt[0] = Jt[1] = r[0] = r[1] = 0;
        }
        D.costf[(size_t) w * C.F + f] = cost;
        double *sr = s_rec[tid];
#pragma unroll
        for (int k = 0; k < 12; k++) sr[k] = Ji[k], sr[12 + k] = Jj[k], sr[24 + k] = Je[k];
        sr[36] = Jt[0], sr[37] = Jt[1], sr[38] = r[0], sr[39] = r[1];
        sr[40] = Jr[0], sr[41] = Jr[1], sr[42] = (double) j, sr[43] = (double) i;
    }
    __syncthreads();
    // ---- phase 2
    {
        double *gj = D.jcomp + ((size_t) w * C.F + s0) * 40;
        for (int idx = tid; idx < nslot * 40; idx += 128) {
            const int rr = idx / 40, k = idx - 40 * rr;
            gj[idx] = s_rec[rr][k];
        }
    }
    // ---- phase 3
    const int K = dm.K, NCV = 6 * K + 7, NCA = 4 * ((NCV + 1 + 3) / 4);
    const int grp = tid >> 3, sl = tid & 7;
    int o0[3], o1[3];
#pragma unroll
    for (int t = 0; t < 3; t++) {
        const int c = sl + 8 * t;  // 0..23; 19 -> residual pair (g_l); 20 -> h_l from j_rho; > 20 unused
        o0[t] = c < 19 ? jc_off(c) : 38, o1[t] = c < 19 ? o0[t] + jc_row1(c) : 39;
    }
    for (int l = lmA + grp; l < lmB; l += 16) {
        const int f0 = off[l] - s0, nf = off[l + 1] - off[l];
        double *row = D.AW + ((size_t) w * C.LP + l) * C.NCA;
        for (int c = sl; c < NCA; c += 8) row[c] = 0.0;
        __syncwarp(0xffu << (tid & 24));  // the landmark's eight lanes: zeros land before the values
        double acc[3] = {0, 0, 0};
        for (int q = 0; q < nf; q++) {
            const double *rec = s_rec[f0 + q];
            const double r0 = rec[40], r1 = rec[41];
            const int ob = (int) rec[42];
#pragma unroll
            for (int t = 0; t < 3; t++) {
                const int c = sl + 8 * t;
                if (c == 20) {
                    acc[t] += r0 * r0 + r1 * r1;
                } else if (c < 20) {
                    const double v = rec[o0[t]] * r0 + rec[o1[t]] * r1;
                    if (c >= 6 && c < 12)
                        row[col_pose(ob) + c - 6] = v;
                    else
                        acc[t] += v;
                }
            }
        }
        const int ref = nf > 0 ? (int) s_rec[f0][43] : 0;
#pragma unroll
        for (int t = 0; t < 3; t++) {
            const int c = sl + 8 * t;
            if (nf > 0) {
                if (c < 6) row[col_pose(ref) + c] = acc[t];
                else if (c >= 12 && c < 18) row[col_ext(K) + c - 12] = acc[t];
                else if (c == 18) row[col_td(K)] = acc[t];
            }
            if (c == 19) {
                row[NCV] = acc[t];
                D.gl[(size_t) w * C.L + l] = acc[t];
            } else if (c == 20) {
                D.hl[(size_t) w * C.L + l] = acc[t];
                if (st.first) D.scale_l[(size_t) w * C.L + l] = 1.0 / (1.0 + sqrt(acc[t]));  // jacobi_scaling, once (iteration 0)
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------ pair_gram: vision part of H_cc, g_c
// Factors are grouped by (reference node, observing node).  Within a group every factor has the same 19 camera-side columns
// [ref pose 6 | obs pose 6 | extrinsic 6 | td 1] (+ the residual as a 20th column), so the group's contribution is the dense
// 20x20 Gram matrix of its stacked 2x20 rows: stage 1 (warp / group) computes it, stage 2 (thread / output entry) gathers the
// groups into the symmetric (NCV+1)^2 matrix [H_vis g_vis; g_vis^T r^T r].  No atomics: every output has one writer.
__device__ __forceinline__ int tri20(int la, int lb) {  // index of (la <= lb) in the packed upper 20x20
    return la * 20 - la * (la - 1) / 2 + (lb - la);
}
// stage 1: one warp per (window, group): the group's packed 20x20 Gram matrix -> Mp (global, L2 resident).
// FP64 tensor cores (DMMA.8x8x4): the stacked 2x20 rows X of the group are multiplied as X^T X, 4 rows (2 factors) per k-step.
// With the m8n8k4 fragment layout (A: lane -> (row lane/4, k lane%4); B: lane -> (k lane%4, col lane/4)) the A operand of
// X^T X and the B operand are the SAME register: lane loads X[k = lane%4][8 t + lane/4] for the three column tiles t and issues
// the six upper-triangular tile products.  Records are read straight from L2 (each 320-byte record is consumed whole by the warp).
__device__ __forceinline__ void dmma884(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
__device__ __forceinline__ void gram1_body(const BaCaps &C, const BaDev &D, int w, int pblock) {
    const LmState &st = D.st[w];
    if (st.done || !st.need_lin) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int PM = C.K * (C.K - 1);
    const int P = D.npairs[w];
    const int p = pblock * 8 + warp;
    if (p >= P) return;
    const int *poff = D.pair_off + (size_t) w * (PM + 1), *pfidx = D.pair_fidx + (size_t) w * C.F;
    double *Mp = D.Mp + (size_t) w * PM * 210;
    const int kk = lane & 3, g = lane >> 2;  // k index inside the step (factor kk/2, residual row kk%2), column inside the tile
    int o[3];
#pragma unroll
    for (int t = 0; t < 3; t++) {
        const int a = 8 * t + g;
        o[t] = a < 20 ? jc_off(a) + (kk & 1) * jc_row1(a) : -1;
    }
    double c00[2] = {0, 0}, c01[2] = {0, 0}, c02[2] = {0, 0}, c11[2] = {0, 0}, c12[2] = {0, 0}, c22[2] = {0, 0};
    const int pbeg = poff[p], pend = poff[p + 1];
    const double *rec = D.jcomp + (size_t) w * C.F * 40;
    constexpr int UNR = 4;  // k-steps in flight (8 factors)
    for (int base = pbeg; base < pend; base += 2 * UNR) {
        double x[UNR][3];
#pragma unroll
        for (int u = 0; u < UNR; u++) {
            const int q = base + 2 * u + (kk >> 1);
            const bool ok = q < pend;
            const int f = ok ? pfidx[q] : 0;
#pragma unroll
            for (int t = 0; t < 3; t++) x[u][t] = (ok && o[t] >= 0) ? rec[(size_t) f * 40 + o[t]] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < UNR; u++) {
            dmma884(c00[0], c00[1], x[u][0], x[u][0]);
            dmma884(c01[0], c01[1], x[u][0], x[u][1]);
            dmma884(c02[0], c02[1], x[u][0], x[u][2]);
            dmma884(c11[0], c11[1], x[u][1], x[u][1]);
            dmma884(c12[0], c12[1], x[u][1], x[u][2]);
            dmma884(c22[0], c22[1], x[u][2], x[u][2]);
        }
    }
    // C fragment: lane holds (row lane/4, cols 2 (lane%4) + {0,1}) of each 8x8 tile
    auto put = [&](int ti, int tj, const double *c) {
#pragma unroll
        for (int e = 0; e < 2; e++) {
            const int la = 8 * ti + g, lb = 8 * tj + 2 * kk + e;
            if (la <= lb && lb < 20) Mp[(size_t) p * 210 + tri20(la, lb)] = c[e];
        }
    };
    put(0, 0, c00), put(0, 1, c01), put(0, 2, c02), put(1, 1, c11), put(1, 2, c12), put(2, 2, c22);
}

__global__ void __launch_bounds__(256) ba_pair_gram1(BaCaps C, BaDev D) { gram1_body(C, D, blockIdx.y, blockIdx.x); }

// stage 2: one thread per output entry gathers the groups that touch both of its blocks (one writer per entry, no atomics)
// gather of one entry (A <= B) of the symmetric (NCV+1)^2 matrix [H_vis g_vis; g_vis^T r^T r] from the per-pair Gram matrices
__device__ __forceinline__ void gram2_slots(const BaCaps &C, const BaDev &D, int w, int K, short *s_slot) {
    const int PM = C.K * (C.K - 1), P = D.npairs[w];
    const int *pro = D.pair_ro + (size_t) w * PM;
    for (int e = threadIdx.x; e < K * K; e += blockDim.x) s_slot[e] = -1;
    __syncthreads();
    for (int p = threadIdx.x; p < P; p += blockDim.x) s_slot[(pro[p] >> 8) * K + (pro[p] & 255)] = (short) p;
    __syncthreads();
}
__device__ __forceinline__ double gram2_entry(const BaCaps &C, const BaDev &D, int w, int K, const short *s_slot, int A, int B) {
    const int PM = C.K * (C.K - 1), P = D.npairs[w];
    const double *Mp = D.Mp + (size_t) w * PM * 210;
    const int bA = A < 6 * K ? A / 6 : K, bB = B < 6 * K ? B / 6 : K;
    const int a = A - 6 * bA, b = B - 6 * bB;  // offsets inside the block (global block: 0..7 = ext 6, td, residual)
    const int ga = 12 + a, gb = 12 + b;          // local column of a global-block column
    double sum = 0;
    if (bA == K) {  // (global, global): every group
        // up to K (K - 1) groups: eight loads in flight and four partial sums in a fixed order (these 36 entries are the tail of the kernel:
        // a serial sum is 90 dependent L2 round trips)
        const int idx = tri20(ga, gb);
        double s4[4] = {0, 0, 0, 0};
        int p = 0;
        for (; p + 8 <= P; p += 8) {
            double v[8];
#pragma unroll
            for (int u = 0; u < 8; u++) v[u] = Mp[(size_t) (p + u) * 210 + idx];
#pragma unroll
            for (int u = 0; u < 8; u++) s4[u & 3] += v[u];
        }
        for (; p < P; p++) s4[p & 3] += Mp[(size_t) p * 210 + idx];
        sum = (s4[0] + s4[1]) + (s4[2] + s4[3]);
    } else if (bB == K || bB == bA) {  // (pose, global) or the pose's diagonal block
        const int i1 = tri20(a, bB == K ? gb : b), i2 = tri20(6 + a, bB == K ? gb : 6 + b);
        for (int o0 = 0; o0 < K; o0 += 4) {  // 8 loads in flight; same summation order as a serial loop
            double v1[4], v2[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int o = o0 + u;
                const int p1 = o < K ? s_slot[bA * K + o] : -1, p2 = o < K ? s_slot[o * K + bA] : -1;  // bA as reference node / as observing node
                v1[u] = p1 >= 0 ? Mp[(size_t) p1 * 210 + i1] : 0.0;
                v2[u] = p2 >= 0 ? Mp[(size_t) p2 * 210 + i2] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < 4; u++) sum += v1[u], sum += v2[u];
        }
    } else {  // two different poses: the (bA -> bB) and (bB -> bA) groups
        const int p1 = s_slot[bA * K + bB], p2 = s_slot[bB * K + bA];
        if (p1 >= 0) sum += Mp[(size_t) p1 * 210 + tri20(a, 6 + b)];
        if (p2 >= 0) sum += Mp[(size_t) p2 * 210 + tri20(b, 6 + a)];
    }
    return sum;
}

// ------------------------------------------------------------------------------------------------ Schur term
// Schur SYRK on the FP64 tensor cores: CW[split] = sum over the split's landmarks of phi_l w_l w_l^T (stored symmetric), with
// phi_l = s_l^2 / (s_l^2 h_l + clamp(s_l^2 h_l) / radius) the LM-damped landmark pivot.  DMMA.8x8x4 with k = 4 landmarks per step; as in
// ba_pair_gram1 the A and B fragments of X^T X share one layout: lane reads A_W[l0 + lane%4][8 t + lane/4].  The CTA stages its
// landmark rows (and phi) in shared memory once per pass -- leading dimension = 8 mod 16 doubles, so a fragment read is the minimal
// two wavefronts -- and every warp accumulates two 16x16 super-tiles (2x2 DMMA tiles each) of the upper triangle per pass.
// The BA_SPLIT_W landmark splits are separate CTAs whose partials ba_hsum / ba_export sum in fixed order (deterministic).
constexpr int SCHUR_RCH = 80;  // landmark rows staged per chunk (multiple of 4)
__device__ __forceinline__ void schur_body(const BaCaps &C, const BaDev &D, int w, int split, int ld, double *sA /* [SCHUR_RCH][ld] rows, then phi[SCHUR_RCH] */) {
    const LmState &st = D.st[w];
    if (st.done) return;
    const WinDims dm = D.dims[w];
    const int NCV = 6 * dm.K + 7, NCA = 4 * ((NCV + 1 + 3) / 4);
    const int T2 = (NCA + 15) / 16, nsuper = T2 * (T2 + 1) / 2;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, kk = lane & 3;
    double *sphi = sA + (size_t) SCHUR_RCH * ld;
    const double *A = D.AW + (size_t) w * C.LP * C.NCA;
    double *Cout = D.CW + ((size_t) w * BA_SPLIT_W + split) * C.NCA * C.NCA;
    const double radius = st.radius;
    const int nsteps = (dm.L + 3) / 4;
    const int r_beg = 4 * (int) ((long long) nsteps * split / BA_SPLIT_W), r_end = min(dm.L, 4 * (int) ((long long) nsteps * (split + 1) / BA_SPLIT_W));
    const int npass = (nsuper + 15) / 16;
    for (int pass = 0; pass < npass; pass++) {
        int si[2], sj[2];
        bool on[2];
#pragma unroll
        for (int h2 = 0; h2 < 2; h2++) {
            const int su = (2 * pass + h2) * 8 + warp;
            on[h2] = su < nsuper;
            int a = 0, e = on[h2] ? su : 0;
            while (e >= T2 - a) e -= T2 - a, a++;
            si[h2] = a, sj[h2] = a + e;
        }
        double acc[2][4][2];
#pragma unroll
        for (int h2 = 0; h2 < 2; h2++)
#pragma unroll
            for (int q = 0; q < 4; q++) acc[h2][q][0] = acc[h2][q][1] = 0;
        for (int r0 = r_beg; r0 < r_end; r0 += SCHUR_RCH) {
            const int nr = min(SCHUR_RCH, r_end - r0), nr4 = (nr + 3) & ~3;
            __syncthreads();
            for (int rb = warp; rb < nr4; rb += 8 * 4) {  // warp stages rows rb, rb + 8, rb + 16, rb + 24: 4 rows x 3 column chunks in flight
                double v[4][3];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int rr = rb + 8 * u;
#pragma unroll
                    for (int cchunk = 0; cchunk < 3; cchunk++) {
                        const int c = lane + 32 * cchunk;
                        v[u][cchunk] = (rr < nr && c < NCA) ? A[(size_t) (r0 + rr) * C.NCA + c] : 0.0;
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int rr = rb + 8 * u;
#pragma unroll
                    for (int cchunk = 0; cchunk < 3; cchunk++) {
                        const int c = lane + 32 * cchunk;
                        if (rr < nr4 && c < ld) sA[(size_t) rr * ld + c] = v[u][cchunk];
                    }
                }
                for (int c = lane + 96; c < ld; c += 32)  // wider rows (K > 12): remaining columns
                    for (int u = 0; u < 4; u++) {
                        const int rr = rb + 8 * u;
                        if (rr < nr4) sA[(size_t) rr * ld + c] = (rr < nr && c < NCA) ? A[(size_t) (r0 + rr) * C.NCA + c] : 0.0;
                    }
            }
            for (int rr = tid; rr < nr4; rr += 256) {
                double ph = 0;
                if (rr < nr) {
                    const int l = r0 + rr;
                    const double sl = D.scale_l[(size_t) w * C.L + l], hs = sl * sl * D.hl[(size_t) w * C.L + l];
                    ph = sl * sl / (hs + fmin(fmax(hs, 1e-6), 1e32) / radius);
                }
                sphi[rr] = ph;
            }
            __syncthreads();
            for (int ks = 0; ks < nr4 / 4; ks++) {
                const double *row = sA + (size_t) (4 * ks + kk) * ld;
                const double ph = sphi[4 * ks + kk];
#pragma unroll
                for (int h2 = 0; h2 < 2; h2++) {
                    if (!on[h2]) continue;
                    const double xb0 = row[16 * sj[h2] + g], xb1 = row[16 * sj[h2] + 8 + g];
                    const double a0 = row[16 * si[h2] + g] * ph, a1 = row[16 * si[h2] + 8 + g] * ph;
                    dmma884(acc[h2][0][0], acc[h2][0][1], a0, xb0);
                    dmma884(acc[h2][1][0], acc[h2][1][1], a0, xb1);
                    dmma884(acc[h2][2][0], acc[h2][2][1], a1, xb0);
                    dmma884(acc[h2][3][0], acc[h2][3][1], a1, xb1);
                }
            }
        }
#pragma unroll
        for (int h2 = 0; h2 < 2; h2++) {
            if (!on[h2]) continue;
#pragma unroll
            for (int q = 0; q < 4; q++) {  // C fragment: (row g, cols 2 kk + {0, 1}) of tile (2 si + q/2, 2 sj + q%2)
#pragma unroll
                for (int e = 0; e < 2; e++) {
                    const int r = 8 * (2 * si[h2] + (q >> 1)) + g, cc = 8 * (2 * sj[h2] + (q & 1)) + 2 * kk + e;
                    if (r <= cc && cc < NCA) {
                        Cout[(size_t) r * C.NCA + cc] = acc[h2][q][e];
                        Cout[(size_t) cc * C.NCA + r] = acc[h2][q][e];  // stored symmetric: ba_solve reads rows contiguously
                    }
                }
            }
        }
    }
}

__global__ void __launch_bounds__(256) ba_schur_dmma(BaCaps C, BaDev D, int ld) {
    extern __shared__ double sA[];
    schur_body(C, D, blockIdx.y, blockIdx.x, ld, sA);
}

// symmetric read of the summed SYRK partials (upper tiles hold the data)
__device__ __forceinline__ double syrk_get(const double *Cp, int nsplit, int NCAcap, int a, int b) {
    if (a > b) {
        int t = a;
        a = b, b = t;
    }
    // tiles with ti <= tj are stored; within a diagonal tile both triangles are present
    double s = 0;
    for (int k = 0; k < nsplit; k++) s += Cp[(size_t) k * NCAcap * NCAcap + (size_t) a * NCAcap + b];
    return s;
}

// ------------------------------------------------------------------------------------------------ camera-only factors
constexpr double IMU_GB_STD = 7200 / 3600.0 * 3.14159265358979323846 / 180.0;  // IG/preintegration/imu_error_factor.h:89-91
constexpr double IMU_AB_STD = 2.0e4 * 1.0e-5;

// one warp evaluates one IMU factor: whitened residual rw[15] and (optionally) whitened local Jacobian Jw[15x30] in shared memory
__device__ void imu_factor_warp(const double *blob, const double *U, const double *pose0, const double *mix0, const double *pose1,
                                const double *mix1, bool want_j, double *rw, double *Jw, int lane) {
    __shared__ ImuMid s_mid[16];
    double *raw_r = rw + 15;  // scratch behind rw (caller provides 30 doubles)
    const int wslot = (threadIdx.x >> 5) & 15;
    if (want_j)
        for (int e = lane; e < 450; e += 32) Jw[e] = 0;
    __syncwarp();
    if (lane == 0) {
        ImuMid M;
        imu_residual_raw(blob, pose0, mix0, pose1, mix1, raw_r, M);
        if (want_j) imu_jacobian_raw(blob, M, Jw);
        s_mid[wslot] = M;
    }
    __syncwarp();
    // whitening by the upper-triangular sqrt information: out[i] = sum_{k >= i} U[i][k] in[k]  (in place, rows ascending)
    if (want_j && lane < 30) {
        for (int i = 0; i < 15; i++) {
            double s = 0;
            for (int k = i; k < 15; k++) s += U[i * 15 + k] * Jw[k * 30 + lane];
            Jw[i * 30 + lane] = s;
        }
    }
    if (lane < 15) {
        double s = 0;
        for (int k = lane; k < 15; k++) s += U[lane * 15 + k] * raw_r[k];
        rw[lane] = s;
    }
    __syncwarp();
}

// marginalization prior (IG/factors/marginalization_factor.h:47-101): dx of every remained block
__device__ void marg_dx(const BaCaps &C, const BaDev &D, int w, const WinDims &dm, const double *pose, const double *mix, const double *ext, double *dx,
                        int *colmap, int tid, int nthreads) {
    const int *type = D.marg_type + (size_t) w * BA_MARG_MAXB, *node = D.marg_node + (size_t) w * BA_MARG_MAXB;
    const double *x0 = D.marg_x0 + (size_t) w * BA_MARG_MAXB * 9;
    if (tid == 0) {
        int col = 0, xo = 0;
        for (int b = 0; b < dm.marg_nb; b++) {
            int t = type[b], nd = node[b];
            if (t == 0 || t == 2) {
                const double *x = t == 0 ? pose + nd * 7 : ext;
                const double *xl = x0 + xo;
                Q dq = qmul(qinv(pose_q(xl)), pose_q(x));
                V3 a = 2.0 * qv(dq);
                if (dq.w < 0) a = -a;
                for (int k = 0; k < 3; k++) dx[col + k] = x[k] - xl[k];
                dx[col + 3] = a.x, dx[col + 4] = a.y, dx[col + 5] = a.z;
                int base = t == 0 ? col_pose(nd) : col_ext(dm.K);
                for (int k = 0; k < 6; k++) colmap[col + k] = (t == 2 && dm.ext_const) ? -1 : base + k;
                col += 6, xo += 7;
            } else if (t == 1) {
                for (int k = 0; k < 9; k++) dx[col + k] = mix[nd * 9 + k] - x0[xo + k], colmap[col + k] = col_mix(dm.K, nd) + k;
                col += 9, xo += 9;
            } else {
                dx[col] = ext[7] - x0[xo];
                colmap[col] = dm.td_const ? -1 : col_td(dm.K);
                col += 1, xo += 1;
            }
        }
    }
}

// cost of all camera-only factors at (pose, mix, ext); optionally the linearisation (H_c, g_c).  One CTA (256 threads).
// smem: per IMU factor 30 + 450 doubles; GNSS 3 + 18 each; misc.
// x += v on a global accumulator whose value the thread does not need back: one fire-and-forget reduction at the L2 (RED.ADD.F64) instead of a
// load -> add -> store chain (a dependent L2 round trip per entry: measured 50 k of ba_lin_cam's 123 k cycles in the IMU block accumulation).
// Every entry has ONE writer per phase and the phases are separated by block barriers, so the summation order is fixed (deterministic).
__device__ __forceinline__ void red_add(double *p, double v) { asm volatile("red.global.add.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory"); }

__device__ double cam_factors(const BaCaps &C, const BaDev &D, int w, const WinDims &dm, const double *pose, const double *mix, const double *ext,
                              bool lin, double *smem) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int K = dm.K, N = 15 * K + 7;
    double *Hc = D.Hc + (size_t) w * C.NS * C.NS, *gc = D.gc + (size_t) w * C.NS;
    double *s_imu = smem;                              // n_imu * 480
    double *s_gnss = s_imu + (size_t) C.K * 480;       // G * 24 : r[3] J[18] cost scale
    double *s_misc = s_gnss + (size_t) C.G * 24;       // pose prior r[6] J[36] | mix prior r[9] | marg dx[R] y[R] | costs
    double *s_pp = s_misc, *s_mp = s_misc + 48, *s_dx = s_mp + 16, *s_y = s_dx + C.R, *s_cost = s_y + C.R;
    int *s_colmap = (int *) (s_cost + 8);
    __shared__ double s_total;
#ifdef ICG_BA_PHASE_CLOCKS
    unsigned long long cclk = D.clk ? clock64() : 0ull;  // profiling build: phase clocks of the linearising call, window 0
#define CAM_CLK(k)                                                 \
    if (D.clk && lin && w == 0 && tid == 0) {                      \
        const unsigned long long t_ = clock64();                   \
        atomicAdd(&D.clk[16 + (k)], t_ - cclk), atomicAdd(&D.clk[24 + (k)], 1ull); \
        cclk = t_;                                                 \
    }
#else
#define CAM_CLK(k)
#endif
    // ---- phase 1: evaluate
    for (int k = warp; k < dm.n_imu; k += nwarps)
        imu_factor_warp(D.imu_blob + ((size_t) w * C.K + k) * ICG_IMU_BLOB_DOUBLES, D.imu_U + ((size_t) w * C.K + k) * 225, pose + k * 7, mix + k * 9,
                        pose + (k + 1) * 7, mix + (k + 1) * 9, lin, s_imu + (size_t) k * 480, s_imu + (size_t) k * 480 + 30, lane);
    if (tid < dm.n_gnss) {
        const int nd = D.gnss_node[(size_t) w * C.G + tid];
        double *o = s_gnss + tid * 24;
        gnss_eval(pose + nd * 7, D.gnss_blh + ((size_t) w * C.G + tid) * 3, D.gnss_std + ((size_t) w * C.G + tid) * 3, D.lever + (size_t) w * 3, lin, o, o + 3);
        double sq = o[0] * o[0] + o[1] * o[1] + o[2] * o[2], cost, sc = 1.0;
        if (dm.gnss_huber)
            huber(sq, cost, sc);
        else
            cost = 0.5 * sq;
        if (sc != 1.0) {
            for (int e = 0; e < 3; e++) o[e] *= sc;
            if (lin)
                for (int e = 0; e < 18; e++) o[3 + e] *= sc;
        }
        o[21] = cost;
    }
    if (tid == 64 && dm.has_pose_prior) pose_prior_eval(pose, D.pose_prior + (size_t) w * 7, D.pose_prior_sinfo + (size_t) w * 6, lin, s_pp, s_pp + 6);
    if (tid == 96 && dm.has_mix_prior)
        for (int k = 0; k < 9; k++) s_mp[k] = (mix[k] - D.mix_prior[(size_t) w * 9 + k]) / D.mix_prior_std[(size_t) w * 9 + k];
    if (dm.marg_r > 0) marg_dx(C, D, w, dm, pose, mix, ext, s_dx, s_colmap, tid, blockDim.x);
    __syncthreads();
    CAM_CLK(0)  // factor evaluation
    const double *H0 = D.marg_H0 + (size_t) w * C.R * C.R, *b0 = D.marg_b0 + (size_t) w * C.R;
    if (dm.marg_r > 0) {
        for (int i = tid; i < dm.marg_r; i += blockDim.x) {
            double s = 0;
            for (int k = 0; k < dm.marg_r; k++) s += H0[(size_t) i * dm.marg_r + k] * s_dx[k];
            s_y[i] = s;
        }
    }
    __syncthreads();
    // ---- cost (single thread, fixed order -> deterministic)
    if (tid == 0) {
        double c = 0;
        for (int k = 0; k < dm.n_imu; k++) {
            const double *r = s_imu + (size_t) k * 480;
            double sq = 0;
            for (int e = 0; e < 15; e++) sq += r[e] * r[e];
            c += 0.5 * sq;
        }
        for (int g = 0; g < dm.n_gnss; g++) c += s_gnss[g * 24 + 21];
        if (dm.has_imu_error) {
            const double *m = mix + dm.n_imu * 9;
            double sq = 0;
            for (int e = 0; e < 3; e++) sq += (m[3 + e] / IMU_GB_STD) * (m[3 + e] / IMU_GB_STD) + (m[6 + e] / IMU_AB_STD) * (m[6 + e] / IMU_AB_STD);
            c += 0.5 * sq;
        }
        if (dm.has_pose_prior) {
            double sq = 0;
            for (int e = 0; e < 6; e++) sq += s_pp[e] * s_pp[e];
            c += 0.5 * sq;
        }
        if (dm.has_mix_prior) {
            double sq = 0;
            for (int e = 0; e < 9; e++) sq += s_mp[e] * s_mp[e];
            c += 0.5 * sq;
        }
        if (dm.marg_r > 0) {
            // 0.5 |e0 + J0 dx|^2 = 0.5 (e0.e0 + 2 b0.dx + dx.H0.dx)
            double q = D.marg_c0[w];
            for (int i = 0; i < dm.marg_r; i++) q += (2.0 * b0[i] + s_y[i]) * s_dx[i];
            c += 0.5 * q;
        }
        s_total = c;
    }
    if (!lin) {
        __syncthreads();
        return s_total;
    }
    CAM_CLK(1)  // prior product + cost
    // ---- phase 2: H_c = sum J^T J, g_c = sum J^T r   (every entry has exactly one writer per round -> deterministic)
    for (int e = tid; e < N * C.NS; e += blockDim.x) Hc[e] = 0;
    for (int e = tid; e < N; e += blockDim.x) gc[e] = 0;
    __syncthreads();
    CAM_CLK(2)  // zero H_c
    if (dm.marg_r > 0) {
        const int r = dm.marg_r;
        for (int e = tid; e < r * r; e += blockDim.x) {
            int i = e / r, j = e - i * r;
            int ci = s_colmap[i], cj = s_colmap[j];
            if (ci >= 0 && cj >= 0) Hc[(size_t) ci * C.NS + cj] = H0[e];
        }
        for (int i = tid; i < r; i += blockDim.x)
            if (s_colmap[i] >= 0) gc[s_colmap[i]] = b0[i] + s_y[i];
    }
    __syncthreads();
    CAM_CLK(3)  // prior blocks
    for (int parity = 0; parity < 2; parity++) {  // IMU factors k and k+2 touch disjoint nodes
        const int nf = (dm.n_imu - parity + 1) / 2;
        for (int e = tid; e < nf * 930; e += blockDim.x) {
            const int k = parity + 2 * (e / 930), q = e % 930;
            const double *rw = s_imu + (size_t) k * 480, *Jw = rw + 30;
            auto gcol = [&](int c) { return c < 6 ? col_pose(k) + c : c < 15 ? col_mix(K, k) + c - 6 : c < 21 ? col_pose(k + 1) + c - 15 : col_mix(K, k + 1) + c - 21; };
            if (q < 900) {
                int a = q / 30, b = q - a * 30;
                double s = 0;
                for (int m = 0; m < 15; m++) s += Jw[m * 30 + a] * Jw[m * 30 + b];
                red_add(&Hc[(size_t) gcol(a) * C.NS + gcol(b)], s);
            } else {
                int a = q - 900;
                double s = 0;
                for (int m = 0; m < 15; m++) s += Jw[m * 30 + a] * rw[m];
                red_add(&gc[gcol(a)], s);
            }
        }
        __syncthreads();
    }
    CAM_CLK(4)  // IMU J^T J
    // pose-diagonal blocks: GNSS + pose prior; mix-diagonal: bias-magnitude factor + mix prior
    for (int e = tid; e < K * 42; e += blockDim.x) {
        const int k = e / 42, q = e % 42;
        double s = 0;
        if (q < 36) {
            const int a = q / 6, b = q % 6;
            for (int g = 0; g < dm.n_gnss; g++)
                if (D.gnss_node[(size_t) w * C.G + g] == k) {
                    const double *J = s_gnss + g * 24 + 3;
                    s += J[a] * J[b] + J[6 + a] * J[6 + b] + J[12 + a] * J[12 + b];
                }
            if (k == 0 && dm.has_pose_prior)
                for (int m = 0; m < 6; m++) s += s_pp[6 + m * 6 + a] * s_pp[6 + m * 6 + b];
            red_add(&Hc[(size_t) (col_pose(k) + a) * C.NS + col_pose(k) + b], s);
        } else {
            const int a = q - 36;
            for (int g = 0; g < dm.n_gnss; g++)
                if (D.gnss_node[(size_t) w * C.G + g] == k) {
                    const double *o = s_gnss + g * 24;
                    s += o[3 + a] * o[0] + o[9 + a] * o[1] + o[15 + a] * o[2];
                }
            if (k == 0 && dm.has_pose_prior)
                for (int m = 0; m < 6; m++) s += s_pp[6 + m * 6 + a] * s_pp[m];
            red_add(&gc[col_pose(k) + a], s);
        }
    }
    if (tid < 9) {
        if (dm.has_imu_error && tid >= 3) {
            const int k = dm.n_imu;
            const double sd = tid < 6 ? IMU_GB_STD : IMU_AB_STD;
            Hc[(size_t) (col_mix(K, k) + tid) * C.NS + col_mix(K, k) + tid] += 1.0 / (sd * sd);
            gc[col_mix(K, k) + tid] += mix[k * 9 + tid] / (sd * sd);
        }
    }
    __syncthreads();
    if (tid < 9 && dm.has_mix_prior) {
        const double sd = D.mix_prior_std[(size_t) w * 9 + tid];
        Hc[(size_t) (col_mix(K, 0) + tid) * C.NS + col_mix(K, 0) + tid] += 1.0 / (sd * sd);
        gc[col_mix(K, 0) + tid] += s_mp[tid] / sd;
    }
    __syncthreads();
    CAM_CLK(5)  // GNSS / prior diagonal blocks
#undef CAM_CLK
    return s_total;
}

constexpr int CAM_THREADS = 320;  // 10 warps: the K - 1 = 9 IMU factors of a 10-node window are evaluated in one round (warp per factor)
__global__ void __launch_bounds__(CAM_THREADS) ba_lin_cam(BaCaps C, BaDev D) {
    extern __shared__ double smem[];
    const int w = blockIdx.x;
    LmState &st = D.st[w];
    if (st.done || !st.need_lin) return;
    if (D.S.split && (w % D.world) != D.rank) return;  // split pipeline: the window's owner handles the camera-only factors
    const WinDims dm = D.dims[w];
    double c = cam_factors(C, D, w, dm, D.pose + (size_t) w * C.K * 7, D.mix + (size_t) w * C.K * 9, D.ext + (size_t) w * 8, true, smem);
    if (threadIdx.x == 0) st.cost_cam = c;
}

// ------------------------------------------------------------------------------------------------ reduced camera matrix
// Hs = H_c + H_vis - Schur term, lower triangle, one thread per entry (wide and coalesced; ba_solve then reads ONE operand per entry
// instead of gathering 2 + BA_SPLIT_W).  The gather of the per-pair Gram matrices happens here too, one kernel less on the path.
__global__ void __launch_bounds__(256) ba_hsum(BaCaps C, BaDev D) {
    __shared__ short s_slot[32 * 32];
    const int w = blockIdx.y;
    if (D.st[w].done) return;
    const int K = D.dims[w].K, NCV = 6 * K + 7, nn = NCV + 1;
    const int NN = C.NCA * C.NCA;
    if ((int) blockIdx.x * 256 >= nn * nn) return;
    gram2_slots(C, D, w, K, s_slot);
    const int t = blockIdx.x * 256 + threadIdx.x;
    if (t >= nn * nn) return;
    const int A = t / nn, B = t - A * nn;  // A <= B: entry (row B, column A) of the lower triangle
    if (B < A) return;
    const double cj = gram2_entry(C, D, w, K, s_slot, A, B);
    double *Cout = D.CJ + (size_t) w * NN;
    Cout[(size_t) A * C.NCA + B] = cj;
    Cout[(size_t) B * C.NCA + A] = cj;
    const double *CWp = D.CW + (size_t) w * BA_SPLIT_W * NN;
    double cw = 0;
#pragma unroll
    for (int k = 0; k < BA_SPLIT_W; k++) cw += CWp[(size_t) k * NN + (size_t) B * C.NCA + A];
    if (B < NCV) D.Hs[(size_t) w * C.NS * C.NS + (size_t) B * C.NS + A] = D.Hc[(size_t) w * C.NS * C.NS + (size_t) B * C.NS + A] + (cj - cw);
}

// ------------------------------------------------------------------------------------------------ solve (one CTA per window)
constexpr int SOLVE_THREADS = 256;  // 2 CTAs (windows) per SM: 107 KB shared memory and <= 128 registers each

__device__ __forceinline__ double block_sum(double v, double *s_red) {
    // deterministic block reduction (fixed tree)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    __syncthreads();
    if (lane == 0) s_red[warp] = v;
    __syncthreads();
    double t = 0;
    if (tid == 0) {
        for (int k = 0; k < (int) (blockDim.x >> 5); k++) t += s_red[k];
        s_red[32] = t;
    }
    __syncthreads();
    return s_red[32];
}
__device__ __forceinline__ double block_max(double v, double *s_red) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_down_sync(0xffffffffu, v, o));
    __syncthreads();
    if (lane == 0) s_red[warp] = v;
    __syncthreads();
    if (tid == 0) {
        double t = 0;
        for (int k = 0; k < (int) (blockDim.x >> 5); k++) t = fmax(t, s_red[k]);
        s_red[32] = t;
    }
    __syncthreads();
    return s_red[32];
}

__global__ void __launch_bounds__(SOLVE_THREADS, 2) ba_solve(BaCaps C, BaDev D) {
    extern __shared__ double sm[];
    const int w = blockIdx.x, tid = threadIdx.x;
    LmState &st = D.st[w];
    if (st.done) return;
    // phase clocks (profiling BUILD only, -DICG_BA_PHASE_CLOCKS: the instrumentation perturbs register allocation): thread 0 of window 0 adds
    // the SM cycles since the previous mark
#ifdef ICG_BA_PHASE_CLOCKS
    unsigned long long clk_prev = D.clk ? clock64() : 0ull;
#define SOLVE_CLK(k)                                              \
    if (D.clk && w == 0 && tid == 0) {                            \
        const unsigned long long t_ = clock64();                  \
        atomicAdd(&D.clk[k], t_ - clk_prev), atomicAdd(&D.clk[8 + (k)], 1ull); \
        clk_prev = t_;                                            \
    }
#define SOLVE_CLK_NOW() (D.clk ? clock64() : 0ull)
#define SOLVE_CLK_ADD(k, t0)                                      \
    if (D.clk && w == 0 && tid == 0) atomicAdd(&D.clk[k], clock64() - (t0)), atomicAdd(&D.clk[8 + (k)], 1ull);
#else
#define SOLVE_CLK(k)
#define SOLVE_CLK_NOW() 0ull
#define SOLVE_CLK_ADD(k, t0)
#endif
    const WinDims dm = D.dims[w];
    const int K = dm.K, L = dm.L, NCV = 6 * K + 7, N = 15 * K + 7;
    const int f_first = st.first, f_fresh = st.fresh_lin, f_last = st.last_success, f_iter = st.iter;
    const double f_gmax_old = st.gmax;
    (void) f_gmax_old;
    // shared layout: vectors first, packed matrix last
    double *s_red = sm;                 // 40
    double *s_scale = s_red + 40;       // N
    double *s_g = s_scale + C.NS;       // N   full camera gradient (unscaled)
    double *s_rhs = s_g + C.NS;         // N   -> step' (scaled space)
    double *s_d2 = s_rhs + C.NS;        // N
    double *s_diag = s_d2 + C.NS;       // N   Cholesky diagonal
    // packed lower triangle, N + 1 rows, ALWAYS in shared memory (systems that do not fit are driven by the split pipeline, ba_solve_cam): a
    // pointer that could also be global made every access a generic LD / ST (longer latency, long-scoreboard tracked)
    double *S = s_diag + C.NS;
    const double *Hc = D.Hc + (size_t) w * C.NS * C.NS, *gcam = D.gc + (size_t) w * C.NS, *Hs = D.Hs + (size_t) w * C.NS * C.NS;
    // Reduction operands: the producers' outputs, read directly (vision Gram matrix; the BA_SPLIT_W Schur partials summed in fixed order).
    const int NN = C.NCA * C.NCA;
    const double *CJ = D.CJ + (size_t) w * BA_SPLIT_J * NN;
    const double *CWp = D.CW + (size_t) w * BA_SPLIT_W * NN;
    auto cw_get = [&](int a, int b) {  // symmetric storage: any (a, b)
        double s2 = 0;
#pragma unroll
        for (int k = 0; k < BA_SPLIT_W; k++) s2 += CWp[(size_t) k * NN + (size_t) a * C.NCA + b];
        return s2;
    };
    if (tid == 0 && st.need_lin) st.need_lin = 0;      // the linearisation kernels of this iteration have run (stream order)
    double *scale_c = D.scale_c + (size_t) w * C.NS;
    const double *hl = D.hl + (size_t) w * C.L, *gl = D.gl + (size_t) w * C.L, *scale_l = D.scale_l + (size_t) w * C.L;

    // ---- after a fresh linearisation: total cost, gradient, (first time) Jacobi scaling
    for (int a = tid; a < N; a += SOLVE_THREADS) {
        double g = gcam[a];
        if (a < NCV) g += syrk_get(CJ, 1, C.NCA, a, NCV);
        s_g[a] = g;
        if (f_first) {
            double h = Hc[(size_t) a * C.NS + a] + (a < NCV ? syrk_get(CJ, 1, C.NCA, a, a) : 0.0);
            scale_c[a] = 1.0 / (1.0 + sqrt(h));
        }
    }
    __syncthreads();
    for (int a = tid; a < N; a += SOLVE_THREADS) s_scale[a] = scale_c[a];
    double gmax_now = st.gmax;
    if (f_fresh) {
        double cs = 0, gq = 0;
        for (int f = tid; f < dm.F; f += SOLVE_THREADS) cs += D.costf[(size_t) w * C.F + f];
        for (int l = tid; l < L; l += SOLVE_THREADS) gq = fmax(gq, fabs(gl[l]));
        const double c = block_sum(cs, s_red);
        const double gml = block_max(gq, s_red);
        double gm = 0;
        for (int a = tid; a < N; a += SOLVE_THREADS) gm = fmax(gm, fabs(s_g[a]));
        gm = fmax(block_max(gm, s_red), gml);
        gmax_now = gm;
        if (tid == 0) {
            st.x_cost = c + st.cost_cam;
            st.gmax = gm;
            if (f_first) st.initial_cost = st.x_cost;
            st.fresh_lin = 0;
        }
        __syncthreads();
    }
    if (f_first) {
        __syncthreads();
        if (tid == 0) st.first = 0;
    }
    // ---- TrustRegionMinimizer::FinalizeIterationAndCheckIfMinimizerCanContinue
    {
        int term = 0;
        if (f_iter >= st.max_iter) term = 1;                                    // NO_CONVERGENCE
        else if (f_last && gmax_now <= 1e-10) term = 2;                         // gradient tolerance
        else if (f_last && st.radius <= 1e-32) term = 2;                        // min trust region radius
        if (term) {
            __syncthreads();
            if (tid == 0) st.done = term, st.step_valid = 0;
            return;
        }
    }
    __syncthreads();
    if (tid == 0) st.iter++;
    const double radius = st.radius;
    SOLVE_CLK(0)  // gradient, cost, termination tests

    // ---- assemble S' = s (H - Schur) s + D^2 (packed lower), rhs' = -s (g - W phi g_l)
    // The reduced camera matrix (ba_hsum's output, row i contiguous) goes global -> packed shared rows with 8-byte cp.async: every element of
    // the lower triangle is in flight at once (one L2 round trip for the whole matrix instead of one per row and warp), the vector part below
    // overlaps the copy, and the Jacobi scaling + LM diagonal are applied in place afterwards.
    constexpr bool async_fill = true;
    if (async_fill) {
        for (int i = tid >> 5; i < N; i += SOLVE_THREADS / 32) {
            const double *src = (i < NCV ? Hs : Hc) + (size_t) i * C.NS;
            const unsigned dst = (unsigned) __cvta_generic_to_shared(S + i * (i + 1) / 2);
            for (int j = tid & 31; j <= i; j += 32)
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + 8u * j), "l"(src + j) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
    for (int a = tid; a < N; a += SOLVE_THREADS) {
        double h = Hc[(size_t) a * C.NS + a] + (a < NCV ? syrk_get(CJ, 1, C.NCA, a, a) : 0.0);
        double hs = s_scale[a] * s_scale[a] * h;
        s_d2[a] = fmin(fmax(hs, 1e-6), 1e32) / radius;
        double gw = a < NCV ? cw_get(a, NCV) : 0.0;
        s_rhs[a] = -s_scale[a] * (s_g[a] - gw);
    }
    if (async_fill) asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();
    if (async_fill) {
        for (int i = tid >> 5; i < N; i += SOLVE_THREADS / 32) {
            double *row = S + i * (i + 1) / 2;
            const double si = s_scale[i];
            for (int j = tid & 31; j <= i; j += 32) {
                double v = si * s_scale[j] * row[j];
                if (i == j) v += s_d2[i];
                row[j] = v;
            }
        }
    } else {
        for (int i = tid >> 5; i < N; i += SOLVE_THREADS / 32) {
            // one warp per row; all global loads of the row are issued before the first store (memory-level parallelism)
            constexpr int MAXQ = 16;  // N <= 512
            double hv[MAXQ];
            const int nq = i / 32 + 1;
#pragma unroll
            for (int q = 0; q < MAXQ; q++) {
                const int j = (tid & 31) + 32 * q;
                hv[q] = 0;
                if (q < nq && j <= i) hv[q] = (i < NCV ? Hs : Hc)[(size_t) i * C.NS + j];  // ba_hsum: H_c + vision Gram - Schur (vision rows); row i contiguous
            }
#pragma unroll
            for (int q = 0; q < MAXQ; q++) {
                const int j = (tid & 31) + 32 * q;
                if (q < nq && j <= i) {
                    double v = s_scale[i] * s_scale[j] * hv[q];
                    if (i == j) v += s_d2[i];
                    S[i * (i + 1) / 2 + j] = v;
                }
            }
        }
    }
    // augmented row N = rhs': the factorisation then leaves y = L^-1 rhs' in it (forward substitution for free)
    for (int a = tid; a < N; a += SOLVE_THREADS) S[N * (N + 1) / 2 + a] = s_rhs[a];
    __syncthreads();
    SOLVE_CLK(1)  // assembly
    // ---- blocked left-looking Cholesky on the packed lower triangle (two barriers per 8 columns); failure -> invalid step.
    // Per panel J (columns J0 .. J0 + 7):
    //   (1) panel update with all previous columns on the FP64 tensor cores, S[J0:, J0:J0+8] -= L[J0:, :J0] L[J0:J0+8, :J0]^T, one warp per
    //       8-row tile (A fragment = L[i0 + g][k0 + kk], B fragment = L[J0 + g][k0 + kk], DMMA.8x8x4, J0 % 8 == 0).  WARP 0 takes the
    //       diagonal tile alone and FACTORS it straight away (in registers: the 8-column pivot chain, ~8 x (DFMA + rsqrt + DMUL) = 600 cycles of
    //       pure latency) while warps 1..7 are still updating the tiles below -- the chain hides behind their tensor-core work.  (The
    //       previous version let every thread factor the block redundantly to save a barrier: measured, a barrier costs ~30 cycles here,
    //       the redundant factorisation ~3 000 issue slots per panel -- 58 % of the kernel.)
    //   (2) barrier; every row below the block (and the augmented rhs row) is solved against the factored block by its own thread; barrier.
    // 1/sqrt(d) comes from rsqrt (one dependent op per column instead of sqrt + divide); the row solve multiplies by it.
    __shared__ int s_fail;
    if (tid == 0) s_fail = 0;
    __syncthreads();
    const int NR = N + 1;
    for (int J0 = 0; J0 < N; J0 += BA_CHOL_NB) {
        const int nb = min(BA_CHOL_NB, N - J0);
        const int lane = tid & 31, warp = tid >> 5, g = lane >> 2, kk = lane & 3;
        const int ntile = (NR - J0 + 7) / 8;
        const unsigned long long pc0 = SOLVE_CLK_NOW();  // profiling: warp 0's own work / the row-solve phase of this panel
        (void) pc0;
        const int cb = J0 + g;                                     // row of L that is the B operand's column
        const double *rb = S + (cb < NR ? cb * (cb + 1) / 2 : 0);
        const bool okb = cb < NR;
        if (warp == 0) {
            if (J0 > 0) {  // diagonal tile: rows J0 + g; four accumulator chains over the k range
                const double *ra = rb;
                double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
                int k0 = 0;
                for (; k0 + 16 <= J0; k0 += 16) {
                    const double x0 = okb ? ra[k0 + kk] : 0.0, x1 = okb ? ra[k0 + 4 + kk] : 0.0, x2 = okb ? ra[k0 + 8 + kk] : 0.0, x3 = okb ? ra[k0 + 12 + kk] : 0.0;
                    dmma884(acc[0], acc[1], x0, x0);
                    dmma884(acc[2], acc[3], x1, x1);
                    dmma884(acc[4], acc[5], x2, x2);
                    dmma884(acc[6], acc[7], x3, x3);
                }
                for (; k0 + 8 <= J0; k0 += 8) {
                    const double x0 = okb ? ra[k0 + kk] : 0.0, x1 = okb ? ra[k0 + 4 + kk] : 0.0;
                    dmma884(acc[0], acc[1], x0, x0);
                    dmma884(acc[2], acc[3], x1, x1);
                }
                const double c0 = (acc[0] + acc[2]) + (acc[4] + acc[6]), c1 = (acc[1] + acc[3]) + (acc[5] + acc[7]);
                const int i = J0 + g;
                if (i < NR) {
                    const int ca = J0 + 2 * kk;
                    if (ca < J0 + nb && ca <= i) S[i * (i + 1) / 2 + ca] -= c0;
                    if (ca + 1 < J0 + nb && ca + 1 <= i) S[i * (i + 1) / 2 + ca + 1] -= c1;
                }
                __syncwarp();
            }
            // factor the nb x nb diagonal block: every lane of warp 0 runs the same register code on broadcast loads (no divergence, no
            // shuffles on the chain); lane a writes row a of L_JJ and its pivot reciprocal back
            double Ld[BA_CHOL_NB][BA_CHOL_NB], dinv[BA_CHOL_NB];
            bool bad = false;
#pragma unroll
            for (int a = 0; a < BA_CHOL_NB; a++)
#pragma unroll
                for (int b = 0; b < BA_CHOL_NB; b++) Ld[a][b] = (a < nb && b <= a) ? S[(J0 + a) * (J0 + a + 1) / 2 + J0 + b] : (a == b ? 1.0 : 0.0);
#pragma unroll
            for (int j = 0; j < BA_CHOL_NB; j++) {
                double d = Ld[j][j];
#pragma unroll
                for (int k = 0; k < j; k++) d -= Ld[j][k] * Ld[j][k];
                if (!(d > 0.0) || !isfinite(d)) bad = true;
                const double di = rsqrt(d);
                dinv[j] = di;
                Ld[j][j] = d * di;
#pragma unroll
                for (int a = j + 1; a < BA_CHOL_NB; a++) {
                    double sum = Ld[a][j];
#pragma unroll
                    for (int k = 0; k < j; k++) sum -= Ld[a][k] * Ld[j][k];
                    Ld[a][j] = sum * di;
                }
            }
            __syncwarp();  // every lane has read the unfactored block
            if (bad && lane == 0) s_fail = 1;
#pragma unroll
            for (int a2 = 0; a2 < BA_CHOL_NB; a2++) {
                // every lane holds the whole factor: entry (a2, b) is stored by ONE lane under a predicate -- statically indexed registers and no
                // divergent code.  ("lane a writes row a" was compiled into a switch on the lane, eight serial paths: 1 640 cycles per panel in
                // ba_solve_cam_dsm's phase clocks against 480 for this form, profiles/r2_ba_solve_cam_dsm.md.)
                double *ri = S + (J0 + a2) * (J0 + a2 + 1) / 2 + J0;
#pragma unroll
                for (int b = 0; b <= a2; b++)
                    if (lane == ((a2 * 8 + b) & 31) && a2 < nb) ri[b] = Ld[a2][b];
                if (lane == 8 + a2 && a2 < nb) s_diag[J0 + a2] = dinv[a2];
            }
            SOLVE_CLK_ADD(6, pc0)
        } else if (J0 > 0 && warp != 4) {
            // tiles 1 .. ntile-1 over warps 1, 2, 3, 5, 6, 7, up to four row tiles per warp in flight (they share the B fragment): N = 157 gives
            // <= 19 such tiles, so the whole panel update is ONE round of the k loop, and eight independent DMMA chains hide the tensor-pipe
            // latency.  Warp 4 sits out: it shares warp 0's scheduler and FP64 pipe (warp id mod 4), and every DMMA holds that pipe for 16
            // cycles -- measured, warp 0's 130-operation pivot chain took 3 600 cycles per panel queuing behind warp 4's tiles.
            constexpr int TPW = 4, NWARP = 6;
            const int wslot = warp < 4 ? warp - 1 : warp - 2;  // 0..5
            for (int t0 = 1 + wslot; t0 < ntile; t0 += TPW * NWARP) {
                const double *ra[TPW];
                bool oka[TPW];
                double acc[TPW][4];
#pragma unroll
                for (int u = 0; u < TPW; u++) {
                    const int ia = J0 + 8 * (t0 + u * NWARP) + g;
                    oka[u] = (t0 + u * NWARP) < ntile && ia < NR;
                    ra[u] = S + (oka[u] ? ia * (ia + 1) / 2 : 0);
                    acc[u][0] = acc[u][1] = acc[u][2] = acc[u][3] = 0;
                }
                for (int k0 = 0; k0 + 8 <= J0; k0 += 8) {
                    const double b0 = okb ? rb[k0 + kk] : 0.0, b1 = okb ? rb[k0 + 4 + kk] : 0.0;
                    double a0[TPW], a1[TPW];
#pragma unroll
                    for (int u = 0; u < TPW; u++) a0[u] = oka[u] ? ra[u][k0 + kk] : 0.0, a1[u] = oka[u] ? ra[u][k0 + 4 + kk] : 0.0;
#pragma unroll
                    for (int u = 0; u < TPW; u++) {
                        dmma884(acc[u][0], acc[u][1], a0[u], b0);
                        dmma884(acc[u][2], acc[u][3], a1[u], b1);
                    }
                }
#pragma unroll
                for (int u = 0; u < TPW; u++) {
                    const double c0 = acc[u][0] + acc[u][2], c1 = acc[u][1] + acc[u][3];
                    const int i = J0 + 8 * (t0 + u * NWARP) + g;
                    if (oka[u]) {
                        const int ca = J0 + 2 * kk;
                        if (ca < J0 + nb && ca <= i) S[i * (i + 1) / 2 + ca] -= c0;
                        if (ca + 1 < J0 + nb && ca + 1 <= i) S[i * (i + 1) / 2 + ca + 1] -= c1;
                    }
                }
            }
        }
        __syncthreads();
        const unsigned long long pc1 = SOLVE_CLK_NOW();
        (void) pc1;
        if (s_fail) break;
        // rows below the block (incl. the augmented rhs row): solve against the factored block, one row per thread.  L_JJ and the pivot
        // reciprocals are read from shared memory as the chain needs them (every thread reads the same address: broadcast, off the
        // dependent chain) instead of being staged in 36 + 8 registers
        for (int i = J0 + nb + tid; i < NR; i += SOLVE_THREADS) {
            double *ri = S + i * (i + 1) / 2 + J0;
            double x[BA_CHOL_NB];
#pragma unroll
            for (int c = 0; c < BA_CHOL_NB; c++) x[c] = c < nb ? ri[c] : 0.0;
#pragma unroll
            for (int c = 0; c < BA_CHOL_NB; c++) {
                if (c < nb) {
                    const double *lc = S + (J0 + c) * (J0 + c + 1) / 2 + J0;
                    double sum = x[c];
#pragma unroll
                    for (int k = 0; k < c; k++) sum -= x[k] * lc[k];
                    x[c] = sum * s_diag[J0 + c];
                }
            }
#pragma unroll
            for (int c = 0; c < BA_CHOL_NB; c++)
                if (c < nb) ri[c] = x[c];
        }
        __syncthreads();
        SOLVE_CLK_ADD(7, pc1)
    }
    __syncthreads();
    bool valid = !s_fail;
    SOLVE_CLK(2)  // Cholesky
    // ---- backward substitution L^T x = y, blocked by the factorisation's 8-column panels, last panel first:
    //   (a) warp 0 solves the panel's 8 x 8 triangle L_JJ^T x_J = y_J in registers (every lane the same code on broadcast loads; the
    //       dependent chain is 8 x (DFMA + DMUL));
    //   (b) barrier; every thread i < J0 applies the panel to its own entry, y_i -= sum_c L[J0 + c][i] x_{J0 + c} -- row J0 + c of the
    //       packed triangle is contiguous in i, so the reads are coalesced; barrier.
    // Same operations in the same order as a column-by-column substitution (c descending), on 256 threads instead of one warp:
    // measured 185 cycles per COLUMN for the single-warp form (29 k cycles at N = 157), about 400 cycles per PANEL for this one.
    if (valid) {
        double *y = S + N * (N + 1) / 2;
        const int lane = tid & 31;
        for (int J0 = ((N - 1) / BA_CHOL_NB) * BA_CHOL_NB; J0 >= 0; J0 -= BA_CHOL_NB) {
            const int nb = min(BA_CHOL_NB, N - J0);
            if (tid < 32) {
                double x[BA_CHOL_NB];
#pragma unroll
                for (int c = BA_CHOL_NB - 1; c >= 0; c--) {
                    x[c] = 0.0;
                    if (c < nb) {
                        double sum = y[J0 + c];
#pragma unroll
                        for (int k = BA_CHOL_NB - 1; k > c; k--)
                            if (k < nb) sum -= S[(J0 + k) * (J0 + k + 1) / 2 + J0 + c] * x[k];
                        x[c] = sum * s_diag[J0 + c];
                    }
                }
#pragma unroll
                for (int c = 0; c < BA_CHOL_NB; c++)
                    if (c == lane && c < nb) s_rhs[J0 + c] = x[c];
            }
            __syncthreads();
            for (int i = tid; i < J0; i += SOLVE_THREADS) {
                double acc = y[i];
#pragma unroll
                for (int c = BA_CHOL_NB - 1; c >= 0; c--)
                    if (c < nb) acc -= S[(J0 + c) * (J0 + c + 1) / 2 + i] * s_rhs[J0 + c];
                y[i] = acc;
            }
            __syncthreads();
        }
    }
    __syncthreads();
    SOLVE_CLK(3)  // camera back-substitution
    // ---- landmark back-substitution + model cost change  (-1/2 step'.g' + 1/2 step'.D^2 step', exact identity of
    //      Ceres' -(J' step)^T (r + J' step / 2) for the damped normal-equation solution)
    double *step_l = D.step_l + (size_t) w * C.L;
    const double *AW = D.AW + (size_t) w * C.LP * C.NCA;  // landmark-major
    double part = 0;
    bool finite = true;
    double *R2 = D.red2 + (size_t) w * 4;
    if (!valid) {
        // Cholesky breakdown: the step is invalid; ba_accept applies HandleInvalidStep
        if (tid == 0) {
            st.chol_ok = 0, st.step_valid = 0;
            R2[0] = 0, R2[1] = 0, R2[2] = 1, R2[3] = 0;
        }
        return;
    }
    for (int a = tid; a < N; a += SOLVE_THREADS) {
        double sp = s_rhs[a];
        finite = finite && isfinite(sp);
        part += -0.5 * sp * (s_scale[a] * s_g[a]) + 0.5 * s_d2[a] * sp * sp;
    }
    // landmark back-substitution: one warp per landmark, the coupling row is read coalesced (two landmarks in flight per warp)
    double *s_sx = s_diag;  // s_diag is dead after the back-substitution: scaled camera step s_c * step'_c
    __syncthreads();
    for (int a = tid; a < NCV; a += SOLVE_THREADS) s_sx[a] = s_scale[a] * s_rhs[a];
    __syncthreads();
    {
        const int lane = tid & 31, warp = tid >> 5;
        constexpr int LB = 8;  // landmarks in flight per warp (the coupling rows come from L2: 24 loads per lane outstanding)
        // after the transposing reduction below, lane holds the dot product of landmark l0 + lu; its per-landmark scalars are loaded at the top
        // of the round, together with the coupling rows (one L2 round trip per round instead of two)
        const int lu = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
        for (int l0 = LB * warp; l0 < L; l0 += LB * (SOLVE_THREADS / 32)) {
            const int l = l0 + lu;
            const bool lok = l < L;
            const double sl = lok ? scale_l[l] : 0.0, hh = lok ? hl[l] : 0.0, gg = lok ? gl[l] : 0.0;
            double d[LB];
#pragma unroll
            for (int u = 0; u < LB; u++) d[u] = 0;
            for (int c = lane; c < NCV; c += 32) {
                const double sx = s_sx[c];
#pragma unroll
                for (int u = 0; u < LB; u++) d[u] += (l0 + u < L ? AW[(size_t) (l0 + u) * C.NCA + c] : 0.0) * sx;
            }
            const double hs = sl * sl * hh, d2 = fmin(fmax(hs, 1e-6), 1e32) / radius, den = hs + d2, sg = sl * gg;
            // transposing butterfly: 8 values x 32 lanes -> 1 value per lane in 4 + 2 + 1 + 1 + 1 exchanges (a plain butterfly needs 8 x 5)
            double e4[4], e2[2];
            {
                const bool hi = lane & 16;
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const double keep = hi ? d[u + 4] : d[u], send = hi ? d[u] : d[u + 4];
                    e4[u] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
                }
            }
            {
                const bool hi = lane & 8;
#pragma unroll
                for (int u = 0; u < 2; u++) {
                    const double keep = hi ? e4[u + 2] : e4[u], send = hi ? e4[u] : e4[u + 2];
                    e2[u] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
                }
            }
            double mine;
            {
                const bool hi = lane & 4;
                const double keep = hi ? e2[1] : e2[0], send = hi ? e2[0] : e2[1];
                mine = keep + __shfl_xor_sync(0xffffffffu, send, 4);
            }
            mine += __shfl_xor_sync(0xffffffffu, mine, 2);
            mine += __shfl_xor_sync(0xffffffffu, mine, 1);
            if ((lane & 3) == 0 && lok) {
                double sp = (-sg - sl * mine) / den;
                finite = finite && isfinite(sp);
                step_l[l] = sp;
                part += -0.5 * sp * sg + 0.5 * d2 * sp * sp;
            }
        }
    }
    __syncthreads();
    SOLVE_CLK(4)  // landmark back-substitution
    const double mcc = block_sum(part, s_red);
    const double nfin = block_sum(finite ? 0.0 : 1.0, s_red);
    // ---- candidate point x (+) delta, delta = step' * scale; |x - x_cand|^2 over active blocks
    const double *pose = D.pose + (size_t) w * C.K * 7, *mix = D.mix + (size_t) w * C.K * 9, *ext = D.ext + (size_t) w * 8, *rho = D.rho + (size_t) w * C.L;
    double *pose_c = D.pose_c + (size_t) w * C.K * 7, *mix_c = D.mix_c + (size_t) w * C.K * 9, *ext_c = D.ext_c + (size_t) w * 8, *rho_c = D.rho_c + (size_t) w * C.L;
    double sn = 0;
    for (int k = tid; k <= K; k += SOLVE_THREADS) {  // K poses + the extrinsic
        const bool is_ext = (k == K);
        const double *x = is_ext ? ext : pose + k * 7;
        double *xc = is_ext ? ext_c : pose_c + k * 7;
        if (is_ext && dm.ext_const) {
            for (int e = 0; e < 7; e++) xc[e] = x[e];
        } else {
            const int c0 = is_ext ? col_ext(K) : col_pose(k);
            double d[6];
            for (int e = 0; e < 6; e++) d[e] = s_rhs[c0 + e] * s_scale[c0 + e];
            pose_plus(x, d, xc);
            for (int e = 0; e < 7; e++) sn += (x[e] - xc[e]) * (x[e] - xc[e]);
        }
    }
    for (int e = tid; e < K * 9; e += SOLVE_THREADS) {
        int k = e / 9, q = e - 9 * k, c = col_mix(K, k) + q;
        double v = mix[e] + s_rhs[c] * s_scale[c];
        mix_c[e] = v;
        sn += (mix[e] - v) * (mix[e] - v);
    }
    if (tid == 0) {
        if (dm.td_const) {
            ext_c[7] = ext[7];
        } else {
            double v = ext[7] + s_rhs[col_td(K)] * s_scale[col_td(K)];
            ext_c[7] = v;
            sn += (ext[7] - v) * (ext[7] - v);
        }
    }
    for (int l = tid; l < L; l += SOLVE_THREADS) {
        double v = rho[l] + step_l[l] * scale_l[l];
        rho_c[l] = v;
        sn += (rho[l] - v) * (rho[l] - v);
    }
    sn = block_sum(sn, s_red);
    if (tid == 0) {
        st.chol_ok = 1, st.step_valid = 1;  // provisional: ba_accept validates with the reduced model cost change
        R2[0] = mcc, R2[1] = sn, R2[2] = nfin, R2[3] = 0;
    }
    SOLVE_CLK(5)  // candidate point, reductions
#undef SOLVE_CLK
#undef SOLVE_CLK_NOW
#undef SOLVE_CLK_ADD
}

// ------------------------------------------------------------------------------------------------ candidate cost
// camera-only factors at the candidate point (one CTA per window; runs beside the vision blocks on the handle's second stream)
__global__ void __launch_bounds__(CAM_THREADS) ba_cost_cam(BaCaps C, BaDev D, int nblk_vis) {
    extern __shared__ double smem[];
    const int w = blockIdx.x;
    const LmState &st = D.st[w];
    if (st.done || !st.step_valid) return;
    if (D.S.split && (w % D.world) != D.rank) return;
    const WinDims dm = D.dims[w];
    double c = cam_factors(C, D, w, dm, D.pose_c + (size_t) w * C.K * 7, D.mix_c + (size_t) w * C.K * 9, D.ext_c + (size_t) w * 8, false, smem);
    if (threadIdx.x == 0) D.cost_part[(size_t) w * (nblk_vis + 1) + nblk_vis] = c;
}
__global__ void __launch_bounds__(256) ba_cost(BaCaps C, BaDev D, int nblk_vis) {
    __shared__ double s_red[40];
    const int w = blockIdx.y;
    const LmState &st = D.st[w];
    if (st.done || !st.step_valid) return;
    const WinDims dm = D.dims[w];
    const double *pose = D.pose_c + (size_t) w * C.K * 7, *ext = D.ext_c + (size_t) w * 8, *rho = D.rho_c + (size_t) w * C.L;
    double *part = D.cost_part + (size_t) w * (nblk_vis + 1);
    const int q = blockIdx.x * 256 + threadIdx.x;  // record slot (landmark-CSR order): the slot-ordered copies are the only factor data on the device
    __shared__ double s_frame[BA_MAX_NODES + 1][NODE_FRAME_LD];  // node frames of the candidate point (see ba_lin_vis)
    if ((int) threadIdx.x <= dm.K) node_frame((int) threadIdx.x < dm.K ? pose + threadIdx.x * 7 : ext, s_frame[threadIdx.x]);
    __syncthreads();
    double cost = 0;
    int4 meta = make_int4(0, 0, 0, 0);
    if (q < dm.F) meta = ((const int4 *) D.f_meta_s)[(size_t) w * C.F + q];  // (landmark, reference node, observing node, factor id)
    if (q < dm.F && D.f_active[(size_t) w * C.F + meta.w]) {
        double r[2];
        reproj_eval_frames(s_frame[meta.y], s_frame[meta.z], s_frame[dm.K], rho[meta.x], ext[7], D.f_const_s + ((size_t) w * C.F + q) * 14, dm.reproj_sinv,
                           false, r, nullptr, nullptr, nullptr, nullptr, nullptr);
        double sq = r[0] * r[0] + r[1] * r[1], sc;
        if (dm.reproj_huber)
            huber(sq, cost, sc);
        else
            cost = 0.5 * sq;
    }
    cost = block_sum(cost, s_red);
    if (threadIdx.x == 0) part[blockIdx.x] = cost;
}

// ------------------------------------------------------------------------------------------------ accept / reject
__global__ void __launch_bounds__(128) ba_accept(BaCaps C, BaDev D, int nblk_vis) {
    __shared__ int s_accept;
    __shared__ double s_camsq, s_rhosq;
    __shared__ double s_red[40];
    const int w = blockIdx.x, tid = threadIdx.x;
    LmState &st = D.st[w];
    if (st.done) return;
    const WinDims dm = D.dims[w];
    const int chol_ok = st.chol_ok;
    const double *R2 = D.red2 + (size_t) w * 4;
    // |x|^2 of the camera-side blocks and of the inverse depths
    {
        const double *pose = D.pose + (size_t) w * C.K * 7, *mix = D.mix + (size_t) w * C.K * 9, *ext = D.ext + (size_t) w * 8;
        double s = 0;
        for (int e = tid; e < dm.K * 7; e += 128) s += pose[e] * pose[e];
        for (int e = tid; e < dm.K * 9; e += 128) s += mix[e] * mix[e];
        if (tid < 7 && !dm.ext_const) s += ext[tid] * ext[tid];
        if (tid == 7 && !dm.td_const) s += ext[7] * ext[7];
        s = block_sum(s, s_red);
        double q = 0;
        for (int l = tid; l < dm.L; l += 128) q += D.rho[(size_t) w * C.L + l] * D.rho[(size_t) w * C.L + l];
        q = block_sum(q, s_red);
        if (tid == 0) s_camsq = s, s_rhosq = q;
    }
    __syncthreads();
    if (tid == 0) {
        s_accept = 0;
        const double mcc = R2[0], sn = R2[1], nfin = R2[2];
        double cand = R2[3];
        if (st.step_valid) {  // sum the candidate-cost partials (vision blocks, then the camera-only factors)
            const double *part = D.cost_part + (size_t) w * (nblk_vis + 1);
            cand = 0;
            const int nb = (dm.F + 255) / 256;
            for (int b = 0; b < nb; b++) cand += part[b];
            cand += part[nblk_vis];
        }
        if (!chol_ok || nfin != 0.0 || !(mcc > 0.0)) {
            // HandleInvalidStep + LevenbergMarquardtStrategy::StepIsInvalid
            st.step_valid = 0;
            st.n_invalid++;
            if (st.n_invalid >= 5) st.done = 3;  // FAILURE
            st.radius *= 0.5;
            st.last_success = 0;
        } else {
            st.n_invalid = 0;
            st.model_cost_change = mcc;
            st.step_norm = sqrt(sn);
            st.x_norm = sqrt(s_camsq + s_rhosq);
            st.cand_cost = cand;
            // ParameterToleranceReached / FunctionToleranceReached (Ceres trust_region_minimizer.cc)
            if (st.step_norm <= 1e-8 * (st.x_norm + 1e-8)) {
                st.done = 2;
            } else if (fabs(st.x_cost - cand) <= 1e-6 * st.x_cost) {
                st.done = 2;
            } else {
                const double rel = (st.x_cost - cand) / mcc;
                if (rel > 1e-3) {
                    s_accept = 1;
                    st.n_success++;
                    // LevenbergMarquardtStrategy::StepAccepted
                    double t = 2.0 * rel - 1.0;
                    st.radius = fmin(1e16, st.radius / fmax(1.0 / 3.0, 1.0 - t * t * t));
                    st.decrease_factor = 2.0;
                    st.last_success = 1;
                    st.need_lin = 1;
                    st.fresh_lin = 1;
                } else {
                    // StepRejected
                    st.radius = st.radius / st.decrease_factor;
                    st.decrease_factor *= 2.0;
                    st.last_success = 0;
                    st.need_lin = 0;
                }
            }
        }
    }
    __syncthreads();
    if (!s_accept) return;
    double *pose = D.pose + (size_t) w * C.K * 7, *mix = D.mix + (size_t) w * C.K * 9, *ext = D.ext + (size_t) w * 8, *rho = D.rho + (size_t) w * C.L;
    const double *pose_c = D.pose_c + (size_t) w * C.K * 7, *mix_c = D.mix_c + (size_t) w * C.K * 9, *ext_c = D.ext_c + (size_t) w * 8, *rho_c = D.rho_c + (size_t) w * C.L;
    for (int e = tid; e < dm.K * 7; e += 128) pose[e] = pose_c[e];
    for (int e = tid; e < dm.K * 9; e += 128) mix[e] = mix_c[e];
    if (tid < 8) ext[tid] = ext_c[tid];
    for (int e = tid; e < dm.L; e += 128) rho[e] = rho_c[e];
}

// ------------------------------------------------------------------------------------------------ LM state reset (device side)
__global__ void ba_reset_state(BaDev D, LmState *save, int n, int max_iter) {
    int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n) return;
    if (save) save[w] = D.st[w];
    LmState st;
    memset(&st, 0, sizeof(st));
    st.radius = 1e4, st.decrease_factor = 2.0;  // Ceres initial_trust_region_radius
    st.need_lin = 1, st.fresh_lin = 1, st.first = 1, st.last_success = 1, st.max_iter = max_iter;
    D.st[w] = st;
}

// The outlier pass between the two solves of GVINS::gvinsOptimization (IG/ic_gvins.cc:1196-1207):
//   gnssOutlierCullingByChi2 (:1241-1267): chi2 = 2 cost > 7.815 -> std *= sqrt(chi2 / 7.815)
//   removeReprojectionFactorsByChi2 (:1269-1297): chi2 = 2 cost > 5.991 -> RemoveResidualBlock
//   GNSS factors re-added without loss function (:1202-1207)
__global__ void __launch_bounds__(128) ba_chi2_cull(BaCaps C, BaDev D, int *counters) {
    const int w = blockIdx.y;
    WinDims &dm = D.dims[w];
    const int t = blockIdx.x * 128 + threadIdx.x;
    const double *pose = D.pose + (size_t) w * C.K * 7, *ext = D.ext + (size_t) w * 8, *rho = D.rho + (size_t) w * C.L;
    int4 meta = make_int4(0, 0, 0, 0);
    if (t < dm.F) meta = ((const int4 *) D.f_meta_s)[(size_t) w * C.F + t];  // record slot t
    if (t < dm.F && D.f_active[(size_t) w * C.F + meta.w]) {
        double r[2];
        reproj_eval(pose + meta.y * 7, pose + meta.z * 7, ext, rho[meta.x], ext[7], D.f_const_s + ((size_t) w * C.F + t) * 14, dm.reproj_sinv, false, r, nullptr,
                    nullptr, nullptr, nullptr, nullptr);
        if ((r[0] * r[0] + r[1] * r[1]) > 5.991) {
            D.f_active[(size_t) w * C.F + meta.w] = 0;
            atomicAdd(&counters[2 * w], 1);
        }
    }
    if (t < dm.n_gnss) {
        double r[3];
        double *sd = D.gnss_std + ((size_t) w * C.G + t) * 3;
        gnss_eval(pose + D.gnss_node[(size_t) w * C.G + t] * 7, D.gnss_blh + ((size_t) w * C.G + t) * 3, sd, D.lever + (size_t) w * 3, false, r, nullptr);
        double chi2 = r[0] * r[0] + r[1] * r[1] + r[2] * r[2];
        if (chi2 > 7.815) {
            double sc = sqrt(chi2 / 7.815);
            sd[0] *= sc, sd[1] *= sc, sd[2] *= sc;
            atomicAdd(&counters[2 * w + 1], 1);
        }
    }
}
__global__ void ba_set_gnss_huber(BaDev D, int n, int v) {
    int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w < n) D.dims[w].gnss_huber = v;
}

// ------------------------------------------------------------------------------------------------ utility kernels
__global__ void ba_residual_costs_kernel(BaCaps C, BaDev D, double *reproj_cost, double *gnss_cost) {
    const int w = 0;
    const WinDims dm = D.dims[w];
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const double *pose = D.pose, *ext = D.ext, *rho = D.rho;
    if (t < dm.F) {
        double r[2];
        const int4 meta = ((const int4 *) D.f_meta_s)[t];  // record slot t -> (landmark, reference node, observing node, factor id)
        reproj_eval(pose + meta.y * 7, pose + meta.z * 7, ext, rho[meta.x], ext[7], D.f_const_s + (size_t) t * 14, dm.reproj_sinv, false, r, nullptr, nullptr,
                    nullptr, nullptr, nullptr);
        reproj_cost[meta.w] = 0.5 * (r[0] * r[0] + r[1] * r[1]);  // EvaluateResidualBlock(id, false, &cost, ...) (IG/ic_gvins.cc:1278)
    }
    if (t < dm.n_gnss) {
        double r[3];
        gnss_eval(pose + D.gnss_node[t] * 7, D.gnss_blh + t * 3, D.gnss_std + t * 3, D.lever, false, r, nullptr);
        gnss_cost[t] = 0.5 * (r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
    }
}

__global__ void ba_reproj_eval_kernel(const double *in /* 7+7+8+1+1+14+1 */, double *out /* 2 + 14+14+14+2+2 */) {
    double r[2], Ji[12], Jj[12], Je[12], Jr[2], Jt[2];
    reproj_eval(in, in + 7, in + 14, in[22], in[23], in + 24, 1.0 / in[38], true, r, Ji, Jj, Je, Jr, Jt);
    out[0] = r[0], out[1] = r[1];
    double *o = out + 2;
    const double *src[3] = {Ji, Jj, Je};
    for (int b = 0; b < 3; b++)
        for (int rr = 0; rr < 2; rr++) {
            for (int c = 0; c < 6; c++) o[b * 14 + rr * 7 + c] = src[b][rr * 6 + c];
            o[b * 14 + rr * 7 + 6] = 0.0;  // the quaternion-w column of the global Jacobian is zero (reprojection_factor.h:103,114,131)
        }
    o[42] = Jr[0], o[43] = Jr[1], o[44] = Jt[0], o[45] = Jt[1];
}

__global__ void ba_imu_eval_kernel(const double *blob, const double *U, const double *x /* 7 9 7 9 */, double *out /* 15 + 450 */) {
    __shared__ double s_buf[480];
    imu_factor_warp(blob, U, x, x + 7, x + 16, x + 23, true, s_buf, s_buf + 30, threadIdx.x);
    for (int e = threadIdx.x; e < 15; e += 32) out[e] = s_buf[e];
    for (int e = threadIdx.x; e < 450; e += 32) out[15 + e] = s_buf[30 + e];
}

// GnssFactor / ImuPosePriorFactor / ImuMixPriorFactor / ImuErrorFactor (kind 0..3), one thread; in / out layouts in the callers below
__global__ void ba_small_factor_eval_kernel(int kind, const double *in, double *out) {
    if (kind == 0) {         // in: pose7 blh3 std3 lever3 -> r[3], J local 3x6
        gnss_eval(in, in + 7, in + 10, in + 13, true, out, out + 3);
    } else if (kind == 1) {  // in: pose7 prior7 sinfo6 -> r[6], J local 6x6
        pose_prior_eval(in, in + 7, in + 14, true, out, out + 6);
    } else if (kind == 2) {  // in: mix9 prior9 std9 -> r[9], diag J[9]   (ImuMixPriorFactor, imu_mix_prior_factor.h:40-75)
        for (int k = 0; k < 9; k++) out[k] = (in[k] - in[9 + k]) / in[18 + k], out[9 + k] = 1.0 / in[18 + k];
    } else {                 // in: mix9 -> r[6], diag J[6]                (ImuErrorFactor, imu_error_factor.h:45-91)
        for (int k = 0; k < 3; k++) {
            out[k] = in[3 + k] / IMU_GB_STD, out[3 + k] = in[6 + k] / IMU_AB_STD;
            out[6 + k] = 1.0 / IMU_GB_STD, out[9 + k] = 1.0 / IMU_AB_STD;
        }
    }
}

// MarginalizationFactor::Evaluate (IG/factors/marginalization_factor.h:47-101): e = e0 + J0 dx with dx the local difference of every
// remained block to its linearisation point (quaternion blocks: 2 vec(q0^-1 q), sign-fixed).  One CTA; thread per residual row.
// in: [r, nb, types[nb], x (global sizes, concatenated), x0 (same), e0[r], J0[r*r]] as doubles; out: residuals[r]
__global__ void ba_marg_factor_eval_kernel(const double *in, double *out) {
    extern __shared__ double s_dx[];
    const int r = (int) in[0], nb = (int) in[1];
    const double *types = in + 2;
    int tot = 0;
    for (int b = 0; b < nb; b++) tot += ((int) types[b] == 1) ? 9 : ((int) types[b] == 3) ? 1 : 7;
    const double *x = types + nb, *x0 = x + tot, *e0 = x0 + tot, *J0 = e0 + r;
    if (threadIdx.x == 0) {
        int col = 0, xo = 0;
        for (int b = 0; b < nb; b++) {
            const int t = (int) types[b];
            if (t == 0 || t == 2) {
                Q dq = qmul(qinv(pose_q(x0 + xo)), pose_q(x + xo));
                V3 a = 2.0 * qv(dq);
                if (dq.w < 0) a = -a;
                for (int k = 0; k < 3; k++) s_dx[col + k] = x[xo + k] - x0[xo + k];
                s_dx[col + 3] = a.x, s_dx[col + 4] = a.y, s_dx[col + 5] = a.z;
                col += 6, xo += 7;
            } else {
                const int g = t == 1 ? 9 : 1;
                for (int k = 0; k < g; k++) s_dx[col + k] = x[xo + k] - x0[xo + k];
                col += g, xo += g;
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < r; i += blockDim.x) {
        double sum = e0[i];
        for (int k = 0; k < r; k++) sum += J0[(size_t) i * r + k] * s_dx[k];
        out[i] = sum;
    }
}

}  // namespace icg

#include "ba_split.cuh"
#include "ba_marg.cuh"

// ======================================================================================================= host side
using namespace icg;

namespace {
// ---- host helpers: IMU sqrt information  U = LLT(cov^-1).matrixL().transpose()  (IG/preintegration/preintegration_earth.cc:39-40)
bool host_invert(const double *A, double *Ai, int n) {
    std::vector<double> a(A, A + n * n);
    for (int i = 0; i < n * n; i++) Ai[i] = 0;
    for (int i = 0; i < n; i++) Ai[i * n + i] = 1;
    for (int c = 0; c < n; c++) {
        int p = c;
        for (int r = c + 1; r < n; r++)
            if (fabs(a[r * n + c]) > fabs(a[p * n + c])) p = r;
        if (a[p * n + c] == 0) return false;
        if (p != c)
            for (int k = 0; k < n; k++) std::swap(a[c * n + k], a[p * n + k]), std::swap(Ai[c * n + k], Ai[p * n + k]);
        double d = a[c * n + c];
        for (int k = 0; k < n; k++) a[c * n + k] /= d, Ai[c * n + k] /= d;
        for (int r = 0; r < n; r++) {
            if (r == c) continue;
            double f = a[r * n + c];
            if (f == 0) continue;
            for (int k = 0; k < n; k++) a[r * n + k] -= f * a[c * n + k], Ai[r * n + k] -= f * Ai[c * n + k];
        }
    }
    return true;
}
bool host_imu_sqrt_info(const double *cov, double *U) {
    double inv[225], Lm[225];
    if (!host_invert(cov, inv, 15)) return false;
    for (int i = 0; i < 15; i++)
        for (int j = 0; j < 15; j++) Lm[i * 15 + j] = 0.5 * (inv[i * 15 + j] + inv[j * 15 + i]);
    for (int j = 0; j < 15; j++) {
        double d = Lm[j * 15 + j];
        for (int k = 0; k < j; k++) d -= Lm[j * 15 + k] * Lm[j * 15 + k];
        if (!(d > 0)) return false;
        d = sqrt(d);
        Lm[j * 15 + j] = d;
        for (int i = j + 1; i < 15; i++) {
            double s = Lm[i * 15 + j];
            for (int k = 0; k < j; k++) s -= Lm[i * 15 + k] * Lm[j * 15 + k];
            Lm[i * 15 + j] = s / d;
        }
    }
    for (int i = 0; i < 15; i++)
        for (int j = 0; j < 15; j++) U[i * 15 + j] = j >= i ? Lm[j * 15 + i] : 0.0;
    return true;
}

template <typename T>
struct HostDev {  // pinned host staging + device array
    T *h = nullptr, *d = nullptr;
    size_t n = 0;
    int alloc(size_t count) {
        n = count;
        if (cudaMallocHost(&h, sizeof(T) * count) != cudaSuccess) return ICG_ENOMEM;
        if (cudaMalloc(&d, sizeof(T) * count) != cudaSuccess) return ICG_ENOMEM;
        memset(h, 0, sizeof(T) * count);
        return ICG_OK;
    }
    void release() {
        if (h) cudaFreeHost(h);
        if (d) cudaFree(d);
        h = d = nullptr;
    }
    cudaError_t up(cudaStream_t s, size_t count = 0) { return cudaMemcpyAsync(d, h, sizeof(T) * (count ? count : n), cudaMemcpyHostToDevice, s); }
    cudaError_t down(cudaStream_t s, size_t count = 0) { return cudaMemcpyAsync(h, d, sizeof(T) * (count ? count : n), cudaMemcpyDeviceToHost, s); }
};
}  // namespace

struct icg_ba {
    BaCaps C;
    BaDev D;
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t stream_cam = nullptr;  // the camera-only factors are linearised concurrently with the vision chain
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    bool own_stream = false;
    int nblk_vis = 0;
    int cur_windows = 0;
    int cam_threads = 160;  // CTA size of the camera-only factor kernels (<= CAM_THREADS): 160 x 168 registers leave room for two
                            // ba_lin_vis CTAs on the SM (320 threads take 82 % of the register file: nothing else fits beside them)
    size_t smem_cam, smem_solve, smem_schur;
    int ld_schur;
    int use_global_S;
    HostDev<WinDims> dims;
    HostDev<LmState> st;
    HostDev<double> pose, mix, ext, rho, imu_blob, imu_U, gnss_blh, gnss_std, lever, pose_prior, pose_prior_sinfo, mix_prior, mix_prior_std, marg_x0,
        marg_H0, marg_b0, marg_c0;
    HostDev<int> f_slot, f_meta_s, vb_lm0;  // f_slot / lm_fidx: host-side packing helpers only (factor id <-> record slot)
    HostDev<double> f_const_s;
    HostDev<int> lm_off, lm_fidx, gnss_node, marg_type, marg_node, pair_off, pair_ro, pair_fidx, npairs;
    HostDev<uint8_t> f_active;
    std::vector<void *> dev_only;
    HostDev<double> scratch;  // single-factor evaluation
    HostDev<LmState> st_save;   // pass-1 LM state of the two-pass protocol
    HostDev<int> cull_counters; // per window: reprojection factors removed, GNSS fixes re-weighted
    // split pipeline (ba_split.cuh): exchange buffer of this rank, peers' buffers opened through CUDA IPC, epoch counter of the flags
    double *xbuf = nullptr;
    size_t xbuf_doubles = 0;
    void *ipc_opened[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    unsigned long long epoch = 0;
    size_t smem_solve_cam = 0, smem_step_lm = 0;
    bool solve_cam_stage_a = false;  // per-warp shared-memory strips for the DMMA A operand (ba_solve_cam)
    bool solve_cam_dsm = false;      // the packed system fits the cluster's shared memory: ba_solve_cam_dsm (max_K <= 22)
    size_t smem_solve_cam_dsm = 0;
    // in-situ stage timing (ICG_BA_PROFILE=1): events between the kernels of the LM sequence on the main stream, read back in
    // icg_ba_sync / icg_ba_download and printed by icg_ba_destroy (warm caches, real launch gaps -- unlike an ncu replay)
    bool prof = false;
    std::vector<cudaEvent_t> prof_ev;
    std::vector<int> prof_tag;
    size_t prof_used = 0;
    int prof_skip = 1;  // LM sequences to discard first (lazy module loading puts a one-off multi-ms cost on every kernel's first launch)
    double prof_ms[16] = {0};
    long prof_cnt[16] = {0};
    // marginalization workspace (allocated on the first icg_ba_marginalize call)
    bool marg_ready = false;
    MargDev M;
    HostDev<int> marg_map;
    HostDev<double> marg_oJ0, marg_oe0, marg_oHp, marg_obp;
    // outlier-culling staging buffer (ba_cull.cuh layout; allocated on the first icg_ba_outlier_culling_resident call)
    HostDev<unsigned char> cull_buf;
};

extern "C" {
static void prof_collect(icg_ba *h);
static void prof_print(icg_ba *h);
}

static int dmalloc(icg_ba *h, double **p, size_t n) {
    if (cudaMalloc(p, sizeof(double) * n) != cudaSuccess) {
        set_error("icg_ba_create: cudaMalloc of %zu doubles failed", n);
        return ICG_ENOMEM;
    }
    cudaMemsetAsync(*p, 0, sizeof(double) * n, h->stream);
    h->dev_only.push_back(*p);
    return ICG_OK;
}

extern "C" {
static int split_setup(icg_ba *h, int rank, int world);
static void split_release(icg_ba *h);

int icg_imu_preintegrate(const double *state16, const double *iewn3, const double *gravity3, const double *noise5, const double *imu, int n, double *blob,
                         double *end_state10) {
    // PreintegrationEarth: resetState (:305-324), setNoiseMatrix (:326-334), integrationProcess (:205-260),
    // updateJacobianAndCovariance (:266-303) of IG/preintegration/preintegration_earth.cc.  Host code (sequential recurrence).
    // iewn3 == NULL selects PreintegrationNormal (`iswithearth: false`, IG/preintegration/preintegration_normal.cc:155-232 +
    // PreintegrationBase::integration, preintegration_base.cc:39-70): no Earth-rotation / Coriolis terms; the blob is tagged (blob[477] = 1)
    // so that the factor evaluates PreintegrationNormal::evaluate.
    if (!state16 || !gravity3 || !noise5 || !imu || !blob || n < 1) {
        set_error("icg_imu_preintegrate: bad arguments");
        return ICG_EINVAL;
    }
    gc::preintegrate_core(state16, iewn3, gravity3, noise5, imu, n, blob, end_state10);  // one definition for host and device (geom_core.cuh)
    return ICG_OK;
}

static int ba_create_body(icg_ba *h, int max_windows, int max_K, int max_L, int max_F, int max_gnss, int max_marg_r, void *stream);

int icg_ba_create(icg_ba **out, int max_windows, int max_K, int max_L, int max_F, int max_gnss, int max_marg_r, int device, void *stream) {
    if (!out || max_windows < 1 || max_K < 2 || max_K > 32 || max_L < 0 || max_F < 0 || max_gnss < 0 || max_marg_r < 0) {
        set_error("icg_ba_create: bad arguments");
        return ICG_EINVAL;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        set_error("icg_ba_create: no CUDA device (this library has no CPU fallback)");
        return ICG_ENODEVICE;
    }
    if (device < 0 || device >= ndev) {
        set_error("icg_ba_create: device %d out of range", device);
        return ICG_EINVAL;
    }
    ICG_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    ICG_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        set_error("icg_ba_create: device is sm_%d%d; this library is built for sm_100a only", prop.major, prop.minor);
        return ICG_ENODEVICE;
    }
    icg_ba *h = new icg_ba();
    h->device = device;
    const int rc_init = ba_create_body(h, max_windows, max_K, max_L, max_F, max_gnss, max_marg_r, stream);
    if (rc_init != ICG_OK) {  // every failure path releases what was already allocated (streams, events, pinned + device memory)
        icg_ba_destroy(h);
        return rc_init;
    }
    *out = h;
    return ICG_OK;
}

static int ba_create_body(icg_ba *h, int max_windows, int max_K, int max_L, int max_F, int max_gnss, int max_marg_r, void *stream) {
    if (stream) {
        h->stream = (cudaStream_t) stream;
    } else {
        ICG_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
        h->own_stream = true;
    }
    {   // the forked camera-factor kernels are one latency-bound CTA per window: give them priority so that they are placed before the
        // wide vision kernels fill the SMs (otherwise they start late and then contend with the Schur / Gram kernels)
        int prio_lo = 0, prio_hi = 0;
        ICG_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        ICG_CUDA(cudaStreamCreateWithPriority(&h->stream_cam, cudaStreamNonBlocking, prio_hi));
    }
    ICG_CUDA(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    ICG_CUDA(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    h->prof = getenv("ICG_BA_PROFILE") != nullptr;
    if (h->prof) {
        double *ck = nullptr;
        if (dmalloc(h, &ck, 48) != ICG_OK) return ICG_ENOMEM;
        h->D.clk = (unsigned long long *) ck;
    }
    if (getenv("ICG_BA_PROFILE_SKIP")) h->prof_skip = atoi(getenv("ICG_BA_PROFILE_SKIP"));
    BaCaps &C = h->C;
    max_L = std::max(1, max_L), max_F = std::max(1, max_F);  // capacities stay >= 1; windows without landmarks (first keyframes, IG/ic_gvins.cc:1698) are accepted
    C.NW = max_windows, C.K = max_K, C.L = max_L, C.F = max_F, C.G = std::max(1, max_gnss), C.R = std::max(1, max_marg_r);
    C.NCV = 6 * max_K + 7, C.N = 15 * max_K + 7, C.NS = (C.N + 3) & ~3, C.NCA = 4 * ((C.NCV + 1 + 3) / 4);
    C.RJ = (2 * max_F + 31) & ~31, C.LP = (max_L + 31) & ~31;
    C.NVB = (max_F + 127 - max_K) / (128 - max_K) + max_L / 128 + 4;  // worst case: every run is cut short by one landmark's K - 1 factors
    h->nblk_vis = (max_F + 255) / 256;
    const size_t NW = max_windows;
#define HD(field, count)                                                       \
    if (h->field.alloc(count) != ICG_OK) {                                     \
        set_error("icg_ba_create: allocation of " #field " failed");           \
        return ICG_ENOMEM;                                                     \
    }
    HD(dims, NW) HD(st, NW) HD(pose, NW * C.K * 7) HD(mix, NW * C.K * 9) HD(ext, NW * 8) HD(rho, NW * C.L)
    HD(imu_blob, NW * C.K * ICG_IMU_BLOB_DOUBLES) HD(imu_U, NW * C.K * 225) HD(gnss_blh, NW * C.G * 3) HD(gnss_std, NW * C.G * 3) HD(lever, NW * 3)
    HD(pose_prior, NW * 7) HD(pose_prior_sinfo, NW * 6) HD(mix_prior, NW * 9) HD(mix_prior_std, NW * 9) HD(marg_x0, NW * BA_MARG_MAXB * 9)
    HD(marg_H0, NW * C.R * C.R) HD(marg_b0, NW * C.R) HD(marg_c0, NW)
    HD(lm_off, NW * (C.L + 1)) HD(lm_fidx, NW * C.F) HD(gnss_node, NW * C.G) HD(marg_type, NW * BA_MARG_MAXB) HD(marg_node, NW * BA_MARG_MAXB) HD(f_active, NW * C.F)
    HD(scratch, 1024) HD(st_save, NW) HD(cull_counters, 2 * NW) HD(f_slot, NW * C.F) HD(f_meta_s, NW * C.F * 4) HD(vb_lm0, NW * C.NVB) HD(f_const_s, NW * C.F * 14)
    HD(pair_off, NW * ((size_t) C.K * (C.K - 1) + 1)) HD(pair_ro, NW * (size_t) C.K * (C.K - 1)) HD(pair_fidx, NW * C.F) HD(npairs, NW)
#undef HD
    BaDev &D = h->D;
    D.rank = 0, D.world = 1;
    D.dims = h->dims.d, D.st = h->st.d, D.pose = h->pose.d, D.mix = h->mix.d, D.ext = h->ext.d, D.rho = h->rho.d;
    D.f_active = h->f_active.d;
    D.pair_off = h->pair_off.d, D.pair_ro = h->pair_ro.d, D.pair_fidx = h->pair_fidx.d, D.npairs = h->npairs.d;
    D.f_meta_s = h->f_meta_s.d, D.vb_lm0 = h->vb_lm0.d, D.f_const_s = h->f_const_s.d;
    D.lm_off = h->lm_off.d, D.imu_blob = h->imu_blob.d, D.imu_U = h->imu_U.d;
    D.gnss_node = h->gnss_node.d, D.gnss_blh = h->gnss_blh.d, D.gnss_std = h->gnss_std.d, D.lever = h->lever.d;
    D.pose_prior = h->pose_prior.d, D.pose_prior_sinfo = h->pose_prior_sinfo.d, D.mix_prior = h->mix_prior.d, D.mix_prior_std = h->mix_prior_std.d;
    D.marg_type = h->marg_type.d, D.marg_node = h->marg_node.d, D.marg_x0 = h->marg_x0.d, D.marg_H0 = h->marg_H0.d, D.marg_b0 = h->marg_b0.d, D.marg_c0 = h->marg_c0.d;
    int rc = ICG_OK;
#define DM(field, count) \
    if (rc == ICG_OK) rc = dmalloc(h, &D.field, count);
    DM(pose_c, NW * C.K * 7) DM(mix_c, NW * C.K * 9) DM(ext_c, NW * 8) DM(rho_c, NW * C.L)
    DM(pose_0, NW * C.K * 7) DM(mix_0, NW * C.K * 9) DM(ext_0, NW * 8) DM(rho_0, NW * C.L)
    DM(AW, NW * C.NCA * C.LP) DM(Mp, NW * (size_t) C.K * (C.K - 1) * 210) DM(CJ, NW * BA_SPLIT_J * C.NCA * C.NCA) DM(CW, NW * BA_SPLIT_W * C.NCA * C.NCA)
    DM(jcomp, NW * C.F * 40) DM(costf, NW * C.F) DM(hl, NW * C.L) DM(gl, NW * C.L) DM(scale_l, NW * C.L) DM(scale_c, NW * C.NS)
    DM(Hc, NW * C.NS * C.NS) DM(gc, NW * C.NS) DM(Hs, NW * C.NS * C.NS) DM(cost_part, NW * (h->nblk_vis + 1)) DM(red2, NW * 4) DM(step_c, NW * C.NS) DM(step_l, NW * C.L)
#undef DM
    if (rc == ICG_OK) rc = dmalloc(h, &D.gnss_std_0, NW * C.G * 3);
    if (rc == ICG_OK) {
        double *fa0 = nullptr;
        rc = dmalloc(h, &fa0, (NW * C.F + 7) / 8 + 1);
        D.f_active_0 = (uint8_t *) fa0;
    }
    if (rc != ICG_OK) return rc;
    // shared-memory budgets
    h->smem_cam = sizeof(double) * ((size_t) C.K * 480 + (size_t) C.G * 24 + 48 + 16 + 2 * (size_t) C.R + 8) + sizeof(int) * (size_t) C.R + 64;
    size_t vec = sizeof(double) * (40 + 5 * (size_t) C.NS);
    size_t packed = sizeof(double) * ((size_t) (C.N + 1) * (C.N + 2) / 2);
    h->use_global_S = (vec + packed > 220 * 1024) ? 1 : 0;
    h->smem_solve = vec + (h->use_global_S ? 0 : packed);
    D.Sglobal = nullptr;
    memset(&D.S, 0, sizeof(D.S));
    if (h->use_global_S) {  // the reduced system does not fit one CTA: the split pipeline (cluster solve, S in L2) drives this handle
        rc = split_setup(h, 0, 1);
        if (rc != ICG_OK) return rc;
    } else {
        ICG_CUDA(raise_dynamic_smem((const void *) ba_solve, (size_t) (h->smem_solve)));
    }
    h->ld_schur = 16 * ((C.NCA + 15) / 16) + 8;  // = 8 mod 16 doubles: conflict-free fragment reads
    h->smem_schur = sizeof(double) * ((size_t) SCHUR_RCH * h->ld_schur + SCHUR_RCH);
    ICG_CUDA(raise_dynamic_smem((const void *) ba_schur_dmma, (size_t) (h->smem_schur)));
    ICG_CUDA(cudaFuncSetAttribute(ba_schur_dmma, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    ICG_CUDA(raise_dynamic_smem((const void *) ba_lin_cam, (size_t) (h->smem_cam)));
    ICG_CUDA(raise_dynamic_smem((const void *) ba_cost_cam, (size_t) (h->smem_cam)));
    ICG_CUDA(raise_dynamic_smem((const void *) ba_lin_vis, LV_SMEM));
    ICG_CUDA(cudaStreamSynchronize(h->stream));
    h->cur_windows = 0;
    return ICG_OK;
}

void icg_ba_destroy(icg_ba *h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    prof_collect(h);
    prof_print(h);
    for (cudaEvent_t e : h->prof_ev) cudaEventDestroy(e);
    h->dims.release(), h->st.release(), h->pose.release(), h->mix.release(), h->ext.release(), h->rho.release();
    h->imu_blob.release(), h->imu_U.release(), h->gnss_blh.release(), h->gnss_std.release(), h->lever.release(), h->pose_prior.release();
    h->pose_prior_sinfo.release(), h->mix_prior.release(), h->mix_prior_std.release(), h->marg_x0.release(), h->marg_H0.release(), h->marg_b0.release();
    h->marg_c0.release(), h->lm_off.release(), h->lm_fidx.release(), h->gnss_node.release();
    h->f_slot.release(), h->f_meta_s.release(), h->vb_lm0.release(), h->f_const_s.release(), h->marg_type.release(), h->marg_node.release(), h->f_active.release(), h->scratch.release(), h->st_save.release(), h->cull_counters.release(), h->pair_off.release(), h->pair_ro.release(), h->pair_fidx.release(), h->npairs.release();
    split_release(h);
    if (h->marg_ready) h->marg_map.release(), h->marg_oJ0.release(), h->marg_oe0.release(), h->marg_oHp.release(), h->marg_obp.release();
    h->cull_buf.release();
    for (void *p : h->dev_only) cudaFree(p);
    if (h->stream_cam) cudaStreamSynchronize(h->stream_cam), cudaStreamDestroy(h->stream_cam);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

// pack + upload n problems (host side of the seam: what AddParameterBlock / AddResidualBlock do in IG/ic_gvins.cc:1697-1909)
int icg_ba_upload(icg_ba *h, int n, const icg_ba_problem *P) {
    if (!h || !P || n < 1 || n > h->C.NW) {
        set_error("icg_ba_upload: bad arguments (n=%d, capacity %d)", n, h ? h->C.NW : 0);
        return ICG_EINVAL;
    }
    ICG_CUDA(cudaSetDevice(h->device));
    const BaCaps &C = h->C;
    // per-window packing is independent (disjoint slices of the pinned staging arrays): spread it over a few host threads -- it is
    // memcpy-bound (about 0.4 MB per cfg-3 window) and sits inside the end-to-end path of every keyframe
#define PK_FAIL(code, ...)                          \
    do {                                            \
        char eb_[512];                              \
        snprintf(eb_, sizeof(eb_), __VA_ARGS__);    \
        err = eb_;                                  \
        return code;                                \
    } while (0)
    auto pack_one = [&](int w, std::string &err) -> int {
        const icg_ba_problem &p = P[w];
        if (p.K < 2 || p.K > C.K || p.L < 0 || p.L > C.L || p.F < 0 || p.F > C.F || p.n_imu < 0 || p.n_imu > p.K - 1 || p.n_gnss < 0 || p.n_gnss > C.G ||
            p.marg_r < 0 || p.marg_r > C.R || p.marg_nblocks < 0 || p.marg_nblocks > 2 * C.K + 2 || !p.pose || !p.mix || !p.ext || (p.L > 0 && !p.invdepth) ||
            (p.F > 0 && (!p.f_lm || !p.f_ref || !p.f_obs || !p.f_const))) {
            PK_FAIL(ICG_EINVAL, "icg_ba_upload: window %d exceeds the handle's capacity or has null parameter arrays (K=%d L=%d F=%d gnss=%d marg_r=%d)", w, p.K, p.L, p.F,
                      p.n_gnss, p.marg_r);
        }
        WinDims &d = h->dims.h[w];
        d.K = p.K, d.L = p.L, d.F = p.F, d.n_imu = p.n_imu, d.n_gnss = p.n_gnss, d.marg_r = p.marg_r, d.marg_nb = p.marg_nblocks;
        d.ext_const = p.ext_const != 0, d.td_const = p.td_const != 0, d.reproj_huber = p.reproj_huber != 0, d.gnss_huber = p.gnss_huber != 0;
        d.has_imu_error = p.has_imu_error != 0, d.has_pose_prior = p.has_pose_prior != 0, d.has_mix_prior = p.has_mix_prior != 0;
        d.reproj_sinv = 1.0 / p.reproj_std;
        memcpy(h->pose.h + (size_t) w * C.K * 7, p.pose, sizeof(double) * 7 * p.K);
        memcpy(h->mix.h + (size_t) w * C.K * 9, p.mix, sizeof(double) * 9 * p.K);
        memcpy(h->ext.h + (size_t) w * 8, p.ext, sizeof(double) * 8);
        if (p.L > 0) memcpy(h->rho.h + (size_t) w * C.L, p.invdepth, sizeof(double) * p.L);
        for (int f = 0; f < p.F; f++) {
            if (p.f_lm[f] < 0 || p.f_lm[f] >= p.L || p.f_ref[f] < 0 || p.f_ref[f] >= p.K || p.f_obs[f] < 0 || p.f_obs[f] >= p.K || p.f_ref[f] == p.f_obs[f]) {
                PK_FAIL(ICG_EINVAL, "icg_ba_upload: window %d factor %d has invalid indices", w, f);
            }
        }
        {   // a map point has one reference frame and at most one observation per keyframe (IG/ic_gvins.cc:1777-1834): lin_lm relies on it
            std::vector<int> refof(p.L, -1);
            std::vector<unsigned> seen((size_t) p.L, 0u);
            for (int f = 0; f < p.F; f++) {
                const int l = p.f_lm[f];
                if (refof[l] < 0) refof[l] = p.f_ref[f];
                if (refof[l] != p.f_ref[f] || (seen[l] >> p.f_obs[f]) & 1u) {
                    PK_FAIL(ICG_EINVAL, "icg_ba_upload: window %d factor %d: landmark %d has two reference nodes or two observations in node %d", w, f, l, p.f_obs[f]);
                }
                seen[l] |= 1u << p.f_obs[f];
            }
        }
        if (p.f_active)
            memcpy(h->f_active.h + (size_t) w * C.F, p.f_active, p.F);
        else
            memset(h->f_active.h + (size_t) w * C.F, 1, p.F);
        // CSR by landmark
        int *off = h->lm_off.h + (size_t) w * (C.L + 1), *fidx = h->lm_fidx.h + (size_t) w * C.F;
        for (int l = 0; l <= p.L; l++) off[l] = 0;
        for (int f = 0; f < p.F; f++) off[p.f_lm[f] + 1]++;
        for (int l = 0; l < p.L; l++) off[l + 1] += off[l];
        int *fslot = h->f_slot.h + (size_t) w * C.F;
        {
            std::vector<int> cur(off, off + p.L);
            for (int f = 0; f < p.F; f++) fslot[f] = cur[p.f_lm[f]], fidx[cur[p.f_lm[f]]++] = f;
            // lin_vis runs: greedy packing of whole landmarks into <= 128 record slots
            int *vbh = h->vb_lm0.h + (size_t) w * C.NVB;
            int nrun = 0, l0 = 0;
            while (l0 < p.L) {
                int l1 = l0;
                while (l1 < p.L && off[l1 + 1] - off[l0] <= 128) l1++;
                if (l1 == l0 || nrun >= C.NVB - 2) PK_FAIL(ICG_EINVAL, "icg_ba_upload: window %d: landmark %d has more than 128 factors or the run table overflows", w, l0);
                vbh[nrun++] = l0;
                l0 = l1;
            }
            vbh[nrun] = p.L;
            vbh[C.NVB - 1] = nrun;
            int *meta = h->f_meta_s.h + (size_t) w * C.F * 4;
            double *fcs = h->f_const_s.h + (size_t) w * C.F * 14;
            for (int q = 0; q < p.F; q++) {
                const int f = fidx[q];
                meta[4 * q] = p.f_lm[f], meta[4 * q + 1] = p.f_ref[f], meta[4 * q + 2] = p.f_obs[f], meta[4 * q + 3] = f;
                memcpy(fcs + (size_t) q * 14, p.f_const + (size_t) f * 14, sizeof(double) * 14);
            }
        }
        // CSR by (reference node, observing node) pair
        {
            const int PM = C.K * (C.K - 1);
            int *poff = h->pair_off.h + (size_t) w * (PM + 1), *pro = h->pair_ro.h + (size_t) w * PM, *pfidx = h->pair_fidx.h + (size_t) w * C.F;
            std::vector<int> cnt((size_t) p.K * p.K, 0), slot((size_t) p.K * p.K, -1);
            for (int f = 0; f < p.F; f++) cnt[(size_t) p.f_ref[f] * p.K + p.f_obs[f]]++;
            int P = 0;
            poff[0] = 0;
            for (int key = 0; key < p.K * p.K; key++)
                if (cnt[key]) {
                    slot[key] = P;
                    pro[P] = ((key / p.K) << 8) | (key % p.K);
                    poff[P + 1] = poff[P] + cnt[key];
                    P++;
                }
            std::vector<int> cur(poff, poff + P);
            for (int f = 0; f < p.F; f++) pfidx[cur[slot[(size_t) p.f_ref[f] * p.K + p.f_obs[f]]]++] = fslot[f];  // record slots, not factor ids
            h->npairs.h[w] = P;
        }
        for (int k = 0; k < p.n_imu; k++) {
            const double *b = p.imu_blob + (size_t) k * ICG_IMU_BLOB_DOUBLES;
            memcpy(h->imu_blob.h + ((size_t) w * C.K + k) * ICG_IMU_BLOB_DOUBLES, b, sizeof(double) * ICG_IMU_BLOB_DOUBLES);
            if (!host_imu_sqrt_info(b + 252, h->imu_U.h + ((size_t) w * C.K + k) * 225)) {
                PK_FAIL(ICG_EINVAL, "icg_ba_upload: window %d IMU factor %d has a non positive-definite covariance", w, k);
            }
        }
        for (int g = 0; g < p.n_gnss; g++) {
            if (p.gnss_node[g] < 0 || p.gnss_node[g] >= p.K) {
                PK_FAIL(ICG_EINVAL, "icg_ba_upload: window %d GNSS factor %d has an invalid node", w, g);
            }
            h->gnss_node.h[(size_t) w * C.G + g] = p.gnss_node[g];
        }
        if (p.n_gnss) {
            memcpy(h->gnss_blh.h + (size_t) w * C.G * 3, p.gnss_blh, sizeof(double) * 3 * p.n_gnss);
            memcpy(h->gnss_std.h + (size_t) w * C.G * 3, p.gnss_std, sizeof(double) * 3 * p.n_gnss);
        }
        memcpy(h->lever.h + (size_t) w * 3, p.lever, sizeof(double) * 3);
        if (p.has_pose_prior) {
            memcpy(h->pose_prior.h + (size_t) w * 7, p.pose_prior, sizeof(double) * 7);
            for (int k = 0; k < 6; k++) h->pose_prior_sinfo.h[(size_t) w * 6 + k] = 1.0 / p.pose_prior_std[k];
        }
        if (p.has_mix_prior) {
            memcpy(h->mix_prior.h + (size_t) w * 9, p.mix_prior, sizeof(double) * 9);
            memcpy(h->mix_prior_std.h + (size_t) w * 9, p.mix_prior_std, sizeof(double) * 9);
        }
        if (p.marg_r > 0) {
            // the prior is linear: H0 = J0^T J0, b0 = J0^T e0, c0 = e0.e0 are constant over the solve (marginalization_factor.h:79-81)
            const int r = p.marg_r;
            int tot = 0, cols = 0;
            for (int b = 0; b < p.marg_nblocks; b++) {
                int t = p.marg_block_type[b];
                if (t < 0 || t > 3 || ((t == 0 || t == 1) && (p.marg_block_node[b] < 0 || p.marg_block_node[b] >= p.K))) {
                    PK_FAIL(ICG_EINVAL, "icg_ba_upload: window %d marginalization block %d invalid", w, b);
                }
                tot += (t == 0 || t == 2) ? 7 : t == 1 ? 9 : 1;
                cols += (t == 0 || t == 2) ? 6 : t == 1 ? 9 : 1;
                h->marg_type.h[(size_t) w * BA_MARG_MAXB + b] = t;
                h->marg_node.h[(size_t) w * BA_MARG_MAXB + b] = p.marg_block_node[b];
            }
            if (cols != r || tot > BA_MARG_MAXB * 9) {
                PK_FAIL(ICG_EINVAL, "icg_ba_upload: window %d marginalization prior size mismatch (blocks give %d columns, marg_r=%d)", w, cols, r);
            }
            memcpy(h->marg_x0.h + (size_t) w * BA_MARG_MAXB * 9, p.marg_x0, sizeof(double) * tot);
            double *H0 = h->marg_H0.h + (size_t) w * C.R * C.R, *b0 = h->marg_b0.h + (size_t) w * C.R;
            for (int i = 0; i < r; i++) {
                for (int j = i; j < r; j++) {
                    double s = 0;
                    for (int k = 0; k < r; k++) s += p.marg_J0[(size_t) k * r + i] * p.marg_J0[(size_t) k * r + j];
                    H0[(size_t) i * r + j] = H0[(size_t) j * r + i] = s;
                }
                double s = 0;
                for (int k = 0; k < r; k++) s += p.marg_J0[(size_t) k * r + i] * p.marg_e0[k];
                b0[i] = s;
            }
            double c0 = 0;
            for (int k = 0; k < r; k++) c0 += p.marg_e0[k] * p.marg_e0[k];
            h->marg_c0.h[w] = c0;
        }
            return ICG_OK;
    };
#undef PK_FAIL
    {
        const int nthreads = std::max(1, std::min({n / 4, 16, (int) std::thread::hardware_concurrency()}));
        std::vector<int> rcs(nthreads, ICG_OK);
        std::vector<std::string> errs(nthreads);
        auto worker = [&](int t) {
            for (int w = t; w < n; w += nthreads) {
                const int rc = pack_one(w, errs[t]);
                if (rc != ICG_OK) {
                    rcs[t] = rc;
                    return;
                }
            }
        };
        std::vector<std::thread> th;
        for (int t = 1; t < nthreads; t++) th.emplace_back(worker, t);
        worker(0);
        for (auto &x : th) x.join();
        for (int t = 0; t < nthreads; t++)
            if (rcs[t] != ICG_OK) {
                set_error("%s", errs[t].c_str());
                return rcs[t];
            }
    }
    cudaStream_t s = h->stream;
    {   // H2D of the n uploaded windows only (the arrays are capacity-strided by window; a partially filled handle moves a prefix)
        const size_t nn = (size_t) n, PM = (size_t) C.K * (C.K - 1);
#define UP(field, stride) ICG_CUDA(h->field.up(s, nn * (size_t) (stride)))
        UP(dims, 1); UP(pose, C.K * 7); UP(mix, C.K * 9); UP(ext, 8); UP(rho, C.L);
        UP(f_active, C.F);  // factor constants and indices travel once, in record-slot order (f_meta_s / f_const_s)
        UP(f_meta_s, C.F * 4); UP(vb_lm0, C.NVB); UP(f_const_s, C.F * 14); UP(lm_off, C.L + 1); UP(pair_off, PM + 1); UP(pair_ro, PM); UP(pair_fidx, C.F);
        UP(npairs, 1); UP(imu_blob, C.K * ICG_IMU_BLOB_DOUBLES); UP(imu_U, C.K * 225);
        UP(gnss_node, C.G); UP(gnss_blh, C.G * 3); UP(gnss_std, C.G * 3); UP(lever, 3);
        UP(pose_prior, 7); UP(pose_prior_sinfo, 6); UP(mix_prior, 9); UP(mix_prior_std, 9);
        UP(marg_type, BA_MARG_MAXB); UP(marg_node, BA_MARG_MAXB); UP(marg_x0, BA_MARG_MAXB * 9); UP(marg_H0, (size_t) C.R * C.R); UP(marg_b0, C.R); UP(marg_c0, 1);
#undef UP
    }
    // keep a pristine copy of the parameters (icg_ba_run(restart=1) re-solves the same problems: bench / repeated solves)
    const BaDev &D = h->D;
    ICG_CUDA(cudaMemcpyAsync(D.pose_0, D.pose, sizeof(double) * (size_t) n * C.K * 7, cudaMemcpyDeviceToDevice, s));
    ICG_CUDA(cudaMemcpyAsync(D.mix_0, D.mix, sizeof(double) * (size_t) n * C.K * 9, cudaMemcpyDeviceToDevice, s));
    ICG_CUDA(cudaMemcpyAsync(D.ext_0, D.ext, sizeof(double) * (size_t) n * 8, cudaMemcpyDeviceToDevice, s));
    ICG_CUDA(cudaMemcpyAsync(D.rho_0, D.rho, sizeof(double) * (size_t) n * C.L, cudaMemcpyDeviceToDevice, s));
    ICG_CUDA(cudaMemcpyAsync(D.f_active_0, D.f_active, (size_t) n * C.F, cudaMemcpyDeviceToDevice, s));
    ICG_CUDA(cudaMemcpyAsync(D.gnss_std_0, D.gnss_std, sizeof(double) * (size_t) n * C.G * 3, cudaMemcpyDeviceToDevice, s));
    // the dense SYRK operands keep a fixed sparsity pattern per problem: zero them once here
    h->cur_windows = n;
    return ICG_OK;
}

// ---- in-situ stage timing
static const char *PROF_NAMES[16] = {"(gap/other)", "lin_vis", "lin_lm", "pair_gram1", "", "schur_dmma", "join lin_cam + lin_done",
                                     "export + signal", "solve", "cost (+cost_cam)", "exchange", "accept", "hsum / reduce", "join gram chain", "step_lm", ""};
static void prof_mark(icg_ba *h, int tag) {
    if (!h->prof) return;
    if (h->prof_used == h->prof_ev.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        h->prof_ev.push_back(e);
        h->prof_tag.push_back(0);
    }
    h->prof_tag[h->prof_used] = tag;
    cudaEventRecord(h->prof_ev[h->prof_used++], h->stream);
}
static void prof_collect(icg_ba *h) {  // call after the stream has been synchronised
    if (!h->prof) return;
    if (h->prof_used && h->prof_skip > 0) {
        h->prof_skip--;
        h->prof_used = 0;
        return;
    }
    for (size_t i = 1; i < h->prof_used; i++) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, h->prof_ev[i - 1], h->prof_ev[i]) == cudaSuccess) {
            h->prof_ms[h->prof_tag[i]] += ms;
            h->prof_cnt[h->prof_tag[i]]++;
        }
    }
    h->prof_used = 0;
}
static void prof_print(icg_ba *h) {
    if (!h->prof) return;
    double tot = 0;
    for (int t = 0; t < 16; t++) tot += h->prof_ms[t];
    fprintf(stderr, "[icg_ba profile] handle %p, %d windows: stage totals over all recorded LM sequences (ms, mean us, share)\n", (void *) h, h->cur_windows);
    for (int t = 0; t < 16; t++)
        if (h->prof_cnt[t])
            fprintf(stderr, "  %-28s %9.3f ms  %8.1f us  %5.1f %%\n", PROF_NAMES[t], h->prof_ms[t], 1e3 * h->prof_ms[t] / h->prof_cnt[t], 100.0 * h->prof_ms[t] / tot);
    if (h->D.clk) {
        unsigned long long ck[48];
        if (cudaMemcpy(ck, h->D.clk, sizeof(ck), cudaMemcpyDeviceToHost) == cudaSuccess) {
            static const char *cn[6] = {"factor evaluation", "prior product + cost", "zero H_c", "prior blocks", "IMU J^T J", "GNSS / prior diagonals"};
            fprintf(stderr, "[icg_ba profile] ba_lin_cam phases of window 0 (SM cycles per call, mean):\n");
            for (int k = 0; k < 6; k++)
                if (ck[24 + k]) fprintf(stderr, "  %-28s %9.0f cycles\n", cn[k], (double) ck[16 + k] / (double) ck[24 + k]);
            if (h->D.S.split) {
                static const char *sn_l2[6] = {"per panel: stage B operand", "per panel: warp 0 tile + factor", "per panel: tiles + barrier 1", "per panel: row solve + barrier 2", "whole factorisation", ""};
                static const char *sn_dsm[6] = {"assembly", "per panel: warp 0 tile + factor", "per panel: until block barrier", "per panel: row solve + cl. barrier", "whole factorisation", "backward substitution"};
                const char **sn = h->solve_cam_dsm ? sn_dsm : sn_l2;
                fprintf(stderr, "[icg_ba profile] %s phases of window 0 (SM cycles, mean):\n", h->solve_cam_dsm ? "ba_solve_cam_dsm" : "ba_solve_cam");
                for (int k = 0; k < 6; k++)
                    if (ck[8 + k]) fprintf(stderr, "  %-34s %9.0f cycles\n", sn[k], (double) ck[k] / (double) ck[8 + k]);
                static const char *sn2[5] = {"per panel: wait for the panel column", "(unused)", "per panel: warp 0 diagonal-tile update", "per panel: warp 0 loads + 8x8 factorisation", "per panel: warp 0 write-back"};
                for (int k = 0; k < 5 && h->solve_cam_dsm; k++)
                    if (ck[40 + k]) fprintf(stderr, "  %-50s %9.0f cycles\n", sn2[k], (double) ck[32 + k] / (double) ck[40 + k]);
            }
            static const char *nm[8] = {"gradient / cost / tests", "assembly", "Cholesky", "camera back-substitution", "landmark back-substitution", "candidate + reductions",
                                        "  per panel: warp 0 tile+factor", "  per panel: row solve phase"};
            if (!h->D.S.split) fprintf(stderr, "[icg_ba profile] ba_solve phases of window 0 (SM cycles per call, mean):\n");
            for (int k = 0; k < 8 && !h->D.S.split; k++)
                if (ck[8 + k]) fprintf(stderr, "  %-28s %9.0f cycles\n", nm[k], (double) ck[k] / (double) ck[8 + k]);
        }
    }
}

static int enqueue_lm_split(icg_ba *h, int max_num_iterations);

static int enqueue_lm(icg_ba *h, int max_num_iterations) {
    if (h->D.S.split) return enqueue_lm_split(h, max_num_iterations);
    const BaCaps &C = h->C;
    const BaDev &D = h->D;
    const int n = h->cur_windows;
    cudaStream_t s = h->stream;
    const dim3 g_vis(C.NVB - 2, n), g_cost(h->nblk_vis, n);
    // iteration 0 linearisation + (max_iter) x [schur syrk, solve, cost, accept, re-linearise]; one extra solve call
    // performs the final termination bookkeeping.
    for (int it = 0; it <= max_num_iterations; it++) {
        // fork: IMU / GNSS / prior factors (one latency-bound CTA per window) run beside the vision chain, from ba_lin_vis on (measured
        // against forking them beside the Schur / Gram kernels instead: profiles/r2_ba_stages.md)
        ICG_CUDA(cudaEventRecord(h->ev_fork, s));
        ICG_CUDA(cudaStreamWaitEvent(h->stream_cam, h->ev_fork, 0));
        ba_lin_cam<<<n, h->cam_threads, h->smem_cam, h->stream_cam>>>(C, D);
        ICG_CUDA(cudaEventRecord(h->ev_join, h->stream_cam));
        prof_mark(h, 0);
        ba_lin_vis<<<g_vis, 128, LV_SMEM, s>>>(C, D);
        prof_mark(h, 1);
        // (measured: one fused launch or two streams are both slower -- the Schur CTAs' shared memory throttles the latency-bound
        //  Gram warps when they share SMs)
        ba_schur_dmma<<<dim3(BA_SPLIT_W, n), 256, h->smem_schur, s>>>(C, D, h->ld_schur);
        prof_mark(h, 5);
        ba_pair_gram1<<<dim3((C.K * (C.K - 1) + 7) / 8, n), 256, 0, s>>>(C, D);
        prof_mark(h, 3);
        ICG_CUDA(cudaStreamWaitEvent(s, h->ev_join, 0));
        prof_mark(h, 6);
        ba_hsum<<<dim3(((C.NCV + 1) * (C.NCV + 1) + 255) / 256, n), 256, 0, s>>>(C, D);
        prof_mark(h, 12);
        ba_solve<<<n, SOLVE_THREADS, h->smem_solve, s>>>(C, D);
        prof_mark(h, 8);
        count_launch(6);
        if (it == max_num_iterations) break;
        ICG_CUDA(cudaEventRecord(h->ev_fork, s));
        ICG_CUDA(cudaStreamWaitEvent(h->stream_cam, h->ev_fork, 0));
        ba_cost_cam<<<n, h->cam_threads, h->smem_cam, h->stream_cam>>>(C, D, h->nblk_vis);
        ICG_CUDA(cudaEventRecord(h->ev_join, h->stream_cam));
        ba_cost<<<g_cost, 256, 0, s>>>(C, D, h->nblk_vis);
        ICG_CUDA(cudaStreamWaitEvent(s, h->ev_join, 0));
        prof_mark(h, 9);
        ba_accept<<<n, 128, 0, s>>>(C, D, h->nblk_vis);
        prof_mark(h, 11);
        count_launch(3);
    }
    ICG_CHECK_LAUNCH();
    return ICG_OK;
}

// ---- split pipeline: host side
static void split_release(icg_ba *h) {
    for (int r = 0; r < 8; r++)
        if (h->ipc_opened[r]) cudaIpcCloseMemHandle(h->ipc_opened[r]), h->ipc_opened[r] = nullptr;
    if (h->xbuf) cudaFree(h->xbuf), h->xbuf = nullptr;
    if (h->D.S.redv) cudaFree(h->D.S.redv), h->D.S.redv = nullptr;
    if (h->D.S.err) cudaFree(h->D.S.err), h->D.S.err = nullptr;
    if (h->D.S.slm) cudaFree(h->D.S.slm), h->D.S.slm = nullptr;
    if (h->D.S.slm_cnt) cudaFree(h->D.S.slm_cnt), h->D.S.slm_cnt = nullptr;
    if (h->D.Sglobal) cudaFree(h->D.Sglobal), h->D.Sglobal = nullptr;
    h->D.S.split = 0;
}

// (re)allocate the exchange buffer of this rank for a group of `world` ranks and switch the handle to the split pipeline.  The layout
// depends only on (max_windows, max_K, world), so every rank computes the same offsets.
static int split_setup(icg_ba *h, int rank, int world) {
    if (world < 1 || world > 8 || rank < 0 || rank >= world) {
        set_error("split pipeline: rank %d / world %d out of range (<= 8 GPUs of one box)", rank, world);
        return ICG_EINVAL;
    }
    ICG_CUDA(cudaSetDevice(h->device));
    ICG_CUDA(cudaStreamSynchronize(h->stream));
    split_release(h);
    const BaCaps &C = h->C;
    ShardDev &S = h->D.S;
    const size_t NW = C.NW, G = world;
    const size_t TRI = (size_t) C.NCV * (C.NCV + 1) / 2;
    S.PK = (int) ((TRI + 3 * (size_t) C.NCV + 4 + 3) & ~(size_t) 3);
    S.BS = (SPLIT_HDR + C.NS + 3) & ~3;
    S.RV = (3 * C.NCV + 4 + 3) & ~3;
    const size_t NWo = (NW + G - 1) / G;
    size_t off = 0;
    S.off_inbox = off, off += NWo * G * S.PK;
    S.off_bcast = off, off += NW * S.BS;
    S.off_scal = off, off += NW * G * SPLIT_SCAL;
    S.off_flagA = off, off += 8;
    S.off_flagB = off, off += (NW + 3) & ~(size_t) 3;
    S.off_flagC = off, off += (NW * G + 3) & ~(size_t) 3;
    h->xbuf_doubles = off;
    if (cudaMalloc(&h->xbuf, sizeof(double) * off) != cudaSuccess || cudaMalloc(&S.redv, sizeof(double) * NW * S.RV) != cudaSuccess ||
        cudaMalloc(&S.err, sizeof(int) * 4) != cudaSuccess || cudaMalloc(&S.slm, sizeof(double) * NW * STEP_SLICES * 8) != cudaSuccess ||
        cudaMalloc(&S.slm_cnt, sizeof(int) * NW) != cudaSuccess ||
        cudaMalloc(&h->D.Sglobal, sizeof(double) * NWo * split_S_stride(C)) != cudaSuccess) {
        set_error("split pipeline: allocation of the exchange buffers failed (%zu doubles)", off);
        return ICG_ENOMEM;
    }
    ICG_CUDA(cudaMemset(h->xbuf, 0, sizeof(double) * off));
    ICG_CUDA(cudaMemset(S.redv, 0, sizeof(double) * NW * S.RV));
    ICG_CUDA(cudaMemset(S.err, 0, sizeof(int) * 4));
    ICG_CUDA(cudaMemset(S.slm, 0, sizeof(double) * NW * STEP_SLICES * 8));
    ICG_CUDA(cudaMemset(S.slm_cnt, 0, sizeof(int) * NW));
    for (int r = 0; r < 8; r++) S.peer[r] = nullptr;
    S.peer[rank] = h->xbuf;
    S.split = 1;
    h->D.rank = rank, h->D.world = world;
    // four or more landmark shards: the owner's camera-only kernels are on the attempt's critical path (the vision kernels shrink with the
    // shard -- 410 us at one rank, ~100 at four --, the per-window IMU chain of ~118 us does not): all 10 warps, two rounds of IMU factors at
    // K = 20 instead of four
    h->cam_threads = world >= 4 ? CAM_THREADS : 160;
    h->epoch = 0;
    {   // ba_solve_cam: vectors + the larger of the back-substitution staging and [B rows | 8 x 8 hand-over | one A strip per warp]; the A strips are
        // dropped when they do not fit (max_K > 20)
        const size_t ldbp = ((size_t) (C.N + 15) / 16) * 16 + 8;
        const size_t bs = (size_t) SPLIT_BS_ROWS * (C.NS + 1), base = 8 * ldbp + 64, strips = (size_t) (SOLVE_THREADS / 32) * 8 * ldbp;
        h->solve_cam_stage_a = sizeof(double) * (40 + 4 * (size_t) C.NS + std::max(bs, base + strips)) <= 220 * 1024;
        h->smem_solve_cam = sizeof(double) * (40 + 4 * (size_t) C.NS + std::max(bs, base + (h->solve_cam_stage_a ? strips : 0)));
    }
    h->smem_step_lm = sizeof(double) * (40 + (size_t) C.NS);
    h->smem_solve_cam_dsm = sizeof(double) * dsm_smem_doubles(C);
    h->solve_cam_dsm = h->smem_solve_cam_dsm <= 227 * 1024 && C.N <= 32 * 11;  // (the assembly stages <= 11 chunks of 32 columns per row)
    if (h->solve_cam_dsm) ICG_CUDA(raise_dynamic_smem((const void *) ba_solve_cam_dsm, h->smem_solve_cam_dsm));
    ICG_CUDA(raise_dynamic_smem((const void *) ba_solve_cam, (size_t) (h->smem_solve_cam)));
    ICG_CUDA(cudaFuncSetAttribute(ba_solve_cam, cudaFuncAttributeNonPortableClusterSizeAllowed, 0));
    ICG_CUDA(raise_dynamic_smem((const void *) ba_step_lm, (size_t) (h->smem_step_lm)));
    return ICG_OK;
}

static int launch_solve_cam(icg_ba *h, int n, unsigned long long epoch) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned) (n * SPLIT_CLUSTER)), cfg.blockDim = dim3(SOLVE_THREADS);
    cfg.dynamicSmemBytes = h->solve_cam_dsm ? h->smem_solve_cam_dsm : h->smem_solve_cam, cfg.stream = h->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = SPLIT_CLUSTER, at[0].val.clusterDim.y = 1, at[0].val.clusterDim.z = 1;
    cfg.attrs = at, cfg.numAttrs = 1;
    if (h->solve_cam_dsm) ICG_CUDA(cudaLaunchKernelEx(&cfg, ba_solve_cam_dsm, h->C, h->D, epoch));
    else ICG_CUDA(cudaLaunchKernelEx(&cfg, ba_solve_cam, h->C, h->D, epoch, (int) h->solve_cam_stage_a));
    return ICG_OK;
}

// One LM sequence of the split pipeline (see ba_split.cuh).  Window w of a sharded group is solved by rank w mod world; the solve kernel
// is launched over all windows and the clusters of windows owned elsewhere return at once.
static int enqueue_lm_split(icg_ba *h, int max_num_iterations) {
    const BaCaps &C = h->C;
    const BaDev &D = h->D;
    const int n = h->cur_windows;
    cudaStream_t s = h->stream;
    for (int r = 0; r < D.world; r++)
        if (!D.S.peer[r]) {
            set_error("landmark-sharded solve: peer %d is not connected (icg_ba_shard_connect)", r);
            return ICG_EINVAL;
        }
    const dim3 g_vis(C.NVB - 2, n), g_cost(h->nblk_vis, n), g_nn(((C.NCV + 1) * (C.NCV + 1) + 255) / 256, n);
    for (int it = 0; it <= max_num_iterations; it++) {
        const unsigned long long epoch = ++h->epoch;
        ICG_CUDA(cudaEventRecord(h->ev_fork, s));
        ICG_CUDA(cudaStreamWaitEvent(h->stream_cam, h->ev_fork, 0));
        ba_lin_cam<<<n, h->cam_threads, h->smem_cam, h->stream_cam>>>(C, D);
        ICG_CUDA(cudaEventRecord(h->ev_join, h->stream_cam));
        prof_mark(h, 0);
        ba_lin_vis<<<g_vis, 128, LV_SMEM, s>>>(C, D);
        prof_mark(h, 1);
        ba_schur_dmma<<<dim3(BA_SPLIT_W, n), 256, h->smem_schur, s>>>(C, D, h->ld_schur);
        prof_mark(h, 5);
        ba_pair_gram1<<<dim3((C.K * (C.K - 1) + 7) / 8, n), 256, 0, s>>>(C, D);
        prof_mark(h, 3);
        ba_export<<<g_nn, 256, 0, s>>>(C, D);
        ba_signal<<<1, 32, 0, s>>>(D, epoch);
        prof_mark(h, 7);
        ICG_CUDA(cudaStreamWaitEvent(s, h->ev_join, 0));
        prof_mark(h, 6);
        ba_reduce<<<g_nn, 256, 0, s>>>(C, D, epoch);
        prof_mark(h, 12);
        int rc = launch_solve_cam(h, n, epoch);
        if (rc != ICG_OK) return rc;
        prof_mark(h, 8);
        ba_step_lm<<<dim3(n, STEP_SLICES), SOLVE_THREADS, h->smem_step_lm, s>>>(C, D, epoch);
        prof_mark(h, 14);
        count_launch(9);
        if (it == max_num_iterations) break;
        ICG_CUDA(cudaEventRecord(h->ev_fork, s));
        ICG_CUDA(cudaStreamWaitEvent(h->stream_cam, h->ev_fork, 0));
        ba_cost_cam<<<n, h->cam_threads, h->smem_cam, h->stream_cam>>>(C, D, h->nblk_vis);
        ICG_CUDA(cudaEventRecord(h->ev_join, h->stream_cam));
        ba_cost<<<g_cost, 256, 0, s>>>(C, D, h->nblk_vis);
        ICG_CUDA(cudaStreamWaitEvent(s, h->ev_join, 0));
        prof_mark(h, 9);
        ba_exchange<<<(n + 63) / 64, 64, 0, s>>>(C, D, n, h->nblk_vis, epoch);
        prof_mark(h, 10);
        ba_accept_split<<<n, 128, 0, s>>>(C, D, epoch);
        prof_mark(h, 11);
        count_launch(4);
    }
    ICG_CHECK_LAUNCH();
    return ICG_OK;
}

static int restore_params(icg_ba *h) {
    const BaCaps &C = h->C;
    const BaDev &D = h->D;
    const int n = h->cur_windows;
    cudaStream_t s = h->stream;
    ICG_CUDA(cudaMemcpyAsync(D.pose, D.pose_0, sizeof(double) * (size_t) n * C.K * 7, cudaMemcpyDeviceToDevice, s));
    ICG_CUDA(cudaMemcpyAsync(D.mix, D.mix_0, sizeof(double) * (size_t) n * C.K * 9, cudaMemcpyDeviceToDevice, s));
    ICG_CUDA(cudaMemcpyAsync(D.ext, D.ext_0, sizeof(double) * (size_t) n * 8, cudaMemcpyDeviceToDevice, s));
    ICG_CUDA(cudaMemcpyAsync(D.rho, D.rho_0, sizeof(double) * (size_t) n * C.L, cudaMemcpyDeviceToDevice, s));
    // problem data the two-pass protocol mutates: factor activity, GNSS std (device-side pristine copies: the pinned staging buffers
    // receive the culled / re-weighted results in icg_ba_gvins_optimization_end), GNSS loss flag
    ICG_CUDA(cudaMemcpyAsync(D.f_active, D.f_active_0, (size_t) n * C.F, cudaMemcpyDeviceToDevice, s));
    ICG_CUDA(cudaMemcpyAsync(D.gnss_std, D.gnss_std_0, sizeof(double) * (size_t) n * C.G * 3, cudaMemcpyDeviceToDevice, s));
    ICG_CUDA(h->dims.up(s, n));
    return ICG_OK;
}

// enqueue the LM iterations for the uploaded problems (asynchronous; device-resident decisions)
int icg_ba_run(icg_ba *h, int max_num_iterations, int restart) {
    if (!h || h->cur_windows < 1 || max_num_iterations < 0) {
        set_error("icg_ba_run: no problems uploaded");
        return ICG_EINVAL;
    }
    ICG_CUDA(cudaSetDevice(h->device));
    const int n = h->cur_windows;
    if (restart) {
        int rc = restore_params(h);
        if (rc != ICG_OK) return rc;
    }
    ba_reset_state<<<(n + 127) / 128, 128, 0, h->stream>>>(h->D, nullptr, n, max_num_iterations);
    count_launch();
    return enqueue_lm(h, max_num_iterations);
}

// GVINS::gvinsOptimization (IG/ic_gvins.cc:1130-1239) entirely on the stream: pass 1 (N/4 iterations, Huber on GNSS),
// chi-square culling, pass 2 (N - N/4 iterations, GNSS without loss).  No host round trip between the passes.
int icg_ba_run_gvins(icg_ba *h, int num_iterations, int restart) {
    if (!h || h->cur_windows < 1 || num_iterations < 1) {
        set_error("icg_ba_run_gvins: no problems uploaded");
        return ICG_EINVAL;
    }
    ICG_CUDA(cudaSetDevice(h->device));
    const BaCaps &C = h->C;
    const int n = h->cur_windows;
    const int first = num_iterations / 4, second = num_iterations - first;  // IG/ic_gvins.cc:1131-1132
    if (restart) {
        int rc = restore_params(h);
        if (rc != ICG_OK) return rc;
    }
    cudaStream_t s = h->stream;
    ba_set_gnss_huber<<<(n + 127) / 128, 128, 0, s>>>(h->D, n, 1);
    ba_reset_state<<<(n + 127) / 128, 128, 0, s>>>(h->D, nullptr, n, first);
    count_launch(2);
    int rc = enqueue_lm(h, first);
    if (rc != ICG_OK) return rc;
    ICG_CUDA(cudaMemsetAsync(h->cull_counters.d, 0, sizeof(int) * 2 * (size_t) n, s));
    const dim3 g_cull((std::max(C.F, C.G) + 127) / 128, n);
    ba_chi2_cull<<<g_cull, 128, 0, s>>>(C, h->D, h->cull_counters.d);
    ba_set_gnss_huber<<<(n + 127) / 128, 128, 0, s>>>(h->D, n, 0);
    ba_reset_state<<<(n + 127) / 128, 128, 0, s>>>(h->D, h->st_save.d, n, second);
    count_launch(3);
    return enqueue_lm(h, second);
}

int icg_ba_download(icg_ba *h, int n, const icg_ba_problem *P, icg_ba_summary *summaries) {
    if (!h || n < 1 || n > h->cur_windows) {
        set_error("icg_ba_download: bad arguments");
        return ICG_EINVAL;
    }
    ICG_CUDA(cudaSetDevice(h->device));
    const BaCaps &C = h->C;
    cudaStream_t s = h->stream;
    ICG_CUDA(h->pose.down(s, (size_t) n * C.K * 7)); ICG_CUDA(h->mix.down(s, (size_t) n * C.K * 9)); ICG_CUDA(h->ext.down(s, (size_t) n * 8));
    ICG_CUDA(h->rho.down(s, (size_t) n * C.L)); ICG_CUDA(h->st.down(s, n));
    ICG_CUDA(cudaStreamSynchronize(s));
    if (h->D.S.split && icg_ba_shard_error(h) != 0) {
        set_error("icg_ba_download: a peer exchange of the split pipeline timed out (a rank of the shard group did not run the same sequence)");
        return ICG_ECUDA;
    }
    for (int w = 0; w < n; w++) {
        if (P) {
            const icg_ba_problem &p = P[w];
            memcpy(p.pose, h->pose.h + (size_t) w * C.K * 7, sizeof(double) * 7 * p.K);
            memcpy(p.mix, h->mix.h + (size_t) w * C.K * 9, sizeof(double) * 9 * p.K);
            memcpy(p.ext, h->ext.h + (size_t) w * 8, sizeof(double) * 8);
            if (p.L > 0) memcpy(p.invdepth, h->rho.h + (size_t) w * C.L, sizeof(double) * p.L);
        }
        if (summaries) {
            const LmState &st = h->st.h[w];
            icg_ba_summary &o = summaries[w];
            o.iterations = st.iter, o.num_successful_steps = st.n_success;
            o.termination = st.done == 2 ? 1 : st.done == 3 ? 2 : 0;
            o.reserved = 0;
            o.initial_cost = st.initial_cost, o.final_cost = st.x_cost, o.final_radius = st.radius;
        }
    }
    return ICG_OK;
}

int icg_ba_solve(icg_ba *h, int n_windows, const icg_ba_problem *problems, int max_num_iterations, icg_ba_summary *summaries) {
    int rc = icg_ba_upload(h, n_windows, problems);
    if (rc != ICG_OK) return rc;
    rc = icg_ba_run(h, max_num_iterations, 0);
    if (rc != ICG_OK) return rc;
    return icg_ba_download(h, n_windows, problems, summaries);
}

static void fill_summary(const LmState &st, icg_ba_summary &o) {
    o.iterations = st.iter, o.num_successful_steps = st.n_success;
    o.termination = st.done == 2 ? 1 : st.done == 3 ? 2 : 0;
    o.reserved = 0;
    o.initial_cost = st.initial_cost, o.final_cost = st.x_cost, o.final_radius = st.radius;
}

int icg_ba_gvins_optimization_begin(icg_ba *h, int n_windows, const icg_ba_problem *problems, int num_iterations) {
    int rc = icg_ba_upload(h, n_windows, problems);
    if (rc != ICG_OK) return rc;
    return icg_ba_run_gvins(h, num_iterations, 0);
}

int icg_ba_gvins_optimization_end(icg_ba *h, int n_windows, const icg_ba_problem *problems, icg_ba_summary *summaries, int32_t *culled) {
    if (!h || !problems || n_windows < 1 || n_windows > h->cur_windows) {
        set_error("icg_ba_gvins_optimization_end: bad arguments");
        return ICG_EINVAL;
    }
    ICG_CUDA(cudaSetDevice(h->device));
    const BaCaps &C = h->C;
    cudaStream_t s = h->stream;
    ICG_CUDA(h->st_save.down(s, n_windows));
    ICG_CUDA(h->cull_counters.down(s, 2 * (size_t) n_windows));
    ICG_CUDA(h->f_active.down(s, (size_t) n_windows * C.F));
    ICG_CUDA(h->gnss_std.down(s, (size_t) n_windows * C.G * 3));
    std::vector<icg_ba_summary> second(n_windows);
    int rc = icg_ba_download(h, n_windows, problems, second.data());
    if (rc != ICG_OK) return rc;
    for (int w = 0; w < n_windows; w++) {
        const icg_ba_problem &p = problems[w];
        // the reference mutates gnss->std in place and removes residual blocks from the problem: mirror both
        if (p.f_active) memcpy(const_cast<uint8_t *>(p.f_active), h->f_active.h + (size_t) w * C.F, p.F);
        if (p.n_gnss) memcpy(const_cast<double *>(p.gnss_std), h->gnss_std.h + (size_t) w * C.G * 3, sizeof(double) * 3 * p.n_gnss);
        if (summaries) {
            fill_summary(h->st_save.h[w], summaries[2 * w]);
            summaries[2 * w + 1] = second[w];
        }
        if (culled) culled[2 * w] = h->cull_counters.h[2 * w], culled[2 * w + 1] = h->cull_counters.h[2 * w + 1];
    }
    return ICG_OK;
}

int icg_ba_gvins_optimization(icg_ba *h, int n_windows, const icg_ba_problem *problems, int num_iterations, icg_ba_summary *summaries,
                              int32_t *culled) {
    int rc = icg_ba_gvins_optimization_begin(h, n_windows, problems, num_iterations);
    if (rc != ICG_OK) return rc;
    return icg_ba_gvins_optimization_end(h, n_windows, problems, summaries, culled);
}

// ---- marginalization (B10)
static int marg_alloc(icg_ba *h) {
    if (h->marg_ready) return ICG_OK;
    const BaCaps &C = h->C;
    MargDev &M = h->M;
    const size_t NW = C.NW;
    M.rcap = C.N, M.mcap = 15 * C.K + C.L, M.n0cap = C.N + C.L;
    if (M.mcap > 512) {
        set_error("icg_ba_marginalize: max_K=%d / max_L=%d exceed the Jacobi kernel's 512-row limit", C.K, C.L);
        return ICG_EUNSUPPORTED;
    }
    M.map_stride = MARG_MAP_HDR + 2 * C.K + C.L;
    if (h->marg_map.alloc(NW * M.map_stride) != ICG_OK || h->marg_oJ0.alloc(NW * (size_t) M.rcap * M.rcap) != ICG_OK || h->marg_oe0.alloc(NW * M.rcap) != ICG_OK ||
        h->marg_oHp.alloc(NW * (size_t) M.rcap * M.rcap) != ICG_OK || h->marg_obp.alloc(NW * M.rcap) != ICG_OK) {
        set_error("icg_ba_marginalize: workspace allocation failed");
        return ICG_ENOMEM;
    }
    M.map = h->marg_map.d, M.J0 = h->marg_oJ0.d, M.e0 = h->marg_oe0.d, M.Hp = h->marg_oHp.d, M.bp = h->marg_obp.d;
    int rc = ICG_OK;
    double *fl = nullptr;
#define DM(ptr, count) \
    if (rc == ICG_OK) rc = dmalloc(h, &ptr, count);
    DM(M.H0, NW * (size_t) M.n0cap * M.n0cap) DM(M.b0, NW * M.n0cap) DM(M.G1, NW * (size_t) M.mcap * M.mcap) DM(M.V1, NW * (size_t) M.mcap * M.mcap)
    DM(M.G2, NW * (size_t) M.rcap * M.rcap) DM(M.V2, NW * (size_t) M.rcap * M.rcap) DM(M.lam1, NW * M.mcap) DM(M.lam2, NW * M.rcap)
    DM(M.Z, NW * (size_t) M.mcap * (M.rcap + 1)) DM(fl, NW * 2)
#undef DM
    if (rc != ICG_OK) return rc;
    M.flags = (int *) fl;
    const size_t smem = sizeof(double) * (8 * 480 + 2 * (size_t) C.R) + sizeof(int) * (size_t) C.R + 64;
    ICG_CUDA(raise_dynamic_smem((const void *) marg_assemble, (size_t) (smem)));
    h->marg_ready = true;
    return ICG_OK;
}

static int marginalize_body(icg_ba *h, int n_windows, const icg_ba_problem *problems, const int32_t *num_marg, icg_ba_prior *out, bool resident) {
    if (!h || !problems || !num_marg || !out || n_windows < 1 || n_windows > h->C.NW) {
        set_error("icg_ba_marginalize: bad arguments");
        return ICG_EINVAL;
    }
    if (h->D.world > 1) {
        set_error("icg_ba_marginalize: not available on a landmark-sharded handle");
        return ICG_EUNSUPPORTED;
    }
    int rc = ICG_OK;
    if (resident) {
        // the windows of the last upload / solve are still on the device (parameters at their optimised values, factor activity and GNSS
        // weights as the two-pass solve left them): `problems` is read for the structure and for x0 only
        if (h->cur_windows != n_windows) {
            set_error("icg_ba_marginalize_resident: the handle holds %d uploaded windows, the call names %d", h->cur_windows, n_windows);
            return ICG_EINVAL;
        }
        ICG_CUDA(cudaSetDevice(h->device));
    } else {
        rc = icg_ba_upload(h, n_windows, problems);
        if (rc != ICG_OK) return rc;
    }
    rc = marg_alloc(h);
    if (rc != ICG_OK) return rc;
    const BaCaps &C = h->C;
    MargDev &M = h->M;
    const int n = n_windows;
    // ---- updateParameterBlocksIndex (marginalization_info.h:228-251) on the host: structure only.  The reference iterates
    //      unordered_maps (implementation-defined order inside each group); here: marginalized = [pose_k, mix_k (k < num_marg),
    //      landmarks ascending], remained = [pose_k, mix_k (k >= num_marg, only blocks some factor touches), ext, td].
    for (int w = 0; w < n; w++) {
        const icg_ba_problem &p = problems[w];
        const int nm = num_marg[w];
        icg_ba_prior &o = out[w];
        if (nm < 1 || nm >= p.K || !o.block_type || !o.block_node || !o.x0 || !o.J0 || !o.e0 || o.rcap < 15 * (p.K - nm) + 7) {
            set_error("icg_ba_marginalize: window %d: num_marg=%d out of range or output arrays missing / too small (rcap=%d)", w, nm, o.rcap);
            return ICG_EINVAL;
        }
        int *map = h->marg_map.h + (size_t) w * M.map_stride;
        int *pose_col = map + MARG_MAP_HDR, *mix_col = pose_col + C.K, *lm_col = mix_col + C.K;
        std::vector<char> tp(p.K, 0), tm(p.K, 0), tl(p.L, 0);
        bool any_vis = false;
        for (int f = 0; f < p.F; f++) {
            if ((p.f_active && !p.f_active[f]) || p.f_ref[f] >= nm) continue;
            tl[p.f_lm[f]] = 1, tp[p.f_obs[f]] = 1, any_vis = true;
        }
        bool has_ext = any_vis, has_td = any_vis;
        // a block exists in the marginalization problem only if some factor touches it (MarginalizationInfo::addResidualBlockInfo,
        // marginalization_info.h:103-121): removed nodes without any factor get no columns
        for (int f = 0; f < p.F; f++)
            if (!(p.f_active && !p.f_active[f]) && p.f_ref[f] < nm) tp[p.f_ref[f]] = 1;
        for (int k = 0; k < nm && k < p.n_imu; k++) tp[k] = tm[k] = tp[k + 1] = tm[k + 1] = 1;  // factor k joins node k and node k + 1
        for (int g = 0; g < p.n_gnss; g++)
            if (p.gnss_node[g] < nm) tp[p.gnss_node[g]] = 1;
        if (p.has_pose_prior) tp[0] = 1;
        if (p.has_mix_prior) tm[0] = 1;
        for (int b = 0; b < p.marg_nblocks && p.marg_r > 0; b++) {
            const int t = p.marg_block_type[b], nd = p.marg_block_node[b];
            if (t == 0) tp[nd] = 1;
            else if (t == 1) tm[nd] = 1;
            else if (t == 2) has_ext = true;
            else has_td = true;
        }
        int idx = 0;
        for (int k = 0; k < C.K; k++) pose_col[k] = mix_col[k] = -1;
        for (int k = 0; k < nm; k++) {
            if (tp[k]) pose_col[k] = idx, idx += 6;
            if (tm[k]) mix_col[k] = idx, idx += 9;
        }
        for (int l = 0; l < C.L; l++) lm_col[l] = -1;
        for (int l = 0; l < p.L; l++)
            if (tl[l]) lm_col[l] = idx++;
        const int m = idx;
        int nb = 0, xo = 0;
        for (int k = nm; k < p.K; k++) {
            if (tp[k]) pose_col[k] = idx, idx += 6, o.block_type[nb] = 0, o.block_node[nb++] = k - nm, xo += 7;
            if (tm[k]) mix_col[k] = idx, idx += 9, o.block_type[nb] = 1, o.block_node[nb++] = k - nm, xo += 9;
        }
        int ext_col = -1, td_col = -1;
        if (has_ext) ext_col = idx, idx += 6, o.block_type[nb] = 2, o.block_node[nb++] = 0, xo += 7;
        if (has_td) td_col = idx, idx += 1, o.block_type[nb] = 3, o.block_node[nb++] = 0, xo += 1;
        // a reprojection factor always carries ext and td columns; give them (unused) columns when only camera factors exist
        if (ext_col < 0) ext_col = 0;
        if (td_col < 0) td_col = 0;
        map[0] = m, map[1] = idx - m, map[2] = idx, map[3] = nm, map[4] = ext_col, map[5] = td_col, map[6] = map[7] = 0;
        o.m = m, o.r = idx - m, o.nblocks = nb;
    }
    cudaStream_t s = h->stream;
    ICG_CUDA(h->marg_map.up(s, (size_t) n * M.map_stride));
    const BaDev &D = h->D;
    const size_t smem = sizeof(double) * (8 * 480 + 2 * (size_t) C.R) + sizeof(int) * (size_t) C.R + 64;
    marg_prepare<<<(n + 127) / 128, 128, 0, s>>>(D, M, n, 0);
    ba_lin_vis<<<dim3(C.NVB - 2, n), 128, LV_SMEM, s>>>(C, D);
    ba_pair_gram1<<<dim3((C.K * (C.K - 1) + 7) / 8, n), 256, 0, s>>>(C, D);
    marg_assemble<<<n, 256, smem, s>>>(C, D, M);
    // eigendecompositions: on-chip cluster-pair kernel when every block of the batch fits (n <= MARG_PAIR_MAXN), global-memory kernel otherwise
    int max_m = 0, max_r = 0;
    for (int w = 0; w < n; w++) max_m = std::max(max_m, out[w].m), max_r = std::max(max_r, out[w].r);
    auto jacobi = [&](int which, int nmax) -> int {
        if (nmax <= MARG_CTA_MAXN && !getenv("ICG_MARG_GLOBAL_JACOBI") && !getenv("ICG_MARG_PAIR_JACOBI")) {
            const size_t smem = sizeof(double) * 2 * (size_t) nmax * nmax;
            ICG_CUDA(raise_dynamic_smem((const void *) marg_jacobi_cta, smem));
            marg_jacobi_cta<<<n, MARG_CTA_THREADS, smem, s>>>(M, which);
        } else if (nmax <= MARG_PAIR_MAXN && !getenv("ICG_MARG_GLOBAL_JACOBI")) {
            const size_t smem = sizeof(double) * ((size_t) nmax * nmax + 2 * (size_t) (nmax + 2));
            cudaLaunchConfig_t cfg;
            memset(&cfg, 0, sizeof(cfg));
            cfg.gridDim = dim3((unsigned) (2 * n)), cfg.blockDim = dim3(MARG_THREADS), cfg.dynamicSmemBytes = smem, cfg.stream = s;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = 2, at[0].val.clusterDim.y = 1, at[0].val.clusterDim.z = 1;
            cfg.attrs = at, cfg.numAttrs = 1;
            ICG_CUDA(raise_dynamic_smem((const void *) marg_jacobi_pair, (size_t) (smem)));
            ICG_CUDA(cudaLaunchKernelEx(&cfg, marg_jacobi_pair, M, which));
        } else {
            marg_jacobi<<<n, MARG_THREADS, 0, s>>>(M, which);
        }
        return ICG_OK;
    };
    rc = jacobi(0, max_m);
    if (rc != ICG_OK) return rc;
    marg_schur<<<n, MARG_THREADS, 0, s>>>(M);
    rc = jacobi(1, max_r);
    if (rc != ICG_OK) return rc;
    marg_finish<<<n, MARG_THREADS, 0, s>>>(M);
    marg_prepare<<<(n + 127) / 128, 128, 0, s>>>(D, M, n, 1);
    ICG_CHECK_LAUNCH();
    count_launch(10);
    // D2H: every window's r x r result sits at the start of its rcap^2 slot -- move the used prefix of each slot only (one strided copy)
    {
        const size_t pitch = sizeof(double) * (size_t) M.rcap * M.rcap, used = sizeof(double) * (size_t) max_r * max_r;
        bool want_Hp = false;
        for (int w = 0; w < n; w++) want_Hp = want_Hp || out[w].Hp != nullptr;
        if (used) ICG_CUDA(cudaMemcpy2DAsync(h->marg_oJ0.h, pitch, h->marg_oJ0.d, pitch, used, (size_t) n, cudaMemcpyDeviceToHost, s));
        ICG_CUDA(h->marg_oe0.down(s, (size_t) n * M.rcap));
        if (want_Hp && used) ICG_CUDA(cudaMemcpy2DAsync(h->marg_oHp.h, pitch, h->marg_oHp.d, pitch, used, (size_t) n, cudaMemcpyDeviceToHost, s));
        ICG_CUDA(h->marg_obp.down(s, (size_t) n * M.rcap));
    }
    ICG_CUDA(cudaStreamSynchronize(s));
    auto write_back = [&](int w) {
        const icg_ba_problem &p = problems[w];
        icg_ba_prior &o = out[w];
        const int nm = num_marg[w], r = o.r;
        // preMarginalization copies the parameter data of every block: x0 of the remained blocks (marginalization_info.h:270-283)
        int xo = 0;
        for (int b = 0; b < o.nblocks; b++) {
            const int t = o.block_type[b], nd = o.block_node[b] + nm;
            const double *src = t == 0 ? p.pose + 7 * nd : t == 1 ? p.mix + 9 * nd : t == 2 ? p.ext : p.ext + 7;
            const int gs = t == 1 ? 9 : t == 3 ? 1 : 7;
            memcpy(o.x0 + xo, src, sizeof(double) * gs);
            xo += gs;
        }
        if (o.m <= 0) return;
        memcpy(o.J0, h->marg_oJ0.h + (size_t) w * M.rcap * M.rcap, sizeof(double) * (size_t) r * r);
        memcpy(o.e0, h->marg_oe0.h + (size_t) w * M.rcap, sizeof(double) * r);
        if (o.Hp) memcpy(o.Hp, h->marg_oHp.h + (size_t) w * M.rcap * M.rcap, sizeof(double) * (size_t) r * r);
        if (o.bp) memcpy(o.bp, h->marg_obp.h + (size_t) w * M.rcap, sizeof(double) * r);
    };
    {   // the copies into the caller's arrays are memcpy-bound (r^2 doubles per window): a few host threads, like the packing of icg_ba_upload
        const int nthreads = std::max(1, std::min({n / 8, 8, (int) std::thread::hardware_concurrency()}));
        auto worker = [&](int t) {
            for (int w = t; w < n; w += nthreads) write_back(w);
        };
        std::vector<std::thread> th;
        for (int t = 1; t < nthreads; t++) th.emplace_back(worker, t);
        worker(0);
        for (auto &x : th) x.join();
    }
    return ICG_OK;
}

int icg_ba_marginalize(icg_ba *h, int n_windows, const icg_ba_problem *problems, const int32_t *num_marg, icg_ba_prior *out) {
    return marginalize_body(h, n_windows, problems, num_marg, out, false);
}

int icg_ba_marginalize_resident(icg_ba *h, int n_windows, const icg_ba_problem *problems, const int32_t *num_marg, icg_ba_prior *out) {
    return marginalize_body(h, n_windows, problems, num_marg, out, true);
}

// ---- post-solve outlier culling (updateParametersFromOptimizer + gvinsOutlierCulling, kernel in ba_cull.cu)
static size_t cull_layout(int n, size_t Ft, size_t Lt, size_t Kt, CullLaunch &A) {  // byte offsets of the sections (ba_cull.cuh); returns the end
    auto al = [](size_t x) { return (x + 15) & ~(size_t) 15; };
    size_t o = 0;
    A.o_win = o, o = al(o + n * sizeof(CullWin));
    A.o_fkp = o, o = al(o + Ft * 2 * sizeof(float));
    A.o_lkp = o, o = al(o + Lt * 2 * sizeof(float));
    A.o_lnode = o, o = al(o + Lt * sizeof(int));
    A.o_lpos = o, o = al(o + Lt * sizeof(int));
    A.o_wout = o, o = al(o + n * sizeof(CullWinOut));
    A.o_fout = o, o = al(o + Ft);
    A.o_lrout = o, o = al(o + Lt);
    A.o_lout = o, o = al(o + Lt);
    A.o_cam = o, o = al(o + Kt * 12 * sizeof(double));
    A.o_depth = o, o = al(o + Lt * sizeof(double));
    A.o_pos = o, o = al(o + Lt * 3 * sizeof(double));
    return o;
}

int icg_ba_outlier_culling_resident(icg_ba *h, int n_windows, const icg_ba_problem *problems, const icg_ba_cull_input *in, icg_ba_cull_output *out) {
    if (!h || !problems || !in || !out || n_windows < 1) {
        set_error("icg_ba_outlier_culling_resident: bad arguments");
        return ICG_EINVAL;
    }
    if (h->D.world > 1) {
        set_error("icg_ba_outlier_culling_resident: not available on a landmark-sharded handle");
        return ICG_EUNSUPPORTED;
    }
    if (h->cur_windows != n_windows) {
        set_error("icg_ba_outlier_culling_resident: the handle holds %d uploaded windows, the call names %d", h->cur_windows, n_windows);
        return ICG_EINVAL;
    }
    const BaCaps &C = h->C;
    const int n = n_windows;
    // ---- argument checks (nothing is launched on failure)
    size_t Ft = 0, Lt = 0, Kt = 0;
    int max_L = 0;
    for (int w = 0; w < n; w++) {
        const icg_ba_problem &p = problems[w];
        const icg_ba_cull_input &c = in[w];
        const icg_ba_cull_output &o = out[w];
        const WinDims &d = h->dims.h[w];
        if (p.K != d.K || p.L != d.L || p.F != d.F) {
            set_error("icg_ba_outlier_culling_resident: window %d is not the uploaded one (K=%d L=%d F=%d, uploaded %d %d %d)", w, p.K, p.L, p.F, d.K, d.L, d.F);
            return ICG_EINVAL;
        }
        if ((p.F > 0 && (!p.f_lm || !p.f_ref || !p.f_active || !c.f_kp || !o.f_outlier)) ||
            (p.L > 0 && (!c.lm_ref_kp || !c.lm_ref_node || !c.lm_ref_pos || !o.lm_ref_outlier || !o.lm_outlier)) || !(c.reprojection_error_std > 0)) {
            set_error("icg_ba_outlier_culling_resident: window %d: a required array is NULL or reprojection_error_std <= 0", w);
            return ICG_EINVAL;
        }
        const int *off = h->lm_off.h + (size_t) w * (C.L + 1);
        for (int l = 0; l < p.L; l++) {
            if (c.lm_ref_node[l] < 0 || c.lm_ref_node[l] >= p.K || c.lm_ref_pos[l] < 0 || c.lm_ref_pos[l] > off[l + 1] - off[l]) {
                set_error("icg_ba_outlier_culling_resident: window %d landmark %d: lm_ref_node %d / lm_ref_pos %d out of range (%d factors)", w, l, c.lm_ref_node[l],
                          c.lm_ref_pos[l], off[l + 1] - off[l]);
                return ICG_EINVAL;
            }
        }
        for (int f = 0; f < p.F; f++) {
            if (p.f_ref[f] != c.lm_ref_node[p.f_lm[f]]) {
                set_error("icg_ba_outlier_culling_resident: window %d factor %d: f_ref %d differs from the landmark's reference node %d", w, f, p.f_ref[f],
                          c.lm_ref_node[p.f_lm[f]]);
                return ICG_EINVAL;
            }
        }
        Ft += p.F, Lt += p.L, Kt += p.K, max_L = std::max(max_L, p.L);
    }
    ICG_CUDA(cudaSetDevice(h->device));
    CullLaunch A;
    if (!h->cull_buf.h) {
        const size_t cap = cull_layout(C.NW, (size_t) C.NW * C.F, (size_t) C.NW * C.L, (size_t) C.NW * C.K, A);
        if (h->cull_buf.alloc(cap) != ICG_OK) {
            h->cull_buf.release();
            set_error("icg_ba_outlier_culling_resident: staging allocation failed");
            return ICG_ENOMEM;
        }
    }
    const size_t end = cull_layout(n, Ft, Lt, Kt, A);
    // ---- pack the inputs (+ zeroed per-window output records: the counters start at zero)
    unsigned char *hb = h->cull_buf.h;
    {
        size_t f0 = 0, l0 = 0, k0 = 0;
        for (int w = 0; w < n; w++) {
            const icg_ba_problem &p = problems[w];
            const icg_ba_cull_input &c = in[w];
            CullWin &W = ((CullWin *) (hb + A.o_win))[w];
            W.cam = c.cam, W.reproj_std = c.reprojection_error_std;
            memcpy(W.R_bc, c.R_bc, sizeof(W.R_bc)), memcpy(W.t_bc, c.t_bc, sizeof(W.t_bc));
            W.estimate_extrinsic = c.estimate_extrinsic != 0, W.K = p.K, W.L = p.L, W.F = p.F;
            W.f0 = (int) f0, W.l0 = (int) l0, W.k0 = (int) k0, W.pad = 0;
            if (p.F) memcpy(hb + A.o_fkp + f0 * 8, c.f_kp, (size_t) p.F * 8);
            if (p.L) {
                memcpy(hb + A.o_lkp + l0 * 8, c.lm_ref_kp, (size_t) p.L * 8);
                memcpy(hb + A.o_lnode + l0 * 4, c.lm_ref_node, (size_t) p.L * 4);
                memcpy(hb + A.o_lpos + l0 * 4, c.lm_ref_pos, (size_t) p.L * 4);
            }
            f0 += p.F, l0 += p.L, k0 += p.K;
        }
        memset(hb + A.o_wout, 0, n * sizeof(CullWinOut));
    }
    const BaDev &D = h->D;
    A.pose = D.pose, A.ext = D.ext, A.rho = D.rho, A.lm_off = D.lm_off, A.f_meta_s = D.f_meta_s, A.f_active = D.f_active;
    A.capK = C.K, A.capL = C.L, A.capF = C.F, A.buf = h->cull_buf.d;
    size_t d2h_end = A.o_cam;  // the D2H stops after the last section some window asked for
    for (int w = 0; w < n; w++) {
        if (out[w].lm_pos) d2h_end = std::max(d2h_end, end);
        else if (out[w].lm_depth) d2h_end = std::max(d2h_end, A.o_pos);
        else if (out[w].cam_pose) d2h_end = std::max(d2h_end, A.o_depth);
    }
    cudaStream_t s = h->stream;
    ICG_CUDA(cudaMemcpyAsync(h->cull_buf.d, hb, A.o_wout + n * sizeof(CullWinOut), cudaMemcpyHostToDevice, s));
    ICG_CUDA(launch_outlier_cull(A, n, max_L, s));
    ICG_CUDA(cudaMemcpyAsync(hb + A.o_wout, h->cull_buf.d + A.o_wout, d2h_end - A.o_wout, cudaMemcpyDeviceToHost, s));
    ICG_CUDA(cudaStreamSynchronize(s));
    // ---- results into the caller's arrays; f_active of the problems mirrors the device copy
    size_t f0 = 0, l0 = 0, k0 = 0;
    for (int w = 0; w < n; w++) {
        const icg_ba_problem &p = problems[w];
        icg_ba_cull_output &o = out[w];
        const CullWinOut &WO = ((const CullWinOut *) (hb + A.o_wout))[w];
        o.ext_updated = WO.ext_updated;
        memcpy(o.counts, WO.counts, sizeof(o.counts)), memcpy(o.R_bc, WO.R_bc, sizeof(o.R_bc)), memcpy(o.t_bc, WO.t_bc, sizeof(o.t_bc));
        const uint8_t *fo = hb + A.o_fout + f0, *lo = hb + A.o_lout + l0;
        if (p.F) memcpy(o.f_outlier, fo, p.F);
        if (p.L) memcpy(o.lm_ref_outlier, hb + A.o_lrout + l0, p.L), memcpy(o.lm_outlier, lo, p.L);
        if (o.cam_pose) memcpy(o.cam_pose, hb + A.o_cam + k0 * 96, (size_t) p.K * 96);
        if (o.lm_depth && p.L) memcpy(o.lm_depth, hb + A.o_depth + l0 * 8, (size_t) p.L * 8);
        if (o.lm_pos && p.L) memcpy(o.lm_pos, hb + A.o_pos + l0 * 24, (size_t) p.L * 24);
        uint8_t *act = const_cast<uint8_t *>(p.f_active);
        for (int f = 0; f < p.F; f++) act[f] = (uint8_t) (!fo[f] && !lo[p.f_lm[f]]);
        f0 += p.F, l0 += p.L, k0 += p.K;
    }
    return ICG_OK;
}

// ---- landmark shards over peer memory (transport "p2p")
struct ShardBlob {  // what a rank publishes to the others (ICG_SHARD_BLOB_BYTES)
    uint64_t magic, pid, ptr, doubles;
    int32_t rank, world, device, pad;
    cudaIpcMemHandle_t ipc;
};
static_assert(sizeof(ShardBlob) <= ICG_SHARD_BLOB_BYTES, "ShardBlob size");

int icg_ba_shard_export(icg_ba *h, int rank, int world, uint8_t *blob) {
    if (!h || !blob) {
        set_error("icg_ba_shard_export: bad arguments");
        return ICG_EINVAL;
    }
    int rc = split_setup(h, rank, world);
    if (rc != ICG_OK) return rc;
    ShardBlob b;
    memset(&b, 0, sizeof(b));
    b.magic = 0x49434753484152ull, b.pid = (uint64_t) getpid(), b.ptr = (uint64_t) (uintptr_t) h->xbuf, b.doubles = h->xbuf_doubles;
    b.rank = rank, b.world = world, b.device = h->device;
    if (world > 1) ICG_CUDA(cudaIpcGetMemHandle(&b.ipc, h->xbuf));
    memset(blob, 0, ICG_SHARD_BLOB_BYTES);
    memcpy(blob, &b, sizeof(b));
    return ICG_OK;
}

int icg_ba_shard_connect(icg_ba *h, const uint8_t *blobs) {
    if (!h || !blobs || !h->D.S.split) {
        set_error("icg_ba_shard_connect: call icg_ba_shard_export first");
        return ICG_EINVAL;
    }
    ICG_CUDA(cudaSetDevice(h->device));
    const int world = h->D.world, rank = h->D.rank;
    for (int r = 0; r < world; r++) {
        ShardBlob b;
        memcpy(&b, blobs + (size_t) r * ICG_SHARD_BLOB_BYTES, sizeof(b));
        if (b.magic != 0x49434753484152ull || b.rank != r || b.world != world || b.doubles != h->xbuf_doubles) {
            set_error("icg_ba_shard_connect: blob %d does not describe rank %d of %d with the same window capacity", r, r, world);
            return ICG_EINVAL;
        }
        if (r == rank) continue;
        if (b.pid == (uint64_t) getpid()) {  // same process (several handles driven by one host process): plain device pointers
            if (b.device != h->device) {
                int can = 0;
                ICG_CUDA(cudaDeviceCanAccessPeer(&can, h->device, b.device));
                if (!can) {
                    set_error("icg_ba_shard_connect: device %d cannot access device %d", h->device, b.device);
                    return ICG_EUNSUPPORTED;
                }
                cudaError_t e = cudaDeviceEnablePeerAccess(b.device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) ICG_CUDA(e);
                cudaGetLastError();
            }
            h->D.S.peer[r] = (double *) (uintptr_t) b.ptr;
        } else {  // one process per GPU: map the peer's buffer through CUDA IPC (NVLink peer memory)
            void *p = nullptr;
            ICG_CUDA(cudaIpcOpenMemHandle(&p, b.ipc, cudaIpcMemLazyEnablePeerAccess));
            h->ipc_opened[r] = p;
            h->D.S.peer[r] = (double *) p;
        }
    }
    return ICG_OK;
}

int icg_ba_shard_error(icg_ba *h) {
    if (!h || !h->D.S.split) return 0;
    int e = 0;
    cudaSetDevice(h->device);
    if (cudaMemcpy(&e, h->D.S.err, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    return e;
}

int icg_ba_sync(icg_ba *h) {
    if (!h) return ICG_EINVAL;
    ICG_CUDA(cudaSetDevice(h->device));
    ICG_CUDA(cudaStreamSynchronize(h->stream));
    prof_collect(h);
    return ICG_OK;
}

int icg_ba_residual_costs(icg_ba *h, const icg_ba_problem *problem, double *reproj_cost, double *gnss_cost) {
    if (!h || !problem) {
        set_error("icg_ba_residual_costs: bad arguments");
        return ICG_EINVAL;
    }
    int rc = icg_ba_upload(h, 1, problem);
    if (rc != ICG_OK) return rc;
    const int F = problem->F, G = problem->n_gnss;
    double *d_out;
    ICG_CUDA(cudaMalloc(&d_out, sizeof(double) * (size_t) (F + G + 1)));
    const int nthreads = std::max(F, G);
    if (nthreads > 0) {
        ba_residual_costs_kernel<<<(nthreads + 127) / 128, 128, 0, h->stream>>>(h->C, h->D, d_out, d_out + F);
        count_launch();
    }
    std::vector<double> host(F + G + 1);
    ICG_CUDA(cudaMemcpyAsync(host.data(), d_out, sizeof(double) * (size_t) (F + G), cudaMemcpyDeviceToHost, h->stream));
    ICG_CUDA(cudaStreamSynchronize(h->stream));
    cudaFree(d_out);
    if (reproj_cost) memcpy(reproj_cost, host.data(), sizeof(double) * F);
    if (gnss_cost) memcpy(gnss_cost, host.data() + F, sizeof(double) * G);
    return ICG_OK;
}

int icg_ba_reproj_evaluate(icg_ba *h, const double *pose0, const double *pose1, const double *ext, const double *invdepth, const double *td,
                           const double *c14, double std_, double *residuals, double **jacobians) {
    if (!h || !pose0 || !pose1 || !ext || !invdepth || !td || !c14 || !residuals) {
        set_error("icg_ba_reproj_evaluate: bad arguments");
        return ICG_EINVAL;
    }
    ICG_CUDA(cudaSetDevice(h->device));
    double *in = h->scratch.h;
    memcpy(in, pose0, 56), memcpy(in + 7, pose1, 56), memcpy(in + 14, ext, 56);
    in[21] = 0, in[22] = *invdepth, in[23] = *td;
    memcpy(in + 24, c14, 112);
    in[38] = std_;
    ICG_CUDA(cudaMemcpyAsync(h->scratch.d, in, sizeof(double) * 40, cudaMemcpyHostToDevice, h->stream));
    ba_reproj_eval_kernel<<<1, 1, 0, h->stream>>>(h->scratch.d, h->scratch.d + 64);
    count_launch();
    ICG_CUDA(cudaMemcpyAsync(h->scratch.h + 64, h->scratch.d + 64, sizeof(double) * 48, cudaMemcpyDeviceToHost, h->stream));
    ICG_CUDA(cudaStreamSynchronize(h->stream));
    const double *o = h->scratch.h + 64;
    residuals[0] = o[0], residuals[1] = o[1];
    if (jacobians) {
        for (int b = 0; b < 3; b++)
            if (jacobians[b]) memcpy(jacobians[b], o + 2 + 14 * b, sizeof(double) * 14);
        if (jacobians[3]) jacobians[3][0] = o[44], jacobians[3][1] = o[45];
        if (jacobians[4]) jacobians[4][0] = o[46], jacobians[4][1] = o[47];
    }
    return ICG_OK;
}

int icg_ba_imu_evaluate(icg_ba *h, const double *blob, const double *pose0, const double *mix0, const double *pose1, const double *mix1,
                        double *residuals, double **jacobians) {
    if (!h || !blob || !pose0 || !mix0 || !pose1 || !mix1 || !residuals) {
        set_error("icg_ba_imu_evaluate: bad arguments");
        return ICG_EINVAL;
    }
    ICG_CUDA(cudaSetDevice(h->device));
    double *in = h->scratch.h;
    memcpy(in, pose0, 56), memcpy(in + 7, mix0, 72), memcpy(in + 16, pose1, 56), memcpy(in + 23, mix1, 72);
    if (!host_imu_sqrt_info(blob + 252, in + 32)) {
        set_error("icg_ba_imu_evaluate: covariance is not positive definite");
        return ICG_EINVAL;
    }
    double *d_blob;
    ICG_CUDA(cudaMalloc(&d_blob, sizeof(double) * (ICG_IMU_BLOB_DOUBLES + 480)));
    ICG_CUDA(cudaMemcpyAsync(d_blob, blob, sizeof(double) * ICG_IMU_BLOB_DOUBLES, cudaMemcpyHostToDevice, h->stream));
    ICG_CUDA(cudaMemcpyAsync(h->scratch.d, in, sizeof(double) * (32 + 225), cudaMemcpyHostToDevice, h->stream));
    ba_imu_eval_kernel<<<1, 32, 0, h->stream>>>(d_blob, h->scratch.d + 32, h->scratch.d, d_blob + ICG_IMU_BLOB_DOUBLES);
    count_launch();
    std::vector<double> out(465);
    ICG_CUDA(cudaMemcpyAsync(out.data(), d_blob + ICG_IMU_BLOB_DOUBLES, sizeof(double) * 465, cudaMemcpyDeviceToHost, h->stream));
    ICG_CUDA(cudaStreamSynchronize(h->stream));
    cudaFree(d_blob);
    memcpy(residuals, out.data(), sizeof(double) * 15);
    if (jacobians) {
        // local 15x30 [pose0 6 | mix0 9 | pose1 6 | mix1 9] -> global row-major 15x7, 15x9, 15x7, 15x9
        const double *J = out.data() + 15;
        const int c0[4] = {0, 6, 15, 21}, ls[4] = {6, 9, 6, 9}, gs[4] = {7, 9, 7, 9};
        for (int b = 0; b < 4; b++) {
            if (!jacobians[b]) continue;
            for (int r = 0; r < 15; r++)
                for (int c = 0; c < gs[b]; c++) jacobians[b][r * gs[b] + c] = c < ls[b] ? J[r * 30 + c0[b] + c] : 0.0;
        }
    }
    return ICG_OK;
}

// host helper of the small single-factor seams: upload `nin` doubles, run, download `nout` doubles (through the handle's scratch buffers)
static int small_factor_eval(icg_ba *h, int kind, const double *in, int nin, double *out, int nout) {
    ICG_CUDA(cudaSetDevice(h->device));
    memcpy(h->scratch.h, in, sizeof(double) * nin);
    ICG_CUDA(cudaMemcpyAsync(h->scratch.d, h->scratch.h, sizeof(double) * nin, cudaMemcpyHostToDevice, h->stream));
    ba_small_factor_eval_kernel<<<1, 1, 0, h->stream>>>(kind, h->scratch.d, h->scratch.d + 128);
    count_launch();
    ICG_CUDA(cudaMemcpyAsync(h->scratch.h + 128, h->scratch.d + 128, sizeof(double) * nout, cudaMemcpyDeviceToHost, h->stream));
    ICG_CUDA(cudaStreamSynchronize(h->stream));
    memcpy(out, h->scratch.h + 128, sizeof(double) * nout);
    return ICG_OK;
}

int icg_ba_gnss_evaluate(icg_ba *h, const double *pose, const double *blh, const double *std3, const double *lever, double *residuals, double **jacobians) {
    if (!h || !pose || !blh || !std3 || !lever || !residuals) {
        set_error("icg_ba_gnss_evaluate: bad arguments");
        return ICG_EINVAL;
    }
    double in[16], out[21];
    memcpy(in, pose, 56), memcpy(in + 7, blh, 24), memcpy(in + 10, std3, 24), memcpy(in + 13, lever, 24);
    int rc = small_factor_eval(h, 0, in, 16, out, 21);
    if (rc != ICG_OK) return rc;
    memcpy(residuals, out, 24);
    if (jacobians && jacobians[0])  // global 3x7 row-major; the quaternion-w column is zero (gnss_factor.h:60-68)
        for (int r = 0; r < 3; r++)
            for (int c = 0; c < 7; c++) jacobians[0][r * 7 + c] = c < 6 ? out[3 + r * 6 + c] : 0.0;
    return ICG_OK;
}

int icg_ba_pose_prior_evaluate(icg_ba *h, const double *pose, const double *prior7, const double *std6, double *residuals, double **jacobians) {
    if (!h || !pose || !prior7 || !std6 || !residuals) {
        set_error("icg_ba_pose_prior_evaluate: bad arguments");
        return ICG_EINVAL;
    }
    double in[20], out[42];
    memcpy(in, pose, 56), memcpy(in + 7, prior7, 56);
    for (int k = 0; k < 6; k++) in[14 + k] = 1.0 / std6[k];
    int rc = small_factor_eval(h, 1, in, 20, out, 42);
    if (rc != ICG_OK) return rc;
    memcpy(residuals, out, 48);
    if (jacobians && jacobians[0])
        for (int r = 0; r < 6; r++)
            for (int c = 0; c < 7; c++) jacobians[0][r * 7 + c] = c < 6 ? out[6 + r * 6 + c] : 0.0;
    return ICG_OK;
}

int icg_ba_mix_prior_evaluate(icg_ba *h, const double *mix, const double *prior9, const double *std9, double *residuals, double **jacobians) {
    if (!h || !mix || !prior9 || !std9 || !residuals) {
        set_error("icg_ba_mix_prior_evaluate: bad arguments");
        return ICG_EINVAL;
    }
    double in[27], out[18];
    memcpy(in, mix, 72), memcpy(in + 9, prior9, 72), memcpy(in + 18, std9, 72);
    int rc = small_factor_eval(h, 2, in, 27, out, 18);
    if (rc != ICG_OK) return rc;
    memcpy(residuals, out, 72);
    if (jacobians && jacobians[0]) {
        memset(jacobians[0], 0, sizeof(double) * 81);
        for (int k = 0; k < 9; k++) jacobians[0][k * 9 + k] = out[9 + k];
    }
    return ICG_OK;
}

int icg_ba_imu_error_evaluate(icg_ba *h, const double *mix, double *residuals, double **jacobians) {
    if (!h || !mix || !residuals) {
        set_error("icg_ba_imu_error_evaluate: bad arguments");
        return ICG_EINVAL;
    }
    double out[12];
    int rc = small_factor_eval(h, 3, mix, 9, out, 12);
    if (rc != ICG_OK) return rc;
    memcpy(residuals, out, 48);
    if (jacobians && jacobians[0]) {  // 6x9: rows 0..2 on bg (columns 3..5), rows 3..5 on ba (columns 6..8)
        memset(jacobians[0], 0, sizeof(double) * 54);
        for (int k = 0; k < 3; k++) jacobians[0][k * 9 + 3 + k] = out[6 + k], jacobians[0][(3 + k) * 9 + 6 + k] = out[9 + k];
    }
    return ICG_OK;
}

int icg_ba_marg_factor_evaluate(icg_ba *h, int r, int nblocks, const int32_t *block_type, const double *const *parameters, const double *x0,
                                const double *J0, const double *e0, double *residuals, double **jacobians) {
    if (!h || r < 1 || nblocks < 1 || !block_type || !parameters || !x0 || !J0 || !e0 || !residuals) {
        set_error("icg_ba_marg_factor_evaluate: bad arguments");
        return ICG_EINVAL;
    }
    ICG_CUDA(cudaSetDevice(h->device));
    int tot = 0, cols = 0;
    for (int b = 0; b < nblocks; b++) {
        const int t = block_type[b];
        if (t < 0 || t > 3 || !parameters[b]) {
            set_error("icg_ba_marg_factor_evaluate: block %d invalid", b);
            return ICG_EINVAL;
        }
        tot += t == 1 ? 9 : t == 3 ? 1 : 7, cols += t == 1 ? 9 : t == 3 ? 1 : 6;
    }
    if (cols != r) {
        set_error("icg_ba_marg_factor_evaluate: the blocks give %d local columns, r = %d", cols, r);
        return ICG_EINVAL;
    }
    const size_t nin = 2 + (size_t) nblocks + 2 * (size_t) tot + r + (size_t) r * r;
    std::vector<double> in(nin);
    in[0] = r, in[1] = nblocks;
    for (int b = 0; b < nblocks; b++) in[2 + b] = block_type[b];
    double *px = in.data() + 2 + nblocks;
    int xo = 0;
    for (int b = 0; b < nblocks; b++) {
        const int g = block_type[b] == 1 ? 9 : block_type[b] == 3 ? 1 : 7;
        memcpy(px + xo, parameters[b], sizeof(double) * g);
        xo += g;
    }
    memcpy(px + tot, x0, sizeof(double) * tot);
    memcpy(px + 2 * tot, e0, sizeof(double) * r);
    memcpy(px + 2 * tot + r, J0, sizeof(double) * (size_t) r * r);
    double *d = nullptr;
    ICG_CUDA(cudaMalloc(&d, sizeof(double) * (nin + r)));
    ICG_CUDA(cudaMemcpyAsync(d, in.data(), sizeof(double) * nin, cudaMemcpyHostToDevice, h->stream));
    ba_marg_factor_eval_kernel<<<1, 256, sizeof(double) * r, h->stream>>>(d, d + nin);
    count_launch();
    ICG_CUDA(cudaMemcpyAsync(residuals, d + nin, sizeof(double) * r, cudaMemcpyDeviceToHost, h->stream));
    ICG_CUDA(cudaStreamSynchronize(h->stream));
    cudaFree(d);
    if (jacobians) {  // the factor is linear: d e / d (block b) = J0[:, columns of b], quaternion-w column zero (marginalization_factor.h:84-97)
        int col = 0;
        for (int b = 0; b < nblocks; b++) {
            const int t = block_type[b], g = t == 1 ? 9 : t == 3 ? 1 : 7, l = t == 1 ? 9 : t == 3 ? 1 : 6;
            if (jacobians[b])
                for (int i = 0; i < r; i++)
                    for (int c = 0; c < g; c++) jacobians[b][(size_t) i * g + c] = c < l ? J0[(size_t) i * r + col + c] : 0.0;
            col += l;
        }
    }
    return ICG_OK;
}

}  // extern "C"
