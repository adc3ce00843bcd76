// ba_cull.cu -- post-solve outlier culling on the device: GVINS::updateParametersFromOptimizer (IG/ic_gvins.cc:1299-1389) followed by
// GVINS::gvinsOutlierCulling (:1035-1128) for every window of a batch in one launch (host side: icg_ba_outlier_culling_resident, ba.cu).
// Built with -fmad=false: cam2pixel rounds a double to float, so a contracted multiply-add could move a key point across a decision.
#include "ba_cull.cuh"
#include "common.cuh"
#include "geom_core.cuh"

namespace icg {

// CTA = CULL_WARPS landmarks of one window (blockIdx.y).  Thread 0 applies the extrinsic gate, one thread per node turns the solved states into
// camera poses (kept in shared memory; CTA 0 of the window also writes both out).  Then one warp per landmark: lane i evaluates observation i
// of the landmark's observations() sequence (the reference observation at lm_ref_pos, the factors in ascending factor id around it; at most
// K <= 32 observations).  A ballot finds the first bad reference observation -- the reference loop breaks there, so the lanes behind it are
// not evaluated -- and the surviving errors are summed in sequence order (std::accumulate) by shuffles.  Counters are integer atomics.
__global__ void __launch_bounds__(CULL_WARPS * 32) ba_outlier_cull(CullLaunch A) {
    __shared__ double sR[32 * 9], sT[32 * 3], gR[9], gT[3];
    const int w = blockIdx.y;
    const CullWin &W = ((const CullWin *) (A.buf + A.o_win))[w];
    CullWinOut &WO = ((CullWinOut *) (A.buf + A.o_wout))[w];
    if (threadIdx.x == 0) {
        double R[9], t[3];
        for (int i = 0; i < 9; i++) R[i] = W.R_bc[i];
        for (int i = 0; i < 3; i++) t[i] = W.t_bc[i];
        const int upd = W.estimate_extrinsic ? gc::extrinsic_gate(A.ext + (size_t) w * 8, R, t) : 0;
        for (int i = 0; i < 9; i++) gR[i] = R[i];
        for (int i = 0; i < 3; i++) gT[i] = t[i];
        if (blockIdx.x == 0) {
            WO.ext_updated = upd;
            for (int i = 0; i < 9; i++) WO.R_bc[i] = R[i];
            for (int i = 0; i < 3; i++) WO.t_bc[i] = t[i];
        }
    }
    __syncthreads();
    if ((int) threadIdx.x < W.K) {
        const int k = threadIdx.x;
        gc::camera_pose(A.pose + ((size_t) w * A.capK + k) * 7, gR, gT, sR + 9 * k, sT + 3 * k);
        if (blockIdx.x == 0) {
            double *cp = (double *) (A.buf + A.o_cam) + (size_t) (W.k0 + k) * 12;
            for (int i = 0; i < 9; i++) cp[i] = sR[9 * k + i];
            for (int i = 0; i < 3; i++) cp[9 + i] = sT[3 * k + i];
        }
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, l = blockIdx.x * CULL_WARPS + (threadIdx.x >> 5);
    if (l >= W.L) return;  // warp-uniform
    const int lg = W.l0 + l;
    const float2 *fkp = (const float2 *) (A.buf + A.o_fkp) + W.f0;
    const float2 rkp = ((const float2 *) (A.buf + A.o_lkp))[lg];
    const int ref_node = ((const int *) (A.buf + A.o_lnode))[lg], ref_pos = ((const int *) (A.buf + A.o_lpos))[lg];
    const int *off = A.lm_off + (size_t) w * (A.capL + 1);
    const int s0 = off[l], nobs = off[l + 1] - s0 + 1;
    double pos[3], depth;
    gc::mappoint_position(W.cam, sR + 9 * ref_node, sT + 3 * ref_node, rkp.x, rkp.y, A.rho[(size_t) w * A.capL + l], pos, depth);
    bool bad = false;
    double err = 0.0;
    int f = -1;
    if (lane < nobs) {
        int node;
        float2 kp;
        if (lane == ref_pos) {
            node = ref_node, kp = rkp;
        } else {
            const int *m = A.f_meta_s + ((size_t) w * A.capF + s0 + (lane < ref_pos ? lane : lane - 1)) * 4;
            node = m[2], f = m[3], kp = fkp[f];
        }
        bad = !gc::good_to_track(W.cam, sR + 9 * node, sT + 3 * node, pos, kp.x, kp.y, W.reproj_std * 3.0, err);
    }
    const unsigned badm = __ballot_sync(0xffffffffu, bad);
    const bool ref_bad = (badm >> ref_pos) & 1u;
    const int last = ref_bad ? ref_pos : nobs - 1;             // the loop breaks at a bad reference observation
    const unsigned evalm = (unsigned) ((2ull << last) - 1ull);  // evaluated sequence positions 0..last
    const unsigned flagged = badm & evalm, goodm = evalm & ~badm;
    const int n_err = __popc(goodm);
    const double mine = (goodm >> lane) & 1u ? err : 0.0;
    double sum = 0.0;
    for (int i = 0; i <= last; i++) {
        const double e = __shfl_sync(0xffffffffu, mine, i);
        if ((goodm >> i) & 1u) sum = sum + e;
    }
    const int num1 = ref_bad, num2 = n_err < 2, num3 = !num2 && sum / (double) n_err > W.reproj_std;
    const int bits = num1 | num2 << 1 | num3 << 2;
    if (f >= 0) {
        const int fo = (flagged >> lane) & 1u;
        (A.buf + A.o_fout)[W.f0 + f] = (unsigned char) fo;
        A.f_active[(size_t) w * A.capF + f] = (uint8_t) (!fo && !bits);
    }
    if (lane == 0) {
        (A.buf + A.o_lrout)[lg] = (unsigned char) num1;
        (A.buf + A.o_lout)[lg] = (unsigned char) bits;
        ((double *) (A.buf + A.o_depth))[lg] = depth;
        double *pp = (double *) (A.buf + A.o_pos) + (size_t) lg * 3;
        pp[0] = pos[0], pp[1] = pos[1], pp[2] = pos[2];
        const int n_feat = __popc(flagged & ~(1u << ref_pos)), n_map = num1 + (num2 | num3);
        if (n_map) atomicAdd(&WO.counts[0], n_map);
        if (n_feat) atomicAdd(&WO.counts[1], n_feat);
        if (num1) atomicAdd(&WO.counts[2], 1);
        if (num2) atomicAdd(&WO.counts[3], 1);
        if (num3) atomicAdd(&WO.counts[4], 1);
    }
}

cudaError_t launch_outlier_cull(const CullLaunch &A, int n, int max_L, cudaStream_t s) {
    const dim3 grid((unsigned) ((max_L + CULL_WARPS - 1) / CULL_WARPS > 0 ? (max_L + CULL_WARPS - 1) / CULL_WARPS : 1), (unsigned) n);
    ba_outlier_cull<<<grid, CULL_WARPS * 32, 0, s>>>(A);
    count_launch();
    return cudaGetLastError();
}

}  // namespace icg
