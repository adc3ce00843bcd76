// ba_cull.cuh -- interface between the host side of icg_ba_outlier_culling_resident (ba.cu) and its kernel (ba_cull.cu, built with
// -fmad=false).  GVINS::updateParametersFromOptimizer + GVINS::gvinsOutlierCulling (IG/ic_gvins.cc:1299-1389, 1035-1128) on the windows a
// handle holds.
//
// One staging buffer per handle, in two parts that meet in the middle:
//   inputs  [CullWin x n | f_kp float2 x sum F | lm_ref_kp float2 x sum L | lm_ref_node int x sum L | lm_ref_pos int x sum L]
//   outputs [CullWinOut x n | f_outlier u8 x sum F | lm_ref_outlier u8 x sum L | lm_outlier u8 x sum L | cam_pose 12 x sum K | lm_depth x sum L | lm_pos 3 x sum L]
// One H2D copy moves the inputs together with the zeroed CullWinOut records (the per-window counters start at zero without a memset);
// one D2H copy brings back the outputs from CullWinOut up to the last section the caller asked for.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/icgvins_b200.h"

namespace icg {

struct CullWin {          // per-window inputs
    icg_camera cam;
    double reproj_std;
    double R_bc[9], t_bc[3];  // gate baseline
    int32_t estimate_extrinsic, K, L, F;
    int32_t f0, l0, k0, pad;  // offsets of the window's factors / landmarks / nodes in the concatenated sections
};
struct CullWinOut {       // per-window outputs (128 bytes)
    int32_t counts[5];    // outliers_[0], outliers_[1], num1, num2, num3
    int32_t ext_updated, pad[2];
    double R_bc[9], t_bc[3];
};

struct CullLaunch {
    const double *pose, *ext, *rho;  // the handle's current parameters (capacity-strided by window)
    const int *lm_off, *f_meta_s;    // landmark CSR of the factor records; per record (landmark, reference node, observing node, factor id)
    uint8_t *f_active;               // by factor id, capacity-strided; rewritten for every factor of the window
    int capK, capL, capF;
    unsigned char *buf;              // device staging buffer
    size_t o_win, o_fkp, o_lkp, o_lnode, o_lpos;              // input sections (bytes)
    size_t o_wout, o_fout, o_lrout, o_lout, o_cam, o_depth, o_pos;  // output sections (bytes)
};

constexpr int CULL_WARPS = 8;  // landmarks per CTA (one warp each)

// one launch: grid (ceil(max L / CULL_WARPS), n windows)
cudaError_t launch_outlier_cull(const CullLaunch &A, int n, int max_L, cudaStream_t s);

}  // namespace icg
