// ba_split.cuh -- the "split" LM pipeline of the window solve: large reduced systems (n = 15K + 7 beyond one CTA's shared memory, cfg 4)
// and landmark-sharded solves over the GPUs of one box (SURVEY.md 8e).  Included by ba.cu.
//
// One LM attempt, rank g of G (G = 1: everything is local), windows w = 0 .. W-1, owner(w) = w mod G:
//
//   every rank   ba_lin_vis / ba_schur_dmma / ba_pair_gram1     its landmark shard of every window (the kernels of the fused pipeline)
//   every rank   ba_export        packs [tri(H_vis - Schur) | diag H_vis | g_vis | W phi g_l | cost, sum rho^2, max |g_l|] of window w and
//                                 STORES it into the inbox of owner(w) -- peer memory over NVLink (P2P stores), slot [w / G][g]
//                ba_signal        release-flag "my partials of this epoch have landed" on every peer
//   owner        ba_reduce        waits for the G flags, sums the G slots in rank order (deterministic, identical regardless of arrival
//                                 order) into Hs = H_c + sum; the reduction is fused into the assembly of the solve's operand
//   owner        ba_solve_cam     thread-block CLUSTER per window: Jacobi scaling, LM diagonal, packed S in global memory (L2), blocked
//                                 Cholesky (DMMA panel updates spread over the cluster's CTAs, cluster barriers), blocked back-substitution;
//                                 broadcasts [header | camera step] into every rank's step buffer (P2P stores + per-window release flag)
//   every rank   ba_step_lm       waits for the window's flag; candidate camera blocks x (+) delta (redundantly, bit-identical), landmark
//                                 back-substitution + candidates of its own landmarks, its parts of the model cost change and step norm
//   every rank   ba_cost (+ ba_cost_cam on the owner)
//   every rank   ba_exchange      [model cost change, |step|^2, non-finite, candidate cost, sum rho^2] of its shard -> slot [w][g] of EVERY rank
//   every rank   ba_accept_split  waits for the G slots, sums them in rank order: identical inputs -> identical accept / reject, radius and
//                                 termination decisions on every rank, no broadcast of the LM state
//
// Three flag synchronisations per attempt, no collective library on the data path, no host round trip.  The flags are monotonically
// increasing epoch counters (one per LM attempt over the life of the handle); a consumer that does not see its flag within ~2 s raises the
// handle's device-side error word instead of hanging the GPU.
#pragma once
#include <cooperative_groups.h>

namespace icg {
namespace cg = cooperative_groups;

constexpr int SPLIT_CLUSTER = 4;      // CTAs per window in ba_solve_cam
constexpr int SPLIT_HDR = 16;         // header doubles of the step broadcast
constexpr int SPLIT_SCAL = 8;         // doubles per (window, rank) slot of the scalar exchange
constexpr int SPLIT_BS_ROWS = 32;     // rows per block of the blocked back-substitution

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// spin until *f >= epoch (flags only grow); ~2 s budget, then the error word is raised and the caller proceeds (results are discarded by
// the host, which reports ICG_ECUDA): a lost peer must not hang the GPU
__device__ __forceinline__ void wait_flag(const unsigned long long *f, unsigned long long epoch, int *err) {
    const long long t0 = clock64();
    while (ld_acquire_sys(f) < epoch) {
        if (clock64() - t0 > 4000000000ll) {
            atomicExch(err, 1);
            break;
        }
        __nanosleep(64);
    }
}

__device__ __forceinline__ double *x_inbox(const BaDev &D, int peer, int w, int from) {
    const ShardDev &S = D.S;
    return S.peer[peer] + S.off_inbox + ((size_t) (w / D.world) * D.world + from) * S.PK;
}
__device__ __forceinline__ double *x_bcast(const BaDev &D, int peer, int w) { return D.S.peer[peer] + D.S.off_bcast + (size_t) w * D.S.BS; }
__device__ __forceinline__ double *x_scal(const BaDev &D, int peer, int w, int from) {
    return D.S.peer[peer] + D.S.off_scal + ((size_t) w * D.world + from) * SPLIT_SCAL;
}
__device__ __forceinline__ unsigned long long *x_flagA(const BaDev &D, int peer, int from) {
    return (unsigned long long *) (D.S.peer[peer] + D.S.off_flagA) + from;
}
__device__ __forceinline__ unsigned long long *x_flagB(const BaDev &D, int peer, int w) {
    return (unsigned long long *) (D.S.peer[peer] + D.S.off_flagB) + w;
}
__device__ __forceinline__ unsigned long long *x_flagC(const BaDev &D, int peer, int w, int from) {
    return (unsigned long long *) (D.S.peer[peer] + D.S.off_flagC) + (size_t) w * D.world + from;
}
__device__ __forceinline__ int tri_idx(int A, int B, int ncv) { return A * ncv - A * (A - 1) / 2 + (B - A); }  // A <= B < ncv

// ------------------------------------------------------------------------------------------------ export (every rank)
// thread per entry (A <= B) of the symmetric (NCV+1)^2 matrix [H_vis g_vis; g_vis^T .]: gathers the per-pair Gram matrices (ba_hsum's job in the
// fused pipeline), subtracts the Schur partials and stores into the owner's inbox.  Block 0 of a window also reduces the scalars.
__global__ void __launch_bounds__(256) ba_export(BaCaps C, BaDev D) {
    __shared__ short s_slot[32 * 32];
    __shared__ double s_red[40];
    const int w = blockIdx.y, tid = threadIdx.x;
    const LmState &st = D.st[w];
    if (st.done) return;
    const WinDims dm = D.dims[w];
    const int K = dm.K, NCV = 6 * K + 7, nn = NCV + 1;
    if ((int) blockIdx.x * 256 >= nn * nn) return;
    const int owner = w % D.world;
    double *P = x_inbox(D, owner, w, D.rank);
    const int TRI = NCV * (NCV + 1) / 2;
    gram2_slots(C, D, w, K, s_slot);
    const int t = blockIdx.x * 256 + tid;
    if (t < nn * nn) {
        const int A = t / nn, B = t - A * nn;
        if (B >= A && A < NCV) {
            const double cj = gram2_entry(C, D, w, K, s_slot, A, B);
            const double *CWp = D.CW + (size_t) w * BA_SPLIT_W * C.NCA * C.NCA;
            double cw = 0;
#pragma unroll
            for (int k = 0; k < BA_SPLIT_W; k++) cw += CWp[(size_t) k * C.NCA * C.NCA + (size_t) B * C.NCA + A];
            if (B < NCV) {
                P[tri_idx(A, B, NCV)] = cj - cw;
                if (A == B) P[TRI + A] = cj;
            } else {
                P[TRI + NCV + A] = cj;       // g_vis
                P[TRI + 2 * NCV + A] = cw;   // W phi g_l
            }
        }
    }
    if (blockIdx.x != 0) return;
    double c = 0, q = 0, gm = 0;
    for (int f = tid; f < dm.F; f += 256) c += D.costf[(size_t) w * C.F + f];
    for (int l = tid; l < dm.L; l += 256) {
        const double r = D.rho[(size_t) w * C.L + l];
        q += r * r;
        gm = fmax(gm, fabs(D.gl[(size_t) w * C.L + l]));
    }
    c = block_sum(c, s_red);
    q = block_sum(q, s_red);
    gm = block_max(gm, s_red);
    if (tid == 0) P[TRI + 3 * NCV] = c, P[TRI + 3 * NCV + 1] = q, P[TRI + 3 * NCV + 2] = gm;
}

// everything this rank stored for `epoch` has been issued by earlier kernels of the stream: publish (one thread per peer)
__global__ void ba_signal(BaDev D, unsigned long long epoch) {
    const int q = threadIdx.x;
    if (q >= D.world) return;
    __threadfence_system();
    st_release_sys(x_flagA(D, q, D.rank), epoch);
}

// ------------------------------------------------------------------------------------------------ reduce (owner)
__global__ void __launch_bounds__(256) ba_reduce(BaCaps C, BaDev D, unsigned long long epoch) {
    const int w = blockIdx.y, tid = threadIdx.x;
    if (w % D.world != D.rank) return;
    if (D.st[w].done) return;
    const int K = D.dims[w].K, NCV = 6 * K + 7, nn = NCV + 1, TRI = NCV * (NCV + 1) / 2;
    if ((int) blockIdx.x * 256 >= nn * nn) return;
    if (tid < D.world) wait_flag(x_flagA(D, D.rank, tid), epoch, D.S.err);
    __syncthreads();
    const int t = blockIdx.x * 256 + tid;
    if (t >= nn * nn) return;
    const int A = t / nn, B = t - A * nn;  // same thread -> entry map as ba_export
    if (B < A) return;
    const double *P0 = x_inbox(D, D.rank, w, 0);
    const size_t PK = D.S.PK;
    auto rsum = [&](int e) {  // fixed rank order: identical on every run and on every rank count
        double s = 0;
        for (int r = 0; r < D.world; r++) s += __ldcg(P0 + (size_t) r * PK + e);
        return s;
    };
    double *rv = D.S.redv + (size_t) w * D.S.RV;
    if (A < NCV && B < NCV) {
        D.Hs[(size_t) w * C.NS * C.NS + (size_t) B * C.NS + A] = D.Hc[(size_t) w * C.NS * C.NS + (size_t) B * C.NS + A] + rsum(tri_idx(A, B, NCV));
        if (A == B) rv[A] = rsum(TRI + A);
    } else if (A < NCV) {  // B == NCV: the gradient column
        rv[NCV + A] = rsum(TRI + NCV + A);
        rv[2 * NCV + A] = rsum(TRI + 2 * NCV + A);
    } else {               // A == B == NCV: the scalars
        rv[3 * NCV] = rsum(TRI + 3 * NCV);
        rv[3 * NCV + 1] = rsum(TRI + 3 * NCV + 1);
        double m = 0;
        for (int r = 0; r < D.world; r++) m = fmax(m, __ldcg(P0 + (size_t) r * PK + TRI + 3 * NCV + 2));
        rv[3 * NCV + 2] = m;
    }
}

__host__ __device__ inline size_t split_S_stride(const BaCaps &C) { return (size_t) (C.N + 1) * (C.N + 2) / 2 + (size_t) C.NS; }

// ------------------------------------------------------------------------------------------------ solve_cam (owner, cluster per window)
// The camera-side half of ba_solve for systems that do not fit one CTA: S lives packed in global memory (L2-resident, written and read by all
// CTAs of the cluster between cluster barriers -- cluster.sync orders the global accesses at cluster scope and invalidates L1).
// Row i of the packed lower triangle starts at i (i + 1) / 2; the augmented row N carries the right-hand side.
__global__ void __launch_bounds__(SOLVE_THREADS) ba_solve_cam(BaCaps C, BaDev D, unsigned long long epoch, int stage_a) {
    extern __shared__ double sm[];
    cg::cluster_group cluster = cg::this_cluster();
    const int CL = (int) cluster.num_blocks(), cr = (int) cluster.block_rank();
    const int w = blockIdx.x / CL, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (w % D.world != D.rank) return;   // uniform over the cluster
    LmState &st = D.st[w];
    if (st.done) return;
    const WinDims dm = D.dims[w];
    const int K = dm.K, NCV = 6 * K + 7, N = 15 * K + 7, NR = N + 1;
    const int CT = CL * SOLVE_THREADS, ctid = cr * SOLVE_THREADS + tid, cwarp = ctid >> 5, ncwarps = CT / 32;
    // snapshot of the LM state (CTA 0 updates it after the first cluster barrier)
    const int f_first = st.first, f_fresh = st.fresh_lin, f_last = st.last_success, f_iter = st.iter, f_maxit = st.max_iter;
    const double radius = st.radius, cost_cam = st.cost_cam, gmax_old = st.gmax, xcost_old = st.x_cost, init_old = st.initial_cost;
    double *s_red = sm;                  // 40
    double *s_scale = s_red + 40;        // N
    double *s_g = s_scale + C.NS;        // N
    double *s_rhs = s_g + C.NS;          // N   rhs' then step'
    double *s_d2 = s_rhs + C.NS;         // N
    double *s_blk = s_d2 + C.NS;         // SPLIT_BS_ROWS x (NS + 1): row block of L for the back-substitution (CTA 0)
    double *S = D.Sglobal + (size_t) (w / D.world) * split_S_stride(C);  // one workspace per OWNED window: packed triangle | pivot reciprocals
    const double *Hc = D.Hc + (size_t) w * C.NS * C.NS, *gcam = D.gc + (size_t) w * C.NS, *Hs = D.Hs + (size_t) w * C.NS * C.NS;
    const double *rv = D.S.redv + (size_t) w * D.S.RV;   // [diag H_vis | g_vis | W phi g_l | cost, sum rho^2, max |g_l|]
    double *scale_c = D.scale_c + (size_t) w * C.NS;
    // ---- gradient, Jacobi scaling (first linearisation), LM diagonal, rhs: every CTA keeps its own copy (no DSMEM traffic)
    for (int a = tid; a < N; a += SOLVE_THREADS) {
        const double g = gcam[a] + (a < NCV ? rv[NCV + a] : 0.0);
        s_g[a] = g;
        const double h = Hc[(size_t) a * C.NS + a] + (a < NCV ? rv[a] : 0.0);
        const double sc = f_first ? 1.0 / (1.0 + sqrt(h)) : scale_c[a];
        s_scale[a] = sc;
        const double hs = sc * sc * h;
        s_d2[a] = fmin(fmax(hs, 1e-6), 1e32) / radius;
        s_rhs[a] = -sc * (g - (a < NCV ? rv[2 * NCV + a] : 0.0));
    }
    __syncthreads();
    double gmax_now = gmax_old, x_cost = xcost_old;
    if (f_fresh) {
        double gm = 0;
        for (int a = tid; a < N; a += SOLVE_THREADS) gm = fmax(gm, fabs(s_g[a]));
        gm = fmax(block_max(gm, s_red), rv[3 * NCV + 2]);
        gmax_now = gm;
        x_cost = rv[3 * NCV] + cost_cam;
    }
    int term = 0;
    if (f_iter >= f_maxit) term = 1;                               // NO_CONVERGENCE
    else if (f_last && gmax_now <= 1e-10) term = 2;                // gradient tolerance
    else if (f_last && radius <= 1e-32) term = 2;                  // min trust region radius
    cluster.sync();  // every CTA has read the state it needs
    if (cr == 0 && tid == 0) {
        st.x_cost = x_cost, st.gmax = gmax_now;
        if (f_first) st.initial_cost = x_cost;
        st.fresh_lin = 0, st.first = 0, st.need_lin = 0;
        if (term) st.done = term, st.step_valid = 0;
        else st.iter = f_iter + 1;
    }
    if (cr == 0 && f_first)
        for (int a = tid; a < N; a += SOLVE_THREADS) scale_c[a] = s_scale[a];
    double *BC = nullptr;
    if (term) {
        // broadcast the termination (header only) and leave
        if (cr == 0) {
            __syncthreads();
            for (int q = tid; q < D.world; q += SOLVE_THREADS) {
                BC = x_bcast(D, q, w);
                BC[0] = (double) term, BC[1] = 0.0, BC[2] = x_cost, BC[3] = gmax_now, BC[4] = f_first ? x_cost : init_old, BC[5] = 0.0;
                __threadfence_system();
                st_release_sys(x_flagB(D, q, w), epoch);
            }
        }
        return;
    }
    // ---- assemble S' = s H s + D^2 (packed lower, global), warp per row over the whole cluster
    for (int i = cwarp; i < N; i += ncwarps) {
        const double *src = (i < NCV ? Hs : Hc) + (size_t) i * C.NS;
        double *dst = S + (size_t) i * (i + 1) / 2;
        const double si = s_scale[i];
        for (int j = lane; j <= i; j += 32) {
            double v = si * s_scale[j] * src[j];
            if (i == j) v += s_d2[i];
            dst[j] = v;
        }
    }
    for (int a = ctid; a < N; a += CT) S[(size_t) N * (N + 1) / 2 + a] = s_rhs[a];
    cluster.sync();
    // ---- blocked left-looking Cholesky, 8 columns per step; panel update (DMMA) and row solves spread over the cluster.  Per panel:
    //   (0) every CTA stages the panel's B operand (rows J0 .. J0 + 7 of L, columns < J0) in its shared memory: one coalesced L2 sweep
    //       instead of a dependent L2 round trip per k-step and warp;
    //   (1) DMMA update of the 8-row tiles: A operands from L2, 64 columns (16 loads per lane) in flight per pass.  Cluster warp 0 takes the
    //       diagonal tile and FACTORS it straight away (registers), writes L_JJ back in place and the pivot reciprocals to dinv[] (a negative
    //       entry = breakdown), while the other 31 cluster warps update the tiles below;
    //   (2) cluster barrier; every row below is solved by its own thread against L_JJ / dinv read from L2; cluster barrier.
    // The round-2-start form read both DMMA operands from L2 four columns at a time and let all 1 024 threads factor the block redundantly
    // (each loading it from L2): 20 k cycles per panel, 392 us per launch at N = 307.
    double *dinvg = S + (size_t) (C.N + 1) * (C.N + 2) / 2;  // [NS] behind the capacity-sized triangle of this window's workspace
    double *s_b = s_blk;                                      // [8][ldbp]: aliases the back-substitution staging (used after the factorisation)
    const int ldbp = ((C.N + 15) / 16) * 16 + 8;              // = 8 mod 16 doubles: conflict-free fragment reads
    int fail = 0;
#ifdef ICG_BA_PHASE_CLOCKS
#define CAMS_CLK(k, t0)                                                                                             \
    if (D.clk && w == 0 && ctid == 0) atomicAdd(&D.clk[k], clock64() - (t0)), atomicAdd(&D.clk[8 + (k)], 1ull);
#define CAMS_NOW() clock64()
#else
#define CAMS_CLK(k, t0)
#define CAMS_NOW() 0ull
#endif
    const unsigned long long tc_all = CAMS_NOW();
    (void) tc_all;
    for (int J0 = 0; J0 < N; J0 += BA_CHOL_NB) {
        const int nb = min(BA_CHOL_NB, N - J0);
        const int g = lane >> 2, kk = lane & 3;
        const int ntile = (NR - J0 + 7) / 8;
        const unsigned long long tc0 = CAMS_NOW();
        (void) tc0;
        if (J0 > 0) {
            for (int e = tid; e < 8 * J0; e += SOLVE_THREADS) {
                const int r = e / J0, c = e - r * J0, row = J0 + r;
                s_b[r * ldbp + c] = row < NR ? S[(size_t) row * (row + 1) / 2 + c] : 0.0;
            }
            __syncthreads();
        }
        CAMS_CLK(0, tc0)  // staging of the B operand
        const unsigned long long tc1 = CAMS_NOW();
        (void) tc1;
        // one 8-row tile: S[rows, J0 : J0 + 8] -= L[rows, : J0] L[J0 : J0 + 8, : J0]^T.
        // stage_a (the launch gave every warp an 8 x ldbp shared-memory strip): the tile's A rows come in with 8-byte cp.async, ALL columns in
        // flight at once (one L2 round trip per tile; measured 2 k cycles per 64-column pass when the operand is read from L2 in the k loop),
        // then both DMMA operands are conflict-free shared-memory reads.  Without the strips (max_K beyond the shared-memory budget): 64 columns
        // (16 loads per lane) in flight per pass.
        auto tile_update = [&](int tI) {
            const int ia = J0 + 8 * tI + g;
            const bool oka = ia < NR;
            const double *ra = S + (oka ? (size_t) ia * (ia + 1) / 2 : 0);
            const double *sb = s_b + g * ldbp;
            double c0 = 0, c1 = 0, d0 = 0, d1 = 0, e0 = 0, e1 = 0, f0 = 0, f1 = 0;
            if (stage_a) {
                double *sw = s_b + 8 * ldbp + 64 + (size_t) warp * 8 * ldbp;  // this warp's strip (behind the B rows and the 8 x 8 hand-over buffer)
                __syncwarp();  // the strip's previous tile has been consumed
#pragma unroll 1
                for (int r = 0; r < 8; r++) {
                    const int row = J0 + 8 * tI + r;
                    if (row < NR) {
                        const double *src = S + (size_t) row * (row + 1) / 2;
                        const unsigned dst = (unsigned) __cvta_generic_to_shared(sw + r * ldbp);
                        for (int c = lane; c < J0; c += 32) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + 8u * c), "l"(src + c) : "memory");
                    }
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
                asm volatile("cp.async.wait_all;" ::: "memory");
                __syncwarp();
                const double *sa = sw + g * ldbp;
                int k0 = 0;
                for (; k0 + 16 <= J0; k0 += 16) {
                    const double a0 = oka ? sa[k0 + kk] : 0.0, a1 = oka ? sa[k0 + 4 + kk] : 0.0, a2 = oka ? sa[k0 + 8 + kk] : 0.0, a3 = oka ? sa[k0 + 12 + kk] : 0.0;
                    dmma884(c0, c1, a0, sb[k0 + kk]);
                    dmma884(d0, d1, a1, sb[k0 + 4 + kk]);
                    dmma884(e0, e1, a2, sb[k0 + 8 + kk]);
                    dmma884(f0, f1, a3, sb[k0 + 12 + kk]);
                }
                for (; k0 + 4 <= J0; k0 += 4) {
                    const double a0 = oka ? sa[k0 + kk] : 0.0;
                    dmma884(c0, c1, a0, sb[k0 + kk]);
                }
            } else {
                for (int k0 = 0; k0 < J0; k0 += 64) {
                    double a[16];
#pragma unroll
                    for (int u = 0; u < 16; u++) a[u] = (oka && k0 + 4 * u < J0) ? ra[k0 + 4 * u + kk] : 0.0;
#pragma unroll
                    for (int u = 0; u < 16; u += 4) {
                        if (k0 + 4 * u < J0) {  // J0 is a multiple of 8: k-steps come in pairs; zero-padded beyond J0
                            const double b0 = sb[k0 + 4 * u + kk], b1 = k0 + 4 * u + 4 < J0 ? sb[k0 + 4 * u + 4 + kk] : 0.0;
                            const double b2 = k0 + 4 * u + 8 < J0 ? sb[k0 + 4 * u + 8 + kk] : 0.0, b3 = k0 + 4 * u + 12 < J0 ? sb[k0 + 4 * u + 12 + kk] : 0.0;
                            dmma884(c0, c1, a[u], b0);
                            dmma884(d0, d1, a[u + 1], b1);
                            dmma884(e0, e1, a[u + 2], b2);
                            dmma884(f0, f1, a[u + 3], b3);
                        }
                    }
                }
            }
            c0 += d0 + (e0 + f0), c1 += d1 + (e1 + f1);
            if (oka) {
                const int ca = J0 + 2 * kk;
                double *ri = S + (size_t) ia * (ia + 1) / 2;
                if (ca < J0 + nb && ca <= ia) ri[ca] -= c0;
                if (ca + 1 < J0 + nb && ca + 1 <= ia) ri[ca + 1] -= c1;
            }
        };
        if (cwarp == 0) {
            // diagonal tile: its A operand IS the staged B operand (shared memory, no L2 round trip on the k loop); the block's current values are
            // fetched from L2 before the loop (they arrive while it runs), updated in registers and handed to the factorisation through a
            // 64-double shared buffer instead of a global write + read
            double *s_jj = s_b + 8 * ldbp;  // [8][8] behind the B rows
            {
                const int ia = J0 + g;
                const bool oka = ia < NR;
                const int ca = J0 + 2 * kk;
                double v0 = 0, v1 = 0;
                if (oka && ca <= ia && ca < J0 + nb) v0 = S[(size_t) ia * (ia + 1) / 2 + ca];
                if (oka && ca + 1 <= ia && ca + 1 < J0 + nb) v1 = S[(size_t) ia * (ia + 1) / 2 + ca + 1];
                if (J0 > 0) {
                    const double *sa = s_b + g * ldbp;
                    double c0 = 0, c1 = 0, d0 = 0, d1 = 0, e0 = 0, e1 = 0, f0 = 0, f1 = 0;
                    int k0 = 0;
                    for (; k0 + 16 <= J0; k0 += 16) {
                        const double x0 = sa[k0 + kk], x1 = sa[k0 + 4 + kk], x2 = sa[k0 + 8 + kk], x3 = sa[k0 + 12 + kk];
                        dmma884(c0, c1, x0, x0);
                        dmma884(d0, d1, x1, x1);
                        dmma884(e0, e1, x2, x2);
                        dmma884(f0, f1, x3, x3);
                    }
                    for (; k0 + 4 <= J0; k0 += 4) {
                        const double x0 = sa[k0 + kk];
                        dmma884(c0, c1, x0, x0);
                    }
                    v0 -= c0 + d0 + (e0 + f0), v1 -= c1 + d1 + (e1 + f1);
                }
                s_jj[g * 8 + 2 * kk] = v0, s_jj[g * 8 + 2 * kk + 1] = v1;
                if (oka && ia >= J0 + nb) {  // last panel (nb < 8): the tile also holds rows BELOW the block (the augmented rhs row): back to S
                    if (ca < J0 + nb) S[(size_t) ia * (ia + 1) / 2 + ca] = v0;
                    if (ca + 1 < J0 + nb) S[(size_t) ia * (ia + 1) / 2 + ca + 1] = v1;
                }
                __syncwarp();
            }
            double Ld[BA_CHOL_NB][BA_CHOL_NB], dinv[BA_CHOL_NB];
            bool bad = false;
#pragma unroll
            for (int a = 0; a < BA_CHOL_NB; a++)
#pragma unroll
                for (int b = 0; b < BA_CHOL_NB; b++) Ld[a][b] = (a < nb && b <= a) ? s_jj[a * 8 + b] : (a == b ? 1.0 : 0.0);
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
#pragma unroll
            for (int a2 = 0; a2 < BA_CHOL_NB; a2++) {  // statically indexed registers, one lane per store under a predicate (no switch on the lane)
                double *ri = S + (size_t) (J0 + a2) * (J0 + a2 + 1) / 2 + J0;
#pragma unroll
                for (int b = 0; b <= a2; b++)
                    if (lane == ((a2 * 8 + b) & 31) && a2 < nb) ri[b] = Ld[a2][b];
                if (lane == 8 + a2 && a2 < nb) dinvg[J0 + a2] = bad ? -1.0 : dinv[a2];
            }
            CAMS_CLK(1, tc1)  // cluster warp 0: diagonal tile + factorisation
        } else if (J0 > 0) {
            for (int tI = cwarp; tI < ntile; tI += ncwarps - 1) tile_update(tI);
        }
        cluster.sync();
        CAMS_CLK(2, tc1)  // tile updates + first cluster barrier
        const unsigned long long tc2 = CAMS_NOW();
        (void) tc2;
        fail = dinvg[J0] < 0.0;  // identical on every thread of the cluster
        if (fail) break;
        // rows below the block (incl. the augmented rhs row): solve against the factored block, one row per thread of the cluster
        for (int i = J0 + nb + ctid; i < NR; i += CT) {
            double *ri = S + (size_t) i * (i + 1) / 2 + J0;
            double x[BA_CHOL_NB], Lb[BA_CHOL_NB * (BA_CHOL_NB - 1) / 2], dv[BA_CHOL_NB];
#pragma unroll
            for (int c = 0; c < BA_CHOL_NB; c++) {
                x[c] = c < nb ? ri[c] : 0.0;
                dv[c] = c < nb ? dinvg[J0 + c] : 1.0;
#pragma unroll
                for (int k = 0; k < c; k++) Lb[c * (c - 1) / 2 + k] = c < nb ? S[(size_t) (J0 + c) * (J0 + c + 1) / 2 + J0 + k] : 0.0;
            }
#pragma unroll
            for (int c = 0; c < BA_CHOL_NB; c++) {
                double sum = x[c];
#pragma unroll
                for (int k = 0; k < c; k++) sum -= x[k] * Lb[c * (c - 1) / 2 + k];
                x[c] = sum * dv[c];
            }
#pragma unroll
            for (int c = 0; c < BA_CHOL_NB; c++)
                if (c < nb) ri[c] = x[c];
        }
        cluster.sync();
        CAMS_CLK(3, tc2)  // row solves + second cluster barrier
    }
    CAMS_CLK(4, tc_all)   // whole factorisation
    if (cr != 0) return;
    // ---- CTA 0: blocked backward substitution L^T x = y.  Blocks of SPLIT_BS_ROWS rows, last block first: the block's rows (all columns
    //      up to the diagonal) are staged in shared memory with one coalesced sweep; one warp solves the triangle, every thread then
    //      subtracts the block's contribution from the y entries above it.
    const bool valid = !fail;
    double *y = s_rhs;  // y = L^-1 rhs' sits in the augmented row
    __syncthreads();
    if (valid) {
        for (int a = tid; a < N; a += SOLVE_THREADS) y[a] = S[(size_t) N * (N + 1) / 2 + a];
        __syncthreads();
        const int ldb = C.NS + 1;
        for (int j1 = N; j1 > 0; j1 -= SPLIT_BS_ROWS) {
            const int j0 = max(0, j1 - SPLIT_BS_ROWS), nr = j1 - j0;
            for (int e = tid; e < nr * j1; e += SOLVE_THREADS) {
                const int r = e / j1, c = e - r * j1;
                const int row = j0 + r;
                s_blk[r * ldb + c] = c <= row ? S[(size_t) row * (row + 1) / 2 + c] : 0.0;
            }
            __syncthreads();
            if (warp == 0) {  // triangle: x_j = (y_j - sum_{i > j in block} L_ij x_i) / L_jj, j descending
                double xv = lane < nr ? y[j0 + lane] : 0.0;
                for (int r = nr - 1; r >= 0; r--) {
                    const double xj = __shfl_sync(0xffffffffu, xv, r) / s_blk[r * ldb + j0 + r];
                    if (lane == r) xv = xj;
                    if (lane < r) xv -= s_blk[r * ldb + j0 + lane] * xj;
                }
                if (lane < nr) y[j0 + lane] = xv;
            }
            __syncthreads();
            for (int c = tid; c < j0; c += SOLVE_THREADS) {
                double acc = y[c];
                for (int r = 0; r < nr; r++) acc -= s_blk[r * ldb + c] * y[j0 + r];
                y[c] = acc;
            }
            __syncthreads();
        }
    }
    // ---- camera part of the model cost change, broadcast of [header | delta = step' * scale]
    double part = 0;
    bool finite = true;
    if (valid)
        for (int a = tid; a < N; a += SOLVE_THREADS) {
            const double sp = y[a];
            finite = finite && isfinite(sp);
            part += -0.5 * sp * (s_scale[a] * s_g[a]) + 0.5 * s_d2[a] * sp * sp;
        }
    const double mcc = block_sum(part, s_red);
    const double nfin = block_sum(finite ? 0.0 : 1.0, s_red);
    for (int q = 0; q < D.world; q++) {
        BC = x_bcast(D, q, w);
        if (valid)
            for (int a = tid; a < N; a += SOLVE_THREADS) BC[SPLIT_HDR + a] = y[a] * s_scale[a];
        if (tid == 0) {
            BC[0] = 0.0, BC[1] = (valid && nfin == 0.0) ? 1.0 : 0.0, BC[2] = x_cost, BC[3] = gmax_now, BC[4] = f_first ? x_cost : init_old, BC[5] = mcc;
        }
    }
    __threadfence_system();
    __syncthreads();
    for (int q = tid; q < D.world; q += SOLVE_THREADS) st_release_sys(x_flagB(D, q, w), epoch);
}

// ------------------------------------------------------------------------------------------------ solve_cam, distributed-shared-memory form
// The same job as ba_solve_cam with the packed system RESIDENT IN THE CLUSTER'S SHARED MEMORY: nothing of the factorisation touches L2.
// (The L2 form above spends 15 k cycles per 8-column panel -- 2 cluster barriers, the B operand, the A strips and the factored block all
// fetched from L2 behind them; profiles/r2_ba_solve_cam_dsm.md.)
//
// Layout.  The (N + 1) x (N + 1) augmented lower triangle (row N = right-hand side) is cut into 8 x 8 tiles, each stored row-major (64 doubles:
// the DMMA C fragment of lane l is the 16 bytes at 2 l -- one conflict-free 128-bit access per lane).  Tile row T lives on CTA T mod 4; a CTA
// keeps the strictly-lower tiles (T, tc < T) of its tile rows.  The DIAGONAL tiles are replicated: every CTA keeps all of them and applies every
// update to them redundantly (bit-identical), so the 8 x 8 factorisation of a panel needs no hand-over between CTAs.
//
// Right-looking blocked Cholesky, ONE cluster barrier per panel:
//   (1) warp 0: Dg[J] -= P_J P_J^T (the previous panel's update of the tile it is about to factor), 8 x 8 factorisation in registers ->
//       L_JJ, reciprocal pivots; meanwhile warps 1,2,3,5,6,7 apply the previous panel's rank-8 update to the CTA's tiles and to the other
//       diagonal replicas: 2 DMMAs per tile, operands = the panel column P (all-gathered, below), k permuted so that a lane's two operand
//       values are adjacent (128-bit loads).  Warp 4 sits out: it shares warp 0's scheduler and FP64 pipe.
//   (2) block barrier; a thread per local row below the panel solves its 8 entries against L_JJ and STORES THE SOLVED ROW INTO THE PANEL-COLUMN
//       BUFFER OF ALL FOUR CTAs (distributed shared memory, fire-and-forget); P is double-buffered by panel parity.
//   (3) cluster barrier (the stores have landed); the right-hand-side row's entries of the panel are y = L^-1 rhs.
// Backward substitution L^T x = y, distributed: tile rows last to first; the owner of tile row T solves the 8 x 8 triangle (one warp), adds the
// row's contributions to its own partial sums for the columns on the left and pushes the partial sums of the next three tile rows (final by
// construction: its next own tile row is T - 4) to their owners' inboxes by st.async; the owner's inbox mbarrier counts the bytes, no cluster
// barrier per tile row.
constexpr int DSM_CL = 4;
static_assert(SOLVE_THREADS == 256 && DSM_CL == SPLIT_CLUSTER, "ba_solve_cam_dsm: warp r assembles row r of a tile row; one launch geometry for both forms");
__host__ __device__ inline int dsm_tile_off(int cr, int m) { return m * cr + 2 * m * (m - 1); }  // tiles ahead of local tile row m (T = cr + 4 m)
__host__ __device__ constexpr int dsm_ntiles(int NR) { return (NR + 7) / 8; }
__host__ inline size_t dsm_smem_doubles(const BaCaps &C) {
    const int nt = dsm_ntiles(C.N + 1);
    int mx = 0;
    for (int cr = 0; cr < DSM_CL; cr++) {
        int s = 0;
        for (int T = cr; T < nt; T += DSM_CL) s += T;
        mx = s > mx ? s : mx;
    }
    return 40 + 8 * (size_t) nt * 8 + 64 + 8 + 8 * DSM_CL + 8 + 8 + (size_t) nt * 64 * 3 + (size_t) mx * 64;
}

// ---- distributed-shared-memory plumbing: cluster addresses, mbarriers with transaction counts, asynchronous remote stores
__device__ __forceinline__ unsigned mapa_u32(unsigned addr, unsigned rank) {
    unsigned r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void dsm_mbar_init(unsigned bar, unsigned count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory"); }
__device__ __forceinline__ void dsm_mbar_arrive_local(unsigned bar) { asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
// arrive on a barrier of another CTA of the cluster and announce the bytes this CTA has sent towards it (st.async below completes them)
__device__ __forceinline__ void dsm_mbar_arrive_expect_tx_remote(unsigned bar_cluster, unsigned tx) {
    asm volatile("mbarrier.arrive.expect_tx.release.cluster.shared::cluster.b64 _, [%0], %1;" ::"r"(bar_cluster), "r"(tx) : "memory");
}
__device__ __forceinline__ void st_async_f64(unsigned dst_cluster, double a, unsigned bar_cluster) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.f64 [%0], %1, [%2];" ::"r"(dst_cluster), "d"(a), "r"(bar_cluster) : "memory");
}
__device__ __forceinline__ bool dsm_mbar_try_wait(unsigned bar, unsigned parity) {
    unsigned ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// bounded wait (~0.2 s): a protocol error raises the handle's error word and poisons the later waits of this CTA instead of hanging the GPU
__device__ __forceinline__ void dsm_mbar_wait(unsigned bar, unsigned parity, volatile int *s_dead, int *err) {
    if (dsm_mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!dsm_mbar_try_wait(bar, parity)) {
        if (*s_dead) return;
        if (clock64() - t0 > 400000000ll) {
            *s_dead = 1;
            atomicExch(err, 1);
            return;
        }
    }
}

// Hand-over forms, measured (profiles/r2_ba_solve_cam_dsm.md): the panel column is bound by the SM-to-SM bandwidth, and st.async + mbarriers
// were no cheaper there than plain stores + the cluster barrier; in the back-substitution chain the point-to-point form gains 15 %.
__global__ void __launch_bounds__(SOLVE_THREADS, 1) ba_solve_cam_dsm(BaCaps C, BaDev D, unsigned long long epoch) {
    extern __shared__ double sm[];
    cg::cluster_group cluster = cg::this_cluster();
    constexpr int CL = DSM_CL;
    const int cr = (int) cluster.block_rank();
    const int w = blockIdx.x / CL, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (w % D.world != D.rank) return;   // uniform over the cluster
    LmState &st = D.st[w];
    if (st.done) return;
    const WinDims dm = D.dims[w];
    const int K = dm.K, NCV = 6 * K + 7, N = 15 * K + 7, NR = N + 1;
    const int ntc = dsm_ntiles(C.N + 1), VL = ntc * 8;   // capacity: tiles per side, vector length
    const int nt = dsm_ntiles(NR), npan = (N + 7) / 8;   // this window: tile rows (incl. the rhs row), column panels
    const int Tn = N >> 3, rn = N & 7;                   // tile row / row in the tile of the augmented right-hand-side row
    const int f_first = st.first, f_fresh = st.fresh_lin, f_last = st.last_success, f_iter = st.iter, f_maxit = st.max_iter;
    const double radius = st.radius, cost_cam = st.cost_cam, gmax_old = st.gmax, xcost_old = st.x_cost, init_old = st.initial_cost;
    double *s_red = sm;                       // 40
    double *s_scale = s_red + 40;             // VL each
    double *s_g = s_scale + VL;
    double *s_rhs = s_g + VL;
    double *s_d2 = s_rhs + VL;
    double *s_y = s_d2 + VL;                  // y = L^-1 rhs'
    double *s_contrib = s_y + VL;             // back-substitution: this CTA's partial sums  sum_rows L[row][c] x[row]
    double *s_x = s_contrib + VL;             // the solution (complete on CTA 0)
    double *s_dinv = s_x + VL;                // reciprocal pivots (0 beyond N)
    double *s_Lf = s_dinv + VL;               // 64: the panel's factored diagonal block, identity-padded
    double *s_dv = s_Lf + 64;                 // 8: its reciprocal pivots
    double *s_inbox = s_dv + 8;               // [CL][8]
    double *s_xT = s_inbox + 8 * CL;          // 8
    int *s_fail = (int *) (s_xT + 8);         // [0] breakdown, [1] a bounded wait ran out; then the mbarrier (8 doubles reserved)
    unsigned long long *s_bar = (unsigned long long *) (s_xT + 12);  // the back-substitution inbox's mbarrier
    double *s_dg = s_xT + 16;                 // [ntc][64] replicated diagonal tiles
    double *s_P = s_dg + (size_t) ntc * 64;   // [2][ntc][64] panel column, by panel parity
    double *s_tiles = s_P + (size_t) 2 * ntc * 64;
    const double *Hc = D.Hc + (size_t) w * C.NS * C.NS, *gcam = D.gc + (size_t) w * C.NS, *Hs = D.Hs + (size_t) w * C.NS * C.NS;
    const double *rv = D.S.redv + (size_t) w * D.S.RV;   // [diag H_vis | g_vis | W phi g_l | cost, sum rho^2, max |g_l|]
    double *scale_c = D.scale_c + (size_t) w * C.NS;
    // ---- gradient, Jacobi scaling (first linearisation), LM diagonal, rhs: every CTA keeps its own copy
    for (int a = tid; a < VL; a += SOLVE_THREADS) {
        double g = 0, sc = 0, d2 = 0, rh = 0;
        if (a < N) {
            g = gcam[a] + (a < NCV ? rv[NCV + a] : 0.0);
            const double h = Hc[(size_t) a * C.NS + a] + (a < NCV ? rv[a] : 0.0);
            sc = f_first ? 1.0 / (1.0 + sqrt(h)) : scale_c[a];
            const double hs = sc * sc * h;
            d2 = fmin(fmax(hs, 1e-6), 1e32) / radius;
            rh = -sc * (g - (a < NCV ? rv[2 * NCV + a] : 0.0));
        }
        s_g[a] = g, s_scale[a] = sc, s_d2[a] = d2, s_rhs[a] = rh;
        s_y[a] = 0, s_contrib[a] = 0, s_x[a] = 0, s_dinv[a] = 0;
    }
    if (tid < 8 * CL) s_inbox[tid] = 0;
    if (tid == 0) {
        s_fail[0] = 0, s_fail[1] = 0;
        dsm_mbar_init(smem_u32(s_bar), CL - 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    double gmax_now = gmax_old, x_cost = xcost_old;
    if (f_fresh) {
        double gm = 0;
        for (int a = tid; a < N; a += SOLVE_THREADS) gm = fmax(gm, fabs(s_g[a]));
        gm = fmax(block_max(gm, s_red), rv[3 * NCV + 2]);
        gmax_now = gm;
        x_cost = rv[3 * NCV] + cost_cam;
    }
    int term = 0;
    if (f_iter >= f_maxit) term = 1;                               // NO_CONVERGENCE
    else if (f_last && gmax_now <= 1e-10) term = 2;                // gradient tolerance
    else if (f_last && radius <= 1e-32) term = 2;                  // min trust region radius
    cluster.sync();  // every CTA has read the state it needs (and is running: its shared memory and barriers may be used from now on)
    if (cr == 0 && tid == 0) {
        st.x_cost = x_cost, st.gmax = gmax_now;
        if (f_first) st.initial_cost = x_cost;
        st.fresh_lin = 0, st.first = 0, st.need_lin = 0;
        if (term) st.done = term, st.step_valid = 0;
        else st.iter = f_iter + 1;
    }
    if (cr == 0 && f_first)
        for (int a = tid; a < N; a += SOLVE_THREADS) scale_c[a] = s_scale[a];
    double *BC = nullptr;
    if (term) {
        if (cr == 0) {
            __syncthreads();
            for (int q = tid; q < D.world; q += SOLVE_THREADS) {
                BC = x_bcast(D, q, w);
                BC[0] = (double) term, BC[1] = 0.0, BC[2] = x_cost, BC[3] = gmax_now, BC[4] = f_first ? x_cost : init_old, BC[5] = 0.0;
                __threadfence_system();
                st_release_sys(x_flagB(D, q, w), epoch);
            }
        }
        return;
    }
#ifdef ICG_BA_PHASE_CLOCKS
#define DSM_CLK(k, t0)                                                                                             \
    if (D.clk && w == 0 && cr == 0 && tid == 0) atomicAdd(&D.clk[k], clock64() - (t0)), atomicAdd(&D.clk[8 + (k)], 1ull);
#define DSM_CLK2(k, t0)                                                                                            \
    if (D.clk && w == 0 && cr == 0 && tid == 0) atomicAdd(&D.clk[32 + (k)], clock64() - (t0)), atomicAdd(&D.clk[40 + (k)], 1ull);
#define DSM_NOW() clock64()
#else
#define DSM_CLK(k, t0)
#define DSM_CLK2(k, t0)
#define DSM_NOW() 0ull
#endif
    const unsigned long long tq0 = DSM_NOW();
    (void) tq0;
    // ---- assembly of S' = s H s + D^2 into the tiles: warp r takes row r of every local tile row (coalesced row reads; the loads of two tile
    //      rows -- up to 20 per lane -- are in flight together: the phase is L2 latency, 24 k cycles with one row at a time)
    for (int m = 0, T = cr; T < nt; m += 2, T += 2 * CL) {
        constexpr int NCH = (15 * 22 + 7 + 31) / 32;   // 32-column chunks of the longest row the shared-memory form admits (max_K = 22)
        double v[2][NCH];
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int Th = T + h * CL, i = 8 * Th + warp, ncol = 8 * Th;
            const double *src = (i < NCV ? Hs : Hc) + (size_t) (i < N ? i : 0) * C.NS;
#pragma unroll
            for (int u = 0; u < NCH; u++) {
                const int j = 32 * u + lane;
                v[h][u] = (Th < nt && j < ncol && i < N) ? __ldcg(src + j) : 0.0;
            }
        }
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int Th = T + h * CL, i = 8 * Th + warp, ncol = 8 * Th;
            if (Th >= nt) continue;
            double *trow = s_tiles + (size_t) dsm_tile_off(cr, m + h) * 64 + warp * 8;
            const double si = i < N ? s_scale[i] : 0.0;
#pragma unroll
            for (int u = 0; u < NCH; u++) {
                const int j = 32 * u + lane;
                if (j < ncol) trow[(j >> 3) * 64 + (j & 7)] = i < N ? si * s_scale[j] * v[h][u] : (i == N ? s_rhs[j] : 0.0);
            }
        }
    }
    {   // every diagonal tile, on every CTA: all of a thread's loads in flight (one dependent L2 round trip instead of one per element)
        constexpr int NDG = (dsm_ntiles(15 * 22 + 8) * 64 + SOLVE_THREADS - 1) / SOLVE_THREADS;
        double v[NDG];
#pragma unroll
        for (int u = 0; u < NDG; u++) {
            const int e = tid + u * SOLVE_THREADS, T = e >> 6, r = (e >> 3) & 7, c = e & 7, i = 8 * T + r, j = 8 * T + c;
            v[u] = (e < nt * 64 && c <= r && i < N) ? __ldcg((i < NCV ? Hs : Hc) + (size_t) i * C.NS + j) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < NDG; u++) {
            const int e = tid + u * SOLVE_THREADS, T = e >> 6, r = (e >> 3) & 7, c = e & 7, i = 8 * T + r, j = 8 * T + c;
            if (e >= nt * 64) continue;
            double x = 0;
            if (c <= r) {
                if (i < N) x = s_scale[i] * s_scale[j] * v[u] + (i == j ? s_d2[i] : 0.0);
                else if (i == N && j < N) x = s_rhs[j];
            }
            s_dg[e] = x;
        }
    }
    volatile int *s_dead = s_fail + 1;
    __syncthreads();
    DSM_CLK(0, tq0)  // assembly
    const int wi = warp < 4 ? warp - 1 : warp - 2;   // worker index 0 .. 5 of warps 1,2,3,5,6,7 (warp 4 shares warp 0's scheduler and FP64 pipe: it sits out)
    const bool worker = warp != 0 && warp != 4;
    int fail = 0;
    const unsigned long long tc_all = DSM_NOW();
    (void) tc_all;
    for (int J = 0; J < npan; J++) {
        const int nb = min(8, N - 8 * J);
        const double *PJ = s_P + (size_t) ((J - 1) & 1) * ntc * 64;   // panel J - 1's solved rows (J > 0)
        const unsigned long long tc0 = DSM_NOW();
        (void) tc0;
        if (J > 0 && tid < 8 && Tn > J - 1) s_y[8 * (J - 1) + tid] = PJ[(size_t) Tn * 64 + rn * 8 + tid];   // panel J - 1's right-hand-side entries: y
        DSM_CLK2(0, tc0)  // wait for the panel column
        const unsigned long long tc1 = DSM_NOW();
        (void) tc1;
        if (J > 0 && worker) {
            // Trailing update of panel Jp = J - 1: the CTA's tiles (T, tc), Jp < tc < T, and the diagonal replicas T >= Jp + 2 (every tile row).
            // Workers 0 .. 4 take PAIRS of local tile rows -- the i-th shortest with the i-th longest: equal work per pair --, worker 5 the
            // diagonal replicas (about as many tiles as a pair).  A row is a unit-stride walk (A fragment loaded once, pointers advance by a
            // tile), four tiles in flight: 8 operand loads, 8 DMMAs in four independent chains, 4 stores.  (A flattened work list with per-item
            // row look-up cost ~250 cycles per tile on these one-or-two-warp schedulers: the bookkeeping, not the arithmetic.)
            const int Jp = J - 1;
            auto run = [&](double a0, double a1, bool diag, const double *pb, double *pc, int n) {
                // n tiles from pb (B fragments) / pc (C tiles); diag: the A fragment is the tile's own B fragment
                for (; n > 0; n -= 4, pb += 256, pc += 256) {
                    double2 bq[4], cq[4];
#pragma unroll
                    for (int u = 0; u < 4; u++)
                        if (u < n) bq[u] = *(const double2 *) (pb + 64 * u), cq[u] = *(double2 *) (pc + 64 * u);
#pragma unroll
                    for (int u = 0; u < 4; u++)
                        if (u < n) dmma884(cq[u].x, cq[u].y, diag ? -bq[u].x : a0, bq[u].x);
#pragma unroll
                    for (int u = 0; u < 4; u++)
                        if (u < n) dmma884(cq[u].x, cq[u].y, diag ? -bq[u].y : a1, bq[u].y);
#pragma unroll
                    for (int u = 0; u < 4; u++)
                        if (u < n) *(double2 *) (pc + 64 * u) = cq[u];
                }
            };
            // both rows of a pair over their common columns: ONE B fragment per tile column feeds both rows (a third less shared-memory traffic
            // -- the update is bound by the shared-memory pipe as much as by the FP64 pipe) and eight DMMA chains are in flight
            auto run2 = [&](double a10, double a11, double a20, double a21, const double *pb, double *pc1, double *pc2, int n) {
                for (; n > 0; n -= 4, pb += 256, pc1 += 256, pc2 += 256) {
                    double2 bq[4], c1[4], c2[4];
#pragma unroll
                    for (int u = 0; u < 4; u++)
                        if (u < n) bq[u] = *(const double2 *) (pb + 64 * u), c1[u] = *(double2 *) (pc1 + 64 * u), c2[u] = *(double2 *) (pc2 + 64 * u);
#pragma unroll
                    for (int u = 0; u < 4; u++)
                        if (u < n) dmma884(c1[u].x, c1[u].y, a10, bq[u].x), dmma884(c2[u].x, c2[u].y, a20, bq[u].x);
#pragma unroll
                    for (int u = 0; u < 4; u++)
                        if (u < n) dmma884(c1[u].x, c1[u].y, a11, bq[u].y), dmma884(c2[u].x, c2[u].y, a21, bq[u].y);
#pragma unroll
                    for (int u = 0; u < 4; u++)
                        if (u < n) *(double2 *) (pc1 + 64 * u) = c1[u], *(double2 *) (pc2 + 64 * u) = c2[u];
                }
            };
            if (wi < 5) {
                const int m_lo = (Jp + 2 - cr + CL - 1) / CL, m_hi = cr < nt ? (nt - 1 - cr) / CL : -1;   // local tile rows T = cr + 4 m with Jp + 2 <= T < nt
                for (int i = wi; m_lo + i <= m_hi - i; i += 5) {
                    const int m1 = m_lo + i, m2 = m_hi - i, T1 = cr + CL * m1, T2 = cr + CL * m2;
                    const double2 pa1 = *(const double2 *) (PJ + (size_t) T1 * 64 + 2 * lane);
                    double *t1 = s_tiles + (size_t) dsm_tile_off(cr, m1) * 64 + 2 * lane;
                    const double *pb0 = PJ + (size_t) (Jp + 1) * 64 + 2 * lane;
                    if (m1 == m2) {
                        run(-pa1.x, -pa1.y, false, pb0, t1 + (size_t) (Jp + 1) * 64, T1 - (Jp + 1));
                    } else {
                        const double2 pa2 = *(const double2 *) (PJ + (size_t) T2 * 64 + 2 * lane);
                        double *t2 = s_tiles + (size_t) dsm_tile_off(cr, m2) * 64 + 2 * lane;
                        run2(-pa1.x, -pa1.y, -pa2.x, -pa2.y, pb0, t1 + (size_t) (Jp + 1) * 64, t2 + (size_t) (Jp + 1) * 64, T1 - (Jp + 1));
                        run(-pa2.x, -pa2.y, false, PJ + (size_t) T1 * 64 + 2 * lane, t2 + (size_t) T1 * 64, T2 - T1);   // the longer row's own columns
                    }
                }
            } else {
                run(0.0, 0.0, true, PJ + (size_t) (Jp + 2) * 64 + 2 * lane, s_dg + (size_t) (Jp + 2) * 64 + 2 * lane, nt - (Jp + 2));
            }
        }
        if (warp == 0) {
            const unsigned long long tf0 = DSM_NOW();
            (void) tf0;
            double *dg = s_dg + (size_t) J * 64;
            if (J > 0) {   // the previous panel's update of the tile about to be factored
                const double2 p = *(const double2 *) (PJ + (size_t) J * 64 + 2 * lane);
                double2 c = *(double2 *) (dg + 2 * lane);
                dmma884(c.x, c.y, -p.x, p.x);
                dmma884(c.x, c.y, -p.y, p.y);
                *(double2 *) (dg + 2 * lane) = c;
                __syncwarp();
            }
            DSM_CLK2(2, tf0)  // warp 0: update of the diagonal tile
            const unsigned long long tf1 = DSM_NOW();
            (void) tf1;
            double Ld[8][8], dinv[8];
            bool bad = false;
#pragma unroll
            for (int a = 0; a < 8; a++)
#pragma unroll
                for (int b = 0; b < 8; b++) Ld[a][b] = (a < nb && b <= a) ? dg[a * 8 + b] : (a == b ? 1.0 : 0.0);
#pragma unroll
            for (int j = 0; j < 8; j++) {
                double d = Ld[j][j];
#pragma unroll
                for (int k = 0; k < j; k++) d -= Ld[j][k] * Ld[j][k];
                if (!(d > 0.0) || !isfinite(d)) bad = true;
                const double di = rsqrt(d);
                dinv[j] = di;
                Ld[j][j] = d * di;
#pragma unroll
                for (int a = j + 1; a < 8; a++) {
                    double sum = Ld[a][j];
#pragma unroll
                    for (int k = 0; k < j; k++) sum -= Ld[a][k] * Ld[j][k];
                    Ld[a][j] = sum * di;
                }
            }
#ifdef ICG_BA_PHASE_CLOCKS
            if (Ld[7][7] == 12345.678) bad = true;  // the clock below is read after the arithmetic
#endif
            DSM_CLK2(3, tf1)  // warp 0: block loads + 8 x 8 factorisation in registers
            const unsigned long long tf2 = DSM_NOW();
            (void) tf2;
            __syncwarp();  // every lane has read the unfactored block
            // write-back: every lane holds the whole factor; entry e is stored by lane e mod 32 under a predicate -- statically indexed registers,
            // no divergent code.  (A switch on the lane, one path per row, cost 1 640 cycles; pairs of entries as 128-bit stores 1 010 -- the
            // register pairs have to be assembled first; scalar predicated stores 480.)
#pragma unroll
            for (int a2 = 0; a2 < 8; a2++) {
#pragma unroll
                for (int b = 0; b <= a2; b++)
                    if (lane == ((a2 * 8 + b) & 31) && a2 < nb) dg[a2 * 8 + b] = Ld[a2][b];
                if (lane == 8 + a2) s_dv[a2] = dinv[a2];
                if (lane == 16 + a2 && a2 < nb) s_dinv[8 * J + a2] = dinv[a2];
            }
            if (lane == 0 && bad) s_fail[0] = 1;
            DSM_CLK2(4, tf2)  // warp 0: write-back
            DSM_CLK(1, tf0)   // warp 0: diagonal-tile update + factorisation
        }
        __syncthreads();
        DSM_CLK(2, tc1)  // ... until the slower of factorisation and trailing update is through
        const unsigned long long tc2 = DSM_NOW();
        (void) tc2;
        fail = s_fail[0];  // identical on every CTA of the cluster (redundant bit-identical factorisations)
        if (fail) break;
        {   // rows below the panel: one thread per row of the local tile rows T > J
            const int m0 = (J + 1 - cr + CL - 1) / CL;
            const int m = m0 + (tid >> 3), r = tid & 7, T = cr + CL * m;
            if (T < nt) {
                double *tp = s_tiles + ((size_t) dsm_tile_off(cr, m) + J) * 64 + r * 8;
                const double *s_Ljj = s_dg + (size_t) J * 64;   // the factored block (nb = 8 whenever there are rows below)
                double x[8];
#pragma unroll
                for (int c = 0; c < 8; c += 2) {
                    const double2 t2 = *(const double2 *) (tp + c);
                    x[c] = t2.x, x[c + 1] = t2.y;
                }
#pragma unroll
                for (int c = 0; c < 8; c++) {
                    double sum = x[c];
#pragma unroll
                    for (int k = 0; k < c; k++) sum -= x[k] * s_Ljj[c * 8 + k];
                    x[c] = sum * s_dv[c];
                }
                // the solved row goes into the panel-column buffer of all four CTAs (addresses of the cluster window formed here: nothing of
                // this is live across the factorisation, whose 8 x 8 block fills the register file)
                double *dstP = s_P + (size_t) (J & 1) * ntc * 64 + (size_t) T * 64 + r * 8;
#pragma unroll
                for (int c = 0; c < 8; c += 2) *(double2 *) (tp + c) = make_double2(x[c], x[c + 1]);
#pragma unroll
                for (int q = 0; q < CL; q++) {
                    double *rp = cluster.map_shared_rank(dstP, q);
#pragma unroll
                    for (int c = 0; c < 8; c += 2) *(double2 *) (rp + c) = make_double2(x[c], x[c + 1]);
                }
            }
            cluster.sync();
        }
        DSM_CLK(3, tc2)  // row solves + hand-over
    }
    DSM_CLK(4, tc_all)   // whole factorisation
    const bool valid = !fail;
    const unsigned long long tb0 = DSM_NOW();
    (void) tb0;
    if (valid) {
        {   // the last panel's column (only the right-hand-side row can be below it)
            const int J = npan - 1;
            if (tid < 8 && Tn > J) s_y[8 * J + tid] = s_P[(size_t) (J & 1) * ntc * 64 + (size_t) Tn * 64 + rn * 8 + tid];
        }
        if (rn > 0 && tid == 0) {   // the right-hand-side row shares the last diagonal tile with the last rn columns
            double x[8];
            for (int c = 0; c < rn; c++) {
                double sum = s_dg[(size_t) Tn * 64 + rn * 8 + c];
                for (int k = 0; k < c; k++) sum -= x[k] * s_dg[(size_t) Tn * 64 + c * 8 + k];
                x[c] = sum * s_dv[c];
                s_y[8 * Tn + c] = x[c];
            }
        }
        __syncthreads();
        // ---- distributed backward substitution
        double *rX0 = cluster.map_shared_rank(s_x, 0);
        for (int T = npan - 1; T >= 0; T--) {
            if (cr == T % CL) {
                const int nbT = min(8, N - 8 * T), m = T / CL;
                const double *trow = s_tiles + (size_t) dsm_tile_off(cr, m) * 64;
                // The chain of the substitution stays inside warp 0: wait for the three partial-sum messages, 8 x 8 triangle, the row's
                // contribution to the next three tile rows (their columns of the row's tiles are loaded before the wait; x travels by shuffle),
                // send.  The other warps join at the block barrier and add the row's contribution to the columns further left.
                const int c0 = max(0, 8 * (T - 3)), ncrit = 8 * T - c0;
                if (warp == 0) {
                    const int c = lane & 7, col = c0 + lane;
                    double lcol[8], tcr[8], acc = 0;
#pragma unroll
                    for (int r = 0; r < 8; r++) lcol[r] = s_dg[(size_t) T * 64 + r * 8 + c];
                    if (lane < ncrit) {
                        const double *tp = trow + (col >> 3) * 64 + (col & 7);
#pragma unroll
                        for (int r = 0; r < 8; r++) tcr[r] = tp[r * 8];
                        acc = s_contrib[col];
                    } else {
#pragma unroll
                        for (int r = 0; r < 8; r++) tcr[r] = 0;
                    }
                    // three messages per tile row (from the owners of T + 1 .. T + 3); the ones that do not exist are arrived here
                    const int nmiss = max(0, 3 - (npan - 1 - T));
                    if (lane < nmiss) dsm_mbar_arrive_local(smem_u32(s_bar));
                    dsm_mbar_wait(smem_u32(s_bar), ((npan - 1 - T) / CL) & 1, s_dead, D.S.err);
                    double v = 0;
                    if (lane < nbT) {
                        v = s_y[8 * T + c] - s_contrib[8 * T + c];
#pragma unroll
                        for (int q = 0; q < CL; q++)
                            if (q != cr) v -= s_inbox[q * 8 + c];
                    }
#pragma unroll
                    for (int r = 7; r >= 0; r--) {   // x_r = (v_r - sum_{i > r} L_ir x_i) / L_rr; rows beyond N have a zero reciprocal pivot
                        const double xr = __shfl_sync(0xffffffffu, v, r) * s_dinv[8 * T + r];
                        if (lane == r) v = xr;
                        else if (lane < r) v -= lcol[r] * xr;
                    }
                    if (lane < 8) s_xT[lane] = v, rX0[8 * T + lane] = v;
#pragma unroll
                    for (int r = 0; r < 8; r++) acc += tcr[r] * __shfl_sync(0xffffffffu, v, r);
                    if (lane < ncrit) {
                        s_contrib[col] = acc;
                        const int q = (col >> 3) % CL;
                        const unsigned abar = mapa_u32(smem_u32(s_bar), q);
                        st_async_f64(mapa_u32(smem_u32(s_inbox + cr * 8 + (col & 7)), q), acc, abar);
                        if ((col & 7) == 0) dsm_mbar_arrive_expect_tx_remote(abar, 64u);
                    }
                }
                __syncthreads();
                for (int col = tid; col < c0; col += SOLVE_THREADS) {
                    const double *tp = trow + (col >> 3) * 64 + (col & 7);
                    double acc = s_contrib[col];
#pragma unroll
                    for (int r = 0; r < 8; r++) acc += tp[r * 8] * s_xT[r];
                    s_contrib[col] = acc;
                }
                __syncthreads();
            }
        }
    }
    cluster.sync();  // the solution has landed on CTA 0; no CTA leaves while its shared memory may still be written
    DSM_CLK(5, tb0)  // backward substitution
    if (cr != 0) return;
    // ---- camera part of the model cost change, broadcast of [header | delta = step' * scale]
    double part = 0;
    bool finite = true;
    if (valid)
        for (int a = tid; a < N; a += SOLVE_THREADS) {
            const double sp = s_x[a];
            finite = finite && isfinite(sp);
            part += -0.5 * sp * (s_scale[a] * s_g[a]) + 0.5 * s_d2[a] * sp * sp;
        }
    const double mcc = block_sum(part, s_red);
    const double nfin = block_sum(finite ? 0.0 : 1.0, s_red);
    for (int q = 0; q < D.world; q++) {
        BC = x_bcast(D, q, w);
        if (valid)
            for (int a = tid; a < N; a += SOLVE_THREADS) BC[SPLIT_HDR + a] = s_x[a] * s_scale[a];
        if (tid == 0) {
            BC[0] = 0.0, BC[1] = (valid && nfin == 0.0) ? 1.0 : 0.0, BC[2] = x_cost, BC[3] = gmax_now, BC[4] = f_first ? x_cost : init_old, BC[5] = mcc;
        }
    }
    __threadfence_system();
    __syncthreads();
    for (int q = tid; q < D.world; q += SOLVE_THREADS) st_release_sys(x_flagB(D, q, w), epoch);
}

// ------------------------------------------------------------------------------------------------ step_lm (every rank, STEP_SLICES CTAs per window)
// Landmark back-substitution (a 2 MB matrix-vector product per cfg-4 window: latency-bound on one CTA, 190 us at 2000 landmarks) is cut into
// STEP_SLICES contiguous landmark slices, one CTA each; slice 0 also forms the candidate camera blocks.  The slices' partial sums meet in
// slot order in the CTA that finishes last (a per-window counter that resets itself): the same bits whatever the arrival order and whatever
// the batch size.
constexpr int STEP_SLICES = 4;
__global__ void __launch_bounds__(SOLVE_THREADS) ba_step_lm(BaCaps C, BaDev D, unsigned long long epoch) {
    extern __shared__ double sm[];
    __shared__ int s_last;
    const int w = blockIdx.x, sl_id = blockIdx.y, tid = threadIdx.x;
    LmState &st = D.st[w];
    const WinDims dm = D.dims[w];
    const int K = dm.K, L = dm.L, NCV = 6 * K + 7, N = 15 * K + 7;
    const bool owner = (w % D.world) == D.rank;
    double *s_red = sm, *s_dl = s_red + 40;  // delta (N)
    // st.done: set in an earlier attempt (the owner's solve then returns without a broadcast: nothing to wait for), or in THIS attempt -- by the
    // owner's solve earlier in the stream, or by slice 0 of a non-owner mirroring the header while the other slices are still starting; in every
    // case all slices of the window leave without touching the slice counter
    if (st.done) return;
    const double *BC = x_bcast(D, D.rank, w);
    if (tid == 0) wait_flag(x_flagB(D, D.rank, w), epoch, D.S.err);
    __syncthreads();
    const int term = (int) __ldcg(BC + 0), valid = (int) __ldcg(BC + 1);
    double *R3 = D.red2 + (size_t) w * 4;
    if (!owner && tid == 0 && sl_id == 0) {  // mirror what the owner's solve did to the LM state
        st.x_cost = __ldcg(BC + 2), st.gmax = __ldcg(BC + 3), st.initial_cost = __ldcg(BC + 4);
        st.fresh_lin = 0, st.first = 0, st.need_lin = 0;
        if (term) st.done = term, st.step_valid = 0;
        else st.iter = st.iter + 1;
    }
    if (term) return;
    if (!valid) {
        if (tid == 0 && sl_id == 0) {
            st.chol_ok = 0, st.step_valid = 0;
            R3[0] = 0, R3[1] = 0, R3[2] = 1, R3[3] = 0;
        }
        return;
    }
    for (int a = tid; a < N; a += SOLVE_THREADS) s_dl[a] = __ldcg(BC + SPLIT_HDR + a);
    __syncthreads();
    const double radius = st.radius;
    const double *hl = D.hl + (size_t) w * C.L, *gl = D.gl + (size_t) w * C.L, *scale_l = D.scale_l + (size_t) w * C.L;
    double *step_l = D.step_l + (size_t) w * C.L;
    const double *AW = D.AW + (size_t) w * C.LP * C.NCA;
    const double *rho = D.rho + (size_t) w * C.L;
    double *rho_c = D.rho_c + (size_t) w * C.L;
    constexpr int LB = 4;
    const int per = ((L + STEP_SLICES - 1) / STEP_SLICES + LB - 1) / LB * LB;   // landmarks per slice (groups of LB stay whole)
    const int lbeg = min(L, sl_id * per), lend = min(L, lbeg + per);
    double part = 0, sn_l = 0, rho2 = 0;
    bool finite = true;
    {
        const int lane = tid & 31, warp = tid >> 5;
        for (int l0 = lbeg + LB * warp; l0 < lend; l0 += LB * (SOLVE_THREADS / 32)) {
            double d[LB];
#pragma unroll
            for (int u = 0; u < LB; u++) d[u] = 0;
            for (int c = lane; c < NCV; c += 32) {
                const double sx = s_dl[c];
#pragma unroll
                for (int u = 0; u < LB; u++) d[u] += (l0 + u < lend ? AW[(size_t) (l0 + u) * C.NCA + c] : 0.0) * sx;
            }
            double mine = 0;
#pragma unroll
            for (int u = 0; u < LB; u++) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) d[u] += __shfl_xor_sync(0xffffffffu, d[u], o);
                if (lane == u) mine = d[u];
            }
            if (lane < LB && l0 + lane < lend) {
                const int l = l0 + lane;
                const double sl = scale_l[l], hs = sl * sl * hl[l], d2 = fmin(fmax(hs, 1e-6), 1e32) / radius;
                const double sp = (-sl * gl[l] - sl * mine) / (hs + d2);
                finite = finite && isfinite(sp);
                step_l[l] = sp;
                part += -0.5 * sp * (sl * gl[l]) + 0.5 * d2 * sp * sp;
                // candidate inverse depth, |step|^2 and |rho|^2 (x_norm of the parameter tolerance test) of this landmark
                const double r0 = rho[l], v = r0 + sp * sl;
                rho_c[l] = v;
                sn_l += (r0 - v) * (r0 - v);
                rho2 += r0 * r0;
            }
        }
    }
    __syncthreads();
    const double mcc_l = block_sum(part, s_red);
    const double nfin = block_sum(finite ? 0.0 : 1.0, s_red);
    sn_l = block_sum(sn_l, s_red);
    rho2 = block_sum(rho2, s_red);
    // candidate point: camera blocks on every rank (bit-identical), by slice 0
    double sn_cam = 0;
    if (sl_id == 0) {
        const double *pose = D.pose + (size_t) w * C.K * 7, *mix = D.mix + (size_t) w * C.K * 9, *ext = D.ext + (size_t) w * 8;
        double *pose_c = D.pose_c + (size_t) w * C.K * 7, *mix_c = D.mix_c + (size_t) w * C.K * 9, *ext_c = D.ext_c + (size_t) w * 8;
        for (int k = tid; k <= K; k += SOLVE_THREADS) {
            const bool is_ext = (k == K);
            const double *x = is_ext ? ext : pose + k * 7;
            double *xc = is_ext ? ext_c : pose_c + k * 7;
            if (is_ext && dm.ext_const) {
                for (int e = 0; e < 7; e++) xc[e] = x[e];
            } else {
                const int c0 = is_ext ? col_ext(K) : col_pose(k);
                double d[6];
                for (int e = 0; e < 6; e++) d[e] = s_dl[c0 + e];
                pose_plus(x, d, xc);
                for (int e = 0; e < 7; e++) sn_cam += (x[e] - xc[e]) * (x[e] - xc[e]);
            }
        }
        for (int e = tid; e < K * 9; e += SOLVE_THREADS) {
            const int k = e / 9, q = e - 9 * k;
            const double v = mix[e] + s_dl[col_mix(K, k) + q];
            mix_c[e] = v;
            sn_cam += (mix[e] - v) * (mix[e] - v);
        }
        if (tid == 0) {
            if (dm.td_const) {
                ext_c[7] = ext[7];
            } else {
                const double v = ext[7] + s_dl[col_td(K)];
                ext_c[7] = v;
                sn_cam += (ext[7] - v) * (ext[7] - v);
            }
        }
    }
    sn_cam = block_sum(sn_cam, s_red);
    // the slices meet: slot [w][slice] = {model cost change, |step_l|^2, non-finite count, |rho|^2, |step_cam|^2}
    double *slot = D.S.slm + ((size_t) w * STEP_SLICES + sl_id) * 8;
    if (tid == 0) {
        slot[0] = mcc_l, slot[1] = sn_l, slot[2] = nfin, slot[3] = rho2, slot[4] = sn_cam;
        __threadfence();
        s_last = atomicAdd(D.S.slm_cnt + w, 1) == STEP_SLICES - 1;
    }
    __syncthreads();
    if (!s_last || tid != 0) return;
    __threadfence();
    D.S.slm_cnt[w] = 0;
    double m = 0, sl2 = 0, nf = 0, r2 = 0, sc2 = 0;
    const double *s0 = D.S.slm + (size_t) w * STEP_SLICES * 8;
    for (int q = 0; q < STEP_SLICES; q++) m += __ldcg(s0 + q * 8), sl2 += __ldcg(s0 + q * 8 + 1), nf += __ldcg(s0 + q * 8 + 2), r2 += __ldcg(s0 + q * 8 + 3), sc2 += __ldcg(s0 + q * 8 + 4);
    st.chol_ok = 1, st.step_valid = 1;
    R3[0] = m + (owner ? __ldcg(BC + 5) : 0.0), R3[1] = sl2 + (owner ? sc2 : 0.0), R3[2] = nf, R3[3] = r2;
}

// ------------------------------------------------------------------------------------------------ exchange + accept (every rank)
__global__ void ba_exchange(BaCaps C, BaDev D, int n, int nblk_vis, unsigned long long epoch) {
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n) return;
    const LmState &st = D.st[w];
    if (st.done) return;
    const WinDims dm = D.dims[w];
    const bool owner = (w % D.world) == D.rank;
    double cand = 0;
    if (st.step_valid) {
        const double *part = D.cost_part + (size_t) w * (nblk_vis + 1);
        const int nb = (dm.F + 255) / 256;
        for (int b = 0; b < nb; b++) cand += part[b];
        if (owner) cand += part[nblk_vis];
    }
    const double *R3 = D.red2 + (size_t) w * 4;
    for (int q = 0; q < D.world; q++) {
        double *s = x_scal(D, q, w, D.rank);
        s[0] = R3[0], s[1] = R3[1], s[2] = R3[2], s[3] = cand, s[4] = R3[3];
        __threadfence_system();
        st_release_sys(x_flagC(D, q, w, D.rank), epoch);
    }
}

__global__ void __launch_bounds__(128) ba_accept_split(BaCaps C, BaDev D, unsigned long long epoch) {
    __shared__ int s_accept;
    __shared__ double s_camsq;
    __shared__ double s_red[40];
    const int w = blockIdx.x, tid = threadIdx.x;
    LmState &st = D.st[w];
    if (st.done) return;
    const WinDims dm = D.dims[w];
    if (tid < D.world) wait_flag(x_flagC(D, D.rank, w, tid), epoch, D.S.err);
    {
        const double *pose = D.pose + (size_t) w * C.K * 7, *mix = D.mix + (size_t) w * C.K * 9, *ext = D.ext + (size_t) w * 8;
        double s = 0;
        for (int e = tid; e < dm.K * 7; e += 128) s += pose[e] * pose[e];
        for (int e = tid; e < dm.K * 9; e += 128) s += mix[e] * mix[e];
        if (tid < 7 && !dm.ext_const) s += ext[tid] * ext[tid];
        if (tid == 7 && !dm.td_const) s += ext[7] * ext[7];
        s = block_sum(s, s_red);
        if (tid == 0) s_camsq = s;
    }
    __syncthreads();
    if (tid == 0) {
        s_accept = 0;
        double mcc = 0, sn = 0, nfin = 0, cand = 0, rho2 = 0;
        for (int r = 0; r < D.world; r++) {  // fixed rank order on every rank
            const double *s = x_scal(D, D.rank, w, r);
            mcc += __ldcg(s + 0), sn += __ldcg(s + 1), nfin += __ldcg(s + 2), cand += __ldcg(s + 3), rho2 += __ldcg(s + 4);
        }
        if (!st.chol_ok || nfin != 0.0 || !(mcc > 0.0)) {
            st.step_valid = 0;
            st.n_invalid++;
            if (st.n_invalid >= 5) st.done = 3;
            st.radius *= 0.5;
            st.last_success = 0;
        } else {
            st.n_invalid = 0;
            st.model_cost_change = mcc;
            st.step_norm = sqrt(sn);
            st.x_norm = sqrt(s_camsq + rho2);
            st.cand_cost = cand;
            if (st.step_norm <= 1e-8 * (st.x_norm + 1e-8)) {
                st.done = 2;
            } else if (fabs(st.x_cost - cand) <= 1e-6 * st.x_cost) {
                st.done = 2;
            } else {
                const double rel = (st.x_cost - cand) / mcc;
                if (rel > 1e-3) {
                    s_accept = 1;
                    st.n_success++;
                    const double t = 2.0 * rel - 1.0;
                    st.radius = fmin(1e16, st.radius / fmax(1.0 / 3.0, 1.0 - t * t * t));
                    st.decrease_factor = 2.0;
                    st.last_success = 1;
                    st.need_lin = 1;
                    st.fresh_lin = 1;
                } else {
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

}  // namespace icg
