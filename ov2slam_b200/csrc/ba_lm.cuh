// Shared declarations of the persistent local-BA solve (ba_lm.cu) and its multi-GPU exchange (ba_comm.cu).
#pragma once
#include <stdint.h>

#include "ov2_common.cuh"

namespace balm {

constexpr unsigned FULL = 0xffffffffu;
constexpr int THREADS = 256, WARPS = THREADS / 32;
constexpr int MAX_VAR_CAMS = 64;            // optimised keyframes per window (ba_lm_kernel; larger windows: ba_large.cu)
constexpr int MAX_N = 6 * MAX_VAR_CAMS;     // reduced camera system
constexpr int MAX_CAMS = 256;               // keyframes per window (optimised + constant)
constexpr int CH_NB = 32;                   // block size of the blocked Cholesky
constexpr double SOPHUS_EPS = 1e-10;
constexpr int MAX_RANKS = 8;

// reduced scalars of one LM iteration (two parities)
enum { SC_COST = 0, SC_CAND_COST, SC_MCC, SC_STEP2, SC_CANDX2, SC_GMAX_LM, SC_GMAX_CAM, SC_CHOL_FAIL, SC_COUNT = 16 };

struct Result {
    int iters_robust, iters_refine;
    double initial_cost, final_cost;
    int n_outliers_first, n_outliers_second, termination, aborted;
};

// One window, as the kernel sees it (all pointers device memory).
struct Prob {
    int ncam, npts, nobs;
    double fx, fy, cx, cy, rfx, rfy, rcx, rcy, Rrl[9], trl[3];
    double huber_a, huber_b, ftol;
    float th_f;
    int use_robust, apply_l2, refine_loss, max_it1, max_it2;
    const int* stop_flag;              // device-visible int (mapped pinned host memory) or NULL: polled before solve #2
    const uint8_t* pose_const; const int32_t* lm_anchor_cam; const double* lm_anchor_px;
    const int32_t* obs_cam; const int32_t* obs_lm; const double* obs_px; const uint8_t* obs_type; const int32_t* lm_ptr;
    double* pose[2]; double* invd[2];  // x / candidate ping-pong
    uint8_t* active; uint8_t* flags; uint8_t* cam_used; int32_t* cam_slot;
    double *Jr, *Ja, *Jo, *Jl, *chi2; uint8_t* dpos;
    double *sc_lm, *ete, *ge;
    double* acc;                       // [ncopy][blk]: rhs | F'r | column norms | S
    double* total;                     // [blk]: folded / all-rank system
    double* scal;                      // [2][SC_COUNT]
    double *z, *sc_cam, *counts;
    double* panel;                     // [CH_NB][n + 24]: row panel of the blocked Cholesky (read by every CTA of the group)
    unsigned* bar;                     // [0] group barrier counter, [1] abort flag
    Result* result;
    unsigned long long* trace;         // optional [16] per-phase nanoseconds (OV2_BA_TRACE=1), NULL otherwise
    int ncv_max, ncopy, solve_blocked, smem_work_off, schur_smem, smem_sacc_off;
    int sg;                            // lanes per landmark in the per-landmark phases (4, 8 or 32)
    const int32_t* pair_perm;          // [nobs] observation indices sorted by (anchor keyframe, observing keyframe)   (owner mode)
    const int2* pair_chunk;            // [npchunk] (begin, end) into pair_perm, <= PCH observations of ONE pair each
    int npchunk;
    int gj2;                           // reduced solve n <= 48: two pivots per barrier
    size_t blk;
};

// Multi-GPU exchange buffer exported by every rank (one cudaMalloc, opened by the peers through CUDA IPC or, inside one
// process, used directly).  Byte offsets:
constexpr size_t XB_FLAGS = 0;          // unsigned long long [MAX_RANKS]: slot r = last epoch rank r has announced to us
constexpr size_t XB_SC4 = 256;          // double [2][8] candidate scalars per parity, + [16..18] outlier counts
constexpr size_t XB_CAMUSED = 1024;     // uint8 [2][MAX_CAMS]
constexpr size_t XB_PARTIAL = 4096;     // double [2][SC_COUNT + blk_max]: this rank's partial reduced system per parity
constexpr size_t XB_BLK_MAX = 3 * (size_t)MAX_N + (size_t)MAX_N * MAX_N;
constexpr size_t XB_BYTES = XB_PARTIAL + 2 * (SC_COUNT + XB_BLK_MAX) * sizeof(double);

struct Peers {
    int world, rank;
    unsigned long long epoch0;          // first epoch of this launch (host-side launch sequence << 20)
    void* base[MAX_RANKS];              // exported buffer of every rank, as mapped in THIS process
};

}  // namespace balm

// Solves `nprob` windows with one launch (peers == NULL: single GPU).  ba_lm.cu
ov2_status balm_solve(ov2_ctx* ctx, int nprob, const ov2_ba_problem* pbs, const ov2_ba_opts* opts, ov2_ba_result* results,
                      uint8_t* const* outlier_outs, const balm::Peers* peers, const int* stop_flag_dev);

// One window with more than MAX_VAR_CAMS optimised keyframes (up to OV2_BA_MAX_OPT_KEYFRAMES).  ba_large.cu
ov2_status balm_solve_large(ov2_ctx* ctx, const ov2_ba_problem* pb, const ov2_ba_opts* opts, ov2_ba_result* res,
                            uint8_t* outlier_out, const int* stop_flag_dev);
