// L (large windows): the two-stage local-BA solve of ov2_localba_solve for windows with more than 64 optimised keyframes
// (loop-closure looseBA, fullBA over a long run): up to OV2_BA_MAX_OPT_KEYFRAMES optimised and OV2_BA_MAX_KEYFRAMES
// keyframes in total.  Same algorithm, same phases and the same device-side trust-region controller (ba_lm_ctl.cuh) as
// ba_lm_kernel (ba_lm.cu, see its header comment); what is sized by the window lives in global memory / L2 instead of
// shared memory:
//
//   keyframe table   Rwc | twc of every keyframe, built once per evaluation by the whole group (x in phase A, the
//                    candidate in phase D) and read by the residual blocks from L2
//   Schur (B)        one warp per landmark (schur_landmark); the landmark's E'F rows are staged in a global slice indexed
//                    by its observations (lm_ptr[l] + l .. : at most one entry per observation + the anchor), the
//                    contributions leave as fp64 RED into the reduced system
//   reduced system   upper triangle of a dense np x np fp64 array (np = n rounded up to 32, n = 6 x optimised keyframes in
//                    trajectory order), cut into 32 x 32 tiles.  The host derives the keyframe block pattern from the
//                    observations and its tile-level symbolic Cholesky fill (ba_fill.cuh); only the tiles of the fill are
//                    zeroed, accumulated, factored and updated.  The pattern of the first stage is kept for the refinement
//                    (it only removes observations); keyframes that drop out of the second stage's program keep their
//                    rows, which become identity rows with a zero right-hand side.
//   solve (C)        right-looking blocked Cholesky A = U'U, one 32-wide block step per tile row, over the fill tiles only:
//                      F1  every CTA with work factors the diagonal tile in its own shared memory (one warp, registers),
//                          then its warps solve the panel tiles (k, j) and the right-hand side segment (forward substitution)
//                      F2  trailing update A(i, j) -= U(k, i)' U(k, j) of every pair of panel tiles on the FP64 tensor cores
//                          (DMMA m8n8k4), one warp per tile pair over the whole group; the diagonal pairs also carry the
//                          forward substitution into the later right-hand side segments
//                    two group barriers per block step; the backward substitution goes column by column (the diagonal solve
//                    redundantly in every CTA with work, the column's tiles spread over the group), one barrier per step.
//                    No part of a block step whose work grows with n runs on one CTA.
//   D                candidate keyframes (group) -> keyframe table -> back-substitution + candidate cost (sub-group per
//                    landmark, backsub_landmarks_sg), z read from global memory
//   E                the controller, replayed by every CTA.
//
// One launch per solve, one group made of every co-resident CTA.
#include "ov2_common.cuh"
#include "ba_lm.cuh"
#include "ba_lm_ctl.cuh"
#include "ba_lm_dev.cuh"
#include "ba_fill.cuh"

#include <float.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <mutex>
#include <vector>

namespace balm {

constexpr int TB = bafill::TILE;

struct LargeProb {
    Prob p;                            // window, work arrays and scalars as ba_lm_kernel uses them (p.acc: the system below)
    int n, np, nt, nlay;               // n = 6 nlay unknowns, np = 32 nt: pitch of the dense array
    const int32_t* lay;                // [ncam] position of the keyframe in the system (first stage's program), -1: not in it
    const int32_t* rptr;               // [nt + 1] fill tiles by tile row: rcol[rptr[k]] = k, then the columns j > k ascending
    const int32_t* rcol;
    const int32_t* cptr;               // [nt + 1] fill tiles by tile column, strictly above the diagonal: rows i < k
    const int32_t* crow;
    const int2* ftile; int nfill;      // every fill tile (row, column)
    double* cam;                       // [ncam][12] keyframe table (Rwc, twc)
    double* etf; int32_t* eslot;       // [nobs + npts] E'F staging (6 doubles / 1 slot per entry)
    uint8_t* live;                     // [nlay] keyframe in this stage's program
    double* idiag;                     // [np] 1 / U(i, i)
    double* y;                         // [np] right-hand side -> forward substitution (the step goes to p.z)
};

__device__ __forceinline__ void cam_entry(const double* pose7, double* out12) {
    double t[3], q[4], R[9];
    load_pose(pose7, t, q);
    quat_to_rot(q, R);
#pragma unroll
    for (int k = 0; k < 9; ++k) out12[k] = R[k];
    out12[9] = t[0]; out12[10] = t[1]; out12[11] = t[2];
}

// Diagonal tile (kb, kb) -> U_kk in sU (upper), 1 / U(i, i) in s_id; the whole CTA loads, warp 0 factors with the column
// of lane j in registers (pivot chain: shuffle -> rsqrt seed + two Newton steps -> one shared-memory row broadcast).
// Returns true when a pivot is not positive and finite (LLT failure).
__device__ __forceinline__ bool factor_diag(const double* A, size_t np, int kb, double (*sU)[TB + 1], double* s_id, int* s_bad) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int e = tid; e < TB * TB; e += THREADS) {
        const int i = e >> 5, j = e & 31;
        sU[i][j] = i <= j ? A[(size_t)(kb + i) * np + kb + j] : 0.0;
    }
    __syncthreads();
    if (warp == 0) {
        bool bad = false;
        double a[TB];
#pragma unroll
        for (int r = 0; r < TB; ++r) a[r] = sU[r][lane];
#pragma unroll
        for (int j = 0; j < TB; ++j) {
            const double d = __shfl_sync(FULL, a[j], j);
            bad = bad || !(d > 1e-30) || !(d < 1e30);
            double is;
            asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(is) : "d"(d));
            is = fma(0.5 * is, fma(-d * is, is, 1.0), is);
            is = fma(0.5 * is, fma(-d * is, is, 1.0), is);
            const double ujc = lane >= j ? a[j] * is : 0.0;
            sU[j][lane] = ujc;
            if (lane == j) s_id[j] = is;
            __syncwarp();
#pragma unroll
            for (int r = j + 1; r < TB; ++r) a[r] = fma(-sU[j][r], ujc, a[r]);
        }
        if (lane == 0) *s_bad = bad ? 1 : 0;
    }
    __syncthreads();
    return *s_bad != 0;
}

// U_kk' x = b for one column held by this thread (32 values in registers)
__device__ __forceinline__ void trsm_col(double (&a)[TB], const double (*sU)[TB + 1], const double* s_id) {
#pragma unroll
    for (int k = 0; k < TB; ++k) {
        const double x = a[k] * s_id[k];
        a[k] = x;
#pragma unroll
        for (int i = k + 1; i < TB; ++i) a[i] = fma(-sU[k][i], x, a[i]);
    }
}

// Reduced camera system: the caller has applied the damping and put the right-hand side into L.y; on return P.z holds the
// step (system order) or scal[SC_CHOL_FAIL] is set.  Must be called by every CTA of the group.  The barrier goes in by value
// (a reference would keep it in local memory across the call) and its epoch comes back.
__device__ __noinline__ unsigned large_solve(const LargeProb& L, GroupBar bar, int bid, int G, double* scal) {
    const Prob& P = L.p;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int gwarps = G * WARPS, gwarp = bid * WARPS + warp;
    const size_t np = (size_t)L.np;
    double* A = P.acc + 3 * np;
    double* z = P.z;
    double* y = L.y;
    __shared__ double sU[TB][TB + 1];
    __shared__ double s_id[TB];
    __shared__ double s_z[TB];
    __shared__ int s_bad;
    const bool tr = P.trace != nullptr && bid == 0 && tid == 0;
    unsigned long long tr_t = tr ? global_ns() : 0;
#define TRS(k) do { if (tr) { const unsigned long long t_ = global_ns(); P.trace[k] += t_ - tr_t; tr_t = t_; } } while (0)
    for (int k = 0; k < L.nt; ++k) {
        const int kb = k * TB;
        const int r0 = L.rptr[k], nr = L.rptr[k + 1] - r0;     // item 0: diagonal tile + right-hand side, items 1..: panel tiles
        if (bid < nr) {
            const bool bad = factor_diag(A, np, kb, sU, s_id, &s_bad);
            if (bad) {
                if (bid == 0 && tid == 0) scal[SC_CHOL_FAIL] = 1.0;
            } else {
                for (int t = bid + G * warp; t < nr; t += G * WARPS) {
                    if (t == 0) {                                // right-hand side segment (its U_kk goes back after the barrier)
                        double a[TB];
#pragma unroll
                        for (int i = 0; i < TB; ++i) a[i] = y[kb + i];
                        trsm_col(a, sU, s_id);
                        if (lane == 0) {
#pragma unroll
                            for (int i = 0; i < TB; ++i) y[kb + i] = a[i];
                        }
                    } else {
                        double* col = A + (size_t)kb * np + (size_t)L.rcol[r0 + t] * TB + lane;
                        double a[TB];
#pragma unroll
                        for (int i = 0; i < TB; ++i) a[i] = col[(size_t)i * np];
                        trsm_col(a, sU, s_id);
#pragma unroll
                        for (int i = 0; i < TB; ++i) col[(size_t)i * np] = a[i];
                    }
                }
            }
        }
        TRS(12);
        bar.sync();
        TRS(13);
        if (scal[SC_CHOL_FAIL] != 0.0) return bar.epoch;                 // uniform across the group (written before the barrier)
        if (bid == 0) {                 // U_kk into the array: every CTA of F1 has read the diagonal tile by now
            for (int e = tid; e < TB * TB; e += THREADS) {
                const int i = e >> 5, j = e & 31;
                if (i <= j) A[(size_t)(kb + i) * np + kb + j] = sU[i][j];
            }
            if (tid < TB) L.idiag[kb + tid] = s_id[tid];
        }
        // F2: every pair a <= b of panel tiles (items 1..nr-1)
        const int m = nr - 1, npair = m * (m + 1) / 2;
        const int g = lane >> 2, t4 = lane & 3;
        for (int p = gwarp; p < npair; p += gwarps) {
            int a = 0, rem = p;
            while (rem >= m - a) { rem -= m - a; ++a; }
            const int b = a + rem;
            const int ja = L.rcol[r0 + 1 + a], jb = L.rcol[r0 + 1 + b];
            const double* Ua = A + (size_t)kb * np + (size_t)ja * TB;
            const double* Ub = A + (size_t)kb * np + (size_t)jb * TB;
            const bool diag = ja == jb;
            double acc[4][4][2];
#pragma unroll
            for (int hi = 0; hi < 4; ++hi)
#pragma unroll
                for (int hj = 0; hj < 4; ++hj) { acc[hi][hj][0] = 0.0; acc[hi][hj][1] = 0.0; }
#pragma unroll
            for (int k0 = 0; k0 < TB; k0 += 4) {
                const size_t ro = (size_t)(k0 + t4) * np;
                double av[4], bv[4];
#pragma unroll
                for (int h = 0; h < 4; ++h) { av[h] = Ua[ro + 8 * h + g]; bv[h] = Ub[ro + 8 * h + g]; }
#pragma unroll
                for (int hi = 0; hi < 4; ++hi)
#pragma unroll
                    for (int hj = 0; hj < 4; ++hj)
                        if (!diag || hi <= hj) dmma_884(acc[hi][hj][0], acc[hi][hj][1], av[hi], bv[hj]);
            }
            double* D = A + (size_t)ja * TB * np + (size_t)jb * TB;
#pragma unroll
            for (int hi = 0; hi < 4; ++hi)
#pragma unroll
                for (int hj = 0; hj < 4; ++hj) {
                    if (diag && hi > hj) continue;
#pragma unroll
                    for (int e = 0; e < 2; ++e) D[(size_t)(8 * hi + g) * np + 8 * hj + 2 * t4 + e] -= acc[hi][hj][e];
                }
            if (diag) {                                                   // forward substitution: z_j -= U(k, j)' y_k
                double s = 0.0;
#pragma unroll 8
                for (int i = 0; i < TB; ++i) s += Ub[(size_t)i * np + lane] * y[kb + i];
                y[(size_t)jb * TB + lane] -= s;
            }
        }
        TRS(14);
        bar.sync();
        TRS(13);
    }
    // backward substitution U z = y, last tile column first: z_k = U_kk^-1 y_k (every CTA with work), then
    // y_i -= U(i, k) z_k for the fill tiles of column k (spread over the group)
    for (int k = L.nt - 1; k >= 0; --k) {
        const int kb = k * TB;
        const int c0 = L.cptr[k], nitem = L.cptr[k + 1] - c0 + 1;    // item 0: store z_k
        if (bid < nitem) {
            for (int e = tid; e < TB * TB; e += THREADS) {
                const int i = e >> 5, j = e & 31;
                sU[i][j] = i <= j ? A[(size_t)(kb + i) * np + kb + j] : 0.0;
            }
            __syncthreads();
            if (warp == 0) {
                double ti = y[kb + lane], zm = 0.0;
                const double idg = L.idiag[kb + lane];
#pragma unroll
                for (int j = TB - 1; j >= 0; --j) {
                    const double zj = __shfl_sync(FULL, ti * idg, j);
                    if (lane < j) ti -= sU[lane][j] * zj;
                    if (lane == j) zm = zj;
                }
                s_z[lane] = zm;
            }
            __syncthreads();
            for (int t = bid + G * warp; t < nitem; t += G * WARPS) {
                if (t == 0) {
                    z[kb + lane] = s_z[lane];
                } else {
                    const int ib = L.crow[c0 + t - 1] * TB;
                    const double* row = A + (size_t)(ib + lane) * np + kb;
                    double s = 0.0;
#pragma unroll 8
                    for (int c = 0; c < TB; ++c) s += row[c] * s_z[c];
                    y[ib + lane] -= s;
                }
            }
        }
        bar.sync();
    }
    TRS(15);
#undef TRS
    return bar.epoch;
}

// B: Schur elimination, warp per landmark, fp64 RED into the dense system (E'F rows staged at lm_ptr[l] + l)
// (per-warp Jacobian staging: [WARPS][28 SCH] doubles, then [WARPS][SCH] ints, behind the keyframe slots in dynamic shared memory)
__device__ __forceinline__ void large_schur(const LargeProb& L, unsigned char* smem, int* s_slot, int gwarp, int gwarps, double radius,
                                            int first_iter, double* scal) {
    const Prob& P = L.p;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* const sJ0 = reinterpret_cast<double*>(smem + (((size_t)P.ncam * sizeof(int) + 15) & ~(size_t)15));
    double* const sJ = sJ0 + (size_t)warp * (28 * SCH);
    int* const smeta = reinterpret_cast<int*>(sJ0 + (size_t)WARPS * 28 * SCH) + warp * SCH;
    double gmax_lm = 0.0;
    for (int l = gwarp; l < P.npts; l += gwarps) {
        const size_t e0 = (size_t)P.lm_ptr[l] + l;
        schur_landmark<false>(P, s_slot, L.etf + 6 * e0, L.eslot + e0, sJ, smeta, l, lane, radius, first_iter, P.acc, L.np, gmax_lm, nullptr);
    }
    if (lane == 0 && gmax_lm > 0.0) atomic_max_pos(scal + SC_GMAX_LM, gmax_lm);
}

// D: back-substitution, candidate point and candidate cost (keyframe table: the candidate's)
__device__ __forceinline__ void large_backsub(const LargeProb& L, const int* s_slot, int gwarp, int gwarps, const double* x_invd, double* c_invd,
                                           int use_huber, double& mcc, double& lst2, double& lcx2, double& cost) {
    const Prob& P = L.p;
    const int lane = threadIdx.x & 31;
    if (P.sg == 4) {
        for (int l0 = gwarp * 8; l0 < P.npts; l0 += gwarps * 8)
            backsub_landmarks_sg<4>(P, s_slot, L.cam, l0, lane, x_invd, c_invd, use_huber, mcc, lst2, lcx2, cost);
    } else if (P.sg == 8) {
        for (int l0 = gwarp * 4; l0 < P.npts; l0 += gwarps * 4)
            backsub_landmarks_sg<8>(P, s_slot, L.cam, l0, lane, x_invd, c_invd, use_huber, mcc, lst2, lcx2, cost);
    } else {
        for (int l = gwarp; l < P.npts; l += gwarps)
            backsub_landmark(P, s_slot, L.cam, l, lane, x_invd, c_invd, use_huber, mcc, lst2, lcx2, cost);
    }
}

__global__ void __launch_bounds__(THREADS, 1) ba_large_kernel(const LargeProb* __restrict__ lp, int G) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ LargeProb L;
    __shared__ lmctl::State S;
    __shared__ int s_action, s_refine, s_trivial;
    __shared__ double s_red[WARPS][4];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int bid = blockIdx.x;
    if (bid >= G) return;
    for (int i = tid; i < (int)(sizeof(LargeProb) / sizeof(int)); i += THREADS)
        reinterpret_cast<int*>(&L)[i] = reinterpret_cast<const int*>(lp)[i];
    __syncthreads();
    const Prob& P = L.p;
    GroupBar bar{P.bar, P.bar + 1, (unsigned)G, 0u};
    // optional phase trace (CTA 0 / thread 0, straight into the zero-initialised trace record)
    unsigned long long tr_last = 0;
    const bool tracing = P.trace != nullptr && bid == 0 && tid == 0;
    if (tracing) tr_last = global_ns();
#define TR(k) do { if (tracing) { const unsigned long long t_ = global_ns(); P.trace[k] += t_ - tr_last; tr_last = t_; } } while (0)
    int* s_slot = reinterpret_cast<int*>(smem_raw);                                                    // [ncam]
    // (the Schur staging slices behind s_slot are carved out inside large_schur: pointers kept live across the whole kernel
    //  were what it spilled)
    const int gthreads = G * THREADS, gtid = bid * THREADS + tid;
    const int gwarps = G * WARPS, gwarp = bid * WARPS + warp;
    const size_t np = (size_t)L.np;
    double* const cRhs = P.acc; double* const cG = P.acc + np; double* const cCn = P.acc + 2 * np; double* const A = P.acc + 3 * np;
    int xi = 0;
    int use_huber = P.use_robust;
    int n_out1 = 0, n_out2 = 0;
    int it0 = 0, it1 = 0, term_last = 0;
    double cost0_last = 0.0, cost1_last = 0.0;
    int ran_refine = 0;
    // zeroes the fill tiles and the vectors of the system (whole group)
    auto clear_system = [&]() {
        for (int e = gtid; e < 3 * L.np; e += gthreads) P.acc[e] = 0.0;
        for (int f = gwarp; f < L.nfill; f += gwarps) {
            const int2 tl = L.ftile[f];
            double* base = A + (size_t)tl.x * TB * np + (size_t)tl.y * TB + lane;
            for (int r = 0; r < TB; ++r) base[(size_t)r * np] = 0.0;
        }
    };
    for (int stage = 0; stage < 2; ++stage) {
        const int max_iters = stage == 0 ? P.max_it1 : P.max_it2;
        uint8_t* cam_used = P.cam_used + (size_t)stage * P.ncam;
        double* x_pose = P.pose[xi]; double* c_pose = P.pose[xi ^ 1];
        double* x_invd = P.invd[xi]; double* c_invd = P.invd[xi ^ 1];
        // ---- set-up: the keyframes this stage's program uses (Program::RemoveFixedBlocks), candidate := x, system zeroed
        for (int c = tid; c < P.ncam; c += THREADS) s_slot[c] = 0;
        __syncthreads();
        for (int i = gtid; i < P.nobs; i += gthreads)
            if (P.active[i] && !(P.obs_type && P.obs_type[i] == 2)) {
                s_slot[P.obs_cam[i]] = 1;
                s_slot[P.lm_anchor_cam[P.obs_lm[i]]] = 1;
            }
        __syncthreads();
        for (int c = tid; c < P.ncam; c += THREADS)
            if (s_slot[c]) cam_used[c] = 1;
        for (int i = gtid; i < 7 * P.ncam; i += gthreads) c_pose[i] = x_pose[i];
        for (int i = gtid; i < P.npts; i += gthreads) c_invd[i] = x_invd[i];
        clear_system();
        for (int i = gtid; i < 2 * SC_COUNT; i += gthreads) P.scal[i] = 0.0;
        TR(stage == 0 ? 0 : 10);
        bar.sync();
        TR(stage == 0 ? 11 : 10);
        int any = 0;
        for (int c = tid; c < P.ncam; c += THREADS) {
            const int u = cam_used[c];
            any |= u;
            s_slot[c] = (u && !P.pose_const[c]) ? L.lay[c] : -1;   // position in the (first stage's) system
        }
        any = __syncthreads_or(any);
        if (!any) { if (stage == 0) break; else continue; }
        for (int c = gtid; c < P.ncam; c += gthreads)
            if (L.lay[c] >= 0) L.live[L.lay[c]] = s_slot[c] >= 0 ? 1 : 0;
        if (tid == 0) lmctl::init(S);
        __syncthreads();
        TR(0);
        for (;;) {
            if (tid == 0) s_action = lmctl::begin_iteration(S, max_iters) ? 1 : 0;
            __syncthreads();
            if (!s_action) break;
            const int par = S.iteration & 1, first_iter = S.first_iter, x_is_new = S.x_is_new;
            const double radius = S.radius;
            double* scal = P.scal + par * SC_COUNT;
            // ---- A: keyframe table at x, residual blocks + Jacobians
            if (x_is_new) {
                for (int c = gtid; c < P.ncam; c += gthreads) cam_entry(x_pose + 7 * c, L.cam + 12 * (size_t)c);
                bar.sync();
                double cost = 0.0;
                for (int i = gtid; i < P.nobs; i += gthreads)
                    if (P.active[i]) cost += eval_block<true>(P, i, P.obs_lm[i], L.cam, x_invd[P.obs_lm[i]], use_huber);
                cost = warp_sum(cost);
                if (lane == 0) s_red[warp][0] = cost;
                __syncthreads();
                if (tid == 0) {
                    double a = 0.0;
                    for (int w_ = 0; w_ < WARPS; ++w_) a += s_red[w_][0];
                    if (a != 0.0) red_add_f64(scal + SC_COST, a);
                }
            }
            bar.sync();
            TR(1);
            // ---- B: Schur elimination, warp per landmark, RED into the dense system
            large_schur(L, smem_raw, s_slot, gwarp, gwarps, radius, first_iter, scal);
            bar.sync();
            TR(2);
            // ---- C: gradient projection |x - Plus(x, -g)|_inf, LM damping + Jacobi scaling, then the blocked factorisation
            if (x_is_new) {
                double gm = 0.0;
                for (int c = gtid; c < P.ncam; c += gthreads) {
                    const int s = s_slot[c];
                    if (s < 0) continue;
                    double d[6], out[7];
                    for (int k = 0; k < 6; ++k) d[k] = -cG[6 * s + k];
                    pose_plus(x_pose + 7 * c, d, out);
                    for (int k = 0; k < 7; ++k) gm = fmax(gm, fabs(x_pose[7 * c + k] - out[k]));
                }
                gm = warp_max(gm);
                if (lane == 0 && gm > 0.0) atomic_max_pos(scal + SC_GMAX_CAM, gm);
            }
            for (int i = gtid; i < L.np; i += gthreads) {
                double* aii = A + (size_t)i * np + i;
                if (i < L.n && L.live[i / 6]) {
                    const double cn = cCn[i];
                    double sc = P.sc_cam[i];
                    if (first_iter) {
                        sc = 1.0 / (1.0 + sqrt(cn));
                        P.sc_cam[i] = sc;
                    }
                    const double diag = fmin(fmax(cn * sc * sc, 1e-6), 1e32);
                    *aii += diag / (radius * sc * sc);
                    L.y[i] = cG[i] + cRhs[i];
                } else {                                   // padding, or a keyframe outside this stage's program
                    *aii = 1.0;
                    L.y[i] = 0.0;
                }
            }
            bar.sync();
            TR(3);
            bar.epoch = large_solve(L, bar, bid, G, scal);
            TR(4);
            bar.sync();
            TR(5);
            // ---- D: candidate keyframes -> keyframe table; back-substitution, candidate point and cost
            {
                double st2 = 0.0, cx2 = 0.0;
                const bool ok = scal[SC_CHOL_FAIL] == 0.0;
                for (int c = gtid; c < P.ncam; c += gthreads) {
                    const int s = s_slot[c];
                    double out[7];
                    if (s >= 0 && ok) {
                        double d[6];
                        for (int k = 0; k < 6; ++k) d[k] = -P.z[6 * s + k];
                        pose_plus(x_pose + 7 * c, d, out);
                        for (int k = 0; k < 7; ++k) {
                            const double df = x_pose[7 * c + k] - out[k];
                            st2 += df * df; cx2 += out[k] * out[k];
                            c_pose[7 * c + k] = out[k];
                        }
                    } else {
                        for (int k = 0; k < 7; ++k) out[k] = x_pose[7 * c + k];
                    }
                    cam_entry(out, L.cam + 12 * (size_t)c);
                }
                bar.sync();
                double mcc = 0.0, cost = 0.0, lst2 = st2, lcx2 = cx2;
                if (ok) large_backsub(L, s_slot, gwarp, gwarps, x_invd, c_invd, use_huber, mcc, lst2, lcx2, cost);
                mcc = warp_sum(mcc); cost = warp_sum(cost); lst2 = warp_sum(lst2); lcx2 = warp_sum(lcx2);
                if (lane == 0) { s_red[warp][0] = cost; s_red[warp][1] = mcc; s_red[warp][2] = lst2; s_red[warp][3] = lcx2; }
                __syncthreads();
                if (tid < 4) {
                    double a = 0.0;
                    for (int w_ = 0; w_ < WARPS; ++w_) a += s_red[w_][tid];
                    if (a != 0.0) red_add_f64(scal + SC_CAND_COST + tid, a);
                }
                clear_system();                              // for the next iteration
                double* oscal = P.scal + (par ^ 1) * SC_COUNT;
                if (gtid < SC_COUNT) oscal[gtid] = 0.0;
            }
            bar.sync();
            TR(6);
            // ---- E: trust-region controller, replayed by every CTA
            if (tid == 0) {
                const double gmax = fmax(scal[SC_GMAX_LM], scal[SC_GMAX_CAM]);
                s_action = (int)lmctl::end_iteration(S, scal[SC_COST], scal[SC_CAND_COST], scal[SC_MCC], scal[SC_STEP2], scal[SC_CANDX2], gmax,
                                                     scal[SC_CHOL_FAIL] != 0.0, P.ftol);
            }
            __syncthreads();
            const int action = s_action;
            TR(7);
            if (action == lmctl::ACT_CONTINUE_ACCEPTED) {
                xi ^= 1;
                x_pose = P.pose[xi]; c_pose = P.pose[xi ^ 1];
                x_invd = P.invd[xi]; c_invd = P.invd[xi ^ 1];
            }
            if (action == lmctl::ACT_STOP) break;
        }
        if (stage == 0) it0 = S.iteration; else it1 = S.iteration;
        cost0_last = S.initial_cost;                 // (the result record reports the last solve that ran)
        cost1_last = lmctl::final_cost(S);
        term_last = S.termination;
        if (stage == 1) ran_refine = 1;
        bar.sync();
        // ---- outlier scan on the values the last evaluation left behind (as ba_lm_kernel)
        {
            double* cnt = P.counts + 4 * stage;
            const int bit = stage == 0 ? 1 : 2;
            const int deact = stage == 0 && P.apply_l2;
            int bad_t = 0, left_t = 0, right_t = 0;
            for (int i = gtid; i < P.nobs; i += gthreads) {
                if (!P.active[i]) continue;
                const bool bad = (P.chi2[i] > (double)P.th_f) || !P.dpos[i];
                if (bad) {
                    P.flags[i] |= (uint8_t)bit;
                    if (deact) P.active[i] = 0;
                    bad_t++;
                } else {
                    const int typ = P.obs_type ? (int)P.obs_type[i] : 0;
                    left_t += typ == 0;
                    right_t += typ == 1;
                }
            }
            bad_t = __reduce_add_sync(FULL, bad_t); left_t = __reduce_add_sync(FULL, left_t); right_t = __reduce_add_sync(FULL, right_t);
            if (lane == 0) { s_red[warp][0] = (double)bad_t; s_red[warp][1] = (double)left_t; s_red[warp][2] = (double)right_t; }
            __syncthreads();
            if (tid < 3) {
                double a = 0.0;
                for (int w_ = 0; w_ < WARPS; ++w_) a += s_red[w_][tid];
                if (a != 0.0) red_add_f64(cnt + tid, a);
            }
            if (stage == 0 && bid == 0 && tid == 0)
                cnt[3] = (P.stop_flag && *reinterpret_cast<volatile const int*>(P.stop_flag) != 0) ? 1.0 : 0.0;
            bar.sync();
            if (stage == 0) {
                n_out1 = (int)cnt[0];
                int refine = P.apply_l2 && P.use_robust && cnt[0] > 0.0;
                if (refine && cnt[3] != 0.0) refine = 0;
                int trivial = P.refine_loss;
                if (trivial < 0) trivial = (cnt[1] > 0.0 && cnt[2] > 0.0) ? 1 : 0;
                if (tid == 0) { s_refine = refine; s_trivial = trivial; }
                __syncthreads();
                if (!s_refine) break;
                use_huber = s_trivial ? 0 : 1;
            } else {
                n_out2 = (int)cnt[0];
            }
        }
    }
    TR(8);
    bar.sync();
    if (xi == 1) {
        for (int i = gtid; i < 7 * P.ncam; i += gthreads) P.pose[0][i] = P.pose[1][i];
        for (int i = gtid; i < P.npts; i += gthreads) P.invd[0][i] = P.invd[1][i];
    }
    if (bid == 0 && tid == 0) {
        Result* R = P.result;
        R->iters_robust = it0;
        R->iters_refine = ran_refine ? it1 : 0;
        R->initial_cost = cost0_last;
        R->final_cost = cost1_last;
        R->termination = term_last;
        R->n_outliers_first = n_out1;
        R->n_outliers_second = n_out2;
        R->aborted = (int)ld_acquire_gpu(P.bar + 1);
    }
    TR(9);
#undef TR
}

}  // namespace balm

// ====================================================================== host side
using namespace balm;

namespace {

size_t take_l(size_t& off, size_t bytes, size_t align = 256) {
    off = (off + align - 1) & ~(align - 1);
    const size_t o = off;
    off += bytes ? bytes : 1;
    return o;
}

}  // namespace

// The tile pattern of a window's reduced system: the keyframe blocks every landmark couples (anchor x observer,
// observer x observer, in the first stage's program), closed under the symbolic factorisation.
static void window_fill(const ov2_ba_problem* pb, const std::vector<int32_t>& lay, int nt, std::vector<uint8_t>& T) {
    T.assign((size_t)nt * nt, 0);
    std::vector<int> sl;
    for (int i = 0, l = -1; i <= pb->nobs; ++i) {
        if (i == pb->nobs || pb->obs_lm[i] != l) {
            if (!sl.empty()) {
                std::sort(sl.begin(), sl.end());
                sl.erase(std::unique(sl.begin(), sl.end()), sl.end());
                for (size_t a = 0; a < sl.size(); ++a)
                    for (size_t b = a; b < sl.size(); ++b) bafill::mark_block(nt, T.data(), sl[a], sl[b]);
            }
            sl.clear();
            if (i == pb->nobs) break;
            l = pb->obs_lm[i];
            const int a = lay[pb->lm_anchor_cam[l]];
            if (a >= 0) sl.push_back(a);
        }
        if (pb->obs_type && pb->obs_type[i] == 2) continue;
        const int o = lay[pb->obs_cam[i]];
        if (o >= 0) sl.push_back(o);
    }
    bafill::symbolic_fill(nt, T.data());
}

void balm_prob_scalars(const ov2_ba_problem* pb, const ov2_ba_opts* opts, Prob& P, const double* Kh, const double* krh, const double* trlh);

// The single-window solve for windows with more than 64 optimised keyframes (ov2_localba_solve routes them here).
// `pb` arrays: host memory, or device memory when pb->pose is device memory (each array is then inspected).
ov2_status balm_solve_large(ov2_ctx* ctx, const ov2_ba_problem* pb_in, const ov2_ba_opts* opts, ov2_ba_result* res,
                            uint8_t* outlier_out, const int* stop_flag_dev) {
    if (!ctx || !pb_in || !opts || !res) return ov2_fail(ctx, OV2_ERR_INVALID, "ov2_localba_solve: bad arguments");
    memset(res, 0, sizeof(*res));
    ov2_status st = ov2_begin(ctx);
    if (st != OV2_OK) return st;
    ov2_ba_problem pb = *pb_in;
    const int ncam = pb.ncam, npts = pb.npts, nobs = pb.nobs;
    if (ncam <= 0 || npts < 0 || nobs < 0) return ov2_fail(ctx, OV2_ERR_INVALID, "ov2_localba_solve: bad arguments");
    if (ncam > OV2_BA_MAX_KEYFRAMES) return ov2_fail(ctx, OV2_ERR_CAPACITY, "ov2_localba_solve: more than OV2_BA_MAX_KEYFRAMES (4096) keyframes in the window");
    // device-resident windows are staged through the host once (the packing below needs the observation graph)
    const bool win_dev = ov2_is_device_ptr(pb.pose);
    std::vector<std::vector<char>> hold;
    cudaError_t pull_err = cudaSuccess;
    auto pull = [&](const void* p, size_t bytes) -> const void* {
        if (!p || bytes == 0 || !win_dev || !ov2_is_device_ptr(p)) return p;
        hold.emplace_back(bytes);
        const cudaError_t ce = cudaMemcpy(hold.back().data(), p, bytes, cudaMemcpyDeviceToHost);
        if (ce != cudaSuccess) pull_err = ce;
        return hold.back().data();
    };
    pb.K = (const double*)pull(pb.K, 32);
    pb.pose_const = (const uint8_t*)pull(pb.pose_const, ncam);
    pb.lm_anchor_cam = (const int32_t*)pull(pb.lm_anchor_cam, sizeof(int32_t) * (size_t)npts);
    pb.lm_anchor_px = (const double*)pull(pb.lm_anchor_px, sizeof(double) * 2 * (size_t)npts);
    pb.obs_cam = (const int32_t*)pull(pb.obs_cam, sizeof(int32_t) * (size_t)nobs);
    pb.obs_lm = (const int32_t*)pull(pb.obs_lm, sizeof(int32_t) * (size_t)nobs);
    pb.obs_px = (const double*)pull(pb.obs_px, sizeof(double) * 2 * (size_t)nobs);
    pb.obs_type = (const uint8_t*)pull(pb.obs_type, (size_t)nobs);
    pb.Kr = (const double*)pull(pb.Kr, 32);
    pb.Trl = (const double*)pull(pb.Trl, 56);
    const double* pose_h = (const double*)pull(pb.pose, sizeof(double) * 7 * (size_t)ncam);
    const double* invd_h = (const double*)pull(pb.lm_invdepth, sizeof(double) * (size_t)npts);
    if (pull_err != cudaSuccess) return ov2_fail(ctx, OV2_ERR_CUDA, "ov2_localba_solve: staging a device-resident window", pull_err);
    if (pb.obs_type && (!pb.Kr || !pb.Trl)) return ov2_fail(ctx, OV2_ERR_INVALID, "ov2_localba_solve: obs_type given without Kr / Trl");
    int ncv = 0;
    for (int c = 0; c < ncam; ++c) ncv += pb.pose_const[c] ? 0 : 1;
    if (ncv > OV2_BA_MAX_OPT_KEYFRAMES) return ov2_fail(ctx, OV2_ERR_CAPACITY, "ov2_localba_solve: more than OV2_BA_MAX_OPT_KEYFRAMES (1024) optimised keyframes");
    if (nobs == 0) return OV2_OK;                          // nothing to solve (as ov2_localba_solve for small windows)
    // validation + CSR by landmark
    std::vector<int32_t> lp((size_t)npts + 1, 0);
    for (int i = 0; i < nobs; ++i) {
        const int l = pb.obs_lm[i];
        if (l < 0 || l >= npts || (i > 0 && l < pb.obs_lm[i - 1])) return ov2_fail(ctx, OV2_ERR_INVALID, "ov2_localba_solve: obs_lm must be sorted ascending and in range");
        if (pb.obs_cam[i] < 0 || pb.obs_cam[i] >= ncam) return ov2_fail(ctx, OV2_ERR_INVALID, "ov2_localba_solve: obs_cam out of range");
        lp[l + 1]++;
    }
    for (int l = 0; l < npts; ++l) lp[l + 1] += lp[l];
    for (int l = 0; l < npts; ++l)
        if (pb.lm_anchor_cam[l] < 0 || pb.lm_anchor_cam[l] >= ncam) return ov2_fail(ctx, OV2_ERR_INVALID, "ov2_localba_solve: lm_anchor_cam out of range");
    // the first stage's program (the kernel derives the same set): optimised keyframes touched by a residual block that
    // has a pose block, in keyframe order
    std::vector<uint8_t> used(ncam, 0);
    for (int i = 0; i < nobs; ++i)
        if (!(pb.obs_type && pb.obs_type[i] == 2)) { used[pb.obs_cam[i]] = 1; used[pb.lm_anchor_cam[pb.obs_lm[i]]] = 1; }
    std::vector<int32_t> lay(ncam, -1);
    int nlay = 0;
    for (int c = 0; c < ncam; ++c)
        if (used[c] && !pb.pose_const[c]) lay[c] = nlay++;
    const int n = 6 * nlay, nt = n > 0 ? (n + TB - 1) / TB : 1, npd = nt * TB;
    std::vector<uint8_t> T;
    window_fill(&pb, lay, nt, T);
    std::vector<int32_t> rptr(nt + 1, 0), rcol, cptr(nt + 1, 0), crow;
    std::vector<int2> ftile;
    for (int k = 0; k < nt; ++k) {
        rcol.push_back(k);
        for (int j = k + 1; j < nt; ++j)
            if (T[(size_t)k * nt + j]) rcol.push_back(j);
        rptr[k + 1] = (int32_t)rcol.size();
    }
    for (int k = 0; k < nt; ++k) {
        for (int i = 0; i < k; ++i)
            if (T[(size_t)i * nt + k]) crow.push_back(i);
        cptr[k + 1] = (int32_t)crow.size();
    }
    for (int k = 0; k < nt; ++k)
        for (int j = k; j < nt; ++j)
            if (T[(size_t)k * nt + j]) ftile.push_back(make_int2(k, j));
    // ---- memory plan: one device block
    const size_t no = nobs, nq = npts, nc = ncam;
    size_t off = 0;
    const size_t o_lp = take_l(off, sizeof(int32_t) * (nq + 1)), o_pose0 = take_l(off, sizeof(double) * 7 * nc), o_pose1 = take_l(off, sizeof(double) * 7 * nc);
    const size_t o_invd0 = take_l(off, sizeof(double) * nq), o_invd1 = take_l(off, sizeof(double) * nq);
    const size_t o_apx = take_l(off, sizeof(double) * 2 * nq), o_opx = take_l(off, sizeof(double) * 2 * no);
    const size_t o_lac = take_l(off, sizeof(int32_t) * nq), o_oc = take_l(off, sizeof(int32_t) * no), o_ol = take_l(off, sizeof(int32_t) * no);
    const size_t o_pc = take_l(off, nc), o_ty = take_l(off, pb.obs_type ? no : 0), o_lay = take_l(off, sizeof(int32_t) * nc);
    const size_t o_rptr = take_l(off, sizeof(int32_t) * (nt + 1)), o_rcol = take_l(off, sizeof(int32_t) * rcol.size());
    const size_t o_cptr = take_l(off, sizeof(int32_t) * (nt + 1)), o_crow = take_l(off, sizeof(int32_t) * crow.size());
    const size_t o_ft = take_l(off, sizeof(int2) * ftile.size()), o_lpr = take_l(off, sizeof(LargeProb));
    const size_t in_bytes = off;
    const size_t z0 = take_l(off, 0);                      // zero-initialised region
    const size_t o_flags = take_l(off, no), o_camused = take_l(off, 2 * nc), o_counts = take_l(off, sizeof(double) * 8);
    const size_t o_bar = take_l(off, sizeof(unsigned) * 4), o_trace = take_l(off, sizeof(unsigned long long) * 16);
    const size_t o_sclm = take_l(off, sizeof(double) * nq), o_result = take_l(off, sizeof(Result));
    const size_t zbytes = off - z0;
    const size_t o_active = take_l(off, no);
    const size_t o_Jr = take_l(off, sizeof(double) * 2 * no), o_Ja = take_l(off, sizeof(double) * 12 * no), o_Jo = take_l(off, sizeof(double) * 12 * no);
    const size_t o_Jl = take_l(off, sizeof(double) * 2 * no), o_chi2 = take_l(off, sizeof(double) * no), o_dpos = take_l(off, no);
    const size_t o_ete = take_l(off, sizeof(double) * nq), o_ge = take_l(off, sizeof(double) * nq);
    const size_t o_scal = take_l(off, sizeof(double) * 2 * SC_COUNT), o_z = take_l(off, sizeof(double) * npd), o_sccam = take_l(off, sizeof(double) * npd);
    const size_t o_idiag = take_l(off, sizeof(double) * npd), o_y = take_l(off, sizeof(double) * npd), o_live = take_l(off, (size_t)nlay);
    const size_t o_cam = take_l(off, sizeof(double) * 12 * nc), o_etf = take_l(off, sizeof(double) * 6 * (no + nq)), o_eslot = take_l(off, sizeof(int32_t) * (no + nq));
    const size_t o_acc = take_l(off, sizeof(double) * (3 * (size_t)npd + (size_t)npd * npd));
    const size_t total = off + 256;
    if (total > OV2_BA_LARGE_MAX_BYTES)
        return ov2_fail(ctx, OV2_ERR_CAPACITY, "ov2_localba_solve: the window's device memory plan exceeds OV2_BA_LARGE_MAX_BYTES");
    void* o = nullptr;
    if ((st = ov2_scratch(ctx, total, &o)) != OV2_OK) return st;
    char* d = (char*)o;
    std::vector<char> h(in_bytes);
    memcpy(h.data() + o_lp, lp.data(), sizeof(int32_t) * (nq + 1));
    memcpy(h.data() + o_pose0, pose_h, sizeof(double) * 7 * nc);
    memcpy(h.data() + o_invd0, invd_h, sizeof(double) * nq);
    memcpy(h.data() + o_apx, pb.lm_anchor_px, sizeof(double) * 2 * nq);
    memcpy(h.data() + o_opx, pb.obs_px, sizeof(double) * 2 * no);
    memcpy(h.data() + o_lac, pb.lm_anchor_cam, sizeof(int32_t) * nq);
    memcpy(h.data() + o_oc, pb.obs_cam, sizeof(int32_t) * no);
    memcpy(h.data() + o_ol, pb.obs_lm, sizeof(int32_t) * no);
    memcpy(h.data() + o_pc, pb.pose_const, nc);
    if (pb.obs_type) memcpy(h.data() + o_ty, pb.obs_type, no);
    memcpy(h.data() + o_lay, lay.data(), sizeof(int32_t) * nc);
    memcpy(h.data() + o_rptr, rptr.data(), sizeof(int32_t) * (nt + 1));
    memcpy(h.data() + o_rcol, rcol.data(), sizeof(int32_t) * rcol.size());
    memcpy(h.data() + o_cptr, cptr.data(), sizeof(int32_t) * (nt + 1));
    if (!crow.empty()) memcpy(h.data() + o_crow, crow.data(), sizeof(int32_t) * crow.size());
    memcpy(h.data() + o_ft, ftile.data(), sizeof(int2) * ftile.size());
    LargeProb L;
    memset(&L, 0, sizeof(L));
    Prob& P = L.p;
    balm_prob_scalars(&pb, opts, P, pb.K, pb.Kr, pb.Trl);
    P.stop_flag = stop_flag_dev;
    P.pose_const = (const uint8_t*)(d + o_pc);
    P.lm_anchor_cam = (const int32_t*)(d + o_lac);
    P.lm_anchor_px = (const double*)(d + o_apx);
    P.obs_cam = (const int32_t*)(d + o_oc);
    P.obs_lm = (const int32_t*)(d + o_ol);
    P.obs_px = (const double*)(d + o_opx);
    P.obs_type = pb.obs_type ? (const uint8_t*)(d + o_ty) : nullptr;
    P.lm_ptr = (const int32_t*)(d + o_lp);
    P.pose[0] = (double*)(d + o_pose0); P.pose[1] = (double*)(d + o_pose1);
    P.invd[0] = (double*)(d + o_invd0); P.invd[1] = (double*)(d + o_invd1);
    P.active = (uint8_t*)(d + o_active); P.flags = (uint8_t*)(d + o_flags);
    P.cam_used = (uint8_t*)(d + o_camused);
    P.Jr = (double*)(d + o_Jr); P.Ja = (double*)(d + o_Ja); P.Jo = (double*)(d + o_Jo); P.Jl = (double*)(d + o_Jl);
    P.chi2 = (double*)(d + o_chi2); P.dpos = (uint8_t*)(d + o_dpos);
    P.sc_lm = (double*)(d + o_sclm); P.ete = (double*)(d + o_ete); P.ge = (double*)(d + o_ge);
    P.acc = (double*)(d + o_acc); P.scal = (double*)(d + o_scal);
    P.z = (double*)(d + o_z); P.sc_cam = (double*)(d + o_sccam);
    P.counts = (double*)(d + o_counts); P.bar = (unsigned*)(d + o_bar); P.result = (Result*)(d + o_result);
    P.trace = getenv("OV2_BA_TRACE") ? (unsigned long long*)(d + o_trace) : nullptr;
    P.ncv_max = nlay; P.ncopy = 1;
    const double avg = (double)nobs / (double)npts;
    P.sg = avg <= 5.0 ? 4 : (avg <= 12.0 ? 8 : 32);
    if (getenv("OV2_BA_SG")) { const int e = atoi(getenv("OV2_BA_SG")); if (e == 4 || e == 8 || e == 32) P.sg = e; }
    L.n = n; L.np = npd; L.nt = nt; L.nlay = nlay;
    L.lay = (const int32_t*)(d + o_lay);
    L.rptr = (const int32_t*)(d + o_rptr); L.rcol = (const int32_t*)(d + o_rcol);
    L.cptr = (const int32_t*)(d + o_cptr); L.crow = (const int32_t*)(d + o_crow);
    L.ftile = (const int2*)(d + o_ft); L.nfill = (int)ftile.size();
    L.cam = (double*)(d + o_cam); L.etf = (double*)(d + o_etf); L.eslot = (int32_t*)(d + o_eslot);
    L.live = (uint8_t*)(d + o_live); L.idiag = (double*)(d + o_idiag); L.y = (double*)(d + o_y);
    memcpy(h.data() + o_lpr, &L, sizeof(L));
    cudaStream_t s = ctx->stream;
    OV2_CUDA(ctx, cudaMemcpyAsync(d, h.data(), in_bytes, cudaMemcpyHostToDevice, s));
    OV2_CUDA(ctx, cudaMemsetAsync(d + z0, 0, zbytes, s));
    OV2_CUDA(ctx, cudaMemsetAsync(d + o_active, 1, no, s));
    // ---- launch: one group of co-resident CTAs
    const size_t smem = (((size_t)ncam * sizeof(int) + 15) & ~(size_t)15) + (size_t)WARPS * 28 * SCH * sizeof(double) + (size_t)WARPS * SCH * sizeof(int) + 16;
    {
        static size_t attr_smem[16] = {0};
        static std::mutex attr_mu;
        std::lock_guard<std::mutex> attr_lock(attr_mu);
        const int dv = ctx->device & 15;
        if (smem > attr_smem[dv]) {
            OV2_CUDA(ctx, cudaFuncSetAttribute(ba_large_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            attr_smem[dv] = smem;
        }
    }
    int per_sm = 0;
    OV2_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ba_large_kernel, THREADS, smem));
    if (per_sm < 1) return ov2_fail(ctx, OV2_ERR_CAPACITY, "ov2_localba_solve: kernel does not fit an SM");
    const int resident = per_sm * ctx->sm_count;
    const int wk = (nobs + THREADS - 1) / THREADS, wl = (npts + WARPS - 1) / WARPS;
    int G = wk > wl ? wk : wl;
    if (G > resident) G = resident;
    if (G < 1) G = 1;
    if (getenv("OV2_BA_CTAS")) { const int e = atoi(getenv("OV2_BA_CTAS")); if (e >= 1 && e <= resident) G = e; }
    const LargeProb* dl = (const LargeProb*)(d + o_lpr);
    if (ctx->profiling) ov2_prof_begin(ctx);
    ba_large_kernel<<<G, THREADS, smem, s>>>(dl, G);
    const cudaError_t le = cudaGetLastError();
    ctx->launches++;
    if (le != cudaSuccess) return ov2_fail(ctx, OV2_ERR_CUDA, "ba_large_kernel launch", le);
    if (ctx->profiling) ov2_prof_end(ctx, "ba_large_kernel");
    // ---- results
    std::vector<double> pose_out(7 * nc), invd_out(nq);
    std::vector<uint8_t> flags_out(no);
    Result hr;
    OV2_CUDA(ctx, cudaMemcpyAsync(pose_out.data(), d + o_pose0, sizeof(double) * 7 * nc, cudaMemcpyDeviceToHost, s));
    OV2_CUDA(ctx, cudaMemcpyAsync(invd_out.data(), d + o_invd0, sizeof(double) * nq, cudaMemcpyDeviceToHost, s));
    OV2_CUDA(ctx, cudaMemcpyAsync(flags_out.data(), d + o_flags, no, cudaMemcpyDeviceToHost, s));
    OV2_CUDA(ctx, cudaMemcpyAsync(&hr, d + o_result, sizeof(Result), cudaMemcpyDeviceToHost, s));
    OV2_CUDA(ctx, cudaStreamSynchronize(s));
    if (getenv("OV2_BA_TRACE")) {
        unsigned long long tr[16];
        cudaMemcpy(tr, d + o_trace, sizeof(tr), cudaMemcpyDeviceToHost);
        static const char* names[16] = {"setup0", "A:eval", "B:schur", "C:damp", "C:solve", "C:wait", "D:backsub", "E:ctl", "scan", "wb", "setup1", "bar0",
                                        "chol:panel", "chol:bar", "chol:update", "chol:back"};
        fprintf(stderr, "[ba trace] large G=%d smem=%zu n=%d tiles=%d/%d |", G, smem, n, (int)ftile.size(), nt * (nt + 1) / 2);
        for (int k = 0; k < 16; ++k) fprintf(stderr, " %s %.1fus", names[k], tr[k] / 1e3);
        fprintf(stderr, "\n");
    }
    const size_t pbytes = sizeof(double) * 7 * nc, ibytes = sizeof(double) * nq;
    if (win_dev) OV2_CUDA(ctx, cudaMemcpy(pb_in->pose, pose_out.data(), pbytes, cudaMemcpyHostToDevice));
    else memcpy(pb_in->pose, pose_out.data(), pbytes);
    if (win_dev && ov2_is_device_ptr(pb_in->lm_invdepth)) OV2_CUDA(ctx, cudaMemcpy(pb_in->lm_invdepth, invd_out.data(), ibytes, cudaMemcpyHostToDevice));
    else memcpy(pb_in->lm_invdepth, invd_out.data(), ibytes);
    if (outlier_out) {
        if (win_dev && ov2_is_device_ptr(outlier_out)) OV2_CUDA(ctx, cudaMemcpy(outlier_out, flags_out.data(), no, cudaMemcpyHostToDevice));
        else memcpy(outlier_out, flags_out.data(), no);
    }
    res->iters_robust = hr.iters_robust; res->iters_refine = hr.iters_refine;
    res->initial_cost = hr.initial_cost; res->final_cost = hr.final_cost;
    res->n_outliers_first = hr.n_outliers_first; res->n_outliers_second = hr.n_outliers_second;
    res->termination = hr.termination;
    if (hr.aborted) return ov2_fail(ctx, OV2_ERR_CUDA, "ov2_localba_solve: a barrier timed out");
    if (res->termination == 2) return ov2_fail(ctx, OV2_ERR_NUMERIC, "ov2_localba_solve: 5 consecutive invalid steps");
    return OV2_OK;
}
