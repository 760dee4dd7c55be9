// L: local bundle adjustment as ONE persistent kernel per solve (float64), device-side LM controller.
//
// Reference behaviour replaced: the solve sections of Optimizer::localBA
// (/root/reference/src/optimizer.cpp:436-479 robust solve, :492-594 outlier scan, :603-627 refinement,
// :637-735 second scan), i.e. Ceres 2.0's TrustRegionMinimizer (trust_region_minimizer.cc:67-134) +
// LevenbergMarquardtStrategy (levenberg_marquardt_strategy.cc:66-160) + Schur linear solver
// (schur_eliminator_impl.h:179-377) on the anchored inverse-depth residual blocks
// (src/ceres_parametrization.cpp:361-712) with SE3LeftParameterization (se3left_parametrization.hpp:41-60).
//
// Design (B200): a solve is launch/sync-latency bound (C3: 0.66 MB per LM iteration, all of it L2 resident), so
// the whole two-stage solve - both Ceres solves, both outlier scans, every LM iteration - is ONE cooperative
// launch.  A "group" of G CTAs works on one window; the phases of an LM iteration are separated by a group
// barrier (monotonic counter in global memory, release/acquire), not by kernel boundaries:
//
//   A  residual blocks + analytic Jacobians at x (thread per observation, keyframe rotations staged in shared
//      memory), cost                                                       [only when x changed]
//   B  Schur elimination, one warp per landmark, fp64 RED into the reduced camera system
//   B2 fold of the privatised accumulation copies (multi-GPU: the partial systems of all ranks are summed here
//      straight out of peer memory over NVLink - no NCCL call, no host round trip)
//   C  reduced camera system: LM damping + solve (n <= 96: Gauss-Jordan in CTA 0's shared memory; larger: blocked
//      Cholesky, sequential part on CTA 0, FP64 tensor-core trailing update spread over the group), gradient
//      projection by the last CTA
//   D  back-substitution + candidate point + candidate cost (warp per landmark; candidate poses are computed
//      redundantly by every CTA into shared memory)
//   E  the trust-region controller (ba_lm_ctl.cuh) replayed by every CTA from the same reduced scalars: all CTAs
//      take the same accept / reject / stop decision without a broadcast and without the host.
//
// K windows can be solved by one launch (ov2_localba_solve_batch): groups pull windows round-robin.
#include "ov2_common.cuh"
#include "ba_lm.cuh"
#include "ba_lm_ctl.cuh"
#include "ba_lm_dev.cuh"

#include <float.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <atomic>
#include <mutex>
#include <thread>

namespace balm {

// ------------------------------------------------------------------ Schur elimination, "owner" mode (reduced systems up to n = 96)
// The RED path above sends ~900 fp64 reductions per landmark to the global block and a B200 SM retires one fp64 RED lane
// every ~2.4-3.6 cycles: a batched C3 solve spent 6.7 of its 11.9 ms there (OV2_BA_TRACE, round 2).  This mode forms the
// same sums where nothing has to be shared:
//   B1  camera part F'F, F'r, column norms: the observations are pre-sorted by (anchor keyframe, observing keyframe)
//       (host: pack_window), so a chunk of <= PCH observations touches ONE 12 x 12 Gram block [Ja | Jo]'[Ja | Jo]; a warp
//       owns a chunk, its lanes own the 78 + 12 entries (upper triangle + gradient), the chunk's Jacobian rows pass through the
//       warp's staging slice of shared memory, and the chunk's totals leave as <= 102 REDs (was ~89 per observation).
//   B2  landmark part: SG lanes per landmark form ete / g_e and the landmark's E'F row as a DENSE n-vector in a shared-memory
//       tile (one row per landmark, 32 / SG rows per warp); then S -= sum_rows w y y', rhs -= sum_rows w g_e y on the FP64
//       tensor cores, every warp owning 8 x 8 tiles of the upper triangle over ALL rounds (no atomics at all), flushed once.
constexpr int PCH = 32;           // observations per pair chunk

// pitch (doubles) of the owner-mode landmark tile: >= n rounded up to 8, congruent 4 mod 16
__host__ __device__ __forceinline__ int owner_tile_pitch(int n) {
    const int n8 = (n + 7) & ~7;
    return n8 + ((4 - n8) % 16 + 16) % 16;
}

template <int SG>
__device__ __forceinline__ void owner_fill_row(const Prob& P, const int* __restrict__ s_slot, int l, int sl, bool in, double radius, int first_iter,
                                               double* row, double& w_out, double& ge_out, double& gmax_lm) {
    const int p0 = in ? P.lm_ptr[l] : 0, p1 = in ? P.lm_ptr[l + 1] : 0;
    const int sa = in ? s_slot[P.lm_anchor_cam[l]] : -1;
    double cnl = 0.0, ge = 0.0, aE[6] = {0, 0, 0, 0, 0, 0};
    int nact = 0;
    for (int p = p0 + sl; p < p1; p += SG) {
        const uint8_t act = P.active[p];
        const double2 jl = *reinterpret_cast<const double2*>(P.Jl + 2 * (size_t)p);
        const double2 jr = *reinterpret_cast<const double2*>(P.Jr + 2 * (size_t)p);
        if (!act) continue;
        cnl += jl.x * jl.x + jl.y * jl.y;
        ge += jl.x * jr.x + jl.y * jr.y;
        nact++;
        if (P.obs_type && P.obs_type[p] == 2) continue;          // e-block-only row (schur_eliminator_impl.h:196-217)
        const double* Ja = P.Ja + 12 * (size_t)p;
        if (sa >= 0) {
#pragma unroll
            for (int k = 0; k < 6; ++k) aE[k] += jl.x * Ja[k] + jl.y * Ja[6 + k];
        }
        const int so = s_slot[P.obs_cam[p]];
        if (so >= 0) {
            const double* Jo = P.Jo + 12 * (size_t)p;
#pragma unroll
            for (int k = 0; k < 6; ++k) atomicAdd(row + 6 * so + k, jl.x * Jo[k] + jl.y * Jo[6 + k]);   // a stereo keyframe observes twice
        }
    }
#pragma unroll
    for (int o = SG / 2; o > 0; o >>= 1) {
        cnl += __shfl_xor_sync(FULL, cnl, o);
        ge += __shfl_xor_sync(FULL, ge, o);
        nact += __shfl_xor_sync(FULL, nact, o);
#pragma unroll
        for (int k = 0; k < 6; ++k) aE[k] += __shfl_xor_sync(FULL, aE[k], o);
    }
    w_out = 0.0;
    ge_out = 0.0;
    if (!in) return;
    if (nact == 0) {   // unused parameter block: dropped from the program (program.cc:305-387)
        if (sl == 0) { P.ete[l] = 0.0; P.ge[l] = 0.0; }
        return;
    }
    double sc = P.sc_lm[l];
    if (first_iter) {
        sc = 1.0 / (1.0 + sqrt(cnl));
        if (sl == 0) P.sc_lm[l] = sc;
    }
    const double diag = fmin(fmax(cnl * sc * sc, 1e-6), 1e32);
    const double ete = cnl + diag / (radius * sc * sc);
    if (sl == 0) {
        P.ete[l] = ete;
        P.ge[l] = ge;
        if (sa >= 0) {
#pragma unroll
            for (int k = 0; k < 6; ++k) atomicAdd(row + 6 * sa + k, aE[k]);
        }
    }
    gmax_lm = fmax(gmax_lm, fabs(ge));
    w_out = 1.0 / ete;
    ge_out = ge;
}

template <int NT, int SG>
__device__ __noinline__ void schur_owner_phase(const Prob& P, const int* __restrict__ s_slot, double* s_tile, int n, double radius, int first_iter,
                                               int bid, int G, double* scal) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int gwarps = G * WARPS, gwarp = bid * WARPS + warp;
    double* const cRhs = P.acc; double* const cG = P.acc + n; double* const cCn = P.acc + 2 * n; double* const cS = P.acc + 3 * n;
    // ---------------- B1: camera part, one pair chunk per warp
    const bool tracing = P.trace != nullptr && bid == 0 && tid == 0;
    const unsigned long long t_b1 = tracing ? global_ns() : 0;
    {
        double* st = s_tile + (size_t)warp * (PCH * 26);
        int ia0[3], ja0[3], ja1[3], ei[3], ej[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int e = lane + 32 * k;
            ei[k] = -1; ej[k] = -1; ia0[k] = 0; ja0[k] = 0; ja1[k] = 0;
            if (e < 78) {
                int i = 0, rem = e;
                while (rem >= 12 - i) { rem -= 12 - i; ++i; }
                const int j = i + rem;
                ei[k] = i; ej[k] = j;
                ia0[k] = i < 6 ? i : i + 6;
                ja0[k] = j < 6 ? j : j + 6;
                ja1[k] = ja0[k] + 6;
            } else if (e < 90) {
                const int i = e - 78;
                ei[k] = i; ej[k] = 12;                              // gradient entry: [Ja | Jo]' r
                ia0[k] = i < 6 ? i : i + 6;
                ja0[k] = 24; ja1[k] = 25;
            }
        }
        for (int c = gwarp; c < P.npchunk; c += gwarps) {
            const int2 ch = P.pair_chunk[c];
            const int cnt = ch.y - ch.x;                             // <= PCH = 32: lane q looks after observation q
            int pq = 0, onq = 0;
            if (lane < cnt) {
                pq = P.pair_perm[ch.x + lane];
                onq = (P.active[pq] && !(P.obs_type && P.obs_type[pq] == 2)) ? 1 : 0;
            }
            const int pf = __shfl_sync(FULL, pq, 0);
            const int sa = s_slot[P.lm_anchor_cam[P.obs_lm[pf]]], so = s_slot[P.obs_cam[pf]];
            if (sa < 0 && so < 0) continue;                         // both keyframes constant / unused (warp-uniform)
            // the whole chunk's rows [Ja | Jo | r] go to this warp's staging slice with every load in flight at once (staging
            // four observations at a time left the phase waiting on one L2 round trip per stage: 4.1 ms of a batched C3 solve)
            __syncwarp();
            // (two unrolled halves of 13 loads per lane: every load of a half is issued before the first store needs its value -
            //  a rolled load -> store loop waited one L2 round trip per element, 14.6 us per chunk)
            const int tot = cnt * 26;
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                double vals[13];
#pragma unroll
                for (int j = 0; j < 13; ++j) {
                    const int e = (half * 13 + j) * 32 + lane;
                    const bool ok = e < tot;
                    const int q = ok ? e / 26 : 0, k = e - 26 * q;
                    const int p = __shfl_sync(FULL, pq, q);
                    const int on = __shfl_sync(FULL, onq, q);
                    const double* src = k < 12 ? P.Ja + 12 * (size_t)p + k : (k < 24 ? P.Jo + 12 * (size_t)p + (k - 12) : P.Jr + 2 * (size_t)p + (k - 24));
                    vals[j] = (ok && on) ? *src : 0.0;
                }
#pragma unroll
                for (int j = 0; j < 13; ++j) {
                    const int e = (half * 13 + j) * 32 + lane;
                    if (e < tot) st[e] = vals[j];
                }
            }
            __syncwarp();
            double a[3] = {0.0, 0.0, 0.0};
            for (int q = 0; q < cnt; ++q) {
                const double* v = st + 26 * q;
#pragma unroll
                for (int k = 0; k < 3; ++k) a[k] += v[ia0[k]] * v[ja0[k]] + v[ia0[k] + 6] * v[ja1[k]];
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const int i = ei[k], j = ej[k];
                double v = a[k];
                if (i < 0 || v == 0.0) continue;
                if (j == 12) {                                      // F'r
                    if (i < 6) { if (sa >= 0) red_add_f64(cG + 6 * sa + i, v); }
                    else if (so >= 0) red_add_f64(cG + 6 * so + (i - 6), v);
                } else if (j < 6) {                                 // anchor diagonal block (i <= j < 6)
                    if (sa >= 0) {
                        red_add_f64(cS + (size_t)(6 * sa + i) * n + 6 * sa + j, v);
                        if (i == j) red_add_f64(cCn + 6 * sa + i, v);
                    }
                } else if (i >= 6) {                                // observer diagonal block
                    if (so >= 0) {
                        red_add_f64(cS + (size_t)(6 * so + (i - 6)) * n + 6 * so + (j - 6), v);
                        if (i == j) red_add_f64(cCn + 6 * so + (i - 6), v);
                    }
                } else if (sa >= 0 && so >= 0) {                    // cross block Ja' Jo into the upper block (min slot, max slot)
                    const int ca = i, cb = j - 6;
                    if (sa < so) red_add_f64(cS + (size_t)(6 * sa + ca) * n + 6 * so + cb, v);
                    else if (sa > so) red_add_f64(cS + (size_t)(6 * so + cb) * n + 6 * sa + ca, v);
                    else {                                          // same pose block twice: Ja'Jo + Jo'Ja lands in its diagonal block
                        if (ca == cb) { v *= 2.0; red_add_f64(cCn + 6 * sa + ca, v); }
                        const int lo = ca < cb ? ca : cb, hi = ca < cb ? cb : ca;
                        red_add_f64(cS + (size_t)(6 * sa + lo) * n + 6 * sa + hi, v);
                    }
                }
            }
        }
    }
    __syncthreads();
    if (tracing) P.trace[15] += global_ns() - t_b1;                 // trace slot 15 = B1 share of B:schur in this mode
    // ---------------- B2: landmark part
    // S -= sum_rows w y y' is the one contraction of this phase: FP64 tensor cores (DMMA m8n8k4), a warp owns up to NT 8 x 8
    // tiles of the upper triangle and keeps their accumulators in registers over ALL rounds; per 4-row step and tile two
    // shared-memory loads (tile pitch = 4 mod 16 doubles: conflict-free half-warps) and one DMMA.
    constexpr int R = WARPS * (32 / SG);                            // tile rows (landmarks per round and CTA)
    const int TP = owner_tile_pitch(n);
    double* tw = s_tile + (size_t)R * TP;
    double* tg = tw + R;
    const int nb8 = (n + 7) >> 3, ntile = nb8 * (nb8 + 1) / 2;
    int bi[NT], bj[NT];
    double acc[NT][2];
#pragma unroll
    for (int k = 0; k < NT; ++k) {
        const int t = warp + WARPS * k;
        bi[k] = -1; bj[k] = 0;
        if (t < ntile) {
            int i = 0, rem = t;
            while (rem >= nb8 - i) { rem -= nb8 - i; ++i; }
            bi[k] = i; bj[k] = i + rem;
        }
        acc[k][0] = 0.0; acc[k][1] = 0.0;
    }
    double racc = 0.0, gmax_lm = 0.0;
    const int sub = lane / SG, sl = lane - sub * SG;
    const int myrow = warp * (32 / SG) + sub;
    const int fg = lane >> 2, ft = lane & 3;                        // DMMA fragment coordinates
    for (int l0 = bid * R; l0 < P.npts; l0 += G * R) {
        for (int e = tid; e < R * TP + 2 * R; e += THREADS) s_tile[e] = 0.0;
        __syncthreads();
        {
            const int l = l0 + myrow;
            double w, g;
            owner_fill_row<SG>(P, s_slot, l, sl, l < P.npts, radius, first_iter, s_tile + (size_t)myrow * TP, w, g, gmax_lm);
            if (sl == 0) { tw[myrow] = w; tg[myrow] = g; }
        }
        __syncthreads();
        const int rows = min(R, P.npts - l0);
        for (int k0 = 0; k0 < rows; k0 += 4) {                      // rows beyond `rows` are zero rows with w = 0
            const double* yk = s_tile + (size_t)(k0 + ft) * TP;
            const double wv = tw[k0 + ft];
#pragma unroll
            for (int k = 0; k < NT; ++k) {
                if (bi[k] < 0) continue;                            // warp-uniform
                dmma_884(acc[k][0], acc[k][1], yk[8 * bi[k] + fg] * wv, yk[8 * bj[k] + fg]);
            }
        }
        if (tid < n) {
            double ra = 0.0;
            for (int r = 0; r < rows; ++r) ra += s_tile[(size_t)r * TP + tid] * (tw[r] * tg[r]);
            racc -= ra;
        }
        __syncthreads();
    }
    // flush: every upper-triangle entry of this CTA's partial system has exactly one owner
#pragma unroll
    for (int k = 0; k < NT; ++k) {
        if (bi[k] < 0) continue;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int r = 8 * bi[k] + fg, c = 8 * bj[k] + 2 * ft + e;
            const double v = acc[k][e];
            if (r <= c && c < n && v != 0.0) red_add_f64(cS + (size_t)r * n + c, -v);
        }
    }
    if (tid < n && racc != 0.0) red_add_f64(cRhs + tid, racc);
    gmax_lm = warp_max(gmax_lm);
    if (lane == 0 && gmax_lm > 0.0) atomic_max_pos(scal + SC_GMAX_LM, gmax_lm);
}

// ------------------------------------------------------------------ reduced camera system, n <= 96: CTA-wide Gauss-Jordan in shared memory
// Augmented system [S + D | b] in shared memory (row pitch n + 2); pivot step j updates every row r != j for the columns
// c > j: A[r][c] -= (A[r][j] / A[j][j]) A[j][c].  Row j and column j are not written in step j, so ONE block barrier per
// pivot suffices and no substitution passes follow (a Cholesky + two triangular solves is 3n dependent steps).  Pivots
// equal those of the LDL' / Cholesky factorisation (no pivoting: S is SPD after LM damping), so "pivot <= 0" is the
// failure test Ceres' LLT applies.  Four threads per row; a thread stages the pivot-row and own-row entries of its
// columns in registers first (all shared-memory loads in flight together), then updates and stores.
template <int QMAX>
__device__ __forceinline__ void gj_pivots(double* sA, int n, int PIT, int* s_fail) {
    const int tid = threadIdx.x, nt = blockDim.x;
    const int sub = tid & 3, r0 = tid >> 2, rows_per_pass = nt >> 2;
    for (int j = 0; j < n; ++j) {
        const double p = sA[j * PIT + j];
        if (!(p > 0.0) || !isfinite(p)) { if (tid == 0) *s_fail = 1; break; }   // uniform: every thread reads the same pivot
        // 1 / p sits on the critical path of every pivot (B200: ~50 cycles per DEPENDENT fp64 operation - the 48-pivot loop
        // is latency bound on this chain): MUFU double-precision seed (2^-23) + two Newton steps, no float round trip
        double ip;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(ip) : "d"(p));
        ip = fma(ip, fma(-p, ip, 1.0), ip);
        ip = fma(ip, fma(-p, ip, 1.0), ip);
        const double* rowj = sA + j * PIT;
        const int c0 = j + 1 + sub;
        const int nq = (n - j + 3 - sub) >> 2;              // columns c = c0 + 4 q <= n
        double pj[QMAX];
#pragma unroll
        for (int q = 0; q < QMAX; ++q) pj[q] = q < nq ? rowj[c0 + 4 * q] : 0.0;
        for (int r = r0; r < n; r += rows_per_pass) {
            if (r == j) continue;
            double* rowr = sA + r * PIT;
            const double f = rowr[j] * ip;
            double a[QMAX];
#pragma unroll
            for (int q = 0; q < QMAX; ++q) a[q] = q < nq ? rowr[c0 + 4 * q] : 0.0;
#pragma unroll
            for (int q = 0; q < QMAX; ++q) a[q] -= f * pj[q];
#pragma unroll
            for (int q = 0; q < QMAX; ++q)
                if (q < nq) rowr[c0 + 4 * q] = a[q];
        }
        __syncthreads();
    }
}

// Two pivots per barrier (n <= 48).  The 48-pivot loop above is a latency chain: barrier -> pivot read -> reciprocal ->
// row factor -> update -> store, ~0.5 us per pivot, 24 us of a 75 us LM iteration of a single C3 window.  Eliminating
// columns j and j+1 in one step halves the barriers and overlaps the second reciprocal with the first update's loads:
//   a = A[j][j], b = A[j][j+1], c = A[j+1][j], d = A[j+1][j+1];   m = c / a;   d' = d - m b   (the SAME second pivot the
//   scalar loop meets);   row j+1 := row j+1 - m row j;   row j := row j - (b / d') row j+1;   every other row r:
//   f0 = A[r][j] / a,  f1 = (A[r][j+1] - f0 b) / d',  row r -= f0 row j(old) + f1 row j+1(new).
// Rows j and j+1 are rewritten in their own step, so the step's readers take them from a double-buffered copy (pbuf) that
// the rows' owners filled at the end of the previous step.
template <int QMAX>
__device__ __forceinline__ void gj_pivots2(double* sA, int n, int PIT, double* pbuf, int* s_fail) {
    const int tid = threadIdx.x, nt = blockDim.x;
    const int sub = tid & 3, r0 = tid >> 2, rows_per_pass = nt >> 2;
    for (int e = tid; e < 2 * PIT; e += nt) pbuf[e] = sA[e];        // rows 0 and 1 -> parity 0
    __syncthreads();
    for (int j = 0; j < n; j += 2) {
        const int par = (j >> 1) & 1;
        const double* P0 = pbuf + (size_t)(2 * par) * PIT;
        const double* P1 = P0 + PIT;
        double* N0 = pbuf + (size_t)(2 * (par ^ 1)) * PIT;
        double* N1 = N0 + PIT;
        const double a = P0[j], b = P0[j + 1], c = P1[j], d = P1[j + 1];
        if (!(a > 0.0) || !isfinite(a)) { if (tid == 0) *s_fail = 1; break; }   // uniform: every thread reads the same pivots
        double ip0;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(ip0) : "d"(a));
        ip0 = fma(ip0, fma(-a, ip0, 1.0), ip0);
        ip0 = fma(ip0, fma(-a, ip0, 1.0), ip0);
        const double m = c * ip0;
        const double d2 = d - m * b;
        if (!(d2 > 0.0) || !isfinite(d2)) { if (tid == 0) *s_fail = 1; break; }
        double ip1;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(ip1) : "d"(d2));
        ip1 = fma(ip1, fma(-d2, ip1, 1.0), ip1);
        ip1 = fma(ip1, fma(-d2, ip1, 1.0), ip1);
        const double g = b * ip1;
        const int c0 = j + 2 + sub;
        const int nq = (n - j + 2 - sub) >> 2;              // columns c = c0 + 4 q <= n
        double p0[QMAX], p1[QMAX];
#pragma unroll
        for (int q = 0; q < QMAX; ++q) {
            p0[q] = q < nq ? P0[c0 + 4 * q] : 0.0;
            p1[q] = q < nq ? P1[c0 + 4 * q] - m * p0[q] : 0.0;
        }
        for (int r = r0; r < n; r += rows_per_pass) {
            double* rowr = sA + r * PIT;
            double v[QMAX];
            if (r == j) {
#pragma unroll
                for (int q = 0; q < QMAX; ++q) v[q] = p0[q] - g * p1[q];
            } else if (r == j + 1) {
#pragma unroll
                for (int q = 0; q < QMAX; ++q) v[q] = p1[q];
                if (sub == 0) rowr[j + 1] = d2;              // the diagonal holds the second pivot (z = A[i][n] / A[i][i])
            } else {
                const double f0 = rowr[j] * ip0;
                const double f1 = (rowr[j + 1] - f0 * b) * ip1;
#pragma unroll
                for (int q = 0; q < QMAX; ++q) v[q] = q < nq ? rowr[c0 + 4 * q] : 0.0;
#pragma unroll
                for (int q = 0; q < QMAX; ++q) v[q] -= f0 * p0[q] + f1 * p1[q];
            }
            double* nxt = r == j + 2 ? N0 : (r == j + 3 ? N1 : nullptr);
#pragma unroll
            for (int q = 0; q < QMAX; ++q)
                if (q < nq) {
                    rowr[c0 + 4 * q] = v[q];
                    if (nxt) nxt[c0 + 4 * q] = v[q];
                }
        }
        __syncthreads();
    }
}

__device__ void reduced_solve_small(const Prob& P, double* T, int n, double radius, int first_iter, double* sA, double* scal) {
    const int tid = threadIdx.x, nt = blockDim.x;
    const int PIT = n + 2;
    const bool tr = P.trace != nullptr && tid == 0;          // (CTA 0 only runs this) trace slots 12: load + damping, 13: pivots, 14: solution
    unsigned long long tr_t = tr ? global_ns() : 0;
#define TRS(k) do { if (tr) { const unsigned long long t_ = global_ns(); P.trace[k] += t_ - tr_t; tr_t = t_; } } while (0)
    double* cRhs = T; double* cG = T + n; double* cCn = T + 2 * n; double* cS = T + 3 * n;
    __shared__ int s_fail;
    if (tid == 0) s_fail = 0;
    for (int e = tid; e < n * n; e += nt) {
        const int r = e / n, c = e - r * n;
        sA[r * PIT + c] = r <= c ? cS[(size_t)r * n + c] : cS[(size_t)c * n + r];
    }
    __syncthreads();
    for (int i = tid; i < n; i += nt) {
        const double cn = cCn[i];
        double sc = P.sc_cam[i];
        if (first_iter) {
            sc = 1.0 / (1.0 + sqrt(cn));
            P.sc_cam[i] = sc;
        }
        const double diag = fmin(fmax(cn * sc * sc, 1e-6), 1e32);
        sA[i * PIT + i] += diag / (radius * sc * sc);
        sA[i * PIT + n] = cG[i] + cRhs[i];
    }
    __syncthreads();
    TRS(12);
    if (n <= 48 && P.gj2) gj_pivots2<13>(sA, n, PIT, sA + (size_t)n * PIT, &s_fail);   // two pivots per barrier
    else if (n <= 48) gj_pivots<13>(sA, n, PIT, &s_fail);    // (n + 1 + 3) / 4 columns per thread
    else if (n <= 64) gj_pivots<17>(sA, n, PIT, &s_fail);
    else gj_pivots<25>(sA, n, PIT, &s_fail);
    __syncthreads();
    TRS(13);
    if (s_fail) {
        if (tid == 0) scal[SC_CHOL_FAIL] = 1.0;
        return;
    }
    for (int i = tid; i < n; i += nt) P.z[i] = sA[i * PIT + n] / sA[i * PIT + i];
    TRS(14);
#undef TRS
}

// ------------------------------------------------------------------ reduced camera system, n > 96: blocked Cholesky (one CTA)

// ------------------------------------------------------------------ reduced camera system, n > 96: blocked Cholesky across the group
// Same factorisation as reduced_solve_blocked, but only the sequential part of a block step stays on CTA 0 (diagonal
// block, row panel, forward substitution); the trailing update A22 -= U12' U12 - the one real contraction, (n - c1)^2 x 32
// flops - is spread over every warp of the group (FP64 tensor cores, operands read from the row panel in L2).  Two group
// barriers per block step; 9 steps for the 288 x 288 system of a 48-keyframe window.
__device__ void reduced_solve_blocked_group(const Prob& P, double* T, int n, double radius, int first_iter, double* sP, double* scal,
                                            GroupBar& bar, int bid, int G) {
    const int tid = threadIdx.x, nt = blockDim.x;
    double* cRhs = T; double* cG = T + n; double* cCn = T + 2 * n; double* A = T + 3 * n;
    __shared__ double s_w[MAX_N];
    __shared__ double sU[CH_NB][CH_NB + 1];
    __shared__ double s_idiag_all[MAX_N + CH_NB];
    __shared__ double s_t[CH_NB];
    __shared__ int s_bad;
    double* w = s_w;
    const int PW = ((n + 15) & ~15) + 8;                 // row pitch of the panel (doubles)
    double* Pan = P.panel;                               // [CH_NB][PW] in global memory: what the other CTAs read
    const int warp = tid >> 5, lane = tid & 31, nwarp = nt >> 5;
    const int gwarps = G * nwarp, gwarp = bid * nwarp + warp;
    const bool tr = P.trace != nullptr && bid == 0 && tid == 0;
    unsigned long long tr_t = tr ? global_ns() : 0;
#define TRS(k) do { if (tr) { const unsigned long long t_ = global_ns(); P.trace[k] += t_ - tr_t; tr_t = t_; } } while (0)
    if (bid == 0) {
        if (tid == 0) s_bad = 0;
        for (int i = tid; i < n; i += nt) {
            const double cn = cCn[i];
            double sc = P.sc_cam[i];
            if (first_iter) {
                sc = 1.0 / (1.0 + sqrt(cn));
                P.sc_cam[i] = sc;
            }
            const double diag = fmin(fmax(cn * sc * sc, 1e-6), 1e32);
            A[(size_t)i * n + i] += diag / (radius * sc * sc);
            w[i] = cG[i] + cRhs[i];
        }
        __syncthreads();
    }
    for (int kb = 0; kb < n; kb += CH_NB) {
        const int nb = min(CH_NB, n - kb), c1 = kb + nb, m = n - c1;
        const int m16 = (m + 15) & ~15;
        if (bid == 0) {
            double* s_idiag = s_idiag_all + kb;
            for (int e = tid; e < CH_NB * CH_NB; e += nt) {
                const int i = e >> 5, j = e & 31;
                sU[i][j] = (i < nb && j < nb && i <= j) ? A[(size_t)(kb + i) * n + kb + j] : (i == j ? 1.0 : 0.0);
            }
            __syncthreads();
            if (warp == 0) {
                // One warp, lane = column, the column's 32 rows in REGISTERS (fully unrolled): per pivot the dependent
                // chain is shuffle -> MUFU rsqrt seed + two Newton steps -> scale -> one shared-memory row broadcast ->
                // 31 independent FMAs.  (The shared-memory read-modify-write form this replaces serialised ~16 row
                // updates per pivot on the ~50-cycle fp64 latency: 1.5 k cycles per pivot, 25 us per block step.)
                bool bad = false;
                double a[CH_NB];
#pragma unroll
                for (int r = 0; r < CH_NB; ++r) a[r] = sU[r][lane];
#pragma unroll
                for (int j = 0; j < CH_NB; ++j) {
                    const double d = __shfl_sync(FULL, a[j], j);
                    bad = bad || !(d > 1e-30) || !(d < 1e30);
                    double is;
                    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(is) : "d"(d));
                    is = fma(0.5 * is, fma(-d * is, is, 1.0), is);
                    is = fma(0.5 * is, fma(-d * is, is, 1.0), is);
                    const double ujc = lane >= j ? a[j] * is : 0.0;
                    sU[j][lane] = ujc;                     // row j of U: final value, and the broadcast source below
                    if (lane == j) s_idiag[j] = is;
                    __syncwarp();
                    // (measured alternatives, both slower: broadcasting U[j][r] by shuffle - no warp barrier in the chain, but
                    // 62 SHFL per pivot: +40 %; for the Gauss-Jordan above, forming the next pivot's reciprocal one step ahead,
                    // redundantly in every thread or in a dedicated warp: +10 % - the pivot chain is not what bounds a step)
#pragma unroll
                    for (int r = j + 1; r < CH_NB; ++r) a[r] = fma(-sU[j][r], ujc, a[r]);   // entries below the diagonal (r > lane) are never read
                }
                if (bad && lane == 0) { s_bad = 1; scal[SC_CHOL_FAIL] = 1.0; }
            }
            __syncthreads();
            if (!s_bad) {
                for (int e = tid; e < CH_NB * CH_NB; e += nt) {
                    const int i = e >> 5, j = e & 31;
                    if (i < nb && j < nb && i <= j) A[(size_t)(kb + i) * n + kb + j] = sU[i][j];
                }
                for (int cc = tid; cc <= m16; cc += nt) {
                    if (cc >= m && cc < m16) {                                   // zero padding of the operand panel
#pragma unroll
                        for (int i = 0; i < CH_NB; ++i) { sP[i * PW + cc] = 0.0; Pan[i * PW + cc] = 0.0; }
                        continue;
                    }
                    const bool is_rhs = cc == m16;
                    if (!is_rhs && cc >= m) continue;
                    double a[CH_NB];
#pragma unroll
                    for (int i = 0; i < CH_NB; ++i)
                        a[i] = i < nb ? (is_rhs ? w[kb + i] : A[(size_t)(kb + i) * n + c1 + cc]) : 0.0;
#pragma unroll
                    for (int k = 0; k < CH_NB; ++k) {
                        const double x = a[k] * s_idiag[k];
                        a[k] = x;
#pragma unroll
                        for (int i = k + 1; i < CH_NB; ++i) a[i] -= sU[k][i] * x;
                    }
                    if (is_rhs) {
#pragma unroll
                        for (int i = 0; i < CH_NB; ++i) if (i < nb) { w[kb + i] = a[i]; s_t[i] = a[i]; }
                    } else {
#pragma unroll
                        for (int i = 0; i < CH_NB; ++i) {
                            sP[i * PW + cc] = a[i];
                            Pan[i * PW + cc] = a[i];
                            if (i < nb) A[(size_t)(kb + i) * n + c1 + cc] = a[i];
                        }
                    }
                }
            }
        }
        TRS(12);
        bar.sync();
        TRS(13);
        if (scal[SC_CHOL_FAIL] != 0.0) return;                           // uniform across the group (written before the barrier)
        if (bid == 0) {
            for (int r = tid; r < m; r += nt) {
                double acc = 0.0;
#pragma unroll 8
                for (int k = 0; k < CH_NB; ++k) acc += sP[k * PW + r] * s_t[k];
                w[c1 + r] -= acc;
            }
        }
        {
            const int mt = m16 >> 4, g = lane >> 2, t = lane & 3;
            for (int idx = gwarp; idx < mt * mt; idx += gwarps) {
                const int tr = idx / mt, tc = idx - tr * mt;
                if (tr > tc) continue;
                const int r0 = tr * 16, q0 = tc * 16;
                double acc[2][2][2] = {{{0.0, 0.0}, {0.0, 0.0}}, {{0.0, 0.0}, {0.0, 0.0}}};
#pragma unroll
                for (int k0 = 0; k0 < CH_NB; k0 += 4) {
                    const double* pk = Pan + (size_t)(k0 + t) * PW;
                    const double a0 = pk[r0 + g], a1 = pk[r0 + 8 + g];
                    const double b0 = pk[q0 + g], b1 = pk[q0 + 8 + g];
                    dmma_884(acc[0][0][0], acc[0][0][1], a0, b0);
                    dmma_884(acc[0][1][0], acc[0][1][1], a0, b1);
                    dmma_884(acc[1][0][0], acc[1][0][1], a1, b0);
                    dmma_884(acc[1][1][0], acc[1][1][1], a1, b1);
                }
#pragma unroll
                for (int hi = 0; hi < 2; ++hi)
#pragma unroll
                    for (int hj = 0; hj < 2; ++hj)
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const int r = r0 + 8 * hi + g, c = q0 + 8 * hj + 2 * t + e;
                            if (r <= c && c < m) A[(size_t)(c1 + r) * n + c1 + c] -= acc[hi][hj][e];
                        }
            }
        }
        TRS(14);
        bar.sync();
        TRS(13);
    }
    if (bid != 0) return;
    // ---- backward substitution U z = y, last block first (CTA 0)
    for (int kb = ((n - 1) / CH_NB) * CH_NB; kb >= 0; kb -= CH_NB) {
        const int nb = min(CH_NB, n - kb), c1 = kb + nb;
        for (int e = tid; e < CH_NB * CH_NB; e += nt) {
            const int i = e >> 5, j = e & 31;
            sU[i][j] = (i < nb && j < nb && i <= j) ? A[(size_t)(kb + i) * n + kb + j] : (i == j ? 1.0 : 0.0);
        }
        for (int i = warp; i < nb; i += nwarp) {
            double acc = 0.0;
            for (int c = c1 + lane; c < n; c += 32) acc += A[(size_t)(kb + i) * n + c] * w[c];
            acc = warp_sum(acc);
            if (lane == 0) s_t[i] = w[kb + i] - acc;
        }
        __syncthreads();
        if (warp == 0) {
            double ti = lane < nb ? s_t[lane] : 0.0;
            const double idg = lane < nb ? s_idiag_all[kb + lane] : 1.0;
#pragma unroll
            for (int j = CH_NB - 1; j >= 0; --j) {
                const double zj = __shfl_sync(FULL, ti * idg, j);
                if (lane < j) ti -= sU[lane][j] * zj;
                if (lane == j && j < nb) w[kb + j] = zj;
            }
        }
        __syncthreads();
    }
    for (int i = tid; i < n; i += nt) P.z[i] = w[i];
    TRS(15);
#undef TRS
}

// ------------------------------------------------------------------ multi-GPU exchange (peer memory over NVLink)
// Every rank exports one buffer (see ba_lm.cuh); xsync() is a barrier between the ranks' kernels: CTA 0 / thread 0
// writes its epoch into slot `rank` of every peer's flag array (release, system scope) and waits until every peer
// has written the same epoch into ours.  Must be bracketed by group barriers.
__device__ __forceinline__ void xsync(const Peers& X, unsigned long long& xepoch, unsigned* abort) {
    xepoch++;
    __threadfence_system();
    for (int r = 0; r < X.world; ++r)
        if (r != X.rank) st_release_sys(reinterpret_cast<unsigned long long*>(X.base[r]) + X.rank, xepoch);
    for (int r = 0; r < X.world; ++r) {
        if (r == X.rank) continue;
        const unsigned long long* f = reinterpret_cast<const unsigned long long*>(X.base[X.rank]) + r;
        unsigned spins = 0;
        unsigned long long t0 = 0;
        while (ld_acquire_sys(f) < xepoch) {
            if ((++spins & 255u) == 0) {
                if (ld_acquire_gpu(abort)) break;
                const unsigned long long t = global_ns();
                if (t0 == 0) t0 = t;
                else if (t - t0 > XSYNC_TIMEOUT_NS) { atomicExch(abort, 1u); break; }
            }
        }
    }
    __threadfence_system();
}

__device__ __forceinline__ double ld_peer(const double* p) {
    double v;
    asm volatile("ld.volatile.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}

// ------------------------------------------------------------------ the persistent solve kernel
struct SolveOut { int iterations; double initial_cost, final_cost; int termination; };

__global__ void __launch_bounds__(THREADS, 2) ba_lm_kernel(const Prob* __restrict__ probs, int nprob, int G, Peers X) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ lmctl::State S;
    __shared__ int s_action, s_ncv, s_any, s_refine, s_trivial, s_lock;
    __shared__ double s_red[WARPS][4];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int group = blockIdx.x / G, bid = blockIdx.x - group * G, ngroups = gridDim.x / G;
    if (group >= ngroups) return;
    unsigned long long xepoch = X.epoch0;
    __shared__ Prob sProb;
    for (int pi = group; pi < nprob; pi += ngroups) {
        __syncthreads();
        for (int i = tid; i < (int)(sizeof(Prob) / sizeof(int)); i += THREADS)
            reinterpret_cast<int*>(&sProb)[i] = reinterpret_cast<const int*>(probs + pi)[i];
        __syncthreads();
        const Prob& P = sProb;
        GroupBar bar{P.bar, P.bar + 1, (unsigned)G, 0u};
        // optional phase trace (CTA 0 / thread 0): time since the previous mark is charged to phase k
        unsigned long long tr_last = 0, tr_acc[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
        const bool tracing = P.trace != nullptr && bid == 0 && tid == 0;
        if (tracing) tr_last = global_ns();
#define TR(k) do { if (tracing) { const unsigned long long t_ = global_ns(); tr_acc[k] += t_ - tr_last; tr_last = t_; } } while (0)
        // shared memory carve-up
        double* s_cam = reinterpret_cast<double*>(smem_raw);                       // [ncam][12]
        int* s_slot = reinterpret_cast<int*>(s_cam + 12 * (size_t)P.ncam);         // [ncam]
        double* s_work = reinterpret_cast<double*>(smem_raw + P.smem_work_off);    // Schur scratch / solve area (union)
        const int etf_stride = 6 * (P.ncv_max + 1);
        double* s_etf = s_work + (size_t)warp * etf_stride;
        int* s_eslot = reinterpret_cast<int*>(s_work + (size_t)WARPS * etf_stride) + warp * (P.ncv_max + 1);
        double* sJ = s_work + (size_t)WARPS * etf_stride + (((size_t)WARPS * (P.ncv_max + 1) + 1) >> 1) + (size_t)warp * (28 * SCH);
        int* smeta = reinterpret_cast<int*>(s_work + (size_t)WARPS * etf_stride + (((size_t)WARPS * (P.ncv_max + 1) + 1) >> 1) + (size_t)WARPS * (28 * SCH)) + warp * SCH;
        const int gthreads = G * THREADS, gtid = bid * THREADS + tid;
        const int gwarps = G * WARPS, gwarp = bid * WARPS + warp;
        const size_t blk = P.blk;                                                  // doubles per accumulation copy (n_max based)
        int xi = 0;                                                                // index of the buffer holding x
        int use_huber = P.use_robust;
        int n_out1 = 0, n_out2 = 0;
        SolveOut so[2];
        so[0] = SolveOut{0, 0.0, 0.0, 0};
        so[1] = SolveOut{0, 0.0, 0.0, 0};
        int ran_refine = 0;
        for (int stage = 0; stage < 2; ++stage) {
            const int max_iters = stage == 0 ? P.max_it1 : P.max_it2;
            uint8_t* cam_used = P.cam_used + (size_t)stage * P.ncam;
            double* x_pose = P.pose[xi]; double* c_pose = P.pose[xi ^ 1];
            double* x_invd = P.invd[xi]; double* c_invd = P.invd[xi ^ 1];
            // ---- set-up: Program::RemoveFixedBlocks (keyframes that are constant or touch no active residual drop out),
            //      candidate := x for the blocks that are not in this solve's program, accumulators zeroed
            // (flags are collected per CTA in shared memory first: thousands of stores from every SM to the same few bytes
            //  serialise in L2 - measured 7 us per CTA of the group)
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
            for (size_t i = gtid; i < (size_t)P.ncopy * blk; i += gthreads) P.acc[i] = 0.0;
            for (int i = gtid; i < 2 * SC_COUNT; i += gthreads) P.scal[i] = 0.0;
            TR(stage == 0 ? 0 : 10);
            bar.sync();
            TR(stage == 0 ? 11 : 10);
            if (X.world > 1) {
                // a keyframe is in the program if ANY rank has an active residual touching it
                uint8_t* mine = reinterpret_cast<uint8_t*>(X.base[X.rank]) + XB_CAMUSED + (size_t)stage * MAX_CAMS;
                for (int i = gtid; i < P.ncam; i += gthreads) mine[i] = cam_used[i];
                bar.sync();
                if (bid == 0 && tid == 0) xsync(X, xepoch, P.bar + 1);
                bar.sync();
                for (int c = tid; c < P.ncam; c += THREADS) {
                    int u = 0;
                    for (int r = 0; r < X.world; ++r)
                        u |= *reinterpret_cast<volatile const uint8_t*>(reinterpret_cast<const uint8_t*>(X.base[r]) + XB_CAMUSED + (size_t)stage * MAX_CAMS + c);
                    s_slot[c] = (u ? 1 : 0) | (P.pose_const[c] ? 2 : 0);          // temporarily: used / constant flags
                }
            } else {
                for (int c = tid; c < P.ncam; c += THREADS) s_slot[c] = (cam_used[c] ? 1 : 0) | (P.pose_const[c] ? 2 : 0);
            }
            __syncthreads();
            if (tid == 0) {
                int ncv = 0, any = 0;
                for (int c = 0; c < P.ncam; ++c) {
                    const int u = s_slot[c];
                    any |= u & 1;
                    s_slot[c] = u == 1 ? ncv++ : -1;
                }
                s_ncv = ncv; s_any = any;
                lmctl::init(S);
            }
            __syncthreads();
            const int ncv = s_ncv, n = 6 * ncv;
            if (!s_any) { if (stage == 0) break; else continue; }   // no residual blocks (on any rank)
            if (bid == 0)
                for (int c = tid; c < P.ncam; c += THREADS) P.cam_slot[c] = s_slot[c];
            double* T = (P.ncopy > 1 || X.world > 1) ? P.total : P.acc;      // the system the solve reads
            TR(0);
            // ---- LM iterations
            for (;;) {
                if (tid == 0) s_action = lmctl::begin_iteration(S, max_iters) ? 1 : 0;
                __syncthreads();
                if (!s_action) break;
                const int par = S.iteration & 1, first_iter = S.first_iter, x_is_new = S.x_is_new;
                const double radius = S.radius;
                double* scal = P.scal + par * SC_COUNT;
                // ---- A: residual blocks + Jacobians at x
                if (x_is_new) {
                    stage_cams(P, x_pose, s_cam);
                    __syncthreads();
                    double cost = 0.0;
                    for (int i = gtid; i < P.nobs; i += gthreads)
                        if (P.active[i]) cost += eval_block<true>(P, i, P.obs_lm[i], s_cam, x_invd[P.obs_lm[i]], use_huber);
                    cost = warp_sum(cost);
                    if (lane == 0) s_red[warp][0] = cost;
                    __syncthreads();
                    if (tid == 0) {                               // one atomic per CTA: they all hit one address
                        double a = 0.0;
                        for (int w_ = 0; w_ < WARPS; ++w_) a += s_red[w_][0];
                        if (a != 0.0) red_add_f64(scal + SC_COST, a);
                    }
                }
                bar.sync();
                TR(1);
                // ---- B: Schur elimination into this CTA's accumulation copy (global, RED) or shared-memory block (lock)
                if (P.schur_smem == 3) {
                    // owner mode (n <= 96): pair-sorted Gram blocks + dense landmark rows, no per-observation reductions
#define OV2_OWNER(NT_) do { if (P.sg == 4) schur_owner_phase<NT_, 4>(P, s_slot, s_work, n, radius, first_iter, bid, G, scal); \
                            else if (P.sg == 8) schur_owner_phase<NT_, 8>(P, s_slot, s_work, n, radius, first_iter, bid, G, scal); \
                            else schur_owner_phase<NT_, 32>(P, s_slot, s_work, n, radius, first_iter, bid, G, scal); } while (0)
                    if (n <= 48) OV2_OWNER(3);            // 21 upper 8 x 8 tiles over 8 warps
                    else if (n <= 72) OV2_OWNER(6);       // 45
                    else OV2_OWNER(10);                   // 78 (n = 96)
#undef OV2_OWNER
                } else if (P.schur_smem == 2) {
                    // per-WARP private copies of [rhs | F'r | column norms | S] in shared memory: plain read-modify-writes, no
                    // lock, no RED; the CTA sums its copies and sends the non-zeros to the global block once per phase
                    const int live_s = 3 * n + n * n;
                    double* mine = s_work + P.smem_sacc_off + (size_t)warp * live_s;
                    for (int e = lane; e < live_s; e += 32) mine[e] = 0.0;
                    __syncwarp();
                    double gmax_lm = 0.0;
                    for (int l = gwarp; l < P.npts; l += gwarps) schur_landmark<true>(P, s_slot, s_etf, s_eslot, sJ, smeta, l, lane, radius, first_iter, mine, n, gmax_lm, nullptr);
                    if (lane == 0 && gmax_lm > 0.0) atomic_max_pos(scal + SC_GMAX_LM, gmax_lm);
                    __syncthreads();
                    const double* all = s_work + P.smem_sacc_off;
                    for (int e = tid; e < live_s; e += THREADS) {
                        double v = 0.0;
#pragma unroll
                        for (int w_ = 0; w_ < WARPS; ++w_) v += all[(size_t)w_ * live_s + e];
                        if (v != 0.0) red_add_f64(P.acc + e, v);
                    }
                } else if (P.schur_smem) {
                    double* sS = s_work + P.smem_sacc_off;
                    const int live_s = 3 * n + n * n;
                    for (int e = tid; e < live_s; e += THREADS) sS[e] = 0.0;
                    if (tid == 0) s_lock = 0;
                    __syncthreads();
                    double gmax_lm = 0.0;
                    for (int l = gwarp; l < P.npts; l += gwarps) schur_landmark<true>(P, s_slot, s_etf, s_eslot, sJ, smeta, l, lane, radius, first_iter, sS, n, gmax_lm, &s_lock);
                    if (lane == 0 && gmax_lm > 0.0) atomic_max_pos(scal + SC_GMAX_LM, gmax_lm);
                    __syncthreads();
                    for (int e = tid; e < live_s; e += THREADS) {
                        const double v = sS[e];
                        if (v != 0.0) red_add_f64(P.acc + e, v);
                    }
                } else {
                    double* acc = P.acc + (size_t)(bid % P.ncopy) * blk;
                    double gmax_lm = 0.0;
                    for (int l = gwarp; l < P.npts; l += gwarps) schur_landmark<false>(P, s_slot, s_etf, s_eslot, sJ, smeta, l, lane, radius, first_iter, acc, n, gmax_lm, nullptr);
                    if (lane == 0 && gmax_lm > 0.0) atomic_max_pos(scal + SC_GMAX_LM, gmax_lm);
                }
                bar.sync();
                TR(2);
                // ---- B2: fold the copies; multi-GPU: sum the ranks' partial systems out of peer memory
                const int live = 3 * n + n * n;
                if (X.world > 1) {
                    double* mine = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(X.base[X.rank]) + XB_PARTIAL) + (size_t)par * (SC_COUNT + blk);
                    for (int e = gtid; e < live; e += gthreads) {
                        double a = P.acc[e];
                        for (int k = 1; k < P.ncopy; ++k) a += P.acc[e + (size_t)k * blk];
                        mine[SC_COUNT + e] = a;
                    }
                    if (gtid < SC_COUNT) mine[gtid] = scal[gtid];
                    bar.sync();
                    if (bid == 0 && tid == 0) xsync(X, xepoch, P.bar + 1);
                    bar.sync();
                    for (int e = gtid; e < live; e += gthreads) {
                        double a = 0.0;
                        for (int r = 0; r < X.world; ++r)
                            a += ld_peer(reinterpret_cast<const double*>(reinterpret_cast<const unsigned char*>(X.base[r]) + XB_PARTIAL) + (size_t)par * (SC_COUNT + blk) + SC_COUNT + e);
                        T[e] = a;
                    }
                    if (gtid == 0) {
                        double c = 0.0, g = 0.0;
                        for (int r = 0; r < X.world; ++r) {
                            const double* pr = reinterpret_cast<const double*>(reinterpret_cast<const unsigned char*>(X.base[r]) + XB_PARTIAL) + (size_t)par * (SC_COUNT + blk);
                            c += ld_peer(pr + SC_COST);
                            g = fmax(g, ld_peer(pr + SC_GMAX_LM));
                        }
                        scal[SC_COST] = c;        // the whole window's cost / gradient bound, identical on every rank
                        scal[SC_GMAX_LM] = g;
                    }
                    bar.sync();
                } else if (P.ncopy > 1) {
                    for (int e = gtid; e < live; e += gthreads) {
                        double a = P.acc[e];
                        for (int k = 1; k < P.ncopy; ++k) a += P.acc[e + (size_t)k * blk];
                        T[e] = a;
                    }
                    bar.sync();
                }
                TR(3);
                // ---- C: reduced camera system (CTA 0); gradient projection |x - Plus(x, -g)|_inf (last CTA); the other
                //      CTAs clear the accumulation copies for the next iteration (T is separate whenever ncopy > 1)
                const bool group_solve = P.solve_blocked && n > 0;
                if (bid == 0 && !group_solve && n > 0) reduced_solve_small(P, T, n, radius, first_iter, s_work, scal);
                if (bid == G - 1 && x_is_new && n > 0) {
                    if (bid == 0) __syncthreads();
                    double gm = 0.0;
                    for (int c = tid; c < P.ncam; c += THREADS) {
                        const int s = s_slot[c];
                        if (s < 0) continue;
                        double d[6], out[7];
                        for (int k = 0; k < 6; ++k) d[k] = -T[n + 6 * s + k];
                        pose_plus(x_pose + 7 * c, d, out);
                        for (int k = 0; k < 7; ++k) gm = fmax(gm, fabs(x_pose[7 * c + k] - out[k]));
                    }
                    gm = warp_max(gm);
                    if (lane == 0) atomic_max_pos(scal + SC_GMAX_CAM, gm);
                }
                if (group_solve) reduced_solve_blocked_group(P, T, n, radius, first_iter, s_work, scal, bar, bid, G);
                TR(4);
                bar.sync();
                TR(5);
                // ---- D: candidate keyframe poses (every CTA, into shared memory), back-substitution, candidate cost
                {
                    double st2 = 0.0, cx2 = 0.0;
                    for (int c = tid; c < P.ncam; c += THREADS) {
                        const int s = s_slot[c];
                        double out[7];
                        if (s >= 0) {
                            double d[6];
                            for (int k = 0; k < 6; ++k) d[k] = -P.z[6 * s + k];
                            pose_plus(x_pose + 7 * c, d, out);
                            for (int k = 0; k < 7; ++k) {
                                const double df = x_pose[7 * c + k] - out[k];
                                st2 += df * df; cx2 += out[k] * out[k];
                            }
                            if (bid == 0)
                                for (int k = 0; k < 7; ++k) c_pose[7 * c + k] = out[k];
                        } else {
                            for (int k = 0; k < 7; ++k) out[k] = x_pose[7 * c + k];
                        }
                        double t[3], q[4], R[9];
                        load_pose(out, t, q);
                        quat_to_rot(q, R);
                        for (int k = 0; k < 9; ++k) s_cam[12 * c + k] = R[k];
                        s_cam[12 * c + 9] = t[0]; s_cam[12 * c + 10] = t[1]; s_cam[12 * c + 11] = t[2];
                    }
                    __syncthreads();
                    double mcc = 0.0, cost = 0.0, lst2 = 0.0, lcx2 = 0.0;
                    if (P.sg == 4) {
                        for (int l0 = gwarp * 8; l0 < P.npts; l0 += gwarps * 8)
                            backsub_landmarks_sg<4>(P, s_slot, s_cam, l0, lane, x_invd, c_invd, use_huber, mcc, lst2, lcx2, cost);
                    } else if (P.sg == 8) {
                        for (int l0 = gwarp * 4; l0 < P.npts; l0 += gwarps * 4)
                            backsub_landmarks_sg<8>(P, s_slot, s_cam, l0, lane, x_invd, c_invd, use_huber, mcc, lst2, lcx2, cost);
                    } else {
                        for (int l = gwarp; l < P.npts; l += gwarps)
                            backsub_landmark(P, s_slot, s_cam, l, lane, x_invd, c_invd, use_huber, mcc, lst2, lcx2, cost);
                    }
                    // the keyframe part of the norms counts once per window (rank 0, CTA 0)
                    if (bid == 0 && X.rank == 0) { lst2 += st2; lcx2 += cx2; }
                    mcc = warp_sum(mcc); cost = warp_sum(cost); lst2 = warp_sum(lst2); lcx2 = warp_sum(lcx2);
                    if (lane == 0) { s_red[warp][0] = cost; s_red[warp][1] = mcc; s_red[warp][2] = lst2; s_red[warp][3] = lcx2; }
                    __syncthreads();
                    if (tid < 4) {
                        double a = 0.0;
                        for (int w_ = 0; w_ < WARPS; ++w_) a += s_red[w_][tid];
                        if (a != 0.0) red_add_f64(scal + SC_CAND_COST + tid, a);
                    }
                    // clear for the next iteration: accumulation copies and the other parity's scalars
                    for (size_t i = gtid; i < (size_t)P.ncopy * blk; i += gthreads) P.acc[i] = 0.0;
                    double* oscal = P.scal + (par ^ 1) * SC_COUNT;
                    if (gtid < SC_COUNT) oscal[gtid] = 0.0;
                }
                bar.sync();
                TR(6);
                if (X.world > 1) {
                    // second, tiny exchange: candidate cost, model cost change, step / candidate norms (rank order sum)
                    double* mine = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(X.base[X.rank]) + XB_SC4) + par * 8;
                    if (gtid < 4) mine[gtid] = scal[SC_CAND_COST + gtid];
                    bar.sync();
                    if (bid == 0 && tid == 0) xsync(X, xepoch, P.bar + 1);
                    bar.sync();
                }
                // ---- E: trust-region controller, replayed by every CTA
                if (tid == 0) {
                    double v[4];
                    if (X.world > 1) {
                        for (int k = 0; k < 4; ++k) {
                            double a = 0.0;
                            for (int r = 0; r < X.world; ++r)
                                a += ld_peer(reinterpret_cast<const double*>(reinterpret_cast<const unsigned char*>(X.base[r]) + XB_SC4) + par * 8 + k);
                            v[k] = a;
                        }
                    } else {
                        for (int k = 0; k < 4; ++k) v[k] = scal[SC_CAND_COST + k];
                    }
                    const double gmax = fmax(scal[SC_GMAX_LM], scal[SC_GMAX_CAM]);
                    s_action = (int)lmctl::end_iteration(S, scal[SC_COST], v[0], v[1], v[2], v[3], gmax, scal[SC_CHOL_FAIL] != 0.0, P.ftol);
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
            so[stage].iterations = S.iteration;
            so[stage].initial_cost = S.initial_cost;
            so[stage].final_cost = lmctl::final_cost(S);
            so[stage].termination = S.termination;
            if (stage == 1) ran_refine = 1;
            // a stop while a candidate was pending leaves buffers unequal for out-of-program blocks only at the
            // next set-up (which copies x over the candidate), so nothing to repair here
            bar.sync();
            // ---- outlier scan on the values the LAST evaluation left behind (optimizer.cpp:500-530, :637-735)
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
                        if (deact) P.active[i] = 0;   // problem.RemoveResidualBlock
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
                if (tid < 3) {                                   // one atomic per CTA and counter
                    double a = 0.0;
                    for (int w_ = 0; w_ < WARPS; ++w_) a += s_red[w_][tid];
                    if (a != 0.0) red_add_f64(cnt + tid, a);
                }
                // the stop request lives in mapped HOST memory: ONE thread of the group reads it (every thread of every CTA
                // polling it over PCIe cost 7 us per CTA of the group) and publishes it next to the counters
                if (stage == 0 && bid == 0 && tid == 0)
                    cnt[3] = (P.stop_flag && *reinterpret_cast<volatile const int*>(P.stop_flag) != 0) ? 1.0 : 0.0;
                bar.sync();
                if (stage == 0) {
                    double nbad = cnt[0], nleft = cnt[1], nright = cnt[2];
                    n_out1 = (int)nbad;
                    if (X.world > 1) {
                        // every rank must take the same branch: counts summed over the ranks
                        double* mine = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(X.base[X.rank]) + XB_SC4) + 16;
                        if (gtid < 3) mine[gtid] = cnt[gtid];
                        bar.sync();
                        if (bid == 0 && tid == 0) xsync(X, xepoch, P.bar + 1);
                        bar.sync();
                        nbad = nleft = nright = 0.0;
                        for (int r = 0; r < X.world; ++r) {
                            const double* pr = reinterpret_cast<const double*>(reinterpret_cast<const unsigned char*>(X.base[r]) + XB_SC4) + 16;
                            nbad += ld_peer(pr); nleft += ld_peer(pr + 1); nright += ld_peer(pr + 2);
                        }
                    }
                    // solve #2 only if residual blocks were removed and no stop was requested meanwhile (optimizer.cpp:603-604)
                    int refine = P.apply_l2 && P.use_robust && nbad > 0.0;
                    if (refine && cnt[3] != 0.0) refine = 0;        // (sharded callers pass no stop flag: ranks could disagree)
                    // mono windows keep the Huber loss in the refinement; the wrapper is reset to the trivial loss only when
                    // left-camera and other-frame right-camera residual lists are both non-empty (optimizer.cpp:606-608)
                    int trivial = P.refine_loss;
                    if (trivial < 0) trivial = (nleft > 0.0 && nright > 0.0) ? 1 : 0;
                    if (tid == 0) { s_refine = refine; s_trivial = trivial; }
                    __syncthreads();
                    if (!s_refine) break;
                    use_huber = s_trivial ? 0 : 1;
                } else {
                    n_out2 = (int)cnt[0];
                }
            }
        }
        // ---- write-back: x into buffer 0, result record
        TR(8);
        bar.sync();
        if (xi == 1) {
            for (int i = gtid; i < 7 * P.ncam; i += gthreads) P.pose[0][i] = P.pose[1][i];
            for (int i = gtid; i < P.npts; i += gthreads) P.invd[0][i] = P.invd[1][i];
        }
        if (bid == 0 && tid == 0) {
            Result* R = P.result;
            R->iters_robust = so[0].iterations;
            R->iters_refine = ran_refine ? so[1].iterations : 0;
            const SolveOut& last = ran_refine ? so[1] : so[0];
            R->initial_cost = last.initial_cost;
            R->final_cost = last.final_cost;
            R->termination = last.termination;
            R->n_outliers_first = n_out1;
            R->n_outliers_second = n_out2;
            R->aborted = (int)ld_acquire_gpu(P.bar + 1);
        }
        TR(9);
        if (tracing)
            for (int k = 0; k < 12; ++k) P.trace[k] = tr_acc[k];
#undef TR
    }
}

}  // namespace balm

// ====================================================================== host side
using namespace balm;

namespace {

struct HostPlan {
    size_t off_prob, off_pose, off_invd, off_apx, off_opx, off_lac, off_oc, off_ol, off_lp, off_pc, off_ty, in_bytes;   // uploaded block
    size_t off_pp, off_pch; int pch_cap, sg;   // owner mode: pair-sorted permutation, chunk table (capacity), lanes per landmark
    // device-only work areas (offsets into the work block)
    size_t w_pose1, w_invd1, w_active, w_flags, w_camused, w_camslot, w_Jr, w_Ja, w_Jo, w_Jl, w_chi2, w_dpos, w_sclm, w_ete, w_ge,
           w_acc, w_total, w_scal, w_z, w_panel, w_sccam, w_counts, w_bar, w_result, w_trace, work_bytes, zero_off, zero_bytes;
    size_t out_result, out_flags, act_rel;   // offsets inside the batch's output region / 'active' region (set up by balm_solve)
    int ncv_max, n_max, ncopy, solve_blocked, schur_smem;
    size_t blk, smem_work_off, smem_bytes, smem_sacc_off;
};

size_t take(size_t& off, size_t bytes, size_t align = 256) {
    off = (off + align - 1) & ~(align - 1);
    const size_t o = off;
    off += bytes;
    return o;
}

}  // namespace

// Plans one window: offsets of its inputs inside the upload block and of its work areas inside the work block.
static ov2_status plan_window(ov2_ctx* ctx, const ov2_ba_problem* pb, int world, size_t& st_off, size_t& in_off, size_t& work_off,
                              size_t& zero_off, size_t& out_off, size_t& act_off, HostPlan& H, int ncopy_cap, bool single_window) {
    const int ncam = pb->ncam, npts = pb->npts, nobs = pb->nobs;
    int ncv = 0;
    for (int c = 0; c < ncam; ++c) ncv += pb->pose_const[c] ? 0 : 1;
    if (ncv > MAX_VAR_CAMS) return ov2_fail(ctx, OV2_ERR_CAPACITY, "ov2_localba_solve: more than 64 optimised keyframes");
    if (ncam > MAX_CAMS) return ov2_fail(ctx, OV2_ERR_CAPACITY, "ov2_localba_solve: more than 256 keyframes in the window");
    H.ncv_max = ncv; H.n_max = 6 * ncv;
    H.blk = 3 * (size_t)H.n_max + (size_t)H.n_max * H.n_max;
    if (H.blk == 0) H.blk = 1;
    // ONE accumulation block: privatised copies (round 1 used up to 8) do not pay on a B200 - the phase is bound by the
    // rate at which an SM retires fp64 REDs, not by same-address contention (measured: identical time with 1 and 8 copies)
    // - and a single copy needs no fold phase.  OV2_BA_NCOPY = 2..8 brings the copies back for experiments.
    (void)ncopy_cap;
    H.ncopy = 1;
    if (getenv("OV2_BA_NCOPY")) { int e = atoi(getenv("OV2_BA_NCOPY")); if (e >= 1 && e <= 8 && (size_t)e * H.blk <= (size_t)(3 * MAX_N + MAX_N * MAX_N)) H.ncopy = e; }
    H.solve_blocked = H.n_max > 96 ? 1 : 0;
    // states (pose, inverse depth) of all windows sit together at the head of the block: they are what comes back
    H.off_pose = take(st_off, sizeof(double) * 7 * ncam, 16);
    H.off_invd = take(st_off, sizeof(double) * (size_t)(npts > 0 ? npts : 1), 16);
    H.off_prob = take(in_off, sizeof(Prob));
    H.off_apx = take(in_off, sizeof(double) * 2 * (size_t)(npts > 0 ? npts : 1));
    H.off_opx = take(in_off, sizeof(double) * 2 * (size_t)(nobs > 0 ? nobs : 1));
    H.off_lac = take(in_off, sizeof(int32_t) * (size_t)(npts > 0 ? npts : 1));
    H.off_oc = take(in_off, sizeof(int32_t) * (size_t)(nobs > 0 ? nobs : 1));
    H.off_ol = take(in_off, sizeof(int32_t) * (size_t)(nobs > 0 ? nobs : 1));
    H.off_lp = take(in_off, sizeof(int32_t) * (size_t)(npts + 1));
    H.off_pc = take(in_off, (size_t)ncam);
    H.off_ty = take(in_off, pb->obs_type ? (size_t)(nobs > 0 ? nobs : 1) : 0);
    {
        // owner-mode Schur (n <= 96): observations sorted by (anchor keyframe, observing keyframe) + chunk table
        const size_t ngmax = (size_t)ncam * ncam < (size_t)(nobs > 0 ? nobs : 1) ? (size_t)ncam * ncam : (size_t)(nobs > 0 ? nobs : 1);
        H.pch_cap = (int)((size_t)(nobs > 0 ? nobs : 1) / PCH + ngmax + 1);
        H.off_pp = take(in_off, sizeof(int32_t) * (size_t)(nobs > 0 ? nobs : 1));
        H.off_pch = take(in_off, sizeof(int2) * (size_t)H.pch_cap);
        const double avg = npts > 0 ? (double)nobs / (double)npts : 0.0;
        H.sg = avg <= 5.0 ? 4 : (avg <= 12.0 ? 8 : 32);
        if (getenv("OV2_BA_SG")) { const int e = atoi(getenv("OV2_BA_SG")); if (e == 4 || e == 8 || e == 32) H.sg = e; }
    }
    const size_t no = nobs > 0 ? nobs : 1, np = npts > 0 ? npts : 1;
    // results (Result record + outlier flags) of all windows sit together in the output region, the 'active' bytes of all
    // windows in another: one memset each and ONE D2H for a whole batch (w_flags / w_result / w_active are made absolute
    // offsets by balm_solve once every window is planned)
    H.out_result = take(out_off, sizeof(Result), 64);
    H.out_flags = take(out_off, no, 64);
    H.act_rel = take(act_off, no, 64);
    // zero-initialised small arrays of all windows: a region of their own (relative offsets until balm_solve places it)
    H.w_camused = take(zero_off, 2 * (size_t)ncam);
    H.w_counts = take(zero_off, sizeof(double) * 8);
    H.w_bar = take(zero_off, sizeof(unsigned) * 4);
    H.w_trace = take(zero_off, sizeof(unsigned long long) * 16);
    H.w_sclm = take(zero_off, sizeof(double) * np);
    H.w_sccam = take(zero_off, sizeof(double) * MAX_N);
    H.w_pose1 = take(work_off, sizeof(double) * 7 * ncam);
    H.w_invd1 = take(work_off, sizeof(double) * np);
    H.w_camslot = take(work_off, sizeof(int32_t) * ncam);
    H.w_Jr = take(work_off, sizeof(double) * 2 * no);
    H.w_Ja = take(work_off, sizeof(double) * 12 * no);
    H.w_Jo = take(work_off, sizeof(double) * 12 * no);
    H.w_Jl = take(work_off, sizeof(double) * 2 * no);
    H.w_chi2 = take(work_off, sizeof(double) * no);
    H.w_dpos = take(work_off, no);
    H.w_ete = take(work_off, sizeof(double) * np);
    H.w_ge = take(work_off, sizeof(double) * np);
    H.w_acc = take(work_off, sizeof(double) * (size_t)H.ncopy * H.blk);
    H.w_total = take(work_off, sizeof(double) * H.blk);
    H.w_scal = take(work_off, sizeof(double) * 2 * SC_COUNT);
    H.w_z = take(work_off, sizeof(double) * MAX_N);
    H.w_panel = take(work_off, sizeof(double) * CH_NB * (size_t)(MAX_N + 24));
    // dynamic shared memory: [keyframes 12 doubles each][slots][union: Schur scratch | solve area]
    size_t s = sizeof(double) * 12 * (size_t)ncam + sizeof(int) * (size_t)ncam;
    s = (s + 15) & ~(size_t)15;
    H.smem_work_off = s;
    size_t schur = (size_t)WARPS * 6 * (size_t)(ncv + 1) * sizeof(double) + ((((size_t)WARPS * (ncv + 1) + 1) >> 1) << 3) +
                   (size_t)WARPS * 28 * SCH * sizeof(double) + (size_t)WARPS * SCH * sizeof(int) + 16;
    schur = (schur + 15) & ~(size_t)15;
    const size_t solve = H.solve_blocked ? (size_t)CH_NB * (size_t)((((size_t)H.n_max + 15) & ~(size_t)15) + 8) * sizeof(double)
                                         : (size_t)(H.n_max + 4) * (size_t)(H.n_max + 2) * sizeof(double);   // + 4 rows: pivot-row double buffer of gj_pivots2
    // shared-memory accumulation of the reduced system (behind the Schur scratch) when the whole block fits next to it
    // with two CTAs per SM still possible
    H.smem_sacc_off = schur / sizeof(double);
    H.schur_smem = 0;
    // (opt-in, OV2_BA_SCHUR_SMEM=1: measured 6x SLOWER than the RED path on a B200 - C3, 64 CTAs: 317 us vs 53 us per
    //  Schur phase; the lock serialises the eight warps of a CTA for the whole commit.  Kept because it is tested and
    //  documents the negative result.)
    const char* ssm = getenv("OV2_BA_SCHUR_SMEM");
    if (H.n_max > 0 && s + schur + H.blk * sizeof(double) <= 100 * 1024 && ssm && atoi(ssm) == 1) {
        H.schur_smem = 1;
        H.ncopy = 1;
        schur += H.blk * sizeof(double);
    } else if (H.n_max > 0 && s + schur + (size_t)WARPS * H.blk * sizeof(double) <= 190 * 1024 && !(ssm && atoi(ssm) == 0) &&
               (single_window || (ssm && atoi(ssm) == 2))) {
        // mode 2 (default for a single window when it fits: reduced systems up to n = 54): one private block per warp, one
        // CTA per SM.  Batches keep the RED path: there two CTAs per SM (different windows overlapping their latency-bound
        // phases) are worth more than the faster accumulation - measured 5.1 k vs 4.1 k solves/s on the C3 batch.
        H.schur_smem = 2;
        H.ncopy = 1;
        schur += (size_t)WARPS * H.blk * sizeof(double);
    }
    // mode 3 (default up to n = 96, single windows and batches): owner mode, see schur_owner_phase
    // Single windows spread over many CTAs stay on mode 2 when it fits (measured C3: 119 us vs 236 us per solve in the
    // Schur phase at 148 CTAs - there the phase is latency, not RED bound); batches (1-2 CTAs per window) take mode 3.
    if (H.n_max > 0 && H.n_max <= 96 && ((ssm && atoi(ssm) == 3) || (!ssm && !(single_window && H.schur_smem == 2)))) {
        const size_t R = (size_t)WARPS * (32 / H.sg);
        size_t tile = (R * (size_t)owner_tile_pitch(H.n_max) + 2 * R) * sizeof(double);
        const size_t stage = (size_t)WARPS * PCH * 26 * sizeof(double);
        if (tile < stage) tile = stage;
        H.schur_smem = 3;
        H.ncopy = 1;
        schur = (tile + 15) & ~(size_t)15;
    }
    H.smem_bytes = s + (schur > solve ? schur : solve) + 16;
    (void)world;
    return OV2_OK;
}

// The scalar part of a window's Prob record: sizes, calibration, stereo extrinsic, loss and solver options.
void balm_prob_scalars(const ov2_ba_problem* pb, const ov2_ba_opts* opts, Prob& P, const double* Kh, const double* krh, const double* trlh) {
    memset(&P, 0, sizeof(P));
    P.ncam = pb->ncam; P.npts = pb->npts; P.nobs = pb->nobs;
    P.fx = Kh[0]; P.fy = Kh[1]; P.cx = Kh[2]; P.cy = Kh[3];
    P.rfx = P.fx; P.rfy = P.fy; P.rcx = P.cx; P.rcy = P.cy;
    for (int k = 0; k < 9; ++k) P.Rrl[k] = (k % 4 == 0) ? 1.0 : 0.0;
    if (pb->obs_type) {
        P.rfx = krh[0]; P.rfy = krh[1]; P.rcx = krh[2]; P.rcy = krh[3];
        const double qn = sqrt(trlh[3] * trlh[3] + trlh[4] * trlh[4] + trlh[5] * trlh[5] + trlh[6] * trlh[6]);
        const double x = trlh[3] / qn, y = trlh[4] / qn, z = trlh[5] / qn, w = trlh[6] / qn;
        const double R[9] = {1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                             2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                             2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)};
        for (int k = 0; k < 9; ++k) P.Rrl[k] = R[k];
        P.trl[0] = trlh[0]; P.trl[1] = trlh[1]; P.trl[2] = trlh[2];
    }
    P.th_f = (float)opts->huber_th;                       // const float mono_th (optimizer.cpp:47)
    P.huber_a = (double)sqrtf(P.th_f);                    // HuberLoss(std::sqrt(mono_th))
    P.huber_b = P.huber_a * P.huber_a;
    P.use_robust = opts->use_robust ? 1 : 0;
    P.apply_l2 = opts->apply_l2_after_robust ? 1 : 0;
    P.refine_loss = opts->refine_loss;
    P.max_it1 = opts->max_iters_robust; P.max_it2 = opts->max_iters_refine;
    P.ftol = opts->function_tolerance;
}

static void fill_prob(const ov2_ba_problem* pb, const ov2_ba_opts* opts, const HostPlan& H, char* din, char* dwork, Prob& P,
                      const double* Kh, const double* krh, const double* trlh, const int* stop_flag_dev) {
    balm_prob_scalars(pb, opts, P, Kh, krh, trlh);
    P.stop_flag = stop_flag_dev;
    P.pose_const = (const uint8_t*)(din + H.off_pc);
    P.lm_anchor_cam = (const int32_t*)(din + H.off_lac);
    P.lm_anchor_px = (const double*)(din + H.off_apx);
    P.obs_cam = (const int32_t*)(din + H.off_oc);
    P.obs_lm = (const int32_t*)(din + H.off_ol);
    P.obs_px = (const double*)(din + H.off_opx);
    P.obs_type = pb->obs_type ? (const uint8_t*)(din + H.off_ty) : nullptr;
    P.lm_ptr = (const int32_t*)(din + H.off_lp);
    P.pose[0] = (double*)(din + H.off_pose); P.pose[1] = (double*)(dwork + H.w_pose1);
    P.invd[0] = (double*)(din + H.off_invd); P.invd[1] = (double*)(dwork + H.w_invd1);
    P.active = (uint8_t*)(dwork + H.w_active); P.flags = (uint8_t*)(dwork + H.w_flags);
    P.cam_used = (uint8_t*)(dwork + H.w_camused); P.cam_slot = (int32_t*)(dwork + H.w_camslot);
    P.Jr = (double*)(dwork + H.w_Jr); P.Ja = (double*)(dwork + H.w_Ja); P.Jo = (double*)(dwork + H.w_Jo); P.Jl = (double*)(dwork + H.w_Jl);
    P.chi2 = (double*)(dwork + H.w_chi2); P.dpos = (uint8_t*)(dwork + H.w_dpos);
    P.sc_lm = (double*)(dwork + H.w_sclm); P.ete = (double*)(dwork + H.w_ete); P.ge = (double*)(dwork + H.w_ge);
    P.acc = (double*)(dwork + H.w_acc); P.total = (double*)(dwork + H.w_total); P.scal = (double*)(dwork + H.w_scal);
    P.z = (double*)(dwork + H.w_z); P.sc_cam = (double*)(dwork + H.w_sccam); P.panel = (double*)(dwork + H.w_panel);
    P.counts = (double*)(dwork + H.w_counts); P.bar = (unsigned*)(dwork + H.w_bar); P.result = (Result*)(dwork + H.w_result);
    P.trace = getenv("OV2_BA_TRACE") ? (unsigned long long*)(dwork + H.w_trace) : nullptr;
    P.ncv_max = H.ncv_max; P.ncopy = H.ncopy; P.blk = H.blk; P.solve_blocked = H.solve_blocked;
    P.sg = H.sg;   // lanes per landmark in the per-landmark phases
    // two-pivot Gauss-Jordan steps for n <= 48: opt-in (OV2_BA_GJ2=1).  Measured on a B200 (C3, 148 CTAs): pivot loop 172 us vs
    // 152 us per solve with one pivot per barrier - the longer dependent chain of a step (two reciprocals + the second
    // pivot's elimination) and 26 more live registers cost more than the 24 saved barriers.  Kept: tested, documents the result.
    P.gj2 = getenv("OV2_BA_GJ2") ? atoi(getenv("OV2_BA_GJ2")) : 0;
    P.schur_smem = H.schur_smem; P.smem_sacc_off = (int)H.smem_sacc_off;
    P.pair_perm = (const int32_t*)(din + H.off_pp); P.pair_chunk = (const int2*)(din + H.off_pch); P.npchunk = 0;
    P.smem_work_off = (int)H.smem_work_off;
}

static ov2_status host_copy(ov2_ctx* ctx, void* dst, const void* src, size_t bytes, bool maybe_device = true) {
    if (bytes == 0) return OV2_OK;
    if (maybe_device && ov2_is_device_ptr(src)) OV2_CUDA(ctx, cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
    else memcpy(dst, src, bytes);
    return OV2_OK;
}

// Solves `nprob` windows with one launch.  peers: multi-GPU exchange description (world 1 = none).
ov2_status balm_solve(ov2_ctx* ctx, int nprob, const ov2_ba_problem* pbs, const ov2_ba_opts* opts, ov2_ba_result* results,
                      uint8_t* const* outlier_outs, const Peers* peers, const int* stop_flag_dev) {
    if (!ctx || nprob <= 0 || !pbs || !opts || !results) return ov2_fail(ctx, OV2_ERR_INVALID, "ov2_localba_solve: bad arguments");
    ov2_status st = ov2_begin(ctx);
    if (st != OV2_OK) return st;
    const int world = peers ? peers->world : 1;
    std::vector<HostPlan> plans(nprob);
    std::vector<ov2_ba_problem> hp(nprob);           // host-resident views of every window (device inputs are copied down)
    std::vector<std::vector<char>> hold;              // storage for inputs that came as device pointers
    std::vector<char> win_on_device(nprob, 0);
    size_t st_off = 0, in_off = 0, work_off = 0, zero_off = 0, out_off = 0, act_off = 0;
    size_t smem_max = 0;
    int gmax_work = 1;
    for (int k = 0; k < nprob; ++k) {
        const ov2_ba_problem& pb = pbs[k];
        if (pb.ncam <= 0 || pb.npts < 0 || pb.nobs < 0 || (world == 1 && pb.npts <= 0))
            return ov2_fail(ctx, OV2_ERR_INVALID, "ov2_localba_solve: bad arguments");
        hp[k] = pb;
        // the flattened window is host data in the reference's flow (optimizer.cpp:43-430); device-resident inputs are
        // accepted and staged through the host once (the solve itself never leaves the device)
        // cudaPointerGetAttributes costs ~1.5 us on a plain host pointer: 15 queries per window were 6 ms of a 296-window batch.
        // One query per window: a window whose `pose` array is host memory is taken to be host memory throughout (the
        // reference's flow, optimizer.cpp:43-430); only windows whose poses live on the device are inspected array by array.
        const bool win_dev = ov2_is_device_ptr(pb.pose);
        win_on_device[k] = win_dev ? 1 : 0;
        cudaError_t pull_err = cudaSuccess;
        auto pull = [&](const void* p, size_t bytes) -> const void* {
            if (!p || bytes == 0 || !win_dev || !ov2_is_device_ptr(p)) return p;
            hold.emplace_back(bytes);
            const cudaError_t ce = cudaMemcpy(hold.back().data(), p, bytes, cudaMemcpyDeviceToHost);
            if (ce != cudaSuccess) pull_err = ce;
            return hold.back().data();
        };
        hp[k].K = (const double*)pull(pb.K, 32);
        hp[k].pose_const = (const uint8_t*)pull(pb.pose_const, pb.ncam);
        hp[k].lm_anchor_cam = (const int32_t*)pull(pb.lm_anchor_cam, sizeof(int32_t) * (size_t)pb.npts);
        hp[k].lm_anchor_px = (const double*)pull(pb.lm_anchor_px, sizeof(double) * 2 * (size_t)pb.npts);
        hp[k].obs_cam = (const int32_t*)pull(pb.obs_cam, sizeof(int32_t) * (size_t)pb.nobs);
        hp[k].obs_lm = (const int32_t*)pull(pb.obs_lm, sizeof(int32_t) * (size_t)pb.nobs);
        hp[k].obs_px = (const double*)pull(pb.obs_px, sizeof(double) * 2 * (size_t)pb.nobs);
        hp[k].obs_type = (const uint8_t*)pull(pb.obs_type, (size_t)pb.nobs);
        hp[k].Kr = (const double*)pull(pb.Kr, 32);
        hp[k].Trl = (const double*)pull(pb.Trl, 56);
        if (pull_err != cudaSuccess) return ov2_fail(ctx, OV2_ERR_CUDA, "ov2_localba_solve: staging a device-resident window", pull_err);
        if (pb.obs_type && (!pb.Kr || !pb.Trl)) return ov2_fail(ctx, OV2_ERR_INVALID, "ov2_localba_solve: obs_type given without Kr / Trl");
        if ((st = plan_window(ctx, &hp[k], world, st_off, in_off, work_off, zero_off, out_off, act_off, plans[k], 8, nprob == 1)) != OV2_OK) return st;
        if (plans[k].smem_bytes > smem_max) smem_max = plans[k].smem_bytes;
        const int wk = (pb.nobs + THREADS - 1) / THREADS;
        const int wl = (pb.npts + WARPS - 1) / WARPS;                  // a landmark per warp and phase (single window: every SM helps)
        const int w = wk > wl ? wk : wl;
        if (w > gmax_work) gmax_work = w;
    }
    if (smem_max > 200 * 1024) return ov2_fail(ctx, OV2_ERR_CAPACITY, "ov2_localba_solve: window needs more than 200 KB of shared memory");
    // ---- pack the inputs into one pinned block: ONE H2D copy for the whole batch.  Layout: [states | everything else]
    const size_t st_bytes = (st_off + 255) & ~(size_t)255;
    for (int k = 0; k < nprob; ++k) {
        HostPlan& H = plans[k];
        for (size_t* f : {&H.off_prob, &H.off_apx, &H.off_opx, &H.off_lac, &H.off_oc, &H.off_ol, &H.off_lp, &H.off_pc, &H.off_ty, &H.off_pp, &H.off_pch}) *f += st_bytes;
    }
    const size_t in_bytes = st_bytes + ((in_off + 255) & ~(size_t)255);
    // work block layout: [per-window work areas | zero region | output region (Result + flags) | 'active' region]
    auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t zbase = al(work_off), zbytes = al(zero_off);
    const size_t obase = zbase + zbytes, obytes = al(out_off);
    const size_t abase = obase + obytes, abytes = al(act_off);
    for (int k = 0; k < nprob; ++k) {
        HostPlan& H = plans[k];
        for (size_t* f : {&H.w_camused, &H.w_counts, &H.w_bar, &H.w_trace, &H.w_sclm, &H.w_sccam}) *f += zbase;
        H.w_result = obase + H.out_result;
        H.w_flags = obase + H.out_flags;
        H.w_active = abase + H.act_rel;
    }
    const size_t host_need = in_bytes + obytes;      // pinned: [packed inputs / returned states | returned output region]
    if (ctx->ba_ws_cap < host_need) {
        if (ctx->ba_ws) cudaFreeHost(ctx->ba_ws);
        ctx->ba_ws = nullptr; ctx->ba_ws_cap = 0;
        OV2_CUDA(ctx, cudaHostAlloc(&ctx->ba_ws, host_need * 2, cudaHostAllocDefault));
        ctx->ba_ws_cap = host_need * 2;
    }
    char* hpk = (char*)ctx->ba_ws;
    char* hout = hpk + in_bytes;
    void* o = nullptr;
    if ((st = ov2_scratch(ctx, in_bytes, &o)) != OV2_OK) return st;
    char* din = (char*)o;
    if ((st = ov2_scratch(ctx, abase + abytes + 256, &o)) != OV2_OK) return st;
    char* dwork = (char*)o;
    // one window's share of the packing: validation, CSR by landmark, copies into the pinned block, the Prob record.
    // Windows write disjoint parts of the block, so a batch is packed by a few host threads.  Returns an error text.
    auto pack_window = [&](int k) -> const char* {
        const ov2_ba_problem& pb = hp[k];
        const HostPlan& H = plans[k];
        const int ncam = pb.ncam, npts = pb.npts, nobs = pb.nobs;
        // CSR by landmark (observations must be sorted by landmark)
        int32_t* lp = (int32_t*)(hpk + H.off_lp);
        memset(lp, 0, sizeof(int32_t) * (size_t)(npts + 1));
        for (int i = 0; i < nobs; ++i) {
            const int l = pb.obs_lm[i];
            if (l < 0 || l >= npts || (i > 0 && l < pb.obs_lm[i - 1])) return "ov2_localba_solve: obs_lm must be sorted ascending and in range";
            lp[l + 1]++;
        }
        for (int l = 0; l < npts; ++l) lp[l + 1] += lp[l];
        for (int i = 0; i < nobs; ++i)
            if (pb.obs_cam[i] < 0 || pb.obs_cam[i] >= ncam) return "ov2_localba_solve: obs_cam out of range";
        for (int l = 0; l < npts; ++l)
            if (pb.lm_anchor_cam[l] < 0 || pb.lm_anchor_cam[l] >= ncam) return "ov2_localba_solve: lm_anchor_cam out of range";
        if (host_copy(ctx, hpk + H.off_pose, pbs[k].pose, sizeof(double) * 7 * ncam, win_on_device[k] != 0) != OV2_OK) return "ov2_localba_solve: copying the poses failed";
        if (host_copy(ctx, hpk + H.off_invd, pbs[k].lm_invdepth, sizeof(double) * (size_t)npts, win_on_device[k] != 0) != OV2_OK) return "ov2_localba_solve: copying the inverse depths failed";
        memcpy(hpk + H.off_apx, pb.lm_anchor_px, sizeof(double) * 2 * (size_t)npts);
        memcpy(hpk + H.off_opx, pb.obs_px, sizeof(double) * 2 * (size_t)nobs);
        memcpy(hpk + H.off_lac, pb.lm_anchor_cam, sizeof(int32_t) * (size_t)npts);
        memcpy(hpk + H.off_oc, pb.obs_cam, sizeof(int32_t) * (size_t)nobs);
        memcpy(hpk + H.off_ol, pb.obs_lm, sizeof(int32_t) * (size_t)nobs);
        memcpy(hpk + H.off_pc, pb.pose_const, (size_t)ncam);
        if (pb.obs_type) memcpy(hpk + H.off_ty, pb.obs_type, (size_t)nobs);
        Prob P;
        fill_prob(&pb, opts, H, din, dwork, P, pb.K, pb.Kr, pb.Trl, stop_flag_dev);
        if (H.schur_smem == 3) {
            // stable counting sort of the observations by (anchor keyframe, observing keyframe), cut into chunks of <= PCH
            int32_t* perm = (int32_t*)(hpk + H.off_pp);
            int2* chunks = (int2*)(hpk + H.off_pch);
            std::vector<int32_t> head((size_t)ncam * ncam + 1, 0);
            for (int i = 0; i < nobs; ++i) head[(size_t)pb.lm_anchor_cam[pb.obs_lm[i]] * ncam + pb.obs_cam[i] + 1]++;
            for (size_t g = 0; g < (size_t)ncam * ncam; ++g) head[g + 1] += head[g];
            {
                std::vector<int32_t> cur(head.begin(), head.end() - 1);
                for (int i = 0; i < nobs; ++i) perm[cur[(size_t)pb.lm_anchor_cam[pb.obs_lm[i]] * ncam + pb.obs_cam[i]]++] = i;
            }
            int nch = 0;
            for (size_t g = 0; g < (size_t)ncam * ncam; ++g)
                for (int b = head[g]; b < head[g + 1]; b += PCH) {
                    if (nch >= H.pch_cap) return "ov2_localba_solve: pair chunk table overflow";
                    chunks[nch++] = make_int2(b, b + PCH < head[g + 1] ? b + PCH : head[g + 1]);
                }
            P.npchunk = nch;
        }
        memcpy(hpk + H.off_prob, &P, sizeof(P));
        return nullptr;
    };
    {
        int nthr = nprob >= 8 ? 8 : 1;
        const unsigned hc = std::thread::hardware_concurrency();
        if (hc > 0 && (unsigned)nthr > hc) nthr = (int)hc;
        if (getenv("OV2_BA_PACK_THREADS")) { const int e = atoi(getenv("OV2_BA_PACK_THREADS")); if (e >= 1 && e <= 64) nthr = e; }
        std::atomic<int> next(0);
        std::atomic<const char*> perr(nullptr);
        auto worker = [&]() {
            for (int k = next.fetch_add(1); k < nprob; k = next.fetch_add(1)) {
                const char* e = pack_window(k);
                if (e) { perr.store(e); return; }
            }
        };
        if (nthr <= 1) worker();
        else {
            std::vector<std::thread> pool;
            for (int t = 1; t < nthr; ++t) pool.emplace_back(worker);
            worker();
            for (auto& t : pool) t.join();
        }
        if (perr.load()) return ov2_fail(ctx, OV2_ERR_INVALID, perr.load());
    }
    // the Prob records must be contiguous for the kernel: they are the first thing of each window's block, so gather them
    std::vector<Prob> parr(nprob);
    for (int k = 0; k < nprob; ++k) memcpy(&parr[k], hpk + plans[k].off_prob, sizeof(Prob));
    if ((st = ov2_scratch(ctx, sizeof(Prob) * (size_t)nprob, &o)) != OV2_OK) return st;
    Prob* dprobs = (Prob*)o;
    cudaStream_t s = ctx->stream;
    OV2_CUDA(ctx, cudaMemcpyAsync(din, hpk, in_bytes, cudaMemcpyHostToDevice, s));
    if (nprob == 1) dprobs = (Prob*)(din + plans[0].off_prob);
    else OV2_CUDA(ctx, cudaMemcpyAsync(dprobs, parr.data(), sizeof(Prob) * (size_t)nprob, cudaMemcpyHostToDevice, s));   // parr outlives the sync below
    OV2_CUDA(ctx, cudaMemsetAsync(dwork + zbase, 0, zbytes + obytes, s));   // zero region + output region of every window
    OV2_CUDA(ctx, cudaMemsetAsync(dwork + abase, 1, abytes, s));            // every observation starts active
    // ---- launch geometry: G CTAs per window, all groups co-resident (cooperative launch)
    {
        // raised only when a window needs more than any before (a function-attribute change while another stream runs the
        // kernel may serialise with it)
        // (check + set + record under one lock: two host threads with their own contexts may make their first solves concurrently)
        static size_t attr_smem[16] = {0};
        static std::mutex attr_mu;
        std::lock_guard<std::mutex> attr_lock(attr_mu);
        const int dv = ctx->device & 15;
        if (smem_max > attr_smem[dv]) {
            OV2_CUDA(ctx, cudaFuncSetAttribute(ba_lm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
            attr_smem[dv] = smem_max;
        }
    }
    int per_sm = 0;
    OV2_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ba_lm_kernel, THREADS, smem_max));
    if (per_sm < 1) return ov2_fail(ctx, OV2_ERR_CAPACITY, "ov2_localba_solve: kernel does not fit an SM");
    const int resident = per_sm * ctx->sm_count;
    int G = gmax_work < 1 ? 1 : gmax_work;
    // one wave of work per phase at most; more CTAs only add barrier latency
    int gcap = nprob == 1 ? resident : (resident / nprob < 1 ? 1 : resident / nprob);
    if (nprob > 1 && gcap > 16) gcap = 16;
    if (G > gcap) G = gcap;
    if (getenv("OV2_BA_CTAS")) { int e = atoi(getenv("OV2_BA_CTAS")); if (e >= 1 && e <= gcap) G = e; }
    if (world > 1 && G < 2) G = 2;
    int ngroups = nprob < resident / G ? nprob : resident / G;
    if (ngroups < 1) ngroups = 1;
    int grid = ngroups * G;
    Peers X;
    memset(&X, 0, sizeof(X));
    X.world = 1;
    if (peers) X = *peers;
    const Prob* dp = dprobs;
    void* kargs[] = {(void*)&dp, (void*)&nprob, (void*)&G, (void*)&X};
    if (ctx->profiling) ov2_prof_begin(ctx);
    // grid <= resident capacity, so on a GPU this process owns every CTA starts at once whichever launch API is used.  The
    // plain launch is the default: cooperative launches were measured to start their CTAs one after the other (~4 us each)
    // and are not run concurrently with another cooperative kernel (ranks sharing one GPU in the tests); OV2_BA_COOP=1
    // selects cudaLaunchCooperativeKernel (co-residency guaranteed by the driver).  A CTA that never arrives trips the
    // barrier timeout instead of hanging the device.
    const char* coop = getenv("OV2_BA_COOP");
    cudaError_t le;
    if (coop && atoi(coop) != 0) {
        le = cudaLaunchCooperativeKernel((const void*)ba_lm_kernel, dim3(grid), dim3(THREADS), kargs, smem_max, s);
    } else {
        ba_lm_kernel<<<grid, THREADS, smem_max, s>>>(dp, nprob, G, X);
        le = cudaGetLastError();
    }
    ctx->launches++;
    if (le != cudaSuccess) return ov2_fail(ctx, OV2_ERR_CUDA, "ba_lm_kernel launch", le);
    if (ctx->profiling) ov2_prof_end(ctx, "ba_lm_kernel");
    // ---- results: [pose | invd] live in the input block (buffer 0), flags + result record in the work block
    OV2_CUDA(ctx, cudaMemcpyAsync(hpk, din, st_bytes, cudaMemcpyDeviceToHost, s));   // poses and inverse depths of every window: one copy
    OV2_CUDA(ctx, cudaMemcpyAsync(hout, dwork + obase, obytes, cudaMemcpyDeviceToHost, s));   // Result records + outlier flags: one copy
    std::vector<Result> hres(nprob);
    std::vector<char> flags_to_host(nprob, 0);
    for (int k = 0; k < nprob; ++k) {
        if (outlier_outs && outlier_outs[k] && pbs[k].nobs > 0) {
            if (win_on_device[k] && ov2_is_device_ptr(outlier_outs[k])) {
                OV2_CUDA(ctx, cudaMemcpyAsync(outlier_outs[k], dwork + plans[k].w_flags, (size_t)pbs[k].nobs, cudaMemcpyDeviceToDevice, s));
            } else {
                flags_to_host[k] = 1;
            }
        }
    }
    OV2_CUDA(ctx, cudaStreamSynchronize(s));
    for (int k = 0; k < nprob; ++k) memcpy(&hres[k], hout + plans[k].out_result, sizeof(Result));
    if (getenv("OV2_BA_TRACE")) {
        unsigned long long tr[16];
        cudaMemcpy(tr, dwork + plans[0].w_trace, sizeof(tr), cudaMemcpyDeviceToHost);
        static const char* names[16] = {"setup0", "A:eval", "B:schur", "B2:fold", "C:solve", "C:wait", "D:backsub", "E:ctl", "scan", "wb", "setup1", "bar0",
                                        "chol:P1", "chol:bar", "chol:P2", "chol:back|ownerB1"};
        fprintf(stderr, "[ba trace] G=%d grid=%d smem=%zu ncopy=%d smemS=%d |", G, grid, smem_max, plans[0].ncopy, plans[0].schur_smem);
        for (int k = 0; k < 16; ++k) fprintf(stderr, " %s %.1fus", names[k], tr[k] / 1e3);
        fprintf(stderr, "\n");
    }
    bool numeric_fail = false, aborted = false;
    for (int k = 0; k < nprob; ++k) {
        const HostPlan& H = plans[k];
        const size_t pb_bytes = sizeof(double) * 7 * pbs[k].ncam, ib = sizeof(double) * (size_t)pbs[k].npts;
        if (win_on_device[k]) cudaMemcpy(pbs[k].pose, hpk + H.off_pose, pb_bytes, cudaMemcpyHostToDevice);
        else memcpy(pbs[k].pose, hpk + H.off_pose, pb_bytes);
        if (ib) {
            if (win_on_device[k] && ov2_is_device_ptr(pbs[k].lm_invdepth)) cudaMemcpy(pbs[k].lm_invdepth, hpk + H.off_invd, ib, cudaMemcpyHostToDevice);
            else memcpy(pbs[k].lm_invdepth, hpk + H.off_invd, ib);
        }
        if (flags_to_host[k]) memcpy(outlier_outs[k], hout + plans[k].out_flags, (size_t)pbs[k].nobs);
        ov2_ba_result& r = results[k];
        memset(&r, 0, sizeof(r));
        r.iters_robust = hres[k].iters_robust; r.iters_refine = hres[k].iters_refine;
        r.initial_cost = hres[k].initial_cost; r.final_cost = hres[k].final_cost;
        r.n_outliers_first = hres[k].n_outliers_first; r.n_outliers_second = hres[k].n_outliers_second;
        r.termination = hres[k].termination;
        if (r.termination == 2) numeric_fail = true;
        if (hres[k].aborted) aborted = true;
    }
    if (aborted) return ov2_fail(ctx, OV2_ERR_CUDA, "ov2_localba_solve: a barrier timed out (peer rank missing?)");
    if (numeric_fail) return ov2_fail(ctx, OV2_ERR_NUMERIC, "ov2_localba_solve: 5 consecutive invalid steps");
    return OV2_OK;
}
