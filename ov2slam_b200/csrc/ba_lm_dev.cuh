// Device building blocks shared by the persistent local-BA solve kernels: ba_lm_kernel (ba_lm.cu, windows of up to
// 64 optimised keyframes) and ba_large_kernel (ba_large.cu, larger windows).  SE3 helpers, the group barrier, the
// residual blocks, the per-landmark Schur elimination and back-substitution.
#pragma once
#include "ba_lm.cuh"

#include <float.h>
#include <math.h>

namespace balm {

// ------------------------------------------------------------------ small SE3 helpers
__device__ __forceinline__ void quat_to_rot(const double* q, double R[9]) {
    const double x = q[0], y = q[1], z = q[2], w = q[3];
    const double tx = 2 * x, ty = 2 * y, tz = 2 * z;
    const double twx = tx * w, twy = ty * w, twz = tz * w;
    const double txx = tx * x, txy = ty * x, txz = tz * x;
    const double tyy = ty * y, tyz = tz * y, tzz = tz * z;
    R[0] = 1 - (tyy + tzz); R[1] = txy - twz; R[2] = txz + twy;
    R[3] = txy + twz; R[4] = 1 - (txx + tzz); R[5] = tyz - twx;
    R[6] = txz - twy; R[7] = tyz + twx; R[8] = 1 - (txx + tyy);
}

__device__ __forceinline__ void load_pose(const double* p, double t[3], double q[4]) {
    t[0] = p[0]; t[1] = p[1]; t[2] = p[2];
    const double n = 1.0 / sqrt(p[3] * p[3] + p[4] * p[4] + p[5] * p[5] + p[6] * p[6]);  // SE3d(q, t) normalises
    q[0] = p[3] * n; q[1] = p[4] * n; q[2] = p[5] * n; q[3] = p[6] * n;
}

// SE3LeftParameterization::Plus: out = Sophus::SE3d::exp(delta) * (q, t)   (sophus/se3.hpp:763-784, so3.hpp:585-620)
__device__ __noinline__ inline void pose_plus(const double* pose, const double* d, double* out) {
    double t[3], q[4];
    load_pose(pose, t, q);
    const double ox = d[3], oy = d[4], oz = d[5];
    const double th2 = ox * ox + oy * oy + oz * oz;
    double imag, real, theta;
    if (th2 < SOPHUS_EPS * SOPHUS_EPS) {
        theta = 0.0;
        const double th4 = th2 * th2;
        imag = 0.5 - (1.0 / 48.0) * th2 + (1.0 / 3840.0) * th4;
        real = 1.0 - (1.0 / 8.0) * th2 + (1.0 / 384.0) * th4;
    } else {
        theta = sqrt(th2);
        double sh_, ch_;
        sincos(0.5 * theta, &sh_, &ch_);
        imag = sh_ / theta;
        real = ch_;
    }
    const double e[4] = {imag * ox, imag * oy, imag * oz, real};
    double Re[9];
    quat_to_rot(e, Re);
    double V[9];
    if (theta < SOPHUS_EPS) {
        for (int i = 0; i < 9; ++i) V[i] = Re[i];
    } else {
        const double a = (1.0 - cos(theta)) / th2;
        const double b = (theta - sin(theta)) / (th2 * theta);
        const double O[9] = {0, -oz, oy, oz, 0, -ox, -oy, ox, 0};
        double O2[9];
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) O2[3 * i + j] = O[3 * i] * O[j] + O[3 * i + 1] * O[3 + j] + O[3 * i + 2] * O[6 + j];
        for (int i = 0; i < 9; ++i) V[i] = a * O[i] + b * O2[i];
        V[0] += 1.0; V[4] += 1.0; V[8] += 1.0;
    }
    const double et[3] = {V[0] * d[0] + V[1] * d[1] + V[2] * d[2], V[3] * d[0] + V[4] * d[1] + V[5] * d[2],
                          V[6] * d[0] + V[7] * d[1] + V[8] * d[2]};
    double r[4];   // quaternion product (so3.hpp:338-342), then normalisation
    r[3] = e[3] * q[3] - e[0] * q[0] - e[1] * q[1] - e[2] * q[2];
    r[0] = e[3] * q[0] + e[0] * q[3] + e[1] * q[2] - e[2] * q[1];
    r[1] = e[3] * q[1] + e[1] * q[3] + e[2] * q[0] - e[0] * q[2];
    r[2] = e[3] * q[2] + e[2] * q[3] + e[0] * q[1] - e[1] * q[0];
    const double n = 1.0 / sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2] + r[3] * r[3]);
    out[0] = et[0] + Re[0] * t[0] + Re[1] * t[1] + Re[2] * t[2];
    out[1] = et[1] + Re[3] * t[0] + Re[4] * t[1] + Re[5] * t[2];
    out[2] = et[2] + Re[6] * t[0] + Re[7] * t[1] + Re[8] * t[2];
    out[3] = r[0] * n; out[4] = r[1] * n; out[5] = r[2] * n; out[6] = r[3] * n;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(FULL, v, o));
    return v;
}
__device__ __forceinline__ void atomic_max_pos(double* addr, double v) {
    // for non-negative doubles the bit pattern orders like an unsigned integer
    atomicMax(reinterpret_cast<unsigned long long*>(addr), (unsigned long long)__double_as_longlong(v));
}

// ------------------------------------------------------------------ barriers
__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}

// Group barrier: monotonic arrival counter (zeroed by the host before the launch); barrier k completes when the
// counter reaches k * G.  Thread 0 arrives / spins, the rest of the CTA waits at the block barrier.  The gpu-scope
// fences publish this CTA's writes and invalidate its L1 (same construction as cooperative-groups grid.sync()).
// A spin that lasts ~seconds means a peer died: it raises `abort` (sticky) so that every later barrier falls
// through and the kernel drains instead of hanging the device.
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
constexpr unsigned long long BARRIER_TIMEOUT_NS = 30000000000ull;   // 30 s: a CTA that never arrives (includes waiting for CTA 0 inside a rank exchange)
constexpr unsigned long long XSYNC_TIMEOUT_NS = 20000000000ull;     // 20 s: a peer rank that never arrives

struct GroupBar {
    unsigned* count; unsigned* abort; unsigned G; unsigned epoch;
    __device__ __forceinline__ void sync() {
        __syncthreads();
        if (G > 1) {
            if (threadIdx.x == 0) {
                epoch += G;
                __threadfence();
                atomicAdd(count, 1u);
                unsigned spins = 0;
                unsigned long long t0 = 0;
                while (ld_acquire_gpu(count) < epoch) {
                    if ((++spins & 1023u) == 0) {
                        if (ld_acquire_gpu(abort)) break;
                        const unsigned long long t = global_ns();
                        if (t0 == 0) t0 = t;
                        else if (t - t0 > BARRIER_TIMEOUT_NS) { atomicExch(abort, 1u); break; }
                    }
                }
                __threadfence();
            }
            __syncthreads();
        }
    }
};

// ------------------------------------------------------------------ keyframe staging
// Rwc (9) + twc (3) of every keyframe of the window in shared memory: one normalisation + quaternion-to-rotation
// per keyframe and CTA instead of two per residual block.
__device__ __forceinline__ void stage_cams(const Prob& P, const double* __restrict__ pose, double* s_cam) {
    for (int c = threadIdx.x; c < P.ncam; c += blockDim.x) {
        double t[3], q[4], R[9];
        load_pose(pose + 7 * c, t, q);
        quat_to_rot(q, R);
#pragma unroll
        for (int k = 0; k < 9; ++k) s_cam[12 * c + k] = R[k];
        s_cam[12 * c + 9] = t[0]; s_cam[12 * c + 10] = t[1]; s_cam[12 * c + 11] = t[2];
    }
}

// ------------------------------------------------------------------ residual blocks
// One residual block (src/ceres_parametrization.cpp:361-473 left camera; :579-712 right camera, other keyframe;
// :476-577 right camera in the anchor keyframe).  Returns the robustified cost 1/2 rho(s); writes chi2 / depth flag
// (the mutable members the reference's outlier scan reads afterwards) and, with JAC, the corrected Jacobian rows.
template <bool JAC>
__device__ __forceinline__ double eval_block(const Prob& P, int i, int lm, const double* __restrict__ s_cam, double lam, int use_huber) {
    const int ca = P.lm_anchor_cam[lm], co = P.obs_cam[i];
    const double* Rwa = s_cam + 12 * ca; const double* ta = Rwa + 9;
    const double* Rwc = s_cam + 12 * co; const double* to = Rwc + 9;
    const double zanch = 1.0 / lam;
    const double bx = (P.lm_anchor_px[2 * lm] - P.cx) / P.fx, by = (P.lm_anchor_px[2 * lm + 1] - P.cy) / P.fy;
    const double ap[3] = {zanch * bx, zanch * by, zanch};
    const double rp[3] = {Rwa[0] * ap[0] + Rwa[1] * ap[1] + Rwa[2] * ap[2], Rwa[3] * ap[0] + Rwa[4] * ap[1] + Rwa[5] * ap[2],
                          Rwa[6] * ap[0] + Rwa[7] * ap[1] + Rwa[8] * ap[2]};  // Rwanch * anchpt
    const double wp[3] = {rp[0] + ta[0], rp[1] + ta[1], rp[2] + ta[2]};
    const double dv[3] = {wp[0] - to[0], wp[1] - to[1], wp[2] - to[2]};
    const double lc[3] = {Rwc[0] * dv[0] + Rwc[3] * dv[1] + Rwc[6] * dv[2], Rwc[1] * dv[0] + Rwc[4] * dv[1] + Rwc[7] * dv[2],
                          Rwc[2] * dv[0] + Rwc[5] * dv[1] + Rwc[8] * dv[2]};   // Rcw = Rwc^T
    const int typ = P.obs_type ? (int)P.obs_type[i] : 0;
    double cp[3] = {lc[0], lc[1], lc[2]};
    double kfx = P.fx, kfy = P.fy, kcx = P.cx, kcy = P.cy;
    if (typ != 0) {
        const double* sv = typ == 2 ? ap : lc;
        for (int k = 0; k < 3; ++k) cp[k] = P.Rrl[3 * k] * sv[0] + P.Rrl[3 * k + 1] * sv[1] + P.Rrl[3 * k + 2] * sv[2] + P.trl[k];
        kfx = P.rfx; kfy = P.rfy; kcx = P.rcx; kcy = P.rcy;
    }
    const double linvz = 1.0 / cp[2];
    const double r0 = kfx * cp[0] * linvz + kcx - P.obs_px[2 * i];
    const double r1 = kfy * cp[1] * linvz + kcy - P.obs_px[2 * i + 1];
    const double s = r0 * r0 + r1 * r1;
    P.chi2[i] = s;
    P.dpos[i] = cp[2] > 0.0 ? 1 : 0;
    double w = 1.0, cost;
    if (use_huber && s > P.huber_b) {
        const double rs = sqrt(s);
        const double rho1 = fmax(DBL_MIN, P.huber_a / rs);
        cost = 0.5 * (2.0 * P.huber_a * rs - P.huber_b);
        w = sqrt(rho1);
    } else {
        cost = 0.5 * s;
    }
    if (JAC) {
        const double linvz2 = linvz * linvz;
        const double jc[6] = {linvz * kfx, 0.0, -cp[0] * linvz2 * kfx, 0.0, linvz * kfy, -cp[1] * linvz2 * kfy};
        // M = d(camera point)/d(world point): Rcw (left), Rrl Rcw (right, other frame), Rrl (right, anchor frame)
        double M[9];
        if (typ == 0) {
            for (int a = 0; a < 3; ++a)
                for (int b = 0; b < 3; ++b) M[3 * a + b] = Rwc[3 * b + a];
        } else if (typ == 1) {
            for (int a = 0; a < 3; ++a)
                for (int b = 0; b < 3; ++b)
                    M[3 * a + b] = P.Rrl[3 * a] * Rwc[3 * b] + P.Rrl[3 * a + 1] * Rwc[3 * b + 1] + P.Rrl[3 * a + 2] * Rwc[3 * b + 2];
        } else {
            for (int k = 0; k < 9; ++k) M[k] = P.Rrl[k];
        }
        double JR[6];  // J_cam * M  (2x3)
        for (int a = 0; a < 2; ++a)
            for (int b = 0; b < 3; ++b)
                JR[3 * a + b] = jc[3 * a] * M[b] + jc[3 * a + 1] * M[3 + b] + jc[3 * a + 2] * M[6 + b];
        double JS[6];  // JR * hat(wpt)
        for (int a = 0; a < 2; ++a) {
            const double j0 = JR[3 * a], j1 = JR[3 * a + 1], j2 = JR[3 * a + 2];
            JS[3 * a] = j1 * wp[2] - j2 * wp[1];
            JS[3 * a + 1] = j2 * wp[0] - j0 * wp[2];
            JS[3 * a + 2] = j0 * wp[1] - j1 * wp[0];
        }
        double* Ja = P.Ja + 12 * (size_t)i;
        double* Jo = P.Jo + 12 * (size_t)i;
        const double wp_ = typ == 2 ? 0.0 : w;   // anchor-frame right-camera block: no pose block at all
        for (int a = 0; a < 2; ++a)
            for (int b = 0; b < 3; ++b) {
                Ja[6 * a + b] = wp_ * JR[3 * a + b];
                Ja[6 * a + 3 + b] = -wp_ * JS[3 * a + b];
                Jo[6 * a + b] = -wp_ * JR[3 * a + b];
                Jo[6 * a + 3 + b] = wp_ * JS[3 * a + b];
            }
        // J_lambda = -zanch * Rwanch * anchpt   (type 2: -zanch * anchpt, the point never leaves the anchor frame)
        const double* lp = typ == 2 ? ap : rp;
        const double jl[3] = {-zanch * lp[0], -zanch * lp[1], -zanch * lp[2]};
        P.Jl[2 * (size_t)i] = w * (JR[0] * jl[0] + JR[1] * jl[1] + JR[2] * jl[2]);
        P.Jl[2 * (size_t)i + 1] = w * (JR[3] * jl[0] + JR[4] * jl[1] + JR[5] * jl[2]);
        P.Jr[2 * (size_t)i] = w * r0;
        P.Jr[2 * (size_t)i + 1] = w * r1;
    }
    return cost;
}

// ------------------------------------------------------------------ Schur elimination (warp / landmark)

// Fire-and-forget fp64 add into GLOBAL memory.  atomicAdd(double*) on a generic pointer compiles to a run-time address-space
// test + ATOM.E.ADD.F64 (value returned) + a shared-memory CAS loop for the other branch; naming the state space gives one
// RED.E.ADD.F64 and nothing else.
__device__ __forceinline__ void red_add_f64(double* p, double v) {
    asm volatile("red.global.add.f64 [%0], %1;" ::"l"(__cvta_generic_to_global(p)), "d"(v) : "memory");
}

// schur_eliminator_impl.h:179-308 for a scalar e-block: E'E, E'r, F'F, F'r, E'F per touching keyframe, then
// S -= (E'F)' (E'E)^-1 (E'F), rhs -= (E'F)' (E'E)^-1 E'r.  The anchor keyframe's F'F / F'r / column norms are summed
// over the landmark's observations in registers and leave the warp once.
constexpr int SCH = 8;   // observations staged per chunk (C3: 4 per landmark, C5: 7.5)

// CTA-local lock for the shared-memory accumulation mode: lane 0 spins on a shared-memory CAS, the warp follows.
__device__ __forceinline__ void warp_lock(int* lock, int lane) {
    if (!lock) return;                       // per-warp private block: nothing to serialise
    if (lane == 0)
        while (atomicCAS(lock, 0, 1) != 0) __nanosleep(20);
    __syncwarp();
    __threadfence_block();
}
__device__ __forceinline__ void warp_unlock(int* lock, int lane) {
    if (!lock) return;
    __threadfence_block();
    __syncwarp();
    if (lane == 0) atomicExch(lock, 0);
}

// SM = false: contributions leave the warp as fp64 RED into the (privatised) global accumulation block.  B200 retires an
// fp64 RED at ~2.4-3.6 cycles per lane and SM (measured: the phase scales 1/SMs and not with warps per SM), which bounds
// this phase at ~900 REDs per landmark.  SM = true (reduced systems that fit shared memory, n <= ~100): the CTA keeps ONE
// copy of [rhs | F'r | column norms | S] in shared memory, warps commit under a CTA-local lock with plain
// read-modify-writes (shared-memory fp64 atomics are CAS loops, slower than RED) and the CTA flushes the non-zeros once.
template <bool SM>
__device__ __forceinline__ void schur_landmark(const Prob& P, const int* __restrict__ s_slot, double* s_etf, int* s_eslot, double* sJ, int* smeta,
                                               int l, int lane, double radius, int first_iter, double* acc, int n, double& gmax_lm, int* lock) {
#define ACC(ptr, v) do { if (SM) *(ptr) += (v); else red_add_f64((ptr), (v)); } while (0)
    const int p0 = P.lm_ptr[l], p1 = P.lm_ptr[l + 1];
    double* const cRhs = acc; double* const cG = acc + n; double* const cCn = acc + 2 * n; double* const cS = acc + 3 * n;
    double cnl = 0.0, ge = 0.0;
    int nact = 0;
    for (int p = p0 + lane; p < p1; p += 32) {
        const uint8_t act = P.active[p];                                   // loads issued together, selected after
        const double2 jl = *reinterpret_cast<const double2*>(P.Jl + 2 * (size_t)p);
        const double2 jr = *reinterpret_cast<const double2*>(P.Jr + 2 * (size_t)p);
        if (!act) continue;
        cnl += jl.x * jl.x + jl.y * jl.y;
        ge += jl.x * jr.x + jl.y * jr.y;
        nact++;
    }
    cnl = warp_sum(cnl);
    ge = warp_sum(ge);
    nact = __reduce_add_sync(FULL, nact);
    if (nact == 0) {   // unused parameter block: dropped from the program (program.cc:305-387)
        if (lane == 0) { P.ete[l] = 0.0; P.ge[l] = 0.0; }
        return;
    }
    double sc = P.sc_lm[l];
    if (first_iter) {
        sc = 1.0 / (1.0 + sqrt(cnl));
        if (lane == 0) P.sc_lm[l] = sc;
    }
    const double diag = fmin(fmax(cnl * sc * sc, 1e-6), 1e32);
    const double ete = cnl + diag / (radius * sc * sc);
    const double inv_ete = 1.0 / ete;
    if (lane == 0) {
        P.ete[l] = ete;
        P.ge[l] = ge;
    }
    gmax_lm = fmax(gmax_lm, fabs(ge));      // one atomicMax per warp and phase (per landmark they all hit ONE address: ~20 cycles each, serialised in L2)
    const int sa = s_slot[P.lm_anchor_cam[l]];
    int m = 0;   // number of E'F entries (uniform across the warp); entry 0 = anchor
    if (sa >= 0) {
        if (lane < 6) s_etf[lane] = 0.0;
        if (lane == 0) s_eslot[0] = sa;
        m = 1;
    }
    __syncwarp();
    // anchor accumulators: lane owns entries e = lane and lane + 32 of the 6x6 (a = e / 6, b = e % 6, a <= b kept)
    double aFF0 = 0.0, aFF1 = 0.0, aG = 0.0, aCn = 0.0, aE = 0.0;
    const int e0a = lane / 6, e0b = lane - 6 * e0a;
    const int e1 = lane + 32, e1a = e1 / 6, e1b = e1 - 6 * e1a;
    // The Jacobian rows of the landmark's observations are staged in this warp's shared-memory slice SCH at a time (coalesced
    // loads, all in flight together): the per-observation loop below then never waits on L2 (with one dependent global
    // load chain per observation and 8-16 warps per SM the phase was latency bound, 2.4x slower than the RED issue rate).
    double* sJa = sJ; double* sJo = sJ + 12 * SCH; double* sJl = sJ + 24 * SCH; double* sJr = sJ + 26 * SCH;
    for (int pb = p0; pb < p1; pb += SCH) {
        const int cnt = min(SCH, p1 - pb);
        __syncwarp();
        for (int e = lane; e < 12 * cnt; e += 32) { sJa[e] = P.Ja[12 * (size_t)pb + e]; sJo[e] = P.Jo[12 * (size_t)pb + e]; }
        if (lane < 2 * cnt) { sJl[lane] = P.Jl[2 * (size_t)pb + lane]; sJr[lane] = P.Jr[2 * (size_t)pb + lane]; }
        if (lane < cnt) {
            const int p = pb + lane;
            const uint8_t act = P.active[p], ty = P.obs_type ? P.obs_type[p] : 0;
            const int cam = P.obs_cam[p];
            smeta[lane] = !act ? -3 : (ty == 2 ? -2 : s_slot[cam]);   // -3: inactive, -2: e-block-only row (schur_eliminator_impl.h:196-217)
        }
        __syncwarp();
        if (SM) warp_lock(lock, lane);
    for (int q = 0; q < cnt; ++q) {
        const int so = smeta[q];
        if (so < -1) continue;
        const double* Ja = sJa + 12 * q;
        const double* Jo = sJo + 12 * q;
        const double jl0 = sJl[2 * q], jl1 = sJl[2 * q + 1];
        const double r0 = sJr[2 * q], r1 = sJr[2 * q + 1];
        if (sa >= 0) {
            aFF0 += Ja[e0a] * Ja[e0b] + Ja[6 + e0a] * Ja[6 + e0b];
            if (e1 < 36) aFF1 += Ja[e1a] * Ja[e1b] + Ja[6 + e1a] * Ja[6 + e1b];
            if (lane < 6) {
                aG += Ja[lane] * r0 + Ja[6 + lane] * r1;
                aCn += Ja[lane] * Ja[lane] + Ja[6 + lane] * Ja[6 + lane];
                aE += jl0 * Ja[lane] + jl1 * Ja[6 + lane];
            }
        }
        if (so >= 0) {
            // E'F row of this keyframe: a stereo keyframe contributes two residual blocks (left and right camera) to the
            // same pose block, so look the slot up before appending a new entry
            int idx = -1;
            for (int qq = lane; qq < m; qq += 32)
                if (s_eslot[qq] == so) idx = qq;
            idx = __reduce_max_sync(FULL, idx);
            const bool fresh = idx < 0;
            if (fresh) idx = m;
            if (lane < 6) {
                const double e = jl0 * Jo[lane] + jl1 * Jo[6 + lane];
                s_etf[6 * idx + lane] = fresh ? e : s_etf[6 * idx + lane] + e;
            }
            if (lane == 0 && fresh) s_eslot[idx] = so;
            // The observation's six contributions per lane (observer diagonal block: 32 + 1 entries, F'r, column norms, cross
            // block Ja' Jo: 32 + 4 entries) go to DISTINCT addresses: addresses and values first, then all the loads, then all
            // the stores - the shared-memory mode pays one read-modify-write latency per observation instead of six.
            const int l6 = lane < 6 ? lane : 0, l4 = lane & 3;
            double* qp[6]; double qv[6]; bool qk[6];
            qk[0] = e0a <= e0b; qp[0] = cS + (size_t)(6 * so + e0a) * n + 6 * so + e0b; qv[0] = Jo[e0a] * Jo[e0b] + Jo[6 + e0a] * Jo[6 + e0b];
            qk[1] = lane == 3;  qp[1] = cS + (size_t)(6 * so + 5) * n + 6 * so + 5;     qv[1] = Jo[5] * Jo[5] + Jo[11] * Jo[11];
            qk[2] = lane < 6;   qp[2] = cG + 6 * so + l6;                               qv[2] = Jo[l6] * r0 + Jo[6 + l6] * r1;
            qk[3] = lane < 6;   qp[3] = cCn + 6 * so + l6;                              qv[3] = Jo[l6] * Jo[l6] + Jo[6 + l6] * Jo[6 + l6];
            // cross block Ja' Jo into the upper block (min slot, max slot); a: anchor column, b: observer column
            qk[4] = sa >= 0;             qv[4] = Ja[e0a] * Jo[e0b] + Ja[6 + e0a] * Jo[6 + e0b];
            qk[5] = sa >= 0 && lane < 4; qv[5] = Ja[5] * Jo[2 + l4] + Ja[11] * Jo[8 + l4];
            const int sa0 = sa >= 0 ? sa : 0;
            if (sa0 < so) { qp[4] = cS + (size_t)(6 * sa0 + e0a) * n + 6 * so + e0b; qp[5] = cS + (size_t)(6 * sa0 + 5) * n + 6 * so + 2 + l4; }
            else          { qp[4] = cS + (size_t)(6 * so + e0b) * n + 6 * sa0 + e0a; qp[5] = cS + (size_t)(6 * so + 2 + l4) * n + 6 * sa0 + 5; }
            if (SM) {
                double qo[6];
#pragma unroll
                for (int u = 0; u < 6; ++u) qo[u] = qk[u] ? *qp[u] : 0.0;
#pragma unroll
                for (int u = 0; u < 6; ++u) if (qk[u]) *qp[u] = qo[u] + qv[u];
            } else {
#pragma unroll
                for (int u = 0; u < 6; ++u) if (qk[u]) red_add_f64(qp[u], qv[u]);
            }
            if (fresh) m++;
        }
        __syncwarp();
    }
        if (SM) warp_unlock(lock, lane);
    }
    if (SM) warp_lock(lock, lane);
    if (sa >= 0) {
        if (e0a <= e0b) ACC(cS + (size_t)(6 * sa + e0a) * n + 6 * sa + e0b, aFF0);
        if (e1 < 36 && e1a <= e1b) ACC(cS + (size_t)(6 * sa + e1a) * n + 6 * sa + e1b, aFF1);
        if (lane < 6) { ACC(cG + 6 * sa + lane, aG); ACC(cCn + 6 * sa + lane, aCn); }
    }
    if (sa >= 0 && lane < 6) s_etf[lane] += aE;     // the anchor's E'F row was summed in registers
    __syncwarp();
    // Schur complement: S[i,j] -= EtF_i' EtF_j / ete (upper blocks), rhs_i -= EtF_i ge / ete.  Pair-major: every unordered
    // pair of touching keyframes once, oriented by slot (the upper block), the 36 entries of a block on lanes 0..31 + a
    // second pass of 4 lanes - no per-entry divisions, no skipped iterations.
    {
        const int a0 = lane / 6, b0 = lane - 6 * a0;            // entry of pass 1
        const int a1 = 5, b1 = 2 + (lane & 3);                  // entries 32..35 of pass 2 (lanes 0..3)
        constexpr int U = 4;                                    // pairs per batch: 2 U independent read-modify-writes in flight
        const int npair = m * (m + 1) / 2;
        int i = 0, j = 0;
        for (int t0 = 0; t0 < npair; t0 += U) {
            double* q0[U]; double* q1[U]; double v0[U], v1[U]; bool k0[U], k1[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const bool live = t0 + u < npair;
                const int ii = live ? i : 0, jj = live ? j : 0;
                const int si = s_eslot[ii], sj = s_eslot[jj];
                const bool swap = si > sj;                      // block (lo, hi) with lo <= hi; entry (a, b) = etf_lo[a] etf_hi[b]
                const double* el = s_etf + 6 * (swap ? jj : ii);
                const double* eh = s_etf + 6 * (swap ? ii : jj);
                const int lo = swap ? sj : si, hi = swap ? si : sj;
                double* blkp = cS + (size_t)(6 * lo) * n + 6 * hi;
                q0[u] = blkp + (size_t)a0 * n + b0;
                q1[u] = blkp + (size_t)a1 * n + b1;
                k0[u] = live && (ii != jj || a0 <= b0);
                k1[u] = live && lane < 4 && (ii != jj || a1 <= b1);
                v0[u] = -(el[a0] * eh[b0] * inv_ete);
                v1[u] = -(el[a1] * eh[b1] * inv_ete);
                if (live && ++j == m) { ++i; j = i; }
            }
            if (SM) {
                double o0[U], o1[U];
#pragma unroll
                for (int u = 0; u < U; ++u) { o0[u] = k0[u] ? *q0[u] : 0.0; o1[u] = k1[u] ? *q1[u] : 0.0; }
#pragma unroll
                for (int u = 0; u < U; ++u) { if (k0[u]) *q0[u] = o0[u] + v0[u]; if (k1[u]) *q1[u] = o1[u] + v1[u]; }
            } else {
#pragma unroll
                for (int u = 0; u < U; ++u) { if (k0[u]) red_add_f64(q0[u], v0[u]); if (k1[u]) red_add_f64(q1[u], v1[u]); }
            }
        }
    }
    for (int e = lane; e < m * 6; e += 32) {
        const int i = e / 6, a = e - 6 * i;
        ACC(cRhs + 6 * s_eslot[i] + a, -s_etf[6 * i + a] * ge * inv_ete);
    }
    if (SM) warp_unlock(lock, lane);
    __syncwarp();
#undef ACC
}

// FP64 tensor-core tile product (DMMA): D(8x8) = A(8x4) B(4x8) + C.  Fragment layout (PTX ISA, mma.m8n8k4 .f64):
// lane = 4 g + t; A: (row g, col t); B: (row t, col g); C/D: (row g, cols 2t, 2t+1).
__device__ __forceinline__ void dmma_884(double& d0, double& d1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// ------------------------------------------------------------------ back-substitution + candidate cost (warp / landmark)
// schur_eliminator_impl.h:311-377: y_e = (E'E)^-1 (E'r - sum_k (E'F_k) z_k); model cost change
// -(J delta)'(r + J delta / 2) (trust_region_minimizer.cc:424-427); candidate inverse depth; then the residual blocks of
// the landmark at the candidate point (cost only).
__device__ __forceinline__ void backsub_landmark(const Prob& P, const int* __restrict__ s_slot, const double* __restrict__ s_cam,
                                                 int l, int lane, const double* __restrict__ invd, double* __restrict__ cand_invd,
                                                 int use_huber, double& mcc_out, double& st2_out, double& cx2_out, double& cost_out) {
    const double ete = P.ete[l];
    if (ete == 0.0) return;   // landmark not in the program: candidate stays equal
    const int p0 = P.lm_ptr[l], p1 = P.lm_ptr[l + 1];
    const int sa = s_slot[P.lm_anchor_cam[l]];
    double za[6] = {0, 0, 0, 0, 0, 0};
    if (sa >= 0)
        for (int k = 0; k < 6; ++k) za[k] = P.z[6 * sa + k];
    double acc = 0.0;
    for (int p = p0 + lane; p < p1; p += 32) {
        if (!P.active[p]) continue;
        const int so = (P.obs_type && P.obs_type[p] == 2) ? -1 : s_slot[P.obs_cam[p]];
        const double* Ja = P.Ja + 12 * (size_t)p;
        const double* Jo = P.Jo + 12 * (size_t)p;
        double f0 = 0.0, f1 = 0.0;
        if (sa >= 0)
            for (int k = 0; k < 6; ++k) { f0 += Ja[k] * za[k]; f1 += Ja[6 + k] * za[k]; }
        if (so >= 0)
            for (int k = 0; k < 6; ++k) { const double zk = P.z[6 * so + k]; f0 += Jo[k] * zk; f1 += Jo[6 + k] * zk; }
        acc += P.Jl[2 * (size_t)p] * f0 + P.Jl[2 * (size_t)p + 1] * f1;
    }
    acc = warp_sum(acc);
    const double y = (P.ge[l] - acc) / ete;
    const double dl = -y;
    const double cl = invd[l] + dl;
    double mcc = 0.0, cost = 0.0;
    for (int p = p0 + lane; p < p1; p += 32) {
        if (!P.active[p]) continue;
        const int so = (P.obs_type && P.obs_type[p] == 2) ? -1 : s_slot[P.obs_cam[p]];
        const double* Ja = P.Ja + 12 * (size_t)p;
        const double* Jo = P.Jo + 12 * (size_t)p;
        double f0 = P.Jl[2 * (size_t)p] * dl, f1 = P.Jl[2 * (size_t)p + 1] * dl;
        if (sa >= 0)
            for (int k = 0; k < 6; ++k) { f0 -= Ja[k] * za[k]; f1 -= Ja[6 + k] * za[k]; }
        if (so >= 0)
            for (int k = 0; k < 6; ++k) { const double zk = P.z[6 * so + k]; f0 -= Jo[k] * zk; f1 -= Jo[6 + k] * zk; }
        mcc -= f0 * (P.Jr[2 * (size_t)p] + 0.5 * f0) + f1 * (P.Jr[2 * (size_t)p + 1] + 0.5 * f1);
        cost += eval_block<false>(P, p, l, s_cam, cl, use_huber);
    }
    if (lane == 0) {
        cand_invd[l] = cl;
        st2_out += dl * dl;
        cx2_out += cl * cl;
    }
    mcc_out += mcc;
    cost_out += cost;
}

// Sub-group variant: SG lanes per landmark, 32 / SG landmarks per warp in flight.  A landmark has ~4 (C3) to ~8 (C5)
// observations, so one warp per landmark leaves most lanes idle and - worse - strings the landmarks' dependent load chains
// (CSR pointers -> Jacobian rows -> reduction -> second pass) one after the other: measured 3.9 ms of a 11.9 ms batched C3
// solve.  Same arithmetic per observation; the per-landmark sums are formed inside the sub-group.
template <int SG>
__device__ __forceinline__ void backsub_landmarks_sg(const Prob& P, const int* __restrict__ s_slot, const double* __restrict__ s_cam,
                                                     int l0, int lane, const double* __restrict__ invd, double* __restrict__ cand_invd,
                                                     int use_huber, double& mcc_out, double& st2_out, double& cx2_out, double& cost_out) {
    const int sub = lane / SG, sl = lane - sub * SG;
    const int l = l0 + sub;
    const bool in = l < P.npts;
    const double ete = in ? P.ete[l] : 0.0;
    const bool live = in && ete != 0.0;     // ete == 0: landmark not in the program, candidate stays equal
    const int p0 = live ? P.lm_ptr[l] : 0, p1 = live ? P.lm_ptr[l + 1] : 0;
    const int sa = live ? s_slot[P.lm_anchor_cam[l]] : -1;
    double za[6] = {0, 0, 0, 0, 0, 0};
    if (sa >= 0)
        for (int k = 0; k < 6; ++k) za[k] = P.z[6 * sa + k];
    double acc = 0.0;
    for (int p = p0 + sl; p < p1; p += SG) {
        if (!P.active[p]) continue;
        const int so = (P.obs_type && P.obs_type[p] == 2) ? -1 : s_slot[P.obs_cam[p]];
        const double* Ja = P.Ja + 12 * (size_t)p;
        const double* Jo = P.Jo + 12 * (size_t)p;
        double f0 = 0.0, f1 = 0.0;
        if (sa >= 0)
            for (int k = 0; k < 6; ++k) { f0 += Ja[k] * za[k]; f1 += Ja[6 + k] * za[k]; }
        if (so >= 0)
            for (int k = 0; k < 6; ++k) { const double zk = P.z[6 * so + k]; f0 += Jo[k] * zk; f1 += Jo[6 + k] * zk; }
        acc += P.Jl[2 * (size_t)p] * f0 + P.Jl[2 * (size_t)p + 1] * f1;
    }
#pragma unroll
    for (int o = SG / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(FULL, acc, o);
    const double y = live ? (P.ge[l] - acc) / ete : 0.0;
    const double dl = -y;
    const double cl = live ? invd[l] + dl : 0.0;
    double mcc = 0.0, cost = 0.0;
    for (int p = p0 + sl; p < p1; p += SG) {
        if (!P.active[p]) continue;
        const int so = (P.obs_type && P.obs_type[p] == 2) ? -1 : s_slot[P.obs_cam[p]];
        const double* Ja = P.Ja + 12 * (size_t)p;
        const double* Jo = P.Jo + 12 * (size_t)p;
        double f0 = P.Jl[2 * (size_t)p] * dl, f1 = P.Jl[2 * (size_t)p + 1] * dl;
        if (sa >= 0)
            for (int k = 0; k < 6; ++k) { f0 -= Ja[k] * za[k]; f1 -= Ja[6 + k] * za[k]; }
        if (so >= 0)
            for (int k = 0; k < 6; ++k) { const double zk = P.z[6 * so + k]; f0 -= Jo[k] * zk; f1 -= Jo[6 + k] * zk; }
        mcc -= f0 * (P.Jr[2 * (size_t)p] + 0.5 * f0) + f1 * (P.Jr[2 * (size_t)p + 1] + 0.5 * f1);
        cost += eval_block<false>(P, p, l, s_cam, cl, use_huber);
    }
    if (live && sl == 0) {
        cand_invd[l] = cl;
        st2_out += dl * dl;
        cx2_out += cl * cl;
    }
    mcc_out += mcc;
    cost_out += cost;
}

}  // namespace balm
