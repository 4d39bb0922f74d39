// ste_filter.cuh - per-track predict / update / smoother-step device functions (fp64, n = 4).
//
// One thread owns one track: the 4-vector mean and the 10 unique entries of the symmetric
// covariance live in registers across the whole time loop.  Citations are to
// /root/reference/src/track_estimators/kalman_filters/unscented.py unless stated.
#pragma once
#include "ste_math.cuh"
#include "../../include/ste_ukf.h"

namespace ste {

// Shared (per launch) matrices, read through the constant bank of the kernel parameters.
struct Model {
    const double *H;   // [16] row-major
    const double *Q;   // [16]
    const double *R;   // [16]
};

// Per-thread scratch slots (struct Scratch, ste_math.cuh): shared memory on the device.  They hold
// the square-root factor so that the sigma-point loop can stay ROLLED (one instance of the
// trigonometric code in the instruction cache) and index its columns at run time, the parked
// deviations of the sigma pairs, and - while the root is being taken, when those are dead - the
// rotation parameters of the Jacobi sweeps.  One layout for the forward and the backward pass:
//   [0, 14)   forward: observation staged for this step's update (4), dt and the two rates staged
//             for the next step (3); backward: the carried smoothed state xs (4), Ps (10)
//   [14, 30)  root M, column-major: M[r][c] at kScratchRoot + c * 4 + r
//   [30, 46)  forward: Sigma_c / Delta_c of the pair loop; backward by recomputation: Delta_c
//   [14, 62)  rotation parameters during sqrt_psd4 (kSqrtRotSlots = 48: four sweeps)
constexpr int kScratchObs = 0;             // 4 slots
constexpr int kScratchIn = 4;              // 3 slots
constexpr int kScratchXs = 0;              // 4 slots  (backward)
constexpr int kScratchPs = 4;              // 10 slots (backward)
constexpr int kScratchRoot = 14;           // 16 slots
constexpr int kScratchDeltaFwd = 30;       // 16 slots
constexpr int kScratchDelta = 30;          // 16 slots (backward by recomputation)
constexpr int kScratchRot = kScratchRoot;  // kSqrtRotSlots slots, live only inside sqrt_psd4
constexpr int kScratchSlots = kScratchRot + kSqrtRotSlots;   // 62
constexpr int kScratchSlotsFwd = kScratchSlots;
constexpr int kScratchSlotsBwd = kScratchSlots;

// Smoother statistics ("tape") the forward pass can emit for every predict, so that the backward
// pass need not regenerate and re-propagate the sigma points of the same filtered state (the
// reference recomputes them, unscented.py:299-330; they are the same numbers).  Per step, 15 planes:
//   [0..3]   delta = sum W_i f(X_i) - x          noise-free predicted mean minus the filtered mean
//   [4..6]   P_b   = sum W_i d_i d_i^T + Q        about the filtered mean: its position block 00 01 11
//   [7..14]  D[q][r], q = 0..3, r = 0..1          cross covariance sum W_i (X_i - x) f(X_i)^T, its
//                                                 longitude and latitude columns (plane 7 + 2 q + r)
// What is NOT on the tape follows from these and from the filtered covariance P the backward pass
// reads anyway: speed and course propagate linearly (y_2 = x_2 + sog_rate dt, y_3 = x_3 + cog_rate dt,
// non_linear_process.py:72-78), so their sigma-point deviations are +-m_c exactly and, with
// M M = 3 P and 2 W_i = 1/3,
//   D[q][r]   = 2 W_i sum_c m_c[q] m_c[r] = P[q][r]                       (r = 2, 3)
//   P_b[r][q] = D[q][r] + Q[r][q] + delta_r delta_q                       (r in {0, 1}, q in {2, 3})
//   P_b[q][r] = P[q][r] + Q[q][r] + delta_q delta_r                       (q, r in {2, 3})
// (the reference forms the same sums numerically and lands within rounding of these values).  The
// identities need M M = 3 P, i.e. no clamped negative eigenvalue: a step whose root clamped one
// marks its tape entry invalid (delta_0 = NaN) and the backward pass recomputes that step.
constexpr int kStatsPlanes = 15;
constexpr int kStatsPb = 4;     // 3 planes: 00 01 11
constexpr int kStatsD = 7;      // 8 planes

STE_DEV void stash_root(const Scratch &sc, const double (&M)[10]) {
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int r = 0; r < 4; ++r) sc.at(kScratchRoot + c * 4 + r) = M[SYM(r, c)];
}

// The rolled sigma-point loop walks the four columns of the root; each iteration propagates the
// mirror pair x + m_c, x - m_c together: the sincos of the offset column is computed once, and
// the two independent evaluations interleave in the FP64 pipe (DFMA latency ~9 cycles, issue
// interval 2: a warp needs 4-5 independent operations in flight to keep the pipe busy).
// Reference column order (unscented.py:100-105): X[:, 0] = x, X[:, 1+c] = x + m_c, X[:, 5+c] = x - m_c.

// Range of the branch-free trigonometry for this step: every angle the nine sigma points can
// produce stays below kSinCosMaxArg.  |m_rc| <= sqrt(lambda_max(3P)) <= sqrt(3 trace P).
STE_DEV bool step_in_fast_range(const double (&x)[4], const double (&P)[10], double dtR) {
    const double tr3 = 3.0 * (P[SYM(0, 0)] + P[SYM(1, 1)] + P[SYM(2, 2)] + P[SYM(3, 3)]);
    const double lim = 1.0e4;   // radians; two orders of magnitude inside kSinCosMaxArg
    // offsets bounded by sqrt(tr3): compare squares to avoid the root
    const double oa = tr3 * (kDegToRad * kDegToRad), od = tr3 * (dtR * dtR);
    return (fabs(x[1]) * kDegToRad < lim) && (fabs(x[3]) * kDegToRad < lim) && (fabs(x[2] * dtR) < lim) &&
           (oa < lim * lim) && (od < lim * lim);   // false on NaN
}

// Small-displacement tier (geodetic_finish_n<.., SMALL>): every sigma point moves at most 2^-6 rad
// and starts within 75 degrees of latitude.  The root M of 3P is symmetric with M M = 3P, so row r
// of M has norm sqrt(3 P_rr) and every offset of component r is bounded by it: |u_i| <= |u| +
// sqrt(3 P_22) (times |dt|/R for the distance), |lat_i| <= |lat| + sqrt(3 P_11); squares are
// compared so that no root is taken.  Then |tan(dlon)| <= sin(2^-6) / cos(75.9 deg) / cos(dlon)
// = 0.0643 as the series assume.  (A negative diagonal entry - indefinite P - fails the test.)
STE_DEV bool step_is_small(const double (&x)[4], const double (&P)[10], double dtR) {
    const double su2 = 3.0 * P[SYM(2, 2)], sl2 = 3.0 * P[SYM(1, 1)];
    const double a = kSmallAsinMax - fabs(x[2] * dtR);     // room left for the speed offset, in radians
    const double b = kSmallLatMaxDeg - fabs(x[1]);         // room left for the latitude offset, in degrees
    // ... and the three offset angles of every root column stay within the short sincos series (kSmallAngle): the
    // distance offset already does (a <= 2^-6), latitude and course offsets are bounded by sqrt(3 P_11), sqrt(3 P_33)
    const double sc2 = 3.0 * P[SYM(3, 3)];
    constexpr double kOff2 = (kSmallAngle * kRadToDeg) * (kSmallAngle * kRadToDeg);   // (7.16 degrees)^2
    return (a > 0.0) && (b > 0.0) && (su2 >= 0.0) && (sl2 >= 0.0) && (su2 * (dtR * dtR) <= a * a) && (sl2 <= b * b) &&
           (sl2 <= kOff2) && (sc2 <= kOff2);   // false on NaN
}

// ------------------------------------------------------------------------------------------ //
// predict (:144-207).  Unscented transform of (x, P) through the geodetic model.
//
// Moments are accumulated in one pass about the propagated centre point c = f(x):
//   d_i = f(X_i) - c,  mu = Wi * sum d_i,   mean = c + mu            (W0 + 8 Wi = 1, d_0 = 0)
//   P'  = sum_i W_i (f(X_i) - mean - e)(...)^T + Q = Wi * sum d_i d_i^T - mu mu^T + e e^T + Q
// with e the additive noise the reference adds to the mean BEFORE forming deviations (:198-205).
// This needs no storage for the 9 propagated points.  The root M must already be in scratch.
// ------------------------------------------------------------------------------------------ //
// The rolled loop over the four root columns, one instance per tier of the geodetic step (SMALL:
// see step_is_small) so that the hot tier is straight-line code in the instruction stream.
//
// Only longitude and latitude are non-linear.  Speed and course of a propagated sigma point are
// y_2 = x_2 +- m_2 + sog_rate dt and y_3 = x_3 +- m_3 + cog_rate dt, so their deviations from the
// propagated centre are +-m_c[2], +-m_c[3] and never have to be formed.  The loop therefore only
// PARKS, per column c, the sums and differences of the mirror pair's longitude / latitude deviations
//     Sigma_c[r] = (y+[r] - c[r]) + (y-[r] - c[r]),   Delta_c[r] = y+[r] - y-[r]      (r = 0, 1)
// (4 scratch slots per column); every moment is assembled after the loop from these 16 numbers and
// the root itself, with no accumulator live across the trigonometry.
#ifndef STE_PAIR_COLS
#define STE_PAIR_COLS 1   // root columns (mirror pairs) propagated in lock-step per loop iteration: 1, 2 or 4
#endif
template <bool LIB, bool SMALL>
STE_DEV void sigma_pair_loop(const double (&x)[4], const AngleTrig &base, const double (&c)[4], double dt, double dtR,
                             double sog_rate, double cog_rate, const Scratch &sc, double *sig_prior, double *sig_post,
                             int64_t ld) {
    constexpr int NC = STE_PAIR_COLS, NP = 2 * NC;
#ifndef STE_PAIR_UNROLL
#define STE_PAIR_UNROLL 1
#endif
    STE_UNROLL(STE_PAIR_UNROLL)
    for (int col = 0; col < 4; col += NC) {
#if defined(STE_STEP_SYNC) && (STE_STEP_SYNC >= 2) && defined(__CUDA_ARCH__)
        __syncthreads();
#endif
        // points 2k, 2k+1 are the mirror pair x + m, x - m of column col + k
        double m[NC][4], xx[NP][4], yy[NP][4];
        AngleTrig tt[NP];
#pragma unroll
        for (int k = 0; k < NC; ++k)
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                m[k][r] = sc.at(kScratchRoot + (col + k) * 4 + r);
                xx[2 * k][r] = x[r] + m[k][r];
                xx[2 * k + 1][r] = x[r] - m[k][r];
            }
        if constexpr (LIB || NC == 1) {
#pragma unroll
            for (int k = 0; k < NC; ++k) angle_add_pair(base, offset_trig<LIB, SMALL>(m[k][1], m[k][3], m[k][2], dtR), tt[2 * k], tt[2 * k + 1]);
        } else {
            // the offsets of all NC columns through one lock-step series; the full-range evaluation replaces it
            // (for all of them) only when some offset is not small
            double ang[3 * NC], sn[3 * NC], cs[3 * NC];
            bool small = true;
#pragma unroll
            for (int k = 0; k < NC; ++k) {
                ang[3 * k] = m[k][1] * kDegToRad;
                ang[3 * k + 1] = m[k][3] * kDegToRad;
                ang[3 * k + 2] = m[k][2] * dtR;
            }
#pragma unroll
            for (int i = 0; i < 3 * NC; ++i) small &= fabs(ang[i]) <= kSmallAngle;
            small_sincos_v<3 * NC>(ang, sn, cs);
            if (__builtin_expect(!small, 0)) fast_sincos_v<3 * NC>(ang, sn, cs);
#pragma unroll
            for (int k = 0; k < NC; ++k) {
                AngleTrig off;
                off.sp = sn[3 * k]; off.cp = cs[3 * k]; off.sa = sn[3 * k + 1]; off.ca = cs[3 * k + 1]; off.sd = sn[3 * k + 2]; off.cd = cs[3 * k + 2];
                angle_add_pair(base, off, tt[2 * k], tt[2 * k + 1]);
            }
        }
        geodetic_finish_n<LIB, NP, SMALL>(xx, tt, dt, sog_rate, cog_rate, yy);
#pragma unroll
        for (int k = 0; k < NC; ++k) {
            if (sig_prior) {
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    sig_prior[(r * 9 + 1 + col + k) * ld] = xx[2 * k][r];
                    sig_post[(r * 9 + 1 + col + k) * ld] = yy[2 * k][r];
                    sig_prior[(r * 9 + 5 + col + k) * ld] = xx[2 * k + 1][r];
                    sig_post[(r * 9 + 5 + col + k) * ld] = yy[2 * k + 1][r];
                }
            }
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                sc.at(kScratchDeltaFwd + (col + k) * 4 + r) = (yy[2 * k][r] - c[r]) + (yy[2 * k + 1][r] - c[r]);
                sc.at(kScratchDeltaFwd + (col + k) * 4 + 2 + r) = yy[2 * k][r] - yy[2 * k + 1][r];
            }
        }
    }
}

// `clamped`: the root dropped a negative eigenvalue (M M != 3 P); the speed/course block of the
// predicted covariance is then summed from the root's columns as the reference does.
template <bool LIB>
STE_DEV void predict_moments(double (&x)[4], double (&P)[10], const double *Q, double dt, double dtR,
                             double sog_rate, double cog_rate, const double (&e)[4], const Scratch &sc,
                             double *sig_prior, double *sig_post, double *stats, int64_t ld, const bool small = false,
                             const bool clamped = false, const bool noisy = true) {
    AngleTrig base;
    double c[4];
    if (!LIB && small) {
        base = angle_trig<LIB, true>(x[1], x[3], x[2], dtR);
        geodetic_finish<LIB, true>(x, base, dt, sog_rate, cog_rate, c);
        if (sig_prior) {
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                sig_prior[(r * 9) * ld] = x[r];
                sig_post[(r * 9) * ld] = c[r];
            }
        }
        sigma_pair_loop<LIB, true>(x, base, c, dt, dtR, sog_rate, cog_rate, sc, sig_prior, sig_post, ld);
    } else {
        base = angle_trig<LIB>(x[1], x[3], x[2], dtR);
        geodetic_finish<LIB, false>(x, base, dt, sog_rate, cog_rate, c);
        if (sig_prior) {
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                sig_prior[(r * 9) * ld] = x[r];
                sig_post[(r * 9) * ld] = c[r];
            }
        }
        sigma_pair_loop<LIB, false>(x, base, c, dt, dtR, sog_rate, cog_rate, sc, sig_prior, sig_post, ld);
    }
    // ---- moments from the parked Sigma_c, Delta_c (r = 0, 1) and the root columns m_c ---- //
    double sg[4][2], dl[4][2], mc[4][4];
#pragma unroll
    for (int col = 0; col < 4; ++col) {
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            sg[col][r] = sc.at(kScratchDeltaFwd + col * 4 + r);
            dl[col][r] = sc.at(kScratchDeltaFwd + col * 4 + 2 + r);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) mc[col][q] = sc.at(kScratchRoot + col * 4 + q);
    }
    // mean: mu = Wi sum_i d_i (zero for speed and course), delta = mean - x (noise-free)
    double mu[2], delta[4];
#pragma unroll
    for (int r = 0; r < 2; ++r) mu[r] = kWi * ((sg[0][r] + sg[1][r]) + (sg[2][r] + sg[3][r]));
#pragma unroll
    for (int r = 0; r < 4; ++r) delta[r] = (c[r] - x[r]) + (r < 2 ? mu[r] : 0.0);
    // G[q][r] = sum_c m_c[q] Delta_c[r]: Wi G is the cross covariance D[q][r] and, for q >= 2, also
    // the predicted covariance between position row r and speed / course
    double G[4][2];
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            double acc = mc[0][q] * dl[0][r];
#pragma unroll
            for (int col = 1; col < 4; ++col) acc = fma(mc[col][q], dl[col][r], acc);
            G[q][r] = kWi * acc;
        }
    double cov[10];
    // position block: sum_i d_i d_i^T = 1/2 sum_c (Sigma_c Sigma_c^T + Delta_c Delta_c^T)
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int q = r; q < 2; ++q) {
            double acc = sg[0][r] * sg[0][q];
            acc = fma(dl[0][r], dl[0][q], acc);
#pragma unroll
            for (int col = 1; col < 4; ++col) acc = fma(sg[col][r], sg[col][q], fma(dl[col][r], dl[col][q], acc));
            cov[SYM(r, q)] = fma(0.5 * kWi, acc, fma(-mu[r], mu[q], Q[r * 4 + q]));
        }
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int q = 2; q < 4; ++q) cov[SYM(r, q)] = G[q][r] + Q[r * 4 + q];
    // speed / course block: 2 Wi sum_c m_c m_c^T = 2 Wi (M M) = P when the root is exact
    if (!clamped) {
#pragma unroll
        for (int r = 2; r < 4; ++r)
#pragma unroll
            for (int q = r; q < 4; ++q) cov[SYM(r, q)] = P[SYM(r, q)] + Q[r * 4 + q];
    } else {
#pragma unroll
        for (int r = 2; r < 4; ++r)
#pragma unroll
            for (int q = r; q < 4; ++q) {
                double acc = mc[0][r] * mc[0][q];
#pragma unroll
                for (int col = 1; col < 4; ++col) acc = fma(mc[col][r], mc[col][q], acc);
                cov[SYM(r, q)] = fma(2.0 * kWi, acc, Q[r * 4 + q]);
            }
    }
    if (noisy) {   // launch-uniform: a noise tape is present
#pragma unroll
        for (int r = 0; r < 4; ++r) x[r] = c[r] + ((r < 2 ? mu[r] : 0.0) + e[r]);
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int q = r; q < 4; ++q) P[SYM(r, q)] = fma(e[r], e[q], cov[SYM(r, q)]);
    } else {
#pragma unroll
        for (int r = 0; r < 4; ++r) x[r] = r < 2 ? c[r] + mu[r] : c[r];
#pragma unroll
        for (int k = 0; k < 10; ++k) P[k] = cov[k];
    }
    if (stats) {
        // position block of P_b (about x); a clamped root invalidates the entry (see kStatsPlanes)
        const uint32_t ldb = (uint32_t)ld * 8u;
        STE_STORE_STREAM(plane_ptr(stats, ldb, kStatsPb + 0), fma(delta[0], delta[0], cov[SYM(0, 0)]));
        STE_STORE_STREAM(plane_ptr(stats, ldb, kStatsPb + 1), fma(delta[0], delta[1], cov[SYM(0, 1)]));
        STE_STORE_STREAM(plane_ptr(stats, ldb, kStatsPb + 2), fma(delta[1], delta[1], cov[SYM(1, 1)]));
        STE_STORE_STREAM(stats, clamped ? f64_from_bits(0x7ff8000000000000ull) : delta[0]);
#pragma unroll
        for (int r = 1; r < 4; ++r) STE_STORE_STREAM(plane_ptr(stats, ldb, r), delta[r]);
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
            for (int r = 0; r < 2; ++r) STE_STORE_STREAM(plane_ptr(stats, ldb, kStatsD + q * 2 + r), G[q][r]);
    }
}

// library-math version of the same step for out-of-range arguments; out of line (never hot)
STE_COLD void predict_moments_cold(double *x_io, double *P_out, const double *Q, double dt, double dtR, double sog_rate,
                                   double cog_rate, const double *e_in, Scratch sc, double *sig_prior, double *sig_post,
                                   double *stats, int64_t ld, bool clamped) {
    double x[4], P[10], e[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        x[r] = x_io[r];
        e[r] = e_in[r];
    }
#pragma unroll
    for (int k = 0; k < 10; ++k) P[k] = P_out[k];
    predict_moments<true>(x, P, Q, dt, dtR, sog_rate, cog_rate, e, sc, sig_prior, sig_post, stats, ld, false, clamped);
#pragma unroll
    for (int r = 0; r < 4; ++r) x_io[r] = x[r];
#pragma unroll
    for (int k = 0; k < 10; ++k) P_out[k] = P[k];
}

STE_DEV void ukf_predict(double (&x)[4], double (&P)[10], const double *Q, double dt,
                         double sog_rate, double cog_rate, const double (&e)[4],
                         int &status, const Scratch &sc, double *sig_prior, double *sig_post, double *stats,
                         int64_t ld, const bool allow_small = true, const bool noisy = true) {
    const double dtR = dt * (1.0 / kEarthRadiusKm);
    const bool fast = step_in_fast_range(x, P, dtR);
    bool clamped;
    {
        double M[10];
        clamped = sqrt_psd4(P, kSigmaScale, M, sc, kScratchRot);
        if (clamped) status |= STE_STATUS_INDEFINITE;
        stash_root(sc, M);
    }
    if (fast) {
        predict_moments<false>(x, P, Q, dt, dtR, sog_rate, cog_rate, e, sc, sig_prior, sig_post, stats, ld,
                               allow_small && !clamped && step_is_small(x, P, dtR), clamped, noisy);   // a clamped root is not bounded by P's diagonal
    } else {
        double xt[4], Pt[10], et[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            xt[r] = x[r];
            et[r] = e[r];
        }
#pragma unroll
        for (int k = 0; k < 10; ++k) Pt[k] = P[k];
        predict_moments_cold(xt, Pt, Q, dt, dtR, sog_rate, cog_rate, et, sc, sig_prior, sig_post, stats, ld, clamped);
#pragma unroll
        for (int r = 0; r < 4; ++r) x[r] = xt[r];
#pragma unroll
        for (int k = 0; k < 10; ++k) P[k] = Pt[k];
    }
}

// ------------------------------------------------------------------------------------------ //
// Robustification (:353-511, dead code in the reference, enabled for BASELINE config 4).
// gamma = |y^T S^+ y| with y = z - x (NOT z - Hx, no angle wrap, :420-426); while gamma > chi:
// lambda += (gamma - chi) / (y^T S^+ R S^+ y); R *= lambda (compounding); zero noise.
// `rs` is the accumulated scale of R.  GENERIC: any H, R.
// ------------------------------------------------------------------------------------------ //
STE_DEV void innovation_cov(const double (&P)[10], const double *H, const double *R,
                                               double rs, double (&HP)[16], double (&S)[10]) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double acc = 0.0;
#pragma unroll
            for (int k = 0; k < 4; ++k) acc = fma(H[i * 4 + k], P[SYM(k, j)], acc);
            HP[i * 4 + j] = acc;
        }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = i; j < 4; ++j) {
            double acc = rs * R[i * 4 + j];
#pragma unroll
            for (int k = 0; k < 4; ++k) acc = fma(HP[i * 4 + k], H[j * 4 + k], acc);
            S[SYM(i, j)] = acc;
        }
}

STE_DEV double quad_form(const double (&A)[10], const double (&y)[4]) {
    double acc = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        double row = 0.0;
#pragma unroll
        for (int j = 0; j < 4; ++j) row = fma(A[SYM(i, j)], y[j], row);
        acc = fma(y[i], row, acc);
    }
    return acc;
}

// update (:209-265), generic H / R.  z is consumed (noise added in place as the reference does).
template <bool GATING, bool INNOV = false>
STE_DEV void ukf_update_generic(double (&x)[4], double (&P)[10], const Model &m,
                                                   double (&z)[4], const double *unit_noise /*[4] or null*/,
                                                   double chi, int max_iter, int &status, int &gate_it,
                                                   double &gate_lam, double &rs, Innov *iv = nullptr) {
    const double *H = m.H, *R = m.R;
    double HP[16], S[10], Sinv[10], lpd;
    rs = 1.0;
    innovation_cov(P, H, R, rs, HP, S);
    int dropped = pinv_sym4<INNOV>(S, Sinv, &lpd);
    gate_it = 0;
    gate_lam = 1.0;
    if (GATING) {
        double yg[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) yg[i] = z[i] - x[i];
        double gamma = fabs(quad_form(Sinv, yg));
        while (gamma > chi) {
            if (gate_it >= max_iter) {
                status |= STE_STATUS_GATE_CAP;
                break;
            }
            // v = S^+ y ; den = v^T (rs R) v
            double v[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                double acc = 0.0;
#pragma unroll
                for (int j = 0; j < 4; ++j) acc = fma(Sinv[SYM(i, j)], yg[j], acc);
                v[i] = acc;
            }
            double den = 0.0;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                double row = 0.0;
#pragma unroll
                for (int j = 0; j < 4; ++j) row = fma(R[i * 4 + j], v[j], row);
                den = fma(v[i], row, den);
            }
            den *= rs;
            gate_lam = gate_lam + (gamma - chi) / den;
            rs *= gate_lam;
            innovation_cov(P, H, R, rs, HP, S);
            dropped = pinv_sym4<INNOV>(S, Sinv, &lpd);
            gamma = fabs(quad_form(Sinv, yg));
            ++gate_it;
        }
    }
    if (unit_noise) {
#pragma unroll
        for (int i = 0; i < 4; ++i) z[i] = fma(unit_noise[i], sqrt(rs * R[i * 4 + i]), z[i]);
    }
    // K = P H^T S^+  with P H^T = (H P)^T
    double K[16];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double acc = 0.0;
#pragma unroll
            for (int k = 0; k < 4; ++k) acc = fma(HP[k * 4 + i], Sinv[SYM(k, j)], acc);
            K[i * 4 + j] = acc;
        }
    double y[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        double acc = z[i];
#pragma unroll
        for (int k = 0; k < 4; ++k) acc = fma(-H[i * 4 + k], x[k], acc);
        y[i] = acc;
    }
    y[3] = wrap180(y[3]);  // :250
    if constexpr (INNOV) *iv = Innov{quad_form(Sinv, y), lpd, 4 - dropped};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        double acc = x[i];
#pragma unroll
        for (int k = 0; k < 4; ++k) acc = fma(K[i * 4 + k], y[k], acc);
        x[i] = acc;
    }
    x[3] = py_mod360(x[3]);  // :257
    // Joseph form (:260-265): (I - K H) P (I - K H)^T + K R K^T
    double A[16], AP[16], KR[16];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double acc = (i == j) ? 1.0 : 0.0;
#pragma unroll
            for (int k = 0; k < 4; ++k) acc = fma(-K[i * 4 + k], H[k * 4 + j], acc);
            A[i * 4 + j] = acc;
        }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double acc = 0.0, acc2 = 0.0;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                acc = fma(A[i * 4 + k], P[SYM(k, j)], acc);
                acc2 = fma(K[i * 4 + k], R[k * 4 + j], acc2);
            }
            AP[i * 4 + j] = acc;
            KR[i * 4 + j] = acc2 * rs;
        }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = i; j < 4; ++j) {
            double acc = 0.0;
#pragma unroll
            for (int k = 0; k < 4; ++k) acc = fma(AP[i * 4 + k], A[j * 4 + k], fma(KR[i * 4 + k], K[j * 4 + k], acc));
            P[SYM(i, j)] = acc;
        }
}

// update for the position-only measurement H = diag(1,1,0,0) with R zero outside its leading
// 2x2 block (every example and the CLI input.json of the reference).  S = H P H^T + R is then
// block-diagonal with an exactly-zero trailing block, pinv(S) = [pinv(S22) 0; 0 0], and K has two
// non-zero columns; the arithmetic below is the generic path with the zeros removed.
// INNOV: the statistics of rows 0 and 1, the only ones S^+ does not zero.
template <bool GATING, bool INNOV = false>
STE_DEV void ukf_update_position(double (&x)[4], double (&P)[10], const Model &m,
                                                    double (&z)[4], const double *unit_noise, double chi,
                                                    int max_iter, int &status, int &gate_it,
                                                    double &gate_lam, double &rs, Innov *iv = nullptr) {
    const double r00 = m.R[0], r01 = m.R[1], r11 = m.R[5];
    rs = 1.0;
    double Si[3], lpd;
    int dropped;
    gate_it = 0;
    gate_lam = 1.0;
    if (GATING) {
        // one copy of the inverse and of the criterion in the instruction stream (the loop is entered at its test):
        // the gated kernel's executed path sits at the size of the instruction cache
        const double y0 = z[0] - x[0], y1 = z[1] - x[1];
#pragma unroll 1
        for (;;) {
            dropped = pinv_sym2<INNOV>(fma(rs, r00, P[SYM(0, 0)]), fma(rs, r01, P[SYM(0, 1)]), fma(rs, r11, P[SYM(1, 1)]), Si, &lpd);
            const double v0 = fma(Si[0], y0, Si[1] * y1), v1 = fma(Si[1], y0, Si[2] * y1);
            const double gamma = fabs(fma(y0, v0, y1 * v1));
            if (!(gamma > chi)) break;
            if (gate_it >= max_iter) {
                status |= STE_STATUS_GATE_CAP;
                break;
            }
            const double den = rs * fma(v0, fma(r00, v0, r01 * v1), v1 * fma(r01, v0, r11 * v1));
            gate_lam = gate_lam + (gamma - chi) / den;
            rs *= gate_lam;
            ++gate_it;
        }
    } else {
        dropped = pinv_sym2<INNOV>(fma(rs, r00, P[SYM(0, 0)]), fma(rs, r01, P[SYM(0, 1)]), fma(rs, r11, P[SYM(1, 1)]), Si, &lpd);
    }
    if (unit_noise) {
        z[0] = fma(unit_noise[0], sqrt(rs * r00), z[0]);
        z[1] = fma(unit_noise[1], sqrt(rs * r11), z[1]);
    }
    double K0[4], K1[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        K0[r] = fma(P[SYM(r, 0)], Si[0], P[SYM(r, 1)] * Si[1]);
        K1[r] = fma(P[SYM(r, 0)], Si[1], P[SYM(r, 1)] * Si[2]);
    }
    const double y0 = z[0] - x[0], y1 = z[1] - x[1];
    if constexpr (INNOV) *iv = Innov{fma(y0, fma(Si[0], y0, Si[1] * y1), y1 * fma(Si[1], y0, Si[2] * y1)), lpd, 2 - dropped};
#pragma unroll
    for (int r = 0; r < 4; ++r) x[r] = fma(K0[r], y0, fma(K1[r], y1, x[r]));
    x[3] = py_mod360(x[3]);
    // Joseph form (I - K H) P (I - K H)^T + K (rs R) K^T (:260-265) with AP = (I - K H) P = P - K P[0:2, :]:
    //     AP A^T + KR K^T = AP + (KR - AP[:, 0:2]) K^T
    // the same sum with the two rank-2 products merged (W = KR - AP[:, 0:2] is the gain's optimality residual: the
    // errors of AP's position columns still meet their cancelling partner, as in the four-product form)
    double AP[16];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (j < 2 || j >= i) AP[i * 4 + j] = fma(-K0[i], P[SYM(0, j)], fma(-K1[i], P[SYM(1, j)], P[SYM(i, j)]));
    const double q00 = rs * r00, q01 = rs * r01, q11 = rs * r11;
    double W0[4], W1[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        W0[r] = fma(K0[r], q00, K1[r] * q01) - AP[r * 4 + 0];
        W1[r] = fma(K0[r], q01, K1[r] * q11) - AP[r * 4 + 1];
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = i; j < 4; ++j) P[SYM(i, j)] = fma(W0[i], K0[j], fma(W1[i], K1[j], AP[i * 4 + j]));
}

// ------------------------------------------------------------------------------------------ //
// One URTSS backward iteration (rts_step, :297-349), in two phases so that the long sigma-point
// loop runs with few live registers:
//
//  phase 1  urtss_moments   sigma points of the filtered state (xf, Pf) -> weighted sums
//      x_b - xf = sum W_i d_i,            d_i = f(X_i) - xf
//      P_b      = sum W_i d_i d_i^T + Q   (about the FILTERED mean: reference quirk, :324-325)
//      Delta_c  = d(x + m_c) - d(x - m_c) (c = 0..3, parked in scratch; mirror pairs are
//                 propagated together, see predict_moments)
//  phase 2  urtss_gain      cross covariance, gain and the smoothed state
//      D = sum W_i (X_i - xf)(f(X_i) - x_b)^T = Wi sum_c m_c Delta_c^T
//          (X_0 - xf = 0 and sum W_i (X_i - xf) = 0, so neither x_b nor the centre point enters)
//      K = D pinv(P_b) = Wi sum_c m_c (pinv(P_b) Delta_c)^T
//      xs = xf + K wrap(xs - x_b);   Ps = Pf + K (Ps - P_b) K^T
//
// The smoothed state of step+1 (xs, Ps) is only touched in phase 2 and lives in scratch between
// steps; Pf is re-read by the caller for phase 2 instead of being held across phase 1.
// ------------------------------------------------------------------------------------------ //

template <bool LIB>
STE_DEV void urtss_moments_impl(const double (&xf)[4], const double *Q, double dt, double dtR, double sog_rate,
                                double cog_rate, double (&s1)[4], double (&Pb)[10], const Scratch &sc) {
    const AngleTrig base = angle_trig<LIB>(xf[1], xf[3], xf[2], dtR);
    {
        double d0[4];
        geodetic_finish<LIB>(xf, base, dt, sog_rate, cog_rate, d0);
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            d0[r] -= xf[r];
            s1[r] = kW0 * d0[r];
        }
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int q = r; q < 4; ++q) Pb[SYM(r, q)] = fma(kW0 * d0[r], d0[q], Q[r * 4 + q]);
    }
#pragma unroll 1
    for (int col = 0; col < 4; ++col) {
        double m[4], xx[2][4], dd[2][4];
        double (&xp)[4] = xx[0], (&xm)[4] = xx[1], (&dp)[4] = dd[0], (&dm)[4] = dd[1];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            m[r] = sc.at(kScratchRoot + col * 4 + r);
            xp[r] = xf[r] + m[r];
            xm[r] = xf[r] - m[r];
        }
        {
            const AngleTrig off = offset_trig<LIB>(m[1], m[3], m[2], dtR);
            AngleTrig tt[2];
            angle_add_pair(base, off, tt[0], tt[1]);
            geodetic_finish_n<LIB, 2>(xx, tt, dt, sog_rate, cog_rate, dd);
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            dp[r] -= xf[r];
            dm[r] -= xf[r];
            s1[r] = fma(kWi, dp[r] + dm[r], s1[r]);
            sc.at(kScratchDelta + col * 4 + r) = dp[r] - dm[r];
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const double wp = kWi * dp[r], wm = kWi * dm[r];
#pragma unroll
            for (int q = r; q < 4; ++q) Pb[SYM(r, q)] = fma(wp, dp[q], fma(wm, dm[q], Pb[SYM(r, q)]));
        }
    }
}

// PER_Q: a clone of its own for callers whose Q lives in thread-local memory (a track's own Q), so that the clone
// the other callers share keeps reading Q from the kernel parameters
template <bool PER_Q = false>
STE_COLD void urtss_moments_cold(const double *xf_in, const double *Q, double dt, double dtR, double sog_rate,
                                 double cog_rate, double *s1_out, double *Pb_out, Scratch sc) {
    double xf[4], s1[4], Pb[10];
#pragma unroll
    for (int r = 0; r < 4; ++r) xf[r] = xf_in[r];
    urtss_moments_impl<true>(xf, Q, dt, dtR, sog_rate, cog_rate, s1, Pb, sc);
#pragma unroll
    for (int r = 0; r < 4; ++r) s1_out[r] = s1[r];
#pragma unroll
    for (int k = 0; k < 10; ++k) Pb_out[k] = Pb[k];
}

template <bool PER_Q = false>
STE_DEV void urtss_moments(const double (&xf)[4], const double (&Pf)[10], const double *Q, double dt,
                           double sog_rate, double cog_rate, double (&s1)[4], double (&Pb)[10], int &status,
                           const Scratch &sc) {
    const double dtR = dt * (1.0 / kEarthRadiusKm);
    const bool fast = step_in_fast_range(xf, Pf, dtR);
    {
        double M[10];
        if (sqrt_psd4(Pf, kSigmaScale, M, sc, kScratchRot)) status |= STE_STATUS_INDEFINITE;
        stash_root(sc, M);
    }
    if (fast) {
        urtss_moments_impl<false>(xf, Q, dt, dtR, sog_rate, cog_rate, s1, Pb, sc);
    } else {
        double xt[4], st[4], Pt[10];
#pragma unroll
        for (int r = 0; r < 4; ++r) xt[r] = xf[r];
        urtss_moments_cold<PER_Q>(xt, Q, dt, dtR, sog_rate, cog_rate, st, Pt, sc);
#pragma unroll
        for (int r = 0; r < 4; ++r) s1[r] = st[r];
#pragma unroll
        for (int k = 0; k < 10; ++k) Pb[k] = Pt[k];
    }
}

// xs <- xf + K wrap(xs - x_b), Ps <- Pf + K (Ps - P_b) K^T with (xs, Ps) carried in scratch (:337-349)
STE_DEV void urtss_apply(const double (&xf)[4], const double (&Pf)[10], const double (&xb_minus_xf)[4],
                         const double (&Pb)[10], const double (&K)[16], double (&xs)[4], double (&Ps)[10],
                         const Scratch &sc) {
#pragma unroll
    for (int r = 0; r < 4; ++r) xs[r] = sc.at(kScratchXs + r);
#pragma unroll
    for (int k = 0; k < 10; ++k) Ps[k] = sc.at(kScratchPs + k);
    double y[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) y[r] = xs[r] - (xf[r] + xb_minus_xf[r]);
    y[3] = wrap180(y[3]);  // :340
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        double acc = xf[i];
#pragma unroll
        for (int k = 0; k < 4; ++k) acc = fma(K[i * 4 + k], y[k], acc);
        xs[i] = acc;
    }
    xs[3] = py_mod360(xs[3]);  // :346
    double KG[16];
#pragma unroll
    for (int k = 0; k < 10; ++k) Ps[k] -= Pb[k];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double acc = 0.0;
#pragma unroll
            for (int k = 0; k < 4; ++k) acc = fma(K[i * 4 + k], Ps[SYM(k, j)], acc);
            KG[i * 4 + j] = acc;
        }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = i; j < 4; ++j) {
            double acc = Pf[SYM(i, j)];
#pragma unroll
            for (int k = 0; k < 4; ++k) acc = fma(KG[i * 4 + k], K[j * 4 + k], acc);
            Ps[SYM(i, j)] = acc;
        }
#pragma unroll
    for (int r = 0; r < 4; ++r) sc.at(kScratchXs + r) = xs[r];
#pragma unroll
    for (int k = 0; k < 10; ++k) sc.at(kScratchPs + k) = Ps[k];
}

// phase 2 after urtss_moments (root and Delta_c in scratch)
STE_DEV void urtss_gain(const double (&xf)[4], const double (&Pf)[10], const double (&s1)[4], const double (&Pb)[10],
                        const double (&e)[4], double (&xs)[4], double (&Ps)[10], int &status, const Scratch &sc) {
    double Pbinv[10];
    if (pinv_spd4(Pb, Pbinv) > 0) status |= STE_STATUS_RANK_DEFICIENT;
    double K[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) K[k] = 0.0;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        double dl[4], v[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) dl[r] = sc.at(kScratchDelta + c * 4 + r);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double acc = 0.0;
#pragma unroll
            for (int k = 0; k < 4; ++k) acc = fma(Pbinv[SYM(j, k)], dl[k], acc);
            v[j] = acc;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const double wm = kWi * sc.at(kScratchRoot + c * 4 + i);
#pragma unroll
            for (int j = 0; j < 4; ++j) K[i * 4 + j] = fma(wm, v[j], K[i * 4 + j]);
        }
    }
    double xb[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) xb[r] = s1[r] + e[r];
    urtss_apply(xf, Pf, xb, Pb, K, xs, Ps, sc);
}

// One backward iteration from the statistics the forward pass stored for this step (kStatsPlanes
// planes at `stats`): no sigma points, no square root - a pseudo-inverse and three small products.
// What the tape leaves out comes from the filtered covariance and Q (see kStatsPlanes).
// Returns false, with nothing changed, when the entry is marked invalid (delta_0 = NaN: the forward
// pass's root clamped an eigenvalue at this step); the caller then recomputes the step.
// The pass is bound by HBM latency and bandwidth, so all 29 loads of a step must be in flight
// before that first decision; left alone, ptxas sinks the other 28 below the branch on delta_0
// (measured: +10 % run time).  The decision is therefore made to depend on every loaded word
// through `guard`, a run-time zero the compiler cannot see through (SteProblem.reserved).
STE_DEV bool urtss_step_from_stats(const double *mf, const double *cf, bool packed, const double *stats, int64_t ld,
                                   const double *Q, const double (&e)[4], double (&xs)[4], double (&Ps)[10], int &status,
                                   const Scratch &sc, const unsigned guard) {
    double xf[4], Pf[10], dlt[4], xb[4], Pb[10], D[16];
#pragma unroll
    for (int r = 0; r < 4; ++r) dlt[r] = STE_LOAD_STREAM_PINNED(stats + r * ld);
#pragma unroll
    for (int k = 0; k < 3; ++k) Pb[k == 2 ? SYM(1, 1) : k] = STE_LOAD_STREAM_PINNED(stats + (kStatsPb + k) * ld);
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int r = 0; r < 2; ++r) D[q * 4 + r] = STE_LOAD_STREAM_PINNED(stats + (kStatsD + q * 2 + r) * ld);
#pragma unroll
    for (int r = 0; r < 4; ++r) xf[r] = STE_LOAD_STREAM_PINNED(mf + r * ld);
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = i; j < 4; ++j) Pf[SYM(i, j)] = STE_LOAD_STREAM_PINNED(cf + (packed ? SYM(i, j) : i * 4 + j) * ld);
    unsigned seen = 0;
#pragma unroll
    for (int r = 0; r < 4; ++r) seen |= (unsigned)(f64_bits(dlt[r]) >> 32) | (unsigned)(f64_bits(xf[r]) >> 32);
#pragma unroll
    for (int k = 0; k < 10; ++k) seen |= (unsigned)(f64_bits(Pf[k]) >> 32);
    seen |= (unsigned)(f64_bits(Pb[SYM(0, 0)]) >> 32) | (unsigned)(f64_bits(Pb[SYM(0, 1)]) >> 32) | (unsigned)(f64_bits(Pb[SYM(1, 1)]) >> 32);
#pragma unroll
    for (int q = 0; q < 4; ++q) seen |= (unsigned)(f64_bits(D[q * 4]) >> 32) | (unsigned)(f64_bits(D[q * 4 + 1]) >> 32);
    if (!(dlt[0] == dlt[0]) || (seen & guard) != 0u) return false;
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int r = 2; r < 4; ++r) D[q * 4 + r] = Pf[SYM(q, r)];
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int q = 2; q < 4; ++q) Pb[SYM(r, q)] = fma(dlt[r], dlt[q], D[q * 4 + r] + Q[r * 4 + q]);
#pragma unroll
    for (int r = 2; r < 4; ++r)
#pragma unroll
        for (int q = r; q < 4; ++q) Pb[SYM(r, q)] = fma(dlt[r], dlt[q], Pf[SYM(r, q)] + Q[r * 4 + q]);
#pragma unroll
    for (int r = 0; r < 4; ++r) xb[r] = dlt[r] + e[r];
    double Pbinv[10];
    if (pinv_spd4(Pb, Pbinv) > 0) status |= STE_STATUS_RANK_DEFICIENT;
    double K[16];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double acc = 0.0;
#pragma unroll
            for (int k = 0; k < 4; ++k) acc = fma(D[i * 4 + k], Pbinv[SYM(k, j)], acc);
            K[i * 4 + j] = acc;
        }
    urtss_apply(xf, Pf, xb, Pb, K, xs, Ps, sc);
    return true;
}

}  // namespace ste
