// ste_generic.cuh - dimension-generic (n <= 8) unscented predict / update / smoother.
//
// The batched n = 4 hot path (ste_tracks.cuh) is specialised for the geodetic state; the reference's
// class, however, takes its dimension from H (unscented.py:52-62) and any process callable.  This file
// covers that surface for the process models the library ships: one thread per filter, matrices in
// thread-local arrays, arithmetic written literally after the reference (two-pass moments about the
// noisy mean, Joseph-form update, state index 3 treated as the heading exactly as unscented.py:250, 257
// hard-code it).
//
// Every function is a template on a compile-time dimension NC: NC = 0 takes n from ProblemN.n and sizes
// the arrays for kMaxN (the single-step kernels of the class API); NC > 0 fixes n = NC and sizes the
// arrays for it (the whole-track fleet kernels, NC = 5).  Both instantiations run the same operations
// in the same order - every FMA is an explicit fma() and the library builds with -fmad=false - so they
// round identically: the fleet kernels are bit-identical to the single-step kernels.
#pragma once
#include "ste_math.cuh"

namespace ste {

constexpr int kMaxN = 8;

// leading dimension of the thread-local matrices and the largest n of an instantiation
template <int NC>
struct DimN {
    static constexpr int LD = NC > 0 ? NC : kMaxN;
    static constexpr int LL = 2 * LD + 1;   // sigma points
};

// process models selectable on the device (SteProblemN.model)
//   0  geodetic_dynamics        n = 4: [lon, lat, sog, cog], rates from the call's arguments
//   1  geodetic_dynamics_turn   n = 5: [lon, lat, sog, cog, cog_rate], the turn rate is a state that persists
// (the reference's default weights W0 = 1 - n/3 must lie in (-1, 1), unscented.py:125-129, so its class runs n <= 5)
STE_DEV void process_n(int model, int n, const double *x, double dt, double sog_rate, double cog_rate, double *y) {
    double x4[4] = {x[0], x[1], x[2], x[3]}, y4[4];
    const double sr = sog_rate, cr = model == 1 ? x[4] : cog_rate;
    geodetic_step(x4, dt, dt / kEarthRadiusKm, sr, cr, y4);
    for (int r = 0; r < 4; ++r) y[r] = y4[r];
    for (int r = 4; r < n; ++r) y[r] = x[r];
}

// cyclic Jacobi on a symmetric n x n (leading dimension DimN<NC>::LD): A -> diagonal, V = eigenvectors
template <int NC>
STE_DEV void eig_sym_n(int n, double *A, double *V) {
    constexpr int D = DimN<NC>::LD;
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) V[i * D + j] = (i == j) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 30; ++sweep) {
        double off = 0.0, dia = 0.0;
        for (int i = 0; i < n; ++i) {
            dia += A[i * D + i] * A[i * D + i];
            for (int j = i + 1; j < n; ++j) off += A[i * D + j] * A[i * D + j];
        }
        if (!(off > 1e-36 * dia)) break;
        for (int p = 0; p < n - 1; ++p)
            for (int q = p + 1; q < n; ++q) {
                const double apq = A[p * D + q];
                if (apq == 0.0) continue;
                const double d = A[q * D + q] - A[p * D + p], b = apq + apq;
                const double tt = (d >= 0.0 ? b : -b) / (fabs(d) + sqrt(fma(d, d, b * b)));
                const double c = 1.0 / sqrt(fma(tt, tt, 1.0)), s = tt * c;
                for (int r = 0; r < n; ++r) {  // columns p, q of A and V
                    const double arp = A[r * D + p], arq = A[r * D + q];
                    A[r * D + p] = fma(c, arp, -s * arq);
                    A[r * D + q] = fma(s, arp, c * arq);
                    const double vrp = V[r * D + p], vrq = V[r * D + q];
                    V[r * D + p] = fma(c, vrp, -s * vrq);
                    V[r * D + q] = fma(s, vrp, c * vrq);
                }
                for (int r = 0; r < n; ++r) {  // rows p, q of A
                    const double apr = A[p * D + r], aqr = A[q * D + r];
                    A[p * D + r] = fma(c, apr, -s * aqr);
                    A[q * D + r] = fma(s, apr, c * aqr);
                }
                A[p * D + q] = 0.0;
                A[q * D + p] = 0.0;
            }
    }
}

// F = V f(diag) V^T of the symmetric part of A.  inverse: Moore-Penrose with numpy's rcond 1e-15;
// otherwise Re sqrtm (negative eigenvalues contribute 0; returns true when one was clamped).
// INNOV (inverse only): also the log pseudo-determinant and the rank of the kept spectrum (struct Innov).
template <int NC, bool INNOV = false>
STE_DEV bool fun_sym_n(int n, const double *Ain, bool inverse, double *F, Innov *iv = nullptr) {
    constexpr int D = DimN<NC>::LD;
    double A[D * D], V[D * D], f[D];
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) A[i * D + j] = 0.5 * (Ain[i * D + j] + Ain[j * D + i]);
    eig_sym_n<NC>(n, A, V);
    double wmax = 0.0;
    for (int k = 0; k < n; ++k) wmax = fmax(wmax, fabs(A[k * D + k]));
    bool flagged = false;
    if constexpr (INNOV) {
        iv->log_pdet = 0.0;
        iv->rank = 0;
    }
    for (int k = 0; k < n; ++k) {
        const double w = A[k * D + k];
        if (inverse) {
            f[k] = fabs(w) > kPinvRcond * wmax ? 1.0 / w : 0.0;
            if constexpr (INNOV) {
                if (fabs(w) > kPinvRcond * wmax) {
                    iv->log_pdet += log(w);
                    ++iv->rank;
                }
            }
        } else {
            flagged |= w < -1e-13 * wmax;
            f[k] = sqrt(fmax(w, 0.0));
        }
    }
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            double acc = 0.0;
            for (int k = 0; k < n; ++k) acc = fma(V[i * D + k] * f[k], V[j * D + k], acc);
            F[i * D + j] = acc;
        }
    return flagged;
}

// n x n matrices of a generic launch travel in the kernel parameters (row-major, leading dimension n)
struct ProblemN {
    int32_t n, model, n_tracks, reserved;
    int64_t ld;
    double H[kMaxN * kMaxN], Q[kMaxN * kMaxN], R[kMaxN * kMaxN];
};

// UnscentedKalmanFilter.predict (unscented.py:144-207) on a thread-local state: x [n], P [n][D] in place; Q row-major
// n x n (p.Q, or a track's own).  noise: unit normals noise[r * ns] or NULL, scaled by sqrt(diag Q); sigma_prior /
// sigma_post: planes [n*(2n+1)] at stride ss, or NULL.  Returns STE_STATUS_* bits.
template <int NC>
STE_DEV int predict_core(const ProblemN &p, const double *Q, double *x, double *P, double d, double sr, double cr, const double *noise, int64_t ns,
                         double *sigma_prior, double *sigma_post, int64_t ss) {
    constexpr int D = DimN<NC>::LD, DL = DimN<NC>::LL;
    const int n = NC > 0 ? NC : p.n, L = 2 * n + 1;
    double S[D * D], M[D * D], Y[D * DL], mean[D];
    const double w0 = 1.0 - n / 3.0, wi = (1.0 - w0) / (2.0 * n);   // unscented.py:125, 132
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) S[i * D + j] = (n / (1.0 - w0)) * P[i * D + j];
    const int st = fun_sym_n<NC>(n, S, false, M) ? STE_STATUS_INDEFINITE : 0;
    for (int j = 0; j < L; ++j) {
        double xi[D], yi[D];
        for (int r = 0; r < n; ++r) {
            xi[r] = x[r];
            if (j >= 1 && j <= n) xi[r] = x[r] + M[r * D + (j - 1)];
            if (j > n) xi[r] = x[r] - M[r * D + (j - 1 - n)];
        }
        process_n(p.model, n, xi, d, sr, cr, yi);
        for (int r = 0; r < n; ++r) {
            Y[r * DL + j] = yi[r];
            if (sigma_prior) sigma_prior[(r * L + j) * ss] = xi[r];
            if (sigma_post) sigma_post[(r * L + j) * ss] = yi[r];
        }
    }
    for (int r = 0; r < n; ++r) {
        double acc = w0 * Y[r * DL];
        for (int j = 1; j < L; ++j) acc = fma(wi, Y[r * DL + j], acc);
        mean[r] = acc + (noise ? noise[r * ns] * sqrt(Q[r * n + r]) : 0.0);   // :195-202
    }
    bool bad = false;
    for (int r = 0; r < n; ++r) {
        for (int q = 0; q < n; ++q) {
            double acc = w0 * (Y[r * DL] - mean[r]) * (Y[q * DL] - mean[q]);
            for (int j = 1; j < L; ++j) acc = fma(wi * (Y[r * DL + j] - mean[r]), Y[q * DL + j] - mean[q], acc);
            const double v = acc + Q[r * n + q];   // :205-207, about the noisy mean
            P[r * D + q] = v;
            bad |= !(v * 0.0 == 0.0);
        }
        x[r] = mean[r];
        bad |= !(mean[r] * 0.0 == 0.0);
    }
    return st | (bad ? STE_STATUS_NONFINITE : 0);
}

// UnscentedKalmanFilter.update (unscented.py:209-265) on a thread-local state, dense H and R: x [n], P [n][D] in place;
// R row-major n x n (p.R, or a track's own); zin [n] the observation, noise unit normals noise[r * ns] or NULL, scaled
// by sqrt(diag R).  Returns STE_STATUS_* bits.  INNOV: also the update's innovation statistics into *iv (struct Innov).
template <int NC, bool INNOV = false>
STE_DEV int update_core(const ProblemN &p, const double *R, double *x, double *P, const double *zin, const double *noise, int64_t ns,
                        Innov *iv = nullptr) {
    constexpr int D = DimN<NC>::LD;
    const int n = NC > 0 ? NC : p.n;
    double z[D], y[D], PHt[D * D], S[D * D], Si[D * D], K[D * D], A[D * D], AP[D * D];
    for (int r = 0; r < n; ++r) z[r] = zin[r] + (noise ? noise[r * ns] * sqrt(R[r * n + r]) : 0.0);   // :232-236
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            double acc = 0.0;
            for (int k = 0; k < n; ++k) acc = fma(P[i * D + k], p.H[j * n + k], acc);
            PHt[i * D + j] = acc;
        }
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            double acc = R[i * n + j];
            for (int k = 0; k < n; ++k) acc = fma(p.H[i * n + k], PHt[k * D + j], acc);
            S[i * D + j] = acc;
        }
    fun_sym_n<NC, INNOV>(n, S, true, Si, iv);
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            double acc = 0.0;
            for (int k = 0; k < n; ++k) acc = fma(PHt[i * D + k], Si[k * D + j], acc);
            K[i * D + j] = acc;
        }
    for (int i = 0; i < n; ++i) {
        double acc = z[i];
        for (int k = 0; k < n; ++k) acc = fma(-p.H[i * n + k], x[k], acc);
        y[i] = acc;
    }
    if (n > 3) y[3] = wrap180(y[3]);   // :250 (the reference indexes state 3 unconditionally)
    if constexpr (INNOV) {
        double nis = 0.0;
        for (int i = 0; i < n; ++i) {
            double row = 0.0;
            for (int j = 0; j < n; ++j) row = fma(Si[i * D + j], y[j], row);
            nis = fma(y[i], row, nis);
        }
        iv->nis = nis;
    }
    for (int i = 0; i < n; ++i) {
        double acc = x[i];
        for (int k = 0; k < n; ++k) acc = fma(K[i * D + k], y[k], acc);
        x[i] = acc;
    }
    if (n > 3) x[3] = py_mod360(x[3]);   // :257
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            double acc = (i == j) ? 1.0 : 0.0;
            for (int k = 0; k < n; ++k) acc = fma(-K[i * D + k], p.H[k * n + j], acc);
            A[i * D + j] = acc;
        }
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            double acc = 0.0;
            for (int k = 0; k < n; ++k) acc = fma(A[i * D + k], P[k * D + j], acc);
            AP[i * D + j] = acc;
        }
    // K R, kept in PHt (dead)
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            double acc = 0.0;
            for (int k = 0; k < n; ++k) acc = fma(K[i * D + k], R[k * n + j], acc);
            PHt[i * D + j] = acc;
        }
    bool bad = false;
    for (int i = 0; i < n; ++i) {
        for (int j = 0; j < n; ++j) {
            double acc = 0.0;
            for (int k = 0; k < n; ++k) acc = fma(AP[i * D + k], A[j * D + k], fma(PHt[i * D + k], K[j * D + k], acc));
            P[i * D + j] = acc;   // Joseph form, :260-265
            bad |= !(acc * 0.0 == 0.0);
        }
        bad |= !(x[i] * 0.0 == 0.0);
    }
    return bad ? STE_STATUS_NONFINITE : 0;
}

// Single-step wrappers of the class API: x [n][ld], P [n*n][ld] of track t in place around the cores.
// predict: dt / sog_rate / cog_rate [T]; noise [n][ld] unit normals or NULL; sigma_prior / sigma_post [n*(2n+1)][ld] or NULL.
STE_DEV void predict_n(const ProblemN &p, int t, double *x_io, double *P_io, const double *dt, const double *sog_rate,
                       const double *cog_rate, const double *noise, double *sigma_prior, double *sigma_post, int32_t *status) {
    const int n = p.n;
    const int64_t ld = p.ld;
    double x[kMaxN], P[kMaxN * kMaxN];
    for (int r = 0; r < n; ++r) x[r] = x_io[r * ld + t];
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) P[i * kMaxN + j] = P_io[(i * n + j) * ld + t];
    const double d = dt[t], sr = sog_rate ? sog_rate[t] : 0.0, cr = cog_rate ? cog_rate[t] : 0.0;
    const int st = predict_core<0>(p, p.Q, x, P, d, sr, cr, noise ? noise + t : nullptr, ld, sigma_prior ? sigma_prior + t : nullptr,
                                   sigma_post ? sigma_post + t : nullptr, ld);
    for (int r = 0; r < n; ++r) {
        for (int q = 0; q < n; ++q) P_io[(r * n + q) * ld + t] = P[r * kMaxN + q];
        x_io[r * ld + t] = x[r];
    }
    if (status) status[t] = st;
}

// update: z [n][ld]; noise [n][ld] unit normals or NULL.
STE_DEV void update_n(const ProblemN &p, int t, double *x_io, double *P_io, const double *z_in, const double *noise, int32_t *status) {
    const int n = p.n;
    const int64_t ld = p.ld;
    double x[kMaxN], z[kMaxN], P[kMaxN * kMaxN];
    for (int r = 0; r < n; ++r) {
        x[r] = x_io[r * ld + t];
        z[r] = z_in[r * ld + t];
        for (int q = 0; q < n; ++q) P[r * kMaxN + q] = P_io[(r * n + q) * ld + t];
    }
    const int st = update_core<0>(p, p.R, x, P, z, noise ? noise + t : nullptr, ld);
    for (int i = 0; i < n; ++i) {
        for (int j = 0; j < n; ++j) P_io[(i * n + j) * ld + t] = P[i * kMaxN + j];
        x_io[i * ld + t] = x[i];
    }
    if (status) status[t] = st;
}

// UnscentedKalmanFilter.rts_step (unscented.py:267-351) for any n <= 8 and a device process model: the whole backward
// loop of one track.  mean_f / mean_s [S][n][ld], cov_f / cov_s [S][n*n][ld] with S = n_states; dt [S-1][ld]; the rates
// [n_rates][ld], indexed by step / rate_repeat as the reference's np.repeat expansion does (:287-292); noise [S-1][n][ld]
// unit normals in step order or NULL.  The last state is copied (the loop starts at S - 2, :297).  Arithmetic written
// literally after the reference: P_b about the FILTERED mean (:324-325), the cross covariance about the noisy x_b
// (:328-330), pinv(P_b), state index 3 wrapped as the heading (:340, 346).  Q row-major n x n (p.Q, or the track's own),
// the noise scaled by sqrt(diag Q).  Returns STE_STATUS_* bits.
template <int NC>
STE_DEV int rts_n(const ProblemN &p, const double *Q, int t, int n_states, int rate_repeat, int n_rates, const double *mean_f, const double *cov_f,
                  const double *dt, const double *sog_rate, const double *cog_rate, const double *noise, double *mean_s,
                  double *cov_s) {
    constexpr int D = DimN<NC>::LD, DL = DimN<NC>::LL;
    const int n = NC > 0 ? NC : p.n, L = 2 * n + 1;
    const int64_t ld = p.ld;
    const double w0 = 1.0 - n / 3.0, wi = (1.0 - w0) / (2.0 * n);
    double xs[D], Ps[D * D];
    int st = 0;
    bool bad = false;
    for (int r = 0; r < n; ++r) {
        xs[r] = mean_f[((int64_t)(n_states - 1) * n + r) * ld + t];
        mean_s[((int64_t)(n_states - 1) * n + r) * ld + t] = xs[r];
        for (int q = 0; q < n; ++q) {
            Ps[r * D + q] = cov_f[((int64_t)(n_states - 1) * n * n + r * n + q) * ld + t];
            cov_s[((int64_t)(n_states - 1) * n * n + r * n + q) * ld + t] = Ps[r * D + q];
        }
    }
    for (int step = n_states - 2; step >= 0; --step) {
        double xf[D], Pf[D * D], S[D * D], M[D * D], X[D * DL], Y[D * DL], xb[D], Pb[D * D], Pbi[D * D], Dc[D * D], K[D * D], y[D];
        for (int r = 0; r < n; ++r) {
            xf[r] = mean_f[((int64_t)step * n + r) * ld + t];
            for (int q = 0; q < n; ++q) Pf[r * D + q] = cov_f[((int64_t)step * n * n + r * n + q) * ld + t];
        }
        for (int i = 0; i < n; ++i)
            for (int j = 0; j < n; ++j) S[i * D + j] = (n / (1.0 - w0)) * Pf[i * D + j];
        if (fun_sym_n<NC>(n, S, false, M)) st |= STE_STATUS_INDEFINITE;
        int ri = step / rate_repeat;
        ri = ri < n_rates ? ri : n_rates - 1;
        const double d = dt[(int64_t)step * ld + t], sr = sog_rate ? sog_rate[(int64_t)ri * ld + t] : 0.0,
                     cr = cog_rate ? cog_rate[(int64_t)ri * ld + t] : 0.0;
        for (int j = 0; j < L; ++j) {
            double xi[D], yi[D];
            for (int r = 0; r < n; ++r) {
                xi[r] = xf[r];
                if (j >= 1 && j <= n) xi[r] = xf[r] + M[r * D + (j - 1)];
                if (j > n) xi[r] = xf[r] - M[r * D + (j - 1 - n)];
            }
            process_n(p.model, n, xi, d, sr, cr, yi);
            for (int r = 0; r < n; ++r) {
                X[r * DL + j] = xi[r];
                Y[r * DL + j] = yi[r];
            }
        }
        for (int r = 0; r < n; ++r) {
            double acc = w0 * Y[r * DL];
            for (int j = 1; j < L; ++j) acc = fma(wi, Y[r * DL + j], acc);
            xb[r] = acc + (noise ? noise[((int64_t)step * n + r) * ld + t] * sqrt(Q[r * n + r]) : 0.0);   // :313-322
        }
        for (int r = 0; r < n; ++r)
            for (int q = 0; q < n; ++q) {
                double pb = w0 * (Y[r * DL] - xf[r]) * (Y[q * DL] - xf[q]);     // :324-325
                double dd = w0 * (X[r * DL] - xf[r]) * (Y[q * DL] - xb[q]);     // :328-330
                for (int j = 1; j < L; ++j) {
                    pb = fma(wi * (Y[r * DL + j] - xf[r]), Y[q * DL + j] - xf[q], pb);
                    dd = fma(wi * (X[r * DL + j] - xf[r]), Y[q * DL + j] - xb[q], dd);
                }
                Pb[r * D + q] = pb + Q[r * n + q];
                Dc[r * D + q] = dd;
            }
        fun_sym_n<NC>(n, Pb, true, Pbi);
        for (int i = 0; i < n; ++i)
            for (int j = 0; j < n; ++j) {
                double acc = 0.0;
                for (int k = 0; k < n; ++k) acc = fma(Dc[i * D + k], Pbi[k * D + j], acc);
                K[i * D + j] = acc;     // :333
            }
        for (int r = 0; r < n; ++r) y[r] = xs[r] - xb[r];
        if (n > 3) y[3] = wrap180(y[3]);    // :340
        for (int i = 0; i < n; ++i) {
            double acc = xf[i];
            for (int k = 0; k < n; ++k) acc = fma(K[i * D + k], y[k], acc);
            xs[i] = acc;                    // :343
        }
        if (n > 3) xs[3] = py_mod360(xs[3]);   // :346
        // Ps <- Pf + K (Ps - P_b) K^T (:349); S holds K (Ps - P_b)
        for (int i = 0; i < n; ++i)
            for (int j = 0; j < n; ++j) {
                double acc = 0.0;
                for (int k = 0; k < n; ++k) acc = fma(K[i * D + k], Ps[k * D + j] - Pb[k * D + j], acc);
                S[i * D + j] = acc;
            }
        for (int i = 0; i < n; ++i)
            for (int j = 0; j < n; ++j) {
                double acc = Pf[i * D + j];
                for (int k = 0; k < n; ++k) acc = fma(S[i * D + k], K[j * D + k], acc);
                M[i * D + j] = acc;
            }
        for (int r = 0; r < n; ++r) {
            mean_s[((int64_t)step * n + r) * ld + t] = xs[r];
            bad |= !(xs[r] * 0.0 == 0.0);
            for (int q = 0; q < n; ++q) {
                Ps[r * D + q] = M[r * D + q];
                cov_s[((int64_t)step * n * n + r * n + q) * ld + t] = Ps[r * D + q];
                bad |= !(Ps[r * D + q] * 0.0 == 0.0);
            }
        }
    }
    return st | (bad ? STE_STATUS_NONFINITE : 0);
}

}  // namespace ste
