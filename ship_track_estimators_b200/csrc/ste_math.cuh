// ste_math.cuh - register-resident fp64 building blocks of the UKF/URTSS kernels (sm_100a).
//
// Everything here is per-thread scalar code on fully unrolled fixed-size arrays, so that the
// compiler keeps all matrices in registers (no local memory).  Symmetric 4x4 matrices are held
// as their 10 upper-triangle entries in the order
//     [00 01 02 03 11 12 13 22 23 33]            (SYM(i,j), i <= j)
//
// Reference arithmetic being restated (file:line under /root/reference/src/track_estimators/):
//   sqrtm(3P)            kalman_filters/unscented.py:95-97   -> sqrt_psd4   (principal root)
//   np.linalg.pinv(S)    kalman_filters/unscented.py:243,333 -> pinv_sym4   (rcond 1e-15)
//   geodetic_dynamics    kalman_filters/non_linear_process.py:54-78 -> geodetic_step
//   x % 360, wrap        kalman_filters/unscented.py:250,257,340,346 -> py_mod360, wrap180
#pragma once
// A plain C++ build of these headers exists only for the developer-side numerical sandbox
// (tools/host_emul); the shipped library is always built by nvcc for sm_100a.
#include "ste_fastmath.cuh"

namespace ste {

constexpr double kEarthRadiusKm = 6378.137;           // constants.py:1
constexpr double kDegToRad = 0.017453292519943295;    // numpy radians(): x * (pi / 180)
constexpr double kRadToDeg = 57.29577951308232;       // numpy degrees(): x * (180 / pi)
constexpr double kW0 = 1.0 - 4.0 / 3.0;               // unscented.py:125  (n = 4)
constexpr double kWi = (1.0 - kW0) / 8.0;             // unscented.py:132
constexpr double kSigmaScale = 4.0 / (1.0 - kW0);     // unscented.py:95   (= 3)
constexpr double kPinvRcond = 1e-15;                  // numpy.linalg.pinv default rcond
constexpr double kLog2Pi = 1.8378770664093454835606594728112;   // log(2 pi): Gaussian log-likelihood of an innovation

STE_HD constexpr int SYM(int i, int j) {
    return i <= j ? (i * 4 - (i * (i - 1)) / 2 + (j - i)) : (j * 4 - (j * (j - 1)) / 2 + (i - j));
}

// Per-thread scratch slots outside the register file (shared memory on the device, a plain
// array in the host sandbox).  Slot k of this thread lives at base[k * stride].
struct Scratch {
    double *base;
    int stride;
    STE_DEV double &at(int slot) const { return base[(long)slot * stride]; }
};

// Plane k (a compile-time index) of a [plane][track] array whose plane stride is ld_bytes: base + k * ld_bytes as ONE
// integer instruction (32-bit stride x immediate + 64-bit base; the C ABI limits ld to 2^29 - 1 tracks for this).
STE_DEV double *plane_ptr(double *base, uint32_t ld_bytes, uint32_t k) {
    return reinterpret_cast<double *>(reinterpret_cast<char *>(base) + (uint64_t)ld_bytes * k);
}
STE_DEV const double *plane_ptr(const double *base, uint32_t ld_bytes, uint32_t k) {
    return reinterpret_cast<const double *>(reinterpret_cast<const char *>(base) + (uint64_t)ld_bytes * k);
}

// Python / numpy floored modulo by 360 (result in [0, 360], sign of the divisor).
STE_COLD double py_mod360_general(double a) {
    double r = fmod(a, 360.0);
    if (r != 0.0) {
        if (r < 0.0) r += 360.0;
    } else {
        r = 0.0;  // copysign(0, 360)
    }
    return r;
}
// a course that is already in [0, 360) - nearly every call - comes back unchanged (a + 0.0: -0.0 -> +0.0 as Python gives)
STE_DEV double py_mod360(double a) {
    if (a >= 0.0 && a < 360.0) return a + 0.0;
    return py_mod360_general(a);
}
STE_DEV double wrap180(double a) { return py_mod360(a + 180.0) - 180.0; }

// ------------------------------------------------------------------------------------------ //
// Cyclic Jacobi eigen-decomposition of a symmetric 4x4:  A = V diag(w) V^T.
// On return a[SYM(i,i)] hold the eigenvalues, V (row-major 4x4) the eigenvectors as columns.
// A rotation on an exactly-zero off-diagonal has s = t = 0 exactly (and c within an ulp of 1), so structurally
// block-diagonal inputs (S = H P H^T + R with zero rows/columns) keep their exact zeros.
// ------------------------------------------------------------------------------------------ //
// Rotation parameters for L disjoint index pairs at once (lock-step: the L dependency chains
// interleave in the FP64 pipe).  Angle theta in (-pi/4, pi/4] with tan 2 theta = 2 a_pq / (a_qq - a_pp):
//   cos 2theta = |d| / h,  sin 2theta = sign(d) b / h,   h = hypot(d, b)
//   cos theta = sqrt((1 + cos 2theta) / 2),  sin theta = sin 2theta / (2 cos theta),  t = tan theta
// two reciprocal square roots, no division; sin theta keeps full RELATIVE accuracy for tiny
// rotations because it is a product of accurately rounded factors.
template <int N>
STE_DEV void jacobi_params(const double (&app)[N], const double (&aqq)[N], const double (&apq)[N], double (&c)[N],
                           double (&s)[N], double (&t)[N]) {
    double d[N], b[N], v[N], rh[N], cc[N], rc[N];
    STE_LANES { d[l] = aqq[l] - app[l]; b[l] = apq[l] + apq[l]; }
    STE_LANES v[l] = fma(d[l], d[l], b[l] * b[l]);
    fast_rsqrt_v<N>(v, rh);
    // identity on a vanishing pivot block (d == b == 0, or underflow) from TWO selects: 1/h := 0 makes sin 2theta = 0, and
    // cos^2 theta := 1 makes cos theta = 1 (rsqrt(1) is exactly 1: its residual is 0), so c = 1, s = t = 0
    bool skip[N];
    STE_LANES {
        // a zero pivot with d != 0 needs no test: b = 0 gives s = t = 0 exactly and c within an ulp of 1, which leaves
        // exact zeros exact; only v = d^2 + b^2 == 0 (or underflowed) has no finite 1/h
        skip[l] = !(v[l] > 1e-290);
        rh[l] = skip[l] ? 0.0 : rh[l];
        cc[l] = skip[l] ? 1.0 : fma(0.5, fabs(d[l]) * rh[l], 0.5);
    }
    fast_rsqrt_v<N>(cc, rc);
    STE_LANES {
        // sign(d) b through the integer pipe (d = -0.0 counts as negative: either 45-degree rotation annihilates the pivot)
        const double s2t = f64_from_bits(f64_bits(b[l]) ^ (f64_bits(d[l]) & 0x8000000000000000ull)) * rh[l];
        c[l] = cc[l] * rc[l];
        s[l] = (0.5 * s2t) * rc[l];
        t[l] = s[l] * rc[l];
    }
}

template <int P_, int Q_>
STE_DEV void jacobi_apply_a(double (&a)[10], double c, double s, double t) {
    const double apq = a[SYM(P_, Q_)];
    a[SYM(P_, P_)] = fma(-t, apq, a[SYM(P_, P_)]);
    a[SYM(Q_, Q_)] = fma(t, apq, a[SYM(Q_, Q_)]);
    a[SYM(P_, Q_)] = 0.0;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        if (r != P_ && r != Q_) {
            const double arp = a[SYM(r, P_)], arq = a[SYM(r, Q_)];
            a[SYM(r, P_)] = fma(c, arp, -s * arq);
            a[SYM(r, Q_)] = fma(s, arp, c * arq);
        }
    }
}

// S <- J S J^T for the rotation J that jacobi_apply_a used as a <- J^T a J (undoes the change of
// basis on a symmetric matrix expressed in the rotated basis).  With d = S_qq - S_pp:
//   S_pp += h, S_qq -= h, h = s^2 d + 2cs S_pq;   S_pq <- (c^2 - s^2) S_pq + cs d
template <int P_, int Q_>
STE_DEV void jacobi_unapply(double (&S)[10], double c, double s) {
    const double cs = c * s, s2 = s * s;
    const double w = fma(c, c, -s2), u = cs + cs;
    const double spq = S[SYM(P_, Q_)], d = S[SYM(Q_, Q_)] - S[SYM(P_, P_)];
    const double h = fma(s2, d, u * spq);
    S[SYM(P_, P_)] += h;
    S[SYM(Q_, Q_)] -= h;
    S[SYM(P_, Q_)] = fma(w, spq, cs * d);
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        if (r != P_ && r != Q_) {
            const double srp = S[SYM(r, P_)], srq = S[SYM(r, Q_)];
            S[SYM(r, P_)] = fma(c, srp, s * srq);
            S[SYM(r, Q_)] = fma(c, srq, -s * srp);
        }
    }
}

template <int P_, int Q_>
STE_DEV void jacobi_apply(double (&a)[10], double (&V)[16], double c, double s, double t) {
    const double apq = a[SYM(P_, Q_)];
    a[SYM(P_, P_)] = fma(-t, apq, a[SYM(P_, P_)]);
    a[SYM(Q_, Q_)] = fma(t, apq, a[SYM(Q_, Q_)]);
    a[SYM(P_, Q_)] = 0.0;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        if (r != P_ && r != Q_) {
            const double arp = a[SYM(r, P_)], arq = a[SYM(r, Q_)];
            a[SYM(r, P_)] = fma(c, arp, -s * arq);
            a[SYM(r, Q_)] = fma(s, arp, c * arq);
        }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const double vrp = V[r * 4 + P_], vrq = V[r * 4 + Q_];
        V[r * 4 + P_] = fma(c, vrp, -s * vrq);
        V[r * 4 + Q_] = fma(s, vrp, c * vrq);
    }
}

// two rotations on disjoint index pairs {P1,Q1}, {P2,Q2}: they commute, so their parameters are
// taken from the same matrix and computed side by side
template <int P1, int Q1, int P2, int Q2>
STE_DEV void jacobi_rotate2(double (&a)[10], double (&V)[16]) {
    const double app[2] = {a[SYM(P1, P1)], a[SYM(P2, P2)]}, aqq[2] = {a[SYM(Q1, Q1)], a[SYM(Q2, Q2)]},
                 apq[2] = {a[SYM(P1, Q1)], a[SYM(P2, Q2)]};
    double c[2], s[2], t[2];
    jacobi_params<2>(app, aqq, apq, c, s, t);
    jacobi_apply<P1, Q1>(a, V, c[0], s[0], t[0]);
    jacobi_apply<P2, Q2>(a, V, c[1], s[1], t[1]);
}

// The same pair of rotations without an eigenvector matrix: (c, s) of both go to four scratch
// slots so that the change of basis can be undone later (jacobi_unrotate2).
template <int P1, int Q1, int P2, int Q2>
STE_DEV void jacobi_rotate2_store(double (&a)[10], const Scratch &sc, int slot) {
    const double app[2] = {a[SYM(P1, P1)], a[SYM(P2, P2)]}, aqq[2] = {a[SYM(Q1, Q1)], a[SYM(Q2, Q2)]},
                 apq[2] = {a[SYM(P1, Q1)], a[SYM(P2, Q2)]};
    double c[2], s[2], t[2];
    jacobi_params<2>(app, aqq, apq, c, s, t);
    jacobi_apply_a<P1, Q1>(a, c[0], s[0], t[0]);
    jacobi_apply_a<P2, Q2>(a, c[1], s[1], t[1]);
    sc.at(slot + 0) = c[0];
    sc.at(slot + 1) = s[0];
    sc.at(slot + 2) = c[1];
    sc.at(slot + 3) = s[1];
}
template <int P1, int Q1, int P2, int Q2>
STE_DEV void jacobi_unrotate2(double (&S)[10], const Scratch &sc, int slot) {
    const double c0 = sc.at(slot + 0), s0 = sc.at(slot + 1), c1 = sc.at(slot + 2), s1 = sc.at(slot + 3);
    jacobi_unapply<P1, Q1>(S, c0, s0);   // disjoint index pairs: the two commute
    jacobi_unapply<P2, Q2>(S, c1, s1);
}
constexpr int kSweepSlots = 12;   // scratch slots one sweep's rotation parameters take
// Stage order (0,1)(2,3) -> (0,3)(1,2) -> (0,2)(1,3).  Measured on the host build (tools/sweep_stats.py): the uniform shape
// needs the (0,1)(2,3) stage first (one sweep per root; two with any other first stage), and on the config-4 shape this
// order of the other two takes 2.42 sweeps per root / 3.06 per warp against 2.57 / 3.16 the other way round.
STE_DEV void jacobi_sweep_store(double (&a)[10], const Scratch &sc, int slot) {
    jacobi_rotate2_store<0, 1, 2, 3>(a, sc, slot);
    jacobi_rotate2_store<0, 3, 1, 2>(a, sc, slot + 4);
    jacobi_rotate2_store<0, 2, 1, 3>(a, sc, slot + 8);
}
STE_DEV void jacobi_unsweep(double (&S)[10], const Scratch &sc, int slot) {
    jacobi_unrotate2<0, 2, 1, 3>(S, sc, slot + 8);
    jacobi_unrotate2<0, 3, 1, 2>(S, sc, slot + 4);
    jacobi_unrotate2<0, 1, 2, 3>(S, sc, slot);
}

STE_DEV void jacobi_sweep(double (&a)[10], double (&V)[16]) {
    jacobi_rotate2<0, 1, 2, 3>(a, V);
    jacobi_rotate2<0, 2, 1, 3>(a, V);
    jacobi_rotate2<0, 3, 1, 2>(a, V);
}

// tol2: a pair (p,q) counts as converged when a_pq^2 <= tol2 |a_pp a_qq| (keeps the small
// eigen-directions of badly scaled covariances accurate) or a_pq is negligible against the whole
// matrix.  kJacobiTight drives the off-diagonals to rounding level.
constexpr double kJacobiTight = 1e-33;

template <bool INIT>
STE_DEV void jacobi_eig4(double (&a)[10], double (&V)[16], double tol2) {
    if (INIT) {
#pragma unroll
        for (int i = 0; i < 16; ++i) V[i] = (i % 5 == 0) ? 1.0 : 0.0;
    }
    // Quadratic convergence: nearly diagonal covariances need 2-3 sweeps.
#pragma unroll 1
    for (int sweep = 0; sweep < 12; ++sweep) {
        const double dia = a[0] * a[0] + a[4] * a[4] + a[7] * a[7] + a[9] * a[9];
        const double floor2 = 1e-40 * dia;
        bool more = false;
#pragma unroll
        for (int p = 0; p < 3; ++p)
#pragma unroll
            for (int q = p + 1; q < 4; ++q) {
                const double o2 = a[SYM(p, q)] * a[SYM(p, q)];
                more |= (o2 > tol2 * fabs(a[SYM(p, p)] * a[SYM(q, q)])) && (o2 > floor2);
            }
        if (!more) break;   // also leaves on NaN
        jacobi_sweep(a, V);
    }
}

// out = V diag(f) V^T (symmetric, 10 entries)
STE_DEV void sym_from_eig(const double (&V)[16], const double (&f)[4], double (&out)[10]) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = i; j < 4; ++j) {
            double acc = 0.0;
#pragma unroll
            for (int k = 0; k < 4; ++k) acc = fma(V[i * 4 + k] * f[k], V[j * 4 + k], acc);
            out[SYM(i, j)] = acc;
        }
}

// Rare path of sqrt_psd4 for slowly converging, (near-)singular or indefinite matrices: a fresh
// Jacobi iteration to rounding level and the root of the clamped spectrum.  Out of line, and fed
// BY VALUE, so that the hot path keeps its matrices in registers (taking the address of the hot
// arrays made the compiler mirror them on the stack every step).
STE_COLD bool sqrt_psd4_cold(double a0, double a1, double a2, double a3, double a4, double a5, double a6, double a7,
                             double a8, double a9, double *M_out) {
    double a[10] = {a0, a1, a2, a3, a4, a5, a6, a7, a8, a9}, V[16], f[4], M[10];
    jacobi_eig4<true>(a, V, kJacobiTight);
    const double w[4] = {a[SYM(0, 0)], a[SYM(1, 1)], a[SYM(2, 2)], a[SYM(3, 3)]};
    const double wmax = fmax(fmax(fabs(w[0]), fabs(w[1])), fmax(fabs(w[2]), fabs(w[3])));
    bool clamped = false;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        clamped |= (w[k] < -1e-13 * wmax);
        f[k] = fast_sqrt(fmax(w[k], 0.0));
    }
    sym_from_eig(V, f, M);
#pragma unroll
    for (int i = 0; i < 10; ++i) M_out[i] = M[i];
    return clamped;
}

// M = Re sqrtm(scale * A): principal square root with negative eigenvalues contributing 0
// (scipy returns a complex root there and numpy's float assignment drops the imaginary part,
// unscented.py:104-105).  Returns true if a negative eigenvalue was clamped.
//
// Covariances of a running filter are strongly graded and cyclic Jacobi converges faster than
// quadratically on them, so the sweeps stop as soon as the matrix is ALMOST diagonal,
// eps = max |a_pq| / sqrt(a_pp a_qq) <= 1e-4, and the root of D + E is finished by its
// perturbation series, which has no small denominators (sums of root eigenvalues, never gaps):
//     sqrt(D + E) = sqrt(D) + X1 + X2 + O(eps^3),   X1_ij = E_ij / (s_i + s_j),
//     X2_ij = -(X1 X1)_ij / (s_i + s_j),             s = sqrt(diag D);
// the neglected term is below 1e-12 of the smaller root eigenvalue (measured on filter
// covariances: 4e-14).  One sweep is enough when every predict follows an update (eps at a median
// of 2.5e-6 then, 99.98 % below 1e-4 on the benchmark tracks), two to four with sub-steps or
// irregular updates (config-4 shape, measured on the host build: 1 % / 46 % / 52 % / 0.6 % of the
// roots take 1 / 2 / 3 / 4 sweeps, 0.01 % the out-of-line finish).  No eigenvector matrix is accumulated: the sweeps leave their rotation
// parameters (c, s) in scratch (kSweepSlots per sweep, kSqrtRotSlots in all, starting at slot
// `rot`) and the root S of the rotated matrix is carried back, M = J_1 (... (J_n S J_n^T) ...) J_1^T,
// rotation by rotation on its 10 unique entries - 114 FP64 operations per sweep instead of 96 for
// the accumulation plus 104 for V S V^T, and 32 registers fewer across the sweeps.
// Anything else - singular, indefinite, slowly converging - goes to the out-of-line finish.
#ifndef STE_SQRT_SERIES_EPS2
#define STE_SQRT_SERIES_EPS2 1e-8
#endif
#if defined(STE_EMUL_STATS) && !defined(__CUDA_ARCH__)
static long long ste_emul_sweep_hist[8] = {0, 0, 0, 0, 0, 0, 0, 0};
static unsigned char *ste_emul_sweep_log = nullptr;   // developer sandbox only: sweeps of every root in call order (0 = cold path)
static long long ste_emul_sweep_log_n = 0, ste_emul_sweep_log_cap = 0;
#endif
constexpr double kSqrtSeriesEps2 = STE_SQRT_SERIES_EPS2;     // eps^2 limit of the series finish
#ifndef STE_SQRT_MAX_SWEEPS
#define STE_SQRT_MAX_SWEEPS 4
#endif
constexpr int kSqrtMaxSweeps = STE_SQRT_MAX_SWEEPS;
constexpr int kSqrtRotSlots = kSqrtMaxSweeps * kSweepSlots;

STE_DEV bool jacobi_off_within(const double (&a)[10], double eps2) {
    const double w[4] = {a[SYM(0, 0)], a[SYM(1, 1)], a[SYM(2, 2)], a[SYM(3, 3)]};
    // every diagonal entry against 1e-12 of the trace (wmax <= trace <= 4 wmax on a positive diagonal): no max / min chains
    const double lim = 1e-12 * ((w[0] + w[1]) + (w[2] + w[3]));
    bool ok = lim > 0.0;             // false on NaN and on a non-positive trace
#pragma unroll
    for (int k = 0; k < 4; ++k) ok &= w[k] > lim;
#pragma unroll
    for (int p = 0; p < 3; ++p)
#pragma unroll
        for (int q = p + 1; q < 4; ++q) ok &= (a[SYM(p, q)] * a[SYM(p, q)] <= eps2 * (w[p] * w[q]));
    return ok;
}

STE_DEV bool sqrt_psd4(const double (&A)[10], double scale, double (&M)[10], const Scratch &sc, const int rot) {
    double a[10];
#pragma unroll
    for (int i = 0; i < 10; ++i) a[i] = A[i] * scale;
    bool series_ok = false;
    int sweeps = 0;
#pragma unroll 1
    while (sweeps < kSqrtMaxSweeps) {
        jacobi_sweep_store(a, sc, rot + sweeps * kSweepSlots);
        ++sweeps;
        if ((series_ok = jacobi_off_within(a, kSqrtSeriesEps2))) break;
    }
#if defined(STE_EMUL_STATS) && !defined(__CUDA_ARCH__)
    ++ste_emul_sweep_hist[series_ok ? sweeps : 0];   // developer sandbox only: sweeps per root, [0] = cold path
    if (ste_emul_sweep_log && ste_emul_sweep_log_n < ste_emul_sweep_log_cap) ste_emul_sweep_log[ste_emul_sweep_log_n++] = (unsigned char)(series_ok ? sweeps : 0);
    if (!series_ok) {
        const double wmx = fmax(fmax(a[0], a[4]), fmax(a[7], a[9])), wmn = fmin(fmin(a[0], a[4]), fmin(a[7], a[9]));
        ++ste_emul_sweep_hist[wmn < 0.0 ? 4 : (wmn > 1e-12 * wmx ? 6 : 5)];   // negative / tiny / off-diagonals still large
    }
#endif
    if (!series_ok) {
        double Mt[10];
        const bool clamped = sqrt_psd4_cold(A[0] * scale, A[1] * scale, A[2] * scale, A[3] * scale, A[4] * scale, A[5] * scale,
                                            A[6] * scale, A[7] * scale, A[8] * scale, A[9] * scale, Mt);
#pragma unroll
        for (int i = 0; i < 10; ++i) M[i] = Mt[i];
        return clamped;
    }
    // s_i = sqrt(d_i) and 1 / s_i from one reciprocal square root each
    double w[4], rs[4], sd[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) w[k] = a[SYM(k, k)];
    fast_rsqrt_v<4>(w, rs);
#pragma unroll
    for (int k = 0; k < 4; ++k) sd[k] = w[k] * rs[k];   // within 2 ulp of the root (rs is good to 2^-60); no correction step
    // pair sums and their reciprocals, pairs in SYM order: (0,1) (0,2) (0,3) (1,2) (1,3) (2,3)
    double ssum[6], rsum[6], X[10], G[10];
    {
        int k = 0;
#pragma unroll
        for (int p = 0; p < 3; ++p)
#pragma unroll
            for (int q = p + 1; q < 4; ++q) ssum[k++] = sd[p] + sd[q];
    }
    // 2^-40 relative is enough: the reciprocals only multiply off-diagonal terms that are <= 1e-4 of the smaller root
    // eigenvalue of their pair, so their error stays below 1e-16 of it
    fast_rcp_v<6, 1>(ssum, rsum);
    {
        int k = 0;
#pragma unroll
        for (int p = 0; p < 3; ++p)
#pragma unroll
            for (int q = p + 1; q < 4; ++q) X[SYM(p, q)] = a[SYM(p, q)] * rsum[k++];   // X1 (zero diagonal)
    }
#pragma unroll
    for (int p = 0; p < 4; ++p) X[SYM(p, p)] = 0.0;
    // G = X1 X1 (symmetric)
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
        for (int q = p; q < 4; ++q) {
            double acc = 0.0;
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (k != p && k != q) acc = fma(X[SYM(p, k)], X[SYM(k, q)], acc);
            G[SYM(p, q)] = acc;
        }
    // S = sqrt(D) + X1 + X2, written into M and carried back to the original basis in place
    {
        int k = 0;
#pragma unroll
        for (int p = 0; p < 3; ++p)
#pragma unroll
            for (int q = p + 1; q < 4; ++q) M[SYM(p, q)] = fma(-G[SYM(p, q)], rsum[k++], X[SYM(p, q)]);
    }
#pragma unroll
    for (int p = 0; p < 4; ++p) M[SYM(p, p)] = fma(-G[SYM(p, p)], 0.5 * rs[p], sd[p]);
#pragma unroll 1
    while (sweeps > 0) {
        --sweeps;
        jacobi_unsweep(M, sc, rot + sweeps * kSweepSlots);
    }
    return false;
}

// Innovation statistics of one update, formed by the INNOV instantiations from what the update already holds: the
// innovation y = z - H x (after the noise draw and the heading wrap), the S = H P H^T + rs R whose pseudo-inverse it
// applied, and that pseudo-inverse's factorisation.  nis = y^T S^+ y; log_pdet = sum of log(lambda) over the rank
// eigenvalues S^+ kept (NaN when one of them is negative).
struct Innov {
    double nis, log_pdet;
    int rank;
};

// Moore-Penrose inverse of a symmetric 4x4 with numpy's cutoff: singular values (|eigenvalues|)
// <= rcond * max are treated as zero.  Returns the number of dropped eigenvalues.  INNOV: also the
// log pseudo-determinant, the sum of log(w) over the kept eigenvalues (NaN when one is negative).
template <bool INNOV = false>
STE_DEV int pinv_sym4(const double (&A)[10], double (&Ainv)[10], double *log_pdet = nullptr) {
    double a[10], V[16], f[4];
#pragma unroll
    for (int i = 0; i < 10; ++i) a[i] = A[i];
    jacobi_eig4<true>(a, V, kJacobiTight);
    const double w[4] = {a[SYM(0, 0)], a[SYM(1, 1)], a[SYM(2, 2)], a[SYM(3, 3)]};
    const double wmax = fmax(fmax(fabs(w[0]), fabs(w[1])), fmax(fabs(w[2]), fabs(w[3])));
    const double cut = kPinvRcond * wmax;
    int dropped = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const bool keep = fabs(w[k]) > cut;
        f[k] = keep ? fast_rcp(w[k]) : 0.0;
        dropped += keep ? 0 : 1;
    }
    if constexpr (INNOV) {
        double lp = 0.0;
#pragma unroll
        for (int k = 0; k < 4; ++k) lp += fabs(w[k]) > cut ? log(w[k]) : 0.0;
        *log_pdet = lp;
    }
    sym_from_eig(V, f, Ainv);
    return dropped;
}

STE_COLD int pinv_sym4_cold(const double *A_in, double *Ainv_out) {
    double A[10], Ainv[10];
#pragma unroll
    for (int i = 0; i < 10; ++i) A[i] = A_in[i];
    const int dropped = pinv_sym4(A, Ainv);
#pragma unroll
    for (int i = 0; i < 10; ++i) Ainv_out[i] = Ainv[i];
    return dropped;
}

// pinv of a symmetric 4x4 that is normally positive definite and well conditioned (the smoother's
// P_b): root-free LDL^T, A^-1 = L^-T D^-1 L^-1, ~90 FP64 operations.  For a full-rank matrix the
// pseudo-inverse IS the inverse.  If a pivot loses more than ~7 digits against its diagonal entry
// (ill-conditioned, singular or indefinite matrix) the eigen-decomposition path with numpy's
// cutoff semantics takes over.  Returns the number of dropped eigenvalues.
STE_DEV int pinv_spd4(const double (&A)[10], double (&Ainv)[10]) {
    const double a00 = A[0], a10 = A[1], a20 = A[2], a30 = A[3], a11 = A[4], a21 = A[5], a31 = A[6], a22 = A[7],
                 a32 = A[8], a33 = A[9];
    const double d0 = a00, r0 = fast_rcp(d0);
    const double l10 = a10 * r0, l20 = a20 * r0, l30 = a30 * r0;
    const double d1 = fma(-l10, a10, a11), r1 = fast_rcp(d1);
    const double l21 = fma(-l20, a10, a21) * r1, l31 = fma(-l30, a10, a31) * r1;
    const double d2 = fma(-l21 * d1, l21, fma(-l20, a20, a22)), r2 = fast_rcp(d2);
    const double l32 = fma(-l31 * d1, l21, fma(-l30, a20, a32)) * r2;
    const double d3 = fma(-l32 * d2, l32, fma(-l31 * d1, l31, fma(-l30, a30, a33)));
    const double r3 = fast_rcp(d3);
    const double kTol = 1e-7;
    const bool ok = (d0 > 0.0) && (d1 > kTol * a11) && (d2 > kTol * a22) && (d3 > kTol * a33) && (d0 < 1e300);
    if (!ok) {
        double tmp_in[10], tmp_out[10];
#pragma unroll
        for (int i = 0; i < 10; ++i) tmp_in[i] = A[i];
        const int dropped = pinv_sym4_cold(tmp_in, tmp_out);
#pragma unroll
        for (int i = 0; i < 10; ++i) Ainv[i] = tmp_out[i];
        return dropped;
    }
    // N = L^-1 (unit lower triangular): n10, n20, n21, n30, n31, n32
    const double n10 = -l10, n21 = -l21, n32 = -l32;
    const double n20 = fma(l21, l10, -l20);
    const double n31 = fma(l32, l21, -l31);
    const double n30 = fma(-l32, n20, fma(l31, l10, -l30));
    // A^-1 = N^T diag(r) N
    const double t10 = n10 * r1, t20 = n20 * r2, t21 = n21 * r2, t30 = n30 * r3, t31 = n31 * r3, t32 = n32 * r3;
    Ainv[SYM(3, 3)] = r3;
    Ainv[SYM(2, 3)] = t32;
    Ainv[SYM(1, 3)] = t31;
    Ainv[SYM(0, 3)] = t30;
    Ainv[SYM(2, 2)] = fma(t32, n32, r2);
    Ainv[SYM(1, 2)] = fma(t31, n32, t21);
    Ainv[SYM(0, 2)] = fma(t30, n32, t20);
    Ainv[SYM(1, 1)] = fma(t31, n31, fma(t21, n21, r1));
    Ainv[SYM(0, 1)] = fma(t30, n31, fma(t20, n21, t10));
    Ainv[SYM(0, 0)] = fma(t30, n30, fma(t20, n20, fma(t10, n10, r0)));
    return 0;
}

// Pseudo-inverse of a symmetric 2x2 [a b; b c] with the same cutoff rule (one Jacobi rotation
// diagonalises a 2x2 exactly).  `floor_sv` is an extra singular value taking part in the
// max (0 when the 2x2 is the only non-zero block of the full matrix).
template <bool INNOV>
STE_DEV int pinv_sym2_eig_impl(double a, double b, double c, double *inv, double *log_pdet) {
    const double d = c - a;
    const double bb = b + b;
    const double h = fast_sqrt(fma(d, d, bb * bb));
    double t = fast_div(d >= 0.0 ? bb : -bb, fabs(d) + h);
    t = (b == 0.0) ? 0.0 : t;
    const double cs = fast_rsqrt(fma(t, t, 1.0));
    const double sn = t * cs;
    const double w0 = fma(-t, b, a), w1 = fma(t, b, c);
    const double cut = kPinvRcond * fmax(fabs(w0), fabs(w1));
    const bool k0 = fabs(w0) > cut, k1 = fabs(w1) > cut;
    const double f0 = k0 ? fast_rcp(w0) : 0.0, f1 = k1 ? fast_rcp(w1) : 0.0;
    // eigenvectors: v0 = (c, -s), v1 = (s, c)
    inv[0] = fma(cs * f0, cs, sn * f1 * sn);
    inv[1] = fma(-cs * f0, sn, sn * f1 * cs);
    inv[2] = fma(sn * f0, sn, cs * f1 * cs);
    if constexpr (INNOV) *log_pdet = (k0 ? log(w0) : 0.0) + (k1 ? log(w1) : 0.0);
    return (k0 ? 0 : 1) + (k1 ? 0 : 1);
}
STE_COLD int pinv_sym2_eig(double a, double b, double c, double *inv) { return pinv_sym2_eig_impl<false>(a, b, c, inv, nullptr); }
STE_COLD int pinv_sym2_eig_innov(double a, double b, double c, double *inv, double *log_pdet) {
    return pinv_sym2_eig_impl<true>(a, b, c, inv, log_pdet);
}

// Hot path: S22 = P22 + R22 of a running filter is positive definite and well conditioned (R adds
// to its diagonal), so the pseudo-inverse is the inverse, adj(S) / det(S): one reciprocal on the
// critical path instead of two dependent square roots.  det = a c - b^2 is formed with an exact
// product error term; anything that is not clearly positive definite (det <= 1e-8 a c, i.e. the
// two rows closer than ~1e-4 rad to parallel, or a non-positive diagonal) takes the
// eigen-decomposition with numpy's cutoff semantics.  INNOV: also the log pseudo-determinant of the
// factorisation taken (log det here, the kept eigenvalues' logs on the eigen branch).
template <bool INNOV = false>
STE_DEV int pinv_sym2(double a, double b, double c, double (&inv)[3], double *log_pdet = nullptr) {
    const double ac = a * c;
    const double det = fma(-b, b, ac) + fma(a, c, -ac);
    if (!(a > 0.0 && c > 0.0 && det > 1e-8 * ac)) {
        double t[3];
        int dropped;
        if constexpr (INNOV) dropped = pinv_sym2_eig_innov(a, b, c, t, log_pdet);
        else dropped = pinv_sym2_eig(a, b, c, t);
        inv[0] = t[0];
        inv[1] = t[1];
        inv[2] = t[2];
        return dropped;
    }
    if constexpr (INNOV) *log_pdet = log(det);
    const double r = fast_rcp(det);
    inv[0] = c * r;
    inv[1] = -b * r;
    inv[2] = a * r;
    return 0;
}

// ------------------------------------------------------------------------------------------ //
// Process model: great-circle propagation on the sphere (non_linear_process.py:54-78).
//
// The reference evaluates lat' = asin(s), s = sin(phi) cos(delta) + cos(phi) sin(delta) cos(alpha).
// (east, north, s) is the unit vector of the new position in the frame of the old meridian, so
// cos(lat') = hypot(east, north) and lat' = atan2(s, hypot(east, north)): the same angle, well
// conditioned up to the poles, and it reuses the one-division atan2 (no separate asin code).
//
// The nine sigma points of a step are x, x + m_c, x - m_c (c = 0..3).  Their three angles
// (latitude, course, angular distance) are therefore theta_0 and theta_0 +/- eps_c, and
//     sin(theta_0 +/- eps) = sin theta_0 cos eps +/- cos theta_0 sin eps          (same for cos)
// so a step needs sincos of 3 centre angles and 12 offsets (15 evaluations) instead of 27.
// AngleTrig carries (sin, cos) of the three angles.
//
// LIB = false: the branch-free functions of ste_fastmath.cuh (hot path; the caller has checked
// the argument range for this step).  LIB = true: the CUDA math library, same formulas (cold path).
// ------------------------------------------------------------------------------------------ //
struct AngleTrig {
    double sp, cp;   // latitude
    double sa, ca;   // course over ground
    double sd, cd;   // angular distance u dt / R
};

// SMALL_DIST: the caller has bounded the angular distance |u dt / R| by kSmallAngle (step_is_small: 2^-6), so its sine and
// cosine come from the short series (no range reduction, no quadrant selects)
template <bool LIB, bool SMALL_DIST = false>
STE_DEV AngleTrig angle_trig(double lat_deg, double cog_deg, double u, double dtR) {
    AngleTrig t;
    if (LIB) {
        sincos(lat_deg * kDegToRad, &t.sp, &t.cp);
        sincos(cog_deg * kDegToRad, &t.sa, &t.ca);
        sincos(u * dtR, &t.sd, &t.cd);
    } else if constexpr (SMALL_DIST) {
        const double ang[2] = {lat_deg * kDegToRad, cog_deg * kDegToRad}, dist[1] = {u * dtR};
        double sn[2], cs[2], sd[1], cd[1];
        fast_sincos_v<2>(ang, sn, cs);
        small_sincos_v<1>(dist, sd, cd);
        t.sp = sn[0]; t.cp = cs[0]; t.sa = sn[1]; t.ca = cs[1]; t.sd = sd[0]; t.cd = cd[0];
    } else {
        const double ang[3] = {lat_deg * kDegToRad, cog_deg * kDegToRad, u * dtR};
        double sn[3], cs[3];
        fast_sincos_v<3>(ang, sn, cs);
        t.sp = sn[0]; t.cp = cs[0]; t.sa = sn[1]; t.ca = cs[1]; t.sd = sn[2]; t.cd = cs[2];
    }
    return t;
}

// trig of the three offset angles of one root column: the short series, replaced by the full-range
// evaluation only when an offset is not small (a wide course or latitude spread)
// KNOWN_SMALL: the caller has bounded all three offsets by kSmallAngle for this step (step_is_small)
template <bool LIB, bool KNOWN_SMALL = false>
STE_DEV AngleTrig offset_trig(double dlat_deg, double dcog_deg, double du, double dtR) {
    if (LIB) return angle_trig<LIB>(dlat_deg, dcog_deg, du, dtR);
    const double ang[3] = {dlat_deg * kDegToRad, dcog_deg * kDegToRad, du * dtR};
    AngleTrig t;
    double sn[3], cs[3];
    if constexpr (KNOWN_SMALL) {
        small_sincos_v<3>(ang, sn, cs);
    } else {
        // decide first, then evaluate ONE of the two: both arms write the same six values (no merge copies on the common arm)
        const bool small = fabs(ang[0]) <= kSmallAngle && fabs(ang[1]) <= kSmallAngle && fabs(ang[2]) <= kSmallAngle;
        if (__builtin_expect(small, 1)) small_sincos_v<3>(ang, sn, cs);
        else fast_sincos_v<3>(ang, sn, cs);
    }
    t.sp = sn[0]; t.cp = cs[0]; t.sa = sn[1]; t.ca = cs[1]; t.sd = sn[2]; t.cd = cs[2];
    return t;
}

// trig of (base + off) and (base - off) from the four shared products per angle
STE_DEV void angle_add_pair(const AngleTrig &b, const AngleTrig &o, AngleTrig &plus, AngleTrig &minus) {
    double sc_, cs_, cc_, ss_;
    sc_ = b.sp * o.cp; cs_ = b.cp * o.sp; cc_ = b.cp * o.cp; ss_ = b.sp * o.sp;
    plus.sp = sc_ + cs_; minus.sp = sc_ - cs_; plus.cp = cc_ - ss_; minus.cp = cc_ + ss_;
    sc_ = b.sa * o.ca; cs_ = b.ca * o.sa; cc_ = b.ca * o.ca; ss_ = b.sa * o.sa;
    plus.sa = sc_ + cs_; minus.sa = sc_ - cs_; plus.ca = cc_ - ss_; minus.ca = cc_ + ss_;
    sc_ = b.sd * o.cd; cs_ = b.cd * o.sd; cc_ = b.cd * o.cd; ss_ = b.sd * o.sd;
    plus.sd = sc_ + cs_; minus.sd = sc_ - cs_; plus.cd = cc_ - ss_; minus.cd = cc_ + ss_;
}

// Propagate NP sigma points at once: x[i] = [lon, lat, u, cog], t[i] = trig of its (lat, cog, u dt/R).
// All 2*NP angles (longitude increments, latitudes) go through one lock-step atan2.
//
// SMALL (the caller has checked step_is_small): every point moves by an angular distance
// <= 2^-6 rad (100 km) and stays below 76 degrees of latitude.  Then the longitude increment is
// atan(east/north) with |east/north| <= 0.0645, cos(lat2) = north sqrt(1 + (east/north)^2), and the
// latitude INCREMENT is asin(up cos(lat1) - cos(lat2) sin(lat1)) with |.| <= 2^-6: three short
// Maclaurin series replace the square root and the two full-range atan2 (no selects, 40 % fewer
// FP64 operations per point).
template <bool LIB, int NP, bool SMALL = false>
STE_DEV void geodetic_finish_n(const double (&x)[NP][4], const AngleTrig (&t)[NP], double dt, double sog_rate,
                               double cog_rate, double (&y)[NP][4]) {
    if constexpr (!LIB && SMALL) {
        // sin(lat2 - lat1) = up cos(lat1) - cos(lat2) sin(lat1) with cos(lat2) = north sqrt(1 + q^2).  Since
        // up cos(lat1) - north sin(lat1) = sin(delta) cos(alpha) identically, it equals
        //     sin(delta) cos(alpha) - sin(lat1) north (sqrt(1 + q^2) - 1):
        // no cancellation between two O(1) products, and `up` is never formed.
        double east[NP], north[NP], sdca[NP], q[NP], e[NP], g[NP], dlon[NP], sdel[NP], dlat[NP];
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            sdca[i] = t[i].sd * t[i].ca;
            east[i] = t[i].sd * t[i].sa;
            north[i] = fma(t[i].cp, t[i].cd, -t[i].sp * sdca[i]);
        }
        fast_div_v<NP>(east, north, q);
#pragma unroll
        for (int i = 0; i < NP; ++i) e[i] = q[i] * q[i];
        small_hypot_excess_v<NP>(north, e, g);     // cos(lat2) - north
        small_atan_v<NP>(q, e, dlon);
#pragma unroll
        for (int i = 0; i < NP; ++i) sdel[i] = fma(-t[i].sp, g[i], sdca[i]);
        small_asin_v<NP>(sdel, dlat);
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            y[i][0] = fma(x[i][0], kDegToRad, dlon[i]) * kRadToDeg;
            y[i][1] = fma(dlat[i], kRadToDeg, x[i][1]);
            y[i][2] = fma(sog_rate, dt, x[i][2]);
            y[i][3] = fma(cog_rate, dt, (x[i][3] * kDegToRad) * kRadToDeg);
        }
    } else {
        double ay[2 * NP], ax[2 * NP], ang[2 * NP], h2[NP], h[NP];
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            const double east = t[i].sd * t[i].sa;
            const double sdca = t[i].sd * t[i].ca;
            const double north = fma(t[i].cp, t[i].cd, -t[i].sp * sdca);
            ay[i] = east;
            ax[i] = north;
            ay[NP + i] = fma(t[i].sp, t[i].cd, t[i].cp * sdca);   // up
            h2[i] = fma(east, east, north * north);
        }
        if (LIB) {
#pragma unroll
            for (int i = 0; i < NP; ++i) ax[NP + i] = sqrt(h2[i]);
#pragma unroll
            for (int i = 0; i < 2 * NP; ++i) ang[i] = atan2(ay[i], ax[i]);
        } else {
            fast_sqrt_v<NP>(h2, h);
#pragma unroll
            for (int i = 0; i < NP; ++i) ax[NP + i] = h[i];
            fast_atan2_v<2 * NP, NP>(ay, ax, ang);   // lanes NP.. are latitudes: (up, hypot) is a unit vector with hypot >= 0
        }
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            y[i][0] = fma(x[i][0], kDegToRad, ang[i]) * kRadToDeg;
            y[i][1] = ang[NP + i] * kRadToDeg;
            y[i][2] = fma(sog_rate, dt, x[i][2]);
            y[i][3] = fma(cog_rate, dt, (x[i][3] * kDegToRad) * kRadToDeg);
        }
    }
}

template <bool LIB, bool SMALL = false>
STE_DEV void geodetic_finish(const double (&x)[4], const AngleTrig &t, double dt, double sog_rate,
                             double cog_rate, double (&y)[4]) {
    double xs[1][4], ys[1][4];
    AngleTrig ts[1] = {t};
#pragma unroll
    for (int r = 0; r < 4; ++r) xs[0][r] = x[r];
    geodetic_finish_n<LIB, 1, SMALL>(xs, ts, dt, sog_rate, cog_rate, ys);
#pragma unroll
    for (int r = 0; r < 4; ++r) y[r] = ys[0][r];
}

// one stand-alone evaluation (geodetic_dynamics called directly, ste_geodetic_f64)
STE_DEV void geodetic_step(const double (&x)[4], double dt, double dtR, double sog_rate,
                           double cog_rate, double (&y)[4]) {
    const bool in_range = fabs(x[1]) * kDegToRad <= kSinCosMaxArg && fabs(x[3]) * kDegToRad <= kSinCosMaxArg &&
                          fabs(x[2] * dtR) <= kSinCosMaxArg;
    if (in_range)
        geodetic_finish<false>(x, angle_trig<false>(x[1], x[3], x[2], dtR), dt, sog_rate, cog_rate, y);
    else
        geodetic_finish<true>(x, angle_trig<true>(x[1], x[3], x[2], dtR), dt, sog_rate, cog_rate, y);
}

}  // namespace ste
